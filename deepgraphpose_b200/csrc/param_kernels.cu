// Parameter-arena kernels (sm_100a): fp32 master -> 16-bit tensor-core operands, frozen-BN scale/shift, the transposed
// (dgrad) weight matrices, and the optimizer of fit_dgp (reference: src/deepgraphpose/models/fitdgp.py:706-713 --
// MomentumOptimizer(lr, 0.9) on gradients clipped by global norm 10).  All of them are flat, HBM-bound passes over the
// arena with 128-bit accesses; reductions use a fixed two-stage order (bitwise reproducible).
#include "half_utils.cuh"
#include "kernels.cuh"

namespace dgp {

namespace {

__device__ __forceinline__ uint32_t pack16(float a, float b, int fp16) { return h16::pack2(a, b, fp16); }
__device__ __forceinline__ uint16_t cvt16(float a, int fp16) { return h16::cvt1(a, fp16); }

// w16[i] = round16(master[i]) over the weight part of the arena (n multiple of 8)
__global__ void refresh_w16_kernel(const float4* __restrict__ master, uint4* __restrict__ w16, size_t n8, int fp16) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
    const float4 a = master[2 * i], b = master[2 * i + 1];
    w16[i] = make_uint4(pack16(a.x, a.y, fp16), pack16(a.z, a.w, fp16), pack16(b.x, b.y, fp16), pack16(b.z, b.w, fp16));
  }
}

// slim batch_norm(is_training=False): scale = gamma / sqrt(var + eps), shift = beta - mean * scale
__global__ void refresh_bn_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                                  const float* __restrict__ mean, const float* __restrict__ var, float eps, int n,
                                  float* __restrict__ scale, float* __restrict__ shift) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float s = gamma[i] / sqrtf(var[i] + eps);
  scale[i] = s;
  shift[i] = beta[i] - mean[i] * s;
}

// Data-gradient operand of one conv: wd[ci][T-1-tap][co] = round16(w[co][tap][ci] * scale[co])  (the BN scale of the
// output channel is folded in, so the dgrad GEMM consumes dy = dL/d(BN output) directly).  Per tap this is a
// Cout x Cin -> Cin x Cout transpose: 32 x 32 tiles through shared memory, coalesced on both sides.
__global__ void __launch_bounds__(256) build_dgrad_w_kernel(const DgradWJob* __restrict__ jobs, int njobs,
                                                            const float* __restrict__ master,
                                                            const float* __restrict__ scale_arena, int fp16) {
  __shared__ float tile[32][33];
  // all layers in ONE launch: a block finds its layer from the prefix of 32x32-tile counts (<= kDgradWMaxJobs entries,
  // ascending, first one 0; 52 at ResNet-50, 154 at ResNet-152).  Thread t tests entry t and the block counts the hits -- one
  // load latency instead of a serial walk of up to njobs dependent loads per block (that walk was most of this kernel's 90 us).
  const int hit = (int)threadIdx.x < njobs && (int)blockIdx.x >= jobs[threadIdx.x].tile_start;
  const int job = __syncthreads_count(hit) - 1;
  const DgradWJob jb = jobs[job];
  const int local = (int)blockIdx.x - jb.tile_start;
  const int tx_n = jb.Cin / 32, ty_n = jb.Cout / 32;
  const int tap = local / (tx_n * ty_n);
  const int rem = local - tap * (tx_n * ty_n);
  const int co0 = (rem / tx_n) * 32, ci0 = (rem - (rem / tx_n) * tx_n) * 32;
  const float* w = master + jb.w_off;
  const float* scale = scale_arena + jb.ch_off;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const size_t K = (size_t)jb.taps * jb.Cin, Kd = (size_t)jb.taps * jb.Cout;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int co = co0 + ty + 8 * j;
    tile[ty + 8 * j][tx] = w[(size_t)co * K + (size_t)tap * jb.Cin + ci0 + tx] * scale[co];
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int ci = ci0 + ty + 8 * j;
    jb.wd[(size_t)ci * Kd + (size_t)(jb.taps - 1 - tap) * jb.Cout + co0 + tx] = cvt16(tile[tx][ty + 8 * j], fp16);
  }
}

// Head dgrad operand: whT[c][r] = round16(wh[r][c]) for r < rows, zero for rows <= r < Kd.
__global__ void build_head_dgrad_w_kernel(const float* __restrict__ wh, int rows, int C, uint16_t* __restrict__ whT,
                                          int Kd, int fp16) {
  const size_t total = (size_t)C * Kd;
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(t % (size_t)Kd);
    const int c = (int)(t / (size_t)Kd);
    whT[t] = cvt16(r < rows ? wh[(size_t)r * C + c] : 0.0f, fp16);
  }
}

constexpr int kNormBlocks = 592;  // 4 per SM

__global__ void sqnorm_partial_kernel(const float4* __restrict__ g, size_t n4, float* __restrict__ partial) {
  float acc = 0.0f;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 v = g[i];
    acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  __shared__ float sm[256];
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) sm[threadIdx.x] += sm[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[blockIdx.x] = sm[0];
}

// out[0] = global norm, out[1] = clip factor clip / max(norm, clip)  (tf.clip_by_global_norm)
__global__ void sqnorm_final_kernel(const float* __restrict__ partial, int n, float grad_scale, float clip,
                                    float* __restrict__ out) {
  __shared__ float sm[1024];
  float acc = 0.0f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += partial[i];
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) sm[threadIdx.x] += sm[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const float norm = sqrtf(sm[0]) * fabsf(grad_scale);
    out[0] = norm;
    out[1] = clip > 0.0f ? clip / fmaxf(norm, clip) : 1.0f;
  }
}

// accum = momentum * accum + g';  w -= lr * accum;  g' = g * grad_scale * clip_factor
__global__ void momentum_step_kernel(float4* __restrict__ w, float4* __restrict__ accum, const float4* __restrict__ g,
                                     size_t n4, float lr, float momentum, float grad_scale,
                                     const float* __restrict__ norm_clip) {
  const float f = grad_scale * norm_clip[1];
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 gg = g[i];
    float4 a = accum[i];
    float4 ww = w[i];
    a.x = momentum * a.x + gg.x * f; a.y = momentum * a.y + gg.y * f;
    a.z = momentum * a.z + gg.z * f; a.w = momentum * a.w + gg.w * f;
    ww.x -= lr * a.x; ww.y -= lr * a.y; ww.z -= lr * a.z; ww.w -= lr * a.w;
    accum[i] = a;
    w[i] = ww;
  }
}

int flat_grid(size_t n, int threads) {
  size_t g = (n + threads - 1) / threads;
  if (g > 148 * 8) g = 148 * 8;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

cudaError_t launch_refresh_w16(const float* master, void* w16, size_t n, int fp16, cudaStream_t s) {
  if (n % 8) return cudaErrorInvalidValue;
  refresh_w16_kernel<<<flat_grid(n / 8, 256), 256, 0, s>>>(reinterpret_cast<const float4*>(master),
                                                           reinterpret_cast<uint4*>(w16), n / 8, fp16);
  return cudaGetLastError();
}

cudaError_t launch_refresh_bn(const float* gamma, const float* beta, const float* mean, const float* var, float eps, int n,
                              float* scale, float* shift, cudaStream_t s) {
  refresh_bn_kernel<<<(n + 255) / 256, 256, 0, s>>>(gamma, beta, mean, var, eps, n, scale, shift);
  return cudaGetLastError();
}

cudaError_t launch_build_dgrad_w(const DgradWJob* jobs_dev, int njobs, int total_tiles, const float* master,
                                 const float* scale_arena, int fp16, cudaStream_t s) {
  if (njobs < 1 || total_tiles < 1) return cudaSuccess;
  if (njobs > kDgradWMaxJobs) return cudaErrorInvalidValue;   // the kernel's job lookup is one thread per job
  build_dgrad_w_kernel<<<total_tiles, 256, 0, s>>>(jobs_dev, njobs, master, scale_arena, fp16);
  return cudaGetLastError();
}

cudaError_t launch_build_head_dgrad_w(const float* wh, int rows, int C, void* whT, int Kd, int fp16, cudaStream_t s) {
  build_head_dgrad_w_kernel<<<flat_grid((size_t)C * Kd, 256), 256, 0, s>>>(wh, rows, C, reinterpret_cast<uint16_t*>(whT),
                                                                            Kd, fp16);
  return cudaGetLastError();
}

int sqnorm_partials() { return kNormBlocks; }

cudaError_t launch_global_norm(const float* g, size_t n, float grad_scale, float clip, float* partial, float* norm_clip,
                               cudaStream_t s) {
  if (n % 4) return cudaErrorInvalidValue;
  sqnorm_partial_kernel<<<kNormBlocks, 256, 0, s>>>(reinterpret_cast<const float4*>(g), n / 4, partial);
  sqnorm_final_kernel<<<1, 1024, 0, s>>>(partial, kNormBlocks, grad_scale, clip, norm_clip);
  return cudaGetLastError();
}

cudaError_t launch_momentum_step(float* w, float* accum, const float* g, size_t n, float lr, float momentum,
                                 float grad_scale, const float* norm_clip, cudaStream_t s) {
  if (n % 4) return cudaErrorInvalidValue;
  momentum_step_kernel<<<flat_grid(n / 4, 256), 256, 0, s>>>(reinterpret_cast<float4*>(w), reinterpret_cast<float4*>(accum),
                                                             reinterpret_cast<const float4*>(g), n / 4, lr, momentum,
                                                             grad_scale, norm_clip);
  return cudaGetLastError();
}

}  // namespace dgp
