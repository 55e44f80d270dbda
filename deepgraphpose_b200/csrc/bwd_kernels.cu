// Bandwidth-class kernels of the network backward pass (sm_100a); the GEMM-shaped parts (dgrad, wgrad) run on
// conv_gemm_sm100.cu / wgrad_gemm_sm100.cu.  Reference: the gradients TF derives for
// optimizer.compute_gradients(total_loss, TF.trainable_variables()) (src/deepgraphpose/models/fitdgp.py:706-713) through
// slim resnet_v1_50 with is_training=False (frozen moving statistics; gamma, beta and conv weights trainable).
//
//   relu_bn_bwd   : dy = g * [a > 0] in place, plus the per-channel sum of dy (dbeta of the frozen BN; at a bottleneck junction
//                   out = relu(shortcut + bn3(conv3)) conv3 and the projection shortcut share it).  dgamma is taken from the
//                   weight gradient: sum_p dy*z = <W[c,:], dW_raw[c,:]> with z the conv output, so
//                   dgamma = (<W, dW_raw> - mean * dbeta) / sigma -- exact for gamma = 0 too (wgrad_gemm_sm100.cu).
//                   It also adds the gradient of resnet_utils.subsample (identity shortcut of a stride-2 unit):
//                   g_x[2p,2q] += d[p,q].
//   maxpool_relu_bwd : gradient of slim.max_pool2d(3x3, stride 2, SAME), routed to the first maximum of each window,
//                   with conv1's ReLU mask and dy sums.
//   upsample2     : zero insertion that turns the stride-2 3x3 dgrad into a stride-1 conv.
//   col2im_bwd    : gradient of the deconv heads' col2im (gather of the head gradients per (pixel, tap, channel)).
// Reductions are two-stage with a fixed order (bitwise reproducible).
#include "half_utils.cuh"
#include "kernels.cuh"

namespace dgp {

namespace {

using h16::unpack8;
__device__ __forceinline__ uint4 pack8v(const float* f, int fp16) { return h16::pack8(f, fp16); }

// dy = g * [act > 0] in place + per-channel partial sums of dy (-> dbeta).  The same kernel serves plain ReLU layers and the
// bottleneck junctions out = relu(shortcut + bn3(conv3)): dgamma no longer needs the BN output (bn_finalize_all_kernel takes it
// from the wgrad reduce's row-dot products <W, dW_raw>), so neither the shortcut tensor nor a division by gamma is involved.
// d != nullptr: g first receives the gradient of resnet_utils.subsample (the identity shortcut of the stride-2 unit behind this
// junction): g[n,2p,2q] += d[n,p,q] with g (N,H,W,C), d (N,P,Q,C) -- one pass instead of a scatter-add pass plus this one.
__global__ void __launch_bounds__(256) relu_bn_bwd_kernel(uint4* __restrict__ g, const uint4* __restrict__ act, int M, int C8,
                                                          float* __restrict__ partial, int fp16, const uint4* __restrict__ d,
                                                          int H, int W, int P, int Q) {
  const int my_cg = threadIdx.x % C8;
  const int my_r = threadIdx.x / C8;
  const int rpb = 256 / C8;
  float S[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) S[j] = 0.0f;
  for (int r = blockIdx.x * rpb + my_r; r < M; r += gridDim.x * rpb) {
    const size_t idx = (size_t)r * C8 + my_cg;
    float gv[8], av[8];
    unpack8(g[idx], gv, fp16);
    unpack8(__ldg(act + idx), av, fp16);
    if (d != nullptr) {
      const int xx = r % W, y = (r / W) % H, n = r / (W * H);
      if (!(xx & 1) && !(y & 1) && (y >> 1) < P && (xx >> 1) < Q) {
        float dv[8];
        unpack8(__ldg(d + (((size_t)n * P + (y >> 1)) * Q + (xx >> 1)) * C8 + my_cg), dv, fp16);
#pragma unroll
        for (int j = 0; j < 8; ++j) gv[j] += dv[j];
      }
    }
    float dyv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) dyv[j] = av[j] > 0.0f ? gv[j] : 0.0f;
    const uint4 o = pack8v(dyv, fp16);
    g[idx] = o;
    // the sums are those of dy as stored (what the wgrad GEMM consumes, so that dgamma's <W, dW_raw> - mean * dbeta cancels
    // exactly): with the scatter, g + d is rounded on the store
    unpack8(o, dyv, fp16);
#pragma unroll
    for (int j = 0; j < 8; ++j) S[j] += dyv[j];
  }
  __shared__ float sm[256][9];
#pragma unroll
  for (int j = 0; j < 8; ++j) sm[threadIdx.x][j] = S[j];
  __syncthreads();
  if (my_r == 0) {
    const int C = C8 * 8;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float acc = 0.0f;
      for (int rr = 0; rr < rpb; ++rr) acc += sm[rr * C8 + my_cg][j];
      partial[(size_t)blockIdx.x * C + my_cg * 8 + j] = acc;
    }
  }
}

// All frozen-BN parameter gradients of the network in one launch (one block per 8 channels, 128 row groups x 8 channels):
// dbeta = sum over the row blocks of the dy sums its mask site left, dgamma = (sum_kk <W, dW_raw> - mean * dbeta) / sigma.
// Fixed summation order (strided partial sums, then a tree over the row groups): bitwise reproducible.
__global__ void __launch_bounds__(1024) bn_finalize_all_kernel(const BnGroup* __restrict__ table, const float* __restrict__ part,
                                                               const float* __restrict__ rowdot, const float* __restrict__ mean,
                                                               const float* __restrict__ var, float eps,
                                                               float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                               const GradMode* __restrict__ mode) {
  const BnGroup g = table[blockIdx.x];
  const int cl = threadIdx.x & 7, rg = threadIdx.x >> 3;
  const float* pp = part + g.part_off + g.col + cl;
  float s0 = 0.0f, s1 = 0.0f;
#pragma unroll 8
  for (int b = rg; b < g.rows; b += 128) s0 += __ldg(pp + (size_t)b * g.C);   // up to ~100 independent loads per thread
  const float* rd = rowdot + g.rd_off + (size_t)cl * g.K4;
#pragma unroll 4
  for (int i = rg; i < g.K4; i += 128) s1 += __ldg(rd + i);
  __shared__ float sm0[128][9], sm1[128][9];
  sm0[rg][cl] = s0;
  sm1[rg][cl] = s1;
  __syncthreads();
  for (int st = 64; st > 0; st >>= 1) {
    if (rg < st) {
      sm0[rg][cl] += sm0[rg + st][cl];
      sm1[rg][cl] += sm1[rg + st][cl];
    }
    __syncthreads();
  }
  if (rg == 0) {
    const int c = blockIdx.x * 8 + cl;
    const float db = sm0[0][cl];
    store_grad(dbeta + c, db, mode);
    store_grad(dgamma + c, (sm1[0][cl] - mean[c] * db) * rsqrtf(var[c] + eps), mode);
  }
}

// Root of the backward pass in ONE pass: gradient of slim.max_pool2d(3x3, stride 2, SAME) routed to the first maximum of each
// window, conv1's ReLU mask, and the per-channel sums of the masked gradient (-> dbeta of conv1's BN).  64 channels.
// A CTA owns an 8 x 32 tile of conv1-output pixels: it stages the (<= 11 x 35)-pixel neighbourhood of x = relu(bn(conv1)) in
// shared memory, finds the argmax of the (<= 5 x 17) windows that touch the tile there (stage A; their pooled gradients are
// fetched alongside), and every pixel then gathers from its <= 2 x 2 windows (stage B).  x is read ~1.5 x (halo, L2 hits), the
// pooled gradient once, dy written once: ~0.5 GB per 10 frames of 747 x 832 instead of the 1.5 GB of argmax + gather + mask
// passes over HBM-resident tensors.
constexpr int kPoolTileH = 8, kPoolTileW = 32, kPoolRows = 11, kPoolCols = 35, kPoolP = 5, kPoolQ = 17;
constexpr int kPoolBwdSmem = (kPoolRows * kPoolCols * 8 + 2 * kPoolP * kPoolQ * 8) * 16;

// packed 16-bit helpers of the kernel below: per-half masks (0xFFFF where true)
template <bool kFp16>
__device__ __forceinline__ uint32_t gt_mask16x2(uint32_t a, uint32_t b) {
  if (kFp16) return __hgt2_mask(*reinterpret_cast<const __half2*>(&a), *reinterpret_cast<const __half2*>(&b));
  return __hgt2_mask(*reinterpret_cast<const __nv_bfloat162*>(&a), *reinterpret_cast<const __nv_bfloat162*>(&b));
}
template <bool kFp16>
__device__ __forceinline__ float2 unpack16x2(uint32_t w) {
  if (kFp16) return __half22float2(*reinterpret_cast<const __half2*>(&w));
  return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}

// ncu (first version, profiles/r02_ncu_bwd_kernels.md): issue-bound (78 % issue utilisation, DRAM 18 %) at ~3000 instructions
// per thread, so this version counts instructions: all index arithmetic divides by compile-time constants (fixed shared-memory
// strides), the arg-max scan of stage A runs on packed 16-bit pairs (one mask + two selects per pair and position instead of
// unpack + 2 x (compare, select, select)), the winner is kept as a ONE-HOT position bit per 16-bit lane so that stage B turns
// "is this pixel the winner of that window" into shift / and / multiply on two channels at a time.
template <bool kFp16>
__global__ void __launch_bounds__(256) maxpool_relu_bwd_kernel(const uint4* __restrict__ x, const uint4* __restrict__ gout, int H,
                                                               int W, int Ho, int Wo, int pad_t, int pad_l, uint4* __restrict__ gx,
                                                               float* __restrict__ partial) {
  extern __shared__ uint4 pool_sm[];
  uint4* xs = pool_sm;                                   // [kPoolRows][kPoolCols][8]
  uint4* gs = pool_sm + kPoolRows * kPoolCols * 8;       // [kPoolP][kPoolQ][8] pooled gradients
  uint4* as = gs + kPoolP * kPoolQ * 8;                  // [kPoolP][kPoolQ][8] one-hot winner position per 16-bit lane
  const int n = blockIdx.z, y0 = blockIdx.y * kPoolTileH, x0 = blockIdx.x * kPoolTileW;
  const int y1 = min(y0 + kPoolTileH, H) - 1, x1 = min(x0 + kPoolTileW, W) - 1;
  const int p_lo = max(0, (y0 + pad_t - 1) >> 1), p_hi = min(Ho - 1, (y1 + pad_t) >> 1);
  const int q_lo = max(0, (x0 + pad_l - 1) >> 1), q_hi = min(Wo - 1, (x1 + pad_l) >> 1);
  const int nP = p_hi - p_lo + 1, nQ = q_hi - q_lo + 1;
  const int ys0 = min(2 * p_lo - pad_t, y0), xs0 = min(2 * q_lo - pad_l, x0);
  const int tid = threadIdx.x;
  const int cg = tid & 7;
  for (int it = tid; it < kPoolRows * kPoolCols * 8; it += 256) {
    const int px = it >> 3, col = px % kPoolCols, row = px / kPoolCols;
    const int y = ys0 + row, xx = xs0 + col;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (y >= 0 && y < H && xx >= 0 && xx < W) v = __ldg(x + (((size_t)n * H + y) * W + xx) * 8 + cg);
    xs[it] = v;
  }
  __syncthreads();
  // ---- stage A: first maximum of every window (row-major over its valid positions, strict >), packed
  const uint32_t ninf = kFp16 ? 0xFC00FC00u : 0xFF80FF80u;
  for (int it = tid; it < kPoolP * kPoolQ * 8; it += 256) {
    const int wi = it >> 3, wq = wi % kPoolQ, wp = wi / kPoolQ;
    if (wp >= nP || wq >= nQ) continue;
    const int p = p_lo + wp, q = q_lo + wq;
    uint32_t best[4] = {ninf, ninf, ninf, ninf}, oh[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
      const int y = 2 * p - pad_t + dy;
      if (y < 0 || y >= H) continue;
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        const int xx = 2 * q - pad_l + dx;
        if (xx < 0 || xx >= W) continue;
        const uint4 v = xs[((y - ys0) * kPoolCols + (xx - xs0)) * 8 + cg];
        const uint32_t vw[4] = {v.x, v.y, v.z, v.w};
        const uint32_t pos2 = 0x00010001u << (dy * 3 + dx);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint32_t m = gt_mask16x2<kFp16>(vw[k], best[k]);
          best[k] = (vw[k] & m) | (best[k] & ~m);
          oh[k] = (pos2 & m) | (oh[k] & ~m);
        }
      }
    }
    as[it] = make_uint4(oh[0], oh[1], oh[2], oh[3]);
    gs[it] = __ldg(gout + (((size_t)n * Ho + p) * Wo + q) * 8 + cg);
  }
  __syncthreads();
  // ---- stage B: every pixel of the tile gathers from the windows that contain it, masks, stores, sums
  float S[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) S[j] = 0.0f;
#pragma unroll 2
  for (int it = tid; it < kPoolTileH * kPoolTileW * 8; it += 256) {
    const int col = (it >> 3) % kPoolTileW, row = (it >> 3) / kPoolTileW;
    const int y = y0 + row, xx = x0 + col;
    if (y >= H || xx >= W) continue;
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.0f;
    const int pa = max(0, (y + pad_t - 1) >> 1), pb = min(Ho - 1, (y + pad_t) >> 1);
    const int qa = max(0, (xx + pad_l - 1) >> 1), qb = min(Wo - 1, (xx + pad_l) >> 1);
    for (int p = pa; p <= pb; ++p)
      for (int q = qa; q <= qb; ++q) {
        const int mine = (y - (2 * p - pad_t)) * 3 + (xx - (2 * q - pad_l));
        const int w = ((p - p_lo) * kPoolQ + (q - q_lo)) * 8 + cg;
        const uint4 a = as[w], g = gs[w];
        const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, gw[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint32_t hit = ((aw[k] >> mine) & 0x00010001u) * 0xFFFFu;   // 0xFFFF per 16-bit lane this pixel won
          const float2 f = unpack16x2<kFp16>(gw[k] & hit);
          acc[2 * k] += f.x;
          acc[2 * k + 1] += f.y;
        }
      }
    const uint4 xv = xs[((y - ys0) * kPoolCols + (xx - xs0)) * 8 + cg];
    uint4 o = pack8v(acc, kFp16 ? 1 : 0);
    o.x &= gt_mask16x2<kFp16>(xv.x, 0u); o.y &= gt_mask16x2<kFp16>(xv.y, 0u);
    o.z &= gt_mask16x2<kFp16>(xv.z, 0u); o.w &= gt_mask16x2<kFp16>(xv.w, 0u);
    gx[(((size_t)n * H + y) * W + xx) * 8 + cg] = o;
    // the sums are those of dy as stored (what the wgrad GEMM consumes)
    const uint32_t ow[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 f = unpack16x2<kFp16>(ow[k]);
      S[2 * k] += f.x;
      S[2 * k + 1] += f.y;
    }
  }
  __syncthreads();   // xs is dead: reuse it for the fixed-order column reduction
  float* red = reinterpret_cast<float*>(pool_sm);   // [256][9]
#pragma unroll
  for (int j = 0; j < 8; ++j) red[tid * 9 + j] = S[j];
  __syncthreads();
  if (tid < 64) {
    const int c8 = tid >> 3, j = tid & 7;
    float acc = 0.0f;
    for (int r = 0; r < 32; ++r) acc += red[(r * 8 + c8) * 9 + j];
    const size_t blk = ((size_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    partial[blk * 64 + tid] = acc;
  }
}

// out (N,H,W,C) = zero-inserted in (N,P,Q,C): out[n,2p,2q] = in[n,p,q]
__global__ void upsample2_kernel(const uint4* __restrict__ in, int N, int P, int Q, int C8, uint4* __restrict__ out, int H,
                                 int W) {
  const size_t total = (size_t)N * H * W * C8;
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(t % C8);
    size_t r = t / C8;
    const int x = (int)(r % W);
    r /= W;
    const int y = (int)(r % H);
    const int n = (int)(r / H);
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (!(y & 1) && !(x & 1) && (y >> 1) < P && (x >> 1) < Q) v = __ldg(in + (((size_t)n * P + (y >> 1)) * Q + (x >> 1)) * C8 + c);
    out[t] = v;
  }
}

// dG[m][kk] (16-bit, Kd columns) = head gradient at (2i+kh, 2j+kw), kk = (kh*3+kw)*ctot + co; zero outside / padding.
__global__ void col2im_bwd_kernel(const float* __restrict__ g_logits, const float* __restrict__ g_locref, int N, int h, int w,
                                  int ctot, int nj, uint16_t* __restrict__ dG, int Kd, int fp16) {
  const size_t total = (size_t)N * h * w * Kd;
  const int Ho = 2 * h, Wo = 2 * w;
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const int kk = (int)(t % (size_t)Kd);
    size_t m = t / (size_t)Kd;
    const int j = (int)(m % w);
    m /= w;
    const int i = (int)(m % h);
    const int n = (int)(m / h);
    float v = 0.0f;
    if (kk < 9 * ctot) {
      const int tap = kk / ctot;
      const int co = kk - tap * ctot;
      const int y = 2 * i + tap / 3, x = 2 * j + tap % 3;
      if (y < Ho && x < Wo) {
        if (co < nj) v = g_logits[(((size_t)n * Ho + y) * Wo + x) * nj + co];
        else if (g_locref) v = g_locref[(((size_t)n * Ho + y) * Wo + x) * (size_t)(ctot - nj) + (co - nj)];
      }
    }
    dG[t] = h16::cvt1(v, fp16);
  }
}

// Head bias gradient, stage 1: block b sums a contiguous slice of the (npix, C) gradient per channel.  The thread
// count is a multiple of C, so a thread's elements all belong to channel (global thread id) % C.
__global__ void __launch_bounds__(256) head_bias_partial_kernel(const float* __restrict__ g, size_t n, int C, int nthreads,
                                                                float* __restrict__ partial) {
  const int gid = blockIdx.x * 256 + threadIdx.x;
  float acc = 0.0f;
  if (gid < nthreads)
    for (size_t i = gid; i < n; i += (size_t)nthreads) acc += g[i];
  __shared__ float sm[256];
  sm[threadIdx.x] = acc;
  __syncthreads();
  if ((int)threadIdx.x < C) {
    // threads t of this block with (blockIdx.x * 256 + t) % C == threadIdx.x
    const int base = (blockIdx.x * 256) % C;
    int t0 = (int)threadIdx.x - base;
    if (t0 < 0) t0 += C;
    float s = 0.0f;
    for (int t = t0; t < 256; t += C) s += sm[t];
    partial[(size_t)blockIdx.x * C + threadIdx.x] = s;
  }
}
__global__ void head_bias_final_kernel(const float* __restrict__ partial, int nblocks, int C, float* __restrict__ dbias,
                                       const GradMode* __restrict__ mode) {
  const int c = threadIdx.x;
  if (c >= C) return;
  float s = 0.0f;
  for (int b = 0; b < nblocks; ++b) s += partial[(size_t)b * C + c];
  store_grad(dbias + c, s, mode);
}

__global__ void scale_inplace_kernel(float* __restrict__ x, size_t n, float s) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) x[i] *= s;
}

int flat_grid(size_t n, int threads) {
  size_t g = (n + threads - 1) / threads;
  if (g > 148 * 16) g = 148 * 16;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

int relu_bn_bwd_blocks(int M, int C) {
  const int rpb = 256 / (C / 8);
  int blocks = (M + rpb - 1) / rpb;
  if (blocks > 148 * 4) blocks = 148 * 4;
  return blocks < 1 ? 1 : blocks;
}

cudaError_t launch_relu_bn_bwd(void* g, const void* act, int M, int C, float* partial, int fp16, cudaStream_t s,
                               const void* scatter_d, int H, int W, int P, int Q) {
  if (C % 8 || 256 % (C / 8) || C / 8 > 256) return cudaErrorInvalidValue;
  if (scatter_d != nullptr && (H < 1 || W < 1 || M % (H * W))) return cudaErrorInvalidValue;
  const int blocks = relu_bn_bwd_blocks(M, C);
  relu_bn_bwd_kernel<<<blocks, 256, 0, s>>>(reinterpret_cast<uint4*>(g), reinterpret_cast<const uint4*>(act), M, C / 8, partial, fp16,
                                            reinterpret_cast<const uint4*>(scatter_d), H, W, P, Q);
  return cudaGetLastError();
}

cudaError_t launch_bn_finalize_all(const BnGroup* table, int ngroups, const float* part, const float* rowdot, const float* mean,
                                   const float* var, float eps, float* dgamma, float* dbeta, const GradMode* mode, cudaStream_t s) {
  bn_finalize_all_kernel<<<ngroups, 1024, 0, s>>>(table, part, rowdot, mean, var, eps, dgamma, dbeta, mode);
  return cudaGetLastError();
}

int maxpool_relu_bwd_rows(int N, int H, int W) {
  return N * ((H + kPoolTileH - 1) / kPoolTileH) * ((W + kPoolTileW - 1) / kPoolTileW);
}

cudaError_t launch_maxpool_relu_bwd(const void* x, const void* gout, int N, int H, int W, int C, int Ho, int Wo, int pad_t,
                                    int pad_l, void* gx, float* partial, int fp16, cudaStream_t s) {
  if (C != 64 || pad_t < 0 || pad_t > 1 || pad_l < 0 || pad_l > 1 || N > 65535) return cudaErrorInvalidValue;
  dim3 grid((W + kPoolTileW - 1) / kPoolTileW, (H + kPoolTileH - 1) / kPoolTileH, N);
  cudaError_t e;
  if (fp16) {
    e = cudaFuncSetAttribute(maxpool_relu_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPoolBwdSmem);
    if (e != cudaSuccess) return e;
    maxpool_relu_bwd_kernel<true><<<grid, 256, kPoolBwdSmem, s>>>(reinterpret_cast<const uint4*>(x), reinterpret_cast<const uint4*>(gout),
                                                                  H, W, Ho, Wo, pad_t, pad_l, reinterpret_cast<uint4*>(gx), partial);
  } else {
    e = cudaFuncSetAttribute(maxpool_relu_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPoolBwdSmem);
    if (e != cudaSuccess) return e;
    maxpool_relu_bwd_kernel<false><<<grid, 256, kPoolBwdSmem, s>>>(reinterpret_cast<const uint4*>(x), reinterpret_cast<const uint4*>(gout),
                                                                   H, W, Ho, Wo, pad_t, pad_l, reinterpret_cast<uint4*>(gx), partial);
  }
  return cudaGetLastError();
}

cudaError_t launch_upsample2(const void* in, int N, int P, int Q, int C, void* out, int H, int W, cudaStream_t s) {
  const size_t total = (size_t)N * H * W * (C / 8);
  upsample2_kernel<<<flat_grid(total, 256), 256, 0, s>>>(reinterpret_cast<const uint4*>(in), N, P, Q, C / 8,
                                                         reinterpret_cast<uint4*>(out), H, W);
  return cudaGetLastError();
}

cudaError_t launch_col2im_bwd(const float* g_logits, const float* g_locref, int N, int h, int w, int ctot, int nj,
                              void* dG, int Kd, int fp16, cudaStream_t s) {
  const size_t total = (size_t)N * h * w * Kd;
  col2im_bwd_kernel<<<flat_grid(total, 256), 256, 0, s>>>(g_logits, g_locref, N, h, w, ctot, nj,
                                                          reinterpret_cast<uint16_t*>(dG), Kd, fp16);
  return cudaGetLastError();
}

int head_bias_blocks() { return 148; }

// g: (npix, C) fp32; partial: [head_bias_blocks()][C] workspace
cudaError_t launch_head_bias_grad(const float* g, size_t npix, int C, float* partial, float* dbias, const GradMode* mode,
                                  cudaStream_t s) {
  if (C > 256) return cudaErrorInvalidValue;
  const int nthreads = (148 * 256 / C) * C;
  head_bias_partial_kernel<<<148, 256, 0, s>>>(g, npix * (size_t)C, C, nthreads, partial);
  head_bias_final_kernel<<<1, 256, 0, s>>>(partial, 148, C, dbias, mode);
  return cudaGetLastError();
}

cudaError_t launch_scale_inplace(float* x, size_t n, float scale, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  scale_inplace_kernel<<<flat_grid(n, 256), 256, 0, s>>>(x, n, scale);
  return cudaGetLastError();
}

}  // namespace dgp
