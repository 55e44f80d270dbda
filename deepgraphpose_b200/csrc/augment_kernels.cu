// Augmentation of fit_dgp's labelled training frames on the device (reference data_aug / build_aug, fitdgp_util.py:412-451,
// called at fitdgp.py:773-779): rotation, motion blur, coarse dropout and elastic deformation, applied in that order to the
// frames a batch lists, with their labels moved alongside.  Every pixel operation is integer arithmetic pinned to an oracle:
//  - rotation is cv2.warpAffine(INTER_LINEAR, BORDER_CONSTANT 0) and elastic sampling cv2.remap(INTER_LINEAR, BORDER_CONSTANT 0),
//    both through OpenCV's fixed-point bilinear path (5 fraction bits, int16 weights summing to 2^15), bit for bit;
//  - motion blur is an integer correlation with weights summing to 2^14 and a reflect-101 border;
//  - dropout zeroes the pixels of dropped cells of a coarse grid upsampled as cv2.resize(INTER_NEAREST) indexes it.
// The random fields (elastic displacement noise, dropout cells) come from a counter hash of (seed, plane, row, col)
// (include/dgp_b200.h), so no frame-sized random array is drawn on the host.  A sampler cannot work in place: each
// geometric pass writes into handle-owned scratch frames and the last pass of every frame writes back into the caller's.
#include "../../include/dgp_b200.h"

#include <cuda_runtime.h>

#include <cmath>
#include <vector>

#include "handle.cuh"

namespace {

constexpr int kChunk = 16;         // frames per launch (per-frame arguments travel in the kernel parameters)
constexpr int kMaxBlurK = 15;
constexpr int kMaxRadius = 64;     // elastic Gaussian radius ceil(4 sigma): sigma <= 16
constexpr int kSampThreads = 128;
constexpr int kBlurTX = 32, kBlurTY = 8;
constexpr int kFieldThreads = 256;
constexpr int kLabelThreads = 128;
constexpr int kElasticIters = 20;

__host__ __device__ inline uint64_t aug_hash(uint64_t seed, uint32_t plane, uint32_t row, uint32_t col) {
  const uint64_t c = ((uint64_t)plane << 48) | ((uint64_t)row << 24) | (uint64_t)col;
  uint64_t z = seed + (c + 1) * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// uniform in [-1, 1): (b + 0.5) / 2^23 - 1 of the top 24 bits b, exact in float32
__device__ inline float noise_pm1(uint64_t z) {
  const int b = (int)(z >> 40);
  return (float)(2 * b + 1 - (1 << 24)) * 0x1p-24f;
}

// cv::borderInterpolate for BORDER_REFLECT_101
__host__ __device__ inline int reflect101(int p, int len) {
  if ((unsigned)p < (unsigned)len) return p;
  if (len == 1) return 0;
  do {
    p = p < 0 ? -p : 2 * len - 2 - p;
  } while ((unsigned)p >= (unsigned)len);
  return p;
}

// OpenCV's bilinear int16 weight table entry (initInterTab2D, INTER_LINEAR): products of the 1-D float weights scaled by
// 2^15 and rounded half-even, then the sum fixed up to 2^15 on the smallest / largest entry.  w[dy * 2 + dx].
__device__ inline void bilinear_weights(int fx, int fy, int w[4]) {
  const float ax = (float)fx * (1.f / 32), ay = (float)fy * (1.f / 32);
  const float vx[2] = {1.f - ax, ax}, vy[2] = {1.f - ay, ay};
  int sum = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    w[k] = __float2int_rn(__fmul_rn(__fmul_rn(vy[k >> 1], vx[k & 1]), 32768.f));
    sum += w[k];
  }
  if (sum != 32768) {
    int mk = 0, Mk = 0, mv = w[0], Mv = w[0];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (w[k] < mv) { mk = k; mv = w[k]; }
      else if (w[k] > Mv) { Mk = k; Mv = w[k]; }
    }
    const int diff = sum - 32768;
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (k == (diff < 0 ? Mk : mk)) w[k] -= diff;
  }
}

__device__ inline int sat16(int v) { return min(max(v, -32768), 32767); }

struct SampFrame {
  const uint8_t* src;
  uint8_t* dst;
  double m[6];                 // warpAffine: the inverted matrix
  const float *dx, *dy;        // remap: displacement fields
};
struct SampArgs {
  SampFrame f[kChunk];
  int H, W, chunks;            // chunks: 16-byte pieces of an output row
};

// One thread per 16 output bytes of a row: the pixels those bytes belong to are sampled with OpenCV's fixed-point
// bilinear arithmetic (coordinates from the per-row / per-column warpAffine terms, or from the float remap maps x + dx,
// y + dy), taps outside the frame read 0.  The source frame is read through L2; the result is stored with one 16 B store
// when the row piece is aligned.
template <bool kRemap>
__global__ void __launch_bounds__(kSampThreads) aug_sample_kernel(const SampArgs a) {
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (int64_t)a.H * a.chunks) return;
  const SampFrame& F = a.f[blockIdx.y];
  const int H = a.H, W = a.W;
  const int y = (int)(gid / a.chunks), o = (int)(gid % a.chunks) * 16;
  const int row_bytes = 3 * W;
  const int x0 = o / 3, x1 = min((o + 15) / 3, W - 1);
  int X0 = 0, Y0 = 0;
  if (!kRemap) {
    X0 = __double2int_rn(__dmul_rn(__dadd_rn(__dmul_rn(F.m[1], (double)y), F.m[2]), 1024.0)) + 16;
    Y0 = __double2int_rn(__dmul_rn(__dadd_rn(__dmul_rn(F.m[4], (double)y), F.m[5]), 1024.0)) + 16;
  }
  // bytes of pixels x0 .. x0 + 5 at fixed positions, shifted by the row piece's offset o - 3 x0 at the end
  uint32_t buf[5] = {0u, 0u, 0u, 0u, 0u};
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const int x = x0 + i;
    if (x > x1) continue;
    int X, Y;
    if (kRemap) {
      const size_t pi = (size_t)y * W + x;
      const float mx = __fadd_rn((float)x, __ldg(F.dx + pi)), my = __fadd_rn((float)y, __ldg(F.dy + pi));
      X = __float2int_rn(__fmul_rn(mx, 32.f));
      Y = __float2int_rn(__fmul_rn(my, 32.f));
    } else {
      X = (X0 + __double2int_rn(__dmul_rn(__dmul_rn(F.m[0], (double)x), 1024.0))) >> 5;
      Y = (Y0 + __double2int_rn(__dmul_rn(__dmul_rn(F.m[3], (double)x), 1024.0))) >> 5;
    }
    const int sx = sat16(X >> 5), sy = sat16(Y >> 5);
    int w[4];
    bilinear_weights(X & 31, Y & 31, w);
    int acc0 = 1 << 14, acc1 = 1 << 14, acc2 = 1 << 14;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int py = sy + (k >> 1), px = sx + (k & 1);
      if (py >= 0 && py < H && px >= 0 && px < W) {
        const uint8_t* p = F.src + ((size_t)py * W + px) * 3;
        acc0 += w[k] * (int)__ldg(p);
        acc1 += w[k] * (int)__ldg(p + 1);
        acc2 += w[k] * (int)__ldg(p + 2);
      }
    }
    const int v[3] = {min(acc0 >> 15, 255), min(acc1 >> 15, 255), min(acc2 >> 15, 255)};
#pragma unroll
    for (int c = 0; c < 3; ++c) buf[(3 * i + c) >> 2] |= (uint32_t)v[c] << (8 * ((3 * i + c) & 3));
  }
  const int sh = 8 * (o - 3 * x0);
  uint32_t out[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) out[j] = __funnelshift_r(buf[j], buf[j + 1], sh);
  uint8_t* dst = F.dst + (size_t)y * row_bytes + o;
  if (o + 16 <= row_bytes && ((uintptr_t)dst & 15) == 0) {
    *reinterpret_cast<uint4*>(dst) = make_uint4(out[0], out[1], out[2], out[3]);
  } else {
    const int m = min(16, row_bytes - o);
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (j < m) dst[j] = (uint8_t)(out[j >> 2] >> (8 * (j & 3)));
  }
}

struct BlurFrame {
  const uint8_t* src;
  uint8_t* dst;
  int k;                       // odd kernel size (1 = identity, for dropout alone)
  int gh, gw;                  // dropout grid (0 = no dropout)
  double ify, ifx;             // cv2.resize(INTER_NEAREST) scales 1 / (H / gh), 1 / (W / gw)
  double p;                    // a cell is dropped when its uniform is below p
  uint64_t seed;
  int32_t w[kMaxBlurK * kMaxBlurK];  // row-major, sum 2^14
};
struct BlurArgs {
  BlurFrame f[kChunk];
  int H, W;
};

// Integer k x k correlation (sum w * p + 2^13) >> 14 with a reflect-101 border, the frame tile and its halo staged in shared
// memory, and the dropout mask applied at the store.
__global__ void __launch_bounds__(kBlurTX * kBlurTY) aug_blur_drop_kernel(const BlurArgs a) {
  __shared__ uint8_t tile[(kBlurTY + kMaxBlurK - 1) * (kBlurTX + kMaxBlurK - 1) * 3];
  const BlurFrame& F = a.f[blockIdx.z];
  const int H = a.H, W = a.W;
  const int k = F.k, r = k >> 1;
  const int tw = kBlurTX + 2 * r, th = kBlurTY + 2 * r;
  const int bx0 = blockIdx.x * kBlurTX, by0 = blockIdx.y * kBlurTY;
  const int tid = threadIdx.y * kBlurTX + threadIdx.x;
  for (int i = tid; i < tw * th; i += kBlurTX * kBlurTY) {
    const int ty = i / tw, tx = i - ty * tw;
    const int gy = reflect101(by0 + ty - r, H), gx = reflect101(bx0 + tx - r, W);
    const uint8_t* p = F.src + ((size_t)gy * W + gx) * 3;
    tile[3 * i] = __ldg(p);
    tile[3 * i + 1] = __ldg(p + 1);
    tile[3 * i + 2] = __ldg(p + 2);
  }
  __syncthreads();
  const int x = bx0 + threadIdx.x, y = by0 + threadIdx.y;
  if (x >= W || y >= H) return;
  int a0 = 1 << 13, a1 = 1 << 13, a2 = 1 << 13;
  for (int i = 0; i < k; ++i) {
    const uint8_t* t = tile + ((threadIdx.y + i) * tw + threadIdx.x) * 3;
    const int32_t* wr = F.w + i * k;
    for (int j = 0; j < k; ++j) {
      const int wt = wr[j];
      a0 += wt * t[3 * j];
      a1 += wt * t[3 * j + 1];
      a2 += wt * t[3 * j + 2];
    }
  }
  int v0 = min(max(a0 >> 14, 0), 255), v1 = min(max(a1 >> 14, 0), 255), v2 = min(max(a2 >> 14, 0), 255);
  if (F.gh) {
    const int iy = min((int)floor(__dmul_rn((double)y, F.ify)), F.gh - 1);
    const int ix = min((int)floor(__dmul_rn((double)x, F.ifx)), F.gw - 1);
    const double u = ((double)(aug_hash(F.seed, 2, iy, ix) >> 40) + 0.5) * 0x1p-24;
    if (u < F.p) v0 = v1 = v2 = 0;
  }
  uint8_t* d = F.dst + ((size_t)y * W + x) * 3;
  d[0] = (uint8_t)v0;
  d[1] = (uint8_t)v1;
  d[2] = (uint8_t)v2;
}

struct Gauss {
  float w[2 * kMaxRadius + 1];
  int R;
};

// Horizontal pass of the elastic field: the hash noise of planes 0 (dx) and 1 (dy) of one row segment and its reflect-101
// halo is staged in shared memory, then smoothed with the float32 Gaussian.
__global__ void __launch_bounds__(kFieldThreads) aug_field_h_kernel(uint64_t seed, int H, int W, const Gauss g, float* tx,
                                                                    float* ty) {
  extern __shared__ float sn[];
  const int R = g.R, span = kFieldThreads + 2 * R;
  const int row = blockIdx.y, x0 = blockIdx.x * kFieldThreads;
  for (int i = threadIdx.x; i < span; i += kFieldThreads) {
    const int col = reflect101(x0 + i - R, W);
    sn[i] = noise_pm1(aug_hash(seed, 0, row, col));
    sn[span + i] = noise_pm1(aug_hash(seed, 1, row, col));
  }
  __syncthreads();
  const int x = x0 + threadIdx.x;
  if (x >= W) return;
  float sx = 0.f, sy = 0.f;
  for (int k = 0; k <= 2 * R; ++k) {
    sx = fmaf(g.w[k], sn[threadIdx.x + k], sx);
    sy = fmaf(g.w[k], sn[span + threadIdx.x + k], sy);
  }
  tx[(size_t)row * W + x] = sx;
  ty[(size_t)row * W + x] = sy;
}

// Vertical pass: Gaussian over rows (reflect-101), scaled by alpha.
__global__ void __launch_bounds__(kFieldThreads) aug_field_v_kernel(int H, int W, const Gauss g, float alpha,
                                                                    const float* __restrict__ tx, const float* __restrict__ ty,
                                                                    float* __restrict__ dx, float* __restrict__ dy) {
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (int64_t)H * W) return;
  const int y = (int)(gid / W), x = (int)(gid % W);
  const int R = g.R;
  float sx = 0.f, sy = 0.f;
  for (int k = 0; k <= 2 * R; ++k) {
    const size_t q = (size_t)reflect101(y + k - R, H) * W + x;
    sx = fmaf(g.w[k], __ldg(tx + q), sx);
    sy = fmaf(g.w[k], __ldg(ty + q), sy);
  }
  dx[gid] = alpha * sx;
  dy[gid] = alpha * sy;
}

struct LabelFrame {
  double* jl;                  // (nj, 2) scoremap (row, col) labels of the frame
  double m[6];                 // forward rotation matrix (rot != 0)
  const float *dx, *dy;        // elastic fields (NULL = no elastic)
  int rot;
};
struct LabelArgs {
  LabelFrame f[kChunk];
  int nj, H, W;
  double stride;
};

__device__ inline double bilinear_field(const float* f, int H, int W, double px, double py) {
  const double cx = fmin(fmax(px, 0.0), (double)(W - 1)), cy = fmin(fmax(py, 0.0), (double)(H - 1));
  const int x0 = min((int)floor(cx), max(W - 2, 0)), y0 = min((int)floor(cy), max(H - 2, 0));
  const int x1 = min(x0 + 1, W - 1), y1 = min(y0 + 1, H - 1);
  const double fx = cx - x0, fy = cy - y0;
  const double f00 = f[(size_t)y0 * W + x0], f01 = f[(size_t)y0 * W + x1];
  const double f10 = f[(size_t)y1 * W + x0], f11 = f[(size_t)y1 * W + x1];
  return (1.0 - fy) * ((1.0 - fx) * f00 + fx * f01) + fy * ((1.0 - fx) * f10 + fx * f11);
}

// One thread per label: to pixels, rotation by the forward matrix, inversion of the elastic backward map by the fixed
// iteration p <- q - d(p), back to scoremap units.  NaN labels stay NaN; labels outside the frame are kept.
__global__ void __launch_bounds__(kLabelThreads) aug_labels_kernel(const LabelArgs a) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= a.nj) return;
  const LabelFrame& F = a.f[blockIdx.y];
  double* p = F.jl + 2 * j;
  const double row = p[0], col = p[1];
  if (isnan(row) || isnan(col)) return;
  const double s = a.stride;
  double x = col * s + s * 0.5, y = row * s + s * 0.5;
  if (F.rot) {
    const double xr = F.m[0] * x + F.m[1] * y + F.m[2];
    const double yr = F.m[3] * x + F.m[4] * y + F.m[5];
    x = xr;
    y = yr;
  }
  if (F.dx) {
    double px = x, py = y;
    for (int it = 0; it < kElasticIters; ++it) {
      const double nx = x - bilinear_field(F.dx, a.H, a.W, px, py);
      const double ny = y - bilinear_field(F.dy, a.H, a.W, px, py);
      px = nx;
      py = ny;
    }
    x = px;
    y = py;
  }
  p[0] = (y - s * 0.5) / s;
  p[1] = (x - s * 0.5) / s;
}

// ---------------------------------------------------------------------------------------------------------------- host
void rotation_matrix(double deg, int H, int W, double m[6]) {
  const double t = deg * (M_PI / 180.0);
  const double c = std::cos(t), s = std::sin(t);
  const double cx = W / 2.0 - 0.5, cy = H / 2.0 - 0.5;
  m[0] = c; m[1] = -s; m[2] = cx - c * cx + s * cy;
  m[3] = s; m[4] = c;  m[5] = cy - s * cx - c * cy;
}

// cv::warpAffine's inversion of the forward matrix (no WARP_INVERSE_MAP)
void invert_affine(const double f[6], double m[6]) {
  for (int i = 0; i < 6; ++i) m[i] = f[i];
  double D = m[0] * m[4] - m[1] * m[3];
  D = D != 0 ? 1. / D : 0;
  const double A11 = m[4] * D, A22 = m[0] * D;
  m[0] = A11; m[1] *= -D;
  m[3] *= -D; m[4] = A22;
  const double b1 = -m[0] * m[2] - m[1] * m[5];
  const double b2 = -m[3] * m[2] - m[4] * m[5];
  m[2] = b1; m[5] = b2;
}

void motion_blur_weights(int k, double angle_deg, double direction, int32_t* w) {
  const double d = (direction + 1.0) / 2.0;
  std::vector<double> img((size_t)k * k, 0.0), rot((size_t)k * k, 0.0);
  const double step = ((1.0 - d) - d) / (k - 1);
  for (int i = 0; i < k; ++i) img[(size_t)i * k + k / 2] = i == k - 1 ? 1.0 - d : i * step + d;
  const double t = angle_deg * (M_PI / 180.0);
  const double ca = std::cos(t), sa = std::sin(t), c = (k - 1) / 2.0;
  auto at = [&](int yy, int xx) { return (yy >= 0 && yy < k && xx >= 0 && xx < k) ? img[(size_t)yy * k + xx] : 0.0; };
  double sum = 0.0;
  for (int i = 0; i < k; ++i)
    for (int j = 0; j < k; ++j) {
      const double u = j - c, v = i - c;
      const double sx = ca * u + sa * v + c, sy = -sa * u + ca * v + c;
      const double fx0 = std::floor(sx), fy0 = std::floor(sy);
      const int x0 = (int)fx0, y0 = (int)fy0;
      const double fx = sx - fx0, fy = sy - fy0;
      const double val = (1.0 - fy) * ((1.0 - fx) * at(y0, x0) + fx * at(y0, x0 + 1)) +
                         fy * ((1.0 - fx) * at(y0 + 1, x0) + fx * at(y0 + 1, x0 + 1));
      rot[(size_t)i * k + j] = val;
      sum += val;
    }
  int64_t total = 0;
  size_t imax = 0;
  for (size_t i = 0; i < rot.size(); ++i) {
    w[i] = (int32_t)std::nearbyint(rot[i] / sum * 16384.0);
    total += w[i];
    if (w[i] > w[imax]) imax = i;
  }
  w[imax] += (int32_t)(16384 - total);
}

void gaussian(double sigma, Gauss* g) {
  const int R = (int)std::ceil(4.0 * sigma);
  std::vector<double> e(2 * R + 1);
  double sum = 0.0;
  for (int k = -R; k <= R; ++k) {
    e[k + R] = std::exp(-(double)(k * k) / (2.0 * sigma * sigma));
    sum += e[k + R];
  }
  g->R = R;
  for (int k = 0; k <= 2 * R; ++k) g->w[k] = (float)(e[k] / sum);
}

bool is_finite(double v) { return std::isfinite(v); }

bool frame_size_ok(int H, int W) {
  return H >= 1 && W >= 1 && H <= 32767 && W <= 32767 && (int64_t)H * W * 3 <= INT32_MAX;
}

bool params_ok(const dgp_augment_params& p) {
  if (!is_finite(p.rotate_deg) || !is_finite(p.blur_angle_deg) || !is_finite(p.blur_direction) || !is_finite(p.drop_p) ||
      !is_finite(p.drop_size_percent) || !is_finite(p.elastic_alpha) || !is_finite(p.elastic_sigma))
    return false;
  if (p.blur_k != 0 && (p.blur_k < 3 || p.blur_k > kMaxBlurK || (p.blur_k & 1) == 0)) return false;
  if (p.blur_k && (p.blur_direction < -1.0 || p.blur_direction > 1.0)) return false;
  if (p.drop_p < 0.0 || p.drop_p > 1.0 || p.drop_size_percent < 0.0 || p.drop_size_percent > 1.0) return false;
  if (p.elastic_alpha != 0.0 && (!(p.elastic_sigma > 0.0) || std::ceil(4.0 * p.elastic_sigma) > kMaxRadius)) return false;
  return true;
}

int launch_field(dgp_handle* h, int H, int W, double alpha, double sigma, uint64_t seed, float* tx, float* ty, float* dx,
                 float* dy, cudaStream_t s) {
  Gauss g;
  gaussian(sigma, &g);
  const size_t smem = (size_t)2 * (kFieldThreads + 2 * g.R) * sizeof(float);
  aug_field_h_kernel<<<dim3((W + kFieldThreads - 1) / kFieldThreads, H), kFieldThreads, smem, s>>>(seed, H, W, g, tx, ty);
  CU_OK(h, cudaGetLastError());
  const int64_t blocks = ((int64_t)H * W + kFieldThreads - 1) / kFieldThreads;
  aug_field_v_kernel<<<(unsigned)blocks, kFieldThreads, 0, s>>>(H, W, g, (float)alpha, tx, ty, dx, dy);
  CU_OK(h, cudaGetLastError());
  h->launches += 2;
  return DGP_OK;
}

}  // namespace

extern "C" {

int dgp_motion_blur_kernel(int k, double angle_deg, double direction, int32_t* weights) {
  if (k < 3 || k > kMaxBlurK || (k & 1) == 0 || !weights || !is_finite(angle_deg) || !is_finite(direction) || direction < -1.0 ||
      direction > 1.0)
    return DGP_ERR_INVALID;
  motion_blur_weights(k, angle_deg, direction, weights);
  return DGP_OK;
}

int dgp_elastic_field(dgp_handle* h, int H, int W, double alpha, double sigma, uint64_t seed, float* dx_dev, float* dy_dev,
                      void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!frame_size_ok(H, W) || !dx_dev || !dy_dev || !is_finite(alpha) || !is_finite(sigma) || !(sigma > 0.0) ||
      std::ceil(4.0 * sigma) > kMaxRadius)
    return fail(h, DGP_ERR_INVALID, "dgp_elastic_field: bad argument");
  CU_OK(h, cudaSetDevice(h->device));
  if (int rc = ensure(h, &h->aug_tmp, (size_t)2 * H * W * sizeof(float))) return rc;
  float* t = h->aug_tmp.get<float>();
  return launch_field(h, H, W, alpha, sigma, seed, t, t + (size_t)H * W, dx_dev, dy_dev, (cudaStream_t)stream);
}

int dgp_augment(dgp_handle* h, uint8_t* frames_dev, int nt, int H, int W, const int32_t* frame_idx_host, int n,
                const dgp_augment_params* params_host, double* joint_loc_dev, double stride, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (n < 0 || nt < 0 || !frame_size_ok(H, W)) return fail(h, DGP_ERR_INVALID, "dgp_augment: bad size");
  if (n == 0) return DGP_OK;
  if (!frames_dev || !frame_idx_host || !params_host) return fail(h, DGP_ERR_INVALID, "dgp_augment: NULL argument");
  if (joint_loc_dev && !(stride > 0.0 && is_finite(stride))) return fail(h, DGP_ERR_INVALID, "dgp_augment: stride must be > 0");
  std::vector<char> seen(nt, 0);
  for (int k = 0; k < n; ++k) {
    const int i = frame_idx_host[k];
    if (i < 0 || i >= nt) return fail(h, DGP_ERR_INVALID, "dgp_augment: frame index %d outside [0, %d)", i, nt);
    if (seen[i]) return fail(h, DGP_ERR_INVALID, "dgp_augment: frame index %d listed twice", i);
    seen[i] = 1;
    if (!params_ok(params_host[k])) return fail(h, DGP_ERR_INVALID, "dgp_augment: invalid parameters for frame %d", k);
  }
  const cudaStream_t s = (cudaStream_t)stream;
  const size_t fb = (size_t)H * W * 3, plane = (size_t)H * W;
  // per frame: the passes it runs (rotation, blur / dropout, elastic) and the buffer chain frames -> scratch -> frames
  struct Plan {
    bool rot, bd, el;
    int m;
    uint8_t* chain[4];
    int field;  // slot of the elastic fields
  };
  std::vector<Plan> plan(n);
  int n_el = 0, max_m = 0;
  bool any_label = false;
  for (int k = 0; k < n; ++k) {
    const dgp_augment_params& p = params_host[k];
    Plan& f = plan[k];
    f.rot = p.rotate_deg != 0.0;
    f.bd = p.blur_k != 0 || (p.drop_p > 0.0 && p.drop_size_percent > 0.0);
    f.el = p.elastic_alpha != 0.0;
    f.m = (int)f.rot + (int)f.bd + (int)f.el;
    f.field = f.el ? n_el++ : -1;
    max_m = max_m > f.m ? max_m : f.m;
    any_label |= f.rot || f.el;
  }
  if (max_m == 0) return DGP_OK;  // every op off for every frame: nothing is launched
  CU_OK(h, cudaSetDevice(h->device));
  int rc;
  if ((rc = ensure(h, &h->aug_scratch[0], fb * n))) return rc;
  if (max_m == 3 && (rc = ensure(h, &h->aug_scratch[1], fb * n))) return rc;
  if (n_el) {
    if ((rc = ensure(h, &h->aug_fields, plane * 2 * n_el * sizeof(float)))) return rc;
    if ((rc = ensure(h, &h->aug_tmp, plane * 2 * sizeof(float)))) return rc;
  }
  uint8_t* B = h->aug_scratch[0].get<uint8_t>();
  uint8_t* Cb = h->aug_scratch[1].get<uint8_t>();
  float* fields = h->aug_fields.get<float>();
  for (int k = 0; k < n; ++k) {
    Plan& f = plan[k];
    uint8_t* A = frames_dev + (size_t)frame_idx_host[k] * fb;
    f.chain[0] = f.chain[f.m] = A;
    if (f.m == 1) {  // one pass cannot run in place: it reads a scratch copy
      f.chain[0] = B + k * fb;
      CU_OK(h, cudaMemcpyAsync(f.chain[0], A, fb, cudaMemcpyDeviceToDevice, s));
    } else if (f.m >= 2) {
      f.chain[1] = B + k * fb;
      if (f.m == 3) f.chain[2] = Cb + k * fb;
    }
  }
  for (int k = 0; k < n; ++k) {
    const dgp_augment_params& p = params_host[k];
    if (!plan[k].el) continue;
    float* dx = fields + (size_t)plan[k].field * 2 * plane;
    float* t = h->aug_tmp.get<float>();
    if ((rc = launch_field(h, H, W, p.elastic_alpha, p.elastic_sigma, p.seed, t, t + plane, dx, dx + plane, s))) return rc;
  }
  std::vector<int> step(n, 0);  // passes each frame has run so far
  const int chunks = (3 * W + 15) / 16;
  const int64_t samp_blocks = ((int64_t)H * chunks + kSampThreads - 1) / kSampThreads;
  if (samp_blocks > INT32_MAX) return fail(h, DGP_ERR_UNSUPPORTED, "dgp_augment: frame too large");
  // rotation
  {
    SampArgs a;
    a.H = H; a.W = W; a.chunks = chunks;
    int c = 0;
    for (int k = 0; k <= n; ++k) {
      if (k < n && plan[k].rot) {
        SampFrame& F = a.f[c++];
        F.src = plan[k].chain[step[k]];
        F.dst = plan[k].chain[step[k] + 1];
        step[k]++;
        double fwd[6];
        rotation_matrix(params_host[k].rotate_deg, H, W, fwd);
        invert_affine(fwd, F.m);
        F.dx = F.dy = nullptr;
      }
      if (c == kChunk || (k == n && c > 0)) {
        aug_sample_kernel<false><<<dim3((unsigned)samp_blocks, c), kSampThreads, 0, s>>>(a);
        CU_OK(h, cudaGetLastError());
        h->launches++;
        c = 0;
      }
    }
  }
  // motion blur and / or dropout
  {
    BlurArgs a;
    a.H = H; a.W = W;
    int c = 0;
    for (int k = 0; k <= n; ++k) {
      if (k < n && plan[k].bd) {
        const dgp_augment_params& p = params_host[k];
        BlurFrame& F = a.f[c++];
        F.src = plan[k].chain[step[k]];
        F.dst = plan[k].chain[step[k] + 1];
        step[k]++;
        if (p.blur_k) {
          F.k = p.blur_k;
          motion_blur_weights(p.blur_k, p.blur_angle_deg, p.blur_direction, F.w);
        } else {
          F.k = 1;
          F.w[0] = 1 << 14;
        }
        F.gh = F.gw = 0;
        F.ify = F.ifx = 0.0;
        F.p = p.drop_p;
        F.seed = p.seed;
        if (p.drop_p > 0.0 && p.drop_size_percent > 0.0) {
          F.gh = std::max(1, (int)std::nearbyint(H * p.drop_size_percent));
          F.gw = std::max(1, (int)std::nearbyint(W * p.drop_size_percent));
          F.ify = 1.0 / ((double)H / F.gh);
          F.ifx = 1.0 / ((double)W / F.gw);
        }
      }
      if (c == kChunk || (k == n && c > 0)) {
        aug_blur_drop_kernel<<<dim3((W + kBlurTX - 1) / kBlurTX, (H + kBlurTY - 1) / kBlurTY, c), dim3(kBlurTX, kBlurTY), 0,
                               s>>>(a);
        CU_OK(h, cudaGetLastError());
        h->launches++;
        c = 0;
      }
    }
  }
  // elastic deformation
  {
    SampArgs a;
    a.H = H; a.W = W; a.chunks = chunks;
    int c = 0;
    for (int k = 0; k <= n; ++k) {
      if (k < n && plan[k].el) {
        SampFrame& F = a.f[c++];
        F.src = plan[k].chain[step[k]];
        F.dst = plan[k].chain[step[k] + 1];
        step[k]++;
        F.dx = fields + (size_t)plan[k].field * 2 * plane;
        F.dy = F.dx + plane;
        for (int i = 0; i < 6; ++i) F.m[i] = 0.0;
      }
      if (c == kChunk || (k == n && c > 0)) {
        aug_sample_kernel<true><<<dim3((unsigned)samp_blocks, c), kSampThreads, 0, s>>>(a);
        CU_OK(h, cudaGetLastError());
        h->launches++;
        c = 0;
      }
    }
  }
  // labels
  const int nj = h->cfg.num_joints;
  if (joint_loc_dev && any_label && nj > 0) {
    LabelArgs a;
    a.nj = nj; a.H = H; a.W = W; a.stride = stride;
    int c = 0;
    for (int k = 0; k <= n; ++k) {
      if (k < n && (plan[k].rot || plan[k].el)) {
        LabelFrame& F = a.f[c++];
        F.jl = joint_loc_dev + (size_t)k * nj * 2;
        F.rot = plan[k].rot;
        if (F.rot) rotation_matrix(params_host[k].rotate_deg, H, W, F.m);
        F.dx = plan[k].el ? fields + (size_t)plan[k].field * 2 * plane : nullptr;
        F.dy = F.dx ? F.dx + plane : nullptr;
      }
      if (c == kChunk || (k == n && c > 0)) {
        aug_labels_kernel<<<dim3((nj + kLabelThreads - 1) / kLabelThreads, c), kLabelThreads, 0, s>>>(a);
        CU_OK(h, cudaGetLastError());
        h->launches++;
        c = 0;
      }
    }
  }
  return DGP_OK;
}

}  // extern "C"
