// Frame resize + crop on the device, bit-exact to Pillow's 8-bit resample (Image.resize with its default filter for RGB,
// BICUBIC, then Image.crop): the `new_size` / `crop_size` options of estimate_pose (reference eval.py:309-326).
//
// Pillow's 8-bit path (libImaging/Resample.c) is integer arithmetic on a table of fixed-point weights built in double, so
// the host builds the same table once per (in, out) size pair and two table-driven uint8 1-D passes reproduce it exactly:
// horizontal first (into a uint8 intermediate), then vertical, a pass being skipped when its size does not change.  Only
// the part of the resized frame that the crop box covers is computed; box pixels outside the resized frame are 0.
#include "../../include/dgp_b200.h"

#include <cuda_runtime.h>

#include <cmath>
#include <vector>

#include "handle.cuh"

namespace {

constexpr int kPrecisionBits = 22;  // Pillow's PRECISION_BITS for 8-bit images
constexpr int kHThreads = 256;
constexpr int kVThreads = 128;
constexpr int kMaxSmem = 227 * 1024;

double bicubic_filter(double x) {  // Resample.c bicubic_filter, a = -0.5
  const double a = -0.5;
  if (x < 0.0) x = -x;
  if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
  if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
  return 0.0;
}

// Resample.c precompute_coeffs + normalize_coeffs_8bpc for BICUBIC (support 2).  The operations and their order are
// Pillow's, in double, so the rounded weights are the same integers.
int pillow_taps(int in_size, int out_size) {
  const double scale = (double)in_size / out_size;
  const double fs = scale < 1.0 ? 1.0 : scale;
  return (int)std::ceil(2.0 * fs) * 2 + 1;
}

void pillow_coeffs(int in_size, int out_size, int ksize, int32_t* first, int32_t* count, int32_t* weights) {
  const double scale = (double)in_size / out_size;
  const double fs = scale < 1.0 ? 1.0 : scale;
  const double support = 2.0 * fs;
  const double ss = 1.0 / fs;
  std::vector<double> k(ksize);
  for (int xx = 0; xx < out_size; ++xx) {
    const double center = (xx + 0.5) * scale;
    int xmin = (int)(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)(center + support + 0.5);
    if (xmax > in_size) xmax = in_size;
    xmax -= xmin;
    double ww = 0.0;
    for (int x = 0; x < xmax; ++x) {
      k[x] = bicubic_filter((x + xmin - center + 0.5) * ss);
      ww += k[x];
    }
    int32_t* row = weights + (size_t)xx * ksize;
    for (int x = 0; x < ksize; ++x) {
      double w = x < xmax ? k[x] : 0.0;
      if (x < xmax && ww != 0.0) w /= ww;
      row[x] = w < 0 ? (int32_t)(-0.5 + w * (1 << kPrecisionBits)) : (int32_t)(0.5 + w * (1 << kPrecisionBits));
    }
    first[xx] = xmin;
    count[xx] = xmax;
  }
}

struct Geometry {
  int H0, W0;            // source frame
  int Hr, Wr;            // resized frame (= source when there is no resize)
  int x0, y0, Hout, Wout;  // crop box origin in the resized frame, output frame
  int cx0, cx1, cy0, cy1;  // part of the box inside the resized frame (empty when cx1 <= cx0 or cy1 <= cy0)
};

// Validates a transform; the NULL / all-zero transform is the identity.
int geometry(int H0, int W0, const dgp_frame_transform* t, Geometry* g) {
  if (H0 < 1 || W0 < 1) return DGP_ERR_INVALID;
  g->H0 = H0; g->W0 = W0;
  g->Hr = H0; g->Wr = W0;
  if (t && (t->resize_h != 0 || t->resize_w != 0)) {
    if (t->resize_h < 1 || t->resize_w < 1) return DGP_ERR_INVALID;
    g->Hr = t->resize_h; g->Wr = t->resize_w;
  }
  int64_t x0 = 0, y0 = 0, x1 = g->Wr, y1 = g->Hr;
  if (t && (t->crop_x0 || t->crop_y0 || t->crop_x1 || t->crop_y1)) {
    x0 = t->crop_x0; y0 = t->crop_y0; x1 = t->crop_x1; y1 = t->crop_y1;
    if (x1 <= x0 || y1 <= y0) return DGP_ERR_INVALID;
  }
  // frame bytes (and every index within a frame) must fit an int
  if ((int64_t)H0 * W0 * 3 > INT32_MAX || (x1 - x0) * (y1 - y0) * 3 > INT32_MAX || (int64_t)g->Hr * g->Wr * 3 > INT32_MAX)
    return DGP_ERR_INVALID;
  auto clampi = [](int64_t v, int hi) { return (int)(v < 0 ? 0 : (v > hi ? hi : v)); };
  g->x0 = (int)x0; g->y0 = (int)y0;
  g->Wout = (int)(x1 - x0); g->Hout = (int)(y1 - y0);
  g->cx0 = clampi(x0, g->Wr); g->cx1 = clampi(x1, g->Wr);
  g->cy0 = clampi(y0, g->Hr); g->cy1 = clampi(y1, g->Hr);
  return DGP_OK;
}

// One block per source row (n, r): stage the row's needed byte span in shared memory (16 B loads between the unaligned
// head and tail), resample columns [0, Wv) of the table, and store the uint8 row with 16 B stores (the intermediate's
// pitch is a multiple of 16).
__global__ void __launch_bounds__(kHThreads) resize_h_kernel(const uint8_t* __restrict__ src, int H0, int W0, int r0, int R,
                                                            const int32_t* __restrict__ first, const int32_t* __restrict__ count,
                                                            const int32_t* __restrict__ weights, int ksize, int Wv, int span0,
                                                            int span_bytes, uint8_t* __restrict__ tmp, int tmp_pitch) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int n = blockIdx.x / R, r = blockIdx.x - n * R;
  const uint8_t* g = src + ((size_t)n * H0 + r0 + r) * W0 * 3 + (size_t)span0 * 3;
  const int shift = (int)((uintptr_t)g & 15);
  uint8_t* srow = smem;                                // row bytes at srow[shift + k], k < span_bytes
  uint8_t* orow = smem + ((shift + span_bytes + 15) & ~15);
  const int head = (16 - shift) & 15;
  const int n16 = span_bytes > head ? (span_bytes - head) >> 4 : 0;
  for (int k = threadIdx.x; k < span_bytes; k += blockDim.x) {
    if (k < head || k >= head + 16 * n16) srow[shift + k] = g[k];
  }
  for (int i = threadIdx.x; i < n16; i += blockDim.x)
    reinterpret_cast<uint4*>(srow + shift + head)[i] = __ldg(reinterpret_cast<const uint4*>(g + head) + i);
  __syncthreads();
  for (int j = threadIdx.x; j < Wv; j += blockDim.x) {
    const uint8_t* p = srow + shift + (first[j] - span0) * 3;
    const int32_t* w = weights + (size_t)j * ksize;
    const int c = count[j];
    int a0 = 1 << (kPrecisionBits - 1), a1 = a0, a2 = a0;
    for (int t = 0; t < c; ++t) {
      const int wt = __ldg(w + t);
      a0 += p[3 * t] * wt;
      a1 += p[3 * t + 1] * wt;
      a2 += p[3 * t + 2] * wt;
    }
    orow[3 * j] = (uint8_t)min(max(a0 >> kPrecisionBits, 0), 255);
    orow[3 * j + 1] = (uint8_t)min(max(a1 >> kPrecisionBits, 0), 255);
    orow[3 * j + 2] = (uint8_t)min(max(a2 >> kPrecisionBits, 0), 255);
  }
  __syncthreads();
  uint4* dst = reinterpret_cast<uint4*>(tmp + ((size_t)n * R + r) * tmp_pitch);
  for (int i = threadIdx.x; i < tmp_pitch / 16; i += blockDim.x) dst[i] = reinterpret_cast<const uint4*>(orow)[i];
}

struct VArgs {
  const uint8_t* in;   // row 0 of frame 0 of the input, at the byte of the first valid column
  size_t in_frame;     // bytes per input frame
  int in_pitch;        // bytes per input row
  int in_readable;     // bytes readable from a row's first valid column (>= the valid bytes)
  int in_row0;         // resized-frame row of input row 0
  const int32_t *first, *count, *weights;  // vertical table (NULL: rows are copied)
  int ksize;
  uint8_t* out;
  int Hout, row_bytes;  // output frame
  int vy0, vy1;        // valid output rows
  int vo, vlen;        // valid output bytes of a row: [vo, vo + vlen)
  int y0;              // resized-frame row of output row 0
  int chunks;          // 16-byte chunks per output row
};

// One thread per 16 output bytes of a row: a vertical resample (or a copy) of the valid part, 0 elsewhere.  Input rows
// are read with 16 B loads when the address is aligned, which the intermediate's layout guarantees whenever the box does
// not start left of the frame.
__global__ void __launch_bounds__(kVThreads) resize_v_kernel(VArgs a, int64_t total) {
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= total) return;
  const int ci = (int)(gid % a.chunks);
  const int64_t rowid = gid / a.chunks;
  const int oy = (int)(rowid % a.Hout);
  const int n = (int)(rowid / a.Hout);
  const int o = ci * 16;
  const int q = o - a.vo;  // input byte of output byte o, relative to the first valid column
  int acc[16];
  const bool row_ok = oy >= a.vy0 && oy < a.vy1 && q + 16 > 0 && q < a.vlen;
  if (row_ok) {
    const int yy = a.y0 + oy;
    int first = yy, cnt = 1;
    const int32_t* w = nullptr;
    if (a.first) { first = a.first[yy]; cnt = a.count[yy]; w = a.weights + (size_t)yy * a.ksize; }
    const uint8_t* base = a.in + (size_t)n * a.in_frame + (size_t)(first - a.in_row0) * a.in_pitch;
#pragma unroll
    for (int j = 0; j < 16; ++j) acc[j] = w ? 1 << (kPrecisionBits - 1) : 0;
    const bool vec = q >= 0 && q + 16 <= a.in_readable && (((uintptr_t)(base + q) | (uintptr_t)a.in_pitch) & 15) == 0;
    for (int t = 0; t < cnt; ++t) {
      const uint8_t* p = base + (size_t)t * a.in_pitch + q;
      const int wt = w ? __ldg(w + t) : 1;
      uint4 v;
      if (vec) {
        v = __ldg(reinterpret_cast<const uint4*>(p));
      } else {
        uint32_t* vw = &v.x;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          uint32_t word = 0;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int j = 4 * i + k;
            if (q + j >= 0 && q + j < a.vlen) word |= (uint32_t)p[j] << (8 * k);
          }
          vw[i] = word;
        }
      }
      const uint32_t* vw = &v.x;
#pragma unroll
      for (int j = 0; j < 16; ++j) acc[j] += (int)((vw[j >> 2] >> (8 * (j & 3))) & 255u) * wt;
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int v = w ? min(max(acc[j] >> kPrecisionBits, 0), 255) : acc[j];
      acc[j] = (q + j >= 0 && q + j < a.vlen) ? v : 0;
    }
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) acc[j] = 0;
  }
  uint8_t* dst = a.out + ((size_t)n * a.Hout + oy) * a.row_bytes + o;
  if (o + 16 <= a.row_bytes && ((uintptr_t)dst & 15) == 0) {
    uint4 v;
    uint32_t* vw = &v.x;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      vw[i] = (uint32_t)acc[4 * i] | ((uint32_t)acc[4 * i + 1] << 8) | ((uint32_t)acc[4 * i + 2] << 16) |
              ((uint32_t)acc[4 * i + 3] << 24);
    *reinterpret_cast<uint4*>(dst) = v;
  } else {
    const int m = min(16, a.row_bytes - o);
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (j < m) dst[j] = (uint8_t)acc[j];
  }
}

}  // namespace

namespace dgp {

// The table of one (in, out) size pair, built on first use and kept on the handle: device copy for the kernels, host copy
// of the bounds for the launch geometry.
static int resize_table(dgp_handle* h, int in_size, int out_size, const ResizeTable** out) {
  auto key = std::make_pair(in_size, out_size);
  auto it = h->resize_tables.find(key);
  if (it == h->resize_tables.end()) {
    ResizeTable t;
    t.ksize = pillow_taps(in_size, out_size);
    std::vector<int32_t> host((size_t)out_size * (2 + t.ksize));
    pillow_coeffs(in_size, out_size, t.ksize, host.data(), host.data() + out_size, host.data() + 2 * (size_t)out_size);
    t.first.assign(host.begin(), host.begin() + out_size);
    t.count.assign(host.begin() + out_size, host.begin() + 2 * out_size);
    CU_OK(h, t.dev.alloc(host.size() * 4));
    CU_OK(h, cudaMemcpy(t.dev.get(), host.data(), host.size() * 4, cudaMemcpyHostToDevice));
    it =h->resize_tables.emplace(key, std::move(t)).first;
  }
  *out = &it->second;
  return DGP_OK;
}

int resize_crop_impl(dgp_handle* h, const uint8_t* src, int N, int H0, int W0, const dgp_frame_transform* tf, uint8_t* dst,
                     cudaStream_t s) {
  Geometry g;
  if (geometry(H0, W0, tf, &g)) return fail(h, DGP_ERR_INVALID, "dgp_resize_crop: invalid frame size or transform");
  if (N < 0 || (N > 0 && (!src || !dst))) return fail(h, DGP_ERR_INVALID, "dgp_resize_crop: bad argument");
  if (N == 0) return DGP_OK;
  const bool empty = g.cx1 <= g.cx0 || g.cy1 <= g.cy0;  // the box lies outside the resized frame: all zeros
  const bool hpass = g.Wr != W0 && !empty, vpass = g.Hr != H0 && !empty;
  const ResizeTable *th = nullptr, *tv = nullptr;
  int rc;
  if (hpass && (rc = resize_table(h, W0, g.Wr, &th))) return rc;
  if (vpass && (rc = resize_table(h, H0, g.Hr, &tv))) return rc;
  const int Wv = empty ? 0 : g.cx1 - g.cx0;
  VArgs a;
  a.first = a.count = a.weights = nullptr;
  a.ksize = 0;
  if (vpass) {
    a.first = tv->dev.get<int32_t>();
    a.count = a.first + g.Hr;
    a.weights = a.first + 2 * (size_t)g.Hr;
    a.ksize = tv->ksize;
  }
  a.out = dst;
  a.Hout = g.Hout;
  a.row_bytes = g.Wout * 3;
  a.vy0 = empty ? 0 : g.cy0 - g.y0;
  a.vy1 = empty ? 0 : g.cy1 - g.y0;
  a.vo = (g.cx0 - g.x0) * 3;
  a.vlen = Wv * 3;
  a.y0 = g.y0;
  a.chunks = (a.row_bytes + 15) / 16;
  // without a horizontal pass the vertical pass reads the source frames themselves
  a.in = src + (size_t)g.cx0 * 3;
  a.in_frame = (size_t)H0 * W0 * 3;
  a.in_pitch = W0 * 3;
  a.in_readable = (W0 - g.cx0) * 3;
  a.in_row0 = 0;
  if (hpass) {
    // source rows the vertical pass reads: first and first + count are non-decreasing in the output row
    int r0 = g.cy0, r1 = g.cy1;
    if (vpass) {
      r0 = tv->first[g.cy0];
      r1 = tv->first[g.cy1 - 1] + tv->count[g.cy1 - 1];
    }
    const int R = r1 - r0;
    const int span0 = th->first[g.cx0];
    const int span_bytes = (th->first[g.cx1 - 1] + th->count[g.cx1 - 1] - span0) * 3;
    const int pitch = (Wv * 3 + 15) & ~15;
    const size_t smem = (size_t)((15 + span_bytes + 15) & ~15) + pitch;
    if (smem > (size_t)kMaxSmem)
      return fail(h, DGP_ERR_UNSUPPORTED, "dgp_resize_crop: a %d-pixel source row does not fit in shared memory", W0);
    if ((int64_t)R * N > INT32_MAX) return fail(h, DGP_ERR_UNSUPPORTED, "dgp_resize_crop: too many rows in one call");
    if ((rc = ensure(h, &h->resize_tmp, (size_t)N * R * pitch))) return rc;
    if (smem > 48 * 1024)
      CU_OK(h, cudaFuncSetAttribute(resize_h_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int32_t* tab = th->dev.get<int32_t>();
    resize_h_kernel<<<R * N, kHThreads, smem, s>>>(src, H0, W0, r0, R, tab + g.cx0, tab + g.Wr + g.cx0,
                                                   tab + 2 * (size_t)g.Wr + (size_t)g.cx0 * th->ksize, th->ksize, Wv,
                                                   span0, span_bytes, h->resize_tmp.get<uint8_t>(), pitch);
    CU_OK(h, cudaGetLastError());
    h->launches++;
    a.in = h->resize_tmp.get<uint8_t>();
    a.in_frame = (size_t)R * pitch;
    a.in_pitch = pitch;
    a.in_readable = pitch;
    a.in_row0 = r0;
  }
  const int64_t total = (int64_t)N * g.Hout * a.chunks;
  const int64_t blocks = (total + kVThreads - 1) / kVThreads;
  if (blocks > INT32_MAX) return fail(h, DGP_ERR_UNSUPPORTED, "dgp_resize_crop: output too large for one call");
  resize_v_kernel<<<(unsigned)blocks, kVThreads, 0, s>>>(a, total);
  CU_OK(h, cudaGetLastError());
  h->launches++;
  return DGP_OK;
}

int transform_dims(int H0, int W0, const dgp_frame_transform* t, int* H, int* W, bool* identity) {
  Geometry g;
  if (geometry(H0, W0, t, &g)) return DGP_ERR_INVALID;
  *H = g.Hout;
  *W = g.Wout;
  *identity = g.Hr == H0 && g.Wr == W0 && g.x0 == 0 && g.y0 == 0 && g.Hout == H0 && g.Wout == W0;
  return DGP_OK;
}

}  // namespace dgp

extern "C" {

int dgp_transform_dims(int H0, int W0, const dgp_frame_transform* t, int* H, int* W) {
  Geometry g;
  if (geometry(H0, W0, t, &g)) return DGP_ERR_INVALID;
  if (H) *H = g.Hout;
  if (W) *W = g.Wout;
  return DGP_OK;
}

int dgp_resize_coefficients(int in_size, int out_size, int max_taps, int32_t* first, int32_t* count, int32_t* weights) {
  if (in_size < 1 || out_size < 1 || !first || !count || !weights) return DGP_ERR_INVALID;
  const int ksize = pillow_taps(in_size, out_size);
  if (max_taps < 1) return DGP_ERR_INVALID;
  std::vector<int32_t> w((size_t)out_size * ksize);
  pillow_coeffs(in_size, out_size, ksize, first, count, w.data());
  for (int xx = 0; xx < out_size; ++xx) {
    if (count[xx] > max_taps) return DGP_ERR_INVALID;
    for (int x = 0; x < max_taps; ++x) weights[(size_t)xx * max_taps + x] = x < ksize ? w[(size_t)xx * ksize + x] : 0;
  }
  return DGP_OK;
}

int dgp_resize_crop(dgp_handle* h, const uint8_t* src_dev, int N, int H0, int W0, const dgp_frame_transform* t,
                    uint8_t* dst_dev, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  CU_OK(h, cudaSetDevice(h->device));
  return resize_crop_impl(h, src_dev, N, H0, W0, t, dst_dev, (cudaStream_t)stream);
}

}  // extern "C"
