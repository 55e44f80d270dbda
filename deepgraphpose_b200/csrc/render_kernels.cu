// Markers of the labelled video (plot_dgp / create_annotated_movie, src/deepgraphpose/models/eval.py): the reference draws
// each frame on the host, one joint at a time (DLC's skimage circle); here one CTA per frame walks the frame's paint sequence
// (trail discs, skeleton lines, discs) in order.  The threads first resolve up to 256 paints at once, one each (mask, centre,
// clipped box or visible line range), into shared memory; then the CTA paints them one after another, with a barrier after
// each, so that overlapping paints resolve the same way on every run (the later one wins).  Only painted pixels are written.
// The drawing contract is in include/dgp_b200.h.
#include "../../include/dgp_b200.h"

#include <cuda_runtime.h>
#include <math.h>

#include "handle.cuh"

namespace dgp {
namespace {

constexpr int kMarkerThreads = 256;
constexpr int kTableThreads = 256;
constexpr double kMinLineCentre = -1048576.0;  // -2^20: keeps the line arithmetic in int64
constexpr int kMaxLineFrame = 1 << 30;

enum PaintKind { PAINT_NONE = 0, PAINT_DISC = 1, PAINT_LINE = 2 };

// One resolved paint.  Disc: p = {r0, c0, box width, box pixels, xc, yc}.  Line: p = {ra, ca, dr, dc, n, k0, k1}, the
// pixels k0..k1 of the line being the ones inside the frame.
struct Paint {
  int kind;
  int p[7];
  uint8_t rgb[4];
};

__device__ __forceinline__ int64_t floor_div(int64_t a, int64_t b) {  // b > 0
  const int64_t q = a / b;
  return (a % b != 0 && a < 0) ? q - 1 : q;
}
__device__ __forceinline__ int64_t ceil_div64(int64_t a, int64_t b) { return -floor_div(-a, b); }

// The mask and the centre of the contract; false when the joint is not drawn (lines also need finite coordinates).
__device__ __forceinline__ bool centre(double x, double y, double l, const MarkerArgs& a, int H, int W, double* xt,
                                       double* yt) {
  if (!(l > a.mask_threshold) || isnan(x) || isnan(y)) return false;
  *xt = fmin(trunc(x), (double)(W - 1));
  *yt = fmin(trunc(y), (double)(H - 1));
  return true;
}

__device__ bool resolve_disc(double x, double y, double l, const uint8_t* rgb, const MarkerArgs& a, int H, int W, Paint* o) {
  double xt, yt;
  const int d = a.dotsize;
  if (!centre(x, y, l, a, H, W, &xt, &yt)) return false;
  if (xt <= -d || yt <= -d) return false;  // the disc lies left of / above the frame (and the centre may not fit an int)
  const int xc = (int)xt, yc = (int)yt;
  const int r0 = max(yc - d + 1, 0), r1 = min(yc + d - 1, H - 1);
  const int c0 = max(xc - d + 1, 0), c1 = min(xc + d - 1, W - 1);
  if (r0 > r1 || c0 > c1) return false;
  const int bw = c1 - c0 + 1;
  o->p[0] = r0; o->p[1] = c0; o->p[2] = bw; o->p[3] = bw * (r1 - r0 + 1); o->p[4] = xc; o->p[5] = yc;
  o->rgb[0] = rgb[0]; o->rgb[1] = rgb[1]; o->rgb[2] = rgb[2];
  return true;
}

// Offset of the line's pixel k along an axis moving by d over n steps: floor((2 k d + n) / 2n).  Exact in int32 while
// 2 n^2 + n < 2^31; the axis that moves by n is k itself.
__device__ __forceinline__ int line_offset(int64_t k, int64_t d, int64_t n) {
  if (d == n) return (int)k;
  if (d == -n) return (int)-k;
  if (n < 32768) {
    const int num = (int)(2 * k * d + n), den = (int)(2 * n);
    const int q = num / den;
    return (num % den != 0 && num < 0) ? q - 1 : q;
  }
  return (int)floor_div(2 * k * d + n, 2 * n);
}

// Narrows [*k0, *k1] to the k whose coordinate p0 + line_offset(k, d, n) lies in [0, hi]: the offset is monotone in k, so
// the set is an interval, found from floor(v) >= m <=> v >= m and floor(v) <= m <=> v < m + 1.
__device__ void clip_axis(int64_t p0, int64_t d, int64_t n, int64_t hi, int64_t* k0, int64_t* k1) {
  if (d == 0) {
    if (p0 < 0 || p0 > hi) *k1 = -1;
    return;
  }
  int64_t lo_k, hi_k;
  if (d > 0) {  // 2kd + n >= -2n p0  and  2kd + n < 2n (hi + 1 - p0)
    lo_k = ceil_div64(-2 * n * p0 - n, 2 * d);
    hi_k = floor_div(2 * n * (hi + 1 - p0) - n - 1, 2 * d);
  } else {      // with e = -d: n - 2ke >= -2n p0  and  n - 2ke < 2n (hi + 1 - p0)
    const int64_t e = -d;
    lo_k = ceil_div64(n - 2 * n * (hi + 1 - p0) + 1, 2 * e);
    hi_k = floor_div(n + 2 * n * p0, 2 * e);
  }
  *k0 = max(*k0, lo_k);
  *k1 = min(*k1, hi_k);
}

__device__ bool resolve_line(double xa, double ya, double la, double xb, double yb, double lb, const MarkerArgs& a, int H,
                             int W, Paint* o) {
  double xta, yta, xtb, ytb;
  if (!centre(xa, ya, la, a, H, W, &xta, &yta) || !centre(xb, yb, lb, a, H, W, &xtb, &ytb)) return false;
  if (isinf(xa) || isinf(ya) || isinf(xb) || isinf(yb)) return false;
  if (xta < kMinLineCentre || yta < kMinLineCentre || xtb < kMinLineCentre || ytb < kMinLineCentre) return false;
  const int64_t ra = (int64_t)yta, ca = (int64_t)xta;
  const int64_t dr = (int64_t)ytb - ra, dc = (int64_t)xtb - ca;
  const int64_t n = max(dr < 0 ? -dr : dr, dc < 0 ? -dc : dc);
  int64_t k0 = 0, k1 = n;
  clip_axis(ra, dr, n, H - 1, &k0, &k1);
  clip_axis(ca, dc, n, W - 1, &k0, &k1);
  if (k0 > k1) return false;
  o->p[0] = (int)ra; o->p[1] = (int)ca; o->p[2] = (int)dr; o->p[3] = (int)dc; o->p[4] = (int)n;
  o->p[5] = (int)k0; o->p[6] = (int)k1;
  o->rgb[0] = a.skeleton_color[0]; o->rgb[1] = a.skeleton_color[1]; o->rgb[2] = a.skeleton_color[2];
  return true;
}

// Paint s of frame t: the trail discs (s < n_trail), the skeleton edges, then the discs of frame t.  Rows of xs / ys / liks
// are frames relative to the CTA's; rows from -history are valid.
__device__ Paint resolve(int s, int t, int n_trail, int H, int W, const double* __restrict__ xs,
                         const double* __restrict__ ys, const double* __restrict__ liks, int history, const MarkerArgs& a) {
  Paint o;
  o.kind = PAINT_NONE;
  const int nj = a.nj;
  if (s < n_trail) {
    const int k = a.trailpoints - 1 - s / nj, j = s % nj;
    if (t - k < -history) return o;
    const ptrdiff_t i = (ptrdiff_t)(t - k) * nj + j;
    if (resolve_disc(xs[i], ys[i], liks[i], a.colors + 3 * j, a, H, W, &o)) o.kind = PAINT_DISC;
  } else if (s < n_trail + a.n_edges) {
    const int e = s - n_trail;
    const ptrdiff_t i = (ptrdiff_t)t * nj + a.edges[2 * e], k = (ptrdiff_t)t * nj + a.edges[2 * e + 1];
    if (resolve_line(xs[i], ys[i], liks[i], xs[k], ys[k], liks[k], a, H, W, &o)) o.kind = PAINT_LINE;
  } else {
    const int j = s - n_trail - a.n_edges;
    const ptrdiff_t i = (ptrdiff_t)t * nj + j;
    if (resolve_disc(xs[i], ys[i], liks[i], a.colors + 3 * j, a, H, W, &o)) o.kind = PAINT_DISC;
  }
  return o;
}

__global__ void __launch_bounds__(kMarkerThreads) draw_markers_kernel(uint8_t* __restrict__ frames, int H, int W,
                                                                     const double* __restrict__ xs,
                                                                     const double* __restrict__ ys,
                                                                     const double* __restrict__ liks, int history,
                                                                     const MarkerArgs a) {
  __shared__ Paint paints[kMarkerThreads];
  const int t = blockIdx.x;
  uint8_t* f = frames + (size_t)t * H * W * 3;
  const int n_trail = a.trailpoints >= 2 ? (a.trailpoints - 1) * a.nj : 0;
  const int n_paints = n_trail + a.n_edges + a.nj;
  const int d2 = a.dotsize * a.dotsize;
  for (int base = 0; base < n_paints; base += kMarkerThreads) {
    const int s = base + threadIdx.x;
    if (s < n_paints) paints[threadIdx.x] = resolve(s, t, n_trail, H, W, xs, ys, liks, history, a);
    __syncthreads();
    const int m = min(kMarkerThreads, n_paints - base);
    for (int i = 0; i < m; ++i) {
      const Paint& o = paints[i];
      // every thread reads the same record, so the skip (and the barrier below) is uniform over the CTA
      if (o.kind == PAINT_NONE) continue;
      const uint8_t cr = o.rgb[0], cg = o.rgb[1], cb = o.rgb[2];
      if (o.kind == PAINT_DISC) {
        const int r0 = o.p[0], c0 = o.p[1], bw = o.p[2], nbox = o.p[3], xc = o.p[4], yc = o.p[5];
        for (int q = threadIdx.x; q < nbox; q += kMarkerThreads) {
          const int r = r0 + q / bw, c = c0 + q % bw;
          const int dr = r - yc, dc = c - xc;
          if (dr * dr + dc * dc < d2) {
            uint8_t* p = f + ((size_t)r * W + c) * 3;
            p[0] = cr;
            p[1] = cg;
            p[2] = cb;
          }
        }
      } else {
        const int ra = o.p[0], ca = o.p[1], dr = o.p[2], dc = o.p[3], n = o.p[4], k1 = o.p[6];
        for (int k = o.p[5] + threadIdx.x; k <= k1; k += kMarkerThreads) {
          const int r = ra + line_offset(k, dr, n), c = ca + line_offset(k, dc, n);
          uint8_t* p = f + ((size_t)r * W + c) * 3;
          p[0] = cr;
          p[1] = cg;
          p[2] = cb;
        }
      }
      __syncthreads();
    }
    __syncthreads();  // the next chunk overwrites `paints`
  }
}

// x, y in video pixels exactly as eval.estimate_pose forms them on the host (float64, unfused multiply then add, then the
// scale), and lik widened.
__global__ void __launch_bounds__(kTableThreads) marker_table_kernel(const float* __restrict__ mu,
                                                                     const float* __restrict__ likf, int count, double stride,
                                                                     double half_stride, double scale_x, double scale_y,
                                                                     double* __restrict__ xs, double* __restrict__ ys,
                                                                     double* __restrict__ liks) {
  const int i = blockIdx.x * kTableThreads + threadIdx.x;
  if (i >= count) return;
  xs[i] = __dmul_rn(__dadd_rn(__dmul_rn((double)mu[2 * i + 1], stride), half_stride), scale_x);
  ys[i] = __dmul_rn(__dadd_rn(__dmul_rn((double)mu[2 * i], stride), half_stride), scale_y);
  liks[i] = (double)likf[i];
}

}  // namespace

int marker_args(dgp_handle* h, const dgp_marker_style* st, int H, int W, MarkerArgs* a) {
  if (!st || !st->colors) return fail(h, DGP_ERR_INVALID, "dgp_marker_style: null style or colour table");
  if (st->dotsize < 0 || st->dotsize > kMaxDotsize)
    return fail(h, DGP_ERR_INVALID, "dgp_marker_style: dotsize %d outside [0, %d]", st->dotsize, kMaxDotsize);
  a->nj = h->cfg.num_joints;
  if (st->n_edges < 0 || st->n_edges > kMaxEdges || (st->n_edges > 0 && !st->edges))
    return fail(h, DGP_ERR_INVALID, "dgp_marker_style: %d edges (at most %d, and a table for any)", st->n_edges, kMaxEdges);
  for (int e = 0; e < st->n_edges; ++e)
    for (int s = 0; s < 2; ++s) {
      const int32_t j = st->edges[2 * e + s];
      if (j < 0 || j >= a->nj)
        return fail(h, DGP_ERR_INVALID, "dgp_marker_style: edge %d joint %d outside [0, %d)", e, (int)j, a->nj);
      a->edges[2 * e + s] = (uint8_t)j;
    }
  if (st->n_edges > 0 && (H > kMaxLineFrame || W > kMaxLineFrame))
    return fail(h, DGP_ERR_INVALID, "dgp_marker_style: skeleton lines on a %dx%d frame (at most %d a side)", H, W,
                kMaxLineFrame);
  if (st->trailpoints < 0 || st->trailpoints > kMaxTrailpoints)
    return fail(h, DGP_ERR_INVALID, "dgp_marker_style: trailpoints %d outside [0, %d]", st->trailpoints, kMaxTrailpoints);
  a->dotsize = st->dotsize;
  a->n_edges = st->n_edges;
  a->trailpoints = st->trailpoints;
  a->mask_threshold = st->mask_threshold;
  a->scale_x = st->scale_x;
  a->scale_y = st->scale_y;
  a->stride = (double)h->cfg.stride;
  a->half_stride = 0.5 * a->stride;
  for (int i = 0; i < 3 * a->nj; ++i) a->colors[i] = st->colors[i];
  for (int i = 0; i < 3; ++i) a->skeleton_color[i] = st->skeleton_color[i];
  return DGP_OK;
}

int draw_markers_impl(dgp_handle* h, uint8_t* frames, int N, int H, int W, const double* xs, const double* ys,
                      const double* liks, int history, const MarkerArgs& a, cudaStream_t s) {
  if (N == 0 || (a.dotsize == 0 && a.n_edges == 0)) return DGP_OK;
  draw_markers_kernel<<<N, kMarkerThreads, 0, s>>>(frames, H, W, xs, ys, liks, history, a);
  CU_OK(h, cudaGetLastError());
  h->launches++;
  return DGP_OK;
}

int marker_table_fused(dgp_handle* h, const float* mu, const float* lik, int n, const MarkerArgs& a, double* xs, double* ys,
                       double* liks, cudaStream_t s) {
  const int count = n * a.nj;
  if (count == 0) return DGP_OK;
  marker_table_kernel<<<(count + kTableThreads - 1) / kTableThreads, kTableThreads, 0, s>>>(
      mu, lik, count, a.stride, a.half_stride, a.scale_x, a.scale_y, xs, ys, liks);
  CU_OK(h, cudaGetLastError());
  h->launches++;
  return DGP_OK;
}

}  // namespace dgp

extern "C" {

int dgp_draw_markers(dgp_handle* h, uint8_t* frames_dev, int N, int H, int W, const double* x_dev, const double* y_dev,
                     const double* lik_dev, const dgp_marker_style* style, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (N < 0 || H < 1 || W < 1 || (N > 0 && (!frames_dev || !x_dev || !y_dev || !lik_dev)))
    return fail(h, DGP_ERR_INVALID, "dgp_draw_markers: bad argument");
  MarkerArgs a;
  int rc = marker_args(h, style, H, W, &a);
  if (rc) return rc;
  const int max_history = a.trailpoints > 1 ? a.trailpoints - 1 : 0;
  if (style->history < 0 || style->history > max_history)
    return fail(h, DGP_ERR_INVALID, "dgp_draw_markers: history %d outside [0, %d] (trailpoints - 1)", style->history,
                max_history);
  if (N == 0) return DGP_OK;
  CU_OK(h, cudaSetDevice(h->device));
  const size_t off = (size_t)style->history * a.nj;
  return draw_markers_impl(h, frames_dev, N, H, W, x_dev + off, y_dev + off, lik_dev + off, style->history, a,
                           (cudaStream_t)stream);
}

}  // extern "C"
