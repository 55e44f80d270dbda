// Markers of the labelled video (plot_dgp / create_annotated_movie, src/deepgraphpose/models/eval.py): the reference draws
// each frame on the host, one joint at a time (DLC's skimage circle); here one CTA per frame walks the joints in index order
// and paints each disc's bounding box, with a barrier between joints so that overlapping discs resolve the same way on every
// run (the higher joint index wins).  Only disc pixels are written.  The drawing contract is in include/dgp_b200.h.
#include "../../include/dgp_b200.h"

#include <cuda_runtime.h>
#include <math.h>

#include "handle.cuh"

namespace dgp {
namespace {

constexpr int kMarkerThreads = 256;

// kFused: the coordinates come from the float32 soft-argmax of estimate_pose's batch, converted to video pixels exactly as
// eval.estimate_pose does on the host (float64, unfused multiply then add, then the scale); otherwise from float64 arrays.
template <bool kFused>
__global__ void __launch_bounds__(kMarkerThreads) draw_markers_kernel(uint8_t* __restrict__ frames, int H, int W,
                                                                     const double* __restrict__ xs,
                                                                     const double* __restrict__ ys,
                                                                     const double* __restrict__ liks,
                                                                     const float* __restrict__ mu,
                                                                     const float* __restrict__ likf, const MarkerArgs a) {
  const int t = blockIdx.x;
  uint8_t* f = frames + (size_t)t * H * W * 3;
  const int d = a.dotsize;
  for (int j = 0; j < a.nj; ++j) {
    const size_t k = (size_t)t * a.nj + j;
    double x, y, l;
    if (kFused) {
      x = __dmul_rn(__dadd_rn(__dmul_rn((double)mu[2 * k + 1], a.stride), a.half_stride), a.scale_x);
      y = __dmul_rn(__dadd_rn(__dmul_rn((double)mu[2 * k], a.stride), a.half_stride), a.scale_y);
      l = (double)likf[k];
    } else {
      x = xs[k];
      y = ys[k];
      l = liks[k];
    }
    // every thread computes the same decision, so the skip (and the barrier below) is uniform over the CTA
    if (!(l > a.mask_threshold) || isnan(x) || isnan(y)) continue;
    const double xt = fmin(trunc(x), (double)(W - 1)), yt = fmin(trunc(y), (double)(H - 1));
    if (xt <= -d || yt <= -d) continue;  // the disc lies left of / above the frame (and the centre may not fit an int)
    const int xc = (int)xt, yc = (int)yt;
    const int r0 = max(yc - d + 1, 0), r1 = min(yc + d - 1, H - 1);
    const int c0 = max(xc - d + 1, 0), c1 = min(xc + d - 1, W - 1);
    if (r0 > r1 || c0 > c1) continue;
    const int bw = c1 - c0 + 1, nbox = bw * (r1 - r0 + 1);
    const uint8_t cr = a.colors[3 * j], cg = a.colors[3 * j + 1], cb = a.colors[3 * j + 2];
    for (int i = threadIdx.x; i < nbox; i += kMarkerThreads) {
      const int r = r0 + i / bw, c = c0 + i % bw;
      const int dr = r - yc, dc = c - xc;
      if (dr * dr + dc * dc < d * d) {
        uint8_t* p = f + ((size_t)r * W + c) * 3;
        p[0] = cr;
        p[1] = cg;
        p[2] = cb;
      }
    }
    __syncthreads();
  }
}

}  // namespace

int marker_args(dgp_handle* h, const dgp_marker_style* st, MarkerArgs* a) {
  if (!st || !st->colors) return fail(h, DGP_ERR_INVALID, "dgp_marker_style: null style or colour table");
  if (st->dotsize < 0 || st->dotsize > kMaxDotsize)
    return fail(h, DGP_ERR_INVALID, "dgp_marker_style: dotsize %d outside [0, %d]", st->dotsize, kMaxDotsize);
  a->nj = h->cfg.num_joints;
  a->dotsize = st->dotsize;
  a->mask_threshold = st->mask_threshold;
  a->scale_x = st->scale_x;
  a->scale_y = st->scale_y;
  a->stride = (double)h->cfg.stride;
  a->half_stride = 0.5 * a->stride;
  for (int i = 0; i < 3 * a->nj; ++i) a->colors[i] = st->colors[i];
  return DGP_OK;
}

int draw_markers_fused(dgp_handle* h, uint8_t* frames, int N, int H, int W, const float* mu, const float* lik,
                       const MarkerArgs& a, cudaStream_t s) {
  if (N == 0 || a.dotsize == 0) return DGP_OK;
  draw_markers_kernel<true><<<N, kMarkerThreads, 0, s>>>(frames, H, W, nullptr, nullptr, nullptr, mu, lik, a);
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
  int rc = marker_args(h, style, &a);
  if (rc) return rc;
  if (N == 0 || a.dotsize == 0) return DGP_OK;
  CU_OK(h, cudaSetDevice(h->device));
  draw_markers_kernel<false><<<N, kMarkerThreads, 0, (cudaStream_t)stream>>>(frames_dev, H, W, x_dev, y_dev, lik_dev, nullptr,
                                                                            nullptr, a);
  CU_OK(h, cudaGetLastError());
  h->launches++;
  return DGP_OK;
}

}  // extern "C"
