// Launchers of the bandwidth-class kernels (softargmax.cu, aux_kernels.cu).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace dgp {

struct SaPartial {  // per (frame, row-split, joint) partial of the online softmax + DLC peak search
  float m, s0, sr, sc, bsig;
  int bidx;
  int pad0, pad1;
};

int softargmax_tact(int nj);
int softargmax_splits(int H, int W, int nj);  // segments per frame (workspace = B * splits * nj SaPartial)
cudaError_t launch_softargmax(const float* logits, const float* locref, int B, int H, int W, int nj, float gamma,
                              float gauss_len, float stride, float locref_stdev, SaPartial* workspace, int splits,
                              float* mu, int* peak, float* lik, int* dlc_peak, float* dlc_pose, float* norm,
                              cudaStream_t stream);
cudaError_t launch_softmax_map(const float* logits, const float* norm, int B, int H, int W, int nj, float gamma,
                               float gauss_len, float* out, int num_sms, cudaStream_t stream);
cudaError_t launch_sigmoid_map(const float* x, float* y, size_t n, int num_sms, cudaStream_t stream);
cudaError_t launch_potentials(const float* mu, const float* halo_next, int T, int nj, const int* edges, int nl,
                              float stride, const float* ws, const float* ws_max, float wt_max, float* skel,
                              float* temporal, float* e_skel, float* e_temp, cudaStream_t stream);

// u8 RGB frames (N,H,W,3) -> mean-subtracted, zero-padded, space-to-depth bf16 (N,Hs,Ws,16), Hs=ceil(H/2)+3.
cudaError_t launch_prep_s2d(const uint8_t* frames, int N, int H, int W, const float* mean3, __nv_bfloat16* out,
                            int Hs, int Ws, int fp16, cudaStream_t stream);
// 3x3 stride-2 max-pool with TF SAME padding on NHWC bf16 (C multiple of 8).
cudaError_t launch_maxpool3x3s2(const __nv_bfloat16* in, int N, int H, int W, int C, __nv_bfloat16* out, int Ho,
                                int Wo, int pad_t, int pad_l, int fp16, cudaStream_t stream);
// col2im of the head GEMM: contrib (N*h*w, ldn) fp32 with column (kh*3+kw)*ctot + co ->
// part logits (N,2h,2w,nj) [+ locref (N,2h,2w,2nj)] with bias.
cudaError_t launch_deconv_col2im(const float* contrib, int N, int h, int w, int ldn, int ctot, int nj,
                                 const float* bias, float* logits, float* locref, cudaStream_t stream);

// argmax_2d_from_cm(th=...): threshold + renormalise the blurred softmax map in place and return E[(row, col)] (B,nj,2).
cudaError_t launch_softmax_threshold(float* map, int B, int H, int W, int nj, float th, float* mu, cudaStream_t stream);

// 16-bit storage (bf16 / fp16) <-> float32, elementwise (boundary entry points that hand activations to the caller).
cudaError_t launch_cvt16_to_f32(const void* in, float* out, size_t n, int fp16, cudaStream_t stream);
cudaError_t launch_f32_to_cvt16(const float* in, void* out, size_t n, int fp16, cudaStream_t stream);

// Forward DGP loss on the head outputs (loss_kernels.cu).  All pointers are device pointers.
struct LossArgs {
  const float* pred; const float* locref; const float* mu;  // (nt,H,W,nj), (nt,H,W,2nj) or null, (nt,nj,2)
  int nt, H, W, nj;
  const float* targets;                                     // (nv,nj,2), NaN = missing label
  const float* locref_map; const float* locref_mask;        // (nt,H,W,2nj)
  const int* visible; int nbv; const int* hidden; int nbh; const int* vis_in_targets;
  const int* edges; int nl; const float* ws; const float* ws_max;
  const float* flow; int Hin, Win; const float* wt_batch;   // (nt-1,Hin,Win), (nt-1) = wt * mask
  float stride, lengthscale, wt, wt_max, wn_visible, wn_hidden, locref_weight, n_vis_total, n_hid_total;
  int gm2, gm3;
  int locref_mse;       // 0 = Huber (k = 1) locref loss, 1 = mean squared error (dgp_cfg.locref_huber_loss False)
  float* all_markers;   // scratch (nt*nj,2): targets_all_marker
  float4* partials;     // scratch (nbv+nbh)
  float* meanflow;      // scratch ((nt-1)*nj)
  float* flow_part;     // scratch ((nt-1)*nj * ceil(Hin/16) * 8): per row-slab partial sums of the flow box means
  float4* boxgrad;      // scratch ((nt-1)*nj): d meanflow / d (y1, x1, y2, x2) of the crop box, or nullptr (forward only)
  float* out;           // [6]
};
cudaError_t launch_dgp_loss(const LossArgs& a, cudaStream_t stream);
// Gradients of total_loss (or total_loss_visible) w.r.t. pred / locref; needs launch_dgp_loss's partials + all_markers.
cudaError_t launch_dgp_loss_backward(const LossArgs& a, const float* norm, float gamma, float gauss_len, int visible_only,
                                     float* g_pred, float* g_locref, cudaStream_t stream);

// ---- parameter arena / optimizer (param_kernels.cu)
cudaError_t launch_refresh_w16(const float* master, void* w16, size_t n, int fp16, cudaStream_t s);
cudaError_t launch_refresh_bn(const float* gamma, const float* beta, const float* mean, const float* var, float eps, int n,
                              float* scale, float* shift, cudaStream_t s);
// wd[ci][T-1-tap][co] = round16(w[co][tap][ci] * scale[co]) for every conv layer in one launch: one job per layer,
// tile_start = prefix sum of (Cin/32)*(Cout/32)*taps over the jobs (Cin, Cout multiples of 32).
struct DgradWJob {
  size_t w_off;     // offset of w [Cout][taps*Cin] in the master arena
  uint16_t* wd;     // [Cin][taps*Cout]
  int ch_off;       // offset of the layer's channels in the BN scale arena
  int Cout, taps, Cin;
  int tile_start;
};
constexpr int kDgradWMaxJobs = 256;  // build_dgrad_w_kernel looks a block's job up with one thread per job (256 threads)
cudaError_t launch_build_dgrad_w(const DgradWJob* jobs_dev, int njobs, int total_tiles, const float* master,
                                 const float* scale_arena, int fp16, cudaStream_t s);
cudaError_t launch_build_head_dgrad_w(const float* wh, int rows, int C, void* whT, int Kd, int fp16, cudaStream_t s);
int sqnorm_partials();
// norm_clip[0] = |grad_scale| * ||g||_2, norm_clip[1] = clip / max(norm, clip) (1 if clip <= 0)
cudaError_t launch_global_norm(const float* g, size_t n, float grad_scale, float clip, float* partial, float* norm_clip,
                               cudaStream_t s);
cudaError_t launch_momentum_step(float* w, float* accum, const float* g, size_t n, float lr, float momentum,
                                 float grad_scale, const float* norm_clip, cudaStream_t s);

// ---- network backward, bandwidth-class parts (bwd_kernels.cu)
// How the kernels that finish a gradient write it into the gradient arena (wgrad_reduce_kernel, bn_finalize_all_kernel,
// head_bias_final_kernel): arena = (accumulate ? arena : 0) + out_scale * finished value, the add after the fixed-order sum.
// A device word read at run time, so that one captured backward graph serves both training entries; nullptr = overwrite
// with out_scale 1.
struct GradMode {
  int accumulate;
  float out_scale;
};
#ifdef __CUDACC__
__device__ __forceinline__ void store_grad(float* dst, float v, const GradMode* mode) {
  if (mode != nullptr) {
    const GradMode m = *mode;
    v *= m.out_scale;
    if (m.accumulate) v = *dst + v;
  }
  *dst = v;
}
#endif
// One entry per 8 consecutive BatchNorm channels (always one layer): where their dy sums ([rows][C] floats, this group at column
// `col`) and their <W, dW_raw> products ([8][K4] floats) were left by the backward pass.
struct BnGroup {
  unsigned long long part_off = 0, rd_off = 0;
  int rows = 0, C = 0, col = 0, K4 = 0;
};
// dbeta[c] = sum of the dy sums, dgamma[c] = (sum of the row-dot products - mean * dbeta) / sqrt(var + eps), all channels at once
cudaError_t launch_bn_finalize_all(const BnGroup* table, int ngroups, const float* part, const float* rowdot, const float* mean,
                                   const float* var, float eps, float* dgamma, float* dbeta, const GradMode* mode, cudaStream_t s);
int relu_bn_bwd_blocks(int M, int C);  // rows of `partial` ([blocks][C])
// scatter_d != nullptr: g (N,H,W,C) += zero-inserted scatter_d (N,P,Q,C) first (gradient of the stride-2 identity shortcut)
cudaError_t launch_relu_bn_bwd(void* g, const void* act, int M, int C, float* partial, int fp16, cudaStream_t s,
                               const void* scatter_d = nullptr, int H = 0, int W = 0, int P = 0, int Q = 0);
// fused root of the backward: max-pool gradient + conv1 ReLU mask + dy sums ([maxpool_relu_bwd_rows][64] partial rows)
int maxpool_relu_bwd_rows(int N, int H, int W);
cudaError_t launch_maxpool_relu_bwd(const void* x, const void* gout, int N, int H, int W, int C, int Ho, int Wo, int pad_t,
                                    int pad_l, void* gx, float* partial, int fp16, cudaStream_t s);
cudaError_t launch_upsample2(const void* in, int N, int P, int Q, int C, void* out, int H, int W, cudaStream_t s);
cudaError_t launch_col2im_bwd(const float* g_logits, const float* g_locref, int N, int h, int w, int ctot, int nj,
                              void* dG, int Kd, int fp16, cudaStream_t s);
int head_bias_blocks();
// g (npix, C) fp32 -> dbias[C]; partial: [head_bias_blocks()][C] floats of workspace
cudaError_t launch_head_bias_grad(const float* g, size_t npix, int C, float* partial, float* dbias, const GradMode* mode,
                                  cudaStream_t s);

cudaError_t launch_scale_inplace(float* x, size_t n, float scale, cudaStream_t s);

// evaluate_dgp 'dgp' locref read-out: st (B,H,W,nj) blurred softmax, locref (B,H,W,2nj) raw -> pose (B,nj,3) = (x,y,1)
cudaError_t launch_soft_pose(const float* st, const float* locref, int B, int H, int W, int nj, float stride,
                             float locref_stdev, int swap_offsets, float* pose, cudaStream_t stream);

// ---- host-feeder replacements (feeder_kernels.cu)
// coord2map + scatter over the batch: joint_loc (n_vis,nj,2) double scoremap (row,col), NaN = missing; frame_idx (n_vis)
// position of each visible frame in the batch; lmap / lmask (nt,H,W,2nj) float32 are fully overwritten.
// learn_wt (fitdgp_util.py:454-467): |u| + |v| of OpenCV's dense Farneback flow (0.5, 3, 15, 3, 5, 1.2, 0) between consecutive
// BGR2GRAY-converted frames, all T-1 pairs per launch sequence (flow_kernels.cu).  out: float32 (T-1, H, W).
size_t learn_wt_workspace_bytes(int T, int H, int W);
cudaError_t launch_learn_wt(const uint8_t* frames, int T, int H, int W, float* out, void* workspace, int* launches, cudaStream_t s);
// gen_idx_chunk (dataset.py:187-239): sorted marker index vectors of a batch (visible_marker, hidden_marker,
// visible_marker_in_targets) + counts[2]; vis_frames sorted ascending (joint_loc rows follow that order), nt <= ~11 k frames
cudaError_t launch_marker_indices(const int* vis_frames, int n_vis, const int* hid_frames, int n_hid, const double* joint_loc, int nj,
                                  int nt, int* visible_marker, int* hidden_marker, int* visible_in_targets, int* counts,
                                  cudaStream_t s);
// sums[t] = sum over the bytes of (frames[t] - frames[t-1]) & 0xFF (sums[0] = 0): calculate_motion_energy, dataset.py:29-43
cudaError_t launch_motion_energy(const uint8_t* frames, int T, size_t frame_bytes, unsigned long long* sums, int num_sms,
                                 cudaStream_t s);
cudaError_t launch_locref_targets(const double* joint_loc, const int* frame_idx, int n_vis, int nt, int nj, int H, int W,
                                  double stride, double pos_dist_thresh, double locref_stdev, float* lmap, float* lmask,
                                  cudaStream_t s);

}  // namespace dgp
