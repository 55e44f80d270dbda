/*
 * dgp_b200.h -- C ABI of libdgp_b200.so: the B200-native (sm_100a) implementation of Deep Graph Pose's
 * per-frame scoremap-and-graph hot path.
 *
 * The reference (paninski-lab/deepgraphpose) has no FFI: its boundary is the TF1 graph-handle tuple returned by
 * `setup_dgp_eval_graph` / `dgp_loss` plus `sess.run(fetches, feed_dict)`.  Each entry point below names the
 * reference interface it replaces (paths relative to the reference root).  The Python shims in
 * `deepgraphpose_b200/` bind these with ctypes and re-create the reference call surface on top of them; see
 * INTEGRATION.md for the stub a reference maintainer would add.
 *
 * Conventions
 *  - All `*_dev` pointers are CUDA device pointers owned by the caller (PyTorch tensors in the shims);
 *    all tensors are dense, NHWC, (row, col) coordinate order, exactly as the reference's TF tensors.
 *  - `stream` is a `cudaStream_t` passed as `void*` (NULL = legacy default stream).  Calls are asynchronous on it.
 *  - Return value: DGP_OK (0) or a negative dgp_status; `dgp_last_error` gives the message.
 *  - There is NO CPU fallback and no alternate backend: a device that is not sm_100 is DGP_ERR_UNSUPPORTED.
 *  - A handle is bound to one device and is not thread-safe (one handle per GPU / rank).
 */
#ifndef DGP_B200_H_
#define DGP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum dgp_status {
  DGP_OK = 0,
  DGP_ERR_INVALID = -1,      /* bad argument / shape */
  DGP_ERR_CUDA = -2,         /* CUDA runtime or driver error */
  DGP_ERR_UNSUPPORTED = -3,  /* not an sm_100 device, or a configuration outside the path */
  DGP_ERR_STATE = -4,        /* call order (e.g. forward before finalize_weights) */
  DGP_ERR_NOMEM = -5
} dgp_status;

typedef struct dgp_handle dgp_handle;

/* Constants of PTF/default_config.py:16-59 and pose_cfg.yaml that parameterise the path. */
typedef struct dgp_config {
  int32_t num_joints;          /* cfg.num_joints */
  int32_t location_refinement; /* build the locref_pred head (pose_net.py:66-68) */
  int32_t device;              /* CUDA device ordinal */
  float stride;                /* default_config.py:18  (8.0) */
  float locref_stdev;          /* default_config.py:29  (7.2801) */
  float mean_pixel[3];         /* default_config.py:23  (123.68, 116.779, 103.939), RGB */
  float bn_epsilon;            /* slim resnet_arg_scope batch_norm_epsilon (1e-5) */
  int32_t precision;           /* 16-bit storage type of the activations / weights fed to the tensor cores (fp32 accumulate,
                                  fp32 BN epilogue, fp32 logits either way; same tcgen05 kind::f16 kernels, same speed):
                                  1 = fp16 -- what the Python shims and bench.py select: 11-bit mantissa, meets BASELINE.json's
                                      parity tolerances (sigmoid 1e-2, soft-argmax 0.5 px, loss 1e-3); values saturate at 65504;
                                  0 = bf16 -- fp32's exponent range, 8-bit mantissa: sigmoid scoremaps differ by up to ~4e-2 */
} dgp_config;

/* Replaces the graph construction in setup_dgp_eval_graph (src/deepgraphpose/models/eval.py:147-214) and in
 * dgp_loss (src/deepgraphpose/models/fitdgp.py:934-944): PoseNet(cfg) + prediction layers. */
int dgp_create(const dgp_config* cfg, dgp_handle** out);
void dgp_destroy(dgp_handle* h);
/* Message of the last failing call on `h` (or of the last failing dgp_create when h == NULL). */
const char* dgp_last_error(const dgp_handle* h);

/* Replaces TF.train.Saver.restore (eval.py:194-211, fitdgp.py:689-720): hand over one variable under its TF/slim
 * name and TF layout (conv HWIO [kh,kw,cin,cout]; deconv [kh,kw,cout,cin]; BN vectors [c]; biases [c]).
 * dtype: 0 = float32.  The data is copied; call dgp_finalize_weights once all variables are loaded. */
int dgp_load_weights(dgp_handle* h, const char* tf_var_name, const void* host_ptr, const int64_t* shape, int ndim,
                     int dtype);
/* Converts to kernel layouts (bf16 [cout][kh*kw*cin] K-major, fp32 BN scale/shift) and uploads.  The backbone is the one
 * the loaded names describe: every backbone variable must sit under exactly one of the slim scopes resnet_v1_50,
 * resnet_v1_101 or resnet_v1_152 (units per block (3,4,6,3), (3,4,23,3), (3,8,36,3)); mixed scopes or none at all are
 * DGP_ERR_INVALID. */
int dgp_finalize_weights(dgp_handle* h);
/* Depth of the backbone built by dgp_finalize_weights: 50, 101 or 152. */
int dgp_net_depth(const dgp_handle* h, int* depth);

/* slim's output_stride of the backbone (pose_cfg.yaml `output_stride`, pose_net.py:31-34): 8 or 16 (the default), set
 * before dgp_finalize_weights.  At 8, block 2 runs at stride 1, block 3 at rate 2 and block 4 at rate 4 (slim
 * stack_blocks_dense), so features and scoremaps have twice the resolution on each axis; pose_cfg's `stride` is then 4.0.
 * The weights are the same variables at either stride.  Other values are DGP_ERR_UNSUPPORTED; a call after
 * dgp_finalize_weights is DGP_ERR_STATE. */
int dgp_set_output_stride(dgp_handle* h, int output_stride);
int dgp_get_output_stride(const dgp_handle* h, int* output_stride);

/* Closed form of Dataset._compute_pred_dims (src/deepgraphpose/dataset.py:348-371) at output_stride 16. */
int dgp_output_dims(int H, int W, int* h_feat, int* w_feat, int* h_out, int* w_out);
/* The same at output_stride 8 or 16: h_feat = ceil(H / output_stride) by repeated SAME halving, h_out = 2 * h_feat. */
int dgp_output_dims_os(int H, int W, int output_stride, int* h_feat, int* w_feat, int* h_out, int* w_out);

/* Replaces sess.run([scmap(, locref)], {inputs: frames}) (eval.py:328, 746): PoseNet.extract_features
 * (pose_net.py:36-54: mean subtraction + slim resnet_v1_<depth> OS16, frozen BN) and the 3x3 stride-2 deconv heads
 * (pose_net.py:18-26).  frames_dev: uint8 (B,H,W,3) RGB.  logits_dev: float32 (B,2h,2w,nj) part_pred logits.
 * locref_dev: float32 (B,2h,2w,2nj) or NULL. */
int dgp_forward(dgp_handle* h, const uint8_t* frames_dev, int B, int H, int W, float* logits_dev, float* locref_dev,
                void* stream);

/* The two halves of dgp_forward under the reference's method names.
 * dgp_extract_features replaces PoseNet.extract_features (PTF/nnet/pose_net.py:36-54): net_dev float32 (B,hf,wf,2048) =
 * the block4 output `net` (hf, wf from dgp_output_dims).
 * dgp_prediction_layers replaces PoseNet.prediction_layers / prediction_layer (pose_net.py:18-26, 56-78) with the
 * handle's own pose/part_pred and pose/locref_pred variables: net_dev float32 (B,hf,wf,2048) -> logits_dev (B,2hf,2wf,nj)
 * and locref_dev (B,2hf,2wf,2nj) or NULL.  Both round `net` to the handle's 16-bit storage type exactly as dgp_forward
 * does, so extract_features followed by prediction_layers is bit-identical to dgp_forward.  Synchronous. */
int dgp_extract_features(dgp_handle* h, const uint8_t* frames_dev, int B, int H, int W, float* net_dev, void* stream);
int dgp_prediction_layers(dgp_handle* h, const float* net_dev, int B, int hf, int wf, float* logits_dev, float* locref_dev,
                          void* stream);
/* Replaces slim.conv2d_transpose(inputs, num_outputs, kernel_size=[3,3], stride=2, padding='SAME') + bias as built by
 * prediction_layer (pose_net.py:18-26) and dgp_prediction_layer (src/deepgraphpose/models/fitdgp_util.py:18-74, whose
 * init_flag hands the kernel in as constants): x_dev float32 (N,H,W,Cin), Cin a multiple of 64; w_host float32 in the TF
 * layout [3,3,Cout,Cin]; bias_host [Cout] or NULL; out_dev float32 (N,2H,2W,Cout).  One tcgen05 GEMM over the input
 * pixels + col2im (out[2i+k] += x[i] w[k], cropped to 2H x 2W).  Synchronous. */
int dgp_deconv2d(dgp_handle* h, const float* x_dev, int N, int H, int W, int Cin, const float* w_host, const float* bias_host,
                 int Cout, float* out_dev, void* stream);

/* Replaces argmax_2d_from_cm (src/deepgraphpose/models/fitdgp_util.py:342-402) fused with the per-frame read-outs
 * that consume it: estimate_pose's windowed peak + likelihood (eval.py:331-343) and DLC's global-argmax pose
 * (PTF/nnet/predict.py:62-77, pose_net.py:92-163).  Any output pointer may be NULL.
 *  mu_dev       float32 (B,nj,2)  soft-argmax (row, col) in scoremap pixels
 *  peak_dev     int32   (B,nj,2)  estimate_pose `mu_likelihoods` (row, col)
 *  lik_dev      float32 (B,nj)    estimate_pose `likelihoods`
 *  dlc_peak_dev int32   (B,nj,2)  argmax_pose_predict integer peak (row, col)
 *  dlc_pose_dev float32 (B,nj,3)  argmax_pose_predict (x, y, likelihood), locref offset applied iff locref_dev */
int dgp_softargmax(dgp_handle* h, const float* logits_dev, const float* locref_dev, int B, int H, int W, int nj,
                   float gamma, float gauss_len, float* mu_dev, int32_t* peak_dev, float* lik_dev,
                   int32_t* dlc_peak_dev, float* dlc_pose_dev, void* stream);

/* Second return value of argmax_2d_from_cm (fitdgp_util.py:391, consumed by evaluate_dgp eval.py:752): the
 * Gaussian-blurred, renormalised spatial softmax, float32 (B,H,W,nj). */
int dgp_softmax_map(dgp_handle* h, const float* logits_dev, int B, int H, int W, int nj, float gamma, float gauss_len,
                    float* map_dev, void* stream);

/* The `th` branch of argmax_2d_from_cm (fitdgp_util.py:379-399; no reference caller passes it): on the map written by
 * dgp_softmax_map, zero every entry below th * (the joint's maximum), renormalise, and return the soft-argmax of the
 * thresholded map.  map_dev float32 (B,H,W,nj) is rewritten in place; mu_dev float32 (B,nj,2) (row, col) or NULL. */
int dgp_softmax_threshold(dgp_handle* h, float* map_dev, int B, int H, int W, int nj, float th, float* mu_dev, void* stream);

/* Replaces evaluate_dgp's 'dgp' locref read-out (src/deepgraphpose/models/eval.py:751-785): blurred spatial softmax of the
 * logits, then pose = (sum st * (row, col) * stride + stride/2 + sum st * locref * locref_stdev)[::-1] -> float32 (B,nj,3) =
 * (x, y, 1).  swap_offsets = 0 reproduces the reference (locref's first component is added to the row coordinate),
 * 1 applies the offsets as DLC's argmax_pose_predict does.  map_ws_dev: float32 (B,H,W,nj) workspace (receives the map). */
int dgp_soft_pose(dgp_handle* h, const float* logits_dev, const float* locref_dev, int B, int H, int W, int nj, float gamma,
                  float gauss_len, int swap_offsets, float* map_ws_dev, float* pose_dev, void* stream);

/* Replaces the host feeder coord2map (src/deepgraphpose/dataset.py:246-271 -> PoseDataset.compute_target_part_scoremap,
 * PTF/dataset/pose_defaultdataset.py:220-266) and the scatter of its output over the batch (fitdgp.py:781-795): the
 * `locref_map` / `locref_mask` feeds are generated on the device.  joint_loc_dev: float64 (n_vis,nj,2) labels in scoremap
 * (row, col) units, NaN = missing; frame_idx_dev: int32 (n_vis) = visible_frame_within_batch; outputs float32
 * (nt,H,W,2nj), fully overwritten; locref_stdev as a double (0 = the handle's float config value).  Bit-identical to the
 * reference's float64 arrays cast to the float32 placeholders. */
int dgp_locref_targets(dgp_handle* h, const double* joint_loc_dev, const int32_t* frame_idx_dev, int n_vis, int nt, int H,
                       int W, double pos_dist_thresh, double locref_stdev, float* locref_map_dev, float* locref_mask_dev,
                       void* stream);

/* Replaces gen_idx_chunk / find_marker_index (src/deepgraphpose/dataset.py:157-239), the marker bookkeeping of every training
 * batch: marker id = frame_position * nj + joint; visible_frames_dev (ascending; joint_loc_dev float64 (n_vis,nj,2) rows in that
 * order, NaN = unlabelled) and hidden_frames_dev are positions within the nt-frame batch.  Outputs (capacity nt * nj each),
 * sorted ascending as the reference's np.sort / np.setdiff1d produce them: visible_marker, hidden_marker (hidden frames' markers
 * + the NaN-labelled markers of visible frames), visible_marker_in_targets (row * nj + joint of each visible marker in the
 * targets array); counts_dev[0..1] = their lengths.  Integer work, bit-exact. */
int dgp_marker_indices(dgp_handle* h, const int32_t* visible_frames_dev, int n_vis, const int32_t* hidden_frames_dev, int n_hid,
                       const double* joint_loc_dev, int nt, int32_t* visible_marker_dev, int32_t* hidden_marker_dev,
                       int32_t* visible_in_targets_dev, int32_t* counts_dev, void* stream);

/* Replaces learn_wt (src/deepgraphpose/models/fitdgp_util.py:454-467), the host feeder of the temporal clique's
 * `vector_field_tf`: for every consecutive pair of the T frames (uint8 (T,H,W,3) on the device, as fed to the network),
 * cv2.cvtColor(BGR2GRAY) -> cv2.calcOpticalFlowFarneback(prev, next, None, 0.5, 3, 15, 3, 5, 1.2, 0) -> |u| + |v|.
 * field_dev: float32 (T-1, H, W).  OpenCV is an un-vendored dependency of the reference; the algorithm is restated from the
 * published method / OpenCV 4.x semantics and agrees with cv2 4.13 to ~1e-5 px (tests/test_flow.py). */
int dgp_learn_wt(dgp_handle* h, const uint8_t* frames_dev, int T, int H, int W, float* field_dev, void* stream);

/* Replaces the per-frame arithmetic of calculate_motion_energy (src/deepgraphpose/dataset.py:29-43), the score that ranks
 * hidden frames for training: motion_energy[t] = np.mean(np.abs(frame[t] - frame[t-1])) on uint8 frames, i.e. the mean of the
 * byte differences MODULO 256 (uint8 subtraction wraps, abs is the identity).  frames_dev: uint8 (T, frame_bytes), T consecutive
 * frames; sums_dev: uint64 (T) <- exact byte sums (sums[0] = 0 -- pass the last frame of the previous chunk first to continue a
 * video).  The caller divides by frame_bytes in double: bit-identical to the reference's float64 mean. */
int dgp_motion_energy(dgp_handle* h, const uint8_t* frames_dev, int T, size_t frame_bytes, uint64_t* sums_dev, void* stream);

/* Replaces PoseNet.test's tf.sigmoid(part_pred) (pose_net.py:84-90). n = number of floats (multiple of 4). */
int dgp_sigmoid(dgp_handle* h, const float* logits_dev, float* prob_dev, size_t n, void* stream);

/* Replaces the clique distance terms of dgp_loss: skeleton d[l,t] = ||S (mu_t*stride + stride/2)||_2
 * (fitdgp.py:1063-1069) and temporal delta[t,j] = ||mu_t - mu_{t+1}||_2 * stride (fitdgp.py:1079-1083).
 *  mu_dev (T,nj,2); mu_halo_next_dev (nj,2) = first frame of the next shard or NULL (then row T-1 of temporal is
 *  not written); edges_dev int32 (nl,2) = (+1 joint, -1 joint) rows of S0 (fitdgp.py:607-617);
 *  ws_dev / ws_max_dev (nl) or NULL; skel_dist_dev (nl,T); temporal_dev (T,nj);
 *  e_skel_dev (T) = sum_l ws_l * max(d, ws_max_l); e_temp_dev (T) = sum_j max(delta, wt_max)^2.  Outputs may be NULL. */
int dgp_potentials(dgp_handle* h, const float* mu_dev, const float* mu_halo_next_dev, int T, int nj,
                   const int32_t* edges_dev, int nl, const float* ws_dev, const float* ws_max_dev, float wt_max,
                   float* skel_dist_dev, float* temporal_dev, float* e_skel_dev, float* e_temp_dev, void* stream);

/* Hyper-parameters fit_dgp writes onto dlc_cfg (fitdgp.py:637-654) plus the demo's gm2/gm3 flags. */
typedef struct dgp_loss_cfg {
  float gamma, gauss_len, lengthscale;       /* 1, 1, 1 */
  float wt, wt_max;                          /* temporal clique (0 = off), upper bound */
  float wn_visible, wn_hidden;               /* 5, 3 */
  float locref_loss_weight;                  /* 0.05 */
  float n_frames_total, n_visible_frames_total;
  int32_t gm2, gm3;                          /* {0,1,2}, {0,3} */
  int32_t locref_mse;                        /* 0 = losses.huber_loss (dlc_cfg.locref_huber_loss True, the DLC default),
                                                1 = tf.losses.mean_squared_error (fitdgp.py:1053) */
} dgp_loss_cfg;

/* The feeds of dgp_loss's placeholders (fitdgp.py:1130-1142), as device pointers.  Index vectors are int32. */
typedef struct dgp_loss_batch {
  const float* pred_dev;        /* (nt,H,W,nj) part_pred logits (output of dgp_forward) */
  const float* locref_dev;      /* (nt,H,W,2nj) locref_pred, or NULL to skip the locref term */
  int32_t nt, H, W;
  const float* targets_dev;     /* (nv,nj,2) labels in scoremap (row, col) units, NaN = missing */
  int32_t nv;
  const float* locref_map_dev;  /* (nt,H,W,2nj) */
  const float* locref_mask_dev; /* (nt,H,W,2nj) */
  const int32_t* visible_marker_dev; int32_t nbv;
  const int32_t* hidden_marker_dev;  int32_t nbh;
  const int32_t* visible_marker_in_targets_dev;
  const int32_t* edges_dev; int32_t nl;   /* skeleton: rows of S0 as (+1 joint, -1 joint) */
  const float* ws_dev; const float* ws_max_dev;  /* (nl) from the host precompute fitdgp.py:874-892 */
  const float* vector_field_dev; int32_t Hin, Win;  /* (nt-1,Hin,Win) optical-flow magnitude, or NULL */
  const float* wt_batch_dev;    /* (nt-1) = wt_batch_pl * wt_batch_mask_pl */
  void* vector_field_ready_event; /* optional cudaEvent_t recorded behind the producer of vector_field_dev (dgp_learn_wt on
                                     another stream): the loss waits for it on its own stream, so the Farneback flow of the
                                     batch overlaps the forward pass of dgp_train_forward_backward.  NULL: already ordered. */
} dgp_loss_batch;

/* Replaces the loss part of sess.run([loss, ...]) in fit_dgp (fitdgp.py:817-818, graph :947-1128): soft-argmax of
 * the hidden markers, visible/hidden marker scatter, Gaussian-target sigmoid cross-entropies with the gm2/gm3
 * confidence scaling, locref Huber, skeleton (spatial) and temporal cliques (forward).
 * losses_dev[6] = {visible_loss_pred, hidden_loss_pred, visible_loss_locref, ws_loss, wt_loss, total_loss};
 * targets_all_dev (nt*nj,2) optionally receives targets_all_marker. */
int dgp_loss_forward(dgp_handle* h, const dgp_loss_cfg* cfg, const dgp_loss_batch* batch, float* losses_dev,
                     float* targets_all_dev, void* stream);

/* Forward + the loss-side half of the backward pass of fit_dgp's train_op (fitdgp.py:706-713 differentiates total_loss;
 * fit_dgp_labeledonly differentiates total_loss_visible, fitdgp.py:416 -> visible_only = 1): gradients of the loss
 * w.r.t. the head outputs, float32 (nt,H,W,nj) and (nt,H,W,2nj) (grad_locref_dev may be NULL).  They flow through the
 * cross-entropy labels (Gaussian targets -> soft-argmax), the confidence max and the (1 - c) weights exactly as in the
 * TF graph, including the temporal clique's path through tf.image.crop_and_resize's box gradient (wt > 0).  The network
 * backward and the Momentum step are dgp_train_forward_backward / dgp_optimizer_step below. */
int dgp_loss_backward(dgp_handle* h, const dgp_loss_cfg* cfg, const dgp_loss_batch* batch, float* losses_dev,
                      float* grad_pred_dev, float* grad_locref_dev, int visible_only, void* stream);

/* ---- frame resize + crop (estimate_pose's new_size / crop_size, eval.py:309-326) ----
 * The reference resizes each frame with PIL's Image.resize((resize_w, resize_h)) -- Pillow's default filter for RGB images,
 * BICUBIC (a = -0.5) since Pillow 7.0 -- and then crops it with Image.crop((crop_x0, crop_y0, crop_x1, crop_y1)).  The
 * entries below compute the same bytes on the device: Pillow's 8-bit resample is integer arithmetic on fixed-point weights
 * (22 fraction bits) computed in double, horizontal pass first, a pass skipped when its size does not change, and the
 * crop taken on the resized frame with box pixels outside that frame set to 0.
 *  resize_h = resize_w = 0: no resize (else both > 0).  All four crop fields 0: no crop (else crop_x1 > crop_x0 and
 *  crop_y1 > crop_y0; the box may extend past the resized frame).  Anything else is DGP_ERR_INVALID and launches nothing. */
typedef struct dgp_frame_transform {
  int32_t resize_h, resize_w;
  int32_t crop_x0, crop_y0, crop_x1, crop_y1;
} dgp_frame_transform;
/* Size (H, W) of a transformed H0 x W0 frame; `t` NULL = identity.  Handle-free, like dgp_output_dims. */
int dgp_transform_dims(int H0, int W0, const dgp_frame_transform* t, int* H, int* W);
/* Pillow's resample table for one axis, in_size -> out_size (handle-free; what the device passes use): output index i reads
 * count[i] inputs from first[i] with int32 weights[i * max_taps + k] (weights past count[i] are 0).  ceil(2 * max(in_size /
 * out_size, 1)) * 2 + 1 taps always suffice; a max_taps below some count[i] is DGP_ERR_INVALID. */
int dgp_resize_coefficients(int in_size, int out_size, int max_taps, int32_t* first, int32_t* count, int32_t* weights);
/* src_dev uint8 (N,H0,W0,3) RGB -> dst_dev uint8 (N,H,W,3), (H, W) from dgp_transform_dims.  Asynchronous on `stream`.
 * The size tables are built on the host at the first use of a size pair and kept on the handle. */
int dgp_resize_crop(dgp_handle* h, const uint8_t* src_dev, int N, int H0, int W0, const dgp_frame_transform* t,
                    uint8_t* dst_dev, void* stream);

/* ---- augmentation of labelled training frames (fit_dgp's data_aug, fitdgp.py:773-779; pipeline of build_aug,
 * fitdgp_util.py:412-451) ----
 * Per frame, in this order, each op switched on by its parameters:
 *  1. rotation by rotate_deg (0 = off) about the frame centre: forward matrix, in double, with t = rotate_deg * (pi / 180),
 *     c = cos t, s = sin t, cx = W / 2 - 0.5, cy = H / 2 - 0.5:  M = [[c, -s, cx - c cx + s cy], [s, c, cy - s cx - c cy]].
 *     Pixels: bit-exact to cv2.warpAffine(img, M, (W, H), INTER_LINEAR, BORDER_CONSTANT, 0) -- OpenCV's fixed-point path
 *     (M inverted in double; X0 = rint((M1 y + M2) 1024) + 16 per row, X = (X0 + rint(M0 x 1024)) >> 5 per column; 5
 *     fraction bits select 2x2 int16 weights summing to 2^15; (sum w p + 2^14) >> 15, saturated; taps outside read 0).
 *  2. motion blur with the k x k table of dgp_motion_blur_kernel(blur_k, blur_angle_deg, blur_direction) (blur_k 0 = off,
 *     else odd in [3, 15]): (sum w p + 2^13) >> 14 per channel, saturated, correlation with a reflect-101 border.
 *  3. coarse dropout (drop_p = 0 or drop_size_percent = 0: off): grid gh = max(1, rint(H sp)), gw = max(1, rint(W sp)),
 *     sp = drop_size_percent; cell (i, j) is dropped when u01(seed, 2, i, j) < drop_p; pixel (y, x) lies in cell
 *     (min(floor(y * (1 / (H / gh))), gh - 1), min(floor(x * (1 / (W / gw))), gw - 1)), in double -- the indexing of
 *     cv2.resize(mask, (W, H), INTER_NEAREST); the pixels of dropped cells become 0 in all channels.
 *  4. elastic deformation (elastic_alpha 0 = off) with the fields of dgp_elastic_field(alpha, sigma, seed):
 *     out(x, y) = in(x + dx, y + dy), bit-exact to cv2.remap(img, x + dx, y + dy, INTER_LINEAR, BORDER_CONSTANT, 0) fed
 *     the same float32 maps (map = float32(x) + dx in float32; X = rint(map * 32); the weights of rotation).
 * Counter hash (splitmix64) of (seed, plane, row, col):
 *     c = plane << 48 | row << 24 | col;  z = seed + (c + 1) * 0x9E3779B97F4A7C15;
 *     z = (z ^ z >> 30) * 0xBF58476D1CE4E5B9;  z = (z ^ z >> 27) * 0x94D049BB133111EB;  z ^= z >> 31;  b = z >> 40
 *   (all mod 2^64); noise(seed, plane, row, col) = (b + 0.5) / 2^23 - 1 (float32, exact), u01 = (b + 0.5) / 2^24 (double). */
typedef struct dgp_augment_params {
  double rotate_deg;
  int32_t blur_k;
  double blur_angle_deg;
  double blur_direction;     /* in [-1, 1] */
  double drop_p;             /* in [0, 1] */
  double drop_size_percent;  /* in [0, 1] */
  double elastic_alpha;
  double elastic_sigma;      /* in (0, 16] when elastic_alpha != 0 */
  uint64_t seed;             /* of the dropout cells and the elastic noise */
} dgp_augment_params;
/* The motion-blur table (handle-free): a k x k float64 image whose middle column is numpy.linspace(d, 1 - d, k),
 * d = (direction + 1) / 2, rotated by angle_deg about its centre c = (k - 1) / 2 with bilinear sampling (constant 0 outside):
 * out(i, j) = img at (x, y) = (ca u + sa v + c, -sa u + ca v + c), u = j - c, v = i - c, ca = cos, sa = sin of
 * angle_deg * (pi / 180); divided by its sum (row-major, sequential); w = rint(out * 2^14) and 2^14 - sum(w) added to the
 * first largest weight, so the k * k int32 weights (row-major) sum to exactly 2^14.  k odd in [3, 15]. */
int dgp_motion_blur_kernel(int k, double angle_deg, double direction, int32_t* weights);
/* Elastic displacement fields of one H x W frame into float32 dx_dev, dy_dev (H, W): the noise planes 0 (dx) and 1 (dy) of
 * `seed` are smoothed by a separable float32 Gaussian of radius R = ceil(4 sigma) (weights exp(-k^2 / (2 sigma^2)) divided
 * by their sum in double, reflect-101 border, rows then columns) and multiplied by alpha.  sigma in (0, 16]. */
int dgp_elastic_field(dgp_handle* h, int H, int W, double alpha, double sigma, uint64_t seed, float* dx_dev, float* dy_dev,
                      void* stream);
/* Augments frames_dev uint8 (nt, H, W, 3) in place: frame frame_idx_host[k] (k < n, distinct, in [0, nt)) with
 * params_host[k]; other frames are not touched.  joint_loc_dev (NULL = no labels): float64 (n, nj) (row, col) scoremap
 * labels of those frames, moved in place -- to pixels x = col stride + stride / 2, by M under rotation, under elastic by the
 * inverse of the backward map (p <- q - d(p) from p = q, 20 iterations, d bilinear in the frame's float32 fields with
 * coordinates clamped to the frame), and back; NaN labels stay NaN, labels leaving the frame are kept.  Blur and dropout
 * leave labels alone.  Asynchronous on `stream`: per-frame matrices and tables travel as kernel arguments; a pass no frame
 * needs is not launched.  Invalid arguments return DGP_ERR_INVALID before anything is launched. */
int dgp_augment(dgp_handle* h, uint8_t* frames_dev, int nt, int H, int W, const int32_t* frame_idx_host, int n,
                const dgp_augment_params* params_host, double* joint_loc_dev, double stride, void* stream);

/* Replaces the estimate_pose frame loop (eval.py:306-345) end to end with HOST buffers: per batch of `batch`
 * frames H2D copy, dgp_forward, dgp_softargmax, D2H of the results.  frames_host uint8 (T,H,W,3) (pinned memory
 * gives asynchronous copies); mu_host float32 (T,nj,2); peak_host int32 (T,nj,2); lik_host float32 (T,nj). */
int dgp_estimate_pose_host(dgp_handle* h, const uint8_t* frames_host, int T, int H, int W, int batch, float gamma,
                           float gauss_len, float* mu_host, int32_t* peak_host, float* lik_host);
/* dgp_estimate_pose_host on frames that `transform` resizes / crops on the device first (NULL = identity, which is
 * dgp_estimate_pose_host): frames_host holds (T,H0,W0,3) source frames, the H2D copy carries them at that size, and
 * dgp_resize_crop turns each batch into the (H,W) frames of dgp_transform_dims on the compute stream. */
int dgp_estimate_pose_host_transform(dgp_handle* h, const uint8_t* frames_host, int T, int H0, int W0,
                                     const dgp_frame_transform* transform, int batch, float gamma, float gauss_len,
                                     float* mu_host, int32_t* peak_host, float* lik_host);

/* Streaming form of the estimate_pose frame loop (eval.py:256, 306-345: `for frame in clip.iter_frames()`), for videos that
 * do not fit in host memory.  A reader thread owned by the call asks `reader` for up to `max_frames` frames at a time and
 * stages them in a ring of 3 pinned host slots of `batch` frames; the calling thread copies filled slots to the device and
 * runs dgp_forward + dgp_softargmax on them, so decode, H2D and compute overlap and host memory is bounded by the ring.
 *  reader(user, slot, max_frames, &direct): write n <= max_frames uint8 (H,W,3) RGB frames into `slot` (pinned) and return n,
 *    or leave `slot` alone, point *direct at n frames the source already holds in (ideally pinned) host memory, and return n;
 *    return 0 at the end of the video, < 0 on error.  It is called from the reader thread, never concurrently.
 *  max_frames: capacity of the output arrays (frames beyond it are not read); *frames_done receives the number processed.
 *  Outputs as in dgp_estimate_pose_host.  Synchronous: returns when every result is in the host arrays. */
typedef int (*dgp_frame_reader)(void* user, uint8_t* slot, int max_frames, const uint8_t** direct);
int dgp_estimate_pose_stream(dgp_handle* h, dgp_frame_reader reader, void* user, int H, int W, int batch, float gamma,
                             float gauss_len, int64_t max_frames, float* mu_host, int32_t* peak_host, float* lik_host,
                             int64_t* frames_done);
/* dgp_estimate_pose_stream on (H0,W0,3) source frames that `transform` resizes / crops on the device (NULL = identity):
 * the reader delivers source-size frames, the pinned ring and the H2D copy carry them, and dgp_resize_crop runs on the
 * compute stream into the device buffer that dgp_forward consumes. */
int dgp_estimate_pose_stream_transform(dgp_handle* h, dgp_frame_reader reader, void* user, int H0, int W0,
                                       const dgp_frame_transform* transform, int batch, float gamma, float gauss_len,
                                       int64_t max_frames, float* mu_host, int32_t* peak_host, float* lik_host,
                                       int64_t* frames_done);
/* A ready-made reader for frames already resident in (pinned) host memory, e.g. a decoded clip kept in RAM or bench.py's
 * synthetic video: serves `total_frames` frames by cycling over pool[0 .. pool_frames) in direct (zero-copy) mode. */
typedef struct dgp_cyclic_source {
  const uint8_t* pool;     /* pool_frames frames of frame_bytes each */
  int64_t pool_frames;
  int64_t total_frames;    /* length of the video to serve */
  int64_t position;        /* next frame to serve (start at 0) */
  size_t frame_bytes;      /* H * W * 3 */
} dgp_cyclic_source;
int dgp_cyclic_reader(void* user, uint8_t* slot, int max_frames, const uint8_t** direct);

/* ---- labelled video (plot_dgp / create_annotated_movie, src/deepgraphpose/models/eval.py) ----
 * Markers drawn into uint8 (N,H,W,3) RGB frames.  For frame t and joint j with video-pixel coordinates x, y (float64) and
 * likelihood lik: the joint is drawn iff (double)lik > mask_threshold (strictly; NaN in x, y or lik: not drawn); centre
 * xc = min(trunc(x), W - 1), yc = min(trunc(y), H - 1) in double (truncation toward zero, negative centres kept, +inf
 * clamps to the last row / column); the disc is every pixel (r, c) of the frame with (r - yc)^2 + (c - xc)^2 < dotsize^2 in
 * integers, painted colors[j].  Joints are drawn in index order (where discs overlap the higher index wins); pixels outside
 * every disc keep their bytes.  dotsize in [0, 64] (0 draws nothing).
 * Skeleton and trails (zero-initialised fields draw neither).  Frame t is painted in this order:
 *  1. trails, when trailpoints = K >= 2: for k = K-1 down to 1, and within each k for j = 0..nj-1, the disc of joint j of
 *     frame t-k by the rule above (dotsize, colors[j], the mask of frame t-k's own lik); frames t-k < 0 are skipped.  Frame
 *     indices count from the first frame of the call (in dgp_draw_markers, from its first history row).  K in [0, 64].
 *  2. skeleton: for each edge (a, b) in the order given, a line in skeleton_color, drawn iff both joints of frame t pass the
 *     mask, their x and y are finite and both centres (xc, yc above) are >= -2^20.  With dr = yc_b - yc_a, dc = xc_b - xc_a,
 *     n = max(|dr|, |dc|), the line is the pixels k = 0..n with r = yc_a + floor((2 k dr + n) / 2n),
 *     c = xc_a + floor((2 k dc + n) / 2n) (integer floor division; n = 0 is one pixel), those inside the frame written.  At
 *     most 256 edges, joints in [0, nj); frames with an edge are at most 2^30 pixels high and wide.
 *  3. the discs of frame t, as without an overlay, so that they stay on top.
 * With no edges and K <= 1 the bytes are those of the markers alone. */
typedef struct dgp_marker_style {
  int32_t dotsize;
  double mask_threshold;
  double scale_x, scale_y;  /* fused pass only: soft-argmax coordinates -> video pixels (W0 / new_w, H0 / new_h, else 1) */
  const uint8_t* colors;    /* host (nj,3) RGB, nj = the handle's num_joints */
  const int32_t* edges;     /* host (n_edges,2) joint index pairs of the skeleton */
  int32_t n_edges;
  uint8_t skeleton_color[3];
  int32_t trailpoints;      /* K: frames of a joint's trail, the current one included (0 or 1: no trail) */
  int32_t history;          /* dgp_draw_markers only: rows before frames_dev[0] in x_dev / y_dev / lik_dev, <= K - 1 */
} dgp_marker_style;
/* Draws the markers of x_dev, y_dev, lik_dev (float64 (history + N, nj) on the device; row history + t is frame t of
 * frames_dev, the first `history` rows are the frames before it) into frames_dev (N,H,W,3) in place; `scale_x` and
 * `scale_y` are not used (the coordinates are video pixels already).  Asynchronous on `stream`; the colour and edge tables
 * travel as kernel arguments.  The render-only entry, for labels that already exist (a DLC csv). */
int dgp_draw_markers(dgp_handle* h, uint8_t* frames_dev, int N, int H, int W, const double* x_dev, const double* y_dev,
                     const double* lik_dev, const dgp_marker_style* style, void* stream);
/* writer(user, frames, n): n uint8 (H0,W0,3) RGB annotated frames, valid only during the call; return < 0 to abort.  Called
 * from a thread owned by the call, never concurrently, with frames in video order. */
typedef int (*dgp_frame_writer)(void* user, const uint8_t* frames, int n);
/* dgp_estimate_pose_stream_transform that also renders the labelled video in the same pass: per batch, after the
 * soft-argmax, the markers of x = ((double)mu[..,1] * stride + 0.5 * stride) * scale_x, y likewise with mu[..,0] and
 * scale_y, and lik are drawn into the batch's (H0,W0) source frames on the device (stride = the handle's, as a double),
 * the n real frames are copied into a ring of 3 pinned writer slots and handed to `writer` on a writer thread.  Trails
 * reach back across batches to the first frame of the call, so the frames do not depend on `batch`.  Read-outs as in
 * dgp_estimate_pose_stream_transform.  A failing writer aborts the call like a failing reader (DGP_ERR_INVALID). */
int dgp_estimate_pose_stream_render(dgp_handle* h, dgp_frame_reader reader, void* user, int H0, int W0,
                                    const dgp_frame_transform* transform, int batch, float gamma, float gauss_len,
                                    int64_t max_frames, float* mu_host, int32_t* peak_host, float* lik_host,
                                    int64_t* frames_done, const dgp_marker_style* style, dgp_frame_writer writer,
                                    void* writer_user);

/* ---- Motion-JPEG of the labelled video ----
 * Each uint8 (H,W,3) RGB frame becomes exactly the bytes of Pillow's (libjpeg-turbo's)
 *   Image.fromarray(frame).save(buf, format="JPEG", quality=quality, subsampling=2, restart_marker_rows=1)
 * for 1 <= H, W <= 16383 and quality 1..100: baseline JPEG, JFIF 1.01 APP0, the Annex K quantisation tables scaled by
 * libjpeg's quality rule, 4:2:0 (Y 2x2, Cb / Cr 1x1), the Annex K Huffman tables, one restart interval per MCU row (RST0..7
 * between rows).  The contract, down to the fixed-point colour conversion and the islow DCT, is in DESIGN.md §4.5. */
/* Bytes one frame's file can take at most (the header, 64 x (16 + 11) bits per 8x8 block doubled for 0xFF stuffing, the
 * markers); -1 for a size outside 1..16383. */
int64_t dgp_jpeg_capacity(int H, int W);
/* Encodes N frames of frames_dev (device (N,H,W,3)) into out_dev (device, `capacity` >= N * dgp_jpeg_capacity(H, W) bytes):
 * the files are packed in frame order, frame i at out_dev + offsets_dev[i] with sizes_dev[i] bytes (device int64 (N)).  A
 * frame's bytes do not depend on N or on its position.  A frame that would exceed its bound (never, for valid input) gets
 * size -1 and is not written.  Asynchronous on `stream`; scratch and the (H, W, quality) header template are kept on the
 * handle, so calls on one handle are ordered on one stream. */
int dgp_encode_jpeg(dgp_handle* h, const uint8_t* frames_dev, int N, int H, int W, int quality, uint8_t* out_dev,
                    int64_t capacity, int64_t* offsets_dev, int64_t* sizes_dev, void* stream);
/* writer(user, data, sizes, n): the JPEG files of n frames, packed back to back in video order at `data` (frame i has
 * sizes[i] bytes), valid only during the call; return < 0 to abort.  Called from a thread owned by the call, never
 * concurrently. */
typedef int (*dgp_packet_writer)(void* user, const uint8_t* data, const int64_t* sizes, int n);
/* dgp_estimate_pose_stream_render whose annotated frames are encoded on the device (dgp_encode_jpeg at `quality`) right
 * after the markers are drawn: only the encoded bytes cross to the host, into a ring of 3 pinned writer slots that a writer
 * thread hands to `writer`.  Read-outs, markers and failure handling as in dgp_estimate_pose_stream_render. */
int dgp_estimate_pose_stream_render_jpeg(dgp_handle* h, dgp_frame_reader reader, void* user, int H0, int W0,
                                         const dgp_frame_transform* transform, int batch, float gamma, float gauss_len,
                                         int64_t max_frames, float* mu_host, int32_t* peak_host, float* lik_host,
                                         int64_t* frames_done, const dgp_marker_style* style, int quality,
                                         dgp_packet_writer writer, void* writer_user);

/* ---- training step (fit_dgp, src/deepgraphpose/models/fitdgp.py:706-713 and :817-818) ----
 * Replaces sess.run([train_op, loss], feed_dict): dgp_train_forward_backward computes the loss and the gradients of
 * total_loss (visible_only = 1: total_loss_visible, fit_dgp_labeledonly fitdgp.py:416) w.r.t. every trainable variable
 * (conv weights, BatchNorm gamma/beta with frozen moving statistics, deconv weights + biases); dgp_optimizer_step applies
 * tf.clip_by_global_norm(clip_norm) + MomentumOptimizer(lr, momentum).  Between the two calls a data-parallel caller
 * all-reduces (sums) the flat gradient buffer of dgp_get_grad_buffer with NCCL and passes grad_scale = 1 / world_size
 * (the tower averaging of src/deepgraphpose/helpers/utils_tf.py:4-39).
 * From its second run at a given input shape the network backward (about 280 launches with fixed arguments) is replayed as
 * one CUDA graph; it is launched kernel by kernel while dgp_set_profiling is on. */
/* Allocates gradients, momentum accumulators and the transposed (dgrad) weight operands. Call after finalize. */
int dgp_train_enable(dgp_handle* h);
/* frames_dev uint8 (nt,H,W,3); batch->pred_dev / locref_dev are ignored (the handle's own head outputs are used), all other
 * members as in dgp_loss_forward.  losses_dev[6] as in dgp_loss_forward. */
int dgp_train_forward_backward(dgp_handle* h, const uint8_t* frames_dev, int nt, int H, int W, const dgp_loss_cfg* cfg,
                               const dgp_loss_batch* batch, int visible_only, float* losses_dev, void* stream);
/* The same step split in two, for a loss (and optimizer) written by the caller:
 *  dgp_train_forward: the training forward of frames_dev uint8 (nt,H,W,3), keeping every activation.  The head outputs go to
 *    logits_dev float32 (nt,2h,2w,nj) and locref_dev (nt,2h,2w,2nj); locref_dev may be NULL.  *token names this forward.
 *    At most one forward per input shape is live: the next training forward at that shape (either entry), the eviction of
 *    the shape's plan (more than 3 training shapes) or a weight change (dgp_set_variable, dgp_optimizer_step,
 *    dgp_params_changed) makes the token stale.
 *  dgp_train_backward: the network backward of that forward from the caller's loss gradients w.r.t. the head outputs
 *    (float32, shapes as above; NULL = zeros).  They are loss-scaled like the fused step's, and the finished gradients are
 *    divided by the loss scale again as they are stored, so the gradient buffer holds the TRUE gradient.  accumulate = 0
 *    overwrites the buffer, 1 adds to it (the add comes after every fixed-order sum: batch A then B == gA + gB in fp32, bit
 *    for bit); adding onto the loss-scaled buffer of dgp_train_forward_backward is DGP_ERR_STATE.  A stale token is
 *    DGP_ERR_STATE and launches nothing.  The same token may be differentiated more than once.
 * Readers of the gradient buffer (dgp_optimizer_step, dgp_get_variable(what = 1), dgp_get_grad_norm) divide by the scale
 * the buffer holds: loss_scale after dgp_train_forward_backward, 1 after dgp_train_backward. */
int dgp_train_forward(dgp_handle* h, const uint8_t* frames_dev, int nt, int H, int W, float* logits_dev, float* locref_dev,
                      uint64_t* token, void* stream);
int dgp_train_backward(dgp_handle* h, uint64_t token, const float* g_logits_dev, const float* g_locref_dev, int accumulate,
                       void* stream);
/* g' = g * grad_scale; g' *= clip_norm / max(||g'||, clip_norm) (clip_norm <= 0: no clipping);
 * accum = momentum * accum + g'; var -= lr * accum; then refreshes the 16-bit operands and BN scale/shift. */
int dgp_optimizer_step(dgp_handle* h, float lr, float momentum, float clip_norm, float grad_scale, void* stream);
/* Flat float32 parameter arena (fp32 master copy, kernel layouts: [weights | gamma | beta | head bias], the layout of the
 * gradient buffer) for an optimizer outside the library.  After changing it in place, call dgp_params_changed: it re-derives
 * the 16-bit weights, the BatchNorm scale / shift and the dgrad operands on `stream` (what dgp_optimizer_step does at its
 * end).  Padding of the layouts (conv1's space-to-depth taps, head rows beyond 3nj) must stay 0. */
int dgp_get_param_buffer(dgp_handle* h, void** dev_ptr, size_t* bytes);
int dgp_params_changed(dgp_handle* h, void* stream);
/* Loss scaling for fp16 storage (precision = 1): the head gradients are multiplied by loss_scale before the network
 * backward so that small activation gradients stay above fp16's subnormal range; dgp_optimizer_step divides it out again and
 * dgp_get_variable(what = 1) returns unscaled gradients (after dgp_train_forward_backward the raw buffer of
 * dgp_get_grad_buffer holds loss_scale * gradient; after dgp_train_backward the gradient itself).
 * Default 1 (bf16 storage has fp32's exponent range and needs none). */
int dgp_train_set_loss_scale(dgp_handle* h, float loss_scale);
/* Flat float32 gradient buffer (kernel layouts: [weights | gamma | beta | head bias]) for ncclAllReduce. */
int dgp_get_grad_buffer(dgp_handle* h, void** dev_ptr, size_t* bytes);
/* ---- data-parallel training inside the C ABI (SURVEY 8b: dgp_attach_comm).  The reference's only multi-GPU design averages
 * tower gradients (src/deepgraphpose/helpers/utils_tf.py:4-39, average_gradients); here one process per GPU owns a handle and
 * an NCCL communicator, and the library itself all-reduces the flat gradient arena -- no Python, no torch.distributed on the
 * data path.  NCCL is resolved at run time (dlopen of libnccl.so.2, the copy already in the process if there is one).
 *  dgp_comm_unique_id: rank 0 creates the 128-byte ncclUniqueId and the host distributes it (MPI, a file, a torch store ...).
 *  dgp_comm_init_rank: every rank creates the communicator (owned and destroyed by the handle).
 *  dgp_attach_comm:    alternatively hand over an existing ncclComm_t (not owned; NULL detaches).
 *  dgp_allreduce_gradients: SUM all-reduce of the gradient arena of the LAST dgp_train_forward_backward in four buckets in
 *    backward order -- [block4 + heads], [block3], [block2], [conv1 + block1 + gamma / beta / bias] -- on the handle's
 *    communication stream, each bucket behind an event recorded at the point of the backward pass where it became final, so
 *    the first three overlap the rest of the backward; `stream` (the stream of the training calls) is made to wait for the
 *    last one.  *grad_scale receives 1 / world_size for dgp_optimizer_step (mean semantics of average_gradients; replicas stay
 *    bit-identical because every rank applies the same reduced gradient).  Without a communicator it is a no-op with
 *    *grad_scale = 1.
 *  dgp_allreduce_exposed_ms: time between the end of the last backward pass and the end of its all-reduce (the part of the
 *    communication that was NOT hidden behind compute).  Synchronises with the communication stream. */
int dgp_comm_unique_id(char* id128);
int dgp_comm_init_rank(dgp_handle* h, const char* id128, int nranks, int rank);
int dgp_attach_comm(dgp_handle* h, void* nccl_comm);
int dgp_comm_world_size(dgp_handle* h);
int dgp_allreduce_gradients(dgp_handle* h, void* stream, float* grad_scale);
int dgp_allreduce_exposed_ms(dgp_handle* h, float* ms);
/* Global gradient norm computed by the last dgp_optimizer_step (after grad_scale, before clipping). Synchronises. */
int dgp_get_grad_norm(dgp_handle* h, float* norm_host);
/* Device pointers of the head outputs (nt,2h,2w,nj) / (nt,2h,2w,2nj) written by the last dgp_train_forward_backward at this
 * shape (dgp_train_forward writes into the caller's buffers instead). */
int dgp_train_outputs(dgp_handle* h, int nt, int H, int W, float** logits_dev, float** locref_dev);
/* Replaces sess.run(variable) / TF.train.Saver.save (fitdgp.py:830-839): copies a trainable variable back to the host under
 * its TF name and TF layout.  what: 0 = value, 1 = gradient of the last step, 2 = momentum accumulator.
 * host_out may be NULL to query shape4 / ndim only. */
int dgp_get_variable(dgp_handle* h, const char* tf_var_name, int what, float* host_out, size_t max_elems, int64_t* shape4,
                     int* ndim);

/* Replaces TF.train.Saver.restore on a live session (resuming fit_dgp from a snapshot, fitdgp.py:689-720): overwrite a
 * trainable variable (what = 0; the 16-bit operands and BN scale/shift are refreshed) or its Momentum accumulator
 * (what = 2) from a host array in TF layout.  Together with dgp_get_variable this is checkpoint / resume. */
int dgp_set_variable(dgp_handle* h, const char* tf_var_name, int what, const float* host_in, size_t n_elems);

/* ---- test / profiling hooks (not part of the reference surface) ---- */
/* Keep every end_point (slim names, e.g. "resnet_v1_50/block1/unit_1/bottleneck_v1") of the next dgp_forward. */
int dgp_debug_keep_activations(dgp_handle* h, int enable);
/* Copy a kept end_point to host as float32 NHWC; shape4 receives (N,H,W,C). Returns DGP_ERR_INVALID if unknown. */
int dgp_debug_get_activation(dgp_handle* h, const char* end_point, float* host_out, size_t max_elems,
                             int64_t* shape4);
/* Process-wide count of the CUDA resources the library holds (buffers, pinned host memory, events, streams, graphs) and
 * of their device bytes, over all handles.  Either pointer may be NULL.  A handle's dgp_destroy returns both counts to
 * their value before its dgp_create. */
int dgp_debug_live_resources(int64_t* objects, int64_t* device_bytes);
/* One conv layer through the tcgen05 implicit-GEMM kernel (unit tests): x_dev bf16 NHWC (N,H,W,Cin), w_host float32
 * HWIO, scale/shift host float32 [Cout] or NULL, residual_dev bf16 or NULL (res_sub 1|2), out_dev bf16 or fp32.
 * pad_mode: 0 = TF SAME (stride 1), 1 = slim conv2d_same explicit padding, 2 = VALID. */
int dgp_conv2d(dgp_handle* h, const void* x_dev, int N, int H, int W, int Cin, const float* w_host, int R, int S,
               int Cout, int stride, int dilation, int pad_mode, const float* scale_host, const float* shift_host,
               const void* residual_dev, int res_sub, int res_H, int res_W, int relu, void* out_dev, int out_f32,
               int block_n, void* stream);
/* Weight gradient of one conv layer through the tcgen05 wgrad GEMM (unit tests): x_dev (N,H,W,Cin) and dy_dev
 * (N,P,Q,Cout) 16-bit NHWC; dw_dev float32 [Cout][R*S*Cin] (the kernel's weight layout, tap-major then channel).
 * dbg3 = NULL, or 3 descriptor overrides {LBO, SBO, k-step bytes} (0 = default) used during bring-up. */
int dgp_conv2d_wgrad(dgp_handle* h, const void* x_dev, int N, int H, int W, int Cin, const void* dy_dev, int R, int S,
                     int Cout, int stride, int dilation, int pad_mode, float* dw_dev, const int32_t* dbg3, void* stream);
/* CUDA-event timing per kernel family, recorded on the launching stream around every launch while enabled.
 * kinds: 0 = u8->bf16 space-to-depth prep, 1 = tcgen05 conv GEMM, 2 = max-pool, 3 = deconv col2im, 4 = soft-argmax,
 * 5 = dgrad GEMM, 6 = wgrad GEMM + reduce, 7 = bandwidth-class backward kernels.
 * dgp_get_profile synchronises the device, sums the elapsed ms and launch counts per kind and clears the records.
 * enable = 2 ("bracket" mode): ONE event pair around every run of consecutive same-kind launches (the 54 GEMM layers of a
 * forward pass are one run) -- the launches inside keep their programmatic-dependent-launch overlap, which an event record
 * between two of them would break. */
int dgp_set_profiling(dgp_handle* h, int enable);
int dgp_get_profile(dgp_handle* h, double* ms_by_kind, int64_t* count_by_kind, int nkinds);
/* The same records one by one, in launch order (elapsed ms and kind of up to max_records launches; clears the records):
 * the in-step duration of every layer, at the clocks and power state of the real step (tools/instep_layers.py). */
int dgp_get_profile_records(dgp_handle* h, float* ms, int32_t* kind, int max_records, int* n_records);
/* Host helper: CRC-32C of a byte range (the tensor checksums of TensorFlow checkpoint bundles, tf_checkpoint.py). */
uint32_t dgp_crc32c(const void* data, size_t n);
/* Number of kernels this handle has launched since creation. */
int64_t dgp_launch_count(const dgp_handle* h);
/* Number of SMs of the handle's device. */
int dgp_num_sms(const dgp_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* DGP_B200_H_ */
