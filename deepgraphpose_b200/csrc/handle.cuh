// Internal declarations shared by capi.cu (inference entry points) and train.cu (training step): the handle, the
// per-shape execution plan and the host helpers that build GEMM / wgrad launch parameters.
#pragma once
#include "../../include/dgp_b200.h"

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

#include "conv_gemm_sm100.cuh"
#include "kernels.cuh"
#include "owned.cuh"

namespace dgp {

struct TrainState;  // train.cu
struct TrainStateDeleter {
  void operator()(TrainState* ts) const;  // train.cu
};
typedef __nv_bfloat16 W16;  // opaque 16-bit storage element (bf16 or fp16 bits)

struct HostVar {
  std::vector<float> data;
  std::vector<int64_t> shape;
};

// How a trainable variable's TF layout maps onto its span of the parameter arena (variables.cu):
//   VAR_VECTOR     gamma, beta, biases: the same order
//   VAR_CONV       HWIO [R,S,Cin,Cout] <-> GEMM rows [Cout][R*S*Cin]
//   VAR_CONV1_S2D  [7,7,3,64] <-> the [64][256] space-to-depth matrix of conv1
//   VAR_HEAD       [3,3,cn,Cin] <-> rows t*ctot + c0 + cc (tap t, cc < cn) of the deconv heads' [Npad][Cin] GEMM matrix
enum VarLayout { VAR_VECTOR, VAR_CONV, VAR_CONV1_S2D, VAR_HEAD };

struct ArenaVar {
  std::string name;                  // TF name
  int ndim = 1;
  int64_t shape[4] = {0, 0, 0, 0};   // TF shape
  VarLayout layout = VAR_VECTOR;
  size_t off = 0, len = 0;           // arena span [off, off + len); pack writes only the variable's own elements of it
  int ctot = 0, c0 = 0;              // VAR_HEAD (cn = shape[2], Cin = shape[3])
};

struct ConvLayer {
  std::string scope;
  int R = 1, S = 1, Cin = 0, Cout = 0, stride = 1, dil = 1;
  bool relu = true;
  int K = 0;        // GEMM K (multiple of 64)
  int Npad = 0;     // rows of the weight matrix (multiple of block_n)
  int block_n = 0;
  __nv_bfloat16* w = nullptr;  // [Npad][K]  (points into the handle's 16-bit arena)
  float* scale = nullptr;      // [Npad] or nullptr
  float* shift = nullptr;
  size_t w_off = 0;            // offset of the fp32 master copy [Npad][K] in the parameter arena
  int ch_off = -1;             // offset of this layer's channels in the BN blocks (gamma / beta / mean / var / scale / shift)
};

struct UnitDesc {
  std::string scope;
  int depth, base, stride, rate;
  int shortcut = -1, conv1 = -1, conv2 = -1, conv3 = -1;  // indices into layers
};

enum StepKind { STEP_PREP = 0, STEP_GEMM = 1, STEP_POOL = 2, STEP_COL2IM = 3 };

struct Step {
  StepKind kind;
  ConvGemmParams gp;      // STEP_GEMM
  std::string end_point;  // name under which the output is kept in debug mode ("" = none)
  const void* out_ptr = nullptr;
  int oN = 0, oH = 0, oW = 0, oC = 0;  // output shape (bf16 NHWC) for debug dumps
  // pool
  const __nv_bfloat16* pin = nullptr;
  int pN = 0, pH = 0, pW = 0, pC = 0, pad_t = 0, pad_l = 0;
};

struct Plan {
  int B = 0, H = 0, W = 0;
  uint64_t last_use = 0;               // plan-cache LRU clock
  int H1 = 0, W1 = 0, Hs = 0, Ws = 0;  // conv1 output / s2d dims
  int hf = 0, wf = 0;                  // feature map (stride 16)
  std::vector<DevBuf> bufs;
  __nv_bfloat16* s2d = nullptr;
  float* contrib = nullptr;
  int contrib_ld = 0;
  std::vector<Step> steps;
  int head_step = 0;                   // index of the head GEMM in `steps` (everything before it is extract_features)
  // training plans keep every activation (no buffer rotation) and own the fp32 head outputs
  bool train = false;
  struct UnitBufs {
    void *x = nullptr, *sc = nullptr, *t1 = nullptr, *t2 = nullptr, *out = nullptr;  // unit input, projection shortcut, conv1/conv2/unit outputs
    int H = 0, W = 0, Ho = 0, Wo = 0, Cin = 0;
  };
  std::vector<UnitBufs> ub;
  void *c1 = nullptr, *pool = nullptr, *feat = nullptr;  // conv1 output, pool1 output, block4 output
  int Hp = 0, Wp = 0, pool_pad_t = 0, pool_pad_l = 0;
  float *logits = nullptr, *locref = nullptr;
  std::shared_ptr<void> bwd;  // train.cu: backward step list
  uint64_t fwd_token = 0;     // train.cu: token of the dgp_train_forward whose activations the plan holds (0 = none)
};

// Pillow's fixed-point resample table of one (in, out) size pair (resize_kernels.cu): dev holds first[out] | count[out] |
// weights[out][ksize] as int32; first / count are kept on the host for the launch geometry.
struct ResizeTable {
  int ksize = 0;
  std::vector<int32_t> first, count;
  DevBuf dev;
};

// What one dgp_estimate_pose_host / _stream call reads and writes, besides its frames.
struct PoseJob {
  int H0, W0;       // source frame size
  int H, W;         // size of the frames the network sees (after the transform)
  bool identity;    // the transform leaves frames unchanged
  const dgp_frame_transform* transform;
  float gamma, gauss_len;
  float* mu_host;
  int32_t* peak_host;
  float* lik_host;
};

// Kernel argument of the marker drawing (render_kernels.cu): the style of dgp_marker_style with its colour and edge tables
// by value, so a launch needs no allocation.
constexpr int kMaxDotsize = 64;
constexpr int kMaxEdges = 256;
constexpr int kMaxTrailpoints = 64;
struct MarkerArgs {
  int nj, dotsize, n_edges, trailpoints;
  double mask_threshold, scale_x, scale_y, stride, half_stride;
  uint8_t colors[3 * 256];
  uint8_t edges[2 * kMaxEdges];
  uint8_t skeleton_color[3];
};
// Validates `st` for (H, W) frames and fills `a` for the handle's joints and stride.
int marker_args(dgp_handle* h, const dgp_marker_style* st, int H, int W, MarkerArgs* a);
// Paints N frames from the float64 tables xs / ys / liks (rows of nj; row t is frame t, rows -history .. -1 the frames
// before it).
int draw_markers_impl(dgp_handle* h, uint8_t* frames, int N, int H, int W, const double* xs, const double* ys,
                      const double* liks, int history, const MarkerArgs& a, cudaStream_t s);
// The fused pass's table rows of an estimate_pose batch: x, y, lik of the soft-argmax read-outs mu (n,nj,2) / lik (n,nj) in
// video pixels, as eval.estimate_pose forms them on the host.
int marker_table_fused(dgp_handle* h, const float* mu, const float* lik, int n, const MarkerArgs& a, double* xs, double* ys,
                       double* liks, cudaStream_t s);

// Motion-JPEG (jpeg_kernels.cu): bytes of the header template (SOI .. SOS) and the largest frame side.
constexpr int kJpegHeaderBytes = 629;
constexpr int kJpegMaxDim = 16383;
// dgp_jpeg_capacity (-1 for an invalid size)
int64_t jpeg_capacity(int H, int W);
// dgp_encode_jpeg without the device switch
int encode_jpeg_impl(dgp_handle* h, const uint8_t* frames, int N, int H, int W, int quality, uint8_t* out, int64_t capacity,
                     int64_t* offsets, int64_t* sizes, cudaStream_t s);

// The rendering half of a dgp_estimate_pose_stream_render batch: markers drawn into the batch's source frames, the n real
// frames copied to the pinned writer slot `dst`, then handoff(handoff_arg) on the D2H stream.  With quality > 0
// (dgp_estimate_pose_stream_render_jpeg) the frames are encoded into `packets` instead (offsets | sizes of the n frames at
// `meta`), and only offsets | sizes go to `dst`; the writer thread copies the packets themselves.
struct RenderBatch {
  const MarkerArgs* args;
  uint8_t* dst;
  cudaHostFn_t handoff;
  void* handoff_arg;
  int quality;
  uint8_t* packets;
  int64_t packets_bytes;
  int64_t* meta;
};

// estimate_pose staging: source frames double-buffered between the H2D of the copy stream and the compute stream (slot =
// batch index & 1), the transformed batch that dgp_forward consumes when a frame transform is given, and the read-outs.
struct PoseStaging {
  Stream copy_stream;  // H2D of the next batch overlaps the current batch's kernels
  Event ev_copied[2], ev_consumed[2];
  DevBuf frames[2], xf, logits, mu, peak, lik;
  // rendering: the annotated frames leave on their own stream so that their D2H overlaps the next batch's forward
  Stream d2h_stream;
  Event ev_drawn[2];
  // Motion-JPEG rendering: the writer thread's copies of the encoded packets
  Stream packet_stream;
  // rendering: the float64 marker table, two halves used by alternate batches, each three planes (x | y | lik) of
  // marker_rows = K - 1 + batch rows of nj.  Rows [0, K-1) of a half hold the last frames before the batch (carried from
  // the other half), rows [K-1, K-1+n) the batch's own.
  DevBuf marker_table;
  int marker_rows = 0;
  int reserve(dgp_handle* h, int batch, int H0, int W0, int H, int W, bool identity);
  // Batch number `it` (n frames at host_frames, output rows [t0, t0 + n)): H2D, transform, forward + soft-argmax of run_n
  // rows, D2H of n read-outs.  release(release_arg) runs on the copy stream once host_frames has been copied.  With
  // `render`, the slot's source frames are annotated and copied out as well, and the slot counts as consumed only after that
  // copy.
  int run_batch(dgp_handle* h, const PoseJob& j, const uint8_t* host_frames, int n, int run_n, int it, int64_t t0,
                cudaHostFn_t release, void* release_arg, const RenderBatch* render = nullptr);
  // the D2H stream and events of run_batch's `render` step (created at the first rendering call), with `jpeg` the packet
  // stream, and the marker table for `batch` frames and `trailpoints`
  int reserve_render(dgp_handle* h, bool jpeg, int batch, int trailpoints);
};

}  // namespace dgp

using namespace dgp;  // internal header: the handle's members are dgp:: types

struct dgp_handle {
  std::unique_ptr<TrainState, TrainStateDeleter> train;  // set by dgp_train_enable
  dgp_config cfg;
  int device = 0;
  int num_sms = 0;
  int fp16 = 0;  // storage precision of activations / weights: 0 = bf16, 1 = fp16
  char err[512] = "";
  std::map<std::string, HostVar> host_vars;
  bool finalized = false;
  int depth = 0;             // 50, 101 or 152: slim resnet_v1_<depth>, read from the variable names at finalize
  int output_stride = 16;    // 8 or 16: slim's output_stride (dgp_set_output_stride, before finalize)
  std::string net_scope;     // "resnet_v1_<depth>": prefix of every backbone variable and end point
  std::vector<ConvLayer> layers;
  int conv1_layer = -1, head_layer = -1;
  std::vector<UnitDesc> units;
  float* head_bias = nullptr;  // points into the arena
  int ctot = 0;
  // Parameter arena (fp32 master, kernel layouts): [weights n_w | gamma n_ch | beta n_ch | head bias n_bias]
  DevBuf master;
  DevBuf w16;          // W16: 16-bit copy of the weight part (tensor-core operands)
  DevBuf bn_mean;      // frozen moving statistics [n_ch]
  DevBuf bn_var;
  DevBuf bn_ss;        // [scale n_ch | shift n_ch]
  DevBuf conv1_mask;   // [64][256] 1 = real 7x7x3 tap of the space-to-depth conv1 matrix
  size_t n_w = 0, n_ch = 0, n_bias = 0, n_params = 0;
  std::vector<ArenaVar> vars;              // the trainable variables in layer order (variables.cu)
  std::map<std::string, int> var_index;    // TF name -> index into vars
  std::map<std::tuple<int, int, int>, std::unique_ptr<Plan>> plans, train_plans;  // inference key (-B,..) = unchunked debug plan
  uint64_t plan_clock = 0;
  bool debug_keep = false;
  struct Kept {
    DevBuf buf;
    int N, H, W, C;
  };
  std::map<std::string, Kept> kept;
  int64_t launches = 0;
  // per-kernel-family CUDA-event profiling (bench.py roofline numbers)
  bool profiling = false;
  struct ProfRec {
    int kind;
    int count = 1;   // launches bracketed by the event pair (> 1 in bracket mode)
    Event a, b;
  };
  bool profile_brackets = false;  // dgp_set_profiling(h, 2): one event pair around every RUN of same-kind launches
  std::vector<ProfRec> prof;
  std::vector<Event> ev_pool;
  DevBuf flow_ws;   // dgp_learn_wt workspace
  DevBuf sa_ws;     // SaPartial: softargmax workspace
  DevBuf loss_ws;
  Stream stream;    // the handle's own stream: estimate_pose computes and the backward graph is captured on it
  PoseStaging pose;
  // dgp_resize_crop: tables per (in, out) size pair and the uint8 intermediate of the horizontal pass
  std::map<std::pair<int, int>, ResizeTable> resize_tables;
  DevBuf resize_tmp;
  // dgp_augment: two scratch frame sets of the ping-pong between passes, elastic fields (dx | dy per frame) and the
  // intermediate of the field's horizontal pass
  DevBuf aug_scratch[2], aug_fields, aug_tmp;
  // dgp_estimate_pose_stream: pinned host ring the reader thread decodes into (stream.cu)
  PinnedBuf ring_slot[3];
  // dgp_estimate_pose_stream_render: pinned host ring of annotated frames the writer thread drains (stream.cu)
  PinnedBuf writer_slot[3];
  // dgp_encode_jpeg: header template + Huffman codes per (H, W, quality), and the scratch of its launches (coefficients,
  // block bit offsets, segment bit buffers, segment sizes / offsets)
  std::map<std::tuple<int, int, int>, DevBuf> jpeg_tables;
  DevBuf jpeg_coef, jpeg_bitoff, jpeg_raw, jpeg_seg;
  // dgp_estimate_pose_stream_render_jpeg, per writer slot: device packets and their offsets | sizes, and the pinned copy of
  // the packets (grown by the writer thread to what a batch needs)
  DevBuf jpeg_packets[3], jpeg_meta[3];
  PinnedBuf jpeg_host[3];
};

// loss forward (+ optional loss-side backward) shared by dgp_loss_forward / dgp_loss_backward / the training step
extern "C" int dgp_run_loss_impl(dgp_handle* h, const dgp_loss_cfg* cfg, const dgp_loss_batch* b, float* losses_dev,
                                   float* targets_all_dev, float* grad_pred_dev, float* grad_locref_dev, int visible_only,
                                   void* stream);

namespace dgp {

W16 cvt16(const dgp_handle* h, float f);
float cvt16_to_float(const dgp_handle* h, W16 v);
int fail(dgp_handle* h, int code, const char* fmt, ...);

#define CU_OK(h, expr)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess)                                                                      \
      return fail(h, DGP_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

int ceil_div(int a, int b);
void same_pad(int in, int k, int stride, int rate, int* beg, int* out);
int pick_block_n(int n);
int tmem_cols_for(int block_n);
void conv_geometry(int R, int S, int stride, int dil, int H, int W, int pad_mode, int* Pout, int* Qout, int* lower_h_,
                   int* lower_w_, int* upper_h_, int* upper_w_);
int setup_epilogue(dgp_handle* h, ConvGemmParams& g, const char* scope, int n_img);
int make_gemm_step(dgp_handle* h, const ConvLayer& L, const void* x, int N, int H, int W, int pad_mode, void* out,
                   bool out_f32, const __nv_bfloat16* residual, int res_sub, int res_H, int res_W, int block_n_override,
                   Step* st, int* Ho, int* Wo);
int make_wgrad_params(dgp_handle* h, const char* scope, int R, int S, int Cin, int Cout, int stride, int dil,
                      const void* x, int N, int H, int W, int pad_mode, const void* dy, WgradParams* wp);
// conv1's wgrad params: dy (B*H1*W1, 64) 16-bit against the space-to-depth input s2d (B, Hs, Ws, 16) of launch_prep_s2d
int make_conv1_wgrad_params(dgp_handle* h, const void* dy, const void* s2d, int B, int H1, int W1, int Hs, int Ws,
                            WgradParams* wp);
int alloc_buf(dgp_handle* h, std::vector<DevBuf>* bufs, size_t bytes, void** out);
int build_plan(dgp_handle* h, int B, int H, int W, bool train, Plan** out);
int run_forward_plan(dgp_handle* h, Plan* pl, const uint8_t* frames_dev, float* logits_dev, float* locref_dev,
                     cudaStream_t s, int first_step = 0, int last_step = -1);
int ensure(dgp_handle* h, DevBuf* b, size_t bytes);
int refresh_operands(dgp_handle* h, cudaStream_t s);

// variables.cu
size_t tf_elems(const ArenaVar& v);
std::string shape_str(const ArenaVar& v);  // "[7,7,3,64]"
// TF layout <-> the variable's span (span = arena + v.off)
void pack(const ArenaVar& v, const float* tf, float* span);
void unpack(const ArenaVar& v, const float* span, float* tf);
// Fills h->vars / h->var_index from the finalized layers: arena [weights n_w | gamma n_ch | beta n_ch | head bias n_bias].
// *frozen gets the moving statistics, with spans in [moving_mean n_ch | moving_variance n_ch].
void build_variable_table(dgp_handle* h, std::vector<ArenaVar>* frozen);
// train.cu: the arena dgp_get_variable / dgp_set_variable address with `what` (0 value, 1 gradient, 2 momentum) and the
// factor that turns a stored element into the variable's value (gradients are stored multiplied by arena_scale).
float* variable_arena(dgp_handle* h, int what, float* unscale);
// train.cu: dgp_set_variable changed the weights: every dgp_train_forward token is stale, the dgrad operands too.
void weights_changed(dgp_handle* h);
// Size of a transformed frame (DGP_ERR_INVALID for an invalid transform); *identity: the transform leaves frames unchanged.
int transform_dims(int H0, int W0, const dgp_frame_transform* t, int* H, int* W, bool* identity);
// dgp_resize_crop without the device switch (resize_kernels.cu)
int resize_crop_impl(dgp_handle* h, const uint8_t* src, int N, int H0, int W0, const dgp_frame_transform* t, uint8_t* dst,
                     cudaStream_t s);

inline Event prof_event(dgp_handle* h) {
  Event e;
  if (!h->ev_pool.empty()) {
    e = std::move(h->ev_pool.back());
    h->ev_pool.pop_back();
  } else {
    create(&e, cudaEventDefault);
  }
  return e;
}

struct ProfScope {
  dgp_handle* h;
  cudaStream_t s;
  int idx = -1;
  ProfScope(dgp_handle* h_, int kind, cudaStream_t s_, int count = 1) : h(h_), s(s_) {
    if (!h->profiling) return;
    dgp_handle::ProfRec r;
    r.kind = kind;
    r.count = count;
    r.a = prof_event(h);
    r.b = prof_event(h);
    cudaEventRecord(r.a.get(), s);
    idx = (int)h->prof.size();
    h->prof.push_back(std::move(r));
  }
  ~ProfScope() {
    if (idx >= 0) cudaEventRecord(h->prof[idx].b.get(), s);
  }
};

}  // namespace dgp
