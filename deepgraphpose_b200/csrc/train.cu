// Training step of fit_dgp on the GPU: network backward (dgrad / wgrad of the 53 / 104 / 155 convs of
// ResNet-50 / 101 / 152 + deconv heads), frozen-BN
// parameter gradients, global-norm clipping and the Momentum update.
// Reference: src/deepgraphpose/models/fitdgp.py:706-713
//   optimizer = MomentumOptimizer(lr, 0.9); grads = compute_gradients(total_loss, TF.trainable_variables());
//   grads, _ = clip_by_global_norm(grads, 10.0); train_op = apply_gradients(...)
// with the graph of fitdgp.py:934-1128 (PoseNet with is_training=False -> frozen moving statistics, trainable
// gamma / beta / conv weights / deconv weights + biases).
//
// Data flow per bottleneck unit (all tensors 16-bit NHWC, gradients w.r.t. BN outputs "dy"):
//   junction  : d = g_out * [out > 0]                      (relu_bn_bwd, + BN sums of conv3 / projection shortcut)
//   conv3     : wgrad(t2, d) ; g_t2 = dgrad(d)             (tcgen05 GEMMs)
//   conv2     : dy2 = g_t2 * [t2 > 0] ; wgrad(t1, dy2) ; g_t1 = dgrad(dy2)   (stride 2: zero-inserted dy2, stride-1 conv)
//   conv1     : dy1 = g_t1 * [t1 > 0] ; wgrad(x, dy1) ; g_x = dgrad(dy1) + shortcut path
//   shortcut  : identity: + d (GEMM residual; stride 2: scatter-add)   projection: wgrad(x, d), g_x += dgrad(d)
// The BN scale of a layer is folded into its dgrad operand (build_dgrad_w_kernel) and applied per output row in the
// wgrad reduction, so every GEMM consumes the same dy tensor.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <dlfcn.h>

#include <algorithm>
#include <functional>

#include "handle.cuh"

using namespace dgp;

namespace dgp {

struct BStep {
  int kind;      // profiling family: 5 = dgrad GEMM, 6 = wgrad GEMM (+ reduce), 7 = bandwidth-class backward kernel
  int launches;
  std::function<cudaError_t(cudaStream_t)> run;
  // Hazard notes for the two-branch capture (see dgp_train_forward_backward): a wgrad step (kind 6) only READS the gradient
  // buffer `rd` (plus forward activations, which the backward never writes) and may run on the side branch until a main-branch
  // step WRITES that buffer (`wr`); `join` = the step consumes what the wgrads produced (rowdot -> dgamma).
  const void* wr = nullptr;
  const void* rd = nullptr;
  bool join = false;
};

struct Backward {
  std::vector<DevBuf> bufs;  // gradient buffers (declared first: the graph exec that references them goes before them)
  std::vector<BStep> steps;
  float *g_logits = nullptr, *g_locref = nullptr;
  // Deferred frozen-BN gradients: every mask site leaves its per-row-block sums of dy in its own region of `bn_part`, every
  // wgrad its <W, dW_raw> products in its slice of `rowdot`; ONE kernel at the end of the backward turns both into dbeta / dgamma
  // for every channel (26 560 at ResNet-50, 75 712 at ResNet-152; instead of ~100 latency-bound launches of 3-7 us each inside the pass).
  float* bn_part = nullptr;
  float* rowdot = nullptr;
  BnGroup* bn_table = nullptr;
  size_t bn_part_floats = 0;
  std::vector<BnGroup> bn_groups;   // host copy, one entry per 8 channels
  int bucket_step[3] = {-1, -1, -1};  // steps after which buckets 0 (block4 + heads), 1 (block3), 2 (block2) are final
  // The ~280 launches of the network backward have fixed arguments per plan: after the first (eager) step they are
  // replayed as one CUDA graph, which removes the launch gaps between the many small bandwidth-class kernels.
  int runs = 0;
  int launches = 0;
  uint64_t graph_gen = 0;
  GraphExec graph_exec;
};

struct TrainState {
  DevBuf grads, accum;  // float, n_params each
  DevBuf norm_partial;
  DevBuf norm_clip;     // float [0] = global norm of the last step, [1] = clip factor
  DevBuf bn_partial, wgrad_ws;
  std::vector<DevBuf> wd;  // per layer: W16 dgrad operand [Cin][taps*Cout] (empty for conv1 / head)
  DevBuf head_wd;
  int head_Kd = 0;
  bool wd_fresh = false;
  uint64_t ws_gen = 1;           // bumped whenever a shared workspace is reallocated (captured graphs hold its address)
  float loss_scale = 1.0f;       // head gradients are multiplied by this before the network backward (fp16 storage)
  // What the gradient arena holds: arena_scale x the true gradient (loss_scale after dgp_train_forward_backward, 1 after
  // dgp_train_backward); every reader divides by it.  grad_mode is the device word the arena-writing kernels read
  // (GradMode), grad_mode_host the value last stored there.
  float arena_scale = 1.0f;
  bool arena_fused = false;      // the last backward was dgp_train_forward_backward's (no accumulation onto it)
  DevBuf grad_mode;              // GradMode
  GradMode grad_mode_host = {0, 1.0f};
  uint64_t fwd_seq = 0;          // tokens handed out by dgp_train_forward
  DevBuf wd_jobs;                // DgradWJob: device table for the one-launch rebuild of every dgrad operand
  int n_wd_jobs = 0, wd_tiles = 0;
  // Data-parallel all-reduce owned by the library (dgp_attach_comm / dgp_comm_init_rank + dgp_allreduce_gradients): the
  // weight gradients of a block are final once the backward has passed its first unit, so the arena is reduced in four
  // buckets in backward order -- [block4 + heads], [block3], [block2], [conv1 + block1 + gamma/beta/bias] -- each on the
  // communication stream behind an event recorded at that point of the backward.  Bucket 0 holds about two thirds of the
  // arena and is final after the first quarter of the backward pass.
  static constexpr int kBuckets = 4;
  size_t bucket_off[kBuckets + 1] = {0, 0, 0, 0, 0};   // weight-part offsets: bucket k = [bucket_off[k+1], bucket_off[k])
  Event ev_bucket[kBuckets - 1];
  void* comm = nullptr;           // ncclComm_t
  bool comm_owned = false;
  int comm_world = 1;
  Stream comm_stream;
  Event ev_bwd_done, ev_comm_done;   // timing enabled: exposed all-reduce time
  bool bwd_ran = false;           // a backward has recorded the bucket events on some stream
  // second branch of the captured backward: the wgrad chain (see dgp_train_forward_backward)
  Stream side_stream;
  std::vector<Event> branch_events;

  void release_comm();
  ~TrainState() { release_comm(); }
};

void TrainStateDeleter::operator()(TrainState* ts) const { delete ts; }

// ---- NCCL, resolved at run time from the process (the copy PyTorch loaded, if any) or the system library: the .so has no
// link-time NCCL dependency, and a host that never calls dgp_attach_comm / dgp_comm_init_rank never needs it.
namespace nccl {
typedef struct { char internal[128]; } UniqueId;     // ncclUniqueId (NCCL_UNIQUE_ID_BYTES = 128)
typedef int (*GetUniqueIdFn)(UniqueId*);
typedef int (*CommInitRankFn)(void**, int, UniqueId, int);
typedef int (*CommDestroyFn)(void*);
typedef int (*CommCountFn)(void*, int*);
typedef int (*AllReduceFn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef int (*GroupFn)();
typedef const char* (*ErrStrFn)(int);
constexpr int kFloat = 7, kSum = 0;                  // ncclFloat32, ncclSum
struct Api {
  GetUniqueIdFn get_unique_id = nullptr;
  CommInitRankFn comm_init_rank = nullptr;
  CommDestroyFn comm_destroy = nullptr;
  CommCountFn comm_count = nullptr;
  AllReduceFn all_reduce = nullptr;
  GroupFn group_start = nullptr, group_end = nullptr;
  ErrStrFn err_str = nullptr;
  bool ok = false;
};
const Api& api() {
  static Api a;
  static bool tried = false;
  if (tried) return a;
  tried = true;
  void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);   // already in the process (torch's bundled NCCL)
  if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) return a;
  a.get_unique_id = (GetUniqueIdFn)dlsym(lib, "ncclGetUniqueId");
  a.comm_init_rank = (CommInitRankFn)dlsym(lib, "ncclCommInitRank");
  a.comm_destroy = (CommDestroyFn)dlsym(lib, "ncclCommDestroy");
  a.comm_count = (CommCountFn)dlsym(lib, "ncclCommCount");
  a.all_reduce = (AllReduceFn)dlsym(lib, "ncclAllReduce");
  a.group_start = (GroupFn)dlsym(lib, "ncclGroupStart");
  a.group_end = (GroupFn)dlsym(lib, "ncclGroupEnd");
  a.err_str = (ErrStrFn)dlsym(lib, "ncclGetErrorString");
  a.ok = a.get_unique_id && a.comm_init_rank && a.comm_destroy && a.comm_count && a.all_reduce && a.group_start &&
         a.group_end && a.err_str;
  return a;
}
}  // namespace nccl

void TrainState::release_comm() {
  if (!comm) return;
  if (comm_owned && nccl::api().ok) nccl::api().comm_destroy(comm);
  comm = nullptr;
  comm_owned = false;
  comm_world = 1;
}

namespace {

int refresh_dgrad_weights(dgp_handle* h, cudaStream_t s) {
  TrainState* ts = h->train.get();
  const float* master = h->master.get<float>();
  CU_OK(h, launch_build_dgrad_w(ts->wd_jobs.get<DgradWJob>(), ts->n_wd_jobs, ts->wd_tiles, master, h->bn_ss.get<float>(), h->fp16,
                                s));
  const ConvLayer& Lh = h->layers[h->head_layer];
  CU_OK(h, launch_build_head_dgrad_w(master + Lh.w_off, 9 * h->ctot, 2048, ts->head_wd.get<W16>(), ts->head_Kd, h->fp16, s));
  h->launches += 2;
  ts->wd_fresh = true;
  return DGP_OK;
}

// Pushes the dgrad GEMM `gp`, which writes `out`.  mask_act != nullptr: `out` is the gradient w.r.t. the post-ReLU tensor
// mask_act (same shape); when the GEMM runs the staged epilogue, that epilogue also applies its consumer's dy = g * [act > 0]
// and leaves the per-channel sums of dy (conv_gemm_kernel kMask) in a [ceil(M/32)][N] region of bw->bn_part reserved here.
// Returns the region's offset, or -1 when the caller has to add the stand-alone mask pass.
long long push_dgrad_gemm(dgp_handle* h, Backward* bw, ConvGemmParams gp, void* out, const void* mask_act) {
  long long off = -1;
  if (mask_act != nullptr && gp.epi_mode == 1) {
    off = (long long)bw->bn_part_floats;
    bw->bn_part_floats += (size_t)ceil_div(gp.M, 32) * gp.N;
    gp.mask_act = mask_act;
  }
  const int sms = h->num_sms;
  bw->steps.push_back({5, 1, [gp, sms, bw, off](cudaStream_t s) {
                         ConvGemmParams g = gp;
                         if (off >= 0) g.colsum_part = bw->bn_part + off;
                         return launch_conv_gemm(g, sms, s);
                       }});
  bw->steps.back().wr = out;
  return off;
}

// dgrad of layer L as a stride-1 conv of dy (N,H,W,L.Cout) with the transposed / flipped operand -> out (N,H,W,L.Cin).
// mask_act / *site: see push_dgrad_gemm.
int add_dgrad(dgp_handle* h, Backward* bw, const ConvLayer& L, const DevBuf& wd, const void* dy, int N, int H, int W, void* out,
              const void* residual, const void* mask_act = nullptr, long long* site = nullptr) {
  ConvLayer D;
  D.scope = L.scope + "/dgrad";
  D.R = L.R; D.S = L.S; D.Cin = L.Cout; D.Cout = L.Cin; D.stride = 1; D.dil = L.dil; D.relu = false;
  D.K = L.R * L.S * L.Cout;
  D.Npad = L.Cin;
  D.block_n = L.Cin >= 256 ? 256 : L.Cin;
  D.w = wd.get<W16>();
  Step st;
  int Ho, Wo;
  int rc = make_gemm_step(h, D, dy, N, H, W, (L.R == 1 && L.S == 1) ? 0 : 1, out, false, (const __nv_bfloat16*)residual, 1, H,
                          W, 0, &st, &Ho, &Wo);
  if (rc) return rc;
  const long long off = push_dgrad_gemm(h, bw, st.gp, out, mask_act);
  if (site) *site = off;
  return DGP_OK;
}

// bn_layer: the conv's frozen BN -- the reduce also leaves <W[co, 4 kk], dW_raw[co, 4 kk]> in the layer's slice of bw->rowdot
// (-> dgamma in the final bn_finalize_all pass), or nullptr (heads)
int add_wgrad_params(dgp_handle* h, Backward* bw, const WgradParams& wp0, const void* dy_buf, const float* rowscale,
                     const float* mask, float* grad, size_t* ws_need, const ConvLayer* bn_layer = nullptr) {
  TrainState* ts = h->train.get();
  const size_t need = wgrad_workspace_bytes(wp0);
  if (need > *ws_need) *ws_need = need;
  const int sms = h->num_sms;
  const float* wmaster = bn_layer ? h->master.get<float>() + bn_layer->w_off : nullptr;
  const size_t rd_off = bn_layer ? bn_layer->w_off / 4 : 0;
  if (bn_layer) {
    for (int c = 0; c < wp0.Cout; c += 8) {
      BnGroup& g = bw->bn_groups[(bn_layer->ch_off + c) / 8];
      g.rd_off = rd_off + (unsigned long long)c * (wp0.Kw / 4);
      g.K4 = wp0.Kw / 4;
    }
  }
  bw->steps.push_back({6, 2, [=](cudaStream_t s) {
                         WgradParams wp = wp0;
                         wp.partials = ts->wgrad_ws.get<float>();
                         cudaError_t e = launch_wgrad_gemm(wp, sms, s);
                         if (e != cudaSuccess) return e;
                         return launch_wgrad_reduce(wp, rowscale, mask, grad, ts->grad_mode.get<GradMode>(), s, wmaster,
                                                    wmaster ? bw->rowdot + rd_off : nullptr);
                       }});
  bw->steps.back().rd = dy_buf;
  return DGP_OK;
}

int add_wgrad(dgp_handle* h, Backward* bw, const ConvLayer& L, const void* x, int N, int H, int W, int pad_mode,
              const void* dy, size_t* ws_need) {
  WgradParams wp;
  int rc = make_wgrad_params(h, L.scope.c_str(), L.R, L.S, L.Cin, L.Cout, L.stride, L.dil, x, N, H, W, pad_mode, dy, &wp);
  if (rc) return rc;
  return add_wgrad_params(h, bw, wp, dy, L.scale, nullptr, h->train->grads.get<float>() + L.w_off, ws_need, &L);
}

// dy = g * [act > 0] in place and the dy sums of up to two layers (conv3 and the projection shortcut share dy at a junction).
// site >= 0: the dgrad GEMM that produced g already applied the mask and writes the [ceil(M/32)][C] sums into that region of
// bw->bn_part; otherwise a stand-alone relu_bn_bwd pass does both into a region of its own.
struct ScatterSrc {   // pending gradient of a stride-2 identity shortcut, folded into the next stand-alone junction mask
  const void* d = nullptr;
  int H = 0, W = 0, P = 0, Q = 0;
};

void add_mask(dgp_handle* h, Backward* bw, void* g, const void* act, int M, int C, const ConvLayer* la, const ConvLayer* lb,
              long long site = -1, int site_rows = 0, ScatterSrc sc = ScatterSrc()) {
  int rows;
  if (site >= 0) {
    rows = site_rows > 0 ? site_rows : ceil_div(M, 32);
  } else {
    rows = relu_bn_bwd_blocks(M, C);
    site = (long long)bw->bn_part_floats;
    bw->bn_part_floats += (size_t)rows * C;
    const int fp16 = h->fp16;
    const long long off = site;
    bw->steps.push_back({7, 1, [=](cudaStream_t s) {
                           return launch_relu_bn_bwd(g, act, M, C, bw->bn_part + off, fp16, s, sc.d, sc.H, sc.W, sc.P, sc.Q);
                         }});
    bw->steps.back().wr = g;
  }
  for (const ConvLayer* L : {la, lb}) {
    if (!L) continue;
    for (int c = 0; c < C; c += 8) {
      BnGroup& grp = bw->bn_groups[(L->ch_off + c) / 8];
      grp.part_off = (unsigned long long)site;
      grp.rows = rows; grp.C = C; grp.col = c;
    }
  }
}

int build_backward(dgp_handle* h, Plan* pl) {
  TrainState* ts = h->train.get();
  std::shared_ptr<Backward> bw(new Backward());
  const int B = pl->B, nj = h->cfg.num_joints, fp16 = h->fp16;
  const int hf = pl->hf, wf = pl->wf;
  int rc;
  void* p = nullptr;
  size_t ws_need = 0, bn_need = 0;
  long long g_site = -1;   // >= 0: the gradient w.r.t. the current unit's output already carries its junction mask; its dy sums live there
  bw->bn_groups.assign((h->n_ch + 7) / 8, BnGroup());
  // ---- gradient buffers
  size_t max_unit = (size_t)pl->Hp * pl->Wp * 64, max_t1 = 0, max_t2 = 0, max_up = 0;
  for (size_t i = 0; i < h->units.size(); ++i) {
    const UnitDesc& u = h->units[i];
    const Plan::UnitBufs& ub = pl->ub[i];
    max_unit = std::max(max_unit, (size_t)ub.Ho * ub.Wo * u.depth);
    max_unit = std::max(max_unit, (size_t)ub.H * ub.W * ub.Cin);
    max_t1 = std::max(max_t1, (size_t)ub.H * ub.W * u.base);
    max_t2 = std::max(max_t2, (size_t)ub.Ho * ub.Wo * u.base);
    if (u.stride == 2) max_up = std::max(max_up, (size_t)ub.H * ub.W * u.base);
  }
  void *gbuf[3], *gt1 = nullptr, *gt2 = nullptr, *gup = nullptr, *g_c1 = nullptr, *dG = nullptr;
  for (int i = 0; i < 3; ++i)
    if ((rc = alloc_buf(h, &bw->bufs, (size_t)B * max_unit * 2 + 1024, &gbuf[i]))) return rc;
  if ((rc = alloc_buf(h, &bw->bufs, (size_t)B * max_t1 * 2 + 1024, &gt1))) return rc;
  if ((rc = alloc_buf(h, &bw->bufs, (size_t)B * max_t2 * 2 + 1024, &gt2))) return rc;
  if (max_up && (rc = alloc_buf(h, &bw->bufs, (size_t)B * max_up * 2 + 1024, &gup))) return rc;
  if ((rc = alloc_buf(h, &bw->bufs, (size_t)B * pl->H1 * pl->W1 * 64 * 2 + 1024, &g_c1))) return rc;
  const int Kd = ts->head_Kd;
  const int Mf = B * hf * wf;
  if ((rc = alloc_buf(h, &bw->bufs, (size_t)Mf * Kd * 2 + 1024, &dG))) return rc;
  if ((rc = alloc_buf(h, &bw->bufs, (size_t)B * 4 * hf * wf * nj * 4, &p))) return rc;
  bw->g_logits = (float*)p;
  if (pl->locref) {
    if ((rc = alloc_buf(h, &bw->bufs, (size_t)B * 4 * hf * wf * 2 * nj * 4, &p))) return rc;
    bw->g_locref = (float*)p;
  }
  float* g_logits = bw->g_logits;
  float* g_locref = bw->g_locref;
  const int ctot = h->ctot;

  // ---- heads: col2im gather, bias gradient, wgrad, dgrad
  bw->steps.push_back({7, 1, [=](cudaStream_t s) { return launch_col2im_bwd(g_logits, g_locref, B, hf, wf, ctot, nj, dG, Kd, fp16, s); }});
  bw->steps.back().wr = dG;
  {
    float* dbias = ts->grads.get<float>() + h->n_w + 2 * h->n_ch;
    const size_t npix = (size_t)B * 4 * hf * wf;
    bn_need = std::max(bn_need, (size_t)head_bias_blocks() * 256 * sizeof(float));
    bw->steps.push_back({7, g_locref ? 4 : 2, [=](cudaStream_t s) {
                           float* partial = ts->bn_partial.get<float>();
                           const GradMode* mode = ts->grad_mode.get<GradMode>();
                           cudaError_t e = launch_head_bias_grad(g_logits, npix, nj, partial, dbias, mode, s);
                           if (e == cudaSuccess && g_locref)
                             e = launch_head_bias_grad(g_locref, npix, 2 * nj, partial, dbias + nj, mode, s);
                           return e;
                         }});
  }
  {
    const ConvLayer& Lh = h->layers[h->head_layer];
    WgradParams wp;
    // gradient rows = Npad rows of the head matrix; dy = dG (Kd >= Npad columns, zero beyond 9 * ctot)
    rc = make_wgrad_params(h, "pose/heads", 1, 1, 2048, Kd, 1, 1, pl->feat, B, hf, wf, 0, dG, &wp);
    if (rc) return rc;
    wp.Cout = Lh.Npad;
    wgrad_plan(&wp, h->num_sms);
    if ((rc = add_wgrad_params(h, bw.get(), wp, dG, nullptr, nullptr, ts->grads.get<float>() + Lh.w_off, &ws_need))) return rc;
    ConvLayer D;
    D.scope = "pose/heads/dgrad"; D.R = 1; D.S = 1; D.Cin = Kd; D.Cout = 2048; D.relu = false;
    D.K = Kd; D.Npad = 2048; D.block_n = 256; D.w = ts->head_wd.get<W16>();
    Step st;
    int Ho, Wo;
    rc = make_gemm_step(h, D, dG, B, hf, wf, 0, gbuf[0], false, nullptr, 1, 0, 0, 0, &st, &Ho, &Wo);
    if (rc) return rc;
    // gbuf[0] is the gradient w.r.t. block4's output: the last unit's junction mask rides in this GEMM's epilogue
    g_site = push_dgrad_gemm(h, bw.get(), st.gp, gbuf[0], pl->feat);
  }

  // ---- bottleneck units, last to first.  G = gradient w.r.t. the unit output (then d in place).
  int gi = 0;  // index of G in gbuf
  ScatterSrc scatter;
  for (int i = (int)h->units.size() - 1; i >= 0; --i) {
    const UnitDesc& u = h->units[i];
    const Plan::UnitBufs& ub = pl->ub[i];
    const ConvLayer& L1 = h->layers[u.conv1];
    const ConvLayer& L2 = h->layers[u.conv2];
    const ConvLayer& L3 = h->layers[u.conv3];
    const ConvLayer* Ls = u.shortcut >= 0 ? &h->layers[u.shortcut] : nullptr;
    void* G = gbuf[gi];
    void* Gx = gbuf[(gi + 1) % 3];
    void* Gy = gbuf[(gi + 2) % 3];
    const int Mo = B * ub.Ho * ub.Wo, Mi = B * ub.H * ub.W;
    // junction
    add_mask(h, bw.get(), G, ub.out, Mo, u.depth, &L3, Ls, g_site, 0, g_site < 0 ? scatter : ScatterSrc());
    scatter = ScatterSrc();
    // conv3 (its dgrad's epilogue applies conv2's ReLU mask and leaves the dy sums)
    long long site = -1;
    if ((rc = add_wgrad(h, bw.get(), L3, ub.t2, B, ub.Ho, ub.Wo, 0, G, &ws_need))) return rc;
    if ((rc = add_dgrad(h, bw.get(), L3, ts->wd[u.conv3], G, B, ub.Ho, ub.Wo, gt2, nullptr, ub.t2, &site))) return rc;
    // conv2
    add_mask(h, bw.get(), gt2, ub.t2, Mo, u.base, &L2, nullptr, site);
    if ((rc = add_wgrad(h, bw.get(), L2, ub.t1, B, ub.H, ub.W, 1, gt2, &ws_need))) return rc;
    if (u.stride == 1) {
      if ((rc = add_dgrad(h, bw.get(), L2, ts->wd[u.conv2], gt2, B, ub.H, ub.W, gt1, nullptr, ub.t1, &site))) return rc;
    } else {
      const int P = ub.Ho, Q = ub.Wo, H = ub.H, W = ub.W, C = u.base;
      bw->steps.push_back({7, 1, [=](cudaStream_t s) { return launch_upsample2(gt2, B, P, Q, C, gup, H, W, s); }});
      bw->steps.back().wr = gup;
      if ((rc = add_dgrad(h, bw.get(), L2, ts->wd[u.conv2], gup, B, ub.H, ub.W, gt1, nullptr, ub.t1, &site))) return rc;
    }
    // conv1
    add_mask(h, bw.get(), gt1, ub.t1, Mi, u.base, &L1, nullptr, site);
    if ((rc = add_wgrad(h, bw.get(), L1, ub.x, B, ub.H, ub.W, 0, gt1, &ws_need))) return rc;
    // the GEMM that completes Gx (gradient w.r.t. this unit's input = the previous unit's post-ReLU output) also applies that
    // unit's junction mask -- except for the first unit (its input is the max-pool output) and the stride-2 identity shortcuts
    // (their scatter-add into Gx rides in the previous unit's stand-alone junction mask)
    const void* junction_act = i > 0 ? ub.x : nullptr;
    g_site = -1;
    if (Ls) {
      if ((rc = add_dgrad(h, bw.get(), L1, ts->wd[u.conv1], gt1, B, ub.H, ub.W, Gy, nullptr))) return rc;
      if ((rc = add_wgrad(h, bw.get(), *Ls, ub.x, B, ub.H, ub.W, 0, G, &ws_need))) return rc;
      if ((rc = add_dgrad(h, bw.get(), *Ls, ts->wd[u.shortcut], G, B, ub.H, ub.W, Gx, Gy, junction_act, &g_site))) return rc;
    } else if (u.stride == 1) {
      if ((rc = add_dgrad(h, bw.get(), L1, ts->wd[u.conv1], gt1, B, ub.H, ub.W, Gx, G, junction_act, &g_site))) return rc;
    } else {
      if (i == 0)
        return fail(h, DGP_ERR_STATE, "backward plan: %s: a stride-2 identity shortcut in the first unit is not supported",
                    u.scope.c_str());
      if ((rc = add_dgrad(h, bw.get(), L1, ts->wd[u.conv1], gt1, B, ub.H, ub.W, Gx, nullptr))) return rc;
      // Gx[n,2p,2q] += G[n,p,q] rides in the previous unit's junction mask (the next step of this plan; G stays intact until
      // then: it is that unit's third buffer, written only after its mask)
      scatter.d = G; scatter.H = ub.H; scatter.W = ub.W; scatter.P = ub.Ho; scatter.Q = ub.Wo;
    }
    gi = (gi + 1) % 3;
    if (u.shortcut >= 0)
      for (int k = 0; k < 3; ++k)
        if (h->layers[u.shortcut].w_off == ts->bucket_off[k + 1]) bw->bucket_step[k] = (int)bw->steps.size();
  }
  // ---- root: max-pool backward, conv1 ReLU/BN, conv1 wgrad (no dgrad: the input is the image)
  {
    void* Gp = gbuf[gi];
    const void* c1 = pl->c1;
    const int H1 = pl->H1, W1 = pl->W1, Hp = pl->Hp, Wp = pl->Wp, pt = pl->pool_pad_t, plft = pl->pool_pad_l;
    const ConvLayer& L = h->layers[h->conv1_layer];
    // max-pool gradient + conv1's ReLU mask + dy sums in one pass (bwd_kernels.cu: maxpool_relu_bwd_kernel)
    const long long site = (long long)bw->bn_part_floats;
    const int rows = maxpool_relu_bwd_rows(B, H1, W1);
    bw->bn_part_floats += (size_t)rows * 64;
    Backward* bwp = bw.get();
    bw->steps.push_back({7, 1, [=](cudaStream_t s) {
                           return launch_maxpool_relu_bwd(c1, Gp, B, H1, W1, 64, Hp, Wp, pt, plft, g_c1, bwp->bn_part + site, fp16, s);
                         }});
    bw->steps.back().wr = g_c1;
    add_mask(h, bw.get(), g_c1, c1, B * H1 * W1, 64, &L, nullptr, site, rows);
    WgradParams wp;
    if ((rc = make_conv1_wgrad_params(h, g_c1, pl->s2d, B, H1, W1, pl->Hs, pl->Ws, &wp))) return rc;
    if ((rc = add_wgrad_params(h, bw.get(), wp, g_c1, L.scale, h->conv1_mask.get<float>(), ts->grads.get<float>() + L.w_off,
                               &ws_need, &L)))
      return rc;
  }
  // ---- every channel's dbeta / dgamma in one pass at the end
  {
    if ((rc = alloc_buf(h, &bw->bufs, bw->bn_part_floats * sizeof(float) + 1024, &p))) return rc;
    bw->bn_part = (float*)p;
    if ((rc = alloc_buf(h, &bw->bufs, (h->n_w / 4 + 64) * sizeof(float), &p))) return rc;
    bw->rowdot = (float*)p;
    if ((rc = alloc_buf(h, &bw->bufs, bw->bn_groups.size() * sizeof(BnGroup), &p))) return rc;
    bw->bn_table = (BnGroup*)p;
    for (const BnGroup& g : bw->bn_groups)
      if (g.rows <= 0 || g.K4 <= 0) return fail(h, DGP_ERR_STATE, "backward plan: a BatchNorm channel group has no gradient source");
    CU_OK(h, cudaMemcpy(bw->bn_table, bw->bn_groups.data(), bw->bn_groups.size() * sizeof(BnGroup), cudaMemcpyHostToDevice));
    const int ngroups = (int)bw->bn_groups.size();
    Backward* bwp = bw.get();
    const float *mean = h->bn_mean.get<float>(), *var = h->bn_var.get<float>();
    const float eps = h->cfg.bn_epsilon;
    float* dgam = ts->grads.get<float>() + h->n_w;
    float* dbet = ts->grads.get<float>() + h->n_w + h->n_ch;
    const GradMode* mode = ts->grad_mode.get<GradMode>();
    bw->steps.push_back({7, 1, [=](cudaStream_t s) {
                           return launch_bn_finalize_all(bwp->bn_table, ngroups, bwp->bn_part, bwp->rowdot, mean, var, eps, dgam, dbet,
                                                         mode, s);
                         }});
    bw->steps.back().join = true;
  }
  const void *p0 = ts->wgrad_ws.get(), *p1 = ts->bn_partial.get();
  if ((rc = ensure(h, &ts->wgrad_ws, ws_need))) return rc;
  if ((rc = ensure(h, &ts->bn_partial, bn_need))) return rc;
  if (p0 != ts->wgrad_ws.get() || p1 != ts->bn_partial.get()) ++ts->ws_gen;
  for (const BStep& st : bw->steps) bw->launches += st.launches;
  pl->bwd = bw;
  return DGP_OK;
}

// Stores the arena write mode the backward kernels read (GradMode) on `s`, when it differs from the stored one.
int set_grad_mode(dgp_handle* h, int accumulate, float out_scale, cudaStream_t s) {
  TrainState* ts = h->train.get();
  if (ts->grad_mode_host.accumulate == accumulate && ts->grad_mode_host.out_scale == out_scale) return DGP_OK;
  ts->grad_mode_host.accumulate = accumulate;
  ts->grad_mode_host.out_scale = out_scale;
  CU_OK(h, cudaMemcpyAsync(ts->grad_mode.get(), &ts->grad_mode_host, sizeof(GradMode), cudaMemcpyHostToDevice, s));
  return DGP_OK;
}

// A change of the weights makes every outstanding dgp_train_forward token stale.
void drop_train_tokens(dgp_handle* h) {
  for (auto& kv : h->train_plans) kv.second->fwd_token = 0;
}

// Loss scaling of the head gradients before the network backward (dgp_train_set_loss_scale).
int scale_head_grads(dgp_handle* h, const Plan* pl, Backward* bw, cudaStream_t s) {
  const float ls = h->train->loss_scale;
  if (ls == 1.0f) return DGP_OK;
  const size_t n = (size_t)pl->B * 4 * pl->hf * pl->wf * h->cfg.num_joints;
  CU_OK(h, launch_scale_inplace(bw->g_logits, n, ls, s));
  if (bw->g_locref) CU_OK(h, launch_scale_inplace(bw->g_locref, 2 * n, ls, s));
  h->launches += bw->g_locref ? 2 : 1;
  return DGP_OK;
}

// The network backward of `bw` from its g_logits / g_locref: eager on the first run of a plan, a captured graph afterwards.
int run_backward(dgp_handle* h, Backward* bw, cudaStream_t s) {
  TrainState* ts = h->train.get();
  const bool graphs = !h->profiling && bw->runs > 0;
  if (graphs && (!bw->graph_exec || bw->graph_gen != ts->ws_gen)) {
    // (re)capture on the handle's private stream; the first step ran eagerly, so every lazy cudaFuncSetAttribute is done
    bw->graph_exec.reset();
    cudaStream_t hs = h->stream.get();
    CU_OK(h, cudaStreamBeginCapture(hs, cudaStreamCaptureModeThreadLocal));
    // Two branches: the wgrad GEMMs only read a gradient buffer that the dgrad chain has finished writing, and nothing
    // downstream of them is needed before the end of the pass (or the bucket boundaries of the data-parallel all-reduce), so
    // they are captured on a side stream forked from the main branch.  A wgrad of blocks 2-3 is a short kernel (a few k-blocks
    // per CTA after the split over pixel ranges, then a latency-bound reduce): as a parallel branch its launch latency, ramp and
    // tail hide under the dgrad GEMMs instead of being serialised between them.  Joins: before a main-branch step that
    // overwrites the buffer a pending wgrad reads, before every bucket event, before the final gamma/beta pass.
    cudaError_t ce = cudaSuccess;
    if (!ts->side_stream) ce = create(&ts->side_stream, cudaStreamNonBlocking);
    cudaStream_t ss = ts->side_stream.get();
    size_t ev_next = 0;
    auto next_event = [&](cudaEvent_t* out) -> cudaError_t {
      if (ev_next == ts->branch_events.size()) {
        Event e;
        cudaError_t r = create(&e, cudaEventDisableTiming);
        if (r != cudaSuccess) return r;
        ts->branch_events.push_back(std::move(e));
      }
      *out = ts->branch_events[ev_next++].get();
      return cudaSuccess;
    };
    struct Pending { const void* rd; cudaEvent_t done; };
    std::vector<Pending> pending;   // in side-stream order: waiting for entry i covers entries 0..i
    auto join_through = [&](size_t i) -> cudaError_t {
      cudaError_t r = cudaStreamWaitEvent(hs, pending[i].done, 0);
      pending.erase(pending.begin(), pending.begin() + i + 1);
      return r;
    };
    int k = 0;
    for (const BStep& st : bw->steps) {
      if (ce != cudaSuccess) break;
      if (st.kind == 6 && st.rd != nullptr) {
        cudaEvent_t fork = nullptr, done = nullptr;
        if ((ce = next_event(&fork)) != cudaSuccess || (ce = next_event(&done)) != cudaSuccess) break;
        if ((ce = cudaEventRecord(fork, hs)) != cudaSuccess) break;
        if ((ce = cudaStreamWaitEvent(ss, fork, 0)) != cudaSuccess) break;
        if ((ce = st.run(ss)) != cudaSuccess) break;
        if ((ce = cudaEventRecord(done, ss)) != cudaSuccess) break;
        pending.push_back({st.rd, done});
      } else {
        if (st.join && !pending.empty()) ce = join_through(pending.size() - 1);
        if (ce == cudaSuccess && st.wr != nullptr)
          for (size_t i = pending.size(); i-- > 0;)
            if (pending[i].rd == st.wr) { ce = join_through(i); break; }
        if (ce == cudaSuccess) ce = st.run(hs);
        if (ce != cudaSuccess) break;
      }
      ++k;
      const bool boundary = k == bw->bucket_step[0] || k == bw->bucket_step[1] || k == bw->bucket_step[2];
      if (boundary && !pending.empty() && (ce = join_through(pending.size() - 1)) != cudaSuccess) break;
      for (int b = 0; b < 3 && ce == cudaSuccess; ++b)
        if (k == bw->bucket_step[b]) ce = cudaEventRecordWithFlags(ts->ev_bucket[b].get(), hs, cudaEventRecordExternal);
      if (ce != cudaSuccess) break;
    }
    if (!pending.empty()) {
      cudaError_t je = join_through(pending.size() - 1);   // every forked branch rejoins before the capture ends
      if (ce == cudaSuccess) ce = je;
    }
    cudaGraph_t g = nullptr;
    cudaError_t ee = cudaStreamEndCapture(hs, &g);
    Graph graph;
    if (g) adopt(&graph, g);
    if (ce == cudaSuccess) ce = ee;
    cudaGraphExec_t exec = nullptr;
    if (ce == cudaSuccess) ce = cudaGraphInstantiate(&exec, g, 0);
    if (ce != cudaSuccess) {
      cudaGetLastError();
      return fail(h, DGP_ERR_CUDA, "capturing the backward graph failed: %s", cudaGetErrorString(ce));
    }
    adopt(&bw->graph_exec, exec);
    bw->graph_gen = ts->ws_gen;
  }
  if (graphs) {
    CU_OK(h, cudaGraphLaunch(bw->graph_exec.get(), s));
    h->launches += bw->launches;
  } else {
    int k = 0;
    for (const BStep& st : bw->steps) {
      {
        ProfScope prof(h, st.kind, s);
        CU_OK(h, st.run(s));
      }
      h->launches += st.launches;
      ++k;
      for (int b = 0; b < 3; ++b)
        if (k == bw->bucket_step[b]) CU_OK(h, cudaEventRecord(ts->ev_bucket[b].get(), s));
    }
  }
  ts->bwd_ran = bw->bucket_step[0] > 0;
  bw->runs++;
  return DGP_OK;
}

}  // namespace

float* variable_arena(dgp_handle* h, int what, float* unscale) {
  *unscale = what == 1 ? 1.0f / h->train->arena_scale : 1.0f;
  return (what == 0 ? h->master : (what == 1 ? h->train->grads : h->train->accum)).get<float>();
}

void weights_changed(dgp_handle* h) {
  drop_train_tokens(h);
  if (h->train) h->train->wd_fresh = false;
}

}  // namespace dgp

extern "C" {

int dgp_train_enable(dgp_handle* h) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->finalized) return fail(h, DGP_ERR_STATE, "dgp_train_enable before dgp_finalize_weights");
  if (h->train) return DGP_OK;
  CU_OK(h, cudaSetDevice(h->device));
  std::unique_ptr<TrainState, TrainStateDeleter> ts(new TrainState());
  CU_OK(h, ts->grads.alloc(h->n_params * sizeof(float)));
  CU_OK(h, ts->accum.alloc(h->n_params * sizeof(float)));
  CU_OK(h, cudaMemset(ts->grads.get(), 0, h->n_params * sizeof(float)));
  CU_OK(h, cudaMemset(ts->accum.get(), 0, h->n_params * sizeof(float)));
  CU_OK(h, ts->norm_partial.alloc(sqnorm_partials() * sizeof(float)));
  CU_OK(h, ts->norm_clip.alloc(2 * sizeof(float)));
  CU_OK(h, cudaMemset(ts->norm_clip.get(), 0, 2 * sizeof(float)));
  CU_OK(h, ts->grad_mode.alloc(sizeof(GradMode)));
  CU_OK(h, cudaMemcpy(ts->grad_mode.get(), &ts->grad_mode_host, sizeof(GradMode), cudaMemcpyHostToDevice));
  ts->wd.resize(h->layers.size());
  std::vector<DgradWJob> jobs;
  for (size_t i = 0; i < h->layers.size(); ++i) {
    if ((int)i == h->conv1_layer || (int)i == h->head_layer) continue;
    const ConvLayer& L = h->layers[i];
    if (L.Cin % 32 || L.Cout % 32 || L.ch_off < 0) return fail(h, DGP_ERR_UNSUPPORTED, "%s: dgrad operand needs 32-aligned channels", L.scope.c_str());
    CU_OK(h, ts->wd[i].alloc((size_t)L.Cin * L.R * L.S * L.Cout * sizeof(W16)));
    DgradWJob jb;
    jb.w_off = L.w_off; jb.wd = ts->wd[i].get<uint16_t>(); jb.ch_off = L.ch_off;
    jb.Cout = L.Cout; jb.taps = L.R * L.S; jb.Cin = L.Cin; jb.tile_start = ts->wd_tiles;
    ts->wd_tiles += (L.Cin / 32) * (L.Cout / 32) * L.R * L.S;
    jobs.push_back(jb);
  }
  if (jobs.size() > (size_t)kDgradWMaxJobs)
    return fail(h, DGP_ERR_UNSUPPORTED, "%zu conv layers exceed the %d of the one-launch dgrad operand rebuild", jobs.size(),
                kDgradWMaxJobs);
  ts->n_wd_jobs = (int)jobs.size();
  CU_OK(h, ts->wd_jobs.alloc(jobs.size() * sizeof(DgradWJob)));
  CU_OK(h, cudaMemcpy(ts->wd_jobs.get(), jobs.data(), jobs.size() * sizeof(DgradWJob), cudaMemcpyHostToDevice));
  {
    // bucket k = the weight gradients of one block (k = 0: block4 + heads ... k = 3: conv1 + block1 + the BN / bias tail)
    const char* first[3] = {"/block4/unit_1/", "/block3/unit_1/", "/block2/unit_1/"};
    ts->bucket_off[0] = h->n_w;
    for (int k = 0; k < 3; ++k)
      for (const UnitDesc& u : h->units)
        if (u.scope.find(first[k]) != std::string::npos && u.shortcut >= 0) ts->bucket_off[k + 1] = h->layers[u.shortcut].w_off;
    ts->bucket_off[4] = 0;
    for (int k = 0; k < 3; ++k) CU_OK(h, create(&ts->ev_bucket[k], cudaEventDisableTiming));
    CU_OK(h, create(&ts->ev_bwd_done, cudaEventDefault));
    CU_OK(h, create(&ts->ev_comm_done, cudaEventDefault));
    CU_OK(h, create(&ts->comm_stream, cudaStreamNonBlocking));
  }
  ts->head_Kd = ceil_div(std::max(9 * h->ctot, h->layers[h->head_layer].Npad), 64) * 64;
  CU_OK(h, ts->head_wd.alloc((size_t)2048 * ts->head_Kd * sizeof(W16)));
  h->train = std::move(ts);
  return DGP_OK;
}

int dgp_train_forward_backward(dgp_handle* h, const uint8_t* frames_dev, int nt, int H, int W, const dgp_loss_cfg* cfg,
                               const dgp_loss_batch* batch, int visible_only, float* losses_dev, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->train) return fail(h, DGP_ERR_STATE, "dgp_train_forward_backward before dgp_train_enable");
  if (!frames_dev || !cfg || !batch || !losses_dev || nt < 1 || H < 32 || W < 32)
    return fail(h, DGP_ERR_INVALID, "dgp_train_forward_backward: bad argument");
  CU_OK(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  TrainState* ts = h->train.get();
  Plan* pl = nullptr;
  int rc = build_plan(h, nt, H, W, true, &pl);
  if (rc) return rc;
  if (!pl->bwd && (rc = build_backward(h, pl))) return rc;
  Backward* bw = static_cast<Backward*>(pl->bwd.get());
  if (batch->nt != nt || batch->H != 2 * pl->hf || batch->W != 2 * pl->wf)
    return fail(h, DGP_ERR_INVALID, "dgp_train_forward_backward: batch dims (%d,%d,%d) do not match the network output (%d,%d,%d)",
                batch->nt, batch->H, batch->W, nt, 2 * pl->hf, 2 * pl->wf);
  if (!ts->wd_fresh && (rc = refresh_dgrad_weights(h, s))) return rc;
  pl->fwd_token = 0;   // the activations are this step's from here on
  if ((rc = run_forward_plan(h, pl, frames_dev, pl->logits, pl->locref, s))) return rc;
  dgp_loss_batch b = *batch;
  b.pred_dev = pl->logits;
  b.locref_dev = pl->locref;
  if ((rc = dgp_run_loss_impl(h, cfg, &b, losses_dev, nullptr, bw->g_logits, bw->g_locref, visible_only, stream))) return rc;
  if ((rc = scale_head_grads(h, pl, bw, s))) return rc;
  if ((rc = set_grad_mode(h, 0, 1.0f, s))) return rc;
  if ((rc = run_backward(h, bw, s))) return rc;
  ts->arena_scale = ts->loss_scale;
  ts->arena_fused = true;
  return DGP_OK;
}

int dgp_train_forward(dgp_handle* h, const uint8_t* frames_dev, int nt, int H, int W, float* logits_dev, float* locref_dev,
                      uint64_t* token, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->train) return fail(h, DGP_ERR_STATE, "dgp_train_forward before dgp_train_enable");
  if (!frames_dev || !logits_dev || !token || nt < 1 || H < 32 || W < 32)
    return fail(h, DGP_ERR_INVALID, "dgp_train_forward: bad argument");
  if (locref_dev && !h->cfg.location_refinement)
    return fail(h, DGP_ERR_INVALID, "dgp_train_forward: locref_dev given but the network has no locref head");
  CU_OK(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  TrainState* ts = h->train.get();
  Plan* pl = nullptr;
  int rc = build_plan(h, nt, H, W, true, &pl);
  if (rc) return rc;
  if (!pl->bwd && (rc = build_backward(h, pl))) return rc;
  if (!ts->wd_fresh && (rc = refresh_dgrad_weights(h, s))) return rc;
  pl->fwd_token = 0;
  // the head GEMM's col2im writes straight into the caller's buffers; the backward needs only the kept activations
  if ((rc = run_forward_plan(h, pl, frames_dev, logits_dev, locref_dev, s))) return rc;
  pl->fwd_token = ++ts->fwd_seq;
  *token = pl->fwd_token;
  return DGP_OK;
}

int dgp_train_backward(dgp_handle* h, uint64_t token, const float* g_logits_dev, const float* g_locref_dev, int accumulate,
                       void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->train) return fail(h, DGP_ERR_STATE, "dgp_train_backward before dgp_train_enable");
  TrainState* ts = h->train.get();
  Plan* pl = nullptr;
  for (auto& kv : h->train_plans)
    if (token != 0 && kv.second->fwd_token == token) pl = kv.second.get();
  if (!pl)
    return fail(h, DGP_ERR_STATE, "dgp_train_backward: stale token (a later training forward of this shape, a plan eviction or a "
                                  "weight change has overwritten the activations of that forward)");
  Backward* bw = static_cast<Backward*>(pl->bwd.get());
  if (g_locref_dev && !bw->g_locref)
    return fail(h, DGP_ERR_INVALID, "dgp_train_backward: g_locref_dev given but the network has no locref head");
  if (accumulate && ts->arena_fused)
    return fail(h, DGP_ERR_STATE, "dgp_train_backward: cannot accumulate onto the loss-scaled gradients of dgp_train_forward_backward");
  CU_OK(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)pl->B * 4 * pl->hf * pl->wf * h->cfg.num_joints;
  if (g_logits_dev) CU_OK(h, cudaMemcpyAsync(bw->g_logits, g_logits_dev, n * sizeof(float), cudaMemcpyDeviceToDevice, s));
  else CU_OK(h, cudaMemsetAsync(bw->g_logits, 0, n * sizeof(float), s));
  if (bw->g_locref) {
    if (g_locref_dev) CU_OK(h, cudaMemcpyAsync(bw->g_locref, g_locref_dev, 2 * n * sizeof(float), cudaMemcpyDeviceToDevice, s));
    else CU_OK(h, cudaMemsetAsync(bw->g_locref, 0, 2 * n * sizeof(float), s));
  }
  int rc;
  if ((rc = scale_head_grads(h, pl, bw, s))) return rc;
  // the loss scale is divided out again as the finished gradients are stored: the arena holds the true gradient
  if ((rc = set_grad_mode(h, accumulate ? 1 : 0, 1.0f / ts->loss_scale, s))) return rc;
  if ((rc = run_backward(h, bw, s))) return rc;
  ts->arena_scale = 1.0f;
  ts->arena_fused = false;
  return DGP_OK;
}

int dgp_optimizer_step(dgp_handle* h, float lr, float momentum, float clip_norm, float grad_scale, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->train) return fail(h, DGP_ERR_STATE, "dgp_optimizer_step before dgp_train_enable");
  CU_OK(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  TrainState* ts = h->train.get();
  grad_scale /= ts->arena_scale;  // the buffer holds arena_scale * gradient
  float *grads = ts->grads.get<float>(), *norm_clip = ts->norm_clip.get<float>();
  CU_OK(h, launch_global_norm(grads, h->n_params, grad_scale, clip_norm, ts->norm_partial.get<float>(), norm_clip, s));
  CU_OK(h, launch_momentum_step(h->master.get<float>(), ts->accum.get<float>(), grads, h->n_params, lr, momentum, grad_scale,
                                norm_clip, s));
  h->launches += 3;
  drop_train_tokens(h);
  int rc = refresh_operands(h, s);
  if (rc) return rc;
  return refresh_dgrad_weights(h, s);
}

int dgp_params_changed(dgp_handle* h, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->finalized) return fail(h, DGP_ERR_STATE, "dgp_params_changed before dgp_finalize_weights");
  CU_OK(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  drop_train_tokens(h);
  int rc = refresh_operands(h, s);
  if (rc || !h->train) return rc;
  return refresh_dgrad_weights(h, s);
}

int dgp_get_param_buffer(dgp_handle* h, void** dev_ptr, size_t* bytes) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->finalized) return fail(h, DGP_ERR_STATE, "dgp_get_param_buffer before dgp_finalize_weights");
  if (dev_ptr) *dev_ptr = h->master.get();
  if (bytes) *bytes = h->n_params * sizeof(float);
  return DGP_OK;
}

int dgp_train_set_loss_scale(dgp_handle* h, float loss_scale) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->train) return fail(h, DGP_ERR_STATE, "dgp_train_set_loss_scale before dgp_train_enable");
  if (!(loss_scale > 0.0f) || !isfinite(loss_scale)) return fail(h, DGP_ERR_INVALID, "dgp_train_set_loss_scale: scale must be positive and finite");
  h->train->loss_scale = loss_scale;
  return DGP_OK;
}

int dgp_get_grad_buffer(dgp_handle* h, void** dev_ptr, size_t* bytes) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->train) return fail(h, DGP_ERR_STATE, "dgp_get_grad_buffer before dgp_train_enable");
  if (dev_ptr) *dev_ptr = h->train->grads.get();
  if (bytes) *bytes = h->n_params * sizeof(float);
  return DGP_OK;
}

int dgp_get_grad_norm(dgp_handle* h, float* norm_host) {
  if (!h || !norm_host) return DGP_ERR_INVALID;
  if (!h->train) return fail(h, DGP_ERR_STATE, "dgp_get_grad_norm before dgp_train_enable");
  CU_OK(h, cudaSetDevice(h->device));
  CU_OK(h, cudaDeviceSynchronize());
  CU_OK(h, cudaMemcpy(norm_host, h->train->norm_clip.get(), sizeof(float), cudaMemcpyDeviceToHost));
  return DGP_OK;
}

int dgp_train_outputs(dgp_handle* h, int nt, int H, int W, float** logits_dev, float** locref_dev) {
  if (!h) return DGP_ERR_INVALID;
  auto it = h->train_plans.find(std::make_tuple(nt, H, W));
  if (it == h->train_plans.end()) return fail(h, DGP_ERR_STATE, "dgp_train_outputs: no training step has run at this shape");
  if (logits_dev) *logits_dev = it->second->logits;
  if (locref_dev) *locref_dev = it->second->locref;
  return DGP_OK;
}

// ---------------------------------------------------------------- data-parallel all-reduce inside the C ABI
#define NCCL_OK(h, expr)                                                                                       \
  do {                                                                                                         \
    int _r = (expr);                                                                                           \
    if (_r != 0) return fail(h, DGP_ERR_CUDA, "%s failed: %s", #expr, nccl::api().err_str(_r));                \
  } while (0)

int dgp_comm_unique_id(char* id128) {
  if (!id128) return DGP_ERR_INVALID;
  if (!nccl::api().ok) return fail(nullptr, DGP_ERR_UNSUPPORTED, "dgp_comm_unique_id: libnccl.so.2 could not be loaded");
  nccl::UniqueId id;
  const int r = nccl::api().get_unique_id(&id);
  if (r != 0) return fail(nullptr, DGP_ERR_CUDA, "ncclGetUniqueId failed: %s", nccl::api().err_str(r));
  memcpy(id128, id.internal, 128);
  return DGP_OK;
}

int dgp_comm_init_rank(dgp_handle* h, const char* id128, int nranks, int rank) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->train) return fail(h, DGP_ERR_STATE, "dgp_comm_init_rank before dgp_train_enable");
  if (!id128 || nranks < 1 || rank < 0 || rank >= nranks) return fail(h, DGP_ERR_INVALID, "dgp_comm_init_rank: bad argument");
  if (!nccl::api().ok) return fail(h, DGP_ERR_UNSUPPORTED, "dgp_comm_init_rank: libnccl.so.2 could not be loaded");
  CU_OK(h, cudaSetDevice(h->device));
  h->train->release_comm();
  nccl::UniqueId id;
  memcpy(id.internal, id128, 128);
  void* comm = nullptr;
  NCCL_OK(h, nccl::api().comm_init_rank(&comm, nranks, id, rank));
  h->train->comm = comm;
  h->train->comm_owned = true;
  h->train->comm_world = nranks;
  return DGP_OK;
}

int dgp_attach_comm(dgp_handle* h, void* nccl_comm) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->train) return fail(h, DGP_ERR_STATE, "dgp_attach_comm before dgp_train_enable");
  h->train->release_comm();
  if (!nccl_comm) return DGP_OK;   // detach
  if (!nccl::api().ok) return fail(h, DGP_ERR_UNSUPPORTED, "dgp_attach_comm: libnccl.so.2 could not be loaded");
  int n = 0;
  NCCL_OK(h, nccl::api().comm_count(nccl_comm, &n));
  h->train->comm = nccl_comm;
  h->train->comm_owned = false;
  h->train->comm_world = n;
  return DGP_OK;
}

int dgp_comm_world_size(dgp_handle* h) { return (h && h->train && h->train->comm) ? h->train->comm_world : 1; }

int dgp_allreduce_gradients(dgp_handle* h, void* stream, float* grad_scale) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->train) return fail(h, DGP_ERR_STATE, "dgp_allreduce_gradients before dgp_train_enable");
  TrainState* ts = h->train.get();
  if (grad_scale) *grad_scale = 1.0f / (float)ts->comm_world;
  if (!ts->comm || ts->comm_world == 1) return DGP_OK;
  if (!ts->bwd_ran) return fail(h, DGP_ERR_STATE, "dgp_allreduce_gradients: no backward pass has run");
  CU_OK(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream, cs = ts->comm_stream.get();
  const nccl::Api& nc = nccl::api();
  float* grads = ts->grads.get<float>();
  CU_OK(h, cudaEventRecord(ts->ev_bwd_done.get(), s));                    // the end of the backward on the caller's stream
  for (int k = 0; k < 3; ++k) {                                      // buckets that were final before the backward ended
    const size_t lo = ts->bucket_off[k + 1], hi = ts->bucket_off[k];
    if (hi <= lo) continue;
    CU_OK(h, cudaStreamWaitEvent(cs, ts->ev_bucket[k].get(), 0));
    NCCL_OK(h, nc.all_reduce(grads + lo, grads + lo, hi - lo, nccl::kFloat, nccl::kSum, ts->comm, cs));
  }
  CU_OK(h, cudaStreamWaitEvent(cs, ts->ev_bwd_done.get(), 0));       // conv1 + block1 weights, then gamma / beta / head bias
  NCCL_OK(h, nc.group_start());
  if (ts->bucket_off[3] > 0)
    NCCL_OK(h, nc.all_reduce(grads, grads, ts->bucket_off[3], nccl::kFloat, nccl::kSum, ts->comm, cs));
  NCCL_OK(h, nc.all_reduce(grads + h->n_w, grads + h->n_w, h->n_params - h->n_w, nccl::kFloat, nccl::kSum, ts->comm, cs));
  NCCL_OK(h, nc.group_end());
  CU_OK(h, cudaEventRecord(ts->ev_comm_done.get(), cs));
  CU_OK(h, cudaStreamWaitEvent(s, ts->ev_comm_done.get(), 0));       // the optimizer step on `s` follows the reduced gradients
  return DGP_OK;
}

int dgp_allreduce_exposed_ms(dgp_handle* h, float* ms) {
  if (!h || !ms) return DGP_ERR_INVALID;
  if (!h->train) return fail(h, DGP_ERR_STATE, "dgp_allreduce_exposed_ms before dgp_train_enable");
  *ms = 0.0f;
  if (!h->train->comm || h->train->comm_world == 1) return DGP_OK;
  CU_OK(h, cudaSetDevice(h->device));
  CU_OK(h, cudaEventSynchronize(h->train->ev_comm_done.get()));
  CU_OK(h, cudaEventElapsedTime(ms, h->train->ev_bwd_done.get(), h->train->ev_comm_done.get()));
  return DGP_OK;
}

}  // extern "C"
