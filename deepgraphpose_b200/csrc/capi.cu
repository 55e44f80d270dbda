// libdgp_b200.so -- handle, weight loading, per-shape execution plans and the C ABI of include/dgp_b200.h.
#include "../../include/dgp_b200.h"

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include "handle.cuh"

using namespace dgp;

namespace dgp {

char g_create_error[512] = "";
std::atomic<int64_t> g_live_objects{0}, g_live_device_bytes{0};


W16 cvt16(const dgp_handle* h, float f) {
  W16 out;
  if (h->fp16) {
    const float c = f > 65504.0f ? 65504.0f : (f < -65504.0f ? -65504.0f : f);
    __half v = __float2half_rn(c);
    memcpy(&out, &v, 2);
  } else {
    out = __float2bfloat16_rn(f);
  }
  return out;
}
float cvt16_to_float(const dgp_handle* h, W16 v) {
  if (h->fp16) {
    __half x;
    memcpy(&x, &v, 2);
    return __half2float(x);
  }
  return __bfloat162float(v);
}

int fail(dgp_handle* h, int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(h ? h->err : g_create_error, 512, fmt, ap);
  va_end(ap);
  return code;
}


int ceil_div(int a, int b) { return (a + b - 1) / b; }

void same_pad(int in, int k, int stride, int rate, int* beg, int* out) {
  const int o = ceil_div(in, stride);
  const int keff = (k - 1) * rate + 1;
  int total = (o - 1) * stride + keff - in;
  if (total < 0) total = 0;
  *beg = total / 2;
  *out = o;
}

int pick_block_n(int n) {
  // largest UMMA N (multiple of 16, <= 256) that tiles n with the least padding
  const int nb = ceil_div(n, 256);
  int bn = ceil_div(ceil_div(n, nb), 16) * 16;
  if (bn > 256) bn = 256;
  return bn;
}

int tmem_cols_for(int block_n) {
  int need = 2 * block_n, c = 32;
  while (c < need) c <<= 1;
  return c;
}

const HostVar* find_var(dgp_handle* h, const std::string& name) {
  auto it = h->host_vars.find(name);
  return it == h->host_vars.end() ? nullptr : &it->second;
}

// master fp32 -> 16-bit GEMM operands + BN scale/shift (after loading and after every optimizer step)
int refresh_operands(dgp_handle* h, cudaStream_t s) {
  const float* master = h->master.get<float>();
  float* bn_ss = h->bn_ss.get<float>();
  CU_OK(h, launch_refresh_w16(master, h->w16.get<W16>(), h->n_w, h->fp16, s));
  CU_OK(h, launch_refresh_bn(master + h->n_w, master + h->n_w + h->n_ch, h->bn_mean.get<float>(), h->bn_var.get<float>(),
                             h->cfg.bn_epsilon, (int)h->n_ch, bn_ss, bn_ss + h->n_ch, s));
  h->launches += 2;
  return DGP_OK;
}

// Frozen batch norm (slim batch_norm, is_training=False): gamma / beta are trainable and live in the parameter arena,
// the moving statistics are constants; the fp32 scale/shift applied in the GEMM epilogue are derived on the device
// (refresh_bn_kernel), never folded into the 16-bit weights.  A missing gamma is slim's default scale, 1.
int append_bn(dgp_handle* h, const std::string& scope, int C, int* ch_off) {
  const std::string bn = scope + "/BatchNorm/";
  if (!find_var(h, bn + "beta") || !find_var(h, bn + "moving_mean") || !find_var(h, bn + "moving_variance"))
    return fail(h, DGP_ERR_STATE, "missing BatchNorm variables for %s", scope.c_str());
  if (!find_var(h, bn + "gamma")) h->host_vars[bn + "gamma"] = HostVar{std::vector<float>(C, 1.0f), {C}};
  *ch_off = (int)h->n_ch;
  h->n_ch += C;
  return DGP_OK;
}

int build_conv_layer(dgp_handle* h, const std::string& scope, int R, int S, int Cin, int Cout, int stride, int dil,
                     bool relu, int* index) {
  if (!find_var(h, scope + "/weights")) return fail(h, DGP_ERR_STATE, "missing variable %s/weights", scope.c_str());
  if (Cin % 64 != 0 || Cout % 16 != 0) return fail(h, DGP_ERR_UNSUPPORTED, "%s: channels not tileable", scope.c_str());
  ConvLayer L;
  L.scope = scope; L.R = R; L.S = S; L.Cin = Cin; L.Cout = Cout; L.stride = stride; L.dil = dil; L.relu = relu;
  L.K = R * S * Cin;
  L.block_n = Cout >= 256 ? 256 : Cout;
  L.Npad = Cout;
  L.w_off = h->n_w;
  h->n_w += (size_t)Cout * L.K;
  int rc = append_bn(h, scope, Cout, &L.ch_off);
  if (rc) return rc;
  *index = (int)h->layers.size();
  h->layers.push_back(L);
  return DGP_OK;
}

// conv1: 7x7 stride 2 on 3 channels == 4x4 stride-1 conv on the 2x2 space-to-depth image (12 -> 16 channels);
// one TMA "pixel" is a window of 4 horizontally adjacent s2d pixels (64 channels), the 4 window rows are the taps.
int build_conv1_layer(dgp_handle* h) {
  const std::string scope = h->net_scope + "/conv1";
  if (!find_var(h, scope + "/weights")) return fail(h, DGP_ERR_STATE, "missing variable %s/weights", scope.c_str());
  ConvLayer L;
  L.scope = scope; L.R = 4; L.S = 1; L.Cin = 64; L.Cout = 64; L.stride = 1; L.dil = 1; L.relu = true;
  L.K = 256; L.block_n = 64; L.Npad = 64;
  L.w_off = h->n_w;
  h->n_w += (size_t)64 * 256;
  int rc = append_bn(h, scope, 64, &L.ch_off);
  if (rc) return rc;
  h->conv1_layer = (int)h->layers.size();
  h->layers.push_back(L);
  return DGP_OK;
}

// Both deconv heads as ONE GEMM over input pixels: column (kh*3+kw)*ctot + co, co = [part_pred | locref_pred].
int build_head_layer(dgp_handle* h) {
  const int nj = h->cfg.num_joints;
  const int ctot = h->cfg.location_refinement ? 3 * nj : nj;
  if (!find_var(h, "pose/part_pred/block4/weights") || !find_var(h, "pose/part_pred/block4/biases"))
    return fail(h, DGP_ERR_STATE, "missing pose/part_pred/block4 variables");
  if (h->cfg.location_refinement &&
      (!find_var(h, "pose/locref_pred/block4/weights") || !find_var(h, "pose/locref_pred/block4/biases")))
    return fail(h, DGP_ERR_STATE, "missing pose/locref_pred/block4 variables");
  ConvLayer L;
  L.scope = "pose/heads"; L.R = 1; L.S = 1; L.Cin = 2048; L.Cout = 9 * ctot; L.relu = false;
  L.K = 2048;
  L.block_n = pick_block_n(9 * ctot);
  L.Npad = ceil_div(9 * ctot, L.block_n) * L.block_n;
  L.w_off = h->n_w;
  h->n_w += (size_t)L.Npad * 2048;
  h->n_bias = (size_t)ceil_div(ctot, 8) * 8;
  h->ctot = ctot;
  h->head_layer = (int)h->layers.size();
  h->layers.push_back(L);
  return DGP_OK;
}

// Checks every loaded variable of `vars` against its TF shape and packs it into its span of `base`.
int pack_loaded(dgp_handle* h, const std::vector<ArenaVar>& vars, float* base) {
  for (const ArenaVar& v : vars) {
    const HostVar* x = find_var(h, v.name);  // present: the layer walk checked every name
    bool same = x && (int)x->shape.size() == v.ndim;
    for (int i = 0; same && i < v.ndim; ++i) same = x->shape[i] == v.shape[i];
    if (!same) return fail(h, DGP_ERR_INVALID, "%s has the wrong shape (want %s)", v.name.c_str(), shape_str(v).c_str());
    pack(v, x->data.data(), base + v.off);
  }
  return DGP_OK;
}

// Packs the loaded variables into the parameter arena [weights | gamma | beta | head bias] (fp32 master copy) and the
// frozen moving statistics, uploads both and derives the tensor-core operands on the device.
int upload_arena(dgp_handle* h) {
  h->n_params = h->n_w + 2 * h->n_ch + h->n_bias;
  if (h->n_w % 8 || h->n_ch % 4) return fail(h, DGP_ERR_STATE, "parameter arena is not vector aligned");
  std::vector<ArenaVar> frozen;
  build_variable_table(h, &frozen);
  std::vector<float> arena(h->n_params, 0.0f), stats(2 * h->n_ch);  // stats: [moving_mean | moving_variance]
  int rc;
  if ((rc = pack_loaded(h, h->vars, arena.data())) || (rc = pack_loaded(h, frozen, stats.data()))) return rc;
  const ArenaVar& conv1 = h->vars[h->var_index[h->net_scope + "/conv1/weights"]];
  std::vector<float> ones(tf_elems(conv1), 1.0f), mask(conv1.len, 0.0f);
  pack(conv1, ones.data(), mask.data());
  CU_OK(h, h->master.alloc(h->n_params * sizeof(float)));
  CU_OK(h, h->w16.alloc(h->n_w * sizeof(W16)));
  CU_OK(h, h->bn_mean.alloc(h->n_ch * sizeof(float)));
  CU_OK(h, h->bn_var.alloc(h->n_ch * sizeof(float)));
  CU_OK(h, h->bn_ss.alloc(2 * h->n_ch * sizeof(float)));
  CU_OK(h, h->conv1_mask.alloc(mask.size() * sizeof(float)));
  float* master = h->master.get<float>();
  CU_OK(h, cudaMemcpy(master, arena.data(), h->n_params * 4, cudaMemcpyHostToDevice));
  CU_OK(h, cudaMemcpy(h->bn_mean.get(), stats.data(), h->n_ch * 4, cudaMemcpyHostToDevice));
  CU_OK(h, cudaMemcpy(h->bn_var.get(), stats.data() + h->n_ch, h->n_ch * 4, cudaMemcpyHostToDevice));
  CU_OK(h, cudaMemcpy(h->conv1_mask.get(), mask.data(), mask.size() * 4, cudaMemcpyHostToDevice));
  float* bn_ss = h->bn_ss.get<float>();
  for (ConvLayer& L : h->layers) {
    L.w = h->w16.get<W16>() + L.w_off;
    if (L.ch_off >= 0) {
      L.scale = bn_ss + L.ch_off;
      L.shift = bn_ss + h->n_ch + L.ch_off;
    }
  }
  h->head_bias = master + h->n_w + 2 * h->n_ch;
  if ((rc = refresh_operands(h, nullptr))) return rc;
  CU_OK(h, cudaDeviceSynchronize());
  return DGP_OK;
}

int alloc_buf(dgp_handle* h, std::vector<DevBuf>* bufs, size_t bytes, void** out) {
  DevBuf b;
  CU_OK(h, b.alloc(bytes));
  *out = b.get();
  bufs->push_back(std::move(b));
  return DGP_OK;
}

// Staging buffers per epilogue warp (2 KB each, 16 warps): the residual prefetch runs epi_bufs-1 units ahead.
int epi_bufs_for(bool residual, int block_n) {
  // 64-wide layers (256-row tiles, one unit per warp and tile): a single buffer leaves room for a fourth smem stage
  return (!residual && block_n == 64) ? 1 : 2;
}

// Epilogue configuration: bf16 outputs whose tile width is a multiple of 64 go through the TMA-staged epilogue
// (TMA store of the output, TMA load of the residual); everything else uses direct register->global stores.
int setup_epilogue(dgp_handle* h, ConvGemmParams& g, const char* scope, int n_img) {
  const bool staged = !g.out_f32 && (g.block_n == 64 || g.block_n == 128 || g.block_n == 256);
  if (!staged) {
    if (g.residual) return fail(h, DGP_ERR_UNSUPPORTED, "%s: residual needs a 16-bit output with block_n 64, 128 or 256", scope);
    g.epi_mode = 0;
    g.epi_bufs = 0;
  } else {
    g.epi_mode = 1;
    g.epi_bufs = epi_bufs_for(g.residual != nullptr, g.block_n);
    const char* e = make_tmap_2d(&g.tmap_out, g.out, (uint64_t)g.M, (uint64_t)g.N, (uint64_t)g.ldc * 2, 32, kEpiUnitCols);
    if (e) return fail(h, DGP_ERR_CUDA, "%s (out map): %s", scope, e);
    if (g.residual) {
      if (g.res_sub == 1) {
        e = make_tmap_2d(&g.tmap_res, g.residual, (uint64_t)g.M, (uint64_t)g.N, (uint64_t)g.ldres * 2, 32, kEpiUnitCols);
      } else {
        e = make_tmap_im2col(&g.tmap_res, g.residual, (uint64_t)g.N, (uint64_t)g.res_W, (uint64_t)g.res_H, (uint64_t)n_img,
                             (uint64_t)g.ldres * 2, (uint64_t)g.res_W * g.ldres * 2,
                             (uint64_t)g.res_H * g.res_W * g.ldres * 2, 0, 0, 0, 0, g.res_sub,
                             (uint64_t)n_img * g.res_H * g.res_W * g.ldres * 2, 32, kEpiUnitCols);
      }
      if (e) return fail(h, DGP_ERR_CUDA, "%s (residual map): %s", scope, e);
    }
  }
  // narrow layers (N tile <= 128) run 256-row CTA tiles: one TMA + two UMMAs per k-step halves the per-k-block
  // issue overhead of the single-warp producer / MMA loops (see DESIGN.md "BLOCK_M = 256")
  g.msub = (g.epi_mode == 1 && g.block_n <= 128 && g.M > kBlockM) ? 2 : 1;
  // 256-wide tiles of big layers run as CTA pairs (cta_group::2): a single-CTA M=128 x N=256 MMA reads 12 KB of operands
  // from shared memory per K=16 step and is bound by that, the pair reads 8 KB per CTA.
  g.cta2 = (g.epi_mode == 1 && g.block_n == 256 && g.M >= 4 * kBlockM) ? 1 : 0;
  g.num_m_blocks = ceil_div(g.M, g.cta2 ? 2 * kBlockM : kBlockM * g.msub);
  g.tmem_cols = tmem_cols_for(g.block_n * g.msub);
  g.num_stages = conv_gemm_pick_stages(g);
  return DGP_OK;
}

// Output size and padding of one conv: pad_mode 0 = TF SAME, 1 = slim conv2d_same (explicit pad + VALID), 2 = VALID.
void conv_geometry(int R, int S, int stride, int dil, int H, int W, int pad_mode, int* Pout, int* Qout, int* lower_h_,
                   int* lower_w_, int* upper_h_, int* upper_w_) {
  int P, Q, lower_h = 0, lower_w = 0, upper_h = 0, upper_w = 0;
  const int keff_h = (R - 1) * dil + 1, keff_w = (S - 1) * dil + 1;
  if (pad_mode == 0) {  // TF SAME
    same_pad(H, R, stride, dil, &lower_h, &P);
    same_pad(W, S, stride, dil, &lower_w, &Q);
    const int tot_h = (P - 1) * stride + keff_h - H, tot_w = (Q - 1) * stride + keff_w - W;
    upper_h = (tot_h > 0 ? tot_h : 0) - lower_h;
    upper_w = (tot_w > 0 ? tot_w : 0) - lower_w;
  } else if (pad_mode == 1) {  // slim conv2d_same: explicit (keff-1) padding, beg = (keff-1)/2, then VALID
    if (stride == 1) {
      same_pad(H, R, 1, dil, &lower_h, &P);
      same_pad(W, S, 1, dil, &lower_w, &Q);
      upper_h = (keff_h - 1) - lower_h;
      upper_w = (keff_w - 1) - lower_w;
    } else {
      lower_h = (keff_h - 1) / 2; upper_h = (keff_h - 1) - lower_h;
      lower_w = (keff_w - 1) / 2; upper_w = (keff_w - 1) - lower_w;
      P = (H + keff_h - 1 - keff_h) / stride + 1;
      Q = (W + keff_w - 1 - keff_w) / stride + 1;
    }
  } else {  // VALID
    P = (H - keff_h) / stride + 1;
    Q = (W - keff_w) / stride + 1;
  }
  *Pout = P; *Qout = Q; *lower_h_ = lower_h; *lower_w_ = lower_w; *upper_h_ = upper_h; *upper_w_ = upper_w;
}

// Fill the GEMM params of one conv layer. x: input NHWC bf16 (N,H,W,Cin). Returns output dims via Ho/Wo.
int make_gemm_step(dgp_handle* h, const ConvLayer& L, const void* x, int N, int H, int W, int pad_mode, void* out,
                   bool out_f32, const __nv_bfloat16* residual, int res_sub, int res_H, int res_W, int block_n_override,
                   Step* st, int* Ho, int* Wo) {
  memset(&st->gp, 0, sizeof(st->gp));
  ConvGemmParams& g = st->gp;
  g.fp16 = h->fp16;
  tmap_set_fp16(h->fp16);
  int P, Q, lower_h = 0, lower_w = 0, upper_h = 0, upper_w = 0;
  conv_geometry(L.R, L.S, L.stride, L.dil, H, W, pad_mode, &P, &Q, &lower_h, &lower_w, &upper_h, &upper_w);
  *Ho = P;
  *Wo = Q;
  const int bn = block_n_override > 0 ? block_n_override : L.block_n;
  if (L.Npad % bn) return fail(h, DGP_ERR_INVALID, "%s: block_n %d does not divide N %d", L.scope.c_str(), bn, L.Npad);
  g.M = N * P * Q;
  g.N = L.Npad;
  g.block_n = bn;
  g.num_k_blocks = L.K / kBlockK;
  g.P = P; g.Q = Q;
  g.conv_stride = L.stride;
  g.lower_h = -lower_h; g.lower_w = -lower_w;
  g.S = L.S; g.dil = L.dil; g.cblocks = L.Cin / kBlockK;
  g.scale = L.scale; g.shift = L.shift;
  g.residual = residual; g.res_sub = res_sub; g.res_H = res_H; g.res_W = res_W; g.ldres = L.Npad;
  g.relu = L.relu ? 1 : 0;
  g.out = out; g.out_f32 = out_f32 ? 1 : 0; g.ldc = L.Npad;
  g.num_m_blocks = ceil_div(g.M, kBlockM);
  g.num_n_blocks = L.Npad / bn;
  g.tmem_cols = tmem_cols_for(bn);
  const char* e = nullptr;
  // 3x3 stride-1 convs over 64 channels (block 1 conv2 and its dgrad) run from a shared-memory resident input patch: the
  // im2col form re-reads every activation nine times from the L2 and is bound by the L2 -> SM fabric (~11 TB/s of
  // distinct lines), not by the tensor pipe.
  const bool patch = L.R == 3 && L.S == 3 && L.stride == 1 && L.Cin == 64 && bn == 64 && L.Npad == 64 && !out_f32 && !residual &&
                     lower_h == L.dil && lower_w == L.dil;
  if (patch) {
    g.a_mode = 3; g.epi_mode = 3; g.epi_bufs = 0; g.msub = 2;
    g.pt_rows = 14; g.pt_cols = 16;
    if (L.dil > 1) { g.pt_rows = 12; g.pt_cols = 16; }
    g.pt_wp = g.pt_cols + 2 * L.dil;
    while (g.pt_rows * g.pt_wp > 256) --g.pt_rows;
    g.pt_stage_bytes = conv_patch_stage_bytes(g.pt_wp, L.dil);
    g.pt_base_offset_mode = 0;  // measured: the UMMA swizzle is a function of the absolute smem address; base_offset stays 0
    g.pool_tiles_i = ceil_div(P, g.pt_rows); g.pool_tiles_j = ceil_div(Q, g.pt_cols);
    g.num_m_blocks = N * g.pool_tiles_i * g.pool_tiles_j;
    g.num_n_blocks = 1;
    g.tmem_cols = tmem_cols_for(bn * 2);
    g.num_stages = 2;
    if (conv_gemm_smem_bytes(g) > 227 * 1024) return fail(h, DGP_ERR_UNSUPPORTED, "%s: patch conv does not fit shared memory", L.scope.c_str());
    e = make_tmap_tiled4d(&g.tmap_a, x, 64, (uint64_t)W, (uint64_t)H, (uint64_t)N, 128, (uint64_t)W * 128, (uint64_t)H * W * 128,
                          (uint32_t)g.pt_wp, (uint32_t)(g.pt_rows + 2 * L.dil));
    if (e) return fail(h, DGP_ERR_CUDA, "%s: %s", L.scope.c_str(), e);
    e = make_tmap_2d(&g.tmap_b, L.w, (uint64_t)L.Npad, (uint64_t)L.K, (uint64_t)L.K * 2, (uint32_t)bn);
    if (e) return fail(h, DGP_ERR_CUDA, "%s: %s", L.scope.c_str(), e);
    st->kind = STEP_GEMM;
    st->out_ptr = out;
    st->oN = N; st->oH = P; st->oW = Q; st->oC = L.Npad;
    return DGP_OK;
  }
  if (int rc = setup_epilogue(h, g, L.scope.c_str(), N)) return rc;
  const bool pointwise = (L.R == 1 && L.S == 1 && L.stride == 1);
  if (pointwise) {
    g.a_mode = 0;
    e = make_tmap_2d(&g.tmap_a, x, (uint64_t)g.M, (uint64_t)L.K, (uint64_t)L.K * 2, kBlockM * g.msub);
  } else {
    g.a_mode = 1;
    const int up_h = upper_h - (L.R - 1) * L.dil, up_w = upper_w - (L.S - 1) * L.dil;
    e = make_tmap_im2col(&g.tmap_a, x, (uint64_t)L.Cin, (uint64_t)W, (uint64_t)H, (uint64_t)N, (uint64_t)L.Cin * 2,
                         (uint64_t)W * L.Cin * 2, (uint64_t)H * W * L.Cin * 2, -lower_w, -lower_h, up_w, up_h, L.stride,
                         (uint64_t)N * H * W * L.Cin * 2, kBlockM * g.msub);
  }
  if (e) return fail(h, DGP_ERR_CUDA, "%s: %s", L.scope.c_str(), e);
  e = make_tmap_2d(&g.tmap_b, L.w, (uint64_t)L.Npad, (uint64_t)L.K, (uint64_t)L.K * 2, (uint32_t)(g.cta2 ? bn / 2 : bn));
  if (e) return fail(h, DGP_ERR_CUDA, "%s: %s", L.scope.c_str(), e);
  st->kind = STEP_GEMM;
  st->out_ptr = out;
  st->oN = N; st->oH = P; st->oW = Q; st->oC = L.Npad;
  return DGP_OK;
}

// Weight-gradient GEMM params of one conv: x NHWC (N,H,W,Cin), dy (N,P,Q,Cout) 16-bit; the im2col geometry is the forward's.
int make_wgrad_params(dgp_handle* h, const char* scope, int R, int S, int Cin, int Cout, int stride, int dil,
                      const void* x, int N, int H, int W, int pad_mode, const void* dy, WgradParams* wp) {
  memset(wp, 0, sizeof(*wp));
  tmap_set_fp16(h->fp16);
  wp->fp16 = h->fp16;
  int P, Q, lower_h, lower_w, upper_h, upper_w;
  conv_geometry(R, S, stride, dil, H, W, pad_mode, &P, &Q, &lower_h, &lower_w, &upper_h, &upper_w);
  const int M = N * P * Q;
  wp->Cout = Cout; wp->Kw = R * S * Cin;
  wp->num_pix_blocks = ceil_div(M, 64);
  wp->P = P; wp->Q = Q; wp->conv_stride = stride; wp->lower_h = -lower_h; wp->lower_w = -lower_w;
  wp->S = S; wp->dil = dil; wp->cblocks = Cin / 64;
  const char* e = make_tmap_2d(&wp->tmap_dy, dy, (uint64_t)M, (uint64_t)Cout, (uint64_t)Cout * 2, 64);
  if (e) return fail(h, DGP_ERR_CUDA, "%s wgrad (dy map): %s", scope, e);
  if (R == 1 && S == 1 && stride == 1) {
    wp->x_mode = 0;
    e = make_tmap_2d(&wp->tmap_x, x, (uint64_t)M, (uint64_t)Cin, (uint64_t)Cin * 2, 64);
  } else {
    wp->x_mode = 1;
    const int up_h = upper_h - (R - 1) * dil, up_w = upper_w - (S - 1) * dil;
    e = make_tmap_im2col(&wp->tmap_x, x, (uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)N, (uint64_t)Cin * 2,
                         (uint64_t)W * Cin * 2, (uint64_t)H * W * Cin * 2, -lower_w, -lower_h, up_w, up_h, stride,
                         (uint64_t)N * H * W * Cin * 2, 64);
  }
  if (e) return fail(h, DGP_ERR_CUDA, "%s wgrad (x map): %s", scope, e);
  wgrad_plan(wp, h->num_sms);
  return DGP_OK;
}

// conv1's weight gradient in the space-to-depth form of build_conv1_layer: dy (B*H1*W1, 64) against the im2col view of s2d
// (B, Hs, Ws, 16) in which one 64-channel pixel is a window of 4 horizontally adjacent s2d pixels and the 4 window rows are
// the taps, exactly as the forward's conv1 map reads it.
int make_conv1_wgrad_params(dgp_handle* h, const void* dy, const void* s2d, int B, int H1, int W1, int Hs, int Ws,
                            WgradParams* wp) {
  memset(wp, 0, sizeof(*wp));
  tmap_set_fp16(h->fp16);
  wp->fp16 = h->fp16;
  const int M = B * H1 * W1;
  wp->Cout = 64; wp->Kw = 256; wp->num_pix_blocks = ceil_div(M, 64);
  wp->x_mode = 1; wp->P = H1; wp->Q = W1; wp->conv_stride = 1; wp->lower_h = 0; wp->lower_w = 0; wp->S = 1; wp->dil = 1;
  wp->cblocks = 1;
  const char* e = make_tmap_2d(&wp->tmap_dy, dy, (uint64_t)M, 64, 128, 64);
  if (e) return fail(h, DGP_ERR_CUDA, "conv1 wgrad (dy map): %s", e);
  e = make_tmap_im2col(&wp->tmap_x, s2d, 64, (uint64_t)W1, (uint64_t)Hs, (uint64_t)B, 32, (uint64_t)Ws * 32,
                       (uint64_t)Hs * Ws * 32, 0, 0, 0, -3, 1, (uint64_t)B * Hs * Ws * 32, 64);
  if (e) return fail(h, DGP_ERR_CUDA, "conv1 wgrad (x map): %s", e);
  wgrad_plan(wp, h->num_sms);
  return DGP_OK;
}

int keep_activation(dgp_handle* h, const Step& st, cudaStream_t s);

int build_plan(dgp_handle* h, int B, int H, int W, bool train, Plan** out) {
  // Inference plans run conv1 fused with pool1 (conv_gemm_kernel a_mode / epi_mode 2): conv1's output -- 20 MB per 747x832
  // frame, the largest tensor of the net -- never reaches HBM.  Training keeps it for the backward pass and debug runs
  // (dgp_debug_keep_activations) dump it: those plans (key -B for the debug one) run conv1 and the pool as two launches.
  const bool unfused = train || h->debug_keep;
  auto key = std::make_tuple((!train && h->debug_keep) ? -B : B, H, W);
  auto& plans = train ? h->train_plans : h->plans;
  auto it = plans.find(key);
  if (it != plans.end()) {
    it->second->last_use = ++h->plan_clock;
    *out = it->second.get();
    return DGP_OK;
  }
  // Plans own gigabytes of activation buffers: keep at most a handful per kind (fit_dgp's last batch of an epoch and
  // videos of different sizes create new shapes), dropping the least recently used one once the device is idle.
  const size_t max_plans = train ? 3 : 6;
  if (plans.size() >= max_plans) {
    CU_OK(h, cudaDeviceSynchronize());
    auto victim = plans.begin();
    for (auto jt = plans.begin(); jt != plans.end(); ++jt)
      if (jt->second->last_use < victim->second->last_use) victim = jt;
    plans.erase(victim);
  }
  std::unique_ptr<Plan> pl(new Plan());
  pl->last_use = ++h->plan_clock;
  pl->train = train;
  pl->B = B; pl->H = H; pl->W = W;
  pl->H1 = ceil_div(H, 2); pl->W1 = ceil_div(W, 2);
  pl->Hs = pl->H1 + 3; pl->Ws = pl->W1 + 3;
  int rc;
  void* p = nullptr;
  // ---- conv1 (s2d + windowed im2col GEMM)
  rc = alloc_buf(h, &pl->bufs, (size_t)B * pl->Hs * pl->Ws * 16 * 2, &p);
  if (rc) return rc;
  pl->s2d = (__nv_bfloat16*)p;
  {
    Step st; st.kind = STEP_PREP;
    pl->steps.push_back(st);
  }
  // ---- shape pre-pass: sizes of the rotating activation buffers
  size_t max_x = 0, max_t = 0, max_sc = 0;
  {
    int hh, ww, d;
    same_pad(pl->H1, 3, 2, 1, &d, &hh);
    same_pad(pl->W1, 3, 2, 1, &d, &ww);
    max_x = (size_t)hh * ww * 64;
    int cin = 64;
    for (const UnitDesc& u : h->units) {
      const int ho = ceil_div(hh, u.stride), wo = ceil_div(ww, u.stride);
      if ((size_t)hh * ww * u.base > max_t) max_t = (size_t)hh * ww * u.base;
      if (cin != u.depth && (size_t)hh * ww * u.depth > max_sc) max_sc = (size_t)hh * ww * u.depth;
      if ((size_t)ho * wo * u.depth > max_x) max_x = (size_t)ho * wo * u.depth;
      hh = ho; ww = wo; cin = u.depth;
    }
  }
  const size_t big = (size_t)B * pl->H1 * pl->W1 * 64 * 2;
  const size_t x_bytes = (size_t)B * max_x * 2 + 1024, t_bytes = (size_t)B * max_t * 2 + 1024,
               sc_bytes = (size_t)B * max_sc * 2 + 1024;
  void *c1 = nullptr, *xa = nullptr, *xb = nullptr, *t1 = nullptr, *t2 = nullptr, *sc = nullptr;
  if (unfused && (rc = alloc_buf(h, &pl->bufs, big, &c1))) return rc;
  int Hc, Wc, pad_t, pad_l;
  same_pad(pl->H1, 3, 2, 1, &pad_t, &Hc);
  same_pad(pl->W1, 3, 2, 1, &pad_l, &Wc);
  if (!train) {
    if ((rc = alloc_buf(h, &pl->bufs, x_bytes, &xa))) return rc;
    if ((rc = alloc_buf(h, &pl->bufs, x_bytes, &xb))) return rc;
    if ((rc = alloc_buf(h, &pl->bufs, sc_bytes, &sc))) return rc;
    if ((rc = alloc_buf(h, &pl->bufs, t_bytes, &t1))) return rc;
    if ((rc = alloc_buf(h, &pl->bufs, t_bytes, &t2))) return rc;
  } else {
    // training keeps every activation for the backward pass: each tensor gets its own buffer
    if ((rc = alloc_buf(h, &pl->bufs, (size_t)B * Hc * Wc * 64 * 2 + 1024, &xa))) return rc;
  }
  pl->c1 = c1; pl->pool = xa; pl->Hp = Hc; pl->Wp = Wc; pl->pool_pad_t = pad_t; pl->pool_pad_l = pad_l;
  {
    const ConvLayer& L = h->layers[h->conv1_layer];
    Step st;
    memset(&st.gp, 0, sizeof(st.gp));
    ConvGemmParams& g = st.gp;
    g.fp16 = h->fp16;
    tmap_set_fp16(h->fp16);
    g.M = B * pl->H1 * pl->W1; g.N = 64; g.block_n = 64; g.num_k_blocks = 4;
    g.P = pl->H1; g.Q = pl->W1; g.conv_stride = 1; g.lower_h = 0; g.lower_w = 0; g.S = 1; g.dil = 1; g.cblocks = 1;
    g.scale = L.scale; g.shift = L.shift; g.residual = nullptr; g.res_sub = 1; g.relu = 1;
    g.out_f32 = 0; g.ldc = 64; g.num_n_blocks = 1;
    uint32_t pixels_per_load;
    if (unfused) {
      g.a_mode = 1;
      g.out = c1;
      g.num_m_blocks = ceil_div(g.M, kBlockM);
      g.tmem_cols = tmem_cols_for(64);
      if ((rc = setup_epilogue(h, g, "conv1", B))) return rc;
      pixels_per_load = kBlockM * g.msub;
    } else {
      g.epi_mode = 2; g.epi_bufs = 0; g.msub = 2;
      g.out = xa;
      g.pool_H = Hc; g.pool_W = Wc; g.pool_pad_t = pad_t; g.pool_pad_l = pad_l;
      // a tile = the 15 x 17 patch of conv1 outputs (255 of the 256 accumulator rows) under 7 x 8 pooled pixels, loaded
      // per filter row as one tiled box of overlapping 4-pixel windows (10x read amplification out of the L2).  Measured
      // (profiles/r02_conv1_variants.md) against a since-removed variant that kept a patch of space-to-depth pixels resident
      // in shared memory: both are bound by the SM's shared-memory port, and the resident one needed 20 % more tiles.
      g.a_mode = 2; g.pool_R = 7; g.pool_C = 8;
      g.pool_tiles_i = ceil_div(Hc, g.pool_R); g.pool_tiles_j = ceil_div(Wc, g.pool_C);
      g.num_m_blocks = B * g.pool_tiles_i * g.pool_tiles_j;
      g.tmem_cols = tmem_cols_for(64 * g.msub);
      g.num_stages = conv_gemm_pick_stages(g);
      pixels_per_load = 0;
    }
    const char* e = unfused
        ? make_tmap_im2col(&g.tmap_a, pl->s2d, 64, (uint64_t)pl->W1, (uint64_t)pl->Hs, (uint64_t)B, 32, (uint64_t)pl->Ws * 32,
                           (uint64_t)pl->Hs * pl->Ws * 32, 0, 0, 0, -3, 1, (uint64_t)B * pl->Hs * pl->Ws * 32, pixels_per_load)
        : make_tmap_tiled4d(&g.tmap_a, pl->s2d, 64, (uint64_t)pl->W1, (uint64_t)pl->Hs, (uint64_t)B, 32, (uint64_t)pl->Ws * 32,
                            (uint64_t)pl->Hs * pl->Ws * 32, (uint32_t)(2 * g.pool_C + 1), (uint32_t)(2 * g.pool_R + 1));
    if (e) return fail(h, DGP_ERR_CUDA, "conv1: %s", e);
    e = make_tmap_2d(&g.tmap_b, L.w, 64, 256, 512, 64);
    if (e) return fail(h, DGP_ERR_CUDA, "conv1: %s", e);
    st.kind = STEP_GEMM;
    if (unfused) {
      st.out_ptr = c1;
      st.end_point = h->net_scope + "/conv1";
      st.oN = B; st.oH = pl->H1; st.oW = pl->W1; st.oC = 64;
    } else {
      st.out_ptr = xa;
      st.oN = B; st.oH = Hc; st.oW = Wc; st.oC = 64;
    }
    pl->steps.push_back(st);
  }
  if (unfused) {
    Step st; st.kind = STEP_POOL;
    st.pin = (const __nv_bfloat16*)c1; st.pN = B; st.pH = pl->H1; st.pW = pl->W1; st.pC = 64; st.pad_t = pad_t; st.pad_l = pad_l;
    st.out_ptr = xa;
    st.end_point = h->net_scope + "/pool1";
    st.oN = B; st.oH = Hc; st.oW = Wc; st.oC = 64;
    pl->steps.push_back(st);
  }
  // ---- bottleneck units
  void* x = xa;
  void* y = xb;
  int Cin = 64;
  for (const UnitDesc& u : h->units) {
    const void* shortcut = nullptr;
    int res_sub = 1, res_H = Hc, res_W = Wc;
    int Ho, Wo, dh, dw;
    if (train) {
      const int ho = ceil_div(Hc, u.stride), wo = ceil_div(Wc, u.stride);
      sc = nullptr;
      if (u.shortcut >= 0 && (rc = alloc_buf(h, &pl->bufs, (size_t)B * Hc * Wc * u.depth * 2 + 1024, &sc))) return rc;
      if ((rc = alloc_buf(h, &pl->bufs, (size_t)B * Hc * Wc * u.base * 2 + 1024, &t1))) return rc;
      if ((rc = alloc_buf(h, &pl->bufs, (size_t)B * ho * wo * u.base * 2 + 1024, &t2))) return rc;
      if ((rc = alloc_buf(h, &pl->bufs, (size_t)B * ho * wo * u.depth * 2 + 1024, &y))) return rc;
      Plan::UnitBufs ub;
      ub.x = x; ub.sc = sc; ub.t1 = t1; ub.t2 = t2; ub.out = y; ub.H = Hc; ub.W = Wc; ub.Ho = ho; ub.Wo = wo; ub.Cin = Cin;
      pl->ub.push_back(ub);
    }
    if (u.shortcut >= 0) {
      Step st;
      rc = make_gemm_step(h, h->layers[u.shortcut], x, B, Hc, Wc, 0, sc, false, nullptr, 1, 0, 0, 0, &st, &dh, &dw);
      if (rc) return rc;
      st.end_point = u.scope + "/shortcut";
      pl->steps.push_back(st);
      shortcut = sc;
    } else {
      shortcut = x;
      res_sub = u.stride;
    }
    {
      Step st;
      rc = make_gemm_step(h, h->layers[u.conv1], x, B, Hc, Wc, 0, t1, false, nullptr, 1, 0, 0, 0, &st, &dh, &dw);
      if (rc) return rc;
      st.end_point = u.scope + "/conv1";
      pl->steps.push_back(st);
    }
    {
      Step st;
      rc = make_gemm_step(h, h->layers[u.conv2], t1, B, Hc, Wc, 1, t2, false, nullptr, 1, 0, 0, 0, &st, &Ho, &Wo);
      if (rc) return rc;
      st.end_point = u.scope + "/conv2";
      pl->steps.push_back(st);
    }
    {
      Step st;
      rc = make_gemm_step(h, h->layers[u.conv3], t2, B, Ho, Wo, 0, y, false, (const __nv_bfloat16*)shortcut, res_sub,
                          res_H, res_W, 0, &st, &dh, &dw);
      if (rc) return rc;
      st.end_point = u.scope;
      pl->steps.push_back(st);
    }
    Hc = Ho; Wc = Wo; Cin = u.depth;
    std::swap(x, y);
  }
  (void)Cin;
  pl->feat = x;
  pl->hf = Hc; pl->wf = Wc;
  // ---- heads: GEMM over feature pixels + col2im
  {
    const ConvLayer& L = h->layers[h->head_layer];
    if ((rc = alloc_buf(h, &pl->bufs, (size_t)B * Hc * Wc * L.Npad * 4, &p))) return rc;
    pl->contrib = (float*)p;
    pl->contrib_ld = L.Npad;
    Step st;
    int dh, dw;
    rc = make_gemm_step(h, L, x, B, Hc, Wc, 0, pl->contrib, true, nullptr, 1, 0, 0, 0, &st, &dh, &dw);
    if (rc) return rc;
    pl->head_step = (int)pl->steps.size();
    pl->steps.push_back(st);
    Step c; c.kind = STEP_COL2IM;
    pl->steps.push_back(c);
  }
  if (train) {
    const int nj = h->cfg.num_joints;
    if ((rc = alloc_buf(h, &pl->bufs, (size_t)B * 4 * Hc * Wc * nj * 4, &p))) return rc;
    pl->logits = (float*)p;
    if (h->cfg.location_refinement) {
      if ((rc = alloc_buf(h, &pl->bufs, (size_t)B * 4 * Hc * Wc * 2 * nj * 4, &p))) return rc;
      pl->locref = (float*)p;
    }
  }
  if (getenv("DGP_DEBUG_PLAN")) {
    for (size_t i = 0; i < pl->steps.size(); ++i) {
      const Step& st = pl->steps[i];
      if (st.kind != STEP_GEMM) continue;
      const ConvGemmParams& g = st.gp;
      fprintf(stderr, "dgp plan B=%d %dx%d step %2zu %-50s M=%d N=%d K=%d block_n=%d a_mode=%d epi=%d msub=%d cta2=%d stages=%d epi_bufs=%d smem=%zu\n",
              B, H, W, i, st.end_point.c_str(), g.M, g.N, g.num_k_blocks * 64, g.block_n, g.a_mode, g.epi_mode, g.msub, g.cta2,
              g.num_stages, g.epi_bufs, conv_gemm_smem_bytes(g));
    }
  }
  *out = pl.get();
  plans[key] = std::move(pl);
  return DGP_OK;
}

// first_step / last_step select a slice of the plan: [0, head_step) is PoseNet.extract_features, [head_step, end) the
// prediction layers (dgp_extract_features / dgp_prediction_layers); the default runs everything.
int run_forward_plan(dgp_handle* h, Plan* pl, const uint8_t* frames_dev, float* logits_dev, float* locref_dev,
                     cudaStream_t s, int first_step, int last_step) {
  int rc;
  if (last_step < 0) last_step = (int)pl->steps.size();
  int si = first_step;
  while (si < last_step) {
    // bracket mode: one event pair around the whole run of same-kind launches (the 54 GEMM layers are one run), so that the
    // launches inside keep their programmatic-dependent-launch overlap while they are timed
    int sj = si;
    if (h->profiling && h->profile_brackets)
      while (sj + 1 < last_step && pl->steps[sj + 1].kind == pl->steps[si].kind) ++sj;
    ProfScope prof(h, (int)pl->steps[si].kind, s, sj - si + 1);
    for (; si <= sj; ++si) {
      const Step& st = pl->steps[si];
      switch (st.kind) {
        case STEP_PREP:
          CU_OK(h, launch_prep_s2d(frames_dev, pl->B, pl->H, pl->W, h->cfg.mean_pixel, pl->s2d, pl->Hs, pl->Ws, h->fp16, s));
          break;
        case STEP_GEMM:
          CU_OK(h, launch_conv_gemm(st.gp, h->num_sms, s));
          break;
        case STEP_POOL:
          CU_OK(h, launch_maxpool3x3s2(st.pin, st.pN, st.pH, st.pW, st.pC, (__nv_bfloat16*)st.out_ptr, st.oH, st.oW, st.pad_t,
                                       st.pad_l, h->fp16, s));
          break;
        case STEP_COL2IM:
          CU_OK(h, launch_deconv_col2im(pl->contrib, pl->B, pl->hf, pl->wf, pl->contrib_ld, h->ctot, h->cfg.num_joints,
                                        h->head_bias, logits_dev, locref_dev, s));
          break;
      }
      h->launches++;
      if ((rc = keep_activation(h, st, s))) return rc;
    }
  }
  return DGP_OK;
}

int keep_activation(dgp_handle* h, const Step& st, cudaStream_t s) {
  if (!h->debug_keep || st.end_point.empty() || !st.out_ptr) return DGP_OK;
  const size_t bytes = (size_t)st.oN * st.oH * st.oW * st.oC * 2;
  h->kept.erase(st.end_point);
  dgp_handle::Kept k;
  k.N = st.oN; k.H = st.oH; k.W = st.oW; k.C = st.oC;
  CU_OK(h, k.buf.alloc(bytes));
  CU_OK(h, cudaMemcpyAsync(k.buf.get(), st.out_ptr, bytes, cudaMemcpyDeviceToDevice, s));
  h->kept[st.end_point] = std::move(k);
  return DGP_OK;
}

int ensure(dgp_handle* h, DevBuf* b, size_t bytes) {
  if (b->bytes() >= bytes) return DGP_OK;
  CU_OK(h, b->alloc(bytes));
  return DGP_OK;
}

// The ring of dgp_estimate_pose_stream, the H2D copies and `frames` carry source-size frames; the transform writes `xf`
// on the compute stream.
int PoseStaging::reserve(dgp_handle* h, int batch, int H0, int W0, int H, int W, bool identity) {
  const int nj = h->cfg.num_joints;
  int hf, wf, ho, wo;
  dgp_output_dims_os(H, W, h->output_stride, &hf, &wf, &ho, &wo);
  const size_t frame_bytes = (size_t)H0 * W0 * 3;
  int rc;
  if ((rc = ensure(h, &frames[0], frame_bytes * batch))) return rc;
  if ((rc = ensure(h, &frames[1], frame_bytes * batch))) return rc;
  if (!identity && (rc = ensure(h, &xf, (size_t)H * W * 3 * batch))) return rc;
  if ((rc = ensure(h, &logits, (size_t)batch * ho * wo * nj * 4))) return rc;
  if ((rc = ensure(h, &mu, (size_t)batch * nj * 2 * 4))) return rc;
  if ((rc = ensure(h, &peak, (size_t)batch * nj * 2 * 4))) return rc;
  if ((rc = ensure(h, &lik, (size_t)batch * nj * 4))) return rc;
  if (!copy_stream) CU_OK(h, create(&copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    if (!ev_copied[i]) CU_OK(h, create(&ev_copied[i], cudaEventDisableTiming));
    if (!ev_consumed[i]) CU_OK(h, create(&ev_consumed[i], cudaEventDisableTiming));
  }
  return DGP_OK;
}

int PoseStaging::reserve_render(dgp_handle* h, bool jpeg, int batch, int trailpoints) {
  if (!d2h_stream) CU_OK(h, create(&d2h_stream, cudaStreamNonBlocking));
  if (jpeg && !packet_stream) CU_OK(h, create(&packet_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i)
    if (!ev_drawn[i]) CU_OK(h, create(&ev_drawn[i], cudaEventDisableTiming));
  marker_rows = (trailpoints > 1 ? trailpoints - 1 : 0) + batch;
  return ensure(h, &marker_table, (size_t)2 * 3 * marker_rows * h->cfg.num_joints * sizeof(double));
}

int PoseStaging::run_batch(dgp_handle* h, const PoseJob& j, const uint8_t* host_frames, int n, int run_n, int it, int64_t t0,
                           cudaHostFn_t release, void* release_arg, const RenderBatch* render) {
  const int nj = h->cfg.num_joints;
  int hf, wf, ho, wo;
  dgp_output_dims_os(j.H, j.W, h->output_stride, &hf, &wf, &ho, &wo);
  cudaStream_t s = h->stream.get(), cs = copy_stream.get();
  const int slot = it & 1;
  // H2D of this batch on the copy stream, as soon as the batch that last used this slot has been consumed
  if (it >= 2) CU_OK(h, cudaStreamWaitEvent(cs, ev_consumed[slot].get(), 0));
  CU_OK(h, cudaMemcpyAsync(frames[slot].get(), host_frames, (size_t)j.H0 * j.W0 * 3 * n, cudaMemcpyHostToDevice, cs));
  if (release) CU_OK(h, cudaLaunchHostFunc(cs, release, release_arg));
  CU_OK(h, cudaEventRecord(ev_copied[slot].get(), cs));
  CU_OK(h, cudaStreamWaitEvent(s, ev_copied[slot].get(), 0));
  const uint8_t* x = frames[slot].get<uint8_t>();
  int rc;
  if (!j.identity) {
    if ((rc = resize_crop_impl(h, x, n, j.H0, j.W0, j.transform, xf.get<uint8_t>(), s))) return rc;
    x = xf.get<uint8_t>();
  }
  if ((rc = dgp_forward(h, x, run_n, j.H, j.W, logits.get<float>(), nullptr, s))) return rc;
  if (!render) CU_OK(h, cudaEventRecord(ev_consumed[slot].get(), s));
  if ((rc = dgp_softargmax(h, logits.get<float>(), nullptr, run_n, ho, wo, nj, j.gamma, j.gauss_len, mu.get<float>(),
                           peak.get<int32_t>(), lik.get<float>(), nullptr, nullptr, s)))
    return rc;
  if (render) {
    // the next H2D into this slot waits for ev_consumed, so it must follow the copy of the annotated frames, not the forward
    cudaStream_t ds = d2h_stream.get();
    const MarkerArgs& ma = *render->args;
    // the batch's rows go after the carried ones; the last `carry` rows of the sequence are copied to the front of the other
    // half for the next batch (two halves, because for a batch shorter than the trail the rows would overlap in one)
    const int trail = ma.trailpoints > 1 ? ma.trailpoints - 1 : 0;
    const int history = (int)std::min<int64_t>(trail, t0), carry = std::min(trail, history + n);
    const size_t plane = (size_t)marker_rows * nj;
    double* xs = marker_table.get<double>() + (size_t)(it & 1) * 3 * plane + (size_t)trail * nj;
    if ((rc = marker_table_fused(h, mu.get<float>(), lik.get<float>(), n, ma, xs, xs + plane, xs + 2 * plane, s))) return rc;
    if ((rc = draw_markers_impl(h, frames[slot].get<uint8_t>(), n, j.H0, j.W0, xs, xs + plane, xs + 2 * plane, history, ma,
                                s)))
      return rc;
    if (carry > 0) {
      double* next = marker_table.get<double>() + (size_t)((it + 1) & 1) * 3 * plane + (size_t)(trail - carry) * nj;
      CU_OK(h, cudaMemcpy2DAsync(next, plane * sizeof(double), xs + (ptrdiff_t)(n - carry) * nj, plane * sizeof(double),
                                 (size_t)carry * nj * sizeof(double), 3, cudaMemcpyDeviceToDevice, s));
    }
    if (render->quality) {
      // the encode is the last reader of the slot; only the packets' offsets | sizes go D2H here, the writer thread copies
      // the packets themselves once it knows their total
      if ((rc = encode_jpeg_impl(h, frames[slot].get<uint8_t>(), n, j.H0, j.W0, render->quality, render->packets,
                                 render->packets_bytes, render->meta, render->meta + n, s)))
        return rc;
      CU_OK(h, cudaEventRecord(ev_consumed[slot].get(), s));
      CU_OK(h, cudaStreamWaitEvent(ds, ev_consumed[slot].get(), 0));
      CU_OK(h, cudaMemcpyAsync(render->dst, render->meta, (size_t)2 * n * sizeof(int64_t), cudaMemcpyDeviceToHost, ds));
    } else {
      CU_OK(h, cudaEventRecord(ev_drawn[slot].get(), s));
      CU_OK(h, cudaStreamWaitEvent(ds, ev_drawn[slot].get(), 0));
      CU_OK(h, cudaMemcpyAsync(render->dst, frames[slot].get(), (size_t)j.H0 * j.W0 * 3 * n, cudaMemcpyDeviceToHost, ds));
      CU_OK(h, cudaEventRecord(ev_consumed[slot].get(), ds));
    }
    CU_OK(h, cudaLaunchHostFunc(ds, render->handoff, render->handoff_arg));
  }
  CU_OK(h, cudaMemcpyAsync(j.mu_host + (size_t)t0 * nj * 2, mu.get(), (size_t)n * nj * 2 * 4, cudaMemcpyDeviceToHost, s));
  if (j.peak_host)
    CU_OK(h, cudaMemcpyAsync(j.peak_host + (size_t)t0 * nj * 2, peak.get(), (size_t)n * nj * 2 * 4, cudaMemcpyDeviceToHost, s));
  if (j.lik_host)
    CU_OK(h, cudaMemcpyAsync(j.lik_host + (size_t)t0 * nj, lik.get(), (size_t)n * nj * 4, cudaMemcpyDeviceToHost, s));
  return DGP_OK;
}

}  // namespace dgp

extern "C" {

int dgp_create(const dgp_config* cfg, dgp_handle** out) {
  if (!cfg || !out) return fail(nullptr, DGP_ERR_INVALID, "dgp_create: null argument");
  if (cfg->num_joints < 1 || cfg->num_joints > 256) return fail(nullptr, DGP_ERR_INVALID, "dgp_create: num_joints out of range");
  if (cfg->precision != 0 && cfg->precision != 1) return fail(nullptr, DGP_ERR_INVALID, "dgp_create: precision must be 0 (bf16) or 1 (fp16)");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, DGP_ERR_CUDA, "dgp_create: no CUDA device (%s); this library has no CPU fallback",
                cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, DGP_ERR_INVALID, "dgp_create: bad device ordinal");
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, cfg->device);
  if (e != cudaSuccess) return fail(nullptr, DGP_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, DGP_ERR_UNSUPPORTED, "dgp_create: device is sm_%d%d; this library only runs on sm_100 (B200)",
                prop.major, prop.minor);
  e = cudaSetDevice(cfg->device);
  if (e != cudaSuccess) return fail(nullptr, DGP_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
  if (const char* te = tma_init()) return fail(nullptr, DGP_ERR_CUDA, "dgp_create: %s", te);
  dgp_handle* h = new dgp_handle();
  h->cfg = *cfg;
  h->fp16 = cfg->precision == 1 ? 1 : 0;
  if (h->cfg.bn_epsilon <= 0) h->cfg.bn_epsilon = 1e-5f;
  h->device = cfg->device;
  h->num_sms = prop.multiProcessorCount;
  e = create(&h->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    delete h;
    return fail(nullptr, DGP_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
  }
  *out = h;
  return DGP_OK;
}

void dgp_destroy(dgp_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();  // nothing in flight uses what the owners release
  delete h;
}

const char* dgp_last_error(const dgp_handle* h) { return h ? h->err : g_create_error; }

int dgp_load_weights(dgp_handle* h, const char* name, const void* host_ptr, const int64_t* shape, int ndim, int dtype) {
  if (!h) return DGP_ERR_INVALID;
  if (!name || !host_ptr || !shape || ndim < 1 || ndim > 4) return fail(h, DGP_ERR_INVALID, "dgp_load_weights: bad argument");
  if (dtype != 0) return fail(h, DGP_ERR_UNSUPPORTED, "dgp_load_weights: only float32 (dtype 0) is accepted");
  if (h->finalized) return fail(h, DGP_ERR_STATE, "dgp_load_weights after dgp_finalize_weights");
  HostVar v;
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) {
    if (shape[i] <= 0) return fail(h, DGP_ERR_INVALID, "dgp_load_weights: bad shape for %s", name);
    v.shape.push_back(shape[i]);
    n *= (size_t)shape[i];
  }
  v.data.assign((const float*)host_ptr, (const float*)host_ptr + n);
  h->host_vars[name] = std::move(v);
  return DGP_OK;
}

int dgp_finalize_weights(dgp_handle* h) {
  if (!h) return DGP_ERR_INVALID;
  if (h->finalized) return fail(h, DGP_ERR_STATE, "weights already finalized");
  CU_OK(h, cudaSetDevice(h->device));
  // The backbone is the one the variable names describe (as Saver.restore works off names): slim's resnet_v1_50 / _101 /
  // _152 differ only in the number of units of blocks 2 and 3; every layer of the deeper nets has a ResNet-50 shape.
  static const struct { const char* scope; int depth, units[4]; } nets[3] = {
      {"resnet_v1_50", 50, {3, 4, 6, 3}}, {"resnet_v1_101", 101, {3, 4, 23, 3}}, {"resnet_v1_152", 152, {3, 8, 36, 3}}};
  std::string scope;
  for (const auto& kv : h->host_vars) {
    if (kv.first.compare(0, 10, "resnet_v1_") != 0) continue;
    const std::string p = kv.first.substr(0, kv.first.find('/'));
    if (scope.empty()) scope = p;
    else if (p != scope)
      return fail(h, DGP_ERR_INVALID, "the weights mix the backbone scopes %s and %s", scope.c_str(), p.c_str());
  }
  const int* units = nullptr;
  for (const auto& n : nets)
    if (scope == n.scope) { h->depth = n.depth; units = n.units; }
  if (!units) {
    if (scope.empty())
      return fail(h, DGP_ERR_INVALID, "no backbone variables: expected names under resnet_v1_50/, resnet_v1_101/ or resnet_v1_152/");
    return fail(h, DGP_ERR_INVALID, "unsupported backbone scope %s (resnet_v1_50, resnet_v1_101 or resnet_v1_152)", scope.c_str());
  }
  h->net_scope = scope;
  int rc = build_conv1_layer(h);
  if (rc) return rc;
  // slim resnet_v1_<depth> + stack_blocks_dense(output_stride): see oracle/resnet_v1.py::unit_plan.  The root block has
  // stride 4; once the units reach output_stride / 4, every later unit runs at stride 1 and its rate takes the stride over.
  static const struct { const char* name; int base, stride; } blocks[4] = {
      {"block1", 64, 2}, {"block2", 128, 2}, {"block3", 256, 2}, {"block4", 512, 1}};
  int cin = 64, current_stride = 1, rate = 1;
  const int target = h->output_stride / 4;
  for (int bi = 0; bi < 4; ++bi) {
    const auto& b = blocks[bi];
    for (int u = 0; u < units[bi]; ++u) {
      const int ustride = (u == units[bi] - 1) ? b.stride : 1;
      UnitDesc ud;
      char sc[128];
      snprintf(sc, sizeof(sc), "%s/%s/unit_%d/bottleneck_v1", scope.c_str(), b.name, u + 1);
      ud.scope = sc; ud.depth = b.base * 4; ud.base = b.base;
      if (current_stride == target) { ud.stride = 1; ud.rate = rate; rate *= ustride; }
      else { ud.stride = ustride; ud.rate = 1; current_stride *= ustride; }
      if (cin != ud.depth) {
        if (ud.stride != 1) return fail(h, DGP_ERR_UNSUPPORTED, "strided projection shortcut not on this path");
        if ((rc = build_conv_layer(h, ud.scope + "/shortcut", 1, 1, cin, ud.depth, 1, 1, false, &ud.shortcut))) return rc;
      }
      if ((rc = build_conv_layer(h, ud.scope + "/conv1", 1, 1, cin, ud.base, 1, 1, true, &ud.conv1))) return rc;
      if ((rc = build_conv_layer(h, ud.scope + "/conv2", 3, 3, ud.base, ud.base, ud.stride, ud.rate, true, &ud.conv2))) return rc;
      if ((rc = build_conv_layer(h, ud.scope + "/conv3", 1, 1, ud.base, ud.depth, 1, 1, true, &ud.conv3))) return rc;
      cin = ud.depth;
      h->units.push_back(ud);
    }
  }
  if ((rc = build_head_layer(h))) return rc;
  if ((rc = upload_arena(h))) return rc;
  h->host_vars.clear();
  h->finalized = true;
  return DGP_OK;
}

int dgp_net_depth(const dgp_handle* h, int* depth) {
  if (!h || !depth) return DGP_ERR_INVALID;
  if (!h->finalized) return fail(const_cast<dgp_handle*>(h), DGP_ERR_STATE, "dgp_net_depth before dgp_finalize_weights");
  *depth = h->depth;
  return DGP_OK;
}

int dgp_set_output_stride(dgp_handle* h, int output_stride) {
  if (!h) return DGP_ERR_INVALID;
  if (output_stride != 8 && output_stride != 16)
    return fail(h, DGP_ERR_UNSUPPORTED, "dgp_set_output_stride: output_stride must be 8 or 16, got %d", output_stride);
  if (h->finalized) return fail(h, DGP_ERR_STATE, "dgp_set_output_stride after dgp_finalize_weights");
  h->output_stride = output_stride;
  return DGP_OK;
}

int dgp_get_output_stride(const dgp_handle* h, int* output_stride) {
  if (!h || !output_stride) return DGP_ERR_INVALID;
  *output_stride = h->output_stride;
  return DGP_OK;
}

int dgp_output_dims(int H, int W, int* h_feat, int* w_feat, int* h_out, int* w_out) {
  return dgp_output_dims_os(H, W, 16, h_feat, w_feat, h_out, w_out);
}

int dgp_output_dims_os(int H, int W, int output_stride, int* h_feat, int* w_feat, int* h_out, int* w_out) {
  if (H < 1 || W < 1 || (output_stride != 8 && output_stride != 16)) return DGP_ERR_INVALID;
  // every stride-2 layer (conv1, pool1 and the last unit of each block before output_stride is reached) is SAME: ceil(v / 2)
  const int halvings = output_stride == 16 ? 4 : 3;
  int a = H, b = W;
  for (int i = 0; i < halvings; ++i) { a = (a + 1) / 2; b = (b + 1) / 2; }
  if (h_feat) *h_feat = a;
  if (w_feat) *w_feat = b;
  if (h_out) *h_out = 2 * a;
  if (w_out) *w_out = 2 * b;
  return DGP_OK;
}

int dgp_forward(dgp_handle* h, const uint8_t* frames_dev, int B, int H, int W, float* logits_dev, float* locref_dev,
                void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->finalized) return fail(h, DGP_ERR_STATE, "dgp_forward before dgp_finalize_weights");
  if (!frames_dev || !logits_dev || B < 1 || H < 32 || W < 32) return fail(h, DGP_ERR_INVALID, "dgp_forward: bad argument");
  if (locref_dev && !h->cfg.location_refinement) return fail(h, DGP_ERR_INVALID, "dgp_forward: locref requested but the head was not built");
  CU_OK(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  Plan* pl = nullptr;
  int rc = build_plan(h, B, H, W, false, &pl);
  if (rc) return rc;
  return run_forward_plan(h, pl, frames_dev, logits_dev, locref_dev, s);
}

int dgp_softargmax(dgp_handle* h, const float* logits_dev, const float* locref_dev, int B, int H, int W, int nj,
                   float gamma, float gauss_len, float* mu_dev, int32_t* peak_dev, float* lik_dev,
                   int32_t* dlc_peak_dev, float* dlc_pose_dev, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (B == 0) return DGP_OK;
  if (!logits_dev || B < 0 || H < 2 || W < 2 || nj < 1) return fail(h, DGP_ERR_INVALID, "dgp_softargmax: bad argument");
  if ((H & 1) || (W & 1)) return fail(h, DGP_ERR_INVALID, "dgp_softargmax: scoremap dims must be even (they are 2*ceil(./16))");
  if (gauss_len < 1.0f || gauss_len >= 5.0f) return fail(h, DGP_ERR_INVALID, "dgp_softargmax: gauss_len must be in [1, 5)");
  if (!(gamma > 0.0f)) return fail(h, DGP_ERR_INVALID, "dgp_softargmax: gamma must be > 0");
  if (((uintptr_t)logits_dev & 15) != 0) return fail(h, DGP_ERR_INVALID, "dgp_softargmax: logits must be 16-byte aligned");
  if (nj > 128 || softargmax_tact(nj) <= 0)
    return fail(h, DGP_ERR_UNSUPPORTED, "dgp_softargmax: num_joints must be <= 128 with num_joints / gcd(num_joints, 4) <= 32");
  CU_OK(h, cudaSetDevice(h->device));
  const int splits = softargmax_splits(H, W, nj);
  if (int rc = ensure(h, &h->sa_ws, (size_t)B * splits * nj * sizeof(SaPartial))) return rc;
  ProfScope prof(h, 4, (cudaStream_t)stream);
  CU_OK(h, launch_softargmax(logits_dev, locref_dev, B, H, W, nj, gamma, gauss_len, h->cfg.stride, h->cfg.locref_stdev,
                             h->sa_ws.get<SaPartial>(), splits, mu_dev, peak_dev, lik_dev, dlc_peak_dev, dlc_pose_dev, nullptr,
                             (cudaStream_t)stream));
  h->launches += 2;
  return DGP_OK;
}

int dgp_softmax_map(dgp_handle* h, const float* logits_dev, int B, int H, int W, int nj, float gamma, float gauss_len,
                    float* map_dev, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (B == 0) return DGP_OK;
  if (!logits_dev || !map_dev || B < 0 || nj < 1 || (H & 1) || (W & 1) || gauss_len < 1.0f || gauss_len >= 5.0f)
    return fail(h, DGP_ERR_INVALID, "dgp_softmax_map: bad argument");
  CU_OK(h, cudaSetDevice(h->device));
  const int splits = softargmax_splits(H, W, nj);
  const size_t need = (size_t)B * splits * nj * sizeof(SaPartial) + (size_t)B * nj * 2 * sizeof(float);
  if (int rc = ensure(h, &h->sa_ws, need)) return rc;
  SaPartial* ws = h->sa_ws.get<SaPartial>();
  float* norm = reinterpret_cast<float*>(ws + (size_t)B * splits * nj);
  CU_OK(h, launch_softargmax(logits_dev, nullptr, B, H, W, nj, gamma, gauss_len, h->cfg.stride, h->cfg.locref_stdev, ws, splits,
                             nullptr, nullptr, nullptr, nullptr, nullptr, norm, (cudaStream_t)stream));
  CU_OK(h, launch_softmax_map(logits_dev, norm, B, H, W, nj, gamma, gauss_len, map_dev, h->num_sms, (cudaStream_t)stream));
  h->launches += 3;
  return DGP_OK;
}

int dgp_run_loss_impl(dgp_handle* h, const dgp_loss_cfg* cfg, const dgp_loss_batch* b, float* losses_dev,
                    float* targets_all_dev, float* grad_pred_dev, float* grad_locref_dev, int visible_only, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!cfg || !b || !losses_dev || !b->pred_dev) return fail(h, DGP_ERR_INVALID, "dgp_loss_forward: null argument");
  const int nj = h->cfg.num_joints;
  if (b->nt < 1 || b->nbv < 0 || b->nbh < 0 || b->nbv + b->nbh > b->nt * nj)
    return fail(h, DGP_ERR_INVALID, "dgp_loss_forward: bad marker counts");
  if (cfg->gm2 < 0 || cfg->gm2 > 2 || (cfg->gm3 != 0 && cfg->gm3 != 3))
    return fail(h, DGP_ERR_INVALID, "dgp_loss_forward: Not implemented (gm2 in {0,1,2}, gm3 in {0,3}; fitdgp.py:1021,1037)");
  if (cfg->gm3 == 3 && cfg->gm2 == 0)
    return fail(h, DGP_ERR_INVALID, "dgp_loss_forward: gm3=3 needs gm2 in {1,2} (pred_h_scaled1 is undefined in the reference)");
  if (b->nbv > 0 && (!b->targets_dev || !b->visible_marker_dev || !b->visible_marker_in_targets_dev))
    return fail(h, DGP_ERR_INVALID, "dgp_loss_forward: visible markers without targets");
  if (b->locref_dev && (!b->locref_map_dev || !b->locref_mask_dev))
    return fail(h, DGP_ERR_INVALID, "dgp_loss_forward: locref without map/mask");
  if (b->nl > 0 && (!b->edges_dev || !b->ws_dev || !b->ws_max_dev))
    return fail(h, DGP_ERR_INVALID, "dgp_loss_forward: skeleton without ws/ws_max");
  CU_OK(h, cudaSetDevice(h->device));
  const int nm = b->nt * nj;
  const size_t flow_part_bytes = (size_t)nm * ((b->Hin + 15) / 16 + 1) * 8 * 4;
  const size_t need = (size_t)nm * 2 * 4 * 3 + (size_t)(b->nbv + b->nbh + 1) * 16 + (size_t)nm * 4 + (size_t)nm * 16 + 512 + flow_part_bytes;
  int rc = ensure(h, &h->loss_ws, need);
  if (rc) return rc;
  char* w = h->loss_ws.get<char>();
  float* mu = (float*)w; w += (size_t)nm * 2 * 4;
  float* all = (float*)w; w += (size_t)nm * 2 * 4;
  float* norm = (float*)w; w += (size_t)nm * 2 * 4;
  w = (char*)(((uintptr_t)w + 15) & ~(uintptr_t)15);
  float4* partials = (float4*)w; w += (size_t)(b->nbv + b->nbh + 1) * 16;
  float* meanflow = (float*)w; w += (size_t)nm * 4;
  w = (char*)(((uintptr_t)w + 15) & ~(uintptr_t)15);
  float4* boxgrad = (float4*)w; w += (size_t)nm * 16;
  float* flow_part = (float*)w;
  if ((b->H & 1) || (b->W & 1) || cfg->gauss_len < 1.0f || cfg->gauss_len >= 5.0f || !(cfg->gamma > 0.0f))
    return fail(h, DGP_ERR_INVALID, "dgp_loss: scoremap dims must be even, gauss_len in [1,5), gamma > 0");
  {
    const int splits = softargmax_splits(b->H, b->W, nj);
    if ((rc = ensure(h, &h->sa_ws, (size_t)b->nt * splits * nj * sizeof(SaPartial)))) return rc;
    CU_OK(h, launch_softargmax(b->pred_dev, nullptr, b->nt, b->H, b->W, nj, cfg->gamma, cfg->gauss_len, h->cfg.stride,
                               h->cfg.locref_stdev, h->sa_ws.get<SaPartial>(), splits, mu, nullptr, nullptr, nullptr, nullptr,
                               norm, (cudaStream_t)stream));
    h->launches += 2;
  }
  LossArgs a;
  a.pred = b->pred_dev; a.locref = b->locref_dev; a.mu = mu;
  a.nt = b->nt; a.H = b->H; a.W = b->W; a.nj = nj;
  a.targets = b->targets_dev; a.locref_map = b->locref_map_dev; a.locref_mask = b->locref_mask_dev;
  a.visible = b->visible_marker_dev; a.nbv = b->nbv; a.hidden = b->hidden_marker_dev; a.nbh = b->nbh;
  a.vis_in_targets = b->visible_marker_in_targets_dev;
  a.edges = b->edges_dev; a.nl = b->nl; a.ws = b->ws_dev; a.ws_max = b->ws_max_dev;
  a.flow = b->vector_field_dev; a.Hin = b->Hin; a.Win = b->Win; a.wt_batch = b->wt_batch_dev;
  a.stride = h->cfg.stride; a.lengthscale = cfg->lengthscale; a.wt = cfg->wt; a.wt_max = cfg->wt_max;
  a.wn_visible = cfg->wn_visible; a.wn_hidden = cfg->wn_hidden; a.locref_weight = cfg->locref_loss_weight;
  a.n_vis_total = cfg->n_visible_frames_total; a.n_hid_total = cfg->n_frames_total - cfg->n_visible_frames_total;
  a.gm2 = cfg->gm2; a.gm3 = cfg->gm3; a.locref_mse = cfg->locref_mse ? 1 : 0;
  a.all_markers = all; a.partials = partials; a.meanflow = meanflow; a.out = losses_dev;
  a.boxgrad = grad_pred_dev ? boxgrad : nullptr;
  a.flow_part = flow_part;
  if (a.wt > 0.0f && a.flow != nullptr && !a.wt_batch) return fail(h, DGP_ERR_INVALID, "dgp_loss_forward: wt > 0 needs wt_batch");
  if (b->vector_field_ready_event && b->vector_field_dev)   // the flow field comes from another stream (dgp_learn_wt overlapped)
    CU_OK(h, cudaStreamWaitEvent((cudaStream_t)stream, (cudaEvent_t)b->vector_field_ready_event, 0));
  CU_OK(h, launch_dgp_loss(a, (cudaStream_t)stream));
  h->launches += 4;
  if (targets_all_dev)
    CU_OK(h, cudaMemcpyAsync(targets_all_dev, all, (size_t)nm * 2 * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (grad_pred_dev) {
    CU_OK(h, launch_dgp_loss_backward(a, norm, cfg->gamma, cfg->gauss_len, visible_only, grad_pred_dev, grad_locref_dev,
                                      (cudaStream_t)stream));
    h->launches += 1;
  }
  return DGP_OK;
}

int dgp_loss_forward(dgp_handle* h, const dgp_loss_cfg* cfg, const dgp_loss_batch* b, float* losses_dev,
                     float* targets_all_dev, void* stream) {
  return dgp_run_loss_impl(h, cfg, b, losses_dev, targets_all_dev, nullptr, nullptr, 0, stream);
}

int dgp_loss_backward(dgp_handle* h, const dgp_loss_cfg* cfg, const dgp_loss_batch* b, float* losses_dev,
                      float* grad_pred_dev, float* grad_locref_dev, int visible_only, void* stream) {
  if (h && !grad_pred_dev) return fail(h, DGP_ERR_INVALID, "dgp_loss_backward: grad_pred_dev is required");
  return dgp_run_loss_impl(h, cfg, b, losses_dev, nullptr, grad_pred_dev, grad_locref_dev, visible_only, stream);
}

int dgp_soft_pose(dgp_handle* h, const float* logits_dev, const float* locref_dev, int B, int H, int W, int nj, float gamma,
                  float gauss_len, int swap_offsets, float* map_ws_dev, float* pose_dev, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (B == 0) return DGP_OK;
  if (!logits_dev || !locref_dev || !map_ws_dev || !pose_dev || B < 0 || nj < 1)
    return fail(h, DGP_ERR_INVALID, "dgp_soft_pose: bad argument");
  if (((uintptr_t)locref_dev & 7) != 0) return fail(h, DGP_ERR_INVALID, "dgp_soft_pose: locref must be 8-byte aligned");
  int rc = dgp_softmax_map(h, logits_dev, B, H, W, nj, gamma, gauss_len, map_ws_dev, stream);
  if (rc) return rc;
  CU_OK(h, launch_soft_pose(map_ws_dev, locref_dev, B, H, W, nj, h->cfg.stride, h->cfg.locref_stdev, swap_offsets, pose_dev,
                            (cudaStream_t)stream));
  h->launches++;
  return DGP_OK;
}

int dgp_locref_targets(dgp_handle* h, const double* joint_loc_dev, const int32_t* frame_idx_dev, int n_vis, int nt, int H,
                       int W, double pos_dist_thresh, double locref_stdev, float* locref_map_dev, float* locref_mask_dev,
                       void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (n_vis < 0 || nt < 1 || n_vis > nt || H < 1 || W < 1 || !locref_map_dev || !locref_mask_dev || !(pos_dist_thresh > 0) ||
      (n_vis > 0 && (!joint_loc_dev || !frame_idx_dev)))
    return fail(h, DGP_ERR_INVALID, "dgp_locref_targets: bad argument");
  CU_OK(h, cudaSetDevice(h->device));
  CU_OK(h, launch_locref_targets(joint_loc_dev, frame_idx_dev, n_vis, nt, h->cfg.num_joints, H, W, (double)h->cfg.stride,
                                 pos_dist_thresh, locref_stdev > 0 ? locref_stdev : (double)h->cfg.locref_stdev, locref_map_dev, locref_mask_dev,
                                 (cudaStream_t)stream));
  h->launches += n_vis > 0 ? 1 : 0;
  return DGP_OK;
}

int dgp_marker_indices(dgp_handle* h, const int32_t* visible_frames_dev, int n_vis, const int32_t* hidden_frames_dev, int n_hid,
                       const double* joint_loc_dev, int nt, int32_t* visible_marker_dev, int32_t* hidden_marker_dev,
                       int32_t* visible_in_targets_dev, int32_t* counts_dev, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (n_vis < 0 || n_hid < 0 || nt < 1 || n_vis + n_hid > nt || !visible_marker_dev || !hidden_marker_dev || !visible_in_targets_dev ||
      !counts_dev || (n_vis > 0 && (!visible_frames_dev || !joint_loc_dev)) || (n_hid > 0 && !hidden_frames_dev))
    return fail(h, DGP_ERR_INVALID, "dgp_marker_indices: bad argument");
  CU_OK(h, cudaSetDevice(h->device));
  CU_OK(h, launch_marker_indices(visible_frames_dev, n_vis, hidden_frames_dev, n_hid, joint_loc_dev, h->cfg.num_joints, nt,
                                 visible_marker_dev, hidden_marker_dev, visible_in_targets_dev, counts_dev, (cudaStream_t)stream));
  h->launches++;
  return DGP_OK;
}

int dgp_learn_wt(dgp_handle* h, const uint8_t* frames_dev, int T, int H, int W, float* field_dev, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (T < 0 || H < 1 || W < 1 || (T > 1 && (!frames_dev || !field_dev))) return fail(h, DGP_ERR_INVALID, "dgp_learn_wt: bad argument");
  if (T < 2) return DGP_OK;
  CU_OK(h, cudaSetDevice(h->device));
  if (int rc = ensure(h, &h->flow_ws, learn_wt_workspace_bytes(T, H, W))) return rc;
  int nl = 0;
  CU_OK(h, launch_learn_wt(frames_dev, T, H, W, field_dev, h->flow_ws.get(), &nl, (cudaStream_t)stream));
  h->launches += nl;
  return DGP_OK;
}

int dgp_motion_energy(dgp_handle* h, const uint8_t* frames_dev, int T, size_t frame_bytes, uint64_t* sums_dev, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (T < 0 || frame_bytes == 0 || (T > 0 && (!frames_dev || !sums_dev))) return fail(h, DGP_ERR_INVALID, "dgp_motion_energy: bad argument");
  if (T == 0) return DGP_OK;
  CU_OK(h, cudaSetDevice(h->device));
  CU_OK(h, launch_motion_energy(frames_dev, T, frame_bytes, reinterpret_cast<unsigned long long*>(sums_dev), h->num_sms,
                                (cudaStream_t)stream));
  h->launches += T > 1 ? 1 : 0;
  return DGP_OK;
}

int dgp_sigmoid(dgp_handle* h, const float* logits_dev, float* prob_dev, size_t n, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!logits_dev || !prob_dev || (n % 4)) return fail(h, DGP_ERR_INVALID, "dgp_sigmoid: bad argument");
  if (n == 0) return DGP_OK;
  CU_OK(h, cudaSetDevice(h->device));
  CU_OK(h, launch_sigmoid_map(logits_dev, prob_dev, n, h->num_sms, (cudaStream_t)stream));
  h->launches++;
  return DGP_OK;
}

int dgp_potentials(dgp_handle* h, const float* mu_dev, const float* mu_halo_next_dev, int T, int nj,
                   const int32_t* edges_dev, int nl, const float* ws_dev, const float* ws_max_dev, float wt_max,
                   float* skel_dist_dev, float* temporal_dev, float* e_skel_dev, float* e_temp_dev, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (T == 0) return DGP_OK;
  if (!mu_dev || T < 0 || nj < 1 || nl < 0 || (nl > 0 && !edges_dev)) return fail(h, DGP_ERR_INVALID, "dgp_potentials: bad argument");
  if ((ws_dev == nullptr) != (ws_max_dev == nullptr)) return fail(h, DGP_ERR_INVALID, "dgp_potentials: ws and ws_max go together");
  CU_OK(h, cudaSetDevice(h->device));
  CU_OK(h, launch_potentials(mu_dev, mu_halo_next_dev, T, nj, edges_dev, nl, h->cfg.stride, ws_dev, ws_max_dev, wt_max,
                             skel_dist_dev, temporal_dev, e_skel_dev, e_temp_dev, (cudaStream_t)stream));
  h->launches++;
  return DGP_OK;
}

int dgp_estimate_pose_host(dgp_handle* h, const uint8_t* frames_host, int T, int H, int W, int batch, float gamma,
                           float gauss_len, float* mu_host, int32_t* peak_host, float* lik_host) {
  return dgp_estimate_pose_host_transform(h, frames_host, T, H, W, nullptr, batch, gamma, gauss_len, mu_host, peak_host,
                                          lik_host);
}

int dgp_estimate_pose_host_transform(dgp_handle* h, const uint8_t* frames_host, int T, int H0, int W0,
                                     const dgp_frame_transform* transform, int batch, float gamma, float gauss_len,
                                     float* mu_host, int32_t* peak_host, float* lik_host) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->finalized) return fail(h, DGP_ERR_STATE, "dgp_estimate_pose_host before dgp_finalize_weights");
  if (!frames_host || T < 0 || batch < 1 || !mu_host) return fail(h, DGP_ERR_INVALID, "dgp_estimate_pose_host: bad argument");
  int H, W;
  bool identity;
  if (transform_dims(H0, W0, transform, &H, &W, &identity))
    return fail(h, DGP_ERR_INVALID, "dgp_estimate_pose_host: invalid frame size or transform");
  if (T == 0) return DGP_OK;
  CU_OK(h, cudaSetDevice(h->device));
  int rc = h->pose.reserve(h, batch, H0, W0, H, W, identity);
  if (rc) return rc;
  const PoseJob job = {H0, W0, H, W, identity, transform, gamma, gauss_len, mu_host, peak_host, lik_host};
  const size_t frame_bytes = (size_t)H0 * W0 * 3;
  int it = 0;
  for (int t0 = 0; t0 < T; t0 += batch, ++it) {
    const int b = (T - t0) < batch ? (T - t0) : batch;
    // the tail batch of a multi-batch video reuses the full-batch plan (see dgp_estimate_pose_stream): surplus rows hold an
    // earlier batch's frames and their read-outs are not copied back
    const int run_b = (b < batch && it > 0) ? batch : b;
    if ((rc = h->pose.run_batch(h, job, frames_host + (size_t)t0 * frame_bytes, b, run_b, it, t0, nullptr, nullptr))) return rc;
  }
  CU_OK(h, cudaStreamSynchronize(h->stream.get()));
  return DGP_OK;
}

int dgp_debug_keep_activations(dgp_handle* h, int enable) {
  if (!h) return DGP_ERR_INVALID;
  h->debug_keep = enable != 0;
  return DGP_OK;
}

int dgp_debug_get_activation(dgp_handle* h, const char* end_point, float* host_out, size_t max_elems, int64_t* shape4) {
  if (!h || !end_point) return DGP_ERR_INVALID;
  auto it = h->kept.find(end_point);
  if (it == h->kept.end()) return fail(h, DGP_ERR_INVALID, "no kept activation named %s", end_point);
  const auto& k = it->second;
  const size_t n = (size_t)k.N * k.H * k.W * k.C;
  if (shape4) { shape4[0] = k.N; shape4[1] = k.H; shape4[2] = k.W; shape4[3] = k.C; }
  if (!host_out) return DGP_OK;
  if (n > max_elems) return fail(h, DGP_ERR_INVALID, "buffer too small for %s", end_point);
  CU_OK(h, cudaSetDevice(h->device));
  CU_OK(h, cudaDeviceSynchronize());
  std::vector<__nv_bfloat16> tmp(n);
  CU_OK(h, cudaMemcpy(tmp.data(), k.buf.get(), n * 2, cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < n; ++i) host_out[i] = cvt16_to_float(h, tmp[i]);
  return DGP_OK;
}

int dgp_conv2d(dgp_handle* h, const void* x_dev, int N, int H, int W, int Cin, const float* w_host, int R, int S,
               int Cout, int stride, int dilation, int pad_mode, const float* scale_host, const float* shift_host,
               const void* residual_dev, int res_sub, int res_H, int res_W, int relu, void* out_dev, int out_f32,
               int block_n, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!x_dev || !w_host || !out_dev) return fail(h, DGP_ERR_INVALID, "dgp_conv2d: null argument");
  if (Cin % 64 || Cout % 16) return fail(h, DGP_ERR_UNSUPPORTED, "dgp_conv2d: Cin must be a multiple of 64 and Cout of 16");
  CU_OK(h, cudaSetDevice(h->device));
  ConvLayer L;
  L.scope = "dgp_conv2d"; L.R = R; L.S = S; L.Cin = Cin; L.Cout = Cout; L.stride = stride; L.dil = dilation;
  L.relu = relu != 0;
  L.K = R * S * Cin;
  L.block_n = block_n > 0 ? block_n : pick_block_n(Cout);
  L.Npad = ceil_div(Cout, L.block_n) * L.block_n;
  if (L.Npad != Cout) return fail(h, DGP_ERR_INVALID, "dgp_conv2d: block_n must divide Cout");
  std::vector<float> wf((size_t)L.Npad * L.K, 0.0f);
  pack({L.scope, 4, {R, S, Cin, Cout}, VAR_CONV, 0, wf.size()}, w_host, wf.data());
  std::vector<W16> wm(wf.size());
  for (size_t i = 0; i < wf.size(); ++i) wm[i] = cvt16(h, wf[i]);
  DevBuf w, scale, shift;
  CU_OK(h, w.alloc(wm.size() * sizeof(__nv_bfloat16)));
  CU_OK(h, cudaMemcpy(w.get(), wm.data(), wm.size() * sizeof(__nv_bfloat16), cudaMemcpyHostToDevice));
  if (scale_host) {
    CU_OK(h, scale.alloc(Cout * sizeof(float)));
    CU_OK(h, cudaMemcpy(scale.get(), scale_host, Cout * sizeof(float), cudaMemcpyHostToDevice));
  }
  if (shift_host) {
    CU_OK(h, shift.alloc(Cout * sizeof(float)));
    CU_OK(h, cudaMemcpy(shift.get(), shift_host, Cout * sizeof(float), cudaMemcpyHostToDevice));
  }
  L.w = w.get<__nv_bfloat16>();
  L.scale = scale.get<float>();
  L.shift = shift.get<float>();
  Step st;
  int Ho, Wo;
  int rc = make_gemm_step(h, L, x_dev, N, H, W, pad_mode, out_dev, out_f32 != 0, (const __nv_bfloat16*)residual_dev,
                          res_sub > 0 ? res_sub : 1, res_H, res_W, 0, &st, &Ho, &Wo);
  if (rc) return rc;
  h->launches++;
  CU_OK(h, launch_conv_gemm(st.gp, h->num_sms, (cudaStream_t)stream));
  CU_OK(h, cudaStreamSynchronize((cudaStream_t)stream));
  return DGP_OK;
}

int dgp_conv2d_wgrad(dgp_handle* h, const void* x_dev, int N, int H, int W, int Cin, const void* dy_dev, int R, int S,
                     int Cout, int stride, int dilation, int pad_mode, float* dw_dev, const int32_t* dbg3, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!x_dev || !dy_dev || !dw_dev) return fail(h, DGP_ERR_INVALID, "dgp_conv2d_wgrad: null argument");
  if (Cin % 64 || Cout % 8) return fail(h, DGP_ERR_UNSUPPORTED, "dgp_conv2d_wgrad: Cin must be a multiple of 64 and Cout of 8");
  CU_OK(h, cudaSetDevice(h->device));
  WgradParams wp;
  int rc = make_wgrad_params(h, "dgp_conv2d_wgrad", R, S, Cin, Cout, stride, dilation, x_dev, N, H, W, pad_mode, dy_dev, &wp);
  if (rc) return rc;
  if (dbg3) { wp.dbg_lbo = (uint32_t)dbg3[0]; wp.dbg_sbo = (uint32_t)dbg3[1]; wp.dbg_kstep = (uint32_t)dbg3[2]; }
  DevBuf ws;
  CU_OK(h, ws.alloc(wgrad_workspace_bytes(wp)));
  wp.partials = ws.get<float>();
  h->launches += 2;
  CU_OK(h, launch_wgrad_gemm(wp, h->num_sms, (cudaStream_t)stream));
  CU_OK(h, launch_wgrad_reduce(wp, nullptr, nullptr, dw_dev, nullptr, (cudaStream_t)stream));
  CU_OK(h, cudaStreamSynchronize((cudaStream_t)stream));
  return DGP_OK;
}

int dgp_set_profiling(dgp_handle* h, int enable) {
  if (!h) return DGP_ERR_INVALID;
  h->profiling = enable != 0;
  h->profile_brackets = enable == 2;
  return DGP_OK;
}

int dgp_get_profile(dgp_handle* h, double* ms_by_kind, int64_t* count_by_kind, int nkinds) {
  if (!h || !ms_by_kind || !count_by_kind || nkinds < 1) return DGP_ERR_INVALID;
  CU_OK(h, cudaSetDevice(h->device));
  CU_OK(h, cudaDeviceSynchronize());
  for (int i = 0; i < nkinds; ++i) { ms_by_kind[i] = 0.0; count_by_kind[i] = 0; }
  for (auto& r : h->prof) {
    float ms = 0.0f;
    if (cudaEventElapsedTime(&ms, r.a.get(), r.b.get()) == cudaSuccess && r.kind < nkinds) {
      ms_by_kind[r.kind] += ms;
      count_by_kind[r.kind] += r.count;
    }
    h->ev_pool.push_back(std::move(r.a));
    h->ev_pool.push_back(std::move(r.b));
  }
  h->prof.clear();
  return DGP_OK;
}

int dgp_get_profile_records(dgp_handle* h, float* ms, int32_t* kind, int max_records, int* n_records) {
  if (!h || !ms || !kind || !n_records || max_records < 0) return DGP_ERR_INVALID;
  CU_OK(h, cudaSetDevice(h->device));
  CU_OK(h, cudaDeviceSynchronize());
  int n = 0;
  for (auto& r : h->prof) {
    float t = 0.0f;
    if (n < max_records && cudaEventElapsedTime(&t, r.a.get(), r.b.get()) == cudaSuccess) {
      ms[n] = t;
      kind[n] = r.kind;
      ++n;
    }
    h->ev_pool.push_back(std::move(r.a));
    h->ev_pool.push_back(std::move(r.b));
  }
  h->prof.clear();
  *n_records = n;
  return DGP_OK;
}

uint32_t dgp_crc32c(const void* data, size_t n) {
  // CRC-32C (Castagnoli, reflected polynomial 0x82F63B78), host only: the per-tensor checksums of TensorFlow checkpoint bundles
  static uint32_t table[256];
  static bool init = false;
  if (!init) {
    for (uint32_t i = 0; i < 256; ++i) {
      uint32_t c = i;
      for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ 0x82F63B78u : c >> 1;
      table[i] = c;
    }
    init = true;
  }
  const unsigned char* p = static_cast<const unsigned char*>(data);
  uint32_t crc = 0xFFFFFFFFu;
  for (size_t i = 0; i < n; ++i) crc = table[(crc ^ p[i]) & 0xFF] ^ (crc >> 8);
  return crc ^ 0xFFFFFFFFu;
}

int64_t dgp_launch_count(const dgp_handle* h) { return h ? h->launches : 0; }
int dgp_num_sms(const dgp_handle* h) { return h ? h->num_sms : 0; }

int dgp_debug_live_resources(int64_t* objects, int64_t* device_bytes) {
  if (objects) *objects = g_live_objects;
  if (device_bytes) *device_bytes = g_live_device_bytes;
  return DGP_OK;
}

}  // extern "C"
