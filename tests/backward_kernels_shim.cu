// Test-only C wrappers around the library's internal launchers (namespace dgp of libdgp_b200.so), so that
// tests/test_gpu_backward_kernels.py can run each training-backward and parameter kernel on its own.  Every pointer is a
// device pointer owned by torch; nothing here allocates or copies.  Return values are the launchers' own (cudaError_t or
// DGP status).
#include "../deepgraphpose_b200/csrc/handle.cuh"

namespace {
cudaStream_t st(void* s) { return reinterpret_cast<cudaStream_t>(s); }
}  // namespace

extern "C" {

int shim_sizeof_wgrad_params() { return (int)sizeof(WgradParams); }
int shim_sizeof_bn_group() { return (int)sizeof(BnGroup); }
int shim_sizeof_dgrad_w_job() { return (int)sizeof(DgradWJob); }
int shim_max_dgrad_w_jobs() { return kDgradWMaxJobs; }

// The dgrad GEMM of a backward step with its consumer's ReLU mask: the step as add_dgrad builds it (stride 1, R x R taps at
// dilation dil, weights w [N][R*R*K]) and mask_act / colsum_part set as push_dgrad_gemm sets them.  info = {epi_mode, msub,
// cta2}; the mask rides in the epilogue only with epi_mode 1.
int shim_masked_dgrad(dgp_handle* h, const void* dy, int nimg, int H, int W, int K, void* w, int N, int R, int dil, void* out,
                      const void* mask_act, float* colsum_part, const void* residual, void* s, int* info) {
  ConvLayer D;
  D.scope = "shim/dgrad";
  D.R = R; D.S = R; D.Cin = K; D.Cout = N; D.stride = 1; D.dil = dil; D.relu = false;
  D.K = R * R * K; D.Npad = N; D.block_n = N >= 256 ? 256 : N;
  D.w = reinterpret_cast<W16*>(w);
  Step step;
  int Ho, Wo;
  int rc = make_gemm_step(h, D, dy, nimg, H, W, R > 1 ? 1 : 0, out, false, reinterpret_cast<const __nv_bfloat16*>(residual), 1, H,
                          W, 0, &step, &Ho, &Wo);
  if (rc) return rc;
  ConvGemmParams g = step.gp;
  info[0] = g.epi_mode; info[1] = g.msub; info[2] = g.cta2;
  if (mask_act != nullptr && g.epi_mode == 1) {
    g.mask_act = mask_act;
    g.colsum_part = colsum_part;
  }
  return (int)launch_conv_gemm(g, dgp_num_sms(h), st(s));
}

// wp: sizeof(WgradParams) bytes of host memory, filled here and read back by the calls below
int shim_make_wgrad_params(dgp_handle* h, int R, int Cin, int Cout, int stride, int dil, const void* x, int nimg, int H, int W,
                           int pad_mode, const void* dy, void* wp) {
  return make_wgrad_params(h, "shim", R, R, Cin, Cout, stride, dil, x, nimg, H, W, pad_mode, dy,
                           reinterpret_cast<WgradParams*>(wp));
}
int shim_make_conv1_wgrad_params(dgp_handle* h, const void* dy, const void* s2d, int B, int H1, int W1, int Hs, int Ws,
                                 void* wp) {
  return make_conv1_wgrad_params(h, dy, s2d, B, H1, W1, Hs, Ws, reinterpret_cast<WgradParams*>(wp));
}
// info = {Cout, Kw, num_m_blocks, num_n_blocks, splits}; returns the workspace bytes
long long shim_wgrad_info(const void* wp, int* info) {
  const WgradParams& p = *reinterpret_cast<const WgradParams*>(wp);
  info[0] = p.Cout; info[1] = p.Kw; info[2] = p.num_m_blocks; info[3] = p.num_n_blocks; info[4] = p.splits;
  return (long long)wgrad_workspace_bytes(p);
}
int shim_wgrad_gemm(dgp_handle* h, const void* wp, float* partials, void* s) {
  WgradParams p = *reinterpret_cast<const WgradParams*>(wp);
  p.partials = partials;
  return (int)launch_wgrad_gemm(p, dgp_num_sms(h), st(s));
}
int shim_wgrad_reduce(const void* wp, float* partials, const float* rowscale, const float* mask, float* grad,
                      const GradMode* mode, const float* wmaster, float* rowdot_part, void* s) {
  WgradParams p = *reinterpret_cast<const WgradParams*>(wp);
  p.partials = partials;
  return (int)launch_wgrad_reduce(p, rowscale, mask, grad, mode, st(s), wmaster, rowdot_part);
}

int shim_prep_s2d(const uint8_t* frames, int N, int H, int W, const float* mean3_host, void* out, int Hs, int Ws, int fp16,
                  void* s) {
  return (int)launch_prep_s2d(frames, N, H, W, mean3_host, reinterpret_cast<__nv_bfloat16*>(out), Hs, Ws, fp16, st(s));
}

int shim_relu_bn_bwd_blocks(int M, int C) { return relu_bn_bwd_blocks(M, C); }
int shim_relu_bn_bwd(void* g, const void* act, int M, int C, float* partial, int fp16, const void* d, int H, int W, int P, int Q,
                     void* s) {
  return (int)launch_relu_bn_bwd(g, act, M, C, partial, fp16, st(s), d, H, W, P, Q);
}

int shim_maxpool_relu_bwd_rows(int N, int H, int W) { return maxpool_relu_bwd_rows(N, H, W); }
int shim_maxpool_relu_bwd(const void* x, const void* gout, int N, int H, int W, int Ho, int Wo, int pad_t, int pad_l, void* gx,
                          float* partial, int fp16, void* s) {
  return (int)launch_maxpool_relu_bwd(x, gout, N, H, W, 64, Ho, Wo, pad_t, pad_l, gx, partial, fp16, st(s));
}

int shim_bn_finalize_all(const BnGroup* table, int ngroups, const float* part, const float* rowdot, const float* mean,
                         const float* var, float eps, float* dgamma, float* dbeta, const GradMode* mode, void* s) {
  return (int)launch_bn_finalize_all(table, ngroups, part, rowdot, mean, var, eps, dgamma, dbeta, mode, st(s));
}

int shim_upsample2(const void* in, int N, int P, int Q, int C, void* out, int H, int W, void* s) {
  return (int)launch_upsample2(in, N, P, Q, C, out, H, W, st(s));
}
int shim_col2im_bwd(const float* g_logits, const float* g_locref, int N, int h, int w, int ctot, int nj, void* dG, int Kd, int fp16,
                    void* s) {
  return (int)launch_col2im_bwd(g_logits, g_locref, N, h, w, ctot, nj, dG, Kd, fp16, st(s));
}
int shim_head_bias_blocks() { return head_bias_blocks(); }
int shim_head_bias_grad(const float* g, long long npix, int C, float* partial, float* dbias, const GradMode* mode, void* s) {
  return (int)launch_head_bias_grad(g, (size_t)npix, C, partial, dbias, mode, st(s));
}
int shim_scale_inplace(float* x, long long n, float scale, void* s) {
  return (int)launch_scale_inplace(x, (size_t)n, scale, st(s));
}

int shim_build_dgrad_w(const DgradWJob* jobs, int njobs, int total_tiles, const float* master, const float* scale, int fp16,
                       void* s) {
  return (int)launch_build_dgrad_w(jobs, njobs, total_tiles, master, scale, fp16, st(s));
}
int shim_build_head_dgrad_w(const float* wh, int rows, int C, void* whT, int Kd, int fp16, void* s) {
  return (int)launch_build_head_dgrad_w(wh, rows, C, whT, Kd, fp16, st(s));
}
int shim_refresh_w16(const float* master, void* w16, long long n, int fp16, void* s) {
  return (int)launch_refresh_w16(master, w16, (size_t)n, fp16, st(s));
}
int shim_refresh_bn(const float* gamma, const float* beta, const float* mean, const float* var, float eps, int n, float* scale,
                    float* shift, void* s) {
  return (int)launch_refresh_bn(gamma, beta, mean, var, eps, n, scale, shift, st(s));
}
int shim_sqnorm_partials() { return sqnorm_partials(); }
int shim_global_norm(const float* g, long long n, float grad_scale, float clip, float* partial, float* norm_clip, void* s) {
  return (int)launch_global_norm(g, (size_t)n, grad_scale, clip, partial, norm_clip, st(s));
}

}  // extern "C"
