// Boundary entry points that expose the two halves of the forward the way the reference's PoseNet does
// (PTF/nnet/pose_net.py:36-54 extract_features, :18-26 / :56-78 prediction_layer(s)) and a stand-alone 3x3 stride-2
// transposed convolution for dgp_prediction_layer (src/deepgraphpose/models/fitdgp_util.py:18-74).  The hot path keeps using
// the fused dgp_forward; these exist so that code written against the reference's method names finds them.
#include "../../include/dgp_b200.h"

#include <cuda_runtime.h>

#include <vector>

#include "handle.cuh"

using namespace dgp;

extern "C" {

int dgp_extract_features(dgp_handle* h, const uint8_t* frames_dev, int B, int H, int W, float* net_dev, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->finalized) return fail(h, DGP_ERR_STATE, "dgp_extract_features before dgp_finalize_weights");
  if (!frames_dev || !net_dev || B < 1 || H < 32 || W < 32) return fail(h, DGP_ERR_INVALID, "dgp_extract_features: bad argument");
  CU_OK(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  Plan* pl = nullptr;
  int rc = build_plan(h, B, H, W, false, &pl);
  if (rc) return rc;
  if ((rc = run_forward_plan(h, pl, frames_dev, nullptr, nullptr, s, 0, pl->head_step))) return rc;
  CU_OK(h, launch_cvt16_to_f32(pl->feat, net_dev, (size_t)B * pl->hf * pl->wf * 2048, h->fp16, s));
  h->launches++;
  return DGP_OK;
}

int dgp_prediction_layers(dgp_handle* h, const float* net_dev, int B, int hf, int wf, float* logits_dev, float* locref_dev,
                          void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!h->finalized) return fail(h, DGP_ERR_STATE, "dgp_prediction_layers before dgp_finalize_weights");
  if (!net_dev || !logits_dev || B < 1 || hf < 1 || wf < 1) return fail(h, DGP_ERR_INVALID, "dgp_prediction_layers: bad argument");
  if (locref_dev && !h->cfg.location_refinement)
    return fail(h, DGP_ERR_INVALID, "dgp_prediction_layers: locref requested but the head was not built");
  CU_OK(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  const ConvLayer& L = h->layers[h->head_layer];
  const size_t npix = (size_t)B * hf * wf;
  DevBuf x16, contrib;
  CU_OK(h, x16.alloc(npix * 2048 * 2 + 1024));
  CU_OK(h, contrib.alloc(npix * L.Npad * 4));
  Step st;
  int dh, dw;
  CU_OK(h, launch_f32_to_cvt16(net_dev, x16.get(), npix * 2048, h->fp16, s));
  int rc = make_gemm_step(h, L, x16.get(), B, hf, wf, 0, contrib.get(), true, nullptr, 1, 0, 0, 0, &st, &dh, &dw);
  if (rc) return rc;
  h->launches += 3;
  CU_OK(h, launch_conv_gemm(st.gp, h->num_sms, s));
  CU_OK(h, launch_deconv_col2im(contrib.get<float>(), B, hf, wf, L.Npad, h->ctot, h->cfg.num_joints, h->head_bias, logits_dev,
                                locref_dev, s));
  CU_OK(h, cudaStreamSynchronize(s));
  return DGP_OK;
}

int dgp_softmax_threshold(dgp_handle* h, float* map_dev, int B, int H, int W, int nj, float th, float* mu_dev, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (B == 0) return DGP_OK;
  if (!map_dev || B < 0 || H < 1 || W < 1 || nj < 1 || !(th >= 0.0f))
    return fail(h, DGP_ERR_INVALID, "dgp_softmax_threshold: bad argument");
  CU_OK(h, cudaSetDevice(h->device));
  CU_OK(h, launch_softmax_threshold(map_dev, B, H, W, nj, th, mu_dev, (cudaStream_t)stream));
  h->launches++;
  return DGP_OK;
}

int dgp_deconv2d(dgp_handle* h, const float* x_dev, int N, int H, int W, int Cin, const float* w_host, const float* bias_host,
                 int Cout, float* out_dev, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  if (!x_dev || !w_host || !out_dev || N < 1 || H < 1 || W < 1 || Cout < 1)
    return fail(h, DGP_ERR_INVALID, "dgp_deconv2d: bad argument");
  if (Cin % 64) return fail(h, DGP_ERR_UNSUPPORTED, "dgp_deconv2d: input channels must be a multiple of 64");
  CU_OK(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  // the same packing as the network's own heads, with this one head as all of the GEMM's channels
  ConvLayer L;
  L.scope = "dgp_deconv2d"; L.R = 1; L.S = 1; L.Cin = Cin; L.Cout = 9 * Cout; L.relu = false;
  L.K = Cin;
  L.block_n = pick_block_n(9 * Cout);
  L.Npad = ceil_div(9 * Cout, L.block_n) * L.block_n;
  std::vector<float> wf((size_t)L.Npad * Cin, 0.0f);
  pack({L.scope, 4, {3, 3, Cout, Cin}, VAR_HEAD, 0, wf.size(), Cout, 0}, w_host, wf.data());
  std::vector<W16> wm(wf.size());
  for (size_t i = 0; i < wf.size(); ++i) wm[i] = cvt16(h, wf[i]);
  const size_t npix = (size_t)N * H * W;
  DevBuf x16, w16, contrib, bias;
  CU_OK(h, x16.alloc(npix * Cin * 2 + 1024));
  CU_OK(h, w16.alloc(wm.size() * 2));
  CU_OK(h, contrib.alloc(npix * L.Npad * 4));
  if (bias_host) CU_OK(h, bias.alloc((size_t)Cout * 4));
  CU_OK(h, cudaMemcpyAsync(w16.get(), wm.data(), wm.size() * 2, cudaMemcpyHostToDevice, s));
  if (bias_host) CU_OK(h, cudaMemcpyAsync(bias.get(), bias_host, (size_t)Cout * 4, cudaMemcpyHostToDevice, s));
  CU_OK(h, launch_f32_to_cvt16(x_dev, x16.get(), npix * Cin, h->fp16, s));
  L.w = w16.get<__nv_bfloat16>();
  Step st;
  int dh, dw;
  int rc = make_gemm_step(h, L, x16.get(), N, H, W, 0, contrib.get(), true, nullptr, 1, 0, 0, 0, &st, &dh, &dw);
  if (rc) return rc;
  h->launches += 3;
  CU_OK(h, launch_conv_gemm(st.gp, h->num_sms, s));
  CU_OK(h, launch_deconv_col2im(contrib.get<float>(), N, H, W, L.Npad, Cout, Cout, bias.get<float>(), out_dev, nullptr, s));
  CU_OK(h, cudaStreamSynchronize(s));
  return DGP_OK;
}

}  // extern "C"
