// The handle's trainable variables: their TF names and shapes, where each lives in the parameter arena, and the one
// conversion between a variable's TF / slim layout and its arena span.  dgp_finalize_weights packs the loaded checkpoint
// with it, dgp_get_variable / dgp_set_variable read and write single variables through it.
#include "../../include/dgp_b200.h"

#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "handle.cuh"

using namespace dgp;

namespace dgp {

size_t tf_elems(const ArenaVar& v) {
  size_t n = 1;
  for (int i = 0; i < v.ndim; ++i) n *= (size_t)v.shape[i];
  return n;
}

std::string shape_str(const ArenaVar& v) {
  std::string s = "[";
  for (int i = 0; i < v.ndim; ++i) s += (i ? "," : "") + std::to_string(v.shape[i]);
  return s + "]";
}

namespace {

// f(tf index, span index) for every element of the variable: the index arithmetic of each layout, written once.
template <class F>
void for_each_element(const ArenaVar& v, F f) {
  switch (v.layout) {
    case VAR_VECTOR:
      for (size_t i = 0; i < (size_t)v.shape[0]; ++i) f(i, i);
      break;
    case VAR_CONV: {
      const size_t K = (size_t)v.shape[0] * v.shape[1] * v.shape[2], cout = (size_t)v.shape[3];
      for (size_t k = 0; k < K; ++k)
        for (size_t o = 0; o < cout; ++o) f(k * cout + o, o * K + k);
      break;
    }
    case VAR_CONV1_S2D:
      // conv1 runs as a 4x4 stride-1 conv on the 2x2 space-to-depth image (build_conv1_layer): tap (kh, kw) is window
      // row kh/2, window pixel kw/2 and s2d channel ((kh%2)*2 + kw%2)*3 + c of the 256-wide row; taps past 7 stay zero.
      for (int kh = 0; kh < 7; ++kh)
        for (int kw = 0; kw < 7; ++kw)
          for (int c = 0; c < 3; ++c)
            for (int o = 0; o < 64; ++o)
              f((((size_t)kh * 7 + kw) * 3 + c) * 64 + o,
                (size_t)o * 256 + (kh >> 1) * 64 + (kw >> 1) * 16 + ((kh & 1) * 2 + (kw & 1)) * 3 + c);
      break;
    case VAR_HEAD: {
      const size_t cn = (size_t)v.shape[2], cin = (size_t)v.shape[3];
      for (size_t t = 0; t < 9; ++t)
        for (size_t cc = 0; cc < cn; ++cc)
          for (size_t c = 0; c < cin; ++c) f((t * cn + cc) * cin + c, (t * v.ctot + v.c0 + cc) * cin + c);
      break;
    }
  }
}

}  // namespace

void pack(const ArenaVar& v, const float* tf, float* span) {
  for_each_element(v, [&](size_t t, size_t s) { span[s] = tf[t]; });
}

void unpack(const ArenaVar& v, const float* span, float* tf) {
  for_each_element(v, [&](size_t t, size_t s) { tf[t] = span[s]; });
}

void build_variable_table(dgp_handle* h, std::vector<ArenaVar>* frozen) {
  auto add = [h](ArenaVar&& v) {
    h->var_index[v.name] = (int)h->vars.size();
    h->vars.push_back(std::move(v));
  };
  const size_t gamma = h->n_w, beta = h->n_w + h->n_ch, bias = h->n_w + 2 * h->n_ch;
  for (int i = 0; i < (int)h->layers.size(); ++i) {
    if (i == h->head_layer) continue;
    const ConvLayer& L = h->layers[i];
    const size_t C = (size_t)L.Cout;
    if (i == h->conv1_layer) add({L.scope + "/weights", 4, {7, 7, 3, 64}, VAR_CONV1_S2D, L.w_off, 64 * 256});
    else add({L.scope + "/weights", 4, {L.R, L.S, L.Cin, L.Cout}, VAR_CONV, L.w_off, C * L.K});
    add({L.scope + "/BatchNorm/gamma", 1, {L.Cout}, VAR_VECTOR, gamma + L.ch_off, C});
    add({L.scope + "/BatchNorm/beta", 1, {L.Cout}, VAR_VECTOR, beta + L.ch_off, C});
    frozen->push_back({L.scope + "/BatchNorm/moving_mean", 1, {L.Cout}, VAR_VECTOR, (size_t)L.ch_off, C});
    frozen->push_back({L.scope + "/BatchNorm/moving_variance", 1, {L.Cout}, VAR_VECTOR, h->n_ch + L.ch_off, C});
  }
  // both heads share one GEMM matrix and one bias vector: part_pred is channels [0, nj), locref_pred [nj, 3 nj)
  const ConvLayer& L = h->layers[h->head_layer];
  const int nj = h->cfg.num_joints;
  for (int part = 0; part < (h->cfg.location_refinement ? 2 : 1); ++part) {
    const std::string scope = part ? "pose/locref_pred/block4/" : "pose/part_pred/block4/";
    const int cn = part ? 2 * nj : nj, c0 = part ? nj : 0;
    add({scope + "weights", 4, {3, 3, cn, L.Cin}, VAR_HEAD, L.w_off, (size_t)L.Npad * L.Cin, h->ctot, c0});
    add({scope + "biases", 1, {cn}, VAR_VECTOR, bias + c0, (size_t)cn});
  }
}

}  // namespace dgp

extern "C" {

int dgp_get_variable(dgp_handle* h, const char* tf_var_name, int what, float* host_out, size_t max_elems, int64_t* shape4,
                     int* ndim) {
  if (!h || !tf_var_name) return DGP_ERR_INVALID;
  if (!h->finalized) return fail(h, DGP_ERR_STATE, "dgp_get_variable before dgp_finalize_weights");
  if (what < 0 || what > 2) return fail(h, DGP_ERR_INVALID, "dgp_get_variable: what must be 0 (value), 1 (gradient) or 2 (momentum)");
  if (what > 0 && !h->train) return fail(h, DGP_ERR_STATE, "dgp_get_variable: gradients need dgp_train_enable");
  auto it = h->var_index.find(tf_var_name);
  if (it == h->var_index.end()) return fail(h, DGP_ERR_INVALID, "unknown variable %s", tf_var_name);
  const ArenaVar& v = h->vars[it->second];
  const size_t n = tf_elems(v);
  if (shape4) for (int i = 0; i < 4; ++i) shape4[i] = v.shape[i];
  if (ndim) *ndim = v.ndim;
  if (!host_out) return DGP_OK;
  if (n > max_elems) return fail(h, DGP_ERR_INVALID, "buffer too small for %s", tf_var_name);
  float unscale;
  const float* arena = variable_arena(h, what, &unscale);
  CU_OK(h, cudaSetDevice(h->device));
  CU_OK(h, cudaDeviceSynchronize());
  std::vector<float> span(v.len);
  CU_OK(h, cudaMemcpy(span.data(), arena + v.off, v.len * sizeof(float), cudaMemcpyDeviceToHost));
  unpack(v, span.data(), host_out);
  if (unscale != 1.0f)
    for (size_t i = 0; i < n; ++i) host_out[i] *= unscale;
  return DGP_OK;
}

int dgp_set_variable(dgp_handle* h, const char* tf_var_name, int what, const float* host_in, size_t n_elems) {
  if (!h || !tf_var_name || !host_in) return DGP_ERR_INVALID;
  if (!h->finalized) return fail(h, DGP_ERR_STATE, "dgp_set_variable before dgp_finalize_weights");
  if (what != 0 && what != 2) return fail(h, DGP_ERR_INVALID, "dgp_set_variable: what must be 0 (value) or 2 (momentum)");
  if (what == 2 && !h->train) return fail(h, DGP_ERR_STATE, "dgp_set_variable: momentum needs dgp_train_enable");
  auto it = h->var_index.find(tf_var_name);
  if (it == h->var_index.end()) return fail(h, DGP_ERR_INVALID, "unknown variable %s", tf_var_name);
  const ArenaVar& v = h->vars[it->second];
  if (n_elems != tf_elems(v)) return fail(h, DGP_ERR_INVALID, "%s: expected %zu elements", tf_var_name, tf_elems(v));
  float unscale;
  float* arena = variable_arena(h, what, &unscale);
  CU_OK(h, cudaSetDevice(h->device));
  CU_OK(h, cudaDeviceSynchronize());
  std::vector<float> span(v.len);
  CU_OK(h, cudaMemcpy(span.data(), arena + v.off, v.len * sizeof(float), cudaMemcpyDeviceToHost));
  pack(v, host_in, span.data());
  CU_OK(h, cudaMemcpy(arena + v.off, span.data(), v.len * sizeof(float), cudaMemcpyHostToDevice));
  if (what == 0) {  // the tensor-core operands are derived from the master copy
    weights_changed(h);
    int rc = refresh_operands(h, nullptr);
    if (rc) return rc;
    CU_OK(h, cudaDeviceSynchronize());
  }
  return DGP_OK;
}

}  // extern "C"
