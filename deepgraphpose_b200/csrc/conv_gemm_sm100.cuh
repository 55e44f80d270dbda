// Implicit-GEMM convolution on tcgen05 tensor cores (sm_100a) -- host-visible declarations.
//
// One kernel serves every GEMM-shaped layer of the DLC ResNet-50 pose net
// (reference: slim resnet_v1_50 called at
//  /root/reference/src/DeepLabCut/deeplabcut/pose_estimation_tensorflow/nnet/pose_net.py:50-52 and the
//  deconv heads at pose_net.py:18-26):
//    D[m, n] = sum_k A[m, k] * B[n, k],  m = output pixel (n_img, p, q) linearised, n = output channel,
//    k = (r, s, c) with the channel innermost.
//  A is fetched by TMA either as a plain [M, K] matrix (1x1 convs, deconv-as-GEMM) or in im2col mode
//  (3x3 convs with stride / dilation / TF padding, and conv1 after the space-to-depth transform);
//  B (weights, [Cout, K] K-major bf16) is a plain 2-D TMA tile.  Accumulation is fp32 in TMEM; the
//  epilogue applies the frozen-BN scale/shift in fp32, adds the (optionally 2x-subsampled) residual,
//  applies ReLU and stores bf16 (or fp32 for the head GEMM).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.cuh"

namespace dgp {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;  // 64 bf16 = 128 B = one SWIZZLE_128B row

constexpr int kEpiUnitCols = 32;    // 16-bit columns per epilogue staging unit (64 B rows, SWIZZLE_64B)

struct ConvGemmParams {
  CUtensorMap tmap_a;
  CUtensorMap tmap_b;
  CUtensorMap tmap_out;  // epi_mode 1: [M, N] 16-bit, box 32 columns x 32 rows, SWIZZLE_64B
  CUtensorMap tmap_res;  // epi_mode 1 with residual: same box over the residual tensor (tiled or im2col stride 2)
  int M;             // output pixels
  int N;             // output channels (multiple of block_n)
  int block_n;       // UMMA N (multiple of 16, 16..256)
  int msub;          // 128-row sub-tiles per CTA tile: 1, or 2 (BLOCK_M = 256) for narrow layers (block_n <= 128)
  int num_k_blocks;  // K / 64
  int a_mode;        // 0 = tiled [M,K], 1 = im2col, 2 = im2col by 2-D patches (conv1 fused with the 3x3/2 max-pool),
                     // 3 = shared-memory resident input patch (3x3 stride-1 convs with 64 input channels): ONE tiled TMA box
                     //     per tile, the nine taps are row-shifted UMMA descriptors over it, all weights stay resident
  int fp16;          // 0 = bf16 activations/weights (default), 1 = fp16 storage (same kind::f16 MMA, fp32 accumulate)
  // im2col geometry (a_mode == 1)
  int P, Q;          // output height / width
  int conv_stride;
  int lower_h, lower_w;  // TMA lower corner = -pad_beg
  int S;             // filter width (taps are enumerated r-major: tap = r * S + s)
  int dil;
  int cblocks;       // Cin / 64
  // epilogue
  const float* scale;  // [N] or nullptr (=1)
  const float* shift;  // [N] or nullptr (=0)
  int epi_mode;      // 0 = direct register->global stores (fp32 head GEMM), 1 = TMA-staged 16-bit (+ TMA residual),
                     // 2 = BN + ReLU + 3x3 stride-2 max-pool of a 2-D patch (a_mode 2), pooled pixels stored directly,
                     // 3 = direct masked 16-bit stores of a patch tile (a_mode 3)
  int epi_bufs;      // 2 KB staging buffers per epilogue warp (epi_mode 1): 1 or 2; the residual prefetch runs epi_bufs-1 units ahead
  const __nv_bfloat16* residual;  // nullptr = none
  int res_sub;       // 1 = same pixel grid as the output, 2 = residual grid is (res_H, res_W), read at (2p, 2q)
  int res_H, res_W;
  int ldres;         // residual row stride (elements)
  int relu;
  // epi_mode 1, backward pass: the consumer's ReLU mask and dbeta sums fused into this (dgrad) GEMM's epilogue --
  // out = value * [mask_act > 0] and colsum_part[row / 32][n] = sum over the 32 rows of a unit of the stored 16-bit values
  const void* mask_act;   // 16-bit [M, ldc] post-ReLU activation of the tensor whose gradient this GEMM produces, or nullptr
  float* colsum_part;     // fp32 [ceil(M / 32), N]
  void* out;         // bf16 or fp32, row-major [M, ldc]
  int out_f32;
  int ldc;
  int num_m_blocks, num_n_blocks;
  int num_stages;
  int cta2;          // 1 = CTA-pair kernel (cluster of 2, tcgen05 cta_group::2): tiles of 256 rows x 256 columns, each CTA stages
                     // its 128 rows of A and 128 of the 256 weight rows; num_m_blocks counts 256-row tiles
  int tmem_cols;     // power of two >= 2 * block_n
  // a_mode / epi_mode 2 (conv1 + pool1): a tile is the (2R+1) x (2C+1) patch of conv outputs under R x C pooled pixels;
  // P, Q are the conv output dims, pool_H / pool_W the pooled dims, pool_pad_* the TF SAME padding of the pool (0 or 1)
  int pool_R, pool_C, pool_H, pool_W, pool_pad_t, pool_pad_l, pool_tiles_i, pool_tiles_j;
  // a_mode 3: output tile = pt_rows x pt_cols pixels (tile grid pool_tiles_i x pool_tiles_j per image); accumulator row
  // m = r * pt_wp + c over the INPUT patch grid (pt_wp = pt_cols + 2 * dil columns), so tap (kr, ks) reads smem rows
  // m + (kr * pt_wp + ks) * dil: a constant shift of the descriptor start address
  int pt_rows, pt_cols, pt_wp, pt_stage_bytes, pt_base_offset_mode;
};

// Weight-gradient GEMM (wgrad_gemm_sm100.cu): dW[co, kk] = sum_p dy[p, co] * xcol[p, kk], kk = (tap, ci).
struct WgradParams {
  CUtensorMap tmap_dy;  // [pixels, Cout] 16-bit, box 64 ch x 64 pixels, SWIZZLE_128B (rows/cols past the end read as zero)
  CUtensorMap tmap_x;   // x_mode 0: [pixels, Cin] tiled; x_mode 1: im2col (same geometry as the forward conv), 64 pixels per column
  int Cout, Kw;         // gradient matrix [Cout][Kw], Kw = taps * Cin (multiple of 64)
  int num_pix_blocks;   // ceil(pixels / 64)
  int x_mode;
  int fp16;
  int P, Q, conv_stride, lower_h, lower_w, S, dil, cblocks;  // im2col geometry (x_mode 1); cblocks = Cin / 64
  int num_m_blocks, num_n_blocks, splits, kb_per_split;      // filled by wgrad_plan
  float* partials;      // workspace: [num_m_blocks * num_n_blocks * splits][128][256] fp32
  uint32_t dbg_lbo, dbg_sbo, dbg_kstep;  // 0 = defaults (descriptor bring-up hooks)
};
void wgrad_plan(WgradParams* p, int num_sms);
size_t wgrad_workspace_bytes(const WgradParams& p);
cudaError_t launch_wgrad_gemm(const WgradParams& p, int num_sms, cudaStream_t stream);
// grad[co][kk] = rowscale[co] * mask[co][kk] * sum over splits (fixed order), stored through `mode` (nullptr: overwrite);
// rowscale / mask may be null.
// wmaster / rowdot_part (optional): also write <W[co, 4 kk], dW_raw[co, 4 kk]> per float4 of the row (Cout * Kw / 4 floats)
cudaError_t launch_wgrad_reduce(const WgradParams& p, const float* rowscale, const float* mask, float* grad,
                                const GradMode* mode, cudaStream_t stream, const float* wmaster = nullptr,
                                float* rowdot_part = nullptr);

// Host helpers (conv_gemm_sm100.cu)
void tmap_set_fp16(int fp16);  // element type of subsequently encoded tensor maps
const char* tma_init();  // resolves the driver's tensor-map encoders; returns nullptr on success, else an error string
// [rows, k] row-major 16-bit matrix, box = [box_rows, box_cols]: 64 columns -> SWIZZLE_128B, 32 columns -> SWIZZLE_64B.
const char* make_tmap_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t k, uint64_t row_stride_bytes,
                         uint32_t box_rows, uint32_t box_cols = kBlockK);
// NHWC-like activation tensor for im2col loads: dims (C, W, H, N) with explicit byte strides for W, H, N.
const char* make_tmap_im2col(CUtensorMap* out, const void* base, uint64_t C, uint64_t W, uint64_t H, uint64_t N,
                             uint64_t stride_w_bytes, uint64_t stride_h_bytes, uint64_t stride_n_bytes, int lower_w,
                             int lower_h, int upper_w, int upper_h, int conv_stride, uint64_t total_bytes,
                             uint32_t pixels_per_column = kBlockM, uint32_t channels_per_pixel = kBlockK);
// a_mode 3: patch stage bytes (1024-aligned) for a tile geometry, and the tiled 4-D activation map (box = whole input patch)
int conv_patch_stage_bytes(int pt_wp, int dil);
// C = 64 channels per pixel (128 B rows, SWIZZLE_128B)
const char* make_tmap_tiled4d(CUtensorMap* out, const void* base, uint64_t C, uint64_t W, uint64_t H, uint64_t N,
                              uint64_t stride_w_bytes, uint64_t stride_h_bytes, uint64_t stride_n_bytes, uint32_t box_w,
                              uint32_t box_h);
size_t conv_gemm_smem_bytes(const ConvGemmParams& p);   // uses block_n, num_stages, epi_*, msub, a_mode, pt_stage_bytes, num_k_blocks
int conv_gemm_pick_stages(ConvGemmParams p);            // largest num_stages (<= 8) that fits 227 KB
cudaError_t launch_conv_gemm(const ConvGemmParams& p, int num_sms, cudaStream_t stream);

}  // namespace dgp
