// Weight-gradient GEMM of the conv layers on tcgen05 / TMEM / TMA (sm_100a).  See conv_gemm_sm100.cuh (WgradParams).
//
// dW[co, kk] = sum_p dy[p, co] * xcol[p, kk],  kk = (tap, ci) exactly as the forward weight matrix [Cout][taps*Cin],
// p = output pixel.  The reduction dimension is the PIXEL axis, which is the strided axis of both NHWC operands, so
// both shared-memory operands are "MN-major" (channel-contiguous) UMMA tiles: the very same TMA boxes the forward
// kernel loads (64 pixels x 64 channels, SWIZZLE_128B; tiled for dy and 1x1 convs, im2col mode for k x k convs with
// stride / dilation / padding resolved by the TMA unit) are consumed with a transposed interpretation:
//     A = dy tile   [64 pixels (K)] x [128 co (M)]      = 2 boxes,
//     B = xcol tile [64 pixels (K)] x [<=256 kk (N)]    = up to 4 boxes, one per (tap, 64-channel block).
// Work item = (128-row block of Cout, 256-column block of kk, pixel split).  Each item accumulates its pixel range in
// TMEM and writes ONE fp32 partial tile to a workspace; wgrad_reduce_kernel then sums the splits in a fixed order
// (deterministic: no atomics), applies the frozen-BN scale of the output channel (dz = scale * dy) and the optional
// structural mask (conv1's space-to-depth zero taps, padded head rows) and stores the gradient in the parameter arena.
//
// CTA = 192 threads: warp 0 TMA producer, warp 1 MMA issuer, warps 2..5 epilogue (one per TMEM lane quadrant).
#include "conv_gemm_sm100.cuh"

#include <stdio.h>

#include "ptx_sm100.cuh"

namespace dgp {

namespace {

constexpr int kWgThreads = 192;
constexpr int kWgStages = 4;
constexpr int kBoxBytes = 64 * 64 * 2;            // 64 pixels x 64 channels, 8 KiB
constexpr int kWgABytes = 2 * kBoxBytes;          // 128 output channels
constexpr int kWgBBytes = 4 * kBoxBytes;          // up to 256 kk columns
constexpr int kWgStageBytes = kWgABytes + kWgBBytes;

// MN-major SWIZZLE_128B operand descriptor: 64 contiguous elements along M/N per 128 B row, 8-row (K) atoms `sbo`
// bytes apart, 64-element M/N blocks `lbo` bytes apart (cute::UMMA canonical layout ((T,8,m),(8,k)):((1,T,LBO),(8T,SBO))).
__device__ __forceinline__ uint64_t make_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

template <bool kFp16>
__global__ void __launch_bounds__(kWgThreads, 1) wgrad_gemm_kernel(const __grid_constant__ WgradParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kWgStages * kWgStageBytes);
  uint64_t* empty_bar = full_bar + kWgStages;
  uint64_t* tmem_full_bar = empty_bar + kWgStages;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&p.tmap_dy);
    ptx::prefetch_tmap(&p.tmap_x);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kWgStages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tmem_full_bar[a], 1);
      ptx::mbar_init(&tmem_empty_bar[a], 4);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, 512u);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int splits = p.splits, nnb = p.num_n_blocks;
  const int num_items = p.num_m_blocks * nnb * splits;
  const int total_chunks = p.Kw >> 6;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    int stage = 0;
    uint32_t phase = 0;
    const int PQ = p.P * p.Q, Q = p.Q;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
      const int s = item % splits;
      const int t = item / splits;
      const int n_blk = t % nnb;
      const int m_blk = t / nnb;
      const int rem_chunks = total_chunks - n_blk * 4;
      const int nchunks = rem_chunks < 4 ? rem_chunks : 4;
      const int kb0 = s * p.kb_per_split;
      int kb1 = kb0 + p.kb_per_split;
      if (kb1 > p.num_pix_blocks) kb1 = p.num_pix_blocks;
      const uint32_t tx_bytes = (uint32_t)((2 + nchunks) * kBoxBytes);
      // Lane-parallel issue: lanes 0..3 own the (up to 4) x boxes, lanes 4 and 5 the two dy boxes.  Everything that does not
      // depend on the pixel block (channel block, tap offsets, smem slot) is computed once per item; the pixel coordinates
      // advance incrementally (no divisions inside the k loop -- they sat on the single-warp critical path).
      const bool x_lane = lane < nchunks, dy_lane = lane == 4 || lane == 5;
      int my_c0 = 0, my_off_w = 0, my_off_h = 0, my_slot = 0;
      if (x_lane) {
        const int gc = n_blk * 4 + lane;
        const int tap = gc / p.cblocks;
        my_c0 = (gc - tap * p.cblocks) * 64;
        const int tr = tap / p.S;
        my_off_w = (tap - tr * p.S) * p.dil;
        my_off_h = tr * p.dil;
        my_slot = kWgABytes + lane * kBoxBytes;
      } else if (dy_lane) {
        my_c0 = m_blk * 128 + (lane - 4) * 64;
        my_slot = (lane - 4) * kBoxBytes;
      }
      int pix0 = kb0 * 64;
      int img = pix0 / PQ;
      int pp = (pix0 - img * PQ) / Q;
      int qq = pix0 - img * PQ - pp * Q;
      for (int kb = kb0; kb < kb1; ++kb) {
        ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* st = smem + stage * kWgStageBytes;
        if (lane == 0) ptx::mbar_arrive_expect_tx(&full_bar[stage], tx_bytes);
        __syncwarp();
        if (dy_lane || (x_lane && p.x_mode == 0)) {
          ptx::tma_load_2d(st + my_slot, dy_lane ? &p.tmap_dy : &p.tmap_x, &full_bar[stage], my_c0, pix0);
        } else if (x_lane) {
          ptx::tma_load_im2col_4d(st + my_slot, &p.tmap_x, &full_bar[stage], my_c0, qq * p.conv_stride + p.lower_w,
                                  pp * p.conv_stride + p.lower_h, img, (uint16_t)my_off_w, (uint16_t)my_off_h);
        }
        pix0 += 64;
        qq += 64;
        while (qq >= Q) {
          qq -= Q;
          if (++pp == p.P) {
            pp = 0;
            ++img;
          }
        }
        if (++stage == kWgStages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    const uint32_t smem_base = ptx::smem_u32(smem);
    const uint32_t kstep = p.dbg_kstep ? p.dbg_kstep : 2048u;  // 16 pixel rows of 128 B
    const uint32_t lbo = p.dbg_lbo ? p.dbg_lbo : (uint32_t)kBoxBytes;
    const uint32_t sbo = p.dbg_sbo ? p.dbg_sbo : 1024u;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
      const int s = item % splits;
      const int t = item / splits;
      const int n_blk = t % nnb;
      const int rem_chunks = total_chunks - n_blk * 4;
      const int nchunks = rem_chunks < 4 ? rem_chunks : 4;
      const int kb0 = s * p.kb_per_split;
      int kb1 = kb0 + p.kb_per_split;
      if (kb1 > p.num_pix_blocks) kb1 = p.num_pix_blocks;
      // kind::f16, D = fp32, A and B both MN-major (bits 15 / 16), M = 128, N = 64 * nchunks
      const uint32_t idesc = ptx::make_idesc_bf16_f32(128, 64 * nchunks, kFp16 ? 1 : 0) | (1u << 15) | (1u << 16);
      ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
      ptx::tc_fence_after();
      const uint32_t tmem_d = tmem_base + (uint32_t)acc * 256u;
      for (int kb = kb0; kb < kb1; ++kb) {
        ptx::mbar_wait(&full_bar[stage], phase);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
          const uint32_t a_addr = smem_base + (uint32_t)(stage * kWgStageBytes);
          const uint32_t b_addr = a_addr + (uint32_t)kWgABytes;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t adesc = make_desc_mn_sw128(a_addr + (uint32_t)k * kstep, lbo, sbo);
            const uint64_t bdesc = make_desc_mn_sw128(b_addr + (uint32_t)k * kstep, lbo, sbo);
            ptx::umma_bf16(tmem_d, adesc, bdesc, idesc, (uint32_t)((kb != kb0) | (k != 0)));
          }
          ptx::umma_commit(&empty_bar[stage]);
          if (kb == kb1 - 1) ptx::umma_commit(&tmem_full_bar[acc]);
        }
        __syncwarp();
        if (++stage == kWgStages) {
          stage = 0;
          phase ^= 1;
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else {
    // ------------------------------------------------------------ epilogue: TMEM -> fp32 partial tile
    const int quad = warp & 3;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
      const int t = item / splits;
      const int n_blk = t % nnb;
      const int rem_chunks = total_chunks - n_blk * 4;
      const int nchunks = rem_chunks < 4 ? rem_chunks : 4;
      const int ncols = 64 * nchunks;
      float* dst = p.partials + ((size_t)item * 128 + (size_t)(quad * 32 + lane)) * 256;
      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)acc * 256u;
      for (int c0 = 0; c0 < ncols; c0 += 32) {
        uint32_t v0[16], v1[16];
        ptx::tmem_ld_x16(taddr + (uint32_t)c0, v0);
        ptx::tmem_ld_x16(taddr + (uint32_t)c0 + 16u, v1);
        ptx::tmem_ld_wait();
        float4* o = reinterpret_cast<float4*>(dst + c0);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          o[i] = make_float4(__uint_as_float(v0[4 * i]), __uint_as_float(v0[4 * i + 1]), __uint_as_float(v0[4 * i + 2]),
                             __uint_as_float(v0[4 * i + 3]));
#pragma unroll
        for (int i = 0; i < 4; ++i)
          o[4 + i] = make_float4(__uint_as_float(v1[4 * i]), __uint_as_float(v1[4 * i + 1]),
                                 __uint_as_float(v1[4 * i + 2]), __uint_as_float(v1[4 * i + 3]));
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tmem_empty_bar[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512u);
  }
}

// grad[co][kk] = rowscale[co] * mask[co][kk] * sum_s partial[(m_blk, n_blk, s)][co % 128][kk % 256], stored through `mode`
// (scaled, then optionally added to what the arena holds).
// SG threads share one float4 of the gradient: thread (e, sg) sums the splits sg, sg + SG, ...; the SG partial sums are
// then added in index order by one thread (fixed order: bitwise reproducible, no atomics).
template <int SG>
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ partials, int Cout, int Kw, int nnb,
                                                           int splits, const float* __restrict__ rowscale,
                                                           const float* __restrict__ mask, float* __restrict__ grad,
                                                           const GradMode* __restrict__ mode, const float* __restrict__ wmaster,
                                                           float* __restrict__ rowdot_part) {
  constexpr int EPB = 256 / SG;  // float4 elements per block
  const int e = threadIdx.x % EPB, sg = threadIdx.x / EPB;
  const size_t total = (size_t)Cout * (Kw >> 2);
  const size_t t = (size_t)blockIdx.x * EPB + e;
  __shared__ float4 sm[SG > 1 ? 256 : 1];
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int co = 0, kk = 0;
  if (t < total) {
    kk = (int)(t % (size_t)(Kw >> 2)) * 4;
    co = (int)(t / (size_t)(Kw >> 2));
    const int m_blk = co >> 7, n_blk = kk >> 8;
    const float* src = partials + ((size_t)(m_blk * nnb + n_blk) * splits * 128 + (size_t)(co & 127)) * 256 + (kk & 255);
    for (int s = sg; s < splits; s += SG) {
      const float4 v = *reinterpret_cast<const float4*>(src + (size_t)s * 128 * 256);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  if (SG > 1) {
    sm[threadIdx.x] = acc;
    __syncthreads();
    if (sg != 0) return;
    for (int j = 1; j < SG; ++j) {
      const float4 v = sm[j * EPB + e];
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  if (t >= total) return;
  if (rowdot_part != nullptr) {
    // <W[co, kk..kk+3], dW_raw[co, kk..kk+3]>: summed over the row this is sum_p dy[p,co] * z[p,co] (z = conv output)
    const float4 w = *reinterpret_cast<const float4*>(wmaster + (size_t)co * Kw + kk);
    rowdot_part[t] = (acc.x * w.x + acc.y * w.y) + (acc.z * w.z + acc.w * w.w);
  }
  const float rs = rowscale ? rowscale[co] : 1.0f;
  acc.x *= rs; acc.y *= rs; acc.z *= rs; acc.w *= rs;
  float4* g = reinterpret_cast<float4*>(grad + (size_t)co * Kw + kk);
  if (mask) {
    const float4 m = *reinterpret_cast<const float4*>(mask + (size_t)co * Kw + kk);
    acc.x *= m.x; acc.y *= m.y; acc.z *= m.z; acc.w *= m.w;
  }
  if (mode != nullptr) {
    const GradMode md = *mode;
    acc.x *= md.out_scale; acc.y *= md.out_scale; acc.z *= md.out_scale; acc.w *= md.out_scale;
    if (md.accumulate) {
      const float4 o = *g;
      acc.x = o.x + acc.x; acc.y = o.y + acc.y; acc.z = o.z + acc.z; acc.w = o.w + acc.w;
    }
  }
  *g = acc;
}

}  // namespace

void wgrad_plan(WgradParams* p, int num_sms) {
  p->num_m_blocks = (p->Cout + 127) / 128;
  p->num_n_blocks = (p->Kw + 255) / 256;
  const int base = p->num_m_blocks * p->num_n_blocks;
  int splits = num_sms / base;  // one wave of work items
  if (splits < 1) splits = 1;
  const int max_splits = (p->num_pix_blocks + 3) / 4;  // at least 4 pixel blocks per split
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  p->kb_per_split = (p->num_pix_blocks + splits - 1) / splits;
  p->splits = (p->num_pix_blocks + p->kb_per_split - 1) / p->kb_per_split;
}

size_t wgrad_workspace_bytes(const WgradParams& p) {
  return (size_t)p.num_m_blocks * p.num_n_blocks * p.splits * 128 * 256 * sizeof(float);
}

cudaError_t launch_wgrad_gemm(const WgradParams& p, int num_sms, cudaStream_t stream) {
  static bool attr_set = false;
  const size_t smem = 1024 + (size_t)kWgStages * kWgStageBytes + (2 * kWgStages + 4) * 8 + 16;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(wgrad_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(wgrad_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  const int items = p.num_m_blocks * p.num_n_blocks * p.splits;
  const int grid = items < num_sms ? items : num_sms;
  if (p.fp16) wgrad_gemm_kernel<true><<<grid, kWgThreads, smem, stream>>>(p);
  else wgrad_gemm_kernel<false><<<grid, kWgThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_wgrad_reduce(const WgradParams& p, const float* rowscale, const float* mask, float* grad,
                                const GradMode* mode, cudaStream_t stream, const float* wmaster, float* rowdot_part) {
  const size_t total = (size_t)p.Cout * (p.Kw / 4);
  // few elements and many splits (the narrow, pixel-rich layers of block 1/2): spread the split loop over threads
  if (p.splits >= 32 && total <= 32768) {
    wgrad_reduce_kernel<16><<<(unsigned)((total + 15) / 16), 256, 0, stream>>>(p.partials, p.Cout, p.Kw, p.num_n_blocks,
                                                                             p.splits, rowscale, mask, grad, mode, wmaster, rowdot_part);
  } else if (p.splits >= 8 && total <= 262144) {
    wgrad_reduce_kernel<4><<<(unsigned)((total + 63) / 64), 256, 0, stream>>>(p.partials, p.Cout, p.Kw, p.num_n_blocks,
                                                                            p.splits, rowscale, mask, grad, mode, wmaster, rowdot_part);
  } else {
    wgrad_reduce_kernel<1><<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(p.partials, p.Cout, p.Kw, p.num_n_blocks,
                                                                              p.splits, rowscale, mask, grad, mode, wmaster, rowdot_part);
  }
  return cudaGetLastError();
}

}  // namespace dgp
