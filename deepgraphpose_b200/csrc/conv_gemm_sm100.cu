// Implicit-GEMM convolution on tcgen05 / TMEM / TMA (sm_100a).  See conv_gemm_sm100.cuh.
//
// CTA = 576 threads, persistent over (m_blk, n_blk) tiles:
//   warp 0       TMA producer   (one lane): A tile 128 x 64 (tiled or im2col) + B tile block_n x 64 per stage
//   warp 1       MMA issuer     (one lane): 4 x tcgen05.mma (K=16) per stage into a double-buffered TMEM accumulator
//   warps 2..17  epilogue: tcgen05.ld -> fp32 BN scale/shift (+residual)(+ReLU) -> 16 bit (four warps per TMEM quadrant)
// Pipelines: smem full/empty ring (TMA <-> MMA), TMEM full/empty pair (MMA <-> epilogue), and per epilogue warp a
// ring of 2 KB staging buffers (32 rows x 32 channels, SWIZZLE_64B): the residual tile is TMA-loaded into a buffer
// ahead of time, the warp adds it to the accumulator in place and the buffer is TMA-stored to the output, so that
// every byte of residual / output traffic is moved by the copy engine, not by the LSU, and no epilogue warp ever
// waits for another one (round 1 ran 8 warps in pairs around named barriers: latency-bound at 35 % issue activity).
#include "conv_gemm_sm100.cuh"

#include <stdio.h>

#include <type_traits>

#include "ptx_sm100.cuh"

namespace dgp {

namespace {

constexpr int kEpiWarps = 16;
constexpr int kThreads = 64 + 32 * kEpiWarps;  // TMA warp + MMA warp + 16 epilogue warps
constexpr int kABytes = kBlockM * kBlockK * 2;  // 16 KiB
constexpr int kMaxStages = 8;
constexpr int kMaxEpiBufs = 4;
constexpr int kEpiUnitBytes = 32 * kEpiUnitCols * 2;  // one warp's 32 rows x 32 columns
constexpr int kPatchBytes = 256 * 128;                 // epi_mode 2: one 256-pixel x 64-channel patch of conv1 outputs

__device__ __forceinline__ float bf16lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
// fp16 storage mode (same tcgen05 kind::f16 path, 11-bit mantissa): saturate instead of overflowing to inf
__device__ __forceinline__ uint32_t pack_fp16(float a, float b) {
  __half2 h = __floats2half2_rn(fminf(fmaxf(a, -65504.0f), 65504.0f), fminf(fmaxf(b, -65504.0f), 65504.0f));
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint4 pack8(const float* f, int fp16) {
  if (fp16) return make_uint4(pack_fp16(f[0], f[1]), pack_fp16(f[2], f[3]), pack_fp16(f[4], f[5]), pack_fp16(f[6], f[7]));
  return make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
}
// packed maximum of two 16-bit pairs (fp16 / bf16)
template <bool kFp16>
__device__ __forceinline__ uint32_t max16x2(uint32_t a, uint32_t b) {
  if (kFp16) {
    const __half2 z = __hmax2(*reinterpret_cast<const __half2*>(&a), *reinterpret_cast<const __half2*>(&b));
    return *reinterpret_cast<const uint32_t*>(&z);
  }
  const __nv_bfloat162 z = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(&a), *reinterpret_cast<const __nv_bfloat162*>(&b));
  return *reinterpret_cast<const uint32_t*>(&z);
}

// One epilogue unit = this warp's 32 accumulator rows x 32 columns: BN scale/shift (fp32, packed FFMA2) (+ residual)
// (+ ReLU, folded into the float -> 16-bit conversion) written in place into the warp's 2 KB staging buffer
// (32 rows x 64 B, SWIZZLE_64B: 16-byte unit u of row r lives at u ^ ((r >> 1) & 3), conflict-free for LDS/STS.128).
// per-pair mask 0xFFFF where the 16-bit activation is > 0 (post-ReLU tensors: > 0 <=> != 0)
template <bool kFp16>
__device__ __forceinline__ uint32_t gt0_mask16x2(uint32_t a) {
  if (kFp16) return __hgt2_mask(*reinterpret_cast<const __half2*>(&a), __float2half2_rn(0.0f));
  return __hgt2_mask(*reinterpret_cast<const __nv_bfloat162*>(&a), __float2bfloat162_rn(0.0f));
}
template <bool kFp16>
__device__ __forceinline__ float2 unpack16x2(uint32_t v) {
  if (kFp16) return __half22float2(*reinterpret_cast<const __half2*>(&v));
  return make_float2(bf16lo(v), bf16hi(v));
}

// Per-channel sums over the 32 rows of a unit that sits in its staging buffer (32 rows x 64 B, SWIZZLE_64B): lane (j = lane & 15,
// h = lane >> 4) walks the 16 rows h*16.. of channel pair j -- per step the warp reads two whole rows (128 B, conflict free) --
// then the two halves meet in one shuffle.  Fixed order: bitwise reproducible.  Lanes 0..15 return the sums of channels 2j, 2j+1.
template <bool kFp16>
__device__ __forceinline__ float2 unit_colsum(const uint8_t* buf, int lane) {
  const int j = lane & 15, h = lane >> 4;
  const int u = j >> 2, w = j & 3;
  float sx = 0.0f, sy = 0.0f;
#pragma unroll
  for (int it = 0; it < 16; ++it) {
    const int r = h * 16 + it;
    const uint32_t v = *reinterpret_cast<const uint32_t*>(buf + r * 64 + ((u ^ ((r >> 1) & 3)) << 4) + w * 4);
    const float2 d = unpack16x2<kFp16>(v);
    sx += d.x;
    sy += d.y;
  }
  sx += __shfl_xor_sync(0xffffffffu, sx, 16);
  sy += __shfl_xor_sync(0xffffffffu, sy, 16);
  return make_float2(sx, sy);
}

// kMask: the unit is a dgrad tile whose consumer would apply dy = g * [act > 0] (and sum dy per channel, unit_colsum above):
// `act` holds this lane's 32 activations (64 B), the masked 16-bit values go to the staging row.
template <bool kFp16, bool kRelu, bool kRes, bool kMask>
__device__ __forceinline__ void epi_unit_math(const uint32_t (&v)[2][16], uint8_t* my_row, int lane, const float* ss,
                                              const uint4* act = nullptr) {
  const int sw = (lane >> 1) & 3;
#pragma unroll
  for (int s2 = 0; s2 < 2; ++s2) {
    uint4* s0 = reinterpret_cast<uint4*>(my_row + (((2 * s2) ^ sw) << 4));
    uint4* s1 = reinterpret_cast<uint4*>(my_row + (((2 * s2 + 1) ^ sw) << 4));
    const float* scp = ss + s2 * 16;
    const float* shp = ss + 32 + s2 * 16;
    uint32_t rr[8];
    if (kRes) {
      const uint4 r0 = *s0;
      const uint4 r1 = *s1;
      rr[0] = r0.x; rr[1] = r0.y; rr[2] = r0.z; rr[3] = r0.w; rr[4] = r1.x; rr[5] = r1.y; rr[6] = r1.z; rr[7] = r1.w;
    }
    uint32_t o[8];
#pragma unroll
    for (int i = 0; i < 8; i += 2) {
      ptx::f32x2 q0 = ptx::pk2(__uint_as_float(v[s2][2 * i]), __uint_as_float(v[s2][2 * i + 1]));
      ptx::f32x2 q1 = ptx::pk2(__uint_as_float(v[s2][2 * i + 2]), __uint_as_float(v[s2][2 * i + 3]));
      if (!kMask) {   // the backward GEMMs (kMask) carry no BatchNorm: the scale is folded into their weights
        const float4 sc = *reinterpret_cast<const float4*>(scp + 2 * i);
        const float4 sh = *reinterpret_cast<const float4*>(shp + 2 * i);
        q0 = ptx::fma2(q0, ptx::pk2(sc.x, sc.y), ptx::pk2(sh.x, sh.y));
        q1 = ptx::fma2(q1, ptx::pk2(sc.z, sc.w), ptx::pk2(sh.z, sh.w));
      }
      if (kRes) {
        if (kFp16) {
          const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&rr[i]));
          const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&rr[i + 1]));
          q0 = ptx::add2(q0, ptx::pk2(a.x, a.y));
          q1 = ptx::add2(q1, ptx::pk2(b.x, b.y));
        } else {
          q0 = ptx::add2(q0, ptx::pk2(bf16lo(rr[i]), bf16hi(rr[i])));
          q1 = ptx::add2(q1, ptx::pk2(bf16lo(rr[i + 1]), bf16hi(rr[i + 1])));
        }
      }
      float a0, a1, b0, b1;
      ptx::upk2(q0, a0, a1);
      ptx::upk2(q1, b0, b1);
      o[i] = ptx::cvt_pack16<kFp16, kRelu>(a0, a1);
      o[i + 1] = ptx::cvt_pack16<kFp16, kRelu>(b0, b1);
    }
    if (kMask) {
      const uint4 m0 = act[2 * s2], m1 = act[2 * s2 + 1];
      const uint32_t mm[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] &= gt0_mask16x2<kFp16>(mm[i]);
    }
    *s0 = make_uint4(o[0], o[1], o[2], o[3]);
    *s1 = make_uint4(o[4], o[5], o[6], o[7]);
  }
}

// kFp16 selects the 16-bit storage type at compile time (bf16 / fp16): no dtype branches in the epilogue.
// kCta2: CTA-pair variant (cluster of 2, tcgen05 cta_group::2): one 256-row x 256-column tile per pair, each CTA stages its
// own 128 rows of A and half of the weight tile (half the shared-memory operand traffic per MMA), the leader issues the MMA.
// kMask: backward-pass variant whose epilogue applies the consumer's ReLU mask and writes dbeta partial sums (own
// instantiation so that the forward kernels keep their register allocation).
template <bool kFp16, bool kCta2, bool kMask>
__global__ void __launch_bounds__(kThreads, 1) conv_gemm_kernel(const __grid_constant__ ConvGemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t cta_rank = kCta2 ? ptx::cluster_ctarank() : 0u;
  const int tile0 = kCta2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;     // first tile / tile stride of this CTA (pair)
  const int tstep = kCta2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int stages = p.num_stages;
  const int msub = p.msub;                     // 128-row sub-tiles per CTA tile (BLOCK_M = 128 * msub)
  const int a_bytes = p.a_mode == 3 ? p.pt_stage_bytes : msub * kABytes;
  const int b_bytes = (kCta2 ? p.block_n / 2 : p.block_n) * kBlockK * 2;   // a CTA pair splits the weight tile
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + stages * a_bytes;
  uint8_t* smem_epi = smem_b + (p.a_mode == 3 ? p.num_k_blocks : stages) * b_bytes;  // [16 warps][epi_bufs][2 KiB], 1024 B aligned
  const int epi_bufs = p.epi_mode == 1 ? p.epi_bufs : 0;
  float* smem_ss = reinterpret_cast<float*>(smem_epi + (p.epi_mode == 2 ? 2 * kPatchBytes : kEpiWarps * epi_bufs * kEpiUnitBytes));  // [16 warps][2 sets][scale 32 | shift 32]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_ss + kEpiWarps * 128);
  uint64_t* empty_bar = full_bar + kMaxStages;
  uint64_t* tmem_full_bar = empty_bar + kMaxStages;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint64_t* res_bar = tmem_empty_bar + 2;  // [16 warps][kMaxEpiBufs]
  uint64_t* b_bar = res_bar + kEpiWarps * kMaxEpiBufs;  // a_mode 3: the resident weight matrix has landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(b_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&p.tmap_a);
    ptx::prefetch_tmap(&p.tmap_b);
    if (p.epi_mode == 1) {
      ptx::prefetch_tmap(&p.tmap_out);
      if (p.residual != nullptr) ptx::prefetch_tmap(&p.tmap_res);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < stages; ++s) {
      ptx::mbar_init(&full_bar[s], kCta2 ? 2 : 1);   // pair: the leader's expect_tx arrive + the peer's remote arrive
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tmem_full_bar[a], 1);
      // arrivals per accumulator buffer: every epilogue warp (both CTAs' in a pair); the pooling epilogue splits the warps
      // into two groups, one per buffer
      ptx::mbar_init(&tmem_empty_bar[a], kCta2 ? 2 * kEpiWarps : (p.epi_mode == 2 ? kEpiWarps / 2 : kEpiWarps));
    }
    for (int i = 0; i < kEpiWarps * kMaxEpiBufs; ++i) ptx::mbar_init(&res_bar[i], 1);
    ptx::mbar_init(b_bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    if (kCta2) {
      ptx::tmem_alloc_2sm(tmem_slot, (uint32_t)p.tmem_cols);
      ptx::tmem_relinquish_2sm();
    } else {
      ptx::tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before();
  if (kCta2) ptx::cluster_sync_all();   // the peer's barriers must be initialised before anything signals them
  else __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Programmatic dependent launch: everything above (smem carve-up, barrier init, TMEM alloc, descriptor prefetch)
  // overlapped the previous layer's tail; from here on we touch its output, so wait for it to complete and flush.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  const int num_tiles = p.num_m_blocks * p.num_n_blocks;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (whole warp loops, one lane issues)
    // Kernel parameters used inside the k loop are copied to registers first: every c[0x0][..] re-read is a
    // ~10-cycle uniform load on the single-warp critical path.
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t tx_bytes = (uint32_t)(a_bytes + b_bytes);
    const int PQ = p.P * p.Q, Q = p.Q, nnb = p.num_n_blocks, nkb = p.num_k_blocks, block_n = p.block_n;
    const int a_mode = p.a_mode, cblocks = p.cblocks, S = p.S, dil = p.dil, cstride = p.conv_stride;
    const int lower_w = p.lower_w, lower_h = p.lower_h, block_m = kCta2 ? 2 * kBlockM : kBlockM * msub;
    if (!kCta2 && a_mode == 3) {
      // shared-memory resident input patch: the whole weight matrix once, then ONE tiled box (patch + halo, zero filled
      // outside the image) per tile
      const int tiles_j = p.pool_tiles_j, tiles_ij = p.pool_tiles_i * tiles_j;
      const uint32_t box_bytes = (uint32_t)(p.pt_wp * (p.pt_rows + 2 * dil) * 128);
      if (lane == 0) {
        ptx::mbar_arrive_expect_tx(b_bar, (uint32_t)(nkb * b_bytes));
        for (int kb = 0; kb < nkb; ++kb) ptx::tma_load_2d(smem_b + kb * b_bytes, &p.tmap_b, b_bar, kb * kBlockK, 0);
      }
      __syncwarp();
      for (int tile = tile0; tile < num_tiles; tile += tstep) {
        const int img = tile / tiles_ij;
        const int rem = tile - img * tiles_ij;
        const int ti = rem / tiles_j;
        const int tj = rem - ti * tiles_j;
        ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
        if (lane == 0) {
          ptx::mbar_arrive_expect_tx(&full_bar[stage], box_bytes);
          ptx::tma_load_4d(smem_a + stage * a_bytes, &p.tmap_a, &full_bar[stage], 0, tj * p.pt_cols - dil, ti * p.pt_rows - dil, img);
        }
        __syncwarp();
        if (++stage == stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    } else if (!kCta2 && a_mode == 2) {
      // conv1 + pool1: the A tile is a 2-D patch of conv outputs = ONE tiled box per filter-row tap (the tensor map's
      // "pixels" are overlapping 4-pixel windows of the space-to-depth input; rows / columns past the end read as zero)
      const int tiles_j = p.pool_tiles_j, tiles_ij = p.pool_tiles_i * tiles_j;
      const uint32_t tx = (uint32_t)((2 * p.pool_R + 1) * (2 * p.pool_C + 1) * 128 + b_bytes);
      for (int tile = tile0; tile < num_tiles; tile += tstep) {
        const int img = tile / tiles_ij;
        const int rem = tile - img * tiles_ij;
        const int ti = rem / tiles_j;
        const int tj = rem - ti * tiles_j;
        const int ra = max(0, 2 * ti * p.pool_R - p.pool_pad_t), ca = max(0, 2 * tj * p.pool_C - p.pool_pad_l);
        for (int kb = 0; kb < nkb; ++kb) {
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
          if (lane == 0) {
            ptx::mbar_arrive_expect_tx(&full_bar[stage], tx);
            ptx::tma_load_4d(smem_a + stage * a_bytes, &p.tmap_a, &full_bar[stage], 0, ca, ra + kb, img);
            ptx::tma_load_2d(smem_b + stage * b_bytes, &p.tmap_b, &full_bar[stage], kb * kBlockK, 0);
          }
          __syncwarp();
          if (++stage == stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    } else
    for (int tile = tile0; tile < num_tiles; tile += tstep) {
      const int m_blk = tile / nnb;
      const int n_blk = tile - m_blk * nnb;
      const int m0 = m_blk * block_m + (int)cta_rank * kBlockM;              // pair: this CTA's 128 rows
      const int n0 = n_blk * block_n + (int)cta_rank * (block_n >> 1) * (kCta2 ? 1 : 0);   // ... and its half of the weights
      int img = 0, cw = 0, ch = 0;
      if (a_mode == 1) {
        img = m0 / PQ;
        const int rem = m0 - img * PQ;
        const int pp = rem / Q;
        const int qq = rem - pp * Q;
        cw = qq * cstride + lower_w;
        ch = pp * cstride + lower_h;
      }
      int cb = 0, off_w = 0, off_h = 0, tap_s = 0;  // incremental (channel block, tap) counters: no divides in the loop
      for (int kb = 0; kb < nkb; ++kb) {
        ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
        if (ptx::elect_one()) {
          if (kCta2) {
            // both CTAs count their bytes on the LEADER's barrier (it alone feeds the MMA issuer)
            const uint32_t lbar = ptx::mapa_u32(&full_bar[stage], 0);
            if (cta_rank == 0) ptx::mbar_arrive_expect_tx(&full_bar[stage], 2 * tx_bytes);
            if (a_mode == 0) {
              ptx::tma_load_2d_2sm(smem_a + stage * a_bytes, &p.tmap_a, lbar, kb * kBlockK, m0);
            } else {
              ptx::tma_load_im2col_4d_2sm(smem_a + stage * a_bytes, &p.tmap_a, lbar, cb * kBlockK, cw, ch, img, (uint16_t)off_w,
                                          (uint16_t)off_h);
            }
            ptx::tma_load_2d_2sm(smem_b + stage * b_bytes, &p.tmap_b, lbar, kb * kBlockK, n0);
            if (cta_rank != 0) ptx::mbar_arrive_cluster(lbar);
          } else {
            ptx::mbar_arrive_expect_tx(&full_bar[stage], tx_bytes);
            if (a_mode == 0) {
              ptx::tma_load_2d(smem_a + stage * a_bytes, &p.tmap_a, &full_bar[stage], kb * kBlockK, m0);
            } else {
              ptx::tma_load_im2col_4d(smem_a + stage * a_bytes, &p.tmap_a, &full_bar[stage], cb * kBlockK, cw, ch, img,
                                      (uint16_t)off_w, (uint16_t)off_h);
            }
            ptx::tma_load_2d(smem_b + stage * b_bytes, &p.tmap_b, &full_bar[stage], kb * kBlockK, n0);
          }
        }
        __syncwarp();
        if (++cb == cblocks) {
          cb = 0;
          off_w += dil;
          if (++tap_s == S) {
            tap_s = 0;
            off_w = 0;
            off_h += dil;
          }
        }
        if (++stage == stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    if (!kCta2 || cta_rank == 0) {
    // ------------------------------------------------------------ MMA issuer (whole warp loops, one lane issues)
    const int block_n = p.block_n, nkb = p.num_k_blocks;
    const uint32_t idesc = ptx::make_idesc_bf16_f32(kCta2 ? 2 * kBlockM : kBlockM, block_n, kFp16 ? 1 : 0);
    const uint64_t adesc0 = ptx::make_desc_k_sw128(ptx::smem_u32(smem_a));
    const uint64_t bdesc0 = ptx::make_desc_k_sw128(ptx::smem_u32(smem_b));
    const uint32_t a_step = (uint32_t)a_bytes >> 4, b_step = (uint32_t)b_bytes >> 4;
    const uint32_t acc_cols = (uint32_t)(msub * block_n);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    // The two tile heights get separate, branch-free issue loops (a predicate between UTCHMMAs costs issue slots).
    auto run = [&](auto msub_tag) {
      constexpr int kMsub = decltype(msub_tag)::value;
      for (int tile = tile0; tile < num_tiles; tile += tstep) {
        ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
        ptx::tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)acc * acc_cols;
        for (int kb = 0; kb < nkb; ++kb) {
          ptx::mbar_wait(&full_bar[stage], phase);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            const uint64_t adesc = adesc0 + (uint64_t)(stage * a_step);
            const uint64_t bdesc = bdesc0 + (uint64_t)(stage * b_step);
#pragma unroll
            for (int k = 0; k < kBlockK / 16; ++k) {
              // advance 16 bf16 = 32 B along K inside the 128 B swizzle row: +2 in the (addr >> 4) field
              if (kCta2) {
                ptx::umma_bf16_2sm(tmem_d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0);
              } else {
                ptx::umma_bf16(tmem_d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0);
                if (kMsub == 2)  // rows 128..255 of a 256-row tile: A 16 KiB further, D block_n columns further
                  ptx::umma_bf16(tmem_d + (uint32_t)block_n, adesc + (uint64_t)((kABytes >> 4) + k * 2),
                                 bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0);
              }
            }
            if (kCta2) {
              ptx::umma_commit_2sm(&empty_bar[stage]);                           // frees the stage in BOTH CTAs
              if (kb == nkb - 1) ptx::umma_commit_2sm(&tmem_full_bar[acc]);      // ... and wakes both epilogues
            } else {
              ptx::umma_commit(&empty_bar[stage]);
              if (kb == nkb - 1) ptx::umma_commit(&tmem_full_bar[acc]);
            }
          }
          __syncwarp();
          if (++stage == stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    };
    if (!kCta2 && p.a_mode == 3) {
      // 3x3 taps as row-shifted views of the resident patch: accumulator row m reads patch row m + (kr*Wp + ks)*dil
      const int Wp = p.pt_wp, dil = p.dil, bo_mode = p.pt_base_offset_mode;
      const uint32_t a0 = ptx::smem_u32(smem_a);
      ptx::mbar_wait(b_bar, 0);
      ptx::tc_fence_after();
      for (int tile = tile0; tile < num_tiles; tile += tstep) {
        ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
        ptx::mbar_wait(&full_bar[stage], phase);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
          const uint32_t tmem_d = tmem_base + (uint32_t)acc * acc_cols;
          const uint32_t abase = a0 + (uint32_t)(stage * a_bytes);
#pragma unroll 1
          for (int tap = 0; tap < 9; ++tap) {
            const int kr = tap / 3, ks = tap - kr * 3;
            const uint32_t shift = (uint32_t)((kr * Wp + ks) * dil) * 128u;
            const uint64_t bdesc = bdesc0 + (uint64_t)(tap * b_step);
#pragma unroll
            for (int sub = 0; sub < 2; ++sub) {
              const uint32_t start = abase + shift + (uint32_t)sub * (uint32_t)kABytes;
              const uint64_t adesc = ptx::make_desc_k_sw128(start, bo_mode ? (start >> 7) : 0u);
#pragma unroll
              for (int k = 0; k < kBlockK / 16; ++k)
                ptx::umma_bf16(tmem_d + (uint32_t)(sub * block_n), adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc,
                               (tap | k) != 0);
            }
          }
          ptx::umma_commit(&empty_bar[stage]);
          ptx::umma_commit(&tmem_full_bar[acc]);
        }
        __syncwarp();
        if (++stage == stages) {
          stage = 0;
          phase ^= 1;
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    } else if (!kCta2 && msub == 2) run(std::integral_constant<int, 2>{});
    else run(std::integral_constant<int, 1>{});
    }  // leader CTA (or single-CTA kernel)
  } else if (!kCta2 && p.epi_mode == 0) {
    // -------------------------------------------------------------- epilogue, direct stores (fp32 head GEMM)
    // 16 epilogue warps: four per TMEM lane quadrant, taking every fourth 16-column group.
    const int quad = warp & 3;  // TMEM lane quadrant this warp may access
    const int cg = (warp - 2) >> 2;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = tile0; tile < num_tiles; tile += tstep) {
      const int m_blk = tile / p.num_n_blocks;
      const int n_blk = tile - m_blk * p.num_n_blocks;
      const int row = m_blk * kBlockM + quad * 32 + lane;
      const int n0 = n_blk * p.block_n;
      const bool row_ok = row < p.M;
      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * p.block_n);
      for (int c0 = cg * 16; c0 < p.block_n; c0 += 64) {
        uint32_t v[16];
        ptx::tmem_ld_x16(taddr + (uint32_t)c0, v);
        ptx::tmem_ld_wait();
        if (row_ok) {
          float f[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) f[i] = __uint_as_float(v[i]);
          const int n = n0 + c0;
          if (p.scale != nullptr) {
#pragma unroll
            for (int i = 0; i < 16; ++i) f[i] *= __ldg(p.scale + n + i);
          }
          if (p.shift != nullptr) {
#pragma unroll
            for (int i = 0; i < 16; ++i) f[i] += __ldg(p.shift + n + i);
          }
          if (p.relu) {
#pragma unroll
            for (int i = 0; i < 16; ++i) f[i] = fmaxf(f[i], 0.0f);
          }
          if (p.out_f32) {
            float4* op = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + (size_t)row * p.ldc + n);
#pragma unroll
            for (int i = 0; i < 4; ++i) op[i] = make_float4(f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]);
          } else {
            uint4* op = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + (size_t)row * p.ldc + n);
            op[0] = pack8(f, kFp16);
            op[1] = pack8(f + 8, kFp16);
          }
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tmem_empty_bar[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else if (!kCta2 && p.epi_mode == 3) {
    // -------------------------------------------------------------- epilogue of a patch tile (a_mode 3): direct stores
    // accumulator row m = pr * Wp + pc lies on the input-patch grid; rows with pc >= pt_cols or pr >= pt_rows are halo
    // positions (junk) and are not stored.  Every lane owns one pixel x 32 channels = 64 contiguous bytes of the output.
    const int quad = warp & 3;
    const int ew = warp - 2;
    const int cg = ew >> 2;
    const int sub = cg >> 1, colg = cg & 1;
    float* ss = smem_ss + ew * 128;
    if (lane < 16) {
      const int is_shift = lane >> 3, i = (lane & 7) * 4;
      const float* src = is_shift ? p.shift : p.scale;
      const float fill = is_shift ? 0.f : 1.f;
      const float4 val = src ? __ldg(reinterpret_cast<const float4*>(src + colg * 32 + i)) : make_float4(fill, fill, fill, fill);
      *reinterpret_cast<float4*>(ss + is_shift * 32 + i) = val;
    }
    __syncwarp();
    const int tiles_j = p.pool_tiles_j, tiles_ij = p.pool_tiles_i * tiles_j;
    const int m = sub * 128 + quad * 32 + lane;
    const int pr = m / p.pt_wp, pc = m - pr * p.pt_wp;
    const bool in_tile = pr < p.pt_rows && pc < p.pt_cols;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = tile0; tile < num_tiles; tile += tstep) {
      const int img = tile / tiles_ij;
      const int rem = tile - img * tiles_ij;
      const int ti = rem / tiles_j;
      const int tj = rem - ti * tiles_j;
      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)((acc * 2 + sub) * 64 + colg * 32);
      uint32_t v[2][16];
      ptx::tmem_ld_x16(taddr, v[0]);
      ptx::tmem_ld_x16(taddr + 16, v[1]);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tmem_empty_bar[acc]);
      const int r = ti * p.pt_rows + pr, c = tj * p.pt_cols + pc;
      if (in_tile && r < p.P && c < p.Q) {
        uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(p.out) +
                                              ((((size_t)img * p.P + r) * p.Q + c) * p.ldc + colg * 32) * 2);
#pragma unroll
        for (int s2 = 0; s2 < 2; ++s2) {
          uint32_t o[8];
#pragma unroll
          for (int i = 0; i < 8; i += 2) {
            const float4 sc = *reinterpret_cast<const float4*>(ss + s2 * 16 + 2 * i);
            const float4 sh = *reinterpret_cast<const float4*>(ss + 32 + s2 * 16 + 2 * i);
            const ptx::f32x2 q0 = ptx::fma2(ptx::pk2(__uint_as_float(v[s2][2 * i]), __uint_as_float(v[s2][2 * i + 1])),
                                            ptx::pk2(sc.x, sc.y), ptx::pk2(sh.x, sh.y));
            const ptx::f32x2 q1 = ptx::fma2(ptx::pk2(__uint_as_float(v[s2][2 * i + 2]), __uint_as_float(v[s2][2 * i + 3])),
                                            ptx::pk2(sc.z, sc.w), ptx::pk2(sh.z, sh.w));
            float a0, a1, b0, b1;
            ptx::upk2(q0, a0, a1);
            ptx::upk2(q1, b0, b1);
            if (p.relu) {
              o[i] = ptx::cvt_pack16<kFp16, true>(a0, a1);
              o[i + 1] = ptx::cvt_pack16<kFp16, true>(b0, b1);
            } else {
              o[i] = ptx::cvt_pack16<kFp16, false>(a0, a1);
              o[i + 1] = ptx::cvt_pack16<kFp16, false>(b0, b1);
            }
          }
          dst[2 * s2] = make_uint4(o[0], o[1], o[2], o[3]);
          dst[2 * s2 + 1] = make_uint4(o[4], o[5], o[6], o[7]);
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else if (!kCta2 && p.epi_mode == 2) {
    // -------------------------------------------------------------- epilogue, conv1 + BN + ReLU + 3x3/2 max-pool
    // The 256 accumulator rows are the pixels of a 2-D patch of conv1 outputs (row-major, `Cw` accumulator rows per patch
    // row).  The 16 epilogue warps form TWO groups of 8 that take alternate tiles (group g owns accumulator buffer g and
    // patch buffer g), so two tiles are in flight per SM and one group's barrier / load latencies hide under the other's
    // arithmetic.  Per tile a group turns the accumulator (each warp: 32 rows x 32 channels of both 128-row halves) into
    // 16-bit activations in its shared-memory patch (128 B per pixel, 16-byte units XOR-swizzled by the pixel index), meets
    // on its own named barrier, and its 256 threads reduce the R x C pooled pixels (one 16-byte channel group each, nine
    // LDS.128 + packed max) straight to global memory.  conv1's 20 MB-per-frame output never reaches HBM.
    const int quad = warp & 3;
    const int ew = warp - 2;
    const int grp = ew >> 3;
    const int colg = (ew >> 2) & 1;
    float* ss = smem_ss + ew * 128;
    if (lane < 16) {
      const int is_shift = lane >> 3, i = (lane & 7) * 4;
      const float* src = is_shift ? p.shift : p.scale;
      const float fill = is_shift ? 0.f : 1.f;
      const float4 val = src ? __ldg(reinterpret_cast<const float4*>(src + colg * 32 + i)) : make_float4(fill, fill, fill, fill);
      *reinterpret_cast<float4*>(ss + is_shift * 32 + i) = val;
    }
    __syncwarp();
    const int R = p.pool_R, Cp = p.pool_C, H1 = p.P, W1 = p.Q;
    const int Cw = 2 * p.pool_C + 1;   // accumulator rows per patch row
    const int tiles_i = p.pool_tiles_i, tiles_j = p.pool_tiles_j;
    uint8_t* patch = smem_epi + grp * kPatchBytes;
    const uint32_t bar_id = 1u + (uint32_t)grp;
    // pooling work items of this thread: (pooled pixel, 16-byte channel group), items t and t + 256 of R * C * 8
    const int t = (int)threadIdx.x - 64 - grp * 256;
    const int pv = t & 7;
    int pi[2], pj[2], q0[2];
    bool pool_item[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int pp = (t >> 3) + 32 * k;
      pi[k] = pp / Cp;
      pj[k] = pp - pi[k] * Cp;
      pool_item[k] = pp < R * Cp;
      q0[k] = 2 * pi[k] * Cw + 2 * pj[k];       // first patch pixel of the window in an interior tile
    }
    // this group's tile sequence: tile0 + grp * tstep, then every 2 * tstep; (img, ti, tj) advance without divisions
    int tile = tile0 + grp * tstep;
    int img = tile / (tiles_i * tiles_j);
    int ti = (tile - img * tiles_i * tiles_j) / tiles_j;
    int tj = tile - (img * tiles_i + ti) * tiles_j;
    const int step = 2 * tstep;
    const int d_img = step / (tiles_i * tiles_j);
    const int d_ti = (step - d_img * tiles_i * tiles_j) / tiles_j;
    const int d_tj = step - (d_img * tiles_i + d_ti) * tiles_j;
    const int acc = grp;
    uint32_t acc_phase = 0;
    for (; tile < num_tiles; tile += step) {
      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
      ptx::tc_fence_after();
#pragma unroll
      for (int sub = 0; sub < 2; ++sub) {
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)((acc * 2 + sub) * 64 + colg * 32);
        uint32_t v[2][16];
        ptx::tmem_ld_x16(taddr, v[0]);
        ptx::tmem_ld_x16(taddr + 16, v[1]);
        ptx::tmem_ld_wait();
        if (sub == 1) {
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&tmem_empty_bar[acc]);   // the accumulator is in registers: the MMA may reuse it
        }
        const int px = sub * 128 + quad * 32 + lane;
        uint8_t* my_row = patch + px * 128;
#pragma unroll
        for (int s2 = 0; s2 < 2; ++s2) {
          uint32_t o[8];
#pragma unroll
          for (int i = 0; i < 8; i += 2) {
            const float4 sc = *reinterpret_cast<const float4*>(ss + s2 * 16 + 2 * i);
            const float4 sh = *reinterpret_cast<const float4*>(ss + 32 + s2 * 16 + 2 * i);
            const ptx::f32x2 r0 = ptx::fma2(ptx::pk2(__uint_as_float(v[s2][2 * i]), __uint_as_float(v[s2][2 * i + 1])),
                                            ptx::pk2(sc.x, sc.y), ptx::pk2(sh.x, sh.y));
            const ptx::f32x2 r1 = ptx::fma2(ptx::pk2(__uint_as_float(v[s2][2 * i + 2]), __uint_as_float(v[s2][2 * i + 3])),
                                            ptx::pk2(sc.z, sc.w), ptx::pk2(sh.z, sh.w));
            float a0, a1, b0, b1;
            ptx::upk2(r0, a0, a1);
            ptx::upk2(r1, b0, b1);
            o[i] = ptx::cvt_pack16<kFp16, true>(a0, a1);
            o[i + 1] = ptx::cvt_pack16<kFp16, true>(b0, b1);
          }
          const int u = colg * 4 + 2 * s2;
          *reinterpret_cast<uint4*>(my_row + ((u ^ (px & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
          *reinterpret_cast<uint4*>(my_row + (((u + 1) ^ (px & 7)) << 4)) = make_uint4(o[4], o[5], o[6], o[7]);
        }
      }
      ptx::named_bar_sync(bar_id, 256);
      // interior tiles (patch origin not clamped, no window row / column outside the image): constant patch offsets
      const bool interior = 2 * ti * R >= p.pool_pad_t && 2 * tj * Cp >= p.pool_pad_l &&
                            2 * (ti * R + R - 1) - p.pool_pad_t + 2 < H1 && 2 * (tj * Cp + Cp - 1) - p.pool_pad_l + 2 < W1;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        if (!pool_item[k]) continue;
        const int i = ti * R + pi[k], j = tj * Cp + pj[k];
        uint32_t m[4] = {0u, 0u, 0u, 0u};          // post-ReLU values are >= 0 and every window holds a valid pixel
        if (interior) {
#pragma unroll
          for (int w = 0; w < 9; ++w) {
            const int q = q0[k] + (w / 3) * Cw + w % 3;
            const uint4 x = *reinterpret_cast<const uint4*>(patch + q * 128 + ((pv ^ (q & 7)) << 4));
            const uint32_t xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int c = 0; c < 4; ++c) m[c] = max16x2<kFp16>(m[c], xs[c]);
          }
        } else {
          if (i >= p.pool_H || j >= p.pool_W) continue;
          const int ra = max(0, 2 * ti * R - p.pool_pad_t), ca = max(0, 2 * tj * Cp - p.pool_pad_l);
#pragma unroll
          for (int dr = 0; dr < 3; ++dr) {
            const int rr = 2 * i - p.pool_pad_t + dr;
            if (rr < 0 || rr >= H1) continue;
#pragma unroll
            for (int dc = 0; dc < 3; ++dc) {
              const int cc = 2 * j - p.pool_pad_l + dc;
              if (cc < 0 || cc >= W1) continue;
              const int q = (rr - ra) * Cw + (cc - ca);
              const uint4 x = *reinterpret_cast<const uint4*>(patch + q * 128 + ((pv ^ (q & 7)) << 4));
              const uint32_t xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
              for (int c = 0; c < 4; ++c) m[c] = max16x2<kFp16>(m[c], xs[c]);
            }
          }
        }
        uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(p.out) +
                                              ((((size_t)img * p.pool_H + i) * p.pool_W + j) * 64 + pv * 8) * 2);
        *dst = make_uint4(m[0], m[1], m[2], m[3]);
      }
      // the group's next write into this patch buffer happens after its next barrier-free phase; the barrier below keeps
      // a fast warp from overwriting pixels a slow one is still pooling
      ptx::named_bar_sync(bar_id, 256);
      acc_phase ^= 1;
      tj += d_tj;
      if (tj >= tiles_j) { tj -= tiles_j; ++ti; }
      ti += d_ti;
      if (ti >= tiles_i) { ti -= tiles_i; ++img; }
      img += d_img;
    }
  } else {
    // -------------------------------------------------------------- epilogue, TMA-staged 16-bit (+ TMA residual)
    // 16 INDEPENDENT epilogue warps, four per TMEM lane quadrant.  A tile is cut into units of 32 rows x 32 columns
    // (one warp's TMEM rows x two tcgen05.ld.x16); the warp with column-group index cg takes units cg, cg+4, ... of
    // the (sub-tile, column group) sequence.  Each warp owns a small ring of 2 KB staging buffers (32 rows x 64 B,
    // SWIZZLE_64B), TMA-loads the residual tile into a buffer ahead of time, combines in place and TMA-stores the
    // buffer: no barrier between warps anywhere in the epilogue, 16 units in flight per SM.
    const int quad = warp & 3;
    const int ew = warp - 2;
    const int cg = ew >> 2;
    const int nb = p.epi_bufs;
    uint8_t* ebuf = smem_epi + (size_t)ew * nb * kEpiUnitBytes;
    uint64_t* rbar = res_bar + ew * kMaxEpiBufs;
    const bool has_res = p.residual != nullptr;
    const int block_n = p.block_n, nnb = p.num_n_blocks;
    const int ncg = block_n >> 5;                                   // 32-column groups per tile row: 2, 4 or 8
    const int ncg_shift = ncg == 8 ? 3 : (ncg == 4 ? 2 : 1);
    const int units = msub * ncg;
    const int nsets = ncg == 8 ? 2 : 1;                             // distinct column groups this warp ever touches
    const int PQ = p.P * p.Q;
    float* ss = smem_ss + ew * 128;
    int ss_n0 = -1;

    // Residual prefetch cursor: walks this warp's (tile, unit) sequence nb-1 units ahead of the consumer.  All lanes
    // keep the (uniform) cursor; lane 0 issues.
    int pf_tile = tile0, pf_u = cg, pf_buf = 0, pf_mblk = 0, pf_n0 = 0;
    auto pf_setup_tile = [&]() {
      pf_mblk = pf_tile / nnb;
      pf_n0 = (pf_tile - pf_mblk * nnb) * block_n;
    };
    auto issue_residual = [&]() {
      if (pf_tile >= num_tiles) return;
      const int sub = pf_u >> ncg_shift;
      const int row0 = (kCta2 ? pf_mblk * 2 + (int)cta_rank : pf_mblk * msub + sub) * kBlockM + quad * 32;
      const int col0 = pf_n0 + ((pf_u & (ncg - 1)) << 5);
      if (lane == 0) {
        ptx::mbar_arrive_expect_tx(&rbar[pf_buf], (uint32_t)kEpiUnitBytes);
        if (p.res_sub == 1) {
          ptx::tma_load_2d(ebuf + pf_buf * kEpiUnitBytes, &p.tmap_res, &rbar[pf_buf], col0, row0);
        } else {
          const int img = row0 / PQ;
          const int rem = row0 - img * PQ;
          const int pp = rem / p.Q;
          ptx::tma_load_im2col_4d(ebuf + pf_buf * kEpiUnitBytes, &p.tmap_res, &rbar[pf_buf], col0,
                                  (rem - pp * p.Q) * p.res_sub, pp * p.res_sub, img, 0, 0);
        }
      }
      if (++pf_buf == nb) pf_buf = 0;
      pf_u += 4;
      if (pf_u >= units) {
        pf_u = cg;
        pf_tile += tstep;
        if (pf_tile < num_tiles) pf_setup_tile();
      }
    };

    const bool active = cg < units;  // 128-row tiles of a 64-wide layer have only two units
    if (has_res && active) {
      if (pf_tile < num_tiles) pf_setup_tile();
      for (int i = 0; i < nb - 1; ++i) issue_residual();
      __syncwarp();
    }
    int buf = 0;
    uint32_t buf_phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = tile0; tile < num_tiles; tile += tstep) {
      const int m_blk = tile / nnb;
      const int n0 = (tile - m_blk * nnb) * block_n;
      if (n0 != ss_n0 && active) {
        if (lane < 16 * nsets) {
          const int set = lane >> 4, is_shift = (lane >> 3) & 1, i = (lane & 7) * 4;
          const int col = n0 + (((cg & (ncg - 1)) + 4 * set) << 5) + i;
          const float* src = is_shift ? p.shift : p.scale;
          const float fill = is_shift ? 0.f : 1.f;
          const float4 val = src ? __ldg(reinterpret_cast<const float4*>(src + col)) : make_float4(fill, fill, fill, fill);
          *reinterpret_cast<float4*>(ss + set * 64 + is_shift * 32 + i) = val;
        }
        __syncwarp();
        ss_n0 = n0;
      }
      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
      ptx::tc_fence_after();
      for (int u = cg; u < units; u += 4) {
        const int sub = u >> ncg_shift;
        const int colg = u & (ncg - 1);
        const int row0 = (kCta2 ? m_blk * 2 + (int)cta_rank : m_blk * msub + sub) * kBlockM + quad * 32;
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)((acc * msub + sub) * block_n + (colg << 5));
        uint8_t* my_buf = ebuf + buf * kEpiUnitBytes;
        uint32_t v[2][16];
        ptx::tmem_ld_x16(taddr, v[0]);
        ptx::tmem_ld_x16(taddr + 16, v[1]);
        uint4 act[kMask ? 4 : 1];
        if (kMask) {
          const int row = row0 + lane;
          if (row < p.M) {
            // the lane's 64-byte activation row as two 256-bit loads: every lane touches a different line, so the cost is
            // L1 tag cycles per instruction -- half as many instructions as with 128-bit loads.  (Pulling the next unit's rows
            // towards L2 with prefetch.global.L2 was measured too: slightly slower.)
            const uint8_t* ap = reinterpret_cast<const uint8_t*>(p.mask_act) + ((size_t)row * p.ldc + n0 + (colg << 5)) * 2;
            ptx::ldg_nc_256(ap, act[0], act[1]);
            ptx::ldg_nc_256(ap + 32, act[2], act[3]);
          } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) act[i] = make_uint4(0u, 0u, 0u, 0u);
          }
        }
        if (has_res) {
          // the buffer the next prefetch lands in was last used by the unit before this one: its store must have
          // finished reading shared memory (it was committed a whole unit ago)
          if (lane == 0) ptx::bulk_wait_group_read<0>();
          issue_residual();
          ptx::mbar_wait(&rbar[buf], buf_phase);
        } else {
          // the store that last used this buffer (nb units ago) must have finished reading it
          if (lane == 0) {
            if (nb >= 3) ptx::bulk_wait_group_read<2>();
            else if (nb == 2) ptx::bulk_wait_group_read<1>();
            else ptx::bulk_wait_group_read<0>();
          }
          __syncwarp();
        }
        ptx::tmem_ld_wait();
        const float* ssu = ss + (colg >> 2) * 64;
        uint8_t* my_row = my_buf + lane * 64;
        if (kMask) {
          // dgrad tile with the consumer's ReLU mask and dbeta sums fused (the activation row was requested before the waits)
          if (has_res) epi_unit_math<kFp16, false, true, true>(v, my_row, lane, ssu, act);
          else epi_unit_math<kFp16, false, false, true>(v, my_row, lane, ssu, act);
          __syncwarp();
          const float2 cs = unit_colsum<kFp16>(my_buf, lane);
          if (lane < 16 && row0 < p.M)
            *reinterpret_cast<float2*>(p.colsum_part + (size_t)(row0 >> 5) * p.N + n0 + (colg << 5) + 2 * lane) = cs;
        } else if (has_res) {
          if (p.relu) epi_unit_math<kFp16, true, true, false>(v, my_row, lane, ssu);
          else epi_unit_math<kFp16, false, true, false>(v, my_row, lane, ssu);
        } else {
          if (p.relu) epi_unit_math<kFp16, true, false, false>(v, my_row, lane, ssu);
          else epi_unit_math<kFp16, false, false, false>(v, my_row, lane, ssu);
        }
        ptx::fence_proxy_async_smem();  // my generic-proxy smem writes -> visible to the TMA store (async proxy)
        __syncwarp();
        if (lane == 0) {
          ptx::tma_store_2d(&p.tmap_out, my_buf, n0 + (colg << 5), row0);
          ptx::bulk_commit_group();
        }
        if (++buf == nb) {
          buf = 0;
          buf_phase ^= 1;
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (kCta2) ptx::mbar_arrive_cluster(ptx::mapa_u32(&tmem_empty_bar[acc], 0));   // the leader's MMA issuer waits on it
        else ptx::mbar_arrive(&tmem_empty_bar[acc]);
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (lane == 0) ptx::bulk_wait_group_read<0>();
    __syncwarp();
  }

  ptx::tc_fence_before();
  if (kCta2) ptx::cluster_sync_all();   // the leader's MMAs read the peer's shared memory: nobody leaves early
  else __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    if (kCta2) ptx::tmem_dealloc_2sm(tmem_base, (uint32_t)p.tmem_cols);
    else ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*,
                                   CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                   CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode_tiled = nullptr;
EncodeIm2colFn g_encode_im2col = nullptr;
char g_err[256];

}  // namespace

const char* tma_init() {
  if (g_encode_tiled && g_encode_im2col) return nullptr;
  cudaDriverEntryPointQueryResult q;
  void* fn = nullptr;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
  if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn) return "cuTensorMapEncodeTiled not available";
  g_encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
  fn = nullptr;
  e = cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &q);
  if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn) return "cuTensorMapEncodeIm2col not available";
  g_encode_im2col = reinterpret_cast<EncodeIm2colFn>(fn);
  return nullptr;
}

namespace { int g_tmap_fp16 = 0; }
void tmap_set_fp16(int fp16) { g_tmap_fp16 = fp16; }

const char* make_tmap_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t k, uint64_t row_stride_bytes,
                         uint32_t box_rows, uint32_t box_cols) {
  if (const char* e = tma_init()) return e;
  cuuint64_t dims[2] = {k, rows};
  cuuint64_t strides[1] = {row_stride_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  const CUtensorMapSwizzle swz = box_cols == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;  // 128 B / 64 B rows
  if (box_cols != 64 && box_cols != 32) return "make_tmap_2d: box_cols must be 64 or 32";
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode_tiled(out, g_tmap_fp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box,
                              estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof(g_err), "cuTensorMapEncodeTiled failed: %d (rows=%llu k=%llu stride=%llu box_rows=%u)", (int)r,
             (unsigned long long)rows, (unsigned long long)k, (unsigned long long)row_stride_bytes, box_rows);
    return g_err;
  }
  return nullptr;
}

const char* make_tmap_im2col(CUtensorMap* out, const void* base, uint64_t C, uint64_t W, uint64_t H, uint64_t N,
                             uint64_t stride_w_bytes, uint64_t stride_h_bytes, uint64_t stride_n_bytes, int lower_w,
                             int lower_h, int upper_w, int upper_h, int conv_stride, uint64_t total_bytes,
                             uint32_t pixels_per_column, uint32_t channels_per_pixel) {
  if (const char* e = tma_init()) return e;
  if (channels_per_pixel != 64 && channels_per_pixel != 32) return "make_tmap_im2col: channels_per_pixel must be 64 or 32";
  const CUtensorMapSwizzle swz = channels_per_pixel == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  cuuint64_t dims[4] = {C, W, H, N};
  cuuint64_t strides[3] = {stride_w_bytes, stride_h_bytes, stride_n_bytes};
  int lower[2] = {lower_w, lower_h};
  int upper[2] = {upper_w, upper_h};
  cuuint32_t estr[4] = {1, (cuuint32_t)conv_stride, (cuuint32_t)conv_stride, 1};
  CUresult r = g_encode_im2col(out, g_tmap_fp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, lower,
                               upper, (cuuint32_t)channels_per_pixel, (cuuint32_t)pixels_per_column, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof(g_err),
             "cuTensorMapEncodeIm2col failed: %d (C=%llu W=%llu H=%llu N=%llu sw=%llu sh=%llu sn=%llu lo=(%d,%d) up=(%d,%d) s=%d)",
             (int)r, (unsigned long long)C, (unsigned long long)W, (unsigned long long)H, (unsigned long long)N,
             (unsigned long long)stride_w_bytes, (unsigned long long)stride_h_bytes, (unsigned long long)stride_n_bytes,
             lower_w, lower_h, upper_w, upper_h, conv_stride);
    return g_err;
  }
  // Same driver quirk CUTLASS works around (copy_traits_sm90_im2col.hpp): for tensors < 128 KiB, drivers <= 13.1
  // set a descriptor bit that breaks im2col loads.
  int drv = 0;
  cudaDriverGetVersion(&drv);
  if (drv <= 13010 && total_bytes < 131072) reinterpret_cast<uint64_t*>(out)[1] &= ~(1ull << 21);
  return nullptr;
}

size_t conv_gemm_smem_bytes(const ConvGemmParams& p) {
  const size_t a_bytes = p.a_mode == 3 ? (size_t)p.pt_stage_bytes : (size_t)p.msub * kABytes;
  const size_t b_bytes = (size_t)(p.cta2 ? p.block_n / 2 : p.block_n) * kBlockK * 2;
  const size_t epi = p.epi_mode == 2 ? (size_t)2 * kPatchBytes : (p.epi_mode == 1 ? (size_t)kEpiWarps * p.epi_bufs * kEpiUnitBytes : 0);
  return 1024 + (size_t)p.num_stages * a_bytes + (size_t)(p.a_mode == 3 ? p.num_k_blocks : p.num_stages) * b_bytes + epi +
         kEpiWarps * 128 * sizeof(float) + (2 * kMaxStages + 4 + kEpiWarps * kMaxEpiBufs + 1) * 8 + 16;
}

int conv_gemm_pick_stages(ConvGemmParams p) {
  const size_t budget = 227 * 1024;
  p.num_stages = kMaxStages;
  while (p.num_stages > 2 && conv_gemm_smem_bytes(p) > budget) --p.num_stages;
  return p.num_stages;
}

int conv_patch_stage_bytes(int pt_wp, int dil) {
  // 256 accumulator rows + the largest tap shift, 128 B per row, rounded up to the 1024 B swizzle period
  const int rows = 256 + (2 * pt_wp + 2) * dil;
  return (rows * 128 + 1023) / 1024 * 1024;
}

const char* make_tmap_tiled4d(CUtensorMap* out, const void* base, uint64_t C, uint64_t W, uint64_t H, uint64_t N,
                              uint64_t stride_w_bytes, uint64_t stride_h_bytes, uint64_t stride_n_bytes, uint32_t box_w,
                              uint32_t box_h) {
  if (const char* e = tma_init()) return e;
  if (C != 64) return "make_tmap_tiled4d: 64 channels expected";
  cuuint64_t dims[4] = {C, W, H, N};
  cuuint64_t strides[3] = {stride_w_bytes, stride_h_bytes, stride_n_bytes};
  cuuint32_t box[4] = {(cuuint32_t)C, box_w, box_h, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  if (box_w > 256 || box_h > 256) return "make_tmap_tiled4d: box too large";
  CUresult r = g_encode_tiled(out, g_tmap_fp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims,
                              strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_128B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof(g_err), "cuTensorMapEncodeTiled (4-D) failed: %d", (int)r);
    return g_err;
  }
  return nullptr;
}

cudaError_t launch_conv_gemm(const ConvGemmParams& p, int num_sms, cudaStream_t stream) {
  static bool attr_set = false;
  const void* fns[8] = {(const void*)conv_gemm_kernel<false, false, false>, (const void*)conv_gemm_kernel<true, false, false>,
                        (const void*)conv_gemm_kernel<false, true, false>,  (const void*)conv_gemm_kernel<true, true, false>,
                        (const void*)conv_gemm_kernel<false, false, true>,  (const void*)conv_gemm_kernel<true, false, true>,
                        (const void*)conv_gemm_kernel<false, true, true>,   (const void*)conv_gemm_kernel<true, true, true>};
  if (!attr_set) {
    for (const void* f : fns) {
      cudaError_t e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
      if (e != cudaSuccess) return e;
    }
    attr_set = true;
  }
  if (p.mask_act != nullptr && (p.epi_mode != 1 || p.colsum_part == nullptr || p.scale != nullptr || p.shift != nullptr))
    return cudaErrorInvalidValue;
  const int tiles = p.num_m_blocks * p.num_n_blocks;
  int grid = tiles < num_sms ? tiles : num_sms;
  if (p.cta2) {   // one tile per CTA pair
    grid = 2 * tiles < num_sms ? 2 * tiles : (num_sms & ~1);
  }
  const size_t smem = conv_gemm_smem_bytes(p);
  if (smem > 227 * 1024) return cudaErrorInvalidConfiguration;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (p.cta2) {
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = 2;
    attr[1].val.clusterDim.y = 1;
    attr[1].val.clusterDim.z = 1;
    cfg.numAttrs = 2;
  }
  const void* fn = fns[(p.fp16 ? 1 : 0) + (p.cta2 ? 2 : 0) + (p.mask_act != nullptr ? 4 : 0)];
  void* args[1] = {const_cast<ConvGemmParams*>(&p)};
  return cudaLaunchKernelExC(&cfg, fn, args);
}

}  // namespace dgp
