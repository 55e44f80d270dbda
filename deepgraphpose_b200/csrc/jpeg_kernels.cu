// Motion-JPEG of the labelled video: baseline JPEG, 4:2:0, one restart interval per MCU row, byte-identical to
// `PIL.Image.save(format="JPEG", quality=q, subsampling=2, restart_marker_rows=1)` (libjpeg-turbo).  The contract is in
// include/dgp_b200.h and DESIGN.md §4.5.
//
// Restart markers make every MCU row an independent entropy-coded segment, so one frame is encoded by four launches:
//   1. transform: colour conversion, 2x2 chroma downsampling, islow DCT and quantisation, 8 threads per 8x8 block;
//   2. entropy:   one CTA per segment: bit length of each block, a scan of the lengths, then every thread ORs its codes
//                 into the segment's zeroed bit buffer at its own offset; the CTA counts the 0xFF bytes stuffing will add;
//   3. layout:    a scan over segments (and frames) gives every segment's place in the packed output and every frame's
//                 size and offset; a frame above its proven bound is reported (size -1) and not written;
//   4. pack:      one CTA per segment copies its bytes with 0xFF -> 0xFF 0x00 stuffing behind the header template and
//                 appends RSTn (or EOI).
#include "../../include/dgp_b200.h"

#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

#include "handle.cuh"

namespace dgp {
namespace {

constexpr int kThreads = 256;
constexpr int kBlockBits = 64 * 27;      // 64 coefficients x (16-bit longest code + 11 magnitude bits): a block's bound
constexpr int kBlockBytes = kBlockBits / 8;
constexpr int kTableHeader = 640;        // the header template, padded; the Huffman codes follow it in the table buffer

// natural (row-major) index -> zig-zag position
__constant__ uint8_t c_zigzag_of[64] = {0,  1,  5,  6,  14, 15, 27, 28, 2,  4,  7,  13, 16, 26, 29, 42,
                                        3,  8,  12, 17, 25, 30, 41, 43, 9,  11, 18, 24, 31, 40, 44, 53,
                                        10, 19, 23, 32, 39, 45, 52, 54, 20, 22, 33, 38, 46, 51, 55, 60,
                                        21, 34, 37, 47, 50, 56, 59, 61, 35, 36, 48, 49, 57, 58, 62, 63};

// Annex K tables
const uint8_t kLumaQ[64] = {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
                            14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
                            18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
                            49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
const uint8_t kChromaQ[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99,
                              99, 99, 47, 66, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
                              99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};
const uint8_t kZigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                             41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                             30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
const uint8_t kDcLumaBits[16] = {0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0};
const uint8_t kDcChromaBits[16] = {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0};
const uint8_t kDcVals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
const uint8_t kAcLumaBits[16] = {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d};
const uint8_t kAcLumaVals[162] = {
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14, 0x32, 0x81,
    0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0a, 0x16, 0x17, 0x18,
    0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48,
    0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75,
    0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99,
    0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
    0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5,
    0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
const uint8_t kAcChromaBits[16] = {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77};
const uint8_t kAcChromaVals[162] = {
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32, 0x81, 0x08,
    0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25,
    0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47,
    0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74,
    0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97,
    0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
    0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4,
    0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};

// Frame geometry: MCUs (16x16 pixels: Y0 Y1 Y2 Y3 Cb Cr), luma blocks inside the component, chroma rows.
struct Geom {
  int H, W, mcux, mcuy, ywib, yhib, cH;
  int nbr;          // blocks per MCU row (= per segment)
  int seg_words;    // 32-bit words of one segment's bit buffer
  int64_t nbf;      // blocks per frame
  int64_t frame_cap;
};

Geom geom(int H, int W) {
  Geom g;
  g.H = H;
  g.W = W;
  g.mcux = (W + 15) / 16;
  g.mcuy = (H + 15) / 16;
  g.ywib = (W + 7) / 8;
  g.yhib = (H + 7) / 8;
  g.cH = (H + 1) / 2;
  g.nbr = g.mcux * 6;
  g.seg_words = g.nbr * (kBlockBits / 32) + 1;  // + the 1..7 padding bits
  g.nbf = (int64_t)g.mcuy * g.nbr;
  // header + per segment: its bytes doubled by stuffing, then RSTn; EOI
  g.frame_cap = kJpegHeaderBytes + (int64_t)g.mcuy * (2 * ((int64_t)g.nbr * kBlockBytes + 1) + 2) + 2;
  return g;
}

struct QuantArgs {
  uint16_t div[2][64];  // 8 * Q in natural order: luma, chroma
};

// libjpeg's jccolor.c fixed point (16 scale bits)
__device__ __forceinline__ int luma(int r, int g, int b) { return (19595 * r + 38470 * g + 7471 * b + 32768) >> 16; }
__device__ __forceinline__ int chroma(int r, int g, int b, bool cr) {
  return cr ? (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16
            : (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16;
}

__device__ __forceinline__ int descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }

// One 1-D pass of libjpeg's jfdctint.c (islow: 13 constant bits, 2 pass-1 bits); outputs of the 2-D transform are scaled by 8.
template <bool kFirst>
__device__ __forceinline__ void fdct_pass(const int* d, int* o) {
  constexpr int kSh = kFirst ? 11 : 15;
  int t0 = d[0] + d[7], t7 = d[0] - d[7], t1 = d[1] + d[6], t6 = d[1] - d[6];
  int t2 = d[2] + d[5], t5 = d[2] - d[5], t3 = d[3] + d[4], t4 = d[3] - d[4];
  const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
  if (kFirst) {
    o[0] = (t10 + t11) * 4;
    o[4] = (t10 - t11) * 4;
  } else {
    o[0] = descale(t10 + t11, 2);
    o[4] = descale(t10 - t11, 2);
  }
  int z1 = (t12 + t13) * 4433;
  o[2] = descale(z1 + t13 * 6270, kSh);
  o[6] = descale(z1 - t12 * 15137, kSh);
  z1 = t4 + t7;
  int z2 = t5 + t6, z3 = t4 + t6, z4 = t5 + t7;
  const int z5 = (z3 + z4) * 9633;
  t4 *= 2446;
  t5 *= 16819;
  t6 *= 25172;
  t7 *= 12299;
  z1 *= -7373;
  z2 *= -20995;
  z3 = z3 * -16069 + z5;
  z4 = z4 * -3196 + z5;
  o[7] = descale(t4 + z1 + z3, kSh);
  o[5] = descale(t5 + z2 + z4, kSh);
  o[3] = descale(t6 + z2 + z3, kSh);
  o[1] = descale(t7 + z1 + z4, kSh);
}

// Launch 1: blockIdx.y = frame, 32 blocks per CTA in MCU order, thread = (block, row).  Pass 1 transforms the thread's
// row, pass 2 its column; coefficients are stored in zig-zag order.  Luma blocks outside the component (the right half of
// the last MCU column, the bottom half of the last MCU row) are stored as zeros; their DC is resolved by the entropy coder.
__global__ void __launch_bounds__(kThreads) jpeg_transform_kernel(const uint8_t* __restrict__ frames, const Geom g,
                                                                  const QuantArgs q, int16_t* __restrict__ coef) {
  __shared__ int rows[32][8][9];
  const int lb = threadIdx.x >> 3, r = threadIdx.x & 7;
  const int64_t b = (int64_t)blockIdx.x * 32 + lb;
  const int f = blockIdx.y;
  const bool valid = b < g.nbf;
  int p = 0;
  bool dummy = true;
  if (valid) {
    const int64_t mcu = b / 6;
    p = (int)(b - mcu * 6);
    const int my = (int)(mcu / g.mcux), mx = (int)(mcu - (int64_t)my * g.mcux);
    const uint8_t* img = frames + (size_t)f * g.H * g.W * 3;
    int s[8];
    if (p < 4) {
      const int by = 2 * my + (p >> 1), bx = 2 * mx + (p & 1);
      dummy = bx >= g.ywib || by >= g.yhib;
      if (!dummy) {
        const uint8_t* row = img + (size_t)min(by * 8 + r, g.H - 1) * g.W * 3;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const uint8_t* px = row + (size_t)min(bx * 8 + c, g.W - 1) * 3;
          s[c] = luma(px[0], px[1], px[2]) - 128;
        }
      }
    } else {
      // rows past the last chroma row repeat it (the downsampled plane is padded, not the source)
      dummy = false;
      const bool cr = p == 5;
      const int cy = min(my * 8 + r, g.cH - 1);
      const uint8_t* r0 = img + (size_t)(2 * cy) * g.W * 3;
      const uint8_t* r1 = img + (size_t)min(2 * cy + 1, g.H - 1) * g.W * 3;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int cx = mx * 8 + c;
        const size_t x0 = (size_t)min(2 * cx, g.W - 1) * 3, x1 = (size_t)min(2 * cx + 1, g.W - 1) * 3;
        const int sum = chroma(r0[x0], r0[x0 + 1], r0[x0 + 2], cr) + chroma(r0[x1], r0[x1 + 1], r0[x1 + 2], cr) +
                        chroma(r1[x0], r1[x0 + 1], r1[x0 + 2], cr) + chroma(r1[x1], r1[x1 + 1], r1[x1 + 2], cr);
        s[c] = ((sum + 1 + (cx & 1)) >> 2) - 128;  // bias 1, 2, 1, 2, ... along the row (jcsample.c h2v2_downsample)
      }
    }
    if (!dummy) {
      int o[8];
      fdct_pass<true>(s, o);
#pragma unroll
      for (int k = 0; k < 8; ++k) rows[lb][r][k] = o[k];
    }
  }
  __syncthreads();
  if (!valid) return;
  int16_t* out = coef + ((size_t)f * g.nbf + b) * 64;
  if (dummy) {
#pragma unroll
    for (int i = 0; i < 8; ++i) out[c_zigzag_of[i * 8 + r]] = 0;
    return;
  }
  int d[8], o[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) d[i] = rows[lb][i][r];
  fdct_pass<false>(d, o);
  const uint16_t* div = q.div[p < 4 ? 0 : 1];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int dv = div[i * 8 + r];
    const int a = abs(o[i]);
    const int v = (a + (dv >> 1)) / dv;
    out[c_zigzag_of[i * 8 + r]] = (int16_t)(o[i] < 0 ? -v : v);
  }
}

__device__ __forceinline__ bool luma_dummy(const Geom& g, int my, int mx, int p) {
  return 2 * mx + (p & 1) >= g.ywib || 2 * my + (p >> 1) >= g.yhib;
}

// DC of block p of MCU mx: a dummy luma block takes the DC of the block before it in MCU order (block 0 is always real).
__device__ __forceinline__ int block_dc(const int16_t* seg, const Geom& g, int my, int mx, int p) {
  if (p < 4)
    while (p > 0 && luma_dummy(g, my, mx, p)) --p;
  return seg[((size_t)mx * 6 + p) * 64];
}

__device__ __forceinline__ int nbits(int v) { return v ? 32 - __clz(abs(v)) : 0; }

// Bit writer of one block into the segment's buffer (32-bit words, most significant bit first).  Only the first and the
// last word of a block can be shared with its neighbours; every word is ORed atomically.
struct BitSink {
  uint32_t* words;
  int64_t word;
  uint64_t acc;
  int filled;
  __device__ BitSink(uint32_t* w, int64_t pos) : words(w), word(pos >> 5), acc(0), filled((int)(pos & 31)) {}
  __device__ __forceinline__ void put(uint32_t code, int len) {
    acc = (acc << len) | code;
    filled += len;
    if (filled >= 32) {
      filled -= 32;
      atomicOr(&words[word++], (uint32_t)(acc >> filled));
      acc &= (1ull << filled) - 1;
    }
  }
  __device__ __forceinline__ void flush() {
    if (filled) atomicOr(&words[word], (uint32_t)(acc << (32 - filled)));
  }
};

struct BitCount {
  int64_t bits = 0;
  __device__ __forceinline__ void put(uint32_t, int len) { bits += len; }
};

// huff[t][symbol] = code | length << 16; t: 0 DC luma, 1 AC luma, 2 DC chroma, 3 AC chroma (jchuff.c encode_one_block)
template <class Sink>
__device__ void encode_block(Sink& out, const int16_t* blk, int dc, int pred, const uint32_t* hdc, const uint32_t* hac) {
  const int diff = dc - pred;
  int n = nbits(diff);
  uint32_t h = hdc[n];
  out.put((h & 0xFFFF), h >> 16);
  if (n) out.put((uint32_t)(diff < 0 ? diff - 1 : diff) & ((1u << n) - 1), n);
  int run = 0;
  for (int k = 1; k < 64; ++k) {
    const int v = blk[k];
    if (v == 0) {
      ++run;
      continue;
    }
    while (run > 15) {
      h = hac[0xF0];
      out.put(h & 0xFFFF, h >> 16);
      run -= 16;
    }
    n = nbits(v);
    h = hac[(run << 4) | n];
    out.put(((h & 0xFFFF) << n) | ((uint32_t)(v < 0 ? v - 1 : v) & ((1u << n) - 1)), (h >> 16) + n);
    run = 0;
  }
  if (run) {
    h = hac[0];
    out.put(h & 0xFFFF, h >> 16);
  }
}

// Launch 2: blockIdx = (segment = MCU row, frame).
__global__ void __launch_bounds__(kThreads) jpeg_entropy_kernel(const int16_t* __restrict__ coef, const Geom g,
                                                                const uint32_t* __restrict__ huff_g,
                                                                int64_t* __restrict__ bitoff, uint32_t* __restrict__ raw,
                                                                int64_t* __restrict__ seg_bytes) {
  typedef cub::BlockScan<int64_t, kThreads> Scan;
  typedef cub::BlockReduce<int64_t, kThreads> Reduce;
  __shared__ union {
    typename Scan::TempStorage scan;
    typename Reduce::TempStorage reduce;
  } tmp;
  __shared__ uint32_t huff[4 * 256];
  for (int i = threadIdx.x; i < 4 * 256; i += kThreads) huff[i] = huff_g[i];
  const int my = blockIdx.x, f = blockIdx.y;
  const int64_t seg_id = (int64_t)f * g.mcuy + my;
  const int16_t* seg = coef + ((size_t)f * g.nbf + (size_t)my * g.nbr) * 64;
  int64_t* off = bitoff + seg_id * g.nbr;
  uint32_t* words = raw + seg_id * g.seg_words;
  __syncthreads();
  int64_t running = 0;
  for (int base = 0; base < g.nbr; base += kThreads) {
    const int i = base + threadIdx.x;
    int64_t bits = 0;
    if (i < g.nbr) {
      const int mx = i / 6, p = i - mx * 6;
      const int pred = p < 4 ? (p > 0 ? block_dc(seg, g, my, mx, p - 1) : (mx > 0 ? block_dc(seg, g, my, mx - 1, 3) : 0))
                             : (mx > 0 ? seg[((size_t)(mx - 1) * 6 + p) * 64] : 0);
      const int t = p < 4 ? 0 : 2;
      BitCount c;
      encode_block(c, seg + (size_t)i * 64, block_dc(seg, g, my, mx, p), pred, huff + t * 256, huff + (t + 1) * 256);
      bits = c.bits;
    }
    int64_t ex, tot;
    Scan(tmp.scan).ExclusiveSum(bits, ex, tot);
    if (i < g.nbr) off[i] = running + ex;
    running += tot;
    __syncthreads();
  }
  const int64_t nbytes = (running + 7) >> 3;
  const int64_t nwords = (nbytes + 3) >> 2;
  for (int64_t w = threadIdx.x; w < nwords; w += kThreads) words[w] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < g.nbr; i += kThreads) {
    const int mx = i / 6, p = i - mx * 6;
    const int pred = p < 4 ? (p > 0 ? block_dc(seg, g, my, mx, p - 1) : (mx > 0 ? block_dc(seg, g, my, mx - 1, 3) : 0))
                           : (mx > 0 ? seg[((size_t)(mx - 1) * 6 + p) * 64] : 0);
    const int t = p < 4 ? 0 : 2;
    BitSink s(words, off[i]);
    encode_block(s, seg + (size_t)i * 64, block_dc(seg, g, my, mx, p), pred, huff + t * 256, huff + (t + 1) * 256);
    s.flush();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const int pad = (int)((8 - (running & 7)) & 7);  // 1-bits up to the byte boundary (jchuff.c flush_bits)
    if (pad) {
      BitSink s(words, running);
      s.put((1u << pad) - 1, pad);
      s.flush();
    }
  }
  __syncthreads();
  int64_t ff = 0;
  for (int64_t k = threadIdx.x; k < nbytes; k += kThreads) ff += ((words[k >> 2] >> (24 - 8 * (k & 3))) & 0xFF) == 0xFF;
  ff = Reduce(tmp.reduce).Sum(ff);
  if (threadIdx.x == 0) {
    seg_bytes[2 * seg_id] = nbytes;
    seg_bytes[2 * seg_id + 1] = nbytes + ff + (my < g.mcuy - 1 ? 2 : 0);  // stuffed, with its RSTn
  }
}

// Launch 3 (one CTA): segment offsets inside each frame, frame sizes and the offsets of the packed frames.
__global__ void __launch_bounds__(1024) jpeg_layout_kernel(const Geom g, int N, int64_t* __restrict__ seg_bytes,
                                                           int64_t* __restrict__ offsets, int64_t* __restrict__ sizes) {
  typedef cub::BlockScan<int64_t, 1024> Scan;
  __shared__ typename Scan::TempStorage tmp;
  int64_t packed = 0;
  for (int f = 0; f < N; ++f) {
    int64_t running = kJpegHeaderBytes;
    for (int base = 0; base < g.mcuy; base += 1024) {
      const int s = base + threadIdx.x;
      const int64_t id = (int64_t)f * g.mcuy + s;
      const int64_t len = s < g.mcuy ? seg_bytes[2 * id + 1] : 0;
      int64_t ex, tot;
      Scan(tmp).ExclusiveSum(len, ex, tot);
      if (s < g.mcuy) seg_bytes[2 * id + 1] = running + ex;  // now: the segment's offset in its frame
      running += tot;
      __syncthreads();
    }
    const int64_t size = running + 2;
    const bool ok = size <= g.frame_cap;
    if (threadIdx.x == 0) {
      offsets[f] = packed;
      sizes[f] = ok ? size : -1;
    }
    if (ok) packed += size;
  }
}

// Launch 4: blockIdx = (segment, frame).  The first segment's CTA also writes the header, the last one EOI.
__global__ void __launch_bounds__(kThreads) jpeg_pack_kernel(const Geom g, const uint32_t* __restrict__ raw,
                                                             const int64_t* __restrict__ seg_bytes,
                                                             const uint8_t* __restrict__ header,
                                                             const int64_t* __restrict__ offsets,
                                                             const int64_t* __restrict__ sizes, uint8_t* __restrict__ out) {
  typedef cub::BlockScan<int, kThreads> Scan;
  __shared__ typename Scan::TempStorage tmp;
  const int my = blockIdx.x, f = blockIdx.y;
  const int64_t size = sizes[f];
  if (size < 0) return;
  uint8_t* dst = out + offsets[f];
  if (my == 0)
    for (int i = threadIdx.x; i < kJpegHeaderBytes; i += kThreads) dst[i] = header[i];
  const int64_t seg_id = (int64_t)f * g.mcuy + my;
  const uint32_t* words = raw + seg_id * g.seg_words;
  const int64_t nbytes = seg_bytes[2 * seg_id];
  uint8_t* o = dst + seg_bytes[2 * seg_id + 1];
  int64_t running = 0;
  for (int64_t base = 0; base < nbytes; base += kThreads) {
    const int64_t k = base + threadIdx.x;
    const uint32_t b = k < nbytes ? (words[k >> 2] >> (24 - 8 * (k & 3))) & 0xFF : 0;
    const int ff = k < nbytes && b == 0xFF;
    int ex, tot;
    Scan(tmp).ExclusiveSum(ff, ex, tot);
    if (k < nbytes) {
      const int64_t at = k + running + ex;
      o[at] = (uint8_t)b;
      if (ff) o[at + 1] = 0;
    }
    running += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    uint8_t* m = o + nbytes + running;
    m[0] = 0xFF;
    m[1] = my < g.mcuy - 1 ? (uint8_t)(0xD0 + (my & 7)) : 0xD9;
  }
}

void huff_codes(const uint8_t* bits, const uint8_t* vals, uint32_t* table) {
  uint32_t code = 0;
  int k = 0;
  for (int len = 1; len <= 16; ++len) {
    for (int i = 0; i < bits[len - 1]; ++i) table[vals[k++]] = code++ | (uint32_t)len << 16;
    code <<= 1;
  }
}

void quant_table(const uint8_t* base, int quality, uint16_t* natural) {
  const int scale = quality < 50 ? 5000 / quality : 200 - 2 * quality;
  for (int i = 0; i < 64; ++i) {
    int v = (base[i] * scale + 50) / 100;
    natural[i] = (uint16_t)(v < 1 ? 1 : v > 255 ? 255 : v);
  }
}

void put16(uint8_t*& p, int v) {
  *p++ = (uint8_t)(v >> 8);
  *p++ = (uint8_t)v;
}

// The bytes in front of the entropy-coded data: SOI, APP0 (JFIF 1.01), DQT x2, SOF0, DHT x4, DRI, SOS.
void header_template(int H, int W, const uint16_t q[2][64], uint8_t* out) {
  uint8_t* p = out;
  const uint8_t head[] = {0xFF, 0xD8, 0xFF, 0xE0, 0x00, 0x10, 'J', 'F', 'I', 'F', 0x00, 0x01, 0x01, 0x00, 0x00, 0x01, 0x00, 0x01,
                          0x00, 0x00};
  memcpy(p, head, sizeof(head));
  p += sizeof(head);
  for (int t = 0; t < 2; ++t) {
    *p++ = 0xFF;
    *p++ = 0xDB;
    put16(p, 67);
    *p++ = (uint8_t)t;
    for (int k = 0; k < 64; ++k) *p++ = (uint8_t)q[t][kZigzag[k]];
  }
  const uint8_t sof[] = {0xFF, 0xC0, 0x00, 0x11, 0x08};
  memcpy(p, sof, sizeof(sof));
  p += sizeof(sof);
  put16(p, H);
  put16(p, W);
  const uint8_t comps[] = {0x03, 0x01, 0x22, 0x00, 0x02, 0x11, 0x01, 0x03, 0x11, 0x01};
  memcpy(p, comps, sizeof(comps));
  p += sizeof(comps);
  struct { uint8_t id; const uint8_t* bits; const uint8_t* vals; } dht[4] = {
      {0x00, kDcLumaBits, kDcVals}, {0x10, kAcLumaBits, kAcLumaVals}, {0x01, kDcChromaBits, kDcVals},
      {0x11, kAcChromaBits, kAcChromaVals}};
  for (const auto& d : dht) {
    int n = 0;
    for (int i = 0; i < 16; ++i) n += d.bits[i];
    *p++ = 0xFF;
    *p++ = 0xC4;
    put16(p, 2 + 1 + 16 + n);
    *p++ = d.id;
    memcpy(p, d.bits, 16);
    p += 16;
    memcpy(p, d.vals, n);
    p += n;
  }
  const uint8_t dri[] = {0xFF, 0xDD, 0x00, 0x04};
  memcpy(p, dri, sizeof(dri));
  p += sizeof(dri);
  put16(p, (W + 15) / 16);
  const uint8_t sos[] = {0xFF, 0xDA, 0x00, 0x0C, 0x03, 0x01, 0x00, 0x02, 0x11, 0x03, 0x11, 0x00, 0x3F, 0x00};
  memcpy(p, sos, sizeof(sos));
  p += sizeof(sos);
}

bool valid_dims(int H, int W) { return H >= 1 && W >= 1 && H <= kJpegMaxDim && W <= kJpegMaxDim; }

}  // namespace

static_assert(kJpegHeaderBytes <= kTableHeader, "header template does not fit its slot");

// The header template and Huffman codes of one (H, W, quality), built on first use and kept on the handle.
static int jpeg_table(dgp_handle* h, int H, int W, int quality, QuantArgs* q, const uint8_t** dev) {
  quant_table(kLumaQ, quality, q->div[0]);
  quant_table(kChromaQ, quality, q->div[1]);
  const auto key = std::make_tuple(H, W, quality);
  auto it = h->jpeg_tables.find(key);
  if (it == h->jpeg_tables.end()) {
    std::vector<uint8_t> host(kTableHeader + 4 * 256 * 4, 0);
    header_template(H, W, q->div, host.data());
    uint32_t huff[4 * 256] = {};
    huff_codes(kDcLumaBits, kDcVals, huff);
    huff_codes(kAcLumaBits, kAcLumaVals, huff + 256);
    huff_codes(kDcChromaBits, kDcVals, huff + 512);
    huff_codes(kAcChromaBits, kAcChromaVals, huff + 768);
    memcpy(host.data() + kTableHeader, huff, sizeof(huff));
    DevBuf b;
    CU_OK(h, b.alloc(host.size()));
    CU_OK(h, cudaMemcpy(b.get(), host.data(), host.size(), cudaMemcpyHostToDevice));
    it = h->jpeg_tables.emplace(key, std::move(b)).first;
  }
  for (int t = 0; t < 2; ++t)
    for (int i = 0; i < 64; ++i) q->div[t][i] = (uint16_t)(q->div[t][i] * 8);
  *dev = it->second.get<uint8_t>();
  return DGP_OK;
}

int64_t jpeg_capacity(int H, int W) { return valid_dims(H, W) ? geom(H, W).frame_cap : -1; }

int encode_jpeg_impl(dgp_handle* h, const uint8_t* frames, int N, int H, int W, int quality, uint8_t* out, int64_t capacity,
                     int64_t* offsets, int64_t* sizes, cudaStream_t s) {
  if (N < 0 || N > 65535 || !valid_dims(H, W) || quality < 1 || quality > 100 ||
      (N > 0 && (!frames || !out || !offsets || !sizes)))
    return fail(h, DGP_ERR_INVALID, "dgp_encode_jpeg: bad argument (N %d, %dx%d, quality %d)", N, H, W, quality);
  const Geom g = geom(H, W);
  if (capacity < g.frame_cap * N)
    return fail(h, DGP_ERR_INVALID, "dgp_encode_jpeg: capacity %lld below %d x dgp_jpeg_capacity = %lld", (long long)capacity,
                N, (long long)(g.frame_cap * N));
  if (N == 0) return DGP_OK;
  QuantArgs q;
  const uint8_t* table = nullptr;
  int rc;
  if ((rc = jpeg_table(h, H, W, quality, &q, &table))) return rc;
  const int64_t segs = (int64_t)N * g.mcuy;
  if ((rc = ensure(h, &h->jpeg_coef, (size_t)N * g.nbf * 64 * sizeof(int16_t)))) return rc;
  if ((rc = ensure(h, &h->jpeg_bitoff, (size_t)N * g.nbf * sizeof(int64_t)))) return rc;
  if ((rc = ensure(h, &h->jpeg_raw, (size_t)segs * g.seg_words * sizeof(uint32_t)))) return rc;
  if ((rc = ensure(h, &h->jpeg_seg, (size_t)segs * 2 * sizeof(int64_t)))) return rc;
  int16_t* coef = h->jpeg_coef.get<int16_t>();
  uint32_t* raw = h->jpeg_raw.get<uint32_t>();
  int64_t* seg = h->jpeg_seg.get<int64_t>();
  jpeg_transform_kernel<<<dim3((unsigned)((g.nbf + 31) / 32), N), kThreads, 0, s>>>(frames, g, q, coef);
  CU_OK(h, cudaGetLastError());
  jpeg_entropy_kernel<<<dim3(g.mcuy, N), kThreads, 0, s>>>(coef, g, reinterpret_cast<const uint32_t*>(table + kTableHeader),
                                                           h->jpeg_bitoff.get<int64_t>(), raw, seg);
  CU_OK(h, cudaGetLastError());
  jpeg_layout_kernel<<<1, 1024, 0, s>>>(g, N, seg, offsets, sizes);
  CU_OK(h, cudaGetLastError());
  jpeg_pack_kernel<<<dim3(g.mcuy, N), kThreads, 0, s>>>(g, raw, seg, table, offsets, sizes, out);
  CU_OK(h, cudaGetLastError());
  h->launches += 4;
  return DGP_OK;
}

}  // namespace dgp

extern "C" {

int64_t dgp_jpeg_capacity(int H, int W) { return jpeg_capacity(H, W); }

int dgp_encode_jpeg(dgp_handle* h, const uint8_t* frames_dev, int N, int H, int W, int quality, uint8_t* out_dev,
                    int64_t capacity, int64_t* offsets_dev, int64_t* sizes_dev, void* stream) {
  if (!h) return DGP_ERR_INVALID;
  CU_OK(h, cudaSetDevice(h->device));
  return encode_jpeg_impl(h, frames_dev, N, H, W, quality, out_dev, capacity, offsets_dev, sizes_dev, (cudaStream_t)stream);
}

}  // extern "C"
