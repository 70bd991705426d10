// Fused stem of the inference plan (frozen_encoder.py): one kernel computes
//   out = maxpool3x3/s2/p1( relu( conv7x7/s2/p3(x, W) + bias ) )
// for the folded conv1 + bn1 + relu + maxpool children of the truncated encoder
// (Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:17,37-40), with tf32 operands and fp32 accumulation on tcgen05.
// The three-launch chain it replaces (space-to-depth staging, cuDNN convolution, max pool) moves 2.4 GB through HBM at
// batch 256 x 224^2; this kernel reads the fp32 image once and writes only the pooled (B, 64, H/4, W/4) result.
//
// The convolution is the 4x4 stride-1 one over the 2x2 space-to-depth image (pool.cuh, gh_stem_space_to_depth):
//   conv[y][x][o] = sum_{a,b < 4} sum_{k < 16} z[y + a][x + b][k] * W16[o][k][a][b]
// with z's cell (Y + 2, X + 2) holding, per image channel c, the 2x2 pixel block {x[c][2Y][2X], x[c][2Y][2X+1],
// x[c][2Y+1][2X], x[c][2Y+1][2X+1]} -- a 16-byte "k-chunk" -- and a zero 4th chunk (12 channels padded to 16).
//
// Implicit GEMM by descriptor shift. M = 128 consecutive conv columns of one conv row, N = 64 output channels, K = 16
// taps x 12 (the zero 4th k-chunk is never multiplied). The staged image rows live in shared memory K-major without
// swizzle as [k-chunk plane 0..2][row slot][cell][16 B]: one core matrix is 8 consecutive cells (SBO = 128 B between
// 8-cell groups). Tap (a, b) of the tile is the same staged rows with the descriptor start moved to row slot y + a and
// 16 B per cell of b, so there is no im2col copy. Per tap row a, six tf32 MMAs of 128 x 64 x 8: one per tap b for
// k-chunks 0 and 1 (planes 0 and 1, LBO = plane stride), and one per tap pair (b, b + 1) = (0, 1), (2, 3) for k-chunk 2
// (plane 2 at cell b, LBO = 16 B: the second "k-chunk" of the MMA is the next cell, i.e. tap b + 1). 24 MMAs per conv row.
//
// Tiles: 63 pooled columns per tile need the 127 conv columns 126 j - 1 .. 126 j + 125 (lane l = column 126 j - 1 + l),
// i.e. staged cells 126 j - 1 .. 126 j + 129 of each padded row (131 cells). 224^2 is one tile per row (lanes with no
// conv column are masked); wider images take ceil(PW / 63) tiles. The pooling windows of vertically adjacent pooled rows
// share one conv row; a ring of 8 TMEM accumulators (one 64-column accumulator per conv row) keeps it.
//
// Epilogue: max over the (up to) three conv rows of the window straight from TMEM, then over columns x-1, x, x+1 with
// shuffles (the one neighbour across a warp boundary goes through shared memory), then + bias and ReLU. Pooling the raw
// sums first is exact: fl(a + b) is monotone in a, so max_i fl(a_i + b) = fl(max_i a_i + b), and ReLU is monotone.
// NaN propagates as in nn.MaxPool2d / PoolVec::max_into, and ReLU keeps it, as torch's does.
//
// Work split: persistent CTAs, one per SM, each a contiguous range of (image, tile, pooled row) units; the conv row above
// a range's first pooled row is recomputed (halo). No atomics: an image's result does not depend on its batch.
// Warps: 0-6 producers (one staged row each, round robin), 7-14 epilogue (TMEM lane quadrant warp % 4, output channel
// half (warp - 7) / 4), 15 MMA issuer: 16 warps, so that each thread may hold 128 registers.
//
// Pixel type: fp32 images, or the uint8 pixels of the loaders (functions.uint8_transform) with ToTensor + Normalize
// applied in the producers (reference test_...:64-65, train_best_...:42-43). The uint8 kernel builds a [3][256] table
// of to_tensor_normalize() results in shared memory -- the values gh_normalize_u8 writes -- and looks each byte up, so
// its staged tf32 operands, and hence its output, are bitwise those of the fp32 kernel on the normalize_u8 batch.
// Cells outside the image stay 0: conv1's zero padding applies after Normalize. Only the producers' loads differ.
#pragma once
#include "common.cuh"
#include "preprocess.cuh"

namespace gh {

constexpr int kScProducerWarps = 7;
constexpr int kScEpiWarp0 = kScProducerWarps;
constexpr int kScEpiWarps = 8;                         // two per TMEM lane quadrant, 32 output channels each
constexpr int kScMmaWarp = kScEpiWarp0 + kScEpiWarps;
constexpr int kScThreads = (kScMmaWarp + 1) * 32;
constexpr int kScTileCols = 63;                        // pooled columns per tile
constexpr int kScCells = 131;                          // staged cells per row slot
constexpr int kScItems = 3 * kScCells;                 // (image channel, cell) k-chunks a producer warp stores per row
constexpr int kScItemIters = (kScItems + 31) / 32;
constexpr int kScSlots = 12;                           // staged row ring: 4 rows in use by the MMAs + 8 being produced
constexpr int kScAccSlots = 8;                         // TMEM accumulators (conv rows), 64 columns each
constexpr uint32_t kScSlotBytes = kScCells * 16;       // 2096
constexpr uint32_t kScPlaneBytes = kScSlots * kScSlotBytes;
constexpr uint32_t kScWBytes = 16 * 2 * 2048;          // 16 taps x 2 MMAs x (64 rows x 2 k-chunks x 16 B)
constexpr uint32_t kScAOff = kScWBytes;
constexpr uint32_t kScBiasOff = kScAOff + 3 * kScPlaneBytes;
constexpr uint32_t kScXbufOff = kScBiasOff + 64 * 4;
constexpr uint32_t kScBarOff = kScXbufOff + 2 * 4 * 64 * 4;
constexpr uint32_t kScBarBytes = 8 * (2 * kScSlots + 2 * kScAccSlots) + 16;
constexpr uint32_t kScSmemBytes = kScBarOff + kScBarBytes + 1024;
constexpr uint32_t kScTableOff = kScBarOff + kScBarBytes;        // uint8 pixels: [3][256] fp32 Normalize table
constexpr uint32_t kScSmemBytesU8 = kScSmemBytes + 3 * 256 * 4;

template <typename T>
struct StemConvPoolParams {
  const T* x;                          // float or uint8_t pixels
  long long s_img, s_c, s_y, s_x;      // element strides of x
  const float* w;                      // packed tf32 weights, the shared-memory image of the B operands (kScWBytes)
  const float* bias;                   // [64]
  float* out;                          // (B, PH, PW, 64)
  int B, OH, OW, PH, PW, tiles;        // conv size OH x OW = H/2 x W/2; pooled PH x PW; tiles per pooled row
  int vec2;                            // x-contiguous pixel pairs 2 * sizeof(T) aligned: one load per pair
  int units;                           // B * tiles * PH (the launcher keeps it below 2^30)
  float mean[3], std[3];               // uint8 pixels: Normalize's constants
};

// -DGH_SC_PROFILE: per-role cycle accounting (clock64 around every mbarrier wait, the TMEM loads, the epilogue's
// bar.sync and the store phase of one thread per role, summed over the CTAs into g_sc_prof and read back by
// gh_sc_profile_read; tools/prof_stem_roles.py). Slots: 0 issuer loop, 1 issuer wait aempty, 2 issuer wait full,
// 3 conv rows issued, 4 producer (warp 0) loop, 5 producer wait empty, 6 producer store phase (wait for its loads,
// cvt, STS, arrive), 7 rows staged by warp 0, 8 epilogue (warp kScEpiWarp0) loop, 9 epilogue wait afull, 10 epilogue
// TMEM loads and row max, 11 epilogue bar.sync, 12 epilogue column max + store, 13 pooled rows, 14 CTAs,
// 15 CTA lifetime (thread 0, prologue included).
#ifdef GH_SC_PROFILE
__device__ unsigned long long g_sc_prof[16];
#define GH_SC_DECL(var) long long var = 0
#define GH_SC_CLK(var) const long long var = clock64()
#define GH_SC_ADD(acc, var) acc += clock64() - var
#define GH_SC_FLUSH(slot, acc) atomicAdd(&g_sc_prof[slot], (unsigned long long)(acc))
#define GH_SC_INC(var) ++var
#else
#define GH_SC_DECL(var)
#define GH_SC_CLK(var)
#define GH_SC_ADD(acc, var)
#define GH_SC_FLUSH(slot, acc)
#define GH_SC_INC(var)
#endif

// max that propagates NaN (one FMNMX.NAN): a NaN operand gives a NaN, as in nn.MaxPool2d and torch.relu.
__device__ __forceinline__ float max_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}

// A CTA's range of units, cut where (image, tile) changes: one segment = consecutive pooled rows py0..py1-1 of one
// (image, tile), computed from conv rows y_lo..y_hi, staged from padded rows y_lo..y_hi + 3.
struct ScSeg {
  int b, j, py0, py1, y_lo, y_hi;
};
template <typename T>
__device__ __forceinline__ bool sc_next(const StemConvPoolParams<T>& p, int& u, int u1, ScSeg& s) {
  if (u >= u1) return false;
  const int bj = u / p.PH;
  const int end = (bj + 1) * p.PH < u1 ? (bj + 1) * p.PH : u1;
  s.b = bj / p.tiles;
  s.j = bj - s.b * p.tiles;
  s.py0 = u - bj * p.PH;
  s.py1 = s.py0 + (end - u);
  s.y_lo = 2 * s.py0 - 1 > 0 ? 2 * s.py0 - 1 : 0;
  s.y_hi = 2 * s.py1 - 1 < p.OH - 1 ? 2 * s.py1 - 1 : p.OH - 1;
  u = end;
  return true;
}

// The 2x2 pixel block {(2Y, 2X), (2Y, 2X+1), (2Y+1, 2X), (2Y+1, 2X+1)} of one channel at q, as the fp32 values the
// convolution sees. table: the channel's 256 Normalize results (uint8 pixels only).
__device__ __forceinline__ float4 sc_load_block(const StemConvPoolParams<float>& p, const float* q, const float*) {
  if (p.vec2) {
    const float2 t0 = __ldg(reinterpret_cast<const float2*>(q));
    const float2 t1 = __ldg(reinterpret_cast<const float2*>(q + p.s_y));
    return make_float4(t0.x, t0.y, t1.x, t1.y);
  }
  return make_float4(__ldg(q), __ldg(q + p.s_x), __ldg(q + p.s_y), __ldg(q + p.s_y + p.s_x));
}

__device__ __forceinline__ float4 sc_load_block(const StemConvPoolParams<uint8_t>& p, const uint8_t* q,
                                                const float* table) {
  uint32_t b0, b1, b2, b3;
  if (p.vec2) {
    const uint32_t t0 = __ldg(reinterpret_cast<const unsigned short*>(q));
    const uint32_t t1 = __ldg(reinterpret_cast<const unsigned short*>(q + p.s_y));
    b0 = t0 & 0xffu; b1 = t0 >> 8; b2 = t1 & 0xffu; b3 = t1 >> 8;
  } else {
    b0 = __ldg(q); b1 = __ldg(q + p.s_x); b2 = __ldg(q + p.s_y); b3 = __ldg(q + p.s_y + p.s_x);
  }
  return make_float4(table[b0], table[b1], table[b2], table[b3]);
}

template <typename T>
__global__ void __launch_bounds__(kScThreads, 1) stem_conv_pool_kernel(const StemConvPoolParams<T> p) {
  GH_SC_CLK(prof_cta0);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - raw);
  const uint32_t w_smem = base, a_smem = base + kScAOff;
  const float* bias_s = reinterpret_cast<const float*>(gbase + kScBiasOff);
  float* xbuf = reinterpret_cast<float*>(gbase + kScXbufOff);
  const uint32_t bar_full = base + kScBarOff, bar_empty = bar_full + 8 * kScSlots;
  const uint32_t bar_afull = bar_empty + 8 * kScSlots, bar_aempty = bar_afull + 8 * kScAccSlots;
  const uint32_t tmem_slot = bar_aempty + 8 * kScAccSlots;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + (tmem_slot - base));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // Weights and bias for the CTA's life.
  {
    const float4* wg = reinterpret_cast<const float4*>(p.w);
    float4* ws = reinterpret_cast<float4*>(gbase);
    for (int i = threadIdx.x; i < (int)(kScWBytes / 16); i += kScThreads) ws[i] = __ldg(wg + i);
    if (threadIdx.x < 64) reinterpret_cast<float*>(gbase + kScBiasOff)[threadIdx.x] = __ldg(p.bias + threadIdx.x);
    if constexpr (sizeof(T) == 1) {
      float* table = reinterpret_cast<float*>(gbase + kScTableOff);
      for (int i = threadIdx.x; i < 3 * 256; i += kScThreads) {
        const int c = i >> 8;
        table[i] = to_tensor_normalize((unsigned)(i & 255), c == 0 ? p.mean[0] : c == 1 ? p.mean[1] : p.mean[2],
                                       c == 0 ? p.std[0] : c == 1 ? p.std[1] : p.std[2]);
      }
    }
    fence_proxy_async_smem();
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < kScSlots; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int s = 0; s < kScAccSlots; ++s) {
      mbar_init(bar_afull + 8 * s, 1);
      mbar_init(bar_aempty + 8 * s, kScEpiWarps);
    }
    mbar_fence_init();
  }
  if (warp == kScMmaWarp) tmem_alloc(tmem_slot, 512);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const int u0 = (int)((long long)p.units * blockIdx.x / gridDim.x);
  const int u1 = (int)((long long)p.units * (blockIdx.x + 1) / gridDim.x);

  if (warp < kScProducerWarps) {
    // =========================== producers: one padded s2d row per warp, round robin ===========================
    uint32_t gs = 0;                                   // staged rows so far (all segments)
    int u = u0;
    ScSeg sg;
    GH_SC_DECL(prof_wait);
    GH_SC_DECL(prof_store);
    GH_SC_DECL(prof_n);
    GH_SC_CLK(prof_t0);
    while (sc_next(p, u, u1, sg)) {
      const int n_stage = sg.y_hi - sg.y_lo + 4;
      const T* img = p.x + (long long)sg.b * p.s_img;
      for (int k = 0; k < n_stage; ++k) {
        const uint32_t g = gs + (uint32_t)k;
        if ((int)(g % kScProducerWarps) != warp) continue;
        const uint32_t slot = g % kScSlots;
        const int Y = sg.y_lo + k - 2;                 // image cell row of padded row y_lo + k
        const bool row_ok = Y >= 0 && Y < p.OH;
        float4 v[kScItemIters];
#pragma unroll
        for (int it = 0; it < kScItemIters; ++it) {
          const int i = it * 32 + lane;
          const int c = i / kScCells, s = i - c * kScCells;
          const int X = kScTileCols * 2 * sg.j + s - 3;
          v[it] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (i < kScItems && row_ok && X >= 0 && X < p.OW) {
            const T* q = img + (long long)c * p.s_c + (long long)(2 * Y) * p.s_y + (long long)(2 * X) * p.s_x;
            v[it] = sc_load_block(p, q, reinterpret_cast<const float*>(gbase + kScTableOff) + c * 256);
          }
        }
        GH_SC_CLK(prof_w0);
        mbar_wait(bar_empty + 8 * slot, ((g / kScSlots) & 1u) ^ 1u, 300u + slot);
        GH_SC_ADD(prof_wait, prof_w0);
        GH_SC_CLK(prof_s0);
        GH_SC_INC(prof_n);
#pragma unroll
        for (int it = 0; it < kScItemIters; ++it) {
          const int i = it * 32 + lane;
          if (i < kScItems) {
            const int c = i / kScCells, s = i - c * kScCells;
            sts_u4(a_smem + (uint32_t)c * kScPlaneBytes + slot * kScSlotBytes + (uint32_t)s * 16u, tf32_rna(v[it].x),
                   tf32_rna(v[it].y), tf32_rna(v[it].z), tf32_rna(v[it].w));
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_full + 8 * slot);
        GH_SC_ADD(prof_store, prof_s0);
      }
      gs += (uint32_t)n_stage;
    }
#ifdef GH_SC_PROFILE
    if (warp == 0 && lane == 0) {
      long long prof_tot = 0;
      GH_SC_ADD(prof_tot, prof_t0);
      GH_SC_FLUSH(4, prof_tot);
      GH_SC_FLUSH(5, prof_wait);
      GH_SC_FLUSH(6, prof_store);
      GH_SC_FLUSH(7, prof_n);
    }
#endif
  } else if (warp == kScMmaWarp) {
    // =========================== MMA issuer ===========================
    constexpr uint32_t idesc = make_idesc_tf32(128, 64);
    // k-chunks (0, 1) of a tap: planes 0 and 1 (LBO = one plane) against packed [a][b][h=0][q=0..1] (LBO = 1024 B).
    // k-chunk 2 of the taps b and b + 1: cells b and b + 1 of plane 2 (LBO = 16 B, one cell; the last cell read is
    // 127 + 2 + 1 = 130 < kScCells) against packed [a][b][1][0] and [a][b + 1][1][0] (LBO = 4096 B, one tap).
    const uint64_t adesc0 = make_smem_desc_noswz(a_smem, kScPlaneBytes, 128);
    const uint64_t bdesc0 = make_smem_desc_noswz(w_smem, 1024, 128);
    const uint64_t adesc2 = make_smem_desc_noswz(a_smem + 2 * kScPlaneBytes, 16, 128);
    const uint64_t bdesc2 = make_smem_desc_noswz(w_smem + 2048, 4096, 128);
    uint32_t gs = 0, gc = 0;
    int u = u0;
    ScSeg sg;
    GH_SC_DECL(prof_ae);
    GH_SC_DECL(prof_full);
    GH_SC_CLK(prof_t0);
    while (sc_next(p, u, u1, sg)) {
      const int n_conv = sg.y_hi - sg.y_lo + 1;
      for (int k = 0; k < n_conv; ++k, ++gc) {
        const uint32_t acc = gc % kScAccSlots;
        GH_SC_CLK(prof_w0);
        mbar_wait(bar_aempty + 8 * acc, ((gc / kScAccSlots) & 1u) ^ 1u, 400u + acc);
        GH_SC_ADD(prof_ae, prof_w0);
        GH_SC_CLK(prof_w1);
        uint32_t slot[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          const uint32_t g = gs + (uint32_t)(k + a);
          slot[a] = g % kScSlots;
          mbar_wait(bar_full + 8 * slot[a], (g / kScSlots) & 1u, 500u + slot[a]);
        }
        GH_SC_ADD(prof_full, prof_w1);
        tc_fence_after_sync();
        if (elect_one()) {
          const uint32_t d = tmem_base + acc * 64u;
#pragma unroll
          for (int a = 0; a < 4; ++a) {
            const uint32_t row = (slot[a] * kScSlotBytes) >> 4;
#pragma unroll
            for (int b = 0; b < 4; ++b)
              umma_tf32(d, adesc0 + row + b, bdesc0 + (((a * 4 + b) * 2 * 2048) >> 4), idesc, (a | b) != 0);
#pragma unroll
            for (int b = 0; b < 4; b += 2)
              umma_tf32(d, adesc2 + row + b, bdesc2 + (((a * 4 + b) * 2 * 2048) >> 4), idesc, 1u);
          }
          umma_commit(bar_afull + 8 * acc);
          umma_commit(bar_empty + 8 * slot[0]);        // padded row y is not read by conv rows below y
          if (k == n_conv - 1)
            for (int a = 1; a < 4; ++a) umma_commit(bar_empty + 8 * slot[a]);
        }
        __syncwarp();
      }
      gs += (uint32_t)(n_conv + 3);
    }
#ifdef GH_SC_PROFILE
    if (lane == 0) {
      long long prof_tot = 0;
      GH_SC_ADD(prof_tot, prof_t0);
      GH_SC_FLUSH(0, prof_tot);
      GH_SC_FLUSH(1, prof_ae);
      GH_SC_FLUSH(2, prof_full);
      GH_SC_FLUSH(3, gc);
    }
#endif
  } else {
    // =========================== epilogue: TMEM -> 3x3/s2 max -> + bias, ReLU -> NHWC ===========================
    // A warp reads TMEM lane quadrant warp % 4 (the quadrant a warp may access) and output channels 32 half .. + 31.
    // A window's rows are loaded back to back and waited for once; the window's last row is kept in registers as the
    // next window's first row, so each conv row leaves TMEM once and its accumulator is released as soon as it is read.
    const int quad = warp & 3, half = (warp - kScEpiWarp0) >> 2;
    const uint32_t tlane = tmem_base + ((uint32_t)(32 * quad) << 16) + 32u * (uint32_t)half;
    const float* bias_h = bias_s + 32 * half;
    const float neg_inf = -__int_as_float(0x7f800000);
    uint32_t gc = 0, xb = 0;
    int u = u0;
    ScSeg sg;
    GH_SC_DECL(prof_af);
    GH_SC_DECL(prof_ld);
    GH_SC_DECL(prof_bar);
    GH_SC_DECL(prof_st);
    GH_SC_DECL(prof_n);
    GH_SC_CLK(prof_t0);
    while (sc_next(p, u, u1, sg)) {
      const int x = kScTileCols * 2 * sg.j - 1 + 32 * quad + lane;     // this lane's conv column
      const bool col_ok = x >= 0 && x < p.OW;
      auto acc_of = [&](int y) { return (gc + (uint32_t)(y - sg.y_lo)) % kScAccSlots; };
      auto wait_row = [&](int y) {
        const uint32_t g = gc + (uint32_t)(y - sg.y_lo);
        mbar_wait(bar_afull + 8 * (g % kScAccSlots), (g / kScAccSlots) & 1u, 600u + g % kScAccSlots);
      };
      uint32_t ra[32];                                                 // conv row 2 py - 1 of the current window
      for (int py = sg.py0; py < sg.py1; ++py) {
        const int ya = 2 * py - 1, yb = 2 * py, yc = 2 * py + 1;
        const bool ha = ya >= sg.y_lo, hc = yc <= sg.y_hi, first = py == sg.py0;
        GH_SC_CLK(prof_w0);
        if (first && ha) wait_row(ya);
        wait_row(yb);
        if (hc) wait_row(yc);
        GH_SC_ADD(prof_af, prof_w0);
        GH_SC_CLK(prof_l0);
        GH_SC_INC(prof_n);
        tc_fence_after_sync();
        uint32_t rb[32], rc[32];
        if (first && ha) tmem_ld32_nowait(tlane + acc_of(ya) * 64u, ra);
        tmem_ld32_nowait(tlane + acc_of(yb) * 64u, rb);
        if (hc) tmem_ld32_nowait(tlane + acc_of(yc) * 64u, rc);
        tmem_ld_wait();
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) {
          if (first && ha) mbar_arrive(bar_aempty + 8 * acc_of(ya));
          mbar_arrive(bar_aempty + 8 * acc_of(yb));
          if (hc) mbar_arrive(bar_aempty + 8 * acc_of(yc));
        }
        float m[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          m[i] = __uint_as_float(rb[i]);
          if (ha) m[i] = max_nan(m[i], __uint_as_float(ra[i]));
          if (hc) m[i] = max_nan(m[i], __uint_as_float(rc[i]));
          ra[i] = rc[i];
        }
        GH_SC_ADD(prof_ld, prof_l0);
        if (!col_ok) {
#pragma unroll
          for (int i = 0; i < 32; ++i) m[i] = neg_inf;
        }
        // column x + 2 of lane 30 is lane 0 of the next quadrant
        float* xs = xbuf + xb * 256 + 32 * half;
        if (lane == 0 && quad > 0) {
#pragma unroll
          for (int i = 0; i < 32; i += 4)
            *reinterpret_cast<float4*>(xs + quad * 64 + i) = make_float4(m[i], m[i + 1], m[i + 2], m[i + 3]);
        }
        GH_SC_CLK(prof_b0);
        asm volatile("bar.sync %0, 128;" ::"r"(1 + half) : "memory");   // the four warps of this channel half
        GH_SC_ADD(prof_bar, prof_b0);
        GH_SC_CLK(prof_s0);
        const bool from_next = lane == 30 && quad < 3;
        const int qx = 16 * quad + (lane >> 1);                         // pooled column within the tile
        const int px = kScTileCols * sg.j + qx;
        const bool store = !(lane & 1) && qx < kScTileCols && px < p.PW;
        float4* o = reinterpret_cast<float4*>(p.out + (((long long)sg.b * p.PH + py) * p.PW + px) * 64 + 32 * half);
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          float r4[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float v1 = __shfl_down_sync(0xffffffffu, m[i + e], 1);
            float v2 = __shfl_down_sync(0xffffffffu, m[i + e], 2);
            if (from_next) v2 = xs[(quad + 1) * 64 + i + e];
            float t = max_nan(max_nan(m[i + e], v1), v2) + bias_h[i + e];
            r4[e] = max_nan(t, 0.f);
          }
          if (store) o[i / 4] = make_float4(r4[0], r4[1], r4[2], r4[3]);
        }
        xb ^= 1u;
        GH_SC_ADD(prof_st, prof_s0);
      }
      gc += (uint32_t)(sg.y_hi - sg.y_lo + 1);
    }
#ifdef GH_SC_PROFILE
    if (warp == kScEpiWarp0 && lane == 0) {
      long long prof_tot = 0;
      GH_SC_ADD(prof_tot, prof_t0);
      GH_SC_FLUSH(8, prof_tot);
      GH_SC_FLUSH(9, prof_af);
      GH_SC_FLUSH(10, prof_ld);
      GH_SC_FLUSH(11, prof_bar);
      GH_SC_FLUSH(12, prof_st);
      GH_SC_FLUSH(13, prof_n);
    }
#endif
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == kScMmaWarp) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
#ifdef GH_SC_PROFILE
  if (threadIdx.x == 0) {
    long long prof_tot = 0;
    GH_SC_ADD(prof_tot, prof_cta0);
    GH_SC_FLUSH(14, 1);
    GH_SC_FLUSH(15, prof_tot);
  }
#endif
}

}  // namespace gh
