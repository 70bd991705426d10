// Batched symmetric Gram forward on tcgen05:  G_b = F_b F_b^T * scale,  F_b : C x HW (row-major, K = HW contiguous).
//
// Replaces TruncatedResNet50.gram_matrix (reference Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:26-30,
// bmm + div(h*w)) and, in POOL mode, also the adaptive_avg_pool2d + stack/flatten that follow it (:51-55): the
// C x C Gram only ever exists in TMEM; what reaches HBM is the g x g block-mean written straight into the
// (B, L, g*g) descriptor buffer the attention consumes.
//
// Work decomposition
//   unit      = (image b, 256x256 super-tile (I <= J) of the Gram, K-range kp of ksplit)
//   CTA       = persistent, walks units blockIdx.x, +gridDim.x, ...
//   producers = 16 warps: ld.global fp32/bf16 (coalesced along HW) -> cvt.rn.bf16x2 -> st.shared into the
//               UMMA K-major SWIZZLE_128B layout (no separate cast pass over HBM, any HW, any pitch); the loads of
//               stage s+1 are issued before stage s is converted and stored (register double buffering)
//   epilogue  = 4 warps: tcgen05.ld -> in-register k x k block sums -> descriptor (mirrored for off-diagonal
//               128-col blocks; plain stores when each element has one writer, red.global.add otherwise) or dense G
//   MMA       = 1 warp: TMEM owner + the single MMA-issuing thread
//   smem ring = 6 stages of [256 rows][64 k] bf16 (32 KB). A diagonal super-tile consumes one stage per k-block
//               (A and B tiles are the same rows), an off-diagonal one consumes two (I rows, then J rows).
//   TMEM      = 512 columns: acc0 = rows 0-127 of I x 256 cols, acc1 = rows 128-255 of I x (128 | 256) cols.
//               Only upper-triangle 128x128 blocks are ever issued: 3 of 4 on a diagonal super-tile.
#pragma once
#include "common.cuh"

namespace gh {

constexpr int kGfStages = 6;
constexpr uint32_t kGfStageRows = 256;
constexpr uint32_t kGfStageBytes = kGfStageRows * kRowBytes;   // 32 KB
constexpr uint32_t kGfSmemBytes = kGfStages * kGfStageBytes + 1024 /*align*/ + 256 /*barriers*/;
constexpr uint32_t kGfTmemCols = 512;
constexpr int kGfProducerWarps = 16;
constexpr int kGfProducerThreads = kGfProducerWarps * 32;
constexpr int kGfThreads = (kGfProducerWarps + 4) * 32;   // + 4 epilogue warps

enum GramMode : int { GRAM_POOL = 0, GRAM_DENSE = 1 };

struct GramFwdParams {
  const void* F;
  long long img_stride;   // elements between images
  long long row_stride;   // elements between channel rows
  int B, C, HW;
  int nT;                 // ceil(C / 256)
  int nST;                // nT (nT + 1) / 2 super-tiles per image
  int ksplit;             // K partitions per super-tile
  int nkb;                // ceil(HW / 64)
  int total_units;
  int g;                  // POOL: pooled size
  float* out;             // POOL: (B, L, g*g) slice base for this stage; DENSE: (B, C, C)
  long long out_img_stride;
  float scale;
  int use_atomics;        // outputs meet in red.global.add (ksplit > 1, or pool factor > 32): buffer pre-zeroed
};

struct GramUnit {
  int b, I, J, kb0, kb1;
};

__device__ __forceinline__ GramUnit gram_decode_unit(const GramFwdParams& p, int u) {
  GramUnit w;
  const int kp = u % p.ksplit;
  int t = u / p.ksplit;
  int st = t % p.nST;
  w.b = t / p.nST;
  int I = 0, rowlen = p.nT;
  while (st >= rowlen) { st -= rowlen; ++I; --rowlen; }
  w.I = I;
  w.J = I + st;
  w.kb0 = (int)(((long long)p.nkb * kp) / p.ksplit);
  w.kb1 = (int)(((long long)p.nkb * (kp + 1)) / p.ksplit);
  return w;
}

// ---- producers ----------------------------------------------------------------------------------------------------
// One stage = rows [blk*256, blk*256+256) x k in [kb*64, kb*64+64) of image b.
// 16 threads cover one row (64 elements, 4 each); the 512 producer threads cover 32 rows per pass, 8 passes.
// Loading (global -> registers) and storing (registers -> swizzled smem) are separate steps so that the loads of the
// NEXT stage are in flight while the current one is converted and stored (register double buffering): the memory
// pipe never drains between stages, units or images.
struct GfItem {
  int u, kb, h, nblk;
  GramUnit w;
};
__device__ __forceinline__ bool gf_item_first(GfItem& it, const GramFwdParams& p) {
  it.u = blockIdx.x;
  if (it.u >= p.total_units) return false;
  it.w = gram_decode_unit(p, it.u);
  it.nblk = (it.w.I == it.w.J) ? 1 : 2;
  it.kb = it.w.kb0;
  it.h = 0;
  return true;
}
__device__ __forceinline__ bool gf_item_next(GfItem& it, const GramFwdParams& p) {
  if (++it.h < it.nblk) return true;
  it.h = 0;
  if (++it.kb < it.w.kb1) return true;
  it.u += gridDim.x;
  if (it.u >= p.total_units) return false;
  it.w = gram_decode_unit(p, it.u);
  it.nblk = (it.w.I == it.w.J) ? 1 : 2;
  it.kb = it.w.kb0;
  return true;
}

// SRC: 0 = fp32 vector (16 B aligned rows, HW % 4 == 0), 1 = fp32 scalar (anything), 2 = bf16 vector (8 B), 3 = bf16 scalar.
// Register image of one thread's share of a stage: NL x 4 elements, already packed to bf16x2 pairs for SRC >= 1.
template <int SRC, int NL>
struct GfRegs {
  float4 f[SRC == 0 ? NL : 1];
  uint2 h[SRC == 0 ? 1 : NL];
};

constexpr int kGfLoads = 4096 / kGfProducerThreads;   // 16 B loads per producer thread and stage

template <int SRC>
__device__ __forceinline__ void gf_load(const GramFwdParams& p, const GfItem& it, GfRegs<SRC, kGfLoads>& r, int tid) {
  constexpr int NL = kGfLoads, RPP = kGfProducerThreads / 16;
  const int sub = tid >> 4, q = tid & 15;
  const int k = it.kb * 64 + q * 4;
  const int blk = it.h == 0 ? it.w.I : it.w.J;
  const int c0 = blk * 256 + sub;
  if (SRC == 0) {
    const bool kvalid = k < p.HW;   // HW % 4 == 0 on this path, so k+3 < HW too
    const float* base = reinterpret_cast<const float*>(p.F) + (long long)it.w.b * p.img_stride + k;
#pragma unroll
    for (int i = 0; i < NL; ++i) {
      const int c = c0 + i * RPP;
      if (kvalid && c < p.C) r.f[i] = ldg_stream_f4(base + (long long)c * p.row_stride);
      else r.f[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  } else if (SRC == 1) {
    const float* base = reinterpret_cast<const float*>(p.F) + (long long)it.w.b * p.img_stride + k;
#pragma unroll
    for (int i = 0; i < NL; ++i) {
      const int c = c0 + i * RPP;
      float x[4] = {0.f, 0.f, 0.f, 0.f};
      if (c < p.C) {
        const float* rp = base + (long long)c * p.row_stride;
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (k + e < p.HW) x[e] = __ldg(rp + e);
      }
      r.h[i] = make_uint2(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]));
    }
  } else if (SRC == 2) {
    const bool kvalid = k < p.HW;
    const __nv_bfloat16* base = reinterpret_cast<const __nv_bfloat16*>(p.F) + (long long)it.w.b * p.img_stride + k;
#pragma unroll
    for (int i = 0; i < NL; ++i) {
      const int c = c0 + i * RPP;
      if (kvalid && c < p.C) r.h[i] = ldg_stream_u2(base + (long long)c * p.row_stride);
      else r.h[i] = make_uint2(0u, 0u);
    }
  } else {
    const unsigned short* base = reinterpret_cast<const unsigned short*>(p.F) + (long long)it.w.b * p.img_stride + k;
#pragma unroll
    for (int i = 0; i < NL; ++i) {
      const int c = c0 + i * RPP;
      unsigned int x[4] = {0u, 0u, 0u, 0u};
      if (c < p.C) {
        const unsigned short* rp = base + (long long)c * p.row_stride;
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (k + e < p.HW) x[e] = __ldg(rp + e);
      }
      r.h[i] = make_uint2(x[0] | (x[1] << 16), x[2] | (x[3] << 16));
    }
  }
}

template <int SRC>
__device__ __forceinline__ void gf_store(const GramFwdParams& p, const GfItem& it, const GfRegs<SRC, kGfLoads>& r,
                                         uint32_t stage_smem, int tid) {
  constexpr int NL = kGfLoads, RPP = kGfProducerThreads / 16;
  const int sub = tid >> 4, q = tid & 15;
  // a 16-wide k-step that lies entirely beyond HW is never issued to the tensor core, so it need not be written
  if (it.kb * 64 + (q >> 2) * 16 >= p.HW) return;
#pragma unroll
  for (int i = 0; i < NL; ++i) {
    const uint32_t row = (uint32_t)(sub + i * RPP);
    const uint32_t addr = stage_smem + sw128_off(row, (uint32_t)(q * 4));
    if (SRC == 0) sts_u2(addr, pack_bf16x2(r.f[i].x, r.f[i].y), pack_bf16x2(r.f[i].z, r.f[i].w));
    else sts_u2(addr, r.h[i].x, r.h[i].y);
  }
}

template <int SRC>
__device__ __forceinline__ void gf_publish(const GramFwdParams& p, const GfItem& it, const GfRegs<SRC, kGfLoads>& r,
                                           uint32_t smem_base, uint32_t bar_full, uint32_t bar_empty, uint32_t& stage,
                                           uint32_t& phase, int tid, int lane) {
  mbar_wait(bar_empty + 8 * stage, phase ^ 1u, 100u + stage);
  gf_store<SRC>(p, it, r, smem_base + stage * kGfStageBytes, tid);
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) mbar_arrive(bar_full + 8 * stage);
  if (++stage == kGfStages) { stage = 0; phase ^= 1u; }
}

// ---- epilogue -----------------------------------------------------------------------------------------------------
// One 32-lane x 32-column chunk of an accumulator. Thread = Gram row c_row, v[j] = G[c_row][c_col0 + j] (unscaled).
template <int KP>
__device__ __forceinline__ void gram_epi_pool_chunk(const float (&v)[32], int c_row, int c_col0, int C, int g,
                                                    float scale, float* __restrict__ outp, bool mirror, bool atomics,
                                                    int lane) {
  constexpr int CW = KP < 32 ? KP : 32;   // columns summed in-thread per value
  constexpr int NC = 32 / CW;             // values this chunk yields per row
  constexpr int LK = KP < 32 ? KP : 32;   // rows (lanes) summed by shuffles
  float s[NC];
#pragma unroll
  for (int j = 0; j < NC; ++j) {
    float a = 0.f;
#pragma unroll
    for (int i = 0; i < CW; ++i) a += v[j * CW + i];
    s[j] = a;
  }
#pragma unroll
  for (int off = 1; off < LK; off <<= 1) {
#pragma unroll
    for (int j = 0; j < NC; ++j) s[j] += __shfl_xor_sync(0xffffffffu, s[j], off);
  }
  // Rows/cols >= C were zero-filled by the producers, so the sums need no masks; only the writes do.
  const int lj = lane & (LK - 1);
  const int pi = c_row / KP;
#pragma unroll
  for (int j = 0; j < NC; ++j) {
    if ((j % LK) == lj && c_row < C) {
      const int col = c_col0 + j * CW;
      if (col < C) {
        const int pj = col / KP;
        const float val = s[j] * scale;
        if (atomics) {
          red_add_f32(outp + pi * g + pj, val);
          if (mirror) red_add_f32(outp + pj * g + pi, val);
        } else {
          outp[pi * g + pj] = val;
          if (mirror) outp[pj * g + pi] = val;
        }
      }
    }
  }
}

// Sum of CW consecutive registers starting at v[o], as a balanced tree (short dependency chain).
template <int CW>
__device__ __forceinline__ float tree_sum(const uint32_t (&v)[32], int o) {
  if constexpr (CW == 1) {
    return __uint_as_float(v[o]);
  } else {
    return tree_sum<CW / 2>(v, o) + tree_sum<CW / 2>(v, o + CW / 2);
  }
}

// Pooled epilogue for a group of 128 accumulator columns (4 tcgen05.ld of 32 columns, two in flight at a time), KP >= 8.
// Thread = Gram row c_row. Column pooling is in-thread; row pooling over LK = min(KP, 32) lanes is a halving butterfly:
// at each step a lane hands half of its partial sums to its partner and keeps the other half, so NV values cost
// NV - 1 + (log2 LK - log2 NV) shuffles instead of NV * log2 LK, and every lane ends up owning distinct outputs.
template <int KP>
__device__ __forceinline__ void gram_epi_pool_group128(uint32_t taddr, int c_row, int c_col0, int C, int g, float scale,
                                                       float* __restrict__ outp, bool mirror, bool atomics, int lane) {
  constexpr int CW = KP < 32 ? KP : 32;         // columns summed in-thread per tcgen05.ld chunk value
  constexpr int NCc = 32 / CW;                  // values per 32-column chunk
  constexpr int CPV = KP > 32 ? KP / 32 : 1;    // chunks that fold into one value (KP = 64: 2, 128: 4)
  constexpr int NV = 4 * NCc / CPV;             // values per thread for the 128-column group
  constexpr int LK = KP < 32 ? KP : 32;
  float s[NV];
#pragma unroll
  for (int j = 0; j < NV; ++j) s[j] = 0.f;
  if constexpr (NV <= 8) {
    // two TMEM loads in flight (64 registers): the short-K shapes (C >= 512) are bounded by this drain
#pragma unroll
    for (int pair = 0; pair < 2; ++pair) {
      uint32_t v0[32], v1[32];
      tmem_ld32_nowait(taddr + (uint32_t)(pair * 64), v0);
      tmem_ld32_nowait(taddr + (uint32_t)(pair * 64 + 32), v1);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < NCc; ++j) {
        s[((2 * pair) * NCc + j) / CPV] += tree_sum<CW>(v0, j * CW);
        s[((2 * pair + 1) * NCc + j) / CPV] += tree_sum<CW>(v1, j * CW);
      }
    }
  } else {
    // KP = 8 (C = 256, long K loop, epilogue off the critical path): one load at a time keeps the kernel spill-free
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {
      uint32_t v0[32];
      tmem_ld32_nowait(taddr + (uint32_t)(ch * 32), v0);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < NCc; ++j) s[(ch * NCc + j) / CPV] += tree_sum<CW>(v0, j * CW);
    }
  }
  int nv = NV, base = 0;
#pragma unroll
  for (int off = LK / 2; off >= 1; off >>= 1) {
    if (nv > 1) {
      const int half = nv >> 1;
      const bool upper = (lane & off) != 0;
#pragma unroll
      for (int j = 0; j < NV / 2; ++j) {
        if (j < half) {
          const float send = upper ? s[j] : s[j + half];
          const float keep = upper ? s[j + half] : s[j];
          s[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
      }
      if (upper) base += half;
      nv = half;
    } else {
      s[0] += __shfl_xor_sync(0xffffffffu, s[0], off);
    }
  }
  // lanes that went through plain (non-halving) steps hold copies: the one with those low lane bits clear writes
  constexpr int kHalvings = (NV >= LK) ? /*all steps halve*/ 31 : 0;
  (void)kHalvings;
  int plain_mask = 0;
  {
    int n2 = NV;
#pragma unroll
    for (int off = LK / 2; off >= 1; off >>= 1) {
      if (n2 > 1) n2 >>= 1;
      else plain_mask |= off;
    }
  }
  if ((lane & plain_mask) != 0 || c_row >= C) return;
  const int pi = c_row / KP;
#pragma unroll
  for (int t = 0; t < NV; ++t) {
    if (t < nv) {
      const int jv = base + t;
      if (c_col0 + jv * KP < C) {
        const int pj = c_col0 / KP + jv;
        const float val = s[t] * scale;
        if (atomics) {
          red_add_f32(outp + pi * g + pj, val);
          if (mirror) red_add_f32(outp + pj * g + pi, val);
        } else {
          outp[pi * g + pj] = val;
          if (mirror) outp[pj * g + pi] = val;
        }
      }
    }
  }
}

__device__ __forceinline__ void gram_epi_dense_chunk(const float (&v)[32], int c_row, int c_col0, int C, float scale,
                                                     float* __restrict__ G, bool mirror, bool atomics) {
  if (c_row >= C) return;
  float* rowp = G + (long long)c_row * C + c_col0;
  if (!atomics && c_col0 + 32 <= C && (C & 3) == 0) {
#pragma unroll
    for (int j = 0; j < 32; j += 4)
      *reinterpret_cast<float4*>(rowp + j) = make_float4(v[j] * scale, v[j + 1] * scale, v[j + 2] * scale, v[j + 3] * scale);
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (c_col0 + j < C) {
        if (atomics) red_add_f32(rowp + j, v[j] * scale);
        else rowp[j] = v[j] * scale;
      }
  }
  if (mirror) {
    // lanes = consecutive c_row -> each j is one coalesced 128 B store across the warp
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (c_col0 + j < C) {
        float* mp = G + (long long)(c_col0 + j) * C + c_row;
        if (atomics) red_add_f32(mp, v[j] * scale);
        else *mp = v[j] * scale;
      }
  }
}

// MMAs of one unit, issued by lane 0 of the calling warp (all lanes wait on the barriers).
__device__ __forceinline__ void gf_issue_unit(const GramFwdParams& p, const GramUnit& w, uint32_t smem_base,
                                              uint32_t bar_full, uint32_t bar_empty, uint32_t bar_tfull,
                                              uint32_t bar_tempty, uint32_t tmem_base, uint32_t& stage, uint32_t& phase,
                                              uint32_t acc_phase, int lane) {
  const uint32_t idesc256 = make_idesc_bf16(128, 256), idesc128 = make_idesc_bf16(128, 128);
  const bool diag = (w.I == w.J);
  mbar_wait(bar_tempty, acc_phase ^ 1u, 200u);   // every epilogue warp has drained the previous unit's accumulators
  tc_fence_after_sync();
  for (int kb = w.kb0; kb < w.kb1; ++kb) {
    const uint32_t sA = stage;
    mbar_wait(bar_full + 8 * sA, phase, 300u + sA);
    uint32_t sB = sA, phaseB = phase;
    if (!diag) {
      sB = sA + 1;
      if (sB == kGfStages) { sB = 0; phaseB ^= 1u; }
      mbar_wait(bar_full + 8 * sB, phaseB, 310u + sB);
    }
    tc_fence_after_sync();
    if (elect_one()) {   // elect.sync, not a lane test: see gram_fwd_pair.cuh
      const uint32_t aI = smem_base + sA * kGfStageBytes;   // rows of block I
      const uint32_t aJ = smem_base + sB * kGfStageBytes;   // rows of block J (== I on the diagonal)
      const uint32_t acc = (kb > w.kb0) ? 1u : 0u;
#pragma unroll
      for (uint32_t ks = 0; ks < kTileK / kUmmaK; ++ks) {
        if ((int)(kb * 64 + ks * 16) >= p.HW) break;        // K tail: whole k-steps past HW are skipped
        const uint32_t koff = ks * 32u;
        // acc0: I rows 0-127 x J rows 0-255
        umma_bf16(tmem_base + 0u, make_smem_desc_sw128(aI + koff), make_smem_desc_sw128(aJ + koff), idesc256, acc | ks);
        if (diag) {
          // acc1: I rows 128-255 x I rows 128-255 (the lower-left 128x128 block is never computed)
          umma_bf16(tmem_base + 256u, make_smem_desc_sw128(aI + 128u * kRowBytes + koff),
                    make_smem_desc_sw128(aI + 128u * kRowBytes + koff), idesc128, acc | ks);
        } else {
          // acc1: I rows 128-255 x J rows 0-255
          umma_bf16(tmem_base + 256u, make_smem_desc_sw128(aI + 128u * kRowBytes + koff),
                    make_smem_desc_sw128(aJ + koff), idesc256, acc | ks);
        }
      }
      umma_commit(bar_empty + 8 * sA);
      if (!diag) umma_commit(bar_empty + 8 * sB);
      if (kb + 1 == w.kb1) umma_commit(bar_tfull);
    }
    __syncwarp();
    stage = sB + 1; phase = phaseB;
    if (stage == kGfStages) { stage = 0; phase ^= 1u; }
  }
}

// Drains the accumulators of one unit. q = TMEM lane quarter of this warp.
template <int KP>
__device__ __forceinline__ void gf_epilogue_unit(const GramFwdParams& p, const GramUnit& w, uint32_t tmem_base, int q,
                                                 bool atomics, int lane) {
  const bool diag = (w.I == w.J);
  float* outp = p.out + (long long)w.b * p.out_img_stride;
  const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
  for (int a = 0; a < 2; ++a) {
    const int c_row = w.I * 256 + a * 128 + q * 32 + lane;
    const int ncols = (a == 1 && diag) ? 128 : 256;
    const int colbase = w.J * 256 + ((a == 1 && diag) ? 128 : 0);
    if (w.I * 256 + a * 128 >= p.C) break;   // whole accumulator is padding (C <= 128)
#pragma unroll 1
    for (int g0 = 0; g0 < ncols && colbase + g0 < p.C; g0 += 128) {   // columns >= C are padding
      const int c_grp = colbase + g0;
      // a 128x128 block strictly above the diagonal is mirrored; diagonal blocks are complete on their own
      const bool mirror = (c_grp >> 7) > (c_row >> 7);
      if constexpr (KP >= 8) {
        gram_epi_pool_group128<KP>(lane_addr + (uint32_t)(a * 256 + g0), c_row, c_grp, p.C, p.g, p.scale, outp, mirror,
                                   atomics, lane);
      } else {
#pragma unroll 1
        for (int n0 = 0; n0 < 128; n0 += 32) {
          const int c_col0 = c_grp + n0;
          if (c_col0 >= p.C) break;
          float v[32];
          tmem_ld32(lane_addr + (uint32_t)(a * 256 + g0 + n0), v);
          if (KP > 0)
            gram_epi_pool_chunk<(KP > 0 ? KP : 1)>(v, c_row, c_col0, p.C, p.g, p.scale, outp, mirror, atomics, lane);
          else gram_epi_dense_chunk(v, c_row, c_col0, p.C, p.scale, outp, mirror, atomics);
        }
      }
    }
  }
}

// SRC: see gf_load.  KP = pool factor (POOL) or 0 (DENSE).
// Warp roles: [0, 16) producers, [16, 20) epilogue (warp % 4 is the TMEM lane quarter). The first epilogue warp also
// owns TMEM and issues the MMAs of a unit before joining its epilogue: with one accumulator set in TMEM (384-512 of the
// 512 columns) the two phases of a unit cannot overlap anyway, and 20 warps (a multiple of the 4 SM sub-partitions)
// leave every thread 96 registers for the double-buffered loads. Measured on every ResNet stage shape
// (profiles/r01e_kernel_timings.log), 16 producer warps are as fast as 8 or faster, and 8 epilogue warps (24 warps -> 80
// registers per thread) spill in the producer loop and lose.
template <int SRC, int KP>
__global__ void __launch_bounds__(kGfThreads, 1) gram_fwd_kernel(const GramFwdParams p) {
  constexpr int kEpiWarp0 = kGfProducerWarps, kMmaWarp = kGfProducerWarps;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bars = smem_base + kGfStages * kGfStageBytes;
  // barrier map (8 B each): full[6], empty[6], tmem_full, tmem_empty, then the TMEM base word
  const uint32_t bar_full = bars, bar_empty = bars + 8 * kGfStages;
  const uint32_t bar_tfull = bars + 16 * kGfStages, bar_tempty = bar_tfull + 8;
  const uint32_t tmem_slot = bar_tempty + 8;
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kGfStages; ++s) {
      mbar_init(bar_full + 8 * s, kGfProducerWarps);
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_tfull, 1);
    mbar_init(bar_tempty, 4);
    mbar_fence_init();
  }
  if (warp == kMmaWarp) tmem_alloc(tmem_slot, kGfTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp < kGfProducerWarps) {
    // =========================== producers ===========================
    uint32_t stage = 0, phase = 0;
    const int tid = threadIdx.x;
    GfRegs<SRC, kGfLoads> ra, rb;
    GfItem cur;
    bool have = gf_item_first(cur, p);
    if (have) gf_load<SRC>(p, cur, ra, tid);
    while (have) {
      GfItem n1 = cur;
      const bool h1 = gf_item_next(n1, p);
      if (h1) gf_load<SRC>(p, n1, rb, tid);    // next stage's loads fly while this one is stored
      gf_publish<SRC>(p, cur, ra, smem_base, bar_full, bar_empty, stage, phase, tid, lane);
      if (!h1) break;
      cur = n1;
      have = gf_item_next(cur, p);
      if (have) gf_load<SRC>(p, cur, ra, tid);
      gf_publish<SRC>(p, n1, rb, smem_base, bar_full, bar_empty, stage, phase, tid, lane);
    }
  } else {
    // =========================== MMA issue (first epilogue warp) + epilogue (all of them) ===========================
    const int ew = warp - kEpiWarp0;
    const int q = ew & 3;             // TMEM lane quarter this warp may read (= warp % 4)
    uint32_t acc_phase = 0, stage = 0, phase = 0;
    const bool atomics = p.use_atomics != 0;
    for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
      const GramUnit w = gram_decode_unit(p, u);
      if (ew == 0)
        gf_issue_unit(p, w, smem_base, bar_full, bar_empty, bar_tfull, bar_tempty, tmem_base, stage, phase, acc_phase, lane);
      mbar_wait(bar_tfull, acc_phase, 400u);
      tc_fence_after_sync();
      gf_epilogue_unit<KP>(p, w, tmem_base, q, atomics, lane);
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tempty);
      acc_phase ^= 1u;
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, kGfTmemCols);
  }
}

}  // namespace gh
