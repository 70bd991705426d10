// Single-CTA Gram backward:  dF_b[c][x] = scale * sum_d M_b[c][d] F_b[d][x],   M = dG + dG^T.
//
// This is what autograd derives for the reference's bmm(features, features^T).div(h*w)
// (Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:26-30) followed, on the classification path, by
// adaptive_avg_pool2d (:51-52). In POOL mode dG is never materialised: it is the block-constant upsampling of the
// g x g descriptor gradient, dG[c][d] = dP[c/k][d/k] / k^2, and the symmetrised bf16 operand tile is generated in
// shared memory from the image's dP. In DENSE mode (gram_matrix() used directly, e.g. style transfer) dG is read from
// HBM. F is consumed exactly as it lies in HBM:
//   A tile = M   [128 c][64 d]  K-major SWIZZLE_128B, generated in smem from the image's g x g descriptor gradient
//                               (POOL) or read from the dense dG (DENSE); two of them per stage (256 output channels)
//   B tile = F   [64 d][256 x]  MN-major SWIZZLE_128B: rows of F are contiguous along x, which IS the MN-major
//                               canonical layout ([x/64][d/8][d%8][64 x] with 16 B chunks XOR-swizzled by d%8), so the
//                               producers use the same coalesced ld.global.v4 -> cvt -> st.shared path as the forward
//                               kernel: no transposing gathers, no scalar loads
//   D      = dF  [128 c][256 x] in TMEM: lane = output channel, 32 consecutive x per tcgen05.ld -> 8 x 16 B stores
//   unit   = (image, 256-wide x tile, pair of 128-channel output blocks); every CTA owns a contiguous range of units
//            so the per-image gradient table is rebuilt only at image boundaries
//   TMEM   = one accumulator of 2 x 256 columns per unit
//   warps  = 8 producers, 4 epilogue warps, 1 MMA warp (TMEM owner + the MMA-issuing thread): 13 warps
// Producers double-buffer their loads in registers in batches of 8 x 16 B per thread, two batches per stage.
// At batch 256 on every ResNet stage shape, 256-wide x tiles beat 128-wide ones with two accumulators, and a separate MMA
// warp beats 16 producer warps with the MMAs issued by an epilogue warp (profiles/r01e_kernel_timings.log).
#pragma once
#include "common.cuh"
#include "gram_fwd.cuh"   // GramMode

namespace gh {

constexpr int kB2NHW = 256;                                 // x positions per unit
constexpr int kB2ProducerWarps = 8;
constexpr int kB2ProducerThreads = kB2ProducerWarps * 32;
constexpr int kB2MmaWarp = kB2ProducerWarps + 4;            // after the 4 epilogue warps
constexpr int kB2Threads = (kB2MmaWarp + 1) * 32;           // 13 warps
constexpr int kB2Batches = 2 * kB2NHW / kB2ProducerThreads; // register batches (8 x 16 B per thread) per stage
constexpr uint32_t kB2ATileBytes = 128 * kRowBytes;        // 16 KB
constexpr uint32_t kB2StageBytes = 2 * kB2ATileBytes + kB2NHW * kRowBytes;   // 64 KB
constexpr uint32_t kB2RingBytes = 192 * 1024;
constexpr int kB2Stages = (int)(kB2RingBytes / kB2StageBytes);              // 3
constexpr int kB2MaxStages = 4;
constexpr int kB2MaxG = 64;
constexpr uint32_t kB2SmemBytes = kB2RingBytes + kB2MaxG * kB2MaxG * 4 + 1024 + 256;

struct GramBwd2Params {
  const void* F;
  long long img_stride, row_stride;
  int B, C, HW;
  int mode;                 // GRAM_POOL / GRAM_DENSE
  const float* dP;          // POOL: (B, L, g*g) slice base of this stage
  long long dp_img_stride;
  int g, kshift;
  const float* dG;          // DENSE: (B, C, C)
  float* dF;
  long long df_img_stride, df_row_stride;
  float scale;
  int nHT, nCP, nkb, nA;    // x tiles, output-channel pairs, 64-deep k-blocks over input channels, A tiles in use (1|2)
  int total_units;
  int units_per_cta;
  int df_vec_ok;            // dF rows 16 B aligned and HW % 4 == 0: float4 stores
};

struct GramBwd2Unit {
  int b, ht, cp;
};
__device__ __forceinline__ GramBwd2Unit gb2_decode(const GramBwd2Params& p, int u) {
  GramBwd2Unit w;
  w.cp = u % p.nCP;
  const int t = u / p.nCP;
  w.ht = t % p.nHT;
  w.b = t / p.nHT;
  return w;
}

// smem descriptor for the MN-major SWIZZLE_128B B tile: LBO = distance between 64-wide x blocks (64 k-rows x 128 B),
// SBO = distance between groups of 8 k-rows (1024 B).
__host__ __device__ constexpr uint64_t make_smem_desc_sw128_mn(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(8192u >> 4) << 16) | ((uint64_t)(1024u >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
__host__ __device__ constexpr uint32_t make_idesc_bf16_bmn(uint32_t m, uint32_t n) {
  return make_idesc_bf16(m, n) | (1u << 16);   // B operand MN-major
}

struct Gb2Item {
  int u, kb, half;
  GramBwd2Unit w;
};

__device__ __forceinline__ bool gb2_first(Gb2Item& it, const GramBwd2Params& p, int u0, int u1) {
  it.u = u0;
  if (u0 >= u1) return false;
  it.w = gb2_decode(p, u0);
  it.kb = 0;
  it.half = 0;
  return true;
}
__device__ __forceinline__ bool gb2_next(Gb2Item& it, const GramBwd2Params& p, int u1) {
  if (++it.half < kB2Batches) return true;
  it.half = 0;
  if (++it.kb < p.nkb) return true;
  it.kb = 0;
  if (++it.u >= u1) return false;
  it.w = gb2_decode(p, it.u);
  return true;
}

// One batch = 8 segments per thread; a segment = 4 consecutive x of one F row. Segment index s in [0, 1024) per stage:
// d_local = s / MB, x block = s % MB (MB = 256 / 64), so consecutive segments continue along the same F row.
template <int SRC>
__device__ __forceinline__ void gb2_load(const GramBwd2Params& p, const Gb2Item& it, uint4 (&r)[8], int tid) {
  constexpr int MB = kB2NHW / 64, SPP = kB2ProducerThreads / 16;   // 64-wide x blocks per row; segments per pass
  const int seg = tid >> 4, q = tid & 15;
  const int hw0 = it.w.ht * kB2NHW;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int s = seg + SPP * (i + 8 * it.half);
    const int d = it.kb * 64 + s / MB;
    const int x = hw0 + (s % MB) * 64 + q * 4;
    r[i] = make_uint4(0u, 0u, 0u, 0u);
    if (d < p.C) {
      if (SRC == 0) {
        if (x < p.HW) {
          const float4 v = ldg_stream_f4(reinterpret_cast<const float*>(p.F) + (long long)it.w.b * p.img_stride +
                                         (long long)d * p.row_stride + x);
          r[i] = make_uint4(__float_as_uint(v.x), __float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(v.w));
        }
      } else if (SRC == 1) {
        const float* rp = reinterpret_cast<const float*>(p.F) + (long long)it.w.b * p.img_stride + (long long)d * p.row_stride + x;
        float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (x + e < p.HW) v[e] = __ldg(rp + e);
        r[i] = make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
      } else if (SRC == 2) {
        if (x < p.HW) {
          const uint2 v = ldg_stream_u2(reinterpret_cast<const __nv_bfloat16*>(p.F) + (long long)it.w.b * p.img_stride +
                                        (long long)d * p.row_stride + x);
          r[i].x = v.x; r[i].y = v.y;
        }
      } else {
        const unsigned short* rp = reinterpret_cast<const unsigned short*>(p.F) + (long long)it.w.b * p.img_stride +
                                   (long long)d * p.row_stride + x;
        unsigned int v[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (x + e < p.HW) v[e] = __ldg(rp + e);
        r[i].x = v[0] | (v[1] << 16); r[i].y = v[2] | (v[3] << 16);
      }
    }
  }
}

template <int SRC>
__device__ __forceinline__ void gb2_store_b(const Gb2Item& it, const uint4 (&r)[8], uint32_t b_smem, int tid) {
  constexpr int MB = kB2NHW / 64, SPP = kB2ProducerThreads / 16;
  const int seg = tid >> 4, q = tid & 15;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int s = seg + SPP * (i + 8 * it.half);
    const uint32_t dl = (uint32_t)(s / MB), xb = (uint32_t)(s % MB);
    // [x block][d / 8][d % 8][64 x]: 16 B chunk (q / 2) XOR-swizzled by d % 8, 8 B half (q % 2)
    const uint32_t addr = b_smem + xb * 8192u + (dl >> 3) * 1024u + (dl & 7u) * 128u +
                          ((((uint32_t)q >> 1) ^ (dl & 7u)) << 4) + (((uint32_t)q & 1u) << 3);
    if (SRC < 2)
      sts_u2(addr, pack_bf16x2(__uint_as_float(r[i].x), __uint_as_float(r[i].y)),
             pack_bf16x2(__uint_as_float(r[i].z), __uint_as_float(r[i].w)));
    else sts_u2(addr, r[i].x, r[i].y);
  }
}

// A tiles of one stage: rows n in [0, 256) = output channels cp*256 + n, columns = input channels kb*64 .. +63.
__device__ __forceinline__ void gb2_gen_a(const GramBwd2Params& p, const Gb2Item& it, const float* sym, uint32_t a_smem,
                                          int tid) {
  constexpr int CPT = 8 * 256 / kB2ProducerThreads;   // 16 B chunks per thread
  const int r256 = tid & 255, j0 = (tid >> 8) * CPT;
  const int c = it.w.cp * 256 + r256;
  const uint32_t tile = a_smem + (uint32_t)(r256 >> 7) * kB2ATileBytes;
  const uint32_t row = (uint32_t)(r256 & 127);
  if ((r256 >> 7) >= p.nA) return;
  if (p.mode == GRAM_POOL) {
    const float* srow = sym + (c >> p.kshift) * p.g;
#pragma unroll
    for (int j = j0; j < j0 + CPT; ++j) {
      const int d0 = it.kb * 64 + j * 8;
      uint32_t pk[4];
      if (c >= p.C || d0 >= p.C) {
        pk[0] = pk[1] = pk[2] = pk[3] = 0u;
      } else if (p.kshift >= 3) {
        const float v = srow[d0 >> p.kshift];
        pk[0] = pk[1] = pk[2] = pk[3] = pack_bf16x2(v, v);
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int da = d0 + 2 * e, db = da + 1;
          pk[e] = pack_bf16x2(da < p.C ? srow[da >> p.kshift] : 0.f, db < p.C ? srow[db >> p.kshift] : 0.f);
        }
      }
      sts_u4(tile + sw128_off(row, (uint32_t)(j * 8)), pk[0], pk[1], pk[2], pk[3]);
    }
  } else {
    const float* gb = p.dG + (long long)it.w.b * p.C * p.C;
#pragma unroll
    for (int j = j0; j < j0 + CPT; ++j) {
      float x[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int d = it.kb * 64 + j * 8 + e;
        x[e] = (c < p.C && d < p.C) ? (__ldg(gb + (long long)c * p.C + d) + __ldg(gb + (long long)d * p.C + c)) : 0.f;
      }
      sts_u4(tile + sw128_off(row, (uint32_t)(j * 8)), pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]),
             pack_bf16x2(x[4], x[5]), pack_bf16x2(x[6], x[7]));
    }
  }
}

template <int SRC>
__global__ void __launch_bounds__(kB2Threads, 1) gram_bwd2_kernel(const GramBwd2Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sym_smem = smem_base + kB2RingBytes;
  float* sym = reinterpret_cast<float*>(smem_raw + (sym_smem - smem_u32(smem_raw)));
  const uint32_t bars = sym_smem + kB2MaxG * kB2MaxG * 4;
  const uint32_t bar_full = bars, bar_empty = bars + 8 * kB2MaxStages;
  const uint32_t bar_tfull = bars + 16 * kB2MaxStages, bar_tempty = bar_tfull + 8;
  const uint32_t tmem_slot = bar_tempty + 8;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kB2MaxStages; ++s) {
      mbar_init(bar_full + 8 * s, kB2ProducerWarps);
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_tfull, 1);
    mbar_init(bar_tempty, 4);
    mbar_fence_init();
  }
  if (warp == kB2MmaWarp) tmem_alloc(tmem_slot, 512);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot_ptr;

  // contiguous unit range of this CTA
  const int u0 = blockIdx.x * p.units_per_cta;
  const int u1 = min(u0 + p.units_per_cta, p.total_units);

  if (warp < kB2ProducerWarps) {
    // =========================== producers ===========================
    const int tid = threadIdx.x;
    uint32_t stage = 0, phase = 0;
    int cur_b = -1;
    uint4 ra[8], rb[8];
    Gb2Item cur;
    bool have = gb2_first(cur, p, u0, u1);
    if (have) gb2_load<SRC>(p, cur, ra, tid);

    auto publish = [&](const Gb2Item& it, const uint4 (&r)[8]) {
      if (it.half == 0) {
        if (p.mode == GRAM_POOL && it.w.b != cur_b) {
          // per-image table sym[i][j] = dP[i][j] + dP[j][i]; every producer is done reading the previous image's
          named_bar_sync(1, kB2ProducerThreads);
          const float* dp = p.dP + (long long)it.w.b * p.dp_img_stride;
          const int gg = p.g * p.g;
          for (int i = tid; i < gg; i += kB2ProducerThreads) {
            const int rr = i / p.g, cc = i - rr * p.g;
            sym[i] = __ldg(dp + i) + __ldg(dp + cc * p.g + rr);
          }
          named_bar_sync(1, kB2ProducerThreads);
          cur_b = it.w.b;
        }
        mbar_wait(bar_empty + 8 * stage, phase ^ 1u, 100u + stage);
        gb2_gen_a(p, it, sym, smem_base + stage * kB2StageBytes, tid);
      }
      gb2_store_b<SRC>(it, r, smem_base + stage * kB2StageBytes + 2 * kB2ATileBytes, tid);
      if (it.half == kB2Batches - 1) {
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_full + 8 * stage);
        if ((int)++stage == kB2Stages) { stage = 0; phase ^= 1u; }
      }
    };
    while (have) {
      Gb2Item n1 = cur;
      const bool h1 = gb2_next(n1, p, u1);
      if (h1) gb2_load<SRC>(p, n1, rb, tid);
      publish(cur, ra);
      if (!h1) break;
      cur = n1;
      have = gb2_next(cur, p, u1);
      if (have) gb2_load<SRC>(p, cur, ra, tid);
      publish(n1, rb);
    }
  } else if (warp == kB2MmaWarp) {
    // =========================== MMA issuer: all k-blocks of a unit ===========================
    const uint32_t idesc = make_idesc_bf16_bmn(128, kB2NHW);
    uint32_t stage = 0, phase = 0, it = 0;
    for (int u = u0; u < u1; ++u, ++it) {
      mbar_wait(bar_tempty, (it & 1u) ^ 1u, 200u);
      tc_fence_after_sync();
      for (int kb = 0; kb < p.nkb; ++kb) {
        mbar_wait(bar_full + 8 * stage, phase, 300u + stage);
        tc_fence_after_sync();
        if (elect_one()) {   // elect.sync, not a lane test: see gram_fwd_pair.cuh
          const uint32_t a_smem = smem_base + stage * kB2StageBytes;
          const uint32_t b_smem = a_smem + 2 * kB2ATileBytes;
#pragma unroll
          for (uint32_t ks = 0; ks < kTileK / kUmmaK; ++ks) {
            if ((int)(kb * 64 + ks * 16) >= p.C) break;
            const uint64_t db = make_smem_desc_sw128_mn(b_smem + ks * 2048u);   // 16 k = two 8-row groups of 1 KB
            for (int a = 0; a < p.nA; ++a)
              umma_bf16(tmem_base + (uint32_t)a * kB2NHW,
                        make_smem_desc_sw128(a_smem + (uint32_t)a * kB2ATileBytes + ks * 32u), db, idesc, (uint32_t)kb | ks);
          }
          umma_commit(bar_empty + 8 * stage);
          if (kb + 1 == p.nkb) umma_commit(bar_tfull);
        }
        __syncwarp();
        if ((int)++stage == kB2Stages) { stage = 0; phase ^= 1u; }
      }
    }
  } else {
    // =========================== epilogue ===========================
    const int q = warp - kB2ProducerWarps;
    uint32_t it = 0;
    for (int u = u0; u < u1; ++u, ++it) {
      const GramBwd2Unit w = gb2_decode(p, u);
      mbar_wait(bar_tfull, it & 1u, 400u);
      tc_fence_after_sync();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
      const int x0 = w.ht * kB2NHW;
#pragma unroll 1
      for (int a = 0; a < p.nA; ++a) {
        const int c = w.cp * 256 + a * 128 + q * 32 + lane;
        float* orow = p.dF + (long long)w.b * p.df_img_stride + (long long)c * p.df_row_stride;
#pragma unroll 1
        for (int n0 = 0; n0 < kB2NHW; n0 += 32) {
          const int x = x0 + n0;
          if (x >= p.HW) break;   // warp-uniform
          float v[32];
          tmem_ld32(taddr + (uint32_t)(a * kB2NHW + n0), v);
          if (c < p.C) {
            if (p.df_vec_ok && x + 32 <= p.HW) {
#pragma unroll
              for (int j = 0; j < 32; j += 4)
                *reinterpret_cast<float4*>(orow + x + j) =
                    make_float4(v[j] * p.scale, v[j + 1] * p.scale, v[j + 2] * p.scale, v[j + 3] * p.scale);
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (x + j < p.HW) orow[x + j] = v[j] * p.scale;
            }
          }
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tempty);
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == kB2MmaWarp) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace gh
