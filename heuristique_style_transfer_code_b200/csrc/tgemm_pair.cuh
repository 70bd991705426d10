// Grouped fp32-accurate GEMM on CTA pairs with TMA-fed split-bf16 operands:
//     D[M][N] (+)= A[M][K] * B[N][K]^T (+ bias[N])            for up to kTgMaxProblems problems in one launch.
//
// This is the linear-layer engine of the attention head and of its backward (reference: nn.MultiheadAttention in_proj /
// out_proj, Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:58, and autograd of it through loss.backward(),
// functions/functions_RESNET50_Truncate_Gram_Attention.py:135). The attention scores of a random-init encoder reach
// 1e4-1e5, so one bf16 pass (3e-3 on the embeddings) is not acceptable: every fp32 operand x lives in global memory as
// two bf16 planes, hi = bf16(x) and lo = bf16(x - hi), written ONCE by whoever produced x (weights: once per weight
// version, gh_split_bf16; activations: by the kernel that computes them), and three MMAs per k-step accumulate
// lo*hi + hi*lo + hi*hi in one fp32 TMEM accumulator (products exact to 2^-16; 6e-6 measured on embeddings/logits).
//
// Machine mapping (the CTA-pair protocol of pair.cuh, as in gram_fwd_pair.cuh):
//   unit      = (problem, 256 x TN output tile, K partition), walked by a cluster of two CTAs; TN = 256 or 128
//   MMA       = tcgen05.mma.cta_group::2.kind::f16, M = 256 (128 rows per CTA), N = TN (TN/2 rows of B per CTA)
//   operands  = cp.async.bulk.tensor straight from the bf16 planes, either K-major ([rows][64 k], box 64 x rows) or
//               MN-major ([64 k][64 mn] atoms through one 4-D box): the same planes serve X W^T (K-major weights), dY W
//               (MN-major weights) and dY^T X (both MN-major) without any transposed copy
//   ring      = 3 stages x {A_hi, A_lo, B_hi, B_lo} x 16 KB per CTA (64 k per stage; GH_TG_KB=32: 6 x 4 x 8 KB)
//   D         = two 256-column TMEM accumulators per CTA: the epilogue of unit i overlaps the MMAs of unit i+1
//   epilogue  = tcgen05.ld -> (+ bias) -> swizzled staging tile -> TMA store (fp32), TMA reduce-add (fp32, K split) or
//               TMA store of the hi / lo bf16 planes of the result (when the consumer is another GEMM of this kind)
// Warps: 0 = TMA producer, 1 = TMEM owner + MMA issuer (leader CTA only), 2-5 = epilogue.
#pragma once
#include "pair.cuh"
#include "launch.cuh"

namespace gh {

// K per stage: 64 (three stages of 64 KB per CTA; K-major tiles [rows][128 B], 128 B swizzle) or, with -DGH_TG_KB=32, 32
// (six stages of 32 KB; K-major tiles [rows][64 B] with the 64 B swizzle; MN-major tiles [atom][32 k][128 B]). The deeper
// ring keeps 160 KB instead of 128 KB per SM in flight; measured on B200 at batch 512 it changes nothing that matters
// (attention forward 57.8 vs 59.4 us, backward 94.2 vs 90.1 us, gpurun_out r2s): with one 256 x 256 unit per CTA pair the
// in_proj GEMM is bounded by its exposed prologue + pipeline fill + epilogue (CTA lifetime 51 k cycles for 24.6 k cycles of
// MMAs), not by bytes in flight. Both settings pass the parity tests.
#ifndef GH_TG_KB
#define GH_TG_KB 64
#endif
constexpr int kTgKB = GH_TG_KB;
static_assert(kTgKB == 32 || kTgKB == 64, "tgemm_pair: K block of 32 or 64");
constexpr int kTgStages = kTgKB == 64 ? 3 : 6;
constexpr uint32_t kTgRowB = kTgKB * 2;                      // bytes of one K-major row: 128 | 64
constexpr uint32_t kTgTile = 128 * kTgRowB;                  // [128 rows][row] (or 2 MN-major atoms of [KB k][128 B]): 16 | 8 KB
constexpr uint32_t kTgStageBytes = 4 * kTgTile;              // A_hi | A_lo | B_hi | B_lo, this CTA's halves
constexpr uint32_t kTgKSteps = kTgKB / 16;                   // MMAs (x3) per stage: 4 | 2
// K-major operand descriptor: 8-row groups of kTgRowB bytes; SWIZZLE_128B (layout 2) or SWIZZLE_64B (layout 4)
__host__ __device__ constexpr uint64_t tg_desc_kmajor(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)((8u * kTgRowB) >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)(kTgKB == 64 ? 2 : 4) << 61);
}
constexpr int kTgStoreBufs = 2;                              // staging tiles per epilogue warp
constexpr uint32_t kTgStoreBytes = 4 * kTgStoreBufs * 4096;
constexpr uint32_t kTgSmemBytes = kTgStages * kTgStageBytes + kTgStoreBytes + 1024 + 256;
constexpr int kTgThreads = 6 * 32;
constexpr int kTgMaxProblems = 2;
static_assert(kTgSmemBytes <= 232448, "tgemm_pair: shared memory budget");

enum : int { TG_OUT_F32 = 0, TG_OUT_F32_ADD = 1, TG_OUT_PLANES = 2 };

struct TgProblem {
  int M, N, K;
  int a_mn, b_mn;        // 0 = K-major planes, 1 = MN-major planes
  int tn;                // N tile: 256 or 128
  int tiles_n, ksplit, nkb;
  int unit0, nunits;     // this problem's slice of the unit list
  int out_mode;          // TG_OUT_*
  const float* bias;     // [N] or null; added by K partition 0
};
struct TgParams {
  TgProblem prob[kTgMaxProblems];
  int nprob, total_units;
};
struct alignas(64) TgMaps {
  CUtensorMap a[kTgMaxProblems], b[kTgMaxProblems], d[kTgMaxProblems];
};

struct TgUnit {
  int pi, m0, n0, kb0, kb1, ks;
};
__device__ __forceinline__ TgUnit tg_decode(const TgParams& p, int u) {
  TgUnit w;
  w.pi = (p.nprob > 1 && u >= p.prob[1].unit0) ? 1 : 0;
  const TgProblem& q = p.prob[w.pi];
  const int v = u - q.unit0;
  w.ks = v % q.ksplit;
  const int tile = v / q.ksplit;
  w.m0 = (tile / q.tiles_n) * 256;
  w.n0 = (tile % q.tiles_n) * q.tn;
  w.kb0 = (int)(((long long)q.nkb * w.ks) / q.ksplit);
  w.kb1 = (int)(((long long)q.nkb * (w.ks + 1)) / q.ksplit);
  return w;
}

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tmap, uint32_t src_smem, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tmap)),
               "r"(src_smem), "r"(c0), "r"(c1)
               : "memory");
}
// D += tile (fp32 add performed by the memory system; the order among K partitions is not fixed)
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* tmap, uint32_t src_smem, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tmap)),
               "r"(src_smem), "r"(c0), "r"(c1)
               : "memory");
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kTgThreads, 1)
    tgemm_pair_kernel(const TgParams p, const __grid_constant__ TgMaps maps) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t store_smem = smem_base + kTgStages * kTgStageBytes;
  const uint32_t bars = store_smem + kTgStoreBytes;
  const uint32_t bar_full = bars, bar_empty = bars + 8 * kTgStages;
  const uint32_t bar_tfull = bars + 16 * kTgStages, bar_tempty = bar_tfull + 16;
  const uint32_t tmem_slot = bar_tempty + 16;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = (int)cluster_id_x(), npairs = (int)cluster_nclusters_x();

  pdl_launch_dependents();
  if (threadIdx.x == 0) {
    for (int i = 0; i < p.nprob; ++i) {
      tma_prefetch_desc(&maps.a[i]);
      tma_prefetch_desc(&maps.b[i]);
      tma_prefetch_desc(&maps.d[i]);
    }
    for (int s = 0; s < kTgStages; ++s) {
      mbar_init(bar_full + 8 * s, 1);      // the leader's arrive.expect_tx; both CTAs' TMA bytes complete on it
      mbar_init(bar_empty + 8 * s, 1);     // multicast tcgen05.commit
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_tfull + 8 * a, 1);
      mbar_init(bar_tempty + 8 * a, 8);    // 4 epilogue warps x 2 CTAs
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc2(tmem_slot, 512);
  tc_fence_before_sync();
  cluster_sync_all();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const uint32_t full_leader = mapa_u32(bar_full, 0);
  const uint32_t tempty_leader = mapa_u32(bar_tempty, 0);
  const bool elected = elect_one();        // elect.sync, not a lane test: see gram_fwd_pair.cuh
  pdl_wait();                              // operands and zeroed outputs come from the previous kernels of the chain

  if (warp == 0) {
    // =========================== TMA producer (one thread): this CTA's halves of A and B, both planes ================
    if (elected) {
      uint32_t stage = 0, phase = 0;
      for (int u = pair; u < p.total_units; u += npairs) {
        const TgUnit w = tg_decode(p, u);
        const TgProblem& q = p.prob[w.pi];
        const CUtensorMap* ma = &maps.a[w.pi];
        const CUtensorMap* mb = &maps.b[w.pi];
        const int half = q.tn >> 1;
        const uint32_t tx_bytes = 2u * (2u * kTgTile + 2u * (uint32_t)half * kTgRowB);
        const int rowA = w.m0 + (int)rank * 128, rowB = w.n0 + (int)rank * half;
        for (int kb = w.kb0; kb < w.kb1; ++kb) {
          mbar_wait(bar_empty + 8 * stage, phase ^ 1u, 100u + stage);
          if (rank == 0) mbar_arrive_expect_tx(bar_full + 8 * stage, tx_bytes);
          const uint32_t st = smem_base + stage * kTgStageBytes;
          const uint32_t fb = full_leader + 8 * stage;
#pragma unroll
          for (int pl = 0; pl < 2; ++pl) {
            if (q.a_mn) tma_load_4d_pair(st + pl * kTgTile, ma, fb, 0, kb * kTgKB, rowA >> 6, pl);
            else tma_load_3d_pair(st + pl * kTgTile, ma, fb, kb * kTgKB, rowA, pl);
            if (q.b_mn) tma_load_4d_pair(st + (2 + pl) * kTgTile, mb, fb, 0, kb * kTgKB, rowB >> 6, pl);
            else tma_load_3d_pair(st + (2 + pl) * kTgTile, mb, fb, kb * kTgKB, rowB, pl);
          }
          if (++stage == kTgStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // =========================== MMA issuer (one thread of the leader CTA) ===========================
    if (rank == 0 && elected) {
      constexpr uint64_t kStageInc = kTgStageBytes >> 4, kTileInc = kTgTile >> 4;
      uint32_t stage = 0, phase = 0, it = 0;
      for (int u = pair; u < p.total_units; u += npairs, ++it) {
        const TgUnit w = tg_decode(p, u);
        const TgProblem& q = p.prob[w.pi];
        const uint32_t idesc = make_idesc(1u, 256u, (uint32_t)q.tn, (uint32_t)q.a_mn, (uint32_t)q.b_mn);
        // K-major tiles advance 32 B inside the 128 B row per MMA, MN-major ones by 16 k-rows of 128 B
        const uint64_t dA0 = q.a_mn ? make_smem_desc_sw128_mnmajor(smem_base, kTgKB * 128u) : tg_desc_kmajor(smem_base);
        const uint64_t dB0 = q.b_mn ? make_smem_desc_sw128_mnmajor(smem_base + 2 * kTgTile, kTgKB * 128u)
                                    : tg_desc_kmajor(smem_base + 2 * kTgTile);
        const uint64_t kAInc = q.a_mn ? 128u : 2u, kBInc = q.b_mn ? 128u : 2u;
        const uint32_t ab = it & 1u, use = it >> 1;
        mbar_wait_cl(bar_tempty + 8 * ab, (use & 1u) ^ 1u, 200u + ab);
        tc_fence_after_sync();
        const uint32_t acc = tmem_base + ab * 256u;
        for (int kb = w.kb0; kb < w.kb1; ++kb) {
          mbar_wait_cl(bar_full + 8 * stage, phase, 300u + stage);
          tc_fence_after_sync();
          const uint64_t ah = dA0 + stage * kStageInc, al = ah + kTileInc;
          const uint64_t bh = dB0 + stage * kStageInc, bl = bh + kTileInc;
#pragma unroll
          for (uint32_t ks = 0; ks < kTgKSteps; ++ks) {
            // small terms first, then the dominant hi*hi
            umma2<KIND_BF16>(acc, al + ks * kAInc, bh + ks * kBInc, idesc, (kb != w.kb0 || ks != 0) ? 1u : 0u);
            umma2<KIND_BF16>(acc, ah + ks * kAInc, bl + ks * kBInc, idesc, 1u);
            umma2<KIND_BF16>(acc, ah + ks * kAInc, bh + ks * kBInc, idesc, 1u);
          }
          umma_commit2(bar_empty + 8 * stage);
          if (kb + 1 == w.kb1) umma_commit2(bar_tfull + 8 * ab);
          if (++stage == kTgStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else {
    // =========================== epilogue: TMEM -> (+bias) -> staging -> TMA store / reduce-add ======================
    const int q4 = warp & 3;                                 // TMEM lane quarter this warp may read
    const uint32_t my_store = store_smem + (uint32_t)(warp - 2) * (kTgStoreBufs * 4096u);
    uint32_t it = 0, buf = 0;
    for (int u = pair; u < p.total_units; u += npairs, ++it) {
      const TgUnit w = tg_decode(p, u);
      const TgProblem& q = p.prob[w.pi];
      const CUtensorMap* md = &maps.d[w.pi];
      const uint32_t ab = it & 1u, use = it >> 1;
      mbar_wait(bar_tfull + 8 * ab, use & 1u, 400u + ab);
      tc_fence_after_sync();
      const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + ab * 256u;
      const int row0 = w.m0 + (int)rank * 128 + q4 * 32;
      if (row0 < q.M) {                                      // warp-uniform: rows beyond M are padding
        const bool add_bias = q.bias != nullptr && w.ks == 0;
#pragma unroll 1
        for (int c0 = 0; c0 < q.tn; c0 += 32) {
          const int n = w.n0 + c0;
          if (n >= q.N) break;
          float v[32];
          tmem_ld32(taddr + (uint32_t)c0, v);
          if (add_bias) {                                    // N % 32 == 0: the chunk lies inside [0, N)
            const float4* bp = reinterpret_cast<const float4*>(q.bias + n);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 bv = __ldg(bp + j);
              v[4 * j] += bv.x; v[4 * j + 1] += bv.y; v[4 * j + 2] += bv.z; v[4 * j + 3] += bv.w;
            }
          }
          if (elected) tma_store_wait_read<kTgStoreBufs - 1>();   // the staging tile about to be reused has been read
          __syncwarp();
          const uint32_t tile = my_store + buf * 4096u;
          if (q.out_mode == TG_OUT_PLANES) {
            // two [32 rows][32 bf16 = 64 B] tiles, SWIZZLE_64B: 16 B chunk c of row r sits at chunk c ^ ((r >> 1) & 3)
            const uint32_t rbase = tile + (uint32_t)lane * 64u, sw = ((uint32_t)lane >> 1) & 3u;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              uint32_t hi[4], lo[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float x0 = v[8 * c + 2 * e], x1 = v[8 * c + 2 * e + 1];
                const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
                const float2 f = __bfloat1622float2(h);
                hi[e] = *reinterpret_cast<const uint32_t*>(&h);
                lo[e] = pack_bf16x2(x0 - f.x, x1 - f.y);
              }
              const uint32_t off = (((uint32_t)c ^ sw) << 4);
              sts_u4(rbase + off, hi[0], hi[1], hi[2], hi[3]);
              sts_u4(rbase + 2048u + off, lo[0], lo[1], lo[2], lo[3]);
            }
          } else {
            // [32 rows][32 fp32 = 128 B], SWIZZLE_128B
            const uint32_t rbase = tile + (uint32_t)lane * kRowBytes;
#pragma unroll
            for (int j = 0; j < 8; ++j)
              sts_u4(rbase + ((((uint32_t)j) ^ ((uint32_t)lane & 7u)) << 4), __float_as_uint(v[4 * j]),
                     __float_as_uint(v[4 * j + 1]), __float_as_uint(v[4 * j + 2]), __float_as_uint(v[4 * j + 3]));
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (elected) {
            if (q.out_mode == TG_OUT_PLANES) {
              tma_store_3d(md, tile, n, row0, 0);
              tma_store_3d(md, tile + 2048u, n, row0, 1);
            } else if (q.out_mode == TG_OUT_F32_ADD) {
              tma_reduce_add_2d(md, tile, n, row0);
            } else {
              tma_store_2d(md, tile, n, row0);
            }
            tma_store_commit();
          }
          buf = (buf + 1u) % kTgStoreBufs;
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty_leader + 8 * ab);
    }
    if (elected) tma_store_wait_all<0>();
    __syncwarp();
  }

  __syncwarp();
  tc_fence_before_sync();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc2(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------
// A split operand: two bf16 planes (hi, lo) `plane_stride` elements apart, each a matrix with leading dimension ld.
//   mn_major = 0: element (row, k) at row*ld + k   (rows = the operand's M or N index, k contiguous)
//   mn_major = 1: element (row, k) at k*ld + row   (the operand's M / N index contiguous)
struct TgOperand {
  const void* planes;
  long long ld, plane_stride;
  int mn_major;
};
struct TgSpec {
  TgOperand A, B;
  int M, N, K;
  const float* bias;
  float* D_f32;          // fp32 result (ldd), or null when the result leaves as planes
  void* D_planes;        // bf16 hi/lo planes of the result (ldd, d_plane_stride), or null
  long long ldd, d_plane_stride;
  int max_split;         // 1 = never split K; 2 = at most two partitions (bitwise reproducible: two partial sums meeting
                         // in a zeroed slot add to the same bits in either order); larger = free. Planes output: 1.
  // filled by tg_plan():
  int tn, ksplit;
};

inline bool tg_map_operand(CUtensorMap* map, const TgOperand& o, int rows, int K, int box_rows) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return false;
  if ((reinterpret_cast<uintptr_t>(o.planes) & 15u) || (o.ld * 2) % 16 || (o.plane_stride * 2) % 16) return false;
  if (!o.mn_major) {
    cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)rows, 2};
    cuuint64_t strides[2] = {(cuuint64_t)(o.ld * 2), (cuuint64_t)(o.plane_stride * 2)};
    cuuint32_t box[3] = {(cuuint32_t)kTgKB, (cuuint32_t)box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(o.planes), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, kTgKB == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
  }
  if (rows % 64 != 0 || box_rows % 64 != 0) return false;
  cuuint64_t dims[4] = {64, (cuuint64_t)K, (cuuint64_t)(rows / 64), 2};
  cuuint64_t strides[3] = {(cuuint64_t)(o.ld * 2), 128, (cuuint64_t)(o.plane_stride * 2)};
  cuuint32_t box[4] = {64, (cuuint32_t)kTgKB, (cuuint32_t)(box_rows / 64), 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(o.planes), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
inline bool tg_map_out(CUtensorMap* map, const TgSpec& s) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return false;
  cuuint32_t estr[3] = {1, 1, 1};
  if (s.D_planes) {
    if ((reinterpret_cast<uintptr_t>(s.D_planes) & 15u) || (s.ldd * 2) % 16 || (s.d_plane_stride * 2) % 16) return false;
    cuuint64_t dims[3] = {(cuuint64_t)s.N, (cuuint64_t)s.M, 2};
    cuuint64_t strides[2] = {(cuuint64_t)(s.ldd * 2), (cuuint64_t)(s.d_plane_stride * 2)};
    cuuint32_t box[3] = {32, 32, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, s.D_planes, dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
  }
  if ((reinterpret_cast<uintptr_t>(s.D_f32) & 15u) || (s.ldd * 4) % 16) return false;
  cuuint64_t dims[2] = {(cuuint64_t)s.N, (cuuint64_t)s.M};
  cuuint64_t strides[1] = {(cuuint64_t)(s.ldd * 4)};
  cuuint32_t box[2] = {32, 32};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, s.D_f32, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Tile width and K partitions per problem. Cost model in units of one 256 x 256 x 64 k-block (12 MMAs, ~1 us):
// a unit of `len` k-blocks at width tn costs len * tn/256 + 1.5 (pipeline fill + exposed epilogue); the launch takes ceil(units / pairs) rounds of the longest unit. For every
// target unit length U the largest admissible unit <= U is taken per problem, and the U with the smallest estimate wins.
// Measured against it on B200 (gpurun_out r2t, attention forward / backward at batch 512): forcing tn = 128 everywhere
// 65.9 / 112.6 us, tn = 256 everywhere 72.1 / 122.9 us, this plan 59.4 / 90.1 us -- in particular two 128-wide units per
// pair for the in_proj GEMM (to overlap one epilogue) lose to one 256-wide unit.
static int g_opt_tg_tn = 0;            // 0 = plan; 128 / 256 force the tile width (experiments, gh_set_option "tgemm_tn")
inline void tg_plan(TgSpec* specs, int n, int npairs) {
  static const int kTargets[] = {2, 3, 4, 6, 8, 12, 16, 24, 32, 48, 64, 96, 128, 192, 256};
  double best = 1e30;
  int best_tn[kTgMaxProblems] = {256, 256}, best_ks[kTgMaxProblems] = {1, 1};
  for (int U : kTargets) {
    int tn_c[kTgMaxProblems], ks_c[kTgMaxProblems];
    long long units = 0;
    double longest = 0;
    for (int i = 0; i < n; ++i) {
      const TgSpec& s = specs[i];
      const int nkb = (s.K + kTgKB - 1) / kTgKB;
      double pick_cost = -1;
      int pick_tn = 256, pick_ks = 1;
      double fallback_cost = 1e30;        // nothing fits under U: the shortest admissible unit
      int fb_tn = 256, fb_ks = 1;
      for (int tn = 256; tn >= 128; tn >>= 1) {
        if (tn == 128 && s.N % 128 != 0 && s.N > 128) continue;
        if (g_opt_tg_tn && tn != g_opt_tg_tn) continue;
        for (int ks = 1; ks <= nkb && ks <= (s.max_split > 0 ? s.max_split : 1); ++ks) {
          if (ks > 1 && nkb / ks < 2 * (64 / kTgKB)) break;
          const double cost = (double)((nkb + ks - 1) / ks) * tn / 256.0 * kTgKB / 64.0;
          // equal length: the unsplit (narrower) tiling wins -- no zeroed output, no reduce-add traffic
          if (cost <= U && (cost > pick_cost + 1e-9 || (cost > pick_cost - 1e-9 && ks < pick_ks))) {
            pick_cost = cost; pick_tn = tn; pick_ks = ks;
          }
          if (cost < fallback_cost) { fallback_cost = cost; fb_tn = tn; fb_ks = ks; }
        }
      }
      if (pick_cost < 0) { pick_cost = fallback_cost; pick_tn = fb_tn; pick_ks = fb_ks; }
      tn_c[i] = pick_tn; ks_c[i] = pick_ks;
      units += (long long)((s.M + 255) / 256) * ((s.N + pick_tn - 1) / pick_tn) * pick_ks;
      if (pick_cost > longest) longest = pick_cost;
    }
    const double rounds = (double)((units + npairs - 1) / npairs);
    const double est = rounds * (longest + 1.5);
    if (est < best - 1e-9) {
      best = est;
      for (int i = 0; i < n; ++i) { best_tn[i] = tn_c[i]; best_ks[i] = ks_c[i]; }
    }
  }
  for (int i = 0; i < n; ++i) { specs[i].tn = best_tn[i]; specs[i].ksplit = best_ks[i]; }
}

// A planned launch: parameters and tensor maps, built on the host before anything is enqueued.
struct TgLaunch {
  TgParams p;
  TgMaps maps;
  int npairs;
};

// Supported: K-major operands with ld % 8 == 0; MN-major operands whose M / N extent is a multiple of 64; 16 B aligned
// planes. Returns cudaErrorNotSupported otherwise (the caller then uses the ld.global kernels of umma_gemm.cuh).
// specs[] must have been planned with tg_plan(). Enqueues nothing, so a caller that has more to do before the launch
// (zeroing a K-split output, kernels that feed the GEMM) checks here first and writes nothing when the shape is refused.
inline cudaError_t tg_prepare(const TgSpec* specs, int n, int sms, TgLaunch* out) {
  if (n < 1 || n > kTgMaxProblems || sms < 2) return cudaErrorNotSupported;
  TgParams& p = out->p;
  TgMaps& maps = out->maps;
  p = TgParams{};
  int units = 0;
  for (int i = 0; i < n; ++i) {
    const TgSpec& s = specs[i];
    if (s.M <= 0 || s.N <= 0 || s.K <= 0 || (s.tn != 128 && s.tn != 256) || s.ksplit < 1) return cudaErrorInvalidValue;
    if ((s.D_planes != nullptr) == (s.D_f32 != nullptr)) return cudaErrorInvalidValue;
    if (s.D_planes && s.ksplit != 1) return cudaErrorInvalidValue;
    if (s.N % 32 != 0 || (reinterpret_cast<uintptr_t>(s.bias) & 15u)) return cudaErrorNotSupported;
    TgProblem& q = p.prob[i];
    q.M = s.M; q.N = s.N; q.K = s.K;
    q.a_mn = s.A.mn_major; q.b_mn = s.B.mn_major;
    q.tn = s.tn; q.tiles_n = (s.N + s.tn - 1) / s.tn; q.ksplit = s.ksplit; q.nkb = (s.K + kTgKB - 1) / kTgKB;
    q.unit0 = units;
    q.nunits = ((s.M + 255) / 256) * q.tiles_n * q.ksplit;
    units += q.nunits;
    q.out_mode = s.D_planes ? TG_OUT_PLANES : (s.ksplit > 1 ? TG_OUT_F32_ADD : TG_OUT_F32);
    q.bias = s.bias;
    if (!tg_map_operand(&maps.a[i], s.A, s.M, s.K, 128) || !tg_map_operand(&maps.b[i], s.B, s.N, s.K, s.tn / 2) ||
        !tg_map_out(&maps.d[i], s))
      return cudaErrorNotSupported;
  }
  for (int i = n; i < kTgMaxProblems; ++i) {      // unused slots: valid (never dereferenced) descriptors
    maps.a[i] = maps.a[0]; maps.b[i] = maps.b[0]; maps.d[i] = maps.d[0];
  }
  p.nprob = n;
  p.total_units = units;
  out->npairs = sms / 2;
  if (units < out->npairs) out->npairs = units;
  return cudaSuccess;
}
// A problem with ksplit > 1 accumulates into D_f32, which the caller has zeroed earlier in the stream.
inline cudaError_t tg_launch(const TgLaunch& l, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(tgemm_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTgSmemBytes);
  if (e != cudaSuccess) return e;
  return launch_pdl(tgemm_pair_kernel, dim3(2 * l.npairs), dim3(kTgThreads), kTgSmemBytes, st, l.p, l.maps);
}

}  // namespace gh
