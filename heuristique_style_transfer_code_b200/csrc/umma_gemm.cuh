// fp32-in / fp32-out GEMM on tcgen05 with split-bf16 operands:  D[M][N] = A[M][K] * B[N][K]^T (+ bias[N]).
//
// Used for every linear layer of the attention head and its backward (reference: nn.MultiheadAttention in_proj /
// out_proj, Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:58, and autograd of it). The attention scores of
// a random-init encoder reach 1e4-1e5, so single-pass bf16 (rel. err 3e-3 on the embeddings) is not acceptable here;
// each fp32 operand x is split in the producer as x = hi + lo (hi = bf16(x), lo = bf16(x - hi)) and three MMAs per
// k-step accumulate hi*hi + hi*lo + lo*hi in the same fp32 TMEM accumulator: products are exact to 2^-16, measured
// 6e-6 on embeddings/logits (fp32 FMA level) at a third of the bf16 tensor rate -- still > 10x the fp32 SIMT rate.
//
// Operand storage in global memory (fp32):
//   A_MN = false: A(m, k) = A[m*lda + k]   (k contiguous: activations x weights^T, "NT")
//   A_MN = true : A(m, k) = A[k*lda + m]   (m contiguous: dW = dY^T X reads dY as [k = row][m])
//   B_MN = false: B(n, k) = B[n*ldb + k]   (nn.Linear weight (N, K))
//   B_MN = true : B(n, k) = B[k*ldb + n]   (dX = dY W reads W as [k][n]; dW reads X as [k = row][n])
// K-major operands go to smem as [rows][64 k] SWIZZLE_128B (common.cuh); MN-major ones as [mn/64][k/8][k%8][64 mn]
// with the 16 B chunks XOR-swizzled by k%8 -- in both cases the global reads are coalesced float4 along the
// contiguous axis and the smem writes are conflict-free 8 B stores.
//
// Tiling: CTA tile 128 (M) x 256 (N), K blocks of 64, 2 smem stages of {A_hi, A_lo, B_hi, B_lo} = 96 KB, two 256-column
// TMEM accumulators (epilogue of tile i overlaps the MMAs of tile i+1). Persistent CTAs, work items round-robin; when
// the tiles alone cannot fill the SMs (M = B*L is a few hundred rows) K is split across CTAs and the partial sums meet
// in red.global.add.f32 on a zeroed D (bias added by partition 0).
// Warps: 0-7 producers (register double buffering in batches of 128 rows x 64 k), 8-11 epilogue, 12 MMA issuer.
// Requirements (checked by the launcher, which otherwise uses the fp32 SIMT kernel): the contiguous extent and the
// leading dimension of each operand are multiples of 4 elements and the base pointers are 16 B aligned.
#pragma once
#include "common.cuh"

namespace gh {

constexpr int kUgProducerThreads = 256;
constexpr int kUgEpiWarp0 = 8;
constexpr int kUgMmaWarp = 12;
constexpr int kUgThreads = 13 * 32;
constexpr uint32_t kUgATile = 128 * 128;           // 16 KB: 128 rows (or 2 x 64-wide MN blocks) x 64 k bf16
constexpr uint32_t kUgBTile = 256 * 128;           // 32 KB
constexpr uint32_t kUgStageBytes = 2 * kUgATile + 2 * kUgBTile;   // 96 KB
constexpr int kUgStages = 2;
constexpr uint32_t kUgSmemBytes = kUgStages * kUgStageBytes + 1024 + 256;

struct UmmaGemmParams {
  const float* A; long long lda;
  const float* B; long long ldb;
  const float* bias;     // [N] or null
  float* D; long long ldd;
  int M, N, K;
  int tiles_m, tiles_n, nkb;
  int ksplit;            // K partitions per tile; > 1: partial sums meet in red.global.add.f32 on a zeroed D
  int nwork;             // tiles_m * tiles_n * ksplit
};

__host__ __device__ constexpr uint64_t ug_desc_k(uint32_t addr) { return make_smem_desc_sw128(addr); }
__host__ __device__ constexpr uint64_t ug_desc_mn(uint32_t addr) {
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(8192u >> 4) << 16) | ((uint64_t)(1024u >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}

struct UgWork {
  int m0, n0, kb0, kb1, ks;
};
// work item w -> (tile, K partition); the K partitions of a tile are adjacent so they run concurrently and hit L2
__device__ __forceinline__ UgWork ug_work(const UmmaGemmParams& p, int w) {
  UgWork u;
  u.ks = w % p.ksplit;
  const int tile = w / p.ksplit;
  u.m0 = (tile / p.tiles_n) * 128;
  u.n0 = (tile % p.tiles_n) * 256;
  u.kb0 = (int)(((long long)p.nkb * u.ks) / p.ksplit);
  u.kb1 = (int)(((long long)p.nkb * (u.ks + 1)) / p.ksplit);
  return u;
}
struct UgItem {
  int w, kb, part;   // part 0 = A (128 rows), 1 = B rows 0-127, 2 = B rows 128-255
  int m0, n0, kb1;
};
__device__ __forceinline__ void ug_set_work(UgItem& it, const UmmaGemmParams& p) {
  const UgWork u = ug_work(p, it.w);
  it.m0 = u.m0; it.n0 = u.n0; it.kb = u.kb0; it.kb1 = u.kb1;
}
__device__ __forceinline__ bool ug_first(UgItem& it, const UmmaGemmParams& p) {
  it.w = blockIdx.x;
  if (it.w >= p.nwork) return false;
  it.part = 0;
  ug_set_work(it, p);
  return true;
}
__device__ __forceinline__ bool ug_next(UgItem& it, const UmmaGemmParams& p) {
  if (++it.part < 3) return true;
  it.part = 0;
  if (++it.kb < it.kb1) return true;
  it.w += gridDim.x;
  if (it.w >= p.nwork) return false;
  ug_set_work(it, p);
  return true;
}

// One batch: a 128 (rows of the operand) x 64 (k) block, 8 float4 per thread.
template <bool A_MN, bool B_MN>
__device__ __forceinline__ void ug_load(const UmmaGemmParams& p, const UgItem& it, float4 (&r)[8], int tid) {
  const bool isA = it.part == 0;
  const bool mn = isA ? A_MN : B_MN;
  const float* base = isA ? p.A : p.B;
  const long long ld = isA ? p.lda : p.ldb;
  const int row0 = isA ? it.m0 : it.n0 + (it.part - 1) * 128;   // first operand row (m or n) of this batch
  const int rows = isA ? p.M : p.N;
  const int k0 = it.kb * 64;
  const int seg = tid >> 4, q = tid & 15;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    r[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!mn) {
      // K-major source: 16 threads cover one row's 64 k; 16 rows per pass
      const int row = row0 + seg + 16 * i;
      const int k = k0 + q * 4;
      if (row < rows && k < p.K) r[i] = ldg_stream_f4(base + (long long)row * ld + k);
    } else {
      // MN-major source: segment s = (k row, 64-wide block); 16 threads cover 64 consecutive rows (m or n)
      const int s = seg + 16 * i;              // 0..127
      const int k = k0 + (s >> 1);
      const int row = row0 + (s & 1) * 64 + q * 4;
      if (k < p.K && row < rows) r[i] = ldg_stream_f4(base + (long long)k * ld + row);
    }
  }
}

template <bool A_MN, bool B_MN>
__device__ __forceinline__ void ug_store(const UgItem& it, const float4 (&r)[8], uint32_t stage_smem, int tid) {
  const bool isA = it.part == 0;
  const bool mn = isA ? A_MN : B_MN;
  // stage layout: [A_hi 16K][A_lo 16K][B_hi 32K][B_lo 32K]; B rows 128-255 start 16 KB into each B tile for K-major,
  // and 2 blocks x 8 KB = 16 KB for MN-major as well
  const uint32_t hi = stage_smem + (isA ? 0u : (2u * kUgATile + (uint32_t)(it.part - 1) * 16384u));
  const uint32_t lo_off = isA ? kUgATile : kUgBTile;
  const int seg = tid >> 4, q = tid & 15;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    uint32_t off;
    if (!mn) {
      off = sw128_off((uint32_t)(seg + 16 * i), (uint32_t)(q * 4));
    } else {
      const uint32_t s = (uint32_t)(seg + 16 * i), kl = s >> 1, xb = s & 1u;
      off = xb * 8192u + (kl >> 3) * 1024u + (kl & 7u) * 128u + ((((uint32_t)q >> 1) ^ (kl & 7u)) << 4) + (((uint32_t)q & 1u) << 3);
    }
    const __nv_bfloat162 h01 = __floats2bfloat162_rn(r[i].x, r[i].y), h23 = __floats2bfloat162_rn(r[i].z, r[i].w);
    const float2 f01 = __bfloat1622float2(h01), f23 = __bfloat1622float2(h23);
    sts_u2(hi + off, *reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23));
    sts_u2(hi + lo_off + off, pack_bf16x2(r[i].x - f01.x, r[i].y - f01.y), pack_bf16x2(r[i].z - f23.x, r[i].w - f23.y));
  }
}

template <bool A_MN, bool B_MN>
__global__ void __launch_bounds__(kUgThreads, 1) umma_gemm_kernel(const UmmaGemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bars = smem_base + kUgStages * kUgStageBytes;
  const uint32_t bar_full = bars, bar_empty = bars + 8 * kUgStages;
  const uint32_t bar_tfull = bars + 16 * kUgStages, bar_tempty = bar_tfull + 16;
  const uint32_t tmem_slot = bar_tempty + 16;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kUgStages; ++s) {
      mbar_init(bar_full + 8 * s, 8);
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_tfull + 8 * a, 1);
      mbar_init(bar_tempty + 8 * a, 4);
    }
    mbar_fence_init();
  }
  if (warp == kUgMmaWarp) tmem_alloc(tmem_slot, 512);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp < 8) {
    // =========================== producers ===========================
    const int tid = threadIdx.x;
    uint32_t stage = 0, phase = 0;
    float4 ra[8], rb[8];
    UgItem cur;
    bool have = ug_first(cur, p);
    if (have) ug_load<A_MN, B_MN>(p, cur, ra, tid);
    auto publish = [&](const UgItem& it, const float4 (&r)[8]) {
      if (it.part == 0) mbar_wait(bar_empty + 8 * stage, phase ^ 1u, 100u + stage);
      ug_store<A_MN, B_MN>(it, r, smem_base + stage * kUgStageBytes, tid);
      if (it.part == 2) {
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_full + 8 * stage);
        if (++stage == (uint32_t)kUgStages) { stage = 0; phase ^= 1u; }
      }
    };
    while (have) {
      UgItem n1 = cur;
      const bool h1 = ug_next(n1, p);
      if (h1) ug_load<A_MN, B_MN>(p, n1, rb, tid);
      publish(cur, ra);
      if (!h1) break;
      cur = n1;
      have = ug_next(cur, p);
      if (have) ug_load<A_MN, B_MN>(p, cur, ra, tid);
      publish(n1, rb);
    }
  } else if (warp == kUgMmaWarp) {
    // =========================== MMA issuer ===========================
    uint32_t stage = 0, phase = 0, it = 0;
    const uint32_t idesc = make_idesc_bf16(128, 256) | (A_MN ? (1u << 15) : 0u) | (B_MN ? (1u << 16) : 0u);
    for (int w = blockIdx.x; w < p.nwork; w += gridDim.x, ++it) {
      const UgWork u = ug_work(p, w);
      const uint32_t ab = it & 1u, use = it >> 1;
      mbar_wait(bar_tempty + 8 * ab, (use & 1u) ^ 1u, 200u + ab);
      tc_fence_after_sync();
      for (int kb = u.kb0; kb < u.kb1; ++kb) {
        mbar_wait(bar_full + 8 * stage, phase, 300u + stage);
        tc_fence_after_sync();
        if (elect_one()) {   // elect.sync, not a lane test: see gram_fwd_pair.cuh
          const uint32_t a_hi = smem_base + stage * kUgStageBytes, a_lo = a_hi + kUgATile;
          const uint32_t b_hi = a_hi + 2 * kUgATile, b_lo = b_hi + kUgBTile;
#pragma unroll
          for (uint32_t ks = 0; ks < 4; ++ks) {
            if ((int)(kb * 64 + ks * 16) >= p.K) break;
            const uint32_t ka = A_MN ? ks * 2048u : ks * 32u, kbo = B_MN ? ks * 2048u : ks * 32u;
            const uint64_t dah = A_MN ? ug_desc_mn(a_hi + ka) : ug_desc_k(a_hi + ka);
            const uint64_t dal = A_MN ? ug_desc_mn(a_lo + ka) : ug_desc_k(a_lo + ka);
            const uint64_t dbh = B_MN ? ug_desc_mn(b_hi + kbo) : ug_desc_k(b_hi + kbo);
            const uint64_t dbl = B_MN ? ug_desc_mn(b_lo + kbo) : ug_desc_k(b_lo + kbo);
            const uint32_t d = tmem_base + ab * 256u;
            umma_bf16(d, dal, dbh, idesc, (uint32_t)(kb - u.kb0) | ks);   // small terms first, then the dominant hi*hi
            umma_bf16(d, dah, dbl, idesc, 1u);
            umma_bf16(d, dah, dbh, idesc, 1u);
          }
          umma_commit(bar_empty + 8 * stage);
          if (kb + 1 == u.kb1) umma_commit(bar_tfull + 8 * ab);
        }
        __syncwarp();
        if (++stage == (uint32_t)kUgStages) { stage = 0; phase ^= 1u; }
      }
    }
  } else {
    // =========================== epilogue ===========================
    const int q = warp - kUgEpiWarp0;
    uint32_t it = 0;
    const bool vec = (p.ldd % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.D) & 15u) == 0);
    const bool atomics = p.ksplit > 1;
    for (int w = blockIdx.x; w < p.nwork; w += gridDim.x, ++it) {
      const UgWork u = ug_work(p, w);
      const uint32_t ab = it & 1u, use = it >> 1;
      const int m = u.m0 + q * 32 + lane;
      const int n_tile = u.n0;
      mbar_wait(bar_tfull + 8 * ab, use & 1u, 400u + ab);
      tc_fence_after_sync();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + ab * 256u;
      float* drow = p.D + (long long)m * p.ldd;
#pragma unroll 1
      for (int c0 = 0; c0 < 256; c0 += 32) {
        const int n = n_tile + c0;
        if (n >= p.N) break;
        float v[32];
        tmem_ld32(taddr + (uint32_t)c0, v);
        if (p.bias && u.ks == 0) {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (n + j < p.N) v[j] += __ldg(p.bias + n + j);
        }
        if (m < p.M) {
          if (atomics) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (n + j < p.N) red_add_f32(drow + n + j, v[j]);
          } else if (vec && n + 32 <= p.N) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(drow + n + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (n + j < p.N) drow[n + j] = v[j];
          }
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tempty + 8 * ab);
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == kUgMmaWarp) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
}

// Launcher. Returns cudaErrorNotSupported when the shape needs the SIMT path (caller falls through to launch_sgemm).
// max_split > 0 caps the K split; 1 gives every output tile a single writer (no reduce-adds: the same bits on every run).
inline cudaError_t launch_umma_gemm(const float* A, bool a_mn, long long lda, const float* B, bool b_mn, long long ldb,
                                    const float* bias, float* D, long long ldd, int M, int N, int K, int sms,
                                    cudaStream_t st, int max_split = 0) {
  if (M <= 0 || N <= 0 || K <= 0) return cudaSuccess;
  const bool aligned = (lda % 4 == 0) && (ldb % 4 == 0) && ((reinterpret_cast<uintptr_t>(A) & 15u) == 0) &&
                       ((reinterpret_cast<uintptr_t>(B) & 15u) == 0) && ((a_mn ? M : K) % 4 == 0) &&
                       ((b_mn ? N : K) % 4 == 0);
  if (!aligned || N < 64) return cudaErrorNotSupported;
  UmmaGemmParams p;
  p.A = A; p.lda = lda; p.B = B; p.ldb = ldb; p.bias = bias; p.D = D; p.ldd = ldd;
  p.M = M; p.N = N; p.K = K;
  p.tiles_m = (M + 127) / 128; p.tiles_n = (N + 255) / 256; p.nkb = (K + 63) / 64;
  const int ntiles = p.tiles_m * p.tiles_n;
  // split K when the tiles alone cannot fill the machine; keep at least 2 k-blocks per partition
  int ks = 1;
  if (ntiles < sms) {
    ks = sms / ntiles;
    const int kmax = p.nkb / 2 > 1 ? p.nkb / 2 : 1;
    if (ks > kmax) ks = kmax;
    if (max_split > 0 && ks > max_split) ks = max_split;
    if (ks < 1) ks = 1;
  }
  p.ksplit = ks;
  p.nwork = ntiles * ks;
  const int grid = p.nwork < sms ? p.nwork : sms;
  cudaError_t e;
  if (ks > 1) {
    e = cudaMemset2DAsync(D, (size_t)ldd * 4, 0, (size_t)N * 4, (size_t)M, st);
    if (e != cudaSuccess) return e;
  }
#define GH_UG(AM, BM)                                                                                                  \
  {                                                                                                                    \
    e = cudaFuncSetAttribute(umma_gemm_kernel<AM, BM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kUgSmemBytes); \
    if (e != cudaSuccess) return e;                                                                                    \
    umma_gemm_kernel<AM, BM><<<grid, kUgThreads, kUgSmemBytes, st>>>(p);                                               \
  }
  if (!a_mn && !b_mn) GH_UG(false, false)
  else if (!a_mn && b_mn) GH_UG(false, true)
  else if (a_mn && !b_mn) GH_UG(true, false)
  else GH_UG(true, true)
#undef GH_UG
  return cudaGetLastError();
}

}  // namespace gh
