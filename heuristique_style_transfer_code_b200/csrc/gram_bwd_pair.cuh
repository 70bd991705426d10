// Gram backward on CTA pairs:  dF_b[c][x] = scale * sum_d M_b[c][d] F_b[d][x],   M = dG + dG^T  (C x C, symmetric).
//
// Autograd of reference Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:26-30 (bmm + div) and :51-52
// (adaptive_avg_pool2d), driven by loss.backward() at functions/functions_RESNET50_Truncate_Gram_Attention.py:135.
//
// One cluster of two CTAs (one TPC) produces a 256-channel x NT-position tile of dF per unit with
// tcgen05.mma.cta_group::2 (M = 256, N = NT <= 256):
//   A = M   [256 c][K d]   K-major SWIZZLE_128B; each CTA GENERATES its 128 rows in shared memory from the image's
//                          g x g descriptor gradient (POOL: M[c][d] = dP[c/k][d/k] + dP[d/k][c/k], block-constant) or
//                          from the dense dG (DENSE), so dG never exists in HBM on the classification path
//   B = F   [K d][NT x]    MN-major SWIZZLE_128B: rows of F are contiguous along x, which is the canonical MN-major
//                          layout, so the feature map is TMA-staged exactly as cuDNN left it (fp32 -> kind::tf32,
//                          bf16 -> kind::f16): no cast pass, no register staging; each CTA loads its NT/2 columns
//   D = dF  [128 c][NT x]  per CTA in TMEM, two accumulator buffers: the epilogue of unit i overlaps the MMAs of i+1
//   epilogue: tcgen05.ld (lane = channel, 32 positions) -> *scale -> swizzled staging tile -> TMA store, so the
//             4 B/element gradient leaves the SM as full 128 B lines without occupying the LSU
// Warps: 0 and 22 = TMA producers (even / odd K chunks), 1 = TMEM owner + MMA issuer (leader CTA only), 2-5 and 23-26 =
// epilogue (two sets of four: even / odd 32-column chunks),
// 6-21 = A-tile generators in four groups of four warps; group i generates the K chunks n = i mod 4 (into A-ring stage
// n mod 5), so four chunks are generated concurrently and the per-chunk handshake (mbarrier wait, proxy fence, arrive)
// of one group overlaps the stores of the others. A and B tiles travel in separate rings: 5 stages of generated A, 5 stages (80 KB) of TMA-loaded F, 3 store
// staging tiles per epilogue warp -- the best of the depth sweep in profiles/ (6 B stages are faster for C >= 512 but
// 20 % slower on the HBM-bound C = 256 stage).
#pragma once
#include "pair.cuh"
#include "gram_fwd.cuh"   // GramMode

namespace gh {

// Two rings. The generated A tiles have a short refill round trip (commit -> empty -> 8 stores -> proxy fence -> remote
// arrive, well under a microsecond), the F tiles come from HBM / L2 with 1-2 us of loaded latency: bytes in flight =
// bandwidth x latency, so the B ring is as deep as shared memory allows and the A ring only as deep as it must be.
#ifndef GH_BP_STORE_BUFS
#define GH_BP_STORE_BUFS 2
#endif
// Ring depths are launch parameters (GramBwdPairParams::a_stages / b_stages): a_stages A tiles of 16 KB and as many F
// stages of b_stage_bytes (the x-tile width decides) as fit in the remaining kBpRingTiles - a_stages tiles. The F tiles
// of the C >= 512 stages come mostly from L2 and want the ring as deep as shared memory allows (bytes in flight =
// bandwidth x latency). Measured and rejected (profiles/r2_gram_bwd_experiments.md): ONE ring with a single full / empty
// barrier pair per slot (halves the MMA issuer's waits and commits per chunk, but leaves only 4-5 slots: 5-17 % slower).
// a_stages >= the number of stage lanes (4 generator groups / CH chunks per stage, CH = 1 in the shared-memory form):
// a group produces the stages n = lane (mod lanes); its next stage n + lanes reuses the slot of stage n + lanes -
// a_stages. Before it started stage n it waited for the MMAs of stage n - a_stages, so everything up to there has been
// consumed; with a_stages >= lanes that covers stage n + lanes - 2 * a_stages, the slot's last-but-one occupant: the
// waiter is at most ONE phase ahead of the slot's `empty` barrier. With fewer stages it could be two phases ahead and
// pass on the aliased parity (seen as a deadlock, caught by the bounded waits, when a 3-stage ring was tried).
constexpr int kBpRingTiles = 9;                             // A stages + F tiles, in 16 KB tiles
constexpr int kBpMaxStages = 12;                            // per ring (sizes the barrier arrays)
constexpr uint32_t kBpTileBytes = 16384;                    // A: [128 c][128 B]; B: <= 128 x-columns x (K chunk) x elem
constexpr int kBpStoreBufs = GH_BP_STORE_BUFS;              // staging tiles per epilogue warp = TMA stores it keeps in flight
constexpr int kBpEpiWarps = 8;                              // two sets of four (one warp per TMEM lane quarter): set s drains
                                                            // the 32-column chunks s, s + 2, ... of a unit's accumulator
constexpr uint32_t kBpStoreBytes = kBpEpiWarps * kBpStoreBufs * 4096; // per epilogue warp: kBpStoreBufs [32 c][32 x] fp32 staging tiles
constexpr int kBpMaxG = 32;                                 // pooled size handled here (larger g: the ldg kernels)
constexpr int kBpGroups = 4;                                // generator groups (four warps each); group i generates chunks n = i mod 4
constexpr int kBpTableFloats = kBpMaxG * kBpMaxG + kBpMaxG; // g x g table + one row of zeros (rows beyond C)
constexpr uint32_t kBpSymBytes = 2 * kBpTableFloats * 4;    // current and next image's table, shared by the groups
constexpr uint32_t kBpSmemBytes = kBpRingTiles * kBpTileBytes + kBpStoreBytes + kBpSymBytes + 1024 + 512;
constexpr int kBpGroupThreads = 128;                        // one thread per A row
constexpr int kBpGenThreads = kBpGroups * kBpGroupThreads;
constexpr int kBpProducer2Warp = 6 + kBpGenThreads / 32;    // second TMA producer warp
constexpr int kBpEpi2Warp0 = kBpProducer2Warp + 1;          // second set of epilogue warps: 23..26 (23 & 3 = 3, 24 & 3 = 0, ...)
constexpr int kBpThreads = (kBpEpi2Warp0 + 4) * 32;
static_assert(kBpSmemBytes <= 232448, "gram_bwd_pair: shared memory budget");

struct GramBwdPairParams {
  int B, C, HW;
  int mode;                 // GRAM_POOL / GRAM_DENSE
  const float* dP;          // POOL: (B, L, g*g) slice base of this stage
  long long dp_img_stride;
  int g, kshift;
  const float* dG;          // DENSE: (B, C, C)
  float scale;
  int NT;                   // x-tile width of a pair (multiple of 32, <= 256); each CTA supplies NT/2 columns of B
  int nHT, nCB;             // x tiles, 256-channel output blocks
  int nkc;                  // K stages per unit: CH chunks of 32 (tf32) / 64 (bf16) input channels each
  int total_units;
  int areuse;               // POOL: consecutive k-steps of a chunk whose A data is identical (1, 2 or 4), see below
  int a_stages, b_stages;   // ring depths (A: generated gradient tiles, B: TMA-loaded F tiles)
  int b_stage_bytes;        // bytes of one F stage (a multiple of 1024): the F ring takes the (kBpRingTiles - a_stages)
                            // tiles the A ring leaves, cut into stages of the size the x-tile width needs
  int df_bf16;              // 1: dF leaves as bf16 (tmD is a bf16 map, 64 B swizzle): half the gradient bytes, and the
                            //    gradient a bf16 backbone wants (SURVEY 8(f) n1); 0: fp32
  int a_smem_tiles;         // 16 KB tiles the generated-A ring occupies in shared memory: a_stages, or 0 when the A
                            // operand lives in tensor memory (ATS kernels: the whole ring then belongs to F)
  int a_tmem_cols;          // ATS: TMEM columns of one A stage = CH * 32 / areuse (only the k-steps that differ are stored)
  int d_stride;             // TMEM columns between the two accumulators: 256, or NT rounded up to 32 in the ATS kernels,
  int a_tmem_base;          // whose A ring takes the columns from 2 * d_stride on: stage s at a_tmem_base + s * a_tmem_cols
};

// -DGH_BP_PROFILE: per-role cycle accounting (clock64 around every mbarrier wait of one thread per role, summed over
// the CTAs into g_bp_prof and read back by gh_bp_profile_read) -- where each warp role of the kernel spends its time.
// Slots: 0 issuer loop, 1 issuer wait tmem_empty, 2 wait fullA, 3 wait fullB, 4 chunks issued, 5 epilogue (warp 2) loop,
// 6 wait tmem_full, 7 wait staging tile, 8 generator (warp 6) loop, 9 wait emptyA, 10 producer (warp 0) loop,
// 11 wait emptyB, 12 leader CTAs counted.
#ifdef GH_BP_PROFILE
__device__ unsigned long long g_bp_prof[16];
#define GH_BP_CLK(var) const long long var = clock64()
#define GH_BP_ADD(acc, var) acc += clock64() - var
#define GH_BP_FLUSH(slot, acc) atomicAdd(&g_bp_prof[slot], (unsigned long long)(acc))
#else
#define GH_BP_CLK(var)
#define GH_BP_ADD(acc, var)
#define GH_BP_FLUSH(slot, acc)
#endif

struct GramBwdPairUnit {
  int b, ht, cb;
};
__device__ __forceinline__ GramBwdPairUnit gbp_decode(const GramBwdPairParams& p, int u) {
  GramBwdPairUnit w;
  w.cb = u % p.nCB;
  const int t = u / p.nCB;
  w.ht = t % p.nHT;
  w.b = t / p.nHT;
  return w;
}

__device__ __forceinline__ uint32_t f32_to_tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}

// MODE: GRAM_POOL (A generated from the g x g descriptor gradient) or GRAM_DENSE (A = dG + dG^T read from HBM).
// NHWC = false: F and dF with x contiguous (NCHW): F is the MN-major B operand, dF leaves as [channel rows][32 x] tiles.
// NHWC = true : channels_last F and dF (c contiguous): F[d][x] at x*C + d is K-contiguous, i.e. a K-major B operand
//               [NT/2 position rows][128 B of input channels] fetched by ONE box per chunk; the epilogue transposes
//               through the staging tile ([32 x rows][32 channels]) so that dF is stored NHWC too.
// ATS  = true : (POOL only) the generated gradient tile is written to TENSOR MEMORY (tcgen05.st) and the MMAs take their
//               A operand from there (UTCHMMA tmem, gdesc). Why: per unit the SS form moves through shared memory the A
//               tile twice (generator stores + the tensor core's operand fetch, 4 KB per MMA and CTA whatever N is)
//               on top of the F tiles (TMA write + operand fetch) and the gradient staging (write + TMA read) --
//               872 KB per C = 512 unit against 5 120 cycles of MMAs, i.e. more than the ~90 B/clk the kernels of this
//               library are seen to sustain; with A in TMEM it is 488 KB. The two accumulators sit d_stride = NT (rounded
//               up to 32) columns apart and the A ring takes the columns behind them: stage s at a_tmem_base +
//               s * a_tmem_cols. (Measured: the shared-memory traffic was NOT the limit -- same speed with one chunk per
//               stage; what the TMEM operand buys is room for CH > 1, below.)
// CH          : K chunks (128 B operand rows: 32 tf32 / 64 bf16 input channels) per ring stage. The single thread that
//               issues the MMAs needs ~570 cycles per loop iteration (two mbarrier waits, descriptor arithmetic moved to
//               uniform registers, 4 UTCHMMA, 2-3 UTCBAR -- measured with -DGH_BP_PROFILE: ~185 of them in waits that pass
//               at once), while the four MMAs of a chunk execute in 320 (N = 160) to 448 cycles: with one chunk per
//               stage the ISSUER paces the C >= 512 stages (tensor pipe 57 % active). CH = 2 (ATS only: a doubled A
//               stage fits TMEM, not shared memory) issues eight MMAs per iteration, CH = 4 sixteen. The four generator
//               groups then share a stage: group i writes chunk i % CH of the stages n = i / CH (mod 4 / CH); a_stages
//               >= 4 / CH keeps every waiter at most one phase ahead of its barrier (see kBpRingTiles above).
//               CH = 4 was measured too: its 40 KB F stages leave a 3-deep ring and it loses to CH = 2.
template <int KIND, int MODE, bool NHWC, bool ATS = false, int CH = 1>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kBpThreads, 1)
    gram_bwd_pair_kernel(const GramBwdPairParams p, const __grid_constant__ CUtensorMap tmF,
                         const __grid_constant__ CUtensorMap tmD) {
  static_assert(CH == 1 || ((CH == 2 || CH == 4) && ATS), "a multi-chunk stage needs the A operand in tensor memory");
  using T = KindTraits<KIND>;
  constexpr uint32_t KC = T::kElemsPerRow;                  // input channels per K chunk
  constexpr uint32_t kAtomBytesB = KC * kRowBytes;          // one 128 B-wide x block of the B tile: 4 KB | 8 KB
  constexpr uint32_t kStepBytesB = (T::kUmmaK / 8) * 1024;  // B advance per MMA: K/8 groups of 8 K-rows

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t kBpAStages = (uint32_t)p.a_stages, kBpBStages = (uint32_t)p.b_stages;   // launch parameters
  const uint32_t a_ring = smem_base;                                        // a_stages x 16 KB
  const uint32_t b_ring = a_ring + (uint32_t)p.a_smem_tiles * kBpTileBytes; // b_stages x b_stage_bytes
  const uint32_t store_smem = smem_base + kBpRingTiles * kBpTileBytes;
  const uint32_t sym_smem = store_smem + kBpStoreBytes;
  float* sym = reinterpret_cast<float*>(smem_raw + (sym_smem - smem_u32(smem_raw)));
  const uint32_t bars = sym_smem + kBpSymBytes;
  const uint32_t bar_fullA = bars, bar_emptyA = bar_fullA + 8 * kBpMaxStages;
  const uint32_t bar_fullB = bar_emptyA + 8 * kBpMaxStages, bar_emptyB = bar_fullB + 8 * kBpMaxStages;
  const uint32_t bar_tfull = bar_emptyB + 8 * kBpMaxStages, bar_tempty = bar_tfull + 16;
  const uint32_t tmem_slot = bar_tempty + 16;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = (int)cluster_id_x(), npairs = (int)cluster_nclusters_x();
  // Every pair walks a CONTIGUOUS range of units: consecutive units then belong to the same image (nHT * nCB units per
  // image), so the generators switch gradient tables -- and synchronise among themselves -- only when the image changes,
  // and the two channel blocks of an x tile read the same F tiles back to back (the second time from L2).
  const int u_begin = (int)(((long long)p.total_units * pair) / npairs);
  const int u_end = (int)(((long long)p.total_units * (pair + 1)) / npairs);

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmF);
    tma_prefetch_desc(&tmD);
    for (uint32_t s = 0; s < kBpAStages; ++s) {
      mbar_init(bar_fullA + 8 * s, 2 * CH * (kBpGroupThreads / 32));   // the stage's generator warps of both CTAs
      mbar_init(bar_emptyA + 8 * s, 1);                           // multicast tcgen05.commit
    }
    for (uint32_t s = 0; s < kBpBStages; ++s) {
      mbar_init(bar_fullB + 8 * s, 1);                            // leader's expect_tx; both CTAs' TMA bytes land on it
      mbar_init(bar_emptyB + 8 * s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_tfull + 8 * a, 1);
      mbar_init(bar_tempty + 8 * a, 2 * kBpEpiWarps);              // 8 epilogue warps x 2 CTAs
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc2(tmem_slot, 512);
  tc_fence_before_sync();
  cluster_sync_all();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const uint32_t fullA_leader = mapa_u32(bar_fullA, 0);    // shared::cluster addresses of the leader's barriers
  const uint32_t fullB_leader = mapa_u32(bar_fullB, 0);
  const uint32_t tempty_leader = mapa_u32(bar_tempty, 0);
  const int na = (p.NT / 2 + (int)KC - 1) / (int)KC;       // 128 B-wide x blocks each CTA loads per K chunk
  // One thread per warp issues the TMA / tcgen05 instructions; elect.sync (not `lane == 0`) lets ptxas feed their
  // uniform-register operands directly instead of wrapping each one in an elect-broadcast-retry loop (gram_fwd_pair.cuh).
  const bool elected = elect_one();

  if (warp == 0 || warp == kBpProducer2Warp) {
    // =========================== TMA producers: this CTA's NT/2 columns of F ===========================
    // Two warps, even and odd K chunks (even and odd B stages): per chunk a producer spends a few hundred cycles on
    // the mbarrier round trip and on issuing 3-4 tile loads, about as long as the chunk's MMAs take to execute.
    const uint32_t pidx = (warp == 0) ? 0u : 1u;
    if (elected) {
      uint32_t n = 0;
      [[maybe_unused]] long long prof_wait = 0;
      GH_BP_CLK(prof_t0);
      const uint32_t sub_tx = NHWC ? 2u * (uint32_t)(p.NT / 2) * kRowBytes : 2u * (uint32_t)na * kAtomBytesB;
      const uint32_t sub_bytes = (uint32_t)p.b_stage_bytes / (uint32_t)CH;      // one chunk's F tile inside a stage
      const int nsub_total = (p.C + (int)KC - 1) / (int)KC;                     // chunks that hold any channel < C
      for (int u = u_begin; u < u_end; ++u) {
        const GramBwdPairUnit w = gbp_decode(p, u);
        const int x0 = w.ht * p.NT + (int)rank * (p.NT / 2);
        for (int kc = 0; kc < p.nkc; ++kc, ++n) {
          if ((n & 1u) != pidx) continue;
          const uint32_t stage = n % (uint32_t)kBpBStages, phase = (n / (uint32_t)kBpBStages) & 1u;
          GH_BP_CLK(prof_w);
          mbar_wait(bar_emptyB + 8 * stage, phase ^ 1u, 100u + stage);
          GH_BP_ADD(prof_wait, prof_w);
          const int nsub = (kc * CH + CH <= nsub_total) ? CH : nsub_total - kc * CH;   // chunks of this stage in range
          if (rank == 0) mbar_arrive_expect_tx(bar_fullB + 8 * stage, (uint32_t)nsub * sub_tx);
#pragma unroll
          for (int sc = 0; sc < CH; ++sc) {
            if (sc >= nsub) break;
            const uint32_t b_tile = b_ring + stage * (uint32_t)p.b_stage_bytes + (uint32_t)sc * sub_bytes;
            const int ch0 = (kc * CH + sc) * (int)KC;
            if constexpr (NHWC) {
              tma_load_3d_pair(b_tile, &tmF, fullB_leader + 8 * stage, ch0, x0, w.b);
            } else {
              for (int j = 0; j < na; ++j)
                tma_load_3d_pair(b_tile + (uint32_t)j * kAtomBytesB, &tmF, fullB_leader + 8 * stage, x0 + j * (int)KC, ch0,
                                 w.b);
            }
          }
        }
      }
#ifdef GH_BP_PROFILE
      if (warp == 0 && rank == 0) {
        [[maybe_unused]] long long prof_tot = 0;
        GH_BP_ADD(prof_tot, prof_t0);
        GH_BP_FLUSH(10, prof_tot);
        GH_BP_FLUSH(11, prof_wait);
      }
#endif
    }
    __syncwarp();
  } else if (warp == 1) {
    // =========================== MMA issuer (one thread of the leader CTA) ===========================
    // The loop body is kept to a few dozen instructions: descriptors are a per-ring constant plus small increments
    // (stage * 1024 and k-step * 2 / * 64|128 in 16 B units), a full chunk issues its four MMAs without bound checks.
    // A single thread executes ~10 cycles per dependent instruction; at ~300 instructions per chunk (first version)
    // the issuer, not the tensor pipe, set the pace of the C >= 512 stages.
    if (rank == 0 && elected) {
      const uint32_t idesc = make_idesc(T::kFormat, 256, (uint32_t)p.NT, 0, NHWC ? 0 : 1);
      const uint64_t dA0 = make_smem_desc_sw128(a_ring);
      const uint64_t dB0 = NHWC ? make_smem_desc_sw128(b_ring)
                                : (KIND == KIND_TF32 ? make_smem_desc_sw128b32_mnmajor(b_ring, kAtomBytesB)
                                                     : make_smem_desc_sw128_mnmajor(b_ring, kAtomBytesB));
      constexpr uint64_t kStageInc = kBpTileBytes >> 4, kAInc = 32u >> 4, kBInc = NHWC ? 32u >> 4 : kStepBytesB >> 4;
      const uint64_t kStageIncB = (uint64_t)p.b_stage_bytes >> 4;
      const int full_chunks = p.C / (int)KC;
      const uint32_t amask = (MODE == GRAM_POOL) ? (~((uint32_t)p.areuse - 1u) & 3u) : 3u;
      const uint64_t a1 = (1u & amask) * kAInc, a2 = (2u & amask) * kAInc, a3 = (3u & amask) * kAInc;
      const uint32_t ashift = p.areuse >= 4 ? 2u : (p.areuse == 2 ? 1u : 0u);         // ATS: log2(areuse)
      const uint32_t t1 = 8u * (1u >> ashift), t2 = 8u * (2u >> ashift), t3 = 8u * (3u >> ashift);
      const uint32_t sub_cols = (uint32_t)p.a_tmem_cols / (uint32_t)CH;               // ATS: TMEM columns of one chunk
      const uint64_t kSubIncB = ((uint64_t)p.b_stage_bytes / (uint64_t)CH) >> 4;      // one chunk's F tile inside a stage
      uint32_t sa = 0, pa = 0, sb = 0, pb = 0, it = 0;
      [[maybe_unused]] long long prof_te = 0, prof_fa = 0, prof_fb = 0, prof_n = 0;
      GH_BP_CLK(prof_t0);
      for (int u = u_begin; u < u_end; ++u, ++it) {
        const uint32_t ab = it & 1u, use = it >> 1;
        GH_BP_CLK(prof_w0);
        mbar_wait_cl(bar_tempty + 8 * ab, (use & 1u) ^ 1u, 200u + ab);
        GH_BP_ADD(prof_te, prof_w0);
        tc_fence_after_sync();
        const uint32_t acc = tmem_base + ab * (uint32_t)p.d_stride;
        for (int kc = 0; kc < p.nkc; ++kc) {
          GH_BP_CLK(prof_w1);
          mbar_wait_cl(bar_fullA + 8 * sa, pa, 300u + sa);
          GH_BP_ADD(prof_fa, prof_w1);
          GH_BP_CLK(prof_w2);
          mbar_wait_cl(bar_fullB + 8 * sb, pb, 320u + sb);
          GH_BP_ADD(prof_fb, prof_w2);
#ifdef GH_BP_PROFILE
          ++prof_n;
#endif
          tc_fence_after_sync();
          const uint64_t da = dA0 + sa * kStageInc, db = dB0 + sb * kStageIncB;
          if constexpr (ATS) {
            // A from tensor memory: k-step ks of chunk sc reads the 8 columns of generated k-step ks / areuse
            const uint32_t ta0 = tmem_base + (uint32_t)p.a_tmem_base + sa * (uint32_t)p.a_tmem_cols;
#pragma unroll
            for (int sc = 0; sc < CH; ++sc) {
              const int ch = kc * CH + sc;                                     // chunk index within the unit
              const uint32_t ta = ta0 + (uint32_t)sc * sub_cols;
              const uint64_t dbs = db + (uint64_t)sc * kSubIncB;
              if (ch < full_chunks) {
                umma2_ts<KIND>(acc, ta, dbs, idesc, ch != 0 ? 1u : 0u);
                umma2_ts<KIND>(acc, ta + t1, dbs + kBInc, idesc, 1u);
                umma2_ts<KIND>(acc, ta + t2, dbs + 2 * kBInc, idesc, 1u);
                umma2_ts<KIND>(acc, ta + t3, dbs + 3 * kBInc, idesc, 1u);
              } else {
                for (uint32_t ks = 0; ks < KC / T::kUmmaK; ++ks) {
                  if ((int)(ch * KC + ks * T::kUmmaK) >= p.C) break;
                  umma2_ts<KIND>(acc, ta + 8u * (ks >> ashift), dbs + ks * kBInc, idesc, (uint32_t)ch | ks);
                }
              }
            }
          } else
          // k-step ks reads the A data of k-step (ks & amask): with a pooling factor k >= 2 * UMMA_K the generated rows
          // repeat across k-steps, so only the first k-step of each run is generated (a1..a3 = 0/0/0, 1/2/2 or 1/2/3)
          if (kc < full_chunks) {
            umma2<KIND>(acc, da, db, idesc, kc != 0 ? 1u : 0u);
            umma2<KIND>(acc, da + a1, db + kBInc, idesc, 1u);
            umma2<KIND>(acc, da + a2, db + 2 * kBInc, idesc, 1u);
            umma2<KIND>(acc, da + a3, db + 3 * kBInc, idesc, 1u);
          } else {
            for (uint32_t ks = 0; ks < KC / T::kUmmaK; ++ks) {
              if ((int)(kc * KC + ks * T::kUmmaK) >= p.C) break;
              umma2<KIND>(acc, da + (ks & amask) * kAInc, db + ks * kBInc, idesc, (uint32_t)kc | ks);
            }
          }
          umma_commit2(bar_emptyA + 8 * sa);
          umma_commit2(bar_emptyB + 8 * sb);
          if (kc + 1 == p.nkc) umma_commit2(bar_tfull + 8 * ab);
          if (++sa == kBpAStages) { sa = 0; pa ^= 1u; }
          if (++sb == kBpBStages) { sb = 0; pb ^= 1u; }
        }
      }
#ifdef GH_BP_PROFILE
      {
        long long prof_tot = 0;
        GH_BP_ADD(prof_tot, prof_t0);
        GH_BP_FLUSH(0, prof_tot);
        GH_BP_FLUSH(1, prof_te);
        GH_BP_FLUSH(2, prof_fa);
        GH_BP_FLUSH(3, prof_fb);
        GH_BP_FLUSH(4, prof_n);
        GH_BP_FLUSH(12, 1);
      }
#endif
    }
    __syncwarp();
  } else if (warp < 6 || warp >= kBpEpi2Warp0) {
    // =========================== epilogue: TMEM -> scale -> staging -> TMA store ===========================
    // Eight warps: with four, draining a 128 x 160 accumulator took about as long as the 5 120 cycles of MMAs of a
    // C = 512 unit and the tensor pipe idled 40 % of the time (profiles/r2_bwd512_ncu_summary.txt).
    const int q = warp & 3;                                 // TMEM lane quarter this warp may read
    const int eset = warp < 6 ? 0 : 1;                      // which half of the 32-column chunks
    const int eidx = warp < 6 ? warp - 2 : 4 + (warp - kBpEpi2Warp0);
    const uint32_t my_store = store_smem + (uint32_t)eidx * (kBpStoreBufs * 4096u);
    uint32_t it = 0, buf = 0;
    [[maybe_unused]] long long prof_tf = 0, prof_sb = 0;
    GH_BP_CLK(prof_t0);
    for (int u = u_begin; u < u_end; ++u, ++it) {
      const GramBwdPairUnit w = gbp_decode(p, u);
      const uint32_t ab = it & 1u, use = it >> 1;
      GH_BP_CLK(prof_w0);
      mbar_wait(bar_tfull + 8 * ab, use & 1u, 400u + ab);
      GH_BP_ADD(prof_tf, prof_w0);
      tc_fence_after_sync();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + ab * (uint32_t)p.d_stride;
      const int crow0 = w.cb * 256 + (int)rank * 128 + q * 32;
#pragma unroll 1
      for (int n0 = 32 * eset; n0 < p.NT; n0 += 64) {
        const int x = w.ht * p.NT + n0;
        if (x >= p.HW) break;                               // warp-uniform
        float v[32];
        tmem_ld32(taddr + (uint32_t)n0, v);
        GH_BP_CLK(prof_w1);
        if (elected) tma_store_wait_read<kBpStoreBufs - 1>();     // the staging tile about to be reused has been read
        __syncwarp();
        GH_BP_ADD(prof_sb, prof_w1);
        if (p.df_bf16) {
          // bf16 gradient: 64 B rows, SWIZZLE_64B (16 B chunk c of row r sits at chunk c ^ ((r >> 1) & 3))
          if constexpr (NHWC) {
            // [32 x rows][32 channels]: lane (= channel) writes element `lane` of every row
            const uint32_t tile = my_store + buf * 4096u + (((uint32_t)lane & 7u) << 1);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const uint32_t addr = tile + (uint32_t)j * 64u + (((((uint32_t)lane >> 3) ^ (((uint32_t)j >> 1) & 3u))) << 4);
              const __nv_bfloat16 h = __float2bfloat16_rn(v[j] * p.scale);
              asm volatile("st.shared.b16 [%0], %1;" ::"r"(addr), "h"(*reinterpret_cast<const unsigned short*>(&h)) : "memory");
            }
          } else {
            // [32 channel rows][32 x]: lane (= channel) writes its row as four 16 B chunks
            const uint32_t tile = my_store + buf * 4096u + (uint32_t)lane * 64u, sw64 = ((uint32_t)lane >> 1) & 3u;
#pragma unroll
            for (int c = 0; c < 4; ++c)
              sts_u4(tile + ((((uint32_t)c) ^ sw64) << 4), pack_bf16x2(v[8 * c] * p.scale, v[8 * c + 1] * p.scale),
                     pack_bf16x2(v[8 * c + 2] * p.scale, v[8 * c + 3] * p.scale),
                     pack_bf16x2(v[8 * c + 4] * p.scale, v[8 * c + 5] * p.scale),
                     pack_bf16x2(v[8 * c + 6] * p.scale, v[8 * c + 7] * p.scale));
          }
        } else if constexpr (NHWC) {
          // staging tile = [32 x rows][32 channels]: lane (= channel) writes column `lane` of every row; one row is 32
          // consecutive words across the warp (16 B chunks XOR-swizzled by the row), so the stores are conflict-free
          const uint32_t tile = my_store + buf * 4096u + (((uint32_t)lane & 3u) << 2);
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const uint32_t addr = tile + (uint32_t)j * kRowBytes + (((((uint32_t)lane >> 2) ^ ((uint32_t)j & 7u))) << 4);
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(__float_as_uint(v[j] * p.scale)) : "memory");
          }
        } else {
          const uint32_t tile = my_store + buf * 4096u + (uint32_t)lane * kRowBytes;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            sts_u4(tile + ((((uint32_t)j) ^ ((uint32_t)lane & 7u)) << 4), __float_as_uint(v[4 * j] * p.scale),
                   __float_as_uint(v[4 * j + 1] * p.scale), __float_as_uint(v[4 * j + 2] * p.scale),
                   __float_as_uint(v[4 * j + 3] * p.scale));
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (elected && crow0 < p.C) {
          if constexpr (NHWC) tma_store_3d(&tmD, my_store + buf * 4096u, crow0, x, w.b);
          else tma_store_3d(&tmD, my_store + buf * 4096u, x, crow0, w.b);
          tma_store_commit();
        }
        buf = (buf + 1u) % kBpStoreBufs;
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty_leader + 8 * ab);
    }
#ifdef GH_BP_PROFILE
    if (warp == 2 && rank == 0 && lane == 0) {
      long long prof_tot = 0;
      GH_BP_ADD(prof_tot, prof_t0);
      GH_BP_FLUSH(5, prof_tot);
      GH_BP_FLUSH(6, prof_tf);
      GH_BP_FLUSH(7, prof_sb);
    }
#endif
    if (elected) tma_store_wait_all<0>();
    __syncwarp();
  } else {
    // =========================== A-tile generators: this CTA's 128 rows of M ===========================
    // Group grp fills chunk grp % CH of the stages n = unit_index * nkc + kc with n % (4 / CH) == grp / CH. Thread = A row.
    // POOL: every 16 B chunk of the row is one value of the per-image table sym = dP + dP^T repeated (the pooling
    // factor k is >= the elements of a chunk): 8 shared loads, 8 conversions and 8 16 B stores per K chunk. The
    // table of the NEXT unit's image is fetched into registers (all 512 generator threads share the work) while the
    // current unit is generated, and published through the second table buffer at the unit boundary.
    constexpr int EPC = 16 / (int)T::kElemBytes;            // elements per 16 B chunk: 4 (tf32) / 8 (bf16)
    constexpr int NE = kBpMaxG * kBpMaxG / kBpGenThreads;   // table entries per generator thread
    const int grp = (warp - 6) / (kBpGroupThreads / 32);
    constexpr int kLanes = kBpGroups / CH;                  // groups sharing a stage: CH; stage lanes: 4 / CH
    const int glane = grp / CH, gsub = grp % CH;            // this group: chunk gsub of the stages n = glane (mod kLanes)
    const int gall = threadIdx.x - 6 * 32;                  // 0..511 among all generator threads
    // thread = A row. SS: any assignment works (0..127 in thread order); ATS: a warp can only write the TMEM lanes of
    // its quarter (warp & 3), so the row is that quarter's lane
    const int gt = ATS ? ((warp & 3) * 32 + lane) : (gall - grp * kBpGroupThreads);
    const uint32_t row = (uint32_t)gt, sw = row & 7u;
    const uint32_t row_off = (row >> 3) * kAtomBytes + sw * kRowBytes;
    const int gg = p.g * p.g;
    float* table = sym;
    float pre_a[NE], pre_b[NE];                             // dP[i][j] and dP[j][i]: added only when published, so the
    auto fetch_table = [&](int b) {                         // loads stay in flight while the current unit is generated
      const float* dp = p.dP + (long long)b * p.dp_img_stride;
#pragma unroll
      for (int e = 0; e < NE; ++e) {
        const int i = gall + e * kBpGenThreads;
        pre_a[e] = 0.f;
        pre_b[e] = 0.f;
        if (i < gg) {
          const int r = i / p.g, cc = i - r * p.g;
          pre_a[e] = __ldg(dp + i);
          pre_b[e] = __ldg(dp + cc * p.g + r);
        }
      }
    };
    auto publish_table = [&](int which) {
#pragma unroll
      for (int e = 0; e < NE; ++e) {
        const int i = gall + e * kBpGenThreads;
        if (i < gg) table[which * kBpTableFloats + i] = pre_a[e] + pre_b[e];
      }
    };
    int cur = 0;
    if (MODE == GRAM_POOL) {
      if (gall < kBpMaxG) {                                 // the zero rows
        table[gg + gall] = 0.f;
        table[kBpTableFloats + gg + gall] = 0.f;
      }
      if (u_begin < u_end) {
        fetch_table(gbp_decode(p, u_begin).b);
        publish_table(0);
      }
      named_bar_sync(1, kBpGenThreads);
    }
    int n0 = 0;                                             // sequence number of the unit's first K chunk
    [[maybe_unused]] long long prof_ea = 0;
    GH_BP_CLK(prof_t0);
    for (int u = u_begin; u < u_end; ++u, n0 += p.nkc) {
      const GramBwdPairUnit w = gbp_decode(p, u);
      // the table changes only when the next unit belongs to another image
      const bool switch_table = MODE == GRAM_POOL && u + 1 < u_end && gbp_decode(p, u + 1).b != w.b;
      if (switch_table) fetch_table(gbp_decode(p, u + 1).b);
      const int c = w.cb * 256 + (int)rank * 128 + (int)row;
      const bool row_ok = c < p.C;
      const float* srow = table + cur * kBpTableFloats + (row_ok ? (c >> p.kshift) * p.g : gg);
      for (int kc = (glane - (n0 & (kLanes - 1)) + kLanes) & (kLanes - 1); kc < p.nkc; kc += kLanes) {
        const uint32_t n = (uint32_t)(n0 + kc);
        const uint32_t stage = n % (uint32_t)kBpAStages, phase = (n / (uint32_t)kBpAStages) & 1u;
        GH_BP_CLK(prof_w0);
        mbar_wait(bar_emptyA + 8 * stage, phase ^ 1u, 500u + stage);
        GH_BP_ADD(prof_ea, prof_w0);
        const uint32_t a_row = a_ring + stage * kBpTileBytes + row_off;
        const int dbase = kc * (int)KC;
        if constexpr (ATS) {
          // The same pieces as below (one table value per 16 B = 4 columns), written to this row's TMEM lane: 8 columns
          // per generated k-step, only the k-steps the MMAs read.
          tc_fence_after_sync();                            // the MMAs that read this stage have completed (emptyA)
          const uint32_t t_row = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)p.a_tmem_base +
                                 stage * (uint32_t)p.a_tmem_cols;
          const int jstep = 2 * p.areuse, nd = 4 / p.areuse;         // generated k-steps of a chunk: 4, 2 or 1
          const uint32_t col = (uint32_t)gsub * ((uint32_t)p.a_tmem_cols / (uint32_t)CH);
          const int dsub = (dbase * CH) + gsub * (int)KC;   // first channel of this group's chunk of the stage
          const bool full_chunk = dsub + (int)KC <= p.C;
          uint32_t t[8];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
#pragma unroll
            for (int jj = 0; jj < 2; ++jj) {
              const int d0 = dsub + (i * jstep + jj) * EPC;
              const float v = (i < nd && (full_chunk || d0 < p.C)) ? srow[d0 >> p.kshift] : 0.f;
              t[2 * i + jj] = (KIND == KIND_TF32) ? f32_to_tf32_rna(v) : pack_bf16x2(v, v);
            }
          }
          if (nd == 4) tmem_st32_pairs(t_row + col, t);
          else if (nd == 2) tmem_st16_pairs(t_row + col, t);
          else tmem_st8_pairs(t_row + col, t[0], t[1]);
          tmem_st_wait();
          tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(fullA_leader + 8 * stage);
          continue;
        }
        if (MODE == GRAM_POOL) {
          // A k-step is two 16 B chunks of the row. Only the k-steps the MMAs read are written: all four when the
          // pooling factor equals UMMA_K, every second one / the first one when it is 2x / >= 4x UMMA_K (p.areuse).
          const bool full_chunk = dbase + (int)KC <= p.C;
          const int jstep = 2 * p.areuse;
          for (int j0 = 0; j0 < 8; j0 += jstep) {
#pragma unroll
            for (int jj = 0; jj < 2; ++jj) {
              const int j = j0 + jj;
              const int d0 = dbase + j * EPC;
              const float v = (full_chunk || d0 < p.C) ? srow[d0 >> p.kshift] : 0.f;
              const uint32_t t = (KIND == KIND_TF32) ? f32_to_tf32_rna(v) : pack_bf16x2(v, v);
              sts_u4(a_row + ((((uint32_t)j) ^ sw) << 4), t, t, t, t);
            }
          }
        } else {
          const float* gb = p.dG + (long long)w.b * p.C * p.C;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int d0 = dbase + j * EPC;
            float x[EPC];
#pragma unroll
            for (int e = 0; e < EPC; ++e) {
              const int d = d0 + e;
              x[e] = (row_ok && d < p.C) ? (__ldg(gb + (long long)c * p.C + d) + __ldg(gb + (long long)d * p.C + c)) : 0.f;
            }
            const uint32_t addr = a_row + ((((uint32_t)j) ^ sw) << 4);
            if constexpr (KIND == KIND_TF32) {
              sts_u4(addr, f32_to_tf32_rna(x[0]), f32_to_tf32_rna(x[1]), f32_to_tf32_rna(x[2]), f32_to_tf32_rna(x[3]));
            } else {
              sts_u4(addr, pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]), pack_bf16x2(x[4], x[5]), pack_bf16x2(x[6], x[7]));
            }
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(fullA_leader + 8 * stage);
      }
      if (switch_table) {
        publish_table(cur ^ 1);                             // last read before the barrier of the previous switch
        named_bar_sync(1, kBpGenThreads);                   // every group sees the next table and is done with this one
        cur ^= 1;
      }
    }
#ifdef GH_BP_PROFILE
    if (warp == 6 && rank == 0 && lane == 0) {
      long long prof_tot = 0;
      GH_BP_ADD(prof_tot, prof_t0);
      GH_BP_FLUSH(8, prof_tot);
      GH_BP_FLUSH(9, prof_ea);
    }
#endif
  }

  __syncwarp();
  tc_fence_before_sync();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc2(tmem_base, 512);
  }
}

// x-tile plan: nHT tiles of NT (64 <= NT <= 256) covering HW with the least padded MMA work. NT is a multiple of 32 (the
// epilogue drains 32 columns at a time); a map that fits ONE tile may use a multiple of 16 (the MMA's N granularity):
// the half-filled last chunk then lies beyond HW, where the TMA store clips it (HW = 196 -> NT = 208 instead of 224).
inline void gbp_plan_tiles(int HW, int* NT, int* nHT) {
  int best_nt = 256, best_n = (HW + 255) / 256;
  long long best_cost = (long long)best_nt * best_n;
  const int n0 = (HW + 255) / 256;
  for (int n = n0; n <= n0 + 3; ++n) {
    int nt = ((HW + n - 1) / n + 31) / 32 * 32;
    if (n == 1) nt = (HW + 15) / 16 * 16;
    if (nt < 64) nt = 64;
    if (nt > 256) continue;
    const long long cost = (long long)nt * n;
    if (cost < best_cost) { best_cost = cost; best_nt = nt; best_n = n; }
  }
  *NT = best_nt;
  *nHT = best_n;
}

}  // namespace gh
