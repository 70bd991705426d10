// libgramhead.so - host launchers behind the C ABI in include/gramhead.h. One translation unit:
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -Xcompiler -fPIC -shared gramhead.cu -o libgramhead.so
#include "../../include/gramhead.h"
#include "common.cuh"
#include "gram_fwd.cuh"
#include "gram_fwd_pair.cuh"
#include "gram_bwd2.cuh"
#include "gram_bwd_pair.cuh"
#include "attn_head.cuh"
#include "umma_gemm.cuh"
#include "tgemm_pair.cuh"
#include "attn_head2.cuh"
#include "preprocess.cuh"
#include "transpose.cuh"
#include "patchgan.cuh"
#include "pool.cuh"
#include "stem.cuh"
#include "style_loss.cuh"
#include "jpeg.cuh"
#include <string>

namespace gh {

static int sm_count_cached() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
    error_record_host();       // every launcher passes here first: the device-side error record exists before any kernel runs
  }
  return cached[dev];
}

static int ilog2_exact(int v) {
  if (v <= 0 || (v & (v - 1))) return -1;
  int s = 0;
  while ((1 << s) < v) ++s;
  return s;
}

// K split of the Gram forward. Measured on B200 (profiles/r01*_kernel_timings.log): once there is at least one unit
// per CTA, splitting K only adds atomics and epilogues (C=512: 151 us unsplit vs 179 us split in two), so K is split
// only to fill the machine at small batch (camera mode: 1 image -> 1..10 units), keeping >= 2 k-blocks per part.
static int choose_ksplit(long long base_units, int nkb, int ctas, bool balance = false) {
  if (base_units >= ctas) {
    if (!balance) return 1;   // single-CTA kernel: its epilogue is not overlapped, a second one per unit costs more than it evens out
    // Whole units per worker leave the last round partly empty (256 images on 74 CTA pairs: 4 rounds for 3.46 rounds
    // of work). Two K halves per unit even that out, and two partial sums meeting in a zeroed fp32 slot add to the
    // same bits in either order, so the result stays deterministic.
    const long long r1 = (base_units + ctas - 1) / ctas * 2, r2 = (2 * base_units + ctas - 1) / ctas;
    return (nkb >= 8 && r2 * 100 <= r1 * 93) ? 2 : 1;
  }
  long long ks = (2LL * ctas + base_units - 1) / base_units;
  const int kmax = nkb / 2 > 1 ? nkb / 2 : 1;
  if (ks > kmax) ks = kmax;
  if (ks > 128) ks = 128;
  return ks < 1 ? 1 : (int)ks;
}

// D = A B (+ bias) with strided fp32 operands: tensor-core path when the layout allows it, fp32 FMA kernel otherwise.
// max_split = 1: no K split, so every output element has one writer and the result is the same bits on every run
// (both routes then reduce K in a fixed order).
static cudaError_t gemm_auto(const float* A, long long a_sm, long long a_sk, const float* Bm, long long b_sk,
                             long long b_sn, const float* bias, float* D, long long ldd, int M, int N, int K,
                             int accumulate, cudaStream_t st, int max_split = 0) {
  if (!accumulate && (a_sk == 1 || a_sm == 1) && (b_sk == 1 || b_sn == 1)) {
    const bool a_mn = (a_sk != 1), b_mn = (b_sk != 1);
    cudaError_t e = launch_umma_gemm(A, a_mn, a_mn ? a_sk : a_sm, Bm, b_mn, b_mn ? b_sk : b_sn, bias, D, ldd, M, N, K,
                                     sm_count_cached(), st, max_split);
    if (e != cudaErrorNotSupported) return e;
  }
  return launch_sgemm(A, a_sm, a_sk, Bm, b_sk, b_sn, bias, D, ldd, M, N, K, accumulate, st);
}

template <int SRC, int KP>
static cudaError_t launch_gram_fwd_one(const GramFwdParams& p, int grid, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(gram_fwd_kernel<SRC, KP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)kGfSmemBytes);
  if (e != cudaSuccess) return e;
  gram_fwd_kernel<SRC, KP><<<grid, kGfThreads, kGfSmemBytes, st>>>(p);
  return cudaGetLastError();
}

template <int SRC>
static cudaError_t launch_gram_fwd_kp(const GramFwdParams& p, int kp, int grid, cudaStream_t st) {
  switch (kp) {
    case 0: return launch_gram_fwd_one<SRC, 0>(p, grid, st);
    case 8: return launch_gram_fwd_one<SRC, 8>(p, grid, st);
    case 16: return launch_gram_fwd_one<SRC, 16>(p, grid, st);
    case 32: return launch_gram_fwd_one<SRC, 32>(p, grid, st);
    case 64: return launch_gram_fwd_one<SRC, 64>(p, grid, st);
    case 128: return launch_gram_fwd_one<SRC, 128>(p, grid, st);
    default: return cudaErrorInvalidValue;
  }
}

// Pair (cta_group::2, TMA-staged) kernels. -1 = auto, 0 = never, 1 = whenever TMA can describe the tensors.
static int g_opt_fwd_pair = -1;
static int g_opt_bwd_pair = -1;
static int g_opt_bwd_nt = 0;        // 0 = plan the x-tile width; 64..256 (multiple of 16) forces it (experiments)
static int g_opt_bwd_stages = 0;    // 0 = by shape; a * 16 + b forces the A / B ring depths of the pair backward
static int g_opt_bwd_ats = -1;      // pooled pair backward with the generated gradient tile in TENSOR memory (A operand of
                                    // the MMAs read from TMEM, gram_bwd_pair.cuh ATS): 0 = never, 1 = whenever the free
                                    // TMEM columns beside the two accumulators hold the A ring, -1 = auto (C >= 512)
static int g_opt_bwd_ch = 0;        // K chunks per ring stage of the tensor-memory form, at most: 1, 2 (8 MMAs per iteration
                                    // of the issuing thread, when the widened A ring fits TMEM), 0 = auto (2)

template <int KIND, int KP, bool NHWC>
static cudaError_t launch_gram_fwd_pair_one(const GramFwdParams& p, const CUtensorMap& map, int npairs, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(gram_fwd_pair_kernel<KIND, KP, NHWC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)kFpSmemBytes);
  if (e != cudaSuccess) return e;
  gram_fwd_pair_kernel<KIND, KP, NHWC><<<2 * npairs, kFpThreads, kFpSmemBytes, st>>>(p, map);
  return cudaGetLastError();
}
template <int KIND, bool NHWC>
static cudaError_t launch_gram_fwd_pair(const GramFwdParams& p, const CUtensorMap& map, int kp, int npairs, cudaStream_t st) {
  switch (kp) {
    case 0: return launch_gram_fwd_pair_one<KIND, 0, NHWC>(p, map, npairs, st);
    case 8: return launch_gram_fwd_pair_one<KIND, 8, NHWC>(p, map, npairs, st);
    case 16: return launch_gram_fwd_pair_one<KIND, 16, NHWC>(p, map, npairs, st);
    case 32: return launch_gram_fwd_pair_one<KIND, 32, NHWC>(p, map, npairs, st);
    case 64: return launch_gram_fwd_pair_one<KIND, 64, NHWC>(p, map, npairs, st);
    case 128: return launch_gram_fwd_pair_one<KIND, 128, NHWC>(p, map, npairs, st);
    default: return cudaErrorInvalidValue;
  }
}

static int gram_fwd_common(const void* F, int f_dtype, long long img_stride, long long row_stride, long long x_stride,
                           int B, int C, int HW, int mode, int g, float* out, long long out_img_stride, int ksplit,
                           int max_ctas, cudaStream_t st) {
  if (!F || !out || B <= 0 || C <= 0 || HW <= 0) return GH_ERR_BAD_ARG;
  if (f_dtype != GH_DTYPE_F32 && f_dtype != GH_DTYPE_BF16) return GH_ERR_BAD_ARG;
  // Layouts: x contiguous (NCHW: x_stride == 1, channel rows row_stride apart) or c contiguous (channels_last / NHWC:
  // row_stride == 1, positions x_stride apart). The latter exists on the CTA-pair kernels only.
  const bool nhwc = (x_stride != 1);
  if (x_stride <= 0 || row_stride <= 0 || (nhwc && row_stride != 1)) return GH_ERR_BAD_ARG;
  int kp = 0;
  if (mode == GRAM_POOL) {
    if (g <= 0 || C % g != 0) return GH_ERR_UNSUPPORTED;
    kp = C / g;
    if (ilog2_exact(kp) < 0 || kp > 128 || kp < 8) return GH_ERR_UNSUPPORTED;
  }
  GramFwdParams p;
  p.F = F; p.img_stride = img_stride; p.row_stride = row_stride;
  p.B = B; p.C = C; p.HW = HW;
  p.nT = (C + 255) / 256;
  p.nST = p.nT * (p.nT + 1) / 2;
  p.nkb = (HW + 63) / 64;
  const int sms = sm_count_cached();
  const int ctas = (max_ctas > 0 && max_ctas < sms) ? max_ctas : sms;
  const long long base_units = (long long)B * p.nST;
  const int ksplit_arg = ksplit;
  if (ksplit <= 0) ksplit = choose_ksplit(base_units, p.nkb, ctas);
  if (ksplit > p.nkb) ksplit = p.nkb;
  p.ksplit = ksplit;
  const long long total = base_units * ksplit;
  if (total > 0x7fffffffLL) return GH_ERR_UNSUPPORTED;
  p.total_units = (int)total;
  p.g = g; p.out = out; p.out_img_stride = out_img_stride;
  p.scale = (mode == GRAM_POOL) ? 1.0f / ((float)HW * (float)kp * (float)kp) : 1.0f / (float)HW;

  // ---- CTA-pair kernel with TMA-staged operands (bf16 -> kind::f16, fp32 -> kind::tf32) ----
  const bool is_bf16 = (f_dtype == GH_DTYPE_BF16);
  // auto: whenever TMA can describe the tensor. At C = 256 / fp32 the two families tie at batch 256 (143 us) and the
  // pair kernel wins at larger batches; its tf32 operands are also ~10x closer to fp32 than the ldg kernel's bf16.
  const bool want_pair = g_opt_fwd_pair != 0;
  if (want_pair && sms >= 2) {
    CUtensorMap map;
    const int kb_elems = is_bf16 ? 64 : 32;
    const bool mapped = nhwc ? make_tensor_map_nhwc_mn(&map, F, is_bf16, img_stride, x_stride, B, C, HW, kb_elems, 128,
                                                       /*tf32=*/true)
                             : make_tensor_map_xcb(&map, F, is_bf16, img_stride, row_stride, B, C, HW, kb_elems, 128,
                                                   /*tf32=*/true);
    if (mapped) {
      GramFwdParams q = p;
      q.nkb = (HW + kb_elems - 1) / kb_elems;
      int npairs = ctas / 2;
      if (npairs < 1) npairs = 1;
      int ks = ksplit_arg > 0 ? ksplit_arg : choose_ksplit(base_units, q.nkb, npairs, /*balance=*/true);
      if (ks > q.nkb) ks = q.nkb;
      q.ksplit = ks;
      const long long tot = base_units * ks;
      if (tot <= 0x7fffffffLL) {
        q.total_units = (int)tot;
        q.use_atomics = (ks > 1 || kp > 32) ? 1 : 0;
        cudaError_t e2 = cudaSuccess;
        if (q.use_atomics) {
          if (mode == GRAM_POOL) e2 = cudaMemset2DAsync(out, (size_t)out_img_stride * 4, 0, (size_t)g * g * 4, (size_t)B, st);
          else e2 = cudaMemsetAsync(out, 0, (size_t)B * C * C * 4, st);
          if (e2 != cudaSuccess) return (int)e2;
        }
        if (tot < npairs) npairs = (int)tot;
        if (nhwc)
          e2 = is_bf16 ? launch_gram_fwd_pair<KIND_BF16, true>(q, map, kp, npairs, st)
                       : launch_gram_fwd_pair<KIND_TF32, true>(q, map, kp, npairs, st);
        else
          e2 = is_bf16 ? launch_gram_fwd_pair<KIND_BF16, false>(q, map, kp, npairs, st)
                       : launch_gram_fwd_pair<KIND_TF32, false>(q, map, kp, npairs, st);
        return (int)e2;
      }
    }
  }
  if (nhwc) return GH_ERR_UNSUPPORTED;   // the ld.global kernels read NCHW rows only: the caller transposes (gh_transpose_cast)
  // every output element has exactly one writer unless K is split or a pooled row spans two epilogue warps (k > 32)
  p.use_atomics = (ksplit > 1 || kp > 32) ? 1 : 0;

  cudaError_t e;
  if (mode == GRAM_POOL) {
    if (p.use_atomics) {
      e = cudaMemset2DAsync(out, (size_t)out_img_stride * 4, 0, (size_t)g * g * 4, (size_t)B, st);
      if (e != cudaSuccess) return (int)e;
    }
  } else if (p.use_atomics) {
    e = cudaMemsetAsync(out, 0, (size_t)B * C * C * 4, st);
    if (e != cudaSuccess) return (int)e;
  }
  const int grid = (int)(total < ctas ? total : ctas);
  const uintptr_t addr = (uintptr_t)F;
  const bool s4 = (HW % 4 == 0) && (row_stride % 4 == 0) && (img_stride % 4 == 0);
  if (f_dtype == GH_DTYPE_F32) {
    if (s4 && addr % 16 == 0) e = launch_gram_fwd_kp<0>(p, kp, grid, st);
    else e = launch_gram_fwd_kp<1>(p, kp, grid, st);
  } else {
    if (s4 && addr % 8 == 0) e = launch_gram_fwd_kp<2>(p, kp, grid, st);
    else e = launch_gram_fwd_kp<3>(p, kp, grid, st);
  }
  return (int)e;
}

// Launch plan of the CTA-pair backward (gram_bwd_pair.cuh) from the shape alone: x-tile width, ring depths, and whether the
// generated gradient tile lives in tensor memory (ATS) with how many K chunks per ring stage (CH). Fills the plan fields of
// `q`; false when the shape leaves fewer than two F stages. Also behind gh_gram_bwd_plan (host logic, testable without a GPU).
static bool plan_bwd_pair(int C, int HW, int g, int mode, bool is_bf16, bool nhwc, GramBwdPairParams& q, bool* ats_out,
                          int* ch_out) {
  const int kc_elems = is_bf16 ? 64 : 32;
  gbp_plan_tiles(HW, &q.NT, &q.nHT);
  if (g_opt_bwd_nt) { q.NT = g_opt_bwd_nt; q.nHT = (HW + q.NT - 1) / q.NT; }
  // ring depths: see gram_bwd_pair.cuh. Shared-memory form: four A stages (the generator groups need that many; the
  // generated chunks are cheap), the remaining tiles cut into F stages of the width the x tile needs.
  q.a_stages = 4; q.b_stages = kBpMaxStages;
  if (g_opt_bwd_stages) { q.a_stages = g_opt_bwd_stages >> 4; q.b_stages = g_opt_bwd_stages & 15; }
  {   // k-steps of a chunk that share one generated piece of A: pooling factor / UMMA_K, capped at the 4 of a chunk
    const int umma_k = is_bf16 ? 16 : 8, kfac = (mode == GRAM_POOL && g > 0) ? (C / g) : 1;
    q.areuse = kfac >= 4 * umma_k ? 4 : (kfac >= 2 * umma_k ? 2 : 1);
  }
  bool ats = mode == GRAM_POOL && (g_opt_bwd_ats == 1 || (g_opt_bwd_ats == -1 && C >= 512));
  // one chunk's F tile: NHWC [NT/2 position rows][128 B]; NCHW: ceil(NT/2 / KC) x-blocks of [KC k-rows][128 B]
  long long sb1 = nhwc ? (long long)(q.NT / 2) * 128 : (long long)((q.NT / 2 + kc_elems - 1) / kc_elems) * kc_elems * 128;
  sb1 = (sb1 + 1023) / 1024 * 1024;
  int ch = 1;
  q.a_tmem_cols = 0; q.d_stride = 256; q.a_tmem_base = 0;
  if (ats) {
    // Most chunks per stage first (fewer iterations of the issuing thread per MMA). The accumulators take 2 * NT32
    // columns (NT rounded up to 32), the A ring the rest: stages of c * 32 / areuse columns, at least as many as the
    // 4 / c stage lanes of the generator groups and at least 2; the F ring keeps at least four stages.
    const int scols = 32 / q.areuse, cmax = g_opt_bwd_ch ? g_opt_bwd_ch : 2, nt32 = (q.NT + 31) / 32 * 32;
    bool found = false;
    for (int c = 2; c >= 1 && !found; c >>= 1) {
      if (c > cmax || ((long long)kBpRingTiles * kBpTileBytes) / (c * sb1) < 4) continue;
      int a = (512 - 2 * nt32) / (c * scols);
      if (a > 8) a = 8;
      if (a < 4 / c || a < 2) continue;
      ch = c; q.a_stages = a; found = true;
    }
    if (!found) ats = false;
    else { q.a_tmem_cols = ch * scols; q.d_stride = nt32; q.a_tmem_base = 2 * nt32; }
  }
  q.a_smem_tiles = ats ? 0 : q.a_stages;
  const long long sb = sb1 * ch;
  q.b_stage_bytes = (int)sb;
  const long long fit = ((long long)(kBpRingTiles - q.a_smem_tiles) * kBpTileBytes) / sb;
  if (q.b_stages > fit) q.b_stages = (int)fit;
  if (q.b_stages > kBpMaxStages) q.b_stages = kBpMaxStages;
  q.nCB = (C + 255) / 256;
  q.nkc = (C + kc_elems * ch - 1) / (kc_elems * ch);
  *ats_out = ats;
  *ch_out = ch;
  return q.b_stages >= 2;
}

template <int SRC>
static cudaError_t launch_gram_bwd2(const GramBwd2Params& q, int grid, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(gram_bwd2_kernel<SRC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kB2SmemBytes);
  if (e != cudaSuccess) return e;
  gram_bwd2_kernel<SRC><<<grid, kB2Threads, kB2SmemBytes, st>>>(q);
  return cudaGetLastError();
}

static int gram_bwd_common(const void* F, int f_dtype, long long img_stride, long long row_stride, long long x_stride,
                           int B, int C, int HW, int mode, int g, const float* dP, long long dp_img_stride,
                           const float* dG, void* dF_any, int df_dtype, long long df_img_stride, long long df_row_stride,
                           long long df_x_stride, int max_ctas, cudaStream_t st) {
  float* dF = reinterpret_cast<float*>(dF_any);
  if (!F || !dF || B <= 0 || C <= 0 || HW <= 0) return GH_ERR_BAD_ARG;
  if (f_dtype != GH_DTYPE_F32 && f_dtype != GH_DTYPE_BF16) return GH_ERR_BAD_ARG;
  if (df_dtype != GH_DTYPE_F32 && df_dtype != GH_DTYPE_BF16) return GH_ERR_BAD_ARG;
  const bool df16 = (df_dtype == GH_DTYPE_BF16);   // bf16 gradient: CTA-pair kernels only (GH_ERR_UNSUPPORTED otherwise)
  const bool nhwc = (x_stride != 1);     // F and dF share the layout: both NCHW-like or both channels_last
  if (x_stride <= 0 || row_stride <= 0 || df_x_stride <= 0 || df_row_stride <= 0) return GH_ERR_BAD_ARG;
  if (nhwc != (df_x_stride != 1) || (nhwc && (row_stride != 1 || df_row_stride != 1))) return GH_ERR_BAD_ARG;
  if (C % 16 != 0) return GH_ERR_UNSUPPORTED;
  int kshift = 0;           // POOL: pool factor k = 1 << kshift
  float scale;
  if (mode == GRAM_POOL) {
    if (!dP) return GH_ERR_BAD_ARG;
    if (g <= 0 || g > kB2MaxG || C % g != 0) return GH_ERR_UNSUPPORTED;
    const int k = C / g;
    kshift = ilog2_exact(k);
    if (kshift < 0) return GH_ERR_UNSUPPORTED;
    scale = 1.0f / ((float)HW * (float)k * (float)k);
  } else {
    if (!dG) return GH_ERR_BAD_ARG;
    scale = 1.0f / (float)HW;
  }
  // ---- CTA-pair kernel: F TMA-staged as the MN-major operand, dF written with TMA stores ----
  {
    const bool is_bf16 = (f_dtype == GH_DTYPE_BF16);
    const int sms_p = sm_count_cached();
    const int ctas_p = (max_ctas > 0 && max_ctas < sms_p) ? max_ctas : sms_p;
    // POOL: a 16 B chunk of the generated A tile must lie inside one pooled column (k >= 8 covers bf16 and tf32)
    const bool want_pair = g_opt_bwd_pair != 0 && ctas_p >= 2 && (mode != GRAM_POOL || (g <= kBpMaxG && (C / g) >= 8));
    CUtensorMap tmF, tmD;
    const int kc_elems = is_bf16 ? 64 : 32;
    GramBwdPairParams q;
    bool ats = false;
    int ch = 1;
    const bool planned = plan_bwd_pair(C, HW, g, mode, is_bf16, nhwc, q, &ats, &ch);
    bool mapped = false;
    if (want_pair && planned) {
      if (nhwc)     // F: K-major tiles [NT/2 position rows][128 B of channels]; dF: [32 x][32 c] tiles
        mapped = make_tensor_map_nhwc_cxb(&tmF, F, is_bf16, img_stride, x_stride, B, C, HW, kc_elems, q.NT / 2,
                                          /*tf32=*/true) &&
                 make_tensor_map_nhwc_cxb(&tmD, dF, df16, df_img_stride, df_x_stride, B, C, HW, 32, 32, /*tf32=*/false,
                                          /*swizzle64=*/df16);
      else
        mapped = make_tensor_map_xcb(&tmF, F, is_bf16, img_stride, row_stride, B, C, HW, kc_elems, kc_elems,
                                     /*tf32=*/true, /*atom32=*/!is_bf16) &&
                 make_tensor_map_xcb(&tmD, dF, df16, df_img_stride, df_row_stride, B, C, HW, 32, 32, /*tf32=*/false, false,
                                     /*swizzle64=*/df16);
    }
    if (mapped) {
      q.B = B; q.C = C; q.HW = HW; q.mode = mode;
      q.dP = dP; q.dp_img_stride = dp_img_stride; q.g = g; q.kshift = kshift; q.dG = dG;
      q.scale = scale;
      q.df_bf16 = df16 ? 1 : 0;
      const long long tot = (long long)B * q.nHT * q.nCB;
      if (tot <= 0x7fffffffLL) {
        q.total_units = (int)tot;
        int npairs = ctas_p / 2;
        if (tot < npairs) npairs = (int)tot;
        cudaError_t e3 = cudaErrorInvalidValue;
#define GH_LAUNCH_BP(KIND, MODE, NHWC, ATS, CH)                                                                        \
        {                                                                                                              \
          e3 = cudaFuncSetAttribute(gram_bwd_pair_kernel<KIND, MODE, NHWC, ATS, CH>,                                   \
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBpSmemBytes);                   \
          if (e3 != cudaSuccess) return (int)e3;                                                                       \
          gram_bwd_pair_kernel<KIND, MODE, NHWC, ATS, CH><<<2 * npairs, kBpThreads, kBpSmemBytes, st>>>(q, tmF, tmD);  \
        }
#define GH_LAUNCH_BP2(KIND, MODE, ATS, CH)                                                                             \
        {                                                                                                              \
          if (nhwc) GH_LAUNCH_BP(KIND, MODE, true, ATS, CH) else GH_LAUNCH_BP(KIND, MODE, false, ATS, CH)              \
        }
#define GH_LAUNCH_BP3(KIND)                                                                                            \
        {                                                                                                              \
          if (mode != GRAM_POOL) GH_LAUNCH_BP2(KIND, GRAM_DENSE, false, 1)                                             \
          else if (!ats) GH_LAUNCH_BP2(KIND, GRAM_POOL, false, 1)                                                      \
          else if (ch == 2) GH_LAUNCH_BP2(KIND, GRAM_POOL, true, 2)                                                    \
          else GH_LAUNCH_BP2(KIND, GRAM_POOL, true, 1)                                                                 \
        }
        if (is_bf16) GH_LAUNCH_BP3(KIND_BF16) else GH_LAUNCH_BP3(KIND_TF32)
#undef GH_LAUNCH_BP3
#undef GH_LAUNCH_BP2
#undef GH_LAUNCH_BP
        return (int)cudaGetLastError();
      }
    }
  }
  if (nhwc || df16) return GH_ERR_UNSUPPORTED;   // the ld.global kernel reads / writes fp32 NCHW rows only
  GramBwd2Params q;
  q.F = F; q.img_stride = img_stride; q.row_stride = row_stride;
  q.B = B; q.C = C; q.HW = HW; q.mode = mode;
  q.dP = dP; q.dp_img_stride = dp_img_stride; q.g = g; q.kshift = kshift; q.dG = dG;
  q.dF = dF; q.df_img_stride = df_img_stride; q.df_row_stride = df_row_stride; q.scale = scale;
  q.nHT = (HW + kB2NHW - 1) / kB2NHW;
  q.nCP = (C + 255) / 256;
  q.nkb = (C + 63) / 64;
  q.nA = (C > 128) ? 2 : 1;
  const long long total = (long long)B * q.nHT * q.nCP;
  if (total > 0x7fffffffLL) return GH_ERR_UNSUPPORTED;
  q.total_units = (int)total;
  const int sms = sm_count_cached();
  const int ctas = (max_ctas > 0 && max_ctas < sms) ? max_ctas : sms;
  int grid = (int)(total < ctas ? total : ctas);
  q.units_per_cta = (int)((total + grid - 1) / grid);
  grid = (int)((total + q.units_per_cta - 1) / q.units_per_cta);
  q.df_vec_ok = (HW % 4 == 0 && df_img_stride % 4 == 0 && df_row_stride % 4 == 0 && ((uintptr_t)dF) % 16 == 0) ? 1 : 0;
  const bool s4 = (HW % 4 == 0) && (row_stride % 4 == 0) && (img_stride % 4 == 0);
  cudaError_t e;
  if (f_dtype == GH_DTYPE_F32)
    e = (s4 && ((uintptr_t)F) % 16 == 0) ? launch_gram_bwd2<0>(q, grid, st) : launch_gram_bwd2<1>(q, grid, st);
  else
    e = (s4 && ((uintptr_t)F) % 8 == 0) ? launch_gram_bwd2<2>(q, grid, st) : launch_gram_bwd2<3>(q, grid, st);
  return (int)e;
}

// ---- general-bin adaptive pooling (torch rule), used when C % g != 0 ------------------------------------------------
__device__ __forceinline__ int bin_start(int i, int C, int g) { return (int)(((long long)i * C) / g); }
__device__ __forceinline__ int bin_end(int i, int C, int g) { return (int)((((long long)(i + 1)) * C + g - 1) / g); }

// grid (g, B), 256 threads: block (i, b) produces row i of the pooled matrix.
__global__ void adaptive_pool_fwd_kernel(const float* __restrict__ G, int C, int g, float* __restrict__ desc,
                                         long long desc_img_stride) {
  const int i = blockIdx.x, b = blockIdx.y;
  const int r0 = bin_start(i, C, g), r1 = bin_end(i, C, g);
  const float* Gb = G + (long long)b * C * C;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int j = warp; j < g; j += 8) {
    const int c0 = bin_start(j, C, g), c1 = bin_end(j, C, g);
    const int w = c1 - c0, n = (r1 - r0) * w;
    float s = 0.f;
    for (int t = lane; t < n; t += 32) s += Gb[(long long)(r0 + t / w) * C + c0 + t % w];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) desc[(long long)b * desc_img_stride + i * g + j] = s / (float)n;
  }
}
// grid (ceil(C*C/256), B): one thread per dG element; sums the (at most 2x2) bins that contain (c, d).
__global__ void adaptive_pool_bwd_kernel(const float* __restrict__ d_desc, long long desc_img_stride, int C, int g,
                                         float* __restrict__ dG) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)C * C) return;
  const int b = blockIdx.y;
  const int c = (int)(idx / C), d = (int)(idx % C);
  const float* dp = d_desc + (long long)b * desc_img_stride;
  // bins containing c: i in [ilo, ihi]; start(i) <= c < end(i)
  int ilo = (int)(((long long)c * g) / C);
  while (ilo > 0 && bin_end(ilo - 1, C, g) > c) --ilo;
  int jlo = (int)(((long long)d * g) / C);
  while (jlo > 0 && bin_end(jlo - 1, C, g) > d) --jlo;
  float s = 0.f;
  for (int i = ilo; i < g && bin_start(i, C, g) <= c; ++i) {
    if (bin_end(i, C, g) <= c) continue;
    const float ni = (float)(bin_end(i, C, g) - bin_start(i, C, g));
    for (int j = jlo; j < g && bin_start(j, C, g) <= d; ++j) {
      if (bin_end(j, C, g) <= d) continue;
      const float nj = (float)(bin_end(j, C, g) - bin_start(j, C, g));
      s += dp[i * g + j] / (ni * nj);
    }
  }
  dG[(long long)b * C * C + idx] = s;
}

// Shared by the fp32 and uint8 entry points: p.x, p.w, p.bias, p.out (and p.mean / p.std) are set and checked.
template <typename T>
static int stem_conv_pool_launch(StemConvPoolParams<T>& p, long long img_stride, long long c_stride, long long y_stride,
                                 long long x_stride, int B, int H, int W, void* stream) {
  p.s_img = img_stride; p.s_c = c_stride; p.s_y = y_stride; p.s_x = x_stride;
  p.B = B; p.OH = H / 2; p.OW = W / 2;
  p.PH = (p.OH - 1) / 2 + 1;                                     // nn.MaxPool2d(3, 2, 1), floor mode
  p.PW = (p.OW - 1) / 2 + 1;
  p.tiles = (p.PW + kScTileCols - 1) / kScTileCols;
  p.vec2 = x_stride == 1 && (uintptr_t)p.x % (2 * sizeof(T)) == 0 && (img_stride % 2 == 0) && (c_stride % 2 == 0) &&
           (y_stride % 2 == 0);
  const long long units = (long long)B * p.tiles * p.PH;
  if (units >= (1ll << 30)) return GH_ERR_UNSUPPORTED;          // 256 B of output per unit: 256 GB, more than any GPU
  p.units = (int)units;
  const int sms = sm_count_cached();
  const int grid = p.units < sms ? p.units : sms;
  const uint32_t smem = sizeof(T) == 1 ? kScSmemBytesU8 : kScSmemBytes;
  cudaError_t e = cudaFuncSetAttribute(stem_conv_pool_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  stem_conv_pool_kernel<T><<<grid, kScThreads, smem, (cudaStream_t)stream>>>(p);
  return (int)cudaGetLastError();
}

}  // namespace gh

using namespace gh;

extern "C" {

int gh_version(void) { return 100; }

int gh_sm_count(void) { return sm_count_cached(); }

#ifdef GH_BP_PROFILE
// Profile builds only (not part of include/gramhead.h): copies the 16 role counters of gram_bwd_pair_kernel and clears them.
int gh_bp_profile_read(unsigned long long* out) {
  unsigned long long zero[16] = {0};
  cudaError_t e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpyFromSymbol(out, g_bp_prof, sizeof(zero));
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_bp_prof, zero, sizeof(zero));
  return (int)e;
}
#endif

#ifdef GH_SC_PROFILE
// Profile builds only (not part of include/gramhead.h): copies the 16 role counters of stem_conv_pool_kernel and clears them.
int gh_sc_profile_read(unsigned long long* out) {
  unsigned long long zero[16] = {0};
  cudaError_t e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpyFromSymbol(out, g_sc_prof, sizeof(zero));
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_sc_prof, zero, sizeof(zero));
  return (int)e;
}
#endif

int gh_gram_bwd_plan(int C, int HW, int g, int f_dtype, int channels_last, int* out) {
  if (!out || C <= 0 || HW <= 0 || g <= 0 || (f_dtype != GH_DTYPE_F32 && f_dtype != GH_DTYPE_BF16)) return GH_ERR_BAD_ARG;
  if (C % g != 0 || g > kBpMaxG || C / g < 8 || ilog2_exact(C / g) < 0) return GH_ERR_UNSUPPORTED;
  GramBwdPairParams q;
  bool ats = false;
  int ch = 1;
  if (!plan_bwd_pair(C, HW, g, GRAM_POOL, f_dtype == GH_DTYPE_BF16, channels_last != 0, q, &ats, &ch)) return GH_ERR_UNSUPPORTED;
  out[0] = q.NT; out[1] = q.nHT; out[2] = ats ? 1 : 0; out[3] = ch; out[4] = q.a_stages; out[5] = q.b_stages;
  out[6] = q.a_tmem_base + q.a_stages * q.a_tmem_cols;   // TMEM columns in use (ATS), 0 otherwise
  out[7] = q.b_stages * q.b_stage_bytes + q.a_smem_tiles * (int)kBpTileBytes;   // ring bytes in shared memory
  return 0;
}

int gh_set_option(const char* name, int value) {
  if (!name) return GH_ERR_BAD_ARG;
  const std::string key(name);
  if (key == "gram_fwd_pair") {
    if (value < -1 || value > 1) return GH_ERR_BAD_ARG;
    g_opt_fwd_pair = value;
    return 0;
  }
  if (key == "gram_bwd_pair") {
    if (value < -1 || value > 1) return GH_ERR_BAD_ARG;
    g_opt_bwd_pair = value;
    return 0;
  }
  if (key == "gram_bwd_nt") {
    if (value != 0 && (value < 64 || value > 256 || value % 16)) return GH_ERR_BAD_ARG;
    g_opt_bwd_nt = value;
    return 0;
  }
  if (key == "gram_bwd_stages") {        // value = a_stages * 16 + b_stages (experiments; b is capped by what fits)
    const int a = value >> 4, b = value & 15;
    if (value != 0 && (a < kBpGroups || b < 2 || a > kBpRingTiles - 2 || b > kBpMaxStages)) return GH_ERR_BAD_ARG;
    g_opt_bwd_stages = value;
    return 0;
  }
  if (key == "gram_bwd_ats") {
    if (value < -1 || value > 1) return GH_ERR_BAD_ARG;
    g_opt_bwd_ats = value;
    return 0;
  }
  if (key == "gram_bwd_ch") {
    if (value < 0 || value > 2) return GH_ERR_BAD_ARG;
    g_opt_bwd_ch = value;
    return 0;
  }
  if (key == "tgemm_tn") {
    if (value != 0 && value != 128 && value != 256) return GH_ERR_BAD_ARG;
    g_opt_tg_tn = value;
    return 0;
  }
  if (key == "pdl") {
    if (value != 0 && value != 1) return GH_ERR_BAD_ARG;
    g_opt_pdl = value;
    return 0;
  }
  return GH_ERR_BAD_ARG;
}

int gh_last_device_error(unsigned int* out4) {
  if (!out4) return GH_ERR_BAD_ARG;
  volatile unsigned int* rec = error_record_host();
  if (!rec) return GH_ERR_UNSUPPORTED;
  for (int i = 0; i < 4; ++i) out4[i] = rec[i];
  for (int i = 3; i >= 0; --i) rec[i] = 0u;
  return 0;
}

int gh_gram_pool_fwd(const void* F, int f_dtype, long long img_stride, long long row_stride, long long x_stride, int B,
                     int C, int HW, int g, float* desc, int l, int L, int ksplit, int max_ctas, void* stream) {
  if (!desc || l < 0 || l >= L || g <= 0) return GH_ERR_BAD_ARG;
  return gram_fwd_common(F, f_dtype, img_stride, row_stride, x_stride, B, C, HW, GRAM_POOL, g, desc + (long long)l * g * g,
                         (long long)L * g * g, ksplit, max_ctas, (cudaStream_t)stream);
}

int gh_gram_dense_fwd(const void* F, int f_dtype, long long img_stride, long long row_stride, long long x_stride, int B,
                      int C, int HW, float* G, int ksplit, int max_ctas, void* stream) {
  return gram_fwd_common(F, f_dtype, img_stride, row_stride, x_stride, B, C, HW, GRAM_DENSE, 0, G, (long long)C * C, ksplit,
                         max_ctas, (cudaStream_t)stream);
}

int gh_adaptive_pool_fwd(const float* G, int B, int C, int g, float* desc, int l, int L, void* stream) {
  if (!G || !desc || B <= 0 || C <= 0 || g <= 0 || l < 0 || l >= L) return GH_ERR_BAD_ARG;
  if (B > 65535) return GH_ERR_UNSUPPORTED;
  adaptive_pool_fwd_kernel<<<dim3(g, B), 256, 0, (cudaStream_t)stream>>>(G, C, g, desc + (long long)l * g * g,
                                                                         (long long)L * g * g);
  return (int)cudaGetLastError();
}

int gh_adaptive_pool_bwd(const float* d_desc, int l, int L, int B, int C, int g, float* dG, void* stream) {
  if (!dG || !d_desc || B <= 0 || C <= 0 || g <= 0 || l < 0 || l >= L) return GH_ERR_BAD_ARG;
  if (B > 65535) return GH_ERR_UNSUPPORTED;
  const long long n = (long long)C * C;
  adaptive_pool_bwd_kernel<<<dim3((unsigned)((n + 255) / 256), B), 256, 0, (cudaStream_t)stream>>>(
      d_desc + (long long)l * g * g, (long long)L * g * g, C, g, dG);
  return (int)cudaGetLastError();
}

int gh_gram_pool_bwd(const void* F, int f_dtype, long long img_stride, long long row_stride, long long x_stride, int B,
                     int C, int HW, int g, const float* d_desc, int l, int L, void* dF, int df_dtype,
                     long long df_img_stride, long long df_row_stride, long long df_x_stride, int max_ctas, void* stream) {
  if (!d_desc || l < 0 || l >= L || g <= 0) return GH_ERR_BAD_ARG;
  return gram_bwd_common(F, f_dtype, img_stride, row_stride, x_stride, B, C, HW, GRAM_POOL, g,
                         d_desc + (long long)l * g * g, (long long)L * g * g, nullptr, dF, df_dtype, df_img_stride,
                         df_row_stride, df_x_stride, max_ctas, (cudaStream_t)stream);
}

int gh_gram_dense_bwd(const void* F, int f_dtype, long long img_stride, long long row_stride, long long x_stride, int B,
                      int C, int HW, const float* dG, void* dF, int df_dtype, long long df_img_stride,
                      long long df_row_stride, long long df_x_stride, int max_ctas, void* stream) {
  return gram_bwd_common(F, f_dtype, img_stride, row_stride, x_stride, B, C, HW, GRAM_DENSE, 0, nullptr, 0, dG, dF,
                         df_dtype, df_img_stride, df_row_stride, df_x_stride, max_ctas, (cudaStream_t)stream);
}

int gh_attn_head_fwd(const float* desc, const float* W_in, const float* b_in, const float* W_out, const float* b_out,
                     const float* W_c, const float* b_c, int B, int L, int E, int nc, float* qkv, float* probs,
                     float* obar, float* emb, float* logits, void* stream) {
  if (!desc || !W_in || !W_out || !W_c || !qkv || !probs || !obar || !emb || !logits) return GH_ERR_BAD_ARG;
  if (B <= 0 || L <= 0 || E <= 0 || nc <= 0) return GH_ERR_BAD_ARG;
  if (L > kMaxL) return GH_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e;
  // QKV = X W_in^T + b_in           (B*L, 3E)
  e = gemm_auto(desc, E, 1, W_in, 1, E, b_in, qkv, 3LL * E, B * L, 3 * E, E, 0, st);
  if (e != cudaSuccess) return (int)e;
  if (L <= 4) attn_core_fwd_kernel<4><<<B, 128, 0, st>>>(qkv, probs, obar, L, E);
  else attn_core_fwd_kernel<kMaxL><<<B, 128, 0, st>>>(qkv, probs, obar, L, E);
  e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  // emb = Obar W_out^T + b_out      (B, E)
  e = gemm_auto(obar, E, 1, W_out, 1, E, b_out, emb, E, B, E, E, 0, st);
  if (e != cudaSuccess) return (int)e;
  // logits = emb W_c^T + b_c        (B, nc): nc is a handful of classes -> one warp per (image, class) dot product
  classifier_fwd_kernel<<<(B * nc + 3) / 4, 128, 0, st>>>(emb, W_c, b_c, logits, B, E, nc);
  return (int)cudaGetLastError();
}

int gh_transpose_cast(const void* in, int in_dtype, void* out, int out_dtype, int B, int R, int S, long long out_pitch,
                      void* stream) {
  if (!in || !out || B <= 0 || R <= 0 || S <= 0 || out_pitch < R) return GH_ERR_BAD_ARG;
  if ((in_dtype != GH_DTYPE_F32 && in_dtype != GH_DTYPE_BF16) || (out_dtype != GH_DTYPE_F32 && out_dtype != GH_DTYPE_BF16))
    return GH_ERR_BAD_ARG;
  if (B > 65535 || (R + 63) / 64 > 65535) return GH_ERR_UNSUPPORTED;
  const dim3 grid((S + 63) / 64, (R + 63) / 64, B), block(64, 4);
  cudaStream_t st = (cudaStream_t)stream;
  if (in_dtype == GH_DTYPE_F32 && out_dtype == GH_DTYPE_F32)
    transpose_cast_kernel<float, float><<<grid, block, 0, st>>>((const float*)in, (float*)out, R, S, out_pitch);
  else if (in_dtype == GH_DTYPE_F32)
    transpose_cast_kernel<float, __nv_bfloat16><<<grid, block, 0, st>>>((const float*)in, (__nv_bfloat16*)out, R, S, out_pitch);
  else if (out_dtype == GH_DTYPE_BF16)
    transpose_cast_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, block, 0, st>>>((const __nv_bfloat16*)in, (__nv_bfloat16*)out, R, S, out_pitch);
  else
    transpose_cast_kernel<__nv_bfloat16, float><<<grid, block, 0, st>>>((const __nv_bfloat16*)in, (float*)out, R, S, out_pitch);
  return (int)cudaGetLastError();
}

int gh_preprocess_frame(const unsigned char* frame, long long pitch_bytes, int H, int W, int bgr, const int* hx_min,
                        const int* hx_size, const int* hk, int hkmax, const int* vy_min, const int* vy_size, const int* vk,
                        int vkmax, const float* mean3_host, const float* std3_host, float* out, int OH, int OW,
                        void* stream) {
  if (!frame || !hx_min || !hx_size || !hk || !vy_min || !vy_size || !vk || !mean3_host || !std3_host || !out)
    return GH_ERR_BAD_ARG;
  if (H <= 0 || W <= 0 || OH <= 0 || OW <= 0 || hkmax <= 0 || vkmax <= 0 || pitch_bytes < 3LL * W) return GH_ERR_BAD_ARG;
  if (OH > 65535) return GH_ERR_UNSUPPORTED;
  PreprocParams p;
  p.frame = frame; p.pitch = pitch_bytes; p.H = H; p.W = W; p.OH = OH; p.OW = OW;
  p.hx_min = hx_min; p.hx_size = hx_size; p.hk = hk; p.hkmax = hkmax;
  p.vy_min = vy_min; p.vy_size = vy_size; p.vk = vk; p.vkmax = vkmax;
  p.out = out; p.bgr = bgr ? 1 : 0;
  for (int c = 0; c < 3; ++c) { p.mean[c] = mean3_host[c]; p.std[c] = std3_host[c]; }
  preprocess_frame_kernel<<<dim3((OW + 255) / 256, OH), 256, 0, (cudaStream_t)stream>>>(p);
  return (int)cudaGetLastError();
}

static_assert(sizeof(GhFrameDesc) == 80, "GhFrameDesc is mirrored by streaming.FRAME_DESC_DTYPE");

int gh_preprocess_frames_smem(int OW, int span_rows) {
  if (OW <= 0 || span_rows <= 0) return GH_ERR_BAD_ARG;
  const long long bytes = 3LL * OW * span_rows;
  return bytes > kFramesMaxSmem ? GH_ERR_UNSUPPORTED : (int)bytes;
}

int gh_preprocess_frames(const GhFrameDesc* frames, int N, int OH, int OW, int band_rows, int span_rows, const int* tables,
                         int hkmax, int vkmax, unsigned char* out, void* stream) {
  if (!frames || !tables || !out) return GH_ERR_BAD_ARG;
  if (N <= 0 || OH <= 0 || OW <= 0 || band_rows <= 0 || hkmax <= 0 || vkmax <= 0 || span_rows < vkmax) return GH_ERR_BAD_ARG;
  const int smem = gh_preprocess_frames_smem(OW, span_rows);
  if (smem < 0) return smem;
  const int bands = (int)((OH + (long long)band_rows - 1) / band_rows);
  if (N > 65535 || bands > 65535) return GH_ERR_UNSUPPORTED;
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(preprocess_frames_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return (int)e;
  }
  FramesParams p;
  p.frames = frames; p.tables = tables; p.out = out;
  p.OH = OH; p.OW = OW; p.band_rows = band_rows; p.span_rows = span_rows; p.hkmax = hkmax; p.vkmax = vkmax;
  preprocess_frames_kernel<<<dim3(bands, N), kFramesThreads, smem, (cudaStream_t)stream>>>(p);
  return (int)cudaGetLastError();
}

long long gh_frame_tables_stride(int OH, int OW, int hkmax, int vkmax) {
  if (OH <= 0 || OW <= 0 || hkmax <= 0 || vkmax <= 0) return GH_ERR_BAD_ARG;
  return frame_tables_stride(OH, OW, hkmax, vkmax);
}

int gh_frame_tables(const long long* geom, int N, const unsigned char* base, int OH, int OW, int hkmax, int vkmax,
                    int* tables, GhFrameDesc* frames, void* stream) {
  if (!geom || !base || !tables || !frames) return GH_ERR_BAD_ARG;
  if (N <= 0 || OH <= 0 || OW <= 0 || hkmax <= 0 || vkmax <= 0) return GH_ERR_BAD_ARG;
  const long long coords = (long long)OH + OW;
  if (N > 65535 || coords > 0x7fffffffLL - kFrameTablesThreads) return GH_ERR_UNSUPPORTED;
  FrameTablesParams p;
  p.geom = geom; p.base = base; p.tables = tables; p.frames = frames;
  p.OH = OH; p.OW = OW; p.hkmax = hkmax; p.vkmax = vkmax; p.stride = frame_tables_stride(OH, OW, hkmax, vkmax);
  const dim3 grid((unsigned)((coords + kFrameTablesThreads - 1) / kFrameTablesThreads), (unsigned)N);
  frame_tables_kernel<<<grid, kFrameTablesThreads, 0, (cudaStream_t)stream>>>(p);
  return (int)cudaGetLastError();
}

int gh_normalize_u8(const unsigned char* src, float* dst, long long images, int channels, long long hw,
                    const float* mean_host, const float* std_host, void* stream) {
  if (!src || !dst || !mean_host || !std_host || images <= 0 || hw <= 0) return GH_ERR_BAD_ARG;
  if (channels <= 0 || channels > 4) return GH_ERR_UNSUPPORTED;
  NormalizeU8Params p{};
  p.src = src; p.dst = dst; p.hw = hw; p.C = channels;
  for (int c = 0; c < channels; ++c) {
    if (!(std_host[c] != 0.f)) return GH_ERR_BAD_ARG;             // torchvision's Normalize raises on a zero std
    p.mean[c] = mean_host[c]; p.std[c] = std_host[c];
  }
  const long long planes = images * channels;
  // with hw % 4 == 0 every plane starts 4 B (uint8) / 16 B (fp32) aligned whenever the batch does
  const bool quads = hw % 4 == 0 && (uintptr_t)src % 4 == 0 && (uintptr_t)dst % 16 == 0;
  const long long groups = quads ? hw / 4 : hw;
  const long long chunks = (groups + 256 * kNormUnroll - 1) / (256 * kNormUnroll);
  if (planes > 0x7fffffffLL || chunks > 65535 || groups > 0x7fffffffLL) return GH_ERR_UNSUPPORTED;
  p.groups = (int)groups;
  const dim3 grid((unsigned)planes, (unsigned)chunks);
  if (quads) normalize_u8_kernel<4><<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  else normalize_u8_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  return (int)cudaGetLastError();
}

int gh_gemm_f32(const float* A, long long a_sm, long long a_sk, const float* Bm, long long b_sk, long long b_sn,
                const float* bias, float* D, long long ldd, int M, int N, int K, void* stream) {
  if (!A || !Bm || !D || M <= 0 || N <= 0 || K <= 0) return GH_ERR_BAD_ARG;
  return (int)gemm_auto(A, a_sm, a_sk, Bm, b_sk, b_sn, bias, D, ldd, M, N, K, 0, (cudaStream_t)stream);
}

int gh_gemm_f32_fixed(const float* A, long long a_sm, long long a_sk, const float* Bm, long long b_sk, long long b_sn,
                      const float* bias, float* D, long long ldd, int M, int N, int K, void* stream) {
  if (!A || !Bm || !D || M <= 0 || N <= 0 || K <= 0) return GH_ERR_BAD_ARG;
  return (int)gemm_auto(A, a_sm, a_sk, Bm, b_sk, b_sn, bias, D, ldd, M, N, K, 0, (cudaStream_t)stream, 1);
}

int gh_colsum_f32(const float* X, long long ldx, int M, int N, float* out, void* stream) {
  if (!X || !out || M <= 0 || N <= 0 || ldx < N) return GH_ERR_BAD_ARG;
  colsum_kernel<<<(N + 31) / 32, dim3(32, 8), 0, (cudaStream_t)stream>>>(X, ldx, out, M, N);
  return (int)cudaGetLastError();
}

int gh_maxpool2d_nhwc(const void* in, int dtype, void* out, int B, int H, int W, int C, int k, int stride, int pad,
                      void* stream) {
  if (!in || !out || B <= 0 || H <= 0 || W <= 0 || C <= 0 || k <= 0 || stride <= 0 || pad < 0) return GH_ERR_BAD_ARG;
  if (dtype != GH_DTYPE_F32 && dtype != GH_DTYPE_BF16) return GH_ERR_BAD_ARG;
  if (2 * pad > k) return GH_ERR_BAD_ARG;                       // torch's own constraint: pad <= k / 2
  const int vec = dtype == GH_DTYPE_F32 ? 4 : 8;
  if (C % vec != 0 || (uintptr_t)in % 16 != 0 || (uintptr_t)out % 16 != 0) return GH_ERR_UNSUPPORTED;
  MaxPoolParams p{};
  p.in = in; p.out = out; p.B = B; p.H = H; p.W = W; p.C = C; p.k = k; p.stride = stride; p.pad = pad;
  p.OH = (H + 2 * pad - k) / stride + 1;                         // floor mode (ceil_mode=False), dilation 1
  p.OW = (W + 2 * pad - k) / stride + 1;
  if (p.OH <= 0 || p.OW <= 0) return GH_ERR_BAD_ARG;
  p.total_vec = (long long)B * p.OH * p.OW * (C / vec);
  const int cv = C / vec;
  if (cv > 256 || B > 65535) return GH_ERR_UNSUPPORTED;
  const int ppc = 256 / cv;
  const dim3 grid((p.OW + ppc - 1) / ppc, (p.OH + kPoolRows - 1) / kPoolRows, B);
  if (grid.y > 65535) return GH_ERR_UNSUPPORTED;
  if (dtype == GH_DTYPE_F32) maxpool2d_nhwc_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  else maxpool2d_nhwc_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  return (int)cudaGetLastError();
}

int gh_stem_space_to_depth(const float* x, long long img_stride, long long c_stride, long long y_stride,
                           long long x_stride, int B, int H, int W, void* z, int z_dtype, void* stream) {
  if (!x || !z || B <= 0 || H <= 0 || W <= 0) return GH_ERR_BAD_ARG;
  if (z_dtype != GH_DTYPE_F32 && z_dtype != GH_DTYPE_BF16) return GH_ERR_BAD_ARG;
  if ((H & 1) || (W & 1) || (uintptr_t)z % 16 != 0) return GH_ERR_UNSUPPORTED;
  StemS2DParams p{};
  p.x = x; p.z = z; p.s_img = img_stride; p.s_c = c_stride; p.s_y = y_stride; p.s_x = x_stride;
  p.B = B; p.H = H; p.W = W; p.HP = H / 2 + 3; p.WP = W / 2 + 3;
  p.total = (long long)B * p.HP * p.WP;
  const long long want = (p.total + 255) / 256;
  const long long cap = (long long)gh_sm_count() * 32;
  const int grid = (int)(want < cap ? want : cap);
  if (z_dtype == GH_DTYPE_F32) stem_space_to_depth_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  else stem_space_to_depth_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  return (int)cudaGetLastError();
}

int gh_stem_conv_pool_nhwc(const float* x, long long img_stride, long long c_stride, long long y_stride,
                           long long x_stride, int B, int H, int W, const float* w_packed, const float* bias, float* out,
                           void* stream) {
  if (!x || !w_packed || !bias || !out || B <= 0 || H <= 0 || W <= 0) return GH_ERR_BAD_ARG;
  if ((H & 1) || (W & 1) || (uintptr_t)w_packed % 16 != 0 || (uintptr_t)out % 16 != 0) return GH_ERR_UNSUPPORTED;
  StemConvPoolParams<float> p{};
  p.x = x; p.w = w_packed; p.bias = bias; p.out = out;
  return stem_conv_pool_launch(p, img_stride, c_stride, y_stride, x_stride, B, H, W, stream);
}

int gh_stem_conv_pool_u8_nhwc(const unsigned char* x, long long img_stride, long long c_stride, long long y_stride,
                              long long x_stride, int B, int H, int W, const float* mean3_host, const float* std3_host,
                              const float* w_packed, const float* bias, float* out, void* stream) {
  if (!x || !mean3_host || !std3_host || !w_packed || !bias || !out || B <= 0 || H <= 0 || W <= 0) return GH_ERR_BAD_ARG;
  StemConvPoolParams<uint8_t> p{};
  for (int c = 0; c < 3; ++c) {
    if (!(std3_host[c] != 0.f && std3_host[c] == std3_host[c])) return GH_ERR_BAD_ARG;     // zero or NaN std
    p.mean[c] = mean3_host[c]; p.std[c] = std3_host[c];
  }
  if ((H & 1) || (W & 1) || (uintptr_t)w_packed % 16 != 0 || (uintptr_t)out % 16 != 0) return GH_ERR_UNSUPPORTED;
  p.x = x; p.w = w_packed; p.bias = bias; p.out = out;
  return stem_conv_pool_launch(p, img_stride, c_stride, y_stride, x_stride, B, H, W, stream);
}

int gh_gram_mse_blocks(long long n) {
  if (n <= 0) return 0;
  long long blocks = (n / 4 + kMseThreads - 1) / kMseThreads;
  const long long cap = (long long)sm_count_cached() * 4 < kMseMaxBlocks ? (long long)sm_count_cached() * 4 : kMseMaxBlocks;
  if (blocks > cap) blocks = cap;
  return (int)(blocks < 1 ? 1 : blocks);
}

int gh_gram_mse(const float* G, const float* G_target, long long n, float* dG, float* partial, void* stream) {
  if (!G || !G_target || !dG || !partial || n <= 0) return GH_ERR_BAD_ARG;
  if (((uintptr_t)G | (uintptr_t)G_target | (uintptr_t)dG) % 16 != 0) return GH_ERR_UNSUPPORTED;
  gram_mse_kernel<<<gh_gram_mse_blocks(n), kMseThreads, 0, (cudaStream_t)stream>>>(G, G_target, dG, partial, n,
                                                                                   1.0f / (float)n);
  return (int)cudaGetLastError();
}

int gh_gram_mse_images_blocks(long long n_img) { return gh_gram_mse_blocks(n_img); }

int gh_gram_mse_images(const float* G, const float* G_target, int B, long long n_img, float* dG, float* partial,
                       void* stream) {
  if (!G || !G_target || !dG || !partial || B <= 0 || n_img <= 0) return GH_ERR_BAD_ARG;
  if (B > 65535) return GH_ERR_UNSUPPORTED;                                  // gridDim.y
  const dim3 grid(gh_gram_mse_blocks(n_img), B);
  gram_mse_images_kernel<<<grid, kMseThreads, 0, (cudaStream_t)stream>>>(G, G_target, dG, partial, n_img,
                                                                         1.0f / (float)n_img);
  return (int)cudaGetLastError();
}

long long gh_patch_gram_workspace(int L, int B, int D) {
  if (L <= 0 || B <= 0 || D <= 0) return 0;
  return (long long)L * B * D * (kPatchBins + 4);      // bin means (16 floats) + two doubles per plane
}

int gh_patch_gram_fwd(const float* const* maps, const int* H, const int* W, const long long* strides, int L, int B,
                      int D, int ln_input, float* gram, float* gram_norm, float* workspace, void* stream) {
  if (!maps || !H || !W || !strides || !gram || !gram_norm || !workspace || L <= 0 || B <= 0 || D <= 0)
    return GH_ERR_BAD_ARG;
  if ((uintptr_t)workspace % 8 != 0) return GH_ERR_BAD_ARG;
  if (L > kPatchMaxLayers || D > kPatchMaxD || B > 0x7fffffff / 2) return GH_ERR_UNSUPPORTED;
  PatchGramParams p{};
  for (int l = 0; l < L; ++l) {
    if (!maps[l] || H[l] <= 0 || W[l] <= 0) return GH_ERR_BAD_ARG;
    p.layer[l].x = maps[l];
    p.layer[l].H = H[l];
    p.layer[l].W = W[l];
    p.layer[l].s_img = strides[4 * l + 0];
    p.layer[l].s_c = strides[4 * l + 1];
    p.layer[l].s_y = strides[4 * l + 2];
    p.layer[l].s_x = strides[4 * l + 3];
  }
  p.L = L; p.B = B; p.D = D; p.ln_input = ln_input ? 1 : 0;
  p.gram = gram; p.gram_norm = gram_norm;
  const long long planes = (long long)L * B * D;
  double* stats = reinterpret_cast<double*>(workspace);              // (L, B, D, 2) doubles first: 8 B aligned
  float* pooled = workspace + planes * 4;                            // (L, B, D, 16)
  const long long gx = (long long)B * ((D + 7) / 8);
  if (gx > 0x7fffffffLL) return GH_ERR_UNSUPPORTED;
  patch_pool_kernel<<<dim3((unsigned)gx, L), kPatchThreads, (kPatchThreads / 32) * kPatchSmallPlane * sizeof(float),
                      (cudaStream_t)stream>>>(p, pooled, stats);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  const size_t smem = (size_t)D * kPatchBins * 4 + 32 * sizeof(double);
  patch_gram_kernel<<<dim3(B, L), kPatchThreads, smem, (cudaStream_t)stream>>>(p, pooled, stats);
  return (int)cudaGetLastError();
}

int gh_patch_attn_fwd(const float* feat, const float* W_in1, const float* b_in1, const float* W_out1,
                      const float* b_out1, const float* W_in2, const float* b_in2, const float* W_out2,
                      const float* b_out2, const float* W_c, const float* b_c, int L, int B, int E, int heads, int nc,
                      float* emb, float* logits, void* stream) {
  if (!feat || !W_in1 || !b_in1 || !W_out1 || !b_out1 || !W_in2 || !b_in2 || !W_out2 || !b_out2 || !W_c || !b_c ||
      !emb || !logits)
    return GH_ERR_BAD_ARG;
  if (L <= 0 || B <= 0 || E <= 0 || heads <= 0 || nc <= 0 || E % heads != 0) return GH_ERR_BAD_ARG;
  if (L > kPatchMaxLayers || E > 128 || E % 4 != 0) return GH_ERR_UNSUPPORTED;
  const float* ptrs[6] = {W_in1, W_out1, W_in2, W_out2, feat, W_c};
  for (int i = 0; i < 4; ++i)
    if ((uintptr_t)ptrs[i] % 16 != 0) return GH_ERR_UNSUPPORTED;       // weight rows are read as float4
  PatchAttnParams p{};
  p.feat = feat;
  p.w_in[0] = W_in1; p.b_in[0] = b_in1; p.w_out[0] = W_out1; p.b_out[0] = b_out1;
  p.w_in[1] = W_in2; p.b_in[1] = b_in2; p.w_out[1] = W_out2; p.b_out[1] = b_out2;
  p.w_c = W_c; p.b_c = b_c;
  p.L = L; p.B = B; p.E = E; p.heads = heads; p.nc = nc;
  p.emb = emb; p.logits = logits;
  const size_t smem = ((size_t)L * E * 5 + (size_t)heads * L * L) * 4;
  const int sms = gh_sm_count();
  const int grid = B < 4 * sms ? B : 4 * sms;
  patch_attention_kernel<<<grid, kPatchThreads, smem, (cudaStream_t)stream>>>(p);
  return (int)cudaGetLastError();
}

long long gh_patch_bwd_workspace(int L, int B, int D) {
  if (L <= 0 || B <= 0 || D <= 0) return 0;
  return (long long)L * B * (D * kPatchBins + kPatchBwdScalars);   // coefficient tables, then 4 scalars per image
}

int gh_patch_gram_bwd(const int* H, const int* W, int L, int B, int D, int ln_input, const float* d_gram,
                      const float* d_norm, const float* gram_norm, const float* fwd_workspace, float* bwd_workspace,
                      void* stream) {
  if (!H || !W || !d_gram || !d_norm || !gram_norm || !fwd_workspace || !bwd_workspace || L <= 0 || B <= 0 || D <= 0)
    return GH_ERR_BAD_ARG;
  if ((uintptr_t)fwd_workspace % 8 != 0 || (uintptr_t)bwd_workspace % 16 != 0) return GH_ERR_BAD_ARG;
  if (L > kPatchMaxLayers || D > kPatchMaxD || B > 65535) return GH_ERR_UNSUPPORTED;
  PatchGramParams p{};
  for (int l = 0; l < L; ++l) {
    if (H[l] <= 0 || W[l] <= 0) return GH_ERR_BAD_ARG;
    p.layer[l].H = H[l];
    p.layer[l].W = W[l];
  }
  p.L = L; p.B = B; p.D = D; p.ln_input = ln_input ? 1 : 0;
  p.gram_norm = const_cast<float*>(gram_norm);        // read: the forward's norms
  const long long planes = (long long)L * B * D;
  const double* stats = reinterpret_cast<const double*>(fwd_workspace);   // gh_patch_gram_fwd's layout
  const float* pooled = fwd_workspace + planes * 4;
  float* coef = bwd_workspace;
  float* scal = bwd_workspace + planes * kPatchBins;
  const size_t smem = ((size_t)D * kPatchBins + (size_t)D * (D + 1) + kPatchBins * kPatchBins) * 4 + 32 * sizeof(double);
  cudaError_t e = cudaFuncSetAttribute(patch_gram_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  patch_gram_bwd_kernel<<<dim3(B, L), kPatchThreads, smem, (cudaStream_t)stream>>>(p, pooled, stats, d_gram, d_norm, coef,
                                                                                  scal);
  return (int)cudaGetLastError();
}

int gh_patch_pool_bwd(const float* const* maps, float* const* d_maps, const int* H, const int* W, const long long* strides,
                      const long long* d_strides, int L, int B, int D, int ln_input, const float* bwd_workspace,
                      void* stream) {
  if (!d_maps || !H || !W || !d_strides || !bwd_workspace || L <= 0 || B <= 0 || D <= 0) return GH_ERR_BAD_ARG;
  if (ln_input && (!maps || !strides)) return GH_ERR_BAD_ARG;
  if ((uintptr_t)bwd_workspace % 16 != 0) return GH_ERR_BAD_ARG;
  if (L > kPatchMaxLayers || D > kPatchMaxD || B > 0x7fffffff / 2) return GH_ERR_UNSUPPORTED;
  PatchPoolBwdParams p{};
  for (int l = 0; l < L; ++l) {
    if (!d_maps[l] || H[l] <= 0 || W[l] <= 0 || (ln_input && !maps[l])) return GH_ERR_BAD_ARG;
    p.layer[l].x = ln_input ? maps[l] : nullptr;
    p.layer[l].H = H[l];
    p.layer[l].W = W[l];
    if (ln_input) {
      p.layer[l].s_img = strides[4 * l + 0];
      p.layer[l].s_c = strides[4 * l + 1];
      p.layer[l].s_y = strides[4 * l + 2];
      p.layer[l].s_x = strides[4 * l + 3];
    }
    p.grad[l].dx = d_maps[l];
    p.grad[l].s_img = d_strides[4 * l + 0];
    p.grad[l].s_c = d_strides[4 * l + 1];
    p.grad[l].s_y = d_strides[4 * l + 2];
    p.grad[l].s_x = d_strides[4 * l + 3];
  }
  p.L = L; p.B = B; p.D = D; p.ln_input = ln_input ? 1 : 0;
  const long long planes = (long long)L * B * D;
  p.coef = bwd_workspace;
  p.scal = bwd_workspace + planes * kPatchBins;
  const long long gx = (long long)B * ((D + 7) / 8);
  if (gx > 0x7fffffffLL) return GH_ERR_UNSUPPORTED;
  patch_pool_bwd_kernel<<<dim3((unsigned)gx, L), kPatchThreads, 0, (cudaStream_t)stream>>>(p);
  return (int)cudaGetLastError();
}

int gh_patch_attn_bwd(const float* feat, const float* W_in1, const float* b_in1, const float* W_out1,
                      const float* b_out1, const float* W_in2, const float* b_in2, const float* W_out2,
                      const float* b_out2, const float* W_c, const float* d_emb, const float* d_logits, int L, int B,
                      int E, int heads, int nc, float* d_feat, float* x1, float* dqkv, float* o, float* dy,
                      void* stream) {
  if (!feat || !W_in1 || !b_in1 || !W_out1 || !b_out1 || !W_in2 || !b_in2 || !W_out2 || !b_out2 || !W_c || !d_emb ||
      !d_logits || !d_feat || !x1 || !dqkv || !o || !dy)
    return GH_ERR_BAD_ARG;
  if (L <= 0 || B <= 0 || E <= 0 || heads <= 0 || nc <= 0 || E % heads != 0) return GH_ERR_BAD_ARG;
  if (L > kPatchMaxLayers || E > 128 || E % 4 != 0) return GH_ERR_UNSUPPORTED;
  const float* ptrs[4] = {W_in1, W_out1, W_in2, W_out2};
  for (int i = 0; i < 4; ++i)
    if ((uintptr_t)ptrs[i] % 16 != 0) return GH_ERR_UNSUPPORTED;       // in_proj rows are read as float4
  PatchAttnBwdParams p{};
  p.f.feat = feat;
  p.f.w_in[0] = W_in1; p.f.b_in[0] = b_in1; p.f.w_out[0] = W_out1; p.f.b_out[0] = b_out1;
  p.f.w_in[1] = W_in2; p.f.b_in[1] = b_in2; p.f.w_out[1] = W_out2; p.f.b_out[1] = b_out2;
  p.f.w_c = W_c;
  p.f.L = L; p.f.B = B; p.f.E = E; p.f.heads = heads; p.f.nc = nc;
  p.d_emb = d_emb; p.d_logits = d_logits;
  p.d_feat = d_feat; p.x1 = x1; p.dqkv = dqkv; p.o = o; p.dy = dy;
  const size_t smem = ((size_t)L * E * 15 + (size_t)heads * L * L * 3 + E) * 4;
  cudaError_t e = cudaFuncSetAttribute(patch_attention_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const int sms = gh_sm_count();
  const int grid = B < 2 * sms ? B : 2 * sms;
  patch_attention_bwd_kernel<<<grid, kPatchThreads, smem, (cudaStream_t)stream>>>(p);
  return (int)cudaGetLastError();
}

// ---- attention head on the TMA-fed split-bf16 GEMMs (tgemm_pair.cuh, attn_head2.cuh) --------------------------------
static bool attn2_supported(int B, int L, int E, int nc) {
  return B > 0 && L > 0 && L <= kMaxL && E >= 64 && E % 64 == 0 && E <= 4 * kAttn2Threads && nc > 0 && nc <= kAttn2MaxNc &&
         sm_count_cached() >= 2;
}
static TgOperand tg_op(const void* planes, long long ld, long long rows_total, int mn_major) {
  TgOperand o;
  o.planes = planes; o.ld = ld; o.plane_stride = ld * rows_total; o.mn_major = mn_major;
  return o;
}
static TgSpec tg_spec(TgOperand A, TgOperand Bo, int M, int N, int K, const float* bias, float* D, long long ldd,
                      int max_split) {
  TgSpec s{};
  s.A = A; s.B = Bo; s.M = M; s.N = N; s.K = K; s.bias = bias; s.D_f32 = D; s.D_planes = nullptr; s.ldd = ldd;
  s.d_plane_stride = 0; s.max_split = max_split; s.tn = 256; s.ksplit = 1;
  return s;
}

int gh_split_bf16(const float* src, void* planes, long long n, long long plane_stride, void* stream) {
  if (!src || !planes || n <= 0 || plane_stride < n) return GH_ERR_BAD_ARG;
  if (n % 4 != 0 || plane_stride % 4 != 0 || (uintptr_t)src % 16 != 0 || (uintptr_t)planes % 8 != 0) return GH_ERR_UNSUPPORTED;
  const long long n4 = n / 4;
  long long blocks = (n4 + 255) / 256;
  const long long cap = (long long)sm_count_cached() * 16;
  if (blocks > cap) blocks = cap;
  return (int)launch_pdl(split_bf16_kernel, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, src,
                         (__nv_bfloat16*)planes, n4, plane_stride);
}

int gh_tgemm_plan(int M, int N, int K, int max_split, int npairs, int* tn, int* ksplit, int* units) {
  if (M <= 0 || N <= 0 || K <= 0 || npairs <= 0 || !tn || !ksplit || !units) return GH_ERR_BAD_ARG;
  TgSpec s{};
  s.M = M; s.N = N; s.K = K; s.max_split = max_split < 1 ? 1 : max_split; s.tn = 256; s.ksplit = 1;
  tg_plan(&s, 1, npairs);
  *tn = s.tn;
  *ksplit = s.ksplit;
  *units = ((M + 255) / 256) * ((N + s.tn - 1) / s.tn) * s.ksplit;
  return 0;
}

int gh_gemm_planes(const void* A_planes, long long lda, long long a_plane_stride, int a_mn, const void* B_planes,
                   long long ldb, long long b_plane_stride, int b_mn, const float* bias, float* D, void* D_planes,
                   long long ldd, long long d_plane_stride, int M, int N, int K, int max_split, void* stream) {
  if (!A_planes || !B_planes || (!D && !D_planes) || (D && D_planes) || M <= 0 || N <= 0 || K <= 0) return GH_ERR_BAD_ARG;
  TgSpec s{};
  s.A.planes = A_planes; s.A.ld = lda; s.A.plane_stride = a_plane_stride; s.A.mn_major = a_mn ? 1 : 0;
  s.B.planes = B_planes; s.B.ld = ldb; s.B.plane_stride = b_plane_stride; s.B.mn_major = b_mn ? 1 : 0;
  s.M = M; s.N = N; s.K = K; s.bias = bias; s.D_f32 = D; s.D_planes = D_planes; s.ldd = ldd;
  s.d_plane_stride = d_plane_stride; s.max_split = D_planes ? 1 : (max_split < 1 ? 1 : max_split);
  const int sms = sm_count_cached();
  if (sms < 2) return GH_ERR_UNSUPPORTED;
  tg_plan(&s, 1, sms / 2);
  cudaStream_t st = (cudaStream_t)stream;
  TgLaunch l;
  cudaError_t e = tg_prepare(&s, 1, sms, &l);       // before the K-split zeroing: a refused call writes nothing
  if (e != cudaSuccess) return e == cudaErrorNotSupported ? GH_ERR_UNSUPPORTED : (int)e;
  if (s.ksplit > 1) {
    e = cudaMemset2DAsync(D, (size_t)ldd * 4, 0, (size_t)N * 4, (size_t)M, st);
    if (e != cudaSuccess) return (int)e;
  }
  return (int)tg_launch(l, st);
}

int gh_attn_head_fwd2(const float* desc, const void* w_in_planes, const float* b_in, const void* w_out_planes,
                      const float* b_out, const float* W_c, const float* b_c, int B, int L, int E, int nc, void* x_planes,
                      float* qkv, float* probs, void* obar_planes, float* emb, float* logits, void* stream) {
  if (!desc || !w_in_planes || !w_out_planes || !W_c || !x_planes || !qkv || !probs || !obar_planes || !emb || !logits)
    return GH_ERR_BAD_ARG;
  if (B <= 0 || L <= 0 || E <= 0 || nc <= 0) return GH_ERR_BAD_ARG;
  if (!attn2_supported(B, L, E, nc)) return GH_ERR_UNSUPPORTED;
  if ((uintptr_t)W_c % 16 != 0) return GH_ERR_UNSUPPORTED;      // the classifier reads its rows as float4
  cudaStream_t st = (cudaStream_t)stream;
  const int sms = sm_count_cached();
  const long long BL = (long long)B * L;
  // QKV = X W_in^T + b_in           (B*L, 3E); at most two K partitions, so the sum is bitwise reproducible
  TgSpec s1 = tg_spec(tg_op(x_planes, E, BL, 0), tg_op(w_in_planes, E, 3LL * E, 0), (int)BL, 3 * E, E, b_in, qkv, 3LL * E, 2);
  tg_plan(&s1, 1, sms / 2);
  // emb = Obar W_out^T + b_out      (B, E)
  TgSpec s2 = tg_spec(tg_op(obar_planes, E, B, 0), tg_op(w_out_planes, E, E, 0), B, E, E, b_out, emb, E, 2);
  tg_plan(&s2, 1, sms / 2);
  // both GEMMs are checked (alignment, tensor maps) before the first write, so a refused call writes nothing
  TgLaunch l1, l2;
  cudaError_t e = tg_prepare(&s1, 1, sms, &l1);
  if (e == cudaSuccess) e = tg_prepare(&s2, 1, sms, &l2);
  if (e != cudaSuccess) return e == cudaErrorNotSupported ? GH_ERR_UNSUPPORTED : (int)e;
  // X -> planes (the A operand of the in_proj GEMM, and of dW_in in the backward)
  int rc = gh_split_bf16(desc, x_planes, BL * E, BL * E, stream);
  if (rc != 0) return rc;
  if (s1.ksplit > 1) {
    e = cudaMemsetAsync(qkv, 0, (size_t)BL * 3 * E * 4, st);
    if (e != cudaSuccess) return (int)e;
  }
  e = tg_launch(l1, st);
  if (e != cudaSuccess) return (int)e;
  __nv_bfloat16* ob = (__nv_bfloat16*)obar_planes;
  float* ez = s2.ksplit > 1 ? emb : nullptr;
  if (L <= 4) e = launch_pdl(attn2_core_fwd_kernel<4>, dim3(B), dim3(kAttn2Threads), 0, st, qkv, probs, ob, (long long)B * E, ez, L, E);
  else e = launch_pdl(attn2_core_fwd_kernel<kMaxL>, dim3(B), dim3(kAttn2Threads), 0, st, qkv, probs, ob, (long long)B * E, ez, L, E);
  if (e != cudaSuccess) return (int)e;
  e = tg_launch(l2, st);
  if (e != cudaSuccess) return (int)e;
  return (int)launch_pdl(attn2_classifier_kernel, dim3((B + 3) / 4), dim3(128), 0, st, emb, W_c, b_c, logits, B, E, nc);
}

long long gh_attn_head_bwd2_workspace(int B, int L, int E) {
  if (B <= 0 || L <= 0 || E <= 0) return 0;
  // bytes: demb planes (2 * B*E bf16) | dobar fp32 (B*E) | dQKV planes (2 * B*L*3E bf16) | db_in scratch (3E fp32)
  return 4LL * B * E + 4LL * B * E + 12LL * B * L * E + 12LL * E;
}

int gh_attn_head_bwd2(const void* x_planes, const void* w_in_planes, const void* w_out_planes, const float* W_c,
                      const float* qkv, const float* probs, const void* obar_planes, const float* emb,
                      const float* d_logits, const float* d_emb_ext, int B, int L, int E, int nc, float* d_desc,
                      float* dW_in, float* db_in, float* dW_out, float* db_out, float* dW_c, float* db_c, void* workspace,
                      void* stream) {
  if (!x_planes || !w_in_planes || !w_out_planes || !W_c || !qkv || !probs || !obar_planes || !emb || !d_logits || !workspace)
    return GH_ERR_BAD_ARG;
  if (B <= 0 || L <= 0 || E <= 0 || nc <= 0) return GH_ERR_BAD_ARG;
  if (!attn2_supported(B, L, E, nc) || (uintptr_t)workspace % 16 != 0) return GH_ERR_UNSUPPORTED;
  // read (and db_in zeroed) as float4
  if (((uintptr_t)qkv | (uintptr_t)emb | (uintptr_t)W_c | (uintptr_t)d_emb_ext | (uintptr_t)db_in) % 16 != 0) return GH_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const int sms = sm_count_cached();
  const long long BL = (long long)B * L, BE = (long long)B * E;
  uint8_t* ws = (uint8_t*)workspace;
  __nv_bfloat16* demb = (__nv_bfloat16*)ws;                       // planes (B, E)
  float* dobar = (float*)(ws + 4 * BE);                           // (B, E)
  __nv_bfloat16* dqkv = (__nv_bfloat16*)(ws + 8 * BE);            // planes (B*L, 3E)
  float* dbin_scratch = (float*)(ws + 8 * BE + 12 * BL * E);      // (3E) when the caller does not want db_in

  // G1: dObar = demb W_out (B, E) and dW_out = demb^T Obar (E, E)
  TgSpec g1[2];
  int n1 = 0;
  g1[n1++] = tg_spec(tg_op(demb, E, B, 0), tg_op(w_out_planes, E, E, 1), B, E, E, nullptr, dobar, E, 64);
  if (dW_out) g1[n1++] = tg_spec(tg_op(demb, E, B, 1), tg_op(obar_planes, E, B, 1), E, E, B, nullptr, dW_out, E, 64);
  tg_plan(g1, n1, sms / 2);
  // G2: dW_in = dQKV^T X (3E, E) and dX = dQKV W_in (B*L, E)
  TgSpec g2[2];
  int n2 = 0;
  if (dW_in) g2[n2++] = tg_spec(tg_op(dqkv, 3LL * E, BL, 1), tg_op(x_planes, E, BL, 1), 3 * E, E, (int)BL, nullptr, dW_in, E, 64);
  if (d_desc) g2[n2++] = tg_spec(tg_op(dqkv, 3LL * E, BL, 0), tg_op(w_in_planes, E, 3LL * E, 1), (int)BL, E, 3 * E, nullptr, d_desc, E, 64);
  if (n2) tg_plan(g2, n2, sms / 2);
  // both launches are checked (alignment, tensor maps) before the first write, so a refused call writes nothing
  TgLaunch l1, l2;
  cudaError_t e = tg_prepare(g1, n1, sms, &l1);
  if (e == cudaSuccess && n2) e = tg_prepare(g2, n2, sms, &l2);
  if (e != cudaSuccess) return e == cudaErrorNotSupported ? GH_ERR_UNSUPPORTED : (int)e;

  float* dbin = db_in ? db_in : dbin_scratch;
  ZeroList z0{};
  z0.ptr[0] = g1[0].ksplit > 1 ? dobar : nullptr; z0.n4[0] = BE / 4;
  z0.ptr[1] = (n1 > 1 && g1[1].ksplit > 1) ? dW_out : nullptr; z0.n4[1] = (long long)E * E / 4;
  z0.ptr[2] = dbin; z0.n4[2] = 3LL * E / 4;
  const size_t prep_smem = attn2_prep_smem_bytes(nc);
  if (prep_smem > 48 * 1024) {
    e = cudaFuncSetAttribute(attn2_bwd_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prep_smem);
    if (e != cudaSuccess) return (int)e;
  }
  e = launch_pdl(attn2_bwd_prep_kernel, dim3((E + 127) / 128, kPrepSplit), dim3(kPrepThreads), prep_smem, st, d_logits,
                 d_emb_ext, W_c, emb, demb, BE, db_out, dW_c, db_c, B, E, nc, z0);
  if (e != cudaSuccess) return (int)e;
  e = tg_launch(l1, st);
  if (e != cudaSuccess) return (int)e;
  ZeroList z1{};
  for (int i = 0; i < n2; ++i) {
    z1.ptr[i] = g2[i].ksplit > 1 ? g2[i].D_f32 : nullptr;
    z1.n4[i] = (long long)g2[i].M * g2[i].N / 4;
  }
  int grid = 2 * sms;                              // one resident wave; each CTA adds its db_in column sums once
  if (grid > B) grid = B;
  if (L <= 4) e = launch_pdl(attn2_core_bwd_kernel<4>, dim3(grid), dim3(kAttn2Threads), 0, st, qkv, probs, (const float*)dobar, dqkv, BL * 3 * E, dbin, B, L, E, z1);
  else e = launch_pdl(attn2_core_bwd_kernel<kMaxL>, dim3(grid), dim3(kAttn2Threads), 0, st, qkv, probs, (const float*)dobar, dqkv, BL * 3 * E, dbin, B, L, E, z1);
  if (e != cudaSuccess) return (int)e;
  if (n2) {
    e = tg_launch(l2, st);
    if (e != cudaSuccess) return (int)e;
  }
  return (int)cudaGetLastError();
}

long long gh_attn_head_bwd_workspace(int B, int L, int E) {
  return 2LL * B * E + 3LL * B * L * E;
}

int gh_attn_head_bwd(const float* desc, const float* W_in, const float* W_out, const float* W_c, const float* qkv,
                     const float* probs, const float* obar, const float* emb, const float* d_logits,
                     const float* d_emb_ext, int B, int L, int E, int nc, float* d_desc, float* dW_in, float* db_in,
                     float* dW_out, float* db_out, float* dW_c, float* db_c, float* workspace, void* stream) {
  if (!desc || !W_in || !W_out || !W_c || !qkv || !probs || !obar || !emb || !d_logits || !workspace)
    return GH_ERR_BAD_ARG;
  if (B <= 0 || L <= 0 || E <= 0 || nc <= 0) return GH_ERR_BAD_ARG;
  if (L > kMaxL) return GH_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  float* demb = workspace;                    // (B, E)
  float* dobar = demb + (long long)B * E;     // (B, E)
  float* dqkv = dobar + (long long)B * E;     // (B*L, 3E)
  cudaError_t e;
  // demb = d_logits W_c (+ d_emb_ext)
  if (d_emb_ext) {
    e = cudaMemcpyAsync(demb, d_emb_ext, (size_t)B * E * 4, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return (int)e;
  }
  e = gemm_auto(d_logits, nc, 1, W_c, E, 1, nullptr, demb, E, B, E, nc, d_emb_ext ? 1 : 0, st);
  if (e != cudaSuccess) return (int)e;
  if (dW_c) {   // dW_c = d_logits^T emb   (nc, E)
    e = gemm_auto(d_logits, 1, nc, emb, E, 1, nullptr, dW_c, E, nc, E, B, 0, st);
    if (e != cudaSuccess) return (int)e;
  }
  if (db_c) colsum_kernel<<<(nc + 31) / 32, dim3(32, 8), 0, st>>>(d_logits, nc, db_c, B, nc);
  if (dW_out) {   // dW_out = demb^T Obar  (E, E)
    e = gemm_auto(demb, 1, E, obar, E, 1, nullptr, dW_out, E, E, E, B, 0, st);
    if (e != cudaSuccess) return (int)e;
  }
  if (db_out) colsum_kernel<<<(E + 31) / 32, dim3(32, 8), 0, st>>>(demb, E, db_out, B, E);
  // dObar = demb W_out             (B, E)
  e = gemm_auto(demb, E, 1, W_out, E, 1, nullptr, dobar, E, B, E, E, 0, st);
  if (e != cudaSuccess) return (int)e;
  attn_core_bwd_kernel<<<B, 128, 0, st>>>(qkv, probs, dobar, dqkv, L, E);
  e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  if (dW_in) {   // dW_in = dQKV^T X       (3E, E)
    e = gemm_auto(dqkv, 1, 3LL * E, desc, E, 1, nullptr, dW_in, E, 3 * E, E, B * L, 0, st);
    if (e != cudaSuccess) return (int)e;
  }
  if (db_in) colsum_kernel<<<(3 * E + 31) / 32, dim3(32, 8), 0, st>>>(dqkv, 3LL * E, db_in, B * L, 3 * E);
  if (d_desc) {  // dX = dQKV W_in         (B*L, E)
    e = gemm_auto(dqkv, 3LL * E, 1, W_in, E, 1, nullptr, d_desc, E, B * L, E, 3 * E, 0, st);
    if (e != cudaSuccess) return (int)e;
  }
  return (int)cudaGetLastError();
}


int gh_jpeg_table_ints(void) { return GH_JPEG_TABLE_INTS; }

long long gh_jpeg_records_bytes(long long scan_bytes, int n_segs, int subseq_bytes) {
  if (scan_bytes < 0 || n_segs <= 0 || subseq_bytes <= 0) return GH_ERR_BAD_ARG;
  // segment i's records start at (its first byte / subseq_bytes + i): room for every segment's ceil(len / subseq) ones
  return (scan_bytes / subseq_bytes + n_segs + 1) * (long long)kJpegRecordInts * 4;
}

int gh_jpeg_check(long long scan_bytes, int n_segs, int n_imgs, long long max_blocks, long long max_pixels,
                  int subseq_bytes, int phases) {
  if (scan_bytes <= 0 || n_segs <= 0 || n_imgs <= 0 || max_blocks <= 0 || max_pixels <= 0 || subseq_bytes <= 0)
    return GH_ERR_BAD_ARG;
  if (phases <= 0 || phases > (GH_JPEG_PHASE_HUFFMAN | GH_JPEG_PHASE_IDCT | GH_JPEG_PHASE_COLOR)) return GH_ERR_BAD_ARG;
  // the batch's scan data has no size limit (offsets are 64-bit; a segment's own length is bounded by the caller and by
  // the kernel, GH_JPEG_MAX_SEGMENT_BYTES); grids: images on y, blocks and pixels on x
  if (n_imgs > 65535 || (max_blocks + 31) / 32 > 0x7fffffffLL ||
      (max_pixels + kJpegColorThreads - 1) / kJpegColorThreads > 0x7fffffffLL)
    return GH_ERR_UNSUPPORTED;
  return 0;
}

int gh_jpeg_decode(const unsigned char* scan, long long scan_bytes, const long long* segs, int n_segs,
                   const long long* imgs, int n_imgs, const int* tables, long long max_blocks, long long max_pixels,
                   int subseq_bytes, short* coef, unsigned char* planes, int* records, int* status, unsigned char* arena,
                   int phases, void* stream) {
  if (!scan || !segs || !imgs || !tables || !coef || !planes || !records || !status || !arena) return GH_ERR_BAD_ARG;
  const int rc = gh_jpeg_check(scan_bytes, n_segs, n_imgs, max_blocks, max_pixels, subseq_bytes, phases);
  if (rc != 0) return rc;
  JpegParams p;
  p.scan = scan; p.scan_bytes = scan_bytes; p.segs = segs; p.imgs = imgs; p.tables = tables;
  p.n_segs = n_segs; p.n_imgs = n_imgs; p.subseq = subseq_bytes;
  p.coef = coef; p.planes = planes; p.records = records; p.status = status; p.arena = arena;
  const cudaStream_t st = (cudaStream_t)stream;
  if (phases & GH_JPEG_PHASE_HUFFMAN) {
    const cudaError_t e = cudaMemsetAsync(status, 0, sizeof(int) * (size_t)n_imgs, st);
    if (e != cudaSuccess) return (int)e;
    jpeg_huffman_kernel<<<n_segs, kJpegHuffThreads, 0, st>>>(p);
  }
  if (phases & GH_JPEG_PHASE_IDCT)
    jpeg_idct_kernel<<<dim3((unsigned)((max_blocks + 31) / 32), (unsigned)n_imgs), kJpegIdctThreads, 0, st>>>(p);
  if (phases & GH_JPEG_PHASE_COLOR)
    jpeg_color_kernel<<<dim3((unsigned)((max_pixels + kJpegColorThreads - 1) / kJpegColorThreads), (unsigned)n_imgs),
                        kJpegColorThreads, 0, st>>>(p);
  return (int)cudaGetLastError();
}

}  // extern "C"
