// Building blocks of the CTA-pair (cta_group::2) kernels: cluster helpers, cross-CTA mbarrier signalling, 2-SM TMEM
// allocation / MMA / commit, TMA tile loads and stores, and the host-side tensor-map encoder.
//
// Pair protocol used by gram_fwd_pair.cuh and gram_bwd_pair.cuh (cluster of 2 CTAs on one TPC, rank 0 = leader):
//   * both CTAs lay out shared memory identically; an UMMA descriptor built by the leader addresses the same offset
//     in both CTAs, each of which holds its half of the A rows (M = 256 -> 128 per CTA) and its half of the B rows
//     (N -> N/2 per CTA);
//   * every CTA issues the TMA loads of its own halves, all of them completing on the LEADER's `full` barrier;
//   * one thread of the leader issues tcgen05.mma.cta_group::2 and commits with a multicast arrive, so the `empty`
//     and `tmem_full` barriers fire at the same offset in both CTAs;
//   * each CTA drains its own 128 TMEM lanes and arrives on the leader's `tmem_empty` barrier.
#pragma once
#include <cuda.h>
#include "common.cuh"

namespace gh {

// ---------------------------------------------------------------------------------------------
// cluster
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nclusters_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
  return r;
}
// Every thread of both CTAs. Also orders prior shared-memory writes (barrier inits) before the peer's accesses.
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address of this CTA -> shared::cluster address of the same offset in CTA `rank` of the cluster.
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// Arrive on a barrier given by a shared::cluster address (own or peer CTA).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// Waits on barriers that the peer CTA arrives on use the same default-scope try_wait as local ones (as CUTLASS's
// ClusterBarrier does): what crosses the CTA boundary is ordered by the tcgen05 / async-proxy fences around it, and
// a cluster-scope acquire would cost a MEMBAR.ALL.GPU per wait.
__device__ __forceinline__ void mbar_wait_cl(uint32_t bar, uint32_t parity, uint32_t site) { mbar_wait(bar, parity, site); }

// ---------------------------------------------------------------------------------------------
// tcgen05, cta_group::2
// ---------------------------------------------------------------------------------------------
// One warp in EACH CTA of the pair, same destination offset in both.
__device__ __forceinline__ void tmem_alloc2(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// Operand kinds of the pair kernels.
//   KIND_BF16: bf16 features, kind::f16, 64 elements per 128 B smem row, K = 16 per instruction
//   KIND_TF32: fp32 features consumed as they are by kind::tf32 (the tensor core reads the upper 19 bits),
//              32 elements per 128 B smem row, K = 8 per instruction
enum : int { KIND_BF16 = 0, KIND_TF32 = 1 };

template <int KIND>
struct KindTraits;
template <>
struct KindTraits<KIND_BF16> {
  static constexpr uint32_t kElemBytes = 2, kElemsPerRow = 64, kUmmaK = 16, kFormat = 1;
};
template <>
struct KindTraits<KIND_TF32> {
  static constexpr uint32_t kElemBytes = 4, kElemsPerRow = 32, kUmmaK = 8, kFormat = 2;
};

// Instruction descriptor: D fp32, A/B of format `fmt` (1 = bf16, 2 = tf32), majors 0 = K-major, 1 = MN-major.
__host__ __device__ constexpr uint32_t make_idesc(uint32_t fmt, uint32_t m, uint32_t n, uint32_t a_mn, uint32_t b_mn) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (a_mn << 15) | (b_mn << 16) | ((n >> 3) << 17) | ((m >> 4) << 24);
}
// MN-major SWIZZLE_128B operand: 128 B rows run along MN, 8 consecutive K rows form a 1 KB group (SBO),
// `lbo_bytes` separates successive 128 B-wide MN blocks.
__host__ __device__ constexpr uint64_t make_smem_desc_sw128_mnmajor(uint32_t smem_addr, uint32_t lbo_bytes) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(1024u >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}

// MN-major operand of 32-bit elements (tf32): the only layout the tensor core accepts is the 128 B swizzle with a 32 B
// atom (Swizzle<2,5,2>: 32 B chunks XOR-ed with the row index mod 4; TMA: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B).
// Groups of 4 K rows (512 B) are `sbo` apart, 128 B-wide MN blocks `lbo_bytes` apart.
__host__ __device__ constexpr uint64_t make_smem_desc_sw128b32_mnmajor(uint32_t smem_addr, uint32_t lbo_bytes) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(512u >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)1 << 61);
}

// D[tmem, 256 x N across the pair] (+)= A B^T ; issued by one thread of the leader CTA.
template <int KIND>
__device__ __forceinline__ void umma2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                      uint32_t accumulate) {
  if constexpr (KIND == KIND_BF16) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// Same product with the A operand read from TENSOR MEMORY instead of shared memory: [128 lanes = this CTA's rows][K
// columns of 32 bit: one tf32 or two bf16 elements each], at the same TMEM address in both CTAs of the pair. The MMA
// then fetches only B from shared memory (gram_bwd_pair.cuh, ATS: the generated gradient tile never touches smem).
template <int KIND>
__device__ __forceinline__ void umma2_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                         uint32_t accumulate) {
  if constexpr (KIND == KIND_BF16) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// Warp-collective: lane l writes 8 consecutive 32-bit columns of TMEM lane (lane quarter of taddr) + l: four times `a`,
// then four times `b` (one k-step of a generated operand row whose 16 B pieces are constant).
__device__ __forceinline__ void tmem_st8_pairs(uint32_t taddr, uint32_t a, uint32_t b) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %2, %2, %2, %2};" ::"r"(taddr), "r"(a), "r"(b)
               : "memory");
}
// The same for two and four k-steps in one instruction (16 / 32 columns): a TMEM store costs the issuing warp a few
// hundred cycles under MMA load whatever its width, so a stage's k-steps leave together.
__device__ __forceinline__ void tmem_st16_pairs(uint32_t taddr, const uint32_t (&t)[8]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %1, %1, %1, %2, %2, %2, %2, %3, %3, %3, %3, %4, %4, %4, %4};" ::"r"(taddr),
      "r"(t[0]), "r"(t[1]), "r"(t[2]), "r"(t[3])
      : "memory");
}
__device__ __forceinline__ void tmem_st32_pairs(uint32_t taddr, const uint32_t (&t)[8]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %1, %1, %1, %2, %2, %2, %2, %3, %3, %3, %3, %4, %4, %4, %4, "
      "%5, %5, %5, %5, %6, %6, %6, %6, %7, %7, %7, %7, %8, %8, %8, %8};" ::"r"(taddr),
      "r"(t[0]), "r"(t[1]), "r"(t[2]), "r"(t[3]), "r"(t[4]), "r"(t[5]), "r"(t[6]), "r"(t[7])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// Arrives on the barrier at this offset in BOTH CTAs once every MMA issued so far by this thread has finished.
__device__ __forceinline__ void umma_commit2(uint32_t bar) {
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(mask)
               : "memory");
}

// ---------------------------------------------------------------------------------------------
// TMA
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
// Single-CTA tile load: completes (bytes) on a barrier of this CTA.
__device__ __forceinline__ void tma_load_3d(uint32_t dst_smem, const CUtensorMap* tmap, uint32_t bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// Pair tile load: data lands in this CTA's shared memory, the byte count completes on `bar_cluster`, a
// shared::cluster barrier address that may belong to the peer (the leader's `full` barrier).
__device__ __forceinline__ void tma_load_3d_pair(uint32_t dst_smem, const CUtensorMap* tmap, uint32_t bar_cluster,
                                                 int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(uint32_t dst_smem, const CUtensorMap* tmap, uint32_t bar_cluster,
                                                 int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// Tile store shared -> global (clipped at the tensor bounds), tracked by the issuing thread's bulk async-group.
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tmap, uint32_t src_smem, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tmap)),
               "r"(src_smem), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// Blocks until at most N of this thread's store groups still have to READ their shared-memory source.
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---------------------------------------------------------------------------------------------
// Host: cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda).
// ---------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(ptr);
  }
  return fn;
}

// (B, C, HW) tensor, element (b, c, x) at base[b*img_stride + c*row_stride + x] (strides in elements), viewed as a 3-D
// map (x, c, b) with a box of box_x x box_c x 1 elements and 128 B swizzle (box_x * elem_bytes must be 128).
// Out-of-bounds box elements read as zero and are not written. Returns false when TMA cannot describe the layout
// (base or pitches not multiples of 16 B, extents out of range): the caller then uses a non-TMA kernel.
// tf32: fp32 elements as CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, for tensor-core operands: the TMA unit rounds fp32 to the
//       nearest tf32 on the way in (measured on B200: normwise Gram error 4e-6..7e-6, against 7e-4 for FLOAT32 bits
//       that the tensor core truncates). Otherwise FLOAT32: bits copied (gradient stores).
// atom32: 128 B swizzle with a 32 B atom (MN-major tf32 operands) instead of the plain 128 B swizzle.
inline bool make_tensor_map_xcb(CUtensorMap* map, const void* base, bool is_bf16, long long img_stride,
                                long long row_stride, int B, int C, int HW, int box_x, int box_c, bool tf32,
                                bool atom32 = false, bool swizzle64 = false) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return false;
  const long long es = is_bf16 ? 2 : 4;
  if ((reinterpret_cast<uintptr_t>(base) & 15u) || (row_stride * es) % 16 || (img_stride * es) % 16) return false;
  if (row_stride < HW || img_stride <= 0 || box_x * es != (swizzle64 ? 64 : 128) || box_c > 256 || box_c < 1) return false;
  if (row_stride * es >= (1LL << 40) || img_stride * es >= (1LL << 40)) return false;
  cuuint64_t dims[3] = {(cuuint64_t)HW, (cuuint64_t)C, (cuuint64_t)B};
  cuuint64_t strides[2] = {(cuuint64_t)(row_stride * es), (cuuint64_t)(img_stride * es)};
  cuuint32_t box[3] = {(cuuint32_t)box_x, (cuuint32_t)box_c, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  const CUtensorMapDataType dt = is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                 : (tf32 ? CU_TENSOR_MAP_DATA_TYPE_TFLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32);
  CUresult r = enc(map, dt, 3,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle64 ? CU_TENSOR_MAP_SWIZZLE_64B
                             : (atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B),
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

// ---- channels-last (NHWC) features: element (b, c, x) at base[b*img_stride + x*x_stride + c], c contiguous ----------
// Operand tiles whose MN index is the channel (the Gram forward): 128 B rows run along c, so the canonical MN-major tile
// of R channels x K positions is R/E atoms of [K positions][E channels] (E = 128 B of elements). One 4-D box fetches
// all atoms of a tile: dims (c within atom, x, atom, b), box E x box_x x (R/E) x 1, landing as [atom][x][E].
// tf32 MN-major operands need the 32 B-atom flavour of the 128 B swizzle. tf32: as for make_tensor_map_xcb.
inline bool make_tensor_map_nhwc_mn(CUtensorMap* map, const void* base, bool is_bf16, long long img_stride,
                                    long long x_stride, int B, int C, int HW, int box_x, int rows, bool tf32) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return false;
  const long long es = is_bf16 ? 2 : 4;
  const int E = (int)(128 / es);
  if ((reinterpret_cast<uintptr_t>(base) & 15u) || (x_stride * es) % 16 || (img_stride * es) % 16) return false;
  if (C % E != 0 || rows % E != 0 || x_stride < C || img_stride <= 0 || box_x < 1 || box_x > 256) return false;
  if (x_stride * es >= (1LL << 40) || img_stride * es >= (1LL << 40)) return false;
  cuuint64_t dims[4] = {(cuuint64_t)E, (cuuint64_t)HW, (cuuint64_t)(C / E), (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)(x_stride * es), (cuuint64_t)128, (cuuint64_t)(img_stride * es)};
  cuuint32_t box[4] = {(cuuint32_t)E, (cuuint32_t)box_x, (cuuint32_t)(rows / E), 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUtensorMapDataType dt = is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                 : (tf32 ? CU_TENSOR_MAP_DATA_TYPE_TFLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32);
  CUresult r = enc(map, dt, 4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   is_bf16 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}
// The same tensor as a 3-D map (c, x, b) with a box of box_c x box_x x 1 and the plain 128 B swizzle: K-major operand
// tiles whose K index is the channel (the backward's F operand: [x rows][128 B of channels]) and the NHWC gradient store.
inline bool make_tensor_map_nhwc_cxb(CUtensorMap* map, const void* base, bool is_bf16, long long img_stride,
                                     long long x_stride, int B, int C, int HW, int box_c, int box_x, bool tf32,
                                     bool swizzle64 = false) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return false;
  const long long es = is_bf16 ? 2 : 4;
  if ((reinterpret_cast<uintptr_t>(base) & 15u) || (x_stride * es) % 16 || (img_stride * es) % 16) return false;
  if (x_stride < C || img_stride <= 0 || box_c * es != (swizzle64 ? 64 : 128) || box_x < 1 || box_x > 256) return false;
  if (x_stride * es >= (1LL << 40) || img_stride * es >= (1LL << 40)) return false;
  cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)HW, (cuuint64_t)B};
  cuuint64_t strides[2] = {(cuuint64_t)(x_stride * es), (cuuint64_t)(img_stride * es)};
  cuuint32_t box[3] = {(cuuint32_t)box_c, (cuuint32_t)box_x, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  const CUtensorMapDataType dt = is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                 : (tf32 ? CU_TENSOR_MAP_DATA_TYPE_TFLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32);
  CUresult r = enc(map, dt, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

}  // namespace gh
