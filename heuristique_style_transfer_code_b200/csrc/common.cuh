// Device-side building blocks shared by the sm_100a kernels of the library:
// mbarrier, proxy fences, TMEM allocation, tcgen05.mma / commit / ld wrappers and the
// UMMA shared-memory / instruction descriptors for the two operand layouts in use: bf16, K-major, 128-byte swizzle
// (8-row x 128 B atoms, 1024 B apart; the Gram and attention kernels), and tf32, K-major, no swizzle (8-row x 16 B
// core matrices; the fused stem, stem.cuh).
//
// Nothing here includes torch/ATen headers; the library is a plain C-ABI .so (include/gramhead.h).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace gh {

// ---------------------------------------------------------------------------------------------
// Error reporting from device code. A bounded mbarrier wait that runs out of time records where it happened and
// traps, so a protocol bug surfaces as a launch failure instead of a hung GPU. The record {code, blockIdx.x,
// threadIdx.x, site tag} lives in MAPPED PINNED HOST memory (error_record_host(), below): after a trap the context is in
// a sticky error state and no CUDA call could copy it back, but the host can still read its own memory.
// ---------------------------------------------------------------------------------------------
__device__ unsigned int* g_dev_error_ptr = nullptr;   // device address of the mapped record; null until the library's
                                                      // first launch on this device (error_record_host())

__device__ __forceinline__ void dev_fail(unsigned int code, unsigned int site) {
  unsigned int* rec = g_dev_error_ptr;
  if (rec != nullptr && atomicCAS_system(rec, 0u, code) == 0u) {
    rec[1] = blockIdx.x;
    rec[2] = threadIdx.x;
    rec[3] = site;
    __threadfence_system();
  }
  __trap();
}

// Host side: the record of the current device, allocated and published to g_dev_error_ptr on first use.
inline volatile unsigned int* error_record_host() {
  static unsigned int* host_rec[64] = {nullptr};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  if (host_rec[dev] == nullptr) {
    unsigned int* h = nullptr;
    unsigned int* d = nullptr;
    if (cudaHostAlloc(reinterpret_cast<void**>(&h), 4 * sizeof(unsigned int), cudaHostAllocMapped) != cudaSuccess) return nullptr;
    h[0] = h[1] = h[2] = h[3] = 0u;
    if (cudaHostGetDevicePointer(reinterpret_cast<void**>(&d), h, 0) != cudaSuccess ||
        cudaMemcpyToSymbol(g_dev_error_ptr, &d, sizeof(d)) != cudaSuccess) {
      cudaFreeHost(h);
      return nullptr;
    }
    host_rec[dev] = h;
  }
  return host_rec[dev];
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch (kernels launched with launch_pdl(), gramhead.cu): the next kernel of a chain may
// start -- run its prologue, become resident -- while this one is still executing; pdl_wait() blocks until every
// prerequisite grid has completed and its memory is visible. Every thread calls pdl_wait() before it touches global
// memory a predecessor wrote (or will read: a successor never writes before its own wait).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done != 0;
}
#ifndef GH_WAIT_TIMEOUT_NS
#define GH_WAIT_TIMEOUT_NS 4000000000ull   // 4 s: far beyond any legitimate wait in these kernels
#endif
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, uint32_t site) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = globaltimer_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ffu) == 0u && globaltimer_ns() - t0 > GH_WAIT_TIMEOUT_NS) dev_fail(1u, site);
  }
}

// Generic-proxy writes (st.shared) -> async-proxy readers (tcgen05.mma, TMA store).
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// Barrier among a subset of the CTA's warps (nthreads a multiple of 32); id 0 is __syncthreads'.
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------------------------------------
// tcgen05: TMEM allocation, fences, MMA, commit, load
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// Whole warp. Writes the TMEM base address to *dst_smem.
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]^T ; one thread issues on behalf of the CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrives on `bar` once every tcgen05.mma issued so far by this thread has finished.
// (implies tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread = lane/row).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// Same load without the wait, so that several can be in flight; call tmem_ld_wait() before touching the registers.
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// Descriptors. Operand tiles live in smem as [rows][64] bf16, K-major, SWIZZLE_128B:
//   byte(r, k) = (r/8)*1024 + (r%8)*128 + (((k/8) ^ (r%8)) * 16) + (k%8)*2      (tile base 1024-aligned)
// One UMMA consumes K=16 (32 bytes of each row); stepping K inside the 128-byte row is a plain
// +32 B on the descriptor start address (the hardware applies the XOR on the address bits).
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kTileK = 64;            // bf16 elements per smem row (= one 128 B swizzle row)
constexpr uint32_t kRowBytes = 128;
constexpr uint32_t kAtomBytes = 1024;      // 8 rows
constexpr uint32_t kUmmaK = 16;

__host__ __device__ constexpr uint64_t make_smem_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4)        // start address  [0,14)
         | ((uint64_t)1 << 16)                          // LBO (unused for swizzled K-major) [16,30)
         | ((uint64_t)(kAtomBytes >> 4) << 32)          // SBO = 1024 B between 8-row groups [32,46)
         | ((uint64_t)1 << 46)                          // descriptor version 1 (sm_100)     [46,48)
         | ((uint64_t)2 << 61);                         // SWIZZLE_128B                      [61,64)
}
// kind::f16, A=B=bf16, D=fp32, both operands K-major, dense.
__host__ __device__ constexpr uint32_t make_idesc_bf16(uint32_t m, uint32_t n) {
  return (1u << 4)            // D format f32
         | (1u << 7)          // A format bf16
         | (1u << 10)         // B format bf16
         | ((n >> 3) << 17)   // N
         | ((m >> 4) << 24);  // M
}
// Byte offset of the 8-byte group holding elements k..k+3 (k % 4 == 0) of row r inside a tile.
__device__ __forceinline__ uint32_t sw128_off(uint32_t r, uint32_t k) {
  return (r >> 3) * kAtomBytes + (r & 7u) * kRowBytes + ((((k >> 3) ^ r) & 7u) << 4) + ((k & 7u) << 1);
}
// kind::tf32, D = fp32, both operands K-major, dense.
__host__ __device__ constexpr uint32_t make_idesc_tf32(uint32_t m, uint32_t n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}
// K-major, SWIZZLE_NONE: 8-row x 16 B core matrices, SBO between 8-row groups, LBO between the two k-chunks.
__host__ __device__ constexpr uint64_t make_smem_desc_noswz(uint32_t addr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | ((uint64_t)1 << 46);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ uint32_t tf32_rna(float f) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(f));
  return r;
}

// ---------------------------------------------------------------------------------------------
// Small memory helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 ldg_stream_f4(const float* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::128B.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ uint2 ldg_stream_u2(const void* p) {
  uint2 v;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
  return v;
}
__device__ __forceinline__ void sts_u2(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void sts_u4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ void red_add_f32(float* p, float v) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

}  // namespace gh
