// Per-image and per-column pieces of the attention head around the TMA-fed GEMMs of tgemm_pair.cuh.
//
// Reference: nn.MultiheadAttention(embed_dim = g*g, num_heads = 1)(X, X, X), .mean(dim=0), nn.Linear
// (Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:56-61 / :108-114); math in SURVEY.md Appendix A.
// Every tensor that feeds a GEMM is written here directly as split-bf16 planes (hi = bf16(x), lo = bf16(x - hi),
// `plane` elements apart), so no separate cast pass runs between the kernels:
//   split_bf16_kernel        X (or a weight matrix) fp32 -> planes
//   attn2_core_fwd_kernel    scores, softmax over keys, Obar = mean_l sum_m A[l][m] V[m]  -> probs, Obar planes; zeroes emb
//   attn2_bwd_prep_kernel    demb = dlogits W_c (+ external gradient) -> planes; db_out, dW_c, db_c (fixed summation
//                            order); zeroes the buffers later kernels accumulate into
//   attn2_core_bwd_kernel    softmax / score backward -> dQKV planes; db_in; zeroes the K-split GEMM outputs
#pragma once
#include "common.cuh"
#include "attn_head.cuh"
#include "launch.cuh"

namespace gh {

__device__ __forceinline__ void split2(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

// planes[0 .. n) = hi, planes[plane .. plane + n) = lo. n % 4 == 0, 16 B aligned src, 8 B aligned planes.
__global__ void __launch_bounds__(256) split_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ planes,
                                                         long long n4, long long plane) {
  pdl_launch_dependents();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = ldg_stream_f4(src + 4 * i);
    const __nv_bfloat162 h01 = __floats2bfloat162_rn(v.x, v.y), h23 = __floats2bfloat162_rn(v.z, v.w);
    const float2 f01 = __bfloat1622float2(h01), f23 = __bfloat1622float2(h23);
    uint2 hi, lo;
    hi.x = *reinterpret_cast<const uint32_t*>(&h01);
    hi.y = *reinterpret_cast<const uint32_t*>(&h23);
    lo.x = pack_bf16x2(v.x - f01.x, v.y - f01.y);
    lo.y = pack_bf16x2(v.z - f23.x, v.w - f23.y);
    *reinterpret_cast<uint2*>(planes + 4 * i) = hi;
    *reinterpret_cast<uint2*>(planes + plane + 4 * i) = lo;
  }
}

// A list of fp32 buffers a kernel zeroes on the side (outputs that later kernels in the stream accumulate into).
struct ZeroList {
  float* ptr[3];
  long long n4[3];       // float4 counts (buffers are 16 B aligned, lengths multiples of 4)
};
__device__ __forceinline__ void zero_buffers(const ZeroList& z, long long tid, long long nthreads) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    if (z.ptr[i] == nullptr) continue;
    float4* p = reinterpret_cast<float4*>(z.ptr[i]);
    for (long long j = tid; j < z.n4[i]; j += nthreads) p[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// ---------------------------------------------------------------------------------------------
// Per-image kernels. One CTA of kAttn2Threads threads per image; thread t owns the four consecutive embedding
// coordinates e = 4t .. 4t+3 of every token (E <= 4 * kAttn2Threads), so all of a thread's loads are independent 16 B
// loads issued before the first use: at E = 1024 an image is 36 KB of Q/K/V and the kernels are bandwidth-, not
// latency-bound.
// ---------------------------------------------------------------------------------------------
constexpr int kAttn2Threads = 256;
constexpr int kAttn2Warps = kAttn2Threads / 32;

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float dot4(const float4& a, const float4& b) {
  return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w)));
}
__device__ __forceinline__ void store_planes4(__nv_bfloat16* hi_ptr, long long plane, const float4& v) {
  const __nv_bfloat162 h01 = __floats2bfloat162_rn(v.x, v.y), h23 = __floats2bfloat162_rn(v.z, v.w);
  const float2 f01 = __bfloat1622float2(h01), f23 = __bfloat1622float2(h23);
  uint2 hi, lo;
  hi.x = *reinterpret_cast<const uint32_t*>(&h01);
  hi.y = *reinterpret_cast<const uint32_t*>(&h23);
  lo.x = pack_bf16x2(v.x - f01.x, v.y - f01.y);
  lo.y = pack_bf16x2(v.z - f23.x, v.w - f23.y);
  *reinterpret_cast<uint2*>(hi_ptr) = hi;
  *reinterpret_cast<uint2*>(hi_ptr + plane) = lo;
}
// Sum of NV per-thread values over the CTA, in a fixed order; result in out[0..NV) (shared), valid after the call.
template <int NV>
__device__ __forceinline__ void block_sum_vec(float (&v)[NV], float (*red)[NV], float* out) {
  const int w = threadIdx.x >> 5, ln = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    float x = v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (ln == 0) red[w][i] = x;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < kAttn2Warps; ++i) t += red[i][threadIdx.x];
    out[threadIdx.x] = t;
  }
  __syncthreads();
}

// QKV: (B*L, 3E) rows ordered b*L + l. Writes probs (B, L, L), the Obar planes (B, E) and zeroes emb[b] when the
// out_proj GEMM accumulates two K partitions into it. E % 4 == 0, E <= 4 * kAttn2Threads.
template <int LT>
__global__ void __launch_bounds__(kAttn2Threads) attn2_core_fwd_kernel(const float* __restrict__ QKV, float* __restrict__ probs,
                                                                        __nv_bfloat16* __restrict__ obar, long long obar_plane,
                                                                        float* __restrict__ emb_zero, int L, int E) {
  __shared__ float red[kAttn2Warps][LT * LT];
  __shared__ float sc[LT * LT];
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.x;
  const int e = threadIdx.x * 4;
  const bool ok = e < E;
  const float* base = QKV + (long long)b * L * 3 * E + e;
  const float inv_sqrt_e = rsqrtf((float)E);
  float4 q[LT], k[LT], v[LT];
#pragma unroll
  for (int l = 0; l < LT; ++l) {
    const bool ld = ok && l < L;
    q[l] = ld ? ld4(base + (long long)l * 3 * E) : make_float4(0.f, 0.f, 0.f, 0.f);
    k[l] = ld ? ld4(base + (long long)l * 3 * E + E) : make_float4(0.f, 0.f, 0.f, 0.f);
    v[l] = ld ? ld4(base + (long long)l * 3 * E + 2 * E) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float acc[LT * LT];
#pragma unroll
  for (int l = 0; l < LT; ++l) {
    // torch scales q before the product
    const float4 qs = make_float4(q[l].x * inv_sqrt_e, q[l].y * inv_sqrt_e, q[l].z * inv_sqrt_e, q[l].w * inv_sqrt_e);
#pragma unroll
    for (int m = 0; m < LT; ++m) acc[l * LT + m] = dot4(qs, k[m]);
  }
  block_sum_vec<LT * LT>(acc, red, sc);
  if (threadIdx.x < L) {
    const int l = threadIdx.x;
    float mx = -INFINITY;
    for (int m = 0; m < L; ++m) mx = fmaxf(mx, sc[l * LT + m]);
    float den = 0.f;
    for (int m = 0; m < L; ++m) den += expf(sc[l * LT + m] - mx);
    for (int m = 0; m < L; ++m) {
      const float pr = expf(sc[l * LT + m] - mx) / den;
      sc[l * LT + m] = pr;
      probs[((long long)b * L + l) * L + m] = pr;
    }
  }
  __syncthreads();
  if (!ok) return;
  // Obar[e] = (1/L) sum_l sum_m A[l][m] V[m][e] = sum_m (mean_l A[l][m]) V[m][e]
  float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int m = 0; m < LT; ++m) {
    if (m < L) {
      float a = 0.f;
      for (int l = 0; l < L; ++l) a += sc[l * LT + m];
      const float wm = a / (float)L;
      o.x = fmaf(wm, v[m].x, o.x); o.y = fmaf(wm, v[m].y, o.y); o.z = fmaf(wm, v[m].z, o.z); o.w = fmaf(wm, v[m].w, o.w);
    }
  }
  store_planes4(obar + (long long)b * E + e, obar_plane, o);
  if (emb_zero) *reinterpret_cast<float4*>(emb_zero + (long long)b * E + e) = make_float4(0.f, 0.f, 0.f, 0.f);
}

// logits[b][c] = <emb[b], W_c[c]> + b_c[c]: one warp per image, all classes at once, 16 B loads issued up front.
// E % 4 == 0, E <= 1024, nc <= kAttn2MaxNc.
constexpr int kAttn2MaxNc = 16;
__global__ void __launch_bounds__(128) attn2_classifier_kernel(const float* __restrict__ emb, const float* __restrict__ Wc,
                                                               const float* __restrict__ bc, float* __restrict__ logits,
                                                               int B, int E, int nc) {
  const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  pdl_launch_dependents();
  pdl_wait();
  if (b >= B) return;
  float4 x[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int e = (lane + 32 * i) * 4;
    x[i] = e < E ? ld4(emb + (long long)b * E + e) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (int c = 0; c < nc; ++c) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int e = (lane + 32 * i) * 4;
      if (e < E) s += dot4(x[i], __ldg(reinterpret_cast<const float4*>(Wc + (long long)c * E + e)));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) logits[(long long)b * nc + c] = s + (bc ? bc[c] : 0.f);
  }
}

// demb = d_logits W_c (+ d_emb_ext) as planes; db_out = colsum(demb); dW_c = d_logits^T emb; db_c = colsum(d_logits).
// grid (ceil(E / 128), kPrepSplit) in clusters of kPrepSplit CTAs along y: a cluster owns 128 columns (thread = 4
// consecutive columns x one of 8 row groups), its CTA r the rows b = r + kPrepSplit * (g + 8 i). The column sums are
// reduced across the row groups in shared memory and across the cluster through distributed shared memory, both in a
// fixed order: no atomics, bitwise reproducible. Dynamic shared memory: attn2_prep_smem_bytes(nc).
constexpr int kPrepSplit = 8;
constexpr int kPrepThreads = 256;
inline size_t attn2_prep_smem_bytes(int nc) {
  const size_t nq = 1 + (size_t)nc;
  return (nq * 8 * 128 + kPrepSplit * nq * 128 + kPrepSplit * kAttn2MaxNc + 8 * kAttn2MaxNc) * sizeof(float);
}
__device__ __forceinline__ void st_cluster_f32(const float* local_ptr, uint32_t rank, float v) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(local_ptr)), "r"(rank));
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(remote), "f"(v) : "memory");
}
__global__ void __cluster_dims__(1, kPrepSplit, 1) __launch_bounds__(kPrepThreads)
    attn2_bwd_prep_kernel(const float* __restrict__ d_logits, const float* __restrict__ d_emb_ext, const float* __restrict__ Wc,
                          const float* __restrict__ emb, __nv_bfloat16* __restrict__ demb, long long demb_plane,
                          float* __restrict__ db_out, float* __restrict__ dWc, float* __restrict__ db_c, int B, int E, int nc,
                          ZeroList zl) {
  extern __shared__ float prep_smem[];
  pdl_launch_dependents();
  pdl_wait();
  const int nq = 1 + nc;                                           // quantity 0 = db_out, 1 + c = row c of dW_c
  float* part = prep_smem;                                         // [nq][8 row groups][128 columns]
  float* gather = part + nq * 8 * 128;                             // [kPrepSplit][nq][128]   (used on cluster rank 0)
  float* gather_c = gather + kPrepSplit * nq * 128;                // [kPrepSplit][kAttn2MaxNc] (rank 0, column block 0)
  float* dbc_part = gather_c + kPrepSplit * kAttn2MaxNc;           // [8][kAttn2MaxNc]
  const int tx = threadIdx.x & 31, g = threadIdx.x >> 5;           // 32 threads x 4 columns, 8 row groups
  const int e = blockIdx.x * 128 + tx * 4;
  const bool ok = e < E;
  const uint32_t rank = blockIdx.y;                                // cluster rank (cluster dims (1, kPrepSplit, 1), gridDim.y = kPrepSplit)
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 wc[kAttn2MaxNc], dwc[kAttn2MaxNc];
#pragma unroll
  for (int c = 0; c < kAttn2MaxNc; ++c) {
    wc[c] = (ok && c < nc) ? __ldg(reinterpret_cast<const float4*>(Wc + (long long)c * E + e)) : zero4;
    dwc[c] = zero4;
  }
  float4 csum = zero4;
  float dbc = 0.f;                                                 // lane tx < nc: partial db_c[tx] over this warp's rows
  // four rows per trip: their eight 16 B loads are in flight together
  constexpr int kRowStep = kPrepSplit * 8;
  for (int b0 = (int)rank + kPrepSplit * g; b0 < B; b0 += 4 * kRowStep) {
    float4 d[4], ev[4];
    float my_dl[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int b = b0 + r * kRowStep;
      const bool row = b < B;
      d[r] = (ok && row && d_emb_ext) ? ld4(d_emb_ext + (long long)b * E + e) : zero4;
      ev[r] = (ok && row) ? ld4(emb + (long long)b * E + e) : zero4;
      my_dl[r] = (row && tx < nc) ? __ldg(d_logits + (long long)b * nc + tx) : 0.f;
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int b = b0 + r * kRowStep;
      dbc += my_dl[r];
#pragma unroll
      for (int c = 0; c < kAttn2MaxNc; ++c) {
        if (c < nc) {
          const float dl = __shfl_sync(0xffffffffu, my_dl[r], c);
          d[r].x = fmaf(dl, wc[c].x, d[r].x); d[r].y = fmaf(dl, wc[c].y, d[r].y);
          d[r].z = fmaf(dl, wc[c].z, d[r].z); d[r].w = fmaf(dl, wc[c].w, d[r].w);
          dwc[c].x = fmaf(dl, ev[r].x, dwc[c].x); dwc[c].y = fmaf(dl, ev[r].y, dwc[c].y);
          dwc[c].z = fmaf(dl, ev[r].z, dwc[c].z); dwc[c].w = fmaf(dl, ev[r].w, dwc[c].w);
        }
      }
      if (ok && b < B) store_planes4(demb + (long long)b * E + e, demb_plane, d[r]);
      csum.x += d[r].x; csum.y += d[r].y; csum.z += d[r].z; csum.w += d[r].w;
    }
  }
  *reinterpret_cast<float4*>(part + (0 * 8 + g) * 128 + tx * 4) = csum;
#pragma unroll
  for (int c = 0; c < kAttn2MaxNc; ++c)
    if (c < nc) *reinterpret_cast<float4*>(part + ((1 + c) * 8 + g) * 128 + tx * 4) = dwc[c];
  if (tx < kAttn2MaxNc) dbc_part[g * kAttn2MaxNc + tx] = dbc;
  __syncthreads();
  // this CTA's sums over its 8 row groups -> slot `rank` of the arrays in cluster rank 0's shared memory
  for (int i = threadIdx.x; i < nq * 128; i += kPrepThreads) {
    const int qn = i >> 7, col = i & 127;
    float t = 0.f;
#pragma unroll
    for (int gg = 0; gg < 8; ++gg) t += part[(qn * 8 + gg) * 128 + col];
    st_cluster_f32(gather + ((int)rank * nq + qn) * 128 + col, 0u, t);
  }
  if (threadIdx.x < nc) {
    float t = 0.f;
#pragma unroll
    for (int gg = 0; gg < 8; ++gg) t += dbc_part[gg * kAttn2MaxNc + threadIdx.x];
    st_cluster_f32(gather_c + (int)rank * kAttn2MaxNc + threadIdx.x, 0u, t);
  }
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  if (rank == 0) {
    for (int i = threadIdx.x; i < nq * 128; i += kPrepThreads) {
      const int qn = i >> 7, col = i & 127;
      const int ee = blockIdx.x * 128 + col;
      float t = 0.f;
#pragma unroll
      for (int r = 0; r < kPrepSplit; ++r) t += gather[(r * nq + qn) * 128 + col];
      if (ee < E) {
        if (qn == 0) { if (db_out) db_out[ee] = t; }
        else if (dWc) dWc[(long long)(qn - 1) * E + ee] = t;
      }
    }
    if (blockIdx.x == 0 && db_c && threadIdx.x < nc) {
      float t = 0.f;
#pragma unroll
      for (int r = 0; r < kPrepSplit; ++r) t += gather_c[r * kAttn2MaxNc + threadIdx.x];
      db_c[threadIdx.x] = t;
    }
  }
  zero_buffers(zl, ((long long)blockIdx.y * gridDim.x + blockIdx.x) * kPrepThreads + threadIdx.x,
               (long long)gridDim.x * gridDim.y * kPrepThreads);
}

// Backward of the per-image core; one CTA per image. dObar: (B, E) fp32. Writes the dQKV planes (B*L, 3E) and the
// image's contribution to db_in (3E, zeroed earlier in the stream; the order of the contributions is not fixed) -- the
// latter from a persistent grid: CTA i takes the images i, i + gridDim.x, ... and adds its column sums once.
template <int LT>
__global__ void __launch_bounds__(kAttn2Threads) attn2_core_bwd_kernel(const float* __restrict__ QKV, const float* __restrict__ probs,
                                                                        const float* __restrict__ dobar,
                                                                        __nv_bfloat16* __restrict__ dQKV, long long dqkv_plane,
                                                                        float* __restrict__ db_in, int B, int L, int E,
                                                                        ZeroList zl) {
  __shared__ float red[kAttn2Warps][LT];
  __shared__ float sdAv[LT];
  __shared__ float sA[LT * LT];
  __shared__ float sdS[LT * LT];
  pdl_launch_dependents();
  pdl_wait();
  const int e = threadIdx.x * 4;
  const bool ok = e < E;
  const float inv_l = 1.f / (float)L;
  const float inv_sqrt_e = rsqrtf((float)E);
  float4 bq = make_float4(0.f, 0.f, 0.f, 0.f), bk = bq, bv = bq;
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);

  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const float* base = QKV + (long long)b * L * 3 * E + e;
    __nv_bfloat16* dbase = dQKV + (long long)b * L * 3 * E + e;
    float4 q[LT], k[LT], v[LT];
#pragma unroll
    for (int l = 0; l < LT; ++l) {
      const bool ld = ok && l < L;
      q[l] = ld ? ld4(base + (long long)l * 3 * E) : zero4;
      k[l] = ld ? ld4(base + (long long)l * 3 * E + E) : zero4;
      v[l] = ld ? ld4(base + (long long)l * 3 * E + 2 * E) : zero4;
    }
    const float4 dO = ok ? ld4(dobar + (long long)b * E + e) : zero4;
    __syncthreads();                                        // the previous image's shared tables are no longer read
    if (threadIdx.x < L * L) {
      const int l = threadIdx.x / L, m = threadIdx.x % L;
      sA[l * LT + m] = probs[((long long)b * L + l) * L + m];
    }
    // dA[l][m] = <dO[l], V[m]> with dO[l] = dObar / L for every l  -> depends on m only
    float dav[LT];
#pragma unroll
    for (int m = 0; m < LT; ++m) dav[m] = dot4(dO, v[m]);
    block_sum_vec<LT>(dav, red, sdAv);
    if (threadIdx.x < L) {
      const int l = threadIdx.x;
      float dot = 0.f;
      for (int m = 0; m < L; ++m) dot += __fmul_rn(sdAv[m], inv_l) * sA[l * LT + m];
      // dA[m] - dot rounded once, not contracted into an FMA: on a one-hot row (scores of 1e4 and more) the two are
      // equal and the difference must be exactly 0, not the product's rounding error scaled by the size of the scores
      for (int m = 0; m < L; ++m) sdS[l * LT + m] = sA[l * LT + m] * (__fmul_rn(sdAv[m], inv_l) - dot) * inv_sqrt_e;
    }
    __syncthreads();
    if (ok) {
#pragma unroll
      for (int l = 0; l < LT; ++l) {
        if (l < L) {
          float4 dq = zero4, dk = zero4;
          float colA = 0.f;
#pragma unroll
          for (int m = 0; m < LT; ++m) {
            if (m < L) {
              const float s1 = sdS[l * LT + m], s2 = sdS[m * LT + l];
              dq.x = fmaf(s1, k[m].x, dq.x); dq.y = fmaf(s1, k[m].y, dq.y); dq.z = fmaf(s1, k[m].z, dq.z); dq.w = fmaf(s1, k[m].w, dq.w);
              dk.x = fmaf(s2, q[m].x, dk.x); dk.y = fmaf(s2, q[m].y, dk.y); dk.z = fmaf(s2, q[m].z, dk.z); dk.w = fmaf(s2, q[m].w, dk.w);
              colA += sA[m * LT + l];
            }
          }
          colA *= inv_l;                                    // dV[l] = sum_i A[i][l] dO[i] = colA[l] * dObar
          const float4 dv = make_float4(colA * dO.x, colA * dO.y, colA * dO.z, colA * dO.w);
          __nv_bfloat16* row = dbase + (long long)l * 3 * E;
          store_planes4(row, dqkv_plane, dq);
          store_planes4(row + E, dqkv_plane, dk);
          store_planes4(row + 2 * E, dqkv_plane, dv);
          bq.x += dq.x; bq.y += dq.y; bq.z += dq.z; bq.w += dq.w;
          bk.x += dk.x; bk.y += dk.y; bk.z += dk.z; bk.w += dk.w;
          bv.x += dv.x; bv.y += dv.y; bv.z += dv.z; bv.w += dv.w;
        }
      }
    }
  }
  if (db_in && ok) {
    red_add_f32(db_in + e, bq.x); red_add_f32(db_in + e + 1, bq.y); red_add_f32(db_in + e + 2, bq.z); red_add_f32(db_in + e + 3, bq.w);
    red_add_f32(db_in + E + e, bk.x); red_add_f32(db_in + E + e + 1, bk.y); red_add_f32(db_in + E + e + 2, bk.z); red_add_f32(db_in + E + e + 3, bk.w);
    red_add_f32(db_in + 2 * E + e, bv.x); red_add_f32(db_in + 2 * E + e + 1, bv.y); red_add_f32(db_in + 2 * E + e + 2, bv.z); red_add_f32(db_in + 2 * E + e + 3, bv.w);
  }
  zero_buffers(zl, (long long)blockIdx.x * kAttn2Threads + threadIdx.x, (long long)gridDim.x * kAttn2Threads);
}

}  // namespace gh
