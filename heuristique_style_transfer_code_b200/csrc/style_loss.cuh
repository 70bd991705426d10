// Style-transfer loss on the dense Gram (SURVEY.md section 8(f) n3): mse_loss(G(x), G*) and its gradient w.r.t. G in one
// pass. Reference: functions/functions_RESNET50_Truncate_Gram_Attention.py:286-301 -- `loss = mse_loss(noise_gram,
// original_gram); loss.backward()` -- i.e. loss = mean((G - G*)^2) over all B*C*C entries and, through autograd,
// dG = 2 (G - G*) / (B C C), then dF = (dG + dG^T) F / HW = 4 (G - G*) F / (B C^2 HW) through the Gram backward.
// The forward Gram comes from gh_gram_dense_fwd (split over K at batch 1, so the difference cannot live in its
// epilogue); this kernel reads G and G* once and writes dG and per-block partial sums of the squared difference, which
// replaces the subtract / square / mean kernels of the forward and the three element-wise kernels of their backward.
//
// gram_mse_images_kernel is the same pass with one loss per image (several style-transfer images optimised in one step):
// grid (k, B), and image b's k blocks run exactly the per-block code gram_mse_kernel runs on that image alone, so its
// partials and dG are bitwise those of a batch-1 call.
#pragma once
#include "common.cuh"

namespace gh {

constexpr int kMseThreads = 256;
constexpr int kMseMaxBlocks = 1024;      // partial sums (the caller adds them up in a fixed order)

// Block `block` of `nblocks` over the n elements at G / Gt / dG:
//   *partial = sum over this block's elements of (G - Gt)^2 * inv_n ;  dG = 2 * inv_n * (G - Gt).
// Steps of four elements over the first 4 * (n / 4), block-strided; the n % 4 left are block 0's. kVec: one float4 per
// operand (16 B-aligned G, Gt, dG); otherwise four scalar loads and stores with the same fma chain, so both give the
// same bits.
template <bool kVec>
__device__ __forceinline__ void gram_mse_block(const float* __restrict__ G, const float* __restrict__ Gt,
                                               float* __restrict__ dG, float* __restrict__ partial, long long n,
                                               float inv_n, int block, int nblocks) {
  __shared__ float red[kMseThreads / 32];
  float acc = 0.f;
  const float coef = 2.f * inv_n;
  const long long n4 = n >> 2;
  for (long long i = (long long)block * kMseThreads + threadIdx.x; i < n4; i += (long long)nblocks * kMseThreads) {
    float4 a, b;
    if constexpr (kVec) {
      a = *reinterpret_cast<const float4*>(G + 4 * i);
      b = *reinterpret_cast<const float4*>(Gt + 4 * i);
    } else {
      a = make_float4(G[4 * i], G[4 * i + 1], G[4 * i + 2], G[4 * i + 3]);
      b = make_float4(Gt[4 * i], Gt[4 * i + 1], Gt[4 * i + 2], Gt[4 * i + 3]);
    }
    const float4 d = make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w);
    acc = fmaf(d.x, d.x, fmaf(d.y, d.y, fmaf(d.z, d.z, fmaf(d.w, d.w, acc))));
    const float4 g = make_float4(coef * d.x, coef * d.y, coef * d.z, coef * d.w);
    if constexpr (kVec) {
      *reinterpret_cast<float4*>(dG + 4 * i) = g;
    } else {
      dG[4 * i] = g.x; dG[4 * i + 1] = g.y; dG[4 * i + 2] = g.z; dG[4 * i + 3] = g.w;
    }
  }
  if (block == 0 && threadIdx.x < (int)(n - 4 * n4)) {
    const long long i = 4 * n4 + threadIdx.x;
    const float d = G[i] - Gt[i];
    acc = fmaf(d, d, acc);
    dG[i] = coef * d;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < kMseThreads / 32; ++i) t += red[i];
    *partial = t * inv_n;
  }
}

// n = B*C*C elements, one loss: partial[blockIdx.x].
__global__ void __launch_bounds__(kMseThreads) gram_mse_kernel(const float* __restrict__ G, const float* __restrict__ Gt,
                                                               float* __restrict__ dG, float* __restrict__ partial,
                                                               long long n, float inv_n) {
  gram_mse_block<true>(G, Gt, dG, partial + blockIdx.x, n, inv_n, blockIdx.x, gridDim.x);
}

// gridDim.y images of n_img = C*C elements each, one loss per image: partial[blockIdx.y * gridDim.x + blockIdx.x].
// Image b starts at b * n_img, which is 16 B-aligned only when n_img % 4 == 0 (and the bases are): misaligned images take
// the scalar loads. The choice is per image, hence uniform over a block.
__global__ void __launch_bounds__(kMseThreads) gram_mse_images_kernel(const float* __restrict__ G,
                                                                      const float* __restrict__ Gt,
                                                                      float* __restrict__ dG, float* __restrict__ partial,
                                                                      long long n_img, float inv_n) {
  const long long off = (long long)blockIdx.y * n_img;
  const float* g = G + off;
  const float* gt = Gt + off;
  float* dg = dG + off;
  float* p = partial + (long long)blockIdx.y * gridDim.x + blockIdx.x;
  if (((uintptr_t)g | (uintptr_t)gt | (uintptr_t)dg) % 16 == 0) gram_mse_block<true>(g, gt, dg, p, n_img, inv_n, blockIdx.x, gridDim.x);
  else gram_mse_block<false>(g, gt, dg, p, n_img, inv_n, blockIdx.x, gridDim.x);
}

}  // namespace gh
