// Style-transfer loss on the dense Gram (SURVEY.md section 8(f) n3): mse_loss(G(x), G*) and its gradient w.r.t. G in one
// pass. Reference: functions/functions_RESNET50_Truncate_Gram_Attention.py:286-301 -- `loss = mse_loss(noise_gram,
// original_gram); loss.backward()` -- i.e. loss = mean((G - G*)^2) over all B*C*C entries and, through autograd,
// dG = 2 (G - G*) / (B C C), then dF = (dG + dG^T) F / HW = 4 (G - G*) F / (B C^2 HW) through the Gram backward.
// The forward Gram comes from gh_gram_dense_fwd (split over K at batch 1, so the difference cannot live in its
// epilogue); this kernel reads G and G* once and writes dG and per-block partial sums of the squared difference, which
// replaces the subtract / square / mean kernels of the forward and the three element-wise kernels of their backward.
#pragma once
#include "common.cuh"

namespace gh {

constexpr int kMseThreads = 256;
constexpr int kMseMaxBlocks = 1024;      // partial sums (the caller adds them up in a fixed order)

// partial[blockIdx.x] = sum over this block's elements of (G - Gt)^2 * inv_n ;  dG = 2 * inv_n * (G - Gt).
// float4 steps over the first 4 * (n / 4) elements; the n % 4 left (B*C*C with odd C and B) are block 0's.
__global__ void __launch_bounds__(kMseThreads) gram_mse_kernel(const float* __restrict__ G, const float* __restrict__ Gt,
                                                               float* __restrict__ dG, float* __restrict__ partial,
                                                               long long n, float inv_n) {
  __shared__ float red[kMseThreads / 32];
  float acc = 0.f;
  const float coef = 2.f * inv_n;
  const long long n4 = n >> 2;
  for (long long i = (long long)blockIdx.x * kMseThreads + threadIdx.x; i < n4; i += (long long)gridDim.x * kMseThreads) {
    const float4 a = *reinterpret_cast<const float4*>(G + 4 * i);
    const float4 b = *reinterpret_cast<const float4*>(Gt + 4 * i);
    const float4 d = make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w);
    acc = fmaf(d.x, d.x, fmaf(d.y, d.y, fmaf(d.z, d.z, fmaf(d.w, d.w, acc))));
    *reinterpret_cast<float4*>(dG + 4 * i) = make_float4(coef * d.x, coef * d.y, coef * d.z, coef * d.w);
  }
  if (blockIdx.x == 0 && threadIdx.x < (int)(n - 4 * n4)) {
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
    partial[blockIdx.x] = t * inv_n;
  }
}

}  // namespace gh
