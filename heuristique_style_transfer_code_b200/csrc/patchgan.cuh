// Gram head of the Multi-PatchGAN discriminator (SURVEY 8(f) n4; reference Models/Models_Multi_PatchGAN.py:198-256).
//
//   patch_pool_kernel      one warp per (image, collected layer, channel) plane: a single pass over the projected
//                          feature maps produces the 4x4 adaptive-average bins of every channel and the per-channel
//                          sum / sum of squares the folded-in :198 layer norm needs. HBM-bound: every map is read once
//                          (the reference reads it for layer_norm, writes it, reads it again for the pooling).
//   patch_gram_kernel      one CTA per (image, layer): whole-map layer norm applied to the 16 bin means, layer norm
//                          over (D, 4, 4), the D x D Gram over the 16 positions, its Frobenius norm.
//   patch_attention_kernel the two 8-head nn.MultiheadAttention layers over the L stacked layer tokens, the mean over
//                          layers and the classifier, one image at a time per CTA; every intermediate stays in shared
//                          memory (L <= 8 tokens of ndf <= 128 features), weights come through L1/L2.
// The Linear(D*D -> ndf) between the two is the tcgen05 split-bf16 GEMM (gh_gemm_f32) over all L*B Gram rows at once.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gh {

constexpr int kPatchMaxLayers = 8;
constexpr int kPatchPool = 4;
constexpr int kPatchBins = kPatchPool * kPatchPool;   // 16 positions per channel after pooling
constexpr int kPatchMaxD = 128;
constexpr int kPatchThreads = 256;

struct PatchLayer {
  const float* x;
  int H, W;
  long long s_img, s_c, s_y, s_x;   // element strides (NCHW: C*H*W, H*W, W, 1)
};

struct PatchGramParams {
  PatchLayer layer[kPatchMaxLayers];
  int L, B, D;
  int ln_input;        // 1: apply F.layer_norm(x, x.shape[1:]) (:198) to the map before pooling
  float* gram;         // (L, B, D*D)
  float* gram_norm;    // (L, B)
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// sum over the CTA of one double per thread; result broadcast to every thread. red: >= 32 doubles of shared memory.
__device__ __forceinline__ double block_sum(double v, double* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double t = (lane < (int)(blockDim.x >> 5)) ? red[lane] : 0.0;
  t = warp_sum(t);
  return t;
}

// ---- pass over the maps: one warp per (image, layer, channel) plane ---------------------------------------------------
// Fast path (rows contiguous, W <= 32*KMAX): lane <-> fixed columns x = lane + 32k, so a lane's column-bin membership is
// a constant mask; rows are walked in segments over which the row-bin membership is constant, and inside a segment the
// inner loop is one load, one add and one fma per element. Column sums are folded into the 16 bins once per segment.
template <int KMAX>
__device__ __forceinline__ void pool_plane_rows(const float* __restrict__ plane, int H, int W, long long s_y,
                                                const int* ys, const int* ye, const int* xs, const int* xe,
                                                float* acc, float& sum, float& sq) {
  const int lane = threadIdx.x & 31;
  unsigned colmask[KMAX];
  float colsum[KMAX];
  float rowacc[kPatchPool][KMAX];
#pragma unroll
  for (int i = 0; i < kPatchPool; ++i)
#pragma unroll
    for (int k = 0; k < KMAX; ++k) rowacc[i][k] = 0.f;
#pragma unroll
  for (int k = 0; k < KMAX; ++k) {
    const int x = lane + 32 * k;
    unsigned m = 0;
#pragma unroll
    for (int j = 0; j < kPatchPool; ++j) m |= (x >= xs[j] && x < xe[j] && x < W) ? (1u << j) : 0u;
    colmask[k] = m;
    colsum[k] = 0.f;
  }
  int y = 0;
  while (y < H) {
    unsigned rm = 0;
#pragma unroll
    for (int i = 0; i < kPatchPool; ++i) rm |= (y >= ys[i] && y < ye[i]) ? (1u << i) : 0u;
    int yend = H;                                     // the segment ends at the next bin boundary above y
#pragma unroll
    for (int i = 0; i < kPatchPool; ++i) {
      if (ys[i] > y && ys[i] < yend) yend = ys[i];
      if (ye[i] > y && ye[i] < yend) yend = ye[i];
    }
    for (int yy = y; yy < yend; yy += 4) {
      float v[4][KMAX];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const float* row = plane + (long long)(yy + r) * s_y;
#pragma unroll
        for (int k = 0; k < KMAX; ++k) {
          const int x = lane + 32 * k;
          v[r][k] = (yy + r < yend && x < W) ? __ldg(row + x) : 0.f;
        }
      }
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int k = 0; k < KMAX; ++k) {
          colsum[k] += v[r][k];
          sq = fmaf(v[r][k], v[r][k], sq);
        }
    }
#pragma unroll
    for (int i = 0; i < kPatchPool; ++i)
      if ((rm >> i) & 1u) {                            // warp-uniform
#pragma unroll
        for (int k = 0; k < KMAX; ++k) rowacc[i][k] += colsum[k];
      }
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
      sum += colsum[k];
      colsum[k] = 0.f;
    }
    y = yend;
  }
#pragma unroll
  for (int i = 0; i < kPatchPool; ++i)
#pragma unroll
    for (int j = 0; j < kPatchPool; ++j)
#pragma unroll
      for (int k = 0; k < KMAX; ++k) acc[i * kPatchPool + j] += ((colmask[k] >> j) & 1u) ? rowacc[i][k] : 0.f;
}

// Vector path (rows contiguous and 16 B aligned, W % 4 == 0, W <= 4*LPR): LPR lanes cover one row with a float4 each, so one
// load instruction fetches 32/LPR rows; U of them are in flight per lane before the first add.
template <int LPR, int U>
__device__ __forceinline__ void pool_plane_vec4(const float* __restrict__ plane, int H, int W, long long s_y,
                                                const int* ys, const int* ye, const int* xs, const int* xe,
                                                float* acc, float& sum, float& sq) {
  constexpr int RPI = 32 / LPR;                       // rows per load instruction
  const int lane = threadIdx.x & 31;
  const int cg = (lane % LPR) * 4, rsub = lane / LPR;
  const bool colvalid = cg < W;
  unsigned colmask[4];
  float colsum[4] = {0.f, 0.f, 0.f, 0.f};
  float rowacc[kPatchPool][4];
#pragma unroll
  for (int i = 0; i < kPatchPool; ++i)
#pragma unroll
    for (int e = 0; e < 4; ++e) rowacc[i][e] = 0.f;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int x = cg + e;
    unsigned m = 0;
#pragma unroll
    for (int j = 0; j < kPatchPool; ++j) m |= (x >= xs[j] && x < xe[j] && x < W) ? (1u << j) : 0u;
    colmask[e] = m;
  }
  int y = 0;
  while (y < H) {
    unsigned rm = 0;
#pragma unroll
    for (int i = 0; i < kPatchPool; ++i) rm |= (y >= ys[i] && y < ye[i]) ? (1u << i) : 0u;
    int yend = H;
#pragma unroll
    for (int i = 0; i < kPatchPool; ++i) {
      if (ys[i] > y && ys[i] < yend) yend = ys[i];
      if (ye[i] > y && ye[i] < yend) yend = ye[i];
    }
    for (int yy = y; yy < yend; yy += U * RPI) {
      float4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int row = yy + u * RPI + rsub;
        v[u] = (row < yend && colvalid) ? __ldg(reinterpret_cast<const float4*>(plane + (long long)row * s_y + cg))
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        colsum[0] += v[u].x; colsum[1] += v[u].y; colsum[2] += v[u].z; colsum[3] += v[u].w;
        sq = fmaf(v[u].x, v[u].x, sq); sq = fmaf(v[u].y, v[u].y, sq);
        sq = fmaf(v[u].z, v[u].z, sq); sq = fmaf(v[u].w, v[u].w, sq);
      }
    }
#pragma unroll
    for (int i = 0; i < kPatchPool; ++i)
      if ((rm >> i) & 1u) {                            // warp-uniform
#pragma unroll
        for (int e = 0; e < 4; ++e) rowacc[i][e] += colsum[e];
      }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      sum += colsum[e];
      colsum[e] = 0.f;
    }
    y = yend;
  }
  // once per plane: this lane's four columns into the column bins they belong to
#pragma unroll
  for (int i = 0; i < kPatchPool; ++i)
#pragma unroll
    for (int j = 0; j < kPatchPool; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[i * kPatchPool + j] += ((colmask[e] >> j) & 1u) ? rowacc[i][e] : 0.f;
}

// Small planes (H*W <= kPatchSmallPlane): the walk above costs ~1000 instructions per plane whatever its size. Here
// the warp copies its plane into shared memory (accumulating sum and sum of squares on the way), then lane i < 16 adds
// up the (at most (H/4+1) x (W/4+1)) elements of bin i: ~10x fewer instructions for the 14x14 .. 28x28 maps.
constexpr int kPatchSmallPlane = 1024;

__device__ __forceinline__ float pool_plane_small(const float* __restrict__ plane, int H, int W, long long s_y,
                                                  long long s_x, float* buf, float& sum, float& sq) {
  const int lane = threadIdx.x & 31;
  const int n = H * W;
  if (s_x == 1 && s_y == W) {
    for (int i = lane; i < n; i += 32) {
      const float v = __ldg(plane + i);
      buf[i] = v;
      sum += v;
      sq = fmaf(v, v, sq);
    }
  } else {
    for (int i = lane; i < n; i += 32) {
      const int y = i / W, x = i - y * W;
      const float v = __ldg(plane + (long long)y * s_y + (long long)x * s_x);
      buf[i] = v;
      sum += v;
      sq = fmaf(v, v, sq);
    }
  }
  __syncwarp();
  float mean = 0.f;
  if (lane < kPatchBins) {
    const int by = lane / kPatchPool, bx = lane % kPatchPool;
    const int y0 = (by * H) / kPatchPool, y1 = ((by + 1) * H + kPatchPool - 1) / kPatchPool;
    const int x0 = (bx * W) / kPatchPool, x1 = ((bx + 1) * W + kPatchPool - 1) / kPatchPool;
    float s = 0.f;
    for (int y = y0; y < y1; ++y)
      for (int x = x0; x < x1; ++x) s += buf[y * W + x];
    mean = s / (float)((y1 - y0) * (x1 - x0));
  }
  __syncwarp();
  return mean;
}

// Any strides / any width: lanes along x, every element tested against the four column bins.
__device__ __forceinline__ void pool_plane_generic(const float* __restrict__ plane, int H, int W, long long s_y,
                                                   long long s_x, const int* ys, const int* ye, const int* xs,
                                                   const int* xe, float* acc, float& sum, float& sq) {
  const int lane = threadIdx.x & 31;
  for (int y = 0; y < H; ++y) {
    const float* row = plane + (long long)y * s_y;
    float col[kPatchPool] = {0.f, 0.f, 0.f, 0.f};
    for (int x = lane; x < W; x += 32) {
      const float v = __ldg(row + (long long)x * s_x);
      sum += v;
      sq = fmaf(v, v, sq);
#pragma unroll
      for (int j = 0; j < kPatchPool; ++j) col[j] += (x >= xs[j] && x < xe[j]) ? v : 0.f;
    }
#pragma unroll
    for (int i = 0; i < kPatchPool; ++i)
      if (y >= ys[i] && y < ye[i]) {                 // warp-uniform
#pragma unroll
        for (int j = 0; j < kPatchPool; ++j) acc[i * kPatchPool + j] += col[j];
      }
  }
}

// grid (B * ceil(D / 8), L), 8 warps: warp w of CTA (b, chunk) owns channel chunk*8 + w of image b in layer blockIdx.y.
// pooled: (L, B, D, 16) bin means; stats: (L, B, D, 2) per-channel sum and sum of squares (doubles).
__global__ void __launch_bounds__(kPatchThreads, 3) patch_pool_kernel(const PatchGramParams p, float* __restrict__ pooled,
                                                                   double* __restrict__ stats) {
  const int l = blockIdx.y;
  const PatchLayer ly = p.layer[l];
  const int H = ly.H, W = ly.W, D = p.D;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int chunks = (D + 7) / 8;
  const int b = blockIdx.x / chunks, c = (blockIdx.x % chunks) * 8 + warp;
  if (c >= D) return;
  int ys[kPatchPool], ye[kPatchPool], xs[kPatchPool], xe[kPatchPool];
#pragma unroll
  for (int i = 0; i < kPatchPool; ++i) {            // ATen adaptive bins: floor(i*n/4) .. ceil((i+1)*n/4)
    ys[i] = (i * H) / kPatchPool;  ye[i] = ((i + 1) * H + kPatchPool - 1) / kPatchPool;
    xs[i] = (i * W) / kPatchPool;  xe[i] = ((i + 1) * W + kPatchPool - 1) / kPatchPool;
  }
  const float* plane = ly.x + (long long)b * ly.s_img + (long long)c * ly.s_c;
  const long long plane_id = ((long long)l * p.B + b) * D + c;
  if (H * W <= kPatchSmallPlane) {                    // uniform over the CTA (one layer per blockIdx.y)
    extern __shared__ float small_planes[];
    float sum = 0.f, sq = 0.f;
    const float mean = pool_plane_small(plane, H, W, ly.s_y, ly.s_x, small_planes + warp * kPatchSmallPlane, sum, sq);
    if (lane < kPatchBins) pooled[plane_id * kPatchBins + lane] = mean;
    const float fsum = warp_sum(sum), fsq = warp_sum(sq);
    if (lane == 0) {
      stats[plane_id * 2] = (double)fsum;
      stats[plane_id * 2 + 1] = (double)fsq;
    }
    return;
  }
  float acc[kPatchBins];
#pragma unroll
  for (int i = 0; i < kPatchBins; ++i) acc[i] = 0.f;
  float sum = 0.f, sq = 0.f;
  const bool vec = ly.s_x == 1 && (W & 3) == 0 && (ly.s_y & 3) == 0 && (ly.s_c & 3) == 0 && (ly.s_img & 3) == 0 &&
                   (reinterpret_cast<uintptr_t>(ly.x) & 15) == 0;
  if (vec && W <= 32) pool_plane_vec4<8, 4>(plane, H, W, ly.s_y, ys, ye, xs, xe, acc, sum, sq);
  else if (vec && W <= 64) pool_plane_vec4<16, 7>(plane, H, W, ly.s_y, ys, ye, xs, xe, acc, sum, sq);
  else if (vec && W <= 128) pool_plane_vec4<32, 7>(plane, H, W, ly.s_y, ys, ye, xs, xe, acc, sum, sq);
  else if (ly.s_x == 1 && W <= 32) pool_plane_rows<1>(plane, H, W, ly.s_y, ys, ye, xs, xe, acc, sum, sq);
  else if (ly.s_x == 1 && W <= 64) pool_plane_rows<2>(plane, H, W, ly.s_y, ys, ye, xs, xe, acc, sum, sq);
  else if (ly.s_x == 1 && W <= 128) pool_plane_rows<4>(plane, H, W, ly.s_y, ys, ye, xs, xe, acc, sum, sq);
  else if (ly.s_x == 1 && W <= 256) pool_plane_rows<8>(plane, H, W, ly.s_y, ys, ye, xs, xe, acc, sum, sq);
  else pool_plane_generic(plane, H, W, ly.s_y, ly.s_x, ys, ye, xs, xe, acc, sum, sq);

  // halving butterfly: 16 values per lane -> lane (i << 1) holds bin i summed over the warp (16 shuffles instead of 80)
#pragma unroll
  for (int half = 8, o = 16; half >= 1; half >>= 1, o >>= 1) {
    const bool up = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float send = up ? acc[i] : acc[i + half];
      const float keep = up ? acc[i + half] : acc[i];
      acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
  const float total = acc[0] + __shfl_xor_sync(0xffffffffu, acc[0], 1);
  const int bin = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
  if ((lane & 1) == 0) {
    const int by = bin / kPatchPool, bx = bin % kPatchPool;   // arithmetic, not ys[by]: keeps the bin tables in registers
    const int cnt = (((by + 1) * H + kPatchPool - 1) / kPatchPool - (by * H) / kPatchPool) *
                    (((bx + 1) * W + kPatchPool - 1) / kPatchPool - (bx * W) / kPatchPool);
    pooled[plane_id * kPatchBins + bin] = total / (float)cnt;
  }
  const float fsum = warp_sum(sum), fsq = warp_sum(sq);
  if (lane == 0) {
    stats[plane_id * 2] = (double)fsum;
    stats[plane_id * 2 + 1] = (double)fsq;
  }
}

// The two layer norms of image b, layer l, from the pooling pass's bin means and channel sums: Z[D][16] (shared memory)
// receives LN_(D,4,4)(pool(LN_map(x))) (:198, :210, :213). Shared by the forward and the backward so that the backward
// differentiates the very values the forward produced. fm / fr: mean and rstd of the whole map (0 / 1 without
// ln_input); mean2 / rstd2: those of the pooled map. Ends with the CTA synchronised.
struct PatchBinNorm {
  float fm, fr, mean2, rstd2;
};

__device__ __forceinline__ PatchBinNorm patch_normalise_bins(const PatchGramParams& p, const float* __restrict__ pooled,
                                                             const double* __restrict__ stats, float* Z, double* red,
                                                             int b, int l) {
  const int H = p.layer[l].H, W = p.layer[l].W, D = p.D;
  const int n = D * kPatchBins;
  const long long base = ((long long)l * p.B + b) * D;
  PatchBinNorm r{0.f, 1.f, 0.f, 1.f};
  for (int i = threadIdx.x; i < n; i += blockDim.x) Z[i] = pooled[base * kPatchBins + i];
  if (p.ln_input) {                                  // pool(LN(x)) = (pool(x) - mean) * rstd: pooling is linear
    double tsum = 0.0, tsq = 0.0;
    for (int c = threadIdx.x; c < D; c += blockDim.x) {
      tsum += stats[(base + c) * 2];
      tsq += stats[(base + c) * 2 + 1];
    }
    const double cnt = (double)D * H * W;
    const double s1 = block_sum(tsum, red);
    const double s2 = block_sum(tsq, red);
    const double mean = s1 / cnt;
    double var = s2 / cnt - mean * mean;
    var = var > 0.0 ? var : 0.0;
    const float fm = (float)mean, fr = (float)(1.0 / sqrt(var + 1e-5));
    for (int i = threadIdx.x; i < n; i += blockDim.x) Z[i] = (Z[i] - fm) * fr;   // each thread rewrites what it loaded
    r.fm = fm;
    r.fr = fr;
  }
  __syncthreads();

  // ---- layer norm over the (D, 4, 4) pooled map (:213) ----
  double ps = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) ps += (double)Z[i];
  const float mean2 = (float)(block_sum(ps, red) / n);
  double pv = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) { const float d = Z[i] - mean2; pv += (double)(d * d); }
  const float rstd2 = (float)(1.0 / sqrt(block_sum(pv, red) / n + 1e-5));
  for (int i = threadIdx.x; i < n; i += blockDim.x) Z[i] = (Z[i] - mean2) * rstd2;
  __syncthreads();
  r.mean2 = mean2;
  r.rstd2 = rstd2;
  return r;
}

// grid (B, L): whole-map layer norm folded in (:198), layer norm over (D, 4, 4) (:213), Gram (:217-220), norm (:223).
__global__ void __launch_bounds__(kPatchThreads) patch_gram_kernel(const PatchGramParams p, const float* __restrict__ pooled,
                                                                   const double* __restrict__ stats) {
  extern __shared__ float smem[];
  float* Z = smem;                                   // [D][16] pooled (then normalised) map
  double* red = reinterpret_cast<double*>(Z + p.D * kPatchBins);   // 32 doubles
  const int b = blockIdx.x, l = blockIdx.y;
  const int D = p.D;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  patch_normalise_bins(p, pooled, stats, Z, red, b, l);

  // ---- Gram over the 16 positions (:217-220) and its Frobenius norm (:223) ----
  const float inv = (float)(1.0 / ((double)kPatchBins + 1e-6));
  float* out = p.gram + ((long long)l * p.B + b) * D * D;
  double fro = 0.0;
  for (int d0 = 0; d0 < D; d0 += 32) {               // lane <-> column d (coalesced stores), warp <-> rows c
    const int d = d0 + lane;
    float zd[kPatchBins];
#pragma unroll
    for (int k = 0; k < kPatchBins; ++k) zd[k] = (d < D) ? Z[d * kPatchBins + k] : 0.f;
    for (int c = warp; c < D; c += nwarps) {
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < kPatchBins; k += 4) {
        const float4 t = *reinterpret_cast<const float4*>(&Z[c * kPatchBins + k]);   // broadcast
        s = fmaf(zd[k], t.x, s); s = fmaf(zd[k + 1], t.y, s); s = fmaf(zd[k + 2], t.z, s); s = fmaf(zd[k + 3], t.w, s);
      }
      s *= inv;
      if (d < D) {
        out[c * D + d] = s;
        fro += (double)(s * s);
      }
    }
  }
  const double f2 = block_sum(fro, red);
  if (threadIdx.x == 0) p.gram_norm[(long long)l * p.B + b] = (float)sqrt(f2);
}

// ----------------------------------------------------------------------------------------------------------------------
struct PatchAttnParams {
  const float* feat;                       // (L, B, E) projected Gram features
  const float* w_in[2];  const float* b_in[2];     // (3E, E), (3E)   attention_per_layer, attention_per_patch
  const float* w_out[2]; const float* b_out[2];    // (E, E), (E)
  const float* w_c;      const float* b_c;         // (nc, E), (nc)
  int L, B, E, heads, nc;
  float* emb;                              // (B, E)
  float* logits;                           // (B, nc)
};

// Y[l][j] = bias[j] + sum_k X[l][k] * Wt[j][k]   for l < L, j < N;  X, Y in shared memory (row pitch ldx / ldy), W global.
template <int MAXL>
__device__ __forceinline__ void rows_linear(const float* X, int ldx, const float* __restrict__ Wt, const float* __restrict__ bias,
                                            float* Y, int ldy, int L, int N, int K, float scale_first, int n_scaled) {
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    float acc[MAXL];
#pragma unroll
    for (int l = 0; l < MAXL; ++l) acc[l] = 0.f;
    const float4* w4 = reinterpret_cast<const float4*>(Wt + (long long)j * K);
    for (int k4 = 0; k4 < K / 4; ++k4) {
      const float4 w = __ldg(w4 + k4);
#pragma unroll
      for (int l = 0; l < MAXL; ++l)
        if (l < L) {
          const float4 x = *reinterpret_cast<const float4*>(X + l * ldx + k4 * 4);   // broadcast across the warp
          acc[l] = fmaf(x.x, w.x, acc[l]); acc[l] = fmaf(x.y, w.y, acc[l]);
          acc[l] = fmaf(x.z, w.z, acc[l]); acc[l] = fmaf(x.w, w.w, acc[l]);
        }
    }
    const float bj = bias ? __ldg(bias + j) : 0.f;
    const float sc = (j < n_scaled) ? scale_first : 1.f;
#pragma unroll
    for (int l = 0; l < MAXL; ++l)
      if (l < L) Y[l * ldy + j] = (acc[l] + bj) * sc;
  }
}

// One attention of one image up to the out_proj input: QKV = X W_in^T + b_in (q scaled by sqrt(1/hd)), P = softmax of the
// scores per head, O = P V (all [L][.] rows in shared memory). Shared by the forward and the backward's recomputation.
// Ends with the CTA synchronised.
__device__ __forceinline__ void patch_attention_core(const float* X, float* QKV, float* P, float* O,
                                                     const float* __restrict__ w_in, const float* __restrict__ b_in,
                                                     int L, int E, int H, int hd, float qscale) {
  rows_linear<kPatchMaxLayers>(X, E, w_in, b_in, QKV, 3 * E, L, 3 * E, E, qscale, E);
  __syncthreads();
  for (int i = threadIdx.x; i < H * L * L; i += blockDim.x) {         // scores
    const int h = i / (L * L), r = i - h * L * L, l = r / L, m = r - l * L;
    const float* q = QKV + l * 3 * E + h * hd;
    const float* k = QKV + m * 3 * E + E + h * hd;
    float s = 0.f;
    for (int d = 0; d < hd; ++d) s = fmaf(q[d], k[d], s);
    P[i] = s;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < H * L; i += blockDim.x) {             // softmax over keys
    float* row = P + i * L;
    float mx = row[0];
    for (int m = 1; m < L; ++m) mx = fmaxf(mx, row[m]);
    float sum = 0.f;
    for (int m = 0; m < L; ++m) { const float e = expf(row[m] - mx); row[m] = e; sum += e; }
    const float r = 1.f / sum;
    for (int m = 0; m < L; ++m) row[m] *= r;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < L * E; i += blockDim.x) {             // attention-weighted values
    const int l = i / E, e = i - l * E, h = e / hd;
    const float* pr = P + (h * L + l) * L;
    float s = 0.f;
    for (int m = 0; m < L; ++m) s = fmaf(pr[m], QKV[m * 3 * E + 2 * E + e], s);
    O[i] = s;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kPatchThreads) patch_attention_kernel(const PatchAttnParams p) {
  extern __shared__ float smem[];
  const int L = p.L, E = p.E, H = p.heads, hd = E / H;
  float* X = smem;                       // [L][E]   tokens in / attention output / next tokens
  float* QKV = X + L * E;                // [L][3E]
  float* P = QKV + L * 3 * E;            // [H][L][L]
  float* O = P + H * L * L;              // [L][E]
  const float qscale = sqrtf(1.0f / (float)hd);      // torch: q * math.sqrt(1.0 / head_dim)

  for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
    __syncthreads();
    for (int i = threadIdx.x; i < L * E; i += blockDim.x) {
      const int l = i / E, e = i - l * E;
      X[i] = p.feat[((long long)l * p.B + b) * E + e];
    }
    __syncthreads();
    for (int a = 0; a < 2; ++a) {
      patch_attention_core(X, QKV, P, O, p.w_in[a], p.b_in[a], L, E, H, hd, qscale);
      rows_linear<kPatchMaxLayers>(O, E, p.w_out[a], p.b_out[a], X, E, L, E, E, 1.f, 0);
      __syncthreads();
    }
    for (int e = threadIdx.x; e < E; e += blockDim.x) {                 // mean over the layer tokens (:247)
      float s = 0.f;
      for (int l = 0; l < L; ++l) s += X[l * E + e];
      s /= (float)L;
      O[e] = s;
      p.emb[(long long)b * E + e] = s;
    }
    __syncthreads();
    for (int j = threadIdx.x >> 5; j < p.nc; j += blockDim.x >> 5) {    // classifier (:256): one warp per class
      const float* w = p.w_c + (long long)j * E;
      float s = 0.f;
      for (int e = threadIdx.x & 31; e < E; e += 32) s = fmaf(O[e], __ldg(w + e), s);
      s = warp_sum(s);
      if ((threadIdx.x & 31) == 0) p.logits[(long long)b * p.nc + j] = s + __ldg(p.b_c + j);
    }
  }
}

// ======================================================================================================================
// Backward. Per image and layer, with P the (normalised) pooled map, Z = LN(P), G = Z Z^T / (16 + 1e-6), n = |G|_F:
//   dG <- dG + dn G / n (0 where n == 0);  dZ = (dG + dG^T) Z / (16 + 1e-6);  dP = r2 (dZ - mean dZ - Z mean(dZ Z))
//   dx^(y, x) = sum over the bins i holding (y, x) of dP[i] / |bin i|   (ATen's bins overlap when H % 4 != 0)
//   dX = r (dx^ - sum(dP) / N - x^ sum(dP P) / N)   (ln_input; both whole-map sums come out of the 16 D bin values)
// patch_gram_bwd_kernel reduces that to a per-plane table coef[d][i] = r dP[d][i] / |bin i| and three scalars, so that
//   dX(d, y, x) = sum_{i holding (y, x)} coef[d][i] + a + c (X(d, y, x) - mu)
// and patch_pool_bwd_kernel writes every map's gradient in one pass (X read only with ln_input).
constexpr int kPatchBwdScalars = 4;      // a, c, mu, (pad) per (layer, image)

// grid (B, L). Shared memory: Z [D][16], S = dG + dG^T [D][D+1], M = Z^T Z [16][16], 32 doubles.
__global__ void __launch_bounds__(kPatchThreads) patch_gram_bwd_kernel(const PatchGramParams p, const float* __restrict__ pooled,
                                                                       const double* __restrict__ stats,
                                                                       const float* __restrict__ d_gram,
                                                                       const float* __restrict__ d_norm,
                                                                       float* __restrict__ coef, float* __restrict__ scal) {
  extern __shared__ float smem[];
  const int D = p.D, n = D * kPatchBins, ld = D + 1;
  float* Z = smem;
  float* S = Z + n;
  float* M = S + D * ld;
  double* red = reinterpret_cast<double*>(M + kPatchBins * kPatchBins);   // D (D + 1) is even: 8 B aligned
  const int b = blockIdx.x, l = blockIdx.y;
  const int H = p.layer[l].H, W = p.layer[l].W;
  const PatchBinNorm nb = patch_normalise_bins(p, pooled, stats, Z, red, b, l);
  const long long img = (long long)l * p.B + b;

  const float* dg = d_gram + img * D * D;
  for (int i = threadIdx.x; i < D * D; i += blockDim.x) {
    const int c = i / D, d = i - c * D;
    S[c * ld + d] = dg[i];
  }
  for (int i = threadIdx.x; i < kPatchBins * kPatchBins; i += blockDim.x) {
    const int j = i / kPatchBins, k = i % kPatchBins;
    float s = 0.f;
    for (int c = 0; c < D; ++c) s = fmaf(Z[c * kPatchBins + j], Z[c * kPatchBins + k], s);
    M[i] = s;
  }
  __syncthreads();

  // norm term (:223): dn G / n, with G Z = Z (Z^T Z) / (16 + 1e-6); the forward's n, 0 where n == 0 (torch's convention)
  const float inv = (float)(1.0 / ((double)kPatchBins + 1e-6));
  const float nrm = p.gram_norm[img], dn = d_norm[img];
  const float s_n = nrm > 0.f ? 2.f * dn / nrm * inv * inv : 0.f;
  constexpr int kPer = kPatchMaxD * kPatchBins / kPatchThreads;      // 8 (launched with kPatchThreads threads)
  float dz[kPer];
  double t1 = 0.0, t2 = 0.0;
#pragma unroll
  for (int t = 0; t < kPer; ++t) {
    const int i = threadIdx.x + t * kPatchThreads;
    dz[t] = 0.f;
    if (i < n) {
      const int c = i / kPatchBins, k = i % kPatchBins;
      float acc = 0.f;
      for (int d = 0; d < D; ++d) acc = fmaf(S[c * ld + d] + S[d * ld + c], Z[d * kPatchBins + k], acc);
      float gz = 0.f;
#pragma unroll
      for (int j = 0; j < kPatchBins; ++j) gz = fmaf(Z[c * kPatchBins + j], M[j * kPatchBins + k], gz);
      dz[t] = fmaf(s_n, gz, inv * acc);
      t1 += (double)dz[t];
      t2 += (double)dz[t] * (double)Z[i];
    }
  }
  // layer norm over (D, 4, 4) (:213)
  const double m1 = block_sum(t1, red) / n;
  const double m2 = block_sum(t2, red) / n;
  const float fm1 = (float)m1, fm2 = (float)m2;
  float* cf = coef + img * n;
  double u1 = 0.0, u2 = 0.0;
#pragma unroll
  for (int t = 0; t < kPer; ++t) {
    const int i = threadIdx.x + t * kPatchThreads;
    if (i < n) {
      const float dp = nb.rstd2 * (dz[t] - fm1 - Z[i] * fm2);
      const int k = i % kPatchBins, by = k / kPatchPool, bx = k % kPatchPool;
      const int cnt = (((by + 1) * H + kPatchPool - 1) / kPatchPool - (by * H) / kPatchPool) *
                      (((bx + 1) * W + kPatchPool - 1) / kPatchPool - (bx * W) / kPatchPool);
      cf[i] = nb.fr * dp / (float)cnt;
      if (p.ln_input) {
        const float pv = (pooled[img * n + i] - nb.fm) * nb.fr;     // the forward's pooled value P
        u1 += (double)dp;
        u2 += (double)dp * (double)pv;
      }
    }
  }
  if (p.ln_input) {                                  // whole-map layer norm (:198), folded like the forward folds it
    const double s1 = block_sum(u1, red), s2 = block_sum(u2, red);
    if (threadIdx.x == 0) {
      const double N = (double)D * H * W, r = (double)nb.fr;
      scal[img * kPatchBwdScalars + 0] = (float)(-r * s1 / N);
      scal[img * kPatchBwdScalars + 1] = (float)(-r * r * s2 / N);
      scal[img * kPatchBwdScalars + 2] = nb.fm;
      scal[img * kPatchBwdScalars + 3] = 0.f;
    }
  } else if (threadIdx.x < kPatchBwdScalars) {
    scal[img * kPatchBwdScalars + threadIdx.x] = 0.f;
  }
}

struct PatchGradLayer {
  float* dx;
  long long s_img, s_c, s_y, s_x;   // element strides of the gradient (the layout of the map the forward read)
};

struct PatchPoolBwdParams {
  PatchLayer layer[kPatchMaxLayers];      // x: read only with ln_input
  PatchGradLayer grad[kPatchMaxLayers];
  int L, B, D, ln_input;
  const float* coef;                      // (L, B, D, 16)
  const float* scal;                      // (L, B, 4)
};

// sum of the plane's coefficients over the row bins in rm and the column bins in cm
__device__ __forceinline__ float patch_bin_sum(const float* cf, unsigned rm, unsigned cm) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < kPatchPool; ++i)
#pragma unroll
    for (int j = 0; j < kPatchPool; ++j) s += (((rm >> i) & (cm >> j)) & 1u) ? cf[i * kPatchPool + j] : 0.f;
  return s;
}

__device__ __forceinline__ unsigned patch_bin_mask(int v, const int* s, const int* e) {
  unsigned m = 0;
#pragma unroll
  for (int i = 0; i < kPatchPool; ++i) m |= (v >= s[i] && v < e[i]) ? (1u << i) : 0u;
  return m;
}

// Vector path (x and dX rows contiguous and 16 B aligned, W % 4 == 0, W <= 4*LPR): LPR lanes cover a row with a float4
// each. Rows are walked in segments of constant row-bin membership; inside one, a lane's four values are constant
// (a + bin sums) and each element costs one fma on the loaded x (ln_input) or nothing (a plain store).
template <int LPR, int U, bool LN>
__device__ __forceinline__ void pool_bwd_plane_vec4(const float* __restrict__ plane, float* __restrict__ out, int H, int W,
                                                    long long s_y, long long d_y, const int* ys, const int* ye,
                                                    const int* xs, const int* xe, const float* cf, float a, float c,
                                                    float mu) {
  constexpr int RPI = 32 / LPR;
  const int lane = threadIdx.x & 31;
  const int cg = (lane % LPR) * 4, rsub = lane / LPR;
  const bool colvalid = cg < W;
  unsigned cm[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) cm[e] = patch_bin_mask(cg + e, xs, xe);
  int y = 0;
  while (y < H) {
    const unsigned rm = patch_bin_mask(y, ys, ye);
    int yend = H;
#pragma unroll
    for (int i = 0; i < kPatchPool; ++i) {
      if (ys[i] > y && ys[i] < yend) yend = ys[i];
      if (ye[i] > y && ye[i] < yend) yend = ye[i];
    }
    float base[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) base[e] = a + patch_bin_sum(cf, rm, cm[e]);
    for (int yy = y; yy < yend; yy += U * RPI) {
      float4 v[U];
      if (LN) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int row = yy + u * RPI + rsub;
          v[u] = (row < yend && colvalid) ? __ldg(reinterpret_cast<const float4*>(plane + (long long)row * s_y + cg))
                                          : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int row = yy + u * RPI + rsub;
        if (row < yend && colvalid) {
          float4 o;
          if (LN) {
            o.x = fmaf(c, v[u].x - mu, base[0]); o.y = fmaf(c, v[u].y - mu, base[1]);
            o.z = fmaf(c, v[u].z - mu, base[2]); o.w = fmaf(c, v[u].w - mu, base[3]);
          } else {
            o = make_float4(base[0], base[1], base[2], base[3]);
          }
          __stcs(reinterpret_cast<float4*>(out + (long long)row * d_y + cg), o);
        }
      }
    }
    y = yend;
  }
}

// Any strides / widths: lanes along x, rows in segments of constant row-bin membership.
__device__ __forceinline__ void pool_bwd_plane_generic(const float* __restrict__ plane, float* __restrict__ out, int H,
                                                       int W, long long s_y, long long s_x, long long d_y, long long d_x,
                                                       bool ln, const int* ys, const int* ye, const int* xs,
                                                       const int* xe, const float* cf, float a, float c, float mu) {
  const int lane = threadIdx.x & 31;
  int y = 0;
  while (y < H) {
    const unsigned rm = patch_bin_mask(y, ys, ye);
    int yend = H;
#pragma unroll
    for (int i = 0; i < kPatchPool; ++i) {
      if (ys[i] > y && ys[i] < yend) yend = ys[i];
      if (ye[i] > y && ye[i] < yend) yend = ye[i];
    }
    for (int x = lane; x < W; x += 32) {
      const float base = a + patch_bin_sum(cf, rm, patch_bin_mask(x, xs, xe));
      for (int yy = y; yy < yend; ++yy) {
        float o = base;
        if (ln) o = fmaf(c, __ldg(plane + (long long)yy * s_y + (long long)x * s_x) - mu, base);
        __stcs(out + (long long)yy * d_y + (long long)x * d_x, o);
      }
    }
    y = yend;
  }
}

// Small planes (H*W <= kPatchSmallPlane): lanes over the flattened plane, so that a 14x14 map keeps all 32 lanes busy.
__device__ __forceinline__ void pool_bwd_plane_small(const float* __restrict__ plane, float* __restrict__ out, int H, int W,
                                                     long long s_y, long long s_x, long long d_y, long long d_x, bool ln,
                                                     const int* ys, const int* ye, const int* xs, const int* xe,
                                                     const float* cf, float a, float c, float mu) {
  const int lane = threadIdx.x & 31;
  const int n = H * W;
  for (int i = lane; i < n; i += 32) {
    const int y = i / W, x = i - y * W;
    float o = a + patch_bin_sum(cf, patch_bin_mask(y, ys, ye), patch_bin_mask(x, xs, xe));
    if (ln) o = fmaf(c, __ldg(plane + (long long)y * s_y + (long long)x * s_x) - mu, o);
    __stcs(out + (long long)y * d_y + (long long)x * d_x, o);
  }
}

// grid (B * ceil(D / 8), L), 8 warps: warp w of CTA (b, chunk) writes the gradient of channel chunk*8 + w of image b in
// layer blockIdx.y (the forward's layout of work).
__global__ void __launch_bounds__(kPatchThreads) patch_pool_bwd_kernel(const PatchPoolBwdParams p) {
  const int l = blockIdx.y;
  const PatchLayer ly = p.layer[l];
  const PatchGradLayer gl = p.grad[l];
  const int H = ly.H, W = ly.W, D = p.D;
  const int warp = threadIdx.x >> 5;
  const int chunks = (D + 7) / 8;
  const int b = blockIdx.x / chunks, ch = (blockIdx.x % chunks) * 8 + warp;
  if (ch >= D) return;
  int ys[kPatchPool], ye[kPatchPool], xs[kPatchPool], xe[kPatchPool];
#pragma unroll
  for (int i = 0; i < kPatchPool; ++i) {            // ATen adaptive bins: floor(i*n/4) .. ceil((i+1)*n/4)
    ys[i] = (i * H) / kPatchPool;  ye[i] = ((i + 1) * H + kPatchPool - 1) / kPatchPool;
    xs[i] = (i * W) / kPatchPool;  xe[i] = ((i + 1) * W + kPatchPool - 1) / kPatchPool;
  }
  const long long img = (long long)l * p.B + b;
  float cf[kPatchBins];
  const float4* c4 = reinterpret_cast<const float4*>(p.coef + (img * D + ch) * kPatchBins);
#pragma unroll
  for (int q = 0; q < kPatchBins / 4; ++q) {
    const float4 t = __ldg(c4 + q);
    cf[4 * q] = t.x; cf[4 * q + 1] = t.y; cf[4 * q + 2] = t.z; cf[4 * q + 3] = t.w;
  }
  const float4 sc = __ldg(reinterpret_cast<const float4*>(p.scal) + img);
  const float a = sc.x, c = sc.y, mu = sc.z;
  const bool ln = p.ln_input != 0;
  const float* plane = ln ? ly.x + (long long)b * ly.s_img + (long long)ch * ly.s_c : nullptr;
  float* out = gl.dx + (long long)b * gl.s_img + (long long)ch * gl.s_c;
  if (H * W <= kPatchSmallPlane) {
    pool_bwd_plane_small(plane, out, H, W, ly.s_y, ly.s_x, gl.s_y, gl.s_x, ln, ys, ye, xs, xe, cf, a, c, mu);
    return;
  }
  const bool vec = gl.s_x == 1 && (W & 3) == 0 && (gl.s_y & 3) == 0 && (gl.s_c & 3) == 0 && (gl.s_img & 3) == 0 &&
                   (reinterpret_cast<uintptr_t>(gl.dx) & 15) == 0 &&
                   (!ln || (ly.s_x == 1 && (ly.s_y & 3) == 0 && (ly.s_c & 3) == 0 && (ly.s_img & 3) == 0 &&
                            (reinterpret_cast<uintptr_t>(ly.x) & 15) == 0));
  if (vec && W <= 32) {
    if (ln) pool_bwd_plane_vec4<8, 4, true>(plane, out, H, W, ly.s_y, gl.s_y, ys, ye, xs, xe, cf, a, c, mu);
    else pool_bwd_plane_vec4<8, 4, false>(plane, out, H, W, ly.s_y, gl.s_y, ys, ye, xs, xe, cf, a, c, mu);
  } else if (vec && W <= 64) {
    if (ln) pool_bwd_plane_vec4<16, 4, true>(plane, out, H, W, ly.s_y, gl.s_y, ys, ye, xs, xe, cf, a, c, mu);
    else pool_bwd_plane_vec4<16, 4, false>(plane, out, H, W, ly.s_y, gl.s_y, ys, ye, xs, xe, cf, a, c, mu);
  } else if (vec && W <= 128) {
    if (ln) pool_bwd_plane_vec4<32, 4, true>(plane, out, H, W, ly.s_y, gl.s_y, ys, ye, xs, xe, cf, a, c, mu);
    else pool_bwd_plane_vec4<32, 4, false>(plane, out, H, W, ly.s_y, gl.s_y, ys, ye, xs, xe, cf, a, c, mu);
  } else {
    pool_bwd_plane_generic(plane, out, H, W, ly.s_y, ly.s_x, gl.s_y, gl.s_x, ln, ys, ye, xs, xe, cf, a, c, mu);
  }
}

// ---- attentions, mean over layers and classifier, backward ----------------------------------------------------------
struct PatchAttnBwdParams {
  PatchAttnParams f;                       // the forward's inputs and weights (emb / logits unused)
  const float* d_emb;                      // (B, E)
  const float* d_logits;                   // (B, nc)
  float* d_feat;                           // (L, B, E)
  float* x1;                               // (L, B, E)     input of attention_per_patch
  float* dqkv;                             // (2, L, B, 3E) gradient of each attention's in_proj output
  float* o;                                // (2, L, B, E)  each attention's out_proj input
  float* dy;                               // (2, L, B, E)  gradient of each attention's output
};

// Y[l][k] = sum_{j < N} G[l][j] W[j][k] for l < L, k < K; G, Y in shared memory, W (N, K) row-major in global memory
// (coalesced across k).
template <int MAXL>
__device__ __forceinline__ void rows_linear_t(const float* G, int ldg, const float* __restrict__ Wm, float* Y, int ldy,
                                              int L, int N, int K) {
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    float acc[MAXL];
#pragma unroll
    for (int l = 0; l < MAXL; ++l) acc[l] = 0.f;
    for (int j = 0; j < N; ++j) {
      const float w = __ldg(Wm + (long long)j * K + k);
#pragma unroll
      for (int l = 0; l < MAXL; ++l)
        if (l < L) acc[l] = fmaf(G[l * ldg + j], w, acc[l]);
    }
#pragma unroll
    for (int l = 0; l < MAXL; ++l)
      if (l < L) Y[l * ldy + k] = acc[l];
  }
}

// rows [L][n] of shared memory -> rows l * B + b of a (L, B, n) global tensor
__device__ __forceinline__ void store_rows(const float* src, float* dst, int L, int B, int b, int n) {
  for (int i = threadIdx.x; i < L * n; i += blockDim.x) {
    const int l = i / n, e = i - l * n;
    dst[((long long)l * B + b) * n + e] = src[i];
  }
}

// One CTA per image at a time. The image's forward is recomputed in shared memory (with patch_attention_core, the
// forward's own code), then: classifier, mean, and for attention 2 then 1: out_proj, softmax attention, in_proj.
__global__ void __launch_bounds__(kPatchThreads) patch_attention_bwd_kernel(const PatchAttnBwdParams p) {
  extern __shared__ float smem[];
  const int L = p.f.L, E = p.f.E, H = p.f.heads, hd = E / H, B = p.f.B, nc = p.f.nc;
  const int LE = L * E, HLL = H * L * L;
  // rows read as float4 (X, O) first: every [L][.] buffer starts 16 B aligned (E % 4 == 0), whatever H L L is
  float* X[2] = {smem, smem + LE};                      // inputs of the two attentions [L][E]
  float* QKV[2] = {X[1] + LE, X[1] + LE + 3 * LE};      // [L][3E]
  float* O[2] = {QKV[1] + 3 * LE, QKV[1] + 3 * LE + LE};   // [L][E]
  float* G = O[1] + LE;                                  // [L][E] gradient of the current attention's output
  float* dO = G + LE;                                    // [L][E]
  float* dQKV = dO + LE;                                 // [L][3E]
  float* demb = dQKV + 3 * LE;                           // [E]
  float* P[2] = {demb + E, demb + E + HLL};              // [H][L][L]
  float* dS = P[1] + HLL;                                // [H][L][L]
  const float qscale = sqrtf(1.0f / (float)hd);

  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    __syncthreads();
    for (int i = threadIdx.x; i < LE; i += blockDim.x) {
      const int l = i / E, e = i - l * E;
      X[0][i] = p.f.feat[((long long)l * B + b) * E + e];
    }
    __syncthreads();
    patch_attention_core(X[0], QKV[0], P[0], O[0], p.f.w_in[0], p.f.b_in[0], L, E, H, hd, qscale);
    rows_linear<kPatchMaxLayers>(O[0], E, p.f.w_out[0], p.f.b_out[0], X[1], E, L, E, E, 1.f, 0);
    __syncthreads();
    patch_attention_core(X[1], QKV[1], P[1], O[1], p.f.w_in[1], p.f.b_in[1], L, E, H, hd, qscale);

    // classifier (:256) and mean over the layers (:247)
    for (int e = threadIdx.x; e < E; e += blockDim.x) {
      float s = p.d_emb[(long long)b * E + e];
      for (int j = 0; j < nc; ++j) s = fmaf(p.d_logits[(long long)b * nc + j], __ldg(p.f.w_c + (long long)j * E + e), s);
      demb[e] = s;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < LE; i += blockDim.x) G[i] = demb[i % E] / (float)L;
    store_rows(X[1], p.x1, L, B, b, E);
    __syncthreads();

    for (int a = 1; a >= 0; --a) {
      const float* qkv = QKV[a];
      const float* pr = P[a];
      store_rows(G, p.dy + (long long)a * LE * B, L, B, b, E);
      store_rows(O[a], p.o + (long long)a * LE * B, L, B, b, E);
      rows_linear_t<kPatchMaxLayers>(G, E, p.f.w_out[a], dO, E, L, E, E);          // out_proj
      __syncthreads();
      for (int i = threadIdx.x; i < HLL; i += blockDim.x) {                       // d probabilities
        const int h = i / (L * L), r = i - h * L * L, l = r / L, m = r - l * L;
        const float* go = dO + l * E + h * hd;
        const float* v = qkv + m * 3 * E + 2 * E + h * hd;
        float s = 0.f;
        for (int d = 0; d < hd; ++d) s = fmaf(go[d], v[d], s);
        dS[i] = s;
      }
      __syncthreads();
      for (int i = threadIdx.x; i < H * L; i += blockDim.x) {                     // softmax over keys
        const float* prow = pr + i * L;
        float* drow = dS + i * L;
        float t = 0.f;
        for (int m = 0; m < L; ++m) t = fmaf(prow[m], drow[m], t);
        for (int m = 0; m < L; ++m) drow[m] = prow[m] * (drow[m] - t);
      }
      __syncthreads();
      for (int i = threadIdx.x; i < LE; i += blockDim.x) {                        // scores and values
        const int l = i / E, e = i - l * E, h = e / hd;
        float dq = 0.f, dk = 0.f, dv = 0.f;
        for (int m = 0; m < L; ++m) {
          dq = fmaf(dS[(h * L + l) * L + m], qkv[m * 3 * E + E + e], dq);        // row l of dS times K
          dk = fmaf(dS[(h * L + m) * L + l], qkv[m * 3 * E + e], dk);            // column l of dS times scaled Q
          dv = fmaf(pr[(h * L + m) * L + l], dO[m * E + e], dv);                 // column l of P times dO
        }
        dQKV[l * 3 * E + e] = dq * qscale;
        dQKV[l * 3 * E + E + e] = dk;
        dQKV[l * 3 * E + 2 * E + e] = dv;
      }
      __syncthreads();
      store_rows(dQKV, p.dqkv + (long long)a * 3 * LE * B, L, B, b, 3 * E);
      rows_linear_t<kPatchMaxLayers>(dQKV, 3 * E, p.f.w_in[a], G, E, L, 3 * E, E);   // in_proj
      __syncthreads();
    }
    store_rows(G, p.d_feat, L, B, b, E);
  }
}

}  // namespace gh
