// Camera-mode preprocessing on the GPU: one kernel turns a raw BGR uint8 frame into the normalised fp32 CHW tensor the
// encoder consumes, bit-identically to what the reference does on the host per frame
// (functions/functions_RESNET50_Truncate_Gram_Attention.py:499-501: cv2.cvtColor(BGR2RGB) -> Image.fromarray ->
// transform; test_RESNET50_Truncate_gram_attention.py:61-66: Resize [+ CenterCrop] + ToTensor + Normalize).
//
// torchvision's Resize on a PIL image is Pillow's ImagingResample with the bilinear (triangle) filter: separable,
// support widened by the down-scale factor (antialiasing), 8-bit fixed point -- coefficients with 22 fractional bits,
// a horizontal pass rounded to uint8, then a vertical pass rounded to uint8. The coefficient tables depend only on the
// sizes; the host computes them once (streaming.py) and a CenterCrop is just the sub-range of output coordinates the
// tables are built for. One thread = one output pixel (three channels): for every contributing input row it forms
// the horizontally filtered uint8, then filters those vertically, divides by 255 and normalises in IEEE fp32.
// The frame is read straight from the uploaded uint8 buffer (6 MB at 1080p, L2 resident); nothing else touches HBM.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/gramhead.h"

namespace gh {

constexpr int kPreprocPrecisionBits = 32 - 8 - 2;

struct PreprocParams {
  const uint8_t* frame;     // (H, W, 3) uint8, `pitch` bytes between rows
  long long pitch;
  int H, W;
  int OH, OW;               // output (after crop) extent
  const int* hx_min;        // [OW]   first contributing input column
  const int* hx_size;       // [OW]   number of contributing columns
  const int* hk;            // [OW][hkmax] integer coefficients (sum = 2^22)
  int hkmax;
  const int* vy_min;        // [OH]
  const int* vy_size;       // [OH]
  const int* vk;            // [OH][vkmax]
  int vkmax;
  float* out;               // (3, OH, OW) fp32
  int bgr;                  // 1: the frame is BGR and output channel c reads input channel 2 - c (cv2.cvtColor BGR2RGB)
  float mean[3], std[3];
};

__device__ __forceinline__ int preproc_clip8(int acc) {
  const int v = acc >> kPreprocPrecisionBits;
  return v < 0 ? 0 : (v > 255 ? 255 : v);
}

__global__ void __launch_bounds__(256) preprocess_frame_kernel(const PreprocParams p) {
  const int ox = blockIdx.x * blockDim.x + threadIdx.x;
  const int oy = blockIdx.y;
  if (ox >= p.OW) return;
  const int x0 = p.hx_min[ox], nx = p.hx_size[ox];
  const int y0 = p.vy_min[oy], ny = p.vy_size[oy];
  const int* __restrict__ hk = p.hk + (long long)ox * p.hkmax;
  const int* __restrict__ vk = p.vk + (long long)oy * p.vkmax;
  int acc[3] = {1 << (kPreprocPrecisionBits - 1), 1 << (kPreprocPrecisionBits - 1), 1 << (kPreprocPrecisionBits - 1)};
  for (int j = 0; j < ny; ++j) {
    const uint8_t* __restrict__ row = p.frame + (long long)(y0 + j) * p.pitch + (long long)x0 * 3;
    int h0 = 1 << (kPreprocPrecisionBits - 1), h1 = h0, h2 = h0;
    for (int i = 0; i < nx; ++i) {
      const int k = __ldg(hk + i);
      h0 += (int)__ldg(row + 3 * i) * k;
      h1 += (int)__ldg(row + 3 * i + 1) * k;
      h2 += (int)__ldg(row + 3 * i + 2) * k;
    }
    const int kv = __ldg(vk + j);
    acc[0] += preproc_clip8(h0) * kv;
    acc[1] += preproc_clip8(h1) * kv;
    acc[2] += preproc_clip8(h2) * kv;
  }
  const long long plane = (long long)p.OH * p.OW;
  float* o = p.out + (long long)oy * p.OW + ox;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int src = p.bgr ? 2 - c : c;
    const float v = (float)preproc_clip8(acc[src]) / 255.0f;          // ToTensor
    o[c * plane] = (v - p.mean[c]) / p.std[c];                        // Normalize (IEEE division: no fast-math)
  }
}

// ---- several frames per launch, into one uint8 batch (streaming.FrameBatchPipeline) ------------------------------------
// N frames, each with its own size, pitch, channel order and tables (GhFrameDesc, include/gramhead.h), resampled to one
// common (OH, OW) and written as a dense (N, 3, OH, OW) uint8 batch in RGB order: clip8 of the vertical sum, the byte that
// preprocess_frame_kernel divides by 255 and normalises. The model applies ToTensor + Normalize to it bit for bit as that
// kernel does (to_tensor_normalize), so the batch carries the same information in a quarter of the bytes.
// preprocess_frame_kernel recomputes every horizontal tap sum once per output row that uses its input row (vy_size of
// them: ~6 at 1080p -> 448, ~17 at 2160p -> Resize(256)). Here a CTA owns (band of `band_rows` output rows, frame): it
// filters the band's input rows horizontally once, rounds them to uint8 into shared memory, then filters those vertically.
// Same integer operations in the same order as preprocess_frame_kernel, so the same bytes. A band whose input rows exceed
// the `span_rows` rows of shared memory is done as several runs of consecutive output rows, each of which fits (one
// output row always does: span_rows >= vkmax), so the host's choice of band height is a matter of speed only.
struct FramesParams {
  const GhFrameDesc* frames;    // [N]
  const int* tables;            // the packed tables the descriptors' offsets point into
  uint8_t* out;                 // (N, 3, OH, OW)
  int OH, OW, band_rows, span_rows, hkmax, vkmax;
};

constexpr int kFramesThreads = 256;
constexpr int kFramesMaxSmem = 227 * 1024;

__global__ void __launch_bounds__(kFramesThreads) preprocess_frames_kernel(const FramesParams p) {
  extern __shared__ uint8_t hrows[];     // [span_rows][3][OW]: horizontally filtered input rows, output channel order
  const GhFrameDesc d = p.frames[blockIdx.y];
  const int OW = p.OW;
  const int* __restrict__ hx_min = p.tables + d.hx_min;
  const int* __restrict__ hx_size = p.tables + d.hx_size;
  const int* __restrict__ vy_min = p.tables + d.vy_min;
  const int* __restrict__ vy_size = p.tables + d.vy_size;
  const long long plane = (long long)p.OH * OW;
  uint8_t* __restrict__ out = p.out + (long long)blockIdx.y * 3 * plane;
  const int band_end = min(p.OH, (int)(blockIdx.x + 1) * p.band_rows);
  for (int r = blockIdx.x * p.band_rows; r < band_end;) {
    // output rows [r, re) and the input rows [ylo, yhi) they read: the longest run that fits in shared memory
    int ylo = __ldg(vy_min + r), yhi = ylo + __ldg(vy_size + r), re = r + 1;
    for (; re < band_end; ++re) {
      const int y0 = __ldg(vy_min + re);
      const int lo = min(ylo, y0), hi = max(yhi, y0 + __ldg(vy_size + re));
      if (hi - lo > p.span_rows) break;
      ylo = lo;
      yhi = hi;
    }
    const int items = (yhi - ylo) * OW;
    for (int i = threadIdx.x; i < items; i += kFramesThreads) {
      const int yy = i / OW, ox = i - yy * OW;
      const int x0 = __ldg(hx_min + ox), nx = __ldg(hx_size + ox);
      const int* __restrict__ hk = p.tables + d.hk + (long long)ox * p.hkmax;
      const uint8_t* __restrict__ row = d.frame + (long long)(ylo + yy) * d.pitch + (long long)x0 * 3;
      int h0 = 1 << (kPreprocPrecisionBits - 1), h1 = h0, h2 = h0;
      for (int k = 0; k < nx; ++k) {
        const int c = __ldg(hk + k);
        h0 += (int)__ldg(row + 3 * k) * c;
        h1 += (int)__ldg(row + 3 * k + 1) * c;
        h2 += (int)__ldg(row + 3 * k + 2) * c;
      }
      uint8_t* s = hrows + (long long)yy * 3 * OW + ox;
      s[0] = (uint8_t)preproc_clip8(d.bgr ? h2 : h0);     // output channel c holds input channel bgr ? 2 - c : c
      s[OW] = (uint8_t)preproc_clip8(h1);
      s[2 * OW] = (uint8_t)preproc_clip8(d.bgr ? h0 : h2);
    }
    __syncthreads();
    const int outs = (re - r) * OW;
    for (int i = threadIdx.x; i < outs; i += kFramesThreads) {
      const int dy = i / OW, ox = i - dy * OW, oy = r + dy;
      const int y0 = __ldg(vy_min + oy) - ylo, ny = __ldg(vy_size + oy);
      const int* __restrict__ vk = p.tables + d.vk + (long long)oy * p.vkmax;
      int a0 = 1 << (kPreprocPrecisionBits - 1), a1 = a0, a2 = a0;
      for (int j = 0; j < ny; ++j) {
        const int kv = __ldg(vk + j);
        const uint8_t* s = hrows + (long long)(y0 + j) * 3 * OW + ox;
        a0 += (int)s[0] * kv;
        a1 += (int)s[OW] * kv;
        a2 += (int)s[2 * OW] * kv;
      }
      uint8_t* o = out + (long long)oy * OW + ox;
      o[0] = (uint8_t)preproc_clip8(a0);
      o[plane] = (uint8_t)preproc_clip8(a1);
      o[2 * plane] = (uint8_t)preproc_clip8(a2);
    }
    __syncthreads();
    r = re;
  }
}

// ---- the tables of a loader batch, built on the device (functions.gpu_resize_transform) ---------------------------------
// A loader hands over N decoded images of new sizes in every batch, so the tables preprocess_frames_kernel reads change
// per batch; streaming.resample_tables builds them in Python one output coordinate at a time (over half a second for 256
// mixed images). Here one thread owns one output coordinate of one image -- its column (c < OW) or row (c - OW) -- and
// evaluates Pillow's precompute_coeffs for it in fp64, in Pillow's order of operations, every operation correctly rounded
// and none contracted (__d*_rn: a fused 1 - |t| * ss or center - support + 0.5 rounds differently), so the int tables are
// resample_tables' bit for bit. Each image's tables sit at a fixed stride (frame_tables_stride), laid out as the offsets
// of its GhFrameDesc, which the same launch writes.
struct FrameTablesParams {
  const long long* geom;        // [N][7]: H, W, byte offset of the image in `base`, resized rh, rw, crop top, left
  const uint8_t* base;
  int* tables;                  // [N][stride]
  GhFrameDesc* frames;          // [N]
  int OH, OW, hkmax, vkmax;
  long long stride;
};

constexpr int kFrameTablesThreads = 128;

__host__ __device__ inline long long frame_tables_stride(int OH, int OW, int hkmax, int vkmax) {
  return (2LL + hkmax) * OW + (2LL + vkmax) * OH;
}

// Pillow's bilinear filter at input index `x` for an output coordinate centred at `center`: max(0, 1 - |(x - center + 0.5) * ss|)
__device__ __forceinline__ double resample_tap(int x, double center, double ss) {
  const double w = __dsub_rn(1.0, fabs(__dmul_rn(__dadd_rn(__dsub_rn((double)x, center), 0.5), ss)));
  return w > 0.0 ? w : 0.0;
}

__global__ void __launch_bounds__(kFrameTablesThreads) frame_tables_kernel(const FrameTablesParams p) {
  const long long* g = p.geom + 7LL * blockIdx.y;
  const int H = (int)g[0], W = (int)g[1];
  int* t = p.tables + p.stride * blockIdx.y;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    GhFrameDesc d;
    d.frame = p.base + g[2];
    d.pitch = 3LL * W;
    d.H = H; d.W = W; d.bgr = 0; d.reserved = 0;
    const long long t0 = p.stride * blockIdx.y, v0 = t0 + (2LL + p.hkmax) * p.OW;
    d.hx_min = t0; d.hx_size = t0 + p.OW; d.hk = t0 + 2LL * p.OW;
    d.vy_min = v0; d.vy_size = v0 + p.OH; d.vk = v0 + 2LL * p.OH;
    p.frames[blockIdx.y] = d;
  }
  const int c = blockIdx.x * kFrameTablesThreads + threadIdx.x;
  if (c >= p.OW + p.OH) return;
  const bool col = c < p.OW;
  const int in_size = col ? W : H, out_size = (int)(col ? g[4] : g[3]), kmax = col ? p.hkmax : p.vkmax;
  const int count = col ? p.OW : p.OH, i = col ? c : c - p.OW, xx = i + (int)(col ? g[6] : g[5]);
  if (!col) t += (2LL + p.hkmax) * p.OW;
  const double scale = __ddiv_rn((double)in_size, (double)out_size);
  const double support = scale < 1.0 ? 1.0 : scale;             // filterscale; bilinear support 1.0 * filterscale
  const double ss = __ddiv_rn(1.0, support);
  const double center = __dmul_rn(__dadd_rn((double)xx, 0.5), scale);
  const int lo = max((int)__dadd_rn(__dsub_rn(center, support), 0.5), 0);
  const int hi = min((int)__dadd_rn(__dadd_rn(center, support), 0.5), in_size);
  const int n = max(min(hi - lo, kmax), 0);                     // hi - lo <= kmax when kmax is the image's (the host's)
  double sum = 0.0;
  for (int x = 0; x < n; ++x) sum = __dadd_rn(sum, resample_tap(x + lo, center, ss));
  int* k = t + 2LL * count + (long long)i * kmax;
  for (int x = 0; x < kmax; ++x) {
    int v = 0;
    if (x < n) {
      double w = resample_tap(x + lo, center, ss);
      if (sum != 0.0) w = __ddiv_rn(w, sum);
      v = (int)__dadd_rn(__dmul_rn(w, (double)(1 << kPreprocPrecisionBits)), 0.5);
    }
    k[x] = v;
  }
  t[i] = lo;
  t[count + i] = n;
}

// ---- loader-side counterpart: a uint8 image batch normalised on the device -------------------------------------------------
// The reference's loaders end in ToTensor + Normalize on the host (test_RESNET50_Truncate_gram_attention.py:64-65,
// train_best_RESNET50_Truncate_gram_attention.py:42-43) and every batch crosses PCIe as fp32: 154 MB for 256 images at
// 224 x 224, 2.8 ms at the 55 GB/s the host link gives one GPU -- hidden behind the forward then, but the bound of the step
// when eight ranks share the host (25 GB/s each). Uploading the uint8 pixels (38.5 MB) and applying the two transforms
// here moves a quarter of the bytes; the arithmetic is the host's: float(b) / 255 (ToTensor), (v - mean[c]) / std[c]
// (Normalize), IEEE fp32 with correctly rounded divisions, so the fp32 batch is bit-identical to the loader's.
// A byte has 256 values and a plane one (mean, std): each CTA works inside ONE plane (grid x = plane, grid y = chunk of it,
// so no 64-bit division per element), builds the plane's 256-entry table of results once -- thread t computes
// ((float)t / 255 - mean) / std with the two correctly rounded divisions -- and the pixels become shared-memory lookups:
// the arithmetic per value is the host's, done once per byte value instead of once per pixel (the first version, which
// divided per pixel behind a 64-bit channel computation, reached 0.35 of the HBM roofline:
// profiles/r4b_normalize_u8_timing_first_version.log). One thread = kNormUnroll groups of VEC pixels, 256 threads apart:
// all loads of a thread are issued before the first use; with VEC = 4 a warp loads 128 B and stores 512 B contiguous per
// instruction.
struct NormalizeU8Params {
  const uint8_t* src;       // (N, C, H, W) uint8, dense
  float* dst;               // (N, C, H, W) fp32, dense
  long long hw;             // H * W
  int groups;               // per plane: hw / VEC
  int C;
  float mean[4], std[4];
};

constexpr int kNormUnroll = 8;

// ToTensor (/255) then Normalize ((v - mean) / std) of the byte value t, IEEE fp32 with correctly rounded divisions: the
// host's result. normalize_u8_kernel and the uint8 fused stem (stem.cuh) build their tables with it.
__device__ __forceinline__ float to_tensor_normalize(unsigned t, float mean, float std) {
  return __fdiv_rn(__fdiv_rn((float)t, 255.0f) - mean, std);
}

template <int VEC>
__global__ void __launch_bounds__(256) normalize_u8_kernel(const NormalizeU8Params p) {
  __shared__ float table[256];
  const long long plane = blockIdx.x;
  const int c = (int)(blockIdx.x % (unsigned)p.C);
  const float m = c == 0 ? p.mean[0] : c == 1 ? p.mean[1] : c == 2 ? p.mean[2] : p.mean[3];
  const float s = c == 0 ? p.std[0] : c == 1 ? p.std[1] : c == 2 ? p.std[2] : p.std[3];
  table[threadIdx.x] = to_tensor_normalize(threadIdx.x, m, s);
  __syncthreads();
  const uint8_t* __restrict__ src = p.src + plane * p.hw;
  float* __restrict__ dst = p.dst + plane * p.hw;
  const int first = blockIdx.y * (256 * kNormUnroll) + threadIdx.x;
  if (VEC == 4) {
    unsigned raw[kNormUnroll];
#pragma unroll
    for (int j = 0; j < kNormUnroll; ++j) {
      const int g = first + j * 256;
      raw[j] = g < p.groups ? __ldg(reinterpret_cast<const unsigned*>(src) + g) : 0u;
    }
#pragma unroll
    for (int j = 0; j < kNormUnroll; ++j) {
      const int g = first + j * 256;
      if (g < p.groups) {
        float4 o;
        o.x = table[raw[j] & 0xffu];
        o.y = table[(raw[j] >> 8) & 0xffu];
        o.z = table[(raw[j] >> 16) & 0xffu];
        o.w = table[raw[j] >> 24];
        __stcs(reinterpret_cast<float4*>(dst) + g, o);
      }
    }
  } else {
#pragma unroll
    for (int j = 0; j < kNormUnroll; ++j) {
      const int g = first + j * 256;
      if (g < p.groups) dst[g] = table[__ldg(src + g)];
    }
  }
}

}  // namespace gh
