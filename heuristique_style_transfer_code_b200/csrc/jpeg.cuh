// Baseline JPEG decoding on the GPU for the loaders (functions.gpu_resize_transform(decode="gpu")), bit for bit what
// Pillow's `Image.open(f).convert('RGB')` returns: libjpeg-turbo with JDCT_ISLOW, fancy upsampling and ycc_rgb_convert.
// oracle/jpeg_decode.py restates the arithmetic and is pinned to Pillow on a seeded corpus; the kernels follow it.
//
// The worker (jpeg.py) parses the headers, removes byte stuffing, splits the scan at its restart markers and builds
// each image's tables. Three phases then run on the device:
//   1. jpeg_huffman_kernel, one CTA per restart segment: self-synchronising parallel Huffman decoding (Weissenberger &
//      Schmidt, ICPP 2018). The segment is cut into subsequences of `subseq` bytes; each is decoded speculatively from
//      a guessed state at its first bit, then again from the state its predecessor reaches at the boundary, until no
//      subsequence's exit state (bit position, block within the MCU, coefficient index) changes. Block counts and DC
//      differences per component are then prefix-summed over the subsequences, and each subsequence decodes once more,
//      writing quantised coefficients (DC prediction resolved) into the coefficient workspace.
//   2. jpeg_idct_kernel: the islow IDCT of every block into component planes, as libjpeg-turbo's SIMD routines compute
//      it (16-bit dequantisation and sums, saturation after each pass; see the oracle).
//   3. jpeg_color_kernel: fancy upsampling of the chroma planes and YCbCr -> RGB (or grayscale replicated), written as
//      (H, W, 3) uint8 at the image's offset in the pixel arena that gh_frame_tables / gh_preprocess_frames read.
// Every read of scan data is bounded by its segment and every write by its image's ranges; a segment that runs out
// of bits, meets an invalid code or yields fewer blocks than the frame needs sets the image's status word.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/gramhead.h"

namespace gh {

constexpr int kJpegHuffThreads = 256;
constexpr int kJpegIdctThreads = 256;          // 8 threads per block: 32 blocks per CTA
constexpr int kJpegColorThreads = 256;
constexpr int kJpegLookahead = 9;
constexpr int kJpegRecordInts = 8;             // start_p, start_uz, exit_p, exit_uz, blocks, dc0, dc1, dc2
constexpr int kJpegBroken = 0x7fffffff;        // a bit position: the decoder met an invalid code or ran out of bits

__constant__ unsigned char kJpegNatural[64] = {
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
    28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54,
    47, 55, 62, 63};

struct JpegParams {
  const unsigned char* scan;
  long long scan_bytes;
  const long long* segs;       // [n_segs][GH_JPEG_SEG_COLS]
  const long long* imgs;       // [n_imgs][GH_JPEG_IMG_COLS]
  const int* tables;           // GH_JPEG_TABLE_INTS per image
  int n_segs, n_imgs, subseq;
  short* coef;                 // [blocks][64]
  unsigned char* planes;
  int* records;
  int* status;
  unsigned char* arena;
};

struct JpegImage {
  int H, W, ncomp, h0, v0, mcux, mcuy, bpm;
  long long coef_off, n_blocks, plane_off, arena_off;
  const int* t;
};

__device__ __forceinline__ JpegImage jpeg_image(const JpegParams& p, int i) {
  const long long* d = p.imgs + (long long)i * GH_JPEG_IMG_COLS;
  JpegImage m;
  m.H = (int)d[GH_JPEG_H]; m.W = (int)d[GH_JPEG_W]; m.ncomp = (int)d[GH_JPEG_NCOMP];
  m.h0 = (int)d[GH_JPEG_H0]; m.v0 = (int)d[GH_JPEG_V0]; m.mcux = (int)d[GH_JPEG_MCUX]; m.mcuy = (int)d[GH_JPEG_MCUY];
  m.bpm = m.ncomp == 1 ? 1 : m.h0 * m.v0 + 2;
  m.coef_off = d[GH_JPEG_COEF_OFF]; m.n_blocks = d[GH_JPEG_BLOCKS]; m.plane_off = d[GH_JPEG_PLANE_OFF];
  m.arena_off = d[GH_JPEG_ARENA_OFF];
  m.t = p.tables + d[GH_JPEG_TABLE_OFF];
  return m;
}

// 32 bits of the segment starting at bit p, MSB first; bytes past the segment read as 0xFF
__device__ __forceinline__ uint32_t jpeg_peek(const unsigned char* seg, long long len, long long p) {
  const long long i = p >> 3;
  unsigned long long v = 0;
#pragma unroll
  for (int k = 0; k < 5; ++k) v = (v << 8) | (i + k < len ? (unsigned long long)__ldg(seg + i + k) : 0xFFull);
  return (uint32_t)(v >> (8 - (int)(p & 7)));
}

// one Huffman symbol from the left-aligned bits w with table t (GH_JPEG_HUFF_INTS layout); returns length << 8 | symbol,
// or 0 for a bit pattern that starts no code
__device__ __forceinline__ int jpeg_symbol(const int* t, uint32_t w) {
  const int la = __ldg(t + (w >> (32 - kJpegLookahead)));
  if (la) return la;
  for (int l = kJpegLookahead + 1; l <= 16; ++l) {
    const int code = (int)(w >> (32 - l));
    if (code <= __ldg(t + GH_JPEG_HUFF_MAXCODE + l)) {
      const int idx = code + __ldg(t + GH_JPEG_HUFF_VALOFF + l);
      if (idx < 0 || idx > 255) return 0;
      const int sym = (__ldg(t + GH_JPEG_HUFF_VALS + (idx >> 2)) >> (8 * (idx & 3))) & 255;
      return (l << 8) | sym;
    }
  }
  return 0;
}

__device__ __forceinline__ int jpeg_extend(uint32_t v, int s) {
  return (int)v < (1 << (s - 1)) ? (int)v - (1 << s) + 1 : (int)v;
}

// component of block u of an MCU
__device__ __forceinline__ int jpeg_comp(const JpegImage& m, int u) {
  return m.ncomp == 1 ? 0 : (u < m.h0 * m.v0 ? 0 : u - m.h0 * m.v0 + 1);
}

// Decodes symbols that start in [p, end) from state (u, z). Counts completed blocks and sums DC differences per
// component; with `out`, also writes the coefficients of block `blk` on (DC as pred + diff) and stops after block
// `last`. Returns the bit position of the first symbol at or past `end`, or kJpegBroken.
__device__ __forceinline__ long long jpeg_run(const JpegImage& m, const unsigned char* seg, long long len, long long p,
                                              long long end, int& u, int& z, int& blocks, int& dc0, int& dc1, int& dc2,
                                              short* out, long long blk, long long last) {
  const long long nbits = len * 8;
  while (p < end) {
    const int c = jpeg_comp(m, u);
    const int* ht = m.t + GH_JPEG_QUANT_INTS + (2 * c + (z > 0)) * GH_JPEG_HUFF_INTS;
    const uint32_t w = jpeg_peek(seg, len, p);
    const int ls = jpeg_symbol(ht, w);
    if (!ls) return kJpegBroken;
    const int l = ls >> 8, sym = ls & 255;
    const int r = z ? sym >> 4 : 0, s = z ? sym & 15 : sym;
    if (s > 15 || p + l + s > nbits) return kJpegBroken;
    const int v = s ? jpeg_extend((w << l) >> (32 - s), s) : 0;
    p += l + s;
    short* blkp = out ? out + (blk + blocks) * 64 : nullptr;
    if (z == 0) {
      // the three predictors stay in registers: select and write back instead of indexing an array
      const int pred = (c == 0 ? dc0 : c == 1 ? dc1 : dc2) + v;
      if (c == 0) dc0 = pred; else if (c == 1) dc1 = pred; else dc2 = pred;
      if (blkp) blkp[0] = (short)pred;
      z = 1;
    } else if (s == 0) {
      z = r == 15 ? z + 16 : 64;
    } else {
      z += r;
      if (z > 63) return kJpegBroken;
      if (blkp) blkp[kJpegNatural[z]] = (short)v;
      ++z;
    }
    if (z >= 64) {
      z = 0;
      u = u + 1 == m.bpm ? 0 : u + 1;
      ++blocks;
      if (out && blk + blocks > last) return p;
    }
  }
  return p;
}

__global__ void __launch_bounds__(kJpegHuffThreads) jpeg_huffman_kernel(const JpegParams p) {
  const long long* sd = p.segs + (long long)blockIdx.x * GH_JPEG_SEG_COLS;
  const long long start = sd[GH_JPEG_SEG_START], len = sd[GH_JPEG_SEG_LEN];
  const int img = (int)sd[GH_JPEG_SEG_IMAGE];
  if (len >= GH_JPEG_MAX_SEGMENT_BYTES) {             // bit positions below are ints: refuse, never wrap
    if (threadIdx.x == 0) atomicOr(p.status + img, 1);
    return;
  }
  const JpegImage m = jpeg_image(p, img);
  const long long first_blk = sd[GH_JPEG_SEG_MCU] * m.bpm;
  const long long want = min((long long)sd[GH_JPEG_SEG_MCUS] * m.bpm, m.n_blocks - first_blk);
  const unsigned char* seg = p.scan + start;
  const long long S = (long long)p.subseq * 8;
  const int ns = (int)max(1LL, (len * 8 + S - 1) / S);
  int* rec = p.records + (start / p.subseq + blockIdx.x) * kJpegRecordInts;
  __shared__ int s_sum[kJpegHuffThreads][4];
  __shared__ int s_total;
  // Each thread owns a contiguous chunk of subsequences and decodes it in order, so inside a chunk every subsequence
  // starts from its predecessor's exit; only a chunk's first subsequence starts from a guess (round 0) or from the
  // exit the previous chunk reached in the round before.
  const int chunk = (ns + blockDim.x - 1) / blockDim.x;
  const int k0 = min(ns, (int)threadIdx.x * chunk), k1 = min(ns, k0 + chunk);
  auto decode_chunk = [&](int sp, int suz, bool force) {
    for (int k = k0; k < k1; ++k) {
      int* r = rec + k * kJpegRecordInts;
      if (!force && k > k0 && r[0] == sp && r[1] == suz) break;     // synchronised: the rest of the chunk stands
      int u = suz >> 8, z = suz & 255, blocks = 0, dc0 = 0, dc1 = 0, dc2 = 0;
      const long long q = sp == kJpegBroken ? (long long)kJpegBroken
                          : jpeg_run(m, seg, len, sp, min((k + 1) * S, len * 8), u, z, blocks, dc0, dc1, dc2, nullptr, 0, 0);
      r[0] = sp; r[1] = suz; r[2] = (int)q; r[3] = (u << 8) | z;
      r[4] = blocks; r[5] = dc0; r[6] = dc1; r[7] = dc2;
      sp = r[2]; suz = r[3];
    }
  };
  if (k0 < k1) decode_chunk((int)(k0 * S), 0, true);
  __syncthreads();
  for (;;) {
    int sp = 0, suz = 0, changed = 0;
    if (k0 > 0 && k0 < k1) {
      const int* prev = rec + (k0 - 1) * kJpegRecordInts;
      sp = prev[2]; suz = prev[3];
      changed = sp != rec[k0 * kJpegRecordInts] || suz != rec[k0 * kJpegRecordInts + 1];
    }
    if (!__syncthreads_or(changed)) break;
    if (changed) decode_chunk(sp, suz, false);
    __syncthreads();
  }
  // exclusive prefix sums of blocks and DC differences over the subsequences
  int acc[4] = {0, 0, 0, 0};
  for (int k = k0; k < k1; ++k)
    for (int j = 0; j < 4; ++j) acc[j] += rec[k * kJpegRecordInts + 4 + j];
  for (int j = 0; j < 4; ++j) s_sum[threadIdx.x][j] = acc[j];
  __syncthreads();
  if (threadIdx.x == 0) {
    int run[4] = {0, 0, 0, 0};
    for (int t = 0; t < (int)blockDim.x; ++t)
      for (int j = 0; j < 4; ++j) { const int v = s_sum[t][j]; s_sum[t][j] = run[j]; run[j] += v; }
    s_total = run[0];
  }
  __syncthreads();
  // a broken chain decodes no further blocks, so it shows as too few; padding bits after the last block may add some
  if (threadIdx.x == 0 && s_total < want) atomicOr(p.status + img, 1);
  int base[4];
  for (int j = 0; j < 4; ++j) base[j] = s_sum[threadIdx.x][j];
  for (int k = k0; k < k1; ++k) {
    int* r = rec + k * kJpegRecordInts;
    const int blocks_before = base[0];
    int dc0 = base[1], dc1 = base[2], dc2 = base[3];
    for (int j = 0; j < 4; ++j) base[j] += r[4 + j];
    if (r[0] == kJpegBroken || blocks_before >= want) continue;
    int u = r[1] >> 8, z = r[1] & 255, blocks = 0;
    jpeg_run(m, seg, len, r[0], min((k + 1) * S, len * 8), u, z, blocks, dc0, dc1, dc2,
             p.coef + (m.coef_off + first_blk) * 64,
             blocks_before, want - 1);
  }
}

// ---- phase 2: islow IDCT ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int jpeg_wrap16(int x) { return (int)(short)x; }
__device__ __forceinline__ int jpeg_sat16(int x) { return max(-32768, min(32767, x)); }

// one 1-D pass of the islow IDCT as libjpeg-turbo's SIMD routines compute it (oracle/jpeg_decode.py _idct_1d)
__device__ __forceinline__ void jpeg_idct_1d(const int v[8], int out[8], int shift) {
  const int F0298 = 2446, F0390 = 3196, F0541 = 4433, F0765 = 6270, F0899 = 7373, F1175 = 9633, F1501 = 12299,
            F1847 = 15137, F1961 = 16069, F2053 = 16819, F2562 = 20995, F3072 = 25172;
  const int tmp2 = v[2] * F0541 + v[6] * (F0541 - F1847);
  const int tmp3 = v[2] * (F0541 + F0765) + v[6] * F0541;
  const int tmp0 = jpeg_wrap16(v[0] + v[4]) * (1 << 13);
  const int tmp1 = jpeg_wrap16(v[0] - v[4]) * (1 << 13);
  const int t10 = tmp0 + tmp3, t13 = tmp0 - tmp3, t11 = tmp1 + tmp2, t12 = tmp1 - tmp2;
  const int t0 = v[7], t1 = v[5], t2 = v[3], t3 = v[1];
  const int z3s = jpeg_wrap16(t0 + t2), z4s = jpeg_wrap16(t1 + t3);
  const int z3 = z3s * (F1175 - F1961) + z4s * F1175, z4 = z3s * F1175 + z4s * (F1175 - F0390);
  const int a0 = t0 * (F0298 - F0899) - t3 * F0899 + z3;
  const int a1 = t1 * (F2053 - F2562) - t2 * F2562 + z4;
  const int a2 = -t1 * F2562 + t2 * (F3072 - F2562) + z3;
  const int a3 = -t0 * F0899 + t3 * (F1501 - F0899) + z4;
  const int rnd = 1 << (shift - 1);
  out[0] = jpeg_sat16((t10 + a3 + rnd) >> shift); out[7] = jpeg_sat16((t10 - a3 + rnd) >> shift);
  out[1] = jpeg_sat16((t11 + a2 + rnd) >> shift); out[6] = jpeg_sat16((t11 - a2 + rnd) >> shift);
  out[2] = jpeg_sat16((t12 + a1 + rnd) >> shift); out[5] = jpeg_sat16((t12 - a1 + rnd) >> shift);
  out[3] = jpeg_sat16((t13 + a0 + rnd) >> shift); out[4] = jpeg_sat16((t13 - a0 + rnd) >> shift);
}

// component c's plane: width, height and start within the image's planes
__device__ __forceinline__ void jpeg_plane(const JpegImage& m, int c, int& pw, int& ph, long long& off) {
  const int pw0 = m.mcux * (m.ncomp == 1 ? 1 : m.h0) * 8, ph0 = m.mcuy * (m.ncomp == 1 ? 1 : m.v0) * 8;
  const int pwc = m.mcux * 8, phc = m.mcuy * 8;
  pw = c ? pwc : pw0;
  ph = c ? phc : ph0;
  off = m.plane_off + (c ? (long long)pw0 * ph0 + (long long)(c - 1) * pwc * phc : 0);
}

__global__ void __launch_bounds__(kJpegIdctThreads) jpeg_idct_kernel(const JpegParams p) {
  const int img = blockIdx.y;
  const JpegImage m = jpeg_image(p, img);
  const long long b = (long long)blockIdx.x * (kJpegIdctThreads / 8) + threadIdx.x / 8;
  const int t = threadIdx.x & 7;
  const unsigned group = 0xFFu << (threadIdx.x & 24);
  __shared__ int ws[kJpegIdctThreads / 8][8][9];
  if (b >= m.n_blocks) return;                  // whole 8-thread groups leave together
  const long long mcu = b / m.bpm;
  const int u = (int)(b - mcu * m.bpm), c = jpeg_comp(m, u);
  int by, bx;
  if (m.ncomp == 1) { by = (int)(b / m.mcux); bx = (int)(b % m.mcux); }
  else if (c == 0) { by = (int)(mcu / m.mcux) * m.v0 + u / m.h0; bx = (int)(mcu % m.mcux) * m.h0 + u % m.h0; }
  else { by = (int)(mcu / m.mcux); bx = (int)(mcu % m.mcux); }
  const short* blk = p.coef + (m.coef_off + b) * 64;
  const int* q = m.t + c * 64;
  int (*w)[9] = ws[threadIdx.x / 8];
  // pass 1: column t
  int in[8], out[8], nz = 0;
  for (int r = 0; r < 8; ++r) {
    const int cv = blk[r * 8 + t];
    nz |= r ? cv : 0;
    in[r] = jpeg_wrap16(cv * __ldg(q + r * 8 + t));
  }
  const bool dc_only = (__ballot_sync(group, nz != 0) & group) == 0;
  if (dc_only) {
    const int v = jpeg_wrap16(in[0] * 4);
    for (int r = 0; r < 8; ++r) w[r][t] = v;
  } else {
    jpeg_idct_1d(in, out, 11);
    for (int r = 0; r < 8; ++r) w[r][t] = out[r];
  }
  __syncwarp(group);
  // pass 2: row t
  for (int k = 0; k < 8; ++k) in[k] = w[t][k];
  jpeg_idct_1d(in, out, 18);
  int pw, ph;
  long long off;
  jpeg_plane(m, c, pw, ph, off);
  unsigned char* dst = p.planes + off + (long long)(by * 8 + t) * pw + bx * 8;
  for (int k = 0; k < 8; ++k) dst[k] = (unsigned char)(max(-128, min(127, out[k])) + 128);
}

// ---- phase 3: upsampling and colour ------------------------------------------------------------------------------------
__device__ __forceinline__ int jpeg_chroma(const unsigned char* s, int pw, int dw, int dh, int h0, int v0, int x, int y) {
  if (h0 == 1 && v0 == 1) return s[(long long)y * pw + x];
  if (h0 == 2 && dw <= 2) return s[(long long)(v0 == 2 ? y >> 1 : y) * pw + (x >> 1)];      // h2v1 / h2v2_upsample
  if (h0 == 1) {                                                                              // h1v2_fancy_upsample
    const int j = y >> 1, jf = (y & 1) ? min(j + 1, dh - 1) : max(j - 1, 0);
    return (3 * s[(long long)j * pw + x] + s[(long long)jf * pw + x] + ((y & 1) ? 2 : 1)) >> 2;
  }
  const int i = x >> 1, iff = (x & 1) ? min(i + 1, dw - 1) : max(i - 1, 0);
  if (v0 == 1) {                                                                              // h2v1_fancy_upsample
    const unsigned char* row = s + (long long)y * pw;
    return (3 * row[i] + row[iff] + ((x & 1) ? 2 : 1)) >> 2;
  }
  const int j = y >> 1, jf = (y & 1) ? min(j + 1, dh - 1) : max(j - 1, 0);                 // h2v2_fancy_upsample
  const unsigned char *rn = s + (long long)j * pw, *rf = s + (long long)jf * pw;
  const int cs = 3 * rn[i] + rf[i], cf = 3 * rn[iff] + rf[iff];
  return (3 * cs + cf + ((x & 1) ? 7 : 8)) >> 4;
}

__global__ void __launch_bounds__(kJpegColorThreads) jpeg_color_kernel(const JpegParams p) {
  const JpegImage m = jpeg_image(p, blockIdx.y);
  const long long px = (long long)blockIdx.x * kJpegColorThreads + threadIdx.x;
  if (px >= (long long)m.H * m.W) return;
  const int y = (int)(px / m.W), x = (int)(px - (long long)y * m.W);
  int pw, ph;
  long long off;
  jpeg_plane(m, 0, pw, ph, off);
  const int Y = p.planes[off + (long long)y * pw + x];
  unsigned char* dst = p.arena + m.arena_off + px * 3;
  if (m.ncomp == 1) { dst[0] = dst[1] = dst[2] = (unsigned char)Y; return; }
  const int dw = (m.W + m.h0 - 1) / m.h0, dh = (m.H + m.v0 - 1) / m.v0;
  int pwc, phc;
  long long o1, o2;
  jpeg_plane(m, 1, pwc, phc, o1);
  jpeg_plane(m, 2, pwc, phc, o2);
  const int cb = jpeg_chroma(p.planes + o1, pwc, dw, dh, m.h0, m.v0, x, y) - 128;
  const int cr = jpeg_chroma(p.planes + o2, pwc, dw, dh, m.h0, m.v0, x, y) - 128;
  const int r = Y + ((91881 * cr + 32768) >> 16);
  const int g = Y + ((-22554 * cb + 32768 - 46802 * cr) >> 16);
  const int bl = Y + ((116130 * cb + 32768) >> 16);
  dst[0] = (unsigned char)max(0, min(255, r));
  dst[1] = (unsigned char)max(0, min(255, g));
  dst[2] = (unsigned char)max(0, min(255, bl));
}

}  // namespace gh
