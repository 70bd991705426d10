/* gramhead.h - C ABI of libgramhead.so, the sm_100a implementation of the Gram + attention style-feature head of
 * Hamedkiri/heuristique_style_transfer_code (model "TruncatedResNet50 + Gram + Attention").
 *
 * Every entry point replaces a piece of the reference's Python hot path; the reference interface each one stands
 * in for is cited as file:line relative to the reference tree. The reference has no FFI of its own (it is pure
 * PyTorch), so the binding a maintainer adds is the ctypes stub shown in INTEGRATION.md.
 *
 * Conventions
 *   - all pointers are DEVICE pointers on the current CUDA device unless stated otherwise;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream); calls only enqueue work, they never
 *     synchronise the host and never allocate device memory;
 *   - tensors are dense row-major unless a stride argument says otherwise; fp32 buffers must be 4-byte aligned
 *     (16-byte alignment enables the vector load path);
 *   - return value: 0 = ok; > 0 = a cudaError_t from the launch; < 0 = GH_ERR_* below.
 */
#ifndef GRAMHEAD_H_
#define GRAMHEAD_H_

#ifdef __cplusplus
extern "C" {
#endif

#define GH_ERR_BAD_ARG (-1)       /* null pointer / non-positive size */
#define GH_ERR_UNSUPPORTED (-2)   /* shape outside what this entry point implements; see its comment */

#define GH_DTYPE_F32 0
#define GH_DTYPE_BF16 1

/* Library version (major*10000 + minor*100 + patch). */
int gh_version(void);

/* Number of SMs the launchers size their persistent grids by (cudaDevAttrMultiProcessorCount of the current device). */
int gh_sm_count(void);

/* Launch tuning, process-wide. Known names (unknown name or value outside the allowed set: GH_ERR_BAD_ARG):
 *   "gram_fwd_pair", "gram_bwd_pair"   -1 = CTA-pair (TMA-staged) kernels whenever TMA can describe the tensors (default),
 *                                      0 = never (ld.global-fed kernels), 1 = same as -1
 *   "gram_bwd_nt"                      0 = plan the x-tile width of the pair backward; 64..256 (multiple of 16) forces it
 *   "gram_bwd_stages"                  0 = by shape; a*16 + b = A / F ring depths of the pair backward (a >= 4)
 *   "gram_bwd_ats"                     pooled pair backward with the generated gradient tile in tensor memory (the MMAs read
 *                                      their A operand from TMEM): 0 = never, 1 = whenever the TMEM columns behind the two
 *                                      accumulators hold the A ring, -1 = for C >= 512 only (default)
 *   "gram_bwd_ch"                      K chunks per ring stage of that form (MMAs per iteration of the issuing thread / 4):
 *                                      0 = as many as fit, at most 2 (default), 1, 2
 *   "tgemm_tn"                         tile width of the TMA-fed attention GEMMs: 0 = planned (default), 128, 256
 *   "pdl"                              1 = programmatic dependent launch along the attention kernel chain (default), 0 = off */
int gh_set_option(const char* name, int value);

/* Reads and clears the error record {code, blockIdx.x, threadIdx.x, site} of the current device into host memory `out4`.
 * code 1 = an mbarrier wait inside a kernel ran out of time (the kernel then traps instead of hanging the GPU). The
 * record lives in mapped pinned host memory, so it can be read after the trap, when the CUDA context itself only
 * returns errors; no CUDA call is made once the record exists. GH_ERR_UNSUPPORTED when it could not be allocated. */
int gh_last_device_error(unsigned int* out4);

/* Pooled Gram, forward.  Replaces, for one encoder stage l of L,
 *   gram_matrix():            Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:26-30 (bmm + div(h*w))
 *   adaptive_avg_pool2d:      :51-52
 *   stack/flatten (layout):   :54-55
 * F: (B, C, HW) features, element (b,c,x) at F[b*img_stride + c*row_stride + x*x_stride], dtype f_dtype. Two layouts:
 *   x contiguous (NCHW as cuDNN's default leaves it):  x_stride == 1, row_stride >= HW;
 *   c contiguous (channels_last / NHWC):               row_stride == 1, x_stride >= C  (CTA-pair kernels only:
 *   GH_ERR_UNSUPPORTED when TMA cannot describe the tensor -- transpose with gh_transpose_cast instead).
 * desc: (B, L, g*g) fp32; this call overwrites desc[:, l, :] with vec_rowmajor(pool_g(F F^T / HW)).
 * Requires C % g == 0 and k = C/g a power of two in [8, 128] (returns GH_ERR_UNSUPPORTED otherwise: use
 * gh_gram_dense_fwd + gh_adaptive_pool_fwd, which implement torch's general bin rule).
 * ksplit: number of K (=HW) partitions per tile whose partial sums meet in fp32 atomics; 0 = choose for load balance,
 * 1 = deterministic summation order. max_ctas: 0 = one persistent CTA per SM. */
int gh_gram_pool_fwd(const void* F, int f_dtype, long long img_stride, long long row_stride, long long x_stride, int B,
                     int C, int HW, int g, float* desc, int l, int L, int ksplit, int max_ctas, void* stream);

/* Dense Gram, forward: G[b] = F[b] F[b]^T / HW, (B, C, C) fp32, both triangles written.
 * Replaces gram_matrix() used on its own (:26-30; style-transfer mode,
 * functions/functions_RESNET50_Truncate_Gram_Attention.py:273-275,290-291). */
int gh_gram_dense_fwd(const void* F, int f_dtype, long long img_stride, long long row_stride, long long x_stride, int B,
                      int C, int HW, float* G, int ksplit, int max_ctas, void* stream);

/* torch.nn.functional.adaptive_avg_pool2d(G, (g, g)) on (B, C, C) with torch's bin rule
 * [floor(i*C/g), ceil((i+1)*C/g)), written to desc[:, l, :] of a (B, L, g*g) buffer.  (:51-55) */
int gh_adaptive_pool_fwd(const float* G, int B, int C, int g, float* desc, int l, int L, void* stream);
/* Its backward (AdaptiveAvgPool2DBackward of Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:51-52, reached from
 * loss.backward(), functions/functions_RESNET50_Truncate_Gram_Attention.py:135): dG (B, C, C) from d_desc[:, l, :]. */
int gh_adaptive_pool_bwd(const float* d_desc, int l, int L, int B, int C, int g, float* dG, void* stream);

/* Pooled Gram, backward: what loss.backward() (functions/functions_RESNET50_Truncate_Gram_Attention.py:135) runs for
 * Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:26-30, :51-52, :54-55 (BmmBackward, DivBackward,
 * AdaptiveAvgPool2DBackward, StackBackward):
 *   dF[b] = (dG + dG^T) F[b] / HW,  dG[c][d] = d_desc[b, l, (c/k)*g + d/k] / k^2.
 * dF: dtype df_dtype, element (b,c,x) at dF[b*df_img_stride + c*df_row_stride + x*df_x_stride]; overwritten. F and dF
 * must use the same layout (both x contiguous or both c contiguous, see gh_gram_pool_fwd). df_dtype = GH_DTYPE_BF16
 * writes the gradient as bf16 straight from the accumulators (half the bytes; what a bf16 backbone's backward
 * consumes): CTA-pair kernels only, GH_ERR_UNSUPPORTED when they do not apply (then ask for fp32 and cast).
 * Requires C % g == 0, k a power of two, g <= 64, C % 16 == 0. */
int gh_gram_pool_bwd(const void* F, int f_dtype, long long img_stride, long long row_stride, long long x_stride, int B,
                     int C, int HW, int g, const float* d_desc, int l, int L, void* dF, int df_dtype,
                     long long df_img_stride, long long df_row_stride, long long df_x_stride, int max_ctas, void* stream);

/* Dense Gram, backward (autograd of gram_matrix(), Models/...Attention.py:26-30, as style transfer drives it:
 * functions/functions_RESNET50_Truncate_Gram_Attention.py:293): dF[b] = (dG[b] + dG[b]^T) F[b] / HW with dG (B, C, C) fp32.
 * Requires C % 16 == 0. */
int gh_gram_dense_bwd(const void* F, int f_dtype, long long img_stride, long long row_stride, long long x_stride, int B,
                      int C, int HW, const float* dG, void* dF, int df_dtype, long long df_img_stride,
                      long long df_row_stride, long long df_x_stride, int max_ctas, void* stream);

/* Attention over the L stage descriptors + mean over stages + classifier, forward.  Replaces
 *   permute + self.attention(X, X, X) (nn.MultiheadAttention, 1 head): :56-58
 *   .mean(dim=0):                                                     :59
 *   self.classifier(...):                                             :61 / :113-114
 * desc (B, L, E) fp32 with E = g*g; W_in (3E, E), b_in (3E), W_out (E, E), b_out (E), W_c (nc, E), b_c (nc):
 * the tensors of attention.in_proj_weight/.in_proj_bias/.out_proj.weight/.out_proj.bias and classifier.weight/.bias.
 * Outputs: emb (B, E) (the `embeddings` of TruncatedResNet50_for_test), logits (B, nc); saved for backward:
 * qkv (B*L, 3E), probs (B, L, L), obar (B, E). L <= 8. */
int gh_attn_head_fwd(const float* desc, const float* W_in, const float* b_in, const float* W_out, const float* b_out,
                     const float* W_c, const float* b_c, int B, int L, int E, int nc, float* qkv, float* probs,
                     float* obar, float* emb, float* logits, void* stream);

/* Batched transpose with optional cast: out[b][s][r] = cast(in[b][r][s]); in (B, R, S) dense, out (B, S, out_pitch)
 * with out_pitch >= R elements between rows (padding a C x HW matrix's rows to a multiple of 16 B makes it
 * describable by a TMA tensor map, e.g. HW = 196 in bf16); dtypes GH_DTYPE_F32 / GH_DTYPE_BF16 in any combination. Hand-off with a channels_last (NHWC) backbone: the
 * reference's gram_matrix() begins with activations.view(b, ch, h*w)
 * (Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:27-28) and so needs each image as a C x HW matrix with HW
 * contiguous; an NHWC activation is the HW x C transpose of it (forward: R = HW, S = C), and the fp32 NCHW gradient
 * goes back to NHWC in the activation's dtype (backward: R = C, S = HW). */
int gh_transpose_cast(const void* in, int in_dtype, void* out, int out_dtype, int B, int R, int S, long long out_pitch,
                      void* stream);

/* Camera-mode preprocessing of one frame on the GPU, bit-identical to the reference's per-frame host code
 *   functions/functions_RESNET50_Truncate_Gram_Attention.py:499-501  cv2.cvtColor(BGR2RGB) -> Image.fromarray -> transform
 *   test_RESNET50_Truncate_gram_attention.py:61-66                   Resize [+ CenterCrop] + ToTensor + Normalize
 * (torchvision Resize on a PIL image = Pillow's fixed-point, antialiased bilinear ImagingResample).
 * frame: (H, W, 3) uint8 on the device, pitch_bytes between rows; bgr != 0: channels are B,G,R (OpenCV).
 * hx_min/hx_size [OW], hk [OW][hkmax]: per output column the first contributing input column, their number and
 * the 22-bit fixed-point coefficients; vy_min/vy_size [OH], vk [OH][vkmax]: the same for rows. A centre crop is the
 * sub-range of output coordinates the tables are built for (streaming.py computes them once per geometry).
 * mean3_host / std3_host: HOST pointers to 3 floats. out: (3, OH, OW) fp32 = (x/255 - mean) / std. */
int gh_preprocess_frame(const unsigned char* frame, long long pitch_bytes, int H, int W, int bgr, const int* hx_min,
                        const int* hx_size, const int* hk, int hkmax, const int* vy_min, const int* vy_size, const int* vk,
                        int vkmax, const float* mean3_host, const float* std3_host, float* out, int OH, int OW,
                        void* stream);

/* Several camera or video frames per call: the resize [+ centre crop] of gh_preprocess_frame for N frames of any sizes
 * at once, written as one dense (N, 3, OH, OW) uint8 batch in RGB order -- the rounded bytes gh_preprocess_frame divides
 * by 255 and normalises, so that ToTensor + Normalize applied to this batch (gh_normalize_u8, or the uint8 stem
 * gh_stem_conv_pool_u8_nhwc) gives its fp32 output bit for bit. One record per frame, in DEVICE memory (it does not
 * change between calls, so a CUDA graph can hold it); the table offsets count int elements from `tables`: */
typedef struct GhFrameDesc {
  const unsigned char* frame;   /* (H, W, 3) uint8 on the device, `pitch` bytes between rows */
  long long pitch;
  int H, W;
  int bgr;                      /* != 0: channels are B,G,R (OpenCV); the output is RGB either way */
  int reserved;                 /* 0 */
  long long hx_min, hx_size;    /* [OW] first contributing input column and their number */
  long long hk;                 /* [OW][hkmax] 22-bit fixed-point coefficients, rows padded with zeros to hkmax */
  long long vy_min, vy_size;    /* [OH] the same for rows */
  long long vk;                 /* [OH][vkmax] */
} GhFrameDesc;                  /* 80 bytes */

/* frames: [N] descriptors (device). tables: the packed int tables (device). Each CTA resamples `band_rows` output rows of
 * one frame, holding the horizontally filtered input rows they read in shared memory, at most `span_rows` of them at a
 * time: span_rows >= vkmax (one output row always fits); a band that needs more input rows is done in several runs, so
 * any band_rows is correct and the caller picks it for speed (streaming.py: the most input rows any band of that height
 * needs). out: (N, 3, OH, OW) uint8. N <= 65535 and ceil(OH / band_rows) <= 65535 (GH_ERR_UNSUPPORTED beyond); the
 * shared memory gh_preprocess_frames_smem(OW, span_rows) must be available (GH_ERR_UNSUPPORTED otherwise). */
int gh_preprocess_frames(const GhFrameDesc* frames, int N, int OH, int OW, int band_rows, int span_rows, const int* tables,
                         int hkmax, int vkmax, unsigned char* out, void* stream);
/* Host-only: the shared-memory bytes of one gh_preprocess_frames CTA holding span_rows filtered rows of width OW;
 * GH_ERR_BAD_ARG for non-positive sizes, GH_ERR_UNSUPPORTED above what one CTA can have. No GPU needed. */
int gh_preprocess_frames_smem(int OW, int span_rows);

/* The tables and descriptors of gh_preprocess_frames for a batch of N images of any sizes, built on the device (a loader
 * has new sizes in every batch). geom: [N][7] long long in DEVICE memory, per image H, W, the byte offset of its (H, W, 3)
 * RGB pixels (pitch 3 * W) from `base`, its resized size rh, rw and the centre crop's top, left (OH x OW from there;
 * top + OH <= rh, left + OW <= rw). hkmax / vkmax: at least every image's 2 * ceil(max(W / rw, 1)) + 1, resp. for H / rh.
 * Writes, per image i, the tables of streaming.resample_tables(W, rw, left, OW) and (H, rh, top, OH) -- bit for bit: fp64
 * in Pillow's order of operations, none fused -- at tables + i * gh_frame_tables_stride(...), coefficient rows padded
 * with zeros to hkmax / vkmax, and frames[i] = { base + offset, 3 * W, H, W, RGB, offsets of those tables }.
 * N <= 65535 (GH_ERR_UNSUPPORTED beyond). */
int gh_frame_tables(const long long* geom, int N, const unsigned char* base, int OH, int OW, int hkmax, int vkmax,
                    int* tables, GhFrameDesc* frames, void* stream);
/* Host-only: the ints of one image's tables in gh_frame_tables' layout, (2 + hkmax) * OW + (2 + vkmax) * OH;
 * GH_ERR_BAD_ARG for non-positive sizes. */
long long gh_frame_tables_stride(int OH, int OW, int hkmax, int vkmax);

/* Loader-side counterpart of gh_preprocess_frame: a dense (images, channels, H, W) uint8 batch -> the fp32 batch the
 * reference's loader transforms produce on the host, transforms.ToTensor() + transforms.Normalize(mean, std)
 * (test_RESNET50_Truncate_gram_attention.py:64-65, train_best_RESNET50_Truncate_gram_attention.py:42-43):
 *   dst = (float(src) / 255 - mean[c]) / std[c]   in IEEE fp32, bit-identical to the host result,
 * so that a loader can hand over uint8 pixels (a quarter of the PCIe bytes) and the model still sees the same tensor.
 * mean_host / std_host: HOST pointers to `channels` floats (channels <= 4, std != 0); hw = H * W. */
int gh_normalize_u8(const unsigned char* src, float* dst, long long images, int channels, long long hw,
                    const float* mean_host, const float* std_host, void* stream);

/* The GEMM the attention entry points are built from, exposed for testing and reuse:
 *   D[m*ldd + n] = sum_k A[m*a_sm + k*a_sk] * B[k*b_sk + n*b_sn] (+ bias[n]),   fp32 in, fp32 out.
 * Runs on tcgen05 with split-bf16 operands (hi*hi + hi*lo + lo*hi, fp32 accumulate: ~1e-5 relative) when each operand
 * is contiguous along one of its two axes with 16 B aligned rows and N >= 64; otherwise on the fp32 FMA kernel. Stands in for the F.linear / matmul calls inside
 * torch.nn.functional.multi_head_attention_forward that the reference reaches through self.attention (:58). */
int gh_gemm_f32(const float* A, long long a_sm, long long a_sk, const float* B, long long b_sk, long long b_sn,
                const float* bias, float* D, long long ldd, int M, int N, int K, void* stream);

/* gh_gemm_f32 on the same routes, but K is never split: every output element has one writer and K is reduced in a fixed
 * order, so the result is the same bits on every run (gh_gemm_f32 may split a long K over CTAs that meet in reduce-adds
 * when the output has fewer tiles than the GPU has SMs). For weight gradients, whose K is the batch. */
int gh_gemm_f32_fixed(const float* A, long long a_sm, long long a_sk, const float* B, long long b_sk, long long b_sn,
                      const float* bias, float* D, long long ldd, int M, int N, int K, void* stream);

/* out[n] = sum_{m < M} X[m*ldx + n] for n < N, summed in a fixed order (bias gradients over the rows of a batch). */
int gh_colsum_f32(const float* X, long long ldx, int M, int N, float* out, void* stream);

/* Max pooling of a channels_last activation, values only (inference plan of the encoder, frozen_encoder.py). Replaces the
 * nn.MaxPool2d child of the truncated encoder (torchvision resnet `maxpool`: kernel 3, stride 2, padding 1; child 3 of
 * `self.truncated_encoder`, Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:17,40) under eval + no_grad, where
 * the argmax indices ATen's kernel also produces are not needed. in: (B, H, W, C) dense NHWC storage of a (B, C, H, W)
 * channels_last tensor, fp32 or bf16; out: (B, OH, OW, C) with OH = (H + 2*pad - k)/stride + 1 (floor mode, dilation 1).
 * NaN-propagating like ATen; bit-identical results. C % 4 == 0 (fp32) / C % 8 == 0 (bf16), 16 B aligned pointers. */
int gh_maxpool2d_nhwc(const void* in, int dtype, void* out, int B, int H, int W, int C, int k, int stride, int pad,
                      void* stream);

/* Space-to-depth staging of the image batch for the stem convolution of the inference plan (frozen_encoder.py): the
 * stem `conv1` (7x7, stride 2, padding 3, 3 input channels; child 0 of `self.truncated_encoder`,
 * Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:17,37) is evaluated by cuDNN as the equivalent 4x4 stride-1
 * convolution over z, which this call builds in place of the NCHW -> channels_last conversion of the input:
 *   z[b, Y + 2, X + 2, c*4 + r*2 + s] = x[b, c, 2Y + r, 2X + s],  zero elsewhere,
 * z: dense NHWC storage of a (B, 16, H/2 + 3, W/2 + 3) channels_last tensor, fp32 or bf16 (z_dtype); x: fp32 with the
 * given element strides (NCHW or channels_last). H and W even (GH_ERR_UNSUPPORTED otherwise). */
int gh_stem_space_to_depth(const float* x, long long img_stride, long long c_stride, long long y_stride,
                           long long x_stride, int B, int H, int W, void* z, int z_dtype, void* stream);

/* The whole stem of the inference plan in one kernel (csrc/stem.cuh): conv1 (7x7, stride 2, padding 3) with bn1 folded
 * in, relu and maxpool (3, stride 2, padding 1) -- children 0-3 of `self.truncated_encoder`,
 * Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:17,37-40 -- in place of gh_stem_space_to_depth, the cuDNN
 * convolution and gh_maxpool2d_nhwc. tf32 operands (rounded to nearest, ties away), fp32 accumulation (kind::tf32).
 * x: fp32 (B, 3, H, W) with the given element strides (NCHW, channels_last or strided), H and W even
 * (GH_ERR_UNSUPPORTED otherwise). w_packed: the 64 x 256 folded space-to-depth weights (frozen_encoder.py,
 * _stem_space_to_depth_weight) rounded to tf32 and laid out as the kernel's shared-memory B operands:
 * [tap a*4+b][half h][k-chunk q][out channel n][4] = W16[n][(2h + q)*4 + e][a][b], 16384 floats, 16 B aligned.
 * bias: [64]. out: (B, PH, PW, 64) dense NHWC storage of a channels_last (B, 64, PH, PW) tensor, 16 B aligned,
 * PH = (H/2 - 1)/2 + 1, PW = (W/2 - 1)/2 + 1 (nn.MaxPool2d's floor mode). NaN propagates as in the reference. */
int gh_stem_conv_pool_nhwc(const float* x, long long img_stride, long long c_stride, long long y_stride,
                           long long x_stride, int B, int H, int W, const float* w_packed, const float* bias, float* out,
                           void* stream);

/* gh_stem_conv_pool_nhwc on the uint8 pixels of the loaders (functions.uint8_transform) with ToTensor + Normalize
 * applied inside it -- the transforms of the reference's loaders, test_RESNET50_Truncate_gram_attention.py:64-65 and
 * train_best_RESNET50_Truncate_gram_attention.py:42-43, in front of the stem, children 0-3 of `self.truncated_encoder`,
 * Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:17,37-40 -- in place of gh_normalize_u8 followed by
 * gh_stem_conv_pool_nhwc, without the fp32 batch. Each pixel becomes (float(b) / 255 - mean[c]) / std[c] exactly as in
 * gh_normalize_u8, so `out` is bit for bit what those two calls produce. x: uint8 (B, 3, H, W) with the given element
 * strides; zero padding applies after Normalize. mean3_host / std3_host: HOST pointers to 3 floats each (std neither
 * zero nor NaN: GH_ERR_BAD_ARG). w_packed, bias, out, H, W: as for gh_stem_conv_pool_nhwc. */
int gh_stem_conv_pool_u8_nhwc(const unsigned char* x, long long img_stride, long long c_stride, long long y_stride,
                              long long x_stride, int B, int H, int W, const float* mean3_host, const float* std3_host,
                              const float* w_packed, const float* bias, float* out, void* stream);

/* ---- Gram head of the Multi-PatchGAN discriminator (the *_test classes of Models/Models_Multi_PatchGAN.py) ----------
 * gh_patch_gram_fwd replaces, for all L collected feature maps of one discriminator in one launch,
 *   F.layer_norm(x_proj, x_proj.shape[1:])                  :198   (only when ln_input != 0; otherwise pass the
 *                                                                    already normalised maps of :199)
 *   F.adaptive_avg_pool2d(feature_map, (4, 4))              :210
 *   F.layer_norm(pooled, pooled.shape[1:])                  :213
 *   torch.bmm(fm, fm^T) / (16 + 1e-6)                       :217-220
 *   torch.norm(gram, p='fro', dim=(1, 2))                   :223
 * maps[l]: device pointer to layer l's (B, D, H[l], W[l]) fp32 map; strides[4*l..4*l+3] = its image / channel / row /
 * column strides in elements (any layout; NCHW is the coalesced one). maps, H, W, strides are HOST arrays of length L
 * (4L for strides). L <= 8, D <= 128 (GH_ERR_UNSUPPORTED beyond). gram: (L, B, D*D) row-major flattened as :226 does;
 * gram_norm: (L, B).
 * workspace: gh_patch_gram_workspace(L, B, D) fp32 elements, 8 B aligned (bin means and per-channel sums between the two
 * launches: a pooling pass with one warp per channel plane, then one CTA per (image, layer) for the norms and the Gram). */
long long gh_patch_gram_workspace(int L, int B, int D);
int gh_patch_gram_fwd(const float* const* maps, const int* H, const int* W, const long long* strides, int L, int B,
                      int D, int ln_input, float* gram, float* gram_norm, float* workspace, void* stream);

/* gh_patch_attn_fwd replaces
 *   attention_per_layer(x, x, x), attention_per_patch(y, y, y)   :243-244  (nn.MultiheadAttention(ndf, heads), sequence =
 *                                                                           the L layers, dropout 0, no masks)
 *   torch.mean(..., dim=0)                                       :247
 *   self.classifier(aggregated_features)                         :256
 * feat: (L, B, E) projected Gram features (the stack of :240; the Linear of :229 is gh_gemm_f32 over the L*B rows of
 * gh_patch_gram_fwd's output). W_in* (3E, E), b_in* (3E), W_out* (E, E), b_out* (E): in_proj_weight / in_proj_bias /
 * out_proj.weight / out_proj.bias of the two attention modules; W_c (nc, E), b_c (nc). emb: (B, E) `embeddings`,
 * logits: (B, nc) `output`. L <= 8, E <= 128, E % 4 == 0, E % heads == 0, 16 B-aligned weights. */
int gh_patch_attn_fwd(const float* feat, const float* W_in1, const float* b_in1, const float* W_out1,
                      const float* b_out1, const float* W_in2, const float* b_in2, const float* W_out2,
                      const float* b_out2, const float* W_c, const float* b_c, int L, int B, int E, int heads, int nc,
                      float* emb, float* logits, void* stream);

/* ---- Backward of the Multi-PatchGAN Gram head ------------------------------------------------------------------------
 * Per image and collected layer the forward is x^ = LN(X) (:198, with ln_input), P = pool4x4(x^) (:210),
 * Z = LN(P) over (D, 16) (:213), G = Z Z^T / (16 + 1e-6) (:217-220), n = |G|_F (:223), feat = vec(G) W^T + b (:229).
 *
 * gh_patch_gram_bwd: from d_gram (L, B, D*D) and d_norm (L, B), the backward of :213-223 and of the pooling's bin
 * weights, per (image, layer):  dG += dn G / n (0 where n == 0, as torch's norm backward);  dZ = (dG + dG^T) Z /
 * (16 + 1e-6);  dP = r2 (dZ - mean dZ - Z mean(dZ Z)). It writes bwd_workspace (gh_patch_bwd_workspace(L, B, D) floats,
 * 16 B aligned): the table r dP[d][i] / |bin i| (L, B, D, 16), then per (layer, image) the scalars a = -r sum(dP) / N,
 * c = -r^2 sum(dP P) / N and the map mean mu (0, 0, 0 without ln_input; N = D H W; r: the map's rstd, 1 without
 * ln_input). Z, r and mu are recomputed with the forward's own code from fwd_workspace (gh_patch_gram_fwd's workspace,
 * unchanged since that call); gram_norm is that call's output. H, W: HOST arrays of length L.
 * gh_patch_pool_bwd: one pass that writes the gradient of every map,
 *   dX(d, y, x) = sum over the 4x4 adaptive bins i holding (y, x) of table[d][i] + a + c (X(d, y, x) - mu),
 * i.e. the pooling's backward (ATen's bins overlap when H % 4 != 0) and, with ln_input, the whole-map layer norm's
 * backward r (dx^ - mean dx^ - x^ mean(dx^ x^)), whose two means are exact functions of the 16 D bin values. X (maps,
 * strides as in gh_patch_gram_fwd) is read only when ln_input != 0. d_maps / d_strides: the gradients and their element
 * strides (any layout: pass the map's own layout, channels_last included). L <= 8, D <= 128 (GH_ERR_UNSUPPORTED beyond). */
long long gh_patch_bwd_workspace(int L, int B, int D);
int gh_patch_gram_bwd(const int* H, const int* W, int L, int B, int D, int ln_input, const float* d_gram,
                      const float* d_norm, const float* gram_norm, const float* fwd_workspace, float* bwd_workspace,
                      void* stream);
int gh_patch_pool_bwd(const float* const* maps, float* const* d_maps, const int* H, const int* W,
                      const long long* strides, const long long* d_strides, int L, int B, int D, int ln_input,
                      const float* bwd_workspace, void* stream);

/* gh_patch_attn_bwd: backward of gh_patch_attn_fwd (:243-256) from d_emb (B, E) and d_logits (B, nc), one CTA per image:
 * the image's forward is recomputed in shared memory, then classifier, mean over layers (:247), and for
 * attention_per_patch then attention_per_layer: out_proj, softmax attention (q scaled by sqrt(1/hd)), in_proj. Writes
 * d_feat (L, B, E) and the rows the weight gradients are GEMMs over (gh_gemm_f32_fixed / gh_colsum_f32 over the L*B rows):
 * x1 (L, B, E) the input of attention_per_patch (the input of attention_per_layer is feat), and for a = 0 (per layer), 1
 * (per patch): dqkv[a] (L, B, 3E) the gradient of the in_proj output, o[a] (L, B, E) the out_proj input, dy[a] (L, B, E)
 * the gradient of the attention's output. Same weights and limits as gh_patch_attn_fwd (b_c is not needed). */
int gh_patch_attn_bwd(const float* feat, const float* W_in1, const float* b_in1, const float* W_out1,
                      const float* b_out1, const float* W_in2, const float* b_in2, const float* W_out2,
                      const float* b_out2, const float* W_c, const float* d_emb, const float* d_logits, int L, int B,
                      int E, int heads, int nc, float* d_feat, float* x1, float* dqkv, float* o, float* dy,
                      void* stream);

/* Number of fp32 elements gh_attn_head_bwd needs in `workspace`. */
long long gh_attn_head_bwd_workspace(int B, int L, int E);

/* Backward of gh_attn_head_fwd (what loss.backward() runs for those lines; functions/...Attention.py:135).
 * Inputs: the forward's inputs and saved tensors, d_logits (B, nc), d_emb_ext (B, E) or NULL (gradient arriving
 * directly at the embeddings output). Outputs (each may be NULL to skip it; all are overwritten, not accumulated):
 * d_desc (B, L, E), dW_in, db_in, dW_out, db_out, dW_c, db_c. */
int gh_attn_head_bwd(const float* desc, const float* W_in, const float* W_out, const float* W_c, const float* qkv,
                     const float* probs, const float* obar, const float* emb, const float* d_logits,
                     const float* d_emb_ext, int B, int L, int E, int nc, float* d_desc, float* dW_in, float* db_in,
                     float* dW_out, float* db_out, float* dW_c, float* db_c, float* workspace, void* stream);

/* Style-transfer loss on the dense Gram (SURVEY 8(f) n3). Replaces `loss = mse_loss(noise_gram, original_gram)` and the
 * element-wise part of `loss.backward()` (functions/functions_RESNET50_Truncate_Gram_Attention.py:291-295):
 *   partial[i] = sum over block i's elements of (G - G_target)^2 / n     (loss = sum_i partial[i], i < gh_gram_mse_blocks(n))
 *   dG         = 2 (G - G_target) / n                                      (d loss / d G; feed it to gh_gram_dense_bwd)
 * G, G_target, dG: n = B*C*C fp32 elements, 16 B aligned (any n). */
int gh_gram_mse_blocks(long long n);
int gh_gram_mse(const float* G, const float* G_target, long long n, float* dG, float* partial, void* stream);

/* The same loss with one value per image, for several style-transfer images optimised in one step (the reference's loop
 * of functions/functions_RESNET50_Truncate_Gram_Attention.py:283-299 runs each image's `mse_loss(noise_gram,
 * original_gram)` and `loss.backward()` on its own, :291-295). G, G_target, dG: (B, C, C) fp32, n_img = C*C, k =
 * gh_gram_mse_images_blocks(n_img) (= gh_gram_mse_blocks(n_img)):
 *   partial[b*k + i] = sum over block i of image b of (G - G_target)^2 / n_img     (mse_b = sum_i partial[b*k + i])
 *   dG               = 2 (G - G_target) / n_img                                    (d (sum_b mse_b) / d G)
 * Image b's partials and dG slice are bitwise what gh_gram_mse gives on a 16 B-aligned copy of that image alone. Any
 * n_img: images that do not start on a 16 B boundary (n_img % 4 != 0) are read with scalar loads. B <= 65535. */
int gh_gram_mse_images_blocks(long long n_img);
int gh_gram_mse_images(const float* G, const float* G_target, int B, long long n_img, float* dG, float* partial,
                       void* stream);

/* ---- Attention head on TMA-fed tensor-core GEMMs (the default whenever E % 64 == 0, E <= 1024, L <= 8, nc <= 16) -------
 * Same reference lines as gh_attn_head_fwd / gh_attn_head_bwd (Models/...Attention.py:56-61 and its autograd), other
 * operand format: every matrix that feeds a linear layer travels as "split planes" -- two bf16 matrices of the same
 * shape, hi = bf16(x) and lo = bf16(x - hi), `plane_stride` elements apart -- which tcgen05 consumes straight from
 * TMA-staged shared memory with three MMAs per k-step (lo*hi + hi*lo + hi*hi, fp32 accumulate: fp32-level accuracy).
 *
 * gh_split_bf16: planes[i] = bf16(src[i]), planes[plane_stride + i] = bf16(src[i] - hi) for i < n. Called once per
 * WEIGHT VERSION for attention.in_proj_weight and attention.out_proj.weight (the host caches the planes), and by
 * gh_attn_head_fwd2 for the descriptors. n % 4 == 0, src 16 B aligned. */
int gh_split_bf16(const float* src, void* planes, long long n, long long plane_stride, void* stream);

/* The GEMM gh_attn_head_fwd2 / _bwd2 are built from (the F.linear / matmul calls torch's multi_head_attention_forward makes
 * for self.attention, Models/...Attention.py:58, and their autograd), exposed for testing and reuse:
 *   D[m*ldd + n] (fp32)  or  D_planes (hi/lo bf16, d_plane_stride apart)  =  sum_k A(m,k) B(n,k) (+ bias[n])
 * with split-plane operands. a_mn = 0: A(m,k) at m*lda + k; a_mn = 1: A(m,k) at k*lda + m (M % 64 == 0). Same for B
 * with ldb / N. Exactly one of D, D_planes is non-NULL. K is split in at most max_split partitions (1 for D_planes).
 * lda/ldb % 8 == 0, N % 32 == 0, 16 B aligned bases; GH_ERR_UNSUPPORTED otherwise. */
int gh_gemm_planes(const void* A_planes, long long lda, long long a_plane_stride, int a_mn, const void* B_planes,
                   long long ldb, long long b_plane_stride, int b_mn, const float* bias, float* D, void* D_planes,
                   long long ldd, long long d_plane_stride, int M, int N, int K, int max_split, void* stream);

/* Host-only: the tiling gh_gemm_planes / gh_attn_head_fwd2 / _bwd2 choose for one M x N x K problem on `npairs` CTA pairs
 * (tile width 256 or 128, number of K partitions <= max_split, resulting work units). No GPU needed. */
int gh_tgemm_plan(int M, int N, int K, int max_split, int npairs, int* tn, int* ksplit, int* units);

/* Host-only: the launch plan of the CTA-pair pooled Gram backward (gh_gram_pool_bwd on TMA-describable features) for one
 * stage shape, under the current gh_set_option state. out[0..7] = x-tile width NT, x tiles per image, 1 if the generated
 * gradient tile lives in tensor memory (the MMAs' A operand is read from TMEM) else 0, K chunks per ring stage (1 or 2),
 * A-ring stages, F-ring stages, TMEM columns in use (<= 512; 0 for the shared-memory form), ring bytes in shared memory
 * (<= 147 456). GH_ERR_UNSUPPORTED for shapes the pair kernels do not take (C % g, pooling factor < 8 or not a power of
 * two, g > 32). No GPU needed. */
int gh_gram_bwd_plan(int C, int HW, int g, int f_dtype, int channels_last, int* out);

/* Forward (Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:56-61 / :108-114). w_in_planes: planes of in_proj_weight (2, 3E, E); w_out_planes: planes of out_proj.weight (2, E, E) (dense,
 * plane_stride = rows*E). b_in, b_out, W_c, b_c fp32 as in gh_attn_head_fwd. Outputs: emb (B, E), logits (B, nc); saved
 * for backward: x_planes (2, B*L, E) bf16, qkv (B*L, 3E) fp32, probs (B, L, L) fp32, obar_planes (2, B, E) bf16.
 * Five launches: split X, in_proj GEMM, per-image scores/softmax/value mix, out_proj GEMM, classifier. Results are
 * bitwise reproducible (K is split in at most two partitions). GH_ERR_UNSUPPORTED outside the shape range above. */
int gh_attn_head_fwd2(const float* desc, const void* w_in_planes, const float* b_in, const void* w_out_planes,
                      const float* b_out, const float* W_c, const float* b_c, int B, int L, int E, int nc, void* x_planes,
                      float* qkv, float* probs, void* obar_planes, float* emb, float* logits, void* stream);

/* Bytes of `workspace` gh_attn_head_bwd2 needs (16 B aligned). */
long long gh_attn_head_bwd2_workspace(int B, int L, int E);

/* Backward of gh_attn_head_fwd2 (autograd of Models/...Attention.py:56-61, driven by loss.backward(),
 * functions/functions_RESNET50_Truncate_Gram_Attention.py:135). Outputs as in gh_attn_head_bwd (each may be NULL; overwritten, not accumulated).
 * Four launches: gradient prep (demb planes, db_out, dW_c, db_c), {dObar, dW_out} GEMMs, per-image softmax/score
 * backward (dQKV planes, db_in), {dW_in, d_desc} GEMMs. K partitions of a GEMM meet in fp32 reduce-adds whose order is
 * not fixed: gradients are reproducible to fp32 rounding, not bitwise. */
int gh_attn_head_bwd2(const void* x_planes, const void* w_in_planes, const void* w_out_planes, const float* W_c,
                      const float* qkv, const float* probs, const void* obar_planes, const float* emb,
                      const float* d_logits, const float* d_emb_ext, int B, int L, int E, int nc, float* d_desc,
                      float* dW_in, float* db_in, float* dW_out, float* db_out, float* dW_c, float* db_c, void* workspace,
                      void* stream);

/* ---- Baseline JPEG decoding for the loaders (csrc/jpeg.cuh; functions.gpu_resize_transform(decode="gpu")) ----
 * The output equals `np.asarray(Image.open(f).convert('RGB'))` byte for byte (Pillow + libjpeg-turbo: islow IDCT, fancy
 * upsampling). The worker parses each file (jpeg.py): `scan` holds every restart segment's entropy-coded bytes with
 * stuffing removed, back to back; `segs` one row per segment, `imgs` one row per image, `tables` GH_JPEG_TABLE_INTS
 * ints per image: quantisation tables per component (64 ints, natural order), then per component a DC and an AC
 * Huffman table of GH_JPEG_HUFF_INTS ints (a 9-bit lookahead of length << 8 | symbol, maxcode[17] and valoff[17] per
 * code length, the symbols packed four per int). */
enum { GH_JPEG_SEG_START, GH_JPEG_SEG_LEN, GH_JPEG_SEG_IMAGE, GH_JPEG_SEG_MCU, GH_JPEG_SEG_MCUS, GH_JPEG_SEG_COLS };
enum { GH_JPEG_H, GH_JPEG_W, GH_JPEG_NCOMP, GH_JPEG_H0, GH_JPEG_V0, GH_JPEG_MCUX, GH_JPEG_MCUY, GH_JPEG_COEF_OFF,
       GH_JPEG_BLOCKS, GH_JPEG_PLANE_OFF, GH_JPEG_ARENA_OFF, GH_JPEG_TABLE_OFF, GH_JPEG_BATCH_INDEX, GH_JPEG_IMG_COLS };
#define GH_JPEG_QUANT_INTS 192
#define GH_JPEG_HUFF_MAXCODE 512
#define GH_JPEG_HUFF_VALOFF 530
#define GH_JPEG_HUFF_VALS 547
#define GH_JPEG_HUFF_INTS 612
#define GH_JPEG_TABLE_INTS (GH_JPEG_QUANT_INTS + 6 * GH_JPEG_HUFF_INTS)
#define GH_JPEG_PHASE_HUFFMAN 1
#define GH_JPEG_PHASE_IDCT 2
#define GH_JPEG_PHASE_COLOR 4
/* A segment's length in bytes stays below this (bit positions inside a segment are 32-bit); the batch has no limit. */
#define GH_JPEG_MAX_SEGMENT_BYTES (1LL << 28)

/* Host-only: the ints per image of `tables` (GH_JPEG_TABLE_INTS). */
int gh_jpeg_table_ints(void);
/* Host-only: bytes of `records` gh_jpeg_decode needs for scan_bytes of scan data in n_segs segments cut into
 * subsequences of subseq_bytes; GH_ERR_BAD_ARG for a non-positive count or size. */
long long gh_jpeg_records_bytes(long long scan_bytes, int n_segs, int subseq_bytes);
/* Decodes n_imgs images. All pointers are DEVICE memory. `phases` (GH_JPEG_PHASE_*) selects the launches, so that each
 * can be timed alone: Huffman decoding (one CTA per segment, subsequences of subseq_bytes) into `coef` (int16, 64 per
 * block, zeroed by the caller), which also zeroes and then sets `status[i]` to nonzero for an image whose scan runs out
 * of bits, meets an invalid code or yields fewer blocks than its frame; the IDCT into `planes`; upsampling and colour
 * into `arena`. max_blocks / max_pixels: the largest block count / H * W of an image. The caller checks every range in
 * `segs` / `imgs` against the buffers, and every segment's length against GH_JPEG_MAX_SEGMENT_BYTES (the kernel sets the
 * image's status for a longer one). Arguments as gh_jpeg_check. */
/* Host-only: the argument check of gh_jpeg_decode (0, GH_ERR_BAD_ARG, or GH_ERR_UNSUPPORTED for n_imgs > 65535 or
 * grids beyond the launch limits). The total scan_bytes of a batch is not limited. */
int gh_jpeg_check(long long scan_bytes, int n_segs, int n_imgs, long long max_blocks, long long max_pixels,
                  int subseq_bytes, int phases);
int gh_jpeg_decode(const unsigned char* scan, long long scan_bytes, const long long* segs, int n_segs,
                   const long long* imgs, int n_imgs, const int* tables, long long max_blocks, long long max_pixels,
                   int subseq_bytes, short* coef, unsigned char* planes, int* records, int* status, unsigned char* arena,
                   int phases, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GRAMHEAD_H_ */
