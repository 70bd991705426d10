"""torch-facing wrappers (autograd.Function) over the C ABI in include/gramhead.h.

PyTorch is used for device memory, streams and autograd bookkeeping only; every FLOP of the head runs in
libgramhead.so. All functions require CUDA tensors and raise otherwise: there is no CPU / eager fallback.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import GH_DTYPE_BF16, GH_DTYPE_F32, GramHeadError, check

# Launch knobs (tests and bench sweep them; 0 = library default)
KSPLIT = 0
MAX_CTAS = 0

# Accounting used by bench.py: number of kernels of this library launched, and (when PROFILE is a list) one
# (name, work dict, start event, end event) record per C-ABI call, timed on the stream the call is enqueued on.
LAUNCHES = 0
PROFILE = None


class _Timed:
    def __init__(self, name, kernels, device, **work):
        self.name, self.kernels, self.device, self.work = name, kernels, device, work

    def __enter__(self):
        global LAUNCHES
        LAUNCHES += self.kernels
        if PROFILE is not None:
            self.start = torch.cuda.Event(enable_timing=True)
            self.end = torch.cuda.Event(enable_timing=True)
            self.start.record(torch.cuda.current_stream(self.device))
        return self

    def __exit__(self, *exc):
        if PROFILE is not None and exc[0] is None:
            self.end.record(torch.cuda.current_stream(self.device))
            PROFILE.append((self.name, self.work, self.start, self.end))
        return False


def _stream_ptr(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise GramHeadError(f"gramhead: {what} must be a CUDA tensor (got {t.device}); the head has no CPU path")


def _feature_view(x: torch.Tensor):
    """(B, C, H, W) or (B, C, HW) activation -> (tensor kept alive, dtype code, img / channel / position strides in
    elements, B, C, HW). Dense channels_last (NHWC) 4-D tensors are passed through with channel stride 1; anything
    else is brought to x-contiguous rows (what the reference's .view(b, ch, h*w) requires)."""
    _require_cuda(x, "features")
    if x.dim() == 4:
        b, c, h, w = x.shape
        hw = h * w
        if is_channels_last(x):
            return x, _dtype_code(x), x.stride(0), 1, c, b, c, hw
        if not (x.stride(3) == 1 and x.stride(2) == w):
            x = x.contiguous()
    elif x.dim() == 3:
        b, c, hw = x.shape
        if x.stride(2) != 1:
            x = x.contiguous()
    else:
        raise GramHeadError(f"gramhead: features must be (B,C,H,W) or (B,C,HW), got {tuple(x.shape)}")
    return x, _dtype_code(x), x.stride(0), x.stride(1), 1, b, c, hw


def _dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return GH_DTYPE_F32
    if t.dtype == torch.bfloat16:
        return GH_DTYPE_BF16
    raise GramHeadError(f"gramhead: features must be float32 or bfloat16, got {t.dtype}")


def is_channels_last(x: torch.Tensor) -> bool:
    """Dense NHWC storage of a (B, C, H, W) tensor with more than one channel and more than one position."""
    if x.dim() != 4:
        return False
    b, c, h, w = x.shape
    return (c > 1 and h * w > 1 and x.stride(1) == 1 and x.stride(3) == c and x.stride(2) == w * c
            and x.stride(0) == h * w * c)


def nhwc_to_nchw(x: torch.Tensor) -> torch.Tensor:
    """(B, C, HW)-shaped copy of a channels_last activation (same dtype): the C x HW matrices gram_matrix() views
    (reference Models/...:27-28), produced by the library's transpose kernel in one HBM-bound pass. Rows are padded to
    a multiple of 16 B (HW = 196 in bf16 -> pitch 200) so that every stage qualifies for the TMA-fed kernels."""
    _require_cuda(x, "features")
    b, c, h, w = x.shape
    hw = h * w
    per16 = 16 // x.element_size()                       # rows padded to 16 B: what a TMA tensor map can describe
    pitch = (hw + per16 - 1) // per16 * per16
    buf = torch.empty((b, c, pitch), dtype=x.dtype, device=x.device)
    code = _dtype_code(x)
    work = dict(bytes=2 * x.numel() * x.element_size(), flops=0, kind="transpose")
    with torch.cuda.device(x.device), _Timed(f"nhwc_to_nchw[C={c},HW={hw},{x.dtype}]", 1, x.device, **work):
        rc = _lib.lib().gh_transpose_cast(x.data_ptr(), code, buf.data_ptr(), code, b, hw, c, pitch, _stream_ptr(x))
    check(rc, "gh_transpose_cast")
    return buf[:, :, :hw] if pitch != hw else buf.view(b, c, h, w)


def grad_like_activation(df: torch.Tensor, shape, dtype, channels_last: bool) -> torch.Tensor:
    """(B, C, HW) gradient (fp32 or bf16) -> gradient tensor of the activation's shape and dtype; for a channels_last activation
    the transpose kernel writes it NHWC (and casts) directly, so the cuDNN backward gets the layout it runs in."""
    if not channels_last:
        return df.view(shape).to(dtype)
    b, c, h, w = shape
    out = torch.empty((b, c, h, w), dtype=dtype, device=df.device, memory_format=torch.channels_last)
    work = dict(bytes=df.numel() * (df.element_size() + out.element_size()), flops=0, kind="transpose")
    with torch.cuda.device(df.device), _Timed(f"nchw_to_nhwc[C={c},HW={h * w},{dtype}]", 1, df.device, **work):
        rc = _lib.lib().gh_transpose_cast(df.data_ptr(), _dtype_code(df), out.data_ptr(), _dtype_code(out), b, c, h * w, c,
                                          _stream_ptr(df))
    check(rc, "gh_transpose_cast")
    return out


def _layout_tag(s_x: int) -> str:
    return "" if s_x == 1 else ",nhwc"


def nhwc_native(x: torch.Tensor, g: int = 0) -> bool:
    """True when a channels_last activation can be consumed as it is by the CTA-pair kernels (forward AND backward):
    channels a multiple of one 128 B row, 16 B-aligned storage and, for the pooled path, the shapes the generated
    backward handles (k = C/g a power of two >= 8, g <= 32). Otherwise it goes through nhwc_to_nchw()."""
    if not is_channels_last(x):
        return False
    c = x.shape[1]
    per_row = 128 // x.element_size()
    if c % per_row or x.data_ptr() % 16 or x.dtype not in (torch.float32, torch.bfloat16):
        return False
    if g:
        k = c // g if c % g == 0 else 0
        return g <= 32 and k >= 8 and (k & (k - 1)) == 0 and k <= 128
    return True


def pooled_supported(c: int, g: int) -> bool:
    """True when the fused Gram+pool kernels apply (bins are disjoint k x k blocks, k a power of two in [8, 128])."""
    if g <= 0 or c % g:
        return False
    k = c // g
    return 8 <= k <= 128 and (k & (k - 1)) == 0


# ----------------------------------------------------------------------------------------------------------------------
# raw launches
# ----------------------------------------------------------------------------------------------------------------------
def gram_pool_fwd_(x: torch.Tensor, g: int, desc: torch.Tensor, l: int) -> None:
    """desc[:, l, :] = vec(pool_g(F F^T / HW)) for stage activation x. desc: (B, L, g*g) fp32 contiguous."""
    x, code, s_img, s_row, s_x, b, c, hw = _feature_view(x)
    assert desc.is_contiguous() and desc.dtype == torch.float32 and desc.shape[0] == b and desc.shape[2] == g * g
    work = dict(bytes=b * c * hw * x.element_size() + b * g * g * 4, flops=b * c * (c + 1) * hw, kind="gram_fwd")
    with torch.cuda.device(x.device), _Timed(f"gram_pool_fwd[C={c},HW={hw},{x.dtype}{_layout_tag(s_x)}]", 1, x.device, **work):
        rc = _lib.lib().gh_gram_pool_fwd(x.data_ptr(), code, s_img, s_row, s_x, b, c, hw, g, desc.data_ptr(), l,
                                         desc.shape[1], KSPLIT, MAX_CTAS, _stream_ptr(x))
    check(rc, "gh_gram_pool_fwd")


def gram_dense_fwd(x: torch.Tensor) -> torch.Tensor:
    x, code, s_img, s_row, s_x, b, c, hw = _feature_view(x)
    out = torch.empty((b, c, c), device=x.device, dtype=torch.float32)
    work = dict(bytes=b * c * hw * x.element_size() + b * c * c * 4, flops=b * c * (c + 1) * hw, kind="gram_fwd")
    with torch.cuda.device(x.device), _Timed(f"gram_dense_fwd[C={c},HW={hw},{x.dtype}{_layout_tag(s_x)}]", 1, x.device, **work):
        rc = _lib.lib().gh_gram_dense_fwd(x.data_ptr(), code, s_img, s_row, s_x, b, c, hw, out.data_ptr(), KSPLIT,
                                          MAX_CTAS, _stream_ptr(x))
    check(rc, "gh_gram_dense_fwd")
    return out


def _grad_buffer(x: torch.Tensor, s_x: int, b: int, c: int, hw: int, dtype=torch.float32):
    """dF in the layout of the features: (B, C, HW) rows, or channels_last like x. -> (tensor, img, row, x strides)"""
    if s_x == 1:
        return torch.empty((b, c, hw), device=x.device, dtype=dtype), c * hw, hw, 1
    df = torch.empty(x.shape, device=x.device, dtype=dtype, memory_format=torch.channels_last)
    return df, c * hw, 1, c


# bf16 activations (the opt-in bf16 backbone modes) get their gradient written as bf16 by the backward kernel itself --
# half the HBM bytes of the fp32 gradient and no separate cast pass -- whenever the CTA-pair kernels take the shape.
BF16_GRADIENTS = True


def _gram_bwd_call(entry, name, x, args_mid, work_extra):
    """Shared launch logic of the pooled / dense backward: try the bf16 gradient for bf16 features, fall back to fp32."""
    x, code, s_img, s_row, s_x, b, c, hw = _feature_view(x)
    want16 = BF16_GRADIENTS and x.dtype == torch.bfloat16
    for dtype in ((torch.bfloat16, torch.float32) if want16 else (torch.float32,)):
        df, d_img, d_row, d_x = _grad_buffer(x, s_x, b, c, hw, dtype)
        work = dict(bytes=b * c * hw * (x.element_size() + df.element_size()) + work_extra, flops=2 * b * c * c * hw,
                    kind="gram_bwd")
        tag = ",bf16out" if dtype == torch.bfloat16 else ""
        with torch.cuda.device(x.device), _Timed(f"{name}[C={c},HW={hw},{x.dtype}{_layout_tag(s_x)}{tag}]", 1, x.device, **work):
            rc = entry(x.data_ptr(), code, s_img, s_row, s_x, b, c, hw, *args_mid, df.data_ptr(), _dtype_code(df), d_img, d_row,
                       d_x, MAX_CTAS, _stream_ptr(x))
        if rc == _lib.GH_ERR_UNSUPPORTED and dtype == torch.bfloat16:
            global LAUNCHES                                   # nothing was launched: take the attempt out of the accounting
            LAUNCHES -= 1
            if PROFILE and PROFILE[-1][0].endswith("bf16out]"):
                PROFILE.pop()
            continue
        return rc, df
    return rc, df


def gram_pool_bwd(x: torch.Tensor, g: int, d_desc: torch.Tensor, l: int) -> torch.Tensor:
    """-> dF, (B, C, HW) for x-contiguous features, channels_last (B, C, H, W) for channels_last features; fp32, or bf16
    for bf16 features on the CTA-pair kernels (BF16_GRADIENTS)."""
    d_desc = d_desc.contiguous()
    b = d_desc.shape[0]
    rc, df = _gram_bwd_call(_lib.lib().gh_gram_pool_bwd, "gram_pool_bwd", x, (g, d_desc.data_ptr(), l, d_desc.shape[1]),
                            b * g * g * 4)
    check(rc, "gh_gram_pool_bwd")
    return df


def gram_dense_bwd(x: torch.Tensor, d_gram: torch.Tensor) -> torch.Tensor:
    """-> dF = (dG + dG^T) F / HW, in the layout gram_pool_bwd returns.

    The backward kernels take C % 16 == 0 only (gh_gram_dense_bwd refuses other C). For other C (e.g. 3, 17, 100) F's
    channels and dG's rows and columns are zero-padded to the next multiple of 16 here, and the first C channels of the
    padded gradient are returned: padded channels add exact zeros to every sum of (dG + dG^T) F, so the result is the
    unpadded one. This costs a copy of F and dG; the ResNet stages (C a multiple of 64) never take it. The pooled backward
    is not padded (extra channels would move the pooling bins): style_descriptor sends such stages here through
    adaptive_pool_bwd."""
    d_gram = d_gram.contiguous().float()
    c = x.shape[1]
    if c % 16:
        b, cp = x.shape[0], (c + 15) // 16 * 16
        xp = torch.zeros((b, cp, x[0, 0].numel()), device=x.device, dtype=x.dtype)
        xp[:, :c] = x.reshape(b, c, -1)
        dgp = torch.zeros((b, cp, cp), device=d_gram.device, dtype=torch.float32)
        dgp[:, :c, :c] = d_gram
        df = gram_dense_bwd(xp, dgp)[:, :c]
        if x.dim() == 4 and is_channels_last(x):       # the layout _grad_buffer gives channels_last features
            return df.reshape(x.shape).contiguous(memory_format=torch.channels_last)
        return df.contiguous()
    rc, df = _gram_bwd_call(_lib.lib().gh_gram_dense_bwd, "gram_dense_bwd", x, (d_gram.data_ptr(),), d_gram.numel() * 4)
    check(rc, "gh_gram_dense_bwd")
    return df


def adaptive_pool_fwd_(gram: torch.Tensor, g: int, desc: torch.Tensor, l: int) -> None:
    b, c, _ = gram.shape
    with torch.cuda.device(gram.device), _Timed("adaptive_pool_fwd", 1, gram.device, bytes=b * c * c * 4, flops=0, kind="pool"):
        rc = _lib.lib().gh_adaptive_pool_fwd(gram.data_ptr(), b, c, g, desc.data_ptr(), l, desc.shape[1],
                                             _stream_ptr(gram))
    check(rc, "gh_adaptive_pool_fwd")


def adaptive_pool_bwd(d_desc: torch.Tensor, l: int, c: int, g: int) -> torch.Tensor:
    d_desc = d_desc.contiguous()
    b = d_desc.shape[0]
    dg = torch.empty((b, c, c), device=d_desc.device, dtype=torch.float32)
    with torch.cuda.device(d_desc.device), _Timed("adaptive_pool_bwd", 1, d_desc.device, bytes=b * c * c * 4, flops=0, kind="pool"):
        rc = _lib.lib().gh_adaptive_pool_bwd(d_desc.data_ptr(), l, d_desc.shape[1], b, c, g, dg.data_ptr(),
                                             _stream_ptr(d_desc))
    check(rc, "gh_adaptive_pool_bwd")
    return dg


def gemm_f32(a: torch.Tensor, b: torch.Tensor, bias: torch.Tensor = None) -> torch.Tensor:
    """a (M, K) @ b (K, N) (+ bias) for arbitrarily strided fp32 CUDA views (e.g. w.t()), through gh_gemm_f32."""
    _require_cuda(a, "a")
    m, k = a.shape
    k2, n = b.shape
    assert k == k2 and a.dtype == torch.float32 and b.dtype == torch.float32
    out = torch.empty((m, n), device=a.device, dtype=torch.float32)
    work = dict(bytes=(m * k + k * n + m * n) * 4, flops=2 * m * n * k, kind="gemm")
    with torch.cuda.device(a.device), _Timed(f"gemm_f32[M={m},N={n},K={k}]", 1, a.device, **work):
        rc = _lib.lib().gh_gemm_f32(a.data_ptr(), a.stride(0), a.stride(1), b.data_ptr(), b.stride(0), b.stride(1),
                                    0 if bias is None else bias.data_ptr(), out.data_ptr(), n, m, n, k, _stream_ptr(a))
    check(rc, "gh_gemm_f32")
    return out


def maxpool2d_nhwc(x: torch.Tensor, kernel: int, stride: int, padding: int) -> torch.Tensor:
    """nn.MaxPool2d(kernel, stride, padding) (floor mode, dilation 1) of a channels_last (B, C, H, W) fp32 / bf16
    activation, values only (gh_maxpool2d_nhwc); the result is channels_last again."""
    _require_cuda(x, "x")
    if x.dim() != 4 or not x.is_contiguous(memory_format=torch.channels_last):
        raise GramHeadError("gramhead: maxpool2d_nhwc takes a channels_last (B, C, H, W) tensor")
    b, c, h, w = x.shape
    oh, ow = (h + 2 * padding - kernel) // stride + 1, (w + 2 * padding - kernel) // stride + 1
    out = torch.empty((b, c, oh, ow), device=x.device, dtype=x.dtype, memory_format=torch.channels_last)
    work = dict(bytes=(x.numel() + out.numel()) * x.element_size(), flops=0, kind="maxpool")
    with torch.cuda.device(x.device), _Timed(f"maxpool2d_nhwc[C={c},HW={h}x{w},{x.dtype}]", 1, x.device, **work):
        rc = _lib.lib().gh_maxpool2d_nhwc(x.data_ptr(), _dtype_code(x), out.data_ptr(), b, h, w, c, kernel, stride, padding,
                                          _stream_ptr(x))
    check(rc, "gh_maxpool2d_nhwc")
    return out


def stem_space_to_depth(x: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """(B, 3, H, W) fp32 images (any strides) -> channels_last (B, 16, H/2 + 3, W/2 + 3) in `dtype`: the zero-bordered
    2x2 space-to-depth image over which the stem's 7x7 stride-2 convolution is a 4x4 stride-1 one (gh_stem_space_to_depth)."""
    _require_cuda(x, "x")
    if x.dim() != 4 or x.shape[1] != 3 or x.dtype != torch.float32 or x.shape[2] % 2 or x.shape[3] % 2:
        raise GramHeadError("gramhead: stem_space_to_depth takes fp32 (B, 3, H, W) images with even H and W")
    b, _, h, w = x.shape
    z = torch.empty((b, 16, h // 2 + 3, w // 2 + 3), device=x.device, dtype=dtype, memory_format=torch.channels_last)
    work = dict(bytes=x.numel() * 4 + z.numel() * z.element_size(), flops=0, kind="stem_s2d")
    with torch.cuda.device(x.device), _Timed(f"stem_space_to_depth[HW={h}x{w},{dtype}]", 1, x.device, **work):
        rc = _lib.lib().gh_stem_space_to_depth(x.data_ptr(), x.stride(0), x.stride(1), x.stride(2), x.stride(3), b, h, w,
                                               z.data_ptr(), _dtype_code(z), _stream_ptr(x))
    check(rc, "gh_stem_space_to_depth")
    return z


def stem_conv_pool(x: torch.Tensor, packed_weight: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """(B, 3, H, W) fp32 images (any strides, H and W even) -> channels_last (B, 64, PH, PW) fp32:
    maxpool3x3/s2/p1(relu(conv7x7/s2/p3(x) + bias)) in one kernel with tf32 operands (gh_stem_conv_pool_nhwc).
    packed_weight: frozen_encoder.pack_stem_weight() of the folded weights; bias: the folded (64,) bias."""
    _require_cuda(x, "x")
    if x.dim() != 4 or x.shape[1] != 3 or x.dtype != torch.float32 or x.shape[2] % 2 or x.shape[3] % 2:
        raise GramHeadError("gramhead: stem_conv_pool takes fp32 (B, 3, H, W) images with even H and W")
    if (packed_weight.dtype != torch.float32 or packed_weight.numel() != 16384 or not packed_weight.is_contiguous()
            or bias.dtype != torch.float32 or bias.numel() != 64 or not bias.is_contiguous()
            or packed_weight.device != x.device or bias.device != x.device):
        raise GramHeadError("gramhead: stem_conv_pool takes the packed fp32 stem weights (16384) and bias (64) on x's device")
    b, _, h, w = x.shape
    oh, ow = h // 2, w // 2
    ph, pw = (oh - 1) // 2 + 1, (ow - 1) // 2 + 1
    out = torch.empty((b, 64, ph, pw), device=x.device, dtype=torch.float32, memory_format=torch.channels_last)
    work = dict(bytes=(x.numel() + out.numel()) * 4, flops=2 * b * oh * ow * 64 * 147, kind="stem_conv_pool")
    with torch.cuda.device(x.device), _Timed(f"stem_conv_pool[HW={h}x{w}]", 1, x.device, **work):
        rc = _lib.lib().gh_stem_conv_pool_nhwc(x.data_ptr(), x.stride(0), x.stride(1), x.stride(2), x.stride(3), b, h, w,
                                               packed_weight.data_ptr(), bias.data_ptr(), out.data_ptr(), _stream_ptr(x))
    check(rc, "gh_stem_conv_pool_nhwc")
    return out


def stem_conv_pool_u8(x: torch.Tensor, mean, std, packed_weight: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """stem_conv_pool(normalize_u8(x, mean, std), packed_weight, bias) bit for bit, in one kernel that reads the (B, 3, H, W)
    uint8 pixels (any strides, H and W even) and never builds the fp32 batch (gh_stem_conv_pool_u8_nhwc)."""
    _require_cuda(x, "x")
    if x.dim() != 4 or x.shape[1] != 3 or x.dtype != torch.uint8 or x.shape[2] % 2 or x.shape[3] % 2:
        raise GramHeadError("gramhead: stem_conv_pool_u8 takes uint8 (B, 3, H, W) images with even H and W")
    if (packed_weight.dtype != torch.float32 or packed_weight.numel() != 16384 or not packed_weight.is_contiguous()
            or bias.dtype != torch.float32 or bias.numel() != 64 or not bias.is_contiguous()
            or packed_weight.device != x.device or bias.device != x.device):
        raise GramHeadError("gramhead: stem_conv_pool_u8 takes the packed fp32 stem weights (16384) and bias (64) on x's device")
    mean, std = [float(v) for v in mean], [float(v) for v in std]
    if len(mean) != 3 or len(std) != 3:
        raise GramHeadError("gramhead: stem_conv_pool_u8: 3 channels need 3 means and stds")
    b, _, h, w = x.shape
    oh, ow = h // 2, w // 2
    ph, pw = (oh - 1) // 2 + 1, (ow - 1) // 2 + 1
    out = torch.empty((b, 64, ph, pw), device=x.device, dtype=torch.float32, memory_format=torch.channels_last)
    fl = ctypes.c_float * 3
    work = dict(bytes=x.numel() + out.numel() * 4, flops=2 * b * oh * ow * 64 * 147, kind="stem_conv_pool")
    with torch.cuda.device(x.device), _Timed(f"stem_conv_pool_u8[HW={h}x{w}]", 1, x.device, **work):
        rc = _lib.lib().gh_stem_conv_pool_u8_nhwc(x.data_ptr(), x.stride(0), x.stride(1), x.stride(2), x.stride(3), b, h,
                                                  w, fl(*mean), fl(*std), packed_weight.data_ptr(), bias.data_ptr(),
                                                  out.data_ptr(), _stream_ptr(x))
    check(rc, "gh_stem_conv_pool_u8_nhwc")
    return out


def normalize_u8_host(t: torch.Tensor, mean, std) -> torch.Tensor:
    """ToTensor's scaling + Normalize for a uint8 batch that stays on the host (CPU runs): the same op sequence
    torchvision executes per image (to float32, div 255, sub mean, div std)."""
    shape = (1, -1, 1, 1)
    out = t.to(torch.float32).div_(255)
    return out.sub_(torch.tensor(mean, dtype=torch.float32).view(shape)).div_(torch.tensor(std, dtype=torch.float32).view(shape))


def normalize_u8(x: torch.Tensor, mean, std, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(B, C, H, W) uint8 pixels on the device -> the fp32 batch transforms.ToTensor() + transforms.Normalize(mean, std)
    produce on the host (reference test_RESNET50_Truncate_gram_attention.py:64-65), bit for bit (gh_normalize_u8).
    `out`: optional dense fp32 buffer of at least B images to write into (its first B images are returned)."""
    _require_cuda(x, "x")
    if x.dim() != 4 or x.dtype != torch.uint8 or not 1 <= x.shape[1] <= 4:
        raise GramHeadError("gramhead: normalize_u8 takes a (B, C <= 4, H, W) uint8 batch")
    mean, std = [float(v) for v in mean], [float(v) for v in std]
    b, c, h, w = x.shape
    if len(mean) != c or len(std) != c:
        raise GramHeadError(f"gramhead: normalize_u8: {c} channels need {c} means and stds")
    x = x.contiguous()
    if out is None:
        out = torch.empty((b, c, h, w), device=x.device, dtype=torch.float32)
    else:
        if (out.dtype != torch.float32 or out.device != x.device or out.dim() != 4 or out.shape[0] < b
                or out.shape[1:] != x.shape[1:] or not out.is_contiguous()):
            raise GramHeadError("gramhead: normalize_u8: `out` must be a dense fp32 (>= B, C, H, W) tensor on x's device")
        out = out[:b]
    if b == 0:
        return out
    fl = ctypes.c_float * c
    work = dict(bytes=x.numel() * 5, flops=0, kind="normalize_u8")
    with torch.cuda.device(x.device), _Timed(f"normalize_u8[C={c},HW={h}x{w}]", 1, x.device, **work):
        rc = _lib.lib().gh_normalize_u8(x.data_ptr(), out.data_ptr(), b, c, h * w, fl(*mean), fl(*std), _stream_ptr(x))
    check(rc, "gh_normalize_u8")
    return out


def patch_gram(maps: Sequence[torch.Tensor], ln_input: bool = True):
    """The L collected (B, D, H_l, W_l) fp32 maps of one Multi-PatchGAN discriminator -> (gram (L, B, D*D),
    gram_norm (L, B)) through gh_patch_gram_fwd: [layer norm over the map,] 4x4 adaptive average pooling, layer norm,
    Gram over the 16 positions / (16 + 1e-6), Frobenius norm (Models_Multi_PatchGAN.py:198, :210-223)."""
    import ctypes
    L = len(maps)
    if L == 0:
        raise GramHeadError("gramhead: patch_gram needs at least one feature map")
    for m in maps:
        _require_cuda(m, "feature map")
        if m.dtype != torch.float32 or m.dim() != 4 or m.shape[:2] != maps[0].shape[:2] or m.device != maps[0].device:
            raise GramHeadError("gramhead: patch_gram takes fp32 (B, D, H, W) maps with one B, D and device")
    b, d = maps[0].shape[:2]
    dev = maps[0].device
    gram = torch.empty((L, b, d * d), device=dev, dtype=torch.float32)
    norm = torch.empty((L, b), device=dev, dtype=torch.float32)
    scratch = torch.empty((_lib.lib().gh_patch_gram_workspace(L, b, d) + 1) // 2, device=dev, dtype=torch.float64)
    ptrs = (ctypes.c_void_p * L)(*[m.data_ptr() for m in maps])
    hs = (ctypes.c_int * L)(*[m.shape[2] for m in maps])
    ws = (ctypes.c_int * L)(*[m.shape[3] for m in maps])
    st = (ctypes.c_longlong * (4 * L))(*[v for m in maps for v in m.stride()])
    work = dict(bytes=sum(m.numel() for m in maps) * 4 + gram.numel() * 4, flops=2 * L * b * d * d * 16, kind="patch_gram")
    with torch.cuda.device(dev), _Timed(f"patch_gram[L={L},D={d},HW0={maps[0].shape[2]}x{maps[0].shape[3]}]", 2, dev, **work):
        rc = _lib.lib().gh_patch_gram_fwd(ptrs, hs, ws, st, L, b, d, 1 if ln_input else 0, gram.data_ptr(),
                                          norm.data_ptr(), scratch.data_ptr(), _stream_ptr(maps[0]))
    check(rc, "gh_patch_gram_fwd")
    return gram, norm


def patch_attention(feat: torch.Tensor, attn1: torch.nn.MultiheadAttention, attn2: torch.nn.MultiheadAttention,
                    classifier: torch.nn.Linear):
    """feat (L, B, E) -> (embeddings (B, E), output (B, nc)): the two multi-head attentions over the layer tokens, the
    mean over layers and the classifier (Models_Multi_PatchGAN.py:243-256) in one launch (gh_patch_attn_fwd)."""
    _require_cuda(feat, "feat")
    L, b, e = feat.shape
    feat = feat.contiguous()
    nc = classifier.out_features
    emb = torch.empty((b, e), device=feat.device, dtype=torch.float32)
    out = torch.empty((b, nc), device=feat.device, dtype=torch.float32)
    tensors = []
    for a in (attn1, attn2):
        if a.in_proj_weight is None or a.in_proj_bias is None or a.embed_dim != e or a.num_heads != attn1.num_heads:
            raise GramHeadError("gramhead: patch_attention needs packed in_proj weights with biases and one embed_dim")
        tensors += [a.in_proj_weight, a.in_proj_bias, a.out_proj.weight, a.out_proj.bias]
    tensors += [classifier.weight, classifier.bias]
    tensors = [t.detach().contiguous() for t in tensors]
    for t in tensors:
        _require_cuda(t, "head parameter")
    work = dict(bytes=(feat.numel() + emb.numel() + out.numel() + sum(t.numel() for t in tensors)) * 4,
                flops=2 * b * L * (2 * 4 * e * e) + 2 * b * e * nc, kind="patch_attention")
    with torch.cuda.device(feat.device), _Timed(f"patch_attention[L={L},E={e}]", 1, feat.device, **work):
        rc = _lib.lib().gh_patch_attn_fwd(feat.data_ptr(), *[t.data_ptr() for t in tensors], L, b, e, attn1.num_heads, nc,
                                          emb.data_ptr(), out.data_ptr(), _stream_ptr(feat))
    check(rc, "gh_patch_attn_fwd")
    return emb, out


# ----------------------------------------------------------------------------------------------------------------------
# autograd
# ----------------------------------------------------------------------------------------------------------------------
class _GramDense(torch.autograd.Function):
    """model.gram_matrix(x): (B, C, H, W) -> (B, C, C)."""

    @staticmethod
    def forward(ctx, x):
        ctx.meta = (tuple(x.shape), x.dtype, is_channels_last(x) and not nhwc_native(x))
        if ctx.meta[2]:
            x = nhwc_to_nchw(x)
        ctx.save_for_backward(x)
        return gram_dense_fwd(x)

    @staticmethod
    def backward(ctx, d_gram):
        (x,) = ctx.saved_tensors
        df = gram_dense_bwd(x, d_gram)
        if df.dim() == 4:                       # channels_last features consumed natively: dF is already NHWC
            return df.to(ctx.meta[1])
        return grad_like_activation(df, *ctx.meta)


def gram_matrix(x: torch.Tensor) -> torch.Tensor:
    return _GramDense.apply(x)


class _GramMSE(torch.autograd.Function):
    """mse_loss(gram_matrix(x), target) as one differentiable op (style transfer, reference functions/...:286-301):
    dense Gram forward, one fused pass for the loss and d loss / d G (gh_gram_mse), dense Gram backward."""

    @staticmethod
    def forward(ctx, x, target):
        ctx.meta = (tuple(x.shape), x.dtype, is_channels_last(x) and not nhwc_native(x))
        if ctx.meta[2]:
            x = nhwc_to_nchw(x)
        gram = gram_dense_fwd(x)
        target = target.detach().contiguous().float()
        if target.shape != gram.shape:
            raise GramHeadError(f"gramhead: target Gram {tuple(target.shape)} does not match {tuple(gram.shape)}")
        n = gram.numel()
        lib = _lib.lib()
        d_gram = torch.empty_like(gram)
        partial = torch.empty((lib.gh_gram_mse_blocks(n),), device=gram.device, dtype=torch.float32)
        with torch.cuda.device(x.device), _Timed(f"gram_mse[n={n}]", 1, x.device, bytes=3 * n * 4, flops=3 * n, kind="style"):
            rc = lib.gh_gram_mse(gram.data_ptr(), target.data_ptr(), n, d_gram.data_ptr(), partial.data_ptr(), _stream_ptr(x))
        check(rc, "gh_gram_mse")
        ctx.save_for_backward(x, d_gram)
        return partial.sum()

    @staticmethod
    def backward(ctx, grad_out):
        x, d_gram = ctx.saved_tensors
        df = gram_dense_bwd(x, d_gram * grad_out)            # grad_out is 1 in the style-transfer loop (loss.backward())
        if df.dim() == 4:
            return df.to(ctx.meta[1]), None
        return grad_like_activation(df, *ctx.meta), None


def gram_mse_loss(x: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """mean((gram_matrix(x) - target)^2): x (B, C, H, W) activations, target (B, C, C)."""
    return _GramMSE.apply(x, target)


class _GramMSEPerImage(torch.autograd.Function):
    """[mse_loss(gram_matrix(x[b]), target[b]) for b] as one differentiable op: dense Gram forward, one pass for the B
    losses and d (sum_b loss_b) / d G (gh_gram_mse_images), dense Gram backward. Image b's dG is the one a batch-1
    gram_mse_loss computes for it, so several style-transfer images step together with their own gradients."""

    @staticmethod
    def forward(ctx, x, target):
        ctx.meta = (tuple(x.shape), x.dtype, is_channels_last(x) and not nhwc_native(x))
        if ctx.meta[2]:
            x = nhwc_to_nchw(x)
        gram = gram_dense_fwd(x)
        target = target.detach().contiguous().float()
        if target.shape != gram.shape:
            raise GramHeadError(f"gramhead: target Gram {tuple(target.shape)} does not match {tuple(gram.shape)}")
        b, c, _ = gram.shape
        n = c * c
        lib = _lib.lib()
        k = lib.gh_gram_mse_images_blocks(n)
        d_gram = torch.empty_like(gram)
        partial = torch.empty((b, k), device=gram.device, dtype=torch.float32)
        with torch.cuda.device(x.device), _Timed(f"gram_mse_images[B={b},n={n}]", 1, x.device, bytes=3 * b * n * 4,
                                                 flops=3 * b * n, kind="style"):
            rc = lib.gh_gram_mse_images(gram.data_ptr(), target.data_ptr(), b, n, d_gram.data_ptr(), partial.data_ptr(),
                                        _stream_ptr(x))
        check(rc, "gh_gram_mse_images")
        ctx.save_for_backward(x, d_gram)
        return partial.sum(1)

    @staticmethod
    def backward(ctx, grad_out):
        x, d_gram = ctx.saved_tensors
        df = gram_dense_bwd(x, d_gram * grad_out.view(-1, 1, 1))   # all ones under losses.sum().backward()
        if df.dim() == 4:
            return df.to(ctx.meta[1]), None
        return grad_like_activation(df, *ctx.meta), None


def gram_mse_loss_per_image(x: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """(B,) losses mean((gram_matrix(x)[b] - target[b])^2): x (B, C, H, W) activations, target (B, C, C)."""
    return _GramMSEPerImage.apply(x, target)


class _StyleDescriptor(torch.autograd.Function):
    """L stage activations -> (B, L, g*g) pooled-Gram descriptors (the attention's input, batch-major)."""

    @staticmethod
    def forward(ctx, g, *stages):
        b = stages[0].shape[0]
        L = len(stages)
        desc = torch.empty((b, L, g * g), device=stages[0].device, dtype=torch.float32)
        # channels_last (NHWC) activations are consumed as they are by the CTA-pair kernels (MN-major operand tiles) when
        # nhwc_native() holds; otherwise one transpose pass gives the C x HW matrices the other kernels need, and that
        # NCHW copy is the tensor saved for backward (the backbone keeps the original alive anyway)
        ctx.meta = [(tuple(x.shape), x.dtype, is_channels_last(x) and not nhwc_native(x, g)) for x in stages]
        stages = [nhwc_to_nchw(x) if m[2] else x for x, m in zip(stages, ctx.meta)]
        for l, x in enumerate(stages):
            if pooled_supported(x.shape[1], g):
                gram_pool_fwd_(x, g, desc, l)
            else:   # torch's general (overlapping) bins: dense Gram, then the bin-rule pooling kernel
                adaptive_pool_fwd_(gram_dense_fwd(x), g, desc, l)
        ctx.g = g
        ctx.save_for_backward(*stages)
        return desc

    @staticmethod
    def backward(ctx, d_desc):
        g = ctx.g
        d_desc = d_desc.contiguous().float()
        grads: List[object] = [None]
        for l, x in enumerate(ctx.saved_tensors):
            if not ctx.needs_input_grad[l + 1]:
                grads.append(None)
                continue
            c = x.shape[1]
            if pooled_supported(c, g) and g <= 64 and c % 16 == 0:
                df = gram_pool_bwd(x, g, d_desc, l)
            else:
                df = gram_dense_bwd(x, adaptive_pool_bwd(d_desc, l, c, g))
            if df.dim() == 4:                   # channels_last features consumed natively: dF is already NHWC
                grads.append(df.to(ctx.meta[l][1]))
            else:
                grads.append(grad_like_activation(df, *ctx.meta[l]))
        return tuple(grads)


def style_descriptor(stages: Sequence[torch.Tensor], g: int) -> torch.Tensor:
    return _StyleDescriptor.apply(g, *stages)


# Which kernels run the attention head: "tma" = TMA-fed split-bf16 GEMMs on CTA pairs (gh_attn_head_fwd2 / _bwd2) when
# the shape allows it (E % 64 == 0, E <= 1024, L <= 8, nc <= 16), "ldg" = always the ld.global-fed kernels.
ATTN_IMPL = "tma"


def attn2_supported(L: int, e: int, nc: int) -> bool:
    return ATTN_IMPL == "tma" and e % 64 == 0 and 64 <= e <= 1024 and 1 <= L <= 8 and 1 <= nc <= 16


def split_bf16(x: torch.Tensor) -> torch.Tensor:
    """fp32 tensor -> (2, *x.shape) bf16 planes: hi = bf16(x), lo = bf16(x - hi) (gh_split_bf16)."""
    _require_cuda(x, "x")
    x = x.detach().contiguous().float()
    n = x.numel()
    planes = torch.empty((2,) + tuple(x.shape), device=x.device, dtype=torch.bfloat16)
    with torch.cuda.device(x.device), _Timed(f"split_bf16[n={n}]", 1, x.device, bytes=n * 8, flops=0, kind="split"):
        rc = _lib.lib().gh_split_bf16(x.data_ptr(), planes.data_ptr(), n, n, _stream_ptr(x))
    check(rc, "gh_split_bf16")
    return planes


# Split planes of the attention weights, cached per parameter object FOR INFERENCE ONLY.
# Invalidation cannot rest on tensor version counters alone: fused optimizers (torch.optim.AdamW(fused=True), the default
# of bench.py's training leg) update parameters without bumping `_version`. So:
#   * a forward that may be followed by an update -- autograd enabled and the weight requires grad -- or that is being
#     captured in a CUDA graph always splits afresh and evicts the weight's cache entry;
#   * the modules clear the cache on every train() / eval() switch (modules.py);
#   * otherwise an entry is valid while the parameter object, its storage address and its version counter are unchanged
#     (load_state_dict, .to(), in-place edits, non-fused optimizers). Edits through `.data` bypass all of this: call
#     clear_weight_planes() after them.
_WEIGHT_PLANES = {}


def clear_weight_planes() -> None:
    _WEIGHT_PLANES.clear()


def weight_planes(w: torch.Tensor) -> torch.Tensor:
    import weakref
    key = id(w)
    if torch.cuda.is_current_stream_capturing() or (torch.is_grad_enabled() and w.requires_grad):
        _WEIGHT_PLANES.pop(key, None)
        return split_bf16(w)
    hit = _WEIGHT_PLANES.get(key)
    if hit is not None:
        ref, version, ptr, planes = hit
        if ref() is w and version == w._version and ptr == w.data_ptr() and planes.device == w.device:
            return planes
    if len(_WEIGHT_PLANES) > 64:                       # parameters of models that no longer exist
        for k in [k for k, v in _WEIGHT_PLANES.items() if v[0]() is None]:
            del _WEIGHT_PLANES[k]
    planes = split_bf16(w)
    _WEIGHT_PLANES[key] = (weakref.ref(w), w._version, w.data_ptr(), planes)
    return planes


class _AttnHead(torch.autograd.Function):
    """(B, L, E) descriptors + the six head parameters -> (embeddings (B, E), logits (B, nc)); ld.global-fed kernels."""

    @staticmethod
    def forward(ctx, desc, w_in, b_in, w_out, b_out, w_c, b_c):
        _require_cuda(desc, "descriptors")
        desc = desc.contiguous().float()
        ps = [t.contiguous().float() for t in (w_in, b_in, w_out, b_out, w_c, b_c)]
        b, L, e = desc.shape
        nc = ps[4].shape[0]
        dev = desc.device
        qkv = torch.empty((b * L, 3 * e), device=dev, dtype=torch.float32)
        probs = torch.empty((b, L, L), device=dev, dtype=torch.float32)
        obar = torch.empty((b, e), device=dev, dtype=torch.float32)
        emb = torch.empty((b, e), device=dev, dtype=torch.float32)
        logits = torch.empty((b, nc), device=dev, dtype=torch.float32)
        work = dict(bytes=(3 * e * e + e * e + nc * e) * 4 + b * L * e * 4 * 5, kind="attn",
                    flops=2 * b * L * e * 3 * e + 2 * b * e * e + 2 * b * e * nc + 4 * b * L * L * e)
        with torch.cuda.device(dev), _Timed(f"attn_head_fwd[B={b},L={L},E={e},ldg]", 4, dev, **work):
            rc = _lib.lib().gh_attn_head_fwd(desc.data_ptr(), *[p.data_ptr() for p in ps], b, L, e, nc, qkv.data_ptr(),
                                             probs.data_ptr(), obar.data_ptr(), emb.data_ptr(), logits.data_ptr(),
                                             _stream_ptr(desc))
        check(rc, "gh_attn_head_fwd")
        ctx.save_for_backward(desc, ps[0], ps[2], ps[4], qkv, probs, obar, emb)
        ctx.dims = (b, L, e, nc)
        return emb, logits

    @staticmethod
    def backward(ctx, d_emb, d_logits):
        desc, w_in, w_out, w_c, qkv, probs, obar, emb = ctx.saved_tensors
        b, L, e, nc = ctx.dims
        dev = desc.device
        need = ctx.needs_input_grad
        d_logits = (torch.zeros((b, nc), device=dev) if d_logits is None else d_logits).contiguous().float()
        d_emb = None if d_emb is None else d_emb.contiguous().float()

        def buf(flag, shape):
            return torch.empty(shape, device=dev, dtype=torch.float32) if flag else None

        d_desc = buf(need[0], (b, L, e))
        gw_in, gb_in = buf(need[1], (3 * e, e)), buf(need[2], (3 * e,))
        gw_out, gb_out = buf(need[3], (e, e)), buf(need[4], (e,))
        gw_c, gb_c = buf(need[5], (nc, e)), buf(need[6], (nc,))
        lib = _lib.lib()
        ws = torch.empty((lib.gh_attn_head_bwd_workspace(b, L, e),), device=dev, dtype=torch.float32)
        ptr = lambda t: 0 if t is None else t.data_ptr()
        work = dict(bytes=(3 * e * e + e * e + nc * e) * 4 * 2 + b * L * e * 4 * 8, kind="attn",
                    flops=2 * (2 * b * L * e * 3 * e + 2 * b * e * e + 2 * b * e * nc) + 8 * b * L * L * e)
        with torch.cuda.device(dev), _Timed(f"attn_head_bwd[B={b},L={L},E={e},ldg]", 10, dev, **work):
            rc = lib.gh_attn_head_bwd(desc.data_ptr(), w_in.data_ptr(), w_out.data_ptr(), w_c.data_ptr(), qkv.data_ptr(),
                                      probs.data_ptr(), obar.data_ptr(), emb.data_ptr(), d_logits.data_ptr(), ptr(d_emb),
                                      b, L, e, nc, ptr(d_desc), ptr(gw_in), ptr(gb_in), ptr(gw_out), ptr(gb_out),
                                      ptr(gw_c), ptr(gb_c), ws.data_ptr(), _stream_ptr(desc))
        check(rc, "gh_attn_head_bwd")
        return d_desc, gw_in, gb_in, gw_out, gb_out, gw_c, gb_c


class _AttnHead2(torch.autograd.Function):
    """Same function on the TMA-fed GEMMs (gh_attn_head_fwd2 / gh_attn_head_bwd2). w_in_planes / w_out_planes are the
    cached split planes of in_proj_weight / out_proj.weight (weight_planes())."""

    @staticmethod
    def forward(ctx, desc, w_in, b_in, w_out, b_out, w_c, b_c, w_in_planes, w_out_planes):
        _require_cuda(desc, "descriptors")
        desc = desc.contiguous().float()
        b_in_, b_out_, w_c_, b_c_ = [t.contiguous().float() for t in (b_in, b_out, w_c, b_c)]
        b, L, e = desc.shape
        nc = w_c_.shape[0]
        dev = desc.device
        f32 = dict(device=dev, dtype=torch.float32)
        x_planes = torch.empty((2, b * L, e), device=dev, dtype=torch.bfloat16)
        obar_planes = torch.empty((2, b, e), device=dev, dtype=torch.bfloat16)
        qkv = torch.empty((b * L, 3 * e), **f32)
        probs = torch.empty((b, L, L), **f32)
        emb = torch.empty((b, e), **f32)
        logits = torch.empty((b, nc), **f32)
        work = dict(bytes=(3 * e * e + e * e + nc * e) * 4 + b * L * e * 4 * 5, kind="attn",
                    flops=2 * b * L * e * 3 * e + 2 * b * e * e + 2 * b * e * nc + 4 * b * L * L * e)
        with torch.cuda.device(dev), _Timed(f"attn_head_fwd[B={b},L={L},E={e}]", 5, dev, **work):
            rc = _lib.lib().gh_attn_head_fwd2(desc.data_ptr(), w_in_planes.data_ptr(), b_in_.data_ptr(),
                                              w_out_planes.data_ptr(), b_out_.data_ptr(), w_c_.data_ptr(), b_c_.data_ptr(),
                                              b, L, e, nc, x_planes.data_ptr(), qkv.data_ptr(), probs.data_ptr(),
                                              obar_planes.data_ptr(), emb.data_ptr(), logits.data_ptr(), _stream_ptr(desc))
        check(rc, "gh_attn_head_fwd2")
        ctx.save_for_backward(x_planes, w_in_planes, w_out_planes, w_c_, qkv, probs, obar_planes, emb)
        ctx.dims = (b, L, e, nc)
        return emb, logits

    @staticmethod
    def backward(ctx, d_emb, d_logits):
        x_planes, w_in_planes, w_out_planes, w_c, qkv, probs, obar_planes, emb = ctx.saved_tensors
        b, L, e, nc = ctx.dims
        dev = qkv.device
        need = ctx.needs_input_grad
        d_logits = (torch.zeros((b, nc), device=dev) if d_logits is None else d_logits).contiguous().float()
        d_emb = None if d_emb is None else d_emb.contiguous().float()

        def buf(flag, shape):
            return torch.empty(shape, device=dev, dtype=torch.float32) if flag else None

        d_desc = buf(need[0], (b, L, e))
        gw_in, gb_in = buf(need[1], (3 * e, e)), buf(need[2], (3 * e,))
        gw_out, gb_out = buf(need[3], (e, e)), buf(need[4], (e,))
        gw_c, gb_c = buf(need[5], (nc, e)), buf(need[6], (nc,))
        lib = _lib.lib()
        ws = torch.empty(((lib.gh_attn_head_bwd2_workspace(b, L, e) + 15) // 16 * 4,), device=dev, dtype=torch.float32)
        ptr = lambda t: 0 if t is None else t.data_ptr()
        work = dict(bytes=(3 * e * e + e * e + nc * e) * 4 * 2 + b * L * e * 4 * 8, kind="attn",
                    flops=2 * (2 * b * L * e * 3 * e + 2 * b * e * e + 2 * b * e * nc) + 8 * b * L * L * e)
        with torch.cuda.device(dev), _Timed(f"attn_head_bwd[B={b},L={L},E={e}]", 4, dev, **work):
            rc = lib.gh_attn_head_bwd2(x_planes.data_ptr(), w_in_planes.data_ptr(), w_out_planes.data_ptr(), w_c.data_ptr(),
                                       qkv.data_ptr(), probs.data_ptr(), obar_planes.data_ptr(), emb.data_ptr(),
                                       d_logits.data_ptr(), ptr(d_emb), b, L, e, nc, ptr(d_desc), ptr(gw_in), ptr(gb_in),
                                       ptr(gw_out), ptr(gb_out), ptr(gw_c), ptr(gb_c), ws.data_ptr(), _stream_ptr(qkv))
        check(rc, "gh_attn_head_bwd2")
        return d_desc, gw_in, gb_in, gw_out, gb_out, gw_c, gb_c, None, None


def attention_head(desc, w_in, b_in, w_out, b_out, w_c, b_c):
    L, e, nc = desc.shape[1], desc.shape[2], w_c.shape[0]
    if attn2_supported(L, e, nc) and desc.is_cuda and w_in.dtype == torch.float32 and w_out.dtype == torch.float32:
        return _AttnHead2.apply(desc, w_in, b_in, w_out, b_out, w_c, b_c, weight_planes(w_in), weight_planes(w_out))
    return _AttnHead.apply(desc, w_in, b_in, w_out, b_out, w_c, b_c)


def gemm_planes(a_planes: torch.Tensor, a_mn: bool, b_planes: torch.Tensor, b_mn: bool, bias: torch.Tensor = None,
                planes_out: bool = False, max_split: int = 64) -> torch.Tensor:
    """D = A B^T (+ bias) through gh_gemm_planes. a_planes: (2, M, K) bf16 planes, or (2, K, M) when a_mn (the M index
    contiguous); b_planes: (2, N, K) or (2, K, N) when b_mn. Returns fp32 (M, N), or its (2, M, N) planes."""
    _require_cuda(a_planes, "a_planes")
    assert a_planes.dtype == torch.bfloat16 and b_planes.dtype == torch.bfloat16
    assert a_planes.is_contiguous() and b_planes.is_contiguous()
    m, k = (a_planes.shape[2], a_planes.shape[1]) if a_mn else (a_planes.shape[1], a_planes.shape[2])
    n, k2 = (b_planes.shape[2], b_planes.shape[1]) if b_mn else (b_planes.shape[1], b_planes.shape[2])
    assert k == k2
    dev = a_planes.device
    if planes_out:
        out = torch.empty((2, m, n), device=dev, dtype=torch.bfloat16)
        d, dp = 0, out.data_ptr()
    else:
        out = torch.empty((m, n), device=dev, dtype=torch.float32)
        d, dp = out.data_ptr(), 0
    work = dict(bytes=(m * k + k * n) * 4 + m * n * 4, flops=2 * m * n * k, kind="gemm")
    with torch.cuda.device(dev), _Timed(f"gemm_planes[M={m},N={n},K={k}]", 1, dev, **work):
        rc = _lib.lib().gh_gemm_planes(a_planes.data_ptr(), a_planes.shape[2], a_planes[0].numel(), int(a_mn),
                                       b_planes.data_ptr(), b_planes.shape[2], b_planes[0].numel(), int(b_mn),
                                       0 if bias is None else bias.data_ptr(), d, dp, n, m * n, m, n, k, max_split,
                                       _stream_ptr(a_planes))
    check(rc, "gh_gemm_planes")
    return out
