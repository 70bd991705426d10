"""fp64 numpy model of the fused stem of the inference plan (gh_stem_conv_pool_nhwc, csrc/stem.cuh):
    maxpool3x3/s2/p1( relu( conv7x7/s2/p3(x, w) + bias ) )
on tf32-rounded operands (head_fp64.tf32_round: what cvt.rna.tf32.f32 does to the image, and what the plan does to the
folded weights before packing them). The bias is added in fp32 by the kernel and is not rounded. NaN propagates through
the window as in nn.MaxPool2d, and ReLU keeps it."""
from __future__ import annotations

import numpy as np

from .head_fp64 import tf32_round


def stem_fp64(x: np.ndarray, w: np.ndarray, bias: np.ndarray, round_operands: bool = True) -> np.ndarray:
    """x: (B, 3, H, W), w: (O, 3, 7, 7), bias: (O,) -> (B, O, PH, PW) float64, PH = (H/2 - 1)//2 + 1 (H, W even)."""
    x = np.asarray(x, dtype=np.float32)
    w = np.asarray(w, dtype=np.float32)
    if round_operands:
        x, w = tf32_round(x), tf32_round(w)
    x, w = x.astype(np.float64), w.astype(np.float64)
    b, c, h, wd = x.shape
    o = w.shape[0]
    oh, ow = (h + 6 - 7) // 2 + 1, (wd + 6 - 7) // 2 + 1
    xp = np.zeros((b, c, h + 6, wd + 6))
    xp[:, :, 3:h + 3, 3:wd + 3] = x
    conv = np.zeros((b, o, oh, ow))
    for i in range(7):
        for j in range(7):
            patch = xp[:, :, i:i + 2 * oh:2, j:j + 2 * ow:2]                  # (B, C, OH, OW)
            conv += np.einsum("bchw,oc->bohw", patch, w[:, :, i, j])
    conv += np.asarray(bias, dtype=np.float64).reshape(1, o, 1, 1)
    act = np.where(np.isnan(conv), conv, np.maximum(conv, 0.0))
    ph, pw = (oh + 2 - 3) // 2 + 1, (ow + 2 - 3) // 2 + 1
    ap = np.full((b, o, oh + 2, ow + 2), -np.inf)
    ap[:, :, 1:oh + 1, 1:ow + 1] = act
    out = np.full((b, o, ph, pw), -np.inf)
    for i in range(3):
        for j in range(3):
            out = np.maximum(out, ap[:, :, i:i + 2 * ph:2, j:j + 2 * pw:2])   # np.maximum propagates NaN
    return out
