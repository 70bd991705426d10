"""fp64 statement of the Multi-PatchGAN Gram head's backward  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The gradients of oracle/patchgan_fp64.patch_head (Models/Models_Multi_PatchGAN.py:198-256 of the reference tree) with
respect to the collected feature maps and the head's parameters, written out by hand in numpy fp64:
  patch_gram_grad()           :198-223  whole-map layer norm, 4x4 adaptive pooling, pooled layer norm, Gram, its norm,
                                        in the folded form the CUDA kernels use (csrc/patchgan.cuh)
  multihead_attention_grad()  :243-244  one nn.MultiheadAttention(ndf, 8 heads) over the L layer tokens
  patch_head_grad()           :198-256  all of it, with feature_projection :229, the mean :247 and the classifier :256

It builds on the forward statement in oracle/patchgan_fp64.py. tests/test_patchgan_backward_cpu.py pins it against
torch fp64 autograd of oracle/torch_port.patchgan_forward, and tests/test_gpu_patchgan_backward.py holds the CUDA
backward to it.
"""
from __future__ import annotations

import math
from typing import Dict, Sequence

import numpy as np

from oracle.patchgan_fp64 import GRAM_EPS, LN_EPS, POOL, adaptive_bins, adaptive_pool, multihead_attention, patch_head


def patch_gram_grad(feature_map: np.ndarray, d_gram: np.ndarray, d_norm: np.ndarray, ln_input: bool = False):
    """Backward of patch_gram for one map (B, D, H, W): d_gram (B, D, D), d_norm (B,) -> d_map (B, D, H, W).

    Stated the way the CUDA kernels fold it: with P the pooled (normalised) map, Z = LN(P), G = Z Z^T / (16 + 1e-6),
      dG <- dG + dn G / n              (0 where n == 0, as torch's norm backward)
      dZ  = (dG + dG^T) Z / (16 + 1e-6)
      dP  = r2 (dZ - mean(dZ) - Z mean(dZ * Z))
      dx^(y, x) = sum over the bins i holding (y, x) of dP[i] / |bin i|        (bins overlap when H % 4 != 0)
    and, with ln_input, the whole-map layer norm's two means taken from the 16 D bin values alone
    (sum dx^ = sum dP and sum dx^ * x^ = sum dP * P, overlapping bins included):
      dX  = r (dx^ - sum(dP) / N - x^ sum(dP * P) / N),   N = D H W."""
    x = np.asarray(feature_map, dtype=np.float64)
    b, d, h, w = x.shape
    if ln_input:
        ax = (1, 2, 3)
        mu = x.mean(axis=ax, keepdims=True)
        r = 1.0 / np.sqrt(x.var(axis=ax, keepdims=True) + LN_EPS)
        xh = (x - mu) * r
    else:
        xh = x
    p = adaptive_pool(xh).reshape(b, d, POOL * POOL)
    mean2 = p.mean(axis=(1, 2), keepdims=True)
    r2 = 1.0 / np.sqrt(p.var(axis=(1, 2), keepdims=True) + LN_EPS)
    z = (p - mean2) * r2
    inv = 1.0 / (POOL * POOL + GRAM_EPS)
    g = z @ z.transpose(0, 2, 1) * inv
    n = np.sqrt((g ** 2).sum(axis=(1, 2)))
    scale = np.where(n > 0, np.asarray(d_norm, np.float64) / np.where(n > 0, n, 1.0), 0.0)
    dg = np.asarray(d_gram, np.float64) + scale[:, None, None] * g
    dz = (dg + dg.transpose(0, 2, 1)) @ z * inv
    dp = r2 * (dz - dz.mean(axis=(1, 2), keepdims=True) - z * (dz * z).mean(axis=(1, 2), keepdims=True))
    dp = dp.reshape(b, d, POOL, POOL)
    dxh = np.zeros_like(x)
    for i, (ys, ye) in enumerate(adaptive_bins(h)):
        for j, (xs, xe) in enumerate(adaptive_bins(w)):
            dxh[:, :, ys:ye, xs:xe] += (dp[:, :, i, j] / ((ye - ys) * (xe - xs)))[:, :, None, None]
    if not ln_input:
        return dxh
    n_el = d * h * w
    s1 = dp.sum(axis=(1, 2, 3)).reshape(b, 1, 1, 1)
    s2 = (dp * p.reshape(b, d, POOL, POOL)).sum(axis=(1, 2, 3)).reshape(b, 1, 1, 1)
    return r * (dxh - s1 / n_el - xh * s2 / n_el)


def multihead_attention_grad(x: np.ndarray, dy: np.ndarray, w_in, b_in, w_out, b_out, heads: int):
    """Backward of multihead_attention: dy (L, B, E) -> (dx, dW_in, db_in, dW_out, db_out)."""
    x = np.asarray(x, dtype=np.float64)
    dy = np.asarray(dy, dtype=np.float64)
    w_in, w_out = np.asarray(w_in, np.float64), np.asarray(w_out, np.float64)
    L, B, E = x.shape
    hd = E // heads
    c = math.sqrt(1.0 / hd)
    qkv = x @ w_in.T + np.asarray(b_in, np.float64)
    q, k, v = (qkv[..., i * E:(i + 1) * E].reshape(L, B, heads, hd) for i in range(3))
    s = np.einsum("lbhd,mbhd->bhlm", q * c, k)
    s = s - s.max(axis=-1, keepdims=True)
    p = np.exp(s)
    p /= p.sum(axis=-1, keepdims=True)
    o = np.einsum("bhlm,mbhd->lbhd", p, v).reshape(L, B, E)
    dw_out = dy.reshape(-1, E).T @ o.reshape(-1, E)
    db_out = dy.reshape(-1, E).sum(axis=0)
    do = (dy @ w_out).reshape(L, B, heads, hd)
    dp = np.einsum("lbhd,mbhd->bhlm", do, v)
    dv = np.einsum("bhlm,lbhd->mbhd", p, do)
    ds = p * (dp - (p * dp).sum(axis=-1, keepdims=True))
    dq = np.einsum("bhlm,mbhd->lbhd", ds, k) * c
    dk = np.einsum("bhlm,lbhd->mbhd", ds, q * c)
    dqkv = np.concatenate([t.reshape(L, B, E) for t in (dq, dk, dv)], axis=-1)
    dw_in = dqkv.reshape(-1, 3 * E).T @ x.reshape(-1, E)
    db_in = dqkv.reshape(-1, 3 * E).sum(axis=0)
    return dqkv @ w_in, dw_in, db_in, dw_out, db_out


def patch_head_grad(feature_maps: Sequence[np.ndarray], params: Dict[str, np.ndarray], d_embeddings: np.ndarray,
                    d_output: np.ndarray, d_gram_norms: np.ndarray = None, heads: int = 8,
                    ln_input: bool = False) -> Dict[str, np.ndarray]:
    """Gradients of patch_head's (embeddings, output, gram_norms) cotangents with respect to the L feature maps and the
    parameters named in oracle.patchgan_fp64.HEAD_KEYS. d_gram_norms: (L, B) or None. Returns {"maps": [L arrays],
    "projected": (L, B, E), "grams": (L, B, D, D), <each HEAD_KEYS name>: ...}."""
    f64 = {k: np.asarray(v, dtype=np.float64) for k, v in params.items()}
    fwd = patch_head(feature_maps, params, heads=heads, ln_input=ln_input)
    x0 = fwd["projected"]
    L, B, E = x0.shape
    a1 = [f64["attention_per_layer." + k] for k in ("in_proj_weight", "in_proj_bias", "out_proj.weight", "out_proj.bias")]
    a2 = [f64["attention_per_patch." + k] for k in ("in_proj_weight", "in_proj_bias", "out_proj.weight", "out_proj.bias")]
    x1 = multihead_attention(x0, *a1, heads)
    d_out = np.asarray(d_output, np.float64)
    out = {"classifier.weight": d_out.T @ fwd["embeddings"], "classifier.bias": d_out.sum(axis=0)}
    d_emb = np.asarray(d_embeddings, np.float64) + d_out @ f64["classifier.weight"]
    dy2 = np.broadcast_to(d_emb / L, (L, B, E))
    dx1, *g2 = multihead_attention_grad(x1, dy2, *a2, heads)
    dx0, *g1 = multihead_attention_grad(x0, dx1, *a1, heads)
    for name, grads in (("attention_per_layer", g1), ("attention_per_patch", g2)):
        for key, g in zip(("in_proj_weight", "in_proj_bias", "out_proj.weight", "out_proj.bias"), grads):
            out[f"{name}.{key}"] = g
    grams = fwd["grams"]
    D = grams.shape[-1]
    out["feature_projection.weight"] = dx0.reshape(-1, E).T @ grams.reshape(L * B, D * D)
    out["feature_projection.bias"] = dx0.reshape(-1, E).sum(axis=0)
    d_grams = (dx0 @ f64["feature_projection.weight"]).reshape(L, B, D, D)
    dn = np.zeros((L, B)) if d_gram_norms is None else np.asarray(d_gram_norms, np.float64)
    out["maps"] = [patch_gram_grad(fm, d_grams[l], dn[l], ln_input) for l, fm in enumerate(feature_maps)]
    out["projected"] = dx0
    out["grams"] = d_grams
    return out
