"""fp64 restatement of the reference's Gram + attention head  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this package;
the shipped path (heuristique_style_transfer_code_b200/) never does and has no CPU fallback.

What it restates (file:line relative to the reference tree):
  gram()            Models/Models_RESNET50_TRUNCATE_GRAM_with_Attention.py:26-30   bmm(F, F^T).div(h*w)
  adaptive_pool()   :51-52  F.adaptive_avg_pool2d(gram, (g, g)) on the 3-D (B, C, C) tensor; bins follow ATen's
                    start = floor(i*C/g), end = ceil((i+1)*C/g)
  descriptors()     :54-56  stack(dim=1).flatten(2)  (the permute to (L, B, E) is layout only)
  attention()       :58     nn.MultiheadAttention(embed_dim=g*g, num_heads=1)(X, X, X): packed in_proj, q scaled by
                    1/sqrt(E) before the product, softmax over keys, out_proj, dropout 0
  head_forward()    :59-61 / :110-114  mean over the L stage tokens, classifier Linear
  head_backward()   what loss.backward() (functions/functions_RESNET50_Truncate_Gram_Attention.py:135) derives for the
                    lines above: SURVEY.md Appendix A

Pinning: the reference ships no tests or golden vectors for this path, so this oracle is pinned against outputs of the
unmodified reference module itself, generated in the build container by tests/golden/make_golden.py and committed as
tests/golden/*.npz (tests/test_oracle_golden.py).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence

import numpy as np


def bf16_round(x: np.ndarray) -> np.ndarray:
    """Round-to-nearest-even fp32 -> bf16 -> back, as cvt.rn.bf16.f32 does (operand rounding of the CUDA Gram kernels)."""
    a = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    lsb = (a >> 16) & 1
    a = (a + 0x7FFF + lsb) & 0xFFFF0000
    return a.astype(np.uint32).view(np.float32).reshape(np.shape(x))


def tf32_trunc(x: np.ndarray) -> np.ndarray:
    """fp32 with the low 13 mantissa bits dropped: what a tensor core reading fp32 words as kind::tf32 operands sees."""
    a = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32) & np.uint32(0xFFFFE000)
    return a.view(np.float32).reshape(np.shape(x))


def tf32_round(x: np.ndarray) -> np.ndarray:
    """fp32 rounded to the nearest tf32 (ties away from zero), as cvt.rna.tf32.f32 does."""
    a = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    a = (a + 0x1000) & 0xFFFFE000
    return a.astype(np.uint32).view(np.float32).reshape(np.shape(x))


_OPERAND_ROUNDING = {"bf16": bf16_round, "tf32_trunc": tf32_trunc, "tf32_round": tf32_round}


def gram(features: np.ndarray) -> np.ndarray:
    """(B, C, H, W) or (B, C, HW) -> (B, C, C): F F^T / HW."""
    f = np.asarray(features, dtype=np.float64)
    b, c = f.shape[:2]
    f = f.reshape(b, c, -1)
    return np.einsum("bck,bdk->bcd", f, f, optimize=True) / f.shape[2]


def pool_bins(c: int, g: int):
    starts = [(i * c) // g for i in range(g)]
    ends = [-((-(i + 1) * c) // g) for i in range(g)]
    return starts, ends


def pool_matrix(c: int, g: int) -> np.ndarray:
    """(g, C) averaging matrix: row i holds 1/n_i over bin i."""
    starts, ends = pool_bins(c, g)
    m = np.zeros((g, c), dtype=np.float64)
    for i, (s, e) in enumerate(zip(starts, ends)):
        m[i, s:e] = 1.0 / (e - s)
    return m


def adaptive_pool(gmat: np.ndarray, g: int) -> np.ndarray:
    """(B, C, C) -> (B, g, g)."""
    m = pool_matrix(gmat.shape[-1], g)
    return np.einsum("ic,bcd,jd->bij", m, np.asarray(gmat, dtype=np.float64), m, optimize=True)


def descriptors(features: Sequence[np.ndarray], g: int, operand_rounding: Optional[str] = None) -> np.ndarray:
    """List of L stage feature maps -> (B, L, g*g). operand_rounding in {'bf16', 'tf32_trunc', 'tf32_round'} applies
    that operand model to the Gram operands first (see _OPERAND_ROUNDING)."""
    out = []
    for f in features:
        f = np.asarray(f)
        if operand_rounding is not None:
            f = _OPERAND_ROUNDING[operand_rounding](f.astype(np.float32))
        p = adaptive_pool(gram(f), g)
        out.append(p.reshape(p.shape[0], g * g))
    return np.stack(out, axis=1)


def attention_forward(desc: np.ndarray, w_in, b_in, w_out, b_out, w_c, b_c) -> Dict[str, np.ndarray]:
    x = np.asarray(desc, dtype=np.float64)          # (B, L, E)
    w_in, b_in, w_out, b_out, w_c, b_c = (np.asarray(a, dtype=np.float64) for a in (w_in, b_in, w_out, b_out, w_c, b_c))
    bsz, L, E = x.shape
    qkv = x @ w_in.T + b_in                           # (B, L, 3E)
    q, k, v = qkv[..., :E], qkv[..., E:2 * E], qkv[..., 2 * E:]
    s = np.einsum("ble,bme->blm", q / math.sqrt(E), k)
    s = s - s.max(axis=-1, keepdims=True)
    a = np.exp(s)
    a /= a.sum(axis=-1, keepdims=True)
    o = np.einsum("blm,bme->ble", a, v)
    obar = o.mean(axis=1)                             # mean over stages commutes with out_proj
    emb = obar @ w_out.T + b_out
    logits = emb @ w_c.T + b_c
    return dict(desc=x, qkv=qkv, probs=a, obar=obar, emb=emb, logits=logits)


def head_forward(features: Sequence[np.ndarray], g: int, params: Dict[str, np.ndarray],
                 operand_rounding: Optional[str] = None) -> Dict[str, np.ndarray]:
    """params keys: in_proj_weight, in_proj_bias, out_proj_weight, out_proj_bias, classifier_weight, classifier_bias."""
    desc = descriptors(features, g, operand_rounding)
    return attention_forward(desc, params["in_proj_weight"], params["in_proj_bias"], params["out_proj_weight"],
                             params["out_proj_bias"], params["classifier_weight"], params["classifier_bias"])


def attention_backward(cache: Dict[str, np.ndarray], params: Dict[str, np.ndarray], d_logits: np.ndarray,
                       d_emb_ext: Optional[np.ndarray] = None) -> Dict[str, np.ndarray]:
    x, qkv, a, obar, emb = (cache[k] for k in ("desc", "qkv", "probs", "obar", "emb"))
    w_in = np.asarray(params["in_proj_weight"], dtype=np.float64)
    w_out = np.asarray(params["out_proj_weight"], dtype=np.float64)
    w_c = np.asarray(params["classifier_weight"], dtype=np.float64)
    bsz, L, E = x.shape
    d_logits = np.asarray(d_logits, dtype=np.float64)
    q, k, v = qkv[..., :E], qkv[..., E:2 * E], qkv[..., 2 * E:]
    demb = d_logits @ w_c
    if d_emb_ext is not None:
        demb = demb + np.asarray(d_emb_ext, dtype=np.float64)
    g_wc = d_logits.T @ emb
    g_bc = d_logits.sum(axis=0)
    g_wo = demb.T @ obar
    g_bo = demb.sum(axis=0)
    d_obar = demb @ w_out
    d_o = np.repeat(d_obar[:, None, :], L, axis=1) / L
    d_a = np.einsum("ble,bme->blm", d_o, v)
    d_v = np.einsum("blm,ble->bme", a, d_o)
    d_s = a * (d_a - (d_a * a).sum(axis=-1, keepdims=True)) / math.sqrt(E)
    d_q = np.einsum("blm,bme->ble", d_s, k)
    d_k = np.einsum("blm,ble->bme", d_s, q)
    d_qkv = np.concatenate([d_q, d_k, d_v], axis=-1)             # (B, L, 3E)
    g_win = np.einsum("blo,ble->oe", d_qkv, x)
    g_bin = d_qkv.sum(axis=(0, 1))
    d_desc = d_qkv @ w_in
    return dict(d_desc=d_desc, in_proj_weight=g_win, in_proj_bias=g_bin, out_proj_weight=g_wo, out_proj_bias=g_bo,
                classifier_weight=g_wc, classifier_bias=g_bc)


def gram_pool_backward(features: np.ndarray, g: int, d_pooled: np.ndarray) -> np.ndarray:
    """d_pooled (B, g*g) or (B, g, g) -> dF with the shape of `features`: dF = (dG + dG^T) F / HW, dG = M^T dP M."""
    f = np.asarray(features, dtype=np.float64)
    shape = f.shape
    b, c = shape[:2]
    f = f.reshape(b, c, -1)
    m = pool_matrix(c, g)
    dp = np.asarray(d_pooled, dtype=np.float64).reshape(b, g, g)
    dg = np.einsum("ic,bij,jd->bcd", m, dp, m, optimize=True)
    df = np.einsum("bcd,bdk->bck", dg + dg.transpose(0, 2, 1), f, optimize=True) / f.shape[2]
    return df.reshape(shape)


def gram_dense_backward(features: np.ndarray, d_gram: np.ndarray) -> np.ndarray:
    f = np.asarray(features, dtype=np.float64)
    shape = f.shape
    b, c = shape[:2]
    f = f.reshape(b, c, -1)
    dg = np.asarray(d_gram, dtype=np.float64)
    return (np.einsum("bcd,bdk->bck", dg + dg.transpose(0, 2, 1), f, optimize=True) / f.shape[2]).reshape(shape)


def style_loss_and_grad(features: np.ndarray, target_gram: np.ndarray):
    """Style-transfer objective of one layer (functions/functions_RESNET50_Truncate_Gram_Attention.py:286-295:
    `noise_gram = model.gram_matrix(noise_features); loss = mse_loss(noise_gram, original_gram); loss.backward()`):
    loss = mean over all B*C*C entries of (G - G*)^2 with G = F F^T / HW (Models/...:26-30), and the gradient that reaches
    the activations, dF = (dG + dG^T) F / HW with dG = 2 (G - G*) / (B C C). features (B, C, HW), target (B, C, C).
    -> (loss, dF (B, C, HW))"""
    f = np.asarray(features, np.float64)
    diff = gram(f) - np.asarray(target_gram, np.float64)
    loss = float(np.mean(diff * diff))
    d_gram = 2.0 * diff / diff.size
    return loss, gram_dense_backward(f, d_gram)


def head_backward(features: Sequence[np.ndarray], g: int, params: Dict[str, np.ndarray], cache: Dict[str, np.ndarray],
                  d_logits: np.ndarray, d_emb_ext: Optional[np.ndarray] = None) -> Dict[str, object]:
    grads = attention_backward(cache, params, d_logits, d_emb_ext)
    d_desc = grads["d_desc"]
    grads["d_features"] = [gram_pool_backward(f, g, d_desc[:, l, :]) for l, f in enumerate(features)]
    return grads


def cross_entropy(logits: np.ndarray, labels: np.ndarray):
    """Mean CE and its gradient w.r.t. logits (nn.CrossEntropyLoss default; train script :87)."""
    z = np.asarray(logits, dtype=np.float64)
    z = z - z.max(axis=1, keepdims=True)
    p = np.exp(z)
    p /= p.sum(axis=1, keepdims=True)
    n = z.shape[0]
    loss = -np.log(p[np.arange(n), labels]).mean()
    d = p.copy()
    d[np.arange(n), labels] -= 1.0
    return loss, d / n


def rel_err(a: np.ndarray, b: np.ndarray) -> float:
    """Normwise (Frobenius) relative error of a against reference b."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))
