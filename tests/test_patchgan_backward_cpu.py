"""Backward of the Multi-PatchGAN Gram head without a GPU: the fp64 oracle's gradients against torch fp64 autograd of the
fp32 port's op sequence (run in fp64), the C-ABI argument checks of the backward entry points, and the opt-in switch."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from heuristique_style_transfer_code_b200 import _lib
from heuristique_style_transfer_code_b200.build import build_library
from heuristique_style_transfer_code_b200.patchgan import MultiScaleDiscriminator_test, VariablePatchesNLayerDiscriminator_test
from oracle import patchgan_fp64 as O
from oracle.torch_port import patchgan_forward

import patchgan_backward_fp64 as G


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def torch_map_head(fm, ln_input):
    """The port's per-map op sequence (torch_port.patchgan_forward, :198-223) on one (B, D, H, W) map."""
    if ln_input:
        fm = F.layer_norm(fm, fm.shape[1:])
    pooled = F.adaptive_avg_pool2d(fm, output_size=(4, 4))
    pooled = F.layer_norm(pooled, pooled.shape[1:])
    flat = pooled.view(pooled.size(0), fm.shape[1], -1)
    gram = torch.bmm(flat, flat.transpose(1, 2)) / (flat.size(-1) + 1e-6)
    return gram, torch.norm(gram, p='fro', dim=(1, 2))


@pytest.mark.parametrize("shape", [(3, 5, 12, 16), (2, 24, 13, 9), (2, 7, 5, 3), (1, 4, 2, 1), (2, 6, 1, 1), (2, 3, 31, 30)])
@pytest.mark.parametrize("ln_input", [True, False])
def test_map_gradient_against_torch_autograd(shape, ln_input):
    """Ragged and overlapping bins (H % 4 != 0), maps smaller than the 4x4 grid, D = 24."""
    rng = np.random.default_rng(sum(shape))
    x = rng.standard_normal(shape) * 2.0 + 0.7
    b, d = shape[:2]
    dg = rng.standard_normal((b, d, d))
    dn = rng.standard_normal(b)
    xt = torch.tensor(x, requires_grad=True)
    gram, norm = torch_map_head(xt, ln_input)
    ((gram * torch.tensor(dg)).sum() + (norm * torch.tensor(dn)).sum()).backward()
    got = G.patch_gram_grad(x, dg, dn, ln_input)
    assert rel(got, xt.grad.numpy()) < 1e-12


def test_zero_norm_gets_a_zero_norm_gradient_like_torch():
    """A constant map: Z = 0, G = 0, n = 0. torch's norm backward gives 0 there, and so must the oracle."""
    x = np.full((2, 5, 9, 7), 1.25)
    x[1] = np.random.default_rng(3).standard_normal((5, 9, 7))
    dg = np.random.default_rng(4).standard_normal((2, 5, 5))
    dn = np.array([1.5, -0.5])
    for ln_input in (True, False):
        xt = torch.tensor(x, requires_grad=True)
        gram, norm = torch_map_head(xt, ln_input)
        assert float(norm[0].detach()) == 0.0
        ((gram * torch.tensor(dg)).sum() + (norm * torch.tensor(dn)).sum()).backward()
        got = G.patch_gram_grad(x, dg, dn, ln_input)
        assert np.isfinite(got).all()
        assert rel(got, xt.grad.numpy()) < 1e-12


def head_params(m):
    return {k: v.detach().numpy() for k, v in m.state_dict().items() if k in O.HEAD_KEYS}


@pytest.mark.parametrize("ndf,dim,patch,size", [(8, 24, 150, 256), (16, 16, 10, 45)])
def test_head_gradient_against_autograd_of_the_port(ndf, dim, patch, size):
    """Whole head (:198-256) under autograd of oracle/torch_port.patchgan_forward in fp64 on a small discriminator:
    ndf 8 / patch 150 collects L = 8 maps (down to 2x2) with D = 24; patch 10 at 45x45 gives ragged, overlapping bins."""
    torch.manual_seed(ndf + patch)
    m = VariablePatchesNLayerDiscriminator_test(ndf=ndf, norm="instance", patch_size=patch, num_classes=5,
                                                gram_matrix_dim=dim).double()
    with torch.no_grad():
        for a in (m.attention_per_layer, m.attention_per_patch):
            a.in_proj_bias.normal_(0, 0.2)
            a.out_proj.bias.normal_(0, 0.2)
    maps = []

    def keep(mod, inputs, output):
        output.retain_grad()
        maps.append(output)

    hooks = [p.register_forward_hook(keep) for p in m.projection_layers]
    x = torch.randn(2, 3, size, size, dtype=torch.float64)
    emb, out, norms = patchgan_forward(m, x)
    for h in hooks:
        h.remove()
    if patch == 150:
        assert len(maps) == 8 and maps[-1].shape[2:] == (2, 2)
    rng = np.random.default_rng(0)
    w_emb, w_out = rng.standard_normal(emb.shape), rng.standard_normal(out.shape)
    w_n = rng.standard_normal((len(norms), x.shape[0]))
    loss = (emb * torch.tensor(w_emb)).sum() + (out * torch.tensor(w_out)).sum()
    loss = loss + sum((n * torch.tensor(w)).sum() for n, w in zip(norms, w_n))
    loss.backward()
    got = G.patch_head_grad([t.detach().numpy() for t in maps], head_params(m), w_emb, w_out, w_n, heads=8, ln_input=True)
    for t, g in zip(maps, got["maps"]):
        assert rel(g, t.grad.numpy()) < 1e-12
    named = dict(m.named_parameters())
    for k in O.HEAD_KEYS:
        assert rel(got[k], named[k].grad.numpy()) < 1e-12, k


@pytest.fixture(scope="module")
def library():
    build_library()
    return _lib.lib()


def test_backward_entry_points_validate_before_any_cuda_call(library):
    bad, unsup = _lib.GH_ERR_BAD_ARG, _lib.GH_ERR_UNSUPPORTED
    dummy = ctypes.c_void_p(16)
    ints = lambda n, v: (ctypes.c_int * n)(*([v] * n))
    ptrs = (ctypes.c_void_p * 9)(*([16] * 9))
    st = (ctypes.c_longlong * 36)(*([1] * 36))
    assert library.gh_patch_bwd_workspace(6, 256, 64) == 6 * 256 * (64 * 16 + 4)
    assert library.gh_patch_bwd_workspace(0, 1, 1) == 0
    # gh_patch_gram_bwd
    assert library.gh_patch_gram_bwd(None, None, 1, 1, 64, 1, dummy, dummy, dummy, dummy, dummy, None) == bad
    assert library.gh_patch_gram_bwd(ints(2, 4), ints(2, 4), 2, 1, 64, 1, None, dummy, dummy, dummy, dummy, None) == bad
    assert library.gh_patch_gram_bwd(ints(2, 4), ints(2, 0), 2, 1, 64, 1, dummy, dummy, dummy, dummy, dummy, None) == bad
    assert library.gh_patch_gram_bwd(ints(2, 4), ints(2, 4), 2, 1, 64, 1, dummy, dummy, dummy, ctypes.c_void_p(12),
                                     dummy, None) == bad                                                  # 8 B alignment
    assert library.gh_patch_gram_bwd(ints(9, 4), ints(9, 4), 9, 1, 64, 1, dummy, dummy, dummy, dummy, dummy, None) == unsup
    assert library.gh_patch_gram_bwd(ints(2, 4), ints(2, 4), 2, 1, 160, 1, dummy, dummy, dummy, dummy, dummy, None) == unsup
    # gh_patch_pool_bwd: the maps are needed only with ln_input
    assert library.gh_patch_pool_bwd(None, None, ints(2, 4), ints(2, 4), None, st, 2, 1, 64, 0, dummy, None) == bad
    assert library.gh_patch_pool_bwd(None, ptrs, ints(2, 4), ints(2, 4), None, st, 2, 1, 64, 1, dummy, None) == bad
    assert library.gh_patch_pool_bwd(ptrs, ptrs, ints(2, 4), ints(2, 4), st, st, 2, 1, 64, 1, ctypes.c_void_p(8),
                                     None) == bad                                                         # 16 B alignment
    assert library.gh_patch_pool_bwd(ptrs, ptrs, ints(9, 4), ints(9, 4), st, st, 9, 1, 64, 1, dummy, None) == unsup
    assert library.gh_patch_pool_bwd(ptrs, ptrs, ints(2, 4), ints(2, 4), st, st, 2, 1, 129, 1, dummy, None) == unsup
    # gh_patch_attn_bwd: the forward's limits
    assert library.gh_patch_attn_bwd(*([None] * 12), 4, 2, 64, 8, 3, *([None] * 5), None) == bad
    assert library.gh_patch_attn_bwd(*([dummy] * 12), 4, 2, 60, 8, 3, *([dummy] * 5), None) == bad       # E % heads
    assert library.gh_patch_attn_bwd(*([dummy] * 12), 4, 0, 64, 8, 3, *([dummy] * 5), None) == bad       # B
    assert library.gh_patch_attn_bwd(*([dummy] * 12), 9, 2, 64, 8, 3, *([dummy] * 5), None) == unsup     # L > 8
    assert library.gh_patch_attn_bwd(*([dummy] * 12), 4, 2, 256, 8, 3, *([dummy] * 5), None) == unsup   # E > 128
    # the GEMM without a K split, and the column sums
    assert library.gh_gemm_f32_fixed(None, 1, 1, dummy, 1, 1, None, dummy, 4, 4, 4, 4, None) == bad
    assert library.gh_gemm_f32_fixed(dummy, 1, 1, dummy, 1, 1, None, dummy, 4, 4, 4, 0, None) == bad
    assert library.gh_colsum_f32(None, 4, 4, 4, dummy, None) == bad
    assert library.gh_colsum_f32(dummy, 3, 4, 4, dummy, None) == bad                                     # ldx < N
    assert library.gh_colsum_f32(dummy, 4, 0, 4, dummy, None) == bad


def test_library_backward_is_opt_in(monkeypatch):
    monkeypatch.delenv("GRAMHEAD_PATCHGAN_BACKWARD", raising=False)
    m = VariablePatchesNLayerDiscriminator_test(ndf=16, patch_size=10, gram_matrix_dim=8)
    assert m.library_backward is False
    keys = list(m.state_dict())
    assert m.set_library_backward() is m and m.library_backward is True
    assert list(m.state_dict()) == keys                     # a plain attribute: no state_dict key
    m.set_library_backward(False)
    assert m.library_backward is False
    ms = MultiScaleDiscriminator_test(ndf=16, gram_matrix_dim=8)
    assert not any(d.library_backward for d in ms.scale_discriminators.values())
    keys = list(ms.state_dict())
    ms.set_library_backward(True)
    assert all(d.library_backward for d in ms.scale_discriminators.values()) and list(ms.state_dict()) == keys


@pytest.mark.parametrize("value,expected", [("1", True), ("0", False), ("", False), ("yes", False)])
def test_environment_switch(monkeypatch, value, expected):
    monkeypatch.setenv("GRAMHEAD_PATCHGAN_BACKWARD", value)
    assert VariablePatchesNLayerDiscriminator_test(ndf=16, patch_size=10, gram_matrix_dim=8).library_backward is expected
    ms = MultiScaleDiscriminator_test(ndf=16, gram_matrix_dim=8)
    assert all(d.library_backward is expected for d in ms.scale_discriminators.values())
