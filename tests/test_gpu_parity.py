"""Parity of the sm_100a kernels against the oracle, through the C ABI (ops.py is a thin ctypes layer over it).

Behind every Gram entry point sit two kernel families, forced here one at a time (`path`):
  * "ldg"  - single-CTA kernels whose producer warps convert fp32 -> bf16 (round to nearest even) on the way to smem,
             with four loaders (fp32 / bf16, vector / scalar loads) chosen by the tensor's alignment;
  * "pair" - CTA-pair (cta_group::2) kernels with TMA-staged operands: bf16 features feed kind::f16 as they are,
             fp32 features feed kind::tf32, rounded to the nearest tf32 by the TMA unit (TFLOAT32 tensor maps);
  * "auto" - whatever the library picks for the shape (the shipped default).
This file feeds fresh tensors at the shipped shapes. tests/test_gpu_gram_routes.py covers the routes a tensor's layout
selects (strided and misaligned views, every loader, ragged channel counts) and checks which kernel ran;
tests/test_gpu_attention_routes.py does the same for the attention head (both kernel families, batch edges, token
counts, gradient subsets, launch options, large scores) and for the general GEMMs beneath it.

Tolerances (written next to each assert):
  * Gram / descriptor vs the fp64 oracle on fp32 inputs:            normwise rel. err <= 1e-3  (task statement)
                                                                     -- measured 2e-5 .. 3e-4 (bf16), 4e-6 .. 9e-5 (tf32)
  * same vs the fp64 oracle fed the path's operand model:            <= 1e-5  (only fp32 accumulation order differs)
  * attention head fwd/bwd vs fp64 oracle:                           <= 2e-5
  * Gram backward: bf16 operands incl. the bf16-rounded gradient     <= 6e-3 normwise (measured 1.4e-3 .. 2.4e-3);
                   tf32 operands (pair path on fp32 features)        <= 1e-3 (measured 2.2e-4 .. 2.8e-4)
"""
import numpy as np
import pytest
import torch

from conftest import head_params_from
from oracle import head_fp64 as O

pytestmark = pytest.mark.gpu

STAGES = ("stage0", "stage1", "stage2")


@pytest.fixture(scope="module")
def ops():
    from heuristique_style_transfer_code_b200 import ops as _ops
    from heuristique_style_transfer_code_b200 import _lib
    _lib.lib()          # fails loudly when the .so is missing
    return _ops


def npf(t):
    return t.detach().float().cpu().numpy()


PATHS = ("ldg", "pair", "auto")


class kernel_path:
    """Context manager: force one kernel family for the forward and backward Gram entry points."""

    def __init__(self, path):
        self.value = {"ldg": 0, "pair": 1, "auto": -1}[path]

    def __enter__(self):
        from heuristique_style_transfer_code_b200 import _lib
        assert _lib.lib().gh_set_option(b"gram_fwd_pair", self.value) == 0
        assert _lib.lib().gh_set_option(b"gram_bwd_pair", self.value) == 0
        return self

    def __exit__(self, *exc):
        from heuristique_style_transfer_code_b200 import _lib
        _lib.lib().gh_set_option(b"gram_fwd_pair", -1)
        _lib.lib().gh_set_option(b"gram_bwd_pair", -1)
        return False


_ORACLE_CACHE = {}


def cached_oracle(key, fn):
    """The three kernel families of one parametrisation see the same seeded input: evaluate the fp64 oracle once."""
    if key not in _ORACLE_CACHE:
        if len(_ORACLE_CACHE) > 200:
            _ORACLE_CACHE.clear()
        _ORACLE_CACHE[key] = fn()
    return _ORACLE_CACHE[key]


def operand_model_err(got, ref_fn, xf, path, dtype, key=None):
    """Error of `got` against the fp64 oracle fed the operand model of the kernel family that ran.
    ref_fn(rounded_features) -> reference. bf16 features are exact in every family."""
    def ref(model):
        if key is None:
            return ref_fn(model(xf) if model else xf)
        return cached_oracle(key + (model.__name__ if model else "exact",), lambda: ref_fn(model(xf) if model else xf))
    if dtype == "bf16":
        return O.rel_err(got, ref(None))
    models = {"ldg": (O.bf16_round,), "pair": (O.tf32_round, O.bf16_round), "auto": (O.tf32_round, O.bf16_round)}[path]
    # "pair" falls back to the ldg kernels where TMA cannot describe the tensor (e.g. HW = 49: 196 B pitch)
    return min(O.rel_err(got, ref(m)) for m in models)


def test_cuda_is_present():
    assert torch.cuda.is_available(), "pytest -m gpu must run on a CUDA machine"
    assert torch.cuda.get_device_capability()[0] == 10, "kernels are built for sm_100a only"


@pytest.mark.parametrize("B,C,HW,g,ksplit,dtype", [
    (1, 256, 64, 32, 1, "f32"),            # single K block
    (2, 256, 3136, 32, 1, "f32"),          # layer1 @224
    (3, 512, 784, 32, 1, "f32"),           # layer2: 3 super-tiles, off-diagonal one uses two smem stages per k-block
    (2, 1024, 196, 32, 1, "f32"),          # layer3: K tail 196 = 3*64 + 4
    (2, 2048, 49, 32, 1, "f32"),           # layer4: unaligned rows -> scalar loader, k = 64 -> atomics
    (5, 256, 3136, 32, 0, "f32"),          # auto K split
    (5, 256, 3136, 32, 4, "f32"),          # K split, fp32 atomics
    (2, 256, 3136, 32, 1, "bf16"),         # bf16 features
    (3, 512, 784, 32, 1, "bf16"),          # bf16, off-diagonal super-tiles
    (2, 1024, 200, 32, 0, "bf16"),         # bf16, K tail inside a TMA box
    (2, 384, 200, 48, 1, "f32"),           # C not a multiple of 256: padded rows / columns
    (2, 256, 12544, 32, 0, "f32"),         # layer1 @448 (camera config)
    (2, 1024, 196, 8, 1, "f32"),           # k = 128
    (2, 64, 3136, 8, 1, "f32"),            # C < 128: second accumulator is all padding
    (300, 256, 256, 32, 1, "f32"),         # more units than CTAs: persistent loop, ring wrap
    (1, 256, 3136, 32, 0, "f32"),          # batch 1 (camera): K split fills the SMs
])
@pytest.mark.parametrize("path", PATHS)
def test_pooled_gram_forward(ops, B, C, HW, g, ksplit, dtype, path):
    torch.manual_seed(0)
    x = torch.relu(torch.randn(B, C, HW, device="cuda"))
    if dtype == "bf16":
        x = x.bfloat16()
    desc = torch.full((B, 2, g * g), float("nan"), device="cuda")
    ops.KSPLIT = ksplit
    try:
        with kernel_path(path):
            ops.gram_pool_fwd_(x, g, desc, 1)
    finally:
        ops.KSPLIT = 0
    torch.cuda.synchronize()
    got = npf(desc[:, 1])
    xf = npf(x)
    assert torch.isnan(desc[:, 0]).all(), "the other stage's slice must not be touched"
    key = ("pool_fwd", B, C, HW, g, dtype)
    assert O.rel_err(got, cached_oracle(key + ("exact",), lambda: O.descriptors([xf], g)[:, 0])) <= 1e-3
    assert operand_model_err(got, lambda f: O.descriptors([f], g)[:, 0], xf, path, dtype, key) <= 1e-5
    sym = got.reshape(B, g, g)
    assert np.abs(sym - sym.transpose(0, 2, 1)).max() <= 1e-5 * np.abs(sym).max()


@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (768, 3072, 1024), (100, 200, 72), (3, 1024, 1024), (260, 64, 36)])
def test_split_bf16_gemm_all_layouts(ops, M, N, K):
    """gh_gemm_f32 (tcgen05, hi/lo bf16 operands, split-K with atomics when M*N is small): <= 2e-5 vs fp64."""
    torch.manual_seed(0)
    for a_t in (False, True):
        for b_t in (False, True):
            a = torch.randn(K, M, device="cuda").t() if a_t else torch.randn(M, K, device="cuda")
            b = torch.randn(N, K, device="cuda").t() if b_t else torch.randn(K, N, device="cuda")
            bias = torch.randn(N, device="cuda")
            got = ops.gemm_f32(a, b, bias)
            ref = a.double() @ b.double() + bias.double()
            assert float((got.double() - ref).norm() / ref.norm()) <= 2e-5, (a_t, b_t)


@pytest.mark.parametrize("B,C,HW,ksplit", [(1, 64, 3136, 1), (2, 256, 784, 1), (2, 512, 196, 1), (1, 64, 3136, 0),
                                           (2, 320, 100, 1), (1, 256, 196, 1)])
@pytest.mark.parametrize("path", PATHS)
def test_dense_gram_forward(ops, B, C, HW, ksplit, path):
    torch.manual_seed(0)
    x = torch.relu(torch.randn(B, C, HW, device="cuda"))
    ops.KSPLIT = ksplit
    try:
        with kernel_path(path):
            G = ops.gram_dense_fwd(x)
    finally:
        ops.KSPLIT = 0
    torch.cuda.synchronize()
    assert O.rel_err(npf(G), O.gram(npf(x))) <= 1e-3
    assert operand_model_err(npf(G), O.gram, npf(x), path, "f32") <= 1e-5
    assert float((G - G.transpose(1, 2)).abs().max()) <= 1e-6 * float(G.abs().max())


@pytest.mark.parametrize("B,C,HW,g,dtype", [(1, 256, 128, 32, "f32"), (2, 256, 3136, 32, "f32"), (2, 512, 784, 32, "f32"),
                                            (2, 1024, 196, 32, "f32"), (2, 2048, 49, 32, "f32"),
                                            (2, 256, 3136, 32, "bf16"), (40, 256, 784, 32, "f32"), (2, 64, 100, 16, "f32"),
                                            (2, 1024, 200, 32, "bf16"), (2, 384, 200, 48, "f32"), (2, 64, 100, 8, "f32"),
                                            (1, 256, 12544, 32, "f32")])
@pytest.mark.parametrize("path", PATHS)
def test_pooled_gram_backward(ops, B, C, HW, g, dtype, path):
    torch.manual_seed(0)
    x = torch.relu(torch.randn(B, C, HW, device="cuda"))
    if dtype == "bf16":
        x = x.bfloat16()
    dd = torch.randn(B, 2, g * g, device="cuda")
    with kernel_path(path):
        df = ops.gram_pool_bwd(x, g, dd, 1)
    torch.cuda.synchronize()
    err = O.rel_err(npf(df), O.gram_pool_backward(npf(x), g, npf(dd[:, 1])))
    assert err <= 6e-3
    # fp32 features on the pair kernels are tf32 operands (the generated gradient tile included): 10x tighter.
    # (x-contiguous rows of HW = 49 have a 196 B pitch TMA cannot describe: NCHW (2048, 49) stays on the ldg kernels;
    # channels_last (2048, 7, 7) goes to the pair kernels, test_channels_last_features_forward_backward.)
    # The pair kernels take pooled shapes with k = C/g >= 8 and g <= 32; others stay on the ldg kernels as well.
    if path != "ldg" and dtype == "f32" and (HW * 4) % 16 == 0 and C // g >= 8 and g <= 32:
        assert err <= 1e-3


class bwd_operand_in_tmem:
    """Context manager: pooled pair backward with the generated gradient tile in tensor memory (1), in shared memory (0),
    or as shipped (-1: tensor memory for C >= 512) -- gh_set_option("gram_bwd_ats")."""

    def __init__(self, value):
        self.value = value

    def __enter__(self):
        from heuristique_style_transfer_code_b200 import _lib
        assert _lib.lib().gh_set_option(b"gram_bwd_ats", self.value) == 0
        return self

    def __exit__(self, *exc):
        from heuristique_style_transfer_code_b200 import _lib
        _lib.lib().gh_set_option(b"gram_bwd_ats", BWD_ATS_DEFAULT)
        return False


BWD_ATS_DEFAULT = -1


@pytest.mark.parametrize("B,C,H,W,g,dtype,cl", [
    (2, 512, 28, 28, 32, "f32", True),      # layer2, NHWC: x tile 160, A stage = 16 TMEM columns (k-steps reused twice)
    (2, 1024, 14, 14, 32, "f32", True),     # layer3: one x tile of 208 (not a multiple of 32), 8 columns per stage
    (2, 256, 8, 16, 32, "f32", True),       # pooling factor = UMMA_K: every k-step generated, 32 columns per stage
    (2, 256, 8, 16, 32, "bf16", True),      # pooling factor 8 < UMMA_K 16: a k-step holds two table values
    (2, 512, 28, 28, 32, "bf16", True),     # bf16: four A stages only (2 x 32 columns beside each accumulator)
    (2, 1024, 14, 14, 32, "bf16", True),
    (3, 2048, 14, 14, 32, "f32", True),     # eight 256-channel blocks, pooling factor 64
    (1, 2048, 7, 7, 32, "bf16", True),      # layer4: x tile 64
    (2, 512, 28, 28, 32, "f32", False),     # NCHW: F is the MN-major operand
    (2, 1024, 14, 14, 32, "f32", False),
    (2, 512, 28, 28, 32, "bf16", False),
    (2, 160, 10, 20, 20, "bf16", False),    # C not a multiple of the K chunk: partial last chunk, padded rows
    (2, 144, 10, 20, 18, "f32", False),
    (40, 512, 28, 28, 32, "f32", True),     # several units per CTA pair: ring wrap, gradient-table switches
    (300, 512, 8, 8, 32, "f32", True),
])
def test_pooled_gram_backward_with_the_gradient_tile_in_tensor_memory(ops, B, C, H, W, g, dtype, cl):
    """The A operand (dG + dG^T, generated from the g x g descriptor gradient) written to TMEM by tcgen05.st and read from
    there by the MMAs, against the fp64 oracle and against the shared-memory form: same operand values, same K order, so
    the two agree to rounding of the last bit at most."""
    torch.manual_seed(0)
    x = torch.relu(torch.randn(B, C, H, W, device="cuda"))
    if dtype == "bf16":
        x = x.bfloat16()
    xin = x.contiguous(memory_format=torch.channels_last) if cl else x.reshape(B, C, H * W)
    dd = torch.randn(B, 2, g * g, device="cuda")
    from heuristique_style_transfer_code_b200 import _lib
    with kernel_path("pair"):
        with bwd_operand_in_tmem(0):
            ss = ops.gram_pool_bwd(xin, g, dd, 1)
        ts = {}
        try:
            for chunks in (1, 0):                                  # one K chunk per ring stage / as many as fit (two)
                assert _lib.lib().gh_set_option(b"gram_bwd_ch", chunks) == 0
                with bwd_operand_in_tmem(1):
                    ts[chunks] = ops.gram_pool_bwd(xin, g, dd, 1)
        finally:
            _lib.lib().gh_set_option(b"gram_bwd_ch", 0)
    torch.cuda.synchronize()
    ref = O.gram_pool_backward(npf(x).reshape(B, C, H * W), g, npf(dd[:, 1]))
    for t in ts.values():
        assert O.rel_err(npf(t).reshape(ref.shape), ref) <= (1e-3 if dtype == "f32" else 6e-3)
        assert float((t.float() - ss.float()).norm() / ss.float().norm()) <= 1e-6


@pytest.mark.parametrize("B,C,HW", [(1, 64, 3136), (2, 256, 196), (1, 512, 100)])
@pytest.mark.parametrize("path", PATHS)
def test_dense_gram_backward(ops, B, C, HW, path):
    torch.manual_seed(0)
    x = torch.relu(torch.randn(B, C, HW, device="cuda"))
    dg = torch.randn(B, C, C, device="cuda")
    with kernel_path(path):
        df = ops.gram_dense_bwd(x, dg)
    torch.cuda.synchronize()
    err = O.rel_err(npf(df), O.gram_dense_backward(npf(x), npf(dg)))
    assert err <= (6e-3 if path == "ldg" else 1e-3)


@pytest.mark.parametrize("B,C,HW,g", [(2, 256, 196, 24), (2, 64, 100, 7), (2, 256, 100, 64), (2, 64, 3136, 32)])
def test_general_bins_path(ops, B, C, HW, g):
    """C % g != 0: torch's overlapping bins -> dense Gram kernel + bin-rule pooling kernels (forward and backward)."""
    torch.manual_seed(0)
    x = torch.relu(torch.randn(B, C, HW, device="cuda")).requires_grad_(True)
    desc = ops.style_descriptor([x], g)
    w = torch.randn_like(desc)
    (desc * w).sum().backward()
    torch.cuda.synchronize()
    assert O.rel_err(npf(desc), O.descriptors([npf(x)], g)) <= 1e-3
    assert O.rel_err(npf(x.grad), O.gram_pool_backward(npf(x), g, npf(w[:, 0]))) <= 6e-3


class attention_impl:
    """Context manager: "tma" = TMA-fed split-plane GEMMs on CTA pairs (gh_attn_head_fwd2 / _bwd2, the default whenever the
    shape allows), "ldg" = the ld.global-fed kernels (gh_attn_head_fwd / _bwd)."""

    def __init__(self, impl):
        self.impl = impl

    def __enter__(self):
        from heuristique_style_transfer_code_b200 import ops as _ops
        self.saved, _ops.ATTN_IMPL = _ops.ATTN_IMPL, self.impl
        return self

    def __exit__(self, *exc):
        from heuristique_style_transfer_code_b200 import ops as _ops
        _ops.ATTN_IMPL = self.saved
        return False


@pytest.mark.parametrize("impl", ("tma", "ldg"))
@pytest.mark.parametrize("B,L,g,nc", [(5, 3, 8, 4), (33, 3, 32, 4), (4, 1, 16, 3), (7, 4, 8, 10), (1, 3, 32, 4), (2, 8, 8, 16),
                                      (96, 3, 32, 4), (3, 3, 10, 4), (1, 2, 8, 1), (3, 5, 24, 16), (4, 7, 5, 17),
                                      (2, 6, 12, 100)])
def test_attention_head_forward_backward(ops, B, L, g, nc, impl):
    E = g * g
    torch.manual_seed(0)
    desc = torch.randn(B, L, E, device="cuda") * 2.0
    mha = torch.nn.MultiheadAttention(E, 1).cuda()
    lin = torch.nn.Linear(E, nc).cuda()
    with torch.no_grad():
        mha.in_proj_bias.normal_(0, 0.1)
        mha.out_proj.bias.normal_(0, 0.1)
    ps = [mha.in_proj_weight, mha.in_proj_bias, mha.out_proj.weight, mha.out_proj.bias, lin.weight, lin.bias]
    d = desc.clone().requires_grad_(True)
    with attention_impl(impl):
        assert ops.attn2_supported(L, E, nc) == (impl == "tma" and E % 64 == 0)   # g = 10: E = 100 stays on the ldg kernels
        before = ops.LAUNCHES
        emb, logits = ops.attention_head(d, *ps)
        assert ops.LAUNCHES - before >= 4                  # the library's kernels ran (5 + weight splits on the TMA path)
        labels = torch.arange(B, device="cuda") % nc
        w = torch.randn(B, E, device="cuda") * 0.01
        (torch.nn.functional.cross_entropy(logits, labels) + (emb * w).sum()).backward()
    torch.cuda.synchronize()
    names = ("in_proj_weight", "in_proj_bias", "out_proj_weight", "out_proj_bias", "classifier_weight", "classifier_bias")
    params = {k: npf(p) for k, p in zip(names, ps)}
    c = O.attention_forward(npf(desc), *[params[k] for k in names])
    _, dl = O.cross_entropy(c["logits"], labels.cpu().numpy())
    gr = O.attention_backward(c, params, dl, npf(w))
    assert O.rel_err(npf(emb), c["emb"]) <= 2e-5
    assert O.rel_err(npf(logits), c["logits"]) <= 2e-5
    assert O.rel_err(npf(d.grad), gr["d_desc"]) <= 2e-5
    for k, p in zip(names, ps):
        assert O.rel_err(npf(p.grad), gr[k]) <= 2e-5, k


def test_attention_head_tma_forward_is_bitwise_reproducible_and_follows_weight_updates(ops):
    """The forward splits K in at most two partitions: two runs give the same bits. The cached weight planes are rebuilt
    when a parameter changes in place (optimizer step, load_state_dict) and when only some gradients are requested."""
    torch.manual_seed(0)
    B, L, E, nc = 40, 3, 1024, 4
    desc = torch.randn(B, L, E, device="cuda")
    mha = torch.nn.MultiheadAttention(E, 1).cuda()
    lin = torch.nn.Linear(E, nc).cuda()
    ps = [mha.in_proj_weight, mha.in_proj_bias, mha.out_proj.weight, mha.out_proj.bias, lin.weight, lin.bias]
    with torch.no_grad():
        e1, l1 = ops.attention_head(desc, *ps)
        e2, l2 = ops.attention_head(desc, *ps)
        assert torch.equal(e1, e2) and torch.equal(l1, l2)
        mha.in_proj_weight.mul_(1.5)                       # in-place update: version counter moves, planes are rebuilt
        mha.out_proj.weight.add_(0.01)
        e3, l3 = ops.attention_head(desc, *ps)
    names = ("in_proj_weight", "in_proj_bias", "out_proj_weight", "out_proj_bias", "classifier_weight", "classifier_bias")
    c = O.attention_forward(npf(desc), *[npf(p) for p in ps])
    assert O.rel_err(npf(e3), c["emb"]) <= 2e-5 and O.rel_err(npf(l3), c["logits"]) <= 2e-5
    assert not torch.equal(e1, e3)
    # gradient w.r.t. the descriptors only (frozen head): the weight-gradient GEMMs are skipped
    for p in ps:
        p.requires_grad_(False)
    d = desc.clone().requires_grad_(True)
    emb, logits = ops.attention_head(d, *ps)
    labels = torch.arange(B, device="cuda") % nc
    torch.nn.functional.cross_entropy(logits, labels).backward()
    _, dl = O.cross_entropy(c["logits"], labels.cpu().numpy())
    gr = O.attention_backward(c, dict(zip(names, [npf(p) for p in ps])), dl, np.zeros((B, E)))
    assert O.rel_err(npf(d.grad), gr["d_desc"]) <= 2e-5


@pytest.mark.parametrize("M,N,K", [(256, 256, 64), (100, 192, 320), (1536, 1024, 3072), (15, 64, 64), (768, 3072, 1024)])
@pytest.mark.parametrize("a_mn,b_mn", [(False, False), (False, True), (True, False), (True, True)])
def test_split_plane_gemm(ops, M, N, K, a_mn, b_mn):
    """gh_gemm_planes (TMA-fed, CTA pairs, hi/lo bf16 planes): every operand layout the attention head uses, fp32 output
    (plain, two K partitions, free K split with reduce-adds) and split-plane output: <= 2e-5 vs fp64."""
    if a_mn and M % 64:
        pytest.skip("an M-contiguous operand needs M % 64 == 0")
    torch.manual_seed(1)
    A = torch.randn(M, K, device="cuda")
    Bm = torch.randn(N, K, device="cuda")
    bias = torch.randn(N, device="cuda")
    ap = ops.split_bf16(A.t().contiguous() if a_mn else A)
    bp = ops.split_bf16(Bm.t().contiguous() if b_mn else Bm)
    assert torch.equal(ap[0], (A.t().contiguous() if a_mn else A).bfloat16())
    ref = A.double() @ Bm.double().t() + bias.double()
    for max_split in (1, 2, 64):
        got = ops.gemm_planes(ap, a_mn, bp, b_mn, bias, max_split=max_split)
        assert float((got.double() - ref).norm() / ref.norm()) <= 2e-5, max_split
    planes = ops.gemm_planes(ap, a_mn, bp, b_mn, bias, planes_out=True)
    assert float(((planes[0].double() + planes[1].double()) - ref).norm() / ref.norm()) <= 2e-5


def test_golden_small_head_forward_backward(ops, golden_small):
    """Fixture produced by the unmodified reference (tests/golden/make_golden.py): k = 8/16/32 at g = 8."""
    d = golden_small
    g = int(d["g"])
    feats = [torch.from_numpy(d[s]).cuda().requires_grad_(True) for s in STAGES]
    ps = [torch.from_numpy(v).cuda().requires_grad_(True) for v in head_params_from(d).values()]
    desc = ops.style_descriptor(feats, g)
    emb, logits = ops.attention_head(desc, *ps)
    loss = torch.nn.functional.cross_entropy(logits, torch.from_numpy(d["labels"]).cuda())
    loss.backward()
    torch.cuda.synchronize()
    assert O.rel_err(npf(emb), d["embeddings"]) <= 1e-3
    assert O.rel_err(npf(logits), d["logits"]) <= 1e-3
    assert np.array_equal(npf(logits).argmax(1), d["logits"].argmax(1))
    assert abs(loss.item() - float(d["loss"])) <= 1e-3 * abs(float(d["loss"]))
    for f, s in zip(feats, STAGES):
        assert O.rel_err(npf(f.grad), d["d_" + s]) <= 6e-3, s
    for p, k in zip(ps, head_params_from(d)):
        assert O.rel_err(npf(p.grad), d["grad_" + k]) <= 2e-3, k


def test_golden_resnet_descriptors(ops, golden_resnet):
    d = golden_resnet
    feats = [torch.from_numpy(d[s]).cuda() for s in STAGES]
    desc = ops.style_descriptor(feats, int(d["g"]))
    torch.cuda.synchronize()
    assert O.rel_err(npf(desc), d["descriptors"]) <= 1e-3     # bf16-in / fp32-acc vs the fp32 reference


# ---- size-independent properties at BASELINE.json's full sizes -------------------------------------------------------
def _tf32_round_t(x):
    return ((x.view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


@pytest.mark.parametrize("path", ("ldg", "pair"))
@pytest.mark.parametrize("C,HW", [(256, 3136), (512, 784), (1024, 196)])
def test_full_size_properties(ops, C, HW, path):
    with kernel_path(path):
        _full_size_properties(ops, C, HW, path)


def _full_size_properties(ops, C, HW, path):
    B, g = 256, 32
    torch.manual_seed(0)
    x = torch.relu(torch.randn(B, C, HW, device="cuda"))
    desc = torch.empty((B, 1, g * g), device="cuda")
    ops.KSPLIT = 1
    ops.gram_pool_fwd_(x, g, desc, 0)
    base = desc.clone()
    # (1) images are independent: any batch shard gives the same rows, bit for bit (what multi-GPU sharding relies on)
    part = torch.empty((64, 1, g * g), device="cuda")
    ops.gram_pool_fwd_(x[128:192], g, part, 0)
    assert torch.equal(part, base[128:192])
    # (2) degree-2 homogeneity: scaling by a power of two is exact in bf16 and fp32
    ops.gram_pool_fwd_(x * 2.0, g, desc, 0)
    assert torch.equal(desc, base * 4.0)
    # (3) invariance under a permutation of the spatial positions, up to fp32 summation order
    perm = torch.randperm(HW, device="cuda")
    ops.gram_pool_fwd_(x[:, :, perm].contiguous(), g, desc, 0)
    assert float((desc - base).norm() / base.norm()) <= 1e-5
    # (4) trace identity: sum of the pooled diagonal * k  ==  mean_c of ||F_c||^2 / HW  summed ... checked in fp64 on a slice
    k = C // g
    xs = (x[:8].bfloat16() if path == "ldg" else _tf32_round_t(x[:8])).double()   # the family's operand model
    tr = (xs * xs).sum(dim=(1, 2)) / HW
    diag_blocks = base[:8, 0].double().view(8, g, g)
    # sum over all pooled entries * k^2 = sum_cd G[c][d] = ||sum_c F_c||^2 / HW
    tot = (xs.sum(dim=1) ** 2).sum(dim=1) / HW
    assert torch.allclose(diag_blocks.sum(dim=(1, 2)) * k * k, tot, rtol=1e-5)
    assert (diag_blocks.diagonal(dim1=1, dim2=2).sum(1) * k * k <= tr * k * 1.0001 + 1e-6).all()
    ops.KSPLIT = 0
    # (5) K split (atomics) agrees with the deterministic order
    ops.gram_pool_fwd_(x, g, desc, 0)
    assert float((desc - base).norm() / base.norm()) <= 1e-5
    # (6) against torch's fp32 ops on the GPU (the reference's own call sequence) on a 16-image slice
    xs = x[:16]
    ref = torch.nn.functional.adaptive_avg_pool2d(torch.bmm(xs, xs.transpose(1, 2)).div(HW), (g, g)).flatten(1)
    assert float((base[:16, 0] - ref).norm() / ref.norm()) <= 1e-3


# ---- channels_last (NHWC) features consumed natively by the CTA-pair kernels (MN-major operand tiles) -----------------
@pytest.mark.parametrize("B,C,H,W,g,dtype", [(2, 256, 56, 56, 32, "f32"), (3, 512, 28, 28, 32, "f32"), (2, 1024, 14, 14, 32, "f32"),
                                             (2, 256, 56, 56, 32, "bf16"), (3, 512, 28, 28, 32, "bf16"), (2, 1024, 14, 14, 32, "bf16"),
                                             (2, 384, 10, 20, 48, "f32"), (5, 256, 112, 112, 32, "f32"), (2, 64, 10, 10, 8, "f32"),
                                             (1, 2048, 7, 7, 32, "f32"), (1, 2048, 7, 7, 32, "bf16"),      # k = 64: layer4, NHWC default
                                             (2, 1024, 14, 14, 8, "f32"), (2, 1024, 14, 14, 8, "bf16"),    # k = 128
                                             (1, 2048, 14, 14, 32, "f32")])                                # layer4 at 448 x 448
def test_channels_last_features_forward_backward(ops, B, C, H, W, g, dtype):
    torch.manual_seed(0)
    x = torch.relu(torch.randn(B, C, H, W, device="cuda"))
    if dtype == "bf16":
        x = x.bfloat16()
    xcl = x.contiguous(memory_format=torch.channels_last)
    native = ops.nhwc_native(xcl, g)
    assert native == (C % (32 if dtype == "f32" else 64) == 0 and g <= 32)
    desc = torch.full((B, 2, g * g), float("nan"), device="cuda")
    ops.KSPLIT = 1
    try:
        a = xcl.clone().requires_grad_(True)
        d = ops.style_descriptor([a], g)
        w = torch.randn_like(d)
        (d * w).sum().backward()
        if native:
            ops.gram_pool_fwd_(xcl, g, desc, 1)          # the raw entry point on the NHWC tensor
    finally:
        ops.KSPLIT = 0
    torch.cuda.synchronize()
    xf = npf(x).reshape(B, C, H * W)
    ref = O.descriptors([xf], g)[:, 0]
    assert O.rel_err(npf(d[:, 0]), ref) <= 1e-3
    # one fp32 accumulator over all HW positions (KSPLIT = 1): summation-order error grows with K (12 544 at 112 x 112)
    assert operand_model_err(npf(d[:, 0]), lambda f: O.descriptors([f], g)[:, 0], xf, "pair", dtype) <= (1e-5 if H * W <= 4096 else 1e-4)
    if native:
        assert torch.isnan(desc[:, 0]).all()
        if C // g <= 32:
            assert torch.equal(desc[:, 1], d[:, 0])
        else:     # k > 32: a pooled row spans two epilogue warps whose partial sums meet in fp32 atomics (order not fixed)
            assert float((desc[:, 1] - d[:, 0]).norm() / d[:, 0].norm()) <= 1e-6
    gref = O.gram_pool_backward(xf, g, npf(w[:, 0])).reshape(B, C, H, W)
    assert a.grad.dtype == x.dtype and ops.is_channels_last(a.grad)
    err = O.rel_err(npf(a.grad), gref)
    assert err <= (1e-3 if dtype == "f32" and g <= 32 else 6e-3)


@pytest.mark.parametrize("B,C,H,W", [(1, 64, 56, 56), (2, 256, 14, 14), (1, 512, 10, 10)])
def test_channels_last_dense_gram(ops, B, C, H, W):
    torch.manual_seed(0)
    x = torch.relu(torch.randn(B, C, H, W, device="cuda")).contiguous(memory_format=torch.channels_last)
    a = x.clone().requires_grad_(True)
    ops.KSPLIT = 1
    try:
        G = ops.gram_matrix(a)
        dg = torch.randn_like(G)
        (G * dg).sum().backward()
    finally:
        ops.KSPLIT = 0
    torch.cuda.synchronize()
    xf = npf(x).reshape(B, C, H * W)
    assert O.rel_err(npf(G), O.gram(xf)) <= 1e-3
    assert operand_model_err(npf(G), O.gram, xf, "pair", "f32") <= 1e-5
    assert float((G - G.transpose(1, 2)).abs().max()) <= 1e-6 * float(G.abs().max())
    assert ops.is_channels_last(a.grad)
    assert O.rel_err(npf(a.grad), O.gram_dense_backward(xf, npf(dg)).reshape(B, C, H, W)) <= 1e-3


# ---- SURVEY 8(f) n3: fused style-transfer loss on the dense Gram kernels ---------------------------------------------
@pytest.mark.parametrize("B,C,H,W,layout", [(1, 64, 56, 56, "nchw"), (1, 256, 56, 56, "nhwc"), (1, 512, 28, 28, "nhwc"),
                                            (2, 256, 14, 14, "nchw"), (1, 1024, 14, 14, "nhwc")])
def test_style_loss_forward_backward(ops, B, C, H, W, layout):
    """ops.gram_mse_loss = mse_loss(gram_matrix(x), G*) (reference functions/...:286-295) on the dense tcgen05 Gram
    kernels with the fused loss / dG pass: loss and dF against the fp64 oracle (<= 1e-3; tf32 / bf16 operands) and
    against torch's autograd of the reference's own op sequence in fp64 on the same inputs."""
    torch.manual_seed(0)
    x = torch.relu(torch.randn(B, C, H, W, device="cuda"))
    y = torch.relu(torch.randn(B, C, H, W, device="cuda")) * 1.3
    if layout == "nhwc":
        x = x.contiguous(memory_format=torch.channels_last)
    with torch.no_grad():
        target = ops.gram_matrix(y)
    a = x.clone().requires_grad_(True)
    if layout == "nhwc":
        a = x.clone(memory_format=torch.channels_last).requires_grad_(True)
    loss = ops.gram_mse_loss(a, target)
    loss.backward()
    torch.cuda.synchronize()
    xf = npf(x).reshape(B, C, H * W)
    want_loss, want_df = O.style_loss_and_grad(xf, npf(target))
    assert abs(loss.item() - want_loss) <= 1e-3 * want_loss
    assert a.grad.shape == x.shape and O.rel_err(npf(a.grad).reshape(B, C, H * W), want_df) <= 1e-3
    # the reference's ops through autograd, fp64
    xd = x.double().contiguous().requires_grad_(True)
    feats = xd.view(B, C, H * W)
    gram = torch.bmm(feats, feats.transpose(1, 2)).div(H * W)
    ref_loss = torch.nn.functional.mse_loss(gram, target.double())
    ref_loss.backward()
    assert abs(loss.item() - ref_loss.item()) <= 1e-3 * ref_loss.item()
    assert O.rel_err(npf(a.grad), npf(xd.grad)) <= 1e-3
    # composing the separate ops gives the same numbers
    b2 = x.clone().requires_grad_(True)
    torch.nn.functional.mse_loss(ops.gram_matrix(b2), target).backward()
    assert O.rel_err(npf(a.grad), npf(b2.grad)) <= 1e-5 and abs(loss.item() - want_loss) <= 1e-3 * want_loss
