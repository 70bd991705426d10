"""Every route the Gram entry points can take, against the fp64 oracle.

gram_fwd_common and gram_bwd_common (csrc/gramhead.cu) pick a kernel from the tensor they are given:
  * "pair"      - the CTA-pair kernels, whenever a TMA tensor map can describe the features (and, backward, the gradient);
  * "ldg0".."ldg3" - the single-CTA kernels for every other tensor, by loader (SRC in gram_fwd.cuh / gram_bwd2.cuh):
                  0 fp32 16 B vector loads, 1 fp32 scalar loads, 2 bf16 8 B vector loads, 3 bf16 scalar loads;
  * "unsupported" - refused (GramHeadError).
ops._feature_view hands the strides of any view with x-contiguous rows straight to the library, so the route depends on
the view: channel slices, batch steps, padded pitches and misaligned bases all reach the kernels as they are. Here each
case is built for one route, asserts with expected_route() that the host rules send it there, and checks with
torch.profiler that the kernel of that route is the one that ran. Then:
  1. forward vs the fp64 oracle: <= 1e-3 on exact operands (2^-7 for bf16 operands at HW < 32), <= 1e-5 fed the
     route's operand model (ldg on fp32: bf16 operands, pair on fp32: tf32, bf16 features: exact); the other family's
     model must not fit where the two models differ;
  2. backward vs the fp64 oracle: <= 6e-3 on bf16-operand routes, <= 1e-3 on tf32 routes; the ldg backward also against
     its operand model (bf16 F, bf16 dG + dG^T) at <= 1e-5;
  3. with ops.KSPLIT = 1 and no atomics, the same values through different views on one family give identical bits,
     forward and backward, and so does every grid size (ops.MAX_CTAS);
  4. nothing outside the output is written;
  5. autograd through views of a leaf, and through channel counts the backward kernels do not take (C % 16 != 0, which
     ops.gram_dense_bwd zero-pads).
test_gpu_parity.py covers the shipped shapes on fresh tensors; this file covers the views and the ragged shapes.
"""
import re

import numpy as np
import pytest
import torch

from oracle import head_fp64 as O

pytestmark = pytest.mark.gpu

F32, BF16 = "f32", "bf16"
ENTRIES = ("pool_fwd", "dense_fwd", "pool_bwd", "dense_bwd")
FORCED = {"ldg": 0, "pair": 1, "auto": -1}


@pytest.fixture(scope="module")
def ops():
    from heuristique_style_transfer_code_b200 import ops as _ops
    from heuristique_style_transfer_code_b200 import _lib
    _lib.lib()
    return _ops


def npf(t):
    return t.detach().float().cpu().numpy()


class kernel_path:
    """Force one kernel family for the forward and backward Gram entry points (gram_fwd_pair / gram_bwd_pair), and the
    launch knobs ops.KSPLIT / ops.MAX_CTAS; everything is restored on exit."""

    def __init__(self, forced, ksplit=1, max_ctas=0):
        self.forced, self.ksplit, self.max_ctas = forced, ksplit, max_ctas

    def __enter__(self):
        from heuristique_style_transfer_code_b200 import _lib, ops as _ops
        assert _lib.lib().gh_set_option(b"gram_fwd_pair", self.forced) == 0
        assert _lib.lib().gh_set_option(b"gram_bwd_pair", self.forced) == 0
        self.saved = (_ops.KSPLIT, _ops.MAX_CTAS)
        _ops.KSPLIT, _ops.MAX_CTAS = self.ksplit, self.max_ctas
        return self

    def __exit__(self, *exc):
        from heuristique_style_transfer_code_b200 import _lib, ops as _ops
        _lib.lib().gh_set_option(b"gram_fwd_pair", -1)
        _lib.lib().gh_set_option(b"gram_bwd_pair", -1)
        _ops.KSPLIT, _ops.MAX_CTAS = self.saved
        return False


# ---- the host rules -------------------------------------------------------------------------------------------------
def _tma_ok(addr, img, row, hw, es):
    """make_tensor_map_xcb (csrc/pair.cuh:262-283): 16 B-aligned base, row and image pitches multiples of 16 B, rows at
    least HW long."""
    return addr % 16 == 0 and (row * es) % 16 == 0 and (img * es) % 16 == 0 and row >= hw


def layout(ops, view):
    """(base address, image stride, row stride, B, C, HW) as the op layer passes them; the view itself must reach the
    library (no copy)."""
    t, _, s_img, s_row, s_x, b, c, hw = ops._feature_view(view)
    assert t.data_ptr() == view.data_ptr() and s_x == 1, "ops._feature_view copied the view"
    return view.data_ptr(), s_img, s_row, b, c, hw


def expected_route(view, dtype, mode, g, forced, max_ctas=0):
    """Kernel the library runs for `view` through the ops entry point `mode` (one of ENTRIES) with gram_fwd_pair /
    gram_bwd_pair = `forced` (0 ldg, 1 pair, -1 auto) and ops.MAX_CTAS = max_ctas. Mirrors, in csrc/gramhead.cu:
      gram_fwd_common :129-229  pooled shape check :139-143; pair when a tensor map is made :163-203 (any grid: a single
                                CTA pair when max_ctas < 2); ldg loader by alignment :218-227
      gram_bwd_common :290-405  C % 16 refusal :302; pooled checks (g <= 64, k a power of two) :305-311; pair needs
                                >= 2 CTAs, g <= 32 and k >= 8 when pooled :322, and tensor maps of F AND of the fresh
                                (B, C, HW) gradient :330-341; otherwise the ldg loader by alignment :397-404
    and, in ops.py, _gram_bwd_call (bf16 gradient first for bf16 features, then fp32: either needs HW % 4 == 0 for the
    gradient's map) and gram_dense_bwd (C % 16 != 0: F is copied into a fresh zero-padded (B, C16, HW) tensor first)."""
    from heuristique_style_transfer_code_b200 import ops
    addr, img, row, B, C, HW = layout(ops, view)
    assert (view.dtype == torch.bfloat16) == (dtype == BF16)
    es = 2 if dtype == BF16 else 4
    k = C // g if g and C % g == 0 else 0
    pow2 = k > 0 and k & (k - 1) == 0
    if mode == "dense_bwd" and C % 16:
        C = (C + 15) // 16 * 16
        addr, img, row = 0, C * HW, HW            # torch allocations are 512 B aligned

    def ldg():
        s4 = HW % 4 == 0 and row % 4 == 0 and img % 4 == 0
        if dtype == F32:
            return "ldg0" if s4 and addr % 16 == 0 else "ldg1"
        return "ldg2" if s4 and addr % 8 == 0 else "ldg3"

    if mode in ("pool_fwd", "dense_fwd"):
        if mode == "pool_fwd" and not (pow2 and 8 <= k <= 128):
            return "unsupported"
        return "pair" if forced != 0 and _tma_ok(addr, img, row, HW, es) else ldg()
    if C % 16 or (mode == "pool_bwd" and not (pow2 and g <= 64)):
        return "unsupported"
    want_pair = forced != 0 and max_ctas != 1 and (mode == "dense_bwd" or (g <= 32 and k >= 8))
    if want_pair and _tma_ok(addr, img, row, HW, es) and HW % 4 == 0:
        return "pair"
    return ldg()


_KERNEL_ROUTE = [(re.compile(r"gram_(?:fwd|bwd)_pair_kernel"), lambda m: "pair"),
                 (re.compile(r"gram_(?:fwd|bwd2)_kernel<\(?\w*\)?(\d)"), lambda m: "ldg" + m.group(1))]


def ran(fn):
    """Run fn() under torch.profiler -> (its result, the set of Gram routes whose kernels ran)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    routes = set()
    for name in names:
        for pat, route in _KERNEL_ROUTE:
            m = pat.search(name)
            if m:
                routes.add(route(m))
    return out, routes, names


# ---- views ----------------------------------------------------------------------------------------------------------
def make_view(kind, x, hw_shape=None):
    """x: (B, C, HW) values on the GPU -> a view with x-contiguous rows holding the same values.
    contig     fresh tensor
    offset     base one element past a 16 B boundary
    pitch_tma  rows padded to a multiple of 16 B (what TMA can describe), one 16 B more when HW already is
    pitch4     rows padded to a multiple of 4 elements that is not one of 16 B (bf16: 8 B vector loads, no TMA)
    pitch_odd  rows padded to a pitch that is not a multiple of 4 elements
    chslice3   channels 16 .. 16 + C of a (B, C + 32, HW) tensor
    chslice4   the same of a (B, C + 32, H, W) tensor (hw_shape = (H, W))
    bstep      every other image of a (2B, C, HW) tensor"""
    B, C, HW = x.shape
    per16 = 16 // x.element_size()
    if kind == "contig":
        return x.clone()
    if kind == "offset":
        buf = torch.empty(B * C * HW + per16, device=x.device, dtype=x.dtype)
        v = buf[1:1 + B * C * HW].view(B, C, HW)
        v.copy_(x)
        return v
    if kind.startswith("pitch"):
        if kind == "pitch_tma":
            pitch = (HW // per16 + 1) * per16
        elif kind == "pitch4":
            pitch = (HW // 4 + 1) * 4
            pitch += 4 if pitch % per16 == 0 else 0
        else:
            pitch = HW + 1 + ((HW + 1) % 4 == 0)
        buf = torch.full((B, C, pitch), float("nan"), device=x.device, dtype=x.dtype)
        v = buf[:, :, :HW]
        v.copy_(x)
        return v
    if kind in ("chslice3", "chslice4"):
        full = torch.full((B, C + 32, HW), float("nan"), device=x.device, dtype=x.dtype)
        full[:, 16:16 + C] = x
        if kind == "chslice4":
            full = full.view(B, C + 32, *hw_shape)
        return full[:, 16:16 + C]
    if kind == "bstep":
        full = torch.full((2 * B, C, HW), float("nan"), device=x.device, dtype=x.dtype)
        full[::2] = x
        return full[::2]
    raise ValueError(kind)


def features(B, C, HW, dtype, seed=0):
    torch.manual_seed(seed)
    x = torch.relu(torch.randn(B, C, HW, device="cuda"))
    return x.bfloat16() if dtype == BF16 else x


# ---- one launch of an entry point, with its checks ------------------------------------------------------------------
GUARD = 64


def dense_fwd_guarded(ops, view):
    """ops.gram_dense_fwd through the C ABI into a NaN-filled buffer with GUARD floats on each side: returns (B, C, C) and
    checks that every element of it was written and nothing beside it."""
    from heuristique_style_transfer_code_b200 import _lib
    t, code, s_img, s_row, s_x, b, c, hw = ops._feature_view(view)
    buf = torch.full((b * c * c + 2 * GUARD,), float("nan"), device=view.device)
    out = buf[GUARD:GUARD + b * c * c]
    rc = _lib.lib().gh_gram_dense_fwd(t.data_ptr(), code, s_img, s_row, s_x, b, c, hw, out.data_ptr(), ops.KSPLIT,
                                      ops.MAX_CTAS, torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "gh_gram_dense_fwd")
    torch.cuda.synchronize()
    assert torch.isnan(buf[:GUARD]).all() and torch.isnan(buf[GUARD + b * c * c:]).all(), "written outside the Gram"
    assert not torch.isnan(out).any(), "Gram elements left unwritten"
    return out.view(b, c, c)


def launch(ops, mode, view, g, d_out):
    """Run one entry point on `view`. d_out: the (B, 3, g*g) descriptor gradient (pool_bwd, slice 1 is read) or the
    (B, C, C) Gram gradient (dense_bwd). -> result tensor."""
    B = view.shape[0]
    if mode == "pool_fwd":
        desc = torch.full((B, 3, g * g), float("nan"), device="cuda")
        ops.gram_pool_fwd_(view, g, desc, 1)
        torch.cuda.synchronize()
        assert torch.isnan(desc[:, 0]).all() and torch.isnan(desc[:, 2]).all(), "other stages' slices were written"
        assert not torch.isnan(desc[:, 1]).any()
        return desc[:, 1].clone()
    if mode == "dense_fwd":
        return dense_fwd_guarded(ops, view)
    if mode == "pool_bwd":
        return ops.gram_pool_bwd(view, g, d_out, 1)
    return ops.gram_dense_bwd(view, d_out)


_ORACLE = {}


def oracle(key, fn):
    """fp64 references depend on the values only: evaluated once per input (across views and families)."""
    if key not in _ORACLE:
        if len(_ORACLE) > 64:
            _ORACLE.clear()
        _ORACLE[key] = fn()
    return _ORACLE[key]


def ldg_bwd_model(xf, mode, g, d):
    """What the ldg backward computes, in fp64: bf16(F) and bf16(M), M = dG + dG^T summed in fp32 (dense), or the pooled
    table dP + dP^T summed in fp32 and upsampled by k (pool). dF = M F / HW."""
    B, C, HW = xf.shape
    f = O.bf16_round(xf).astype(np.float64)
    if mode == "pool_bwd":
        dp = d.reshape(B, g, g).astype(np.float32)
        sym = O.bf16_round(dp + dp.transpose(0, 2, 1)).astype(np.float64)
        k = C // g
        m = np.repeat(np.repeat(sym, k, axis=1), k, axis=2) / (k * k)
    else:
        dg = d.astype(np.float32)
        m = O.bf16_round(dg + dg.transpose(0, 2, 1)).astype(np.float64)
    return np.matmul(m, f) / HW


def check_case(ops, mode, x, view, g, route, key):
    """Launch `mode` on `view` (values x) expecting `route`; check against the oracle. -> result (for bitwise checks)."""
    B, C, HW = x.shape
    dtype = BF16 if x.dtype == torch.bfloat16 else F32
    xf = npf(x)
    torch.manual_seed(1)
    d_out = (torch.randn(B, 3, g * g, device="cuda") if mode == "pool_bwd" else
             torch.randn(B, C, C, device="cuda") if mode == "dense_bwd" else None)
    got_t, routes, names = ran(lambda: launch(ops, mode, view, g, d_out))
    assert routes == {route}, f"expected the {route} kernel, ran {routes or sorted(n for n in names if 'gram' in n)}"
    got = npf(got_t)
    if mode.endswith("fwd"):
        ref = (lambda f: O.descriptors([f], g)[:, 0]) if mode == "pool_fwd" else O.gram
        exact = oracle(key + ("exact",), lambda: ref(xf))
        # bf16 operands (ldg on fp32): each product carries up to 2^-7 of rounding error, which sums over HW positions
        # average down below 1e-3 only when there are enough of them (measured 1.7e-3 .. 4.5e-3 at HW = 1, 2, 7)
        bf16_ops = route != "pair" and dtype == F32
        assert O.rel_err(got, exact) <= (2 ** -7 if bf16_ops and HW < 32 else 1e-3)
        if dtype == BF16:
            assert O.rel_err(got, exact) <= 1e-5            # bf16 features are exact operands on every route
        else:
            own, other = (O.tf32_round, O.bf16_round) if route == "pair" else (O.bf16_round, O.tf32_round)
            r_own = oracle(key + (own.__name__,), lambda: ref(own(xf)))
            r_other = oracle(key + (other.__name__,), lambda: ref(other(xf)))
            assert O.rel_err(got, r_own) <= 1e-5
            if O.rel_err(r_own, r_other) >= 1e-4:          # the two operand models are told apart on this input
                assert O.rel_err(got, r_other) > 1e-5, "the other family's operand model fits: wrong kernel family?"
        if mode == "dense_fwd":
            assert float((got_t - got_t.transpose(1, 2)).abs().max()) <= 1e-6 * float(got_t.abs().max())
    else:
        d = npf(d_out[:, 1] if mode == "pool_bwd" else d_out)
        ref = oracle(key + ("bwd",), lambda: O.gram_pool_backward(xf, g, d) if mode == "pool_bwd"
                     else O.gram_dense_backward(xf, d))
        assert got_t.shape == (B, C, HW)
        err = O.rel_err(got, ref)
        assert err <= (1e-3 if route == "pair" and dtype == F32 else 6e-3)
        if route.startswith("ldg"):
            assert O.rel_err(got, oracle(key + ("bwd_ldg",), lambda: ldg_bwd_model(xf, mode, g, d))) <= 1e-5
    return got_t


# ---- 1. views x families x entry points -----------------------------------------------------------------------------
# kind, dtype, HW, (H, W) for the 4-D slice, routes forward (ldg forced, pair forced / auto), backward (the same)
VIEW_CASES = [
    ("contig", F32, 64, None, ("ldg0", "pair"), ("ldg0", "pair")),
    ("offset", F32, 64, None, ("ldg1", "ldg1"), ("ldg1", "ldg1")),
    ("pitch_tma", F32, 64, None, ("ldg0", "pair"), ("ldg0", "pair")),
    ("pitch_odd", F32, 64, None, ("ldg1", "ldg1"), ("ldg1", "ldg1")),
    ("chslice3", F32, 64, None, ("ldg0", "pair"), ("ldg0", "pair")),
    ("chslice4", F32, 64, (8, 8), ("ldg0", "pair"), ("ldg0", "pair")),
    ("bstep", F32, 64, None, ("ldg0", "pair"), ("ldg0", "pair")),
    ("contig", F32, 63, None, ("ldg1", "ldg1"), ("ldg1", "ldg1")),
    ("offset", F32, 63, None, ("ldg1", "ldg1"), ("ldg1", "ldg1")),
    ("pitch_tma", F32, 63, None, ("ldg1", "pair"), ("ldg1", "ldg1")),     # backward: 63-float gradient rows, no TMA
    ("contig", BF16, 64, None, ("ldg2", "pair"), ("ldg2", "pair")),
    ("offset", BF16, 64, None, ("ldg3", "ldg3"), ("ldg3", "ldg3")),
    ("pitch_tma", BF16, 64, None, ("ldg2", "pair"), ("ldg2", "pair")),
    ("pitch4", BF16, 64, None, ("ldg2", "ldg2"), ("ldg2", "ldg2")),
    ("pitch_odd", BF16, 64, None, ("ldg3", "ldg3"), ("ldg3", "ldg3")),
    ("chslice3", BF16, 64, None, ("ldg2", "pair"), ("ldg2", "pair")),
    ("chslice4", BF16, 64, (4, 16), ("ldg2", "pair"), ("ldg2", "pair")),
    ("bstep", BF16, 64, None, ("ldg2", "pair"), ("ldg2", "pair")),
    ("contig", BF16, 63, None, ("ldg3", "ldg3"), ("ldg3", "ldg3")),
    ("offset", BF16, 63, None, ("ldg3", "ldg3"), ("ldg3", "ldg3")),
    ("pitch_tma", BF16, 63, None, ("ldg3", "pair"), ("ldg3", "ldg3")),
]
VIEW_B, VIEW_C, VIEW_G = 2, 160, 20        # k = 8; 160 channels: one partial 256-channel super-tile


def view_routes(family, mode):
    """-> [(kind, dtype, HW, hw_shape, declared route)] of VIEW_CASES for one family and entry point."""
    col = 0 if family == "ldg" else 1
    return [(kind, dt, hw, shp, (fr if mode.endswith("fwd") else br)[col]) for kind, dt, hw, shp, fr, br in VIEW_CASES]


@pytest.mark.parametrize("dtype", (F32, BF16))
@pytest.mark.parametrize("mode", ENTRIES)
@pytest.mark.parametrize("family", ("ldg", "pair", "auto"))
def test_views_take_their_route_and_match_the_oracle(ops, family, mode, dtype):
    """Same values through every view: the declared route, the oracle, and identical bits between views of one HW on one
    family (KSPLIT = 1, pooling factor 8: no atomics)."""
    g = VIEW_G if mode.startswith("pool") else 0
    first = {}
    with kernel_path(FORCED[family]):
        for kind, dt, hw, shp, route in view_routes(family, mode):
            if dt != dtype:
                continue
            x = features(VIEW_B, VIEW_C, hw, dtype)
            v = make_view(kind, x, shp)
            assert expected_route(v, dtype, mode, g, FORCED[family]) == route, (kind, hw)
            got = check_case(ops, mode, x, v, g, route, (mode, dtype, hw, g))
            fam = "pair" if route == "pair" else "ldg"
            ref_kind, ref = first.setdefault((hw, fam), (kind, got))
            assert got.dtype == ref.dtype and torch.equal(got, ref), f"{kind} differs from {ref_kind} on {route}"


# ---- 2. refusals ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", (F32, BF16))
def test_unsupported_shapes_raise_and_write_nothing(ops, dtype):
    from heuristique_style_transfer_code_b200._lib import GramHeadError
    x = features(2, 96, 64, dtype)                        # g = 8: k = 12 is not a power of two
    assert expected_route(x, dtype, "pool_fwd", 8, -1) == "unsupported"
    desc = torch.full((2, 2, 64), float("nan"), device="cuda")
    with pytest.raises(GramHeadError):
        ops.gram_pool_fwd_(x, 8, desc, 1)
    assert torch.isnan(desc).all()
    x = features(2, 40, 64, dtype)                        # C % 16 != 0: the pooled backward is not padded
    assert expected_route(x, dtype, "pool_bwd", 5, -1) == "unsupported"
    with pytest.raises(GramHeadError):
        ops.gram_pool_bwd(x, 5, torch.randn(2, 1, 25, device="cuda"), 0)


# ---- 3. shapes where tiling goes wrong ------------------------------------------------------------------------------
# B, C, HW (g for pooled). Every C has an odd HW, whose K tail also ends inside a 16-wide k-step, most an even one too.
DENSE_SHAPES = [(3, 1, 7), (2, 1, 2), (3, 3, 63), (2, 3, 196), (3, 17, 65), (3, 17, 2), (2, 100, 1), (2, 100, 196),
                (2, 129, 63), (1, 129, 1023), (2, 255, 7), (2, 255, 100), (2, 257, 65), (2, 257, 196), (1, 383, 1023),
                (2, 383, 2), (1, 520, 63), (1, 520, 196)]
POOL_SHAPES = [(2, 96, 12, 63), (2, 96, 12, 196),         # k = 8, C < 128: the second accumulator is padding
               (2, 160, 20, 65), (2, 160, 20, 100),        # k = 8, one partial super-tile
               (2, 224, 28, 7), (2, 224, 28, 196),
               (2, 288, 36, 63), (2, 288, 36, 196),        # g > 32: the backward stays on the ldg kernels
               (2, 640, 40, 65), (2, 640, 40, 196),        # k = 16
               (1, 1536, 48, 63), (1, 1536, 48, 100),      # k = 32
               (1, 2048, 16, 7), (1, 2048, 16, 36)]        # k = 128: pooled rows meet in atomics


def _shape_view(x):
    """Rows padded to 16 B when they are not already (as nhwc_to_nchw pads them), so the pair family can take any HW."""
    return x.clone() if (x.shape[2] * x.element_size()) % 16 == 0 else make_view("pitch_tma", x)


@pytest.mark.parametrize("family", ("ldg", "pair"))
@pytest.mark.parametrize("dtype", (F32, BF16))
@pytest.mark.parametrize("B,C,HW", DENSE_SHAPES)
def test_dense_gram_ragged_shapes(ops, B, C, HW, dtype, family):
    x = features(B, C, HW, dtype)
    v = _shape_view(x)
    with kernel_path(FORCED[family], ksplit=0):
        for mode in ("dense_fwd", "dense_bwd"):
            route = expected_route(v, dtype, mode, 0, FORCED[family])
            assert route != "pair" if family == "ldg" else (route == "pair" or mode == "dense_bwd")
            check_case(ops, mode, x, v, 0, route, ("shape", mode, dtype, B, C, HW))


@pytest.mark.parametrize("family", ("ldg", "pair"))
@pytest.mark.parametrize("dtype", (F32, BF16))
@pytest.mark.parametrize("B,C,g,HW", POOL_SHAPES)
def test_pooled_gram_tiling_shapes(ops, B, C, g, HW, dtype, family):
    x = features(B, C, HW, dtype)
    v = _shape_view(x)
    with kernel_path(FORCED[family], ksplit=0):
        for mode in ("pool_fwd", "pool_bwd"):
            route = expected_route(v, dtype, mode, g, FORCED[family])
            assert route != "pair" if family == "ldg" else (route == "pair" or mode == "pool_bwd")
            check_case(ops, mode, x, v, g, route, ("shape", mode, dtype, B, C, HW, g))


# ---- 4. grid size -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", (F32, BF16))
@pytest.mark.parametrize("family", ("ldg", "pair"))
@pytest.mark.parametrize("mode,B,C,HW,g", [("dense", 3, 257, 136, 0), ("pool", 3, 512, 136, 32)])
def test_grid_size_does_not_change_the_bits(ops, mode, B, C, HW, g, family, dtype):
    """ops.MAX_CTAS = 1, 2, 3, 5 against the default grid, KSPLIT = 1: more units than CTAs (persistent loop, ring and
    phase wrap) with one writer per output element. MAX_CTAS = 1 sends the pair backward to the ldg kernels."""
    x = features(B, C, HW, dtype)
    torch.manual_seed(1)
    d_out = torch.randn(B, 3, g * g, device="cuda") if mode == "pool" else torch.randn(B, C, C, device="cuda")
    fwd, bwd = mode + "_fwd", mode + "_bwd"
    base = {}
    for fam in ("ldg", family):
        with kernel_path(FORCED[fam]):
            base[fam] = (launch(ops, fwd, x, g, None), launch(ops, bwd, x, g, d_out))
    for max_ctas in (1, 2, 3, 5):
        with kernel_path(FORCED[family], max_ctas=max_ctas):
            for i, m in enumerate((fwd, bwd)):
                route = expected_route(x, dtype, m, g, FORCED[family], max_ctas)
                got, routes, _ = ran(lambda: launch(ops, m, x, g, d_out))
                assert routes == {route}
                want = base["pair" if route == "pair" else "ldg"][i]
                assert torch.equal(got, want), (m, max_ctas, route)


# ---- 5. autograd ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", (F32, BF16))
@pytest.mark.parametrize("kind", ("chslice", "bstep"))
@pytest.mark.parametrize("fn", ("style_descriptor", "gram_matrix"))
def test_autograd_through_views_of_a_leaf(ops, fn, kind, dtype):
    """The gradient reaches the leaf inside the view only (exact zeros elsewhere) and matches the oracle there."""
    B, C, H, W, g = 2, 160, 8, 8, 20
    torch.manual_seed(0)
    full = torch.relu(torch.randn((B, C + 32, H, W) if kind == "chslice" else (2 * B, C, H, W), device="cuda"))
    leaf = (full.bfloat16() if dtype == BF16 else full).requires_grad_(True)
    view = leaf[:, 16:16 + C] if kind == "chslice" else leaf[::2]
    out = ops.style_descriptor([view], g) if fn == "style_descriptor" else ops.gram_matrix(view)
    w = torch.randn_like(out)
    (out * w).sum().backward()
    torch.cuda.synchronize()
    xf = npf(view).reshape(B, C, H * W)
    if fn == "style_descriptor":
        assert O.rel_err(npf(out), O.descriptors([xf], g)) <= 1e-3
        ref = O.gram_pool_backward(xf, g, npf(w[:, 0]))
        route = expected_route(view, dtype, "pool_bwd", g, -1)
    else:
        assert O.rel_err(npf(out), O.gram(xf)) <= 1e-3
        ref = O.gram_dense_backward(xf, npf(w))
        route = expected_route(view, dtype, "dense_bwd", 0, -1)
    grad = leaf.grad
    mask = torch.zeros_like(grad, dtype=torch.bool)
    if kind == "chslice":
        mask[:, 16:16 + C] = True
    else:
        mask[::2] = True
    assert grad.dtype == leaf.dtype and (grad[~mask] == 0).all()
    inside = npf(grad[:, 16:16 + C] if kind == "chslice" else grad[::2]).reshape(B, C, H * W)
    assert O.rel_err(inside, ref) <= (1e-3 if route == "pair" and dtype == F32 else 6e-3)


@pytest.mark.parametrize("dtype", (F32, BF16))
@pytest.mark.parametrize("B,C,H,W,cl", [(2, 3, 7, 9, False), (2, 17, 8, 8, False), (2, 17, 7, 7, True),
                                        (1, 100, 14, 14, False), (2, 100, 5, 5, True)])
def test_ragged_channels_autograd(ops, B, C, H, W, cl, dtype):
    """gram_matrix and gram_mse_loss backward at C % 16 != 0 (gram_dense_bwd zero-pads the channels), NCHW and
    channels_last, against the fp64 oracle."""
    torch.manual_seed(0)
    x = torch.relu(torch.randn(B, C, H, W, device="cuda"))
    x = x.bfloat16() if dtype == BF16 else x
    if cl:
        x = x.contiguous(memory_format=torch.channels_last)
    xf = npf(x).reshape(B, C, H * W)
    tol = 6e-3                                             # some of these HW take the ldg kernels (bf16 operands)
    a = x.clone().requires_grad_(True)
    G = ops.gram_matrix(a)
    dg = torch.randn_like(G)
    (G * dg).sum().backward()
    assert a.grad.shape == x.shape and a.grad.dtype == x.dtype and ops.is_channels_last(a.grad) == cl
    assert O.rel_err(npf(G), O.gram(xf)) <= 1e-3
    assert O.rel_err(npf(a.grad).reshape(B, C, H * W), O.gram_dense_backward(xf, npf(dg))) <= tol
    target = O.gram(xf * 1.3).astype(np.float32)
    b = x.clone().requires_grad_(True)
    loss = ops.gram_mse_loss(b, torch.from_numpy(target).cuda())
    loss.backward()
    want_loss, want_df = O.style_loss_and_grad(xf, target)
    assert abs(loss.item() - want_loss) <= 1e-3 * want_loss
    assert O.rel_err(npf(b.grad).reshape(B, C, H * W), want_df) <= tol


@pytest.mark.parametrize("dtype", (F32, BF16))
@pytest.mark.parametrize("B,C,HW,g", [(2, 40, 64, 5), (2, 24, 63, 3), (2, 100, 49, 10)])
def test_style_descriptor_ragged_channels(ops, B, C, HW, g, dtype):
    """Pooled forward with C % 16 != 0 (k = 8 for C = 40 and 24): its backward goes through adaptive_pool_bwd and the
    padded dense backward."""
    x = features(B, C, HW, dtype).requires_grad_(True)
    desc = ops.style_descriptor([x], g)
    w = torch.randn_like(desc)
    (desc * w).sum().backward()
    torch.cuda.synchronize()
    xf = npf(x)
    assert O.rel_err(npf(desc), O.descriptors([xf], g)) <= 1e-3
    assert O.rel_err(npf(x.grad), O.gram_pool_backward(xf, g, npf(w[:, 0]))) <= 6e-3


# ---- 6. coverage ------------------------------------------------------------------------------------------------------
ROUTE_TABLE = {(m, dt, r) for m in ENTRIES for dt, rs in ((F32, ("pair", "ldg0", "ldg1")), (BF16, ("pair", "ldg2", "ldg3")))
               for r in rs} | {(m, dt, "unsupported") for m in ("pool_fwd", "pool_bwd") for dt in (F32, BF16)}


def test_every_route_is_reached():
    """Each route x dtype x entry point is declared by at least one case above (and each case asserts that it gets its
    declared route from expected_route() and from the kernel that ran)."""
    reached = {(m, dt, r) for fam in ("ldg", "pair", "auto") for m in ENTRIES for _, dt, _, _, r in view_routes(fam, m)}
    reached |= {(m, dt, "unsupported") for m in ("pool_fwd", "pool_bwd") for dt in (F32, BF16)}   # the refusal test
    print("reached:", sorted(reached))
    assert reached == ROUTE_TABLE, sorted(ROUTE_TABLE - reached)
