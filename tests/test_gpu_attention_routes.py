"""Every route the attention head and the general GEMMs beneath it can take, against the fp64 oracle.

The head (csrc/gramhead.cu) has two kernel families:
  * "tma" - gh_attn_head_fwd2 / _bwd2: split-bf16 planes fed by TMA to tgemm_pair_kernel on CTA pairs, with the per-image
            kernels of attn_head2.cuh. Taken when ops.attn2_supported and attn2_supported (gramhead.cu) agree:
            E % 64 == 0, 64 <= E <= 1024, L <= 8, nc <= 16.
  * "ldg" - gh_attn_head_fwd / _bwd: every product on gemm_auto, which picks umma_gemm_kernel<A_MN, B_MN> (tcgen05) or
            sgemm_strided_kernel<AK, BK> (fp32 FMA) per product from the strides, alignment, N >= 64 and `accumulate`.
Both instantiate their per-image kernels for L <= 4 (<4>) and 5 <= L <= 8 (<8>, masked tokens); L = 9 is refused.
expected_route() restates these rules; each case asserts that its shape lands on the route it was built for, and
torch.profiler confirms that the route's kernels are the ones that ran. Then:
  1. shape matrix, both families, forward and backward vs oracle/head_fp64: normwise <= 2e-5 on qkv, probs, emb, logits,
     d_desc and every parameter gradient, and per image <= 1e-4 of the batch's RMS row norm on emb / logits / d_desc;
  2. batch independence: an image gives the same emb / logits bits alone and in a batch when the forward GEMMs split K
     alike, else within 4e-5; d_desc within 4e-5; a NaN image leaves every other image finite;
  3. gradient subsets (which outputs the backward is asked for, losses on emb or logits only): only the requested
     gradients are computed (GEMM / column-sum launches counted), and they match the oracle;
  4. launch options of the TMA head (tgemm_tn, pdl): the oracle, and identical forward bits across pdl and repeats;
  5. scores of 1e2 .. 1e5, checked in stages so that near-ties in the softmax do not hide or fake an error;
  6. every output of the C ABI sits inside NaN padding: nothing outside it is written, everything inside it is;
  7. gh_gemm_f32 on each route, gh_gemm_f32_fixed, gh_colsum_f32 and gh_split_bf16 against fp64 / torch;
  8. refusals write nothing.
test_gpu_parity.py::test_attention_head_forward_backward covers small shapes through autograd on fresh tensors.
Measured errors (B200) are written next to each bound.
"""
import ctypes
import math
import re

import numpy as np
import pytest
import torch

from oracle import head_fp64 as O

pytestmark = pytest.mark.gpu

GH_ERR_UNSUPPORTED = -2
ORACLE_NAMES = {"d_desc": "d_desc", "w_in": "in_proj_weight", "b_in": "in_proj_bias", "w_out": "out_proj_weight",
                "b_out": "out_proj_bias", "w_c": "classifier_weight", "b_c": "classifier_bias"}
GRADS = tuple(ORACLE_NAMES)
PARAM_NAMES = ("in_proj_weight", "in_proj_bias", "out_proj_weight", "out_proj_bias", "classifier_weight",
               "classifier_bias")
TOL = 2e-5            # normwise, every tensor of the head (measured <= 1.3e-5 over the matrix)
TOL_IMAGE = 1e-4      # per image, relative to the RMS row norm of the batch (measured <= 3.2e-5)


@pytest.fixture(scope="module")
def ops():
    from heuristique_style_transfer_code_b200 import ops as _ops
    from heuristique_style_transfer_code_b200 import _lib
    _lib.lib()
    return _ops


def lib():
    from heuristique_style_transfer_code_b200 import _lib
    return _lib.lib()


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def npf(t):
    return t.detach().float().cpu().numpy()


def stream():
    return torch.cuda.current_stream().cuda_stream


def batch(b):
    """Batch sizes relative to the SM count: "2S" = one CTA per image in attn2_core_bwd_kernel's single wave, "2S+1" =
    its persistent loop."""
    return {"2S": 2 * sms(), "2S+1": 2 * sms() + 1}.get(b, b)


class options:
    """gh_set_option("tgemm_tn" / "pdl") for the body; both are restored to their defaults (0 = plan, 1 = PDL) on exit."""

    def __init__(self, tn=0, pdl=1):
        self.tn, self.pdl = tn, pdl

    def __enter__(self):
        assert lib().gh_set_option(b"tgemm_tn", self.tn) == 0 and lib().gh_set_option(b"pdl", self.pdl) == 0
        return self

    def __exit__(self, *exc):
        lib().gh_set_option(b"tgemm_tn", 0)
        lib().gh_set_option(b"pdl", 1)
        return False


# ---- the host rules -------------------------------------------------------------------------------------------------
def tgemm_plan(M, N, K, max_split=2):
    """(tn, ksplit) of one forward GEMM: gh_tgemm_plan, the host planner gh_attn_head_fwd2 runs per GEMM
    (gh_attn_head_fwd2 plans each GEMM alone with tg_plan, tgemm_pair.cuh), on sms / 2 CTA pairs."""
    tn, ks, units = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    assert lib().gh_tgemm_plan(M, N, K, max_split, sms() // 2, ctypes.byref(tn), ctypes.byref(ks), ctypes.byref(units)) == 0
    return tn.value, ks.value


def family(L, E, nc, impl="tma"):
    """ops.attention_head's choice (ops.attn2_supported) and the C entry points' own refusals (kMaxL = 8)."""
    if not 1 <= L <= 8:
        return "unsupported"
    if impl == "tma" and E % 64 == 0 and 64 <= E <= 1024 and 1 <= nc <= 16 and sms() >= 2:
        return "tma"
    return "ldg"


def umma_ksplit(M, N, K):
    """K partitions launch_umma_gemm plans (umma_gemm.cuh:311-321)."""
    ntiles, nkb = -(-M // 128) * -(-N // 256), -(-K // 64)
    if ntiles >= sms():
        return 1
    return max(1, min(sms() // ntiles, max(nkb // 2, 1)))


def gemm_route(a_sm, a_sk, b_sk, b_sn, M, N, K, accumulate=False, a_ptr=0, b_ptr=0):
    """gemm_auto (gramhead.cu:65-75) + launch_umma_gemm's alignment rule (umma_gemm.cuh:304-307) ->
    "umma<A_MN,B_MN>" or "sgemm<AK,BK>"."""
    if not accumulate and 1 in (a_sk, a_sm) and 1 in (b_sk, b_sn):
        a_mn, b_mn = a_sk != 1, b_sk != 1
        lda, ldb = (a_sk if a_mn else a_sm), (b_sk if b_mn else b_sn)
        if (lda % 4 == 0 and ldb % 4 == 0 and a_ptr % 16 == 0 and b_ptr % 16 == 0 and (M if a_mn else K) % 4 == 0
                and (N if b_mn else K) % 4 == 0 and N >= 64):
            return f"umma<{str(a_mn).lower()},{str(b_mn).lower()}>"
    return f"sgemm<{str(a_sk == 1).lower()},{str(b_sk == 1).lower()}>"


def ldg_products(B, L, E, nc, d_emb=True, want=GRADS):
    """Each gemm_auto call of gh_attn_head_fwd / _bwd (gramhead.cu:635-642, 1217-1241) -> its kernel. demb accumulates
    onto the external embedding gradient when there is one, which rules out the tensor-core kernel."""
    BL = B * L
    p = {"in_proj": (E, 1, 1, E, BL, 3 * E, E, False), "out_proj": (E, 1, 1, E, B, E, E, False),
         "demb": (nc, 1, E, 1, B, E, nc, d_emb), "dobar": (E, 1, E, 1, B, E, E, False)}
    if "w_c" in want:
        p["dW_c"] = (1, nc, E, 1, nc, E, B, False)
    if "w_out" in want:
        p["dW_out"] = (1, E, E, 1, E, E, B, False)
    if "w_in" in want:
        p["dW_in"] = (1, 3 * E, E, 1, 3 * E, E, BL, False)
    if "d_desc" in want:
        p["d_desc"] = (3 * E, 1, E, 1, BL, E, 3 * E, False)
    return {k: gemm_route(*v) for k, v in p.items()}


def expected_route(B, L, E, nc, impl="tma", d_emb=True, want=GRADS):
    """-> dict: family, the L template, and per family the facts the launch depends on:
    tma: the forward plans (tn, ksplit) of in_proj and out_proj, attn2_bwd_prep_kernel's row-loop trips (one below 257
    images, gramhead.cu attn2_bwd_prep_kernel step 4 * kRowStep = 256), attn2_core_bwd_kernel single wave or persistent
    (grid = min(B, 2 * SMs)); the backward plans two problems per launch, which gh_tgemm_plan does not expose.
    ldg: the kernel of every product."""
    fam = family(L, E, nc, impl)
    r = {"family": fam}
    if fam == "unsupported":
        return r
    r["LT"] = 4 if L <= 4 else 8
    if fam == "tma":
        r["in_proj"] = tgemm_plan(B * L, 3 * E, E)
        r["out_proj"] = tgemm_plan(B, E, E)
        r["prep_trips"] = 1 if B <= 256 else 2
        r["core_bwd"] = "persistent" if B > 2 * sms() else "single"
    else:
        r["products"] = ldg_products(B, L, E, nc, d_emb, want)
    return r


def route_cells(r):
    """The cells of the route table a case reaches."""
    if r["family"] == "unsupported":
        return {("family", "unsupported")}
    f = r["family"]
    cells = {("family", f), (f, "LT", r["LT"])}
    if f == "tma":
        cells |= {("tma", "in_proj") + r["in_proj"], ("tma", "out_proj") + r["out_proj"],
                  ("tma", "prep_trips", r["prep_trips"]), ("tma", "core_bwd", r["core_bwd"])}
    else:
        cells |= {("ldg", k, v) for k, v in r["products"].items()}
    return cells


# ---- profiler -------------------------------------------------------------------------------------------------------
_KERNEL = re.compile(r"(\w+_kernel)(<[^>]*>)?")


OUR_KERNELS = ("tgemm_pair_kernel", "attn2_core_fwd_kernel", "attn2_classifier_kernel", "attn2_bwd_prep_kernel",
               "attn2_core_bwd_kernel", "split_bf16_kernel", "attn_core_fwd_kernel", "classifier_fwd_kernel",
               "attn_core_bwd_kernel", "umma_gemm_kernel", "sgemm_strided_kernel", "colsum_kernel")


def _canon(name):
    m = _KERNEL.search(name)
    if not m or m.group(1) not in OUR_KERNELS:
        return None
    args = (m.group(2) or "").replace(" ", "").replace("(bool)1", "true").replace("(bool)0", "false")
    args = re.sub(r"\(\w+\)", "", args)
    return m.group(1).replace("sgemm_strided_kernel", "sgemm").replace("umma_gemm_kernel", "umma") + args


def ran(fn):
    """Run fn() under torch.profiler -> (result, the library's kernels that ran, one entry per launch, and "memset" per
    device memset; torch's own kernels are left out)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = []
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        if "memset" in e.name.lower():
            names.append("memset")
        else:
            c = _canon(e.name)
            if c:
                names.append(c)
    return out, names


def check_kernels(r, names, direction, ldg_products_run=None):
    """The kernels of the route ran (and no kernel of the other family)."""
    ks = set(names)
    LT = r["LT"]
    if r["family"] == "tma":
        want = ({f"attn2_core_fwd_kernel<{LT}>", "attn2_classifier_kernel", "tgemm_pair_kernel", "split_bf16_kernel"}
                if direction == "fwd" else {"attn2_bwd_prep_kernel", f"attn2_core_bwd_kernel<{LT}>", "tgemm_pair_kernel"})
        assert want <= ks, (want - ks, names)
        assert not any(n.startswith(("umma", "sgemm", "attn_core", "classifier_fwd")) for n in ks), names
        if direction == "fwd":
            assert names.count("tgemm_pair_kernel") == 2
            assert ("memset" in ks) == (r["in_proj"][1] > 1), names    # only a K-split in_proj zeroes qkv first
    else:
        prods = ldg_products_run
        gemms = {v for k, v in prods.items() if (k in ("in_proj", "out_proj")) == (direction == "fwd")}
        want = ({f"attn_core_fwd_kernel<{LT}>", "classifier_fwd_kernel"} if direction == "fwd" else {"attn_core_bwd_kernel"})
        got_gemms = {n for n in ks if n.startswith(("umma<", "sgemm<"))}
        assert want <= ks and got_gemms == gemms, (want, gemms, names)
        assert not any(n.startswith(("tgemm", "attn2")) for n in ks), names


# ---- the C ABI with guarded outputs ---------------------------------------------------------------------------------
PAD_BYTES = 256


class Outputs:
    """Output buffers, each inside NaN padding of PAD_BYTES on both sides (16 B-aligned offsets) and NaN-filled itself.
    check() asserts that the padding is untouched and that every element of every output was written."""

    def __init__(self):
        self.bufs = []

    def __call__(self, shape, dtype=torch.float32, name="", offset=0):
        n = int(np.prod(shape))
        pad = PAD_BYTES // torch.empty((), dtype=dtype).element_size()
        full = torch.full((n + 2 * pad + offset,), float("nan"), device="cuda", dtype=dtype)
        self.bufs.append((name, full, pad + offset, n))
        return full[pad + offset:pad + offset + n].view(shape)

    def untouched(self):
        torch.cuda.synchronize()
        return all(torch.isnan(full).all() for _, full, _, _ in self.bufs)

    def check(self, allow_nan=()):
        torch.cuda.synchronize()
        for name, full, lo, n in self.bufs:
            assert torch.isnan(full[:lo]).all() and torch.isnan(full[lo + n:]).all(), f"{name}: written outside"
            if name not in allow_nan:
                assert not torch.isnan(full[lo:lo + n]).any(), f"{name}: elements left unwritten"


def head_params(E, nc, seed=0):
    """nn.MultiheadAttention / nn.Linear initialisation scales, biases N(0, 0.1)."""
    g = torch.Generator().manual_seed(seed)
    u = lambda *s: torch.rand(*s, generator=g) * 2 - 1
    ps = [u(3 * E, E) * math.sqrt(6 / (4 * E)), torch.randn(3 * E, generator=g) * 0.1, u(E, E) / math.sqrt(E),
          torch.randn(E, generator=g) * 0.1, u(nc, E) / math.sqrt(E), u(nc) / math.sqrt(E)]
    return [p.cuda() for p in ps]


def inputs(B, L, E, nc, seed=0, scale=2.0):
    g = torch.Generator().manual_seed(seed + 1)
    desc = (torch.randn(B, L, E, generator=g) * scale).cuda()
    d_logits = (torch.randn(B, nc, generator=g) * 0.1).cuda()
    d_emb = (torch.randn(B, E, generator=g) * 0.01).cuda()
    return desc, d_logits, d_emb


def fwd(fam, desc, P, out=None):
    """One forward through the C ABI -> (rc, dict of outputs). TMA: the weight planes are made here (ops.split_bf16)."""
    B, L, E = desc.shape
    nc = P[4].shape[0]
    out = out if out is not None else Outputs()
    r = dict(out=out, qkv=out((B * L, 3 * E), name="qkv"), probs=out((B, L, L), name="probs"),
             emb=out((B, E), name="emb"), logits=out((B, nc), name="logits"))
    from heuristique_style_transfer_code_b200 import ops
    if fam == "tma":
        r["w_planes"] = (ops.split_bf16(P[0]), ops.split_bf16(P[2]))
        r["x_planes"] = out((2, B * L, E), torch.bfloat16, "x_planes")
        r["obar_planes"] = out((2, B, E), torch.bfloat16, "obar_planes")
        rc = lib().gh_attn_head_fwd2(desc.data_ptr(), r["w_planes"][0].data_ptr(), P[1].data_ptr(),
                                     r["w_planes"][1].data_ptr(), P[3].data_ptr(), P[4].data_ptr(), P[5].data_ptr(),
                                     B, L, E, nc, r["x_planes"].data_ptr(), r["qkv"].data_ptr(), r["probs"].data_ptr(),
                                     r["obar_planes"].data_ptr(), r["emb"].data_ptr(), r["logits"].data_ptr(), stream())
    else:
        r["obar"] = out((B, E), name="obar")
        rc = lib().gh_attn_head_fwd(desc.data_ptr(), *[p.data_ptr() for p in P], B, L, E, nc, r["qkv"].data_ptr(),
                                    r["probs"].data_ptr(), r["obar"].data_ptr(), r["emb"].data_ptr(),
                                    r["logits"].data_ptr(), stream())
    return rc, r


def bwd(fam, desc, P, r, d_logits, d_emb, want=GRADS, out=None):
    """One backward through the C ABI on the saved tensors of fwd() -> (rc, dict of the requested gradients)."""
    B, L, E = desc.shape
    nc = P[4].shape[0]
    out = out if out is not None else Outputs()
    shapes = {"d_desc": (B, L, E), "w_in": (3 * E, E), "b_in": (3 * E,), "w_out": (E, E), "b_out": (E,),
              "w_c": (nc, E), "b_c": (nc,)}
    g = {k: out(shapes[k], name=k) if k in want else None for k in GRADS}
    g["out"] = out
    ptr = lambda t: 0 if t is None else t.data_ptr()
    gp = [ptr(g[k]) for k in GRADS]
    if fam == "tma":
        ws = torch.empty(((lib().gh_attn_head_bwd2_workspace(B, L, E) + 15) // 16 * 4,), device="cuda")
        rc = lib().gh_attn_head_bwd2(r["x_planes"].data_ptr(), r["w_planes"][0].data_ptr(), r["w_planes"][1].data_ptr(),
                                     P[4].data_ptr(), r["qkv"].data_ptr(), r["probs"].data_ptr(),
                                     r["obar_planes"].data_ptr(), r["emb"].data_ptr(), d_logits.data_ptr(), ptr(d_emb),
                                     B, L, E, nc, *gp, ws.data_ptr(), stream())
    else:
        ws = torch.empty((lib().gh_attn_head_bwd_workspace(B, L, E),), device="cuda")
        rc = lib().gh_attn_head_bwd(desc.data_ptr(), P[0].data_ptr(), P[2].data_ptr(), P[4].data_ptr(),
                                    r["qkv"].data_ptr(), r["probs"].data_ptr(), r["obar"].data_ptr(), r["emb"].data_ptr(),
                                    d_logits.data_ptr(), ptr(d_emb), B, L, E, nc, *gp, ws.data_ptr(), stream())
    return rc, g


def oracle_fwd(desc, P):
    return O.attention_forward(npf(desc), *[npf(p) for p in P])


def oracle_bwd(c, P, d_logits, d_emb):
    return O.attention_backward(c, dict(zip(PARAM_NAMES, [npf(p) for p in P])), npf(d_logits),
                                None if d_emb is None else npf(d_emb))


def close(got, ref, what, tol=TOL, per_image=None):
    """Normwise bound, and optionally per image (rows of the leading axis) relative to the RMS row norm of ref."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    if not np.any(ref):
        assert not np.any(got), f"{what}: nonzero where the oracle is exactly zero"
        return
    err = O.rel_err(got, ref)
    assert err <= tol, f"{what}: normwise error {err:.3g} > {tol:.3g}"
    if per_image:
        B = ref.shape[0]
        rows = np.linalg.norm((got - ref).reshape(B, -1), axis=1)
        scale = math.sqrt(np.mean(np.linalg.norm(ref.reshape(B, -1), axis=1) ** 2))
        worst = int(np.argmax(rows))
        assert rows[worst] <= per_image * scale, f"{what}: image {worst} off by {rows[worst] / scale:.3g} of the RMS row"
        print(f"  {what} per image: {rows[worst] / scale:.2e}")
    print(f"  {what}: {err:.2e}")


# ---- 1. shape matrix ------------------------------------------------------------------------------------------------
# B, L, E, nc, impl (ops.ATTN_IMPL the shape is run under), family it must land on
HEAD_CASES = [
    (1, 1, 64, 1, "tma", "tma"),
    (255, 2, 256, 16, "tma", "tma"),
    (256, 5, 576, 3, "tma", "tma"),            # 144 of 256 threads per image; in_proj N = 1728, out_proj N = 576
    (257, 6, 1024, 16, "tma", "tma"),          # second trip of attn2_bwd_prep_kernel's row loop
    ("2S", 7, 256, 4, "tma", "tma"),
    ("2S+1", 8, 64, 1, "tma", "tma"),          # persistent attn2_core_bwd_kernel
    (512, 3, 1024, 4, "tma", "tma"),
    (5, 1, 4, 1, "tma", "ldg"),                # g = 2: every product on the SIMT kernel
    (255, 2, 16, 17, "tma", "ldg"),            # g = 4: N < 64 everywhere; nc > 16
    (257, 5, 25, 100, "tma", "ldg"),           # g = 5: E % 4 != 0
    ("2S+1", 7, 49, 16, "tma", "ldg"),         # g = 7
    (256, 6, 100, 100, "tma", "ldg"),          # g = 10: tcgen05 products, nc % 4 == 0 as M of dW_c
    (512, 8, 144, 17, "tma", "ldg"),           # g = 12, nc > 16
    (3, 3, 1296, 4, "tma", "ldg"),             # E > 1024 falls to the ldg family
    (40, 3, 256, 17, "tma", "ldg"),            # a TMA width with nc > 16
    (3, 3, 1024, 4, "ldg", "ldg"),
]


def case_id(c):
    return f"B{c[0]}-L{c[1]}-E{c[2]}-nc{c[3]}-{c[4]}"


def run_case(B, L, E, nc, fam, seed=0, want=GRADS, with_d_emb=True):
    """Forward + backward through the C ABI with guarded outputs, under the profiler; checks the kernels and the guards.
    -> (desc, P, d_logits, d_emb, forward outputs, gradients, route)"""
    P = head_params(E, nc, seed)
    desc, d_logits, d_emb = inputs(B, L, E, nc, seed)
    d_emb = d_emb if with_d_emb else None
    r = expected_route(B, L, E, nc, impl=fam, d_emb=with_d_emb, want=want)
    assert r["family"] == fam
    (rc, f), names = ran(lambda: fwd(fam, desc, P))
    assert rc == 0
    check_kernels(r, names, "fwd", r.get("products"))
    f["out"].check()
    (rc, g), names = ran(lambda: bwd(fam, desc, P, f, d_logits, d_emb, want))
    assert rc == 0
    check_kernels(r, names, "bwd", r.get("products"))
    g["out"].check()
    return desc, P, d_logits, d_emb, f, g, r, names


@pytest.mark.parametrize("case", HEAD_CASES, ids=case_id)
def test_head_shape_matrix(case):
    B, L, E, nc, impl, fam = case
    B = batch(B)
    assert family(L, E, nc, impl) == fam
    desc, P, d_logits, d_emb, f, g, r, _ = run_case(B, L, E, nc, fam)
    c = oracle_fwd(desc, P)
    close(npf(f["qkv"]).reshape(B, L, 3 * E), c["qkv"], "qkv")
    close(npf(f["probs"]), c["probs"], "probs")
    close(npf(f["emb"]), c["emb"], "emb", per_image=TOL_IMAGE)
    close(npf(f["logits"]), c["logits"], "logits", per_image=TOL_IMAGE)
    gr = oracle_bwd(c, P, d_logits, d_emb)
    for k in GRADS:
        close(npf(g[k]), gr[ORACLE_NAMES[k]], k, per_image=TOL_IMAGE if k == "d_desc" else None)


# ---- 2. batch independence ------------------------------------------------------------------------------------------
def forward_splits(fam, B, L, E):
    """K partitions of the two forward GEMMs."""
    if fam == "tma":
        return tgemm_plan(B * L, 3 * E, E)[1], tgemm_plan(B, E, E)[1]
    return tuple(umma_ksplit(M, N, K) if gemm_route(E, 1, 1, E, M, N, K).startswith("umma") else 1
                 for M, N, K in ((B * L, 3 * E, E), (B, E, E)))


TOL_ALONE = 4e-5      # an image alone vs in a batch, when K is split differently (measured <= 4.0e-6)


@pytest.mark.parametrize("B,L,E,nc,fam", [(300, 3, 1024, 4, "tma"), (257, 5, 576, 16, "tma"), (100, 3, 100, 10, "ldg"),
                                          (300, 2, 49, 17, "ldg"), (64, 7, 256, 4, "ldg")])
def test_an_image_does_not_depend_on_its_batch(B, L, E, nc, fam):
    P = head_params(E, nc, 3)
    desc, d_logits, d_emb = inputs(B, L, E, nc, 3)
    rc, f = fwd(fam, desc, P)
    assert rc == 0
    rc, g = bwd(fam, desc, P, f, d_logits, d_emb, want=("d_desc",))
    assert rc == 0
    same_splits = forward_splits(fam, B, L, E) == forward_splits(fam, 1, L, E)
    for i in (0, B // 2, B - 1):
        sl = slice(i, i + 1)
        rc, f1 = fwd(fam, desc[sl].contiguous(), P)
        assert rc == 0
        rc, g1 = bwd(fam, desc[sl].contiguous(), P, f1, d_logits[sl].contiguous(), d_emb[sl].contiguous(), want=("d_desc",))
        assert rc == 0
        for k in ("emb", "logits"):
            if same_splits:
                assert torch.equal(f[k][sl], f1[k]), (k, i)
            else:
                close(npf(f[k][sl]), npf(f1[k]), f"{k}[{i}] alone", TOL_ALONE)
        close(npf(g["d_desc"][sl]), npf(g1["d_desc"]), f"d_desc[{i}] alone", TOL_ALONE)
    print(f"  same forward K splits alone and in the batch: {same_splits}")


@pytest.mark.parametrize("fam,E", [("tma", 256), ("ldg", 100), ("ldg", 49)])
def test_a_nan_image_stays_in_its_rows(fam, E):
    B, L, nc, bad = 64, 3, 4, 5
    P = head_params(E, nc)
    desc, d_logits, d_emb = inputs(B, L, E, nc)
    desc[bad, 1, 3] = float("nan")
    rc, f = fwd(fam, desc, P)
    assert rc == 0
    rc, g = bwd(fam, desc, P, f, d_logits, d_emb, want=("d_desc",))
    assert rc == 0
    keep = torch.arange(B, device="cuda") != bad
    for k, t in (("emb", f["emb"]), ("logits", f["logits"]), ("d_desc", g["d_desc"])):
        assert torch.isfinite(t[keep]).all(), k
        assert not torch.isfinite(t[bad]).all(), k


# ---- 3. gradient subsets ----------------------------------------------------------------------------------------------
# which of (desc, w_in, b_in, w_out, b_out, w_c, b_c) require grad; the TMA backward plans its launches by these
# (gramhead.cu gh_attn_head_bwd2: dW_out adds a problem to the first GEMM launch, dW_in / d_desc make the second)
SUBSETS = [GRADS, ("d_desc",), GRADS[1:], ("w_in",), ("w_out", "b_c"), ("d_desc", "b_in", "w_c"), ("b_out",),
           ("d_desc", "w_out")]


@pytest.mark.parametrize("loss", ("both", "emb", "logits"))
@pytest.mark.parametrize("fam,B,L,E,nc", [("tma", 40, 3, 256, 4), ("ldg", 40, 3, 100, 100)])
def test_gradient_subsets(ops, fam, B, L, E, nc, loss):
    P0 = head_params(E, nc, 1)
    desc0, d_logits, d_emb = inputs(B, L, E, nc, 1)
    c = oracle_fwd(desc0, P0)
    gr = oracle_bwd(c, P0, d_logits if loss != "emb" else torch.zeros_like(d_logits), d_emb if loss != "logits" else None)
    saved = ops.ATTN_IMPL
    try:
        ops.ATTN_IMPL = fam
        for want in SUBSETS:
            leaves = [desc0.clone()] + [p.clone() for p in P0]
            for k, t in zip(GRADS, leaves):
                t.requires_grad_(k in want)
            emb, logits = ops.attention_head(*leaves)
            terms = ([(logits * d_logits).sum()] if loss != "emb" else []) + ([(emb * d_emb).sum()] if loss != "logits" else [])
            _, names = ran(lambda: sum(terms).backward())
            # autograd hands the backward a zero gradient for an output the loss does not use, so d_emb is never null
            # here: the logits-only route without it is test_loss_on_the_logits_only_through_the_c_abi's
            r = expected_route(B, L, E, nc, fam, d_emb=True, want=want)
            check_kernels(r, names, "bwd", r.get("products"))
            if fam == "tma":
                n2 = ("w_in" in want) or ("d_desc" in want)
                assert names.count("tgemm_pair_kernel") == 1 + n2, (want, names)
            else:
                n_gemm = 2 + sum(k in want for k in ("w_c", "w_out", "w_in", "d_desc"))
                assert sum(n.startswith(("umma<", "sgemm<")) for n in names) == n_gemm, (want, names)
                assert names.count("colsum_kernel") == sum(k in want for k in ("b_c", "b_out", "b_in")), (want, names)
            for k, t in zip(GRADS, leaves):
                if k in want:
                    close(npf(t.grad), gr[ORACLE_NAMES[k]], f"{k} {want}")
                else:
                    assert t.grad is None
    finally:
        ops.ATTN_IMPL = saved


LOGITS_ONLY = [("tma", 40, 3, 256, 4), ("ldg", 40, 3, 100, 100), ("ldg", 33, 2, 16, 17)]


@pytest.mark.parametrize("fam,B,L,E,nc", LOGITS_ONLY)
def test_loss_on_the_logits_only_through_the_c_abi(fam, B, L, E, nc):
    """d_emb NULL: gh_attn_head_bwd writes demb = d_logits W_c without accumulating, so at nc % 4 == 0 that product takes
    tcgen05 with K = nc (a K tail at nc = 100)."""
    desc, P, d_logits, _, f, g, r, _ = run_case(B, L, E, nc, fam, seed=5, with_d_emb=False)
    c = oracle_fwd(desc, P)
    gr = oracle_bwd(c, P, d_logits, None)
    for k in GRADS:
        close(npf(g[k]), gr[ORACLE_NAMES[k]], k, per_image=TOL_IMAGE if k == "d_desc" else None)


# ---- 4. launch options ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,L,E,nc", [(256, 3, 1024, 4), (100, 5, 576, 16)])
def test_tma_launch_options(B, L, E, nc):
    P = head_params(E, nc, 2)
    desc, d_logits, d_emb = inputs(B, L, E, nc, 2)
    c = oracle_fwd(desc, P)
    gr = oracle_bwd(c, P, d_logits, d_emb)
    for tn in (0, 128, 256):
        first = None
        for pdl in (0, 1, 1):
            with options(tn, pdl):
                plan = tgemm_plan(B * L, 3 * E, E)
                if tn and (3 * E) % tn == 0:
                    assert plan[0] == tn
                rc, f = fwd("tma", desc, P)
                assert rc == 0
                rc, g = bwd("tma", desc, P, f, d_logits, d_emb)
                assert rc == 0
                torch.cuda.synchronize()
            f["out"].check()
            if first is None:
                first = f
                close(npf(f["emb"]), c["emb"], f"emb tn={tn}")
                close(npf(f["logits"]), c["logits"], f"logits tn={tn}")
                close(npf(f["qkv"]).reshape(B, L, 3 * E), c["qkv"], f"qkv tn={tn}")
            else:
                for k in ("qkv", "probs", "emb", "logits", "x_planes", "obar_planes"):
                    assert torch.equal(f[k], first[k]), (k, tn, pdl)
            for k in GRADS:
                close(npf(g[k]), gr[ORACLE_NAMES[k]], f"{k} tn={tn} pdl={pdl}")


# ---- 5. large scores ------------------------------------------------------------------------------------------------
# probs vs a softmax of the kernel's own qkv, in fp64: the fp32 score carries ~|s| * 2^-24 of rounding, which moves a
# probability by as much at a near-tie; measured <= 2.2e-7, 7.9e-6, 4.1e-33 at 1e2, 1e4, 1e5 (at 1e5 every row is
# one-hot). Before attn2_core_bwd_kernel rounded dA / L once (no FMA contraction), d_desc on the TMA family was 8.9e-5 /
# 1.1e-3 off at 1e4 / 1e5: the gradient of a one-hot row, exactly 0, came out as the product's rounding error.
TOL_PROBS = {1e2: TOL, 1e4: TOL, 1e5: TOL}


def attention_given_probs(desc, P, probs):
    """The oracle's forward with the softmax replaced by `probs`."""
    c = oracle_fwd(desc, P)
    a = np.asarray(probs, np.float64)
    E = desc.shape[2]
    v = c["qkv"][..., 2 * E:]
    obar = np.einsum("blm,bme->ble", a, v).mean(axis=1)
    emb = obar @ npf(P[2]).astype(np.float64).T + npf(P[3])
    logits = emb @ npf(P[4]).astype(np.float64).T + npf(P[5])
    return dict(c, probs=a, obar=obar, emb=emb, logits=logits)


@pytest.mark.parametrize("fam,E", [("tma", 256), ("ldg", 100)])
@pytest.mark.parametrize("target", sorted(TOL_PROBS))
def test_large_scores(fam, E, target):
    B, L, nc = 64, 3, 4
    P = head_params(E, nc, 4)
    desc, d_logits, d_emb = inputs(B, L, E, nc, 4, scale=1.0)
    s1 = np.abs(np.einsum("ble,bme->blm", *np.split(oracle_fwd(desc, P)["qkv"], 3, axis=-1)[:2])).max() / math.sqrt(E)
    desc = desc * math.sqrt(target / s1)
    rc, f = fwd(fam, desc, P)
    assert rc == 0
    rc, g = bwd(fam, desc, P, f, d_logits, d_emb)
    assert rc == 0
    f["out"].check()
    c = oracle_fwd(desc, P)
    q, k, _ = np.split(c["qkv"], 3, axis=-1)
    print(f"  max |score| {np.abs(np.einsum('ble,bme->blm', q, k)).max() / math.sqrt(E):.3g}")
    qkv = npf(f["qkv"]).reshape(B, L, 3 * E)
    close(qkv, c["qkv"], "qkv")
    q, k, _ = np.split(qkv.astype(np.float64), 3, axis=-1)
    s = np.einsum("ble,bme->blm", q / math.sqrt(E), k)
    p = np.exp(s - s.max(axis=-1, keepdims=True))
    close(npf(f["probs"]), p / p.sum(axis=-1, keepdims=True), "probs vs softmax(own qkv)", TOL_PROBS[target])
    cp = attention_given_probs(desc, P, npf(f["probs"]))
    close(npf(f["emb"]), cp["emb"], "emb", per_image=TOL_IMAGE)
    close(npf(f["logits"]), cp["logits"], "logits", per_image=TOL_IMAGE)
    gr = oracle_bwd(cp, P, d_logits, d_emb)
    for kk in GRADS:
        close(npf(g[kk]), gr[ORACLE_NAMES[kk]], kk)


# ---- 6. dispatch from ops ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L,E,nc,impl", [(3, 256, 4, "tma"), (3, 100, 4, "tma"), (3, 1296, 4, "tma"), (3, 256, 17, "tma"),
                                         (5, 576, 16, "tma"), (3, 256, 4, "ldg")])
def test_ops_takes_the_modelled_family(ops, L, E, nc, impl):
    B = 6
    P = head_params(E, nc)
    desc, _, _ = inputs(B, L, E, nc)
    saved = ops.ATTN_IMPL
    try:
        ops.ATTN_IMPL = impl
        r = expected_route(B, L, E, nc, impl)
        (emb, logits), names = ran(lambda: ops.attention_head(desc, *P))
    finally:
        ops.ATTN_IMPL = saved
    check_kernels(r, names, "fwd", r.get("products"))
    c = oracle_fwd(desc, P)
    close(npf(emb), c["emb"], "emb")
    close(npf(logits), c["logits"], "logits")


# ---- 7. refusals ------------------------------------------------------------------------------------------------------
def test_nine_tokens_are_refused_and_write_nothing(ops):
    from heuristique_style_transfer_code_b200._lib import GramHeadError
    B, L, E, nc = 4, 9, 256, 4
    assert family(L, E, nc) == "unsupported"
    P = head_params(E, nc)
    desc, d_logits, d_emb = inputs(B, L, E, nc)
    for fam in ("tma", "ldg"):
        rc, f = fwd(fam, desc, P)
        assert rc == GH_ERR_UNSUPPORTED and f["out"].untouched(), fam
        out = Outputs()
        rc, _ = bwd(fam, desc, P, f, d_logits, d_emb, out=out)
        assert rc == GH_ERR_UNSUPPORTED and out.untouched(), fam
        saved = ops.ATTN_IMPL
        try:
            ops.ATTN_IMPL = fam
            with pytest.raises(GramHeadError):
                ops.attention_head(desc, *P)
        finally:
            ops.ATTN_IMPL = saved


@pytest.mark.parametrize("B,L,E,nc,why", [(4, 3, 100, 4, "E % 64"), (4, 3, 1088, 4, "E > 1024"), (4, 3, 256, 17, "nc > 16"),
                                          (4, 3, 32, 4, "E < 64"), (4, 9, 256, 4, "L > 8")])
def test_tma_entry_points_refuse_other_shapes(B, L, E, nc, why):
    P = head_params(E, nc)
    desc, d_logits, d_emb = inputs(B, L, E, nc)
    rc, f = fwd("tma", desc, P)
    assert rc == GH_ERR_UNSUPPORTED and f["out"].untouched(), why
    out = Outputs()
    rc, _ = bwd("tma", desc, P, f, d_logits, d_emb, out=out)
    assert rc == GH_ERR_UNSUPPORTED and out.untouched(), why


def test_tma_entry_points_check_alignment_before_writing():
    """Buffers the tensor maps or the float4 loads cannot take are refused before the first write: a misaligned x_planes
    (TMA), W_c (the classifier's float4 rows); backward, a misaligned d_desc (TMA store) or db_in (zeroed as float4)."""
    B, L, E, nc = 40, 3, 256, 4
    P = head_params(E, nc)
    desc, d_logits, d_emb = inputs(B, L, E, nc)
    # x_planes 8 B past a 16 B boundary; qkv for a plan that splits K (zeroed first): B * L rows at E = 1024 do
    for b_, e_ in ((B, E), (1, 1024)):
        Pp = head_params(e_, nc)
        dsc = inputs(b_, L, e_, nc)[0]
        out = Outputs()
        wp = (ops_split(Pp[0]), ops_split(Pp[2]))
        xp = out((2, b_ * L, e_), torch.bfloat16, "x_planes", offset=4)
        bufs = dict(qkv=out((b_ * L, 3 * e_)), probs=out((b_, L, L)), obar=out((2, b_, e_), torch.bfloat16),
                    emb=out((b_, e_)), logits=out((b_, nc)))
        rc = lib().gh_attn_head_fwd2(dsc.data_ptr(), wp[0].data_ptr(), Pp[1].data_ptr(), wp[1].data_ptr(),
                                     Pp[3].data_ptr(), Pp[4].data_ptr(), Pp[5].data_ptr(), b_, L, e_, nc, xp.data_ptr(),
                                     bufs["qkv"].data_ptr(), bufs["probs"].data_ptr(), bufs["obar"].data_ptr(),
                                     bufs["emb"].data_ptr(), bufs["logits"].data_ptr(), stream())
        assert rc == GH_ERR_UNSUPPORTED and out.untouched(), (b_, e_, tgemm_plan(b_ * L, 3 * e_, e_))
    wc = torch.empty(nc * E + 1, device="cuda")[1:].view(nc, E)
    wc.copy_(P[4])
    rc, f = fwd("tma", desc, P[:4] + [wc, P[5]])
    assert rc == GH_ERR_UNSUPPORTED and f["out"].untouched()
    rc, f = fwd("tma", desc, P)
    assert rc == 0
    torch.cuda.synchronize()
    for name in ("d_desc", "b_in"):
        out = Outputs()
        shapes = {"d_desc": (B, L, E), "w_in": (3 * E, E), "b_in": (3 * E,), "w_out": (E, E), "b_out": (E,),
                  "w_c": (nc, E), "b_c": (nc,)}
        g = {k: out(shapes[k], name=k, offset=1 if k == name else 0) for k in GRADS}
        ws = torch.empty(((lib().gh_attn_head_bwd2_workspace(B, L, E) + 15) // 16 * 4,), device="cuda")
        rc = lib().gh_attn_head_bwd2(f["x_planes"].data_ptr(), f["w_planes"][0].data_ptr(), f["w_planes"][1].data_ptr(),
                                     P[4].data_ptr(), f["qkv"].data_ptr(), f["probs"].data_ptr(),
                                     f["obar_planes"].data_ptr(), f["emb"].data_ptr(), d_logits.data_ptr(),
                                     d_emb.data_ptr(), B, L, E, nc, *[g[k].data_ptr() for k in GRADS], ws.data_ptr(),
                                     stream())
        assert rc == GH_ERR_UNSUPPORTED and out.untouched(), name


def ops_split(w):
    from heuristique_style_transfer_code_b200 import ops
    return ops.split_bf16(w)


def test_refused_split_plane_gemm_writes_nothing(ops):
    """gh_gemm_planes with an MN-major operand whose extent is not a multiple of 64, at a shape whose plan splits K:
    the refusal comes before the output is zeroed."""
    for a_mn, b_mn, M, N in ((True, False, 100, 64), (False, True, 128, 96)):
        K = 4096
        assert tgemm_plan(M, N, K, 64)[1] > 1
        a = ops.split_bf16(torch.randn((K, M) if a_mn else (M, K), device="cuda"))
        b = ops.split_bf16(torch.randn((K, N) if b_mn else (N, K), device="cuda"))
        out = Outputs()
        d = out((M, N))
        rc = lib().gh_gemm_planes(a.data_ptr(), a.shape[2], a[0].numel(), int(a_mn), b.data_ptr(), b.shape[2],
                                  b[0].numel(), int(b_mn), 0, d.data_ptr(), 0, N, M * N, M, N, K, 64, stream())
        assert rc == GH_ERR_UNSUPPORTED
        assert out.untouched(), "a refused call zeroed its output"


# ---- 8. the GEMMs beneath -------------------------------------------------------------------------------------------
def operand(rows, cols, layout, seed):
    """A (rows, cols) fp32 view: "r" rows contiguous (row pitch cols + pad), "c" columns contiguous, "off" rows
    contiguous one element past a 16 B boundary, "strided" no unit stride."""
    g = torch.Generator().manual_seed(seed)
    kind, _, pad = layout.partition("+")
    pad = int(pad or 0)
    if kind == "strided":
        return (torch.randn(2 * rows, 3 * cols, generator=g).cuda())[::2, ::3]
    if kind == "off":
        buf = torch.randn(rows * cols + 4, generator=g).cuda()
        return buf[1:1 + rows * cols].view(rows, cols)
    if kind == "r":
        return torch.randn(rows, cols + pad, generator=g).cuda()[:, :cols]
    return torch.randn(cols, rows + pad, generator=g).cuda()[:, :rows].t()


def gemm_call(entry, a, b, bias, ldd_pad=0):
    """D = a @ b (+ bias) into a guarded (M, N + ldd_pad) buffer -> (rc, D view, Outputs)."""
    M, K = a.shape
    N = b.shape[1]
    out = Outputs()
    full = out((M, N + ldd_pad), name="D")
    fn = getattr(lib(), entry)
    rc = fn(a.data_ptr(), a.stride(0), a.stride(1), b.data_ptr(), b.stride(0), b.stride(1),
            0 if bias is None else bias.data_ptr(), full.data_ptr(), N + ldd_pad, M, N, K, stream())
    return rc, full, out


# name, M, N, K, A layout, B layout (as a (K, N) view: "r" = N contiguous, "c" = K contiguous), bias, ldd - N
GEMM_CASES = [
    ("umma kk split bias vec", 128, 256, 2048, "r", "c", True, 0),
    ("umma kmn nosplit", 2048, 2560, 192, "r", "r", False, 4),
    ("umma mnk split bias scalar", 200, 300, 1000, "c", "c", True, 3),
    ("umma mnmn ktail", 256, 64, 100, "c", "r", True, 0),
    ("umma kk pitched scalar", 100, 130, 68, "r+4", "c+8", False, 1),
    ("sgemm TT K%4", 70, 80, 33, "r", "c", True, 0),
    ("sgemm TF N<64", 65, 63, 64, "r", "r", False, 2),
    ("sgemm FT K%4", 64, 100, 37, "c", "c", True, 0),
    ("sgemm FF strided", 50, 70, 40, "strided", "r", False, 0),
    ("sgemm misaligned", 128, 128, 64, "off", "c", True, 0),
    ("sgemm FF both strided", 33, 65, 17, "strided", "strided", True, 5),
]
TOL_GEMM = 2e-5       # measured <= 4.5e-6 (tcgen05, split-bf16 operands), <= 1.4e-7 (fp32 FMA)


def gemm_case_route(a, b, M, N, K):
    return gemm_route(a.stride(0), a.stride(1), b.stride(0), b.stride(1), M, N, K, a_ptr=a.data_ptr(), b_ptr=b.data_ptr())


@pytest.mark.parametrize("case", GEMM_CASES, ids=lambda c: c[0].replace(" ", "-"))
def test_gemm_f32_routes(case):
    name, M, N, K, la, lb, has_bias, ldd_pad = case
    a, b = operand(M, K, la, 1), operand(K, N, lb, 2)
    bias = torch.randn(N, generator=torch.Generator().manual_seed(N)).cuda() if has_bias else None
    route = gemm_case_route(a, b, M, N, K)
    assert route.split("<")[0] == name.split()[0], route
    (rc, d, out), names = ran(lambda: gemm_call("gh_gemm_f32", a, b, bias, ldd_pad))
    assert rc == 0 and not torch.isnan(d[:, :N]).any()
    assert [n for n in names if n != "memset"] == [route], names
    if route.startswith("umma"):
        split = umma_ksplit(M, N, K) > 1
        assert split == ("nosplit" not in name and "ktail" not in name and "pitched" not in name), umma_ksplit(M, N, K)
        assert ("memset" in names) == split
    out.check(allow_nan=("D",))
    assert torch.isnan(d[:, N:]).all(), "written beyond N inside the row pitch"
    ref = a.double() @ b.double() + (0 if bias is None else bias.double())
    close(npf(d[:, :N]), ref.cpu().numpy(), name, TOL_GEMM)


@pytest.mark.parametrize("M,N,K,la,lb", [(64, 64, 8192, "r", "c"), (128, 256, 6000, "c", "r"), (30, 40, 5000, "r", "r")])
def test_gemm_f32_fixed_is_reproducible(M, N, K, la, lb):
    """One output tile over a long K: gh_gemm_f32 splits K there (reduce-adds in any order), gh_gemm_f32_fixed does not."""
    a, b = operand(M, K, la, 3), operand(K, N, lb, 4)
    route = gemm_case_route(a, b, M, N, K)
    if route.startswith("umma"):
        assert umma_ksplit(M, N, K) > 1
    # one fp32 accumulator over the whole K (no partial sums): measured 2.8e-5 / 2.1e-5 at K = 8192 / 6000 on tcgen05,
    # 1.3e-6 on the FMA kernel; the result is the same bits on every run, so these are exact
    tol = 5e-5
    runs = []
    for _ in range(3):
        (rc, d, out), names = ran(lambda: gemm_call("gh_gemm_f32_fixed", a, b, None, 3))
        assert rc == 0 and names == [route], names      # no zeroing: one writer per output element
        out.check(allow_nan=("D",))
        assert torch.isnan(d[:, N:]).all() and not torch.isnan(d[:, :N]).any()
        runs.append(d[:, :N].clone())
    assert all(torch.equal(runs[0], r) for r in runs[1:])
    close(npf(runs[0]), (a.double() @ b.double()).cpu().numpy(), "fixed", tol)


@pytest.mark.parametrize("M,N,ldx", [(1, 1, 1), (7, 33, 40), (1000, 65, 67), (4097, 3, 3), (300, 1025, 1030)])
def test_colsum_ragged(M, N, ldx):
    x = torch.full((M, ldx), float("nan"), device="cuda")
    x[:, :N] = torch.randn(M, N, generator=torch.Generator().manual_seed(M)).cuda()
    out = Outputs()
    s = out((N,), name="colsum")
    assert lib().gh_colsum_f32(x.data_ptr(), ldx, M, N, s.data_ptr(), stream()) == 0
    out.check()
    # fp32 sums over up to 4097 rows, in eight interleaved partial sums: measured 2.1e-7 .. 7.1e-6 over random draws
    close(npf(s), npf(x[:, :N]).astype(np.float64).sum(axis=0), "colsum", TOL)


@pytest.mark.parametrize("n,pitch_pad", [(4, 0), (1020, 8), (1 << 20, 0), ("cap+", 4)])
def test_split_bf16_planes_bitwise(n, pitch_pad):
    """hi = bf16(x), lo = bf16(x - hi) on every bit pattern class (random finite words, RNE ties, subnormals), below and
    above the grid cap of SMs * 16 blocks (n = "cap+": one grid-stride trip more)."""
    if n == "cap+":
        n = sms() * 16 * 256 * 4 + 12
    g = torch.Generator().manual_seed(n)
    bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (n,), generator=g, dtype=torch.int64).to(torch.int32)
    bits[1::7] = (bits[1::7] & ~0xFFFF) | 0x8000                        # ties at the bf16 boundary
    x = bits.view(torch.float32)
    x[~torch.isfinite(x)] = 1.5
    x = x.cuda()
    out = Outputs()
    planes = out((2 * n + pitch_pad,), torch.bfloat16, "planes")
    assert lib().gh_split_bf16(x.data_ptr(), planes.data_ptr(), n, n + pitch_pad, stream()) == 0
    out.check(allow_nan=("planes",))
    hi = x.bfloat16()
    lo = (x - hi.float()).bfloat16()
    assert torch.equal(planes[:n].view(torch.int16), hi.view(torch.int16))
    assert torch.equal(planes[n + pitch_pad:2 * n + pitch_pad].view(torch.int16), lo.view(torch.int16))
    assert torch.isnan(planes[n:n + pitch_pad]).all()


# ---- 9. coverage ------------------------------------------------------------------------------------------------------
ROUTE_TABLE = (
    {("family", f) for f in ("tma", "ldg", "unsupported")}
    | {(f, "LT", t) for f in ("tma", "ldg") for t in (4, 8)}
    | {("tma", gemm, tn, ks) for gemm in ("in_proj", "out_proj") for tn in (128, 256) for ks in (1, 2)}
    | {("tma", "prep_trips", 1), ("tma", "prep_trips", 2), ("tma", "core_bwd", "single"), ("tma", "core_bwd", "persistent")}
    | {("ldg", p, k) for p in ("in_proj", "out_proj") for k in ("umma<false,false>", "sgemm<true,true>")}
    | {("ldg", p, k) for p in ("demb", "dobar", "d_desc") for k in ("umma<false,true>", "sgemm<true,false>")}
    | {("ldg", p, k) for p in ("dW_out", "dW_in") for k in ("umma<true,true>", "sgemm<false,false>")}
    | {("ldg", "dW_c", k) for k in ("umma<true,true>", "sgemm<false,false>", "sgemm<true,false>")}
    | {("gemm", k) for k in ("umma<false,false>", "umma<false,true>", "umma<true,false>", "umma<true,true>",
                              "sgemm<true,true>", "sgemm<true,false>", "sgemm<false,true>", "sgemm<false,false>")}
)


def test_every_route_is_reached():
    """Each cell is declared by at least one case above, and each case asserts its route from expected_route() and from
    the kernels that ran. The demb product reaches tcgen05 only without an embedding gradient (LOGITS_ONLY)."""
    reached = set()
    for B, L, E, nc, impl, fam in HEAD_CASES:
        reached |= route_cells(expected_route(batch(B), L, E, nc, impl))
    for loss in ("both", "emb", "logits"):
        for fam, B, L, E, nc in (("tma", 40, 3, 256, 4), ("ldg", 40, 3, 100, 100)):
            for want in SUBSETS:
                reached |= route_cells(expected_route(B, L, E, nc, fam, want=want))
    for fam, B, L, E, nc in LOGITS_ONLY:
        reached |= route_cells(expected_route(B, L, E, nc, fam, d_emb=False))
    reached |= route_cells(expected_route(4, 9, 256, 4))
    for name, M, N, K, la, lb, _, _ in GEMM_CASES:
        reached.add(("gemm", gemm_case_route(operand(M, K, la, 1), operand(K, N, lb, 2), M, N, K)))
    print("reached:", sorted(map(str, reached)))
    assert reached == ROUTE_TABLE, (sorted(map(str, ROUTE_TABLE - reached)), sorted(map(str, reached - ROUTE_TABLE)))
