"""The C-ABI shared library loads on a CPU-only machine and exports exactly what include/gramhead.h declares.
No compute call is made here (argument validation returns before any CUDA API is touched)."""
import ctypes
import os
import re

import pytest

from conftest import ROOT
from heuristique_style_transfer_code_b200 import _lib
from heuristique_style_transfer_code_b200.build import build_library


DEFAULT_BWD_ATS = -1      # gramhead.cu: g_opt_bwd_ats (the option state lives in the loaded library, i.e. in the process)


@pytest.fixture(scope="module")
def library():
    build_library()
    return _lib.lib()


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "gramhead.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gh_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree():
    assert declared_symbols() == sorted(_lib.EXPORTED_SYMBOLS)


def test_every_declared_symbol_is_exported(library):
    for name in declared_symbols():
        assert hasattr(library, name), name


def test_version(library):
    assert library.gh_version() >= 100


def test_argument_validation_without_gpu(library):
    assert library.gh_gram_pool_fwd(None, 0, 0, 0, 1, 1, 256, 64, 32, None, 0, 1, 0, 0, None) == _lib.GH_ERR_BAD_ARG
    assert library.gh_gram_dense_fwd(None, 0, 0, 0, 1, 1, 256, 64, None, 0, 0, None) == _lib.GH_ERR_BAD_ARG
    assert library.gh_attn_head_fwd(*([None] * 7), 1, 3, 64, 4, *([None] * 5), None) == _lib.GH_ERR_BAD_ARG
    assert library.gh_gram_pool_bwd(None, 0, 0, 0, 1, 1, 256, 64, 32, None, 0, 1, None, 0, 0, 0, 1, 0, None) == _lib.GH_ERR_BAD_ARG
    dummy = ctypes.c_void_p(16)
    # non-power-of-two pooling factor and oversize g are refused before any launch
    assert library.gh_gram_pool_fwd(dummy, 0, 96 * 64, 64, 1, 1, 96, 64, 32, dummy, 0, 1, 0, 0, None) == _lib.GH_ERR_UNSUPPORTED
    assert library.gh_gram_pool_fwd(dummy, 0, 100 * 64, 64, 1, 1, 100, 64, 32, dummy, 0, 1, 0, 0, None) == _lib.GH_ERR_UNSUPPORTED
    assert library.gh_gram_pool_fwd(dummy, 7, 256 * 64, 64, 1, 1, 256, 64, 32, dummy, 0, 1, 0, 0, None) == _lib.GH_ERR_BAD_ARG
    assert library.gh_gram_pool_fwd(dummy, 0, 128 * 64, 64, 1, 1, 128, 64, 32, dummy, 0, 1, 0, 0, None) == _lib.GH_ERR_UNSUPPORTED   # k = 4
    # a layout that is neither x-contiguous nor c-contiguous is refused
    assert library.gh_gram_pool_fwd(dummy, 0, 256 * 64 * 2, 128, 2, 1, 256, 64, 32, dummy, 0, 1, 0, 0, None) == _lib.GH_ERR_BAD_ARG
    assert library.gh_set_option(b"no_such_option", 1) == _lib.GH_ERR_BAD_ARG
    assert library.gh_set_option(b"gram_bwd_ch", 3) == _lib.GH_ERR_BAD_ARG
    # retired knobs are unknown names now, even with the value that used to be their default
    for name, value in ((b"gram_fwd_producer_warps", 0), (b"gram_fwd_epilogue_warps", 0), (b"gram_bwd_variant", 2),
                        (b"gram_bwd_nhw", 0), (b"gram_bwd_producer_warps", 8), (b"tma_f32_type", 1), (b"attn_gemm", 1)):
        assert library.gh_set_option(name, value) == _lib.GH_ERR_BAD_ARG, name
    assert library.gh_attn_head_bwd_workspace(4, 3, 64) == 2 * 4 * 64 + 3 * 4 * 3 * 64
    # Multi-PatchGAN head and inference-plan entries
    assert library.gh_patch_gram_workspace(6, 256, 64) == 6 * 256 * 64 * 20
    assert library.gh_patch_gram_fwd(None, None, None, None, 1, 1, 64, 1, None, None, None, None) == _lib.GH_ERR_BAD_ARG
    ptrs = (ctypes.c_void_p * 9)(*([16] * 9))
    hw = (ctypes.c_int * 9)(*([4] * 9))
    st = (ctypes.c_longlong * 36)(*([1] * 36))
    assert library.gh_patch_gram_fwd(ptrs, hw, hw, st, 9, 1, 64, 1, dummy, dummy, dummy, None) == _lib.GH_ERR_UNSUPPORTED   # > 8 layers
    assert library.gh_patch_gram_fwd(ptrs, hw, hw, st, 2, 1, 160, 1, dummy, dummy, dummy, None) == _lib.GH_ERR_UNSUPPORTED  # D > 128
    assert library.gh_patch_attn_fwd(*([None] * 11), 4, 2, 64, 8, 3, None, None, None) == _lib.GH_ERR_BAD_ARG
    assert library.gh_patch_attn_fwd(*([dummy] * 11), 4, 2, 60, 8, 3, dummy, dummy, None) == _lib.GH_ERR_BAD_ARG            # E % heads
    assert library.gh_patch_attn_fwd(*([dummy] * 11), 4, 2, 256, 8, 3, dummy, dummy, None) == _lib.GH_ERR_UNSUPPORTED       # E > 128
    assert library.gh_maxpool2d_nhwc(None, 0, None, 1, 8, 8, 64, 3, 2, 1, None) == _lib.GH_ERR_BAD_ARG
    assert library.gh_maxpool2d_nhwc(dummy, 0, dummy, 1, 8, 8, 6, 3, 2, 1, None) == _lib.GH_ERR_UNSUPPORTED                  # C % 4
    assert library.gh_maxpool2d_nhwc(dummy, 0, dummy, 1, 8, 8, 64, 3, 2, 2, None) == _lib.GH_ERR_BAD_ARG                     # pad > k/2
    assert library.gh_stem_space_to_depth(None, 1, 1, 1, 1, 1, 8, 8, None, 0, None) == _lib.GH_ERR_BAD_ARG
    assert library.gh_stem_space_to_depth(dummy, 1, 1, 1, 1, 1, 7, 8, dummy, 0, None) == _lib.GH_ERR_UNSUPPORTED             # odd H
    three = ctypes.c_float * 3
    mean, std = three(0.485, 0.456, 0.406), three(0.229, 0.224, 0.225)
    assert library.gh_normalize_u8(None, None, 1, 3, 16, mean, std, None) == _lib.GH_ERR_BAD_ARG
    assert library.gh_normalize_u8(dummy, dummy, 1, 3, 16, None, std, None) == _lib.GH_ERR_BAD_ARG
    assert library.gh_normalize_u8(dummy, dummy, 0, 3, 16, mean, std, None) == _lib.GH_ERR_BAD_ARG                           # no images
    assert library.gh_normalize_u8(dummy, dummy, 1, 5, 16, mean, std, None) == _lib.GH_ERR_UNSUPPORTED                       # > 4 channels
    assert library.gh_normalize_u8(dummy, dummy, 1, 3, 16, mean, three(0.229, 0.0, 0.225), None) == _lib.GH_ERR_BAD_ARG      # zero std


def test_option_validation_and_environment_hook(monkeypatch, library):
    """gh_set_option refuses values outside each knob's set; GRAMHEAD_OPTIONS applies knobs when the library is loaded and
    fails loudly on anything it cannot apply (a silently ignored knob would make a measurement lie)."""
    for value, want in ((-1, 0), (1, 0), (0, 0), (2, _lib.GH_ERR_BAD_ARG), (-2, _lib.GH_ERR_BAD_ARG)):
        assert library.gh_set_option(b"gram_bwd_ats", value) == want
    assert library.gh_set_option(b"gram_bwd_nt", 100) == _lib.GH_ERR_BAD_ARG         # not a multiple of 16
    assert library.gh_set_option(b"gram_bwd_nt", 224) == 0 and library.gh_set_option(b"gram_bwd_nt", 0) == 0
    monkeypatch.setattr(_lib, "_LIB", None)
    monkeypatch.setenv("GRAMHEAD_OPTIONS", "gram_bwd_ats=1, gram_bwd_nt=0")
    _lib.lib()
    for bad in ("gram_bwd_ats", "gram_bwd_ats=x", "no_such_option=1", "gram_bwd_ats=7"):
        monkeypatch.setattr(_lib, "_LIB", None)
        monkeypatch.setenv("GRAMHEAD_OPTIONS", bad)
        with pytest.raises(_lib.GramHeadError, match="GRAMHEAD_OPTIONS"):
            _lib.lib()
    monkeypatch.delenv("GRAMHEAD_OPTIONS")
    monkeypatch.setattr(_lib, "_LIB", None)
    assert _lib.lib().gh_set_option(b"gram_bwd_ats", DEFAULT_BWD_ATS) == 0           # back to the shipped default


def test_gram_backward_planner_host_logic(library):
    """gh_gram_bwd_plan (no GPU needed): x-tile width, ring depths and the tensor-memory form of the pooled Gram backward.
    Invariants for every shape: TMEM columns <= 512, ring bytes <= 9 tiles of 16 KB, A stages >= the generator groups'
    stage lanes (4 / chunks per stage), at least two F stages, tiles cover HW."""
    import ctypes

    def plan(C, HW, g=32, dtype=_lib.GH_DTYPE_F32, cl=1):
        out = (ctypes.c_int * 8)()
        assert library.gh_gram_bwd_plan(C, HW, g, dtype, cl, out) == 0
        return dict(zip(("NT", "nHT", "ats", "ch", "a_stages", "b_stages", "tmem_cols", "ring_bytes"), out))

    # the three ResNet stages at 224 x 224, fp32 channels_last (the default hand-off)
    s1, s2, s3 = plan(256, 3136), plan(512, 784), plan(1024, 196)
    assert (s1["NT"], s1["nHT"], s1["ats"], s1["ch"]) == (224, 14, 0, 1)        # HBM-bound stage: shared-memory form
    assert (s2["NT"], s2["nHT"], s2["ats"], s2["ch"], s2["a_stages"]) == (160, 5, 1, 2, 6)
    assert (s3["NT"], s3["nHT"], s3["ats"], s3["ch"], s3["a_stages"]) == (208, 1, 1, 2, 4)
    # bf16 features: twice the TMEM columns per chunk (no k-step reuse at pooling factor 16)
    b2 = plan(512, 784, dtype=_lib.GH_DTYPE_BF16)
    assert (b2["ats"], b2["ch"], b2["a_stages"]) == (1, 2, 3)
    for C in (64, 256, 512, 1024, 2048):
        for HW in (49, 64, 100, 196, 784, 3136, 12544):
            for dtype in (_lib.GH_DTYPE_F32, _lib.GH_DTYPE_BF16):
                for cl in (0, 1):
                    for g in (8, 32):
                        if C // g < 8:
                            continue
                        p = plan(C, HW, g, dtype, cl)
                        assert 64 <= p["NT"] <= 256 and p["NT"] % 16 == 0 and p["NT"] * p["nHT"] >= HW
                        assert p["tmem_cols"] <= 512 and p["ring_bytes"] <= 9 * 16384 and p["b_stages"] >= 2
                        assert p["ch"] in (1, 2) and p["a_stages"] >= max(2, 4 // p["ch"])
                        assert p["ats"] == 1 or (p["ch"] == 1 and p["tmem_cols"] == 0)
                        assert p["ats"] == 0 or C >= 512                               # default: tensor-memory form for C >= 512
    try:      # the knobs reach the plan
        assert library.gh_set_option(b"gram_bwd_ats", 0) == 0
        assert plan(512, 784)["ats"] == 0
        assert library.gh_set_option(b"gram_bwd_ats", 1) == 0 and library.gh_set_option(b"gram_bwd_ch", 1) == 0
        p = plan(512, 784)
        assert (p["ats"], p["ch"], p["a_stages"]) == (1, 1, 8)
        assert plan(256, 128)["ats"] == 1                                              # small maps leave TMEM for the A ring
        assert library.gh_set_option(b"gram_bwd_nt", 224) == 0
        assert plan(512, 784)["nHT"] == 4
    finally:
        library.gh_set_option(b"gram_bwd_ats", DEFAULT_BWD_ATS)
        library.gh_set_option(b"gram_bwd_ch", 0)
        library.gh_set_option(b"gram_bwd_nt", 0)
    out = (ctypes.c_int * 8)()
    assert library.gh_gram_bwd_plan(100, 784, 32, 0, 1, out) == _lib.GH_ERR_UNSUPPORTED      # C % g
    assert library.gh_gram_bwd_plan(128, 784, 32, 0, 1, out) == _lib.GH_ERR_UNSUPPORTED      # pooling factor 4
    assert library.gh_gram_bwd_plan(512, 784, 32, 0, 1, None) == _lib.GH_ERR_BAD_ARG


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    monkeypatch.setenv("GRAMHEAD_LIB", str(tmp_path / "nope.so"))
    monkeypatch.setattr(_lib, "_LIB", None)
    with pytest.raises(_lib.GramHeadError, match="no CPU or PyTorch fallback"):
        _lib.lib()


def test_tgemm_planner_host_logic(library):
    """gh_tgemm_plan (no GPU needed): the tiling of the attention GEMMs. The forward never splits K in more than two
    partitions (bitwise reproducibility), big problems fill the 74 CTA pairs of a B200 in whole rounds, small ones are split
    to use the machine, and a partition keeps at least two 64-wide k-blocks."""
    import ctypes

    def plan(M, N, K, max_split, pairs=74):
        tn, ks, units = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        assert library.gh_tgemm_plan(M, N, K, max_split, pairs, ctypes.byref(tn), ctypes.byref(ks), ctypes.byref(units)) == 0
        return tn.value, ks.value, units.value

    # in_proj at batch 512 (B*L = 1536 rows): one 256 x 256 unit per pair, unsplit
    assert plan(1536, 3072, 1024, 2) == (256, 1, 72)
    # in_proj at batch 256: 36 wide tiles would leave half the pairs idle -> 72 narrow, unsplit units
    tn, ks, units = plan(768, 3072, 1024, 2)
    assert (tn, ks, units) == (128, 1, 72)
    # out_proj (M = batch): forward limit of two partitions is respected
    tn, ks, units = plan(512, 1024, 1024, 2)
    assert ks <= 2 and tn in (128, 256) and units >= 16
    # backward problems may split freely, but a partition keeps >= 2 k-blocks
    for (M, N, K) in [(3072, 1024, 1536), (1536, 1024, 3072), (512, 1024, 1024), (1024, 1024, 512), (192, 1024, 3072)]:
        tn, ks, units = plan(M, N, K, 64)
        assert tn in (128, 256) and 1 <= ks <= (K + 63) // 64 // 2 and units == ((M + 255) // 256) * ((N + tn - 1) // tn) * ks
    # tiny problems: a single unit, never more partitions than k-blocks allow
    assert plan(8, 64, 64, 64) == (256, 1, 1) or plan(8, 64, 64, 64)[1] == 1
    assert library.gh_tgemm_plan(0, 64, 64, 1, 74, None, None, None) == _lib.GH_ERR_BAD_ARG
