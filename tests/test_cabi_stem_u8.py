"""C-ABI argument checks of gh_stem_conv_pool_u8_nhwc on a CPU-only machine: every rejection returns before any CUDA
API is touched (the pointers below are never dereferenced on the device)."""
import ctypes

import pytest

from heuristique_style_transfer_code_b200 import _lib
from heuristique_style_transfer_code_b200.build import build_library

BAD, UNSUP = _lib.GH_ERR_BAD_ARG, _lib.GH_ERR_UNSUPPORTED
F3 = ctypes.c_float * 3


@pytest.fixture(scope="module")
def library():
    build_library()
    return _lib.lib()


def _call(library, x=4096, b=1, h=8, w=8, mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225), wp=4096, bias=4096,
          out=4096):
    m = F3(*mean) if mean is not None else None
    s = F3(*std) if std is not None else None
    return library.gh_stem_conv_pool_u8_nhwc(x, 3 * h * w, h * w, w, 1, b, h, w, m, s, wp, bias, out, None)


@pytest.mark.parametrize("kw", [dict(x=None), dict(mean=None), dict(std=None), dict(wp=None), dict(bias=None),
                                dict(out=None), dict(b=0), dict(b=-1), dict(h=0), dict(w=-2)],
                         ids=["no image", "no mean", "no std", "no weights", "no bias", "no output", "no images",
                              "negative batch", "zero height", "negative width"])
def test_null_pointers_and_sizes_are_bad_arguments(library, kw):
    assert _call(library, **kw) == BAD


@pytest.mark.parametrize("std", [(0.229, 0.0, 0.225), (-0.0, 0.224, 0.225), (0.229, 0.224, float("nan"))],
                         ids=["zero", "negative zero", "nan"])
def test_zero_or_nan_std_is_a_bad_argument(library, std):
    assert _call(library, std=std) == BAD


def test_a_std_check_comes_before_the_shape_checks(library):
    assert _call(library, std=(0.0, 1.0, 1.0), h=7, out=4100) == BAD


@pytest.mark.parametrize("kw", [dict(h=7), dict(w=9), dict(out=4100), dict(wp=4104)],
                         ids=["odd H", "odd W", "misaligned output", "misaligned weights"])
def test_unsupported_shapes_and_alignments(library, kw):
    assert _call(library, **kw) == UNSUP
