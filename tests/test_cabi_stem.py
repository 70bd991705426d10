"""C-ABI argument checks of gh_stem_conv_pool_nhwc on a CPU-only machine: validation returns before any CUDA API is
touched."""
import pytest

from heuristique_style_transfer_code_b200 import _lib
from heuristique_style_transfer_code_b200.build import build_library


@pytest.fixture(scope="module")
def library():
    build_library()
    return _lib.lib()


def test_stem_conv_pool_argument_checks(library):
    f = library.gh_stem_conv_pool_nhwc
    d = 4096                                                  # 16 B aligned, never dereferenced
    assert f(None, 1, 1, 1, 1, 1, 8, 8, d, d, d, None) == _lib.GH_ERR_BAD_ARG                     # no image
    assert f(d, 1, 1, 1, 1, 1, 8, 8, None, d, d, None) == _lib.GH_ERR_BAD_ARG                     # no weights
    assert f(d, 1, 1, 1, 1, 1, 8, 8, d, None, d, None) == _lib.GH_ERR_BAD_ARG                     # no bias
    assert f(d, 1, 1, 1, 1, 1, 8, 8, d, d, None, None) == _lib.GH_ERR_BAD_ARG                     # no output
    assert f(d, 1, 1, 1, 1, 0, 8, 8, d, d, d, None) == _lib.GH_ERR_BAD_ARG                        # no images
    assert f(d, 1, 1, 1, 1, 1, 7, 8, d, d, d, None) == _lib.GH_ERR_UNSUPPORTED                    # odd H
    assert f(d, 1, 1, 1, 1, 1, 8, 9, d, d, d, None) == _lib.GH_ERR_UNSUPPORTED                    # odd W
    assert f(d, 1, 1, 1, 1, 1, 8, 8, d, d, d + 4, None) == _lib.GH_ERR_UNSUPPORTED                # misaligned output
    assert f(d, 1, 1, 1, 1, 1, 8, 8, d + 8, d, d, None) == _lib.GH_ERR_UNSUPPORTED                # misaligned weights
