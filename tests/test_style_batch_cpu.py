"""style_transfer's images_per_step and the per-image style loss entry points, without a GPU: the signature, the
argument and environment checks, and the C-ABI validation (which returns before any CUDA call)."""
import ctypes
import inspect

import pytest
import torch

from heuristique_style_transfer_code_b200 import _lib
from heuristique_style_transfer_code_b200 import functions as F
from heuristique_style_transfer_code_b200.build import build_library


def test_images_per_step_is_a_trailing_keyword_defaulting_to_the_environment():
    params = list(inspect.signature(F.style_transfer).parameters.values())
    assert params[-1].name == "images_per_step" and params[-1].default is None


def test_images_per_step_resolution(monkeypatch):
    monkeypatch.delenv("GRAMHEAD_STYLE_IMAGES", raising=False)
    assert F._style_images_per_step(None, "cpu") == 1
    assert F._style_images_per_step(1, "cpu") == 1
    assert F._style_images_per_step(8, "cuda:0") == 8
    assert F._style_images_per_step(8, torch.device("cuda", 1)) == 8
    monkeypatch.setenv("GRAMHEAD_STYLE_IMAGES", " 16 ")
    assert F._style_images_per_step(None, "cuda") == 16
    assert F._style_images_per_step(2, "cuda") == 2           # an explicit value wins over the variable
    monkeypatch.setenv("GRAMHEAD_STYLE_IMAGES", "")
    assert F._style_images_per_step(None, "cpu") == 1
    monkeypatch.setenv("GRAMHEAD_STYLE_IMAGES", "1")
    assert F._style_images_per_step(None, "cpu") == 1


@pytest.mark.parametrize("value,env,device", [(0, None, "cuda"), (-3, None, "cuda"), (2, None, "cpu"),
                                              (None, "0", "cuda"), (None, "four", "cuda"), (None, "2", "cpu"),
                                              (None, "1.5", "cuda")])
def test_images_per_step_refusals(monkeypatch, value, env, device):
    if env is None:
        monkeypatch.delenv("GRAMHEAD_STYLE_IMAGES", raising=False)
    else:
        monkeypatch.setenv("GRAMHEAD_STYLE_IMAGES", env)
    with pytest.raises(ValueError):
        F._style_images_per_step(value, device)


def test_style_transfer_refuses_before_any_work(tmp_path, monkeypatch):
    monkeypatch.delenv("GRAMHEAD_STYLE_IMAGES", raising=False)
    with pytest.raises(ValueError):
        F.style_transfer(None, [], "cpu", str(tmp_path), images_per_step=2)
    with pytest.raises(ValueError):
        F.style_transfer(None, [], "cpu", str(tmp_path), images_per_step=0)
    assert list(tmp_path.iterdir()) == []


def test_per_image_loss_argument_validation_without_gpu():
    build_library()
    lib = _lib.lib()
    dummy = ctypes.c_void_p(16)
    assert lib.gh_gram_mse_images_blocks(0) == 0
    assert lib.gh_gram_mse_images_blocks(-4) == 0
    assert lib.gh_gram_mse_images(None, dummy, 1, 16, dummy, dummy, None) == _lib.GH_ERR_BAD_ARG
    assert lib.gh_gram_mse_images(dummy, dummy, 1, 16, dummy, None, None) == _lib.GH_ERR_BAD_ARG
    assert lib.gh_gram_mse_images(dummy, dummy, 0, 16, dummy, dummy, None) == _lib.GH_ERR_BAD_ARG        # no images
    assert lib.gh_gram_mse_images(dummy, dummy, 2, 0, dummy, dummy, None) == _lib.GH_ERR_BAD_ARG         # n_img <= 0
    assert lib.gh_gram_mse_images(dummy, dummy, 65536, 16, dummy, dummy, None) == _lib.GH_ERR_UNSUPPORTED  # gridDim.y
