"""CPU: the fp64 model of the fused stem (oracle/stem_fp64.py) against torch fp64 conv2d -> relu -> max_pool2d, and
the tf32 B-operand packing of the inference plan against the space-to-depth weights it packs. No GPU needed."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import head_fp64 as O
from oracle.stem_fp64 import stem_fp64


def _torch_fp64(x, w, bias):
    y = F.conv2d(torch.from_numpy(x).double(), torch.from_numpy(w).double(), torch.from_numpy(bias).double(), 2, 3)
    return F.max_pool2d(F.relu(y), 3, 2, 1).numpy()


@pytest.mark.parametrize("shape", [(2, 3, 16, 16), (1, 3, 36, 52), (2, 3, 30, 22), (1, 3, 2, 4)])
def test_stem_oracle_is_torch_fp64_on_rounded_operands(shape):
    rng = np.random.default_rng(sum(shape))
    x = rng.standard_normal(shape).astype(np.float32)
    w = (rng.standard_normal((64, 3, 7, 7)) * 0.1).astype(np.float32)
    bias = rng.standard_normal(64).astype(np.float32)
    got = stem_fp64(x, w, bias, round_operands=False)
    want = _torch_fp64(x, w, bias)
    assert got.shape == want.shape
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
    rounded = stem_fp64(x, w, bias)
    np.testing.assert_allclose(rounded, _torch_fp64(O.tf32_round(x), O.tf32_round(w), bias), rtol=1e-12, atol=1e-12)


def test_stem_oracle_propagates_nan_through_relu_and_pool():
    rng = np.random.default_rng(5)
    x = rng.standard_normal((1, 3, 16, 16)).astype(np.float32)
    x[0, 1, 5, 7] = np.nan
    w = (rng.standard_normal((64, 3, 7, 7)) * 0.1).astype(np.float32)
    bias = np.zeros(64, np.float32)
    got = stem_fp64(x, w, bias, round_operands=False)
    want = _torch_fp64(x, w, bias)
    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.isnan(got).any()


def test_packed_stem_weights_are_the_rounded_space_to_depth_taps():
    from heuristique_style_transfer_code_b200.frozen_encoder import _stem_space_to_depth_weight, pack_stem_weight
    torch.manual_seed(0)
    w = torch.randn(64, 3, 7, 7)
    w16 = _stem_space_to_depth_weight(w)
    packed = pack_stem_weight(w16).view(4, 4, 2, 2, 64, 4)
    ref16 = O.tf32_round(w16.contiguous().numpy())
    for a in range(4):
        for b in range(4):
            for h in range(2):
                for q in range(2):
                    assert np.array_equal(packed[a, b, h, q].numpy(), ref16[:, (2 * h + q) * 4:(2 * h + q) * 4 + 4, a, b])
