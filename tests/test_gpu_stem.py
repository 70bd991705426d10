"""The fused stem of the inference plan (gh_stem_conv_pool_nhwc: conv1 + folded bn1 + relu + maxpool in one tcgen05
kernel with tf32 operands) against the fp64 model of the same arithmetic, against the three-launch chain it replaces
(space-to-depth staging, cuDNN convolution, max pool), and against the unfolded children for NaN / -inf pixels."""
import numpy as np
import pytest
import torch

from oracle import head_fp64 as O
from oracle.stem_fp64 import stem_fp64

pytestmark = pytest.mark.gpu

ORACLE_TOL = 2e-5          # normwise, fused vs fp64 on the same tf32 operands


def npf(t):
    return t.detach().float().cpu().numpy()


def _model(mode="channels_last"):
    from torchvision import models
    from heuristique_style_transfer_code_b200 import TruncatedResNet50_for_test
    torch.manual_seed(0)
    m = TruncatedResNet50_for_test(models.resnet50(weights=None), 7, 4, 32, device="cuda").eval()
    with torch.no_grad():                                    # non-trivial folded bn1
        bn = m.truncated_encoder[1]
        bn.running_mean.uniform_(-0.5, 0.5)
        bn.running_var.uniform_(0.5, 2.0)
        bn.weight.uniform_(0.5, 1.5)
        bn.bias.uniform_(-0.5, 0.5)
    m.set_backbone_mode(mode)
    return m


@pytest.fixture(scope="module")
def plan():
    m = _model()
    with torch.no_grad():
        p = m._inference_plan(torch.zeros(1, 3, 32, 32, device="cuda"))
    assert p is not None and p.stem_packed is not None
    return m, p


def _folded_conv(m):
    from heuristique_style_transfer_code_b200.frozen_encoder import _fold
    w, b, *_ = _fold(m.truncated_encoder[0], m.truncated_encoder[1], torch.float32, False)
    return npf(w), npf(b)


def _fused(p, x):
    from heuristique_style_transfer_code_b200 import ops
    return ops.stem_conv_pool(x, p.stem_packed, p.stem_s2d[1])


def _chain(p, x, tf32):
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = tf32
    p._stem_fused = False
    try:
        with torch.no_grad():
            return p.stem_forward(x)
    finally:
        p._stem_fused = True
        torch.backends.cudnn.allow_tf32 = old


@pytest.mark.parametrize("b,h,w", [(1, 224, 224), (3, 224, 192), (3, 36, 52), (1, 448, 448), (2, 2, 4)])
def test_fused_stem_matches_the_fp64_model(plan, b, h, w):
    m, p = plan
    torch.manual_seed(b * h + w)
    x = torch.randn(b, 3, h, w, device="cuda")
    out = _fused(p, x)
    oh, ow = h // 2, w // 2
    assert out.shape == (b, 64, (oh - 1) // 2 + 1, (ow - 1) // 2 + 1)
    assert out.dtype == torch.float32 and out.is_contiguous(memory_format=torch.channels_last)
    wt, bias = _folded_conv(m)
    want = stem_fp64(npf(x), wt, bias)
    err = O.rel_err(npf(out), want)
    print(f"fused vs fp64 model at {b}x{h}x{w}: {err:.3g}")
    assert err <= ORACLE_TOL


@pytest.mark.parametrize("layout", ["nchw", "channels_last", "strided"])
def test_fused_stem_input_layouts(plan, layout):
    m, p = plan
    torch.manual_seed(3)
    b, h, w = 3, 36, 52
    x = torch.randn(b, 3, h, w, device="cuda")
    if layout == "channels_last":
        x = x.contiguous(memory_format=torch.channels_last)
    elif layout == "strided":
        big = torch.randn(b, 3, h + 2, w + 3, device="cuda")
        big[:, :, 1:h + 1, 1:w + 1] = x
        x = big[:, :, 1:h + 1, 1:w + 1]                      # odd offsets: the scalar-load path
    wt, bias = _folded_conv(m)
    assert O.rel_err(npf(_fused(p, x)), stem_fp64(npf(x), wt, bias)) <= ORACLE_TOL


@pytest.mark.parametrize("b,h,w", [(64, 224, 224), (3, 224, 192), (3, 36, 52), (1, 448, 448)])
def test_fused_stem_matches_the_chain(plan, b, h, w):
    _, p = plan
    torch.manual_seed(7)
    x = torch.randn(b, 3, h, w, device="cuda")
    out = npf(_fused(p, x))
    for tf32 in (True, False):
        ref = _chain(p, x, tf32)
        assert ref.shape == out.shape
        err = O.rel_err(out, npf(ref))
        print(f"fused vs chain (tf32={tf32}) at {b}x{h}x{w}: {err:.3g}")
        assert err <= 1e-3


def test_fused_stem_nan_and_inf_pixels(plan):
    """NaN and -inf pixels land where the unfolded children put them. At an odd (row, column) a pixel meets only the
    real 7x7 taps; at an even one the space-to-depth form also meets a zero tap (0 * NaN, 0 * inf = NaN), exactly as
    the chain it replaces does, so there the fused kernel is compared with the chain."""
    m, p = plan
    torch.manual_seed(11)
    x = torch.randn(2, 3, 64, 48, device="cuda")
    x[0, 1, 21, 13] = float("nan")
    x[1, 0, 5, 33] = float("-inf")
    x[1, 2, 41, 1] = float("nan")
    with torch.no_grad():
        children = m.truncated_encoder[3](m.truncated_encoder[2](m.truncated_encoder[1](m.truncated_encoder[0](x))))
        out = _fused(p, x)
    assert torch.equal(torch.isnan(out), torch.isnan(children)) and torch.isnan(out).any()
    assert torch.equal(torch.isinf(out), torch.isinf(children)) and torch.isinf(out).any()
    fin = torch.isfinite(children)
    assert O.rel_err(npf(out[fin]), npf(children[fin])) <= 1e-3
    x[0, 0, 30, 20] = float("nan")
    x[1, 1, 8, 12] = float("-inf")
    out = _fused(p, x)
    ref = _chain(p, x, True)
    assert torch.equal(torch.isnan(out), torch.isnan(ref)) and torch.equal(torch.isinf(out), torch.isinf(ref))


def test_fused_stem_result_of_an_image_does_not_depend_on_its_batch(plan):
    _, p = plan
    torch.manual_seed(13)
    x = torch.randn(256, 3, 224, 224, device="cuda")
    full = _fused(p, x)
    for i in range(256):
        assert torch.equal(full[i:i + 1], _fused(p, x[i:i + 1])), i


@pytest.mark.parametrize("mode,tf32,fused", [("channels_last", True, True), ("channels_last", False, False),
                                             ("bf16_channels_last", True, False)])
def test_inference_plan_selects_the_stem(mode, tf32, fused):
    from heuristique_style_transfer_code_b200 import ops
    m = _model(mode)
    x = torch.randn(2, 3, 224, 224, device="cuda")
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = tf32
    ops.PROFILE = []
    try:
        with torch.no_grad():
            m(x)
        names = [r[0] for r in ops.PROFILE]
    finally:
        ops.PROFILE = None
        torch.backends.cudnn.allow_tf32 = old
    assert any(n.startswith("stem_conv_pool[HW=224x224]") for n in names) == fused
    assert any(n.startswith("stem_space_to_depth") for n in names) != fused
    assert any(n.startswith("maxpool2d_nhwc") for n in names) != fused
