"""Fused stem shapes at the edges of its tiling and of its epilogue's row carry: a last tile that holds a single pooled
column (W = 256), and an odd number of conv rows (H = 226), whose last pooling window has no third row and takes its first
row from the previous window's registers. Enough images that every CTA computes several consecutive pooled rows, fp32
against the fp64 model and uint8 bit for bit against normalize_u8 followed by the fp32 kernel."""
import numpy as np
import pytest
import torch

from oracle import head_fp64 as O
from oracle.stem_fp64 import stem_fp64

pytestmark = pytest.mark.gpu

ORACLE_TOL = 2e-5          # normwise, fused vs fp64 on the same tf32 operands
IMAGENET = ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))
SHAPES = [(4, 36, 256), (4, 226, 256), (3, 226, 130)]


def npf(t):
    return t.detach().float().cpu().numpy()


@pytest.fixture(scope="module")
def plan():
    from torchvision import models
    from heuristique_style_transfer_code_b200 import TruncatedResNet50_for_test
    from heuristique_style_transfer_code_b200.frozen_encoder import _fold
    torch.manual_seed(0)
    m = TruncatedResNet50_for_test(models.resnet50(weights=None), 7, 4, 32, device="cuda").eval()
    with torch.no_grad():                                    # non-trivial folded bn1
        bn = m.truncated_encoder[1]
        bn.running_mean.uniform_(-0.5, 0.5)
        bn.running_var.uniform_(0.5, 2.0)
        bn.weight.uniform_(0.5, 1.5)
        bn.bias.uniform_(-0.5, 0.5)
    m.set_backbone_mode("channels_last")
    with torch.no_grad():
        p = m._inference_plan(torch.zeros(1, 3, 32, 32, device="cuda"))
    assert p is not None and p.stem_packed is not None
    w, b, *_ = _fold(m.truncated_encoder[0], m.truncated_encoder[1], torch.float32, False)
    return p, npf(w), npf(b)


@pytest.mark.parametrize("b,h,w", SHAPES)
def test_fused_stem_edges_match_the_fp64_model(plan, b, h, w):
    from heuristique_style_transfer_code_b200 import ops
    p, wt, bias = plan
    torch.manual_seed(b * h + w)
    x = torch.randn(b, 3, h, w, device="cuda")
    out = ops.stem_conv_pool(x, p.stem_packed, p.stem_s2d[1])
    assert out.shape == (b, 64, (h // 2 - 1) // 2 + 1, (w // 2 - 1) // 2 + 1)
    err = O.rel_err(npf(out), stem_fp64(npf(x), wt, bias))
    print(f"fused vs fp64 model at {b}x{h}x{w}: {err:.3g}")
    assert err <= ORACLE_TOL


@pytest.mark.parametrize("b,h,w", SHAPES)
def test_uint8_stem_edges_equal_normalize_then_fp32_stem(plan, b, h, w):
    from heuristique_style_transfer_code_b200 import ops
    p, _, _ = plan
    torch.manual_seed(b + h + w)
    x = torch.randint(0, 256, (b, 3, h, w), dtype=torch.uint8, device="cuda")
    got = ops.stem_conv_pool_u8(x, *IMAGENET, p.stem_packed, p.stem_s2d[1])
    want = ops.stem_conv_pool(ops.normalize_u8(x, *IMAGENET), p.stem_packed, p.stem_s2d[1])
    assert torch.equal(got, want)
    assert np.isfinite(npf(got)).all()
