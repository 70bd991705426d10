"""The uint8 fused stem (gh_stem_conv_pool_u8_nhwc: ToTensor + Normalize inside the stem kernel's producers) and
set_input_normalization, all bit for bit: the kernel against normalize_u8 followed by the fp32 fused stem, the model on
every execution path against the same model fed normalize_u8's batch, and the evaluation loop against the fp32 loop."""
import copy

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

IMAGENET = ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))
OTHER = ((-0.75, 0.5, 0.0), (0.3, 1.7, 0.05))                 # a negative mean, a zero mean, a small std
CONSTANTS = {"imagenet": IMAGENET, "other": OTHER}


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
    return p


def _pixels(b, h, w, seed):
    """uint8 (b, 3, h, w) with every byte value in every channel where the channel has 256 pixels."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randint(0, 256, (b, 3, h, w), dtype=torch.uint8, generator=g)
    n = min(256, b * h * w)
    for c in range(3):
        plane = x[:, c].reshape(-1).clone()
        plane[:n] = (torch.arange(n) * (2 * c + 1) + 17 * c) % 256      # a permutation of 0..255 when n = 256
        x[:, c] = plane.view(b, h, w)
    return x.cuda()


def _u8(p, x, consts):
    from heuristique_style_transfer_code_b200 import ops
    return ops.stem_conv_pool_u8(x, *consts, p.stem_packed, p.stem_s2d[1])


def _fp32(p, x, consts):
    from heuristique_style_transfer_code_b200 import ops
    return ops.stem_conv_pool(ops.normalize_u8(x, *consts), p.stem_packed, p.stem_s2d[1])


@pytest.mark.parametrize("consts", ["imagenet", "other"])
@pytest.mark.parametrize("b,h,w", [(1, 224, 224), (3, 224, 192), (3, 36, 52), (1, 448, 448), (2, 2, 4), (64, 224, 224)])
def test_u8_stem_equals_normalize_u8_then_the_fp32_stem(plan, b, h, w, consts):
    x = _pixels(b, h, w, b * h + w)
    if b * h * w >= 256:
        for c in range(3):
            assert torch.unique(x[:, c]).numel() == 256
    got, want = _u8(plan, x, CONSTANTS[consts]), _fp32(plan, x, CONSTANTS[consts])
    assert got.shape == want.shape and got.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(got, want)


@pytest.mark.parametrize("layout", ["nchw", "channels_last", "odd_row_stride", "odd_address"])
def test_u8_stem_input_layouts(plan, layout):
    b, h, w = 3, 36, 52
    x = _pixels(b, h, w, 5)
    if layout == "channels_last":
        x = x.contiguous(memory_format=torch.channels_last)
    elif layout != "nchw":                                  # strided views: the byte-load path
        big = _pixels(b, h + 2, w + (3 if layout == "odd_row_stride" else 4), 6)
        big[:, :, 1:h + 1, 1:w + 1] = x
        x = big[:, :, 1:h + 1, 1:w + 1]
        assert (x.stride(2) % 2 == 1) if layout == "odd_row_stride" else (x.data_ptr() % 2 == 1)
    for consts in (IMAGENET, OTHER):
        assert torch.equal(_u8(plan, x, consts), _fp32(plan, x.contiguous(), consts))


def test_u8_stem_result_of_an_image_does_not_depend_on_its_batch(plan):
    x = _pixels(256, 224, 224, 13)
    full = _u8(plan, x, IMAGENET)
    for i in range(256):
        assert torch.equal(full[i:i + 1], _u8(plan, x[i:i + 1], IMAGENET)), i


def _model_outputs_equal(m, x, consts):
    from heuristique_style_transfer_code_b200 import ops
    with torch.no_grad():
        m.set_input_normalization(None)
        want = m(ops.normalize_u8(x, *consts))
        m.set_input_normalization(*consts)
        got = m(x)
    assert len(got) == len(want) == 2
    for g, w in zip(got, want):
        assert g.shape == w.shape and torch.equal(g, w)


@pytest.mark.parametrize("mode,tf32,fold", [("channels_last", True, True), ("channels_last", False, True),
                                            ("bf16_channels_last", True, True), ("reference", True, True),
                                            ("channels_last", True, False)])
def test_model_on_uint8_input_equals_the_model_on_the_normalised_batch(mode, tf32, fold):
    m = _model(mode)
    m.fold_batchnorm = fold
    x = _pixels(6, 64, 64, 21)
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = tf32
    try:
        for consts in (IMAGENET, OTHER):
            _model_outputs_equal(m, x, consts)
    finally:
        torch.backends.cudnn.allow_tf32 = old


def test_train_mode_forward_on_uint8_input():
    """A gradient-enabled train-mode forward feeds conv1 exactly normalize_u8's batch. Its outputs are compared within
    a tolerance: the train-mode forward (batch-norm batch statistics) is not bitwise reproducible from run to run even
    on identical input and with cudnn.deterministic, so the bits of two runs say nothing about the input."""
    from heuristique_style_transfer_code_b200 import ops
    m = _model().train()
    a, b = copy.deepcopy(m), copy.deepcopy(m)
    a.set_input_normalization(*IMAGENET)
    x = _pixels(6, 64, 64, 22)
    seen = []
    hooks = [c.truncated_encoder[0].register_forward_pre_hook(lambda mod, args: seen.append(args[0].detach().clone()))
             for c in (a, b)]
    old = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        got = a(x)
        want = b(ops.normalize_u8(x, *IMAGENET))
    finally:
        torch.backends.cudnn.deterministic = old
        for h in hooks:
            h.remove()
    assert len(seen) == 2 and seen[0].dtype == torch.float32 and torch.equal(seen[0], seen[1])
    assert got[1].requires_grad
    for g, w in zip(got, want):
        assert float((g - w).norm() / w.norm()) <= 1e-4


@pytest.mark.parametrize("mode,tf32,fold,norm,fused", [
    ("channels_last", True, True, True, True),
    ("channels_last", False, True, True, False),
    ("bf16_channels_last", True, True, True, False),
    ("reference", True, True, True, False),
    ("channels_last", True, False, True, False),
    ("channels_last", True, True, False, False),            # not set: uint8 input runs as before, untransformed
])
def test_path_selection(mode, tf32, fold, norm, fused):
    from heuristique_style_transfer_code_b200 import ops
    m = _model(mode)
    m.fold_batchnorm = fold
    if norm:
        m.set_input_normalization(*IMAGENET)
    x = _pixels(2, 224, 224, 23)
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
    assert ("stem_conv_pool_u8[HW=224x224]" in names) == fused
    assert any(n.startswith("normalize_u8") for n in names) == (norm and not fused)
    assert not any(n.startswith("stem_conv_pool[") for n in names)


def test_evaluation_loop_hands_uint8_pixels_to_a_self_normalising_model():
    """evaluate_model_test over a uint8 loader, with the model normalising its input, returns exactly what the default
    uint8 loop (normalize_u8 in cuda_prefetch) and the fp32 loop (host-normalised batches) return."""
    from torch.utils.data import DataLoader, Dataset
    from heuristique_style_transfer_code_b200 import functions as F, ops

    class Pixels(Dataset):
        def __init__(self, normalised):
            g = torch.Generator().manual_seed(12)
            self.x = torch.randint(0, 256, (15, 3, 64, 64), dtype=torch.uint8, generator=g)
            if normalised:
                self.x = F._normalize_host(self.x, F.IMAGENET_MEAN, F.IMAGENET_STD)
            self.y = torch.arange(15) % 4
            self.samples = [(f"img_{i}.png", int(self.y[i])) for i in range(15)]

        def __len__(self):
            return 15

        def __getitem__(self, i):
            return self.x[i], self.y[i]

    m = _model()
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = True                   # the fused stem's condition
    try:
        u8 = F.evaluate_model_test(m, DataLoader(Pixels(False), batch_size=6, shuffle=False), "cuda")
        fp32 = F.evaluate_model_test(m, DataLoader(Pixels(True), batch_size=6, shuffle=False), "cuda")
        m.set_input_normalization(F.IMAGENET_MEAN, F.IMAGENET_STD)
        ops.PROFILE = []
        inside = F.evaluate_model_test(m, DataLoader(Pixels(False), batch_size=6, shuffle=False), "cuda")
        names = [r[0] for r in ops.PROFILE]
    finally:
        ops.PROFILE = None
        torch.backends.cudnn.allow_tf32 = old
    assert names.count("stem_conv_pool_u8[HW=64x64]") == 3 and not any(n.startswith("normalize_u8") for n in names)
    assert inside[0].shape == (15, 1024) and inside[4] == u8[4] == fp32[4]
    for a, b, c in zip(inside[:4], u8[:4], fp32[:4]):
        assert np.array_equal(a, b) and np.array_equal(a, c)
