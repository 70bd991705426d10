"""set_input_normalization on a CPU machine: the API and its validation, no state_dict change, the host transform on
CPU models, and the loops handing uint8 pixels to a model that normalises them itself."""
import copy

import pytest
import torch
import torch.nn as nn
from torchvision import models

from heuristique_style_transfer_code_b200 import TruncatedResNet50, TruncatedResNet50_for_test
from heuristique_style_transfer_code_b200 import functions as F

MEAN, STD = F.IMAGENET_MEAN, F.IMAGENET_STD


def _model(cls=TruncatedResNet50_for_test, trunc=5):
    torch.manual_seed(0)
    return cls(models.resnet50(weights=None), trunc, 4, 8, device="cpu").eval()


@pytest.mark.parametrize("cls", [TruncatedResNet50, TruncatedResNet50_for_test])
def test_set_and_unset(cls):
    m = _model(cls, trunc=4)
    assert m.input_normalization is None
    assert m.set_input_normalization(MEAN, STD) is m
    assert m.input_normalization == (tuple(MEAN), tuple(STD))
    assert m.set_input_normalization([0.5, -0.25, 1], torch.tensor([2.0, 0.5, 1.0])) is m
    assert m.input_normalization == ((0.5, -0.25, 1.0), (2.0, 0.5, 1.0))
    assert m.set_input_normalization(None) is m and m.input_normalization is None
    with pytest.raises(AttributeError):
        m.input_normalization = (MEAN, STD)


@pytest.mark.parametrize("mean,std", [((0.5, 0.5), (0.2, 0.2, 0.2)), ((0.5, 0.5, 0.5), (0.2, 0.2, 0.2, 0.2)),
                                      ((0.5, 0.5, 0.5), (0.2, 0.0, 0.2)), ((0.5, 0.5, 0.5), (0.2, float("nan"), 0.2)),
                                      (None, (0.2, 0.2, 0.2))])
def test_invalid_normalisation_is_rejected_and_leaves_the_setting(mean, std):
    m = _model(trunc=4).set_input_normalization(MEAN, STD)
    with pytest.raises(ValueError):
        m.set_input_normalization(mean, std)
    assert m.input_normalization == (tuple(MEAN), tuple(STD))


def test_state_dict_keys_and_values_are_unchanged():
    a, b = _model(trunc=5), _model(trunc=5).set_input_normalization(MEAN, STD)
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb)
    assert all(torch.equal(sa[k], sb[k]) for k in sa)
    assert len(list(b.buffers())) == len(list(a.buffers()))
    c = copy.deepcopy(b)
    assert c.input_normalization == b.input_normalization
    a.load_state_dict(sb)
    assert a.input_normalization is None


def test_cpu_model_normalises_uint8_input_like_the_host_transforms():
    m = _model(trunc=5)
    assert m.backbone_mode == "reference"
    g = torch.Generator().manual_seed(3)
    x = torch.randint(0, 256, (2, 3, 32, 40), dtype=torch.uint8, generator=g)
    x.view(-1)[:256] = torch.arange(256, dtype=torch.int64).to(torch.uint8)
    mean, std = (0.3, -0.2, 0.6), (0.2, 0.5, 1.5)
    with torch.no_grad():
        want_last, want_stages = m._stage_activations(F._normalize_host(x, mean, std))
        m.set_input_normalization(mean, std)
        got_last, got_stages = m._stage_activations(x)
        assert torch.equal(got_last, want_last) and len(got_stages) == len(want_stages) == 1
        assert torch.equal(got_stages[0], want_stages[0])
        # fp32 input is untouched by the setting
        xf = F._normalize_host(x, mean, std)
        assert torch.equal(m._stage_activations(xf)[0], want_last)


class _Stub(nn.Module):
    """Stands in for the model classes in the loops: records the dtype it is fed."""

    def __init__(self, norm, returns_embeddings):
        super().__init__()
        self.lin = nn.Linear(2, 4)
        self.returns_embeddings = returns_embeddings
        self.seen = []
        if norm:
            self.input_normalization = (MEAN, STD)

    def forward(self, x):
        self.seen.append(x.dtype)
        emb = x.float().flatten(1)[:, :2]
        return (emb, self.lin(emb)) if self.returns_embeddings else self.lin(emb)


class _Wrapper(nn.Module):
    """The attribute layout of DistributedDataParallel: the model under `.module`."""

    def __init__(self, module):
        super().__init__()
        self.module = module

    def forward(self, x):
        return self.module(x)


class _Pixels(torch.utils.data.Dataset):
    def __init__(self):
        self.x = torch.randint(0, 256, (4, 3, 4, 4), dtype=torch.uint8, generator=torch.Generator().manual_seed(1))
        self.y = torch.arange(4) % 4
        self.samples = [(f"img_{i}.png", int(self.y[i])) for i in range(4)]

    def __len__(self):
        return 4

    def __getitem__(self, i):
        return self.x[i], self.y[i]


@pytest.mark.parametrize("wrapped", [False, True])
@pytest.mark.parametrize("norm", [False, True])
def test_loops_hand_uint8_pixels_to_a_self_normalising_model(monkeypatch, norm, wrapped):
    calls = []
    real = F.cuda_prefetch

    def spy(batches, device, **kw):
        calls.append(kw.get("normalize", "default"))
        return real(batches, device, **kw)

    monkeypatch.setattr(F, "cuda_prefetch", spy)
    monkeypatch.setattr(F, "_default_device", lambda: torch.device("cpu"))
    loader = torch.utils.data.DataLoader(_Pixels(), batch_size=2, shuffle=False)
    crit = nn.CrossEntropyLoss()

    def model(returns_embeddings):
        stub = _Stub(norm, returns_embeddings)
        return (_Wrapper(stub) if wrapped else stub), stub

    m, stub = model(False)
    F.train_model(m, loader, crit, torch.optim.SGD(m.parameters(), lr=0.1), num_epochs=1)
    m2, stub2 = model(False)
    F.evaluate_model(m2, loader, crit)
    m3, stub3 = model(True)
    F.evaluate_model_test(m3, loader, "cpu")
    want = None if norm else "default"
    assert calls == [want] * 3
    dtype = torch.uint8 if norm else torch.float32
    assert stub.seen == stub2.seen == stub3.seen == [dtype] * 2
