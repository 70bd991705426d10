"""Drop-in contract of the module and functions files, checked on CPU (no kernel runs here)."""
import inspect
import json
import os

import pytest
import torch
from torchvision import models

from heuristique_style_transfer_code_b200 import TruncatedResNet50, TruncatedResNet50_for_test
from heuristique_style_transfer_code_b200 import functions as F
from heuristique_style_transfer_code_b200._lib import GramHeadError
from oracle.ref_loader import reference_available, load_reference_models, load_reference_functions

HEAD_KEYS = ["classifier.weight", "classifier.bias", "attention.in_proj_weight", "attention.in_proj_bias",
             "attention.out_proj.weight", "attention.out_proj.bias"]


def build(cls=TruncatedResNet50, trunc=7, nc=4, g=32, seed=0):
    torch.manual_seed(seed)
    return cls(models.resnet50(weights=None), trunc, nc, g)


def test_reference_module_paths_resolve_to_the_b200_classes():
    from Models.Models_RESNET50_TRUNCATE_GRAM_with_Attention import TruncatedResNet50 as A, TruncatedResNet50_for_test as B
    import functions.functions_RESNET50_Truncate_Gram_Attention as fn
    assert A is TruncatedResNet50 and B is TruncatedResNet50_for_test
    for name in ("load_model", "set_parameter_requires_grad", "train_model", "save_model_weights", "evaluate_model",
                 "run_camera", "style_transfer", "load_hyperparameters", "load_model_weights", "evaluate_model_test",
                 "perform_tsne", "plot_tsne_interactive"):
        assert callable(getattr(fn, name)), name


def test_constructor_signature_attributes_and_state_dict():
    for cls in (TruncatedResNet50, TruncatedResNet50_for_test):
        params = list(inspect.signature(cls.__init__).parameters)
        assert params == ["self", "base_encoder", "truncate_after_layer", "num_classes", "gram_matrix_size", "device"]
        assert inspect.signature(cls.__init__).parameters["device"].default == "cpu"
    m = build()
    assert m.device == "cpu" and m.num_classes == 4 and m.gram_matrix_size == 32
    assert isinstance(m.truncated_encoder, torch.nn.Sequential) and len(m.truncated_encoder) == 7
    assert isinstance(m.attention, torch.nn.MultiheadAttention) and isinstance(m.classifier, torch.nn.Linear)
    sd = m.state_dict()
    assert len(sd) == 264
    assert [k for k in sd if not k.startswith("truncated_encoder.")] == HEAD_KEYS
    assert sd["attention.in_proj_weight"].shape == (3 * 1024, 1024)
    assert sd["attention.out_proj.weight"].shape == (1024, 1024)
    assert sd["classifier.weight"].shape == (4, 1024)
    assert sum(p.numel() for p in m.parameters()) == 12_745_796       # SURVEY section 8(a) a1


@pytest.mark.parametrize("name", ["TruncatedResNet50", "TruncatedResNet50_for_test"])
def test_identical_random_init_and_keys_as_reference(name, golden_resnet):
    """Seeded construction against the reference: always against what tests/golden/make_golden.py recorded from its
    TruncatedResNet50_for_test (the head parameters' checksum and the activations its encoder produced, which pin every
    encoder weight), and against the live reference classes when a checkout of the reference is available. Both
    classes here build their submodules in the same order, so the one recording serves both."""
    import hashlib
    from oracle import head_fp64 as O
    d = golden_resnet
    m = build(TruncatedResNet50 if name == "TruncatedResNet50" else TruncatedResNet50_for_test).train()
    head = dict(in_proj_weight=m.attention.in_proj_weight, in_proj_bias=m.attention.in_proj_bias,
                out_proj_weight=m.attention.out_proj.weight, out_proj_bias=m.attention.out_proj.bias,
                classifier_weight=m.classifier.weight, classifier_bias=m.classifier.bias)
    h = hashlib.sha256()
    for k in sorted(head):
        h.update(head[k].detach().numpy().tobytes())
    assert h.hexdigest() == str(d["params_sha256"])
    torch.manual_seed(1)
    x = torch.randn(2, 3, 64, 64)
    with torch.no_grad():
        for i, block in enumerate(m.truncated_encoder):
            x = block(x)
            if i >= 4:
                assert O.rel_err(x.numpy(), d[f"stage{i - 4}"]) <= 1e-6, i
    if not reference_available():
        return
    ref = load_reference_models()
    torch.manual_seed(0)
    a = getattr(ref, name)(models.resnet50(weights=None), 7, 4, 32)
    b = build(TruncatedResNet50 if name == "TruncatedResNet50" else TruncatedResNet50_for_test)
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb)
    assert all(torch.equal(sa[k], sb[k]) for k in sa)
    assert [n for n, _ in a.named_parameters()] == [n for n, _ in b.named_parameters()]


def test_forward_without_cuda_fails_loudly_instead_of_falling_back():
    m = build(trunc=5, g=8)
    with pytest.raises(GramHeadError, match="no CPU path"):
        m(torch.randn(1, 3, 32, 32))
    with pytest.raises(GramHeadError):
        m.gram_matrix(torch.randn(1, 8, 4, 4))


def test_zero_stage_early_return_matches_reference_semantics():
    m = build(trunc=4, nc=3, g=8)
    out = m(torch.randn(2, 3, 32, 32))
    assert out.shape == (2, 3) and float(out.abs().sum()) == 0.0
    t = build(TruncatedResNet50_for_test, trunc=4, nc=3, g=8)
    out = t(torch.randn(2, 3, 32, 32))
    assert isinstance(out, torch.Tensor) and out.shape == (2, 3)
    with pytest.raises(IndexError):
        build(trunc=3, g=8)(torch.randn(1, 3, 32, 32))


def test_importing_does_not_enable_anomaly_mode():
    assert not torch.is_anomaly_enabled()


def test_checkpoint_functions_roundtrip_and_fallback(tmp_path, capsys):
    m = build(TruncatedResNet50_for_test, trunc=5, g=8)
    path = str(tmp_path / "best_model_fold_0.pth")
    F.save_model_weights(m, path)
    blob = torch.load(path)
    assert sorted(blob) == ["attention", "classifier", "truncated_encoder"]
    other = build(TruncatedResNet50_for_test, trunc=5, g=8, seed=7)
    F.load_model_weights(other, path)
    assert all(torch.equal(v, other.state_dict()[k]) for k, v in m.state_dict().items())
    # flat-prefix checkpoint -> second strategy
    flat = str(tmp_path / "flat.pth")
    torch.save(m.state_dict(), flat)
    third = build(TruncatedResNet50_for_test, trunc=5, g=8, seed=9)
    F.load_model_weights(third, flat)
    out = capsys.readouterr().out
    assert "Warning: 'truncated_encoder' not found" in out
    # the reference's direct method "succeeds" on a flat dict without loading anything (all three sections absent)
    assert not torch.equal(third.state_dict()["classifier.weight"], m.state_dict()["classifier.weight"])
    F.load_model_weights(third, str(tmp_path / "missing.pth"))
    assert "No weights file found" in capsys.readouterr().out


def test_load_model_remaps_bare_encoder_keys(tmp_path):
    m = build(trunc=5, g=8)
    donor = build(trunc=5, g=8, seed=3)
    bare = {k: v for k, v in donor.truncated_encoder.state_dict().items()}
    bare["fc.weight"] = torch.zeros(3)                      # ignored
    bare["layer9.bogus"] = torch.zeros(1)                   # unknown keys are dropped silently
    path = str(tmp_path / "encoder.pth")
    torch.save(bare, path)
    before = m.classifier.weight.clone()
    F.load_model(m, path, "cpu")
    assert torch.equal(m.truncated_encoder[0].weight, donor.truncated_encoder[0].weight)
    assert torch.equal(m.classifier.weight, before)
    with pytest.raises(FileNotFoundError):
        F.load_model(m, str(tmp_path / "nope.pth"), "cpu")


def test_set_parameter_requires_grad():
    m = build(trunc=5, g=8)
    F.set_parameter_requires_grad(m, True)
    for n, p in m.named_parameters():
        assert p.requires_grad == (("classifier" in n) or ("attention" in n)), n
    F.set_parameter_requires_grad(m, False)
    assert all(p.requires_grad for p in m.parameters())


def test_load_hyperparameters(tmp_path):
    assert F.load_hyperparameters(str(tmp_path / "none.json")) is None
    cfg = dict(hidden_dims=[256], num_layers=2, batch_size=8, lr=1e-3, truncate_layer=7, gram_matrix_size=32)
    path = tmp_path / "cfg.json"
    path.write_text(json.dumps(cfg))
    assert F.load_hyperparameters(str(path)) == cfg


def test_denormalize_inplace():
    t = torch.zeros(3, 2, 2)
    out = F.denormalize(t, torch.tensor([1.0, 2.0, 3.0]), torch.tensor([0.5, 0.5, 0.5]))
    assert out is t and torch.equal(t[:, 0, 0], torch.tensor([1.0, 2.0, 3.0]))


@pytest.mark.skipif(not reference_available(), reason="needs a checkout of the reference project (GH_REFERENCE_ROOT)")
def test_function_signatures_match_reference():
    ref = load_reference_functions()
    for name in ("load_model", "save_model_weights", "load_model_weights", "train_model", "evaluate_model",
                 "evaluate_model_test", "set_parameter_requires_grad", "denormalize",
                 "load_hyperparameters", "perform_tsne", "plot_tsne_interactive", "create_onpick_function"):
        a = inspect.signature(getattr(ref, name))
        b = inspect.signature(getattr(F, name))
        assert list(a.parameters.items()) == list(b.parameters.items()), name
    for name in ("run_camera", "style_transfer"):            # additions are trailing keyword arguments with defaults
        a = list(inspect.signature(getattr(ref, name)).parameters.items())
        b = list(inspect.signature(getattr(F, name)).parameters.items())
        assert b[:len(a)] == a, name
        assert all(p.default is not inspect.Parameter.empty for _, p in b[len(a):]), name


def test_loops_run_with_a_cpu_stand_in_model(tmp_path):
    """train_model / evaluate_model / evaluate_model_test drive any module with the same forward contract; a CPU
    stand-in (the oracle's port) exercises the host-side loop logic without a GPU."""
    from oracle.torch_port import PortModel
    from torch.utils.data import Dataset, DataLoader

    class Fake(Dataset):
        def __init__(self):
            g = torch.Generator().manual_seed(0)
            self.x = torch.randn(6, 3, 32, 32, generator=g)
            self.y = torch.tensor([0, 1, 2, 0, 1, 2])
            self.samples = [(f"img_{i}.png", int(self.y[i])) for i in range(6)]

        def __len__(self):
            return 6

        def __getitem__(self, i):
            return self.x[i], self.y[i]

    if torch.cuda.is_available():
        pytest.skip("loop uses cuda when present; covered by the GPU integration test")
    torch.manual_seed(0)
    base = models.resnet50(weights=None)
    model = PortModel(base, 5, 3, 8)
    loader = DataLoader(Fake(), batch_size=4, shuffle=False)
    opt = torch.optim.SGD(model.parameters(), lr=1e-3, momentum=0.9)
    crit = torch.nn.CrossEntropyLoss()
    F.train_model(model, loader, crit, opt, num_epochs=1)
    loss, acc, prec, rec = F.evaluate_model(model, loader, crit)
    assert loss > 0 and 0 <= acc <= 1
    tester = PortModel(base, 5, 3, 8, return_embeddings=True)
    emb, preds, labels, probs, paths = F.evaluate_model_test(tester, loader, "cpu")
    assert emb.shape == (6, 64) and probs.shape == (6, 3) and len(paths) == 6 and paths[4] == "img_4.png"


def test_cuda_prefetch_passes_batches_through_in_order_on_cpu():
    import torch
    from heuristique_style_transfer_code_b200.functions import cuda_prefetch
    batches = [(torch.full((2, 3), float(i)), torch.tensor([i, i])) for i in range(5)]
    out = list(cuda_prefetch(iter(batches), "cpu"))
    assert len(out) == 5
    for i, (x, y) in enumerate(out):
        assert torch.equal(x, batches[i][0]) and torch.equal(y, batches[i][1])
    assert list(cuda_prefetch(iter([]), "cpu")) == []


def test_backbone_mode_defaults_and_validation(monkeypatch):
    from torchvision import models
    from heuristique_style_transfer_code_b200.modules import BACKBONE_MODES
    monkeypatch.delenv("GRAMHEAD_BACKBONE", raising=False)
    m = TruncatedResNet50(models.resnet50(weights=None), 5, 4, 8, device="cpu")
    assert m.backbone_mode == "reference"                 # CPU construction keeps the reference's NCHW execution
    assert set(BACKBONE_MODES) == {"reference", "channels_last", "bf16", "bf16_channels_last"}
    keys_before = list(m.state_dict())
    m.set_backbone_mode("channels_last")
    assert m.backbone_mode == "channels_last" and list(m.state_dict()) == keys_before
    with pytest.raises(ValueError):
        m.set_backbone_mode("int8")
    monkeypatch.setenv("GRAMHEAD_BACKBONE", "bf16")
    assert TruncatedResNet50(models.resnet50(weights=None), 5, 4, 8, device="cpu").backbone_mode == "bf16"


def test_inference_plan_is_off_without_cuda_and_never_changes_the_state_dict(monkeypatch):
    monkeypatch.delenv("GRAMHEAD_FOLD_BN", raising=False)
    m = build(trunc=5, g=8).eval()
    assert m.fold_batchnorm is True and m._plan is None
    keys = list(m.state_dict())
    with torch.no_grad():
        assert m._inference_plan(torch.randn(1, 3, 32, 32)) is None        # CPU tensor: children run one by one
    m.set_backbone_mode("channels_last")
    with torch.no_grad():
        assert m._inference_plan(torch.randn(1, 3, 32, 32)) is None
    assert list(m.state_dict()) == keys and not any(k.startswith("_plan") for k in keys)
    from heuristique_style_transfer_code_b200.frozen_encoder import FoldedEncoder, encoder_signature
    assert FoldedEncoder.supported(m.truncated_encoder)
    sig = encoder_signature(m.truncated_encoder)
    with torch.no_grad():
        m.truncated_encoder[1].weight.mul_(2.0)
    assert encoder_signature(m.truncated_encoder) != sig                   # in-place edits are seen
    assert not FoldedEncoder.supported(torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3), torch.nn.ReLU()))
    monkeypatch.setenv("GRAMHEAD_FOLD_BN", "0")
    assert build(trunc=5, g=8).fold_batchnorm is False


def test_host_collector_and_buffer_reusing_prefetch_on_cpu():
    from heuristique_style_transfer_code_b200.functions import HostCollector, cuda_prefetch
    c = HostCollector(depth=2)
    for i in range(5):
        c.push(torch.full((3, 2), float(i)), torch.tensor([i]))
    out = c.finish()
    assert [float(a[0, 0]) for a, _ in out] == [0.0, 1.0, 2.0, 3.0, 4.0] and [int(b[0]) for _, b in out] == list(range(5))
    assert c.finish() == []
    batches = [(torch.full((2, 3), float(i)), torch.tensor([i, i]), "meta") for i in range(4)]
    got = list(cuda_prefetch(iter(batches), "cpu", reuse_buffers=True))
    assert len(got) == 4 and all(torch.equal(g[0], b[0]) and g[2] == "meta" for g, b in zip(got, batches))


def test_uint8_loader_path_matches_the_reference_transforms_on_cpu():
    """Opt-in uint8 upload: uint8_transform() + the normalisation cuda_prefetch applies == the reference's
    Resize / CenterCrop / ToTensor / Normalize (test_RESNET50_Truncate_gram_attention.py:61-66), bit for bit."""
    import numpy as np
    from PIL import Image
    from torchvision import transforms
    from heuristique_style_transfer_code_b200 import functions as F
    rng = np.random.default_rng(5)
    images = [Image.fromarray(rng.integers(0, 256, (300 + 20 * i, 280, 3), dtype=np.uint8)) for i in range(3)]
    reference = transforms.Compose([transforms.Resize(256), transforms.CenterCrop(224), transforms.ToTensor(),
                                    transforms.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])
    want = torch.stack([reference(im) for im in images])
    pixels = torch.stack([F.uint8_transform(256, 224)(im) for im in images])
    assert pixels.dtype == torch.uint8 and pixels.shape == (3, 3, 224, 224)
    labels = torch.tensor([0, 1, 2])
    (got, lab), = list(F.cuda_prefetch(iter([(pixels, labels)]), "cpu"))
    assert got.dtype == torch.float32 and torch.equal(got, want) and torch.equal(lab, labels)
    (raw, _), = list(F.cuda_prefetch(iter([(pixels, labels)]), "cpu", normalize=None))
    assert raw.dtype == torch.uint8 and torch.equal(raw, pixels)                # opt-out leaves the pixels alone
    (half, _), = list(F.cuda_prefetch(iter([(pixels, labels)]), "cpu", normalize=((0.5,) * 3, (0.25,) * 3)))
    assert torch.equal(half, (pixels.float() / 255 - 0.5) / 0.25)
    mask = torch.zeros(2, 8, 8, dtype=torch.uint8)                              # not an image batch: passed through
    (m2,), = list(F.cuda_prefetch(iter([(mask,)]), "cpu"))
    assert m2.dtype == torch.uint8


def test_checkpoint_converters_produce_what_load_model_loads(tmp_path):
    """SURVEY 8(f) n4 / quirk Q2: a torchvision ResNet50 state_dict and a three-section checkpoint match nothing in
    load_model (reference behaviour, preserved); their converted bare-encoder form fills every encoder tensor."""
    import torch
    from torchvision import models
    from heuristique_style_transfer_code_b200 import TruncatedResNet50, checkpoints
    from heuristique_style_transfer_code_b200.functions import load_model, save_model_weights

    torch.manual_seed(3)
    donor = models.resnet50(weights=None)
    model = TruncatedResNet50(models.resnet50(weights=None), 7, 4, 8, device="cpu")
    before = {k: v.clone() for k, v in model.state_dict().items()}
    n_enc = sum(1 for k in before if k.startswith("truncated_encoder."))

    # (1) plain torchvision names: load_model "succeeds" and loads nothing
    plain = tmp_path / "resnet50.pth"
    torch.save(donor.state_dict(), plain)
    assert checkpoints.coverage(model, donor.state_dict()) == {"matched": 0, "encoder": n_enc,
                                                               "dropped": len(donor.state_dict()) - 2}
    load_model(model, str(plain), "cpu")
    assert all(torch.equal(v, before[k]) for k, v in model.state_dict().items())

    # (2) converted: every encoder tensor now comes from the donor
    bare = tmp_path / "bare.pth"
    assert checkpoints.convert_file(str(plain), str(bare)) > 0
    converted = torch.load(bare)
    cov = checkpoints.coverage(model, converted)
    assert cov["matched"] == n_enc                      # layer4 tensors are converted too and dropped by load_model
    load_model(model, str(bare), "cpu")
    sd = model.state_dict()
    assert torch.equal(sd["truncated_encoder.0.weight"], donor.conv1.weight)
    assert torch.equal(sd["truncated_encoder.6.5.bn3.running_var"], donor.layer3[5].bn3.running_var)
    assert torch.equal(sd["classifier.weight"], before["classifier.weight"])        # head untouched

    # (3) the three-section file of save_model_weights (what the README passes to --model_path) and DDP-prefixed dicts
    three = tmp_path / "best_model_all.pth"
    save_model_weights(model, str(three))
    assert checkpoints.coverage(model, torch.load(three))["matched"] == 0
    assert set(checkpoints.to_bare_encoder(torch.load(three))) == {k[len("truncated_encoder."):] for k in before
                                                                   if k.startswith("truncated_encoder.")}
    ddp_like = {"module." + k: v for k, v in model.state_dict().items()}
    assert set(checkpoints.to_bare_encoder(ddp_like)) == set(checkpoints.to_bare_encoder(torch.load(three)))
    assert checkpoints.to_bare_encoder(converted).keys() == converted.keys()        # idempotent


def test_reference_loader_restores_anomaly_mode_and_graphed_step_needs_cuda(tmp_path, monkeypatch):
    """_reference.load_reference_file: the reference files switch torch's anomaly detection on at import
    (Models/...Attention.py:9); the loader must leave the caller's setting untouched. GraphedTrainStep is CUDA-only.
    The file loaded is a stand-in with the same import-time side effect, so no checkout of the reference is needed."""
    import os
    import pytest
    import torch
    from heuristique_style_transfer_code_b200 import _reference
    from heuristique_style_transfer_code_b200.functions import GraphedTrainStep
    rel = os.path.join("Models", "Models_RESNET50_TRUNCATE_GRAM_with_Attention.py")
    (tmp_path / "Models").mkdir()
    (tmp_path / rel).write_text("import torch\ntorch.autograd.set_detect_anomaly(True)\n\n\n"
                                "class TruncatedResNet50:\n    pass\n\n\nclass TruncatedResNet50_for_test:\n    pass\n")
    monkeypatch.setenv("GRAMHEAD_REFERENCE_ROOT", str(tmp_path))
    monkeypatch.setattr(_reference, "_LOADED", {})
    assert _reference.reference_root(rel) == str(tmp_path)
    assert not torch.is_anomaly_enabled()
    mod = _reference.load_reference_file(rel)
    assert not torch.is_anomaly_enabled()
    assert hasattr(mod, "TruncatedResNet50") and hasattr(mod, "TruncatedResNet50_for_test")
    assert _reference.load_reference_file(rel) is mod                     # cached
    with pytest.raises(NotImplementedError):
        _reference.load_reference_file(os.path.join("Models", "does_not_exist.py"))
    lin = torch.nn.Linear(4, 2)
    with pytest.raises(ValueError):
        GraphedTrainStep(lin, torch.nn.CrossEntropyLoss(), torch.optim.SGD(lin.parameters(), lr=0.1), torch.randn(3, 4),
                         torch.zeros(3, dtype=torch.long))
