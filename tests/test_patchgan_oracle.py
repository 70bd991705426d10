"""Multi-PatchGAN Gram head (SURVEY 8(f) n4) on CPU: the fp64 oracle against the committed golden vectors (outputs of the
unmodified reference class) and, in the build container, against the reference run live; the drop-in contract."""
import inspect
import os

import numpy as np
import pytest
import torch

from conftest import ROOT
from heuristique_style_transfer_code_b200 import patchgan as P
from heuristique_style_transfer_code_b200._lib import GramHeadError
from oracle import patchgan_fp64 as O
from oracle.ref_loader import load_reference_patchgan, reference_available
from oracle.torch_port import patchgan_forward, patchgan_multiscale_forward

GOLDEN = os.path.join(ROOT, "tests", "golden", "patchgan_head.npz")
needs_reference = pytest.mark.skipif(not reference_available(),
                                     reason="needs a checkout of the reference project (GH_REFERENCE_ROOT)")


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def load_golden():
    z = np.load(GOLDEN)
    n = sum(1 for k in z.files if k.startswith("x_proj_"))
    return z, [z[f"x_proj_{i}"] for i in range(n)], {k: z["param/" + k] for k in O.HEAD_KEYS}


def test_oracle_reproduces_the_reference_golden_vectors():
    z, maps, params = load_golden()
    assert [m.shape[2:] for m in maps] == [(12, 20), (6, 10), (3, 5), (2, 4), (1, 3)]
    r = O.patch_head(maps, params, heads=8, ln_input=True)
    assert rel(r["gram_norms"], z["gram_norms"]) < 1e-6
    assert rel(r["embeddings"], z["embeddings"]) < 1e-6
    assert rel(r["output"], z["output"]) < 1e-6
    # folding the :198 layer norm in or applying it first is the same function
    r2 = O.patch_head([O.layer_norm_all(m) for m in maps], params, heads=8, ln_input=False)
    assert rel(r2["embeddings"], r["embeddings"]) < 1e-12


def test_adaptive_bins_follow_aten():
    for n in (1, 2, 3, 4, 5, 7, 12, 13, 112):
        x = torch.arange(n, dtype=torch.float64).view(1, 1, n, 1).expand(1, 1, n, n).contiguous()
        want = torch.nn.functional.adaptive_avg_pool2d(x, (4, 4))[0, 0, :, 0].numpy()
        got = np.array([np.arange(n)[s:e].mean() for s, e in O.adaptive_bins(n)])
        assert np.allclose(got, want), n


@needs_reference
@pytest.mark.parametrize("norm,patch,size", [("batch", 30, (64, 64)), ("instance", 70, (96, 128))])
def test_oracle_and_port_against_the_live_reference(norm, patch, size):
    ref = load_reference_patchgan()
    torch.manual_seed(3)
    m = ref.VariablePatchesNLayerDiscriminator_test(ndf=32, norm=norm, patch_size=patch, num_classes=4, gram_matrix_dim=32).eval()
    x = torch.randn(2, 3, *size)
    raw = []
    hooks = [p.register_forward_hook(lambda mod, i, o: raw.append(o.detach())) for p in m.projection_layers]
    with torch.no_grad():
        emb, out = m(x)
        for h in hooks:
            h.remove()
        pe, po, pn = patchgan_forward(m, x)
    assert torch.equal(pe, emb) and torch.equal(po, out)                     # the torch port is the same op sequence
    assert all(torch.equal(a, b) for a, b in zip(pn, m.get_gram_norms()))
    sd = m.state_dict()
    r = O.patch_head([t.numpy() for t in raw], {k: sd[k].numpy() for k in O.HEAD_KEYS}, heads=8, ln_input=True)
    assert rel(r["embeddings"], emb.numpy()) < 2e-6 and rel(r["output"], out.numpy()) < 2e-6
    assert rel(r["gram_norms"], torch.stack(m.get_gram_norms()).numpy()) < 2e-6


def test_drop_in_init_and_port_reproduce_the_recorded_reference():
    """The drop-in class rebuilt the way tests/golden/make_golden_patchgan.py built the reference's: same seed, same
    edits of the batch-norm statistics and attention biases, then the input. Identical random init shows as the same
    input (the constructor consumed the generator identically) and the same head tensors; the same convolution weights
    as the same projections; the port on its submodules as the reference's embeddings, output and Gram norms."""
    z, maps, params = load_golden()
    torch.manual_seed(1234)
    m = P.VariablePatchesNLayerDiscriminator_test(ndf=16, norm='batch', patch_size=30, num_classes=5,
                                                  gram_matrix_dim=16).eval()
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.running_mean.normal_(0, 0.2)
                mod.running_var.uniform_(0.5, 1.5)
        for name in ("attention_per_layer", "attention_per_patch"):
            getattr(m, name).in_proj_bias.normal_(0, 0.1)
            getattr(m, name).out_proj.bias.normal_(0, 0.1)
    x = torch.randn(2, 3, 24, 40)
    assert torch.equal(x, torch.from_numpy(z["input"]))
    sd = m.state_dict()
    assert all(np.array_equal(sd[k].numpy(), params[k]) for k in O.HEAD_KEYS)
    raw = []
    hooks = [p.register_forward_hook(lambda mod, i, o: raw.append(o.detach())) for p in m.projection_layers]
    with torch.no_grad():
        emb, out, norms = patchgan_forward(m, x)
    for h in hooks:
        h.remove()
    assert len(raw) == len(maps) and all(rel(a, b) < 1e-6 for a, b in zip(raw, maps))
    assert rel(emb, z["embeddings"]) < 1e-6 and rel(out, z["output"]) < 1e-6
    assert rel(torch.stack(norms), z["gram_norms"]) < 1e-6


@needs_reference
@pytest.mark.parametrize("name,kw", [
    ("VariablePatchesNLayerDiscriminator_test", dict(ndf=16, norm='batch', patch_size=70, num_classes=5, gram_matrix_dim=16)),
    ("VariablePatchesNLayerDiscriminator_test", dict(patch_size=10)),
    ("MultiScaleDiscriminator_test", dict(ndf=16, gram_matrix_dim=8)),
    ("MultiScaleDiscriminator", dict(ndf=8)),
    ("VariablePatchesNLayerDiscriminator", dict(ndf=8, norm='batch'))])
def test_identical_signature_init_and_state_dict_as_reference(name, kw):
    ref = load_reference_patchgan()
    a_cls, b_cls = getattr(ref, name), getattr(P, name)
    assert list(inspect.signature(a_cls.__init__).parameters.items()) == list(inspect.signature(b_cls.__init__).parameters.items())
    torch.manual_seed(0)
    a = a_cls(**kw)
    torch.manual_seed(0)
    b = b_cls(**kw)
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb)
    assert all(torch.equal(sa[k], sb[k]) for k in sa)
    assert [n for n, _ in a.named_modules()] == [n for n, _ in b.named_modules()]


def _stand_in_reference_tree(root, files):
    """A tree with the reference's layout whose files hold only the given sources: enough to show which file a name
    resolves to, without a checkout of the reference."""
    for rel_path, source in files.items():
        path = root / rel_path
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_text(source)
    return str(root)


def test_reference_module_path_resolves_to_the_b200_classes(tmp_path, monkeypatch):
    import Models.Models_Multi_PatchGAN as M
    from heuristique_style_transfer_code_b200 import _reference
    assert M.MultiScaleDiscriminator_test is P.MultiScaleDiscriminator_test
    assert M.VariablePatchesNLayerDiscriminator_test is P.VariablePatchesNLayerDiscriminator_test
    assert M.PATCH_TYPES == P.PATCH_TYPES
    # the head-less training classes are the reference's own, taken from the reference tree the loader finds
    rel_path = os.path.join("Models", "Models_Multi_PatchGAN.py")
    root = _stand_in_reference_tree(tmp_path, {rel_path: "class MultiScaleDiscriminator:\n    pass\n\n\n"
                                                         "class VariablePatchesNLayerDiscriminator:\n    pass\n"})
    monkeypatch.setenv("GRAMHEAD_REFERENCE_ROOT", root)
    monkeypatch.setattr(_reference, "_LOADED", {})
    ref = _reference.load_reference_file(rel_path)
    assert M.MultiScaleDiscriminator is P.MultiScaleDiscriminator is ref.MultiScaleDiscriminator
    assert M.VariablePatchesNLayerDiscriminator is P.VariablePatchesNLayerDiscriminator is ref.VariablePatchesNLayerDiscriminator


def test_structure_and_loud_failures_without_cuda():
    torch.manual_seed(0)
    m = P.VariablePatchesNLayerDiscriminator_test(ndf=16, norm='batch', patch_size=70, num_classes=5, gram_matrix_dim=16)
    names = [n for n, _ in m.feature_extractor.named_children()]
    assert names[:3] == ["conv0", "norm0", "relu0"] and names[-4:] == ["final_conv", "final_norm", "final_relu", "final_conv_ndf"]
    assert len(m.projection_layers) == sum(isinstance(c, torch.nn.Conv2d) for c in m.feature_extractor)
    assert m.attention_per_layer.num_heads == 8 and m.feature_projection.in_features == 256
    with torch.no_grad(), pytest.raises(GramHeadError, match="no CPU path"):
        m(torch.randn(1, 3, 64, 64))
    assert m.get_gram_norms() == []
    ms = P.MultiScaleDiscriminator_test(ndf=16, gram_matrix_dim=8)
    assert list(ms.scale_discriminators) == ["small", "medium", "large"]
    # the port drives the drop-in's submodules on CPU (what bench / GPU tests use as the checker)
    with torch.no_grad():
        e, o = patchgan_multiscale_forward(ms.eval(), torch.randn(1, 3, 224, 224))
    assert e.shape == (1, 16) and o.shape == (1, 10)


def test_reference_scripts_resolve_the_drop_in_classes_and_keep_their_own_functions_file(tmp_path):
    """What tools/run_ref_script.py arranges for test_Multi_PatchGAN.py: the model classes come from this repository,
    functions.functions_Multi_PatchGAN (not provided here) from the reference tree through the namespace packages."""
    import subprocess
    import sys
    REFERENCE_ROOT = _stand_in_reference_tree(tmp_path / "reference", {
        os.path.join("Models", "Models_Multi_PatchGAN.py"): "raise ImportError('shadowed by the drop-in')\n",
        os.path.join("functions", "functions_Multi_PatchGAN.py"): ""})
    code = (
        "import sys, importlib.util\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "import Models.Models_Multi_PatchGAN as mine\n"
        f"sys.path.insert(0, {REFERENCE_ROOT!r})\n"
        "from Models.Models_Multi_PatchGAN import MultiScaleDiscriminator_test as cls\n"
        "assert cls is mine.MultiScaleDiscriminator_test and cls.__module__.startswith('heuristique_style_transfer_code_b200')\n"
        "spec = importlib.util.find_spec('functions.functions_Multi_PatchGAN')\n"
        f"assert spec is not None and spec.origin.startswith({REFERENCE_ROOT!r}), spec\n"
        "print('ok')\n")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=str(tmp_path))
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stderr
