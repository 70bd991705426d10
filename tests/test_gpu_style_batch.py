"""Style transfer on several images per step: the per-image loss kernel (gh_gram_mse_images), its op
(ops.gram_mse_loss_per_image), the N-image engine (functions._StyleIteration(images=N)) and style_transfer's
images_per_step, on the GPU."""
import contextlib
import io
import os

import numpy as np
import pytest
import torch

from oracle import head_fp64 as O

pytestmark = pytest.mark.gpu


def npf(t):
    return t.detach().double().cpu().numpy()


@pytest.fixture(scope="module")
def ops():
    from heuristique_style_transfer_code_b200 import ops as _ops
    from heuristique_style_transfer_code_b200 import _lib
    _lib.lib()
    return _ops


@contextlib.contextmanager
def deterministic():
    """One K part in the Gram forward (no atomics: at small batch it is split over K and the parts meet in atomics) and
    deterministic cuDNN, so that two runs of the same arithmetic give the same bits."""
    from heuristique_style_transfer_code_b200 import ops as _ops
    saved = (_ops.KSPLIT, torch.backends.cudnn.deterministic, torch.backends.cudnn.allow_tf32)
    _ops.KSPLIT, torch.backends.cudnn.deterministic, torch.backends.cudnn.allow_tf32 = 1, True, False
    try:
        yield
    finally:
        _ops.KSPLIT, torch.backends.cudnn.deterministic, torch.backends.cudnn.allow_tf32 = saved


def mse_images(G, T):
    """Raw gh_gram_mse_images on (B, C, C) fp32 tensors -> (partial (B, k), dG)."""
    from heuristique_style_transfer_code_b200 import _lib
    lib = _lib.lib()
    b, c, _ = G.shape
    k = lib.gh_gram_mse_images_blocks(c * c)
    assert k == lib.gh_gram_mse_blocks(c * c)
    partial = torch.full((b, k), float("nan"), device=G.device)
    dG = torch.full_like(G, float("nan"))
    assert lib.gh_gram_mse_images(G.data_ptr(), T.data_ptr(), b, c * c, dG.data_ptr(), partial.data_ptr(), None) == 0
    torch.cuda.synchronize()
    return partial, dG


def mse_single(g, t):
    """Raw gh_gram_mse on one (C, C) image -> (partial (k,), dG)."""
    from heuristique_style_transfer_code_b200 import _lib
    lib = _lib.lib()
    n = g.numel()
    partial = torch.full((lib.gh_gram_mse_blocks(n),), float("nan"), device=g.device)
    dG = torch.full_like(g, float("nan"))
    assert lib.gh_gram_mse(g.data_ptr(), t.data_ptr(), n, dG.data_ptr(), partial.data_ptr(), None) == 0
    torch.cuda.synchronize()
    return partial, dG


HW_SIDE = {3136: 56, 784: 28, 196: 14, 49: 7}
# B in {1, 3, 8}, C in {3, 17, 64, 256, 1024}, HW in {3136, 784, 196, 49}; C * C % 4 != 0 for C = 3, 17 (misaligned images)
SHAPES = [(1, 64, 3136), (3, 17, 49), (3, 3, 196), (8, 3, 784), (3, 64, 49), (8, 256, 784), (1, 256, 196),
          (3, 1024, 196), (8, 17, 3136), (1, 1024, 49), (3, 256, 3136)]


def features(B, C, HW, layout, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    s = HW_SIDE[HW]
    x = torch.relu(torch.randn(B, C, s, s, generator=g)).cuda()
    return x.contiguous(memory_format=torch.channels_last) if layout == "nhwc" else x


@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("B,C,HW", SHAPES)
def test_per_image_loss_against_fp64(ops, B, C, HW, layout):
    """The kernel on given Grams: per-image loss <= 1e-5 relative to fp64 mean((G - G*)^2) of the same G, dG <= 1e-6.
    The op: per-image losses against oracle.style_loss_and_grad applied to each image's features (<= 1e-3 through the
    tf32 Gram; the fp32 NCHW features with HW % 4 != 0 take the ld.global kernels, bf16 operands: 6e-3 as in
    test_gpu_gram_routes.py), and dF of losses.sum() against each image's oracle dF, normwise, same tolerances."""
    x = features(B, C, HW, layout, seed=B * 1000 + C + HW)
    y = features(B, C, HW, layout, seed=7 + B * 1000 + C + HW) * 1.3
    with torch.no_grad():
        target = ops.gram_matrix(y)
        G = ops.gram_matrix(x)
    partial, dG = mse_images(G, target)
    Gd, Td = npf(G), npf(target)
    for b in range(B):
        want = np.mean((Gd[b] - Td[b]) ** 2)
        assert abs(float(partial[b].double().sum()) - want) <= 1e-5 * want, b
        assert O.rel_err(npf(dG[b]), 2 * (Gd[b] - Td[b]) / (C * C)) <= 1e-6, b
    tol = 6e-3 if HW % 4 else 1e-3
    a = x.clone(memory_format=torch.channels_last if layout == "nhwc" else torch.contiguous_format).requires_grad_(True)
    losses = ops.gram_mse_loss_per_image(a, target)
    assert losses.shape == (B,)
    losses.sum().backward()
    torch.cuda.synchronize()
    assert a.grad.shape == x.shape and ops.is_channels_last(a.grad) == (layout == "nhwc")
    xf = npf(x).reshape(B, C, HW)
    for b in range(B):
        want_loss, want_df = O.style_loss_and_grad(xf[b:b + 1], Td[b:b + 1])
        assert abs(float(losses[b]) - want_loss) <= tol * want_loss, b
        assert O.rel_err(npf(a.grad[b]).reshape(1, C, HW), want_df) <= tol, b


@pytest.mark.parametrize("B,C", [(1, 3), (3, 3), (3, 17), (8, 17), (3, 64), (8, 256), (3, 1024), (2, 100), (5, 1)])
def test_each_image_is_bitwise_its_single_image_call(ops, B, C):
    """Image b's partials and dG slice are the bits gh_gram_mse gives on a fresh (aligned) copy of G[b] alone, whether
    image b starts on a 16 B boundary (C * C % 4 == 0) or not; the other images do not matter."""
    g = torch.Generator(device="cpu").manual_seed(B * 100 + C)
    G = torch.randn(B, C, C, generator=g).cuda()
    T = torch.randn(B, C, C, generator=g).cuda()
    partial, dG = mse_images(G, T)
    assert not partial.isnan().any() and not dG.isnan().any()
    for b in range(B):
        p1, d1 = mse_single(G[b].clone(), T[b].clone())
        assert torch.equal(partial[b], p1), b
        assert torch.equal(dG[b], d1), b
    # another batch around the same image: same bits for it
    if B > 1:
        G2, T2 = torch.randn_like(G), torch.randn_like(T)
        G2[B - 1], T2[B - 1] = G[B - 1], T[B - 1]
        p2, d2 = mse_images(G2, T2)
        assert torch.equal(p2[B - 1], partial[B - 1]) and torch.equal(d2[B - 1], dG[B - 1])


# ---- the engine -------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def model_encoder():
    from torchvision import models
    from heuristique_style_transfer_code_b200 import TruncatedResNet50_for_test
    torch.manual_seed(0)
    model = TruncatedResNet50_for_test(models.resnet50(weights=None), 7, 4, 32, device="cuda:0").eval()
    encoder = torch.nn.Sequential(*list(model.truncated_encoder.children())[:5]).to("cuda:0")
    return model, encoder


def test_engine_one_image_eager_is_bitwise_the_one_image_loop(ops, model_encoder):
    """N = 1, eager: after 5 steps the noise has the bits of the loop before the per-image loss (ops.gram_mse_loss +
    loss.backward() + Adam), restated here."""
    from heuristique_style_transfer_code_b200.functions import _StyleIteration
    model, encoder = model_encoder
    g = torch.Generator(device="cpu").manual_seed(3)
    image = torch.randn(1, 3, 224, 224, generator=g).cuda()
    noise0 = torch.randn(1, 3, 224, 224, generator=g).cuda()
    with deterministic():
        with torch.no_grad():
            target = model.gram_matrix(encoder(image))
        noise = noise0.clone().requires_grad_(True)
        opt = torch.optim.Adam([noise], lr=0.01)
        want_losses = []
        for _ in range(5):
            opt.zero_grad()
            loss = ops.gram_mse_loss(encoder(noise), target)
            loss.backward()
            opt.step()
            want_losses.append(loss.item())
        it = _StyleIteration(model, encoder, "cuda:0", 0.01, use_graph=False)
        it.start(target, noise0)
        got_losses = [it.step() for _ in range(5)]
        torch.cuda.synchronize()
    assert torch.equal(it.noise.detach(), noise.detach())
    for a, b in zip(got_losses, want_losses):
        assert abs(a - b) <= 1e-6 * abs(b), (got_losses, want_losses)


def test_engine_four_images_graph_matches_eager(ops, model_encoder):
    """N = 4: graph replay against eager steps, per-image losses within 2e-3 (the one-image test's tolerance); step()
    returns their sum; restarting reproduces the first run. The Gram forward is not split over K and cuDNN is
    deterministic here: with atomics in the loop, Adam's first, sign-like steps turn last-bit differences of small
    gradients into different trajectories, which at four images moves some per-image losses by more than 2e-3 within
    five steps. The two runs then differ only by Adam's capturable (graph) and host-step (eager) arithmetic."""
    from heuristique_style_transfer_code_b200.functions import _StyleIteration
    model, encoder = model_encoder
    g = torch.Generator(device="cpu").manual_seed(4)
    images = torch.randn(4, 3, 224, 224, generator=g).cuda()
    noise0 = torch.randn(4, 3, 224, 224, generator=g).cuda()
    runs = {}
    with deterministic():
        with torch.no_grad():
            target = model.gram_matrix(encoder(images))
        for use_graph in (False, True):
            it = _StyleIteration(model, encoder, "cuda:0", 0.01, use_graph=use_graph, images=4)
            losses = []
            for rep in range(2):
                it.start(target, noise0)
                losses.append([it.step_losses() for _ in range(5)])
            noise = it.noise.detach().clone()
            total = it.step()
            assert abs(total - sum(it.losses.tolist())) <= 1e-6 * total
            assert (it.graph is not None) == use_graph
            runs[use_graph] = (losses, noise)
    (le, ne), (lg, ng) = runs[False], runs[True]
    assert le[0][0] == lg[0][0]                   # step 0: same noise, same arithmetic before Adam
    for rep in range(2):
        for step, (se, sg) in enumerate(zip(le[rep], lg[rep])):
            rel = max(abs(a - b) / abs(a) for a, b in zip(se, sg))
            assert len(se) == 4 and rel <= 2e-3, (rep, step, rel, se, sg)
    assert all(le[0][0][b] > le[0][-1][b] for b in range(4))          # every image's loss goes down
    assert all(abs(a - b) <= 2e-3 * abs(a) for sa, sb in zip(le[0], le[1]) for a, b in zip(sa, sb))
    assert float((ne - ng).abs().max()) <= 5e-3


@pytest.mark.parametrize("use_graph", [False, True])
def test_converged_image_result_is_fixed_while_the_others_step(ops, model_encoder, use_graph):
    """Image 0's target is the Gram of its own initial noise (scaled by 1 + 1e-4, so that its gradient is not zero), so
    its loss is below the threshold at iteration 0: its result is the noise after step 0 (bits of a separate one-step
    run), although it keeps being stepped with the others, which never reach the threshold."""
    from heuristique_style_transfer_code_b200.functions import _StyleIteration, _optimise_chunk
    model, encoder = model_encoder
    g = torch.Generator(device="cpu").manual_seed(5)
    noise0 = torch.randn(4, 3, 224, 224, generator=g).cuda()
    others = torch.randn(3, 3, 224, 224, generator=g).cuda() * 3
    with deterministic():
        with torch.no_grad():
            target = model.gram_matrix(encoder(torch.cat([noise0[:1], others])))
            target[0] = model.gram_matrix(encoder(noise0))[0] * (1 + 1e-4)
        threshold = 1e-6 * float(target.pow(2).mean())
        it = _StyleIteration(model, encoder, "cuda:0", 0.01, use_graph=use_graph, images=4)
        it.start(target, noise0)
        first = it.step_losses()
        after_step0 = it.noise.detach().clone()
        assert first[0] < threshold and min(first[1:]) > 1e2 * threshold, first
        result, reached = _optimise_chunk(it, target, noise0, threshold, 6)
        torch.cuda.synchronize()
    assert reached == [0, None, None, None]
    assert torch.equal(result[0], after_step0[0])
    assert not torch.equal(it.noise.detach()[0], result[0])               # image 0 kept being stepped
    assert torch.equal(result[1:], it.noise.detach()[1:])                 # the others: the noise after the last step


# ---- style_transfer ---------------------------------------------------------------------------------------------------
def _run_style_transfer(model, loader, save_dir, seed, **kw):
    from PIL import Image
    from heuristique_style_transfer_code_b200.functions import style_transfer
    torch.manual_seed(seed)
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        style_transfer(model, loader, "cuda:0", str(save_dir), layers=5, **kw)
    files = {}
    for root, _, names in os.walk(save_dir):
        for name in names:
            path = os.path.join(root, name)
            files[os.path.relpath(path, save_dir)] = np.asarray(Image.open(path).convert("RGB"), dtype=np.float64) / 255
    return out.getvalue(), files


@pytest.mark.parametrize("threshold,iterations,converged", [(float("inf"), 4, True), (0.0, 5, False)])
def test_style_transfer_images_per_step_matches_the_one_image_loop(ops, model_encoder, tmp_path, monkeypatch,
                                                                   threshold, iterations, converged):
    """5 images in loader batches of 3 and 2 (chunks of 2, 1 and 2 at images_per_step = 2; labels chosen so that no
    two images share a file name, which uses the index within the loader batch): the same files and line
    for line the same stdout as the default loop. threshold = inf stops every image at iteration 0, threshold = 0 never
    stops one. The originals (left halves) are identical; the results differ by the encoder's batch-size-dependent
    rounding only: mean |diff| <= 1/255 and max |diff| <= 0.05 per pixel."""
    from torch.utils.data import DataLoader, TensorDataset
    model, _ = model_encoder
    g = torch.Generator(device="cpu").manual_seed(6)
    data = TensorDataset(torch.randn(5, 3, 224, 224, generator=g), torch.tensor([0, 1, 2, 3, 4]))
    loader = DataLoader(data, batch_size=3, shuffle=False)
    saved = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        monkeypatch.delenv("GRAMHEAD_STYLE_IMAGES", raising=False)
        runs = [_run_style_transfer(model, loader, tmp_path, 11, threshold=threshold, num_iterations=iterations)]
        runs.append(_run_style_transfer(model, loader, tmp_path, 11, threshold=threshold, num_iterations=iterations,
                                        images_per_step=2))
        monkeypatch.setenv("GRAMHEAD_STYLE_IMAGES", "2")
        runs.append(_run_style_transfer(model, loader, tmp_path, 11, threshold=threshold, num_iterations=iterations))
    finally:
        torch.backends.cudnn.allow_tf32 = saved
    (out1, files1) = runs[0]
    lines = out1.splitlines()
    assert len(lines) == (10 if converged else 5), out1
    assert sum("itération 0" in line for line in lines) == (5 if converged else 0)
    assert len(files1) == 5
    for out, files in runs[1:]:
        assert out == out1
        assert sorted(files) == sorted(files1)
        for name, img in files.items():
            ref = files1[name]
            w = ref.shape[1] // 2
            assert np.array_equal(img[:, :w], ref[:, :w]), name
            d = np.abs(img[:, w:] - ref[:, w:])
            assert d.mean() <= 1 / 255 and d.max() <= 0.05, (name, d.mean(), d.max())
