"""Backward of the Multi-PatchGAN Gram head on a B200: the three autograd Functions (ops._PatchGram, _PatchProjection,
_PatchAttention) against the fp64 oracle, guard regions around every buffer the backward entry points write, layouts,
reproducibility, and the drop-in modules with the library backward switched on against autograd of the fp32 port."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle.torch_port import patchgan_forward

import patchgan_backward_fp64 as G

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def npf(t):
    return t.detach().float().cpu().numpy()


def test_cuda_is_present():
    assert torch.cuda.is_available()


def make_head(d, e, nc, seed):
    torch.manual_seed(seed)
    a1 = torch.nn.MultiheadAttention(e, 8).cuda()
    a2 = torch.nn.MultiheadAttention(e, 8).cuda()
    cl = torch.nn.Linear(e, nc).cuda()
    fp = torch.nn.Linear(d * d, e).cuda()
    with torch.no_grad():
        for a in (a1, a2):
            a.in_proj_bias.normal_(0, 0.2)
            a.out_proj.bias.normal_(0, 0.2)
    return a1, a2, cl, fp


def head_named_params(a1, a2, cl, fp):
    out = {}
    for name, mod in (("attention_per_layer", a1), ("attention_per_patch", a2), ("classifier", cl), ("feature_projection", fp)):
        out.update({f"{name}.{k}": v for k, v in mod.named_parameters()})
    return out


def run_head_autograd(maps, a1, a2, cl, fp, ln_input):
    from heuristique_style_transfer_code_b200 import ops
    gram, norms = ops.patch_gram_autograd(maps, ln_input=ln_input)
    feat = ops.patch_projection_autograd(gram, fp)
    emb, out = ops.patch_attention_autograd(feat, a1, a2, cl)
    return gram, norms, feat, emb, out


def cotangents(emb, out, norms, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(emb.shape, device="cuda", generator=g), torch.randn(out.shape, device="cuda", generator=g),
            torch.randn(norms.shape, device="cuda", generator=g))


SHAPES = [
    (64, 64, [(112, 112), (56, 56), (28, 28), (14, 14), (13, 13), (12, 12)], 3),     # patch 70 at 224x224
    (64, 64, [(112, 112), (56, 56), (55, 55), (54, 54)], 2),                         # patch 10 at 224x224
    (32, 32, [(24, 17), (5, 9), (3, 3), (2, 1), (1, 1)], 4),                          # tiny / ragged maps
    (128, 128, [(20, 20), (7, 7)], 2),                                               # the largest D and ndf accepted
    (24, 40, [(9, 31)] * 8, 2)]                                                      # eight layers, D not a multiple of 32


@pytest.mark.parametrize("d,e,shapes,b", SHAPES)
@pytest.mark.parametrize("ln_input", [True, False])
def test_functions_against_the_fp64_oracle(d, e, shapes, b, ln_input):
    """d_maps (the _PatchGram backward), d_gram and d_feat (retained), every head parameter gradient, with a nonzero
    cotangent on the norms. fp32 kernels and split-bf16 GEMMs against fp64: 1e-4 normwise."""
    torch.manual_seed(d + len(shapes))
    maps = [(torch.randn(b, d, h, w, device="cuda") * (1.0 + i) + 0.3 * i).requires_grad_(True)
            for i, (h, w) in enumerate(shapes)]
    a1, a2, cl, fp = make_head(d, e, 7, d + e)
    gram, norms, feat, emb, out = run_head_autograd(maps, a1, a2, cl, fp, ln_input)
    gram.retain_grad()
    feat.retain_grad()
    ce, co, cn = cotangents(emb, out, norms)
    ((emb * ce).sum() + (out * co).sum() + (norms * cn).sum()).backward()
    params = head_named_params(a1, a2, cl, fp)
    want = G.patch_head_grad([npf(m) for m in maps], {k: npf(v) for k, v in params.items()}, npf(ce), npf(co), npf(cn),
                             heads=8, ln_input=ln_input)
    errs = {f"map{i}": rel(npf(m.grad), g) for i, (m, g) in enumerate(zip(maps, want["maps"]))}
    errs["d_gram"] = rel(npf(gram.grad), want["grams"].reshape(gram.shape))
    errs["d_feat"] = rel(npf(feat.grad), want["projected"])
    errs.update({k: rel(npf(v.grad), want[k]) for k, v in params.items()})
    print(f"\nrelative errors d={d} e={e} L={len(shapes)} ln_input={ln_input}: "
          + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    for k, v in errs.items():
        assert v < 1e-4, (k, v)


def guarded(n, pad=64):
    """A length-n fp32 view inside a NaN-filled buffer: pad floats of NaN either side (16 B aligned)."""
    big = torch.full((n + 2 * pad,), float("nan"), device="cuda")
    return big, big[pad:pad + n]


def guards_intact(big, pad=64):
    return bool(torch.isnan(big[:pad]).all()) and bool(torch.isnan(big[-pad:]).all())


def test_guard_regions_around_every_output_buffer():
    from heuristique_style_transfer_code_b200 import _lib, ops
    lib = _lib.lib()
    torch.manual_seed(1)
    L, b, d, e, nc = 3, 2, 24, 40, 5
    shapes = [(20, 18), (9, 7), (3, 2)]
    maps = [torch.randn(b, d, h, w, device="cuda") for h, w in shapes]
    a1, a2, cl, fp = make_head(d, e, nc, 3)
    stream = torch.cuda.current_stream().cuda_stream
    gram, norm, scratch = ops._patch_gram_fwd(maps, True)
    d_gram, d_norm = torch.randn_like(gram), torch.randn_like(norm)
    # gh_patch_gram_bwd
    big_ws, ws = guarded(lib.gh_patch_bwd_workspace(L, b, d))
    _, hs, wsz, st = ops._patch_map_arrays(maps)
    _lib.check(lib.gh_patch_gram_bwd(hs, wsz, L, b, d, 1, d_gram.data_ptr(), d_norm.data_ptr(), norm.data_ptr(),
                                     scratch.data_ptr(), ws.data_ptr(), stream), "gh_patch_gram_bwd")
    # gh_patch_pool_bwd into guarded gradients
    bigs, grads = zip(*[guarded(m.numel()) for m in maps])
    gptrs = (ctypes.c_void_p * L)(*[g.data_ptr() for g in grads])
    ptrs = (ctypes.c_void_p * L)(*[m.data_ptr() for m in maps])
    _lib.check(lib.gh_patch_pool_bwd(ptrs, gptrs, hs, wsz, st, st, L, b, d, 1, ws.data_ptr(), stream), "gh_patch_pool_bwd")
    # gh_patch_attn_bwd into guarded rows
    feat = torch.randn(L, b, e, device="cuda")
    params = [t.detach().contiguous() for t in ops._patch_attention_params(feat, a1, a2, cl)]
    d_emb, d_out = torch.randn(b, e, device="cuda"), torch.randn(b, nc, device="cuda")
    outs = [guarded(n) for n in (L * b * e, L * b * e, 2 * L * b * 3 * e, 2 * L * b * e, 2 * L * b * e)]
    _lib.check(lib.gh_patch_attn_bwd(feat.data_ptr(), *[t.data_ptr() for t in params[:9]], d_emb.data_ptr(), d_out.data_ptr(),
                                     L, b, e, 8, nc, *[v.data_ptr() for _, v in outs], stream), "gh_patch_attn_bwd")
    # gh_gemm_f32_fixed on both routes (tensor-core N >= 64, FMA kernel N < 64) and gh_colsum_f32
    x = torch.randn(48, 80, device="cuda")
    gemms = []
    for n in (80, 40):
        big, out = guarded(64 * n)
        _lib.check(lib.gh_gemm_f32_fixed(x.data_ptr(), 1, 80, x.data_ptr(), 80, 1, None, out.data_ptr(), n, 64, n, 48,
                                         stream), "gh_gemm_f32_fixed")
        gemms.append((big, out, n))
    big_cs, cs = guarded(80)
    _lib.check(lib.gh_colsum_f32(x.data_ptr(), 80, 48, 80, cs.data_ptr(), stream), "gh_colsum_f32")
    torch.cuda.synchronize()
    for big, view in [(big_ws, ws), *zip(bigs, grads), *outs, (big_cs, cs)] + [(g[0], g[1]) for g in gemms]:
        assert guards_intact(big) and bool(torch.isfinite(view).all())
    for big, out, n in gemms:
        assert rel(npf(out.view(64, n)), npf(x[:, :64].t() @ x[:, :n])) < 3e-5
    assert rel(npf(cs), npf(x.sum(0))) < 1e-6


def test_strided_and_channels_last_maps_give_the_same_gradient_in_their_layout():
    from heuristique_style_transfer_code_b200 import ops
    torch.manual_seed(5)
    base = [torch.randn(3, 64, 56, 56, device="cuda"), torch.randn(3, 64, 27, 27, device="cuda"),
            torch.randn(3, 64, 14, 14, device="cuda")]
    wide = [torch.randn(3, 64, h + 4, w + 6, device="cuda") for h, w in ((56, 56), (27, 27), (14, 14))]
    for wd, x in zip(wide, base):
        wd[:, :, 2:-2, 3:-3] = x
    variants = {"contiguous": base, "channels_last": [x.contiguous(memory_format=torch.channels_last) for x in base],
                "strided": [wd[:, :, 2:-2, 3:-3] for wd in wide]}
    dg = torch.randn(3, 3, 64 * 64, device="cuda")
    dn = torch.randn(3, 3, device="cuda")
    for ln_input in (True, False):
        grads = {}
        for name, maps in variants.items():
            maps = [m.detach().requires_grad_(True) for m in maps]
            gram, norm = ops.patch_gram_autograd(maps, ln_input)
            ((gram * dg).sum() + (norm * dn).sum()).backward()
            grads[name] = [m.grad for m in maps]
            if name == "channels_last":
                assert all(g.is_contiguous(memory_format=torch.channels_last) for g in grads[name])
            if name == "contiguous":
                assert all(g.is_contiguous() for g in grads[name])
        for name in ("channels_last", "strided"):
            for g, g0 in zip(grads[name], grads["contiguous"]):
                assert rel(npf(g), npf(g0)) < 1e-6, (name, ln_input)


def test_gradients_are_bitwise_reproducible():
    """The backward of one forward, run three times: the same bits. (Across forwards the values can differ in the last
    bits: the forward's feature_projection GEMM, gh_gemm_f32 with K = D*D, splits K over CTAs that meet in reduce-adds
    when the L*B rows fill fewer tiles than the GPU has SMs. Every backward GEMM runs on gh_gemm_f32_fixed.)"""
    torch.manual_seed(7)
    maps = [torch.randn(64, 64, h, w, device="cuda").requires_grad_(True) for h, w in ((112, 112), (56, 56), (28, 28), (14, 14))]
    a1, a2, cl, fp = make_head(64, 64, 10, 7)
    params = head_named_params(a1, a2, cl, fp)
    gram, norms, feat, emb, out = run_head_autograd(maps, a1, a2, cl, fp, True)
    ce, co, cn = cotangents(emb, out, norms)
    runs = []
    for _ in range(3):
        for t in [*maps, *params.values()]:
            t.grad = None
        torch.autograd.backward([emb, out, norms], [ce, co, cn], retain_graph=True)
        runs.append([t.grad.clone() for t in [*maps, *params.values()]])
    for again in runs[1:]:
        assert all(torch.equal(x, y) for x, y in zip(runs[0], again))


def test_an_image_gradient_does_not_depend_on_the_rest_of_the_batch():
    """Gradients of the first two images, from a batch of 64 and from those two alone, through each Function in turn
    from the same forward values: the same bits (the kernels work per image; the d_gram GEMM has K = ndf and is never
    split). The forward's feature_projection GEMM (gh_gemm_f32, K = D*D) may split K by batch size, so recomputing the
    forward on two images can move its values in the last bits; that is the one route that does."""
    from heuristique_style_transfer_code_b200 import ops
    torch.manual_seed(8)
    maps = [torch.randn(64, 64, h, w, device="cuda") for h, w in ((112, 112), (56, 56), (28, 28), (13, 13))]
    a1, a2, cl, fp = make_head(64, 64, 10, 8)
    g = torch.Generator(device="cuda").manual_seed(3)
    ce, co, cn = torch.randn(64, 64, device="cuda", generator=g), torch.randn(64, 10, device="cuda", generator=g), \
        torch.randn(4, 64, device="cuda", generator=g)
    with torch.no_grad():
        gram, _ = ops.patch_gram(maps)
        feat = ops.patch_projection_autograd(gram, fp)

    def attn(n):
        f = feat[:, :n].clone().requires_grad_(True)
        torch.autograd.backward(list(ops.patch_attention_autograd(f, a1, a2, cl)), [ce[:n], co[:n]])
        return f.grad

    def proj(n, d_feat):
        gr = gram[:, :n].clone().requires_grad_(True)
        ops.patch_projection_autograd(gr, fp).backward(d_feat[:, :n])
        return gr.grad

    def maps_grad(n, d_gram):
        ms = [m[:n].clone().requires_grad_(True) for m in maps]
        torch.autograd.backward(list(ops.patch_gram_autograd(ms)), [d_gram[:, :n], cn[:, :n]])
        return [m.grad for m in ms]

    d_feat = attn(64)
    assert torch.equal(d_feat[:, :2], attn(2))
    d_gram = proj(64, d_feat)
    assert torch.equal(d_gram[:, :2], proj(2, d_feat))
    for a, b in zip(maps_grad(64, d_gram), maps_grad(2, d_gram)):
        assert torch.equal(a[:2], b)


# ---- modules -----------------------------------------------------------------------------------------------------------
def no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def same_forward(e0, o0, n0, e1, o1, n1):
    """A grad-enabled forward runs the no-grad forward's kernels: the Gram norms are the same bits. Embeddings and
    output may differ in the last bits only because the feature_projection GEMM (gh_gemm_f32, K = D*D) splits K over
    CTAs that meet in reduce-adds, on both routes."""
    assert torch.equal(n0, n1.detach())
    assert rel(npf(e1), npf(e0)) < 1e-5 and rel(npf(o1), npf(o0)) < 1e-5


def module_grads(m, x, loss_fn):
    m.zero_grad(set_to_none=True)
    xg = x.detach().clone().requires_grad_(True)
    loss = loss_fn(xg)
    loss.backward()
    return xg.grad.clone(), {k: (p.grad.clone() if p.grad is not None else torch.zeros_like(p))
                             for k, p in m.named_parameters()}


def weighted(emb, out, norms, seed=11):
    g = torch.Generator(device="cuda").manual_seed(seed)
    loss = (emb * torch.randn(emb.shape, device="cuda", generator=g)).sum()
    loss = loss + (out * torch.randn(out.shape, device="cuda", generator=g)).sum()
    for n in norms:
        loss = loss + (n * torch.randn(n.shape, device="cuda", generator=g)).sum()
    return loss


def compare_module_grads(ours, port, tol=1e-3):
    errs = {"input": rel(npf(ours[0]), npf(port[0]))}
    errs.update({k: rel(npf(ours[1][k]), npf(port[1][k])) for k in ours[1]})
    worst = max(errs.items(), key=lambda kv: kv[1])
    print(f"\nworst relative gradient error {worst[0]}: {worst[1]:.2e}; input {errs['input']:.2e}")
    for k, v in errs.items():
        assert v < tol, (k, v)


@pytest.mark.parametrize("norm,patch", [("batch", 70), ("instance", 10), ("batch", 150)])
def test_discriminator_backward_matches_autograd_of_the_port(norm, patch):
    from heuristique_style_transfer_code_b200.patchgan import VariablePatchesNLayerDiscriminator_test
    no_tf32()
    torch.manual_seed(patch)
    m = VariablePatchesNLayerDiscriminator_test(ndf=64, norm=norm, patch_size=patch, num_classes=4, gram_matrix_dim=64).cuda()
    m.set_library_backward(True)
    x = torch.randn(4, 3, 224, 224, device="cuda")
    with torch.no_grad():
        e0, o0 = m(x)
        n0 = torch.stack(m.get_gram_norms())
    e1, o1 = m(x.clone().requires_grad_(True))
    assert e1.requires_grad and o1.requires_grad and m.get_gram_norms()[0].requires_grad
    same_forward(e0, o0, n0, e1, o1, torch.stack(m.get_gram_norms()))

    def ours(xg):
        e, o = m(xg)
        return weighted(e, o, m.get_gram_norms())

    def port(xg):
        return weighted(*patchgan_forward(m, xg))

    compare_module_grads(module_grads(m, x, ours), module_grads(m, x, port))


def test_multiscale_backward_matches_autograd_of_the_port_without_a_reference_copy():
    from heuristique_style_transfer_code_b200 import _reference
    from heuristique_style_transfer_code_b200.patchgan import MultiScaleDiscriminator_test
    no_tf32()
    torch.manual_seed(2)
    m = MultiScaleDiscriminator_test(ndf=64, norm='batch', num_classes=4, gram_matrix_dim=64).cuda().set_library_backward()
    x = torch.randn(2, 3, 224, 224, device="cuda")
    saved_root, saved_loaded = _reference.reference_root, dict(_reference._LOADED)
    try:
        _reference.reference_root = lambda rel_path: None       # no copy of the reference: grad mode still works
        _reference._LOADED.clear()
        with torch.no_grad():
            e0, o0 = m(x)
            n0 = torch.stack(m.get_gram_norms())
        e1, o1 = m(x)
        assert e1.requires_grad
        same_forward(e0, o0, n0, e1, o1, torch.stack(m.get_gram_norms()))

        def ours(xg):
            e, o = m(xg)
            return weighted(e, o, m.get_gram_norms())

        got = module_grads(m, x, ours)
    finally:
        _reference.reference_root = saved_root
        _reference._LOADED.update(saved_loaded)

    def port(xg):
        norms = []
        embs, outs = [], []
        for d in m.scale_discriminators.values():
            e, o, n = patchgan_forward(d, xg)
            embs.append(e)
            outs.append(o)
            norms.extend(n)
        return weighted(torch.stack(embs, 0).mean(0), torch.stack(outs, 0).mean(0), norms)

    compare_module_grads(got, module_grads(m, x, port))


def test_nan_pixel_gives_the_ports_messages_and_gradients(capsys):
    from heuristique_style_transfer_code_b200.patchgan import VariablePatchesNLayerDiscriminator_test
    no_tf32()
    torch.manual_seed(9)
    m = VariablePatchesNLayerDiscriminator_test(ndf=32, norm='batch', patch_size=30, num_classes=3,
                                                gram_matrix_dim=32).cuda().set_library_backward()
    x = torch.randn(2, 3, 64, 64, device="cuda")
    x[1, 0, 5, 7] = float("nan")

    def ours(xg):
        e, o = m(xg)
        return weighted(e, o, m.get_gram_norms())

    def port(xg):
        return weighted(*patchgan_forward(m, xg))

    got = module_grads(m, x, ours)
    ours_msgs = capsys.readouterr().out
    want = module_grads(m, x, port)
    port_msgs = capsys.readouterr().out
    assert "NaN detected after layer 0" in ours_msgs and ours_msgs == port_msgs
    assert torch.isfinite(got[0]).all()
    # the first convolution's weight gradient is NaN on both routes (the NaN pixel times a zeroed gradient); everything
    # else is finite and must agree
    for k in got[1]:
        assert torch.equal(torch.isnan(got[1][k]), torch.isnan(want[1][k])), k
        got[1][k] = torch.nan_to_num(got[1][k], nan=0.0)
        want[1][k] = torch.nan_to_num(want[1][k], nan=0.0)
    compare_module_grads(got, want)


def test_adam_on_a_noise_image_lowers_the_loss():
    """What style_transfer_patches (functions_Multi_PatchGAN.py:272-287) does: optimise an image through the
    discriminator. Where the reference copy is staged, the first step's image gradient matches its own forward's."""
    from heuristique_style_transfer_code_b200 import _reference
    from heuristique_style_transfer_code_b200.patchgan import MultiScaleDiscriminator_test
    no_tf32()
    torch.manual_seed(4)
    m = MultiScaleDiscriminator_test(ndf=64, norm='batch', num_classes=4, gram_matrix_dim=64).cuda().eval()
    m.set_library_backward(True)
    for p in m.parameters():
        p.requires_grad_(False)
    target = torch.tensor([1, 3], device="cuda")
    img = torch.rand(2, 3, 128, 128, device="cuda").requires_grad_(True)
    start = img.detach().clone()
    opt = torch.optim.Adam([img], lr=0.02)
    losses, first_grad = [], None
    for step in range(6):
        opt.zero_grad()
        emb, out = m(img)
        loss = torch.nn.functional.cross_entropy(out, target)
        loss.backward()
        if step == 0:
            first_grad = img.grad.clone()
        losses.append(float(loss))
        opt.step()
    print(f"\nAdam losses: {[round(v, 4) for v in losses]}")
    assert losses[-1] < losses[0]
    if _reference.reference_root(os.path.join("Models", "Models_Multi_PatchGAN.py")) is not None:
        m.set_library_backward(False)
        img0 = start.requires_grad_(True)
        _, out = m(img0)
        torch.nn.functional.cross_entropy(out, target).backward()
        err = rel(npf(first_grad), npf(img0.grad))
        print(f"first-step image gradient against the reference's forward: {err:.2e}")
        assert err < 1e-3
