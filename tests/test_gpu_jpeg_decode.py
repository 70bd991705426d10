"""GPU: baseline JPEG decoding on the device (gh_jpeg_decode behind functions.gpu_resize_transform(decode="gpu")):
every image of the seeded corpus equal to Pillow byte for byte at several subsequence sizes of the parallel Huffman
decoder, batch independence, guard bytes, mixed batches with worker-decoded files, reused buffers, a truncated scan
reported by batch index, and the train / evaluation loops against host-transform loaders.

The bitwise comparisons of model outputs run with ops.KSPLIT = 1: Gram launches may otherwise split K over fp32 atomics,
whose order (and so the last bits) changes from run to run."""
import io

import numpy as np
import pytest
import torch
from PIL import Image

import jpeg_corpus as C
from heuristique_style_transfer_code_b200 import functions as F
from heuristique_style_transfer_code_b200 import jpeg
from heuristique_style_transfer_code_b200._lib import GramHeadError

pytestmark = pytest.mark.gpu

MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
CORPUS = C.corpus()


def test_cuda_is_present():
    assert torch.cuda.is_available()


def _decode(datas, subseq=jpeg.SUBSEQ_BYTES, guard=4096):
    """Decodes the files into one arena with guard bytes around it; returns (images, status, guards intact)."""
    files = [jpeg.parse(d) for d in datas]
    assert all(f is not None for f in files)
    sizes = [f.H * f.W * 3 for f in files]
    offsets = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
    scan, segs, imgs, tables = jpeg.pack(files, offsets, list(range(len(files))))
    total = int(sum(sizes))
    buf = torch.full((total + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda")
    arena = buf[guard:guard + total]
    status = jpeg.decode_batch(scan.cuda(), segs.cuda(), imgs.cuda(), tables.cuda(), imgs.numpy(), segs.numpy(), arena,
                               total, subseq=subseq)
    host = buf.cpu().numpy()
    intact = bool((host[:guard] == 0xA5).all() and (host[guard + total:] == 0xA5).all())
    flat = host[guard:guard + total]
    out = [flat[o:o + s].reshape(f.H, f.W, 3) for f, o, s in zip(files, offsets, sizes)]
    return out, status.cpu().numpy(), intact


@pytest.mark.parametrize("subseq", [1, 5, 64, jpeg.SUBSEQ_BYTES, 1 << 20])
def test_device_is_pillow(subseq):
    names = [n for n, _ in CORPUS]
    got, status, intact = _decode([d for _, d in CORPUS], subseq=subseq)
    assert intact and not status.any()
    bad = [n for n, g, (_, d) in zip(names, got, CORPUS) if not np.array_equal(g, C.pillow(d))]
    assert not bad, bad


def test_batch_independence():
    rng = np.random.default_rng(4)
    datas = []
    for k in range(64):
        h, w = (int(v) for v in rng.integers(8, 700, 2))
        kind = C.KINDS[k % len(C.KINDS)]
        img = C.content(kind, h, w, rng)
        datas.append(C._save(img, "L" if k % 7 == 0 else "RGB", quality=int(rng.integers(30, 100)),
                             subsampling=int(rng.integers(0, 3)), restart_marker_blocks=int(k % 3) * 2))
    together, status, intact = _decode(datas, subseq=32)
    assert intact and not status.any()
    for k in (0, 1, 7, 33, 63):
        alone, st, ok = _decode([datas[k]], subseq=32)
        assert ok and not st.any() and np.array_equal(alone[0], together[k])
        assert np.array_equal(alone[0], C.pillow(datas[k]))


def test_truncated_scan_is_reported_by_batch_index(tmp_path):
    good = C._save(C.content("noise", 64, 80, np.random.default_rng(1)), quality=90)
    hdr_end = good.index(b"\xff\xda")
    cut = good[:hdr_end + (len(good) - hdr_end) // 2] + b"\xff\xd9"
    assert jpeg.parse(cut) is not None
    out, status, intact = _decode([good, cut, good])
    assert intact and status.tolist()[0] == 0 and status[1] != 0 and status[2] == 0
    # the broken image leaves its neighbours in the arena alone
    assert np.array_equal(out[0], C.pillow(good)) and np.array_equal(out[2], C.pillow(good))
    t = F.gpu_resize_transform(48, 40, decode="gpu")
    paths = []
    for i, d in enumerate([good, good, cut]):
        p = tmp_path / f"{i}.jpg"
        p.write_bytes(d)
        paths.append(str(p))
    batch = t.collate([(t(t.loader(p)), i) for i, p in enumerate(paths)]).pin_memory()
    with pytest.raises(GramHeadError, match="batch index 2"):
        list(F.cuda_prefetch([batch], "cuda", normalize=None))


def _files(tmp_path, seed, shapes, png_every=4):
    """JPEG files of several kinds (some the worker decodes: progressive, CMYK) and PNGs."""
    rng = np.random.default_rng(seed)
    paths = []
    for i, (h, w) in enumerate(shapes):
        img = C.content(C.KINDS[i % len(C.KINDS)], h, w, rng)
        p = tmp_path / f"{seed}_{i}"
        if i % png_every == png_every - 1:
            p = p.with_suffix(".png")
            Image.fromarray(img).save(p)
        elif i % 5 == 2:
            p = p.with_suffix(".jpg")
            Image.fromarray(img).save(p, "JPEG", progressive=True)
        elif i % 11 == 5:
            p = p.with_suffix(".jpg")
            Image.fromarray(img).convert("CMYK").save(p, "JPEG")
        else:
            p = p.with_suffix(".jpg")
            Image.fromarray(img).convert("L" if i % 6 == 1 else "RGB").save(p, "JPEG", quality=int(rng.integers(40, 98)),
                                                                            subsampling=i % 3)
        paths.append(str(p))
    return paths


def test_mixed_batches_and_reused_buffers(tmp_path):
    from torchvision import transforms
    from torchvision.datasets.folder import default_loader
    ref = transforms.Compose([transforms.Resize(256), transforms.CenterCrop(224), transforms.PILToTensor()])
    t = F.gpu_resize_transform(256, 224, decode="gpu")
    plan = [[(300, 400), (257, 300), (400, 260)], [(1500, 2000), (1200, 1600), (2000, 1400), (999, 1001), (640, 480),
                                                   (700, 500), (333, 517), (260, 260), (900, 300), (300, 900),
                                                   (512, 512), (480, 640)],
            [(300, 400), (401, 299)], [(1100, 900)] * 3]
    batches = [_files(tmp_path, 10 + k, s) for k, s in enumerate(plan)]
    assert any(isinstance(t.loader(p), jpeg.JpegFile) for p in batches[1])
    assert not all(isinstance(t.loader(p), jpeg.JpegFile) for p in batches[1])
    for reuse in (False, True):
        packed = [t.collate([(t(t.loader(p)), i) for i, p in enumerate(b)]).pin_memory() for b in batches]
        got = [x.clone() for x, _ in F.cuda_prefetch(packed, "cuda", reuse_buffers=reuse, normalize=None)]
        assert len(got) == len(plan)
        for x, paths in zip(got, batches):
            assert torch.equal(x.cpu(), torch.stack([ref(default_loader(p)) for p in paths])), reuse


@pytest.fixture(scope="module")
def kernels_deterministic():
    from heuristique_style_transfer_code_b200 import ops
    saved, ops.KSPLIT = ops.KSPLIT, 1
    yield
    ops.KSPLIT = saved


@pytest.fixture(scope="module")
def image_folder(tmp_path_factory):
    root = tmp_path_factory.mktemp("jpeg_images")
    rng = np.random.default_rng(21)
    shapes = [(300, 400), (517, 333), (256, 341), (341, 256), (120, 90), (1200, 1600), (999, 1001), (224, 224),
              (801, 533), (300, 300), (450, 800), (257, 256), (1000, 750), (333, 517), (612, 408), (350, 700), (287, 301)]
    for i, (h, w) in enumerate(shapes):
        d = root / f"class_{i % 3}"
        d.mkdir(exist_ok=True)
        img = Image.fromarray(C.content(C.KINDS[i % len(C.KINDS)], h, w, rng), "RGB")
        if i % 6 == 5:
            img.save(d / f"img_{i:03d}.png")
        elif i % 6 == 4:
            img.save(d / f"img_{i:03d}.jpg", "JPEG", progressive=True)
        else:
            img.save(d / f"img_{i:03d}.jpg", "JPEG", quality=75 + i, subsampling=i % 3)
    return str(root)


def _loaders(root, host_transform, batch_size=8):
    from torch.utils.data import DataLoader
    from torchvision.datasets import ImageFolder
    t = F.gpu_resize_transform(256, 224, decode="gpu")
    gpu = DataLoader(ImageFolder(root, loader=t.loader, transform=t), batch_size=batch_size, shuffle=False,
                     num_workers=2, pin_memory=True, collate_fn=t.collate)
    host = DataLoader(ImageFolder(root, transform=host_transform), batch_size=batch_size, shuffle=False, num_workers=2,
                      pin_memory=True)
    return gpu, host


def _model(cls, train=False):
    from torchvision import models
    import heuristique_style_transfer_code_b200 as pkg
    torch.manual_seed(0)
    m = getattr(pkg, cls)(models.resnet50(weights=None), 7, 4, 32, device="cuda")
    return m.train() if train else m.eval()


def _host_tf():
    from torchvision import transforms
    return transforms.Compose([transforms.Resize(256), transforms.CenterCrop(224), transforms.ToTensor(),
                               transforms.Normalize(MEAN, STD)])


def test_evaluate_model_test_is_the_host_loader(image_folder, kernels_deterministic):
    m = _model("TruncatedResNet50_for_test")
    gpu, host = _loaders(image_folder, _host_tf())
    got = F.evaluate_model_test(m, gpu, "cuda")
    want = F.evaluate_model_test(m, host, "cuda")
    assert got[4] == want[4] and len(got[4]) == len(gpu.dataset)
    for a, b in zip(got[:4], want[:4]):
        assert a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a, b)


def test_evaluate_model_and_train_model_are_the_host_loader(image_folder, kernels_deterministic):
    from torch.utils.data import DataLoader, Subset
    from torchvision.datasets import ImageFolder
    gpu, host = _loaders(image_folder, _host_tf())
    m = _model("TruncatedResNet50")
    crit = torch.nn.CrossEntropyLoss()
    assert F.evaluate_model(m, gpu, crit) == F.evaluate_model(m, host, crit)
    t = F.gpu_resize_transform(256, 224, decode="gpu")
    first = list(range(8))
    losses = {}
    for name, loader in (("gpu", DataLoader(Subset(ImageFolder(image_folder, loader=t.loader, transform=t), first),
                                            batch_size=8, collate_fn=t.collate, pin_memory=True)),
                         ("host", DataLoader(Subset(ImageFolder(image_folder, transform=_host_tf()), first),
                                             batch_size=8, pin_memory=True))):
        model = _model("TruncatedResNet50", train=True)
        seen = []

        def record(out, y):
            loss = crit(out, y)
            seen.append(loss.detach().clone())
            return loss
        F.train_model(model, loader, record, torch.optim.SGD(model.parameters(), lr=0.01), num_epochs=1)
        losses[name] = seen
    assert len(losses["gpu"]) == len(losses["host"]) == 1
    assert torch.equal(losses["gpu"][0], losses["host"][0])
