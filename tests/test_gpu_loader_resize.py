"""GPU: Resize + CenterCrop of loader batches on the device (gh_frame_tables + gh_preprocess_frames behind
functions.gpu_resize_transform and cuda_prefetch): the device tables against streaming.pack_frame_tables bit for bit, the
resampled batches against torchvision on the PIL images, and the train / evaluation loops against host-transform loaders.

The bitwise comparisons of model outputs run with ops.KSPLIT = 1: Gram launches may otherwise split K over fp32 atomics,
whose order (and so the last bits) changes from run to run."""
import copy

import numpy as np
import pytest
import torch
from PIL import Image

from heuristique_style_transfer_code_b200 import _lib
from heuristique_style_transfer_code_b200 import functions as F
from heuristique_style_transfer_code_b200 import streaming as S

pytestmark = pytest.mark.gpu

MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
# one axis already at 256 (the common case under Resize(256)); downscales from ~1x to 16x and beyond; upscales; 1 x N and
# N x 1; a 40 x 3000 strip; odd sides
TABLE_SHAPES = [(256, 341), (341, 256), (300, 400), (480, 640), (1080, 1920), (4096, 3072), (3000, 4000), (100, 150),
                (224, 224), (1, 300), (300, 1), (40, 3000), (333, 517), (1999, 2001), (257, 256)]
GEOMETRIES = [(256, 224), ((224, 224), None), ((448, 300), (400, 299))]
IMAGE_SHAPES = [(300, 400), (517, 333), (256, 341), (341, 256), (120, 90), (1200, 1600), (2, 300), (999, 1001), (224, 224)]


def test_cuda_is_present():
    assert torch.cuda.is_available()


@pytest.fixture(scope="module")
def kernels_deterministic():
    from heuristique_style_transfer_code_b200 import ops
    saved, ops.KSPLIT = ops.KSPLIT, 1
    yield
    ops.KSPLIT = saved


def _rgb(seed, shapes):
    rng = np.random.default_rng(seed)
    return [Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), "RGB") for h, w in shapes]


@pytest.mark.parametrize("resize,crop", GEOMETRIES)
@pytest.mark.parametrize("pad", [0, 3])
def test_device_tables_are_pack_frame_tables(resize, crop, pad):
    shapes = [(h, w, 3) for h, w in TABLE_SHAPES]
    packed = S.pack_frame_tables(shapes, resize, crop)
    geometry, (oh, ow) = S.frame_geometry(shapes, resize, crop)
    sizes = [h * w * 3 for h, w, _ in shapes]
    offsets = np.concatenate([[0], np.cumsum(sizes)[:-1]])
    geom = torch.tensor([(h, w, int(o), rh, rw, top, left) for (h, w, rh, rw, top, left, _, _), o in zip(geometry, offsets)],
                        dtype=torch.int64, device="cuda")
    hk, vk = packed["hkmax"] + pad, packed["vkmax"] + pad
    n, lib = len(shapes), _lib.lib()
    stride = lib.gh_frame_tables_stride(oh, ow, hk, vk)
    base = torch.empty(16, dtype=torch.uint8, device="cuda")          # only its address goes into the descriptors
    guard = 1024
    tables = torch.full((n * stride + 2 * guard,), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
    frames = torch.full((n * 80 + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda")
    _lib.check(lib.gh_frame_tables(geom.data_ptr(), n, base.data_ptr(), oh, ow, hk, vk, tables[guard:].data_ptr(),
                                   frames[guard:].data_ptr(), None), "gh_frame_tables")
    torch.cuda.synchronize()
    got = tables.cpu().numpy()
    assert (got[:guard] == 0x5A5A5A5A).all() and (got[-guard:] == 0x5A5A5A5A).all()
    got = got[guard:-guard]
    desc = frames.cpu().numpy()
    assert (desc[:guard] == 0xA5).all() and (desc[-guard:] == 0xA5).all()
    desc = desc[guard:-guard].view(S.FRAME_DESC_DTYPE)
    want = packed["tables"]
    for i, (h, w, _) in enumerate(shapes):
        o = packed["offsets"][i]
        mine = got[i * stride:(i + 1) * stride]
        fields = [(ow, 1), (ow, 1), (ow, packed["hkmax"]), (oh, 1), (oh, 1), (oh, packed["vkmax"])]
        pos = 0
        for j, (count, width) in enumerate(fields):
            ref = want[o[j]:o[j] + count * width].reshape(count, width)
            padded = pad if width > 1 else 0
            part = mine[pos:pos + count * (width + padded)].reshape(count, width + padded)
            assert np.array_equal(part[:, :width], ref), (i, h, w, S._TABLE_FIELDS[j])
            assert not part[:, width:].any()                                      # zero padding of coefficient rows
            assert desc[S._TABLE_FIELDS[j]][i] == i * stride + pos
            pos += count * (width + padded)
        assert pos == stride
        d = desc[i]
        assert (d["frame"], d["pitch"], d["H"], d["W"], d["bgr"], d["reserved"]) == \
            (base.data_ptr() + offsets[i], 3 * w, h, w, 0, 0)
    # every image whose kmax is below the batch's has zero-padded rows in the unpadded layout as well
    assert pad or any(S.resample_kmax(w, g[3]) < packed["hkmax"] for (h, w, _), g in zip(shapes, geometry))


def _packed(t, images, labels=None):
    labels = list(range(len(images))) if labels is None else labels
    return t.collate([(t(img), lab) for img, lab in zip(images, labels)]).pin_memory()


def test_batches_are_bitwise_torchvision():
    from torchvision import transforms
    images = _rgb(5, IMAGE_SHAPES)
    t = F.gpu_resize_transform(256, 224)
    u8 = transforms.Compose([transforms.Resize(256), transforms.CenterCrop(224), transforms.PILToTensor()])
    fp32 = transforms.Compose([transforms.Resize(256), transforms.CenterCrop(224), transforms.ToTensor(),
                               transforms.Normalize(MEAN, STD)])
    for normalize, ref in ((None, u8), ("default", fp32)):
        for reuse in (False, True):
            (x, y), = [(a.clone(), b.clone()) for a, b in
                       F.cuda_prefetch([_packed(t, images)], "cuda", reuse_buffers=reuse, normalize=normalize)]
            want = torch.stack([ref(img) for img in images])
            assert x.dtype == want.dtype and torch.equal(x.cpu(), want), (normalize, reuse)
            assert y.tolist() == list(range(len(images)))
    # a transform with a pair resize and no crop, through the same path
    t2 = F.gpu_resize_transform((200, 300), None)
    (x, _), = [(a.clone(), b) for a, b in F.cuda_prefetch([_packed(t2, images)], "cuda", normalize=None)]
    ref2 = transforms.Compose([transforms.Resize((200, 300)), transforms.PILToTensor()])
    assert torch.equal(x.cpu(), torch.stack([ref2(img) for img in images]))


def test_reused_buffers_hold_no_stale_data():
    from torchvision import transforms
    t = F.gpu_resize_transform(256, 224)
    ref = transforms.Compose([transforms.Resize(256), transforms.CenterCrop(224), transforms.PILToTensor()])
    small, big, mid = [(300, 400), (257, 300), (400, 260)], [(1500, 2000), (1200, 1600), (2000, 1400), (999, 1001)], \
        [(700, 500), (640, 480)]
    plan = [small, big, small, big, mid, small]                  # the pixel bytes grow, shrink, grow, shrink
    batches = [_rgb(10 + k, s) for k, s in enumerate(plan)]
    got = [x.clone() for x, _ in F.cuda_prefetch([_packed(t, b) for b in batches], "cuda", reuse_buffers=True,
                                                 normalize=None)]
    assert len(got) == len(plan)
    for x, imgs in zip(got, batches):
        assert torch.equal(x.cpu(), torch.stack([ref(img) for img in imgs]))


@pytest.fixture(scope="module")
def image_folder(tmp_path_factory):
    root = tmp_path_factory.mktemp("images")
    rng = np.random.default_rng(21)
    shapes = IMAGE_SHAPES[:6] + [(999, 1001), (224, 224), (801, 533), (300, 300), (450, 800), (257, 256), (1000, 750),
                                 (333, 517), (612, 408), (350, 700), (287, 301)]
    for i, (h, w) in enumerate(shapes):
        d = root / f"class_{i % 3}"
        d.mkdir(exist_ok=True)
        Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), "RGB").save(d / f"img_{i:03d}.png")
    return str(root)


def _loaders(root, host_transform, batch_size=8, **kw):
    from torch.utils.data import DataLoader
    from torchvision.datasets import ImageFolder
    t = F.gpu_resize_transform(256, 224)
    gpu = DataLoader(ImageFolder(root, transform=t), batch_size=batch_size, shuffle=False, num_workers=2,
                     pin_memory=True, collate_fn=t.collate, **kw)
    host = DataLoader(ImageFolder(root, transform=host_transform), batch_size=batch_size, shuffle=False, num_workers=2,
                      pin_memory=True, **kw)
    return gpu, host


def _model(cls, train=False):
    from torchvision import models
    import heuristique_style_transfer_code_b200 as pkg
    torch.manual_seed(0)
    m = getattr(pkg, cls)(models.resnet50(weights=None), 7, 4, 32, device="cuda")
    return m.train() if train else m.eval()


@pytest.mark.parametrize("inside", [False, True])
def test_evaluate_model_test_is_the_host_loader(image_folder, kernels_deterministic, inside):
    from torchvision import transforms
    m = _model("TruncatedResNet50_for_test")
    if inside:            # the model normalises its uint8 input itself (fused uint8 stem); the host loader hands uint8
        m.set_input_normalization(F.IMAGENET_MEAN, F.IMAGENET_STD)
        host_tf = F.uint8_transform(256, 224)
    else:
        host_tf = transforms.Compose([transforms.Resize(256), transforms.CenterCrop(224), transforms.ToTensor(),
                                      transforms.Normalize(MEAN, STD)])
    gpu, host = _loaders(image_folder, host_tf)
    got = F.evaluate_model_test(m, gpu, "cuda")
    want = F.evaluate_model_test(m, host, "cuda")
    assert got[4] == want[4] and len(got[4]) == len(gpu.dataset)
    for a, b in zip(got[:4], want[:4]):
        assert a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a, b)


def test_evaluate_model_and_train_model_are_the_host_loader(image_folder, kernels_deterministic):
    from torch.utils.data import Subset
    from torchvision import transforms
    host_tf = transforms.Compose([transforms.Resize(256), transforms.CenterCrop(224), transforms.ToTensor(),
                                  transforms.Normalize(MEAN, STD)])
    gpu, host = _loaders(image_folder, host_tf)
    m = _model("TruncatedResNet50")
    crit = torch.nn.CrossEntropyLoss()
    assert F.evaluate_model(m, gpu, crit) == F.evaluate_model(m, host, crit)

    from torch.utils.data import DataLoader
    from torchvision.datasets import ImageFolder
    t = F.gpu_resize_transform(256, 224)
    first = list(range(8))
    losses = {}
    for name, loader in (("gpu", DataLoader(Subset(ImageFolder(image_folder, transform=t), first), batch_size=8,
                                            collate_fn=t.collate, pin_memory=True)),
                         ("host", DataLoader(Subset(ImageFolder(image_folder, transform=host_tf), first), batch_size=8,
                                             pin_memory=True))):
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
