"""Resize + CenterCrop of loader batches on the GPU, the parts that need no GPU: the C-ABI validation of gh_frame_tables
(which returns before any CUDA call), the per-image geometry against torchvision, the band-height bound against the exact
band_span, the worker-side packing (functions.gpu_resize_transform / PackedImages), the refusals, and cuda_prefetch's CPU
path against the reference transform."""
import ctypes

import numpy as np
import pytest
import torch
from PIL import Image

from heuristique_style_transfer_code_b200 import _lib
from heuristique_style_transfer_code_b200 import functions as F
from heuristique_style_transfer_code_b200 import streaming as S
from heuristique_style_transfer_code_b200._lib import GramHeadError
from heuristique_style_transfer_code_b200.build import build_library

MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]


@pytest.fixture(scope="module")
def library():
    build_library()
    return _lib.lib()


def _images(seed, shapes):
    rng = np.random.default_rng(seed)
    return [Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), "RGB") for h, w in shapes]


def test_argument_validation_without_gpu(library):
    d = ctypes.c_void_p(256)
    BAD, UNS = _lib.GH_ERR_BAD_ARG, _lib.GH_ERR_UNSUPPORTED
    f = library.gh_frame_tables
    #       geom N  base OH   OW  hk vk tables frames stream
    assert f(None, 2, d, 224, 224, 9, 5, d, d, None) == BAD
    assert f(d, 2, None, 224, 224, 9, 5, d, d, None) == BAD
    assert f(d, 2, d, 224, 224, 9, 5, None, d, None) == BAD
    assert f(d, 2, d, 224, 224, 9, 5, d, None, None) == BAD
    assert f(d, 0, d, 224, 224, 9, 5, d, d, None) == BAD                     # N <= 0
    assert f(d, -3, d, 224, 224, 9, 5, d, d, None) == BAD
    assert f(d, 2, d, 0, 224, 9, 5, d, d, None) == BAD                       # OH <= 0
    assert f(d, 2, d, 224, -1, 9, 5, d, d, None) == BAD                      # OW <= 0
    assert f(d, 2, d, 224, 224, 0, 5, d, d, None) == BAD                     # hkmax <= 0
    assert f(d, 2, d, 224, 224, 9, 0, d, d, None) == BAD                     # vkmax <= 0
    assert f(d, 65536, d, 224, 224, 9, 5, d, d, None) == UNS                 # gridDim.y
    assert f(d, 2, d, 2**31 - 1, 2**31 - 1, 9, 5, d, d, None) == UNS         # output coordinates beyond one grid row
    q = library.gh_frame_tables_stride
    assert q(224, 224, 9, 5) == 224 * (2 + 9) + 224 * (2 + 5)
    assert q(3, 7, 1, 33) == 7 * 3 + 3 * 35
    assert q(0, 224, 9, 5) == BAD and q(224, 224, 9, 0) == BAD


@pytest.mark.parametrize("resize,crop", [(256, 224), (256, 225), ((300, 200), (250, 151)), (224, (224, 200))])
def test_geometry_is_torchvision(resize, crop):
    from torchvision import transforms
    # landscape, portrait, square, odd sides, one side already at the target, and an upscale
    shapes = [(300, 400), (400, 300), (256, 256), (333, 517), (256, 341), (341, 256), (100, 150), (1, 700), (700, 1)]
    shapes = [s for s in shapes if min(s) > 1 or isinstance(resize, tuple)]
    images = _images(0, shapes)
    geometry, (oh, ow) = S.frame_geometry([(h, w, 3) for h, w in shapes], resize, crop)
    odd = 0
    for img, (h, w, rh, rw, top, left, gh, gw) in zip(images, geometry):
        resized = transforms.Resize(resize)(img)
        assert (h, w) == (img.height, img.width) and (rw, rh) == resized.size and (gh, gw) == (oh, ow)
        want = np.asarray(transforms.CenterCrop(crop)(resized))
        assert np.array_equal(np.asarray(resized)[top:top + oh, left:left + ow], want)
        odd += (rh - oh) % 2 + (rw - ow) % 2
    assert odd > 0                                          # a centre offset of x.5, rounded half to even


def test_span_bound_covers_band_span():
    rng = np.random.default_rng(3)
    for _ in range(300):
        h, w = int(rng.integers(1, 3000)), int(rng.integers(1, 3000))
        resize = int(rng.integers(8, 400)) if rng.random() < 0.7 else (int(rng.integers(8, 400)), int(rng.integers(8, 400)))
        try:
            packed = S.pack_frame_tables([(h, w, 3)], resize, crop=None)
        except GramHeadError:
            continue
        ((_, _, rh, _, _, _, oh, _),), _ = S.frame_geometry([(h, w, 3)], resize)
        rows = np.unique(np.r_[1, 2, 3, rng.integers(1, oh + 1, 4), oh])
        bounds = S.band_span_bound([h], [rh], rows)
        for r, bound in zip(rows, bounds):
            assert bound >= S.band_span(packed["rows"], int(r)), (h, w, resize, r)
            assert bound == S.band_span_bound([h], [rh], int(r))
    # several images: the largest bound of any of them
    assert S.band_span_bound([4000, 300], [256, 256], 5) == max(S.band_span_bound([4000], [256], 5),
                                                               S.band_span_bound([300], [256], 5))


def test_collate_packs_offsets_shapes_and_labels():
    t = F.gpu_resize_transform(256, 224)
    shapes = [(300, 400), (517, 333), (256, 256), (1200, 1600)]
    images = _images(1, shapes)
    batch = [(t(img), label) for img, label in zip(images, [3, 0, 2, 1])]
    assert all(x.shape == (h, w, 3) and x.dtype == torch.uint8 for x, (h, w) in zip([b[0] for b in batch], shapes))
    packed = t.collate(batch)
    assert isinstance(packed, F.PackedImages) and len(packed) == 4
    assert packed.labels.tolist() == [3, 0, 2, 1] and packed.labels.dtype == torch.int64
    assert packed.out_hw == (224, 224) and packed.pixels.numel() == sum(h * w * 3 for h, w in shapes)
    g = packed.geometry
    assert g.dtype == torch.int64 and g.shape == (4, len(S.GEOMETRY_COLUMNS))
    offsets = np.concatenate([[0], np.cumsum([h * w * 3 for h, w in shapes])[:-1]])
    assert g[:, 0].tolist() == [h for h, _ in shapes] and g[:, 1].tolist() == [w for _, w in shapes]
    assert g[:, 2].tolist() == offsets.tolist()
    want = S.frame_geometry([(h, w, 3) for h, w in shapes], 256, 224)[0]
    assert g[:, 3:].tolist() == [[rh, rw, top, left] for _, _, rh, rw, top, left, _, _ in want]
    assert packed.kmax == (max(S.resample_kmax(w, r[3]) for (_, w), r in zip(shapes, want)),
                           max(S.resample_kmax(h, r[2]) for (h, _), r in zip(shapes, want)))
    for img, view in zip(images, packed.images()):
        assert np.array_equal(np.asarray(img), view)


def test_unsupported_transforms_are_refused():
    from torchvision.transforms import InterpolationMode
    for kwargs in (dict(interpolation="nearest"), dict(interpolation=InterpolationMode.BICUBIC), dict(max_size=512),
                   dict(resize=200, crop=224), dict(resize=(224, 180), crop=200), dict(resize=256, crop=None),
                   dict(resize=None), dict(resize=0), dict(crop=0)):
        with pytest.raises(ValueError):
            F.gpu_resize_transform(**kwargs)
    F.gpu_resize_transform((224, 300), None)                # one output size without a crop
    F.gpu_resize_transform(interpolation=InterpolationMode.BILINEAR)
    with pytest.raises(ValueError):
        F.gpu_resize_transform()(Image.new("L", (300, 300)))


def test_resample_images_checks_before_any_cuda_call():
    # CPU tensors: every check below fails before the device is touched
    geometry = torch.tensor([[300, 400, 0, 256, 341, 16, 58]], dtype=torch.int64)
    pixels = torch.zeros(300 * 400 * 3, dtype=torch.uint8)
    out = torch.empty((1, 3, 224, 224), dtype=torch.uint8)
    bad = geometry.clone()
    bad[0, 2] = 1                                                           # pixels past the end of the buffer
    with pytest.raises(GramHeadError):
        S.resample_images(pixels, bad, bad.numpy(), out, 5, 5)
    bad = geometry.clone()
    bad[0, 5] = 40                                                          # crop past the resized image
    with pytest.raises(GramHeadError):
        S.resample_images(pixels, bad, bad.numpy(), out, 5, 5)
    with pytest.raises(GramHeadError):
        S.resample_images(pixels, geometry, geometry.numpy(), out, 4, 5)    # hkmax below the image's 5
    with pytest.raises(GramHeadError):
        S.resample_images(pixels, geometry, geometry.numpy(), out[:, :2], 5, 5)


@pytest.mark.parametrize("normalize", ["default", None])
def test_cpu_prefetch_is_the_reference_transform(normalize):
    from torchvision import transforms
    shapes = [(300, 400), (517, 333), (256, 341), (120, 90), (2, 300), (801, 1200)]
    images = _images(2, shapes)
    labels = [1, 0, 3, 2, 1, 0]
    t = F.gpu_resize_transform(256, 224)
    packed = [t.collate([(t(img), lab) for img, lab in zip(images[i:i + 3], labels[i:i + 3])]) for i in (0, 3)]
    got = list(F.cuda_prefetch(packed, "cpu", normalize=normalize))
    if normalize is None:
        ref = transforms.Compose([transforms.Resize(256), transforms.CenterCrop(224), transforms.PILToTensor()])
    else:
        ref = transforms.Compose([transforms.Resize(256), transforms.CenterCrop(224), transforms.ToTensor(),
                                  transforms.Normalize(MEAN, STD)])
    for k, (x, y) in enumerate(got):
        want = torch.stack([ref(img) for img in images[3 * k:3 * k + 3]])
        assert x.dtype == want.dtype and torch.equal(x, want)
        assert y.tolist() == labels[3 * k:3 * k + 3]
