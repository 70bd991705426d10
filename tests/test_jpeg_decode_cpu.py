"""CPU side of decode="gpu" (functions.gpu_resize_transform, jpeg.py): which files the device decodes and which the
worker decodes, the parsed header against Pillow's, the unstuffed restart segments against the oracle's, the CPU path of
the batches against torchvision, construction errors, and the C ABI's host-only queries and refusals."""
import io

import numpy as np
import pytest
import torch
from PIL import Image

import jpeg_corpus as C
from heuristique_style_transfer_code_b200 import _lib, jpeg
from heuristique_style_transfer_code_b200 import functions as F
from oracle import jpeg_decode as J

SMALL = C.corpus(large=False)


@pytest.mark.parametrize("name,data", SMALL[::3], ids=[n for n, _ in SMALL[::3]])
def test_header_and_segments_are_pillows(name, data):
    f = jpeg.parse(data)
    assert f is not None
    im = Image.open(io.BytesIO(data))
    assert (f.W, f.H) == im.size and len(f.comps) == im.layers
    assert im.mode == ("L" if len(f.comps) == 1 else "RGB")
    for k, c in enumerate(f.comps):
        assert np.array_equal(f.tables[k * 64:(k + 1) * 64], np.asarray(im.quantization[c[3]]))   # natural order both
    hdr = J.parse(data)
    assert [bytes(s) for s in f.segments] == J.segments(data, hdr["scan_start"])[:len(f.segments)]


def _kinds(tmp_path):
    rng = np.random.default_rng(2)
    img = Image.fromarray(C.content("resized", 40, 56, rng))
    out = {}
    for name, kw in (("progressive", dict(progressive=True)), ("cmyk", None), ("baseline", dict(quality=80))):
        b = io.BytesIO()
        (img.convert("CMYK") if kw is None else img).save(b, "JPEG", **(kw or {}))
        out[name] = b.getvalue()
    coef = C.random_coefficients(rng, 16, 16, [(1, 1, 1, 0), (2, 1, 1, 0), (3, 1, 1, 0)])
    out["adobe_rgb"] = C.write(coef, [(1, 1, 1, 0), (2, 1, 1, 0), (3, 1, 1, 0)], {0: np.full(64, 4)}, 16, 16,
                               jfif=False, adobe=0)
    out["rgb_ids"] = C.write(coef, [(82, 1, 1, 0), (71, 1, 1, 0), (66, 1, 1, 0)], {0: np.full(64, 4)}, 16, 16,
                             jfif=False)
    b = io.BytesIO()
    img.save(b, "PNG")
    out["png"] = b.getvalue()
    b = io.BytesIO()
    img.save(b, "JPEG", quality=80, optimize=True)
    out["optimized"] = b.getvalue()
    return out


def test_classification_and_fallback(tmp_path):
    from torchvision.datasets.folder import default_loader
    t = F.gpu_resize_transform(32, 24, decode="gpu")
    device = {"baseline", "optimized"}
    for name, data in _kinds(tmp_path).items():
        p = tmp_path / f"{name}.bin"
        p.write_bytes(data)
        got = t.loader(str(p))
        assert isinstance(got, jpeg.JpegFile) == (name in device), name
        if not isinstance(got, jpeg.JpegFile):
            assert got.mode == "RGB" and np.array_equal(np.asarray(got), np.asarray(default_loader(str(p))))
    p = tmp_path / "text.jpg"
    p.write_bytes(b"not an image")
    with pytest.raises(Exception):
        t.loader(str(p))


def test_host_batch_is_torchvision(tmp_path):
    from torchvision import transforms
    from torchvision.datasets.folder import default_loader
    t = F.gpu_resize_transform(64, 56, decode="gpu")
    paths = []
    for i, (name, data) in enumerate(list(_kinds(tmp_path).items()) + SMALL[::11]):
        p = tmp_path / f"{i}.img"
        p.write_bytes(data)
        paths.append(str(p))
    batch = t.collate([(t(t.loader(p)), i) for i, p in enumerate(paths)])
    assert batch.jpeg is not None and batch.pixels.numel() < batch.arena_bytes
    assert batch.files and all(isinstance(f, str) for f in batch.files)      # paths, not the files' bytes
    pinned = batch.pin_memory() if torch.cuda.is_available() else batch
    ref = transforms.Compose([transforms.Resize(64), transforms.CenterCrop(56), transforms.PILToTensor()])
    want = torch.stack([ref(default_loader(p)) for p in paths])
    (x, y), = list(F.cuda_prefetch([pinned], "cpu", normalize=None))
    assert torch.equal(x, want) and y.tolist() == list(range(len(paths)))


def test_host_decode_is_unchanged():
    t = F.gpu_resize_transform(64, 56)
    assert t.decode == "host"
    with pytest.raises(ValueError):
        t.loader("anything.jpg")
    with pytest.raises(ValueError):
        F.gpu_resize_transform(64, 56, decode="nvjpeg")


def test_cabi_host_queries_and_refusals():
    lib = _lib.lib()
    assert lib.gh_jpeg_table_ints() == jpeg.TABLE_INTS
    assert lib.gh_jpeg_records_bytes(1000, 3, 100) == (10 + 3 + 1) * 8 * 4
    for args in ((1000, 0, 100), (1000, 3, 0), (-1, 3, 100)):
        assert lib.gh_jpeg_records_bytes(*args) == _lib.GH_ERR_BAD_ARG
    p = 16

    def call(**kw):
        a = dict(scan=p, scan_bytes=10, segs=p, n_segs=1, imgs=p, n_imgs=1, tables=p, max_blocks=1, max_pixels=1,
                 subseq=64, coef=p, planes=p, records=p, status=p, arena=p, phases=7)
        a.update(kw)
        return lib.gh_jpeg_decode(*a.values(), None)
    assert call(scan=None) == _lib.GH_ERR_BAD_ARG
    assert call(n_segs=0) == _lib.GH_ERR_BAD_ARG
    assert call(subseq=0) == _lib.GH_ERR_BAD_ARG
    assert call(phases=0) == _lib.GH_ERR_BAD_ARG and call(phases=8) == _lib.GH_ERR_BAD_ARG
    assert call(n_imgs=65536) == _lib.GH_ERR_UNSUPPORTED


def test_validate_refuses_out_of_range_descriptors():
    data = SMALL[5][1]
    f = jpeg.parse(data)
    scan, segs, imgs, tables = jpeg.pack([f], [0], [0])
    jpeg.validate(scan.numel(), segs.numpy(), imgs.numpy(), f.H * f.W * 3)
    with pytest.raises(_lib.GramHeadError):
        jpeg.validate(scan.numel(), segs.numpy(), imgs.numpy(), f.H * f.W * 3 - 1)
    bad = segs.numpy().copy()
    bad[0, 1] = scan.numel() + 1
    with pytest.raises(_lib.GramHeadError):
        jpeg.validate(scan.numel(), bad, imgs.numpy(), f.H * f.W * 3)


def test_batch_scan_data_has_no_size_limit():
    """Only a segment's length is bounded (bit positions inside it are 32-bit); a batch of many large files is not."""
    lib = _lib.lib()
    assert lib.gh_jpeg_check(1 << 28, 64, 64, 1 << 20, 1 << 24, jpeg.SUBSEQ_BYTES, 7) == 0
    assert lib.gh_jpeg_check(5 << 30, 1, 1, 1, 1, 1, 7) == 0
    assert lib.gh_jpeg_check(0, 1, 1, 1, 1, 1, 7) == _lib.GH_ERR_BAD_ARG
    assert lib.gh_jpeg_check(10, 1, 65536, 1, 1, 1, 7) == _lib.GH_ERR_UNSUPPORTED
    assert lib.gh_jpeg_records_bytes(5 << 30, 64, jpeg.SUBSEQ_BYTES) > 0
    imgs = np.array([[8, 8, 1, 1, 1, 1, 1, 0, 1, 0, 0, 0, 0]], np.int64)
    total = 3 << 28
    jpeg.validate(total, np.array([[total - 1000, 1000, 0, 0, 1]], np.int64), imgs, 192)
    with pytest.raises(_lib.GramHeadError):
        jpeg.validate(total, np.array([[0, jpeg.MAX_SEGMENT_BYTES, 0, 0, 1]], np.int64), imgs, 192)


def test_all_ones_huffman_code_is_refused_as_pillow_does(tmp_path):
    """jpeg_make_d_derived_tbl refuses a table whose code words of some length run up to all ones; the worker then
    leaves the file to Pillow, which raises its own error."""
    with pytest.raises(ValueError):
        jpeg._huff_table((2,) + (0,) * 15, (0, 1))
    b = io.BytesIO()
    Image.fromarray(C.content("noise", 16, 16, np.random.default_rng(0))).save(b, "JPEG", quality=90)
    data = bytearray(b.getvalue())
    i = data.index(b"\xff\xc4") + 5                    # bits[] of the first table (DC 0: 0,1,5,1,1,1,1,1,1,0,...)
    assert data[i - 1] == 0x00 and sum(data[i:i + 16]) == 12
    data[i:i + 16] = bytes([2, 0, 5, 1, 1, 1, 1, 1] + [0] * 8)      # still 12 codes, but both 1-bit codes used
    p = tmp_path / "bad.jpg"
    p.write_bytes(bytes(data))
    assert jpeg.parse(bytes(data)) is None
    t = F.gpu_resize_transform(32, 24, decode="gpu")
    with pytest.raises(OSError):
        np.asarray(t.loader(str(p)))
