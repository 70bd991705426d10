"""Batched frame preprocessing without a GPU: the C-ABI validation of gh_preprocess_frames (which returns before any CUDA
call), the host packing of descriptors and tables against resample_tables, and the argument checks of the two loops."""
import ctypes

import numpy as np
import pytest

from heuristique_style_transfer_code_b200 import _lib
from heuristique_style_transfer_code_b200 import functions as F
from heuristique_style_transfer_code_b200 import streaming as S
from heuristique_style_transfer_code_b200._lib import GramHeadError
from heuristique_style_transfer_code_b200.build import build_library

MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
SHAPES = [(1080, 1920, 3), (720, 1280, 3), (640, 480, 3), (333, 517, 3), (150, 200, 3)]


@pytest.fixture(scope="module")
def library():
    build_library()
    return _lib.lib()


def test_argument_validation_without_gpu(library):
    d = ctypes.c_void_p(256)
    BAD, UNS = _lib.GH_ERR_BAD_ARG, _lib.GH_ERR_UNSUPPORTED
    f = library.gh_preprocess_frames
    #       frames N  OH   OW  band span tables hk vk out  stream
    assert f(None, 2, 224, 224, 4, 20, d, 9, 5, d, None) == BAD
    assert f(d, 2, 224, 224, 4, 20, None, 9, 5, d, None) == BAD
    assert f(d, 2, 224, 224, 4, 20, d, 9, 5, None, None) == BAD
    assert f(d, 0, 224, 224, 4, 20, d, 9, 5, d, None) == BAD                 # N <= 0
    assert f(d, -1, 224, 224, 4, 20, d, 9, 5, d, None) == BAD
    assert f(d, 2, 0, 224, 4, 20, d, 9, 5, d, None) == BAD                   # OH <= 0
    assert f(d, 2, 224, 0, 4, 20, d, 9, 5, d, None) == BAD                   # OW <= 0
    assert f(d, 2, 224, 224, 0, 20, d, 9, 5, d, None) == BAD                 # band height <= 0
    assert f(d, 2, 224, 224, 4, 20, d, 0, 5, d, None) == BAD                 # hkmax <= 0
    assert f(d, 2, 224, 224, 4, 20, d, 9, 0, d, None) == BAD                 # vkmax <= 0
    assert f(d, 2, 224, 224, 4, 4, d, 9, 5, d, None) == BAD                  # one output row would not fit
    assert f(d, 65536, 224, 224, 4, 20, d, 9, 5, d, None) == UNS             # gridDim.y
    assert f(d, 2, 65536, 224, 1, 20, d, 9, 5, d, None) == UNS               # bands > 65535
    assert f(d, 2, 224, 100000, 1, 5, d, 9, 5, d, None) == UNS               # shared memory beyond one CTA's


def test_shared_memory_query(library):
    q = library.gh_preprocess_frames_smem
    assert q(448, 30) == 3 * 448 * 30
    assert q(224, 1) == 672
    assert q(0, 5) == _lib.GH_ERR_BAD_ARG and q(448, 0) == _lib.GH_ERR_BAD_ARG
    assert q(100000, 1) == _lib.GH_ERR_UNSUPPORTED
    assert q(1024, 227 // 3) == 3 * 1024 * 75


def test_descriptor_layout_is_the_c_struct():
    dt = S.FRAME_DESC_DTYPE
    assert dt.itemsize == 80
    offsets = {name: dt.fields[name][1] for name in dt.names}
    assert offsets == dict(frame=0, pitch=8, H=16, W=20, bgr=24, reserved=28, hx_min=32, hx_size=40, hk=48, vy_min=56,
                           vy_size=64, vk=72)


@pytest.mark.parametrize("resize,crop", [((448, 448), None), (256, 224), ((224, 300), (200, 256))])
def test_packed_tables_are_resample_tables(resize, crop):
    from oracle import pil_resize as P
    packed = S.pack_frame_tables(SHAPES, resize, crop)
    oh, ow = packed["out_hw"]
    tables, hk, vk = packed["tables"], packed["hkmax"], packed["vkmax"]
    assert tables.dtype == np.int32 and packed["offsets"].shape == (len(SHAPES), 6)
    for (h, w, _), off, rows in zip(SHAPES, packed["offsets"], packed["rows"]):
        rh, rw = P.resize_output_size(h, w, resize)
        top, left = 0, 0
        if crop is not None:
            top, left, th, tw = P.center_crop_box(rh, rw, crop)
            assert (th, tw) == (oh, ow)
        else:
            assert (rh, rw) == (oh, ow)
        for (lo, n, kk), o, count, kmax in ((S.resample_tables(w, rw, left, ow), off[:3], ow, hk),
                                            (S.resample_tables(h, rh, top, oh), off[3:], oh, vk)):
            assert np.array_equal(tables[o[0]:o[0] + count], lo)
            assert np.array_equal(tables[o[1]:o[1] + count], n)
            got = tables[o[2]:o[2] + count * kmax].reshape(count, kmax)
            assert np.array_equal(got[:, :kk.shape[1]], kk) and not got[:, kk.shape[1]:].any()
        assert np.array_equal(rows[0], tables[off[3]:off[3] + oh]) and np.array_equal(rows[1], tables[off[4]:off[4] + oh])
    assert packed["offsets"][-1, 5] + oh * vk == tables.size


def test_band_span_and_height(library):
    packed = S.pack_frame_tables(SHAPES, (448, 448))
    rows = packed["rows"]
    for r in (1, 2, 5, 13, 448):
        want = 0
        for y0, yn in rows:
            for b in range(0, len(y0), r):
                want = max(want, int((y0[b:b + r] + yn[b:b + r]).max() - y0[b:b + r].min()))
        assert S.band_span(rows, r) == want
    assert S.band_span(rows, 1) <= packed["vkmax"]
    top = S.max_band_rows(rows, 448)
    assert top > 1 and library.gh_preprocess_frames_smem(448, S.band_span(rows, top)) <= S._BAND_SMEM_BUDGET
    assert library.gh_preprocess_frames_smem(448, S.band_span(rows, top + 1)) > S._BAND_SMEM_BUDGET
    assert S.max_band_rows(rows, 448, budget=1) == 1                     # one row per band always remains


def test_packing_refusals():
    with pytest.raises(GramHeadError):
        S.pack_frame_tables([(1080, 1920, 3), (480, 640, 3)], 256)          # different sizes out of Resize(256)
    with pytest.raises(GramHeadError):
        S.pack_frame_tables([(100, 100, 3)], (200, 200), crop=224)          # crop larger than the resized frame
    with pytest.raises(GramHeadError):
        S.pack_frame_tables([(100, 100)], (224, 224))
    with pytest.raises(GramHeadError):
        S.pack_frame_tables([], (224, 224))


class _CpuModel:
    device = "cpu"


class _NoReads:
    def isOpened(self):
        return True

    def read(self):
        raise AssertionError("the loop read a frame before checking its arguments")

    def release(self):
        pass


def _transform():
    from torchvision import transforms
    return transforms.Compose([transforms.Resize(256), transforms.CenterCrop(224), transforms.ToTensor(),
                               transforms.Normalize(MEAN, STD)])


def test_loop_argument_checks(tmp_path):
    from torchvision import transforms
    tf = _transform()
    cuda_model = type("M", (), {"device": "cuda:0"})()
    unsupported = transforms.Compose([transforms.Resize(256), transforms.ToTensor()])
    for bad in (0, -2, 1.5, True, None):
        with pytest.raises(ValueError):
            F.classify_video(cuda_model, tf, _NoReads(), frames_per_call=bad)
    with pytest.raises(ValueError):
        F.classify_video(cuda_model, tf, _NoReads(), max_frames=-1)
    with pytest.raises(ValueError):
        F.classify_video(_CpuModel(), tf, _NoReads())
    with pytest.raises(ValueError):
        F.classify_video(cuda_model, unsupported, _NoReads())
    args = (["fog", "rain"], False, str(tmp_path), 0.5, True)
    with pytest.raises(ValueError):
        F.run_cameras(cuda_model, tf, args[0], [], *args[1:])
    with pytest.raises(ValueError):
        F.run_cameras(_CpuModel(), tf, args[0], [_NoReads()], *args[1:])
    with pytest.raises(ValueError):
        F.run_cameras(cuda_model, unsupported, args[0], [_NoReads(), _NoReads()], *args[1:])
    with pytest.raises(ValueError):
        F.run_cameras(cuda_model, tf, args[0], [_NoReads()], *args[1:], max_frames=-1)
    assert list(tmp_path.iterdir()) == []


def test_pipeline_refuses_a_cpu_model():
    with pytest.raises(GramHeadError):
        S.FrameBatchPipeline(_CpuModel(), [(480, 640, 3)], (224, 224))
