"""GPU: several frames per forward (gh_preprocess_frames, streaming.FrameBatchPipeline, functions.run_cameras /
classify_video) against the Pillow oracle (oracle/pil_resize.py), the one-frame kernel and CameraPipeline.

The bitwise comparisons of probabilities run with ops.KSPLIT = 1: batch-1 Gram launches otherwise split K over fp32
atomics, whose order (and so the last bits) changes from run to run."""
import numpy as np
import pytest
import torch

from oracle import pil_resize as P

pytestmark = pytest.mark.gpu

MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
# landscape 1080p and 720p, portrait 480 x 640, odd sizes, and a frame smaller than the output (upscale)
SHAPES = [(1080, 1920, 3), (720, 1280, 3), (640, 480, 3), (333, 517, 3), (150, 200, 3)]
GEOMETRIES = {"resize448": ((448, 448), None), "resize256_crop224": (256, 224)}


def test_cuda_is_present():
    assert torch.cuda.is_available()


@pytest.fixture(scope="module")
def model():
    from torchvision import models
    from heuristique_style_transfer_code_b200 import ops, TruncatedResNet50_for_test
    torch.manual_seed(0)
    m = TruncatedResNet50_for_test(models.resnet50(weights=None), 7, 4, 32, device="cuda:0").eval()
    saved, ops.KSPLIT = ops.KSPLIT, 1
    yield m
    ops.KSPLIT = saved


def _frames(seed, shapes=SHAPES):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, s, dtype=np.uint8) for s in shapes]


_ORACLE = {}


def _oracle(geometry, frames_rgb, key):
    """Pillow's resize [+ centre crop] of each RGB frame as (3, oh, ow) uint8."""
    if (geometry, key) not in _ORACLE:
        resize, crop = GEOMETRIES[geometry]
        out = []
        for f in frames_rgb:
            rh, rw = P.resize_output_size(f.shape[0], f.shape[1], resize)
            img = P.resize_bilinear_u8(np.ascontiguousarray(f), rh, rw)
            if crop is not None:
                top, left, th, tw = P.center_crop_box(rh, rw, crop)
                img = img[top:top + th, left:left + tw]
            out.append(img.transpose(2, 0, 1))
        _ORACLE[(geometry, key)] = np.stack(out)
    return _ORACLE[(geometry, key)]


def _upload(pipe, frames):
    for slot, f in zip(pipe._slots, frames):
        np.copyto(slot, f)
    pipe._frames_dev.copy_(pipe._frames_pin)


@pytest.mark.parametrize("bgr", [True, False])
@pytest.mark.parametrize("geometry", list(GEOMETRIES))
def test_kernel_is_bitwise_pillow(model, geometry, bgr):
    from heuristique_style_transfer_code_b200.streaming import FrameBatchPipeline
    resize, crop = GEOMETRIES[geometry]
    rgb = _frames(1)
    frames = [np.ascontiguousarray(f[:, :, ::-1]) for f in rgb] if bgr else rgb
    want = _oracle(geometry, rgb, 1)
    pipe = FrameBatchPipeline(model, SHAPES, resize, crop, MEAN, STD, bgr=bgr, use_graph=False)
    n, (oh, ow) = len(SHAPES), pipe.out_hw
    assert pipe.max_band_rows > 1
    guard = 4096
    buf = torch.empty(n * 3 * oh * ow + 2 * guard, dtype=torch.uint8, device=model.device)
    pipe._input = buf[guard:guard + n * 3 * oh * ow].view(n, 3, oh, ow)
    _upload(pipe, frames)
    for band in (1, pipe.max_band_rows, pipe.band_rows):
        buf.fill_(0xA5)
        got = pipe.preprocess_(band).cpu().numpy()
        assert got.shape == want.shape and np.array_equal(got, want), band
        edges = torch.cat([buf[:guard], buf[-guard:]])
        assert bool((edges == 0xA5).all()), band


def test_kernel_matches_the_one_frame_kernel(model):
    from heuristique_style_transfer_code_b200 import ops
    from heuristique_style_transfer_code_b200.streaming import CameraPipeline, FrameBatchPipeline
    frames = _frames(2)
    for resize, crop in GEOMETRIES.values():
        pipe = FrameBatchPipeline(model, SHAPES, resize, crop, MEAN, STD, use_graph=False)
        _upload(pipe, frames)
        got = ops.normalize_u8(pipe.preprocess_(), MEAN, STD)
        for i, f in enumerate(frames):
            cam = CameraPipeline(model, f.shape, resize, crop, MEAN, STD, use_graph=False)
            cam._frame_dev.copy_(torch.from_numpy(f))
            assert torch.equal(got[i], cam.preprocess_()[0]), (resize, crop, f.shape)


@pytest.mark.parametrize("tf32", [True, False])
def test_one_frame_is_bitwise_camera_pipeline(model, tf32):
    from heuristique_style_transfer_code_b200.streaming import CameraPipeline, FrameBatchPipeline
    saved = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = tf32              # on: uint8 fused stem; off: normalize_u8 + the conv chain
    try:
        shape = (1080, 1920, 3)
        cam = CameraPipeline(model, shape, (448, 448), None, MEAN, STD)
        batch = FrameBatchPipeline(model, [shape], (448, 448), None, MEAN, STD)
        for seed in (3, 4):
            frame = _frames(seed, [shape])[0]
            got, want = batch([frame]), cam(frame)
            assert got.shape == (1, 4) and np.array_equal(got[0], want)
    finally:
        torch.backends.cudnn.allow_tf32 = saved


@pytest.mark.parametrize("n", [4, 16])
def test_mixed_batch_is_bitwise_the_eager_model(model, n):
    from heuristique_style_transfer_code_b200.streaming import CameraPipeline, FrameBatchPipeline
    shapes = [SHAPES[i % len(SHAPES)] for i in range(n)]
    resize, crop = GEOMETRIES["resize256_crop224"]
    graph = FrameBatchPipeline(model, shapes, resize, crop, MEAN, STD)
    eager = FrameBatchPipeline(model, shapes, resize, crop, MEAN, STD, use_graph=False)
    assert graph._graph is not None
    cams = {s: CameraPipeline(model, s, resize, crop, MEAN, STD, use_graph=False) for s in set(shapes)}
    previous = None
    for seed in (5, 6):                                  # the second call reuses every buffer with other frames
        frames = _frames(seed, shapes)
        xs = []
        for f in frames:
            cams[f.shape]._frame_dev.copy_(torch.from_numpy(f))
            xs.append(cams[f.shape].preprocess_().clone())
        with torch.no_grad():
            want = torch.softmax(model(torch.cat(xs))[1], dim=1).cpu().numpy()
        got = graph(frames)
        assert got.shape == (n, 4)
        assert np.array_equal(got, want)
        assert np.array_equal(eager(frames), got)
        if previous is not None:
            assert not np.array_equal(got, previous)
        previous = got


def test_model_state_and_errors(model):
    from heuristique_style_transfer_code_b200 import TruncatedResNet50
    from heuristique_style_transfer_code_b200._lib import GramHeadError
    from heuristique_style_transfer_code_b200.streaming import FrameBatchPipeline
    from torchvision import models
    shapes = [(480, 640, 3), (720, 1280, 3)]
    assert model.input_normalization is None
    pipe = FrameBatchPipeline(model, shapes, 256, 224, MEAN, STD)
    frames = _frames(7, shapes)
    pipe(frames)
    assert model.input_normalization is None
    with pytest.raises(GramHeadError):
        pipe(frames[:1])                                              # number of frames
    with pytest.raises(GramHeadError):
        pipe([frames[1], frames[0]])                                  # shape of a slot
    with pytest.raises(GramHeadError):
        pipe([frames[0], frames[1].astype(np.float32)])               # dtype
    with pytest.raises(GramHeadError):
        FrameBatchPipeline(model, [(100, 100, 3)], (200, 200), 224)   # crop larger than the resized frame
    torch.manual_seed(0)
    cpu_model = TruncatedResNet50(models.resnet50(weights=None), 7, 4, 32, device="cpu")
    with pytest.raises(GramHeadError):
        FrameBatchPipeline(cpu_model, shapes, 256, 224)
    # the training class (forward -> logits) runs too, with its own normalisation left alone
    train_cls = cpu_model.to("cuda:0")
    train_cls.device = "cuda:0"
    train_cls.eval().set_input_normalization([0.5] * 3, [0.25] * 3)
    probs = FrameBatchPipeline(train_cls, shapes, 256, 224, MEAN, STD)(frames)
    assert probs.shape == (2, 4) and np.allclose(probs.sum(axis=1), 1.0, atol=1e-5)
    assert train_cls.input_normalization == ((0.5,) * 3, (0.25,) * 3)


class Capture:
    def __init__(self, n, shape=(480, 640, 3), seed=0):
        self.frames = [np.random.default_rng(seed + i).integers(0, 256, shape, dtype=np.uint8) for i in range(n)]
        self.i = 0
        self.released = False

    def isOpened(self):
        return True

    def read(self):
        if self.i >= len(self.frames):
            return False, None
        self.i += 1
        return True, self.frames[self.i - 1].copy()

    def release(self):
        self.released = True


def _transform():
    from torchvision import transforms
    return transforms.Compose([transforms.Resize(256), transforms.CenterCrop(224), transforms.ToTensor(),
                               transforms.Normalize(mean=MEAN, std=STD)])


def test_classify_video_matches_run_camera(model, tmp_path, monkeypatch):
    import cv2
    from heuristique_style_transfer_code_b200.functions import classify_video, run_camera
    names = ["fog", "rain", "snow", "sun"]
    labels = []
    real = cv2.putText
    monkeypatch.setattr(cv2, "putText", lambda img, text, *a, **k: (labels.append(text), real(img, text, *a, **k))[1])
    run_camera(model, _transform(), names, False, str(tmp_path), 0.0, False, capture=Capture(7), display=False,
               pipeline="gpu")
    pred1, prob1 = classify_video(model, _transform(), Capture(7), frames_per_call=1)
    assert [f"Pred: {names[p]}, Prob: {q:.4f}" for p, q in zip(pred1, prob1)] == labels
    pred3, prob3 = classify_video(model, _transform(), Capture(7), frames_per_call=3)   # groups of 3, 3 and 1
    assert len(pred3) == len(prob3) == 7 and np.allclose(prob3, prob1, atol=1e-5)
    assert pred3.dtype == np.int64 and prob3.dtype == np.float32
    pred4, _ = classify_video(model, _transform(), Capture(7), frames_per_call=4, max_frames=5)
    assert len(pred4) == 5


def test_run_cameras_writes_one_video_per_stream(model, tmp_path):
    import json
    from heuristique_style_transfer_code_b200.functions import run_cameras
    caps = [Capture(4, (480, 640, 3), 0), Capture(3, (720, 1280, 3), 10), Capture(4, (1080, 1920, 3), 20)]
    names = ["fog", "rain", "snow", "sun"]
    times = run_cameras(model, _transform(), names, caps, True, str(tmp_path), 0.5, True)
    assert len(times) == 3                                    # the second capture ends after three frames
    for i in range(3):
        assert (tmp_path / f"camera_{i}_output.avi").stat().st_size > 0
    assert json.loads((tmp_path / "times_cameras.json").read_text()) == times
    assert all(c.released for c in caps)
    times = run_cameras(model, _transform(), names, [Capture(5), Capture(5, seed=9)], False, str(tmp_path), 0.5, False,
                        max_frames=2)
    assert len(times) == 2
