"""Camera-mode streaming on the GPU (SURVEY.md section 8(f) n2).

The reference handles a camera frame on the host: cv2.cvtColor(BGR2RGB) -> PIL -> torchvision transform (Resize
[+ CenterCrop] + ToTensor + Normalize) -> .to(device) -> model -> softmax -> .cpu()
(functions/functions_RESNET50_Truncate_Gram_Attention.py:494-507). At 1080p the host-side resize alone costs ~9 ms per
frame, four times the forward pass. `CameraPipeline` keeps the same arithmetic but moves it:

  frame (uint8 HWC, BGR) --memcpy--> pinned buffer --H2D (6 MB)--> gh_preprocess_frame (one kernel, bit-identical to
  Pillow's antialiased bilinear resize + ToTensor + Normalize) --> encoder + Gram/attention head --> softmax
  --D2H (num_classes floats)--> pinned buffer

Everything between the two host buffers is captured once in a CUDA graph and replayed per frame, so a batch-1 forward
(~150 kernel launches) costs one graph launch. The coefficient tables of the resize depend only on the geometry and are
computed once here (the same rule as Pillow's precompute_coeffs: triangle filter, support scaled by the down-scale
factor, 22-bit fixed point); a CenterCrop is the sub-range of output coordinates the tables are built for.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import GramHeadError, check

_PRECISION_BITS = 32 - 8 - 2


def resample_kmax(in_size: int, out_size: int) -> int:
    """Coefficients per output coordinate of the antialiased bilinear resample along one axis (Pillow's ksize)."""
    return int(math.ceil(max(in_size / out_size, 1.0))) * 2 + 1


def resample_tables(in_size: int, out_size: int, first: int = 0, count: Optional[int] = None):
    """Integer tables of the antialiased bilinear resample along one axis, for output coordinates [first, first+count):
    (min[count], size[count], coeff[count, kmax]) as int32 arrays."""
    count = out_size - first if count is None else count
    scale = in_size / out_size
    filterscale = max(scale, 1.0)
    support = filterscale                       # bilinear: support 1.0 * filterscale
    kmax = resample_kmax(in_size, out_size)
    lo_a = np.zeros(count, dtype=np.int32)
    n_a = np.zeros(count, dtype=np.int32)
    kk = np.zeros((count, kmax), dtype=np.int32)
    inv = 1.0 / filterscale
    for t in range(count):
        center = (first + t + 0.5) * scale
        lo = max(int(center - support + 0.5), 0)
        hi = min(int(center + support + 0.5), in_size)
        n = hi - lo
        w = [max(0.0, 1.0 - abs((x + lo - center + 0.5) * inv)) for x in range(n)]
        tot = sum(w)
        if tot != 0.0:
            w = [v / tot for v in w]
        lo_a[t], n_a[t] = lo, n
        for x, v in enumerate(w):
            kk[t, x] = int(v * (1 << _PRECISION_BITS) + 0.5)
    return lo_a, n_a, kk


def _resize_output_size(h: int, w: int, size) -> Tuple[int, int]:
    if isinstance(size, (tuple, list)):
        if len(size) == 2:
            return int(size[0]), int(size[1])
        size = size[0]
    short, long_ = (w, h) if w <= h else (h, w)
    new_short, new_long = int(size), int(size * long_ / short)
    return (new_long, new_short) if w <= h else (new_short, new_long)


def parse_transform(transform):
    """Recognises torchvision Compose([Resize(bilinear), [CenterCrop], ToTensor, Normalize]) and returns
    dict(resize=, crop=, mean=, std=) -- or None for anything else (the caller then keeps the host path)."""
    try:
        from torchvision import transforms as T
        from torchvision.transforms import InterpolationMode
    except Exception:
        return None
    steps = list(getattr(transform, "transforms", []))
    if len(steps) not in (3, 4) or not isinstance(steps[0], T.Resize):
        return None
    rz = steps[0]
    if rz.interpolation != InterpolationMode.BILINEAR or getattr(rz, "max_size", None) is not None:
        return None
    crop = None
    rest = steps[1:]
    if len(rest) == 3:
        if not isinstance(rest[0], T.CenterCrop):
            return None
        crop = rest[0].size
        rest = rest[1:]
    if not (isinstance(rest[0], T.ToTensor) and isinstance(rest[1], T.Normalize)):
        return None
    mean, std = [float(v) for v in rest[1].mean], [float(v) for v in rest[1].std]
    if len(mean) != 3 or len(std) != 3:
        return None
    return dict(resize=rz.size, crop=crop, mean=mean, std=std)


class CameraPipeline:
    """frame (H, W, 3) uint8 numpy -> probabilities (num_classes,) numpy; model must be a TruncatedResNet50_for_test
    (forward -> (embeddings, logits)) on a CUDA device."""

    def __init__(self, model, frame_shape: Sequence[int], resize, crop=None, mean=(0.485, 0.456, 0.406),
                 std=(0.229, 0.224, 0.225), bgr: bool = True, use_graph: bool = True):
        self.model = model
        self.device = torch.device(model.device)
        if self.device.type != "cuda":
            raise GramHeadError("gramhead: CameraPipeline needs the model on a CUDA device (there is no CPU path)")
        h, w = int(frame_shape[0]), int(frame_shape[1])
        if len(frame_shape) != 3 or frame_shape[2] != 3:
            raise GramHeadError(f"gramhead: frames must be (H, W, 3) uint8, got shape {tuple(frame_shape)}")
        rh, rw = _resize_output_size(h, w, resize)
        top, left, oh, ow = 0, 0, rh, rw
        if crop is not None:
            oh, ow = (int(crop), int(crop)) if not isinstance(crop, (tuple, list)) else (int(crop[0]), int(crop[-1]))
            if oh > rh or ow > rw:
                raise GramHeadError("gramhead: CenterCrop larger than the resized frame is not supported on the GPU path")
            top, left = int(round((rh - oh) / 2.0)), int(round((rw - ow) / 2.0))
        self.frame_shape, self.out_hw, self.bgr = (h, w, 3), (oh, ow), bool(bgr)
        dev = self.device
        hx = resample_tables(w, rw, left, ow)
        vy = resample_tables(h, rh, top, oh)
        self._tables = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (*hx, *vy)]
        self._hkmax, self._vkmax = int(hx[2].shape[1]), int(vy[2].shape[1])
        self._mean = (torch.tensor(mean, dtype=torch.float32).numpy().copy())
        self._std = (torch.tensor(std, dtype=torch.float32).numpy().copy())
        self._frame_pin = torch.empty((h, w, 3), dtype=torch.uint8).pin_memory()
        self._frame_np = self._frame_pin.numpy()
        self._frame_dev = torch.empty((h, w, 3), dtype=torch.uint8, device=dev)
        self._input = torch.empty((1, 3, oh, ow), dtype=torch.float32, device=dev)
        self._probs_dev = None
        self._probs_pin = None
        self._graph = None
        self._done = torch.cuda.Event()
        model.eval()
        with torch.cuda.device(dev), torch.no_grad():
            self._body()                                  # allocates the output buffers, loads every kernel
            torch.cuda.synchronize(dev)
            if use_graph:
                side = torch.cuda.Stream(device=dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):
                    for _ in range(2):
                        self._body()
                torch.cuda.current_stream(dev).wait_stream(side)
                torch.cuda.synchronize(dev)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    self._body()
                self._graph = graph
                # the graph holds raw addresses of the model's folded inference plan: keep that plan (and its tensors)
                # alive for as long as this pipeline exists, whatever the model does with its own reference later
                self._captured_plan = getattr(model, "_plan", None)

    # the device-side work for one frame; captured into the graph
    def preprocess_(self):
        """Runs the preprocessing kernel on the uploaded frame; result in self._input (1, 3, oh, ow)."""
        h, w, _ = self.frame_shape
        oh, ow = self.out_hw
        t = self._tables
        rc = _lib.lib().gh_preprocess_frame(
            self._frame_dev.data_ptr(), w * 3, h, w, 1 if self.bgr else 0, t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(),
            self._hkmax, t[3].data_ptr(), t[4].data_ptr(), t[5].data_ptr(), self._vkmax, self._mean.ctypes.data,
            self._std.ctypes.data, self._input.data_ptr(), oh, ow, torch.cuda.current_stream(self.device).cuda_stream)
        check(rc, "gh_preprocess_frame")
        return self._input

    def _body(self):
        self._frame_dev.copy_(self._frame_pin, non_blocking=True)
        self.preprocess_()
        out = self.model(self._input)
        logits = out[1] if isinstance(out, (tuple, list)) else out
        probs = torch.softmax(logits, dim=1)
        if self._probs_dev is None:
            self._probs_dev = torch.empty_like(probs)
            self._probs_pin = torch.empty(probs.shape, dtype=probs.dtype).pin_memory()
        self._probs_dev.copy_(probs)
        self._probs_pin.copy_(self._probs_dev, non_blocking=True)

    def __call__(self, frame: np.ndarray) -> np.ndarray:
        if frame.shape != self.frame_shape or frame.dtype != np.uint8:
            raise GramHeadError(f"gramhead: CameraPipeline was built for uint8 frames of shape {self.frame_shape}, "
                                f"got {frame.dtype} {tuple(frame.shape)}")
        np.copyto(self._frame_np, frame)
        with torch.cuda.device(self.device), torch.no_grad():
            if self._graph is not None:
                self._graph.replay()
            else:
                self._body()
            self._done.record(torch.cuda.current_stream(self.device))
        self._done.synchronize()
        return self._probs_pin.numpy()[0].copy()

    @classmethod
    def from_transform(cls, model, transform, frame_shape, bgr: bool = True, use_graph: bool = True):
        """Pipeline equivalent to `transform` applied to a PIL image of the frame, or None when the transform is not the
        Resize [+ CenterCrop] + ToTensor + Normalize chain the GPU kernel reproduces."""
        spec = parse_transform(transform)
        if spec is None:
            return None
        return cls(model, frame_shape, spec["resize"], spec["crop"], spec["mean"], spec["std"], bgr=bgr, use_graph=use_graph)


# ---- several frames per forward ---------------------------------------------------------------------------------------
# GhFrameDesc of include/gramhead.h, one record per frame slot; the table offsets count int32 elements.
FRAME_DESC_DTYPE = np.dtype([("frame", "<u8"), ("pitch", "<i8"), ("H", "<i4"), ("W", "<i4"), ("bgr", "<i4"),
                             ("reserved", "<i4"), ("hx_min", "<i8"), ("hx_size", "<i8"), ("hk", "<i8"), ("vy_min", "<i8"),
                             ("vy_size", "<i8"), ("vk", "<i8")])
_TABLE_FIELDS = ("hx_min", "hx_size", "hk", "vy_min", "vy_size", "vk")
# shared memory a band of gh_preprocess_frames may use when the host picks its height: several CTAs stay resident per SM
_BAND_SMEM_BUDGET = 48 * 1024


def frame_geometry(frame_shapes, resize, crop=None):
    """The geometry of torchvision's Resize(resize) [+ CenterCrop(crop)] for each (H, W, 3) frame shape:
    ([(h, w, rh, rw, top, left, oh, ow)] per frame, (oh, ow)). Every frame must come out at the same (oh, ow)."""
    geometry = []
    for shape in frame_shapes:
        if len(shape) != 3 or int(shape[2]) != 3 or int(shape[0]) <= 0 or int(shape[1]) <= 0:
            raise GramHeadError(f"gramhead: frames must be (H, W, 3) uint8, got shape {tuple(shape)}")
        h, w = int(shape[0]), int(shape[1])
        rh, rw = _resize_output_size(h, w, resize)
        top, left, oh, ow = 0, 0, rh, rw
        if crop is not None:
            oh, ow = (int(crop), int(crop)) if not isinstance(crop, (tuple, list)) else (int(crop[0]), int(crop[-1]))
            if oh > rh or ow > rw:
                raise GramHeadError("gramhead: CenterCrop larger than the resized frame is not supported on the GPU path")
            top, left = int(round((rh - oh) / 2.0)), int(round((rw - ow) / 2.0))     # half to even, as torchvision
        geometry.append((h, w, rh, rw, top, left, oh, ow))
    if not geometry:
        raise GramHeadError("gramhead: a frame batch needs at least one frame slot")
    sizes = sorted({g[6:] for g in geometry})
    if len(sizes) != 1:
        raise GramHeadError(f"gramhead: the frames come out of the transform at different sizes {sizes}; one batch needs "
                            "one size (Resize((h, w)), or a CenterCrop)")
    return geometry, sizes[0]


def pack_frame_tables(frame_shapes, resize, crop=None):
    """Resample tables of N frame slots, packed for gh_preprocess_frames.

    Returns dict(out_hw=(oh, ow), tables=int32 array, offsets=(N, 6) int64 (start of hx_min, hx_size, hk, vy_min,
    vy_size, vk of each slot in `tables`), hkmax, vkmax, rows=[(vy_min, vy_size)] per slot). Coefficient rows are padded
    with zeros to the largest kmax of the batch. Every slot must resize [and crop] to the same size."""
    geometry, (oh, ow) = frame_geometry(frame_shapes, resize, crop)
    hx = [resample_tables(w, rw, left, ow) for h, w, rh, rw, top, left, _, _ in geometry]
    vy = [resample_tables(h, rh, top, oh) for h, w, rh, rw, top, left, _, _ in geometry]
    hkmax = max(t[2].shape[1] for t in hx)
    vkmax = max(t[2].shape[1] for t in vy)
    parts, offsets, pos = [], [], 0
    for (x0, xn, xk), (y0, yn, yk) in zip(hx, vy):
        xk = np.pad(xk, ((0, 0), (0, hkmax - xk.shape[1])))
        yk = np.pad(yk, ((0, 0), (0, vkmax - yk.shape[1])))
        row = []
        for a in (x0, xn, xk, y0, yn, yk):
            row.append(pos)
            parts.append(a.ravel())
            pos += a.size
        offsets.append(row)
    return dict(out_hw=(oh, ow), tables=np.concatenate(parts).astype(np.int32), offsets=np.array(offsets, np.int64),
                hkmax=hkmax, vkmax=vkmax, rows=[(t[0], t[1]) for t in vy])


def band_span(rows, band_rows: int) -> int:
    """The most input rows a band of `band_rows` consecutive output rows (bands start at multiples of band_rows) reads,
    over every slot; rows: pack_frame_tables(...)["rows"]."""
    span = 0
    for y0, yn in rows:
        starts = np.arange(0, len(y0), band_rows)
        lo, hi = np.minimum.reduceat(y0, starts), np.maximum.reduceat(y0 + yn, starts)
        span = max(span, int((hi - lo).max()))
    return span


def max_band_rows(rows, ow: int, budget: int = _BAND_SMEM_BUDGET) -> int:
    """The tallest band whose input rows fit in `budget` bytes of shared memory (gh_preprocess_frames_smem); 1 when even
    one output row needs more (one row always runs if the kernel can hold it at all)."""
    lib = _lib.lib()
    best = 1
    for r in range(2, len(rows[0][0]) + 1):
        smem = lib.gh_preprocess_frames_smem(ow, band_span(rows, r))
        if smem < 0 or smem > budget:
            break
        best = r
    return best


def band_span_bound(h, rh, band_rows):
    """An upper bound of band_span from the shapes alone, for images of heights h resized to rh (arrays): output rows
    y .. y + R - 1 read input rows [int(c(y) - s + 0.5), int(c(y + R - 1) + s + 0.5)) with c(y) = (y + 0.5) * scale and
    s = max(scale, 1), fewer than (R - 1) * scale + 2 s + 1 of them; one more row absorbs the rounding of those fp64
    values, and no band reads more than the image's h rows. band_rows: an int, or an array of them (one bound each)."""
    h, rh = np.asarray(h, dtype=np.int64), np.asarray(rh, dtype=np.int64)
    scale = h / rh
    r = np.asarray(band_rows, dtype=np.int64)[..., None]
    bound = np.ceil((r - 1) * scale) + 2 * np.ceil(np.maximum(scale, 1.0)) + 2
    return np.minimum(bound, h).max(axis=-1).astype(np.int64)


# columns of a loader batch's geometry (functions.PackedImages, gh_frame_tables): per image H, W, the byte offset of its
# pixels in the packed buffer, the resized rh, rw, and the centre crop's top, left
GEOMETRY_COLUMNS = ("H", "W", "offset", "rh", "rw", "top", "left")
_SM_COUNTS = {}


def resample_images(pixels: torch.Tensor, geometry: torch.Tensor, geometry_host: np.ndarray, out: torch.Tensor,
                    hkmax: int, vkmax: int, tables: Optional[torch.Tensor] = None,
                    frames: Optional[torch.Tensor] = None) -> torch.Tensor:
    """N RGB images of any sizes, packed in one flat uint8 device buffer, -> Resize [+ CenterCrop] of each as one
    (N, 3, oh, ow) uint8 batch in `out`, bit for bit torchvision's on the PIL images. The resample tables are built on the
    device from the geometry (gh_frame_tables), then gh_preprocess_frames resamples; nothing per output coordinate runs
    on the host. geometry: (N, 7) int64 on the device (GEOMETRY_COLUMNS), geometry_host: the same values on the host
    (checked here, and used to pick the band height). tables / frames: optional int32 / uint8 device buffers of at least
    N * gh_frame_tables_stride(...) ints / N * 80 bytes (allocated when None). Runs on the current stream."""
    lib = _lib.lib()
    g = np.asarray(geometry_host, dtype=np.int64)
    n = len(g)
    if (out.dim() != 4 or out.dtype != torch.uint8 or not out.is_contiguous() or tuple(out.shape[:2]) != (n, 3)
            or g.shape != (n, 7) or n == 0 or tuple(geometry.shape) != g.shape):
        raise GramHeadError("gramhead: resample_images needs (N, 7) geometry and a dense (N, 3, oh, ow) uint8 output")
    for t, dtype in ((pixels, torch.uint8), (geometry, torch.int64)):
        if t.device != out.device or t.dtype != dtype or not t.is_contiguous():
            raise GramHeadError("gramhead: resample_images: pixels (uint8) and geometry (int64) must be dense, on out's device")
    oh, ow = int(out.shape[2]), int(out.shape[3])
    h, w, off, rh, rw, top, left = g.T
    if (h.min() <= 0 or w.min() <= 0 or off.min() < 0 or int((off + h * w * 3).max()) > pixels.numel()
            or (top < 0).any() or (left < 0).any() or (top + oh > rh).any() or (left + ow > rw).any()
            or max(resample_kmax(a, b) for a, b in zip(w, rw)) > hkmax
            or max(resample_kmax(a, b) for a, b in zip(h, rh)) > vkmax):
        raise GramHeadError("gramhead: resample_images: the geometry does not fit the pixels, the output or kmax")
    stride = lib.gh_frame_tables_stride(oh, ow, hkmax, vkmax)
    if stride < 0:
        check(int(stride), "gh_frame_tables_stride")
    if tables is None:
        tables = torch.empty(n * stride, dtype=torch.int32, device=out.device)
    if frames is None:
        frames = torch.empty(n * FRAME_DESC_DTYPE.itemsize, dtype=torch.uint8, device=out.device)
    if (tables.numel() < n * stride or tables.dtype != torch.int32 or frames.numel() < n * FRAME_DESC_DTYPE.itemsize
            or frames.dtype != torch.uint8 or tables.device != out.device or frames.device != out.device):
        raise GramHeadError("gramhead: resample_images: the tables / frames buffers are too small")
    dev = out.device
    if dev not in _SM_COUNTS:
        _SM_COUNTS[dev] = torch.cuda.get_device_properties(dev).multi_processor_count
    band, span = images_band_rows(h, rh, oh, ow, vkmax, _SM_COUNTS[dev])
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        check(lib.gh_frame_tables(geometry.data_ptr(), n, pixels.data_ptr(), oh, ow, hkmax, vkmax, tables.data_ptr(),
                                  frames.data_ptr(), stream), "gh_frame_tables")
        check(lib.gh_preprocess_frames(frames.data_ptr(), n, oh, ow, band, span, tables.data_ptr(), hkmax, vkmax,
                                       out.data_ptr(), stream), "gh_preprocess_frames")
    return out


def images_band_rows(h, rh, oh: int, ow: int, vkmax: int, sms: int):
    """(band_rows, span_rows) of gh_preprocess_frames for images of heights h resized to rh, from the shapes alone
    (band_span_bound; the host has no tables): bands as tall as the shared-memory budget allows, but not so tall that the
    grid leaves SMs without two CTAs."""
    rows = np.arange(1, oh + 1)
    spans = np.maximum(band_span_bound(h, rh, rows), vkmax)
    fits = np.nonzero(3 * ow * spans <= _BAND_SMEM_BUDGET)[0]
    band = max(1, min(int(fits[-1]) + 1 if fits.size else 1, -(-len(h) * oh // (2 * sms))))
    return band, int(spans[band - 1])


class FrameBatchPipeline:
    """N frames (H_i, W_i, 3) uint8 numpy -> probabilities (N, num_classes) numpy, one forward for all of them: the
    CameraPipeline of several cameras or of consecutive video frames. Slot i takes frames of shape frame_shapes[i]; every
    slot must come out of resize [+ crop] at the same size. The model (either model class, on a CUDA device) is unchanged:
    it gets the uint8 batch with this transform's Normalize for this call only (the fused uint8 stem on the fp32 inference
    plan), which is bit for bit the fp32 batch CameraPipeline would give it.

      frames --memcpy--> one pinned arena --one H2D--> gh_preprocess_frames (N frames -> (N, 3, oh, ow) uint8)
      --> model --> softmax --D2H--> pinned (N, num_classes)

    Everything between the two host buffers is one CUDA graph (use_graph=True), replayed per call."""

    def __init__(self, model, frame_shapes, resize, crop=None, mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225),
                 bgr: bool = True, use_graph: bool = True):
        self.model = model
        self.device = torch.device(model.device)
        if self.device.type != "cuda":
            raise GramHeadError("gramhead: FrameBatchPipeline needs the model on a CUDA device (there is no CPU path)")
        mean, std = tuple(float(v) for v in mean), tuple(float(v) for v in std)
        if len(mean) != 3 or len(std) != 3:
            raise GramHeadError(f"gramhead: Normalize needs 3 means and 3 stds, got {len(mean)} and {len(std)}")
        self._normalize = (mean, std)
        packed = pack_frame_tables(frame_shapes, resize, crop)
        self.frame_shapes = [(int(s[0]), int(s[1]), 3) for s in frame_shapes]
        self.out_hw, self.bgr = packed["out_hw"], bool(bgr)
        self._hkmax, self._vkmax, self._rows = packed["hkmax"], packed["vkmax"], packed["rows"]
        n, dev = len(self.frame_shapes), self.device
        sizes = [h * w * 3 for h, w, _ in self.frame_shapes]
        starts = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        self._frames_pin = torch.empty(int(starts[-1]), dtype=torch.uint8).pin_memory()
        arena = self._frames_pin.numpy()
        self._slots = [arena[starts[i]:starts[i + 1]].reshape(self.frame_shapes[i]) for i in range(n)]
        self._frames_dev = torch.empty(int(starts[-1]), dtype=torch.uint8, device=dev)
        desc = np.zeros(n, dtype=FRAME_DESC_DTYPE)
        desc["frame"] = self._frames_dev.data_ptr() + starts[:-1]
        desc["pitch"] = [w * 3 for _, w, _ in self.frame_shapes]
        desc["H"] = [h for h, _, _ in self.frame_shapes]
        desc["W"] = [w for _, w, _ in self.frame_shapes]
        desc["bgr"] = int(self.bgr)
        for j, name in enumerate(_TABLE_FIELDS):
            desc[name] = packed["offsets"][:, j]
        self._desc = torch.from_numpy(desc.view(np.uint8).copy()).to(dev)
        self._tables = torch.from_numpy(packed["tables"]).to(dev)
        oh, ow = self.out_hw
        self.max_band_rows = max_band_rows(self._rows, ow)
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        # as tall a band as the budget allows, but not so tall that the grid leaves SMs without two CTAs
        self.band_rows = max(1, min(self.max_band_rows, -(-n * oh // (2 * sms))))
        self._input = torch.empty((n, 3, oh, ow), dtype=torch.uint8, device=dev)
        self._probs_dev = None
        self._probs_pin = None
        self._graph = None
        self._done = torch.cuda.Event()
        model.eval()
        with torch.cuda.device(dev), torch.no_grad():
            self._body()                                  # allocates the output buffers, loads every kernel
            torch.cuda.synchronize(dev)
            if use_graph:
                side = torch.cuda.Stream(device=dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):
                    for _ in range(2):
                        self._body()
                torch.cuda.current_stream(dev).wait_stream(side)
                torch.cuda.synchronize(dev)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    self._body()
                self._graph = graph
                # the graph holds raw addresses of the model's folded inference plan: keep it alive with the pipeline
                self._captured_plan = getattr(model, "_plan", None)

    def preprocess_(self, band_rows: Optional[int] = None):
        """Runs gh_preprocess_frames on the uploaded frames; result in self._input (N, 3, oh, ow) uint8, RGB.
        band_rows: output rows per CTA, 1 .. max_band_rows (default: self.band_rows)."""
        r = self.band_rows if band_rows is None else int(band_rows)
        if not 1 <= r <= self.max_band_rows:
            raise GramHeadError(f"gramhead: band_rows must be in [1, {self.max_band_rows}], got {band_rows}")
        oh, ow = self.out_hw
        span = max(band_span(self._rows, r), self._vkmax)
        rc = _lib.lib().gh_preprocess_frames(
            self._desc.data_ptr(), len(self.frame_shapes), oh, ow, r, span, self._tables.data_ptr(), self._hkmax,
            self._vkmax, self._input.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream)
        check(rc, "gh_preprocess_frames")
        return self._input

    def _body(self):
        self._frames_dev.copy_(self._frames_pin, non_blocking=True)
        self.preprocess_()
        out = self.model._head(self._input, normalize=self._normalize)
        logits = out[1] if isinstance(out, (tuple, list)) else out
        probs = torch.softmax(logits, dim=1)
        if self._probs_dev is None:
            self._probs_dev = torch.empty_like(probs)
            self._probs_pin = torch.empty(probs.shape, dtype=probs.dtype).pin_memory()
        self._probs_dev.copy_(probs)
        self._probs_pin.copy_(self._probs_dev, non_blocking=True)

    def __call__(self, frames) -> np.ndarray:
        if len(frames) != len(self._slots):
            raise GramHeadError(f"gramhead: FrameBatchPipeline was built for {len(self._slots)} frames, got {len(frames)}")
        for i, (frame, shape) in enumerate(zip(frames, self.frame_shapes)):
            if not isinstance(frame, np.ndarray) or frame.dtype != np.uint8 or frame.shape != shape:
                got = (getattr(frame, "dtype", type(frame).__name__), tuple(getattr(frame, "shape", ())))
                raise GramHeadError(f"gramhead: frame {i}: slot {i} takes uint8 frames of shape {shape}, got {got}")
        for slot, frame in zip(self._slots, frames):
            np.copyto(slot, frame)
        with torch.cuda.device(self.device), torch.no_grad():
            if self._graph is not None:
                self._graph.replay()
            else:
                self._body()
            self._done.record(torch.cuda.current_stream(self.device))
        self._done.synchronize()
        return self._probs_pin.numpy().copy()

    @classmethod
    def from_transform(cls, model, transform, frame_shapes, bgr: bool = True, use_graph: bool = True):
        """Pipeline equivalent to `transform` applied to a PIL image of each frame, or None when the transform is not the
        Resize [+ CenterCrop] + ToTensor + Normalize chain the GPU kernel reproduces."""
        spec = parse_transform(transform)
        if spec is None:
            return None
        return cls(model, frame_shapes, spec["resize"], spec["crop"], spec["mean"], spec["std"], bgr=bgr,
                   use_graph=use_graph)
