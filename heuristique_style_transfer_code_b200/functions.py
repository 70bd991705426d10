"""Task-level functions around the Gram + attention model: same names, signatures and observable behaviour as the
reference's functions/functions_RESNET50_Truncate_Gram_Attention.py (cited per function as file:line of that file),
re-written for the B200 module. GUI / plotting imports are lazy, so importing this file needs only torch + numpy.

Not replicated on purpose: the reference switches torch.autograd.set_detect_anomaly(True) on at import (:23).
"""
from __future__ import annotations

import json
import os
import time
from datetime import datetime

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, ops, streaming
from ._lib import GramHeadError
from torch.utils.data import Subset


# ---------------------------------------------------------------------------------------------------------------------
# checkpoints  (:30-120)
# ---------------------------------------------------------------------------------------------------------------------
def load_model(model, model_path, device):
    """Initialise the encoder from a bare-encoder state_dict (:30-59): every checkpoint key `k` other than `fc.*` is
    tried as `truncated_encoder.k`; keys that do not exist in the model are silently dropped; the merged dict is then
    loaded strictly. Raises FileNotFoundError when the file is missing."""
    if not os.path.isfile(model_path):
        raise FileNotFoundError(f"No model found at {model_path}")
    print(f"Loading pre-trained ResNet50 model from {model_path}")
    checkpoint = torch.load(model_path, map_location=device)
    merged = model.state_dict()
    for key, value in checkpoint.items():
        if key.startswith('fc.'):
            continue
        target = f"truncated_encoder.{key}"
        if target in merged:
            merged[target] = value
    model.load_state_dict(merged, strict=True)
    print("Model loaded successfully.")


_SECTIONS = ('truncated_encoder', 'classifier', 'attention')


def save_model_weights(model, save_path):
    """Three-section checkpoint {'truncated_encoder', 'classifier', 'attention'} of sub-state-dicts (:63-70)."""
    torch.save({name: getattr(model, name).state_dict() for name in _SECTIONS}, save_path)
    print(f"Model weights saved to {save_path}")


def load_model_weights(model, load_path):
    """Loads a three-section checkpoint strictly, section by section, warning about absent sections; if that raises
    KeyError/RuntimeError, re-reads the file as a flat dict with `<section>.` prefixes (:73-120). A missing file is
    reported and ignored."""
    if not os.path.isfile(load_path):
        print(f"No weights file found at {load_path}. Proceeding without loading weights.")
        return
    state = torch.load(load_path, map_location=model.device)
    try:
        for name in _SECTIONS:
            if name in state:
                getattr(model, name).load_state_dict(state[name], strict=True)
            else:
                print(f"Warning: '{name}' not found in state_dict.")
        print(f"Model weights loaded from {load_path} using direct method.")
    except (KeyError, RuntimeError) as err:
        print(f"Direct loading failed with error: {err}")
        print("Attempting to load weights by processing keys...")
        split = {name: {} for name in _SECTIONS}
        for key, value in state.items():
            for name in _SECTIONS:
                if key.startswith(name):
                    split[name][key.replace(f'{name}.', '')] = value
                    break
        for name in _SECTIONS:
            getattr(model, name).load_state_dict(split[name], strict=True)
        print(f"Model weights loaded from {load_path} by processing keys.")


def set_parameter_requires_grad(model, freeze_encoder):
    """freeze_encoder: only parameters whose name contains 'classifier' or 'attention' stay trainable (:226-236)."""
    for name, param in model.named_parameters():
        if not freeze_encoder:
            param.requires_grad = True
        elif "classifier" in name or "attention" in name:
            param.requires_grad = True
            print(f"Layer {name} is unfrozen.")
        else:
            param.requires_grad = False


# ---------------------------------------------------------------------------------------------------------------------
# training / evaluation loops  (:123-224)
# ---------------------------------------------------------------------------------------------------------------------
def _default_device():
    return torch.device('cuda' if torch.cuda.is_available() else 'cpu')


_COPY_STREAMS = {}


def _copy_stream(device):
    """One upload stream per device for the life of the process: the caching allocator keeps a block pool per stream,
    so a fresh stream per loop would strand the previous loop's staging buffers and allocate new ones."""
    key = (device.type, torch.cuda.current_device() if device.index is None else device.index)
    if key not in _COPY_STREAMS:
        _COPY_STREAMS[key] = torch.cuda.Stream(device=device)
    return _COPY_STREAMS[key]


IMAGENET_MEAN, IMAGENET_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
# What a uint8 image batch handed to cuda_prefetch (and so to the train / evaluation loops) is normalised with on the
# device: the constants of the reference's loaders (test_RESNET50_Truncate_gram_attention.py:65,
# train_best_RESNET50_Truncate_gram_attention.py:43). None leaves uint8 tensors as they are.
UINT8_NORMALIZE = (IMAGENET_MEAN, IMAGENET_STD)


def uint8_transform(resize=256, crop=224):
    """Loader transform for the opt-in uint8 upload: the reference's Resize + CenterCrop (test_...:62-63) followed by
    PILToTensor instead of ToTensor + Normalize (:64-65). The batches are then (B, 3, H, W) uint8 -- a quarter of the
    host->device bytes -- and cuda_prefetch applies ToTensor's /255 and Normalize on the GPU (ops.normalize_u8), giving the
    model bit for bit the fp32 batch the reference's transform would have produced on the host."""
    from torchvision import transforms
    steps = [transforms.Resize(resize)] if resize else []
    if crop:
        steps.append(transforms.CenterCrop(crop))
    return transforms.Compose(steps + [transforms.PILToTensor()])


class PackedImages:
    """A loader batch of decoded RGB images of any sizes, built by GpuResizeTransform.collate in the worker:
    `pixels`, one flat uint8 tensor holding every (H, W, 3) image back to back; `geometry`, (N, 7) int64 per image
    (streaming.GEOMETRY_COLUMNS: H, W, byte offset in `pixels`, resized rh, rw, crop top, left); `labels` as the default
    collate makes them; and what cuda_prefetch needs to resample them: the transform's `resize` / `crop`, the common
    output size `out_hw` and the largest coefficient counts `kmax` = (hkmax, vkmax). pin_memory() lets
    DataLoader(pin_memory=True) pin it like any other batch.

    With decode="gpu", `jpeg` = (scan, segs, imgs, tables) holds the compressed part (jpeg.pack) of the images the device
    decodes, `files` their paths (the bytes of a file parsed without one; only CPU runs read them, with Pillow), and
    `arena_bytes` the size of the pixel arena: `pixels` holds only the images the worker decoded, at the start of the
    arena, and the geometry's offsets place every image in it."""

    def __init__(self, pixels, geometry, labels, resize, crop, out_hw, kmax, jpeg=None, files=None, arena_bytes=None):
        self.pixels, self.geometry, self.labels = pixels, geometry, labels
        self.resize, self.crop, self.out_hw, self.kmax = resize, crop, tuple(out_hw), tuple(kmax)
        self.jpeg, self.files = jpeg, files
        self.arena_bytes = int(pixels.numel()) if arena_bytes is None else int(arena_bytes)

    def __len__(self):
        return int(self.geometry.shape[0])

    def pin_memory(self):
        labels = self.labels.pin_memory() if torch.is_tensor(self.labels) else self.labels
        jpeg = None if self.jpeg is None else tuple(t.pin_memory() for t in self.jpeg)
        return PackedImages(self.pixels.pin_memory(), self.geometry.pin_memory(), labels, self.resize, self.crop,
                            self.out_hw, self.kmax, jpeg, self.files, self.arena_bytes)

    def images(self):
        """The (H, W, 3) uint8 images, as numpy views of `pixels` (decoded with Pillow for the device-decoded files)."""
        flat = self.pixels.numpy()
        out = [None if o + h * w * 3 > flat.size else flat[o:o + h * w * 3].reshape(h, w, 3)
               for h, w, o in self.geometry[:, :3].tolist()]
        if self.jpeg is not None:
            import io
            from PIL import Image
            for row, src in zip(self.jpeg[2][:, 12].tolist(), self.files):
                out[row] = np.asarray(Image.open(io.BytesIO(src) if isinstance(src, bytes) else src).convert("RGB"))
        return out

    def host_batch(self):
        """The (N, 3, oh, ow) uint8 batch torchvision's own Resize + CenterCrop + PILToTensor give on the host (CPU runs)."""
        from PIL import Image
        from torchvision import transforms
        steps = [transforms.Resize(self.resize)] + ([transforms.CenterCrop(self.crop)] if self.crop else [])
        tf = transforms.Compose(steps + [transforms.PILToTensor()])
        return torch.stack([tf(Image.fromarray(img, "RGB")) for img in self.images()])


class GpuResizeTransform:
    """Loader side of Resize + CenterCrop on the GPU (gpu_resize_transform). As the dataset's `transform` it maps an RGB
    PIL image to its decoded (H, W, 3) uint8 pixels, without resampling; `.collate` is the DataLoader's collate_fn and
    packs a batch of them into a PackedImages. cuda_prefetch then uploads the pixels, builds the resample tables on the
    device and resamples the batch there, bit for bit what Resize(resize) + CenterCrop(crop) + PILToTensor give on the
    host, before the usual ToTensor + Normalize of uint8 batches."""

    def __init__(self, resize=256, crop=224, interpolation="bilinear", max_size=None, decode="host"):
        from torchvision.transforms import InterpolationMode
        if decode not in ("host", "gpu"):
            raise ValueError(f"gpu_resize_transform: decode must be 'host' or 'gpu', got {decode!r}")
        self.decode = decode
        if InterpolationMode(interpolation) != InterpolationMode.BILINEAR:
            raise ValueError(f"gpu_resize_transform: only bilinear interpolation is reproduced on the GPU, got {interpolation!r}")
        if max_size is not None:
            raise ValueError("gpu_resize_transform: Resize(max_size=...) is not reproduced on the GPU")
        pair = lambda v: (int(v), int(v)) if not isinstance(v, (tuple, list)) else (int(v[0]), int(v[-1]))
        if resize is None or (isinstance(resize, (tuple, list)) and len(resize) not in (1, 2)):
            raise ValueError(f"gpu_resize_transform: resize must be an int or an (h, w) pair, got {resize!r}")
        if isinstance(resize, (tuple, list)) and len(resize) == 1:
            resize = int(resize[0])
        if crop is None and not isinstance(resize, (tuple, list)):
            raise ValueError("gpu_resize_transform: Resize(int) without a CenterCrop gives each image its own size; one "
                             "batch needs one size (give a crop, or resize to an (h, w) pair)")
        if min(pair(resize)) <= 0 or (crop is not None and min(pair(crop)) <= 0):
            raise ValueError(f"gpu_resize_transform: sizes must be positive, got resize={resize!r}, crop={crop!r}")
        if crop is not None:
            ch, cw = pair(crop)
            # Resize(int) makes the short side `resize` and the long side at least that
            lo_h, lo_w = pair(resize)
            if ch > lo_h or cw > lo_w:
                raise ValueError(f"gpu_resize_transform: CenterCrop({crop!r}) is larger than Resize({resize!r}) can give "
                                 "(torchvision would pad); not reproduced on the GPU")
        self.resize = tuple(int(v) for v in resize) if isinstance(resize, (tuple, list)) else int(resize)
        self.crop = None if crop is None else pair(crop)

    def loader(self, path):
        """decode="gpu": the dataset's loader. Reads the file; Image.open without loading pixels gives Pillow's own
        decompression-bomb check and its error on files that are not images. A baseline JPEG the device decodes comes
        back as a jpeg.JpegFile; any other file is decoded here exactly as torchvision's default_loader does."""
        import io
        from PIL import Image
        from . import jpeg
        if self.decode != "gpu":
            raise ValueError('gpu_resize_transform: .loader is for decode="gpu"')
        with open(path, "rb") as f:
            data = f.read()
        img = Image.open(io.BytesIO(data))
        parsed = jpeg.parse(data) if img.format == "JPEG" else None
        if parsed is not None and parsed.W == img.size[0] and parsed.H == img.size[1]:
            parsed.path = path
            return parsed
        return img.convert("RGB")

    def __call__(self, img):
        from . import jpeg
        if isinstance(img, jpeg.JpegFile):
            return img
        if getattr(img, "mode", None) != "RGB":
            raise ValueError(f"gpu_resize_transform: takes RGB PIL images, got {getattr(img, 'mode', type(img).__name__)!r}")
        return torch.from_numpy(np.array(img, dtype=np.uint8))

    def collate(self, batch):
        """[(pixels (H, W, 3) uint8, label), ...] -> PackedImages (pixels, geometry, labels built here, in the worker).
        decode="gpu": items may be jpeg.JpegFile too; their compressed part goes into PackedImages.jpeg and their pixels
        are placed after the worker-decoded ones in the arena."""
        from torch.utils.data import default_collate
        from . import jpeg
        images = [img for img, _ in batch]
        dev = [isinstance(img, jpeg.JpegFile) for img in images]
        for img, d in zip(images, dev):
            if not d and (not torch.is_tensor(img) or img.dtype != torch.uint8 or img.dim() != 3 or img.shape[2] != 3):
                raise ValueError("gpu_resize_transform.collate: expects the (H, W, 3) uint8 tensors of its transform")
        geometry, out_hw = streaming.frame_geometry([tuple(img.shape) for img in images], self.resize, self.crop)
        sizes = [int(np.prod(img.shape)) for img in images]
        order = [i for i in range(len(images)) if not dev[i]] + [i for i in range(len(images)) if dev[i]]
        offsets = np.zeros(len(images), np.int64)
        offsets[order] = np.concatenate([[0], np.cumsum([sizes[i] for i in order])[:-1]])
        host_bytes = sum(sizes[i] for i in range(len(images)) if not dev[i])
        pixels = torch.empty(host_bytes, dtype=torch.uint8)
        for img, o, s, d in zip(images, offsets, sizes, dev):
            if not d:
                pixels[o:o + s].copy_(img.reshape(-1))
        geom = torch.tensor([(h, w, int(o), rh, rw, top, left) for (h, w, rh, rw, top, left, _, _), o in zip(geometry, offsets)],
                            dtype=torch.int64)
        kmax = (max(streaming.resample_kmax(g[1], g[3]) for g in geometry),
                max(streaming.resample_kmax(g[0], g[2]) for g in geometry))
        packed, files = None, None
        if any(dev):
            rows = [i for i in range(len(images)) if dev[i]]
            packed = jpeg.pack([images[i] for i in rows], offsets[rows], rows)
            files = [images[i].path or images[i].data for i in rows]      # bytes only without a path
        return PackedImages(pixels, geom, default_collate([label for _, label in batch]), self.resize, self.crop, out_hw,
                            kmax, packed, files, sum(sizes))


def gpu_resize_transform(resize=256, crop=224, interpolation="bilinear", max_size=None, decode="host"):
    """Opt-in loader transform that moves Resize + CenterCrop (the reference's test_...:62-63) to the GPU, for loaders
    whose images have any sizes:

        t = functions.gpu_resize_transform(256, 224)
        loader = DataLoader(ImageFolder(root, transform=t), batch_size=..., collate_fn=t.collate, pin_memory=True)

    The workers only decode; cuda_prefetch (and so train_model / evaluate_model / evaluate_model_test) uploads the
    decoded pixels, resamples them on the device bit for bit as the host transforms would, and hands on the same
    (B, 3, oh, ow) batch as a uint8_transform() loader. The upload is the decoded pixels (H * W * 3 bytes per image)
    rather than the resampled ones. Raises ValueError for what the kernel does not reproduce: another interpolation,
    max_size, or a crop larger than the resize.

    decode="gpu" also moves the decoding of baseline JPEG files to the device; give the dataset the transform's loader:

        t = functions.gpu_resize_transform(256, 224, decode="gpu")
        loader = DataLoader(ImageFolder(root, loader=t.loader, transform=t), batch_size=..., collate_fn=t.collate,
                            pin_memory=True)

    The workers then only read those files and parse their headers; the upload is the compressed scan data, and the
    device decodes it bit for bit as Pillow does (csrc/jpeg.cuh). Every other file (progressive, arithmetic-coded, CMYK,
    12-bit, PNG, ...) is decoded in the worker as before."""
    return GpuResizeTransform(resize, crop, interpolation, max_size, decode)


def _is_uint8_images(t):
    return torch.is_tensor(t) and t.dtype == torch.uint8 and t.dim() == 4 and 1 <= t.shape[1] <= 4


_normalize_host = ops.normalize_u8_host       # CPU runs of the loops; models with input normalisation use it too


def cuda_prefetch(batches, device, reuse_buffers=False, normalize="default"):
    """Yields the batches of `batches` (tuples / lists of tensors, e.g. a DataLoader) already on `device`.
    On CUDA, batch i+1 is uploaded on a side stream while batch i is being processed, so the host->device copy
    (154 MB for 256 images at 224x224) leaves the critical path; use pin_memory=True loaders for the copy to be
    asynchronous. The reference moves every batch synchronously inside its loops (functions:129-130, :157-158, :190).

    reuse_buffers=True uploads into two fixed sets of device buffers instead of allocating per batch (no allocator
    traffic, constant memory): a yielded batch is then only valid until the next one is requested -- what loops that
    consume a batch and move on (this package's train / evaluation loops) need; leave it False when batches are kept.

    normalize: (mean, std) applied on the device to every (B, C <= 4, H, W) uint8 tensor of a batch after its upload --
    ToTensor's /255 and Normalize, bit-identical to the host transforms (ops.normalize_u8), for loaders built with
    uint8_transform(); "default" takes functions.UINT8_NORMALIZE (the reference's ImageNet constants), None disables it.

    A PackedImages batch (gpu_resize_transform's collate) is yielded as (images, labels): its decoded pixels and geometry
    are uploaded, resampled on the device (streaming.resample_images) into a (B, 3, oh, ow) uint8 batch, which `normalize`
    then treats as any uint8 batch. With reuse_buffers=True its variable-size buffers (pixels, tables) grow with the
    largest batch seen instead of being allocated per batch. On a CPU device, torchvision's own Resize / CenterCrop /
    PILToTensor resample the images."""
    device = torch.device(device)
    if normalize == "default":
        normalize = UINT8_NORMALIZE
    if device.type != 'cuda':
        for batch in batches:
            if isinstance(batch, PackedImages):
                batch = (batch.host_batch(), batch.labels)
            yield tuple((_normalize_host(t, *normalize) if normalize is not None and _is_uint8_images(t) else t.to(device))
                        if torch.is_tensor(t) else t for t in batch)
        return
    copy_stream = _copy_stream(device)
    # Uploads of this generator start after everything already queued on the consumer's stream: buffers of an earlier
    # generator that the caching allocator hands back to the copy stream may still be read by that queued work.
    copy_stream.wait_stream(torch.cuda.current_stream(device))
    slots = [None, None]              # per slot: list of device buffers (one per tensor position of the batch)
    consumed = [None, None]           # per slot: event on the consumer's stream after its last use of the slot
    count = 0

    def staged(slot, key, shape, dtype):
        bufs = slots[slot]
        buf = bufs.get(key)
        if buf is None or buf.dtype != dtype or buf.shape[1:] != shape[1:] or buf.shape[0] < shape[0]:
            buf = torch.empty(shape, dtype=dtype, device=device)
            bufs[key] = buf
        return buf[:shape[0]]

    def place(slot, pos, t):
        pixels = normalize is not None and _is_uint8_images(t)
        if not reuse_buffers or t.dim() == 0:
            moved = t.to(device, non_blocking=True)
            return ops.normalize_u8(moved, *normalize) if pixels else moved
        view = staged(slot, pos, t.shape, t.dtype)
        view.copy_(t, non_blocking=True)
        if pixels:                                 # the uint8 pixels stay in their own staging buffer of the slot
            return ops.normalize_u8(view, *normalize, out=staged(slot, (pos, "fp32"), t.shape, torch.float32))
        return view

    def grown(slot, key, numel, dtype):
        """A flat buffer of the slot with room for `numel` elements, reallocated (with 1/8 headroom) only to grow."""
        buf = slots[slot].get(key)
        if buf is None or buf.numel() < numel:
            buf = torch.empty(numel + numel // 8, dtype=dtype, device=device)
            slots[slot][key] = buf
        return buf[:numel]

    def resample(slot, packed):
        n, (oh, ow), (hkmax, vkmax) = len(packed), packed.out_hw, packed.kmax
        tables = frames = None
        jp = packed.jpeg
        if reuse_buffers:
            src = grown(slot, "packed", packed.arena_bytes, torch.uint8)
            src[:packed.pixels.numel()].copy_(packed.pixels, non_blocking=True)
            geometry = staged(slot, "geometry", packed.geometry.shape, torch.int64)
            geometry.copy_(packed.geometry, non_blocking=True)
            tables = grown(slot, "tables", n * _lib.lib().gh_frame_tables_stride(oh, ow, hkmax, vkmax), torch.int32)
            frames = grown(slot, "frames", n * streaming.FRAME_DESC_DTYPE.itemsize, torch.uint8)
            out = staged(slot, "images", (n, 3, oh, ow), torch.uint8)
        else:
            if jp is None:
                src = packed.pixels.to(device, non_blocking=True)
            else:
                src = torch.empty(packed.arena_bytes, dtype=torch.uint8, device=device)
                src[:packed.pixels.numel()].copy_(packed.pixels, non_blocking=True)
            geometry = packed.geometry.to(device, non_blocking=True)
            out = torch.empty((n, 3, oh, ow), dtype=torch.uint8, device=device)
        status = None
        if jp is not None:
            status = decode(slot, packed, src)
        streaming.resample_images(src, geometry, packed.geometry.numpy(), out, hkmax, vkmax, tables, frames)
        if normalize is not None:
            out = ops.normalize_u8(out, *normalize,
                                   out=staged(slot, "images_fp32", out.shape, torch.float32) if reuse_buffers else None)
        return out, status

    def decode(slot, packed, arena):
        """Uploads the compressed part of a decode="gpu" batch and decodes it into the arena; returns the images'
        status words (uploaded to pinned host memory, read when the batch is handed on)."""
        from . import jpeg
        scan_h, segs_h, imgs_h, tables_h = packed.jpeg
        imgs_np, segs_np = imgs_h.numpy(), segs_h.numpy()
        if reuse_buffers:
            up = []
            for key, t in zip(("jscan", "jsegs", "jimgs", "jtables"), packed.jpeg):
                buf = grown(slot, key, t.numel(), t.dtype)
                buf.copy_(t.reshape(-1), non_blocking=True)
                up.append(buf.view(t.shape))
            n_coef, n_plane, n_rec = jpeg.workspace(imgs_np, scan_h.numel(), len(segs_np))
            work = dict(coef=grown(slot, "jcoef", n_coef, torch.int16), planes=grown(slot, "jplanes", n_plane, torch.uint8),
                        records=grown(slot, "jrecords", n_rec // 4, torch.int32),
                        status=grown(slot, "jstatus", len(imgs_np), torch.int32))
        else:
            up, work = [t.to(device, non_blocking=True) for t in packed.jpeg], {}
        status = jpeg.decode_batch(*up, imgs_np, segs_np, arena, packed.arena_bytes, **work)
        host = torch.empty(status.shape, dtype=torch.int32, pin_memory=True)
        host.copy_(status, non_blocking=True)
        return host, imgs_np[:, 12]

    def upload(batch):
        nonlocal count
        slot = count % 2
        count += 1
        if slots[slot] is None:
            slots[slot] = {}
        with torch.cuda.stream(copy_stream):
            if reuse_buffers and consumed[slot] is not None:
                copy_stream.wait_event(consumed[slot])       # the batch that last lived in these buffers is done with
            status = None
            if isinstance(batch, PackedImages):
                labels = batch.labels
                images, status = resample(slot, batch)
                moved = (images, place(slot, 1, labels) if torch.is_tensor(labels) else labels)
            else:
                moved = tuple(place(slot, i, t) if torch.is_tensor(t) else t for i, t in enumerate(batch))
        done = torch.cuda.Event()
        done.record(copy_stream)
        return moved, done, slot, status

    it = iter(batches)
    try:
        pending = upload(next(it))
    except StopIteration:
        return
    try:
        while pending is not None:
            current, done, slot, status = pending
            if status is not None:                  # decode="gpu": no batch is handed on with a broken image in it
                done.synchronize()
                bad = np.flatnonzero(status[0].numpy())
                if bad.size:
                    raise GramHeadError("gramhead: gpu JPEG decoding failed for batch index "
                                        f"{', '.join(str(int(status[1][i])) for i in bad)} (corrupt or truncated scan)")
            main = torch.cuda.current_stream(device)
            main.wait_event(done)
            if not reuse_buffers:
                for t in current:
                    if torch.is_tensor(t):
                        t.record_stream(main)
            yield current
            if reuse_buffers:                       # the consumer has queued everything that reads `current`
                ev = torch.cuda.Event()
                ev.record(torch.cuda.current_stream(device))
                consumed[slot] = ev
            # The next upload is issued AFTER the consumer has queued its work on `current`: the copy still overlaps that
            # work on the GPU (other stream), and a copy call that blocks the host -- pageable source, or a driver that
            # stages a large pinned copy -- no longer holds back the launch of the kernels it is meant to hide behind.
            # (Issued before the yield, such a call serialised copy and compute on some boxes: 8.8 ms instead of 6.3 ms
            # per 256-image step.)
            try:
                pending = upload(next(it))
            except StopIteration:
                pending = None
    finally:
        if reuse_buffers:
            # the staging buffers were allocated on the copy stream but read on the consumer's: tell the allocator, so that
            # they are not handed out again before the consumer's queued work is done with them
            main = torch.cuda.current_stream(device)
            for bufs in slots:
                for buf in (bufs or {}).values():
                    buf.record_stream(main)


class HostCollector:
    """Brings per-batch results to the host without stopping the GPU after every batch.

    The reference reads each batch's outputs with `.cpu().numpy()` (functions:196-199), a device synchronisation per
    batch: the host cannot queue batch i+1 before batch i has finished, so the GPU idles while Python launches the next
    forward. push() instead enqueues non-blocking copies into a small ring of pinned buffers and records an event;
    a slot is only waited for when it comes up for reuse, `depth` batches later (by then its copy is long done), and its
    content is then moved to ordinary host memory. finish() drains the ring. On CPU tensors it degenerates to a list."""

    def __init__(self, depth: int = 4):
        self.depth, self.slots, self.count, self.done = depth, [], 0, []

    def _retire(self, slot):
        bufs, shapes, event = slot
        if event is not None:
            event.synchronize()
        self.done.append(tuple(np.array(b[:n].numpy()) for b, n in zip(bufs, shapes)))

    def push(self, *tensors):
        if not tensors[0].is_cuda:
            self.done.append(tuple(t.detach().cpu().numpy() for t in tensors))
            return
        i = self.count % self.depth
        self.count += 1
        if i < len(self.slots) and self.slots[i] is not None and self.slots[i][2] is not None:
            self._retire(self.slots[i])
        rows = [t.shape[0] for t in tensors]
        reuse = i < len(self.slots) and self.slots[i] is not None and all(
            b.shape[0] >= t.shape[0] and b.shape[1:] == t.shape[1:] and b.dtype == t.dtype
            for b, t in zip(self.slots[i][0], tensors))
        bufs = self.slots[i][0] if reuse else tuple(torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in tensors)
        for b, t in zip(bufs, tensors):
            b[:t.shape[0]].copy_(t.detach(), non_blocking=True)
        event = torch.cuda.Event()
        event.record(torch.cuda.current_stream(tensors[0].device))
        slot = (bufs, rows, event)
        if i < len(self.slots):
            self.slots[i] = slot
        else:
            self.slots.append(slot)

    def finish(self):
        """-> list of per-batch tuples of numpy arrays, in push order."""
        if self.slots:
            n = len(self.slots)
            start = self.count % self.depth if self.count >= self.depth else 0
            for k in range(n):
                slot = self.slots[(start + k) % n]
                if slot is not None and slot[2] is not None:
                    self._retire(slot)
            self.slots = []
        out, self.done, self.count = self.done, [], 0
        return out


def _prefetch_normalize(model):
    """cuda_prefetch's `normalize` for the loops: None when the model (or the one a DDP wrapper holds) normalises uint8
    input itself (set_input_normalization), so that the pixels reach it; cuda_prefetch's default otherwise."""
    inner = getattr(model, "module", model)
    return None if getattr(inner, "input_normalization", None) is not None else "default"


def train_model(model, train_loader, criterion, optimizer, num_epochs=25, writer=None, fold=0):
    """SGD loop of the train script (:123-145): per batch zero_grad / forward / loss / backward / step, a loss print per
    batch, the sample-weighted epoch loss printed and logged as Fold_{fold}/Train/Loss. Returns the model."""
    device = _default_device()
    model.to(device)
    model.train()
    n_batches = len(train_loader)
    for epoch in range(num_epochs):
        running = 0.0
        for step, (inputs, labels) in enumerate(cuda_prefetch(train_loader, device, reuse_buffers=True,
                                                              normalize=_prefetch_normalize(model))):
            optimizer.zero_grad()
            loss = criterion(model(inputs), labels)
            loss.backward()
            optimizer.step()
            value = loss.item()
            running += value * inputs.size(0)
            print(f'Fold {fold}, Epoch [{epoch + 1}/{num_epochs}], Batch [{step + 1}/{n_batches}], Loss: {value:.4f}')
        epoch_loss = running / len(train_loader.dataset)
        print(f'Fold {fold}, Epoch [{epoch + 1}/{num_epochs}], Loss: {epoch_loss:.4f}')
        if writer:
            writer.add_scalar(f"Fold_{fold}/Train/Loss", epoch_loss, epoch)
    return model


class GraphedTrainStep:
    """One training step -- forward, loss, backward (Gram / attention kernels, cuDNN, DDP's gradient all-reduce), optimizer
    step -- captured once in a CUDA graph and replayed: `loss = step(inputs, labels)`.

    The loop body of train_model (reference functions/...:129-137) is ~560 kernel launches; at small per-GPU batches
    (64 images per GPU when a global batch of 512 is sharded over 8 GPUs) the host cannot issue them as fast as the GPU
    executes them and the GPU idles 15 % of the step (profiles/r2_ddp_timeline_8gpu.json). Replaying the captured step
    removes the launches; the arithmetic and its order are the eager step's.

    Requirements: fixed batch shape (the example batch's); an optimizer that can be captured (torch.optim.AdamW / Adam with
    capturable=True, SGD as it is). `model` may be wrapped in DistributedDataParallel -- the NCCL all-reduce is then part of
    the graph. For that, torch's rules for capturing DDP apply: TORCH_NCCL_ASYNC_ERROR_HANDLING=0 in the environment before
    init_process_group, DDP constructed on a side stream (distributed.wrap_ddp(..., for_graph_capture=True)), at least 11
    eager iterations before the capture (the default `warmup`), and the graph must be released before the process group is
    destroyed (call release(); destroy_process_group() hangs otherwise). Measured: 64 images per GPU, 2 GPUs, 20.3 ms eager ->
    14.7 ms replayed (tests/tools/try_ddp_graph.py); one GPU at batch 64: 14.89 -> 14.45 ms."""

    def __init__(self, model, criterion, optimizer, example_inputs, example_labels, warmup=11):
        device = example_inputs.device
        if device.type != 'cuda':
            raise ValueError("GraphedTrainStep needs CUDA tensors")
        self.model, self.criterion, self.optimizer = model, criterion, optimizer
        self.inputs = example_inputs.detach().clone()
        self.labels = example_labels.detach().clone()
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._eager()
        torch.cuda.current_stream(device).wait_stream(side)
        torch.cuda.synchronize(device)
        optimizer.zero_grad(set_to_none=True)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss = self._forward_backward_step()

    def _forward_backward_step(self):
        loss = self.criterion(self.model(self.inputs), self.labels)
        loss.backward()
        self.optimizer.step()
        return loss

    def _eager(self):
        self.optimizer.zero_grad(set_to_none=True)
        return self._forward_backward_step()

    def release(self):
        """Drops the captured graph (and the memory pool it owns). Required before torch.distributed.destroy_process_group()
        when the captured step contains NCCL collectives."""
        self.graph = None
        self.loss = None
        torch.cuda.synchronize(self.inputs.device)

    def __call__(self, inputs=None, labels=None):
        """Copies the batch into the captured buffers (skipped when None: the captured tensors are reused) and replays the
        step. Returns the loss tensor of the captured step (read it with .item() when needed: that is the only sync)."""
        if inputs is not None:
            self.inputs.copy_(inputs, non_blocking=True)
        if labels is not None:
            self.labels.copy_(labels, non_blocking=True)
        self.graph.replay()
        return self.loss


def evaluate_model(model, val_loader, criterion, writer=None, fold=0):
    """Validation pass (:148-176) -> (loss, accuracy, weighted precision, weighted recall)."""
    from sklearn.metrics import precision_score, recall_score
    device = _default_device()
    model.to(device)
    model.eval()
    results = HostCollector()
    with torch.no_grad():
        for inputs, labels in cuda_prefetch(val_loader, device, reuse_buffers=True,
                                            normalize=_prefetch_normalize(model)):
            outputs = model(inputs)
            # the reference reads loss.item() and the predictions after every batch (:160-166); here they ride to the
            # host through the pinned ring and are reduced there afterwards, in the same order and precision
            results.push(criterion(outputs, labels).reshape(1), outputs.argmax(dim=1), labels)
    loss_sum, correct, preds_all, labels_all = 0.0, 0, [], []
    for loss, preds, labels in results.finish():
        loss_sum += float(loss[0]) * len(labels)
        correct += int((preds == labels).sum())
        preds_all.extend(preds)
        labels_all.extend(labels)
    n = len(val_loader.dataset)
    total_loss = loss_sum / n
    accuracy = torch.tensor(correct, dtype=torch.float64) / n
    precision = precision_score(labels_all, preds_all, average='weighted', zero_division=0)
    recall = recall_score(labels_all, preds_all, average='weighted', zero_division=0)
    print(f'Fold {fold}, Validation Loss: {total_loss:.4f}, Accuracy: {accuracy:.4f}, Precision: {precision:.4f}, '
          f'Recall: {recall:.4f}')
    if writer:
        writer.add_scalar(f"Fold_{fold}/Validation/Loss", total_loss)
        writer.add_scalar(f"Fold_{fold}/Validation/Accuracy", accuracy)
        writer.add_scalar(f"Fold_{fold}/Validation/Precision", precision)
        writer.add_scalar(f"Fold_{fold}/Validation/Recall", recall)
    return total_loss, accuracy.item(), precision, recall


def evaluate_model_test(model, data_loader, device):
    """Test pass with the `_for_test` model (:178-224) -> (embeddings (N, g*g), preds, labels, probs (N, nc), paths).
    Image paths are recovered from batch_idx * loader.batch_size, i.e. the loader must not shuffle (as in the reference).
    """
    model.eval()
    paths = []
    dataset = data_loader.dataset
    results = HostCollector()
    with torch.no_grad():
        for batch_idx, (inputs, labels) in enumerate(cuda_prefetch(data_loader, device, reuse_buffers=True,
                                                                   normalize=_prefetch_normalize(model))):
            embeddings, outputs = model(inputs)
            probs = F.softmax(outputs, dim=1)
            preds = outputs.argmax(dim=1)
            results.push(embeddings, probs, preds, labels)      # no per-batch synchronisation (the reference's .cpu())
            first = batch_idx * data_loader.batch_size
            for j in range(inputs.size(0)):
                if isinstance(dataset, Subset):
                    paths.append(dataset.dataset.samples[dataset.indices[first + j]][0])
                else:
                    paths.append(dataset.samples[first + j][0])
    batches = results.finish()
    emb_all, prob_all, pred_all, label_all = ([b[k] for b in batches] for k in range(4))
    return (np.concatenate(emb_all, axis=0), np.concatenate(pred_all, axis=0), np.concatenate(label_all, axis=0),
            np.concatenate(prob_all, axis=0), paths)


# ---------------------------------------------------------------------------------------------------------------------
# style transfer  (:241-314)
# ---------------------------------------------------------------------------------------------------------------------
def denormalize(tensor, mean, std):
    """In-place per-channel x*std + mean (:241-246)."""
    mean = mean.to(tensor.device)
    std = std.to(tensor.device)
    for channel, m, s in zip(tensor, mean, std):
        channel.mul_(s).add_(m)
    return tensor


def _save_side_by_side(path, image):
    try:
        import matplotlib.pyplot as plt
        plt.imsave(path, image)
    except Exception:
        from PIL import Image
        Image.fromarray((np.clip(image, 0, 1) * 255).astype(np.uint8)).save(path)


class _StyleIteration:
    """One optimisation step of style_transfer() -- encoder forward, dense Gram, MSE against the target Gram, backward
    to the image, Adam step -- captured once in a CUDA graph and replayed (SURVEY.md section 8(f) n3).

    At batch 1 the step is ~400 small kernels (cuDNN encoder forward + backward, the dense tcgen05 Gram forward and
    backward, the loss, Adam) and is bound by launch latency, not by any kernel; replaying it as one graph removes
    that. The image, the target Gram and the optimiser state live in static buffers: a new image only copies into them.
    The arithmetic and its order are the eager loop's (reference functions/...:283-299).

    `images` = N > 1 optimises N independent images in one step: the loss is the sum of the per-image losses
    (ops.gram_mse_loss_per_image), so each image gets exactly its own batch-1 d loss / d G; the eval-mode encoder and
    Adam act on each image separately."""

    def __init__(self, model, encoder, device, learning_rate, use_graph=True, images=1):
        self.model, self.encoder, self.device = model, encoder, torch.device(device)
        self.noise = torch.zeros((images, 3, 224, 224), device=self.device, requires_grad=True)
        self.use_graph = bool(use_graph) and self.device.type == 'cuda'
        self.optimizer = torch.optim.Adam([self.noise], lr=learning_rate, capturable=self.use_graph)
        self.mse = nn.MSELoss()
        self.target = None
        self.loss = None
        self.losses = None
        self.graph = None

    def _step(self):
        features = self.encoder(self.noise)
        if features.is_cuda:       # Gram forward, fused loss + dG pass, Gram backward (ops.gram_mse_loss_per_image; reference :286-295)
            losses = ops.gram_mse_loss_per_image(features, self.target)
        else:
            gram = self.model.gram_matrix(features)
            losses = torch.stack([self.mse(gram[b], self.target[b]) for b in range(gram.shape[0])])
        loss = losses.sum()
        loss.backward()
        self.optimizer.step()
        return loss, losses

    def _reset_optimizer(self):
        for state in self.optimizer.state.values():
            for v in state.values():
                if torch.is_tensor(v):
                    v.zero_()

    def start(self, target, noise_init):
        """New images: target Grams (N, C, C) and fresh noise (N, 3, 224, 224); Adam restarts from zero moments (a new
        optimiser upstream)."""
        if self.target is None:
            self.target = target.detach().clone()
        else:
            self.target.copy_(target)
        if self.use_graph and self.graph is None:
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):                     # warm-up off the capture stream (allocations, cuDNN plans)
                for _ in range(3):
                    self.optimizer.zero_grad(set_to_none=True)
                    self._step()
            torch.cuda.current_stream(self.device).wait_stream(side)
            torch.cuda.synchronize(self.device)
            self.optimizer.zero_grad(set_to_none=True)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.loss, self.losses = self._step()
        with torch.no_grad():
            self.noise.copy_(noise_init)
        self._reset_optimizer()

    def _run(self):
        if self.graph is not None:
            self.graph.replay()
        else:
            self.optimizer.zero_grad()
            self.loss, self.losses = self._step()

    def step(self):
        """Runs one iteration and returns the loss (summed over the images) as a Python float (the only
        synchronisation, as upstream)."""
        self._run()
        return self.loss.item()

    def step_losses(self):
        """Runs one iteration and returns the N per-image losses (before the Adam step) as Python floats, from one
        synchronisation."""
        self._run()
        return self.losses.tolist()


def _style_images_per_step(images_per_step, device):
    """images_per_step, or $GRAMHEAD_STYLE_IMAGES when it is None (1 when that is unset too)."""
    if images_per_step is None:
        env = os.environ.get("GRAMHEAD_STYLE_IMAGES", "").strip()
        try:
            images_per_step = int(env) if env else 1
        except ValueError:
            raise ValueError(f"GRAMHEAD_STYLE_IMAGES={env!r} is not an integer") from None
    images_per_step = int(images_per_step)
    if images_per_step < 1:
        raise ValueError(f"images_per_step must be >= 1, got {images_per_step}")
    if images_per_step > 1 and torch.device(device).type != 'cuda':
        raise ValueError("images_per_step > 1 needs a CUDA device")
    return images_per_step


def _optimise_chunk(runner, target, noise0, threshold, num_iterations):
    """Steps runner's N images from noise0 until each one's loss has gone below `threshold` or `num_iterations` ran out.
    -> (results (N, 3, 224, 224), reached): reached[b] is the iteration at which image b's pre-step loss was first below
    threshold (None if never) and results[b] the noise after that step -- what upstream saves after its `break` -- or
    after the last step. A converged image keeps being stepped with the others; its result is copied out on the stream
    before the next step, so it no longer changes."""
    runner.start(target, noise0)
    noise = runner.noise.detach()
    result = torch.empty_like(noise)
    reached = [None] * noise.shape[0]
    for iteration in range(num_iterations):
        for b, loss in enumerate(runner.step_losses()):
            if reached[b] is None and loss < threshold:
                reached[b] = iteration
                result[b].copy_(noise[b])
        if None not in reached:
            break
    for b, it in enumerate(reached):
        if it is None:
            result[b].copy_(noise[b])
    return result, reached


def style_transfer(model, data_loader, device, save_dir, layers=None, threshold=1e-4, num_iterations=500,
                   learning_rate=0.01, use_graph=True, images_per_step=None):
    """For every image: optimise a noise image with Adam so that the dense Gram of the first `layers` encoder children
    matches the image's (MSE), stop below `threshold`, save original|result under save_dir/style_transfer_<date>/<label>
    (:247-314). Both Gram evaluations and the gradient through them go through model.gram_matrix(), i.e. the dense
    tcgen05 forward/backward kernels; on a CUDA device the whole iteration is replayed from one CUDA graph
    (`use_graph=False` runs the eager loop, same arithmetic).

    `images_per_step` (default: $GRAMHEAD_STYLE_IMAGES, else 1) optimises that many images of a loader batch together,
    each with its own loss, Adam state and stopping point: image b's result is the noise after the first iteration whose
    loss was below `threshold`, as in the one-image loop, and the chunk runs until every image got there or
    `num_iterations` ran out. The random noise, the printed lines and the files are those of the one-image loop; the
    images differ from it only by the encoder's batch-size-dependent rounding."""
    per_step = _style_images_per_step(images_per_step, device)
    model.eval()
    out_root = os.path.join(save_dir, f'style_transfer_{datetime.now().strftime("%Y-%m-%d")}')
    os.makedirs(out_root, exist_ok=True)
    mean = torch.tensor([0.485, 0.456, 0.406], device=device)
    std = torch.tensor([0.229, 0.224, 0.225], device=device)
    encoder = nn.Sequential(*list(model.truncated_encoder.children())[:layers]).to(device)
    runners = {}                                      # one per chunk size: the full chunk and a smaller last one
    for inputs, labels in data_loader:
        inputs, labels = inputs.to(device), labels.to(device)
        # file names use the index within the loader batch (as upstream), so a chunk never spans two batches
        for first in range(0, inputs.size(0), per_step):
            chunk = inputs[first:first + per_step]
            n = chunk.size(0)
            with torch.no_grad():
                target = model.gram_matrix(encoder(chunk))
            noise0 = torch.cat([torch.randn((1, 3, 224, 224), device=device) for _ in range(n)])   # upstream's draws
            if n not in runners:
                runners[n] = _StyleIteration(model, encoder, device, learning_rate, use_graph=use_graph, images=n)
            result, reached = _optimise_chunk(runners[n], target, noise0, threshold, num_iterations)
            for b in range(n):
                i = first + b
                if reached[b] is not None:
                    print(f"Seuil atteint pour l'image {i}, itération {reached[b]}")
                class_dir = os.path.join(out_root, str(labels[i].item()))
                os.makedirs(class_dir, exist_ok=True)
                res = denormalize(result[b].cpu(), mean, std).clamp_(0, 1).numpy().transpose(1, 2, 0)
                original = denormalize(chunk[b].detach().cpu(), mean, std).clamp_(0, 1).numpy().transpose(1, 2, 0)
                save_path = os.path.join(class_dir, f'style_transfer_{i}.png')
                _save_side_by_side(save_path, np.hstack((original, res)))
                print(f"Style transféré pour l'image {i}, sauvegardée à {save_path}")


# ---------------------------------------------------------------------------------------------------------------------
# config  (:329-337)
# ---------------------------------------------------------------------------------------------------------------------
def load_hyperparameters(hyperparams_path):
    if not os.path.isfile(hyperparams_path):
        print(f"No hyperparameters file found at {hyperparams_path}. Proceeding with default hyperparameters.")
        return None
    with open(hyperparams_path, 'r') as f:
        hyperparams = json.load(f)
    print(f"Hyperparameters loaded from {hyperparams_path}")
    return hyperparams


# ---------------------------------------------------------------------------------------------------------------------
# t-SNE views (:343-474): CPU/GUI post-processing of the embeddings (sklearn + matplotlib + Tk), outside the accelerated
# path. The names resolve for the reference's test script; the calls are delegated to the reference's own file.
# ---------------------------------------------------------------------------------------------------------------------
_REF_FUNCTIONS = os.path.join("functions", "functions_RESNET50_Truncate_Gram_Attention.py")


def perform_tsne(embeddings, labels, save_path, colors=None):
    from ._reference import load_reference_file
    return load_reference_file(_REF_FUNCTIONS).perform_tsne(embeddings, labels, save_path, colors)


def create_onpick_function(dataset, img_paths, img_label, label_text, classes, labels):
    from ._reference import load_reference_file
    return load_reference_file(_REF_FUNCTIONS).create_onpick_function(dataset, img_paths, img_label, label_text, classes,
                                                                      labels)


def plot_tsne_interactive(embeddings, labels, classes, img_paths, dataset, colors=None):
    from ._reference import load_reference_file
    return load_reference_file(_REF_FUNCTIONS).plot_tsne_interactive(embeddings, labels, classes, img_paths, dataset, colors)


# ---------------------------------------------------------------------------------------------------------------------
# camera streaming  (:477-536)
# ---------------------------------------------------------------------------------------------------------------------
def run_camera(model, transform, class_names, save_video, save_dir, prob_threshold, measure_time, capture=None,
               display=True, max_frames=None, pipeline="auto"):
    """Per frame: BGR->RGB -> PIL -> transform -> model -> softmax -> label overlay; optional video file and
    times_camera.json (:477-536). `capture`, `display`, `max_frames` are additions (defaults reproduce the reference:
    cv2.VideoCapture(0), cv2.imshow, run until 'q'): any object with read()/isOpened()/release() can stand in for the
    camera, which is how the streaming benchmark feeds synthetic 1080p frames.

    pipeline: "host" preprocesses every frame on the CPU exactly as the reference does; "gpu" uploads the raw frame and
    runs streaming.CameraPipeline (bit-identical preprocessing kernel + CUDA-graph replay of the whole forward);
    "auto" (default) takes the GPU pipeline when the model is on a CUDA device and `transform` is the
    Resize [+ CenterCrop] + ToTensor + Normalize chain that kernel reproduces, the host path otherwise."""
    import cv2
    from PIL import Image
    model.eval()
    cap = capture if capture is not None else cv2.VideoCapture(0)
    if not cap.isOpened():
        print("Error: Unable to open the camera")
        return
    out = None
    if save_video:
        os.makedirs(save_dir, exist_ok=True)
        out = cv2.VideoWriter(os.path.join(save_dir, "camera_output.avi"), cv2.VideoWriter_fourcc(*'XVID'), 20.0,
                              (640, 480))
    times = []
    frames = 0
    gpu_pipe, tried_pipe = None, False
    with torch.no_grad():
        while max_frames is None or frames < max_frames:
            ok, frame = cap.read()
            if not ok:
                print("Error: Unable to read the image from the camera")
                break
            if gpu_pipe is None and pipeline in ("auto", "gpu") and not tried_pipe:
                tried_pipe = True
                on_cuda = torch.device(model.device).type == "cuda"
                if on_cuda:
                    from .streaming import CameraPipeline
                    gpu_pipe = CameraPipeline.from_transform(model, transform, frame.shape)
                if gpu_pipe is None and pipeline == "gpu":
                    raise ValueError("run_camera(pipeline='gpu') needs a CUDA model and a Resize [+ CenterCrop] + "
                                     "ToTensor + Normalize transform")
            start = time.time()
            if gpu_pipe is not None and frame.shape == gpu_pipe.frame_shape:
                probabilities = gpu_pipe(frame)
            else:
                rgb = cv2.cvtColor(frame, cv2.COLOR_BGR2RGB)
                batch = transform(Image.fromarray(rgb)).unsqueeze(0).to(model.device)
                _, outputs = model(batch)
                probabilities = F.softmax(outputs, dim=1).cpu().numpy()[0]   # the .cpu() is the only sync, as upstream
            best = int(np.argmax(probabilities))
            prob = probabilities[best]
            name = class_names[best] if prob >= prob_threshold else "Unknown"
            times.append(time.time() - start)
            frames += 1
            cv2.putText(frame, f"Pred: {name}, Prob: {prob:.4f}", (10, 25), cv2.FONT_HERSHEY_SIMPLEX, 0.7, (0, 255, 0), 2)
            if display:
                cv2.imshow('Camera', frame)
            if out is not None:
                out.write(frame)
            if display and (cv2.waitKey(1) & 0xFF == ord('q')):
                break
    if measure_time:
        os.makedirs(save_dir, exist_ok=True)
        with open(os.path.join(save_dir, "times_camera.json"), "w") as f:
            json.dump(times, f, indent=4)
        print(f"Average processing time per image: {np.mean(times)} seconds")
        print(f"Total processing time: {np.sum(times)} seconds")
    cap.release()
    if out is not None:
        out.release()
    if display:
        cv2.destroyAllWindows()
    return times


def _frame_batch_spec(model, transform, who):
    """The transform as the batched frame kernel reproduces it; ValueError when it cannot (there is no host fallback)."""
    from .streaming import parse_transform
    if torch.device(model.device).type != "cuda":
        raise ValueError(f"{who} needs the model on a CUDA device")
    if parse_transform(transform) is None:
        raise ValueError(f"{who} needs a Resize [+ CenterCrop] + ToTensor + Normalize transform")


def run_cameras(model, transform, class_names, captures, save_video, save_dir, prob_threshold, measure_time,
                display=False, max_frames=None):
    """run_camera for several cameras in one process: each step reads one frame from every capture, classifies them all
    in one forward (streaming.FrameBatchPipeline: one slot per capture, shaped by its first frame) and overlays the label
    on each frame as run_camera does. save_video writes save_dir/camera_<i>_output.avi per stream; measure_time writes
    save_dir/times_cameras.json, the time of each step (all streams). Stops when any capture fails to read, after
    `max_frames` steps, or on 'q' when displaying. Returns the step times.
    Only the GPU path exists: a model off CUDA or a transform the kernel cannot reproduce raises ValueError."""
    captures = list(captures)
    if not captures:
        raise ValueError("run_cameras needs at least one capture")
    if max_frames is not None and max_frames < 0:
        raise ValueError(f"max_frames must be >= 0, got {max_frames}")
    _frame_batch_spec(model, transform, "run_cameras")
    import cv2
    from .streaming import FrameBatchPipeline
    model.eval()
    times = []
    if not all(cap.isOpened() for cap in captures):
        print("Error: Unable to open the cameras")
        for cap in captures:
            cap.release()
        return times
    pipe, writers, steps = None, [], 0
    with torch.no_grad():
        while max_frames is None or steps < max_frames:
            frames = []
            for cap in captures:
                ok, frame = cap.read()
                if not ok:
                    break
                frames.append(frame)
            if len(frames) < len(captures):
                print(f"Error: Unable to read the image from camera {len(frames)}")
                break
            if pipe is None:
                pipe = FrameBatchPipeline.from_transform(model, transform, [f.shape for f in frames])
                if save_video:
                    os.makedirs(save_dir, exist_ok=True)
                    writers = [cv2.VideoWriter(os.path.join(save_dir, f"camera_{i}_output.avi"),
                                               cv2.VideoWriter_fourcc(*'XVID'), 20.0, (f.shape[1], f.shape[0]))
                               for i, f in enumerate(frames)]
            start = time.time()
            probabilities = pipe(frames)
            times.append(time.time() - start)
            steps += 1
            for i, (frame, probs) in enumerate(zip(frames, probabilities)):
                best = int(np.argmax(probs))
                prob = probs[best]
                name = class_names[best] if prob >= prob_threshold else "Unknown"
                cv2.putText(frame, f"Pred: {name}, Prob: {prob:.4f}", (10, 25), cv2.FONT_HERSHEY_SIMPLEX, 0.7,
                            (0, 255, 0), 2)
                if display:
                    cv2.imshow(f'Camera {i}', frame)
                if writers:
                    writers[i].write(frame)
            if display and (cv2.waitKey(1) & 0xFF == ord('q')):
                break
    if measure_time:
        os.makedirs(save_dir, exist_ok=True)
        with open(os.path.join(save_dir, "times_cameras.json"), "w") as f:
            json.dump(times, f, indent=4)
        if times:
            print(f"Average processing time per step ({len(captures)} frames): {np.mean(times)} seconds")
            print(f"Total processing time: {np.sum(times)} seconds")
    for cap in captures:
        cap.release()
    for w in writers:
        w.release()
    if display:
        cv2.destroyAllWindows()
    return times


def classify_video(model, transform, capture, frames_per_call=16, max_frames=None):
    """Classifies the frames of `capture` (anything with read(), e.g. cv2.VideoCapture("file.mp4")) `frames_per_call` at a
    time, in one forward per group (streaming.FrameBatchPipeline; a shorter last group gets a pipeline of its own).
    Reads until the capture ends or `max_frames` frames. Returns (predictions int64 (F,), probabilities float32 (F,)):
    the arg-max class of each frame and its softmax probability, in frame order. The capture is not released.
    Only the GPU path exists: a model off CUDA or a transform the kernel cannot reproduce raises ValueError."""
    if isinstance(frames_per_call, bool) or not isinstance(frames_per_call, int) or frames_per_call < 1:
        raise ValueError(f"frames_per_call must be a positive integer, got {frames_per_call!r}")
    if max_frames is not None and max_frames < 0:
        raise ValueError(f"max_frames must be >= 0, got {max_frames}")
    _frame_batch_spec(model, transform, "classify_video")
    from .streaming import FrameBatchPipeline
    model.eval()
    pipes, preds, probs, count = {}, [], [], 0
    while max_frames is None or count < max_frames:
        group = []
        while len(group) < frames_per_call and (max_frames is None or count + len(group) < max_frames):
            ok, frame = capture.read()
            if not ok:
                break
            group.append(frame)
        if not group:
            break
        n = len(group)
        if n not in pipes:
            pipes[n] = FrameBatchPipeline.from_transform(model, transform, [group[0].shape] * n)
        p = pipes[n](group)
        best = p.argmax(axis=1)
        preds.append(best.astype(np.int64))
        probs.append(p[np.arange(n), best].astype(np.float32))
        count += n
        if n < frames_per_call:
            break
    if not preds:
        return np.zeros(0, np.int64), np.zeros(0, np.float32)
    return np.concatenate(preds), np.concatenate(probs)
