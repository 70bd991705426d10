"""Worker side of baseline JPEG decoding on the GPU (functions.gpu_resize_transform(decode="gpu"), csrc/jpeg.cuh).

`parse(data)` classifies a file and, for one the device decodes (SOF0 / SOF1, 8-bit, Huffman, one scan with every
component, 1 component or 3 that libjpeg treats as YCbCr, luma sampling (1,1), (2,1), (1,2) or (2,2) with chroma
(1,1)), returns its header, its unstuffed restart segments and its tables in the layout of include/gramhead.h. Every
other file gets None and is decoded by Pillow in the worker. `pack(...)` lays a batch of parsed files out for
gh_jpeg_decode, and `decode_batch(...)` runs it on the current stream."""
from __future__ import annotations

import functools

import numpy as np
import torch

from . import _lib
from ._lib import GramHeadError, check

# include/gramhead.h
SEG_COLS = 5                    # start, len, image, first MCU, MCUs
IMG_COLS = 13                   # H, W, ncomp, h0, v0, mcux, mcuy, coef_off, blocks, plane_off, arena_off, table_off, batch
QUANT_INTS, HUFF_MAXCODE, HUFF_VALOFF, HUFF_VALS, HUFF_INTS = 192, 512, 530, 547, 612
TABLE_INTS = QUANT_INTS + 6 * HUFF_INTS
LOOKAHEAD = 9
MAX_SEGMENT_BYTES = 1 << 28        # GH_JPEG_MAX_SEGMENT_BYTES: bit positions inside a segment are 32-bit
SUBSEQ_BYTES = 16384            # subsequence of the parallel Huffman decoder (profiles/r12_loader_decode_timing.log)

_ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,
                    7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38,
                    31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63], dtype=np.int64)


class JpegFile:
    """A file the device decodes: its bytes, size, layout, restart segments and tables. `path` is set by the loader;
    batches then carry the path instead of the bytes, for CPU runs, which decode the file with Pillow."""

    def __init__(self, data, H, W, comps, dri, segments, tables, path=None):
        self.data, self.H, self.W, self.comps, self.dri = data, H, W, comps, dri
        self.segments, self.tables, self.path = segments, tables, path
        self.shape = (H, W, 3)

    @property
    def layout(self):
        """(ncomp, h0, v0, mcux, mcuy, blocks, plane bytes) of the coefficient and sample planes."""
        nc, (_, h0, v0, _) = len(self.comps), self.comps[0]
        if nc == 1:
            hmax, vmax = h0, v0
            mx, my = -(-(-(-self.W * h0 // hmax)) // 8), -(-(-(-self.H * v0 // vmax)) // 8)
            return 1, 1, 1, mx, my, mx * my, mx * my * 64
        mx, my = -(-self.W // (8 * h0)), -(-self.H // (8 * v0))
        return 3, h0, v0, mx, my, mx * my * (h0 * v0 + 2), mx * my * 64 * (h0 * v0 + 2)


@functools.lru_cache(maxsize=256)
def _huff_table(bits, vals):
    """jpeg_make_d_derived_tbl (jdhuff.c) in the device layout: 9-bit lookahead, maxcode / valoff per length, symbols.
    Raises ValueError where libjpeg raises JERR_BAD_HUFF_TABLE. Cached: most files carry the same few tables."""
    t = np.zeros(HUFF_INTS, np.int64)
    t[HUFF_MAXCODE:HUFF_MAXCODE + 18] = -1
    code, k = 0, 0
    for length in range(1, 17):
        n = bits[length - 1]
        if n:
            t[HUFF_VALOFF + length] = k - code
            if length <= LOOKAHEAD:
                for c in range(code, code + n):
                    lo = c << (LOOKAHEAD - length)
                    t[lo:lo + (1 << (LOOKAHEAD - length))] = (length << 8) | vals[k + c - code]
            code += n
            k += n
            t[HUFF_MAXCODE + length] = code - 1
        if code >= (1 << length):                       # an all-ones code word: JERR_BAD_HUFF_TABLE
            raise ValueError("bad Huffman table")
        code <<= 1
    v = np.zeros(256, np.int64)
    v[:len(vals)] = vals
    t[HUFF_VALS:HUFF_VALS + 64] = (v.reshape(64, 4) << np.array([0, 8, 16, 24])).sum(1).astype(np.uint32).view(np.int32)
    return t


def _unstuff(a):
    """Entropy-coded bytes after SOS -> (bytes without stuffing, fill or RST markers, [segment start offsets]); the scan
    ends at the first other marker (jdhuff.c jpeg_fill_bit_buffer). Only the runs of 0xFF need work, so apart from
    finding them and one copy, nothing here is as long as the scan."""
    n = len(a)
    ff = np.flatnonzero(a == 0xFF)
    if ff.size == 0:
        return a, [0]
    brk = np.flatnonzero(np.diff(ff) != 1)
    starts, ends = ff[np.r_[0, brk + 1]], ff[np.r_[brk, ff.size - 1]]
    nxt = np.where(ends + 1 < n, a[np.minimum(ends + 1, n - 1)].astype(np.int64), -1)
    stuffed, rst = nxt == 0, (nxt >= 0xD0) & (nxt <= 0xD7)
    term = ~(stuffed | rst)
    end = n
    if term.any():
        k = int(np.argmax(term))
        end, starts, ends, stuffed, rst = int(starts[k]), starts[:k], ends[:k], stuffed[:k], rst[:k]
    # dropped per run: its fill bytes (every 0xFF but the last), then the 00 after a stuffed 0xFF or the whole RSTn
    fill = ends - starts
    first = np.repeat(np.cumsum(fill) - fill, fill)
    drop = np.concatenate([np.repeat(starts, fill) + np.arange(first.size) - first, ends[stuffed] + 1, ends[rst],
                           ends[rst] + 1])
    # a segment starts after its RSTn, at the run's first byte less the bytes earlier runs dropped
    dropped = fill + stuffed + 2 * rst
    before = np.cumsum(dropped) - dropped
    return np.delete(a[:end], drop), [0] + (starts[rst] - before[rst]).tolist()


def parse(data: bytes):
    """A JpegFile for a file the device decodes, None for every other file (Pillow decodes it in the worker)."""
    try:
        return _parse(data)
    except (ValueError, IndexError, KeyError):
        return None


def _parse(data: bytes):
    if data[:2] != b"\xff\xd8":
        return None
    pos, n = 2, len(data)
    q, huff, dri, frame, jfif, adobe = {}, {}, 0, None, False, None
    while True:
        while pos < n and data[pos] != 0xFF:
            pos += 1
        while pos < n and data[pos] == 0xFF:
            pos += 1
        if pos >= n:
            return None
        m = data[pos]
        pos += 1
        if m == 0xD8 or 0xD0 <= m <= 0xD7 or m == 0x01:
            continue
        seg_len = int.from_bytes(data[pos:pos + 2], "big")
        if seg_len < 2 or pos + seg_len > n:
            return None
        body = data[pos + 2:pos + seg_len]
        pos += seg_len
        if m == 0xDB:
            i = 0
            while i < len(body):
                if body[i] >> 4:
                    return None                          # 16-bit tables: not baseline 8-bit
                t = np.zeros(64, np.int64)
                t[_ZIGZAG] = np.frombuffer(body[i + 1:i + 65], np.uint8)
                q[body[i] & 15] = t
                i += 65
        elif m == 0xC4:
            i = 0
            while i < len(body):
                bits = list(body[i + 1:i + 17])
                huff[(body[i] >> 4, body[i] & 15)] = (bits, list(body[i + 17:i + 17 + sum(bits)]))
                i += 17 + sum(bits)
        elif m == 0xDD:
            dri = int.from_bytes(body[:2], "big")
        elif m == 0xE0 and body[:5] == b"JFIF\0":
            jfif = True
        elif m == 0xEE and body[:5] == b"Adobe" and len(body) >= 12:
            adobe = body[11]
        elif m in (0xC0, 0xC1):
            if frame is not None or body[0] != 8:
                return None
            H, W, nc = int.from_bytes(body[1:3], "big"), int.from_bytes(body[3:5], "big"), body[5]
            frame = (H, W, [(body[6 + 3 * k], body[7 + 3 * k] >> 4, body[7 + 3 * k] & 15, body[8 + 3 * k])
                            for k in range(nc)])
        elif 0xC2 <= m <= 0xCF and m not in (0xC4, 0xC8, 0xCC):
            return None                                  # progressive, lossless, arithmetic, hierarchical
        elif m == 0xDA:
            if frame is None:
                return None
            scan = [(body[1 + 2 * k], body[2 + 2 * k] >> 4, body[2 + 2 * k] & 15) for k in range(body[0])]
            if bytes(body[1 + 2 * body[0]:4 + 2 * body[0]]) != b"\x00\x3f\x00":
                return None
            break
    H, W, comps = frame
    if H == 0 or W == 0 or len(comps) not in (1, 3) or [c[0] for c in comps] != [s[0] for s in scan]:
        return None
    if len(comps) == 3:
        ids = tuple(c[0] for c in comps)
        # default_decompress_parms (jdapimin.c): the cases it treats as YCbCr without a warning
        if not (jfif or adobe == 1 or (adobe is None and ids == (1, 2, 3))):
            return None
        if (comps[0][1], comps[0][2]) not in ((1, 1), (2, 1), (1, 2), (2, 2)) or \
                any((c[1], c[2]) != (1, 1) for c in comps[1:]):
            return None
    elif not (1 <= comps[0][1] <= 4 and 1 <= comps[0][2] <= 4):
        return None
    tables = np.zeros(TABLE_INTS, np.int64)
    for k, ((_, _, _, tq), (_, td, ta)) in enumerate(zip(comps, scan)):
        tables[k * 64:(k + 1) * 64] = q[tq]
        for j, key in enumerate(((0, td), (1, ta))):
            o = QUANT_INTS + (2 * k + j) * HUFF_INTS
            tables[o:o + HUFF_INTS] = _huff_table(*(tuple(v) for v in huff[key]))
    scan_bytes, starts = _unstuff(np.frombuffer(data, np.uint8, offset=pos))
    f = JpegFile(data, H, W, comps, dri, None, tables.astype(np.int32))
    _, _, _, mx, my, _, _ = f.layout
    n_mcu = mx * my
    n_seg = -(-n_mcu // dri) if dri else 1
    bounds = starts + [len(scan_bytes)]
    segs = [scan_bytes[bounds[i]:bounds[i + 1]] if i + 1 < len(bounds) else scan_bytes[:0] for i in range(n_seg)]
    if any(len(sg) >= MAX_SEGMENT_BYTES for sg in segs):
        return None                                      # Pillow decodes it in the worker
    f.segments = segs
    return f


def pack(files, arena_offsets, batch_index):
    """Lays out parsed files for gh_jpeg_decode: (scan uint8, segs (S, 5) int64, imgs (n, 13) int64, tables int32),
    each a CPU tensor. arena_offsets: each file's byte offset in the pixel arena; batch_index: its row in the batch."""
    seg_rows, img_rows, parts = [], [], []
    pos = coef = plane = 0
    for i, f in enumerate(files):
        nc, h0, v0, mx, my, blocks, plane_bytes = f.layout
        per = f.dri or mx * my
        for s, seg in enumerate(f.segments):
            seg_rows.append((pos, len(seg), i, s * per, per))
            parts.append(seg)
            pos += len(seg)
        img_rows.append((f.H, f.W, nc, h0, v0, mx, my, coef, blocks, plane, int(arena_offsets[i]), i * TABLE_INTS,
                         int(batch_index[i])))
        coef += blocks
        plane += plane_bytes
    scan = np.concatenate(parts) if parts else np.zeros(0, np.uint8)
    if scan.size == 0:
        scan = np.zeros(1, np.uint8)                     # every segment empty: a valid pointer for the kernels
    return (torch.from_numpy(np.ascontiguousarray(scan)), torch.tensor(seg_rows, dtype=torch.int64),
            torch.tensor(img_rows, dtype=torch.int64),
            torch.from_numpy(np.concatenate([f.tables for f in files])))


def workspace(imgs_host: np.ndarray, scan_bytes: int, n_segs: int, subseq: int = SUBSEQ_BYTES):
    """(coefficient int16s, plane bytes, record bytes) gh_jpeg_decode needs for a packed batch."""
    last = imgs_host[-1]
    nc, h0, v0, mx, my = (int(v) for v in last[2:7])
    plane_bytes = mx * my * 64 * (1 if nc == 1 else h0 * v0 + 2)
    rec = int(_lib.lib().gh_jpeg_records_bytes(scan_bytes, n_segs, subseq))
    check(min(rec, 0), "gh_jpeg_records_bytes")
    return int(last[7] + last[8]) * 64, int(last[9]) + plane_bytes, rec


def validate(scan_bytes: int, segs: np.ndarray, imgs: np.ndarray, arena_bytes: int):
    """Every range the kernels read or write, checked on the host before a launch."""
    if segs.ndim != 2 or segs.shape[1] != SEG_COLS or imgs.ndim != 2 or imgs.shape[1] != IMG_COLS or not len(imgs):
        raise GramHeadError("gramhead: jpeg: malformed descriptors")
    st, ln, im, mcu, per = segs.T
    H, W, nc, h0, v0, mx, my, co, bl, po, ao, to, _ = imgs.T
    if ((st < 0) | (ln < 0) | (ln >= MAX_SEGMENT_BYTES) | (st + ln > scan_bytes) | (im < 0) | (im >= len(imgs)) | (mcu < 0) | (per <= 0)).any():
        raise GramHeadError("gramhead: jpeg: a segment lies outside the scan data")
    if ((H <= 0) | (W <= 0) | (ao < 0) | (ao + H * W * 3 > arena_bytes) | (bl <= 0) | (co < 0) | (po < 0)).any():
        raise GramHeadError("gramhead: jpeg: an image lies outside the pixel arena")
    if (~np.isin(nc, (1, 3)) | (mx * 8 * np.where(nc == 1, 1, h0) < W) | (my * 8 * np.where(nc == 1, 1, v0) < H)).any():
        raise GramHeadError("gramhead: jpeg: an image's layout does not cover its size")


def decode_batch(scan, segs, imgs, tables, imgs_host, segs_host, arena, arena_bytes, coef=None, planes=None,
                 records=None, status=None, subseq=SUBSEQ_BYTES, phases=7):
    """Runs gh_jpeg_decode on the current stream: the images of `imgs` into `arena`. Buffers left None are allocated.
    Returns the int32 status tensor (nonzero for an image whose scan is broken)."""
    lib = _lib.lib()
    validate(scan.numel(), segs_host, imgs_host, arena_bytes)
    n_coef, n_plane, n_rec = workspace(imgs_host, scan.numel(), len(segs_host), subseq)
    dev = arena.device
    coef = torch.empty(n_coef, dtype=torch.int16, device=dev) if coef is None else coef[:n_coef]
    planes = torch.empty(n_plane, dtype=torch.uint8, device=dev) if planes is None else planes
    records = torch.empty(n_rec // 4, dtype=torch.int32, device=dev) if records is None else records
    status = torch.empty(len(imgs_host), dtype=torch.int32, device=dev) if status is None else status
    if (coef.numel() < n_coef or planes.numel() < n_plane or records.numel() * 4 < n_rec
            or status.numel() < len(imgs_host)):
        raise GramHeadError("gramhead: jpeg: workspace buffers are too small")
    if phases & 1:
        coef.zero_()
    H, W, bl = imgs_host[:, 0], imgs_host[:, 1], imgs_host[:, 8]
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        check(lib.gh_jpeg_decode(scan.data_ptr(), scan.numel(), segs.data_ptr(), len(segs_host), imgs.data_ptr(),
                                 len(imgs_host), tables.data_ptr(), int(bl.max()), int((H * W).max()), subseq,
                                 coef.data_ptr(), planes.data_ptr(), records.data_ptr(), status.data_ptr(),
                                 arena.data_ptr(), phases, stream), "gh_jpeg_decode")
    return status
