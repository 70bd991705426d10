"""The seeded JPEG corpus of the decoder tests, generated at test time (no data files).

`corpus()` writes files with Pillow: the sizes, qualities, subsamplings, grayscale, optimised Huffman tables, restart
intervals and custom quantisation tables Pillow can write, over noise, flat colour, gradients, resized noise (the content
tools/time_loader_resize.py writes) and saturated black / white noise. `write()` is a minimal baseline writer of given
quantised coefficients, for what Pillow's encoder cannot write: luma sampling (1, 2), coefficients whose IDCT leaves
the 16-bit range of libjpeg-turbo's SIMD arithmetic, files without a JFIF marker and chosen component ids. Its Huffman
tables are the ones Pillow writes by default (the example tables of ITU-T T.81 Annex K), taken from a file it writes,
so no table is typed in here."""
from __future__ import annotations

import io

import numpy as np
from PIL import Image

from oracle import jpeg_decode as J


def standard_tables():
    b = io.BytesIO()
    Image.new("RGB", (8, 8)).save(b, "JPEG", quality=75)
    return J.parse(b.getvalue())["huff"]


def _codes(bits, vals):
    table, code, k = {}, 0, 0
    for length in range(1, 17):
        for _ in range(bits[length - 1]):
            table[vals[k]] = (code, length)
            code += 1
            k += 1
        code <<= 1
    return table


def _category(v):
    a = abs(int(v))
    s = a.bit_length()
    return s, (v if v >= 0 else v + (1 << s) - 1)


class _Bits:
    def __init__(self):
        self.out, self.acc, self.n = bytearray(), 0, 0

    def put(self, code, length):
        self.acc, self.n = (self.acc << length) | code, self.n + length
        while self.n >= 8:
            byte = (self.acc >> (self.n - 8)) & 0xFF
            self.out.append(byte)
            if byte == 0xFF:
                self.out.append(0)
            self.n -= 8
        self.acc &= (1 << self.n) - 1

    def flush(self):
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)


def write(coef, comps, qtables, H, W, dri=0, jfif=True, adobe=None, sof=0xC0):
    """coef: per component (bh, bw, 64) int quantised coefficients in natural order, laid out as
    oracle.jpeg_decode.layout gives; comps: [(id, h, v, tq)]; qtables: {tq: (64,) natural order}."""
    huff = standard_tables()
    dc = [_codes(*huff[(0, 0 if k == 0 else 1)]) for k in range(len(comps))]
    ac = [_codes(*huff[(1, 0 if k == 0 else 1)]) for k in range(len(comps))]
    seg = bytearray(b"\xff\xd8")

    def marker(m, body):
        seg.extend(bytes([0xFF, m]) + (len(body) + 2).to_bytes(2, "big") + body)

    if jfif:
        marker(0xE0, b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    if adobe is not None:
        marker(0xEE, b"Adobe\x00\x64\x00\x00\x00\x00" + bytes([adobe]))
    for tq, t in qtables.items():
        marker(0xDB, bytes([tq]) + bytes(int(v) for v in np.asarray(t)[J.ZIGZAG]))
    marker(sof, bytes([8]) + H.to_bytes(2, "big") + W.to_bytes(2, "big") + bytes([len(comps)]) +
           b"".join(bytes([c, (h << 4) | v, tq]) for c, h, v, tq in comps))
    for (tc, th), (bits, vals) in sorted(huff.items()):
        marker(0xC4, bytes([(tc << 4) | th]) + bytes(bits) + bytes(vals))
    if dri:
        marker(0xDD, dri.to_bytes(2, "big"))
    marker(0xDA, bytes([len(comps)]) + b"".join(bytes([c[0], (0 if k == 0 else 0x11)]) for k, c in enumerate(comps))
           + b"\x00\x3f\x00")
    planes, mx, my, order = J.layout(H, W, comps)
    n_mcu = mx * my
    bits, pred, rst = _Bits(), [0] * len(comps), 0
    for mcu in range(n_mcu):
        if dri and mcu and mcu % dri == 0:
            bits.flush()
            seg.extend(bits.out)
            seg.extend(bytes([0xFF, 0xD0 + rst % 8]))
            bits, pred, rst = _Bits(), [0] * len(comps), rst + 1
        my_, mx_ = divmod(mcu, mx)
        for ci, by, bx in order:
            blk = coef[ci][my_ * comps[ci][2] + by, mx_ * comps[ci][1] + bx] if len(comps) > 1 else coef[0][my_, mx_]
            z = np.asarray(blk)[J.ZIGZAG]
            s, v = _category(z[0] - pred[ci])
            pred[ci] = int(z[0])
            bits.put(*dc[ci][s])
            if s:
                bits.put(v, s)
            run = 0
            for k in range(1, 64):
                if z[k] == 0:
                    run += 1
                    continue
                while run > 15:
                    bits.put(*ac[ci][0xF0])
                    run -= 16
                s, v = _category(z[k])
                bits.put(*ac[ci][(run << 4) | s])
                bits.put(v, s)
                run = 0
            if run:
                bits.put(*ac[ci][0x00])
    bits.flush()
    seg.extend(bits.out)
    seg.extend(b"\xff\xd9")
    return bytes(seg)


def random_coefficients(rng, H, W, comps, amp=30, extreme=False):
    """Per component (bh, bw, 64) coefficients: a random DC walk and decaying AC terms; extreme=True puts the largest
    baseline magnitudes (DC +-1023 after prediction limits, AC +-1023) with one sign per block, so that with a coarse
    quantisation table the IDCT output leaves -512..511 and wraps the range-limit table."""
    planes, _, _, _ = J.layout(H, W, comps)
    out = []
    for bw, bh in planes:
        c = np.zeros((bh, bw, 64), np.int64)
        decay = np.maximum(1, amp // (1 + np.arange(64) // 4))
        c[..., :] = rng.integers(-1, 2, (bh, bw, 64)) * rng.integers(0, decay + 1, (bh, bw, 64))
        c[..., 0] = rng.integers(-60, 61, (bh, bw))
        if extreme:
            sign = rng.choice([-1, 1], (bh, bw, 1))
            c[..., :] = sign * rng.integers(0, 40, (bh, bw, 64))
            c[..., 0] = sign[..., 0] * rng.integers(60, 128, (bh, bw))
        out.append(c)
    return out


SMALL = [(1, 1), (7, 9), (8, 8), (15, 17), (16, 16), (31, 33)]
LARGE = [(300, 2000), (2000, 300), (1999, 2001)]
QUALITIES = [1, 50, 75, 90, 95, 100]
SUBSAMPLING = {0: "444", 1: "422", 2: "420"}


def content(kind, h, w, rng):
    if kind == "noise":
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "flat":
        return np.broadcast_to(rng.integers(0, 256, 3, dtype=np.uint8), (h, w, 3)).copy()
    if kind == "gradient":
        y, x = np.mgrid[0:h, 0:w]
        return np.stack([x * 255 // max(w - 1, 1), y * 255 // max(h - 1, 1), (x + y) * 255 // max(h + w - 2, 1)],
                        -1).astype(np.uint8)
    if kind == "resized":
        base = Image.fromarray(rng.integers(0, 256, (12, 12, 3), dtype=np.uint8), "RGB").resize((w, h), Image.BILINEAR)
        px = np.asarray(base, dtype=np.int16) + rng.integers(-20, 21, (h, w, 3), dtype=np.int16)
        return np.clip(px, 0, 255).astype(np.uint8)
    if kind == "extremes":
        return (rng.integers(0, 2, (h, w, 3)) * 255).astype(np.uint8)
    raise ValueError(kind)


KINDS = ["noise", "flat", "gradient", "resized", "extremes"]


def _save(arr, mode="RGB", **kw):
    b = io.BytesIO()
    Image.fromarray(arr, "RGB").convert(mode).save(b, "JPEG", **kw)
    return b.getvalue()


def corpus(seed=0, large=True):
    """[(name, bytes)] of the seeded corpus; large=False leaves out the three large sizes."""
    rng = np.random.default_rng(seed)
    out = []
    for (h, w) in SMALL:
        for qi, q in enumerate(QUALITIES):
            for ss, sname in SUBSAMPLING.items():
                kind = KINDS[(qi + ss) % len(KINDS)]
                out.append((f"{h}x{w}_q{q}_{sname}_{kind}", _save(content(kind, h, w, rng), quality=q, subsampling=ss)))
            kind = KINDS[qi % len(KINDS)]
            out.append((f"{h}x{w}_q{q}_L_{kind}", _save(content(kind, h, w, rng), "L", quality=q)))
    mid = content("resized", 61, 83, rng)
    for ss, sname in SUBSAMPLING.items():
        out.append((f"optimize_{sname}", _save(mid, quality=85, subsampling=ss, optimize=True)))
        out.append((f"restart_blocks_{sname}", _save(mid, quality=90, subsampling=ss, restart_marker_blocks=3)))
        out.append((f"restart_rows_{sname}", _save(mid, quality=90, subsampling=ss, restart_marker_rows=1)))
        out.append((f"qtables_{sname}", _save(mid, subsampling=ss, qtables=[list(range(1, 65)), [255] * 64])))
        out.append((f"extremes_q1_{sname}", _save(content("extremes", 40, 48, rng), quality=1, subsampling=ss)))
    out.append(("restart_blocks_L", _save(mid, "L", quality=90, restart_marker_blocks=1)))
    out.append(("optimize_L", _save(mid, "L", quality=90, optimize=True)))
    for (h, w), comps in (((23, 37), [(1, 1, 2, 0), (2, 1, 1, 1), (3, 1, 1, 1)]),
                          ((40, 50), [(1, 1, 2, 0), (2, 1, 1, 1), (3, 1, 1, 1)]),
                          ((9, 2), [(1, 1, 2, 0), (2, 1, 1, 1), (3, 1, 1, 1)])):
        for dri in (0, 2):
            coef = random_coefficients(rng, h, w, comps)
            out.append((f"written_h1v2_{h}x{w}_dri{dri}",
                        write(coef, comps, {0: np.arange(1, 65), 1: np.full(64, 3)}, h, w, dri=dri)))
    for qv in (8, 48, 255):
        comps = [(1, 2, 2, 0), (2, 1, 1, 1), (3, 1, 1, 1)]
        coef = random_coefficients(rng, 24, 40, comps, extreme=True)
        out.append((f"written_extreme_q{qv}", write(coef, comps, {0: np.full(64, qv), 1: np.full(64, qv)}, 24, 40)))
    comps = [(1, 2, 1, 0), (2, 1, 1, 1), (3, 1, 1, 1)]
    coef = random_coefficients(rng, 20, 30, comps)
    qt = {0: np.full(64, 4), 1: np.full(64, 6)}
    out.append(("written_ids123_nojfif", write(coef, comps, qt, 20, 30, jfif=False)))
    out.append(("written_adobe1", write(coef, [(7, 2, 1, 0), (8, 1, 1, 1), (9, 1, 1, 1)], qt, 20, 30, jfif=False,
                                        adobe=1)))
    out.append(("written_sof1", write(coef, comps, qt, 20, 30, sof=0xC1)))
    if large:
        for (h, w), kind, q, ss in zip(LARGE, ["resized", "gradient", "resized"], [75, 95, 90], [2, 0, 1]):
            out.append((f"{h}x{w}_q{q}_{SUBSAMPLING[ss]}_{kind}", _save(content(kind, h, w, rng), quality=q,
                                                                          subsampling=ss)))
    return out


def pillow(data):
    """What the reference's loaders see: default_loader's `Image.open(f).convert('RGB')`."""
    return np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))
