"""numpy restatement of baseline JPEG decoding as Pillow does it  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

What it restates: torchvision.datasets.folder.default_loader, i.e. `Image.open(f).convert('RGB')`. Pillow (12.2 here)
decodes through libjpeg-turbo (3.1 here) with the library defaults: JDCT_ISLOW, fancy upsampling, no draft scaling.
Each function names the libjpeg-turbo routine it restates. Only what the device decoder supports is restated: SOF0 /
SOF1, 8-bit, Huffman, one interleaved scan with every component, 1 component or 3 YCbCr ones, luma sampling (1,1),
(2,1), (1,2) or (2,2) with chroma (1,1), any restart interval.

Pinning: tests/test_jpeg_oracle.py checks this restatement for exact equality against Pillow on a seeded corpus.
Where a detail below differs from the C source of libjpeg-turbo, it is what Pillow's build computes: the x86 SIMD
routines libjpeg-turbo runs there are the reference.
"""
from __future__ import annotations

import numpy as np

# jpeg_natural_order (jutils.c): zig-zag index -> natural (row-major) index
ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,
                   7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31,
                   39, 46, 53, 60, 61, 54, 47, 55, 62, 63], dtype=np.int64)


class Unsupported(ValueError):
    """The file is not one the restatement (and the device decoder) covers."""


def parse(data: bytes) -> dict:
    """Marker walk of jdmarker.c (read_markers): SOI, DQT (get_dqt), DHT (get_dht), DRI (get_dri), SOF0/1 (get_sof),
    SOS (get_sos), APP0 JFIF / APP14 Adobe (examine_app0 / examine_app14). Returns the frame, tables and the byte range
    of the entropy-coded data of the (single) scan. Raises Unsupported for anything else."""
    if data[:2] != b"\xff\xd8":
        raise Unsupported("no SOI")
    pos, n = 2, len(data)
    q, huff, dri, frame, jfif, adobe = {}, {}, 0, None, False, None
    while True:
        while pos < n and data[pos] != 0xFF:
            pos += 1
        while pos < n and data[pos] == 0xFF:
            pos += 1
        if pos >= n:
            raise Unsupported("no SOS")
        m = data[pos]
        pos += 1
        if m == 0xD8 or 0xD0 <= m <= 0xD7 or m == 0x01:
            continue
        seg_len = int.from_bytes(data[pos:pos + 2], "big")
        body = data[pos + 2:pos + seg_len]
        pos += seg_len
        if m == 0xDB:
            i = 0
            while i < len(body):
                pq, tq = body[i] >> 4, body[i] & 15
                if pq:
                    raise Unsupported("16-bit quantisation table")
                t = np.zeros(64, np.int64)
                t[ZIGZAG] = np.frombuffer(body[i + 1:i + 65], np.uint8)
                q[tq] = t
                i += 65
        elif m == 0xC4:
            i = 0
            while i < len(body):
                tc, th = body[i] >> 4, body[i] & 15
                bits = list(body[i + 1:i + 17])
                cnt = sum(bits)
                huff[(tc, th)] = (bits, list(body[i + 17:i + 17 + cnt]))
                i += 17 + cnt
        elif m == 0xDD:
            dri = int.from_bytes(body[:2], "big")
        elif m == 0xE0 and body[:5] == b"JFIF\0":
            jfif = True
        elif m == 0xEE and body[:5] == b"Adobe" and len(body) >= 12:
            adobe = body[11]
        elif m in (0xC0, 0xC1):
            if body[0] != 8:
                raise Unsupported("precision")
            H, W, nc = int.from_bytes(body[1:3], "big"), int.from_bytes(body[3:5], "big"), body[5]
            comps = [(body[6 + 3 * k], body[7 + 3 * k] >> 4, body[7 + 3 * k] & 15, body[8 + 3 * k]) for k in range(nc)]
            frame = (H, W, comps)
        elif 0xC2 <= m <= 0xCF and m not in (0xC4, 0xC8, 0xCC):
            raise Unsupported(f"SOF{m - 0xC0}")
        elif m == 0xDA:
            if frame is None:
                raise Unsupported("SOS before SOF")
            ns = body[0]
            scan = [(body[1 + 2 * k], body[2 + 2 * k] >> 4, body[2 + 2 * k] & 15) for k in range(ns)]
            break
    H, W, comps = frame
    if len(comps) not in (1, 3) or [c[0] for c in comps] != [s[0] for s in scan]:
        raise Unsupported("components")
    if len(comps) == 3:
        ids = tuple(c[0] for c in comps)
        # default_decompress_parms (jdapimin.c), restricted to the cases it treats as YCbCr without a warning
        if not (jfif or (adobe == 1) or (adobe is None and ids == (1, 2, 3))):
            raise Unsupported("colour space")
        if (comps[0][1], comps[0][2]) not in ((1, 1), (2, 1), (1, 2), (2, 2)) or any((c[1], c[2]) != (1, 1) for c in comps[1:]):
            raise Unsupported("sampling")
    return dict(H=H, W=W, comps=comps, scan=scan, q=q, huff=huff, dri=dri, scan_start=pos)


def segments(data: bytes, start: int) -> list:
    """The entropy-coded data after SOS, split at RSTn markers, with byte stuffing (FF 00 -> FF) removed; it ends at the
    first other marker (jdhuff.c jpeg_fill_bit_buffer stops there)."""
    out, cur, i, n = [], bytearray(), start, len(data)
    while i < n:
        b = data[i]
        if b != 0xFF:
            cur.append(b)
            i += 1
            continue
        j = i + 1
        while j < n and data[j] == 0xFF:
            j += 1
        if j >= n:
            break
        if data[j] == 0:
            cur.append(0xFF)
            i = j + 1
        elif 0xD0 <= data[j] <= 0xD7:
            out.append(bytes(cur))
            cur = bytearray()
            i = j + 1
        else:
            break
    out.append(bytes(cur))
    return out


def huff_lookup(bits, vals):
    """jdhuff.c jpeg_make_d_derived_tbl, as a 16-bit lookahead: code word left-aligned in 16 bits -> (length, symbol);
    length 0 marks a bit pattern that starts no code."""
    lut_len = np.zeros(1 << 16, np.int64)
    lut_sym = np.zeros(1 << 16, np.int64)
    code, k = 0, 0
    for length in range(1, 17):
        for _ in range(bits[length - 1]):
            lo = code << (16 - length)
            lut_len[lo:lo + (1 << (16 - length))] = length
            lut_sym[lo:lo + (1 << (16 - length))] = vals[k]
            code += 1
            k += 1
        code <<= 1
    return lut_len.tolist(), lut_sym.tolist()


def _extend(v, s):
    """HUFF_EXTEND (jdhuff.h)."""
    return v - (1 << s) + 1 if v < (1 << (s - 1)) else v


def layout(H, W, comps):
    """Per component (blocks wide, blocks high) of its coefficient plane and the order of blocks in the scan: for an
    interleaved scan, MCUs of hmax*8 x vmax*8 pixels, each holding h*v blocks of the luma then one of each chroma plane;
    for one component, its blocks in raster order (jdinput.c per_scan_setup)."""
    hmax, vmax = max(c[1] for c in comps), max(c[2] for c in comps)
    if len(comps) == 1:
        bw, bh = -(-(-(-W * comps[0][1] // hmax)) // 8), -(-(-(-H * comps[0][2] // vmax)) // 8)
        return [(bw, bh)], bw, bh, [(0, 0, 0)]
    mx, my = -(-W // (8 * hmax)), -(-H // (8 * vmax))
    planes = [(mx * c[1], my * c[2]) for c in comps]
    order = [(ci, by, bx) for ci, c in enumerate(comps) for by in range(c[2]) for bx in range(c[1])]
    return planes, mx, my, order


def decode_coefficients(data: bytes, hdr: dict) -> list:
    """jdhuff.c decode_mcu: Huffman decoding of every block, DC prediction per component reset at each restart
    (process_restart). Returns per component the quantised coefficients, shape (bh, bw, 64), natural order."""
    comps, scan = hdr["comps"], hdr["scan"]
    planes, mx, my, order = layout(hdr["H"], hdr["W"], comps)
    coef = [np.zeros((bh, bw, 64), np.int64) for bw, bh in planes]
    luts = [(huff_lookup(*hdr["huff"][(0, td)]), huff_lookup(*hdr["huff"][(1, ta)])) for _, td, ta in scan]
    segs = segments(data, hdr["scan_start"])
    n_mcu = mx * my
    per_seg = hdr["dri"] or n_mcu
    mcu = 0
    for seg in segs:
        if mcu >= n_mcu:
            break
        buf = seg + b"\xff" * 8                     # bits past the segment end read as 1s, like a marker's fill
        nbits = len(seg) * 8
        p = 0
        pred = [0] * len(comps)

        def get(nb):
            nonlocal p
            if nb == 0:
                return 0
            v = (int.from_bytes(buf[p >> 3:(p >> 3) + 4], "big") >> (32 - nb - (p & 7))) & ((1 << nb) - 1)
            p += nb
            return v

        def symbol(lut):
            nonlocal p
            peek = (int.from_bytes(buf[p >> 3:(p >> 3) + 4], "big") >> (16 - (p & 7))) & 0xFFFF
            ln = lut[0][peek]
            if ln == 0:
                raise ValueError("invalid Huffman code")
            p += ln
            return lut[1][peek]

        for _ in range(min(per_seg, n_mcu - mcu)):
            my_, mx_ = divmod(mcu, mx)
            for ci, by, bx in order:
                dc_lut, ac_lut = luts[ci]
                blk = coef[ci][my_ * comps[ci][2] + by, mx_ * comps[ci][1] + bx] if len(comps) > 1 else \
                    coef[0][divmod(mcu, mx)]
                s = symbol(dc_lut)
                pred[ci] += _extend(get(s), s) if s else 0
                blk[0] = pred[ci]
                k = 1
                while k < 64:
                    rs = symbol(ac_lut)
                    r, s = rs >> 4, rs & 15
                    if s == 0:
                        if r != 15:
                            break
                        k += 16
                        continue
                    k += r
                    if k > 63:
                        raise ValueError("coefficient index past 63")
                    blk[ZIGZAG[k]] = _extend(get(s), s)
                    k += 1
            if p > nbits:
                raise ValueError("ran out of bits")
            mcu += 1
    if mcu < n_mcu:
        raise ValueError("fewer MCUs than the frame needs")
    return coef


# jidctint.c constants (CONST_BITS 13)
_F = dict(f0298=2446, f0390=3196, f0541=4433, f0765=6270, f0899=7373, f1175=9633, f1501=12299, f1847=15137,
          f1961=16069, f2053=16819, f2562=20995, f3072=25172)
CONST_BITS, PASS1_BITS = 13, 2


def _wrap16(x):
    return ((x + 32768) & 0xFFFF) - 32768


def _idct_1d(v, shift):
    """One pass of the islow IDCT (jidctint.c jpeg_idct_islow) over the last axis, as the SIMD routines that Pillow's
    libjpeg-turbo runs compute it (jidctint-sse2.asm / -avx2.asm): inputs are int16; the sums in0 + in4, in0 - in4,
    in7 + in3 and in5 + in1 wrap in 16 bits (paddw / psubw); every product and the rest are exact 32-bit integers; the
    DESCALE by `shift` is saturated to int16 (packssdw). Where nothing overflows this is the C routine's arithmetic."""
    f = _F
    z2, z3 = v[..., 2], v[..., 6]
    tmp2 = z2 * f["f0541"] + z3 * (f["f0541"] - f["f1847"])
    tmp3 = z2 * (f["f0541"] + f["f0765"]) + z3 * f["f0541"]
    tmp0 = _wrap16(v[..., 0] + v[..., 4]) << CONST_BITS
    tmp1 = _wrap16(v[..., 0] - v[..., 4]) << CONST_BITS
    t10, t13, t11, t12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    t0, t1, t2, t3 = v[..., 7], v[..., 5], v[..., 3], v[..., 1]
    z3, z4 = _wrap16(t0 + t2), _wrap16(t1 + t3)
    z3, z4 = z3 * (f["f1175"] - f["f1961"]) + z4 * f["f1175"], z3 * f["f1175"] + z4 * (f["f1175"] - f["f0390"])
    a0 = t0 * (f["f0298"] - f["f0899"]) - t3 * f["f0899"] + z3
    a1 = t1 * (f["f2053"] - f["f2562"]) - t2 * f["f2562"] + z4
    a2 = -t1 * f["f2562"] + t2 * (f["f3072"] - f["f2562"]) + z3
    a3 = -t0 * f["f0899"] + t3 * (f["f1501"] - f["f0899"]) + z4
    r = 1 << (shift - 1)
    out = [t10 + a3, t11 + a2, t12 + a1, t13 + a0, t13 - a0, t12 - a1, t11 - a2, t10 - a3]
    return np.clip(np.stack([(o + r) >> shift for o in out], axis=-1), -32768, 32767)


def idct_islow(coef, qt):
    """jpeg_idct_islow on blocks (..., 64) natural order with quantisation table qt (64,) -> (..., 8, 8) uint8 samples,
    as Pillow computes it (see _idct_1d):
      - DEQUANTIZE is a 16-bit product (pmullw);
      - pass 1 over columns, DESCALE by CONST_BITS - PASS1_BITS; when every coefficient outside the first row of the
        block is zero, pass 1 is the shortcut in0 * q << PASS1_BITS for all eight rows, in 16 bits (psllw);
      - pass 2 over rows, DESCALE by CONST_BITS + PASS1_BITS + 3;
      - the result is clamped to -128..127 (packsswb) and centred. The C routine's range_limit[x & RANGE_MASK] instead
        wraps values of 512 and more to 0: Pillow's build does not, and the clamp is what it returns."""
    c = coef.reshape(coef.shape[:-1] + (8, 8))                         # [row (vertical frequency), col]
    d = _wrap16(c * qt.reshape(8, 8))
    ws = np.swapaxes(_idct_1d(np.swapaxes(d, -1, -2), CONST_BITS - PASS1_BITS), -1, -2)
    dc_only = (c[..., 1:, :] == 0).all(axis=(-1, -2))
    ws = np.where(dc_only[..., None, None], _wrap16(d[..., :1, :] << PASS1_BITS), ws)
    x = _idct_1d(ws, CONST_BITS + PASS1_BITS + 3)
    return (np.clip(x, -128, 127) + 128).astype(np.uint8)


def sample_plane(coef, qt):
    """(bh, bw, 64) coefficients of one component -> its (bh*8, bw*8) sample plane."""
    bh, bw = coef.shape[:2]
    blocks = idct_islow(coef, qt)                                       # (bh, bw, 8, 8)
    return blocks.transpose(0, 2, 1, 3).reshape(bh * 8, bw * 8)


def upsample(plane, dw, dh, fh, fv, W, H):
    """jdsample.c for a component of downsampled size (dh, dw) (its real extent; rows and columns past it are never read)
    upsampled by (fh, fv) to at least (H, W), cropped to (H, W):
      (1,1) fullsize_upsample; (2,1) h2v1_fancy_upsample; (1,2) h1v2_fancy_upsample; (2,2) h2v2_fancy_upsample.
    The h2 filters fall back to plain replication (h2v1_upsample / h2v2_upsample) when dw <= 2 (jinit_upsampler)."""
    x = plane[:dh, :dw].astype(np.int64)
    if (fh, fv) == (1, 1):
        return x[:H, :W].astype(np.uint8)
    if fh == 2 and dw <= 2:
        out = np.repeat(np.repeat(x, fv, axis=0), 2, axis=1)
        return out[:H, :W].astype(np.uint8)
    up = np.concatenate([x[:1], x[:-1]], axis=0)                        # row above, first row replicated
    down = np.concatenate([x[1:], x[-1:]], axis=0)                      # row below, last row replicated
    if (fh, fv) == (1, 2):
        out = np.empty((2 * dh, dw), np.int64)
        out[0::2] = (3 * x + up + 1) >> 2
        out[1::2] = (3 * x + down + 2) >> 2
        return out[:H, :W].astype(np.uint8)
    if fv == 2:
        rows = np.empty((2 * dh, dw), np.int64)
        rows[0::2] = 3 * x + up
        rows[1::2] = 3 * x + down
        bias_l, bias_r, sh = 8, 7, 4
    else:
        rows, bias_l, bias_r, sh = x, 1, 2, 2
    left = np.concatenate([rows[:, :1], rows[:, :-1]], axis=1)
    right = np.concatenate([rows[:, 1:], rows[:, -1:]], axis=1)
    out = np.empty((rows.shape[0], 2 * dw), np.int64)
    out[:, 0::2] = (3 * rows + left + bias_l) >> sh
    out[:, 1::2] = (3 * rows + right + bias_r) >> sh
    return out[:H, :W].astype(np.uint8)


def ycc_rgb(y, cb, cr):
    """ycc_rgb_convert (jdcolor.c): build_ycc_rgb_table's fixed-point tables (SCALEBITS 16, ONE_HALF rounding), then
    range_limit (clamp to 0..255)."""
    SCALE, HALF = 16, 1 << 15
    y, cb, cr = (a.astype(np.int64) - np.array([0, 128, 128])[k] for k, a in enumerate((y, cb, cr)))
    r = y + ((91881 * cr + HALF) >> SCALE)
    g = y + ((-22554 * cb + HALF - 46802 * cr) >> SCALE)
    b = y + ((116130 * cb + HALF) >> SCALE)
    return np.clip(np.stack([r, g, b], axis=-1), 0, 255).astype(np.uint8)


def decode(data: bytes) -> np.ndarray:
    """The (H, W, 3) uint8 array `np.asarray(Image.open(f).convert('RGB'))` gives for a supported file."""
    hdr = parse(data)
    H, W, comps = hdr["H"], hdr["W"], hdr["comps"]
    coef = decode_coefficients(data, hdr)
    hmax, vmax = max(c[1] for c in comps), max(c[2] for c in comps)
    out = []
    for (cid, h, v, tq), c in zip(comps, coef):
        plane = sample_plane(c, hdr["q"][tq])
        dw, dh = -(-W * h // hmax), -(-H * v // vmax)
        if len(comps) == 1:
            out.append(plane[:H, :W])
        else:
            out.append(upsample(plane, dw, dh, hmax // h, vmax // v, W, H))
    if len(comps) == 1:
        return np.repeat(out[0][:, :, None], 3, axis=2)
    return ycc_rgb(*out)
