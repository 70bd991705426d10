"""oracle.jpeg_decode against Pillow, byte for byte, on the seeded corpus of tests/jpeg_corpus.py: the numpy
restatement of baseline decoding (Huffman with DC prediction and restarts, the islow IDCT as libjpeg-turbo's SIMD
routines compute it, fancy upsampling, YCbCr -> RGB) that the device decoder is checked against."""
import numpy as np
import pytest

import jpeg_corpus as C
from oracle import jpeg_decode as J

CORPUS = C.corpus()


@pytest.mark.parametrize("name,data", CORPUS, ids=[n for n, _ in CORPUS])
def test_oracle_is_pillow(name, data):
    got, want = J.decode(data), C.pillow(data)
    assert got.shape == want.shape and got.dtype == want.dtype
    assert np.array_equal(got, want), (name, int((got != want).sum()))


def test_corpus_covers_every_supported_layout():
    seen = set()
    for _, data in CORPUS:
        hdr = J.parse(data)
        seen.add((len(hdr["comps"]), hdr["comps"][0][1], hdr["comps"][0][2], hdr["dri"] > 0))
    for lum in ((1, 1), (2, 1), (1, 2), (2, 2)):
        for dri in (False, True):
            assert (3, *lum, dri) in seen
    assert (1, 1, 1, False) in seen and (1, 1, 1, True) in seen


def test_extreme_coefficients_leave_the_16_bit_range():
    """The written extreme files reach what separates libjpeg-turbo's SIMD arithmetic from its C source: IDCT outputs
    past +-512 (the C range-limit table wraps them, Pillow clamps) and pass-1 values past int16."""
    reached_wrap = reached_sat = False
    for name, data in CORPUS:
        if not name.startswith("written_extreme"):
            continue
        hdr = J.parse(data)
        for (_, _, _, tq), c in zip(hdr["comps"], J.decode_coefficients(data, hdr)):
            d = (c * hdr["q"][tq]).reshape(c.shape[:-1] + (8, 8))
            ws = np.swapaxes(J._idct_1d(np.swapaxes(d, -1, -2), 11), -1, -2)
            x = J._idct_1d(ws, 18)
            reached_wrap |= bool((np.abs(x) >= 512).any())
            reached_sat |= bool((np.abs(ws) >= 32767).any())
    assert reached_wrap and reached_sat

