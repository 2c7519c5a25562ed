"""ilf_hash_combine on the host (no GPU): parts of a picture's decoded-picture hash, computed here the way ilf_picture_hash_band
defines them (CRC register contribution of the part's rows from a zero register, checksum partial sum with row masks in picture
coordinates), fold into the oracle's calcCRC / calcChecksum of the whole picture; parts that do not tile one picture are refused."""
import ctypes as C
import random

import numpy as np
import pytest

import synth

ERR_ARG = -1


def _crc_rows(plane, bd):
    """CRC register after the rows' message bits from a zero register (compCRC's bit order: low byte, then high byte, MSB first)."""
    s = 0
    for v in plane.astype(np.uint16).ravel().tolist():
        for b in range(16 if bd > 8 else 8):
            bit = (v >> (7 - b)) & 1 if b < 8 else (v >> (23 - b)) & 1
            s = (((s << 1) | bit) & 0xFFFF) ^ (0x1021 if s >> 15 else 0)
    return s


def _sum_rows(plane, bd, y0):
    h, w = plane.shape
    y = np.arange(y0, y0 + h)[:, None]
    x = np.arange(w)[None, :]
    mask = ((x & 0xFF) ^ (y & 0xFF) ^ (x >> 8) ^ (y >> 8)) & 0xFF
    v = plane.astype(np.int64) & 0xFFFF
    s = ((v & 0xFF) ^ mask).sum() + (((v >> 8) ^ mask).sum() if bd > 8 else 0)
    return int(s) & 0xFFFFFFFF


def _part(lib_mod, pic, bd_luma, bd_chroma, first, n):
    p = lib_mod.IlfHashPart()
    h, w = pic["y"].shape
    p.width, p.height, p.bd_luma, p.bd_chroma, p.first_row, p.num_rows = w, h, bd_luma, bd_chroma, first, n
    for i, (k, sh) in enumerate((("y", 0), ("cb", 1), ("cr", 1))):
        bd = bd_luma if k == "y" else bd_chroma
        rows = pic[k][first >> sh:(first + n) >> sh]
        p.crc[i] = _crc_rows(rows, bd)
        p.sum[i] = _sum_rows(rows, bd, first >> sh)
    return bytes(p)


@pytest.mark.parametrize("w,h,bd_luma,bd_chroma,cuts", [(16, 24, 10, 10, [8, 16]), (24, 16, 8, 12, [2]), (8, 520, 12, 8, [256, 264, 514]), (16, 8, 8, 8, [])])
def test_parts_combine_to_the_whole_picture_hash(w, h, bd_luma, bd_chroma, cuts, ilf_lib, oracle):
    """Rows 256 .. 263 of the tall picture make the checksum's (y >> 8) term differ from a part-local row index."""
    rng = np.random.default_rng(w * h + bd_luma)
    pic = synth.picture(rng, w, h, bd_luma, "noise", bd_chroma=bd_chroma)
    edges = [0] + cuts + [h]
    parts = [_part(ilf_lib, pic, bd_luma, bd_chroma, a, b - a) for a, b in zip(edges, edges[1:])]
    random.Random(h).shuffle(parts)
    for kind in ("crc", "checksum"):
        assert ilf_lib.hash_combine(parts, kind) == oracle.picture_hash(pic, bd_luma, bd_chroma, kind), kind


def _hp(lib_mod, width=64, height=32, bd_luma=10, bd_chroma=10, first_row=0, num_rows=32):
    p = lib_mod.IlfHashPart()
    p.width, p.height, p.bd_luma, p.bd_chroma, p.first_row, p.num_rows = width, height, bd_luma, bd_chroma, first_row, num_rows
    return p


def test_parts_that_do_not_tile_one_picture_are_refused(ilf_lib):
    lib = ilf_lib.load_library()
    P = ilf_lib.IlfHashPart
    out = (C.c_uint32 * 3)()
    hp = lambda **kw: _hp(ilf_lib, **kw)   # noqa: E731

    def combine(parts, kind=1, n=None):
        arr = (P * max(1, len(parts)))(*parts)
        return lib.ilf_hash_combine(arr, len(parts) if n is None else n, kind, C.byref(out))
    ok = [hp(first_row=16, num_rows=16), hp(first_row=0, num_rows=16)]
    assert combine(ok) == 0 and combine(ok, 2) == 0
    assert combine(ok, 3) == ERR_ARG and combine(ok, 0) == ERR_ARG
    assert combine(ok, n=0) == ERR_ARG
    assert combine([hp(num_rows=16)]) == ERR_ARG                                        # gap at the end
    assert combine([hp(num_rows=16), hp(first_row=18, num_rows=14)]) == ERR_ARG          # gap
    assert combine([hp(num_rows=18), hp(first_row=16, num_rows=16)]) == ERR_ARG          # overlap
    assert combine([hp(num_rows=16), hp(first_row=16, num_rows=16, width=72)]) == ERR_ARG
    assert combine([hp(num_rows=16), hp(first_row=16, num_rows=16, height=40)]) == ERR_ARG
    assert combine([hp(num_rows=16), hp(first_row=16, num_rows=16, bd_chroma=8)]) == ERR_ARG
    assert combine([hp(num_rows=15), hp(first_row=15, num_rows=17)]) == ERR_ARG          # odd rows: chroma would not split
    assert combine([hp(first_row=-2, num_rows=2), hp(num_rows=32)]) == ERR_ARG           # before the picture
    big = 0x7FFFFFFE                                                                      # rows that would overflow a running int sum
    assert combine([hp(num_rows=16), hp(first_row=16, num_rows=big), hp(first_row=16 + big, num_rows=big)]) == ERR_ARG
    assert combine([hp(num_rows=16), hp(first_row=16, num_rows=big)]) == ERR_ARG
    assert lib.ilf_hash_combine(None, 1, 1, C.byref(out)) == ERR_ARG
    assert lib.ilf_hash_combine((P * 1)(hp()), 1, 1, None) == ERR_ARG
    with pytest.raises(ilf_lib.IlfError):
        ilf_lib.hash_combine([])
    with pytest.raises(ilf_lib.IlfError, match="unknown hash kind"):
        ilf_lib.hash_combine([bytes(hp())], "md5")
