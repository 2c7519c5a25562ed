"""Pins the oracle's SAO and ALF block functions against the REFERENCE's own functions, driven directly with random
blocks, offsets, availability flags and coefficients (oracle/_ref/libvtm_units.so = extern "C" doors onto
SampleAdaptiveOffset::offsetBlock, AdaptiveLoopFilter::deriveClassificationBlk and filterBlk of the unmodified
reference objects, scalar and x86-SIMD flavours).

Where oracle/_ref was built, the reference runs and the oracle must equal it.  Everywhere else the oracle's result must have
the digest of the reference's result for the same case, stored in tests/golden/oracle_units.json; where the reference runs,
its results must have those digests too, and ILF_GOLDEN_RECORD=1 rewrites the file from them instead."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNITS = os.path.join(ROOT, "oracle", "_ref", "libvtm_units.so")
GOLDEN = os.path.join(ROOT, "tests", "golden", "oracle_units.json")
RECORD = os.environ.get("ILF_GOLDEN_RECORD") == "1"
K = ("y", "cb", "cr")

with open(GOLDEN) as _fh:
    _GOLDEN = json.load(_fh)


def _digest(a):
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()[:32]


def check(key, got, want, detail=None):
    """`got` is the reference's result for case `key`: equal to `want` where the reference ran (want is None where it
    did not), and with the digest stored for the case."""
    if want is None:
        assert _digest(got) == _GOLDEN[key], f"{key}: differs from the reference's result (stored digest)"
        return
    assert np.array_equal(got, want), f"{key}: " + (detail(got, want) if detail else "differs from the reference's result")
    if RECORD:
        _GOLDEN[key] = _digest(want)
    else:
        assert _GOLDEN.get(key) == _digest(want), f"{key}: the stored digest is not the reference's result"


@pytest.fixture(scope="module", autouse=True)
def _record_golden():
    yield
    if RECORD and os.path.exists(UNITS):
        with open(GOLDEN, "w") as fh:
            json.dump(_GOLDEN, fh, indent=0, sort_keys=True)
            fh.write("\n")


@pytest.fixture(scope="module")
def units():
    """The reference's block functions, or None where oracle/_ref was not built (needs the reference sources)."""
    if not os.path.exists(UNITS):
        return None
    lib = C.CDLL(UNITS)
    lib.ref_sao_offset_block.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint]
    lib.ref_alf_classify.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.ref_alf_filter.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.ref_sao_blk_stats.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint, C.c_void_p]
    for fn in (lib.ref_plane_crc, lib.ref_plane_checksum):
        fn.restype = C.c_uint
        fn.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.ref_extend_pic_border.argtypes = [C.c_void_p] * 3 + [C.c_int] * 3 + [C.c_void_p] * 3
    lib.ref_alf_blk_stats.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    return lib


def ref_sao(units, pic, bd, ctu_log2, prm):
    """SAOProcess restated with the reference's offsetBlock per CTU and component (offsetCTU, SampleAdaptiveOffset.cpp:510-562)."""
    P = prm.view(synth.SAO_DT).reshape(-1)
    h, w = pic["y"].shape
    ctu = 1 << ctu_log2
    cw = (w + ctu - 1) // ctu
    out = {}
    for ci, k in enumerate(K):
        sh = 1 if ci else 0
        pad = np.pad(pic[k], 1, mode="constant")          # offsetBlock may read one sample beyond the block
        dst = pad.copy()
        ph, pw = pic[k].shape
        sz = ctu >> sh
        for i in range(len(P)):
            t = int(P["type"][i, ci])
            if t < 0:
                continue
            cx, cy = i % cw, i // cw
            x0, y0 = cx * sz, cy * sz
            bw, bh = min(sz, pw - x0), min(sz, ph - y0)
            off = np.zeros(32, np.int32)
            o4 = P["offset"][i, ci].astype(np.int32)
            if t == 4:
                for j in range(4):
                    off[(int(P["band_pos"][i, ci]) + j) % 32] = o4[j]
            else:
                off[[0, 1, 3, 4]] = o4
            s = pad[1 + y0:, 1 + x0:]
            d = dst[1 + y0:, 1 + x0:]
            units.ref_sao_offset_block(bd, t, off.ctypes.data, s.ctypes.data, d.ctypes.data, pad.shape[1], pad.shape[1], bw, bh, int(P["avail"][i]))
        out[k] = dst[1:-1, 1:-1].copy()
    return out


def _first_diffs(got, want):
    bad = np.argwhere(got != want)
    return f"{len(bad)} samples differ from the reference, first at {bad[:5].tolist()}"


@pytest.mark.parametrize("w,h,bd,ctu_log2,seed", [(416, 240, 10, 7, 1), (200, 136, 10, 7, 2), (264, 72, 8, 6, 3), (136, 264, 12, 5, 4), (520, 392, 10, 7, 7)])
def test_sao_oracle_equals_reference_offset_block(w, h, bd, ctu_log2, seed, units, oracle):
    rng = np.random.default_rng(seed)
    ctu = 1 << ctu_log2
    cw, ch = (w + ctu - 1) // ctu, (h + ctu - 1) // ctu
    for kind in ("mix", "noise"):
        pic = synth.picture(rng, w, h, bd, kind)
        prm = synth.sao_params(rng, cw, ch, bd, p_off=0.2)
        want = ref_sao(units, pic, bd, ctu_log2, prm) if units else None
        got = oracle.sao(pic, bd, bd, ctu_log2, prm)
        for k in K:
            check(f"sao/{w}x{h}/bd{bd}/ctu{ctu_log2}/seed{seed}/{kind}/{k}", got[k], want[k] if want else None, _first_diffs)


@pytest.mark.parametrize("simd", [0, 1])
@pytest.mark.parametrize("w,h,bd,seed", [(64, 48, 10, 1), (136, 72, 8, 2), (96, 96, 10, 3)])
def test_alf_classification_oracle_equals_reference(simd, w, h, bd, seed, units, oracle):
    rng = np.random.default_rng(seed)
    for kind in ("mix", "noise"):
        y = synth.picture(rng, w, h, bd, kind)["y"]
        out = None
        if units:
            pad = np.pad(y, 4, mode="edge")
            out = np.zeros((h // 4, w // 4), np.uint8)
            units.ref_alf_classify(simd, pad[4:, 4:].ctypes.data, pad.shape[1], w, h, bd, out.ctypes.data)
        got = oracle.alf_classify(y, bd)
        check(f"alf_classify/simd{simd}/{w}x{h}/bd{bd}/seed{seed}/{kind}", got, out, lambda g, r: f"{(g != r).sum()} blocks differ")


@pytest.mark.parametrize("simd", [0, 1])
@pytest.mark.parametrize("is7", [True, False])
def test_alf_filter_oracle_equals_reference(simd, is7, units, oracle):
    rng = np.random.default_rng(5 + simd + 2 * is7)
    w, h, bd = 128, 64, 10            # one CTU-sized picture, ALF on
    for kind, big in (("mix", False), ("noise", False)):
        pic = synth.picture(rng, w, h, bd, kind)
        pb, en = synth.alf_params(rng, 1, 1, is7, p_on=1.1, big=big)
        got = oracle.alf(pic, bd, bd, 7, pb, en)
        A = np.frombuffer(pb, synth.ALF_DT)[0]
        cls = oracle.alf_classify(pic["y"], bd)
        for ci, k in enumerate(K):
            want = None
            if units:
                ph, pw = pic[k].shape
                pad = np.pad(pic[k], 4, mode="edge")
                dst = pad.copy()
                coeff = np.ascontiguousarray(A["luma_coeff"] if ci == 0 else A["chroma_coeff"], dtype=np.int16)
                units.ref_alf_filter(simd, int(is7) if ci == 0 else 0, int(ci > 0), pad[4:, 4:].ctypes.data, pad.shape[1], dst[4:, 4:].ctypes.data, pad.shape[1],
                                     pw, ph, bd, cls.ctypes.data, coeff.ctypes.data)
                want = dst[4:-4, 4:-4]
            check(f"alf_filter/simd{simd}/is7{int(is7)}/{kind}/{k}", got[k], want, lambda g, r: f"{(g != r).sum()} samples differ")


@pytest.mark.parametrize("bd,is_chroma,w,h,seed", [(10, 0, 128, 128, 1), (10, 1, 64, 64, 2), (8, 0, 64, 56, 3), (12, 1, 32, 28, 4), (10, 0, 32, 112, 5)])
def test_sao_statistics_block_vs_reference(units, oracle, bd, is_chroma, w, h, seed):
    """Encoder SAO statistics (SURVEY.md 8f): the oracle's block function == EncSampleAdaptiveOffset::getBlkStats of the
    reference for every combination of the six availability flags, on noisy and on flat (many ties) content."""
    rng = np.random.default_rng(seed)
    H, W = h + 16, w + 16
    for kind in ("noise", "flat"):
        if kind == "noise":
            src = rng.integers(0, 1 << bd, (H, W)).astype(np.int16)
        else:
            src = (rng.integers(0, 1 << (bd - 2), (H // 4 + 1, W // 4 + 1)).repeat(4, 0).repeat(4, 1)[:H, :W] * 4 + rng.integers(0, 2, (H, W))).astype(np.int16)
        org = np.clip(src.astype(np.int32) + rng.integers(-9, 10, (H, W)), 0, (1 << bd) - 1).astype(np.int16)
        want = None
        if units:
            want = np.zeros((64, 5, 64), np.int64)
            sp = src.ctypes.data + 2 * (8 * W + 8)
            gp = org.ctypes.data + 2 * (8 * W + 8)
            for avail6 in range(64):
                assert units.ref_sao_blk_stats(is_chroma, bd, sp, gp, W, W, w, h, avail6, want[avail6].ctypes.data) == 0
        got = np.stack([oracle.sao_stats_block(src, org, 8, 8, w, h, bd, is_chroma, avail6) for avail6 in range(64)])
        check(f"sao_stats/bd{bd}/chroma{is_chroma}/{w}x{h}/seed{seed}/{kind}", got, want,
              lambda g, r: "; ".join(f"avail6={a:06b}: types differing {np.nonzero((g[a] != r[a]).any(axis=1))[0]}" for a in range(64) if (g[a] != r[a]).any()))


# ---- post-filter consumers (SURVEY.md 8f rank 4): decoded-picture hash and reference border extension ----
@pytest.mark.parametrize("bd,w,h", [(10, 416, 240), (8, 264, 72), (12, 136, 264), (10, 200, 136), (10, 8, 8)])
def test_oracle_hash_and_border_match_reference(bd, w, h, units, oracle):
    """oracle CRC / checksum == the reference's compCRC / compChecksum (PicYuvMD5.cpp:91-163); oracle border extension ==
    Picture::extendPicBorder run on a real Picture (Picture.cpp:996-1040)."""
    rng = np.random.default_rng(bd * 1000 + w)
    pic = {"y": rng.integers(0, 1 << bd, (h, w)).astype(np.int16), "cb": rng.integers(0, 1 << bd, (h // 2, w // 2)).astype(np.int16),
           "cr": rng.integers(0, 1 << bd, (h // 2, w // 2)).astype(np.int16)}
    for kind, fn in (("crc", "ref_plane_crc"), ("checksum", "ref_plane_checksum")):
        want = None
        if units:
            want = np.array([getattr(units, fn)(pic[k].ctypes.data, pic[k].shape[1], pic[k].shape[1], pic[k].shape[0], bd) for k in K], np.uint32)
        check(f"hash/{kind}/bd{bd}/{w}x{h}", np.array(oracle.picture_hash(pic, bd, bd, kind), np.uint32), want)
    m = 16
    outs = None
    if units:
        outs = [np.zeros((a.shape[0] + 2 * (m >> s), a.shape[1] + 2 * (m >> s)), np.int16) for a, s in ((pic["y"], 0), (pic["cb"], 1), (pic["cr"], 1))]
        assert units.ref_extend_pic_border(pic["y"].ctypes.data, pic["cb"].ctypes.data, pic["cr"].ctypes.data, w, h, m, *(o.ctypes.data for o in outs)) == 0
    for i, (k, s) in enumerate((("y", 0), ("cb", 1), ("cr", 1))):
        check(f"border/bd{bd}/{w}x{h}/{k}", oracle.extend_border(pic[k], m >> s, m >> s), outs[i] if outs else None)


# ---- encoder ALF statistics (SURVEY.md 8f rank 3) ----
@pytest.mark.parametrize("shape7,w,h,bd,classes", [(1, 32, 24, 10, True), (0, 32, 24, 10, True), (0, 24, 16, 10, False), (1, 16, 16, 8, True), (1, 40, 8, 12, True)])
def test_oracle_alf_stats_match_reference_getblkstats(shape7, w, h, bd, classes, units, oracle):
    """oracle == EncAdaptiveLoopFilter::getBlkStats / calcCovariance (EncAdaptiveLoopFilter.cpp:1394-1514) for both filter shapes, all four
    transposes and 25 classes: E, y and pixAcc (the reference's doubles hold exact integers)."""
    rng = np.random.default_rng(shape7 * 100 + w + bd)
    rec = rng.integers(0, 1 << bd, (h, w)).astype(np.int16)
    org = np.clip(rec.astype(np.int32) + rng.integers(-40, 41, (h, w)), 0, (1 << bd) - 1).astype(np.int16)
    m = 4
    rec_pad = np.pad(rec, m, mode="edge")
    n = 13 if shape7 else 7
    words = n * (n + 1) // 2 + n + 1
    if classes:
        cls_u = (rng.integers(0, 25, (h // 4, w // 4)) | (rng.integers(0, 4, (h // 4, w // 4)) << 5)).astype(np.uint8)
        cls_s = np.ascontiguousarray(np.kron(cls_u, np.ones((4, 4), np.uint8)))
    ncl = 25 if classes else 1
    want = None
    if units:
        out = np.zeros((ncl, n * n + n + 1), np.float64)     # per class: E [n][n], y [n], pixAcc
        rp = rec_pad.ctypes.data + 2 * (m * rec_pad.shape[1] + m)
        assert units.ref_alf_blk_stats(shape7, org.ctypes.data, w, rp, rec_pad.shape[1], 0, 0, w, h, cls_s.ctypes.data if classes else None, w, out.ctypes.data) == 0
        assert out.any()
        want = out.astype(np.int64)
    got = np.zeros((ncl, words), np.int64)
    g = oracle.lib().ilf_oracle_alf_stats_block
    g.argtypes = [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_ssize_t, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    assert g(rec.ctypes.data, w, org.ctypes.data, w, w, h, shape7, cls_u.ctypes.data if classes else None, got.ctypes.data) == 0
    unpacked = [oracle.alf_stats_unpack(got[c], n) for c in range(ncl)]
    got_eyp = np.stack([np.concatenate([E.ravel(), y, [pa]]) for E, y, pa in unpacked]).astype(np.int64)
    check(f"alf_stats/shape7{shape7}/{w}x{h}/bd{bd}/classes{int(classes)}", got_eyp, want,
          lambda g_, r: f"classes differing (E, y or pixAcc): {np.nonzero((g_ != r).any(axis=1))[0].tolist()}")
