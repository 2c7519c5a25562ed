"""Synthetic side information and pictures for parity tests (seeded numpy; shapes follow include/ilf_b200.h)."""
import numpy as np
import pytest

SAO_DT = np.dtype([("offset", "<i2", (3, 4)), ("type", "i1", (3,)), ("band_pos", "u1", (3,)), ("avail", "u1"), ("reserved", "u1")])
assert SAO_DT.itemsize == 32
ALF_DT = np.dtype([("luma_coeff", "<i2", (25, 13)), ("chroma_coeff", "<i2", (7,)), ("luma_filter_7x7", "<i2")])
DB_DT = np.dtype([("cb_qp_offset", "<i4"), ("cr_qp_offset", "<i4"), ("mv_threshold", "<i4"), ("num_slices", "<i4"), ("slices", "i1", (64, 4))])


def keep_ids(rows, expand):
    """pytest parameters of cases written before their test took more columns (e.g. one bit depth for both planes): expand(*row)
    gives the test's columns, and each case keeps the id pytest gave the row as written."""
    return [pytest.param(*expand(*r), id="-".join(map(str, r))) for r in rows]


def picture(rng, w, h, bd=10, kind="mix", bd_chroma=None):
    """int16 planes with smooth areas, edges, noise and saturated patches (so clipping paths are hit); luma at `bd` bits,
    chroma at `bd_chroma` (default: `bd`)."""

    def plane(ww, hh, bd):
        mx = (1 << bd) - 1
        y, x = np.mgrid[0:hh, 0:ww]
        base = mx / 2 + mx / 3 * np.sin(x / 9.0) * np.cos(y / 7.0)
        blk = np.kron(rng.integers(-mx // 16, mx // 16 + 1, ((hh + 7) // 8, (ww + 7) // 8)), np.ones((8, 8), np.int64))[:hh, :ww]
        p = base + blk + rng.normal(0, mx / 100, (hh, ww))
        if kind == "noise":
            p = rng.integers(0, mx + 1, (hh, ww)).astype(np.float64)
        p = np.clip(np.rint(p), 0, mx)
        # saturated and flat patches
        for _ in range(4):
            yy, xx = rng.integers(0, hh), rng.integers(0, ww)
            p[yy:yy + 9, xx:xx + 13] = rng.choice([0, mx, mx // 2])
        return p.astype(np.int16)

    bdc = bd if bd_chroma is None else bd_chroma
    return {"y": plane(w, h, bd), "cb": plane(w // 2, h // 2, bdc), "cr": plane(w // 2, h // 2, bdc)}


def sao_params(rng, ctus_w, ctus_h, bd=10, p_off=0.25, all_avail=False, bd_chroma=None):
    """Offsets of each component in the range of its own bit depth (luma `bd`, chroma `bd_chroma`, default `bd`)."""
    n = ctus_w * ctus_h
    a = np.zeros(n, SAO_DT)
    maxo_of = lambda b: min(127, 31 << max(0, b - 10))
    maxos = (maxo_of(bd),) + 2 * (maxo_of(bd if bd_chroma is None else bd_chroma),)
    for i in range(n):
        for c in range(3):
            maxo = maxos[c]
            t = -1 if rng.random() < p_off else int(rng.integers(0, 5))
            a["type"][i, c] = t
            a["band_pos"][i, c] = rng.integers(0, 32)
            a["offset"][i, c] = rng.integers(-maxo, maxo + 1, 4)
        cx, cy = i % ctus_w, i // ctus_w
        av = 0xFF if all_avail else int(rng.integers(0, 256)) | (0xFF if rng.random() < 0.3 else 0)
        # picture borders are never available (deriveLoopFilterBoundaryAvailibility, SampleAdaptiveOffset.cpp:685-760)
        if cx == 0: av &= ~(0x01 | 0x10 | 0x40)
        if cx == ctus_w - 1: av &= ~(0x02 | 0x20 | 0x80)
        if cy == 0: av &= ~(0x04 | 0x10 | 0x20)
        if cy == ctus_h - 1: av &= ~(0x08 | 0x40 | 0x80)
        a["avail"][i] = av
    return a.view(np.uint8).reshape(n, 32)


def alf_params(rng, ctus_w, ctus_h, is7=True, p_on=0.8, big=False, dot=False):
    """big: every coefficient anywhere in +-511 (general arithmetic path).  dot: the limits of the dot-product path -- outer
    coefficients over the whole int8 range with both extremes present, the four neighbours of the centre up to +-1500, the
    centre whatever the normalisation leaves (negative and > 8000 occur)."""
    a = np.zeros(1, ALF_DT)
    lim = 511 if big else 40
    n = 13 if is7 else 7
    lc = np.zeros((25, 13), np.int64)
    lc[:, :n - 1] = rng.integers(-lim, lim + 1, (25, n - 1))
    cc = rng.integers(-lim, lim + 1, 7)
    if dot:
        lc[:, :n - 1] = rng.integers(-128, 128, (25, n - 1))
        lc[rng.integers(0, 25, 8), rng.integers(0, n - 1, 8)] = -128
        lc[rng.integers(0, 25, 8), rng.integers(0, n - 1, 8)] = 127
        inner = (6, 11) if is7 else (2, 5)      # (0, +-1) and (+-1, 0)
        for k in inner:
            lc[:, k] = rng.integers(-1500, 1501, 25)
        cc[:6] = rng.integers(-128, 128, 6)
        cc[0], cc[3] = -128, 127
        cc[2], cc[5] = rng.integers(-1500, 1501, 2)
    lc[:, n - 1] = 512 - 2 * lc[:, :n - 1].sum(axis=1)
    a["luma_coeff"][0] = np.clip(lc, -32768, 32767)
    cc[6] = 512 - 2 * cc[:6].sum()
    a["chroma_coeff"][0] = cc
    a["luma_filter_7x7"][0] = 1 if is7 else 0
    en = (rng.random((3, ctus_w * ctus_h)) < p_on).astype(np.uint8)
    return a.tobytes(), en


def deblock_info(rng, w, h, p_edge=0.5, p_intra=0.4, inter=False):
    """Synthetic per-4x4 grid (include/ilf_b200.h): random 8x8 'coding blocks' -- edge / TU flags on the 8-sample grid
    (never on the picture border), intra and cbf flags and QP per 8x8 block.  With inter=True the non-intra blocks carry
    random reference ids and int16 motion vectors (constant per 8x8 block).  Returns (params_bytes, info, mv16)."""
    uw, uh = w // 4, h // 4
    bw, bh = (uw + 1) // 2, (uh + 1) // 2
    up = lambda a: np.kron(a, np.ones((2, 2), a.dtype))[:uh, :uw]
    intra = up((rng.random((bh, bw)) < p_intra).astype(np.uint32))
    cbf = up((rng.random((bh, bw)) < 0.5).astype(np.uint32))
    qp = up(rng.integers(20, 46, (bh, bw)).astype(np.uint32))
    ev = up((rng.random((bh, bw)) < p_edge).astype(np.uint32))
    eh = up((rng.random((bh, bw)) < p_edge).astype(np.uint32))
    tv = up((rng.random((bh, bw)) < 0.7).astype(np.uint32))
    th = up((rng.random((bh, bw)) < 0.7).astype(np.uint32))
    xs, ys = np.arange(uw)[None, :], np.arange(uh)[:, None]
    ev = ev * ((xs % 2 == 0) & (xs > 0))   # a unit's LEFT border is an edge only on the 8-sample grid, not at x = 0
    eh = eh * ((ys % 2 == 0) & (ys > 0))
    ref0 = up(rng.integers(0, 3, (bh, bw)).astype(np.uint32)) if inter else np.full((uh, uw), 0xFF, np.uint32)
    ref1 = np.full((uh, uw), 0xFF, np.uint32)
    info = (intra | (cbf << 1) | (ev.astype(np.uint32) << 2) | ((tv * ev).astype(np.uint32) << 3) | (eh.astype(np.uint32) << 4) |
            ((th * eh).astype(np.uint32) << 5) | (qp << 8) | (ref0 << 16) | (ref1 << 24)).astype(np.uint32)
    mv16 = None
    if inter:
        mv = rng.integers(-12, 13, (bh, bw, 4)).astype(np.int16)
        mv16 = np.ascontiguousarray(np.kron(mv, np.ones((2, 2, 1), np.int16))[:uh, :uw])
        mv16[..., 2:] = 0
    prm = np.zeros(1, DB_DT)
    prm["cb_qp_offset"], prm["cr_qp_offset"], prm["mv_threshold"], prm["num_slices"] = 1, -1, 4, 1
    return prm.tobytes(), info, mv16


def deblock_info_stress(rng, w, h, ctu_log2=7, mv32=False, bd_luma=8, chroma_qp_offset=6):
    """Side information that real streams of the committed configurations rarely or never carry: several slices with their
    own beta / tc offsets (ctu_slice map), no-filter units (PCM / lossless), B-slice units with two reference ids and four
    motion-vector components, a separate chroma-tree layer, QPs over the whole range, optionally 32-bit motion vectors.
    The QPs of both layers come from [-6 (bd_luma - 8), 63] (negative at 10 and 12 bit, as the QP byte of the grid is signed),
    the PPS chroma QP offsets from +-chroma_qp_offset (the syntax allows +-12).  The defaults keep the draws of the cases
    written before these arguments existed.  Returns a dict with the keys of the bench side information."""
    uw, uh = w // 4, h // 4
    bw, bh = (uw + 1) // 2, (uh + 1) // 2
    up = lambda a: np.kron(a, np.ones((2, 2), a.dtype))[:uh, :uw]
    xs, ys = np.arange(uw)[None, :], np.arange(uh)[:, None]

    def layer(p_intra):
        intra = up((rng.random((bh, bw)) < p_intra).astype(np.uint32))
        cbf = up((rng.random((bh, bw)) < 0.5).astype(np.uint32))
        qp = up((rng.integers(-6 * (bd_luma - 8), 64, (bh, bw)) & 0xFF).astype(np.uint32))
        ev = up((rng.random((bh, bw)) < 0.6).astype(np.uint32)) * ((xs % 2 == 0) & (xs > 0))
        eh = up((rng.random((bh, bw)) < 0.6).astype(np.uint32)) * ((ys % 2 == 0) & (ys > 0))
        tv = up((rng.random((bh, bw)) < 0.7).astype(np.uint32))
        th = up((rng.random((bh, bw)) < 0.7).astype(np.uint32))
        nofilt = up((rng.random((bh, bw)) < 0.08).astype(np.uint32))
        bsl = up((rng.random((bh, bw)) < 0.6).astype(np.uint32))
        ids = np.array([0, 1, 2, 0xFF], np.uint32)
        ref0 = up(ids[rng.integers(0, 3, (bh, bw))])
        ref1 = up(ids[rng.integers(0, 4, (bh, bw))]) * bsl + np.uint32(0xFF) * (1 - bsl)
        return (intra | (cbf << 1) | (ev.astype(np.uint32) << 2) | ((tv * ev).astype(np.uint32) << 3) | (eh.astype(np.uint32) << 4) |
                ((th * eh).astype(np.uint32) << 5) | (nofilt << 6) | (bsl << 7) | (qp << 8) | (ref0 << 16) | (ref1.astype(np.uint32) << 24)).astype(np.uint32)

    info, info_c = layer(0.3), layer(0.6)
    span = 40000 if mv32 else 14
    mv = np.kron(rng.integers(-span, span + 1, (bh, bw, 4)), np.ones((2, 2, 1), np.int64))[:uh, :uw]
    ctu = 1 << ctu_log2
    cw, ch = (w + ctu - 1) // ctu, (h + ctu - 1) // ctu
    prm = np.zeros(1, DB_DT)
    co = chroma_qp_offset
    prm["cb_qp_offset"], prm["cr_qp_offset"], prm["mv_threshold"], prm["num_slices"] = rng.integers(-co, co + 1), rng.integers(-co, co + 1), 16 if mv32 else 4, 3
    prm["slices"][0, :3, 0] = rng.integers(-6, 7, 3)
    prm["slices"][0, :3, 1] = rng.integers(-6, 7, 3)
    d = {"db_params": prm.tobytes(), "db_info": info, "db_info_c": info_c, "ctu_slice": np.sort(rng.integers(0, 3, cw * ch)).astype(np.uint8)}
    d["db_mv32" if mv32 else "db_mv16"] = np.ascontiguousarray(mv.astype(np.int32 if mv32 else np.int16))
    return d
