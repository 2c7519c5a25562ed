"""Consumers of the filtered picture on band contexts (one picture split into CTU-row bands): the decoded-picture hash of a split
picture (ilf_picture_hash_band + ilf_hash_combine), the bordered download of a band (ilf_download_band_extended) and the encoder
passes on a band (ilf_set_original_band, then SAO / ALF statistics, ALF classification and the deblocking offset search).  Every
band result must equal, bit for bit, the matching part of the whole-picture result, which is pinned to the oracle."""
import ctypes as C
import random

import numpy as np
import pytest

import golden_io as G
from band_util import rows
from test_gpu_deblock_search import distortion, with_offsets
from test_gpu_geometry import _db_args, inputs
from vvcsoftware_vtm_b200 import bands

pytestmark = pytest.mark.gpu
K = ("y", "cb", "cr")
ERR_ARG, ERR_STATE = -1, -3
STAGE_DEBLOCK, STAGE_SAO, STAGE_ALF = 1, 2, 4
# candidates whose table index clamps at both ends, next to ordinary ones
CANDS = [(0, 0), (3, -2), (-4, 5), (6, 6), (-128, 127), (127, -128), (20, -20)]
SHIFT = (2, 3)


def _set_side(f, slot, si):
    f.set_deblock_info(slot, *_db_args(si))
    f.set_sao_params(slot, si["sao_ctus"])
    f.set_alf_params(slot, si["alf_params"], si["alf_ctu_enable"])


def _whole(v, w, h, bl, bc, c, cases):
    """Whole-picture context, one slot per (pic, org, si) case, every input set."""
    f = v.InLoopFilter(w, h, bl, bc, c, num_slots=len(cases))
    for slot, (pic, org, si) in enumerate(cases):
        f.upload(slot, *(pic[k] for k in K))
        _set_side(f, slot, si)
        f.set_original(slot, org["y"], org["cb"], org["cr"], si["avail"])
    return f


def _banded(v, w, h, bl, bc, c, cases, n, devices=1):
    """n band contexts (rank r on device r % devices), each with one slot per case: own rows uploaded, halos exchanged in one
    batch, side information and the original of the own rows set.  The way test_gpu_bands._run_banded sets bands up."""
    ctu = 1 << c
    part = bands.band_partition((h + ctu - 1) // ctu, n)
    ctxs = [v.InLoopFilter(w, h, bl, bc, c, band=b, device=r % devices, num_slots=len(cases)) for r, b in enumerate(part)]
    for f in ctxs:
        for slot, (pic, _, _) in enumerate(cases):
            f.upload_band(slot, *rows(pic, f.own_row0, f.own_row0 + f.own_rows).values())
    for f in ctxs:
        f.sync()
    for slot in range(len(cases)):
        handles = [f.band_export(slot) for f in ctxs]
        for r, f in enumerate(ctxs):
            bands.connect_bands(f, slot, r, n, handles)
    for f in ctxs:
        f.band_exchange(0, len(cases))
        for slot, (_, org, si) in enumerate(cases):
            _set_side(f, slot, bands.slice_side_info(si, f.row0, f.rows))
            f.set_original_band(slot, *rows(org, f.own_row0, f.own_row0 + f.own_rows).values(), si["avail"])
    return ctxs


def _close(ctxs):
    for f in ctxs:
        f.close()


def _hash_parts(v, ctxs, slot, rng):
    parts = [f.picture_hash_band(slot) for f in ctxs]
    rng.shuffle(parts)
    return {kind: v.hash_combine(parts, kind) for kind in ("crc", "checksum")}


def _slice_border_on_band_border(si, w, h, c, n):
    """A slice starts at the first CTU row of the second band: A / AL of that row cleared."""
    if n < 2:
        return si
    ctu = 1 << c
    cw = (w + ctu - 1) // ctu
    r = bands.band_partition((h + ctu - 1) // ctu, n)[1][0]
    si = dict(si)
    si["avail"] = si["avail"].copy()
    si["avail"][r * cw:(r + 1) * cw] &= ~np.uint8(0x04 | 0x10)
    return si


def _check_consumers(v, O, w, h, bl, bc, c, cases, n, devices=1, with_oracle=True):
    """Hash (input and chain), statistics, classification, search and bordered download of every band against the whole picture
    (slot 0 also against the oracle)."""
    rng = random.Random(w * 31 + h + n)
    whole = _whole(v, w, h, bl, bc, c, cases)
    ctxs = _banded(v, w, h, bl, bc, c, cases, n, devices)
    S = len(cases)
    try:
        # the freshly exchanged input, before any stage
        for slot, (pic, _, _) in enumerate(cases):
            got = _hash_parts(v, ctxs, slot, rng)
            for kind in ("crc", "checksum"):
                assert got[kind] == whole.picture_hash(slot, kind), f"input, slot {slot}, {kind}"
                if with_oracle and slot == 0:
                    assert got[kind] == O.picture_hash(pic, bl, bc, kind), f"input, {kind} vs oracle"
        # offset search on the uploaded picture: the bands' sums add up to the whole picture's
        whole.deblock_search(CANDS, SHIFT, 0, S)
        for f in ctxs:
            f.deblock_search(CANDS, SHIFT, 0, S)
        for slot in range(S):
            total = sum(f.get_deblock_search(slot) for f in ctxs)
            assert np.array_equal(total, whole.get_deblock_search(slot)), f"search, slot {slot}"
        # SAO statistics of the deblocked picture
        whole.run(0, S, STAGE_DEBLOCK)
        whole.sao_stats(0, S)
        for f in ctxs:
            f.run(0, S, STAGE_DEBLOCK)
            f.sao_stats(0, S)
        for slot in range(S):
            got = np.concatenate([f.get_sao_stats(slot) for f in ctxs])
            assert np.array_equal(got, whole.get_sao_stats(slot)), f"SAO statistics, slot {slot}"
        # ALF statistics and classification of the SAO'd picture
        whole.run(0, S, STAGE_SAO)
        whole.alf_stats(0, S)
        for f in ctxs:
            f.run(0, S, STAGE_SAO)
            f.alf_stats(0, S)
        for slot in range(S):
            got = np.concatenate([f.get_alf_stats(slot) for f in ctxs])
            assert np.array_equal(got, whole.get_alf_stats(slot)), f"ALF statistics, slot {slot}"
            cls = np.concatenate([f.alf_classify(slot) for f in ctxs])
            assert np.array_equal(cls, whole.alf_classify(slot)), f"ALF classes, slot {slot}"
        if with_oracle:
            pic, org, si = cases[0]
            d = O.deblock(pic, bl, bc, c, *_db_args(si))
            assert np.array_equal(whole.get_sao_stats(0), O.sao_stats(d, org, bl, bc, c, si["avail"])), "whole-picture SAO statistics vs oracle"
            s = O.sao(d, bl, bc, c, si["sao_ctus"])
            assert np.array_equal(whole.get_alf_stats(0), O.alf_stats(s, org, bl, c)), "whole-picture ALF statistics vs oracle"
        # the whole chain from the uploaded input (the statistics and the search wrote no picture plane)
        for f in ctxs:
            f.run(0, S, STAGE_DEBLOCK | STAGE_SAO | STAGE_ALF)
        whole.run(0, S, STAGE_DEBLOCK | STAGE_SAO | STAGE_ALF)
        for slot, (pic, _, si) in enumerate(cases):
            got = _hash_parts(v, ctxs, slot, rng)
            for kind in ("crc", "checksum"):
                assert got[kind] == whole.picture_hash(slot, kind), f"chain, slot {slot}, {kind}"
            if with_oracle and slot == 0:
                a = O.alf(O.sao(O.deblock(pic, bl, bc, c, *_db_args(si)), bl, bc, c, si["sao_ctus"]), bl, bc, c, si["alf_params"], si["alf_ctu_enable"])
                for kind in ("crc", "checksum"):
                    assert got[kind] == O.picture_hash(a, bl, bc, kind), f"chain, {kind} vs oracle"
            # bordered download: every band into one sentinel-filled set of planes
            for margin in (0, 2, 144):
                out = None
                for f in ctxs:
                    out = f.download_band_extended(slot, margin, out)
                want = whole.download_extended(slot, margin)
                for k, sh in (("y", 0), ("cb", 1), ("cr", 1)):
                    assert np.array_equal(out[k], want[k]), f"bordered download, slot {slot}, margin {margin}, plane {k}"
                    if with_oracle and slot == 0 and margin:
                        assert np.array_equal(out[k], O.extend_border(a[k], margin >> sh, margin >> sh)), f"bordered download vs oracle, {k}"
    finally:
        whole.close()
        _close(ctxs)


# (w, h, ctu_log2, bd_luma, bd_chroma, motion, chroma-tree layer, bands): the synthetic sizes of test_gpu_bands, the short last CTU
# rows of test_gpu_geometry.BAND_CASES, CTU 32 / 64 / 128, 8 / 10 / 12 bit with unequal depths, 1 .. 5 bands
CASES = [(200, 136, 5, 10, 10, "mv16", False, 2), (200, 136, 5, 10, 10, "none", True, 3), (264, 200, 5, 8, 8, "mv32", True, 4),
         (416, 240, 6, 10, 10, "mv16", False, 2), (1920, 1080, 7, 10, 10, "mv16", True, 3), (264, 200, 5, 12, 8, "mv32", False, 3),
         (264, 136, 6, 8, 12, "mv16", True, 2), (328, 136, 5, 12, 10, "none", False, 3), (24, 1032, 6, 10, 8, "mv32", True, 3),
         (416, 240, 7, 10, 10, "none", False, 1), (256, 256, 7, 8, 10, "mv16", True, 2), (264, 200, 5, 10, 12, "mv16", True, 5)]


@pytest.mark.parametrize("w,h,c,bl,bc,mv,ctree,n", CASES, ids=[f"{w}x{h}-ctu{1 << c}-{bl}-{bc}-{mv}{'-ctree' if t else ''}-bands{n}" for w, h, c, bl, bc, mv, t, n in CASES])
def test_band_consumers_equal_whole_picture(w, h, c, bl, bc, mv, ctree, n, ilf_lib, oracle):
    """Two slots per band context (two pictures in one batch); slot 0 is also checked against the oracle."""
    cases = []
    for slot in range(2):
        pic, org, si = inputs(7000 + 97 * slot + w + h + n, w, h, c, bl, bc, mv, ctree, True, "dot")
        cases.append((pic, org, _slice_border_on_band_border(si, w, h, c, n)))
    _check_consumers(ilf_lib, oracle, w, h, bl, bc, c, cases, n, with_oracle=w * h <= 416 * 240)


def _capture_case(name, seed):
    cap = G.load_golden([p for p in G.golden_files() if name in p][0])
    g = cap["geom"]
    pic = {k: cap["pre_" + k] for k in K}
    rng = np.random.default_rng(seed)
    org = {k: np.clip(pic[k].astype(np.int32) + rng.integers(-12, 13, pic[k].shape), 0, (1 << (g["bd_luma"] if k == "y" else g["bd_chroma"])) - 1).astype(np.int16)
           for k in K}
    ctu = 1 << g["ctu_log2"]
    cw, ch = (g["width"] + ctu - 1) // ctu, (g["height"] + ctu - 1) // ctu
    av = rng.integers(0, 256, cw * ch).astype(np.uint8)
    av[np.arange(cw * ch) % cw == 0] &= ~np.uint8(0x01 | 0x10)
    av[:cw] &= ~np.uint8(0x04 | 0x10)
    si = {"db_params": cap["db_params"].tobytes(), "db_info": cap["db_info"], "db_info_c": cap.get("db_info_c"), "db_mv16": None, "db_mv32": cap["db_mv32"],
          "ctu_slice": cap["ctu_slice"], "sao_ctus": cap["sao_ctus"], "alf_params": cap["alf_params"].tobytes(), "alf_ctu_enable": cap["alf_ctu_enable"], "avail": av}
    return g, (pic, org, si)


def test_band_consumers_on_the_reference_capture(ilf_lib, oracle):
    g, case = _capture_case("ra_416x240_05", 5)
    case = (case[0], case[1], _slice_border_on_band_border(case[2], g["width"], g["height"], g["ctu_log2"], 2))
    _check_consumers(ilf_lib, oracle, g["width"], g["height"], g["bd_luma"], g["bd_chroma"], g["ctu_log2"], [case], 2)


def test_band_consumers_on_two_devices_in_one_process(ilf_lib, oracle):
    """Bands on two GPUs of one process (halo over peer access): the same hash, statistics and search checks.  Skipped on a
    one-GPU box."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    g, case = _capture_case("ra_416x240_05", 6)
    _check_consumers(ilf_lib, oracle, g["width"], g["height"], g["bd_luma"], g["bd_chroma"], g["ctu_log2"], [case], 2, devices=2)


@pytest.mark.parametrize("mv,ctree", [("none", True), ("mv16", False), ("mv32", True)])
def test_band_search_sums_equal_numpy_over_own_rows(mv, ctree, ilf_lib, oracle):
    """Each band's sums = a numpy sum over its own rows of the oracle's picture deblocked with every slice's offsets rewritten."""
    w, h, c, bl, bc, n = 264, 200, 5, 10, 10, 3
    pic, org, si = inputs(8100 + len(mv), w, h, c, bl, bc, mv, ctree, True, "dot")
    ctxs = _banded(ilf_lib, w, h, bl, bc, c, [(pic, org, si)], n)
    try:
        for shift in ((0, 0), SHIFT):
            for f in ctxs:
                f.deblock_search(CANDS, shift)
            got = [f.get_deblock_search(0) for f in ctxs]
            for k, (b, t) in enumerate(CANDS):
                prm, info, info_c, mv16, mv32, slc = _db_args(si)
                d = oracle.deblock(pic, bl, bc, c, with_offsets(prm, b, t), info, info_c, mv16, mv32, slc)
                for f, gb in zip(ctxs, got):
                    y0, y1 = f.own_row0, f.own_row0 + f.own_rows
                    assert np.array_equal(gb[k], distortion(rows(d, y0, y1), rows(org, y0, y1), shift)), f"band at row {y0}, candidate {(b, t)}, shift {shift}"
    finally:
        _close(ctxs)


def test_single_band_writes_only_its_own_part_of_the_bordered_planes(ilf_lib):
    w, h, c, n = 264, 200, 5, 3
    pic, org, si = inputs(8200, w, h, c, 10, 10, "mv16", False, True, "dot")
    whole = _whole(ilf_lib, w, h, 10, 10, c, [(pic, org, si)])
    ctxs = _banded(ilf_lib, w, h, 10, 10, c, [(pic, org, si)], n)
    try:
        whole.run(0, 1, 7)
        for f in ctxs:
            f.run(0, 1, 7)
        for margin in (0, 2, 144):
            want = whole.download_extended(0, margin)
            for f in ctxs:
                got = f.download_band_extended(0, margin)
                for k, sh in (("y", 0), ("cb", 1), ("cr", 1)):
                    m = margin >> sh
                    r0 = m + (f.own_row0 >> sh)
                    r1 = r0 + (f.own_rows >> sh)
                    if f.own_row0 == 0:
                        r0 = 0
                    if f.own_row0 + f.own_rows == h:
                        r1 = got[k].shape[0]
                    mine = np.zeros(got[k].shape[0], bool)
                    mine[r0:r1] = True
                    assert np.array_equal(got[k][mine], want[k][mine]), f"band at row {f.own_row0}, margin {margin}, plane {k}"
                    assert (got[k][~mine] == -1).all(), f"band at row {f.own_row0} wrote outside its rows, margin {margin}, plane {k}"
        for bad in (3, -2):   # the margin must be even and >= 0
            with pytest.raises(ilf_lib.IlfError, match="error -1"):
                ctxs[0].download_band_extended(0, bad)
    finally:
        whole.close()
        _close(ctxs)


def test_states_and_errors(ilf_lib):
    lib = ilf_lib.load_library()
    w, h, c = 200, 136, 5
    pic, org, si = inputs(8300, w, h, c, 10, 10, "mv16", False, True, "dot")
    part = ilf_lib.IlfHashPart()
    cand = (C.c_int8 * 2)(0, 0)
    shift = (C.c_int32 * 2)(0, 0)
    z = np.zeros(16, np.int16)
    zp = z.ctypes.data_as(C.c_void_p)
    av = si["avail"]

    def err(f):
        return lib.ilf_last_error(f._h)
    # whole-picture contexts: the band twins refuse
    with ilf_lib.InLoopFilter(w, h, 10, 10, c) as f:
        f.upload(0, *(pic[k] for k in K))
        assert lib.ilf_picture_hash_band(f._h, 0, C.byref(part)) == ERR_STATE
        assert lib.ilf_download_band_extended(f._h, 0, zp, 8, zp, 8, zp, 8, 0) == ERR_STATE
        assert lib.ilf_set_original_band(f._h, 0, zp, 8, zp, 8, zp, 8, av.ctypes.data_as(C.c_void_p)) == ERR_STATE
    ctxs = [ilf_lib.InLoopFilter(w, h, 10, 10, c, band=b) for b in bands.band_partition(5, 2)]
    try:
        f = ctxs[0]
        own = rows(org, f.own_row0, f.own_row0 + f.own_rows)
        # before an upload
        assert lib.ilf_picture_hash_band(f._h, 0, C.byref(part)) == ERR_STATE
        assert lib.ilf_set_original_band(f._h, 0, *(a for k in K for a in (own[k].ctypes.data_as(C.c_void_p), own[k].shape[1])), av.ctypes.data_as(C.c_void_p)) == ERR_STATE
        with pytest.raises(ilf_lib.IlfError):
            f.download_band_extended(0, 2)
        assert lib.ilf_picture_hash_band(f._h, 5, C.byref(part)) == ERR_ARG
        for g in ctxs:
            g.upload_band(0, *rows(pic, g.own_row0, g.own_row0 + g.own_rows).values())
        handles = [g.band_export(0) for g in ctxs]
        for r, g in enumerate(ctxs):
            bands.connect_bands(g, 0, r, 2, handles)
            g.band_exchange(0)
            _set_side(g, 0, bands.slice_side_info(si, g.row0, g.rows))
        assert lib.ilf_picture_hash_band(f._h, 0, None) == ERR_ARG
        # the existing refusals stay as they were
        assert lib.ilf_picture_hash(f._h, 0, 1, (C.c_uint32 * 3)()) == ERR_STATE and b"part of the picture" in err(f)
        assert lib.ilf_download_extended(f._h, 0, zp, 8, zp, 8, zp, 8, 0) == ERR_STATE and b"not available on band contexts" in err(f)
        with pytest.raises(ilf_lib.IlfError):
            f.set_original(0, org["y"], org["cb"], org["cr"], av)
        # without a band original the encoder passes refuse
        assert lib.ilf_sao_stats(f._h, 0, 1) == ERR_STATE
        assert lib.ilf_alf_stats(f._h, 0, 1) == ERR_STATE and b"not available on band contexts" in err(f)
        assert lib.ilf_deblock_search(f._h, 0, 1, cand, 1, shift) == ERR_STATE and b"not available on band contexts" in err(f)
        out = np.zeros(1 << 20, np.int64)
        assert lib.ilf_get_sao_stats(f._h, 0, out.ctypes.data_as(C.c_void_p)) == ERR_STATE
        assert lib.ilf_get_alf_stats(f._h, 0, out.ctypes.data_as(C.c_void_p)) == ERR_STATE
        assert lib.ilf_get_deblock_search(f._h, 0, out.ctypes.data_as(C.c_void_p), 64) == ERR_STATE
        # with one they run, and leave the picture alone
        f.set_original_band(0, own["y"], own["cb"], own["cr"], av)
        before = f.download_band(0)
        f.sao_stats()
        f.alf_stats()
        f.deblock_search(CANDS)
        after = f.download_band(0)
        assert all(np.array_equal(before[k], after[k]) for k in K)
        # a new upload needs a new band original
        f.upload_band(0, *rows(pic, f.own_row0, f.own_row0 + f.own_rows).values())
        assert lib.ilf_sao_stats(f._h, 0, 1) == ERR_STATE
        assert lib.ilf_deblock_search(f._h, 0, 1, cand, 1, shift) == ERR_STATE and b"not available on band contexts" in err(f)
    finally:
        _close(ctxs)
