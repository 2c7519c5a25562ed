"""Deblocking leaves the chroma planes of a picture without an intra unit alone.

A chroma edge is filtered only when the block on one side is intra (bS = 2, LoopFilter.cpp:769), so in a picture whose chroma
decisions' grid has no intra unit deblocking cannot change Cb or Cr.  ilf_set_deblock_info records that per slot, and the
deblocking launch then skips both chroma planes like SAO and ALF skip a plane that is off: no load, no store, the plane stays
in the upload buffer while luma moves to a work buffer.  These tests check every path that reads a slot after such a run,
the decision itself (intra units at the end of the scan, in the chroma-tree layer, in a band's halo rows, a slot whose side
information changes) and that the skipped bytes are really not moved."""
import os
import sys
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (side-information loader and the synthetic planes of the benchmark)
import synth  # noqa: E402
from test_gpu_bands import _run_banded, _run_whole  # noqa: E402
from vvcsoftware_vtm_b200 import bands  # noqa: E402

pytestmark = pytest.mark.gpu
K = ("y", "cb", "cr")
BD, CTU = 10, 7
EDGE_V, EDGE_H, INTRA = 0x04, 0x10, 0x01
W1080, H1080 = 1920, 1080


def _set_db(f, slot, si):
    f.set_deblock_info(slot, si["db_params"], si["db_info"], si.get("db_info_c"), si.get("db_mv16"), si.get("db_mv32"), si.get("ctu_slice"))


def _set(f, slot, si):
    _set_db(f, slot, si)
    f.set_sao_params(slot, si["sao_ctus"])
    f.set_alf_params(slot, si["alf_params"], si["alf_ctu_enable"])


def _side(si):
    """bench side information with the parameter blocks as bytes, as the tests' helpers pass them."""
    d = dict(si)
    d["db_params"] = si["db_params"].tobytes()
    d["alf_params"] = si["alf_params"].tobytes()
    return d


def _has_intra(si):
    layer = si["db_info_c"] if si.get("db_info_c") is not None else si["db_info"]
    return bool((layer & INTRA).any())


def _oracle_deblock(O, pic, si, bd_luma=BD, bd_chroma=BD, ctu_log2=CTU):
    return O.deblock(pic, bd_luma, bd_chroma, ctu_log2, si["db_params"], si["db_info"], si.get("db_info_c"), si.get("db_mv16"), si.get("db_mv32"), si.get("ctu_slice"))


def _diff(got, want):
    return {k: int((got[k] != want[k]).sum()) for k in K}


def _crc(pic):
    return zlib.crc32(b"".join(np.ascontiguousarray(pic[k]).tobytes() for k in K))


_RA1080 = {}


def _ra1080(oracle):
    """The 8 pictures of the 1080p random-access workload (5 without an intra unit), their planes and the oracle's deblocking."""
    if not _RA1080:
        side = [_side(si) for si in bench.load_sideinfo("ra_1080p")]
        planes = [dict(zip(K, p)) for p in bench.synth_planes(W1080, H1080, len(side), seed=311)]
        _RA1080.update(side=side, planes=planes, deblocked=[_oracle_deblock(oracle, p, si) for p, si in zip(planes, side)])
    return _RA1080


@pytest.mark.parametrize("all_on", [False, True], ids=["stream", "all_on"])
@pytest.mark.parametrize("stages", [1, 7], ids=["deblock", "chain"])
def test_mixed_batch_equals_oracle_and_single_pictures(stages, all_on, ilf_lib, oracle):
    d = _ra1080(oracle)
    side = [_side(si) for si in bench.all_on_sideinfo(bench.load_sideinfo("ra_1080p"))] if all_on else d["side"]
    n = len(side)
    assert [_has_intra(si) for si in side].count(False) == 5
    with ilf_lib.InLoopFilter(W1080, H1080, BD, BD, CTU, num_slots=n) as f:
        for j in range(n):
            f.upload(j, *(d["planes"][j][k] for k in K))
            _set(f, j, side[j])
        f.run(0, n, stages)
        batch = [f.download(j) for j in range(n)]
    for j, (got, si) in enumerate(zip(batch, side)):
        want = d["deblocked"][j]
        if stages == 7:
            want = oracle.alf(oracle.sao(want, BD, BD, CTU, si["sao_ctus"]), BD, BD, CTU, si["alf_params"], si["alf_ctu_enable"])
        bad = _diff(got, want)
        assert not any(bad.values()), f"picture {j} (intra: {_has_intra(si)}): mismatching samples {bad}"
    with ilf_lib.InLoopFilter(W1080, H1080, BD, BD, CTU) as f:
        for j in range(n):
            f.upload(0, *(d["planes"][j][k] for k in K))
            _set(f, 0, side[j])
            f.run(0, 1, stages)
            assert _crc(f.download(0)) == _crc(batch[j]), f"picture {j}: batch != one at a time"


def test_readers_after_deblocking_an_intra_free_picture(ilf_lib, oracle):
    """After ilf_deblock of a picture without intra, luma is in a work buffer and chroma in the upload buffer: every reader
    must pick each plane where it is."""
    d = _ra1080(oracle)
    j = next(i for i, si in enumerate(d["side"]) if not _has_intra(si))
    si, pic, want = d["side"][j], d["planes"][j], d["deblocked"][j]
    assert not np.array_equal(want["y"], pic["y"])
    rng = np.random.default_rng(5)
    org = {k: np.clip(pic[k].astype(np.int32) + rng.integers(-6, 7, pic[k].shape), 0, 1023).astype(np.int16) for k in K}
    cw, ch = (W1080 + 127) // 128, (H1080 + 127) // 128
    avail = np.full(cw * ch, 0x15, np.uint8)
    avail[np.arange(cw * ch) % cw == 0] &= ~np.uint8(0x11)
    avail[:cw] &= ~np.uint8(0x14)
    with ilf_lib.InLoopFilter(W1080, H1080, BD, BD, CTU) as f:
        f.upload(0, *(pic[k] for k in K))
        _set(f, 0, si)
        f.loop_filter_pic(0)
        got = f.download(0)
        assert not any(_diff(got, want).values())
        for k in ("cb", "cr"):
            assert np.array_equal(got[k], pic[k]), f"{k} after deblocking != uploaded {k}"
        margin = 16
        ext = f.download_extended(0, margin)
        for k in K:
            m = margin >> (k != "y")
            assert np.array_equal(ext[k], oracle.extend_border(want[k], m, m)), f"download_extended: plane {k}"
        for kind in ("crc", "checksum"):
            assert f.picture_hash(0, kind) == oracle.picture_hash(want, BD, BD, kind), kind
        f.set_original(0, org["y"], org["cb"], org["cr"], avail)
        f.sao_stats(0, 1)
        assert np.array_equal(f.get_sao_stats(0), oracle.sao_stats(want, org, BD, BD, CTU, avail)), "SAO statistics"
        f.alf_stats(0, 1)
        assert np.array_equal(f.get_alf_stats(0), oracle.alf_stats(want, org, BD, CTU)), "ALF statistics"
        # the later stages one call at a time read luma from the work buffer and chroma from the upload buffer
        f.sao_process(0)
        f.alf_process(0)
        want = oracle.alf(oracle.sao(want, BD, BD, CTU, si["sao_ctus"]), BD, BD, CTU, si["alf_params"], si["alf_ctu_enable"])
        assert not any(_diff(f.download(0), want).values()), "SAO + ALF after deblocking"


def test_flag_follows_set_deblock_info(ilf_lib, oracle):
    """One slot, one uploaded picture; side information without, with and again without an intra unit."""
    w, h, ctu_log2 = 264, 200, 6
    rng = np.random.default_rng(41)
    pic = synth.picture(rng, w, h, BD)
    free = synth.deblock_info(rng, w, h, p_intra=0.0, inter=True)
    intra = synth.deblock_info(rng, w, h, p_intra=0.3, inter=True)
    with ilf_lib.InLoopFilter(w, h, BD, BD, ctu_log2) as f:
        f.upload(0, *(pic[k] for k in K))
        for name, (prm, info, mv16) in (("intra-free", free), ("intra", intra), ("intra-free again", free)):
            si = {"db_params": prm, "db_info": info, "db_mv16": mv16}
            _set_db(f, 0, si)
            f.run(0, 1, 1)
            got = f.download(0)
            want = _oracle_deblock(oracle, pic, si, ctu_log2=ctu_log2)
            assert not any(_diff(got, want).values()), name
            assert np.array_equal(want["cb"], pic["cb"]) != _has_intra(si), name


@pytest.mark.parametrize("tree", ["single", "dual"])
@pytest.mark.parametrize("edge", ["vertical", "horizontal"])
def test_single_intra_unit_at_the_end_of_the_scan(edge, tree, ilf_lib, oracle):
    """An intra-free grid with one intra unit on a chroma edge: in the last unit row on the last vertical chroma edge (66 x 50
    units: one of the last 4 units, past the scan's last whole 16-unit block), or in the last unit column on the last
    horizontal chroma edge.  Dual tree: only the chroma layer carries the intra bit (the luma layer has none)."""
    w, h, ctu_log2 = 264, 200, 6
    uw, uh = w // 4, h // 4
    rng = np.random.default_rng(17 if edge == "vertical" else 18)
    pic = synth.picture(rng, w, h, BD)
    prm, info, mv16 = synth.deblock_info(rng, w, h, p_intra=0.0, inter=True)
    r, c = (uh - 1, 4 * ((uw - 1) // 4)) if edge == "vertical" else (4 * ((uh - 1) // 4), uw - 1)
    assert edge == "horizontal" or uw * uh - (r * uw + c) <= (uw * uh) % 16
    pr, pc = (r, c - 1) if edge == "vertical" else (r - 1, c)
    flag = EDGE_V if edge == "vertical" else EDGE_H
    layer = info.copy()
    for (y, x) in ((r, c), (pr, pc)):
        layer[y, x] = (layer[y, x] & ~np.uint32(0xFF00)) | np.uint32(45 << 8)   # a QP whose chroma tc is not 0
    layer[r, c] |= np.uint32(INTRA | flag)
    si = {"db_params": prm, "db_mv16": mv16}
    if tree == "single":
        si["db_info"] = layer
    else:
        si["db_info"], si["db_info_c"] = info, layer
    assert not (si["db_info"] & INTRA).any() or tree == "single"
    want = _oracle_deblock(oracle, pic, si, ctu_log2=ctu_log2)
    assert not np.array_equal(want["cb"], pic["cb"]) or not np.array_equal(want["cr"], pic["cr"]), "the intra unit must filter chroma"
    with ilf_lib.InLoopFilter(w, h, BD, BD, ctu_log2) as f:
        f.upload(0, *(pic[k] for k in K))
        _set_db(f, 0, si)
        f.run(0, 1, 1)
        assert not any(_diff(f.download(0), want).values())


def test_band_with_its_only_intra_unit_in_a_halo_row(ilf_lib, oracle):
    """The only intra unit sits just below the first band's own rows, on the chroma edge between the bands: the first band
    holds it in its halo rows and must still filter the chroma rows above that edge."""
    w, h, ctu_log2, n = 264, 200, 5, 2
    ctu = 1 << ctu_log2
    cw, ch = (w + ctu - 1) // ctu, (h + ctu - 1) // ctu
    rng = np.random.default_rng(29)
    pic = synth.picture(rng, w, h, BD)
    prm, info, mv16 = synth.deblock_info(rng, w, h, p_intra=0.0, inter=True)
    own0, own_rows, _, _ = bands.band_rows(h, ctu_log2, bands.band_partition(ch, n)[0])
    r, c = (own0 + own_rows) // 4, 10   # first unit row below the first band: a halo row of that band
    for y in (r - 1, r):
        info[y, c] = (info[y, c] & ~np.uint32(0xFF00)) | np.uint32(45 << 8)
    info[r, c] |= np.uint32(INTRA | EDGE_H)
    alf_bytes, en = synth.alf_params(rng, cw, ch, is7=True, p_on=0.9)
    si = {"db_params": prm, "db_info": info, "db_mv16": mv16, "sao_ctus": synth.sao_params(rng, cw, ch, BD, p_off=0.1), "alf_params": alf_bytes,
          "alf_ctu_enable": en}
    dbk = oracle.deblock(pic, BD, BD, ctu_log2, prm, info, None, mv16, None, None)
    cy = (own0 + own_rows) // 2
    assert not np.array_equal(dbk["cb"][cy - 1], pic["cb"][cy - 1]) or not np.array_equal(dbk["cr"][cy - 1], pic["cr"][cy - 1])
    whole = _run_whole(ilf_lib, w, h, BD, BD, ctu_log2, pic, si)
    want = oracle.alf(oracle.sao(dbk, BD, BD, ctu_log2, si["sao_ctus"]), BD, BD, ctu_log2, alf_bytes, en)
    assert not any(_diff(whole, want).values()), "whole picture != oracle"
    banded = _run_banded(ilf_lib, w, h, BD, BD, ctu_log2, pic, si, n)
    assert not any(_diff(banded, whole).values()), "banded != whole picture"


def test_skipped_chroma_is_not_moved(ilf_lib, oracle):
    """The deblocking bytes the library counts: luma only (2 B read + 2 B written per luma sample) for pictures without an
    intra unit, all three planes (6 B per luma sample) for a picture with one."""
    d = _ra1080(oracle)
    free = [j for j, si in enumerate(d["side"]) if not _has_intra(si)]
    mixed = [j for j, si in enumerate(d["side"]) if _has_intra(si)]
    px = W1080 * H1080
    for picks, per_picture in ((free, 4.0 * px), (mixed[:1], 6.0 * px)):
        with ilf_lib.InLoopFilter(W1080, H1080, BD, BD, CTU, num_slots=len(picks)) as f:
            for s, j in enumerate(picks):
                f.upload(s, *(d["planes"][j][k] for k in K))
                _set_db(f, s, d["side"][j])
            f.set_timing(True)
            f.run(0, len(picks), 1)
            ms, launches, nbytes = f.kernel_times()["deblock"]
            f.set_timing(False)
            assert launches == 1
            assert nbytes == len(picks) * per_picture, (picks, nbytes)
            for s, j in enumerate(picks):
                assert not any(_diff(f.download(s), d["deblocked"][j]).values()), f"picture {j}"
