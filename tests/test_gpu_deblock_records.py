"""Deblocking from edge records.

ilf_set_deblock_info derives one record per 4-line edge segment (edge flag, bS, no-filter sides, the QP with the slice's beta / tc
offsets and, for chroma, the plane's QP offset and mapping) on the upload stream, and the deblocking kernel reads those records
instead of the unit grid and the motion vectors.  These tests check, sample for sample against the oracle, the cases where the
records could go stale or be misplaced: unlike motion-vector representations and a chroma-tree picture in one launch, a slot whose
side information is replaced, a run issued right after the setter on a lane, slice offsets and edges a slice boundary disables,
band contexts whose records cover halo rows, and picture widths whose last edge column falls on a tile's border."""
import numpy as np
import pytest

import synth
from test_gpu_bands import _run_banded

pytestmark = pytest.mark.gpu
K = ("y", "cb", "cr")
EDGE_V, EDGE_H = 0x04, 0x10


def _diff(got, want):
    return {k: int((got[k] != want[k]).sum()) for k in K}


def _intra_side(rng, w, h):
    """An all-intra picture given without motion vectors (the representation 'none')."""
    prm, info, _ = synth.deblock_info(rng, w, h, p_intra=1.0)
    return {"db_params": prm, "db_info": info}


def _side(rng, w, h, kind, ctu_log2=7):
    if kind == "none":
        return _intra_side(rng, w, h)
    si = synth.deblock_info_stress(rng, w, h, ctu_log2, mv32=kind == "mv32", bd_luma=10, chroma_qp_offset=12)
    if kind != "ctree":
        si.pop("db_info_c")
    return si


def _set_db(f, slot, si):
    f.set_deblock_info(slot, si["db_params"], si["db_info"], si.get("db_info_c"), si.get("db_mv16"), si.get("db_mv32"), si.get("ctu_slice"))


def _oracle(O, pic, si, ctu_log2=7, bd=10):
    return O.deblock(pic, bd, bd, ctu_log2, si["db_params"], si["db_info"], si.get("db_info_c"), si.get("db_mv16"), si.get("db_mv32"), si.get("ctu_slice"))


def test_mixed_representations_and_chroma_tree_in_one_launch(ilf_lib, oracle):
    rng = np.random.default_rng(71)
    w, h = 416, 240
    kinds = ("none", "mv16", "mv32", "ctree", "mv16")
    pics = [synth.picture(rng, w, h) for _ in kinds]
    sides = [_side(rng, w, h, k) for k in kinds]
    with ilf_lib.InLoopFilter(w, h, 10, 10, 7, num_slots=len(kinds)) as f:
        for i, (p, si) in enumerate(zip(pics, sides)):
            f.upload(i, *(p[k] for k in K))
            _set_db(f, i, si)
        n0 = f.launch_count()
        f.run(0, len(kinds), 1)
        assert f.launch_count() - n0 == 1
        for i, (p, si) in enumerate(zip(pics, sides)):
            assert not any(_diff(f.download(i), _oracle(oracle, p, si)).values()), f"slot {i} ({kinds[i]})"


def test_side_information_replaced_between_runs(ilf_lib, oracle):
    """Each setter call replaces the slot's records, also when the motion-vector representation or the chroma-tree layer changes;
    a second run without a new setter call reads the same records again."""
    rng = np.random.default_rng(72)
    w, h = 264, 136
    pic = synth.picture(rng, w, h)
    with ilf_lib.InLoopFilter(w, h, 10, 10, 7) as f:
        f.upload(0, *(pic[k] for k in K))
        for kind in ("mv32", "mv16", "none", "ctree", "mv32"):
            si = _side(rng, w, h, kind)
            _set_db(f, 0, si)
            want = _oracle(oracle, pic, si)
            for _ in range(2):
                f.run(0, 1, 1)
                assert not any(_diff(f.download(0), want).values()), kind


def test_setter_then_run_on_a_lane_without_host_sync(ilf_lib, oracle, monkeypatch):
    """A deblock + SAO chain over a batch large enough for the lanes, issued right after the setters: the lane's launch is ordered
    behind the record pass on the upload stream by the slot's events alone."""
    monkeypatch.setenv("ILF_RUN_LANES", "2")
    monkeypatch.setenv("ILF_RUN_LANE_MIN", "4")
    rng = np.random.default_rng(73)
    w, h, n = 256, 128, 6
    pics = [synth.picture(rng, w, h) for _ in range(n)]
    sao = synth.sao_params(rng, 2, 1, 10, p_off=0.1)
    with ilf_lib.InLoopFilter(w, h, 10, 10, 7, num_slots=n) as f:
        assert f.run_lanes() == 2
        for i in range(n):
            f.upload(i, *(pics[i][k] for k in K))
            f.set_sao_params(i, sao)
        for rnd in range(2):
            sides = [_side(rng, w, h, ("mv16", "mv32", "ctree")[(i + rnd) % 3]) for i in range(n)]
            for i in range(n):
                _set_db(f, i, sides[i])
            f.run(0, n, 3)
            for i in range(n):
                want = oracle.sao(_oracle(oracle, pics[i], sides[i]), 10, 10, 7, sao)
                assert not any(_diff(f.download(i), want).values()), f"round {rnd} slot {i}"


def test_slice_offsets_and_edges_a_slice_boundary_disables(ilf_lib, oracle):
    """Several slices with their own beta / tc offsets, and every edge on a boundary between two slices removed from the grid (a
    slice whose loop filter must not cross it): the records carry each segment's own offsets."""
    rng = np.random.default_rng(74)
    w, h, ctu_log2 = 320, 192, 5
    ctu = 1 << ctu_log2
    cw, ch = w // ctu, h // ctu
    si = synth.deblock_info_stress(rng, w, h, ctu_log2, bd_luma=10)
    prm = np.frombuffer(si["db_params"], synth.DB_DT).copy()
    prm["num_slices"] = 4
    prm["slices"][0, :4, 0] = (-6, 6, 0, 3)
    prm["slices"][0, :4, 1] = (6, -6, 2, -3)
    si["db_params"] = prm.tobytes()
    ctu_slice = np.repeat(np.arange(4, dtype=np.uint8), (cw * ch + 3) // 4)[:cw * ch]
    si["ctu_slice"] = ctu_slice
    sl = ctu_slice.reshape(ch, cw)
    uy, ux = np.mgrid[0:h // 4, 0:w // 4]
    own = sl[(uy * 4) >> ctu_log2, (ux * 4) >> ctu_log2]
    left = sl[(uy * 4) >> ctu_log2, np.maximum(ux * 4 - 4, 0) >> ctu_log2]
    above = sl[np.maximum(uy * 4 - 4, 0) >> ctu_log2, (ux * 4) >> ctu_log2]
    for layer in ("db_info", "db_info_c"):
        g = si[layer].copy()
        g[own != left] &= ~np.uint32(EDGE_V | 0x08)
        g[own != above] &= ~np.uint32(EDGE_H | 0x20)
        si[layer] = g
    pic = synth.picture(rng, w, h)
    with ilf_lib.InLoopFilter(w, h, 10, 10, ctu_log2) as f:
        f.upload(0, *(pic[k] for k in K))
        _set_db(f, 0, si)
        f.run(0, 1, 1)
        assert not any(_diff(f.download(0), _oracle(oracle, pic, si, ctu_log2)).values())


def test_band_contexts_records_across_the_halo(ilf_lib, oracle):
    """A picture in three CTU-row bands: each context derives the records of its held rows, halo rows included, with slices looked
    up at full-picture rows; the stitched result is the whole picture's."""
    rng = np.random.default_rng(75)
    w, h, ctu_log2 = 264, 200, 5
    ctu = 1 << ctu_log2
    cw, ch = (w + ctu - 1) // ctu, (h + ctu - 1) // ctu
    si = synth.deblock_info_stress(rng, w, h, ctu_log2, bd_luma=10)
    si["sao_ctus"] = synth.sao_params(rng, cw, ch, 10, p_off=0.1)
    si["alf_params"], si["alf_ctu_enable"] = synth.alf_params(rng, cw, ch, is7=True, p_on=0.9)
    pic = synth.picture(rng, w, h)
    got = _run_banded(ilf_lib, w, h, 10, 10, ctu_log2, pic, si, 3)
    want = _oracle(oracle, pic, si, ctu_log2)
    want = oracle.sao(want, 10, 10, ctu_log2, si["sao_ctus"])
    want = oracle.alf(want, 10, 10, ctu_log2, si["alf_params"], si["alf_ctu_enable"])
    assert not any(_diff(got, want).values())


@pytest.mark.parametrize("w,h", [(120, 40), (136, 72), (248, 24), (264, 264), (392, 56), (1032, 48)])
@pytest.mark.parametrize("kind", ["mv16", "mv32", "ctree"])
def test_widths_around_the_tile_edge(w, h, kind, ilf_lib, oracle):
    """Widths of 128 k +- 8 (the record arrays' last edge column W / 8 is the tile's edge 16 or its edge 15) and chroma widths
    that are not a multiple of 8 (W / 16 + 1 chroma edge columns)."""
    rng = np.random.default_rng(w * 1000 + h)
    si = _side(rng, w, h, kind)
    pic = synth.picture(rng, w, h)
    with ilf_lib.InLoopFilter(w, h, 10, 10, 7) as f:
        f.upload(0, *(pic[k] for k in K))
        _set_db(f, 0, si)
        f.run(0, 1, 1)
        assert not any(_diff(f.download(0), _oracle(oracle, pic, si)).values())
