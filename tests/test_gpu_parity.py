"""CUDA path (through the C ABI) vs the reference's captured output and vs the oracle.  Bit-exact."""
import os

import numpy as np
import pytest

import golden_io as G

pytestmark = pytest.mark.gpu
K = G.K


def _ctx(v, c, **kw):
    g = c["geom"]
    return v.InLoopFilter(g["width"], g["height"], g["bd_luma"], g["bd_chroma"], g["ctu_log2"], **kw)


def _set_all(f, slot, c):
    mv = c["db_mv32"]
    fits = np.abs(mv).max(initial=0) < 32768
    f.set_deblock_info(slot, c["db_params"].tobytes(), c["db_info"], c.get("db_info_c"),
                       mv.astype(np.int16) if fits else None, None if fits else mv, c["ctu_slice"])
    if "sao_ctus" in c:
        f.set_sao_params(slot, c["sao_ctus"])
    if "alf_params" in c:
        f.set_alf_params(slot, c["alf_params"].tobytes(), c["alf_ctu_enable"])


def _diff(a, b):
    return {k: int((a[k] != b[k]).sum()) for k in K}


@pytest.mark.parametrize("path", G.golden_files(), ids=os.path.basename)
def test_each_stage_matches_reference_capture(path, ilf_lib):
    """Each stage alone, fed with the reference's own input of that stage."""
    c = G.load_golden(path)
    with _ctx(ilf_lib, c) as f:
        for stage, src in G.stage_inputs(c).items():
            f.upload(0, *(c[f"{src}_{k}"] for k in K))
            _set_all(f, 0, c)
            {"dbk": f.loop_filter_pic, "sao": f.sao_process, "alf": f.alf_process}[stage](0)
            out = f.download(0)
            d = _diff(out, {k: c[f"{stage}_{k}"] for k in K})
            assert not any(d.values()), f"{stage}: mismatching samples {d}"


@pytest.mark.parametrize("path", G.golden_files(), ids=os.path.basename)
def test_chain_matches_reference_capture(path, ilf_lib):
    """deblock -> SAO -> ALF in one ilf_run, device-resident between the stages."""
    c = G.load_golden(path)
    last = [s for s in ("dbk", "sao", "alf") if f"{s}_y" in c][-1]
    with _ctx(ilf_lib, c) as f:
        f.upload(0, *(c[f"pre_{k}"] for k in K))
        _set_all(f, 0, c)
        stages = 1 | (2 if "sao_y" in c else 0) | (4 if "alf_y" in c else 0)
        f.run(0, 1, stages)
        out = f.download(0)
        assert not any(_diff(out, {k: c[f"{last}_{k}"] for k in K}).values())
        f.run(0, 1, stages)                       # the uploaded input is preserved: a second run gives the same
        out2 = f.download(0)
        assert not any(_diff(out, out2).values())


def test_mv32_path_equals_mv16_path(ilf_lib):
    c = G.load_golden([p for p in G.golden_files() if "ra_416x240_05" in p][0])
    res = []
    with _ctx(ilf_lib, c) as f:
        for use32 in (False, True):
            f.upload(0, *(c[f"pre_{k}"] for k in K))
            mv = c["db_mv32"]
            f.set_deblock_info(0, c["db_params"].tobytes(), c["db_info"], c.get("db_info_c"), None if use32 else mv.astype(np.int16), mv if use32 else None, c["ctu_slice"])
            f.loop_filter_pic(0)
            res.append(f.download(0))
    assert not any(_diff(res[0], res[1]).values())
    assert not any(_diff(res[0], {k: c[f"dbk_{k}"] for k in K}).values())


def test_alf_classification_matches_oracle(ilf_lib, oracle):
    c = G.load_golden(G.golden_files()[0])
    with _ctx(ilf_lib, c) as f:
        f.upload(0, *(c[f"sao_{k}"] for k in K))
        got = f.alf_classify(0)
    want = oracle.alf_classify(c["sao_y"], c["geom"]["bd_luma"])
    assert np.array_equal(got, want)


def test_batched_slots(ilf_lib):
    """Several pictures of one geometry in one batched launch per stage."""
    caps = [G.load_golden(p) for p in G.golden_files() if "ra_416x240" in p and not p.endswith("_00.npz")]
    with _ctx(ilf_lib, caps[0], num_slots=len(caps)) as f:
        for i, c in enumerate(caps):
            f.upload(i, *(c[f"pre_{k}"] for k in K))
            _set_all(f, i, c)
        f.run(0, len(caps), 7)
        for i, c in enumerate(caps):
            assert not any(_diff(f.download(i), {k: c[f"alf_{k}"] for k in K}).values()), f"slot {i}"
        assert 1 <= f.launch_count() <= 4    # planes whose stage is off in every picture of the batch are not launched


def test_chain_dealt_to_lanes(ilf_lib, monkeypatch):
    """A chain over a batch at or above the lane threshold is dealt to several compute streams (ilf_run, ILF_RUN_LANES): every
    slot still gets the reference result, also when the grouping changes between runs (a slot moves to another lane), when a
    single-stage run on the compute stream follows, and for the picture hash taken on the compute stream afterwards."""
    monkeypatch.setenv("ILF_RUN_LANES", "3")
    monkeypatch.setenv("ILF_RUN_LANE_MIN", "4")
    caps = [G.load_golden(p) for p in G.golden_files() if "ra_416x240" in p]
    n = 7
    with _ctx(ilf_lib, caps[0], num_slots=n) as f:
        for i in range(n):
            c = caps[i % len(caps)]
            f.upload(i, *(c[f"pre_{k}"] for k in K))
            _set_all(f, i, c)
        for first, cnt in ((0, n), (1, 6), (0, 5), (2, 4)):     # different groupings: slots change lanes between runs
            f.run(first, cnt, 7)
        f.run(0, n, 1)          # single stage: compute stream only, ordered after the lanes
        f.run(0, n, 6)          # SAO + ALF as a chain on the lanes again
        for i in range(n):
            c = caps[i % len(caps)]
            assert not any(_diff(f.download(i), {k: c[f"alf_{k}"] for k in K}).values()), f"slot {i}"
        f.run(0, n, 7)
        crc = f.picture_hash(n - 1, "crc")
        c = caps[(n - 1) % len(caps)]
        with _ctx(ilf_lib, c) as g1:
            g1.upload(0, *(c[f"pre_{k}"] for k in K))
            _set_all(g1, 0, c)
            g1.run(0, 1, 7)
            assert list(crc) == list(g1.picture_hash(0, "crc"))


def test_batch_with_mixed_motion_vector_representations(ilf_lib):
    """One ilf_run over an intra picture given without motion vectors, a picture with int16 and one with int32 vectors: the library
    launches the deblocking kernel once per representation present in the batch."""
    caps = [G.load_golden(p) for p in G.golden_files() if os.path.basename(p) in ("ra_416x240_00.npz", "ra_416x240_01.npz", "ra_416x240_05.npz")]
    assert len(caps) == 3
    with _ctx(ilf_lib, caps[0], num_slots=3) as f:
        for i, c in enumerate(caps):
            f.upload(i, *(c[f"pre_{k}"] for k in K))
            mv = c["db_mv32"]
            mv16, mv32 = (None, None) if i == 0 else ((mv.astype(np.int16), None) if i == 1 else (None, mv))
            if i == 0:
                assert (c["db_info"] & 1).all()          # every unit of the I picture is intra: its motion arrays are never read
            f.set_deblock_info(i, c["db_params"].tobytes(), c["db_info"], c.get("db_info_c"), mv16, mv32, c["ctu_slice"])
            f.set_sao_params(i, c["sao_ctus"])
            f.set_alf_params(i, c["alf_params"].tobytes(), c["alf_ctu_enable"])
        f.run(0, 3, 7)
        for i, c in enumerate(caps):
            assert not any(_diff(f.download(i), {k: c[f"alf_{k}"] for k in K}).values()), f"slot {i}"


def test_run_with_missing_side_information_launches_nothing(ilf_lib):
    """ilf_run validates every stage of every slot first: a slot without SAO parameters fails the call before any kernel runs, and the
    slots' state is untouched (the next complete run gives the reference result)."""
    c = G.load_golden([p for p in G.golden_files() if "ra_416x240_01" in p][0])
    with _ctx(ilf_lib, c, num_slots=2) as f:
        for i in range(2):
            f.upload(i, *(c[f"pre_{k}"] for k in K))
            f.set_deblock_info(i, c["db_params"].tobytes(), c["db_info"], c.get("db_info_c"), c["db_mv32"].astype(np.int16), None, c["ctu_slice"])
            f.set_alf_params(i, c["alf_params"].tobytes(), c["alf_ctu_enable"])
        f.set_sao_params(0, c["sao_ctus"])
        n0 = f.launch_count()
        with pytest.raises(ilf_lib.IlfError):
            f.run(0, 2, 7)
        assert f.launch_count() == n0
        f.set_sao_params(1, c["sao_ctus"])
        f.run(0, 2, 7)
        for i in range(2):
            assert not any(_diff(f.download(i), {k: c[f"alf_{k}"] for k in K}).values())
