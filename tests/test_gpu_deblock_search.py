"""Deblocking offset search on the GPU (ilf_deblock_search; EncGOP::applyDeblockingFilterParameterSelection): the sums of
((D_k - O)^2 >> shift) per candidate and plane must equal the oracle's deblocking with every slice's offsets replaced by the
candidate's, sample for sample -- and the reference's own deblocked picture must score exactly 0 under its own offsets."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import golden_io as G
import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (side information and synthetic planes of the benchmark workloads)

pytestmark = pytest.mark.gpu
K = ("y", "cb", "cr")
GRID = [(b, t) for b in range(-3, 4) for t in range(-3, 4)]
CANDS = GRID + [(6, 6), (6, -6), (-6, 6), (-6, -6)]
ERR_ARG, ERR_STATE = -1, -3


def with_offsets(params_bytes, beta, tc):
    """ilf_deblock_params with beta_offset_div2 / tc_offset_div2 of every slice entry replaced (bytes 16 + 4 i and 17 + 4 i)."""
    pb = bytearray(bytes(params_bytes))
    for i in range(64):
        pb[16 + 4 * i] = beta & 0xFF
        pb[17 + 4 * i] = tc & 0xFF
    return bytes(pb)


def distortion(pic, org, shift):
    return np.array([int(((pic[k].astype(np.int64) - org[k]) ** 2 >> shift[c > 0]).sum()) for c, k in enumerate(K)], np.uint64)


def oracle_search(O, pic, org, bd_l, bd_c, ctu_log2, params_bytes, info, info_c, mv16, mv32, ctu_slice, candidates, shifts):
    """{shift: uint64 [K, 3]}: the oracle's deblocking once per candidate, the distortion in numpy int64."""
    out = {s: np.zeros((len(candidates), 3), np.uint64) for s in shifts}
    for k, (b, t) in enumerate(candidates):
        d = O.deblock(pic, bd_l, bd_c, ctu_log2, with_offsets(params_bytes, b, t), info, info_c, mv16, mv32, ctu_slice)
        for s in shifts:
            out[s][k] = distortion(d, org, s)
    return out


def _org_of(rng, pic, bd, bd_chroma=None):
    """The picture plus noise, each plane clipped to its own range (luma `bd`, chroma `bd_chroma`, default `bd`)."""
    bds = dict(zip(K, (bd,) + 2 * (bd if bd_chroma is None else bd_chroma,)))
    return {k: np.clip(pic[k].astype(np.int32) + rng.integers(-12, 13, pic[k].shape), 0, (1 << bds[k]) - 1).astype(np.int16) for k in K}


def _mv(c):
    mv = c["db_mv32"]
    return (mv.astype(np.int16), None) if np.abs(mv).max(initial=0) < 32768 else (None, mv)


def _capture_ctx(v, c, **kw):
    g = c["geom"]
    return v.InLoopFilter(g["width"], g["height"], g["bd_luma"], g["bd_chroma"], g["ctu_log2"], **kw)


def _load_capture(f, slot, c, org):
    mv16, mv32 = _mv(c)
    f.upload(slot, *(c[f"pre_{k}"] for k in K))
    f.set_deblock_info(slot, c["db_params"].tobytes(), c["db_info"], c.get("db_info_c"), mv16, mv32, c["ctu_slice"])
    f.set_original(slot, org["y"], org["cb"], org["cr"], np.zeros(f.ctus_w * f.ctus_h, np.uint8))


def _own_offsets(c):
    prm = np.frombuffer(c["db_params"].tobytes(), synth.DB_DT)[0]
    off = {(int(s[0]), int(s[1])) for s in prm["slices"][:prm["num_slices"]]}
    assert len(off) == 1, "the captures' slices share their offsets"
    return off.pop()


@pytest.mark.parametrize("path", G.golden_files(), ids=os.path.basename)
def test_reference_offsets_score_zero_against_reference_output(path, ilf_lib):
    """The reference's deblocked picture as the original: its own offsets give 0 in every plane, the neighbours do not."""
    c = G.load_golden(path)
    b, t = _own_offsets(c)
    cands = [(b, t), (b + 1, t), (b - 1, t), (b, t + 1), (b, t - 1)]
    with _capture_ctx(ilf_lib, c) as f:
        _load_capture(f, 0, c, {k: c[f"dbk_{k}"] for k in K})
        f.deblock_search(cands)
        got = f.get_deblock_search(0)
    assert got.shape == (5, 3)
    assert not got[0].any(), f"own offsets ({b}, {t}): {got[0]}"
    # beta +-1 always changes a decision somewhere; tc +-1 can land on a flat step of the tc table on one side, not on both
    assert got[1].sum() > 0 and got[2].sum() > 0, f"a beta neighbour of ({b}, {t}) gives the reference's picture exactly: {got}"
    assert got[3].sum() + got[4].sum() > 0, f"both tc neighbours of ({b}, {t}) give the reference's picture exactly: {got}"


@pytest.mark.parametrize("path", G.golden_files(), ids=os.path.basename)
def test_captures_equal_oracle(path, ilf_lib, oracle):
    """Every capture (I/P/B, dual tree, three slices with chroma QP offsets), 53 candidates, shifts (0, 0) and (4, 4)."""
    c = G.load_golden(path)
    g = c["geom"]
    pic = {k: c[f"pre_{k}"] for k in K}
    org = _org_of(np.random.default_rng(len(path)), pic, g["bd_luma"])
    mv16, mv32 = _mv(c)
    want = oracle_search(oracle, pic, org, g["bd_luma"], g["bd_chroma"], g["ctu_log2"], c["db_params"].tobytes(), c["db_info"], c.get("db_info_c"),
                         mv16, mv32, c["ctu_slice"], CANDS, [(0, 0), (4, 4)])
    with _capture_ctx(ilf_lib, c) as f:
        _load_capture(f, 0, c, org)
        for s in ((0, 0), (4, 4)):
            f.deblock_search(CANDS, s)
            got = f.get_deblock_search(0)
            bad = np.argwhere(got != want[s])
            assert bad.size == 0, f"shift {s}: first mismatch (candidate, plane) {bad[0]}: got {got[tuple(bad[0])]} want {want[s][tuple(bad[0])]}"


# odd sizes (width / 2 not a multiple of 8, partial CTUs and tiles), every CTU size and bit depth, none / int16 / int32 motion, three
# slices with their own base offsets (the candidate must override all of them) and the whole QP range.  The cases at two bit depths
# also draw the negative QPs of their luma depth and chroma QP offsets up to +-12 (the cases at one depth keep their draws).
@pytest.mark.parametrize("w,h,bd_luma,bd_chroma,ctu_log2,mv,seed",
                         synth.keep_ids([(200, 136, 8, 5, "mv16", 1), (264, 72, 10, 6, "none", 2), (136, 264, 12, 7, "mv32", 3),
                                         (392, 72, 10, 6, "mv16", 4), (520, 392, 10, 7, "mv32", 5), (16, 16, 10, 5, "none", 6)],
                                        lambda w, h, bd, c, mv, s: (w, h, bd, bd, c, mv, s)) +
                         [(200, 136, 8, 12, 5, "mv16", 7), (264, 72, 12, 10, 6, "none", 8), (520, 392, 12, 10, 7, "mv32", 9)])
def test_synthetic_matrix_equals_oracle(w, h, bd_luma, bd_chroma, ctu_log2, mv, seed, ilf_lib, oracle):
    rng = np.random.default_rng(seed)
    pic = synth.picture(rng, w, h, bd_luma, "mix", bd_chroma=bd_chroma)
    org = _org_of(rng, pic, bd_luma, bd_chroma)
    wide = {} if bd_luma == bd_chroma else {"bd_luma": bd_luma, "chroma_qp_offset": 12}
    si = synth.deblock_info_stress(rng, w, h, ctu_log2, mv == "mv32", **wide)
    mv16, mv32 = (si.get("db_mv16"), si.get("db_mv32")) if mv != "none" else (None, None)
    cands = [(0, 0), (3, -2), (-4, 5), (6, 6), (-128, 127), (127, -128), (20, -20), (-1, 1)]
    shifts = [(0, 0), (2, 3), (0, 4), (4, 0)]
    want = oracle_search(oracle, pic, org, bd_luma, bd_chroma, ctu_log2, si["db_params"], si["db_info"], si["db_info_c"], mv16, mv32, si["ctu_slice"], cands, shifts)
    with ilf_lib.InLoopFilter(w, h, bd_luma, bd_chroma, ctu_log2) as f:
        f.upload(0, *(pic[k] for k in K))
        f.set_deblock_info(0, si["db_params"], si["db_info"], si["db_info_c"], mv16, mv32, si["ctu_slice"])
        f.set_original(0, org["y"], org["cb"], org["cr"], np.zeros(f.ctus_w * f.ctus_h, np.uint8))
        for s in shifts:
            f.deblock_search(cands, s)
            assert np.array_equal(f.get_deblock_search(0), want[s]), f"shift {s}"
    if w * h > 16 * 16:
        assert len({tuple(r) for r in want[(0, 0)]}) > 1, "the candidates must matter in this picture"


def _motion(si, mode):
    """(mv16, mv32) of the stream's int16 motion given as int16, as int32, or not at all (an all-intra picture needs none)."""
    mv16 = si.get("db_mv16")
    return {"mv16": (mv16, None), "mv32": (None, None if mv16 is None else mv16.astype(np.int32)), "none": (None, None)}[mode]


def _set_4k(f, slot, si, params=None, mode="mv16"):
    f.set_deblock_info(slot, params or si["db_params"].tobytes(), si["db_info"], si.get("db_info_c"), *_motion(si, mode), si.get("ctu_slice"))


def test_4k_batch_equals_deblock_download_and_oracle(ilf_lib, oracle):
    """Three resident 4K pictures with the random-access stream's side information (int16 motion, int32 motion, the intra picture
    with a chroma-tree layer and no motion): one search over 49 candidates == per candidate, the offsets rewritten, ilf_deblock,
    download and the distortion in numpy; two candidates also == the oracle."""
    w, h = 3840, 2160
    side = bench.load_sideinfo("ra_4k")
    sis = [side[3], side[6], side[0]]
    modes = ["mv16", "mv32", "none"]
    assert not (sis[2]["db_info"] & 0x80).any() and (sis[2]["db_info"] & 1).all(), "picture 0 is the intra picture"
    planes = bench.synth_planes(w, h, 3, seed=321)
    rng = np.random.default_rng(5)
    pics = [dict(zip(K, p)) for p in planes]
    orgs = [_org_of(rng, p, 10) for p in pics]
    shift = (0, 1)
    with ilf_lib.InLoopFilter(w, h, 10, 10, 7, num_slots=3) as f:
        for j in range(3):
            f.upload(j, *planes[j])
            _set_4k(f, j, sis[j], mode=modes[j])
            f.set_original(j, orgs[j]["y"], orgs[j]["cb"], orgs[j]["cr"], np.zeros(f.ctus_w * f.ctus_h, np.uint8))
        f.deblock_search(GRID, shift, 0, 3)
        got = [f.get_deblock_search(j) for j in range(3)]
        for j in range(3):
            for k, (b, t) in enumerate(GRID):
                _set_4k(f, j, sis[j], with_offsets(sis[j]["db_params"].tobytes(), b, t), modes[j])
                f.loop_filter_pic(j)
                want = distortion(f.download(j), orgs[j], shift)
                assert np.array_equal(got[j][k], want), f"slot {j} candidate {(b, t)}: {got[j][k]} != {want}"
    for j in range(3):
        si = sis[j]
        want = oracle_search(oracle, pics[j], orgs[j], 10, 10, 7, si["db_params"].tobytes(), si["db_info"], si.get("db_info_c"), *_motion(si, modes[j]),
                             si.get("ctu_slice"), [(2, -1), (-3, 3)], [shift])[shift]
        assert np.array_equal(got[j][[GRID.index((2, -1)), GRID.index((-3, 3))]], want), f"slot {j} vs oracle"


def test_8k_intra_equals_oracle(ilf_lib, oracle):
    w, h = 7680, 4320
    si = bench.load_sideinfo("intra_8k")[0]
    pic = dict(zip(K, bench.synth_planes(w, h, 1, seed=8001)[0]))
    org = _org_of(np.random.default_rng(8), pic, 10)
    with ilf_lib.InLoopFilter(w, h, 10, 10, 7) as f:
        f.upload(0, *(pic[k] for k in K))
        _set_4k(f, 0, si)
        f.set_original(0, org["y"], org["cb"], org["cr"], np.zeros(f.ctus_w * f.ctus_h, np.uint8))
        f.deblock_search([(1, -2)], (1, 1))
        got = f.get_deblock_search(0)
    want = oracle_search(oracle, pic, org, 10, 10, 7, si["db_params"].tobytes(), si["db_info"], si.get("db_info_c"), si.get("db_mv16"), None,
                         si.get("ctu_slice"), [(1, -2)], [(1, 1)])[(1, 1)]
    assert np.array_equal(got, want)


def _capture(name):
    return G.load_golden([p for p in G.golden_files() if name in p][0])


def test_search_leaves_the_slot_state_alone(ilf_lib):
    """A search writes no plane: run(ALL) + download after it equals the same picture without the search; a search after a run
    still scores the uploaded picture; a batch equals its slots searched one by one."""
    c = _capture("ra_416x240_05")
    org = _org_of(np.random.default_rng(3), {k: c[f"pre_{k}"] for k in K}, 10)
    with _capture_ctx(ilf_lib, c, num_slots=3) as f:
        for j in range(3):
            _load_capture(f, j, c, org)
            f.set_sao_params(j, c["sao_ctus"])
            f.set_alf_params(j, c["alf_params"].tobytes(), c["alf_ctu_enable"])
        f.deblock_search(CANDS, (0, 0), 0, 1)
        first = f.get_deblock_search(0)
        f.run(0, 2, 7)
        a, b = f.download(0), f.download(1)
        for k in K:
            assert np.array_equal(a[k], b[k]), f"plane {k}: the search changed what the chain gives"
        assert np.array_equal(a["y"], c["alf_y"])
        f.deblock_search(CANDS, (0, 0), 0, 1)   # after run(ALL): the current buffers hold the ALF output, the search reads the upload
        assert np.array_equal(f.get_deblock_search(0), first)
        a2 = f.download(0)
        assert all(np.array_equal(a[k], a2[k]) for k in K), "download after a search differs"
        f.deblock_search(CANDS[:9], (3, 2), 0, 3)
        batch = [f.get_deblock_search(j) for j in range(3)]
        for j in range(3):
            f.deblock_search(CANDS[:9], (3, 2), j, 1)
            assert np.array_equal(f.get_deblock_search(j), batch[j]), f"slot {j}"


def test_errors(ilf_lib):
    c = _capture("ldp_416x240_04")
    org = {k: c[f"dbk_{k}"] for k in K}
    lib = ilf_lib.load_library()
    cand = (C.c_int8 * 2)(0, 0)
    shift = (C.c_int32 * 2)(0, 0)
    out = (C.c_uint64 * (3 * 64))()
    with _capture_ctx(ilf_lib, c, num_slots=2) as f:
        h = f._h
        # state: no upload, no side information, no original since the upload
        assert lib.ilf_deblock_search(h, 0, 1, cand, 1, shift) == ERR_STATE
        assert lib.ilf_get_deblock_search(h, 0, out, 64) == ERR_STATE
        f.upload(0, *(c[f"pre_{k}"] for k in K))
        assert lib.ilf_deblock_search(h, 0, 1, cand, 1, shift) == ERR_STATE
        mv16, mv32 = _mv(c)
        f.set_deblock_info(0, c["db_params"].tobytes(), c["db_info"], c.get("db_info_c"), mv16, mv32, c["ctu_slice"])
        assert lib.ilf_deblock_search(h, 0, 1, cand, 1, shift) == ERR_STATE
        f.set_original(0, org["y"], org["cb"], org["cr"], np.zeros(f.ctus_w * f.ctus_h, np.uint8))
        f.upload(0, *(c[f"pre_{k}"] for k in K))      # a new picture: side information and original are needed again
        f.set_deblock_info(0, c["db_params"].tobytes(), c["db_info"], c.get("db_info_c"), mv16, mv32, c["ctu_slice"])
        assert lib.ilf_deblock_search(h, 0, 1, cand, 1, shift) == ERR_STATE
        f.set_original(0, org["y"], org["cb"], org["cr"], np.zeros(f.ctus_w * f.ctus_h, np.uint8))
        assert lib.ilf_deblock_search(h, 0, 2, cand, 1, shift) == ERR_STATE     # slot 1 has nothing
        # arguments
        cands64 = (C.c_int8 * 130)()
        assert lib.ilf_deblock_search(h, -1, 1, cand, 1, shift) == ERR_ARG
        assert lib.ilf_deblock_search(h, 0, 0, cand, 1, shift) == ERR_ARG
        assert lib.ilf_deblock_search(h, 1, 2, cand, 1, shift) == ERR_ARG
        assert lib.ilf_deblock_search(h, 0, 1, None, 1, shift) == ERR_ARG
        assert lib.ilf_deblock_search(h, 0, 1, cand, 1, None) == ERR_ARG
        assert lib.ilf_deblock_search(h, 0, 1, cand, 0, shift) == ERR_ARG
        assert lib.ilf_deblock_search(h, 0, 1, cands64, 65, shift) == ERR_ARG
        for bad in ((-1, 0), (0, 32), (32, 0), (0, -1)):
            assert lib.ilf_deblock_search(h, 0, 1, cand, 1, (C.c_int32 * 2)(*bad)) == ERR_ARG, bad
        assert lib.ilf_deblock_search(None, 0, 1, cand, 1, shift) == ERR_ARG
        with pytest.raises(ilf_lib.IlfError):
            f.deblock_search([(200, 0)])
        # the limits are accepted: 64 candidates, shift 31
        assert lib.ilf_deblock_search(h, 0, 1, cands64, 64, (C.c_int32 * 2)(31, 31)) == 0
        assert lib.ilf_get_deblock_search(h, 0, out, 63) == ERR_ARG
        assert lib.ilf_get_deblock_search(h, 0, None, 64) == ERR_ARG
        assert lib.ilf_get_deblock_search(h, 2, out, 64) == ERR_ARG
        assert lib.ilf_get_deblock_search(h, 0, out, 64) == 64
        assert lib.ilf_get_deblock_search(h, 1, out, 64) == ERR_STATE
        f.deblock_search([(0, 0)])
        assert lib.ilf_get_deblock_search(h, 0, out, 1) == 1
        assert not any(out[:3]), "the capture's own output scores 0 under its own offsets"
    # band contexts: the message of the statistics entry points
    g = c["geom"]
    with ilf_lib.InLoopFilter(g["width"], g["height"], 10, 10, 7, band=(0, 1)) as f:
        assert lib.ilf_deblock_search(f._h, 0, 1, cand, 1, shift) == ERR_STATE
        assert b"not available on band contexts" in lib.ilf_last_error(f._h)
