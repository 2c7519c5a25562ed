"""Picture geometry at the edges of the kernels' tiles, bands, segments and batch chunks.

Every kernel walks a picture in fixed pieces: deblocking in tiles of 128 x 32 luma (64 x 16 chroma) drawn from a queue, SAO in
bands of 32 rows cut into tiles of 128 samples, ALF in bands of 32 rows cut into tiles of 64 samples, the statistics, hash and
search kernels on grids of their own.  A band walk is cut into horizontal segments whose number follows the number of bands in
the launch, and a launch covers at most 128 slots.  The cases here put every stage and every reader of a slot at each residue of
those pieces, at pictures smaller than one piece and at the most elongated pictures the library accepts, and move the segment
and chunk borders through the same pictures -- each bit-exact against the oracle.  The tests without the gpu mark pin what the
matrix covers, so that a later edit cannot shrink it quietly."""
import ctypes as C
import os

import numpy as np
import pytest

import synth

K = ("y", "cb", "cr")
INTRA = 0x01                                  # ILF_BI_INTRA
MAX_SIZE = 16384                              # ilf_create's limit on either side
SEARCH_CANDS = [(0, 0), (2, -3), (-5, 4), (-128, 127), (127, -128), (20, -20)]   # the last three clamp the beta / tc index


def _residue_cases(base, h0, phase):
    """One picture per width residue mod 128 (every multiple of 8).  Height residue mod 32 and CTU size are dealt so that the
    first twelve residues meet every (height residue, CTU size) pair; the height adds 32 on every other group of four."""
    return [(base + r, h0 + 8 * (i % 4) + 32 * ((i // 4) % 2), 5 + (i + phase) % 3) for i, r in enumerate(range(0, 128, 8))]


GEOMS = (_residue_cases(256, 128, 0) + _residue_cases(128, 64, 1) +
         # whole CTUs in both directions at CTU 64 and 128 (the residue cases have them at CTU 32)
         [(192, 128, 6), (256, 256, 7)] +
         # narrower than one tile of every kernel: chroma 4 .. 28 samples, fewer rows than a deblocking band plus its shift and
         # fewer than an ALF band plus its halo
         [(8, 8, 5), (16, 16, 6), (24, 24, 7), (32, 16, 5), (40, 8, 6), (56, 24, 7), (8, 24, 6), (24, 8, 5)] +
         # elongated; 16384 x 16 is the widest picture accepted (128 deblocking tiles per row, 256 ALF tiles); 1032 and 1000 rows
         # cut the staging copies into chunks of odd row counts
         [(8, 2048, 5), (16, 4096, 6), (4096, 8, 7), (16384, 16, 5), (24, 1032, 6), (40, 1000, 7)])
LARGEST = (MAX_SIZE, MAX_SIZE, 7)             # the largest deblocking tile id (tx 127, band 512); opt-in, see test_largest_picture

BDS = [(8, 8), (10, 10), (12, 12), (10, 8), (8, 12), (12, 10)]
MVS = ["none", "mv16", "mv32"]


def plan(i):
    """Content of case i: (bd_luma, bd_chroma, motion, chroma-tree layer, 7x7 luma filter, ALF arithmetic path)."""
    bl, bc = BDS[i % 6]
    return bl, bc, MVS[(i // 2) % 3], (i // 3) % 2 == 0, (i // 4) % 2 == 0, ("dot", "big")[(i // 5) % 2]


def _ctus(w, h, ctu_log2):
    ctu = 1 << ctu_log2
    return (w + ctu - 1) // ctu, (h + ctu - 1) // ctu


def _avail(rng, w, h, ctu_log2):
    """Random ILF_AVAIL_L / _A / _AL flags of the statistics, never across the picture's left and top border."""
    cw, ch = _ctus(w, h, ctu_log2)
    av = rng.integers(0, 256, cw * ch).astype(np.uint8)
    av[np.arange(cw * ch) % cw == 0] &= ~np.uint8(0x01 | 0x10)
    av[:cw] &= ~np.uint8(0x04 | 0x10)
    return av


def inputs(seed, w, h, ctu_log2, bl, bc, mv, ctree, is7, alf_kind):
    """Seeded planes, original and side information of every stage (the stress layers of deblocking)."""
    rng = np.random.default_rng(seed)
    pic = synth.picture(rng, w, h, bl, "mix", bd_chroma=bc)
    org = {k: np.clip(pic[k].astype(np.int32) + rng.integers(-12, 13, pic[k].shape), 0, (1 << (bl if k == "y" else bc)) - 1).astype(np.int16) for k in K}
    si = synth.deblock_info_stress(rng, w, h, ctu_log2, mv == "mv32", bd_luma=bl, chroma_qp_offset=12)
    si["db_mv16"], si["db_mv32"] = si.get("db_mv16") if mv == "mv16" else None, si.get("db_mv32") if mv == "mv32" else None
    if not ctree:
        si["db_info_c"] = None
    cw, ch = _ctus(w, h, ctu_log2)
    si["sao_ctus"] = synth.sao_params(rng, cw, ch, bl, p_off=0.2, bd_chroma=bc)
    si["alf_params"], si["alf_ctu_enable"] = synth.alf_params(rng, cw, ch, is7, p_on=0.8, big=alf_kind == "big", dot=alf_kind == "dot")
    si["avail"] = _avail(rng, w, h, ctu_log2)
    return pic, org, si


def case_inputs(i):
    w, h, c = GEOMS[i]
    return inputs(1000 + i, w, h, c, *plan(i))


def _db_args(si):
    return si["db_params"], si["db_info"], si["db_info_c"], si["db_mv16"], si["db_mv32"], si["ctu_slice"]


def oracle_chain(O, pic, bl, bc, ctu_log2, si):
    d = O.deblock(pic, bl, bc, ctu_log2, *_db_args(si))
    d = O.sao(d, bl, bc, ctu_log2, si["sao_ctus"])
    return O.alf(d, bl, bc, ctu_log2, si["alf_params"], si["alf_ctu_enable"])


def load(f, slot, pic, org, si):
    f.upload(slot, *(pic[k] for k in K))
    f.set_deblock_info(slot, *_db_args(si))
    f.set_sao_params(slot, si["sao_ctus"])
    f.set_alf_params(slot, si["alf_params"], si["alf_ctu_enable"])
    f.set_original(slot, org["y"], org["cb"], org["cr"], si["avail"])


def _diff(got, want):
    """Mismatching samples per plane, planes that match left out."""
    d = {k: int((got[k] != want[k]).sum()) for k in K}
    return {k: v for k, v in d.items() if v}


def _intra_free(si):
    s = dict(si)
    s["db_info"] = si["db_info"] & ~np.uint32(INTRA)
    if si["db_info_c"] is not None:
        s["db_info_c"] = si["db_info_c"] & ~np.uint32(INTRA)
    return s


# ---- segment cuts of the band walks (launch_sao in ilf_sao.cu, launch_alf / alf_nseg in ilf_alf.cu, pick_segments in
# ilf_common.cuh): 148 SMs, 4 resident SAO CTAs and 5 ALF CTAs per SM, bands of 32 rows, tiles of 128 (SAO) and 64 (ALF)
def _div_up(a, b):
    return (a + b - 1) // b


def _pick_segments(bands_total, ntx, resident, startup=0.5):
    best, best_score = 1, -1.0
    for nseg in range(1, ntx + 1):
        length = ntx / nseg
        if nseg > 1 and length < 2:
            break
        waves = bands_total * nseg / resident
        score = waves / int(waves + 0.999) * length / (length + startup)
        if score > best_score * 1.02:
            best, best_score = nseg, score
    return best


def segment_cuts(w, h, n):
    """(SAO, ALF luma, ALF chroma) segments per band of a launch over n slots with every plane on."""
    by, bcb = _div_up(h, 32), _div_up(h // 2, 32)
    sao = min(max(_div_up(148 * 4, n * (by + 2 * bcb)), 1), _div_up(w, 128))
    alf_c = min(max(_div_up(148 * 5, 2 * bcb * n), 1), _div_up(w // 2, 64))
    return sao, _pick_segments(by * n, _div_up(w, 64), 148 * 5), alf_c


SEGMENT_GEOMS = [(56, 24, 7), (4096, 8, 7), (16384, 16, 5), GEOMS[9]]
SEGMENT_BATCHES = (1, 2, 17, 64)
# banded == whole picture where the last CTU row is partial and shorter than the 16 halo rows
BAND_CASES = [(264, 136, 6, 2), (328, 136, 5, 3), (24, 1032, 6, 3)]


# ---- CPU: what the matrix covers ---------------------------------------------------------------------------------------------

def test_geometry_matrix_covers_every_tile_edge():
    ws = [w for w, _, _ in GEOMS]
    assert {w % 128 for w in ws} == set(range(0, 128, 8)), "a luma width residue mod 128 is missing"
    assert {(w // 2) % 64 for w in ws} >= set(range(0, 64, 4)), "a chroma width residue mod 64 is missing"
    assert {w % 64 for w in ws} == set(range(0, 64, 8)), "a luma width residue mod 64 (ALF tiles) is missing"
    assert {(h % 32, c) for _, h, c in GEOMS} >= {(r, c) for r in (0, 8, 16, 24) for c in (5, 6, 7)}, "a (height mod 32, CTU) pair is missing"
    for c in (5, 6, 7):
        ctu = 1 << c
        cases = [(w, h) for w, h, cc in GEOMS if cc == c]
        assert any(w % ctu and h % ctu for w, h in cases), f"CTU {ctu}: no case with a partial last CTU row and column"
        assert any(w % ctu == 0 and h % ctu == 0 for w, h in cases), f"CTU {ctu}: no case of whole CTUs"
    assert {w for w, h, _ in GEOMS if h < 32} >= {8, 16, 24, 32, 40, 56}, "a width under one box is missing"
    assert {h for _, h, _ in GEOMS if h < 32} >= {8, 16, 24}, "a height under a band plus its shift is missing"
    assert any(w / 2 < 16 for w, _, _ in GEOMS) and any(16 <= w / 2 < 32 for w, h, _ in GEOMS if h < 32), "chroma under 16 samples wide"
    for w, h in ((8, 2048), (16, 4096), (4096, 8), (MAX_SIZE, 16)):
        assert any(g[:2] == (w, h) for g in GEOMS), f"elongated {w} x {h} is missing"
    assert any(w > 7680 for w, _, _ in GEOMS)
    assert LARGEST[0] == MAX_SIZE and LARGEST[1] >= MAX_SIZE - 128
    # the deblocking tile id packs tx into 8 bits and the band into 12: the largest accepted picture must fit both
    for w, h, _ in GEOMS + [LARGEST]:
        assert _div_up(w, 128) <= 256 and _div_up(h + 4, 32) <= 4096
    for w, h, c in GEOMS + [LARGEST]:
        assert w % 8 == 0 and h % 8 == 0 and 8 <= w <= MAX_SIZE and 8 <= h <= MAX_SIZE and c in (5, 6, 7), (w, h, c)
    assert 40 <= len(GEOMS) <= 60 and len(set(GEOMS)) == len(GEOMS)


def test_content_alternates_across_the_matrix():
    plans = [plan(i) for i in range(len(GEOMS))]
    assert {(bl, bc) for bl, bc, *_ in plans} == set(BDS)
    assert {p[2] for p in plans} == set(MVS)
    assert {p[3] for p in plans} == {True, False} and {p[4] for p in plans} == {True, False} and {p[5] for p in plans} == {"dot", "big"}
    # every width residue is met with and without a chroma-tree layer or with both ALF paths across its two cases
    small = [plan(i) for i, (w, h, _) in enumerate(GEOMS) if h < 32]
    assert {p[5] for p in small} == {"dot", "big"} and {p[0] != p[1] for p in small} == {True, False}


def test_segment_and_band_cases():
    for g in SEGMENT_GEOMS:
        assert g in GEOMS
    assert SEGMENT_GEOMS[0][0] < 64, "one segment case is narrower than one tile"
    for w, h, _ in SEGMENT_GEOMS[1:]:
        cuts = [segment_cuts(w, h, n) for n in SEGMENT_BATCHES]
        for k, what in enumerate(("SAO", "ALF luma", "ALF chroma")):
            assert len({c[k] for c in cuts}) >= (3 if w == MAX_SIZE else 2), f"{w} x {h}: the batch sizes cut the {what} bands into {[c[k] for c in cuts]} segments"
    for w, h, c, n in BAND_CASES:
        ctu = 1 << c
        assert (w, h, c) in GEOMS and 0 < h % ctu < 16 and _div_up(h, ctu) >= n, (w, h, c)


# ---- GPU: every stage and every reader per geometry ---------------------------------------------------------------------------

def _ids(cases):
    return [f"{w}x{h}-ctu{1 << c}" for w, h, c in cases]


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(GEOMS)), ids=_ids(GEOMS))
def test_stages_and_chain_equal_oracle(i, ilf_lib, oracle):
    """Deblocking, SAO and ALF each alone on an uploaded picture, the same picture without an intra unit through deblocking
    (chroma untouched), then the chain twice, its picture hash and its download with replicated borders."""
    w, h, c = GEOMS[i]
    bl, bc, _, _, _, alf_kind = plan(i)
    pic, org, si = case_inputs(i)
    O = oracle
    want_db = O.deblock(pic, bl, bc, c, *_db_args(si))
    free = _intra_free(si)
    want_free = O.deblock(pic, bl, bc, c, *_db_args(free))
    want = oracle_chain(O, pic, bl, bc, c, si)
    margin = (8, 24, 80)[i % 3]
    with ilf_lib.InLoopFilter(w, h, bl, bc, c) as f:
        load(f, 0, pic, org, si)
        assert f.alf_path(0) == (3 if alf_kind == "dot" else 0), f"ALF path {f.alf_path(0)} for {alf_kind} coefficients"
        f.loop_filter_pic(0)
        assert not (d := _diff(f.download(0), want_db)), f"deblocking: mismatching samples {d}"
        f.upload(0, *(pic[k] for k in K))
        f.set_sao_params(0, si["sao_ctus"])
        f.sao_process(0)
        assert not (d := _diff(f.download(0), O.sao(pic, bl, bc, c, si["sao_ctus"]))), f"SAO: mismatching samples {d}"
        f.upload(0, *(pic[k] for k in K))
        f.set_alf_params(0, si["alf_params"], si["alf_ctu_enable"])
        f.alf_process(0)
        assert not (d := _diff(f.download(0), O.alf(pic, bl, bc, c, si["alf_params"], si["alf_ctu_enable"]))), f"ALF: mismatching samples {d}"
        f.upload(0, *(pic[k] for k in K))
        f.set_deblock_info(0, *_db_args(free))
        f.loop_filter_pic(0)
        got = f.download(0)
        assert not (d := _diff(got, want_free)), f"deblocking without intra: mismatching samples {d}"
        assert np.array_equal(got["cb"], pic["cb"]) and np.array_equal(got["cr"], pic["cr"])
        load(f, 0, pic, org, si)
        f.run(0, 1, 7)
        got = f.download(0)
        assert not (d := _diff(got, want)), f"chain: mismatching samples {d}"
        f.run(0, 1, 7)
        assert not _diff(f.download(0), got), "a second run differs"
        for kind in ("crc", "checksum"):
            assert f.picture_hash(0, kind) == O.picture_hash(want, bl, bc, kind), kind
        ext = f.download_extended(0, margin)
    for k, s in (("y", 0), ("cb", 1), ("cr", 1)):
        assert np.array_equal(ext[k], O.extend_border(want[k], margin >> s, margin >> s)), f"download_extended, plane {k}, margin {margin}"


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(GEOMS)), ids=_ids(GEOMS))
def test_readers_equal_oracle(i, ilf_lib, oracle):
    """ALF classification of the uploaded picture; SAO and ALF statistics of the deblocked picture; the deblocking offset search."""
    from test_gpu_deblock_search import oracle_search
    w, h, c = GEOMS[i]
    bl, bc = plan(i)[:2]
    pic, org, si = case_inputs(i)
    O = oracle
    dbk = O.deblock(pic, bl, bc, c, *_db_args(si))
    shift = (1, 2)
    want_search = oracle_search(O, pic, org, bl, bc, c, *_db_args(si), SEARCH_CANDS, [shift])[shift]
    with ilf_lib.InLoopFilter(w, h, bl, bc, c) as f:
        load(f, 0, pic, org, si)
        assert np.array_equal(f.alf_classify(0), O.alf_classify(pic["y"], bl)), "ALF classification"
        f.run(0, 1, 1)
        f.sao_stats(0, 1)
        got = f.get_sao_stats(0)
        want = O.sao_stats(dbk, org, bl, bc, c, si["avail"])
        bad = np.argwhere(got != want)
        assert bad.size == 0, f"SAO statistics: first mismatch (ctu, comp, type, word) {bad[0]}"
        f.alf_stats(0, 1)
        got = f.get_alf_stats(0)
        bad = np.argwhere(got != O.alf_stats(dbk, org, bl, c))
        assert bad.size == 0, f"ALF statistics: first mismatch (ctu, word) {bad[0]}"
        f.deblock_search(SEARCH_CANDS, shift)
        got = f.get_deblock_search(0)
    assert np.array_equal(got, want_search), f"deblocking search: {got} != {want_search}"


def _lib_call(f, name, planes):
    """ilf_upload / ilf_download with each plane's own row stride (the binding makes host planes contiguous first)."""
    args = []
    for a in planes:
        assert a.dtype == np.int16 and a.strides[1] == 2
        args += [C.c_void_p(a.ctypes.data), a.strides[0] // 2]
    f._ck(getattr(f._lib, name)(f._h, 0, *args))


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True], ids=["pageable", "pinned"])
@pytest.mark.parametrize("i", range(len(GEOMS)), ids=_ids(GEOMS))
def test_upload_download_round_trip(i, pinned, ilf_lib):
    """Host planes that are views into wider arrays, in pageable or page-locked memory: the download of a slot no stage has run on
    equals its upload, and leaves the host columns beyond the picture alone."""
    w, h, c = GEOMS[i]
    bl, bc = plan(i)[:2]
    pic = synth.picture(np.random.default_rng(3000 + i), w, h, bl, "noise", bd_chroma=bc)
    pad = 72
    if pinned:
        src_full, dst_full = ilf_lib.pinned_planes(w + 2 * pad, h), ilf_lib.pinned_planes(w + 2 * pad, h)
    else:
        src_full = {k: np.zeros((h >> (k != "y"), (w + 2 * pad) >> (k != "y")), np.int16) for k in K}
        dst_full = {k: np.zeros_like(src_full[k]) for k in K}
    try:
        src = {k: src_full[k][:, : w >> (k != "y")] for k in K}
        dst = {k: dst_full[k][:, : w >> (k != "y")] for k in K}
        for k in K:
            src[k][...] = pic[k]
            dst_full[k][...] = -7
        with ilf_lib.InLoopFilter(w, h, bl, bc, c) as f:
            _lib_call(f, "ilf_upload", [src[k] for k in K])
            _lib_call(f, "ilf_download", [dst[k] for k in K])
            f.sync()
        for k in K:
            assert np.array_equal(dst[k], pic[k]), f"plane {k}: the download differs from the upload"
            assert (dst_full[k][:, w >> (k != "y"):] == -7).all(), f"plane {k}: the download wrote beyond the picture's width"
    finally:
        if pinned:
            for full in (src_full, dst_full):
                for k in K:
                    ilf_lib.load_library().ilf_host_free(C.c_void_p(full[k].ctypes.data))


@pytest.mark.skipif(os.environ.get("ILF_TEST_LARGEST") != "1", reason="16384 x 16384: 2.4 GB of device memory per slot and about 30 s of oracle; set ILF_TEST_LARGEST=1")
@pytest.mark.gpu
def test_largest_picture(ilf_lib, oracle):
    """The largest accepted picture: deblocking tile ids up to tx 127 and band 512, SAO / ALF walks of 128 and 256 tiles per band,
    16384 rows of the picture hash -- deblocking, the chain, the hash and one search candidate against the oracle."""
    from test_gpu_deblock_search import oracle_search
    w, h, c = LARGEST
    bl, bc = 10, 10
    rng = np.random.default_rng(16384)
    tile = synth.picture(rng, 2048, 2048, bl, "mix", bd_chroma=bc)
    pic = {k: np.tile(tile[k], (8, 8)) for k in K}
    pic["y"][-9:, -13:] = 0   # the bottom-right corner differs from the repeated tile
    org = {k: np.clip(pic[k].astype(np.int32) + rng.integers(-12, 13, pic[k].shape, dtype=np.int32), 0, 1023).astype(np.int16) for k in K}
    si = synth.deblock_info_stress(rng, w, h, c, False, bd_luma=bl, chroma_qp_offset=12)
    si["db_mv32"] = None
    cw, ch = _ctus(w, h, c)
    si["sao_ctus"] = synth.sao_params(rng, cw, ch, bl, p_off=0.2, bd_chroma=bc)
    si["alf_params"], si["alf_ctu_enable"] = synth.alf_params(rng, cw, ch, True, p_on=0.8, dot=True)
    si["avail"] = _avail(rng, w, h, c)
    O = oracle
    want_db = O.deblock(pic, bl, bc, c, *_db_args(si))
    want_search = oracle_search(O, pic, org, bl, bc, c, *_db_args(si), [(3, -2)], [(0, 0)])[(0, 0)]
    want = O.alf(O.sao(want_db, bl, bc, c, si["sao_ctus"]), bl, bc, c, si["alf_params"], si["alf_ctu_enable"])
    with ilf_lib.InLoopFilter(w, h, bl, bc, c) as f:
        load(f, 0, pic, org, si)
        f.loop_filter_pic(0)
        assert not (d := _diff(f.download(0), want_db)), f"deblocking: mismatching samples {d}"
        f.deblock_search([(3, -2)], (0, 0))
        assert np.array_equal(f.get_deblock_search(0), want_search)
        f.run(0, 1, 7)
        assert not (d := _diff(f.download(0), want)), f"chain: mismatching samples {d}"
        for kind in ("crc", "checksum"):
            assert f.picture_hash(0, kind) == O.picture_hash(want, bl, bc, kind), kind


# ---- GPU: segment borders, batch chunks and bands -----------------------------------------------------------------------------

def _slot_inputs(w, h, c, j, bl=10, bc=10):
    """Content of slot j of a batch: its own seed, motion representation, chroma-tree layer and ALF shape."""
    return inputs(7000 + 131 * j + w + h, w, h, c, bl, bc, MVS[j % 3], j % 2 == 0, j % 4 < 2, "dot")


def scramble(f, data, first, n, cands, shift):
    """Leave other results in every buffer a slot of [first, first + n) writes (work buffers, statistics, search sums), then
    load its own picture again: a batch that skipped a slot, a tile or a segment cannot pass on what a one-slot run left."""
    for j in range(first, first + n):
        load(f, j, *data[(j + 1) % len(data)])
        f.run(j, 1, 7)
        f.sao_stats(j, 1)
        f.alf_stats(j, 1)
        f.deblock_search(cands, shift, j, 1)
        load(f, j, *data[j])


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,c", SEGMENT_GEOMS, ids=_ids(SEGMENT_GEOMS))
def test_segment_cuts_move_with_the_batch(w, h, c, ilf_lib, oracle):
    """The same 64 pictures as batches of 1, 2, 17 and 64 slots: the SAO and ALF bands are cut into different segments at each
    batch size, and every slot equals its one-slot run and the oracle (chain, deblocking, SAO and ALF statistics)."""
    n_max = max(SEGMENT_BATCHES)
    data = [_slot_inputs(w, h, c, j) for j in range(n_max)]
    with ilf_lib.InLoopFilter(w, h, 10, 10, c, num_slots=n_max) as f:
        for j, (pic, org, si) in enumerate(data):
            load(f, j, pic, org, si)

        def results(first, n):
            f.run(first, n, 1)
            f.sao_stats(first, n)
            f.alf_stats(first, n)
            out = [(f.download(j), f.get_sao_stats(j), f.get_alf_stats(j)) for j in range(first, first + n)]
            f.run(first, n, 7)
            return [o + (f.download(j),) for j, o in zip(range(first, first + n), out)]

        single = [results(j, 1)[0] for j in range(n_max)]
        for j, (pic, org, si) in enumerate(data):
            dbk = oracle.deblock(pic, 10, 10, c, *_db_args(si))
            assert not _diff(single[j][0], dbk), f"slot {j}: deblocking != oracle"
            assert np.array_equal(single[j][1], oracle.sao_stats(dbk, org, 10, 10, c, si["avail"])), f"slot {j}: SAO statistics != oracle"
            assert np.array_equal(single[j][2], oracle.alf_stats(dbk, org, 10, c)), f"slot {j}: ALF statistics != oracle"
            want = oracle.alf(oracle.sao(dbk, 10, 10, c, si["sao_ctus"]), 10, 10, c, si["alf_params"], si["alf_ctu_enable"])
            assert not _diff(single[j][3], want), f"slot {j}: chain != oracle"
        for n in SEGMENT_BATCHES[1:]:
            scramble(f, data, 0, n, SEARCH_CANDS[:1], (0, 0))
            for j, got in enumerate(results(0, n)):
                assert not _diff(got[0], single[j][0]), f"batch {n}, slot {j}: deblocking"
                assert np.array_equal(got[1], single[j][1]) and np.array_equal(got[2], single[j][2]), f"batch {n}, slot {j}: statistics"
                assert not _diff(got[3], single[j][3]), f"batch {n}, slot {j}: chain"


CHUNK_GEOM = (136, 72, 5)
CHUNK_SLOTS = 130


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", ["off", "default"])
def test_batches_over_128_slots(lanes, ilf_lib, oracle, monkeypatch):
    """130 slots, each its own picture: the chain, deblocking alone, both statistics and the offset search over [0, 130) (chunks
    [0, 128) and [128, 130)) and over [1, 130) (chunks [1, 129) and [129, 130)) give every slot its one-slot result; the slots on
    each side of both chunk borders also equal the oracle."""
    from test_gpu_deblock_search import oracle_search
    if lanes == "off":
        monkeypatch.setenv("ILF_RUN_LANES", "1")
    w, h, c = CHUNK_GEOM
    n = CHUNK_SLOTS
    shift = (0, 1)
    cands = SEARCH_CANDS[:4]
    bl, bc = 10, 8
    data = [_slot_inputs(w, h, c, j, bl, bc) for j in range(n)]
    with ilf_lib.InLoopFilter(w, h, bl, bc, c, num_slots=n) as f:
        assert f.run_lanes() == (1 if lanes == "off" else 2)
        for j, (pic, org, si) in enumerate(data):
            load(f, j, pic, org, si)

        def results(first, cnt):
            f.run(first, cnt, 7)
            chain = [f.download(j) for j in range(first, first + cnt)]
            f.run(first, cnt, 1)
            f.sao_stats(first, cnt)
            f.alf_stats(first, cnt)
            f.deblock_search(cands, shift, first, cnt)
            return [(chain[j - first], f.download(j), f.get_sao_stats(j), f.get_alf_stats(j), f.get_deblock_search(j)) for j in range(first, first + cnt)]

        single = [results(j, 1)[0] for j in range(n)]
        for first in (0, 1):
            scramble(f, data, first, n - first, cands[::-1], shift)
            for j, got in zip(range(first, n), results(first, n - first)):
                for what, a, b in zip(("chain", "deblocking"), got[:2], single[j][:2]):
                    assert not _diff(a, b), f"[{first}, {n}) slot {j}: {what} differs from its one-slot run"
                for what, a, b in zip(("SAO statistics", "ALF statistics", "search"), got[2:], single[j][2:]):
                    assert np.array_equal(a, b), f"[{first}, {n}) slot {j}: {what} differs from its one-slot run"
    for j in (0, 1, 127, 128, 129):
        pic, org, si = data[j]
        dbk = oracle.deblock(pic, bl, bc, c, *_db_args(si))
        chain, got_db, sao_s, alf_s, search = single[j]
        assert not _diff(chain, oracle_chain(oracle, pic, bl, bc, c, si)), f"slot {j}: chain != oracle"
        assert not _diff(got_db, dbk), f"slot {j}: deblocking != oracle"
        assert np.array_equal(sao_s, oracle.sao_stats(dbk, org, bl, bc, c, si["avail"])), f"slot {j}: SAO statistics != oracle"
        assert np.array_equal(alf_s, oracle.alf_stats(dbk, org, bl, c)), f"slot {j}: ALF statistics != oracle"
        want = oracle_search(oracle, pic, org, bl, bc, c, *_db_args(si), cands, [shift])[shift]
        assert np.array_equal(search, want), f"slot {j}: search != oracle"


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,c,n", BAND_CASES, ids=[f"{w}x{h}-ctu{1 << c}-bands{n}" for w, h, c, n in BAND_CASES])
def test_bands_with_a_short_last_ctu_row(w, h, c, n, ilf_lib, oracle):
    from test_gpu_bands import _run_banded, _run_whole
    i = GEOMS.index((w, h, c))
    bl, bc = plan(i)[:2]
    pic, _, si = case_inputs(i)
    whole = _run_whole(ilf_lib, w, h, bl, bc, c, pic, si)
    assert not (d := _diff(whole, oracle_chain(oracle, pic, bl, bc, c, si))), f"whole picture != oracle: {d}"
    banded = _run_banded(ilf_lib, w, h, bl, bc, c, pic, si, n)
    assert not (d := _diff(banded, whole)), f"banded != whole picture: {d}"
