"""Luma and chroma at different bit depths (ilf_config.bit_depth_luma / bit_depth_chroma, each 8..12, taken from the SPS) and the
edges of the deblocking QP inputs: negative QPs in the grid (down to -6 (bd_luma - 8) at 10 and 12 bit), PPS chroma QP offsets of
+-12, and with them chroma QPs of 70 and over (the qp - 6 branch of the chroma QP mapping, LoopFilter.cpp:812-817) and below 0.

Every check is bit-exact.  The per-plane checks need no oracle: a context at depths (bl, bc) must give the luma of a context at
(bl, bl) and the chroma of one at (bc, bc) for the same planes and side information, so a kernel that takes the other plane's
depth fails them even where the oracle would make the same mistake.  The tests without the gpu mark pin what the GPU tests rely on:
the generator reaches the QP edges and the oracle itself keeps the planes apart."""
import hashlib

import numpy as np
import pytest

import synth

K = ("y", "cb", "cr")
EDGE_V, EDGE_H, INTRA = 0x04, 0x10, 0x01      # ILF_BI_EDGE_V / _EDGE_H / _INTRA
CANDS = [(0, 0), (3, -2), (-4, 5), (-6, -6), (20, -20), (-128, 127)]


def _ctus(w, h, ctu_log2):
    ctu = 1 << ctu_log2
    return (w + ctu - 1) // ctu, (h + ctu - 1) // ctu


def _inputs(seed, w, h, bl, bc, ctu_log2, pic_bd=None, kind="mix"):
    """Seeded planes and side information of every stage.  Deblocking: the stress layers with the QPs of luma depth `bl` (negative
    below 0 at 10 and 12 bit) and chroma QP offsets up to +-12.  The planes, the original and the SAO offsets are drawn at (bl, bc),
    or all at `pic_bd` when one picture has to be valid at several depths."""
    rng = np.random.default_rng(seed)
    pl, pc = (bl, bc) if pic_bd is None else (pic_bd, pic_bd)
    pic = synth.picture(rng, w, h, pl, kind, bd_chroma=pc)
    org = {k: np.clip(pic[k].astype(np.int32) + rng.integers(-12, 13, pic[k].shape), 0, (1 << (pc if k != "y" else pl)) - 1).astype(np.int16) for k in K}
    si = synth.deblock_info_stress(rng, w, h, ctu_log2, False, bd_luma=bl, chroma_qp_offset=12)
    cw, ch = _ctus(w, h, ctu_log2)
    si["sao_ctus"] = synth.sao_params(rng, cw, ch, pl, p_off=0.2, bd_chroma=pc)
    si["alf_params"], si["alf_ctu_enable"] = synth.alf_params(rng, cw, ch, True, p_on=0.8)
    return pic, org, si


def _db_args(si):
    return si["db_params"], si["db_info"], si["db_info_c"], si.get("db_mv16"), si.get("db_mv32"), si["ctu_slice"]


def _oracle_chain(O, pic, bl, bc, ctu_log2, si):
    d = O.deblock(pic, bl, bc, ctu_log2, *_db_args(si))
    d = O.sao(d, bl, bc, ctu_log2, si["sao_ctus"])
    return O.alf(d, bl, bc, ctu_log2, si["alf_params"], si["alf_ctu_enable"])


def _load(f, pic, org, si):
    f.upload(0, *(pic[k] for k in K))
    f.set_deblock_info(0, *_db_args(si))
    f.set_sao_params(0, si["sao_ctus"])
    f.set_alf_params(0, si["alf_params"], si["alf_ctu_enable"])
    f.set_original(0, org["y"], org["cb"], org["cr"], np.zeros(f.ctus_w * f.ctus_h, np.uint8))


def _at_qp_edges(si):
    """Cb offset +12 and Cr offset -12, so that chroma QPs reach 70 and over and fall below 0; the three slices' tc offsets
    negative, so that the tc index of a chroma QP of 70 and over, qp - 6 + 2 + 2 tc_offset, stays below the end of the table,
    where the mapping's qp - 6 shows."""
    prm = np.frombuffer(bytes(si["db_params"]), synth.DB_DT).copy()
    prm["cb_qp_offset"], prm["cr_qp_offset"] = 12, -12
    prm["slices"][0, :3, 1] = (-1, -3, -6)
    si["db_params"] = prm.tobytes()
    return si


def qp_edge_counts(O, w, h, si):
    """Filtered edges of the picture's side information at the QP edges: chroma edges (16-sample grid, an intra side) whose QP
    plus the Cb or Cr offset is >= 70 and < 0, and luma edges (bS > 0) with a negative QP on either side."""
    prm = np.frombuffer(bytes(si["db_params"]), synth.DB_DT)[0]
    qp_of = lambda a: ((a >> 8) & 0xFF).astype(np.uint8).view(np.int8).astype(np.int32)
    c = si["db_info_c"]
    uh, uw = c.shape
    hi = neg = 0
    for q, p, edge in ((c[:, 4::4], c[:, 3:uw - 1:4], EDGE_V), (c[4::4, :], c[3:uh - 1:4, :], EDGE_H)):
        filt = ((q & edge) != 0) & (((q | p) & INTRA) != 0)
        qp = (qp_of(p) + qp_of(q) + 1) >> 1
        for off in (int(prm["cb_qp_offset"]), int(prm["cr_qp_offset"])):
            hi += int((filt & (qp + off >= 70)).sum())
            neg += int((filt & (qp + off < 0)).sum())
    bs = O.bs_map(w, h, si["db_params"], si["db_info"], si.get("db_mv16"), si.get("db_mv32"))
    neg_y = qp_of(si["db_info"]) < 0
    luma = int(((bs[0][:, 1:] > 0) & (neg_y[:, 1:] | neg_y[:, :-1])).sum() + ((bs[1][1:, :] > 0) & (neg_y[1:, :] | neg_y[:-1, :])).sum())
    return hi, neg, luma


# ---- CPU: the generator and the oracle ------------------------------------------------------------------------------------

# sha256 of deblock_info_stress(default_rng(7), 200, 136, 5, True) at its defaults, as drawn before the QP range and the chroma
# offset range were arguments: the seeded cases written then keep their side information
STRESS_DEFAULT_DIGEST = "8551cf9a4b8dc99ad2b1c931e267dbc442bb922f2c022ff51b5d436c47257311"


def test_stress_generator_defaults_are_unchanged():
    si = synth.deblock_info_stress(np.random.default_rng(7), 200, 136, 5, True)
    h = hashlib.sha256()
    for k in sorted(si):
        h.update(k.encode())
        h.update(bytes(si[k]) if isinstance(si[k], bytes) else np.ascontiguousarray(si[k]).tobytes())
    assert h.hexdigest() == STRESS_DEFAULT_DIGEST


# smooth content with saturated patches (the luma filters' decisions pass) and full-range noise (chroma steps beyond tc)
QP_EDGE_CASES = [(520, 392, 12, 8, 6, "mix", 71), (520, 392, 12, 8, 6, "noise", 72), (1920, 1080, 10, 12, 7, "mix", 73), (1920, 1080, 10, 12, 7, "noise", 74)]


@pytest.mark.parametrize("w,h,bl,bc,ctu_log2,kind,seed", QP_EDGE_CASES)
def test_stress_generator_reaches_the_qp_edges(w, h, bl, bc, ctu_log2, kind, seed, oracle):
    si = _at_qp_edges(_inputs(seed, w, h, bl, bc, ctu_log2, kind=kind)[2])
    hi, neg, luma = qp_edge_counts(oracle, w, h, si)
    assert hi > 0 and neg > 0 and luma > 0, f"chroma QP >= 70: {hi}, chroma QP < 0: {neg}, luma edges with a negative QP: {luma}"


def _assert_planes_follow(mixed, luma_of, chroma_of, what, chroma_reads_depth=True):
    """(luma, chroma) results at (bl, bc), (bl, bl) and (bc, bc): the first takes its luma from the second and its chroma from the
    third, and the two depths give different results (else the check could not see a swapped depth)."""
    assert np.array_equal(mixed[0], luma_of[0]), f"{what}: the luma differs from the context whose chroma has the luma depth"
    assert np.array_equal(mixed[1], chroma_of[1]), f"{what}: the chroma differs from the context whose luma has the chroma depth"
    assert not np.array_equal(luma_of[0], chroma_of[0]), f"{what}: the luma does not depend on the depth"
    if chroma_reads_depth:
        assert not np.array_equal(luma_of[1], chroma_of[1]), f"{what}: the chroma does not depend on the depth"


def _planes(d):
    return d["y"], np.stack([d["cb"], d["cr"]])


@pytest.mark.parametrize("w,h,bl,bc,ctu_log2,seed", [(200, 136, 8, 12, 5, 81), (264, 72, 12, 10, 6, 82)])
def test_oracle_keeps_the_planes_apart(w, h, bl, bc, ctu_log2, seed, oracle):
    pic, _, si = _inputs(seed, w, h, bl, bc, ctu_log2, pic_bd=min(bl, bc))
    run = {(a, b): _planes(_oracle_chain(oracle, pic, a, b, ctu_log2, si)) for a, b in ((bl, bc), (bl, bl), (bc, bc))}
    _assert_planes_follow(run[bl, bc], run[bl, bl], run[bc, bc], "oracle chain")


# ---- GPU ----------------------------------------------------------------------------------------------------------------------

# partial CTUs at CTU 32 / 64 / 128, each geometry with two or three unequal depth pairs
CHAIN_CASES = [(200, 136, 8, 12, 5, 1), (200, 136, 12, 8, 5, 2), (264, 72, 10, 8, 6, 3), (264, 72, 8, 10, 6, 4), (136, 264, 12, 10, 7, 5),
               (136, 264, 8, 12, 7, 6), (392, 72, 12, 8, 6, 7), (392, 72, 10, 12, 6, 8), (520, 392, 8, 12, 7, 9), (520, 392, 12, 8, 7, 10),
               (520, 392, 10, 8, 7, 11), (16, 16, 12, 8, 5, 12), (16, 16, 8, 10, 5, 13), (1920, 1080, 10, 8, 7, 14)]


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,bl,bc,ctu_log2,seed", CHAIN_CASES)
def test_chain_equals_oracle(w, h, bl, bc, ctu_log2, seed, ilf_lib, oracle):
    """deblock -> SAO -> ALF in one ilf_run at two depths, negative QPs and chroma offsets up to +-12; a second run gives the same."""
    pic, org, si = _inputs(seed, w, h, bl, bc, ctu_log2)
    want = _oracle_chain(oracle, pic, bl, bc, ctu_log2, si)
    with ilf_lib.InLoopFilter(w, h, bl, bc, ctu_log2) as f:
        _load(f, pic, org, si)
        f.run(0, 1, 7)
        got = f.download(0)
        f.run(0, 1, 7)
        again = f.download(0)
    d = {k: int((got[k] != want[k]).sum()) for k in K}
    assert not any(d.values()), f"mismatching samples {d}"
    assert all(np.array_equal(got[k], again[k]) for k in K), "a second run differs"
    assert all((got[k] != pic[k]).any() for k in K), "the chain left a plane alone"


def _gpu_results(v, w, h, bl, bc, ctu_log2, pic, org, si):
    """Everything the library computes per plane for one context: {name: (luma, chroma)}."""
    with v.InLoopFilter(w, h, bl, bc, ctu_log2) as f:
        _load(f, pic, org, si)
        out = {}
        for kind in ("crc", "checksum"):
            hv = f.picture_hash(0, kind)
            out[kind] = hv[0], hv[1:]
        f.sao_stats(0, 1)
        s = f.get_sao_stats(0)
        out["sao_stats"] = s[:, 0], s[:, 1:]
        f.alf_stats(0, 1)
        a = f.get_alf_stats(0)
        out["alf_stats"] = a[:, :25 * 105], a[:, 25 * 105:]
        f.deblock_search(CANDS, (1, 2))
        r = f.get_deblock_search(0)
        out["deblock_search"] = r[:, 0], r[:, 1:]
        f.run(0, 1, 7)
        out["chain"] = _planes(f.download(0))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,bl,bc,ctu_log2,seed", [(200, 136, 8, 12, 5, 21), (264, 72, 12, 8, 6, 22), (520, 392, 10, 8, 7, 23)])
def test_each_plane_follows_its_own_depth(w, h, bl, bc, ctu_log2, seed, ilf_lib):
    """Contexts at (bl, bc), (bl, bl) and (bc, bc) on the same planes (valid at both depths) and side information: chain output,
    picture hash, SAO and ALF statistics and the deblocking search of the first take their luma from the second and their chroma
    from the third; and the depth matters for each of them (one depth of each pair is 8, so the hash too; the chroma ALF
    statistics read no depth)."""
    pic, org, si = _inputs(seed, w, h, bl, bc, ctu_log2, pic_bd=min(bl, bc))
    run = {(a, b): _gpu_results(ilf_lib, w, h, a, b, ctu_log2, pic, org, si) for a, b in ((bl, bc), (bl, bl), (bc, bc))}
    for what in run[bl, bc]:
        _assert_planes_follow(run[bl, bc][what], run[bl, bl][what], run[bc, bc][what], what, what != "alf_stats")


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,bl,bc,ctu_log2,kind,seed", QP_EDGE_CASES)
def test_qp_edges_deblock_and_search_equal_oracle(w, h, bl, bc, ctu_log2, kind, seed, ilf_lib, oracle):
    """Chroma QPs >= 70 and < 0 (Cb offset +12, Cr offset -12) and negative luma QPs: ilf_deblock and the offset search == oracle."""
    pic, org, si = _inputs(seed, w, h, bl, bc, ctu_log2, kind=kind)
    si = _at_qp_edges(si)
    assert all(qp_edge_counts(oracle, w, h, si)), "the picture does not reach the QP edges"
    want = oracle.deblock(pic, bl, bc, ctu_log2, *_db_args(si))
    with ilf_lib.InLoopFilter(w, h, bl, bc, ctu_log2) as f:
        _load(f, pic, org, si)
        f.loop_filter_pic(0)
        got = f.download(0)
        f.deblock_search(CANDS, (0, 1))
        search = f.get_deblock_search(0)
    d = {k: int((got[k] != want[k]).sum()) for k in K}
    assert not any(d.values()), f"deblocking: mismatching samples {d}"
    from test_gpu_deblock_search import oracle_search
    want_s = oracle_search(oracle, pic, org, bl, bc, ctu_log2, *_db_args(si), CANDS, [(0, 1)])[(0, 1)]
    assert np.array_equal(search, want_s), f"search: {search} != {want_s}"


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,bl,bc,seed", [(200, 136, 8, 12, 31), (264, 72, 12, 8, 32), (520, 392, 12, 10, 33)])
def test_alf_classification_follows_the_luma_depth(w, h, bl, bc, seed, ilf_lib, oracle):
    pic = synth.picture(np.random.default_rng(seed), w, h, bl, "mix", bd_chroma=bc)
    with ilf_lib.InLoopFilter(w, h, bl, bc, 7) as f:
        f.upload(0, *(pic[k] for k in K))
        got = f.alf_classify(0)
    assert np.array_equal(got, oracle.alf_classify(pic["y"], bl))
