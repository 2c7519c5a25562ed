"""Encoder ALF statistics on the GPU (SURVEY.md 8f rank 3; EncAdaptiveLoopFilter::deriveStatsForFiltering / getBlkStats / calcCovariance)
against the oracle, which tests/test_oracle_units.py pins against the reference's own getBlkStats.  Bit-exact int64 sums."""
import numpy as np
import pytest

import synth

K = ("y", "cb", "cr")


def _org_of(rng, pic, bd, bd_chroma=None):
    """The picture plus noise, each plane clipped to its own range (luma `bd`, chroma `bd_chroma`, default `bd`)."""
    bds = dict(zip(K, (bd,) + 2 * (bd if bd_chroma is None else bd_chroma,)))
    return {k: np.clip(pic[k].astype(np.int32) + rng.integers(-30, 31, pic[k].shape), 0, (1 << bds[k]) - 1).astype(np.int16) for k in K}


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,bd_luma,bd_chroma,ctu_log2,seed",
                         synth.keep_ids([(416, 240, 10, 7, 1), (200, 136, 10, 6, 2), (264, 72, 8, 5, 3), (136, 264, 12, 5, 4), (1920, 1080, 10, 7, 5)],
                                        lambda w, h, bd, c, s: (w, h, bd, bd, c, s)) +
                         [(200, 136, 8, 12, 6, 6), (264, 72, 12, 8, 5, 7)])
def test_alf_statistics_match_oracle(w, h, bd_luma, bd_chroma, ctu_log2, seed, ilf_lib, oracle):
    """Odd sizes with partial CTUs, 8/10/12 bit with luma and chroma at the same or at different depths (the classification
    follows the luma depth), textured content (every class and transposition occurs) and full-range noise."""
    rng = np.random.default_rng(seed)
    with ilf_lib.InLoopFilter(w, h, bd_luma, bd_chroma, ctu_log2) as f:
        for kind in ("mix", "noise"):
            pic = synth.picture(rng, w, h, bd_luma, kind, bd_chroma=bd_chroma)
            org = _org_of(rng, pic, bd_luma, bd_chroma)
            f.upload(0, *(pic[k] for k in K))
            f.set_original(0, org["y"], org["cb"], org["cr"], np.zeros(((w + (1 << ctu_log2) - 1) >> ctu_log2) * ((h + (1 << ctu_log2) - 1) >> ctu_log2), np.uint8))
            f.alf_stats(0, 1)
            got = f.get_alf_stats(0)
            want = oracle.alf_stats(pic, org, bd_luma, ctu_log2)
            bad = np.argwhere(got != want)
            assert bad.size == 0, f"{kind}: first mismatch (ctu, word) {bad[0]}: got {got[tuple(bad[0])]} want {want[tuple(bad[0])]}"
            if kind == "mix":
                cls = oracle.alf_classify(pic["y"], bd_luma)
                assert len(np.unique(cls >> 5)) == 4 and len(np.unique(cls & 31)) >= 5     # the case really covers the transpositions and several classes


def test_5x5_luma_statistics_are_a_slice_of_the_7x7_record(oracle):
    """What include/ilf_b200.h promises the host: under every transposition the 5x5 taps are taps {2, 5, 6, 7, 10, 11, 12} of the 7x7 diamond."""
    import ctypes as C
    rng = np.random.default_rng(3)
    w, h = 32, 24
    rec = rng.integers(0, 1024, (h, w)).astype(np.int16)
    org = rng.integers(0, 1024, (h, w)).astype(np.int16)
    cls = (rng.integers(0, 25, (h // 4, w // 4)) | (rng.integers(0, 4, (h // 4, w // 4)) << 5)).astype(np.uint8)
    g = oracle.lib().ilf_oracle_alf_stats_block
    g.argtypes = [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_ssize_t, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    s7 = np.zeros((25, 105), np.int64)
    s5 = np.zeros((25, 36), np.int64)
    g(rec.ctypes.data, w, org.ctypes.data, w, w, h, 1, cls.ctypes.data, s7.ctypes.data)
    g(rec.ctypes.data, w, org.ctypes.data, w, w, h, 0, cls.ctypes.data, s5.ctypes.data)
    m = list(oracle.ALF_5X5_IN_7X7)
    for c in range(25):
        E7, y7, p7 = oracle.alf_stats_unpack(s7[c], 13)
        E5, y5, p5 = oracle.alf_stats_unpack(s5[c], 7)
        assert np.array_equal(E7[np.ix_(m, m)], E5) and np.array_equal(y7[m], y5) and p7 == p5
