"""Encoder SAO statistics on the GPU (SURVEY.md 8f rank 2; EncSampleAdaptiveOffset::getStatistics / getBlkStats) against the
oracle, which tests/test_oracle_units.py pins against the reference's own getBlkStats.  Bit-exact int64 sums."""
import os
import sys

import numpy as np
import pytest

import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

pytestmark = pytest.mark.gpu
K = ("y", "cb", "cr")


def _org_of(rng, pic, bd, bd_chroma=None):
    """The picture plus noise, each plane clipped to its own range (luma `bd`, chroma `bd_chroma`, default `bd`)."""
    bds = dict(zip(K, (bd,) + 2 * (bd if bd_chroma is None else bd_chroma,)))
    return {k: np.clip(pic[k].astype(np.int32) + rng.integers(-12, 13, pic[k].shape), 0, (1 << bds[k]) - 1).astype(np.int16) for k in K}


@pytest.mark.parametrize("w,h,bd_luma,bd_chroma,ctu_log2,seed",
                         synth.keep_ids([(416, 240, 10, 7, 1), (200, 136, 10, 6, 2), (264, 72, 8, 5, 3), (136, 264, 12, 5, 4), (1920, 1080, 10, 7, 5)],
                                        lambda w, h, bd, c, s: (w, h, bd, bd, c, s)) +
                         [(200, 136, 8, 10, 6, 6), (264, 72, 12, 10, 5, 7)])
def test_statistics_of_the_uploaded_picture(w, h, bd_luma, bd_chroma, ctu_log2, seed, ilf_lib, oracle):
    """Random availability flags (multi-slice patterns), odd sizes with partial CTUs, 8/10/12 bit (luma and chroma at the same or
    at different depths: the band classes of each component follow its own depth), noisy and smooth content."""
    rng = np.random.default_rng(seed)
    ctu = 1 << ctu_log2
    n = ((w + ctu - 1) // ctu) * ((h + ctu - 1) // ctu)
    with ilf_lib.InLoopFilter(w, h, bd_luma, bd_chroma, ctu_log2) as f:
        for kind in ("noise", "smooth"):
            pic = synth.picture(rng, w, h, bd_luma, kind, bd_chroma=bd_chroma)
            org = _org_of(rng, pic, bd_luma, bd_chroma)
            cw = (w + ctu - 1) // ctu
            avail = rng.integers(0, 256, n).astype(np.uint8)
            for i in range(n):      # picture borders are never available
                if i % cw == 0: avail[i] &= ~np.uint8(0x01 | 0x10)
                if i < cw: avail[i] &= ~np.uint8(0x04 | 0x10)
            f.upload(0, *(pic[k] for k in K))
            f.set_original(0, org["y"], org["cb"], org["cr"], avail)
            f.sao_stats(0, 1)
            got = f.get_sao_stats(0)
            want = oracle.sao_stats(pic, org, bd_luma, bd_chroma, ctu_log2, avail)
            bad = np.argwhere(got != want)
            assert bad.size == 0, f"{kind}: first mismatch (ctu, comp, type, word) {bad[0]}: got {got[tuple(bad[0])]} want {want[tuple(bad[0])]}"


def test_statistics_after_deblocking_4k(ilf_lib, oracle):
    """The encoder's order: deblock on the GPU, statistics on the device-resident deblocked picture (4K, real side information)."""
    w, h = 3840, 2160
    side = bench.load_sideinfo("ra_4k")
    planes = bench.synth_planes(w, h, 2, seed=4)
    rng = np.random.default_rng(9)
    n = 30 * 17
    with ilf_lib.InLoopFilter(w, h, 10, 10, 7, num_slots=2) as f:
        want = []
        for j, p in enumerate((0, 6)):
            si = side[p]
            pic = dict(zip(K, planes[j]))
            org = _org_of(rng, pic, 10)
            avail = np.full(n, 0x15, np.uint8)
            avail[np.arange(n) % 30 == 0] &= ~np.uint8(0x11)
            avail[:30] &= ~np.uint8(0x14)
            f.upload(j, *planes[j])
            f.set_deblock_info(j, si["db_params"].tobytes(), si["db_info"], si.get("db_info_c"), si.get("db_mv16"), si.get("db_mv32"), si.get("ctu_slice"))
            f.set_original(j, org["y"], org["cb"], org["cr"], avail)
            dbk = oracle.deblock(pic, 10, 10, 7, si["db_params"].tobytes(), si["db_info"], si.get("db_info_c"), si.get("db_mv16"), si.get("db_mv32"), si.get("ctu_slice"))
            want.append(oracle.sao_stats(dbk, org, 10, 10, 7, avail))
        f.run(0, 2, 1)          # deblocking only, both slots in one launch
        f.sao_stats(0, 2)       # statistics of both slots in one launch
        for j in range(2):
            assert np.array_equal(f.get_sao_stats(j), want[j]), f"slot {j}"
