"""Post-filter consumers on the device (SURVEY.md 8f rank 4): decoded-picture hash CRC / checksum (ilf_picture_hash) and the
download that writes Picture::extendPicBorder's margins (ilf_download_extended) -- CUDA path == oracle (the oracle is pinned to
the reference's own compCRC / compChecksum / extendPicBorder in tests/test_oracle_units.py)."""
import numpy as np
import pytest

import golden_io as G
import synth

pytestmark = pytest.mark.gpu
K = ("y", "cb", "cr")


# (8, 10): one byte per luma sample and two per chroma sample; (12, 8) the other way round
@pytest.mark.parametrize("w,h,bd_luma,bd_chroma,seed",
                         synth.keep_ids([(416, 240, 10, 1), (200, 136, 10, 2), (264, 72, 8, 3), (136, 264, 12, 4), (8, 8, 10, 5), (1920, 1080, 10, 6), (3840, 2160, 10, 7)],
                                        lambda w, h, bd, s: (w, h, bd, bd, s)) +
                         [(200, 136, 8, 10, 8), (264, 72, 12, 8, 9)])
def test_picture_hash_matches_oracle(w, h, bd_luma, bd_chroma, seed, ilf_lib, oracle):
    rng = np.random.default_rng(seed)
    pic = synth.picture(rng, w, h, bd_luma, "noise", bd_chroma=bd_chroma)
    with ilf_lib.InLoopFilter(w, h, bd_luma, bd_chroma, 7) as f:
        f.upload(0, *(pic[k] for k in K))
        for kind in ("crc", "checksum"):
            assert f.picture_hash(0, kind) == oracle.picture_hash(pic, bd_luma, bd_chroma, kind), kind


def test_picture_hash_follows_the_filtered_picture(ilf_lib, oracle):
    """The hash is taken of the slot's CURRENT picture: after the chain it equals the hash of the reference's filtered output."""
    c = G.load_golden([p for p in G.golden_files() if "ra_416x240_01" in p][0])
    g = c["geom"]
    with ilf_lib.InLoopFilter(g["width"], g["height"], g["bd_luma"], g["bd_chroma"], g["ctu_log2"]) as f:
        f.upload(0, *(c[f"pre_{k}"] for k in K))
        f.set_deblock_info(0, c["db_params"].tobytes(), c["db_info"], c.get("db_info_c"), c["db_mv32"].astype(np.int16), None, c["ctu_slice"])
        f.set_sao_params(0, c["sao_ctus"])
        f.set_alf_params(0, c["alf_params"].tobytes(), c["alf_ctu_enable"])
        f.run(0, 1, 7)
        want = {k: c[f"alf_{k}"] for k in K}
        for kind in ("crc", "checksum"):
            assert f.picture_hash(0, kind) == oracle.picture_hash(want, g["bd_luma"], g["bd_chroma"], kind)


@pytest.mark.parametrize("w,h,margin", [(416, 240, 144), (200, 136, 16), (1920, 1080, 144)])
def test_download_extended_matches_oracle(w, h, margin, ilf_lib, oracle):
    rng = np.random.default_rng(w)
    pic = synth.picture(rng, w, h, 10, "noise")
    with ilf_lib.InLoopFilter(w, h) as f:
        f.upload(0, *(pic[k] for k in K))
        got = f.download_extended(0, margin)
    for k, s in (("y", 0), ("cb", 1), ("cr", 1)):
        assert np.array_equal(got[k], oracle.extend_border(pic[k], margin >> s, margin >> s)), k
