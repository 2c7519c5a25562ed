"""CUDA path vs the oracle on seeded synthetic pictures and side information that real streams rarely produce:
every SAO type with random availability patterns, odd picture sizes, 8/10/12-bit with luma and chroma at the same or at different
depths, extreme ALF coefficients."""
import numpy as np
import pytest

import synth

pytestmark = pytest.mark.gpu
K = ("y", "cb", "cr")


def _diff(a, b):
    return {k: int((a[k] != b[k]).sum()) for k in K}


def _one_depth(w, h, bd, *rest):
    return (w, h, bd, bd, *rest)


@pytest.mark.parametrize("w,h,bd_luma,bd_chroma,ctu_log2,seed", synth.keep_ids([(416, 240, 10, 7, 1), (200, 136, 10, 7, 2), (264, 72, 8, 6, 3), (136, 264, 12, 5, 4),
                                                                                 (1920, 1080, 10, 7, 5), (8, 8, 10, 7, 6), (520, 392, 10, 7, 7)], _one_depth) +
                         [(200, 136, 8, 12, 5, 8), (264, 72, 12, 8, 6, 9), (520, 392, 10, 8, 7, 10)])
def test_sao_all_types_random_availability(w, h, bd_luma, bd_chroma, ctu_log2, seed, ilf_lib, oracle):
    rng = np.random.default_rng(seed)
    ctu = 1 << ctu_log2
    cw, ch = (w + ctu - 1) // ctu, (h + ctu - 1) // ctu
    for kind in ("mix", "noise"):
        pic = synth.picture(rng, w, h, bd_luma, kind, bd_chroma=bd_chroma)
        prm = synth.sao_params(rng, cw, ch, bd_luma, p_off=0.2, bd_chroma=bd_chroma)
        want = oracle.sao(pic, bd_luma, bd_chroma, ctu_log2, prm)
        with ilf_lib.InLoopFilter(w, h, bd_luma, bd_chroma, ctu_log2) as f:
            f.upload(0, *(pic[k] for k in K))
            f.set_sao_params(0, prm)
            f.sao_process(0)
            got = f.download(0)
        d = _diff(got, want)
        assert not any(d.values()), f"{kind}: mismatching samples {d}"


def test_sao_component_off_for_whole_picture_is_skipped(ilf_lib, oracle):
    rng = np.random.default_rng(11)
    w, h = 416, 240
    pic = synth.picture(rng, w, h)
    prm = synth.sao_params(rng, 4, 2, p_off=0.0).view(synth.SAO_DT).reshape(-1).copy()
    prm["type"][:, 1] = -1          # Cb off everywhere
    prm = prm.view(np.uint8).reshape(-1, 32)
    want = oracle.sao(pic, 10, 10, 7, prm)
    with ilf_lib.InLoopFilter(w, h) as f:
        f.upload(0, *(pic[k] for k in K))
        f.set_sao_params(0, prm)
        f.sao_process(0)
        got = f.download(0)
    assert not any(_diff(got, want).values())
    assert np.array_equal(got["cb"], pic["cb"])


# (the cases written with one depth run at CTU 128)
@pytest.mark.parametrize("w,h,bd_luma,bd_chroma,ctu_log2,is7,seed",
                         synth.keep_ids([(416, 240, 10, True, 1), (200, 136, 10, False, 2), (264, 72, 8, True, 3), (136, 264, 12, True, 4), (1920, 1080, 10, True, 5)],
                                        lambda w, h, bd, is7, seed: (w, h, bd, bd, 7, is7, seed)) +
                         [(200, 136, 8, 12, 5, True, 6), (264, 72, 12, 8, 6, False, 7), (520, 392, 10, 8, 5, True, 8), (136, 264, 12, 8, 7, True, 9)])
def test_alf_random_coefficients(w, h, bd_luma, bd_chroma, ctu_log2, is7, seed, ilf_lib, oracle):
    rng = np.random.default_rng(seed)
    ctu = 1 << ctu_log2
    cw, ch = (w + ctu - 1) // ctu, (h + ctu - 1) // ctu
    # small coefficients and the limits of the dot-product path (IDP.2A, ilf_alf_tab.cuh); anything in +-511: general path
    for kind, big, dot, path in (("mix", False, False, 3), ("noise", False, True, 3), ("noise", True, False, 0), ("mix", False, True, 3)):
        pic = synth.picture(rng, w, h, bd_luma, kind, bd_chroma=bd_chroma)
        pb, en = synth.alf_params(rng, cw, ch, is7, big=big, dot=dot)
        want = oracle.alf(pic, bd_luma, bd_chroma, ctu_log2, pb, en)
        with ilf_lib.InLoopFilter(w, h, bd_luma, bd_chroma, ctu_log2) as f:
            f.upload(0, *(pic[k] for k in K))
            f.set_alf_params(0, pb, en)
            assert f.alf_path(0) == path, "the arithmetic path the host chose is not the one this case is meant to cover"
            f.alf_process(0)
            got = f.download(0)
            cls = f.alf_classify(0)
        d = _diff(got, want)
        assert not any(d.values()), f"{kind} big={big} dot={dot}: mismatching samples {d}"


# (the small and odd geometries exercise the tile queue of the deblocking kernel: fewer tiles than CTAs or ring stages, a last tile
# of 8 columns, pictures narrower than a tile, the right-hand tile edge on and off the picture border)
@pytest.mark.parametrize("w,h,bd_luma,bd_chroma,ctu_log2,mv32,seed",
                         synth.keep_ids([(416, 240, 10, 7, False, 31), (200, 136, 8, 5, True, 32), (264, 200, 12, 6, False, 33), (1920, 1080, 10, 7, True, 34), (16, 16, 10, 5, False, 35),
                                         (136, 40, 10, 7, False, 36), (128, 32, 8, 6, True, 37), (384, 64, 10, 7, False, 38), (392, 72, 10, 6, True, 39)], _one_depth) +
                         [(200, 136, 8, 12, 5, True, 40), (264, 200, 12, 8, 6, False, 41), (392, 72, 10, 8, 6, True, 42), (520, 392, 12, 10, 7, False, 43)])
def test_deblock_stress_side_information(w, h, bd_luma, bd_chroma, ctu_log2, mv32, seed, ilf_lib, oracle):
    """Deblocking with side information the committed streams do not produce: three slices with their own beta / tc offsets,
    no-filter (PCM / lossless) units, two reference lists with four MV components, a chroma-tree layer, the whole QP range,
    chroma QP offsets, 32-bit MVs with the 1/16-pel threshold -- CUDA == oracle, bit-exact.  The cases at two depths also draw
    the negative QPs of their luma depth and chroma QP offsets up to +-12 (the cases at one depth keep the draws they were
    written with)."""
    rng = np.random.default_rng(seed)
    wide = {} if bd_luma == bd_chroma else {"bd_luma": bd_luma, "chroma_qp_offset": 12}
    for kind in ("mix", "noise"):
        pic = synth.picture(rng, w, h, bd_luma, kind, bd_chroma=bd_chroma)
        si = synth.deblock_info_stress(rng, w, h, ctu_log2, mv32, **wide)
        want = oracle.deblock(pic, bd_luma, bd_chroma, ctu_log2, si["db_params"], si["db_info"], si["db_info_c"], si.get("db_mv16"), si.get("db_mv32"), si["ctu_slice"])
        with ilf_lib.InLoopFilter(w, h, bd_luma, bd_chroma, ctu_log2) as f:
            f.upload(0, *(pic[k] for k in K))
            f.set_deblock_info(0, si["db_params"], si["db_info"], si["db_info_c"], si.get("db_mv16"), si.get("db_mv32"), si["ctu_slice"])
            f.loop_filter_pic(0)
            got = f.download(0)
        d = _diff(got, want)
        assert not any(d.values()), f"{kind}: mismatching samples {d}"
        if kind == "mix":
            assert any((got[k] != pic[k]).any() for k in K)      # and something was filtered
