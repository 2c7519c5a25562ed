"""CTU-row band mode on the GPU (BASELINE config 4): band contexts with 16 halo rows, halo pulled from the neighbouring
contexts' input planes (same process here: device-to-device copies; across processes the same entry points use CUDA IPC),
every band filtered on its own -- the bands' own rows must equal the whole-picture result bit for bit."""
import numpy as np
import pytest

import golden_io as G
import synth
from vvcsoftware_vtm_b200 import bands

pytestmark = pytest.mark.gpu
K = ("y", "cb", "cr")


def _run_whole(v, w, h, bd_luma, bd_chroma, ctu_log2, pic, si):
    with v.InLoopFilter(w, h, bd_luma, bd_chroma, ctu_log2) as f:
        f.upload(0, *(pic[k] for k in K))
        f.set_deblock_info(0, si["db_params"], si["db_info"], si.get("db_info_c"), si.get("db_mv16"), si.get("db_mv32"), si.get("ctu_slice"))
        f.set_sao_params(0, si["sao_ctus"])
        f.set_alf_params(0, si["alf_params"], si["alf_ctu_enable"])
        f.run(0, 1, 7)
        return f.download(0)


def _run_banded(v, w, h, bd_luma, bd_chroma, ctu_log2, pic, si, n, devices=1):
    ctu = 1 << ctu_log2
    part = bands.band_partition((h + ctu - 1) // ctu, n)
    ctxs = [v.InLoopFilter(w, h, bd_luma, bd_chroma, ctu_log2, band=b, device=r % devices) for r, b in enumerate(part)]
    try:
        for f in ctxs:
            assert (f.own_row0, f.own_rows, f.row0, f.rows) == bands.band_rows(h, ctu_log2, part[ctxs.index(f)])
            y0, y1 = f.own_row0, f.own_row0 + f.own_rows
            f.upload_band(0, pic["y"][y0:y1], pic["cb"][y0 // 2:y1 // 2], pic["cr"][y0 // 2:y1 // 2])   # own rows only
        for f in ctxs:
            f.sync()
        handles = [f.band_export(0) for f in ctxs]
        for r, f in enumerate(ctxs):
            bands.connect_bands(f, 0, r, n, handles)
            f.band_exchange(0)
            s = bands.slice_side_info(si, f.row0, f.rows)
            f.set_deblock_info(0, s["db_params"], s["db_info"], s.get("db_info_c"), s.get("db_mv16"), s.get("db_mv32"), s.get("ctu_slice"))
            f.set_sao_params(0, s["sao_ctus"])
            f.set_alf_params(0, s["alf_params"], s["alf_ctu_enable"])
            f.run(0, 1, 7)
        outs = [f.download_band(0) for f in ctxs]
        return {k: np.concatenate([o[k] for o in outs]) for k in K}
    finally:
        for f in ctxs:
            f.close()


# (the cases written before the bit depths were a parameter run at 10 bit)
@pytest.mark.parametrize("w,h,bd_luma,bd_chroma,ctu_log2,n,seed",
                         synth.keep_ids([(200, 136, 5, 2, 21), (200, 136, 5, 3, 22), (264, 200, 5, 4, 23), (416, 240, 6, 2, 24), (1920, 1080, 7, 3, 25)],
                                        lambda w, h, c, n, s: (w, h, 10, 10, c, n, s)) +
                         [(264, 200, 12, 8, 5, 3, 26)])
def test_bands_equal_whole_picture_synthetic(w, h, bd_luma, bd_chroma, ctu_log2, n, seed, ilf_lib, oracle):
    rng = np.random.default_rng(seed)
    ctu = 1 << ctu_log2
    cw, ch = (w + ctu - 1) // ctu, (h + ctu - 1) // ctu
    pic = synth.picture(rng, w, h, bd_luma, bd_chroma=bd_chroma)
    prm, info, mv16 = synth.deblock_info(rng, w, h, inter=True)
    alf_bytes, en = synth.alf_params(rng, cw, ch, is7=True, p_on=0.9)
    si = {"db_params": prm, "db_info": info, "db_mv16": mv16, "sao_ctus": synth.sao_params(rng, cw, ch, bd_luma, p_off=0.1, bd_chroma=bd_chroma),
          "alf_params": alf_bytes, "alf_ctu_enable": en}
    whole = _run_whole(ilf_lib, w, h, bd_luma, bd_chroma, ctu_log2, pic, si)
    banded = _run_banded(ilf_lib, w, h, bd_luma, bd_chroma, ctu_log2, pic, si, n)
    d = {k: int((whole[k] != banded[k]).sum()) for k in K}
    assert not any(d.values()), f"banded != whole picture: {d}"
    if h <= 256:   # and the whole-picture result is the oracle's
        want = oracle.deblock(pic, bd_luma, bd_chroma, ctu_log2, prm, info, None, mv16, None, None)
        want = oracle.sao(want, bd_luma, bd_chroma, ctu_log2, si["sao_ctus"])
        want = oracle.alf(want, bd_luma, bd_chroma, ctu_log2, alf_bytes, en)
        d = {k: int((whole[k] != want[k]).sum()) for k in K}
        assert not any(d.values()), f"whole picture != oracle: {d}"


def test_bands_equal_reference_capture(ilf_lib):
    c = G.load_golden([p for p in G.golden_files() if "ra_416x240_05" in p][0])
    g = c["geom"]
    pic = {k: c["pre_" + k] for k in K}
    si = {"db_params": c["db_params"].tobytes(), "db_info": c["db_info"], "db_info_c": c.get("db_info_c"), "db_mv32": c["db_mv32"], "ctu_slice": c["ctu_slice"],
          "sao_ctus": c["sao_ctus"], "alf_params": c["alf_params"].tobytes(), "alf_ctu_enable": c["alf_ctu_enable"]}
    got = _run_banded(ilf_lib, g["width"], g["height"], g["bd_luma"], g["bd_chroma"], g["ctu_log2"], pic, si, 2)
    for k in K:
        assert np.array_equal(got[k], c["alf_" + k]), f"plane {k}: banded result differs from the reference's picture"


def test_bands_on_two_devices_in_one_process(ilf_lib):
    """Band contexts on different GPUs of ONE process: the halo exchange goes through peer access (NVLink P2P) instead of
    CUDA IPC, and every device needs its own kernel attributes.  Skipped on a one-GPU box."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    c = G.load_golden([p for p in G.golden_files() if "ra_416x240_05" in p][0])
    g = c["geom"]
    pic = {k: c["pre_" + k] for k in K}
    si = {"db_params": c["db_params"].tobytes(), "db_info": c["db_info"], "db_info_c": c.get("db_info_c"), "db_mv32": c["db_mv32"], "ctu_slice": c["ctu_slice"],
          "sao_ctus": c["sao_ctus"], "alf_params": c["alf_params"].tobytes(), "alf_ctu_enable": c["alf_ctu_enable"]}
    got = _run_banded(ilf_lib, g["width"], g["height"], g["bd_luma"], g["bd_chroma"], g["ctu_log2"], pic, si, 2, devices=2)
    for k in K:
        assert np.array_equal(got[k], c["alf_" + k]), f"plane {k}: banded result differs from the reference's picture"
