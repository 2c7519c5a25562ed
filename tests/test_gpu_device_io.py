"""Pictures to and from device memory (ilf_upload_device, ilf_set_original_device, ilf_download_device) against the host path.

The host transfers are pinned to the oracle and the reference captures by the other tests, so every result here is compared with
what ilf_upload / ilf_set_original / ilf_download give for the same picture.  The sample conversion is compared with a numpy
statement of the rule in include/ilf_b200.h.  The error cases only pass arguments the library must refuse before it enqueues
anything."""
import ctypes as C
import os

import numpy as np
import pytest

import golden_io as G
import synth
import test_gpu_geometry as TG
from vvcsoftware_vtm_b200 import bands

pytestmark = pytest.mark.gpu
K = ("y", "cb", "cr")
ERR_ARG, ERR_STATE = -1, -3
CANDS = [(0, 0), (2, -3), (-5, 4), (6, 6)]
SHIFT = (1, 2)


# ---- helpers ---------------------------------------------------------------------------------------
def _torch():
    import torch
    return torch


def _dev(pic, device=0):
    """numpy planes -> int16 / uint8 CUDA tensors (a copy)."""
    torch = _torch()
    return {k: torch.from_numpy(np.ascontiguousarray(pic[k])).to(f"cuda:{device}") for k in K}


def _host(t):
    _torch().cuda.synchronize()
    return {k: t[k].cpu().numpy() for k in K}


def _same(a, b):
    return all(np.array_equal(a[k], b[k]) for k in K)


def _diff(a, b):
    return {k: int((np.asarray(a[k]) != np.asarray(b[k])).sum()) for k in K if not np.array_equal(a[k], b[k])}


def convert(v, src_depth, dst_depth, dst_dtype):
    """The rule of ilf_b200.h: int16 containers hold unsigned samples; d > 0 shifts left, d < 0 rounds, shifts and clips, d = 0
    copies; the result is stored as the destination type (its low bits)."""
    v = np.asarray(v)
    x = (v.view(np.uint16) if v.dtype == np.int16 else v).astype(np.int64)
    d = dst_depth - src_depth
    if d > 0:
        r = x << d
    elif d < 0:
        r = np.clip((x + (1 << (-d - 1))) >> -d, 0, (1 << dst_depth) - 1)
    else:
        r = x
    if dst_dtype == np.int16:
        return (r & 0xFFFF).astype(np.uint16).view(np.int16)
    return (r & 0xFF).astype(np.uint8)


def _cap_inputs(c):
    """Planes, side information (in the form of test_gpu_geometry.inputs) and the stages the capture carries."""
    mv = c["db_mv32"]
    fits = np.abs(mv).max(initial=0) < 32768
    si = {"db_params": c["db_params"].tobytes(), "db_info": c["db_info"], "db_info_c": c.get("db_info_c"),
          "db_mv16": np.ascontiguousarray(mv.astype(np.int16)) if fits else None, "db_mv32": None if fits else mv, "ctu_slice": c["ctu_slice"]}
    stages = 1
    if "sao_ctus" in c:
        si["sao_ctus"], si["alf_params"], si["alf_ctu_enable"] = c["sao_ctus"], c["alf_params"].tobytes(), c["alf_ctu_enable"]
        stages = 7
    return {k: c["pre_" + k] for k in K}, si, stages


def _side(f, slot, si, stages=7):
    f.set_deblock_info(slot, *TG._db_args(si))
    if stages & 2:
        f.set_sao_params(slot, si["sao_ctus"])
    if stages & 4:
        f.set_alf_params(slot, si["alf_params"], si["alf_ctu_enable"])


def _avail(w, h, ctu_log2):
    cw, ch = TG._ctus(w, h, ctu_log2)
    cx, cy = np.meshgrid(np.arange(cw), np.arange(ch))
    return ((cx > 0) * 0x01 | (cy > 0) * 0x04 | ((cx > 0) & (cy > 0)) * 0x10).astype(np.uint8).ravel()


def _three_ways(ilf_lib, w, h, bl, bc, ctu_log2, pic, si, stages):
    """(host upload + run + host download, device upload + run + host download, host upload + run + device download)."""
    out = []
    with ilf_lib.InLoopFilter(w, h, bl, bc, ctu_log2) as f:
        for up_dev, down_dev in ((False, False), (True, False), (False, True)):
            if up_dev:
                f.upload_device(0, *_dev(pic).values())
            else:
                f.upload(0, *(pic[k] for k in K))
            _side(f, 0, si, stages)
            f.run(0, 1, stages)
            out.append(_host(f.download_device(0)) if down_dev else f.download(0))
    return out


# ---- 1. same results as the host path --------------------------------------------------------------------
@pytest.mark.parametrize("path", [os.path.basename(p) for p in G.golden_files()])
def test_captures_equal_host_path(path, ilf_lib):
    c = G.load_golden(os.path.join(G.GOLDEN_DIR, path))
    g = c["geom"]
    pic, si, stages = _cap_inputs(c)
    host, up, down = _three_ways(ilf_lib, g["width"], g["height"], g["bd_luma"], g["bd_chroma"], g["ctu_log2"], pic, si, stages)
    if stages == 7:
        assert _same(host, {k: c["alf_" + k] for k in K}), "host path differs from the reference capture"
    assert _same(up, host), f"device upload: {_diff(up, host)}"
    assert _same(down, host), f"device download: {_diff(down, host)}"


# 416x240 and widths whose half is not a multiple of 8; CTU 32, 64, 128; 8, 10, 12 bit, luma != chroma
SYNTH = [(416, 240, 7, 10, 10), (264, 136, 5, 8, 12), (200, 136, 6, 12, 10), (328, 72, 7, 10, 8), (136, 264, 5, 12, 8), (416, 240, 6, 8, 10)]


@pytest.mark.parametrize("w,h,c,bl,bc", SYNTH, ids=[f"{w}x{h}-ctu{1 << c}-{bl}-{bc}" for w, h, c, bl, bc in SYNTH])
def test_synthetic_equal_host_path(w, h, c, bl, bc, ilf_lib):
    pic, _, si = TG.inputs(4000 + w + h + c, w, h, c, bl, bc, ("none", "mv16", "mv32")[c - 5], c != 6, c != 7, ("dot", "big")[c % 2])
    host, up, down = _three_ways(ilf_lib, w, h, bl, bc, c, pic, si, 7)
    assert _same(up, host), f"device upload: {_diff(up, host)}"
    assert _same(down, host), f"device download: {_diff(down, host)}"


def test_batch_on_lanes_equals_host_path(ilf_lib):
    """Eight slots uploaded from tensors, one batched chain (dealt to the lanes), eight device downloads."""
    caps = [G.load_golden(p) for p in G.golden_files() if os.path.basename(p).startswith(("ra_", "ldp_", "ldb_", "intra_"))]
    assert len(caps) >= 8
    caps = caps[:8]
    g = caps[0]["geom"]
    ins = [_cap_inputs(c) for c in caps]
    with ilf_lib.InLoopFilter(g["width"], g["height"], g["bd_luma"], g["bd_chroma"], g["ctu_log2"], num_slots=8) as f:
        for i, (pic, si, _) in enumerate(ins):
            f.upload_device(i, *_dev(pic).values())
            _side(f, i, si)
        f.run(0, 8, 7)
        got = [f.download_device(i) for i in range(8)]
        got = [_host(t) for t in got]
    for i, c in enumerate(caps):
        assert _same(got[i], {k: c["alf_" + k] for k in K}), f"slot {i}: {_diff(got[i], {k: c['alf_' + k] for k in K})}"


# ---- 2. partial chains and planes left in buffer 0 or 1 ---------------------------------------------------------
def _chroma_off(si, intra):
    s = dict(si) if intra else TG._intra_free(si)
    sao = si["sao_ctus"].reshape(-1).view(synth.SAO_DT).copy()
    sao["type"][:, 1:] = -1
    s["sao_ctus"] = sao.view(np.uint8).reshape(-1, 32)
    en = si["alf_ctu_enable"].copy()
    en[1:] = 0
    s["alf_ctu_enable"] = en
    return s


@pytest.mark.parametrize("case", ["deblock", "deblock_sao", "chroma_in_buffer0", "chroma_in_buffer1"])
def test_partial_chains(case, ilf_lib):
    w, h, c, bl, bc = 264, 136, 6, 10, 8
    pic, _, si = TG.inputs(77, w, h, c, bl, bc, "mv16", True, True, "dot")
    stages = {"deblock": 1, "deblock_sao": 3}.get(case, 7)
    if case.startswith("chroma"):
        si = _chroma_off(si, intra=case.endswith("1"))
    with ilf_lib.InLoopFilter(w, h, bl, bc, c) as f:
        f.upload_device(0, *_dev(pic).values())
        _side(f, 0, si)
        f.run(0, 1, stages)
        got = _host(f.download_device(0))
        want = f.download(0)
    if case == "chroma_in_buffer0":
        assert all(np.array_equal(want[k], pic[k]) for k in ("cb", "cr")), "chroma should be the uploaded planes"
    assert _same(got, want), _diff(got, want)


# ---- 3. conversion -------------------------------------------------------------------------------------------------------
CW, CH, CC = 64, 16, 5


def _edge_values(rng, shape, depth, dtype):
    """Samples over [0, 2^depth - 1] with the top values (where rounding carries) and 0 frequent."""
    top = (1 << depth) - 1
    v = rng.integers(0, top + 1, shape)
    pick = rng.random(shape)
    v[pick < 0.2] = top
    v[(pick >= 0.2) & (pick < 0.3)] = top - 1
    v[(pick >= 0.3) & (pick < 0.35)] = 0
    return v.astype(np.uint16).view(np.int16) if dtype == np.int16 else v.astype(np.uint8)


def _pic_at(rng, depths, dtype, w=CW, h=CH):
    return {k: _edge_values(rng, (h >> (k != "y"), w >> (k != "y")), depths[k != "y"], dtype) for k in K}


def _conv(pic, src, dst, dtype):
    return {k: convert(pic[k], src[k != "y"], dst[k != "y"], dtype) for k in K}


def _stats(f, slot=0):
    f.sao_stats(slot, 1)
    return f.get_sao_stats(slot)


@pytest.mark.parametrize("b", range(8, 13))
def test_conversion_matches_rule(b, ilf_lib):
    """Every caller depth 8..16 (int16) and uint8 against a context of luma depth b (chroma: another depth): upload, original
    (through the SAO statistics it feeds) and download."""
    torch = _torch()
    bc = 8 + (b - 8 + 2) % 5
    ctx_d = (b, bc)
    rng = np.random.default_rng(b)
    avail = _avail(CW, CH, CC)
    with ilf_lib.InLoopFilter(CW, CH, b, bc, CC) as f:
        for dtype, cs in ((np.int16, range(8, 17)), (np.uint8, (8,))):
            tdt = torch.int16 if dtype == np.int16 else torch.uint8
            for cdep in cs:
                for caller in ((cdep, cdep), (cdep, 16 if dtype == np.int16 else 8)):
                    tag = f"context {ctx_d}, caller {caller} {dtype.__name__}"
                    bd = caller if dtype == np.int16 else None
                    # upload: caller -> context
                    src = _pic_at(rng, caller, dtype)
                    f.upload_device(0, *_dev(src).values(), bit_depth=bd)
                    assert _same(f.download(0), _conv(src, caller, ctx_d, np.int16)), f"upload, {tag}"
                    # download: context -> caller
                    pic = _pic_at(rng, ctx_d, np.int16)
                    f.upload(0, *(pic[k] for k in K))
                    got = _host(f.download_device(0, dtype=tdt, bit_depth=bd))
                    assert _same(got, _conv(pic, ctx_d, caller, dtype)), f"download, {tag}"
                    # original: caller -> context, seen through the statistics against the host original
                    org = _pic_at(rng, caller, dtype)
                    f.set_original_device(0, *_dev(org).values(), avail, bit_depth=bd)
                    got = _stats(f)
                    want_org = _conv(org, caller, ctx_d, np.int16)
                    f.set_original(0, *(want_org[k] for k in K), avail)
                    assert np.array_equal(got, _stats(f)), f"original, {tag}"


def test_uint8_round_trip_through_10_bit(ilf_lib):
    torch = _torch()
    rng = np.random.default_rng(8)
    src = _pic_at(rng, (8, 8), np.uint8, 264, 136)
    with ilf_lib.InLoopFilter(264, 136, 10, 10, 6) as f:
        f.upload_device(0, *_dev(src).values())
        assert _same(f.download(0), {k: src[k].astype(np.int16) << 2 for k in K})
        assert _same(_host(f.download_device(0, dtype=torch.uint8)), src)


# ---- 4. original -------------------------------------------------------------------------------------------------------
def _encoder_records(f, pic, si, set_org):
    """SAO statistics of the deblocked picture, ALF statistics of the SAO'd one and the deblocking search, against set_org's original."""
    f.upload(0, *(pic[k] for k in K))
    _side(f, 0, si)
    set_org(f)
    f.run(0, 1, 1)
    sao = _stats(f)
    f.run(0, 1, 2)
    f.alf_stats(0, 1)
    alf = f.get_alf_stats(0)
    f.deblock_search(CANDS, SHIFT)
    return sao, alf, f.get_deblock_search(0)


@pytest.mark.parametrize("case", ["capture", "synthetic-12-8", "uint8-capture", "uint8-synthetic"])
def test_original_equals_host(case, ilf_lib):
    if "capture" in case:
        c = G.load_golden([p for p in G.golden_files() if "ra_416x240_05" in p][0])
        g = c["geom"]
        w, h, ctu, bl, bc = g["width"], g["height"], g["ctu_log2"], g["bd_luma"], g["bd_chroma"]
        pic, si, _ = _cap_inputs(c)
        avail = _avail(w, h, ctu)
        org = {k: np.clip(pic[k].astype(np.int32) + np.random.default_rng(1).integers(-9, 10, pic[k].shape), 0, 1023).astype(np.int16) for k in K}
    else:
        w, h, ctu = 264, 136, 5
        bl, bc = (12, 8) if "12" in case else (10, 10)
        pic, org, si = TG.inputs(91, w, h, ctu, bl, bc, "mv16", True, True, "dot")
        avail = si["avail"]
    if case.startswith("uint8"):
        assert (bl, bc) == (10, 10)
        org8 = {k: (np.random.default_rng(2).integers(0, 256, org[k].shape)).astype(np.uint8) for k in K}
        org8["y"][:4] = 255
        dev_org, host_org = _dev(org8), {k: org8[k].astype(np.int16) << 2 for k in K}
    else:
        dev_org, host_org = _dev(org), org
    with ilf_lib.InLoopFilter(w, h, bl, bc, ctu) as f:
        got = _encoder_records(f, pic, si, lambda f: f.set_original_device(0, *dev_org.values(), avail))
        want = _encoder_records(f, pic, si, lambda f: f.set_original(0, *(host_org[k] for k in K), avail))
    for name, a, b in zip(("SAO statistics", "ALF statistics", "search sums"), got, want):
        assert np.array_equal(a, b), name


# ---- 5. strides and views -------------------------------------------------------------------------------------------------
def _views(full, w, h, col0):
    return {k: full[k][:, (col0 >> (k != "y")):(col0 >> (k != "y")) + (w >> (k != "y"))] for k in K}


def _outside(full, w, col0, sentinel):
    """Every sample of `full` outside the picture's columns still holds `sentinel`."""
    for k in K:
        a = full[k].cpu().numpy()
        c0, cw = col0 >> (k != "y"), w >> (k != "y")
        if not ((a[:, :c0] == sentinel).all() and (a[:, c0 + cw:] == sentinel).all()):
            return k
    return None


def test_slices_of_wider_tensors(ilf_lib):
    torch = _torch()
    w, h, c = 264, 136, 5
    pic = synth.picture(np.random.default_rng(5), w, h, 10, "noise")
    col0, pad = 24, 72
    src_full = {k: torch.full((h >> (k != "y"), (w + pad) >> (k != "y")), -3, dtype=torch.int16, device="cuda:0") for k in K}
    dst_full = {k: torch.full_like(src_full[k], -7) for k in K}
    src, dst = _views(src_full, w, h, col0), _views(dst_full, w, h, col0)
    for k in K:
        src[k].copy_(torch.from_numpy(pic[k]))
    with ilf_lib.InLoopFilter(w, h, 10, 10, c) as f:
        f.upload_device(0, *src.values())
        assert _same(f.download(0), pic)
        f.download_device(0, out=dst)
        assert _same(_host(dst), pic)
    assert _outside(dst_full, w, col0, -7) is None, "the download wrote outside the picture's columns"


def _strided(buf, shape, pitch, offset):
    return buf.as_strided(shape, (pitch, 1), offset)


@pytest.mark.parametrize("dtype", ["uint8", "int16"])
def test_odd_pitches_and_offsets(dtype, ilf_lib):
    """Views with odd pitches (in samples) and base offsets that are not 16-byte aligned: the body of a row cannot be moved in
    16-byte words, or only after a head of samples."""
    torch = _torch()
    w, h, c = 264, 136, 5
    tdt, ndt = (torch.uint8, np.uint8) if dtype == "uint8" else (torch.int16, np.int16)
    rng = np.random.default_rng(11)
    src = _pic_at(rng, (8, 8) if dtype == "uint8" else (10, 10), ndt, w, h)
    with ilf_lib.InLoopFilter(w, h, 10, 10, c) as f:
        for pitch_pad, off in ((3, 5), (1, 1), (17, 9), (16, 8), (0, 3)):
            sentinel = 0x5A
            bufs = {k: torch.full(((h >> (k != "y")) * ((w >> (k != "y")) + pitch_pad) + off + 32,), sentinel, dtype=tdt, device="cuda:0") for k in K}
            views = {k: _strided(bufs[k], (h >> (k != "y"), w >> (k != "y")), (w >> (k != "y")) + pitch_pad, off + (k != "y")) for k in K}
            for k in K:
                views[k].copy_(torch.from_numpy(src[k]))
            f.upload_device(0, *views.values())
            want_ctx = {k: src[k].astype(np.int16) << 2 for k in K} if dtype == "uint8" else src
            assert _same(f.download(0), want_ctx), f"upload, pitch +{pitch_pad}, offset {off}"
            for k in K:
                bufs[k].fill_(sentinel)
            f.download_device(0, out=views)
            got = _host(views)
            assert _same(got, src), f"download, pitch +{pitch_pad}, offset {off}: {_diff(got, src)}"
            for k in K:
                a = bufs[k].cpu().numpy()
                mask = np.ones(a.shape, bool)
                pitch, rows, cols = (w >> (k != "y")) + pitch_pad, h >> (k != "y"), w >> (k != "y")
                base = off + (k != "y")
                for r in range(rows):
                    mask[base + r * pitch: base + r * pitch + cols] = False
                assert (a[mask] == sentinel).all(), f"plane {k}: written outside the view (pitch +{pitch_pad}, offset {off})"


# ---- 6. bands -----------------------------------------------------------------------------------------------------------
def _band_ctxs(ilf_lib, w, h, bl, bc, ctu_log2, n, devices):
    part = bands.band_partition((h + (1 << ctu_log2) - 1) >> ctu_log2, n)
    return [ilf_lib.InLoopFilter(w, h, bl, bc, ctu_log2, band=b, device=r % devices) for r, b in enumerate(part)]


def _own(pic, f):
    y0, y1 = f.own_row0, f.own_row0 + f.own_rows
    return {"y": pic["y"][y0:y1], "cb": pic["cb"][y0 // 2:y1 // 2], "cr": pic["cr"][y0 // 2:y1 // 2]}


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_bands_equal_whole_picture(n, ilf_lib):
    torch = _torch()
    devices = min(n, torch.cuda.device_count())
    w, h, c, bl, bc = 264, 520, 6, 10, 8
    pic, org, si = TG.inputs(300 + n, w, h, c, bl, bc, "mv16", True, True, "dot")
    with ilf_lib.InLoopFilter(w, h, bl, bc, c) as f:
        f.upload(0, *(pic[k] for k in K))
        _side(f, 0, si)
        f.run(0, 1, 7)
        whole = f.download(0)
    ctxs = _band_ctxs(ilf_lib, w, h, bl, bc, c, n, devices)
    try:
        for r, f in enumerate(ctxs):
            with torch.cuda.device(r % devices):
                f.upload_device(0, *_dev(_own(pic, f), r % devices).values())
        for f in ctxs:
            f.sync()
        handles = [f.band_export(0) for f in ctxs]
        for r, f in enumerate(ctxs):
            bands.connect_bands(f, 0, r, n, handles)
            f.band_exchange(0)
            _side(f, 0, bands.slice_side_info(si, f.row0, f.rows))
        # the original of the own rows: the statistics and search of the device call equal those of ilf_set_original_band
        for r, f in enumerate(ctxs):
            own = _own(org, f)
            f.run(0, 1, 1)
            f.set_original_device(0, *_dev(own, r % devices).values(), si["avail"])
            got = (_stats(f), (f.alf_stats(0, 1), f.get_alf_stats(0))[1], (f.deblock_search(CANDS, SHIFT), f.get_deblock_search(0))[1])
            f.set_original_band(0, *(own[k] for k in K), si["avail"])
            want = (_stats(f), (f.alf_stats(0, 1), f.get_alf_stats(0))[1], (f.deblock_search(CANDS, SHIFT), f.get_deblock_search(0))[1])
            for name, a, b in zip(("SAO statistics", "ALF statistics", "search sums"), got, want):
                assert np.array_equal(a, b), f"band {r}: {name}"
            f.run(0, 1, 7)
        outs = [_host(f.download_device(0)) for f in ctxs]
    finally:
        for f in ctxs:
            f.close()
    banded = {k: np.concatenate([o[k] for o in outs]) for k in K}
    assert _same(banded, whole), f"bands != whole picture: {_diff(banded, whole)}"


# ---- 7. ordering without host synchronisation ---------------------------------------------------------------------------------
SLEEP = 20_000_000   # GPU cycles, about 10 ms: far longer than any of the calls below takes to issue


def test_input_produced_on_a_side_stream(ilf_lib):
    torch = _torch()
    c = G.load_golden([p for p in G.golden_files() if "ra_416x240_05" in p][0])
    g = c["geom"]
    pic, si, _ = _cap_inputs(c)
    want = {k: c["alf_" + k] for k in K}
    staged = _dev(pic)
    torch.cuda.synchronize()
    with ilf_lib.InLoopFilter(g["width"], g["height"], g["bd_luma"], g["bd_chroma"], g["ctu_log2"]) as f:
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            # produced behind a sleep
            t = {k: torch.zeros_like(staged[k]) for k in K}
            torch.cuda._sleep(SLEEP)
            for k in K:
                t[k].copy_(staged[k])
            f.upload_device(0, *t.values())
            # overwritten right after the call, on the same stream: the upload has the old content
            for k in K:
                t[k].fill_(0)
        _side(f, 0, si)
        f.run(0, 1, 7)
        assert _same(f.download(0), want), "upload: the result is not that of the produced input"
        # the download waits for work issued before it and is waited for by work issued after it, on the caller's stream
        with torch.cuda.stream(side):
            out = {k: torch.empty_like(staged[k]) for k in K}
            torch.cuda._sleep(SLEEP)
            for k in K:
                out[k].fill_(-1)
            f.download_device(0, out=out)
            consumed = {k: out[k].clone() for k in K}
            for k in K:
                out[k].fill_(-2)
        side.synchronize()
        assert _same({k: consumed[k].cpu().numpy() for k in K}, want), "download: consumer did not see the downloaded picture"


def test_device_and_host_transfers_mixed(ilf_lib, monkeypatch):
    """Four slots, device and host uploads and downloads of the same slots issued back to back with no synchronisation, twice, against
    the same calls one slot at a time with a synchronisation after each."""
    monkeypatch.setenv("ILF_RUN_LANES", "2")
    monkeypatch.setenv("ILF_RUN_LANE_MIN", "2")
    torch = _torch()
    caps = [G.load_golden(p) for p in sorted(G.golden_files()) if os.path.basename(p).startswith("ra_416x240")]
    g = caps[0]["geom"]
    ins = [_cap_inputs(c) for c in caps]
    dev_pics = [_dev(p) for p, _, _ in ins]
    n = 4
    lib = ilf_lib.load_library()
    pinned = [ilf_lib.pinned_planes(g["width"], g["height"]) for _ in range(2 * n)]
    try:
        with ilf_lib.InLoopFilter(g["width"], g["height"], g["bd_luma"], g["bd_chroma"], g["ctu_log2"], num_slots=n) as f:
            got = []
            for rnd in range(2):
                for i in range(n):
                    j = (i + rnd) % 4
                    if (i + rnd) % 2:
                        f.upload_device(i, *dev_pics[j].values())
                    else:
                        f.upload(i, *(ins[j][0][k] for k in K))
                    _side(f, i, ins[j][1])
                f.run(0, n, 7)
                for i in range(n):
                    if (i + rnd) % 2:
                        got.append(f.download_device(i))
                    else:
                        f.download_async(i, pinned[rnd * n + i])
                        got.append(pinned[rnd * n + i])
            f.sync()
            got = [{k: (d[k].cpu().numpy() if isinstance(d[k], torch.Tensor) else np.array(d[k])) for k in K} for d in got]
        for rnd in range(2):
            for i in range(n):
                j = (i + rnd) % 4
                assert _same(got[rnd * n + i], {k: caps[j]["alf_" + k] for k in K}), f"round {rnd}, slot {i}"
    finally:
        for p in pinned:
            for k in K:
                lib.ilf_host_free(C.c_void_p(p[k].ctypes.data))


# ---- 8. errors ---------------------------------------------------------------------------------------------------------------
W8, H8, C8 = 264, 136, 6


@pytest.fixture
def loaded(ilf_lib):
    """A context whose slot 0 holds a filtered picture, and a check that a refused call left the slot's picture and state alone (the
    side information is still set, so a run needs no new upload or parameters, and gives the same picture)."""
    pic, org, si = TG.inputs(55, W8, H8, C8, 10, 10, "mv16", True, True, "dot")
    f = ilf_lib.InLoopFilter(W8, H8, 10, 10, C8)
    f.upload(0, *(pic[k] for k in K))
    _side(f, 0, si)
    f.set_original(0, *(org[k] for k in K), si["avail"])
    f.run(0, 1, 7)
    want = f.download(0)
    f.deblock_search(CANDS, SHIFT)
    want_search = f.get_deblock_search(0)

    def unchanged():
        assert _same(f.download(0), want), "the picture changed"
        f.run(0, 1, 7)
        assert _same(f.download(0), want), "the slot's side information was reset"
        f.deblock_search(CANDS, SHIFT)   # ILF_ERR_STATE if the original had become stale
        assert np.array_equal(f.get_deblock_search(0), want_search)

    yield f, pic, org, si, unchanged
    f.close()


def _args(planes):
    out = []
    for a in planes:
        if isinstance(a, tuple):
            out += [C.c_void_p(a[0]), a[1]]
        elif isinstance(a, np.ndarray):
            out += [C.c_void_p(a.ctypes.data), a.strides[0] // a.itemsize]
        else:
            out += [C.c_void_p(a.data_ptr()), a.stride(0)]
    return out


def _dev_call(f, name, planes, fmt=None, avail=None, stream=None, slot=0):
    """The C entry point `name` on slot `slot` with raw arguments (planes: tensors, numpy arrays or (pointer, stride) pairs)."""
    fp = C.byref(fmt) if fmt is not None else None
    st = C.c_void_p(stream)
    if name == "ilf_set_original_device":
        av = avail if avail is not None else np.zeros(1, np.uint8)
        return getattr(f._lib, name)(f._h, slot, *_args(planes), av.ctypes.data_as(C.c_void_p) if isinstance(av, np.ndarray) else av, fp, st)
    return getattr(f._lib, name)(f._h, slot, *_args(planes), fp, st)


DEVICE_CALLS = ["ilf_upload_device", "ilf_download_device", "ilf_set_original_device"]


@pytest.mark.parametrize("name", DEVICE_CALLS)
@pytest.mark.parametrize("mem", ["pageable", "pinned"])
def test_host_memory_refused_by_device_calls(name, mem, loaded, ilf_lib):
    f, pic, org, si, unchanged = loaded
    planes = {k: np.ascontiguousarray(pic[k]) for k in K}
    keep = None
    if mem == "pinned":
        keep = ilf_lib.pinned_planes(W8, H8)
        for k in K:
            keep[k][...] = pic[k]
        planes = keep
    try:
        assert _dev_call(f, name, [planes[k] for k in K], avail=si["avail"]) == ERR_ARG
        assert "device memory" in f._lib.ilf_last_error(f._h).decode()
        unchanged()
    finally:
        if keep is not None:
            for k in K:
                ilf_lib.load_library().ilf_host_free(C.c_void_p(keep[k].ctypes.data))


@pytest.mark.parametrize("name", ["ilf_upload", "ilf_download_async", "ilf_set_original"])
def test_device_memory_refused_by_host_calls(name, loaded):
    f, pic, org, si, unchanged = loaded
    t = _dev(pic)
    extra = [si["avail"].ctypes.data_as(C.c_void_p)] if name == "ilf_set_original" else []
    assert getattr(f._lib, name)(f._h, 0, *_args([t[k] for k in K]), *extra) == ERR_ARG
    assert "_device" in f._lib.ilf_last_error(f._h).decode()
    unchanged()


def _bad_cases(ilf_lib, t):
    """(id, planes, fmt) of arguments every device call refuses with ILF_ERR_ARG."""
    torch = _torch()
    I16 = ilf_lib.ilf.SAMPLES_I16
    F = lambda ty=I16, bl=0, bc=0: ilf_lib.ilf.IlfSamples(ty, (C.c_int32 * 2)(bl, bc))   # noqa: E731
    y, cb, cr = (t[k] for k in K)
    odd = torch.zeros(y.numel() + 8, dtype=torch.int16, device=y.device)
    mis = (odd.data_ptr() + 1, y.stride(0))
    return [("null_y", [(0, y.stride(0)), cb, cr], None), ("null_cr", [y, cb, (0, cr.stride(0))], None),
            ("short_stride", [(y.data_ptr(), W8 - 8), cb, cr], None), ("short_chroma_stride", [y, (cb.data_ptr(), W8 // 2 - 1), cr], None),
            ("misaligned_i16", [mis, cb, cr], None), ("bad_type", [y, cb, cr], F(2)), ("negative_type", [y, cb, cr], F(-1)),
            ("depth_7", [y, cb, cr], F(I16, 7, 10)), ("depth_17", [y, cb, cr], F(I16, 10, 17)),
            ("u8_depth_10", [y, cb, cr], F(ilf_lib.ilf.SAMPLES_U8, 10, 0))], odd


@pytest.mark.parametrize("name", DEVICE_CALLS)
def test_bad_arguments_refused(name, loaded, ilf_lib):
    f, pic, org, si, unchanged = loaded
    t = _dev(pic)
    cases, _keep = _bad_cases(ilf_lib, t)
    for case, planes, fmt in cases:
        assert _dev_call(f, name, planes, fmt, si["avail"]) == ERR_ARG, case
    # a slot out of range, a NULL ctu_avail
    assert _dev_call(f, name, [t[k] for k in K], None, si["avail"], slot=1) == ERR_ARG
    if name == "ilf_set_original_device":
        assert f._lib.ilf_set_original_device(f._h, 0, *_args([t[k] for k in K]), None, None, None) == ERR_ARG
        assert _dev_call(f, name, [t[k] for k in K], None, C.c_void_p(t["y"].data_ptr())) == ERR_ARG   # ctu_avail on the device
    unchanged()


@pytest.mark.parametrize("name", DEVICE_CALLS)
def test_tensor_on_another_device_refused(name, loaded):
    torch = _torch()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    f, pic, org, si, unchanged = loaded
    t0, t1 = _dev(pic, 0), _dev(pic, 1)
    assert _dev_call(f, name, [t0["y"], t1["cb"], t0["cr"]], avail=si["avail"]) == ERR_ARG
    assert "another device" in f._lib.ilf_last_error(f._h).decode()
    unchanged()


def test_state_errors(ilf_lib):
    w, h, c = 264, 520, 6
    pic = synth.picture(np.random.default_rng(1), w, h, 10)
    with ilf_lib.InLoopFilter(w, h, 10, 10, c) as f:
        t = _dev(pic)
        assert _dev_call(f, "ilf_download_device", [t[k] for k in K]) == ERR_STATE
    part = bands.band_partition((h + 63) // 64, 2)
    with ilf_lib.InLoopFilter(w, h, 10, 10, c, band=part[1]) as f:
        own = _dev(_own(pic, f))
        assert _dev_call(f, "ilf_download_device", [own[k] for k in K]) == ERR_STATE
        assert _dev_call(f, "ilf_set_original_device", [own[k] for k in K], avail=_avail(w, h, c)) == ERR_STATE
        f.upload_device(0, *own.values())
        f.set_original_device(0, *own.values(), _avail(w, h, c))
        assert _same(_host(f.download_device(0)), {k: _own(pic, f)[k] for k in K})
