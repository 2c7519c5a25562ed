"""The per-slot ordering of the library's streams, end to end: uploads, side information and originals on the upload stream,
chains dealt to lanes, encoder passes on the compute stream and downloads on the download stream, issued back to back with no
host synchronisation, must give bit for bit what the same calls give one slot at a time with a synchronisation after each.
A batched call that fails validation must leave every slot's pending upload to be waited for by the next run."""
import ctypes as C
import os

import numpy as np
import pytest

import golden_io as G
import synth

pytestmark = pytest.mark.gpu
K = G.K
CANDS = [(b, t) for b in (-2, 0, 2) for t in (-2, 0, 2)]
SHIFT = (1, 2)


@pytest.fixture
def pinned(ilf_lib):
    """pinned(a) -> a page-locked copy of array `a` (ilf_host_alloc); freed when the test ends, after its contexts are closed."""
    lib = ilf_lib.load_library()
    ptrs = []

    def copy(a):
        a = np.ascontiguousarray(a)
        p = lib.ilf_host_alloc(max(1, a.nbytes))
        if not p:
            raise ilf_lib.IlfError("ilf_host_alloc failed")
        ptrs.append(p)
        out = np.ctypeslib.as_array(C.cast(p, C.POINTER(np.ctypeslib.as_ctypes_type(a.dtype))), shape=a.shape)
        out[...] = a
        return out

    yield copy
    for p in ptrs:
        lib.ilf_host_free(p)


def _lanes(monkeypatch):
    monkeypatch.setenv("ILF_RUN_LANES", "3")
    monkeypatch.setenv("ILF_RUN_LANE_MIN", "4")


def _avail(ctus_w, ctus_h):
    """ILF_AVAIL_L / _A / _AL of every CTU whose neighbour is inside the picture."""
    cx, cy = np.meshgrid(np.arange(ctus_w), np.arange(ctus_h))
    return ((cx > 0) * 0x01 | (cy > 0) * 0x04 | ((cx > 0) & (cy > 0)) * 0x10).astype(np.uint8).ravel()


def _same(a, b):
    return all(np.array_equal(a[k], b[k]) for k in K)


def test_calls_without_host_synchronisation(ilf_lib, monkeypatch, pinned):
    """Six slots of captured pictures: upload, side information and original, a chain on lanes, asynchronous downloads, SAO and ALF
    statistics and the deblocking search over all six, a new picture in three slots, a second chain and download, a picture hash --
    with no synchronisation in between -- against a context that makes the same calls one slot at a time and synchronises after each."""
    _lanes(monkeypatch)
    caps = [G.load_golden(p) for p in sorted(G.golden_files()) if os.path.basename(p).startswith("ra_416x240")]
    assert len(caps) == 4
    g = caps[0]["geom"]
    rng = np.random.default_rng(5)
    pre = [{k: pinned(c[f"pre_{k}"]) for k in K} for c in caps]
    org = [{k: pinned(np.clip(c[f"pre_{k}"].astype(np.int32) + rng.integers(-9, 10, c[f"pre_{k}"].shape), 0, 1023).astype(np.int16)) for k in K}
           for c in caps]
    n, again = 6, (0, 1, 2)
    first = [i % 4 for i in range(n)]
    second = [(i + 2) % 4 if i in again else first[i] for i in range(n)]

    def ctx():
        return ilf_lib.InLoopFilter(g["width"], g["height"], g["bd_luma"], g["bd_chroma"], g["ctu_log2"], num_slots=n)

    def load(f, slot, j, avail, after=lambda: None):
        c = caps[j]
        mv = c["db_mv32"]
        fits = np.abs(mv).max(initial=0) < 32768
        calls = [lambda: f.upload(slot, *(pre[j][k] for k in K)),
                 lambda: f.set_deblock_info(slot, c["db_params"].tobytes(), c["db_info"], c.get("db_info_c"), mv.astype(np.int16) if fits else None,
                                            None if fits else mv, c["ctu_slice"]),
                 lambda: f.set_sao_params(slot, c["sao_ctus"]),
                 lambda: f.set_alf_params(slot, c["alf_params"].tobytes(), c["alf_ctu_enable"]),
                 lambda: f.set_original(slot, org[j]["y"], org[j]["cb"], org[j]["cr"], avail)]
        for call in calls:
            call()
            after()

    def outputs():
        return [{k: pinned(np.zeros_like(caps[0][f"pre_{k}"])) for k in K} for _ in range(n)]

    # every call issued back to back; the page-locked inputs, originals and outputs make the copies asynchronous
    out1, out2 = outputs(), outputs()
    with ctx() as f:
        assert f.run_lanes() == 3
        avail = pinned(_avail(f.ctus_w, f.ctus_h))
        for i in range(n):
            load(f, i, first[i], avail)
        f.run(0, n, 7)
        for i in range(n):
            f.download_async(i, out1[i])
        f.sao_stats(0, n)
        f.alf_stats(0, n)
        f.deblock_search(CANDS, SHIFT, 0, n)
        for i in again:
            load(f, i, second[i], avail)
        f.run(0, n, 7)
        for i in range(n):
            f.download_async(i, out2[i])
        crc = f.picture_hash(n - 1, "crc")
        f.sync()
        got = ([f.get_sao_stats(i) for i in range(n)], [f.get_alf_stats(i) for i in range(n)], [f.get_deblock_search(i) for i in range(n)])

    # the same calls one slot at a time, synchronised after each
    with ctx() as f:
        avail = pinned(_avail(f.ctus_w, f.ctus_h))

        def each(call):
            for i in range(n):
                call(i)
                f.sync()

        each(lambda i: load(f, i, first[i], avail, f.sync))
        each(lambda i: f.run(i, 1, 7))
        ref1 = [f.download(i) for i in range(n)]
        each(lambda i: f.sao_stats(i, 1))
        each(lambda i: f.alf_stats(i, 1))
        each(lambda i: f.deblock_search(CANDS, SHIFT, i, 1))
        for i in again:
            load(f, i, second[i], avail, f.sync)
        each(lambda i: f.run(i, 1, 7))
        ref2 = [f.download(i) for i in range(n)]
        want_crc = f.picture_hash(n - 1, "crc")
        want = ([f.get_sao_stats(i) for i in range(n)], [f.get_alf_stats(i) for i in range(n)], [f.get_deblock_search(i) for i in range(n)])

    for i in range(n):
        assert _same(ref1[i], {k: caps[first[i]][f"alf_{k}"] for k in K}), f"slot {i}: the synchronous context differs from the reference capture"
        assert _same(out1[i], ref1[i]), f"slot {i}: first download"
        assert _same(out2[i], ref2[i]), f"slot {i}: second download"
    for name, a, b in zip(("SAO statistics", "ALF statistics", "search sums"), got, want):
        for i in range(n):
            assert np.array_equal(a[i], b[i]), f"slot {i}: {name}"
    assert crc == want_crc


@pytest.mark.parametrize("stats", ["sao_stats", "alf_stats"])
def test_failed_statistics_call_keeps_uploads_pending(stats, ilf_lib, monkeypatch, pinned):
    """A statistics call over eight slots whose last one has no original fails before it orders anything after the uploads that are
    still in flight (4K pictures from page-locked memory): the chain on lanes that follows still waits for them and gives the planes
    of a synchronous run."""
    _lanes(monkeypatch)
    W, H, n = 3840, 2160, 8
    rng = np.random.default_rng(17)
    pics = [{k: pinned(v) for k, v in synth.picture(rng, W, H, 10).items()} for _ in range(2)]
    org = {k: pinned(v) for k, v in synth.picture(rng, W, H, 10).items()}
    with ilf_lib.InLoopFilter(W, H, 10, 10, 7, num_slots=n) as f:
        cw, ch = f.ctus_w, f.ctus_h
        side = []
        for _ in range(2):
            prm, info, mv16 = synth.deblock_info(rng, W, H, inter=True)
            alf, en = synth.alf_params(rng, cw, ch, is7=True, p_on=0.9)
            side.append((prm, info, mv16, synth.sao_params(rng, cw, ch, 10, p_off=0.1), alf, en))
        avail = pinned(_avail(cw, ch))

        def load(pic):
            for i in range(n):
                prm, info, mv16, sao, alf, en = side[i % 2]
                f.upload(i, *(pics[pic][k] for k in K))
                f.set_deblock_info(i, prm, info, None, mv16, None, None)
                f.set_sao_params(i, sao)
                f.set_alf_params(i, alf, en)
                if i < n - 1:
                    f.set_original(i, org["y"], org["cb"], org["cr"], avail)

        # every slot holds the other picture and the same side information and descriptors first, so that the only thing a run
        # that does not wait for the uploads below could get wrong is sample values
        load(0)
        f.sao_stats(0, n - 1)
        f.alf_stats(0, n - 1)
        f.sync()
        load(1)
        with pytest.raises(ilf_lib.IlfError):
            getattr(f, stats)(0, n)
        f.run(0, n, 7)
        got = [f.download(i) for i in range(n)]
        f.sync()
        for i in range(n):
            f.run(i, 1, 7)
            f.sync()
            assert _same(got[i], f.download(i)), f"slot {i}"
