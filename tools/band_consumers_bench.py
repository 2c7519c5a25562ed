"""Consumers of the filtered picture on band contexts, timed on the device against what a host had to do before they existed.

Workload: the 7680x4320 10-bit intra picture of bench.py (real side information of bench_data/intra_8k.npz with every CTU of every
component on, synthetic planes) in 1 / 2 / 4 / 8 CTU-row bands, every band a context of its own on one GPU, and -- when the box has
several -- one band per GPU.  A noisy copy of the picture is the original of the encoder passes.
  hash      per band ilf_picture_hash_band, then ilf_hash_combine on the host (CRC and checksum: one call gives both)
            against per band ilf_download_band into pageable memory and a host CRC-32 (zlib) of its planes, the way bench.py
            checks band parity today
  encoder   ilf_sao_stats (on the deblocked picture), ilf_alf_stats (on the SAO'd picture), ilf_deblock_search (49 candidates)
            per band against the same call on the whole picture
Times are host clocks around calls that end in a synchronise (median of --steps after --warmup): "bands_serial" runs the bands one
after the other and sums their times, "bands_issued" issues every band's call and then synchronises them all (bands on one GPU
share it; bands on several GPUs run side by side).  Results are checked first: combined hash == whole-picture hash, concatenated
statistics and summed search sums == the whole picture's.  Prints one JSON line (and writes it to --out).  Needs a CUDA device.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import zlib

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

K = ("y", "cb", "cr")
W, H, BD, CTU = 7680, 4320, 10, 7
CANDS = [(b, t) for b in range(-3, 4) for t in range(-3, 4)]


def card():
    """Name and power limit of every GPU, read in the same run as the measurement."""
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return [r.strip() for r in q.stdout.strip().splitlines()] if q.returncode == 0 else ["nvidia-smi unavailable"]


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return round(statistics.median(ts) * 1e3, 3)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--bands", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--out", default=None, help="also write the JSON record here")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("band_consumers_bench.py needs a CUDA device (there is no CPU fallback)")
    import bench
    import vvcsoftware_vtm_b200 as v
    from vvcsoftware_vtm_b200 import bands

    si = bench.all_on_sideinfo(bench.load_sideinfo("intra_8k"))[0]
    pic = dict(zip(K, bench.synth_planes(W, H, 1, seed=8000)[0]))
    rng = np.random.default_rng(8001)
    org = {k: np.clip(pic[k].astype(np.int32) + rng.integers(-12, 13, pic[k].shape), 0, (1 << BD) - 1).astype(np.int16) for k in K}
    cw, ch = (W + 127) // 128, (H + 127) // 128
    avail = np.full(cw * ch, 0xFF, np.uint8)
    avail[np.arange(cw * ch) % cw == 0] &= ~np.uint8(0x01 | 0x10)
    avail[:cw] &= ~np.uint8(0x04 | 0x10)
    shift = (0, 0)

    def set_side(f, s):
        f.set_deblock_info(0, s["db_params"].tobytes(), s["db_info"], s.get("db_info_c"), s.get("db_mv16"), s.get("db_mv32"), s.get("ctu_slice"))
        f.set_sao_params(0, s["sao_ctus"])
        f.set_alf_params(0, s["alf_params"].tobytes(), s["alf_ctu_enable"])

    rec = {"what": __doc__.split("\n")[0], "cards": card(), "picture": f"{W}x{H} 10-bit 4:2:0 intra (bench_data/intra_8k.npz side information, all CTUs on)",
           "steps": args.steps, "warmup": args.warmup, "search_candidates": len(CANDS), "legs": []}
    whole = v.InLoopFilter(W, H, BD, BD, CTU)
    whole.upload(0, *(pic[k] for k in K))
    set_side(whole, si)
    whole.set_original(0, org["y"], org["cb"], org["cr"], avail)

    def whole_pass(name):
        return {"sao_stats": lambda: (whole.sao_stats(), whole.sync()), "alf_stats": lambda: (whole.alf_stats(), whole.sync()),
                "deblock_search": lambda: (whole.deblock_search(CANDS, shift), whole.sync())}[name]

    whole.run(0, 1, 1)
    t_whole = {"sao_stats": timed(whole_pass("sao_stats"), args.steps, args.warmup)}
    want_sao = whole.get_sao_stats()
    whole.run(0, 1, 2)
    t_whole["alf_stats"] = timed(whole_pass("alf_stats"), args.steps, args.warmup)
    want_alf = whole.get_alf_stats()
    t_whole["deblock_search"] = timed(whole_pass("deblock_search"), args.steps, args.warmup)
    want_search = whole.get_deblock_search()
    whole.run(0, 1, 7)
    t_whole["picture_hash"] = timed(lambda: (whole.picture_hash(0, "crc"), whole.picture_hash(0, "checksum")), args.steps, args.warmup)
    want_hash = {kind: whole.picture_hash(0, kind) for kind in ("crc", "checksum")}
    rec["whole_picture_ms"] = t_whole
    whole.close()

    ndev = torch.cuda.device_count()
    layouts = [(n, 1) for n in args.bands] + ([(n, min(n, ndev)) for n in args.bands if n > 1] if ndev > 1 else [])
    for n, devices in layouts:
        part = bands.band_partition(ch, n)
        ctxs = [v.InLoopFilter(W, H, BD, BD, CTU, band=b, device=r % devices) for r, b in enumerate(part)]
        try:
            for f in ctxs:
                y0, y1 = f.own_row0, f.own_row0 + f.own_rows
                f.upload_band(0, pic["y"][y0:y1], pic["cb"][y0 // 2:y1 // 2], pic["cr"][y0 // 2:y1 // 2])
            for f in ctxs:
                f.sync()
            handles = [f.band_export(0) for f in ctxs]
            for r, f in enumerate(ctxs):
                bands.connect_bands(f, 0, r, n, handles)
                f.band_exchange(0)
                set_side(f, bands.slice_side_info(si, f.row0, f.rows))
                y0, y1 = f.own_row0, f.own_row0 + f.own_rows
                f.set_original_band(0, org["y"][y0:y1], org["cb"][y0 // 2:y1 // 2], org["cr"][y0 // 2:y1 // 2], avail)
            leg = {"bands": n, "devices": devices, "rows": [f.own_rows for f in ctxs], "ms": {}}

            def band_pass(name, f):
                return {"sao_stats": f.sao_stats, "alf_stats": f.alf_stats, "deblock_search": lambda: f.deblock_search(CANDS, shift)}[name]

            def measure(name):
                serial = sum(timed(lambda f=f: (band_pass(name, f)(), f.sync()), args.steps, args.warmup) for f in ctxs)

                def issued():
                    for f in ctxs:
                        band_pass(name, f)()
                    for f in ctxs:
                        f.sync()
                leg["ms"][name] = {"bands_serial": round(serial, 3), "bands_issued": timed(issued, args.steps, args.warmup)}

            for f in ctxs:
                f.run(0, 1, 1)
            measure("sao_stats")
            assert np.array_equal(np.concatenate([f.get_sao_stats() for f in ctxs]), want_sao), "SAO statistics: bands != whole picture"
            for f in ctxs:
                f.run(0, 1, 2)
            measure("alf_stats")
            assert np.array_equal(np.concatenate([f.get_alf_stats() for f in ctxs]), want_alf), "ALF statistics: bands != whole picture"
            measure("deblock_search")
            assert np.array_equal(sum(f.get_deblock_search() for f in ctxs), want_search), "search: bands != whole picture"
            for f in ctxs:
                f.run(0, 1, 7)
            for f in ctxs:
                f.sync()

            def device_hash():
                parts = [f.picture_hash_band(0) for f in ctxs]
                return {kind: v.hash_combine(parts, kind) for kind in ("crc", "checksum")}

            def host_crc():
                crcs = []
                for f in ctxs:
                    got = f.download_band(0)
                    crcs.append([zlib.crc32(np.ascontiguousarray(got[k]).tobytes()) for k in K])
                return crcs
            assert device_hash() == want_hash, "hash: combined band parts != whole-picture hash"
            leg["ms"]["hash"] = {"picture_hash_band_and_combine": timed(device_hash, args.steps, args.warmup),
                                 "download_band_and_host_crc32": timed(host_crc, args.steps, args.warmup)}
            rec["legs"].append(leg)
        finally:
            for f in ctxs:
                f.close()
    rec["checks"] = "combined hash == whole-picture hash; concatenated SAO / ALF records and summed search sums == whole picture's"
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
