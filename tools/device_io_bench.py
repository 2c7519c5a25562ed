"""Pictures to and from device memory, timed on the device: ilf_upload_device, ilf_set_original_device and ilf_download_device
against a torch copy_ of the same bytes and the host round trip through page-locked memory, in one run.

Workload: 17 resident 3840x2160 10-bit 4:2:0 pictures (the slot count of bench.py's ra_4k workload, synthetic planes as bench.py
makes them), one context slot each.  Every caller picture is one CUDA tensor holding its three planes back to back (Y, then Cb,
then Cr), so a torch copy_ of a picture is one launch, as a transfer of the library is; 17 pictures of sources and destinations
(850 MB in int16) do not fit the 126 MB L2, so each pass reads HBM.  Times are CUDA events on the caller's stream around 17
calls (one per slot), median of --steps passes after --warmup, divided by 17.  Algorithmic bytes = samples x (source bytes +
destination bytes).  The host leg is a host clock around 17 ilf_upload (then ilf_sync) or 17 ilf_download_async (then ilf_sync)
from / into page-locked planes.  ctu_avail of set_original_device is page-locked, so no call waits for the host.  Results are
checked first: every device transfer equals the host path.  A separate pass under torch.profiler (CUDA activity only) gives the
device time of the conversion kernel and of torch's copy kernel alone, which separates kernel time from the cost of ordering a
call against the caller's stream.  Prints one JSON line (and writes it to --out).  Needs a CUDA device.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

K = ("y", "cb", "cr")
W, H, BD, CTU, N = 3840, 2160, 10, 7, 17


def card():
    """Name, power limit and maximum SM clock of every GPU, read in the same run as the measurement."""
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return [r.strip() for r in q.stdout.strip().splitlines()] if q.returncode == 0 else ["nvidia-smi unavailable"]


def planes_of(buf):
    """Y, Cb, Cr views of one picture's buffer (planes back to back)."""
    ny, nc = W * H, (W // 2) * (H // 2)
    return {"y": buf[:ny].view(H, W), "cb": buf[ny:ny + nc].view(H // 2, W // 2), "cr": buf[ny + nc:].view(H // 2, W // 2)}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON record here")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("device_io_bench.py needs a CUDA device (there is no CPU fallback)")
    import bench
    import vvcsoftware_vtm_b200 as v

    dev = torch.device("cuda", 0)
    samples = W * H * 3 // 2
    pics = bench.synth_planes(W, H, N, seed=600)
    src16 = [torch.from_numpy(np.concatenate([p.ravel() for p in pic])).to(dev) for pic in pics]
    src8 = [(s >> 2).to(torch.uint8) for s in src16]
    dst16 = [torch.empty_like(s) for s in src16]
    dst8 = [torch.empty_like(s) for s in src8]
    cw, ch = (W + 127) // 128, (H + 127) // 128
    lib = v.load_library()
    avail_p = lib.ilf_host_alloc(cw * ch)
    avail = np.ctypeslib.as_array(C.cast(avail_p, C.POINTER(C.c_uint8)), shape=(cw * ch,))
    avail[...] = 0x15
    stream = torch.cuda.current_stream(dev)

    def timed_dev(fn):
        """Median ms per picture of fn(i) over the 17 slots, CUDA events on the caller's stream."""
        for _ in range(args.warmup):
            for i in range(N):
                fn(i)
        ts = []
        for _ in range(args.steps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for i in range(N):
                fn(i)
            b.record(stream)
            b.synchronize()
            ts.append(a.elapsed_time(b) / N)
        return statistics.median(ts), min(ts), max(ts)

    def timed_host(fn, f):
        for _ in range(args.warmup):
            for i in range(N):
                fn(i)
            f.sync()
        ts = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            for i in range(N):
                fn(i)
            f.sync()
            ts.append((time.perf_counter() - t0) * 1e3 / N)
        return statistics.median(ts), min(ts), max(ts)

    def leg(name, t, src_bytes, dst_bytes):
        ms = t[0]
        return {"leg": name, "ms_per_picture": round(ms, 5), "min_ms": round(t[1], 5), "max_ms": round(t[2], 5),
                "algo_bytes_per_picture": samples * (src_bytes + dst_bytes), "algo_gb_per_s": round(samples * (src_bytes + dst_bytes) / (ms * 1e-3) / 1e9, 1)}

    rec = {"what": __doc__.split("\n")[0], "cards": card(), "picture": f"{N} x {W}x{H} {BD}-bit 4:2:0, one slot each", "steps": args.steps,
           "warmup": args.warmup, "timing": "CUDA events on the caller's stream around 17 calls; median over steps, per picture", "legs": []}
    with v.InLoopFilter(W, H, BD, BD, CTU, num_slots=N) as f:
        # checks: device transfers equal the host path
        host = [dict(zip(K, p)) for p in pics]
        for i in range(N):
            f.upload_device(i, *planes_of(src16[i]).values())
        for i in (0, N - 1):
            got = f.download(i)
            assert all(np.array_equal(got[k], host[i][k]) for k in K), "upload_device != host planes"
            f.download_device(i, out=planes_of(dst16[i]))
            f.download_device(i, dtype=torch.uint8, out=planes_of(dst8[i]))
            torch.cuda.synchronize()
            assert torch.equal(dst16[i], src16[i]), "download_device (int16) != upload"
            want8 = torch.clamp((src16[i].to(torch.int32) + 2) >> 2, 0, 255).to(torch.uint8)
            assert torch.equal(dst8[i], want8), "download_device (uint8) != rounded picture"
            f.upload_device(i, *planes_of(src8[i]).values())
            assert all(np.array_equal(f.download(i)[k], planes_of(src8[i])[k].cpu().numpy().astype(np.int16) << 2) for k in K), "uint8 upload"

        rec["legs"].append(leg("upload_device int16", timed_dev(lambda i: f.upload_device(i, *planes_of(src16[i]).values())), 2, 2))
        rec["legs"].append(leg("upload_device uint8 (8-bit caller, << 2)", timed_dev(lambda i: f.upload_device(i, *planes_of(src8[i]).values())), 1, 2))
        rec["legs"].append(leg("set_original_device int16", timed_dev(lambda i: f.set_original_device(i, *planes_of(src16[i]).values(), avail)), 2, 2))
        rec["legs"].append(leg("set_original_device uint8 (8-bit caller, << 2)",
                               timed_dev(lambda i: f.set_original_device(i, *planes_of(src8[i]).values(), avail)), 1, 2))
        for i in range(N):
            f.upload_device(i, *planes_of(src16[i]).values())
        rec["legs"].append(leg("download_device int16", timed_dev(lambda i: f.download_device(i, out=planes_of(dst16[i]))), 2, 2))
        rec["legs"].append(leg("download_device uint8 (rounded, clipped)", timed_dev(lambda i: f.download_device(i, dtype=torch.uint8, out=planes_of(dst8[i]))), 2, 1))
        rec["legs"].append(leg("torch copy_ int16 (same bytes)", timed_dev(lambda i: dst16[i].copy_(src16[i])), 2, 2))
        rec["legs"].append(leg("torch copy_ uint8 -> int16 (same bytes as the uint8 upload)", timed_dev(lambda i: dst16[i].copy_(src8[i])), 1, 2))
        pinned = [v.pinned_planes(W, H) for _ in range(N)]
        try:
            for i in range(N):
                for k in K:
                    pinned[i][k][...] = host[i][k]
            up = timed_host(lambda i: f.upload(i, *(pinned[i][k] for k in K)), f)
            down = timed_host(lambda i: f.download_async(i, pinned[i]), f)
            rec["legs"].append(leg("host round trip: ilf_upload from page-locked planes", up, 2, 2))
            rec["legs"].append(leg("host round trip: ilf_download_async into page-locked planes", down, 2, 2))
            rec["host_round_trip_ms_per_picture"] = round(up[0] + down[0], 4)
        finally:
            for p in pinned:
                for k in K:
                    lib.ilf_host_free(C.c_void_p(p[k].ctypes.data))
        # kernel time alone, in a pass of its own
        from torch.profiler import ProfilerActivity, profile

        def kernel_us(fn, name):
            for i in range(N):
                fn(i)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    for i in range(N):
                        fn(i)
                torch.cuda.synchronize()
            ts = [getattr(e, "device_time", None) or e.cuda_time for e in prof.events()
                  if str(e.device_type).endswith("CUDA") and any(n in e.name.lower() for n in name)]
            return round(statistics.median(ts), 2) if ts else None

        for i in range(N):
            f.upload_device(i, *planes_of(src16[i]).values())
        rec["kernel_only_us_per_picture"] = {
            "upload_device int16 (ilf_io_convert)": kernel_us(lambda i: f.upload_device(i, *planes_of(src16[i]).values()), ("ilf_io_convert",)),
            "download_device int16 (ilf_io_convert)": kernel_us(lambda i: f.download_device(i, out=planes_of(dst16[i])), ("ilf_io_convert",)),
            "download_device uint8 (ilf_io_convert)": kernel_us(lambda i: f.download_device(i, dtype=torch.uint8, out=planes_of(dst8[i])), ("ilf_io_convert",)),
            "torch copy_ int16": kernel_us(lambda i: dst16[i].copy_(src16[i]), ("copy", "memcpy")),
        }
    lib.ilf_host_free(avail_p)
    by = {x["leg"]: x for x in rec["legs"]}
    ref = by["torch copy_ int16 (same bytes)"]["algo_gb_per_s"]
    rec["int16_share_of_torch_copy"] = {n: round(by[n]["algo_gb_per_s"] / ref, 3) for n in ("upload_device int16", "set_original_device int16", "download_device int16")}
    rec["checks"] = "upload_device / download_device (int16, uint8) equal the host path on slots 0 and 16 before timing"
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
