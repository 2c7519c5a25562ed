"""Deblocking offset search (ilf_deblock_search) against the best the library offers without it, on the device.

Workload: the 17 resident 4K random-access pictures of bench.py (real side information of bench_data/ra_4k.npz, synthetic
planes) with a noisy copy of each as the original, 49 candidates (beta, tc offsets in -3..3).
  (a) fused:    one ilf_deblock_search over all slots and candidates;
  (b) baseline: per candidate, the side information re-sent with the offsets rewritten (ilf_set_deblock_info), one batched
                deblocking launch over the resident slots (ilf_run, deblocking only) and the distortion of every plane in torch
                on the slots' output planes.
Both are checked against each other first, then timed with CUDA events on the library's stream after a warm-up.  Prints one JSON
line.  Needs a CUDA device: there is no fallback.
"""
import argparse
import os
import re
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

K = ("y", "cb", "cr")


def with_offsets(params_bytes, beta, tc):
    pb = bytearray(bytes(params_bytes))
    for i in range(64):
        pb[16 + 4 * i] = beta & 0xFF
        pb[17 + 4 * i] = tc & 0xFF
    return bytes(pb)


class DevPlane:
    """A library-owned device plane as a torch tensor (no copy): rows x pitch int16, the first `cols` columns are the picture."""

    def __init__(self, ptr, pitch, rows):
        self.__cuda_array_interface__ = {"shape": (rows, pitch), "typestr": "<i2", "data": (ptr, False), "strides": None, "version": 2}


def kernel_resources(lib_path):
    """Registers of deblock_search_kernel<0/1/2> as the compiler allocated them (cuobjdump -res-usage of the built library)."""
    out = subprocess.run(["cuobjdump", "-res-usage", lib_path], capture_output=True, text=True, check=True).stdout
    regs = {}
    for m in re.finditer(r"Function (\S*deblock_search_kernelILi(\d)E\S*):\s*\n\s*REG:(\d+)", out):
        regs[int(m.group(2))] = int(m.group(3))
    return regs


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=5, help="timed passes of each variant")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--shift", type=int, nargs=2, default=(0, 0), help="per-sample shift of the squared error, luma and chroma")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("deblock_search_bench.py needs a CUDA device (there is no CPU fallback)")
    import bench
    import vvcsoftware_vtm_b200 as v
    from vvcsoftware_vtm_b200.ilf import STAGE_DEBLOCK

    w, h = 3840, 2160
    side = bench.load_sideinfo("ra_4k")
    B = len(side)
    cands = [(b, t) for b in range(-3, 4) for t in range(-3, 4)]
    planes = bench.synth_planes(w, h, 4, seed=1000)
    rng = np.random.default_rng(7)
    orgs = [tuple(np.clip(p.astype(np.int32) + rng.integers(-12, 13, p.shape), 0, 1023).astype(np.int16) for p in trip) for trip in planes]
    f = v.InLoopFilter(w, h, 10, 10, 7, num_slots=B)
    dev = torch.device("cuda", 0)

    def set_side(s, params=None):
        si = side[s]
        f.set_deblock_info(s, params or si["db_params"].tobytes(), si["db_info"], si.get("db_info_c"), si.get("db_mv16"), None, si["ctu_slice"])

    for s in range(B):
        f.upload(s, *planes[s % len(planes)])
        set_side(s)
        o = orgs[s % len(orgs)]
        f.set_original(s, o[0], o[1], o[2], np.zeros(f.ctus_w * f.ctus_h, np.uint8))
    f.sync()
    stream = torch.cuda.ExternalStream(f.stream(), device=dev)
    org_t = [[torch.from_numpy(np.ascontiguousarray(p)).to(dev).to(torch.int32) for p in o] for o in orgs]
    shift = tuple(args.shift)
    params = [[with_offsets(side[s]["db_params"].tobytes(), b, t) for s in range(B)] for b, t in cands]

    def fused():
        f.deblock_search(cands, shift, 0, B)

    out_t = []

    def baseline(acc):
        for k in range(len(cands)):
            for s in range(B):
                set_side(s, params[k][s])
            f.run(0, B, STAGE_DEBLOCK)
            if not out_t:   # deblocking writes buffer 1 of every plane: the views stay valid for the whole run
                for s in range(B):
                    ptrs, pitch = f.output_planes(s)
                    out_t.append([torch.as_tensor(DevPlane(ptrs[c], pitch[c], h >> (c > 0)), device=dev)[:, :w >> (c > 0)] for c in range(3)])
            with torch.cuda.stream(stream):
                for s in range(B):
                    for c in range(3):
                        d = out_t[s][c].to(torch.int32) - org_t[s % len(orgs)][c]
                        acc[k, s, c] = ((d * d) >> shift[c > 0]).sum()

    # parity: the fused search == the per-candidate baseline, every candidate, slot and plane
    acc = torch.zeros((len(cands), B, 3), dtype=torch.int64, device=dev)
    fused()
    got = np.stack([f.get_deblock_search(s) for s in range(B)], axis=1).astype(np.int64)
    baseline(acc)
    f.sync()
    torch.cuda.synchronize()
    want = acc.cpu().numpy()
    if not np.array_equal(got, want):
        bad = np.argwhere(got != want)[0]
        raise SystemExit(f"parity failure at (candidate, slot, plane) {tuple(bad)}: fused {got[tuple(bad)]} baseline {want[tuple(bad)]}")

    def timed(fn, steps):
        for _ in range(args.warmup):
            fn()
        f.sync()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(steps):
            fn()
        ev1.record(stream)
        ev1.synchronize()
        f.sync()
        return ev0.elapsed_time(ev1) / steps

    ms_a = timed(fused, args.steps)
    ms_b = timed(lambda: baseline(acc), max(1, args.steps // 5))
    ms_a2 = timed(fused, args.steps)    # again after the baseline: the spread of (a)
    algo_bytes = 6.0 * w * h            # the picture and the original read once: 2 B x 1.5 samples x 2 pictures per luma pixel
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    regs = kernel_resources(v.lib_path())
    rec = {
        "what": "deblocking offset search, 17 resident 3840x2160 10-bit random-access pictures (bench_data/ra_4k.npz side information), 49 candidates",
        "candidates": len(cands), "pictures": B, "shift": list(shift), "parity": "fused == baseline, every candidate, picture and plane",
        "fused_ms_per_picture": ms_a / B, "fused_ms_per_picture_repeat": ms_a2 / B,
        "baseline_ms_per_picture": ms_b / B, "speedup": ms_b / ms_a,
        "fused_ms_per_picture_per_candidate": ms_a / B / len(cands),
        "algo_bytes_per_picture": algo_bytes, "fused_achieved_GBps": algo_bytes * B / (ms_a * 1e-3) / 1e9,
        "search_kernel_registers": regs, "search_kernel_ctas_per_sm": {mv: min(65536 // (((r + 7) // 8 * 8) * 32 * 5), 4) for mv, r in regs.items()},
        "gpu": gpu[0] if gpu else "unknown", "steps": args.steps, "warmup": args.warmup,
    }
    bench.emit(rec)   # bench points file descriptor 1 at stderr on import; emit writes to the original stdout
    f.close()


if __name__ == "__main__":
    main()
