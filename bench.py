#!/usr/bin/env python3
"""bench.py -- deblock+SAO+ALF Mpixel/s of the B200 in-loop filter library (and of the reference on the host cores).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload ra_4k|ra_1080p]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = the whole filter chain (deblock -> SAO -> ALF, 4 kernel launches) over one batch of `--batch`
pictures that are resident in HBM.  The side information of the pictures (per-4x4 CU/TU grid, motion, SAO and ALF
parameters) is REAL: it was packed by the product packer from pictures of the workload's bitstream
(bench_data/<workload>.npz, written by tools/make_bench_sideinfo.py); the sample planes are synthetic (seeded texture
+ 8x8 blockiness), because reconstructed 4K planes are too large to commit.  Pictures are independent, so N GPUs each
run their own batch with no collective (weak scaling); the timed region is bracketed by barrier + synchronize and
the maximum over ranks is reported.

Output: ONE JSON line on rank 0 (see DESIGN.md "measurement" for every field).
`--impl reference` times the reference's own CPU filters (oracle/_ref/vtm_capture = unmodified VTM 2.1 decoder with a
steady_clock hook around its three filter calls) on the same workload's bitstream, one process per host core.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (which may be read-only)
# This script's stdout is ONE JSON line.  Libraries write to file descriptor 1 behind Python's back (NCCL prints its version
# banner there at VERSION level, whatever the environment says), so descriptor 1 is pointed at stderr for the whole run
# and the line goes to a private copy of the original stdout.
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"
_RESULT_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)
sys.stdout = sys.stderr


def emit(line):
    _RESULT_OUT.write(json.dumps(line) + "\n")
    _RESULT_OUT.flush()


WORKLOADS = {
    "ra_4k": dict(width=3840, height=2160, stream="ra_4k", desc="3840x2160 4:2:0 10-bit random access (VTM 2.1 encoder_randomaccess_vtm.cfg, QP37)"),
    "ra_1080p": dict(width=1920, height=1080, stream="ra_1080p", desc="1920x1080 4:2:0 10-bit random access (VTM 2.1 encoder_randomaccess_vtm.cfg, QP37)"),
    # BASELINE config 5: 64 independent low-delay streams dealt round-robin to the GPUs (two encoded streams replicated to 64 logical ones)
    "ld_1080p_x64": dict(width=1920, height=1080, stream="ld_1080p_s3001", npz=["ld_1080p_s3001", "ld_1080p_s3002"], streams=64, scaling="strong",
                         desc="64 independent 1920x1080 4:2:0 10-bit low-delay streams (VTM 2.1 encoder_lowdelay_vtm.cfg, QP37), 9 pictures each, one stream per GPU at a time"),
    # BASELINE config 4: one 8K picture in CTU-row bands across the GPUs, halo rows over NVLink P2P
    "intra_8k_bands": dict(width=7680, height=4320, stream="intra_8k", npz=["intra_8k"], bands=True, scaling="strong",
                           desc="7680x4320 4:2:0 10-bit intra picture (VTM 2.1 encoder_intra_vtm.cfg, QP37) split into CTU-row bands across the GPUs"),
}
# algorithmic bytes per luma pixel and launch: every sample of the planes a kernel owns read once + written once
# (int16, 4:2:0: luma 2 B, both chroma planes 1 B per luma pixel); side information excluded (SURVEY.md 8d).
ALGO_BYTES_PER_PIXEL = {"deblock": 6.0, "sao": 6.0, "alf": 6.0}
CHAIN_BYTES_PER_PIXEL = 18.0


def default_workload():
    return "ra_4k" if os.path.exists(os.path.join(ROOT, "bench_data", "ra_4k.npz")) else "ra_1080p"


def load_sideinfo(name):
    if name in WORKLOADS and "npz" in WORKLOADS[name]:
        name = WORKLOADS[name]["npz"][0]
    z = np.load(os.path.join(ROOT, "bench_data", name + ".npz"))
    pics = []
    for j in range(int(z["num_pictures"])):
        pics.append({k[len(f"p{j}_"):]: z[k] for k in z.files if k.startswith(f"p{j}_")})
    return pics


def synth_planes(width, height, n, seed):
    """n synthetic 10-bit 4:2:0 pictures: smooth texture + sinusoid + 8x8 block offsets (coding-like blockiness) + noise."""
    rng = np.random.default_rng(seed)
    th, tw = height + 64, width + 64
    g = rng.normal(0, 1, (th, tw)).astype(np.float32)
    ky = np.fft.fftfreq(th)[:, None]
    kx = np.fft.rfftfreq(tw)[None, :]
    t = np.fft.irfft2(np.fft.rfft2(g) / (1 + (60 * np.sqrt(ky * ky + kx * kx)) ** 2), s=(th, tw)).astype(np.float32)
    t /= t.std()
    x = np.arange(width, dtype=np.float32)[None, :]
    out = []
    for f in range(n):
        oy, ox = (7 * f) % 64, (13 * f) % 64
        tex = t[oy:oy + height, ox:ox + width]
        def blocks(hh, ww, amp):
            return np.kron(rng.integers(-amp, amp + 1, ((hh + 7) // 8, (ww + 7) // 8)), np.ones((8, 8), np.int32))[:hh, :ww].astype(np.float32)
        blk = blocks(height, width, 5)
        y = 512 + 220 * tex + 60 * np.sin((x - 4 * f) / 37) + blk + rng.normal(0, 2, (height, width)).astype(np.float32)
        cblk = blocks(height // 2, width // 2, 3)
        cb = 512 + 120 * tex[::2, ::2] + cblk
        cr = 512 - 100 * tex[::2, ::2] - cblk
        out.append(tuple(np.clip(np.rint(p), 0, 1023).astype(np.int16) for p in (y, cb, cr)))
    return out


SAO_DT = np.dtype([("offset", "<i2", (3, 4)), ("type", "i1", (3,)), ("band_pos", "u1", (3,)), ("avail", "u1"), ("reserved", "u1")])
ALF_DT = np.dtype([("luma_coeff", "<i2", (25, 13)), ("chroma_coeff", "<i2", (7,)), ("luma_filter_7x7", "<i2")])


def all_on_sideinfo(side):
    """Worst-case variant of the stream's side information (SURVEY.md 8d): every CTU of every component has SAO on (the
    five types cycled over the CTUs, small offsets) and ALF on (the stream's own filters; pictures whose slice had ALF
    off borrow the coefficients of the stream's first ALF picture).  Deblocking information is unchanged (real)."""
    donor = next((si for si in side if np.frombuffer(si["alf_params"].tobytes(), ALF_DT)["luma_coeff"].any()), None)
    out = []
    for j, si in enumerate(side):
        d = dict(si)
        sao = np.frombuffer(si["sao_ctus"].tobytes(), SAO_DT).copy()
        n = sao.shape[0]
        i = np.arange(n)
        for c in range(3):
            sao["type"][:, c] = (i + c + j) % 5
            sao["band_pos"][:, c] = (i * 7 + 3 * c + j) % 32
            for k in range(4):
                sao["offset"][:, c, k] = ((i + 2 * k + c) % 7) - 3
        d["sao_ctus"] = sao.view(np.uint8).reshape(n, 32)
        alf = np.frombuffer(si["alf_params"].tobytes(), ALF_DT).copy()
        if not alf["luma_coeff"].any():
            if donor is not None:
                alf = np.frombuffer(donor["alf_params"].tobytes(), ALF_DT).copy()
            else:
                alf["luma_coeff"][0, :, :12] = np.array([0, 1, -3, 1, 2, -4, 9, -4, 2, -6, 14, 40])[None, :]
                alf["luma_coeff"][0, :, 12] = 512 - 2 * alf["luma_coeff"][0, :, :12].sum(axis=1)
                alf["luma_filter_7x7"] = 1
        cc = alf["chroma_coeff"][0].astype(np.int64)
        if 2 * cc[:6].sum() + cc[6] != 512:  # chroma ALF was off in this slice: the stream carries no (meaningful) chroma filter
            alf["chroma_coeff"][0] = [-2, 5, -9, 5, 3, 30, 512 - 2 * 32]
        d["alf_params"] = np.frombuffer(alf.tobytes(), np.uint8)
        d["alf_ctu_enable"] = np.ones_like(si["alf_ctu_enable"])
        out.append(d)
    return out



def bind_to_gpu_numa(index):
    """Run this rank on the CPU cores NVML names as local to GPU `index` (its NUMA node): page-locked buffers are then
    allocated next to the GPU's PCIe root and the e2e copies do not cross the socket interconnect.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1}
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return len(allowed)
    except Exception:
        return 0


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index, period=0.05):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_ev = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.nv, self.err = None, str(e)

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap", nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake", nv.nvmlClocksThrottleReasonApplicationsClocksSetting: "applications_clocks"}
        while not self._stop_ev.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop_ev.wait(self.period)

    def finish(self):
        self._stop_ev.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the unmodified reference decoder with the timing hook, one process per core
# ------------------------------------------------------------------------------------------------------------------
def reference_chain_run(stream, width, height, procs, max_pics=None, simd=None):
    """Run `procs` reference decoders concurrently on the stream; return (pictures per proc, [chain seconds per proc],
    per-stage seconds of proc 0)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "vtm_capture")
    path = os.path.join(ROOT, "tests", "golden", "streams", stream + ".bin")
    if not (os.path.exists(exe) and os.path.exists(path)):
        return None
    env = dict(os.environ, ILF_TIMING="1")
    env.pop("ILF_CAPTURE_DIR", None)
    if max_pics:
        env["ILF_EXIT_AFTER"] = str(max_pics)
    ps = []
    for i in range(procs):
        cmd = [exe, "-b", path, "-d", "10", "-o", "/dev/null"] + ([f"--SIMD={simd}"] if simd else [])
        if hasattr(os, "sched_setaffinity"):
            cmd = ["taskset", "-c", str(sorted(os.sched_getaffinity(0))[i % len(os.sched_getaffinity(0))])] + cmd
        ps.append(subprocess.Popen(cmd, env=env, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True))
    chain, stages, npics = [], None, 0
    for i, p in enumerate(ps):
        err = p.communicate()[1]
        us = [tuple(int(v) for v in m) for m in re.findall(r"\[ILFTIME\].*deblock_us=(\d+) sao_us=(\d+) alf_us=(\d+)", err)]
        if p.returncode != 0 or not us:
            raise RuntimeError(f"reference decoder failed ({p.returncode}): {err[-500:]}")
        chain.append(sum(sum(u) for u in us) * 1e-6)
        if i == 0:
            stages = [sum(u[k] for u in us) * 1e-6 for k in range(3)]
            npics = len(us)
    return npics, chain, stages


def oracle_port_run(width, height, pics, planes):
    """Fallback CPU baseline when oracle/_ref is absent: the C restatement (oracle/liboracle.so), single thread."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ilf_oracle as O
    K = ("y", "cb", "cr")
    t0 = time.perf_counter()
    n = 0
    while time.perf_counter() - t0 < 10.0:
        si = pics[n % len(pics)]
        pic = dict(zip(K, planes[n % len(planes)]))
        out = O.deblock(pic, 10, 10, 7, si["db_params"].tobytes(), si["db_info"], si.get("db_info_c"), si.get("db_mv16"), None, si["ctu_slice"])
        out = O.sao(out, 10, 10, 7, si["sao_ctus"])
        out = O.alf(out, 10, 10, 7, si["alf_params"].tobytes(), si["alf_ctu_enable"])
        n += 1
    dt = time.perf_counter() - t0
    return n, dt


def shared_config(wl, workload, world):
    """The part of `config` both arms print verbatim (the driver compares the arms' configs): which pictures a step covers."""
    n = len(load_sideinfo(workload))
    return {"workload": wl["desc"], "stream": f"tests/golden/streams/{wl['stream']}.bin", "pictures_per_step_per_gpu": n,
            "chain": "deblock -> SAO -> ALF with the stream's own per-CTU decisions", "gpus": world}


def cpu_baseline(wl, cores, pics=None, planes=None):
    w, h = wl["width"], wl["height"]
    mpx = w * h / 1e6
    r = reference_chain_run(wl["stream"], w, h, cores)
    if r is not None:
        n, chain, stages = r
        value = sum(n * mpx / c for c in chain)
        single = reference_chain_run(wl["stream"], w, h, 1)
        out = {"value": round(value, 1), "unit": "Mpixel/s", "cores": cores, "kind": "reference",
               "sample": f"all {n} pictures of tests/golden/streams/{wl['stream']}.bin decoded by {cores} concurrent unmodified VTM 2.1 decoders (--SIMD default = best available, "
                         f"AVX2 on this box); filter-chain time only (steady_clock around loopFilterPic/SAOProcess/ALFProcess)",
               "single_thread_value": round(single[0] * mpx / single[1][0], 1),
               "stage_share": [round(s / sum(stages), 3) for s in stages]}
        try:   # BASELINE.md section 4: the same with --SIMD=SCALAR (only ALF has a SIMD path in this reference)
            ns, cs, _ = reference_chain_run(wl["stream"], w, h, cores, simd="SCALAR")
            s1 = reference_chain_run(wl["stream"], w, h, 1, simd="SCALAR")
            out["simd_scalar"] = {"value": round(sum(ns * mpx / c for c in cs), 1), "single_thread_value": round(s1[0] * mpx / s1[1][0], 1)}
        except Exception as e:  # pragma: no cover
            out["simd_scalar"] = {"error": str(e)[:200]}
        return out
    n, dt = oracle_port_run(w, h, pics, planes)
    return {"value": round(n * mpx / dt, 1), "unit": "Mpixel/s", "cores": 1, "kind": "port",
            "sample": f"{n} synthetic pictures through oracle/liboracle.so (scalar C restatement), oracle/_ref absent"}


def dropin_leg():
    """The reference-API path, measured in the reference's own decoder: per-picture time of the three filter calls in DecoderApp with
    the host shim + libilf_b200.so (pack + upload + kernels + download, pageable PelStorage planes) against the stock CPU filters, on
    the committed 1080p and 4K random-access streams; average over ALL pictures after the first (which carries the CUDA context)."""
    shim, stock = os.path.join(ROOT, "oracle", "_ref", "DecoderApp_ilf_b200"), os.path.join(ROOT, "oracle", "_ref", "vtm_capture")
    if not (os.path.exists(shim) and os.path.exists(stock)):
        return {"unavailable": "oracle/_ref binaries did not travel"}
    out = {}
    for name in ("ra_1080p", "ra_4k"):
        bit = os.path.join(ROOT, "tests", "golden", "streams", name + ".bin")
        if not os.path.exists(bit):
            continue
        res = {}
        for label, exe in (("cpu", stock), ("gpu", shim)):
            env = dict(os.environ, ILF_TIMING="1")
            env.pop("ILF_CAPTURE_DIR", None)
            r = subprocess.run([exe, "-b", bit, "-d", "10", "-o", "/dev/null"], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
            us = [tuple(int(v) for v in m) for m in re.findall(r"\[ILFTIME\].*deblock_us=(\d+) sao_us=(\d+) alf_us=(\d+)", r.stderr)]
            if r.returncode != 0 or len(us) < 2:
                res[label] = {"error": (r.stderr or r.stdout)[-200:]}
                continue
            us = us[1:]
            res[label] = {"ms_per_picture": round(sum(sum(u) for u in us) / len(us) / 1e3, 3), "pictures": len(us),
                          "stage_ms": [round(sum(u[k] for u in us) / len(us) / 1e3, 3) for k in range(3)], "hash_sei_ok": r.stdout.count("(OK)")}
        if "ms_per_picture" in res.get("cpu", {}) and "ms_per_picture" in res.get("gpu", {}):
            res["gpu_over_cpu_time"] = round(res["gpu"]["ms_per_picture"] / res["cpu"]["ms_per_picture"], 3)
        out[name] = res
    out["what"] = "filter ms per picture inside DecoderApp: gpu = host shim (ilf_pack + ilf_upload + kernels + ilf_download through the C ABI), cpu = the reference's own filters, one thread"
    return out


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()
    w, h = wl["width"], wl["height"]
    mpx = w * h / 1e6
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if reference_chain_run(wl["stream"], w, h, 1, 1) is None:
        # the reference binary did not travel: time the C restatement instead
        pics = load_sideinfo(args.workload)
        planes = synth_planes(w, h, 2, 7)
        n, dt = oracle_port_run(w, h, pics, planes)
        val, ms, kind, c, smp = n * mpx / dt, dt / n * 1e3, "port", 1, "oracle/liboracle.so, synthetic planes"
    else:
        # a step = the whole stream (the same pictures the B200 arm filters per step) on every core at once
        for _ in range(args.warmup):
            reference_chain_run(wl["stream"], w, h, cores)
        tot_t = 0.0
        vals = []
        for _ in range(args.steps):
            n, chain, _st = reference_chain_run(wl["stream"], w, h, cores)
            vals.append(sum(n * mpx / c for c in chain))
            tot_t += max(chain)
        val = float(np.mean(vals))
        ms = tot_t / args.steps * 1e3
        kind, c = "reference", cores
        smp = f"each step: all {n} pictures of {wl['stream']}.bin on each of {cores} concurrent unmodified VTM 2.1 decoders (one per host core), filter-chain time only"
    line = {"impl": "reference", "metric": "deblock+SAO+ALF Mpixel/s", "value": round(val, 1), "unit": "Mpixel/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16",
            "data": "synthetic", "config": shared_config(wl, args.workload, world),
            "cpu_baseline": {"value": round(val, 1), "unit": "Mpixel/s", "cores": c, "kind": kind, "sample": smp},
            "e2e": {"value": round(val, 1), "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------------------------
def hbm_peak():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    return peak, ("MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)")


def ncu_traffic(kernel, batch):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/*_traffic.json, written by tools/ncu_summary.py),
    if that capture was taken with the same batch; None otherwise."""
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")), reverse=True):
        try:
            k = json.load(open(path))["kernels"].get(kernel)
            if k and (k.get("batch") == batch or k["grid"].strip("()").split(",")[-1].strip() == str(batch)):
                return {"bytes_per_launch": round(k["dram_read_bytes"] + k["dram_write_bytes"]), "read": round(k["dram_read_bytes"]), "write": round(k["dram_write_bytes"]),
                        "source": os.path.relpath(path, ROOT)}
        except Exception:
            pass
    return None


def host_ceiling(world, h2d_bytes_per_picture, mpx):
    """What the box's host side allows for the end-to-end leg with `world` GPUs copying at once (profiles/r02_pcie_probe_mg.json,
    tools/pcie_probe_mg.py on an 8-GPU box of this pool): both-directions GB/s and the Mpixel/s that bounds."""
    try:
        rows = json.load(open(os.path.join(ROOT, "profiles", "r02_pcie_probe_mg.json")))["rows"]
        row = max((r for r in rows if r["gpus_copying"] <= world), key=lambda r: r["gpus_copying"])
        gbs = row["both_each_dir"]["aggregate_gbs"]
        return {"both_directions_gbs_each_way": gbs, "gpus_copying": row["gpus_copying"], "mpixel_per_s": round(gbs * 1e9 / h2d_bytes_per_picture * mpx, 1),
                "source": "profiles/r02_pcie_probe_mg.json (measured on an 8-GPU box of this pool; a smaller lease may sit on a different host)"}
    except Exception:
        return None


def kernel_table(kt, peak, steps=None):
    """Per kernel: average launch duration, algorithmic GB/s and fraction of the HBM peak; with `steps` also the kernel's time per
    step (a stage can take several launches per step: deblocking launches the pictures with a chroma tree apart from the others)."""
    tab = {}
    for k, (ms, n, nbytes) in kt.items():
        if n:
            # algorithmic bytes as counted by the library: 2 B x (read + write) x samples of the planes the launches processed
            tab[k] = {"avg_ms": round(ms / n, 4), "launches": n, "algo_mb_per_launch": round(nbytes / n / 1e6, 1), "algo_gbs": round(nbytes / (ms * 1e-3) / 1e9, 1),
                      "frac": round(nbytes / (ms * 1e-3) / 1e9 / peak, 4)}
            if steps:
                tab[k]["ms_per_step"] = round(ms / steps, 4)
                tab[k]["launches_per_step"] = round(n / steps, 2)
    return tab


def dominant(tab):
    return max(tab, key=lambda k: tab[k].get("ms_per_step", tab[k]["avg_ms"]))


def chain_table(kt, ms_region, steps, pixels_per_step, peak):
    """Whole chain against the roofline: bytes the launched kernels really had to move / time of the timed region."""
    nbytes = sum(v[2] for v in kt.values())
    gbs = nbytes / (ms_region * 1e-3) / 1e9
    return {"algo_mb_per_step": round(nbytes / steps / 1e6, 1), "bytes_per_pixel": round(nbytes / (steps * pixels_per_step), 2), "gbs": round(gbs, 1), "frac": round(gbs / peak, 4)}


def plane_crcs(planes):
    import zlib
    return [zlib.crc32(np.ascontiguousarray(p).tobytes()) for p in planes]


DUMP_BYTES = 64 * 10**6


def dump_outputs(f, num_slots, width, height, out_dir):
    """Write the filtered pictures of slots [0, num_slots) as out_dir/{y,cb,cr}.npy, float32 [slot, row, column].  Whole
    pictures when all of them fit in DUMP_BYTES; otherwise the same seeded sample of chroma rows of every picture, with the two
    luma rows of each, so that two builds run with the same arguments can be compared sample for sample."""
    bytes_per_chroma_row = 4 * (2 * width + 2 * (width // 2))
    n = min(height // 2, (DUMP_BYTES - 4096) // (bytes_per_chroma_row * num_slots))
    if n < 1:
        raise SystemExit(f"bench.py: {num_slots} pictures of {width}x{height} do not fit --dump-outputs' {DUMP_BYTES} bytes")
    rows = np.sort(np.random.default_rng(0).choice(height // 2, n, replace=False))
    luma_rows = np.stack([2 * rows, 2 * rows + 1], axis=1).reshape(-1)
    out = {"y": [], "cb": [], "cr": []}
    for s in range(num_slots):
        pic = f.download(s)
        out["y"].append(pic["y"][luma_rows].astype(np.float32))
        out["cb"].append(pic["cb"][rows].astype(np.float32))
        out["cr"].append(pic["cr"][rows].astype(np.float32))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.stack(a))


def bands_record(args, wl, rank, world, local, dist, torch, v):
    """BASELINE config 4: every rank owns a band of CTU rows of ONE picture (vvcsoftware_vtm_b200.bands), uploads its own rows,
    pulls 16 halo rows per side from its neighbours' input planes (CUDA IPC mapping, device-to-device over NVLink P2P, one copy
    kernel) and runs the chain on its band.  A step = halo exchange + chain for B resident pictures; strong scaling.  The record
    carries a PARITY check -- every rank's own rows after the chain, CRC-32 per plane, against the same rows of the whole picture
    filtered by one context on rank 0 -- and the whole-picture time of rank 0 (the N = 1 figure of the same run).  Returns the
    record on rank 0, None elsewhere; raises on a parity mismatch."""
    from vvcsoftware_vtm_b200 import bands
    w, h = wl["width"], wl["height"]
    mpx = w * h / 1e6
    side = load_sideinfo("intra_8k_bands")
    side_on = all_on_sideinfo(side)
    B = args.bands_batch
    steps = args.steps
    f = bands.make_band_context(w, h, 10, 10, 7, rank, world, local, num_slots=B)
    y0, y1 = f.own_row0, f.own_row0 + f.own_rows
    # synthetic planes: a 4K texture tiled 2 x 2 (every rank builds the picture and keeps its own rows)
    q = synth_planes(w // 2, h // 2, 1, seed=8000)[0]
    pic = [np.tile(p, (2, 2)) for p in q]
    own = [np.ascontiguousarray(pic[0][y0:y1]), np.ascontiguousarray(pic[1][y0 // 2:y1 // 2]), np.ascontiguousarray(pic[2][y0 // 2:y1 // 2])]
    if rank != 0:
        del pic
    pins = [torch.from_numpy(a).pin_memory() for a in own]
    own = [t.numpy() for t in pins]

    def set_side(ctx, slot, si, sliced=True):
        s_ = bands.slice_side_info(si, ctx.row0, ctx.rows) if sliced else si
        ctx.set_deblock_info(slot, s_["db_params"].tobytes(), s_["db_info"], s_.get("db_info_c"), s_.get("db_mv16"), None, s_["ctu_slice"])
        ctx.set_sao_params(slot, s_["sao_ctus"])
        ctx.set_alf_params(slot, s_["alf_params"].tobytes(), s_["alf_ctu_enable"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for s_ in range(B):
        f.upload_band(s_, *own)
    f.sync()
    handles = [None] * world
    for s_ in range(B):
        mine = f.band_export(s_)
        if world > 1:
            dist.all_gather_object(handles, mine)
        else:
            handles = [mine]
        bands.connect_bands(f, s_, rank, world, handles)
    barrier()   # every rank's input planes are resident before anybody pulls halos
    halo_rows = (f.own_row0 - f.row0) + (f.row0 + f.rows - (f.own_row0 + f.own_rows))
    stream = torch.cuda.ExternalStream(f.stream(), device=torch.device("cuda", local))

    def timed(ctx, step_fn, n_steps, strm, sync_ranks=True):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if sync_ranks:
            barrier()
        else:
            torch.cuda.synchronize()
        with torch.cuda.stream(strm):
            ev0.record(strm)
            for _ in range(n_steps):
                step_fn()
            ev1.record(strm)
        if sync_ranks:
            barrier()
        else:
            torch.cuda.synchronize()
        return ev0.elapsed_time(ev1)

    def step():
        f.band_exchange(0, B)
        f.run(0, B, 7)

    def measure(side_set):
        for s_ in range(B):
            set_side(f, s_, side_set[0])
        f.sync()
        for _ in range(max(args.warmup, 3)):
            step()
        f.sync()
        f.set_timing(False)
        l0 = f.launch_count()
        ms = timed(f, step, steps, stream)
        n_launch = f.launch_count() - l0
        f.set_timing(True)
        timed(f, step, steps, stream)
        kt = f.kernel_times()
        f.set_timing(False)
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), kt, n_launch

    ms_total, ktimes, launches = measure(side)
    ms_on, kt_on, _ = measure(side_on)          # leaves the all-on side information and its result in the slots
    value = B * steps * mpx / (ms_total * 1e-3)       # the picture is shared: whole-job pixels = B pictures per step
    value_on = B * steps * mpx / (ms_on * 1e-3)

    # ---- parity: own rows of slot 0 (all CTUs on) against the whole picture filtered by ONE context on rank 0 ----
    got = f.download_band(0)
    crcs = plane_crcs([got["y"], got["cb"], got["cr"]])
    all_crcs = [None] * world
    if world > 1:
        dist.all_gather_object(all_crcs, (y0, y1, crcs))
    else:
        all_crcs = [(y0, y1, crcs)]
    whole = None
    if rank == 0:
        g = v.InLoopFilter(w, h, 10, 10, 7, device=local, num_slots=B)
        pin_full = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in pic]
        for s_ in range(B):
            g.upload(s_, *(t.numpy() for t in pin_full))
            set_side(g, s_, side_on[0], sliced=False)
        g.run(0, 1, 7)
        ref = g.download(0)
        bad = []
        for r_, (a0, a1, c) in enumerate(all_crcs):
            want = plane_crcs([ref["y"][a0:a1], ref["cb"][a0 // 2:a1 // 2], ref["cr"][a0 // 2:a1 // 2]])
            if want != c:
                bad.append(r_)
        if bad:
            raise SystemExit(f"bench.py: band parity FAILED on ranks {bad}: the rows a band context produced differ from the whole-picture result")
        # the N = 1 figure of the same run: the whole picture, B resident copies, on rank 0's GPU alone
        gstream = torch.cuda.ExternalStream(g.stream(), device=torch.device("cuda", local))
        for _ in range(3):
            g.run(0, B, 7)
        g.sync()
        ms1_on = timed(g, lambda: g.run(0, B, 7), steps, gstream, sync_ranks=False)
        for s_ in range(B):
            set_side(g, s_, side[0], sliced=False)
        for _ in range(3):
            g.run(0, B, 7)
        g.sync()
        ms1 = timed(g, lambda: g.run(0, B, 7), steps, gstream, sync_ranks=False)
        whole = {"value": round(B * steps * mpx / (ms1 * 1e-3), 1), "ms_per_step": round(ms1 / steps, 4),
                 "all_on_value": round(B * steps * mpx / (ms1_on * 1e-3), 1), "all_on_ms_per_step": round(ms1_on / steps, 4)}
        g.close()
        del pic
    barrier()

    # end to end: own rows up from page-locked memory, halos from the neighbours, chain, own rows down; one picture at a time,
    # the ranks meet once per picture (uploads done -> halos may be pulled)
    e2e_steps = max(1, min(steps, args.e2e_steps))
    nbytes_own = sum(a.nbytes for a in own)

    def e2e_pic():
        f.upload_band(0, *own)
        set_side(f, 0, side[0])
        f.sync()
        if world > 1:
            dist.barrier()
        f.band_exchange(0)
        f.run(0, 1, 7)
        out = f.download_band(0)
        if world > 1:
            dist.barrier()   # nobody uploads the next picture while a neighbour still pulls halos
        return out

    e2e_pic()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_pic()
    barrier()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = e2e_steps * mpx / float(t.item())
    rec = None
    if rank == 0:
        peak, _src = hbm_peak()
        own_px = f.rows * w   # pixels rank 0 really filters per picture (own rows + redundant halo rows)
        rec = {"what": "BASELINE config 4: ONE 7680x4320 picture in CTU-row bands, one band per GPU; a step = halo exchange + chain for the resident pictures (strong scaling)",
               "value": round(value, 1), "unit": "Mpixel/s", "ms_per_step": round(ms_total / steps, 4), "steps": steps, "pictures_per_step": B,
               "bands": bands.band_partition((h + 127) // 128, world), "halo_rows_per_side": 16, "halo_bytes_per_picture_rank0": halo_rows * w * 3,
               "exchange": "one copy kernel per step reads the neighbours' input planes over NVLink P2P (CUDA IPC mapping between the per-GPU processes), no collective",
               "bands_parity": "ok", "parity_how": "CRC-32 per plane of every rank's own rows (all CTUs on) == the same rows of the whole picture filtered by one context on rank 0",
               "per_kernel": kernel_table(ktimes, peak, steps), "chain": chain_table(ktimes, ms_total, steps, B * own_px, peak),
               "all_on": {"value": round(value_on, 1), "ms_per_step": round(ms_on / steps, 4), "per_kernel": kernel_table(kt_on, peak, steps), "chain": chain_table(kt_on, ms_on, steps, B * own_px, peak)},
               "n1_whole_picture_same_run": whole,
               "strong_scaling_efficiency": {"stream_decisions": round(value / (world * whole["value"]), 3), "all_on": round(value_on / (world * whole["all_on_value"]), 3),
                                             "formula": "value / (n_gpus x whole-picture value of rank 0 in this run)"},
               "e2e": {"value": round(e2e_value, 1), "unit": "Mpixel/s", "h2d_bytes_per_step": nbytes_own, "d2h_bytes_per_step": nbytes_own, "steps": e2e_steps,
                       "path": "per picture and rank: upload_band (own rows, page-locked) + side information + barrier + band_exchange + run + download_band"},
               "gpu_launches": launches}
    f.close()
    return rec


def streams_record(args, rank, world, local, dist, torch, v):
    """BASELINE config 5: 64 independent 1080p low-delay streams dealt round-robin to the GPUs, every picture of every stream resident,
    a step = the chain over all of them (strong scaling: the 64 streams are the fixed job)."""
    from vvcsoftware_vtm_b200 import bands
    wl = WORKLOADS["ld_1080p_x64"]
    w, h = wl["width"], wl["height"]
    mpx = w * h / 1e6
    sets = [load_sideinfo(n) for n in wl["npz"]]
    mine = bands.deal_streams(wl["streams"], world)[rank]
    side = [pic for st in mine for pic in sets[st % len(sets)]]
    B = len(side)
    total_pics = sum(len(sets[st % len(sets)]) for st in range(wl["streams"]))
    steps = args.steps
    planes = synth_planes(w, h, 4, seed=3000 + rank)
    f = v.InLoopFilter(w, h, 10, 10, 7, device=local, num_slots=B)
    pins = [[torch.from_numpy(np.ascontiguousarray(p)).pin_memory() for p in trip] for trip in planes]

    def set_side(slot, si):
        f.set_deblock_info(slot, si["db_params"].tobytes(), si["db_info"], si.get("db_info_c"), si.get("db_mv16"), None, si["ctu_slice"])
        f.set_sao_params(slot, si["sao_ctus"])
        f.set_alf_params(slot, si["alf_params"].tobytes(), si["alf_ctu_enable"])

    for s_ in range(B):
        f.upload(s_, *(t.numpy() for t in pins[s_ % len(pins)]))
    stream = torch.cuda.ExternalStream(f.stream(), device=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    out = {}
    for label, side_set in (("stream_decisions", side), ("all_on", all_on_sideinfo(side))):
        for s_ in range(B):
            set_side(s_, side_set[s_])
        f.sync()
        for _ in range(3):
            f.run(0, B, 7)
        f.sync()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        with torch.cuda.stream(stream):
            ev0.record(stream)
            for _ in range(steps):
                f.run(0, B, 7)
            ev1.record(stream)
        barrier()
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        out[label] = {"value": round(total_pics * steps * mpx / (ms * 1e-3), 1), "ms_per_step": round(ms / steps, 4)}
    f.close()
    if rank != 0:
        return None
    return {"what": "BASELINE config 5: 64 independent 1920x1080 low-delay streams (9 pictures each, two encoded streams replicated) dealt round-robin to the GPUs, no collective; "
                    "a step = the chain over every resident picture of every stream (strong scaling over the fixed 64 streams)",
            "unit": "Mpixel/s", "streams": wl["streams"], "pictures_total": total_pics, "pictures_on_rank0": B, "steps": steps,
            "value": out["stream_decisions"]["value"], "ms_per_step": out["stream_decisions"]["ms_per_step"], "all_on": out["all_on"]}


def run_bands(args, wl):
    """`--workload intra_8k_bands`: the band record as the line of its own."""
    import torch
    import torch.distributed as dist
    import vvcsoftware_vtm_b200 as v
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    if world > 1:
        bind_to_gpu_numa(local)
    v.load_library()
    clocks = ClockSampler(local, period=0.01)
    clocks.start()
    rec = bands_record(args, wl, rank, world, local, dist, torch, v)
    clk = clocks.finish()
    if rank == 0:
        peak, peak_src = hbm_peak()
        pk = rec["per_kernel"]
        dom = dominant(pk)
        line = {"metric": "deblock+SAO+ALF Mpixel/s", "value": rec["value"], "unit": "Mpixel/s", "n_gpus": world, "steps": rec["steps"], "warmup": max(args.warmup, 3),
                "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int16", "data": "synthetic",
                "config": {"workload": wl["desc"], "pictures_per_step": rec["pictures_per_step"], "bands": rec["bands"]},
                "roofline": {"bound": "hbm", "kernel": dom, "achieved": pk[dom]["algo_gbs"], "peak": peak, "unit": "GB/s", "frac": pk[dom]["frac"], "traffic": None, "peak_source": peak_src,
                             "note": "per-kernel numbers of rank 0 (its band incl. halo rows)"},
                "bands_8k": rec, "cpu_baseline": None, "e2e": rec["e2e"], "gpu_launches": rec["gpu_launches"], "clocks": clk}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_b200(args, wl):
    import torch
    import torch.distributed as dist
    import vvcsoftware_vtm_b200 as v

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libilf_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        bind_to_gpu_numa(local)
    v.load_library()

    w, h = wl["width"], wl["height"]
    mpx = w * h / 1e6
    if "streams" in wl:
        # independent streams dealt round-robin to the ranks; every stream brings its own pictures (strong scaling)
        from vvcsoftware_vtm_b200 import bands
        sets = [load_sideinfo(n) for n in wl["npz"]]
        mine = bands.deal_streams(wl["streams"], world)[rank]
        side = [pic for st in mine for pic in sets[st % len(sets)]]
    else:
        side = load_sideinfo(args.workload)
    B = args.batch or len(side)
    planes = synth_planes(w, h, min(B, 4), seed=1000 + rank)
    f = v.InLoopFilter(w, h, 10, 10, 7, device=local, num_slots=B)

    def set_side(slot, si):
        f.set_deblock_info(slot, si["db_params"].tobytes(), si["db_info"], si.get("db_info_c"), si.get("db_mv16"), None, si["ctu_slice"])
        f.set_sao_params(slot, si["sao_ctus"])
        f.set_alf_params(slot, si["alf_params"].tobytes(), si["alf_ctu_enable"])

    pinned_planes_in = [[torch.from_numpy(np.ascontiguousarray(p)).pin_memory() for p in trip] for trip in planes]
    for s in range(B):
        f.upload(s, *(t_.numpy() for t_ in pinned_planes_in[s % len(planes)]))
        set_side(s, side[s % len(side)])
    f.sync()
    stream = torch.cuda.ExternalStream(f.stream(), device=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ----
    def measure(side_set, steps):
        """Time `steps` chain passes over the B resident pictures with the given side information (CUDA events on the
        library's compute stream, barrier + synchronize on both sides, max over ranks)."""
        for s in range(B):
            set_side(s, side_set[s % len(side_set)])
        f.sync()
        for _ in range(max(args.warmup, 3)):
            f.run(0, B, 7)
        f.sync()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def region():
            barrier()
            with torch.cuda.stream(stream):
                ev0.record(stream)
                for _ in range(steps):
                    f.run(0, B, 7)
                ev1.record(stream)
            barrier()
            return ev0.elapsed_time(ev1)
        # pass 1 -- the timed region proper: K steps, nothing on the stream but the library's kernels
        f.set_timing(False)
        l0 = f.launch_count()
        ms = region()
        n_launch = f.launch_count() - l0
        # pass 2 -- the same K steps with an event pair around every launch (the per-kernel durations of the roofline);
        # the pairs cost about 5 us per launch, which is why they are kept out of pass 1
        f.set_timing(True)
        ms_instr = region()
        kt = f.kernel_times()
        f.set_timing(False)
        t = torch.tensor([ms, ms_instr], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0].item()), kt, n_launch, float(t[1].item())

    clocks = ClockSampler(local, period=0.01)
    clocks.start()
    ms_on, kt_on, _, msi_on = measure(all_on_sideinfo(side), args.steps)      # worst case: every CTU filtered by every stage
    ms_total, ktimes, launches, msi_total = measure(side, args.steps)         # the stream's own decisions (headline)
    clk = clocks.finish()
    if args.dump_outputs and rank == 0:
        dump_outputs(f, B, w, h, args.dump_outputs)   # before the encoder-statistics runs below overwrite the slots' results
    value = world * B * args.steps * mpx / (ms_total * 1e-3)
    value_on = world * B * args.steps * mpx / (ms_on * 1e-3)

    # ---- the "next" row of SURVEY.md 8f that is built: encoder SAO statistics on the resident deblocked pictures ----
    # (not part of `value`: the decoder chain does not run it; reported as its own kernel against the HBM roofline)
    rng_o = np.random.default_rng(7)
    cw_, ch_ = (wl["width"] + 127) // 128, (wl["height"] + 127) // 128
    av = np.full(cw_ * ch_, 0x15, np.uint8)
    av[np.arange(cw_ * ch_) % cw_ == 0] &= ~np.uint8(0x11)
    av[:cw_] &= ~np.uint8(0x14)
    for s_ in range(B):
        org = [np.clip(p.astype(np.int32) + rng_o.integers(-6, 7, p.shape), 0, 1023).astype(np.int16) for p in planes[s_ % len(planes)]]
        f.set_original(s_, org[0], org[1], org[2], av)
    f.run(0, B, 1)                     # deblocked pictures in the slots, as in the encoder
    for _ in range(3):
        f.sao_stats(0, B)
    f.sync()
    f.set_timing(True)
    for _ in range(args.steps):
        f.sao_stats(0, B)
    kt_stats = f.kernel_times()["sao_stats"]
    f.set_timing(False)
    # encoder ALF statistics (classification + covariances) on the SAO'd pictures, and the decoded-picture hash of a resident picture
    f.run(0, B, 3)
    for _ in range(2):
        f.alf_stats(0, B)
    f.sync()
    f.set_timing(True)
    for _ in range(args.steps):
        f.alf_stats(0, B)
    kt_alf_stats = f.kernel_times()["alf_stats"]
    f.set_timing(False)
    f.picture_hash(0, "crc")
    t_h = time.perf_counter()
    for _ in range(10):
        f.picture_hash(0, "crc")
    hash_ms = (time.perf_counter() - t_h) / 10 * 1e3

    # ---- end to end through the public API: host planes + side information in, filtered host planes out ----
    # Host buffers are page-locked (what a host integration does with its picture buffers: ilf_host_alloc /
    # ilf_host_register), every picture crosses PCIe in both directions inside the timed region, and the slots are
    # cycled so that upload, kernels and download of neighbouring pictures overlap (include/ilf_b200.h "transfer pipeline").
    def pin(a):
        t_ = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t_, t_.numpy()

    keep = []
    pin_in = []
    for trip in planes:
        tn = [pin(p) for p in trip]
        keep += [t_ for t_, _ in tn]
        pin_in.append(tuple(n for _, n in tn))
    pin_side = []
    for si in side:
        d = {}
        for k, v_ in si.items():
            if isinstance(v_, np.ndarray) and v_.nbytes >= 4096:
                t_, n_ = pin(v_)
                keep.append(t_)
                d[k] = n_
            else:
                d[k] = v_
        pin_side.append(d)
    Be = min(B, 32)   # slots in rotation for the end-to-end leg
    outs = [v.pinned_planes(w, h) for _ in range(Be)]
    h2d = sum(p.nbytes for p in planes[0])
    d2h = h2d

    def side_bytes(si):
        return sum(si[k].nbytes for k in ("db_params", "db_info", "db_info_c", "db_mv16", "ctu_slice", "sao_ctus", "alf_params", "alf_ctu_enable") if k in si)

    def e2e_step():
        nb = 0
        for s in range(Be):
            f.wait(s)                       # the slot's previous result has reached the host
            f.upload(s, *pin_in[s % len(pin_in)])
            si = pin_side[s % len(pin_side)]
            set_side(s, si)
            nb += side_bytes(si)
            f.run(s, 1, 7)
            f.download_async(s, outs[s])
        return nb

    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    for _ in range(2):
        side_b = e2e_step()
    f.sync()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    f.sync()
    barrier()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * Be * e2e_steps * mpx / float(t.item())

    f.close()
    # ---- the other sharded configurations of BASELINE.json, in the same line (the driver's scaling run launches only this command) ----
    sub = {}
    if not args.quick and "streams" not in wl:
        torch.cuda.empty_cache()
        sub["bands_8k"] = bands_record(args, WORKLOADS["intra_8k_bands"], rank, world, local, dist, torch, v)
        sub["streams_64"] = streams_record(args, rank, world, local, dist, torch, v)
    if rank == 0:
        peak, peak_src = hbm_peak()
        per_kernel = kernel_table(ktimes, peak, args.steps)
        dom = dominant(per_kernel)
        ach = per_kernel[dom]["algo_gbs"]
        pk_on = kernel_table(kt_on, peak, args.steps)
        dom_on = dominant(pk_on)
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()
        cpu = cpu_baseline(wl, cores, side, planes) if (world == 1 and not args.no_cpu_baseline and not args.quick) else None
        dropin = dropin_leg() if (world == 1 and not args.quick) else None
        line = {"metric": "deblock+SAO+ALF Mpixel/s", "value": round(value, 1), "unit": "Mpixel/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": round(ms_total / args.steps, 4), "higher_is_better": True, "scaling": wl.get("scaling", "weak"),
                "vs_baseline": None, "dtype": "int16", "data": "synthetic",
                "config": shared_config(wl, args.workload, world),
                "config_detail": {"batch_pictures_per_gpu": B, "side_info": f"real, bench_data/{','.join(wl.get('npz', [args.workload]))}.npz ({len(side)} pictures per GPU)",
                                  "planes": "synthetic texture + 8x8 blockiness", "l2": f"working set {B * 2 * h2d / 1e6:.0f} MB per stage > 126 MB L2 (inputs larger than L2, no flush)",
                                  "parallelism": f"independent pictures, {world} GPU(s), no collective",
                                  "run_lanes": f.run_lanes(),
                                  "run_lanes_what": "ilf_run deals the chain over the resident batch to this many compute streams (groups of pictures of similar cost): value / ms_per_step are measured that way, the per-kernel durations with one kernel at a time on one stream"},
                "roofline": {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                             "traffic": (ncu_traffic(dom, B) or {}).get("bytes_per_launch"), "traffic_detail": ncu_traffic(dom, B),
                             "peak_source": peak_src, "chain": chain_table(ktimes, ms_total, args.steps, B * mpx * 1e6, peak), "per_kernel": per_kernel,
                             "per_kernel_pass": {"what": "per-kernel durations come from a second pass over the same K steps with a CUDA event pair around every launch; the pairs are kept out of the timed region of value / ms_per_step",
                                                 "ms_per_step": round(msi_total / args.steps, 4), "all_on_ms_per_step": round(msi_on / args.steps, 4)},
                             "all_on": {"what": "same pictures and deblocking information, SAO and ALF forced on for every CTU of every component (18 B/pixel)",
                                        "value": round(value_on, 1), "unit": "Mpixel/s", "ms_per_step": round(ms_on / args.steps, 4), "kernel": dom_on,
                                        "chain": chain_table(kt_on, ms_on, args.steps, B * mpx * 1e6, peak), "per_kernel": pk_on}},
                "next_rows": {"sao_stats": dict(kernel_table({"sao_stats": kt_stats}, peak)["sao_stats"],
                                                what="encoder SAO statistics (EncSampleAdaptiveOffset::getStatistics) of the resident deblocked pictures, one launch per step; algorithmic bytes = deblocked + original picture read once (6 B/pixel)",
                                                mpixel_per_s=round(B * mpx / (kt_stats[0] / max(kt_stats[1], 1) * 1e-3), 1)),
                              "alf_stats": dict(kernel_table({"alf_stats": kt_alf_stats}, peak)["alf_stats"],
                                                what="encoder ALF statistics (EncAdaptiveLoopFilter::deriveClassification + deriveStatsForFiltering) of the resident SAO'd pictures: classification + three covariance launches per step; multiply-bound (105 IMAD per luma sample), algorithmic bytes = reconstructed + original picture read once (6 B/pixel)",
                                                mpixel_per_s=round(B * mpx / (kt_alf_stats[0] / max(kt_alf_stats[1], 1) * 1e-3), 1)),
                              "picture_hash": {"ms_per_picture": round(hash_ms, 3), "what": "ilf_picture_hash (CRC of the three planes of one resident picture, host call to host result: two launches + 24 bytes down)"}},
                "cpu_baseline": cpu,
                "e2e": {"value": round(e2e_value, 1), "unit": "Mpixel/s", "h2d_bytes_per_step": Be * h2d + side_b, "d2h_bytes_per_step": Be * d2h, "pictures_per_step": Be,
                        "host_ceiling": host_ceiling(world, (Be * h2d + side_b) / Be, mpx),
                        "steps": e2e_steps, "path": "per picture InLoopFilter.upload + set_deblock_info/set_sao_params/set_alf_params + run + download_async (C ABI ilf_upload / ilf_set_* / ilf_run / ilf_download_async / ilf_wait), page-locked host buffers, slots cycled"},
                "gpu_launches": launches, "clocks": clk}
        if dropin is not None:
            line["dropin"] = dropin
        line.update({k: r for k, r in sub.items() if r is not None})
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=list(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="pictures resident per GPU and filtered per step (default: every picture of the workload's side information once, e.g. the 17 pictures of one 4K random-access GOP)")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="kernel A/B runs: no CPU baseline, no drop-in leg, no bands_8k / streams_64 sub-records")
    ap.add_argument("--bands-batch", type=int, default=16, help="resident 8K pictures per step of the band configuration")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the filtered pictures of the last step as DIR/{y,cb,cr}.npy "
                                                         "(float32 [picture, row, column]; a fixed sample of rows when the batch exceeds 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.workload = args.workload or default_workload()
    wl = WORKLOADS[args.workload]
    if args.dump_outputs and (args.impl != "b200" or wl.get("bands")):
        ap.error("--dump-outputs needs --impl b200 and a workload filtered as whole pictures")
    if args.impl == "reference":
        run_reference(args, wl)
    elif wl.get("bands"):
        run_bands(args, wl)
    else:
        run_b200(args, wl)


if __name__ == "__main__":
    main()
