#!/usr/bin/env python
"""bench.py — whole-encode throughput of the B200 JPEG encode path (BASELINE.json: "encode Mpx/s").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload image16k|frame4k]
                    [--dump-outputs DIR]

A "step" is one complete encode (K1 colour/DCT/quant -> K2 symbol statistics -> host Huffman table build ->
K3 Huffman pack -> K4 byte stuffing) of one synthetic image per GPU.  Default workload: the 16384x16384 (268 Mpx)
image of BASELINE.json configs[3] -- the configuration the metric's target is quoted on; it fits one GPU.
With N > 1 (torchrun, one rank per GPU) every rank encodes its own image (weak scaling, no data-path collective:
a single image is never split, SURVEY.md 8e).

value   = Mpx/s with the RGB already resident in HBM (scan left in HBM)
e2e     = Mpx/s through jpgenc_encode_rgb with pinned HOST buffers: H2D of the pixels and D2H of the JPEG inside the
          timed region
roofline= the K1 kernel (fused colour+subsample+DCT+quant+zigzag): 6 algorithmic bytes per padded pixel / its
          CUDA-event duration, against the measured copy bandwidth in MEASURED_PEAKS.json
extra.batch1080p = BASELINE configs[4] on EVERY N: the 1024 frames of 1920x1080 are partitioned over the ranks (strong
          scaling, no data-path collective) and timed resident, with the files returned, and end to end from pinned host
          memory; sizes of all frames and the SHA-256 of frame 0 are checked against tests/golden/batch1080p.json.
cpu_baseline = the reference encoder itself (oracle/_ref, built from /root/reference by oracle/build_ref.sh) on the box's
          host cores, OMP_NUM_THREADS=1, on a bounded sample (2048x2048) of the same synthetic.
--impl reference = the same binary on the headline workload itself: the 16384x16384 file, OMP_NUM_THREADS=1 (north_star:
          "single-threaded"; its three std::async channel tasks still run), ONE timed encode whatever --steps says (an
          encode takes ~45 s + ~9 s of PPM loading); the best multi-threaded figure is reported beside it.
--dump-outputs DIR = after the timed steps, rank 0 writes what its last timed step produced as float32/float64 .npy files
          in DIR, so that two builds can be compared output for output on the same seeded input: the JPEG file (jpeg.npy,
          one value per byte), and for batch1080p the files of its frames back to back (jpeg.npy) and their sizes
          (sizes.npy).  Past DUMP_BYTES the bytes are a fixed, seeded sample (jpeg_sample.npy, jpeg_sample_offsets.npy).
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "image16k": (16384, 16384, "single 16384x16384 synthetic image (268 Mpx), whole encode"),
    "frame4k": (3840, 2160, "single 3840x2160 synthetic frame, whole encode"),
    "batch1080p": (1920, 1080, "batch of 1024 synthetic 1920x1080 frames sharded by image across the ranks"),
}
BATCH_FRAMES = 1024
CPU_SAMPLE = (2048, 2048)          # bounded sample of the same generator for the CPU arms (~0.7 s per encode)
if os.environ.get("JPGENC_BENCH_CPU_SAMPLE"):                      # tests use a smaller one
    CPU_SAMPLE = tuple(int(x) for x in os.environ["JPGENC_BENCH_CPU_SAMPLE"].split("x"))
METRIC, UNIT = "encode_throughput", "Mpx/s"
DUMP_BYTES = 60 << 20              # --dump-outputs writes at most this much


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons of one GPU while the timed region runs (B200_PROFILING.md recipe).  Sampled through NVML
    inside this process: spawning nvidia-smi every few milliseconds initialises NVML over and over and takes driver locks
    that delay the CUDA calls being timed, on every rank at once.  nvidia-smi is the fallback when pynvml is missing."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = index
            if vis and all(t.strip().isdigit() for t in vis.split(",")) and index < len(vis.split(",")):
                phys = int(vis.split(",")[index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        bits = [n.nvmlClocksThrottleReasonHwSlowdown, n.nvmlClocksThrottleReasonHwThermalSlowdown,
                n.nvmlClocksThrottleReasonSwThermalSlowdown, n.nvmlClocksThrottleReasonSwPowerCap]
        return [str(sm), str(self.max_sm)] + ["Active" if r & b else "Not Active" for b in bits]

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        return [c.strip() for c in out.split(",")] if out else None

    def run(self):
        while not self.stop_flag.is_set():
            try:
                row = self._sample_nvml() if self.nvml else self._sample_smi()
                if row:
                    self.rows.append(row)
            except Exception:
                pass
            self.stop_flag.wait(0.02 if self.nvml else 0.05)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        reasons = sorted({self.NAMES[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml else "nvidia-smi"}


# ---------------------------------------------------------------------------------------------------------------
# CPU arms: the reference encoder on host cores
# ---------------------------------------------------------------------------------------------------------------
def _ref_binary():
    p = os.path.join(ROOT, "oracle", "_ref", "jpgEnc_ref")
    return p if os.path.exists(p) else None


def _shm_dir():
    return "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()


def _write_synth_ppm(w: int, h: int, seed: int = 0) -> str:
    """the synthetic image as a P6 file, generated band by band (a 16384x16384 image is 805 MB)"""
    from concurrent.futures import ThreadPoolExecutor
    from jpgenc_b200.synth import synth_rgb
    path = os.path.join(_shm_dir(), f"jpgenc_bench_{w}x{h}_{os.getpid()}.ppm")
    band = max(16, (8 << 20) // max(1, w * 3))
    starts = list(range(0, h, band))
    with open(path, "wb") as f, ThreadPoolExecutor(min(8, os.cpu_count() or 1)) as ex:
        f.write(b"P6\n%d %d\n255\n" % (w, h))
        for part in ex.map(lambda y0: synth_rgb(w, h, seed, rows=slice(y0, min(h, y0 + band))).tobytes(), starts):
            f.write(part)
    return path


def _run_reference_once(path: str, omp_threads: int):
    """(seconds of Image::writeJPEG -- "Encoding duration", src/Image.cpp:975 --, seconds of loadPPM) for one run of the
    reference CLI"""
    env = dict(os.environ, OMP_NUM_THREADS=str(omp_threads))
    out = subprocess.run([_ref_binary(), path, path + ".jpg"], capture_output=True, text=True, env=env, check=True).stdout
    m = re.search(r"Encoding duration: (\d+) ms", out)
    ld = re.search(r"PPM loading took (\d+) ms", out)
    return int(m.group(1)) / 1e3, (int(ld.group(1)) / 1e3 if ld else None)


def _run_port_once(rgb) -> float:
    from oracle.pyoracle import Oracle
    o = Oracle()
    t = time.perf_counter()
    o.encode_rgb(rgb)
    return time.perf_counter() - t


def cpu_arm(w: int, h: int, steps: int, warmup: int, what: str):
    """The reference on host cores, on a w x h image of the bench's generator (seed 0).
    -> (Mpx/s at OMP_NUM_THREADS=1, ms per encode, dict cpu_baseline).  north_star asks for the single-threaded encoder;
    the figure with all host threads is reported beside it (on small hosts the six OpenMP regions cost more than they
    save: BASELINE.md)."""
    mpx = w * h / 1e6
    nproc = os.cpu_count() or 1
    if _ref_binary():
        path = _write_synth_ppm(w, h, 0)
        try:
            for _ in range(warmup):
                _run_reference_once(path, 1)
            runs = [_run_reference_once(path, 1) for _ in range(steps)]
            multi = _run_reference_once(path, nproc) if nproc > 1 else None
        finally:
            for p in (path, path + ".jpg"):
                if os.path.exists(p):
                    os.remove(p)
        sec = sum(r[0] for r in runs) / len(runs)
        load = [r[1] for r in runs if r[1] is not None]
        cb = {"value": round(mpx / sec, 3), "unit": UNIT, "cores": 1, "kind": "reference",
              "sample": (f"{what}: reference CLI (oracle/_ref/jpgEnc_ref), Image::writeJPEG time ('Encoding duration') on the {w}x{h} synthetic "
                         f"(bench generator, seed 0), OMP_NUM_THREADS=1 (its 3 std::async channel tasks still run), {steps} timed encode(s), {warmup} warm-up"),
              "encode_s": round(sec, 3), "ppm_load_s": round(sum(load) / len(load), 3) if load else None,
              "host_cores_available": nproc}
        if multi:
            cb["all_threads"] = {"value": round(mpx / multi[0], 3), "unit": UNIT, "cores": nproc, "encode_s": round(multi[0], 3),
                                 "note": f"same file, OMP_NUM_THREADS={nproc}, one encode"}
    else:
        from jpgenc_b200.synth import synth_rgb
        rgb = synth_rgb(w, h, 0)
        for _ in range(max(1, warmup)):
            _run_port_once(rgb)
        times = [_run_port_once(rgb) for _ in range(steps)]
        sec = sum(times) / len(times)
        cb = {"value": round(mpx / sec, 3), "unit": UNIT, "cores": 1, "kind": "port",
              "sample": f"{what}: oracle C port (oracle/liboracle.so; oracle/_ref absent) on the {w}x{h} synthetic, single thread, {steps} encodes",
              "host_cores_available": nproc}
    return mpx / sec, sec * 1e3, cb


def headline_config(workload: str, world: int) -> dict:
    """the `config` object of the JSON line -- the same for our arm and for the reference arm"""
    w, h, desc = WORKLOADS[workload]
    return {"workload": desc, "width": w, "height": h, "images_per_gpu": 1,
            "l2": "inputs larger than L2 (805 MB RGB + 805 MB coefficients per step)" if w * h > 50e6 else "inputs smaller than L2",
            "parallelism": f"independent images x{world}", "subsampling": "4:2:0 mean",
            "tables": "image-optimal length-limited Huffman per image"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w, h, _ = WORKLOADS[args.workload]
    if os.environ.get("JPGENC_BENCH_REF_SIZE"):                    # tests use a small image
        w, h = (int(x) for x in os.environ["JPGENC_BENCH_REF_SIZE"].split("x"))
    # ONE timed encode of the workload's own image (268 Mpx: ~45 s + ~9 s load at OMP_NUM_THREADS=1), no warm-up run
    big = w * h > 50e6
    steps_timed = 1 if big else max(1, min(args.steps, 5))
    v, ms, cb = cpu_arm(w, h, steps_timed, 0 if big else 1, "the headline workload itself")
    line = {"impl": "reference", "metric": METRIC, "value": round(v, 3), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "steps_timed": steps_timed, "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": headline_config(args.workload, int(os.environ.get("WORLD_SIZE", str(args.gpus)))),
            "cpu_baseline": cb,
            "note": "same image as our arm (same generator, seed 0, full size); steps_timed encodes were timed -- one encode of this image takes "
                    "about a minute on one thread, so --steps is not honoured beyond that",
            "e2e": {"value": round(v, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ---------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch

    from jpgenc_b200.capi import Encoder, pinned_empty, pinned_free

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(local)

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    w, h, desc = WORKLOADS[args.workload]
    numa = (-1, 0)
    if world > 1 and not os.environ.get("JPGENC_BENCH_NO_NUMA"):
        from jpgenc_b200.capi import bind_host_to_device_numa
        numa = bind_host_to_device_numa(local)       # before any pinned allocation: node-local staging buffers
    enc = Encoder(local)
    npx = w * h
    padded_px = ((w + 15) // 16 * 16) * ((h + 15) // 16 * 16)
    d_rgb = enc.dev_alloc(npx * 3)
    enc.synth_rgb(d_rgb, w, h, rank)                 # a different image per rank
    enc.bind_device_rgb(d_rgb, w, h)
    enc.synchronize()

    # ---- device-resident: K steps of the whole encode, pixels in HBM, scan left in HBM -------------------
    # The library's event records between the kernels cost ~3 us each inside the replayed graphs (include/jpgenc_b200.h,
    # jpgenc_set_stage_timing), so the timed region carries only the two around the roofline kernel (level 1: K1's launch
    # duration is measured over exactly these K steps); the other stage times come from a second loop of K steps at level 2.
    sampler = ClockSampler(local)
    sampler.start()                                   # samples from the first warm-up step to the end of the timed steps
    enc.set_stage_timing(1)
    for _ in range(args.warmup):
        jpeg_bytes = enc.encode_bound(None)
    barrier()
    launches0 = enc.launch_count()
    s0 = enc.stats()                                  # the library keeps running sums of its per-stage CUDA-event times:
    enc.timer_begin()                                 # read once before and once after, no per-step polling in the loop
    for _ in range(args.steps):
        jpeg_bytes = enc.encode_bound(None)
    ms_total = enc.timer_end()
    s1 = enc.stats()
    dump = output_arrays(last_file(enc, jpeg_bytes)) if args.dump_outputs and rank == 0 else None
    n_timed = max(1, s1.timed_encodes - s0.timed_encodes)
    k1_ms = [(s1.sum_ms_k1 - s0.sum_ms_k1) / n_timed]
    launches = enc.launch_count() - launches0
    barrier()
    clocks = sampler.summary()
    ms_total = max_over_ranks(ms_total)
    ms_step = ms_total / args.steps
    value = world * npx / 1e6 / (ms_step / 1e3)
    # the same K steps with every stage's events on (stage_ms), and with none (what a caller gets by default)
    enc.set_stage_timing(2)
    for _ in range(3):
        enc.encode_bound(None)
    s0 = enc.stats()
    enc.timer_begin()
    for _ in range(args.steps):
        enc.encode_bound(None)
    ms_step_all_events = max_over_ranks(enc.timer_end()) / args.steps
    s1 = enc.stats()
    n_timed = max(1, s1.timed_encodes - s0.timed_encodes)
    fwd_ms = [(s1.sum_ms_forward - s0.sum_ms_forward) / n_timed]
    st_ms = [(s1.sum_ms_stats - s0.sum_ms_stats) / n_timed]; en_ms = [(s1.sum_ms_entropy - s0.sum_ms_entropy) / n_timed]
    enc.set_stage_timing(0)
    for _ in range(3):
        enc.encode_bound(None)
    enc.timer_begin()
    for _ in range(args.steps):
        enc.encode_bound(None)
    ms_step_no_events = max_over_ranks(enc.timer_end()) / args.steps
    barrier()
    stats = enc.stats()

    # ---- end to end: pinned host pixels in, JPEG bytes out in pinned host memory ---------------------------
    host_rgb, host_ptr = pinned_empty(npx * 3)
    enc.d2h(host_rgb, d_rgb)
    out_cap = int(jpeg_bytes) + 4096
    host_out, out_ptr = pinned_empty(out_cap)
    e2e_warm = min(args.warmup, 2) if npx > 50e6 else args.warmup
    for _ in range(max(1, e2e_warm)):
        n = enc.encode_rgb_into(host_ptr, w, h, out_ptr, out_cap)
    e2e_steps = min(args.steps, 20) if npx > 50e6 else args.steps      # 16 ms per step at 268 Mpx: bounded, still >= 0.3 s
    barrier()
    enc.timer_begin()
    h2d_ms_steps = []
    for _ in range(e2e_steps):
        n = enc.encode_rgb_into(host_ptr, w, h, out_ptr, out_cap)
        h2d_ms_steps.append(enc.stats().ms_h2d)        # the call has returned: its events are complete, nothing is waited for
    ms_e2e = max_over_ranks(enc.timer_end()) / e2e_steps
    barrier()
    assert n == jpeg_bytes and host_out[0] == 0xFF and host_out[1] == 0xD8 and host_out[n - 1] == 0xD9
    e2e_value = world * npx / 1e6 / (ms_e2e / 1e3)
    st_e2e = enc.stats()
    # the uploads of the timed steps on every rank: the step is as slow as the slowest rank's upload (from four ranks up
    # the simultaneous uploads share the host's memory and PCIe fabric and the ranks' rates differ)
    ms_h2d_mean = sum(h2d_ms_steps) / len(h2d_ms_steps)
    ms_h2d_max = max_over_ranks(ms_h2d_mean)               # mean over the timed steps, slowest / fastest rank
    ms_h2d_min = -max_over_ranks(-ms_h2d_mean)
    # what the link gives on this box: ONE plain copy of the same pinned buffer into the same device buffer, all ranks at the
    # same moment, nothing else running -- the ceiling the end-to-end step is measured against
    ceil_ms = []
    for _ in range(3):
        barrier()
        t = time.perf_counter()
        enc.h2d(d_rgb, host_rgb)
        ceil_ms.append(max_over_ranks((time.perf_counter() - t) * 1e3))
    barrier()
    ms_copy_only = min(ceil_ms)

    # ---- roofline of the dominant kernel (K1) ----------------------------------------------------------------
    peak, peak_src = measured_peak()
    k1 = sum(k1_ms) / len(k1_ms)
    alg_bytes = 6 * padded_px                          # 3 B RGB in + 1.5 samples x int16 out per padded pixel
    achieved = alg_bytes / (k1 / 1e3) / 1e9
    roofline = {"kernel": "forward_kernel (K1: colour+subsample+DCT+quant+zigzag)", "bound": "hbm", "achieved": round(achieved, 1),
                "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": None,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": round(k1, 4)}
    tr = os.path.join(ROOT, "profiles", "k1_traffic.json")     # dram bytes per launch from the committed ncu --set full capture
    if os.path.exists(tr):
        try:
            t = json.load(open(tr))
            # the capture is only quoted while K1's source is the one that was profiled: a changed forward.cu makes it null
            import hashlib
            with open(os.path.join(ROOT, "jpgenc_b200", "csrc", "forward.cu"), "rb") as f:
                same_k1 = hashlib.sha256(f.read()).hexdigest() == t.get("k1_source_sha256_at_capture")
            if t.get("workload") == args.workload and same_k1:
                roofline["traffic"] = t.get("dram_bytes_per_launch")
                roofline["traffic_source"] = t.get("source")
        except Exception:
            pass

    # the other stages against the same peak, from the bytes they must move (DESIGN.md section 3): K2 reads the coefficients
    # (128 B per block) and writes one 4-byte item per symbol (~4.2 per block on this image); K3a/K3b read the items twice and
    # write the raw scan, K4 reads and writes the scan
    n_blocks = int(stats.n_blocks)
    st_k2, st_k34 = sum(st_ms) / len(st_ms), sum(en_ms) / len(en_ms)
    scan_b = int(jpeg_bytes)
    k2_bytes = n_blocks * 128
    roofline["other_kernels"] = {
        "k2_symbol_stats": {"algorithmic_bytes": k2_bytes, "ms": round(st_k2, 4), "achieved": round(k2_bytes / (st_k2 / 1e3) / 1e9, 1),
                            "frac": round(k2_bytes / (st_k2 / 1e3) / 1e9 / peak, 4), "note": "coefficient read only; its item writes (4 B per symbol) not counted"},
        "k3_k4_entropy": {"algorithmic_bytes": 3 * scan_b, "ms": round(st_k34, 4), "achieved": round(3 * scan_b / (st_k34 / 1e3) / 1e9, 1),
                          "frac": round(3 * scan_b / (st_k34 / 1e3) / 1e9 / peak, 4),
                          "note": "raw scan written once, read once, stuffed scan written once; the item reads (~10x the scan) not counted: latency- and issue-bound stage, not HBM-bound"},
        "whole_encode": {"algorithmic_bytes": npx * 3 + scan_b, "ms": round(ms_step, 4), "achieved": round((npx * 3 + scan_b) / (ms_step / 1e3) / 1e9, 1),
                         "frac": round((npx * 3 + scan_b) / (ms_step / 1e3) / 1e9 / peak, 4),
                         "two_pass_floor_bytes": 9 * padded_px, "frac_of_two_pass_floor": round(9 * padded_px / (ms_step / 1e3) / 1e9 / peak, 4)},
    }
    line = {
        "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64",
        "data": "synthetic",
        "config": headline_config(args.workload, world),
        "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": npx * 3, "d2h_bytes_per_step": int(n),
                "ms_per_step": round(ms_e2e, 3), "steps": e2e_steps, "ms_h2d": round(ms_h2d_max, 3), "ms_h2d_fastest_rank": round(ms_h2d_min, 3),
                "ms_d2h": round(st_e2e.ms_d2h, 3),
                "h2d_gbps_per_gpu": round(npx * 3 / max(ms_h2d_max, 1e-6) / 1e6, 2),
                "ms_not_h2d": round(ms_e2e - ms_h2d_max, 3),
                "pcie_ceiling": {"ms_plain_copy": round(ms_copy_only, 3), "gbps_per_gpu": round(npx * 3 / ms_copy_only / 1e6, 2),
                                 "how": "one cudaMemcpy of the same pinned pixels on every rank at the same moment (barrier before), slowest rank, best of 3",
                                 "ms_step_minus_plain_copy": round(ms_e2e - ms_copy_only, 3)}},
        "gpu_launches": int(launches),
        "host": {"cores": os.cpu_count(), "numa_node_rank0": numa[0], "cpus_bound_rank0": numa[1]},
        "clocks": clocks,
        "roofline": roofline,
        "stage_ms": {"k1_forward": round(k1, 4), "k1_plus_refine": round(sum(fwd_ms) / len(fwd_ms), 4),
                     "k2_stats": round(sum(st_ms) / len(st_ms), 4), "k3_k4_entropy": round(sum(en_ms) / len(en_ms), 4),
                     "how": "k1_forward: event records around K1 inside the timed region (stage timing level 1); the others from a "
                            "second loop of the same K steps with every stage's records on (level 2)"},
        "stage_event_cost": {"ms_per_step_k1_events_only": round(ms_step, 4), "ms_per_step_all_stage_events": round(ms_step_all_events, 4),
                             "ms_per_step_no_events": round(ms_step_no_events, 4),
                             "note": "jpgenc_set_stage_timing: the library's default is no event records; each one is a graph node of ~3 us"},
        "jpeg_bytes": int(jpeg_bytes), "refined_blocks": int(stats.refined_blocks), "n_blocks": int(stats.n_blocks),
        "whole_encode_gbps_irreducible": round((npx * 3 + jpeg_bytes) / (ms_step / 1e3) / 1e9, 1),
    }
    pinned_free(host_ptr)
    pinned_free(out_ptr)
    enc.dev_free(d_rgb)

    # BASELINE configs[4] on every N (all ranks take part: strong scaling over the ranks); the other single-GPU
    # configurations and the CPU baseline on rank 0 at N = 1 only
    extra = {}
    if args.workload == "image16k" and not os.environ.get("JPGENC_BENCH_NO_BATCH"):
        try:
            extra["batch1080p"] = batch_section(enc, rank, world, barrier, max_over_ranks, reps=3)
        except AssertionError:
            raise
        except Exception as ex:
            extra["batch1080p"] = {"error": repr(ex)}
    if rank == 0 and world == 1:
        try:
            extra.update(extra_workloads(enc, args, peak))
        except Exception as ex:          # extras never invalidate the headline line
            extra["error"] = repr(ex)
        _, _, line["cpu_baseline"] = cpu_arm(CPU_SAMPLE[0], CPU_SAMPLE[1], steps=3, warmup=1,
                                             what="bounded sample of the workload (the full 16384x16384 image is what --impl reference times)")
    line["extra"] = extra
    enc.close()
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(line)


def last_file(enc, jpeg_bytes: int):
    """the JPEG file of the context's last encode_bound (jpgenc_assemble_last: headers + scan + EOI, no new encode)"""
    import ctypes
    import numpy as np
    out = np.empty(jpeg_bytes, np.uint8)
    n = ctypes.c_uint64()
    enc._check(enc.lib.jpgenc_assemble_last(enc.h, out.ctypes.data, out.size, ctypes.byref(n)))
    return out[: n.value]


def output_arrays(jpeg, budget=DUMP_BYTES):
    """the bytes as float32 values, one per byte; past `budget` a fixed, seeded sample of the bytes and their offsets"""
    import numpy as np
    if jpeg.size * 4 <= budget:
        return {"jpeg": jpeg.astype(np.float32)}
    idx = np.sort(np.random.default_rng(0).choice(jpeg.size, budget // 12, replace=False))
    return {"jpeg_sample": jpeg[idx].astype(np.float32), "jpeg_sample_offsets": idx.astype(np.float64)}


def write_outputs(dirname, arrays):
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def batch_golden():
    try:
        with open(os.path.join(ROOT, "tests", "golden", "batch1080p.json")) as f:
            return json.load(f)
    except Exception:
        return None


def batch_section(enc, rank, world, barrier, max_over_ranks, reps=3, frames_total=BATCH_FRAMES, keep_files=False):
    """BASELINE configs[4]: `frames_total` synthetic 1920x1080 frames (frame k = seed k), frame k encoded by the rank that
    owns it (contiguous shards, no data-path collective) -> strong scaling over the ranks.  Every figure is the host wall
    clock around ONE synchronous library call on this rank's shard, between barriers, max over ranks, mean of `reps`.
      resident        frames in HBM, files left in HBM (sizes and offsets reported)
      files_returned  frames in HBM, complete files back in ONE pinned host buffer (one device-to-host copy per pass)
      e2e             frames in pinned host memory, files back in pinned host memory (H2D + D2H inside)
    keep_files: res["files"] = the files of the last timed call, back to back (the three passes return the same files)"""
    import hashlib
    import numpy as np
    from jpgenc_b200.capi import pinned_empty, pinned_free
    from jpgenc_b200.sharding import frames_for_rank
    w, h, _ = WORKLOADS["batch1080p"]
    mine = frames_for_rank(frames_total, rank, world)
    nf, fbytes = len(mine), w * h * 3
    d_all = enc.dev_alloc(max(1, nf) * fbytes)
    for i, k in enumerate(mine):
        enc.synth_rgb(d_all + i * fbytes, w, h, k)
    enc.synchronize()
    dev_ptrs = [d_all + i * fbytes for i in range(nf)]

    def timed(fn):
        fn()                                           # warm-up with the full shard: buffers are sized by the largest pass seen
        tot = 0.0
        for _ in range(reps):
            barrier()
            t = time.perf_counter()
            res = fn()
            tot += max_over_ranks(time.perf_counter() - t)
        barrier()
        return tot / reps, res

    launches0 = enc.launch_count()
    dt_res, (offs, sizes, total) = timed(lambda: enc.encode_frames_packed(dev_ptrs, w, h, None, 0))
    launches = (enc.launch_count() - launches0) // (reps + 1)
    out, out_ptr = pinned_empty(total + 4096)
    dt_files, res2 = timed(lambda: enc.encode_frames_packed(dev_ptrs, w, h, out_ptr, out.size))
    host, host_ptr = pinned_empty(max(1, nf) * fbytes)
    enc.d2h(host, d_all)
    out[:] = 0
    dt_e2e, res3 = timed(lambda: enc.encode_frames_packed([host_ptr + i * fbytes for i in range(nf)], w, h, out_ptr, out.size, host_frames=True))
    # ---- parity, outside the timed regions: golden sizes of this rank's frames, SHA-256 of frame 0 (rank 0), JFIF framing
    gold = batch_golden()
    parity = {"checked": False}
    ok = res2 == (offs, sizes, total) and res3 == (offs, sizes, total)
    if gold and gold.get("frames", 0) >= frames_total:
        ok = ok and sizes == [gold["sizes"][k] for k in mine]
        parity = {"checked": True, "sizes_equal_golden": sizes == [gold["sizes"][k] for k in mine], "frames_checked": nf}
        if rank == 0 and nf:
            sha0 = hashlib.sha256(out[offs[0]: offs[0] + sizes[0]].tobytes()).hexdigest()
            parity["frame0_sha256_equals_reference_pin"] = sha0 == gold["sha256_frame0"]
            ok = ok and sha0 == gold["sha256_frame0"]
            if world == 1 and frames_total == gold["frames"]:
                hs = "".join(hashlib.sha256(out[offs[k]: offs[k] + sizes[k]].tobytes()).hexdigest() for k in range(nf))
                parity["all_files_sha256_equal_golden"] = hashlib.sha256(hs.encode()).hexdigest() == gold["sha256_of_frame_sha256s"]
                ok = ok and parity["all_files_sha256_equal_golden"]
    for k in range(nf):
        ok = ok and out[offs[k]] == 0xFF and out[offs[k] + 1] == 0xD8 and out[offs[k] + sizes[k] - 1] == 0xD9
    parity["ok"] = bool(ok)
    assert ok, f"batch output differs from the golden/reference data: {parity}"
    files = out[:total].copy() if keep_files else None
    pinned_free(host_ptr); pinned_free(out_ptr); enc.dev_free(d_all)
    mpx = frames_total * w * h / 1e6
    sec = {"resident": dt_res, "files_returned": dt_files, "e2e": dt_e2e}
    res = {"frames": frames_total, "frames_per_gpu": nf, "width": w, "height": h, "n_gpus": world, "scaling": "strong",
           "mode": "passes of 64-128 frames (the library picks the size from the shard), each one asynchronous chain K1 > K2 > device table "
                   "build > device sizes/offsets > K3 > K4 (files assembled on the device), rotating over 4 streams driven by one host "
                   "thread; one host synchronisation per pass",
           "timing": f"host wall clock around one synchronous call per rank, barrier before, max over ranks, mean of {reps}",
           "gpu_launches_per_call": int(launches), "jpeg_bytes_total_this_rank": int(total), "parity": parity}
    for k, dt in sec.items():
        res[k] = {"frames_per_s": round(frames_total / dt, 1), "mpx_per_s": round(mpx / dt, 1), "ms": round(dt * 1e3, 3)}
    res["e2e"]["h2d_bytes_per_gpu"] = nf * fbytes
    res["e2e"]["h2d_gbps_per_gpu"] = round(nf * fbytes / dt_e2e / 1e9, 2)
    if keep_files:
        res["files"], res["sizes"] = files, sizes
    return res


def run_batch(args):
    """--workload batch1080p: BASELINE configs[4] as the headline line (the default workload carries the same measurement in
    extra.batch1080p)."""
    import torch
    from jpgenc_b200.capi import Encoder

    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(local)

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    enc = Encoder(local)
    sampler = ClockSampler(local)
    sampler.start()
    reps = args.steps
    dump = bool(args.dump_outputs) and rank == 0
    b = batch_section(enc, rank, world, barrier, max_over_ranks, reps=reps, keep_files=dump)
    if dump:
        import numpy as np
        sizes = np.array(b.pop("sizes"), np.float64)
        write_outputs(args.dump_outputs, {"sizes": sizes, **output_arrays(b.pop("files"), DUMP_BYTES - sizes.nbytes)})
    clocks = sampler.summary()
    w, h, desc = WORKLOADS["batch1080p"]
    line = {"metric": METRIC, "value": b["resident"]["mpx_per_s"], "unit": UNIT, "n_gpus": world, "steps": reps, "warmup": 1,
            "ms_per_step": b["resident"]["ms"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32+f64", "data": "synthetic",
            "config": {"workload": desc, "frames": BATCH_FRAMES, "frames_per_gpu": b["frames_per_gpu"], "width": w, "height": h,
                       "mode": b["mode"], "timing": b["timing"], "l2": "inputs larger than L2 (%.1f GB of frames per GPU)" % (b["frames_per_gpu"] * w * h * 3 / 1e9)},
            "e2e": {"value": b["e2e"]["mpx_per_s"], "unit": UNIT, "h2d_bytes_per_step": b["e2e"]["h2d_bytes_per_gpu"],
                    "d2h_bytes_per_step": b["jpeg_bytes_total_this_rank"], "ms_per_step": b["e2e"]["ms"], "frames_per_s": b["e2e"]["frames_per_s"]},
            "frames_per_s": b["resident"]["frames_per_s"], "files_returned": b["files_returned"],
            "gpu_launches": b["gpu_launches_per_call"] * reps, "clocks": clocks, "parity": b["parity"]}
    enc.close()
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()
    if rank == 0:
        emit(line)


def extra_workloads(enc, args, peak):
    """the other single-GPU configurations of BASELINE.json, measured the same way (reported, not the headline)"""
    import numpy as np
    from jpgenc_b200.tables import ANNEX_K_LUMA
    out = {}
    # configs[1]: DCT + quant + zigzag microbenchmark, 2^24 blocks, 384 algorithmic bytes per block
    nb = 1 << 24
    d_in, d_out = enc.dev_alloc(nb * 256), enc.dev_alloc(nb * 128)
    enc.synth_blocks(d_in, nb)
    qy = ANNEX_K_LUMA
    for _ in range(3):
        refined = enc.dct_quant_blocks(d_in, d_out, nb, qy)
    enc.synchronize()
    enc.timer_begin()
    reps = 10
    for _ in range(reps):
        enc.dct_quant_blocks(d_in, d_out, nb, qy, want_refined=False)
    ms = enc.timer_end() / reps
    out["dct_microbench"] = {"blocks": nb, "ms": round(ms, 4), "gblocks_per_s": round(nb / ms / 1e6, 3),
                             "roofline": {"bound": "hbm", "achieved": round(nb * 384 / (ms / 1e3) / 1e9, 1), "peak": peak, "unit": "GB/s",
                                          "frac": round(nb * 384 / (ms / 1e3) / 1e9 / peak, 4)},
                             "refined_blocks": int(refined), "includes": "fast kernel + exact refinement kernel"}
    enc.dev_free(d_in)
    enc.dev_free(d_out)
    # configs[2]: one 3840x2160 frame
    if args.workload != "frame4k":
        w, h = 3840, 2160
        d = enc.dev_alloc(w * h * 3)
        enc.synth_rgb(d, w, h, 0)
        enc.bind_device_rgb(d, w, h)
        for _ in range(3):
            enc.encode_bound(None)
        enc.flush_l2()
        enc.synchronize()
        reps = 20
        tot = 0.0
        for _ in range(reps):
            enc.flush_l2()
            enc.timer_begin()
            enc.encode_bound(None)
            tot += enc.timer_end()
        enc.timer_begin()
        for _ in range(200):
            enc.encode_bound(None)
        warm = enc.timer_end() / 200
        enc.set_stage_timing(2)
        for _ in range(4):
            enc.flush_l2()
            enc.encode_bound(None)
        s = enc.stats()
        enc.set_stage_timing(0)
        out["frame4k"] = {"ms_per_frame": round(tot / reps, 4), "mpx_per_s": round(w * h / 1e6 / (tot / reps / 1e3), 1),
                          "ms_per_frame_l2_warm": round(warm, 4),
                          "k1_ms": round(s.ms_k1, 4), "l2": "flushed between iterations (256 MB write); l2_warm: 200 encodes back to back",
                          "stage_timing": "off in the timed loops (library default); k1_ms from separate encodes with it on"}
        enc.dev_free(d)
    # SURVEY 8(d): the high-entropy variant (uniform random u8, numpy default_rng(1)) that stresses K3/K4 -- ~37 AC symbols per
    # block and ~3 bit/px instead of 4.2 symbols per block and 0.32 bit/px
    w = h = 4096
    rng = np.random.default_rng(1)
    rgb = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    d = enc.dev_alloc(w * h * 3)
    enc.h2d(d, rgb)
    enc.bind_device_rgb(d, w, h)
    for _ in range(3):
        nbytes = enc.encode_bound(None)
    enc.synchronize()
    reps = 20
    enc.timer_begin()
    for _ in range(reps):
        enc.encode_bound(None)
    ms = enc.timer_end() / reps
    enc.set_stage_timing(2)
    for _ in range(4):
        enc.encode_bound(None)
    s = enc.stats()
    enc.set_stage_timing(0)
    out["noise4096"] = {"ms_per_image": round(ms, 4), "mpx_per_s": round(w * h / 1e6 / (ms / 1e3), 1), "jpeg_bytes": int(nbytes),
                        "bits_per_px": round(8 * nbytes / (w * h), 3), "k1_plus_refine_ms": round(s.ms_forward, 4), "k2_ms": round(s.ms_stats, 4),
                        "k3_k4_ms": round(s.ms_entropy, 4), "stuffed_ff": int(s.stuffed_ff)}
    enc.dev_free(d)
    return out


_REAL_STDOUT = None


def quiet_stdout():
    """Library chatter (NCCL prints its version to stdout at init) must not mix with the one JSON line: everything that
    writes to fd 1 from here on goes to stderr, emit() writes the result to the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=int(os.environ.get("WORLD_SIZE", "1")))
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="image16k", choices=list(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path computed in its last step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs: --impl ours only")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "batch1080p":
        run_batch(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
