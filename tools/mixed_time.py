"""Images of individual sizes: jpgenc_encode_images_packed against the one-by-one loop (jpgenc_bind_device_rgb +
jpgenc_encode_bound) on the same device-resident images, generated on the device from seeds.

    python tools/mixed_time.py [--reps 5] [--out DIR]

Workloads:
  W1  1024 images, sides uniform in [256, 2048] (seed 0)
  W2  4096 thumbnails, sides uniform in [64, 512] (seed 1)
  W3  1024 frames alternating 1920x1080 and 1920x1088: they differ in real_h only, so the mixed-size kernels run on nearly
      the workload of bench.py's batch1080p; compared with 1024 x 1920x1080 through jpgenc_encode_frames_packed, this is the
      cost of the mixed-size variant itself
For each: images/s and Gpx/s of the new call with sizes only and with the files copied into pinned memory, and of the loop
(files into pinned memory).  The variants alternate within every repetition; the spread over repetitions is reported.
Prints one JSON line per workload and writes them to DIR/mixed_time.json."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from jpgenc_b200.capi import Encoder, pinned_empty, pinned_free  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:                                               # reported, not fatal
        return f"nvidia-smi failed: {e}"


def workloads():
    r0 = np.random.default_rng(0).integers(256, 2049, size=(1024, 2))
    r1 = np.random.default_rng(1).integers(64, 513, size=(4096, 2))
    return {
        "W1_1024_sides_256_2048": [(int(w), int(h)) for w, h in r0],
        "W2_4096_thumbnails_64_512": [(int(w), int(h)) for w, h in r1],
        "W3_1024_alternating_1080_1088": [(1920, 1080 if k % 2 == 0 else 1088) for k in range(1024)],
    }


def timed(fn):
    t0 = time.perf_counter()
    fn()                                                                  # every call returns after its device work is done
    return time.perf_counter() - t0


def stats(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "min": xs[0], "max": xs[-1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    card = gpu_info()
    enc = Encoder(0)
    results = []
    for name, dims in workloads().items():
        sizes = [w * h * 3 for w, h in dims]
        at = np.concatenate([[0], np.cumsum([(s + 255) // 256 * 256 for s in sizes])]).astype(np.int64)
        base = enc.dev_alloc(int(at[-1]) + 256)
        for k, (w, h) in enumerate(dims):
            enc.synth_rgb(base + int(at[k]), w, h, k)
        enc.synchronize()
        ptrs = [base + int(a) for a in at[:-1]]
        ws, hs = [w for w, _ in dims], [h for _, h in dims]
        px = float(sum(w * h for w, h in dims))
        offs, fsizes, total = enc.encode_images_packed(ptrs, ws, hs, None, 0)        # warm-up, and the output size
        out, out_ptr = pinned_empty(total + 4096)
        one, one_ptr = pinned_empty(max(fsizes) + 65536)
        one_arr = one

        def mixed_sizes():
            enc.encode_images_packed(ptrs, ws, hs, None, 0)

        def mixed_files():
            o, s, t = enc.encode_images_packed(ptrs, ws, hs, out_ptr, out.size)
            assert t == total

        def loop():
            for p, w, h in zip(ptrs, ws, hs):
                enc.bind_device_rgb(p, w, h)
                enc.encode_bound(one_arr)

        variants = {"mixed_sizes_only": mixed_sizes, "mixed_files_pinned": mixed_files, "loop_files_pinned": loop}
        if name.startswith("W3"):
            fptrs = [base + int(at[k]) for k in range(0, len(dims), 2)]              # the 1920x1080 frames ...
            fptrs = (fptrs * 2)[: len(dims)]                                          # ... each twice: 1024 frames of one size
            enc.encode_frames_packed(fptrs, 1920, 1080, None, 0)
            px_frames = 1920.0 * 1080 * len(fptrs)
            variants["frames_packed_1080p_sizes_only"] = lambda: enc.encode_frames_packed(fptrs, 1920, 1080, None, 0)
            variants["frames_packed_1080p_files_pinned"] = lambda: enc.encode_frames_packed(fptrs, 1920, 1080, out_ptr, out.size)
        for fn in variants.values():                                                   # warm every path
            fn()
        times = {k: [] for k in variants}
        for rep in range(args.reps):
            for k, fn in variants.items():
                times[k].append(timed(fn))
        # the files of the new call against the loop's, image by image (a sample of 64 images)
        mixed_files()
        for k in range(0, len(dims), max(1, len(dims) // 64)):
            enc.bind_device_rgb(ptrs[k], ws[k], hs[k])
            n = enc.encode_bound(one_arr)
            assert one_arr[:n].tobytes() == out[offs[k]: offs[k] + fsizes[k]].tobytes(), f"{name}: image {k} differs from the loop"
        res = {"workload": name, "images": len(dims), "mpx": px / 1e6, "jpeg_bytes": total, "card": card, "reps": args.reps}
        for k, ts in times.items():
            n_img = len(dims)
            p = px_frames if k.startswith("frames") else px
            st = stats(ts)
            res[k] = {"ms": {q: v * 1e3 for q, v in st.items()}, "images_per_s": n_img / st["median"], "gpx_per_s": p / st["median"] / 1e9}
        res["speedup_files_vs_loop"] = res["loop_files_pinned"]["ms"]["median"] / res["mixed_files_pinned"]["ms"]["median"]
        print(json.dumps(res), flush=True)
        results.append(res)
        pinned_free(out_ptr)
        pinned_free(one_ptr)
        enc.dev_free(base)
    enc.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "mixed_time.json"), "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
