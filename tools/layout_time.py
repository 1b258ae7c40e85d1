"""Pixels in other layouts (row pitch, BGR, RGBA, BGRA) against tight RGB, device-resident unless stated, generated on the
device from seeds (torch does the layout conversions before timing starts).

    python tools/layout_time.py [--reps 5] [--out DIR]

Workloads:
  L1  one 16384x16384 image bound as tight RGB, RGB with pitch = 3w + 64, BGR, RGBA and BGRA: whole encode (host clock around
      jpgenc_encode_bound with the scan left on the device) and K1 alone (stage timing level 1: stats().ms_k1), with K1's
      HBM rate over the bytes it must move: 3 or 4 bytes read and 3 bytes of coefficients written per MCU-padded pixel
  L2  1024 frames of 1920x1080: BGRA through jpgenc_encode_images_packed_layout against tight RGB through
      jpgenc_encode_frames_packed (sizes only)
  L3  the 16384x16384 RGB image cut into 4096 tiles of 256x256: pointers into it plus its pitch through
      jpgenc_encode_images_packed_layout, against what a caller has to do without it -- a cudaMemcpy2DAsync of every tile into
      a packed buffer, then jpgenc_encode_images_packed (files into pinned memory for both)
  L4  16384x16384 RGBA from pinned host memory through jpgenc_encode_image, beside a plain host-to-device copy of the same
      bytes and jpgenc_encode_rgb of the RGB image from pinned memory (files into pinned memory)
The variants of a workload alternate within every repetition; median, min and max over the repetitions are reported, and the
files of the variants are compared with each other.  Prints one JSON line per workload and writes them to
DIR/layout_time.json."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from jpgenc_b200.capi import PIXEL_FORMATS, Encoder, pinned_empty, pinned_free  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:                                               # reported, not fatal
        return f"nvidia-smi failed: {e}"


def stats(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "min": xs[0], "max": xs[-1]}


def timed(fn):
    t0 = time.perf_counter()
    fn()                                                                  # every variant returns after its device work is done
    return (time.perf_counter() - t0) * 1e3


def run_variants(variants, reps):
    for fn in variants.values():                                          # warm every path
        fn()
    times = {k: [] for k in variants}
    for _ in range(reps):
        for k, fn in variants.items():
            times[k].append(timed(fn))
    return {k: stats(v) for k, v in times.items()}


def synth_device(enc, w, h, seed, frames=1):
    """(frames, h, w, 3) uint8 CUDA tensor filled by jpgenc_synth_rgb"""
    t = torch.empty((frames, h, w, 3), dtype=torch.uint8, device="cuda")
    for f in range(frames):
        enc.synth_rgb(t[f].data_ptr(), w, h, seed + f)
    enc.synchronize()
    return t


def with_alpha(rgb, bgr):
    a = torch.randint(0, 256, rgb.shape[:-1] + (1,), dtype=torch.uint8, device=rgb.device)
    return torch.cat([rgb.flip(-1) if bgr else rgb, a], dim=-1).contiguous()


def l1_single_16k(enc, reps, card):
    W = H = 16384
    rgb = synth_device(enc, W, H, 3)[0]
    pitched = torch.randint(0, 256, (H, 3 * W + 64), dtype=torch.uint8, device="cuda")
    pitched[:, : 3 * W] = rgb.reshape(H, 3 * W)
    layouts = {
        "rgb": (rgb, 0, "RGB"),
        "rgb_pitch_3w_plus_64": (pitched, 3 * W + 64, "RGB"),
        "bgr": (rgb.flip(-1).contiguous(), 0, "BGR"),
        "rgba": (with_alpha(rgb, False), 0, "RGBA"),
        "bgra": (with_alpha(rgb, True), 0, "BGRA"),
    }
    torch.cuda.synchronize()
    enc.set_stage_timing(1)
    k1 = {k: [] for k in layouts}

    def variant(name):
        t, pitch, fmt = layouts[name]

        def run():
            enc.bind_device_image(t.data_ptr(), W, H, pitch, fmt)
            enc.encode_bound(None)
            k1[name].append(enc.stats().ms_k1)
        return run
    res = run_variants({k: variant(k) for k in layouts}, reps)
    enc.set_stage_timing(0)
    padded_px = float(W * H)                                              # 16384 is a multiple of 16
    out = {"workload": "L1_16384x16384_single_image", "card": card, "reps": reps}
    files = {}
    cap = W * H * 2
    buf, bptr = pinned_empty(cap)
    try:
        for name, (t, pitch, fmt) in layouts.items():
            enc.bind_device_image(t.data_ptr(), W, H, pitch, fmt)
            n = enc.encode_bound(buf)
            files[name] = buf[:n].tobytes()
    finally:
        pinned_free(bptr)
    for name in layouts:
        ms_k1 = stats(k1[name][1:])                                       # the warm-up encode is not counted
        k1_bytes = padded_px * (PIXEL_FORMATS[layouts[name][2]][1] + 3)
        out[name] = {"encode_ms": res[name], "k1_ms": ms_k1, "k1_bytes_per_px": k1_bytes / padded_px,
                     "k1_gb_per_s": k1_bytes / (ms_k1["median"] * 1e-3) / 1e9, "same_file_as_rgb": files[name] == files["rgb"]}
    del layouts, rgb, pitched
    torch.cuda.empty_cache()
    return out


def l2_frames_1080p(enc, reps, card):
    n, W, H = 1024, 1920, 1080
    rgb = synth_device(enc, W, H, 100, frames=n)
    bgra = with_alpha(rgb, True)
    torch.cuda.synchronize()
    rp = [rgb[f].data_ptr() for f in range(n)]
    bp = [bgra[f].data_ptr() for f in range(n)]
    variants = {
        "rgb_frames_packed": lambda: enc.encode_frames_packed(rp, W, H, None, 0),
        "bgra_images_packed_layout": lambda: enc.encode_images_packed(bp, [W] * n, [H] * n, None, 0, pitches=[0] * n, fmt="BGRA"),
    }
    res = run_variants(variants, reps)
    same = variants["rgb_frames_packed"]()[1] == variants["bgra_images_packed_layout"]()[1]
    out = {"workload": "L2_1024_frames_1920x1080", "card": card, "reps": reps, "file_sizes_equal": same}
    for k, st in res.items():
        out[k] = {"ms": st, "frames_per_s": n / (st["median"] * 1e-3)}
    out["bgra_over_rgb"] = res["bgra_images_packed_layout"]["median"] / res["rgb_frames_packed"]["median"]
    del rgb, bgra
    torch.cuda.empty_cache()
    return out


def l3_tiles(enc, reps, card):
    W = H = 16384
    T = 256
    rgb = synth_device(enc, W, H, 5)[0]
    packed = torch.empty(W * H * 3, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    base, pitch = rgb.data_ptr(), 3 * W
    tiles = [(x, y) for y in range(0, H, T) for x in range(0, W, T)]
    ptrs = [base + y * pitch + 3 * x for x, y in tiles]
    pptrs = [packed.data_ptr() + k * T * T * 3 for k in range(len(tiles))]
    ws, hs = [T] * len(tiles), [T] * len(tiles)
    try:
        cudart = C.CDLL("libcudart.so.12")                               # the runtime torch has loaded
    except OSError:
        cudart = C.CDLL("/usr/local/cuda/lib64/libcudart.so")
    cudart.cudaMemcpy2DAsync.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_void_p]
    _, _, total = enc.encode_images_packed(ptrs, ws, hs, None, 0, pitches=[pitch] * len(tiles), fmt="RGB")
    buf, bptr = pinned_empty(total + 4096)

    def with_pitch():
        return enc.encode_images_packed(ptrs, ws, hs, bptr, buf.size, pitches=[pitch] * len(tiles), fmt="RGB")

    def repack_then_encode():
        for src, dst in zip(ptrs, pptrs):
            rc = cudart.cudaMemcpy2DAsync(dst, T * 3, src, pitch, T * 3, T, 3, None)     # device to device, default stream
            assert rc == 0, rc
        assert cudart.cudaDeviceSynchronize() == 0
        return enc.encode_images_packed(pptrs, ws, hs, bptr, buf.size)
    try:
        res = run_variants({"pointers_with_pitch": with_pitch, "tile_copies_then_images_packed": repack_then_encode}, reps)
        a = with_pitch()
        fa = buf[: a[2]].tobytes()
        b = repack_then_encode()
        same = a == b and buf[: b[2]].tobytes() == fa
    finally:
        pinned_free(bptr)
    out = {"workload": "L3_16384x16384_as_4096_tiles_of_256", "card": card, "reps": reps, "same_files": same}
    for k, st in res.items():
        out[k] = {"ms": st, "gpx_per_s": W * H / (st["median"] * 1e-3) / 1e9}
    out["speedup"] = res["tile_copies_then_images_packed"]["median"] / res["pointers_with_pitch"]["median"]
    del rgb, packed
    torch.cuda.empty_cache()
    return out


def l4_host_rgba(enc, reps, card):
    W = H = 16384
    rgb = synth_device(enc, W, H, 8)[0]
    rgba = with_alpha(rgb, False)
    torch.cuda.synchronize()
    h_rgba, p_rgba = pinned_empty(W * H * 4)
    h_rgb, p_rgb = pinned_empty(W * H * 3)
    out_buf, p_out = pinned_empty(W * H * 2)
    dev = enc.dev_alloc(W * H * 4)
    try:
        enc.d2h(h_rgba, rgba.data_ptr())
        enc.d2h(h_rgb, rgb.data_ptr())
        del rgb, rgba
        torch.cuda.empty_cache()
        n = C.c_uint64()
        files = {}

        def rgba_image():
            enc._check(enc.lib.jpgenc_encode_image(enc.h, p_rgba, W, H, 0, PIXEL_FORMATS["RGBA"][0], 255, p_out, out_buf.size, C.byref(n)))
            files["rgba"] = n.value

        def rgb_encode():
            files["rgb"] = enc.encode_rgb_into(p_rgb, W, H, p_out, out_buf.size)

        variants = {"rgba_encode_image": rgba_image, "rgb_encode_rgb": rgb_encode,
                    "plain_copy_rgba_bytes": lambda: enc.h2d(dev, h_rgba), "plain_copy_rgb_bytes": lambda: enc.h2d(dev, h_rgb)}
        res = run_variants(variants, reps)
        rgba_image()
        fa = out_buf[: files["rgba"]].tobytes()
        rgb_encode()
        same = out_buf[: files["rgb"]].tobytes() == fa
    finally:
        enc.dev_free(dev)
        for p in (p_rgba, p_rgb, p_out):
            pinned_free(p)
    out = {"workload": "L4_16384x16384_pinned_host", "card": card, "reps": reps, "same_files": same}
    for k, st in res.items():
        out[k] = {"ms": st}
    out["rgba_over_rgb"] = res["rgba_encode_image"]["median"] / res["rgb_encode_rgb"]["median"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default=None, help="comma-separated subset of L1,L2,L3,L4")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU only")
    card = gpu_info()
    enc = Encoder(0)
    runs = {"L1": l1_single_16k, "L2": l2_frames_1080p, "L3": l3_tiles, "L4": l4_host_rgba}
    pick = args.only.split(",") if args.only else list(runs)
    results = []
    for k in pick:
        res = runs[k](enc, args.reps, card)
        print(json.dumps(res), flush=True)
        results.append(res)
    enc.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "layout_time.json"), "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
