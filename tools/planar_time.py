"""Greyscale and planar RGB pixels against tight RGB, and against the repacking copy a torch user makes without them.  Pixels are
generated on the device from seeds (torch does the layout conversions before timing starts, except where the conversion is what
is timed).

    python tools/planar_time.py [--reps 5] [--out DIR]

Workloads:
  P1  one 16384x16384 image, device-resident: tight RGB, planar RGB (a (3, H, W) tensor) and GRAY bound in place -- whole encode
      (host clock around jpgenc_encode_bound with the scan left on the device) and K1 alone (stage timing level 1), with K1's
      HBM rate over the bytes it must move (3 / 3 / 1 bytes read and 3 bytes of coefficients written per pixel); and the same
      images the way a torch user encodes them without this: permute(1, 2, 0).contiguous() of the (3, H, W) tensor, or the grey
      plane expanded to (H, W, 3) RGB, then tight RGB -- the conversion inside the timed window
  P2  1024 frames of 1920x1080 as (3, H, W) tensors through Encoder.encode_tensors (files returned to the host) and through
      jpgenc_encode_images_packed_planar (sizes only), against tight RGB frames through jpgenc_encode_frames_packed (files into
      pinned memory / sizes only)
  P3  16384x16384 GRAY and planar RGB from pinned host memory, each beside a plain host-to-device copy of the same bytes, and
      tight RGB through jpgenc_encode_rgb (files into pinned memory)
The variants of a workload alternate within every repetition; median, min and max over the repetitions are reported, and the
files of the variants are compared with each other.  Prints one JSON line per workload and writes them to DIR/planar_time.json."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from jpgenc_b200.capi import PIXEL_FORMATS, Encoder, pinned_empty, pinned_free  # noqa: E402
from layout_time import gpu_info, run_variants, stats, synth_device  # noqa: E402


def p1_single_16k(enc, reps, card):
    W = H = 16384
    rgb = synth_device(enc, W, H, 3)[0]
    chw = rgb.permute(2, 0, 1).contiguous()
    grey = rgb[:, :, 1].contiguous()
    torch.cuda.synchronize()
    n = W * H
    binds = {
        "rgb": lambda: enc.bind_device_image(rgb.data_ptr(), W, H, 0, "RGB"),
        "planar": lambda: enc.bind_device_planar(chw.data_ptr(), chw.data_ptr() + n, chw.data_ptr() + 2 * n, W, H),
        "gray": lambda: enc.bind_device_image(grey.data_ptr(), W, H, 0, "GRAY"),
    }
    scratch = {}

    def repacked(make):
        def run():
            scratch["t"] = make()                                         # what the caller has to do without planar / GRAY input
            torch.cuda.synchronize()
            enc.bind_device_image(scratch["t"].data_ptr(), W, H, 0, "RGB")
            enc.encode_bound(None)
        return run
    enc.set_stage_timing(1)
    k1 = {k: [] for k in binds}

    def in_place(name):
        def run():
            binds[name]()
            enc.encode_bound(None)
            k1[name].append(enc.stats().ms_k1)
        return run
    variants = {k: in_place(k) for k in binds}
    variants["planar_repack_permute_contiguous"] = repacked(lambda: chw.permute(1, 2, 0).contiguous())
    variants["gray_repack_expand_to_rgb"] = repacked(lambda: grey[:, :, None].expand(H, W, 3).contiguous())
    res = run_variants(variants, reps)
    enc.set_stage_timing(0)
    scratch.clear()
    files = {}
    buf, bptr = pinned_empty(W * H * 2)
    try:
        for name, bind in binds.items():
            bind()
            files[name] = buf[: enc.encode_bound(buf)].tobytes()
        gt = grey[:, :, None].expand(H, W, 3).contiguous()
        enc.bind_device_image(gt.data_ptr(), W, H, 0, "RGB")
        gray_as_rgb = buf[: enc.encode_bound(buf)].tobytes()
        del gt
    finally:
        pinned_free(bptr)
    out = {"workload": "P1_16384x16384_single_image", "card": card, "reps": reps,
           "planar_same_file_as_rgb": files["planar"] == files["rgb"], "gray_same_file_as_expanded_rgb": files["gray"] == gray_as_rgb}
    read = {"rgb": 3, "planar": 3, "gray": 1}
    for name in binds:
        ms_k1 = stats(k1[name][1:])                                       # the warm-up encode is not counted
        out[name] = {"encode_ms": res[name], "k1_ms": ms_k1, "k1_bytes_per_px": read[name] + 3,
                     "k1_gb_per_s": n * (read[name] + 3) / (ms_k1["median"] * 1e-3) / 1e9}
    for name in ("planar_repack_permute_contiguous", "gray_repack_expand_to_rgb"):
        out[name] = {"encode_ms": res[name]}
    out["planar_saves_over_repack_ms"] = res["planar_repack_permute_contiguous"]["median"] - res["planar"]["median"]
    out["gray_saves_over_repack_ms"] = res["gray_repack_expand_to_rgb"]["median"] - res["gray"]["median"]
    del rgb, chw, grey
    torch.cuda.empty_cache()
    return out


def p2_frames_1080p(enc, reps, card):
    n, W, H = 1024, 1920, 1080
    rgb = synth_device(enc, W, H, 100, frames=n)
    chw = rgb.permute(0, 3, 1, 2).contiguous()
    torch.cuda.synchronize()
    rp = [rgb[f].data_ptr() for f in range(n)]
    planes = [chw[f, k].data_ptr() for f in range(n) for k in range(3)]
    frames = list(chw)
    _, _, total = enc.encode_frames_packed(rp, W, H, None, 0)
    buf, bptr = pinned_empty(total + 4096)
    try:
        variants = {
            "rgb_frames_packed_sizes_only": lambda: enc.encode_frames_packed(rp, W, H, None, 0),
            "planar_images_packed_planar_sizes_only": lambda: enc.encode_images_packed_planar(planes, [W] * n, [H] * n, None, 0),
            "rgb_frames_packed_files_pinned": lambda: enc.encode_frames_packed(rp, W, H, bptr, buf.size),
            "planar_encode_tensors_files": lambda: enc.encode_tensors(frames),
        }
        res = run_variants(variants, reps)
        offs, sizes, _ = enc.encode_frames_packed(rp, W, H, bptr, buf.size)
        want = [buf[o: o + k].tobytes() for o, k in zip(offs, sizes)]
        same = enc.encode_tensors(frames) == want
    finally:
        pinned_free(bptr)
    out = {"workload": "P2_1024_frames_1920x1080_chw_tensors", "card": card, "reps": reps, "same_files": same}
    for k, st in res.items():
        out[k] = {"ms": st, "frames_per_s": n / (st["median"] * 1e-3)}
    del rgb, chw, frames
    torch.cuda.empty_cache()
    return out


def p3_host(enc, reps, card):
    W = H = 16384
    n = W * H
    rgb = synth_device(enc, W, H, 8)[0]
    chw = rgb.permute(2, 0, 1).contiguous()
    torch.cuda.synchronize()
    h_chw, p_chw = pinned_empty(3 * n)
    h_rgb, p_rgb = pinned_empty(3 * n)
    out_buf, p_out = pinned_empty(n * 2)
    dev = enc.dev_alloc(3 * n)
    try:
        enc.d2h(h_chw, chw.data_ptr())
        enc.d2h(h_rgb, rgb.data_ptr())
        del rgb, chw
        torch.cuda.empty_cache()
        size = C.c_uint64()
        files = {}

        def gray_image():                                                 # the G plane of the (3, H, W) buffer as a grey image
            enc._check(enc.lib.jpgenc_encode_image(enc.h, p_chw + n, W, H, 0, PIXEL_FORMATS["GRAY"][0], 255, p_out, out_buf.size, C.byref(size)))
            files["gray"] = size.value

        def planar_image():
            enc._check(enc.lib.jpgenc_encode_planar(enc.h, p_chw, p_chw + n, p_chw + 2 * n, W, H, 0, 255, p_out, out_buf.size, C.byref(size)))
            files["planar"] = size.value

        def rgb_encode():
            files["rgb"] = enc.encode_rgb_into(p_rgb, W, H, p_out, out_buf.size)

        variants = {"gray_encode_image": gray_image, "plain_copy_gray_bytes": lambda: enc.h2d(dev, h_chw[n: 2 * n]),
                    "planar_encode_planar": planar_image, "plain_copy_planar_bytes": lambda: enc.h2d(dev, h_chw),
                    "rgb_encode_rgb": rgb_encode}
        res = run_variants(variants, reps)
        planar_image()
        fa = out_buf[: files["planar"]].tobytes()
        rgb_encode()
        same = out_buf[: files["rgb"]].tobytes() == fa
    finally:
        enc.dev_free(dev)
        for p in (p_chw, p_rgb, p_out):
            pinned_free(p)
    out = {"workload": "P3_16384x16384_pinned_host", "card": card, "reps": reps, "planar_same_file_as_rgb": same}
    for k, st in res.items():
        out[k] = {"ms": st}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default=None, help="comma-separated subset of P1,P2,P3")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU only")
    card = gpu_info()
    enc = Encoder(0)
    runs = {"P1": p1_single_16k, "P2": p2_frames_1080p, "P3": p3_host}
    pick = args.only.split(",") if args.only else list(runs)
    results = []
    for k in pick:
        res = runs[k](enc, args.reps, card)
        print(json.dumps(res), flush=True)
        results.append(res)
    enc.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "planar_time.json"), "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
