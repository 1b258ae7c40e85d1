"""YUV frames (4:2:0: I420, NV12; 4:2:2: I422, NV16, YUYV; 4:4:4: I444) against tight RGB of the same content.  The RGB frames are
generated on the device from seeds; their YUV (full-range BT.601, 4:2:0 chroma of the top-left pixel of every 2x2 cell, 4:2:2 of
the left pixel of every pair) is computed by torch before timing starts.  UYVY moves the same bytes as YUYV and is not timed.

    python tools/yuv_time.py [--reps 5] [--out DIR]

Workloads:
  Y1  one 16384x16384 frame, device-resident, in every timed layout and as tight RGB: the whole encode (host clock around
      jpgenc_encode_bound with the scan left on the device, stage timing off) with L2 flushed before every timed encode; then,
      in rounds of their own, K1 alone (stage timing level 1) with its HBM rate over the bytes it must move (1.5 bytes read per
      pixel for 4:2:0, 2 for 4:2:2, 3 for 4:4:4 and RGB, and 3 bytes of coefficients written)
  Y2  1024 frames of 1920x1080, device-resident: NV12, I422 and YUYV through jpgenc_encode_images_packed_yuv(420) against RGB
      through jpgenc_encode_images_packed_layout (the same pass pipeline of images of individual sizes, so only the input differs)
      and through jpgenc_encode_images_packed (one size: the batched-frame path), sizes only and files into pinned memory
  Y3  one 16384x16384 frame from pinned host memory, NV12, YUYV and I444 through jpgenc_encode_yuv against RGB through
      jpgenc_encode_rgb, all writing the file into the same pinned buffer
The variants of a workload alternate within every repetition; median, min and max over the repetitions are reported.  Prints the
card (name, power limit, max SM clock) and one JSON line per workload, and writes them to DIR/yuv_time.json."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from jpgenc_b200.capi import YUV_FORMATS, Encoder, pinned_empty, pinned_free  # noqa: E402
from layout_time import gpu_info, run_variants, stats, synth_device  # noqa: E402


def yuv_planes(rgb):
    """(H, W, 3) uint8 CUDA tensor -> Y (H, W), U, V (ceil(H/2), ceil(W/2)) uint8 tensors"""
    f = rgb.float()
    y = 0.299 * f[..., 0] + 0.587 * f[..., 1] + 0.114 * f[..., 2]
    q = lambda p: p.round().clamp(0, 255).to(torch.uint8).contiguous()
    u = q(128 + 0.564 * (f[::2, ::2, 2] - y[::2, ::2]))
    v = q(128 + 0.713 * (f[::2, ::2, 0] - y[::2, ::2]))
    return q(y), u, v


def yuv_full(rgb):
    """(H, W, 3) uint8 CUDA tensor -> Y, U, V (H, W) uint8 tensors (4:4:4; [:, ::2] of U and V is 4:2:2)"""
    f = rgb.float()
    y = 0.299 * f[..., 0] + 0.587 * f[..., 1] + 0.114 * f[..., 2]
    q = lambda p: p.round().clamp(0, 255).to(torch.uint8).contiguous()
    return q(y), q(128 + 0.564 * (f[..., 2] - y)), q(128 + 0.713 * (f[..., 0] - y))


def yuyv(y, u2, v2):
    """one (H, 2 W) YUYV plane (W even) of Y and 4:2:2 chroma"""
    return torch.stack([y[:, 0::2], u2, y[:, 1::2], v2], dim=2).reshape(y.shape[0], -1).contiguous()


def nv12(y, u, v):
    """one (H + ch, W) NV12 surface (W even): Y rows, then the interleaved UV rows"""
    h, w = y.shape
    s = torch.empty((h + u.shape[0], w), dtype=torch.uint8, device=y.device)
    s[:h] = y
    s[h:].view(u.shape[0], -1, 2)[..., 0] = u
    s[h:].view(u.shape[0], -1, 2)[..., 1] = v
    return s


def y1_single_16k(enc, reps, card):
    W = H = 16384
    rgb = synth_device(enc, W, H, 3)[0]
    y, u, v = yuv_planes(rgb)
    s = nv12(y, u, v)
    torch.cuda.synchronize()
    y4, u4, v4 = yuv_full(rgb)
    u2, v2 = u4[:, ::2].contiguous(), v4[:, ::2].contiguous()
    nv16 = torch.stack([u2, v2], dim=2).reshape(H, -1).contiguous()
    yuy = yuyv(y4, u2, v2)
    binds = {
        "nv12": lambda: enc.bind_device_yuv420(s.data_ptr(), s[H:].data_ptr(), None, W, H, 0, 0, "NV12"),
        "i420": lambda: enc.bind_device_yuv420(y.data_ptr(), u.data_ptr(), v.data_ptr(), W, H, 0, 0, "I420"),
        "i422": lambda: enc.bind_device_yuv("I422", y4.data_ptr(), u2.data_ptr(), v2.data_ptr(), W, H),
        "nv16": lambda: enc.bind_device_yuv("NV16", y4.data_ptr(), nv16.data_ptr(), None, W, H),
        "yuyv": lambda: enc.bind_device_yuv("YUYV", yuy.data_ptr(), None, None, W, H),
        "i444": lambda: enc.bind_device_yuv("I444", y4.data_ptr(), u4.data_ptr(), v4.data_ptr(), W, H),
        "rgb": lambda: enc.bind_device_image(rgb.data_ptr(), W, H, 0, "RGB"),
    }
    k1 = {k: [] for k in binds}
    enc_ms = {k: [] for k in binds}
    for rep in range(reps + 1):                                           # the first round warms every path and is not counted
        for name, bind in binds.items():
            enc.flush_l2()
            enc.synchronize()
            t0 = time.perf_counter()
            bind()
            enc.encode_bound(None)
            if rep:
                enc_ms[name].append((time.perf_counter() - t0) * 1e3)
    enc.set_stage_timing(1)                                               # K1's events, in rounds of their own
    for rep in range(reps + 1):
        for name, bind in binds.items():
            enc.flush_l2()
            bind()
            enc.encode_bound(None)
            if rep:
                k1[name].append(enc.stats().ms_k1)
    enc.set_stage_timing(0)
    files = {}
    buf, bptr = pinned_empty(W * H * 2)
    try:
        for name, bind in binds.items():
            bind()
            files[name] = buf[: enc.encode_bound(buf)].tobytes()
    finally:
        pinned_free(bptr)
    n = W * H
    read = {"nv12": 1.5, "i420": 1.5, "i422": 2, "nv16": 2, "yuyv": 2, "i444": 3, "rgb": 3}
    out = {"workload": "Y1_16384x16384_single_frame_device", "card": card, "reps": reps,
           "nv12_same_file_as_i420": files["nv12"] == files["i420"],
           "i422_nv16_yuyv_same_file": files["i422"] == files["nv16"] == files["yuyv"]}
    for name in binds:
        ms_k1 = stats(k1[name])
        out[name] = {"encode_ms_l2_flushed": stats(enc_ms[name]), "k1_ms": ms_k1, "k1_bytes_per_px": read[name] + 3,
                     "k1_gb_per_s": n * (read[name] + 3) / (ms_k1["median"] * 1e-3) / 1e9}
    del rgb, y, u, v, s, y4, u4, v4, u2, v2, nv16, yuy
    torch.cuda.empty_cache()
    return out


def y2_frames_1080p(enc, reps, card):
    n, W, H = 1024, 1920, 1080
    rgb = synth_device(enc, W, H, 100, frames=n)
    surf = torch.stack([nv12(*yuv_planes(rgb[f])) for f in range(n)])
    full = [yuv_full(rgb[f]) for f in range(n)]
    i422 = [(y, u[:, ::2].contiguous(), v[:, ::2].contiguous()) for y, u, v in full]
    del full
    packed = [yuyv(*f) for f in i422]
    torch.cuda.synchronize()
    rp = [rgb[f].data_ptr() for f in range(n)]
    planes = [p for f in range(n) for p in (surf[f].data_ptr(), surf[f, H:].data_ptr(), None)]
    planes422 = [p.data_ptr() for f in i422 for p in f]
    planes_yuyv = [p for f in packed for p in (f.data_ptr(), None, None)]
    ws, hs = [W] * n, [H] * n
    _, _, total_rgb = enc.encode_images_packed(rp, ws, hs, None, 0)
    # RGB through the pass pipeline of images of individual sizes, the one the YUV call takes (the layout call with tight RGB
    # would forward to jpgenc_encode_images_packed: a pitch 16 bytes past the row keeps it on the pass pipeline)
    rp_pad = torch.zeros((n, H, 3 * W + 16), dtype=torch.uint8, device="cuda")
    rp_pad[:, :, : 3 * W] = rgb.view(n, H, 3 * W)
    rpp = [rp_pad[f].data_ptr() for f in range(n)]
    pitches = [3 * W + 16] * n
    _, _, total_rgb_pass = enc.encode_images_packed(rpp, ws, hs, None, 0, pitches=pitches, fmt="RGB")
    _, _, total_yuv = enc.encode_images_packed_yuv420(planes, ws, hs, None, 0, "NV12")
    _, _, total_422 = enc.encode_images_packed_yuv(planes422, ws, hs, None, 0, "I422")
    buf, bptr = pinned_empty(max(total_rgb, total_yuv, total_rgb_pass, total_422) + 4096)
    try:
        variants = {
            "nv12_images_packed_yuv420_sizes_only": lambda: enc.encode_images_packed_yuv420(planes, ws, hs, None, 0, "NV12"),
            "i422_images_packed_yuv_sizes_only": lambda: enc.encode_images_packed_yuv(planes422, ws, hs, None, 0, "I422"),
            "yuyv_images_packed_yuv_sizes_only": lambda: enc.encode_images_packed_yuv(planes_yuyv, ws, hs, None, 0, "YUYV"),
            "rgb_images_packed_layout_pass_pipeline_sizes_only": lambda: enc.encode_images_packed(rpp, ws, hs, None, 0, pitches=pitches, fmt="RGB"),
            "rgb_images_packed_frame_path_sizes_only": lambda: enc.encode_images_packed(rp, ws, hs, None, 0),
            "nv12_images_packed_yuv420_files_pinned": lambda: enc.encode_images_packed_yuv420(planes, ws, hs, bptr, buf.size, "NV12"),
            "i422_images_packed_yuv_files_pinned": lambda: enc.encode_images_packed_yuv(planes422, ws, hs, bptr, buf.size, "I422"),
            "yuyv_images_packed_yuv_files_pinned": lambda: enc.encode_images_packed_yuv(planes_yuyv, ws, hs, bptr, buf.size, "YUYV"),
            "rgb_images_packed_layout_pass_pipeline_files_pinned": lambda: enc.encode_images_packed(rpp, ws, hs, bptr, buf.size, pitches=pitches,
                                                                                                     fmt="RGB"),
            "rgb_images_packed_frame_path_files_pinned": lambda: enc.encode_images_packed(rp, ws, hs, bptr, buf.size),
        }
        res = run_variants(variants, reps)
    finally:
        pinned_free(bptr)
    out = {"workload": "Y2_1024_frames_1920x1080_device", "card": card, "reps": reps, "total_bytes_nv12": total_yuv, "total_bytes_rgb": total_rgb,
           "total_bytes_rgb_pass_pipeline": total_rgb_pass, "total_bytes_i422": total_422}
    for k, st in res.items():
        out[k] = {"ms": st, "frames_per_s": n / (st["median"] * 1e-3)}
    del rgb, surf, rp_pad, i422, packed
    torch.cuda.empty_cache()
    return out


def y3_host(enc, reps, card):
    W = H = 16384
    n = W * H
    rgb = synth_device(enc, W, H, 8)[0]
    s = nv12(*yuv_planes(rgb))
    y4, u4, v4 = yuv_full(rgb)
    yuy = yuyv(y4, u4[:, ::2].contiguous(), v4[:, ::2].contiguous())
    i444 = torch.stack([y4, u4, v4])
    torch.cuda.synchronize()
    h_nv12, p_nv12 = pinned_empty(s.numel())
    h_yuyv, p_yuyv = pinned_empty(yuy.numel())
    h_444, p_444 = pinned_empty(i444.numel())
    h_rgb, p_rgb = pinned_empty(3 * n)
    out_buf, p_out = pinned_empty(n * 2)
    try:
        for h_buf, t in ((h_nv12, s), (h_yuyv, yuy), (h_444, i444), (h_rgb, rgb)):
            enc.d2h(h_buf, t.data_ptr())
        del rgb, s, y4, u4, v4, yuy, i444
        torch.cuda.empty_cache()
        size = C.c_uint64()

        def yuv_encode(layout, y, u, v):                                  # into the pinned output, as encode_rgb_into does
            enc._check(enc.lib.jpgenc_encode_yuv(enc.h, y, u, v, W, H, 0, 0, YUV_FORMATS[layout], p_out, out_buf.size, C.byref(size)))
        variants = {"nv12_encode_yuv": lambda: yuv_encode("NV12", p_nv12, p_nv12 + n, None),
                    "yuyv_encode_yuv": lambda: yuv_encode("YUYV", p_yuyv, None, None),
                    "i444_encode_yuv": lambda: yuv_encode("I444", p_444, p_444 + n, p_444 + 2 * n),
                    "rgb_encode_rgb": lambda: enc.encode_rgb_into(p_rgb, W, H, p_out, out_buf.size)}
        res = run_variants(variants, reps)
    finally:
        for p in (p_nv12, p_yuyv, p_444, p_rgb, p_out):
            pinned_free(p)
    out = {"workload": "Y3_16384x16384_pinned_host", "card": card, "reps": reps, "pcie_bytes_nv12": int(1.5 * n), "pcie_bytes_yuyv": 2 * n,
           "pcie_bytes_i444": 3 * n, "pcie_bytes_rgb": 3 * n}
    for k, st in res.items():
        out[k] = {"ms": st}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default=None, help="comma-separated subset of Y1,Y2,Y3")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU only")
    card = gpu_info()
    print(json.dumps({"card": card}), flush=True)
    enc = Encoder(0)
    runs = {"Y1": y1_single_16k, "Y2": y2_frames_1080p, "Y3": y3_host}
    pick = args.only.split(",") if args.only else list(runs)
    results = []
    for k in pick:
        res = runs[k](enc, args.reps, card)
        print(json.dumps(res), flush=True)
        results.append(res)
    enc.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "yuv_time.json"), "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
