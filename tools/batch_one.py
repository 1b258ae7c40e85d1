"""one batched call over 256 frames of 1920x1080 in passes of 128, single lane (for ncu launch lists) -- development aid"""
import os, sys
os.environ["JPGENC_SLOTS"] = "1"; os.environ["JPGENC_FRAMES_PER_PASS"] = "128"
sys.path.insert(0, ".")
from jpgenc_b200.capi import Encoder
w, h, nf = 1920, 1080, 256
fb = w * h * 3
enc = Encoder(0)
d = enc.dev_alloc(nf * fb)
for k in range(nf):
    enc.synth_rgb(d + k * fb, w, h, k)
enc.synchronize()
ptrs = [d + k * fb for k in range(nf)]
enc.encode_frames_device(ptrs, w, h)
enc.encode_frames_device(ptrs, w, h)
