"""K1 and K2 time and whole-encode time on the 16384^2 synthetic (CUDA events inside the library) -- development aid"""
import sys
sys.path.insert(0, ".")
from jpgenc_b200.capi import Encoder
w = h = 16384
enc = Encoder(0)
enc.set_stage_timing(2)
d = enc.dev_alloc(w * h * 3)
enc.synth_rgb(d, w, h, 0)
enc.bind_device_rgb(d, w, h)
for _ in range(3):
    n = enc.encode_bound(None)
k1, k2, tot = [], [], []
for _ in range(30):
    enc.timer_begin()
    enc.encode_bound(None)
    tot.append(enc.timer_end())
    k1.append(enc.stats().ms_k1); k2.append(enc.stats().ms_stats)
k1.sort(); k2.sort(); tot.sort()
print(f"K1 median {k1[15]:.4f} ms min {k1[0]:.4f}; K2 median {k2[15]:.4f}; whole encode median {tot[15]:.4f} ms; {n} bytes")
