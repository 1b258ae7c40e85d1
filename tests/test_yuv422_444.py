"""YUV 4:2:2 and 4:4:4 frames (I422, NV16, YUYV, UYVY, I444) read in place: jpgenc_bind_device_yuv, jpgenc_encode_yuv,
jpgenc_encode_images_packed_yuv and Encoder.encode_yuv / encode_yuv_many.  The file of a frame is defined as Image::writeJPEG of the
YCbCr image whose level-shifted planes are the samples minus 128 at full resolution (a 4:2:2 chroma sample at both pixels of its
group), padded to whole MCUs by edge replication (expected_planes): the reference's 4:2:0 file, whose chroma is the S420_m mean of
every 2x2 cell.  Every file must be byte-identical to the oracle's (or the GPU's FP64 path's) file of those planes.  The bytes
between rows and around the planes are random, so reading any of them would change the file."""
import os
import subprocess
import sys

import numpy as np
import pytest

from jpgenc_b200.capi import YUV_FORMATS, yuv_layout
from jpgenc_b200.synth import synth_rgb

LAYOUTS = ["I422", "NV16", "YUYV", "UYVY", "I444"]
SIZES = [(1, 1), (17, 9), (3, 30), (208, 120), (1000, 667), (1920, 1080)]


def hsub(layout):
    return 0 if layout == "I444" else 1


def yuv_of(rgb, hs):
    """full-range BT.601 Y, Cb, Cr of an RGB image; 4:2:2 (hs 1): chroma of the left pixel of every pair"""
    f = rgb.astype(np.float64)
    r, g, b = f[:, :, 0], f[:, :, 1], f[:, :, 2]
    y = 0.299 * r + 0.587 * g + 0.114 * b
    q = lambda p: np.clip(np.rint(p), 0, 255).astype(np.uint8)
    return q(y), q(128 + 0.564 * (b - y))[:, :: 1 << hs], q(128 + 0.713 * (r - y))[:, :: 1 << hs]


def noise_yuv(w, h, hs, seed):
    """random planes that reach 0 and 255"""
    rng = np.random.default_rng(seed)
    y = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
    u = rng.integers(0, 256, size=(h, (w + hs) >> hs), dtype=np.uint8)
    v = rng.integers(0, 256, size=u.shape, dtype=np.uint8)
    y.flat[0], u.flat[0], v.flat[-1] = 0, 255, 0
    y.flat[-1], v.flat[0] = 255, 255
    return y, u, v


def expected_planes(y, u, v):
    """the level-shifted (H16, W16) planes Y', Cb', Cr' that define a frame's file (u, v: (H, ceil(W/2)) or (H, W))"""
    h, w = y.shape
    h16, w16 = (h + 15) // 16 * 16, (w + 15) // 16 * 16
    up = lambda c: (c if c.shape[1] == w else np.repeat(c, 2, axis=1))[:, :w]
    pad = lambda p: np.pad(p.astype(np.float64) - 128.0, ((0, h16 - h), (0, w16 - w)), mode="edge")
    return pad(y), pad(up(u)), pad(up(v))


def oracle_file(oracle, y, u, v):
    h, w = y.shape
    return oracle.encode_planes(*expected_planes(y, u, v), w, h, ycbcr=True)


def interleave(*planes, fill_seed=None):
    """(H, n) planes -> (H, k n) rows of their samples in turn; a plane of None gets random bytes"""
    shape = next(p.shape for p in planes if p is not None)
    out = np.empty((shape[0], shape[1] * len(planes)), np.uint8)
    rng = np.random.default_rng(fill_seed)
    for k, p in enumerate(planes):
        out[:, k:: len(planes)] = p if p is not None else rng.integers(0, 256, size=shape, dtype=np.uint8)
    return out


def packed_of(layout, y, u, v):
    """the (H, 4 cw) packed plane of a 4:2:2 frame; odd widths: the last group's second Y is random"""
    h, w = y.shape
    cw = u.shape[1]
    yy = np.random.default_rng(5).integers(0, 256, size=(h, 2 * cw), dtype=np.uint8)
    yy[:, :w] = y
    y0, y1 = yy[:, 0::2], yy[:, 1::2]
    return interleave(y0, u, y1, v) if layout == "YUYV" else interleave(u, y0, v, y1)


def layout_planes(layout, y, u, v):
    """the planes the caller passes, in order (y, u, v; absent ones left out)"""
    if layout in ("I422", "I444"):
        return [y, u, v]
    if layout == "NV16":
        return [y, interleave(u, v)]
    return [packed_of(layout, y, u, v)]


def pitch_kinds(row):
    """tight; a multiple of 16 above the row (bulk copies where the width allows it); tight + 3 (clamped loads)"""
    return {"tight": row, "pitch16": (row + 15) // 16 * 16 + 16, "pitch+3": row + 3}


def plane_bytes(plane, pitch, seed, offset=0):
    """plane (H, W) -> (buffer, view): offset + H * pitch random bytes holding the plane's rows `pitch` bytes apart from `offset` on"""
    h, w = plane.shape
    buf = np.random.default_rng(seed).integers(0, 256, size=offset + h * pitch, dtype=np.uint8)
    view = np.lib.stride_tricks.as_strided(buf[offset:], shape=(h, w), strides=(pitch, 1))
    view[:] = plane
    return buf, view


def _encode_bound(enc, cap):
    out = np.empty(cap, np.uint8)
    return out[: enc.encode_bound(out)].tobytes()


class DeviceFrame:
    """a frame's planes in device memory, each in an allocation of its own laid out by plane_bytes; .ptr = (y, u, v) with None
    where the layout has no such plane"""

    def __init__(self, enc, layout, y, u, v, kind, offset, seed):
        self.enc, self.d = enc, []
        planes = layout_planes(layout, y, u, v)
        self.y_pitch = pitch_kinds(planes[0].shape[1])[kind]
        self.c_pitch = pitch_kinds(planes[1].shape[1])[kind] if len(planes) > 1 else 0
        ptr = []
        for k, p in enumerate(planes):
            buf, _ = plane_bytes(p, self.y_pitch if k == 0 else self.c_pitch, seed + k, offset)
            d = enc.dev_alloc(buf.nbytes + 16)
            enc.h2d(d, buf)
            self.d.append(d)
            ptr.append(d + offset)
        self.ptr = tuple(ptr) + (None,) * (3 - len(ptr))

    def free(self):
        for d in self.d:
            self.enc.dev_free(d)


@pytest.fixture(scope="module")
def frames(oracle):
    """per chroma subsampling (hs) and size: a frame derived from synth_rgb and a noise frame, with the oracle's files"""
    out = {}
    for hs in (0, 1):
        out[hs] = []
        for k, (w, h) in enumerate(SIZES):
            for f in (yuv_of(synth_rgb(w, h, 41 + k), hs), noise_yuv(w, h, hs, 7 + k)):
                out[hs].append((f, oracle_file(oracle, *f)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_single_device_frames(encoder, frames, layout):
    for kind in ("tight", "pitch16", "pitch+3"):
        for offset in (0, 1):
            refined = 0
            for k, ((y, u, v), want) in enumerate(frames[hsub(layout)]):
                h, w = y.shape
                f = DeviceFrame(encoder, layout, y, u, v, kind, offset, seed=3 * k)
                try:
                    encoder.bind_device_yuv(layout, *f.ptr, w, h, f.y_pitch, f.c_pitch)
                    got = _encode_bound(encoder, len(want) + 4096)
                    refined += encoder.stats().refined_blocks
                finally:
                    f.free()
                assert got == want, f"{layout} {w}x{h} ({kind}) offset {offset}"
            assert refined > 0, "no block took the FP64 refinement: its sample gather was not exercised"


@pytest.mark.gpu
def test_fp32_bound_at_scale(encoder):
    """4096 x 4096 noise and synthetic frames: the FP32 path with its exact-input thresholds (plus refinement) equals the GPU's
    independent FP64 path on the defining planes"""
    w = h = 4096
    for hs in (1, 0):
        for y, u, v in (noise_yuv(w, h, hs, 99), yuv_of(synth_rgb(w, h, 5), hs)):
            want = encoder.encode_planes(*expected_planes(y, u, v), w, h, ycbcr=True)
            for layout in (lay for lay in LAYOUTS if hsub(lay) == hs):
                f = DeviceFrame(encoder, layout, y, u, v, "tight", 0, seed=1)
                try:
                    encoder.bind_device_yuv(layout, *f.ptr, w, h, 0, 0)
                    got = _encode_bound(encoder, len(want) + 4096)
                finally:
                    f.free()
                assert got == want, f"{layout} 4096x4096"


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_host_frames_in_several_bands(encoder, layout):
    """4000 x 3000 host frames (several upload bands), tight and pitched: each equals the device path's file"""
    w, h = 4000, 3000
    y, u, v = yuv_of(synth_rgb(w, h, 17), hsub(layout))
    f = DeviceFrame(encoder, layout, y, u, v, "tight", 0, seed=2)
    try:
        encoder.bind_device_yuv(layout, *f.ptr, w, h, 0, 0)
        want = _encode_bound(encoder, w * h)
    finally:
        f.free()
    planes = layout_planes(layout, y, u, v)
    for kind in ("tight", "pitch+3"):
        views = [plane_bytes(p, pitch_kinds(p.shape[1])[kind], 3 + k)[1] for k, p in enumerate(planes)]
        assert encoder.encode_yuv(layout, *views) == want, f"host {layout} ({kind})"


def _tiles(W, H, T):
    return [(x, y, min(T, W - x), min(T, H - y)) for y in range(0, H, T) for x in range(0, W, T)]


class BigFrame:
    """a W x H frame (odd sides: ragged odd-sized edge tiles) with pitched planes in one buffer in device or pinned host memory,
    cut into T x T tiles (T even): plane pointers into it, and the oracle's file of every tile"""

    def __init__(self, enc, oracle, layout, W=1501, H=1099, T=256, host=False, tiles=None):
        from jpgenc_b200.capi import pinned_empty
        self.enc, self.host, self.layout = enc, host, layout
        hs = hsub(layout)
        y, u, v = yuv_of(synth_rgb(W, H, 23), hs)
        planes = layout_planes(layout, y, u, v)
        self.y_pitch = planes[0].shape[1] + 5
        self.c_pitch = planes[1].shape[1] + 3 if len(planes) > 1 else 0
        at = [0]
        for p in planes[1:]:
            at.append(at[-1] + p.shape[0] * (self.y_pitch if len(at) == 1 else self.c_pitch) + 16)
        end = at[-1] + H * (self.c_pitch or self.y_pitch) + 16
        buf = np.random.default_rng(9).integers(0, 256, size=end, dtype=np.uint8)
        for k, (a, p) in enumerate(zip(at, planes)):
            np.lib.stride_tricks.as_strided(buf[a:], shape=p.shape, strides=(self.y_pitch if k == 0 else self.c_pitch, 1))[:] = p
        if host:
            self.view, self.base = pinned_empty(buf.nbytes)
            self.view[:] = buf
        else:
            self.base = enc.dev_alloc(buf.nbytes)
            enc.h2d(self.base, buf)
        tl = _tiles(W, H, T)[:tiles]
        ybytes = 2 if layout in ("YUYV", "UYVY") else 1                    # bytes per pixel of the first plane
        cbytes = 2 if layout == "NV16" else 1                              # bytes per chroma sample of a chroma plane
        self.ptrs = []
        for x, yy, _, _ in tl:
            self.ptrs.append(self.base + yy * self.y_pitch + x * ybytes)
            for a in at[1:]:
                self.ptrs.append(self.base + a + yy * self.c_pitch + (x >> hs) * cbytes)
            self.ptrs += [None] * (3 - len(at))
        self.ws = [w for _, _, w, _ in tl]
        self.hs = [h for _, _, _, h in tl]
        self.want = [oracle_file(oracle, y[yy: yy + h, x: x + w], u[yy: yy + h, x >> hs: (x + w + hs) >> hs],
                                 v[yy: yy + h, x >> hs: (x + w + hs) >> hs]) for x, yy, w, h in tl]

    def free(self):
        from jpgenc_b200.capi import pinned_free
        if self.host:
            pinned_free(self.base)
        else:
            self.enc.dev_free(self.base)


def _check_packed(enc, big):
    """contiguous files in input order, each the oracle's; sizes-only equals the real call; one byte short is refused"""
    from jpgenc_b200.capi import ERR_CAPACITY, JpgencError, pinned_empty, pinned_free
    n = len(big.ws)

    def call(o, c):
        return enc.encode_images_packed_yuv(big.ptrs, big.ws, big.hs, o, c, big.layout, host_images=big.host,
                                            y_pitches=[big.y_pitch] * n, c_pitches=[big.c_pitch] * n)

    offs0, sizes0, total = call(None, 0)
    buf, bptr = pinned_empty(total + 64)
    try:
        offs, sizes, total2 = call(bptr, total)
        assert (offs, sizes, total2) == (offs0, sizes0, total)
        assert offs[0] == 0 and all(offs[i] + sizes[i] == offs[i + 1] for i in range(n - 1)) and offs[-1] + sizes[-1] == total
        for i in range(n):
            assert bytes(buf[offs[i]: offs[i] + sizes[i]]) == big.want[i], f"tile {i} ({big.ws[i]}x{big.hs[i]})"
        with pytest.raises(JpgencError) as e:
            call(bptr, total - 1)
        assert e.value.code == ERR_CAPACITY
    finally:
        pinned_free(bptr)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("host", [False, True])
def test_tiles_of_one_frame(encoder, oracle, layout, host):
    big = BigFrame(encoder, oracle, layout, host=host)
    try:
        _check_packed(encoder, big)
    finally:
        big.free()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("host", [False, True])
def test_many_passes_and_refused_passes(oracle, monkeypatch, layout, host):
    """tiles cut into many passes over several slots; JPGENC_RAW_GUESS_PER_BLOCK=0 makes every first pass too small, so each is
    refused on the device and re-run"""
    from jpgenc_b200.capi import Encoder
    monkeypatch.setenv("JPGENC_FRAMES_PER_PASS", "5")
    monkeypatch.setenv("JPGENC_SLOTS", "3")
    for guess in (None, "0"):
        if guess is not None:
            monkeypatch.setenv("JPGENC_RAW_GUESS_PER_BLOCK", guess)
        enc = Encoder(0)                                  # a fresh context: nothing learnt about scan sizes yet
        big = BigFrame(enc, oracle, layout, W=901, H=777, T=128, host=host, tiles=23)
        try:
            _check_packed(enc, big)
        finally:
            big.free()
            enc.close()


def _graph_cycle():
    """one device buffer bound in all seven layouts with the same first pointer and size, each twice in a row; then I422 with the
    same planes and only a wider chroma pitch"""
    from jpgenc_b200.capi import Encoder
    from oracle.pyoracle import Oracle
    oracle = Oracle()
    enc = Encoder(0)
    w, h = 334, 201
    cw = w // 2
    buf = np.random.default_rng(3).integers(0, 256, size=3 * w * h, dtype=np.uint8)
    d = enc.dev_alloc(buf.nbytes)
    try:
        enc.h2d(d, buf)
        y = buf[: w * h].reshape(h, w)
        at = lambda o, rows, row, pitch=None: np.lib.stride_tricks.as_strided(buf[o:], shape=(rows, row), strides=(pitch or row, 1))
        c0, ch = w * h, (h + 1) // 2
        p = buf[: 4 * cw * h].reshape(h, 4 * cw)
        cp = cw + 3
        binds = {
            "I420": (("I420", d, d + c0, d + c0 + cw * ch, 0), (y, at(c0, ch, cw), at(c0 + cw * ch, ch, cw))),
            "NV12": (("NV12", d, d + c0, None, 0), (y, at(c0, ch, 2 * cw)[:, 0::2], at(c0, ch, 2 * cw)[:, 1::2])),
            "I422": (("I422", d, d + c0, d + c0 + cw * h, 0), (y, at(c0, h, cw), at(c0 + cw * h, h, cw))),
            "I422_pitched": (("I422", d, d + c0, d + c0 + cw * h, cp), (y, at(c0, h, cw, cp), at(c0 + cw * h, h, cw, cp))),
            "NV16": (("NV16", d, d + c0, None, 0), (y, at(c0, h, 2 * cw)[:, 0::2], at(c0, h, 2 * cw)[:, 1::2])),
            "I444": (("I444", d, d + c0, d + 2 * c0, 0), (y, at(c0, h, w), at(2 * c0, h, w))),
            "YUYV": (("YUYV", d, None, None, 0), (interleave(p[:, 0::4], p[:, 2::4]), p[:, 1::4], p[:, 3::4])),
            "UYVY": (("UYVY", d, None, None, 0), (interleave(p[:, 1::4], p[:, 3::4]), p[:, 0::4], p[:, 2::4])),
        }
        want = {}
        for k, (_, planes) in binds.items():
            if k in ("I420", "NV12"):
                yy, uu, vv = planes
                up = lambda c: np.repeat(c, 2, axis=0)[:h]
                want[k] = oracle_file(oracle, yy, up(uu), up(vv))
            else:
                want[k] = oracle_file(oracle, *planes)
        for _ in range(2):
            for kind, ((lay, yp, up_, vp, c_pitch), _) in binds.items():
                for _ in range(2):
                    enc.bind_device_yuv(lay, yp, up_, vp, w, h, 0, c_pitch)
                    assert _encode_bound(enc, 1 << 20) == want[kind], kind
    finally:
        enc.dev_free(d)
        enc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("graphs", ["1", "0"])
def test_graph_cache_keys_on_all_yuv_layouts(graphs):
    # JPGENC_GRAPHS is read once per process: each setting runs in a process of its own
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, JPGENC_GRAPHS=graphs,
               PYTHONPATH=os.pathsep.join([root, os.path.dirname(os.path.abspath(__file__))]))
    r = subprocess.run([sys.executable, "-c", "import test_yuv422_444 as t; t._graph_cycle()"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_argument_errors(encoder):
    from jpgenc_b200.capi import ERR_ARG, OK
    import ctypes as C
    lib, h = encoder.lib, encoder.h
    d = encoder.dev_alloc(1 << 18)
    w, hh = 64, 32
    u, v = d + w * hh, d + 2 * w * hh
    u32 = C.POINTER(C.c_uint32)
    out = np.empty(1 << 16, np.uint8)
    n = C.c_uint64()

    def packed_call(fn, a):
        pl = (C.c_void_p * 3)(*a[:3])
        ws, hs = np.array([a[3]], np.uint32), np.array([a[4]], np.uint32)
        yp, cp = np.array([a[5]], np.uint32), np.array([a[6]], np.uint32)
        offs, sizes, total = (C.c_uint64 * 1)(), (C.c_uint64 * 1)(), C.c_uint64()
        return fn(h, 1, pl, 1, ws.ctypes.data_as(u32), hs.ctypes.data_as(u32), yp.ctypes.data_as(u32), cp.ctypes.data_as(u32), a[7], None, 0,
                  offs, sizes, C.byref(total))

    try:
        bad = [(d, u, v, w, hh, 0, 0, 7), (d, u, v, w, hh, 0, 0, -1),               # unknown layout
               (None, u, v, w, hh, 0, 0, 2), (d, None, v, w, hh, 0, 0, 2),          # I422: null Y, null U
               (d, u, None, w, hh, 0, 0, 2), (d, u, None, w, hh, 0, 0, 4),          # null V (I422, I444)
               (d, None, None, w, hh, 0, 0, 3), (d, u, v, w, hh, 0, 0, 3),          # NV16: null UV, a V
               (d, u, None, w, hh, 0, 0, 5), (d, None, v, w, hh, 0, 0, 6),          # packed: a U, a V
               (d, None, None, w, hh, 0, 128, 5), (None, None, None, w, hh, 0, 0, 6),   # packed: c_pitch != 0, null plane
               (d, u, v, w, hh, w - 1, 0, 2), (d, u, v, w, hh, 0, 31, 2),           # pitches below the row sizes
               (d, u, None, w, hh, 0, 63, 3), (d, u, v, w, hh, 0, 63, 4),
               (d, None, None, w, hh, 2 * w - 1, 0, 5), (d, None, None, 7, hh, 7, 0, 6),   # packed rows are 4 ceil(w/2)
               (d, u, v, 0, hh, 0, 0, 4), (d, u, v, w, 0, 0, 0, 4), (d, None, None, 65536, hh, 0, 0, 5),
               (d, u, v, w, 65536, 0, 0, 2)]
        for a in bad:
            assert lib.jpgenc_bind_device_yuv(h, *a) == ERR_ARG, a
            assert lib.jpgenc_encode_yuv(h, *a, out.ctypes.data, out.size, C.byref(n)) == ERR_ARG, a
            assert packed_call(lib.jpgenc_encode_images_packed_yuv, a) == ERR_ARG, a
        # the 4:2:0 calls keep refusing every other layout, even with planes that would suit it
        for code, a in ((2, (d, u, v)), (3, (d, u, None)), (4, (d, u, v)), (5, (d, None, None)), (6, (d, None, None))):
            args = a + (w, hh, 0, 0, code)
            assert lib.jpgenc_bind_device_yuv420(h, *args) == ERR_ARG, code
            assert lib.jpgenc_encode_yuv420(h, *args, out.ctypes.data, out.size, C.byref(n)) == ERR_ARG, code
            assert packed_call(lib.jpgenc_encode_images_packed_yuv420, args) == ERR_ARG, code
            assert lib.jpgenc_bind_device_yuv(h, *args) == OK, code                 # ... which the generic calls take
        # n = 0 is legal and touches nothing
        total = C.c_uint64(7)
        assert lib.jpgenc_encode_images_packed_yuv(h, 0, None, 1, None, None, None, None, 5, None, 0, None, None, C.byref(total)) == OK
        assert total.value == 0
        assert encoder.encode_yuv_many("I444", []) == []
    finally:
        encoder.dev_free(d)


@pytest.mark.gpu
def test_tensors_on_the_gpu_and_the_cpu(encoder, oracle):
    import torch
    w, h = 643, 481                                                     # odd: the packed rows' last Y1 is not read
    y, u, v = yuv_of(synth_rgb(w, h, 3), 1)
    want = oracle_file(oracle, y, u, v)
    y4, u4, v4 = yuv_of(synth_rgb(300, 201, 4), 0)
    want4 = oracle_file(oracle, y4, u4, v4)
    yuyv = packed_of("YUYV", y, u, v)
    for dev in ("cuda:0", "cpu"):
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        assert encoder.encode_yuv("YUYV", t(yuyv), w=w) == want, dev
        assert encoder.encode_yuv("YUYV", t(yuyv).view(h, -1, 4), w=w) == want, dev
        assert encoder.encode_yuv("I422", t(y), t(u), t(v)) == want, dev
        assert encoder.encode_yuv("NV16", t(y), t(interleave(u, v))) == want, dev
        assert encoder.encode_yuv("I444", t(y4), t(u4), t(v4)) == want4, dev
        got = encoder.encode_yuv_many("UYVY", [(t(packed_of("UYVY", y, u, v)), None, None, w)] * 2)
        assert got == [want, want], dev
        assert encoder.encode_yuv_many("I444", [(t(y4), t(u4), t(v4))]) == [want4], dev


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1, 1), (17, 9), (1001, 667)])
def test_cross_layout_identities(encoder, w, h):
    """no oracle: I422 of an I420 frame's chroma rows repeated, and I444 of its chroma repeated 2x2, give the I420 file; NV16,
    YUYV and UYVY of the same samples give the I422 file"""
    rng = np.random.default_rng(w * h)
    ch, cw = (h + 1) // 2, (w + 1) // 2
    y = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
    u, v = (rng.integers(0, 256, size=(ch, cw), dtype=np.uint8) for _ in range(2))
    rows = lambda c: np.ascontiguousarray(np.repeat(c, 2, axis=0)[:h])
    full = lambda c: np.ascontiguousarray(np.repeat(rows(c), 2, axis=1)[:, :w])
    want420 = encoder.encode_yuv420(y, u, v)
    assert encoder.encode_yuv("I422", y, rows(u), rows(v)) == want420
    assert encoder.encode_yuv("I444", y, full(u), full(v)) == want420
    u2, v2 = (rng.integers(0, 256, size=(h, cw), dtype=np.uint8) for _ in range(2))
    want422 = encoder.encode_yuv("I422", y, u2, v2)
    assert encoder.encode_yuv("NV16", y, interleave(u2, v2)) == want422
    for lay in ("YUYV", "UYVY"):
        assert encoder.encode_yuv(lay, packed_of(lay, y, u2, v2), w=w) == want422, lay


# ---- no GPU -------------------------------------------------------------------------------------------------------------------

def test_yuv_layout_accepts():
    import torch
    h, w = 11, 7
    cw = 4
    assert YUV_FORMATS == {"I420": 0, "NV12": 1, "I422": 2, "NV16": 3, "I444": 4, "YUYV": 5, "UYVY": 6}
    big = np.zeros((3 * h, 32), np.uint8)
    y = big[:h, :w]
    u, v = big[h: 2 * h, :cw], big[2 * h:, 3: 3 + cw]
    assert yuv_layout("I422", y, u, v) == ("I422", (y.ctypes.data, u.ctypes.data, v.ctypes.data), w, h, 32, 32)
    assert yuv_layout("I422", y, u, v, w=7)[2] == 7
    uv = big[h: 2 * h, : 2 * cw]
    assert yuv_layout("NV16", y, uv) == ("NV16", (y.ctypes.data, uv.ctypes.data, 0), w, h, 32, 32)
    uv3 = np.zeros((h, 40), np.uint8)[:, : 2 * cw].reshape(h, cw, 2)
    assert yuv_layout("NV16", y, uv3)[4:] == (32, 40)
    u4, v4 = big[h: 2 * h, :w], big[2 * h:, 1: 1 + w]
    assert yuv_layout("I444", y, u4, v4) == ("I444", (y.ctypes.data, u4.ctypes.data, v4.ctypes.data), w, h, 32, 32)
    pk = np.zeros((h, 40), np.uint8)[:, : 4 * cw]
    for lay in ("YUYV", "UYVY"):
        assert yuv_layout(lay, pk) == (lay, (pk.ctypes.data, 0, 0), 2 * cw, h, 40, 0)
        assert yuv_layout(lay, pk, w=2 * cw - 1)[2] == 2 * cw - 1                 # odd width
        assert yuv_layout(lay, np.zeros((h, cw, 4), np.uint8))[2:] == (2 * cw, h, 4 * cw, 0)
    assert yuv_layout("YUYV", np.zeros((1, 4), np.uint8), w=1)[2:] == (1, 1, 4, 0)
    assert yuv_layout("I444", np.zeros((1, 1), np.uint8), np.zeros((1, 1), np.uint8), np.zeros((1, 1), np.uint8))[2:] == (1, 1, 1, 1)
    # the 4:2:0 layouts by name are yuv420_layout's rule
    i420 = yuv_layout("I420", y, big[h: h + 6, :cw], big[2 * h: 2 * h + 6, :cw])
    assert i420[0] == "I420" and i420[2:] == (w, h, 32, 32)
    t = torch.zeros((2 * h, 16), dtype=torch.uint8)
    assert yuv_layout("NV16", t[:h, :w], t[h:, :8]) == ("NV16", (t.data_ptr(), t.data_ptr() + 16 * h, 0), w, h, 16, 16)
    tp = torch.zeros((h, 3, 16), dtype=torch.uint8)
    assert yuv_layout("UYVY", tp[:, 0, :])[4:] == (48, 0)


def test_yuv_layout_refuses():
    import torch
    y = np.zeros((10, 8), np.uint8)
    u = np.zeros((10, 4), np.uint8)
    u4 = np.zeros((10, 8), np.uint8)
    pk = np.zeros((10, 16), np.uint8)
    bad = [
        ("I411", y, u, u),                                        # unknown layout
        ("I422", y.astype(np.uint16), u, u),                      # dtype
        ("I422", y, np.zeros((5, 4), np.uint8), u),               # 4:2:0 chroma for 4:2:2
        ("I422", y, u, np.zeros((10, 5), np.uint8)),              # V shape
        ("I422", y, u),                                           # V missing
        ("I422", y, u, np.zeros((10, 6), np.uint8)[:, :4]),       # U and V row strides differ
        ("I422", y, np.zeros((10, 8), np.uint8)[:, ::2], u),      # U element stride
        ("I444", y, u, u),                                        # 4:2:2 chroma for 4:4:4
        ("I444", y, u4, u4, 9),                                   # w disagrees
        ("NV16", y, np.zeros((10, 7), np.uint8)),                 # NV16 shape
        ("NV16", y, np.zeros((10, 8), np.uint8), u),              # NV16 with a V
        ("NV16", y, np.zeros((10, 4, 2), np.uint8)[:, :, ::-1]),  # NV16 byte order stride
        ("YUYV", pk, u),                                          # packed with a U
        ("YUYV", np.zeros((10, 15), np.uint8)),                   # not whole groups
        ("UYVY", np.zeros((10, 16), np.uint8)[:, ::2]),           # element stride
        ("UYVY", np.zeros((10, 4, 3), np.uint8)),                 # groups of 3
        ("YUYV", pk, None, None, 6),                              # 4 groups hold 7 or 8 pixels
        ("YUYV", pk, None, None, 9),
        ("YUYV", np.zeros((0, 16), np.uint8)),                    # empty
        ("I420", y, np.zeros((5, 4), np.uint8)),                  # I420 without V
        ("NV12", y, np.zeros((5, 4), np.uint8), np.zeros((5, 4), np.uint8)),   # NV12 with a V
        ("I422", [[0] * 8] * 10, u, u),                           # not an array
        ("I422", torch.zeros((10, 8), dtype=torch.uint8).t(), u, u),   # transposed
    ]
    for a in bad:
        with pytest.raises(ValueError):
            yuv_layout(*a)


@pytest.mark.parametrize("hs", [1, 0])
def test_u_is_cb_and_v_is_cr(oracle, hs):
    """PIL decodes the oracle's file of an odd-sized 4:2:2 / 4:4:4 frame's defining planes back to planes close to Y, U and V
    (at the 2x2 cells of the 4:2:0 file); with U and V swapped the chroma is far off"""
    import io
    from PIL import Image
    w, h = 37, 23
    y, u, v = yuv_of(synth_rgb(w, h, 12), hs)
    im = Image.open(io.BytesIO(oracle_file(oracle, y, u, v)))
    im.draft("YCbCr", (w, h))
    assert im.mode == "YCbCr" and im.size == (w, h)
    dec = np.asarray(im).astype(np.int32)
    cb, cr = dec[::2, ::2, 1], dec[::2, ::2, 2]
    cell = lambda c: (np.repeat(c, 2, axis=1)[:, :w] if hs else c)[::2, ::2].astype(np.int32)
    err_y = np.abs(dec[:, :, 0] - y).mean()
    err_c = (np.abs(cb - cell(u)).mean() + np.abs(cr - cell(v)).mean()) / 2
    err_swapped = (np.abs(cb - cell(v)).mean() + np.abs(cr - cell(u)).mean()) / 2
    assert err_y < 6 and err_c < 8, (err_y, err_c)
    assert err_swapped > 3 * err_c, (err_swapped, err_c)
