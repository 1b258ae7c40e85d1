"""YUV 4:2:0 frames (I420, NV12) read in place: jpgenc_bind_device_yuv420, jpgenc_encode_yuv420, jpgenc_encode_images_packed_yuv420
and Encoder.encode_yuv420 / encode_yuv420_many.  The file of a frame is defined as Image::writeJPEG of the YCbCr image whose
level-shifted planes are the samples minus 128, every chroma sample repeated over its 2x2 pixels and the frame padded to whole
MCUs by edge replication (expected_planes): every file must be byte-identical to the oracle's (or the GPU's FP64 path's) file of
those planes.  The bytes between rows and around the planes are random, so reading any of them would change the file."""
import os
import subprocess
import sys

import numpy as np
import pytest

from jpgenc_b200.capi import YUV_LAYOUTS, yuv420_layout
from jpgenc_b200.synth import synth_rgb

SIZES = [(1, 1), (17, 9), (208, 120), (1000, 667), (1920, 1080)]


def yuv_of(rgb):
    """full-range BT.601 Y, Cb, Cr of an RGB image, chroma taken at the top-left pixel of every 2x2 cell"""
    f = rgb.astype(np.float64)
    r, g, b = f[:, :, 0], f[:, :, 1], f[:, :, 2]
    y = 0.299 * r + 0.587 * g + 0.114 * b
    u = 128 + 0.564 * (b - y)
    v = 128 + 0.713 * (r - y)
    q = lambda p: np.clip(np.rint(p), 0, 255).astype(np.uint8)
    return q(y), q(u[::2, ::2]), q(v[::2, ::2])


def noise_yuv(w, h, seed):
    """random planes that reach 0 and 255"""
    rng = np.random.default_rng(seed)
    y = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
    u = rng.integers(0, 256, size=((h + 1) // 2, (w + 1) // 2), dtype=np.uint8)
    v = rng.integers(0, 256, size=u.shape, dtype=np.uint8)
    y.flat[0], u.flat[0], v.flat[-1] = 0, 255, 0
    y.flat[-1], v.flat[0] = 255, 255
    return y, u, v


def expected_planes(y, u, v):
    """the level-shifted (H16, W16) planes Y', Cb', Cr' that define a frame's file"""
    h, w = y.shape
    h16, w16 = (h + 15) // 16 * 16, (w + 15) // 16 * 16
    up = lambda c: np.repeat(np.repeat(c, 2, axis=0), 2, axis=1)[:h, :w]
    pad = lambda p: np.pad(p.astype(np.float64) - 128.0, ((0, h16 - h), (0, w16 - w)), mode="edge")
    return pad(y), pad(up(u)), pad(up(v))


def oracle_file(oracle, y, u, v):
    h, w = y.shape
    return oracle.encode_planes(*expected_planes(y, u, v), w, h, ycbcr=True)


def nv12_of(u, v):
    """the (ch, 2 cw) interleaved UV plane"""
    uv = np.empty((u.shape[0], 2 * u.shape[1]), np.uint8)
    uv[:, 0::2], uv[:, 1::2] = u, v
    return uv


def pitch_kinds(w):
    """tight; a multiple of 16 above the row (bulk copies where the width allows it); tight + 3 (clamped loads)"""
    return {"tight": w, "pitch16": (w + 15) // 16 * 16 + 16, "pitch+3": w + 3}


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
    """a frame's planes in device memory, each in an allocation of its own laid out by plane_bytes; .ptr = (y, u, v or 0)"""

    def __init__(self, enc, y, u, v, layout, kind, offset, seed):
        self.enc, self.d = enc, []
        planes = [y, u, v] if layout == "I420" else [y, nv12_of(u, v)]
        self.y_pitch = pitch_kinds(y.shape[1])[kind]
        self.c_pitch = pitch_kinds(planes[1].shape[1])[kind]
        ptr = []
        for k, p in enumerate(planes):
            buf, _ = plane_bytes(p, self.y_pitch if k == 0 else self.c_pitch, seed + k, offset)
            d = enc.dev_alloc(buf.nbytes + 16)
            enc.h2d(d, buf)
            self.d.append(d)
            ptr.append(d + offset)
        self.ptr = tuple(ptr) + ((0,) if layout == "NV12" else ())

    def free(self):
        for d in self.d:
            self.enc.dev_free(d)


@pytest.fixture(scope="module")
def frames(oracle):
    """per size: a frame derived from synth_rgb and a noise frame, with the oracle's files (and, for the first, of U, V swapped)"""
    out = []
    for k, (w, h) in enumerate(SIZES):
        syn = yuv_of(synth_rgb(w, h, 41 + k))
        noise = noise_yuv(w, h, 7 + k)
        out.append((syn, oracle_file(oracle, *syn), oracle_file(oracle, syn[0], syn[2], syn[1])))
        out.append((noise, oracle_file(oracle, *noise), None))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["I420", "NV12"])
def test_single_device_frames(encoder, frames, layout):
    for kind in ("tight", "pitch16", "pitch+3"):
        for offset in (0, 1):
            refined = 0
            for k, ((y, u, v), want, want_swapped) in enumerate(frames):
                h, w = y.shape
                f = DeviceFrame(encoder, y, u, v, layout, kind, offset, seed=3 * k)
                try:
                    encoder.bind_device_yuv420(*f.ptr, w, h, f.y_pitch, f.c_pitch, layout)
                    got = _encode_bound(encoder, len(want) + 4096)
                    refined += encoder.stats().refined_blocks
                    got_swapped = None
                    if layout == "I420" and want_swapped is not None:          # YV12: the same call with U and V swapped
                        encoder.bind_device_yuv420(f.ptr[0], f.ptr[2], f.ptr[1], w, h, f.y_pitch, f.c_pitch, layout)
                        got_swapped = _encode_bound(encoder, len(want_swapped) + 4096)
                finally:
                    f.free()
                assert got == want, f"{layout} {w}x{h} ({kind}) offset {offset}"
                if got_swapped is not None:
                    assert got_swapped == want_swapped, f"I420 with U, V swapped {w}x{h} ({kind}) offset {offset}"
            assert refined > 0, "no block took the FP64 refinement: its sample gather was not exercised"


@pytest.mark.gpu
def test_fp32_bound_at_scale(encoder):
    """4096 x 4096 noise and synthetic frames: the FP32 path with its exact-input thresholds (plus refinement) equals the GPU's
    independent FP64 path on the defining planes"""
    w = h = 4096
    for y, u, v in (noise_yuv(w, h, 99), yuv_of(synth_rgb(w, h, 5))):
        want = encoder.encode_planes(*expected_planes(y, u, v), w, h, ycbcr=True)
        for layout in ("I420", "NV12"):
            f = DeviceFrame(encoder, y, u, v, layout, "tight", 0, seed=1)
            try:
                encoder.bind_device_yuv420(*f.ptr, w, h, 0, 0, layout)
                got = _encode_bound(encoder, len(want) + 4096)
            finally:
                f.free()
            assert got == want, f"{layout} 4096x4096"


@pytest.mark.gpu
def test_host_frames_in_several_bands(encoder):
    """4000 x 3000 host frames (several upload bands), tight and pitched: each equals the device path's file"""
    w, h = 4000, 3000
    y, u, v = yuv_of(synth_rgb(w, h, 17))
    for layout in ("I420", "NV12"):
        f = DeviceFrame(encoder, y, u, v, layout, "tight", 0, seed=2)
        try:
            encoder.bind_device_yuv420(*f.ptr, w, h, 0, 0, layout)
            want = _encode_bound(encoder, w * h)
        finally:
            f.free()
        for kind in ("tight", "pitch+3"):
            _, yv = plane_bytes(y, pitch_kinds(w)[kind], 3)
            if layout == "I420":
                _, uv_ = plane_bytes(u, pitch_kinds(u.shape[1])[kind], 4)
                _, vv = plane_bytes(v, pitch_kinds(u.shape[1])[kind], 5)
                got = encoder.encode_yuv420(yv, uv_, vv)
            else:
                c = nv12_of(u, v)
                _, cv = plane_bytes(c, pitch_kinds(c.shape[1])[kind], 4)
                got = encoder.encode_yuv420(yv, cv.reshape(c.shape[0], -1, 2) if kind == "tight" else cv)
            assert got == want, f"host {layout} ({kind})"


def _tiles(W, H, T):
    return [(x, y, min(T, W - x), min(T, H - y)) for y in range(0, H, T) for x in range(0, W, T)]


class BigFrame:
    """a W x H YUV frame (odd sides: ragged odd-sized edge tiles) with pitched planes in one buffer in device or pinned host
    memory, cut into T x T tiles: plane pointers into it, and the oracle's file of every tile"""

    def __init__(self, enc, oracle, layout, W=1501, H=1099, T=256, host=False, tiles=None):
        from jpgenc_b200.capi import pinned_empty
        self.enc, self.host, self.layout = enc, host, layout
        y, u, v = yuv_of(synth_rgb(W, H, 23))
        cplanes = [u, v] if layout == "I420" else [nv12_of(u, v)]
        self.y_pitch, self.c_pitch = W + 5, cplanes[0].shape[1] + 3
        ch = u.shape[0]
        c_at = [H * self.y_pitch + 16 + k * (ch * self.c_pitch + 16) for k in range(len(cplanes))]
        buf = np.random.default_rng(9).integers(0, 256, size=c_at[-1] + ch * self.c_pitch + 16, dtype=np.uint8)
        np.lib.stride_tricks.as_strided(buf, shape=y.shape, strides=(self.y_pitch, 1))[:] = y
        for at, p in zip(c_at, cplanes):
            np.lib.stride_tricks.as_strided(buf[at:], shape=p.shape, strides=(self.c_pitch, 1))[:] = p
        if host:
            self.view, self.base = pinned_empty(buf.nbytes)
            self.view[:] = buf
        else:
            self.base = enc.dev_alloc(buf.nbytes)
            enc.h2d(self.base, buf)
        tl = _tiles(W, H, T)[:tiles]
        es = 1 if layout == "I420" else 2
        self.ptrs = []
        for x, yy, _, _ in tl:
            self.ptrs.append(self.base + yy * self.y_pitch + x)
            for at in c_at:
                self.ptrs.append(self.base + at + yy // 2 * self.c_pitch + x // 2 * es)
            if layout == "NV12":
                self.ptrs.append(None)
        self.ws = [w for _, _, w, _ in tl]
        self.hs = [h for _, _, _, h in tl]
        self.want = [oracle_file(oracle, y[yy: yy + h, x: x + w], u[yy // 2: (yy + h + 1) // 2, x // 2: (x + w + 1) // 2],
                                 v[yy // 2: (yy + h + 1) // 2, x // 2: (x + w + 1) // 2]) for x, yy, w, h in tl]

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
        return enc.encode_images_packed_yuv420(big.ptrs, big.ws, big.hs, o, c, big.layout, host_images=big.host,
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
@pytest.mark.parametrize("layout", ["I420", "NV12"])
@pytest.mark.parametrize("host", [False, True])
def test_tiles_of_one_frame(encoder, oracle, layout, host):
    big = BigFrame(encoder, oracle, layout, host=host)
    try:
        _check_packed(encoder, big)
    finally:
        big.free()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["I420", "NV12"])
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
    """one device buffer bound as RGB, GRAY, I420 and NV12 with the same first pointer and size, each twice in a row; then I420
    with the same planes and only a wider chroma pitch"""
    from jpgenc_b200.capi import Encoder
    from oracle.pyoracle import Oracle
    oracle = Oracle()
    enc = Encoder(0)
    w, h = 333, 201
    cw, ch = (w + 1) // 2, (h + 1) // 2
    buf = np.random.default_rng(3).integers(0, 256, size=3 * w * h, dtype=np.uint8)
    d = enc.dev_alloc(buf.nbytes)
    try:
        enc.h2d(d, buf)
        y = buf[: w * h].reshape(h, w)
        u = buf[w * h: w * h + cw * ch].reshape(ch, cw)
        v = buf[w * h + cw * ch: w * h + 2 * cw * ch].reshape(ch, cw)
        uv = buf[w * h: w * h + 2 * cw * ch].reshape(ch, 2 * cw)
        cp = cw + 3                                                  # I420 at the same plane pointers, rows cp bytes apart
        strided = lambda at: np.lib.stride_tricks.as_strided(buf[at:], shape=(ch, cw), strides=(cp, 1))
        want = {"RGB": oracle.encode_rgb(buf.reshape(h, w, 3)), "GRAY": oracle.encode_rgb(np.repeat(y[:, :, None], 3, axis=2)),
                "I420": oracle_file(oracle, y, u, v), "NV12": oracle_file(oracle, y, uv[:, 0::2], uv[:, 1::2]),
                "I420_pitched": oracle_file(oracle, y, strided(w * h), strided(w * h + cw * ch))}
        for _ in range(2):
            for kind in ("RGB", "GRAY", "I420", "I420_pitched", "NV12"):
                for _ in range(2):
                    if kind == "RGB":
                        enc.bind_device_rgb(d, w, h)
                    elif kind == "GRAY":
                        enc.bind_device_image(d, w, h, 0, "GRAY")
                    elif kind == "I420":
                        enc.bind_device_yuv420(d, d + w * h, d + w * h + cw * ch, w, h, 0, 0, "I420")
                    elif kind == "I420_pitched":
                        enc.bind_device_yuv420(d, d + w * h, d + w * h + cw * ch, w, h, 0, cp, "I420")
                    else:
                        enc.bind_device_yuv420(d, d + w * h, None, w, h, 0, 0, "NV12")
                    assert _encode_bound(enc, 1 << 20) == want[kind], kind
    finally:
        enc.dev_free(d)
        enc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("graphs", ["1", "0"])
def test_graph_cache_keys_on_yuv_layouts(graphs):
    # JPGENC_GRAPHS is read once per process: each setting runs in a process of its own
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, JPGENC_GRAPHS=graphs,
               PYTHONPATH=os.pathsep.join([root, os.path.dirname(os.path.abspath(__file__))]))
    r = subprocess.run([sys.executable, "-c", "import test_yuv420 as t; t._graph_cycle()"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_argument_errors(encoder):
    from jpgenc_b200.capi import ERR_ARG, OK
    import ctypes as C
    lib, h = encoder.lib, encoder.h
    d = encoder.dev_alloc(1 << 16)
    w, hh = 64, 32
    u, v = d + w * hh, d + w * hh + 32 * 16
    try:
        bad = [(d, u, v, w, hh, 0, 0, 2), (d, u, v, w, hh, 0, 0, -1),               # unknown layout
               (None, u, v, w, hh, 0, 0, 0), (d, None, v, w, hh, 0, 0, 0),          # null Y, null U
               (d, u, None, w, hh, 0, 0, 0), (d, u, v, w, hh, 0, 0, 1),             # null V for I420, a V for NV12
               (d, u, v, w, hh, w - 1, 0, 0), (d, u, v, w, hh, 0, 31, 0),           # pitches below the row sizes
               (d, u, None, w, hh, 0, 63, 1),
               (d, u, v, 0, hh, 0, 0, 0), (d, u, v, w, 0, 0, 0, 0), (d, u, v, 65536, hh, 0, 0, 0), (d, u, v, w, 65536, 0, 0, 0)]
        out = np.empty(1 << 16, np.uint8)
        n = C.c_uint64()
        for a in bad:
            assert lib.jpgenc_bind_device_yuv420(h, *a) == ERR_ARG, a
            assert lib.jpgenc_encode_yuv420(h, *a, out.ctypes.data, out.size, C.byref(n)) == ERR_ARG, a
            pl = (C.c_void_p * 3)(*a[:3])
            ws, hs = np.array([a[3]], np.uint32), np.array([a[4]], np.uint32)
            yp, cp = np.array([a[5]], np.uint32), np.array([a[6]], np.uint32)
            offs, sizes, total = (C.c_uint64 * 1)(), (C.c_uint64 * 1)(), C.c_uint64()
            u32 = C.POINTER(C.c_uint32)
            assert lib.jpgenc_encode_images_packed_yuv420(h, 1, pl, 1, ws.ctypes.data_as(u32), hs.ctypes.data_as(u32), yp.ctypes.data_as(u32),
                                                          cp.ctypes.data_as(u32), a[7], None, 0, offs, sizes, C.byref(total)) == ERR_ARG, a
        # n = 0 is legal and touches nothing
        total = C.c_uint64(7)
        assert lib.jpgenc_encode_images_packed_yuv420(h, 0, None, 1, None, None, None, None, 0, None, 0, None, None, C.byref(total)) == OK
        assert total.value == 0
        assert encoder.encode_yuv420_many([]) == []
    finally:
        encoder.dev_free(d)


@pytest.mark.gpu
def test_tensors_on_the_gpu_and_the_cpu(encoder, oracle):
    import torch
    w, h = 642, 481
    y, u, v = yuv_of(synth_rgb(w, h, 3))
    ch = u.shape[0]
    want = oracle_file(oracle, y, u, v)
    buf = np.empty((h + ch, w), np.uint8)                     # an NV12 surface: Y rows, then the UV rows, one pitch
    buf[:h], buf[h:] = y, nv12_of(u, v)
    y2, u2, v2 = yuv_of(synth_rgb(300, 201, 4))
    want2 = oracle_file(oracle, y2, u2, v2)
    for dev in ("cuda:0", "cpu"):
        t = torch.from_numpy(buf).to(dev)
        assert encoder.encode_yuv420(t[:h], t[h:]) == want, dev
        assert encoder.encode_yuv420(t[:h], t[h:].view(ch, w // 2, 2)) == want, dev
        planes = [torch.from_numpy(p).to(dev) for p in (y, u, v)]
        planes2 = [torch.from_numpy(p).to(dev) for p in (y2, u2, v2)]
        assert encoder.encode_yuv420(*planes) == want, dev
        assert encoder.encode_yuv420_many([planes, planes2]) == [want, want2], dev
        assert encoder.encode_yuv420_many([(t[:h], t[h:]), (t[:h], t[h:])]) == [want, want], dev
    with pytest.raises(ValueError):
        encoder.encode_yuv420_many([(y, nv12_of(u, v)), (y, u, v)])           # one layout per call


@pytest.mark.gpu
def test_tensor_written_on_another_stream(encoder, oracle):
    """the planes are filled by work queued on a non-default current stream right before the call: the encoder must read them only
    after that work"""
    import torch
    y, u, v = yuv_of(synth_rgb(1920, 1080, 13))
    src = [torch.from_numpy(p).cuda(0) for p in (y, u, v)]
    dst = [torch.zeros_like(p) for p in src]
    s = torch.cuda.Stream(0)
    s.wait_stream(torch.cuda.current_stream(0))                                               # after the zero fill of dst
    with torch.cuda.stream(s):
        torch.cuda._sleep(20_000_000)                                                          # the copies below start late
        for a, b in zip(dst, src):
            a.copy_(b)
        got = encoder.encode_yuv420(*dst)
    assert got == oracle_file(oracle, y, u, v)


# ---- no GPU -------------------------------------------------------------------------------------------------------------------

def test_yuv420_layout_accepts():
    import torch
    h, w = 11, 7
    ch, cw = 6, 4
    big = np.zeros((h + ch, 16), np.uint8)
    y, uv = big[:h, :w], big[h:, : 2 * cw]
    assert YUV_LAYOUTS == {"I420": 0, "NV12": 1}
    assert yuv420_layout(y, uv) == ("NV12", (y.ctypes.data, uv.ctypes.data, 0), w, h, 16, 16)
    uv3 = np.zeros((ch, 20), np.uint8)[:, :8].reshape(ch, cw, 2)
    assert yuv420_layout(y, uv3)[5] == 20
    u, v = np.zeros((ch, 9), np.uint8)[:, :cw], np.zeros((ch, 9), np.uint8)[:, 1: cw + 1]
    assert yuv420_layout(y, u, v) == ("I420", (y.ctypes.data, u.ctypes.data, v.ctypes.data), w, h, 16, 9)
    t = torch.zeros((h + ch, 16), dtype=torch.uint8)
    assert yuv420_layout(t[:h, :w], t[h:, :8]) == ("NV12", (t.data_ptr(), t.data_ptr() + 16 * h, 0), w, h, 16, 16)
    tp = torch.zeros((3, 8, 8), dtype=torch.uint8)
    lay = yuv420_layout(tp[0, :, :7], tp[1, :4, :4], tp[2, :4, :4])
    assert lay[0] == "I420" and lay[4:] == (8, 8)
    assert yuv420_layout(np.zeros((1, 1), np.uint8), np.zeros((1, 1), np.uint8), np.zeros((1, 1), np.uint8))[2:] == (1, 1, 1, 1)
    assert yuv420_layout(np.zeros((1, 1), np.uint8), np.zeros((1, 2), np.uint8))[2:] == (1, 1, 1, 2)


def test_yuv420_layout_refuses():
    import torch
    y = np.zeros((10, 8), np.uint8)
    u = np.zeros((5, 4), np.uint8)
    bad = [
        (y.astype(np.uint16), u, u),                              # dtype
        (np.zeros((10, 8, 1), np.uint8), u, u),                   # Y shape
        (y[:, ::2], np.zeros((5, 2), np.uint8), np.zeros((5, 2), np.uint8)),   # Y element stride
        (y, np.zeros((5, 5), np.uint8), u),                       # U shape
        (y, u, np.zeros((4, 4), np.uint8)),                       # V shape
        (y, np.zeros((5, 8), np.uint8)[:, ::2], u),               # U element stride
        (y, u, np.zeros((5, 6), np.uint8)[:, :4]),                # U and V row strides differ
        (y, np.zeros((5, 8), np.uint16)),                         # NV12 dtype
        (y, np.zeros((5, 7), np.uint8)),                          # NV12 shape
        (y, np.zeros((5, 4, 2), np.uint8)[:, :, ::-1]),           # NV12 byte order stride
        (y, np.zeros((5, 16), np.uint8)[:, ::2]),                 # NV12 element stride
        (np.zeros((0, 8), np.uint8), u, u),                       # empty
        (y, [[0] * 4] * 5, u),                                    # not an array
        (torch.zeros((10, 8), dtype=torch.int16), u, u),          # tensor dtype
        (torch.zeros((10, 8), dtype=torch.uint8).t(), u, u),      # transposed
    ]
    for a in bad:
        with pytest.raises(ValueError):
            yuv420_layout(*a)


def test_u_is_cb_and_v_is_cr(oracle):
    """PIL decodes the oracle's file of an odd-sized I420 frame back to planes close to Y, U and V; with U and V swapped the
    chroma is far off.  Pins the convention that the byte-identity tests cannot see (they build both sides the same way)."""
    import io
    from PIL import Image
    w, h = 37, 23
    rgb = synth_rgb(w, h, 12)
    y, u, v = yuv_of(rgb)
    im = Image.open(io.BytesIO(oracle_file(oracle, y, u, v)))
    im.draft("YCbCr", (w, h))
    assert im.mode == "YCbCr" and im.size == (w, h)
    dec = np.asarray(im).astype(np.int32)
    cb, cr = dec[::2, ::2, 1], dec[::2, ::2, 2]
    err_y = np.abs(dec[:, :, 0] - y).mean()
    err_c = (np.abs(cb - u).mean() + np.abs(cr - v).mean()) / 2
    err_swapped = (np.abs(cb - v).mean() + np.abs(cr - u).mean()) / 2
    assert err_y < 6 and err_c < 6, (err_y, err_c)
    assert err_swapped > 3 * err_c, (err_swapped, err_c)
