"""Greyscale (JPGENC_PIXEL_GRAY) and planar RGB pixels, and torch tensors read in place (Encoder.encode_tensor / encode_tensors).
A grey image v is encoded as the RGB image (v, v, v) and planar RGB as the interleaved image of its planes: every file must be
byte-identical to the oracle's (or, for images the oracle would be slow on, to jpgenc_encode_rgb) on that tight RGB image.  The
bytes between rows and around the planes are random, so reading any of them would change the file."""
import os
import subprocess
import sys

import numpy as np
import pytest

from jpgenc_b200.capi import image_layout, tensor_layout
from jpgenc_b200.synth import ppm_p6_bytes, synth_rgb

SIZES = [(1, 1), (17, 9), (208, 120), (1000, 667), (1920, 1080)]


def grey_of(rgb):
    return np.ascontiguousarray(rgb[:, :, 1])


def as_rgb(grey):
    return np.repeat(grey[:, :, None], 3, axis=2)


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


@pytest.fixture(scope="module")
def sized(oracle):
    """one synthetic image per size of SIZES, its grey image, and the oracle's files of the RGB image and of the grey one"""
    imgs = [synth_rgb(w, h, 31 + k) for k, (w, h) in enumerate(SIZES)]
    return imgs, [oracle.encode_rgb(a) for a in imgs], [oracle.encode_rgb(as_rgb(grey_of(a))) for a in imgs]


class DevicePlanes:
    """the three planes of `rgb` in device memory, each in an allocation of its own laid out by plane_bytes, allocated in the
    order `alloc_order` (a permutation of 0, 1, 2) so that the pointers are not in R, G, B order in memory"""

    def __init__(self, enc, rgb, pitch, offset, seed, alloc_order=(0, 1, 2)):
        self.enc, self.d, self.ptr = enc, [], [0, 0, 0]
        for k in alloc_order:
            buf, _ = plane_bytes(rgb[:, :, k], pitch, seed + k, offset)
            d = enc.dev_alloc(buf.nbytes + 16)
            enc.h2d(d, buf)
            self.d.append(d)
            self.ptr[k] = d + offset

    def free(self):
        for d in self.d:
            self.enc.dev_free(d)


@pytest.mark.gpu
def test_single_device_grey(encoder, sized):
    imgs, _, want = sized
    for kind in ("tight", "pitch16", "pitch+3"):
        for offset in (0, 1):
            refined = 0
            for k, (rgb, ref) in enumerate(zip(imgs, want)):
                h, w, _ = rgb.shape
                pitch = pitch_kinds(w)[kind]
                buf, _ = plane_bytes(grey_of(rgb), pitch, seed=k, offset=offset)
                d = encoder.dev_alloc(buf.nbytes + 16)
                try:
                    encoder.h2d(d, buf)
                    encoder.bind_device_image(d + offset, w, h, pitch, "GRAY")
                    got = _encode_bound(encoder, len(ref) + 4096)
                    refined += encoder.stats().refined_blocks
                finally:
                    encoder.dev_free(d)
                assert got == ref, f"GRAY {w}x{h} pitch {pitch} ({kind}) offset {offset}"
            assert refined > 0, "no block took the FP64 refinement: its pixel gather was not exercised"


@pytest.mark.gpu
@pytest.mark.parametrize("alloc_order", [(0, 1, 2), (2, 0, 1)])
def test_single_device_planar(encoder, sized, alloc_order):
    imgs, want, want_grey = sized
    for kind in ("tight", "pitch16", "pitch+3"):
        for offset in (0, 1):
            refined = 0
            for k, (rgb, ref) in enumerate(zip(imgs, want)):
                h, w, _ = rgb.shape
                pitch = pitch_kinds(w)[kind]
                pl = DevicePlanes(encoder, rgb, pitch, offset, seed=3 * k, alloc_order=alloc_order)
                try:
                    encoder.bind_device_planar(*pl.ptr, w, h, pitch)
                    got = _encode_bound(encoder, len(ref) + 4096)
                    refined += encoder.stats().refined_blocks
                    # aliased planes: the G plane as R, G and B is the grey file
                    encoder.bind_device_planar(pl.ptr[1], pl.ptr[1], pl.ptr[1], w, h, pitch)
                    got_grey = _encode_bound(encoder, len(want_grey[k]) + 4096)
                finally:
                    pl.free()
                assert got == ref, f"planar {w}x{h} pitch {pitch} ({kind}) offset {offset}"
                assert got_grey == want_grey[k], f"aliased planes {w}x{h} pitch {pitch} ({kind}) offset {offset}"
            assert refined > 0, "no block took the FP64 refinement: its pixel gather was not exercised"


@pytest.mark.gpu
def test_host_images_in_several_bands(encoder):
    """grey and planar host pixels large enough for several upload bands: pitched grey, a tight (3, H, W) buffer (one copy per
    band for all planes), and pitched planes in separate buffers (one copy per plane and band)"""
    rgb = synth_rgb(4000, 3000, 5)
    want = encoder.encode_rgb(rgb)
    _, grey = plane_bytes(grey_of(rgb), 4000 + 40, seed=1)
    assert encoder.encode_image(grey, "GRAY") == encoder.encode_rgb(as_rgb(grey_of(rgb)))
    assert encoder.stats().refined_blocks > 0
    chw = np.ascontiguousarray(rgb.transpose(2, 0, 1))
    n = 4000 * 3000
    assert encoder.encode_planar(chw.ctypes.data, chw.ctypes.data + n, chw.ctypes.data + 2 * n, 4000, 3000) == want
    planes = [plane_bytes(rgb[:, :, k], 4000 + 24, seed=k)[1] for k in range(3)]
    assert encoder.encode_planar(*(p.ctypes.data for p in planes), 4000, 3000, 4000 + 24) == want
    assert encoder.stats().refined_blocks > 0


@pytest.mark.gpu
def test_maxval_below_255(encoder, oracle):
    """the pitch gap (bytes above maxval) is not read by the check; a sample above maxval in any plane is refused"""
    from jpgenc_b200.capi import ERR_FORMAT, JpgencError
    rgb = (synth_rgb(67, 45, 2).astype(np.uint16) * 100 // 255).astype(np.uint8)
    want = oracle.encode_ppm(ppm_p6_bytes(rgb, 100))
    want_grey = oracle.encode_ppm(ppm_p6_bytes(as_rgb(grey_of(rgb)), 100))
    bufs, planes = [], []
    for k in range(3):
        buf, view = plane_bytes(rgb[:, :, k], 67 + 5, seed=k)
        buf[:] = 255
        view[:] = rgb[:, :, k]
        bufs.append(buf)
        planes.append(view)
    ptrs = [p.ctypes.data for p in planes]
    assert encoder.encode_image(planes[1], "GRAY", maxval=100) == want_grey
    assert encoder.encode_images([planes[1]], maxval=100, fmt="GRAY") == [want_grey]
    assert encoder.encode_planar(*ptrs, 67, 45, 72, maxval=100) == want
    out = np.empty(len(want) + 64, np.uint8)
    offs, sizes, _ = encoder.encode_images_packed_planar(ptrs, [67], [45], out.ctypes.data, out.size, 100, host_images=True, pitches=[72])
    assert out[offs[0]: offs[0] + sizes[0]].tobytes() == want
    for k in range(3):
        planes[k][7, 9 + k] = 101
        calls = [lambda: encoder.encode_planar(*ptrs, 67, 45, 72, maxval=100),
                 lambda: encoder.encode_images_packed_planar(ptrs, [67], [45], None, 0, 100, host_images=True, pitches=[72])]
        if k == 1:
            calls += [lambda: encoder.encode_image(planes[1], "GRAY", maxval=100),
                      lambda: encoder.encode_images([planes[1]], maxval=100, fmt="GRAY")]
        for call in calls:
            with pytest.raises(JpgencError) as e:
                call()
            assert e.value.code == ERR_FORMAT, k
        planes[k][7, 9 + k] = rgb[7, 9 + k, k]


def _tiles(W, H, T):
    return [(x, y, min(T, W - x), min(T, H - y)) for y in range(0, H, T) for x in range(0, W, T)]


class BigImage:
    """a W x H synthetic image as grey (one plane) or planar RGB (three planes one after the other in one buffer, rows `pitch`
    bytes apart) in device or pinned host memory, cut into T x T tiles plus the ragged ones: pointers into it, and the oracle's
    file of every tile"""

    def __init__(self, enc, oracle, planar, W=4000, H=3000, T=256, host=False, pitch=None, tiles=None):
        from jpgenc_b200.capi import pinned_empty
        self.enc, self.host = enc, host
        rgb = synth_rgb(W, H, 23)
        if not planar:
            rgb = as_rgb(grey_of(rgb))
        self.pitch = pitch or W
        nplanes = 3 if planar else 1
        plane = H * self.pitch + 32
        buf = np.random.default_rng(9).integers(0, 256, size=nplanes * plane, dtype=np.uint8)
        for k in range(nplanes):
            np.lib.stride_tricks.as_strided(buf[k * plane:], shape=(H, W), strides=(self.pitch, 1))[:] = rgb[:, :, k]
        if host:
            self.view, self.base = pinned_empty(buf.nbytes)
            self.view[:] = buf
        else:
            self.base = enc.dev_alloc(buf.nbytes)
            enc.h2d(self.base, buf)
        tl = _tiles(W, H, T)[:tiles]
        self.ptrs = [self.base + k * plane + y * self.pitch + x for x, y, _, _ in tl for k in range(nplanes)]
        self.ws = [w for _, _, w, _ in tl]
        self.hs = [h for _, _, _, h in tl]
        self.want = [oracle.encode_rgb(np.ascontiguousarray(rgb[y: y + h, x: x + w])) for x, y, w, h in tl]

    def free(self):
        from jpgenc_b200.capi import pinned_free
        if self.host:
            pinned_free(self.base)
        else:
            self.enc.dev_free(self.base)


def _check_packed(enc, big, planar, host=False):
    """contiguous files in input order, each the expected one; sizes-only gives the same offsets and sizes; a buffer one byte
    short is refused"""
    from jpgenc_b200.capi import ERR_CAPACITY, JpgencError, pinned_empty, pinned_free
    n = len(big.ws)
    pitches = [big.pitch] * n

    def call(o, c):
        if planar:
            return enc.encode_images_packed_planar(big.ptrs, big.ws, big.hs, o, c, host_images=host, pitches=pitches)
        return enc.encode_images_packed(big.ptrs, big.ws, big.hs, o, c, host_images=host, pitches=pitches, fmt="GRAY")

    total_want = sum(len(x) for x in big.want)
    buf, bptr = pinned_empty(total_want + 64)
    try:
        buf[:] = 0
        offs, sizes, total = call(bptr, buf.size)
        assert sizes == [len(x) for x in big.want] and total == total_want
        assert offs == [sum(sizes[:i]) for i in range(n)]
        bad = [i for i in range(n) if buf[offs[i]: offs[i] + sizes[i]].tobytes() != big.want[i]]
        assert not bad, f"files differ: {[(i, big.ws[i], big.hs[i]) for i in bad]}"
        assert call(None, 0) == (offs, sizes, total)
        with pytest.raises(JpgencError) as e:
            call(bptr, total - 1)
        assert e.value.code == ERR_CAPACITY
    finally:
        pinned_free(bptr)


@pytest.mark.gpu
@pytest.mark.parametrize("planar", [False, True])
@pytest.mark.parametrize("host", [False, True])
def test_tiles_of_one_image(encoder, oracle, planar, host):
    big = BigImage(encoder, oracle, planar, host=host)
    try:
        assert len(big.ws) == 16 * 12
        _check_packed(encoder, big, planar, host=host)
    finally:
        big.free()


@pytest.mark.gpu
@pytest.mark.parametrize("planar", [False, True])
@pytest.mark.parametrize("host", [False, True])
def test_many_passes_and_refused_passes(oracle, monkeypatch, planar, host):
    """tiles with a ragged pitch cut into many passes over several slots; JPGENC_RAW_GUESS_PER_BLOCK=0 makes every first pass
    reserve too little scan space, so it is refused on the device and its entropy stage re-run"""
    from jpgenc_b200.capi import Encoder
    monkeypatch.setenv("JPGENC_FRAMES_PER_PASS", "5")
    monkeypatch.setenv("JPGENC_SLOTS", "3")
    enc = Encoder(0)
    try:
        big = BigImage(enc, oracle, planar, W=1000, H=600, T=96, host=host, pitch=1000 + 13, tiles=24)
        try:
            _check_packed(enc, big, planar, host=host)
            monkeypatch.setenv("JPGENC_RAW_GUESS_PER_BLOCK", "0")
            _check_packed(enc, big, planar, host=host)
        finally:
            big.free()
    finally:
        enc.close()


def _graph_cycle():
    """One device buffer bound alternately as tight RGB, GRAY and planar RGB (same first pointer, same size), each twice in a row
    so that the phases are captured as graphs and then met again under another layout; every file is checked.  The planar
    binds differ only in their G and B planes."""
    from jpgenc_b200.capi import Encoder
    from oracle.pyoracle import Oracle
    W, H = 200, 120
    raw = np.random.default_rng(4).integers(0, 256, size=W * H * 3, dtype=np.uint8)
    n = W * H
    planes = raw.reshape(3, H, W)
    cases = {
        "RGB": (lambda e, d: e.bind_device_rgb(d, W, H), raw.reshape(H, W, 3)),
        "GRAY": (lambda e, d: e.bind_device_image(d, W, H, 0, "GRAY"), as_rgb(planes[0])),
        "planar": (lambda e, d: e.bind_device_planar(d, d + n, d + 2 * n, W, H), planes.transpose(1, 2, 0)),
        "planar2": (lambda e, d: e.bind_device_planar(d, d + 2 * n, d + n, W, H), planes[[0, 2, 1]].transpose(1, 2, 0)),
    }
    oracle = Oracle()
    want = {k: oracle.encode_rgb(np.ascontiguousarray(v)) for k, (_, v) in cases.items()}
    enc = Encoder(0)
    d = enc.dev_alloc(raw.nbytes)
    try:
        enc.h2d(d, raw)
        for rep in range(3):
            for name, (bind, _) in cases.items():
                for _ in range(2):
                    bind(enc, d)
                    assert _encode_bound(enc, len(want[name]) + 4096) == want[name], f"{name}, round {rep}"
    finally:
        enc.dev_free(d)
        enc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("graphs", ["1", "0"])
def test_graph_cache_keys_on_grey_and_planes(graphs):
    # JPGENC_GRAPHS is read once per process: each setting runs in a process of its own
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, JPGENC_GRAPHS=graphs,
               PYTHONPATH=os.pathsep.join([root, os.path.dirname(os.path.abspath(__file__))]))
    r = subprocess.run([sys.executable, "-c", "import test_planar_gray as t; t._graph_cycle()"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_argument_errors(encoder):
    from jpgenc_b200.capi import ERR_ARG, JpgencError
    d = encoder.dev_alloc(48 * 32 * 3)
    try:
        assert encoder.encode_images_packed_planar([], [], [], None, 0) == ([], [], 0)      # n = 0 touches nothing
        bad = [lambda f=f: encoder.bind_device_image(d, 48, 32, 0, f) for f in range(4, 16)]  # unknown formats: 4 .. 15
        bad += [lambda f=f: encoder.encode_images_packed([d], [48], [32], None, 0, pitches=[0], fmt=f) for f in (4, 15, 17)]
        bad += [
            lambda: encoder.bind_device_image(d, 48, 32, 47, "GRAY"),                        # pitch below the row size
            lambda: encoder.bind_device_planar(d, 0, d, 48, 32),                             # null plane
            lambda: encoder.bind_device_planar(d, d, d, 48, 32, 47),
            lambda: encoder.bind_device_planar(d, d, d, 0, 32),
            lambda: encoder.bind_device_planar(d, d, d, 48, 70000),
            lambda: encoder.encode_images_packed_planar([d, d, 0], [48], [32], None, 0),
            lambda: encoder.encode_images_packed_planar([d] * 6, [48, 16], [32, 8], None, 0, pitches=[0, 15]),
            lambda: encoder.encode_images_packed_planar([d] * 3, [65536], [8], None, 0),
        ]
        for k, call in enumerate(bad):
            with pytest.raises(JpgencError) as e:
                call()
            assert e.value.code == ERR_ARG, k
        lib = encoder.lib
        assert lib.jpgenc_encode_planar(encoder.h, d, None, d, 48, 32, 0, 255, None, 0, None) == ERR_ARG
        assert lib.jpgenc_encode_images_packed_planar(encoder.h, 1, None, 1, None, None, None, 255, None, 0, None, None, None) == ERR_ARG
    finally:
        encoder.dev_free(d)


# ---- torch tensors ------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_tensors_on_the_gpu(encoder, oracle):
    import torch
    rgb = synth_rgb(333, 211, 8)
    chw = torch.from_numpy(np.ascontiguousarray(rgb.transpose(2, 0, 1))).cuda(0)
    want = oracle.encode_rgb(rgb)
    crop = rgb[17:190, 5:300]
    grey = grey_of(rgb)
    want_grey = oracle.encode_rgb(as_rgb(grey))
    g = torch.from_numpy(grey).cuda(0)
    assert encoder.encode_tensor(chw) == want
    assert encoder.stats().refined_blocks > 0
    assert encoder.encode_tensor(chw[:, 17:190, 5:300]) == oracle.encode_rgb(np.ascontiguousarray(crop))
    assert encoder.encode_tensor(chw.flip(0).contiguous(), order="BGR") == want
    assert encoder.encode_tensor(chw.permute(1, 2, 0).contiguous().permute(2, 0, 1)) == want                # channels_last
    assert encoder.encode_tensor(chw.permute(1, 2, 0).flip(2).contiguous(), order="BGR") == want
    rgba = torch.cat([chw.permute(1, 2, 0), torch.full((211, 333, 1), 7, dtype=torch.uint8, device="cuda:0")], 2).contiguous()
    assert encoder.encode_tensor(rgba) == want
    assert encoder.encode_tensor(g) == want_grey
    assert encoder.encode_tensor(g[None]) == want_grey
    assert encoder.encode_tensor(g.expand(3, 211, 333)) == want_grey
    # several tensors of one kind and different sizes through one call
    assert encoder.encode_tensors([chw, chw[:, 17:190, 5:300], chw[:, :9, :17]]) == [
        want, oracle.encode_rgb(np.ascontiguousarray(crop)), oracle.encode_rgb(np.ascontiguousarray(rgb[:9, :17]))]
    assert encoder.encode_tensors([]) == []
    with pytest.raises(ValueError):
        encoder.encode_tensors([chw, g])                                                       # two layout kinds
    with pytest.raises(ValueError):
        encoder.encode_tensors([chw, chw.cpu()])                                               # CPU and CUDA mixed
    with pytest.raises(ValueError):
        encoder.encode_tensor(chw.float())
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            encoder.encode_tensor(chw.cuda(1))


@pytest.mark.gpu
def test_tensors_on_the_cpu(encoder, oracle):
    import torch
    rgb = synth_rgb(640, 360, 12)
    want = oracle.encode_rgb(rgb)
    chw = torch.from_numpy(np.ascontiguousarray(rgb.transpose(2, 0, 1)))
    assert encoder.encode_tensor(chw) == want
    assert encoder.encode_tensor(torch.from_numpy(rgb)) == want
    assert encoder.encode_tensors([chw[:, 10:100, 20:300], chw]) == [oracle.encode_rgb(np.ascontiguousarray(rgb[10:100, 20:300])), want]
    grey = grey_of(rgb)
    assert encoder.encode_tensor(torch.from_numpy(grey)[:, 3:]) == oracle.encode_rgb(as_rgb(np.ascontiguousarray(grey[:, 3:])))


@pytest.mark.gpu
def test_tensor_written_on_another_stream(encoder, oracle):
    """the tensor is filled by work queued on a non-default current stream right before the call: the encoder must read it only
    after that work"""
    import torch
    rgb = synth_rgb(1920, 1080, 13)
    src = torch.from_numpy(np.ascontiguousarray(rgb.transpose(2, 0, 1))).cuda(0)
    dst = torch.zeros_like(src)
    s = torch.cuda.Stream(0)
    with torch.cuda.stream(s):
        torch.cuda._sleep(20_000_000)                                                          # the copy below starts late
        dst.copy_(src)
        got = encoder.encode_tensor(dst)
    assert got == oracle.encode_rgb(rgb)


# ---- layouts (no GPU) -----------------------------------------------------------------------------------------------------------

def test_tensor_layout_accepts():
    import torch
    t = torch.zeros((3, 40, 50), dtype=torch.uint8)
    base = t.data_ptr()
    assert tensor_layout(t) == ("planar", (base, base + 2000, base + 4000), 50, 40, 50)
    assert tensor_layout(t, "BGR") == ("planar", (base + 4000, base + 2000, base), 50, 40, 50)
    c = t[:, 5:30, 7:20]
    assert tensor_layout(c) == ("planar", (base + 257, base + 2257, base + 4257), 13, 25, 50)
    cl = t.permute(1, 2, 0).contiguous().permute(2, 0, 1)      # channels_last: strides (1, 3W, 3)
    assert tensor_layout(cl) == ("RGB", (cl.data_ptr(),), 50, 40, 150)
    assert tensor_layout(cl, "BGR")[0] == "BGR"
    hwc = torch.zeros((40, 50, 4), dtype=torch.uint8)
    assert tensor_layout(hwc) == ("RGBA", (hwc.data_ptr(),), 50, 40, 200)
    assert tensor_layout(hwc[3:9, 2:7], "BGR") == ("BGRA", (hwc.data_ptr() + 3 * 200 + 8,), 5, 6, 200)
    g = torch.zeros((40, 50), dtype=torch.uint8)
    assert tensor_layout(g) == ("GRAY", (g.data_ptr(),), 50, 40, 50)
    assert tensor_layout(g[None]) == ("GRAY", (g.data_ptr(),), 50, 40, 50)
    assert tensor_layout(g.expand(3, 40, 50)) == ("GRAY", (g.data_ptr(),), 50, 40, 50)
    assert tensor_layout(g[2:5, 1:9]) == ("GRAY", (g.data_ptr() + 101,), 8, 3, 50)
    assert tensor_layout(g[:1]) == ("GRAY", (g.data_ptr(),), 50, 1, 50)


def test_tensor_layout_refuses():
    import torch
    t = torch.zeros((3, 40, 50), dtype=torch.uint8)
    bad = [
        t.float(),                                               # not uint8
        t[:, :, ::2],                                            # column stride 2
        t.transpose(1, 2),                                       # (3, W, H) view: columns are not contiguous
        torch.zeros((2, 40, 50), dtype=torch.uint8),             # two channels
        torch.zeros((40, 50, 2), dtype=torch.uint8),
        torch.zeros((40, 50, 3), dtype=torch.uint8)[:, ::2],     # pixel stride 6
        torch.zeros((40, 50, 4), dtype=torch.uint8)[:, :, :3],   # 3 channels 4 bytes apart
        torch.zeros((4, 3, 40, 50), dtype=torch.uint8),          # a batch dimension
        torch.zeros((50,), dtype=torch.uint8),
        torch.zeros((0, 50), dtype=torch.uint8),
        np.zeros((40, 50), np.uint8),                            # not a tensor
    ]
    for k, x in enumerate(bad):
        with pytest.raises(ValueError):
            tensor_layout(x)
            pytest.fail(f"case {k} accepted")
    with pytest.raises(ValueError):
        tensor_layout(t, "GBR")


def test_grey_image_layout():
    a = np.zeros((40, 56), np.uint8)
    assert image_layout(a, "GRAY") == (a.ctypes.data, 56, 40, 56)
    assert image_layout(a[3:9, 5:20], "GRAY") == (a.ctypes.data + 3 * 56 + 5, 15, 6, 56)
    for bad in (a[:, ::2], a[None], a.astype(np.uint16), a.T, np.zeros((0, 4), np.uint8), np.zeros((4, 5, 1), np.uint8)):
        with pytest.raises(ValueError):
            image_layout(bad, "GRAY")
