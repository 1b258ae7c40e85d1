"""Pixels with a row pitch and in BGR, RGBA and BGRA order: jpgenc_bind_device_image, jpgenc_encode_image and
jpgenc_encode_images_packed_layout.  Every file must be byte-identical to the oracle's (or, for images the oracle would be slow
on, to jpgenc_encode_rgb) on the tight RGB copy of the same pixels.  The ignored 4th byte and the bytes between rows are random,
so reading either would change the file."""
import os
import subprocess
import sys

import numpy as np
import pytest

from jpgenc_b200.synth import noise_rgb, ppm_p6_bytes, synth_rgb

FORMATS = ["RGB", "BGR", "RGBA", "BGRA"]
BPP = {"RGB": 3, "BGR": 3, "RGBA": 4, "BGRA": 4}
SIZES = [(1, 1), (17, 9), (208, 120), (1000, 667), (1920, 1080)]


def tight_pitch(w, fmt):
    return w * BPP[fmt]


def pitch_kinds(w, fmt):
    """tight; a multiple of 16 above the row (the bulk-copy / vector path where the width allows it); tight + 3 (clamped loads)"""
    t = tight_pitch(w, fmt)
    return {"tight": t, "pitch16": (t + 15) // 16 * 16 + 16, "pitch+3": t + 3}


def layout_bytes(rgb, fmt, pitch, seed, offset=0):
    """rgb (H, W, 3) -> (buffer, view): a uint8 buffer of offset + H * pitch random bytes holding the pixels in format `fmt`
    with rows `pitch` bytes apart from byte `offset` on, and the (H, W, C) view of them"""
    h, w, _ = rgb.shape
    bpp = BPP[fmt]
    rng = np.random.default_rng(seed)
    buf = rng.integers(0, 256, size=offset + h * pitch, dtype=np.uint8)
    view = np.lib.stride_tricks.as_strided(buf[offset:], shape=(h, w, bpp), strides=(pitch, bpp, 1))
    px = rgb[:, :, ::-1] if fmt.startswith("BGR") else rgb
    view[:, :, :3] = px
    return buf, view


def _image(w, h, k):
    return noise_rgb(w, h, k) if k % 3 == 0 else synth_rgb(w, h, k)


@pytest.fixture(scope="module")
def sized(oracle):
    """one synthetic image per size of SIZES with the oracle's file"""
    imgs = [synth_rgb(w, h, 11 + k) for k, (w, h) in enumerate(SIZES)]
    return imgs, [oracle.encode_rgb(a) for a in imgs]


def _encode_bound(enc, cap):
    out = np.empty(cap, np.uint8)
    return out[: enc.encode_bound(out)].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FORMATS)
def test_single_device_images(encoder, sized, fmt):
    imgs, want = sized
    for kind in ("tight", "pitch16", "pitch+3"):
        for offset in (0, 1):
            refined = 0
            for k, (rgb, ref) in enumerate(zip(imgs, want)):
                h, w, _ = rgb.shape
                pitch = pitch_kinds(w, fmt)[kind]
                buf, _ = layout_bytes(rgb, fmt, pitch, seed=k, offset=offset)
                d = encoder.dev_alloc(buf.nbytes + 16)
                try:
                    encoder.h2d(d, buf)
                    encoder.bind_device_image(d + offset, w, h, pitch, fmt)
                    got = _encode_bound(encoder, len(ref) + 4096)
                    refined += encoder.stats().refined_blocks
                finally:
                    encoder.dev_free(d)
                assert got == ref, f"{fmt} {w}x{h} pitch {pitch} ({kind}) offset {offset}"
            assert refined > 0, "no block took the FP64 refinement: its pixel gather was not exercised"


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FORMATS)
def test_host_images_in_several_bands(encoder, fmt):
    """jpgenc_encode_image of a pitched host view large enough for several upload bands (>= 8 MB each)"""
    rgb = synth_rgb(4000, 3000, 5)
    want = encoder.encode_rgb(rgb)
    pitch = tight_pitch(4000, fmt) + 40
    _, view = layout_bytes(rgb, fmt, pitch, seed=3)
    assert encoder.encode_image(view, fmt) == want
    assert encoder.stats().refined_blocks > 0


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FORMATS)
def test_maxval_below_255(encoder, oracle, fmt):
    """the 4th byte (255) and the pitch gap (bytes above maxval) are not samples; a colour sample above maxval is refused"""
    from jpgenc_b200.capi import ERR_FORMAT, JpgencError
    rgb = (synth_rgb(67, 45, 2).astype(np.uint16) * 100 // 255).astype(np.uint8)
    want = oracle.encode_ppm(ppm_p6_bytes(rgb, 100))
    pitch = tight_pitch(67, fmt) + 5
    buf, view = layout_bytes(rgb, fmt, pitch, seed=1)
    buf[:] = 255
    view[:, :, :3] = rgb[:, :, ::-1] if fmt.startswith("BGR") else rgb
    assert encoder.encode_image(view, fmt, maxval=100) == want
    assert encoder.encode_images([view, view[3:20, 5:40]], maxval=100, fmt=fmt) == [
        want, oracle.encode_ppm(ppm_p6_bytes(np.ascontiguousarray(rgb[3:20, 5:40]), 100))]
    view[7, 9, 1] = 101
    for call in (lambda: encoder.encode_image(view, fmt, maxval=100), lambda: encoder.encode_images([view], maxval=100, fmt=fmt)):
        with pytest.raises(JpgencError) as e:
            call()
        assert e.value.code == ERR_FORMAT


def _tiles(W, H, T):
    return [(x, y, min(T, W - x), min(T, H - y)) for y in range(0, H, T) for x in range(0, W, T)]


def _check_packed(enc, ptrs, ws, hs, pitches, fmt, want, host=False):
    """as tests/test_mixed_size_batches.py: contiguous files in input order, each the expected one; sizes-only gives the same
    offsets and sizes; a buffer one byte short is refused"""
    from jpgenc_b200.capi import ERR_CAPACITY, JpgencError, pinned_empty, pinned_free
    total_want = sum(len(x) for x in want)
    buf, bptr = pinned_empty(total_want + 64)
    kw = dict(host_images=host, pitches=pitches, fmt=fmt)
    try:
        buf[:] = 0
        offs, sizes, total = enc.encode_images_packed(ptrs, ws, hs, bptr, buf.size, **kw)
        assert sizes == [len(x) for x in want] and total == total_want
        assert offs == [sum(sizes[:i]) for i in range(len(ptrs))]
        bad = [i for i in range(len(ptrs)) if buf[offs[i]: offs[i] + sizes[i]].tobytes() != want[i]]
        assert not bad, f"files differ: {[(i, ws[i], hs[i]) for i in bad]}"
        assert enc.encode_images_packed(ptrs, ws, hs, None, 0, **kw) == (offs, sizes, total)
        with pytest.raises(JpgencError) as e:
            enc.encode_images_packed(ptrs, ws, hs, bptr, total - 1, **kw)
        assert e.value.code == ERR_CAPACITY
    finally:
        pinned_free(bptr)


class BigImage:
    """a W x H synthetic image in format `fmt` in one buffer (device, or pinned host) with rows `pitch` bytes apart, cut into
    T x T tiles plus the ragged right and bottom ones: pointers into the big image, and the oracle's file of every tile"""

    def __init__(self, enc, oracle, fmt, W=4000, H=3000, T=256, host=False, pitch=None, tiles=None):
        from jpgenc_b200.capi import pinned_empty
        self.enc, self.host = enc, host
        rgb = synth_rgb(W, H, 21)
        self.pitch = pitch or tight_pitch(W, fmt)
        buf, _ = layout_bytes(rgb, fmt, self.pitch, seed=7)
        if host:
            self.view, self.base = pinned_empty(buf.nbytes)
            self.view[:] = buf
        else:
            self.base = enc.dev_alloc(buf.nbytes)
            enc.h2d(self.base, buf)
        bpp = BPP[fmt]
        tl = _tiles(W, H, T)[:tiles]
        self.ptrs = [self.base + y * self.pitch + x * bpp for x, y, _, _ in tl]
        self.ws = [w for _, _, w, _ in tl]
        self.hs = [h for _, _, _, h in tl]
        self.want = [oracle.encode_rgb(np.ascontiguousarray(rgb[y: y + h, x: x + w])) for x, y, w, h in tl]

    def free(self):
        from jpgenc_b200.capi import pinned_free
        if self.host:
            pinned_free(self.base)
        else:
            self.enc.dev_free(self.base)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["RGB", "BGRA"])
@pytest.mark.parametrize("host", [False, True])
def test_tiles_of_one_image(encoder, oracle, fmt, host):
    big = BigImage(encoder, oracle, fmt, host=host)
    try:
        assert len(big.ptrs) == 16 * 12
        _check_packed(encoder, big.ptrs, big.ws, big.hs, [big.pitch] * len(big.ptrs), fmt, big.want, host=host)
    finally:
        big.free()


@pytest.mark.gpu
@pytest.mark.parametrize("per_pass", [1, 7])
@pytest.mark.parametrize("slots", [1, 3])
def test_many_passes_and_refused_passes(oracle, monkeypatch, per_pass, slots):
    """tiles with a ragged pitch cut into many passes over several slots; JPGENC_RAW_GUESS_PER_BLOCK=0 makes every first pass
    reserve too little scan space, so it is refused on the device and its entropy stage re-run"""
    from jpgenc_b200.capi import Encoder
    monkeypatch.setenv("JPGENC_FRAMES_PER_PASS", str(per_pass))
    monkeypatch.setenv("JPGENC_SLOTS", str(slots))
    enc = Encoder(0)
    try:
        big = BigImage(enc, oracle, "BGRA", W=1000, H=600, T=96, pitch=4000 + 12, tiles=24)
        try:
            args = (big.ptrs, big.ws, big.hs, [big.pitch] * len(big.ptrs), "BGRA", big.want)
            _check_packed(enc, *args)
            monkeypatch.setenv("JPGENC_RAW_GUESS_PER_BLOCK", "0")
            _check_packed(enc, *args)
        finally:
            big.free()
    finally:
        enc.close()


@pytest.mark.gpu
def test_tight_rgb_takes_the_existing_paths(oracle):
    """tight RGB through the layout call: equal sizes are jpgenc_encode_frames_packed (same files, same kernel launches), mixed
    sizes jpgenc_encode_images_packed"""
    from jpgenc_b200.capi import Encoder
    enc = Encoder(0)
    try:
        frames = [synth_rgb(320, 240, k) for k in range(9)]
        mixed = [_image(40 + 37 * k, 30 + 11 * k, k) for k in range(9)]
        want_f = [oracle.encode_rgb(a) for a in frames]
        want_m = [oracle.encode_rgb(a) for a in mixed]
        base = enc.dev_alloc(sum(a.nbytes + 256 for a in frames + mixed))
        try:
            ptrs, o = [], 0
            for a in frames + mixed:
                enc.h2d(base + o, a)
                ptrs.append(base + o)
                o += (a.nbytes + 255) // 256 * 256
            fp, mp = ptrs[:9], ptrs[9:]
            out = np.zeros(sum(len(x) for x in want_f + want_m) + 64, np.uint8)
            enc.encode_frames_packed(fp, 320, 240, out.ctypes.data, out.size)      # learns the scan reservation: no refused pass below
            n0 = enc.launch_count()
            r0 = enc.encode_frames_packed(fp, 320, 240, out.ctypes.data, out.size)
            n1 = enc.launch_count()
            r1 = enc.encode_images_packed(fp, [320] * 9, [240] * 9, out.ctypes.data, out.size, pitches=[0] * 9, fmt="RGB")
            n2 = enc.launch_count()
            assert r0 == r1 and n2 - n1 == n1 - n0
            assert [out[o: o + n].tobytes() for o, n in zip(r1[0], r1[1])] == want_f
            ws, hs = [a.shape[1] for a in mixed], [a.shape[0] for a in mixed]
            r2 = enc.encode_images_packed(mp, ws, hs, out.ctypes.data, out.size, pitches=[w * 3 for w in ws], fmt="RGB")
            assert [out[o: o + n].tobytes() for o, n in zip(r2[0], r2[1])] == want_m
            assert r2 == enc.encode_images_packed(mp, ws, hs, out.ctypes.data, out.size)
        finally:
            enc.dev_free(base)
    finally:
        enc.close()


def _graph_cycle():
    """One device buffer bound alternately as tight RGB, BGRA and pitched RGB (same pointer, same size), each twice in a row so
    that the phases are captured as graphs and then met again under another layout; every file is checked."""
    from jpgenc_b200.capi import Encoder
    from oracle.pyoracle import Oracle
    W, H = 200, 120
    raw = noise_rgb(W * 4, H, 4).reshape(-1)[: W * H * 4].copy()            # the bytes of a BGRA image
    bgra = raw.reshape(H, W, 4)
    as_layout = {
        ("RGB", 0): raw[: W * H * 3].reshape(H, W, 3),
        ("BGRA", 0): np.ascontiguousarray(bgra[:, :, 2::-1]),
        ("RGB", W * 4): np.ascontiguousarray(bgra.reshape(H, W * 4)[:, : W * 3].reshape(H, W, 3)),
    }
    oracle = Oracle()
    want = {k: oracle.encode_rgb(np.ascontiguousarray(v)) for k, v in as_layout.items()}
    enc = Encoder(0)
    d = enc.dev_alloc(raw.nbytes)
    try:
        enc.h2d(d, raw)
        for rep in range(3):
            for (fmt, pitch) in as_layout:
                for _ in range(2):
                    enc.bind_device_image(d, W, H, pitch, fmt)
                    got = _encode_bound(enc, len(want[fmt, pitch]) + 4096)
                    assert got == want[fmt, pitch], f"{fmt} pitch {pitch}, round {rep}"
    finally:
        enc.dev_free(d)
        enc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("graphs", ["1", "0"])
def test_graph_cache_keys_on_the_layout(graphs):
    # JPGENC_GRAPHS is read once per process: each setting runs in a process of its own
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, JPGENC_GRAPHS=graphs,
               PYTHONPATH=os.pathsep.join([root, os.path.dirname(os.path.abspath(__file__))]))
    r = subprocess.run([sys.executable, "-c", "import test_pixel_layouts as t; t._graph_cycle()"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_argument_errors(encoder, oracle):
    from jpgenc_b200.capi import ERR_ARG, JpgencError
    rgb = synth_rgb(48, 32, 3)
    want = oracle.encode_rgb(rgb)
    d = encoder.dev_alloc(rgb.nbytes)
    try:
        encoder.h2d(d, rgb)
        encoder.bind_device_rgb(d, 48, 32)
        assert encoder.encode_images_packed([], [], [], None, 0, pitches=[], fmt="BGRA") == ([], [], 0)   # n = 0 touches nothing
        assert _encode_bound(encoder, len(want) + 64) == want
        bad = [
            lambda: encoder.bind_device_image(d, 48, 32, 0, 4),                          # unknown format
            lambda: encoder.bind_device_image(d, 48, 32, 0, -1),
            lambda: encoder.bind_device_image(d, 48, 32, 48 * 4 - 1, "RGBA"),           # pitch below the row size
            lambda: encoder.bind_device_image(0, 48, 32, 0, "RGB"),                      # null pointer
            lambda: encoder.bind_device_image(d, 0, 32, 0, "RGB"),
            lambda: encoder.bind_device_image(d, 70000, 1, 0, "BGR"),
            lambda: encoder.encode_images_packed([d], [48], [32], None, 0, pitches=[0], fmt=9),
            lambda: encoder.encode_images_packed([d, d], [48, 16], [32, 8], None, 0, pitches=[0, 47], fmt="BGR"),
            lambda: encoder.encode_images_packed([d, 0], [48, 16], [32, 8], None, 0, pitches=None, fmt="BGR"),
        ]
        for k, call in enumerate(bad):
            with pytest.raises(JpgencError) as e:
                call()
            assert e.value.code == ERR_ARG, k
        lib = encoder.lib
        assert lib.jpgenc_encode_image(encoder.h, None, 48, 32, 0, 0, 255, None, 0, None) == ERR_ARG
        assert lib.jpgenc_encode_images_packed_layout(encoder.h, 1, None, 1, None, None, None, 0, 255, None, 0, None, None, None) == ERR_ARG
        with pytest.raises(ValueError):
            encoder.encode_image(np.zeros((4, 8, 3), np.uint8)[:, ::2], "RGB")         # strides (24, 6, 1): not a row-pitch layout
        with pytest.raises(ValueError):
            encoder.encode_image(np.zeros((4, 8, 3), np.uint8), "RGBA")
    finally:
        encoder.dev_free(d)
