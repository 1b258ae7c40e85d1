"""jpgenc_encode_images_packed: batches of images of individual sizes through the batched kernel pipeline.  Every file must be
byte-identical to encoding that image alone (the oracle, or jpgenc_encode_bound where the oracle would be slow)."""
import numpy as np
import pytest

from jpgenc_b200.synth import noise_rgb, synth_rgb

SIZES = [(1, 1), (15, 15), (16, 16), (17, 9), (208, 120), (101, 67), (1000, 667), (3001, 1203), (1920, 1080), (4096, 16), (16, 4096)]


def _image(w, h, k):
    return noise_rgb(w, h, k) if k % 3 == 0 else synth_rgb(w, h, k)


@pytest.fixture(scope="module")
def assorted(oracle):
    """44 images: every size of SIZES four times, contents alternating between the synthetic image and noise (noise gives
    FF-rich scans), with the oracle's files"""
    imgs = [_image(w, h, k) for k, (w, h) in enumerate(SIZES * 4)]
    return imgs, [oracle.encode_rgb(a) for a in imgs]


class DeviceImages:
    """the images in one device allocation, each at a 256-byte boundary plus `shift` bytes"""

    def __init__(self, enc, imgs, shift=0):
        self.enc = enc
        self.at, o = [], 0
        for a in imgs:
            self.at.append(o + shift)
            o += (a.nbytes + shift + 255) // 256 * 256
        self.base = enc.dev_alloc(o + 256)
        for a, at in zip(imgs, self.at):
            enc.h2d(self.base + at, a)
        self.ptrs = [self.base + at for at in self.at]

    def free(self):
        self.enc.dev_free(self.base)


def _dims(imgs):
    return [a.shape[1] for a in imgs], [a.shape[0] for a in imgs]


def _check_packed(enc, ptrs, imgs, want, host=False):
    """one call into a pinned buffer: contiguous files in input order, each the oracle's; sizes-only gives the same offsets
    and sizes; a buffer one byte short is refused"""
    from jpgenc_b200.capi import ERR_CAPACITY, JpgencError, pinned_empty, pinned_free
    ws, hs = _dims(imgs)
    total_want = sum(len(x) for x in want)
    buf, bptr = pinned_empty(total_want + 64)
    try:
        buf[:] = 0
        offs, sizes, total = enc.encode_images_packed(ptrs, ws, hs, bptr, buf.size, host_images=host)
        assert sizes == [len(x) for x in want] and total == total_want
        assert offs == [sum(sizes[:i]) for i in range(len(imgs))]
        bad = [i for i in range(len(imgs)) if buf[offs[i]: offs[i] + sizes[i]].tobytes() != want[i]]
        assert not bad, f"files differ: {[(i, ws[i], hs[i]) for i in bad]}"
        assert enc.encode_images_packed(ptrs, ws, hs, None, 0, host_images=host) == (offs, sizes, total)
        with pytest.raises(JpgencError) as e:
            enc.encode_images_packed(ptrs, ws, hs, bptr, total - 1, host_images=host)
        assert e.value.code == ERR_CAPACITY
    finally:
        pinned_free(bptr)


@pytest.mark.gpu
def test_assorted_sizes_device_host_and_unaligned(encoder, assorted):
    from jpgenc_b200.capi import pinned_empty, pinned_free
    imgs, want = assorted
    for shift in (0, 1):                                          # 1: every pointer off 16-byte alignment (clamped K1 loader)
        dev = DeviceImages(encoder, imgs, shift)
        try:
            _check_packed(encoder, dev.ptrs, imgs, want)
        finally:
            dev.free()
    total = sum(a.nbytes for a in imgs)
    host, hptr = pinned_empty(total)
    try:
        ptrs, o = [], 0
        for a in imgs:
            host[o: o + a.nbytes] = a.reshape(-1)
            ptrs.append(hptr + o)
            o += a.nbytes
        _check_packed(encoder, ptrs, imgs, want, host=True)
    finally:
        pinned_free(hptr)
    assert encoder.encode_images(imgs[:12]) == want[:12]         # the convenience form (pageable host arrays)


@pytest.mark.gpu
@pytest.mark.parametrize("per_pass", [1, 3, 7])
@pytest.mark.parametrize("slots", [1, 3])
def test_many_passes_on_several_slots(oracle, monkeypatch, assorted, per_pass, slots):
    """images cut into many passes rotating over several slots; JPGENC_RAW_GUESS_PER_BLOCK=0 makes every first pass reserve
    too little scan space, so it is refused on the device and its entropy stage re-run"""
    from jpgenc_b200.capi import Encoder
    imgs, want = assorted
    imgs, want = imgs[:22], want[:22]
    monkeypatch.setenv("JPGENC_FRAMES_PER_PASS", str(per_pass))
    monkeypatch.setenv("JPGENC_SLOTS", str(slots))
    enc = Encoder(0)
    try:
        dev = DeviceImages(enc, imgs)
        try:
            _check_packed(enc, dev.ptrs, imgs, want)
            monkeypatch.setenv("JPGENC_RAW_GUESS_PER_BLOCK", "0")
            _check_packed(enc, dev.ptrs, imgs, want)
        finally:
            dev.free()
    finally:
        enc.close()


@pytest.mark.gpu
def test_300_random_sizes_in_one_call(encoder, oracle):
    rng = np.random.default_rng(2026)
    dims = rng.integers(1, 701, size=(300, 2))
    imgs = [_image(int(w), int(h), k) for k, (w, h) in enumerate(dims)]
    want = [oracle.encode_rgb(a) for a in imgs]
    dev = DeviceImages(encoder, imgs)
    try:
        _check_packed(encoder, dev.ptrs, imgs, want)
    finally:
        dev.free()


@pytest.mark.gpu
def test_image_over_the_pass_budget_among_small_ones(encoder, oracle):
    """16384 x 16384 (268 Mpx) exceeds the pass pixel budget (256 Mpx) by itself, so it runs in a pass of its own between
    passes of small images; its file equals jpgenc_encode_bound of the same pixels"""
    W = H = 16384
    small = [_image(int(40 + 13 * k), int(30 + 7 * k), k) for k in range(20)]
    want_small = [oracle.encode_rgb(a) for a in small]
    big = encoder.dev_alloc(W * H * 3)
    dev = DeviceImages(encoder, small)
    try:
        encoder.synth_rgb(big, W, H, 9)
        encoder.bind_device_rgb(big, W, H)
        want_big = np.empty(W * H, np.uint8)
        want_big = want_big[: encoder.encode_bound(want_big)].tobytes()
        ptrs = dev.ptrs[:10] + [big] + dev.ptrs[10:]
        ws, hs = _dims(small)
        ws, hs = ws[:10] + [W] + ws[10:], hs[:10] + [H] + hs[10:]
        out = np.zeros(len(want_big) + sum(len(x) for x in want_small) + 64, np.uint8)
        offs, sizes, total = encoder.encode_images_packed(ptrs, ws, hs, out.ctypes.data, out.size)
        files = [out[o: o + n].tobytes() for o, n in zip(offs, sizes)]
        assert files[10] == want_big
        assert files[:10] + files[11:] == want_small
        assert total == sum(sizes)
    finally:
        dev.free()
        encoder.dev_free(big)


@pytest.mark.gpu
def test_alternating_calls_on_one_context(oracle, assorted):
    """mixed call -> equal frames -> one image -> mixed call: no geometry, table or scan reservation of one call leaks into
    the next"""
    from jpgenc_b200.capi import Encoder
    imgs, want = assorted
    enc = Encoder(0)
    try:
        dev = DeviceImages(enc, imgs)
        frames = [synth_rgb(320, 240, k) for k in range(9)]
        fwant = [oracle.encode_rgb(f) for f in frames]
        fdev = DeviceImages(enc, frames)
        try:
            for rep in range(2):
                _check_packed(enc, dev.ptrs, imgs, want)
                out = np.zeros(sum(len(x) for x in fwant) + 64, np.uint8)
                offs, sizes, total = enc.encode_frames_packed(fdev.ptrs, 320, 240, out.ctypes.data, out.size)
                assert [out[o: o + n].tobytes() for o, n in zip(offs, sizes)] == fwant
                assert enc.encode_rgb(imgs[5]) == want[5]
                _check_packed(enc, dev.ptrs[::-1], imgs[::-1], want[::-1])
        finally:
            dev.free()
            fdev.free()
    finally:
        enc.close()


@pytest.mark.gpu
def test_argument_errors(encoder, oracle):
    from jpgenc_b200.capi import ERR_ARG, ERR_FORMAT, JpgencError
    rgb = synth_rgb(48, 32, 3)
    want = oracle.encode_rgb(rgb)
    d = encoder.dev_alloc(rgb.nbytes)
    try:
        encoder.h2d(d, rgb)
        encoder.bind_device_rgb(d, 48, 32)
        assert encoder.encode_images_packed([], [], [], None, 0) == ([], [], 0)       # touches nothing: the bound image stays
        out = np.empty(len(want) + 64, np.uint8)
        assert out[: encoder.encode_bound(out)].tobytes() == want
        with pytest.raises(JpgencError) as e:
            encoder.encode_images_packed([d, d], [48, 0], [32, 32], None, 0)
        assert e.value.code == ERR_ARG
        with pytest.raises(JpgencError) as e:
            encoder.encode_images_packed([d], [70000], [1], None, 0)
        assert e.value.code == ERR_ARG
        with pytest.raises(JpgencError) as e:
            encoder.encode_images_packed([d], [48], [32], None, 0, maxval=256)
        assert e.value.code == ERR_ARG
        small = np.full((3, 5, 3), 100, np.uint8)
        small[1, 2, 0] = 101
        big = np.full((4, 7, 3), 7, np.uint8)
        with pytest.raises(JpgencError) as e:
            encoder.encode_images_packed([big.ctypes.data, small.ctypes.data], [7, 5], [4, 3], None, 0, maxval=100, host_images=True)
        assert e.value.code == ERR_FORMAT
        small[1, 2, 0] = 100
        from jpgenc_b200.synth import ppm_p6_bytes
        assert encoder.encode_images([big, small], maxval=100) == [oracle.encode_ppm(ppm_p6_bytes(a, 100)) for a in (big, small)]
    finally:
        encoder.dev_free(d)
