"""Parity of the CUDA path against the oracle, through the C-ABI.  Run with `-m gpu` on a B200.

Bar: bit-exact everywhere (integer/byte work; the FP32 DCT fast path is backed by exact FP64 refinement, so the
quantised coefficients must equal the reference's with ZERO mismatches, not +-1)."""
import io
import os

import numpy as np
import pytest

from conftest import random_symbol_stats, table_fields
from jpgenc_b200.synth import noise_rgb, ppm_p6_bytes, synth_rgb

pytestmark = pytest.mark.gpu


def _images():
    flat = np.full((64, 64, 3), 200, np.uint8)
    stripes = np.zeros((48, 80, 3), np.uint8)
    stripes[:, ::2] = 255
    half = np.zeros((32, 32, 3), np.uint8)
    half[...] = (128, 127, 129)
    return {
        "synth_512": (synth_rgb(512, 512, 0), 255),
        "noise_256": (noise_rgb(256, 256, 1), 255),
        "odd_203x117": (synth_rgb(203, 117, 3), 255),
        "odd_noise_100x37": (noise_rgb(100, 37, 2), 255),
        "one_pixel": (noise_rgb(1, 1, 3), 255),
        "tiny_5x3": (synth_rgb(5, 3, 1), 255),
        "w16_h17": (noise_rgb(16, 17, 4), 255),
        "w33_h16": (noise_rgb(33, 16, 5), 255),
        "wide_2000x16": (synth_rgb(2000, 16, 6), 255),
        "tall_16x1000": (synth_rgb(16, 1000, 7), 255),
        "flat": (flat, 255),
        "stripes": (stripes, 255),
        "mid_grey": (half, 255),
        "black": (np.zeros((40, 40, 3), np.uint8), 255),
        "white": (np.full((40, 40, 3), 255, np.uint8), 255),
        "maxval15": (noise_rgb(64, 48, 5) >> 4, 15),
        "maxval100": (noise_rgb(50, 50, 6) % 101, 100),
        # the largest dimensions a baseline JPEG can declare (SOF0 holds 16-bit sizes): 4096 MCUs in a row / in a column
        "max_width_65535x16": (synth_rgb(65535, 16, 8), 255),
        "max_height_16x65535": (synth_rgb(16, 65535, 9), 255),
        # 129 MCUs per row: four full strips (tensor store) and a partial one (per-thread copy-out) in every MCU row
        "strips_2064x48": (noise_rgb(2064, 48, 10), 255),
    }


IMAGES = _images()


@pytest.mark.parametrize("name", list(IMAGES))
def test_k1_coefficients_bit_exact(encoder, oracle, name):
    rgb, maxval = IMAGES[name]
    ref = oracle.forward(rgb, maxval)
    encoder.upload_rgb(rgb, maxval)
    encoder.color_dct_quant()
    got = encoder.get_coefficients()
    mismatches = int(np.count_nonzero(got != ref))
    assert mismatches == 0, f"{mismatches} of {ref.size} coefficients differ (max |d| {np.abs(got.astype(int) - ref).max()})"


@pytest.mark.parametrize("name", list(IMAGES))
def test_entropy_stages_bit_exact_on_reference_coefficients(encoder, oracle, name):
    """K2, host table build, K3, K4 fed with the ORACLE's coefficient array (independent of K1)."""
    rgb, maxval = IMAGES[name]
    h, w, _ = rgb.shape
    _, _, mw, mh = oracle.geometry(w, h)
    d = oracle.forward_planes(rgb, maxval)
    encoder.set_coefficients(d["q_y"], d["q_cb"], d["q_cr"])          # the reference's planar int32 arrays
    ref = oracle.planes_to_mcu(d["q_y"], d["q_cb"], d["q_cr"])
    assert np.array_equal(encoder.get_coefficients(), ref)
    count, first = encoder.symbol_stats()
    ocount, ofirst = oracle.symbol_stats(ref, mw, mh)
    assert np.array_equal(count, ocount)
    assert np.array_equal(first, ofirst)
    tabs = encoder.build_huffman(count, first)
    otabs, _, onbits, ostuffed = oracle.entropy_encode(ref, mw, mh)
    for t in range(4):
        assert table_fields(tabs[t]) == table_fields(otabs[t]), f"table {t}"
    n = encoder.entropy_encode(tabs)
    scan = encoder.download_scan()
    assert n == ostuffed.size and np.array_equal(scan, ostuffed)
    assert encoder.stats().scan_bits + (-encoder.stats().scan_bits) % 8 == onbits


@pytest.mark.parametrize("name", list(IMAGES))
def test_whole_file_byte_identical(encoder, oracle, name):
    rgb, maxval = IMAGES[name]
    mine = encoder.encode_rgb(rgb, maxval)
    from jpgenc_b200.synth import ppm_p6_bytes
    theirs = oracle.encode_ppm(ppm_p6_bytes(rgb, maxval))
    assert mine == theirs


def test_golden_files_from_the_reference(encoder, golden, tmp_path):
    """committed outputs of the compiled reference: PPM file in -> JPEG file out through jpgenc_encode_ppm_file"""
    for name in [str(n) for n in golden["names"]]:
        src, dst = tmp_path / f"{name}.ppm", tmp_path / f"{name}.jpg"
        src.write_bytes(golden[f"{name}/ppm"].tobytes())
        encoder.encode_ppm_file(str(src), str(dst))
        assert dst.read_bytes() == golden[f"{name}/jpg"].tobytes(), name


def test_pr1_image_pin(encoder):
    """config 0: the 512x512 synthetic; sha256 pinned by the reference build (SURVEY.md 8c)"""
    import hashlib
    jpg = encoder.encode_rgb(synth_rgb(512, 512, 0))
    assert len(jpg) == 12323
    assert hashlib.sha256(jpg).hexdigest() == "ceedd1ecae8dbeaf3620f9256abf57c9061167b65f5d574426739cacd82a3c20"


def test_error_behaviour(encoder, tmp_path):
    from jpgenc_b200.capi import ERR_ARG, ERR_FORMAT, ERR_IO, Encoder, JpgencError
    with pytest.raises(JpgencError) as e:
        encoder.encode_ppm_file(str(tmp_path / "missing.ppm"), str(tmp_path / "o.jpg"))
    assert e.value.code == ERR_IO                                   # reference: runtime_error("Failed to open ...")
    bad = tmp_path / "bad.ppm"
    bad.write_bytes(b"P5\n2 2\n255\n....")
    with pytest.raises(JpgencError) as e:
        encoder.encode_ppm_file(str(bad), str(tmp_path / "o.jpg"))
    assert e.value.code == ERR_FORMAT and "P3 and P6" in str(e.value)
    # a sample above maxval: refused (P6 bytes, P3 numbers, host pixels handed to the library directly)
    over6 = tmp_path / "over6.ppm"
    over6.write_bytes(b"P6\n2 2\n63\n" + bytes([1, 2, 3, 4, 5, 6, 7, 8, 200, 9, 10, 11]))
    over3 = tmp_path / "over3.ppm"
    over3.write_bytes(b"P3\n2 1\n100\n1 2 3 4 300 6\n")
    for f in (over6, over3):
        with pytest.raises(JpgencError) as e:
            encoder.encode_ppm_file(str(f), str(tmp_path / "o.jpg"))
        assert e.value.code == ERR_FORMAT, f
    with pytest.raises(JpgencError) as e:
        encoder.encode_rgb(np.full((16, 16, 3), 70, np.uint8), 63)
    assert e.value.code == ERR_FORMAT
    fresh = Encoder(0)
    with pytest.raises(JpgencError) as e:
        fresh.color_dct_quant()                                     # stage called out of pipeline order
    assert e.value.code == ERR_ARG
    fresh.close()


def test_custom_quant_tables(encoder, oracle):
    rgb = noise_rgb(64, 64, 8)
    qy = np.clip(oracle.qy.astype(int) // 4, 1, 255).astype(np.uint8)
    qc = np.ones(64, np.uint8)
    try:
        encoder.set_qtables(qy, qc)
        encoder.upload_rgb(rgb)
        encoder.color_dct_quant()
        assert np.array_equal(encoder.get_coefficients(), oracle.forward(rgb, 255, qy, qc))
    finally:
        encoder.set_qtables(oracle.qy, oracle.qc)


def test_idempotent_and_deterministic(encoder):
    rgb = noise_rgb(320, 240, 12)
    a = encoder.encode_rgb(rgb)
    b = encoder.encode_rgb(synth_rgb(64, 64, 1))
    c = encoder.encode_rgb(rgb)
    assert a == c and a != b


def test_decoded_image_is_close(encoder):
    PIL = pytest.importorskip("PIL.Image")
    rgb = synth_rgb(640, 360, 4)
    img = np.asarray(PIL.open(io.BytesIO(encoder.encode_rgb(rgb))).convert("RGB")).astype(float)
    assert img.shape == rgb.shape and np.abs(img - rgb).mean() < 12


def test_microbench_blocks_bit_exact(encoder, oracle):
    """config 1 at a size the oracle finishes in seconds"""
    nb = 1 << 14
    d_in, d_out = encoder.dev_alloc(nb * 256), encoder.dev_alloc(nb * 128)
    try:
        encoder.synth_blocks(d_in, nb)
        refined = encoder.dct_quant_blocks(d_in, d_out, nb, oracle.qy)
        x = np.empty((nb, 64), np.float32)
        y = np.empty((nb, 64), np.int16)
        encoder.d2h(x, d_in)
        encoder.d2h(y, d_out)
        zz = np.array([oracle.zigzag_index(i) for i in range(64)])
        i = np.arange(nb * 64, dtype=np.uint64)
        v = i ^ (i >> np.uint64(16)); v = (v * np.uint64(0x7FEB352D)) & np.uint64(0xFFFFFFFF)
        v ^= v >> np.uint64(15); v = (v * np.uint64(0x846CA68B)) & np.uint64(0xFFFFFFFF); v ^= v >> np.uint64(16)
        assert np.array_equal(x.reshape(-1), ((v & np.uint64(255)).astype(np.int64) - 128).astype(np.float32))
        bad = 0
        for b in range(0, nb, 7):
            q = oracle.quantize(oracle.dct(x[b].astype(np.float64).reshape(8, 8)), oracle.qy).reshape(64)[zz]
            bad += int(np.count_nonzero(q != y[b]))
        assert bad == 0
        assert 0 < refined < nb // 4
    finally:
        encoder.dev_free(d_in)
        encoder.dev_free(d_out)


def test_device_generator_matches_host_generator(encoder):
    w, h = 300, 200
    d = encoder.dev_alloc(w * h * 3)
    try:
        encoder.synth_rgb(d, w, h, 5)
        out = np.empty((h, w, 3), np.uint8)
        encoder.d2h(out, d)
        assert np.array_equal(out, synth_rgb(w, h, 5))
    finally:
        encoder.dev_free(d)


# ---- full BASELINE sizes: size-independent properties -------------------------------------------------------
@pytest.mark.parametrize("w,h", [(3840, 2160), (16384, 16384)])
def test_full_size_properties(encoder, oracle, w, h):
    """configs 2 and 3.  (a) K1 on random MCU rows == oracle; (b) the device scan == the oracle's entropy coder run on
    the DEVICE's coefficients (table build, Huffman pack, padding, stuffing at full size); (c) JPEG size AND SHA-256 ==
    the pins the compiled reference produced for these files (SURVEY.md 8(c)): the whole file is byte-identical to the
    reference's, not only the sampled rows; (d) FF count consistent with the stuffed length."""
    import hashlib
    pins = {(3840, 2160): 339813, (16384, 16384): 10898928}
    sha = {(3840, 2160): "6a1f9d77ee80e71282e563eda740758fc48cc0962e2f7acaeba6318855a7435d",
           (16384, 16384): "6eddc10c5db418a6be99f0d61ba5ee3643c0c8e93994e45131e868f54b2568fd"}
    d = encoder.dev_alloc(w * h * 3)
    try:
        encoder.synth_rgb(d, w, h, 0)
        encoder.bind_device_rgb(d, w, h)
        out = np.empty(pins[(w, h)] + 1024, np.uint8)
        n = encoder.encode_bound(out)
        assert n == pins[(w, h)]
        assert hashlib.sha256(out[:n].tobytes()).hexdigest() == sha[(w, h)]
        st = encoder.stats()
        coef = encoder.get_coefficients()
        mw, mh = st.mcu_w, st.mcu_h
        # (a)
        rng = np.random.default_rng(0)
        rows = sorted(set([0, mh - 1] + rng.integers(0, mh, 6).tolist()))
        for my in rows:
            band = synth_rgb(w, h, 0, rows=slice(my * 16, min(h, my * 16 + 16)))
            # the oracle needs the image rows at their true y positions: build a cropped image whose MCU row 0 is ours
            ref = oracle.forward(band, 255)
            assert np.array_equal(coef[my * mw:(my + 1) * mw], ref), f"MCU row {my}"
        # (b)
        tabs, raw, nbits, stuffed = oracle.entropy_encode(coef, mw, mh)
        hdr = oracle.headers(w, h, tabs)
        assert np.array_equal(out[: hdr.size], hdr)
        assert np.array_equal(out[hdr.size: n - 2], stuffed)
        assert out[n - 2] == 0xFF and out[n - 1] == 0xD9
        # (d)
        assert st.scan_bytes == (st.scan_bits + 7) // 8 + st.stuffed_ff == stuffed.size
        assert st.stuffed_ff == int(np.count_nonzero(raw == 0xFF))
    finally:
        encoder.dev_free(d)


def test_batch_frames_independent(encoder, oracle):
    """config 4 at reduced count: 1920x1080 frames (padded rows 1080 -> 1088), each with its own tables and DC chains"""
    for k in (0, 1, 2):
        rgb = synth_rgb(1920, 1080, k)
        assert encoder.encode_rgb(rgb) == oracle.encode_rgb(rgb)


@pytest.mark.gpu
def test_batch_api_matches_single_encodes(encoder, oracle):
    """jpgenc_batch_encode: frames handed to several contexts/threads come back byte-identical, in order"""
    from jpgenc_b200.capi import Batch
    frames = [synth_rgb(208, 120, s) for s in range(12)] + [noise_rgb(208, 120, 99)]
    want = [oracle.encode_rgb(f) for f in frames]
    b = Batch(0, workers=4)
    try:
        assert b.encode(frames) == want
        assert b.encode(frames[:1]) == want[:1]                  # fewer frames than workers
        assert b.encode(frames[::-1]) == want[::-1]              # contexts are reusable
    finally:
        b.close()


@pytest.mark.parametrize("w,h", [(4096, 1536), (3001, 1203)])
def test_banded_upload_matches_resident_encode(encoder, oracle, w, h):
    """jpgenc_encode_rgb uploads in bands with K1 per band (several bands here, also with an odd width where K1 takes
    the clamped loader): same bytes as the one-shot upload + encode, and as the oracle"""
    rgb = synth_rgb(w, h, 5)
    banded = encoder.encode_rgb(rgb)
    encoder.upload_rgb(rgb)
    out = np.empty(len(banded) + 64, np.uint8)
    n = encoder.encode_bound(out)
    assert out[:n].tobytes() == banded
    assert banded == oracle.encode_rgb(rgb)


def test_high_entropy_image_byte_identical(encoder, oracle):
    """2048x2048 uniform noise: ~40 AC symbols per block, so K2 needs several descriptor windows per tile, item
    ranges are ~25x longer than on smooth images and the scan has many FF bytes to stuff"""
    rgb = noise_rgb(2048, 2048, 7)
    mine = encoder.encode_rgb(rgb)
    st = encoder.stats()
    assert st.stuffed_ff > 1000 and st.scan_bits > 8 * 2048 * 2048 // 4
    assert mine == oracle.encode_rgb(rgb)


@pytest.mark.parametrize("q", [1, 2, 3, 16])
def test_adversarial_blocks_bit_exact(encoder, oracle, q):
    """The FP32 fast path is only trusted outside a computed error bound around rounding boundaries.  Stress it with
    inputs built to maximise FP32 error and boundary hits: +-128 patterns (largest magnitudes in every butterfly),
    sparse impulses, and flat quantisers q (a flat q=1 table makes every quotient a full-magnitude coefficient, so
    the threshold is at its loosest); blocks with ties (exact x.5 quotients) must round half away like the reference."""
    rng = np.random.default_rng(100 + q)
    blocks = []
    for r in range(8):                                   # separable +-128 sign patterns: extreme magnitudes
        for c in range(8):
            sr = np.where(np.cos((2 * np.arange(8) + 1) * r * np.pi / 16) >= 0, 1.0, -1.0)
            sc = np.where(np.cos((2 * np.arange(8) + 1) * c * np.pi / 16) >= 0, 1.0, -1.0)
            blocks.append(128.0 * np.outer(sr, sc))
            blocks.append(-128.0 * np.outer(sr, sc))
    blocks += [np.full((8, 8), v, np.float64) for v in (-128, -127, -1, 0, 1, 4, 12, 127, 128)]   # DC only: exact ties for q | 8v
    for _ in range(400):                                 # +-128 random signs
        blocks.append(128.0 * rng.choice([-1.0, 1.0], (8, 8)))
    for _ in range(400):                                 # saturated / near-saturated integers
        blocks.append(rng.choice([-128.0, -127.0, 126.0, 127.0], (8, 8)))
    for _ in range(400):                                 # impulses
        b = np.zeros((8, 8)); b[rng.integers(8), rng.integers(8)] = rng.integers(-128, 128); blocks.append(b)
    for _ in range(800):                                 # plain 8-bit noise
        blocks.append(rng.integers(-128, 128, (8, 8)).astype(np.float64))
    x = np.ascontiguousarray(np.stack(blocks).reshape(-1, 64), np.float32)
    nb = x.shape[0]
    table = np.full(64, q, np.uint8)
    d_in, d_out = encoder.dev_alloc(nb * 256), encoder.dev_alloc(nb * 128)
    try:
        encoder.h2d(d_in, x)
        refined = encoder.dct_quant_blocks(d_in, d_out, nb, table)
        y = np.empty((nb, 64), np.int16)
        encoder.d2h(y, d_out)
        zz = np.array([oracle.zigzag_index(i) for i in range(64)])
        qt = table.reshape(8, 8)
        bad = 0
        for b in range(nb):
            want = oracle.quantize(oracle.dct(x[b].astype(np.float64).reshape(8, 8)), qt).reshape(64)[zz]
            bad += int(np.count_nonzero(want != y[b]))
        assert bad == 0, f"{bad} coefficients differ (q={q}, {refined} of {nb} blocks refined)"
    finally:
        encoder.dev_free(d_in)
        encoder.dev_free(d_out)


@pytest.mark.parametrize("w,h,n", [(208, 120, 13), (512, 384, 5), (101, 67, 9), (16, 16, 40)])
def test_frames_through_the_kernels_together(encoder, oracle, w, h, n):
    """jpgenc_encode_frames_device: a batch of frames in ONE pass through every kernel (grid dimension = frame) must give
    the files of n separate encodes: own DC chains, own first-occurrence orders, own tables, own padding and stuffing"""
    frames = [synth_rgb(w, h, s) if s % 3 else noise_rgb(w, h, s) for s in range(n)]
    want = [oracle.encode_rgb(f) for f in frames]
    fb = w * h * 3
    d = encoder.dev_alloc(n * fb + 64)
    try:
        for i, f in enumerate(frames):
            encoder.h2d(d + i * fb, np.ascontiguousarray(f))
        cap = max(len(x) for x in want) + 64
        outs = [np.zeros(cap, np.uint8) for _ in range(n)]
        sizes = encoder.encode_frames_device([d + i * fb for i in range(n)], w, h, [o.ctypes.data for o in outs], [cap] * n)
        assert sizes == [len(x) for x in want]
        for i in range(n):
            assert outs[i][: sizes[i]].tobytes() == want[i], f"frame {i}"
        assert encoder.encode_frames_device([d + i * fb for i in range(n)], w, h) == sizes      # sizes only
        # the same batch from host memory (uploads overlapped with the kernels)
        host = [np.ascontiguousarray(f) for f in frames]
        outs2 = [np.zeros(cap, np.uint8) for _ in range(n)]
        sizes2 = encoder.encode_frames_device([f.ctypes.data for f in host], w, h, [o.ctypes.data for o in outs2], [cap] * n, host_frames=True)
        assert sizes2 == sizes and all(outs2[i][: sizes[i]].tobytes() == want[i] for i in range(n))
        # the context is usable for single images afterwards
        assert encoder.encode_rgb(frames[0]) == want[0]
    finally:
        encoder.dev_free(d)


@pytest.mark.gpu
@pytest.mark.parametrize("per_pass,lanes", [(3, 2), (1, 4), (4, 1), (7, 3), (2, 3), (12, 2)])
def test_frames_in_many_passes_on_several_lanes(encoder, oracle, monkeypatch, per_pass, lanes):
    """The batched-frame calls cut a batch into passes and run them on several pipeline lanes (own streams and buffers, one
    host thread each; uploads of host frames travel through a ring of slices ahead of the kernels).  Forcing tiny passes
    makes every hand-over happen many times: the files must not depend on pass size, lane count or which lane ran a pass.
    (12, 2) gives exactly two passes, the one shape whose second pass waits for the first pass's K1 (staggered)."""
    monkeypatch.setenv("JPGENC_FRAMES_PER_PASS", str(per_pass))
    monkeypatch.setenv("JPGENC_SLOTS", str(lanes))
    w, h, n = 176, 104, 23
    frames = [synth_rgb(w, h, s) if s % 4 else noise_rgb(w, h, s) for s in range(n)]
    want = [oracle.encode_rgb(f) for f in frames]
    fb = w * h * 3
    d = encoder.dev_alloc(n * fb + 64)
    try:
        for i, f in enumerate(frames):
            encoder.h2d(d + i * fb, np.ascontiguousarray(f))
        cap = max(len(x) for x in want) + 64
        for rep in range(2):                                      # second round: lanes and their buffers are reused
            outs = [np.zeros(cap, np.uint8) for _ in range(n)]
            sizes = encoder.encode_frames_device([d + i * fb for i in range(n)], w, h, [o.ctypes.data for o in outs], [cap] * n)
            assert sizes == [len(x) for x in want]
            assert all(outs[i][: sizes[i]].tobytes() == want[i] for i in range(n))
            assert encoder.encode_frames_device([d + i * fb for i in range(n)], w, h) == sizes
            host = [np.ascontiguousarray(f) for f in frames]
            outs2 = [np.zeros(cap, np.uint8) for _ in range(n)]
            sizes2 = encoder.encode_frames_device([f.ctypes.data for f in host], w, h, [o.ctypes.data for o in outs2], [cap] * n, host_frames=True)
            assert sizes2 == sizes and all(outs2[i][: sizes[i]].tobytes() == want[i] for i in range(n))
            # frames that follow each other in host memory travel as one strided copy per run (the frame size is not a
            # multiple of the 256-byte device stride here); a gap after frame 9 splits the run
            block = np.zeros(n * fb + 512, np.uint8)
            offs = [i * fb + (512 if i > 9 else 0) for i in range(n)]
            for i, f in enumerate(frames):
                block[offs[i]: offs[i] + fb] = f.reshape(-1)
            outs3 = [np.zeros(cap, np.uint8) for _ in range(n)]
            sizes3 = encoder.encode_frames_device([block.ctypes.data + o for o in offs], w, h, [o.ctypes.data for o in outs3], [cap] * n, host_frames=True)
            assert sizes3 == sizes and all(outs3[i][: sizes[i]].tobytes() == want[i] for i in range(n))
            assert encoder.encode_frames_device([f.ctypes.data for f in host], w, h, host_frames=True) == sizes   # sizes only
        # a too-small output buffer in a late pass is reported, and the context keeps working
        small = [cap] * n
        small[n - 2] = 16
        outs = [np.zeros(cap, np.uint8) for _ in range(n)]
        with pytest.raises(Exception):
            encoder.encode_frames_device([d + i * fb for i in range(n)], w, h, [o.ctypes.data for o in outs], small)
        assert encoder.encode_rgb(frames[1]) == want[1]
    finally:
        encoder.dev_free(d)


@pytest.mark.gpu
def test_device_table_build_equals_host_build(encoder):
    """build_tables_kernel restates libstdc++'s unordered_map iteration order and heap order on arrays; the host build drives
    the real containers.  Same tables -- codes, lengths, DHT symbol order -- for every alphabet size and weight pattern."""
    rng = np.random.default_rng(2024)
    counts, firsts = [], []
    for nsym in list(range(1, 40)) + [47, 59, 60, 64, 100, 127, 128, 129, 162, 200, 255, 256] + list(rng.integers(2, 257, 120)):
        c, f = random_symbol_stats(rng, int(nsym), int(rng.choice([5, 1000, 10 ** 6, 2 ** 31 - 1])))
        counts.append(c); firsts.append(f)
    dev = encoder.build_huffman_device(np.stack(counts), np.stack(firsts))
    for i, (c, f) in enumerate(zip(counts, firsts)):
        host = encoder.build_huffman([c] * 4, [f] * 4)[0]
        assert table_fields(dev[i]) == table_fields(host), f"table {i} ({int(np.count_nonzero(c))} symbols) differs"


@pytest.mark.gpu
def test_device_table_build_small_alphabets_with_many_ties(encoder):
    """Alphabets of up to 64 symbols with small weights take the loop-free heap operations (LeanHeap, tables_device.cu); equal
    weights are where the heap's layout decides the result, so: tiny weight ranges, hundreds of alphabets, every size."""
    rng = np.random.default_rng(77)
    counts, firsts = [], []
    for rep in range(6):
        for nsym in range(2, 65):
            c, f = random_symbol_stats(rng, nsym, int(rng.choice([2, 3, 4, 7, 40, 5000])))
            counts.append(c); firsts.append(f)
    dev = encoder.build_huffman_device(np.stack(counts), np.stack(firsts))
    for i, (c, f) in enumerate(zip(counts, firsts)):
        host = encoder.build_huffman([c] * 4, [f] * 4)[0]
        assert table_fields(dev[i]) == table_fields(host), f"table {i} ({int(np.count_nonzero(c))} symbols) differs"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["synth_512", "noise_256", "odd_203x117", "one_pixel", "stripes", "maxval15"])
def test_device_table_build_on_image_statistics(encoder, name):
    rgb, maxval = IMAGES[name]
    encoder.upload_rgb(rgb, maxval)
    encoder.color_dct_quant()
    count, first = encoder.symbol_stats()
    host = encoder.build_huffman(count, first)
    dev = encoder.build_huffman_device(count, first)
    for t in range(4):
        assert table_fields(dev[t]) == table_fields(host[t]), f"table {t}"


@pytest.mark.gpu
@pytest.mark.parametrize("guess", ["12", "0"])
def test_frames_packed_output_and_refused_passes(oracle, monkeypatch, guess):
    """jpgenc_encode_frames_packed: complete files (headers written on the device, stuffed scan, EOI) back to back in ONE
    buffer, one device-to-host copy per pass.  With JPGENC_RAW_GUESS_PER_BLOCK=0 the first passes reserve too little scan
    space: finalize_tables_kernel refuses them and the host re-runs their entropy stage with what they asked for."""
    from jpgenc_b200.capi import Encoder, pinned_empty, pinned_free
    monkeypatch.setenv("JPGENC_RAW_GUESS_PER_BLOCK", guess)
    monkeypatch.setenv("JPGENC_FRAMES_PER_PASS", "5")
    enc = Encoder(0)
    try:
        w, h, n = 208, 120, 23
        frames = [synth_rgb(w, h, s) if s % 3 else noise_rgb(w, h, s) for s in range(n)]
        want = [oracle.encode_rgb(f) for f in frames]
        host = [np.ascontiguousarray(f) for f in frames]
        total_want = sum(len(x) for x in want)
        buf, ptr = pinned_empty(total_want + 64)
        try:
            for rep in range(2):
                buf[:] = 0
                offs, sizes, total = enc.encode_frames_packed([f.ctypes.data for f in host], w, h, ptr, buf.size, host_frames=True)
                assert sizes == [len(x) for x in want] and total == total_want
                assert offs == [sum(sizes[:i]) for i in range(n)]             # frame order, no gaps
                assert all(buf[offs[i]: offs[i] + sizes[i]].tobytes() == want[i] for i in range(n))
            # device-resident frames, and sizes/offsets only
            fb = w * h * 3
            d = enc.dev_alloc(n * fb + 64)
            try:
                for i, f in enumerate(host):
                    enc.h2d(d + i * fb, f)
                buf[:] = 0
                offs2, sizes2, total2 = enc.encode_frames_packed([d + i * fb for i in range(n)], w, h, ptr, buf.size)
                assert (offs2, sizes2, total2) == (offs, sizes, total)
                assert buf[:total].tobytes() == b"".join(want)
                assert enc.encode_frames_packed([d + i * fb for i in range(n)], w, h, None, 0) == (offs, sizes, total)
                with pytest.raises(Exception):                              # capacity is checked before anything is copied past it
                    enc.encode_frames_packed([d + i * fb for i in range(n)], w, h, ptr, total - 1)
                assert enc.encode_rgb(frames[2]) == want[2]
            finally:
                enc.dev_free(d)
        finally:
            pinned_free(ptr)
    finally:
        enc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("slots,per_pass", [(None, None), (2, 48)])
def test_batch_of_1080p_frames_at_its_real_size(oracle, monkeypatch, slots, per_pass):
    """BASELINE config 4 at its real frame size and a GPU's share of it: 160 frames of 1920x1080 (1080 -> 1088 bottom
    clamp, a partial fourth strip in every MCU row, K1's prefetch running across frame boundaries, several passes on
    several slots, device-built tables) -- every file is compared with the oracle's, through the per-frame and the packed
    output."""
    from concurrent.futures import ThreadPoolExecutor
    from jpgenc_b200.capi import Encoder, pinned_empty, pinned_free
    if slots:
        monkeypatch.setenv("JPGENC_SLOTS", str(slots))
        monkeypatch.setenv("JPGENC_FRAMES_PER_PASS", str(per_pass))
    enc = Encoder(0)
    w, h, n = 1920, 1080, 160
    fb = w * h * 3
    d = enc.dev_alloc(n * fb)
    host, host_ptr = pinned_empty(n * fb)
    try:
        for k in range(n):
            enc.synth_rgb(d + k * fb, w, h, k)                   # the device generator is checked against synth.py elsewhere
        enc.synchronize()
        enc.d2h(host, d)
        frames = host.reshape(n, h, w, 3)
        with ThreadPoolExecutor(os.cpu_count() or 4) as ex:
            want = list(ex.map(oracle.encode_rgb, frames))
        assert np.array_equal(frames[7], synth_rgb(w, h, 7))
        total_want = sum(len(x) for x in want)
        out, out_ptr = pinned_empty(total_want + 4096)
        try:
            offs, sizes, total = enc.encode_frames_packed([d + k * fb for k in range(n)], w, h, out_ptr, out.size)
            assert sizes == [len(x) for x in want] and total == total_want
            bad = [k for k in range(n) if out[offs[k]: offs[k] + sizes[k]].tobytes() != want[k]]
            assert not bad, f"frames {bad[:8]} differ from the oracle (device-resident, packed)"
            out[:] = 0
            offs2, sizes2, _ = enc.encode_frames_packed([host_ptr + k * fb for k in range(n)], w, h, out_ptr, out.size, host_frames=True)
            assert (offs2, sizes2) == (offs, sizes)
            assert out[:total].tobytes() == b"".join(want), "host frames, packed"
            cap = max(sizes) + 64
            outs = [np.zeros(cap, np.uint8) for _ in range(n)]
            sizes3 = enc.encode_frames_device([d + k * fb for k in range(n)], w, h, [o.ctypes.data for o in outs], [cap] * n)
            assert sizes3 == sizes and all(outs[k][: sizes[k]].tobytes() == want[k] for k in range(n)), "per-frame buffers"
        finally:
            pinned_free(out_ptr)
    finally:
        pinned_free(host_ptr)
        enc.dev_free(d)
        enc.close()


@pytest.mark.parametrize("graphs", ["1", "0"])
def test_repeated_encodes_of_bound_pixels_replay_graphs(oracle, monkeypatch, graphs):
    """jpgenc_encode_bound on pixels that stay bound: from the third encode of a configuration on, both GPU phases are
    replayed as CUDA graphs (captured at the second).  The bytes must not depend on that -- also when the CONTENT behind
    the same pointer changes (other scan length, other tables, other number of K4 tiles), when another size is encoded in
    between, and when the quantisers change."""
    from jpgenc_b200.capi import Encoder
    monkeypatch.setenv("JPGENC_GRAPHS", graphs)
    enc = Encoder(0)
    try:
        w, h = 400, 304
        a, b = synth_rgb(w, h, 1), noise_rgb(w, h, 2)            # very different scan lengths
        want_a, want_b = oracle.encode_rgb(a), oracle.encode_rgb(b)
        d = enc.dev_alloc(w * h * 3)
        out = np.zeros(max(len(want_a), len(want_b)) + 64, np.uint8)
        try:
            enc.h2d(d, a)
            enc.bind_device_rgb(d, w, h)
            for _ in range(5):
                n = enc.encode_bound(out)
                assert out[:n].tobytes() == want_a
            enc.h2d(d, b)                                        # same pointer, new content: the captured graphs stay valid
            for _ in range(4):
                n = enc.encode_bound(out)
                assert out[:n].tobytes() == want_b
            enc.h2d(d, a)
            n = enc.encode_bound(out)
            assert out[:n].tobytes() == want_a
            other = synth_rgb(208, 120, 5)                       # another size in between (upload path), then back
            assert enc.encode_rgb(other) == oracle.encode_rgb(other)
            enc.bind_device_rgb(d, w, h)
            for _ in range(4):
                n = enc.encode_bound(out)
                assert out[:n].tobytes() == want_a
            q = np.full(64, 3, np.uint8)
            enc.set_qtables(q, q)
            out = np.zeros(w * h * 3, np.uint8)
            for _ in range(3):
                n = enc.encode_bound(out)
                got_q = out[:n].tobytes()
            assert got_q != want_a and got_q[:2] == b"\xff\xd8" and got_q[-2:] == b"\xff\xd9"
            # the same quantisers on a fresh context (no graph): identical bytes
            enc2 = Encoder(0)
            try:
                enc2.set_qtables(q, q)
                assert enc2.encode_rgb(a) == got_q
            finally:
                enc2.close()
        finally:
            enc.dev_free(d)
    finally:
        enc.close()


def test_stage_timing_levels_change_times_not_bytes(oracle):
    """jpgenc_set_stage_timing: the event records between the kernels are off by default (stats' stage times stay 0), level 1
    times the K1 fast kernel, level 2 every stage; switching in the middle of a run of encodes re-captures the graphs and
    never changes a byte"""
    from jpgenc_b200.capi import Encoder
    enc = Encoder(0)
    try:
        w, h = 624, 416
        rgb = synth_rgb(w, h, 3)
        want = oracle.encode_rgb(rgb)
        d = enc.dev_alloc(w * h * 3)
        out = np.zeros(len(want) + 64, np.uint8)
        try:
            enc.h2d(d, rgb)
            enc.bind_device_rgb(d, w, h)
            for level in (0, 2, 1, 0, 2):
                enc.set_stage_timing(level)
                for _ in range(4):                                # plain launches, capture, replays
                    n = enc.encode_bound(out)
                    assert out[:n].tobytes() == want
                s = enc.stats()
                if level == 0:
                    assert s.ms_k1 == 0 and s.ms_forward == 0 and s.ms_stats == 0 and s.ms_entropy == 0
                elif level == 1:
                    assert s.ms_k1 > 0 and s.ms_forward == 0 and s.ms_stats == 0 and s.ms_entropy == 0
                else:
                    assert 0 < s.ms_k1 <= s.ms_forward and s.ms_stats > 0 and s.ms_entropy > 0
            with pytest.raises(Exception):
                enc.set_stage_timing(3)
        finally:
            enc.dev_free(d)
    finally:
        enc.close()


def test_entropy_stage_can_run_twice_on_a_large_image(encoder, oracle):
    """K3a accumulates bit counts per 256 groups with atomics into words that K2's launch cleared: a second
    jpgenc_entropy_encode over the same symbol items (here: the same tables again) must not see them doubled.  4096x2304
    has 576 K2 tiles = 2304 item ranges = 288 groups, i.e. more than one super-group."""
    w, h = 4096, 2304
    rgb = synth_rgb(w, h, 11)
    want = oracle.encode_rgb(rgb)
    encoder.upload_rgb(rgb)
    encoder.color_dct_quant()
    count, first = encoder.symbol_stats()
    tabs = encoder.build_huffman(count, first)
    n1 = encoder.entropy_encode(tabs)
    scan1 = encoder.download_scan().copy()
    n2 = encoder.entropy_encode(tabs)
    scan2 = encoder.download_scan().copy()
    assert n1 == n2 and np.array_equal(scan1, scan2)
    hdr = encoder.headers(tabs, w, h, oracle.qy, oracle.qc)
    assert hdr.tobytes() + scan2.tobytes() + b"\xff\xd9" == want


@pytest.mark.gpu
def test_ppm_file_streamed_band_by_band(encoder, oracle, tmp_path):
    """jpgenc_encode_ppm_file streams a P6 payload: every band of rows is read (by several threads) into pinned staging,
    uploaded, and taken through K1 / refinement / K2 while the next band is read.  A file with several bands, a header
    with a comment, an odd width (clamped loader), a truncated payload (error), and an ASCII file through the same call."""
    from jpgenc_b200.capi import ERR_FORMAT, JpgencError
    from jpgenc_b200.synth import write_ppm
    for w, h, seed in ((4096, 2304, 3), (3001, 2999, 4)):
        rgb = synth_rgb(w, h, seed)
        src, dst = tmp_path / f"in_{w}.ppm", tmp_path / f"out_{w}.jpg"
        src.write_bytes(b"P6\n# streamed\n%d %d\n255\n" % (w, h) + rgb.tobytes())
        encoder.encode_ppm_file(str(src), str(dst))
        assert dst.read_bytes() == oracle.encode_rgb(rgb)
        data = src.read_bytes()
        cut = tmp_path / f"cut_{w}.ppm"
        cut.write_bytes(data[:-1000])
        with pytest.raises(JpgencError) as e:
            encoder.encode_ppm_file(str(cut), str(tmp_path / "never.jpg"))
        assert e.value.code == ERR_FORMAT
    small = noise_rgb(37, 21, 5)
    p3 = tmp_path / "ascii.ppm"
    p3.write_text("P3\n37 21\n255\n" + "\n".join(" ".join(str(int(v)) for v in row.reshape(-1)) for row in small) + "\n")
    encoder.encode_ppm_file(str(p3), str(tmp_path / "ascii.jpg"))
    assert (tmp_path / "ascii.jpg").read_bytes() == oracle.encode_rgb(small)
    # the context still works for in-memory images afterwards
    assert encoder.encode_rgb(small) == oracle.encode_rgb(small)


@pytest.mark.gpu
def test_planes_of_doubles_byte_identical(encoder, oracle, golden_planes):
    """jpgenc_encode_planes: an Image assembled or edited in memory (real-valued samples, edited padding, planes that already
    are YCbCr) -- the reference's own bytes for the golden cases, the oracle's for larger ones"""
    for name in [str(n) for n in golden_planes["names"]]:
        planes = golden_planes[f"{name}/planes"]
        w, h, ycc = (int(x) for x in golden_planes[f"{name}/dims"])
        assert encoder.encode_planes(planes[0], planes[1], planes[2], w, h, bool(ycc)) == golden_planes[f"{name}/jpg"].tobytes(), name
    rng = np.random.default_rng(31)
    for (w, h, ycc) in [(333, 201, False), (512, 256, True)]:
        w16, h16 = (w + 15) // 16 * 16, (h + 15) // 16 * 16
        lo, hi = (-128, 127) if ycc else (0, 255)
        planes = [rng.uniform(lo, hi, (h16, w16)) for _ in range(3)]
        assert encoder.encode_planes(planes[0], planes[1], planes[2], w, h, ycc) == oracle.encode_planes(planes[0], planes[1], planes[2], w, h, ycc)
    # 8-bit samples given as planes == the 8-bit path
    rgb = synth_rgb(208, 120, 5)
    pad = np.pad(rgb, ((0, 8), (0, 0), (0, 0)), mode="edge").astype(np.float64)
    assert encoder.encode_planes(pad[..., 0], pad[..., 1], pad[..., 2], 208, 120) == encoder.encode_rgb(rgb)
    with pytest.raises(Exception):
        encoder.encode_planes(pad[:120, :, 0], pad[:120, :, 1], pad[:120, :, 2], 208, 120)      # not padded to whole MCUs


@pytest.mark.gpu
def test_stage_kernels_every_subsampling_and_dct_mode(encoder, oracle):
    """SURVEY 8(f)4: Image::applySubsampling for all six SubsamplingModes and Image::applyDCT for Simple / Matrix / Arai on whole
    planes of doubles -- the device's planes against the oracle's (itself pinned against the compiled reference), exactly"""
    rng = np.random.default_rng(8)
    for (w, h) in [(16, 16), (64, 48), (256, 128), (1920, 1088)]:
        plane = rng.uniform(-128, 127, (h, w))
        plane[0, 0] = -0.0
        for name, mode in oracle.SUBSAMPLING.items():
            got, want = encoder.stage_subsample(plane, mode), oracle.subsample_plane(plane, name)
            assert got.shape == want.shape and np.array_equal(got.view(np.uint64), want.view(np.uint64)), (name, w, h)
        if w * h > 300000:
            plane = plane[:64]
        for name, mode in oracle.DCT_MODES.items():
            got, want = encoder.stage_dct(plane, mode), oracle.dct_plane(plane, name)
            assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), (name, w, h)
    from jpgenc_b200.capi import JpgencError
    with pytest.raises(JpgencError):
        encoder.stage_dct(np.zeros((12, 16)), 2)                     # sides must be multiples of 8
    with pytest.raises(JpgencError):
        encoder.stage_subsample(np.zeros((16, 18)), 2)               # S411 takes four columns at a time


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["dense_extreme", "zrl_runs", "last_only", "mixed", "ff_rich", "outrun"])
def test_entropy_coder_on_synthetic_coefficient_arrays(encoder, oracle, kind):
    """K2 .. K4 on coefficient arrays no image produces: every coefficient non-zero with 15-bit magnitudes (code + magnitude
    longer than the one-lookup path's 27 bits, chunks denser than the warp bit buffer: the straight-to-global path of K3b), runs
    of exactly 15 / 16 / 17 / 31 / 32 / 47 / 48 / 62 zeros (ZRL boundaries), blocks whose only coefficient is the last one (no
    EOB), and a mix; statistics, tables and the stuffed scan against the oracle's entropy coder on the same array"""
    rng = np.random.default_rng({"dense_extreme": 1, "zrl_runs": 2, "last_only": 3, "mixed": 4, "ff_rich": 5, "outrun": 6}[kind])
    mw, mh = (128, 128) if kind == "outrun" else (24, 20)
    nb = mw * mh * 6
    coef = np.zeros((nb, 64), np.int16)
    if kind == "outrun":
        # K3b writes a lane's completed words over the items the lane has consumed; an item of more than 64 bits that is a lane's
        # FIRST item outruns that (its second word has no free slot) and the chunk must take the slow path.  Such an item needs
        # three ZRLs and a 15-bit magnitude behind codes of 15-16 bits: ~100 k light blocks over ~160 symbols make the two
        # heavy blocks' symbols that rare; the heavy blocks sit where their AC item opens a lane's items (K3 cuts this array's tiles
        # into quarters of 287 items, 9 per lane: with the tile's first block DC-only, block 21's AC item is item 63 = 9 x 7).
        coef[:, 0] = rng.integers(-500, 500, nb)
        pos = np.minimum(16, rng.geometric(0.25, nb)); cat = np.minimum(10, rng.geometric(0.45, nb))
        val = ((1 << (cat - 1)) + rng.integers(0, 1 << 14, nb) % (1 << (cat - 1))) * rng.choice([-1, 1], nb)
        coef[np.arange(nb), pos] = val.astype(np.int16)
        for tile in (7, 100):
            coef[384 * tile, 1:] = 0
            coef[384 * tile + 21, 1:] = 0
            coef[384 * tile + 21, 63] = -30000
    elif kind == "dense_extreme":
        coef[:] = rng.integers(8192, 32768, (nb, 64)) * rng.choice([-1, 1], (nb, 64))
        coef[:, 0] = rng.integers(-16000, 16000, nb)              # DC differences stay below 2^15: category 16 is outside the reference's coder
    elif kind == "zrl_runs":
        for b in range(nb):
            gap = int(rng.choice([15, 16, 17, 31, 32, 47, 48, 62]))
            coef[b, 0] = rng.integers(-300, 300)
            coef[b, 1 + gap - 1 if gap < 63 else 63] = rng.integers(1, 40) * rng.choice([-1, 1])
            if gap + 17 < 64 and rng.random() < 0.5:
                coef[b, gap + 17] = rng.integers(1, 5)
    elif kind == "last_only":
        coef[:, 63] = rng.integers(1, 1000, nb) * rng.choice([-1, 1], nb)
        coef[::3, 0] = rng.integers(-1000, 1000, len(coef[::3]))
    elif kind == "ff_rich":
        # magnitudes of all ones behind short codes: more than a quarter of the scan's bytes are FF (8 k of 29 k), runs of them across
        # K4's 4 KB tiles and at the frame's end
        coef[:, :8] = 1023
    else:
        dense = rng.random(nb) < 0.15
        coef[dense] = (rng.integers(1, 2000, (int(dense.sum()), 64)) * rng.choice([-1, 1], (int(dense.sum()), 64))).astype(np.int16)
        sparse = ~dense
        mask = rng.random((nb, 64)) < 0.05
        vals = (rng.integers(1, 30, (nb, 64)) * rng.choice([-1, 1], (nb, 64))).astype(np.int16)
        coef[sparse] = np.where(mask[sparse], vals[sparse], 0)
        coef[:, 0] = rng.integers(-1024, 1024, nb)
    coef = coef.reshape(mw * mh, 6, 64)
    encoder.set_coefficients_mcu(coef, mw, mh)
    count, first = encoder.symbol_stats()
    ocount, ofirst = oracle.symbol_stats(coef, mw, mh)
    assert np.array_equal(count, ocount) and np.array_equal(first, ofirst)
    tabs = encoder.build_huffman(count, first)
    otabs, _, onbits, ostuffed = oracle.entropy_encode(coef, mw, mh)
    for t in range(4):
        assert table_fields(tabs[t]) == table_fields(otabs[t]), f"table {t}"
    n = encoder.entropy_encode(tabs)
    scan = encoder.download_scan()
    assert n == ostuffed.size and np.array_equal(scan, ostuffed), kind
    if kind == "ff_rich":
        assert encoder.stats().stuffed_ff > 5000
    if kind == "outrun":
        assert encoder.debug_counter(6) >= 1, "the slow path of the Huffman packer was not exercised"


@pytest.mark.gpu
def test_random_sizes_and_contents_byte_identical(encoder, oracle):
    """80 images of random size (1 .. 260 pixels a side: every padding amount, single-MCU and single-row images, partial strips
    and tiles) and random content (noise, flat, sparse spikes, saturated checkers, gradients, low maxval): whole files against the
    oracle, through the host-pixel path and -- every fourth -- through bound device pixels"""
    rng = np.random.default_rng(20261019)
    for case in range(80):
        w, h = int(rng.integers(1, 261)), int(rng.integers(1, 261))
        kind = case % 6
        maxval = 255
        if kind == 0:
            rgb = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        elif kind == 1:
            rgb = np.full((h, w, 3), rng.integers(0, 256, 3), np.uint8)
        elif kind == 2:
            rgb = np.zeros((h, w, 3), np.uint8)
            n = max(1, w * h // 50)
            rgb[rng.integers(0, h, n), rng.integers(0, w, n)] = rng.integers(0, 256, (n, 3))
        elif kind == 3:
            yy, xx = np.mgrid[0:h, 0:w]
            rgb = (((yy // int(rng.integers(1, 9)) + xx // int(rng.integers(1, 9))) % 2) * 255).astype(np.uint8)[..., None].repeat(3, 2)
        elif kind == 4:
            yy, xx = np.mgrid[0:h, 0:w]
            rgb = np.stack([(xx * 255 // max(1, w - 1)), (yy * 255 // max(1, h - 1)), ((xx + yy) % 256)], -1).astype(np.uint8)
        else:
            maxval = int(rng.choice([1, 7, 31, 100, 200]))
            rgb = rng.integers(0, maxval + 1, (h, w, 3), dtype=np.uint8)
        want = oracle.encode_ppm(ppm_p6_bytes(rgb, maxval))
        assert encoder.encode_rgb(rgb, maxval) == want, (case, w, h, kind, maxval)
        if case % 4 == 0:
            d = encoder.dev_alloc(rgb.size + 16)
            try:
                encoder.h2d(d, rgb)
                encoder.bind_device_rgb(d, w, h, maxval)
                out = np.empty(len(want) + 64, np.uint8)
                n = encoder.encode_bound(out)
                assert out[:n].tobytes() == want, (case, w, h, kind, "bound")
            finally:
                encoder.dev_free(d)


@pytest.mark.gpu
def test_batched_calls_of_changing_frame_sizes_on_one_context(oracle):
    """One context, batched calls of different frame sizes and contents in a row: what a call learnt about scan sizes (buffer
    reservations, K4 grids) is reused for the same size and dropped for another; a later, much denser batch of a known size is
    refused on the device and re-run; n = 1 and n = 0 are batches too"""
    from jpgenc_b200.capi import Encoder
    enc = Encoder(0)
    try:
        def run(frames):
            n = len(frames)
            h, w, _ = frames[0].shape if n else (16, 16, 3)
            fb = w * h * 3
            d = enc.dev_alloc(max(1, n) * fb + 16)
            try:
                for k, f in enumerate(frames):
                    enc.h2d(d + k * fb, np.ascontiguousarray(f))
                want = [oracle.encode_rgb(f) for f in frames]
                cap = sum(len(x) for x in want) + 4096
                out = np.zeros(cap, np.uint8)
                offs, sizes, total = enc.encode_frames_packed([d + k * fb for k in range(n)], w, h, out.ctypes.data, out.size)
                assert sizes == [len(x) for x in want] and total == sum(sizes)
                for k in range(n):
                    assert out[offs[k]: offs[k] + sizes[k]].tobytes() == want[k], (w, h, k)
            finally:
                enc.dev_free(d)
        smooth = [synth_rgb(320, 240, k) for k in range(20)]
        run(smooth)
        run(smooth[:7])                                             # same size again: the learnt reservation is reused
        run([noise_rgb(208, 120, k) for k in range(9)])             # another size
        run([noise_rgb(320, 240, 100 + k) for k in range(20)])      # the first size again, ~10x the scan bytes: refused and re-run
        run(smooth[:1])
        run([])
    finally:
        enc.close()


def test_empty_batches_and_geometry_changes_leave_no_stale_binding(oracle):
    """An empty batch is legal, reports nothing and leaves an image bound to the context alone (its geometry included);
    the coefficient test hook with ANOTHER geometry unbinds the pixels instead of letting K1 read them with the wrong size."""
    from jpgenc_b200.capi import Encoder, JpgencError
    enc = Encoder(0)
    try:
        w, h = 336, 208
        rgb = synth_rgb(w, h, 4)
        want = oracle.encode_rgb(rgb)
        d = enc.dev_alloc(w * h * 3)
        out = np.zeros(len(want) + 64, np.uint8)
        try:
            enc.h2d(d, rgb)
            enc.bind_device_rgb(d, w, h)
            n = enc.encode_bound(out)
            assert out[:n].tobytes() == want
            # empty batches of a LARGER geometry, in all three forms
            assert enc.encode_frames_device([], 4096, 4096) == []
            assert enc.encode_frames_device([], 4096, 4096, host_frames=True) == []
            assert enc.encode_frames_packed([], 4096, 4096, None, 0) == ([], [], 0)
            with pytest.raises(JpgencError):
                enc.encode_frames_device([], 0, 16)
            for _ in range(3):
                n = enc.encode_bound(out)
                assert out[:n].tobytes() == want
            # coefficients of another geometry through the test hook: the bound pixels no longer apply
            coef = oracle.forward(synth_rgb(64, 48, 1))
            enc.set_coefficients_mcu(coef, 4, 3)
            with pytest.raises(JpgencError):
                enc.encode_bound(out)
            enc.bind_device_rgb(d, w, h)
            n = enc.encode_bound(out)
            assert out[:n].tobytes() == want
        finally:
            enc.dev_free(d)
    finally:
        enc.close()
