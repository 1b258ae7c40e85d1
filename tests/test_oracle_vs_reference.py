"""Pins the oracle against the reference encoder itself.  Not a GPU test.

Every test below checks the oracle against answers stored in tests/golden/oracle_vs_reference.npz: a SHA-256 digest (first
16 bytes) of every array that must match exactly, field by field, and the values of the two DCT modes compared with a
tolerance.  Where oracle/_ref is built (oracle/build_ref.sh, from the reference's source tree), the compiled reference is
checked against the same stored answers, so both sides meet on every input.

Provenance of the committed file: it was written from the ORACLE's outputs, not from a run of the reference, because the
reference's tree was not at hand when these tests were made self-contained.  The oracle and these inputs are the ones that
passed these tests against the compiled reference before (then comparing the two directly).  Where the reference is built,
the reference leg of every test confirms or refutes that; tests/golden/make_oracle_vs_reference.py rewrites the file from
the compiled reference and refuses to run without it."""
import glob
import hashlib
import os
import types

import numpy as np
import pytest

from jpgenc_b200.synth import noise_rgb, ppm_p6_bytes, synth_rgb

ANSWERS = os.path.join(os.path.dirname(__file__), "golden", "oracle_vs_reference.npz")
FIXTURES = sorted(glob.glob("/root/reference/src/test/res/*.ppm"))
APPROX = {"dct/direct", "dct/matrix"}            # different operation orders: compared with atol 1e-9, stored as values


def leaves(key, value):
    """(key/field, array) for every array in `value`: bytes, arrays and ints, and dicts/lists/tuples of them"""
    if isinstance(value, dict):
        for k in sorted(value):
            yield from leaves(f"{key}/{k}", value[k])
    elif isinstance(value, (list, tuple)):
        for i, v in enumerate(value):
            yield from leaves(f"{key}/{i}", v)
    else:
        yield key, np.frombuffer(value, np.uint8) if isinstance(value, bytes) else np.ascontiguousarray(value)


def digest(a: np.ndarray) -> bytes:
    """the first 16 bytes of SHA-256 over dtype, shape and contents"""
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).digest()[:16]


class ReferenceAsOracle:
    """The compiled reference behind the oracle's method names, so that one answer function serves both."""

    def __init__(self, ref, tmp):
        from oracle.pyoracle import Oracle
        self.ref, self.tmp = ref, str(tmp)
        self.SUBSAMPLING, self.DCT_MODES = Oracle.SUBSAMPLING, Oracle.DCT_MODES

    def _ppm(self, ppm_bytes):
        p = os.path.join(self.tmp, "in.ppm")
        with open(p, "wb") as f:
            f.write(ppm_bytes)
        return p

    def encode_ppm(self, ppm_bytes):
        j = os.path.join(self.tmp, "out.jpg")
        rc, _, _ = self.ref.encode_file(self._ppm(ppm_bytes), j)
        assert rc == 0
        with open(j, "rb") as f:
            return f.read()

    def forward_planes(self, rgb):
        return self.ref.stage_dump(self._ppm(ppm_p6_bytes(rgb)))

    def dct(self, blk, mode="arai"):
        return self.ref.dct(blk, mode)

    def quantize(self, d, table):
        return self.ref.quantize(d, table)

    def block_symbols(self, blk):
        return self.ref.block_symbols(blk)

    def huffman_from_text(self, text):
        d = self.ref.huffman(text)
        return types.SimpleNamespace(as_dict=lambda: d)

    def pack_bits(self, msb, nbits, msb_aligned, fill):
        assert msb_aligned
        return self.ref.pack_bits(msb, nbits, fill=fill)

    def encode_planes(self, p0, p1, p2, w, h, ycc):
        j = os.path.join(self.tmp, "planes.jpg")
        assert self.ref.encode_planes(p0, p1, p2, w, h, ycc, j) == 0
        with open(j, "rb") as f:
            return f.read()

    def subsample_plane(self, plane, name):
        return self.ref.subsample_plane(plane, self.SUBSAMPLING[name])

    def dct_plane(self, plane, name):
        return self.ref.dct_plane(plane, self.DCT_MODES[name])


@pytest.fixture(scope="module")
def answers():
    with np.load(ANSWERS) as z:
        out = dict(zip((str(k) for k in z["keys"]), (d.tobytes() for d in z["digests"])))
        out.update({k: z[f"approx/{k}"] for k in APPROX})
    return out


@pytest.fixture(scope="module")
def impls(oracle, reference, tmp_path_factory):
    """the oracle, and the compiled reference where it was built"""
    return [oracle] + ([ReferenceAsOracle(reference, tmp_path_factory.mktemp("ref"))] if reference else [])


def check(answers, impls, fn, *params):
    """every answer of fn(impl, *params) against the stored one; a failure names the implementation and the field"""
    for impl in impls:
        for key, got in fn(impl, *params).items():
            if key in APPROX:
                bad = ~np.isclose(got, answers[key], atol=1e-9)
                assert not bad.any(), (type(impl).__name__, key, "blocks", sorted(set(np.nonzero(bad)[0].tolist())))
                continue
            for leaf, a in leaves(key, got):
                assert digest(a) == answers[leaf], (type(impl).__name__, leaf, a)


@pytest.mark.skipif(not FIXTURES, reason="/root/reference not mounted")
@pytest.mark.parametrize("path", FIXTURES, ids=[os.path.basename(f) for f in FIXTURES])
def test_reference_fixtures_byte_identical(oracle, reference, tmp_path, path):
    if reference is None:
        pytest.skip("oracle/_ref not built")
    data = open(path, "rb").read()
    assert oracle.encode_ppm(data) == ReferenceAsOracle(reference, tmp_path).encode_ppm(data)


# SURVEY.md 8(c) pins (generator of 8(d), seed 0): sha256 of the PPM, size and sha256 of the reference's JPEG
PINS = {
    (512, 512): ("82eac3f4d5808b2ba53ca02b76058b00619eea319ce5482c933a5f560b16e554", 12323,
                 "ceedd1ecae8dbeaf3620f9256abf57c9061167b65f5d574426739cacd82a3c20"),
    (1920, 1080): ("580cec4112d86c1d5cbf13d6ca129bc01f6afee2026e46d070f480bec135e884", 87008,
                   "f6d1960662d092cef9ff642694f089a6142cb3d3e0d45113e0ec0606c6656554"),
}


@pytest.mark.parametrize("size", list(PINS))
def test_synthetic_pins(impls, size):
    w, h = size
    ppm = ppm_p6_bytes(synth_rgb(w, h, 0))
    psha, nbytes, jsha = PINS[size]
    assert hashlib.sha256(ppm).hexdigest() == psha
    for impl in impls:
        jpg = impl.encode_ppm(ppm)
        assert len(jpg) == nbytes and hashlib.sha256(jpg).hexdigest() == jsha, type(impl).__name__


def odd_size_answers(impl, w, h, kind):
    rgb = synth_rgb(w, h, 5) if kind == "synth" else noise_rgb(w, h, 9)
    return {f"odd/{w}x{h}/{kind}": impl.encode_ppm(ppm_p6_bytes(rgb))}


ODD_SIZES = [(256, 256, "noise"), (100, 37, "noise"), (33, 17, "synth"), (1, 1, "noise"), (16, 16, "synth"), (17, 16, "synth"),
             (16, 17, "noise")]


@pytest.mark.parametrize("w,h,kind", ODD_SIZES)
def test_odd_sizes_and_noise(answers, impls, w, h, kind):
    check(answers, impls, odd_size_answers, w, h, kind)


def stage_dump_answers(impl):
    out = {}
    for name, rgb in {"n": noise_rgb(40, 24, 4), "s": synth_rgb(64, 48, 2)}.items():
        d = impl.forward_planes(rgb)
        for k in ("y", "cb", "cr", "dct_y", "dct_cb", "dct_cr", "q_y", "q_cb", "q_cr"):
            out[f"stage/{name}/{k}"] = d[k]
    return out


def test_stage_dumps_match(answers, impls):
    """every intermediate plane of the reference, bit for bit (doubles compared exactly)"""
    check(answers, impls, stage_dump_answers)


def dct_answers(impl):
    from jpgenc_b200.tables import ANNEX_K_LUMA
    rng = np.random.default_rng(3)
    blocks = [rng.uniform(-128, 128, (8, 8)) for _ in range(200)]
    arai = [impl.dct(blk) for blk in blocks]                                            # Arai: exact
    return {"dct/arai": arai, "dct/direct": np.stack([impl.dct(blk, "direct") for blk in blocks]),
            "dct/matrix": np.stack([impl.dct(blk, "matrix") for blk in blocks]),
            "dct/quantize": [impl.quantize(d, ANNEX_K_LUMA) for d in arai]}


def test_dct_and_quantize_blocks(oracle, answers, impls):
    from jpgenc_b200.tables import ANNEX_K_LUMA
    assert np.array_equal(np.asarray(ANNEX_K_LUMA, np.uint8).reshape(64), oracle.qy)
    check(answers, impls, dct_answers)


def block_symbol_answers(impl):
    rng = np.random.default_rng(5)
    out = {}
    for density in (0.02, 0.2, 0.9):
        for i in range(100):
            blk = (rng.integers(-300, 300, 64) * (rng.random(64) < density)).astype(np.int32)
            out[f"symbols/{density}/{i}"] = dict(zip(("symbols", "bits", "nbits"), impl.block_symbols(blk)))
    return out


def test_block_symbols(answers, impls):
    check(answers, impls, block_symbol_answers)


def huffman_answers(impl):
    """code lengths, codes AND the order of symbols inside a length (libstdc++ hash/heap order, SURVEY.md H2)"""
    rng = np.random.default_rng(11)
    out = {}
    for trial in range(300):
        nsym = int(rng.integers(1, 200))
        alphabet = rng.permutation(256)[:nsym]
        n = int(rng.integers(nsym, 4000))
        if trial % 3 == 0:      # many ties
            text = alphabet[rng.integers(0, nsym, n)]
        else:                   # skewed
            p = rng.random(nsym) ** 4
            text = rng.choice(alphabet, n, p=p / p.sum())
        t = impl.huffman_from_text(text).as_dict()
        out[f"huffman/{trial}"] = {k: t[k] for k in ("length", "code_msb", "counts", "symbols")}
    return out


def test_huffman_tables_random_texts(answers, impls):
    check(answers, impls, huffman_answers)


def bitstream_answers(impl):
    rng = np.random.default_rng(13)
    out = {}
    for trial in range(50):
        n = int(rng.integers(1, 300))
        nbits = rng.integers(1, 17, n)
        vals = np.array([int(rng.integers(0, 1 << b)) for b in nbits], np.uint32)
        vals[rng.random(n) < 0.3] = 0xFFFF                   # provoke FF bytes
        vals &= (1 << nbits.astype(np.uint32)) - 1
        msb = vals << (32 - nbits).astype(np.uint32)
        for fill in (False, True):
            packed, nb = impl.pack_bits(msb, nbits, msb_aligned=True, fill=fill)
            out[f"pack/{trial}/{fill}"] = {"bytes": packed, "nbits": np.int64(nb)}
    return out


def test_bitstream_pack(answers, impls):
    check(answers, impls, bitstream_answers)


def planes_answers(impl):
    """Image::writeJPEG on an Image assembled from planes of doubles (src/Image.cpp:831-846: RGB planes are converted, an
    image that already is YCbCr is not)"""
    rng = np.random.default_rng(99)
    out = {}
    for (w, h) in [(16, 16), (40, 24), (19, 50)]:
        w16, h16 = (w + 15) // 16 * 16, (h + 15) // 16 * 16
        for ycc in (False, True):
            lo, hi = (-128, 127) if ycc else (0, 255)
            planes = [rng.uniform(lo, hi, (h16, w16)) for _ in range(3)]
            out[f"planes/{w}x{h}/{ycc}"] = impl.encode_planes(planes[0], planes[1], planes[2], w, h, ycc)
    return out


def test_planes_path_matches_reference(oracle, answers, impls):
    """jo_encode_planes == the compiled reference, byte for byte"""
    check(answers, impls, planes_answers)
    # planes that hold 8-bit samples are the ordinary path
    rgb = synth_rgb(48, 32, 3)
    planes = [rgb[..., k].astype(np.float64) for k in range(3)]
    assert oracle.encode_planes(planes[0], planes[1], planes[2], 48, 32, False) == oracle.encode_rgb(rgb)


def stage_method_answers(impl):
    """Image::applySubsampling for every SubsamplingMode (src/Image.cpp:198-319) and Image::applyDCT for every DCTMode
    (src/Image.cpp:540-595, Dct.hpp:47-276) on whole planes: doubles compared exactly"""
    rng = np.random.default_rng(123)
    out = {}
    for (w, h) in [(16, 16), (32, 48), (64, 16)]:
        plane = rng.uniform(-128, 127, (h, w))
        for name in impl.SUBSAMPLING:
            out[f"subsample/{w}x{h}/{name}"] = impl.subsample_plane(plane, name)
        for name in impl.DCT_MODES:
            out[f"dct_plane/{w}x{h}/{name}"] = impl.dct_plane(plane, name)
    return out


def test_stage_methods_on_planes_match_reference(answers, impls):
    check(answers, impls, stage_method_answers)


# every answer function with the parameter sets its test runs; tests/golden/make_oracle_vs_reference.py stores their answers
CASES = [(odd_size_answers, ODD_SIZES), (stage_dump_answers, [()]), (dct_answers, [()]), (block_symbol_answers, [()]),
         (huffman_answers, [()]), (bitstream_answers, [()]), (planes_answers, [()]), (stage_method_answers, [()])]
