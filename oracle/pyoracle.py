"""ctypes bindings for the CPU oracle (oracle/liboracle.so) and, when it was built, the compiled
reference itself (oracle/_ref/libjpgenc_ref.so).

TEST INFRASTRUCTURE ONLY: import this from tests/, from __graft_entry__.smoke() and from bench.py's
cpu_baseline / --impl reference legs.  The product package (jpgenc_b200/) must never import it.
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ORACLE_SO = HERE / "liboracle.so"
REF_SO = HERE / "_ref" / "libjpgenc_ref.so"
REF_BIN = HERE / "_ref" / "jpgEnc_ref"

u8p = C.POINTER(C.c_uint8)
i16p = C.POINTER(C.c_int16)
i32p = C.POINTER(C.c_int32)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
f64p = C.POINTER(C.c_double)


def build(force: bool = False) -> None:
    """Compile liboracle.so (and oracle/_ref when the reference tree is mounted)."""
    src = HERE / "jpgenc_oracle.c"
    if force or not ORACLE_SO.exists() or ORACLE_SO.stat().st_mtime < src.stat().st_mtime:
        subprocess.run(["make", "-C", str(HERE), "-s", "-B", "liboracle.so"], check=True)
    probe = HERE / "ref_probe.cpp"
    stale = REF_SO.exists() and REF_SO.stat().st_mtime < probe.stat().st_mtime
    if force or stale or not REF_SO.exists():
        # build_ref.sh finds the tree ($JPGENC_REFERENCE or its default) and leaves oracle/_ref alone where it cannot read one
        subprocess.run(["bash", str(HERE / "build_ref.sh")], check=True)


class HuffTable(C.Structure):
    _fields_ = [
        ("code_msb", C.c_uint32 * 256),
        ("length", C.c_uint8 * 256),
        ("counts", C.c_uint8 * 16),
        ("symbols", C.c_uint8 * 256),
        ("nsymbols", C.c_int),
    ]

    def as_dict(self):
        n = int(sum(self.counts))
        return {
            "code_msb": np.array(self.code_msb, dtype=np.uint32),
            "length": np.array(self.length, dtype=np.uint8),
            "counts": np.array(self.counts, dtype=np.uint8),
            "symbols": np.array(self.symbols[:n], dtype=np.uint8),
        }


class Bits(C.Structure):
    _fields_ = [("bytes", u8p), ("cap", C.c_size_t), ("nbits", C.c_uint64)]


class PpmHeader(C.Structure):
    _fields_ = [("magic", C.c_int), ("width", C.c_uint32), ("height", C.c_uint32), ("maxval", C.c_uint32),
                ("payload", C.c_size_t)]


def _ptr(a: np.ndarray, t):
    return a.ctypes.data_as(t)


class Oracle:
    def __init__(self):
        build()
        L = C.CDLL(str(ORACLE_SO))
        self.L = L
        L.jo_ppm_parse.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(PpmHeader)]
        L.jo_ppm_samples.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(PpmHeader), u8p]
        L.jo_dct_arai.argtypes = L.jo_dct_direct.argtypes = L.jo_dct_matrix.argtypes = [f64p, f64p]
        L.jo_quantize.argtypes = [f64p, u8p, i32p]
        L.jo_zigzag_index.argtypes = [C.c_int]
        L.jo_category.argtypes = [C.c_int, C.POINTER(C.c_int), u32p]
        L.jo_block_symbols.argtypes = [i32p, u8p, u32p, u8p]
        L.jo_huffman_from_text.argtypes = [i32p, C.c_size_t, C.POINTER(HuffTable)]
        L.jo_huffman_from_hist.argtypes = [u32p, u8p, C.c_int, C.POINTER(HuffTable)]
        L.jo_bits_init.argtypes = L.jo_bits_free.argtypes = L.jo_bits_fill.argtypes = [C.POINTER(Bits)]
        L.jo_bits_push_msb.argtypes = L.jo_bits_push_lsb.argtypes = [C.POINTER(Bits), C.c_uint32, C.c_int]
        L.jo_bits_stuffed_size.argtypes = [C.POINTER(Bits)]
        L.jo_bits_stuffed_size.restype = C.c_size_t
        L.jo_bits_write_stuffed.argtypes = [C.POINTER(Bits), u8p]
        L.jo_bits_write_stuffed.restype = C.c_size_t
        L.jo_forward_mcu_rows.argtypes = [u8p, C.c_uint32, C.c_uint32, C.c_uint32, u8p, u8p, C.c_uint32, C.c_uint32, i16p]
        L.jo_forward_planes.argtypes = [u8p, C.c_uint32, C.c_uint32, C.c_uint32, u8p, u8p] + [f64p] * 6 + [i32p] * 3
        L.jo_planes_to_mcu.argtypes = [i32p, i32p, i32p, C.c_uint32, C.c_uint32, i16p]
        L.jo_symbol_stats.argtypes = [i16p, C.c_uint32, C.c_uint32, u32p, u64p]
        L.jo_entropy_encode.argtypes = [i16p, C.c_uint32, C.c_uint32, C.POINTER(HuffTable), C.POINTER(Bits)]
        L.jo_write_headers.argtypes = [C.c_uint32, C.c_uint32, u8p, u8p, C.POINTER(HuffTable), u8p]
        L.jo_write_headers.restype = C.c_size_t
        L.jo_encode_ppm.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(u8p), C.POINTER(C.c_size_t)]
        L.jo_encode_rgb.argtypes = [u8p, C.c_uint32, C.c_uint32, C.POINTER(u8p), C.POINTER(C.c_size_t)]
        L.jo_forward_from_planes.argtypes = [f64p, f64p, f64p, C.c_uint32, C.c_uint32, C.c_int, u8p, u8p, i16p]
        L.jo_encode_planes.argtypes = [f64p, f64p, f64p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(u8p), C.POINTER(C.c_size_t)]
        L.jo_subsample_dims.argtypes = [C.c_int, C.c_uint32, C.c_uint32, u32p, u32p]
        L.jo_subsample_plane.argtypes = [f64p, C.c_uint32, C.c_uint32, C.c_int, f64p]
        L.jo_dct_plane.argtypes = [f64p, C.c_uint32, C.c_uint32, C.c_int, f64p]
        L.jo_dct_basis.argtypes = [f64p]
        L.jo_free.argtypes = [C.c_void_p]
        self.qy = np.ctypeslib.as_array((C.c_uint8 * 64).in_dll(L, "jo_qtable_luma")).copy()
        self.qc = np.ctypeslib.as_array((C.c_uint8 * 64).in_dll(L, "jo_qtable_chroma")).copy()

    # -- PPM ---------------------------------------------------------------------------------
    def ppm_parse(self, data: bytes):
        h = PpmHeader()
        rc = self.L.jo_ppm_parse(data, len(data), C.byref(h))
        return rc, h

    def ppm_load(self, data: bytes):
        rc, h = self.ppm_parse(data)
        if rc:
            raise ValueError(f"jo_ppm_parse rc={rc}")
        rgb = np.empty((h.height, h.width, 3), np.uint8)
        rc = self.L.jo_ppm_samples(data, len(data), C.byref(h), _ptr(rgb, u8p))
        if rc:
            raise ValueError(f"jo_ppm_samples rc={rc}")
        return rgb, int(h.maxval)

    # -- block kernels -----------------------------------------------------------------------
    def dct(self, block, mode="arai"):
        x = np.ascontiguousarray(block, np.float64).reshape(64)
        y = np.empty(64, np.float64)
        getattr(self.L, {"arai": "jo_dct_arai", "direct": "jo_dct_direct", "matrix": "jo_dct_matrix"}[mode])(
            _ptr(x, f64p), _ptr(y, f64p))
        return y.reshape(8, 8)

    def quantize(self, block, table):
        x = np.ascontiguousarray(block, np.float64).reshape(64)
        t = np.ascontiguousarray(table, np.uint8).reshape(64)
        o = np.empty(64, np.int32)
        self.L.jo_quantize(_ptr(x, f64p), _ptr(t, u8p), _ptr(o, i32p))
        return o.reshape(8, 8)

    def zigzag_index(self, i):
        return self.L.jo_zigzag_index(i)

    def category(self, v):
        c, b = C.c_int(), C.c_uint32()
        self.L.jo_category(int(v), C.byref(c), C.byref(b))
        return c.value, b.value

    def block_symbols(self, natural):
        x = np.ascontiguousarray(natural, np.int32).reshape(64)
        s, b, n = np.empty(64, np.uint8), np.empty(64, np.uint32), np.empty(64, np.uint8)
        k = self.L.jo_block_symbols(_ptr(x, i32p), _ptr(s, u8p), _ptr(b, u32p), _ptr(n, u8p))
        return s[:k].copy(), b[:k].copy(), n[:k].copy()

    # -- Huffman -----------------------------------------------------------------------------
    def huffman_from_text(self, text):
        t = np.ascontiguousarray(text, np.int32)
        h = HuffTable()
        self.L.jo_huffman_from_text(_ptr(t, i32p), t.size, C.byref(h))
        return h

    def huffman_from_hist(self, count, order):
        c = np.ascontiguousarray(count, np.uint32)
        o = np.ascontiguousarray(order, np.uint8)
        h = HuffTable()
        self.L.jo_huffman_from_hist(_ptr(c, u32p), _ptr(o, u8p), o.size, C.byref(h))
        return h

    # -- bits --------------------------------------------------------------------------------
    def pack_bits(self, values, nbits, msb_aligned=False, fill=True):
        b = Bits()
        self.L.jo_bits_init(C.byref(b))
        for v, n in zip(values, nbits):
            (self.L.jo_bits_push_msb if msb_aligned else self.L.jo_bits_push_lsb)(C.byref(b), int(v), int(n))
        if fill:
            self.L.jo_bits_fill(C.byref(b))
        out = self._stuffed(b)
        nb = int(b.nbits)
        self.L.jo_bits_free(C.byref(b))
        return out, nb

    def _stuffed(self, b):
        n = self.L.jo_bits_stuffed_size(C.byref(b))
        out = np.empty(n, np.uint8)
        self.L.jo_bits_write_stuffed(C.byref(b), _ptr(out, u8p))
        return out

    # -- image stages ------------------------------------------------------------------------
    @staticmethod
    def geometry(w, h):
        w16, h16 = (w + 15) & ~15, (h + 15) & ~15
        return w16, h16, w16 // 16, h16 // 16

    def forward(self, rgb, maxval=255, qy=None, qc=None, mcu_rows=None):
        """rgb (h,w,3) u8 -> MCU-ordered zigzag int16 coefficients (n_mcu, 6, 64)."""
        rgb = np.ascontiguousarray(rgb, np.uint8)
        h, w, _ = rgb.shape
        _, _, mw, mh = self.geometry(w, h)
        y0, y1 = (0, mh) if mcu_rows is None else mcu_rows
        qy = self.qy if qy is None else np.ascontiguousarray(qy, np.uint8).reshape(64)
        qc = self.qc if qc is None else np.ascontiguousarray(qc, np.uint8).reshape(64)
        out = np.empty(((y1 - y0) * mw, 6, 64), np.int16)
        self.L.jo_forward_mcu_rows(_ptr(rgb, u8p), w, h, maxval, _ptr(qy, u8p), _ptr(qc, u8p), y0, y1, _ptr(out, i16p))
        return out

    def forward_planes(self, rgb, maxval=255):
        rgb = np.ascontiguousarray(rgb, np.uint8)
        h, w, _ = rgb.shape
        w16, h16, _, _ = self.geometry(w, h)
        d = {
            "y": np.empty((h16, w16)), "cb": np.empty((h16 // 2, w16 // 2)), "cr": np.empty((h16 // 2, w16 // 2)),
            "dct_y": np.empty((h16, w16)), "dct_cb": np.empty((h16 // 2, w16 // 2)), "dct_cr": np.empty((h16 // 2, w16 // 2)),
            "q_y": np.empty((h16, w16), np.int32), "q_cb": np.empty((h16 // 2, w16 // 2), np.int32),
            "q_cr": np.empty((h16 // 2, w16 // 2), np.int32),
        }
        self.L.jo_forward_planes(_ptr(rgb, u8p), w, h, maxval, _ptr(self.qy, u8p), _ptr(self.qc, u8p),
                                 *[_ptr(d[k], f64p) for k in ("y", "cb", "cr", "dct_y", "dct_cb", "dct_cr")],
                                 *[_ptr(d[k], i32p) for k in ("q_y", "q_cb", "q_cr")])
        return d

    def planes_to_mcu(self, q_y, q_cb, q_cr):
        q_y, q_cb, q_cr = (np.ascontiguousarray(a, np.int32) for a in (q_y, q_cb, q_cr))
        mh, mw = q_y.shape[0] // 16, q_y.shape[1] // 16
        out = np.empty((mh * mw, 6, 64), np.int16)
        self.L.jo_planes_to_mcu(_ptr(q_y, i32p), _ptr(q_cb, i32p), _ptr(q_cr, i32p), mw, mh, _ptr(out, i16p))
        return out

    def symbol_stats(self, coef, mcu_w, mcu_h):
        coef = np.ascontiguousarray(coef, np.int16)
        count = np.zeros((4, 256), np.uint32)
        first = np.zeros((4, 256), np.uint64)
        self.L.jo_symbol_stats(_ptr(coef, i16p), mcu_w, mcu_h, _ptr(count, u32p), _ptr(first, u64p))
        return count, first

    def entropy_encode(self, coef, mcu_w, mcu_h):
        """-> (tables[4], unstuffed scan bytes, nbits, stuffed scan bytes)"""
        coef = np.ascontiguousarray(coef, np.int16)
        tabs = (HuffTable * 4)()
        b = Bits()
        self.L.jo_bits_init(C.byref(b))
        self.L.jo_entropy_encode(_ptr(coef, i16p), mcu_w, mcu_h, tabs, C.byref(b))
        nbits = int(b.nbits)
        raw = np.ctypeslib.as_array(b.bytes, shape=((nbits + 7) // 8,)).copy()
        stuffed = self._stuffed(b)
        self.L.jo_bits_free(C.byref(b))
        return tabs, raw, nbits, stuffed

    def headers(self, w, h, tabs, qy=None, qc=None):
        qy = self.qy if qy is None else np.ascontiguousarray(qy, np.uint8)
        qc = self.qc if qc is None else np.ascontiguousarray(qc, np.uint8)
        n = self.L.jo_write_headers(w, h, _ptr(qy, u8p), _ptr(qc, u8p), tabs, None)
        out = np.empty(n, np.uint8)
        self.L.jo_write_headers(w, h, _ptr(qy, u8p), _ptr(qc, u8p), tabs, _ptr(out, u8p))
        return out

    def encode_ppm(self, data: bytes) -> bytes:
        out, n = u8p(), C.c_size_t()
        rc = self.L.jo_encode_ppm(data, len(data), C.byref(out), C.byref(n))
        if rc:
            raise ValueError(f"jo_encode_ppm rc={rc}")
        res = C.string_at(out, n.value)
        self.L.jo_free(out)
        return res

    def encode_rgb(self, rgb) -> bytes:
        rgb = np.ascontiguousarray(rgb, np.uint8)
        out, n = u8p(), C.c_size_t()
        self.L.jo_encode_rgb(_ptr(rgb, u8p), rgb.shape[1], rgb.shape[0], C.byref(out), C.byref(n))
        res = C.string_at(out, n.value)
        self.L.jo_free(out)
        return res


    SUBSAMPLING = {"S444": 0, "S422": 1, "S411": 2, "S420": 3, "S420_m": 4, "S420_lm": 5}
    DCT_MODES = {"simple": 0, "matrix": 1, "arai": 2}

    def subsample_plane(self, plane, mode):
        """Image::subsample (src/Image.cpp:198-319) of one plane; mode: a key of SUBSAMPLING"""
        plane = np.ascontiguousarray(plane, np.float64)
        h, w = plane.shape
        ow, oh = C.c_uint32(), C.c_uint32()
        self.L.jo_subsample_dims(self.SUBSAMPLING[mode], w, h, C.byref(ow), C.byref(oh))
        out = np.empty((oh.value, ow.value), np.float64)
        self.L.jo_subsample_plane(_ptr(plane, f64p), w, h, self.SUBSAMPLING[mode], _ptr(out, f64p))
        return out

    def dct_plane(self, plane, mode="arai"):
        """Image::applyDCT (src/Image.cpp:540-595) on one plane whose sides are multiples of 8"""
        plane = np.ascontiguousarray(plane, np.float64)
        h, w = plane.shape
        out = np.empty_like(plane)
        self.L.jo_dct_plane(_ptr(plane, f64p), w, h, self.DCT_MODES[mode], _ptr(out, f64p))
        return out

    def dct_basis(self):
        a = np.empty(64, np.float64)
        self.L.jo_dct_basis(_ptr(a, f64p))
        return a

    def forward_from_planes(self, p0, p1, p2, ycbcr=False):
        """three (H16, W16) float64 planes (Image::R/G/B, or Y/Cb/Cr with ycbcr) -> MCU-ordered zigzag int16 coefficients"""
        pl = [np.ascontiguousarray(p, np.float64) for p in (p0, p1, p2)]
        h16, w16 = pl[0].shape
        out = np.empty(((h16 // 16) * (w16 // 16), 6, 64), np.int16)
        self.L.jo_forward_from_planes(_ptr(pl[0], f64p), _ptr(pl[1], f64p), _ptr(pl[2], f64p), w16, h16, 1 if ycbcr else 0,
                                      _ptr(self.qy, u8p), _ptr(self.qc, u8p), _ptr(out, i16p))
        return out

    def encode_planes(self, p0, p1, p2, real_w, real_h, ycbcr=False) -> bytes:
        pl = [np.ascontiguousarray(p, np.float64) for p in (p0, p1, p2)]
        h16, w16 = pl[0].shape
        out, n = u8p(), C.c_size_t()
        rc = self.L.jo_encode_planes(_ptr(pl[0], f64p), _ptr(pl[1], f64p), _ptr(pl[2], f64p), w16, h16, real_w, real_h, 1 if ycbcr else 0,
                                     C.byref(out), C.byref(n))
        if rc:
            raise ValueError("planes are not the image padded to whole MCUs")
        res = C.string_at(out, n.value)
        self.L.jo_free(out)
        return res


class Reference:
    """The compiled reference (oracle/_ref).  `available()` is False when it was never built."""

    @staticmethod
    def available() -> bool:
        return REF_SO.exists()

    def __init__(self):
        if not REF_SO.exists():
            build()
        L = C.CDLL(str(REF_SO))
        self.L = L
        L.ref_encode_file.argtypes = [C.c_char_p, C.c_char_p, f64p, f64p]
        L.ref_padded_dims.argtypes = [C.c_char_p] + [u32p] * 4
        L.ref_stage_dump.argtypes = [C.c_char_p] + [f64p] * 7 + [i32p] * 3
        L.ref_dct_block.argtypes = [f64p, f64p, C.c_int]
        L.ref_quantize_block.argtypes = [f64p, f64p, i32p]
        L.ref_block_symbols.argtypes = [i32p, u8p, u32p, u8p]
        L.ref_generate_huffman.argtypes = [i32p, C.c_int, u32p, u8p, u8p, u8p]
        L.ref_bitstream_pack.argtypes = [u32p, u8p, C.c_int, C.c_int, u8p, C.c_int, u32p]
        if hasattr(L, "ref_subsample_plane"):
            L.ref_subsample_plane.argtypes = [f64p, C.c_uint32, C.c_uint32, C.c_int, f64p, u32p, u32p]
            L.ref_dct_plane.argtypes = [f64p, C.c_uint32, C.c_uint32, C.c_int, f64p]
        if hasattr(L, "ref_encode_planes"):
            L.ref_encode_planes.argtypes = [f64p, f64p, f64p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_char_p]

    def subsample_plane(self, plane, mode: int):
        plane = np.ascontiguousarray(plane, np.float64)
        h, w = plane.shape
        out = np.empty(h * w, np.float64)
        ow, oh = C.c_uint32(), C.c_uint32()
        assert self.L.ref_subsample_plane(_ptr(plane, f64p), w, h, mode, _ptr(out, f64p), C.byref(ow), C.byref(oh)) == 0
        return out[: ow.value * oh.value].reshape(oh.value, ow.value).copy()

    def dct_plane(self, plane, mode: int):
        plane = np.ascontiguousarray(plane, np.float64)
        h, w = plane.shape
        out = np.empty_like(plane)
        assert self.L.ref_dct_plane(_ptr(plane, f64p), w, h, mode, _ptr(out, f64p)) == 0
        return out

    def encode_planes(self, p0, p1, p2, real_w, real_h, ycbcr, jpg_path: str) -> int:
        """Image::writeJPEG on an Image assembled from three (H16, W16) float64 planes"""
        pl = [np.ascontiguousarray(p, np.float64) for p in (p0, p1, p2)]
        h16, w16 = pl[0].shape
        return self.L.ref_encode_planes(_ptr(pl[0], f64p), _ptr(pl[1], f64p), _ptr(pl[2], f64p), w16, h16, real_w, real_h, 1 if ycbcr else 0,
                                        jpg_path.encode())

    def encode_file(self, ppm_path: str, jpg_path: str):
        lo, en = C.c_double(), C.c_double()
        rc = self.L.ref_encode_file(ppm_path.encode(), jpg_path.encode(), C.byref(lo), C.byref(en))
        return rc, lo.value, en.value

    def padded_dims(self, ppm_path):
        v = [C.c_uint32() for _ in range(4)]
        rc = self.L.ref_padded_dims(ppm_path.encode(), *[C.byref(x) for x in v])
        if rc:
            raise ValueError("reference rejected the file")
        return tuple(x.value for x in v)

    def stage_dump(self, ppm_path):
        w16, h16, _, _ = self.padded_dims(ppm_path)
        d = {
            "rgb": np.empty((3, h16, w16)),
            "y": np.empty((h16, w16)), "cb": np.empty((h16 // 2, w16 // 2)), "cr": np.empty((h16 // 2, w16 // 2)),
            "dct_y": np.empty((h16, w16)), "dct_cb": np.empty((h16 // 2, w16 // 2)), "dct_cr": np.empty((h16 // 2, w16 // 2)),
            "q_y": np.empty((h16, w16), np.int32), "q_cb": np.empty((h16 // 2, w16 // 2), np.int32),
            "q_cr": np.empty((h16 // 2, w16 // 2), np.int32),
        }
        rc = self.L.ref_stage_dump(ppm_path.encode(),
                                   *[_ptr(d[k], f64p) for k in ("rgb", "y", "cb", "cr", "dct_y", "dct_cb", "dct_cr")],
                                   *[_ptr(d[k], i32p) for k in ("q_y", "q_cb", "q_cr")])
        if rc:
            raise ValueError("reference rejected the file")
        return d

    def dct(self, block, mode="arai"):
        x = np.ascontiguousarray(block, np.float64).reshape(64)
        y = np.empty(64)
        self.L.ref_dct_block(_ptr(x, f64p), _ptr(y, f64p), {"direct": 0, "matrix": 1, "arai": 2}[mode])
        return y.reshape(8, 8)

    def quantize(self, block, table):
        x = np.ascontiguousarray(block, np.float64).reshape(64)
        t = np.ascontiguousarray(table, np.float64).reshape(64)
        o = np.empty(64, np.int32)
        self.L.ref_quantize_block(_ptr(x, f64p), _ptr(t, f64p), _ptr(o, i32p))
        return o.reshape(8, 8)

    def block_symbols(self, natural):
        x = np.ascontiguousarray(natural, np.int32).reshape(64)
        s, b, n = np.empty(64, np.uint8), np.empty(64, np.uint32), np.empty(64, np.uint8)
        k = self.L.ref_block_symbols(_ptr(x, i32p), _ptr(s, u8p), _ptr(b, u32p), _ptr(n, u8p))
        return s[:k].copy(), b[:k].copy(), n[:k].copy()

    def huffman(self, text):
        t = np.ascontiguousarray(text, np.int32)
        code, ln = np.zeros(256, np.uint32), np.zeros(256, np.uint8)
        counts, syms = np.zeros(16, np.uint8), np.zeros(256, np.uint8)
        self.L.ref_generate_huffman(_ptr(t, i32p), t.size, _ptr(code, u32p), _ptr(ln, u8p), _ptr(counts, u8p),
                                    _ptr(syms, u8p))
        return {"code_msb": code, "length": ln, "counts": counts, "symbols": syms[: int(counts.sum())]}

    def pack_bits(self, msb_aligned_values, nbits, fill=True):
        v = np.ascontiguousarray(msb_aligned_values, np.uint32)
        n = np.ascontiguousarray(nbits, np.uint8)
        cap = int(n.sum()) // 4 + 64
        out = np.zeros(cap, np.uint8)
        sz = C.c_uint32()
        k = self.L.ref_bitstream_pack(_ptr(v, u32p), _ptr(n, u8p), v.size, int(fill), _ptr(out, u8p), cap, C.byref(sz))
        return out[:k].copy(), sz.value
