"""ctypes binding of the C-ABI in include/jpgenc_b200.h (the drop-in boundary of the encode path).

This is the binding a maintainer of the reference would write for a Python harness; the tests and bench.py call
the CUDA path exclusively through it.  There is no fallback of any kind: if the shared library is missing or no
B200 is visible, construction raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

LIB_PATH = Path(__file__).resolve().parent / "lib" / "libjpgenc_b200.so"

OK = 0
ERR_CUDA, ERR_ARG, ERR_NO_DEVICE, ERR_FORMAT, ERR_IO, ERR_CAPACITY, ERR_NOMEM = -1, -2, -3, -4, -5, -6, -7

# JPGENC_PIXEL_*: name -> (code, bytes per pixel); a GRAY pixel v is encoded as the pixel (v, v, v)
PIXEL_FORMATS = {"RGB": (0, 3), "BGR": (1, 3), "RGBA": (2, 4), "BGRA": (3, 4), "GRAY": (16, 1)}
# YUV 4:2:0 frames (JPGENC_YUV_*): Y, U, V planes / Y plane and interleaved UV plane
YUV_LAYOUTS = {"I420": 0, "NV12": 1}
# every JPGENC_YUV_* layout: 4:2:0 as above; 4:2:2 planar (I422), semi-planar (NV16) and packed (YUYV, UYVY); 4:4:4 planar (I444)
YUV_FORMATS = {"I420": 0, "NV12": 1, "I422": 2, "NV16": 3, "I444": 4, "YUYV": 5, "UYVY": 6}

u8p = C.POINTER(C.c_uint8)
i16p = C.POINTER(C.c_int16)
i32p = C.POINTER(C.c_int32)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
f32p = C.POINTER(C.c_float)
f64p = C.POINTER(C.c_double)


class HuffTable(C.Structure):
    _fields_ = [
        ("code_msb", C.c_uint32 * 256),
        ("length", C.c_uint8 * 256),
        ("counts", C.c_uint8 * 16),
        ("symbols", C.c_uint8 * 256),
        ("nsymbols", C.c_int32),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("real_w", C.c_uint32), ("real_h", C.c_uint32), ("mcu_w", C.c_uint32), ("mcu_h", C.c_uint32),
        ("n_blocks", C.c_uint64), ("refined_blocks", C.c_uint64), ("scan_bits", C.c_uint64),
        ("scan_bytes", C.c_uint64), ("stuffed_ff", C.c_uint64),
        ("ms_k1", C.c_float), ("ms_forward", C.c_float), ("ms_stats", C.c_float), ("ms_entropy", C.c_float),
        ("ms_h2d", C.c_float), ("ms_d2h", C.c_float),
        ("sum_ms_k1", C.c_double), ("sum_ms_forward", C.c_double), ("sum_ms_stats", C.c_double), ("sum_ms_entropy", C.c_double),
        ("timed_encodes", C.c_uint64),
    ]


# every symbol the header declares: name -> (restype, argtypes)
_SIGNATURES = {
    "jpgenc_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "jpgenc_destroy": (None, [C.c_void_p]),
    "jpgenc_last_error": (C.c_char_p, [C.c_void_p]),
    "jpgenc_stream": (C.c_void_p, [C.c_void_p]),
    "jpgenc_synchronize": (C.c_int, [C.c_void_p]),
    "jpgenc_get_stats": (C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    "jpgenc_set_qtables": (C.c_int, [C.c_void_p, u8p, u8p]),
    "jpgenc_set_dct_constants": (C.c_int, [C.c_void_p, f64p, f64p]),
    "jpgenc_upload_rgb": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]),
    "jpgenc_bind_device_rgb": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]),
    "jpgenc_bind_device_image": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32]),
    "jpgenc_bind_device_planar": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]),
    "jpgenc_encode_planar": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                       C.c_void_p, C.c_uint64, u64p]),
    "jpgenc_bind_device_yuv420": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                            C.c_int]),
    "jpgenc_encode_yuv420": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int,
                                       C.c_void_p, C.c_uint64, u64p]),
    "jpgenc_bind_device_yuv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                         C.c_int]),
    "jpgenc_encode_yuv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int,
                                    C.c_void_p, C.c_uint64, u64p]),
    "jpgenc_encode_image": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32, C.c_void_p, C.c_uint64,
                                      u64p]),
    "jpgenc_color_dct_quant": (C.c_int, [C.c_void_p]),
    "jpgenc_get_coefficients": (C.c_int, [C.c_void_p, i16p]),
    "jpgenc_set_coefficients": (C.c_int, [C.c_void_p, i32p, i32p, i32p, C.c_uint32, C.c_uint32]),
    "jpgenc_set_coefficients_mcu": (C.c_int, [C.c_void_p, i16p, C.c_uint32, C.c_uint32]),
    "jpgenc_symbol_stats": (C.c_int, [C.c_void_p, u32p, u64p]),
    "jpgenc_set_stage_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "jpgenc_build_huffman": (C.c_int, [u32p, u64p, C.POINTER(HuffTable)]),
    "jpgenc_build_huffman_containers": (C.c_int, [u32p, u64p, C.POINTER(HuffTable)]),
    "jpgenc_build_huffman_arrays": (C.c_int, [u32p, u64p, C.POINTER(HuffTable)]),
    "jpgenc_build_huffman_device": (C.c_int, [C.c_void_p, C.c_uint32, u32p, u64p, C.POINTER(HuffTable)]),
    "jpgenc_entropy_encode": (C.c_int, [C.c_void_p, C.POINTER(HuffTable), u64p]),
    "jpgenc_download_scan": (C.c_int, [C.c_void_p, u8p, C.c_uint64]),
    "jpgenc_ppm_info": (C.c_int, [C.c_char_p, C.c_size_t, u32p, u32p, u32p, C.POINTER(C.c_int), C.POINTER(C.c_size_t)]),
    "jpgenc_ppm_samples": (C.c_int, [C.c_char_p, C.c_size_t, u8p]),
    "jpgenc_write_headers": (C.c_size_t, [C.c_uint32, C.c_uint32, u8p, u8p, C.POINTER(HuffTable), u8p]),
    "jpgenc_encode_bound": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, u64p]),
    "jpgenc_assemble_last": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, u64p]),
    "jpgenc_encode_rgb": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64, u64p]),
    "jpgenc_encode_planes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int,
                                       C.c_void_p, C.c_uint64, u64p]),
    "jpgenc_encode_ppm_file": (C.c_int, [C.c_void_p, C.c_char_p, C.c_char_p]),
    "jpgenc_debug_counter": (C.c_int, [C.c_void_p, C.c_int, u32p]),
    "jpgenc_stage_subsample_dims": (C.c_int, [C.c_int, C.c_uint32, C.c_uint32, u32p, u32p]),
    "jpgenc_stage_subsample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]),
    "jpgenc_stage_dct": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]),
    "jpgenc_dct_quant_blocks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, u8p, u64p]),
    "jpgenc_bind_host_to_device_numa": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "jpgenc_dev_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "jpgenc_dev_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "jpgenc_host_alloc_pinned": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "jpgenc_host_free_pinned": (C.c_int, [C.c_void_p]),
    "jpgenc_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "jpgenc_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "jpgenc_synth_rgb": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]),
    "jpgenc_synth_blocks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "jpgenc_flush_l2": (C.c_int, [C.c_void_p]),
    "jpgenc_timer_begin": (C.c_int, [C.c_void_p]),
    "jpgenc_timer_end": (C.c_int, [C.c_void_p, f32p]),
    "jpgenc_launch_count": (C.c_uint64, [C.c_void_p]),
    "jpgenc_encode_frames_device": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_uint32,
                                              C.POINTER(C.c_void_p), u64p, u64p]),
    "jpgenc_encode_frames": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_uint32,
                                       C.POINTER(C.c_void_p), u64p, u64p]),
    "jpgenc_encode_frames_packed": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.c_int, C.c_uint32, C.c_uint32, C.c_uint32,
                                              C.c_void_p, C.c_uint64, u64p, u64p, u64p]),
    "jpgenc_encode_images_packed": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.c_int, u32p, u32p, C.c_uint32,
                                              C.c_void_p, C.c_uint64, u64p, u64p, u64p]),
    "jpgenc_encode_images_packed_layout": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.c_int, u32p, u32p, u32p, C.c_int,
                                                     C.c_uint32, C.c_void_p, C.c_uint64, u64p, u64p, u64p]),
    "jpgenc_encode_images_packed_planar": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.c_int, u32p, u32p, u32p, C.c_uint32,
                                                     C.c_void_p, C.c_uint64, u64p, u64p, u64p]),
    "jpgenc_encode_images_packed_yuv420": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.c_int, u32p, u32p, u32p, u32p, C.c_int,
                                                     C.c_void_p, C.c_uint64, u64p, u64p, u64p]),
    "jpgenc_encode_images_packed_yuv": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.c_int, u32p, u32p, u32p, u32p, C.c_int,
                                                  C.c_void_p, C.c_uint64, u64p, u64p, u64p]),
    "jpgenc_batch_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "jpgenc_batch_destroy": (None, [C.c_void_p]),
    "jpgenc_batch_last_error": (C.c_char_p, [C.c_void_p]),
    "jpgenc_batch_set_qtables": (C.c_int, [C.c_void_p, u8p, u8p]),
    "jpgenc_batch_encode": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_uint32,
                                      C.POINTER(C.c_void_p), u64p, u64p]),
    "jpgenc_batch_encode_device": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_uint32,
                                             C.POINTER(C.c_void_p), u64p, u64p]),
}

_lib = None


def load_library() -> C.CDLL:
    """Load libjpgenc_b200.so and bind every declared symbol; raises if the library was not built."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError(f"{LIB_PATH} is missing: run `make` (or __graft_entry__.build()); there is no fallback path")
        lib = C.CDLL(str(LIB_PATH))
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError here == the library does not export a declared symbol
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


class JpgencError(RuntimeError):
    def __init__(self, code: int, text: str):
        super().__init__(f"jpgenc error {code}: {text}")
        self.code = code


def _np_ptr(a: np.ndarray, t):
    return a.ctypes.data_as(t)


def _format_code(fmt) -> int:
    """'RGB' / 'BGR' / 'RGBA' / 'BGRA' (or a JPGENC_PIXEL_* code) -> the code"""
    if isinstance(fmt, str):
        if fmt not in PIXEL_FORMATS:
            raise ValueError(f"unknown pixel format {fmt!r}")
        return PIXEL_FORMATS[fmt][0]
    return int(fmt)


def image_layout(a: np.ndarray, fmt: str = "RGB"):
    """(pointer, width, height, row pitch) of a uint8 (H, W, C) array whose strides are (pitch, C, 1) with C the format's
    bytes per pixel -- a tight array or a view such as big[y0:y1, x0:x1]; GRAY: a uint8 (H, W) array with strides (pitch, 1).
    Anything else raises ValueError: the pixels are read where they are, never copied."""
    if fmt not in PIXEL_FORMATS:
        raise ValueError(f"unknown pixel format {fmt!r}")
    bpp = PIXEL_FORMATS[fmt][1]
    if fmt == "GRAY":
        if not isinstance(a, np.ndarray) or a.dtype != np.uint8 or a.ndim != 2 or a.size == 0:
            raise ValueError("GRAY pixels must be a uint8 array of shape (H, W)")
        h, w = a.shape
        pitch = a.strides[0] if h > 1 else w
        if (w > 1 and a.strides[1] != 1) or pitch < w:
            raise ValueError(f"GRAY pixels must have strides (pitch, 1) with pitch >= {w}; got {a.strides}")
        return a.ctypes.data, w, h, pitch
    if not isinstance(a, np.ndarray) or a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != bpp:
        raise ValueError(f"{fmt} pixels must be a uint8 array of shape (H, W, {bpp})")
    h, w, _ = a.shape
    pitch = a.strides[0] if h > 1 else w * bpp
    if a.strides[2] != 1 or (w > 1 and a.strides[1] != bpp) or pitch < w * bpp:
        raise ValueError(f"{fmt} pixels must have strides (pitch, {bpp}, 1) with pitch >= {w * bpp}; got {a.strides}")
    return a.ctypes.data, w, h, pitch


def tensor_layout(t, order: str = "RGB"):
    """How a torch uint8 image tensor is read in place: (fmt, pointers, width, height, row pitch in bytes).

    fmt is "planar" (pointers = the R, G, B planes) or a PIXEL_FORMATS name (one pointer).  Accepted:
      (3, H, W) with stride(2) == 1     planar, one plane per channel (crop views t[:, y0:y1, x0:x1] too);
                                        a channel stride of 0 (g.expand(3, H, W)) is GRAY
      (3, H, W) in channels_last        interleaved RGB (strides (1, pitch, 3))
      (H, W, 3) / (H, W, 4)             interleaved RGB / RGBA with strides (pitch, C, 1)
      (H, W), (1, H, W)                 GRAY with strides (pitch, 1)
    order="BGR" reads the channels as B, G, R (BGR / BGRA, or the planes in that order).  Anything else raises ValueError;
    nothing is ever copied.  Pure: only the tensor's metadata is read."""
    if order not in ("RGB", "BGR"):
        raise ValueError(f"order must be 'RGB' or 'BGR', not {order!r}")
    if type(t).__module__.split(".")[0] != "torch" or not hasattr(t, "stride"):
        raise ValueError("expected a torch.Tensor")
    if str(t.dtype) != "torch.uint8":
        raise ValueError(f"image tensors must be uint8, not {t.dtype}")
    if t.numel() == 0:
        raise ValueError("empty image tensor")
    shape, stride, base = tuple(t.shape), tuple(t.stride()), t.data_ptr()

    def plane(h, w, sh, sw):                  # (H, W) with strides (sh, sw): the row pitch of one byte per pixel, or None
        if w > 1 and sw != 1:
            return None
        pitch = sh if h > 1 else w
        return pitch if pitch >= w else None

    if len(shape) == 2 or (len(shape) == 3 and shape[0] == 1):
        h, w = shape[-2:]
        pitch = plane(h, w, stride[-2], stride[-1])
        if pitch is not None:
            return "GRAY", (base,), w, h, pitch
    elif len(shape) == 3 and shape[0] == 3:
        _, h, w = shape
        pitch = plane(h, w, stride[1], stride[2])
        if pitch is not None:
            if stride[0] == 0:
                return "GRAY", (base,), w, h, pitch
            ptrs = tuple(base + k * stride[0] for k in range(3))
            return "planar", ptrs[::-1] if order == "BGR" else ptrs, w, h, pitch
        pitch = stride[1] if h > 1 else 3 * w
        if stride[0] == 1 and (w == 1 or stride[2] == 3) and pitch >= 3 * w:
            return order, (base,), w, h, pitch
    elif len(shape) == 3 and shape[2] in (3, 4):
        h, w, c = shape
        pitch = stride[0] if h > 1 else c * w
        if stride[2] == 1 and (w == 1 or stride[1] == c) and pitch >= c * w:
            return order + ("A" if c == 4 else ""), (base,), w, h, pitch
    raise ValueError(f"cannot read a tensor of shape {shape} and strides {stride} in place: expected (3, H, W) planes, (3, H, W) "
                     "channels_last, (H, W, 3|4) with strides (pitch, C, 1), or (H, W) / (1, H, W) grey")


def _u8_plane(a, what: str):
    """(pointer, shape, strides in bytes) of a uint8 numpy array or torch tensor (metadata only)"""
    if isinstance(a, np.ndarray):
        if a.dtype != np.uint8:
            raise ValueError(f"{what} must be uint8, not {a.dtype}")
        ptr, shape, strides = a.ctypes.data, tuple(a.shape), tuple(a.strides)
    elif type(a).__module__.split(".")[0] == "torch" and hasattr(a, "stride"):
        if str(a.dtype) != "torch.uint8":
            raise ValueError(f"{what} must be uint8, not {a.dtype}")
        ptr, shape, strides = a.data_ptr(), tuple(a.shape), tuple(a.stride())
    else:
        raise ValueError(f"{what} must be a numpy array or a torch tensor")
    if 0 in shape:
        raise ValueError(f"{what} is empty")
    return ptr, shape, strides


def yuv420_layout(y, u, v=None):
    """How a YUV 4:2:0 frame is read in place: (layout, (y, u, v or 0) pointers, width, height, y_pitch, c_pitch).

    y, u, v are uint8 numpy arrays or torch tensors.  Accepted, for a frame of H x W and ch = ceil(H/2), cw = ceil(W/2):
      Y                        (H, W) with strides (y_pitch, 1)
      I420 (v given)           U and V (ch, cw), strides (c_pitch, 1) with one c_pitch for both
      NV12 (v is None)         UV (ch, cw, 2) with strides (c_pitch, 2, 1), or (ch, 2 cw) with strides (c_pitch, 1)
    Anything else raises ValueError; nothing is ever copied.  Pure: only the metadata is read."""
    yp, ys, yst = _u8_plane(y, "Y")
    if len(ys) != 2:
        raise ValueError(f"Y must be (H, W), not {ys}")
    h, w = ys
    y_pitch = yst[0] if h > 1 else w
    if (w > 1 and yst[1] != 1) or y_pitch < w:
        raise ValueError(f"Y must have strides (pitch, 1) with pitch >= {w}; got {yst}")
    ch, cw = (h + 1) // 2, (w + 1) // 2
    up, us, ust = _u8_plane(u, "U")
    if v is None:
        if us == (ch, cw, 2):
            ok = (cw == 1 or ust[1] == 2) and ust[2] == 1
        elif us == (ch, 2 * cw):
            ok = ust[1] == 1
        else:
            raise ValueError(f"NV12 UV must be ({ch}, {cw}, 2) or ({ch}, {2 * cw}) for a {h} x {w} frame, not {us}")
        c_pitch = ust[0] if ch > 1 else 2 * cw
        if not ok or c_pitch < 2 * cw:
            raise ValueError(f"NV12 UV must have strides (pitch, 2, 1) or (pitch, 1) with pitch >= {2 * cw}; got {ust}")
        return "NV12", (yp, up, 0), w, h, y_pitch, c_pitch
    vp, vs, vst = _u8_plane(v, "V")
    pitches = []
    for name, shape, st in (("U", us, ust), ("V", vs, vst)):
        if shape != (ch, cw):
            raise ValueError(f"I420 {name} must be ({ch}, {cw}) for a {h} x {w} frame, not {shape}")
        pitch = st[0] if ch > 1 else cw
        if (cw > 1 and st[1] != 1) or pitch < cw:
            raise ValueError(f"I420 {name} must have strides (pitch, 1) with pitch >= {cw}; got {st}")
        pitches.append(pitch)
    if pitches[0] != pitches[1]:
        raise ValueError(f"I420 U and V must share one row stride; got {pitches[0]} and {pitches[1]}")
    return "I420", (yp, up, vp), w, h, y_pitch, pitches[0]


def _pitched(name, shape, st, rows, row):
    """the row pitch of a (rows, row) uint8 plane with strides (pitch, 1); ValueError otherwise"""
    if shape != (rows, row):
        raise ValueError(f"{name} must be ({rows}, {row}), not {shape}")
    pitch = st[0] if rows > 1 else row
    if (row > 1 and st[1] != 1) or pitch < row:
        raise ValueError(f"{name} must have strides (pitch, 1) with pitch >= {row}; got {st}")
    return pitch


def _pairs(name, shape, st, rows, n, k):
    """the row pitch of a plane of `rows` rows of n groups of k bytes: (rows, n, k) with strides (pitch, k, 1) or (rows, n k) with
    strides (pitch, 1); ValueError otherwise"""
    if shape == (rows, n, k):
        ok = (n == 1 or st[1] == k) and st[2] == 1
    elif shape == (rows, n * k):
        ok = st[1] == 1
    else:
        raise ValueError(f"{name} must be ({rows}, {n}, {k}) or ({rows}, {n * k}), not {shape}")
    pitch = st[0] if rows > 1 else n * k
    if not ok or pitch < n * k:
        raise ValueError(f"{name} must have strides (pitch, {k}, 1) or (pitch, 1) with pitch >= {n * k}; got {st}")
    return pitch


def yuv_layout(layout, y, u=None, v=None, w=None):
    """How a YUV frame in the named layout (a YUV_FORMATS key) is read in place: (layout, (y, u or 0, v or 0) pointers, width,
    height, y_pitch, c_pitch).

    y, u, v are uint8 numpy arrays or torch tensors.  For a frame of H x W and cw = ceil(W/2):
      I420, NV12               as yuv420_layout (NV12: v is None)
      I422 (YV16: u, v swapped) Y (H, W), U and V (H, cw), strides (pitch, 1), one c_pitch for U and V
      NV16                     Y (H, W); UV (H, cw, 2) with strides (c_pitch, 2, 1), or (H, 2 cw) with strides (c_pitch, 1); v None
      I444                     Y, U, V (H, W), strides (pitch, 1), one c_pitch for U and V
      YUYV, UYVY               one packed plane y, (H, 4 cw) with strides (pitch, 1) or (H, cw, 4) with strides (pitch, 4, 1);
                               u and v None; c_pitch 0.  The width is 2 cw unless w says 2 cw - 1 (the last group's second Y
                               is then not read).
    w, where given, must be the width the planes describe.  Anything else raises ValueError; nothing is ever copied.  Pure: only
    the metadata is read."""
    if layout not in YUV_FORMATS:
        raise ValueError(f"unknown YUV layout {layout!r}; expected one of {sorted(YUV_FORMATS)}")
    if layout in ("YUYV", "UYVY"):
        if u is not None or v is not None:
            raise ValueError(f"{layout} is one packed plane: u and v must be None")
        yp, ys, yst = _u8_plane(y, layout)
        if len(ys) not in (2, 3):
            raise ValueError(f"{layout} must be (H, 4 cw) or (H, cw, 4), not {ys}")
        cw = ys[1] if len(ys) == 3 else ys[1] // 4
        if cw == 0 or (len(ys) == 2 and ys[1] % 4):
            raise ValueError(f"{layout} rows must be whole groups of 4 bytes; got {ys}")
        h = ys[0]
        pitch = _pairs(layout, ys, yst, h, cw, 4)
        width = 2 * cw if w is None else w
        if width not in (2 * cw, 2 * cw - 1):
            raise ValueError(f"{layout} rows of {cw} groups hold {2 * cw - 1} or {2 * cw} pixels, not {width}")
        return layout, (yp, 0, 0), width, h, pitch, 0
    if layout in ("I420", "NV12"):
        if (layout == "NV12") != (v is None):
            raise ValueError(f"{layout} takes {'Y and UV (v None)' if layout == 'NV12' else 'Y, U and V'}")
        got = yuv420_layout(y, u, v)
    else:
        yp, ys, yst = _u8_plane(y, "Y")
        if len(ys) != 2:
            raise ValueError(f"Y must be (H, W), not {ys}")
        h, width = ys
        y_pitch = _pitched("Y", ys, yst, h, width)
        cw = width if layout == "I444" else (width + 1) // 2
        if u is None:
            raise ValueError(f"{layout} needs its chroma plane(s)")
        up, us, ust = _u8_plane(u, "U")
        if layout == "NV16":
            if v is not None:
                raise ValueError("NV16 takes its UV plane as u; v must be None")
            got = ("NV16", (yp, up, 0), width, h, y_pitch, _pairs("NV16 UV", us, ust, h, cw, 2))
        else:
            if v is None:
                raise ValueError(f"{layout} takes Y, U and V")
            vp, vs, vst = _u8_plane(v, "V")
            pu, pv = _pitched(f"{layout} U", us, ust, h, cw), _pitched(f"{layout} V", vs, vst, h, cw)
            if pu != pv:
                raise ValueError(f"{layout} U and V must share one row stride; got {pu} and {pv}")
            got = (layout, (yp, up, vp), width, h, y_pitch, pu)
    if w is not None and w != got[2]:
        raise ValueError(f"w = {w}, but the planes describe a frame {got[2]} wide")
    return got


class Encoder:
    """One GPU context (= one CUDA stream + its device buffers).  Methods mirror the C-ABI one to one."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.jpgenc_create(device, C.byref(h))
        if rc != OK:
            raise JpgencError(rc, (self.lib.jpgenc_last_error(None) or b"").decode())
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.jpgenc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != OK:
            raise JpgencError(rc, (self.lib.jpgenc_last_error(self.h) or b"").decode())

    # ---- parameters -----------------------------------------------------------------------------
    def set_stage_timing(self, level: int):
        """0: no event records between the kernels (default); 1: around the K1 fast kernel; 2: around every stage -- what fills
        stats().ms_k1 / ms_forward / ms_stats / ms_entropy and their running sums"""
        self._check(self.lib.jpgenc_set_stage_timing(self.h, int(level)))

    def set_qtables(self, qy, qc):
        qy = np.ascontiguousarray(qy, np.uint8).reshape(64)
        qc = np.ascontiguousarray(qc, np.uint8).reshape(64)
        self._check(self.lib.jpgenc_set_qtables(self.h, _np_ptr(qy, u8p), _np_ptr(qc, u8p)))

    # ---- input ----------------------------------------------------------------------------------
    def upload_rgb(self, rgb: np.ndarray, maxval: int = 255):
        rgb = np.ascontiguousarray(rgb, np.uint8)
        h, w, _ = rgb.shape
        self._check(self.lib.jpgenc_upload_rgb(self.h, rgb.ctypes.data, w, h, maxval))

    def upload_rgb_ptr(self, host_ptr: int, w: int, h: int, maxval: int = 255):
        self._check(self.lib.jpgenc_upload_rgb(self.h, host_ptr, w, h, maxval))

    def bind_device_rgb(self, dev_ptr: int, w: int, h: int, maxval: int = 255):
        self._check(self.lib.jpgenc_bind_device_rgb(self.h, dev_ptr, w, h, maxval))

    def bind_device_image(self, dev_ptr: int, w: int, h: int, pitch: int = 0, fmt="RGB", maxval: int = 255):
        """device pixels in format fmt ('RGB', 'BGR', 'RGBA', 'BGRA', 'GRAY'), rows `pitch` bytes apart (0: tight)"""
        self._check(self.lib.jpgenc_bind_device_image(self.h, dev_ptr, w, h, pitch, _format_code(fmt), maxval))

    def bind_device_planar(self, r: int, g: int, b: int, w: int, h: int, pitch: int = 0, maxval: int = 255):
        """planar RGB in device memory: three planes of one byte per pixel, rows `pitch` bytes apart (0: tight)"""
        self._check(self.lib.jpgenc_bind_device_planar(self.h, r, g, b, w, h, pitch, maxval))

    # ---- stages ---------------------------------------------------------------------------------
    def bind_device_yuv(self, layout: str, y: int, u: int | None, v: int | None, w: int, h: int, y_pitch: int = 0, c_pitch: int = 0):
        """a YUV frame of any YUV_FORMATS layout in device memory (plane pointers; None where the layout has no such plane)"""
        self._check(self.lib.jpgenc_bind_device_yuv(self.h, y, u or None, v or None, w, h, y_pitch, c_pitch, YUV_FORMATS[layout]))

    def bind_device_yuv420(self, y: int, u: int, v: int | None, w: int, h: int, y_pitch: int = 0, c_pitch: int = 0, layout: str = "I420"):
        """a YUV 4:2:0 frame in device memory (plane pointers; NV12: v None, u the UV plane; pitches 0: tight)"""
        self._check(self.lib.jpgenc_bind_device_yuv420(self.h, y, u, v or None, w, h, y_pitch, c_pitch, YUV_LAYOUTS[layout]))

    def color_dct_quant(self):
        self._check(self.lib.jpgenc_color_dct_quant(self.h))

    def get_coefficients(self) -> np.ndarray:
        st = self.stats()
        out = np.empty((st.n_blocks // 6, 6, 64), np.int16)
        self._check(self.lib.jpgenc_get_coefficients(self.h, _np_ptr(out, i16p)))
        return out

    def set_coefficients(self, q_y, q_cb, q_cr):
        q_y, q_cb, q_cr = (np.ascontiguousarray(a, np.int32) for a in (q_y, q_cb, q_cr))
        mh, mw = q_y.shape[0] // 16, q_y.shape[1] // 16
        self._check(self.lib.jpgenc_set_coefficients(self.h, _np_ptr(q_y, i32p), _np_ptr(q_cb, i32p), _np_ptr(q_cr, i32p), mw, mh))

    def set_coefficients_mcu(self, coef, mcu_w, mcu_h):
        coef = np.ascontiguousarray(coef, np.int16)
        assert coef.size == mcu_w * mcu_h * 6 * 64
        self._check(self.lib.jpgenc_set_coefficients_mcu(self.h, _np_ptr(coef, i16p), mcu_w, mcu_h))

    def symbol_stats(self):
        count = np.zeros((4, 256), np.uint32)
        first = np.zeros((4, 256), np.uint64)
        self._check(self.lib.jpgenc_symbol_stats(self.h, _np_ptr(count, u32p), _np_ptr(first, u64p)))
        return count, first

    def build_huffman(self, count, first):
        tabs = (HuffTable * 4)()
        for t in range(4):
            c = np.ascontiguousarray(count[t], np.uint32)
            f = np.ascontiguousarray(first[t], np.uint64)
            rc = self.lib.jpgenc_build_huffman(_np_ptr(c, u32p), _np_ptr(f, u64p), C.byref(tabs[t]))
            if rc != OK:
                raise JpgencError(rc, f"jpgenc_build_huffman(table {t})")
        return tabs

    def build_huffman_device(self, count, first):
        """n tables at once on the device: count (n, 256) u32, first (n, 256) u64 -> HuffTable array"""
        c = np.ascontiguousarray(count, np.uint32).reshape(-1, 256)
        f = np.ascontiguousarray(first, np.uint64).reshape(-1, 256)
        n = c.shape[0]
        tabs = (HuffTable * n)()
        self._check(self.lib.jpgenc_build_huffman_device(self.h, n, _np_ptr(c, u32p), _np_ptr(f, u64p), tabs))
        return tabs

    def entropy_encode(self, tabs) -> int:
        n = C.c_uint64()
        self._check(self.lib.jpgenc_entropy_encode(self.h, tabs, C.byref(n)))
        return n.value

    def download_scan(self) -> np.ndarray:
        n = self.stats().scan_bytes
        out = np.empty(n, np.uint8)
        self._check(self.lib.jpgenc_download_scan(self.h, _np_ptr(out, u8p), n))
        return out

    def headers(self, tabs, w, h, qy, qc) -> np.ndarray:
        qy = np.ascontiguousarray(qy, np.uint8).reshape(64)
        qc = np.ascontiguousarray(qc, np.uint8).reshape(64)
        n = self.lib.jpgenc_write_headers(w, h, _np_ptr(qy, u8p), _np_ptr(qc, u8p), tabs, None)
        out = np.empty(n, np.uint8)
        self.lib.jpgenc_write_headers(w, h, _np_ptr(qy, u8p), _np_ptr(qc, u8p), tabs, _np_ptr(out, u8p))
        return out

    # ---- whole image ----------------------------------------------------------------------------
    def encode_bound(self, out: np.ndarray | None = None) -> int:
        n = C.c_uint64()
        if out is None:
            self._check(self.lib.jpgenc_encode_bound(self.h, None, 0, C.byref(n)))
        else:
            self._check(self.lib.jpgenc_encode_bound(self.h, out.ctypes.data, out.size, C.byref(n)))
        return n.value

    def _file(self, encode, cap: int) -> bytes:
        """encode(out_ptr, cap, byref(size)) -> rc of a call that writes one file; the buffer grows to the size it reports when
        it is too small"""
        while True:
            out = np.empty(cap, np.uint8)
            n = C.c_uint64()
            rc = encode(out.ctypes.data, cap, C.byref(n))
            if rc == ERR_CAPACITY:
                cap = int(n.value) + 16
                continue
            self._check(rc)
            return out[: n.value].tobytes()

    def encode_rgb(self, rgb: np.ndarray, maxval: int = 255) -> bytes:
        rgb = np.ascontiguousarray(rgb, np.uint8)
        h, w, _ = rgb.shape
        return self._file(lambda out, cap, n: self.lib.jpgenc_encode_rgb(self.h, rgb.ctypes.data, w, h, maxval, out, cap, n),
                          max(4096, rgb.size // 2 + 4096))

    def encode_image(self, arr: np.ndarray, fmt: str = "RGB", maxval: int = 255) -> bytes:
        """host pixels in format fmt: a uint8 (H, W, 3 or 4) array with strides (pitch, C, 1), e.g. a crop view of a larger
        image (see image_layout) -> JPEG bytes"""
        ptr, w, h, pitch = image_layout(arr, fmt)
        code = _format_code(fmt)
        return self._file(lambda out, cap, n: self.lib.jpgenc_encode_image(self.h, ptr, w, h, pitch, code, maxval, out, cap, n),
                          max(4096, w * h * 3 // 2 + 4096))

    def encode_planar(self, r: int, g: int, b: int, w: int, h: int, pitch: int = 0, maxval: int = 255) -> bytes:
        """planar RGB in host memory (three plane pointers, one row pitch; 0: tight) -> JPEG bytes"""
        return self._file(lambda out, cap, n: self.lib.jpgenc_encode_planar(self.h, r, g, b, w, h, pitch, maxval, out, cap, n),
                          max(4096, w * h * 3 // 2 + 4096))

    def encode_yuv420_ptr(self, y: int, u: int, v: int | None, w: int, h: int, y_pitch: int = 0, c_pitch: int = 0,
                          layout: str = "I420") -> bytes:
        """a YUV 4:2:0 frame in host memory (plane pointers, see bind_device_yuv420) -> JPEG bytes"""
        code = YUV_LAYOUTS[layout]
        return self._file(lambda out, cap, n: self.lib.jpgenc_encode_yuv420(self.h, y, u, v or None, w, h, y_pitch, c_pitch, code, out, cap, n),
                          max(4096, w * h * 3 // 2 + 4096))

    def encode_yuv_ptr(self, layout: str, y: int, u: int | None, v: int | None, w: int, h: int, y_pitch: int = 0, c_pitch: int = 0) -> bytes:
        """a YUV frame of any YUV_FORMATS layout in host memory (plane pointers, see bind_device_yuv) -> JPEG bytes"""
        code = YUV_FORMATS[layout]
        return self._file(lambda out, cap, n: self.lib.jpgenc_encode_yuv(self.h, y, u or None, v or None, w, h, y_pitch, c_pitch, code, out, cap, n),
                          max(4096, w * h * 3 // 2 + 4096))

    def encode_planes(self, p0: np.ndarray, p1: np.ndarray, p2: np.ndarray, real_w: int, real_h: int, ycbcr: bool = False) -> bytes:
        """three (H16, W16) float64 planes as the reference's Image holds them -> JPEG bytes (exact FP64 path for every block)"""
        planes = [np.ascontiguousarray(p, np.float64) for p in (p0, p1, p2)]
        h16, w16 = planes[0].shape
        n = C.c_uint64()
        self._check(self.lib.jpgenc_encode_planes(self.h, planes[0].ctypes.data, planes[1].ctypes.data, planes[2].ctypes.data, w16, h16, real_w, real_h,
                                                  1 if ycbcr else 0, None, 0, C.byref(n)))
        out = np.empty(n.value, np.uint8)
        self._check(self.lib.jpgenc_assemble_last(self.h, out.ctypes.data, out.size, C.byref(n)))
        return out[: n.value].tobytes()

    def debug_counter(self, index: int) -> int:
        v = C.c_uint32()
        self._check(self.lib.jpgenc_debug_counter(self.h, index, C.byref(v)))
        return v.value

    def stage_subsample(self, plane: np.ndarray, mode: int) -> np.ndarray:
        """Image::applySubsampling(mode) on one plane of doubles (mode = order of Image::SubsamplingMode)"""
        plane = np.ascontiguousarray(plane, np.float64)
        h, w = plane.shape
        ow, oh = C.c_uint32(), C.c_uint32()
        self._check(self.lib.jpgenc_stage_subsample_dims(mode, w, h, C.byref(ow), C.byref(oh)))
        out = np.empty((oh.value, ow.value), np.float64)
        self._check(self.lib.jpgenc_stage_subsample(self.h, plane.ctypes.data, w, h, mode, out.ctypes.data))
        return out

    def stage_dct(self, plane: np.ndarray, mode: int) -> np.ndarray:
        """Image::applyDCT(mode) on one plane of doubles (mode 0 Simple, 1 Matrix, 2 Arai)"""
        plane = np.ascontiguousarray(plane, np.float64)
        h, w = plane.shape
        out = np.empty_like(plane)
        self._check(self.lib.jpgenc_stage_dct(self.h, plane.ctypes.data, w, h, mode, out.ctypes.data))
        return out

    def encode_rgb_into(self, host_ptr: int, w: int, h: int, out_ptr: int, cap: int, maxval: int = 255) -> int:
        n = C.c_uint64()
        self._check(self.lib.jpgenc_encode_rgb(self.h, host_ptr, w, h, maxval, out_ptr, cap, C.byref(n)))
        return n.value

    def encode_frames_device(self, frame_ptrs, w: int, h: int, out_ptrs=None, caps=None, maxval: int = 255, host_frames=False):
        """equally sized frames (device memory, or host memory with host_frames=True) through every kernel together;
        returns the JPEG sizes"""
        n = len(frame_ptrs)
        frames = (C.c_void_p * n)(*frame_ptrs)
        sizes = (C.c_uint64 * n)()
        outs = (C.c_void_p * n)(*out_ptrs) if out_ptrs is not None else None
        capv = (C.c_uint64 * n)(*caps) if caps is not None else None
        fn = self.lib.jpgenc_encode_frames if host_frames else self.lib.jpgenc_encode_frames_device
        self._check(fn(self.h, n, frames, w, h, maxval, outs, capv, sizes))
        return [int(x) for x in sizes]

    def encode_frames_packed(self, frame_ptrs, w: int, h: int, out_ptr: int | None, cap: int, maxval: int = 255, host_frames=False):
        """equally sized frames -> complete files back to back in ONE buffer (one device-to-host copy per pass);
        returns (offsets, sizes, total bytes)"""
        n = len(frame_ptrs)
        frames = (C.c_void_p * n)(*frame_ptrs)
        sizes = (C.c_uint64 * n)()
        offs = (C.c_uint64 * n)()
        total = C.c_uint64()
        self._check(self.lib.jpgenc_encode_frames_packed(self.h, n, frames, 0 if host_frames else 1, w, h, maxval, out_ptr, cap,
                                                         offs, sizes, C.byref(total)))
        return [int(x) for x in offs], [int(x) for x in sizes], int(total.value)

    def _packed(self, fn, n: int, per_image: int, ptrs, host_images: bool, widths, heights, *args):
        """the marshalling the encode_images_packed* calls share: fn(handle, n, pointers, on_device, widths, heights, *args,
        offsets, sizes, &total); optional per-image arrays in args are lists or None; returns (offsets, sizes, total bytes).
        The pointer array holds per_image * n entries, as the C side reads them; missing ones are NULL."""
        arrays = [np.ascontiguousarray(a, np.uint32) for a in (widths, heights)]
        conv = []
        for a in args:
            if isinstance(a, (list, tuple, np.ndarray)):
                arrays.append(np.ascontiguousarray(a, np.uint32))
                conv.append(_np_ptr(arrays[-1], u32p))
            else:
                conv.append(a)
        sizes = (C.c_uint64 * n)()
        offs = (C.c_uint64 * n)()
        total = C.c_uint64()
        self._check(fn(self.h, n, (C.c_void_p * (per_image * n))(*ptrs), 0 if host_images else 1, _np_ptr(arrays[0], u32p), _np_ptr(arrays[1], u32p),
                       *conv, offs, sizes, C.byref(total)))
        return [int(x) for x in offs], [int(x) for x in sizes], int(total.value)

    def encode_images_packed(self, ptrs, widths, heights, out_ptr: int | None, cap: int, maxval: int = 255, host_images=False,
                             pitches=None, fmt=None):
        """images of individual sizes (device memory, or host memory with host_images=True) -> complete files back to back in
        ONE buffer, in input order; returns (offsets, sizes, total bytes).  pitches (bytes from row to row, per image; None or 0:
        tight) and fmt ('RGB', 'BGR', 'RGBA', 'BGRA') describe pixels in another layout than tight RGB."""
        n = len(ptrs)
        if pitches is None and fmt is None:
            return self._packed(self.lib.jpgenc_encode_images_packed, n, 1, ptrs, host_images, widths, heights, maxval, out_ptr, cap)
        return self._packed(self.lib.jpgenc_encode_images_packed_layout, n, 1, ptrs, host_images, widths, heights,
                            None if pitches is None else list(pitches), _format_code(fmt or "RGB"), maxval, out_ptr, cap)

    def encode_images_packed_planar(self, planes, widths, heights, out_ptr: int | None, cap: int, maxval: int = 255, host_images=False,
                                    pitches=None):
        """planar RGB images of individual sizes: planes[3i:3i + 3] = the R, G, B plane pointers of image i (device memory, or host
        memory with host_images=True), pitches per image (None or 0: tight) -> files back to back as encode_images_packed"""
        return self._packed(self.lib.jpgenc_encode_images_packed_planar, len(widths), 3, planes, host_images, widths, heights,
                            None if pitches is None else list(pitches), maxval, out_ptr, cap)

    def encode_images_packed_yuv420(self, planes, widths, heights, out_ptr: int | None, cap: int, layout: str = "I420", host_images=False,
                                    y_pitches=None, c_pitches=None):
        """YUV 4:2:0 frames of individual sizes: planes[3i:3i + 3] = the Y, U, V plane pointers of frame i (NV12: Y, UV, None;
        device memory, or host memory with host_images=True), pitches per frame (None or 0: tight) -> files back to back as
        encode_images_packed"""
        return self._packed(self.lib.jpgenc_encode_images_packed_yuv420, len(widths), 3, planes, host_images, widths, heights,
                            None if y_pitches is None else list(y_pitches), None if c_pitches is None else list(c_pitches),
                            YUV_LAYOUTS[layout], out_ptr, cap)

    def encode_images_packed_yuv(self, planes, widths, heights, out_ptr: int | None, cap: int, layout: str, host_images=False,
                                 y_pitches=None, c_pitches=None):
        """YUV frames of one YUV_FORMATS layout and individual sizes: planes[3i:3i + 3] = the plane pointers of frame i (None where
        the layout has no such plane) -> files back to back as encode_images_packed"""
        return self._packed(self.lib.jpgenc_encode_images_packed_yuv, len(widths), 3, planes, host_images, widths, heights,
                            None if y_pitches is None else list(y_pitches), None if c_pitches is None else list(c_pitches),
                            YUV_FORMATS[layout], out_ptr, cap)

    def _planes_on_host(self, planes) -> bool:
        """True for numpy arrays and CPU tensors; False for tensors on this encoder's GPU, once the work queued on torch's current
        stream has finished.  Anything else (a mix, another device) raises ValueError."""
        kinds = set()
        for a in planes:
            if isinstance(a, np.ndarray):
                kinds.add("cpu")
            else:
                dev = a.device
                if dev.type == "cuda" and dev.index != self.device:
                    raise ValueError(f"tensor on {dev}, encoder on cuda:{self.device}")
                if dev.type not in ("cpu", "cuda"):
                    raise ValueError(f"tensors on {dev} cannot be read")
                kinds.add(dev.type)
        if len(kinds) != 1:
            raise ValueError("the planes of one call must all be in host memory or all on the encoder's GPU")
        if kinds.pop() == "cpu":
            return True
        import torch

        dev = torch.device("cuda", self.device)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
        ev.synchronize()
        return False

    def encode_yuv420(self, y, u, v=None) -> bytes:
        """one YUV 4:2:0 frame read in place (yuv420_layout: I420 with v, NV12 without) from numpy arrays, CPU tensors or tensors on
        this encoder's GPU -> JPEG bytes"""
        layout, (yp, up, vp), w, h, y_pitch, c_pitch = yuv420_layout(y, u, v)
        if self._planes_on_host([a for a in (y, u, v) if a is not None]):
            return self.encode_yuv420_ptr(yp, up, vp, w, h, y_pitch, c_pitch, layout)
        self.bind_device_yuv420(yp, up, vp, w, h, y_pitch, c_pitch, layout)
        n = self.encode_bound(None)
        out = np.empty(n, np.uint8)
        n = C.c_uint64()
        self._check(self.lib.jpgenc_assemble_last(self.h, out.ctypes.data, out.size, C.byref(n)))
        return out[: n.value].tobytes()

    def encode_yuv420_many(self, frames):
        """(y, u) NV12 or (y, u, v) I420 frames of any sizes, one layout per call, all in host memory or all on this encoder's GPU
        (see encode_yuv420), through one batched call -> list of JPEG byte strings"""
        frames = [tuple(f) for f in frames]
        if not frames:
            return []
        layouts = [yuv420_layout(*f) for f in frames]
        kinds = {x[0] for x in layouts}
        if len(kinds) != 1:
            raise ValueError(f"one YUV layout per call; got {sorted(kinds)}")
        host = self._planes_on_host([a for f in frames for a in f if a is not None])
        planes = [p or None for x in layouts for p in x[1]]
        ws = [x[2] for x in layouts]
        hs = [x[3] for x in layouts]
        yps = [x[4] for x in layouts]
        cps = [x[5] for x in layouts]
        layout = layouts[0][0]
        enc = lambda o, c: self.encode_images_packed_yuv420(planes, ws, hs, o, c, layout, host_images=host, y_pitches=yps, c_pitches=cps)
        return self._files(enc, sum(w * h for w, h in zip(ws, hs)), len(frames))

    def encode_yuv(self, layout: str, y, u=None, v=None, w=None) -> bytes:
        """one YUV frame in the named layout read in place (see yuv_layout) from numpy arrays, CPU tensors or tensors on this
        encoder's GPU -> JPEG bytes"""
        layout, (yp, up, vp), w, h, y_pitch, c_pitch = yuv_layout(layout, y, u, v, w)
        if self._planes_on_host([a for a in (y, u, v) if a is not None]):
            return self.encode_yuv_ptr(layout, yp, up, vp, w, h, y_pitch, c_pitch)
        self.bind_device_yuv(layout, yp, up, vp, w, h, y_pitch, c_pitch)
        n = self.encode_bound(None)
        out = np.empty(n, np.uint8)
        n = C.c_uint64()
        self._check(self.lib.jpgenc_assemble_last(self.h, out.ctypes.data, out.size, C.byref(n)))
        return out[: n.value].tobytes()

    def encode_yuv_many(self, layout: str, frames):
        """frames of one named layout and any sizes, each a tuple (y, u, v, w) or a prefix of it (see yuv_layout), all in host
        memory or all on this encoder's GPU, through one batched call -> list of JPEG byte strings"""
        frames = [tuple(f) for f in frames]
        if not frames:
            return []
        layouts = [yuv_layout(layout, *f) for f in frames]
        host = self._planes_on_host([a for f in frames for a in f[:3] if a is not None])
        planes = [p or None for x in layouts for p in x[1]]
        ws, hs = [x[2] for x in layouts], [x[3] for x in layouts]
        yps, cps = [x[4] for x in layouts], [x[5] for x in layouts]
        enc = lambda o, c: self.encode_images_packed_yuv(planes, ws, hs, o, c, layout, host_images=host, y_pitches=yps, c_pitches=cps)
        return self._files(enc, sum(w * h for w, h in zip(ws, hs)), len(frames))

    def _files(self, encode, pixels: int, n: int):
        """encode(out_ptr, cap) -> (offsets, sizes, total) into a host buffer, again with the reported size when the files
        outgrow the first guess -> list of the files"""
        out = np.empty(pixels * 3 + 4096 * n, np.uint8)
        try:
            offs, sizes, _ = encode(out.ctypes.data, out.size)
        except JpgencError as e:
            if e.code != ERR_CAPACITY:
                raise
            _, _, total = encode(None, 0)
            out = np.empty(total, np.uint8)
            offs, sizes, _ = encode(out.ctypes.data, out.size)
        return [out[o: o + k].tobytes() for o, k in zip(offs, sizes)]

    def encode_tensor(self, t, order: str = "RGB") -> bytes:
        """one torch uint8 image tensor, on the CPU or on this encoder's GPU, read in place (see tensor_layout) -> JPEG bytes"""
        return self.encode_tensors([t], order)[0]

    def encode_tensors(self, ts, order: str = "RGB", maxval: int = 255):
        """torch uint8 image tensors of any sizes, all on the CPU or all on this encoder's GPU and all of one layout kind
        (tensor_layout), through one batched call -> list of JPEG byte strings.  Nothing is copied or converted: any other
        tensor raises ValueError.  CUDA tensors are read once the work queued on torch's current stream has finished."""
        import torch

        ts = list(ts)
        if not ts:
            return []
        layouts = [tensor_layout(t, order) for t in ts]
        kinds = {x[0] for x in layouts}
        if len(kinds) != 1:
            raise ValueError(f"one layout kind per call; got {sorted(kinds)}")
        devices = {t.device for t in ts}
        if len(devices) != 1:
            raise ValueError(f"tensors on several devices in one call: {sorted(str(d) for d in devices)}")
        dev = devices.pop()
        if dev.type == "cuda":
            if dev.index != self.device:
                raise ValueError(f"tensor on {dev}, encoder on cuda:{self.device}")
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(dev))
            ev.synchronize()
        elif dev.type != "cpu":
            raise ValueError(f"tensors on {dev} cannot be read")
        kind = layouts[0][0]
        ws = [x[2] for x in layouts]
        hs = [x[3] for x in layouts]
        pitches = [x[4] for x in layouts]
        host = dev.type == "cpu"
        if kind == "planar":
            planes = [p for x in layouts for p in x[1]]
            enc = lambda o, c: self.encode_images_packed_planar(planes, ws, hs, o, c, maxval, host_images=host, pitches=pitches)
        else:
            ptrs = [x[1][0] for x in layouts]
            enc = lambda o, c: self.encode_images_packed(ptrs, ws, hs, o, c, maxval, host_images=host, pitches=pitches, fmt=kind)
        return self._files(enc, sum(w * h for w, h in zip(ws, hs)), len(ts))

    def encode_images(self, images, maxval: int = 255, fmt: str | None = None):
        """list of HxWx3 uint8 arrays of any sizes -> list of JPEG byte strings, through one call (a second one, sizes first,
        only when the files outgrow the pixels).  With fmt ('RGB', 'BGR', 'RGBA', 'BGRA', 'GRAY') the arrays are read where they
        are, with their row pitch: (H, W, C) arrays with strides (pitch, C, 1), such as crop views of a larger image, or (H, W)
        grey arrays with strides (pitch, 1) (image_layout; anything else raises ValueError)."""
        if fmt is None:
            images = [np.ascontiguousarray(a, np.uint8) for a in images]
            layouts = [(a.ctypes.data, a.shape[1], a.shape[0], 0) for a in images]
        else:
            layouts = [image_layout(a, fmt) for a in images]
        if not images:
            return []
        ptrs = [x[0] for x in layouts]
        ws = [x[1] for x in layouts]
        hs = [x[2] for x in layouts]
        pitches = [x[3] for x in layouts] if fmt is not None else None
        return self._files(lambda o, c: self.encode_images_packed(ptrs, ws, hs, o, c, maxval, host_images=True, pitches=pitches, fmt=fmt),
                           sum(w * h for w, h in zip(ws, hs)), len(images))

    def encode_ppm_file(self, src: str, dst: str):
        self._check(self.lib.jpgenc_encode_ppm_file(self.h, src.encode(), dst.encode()))

    # ---- microbench -----------------------------------------------------------------------------
    def dct_quant_blocks(self, dev_in: int, dev_out: int, nblocks: int, q, want_refined=True) -> int:
        q = np.ascontiguousarray(q, np.uint8).reshape(64)
        n = C.c_uint64()
        self._check(self.lib.jpgenc_dct_quant_blocks(self.h, dev_in, dev_out, nblocks, _np_ptr(q, u8p),
                                                     C.byref(n) if want_refined else None))
        return n.value

    # ---- helpers --------------------------------------------------------------------------------
    def stats(self) -> Stats:
        s = Stats()
        self._check(self.lib.jpgenc_get_stats(self.h, C.byref(s)))
        return s

    def synchronize(self):
        self._check(self.lib.jpgenc_synchronize(self.h))

    def stream(self) -> int:
        return self.lib.jpgenc_stream(self.h)

    def dev_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        self._check(self.lib.jpgenc_dev_alloc(self.h, nbytes, C.byref(p)))
        return p.value

    def dev_free(self, p: int):
        self._check(self.lib.jpgenc_dev_free(self.h, p))

    def h2d(self, dev: int, arr: np.ndarray):
        arr = np.ascontiguousarray(arr)
        self._check(self.lib.jpgenc_memcpy_h2d(self.h, dev, arr.ctypes.data, arr.nbytes))

    def d2h(self, arr: np.ndarray, dev: int):
        assert arr.flags.c_contiguous
        self._check(self.lib.jpgenc_memcpy_d2h(self.h, arr.ctypes.data, dev, arr.nbytes))

    def synth_rgb(self, dev: int, w: int, h: int, seed: int = 0):
        self._check(self.lib.jpgenc_synth_rgb(self.h, dev, w, h, seed))

    def synth_blocks(self, dev: int, nblocks: int):
        self._check(self.lib.jpgenc_synth_blocks(self.h, dev, nblocks))

    def flush_l2(self):
        self._check(self.lib.jpgenc_flush_l2(self.h))

    def timer_begin(self):
        self._check(self.lib.jpgenc_timer_begin(self.h))

    def timer_end(self) -> float:
        ms = C.c_float()
        self._check(self.lib.jpgenc_timer_end(self.h, C.byref(ms)))
        return ms.value

    def launch_count(self) -> int:
        return self.lib.jpgenc_launch_count(self.h)


class Batch:
    """Several contexts on one GPU driven by host threads inside the library: independent frames in, JPEG files out."""

    def __init__(self, device: int = 0, workers: int = 4):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.jpgenc_batch_create(device, workers, C.byref(h))
        if rc != OK:
            raise JpgencError(rc, (self.lib.jpgenc_last_error(None) or b"").decode())
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.jpgenc_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != OK:
            raise JpgencError(rc, (self.lib.jpgenc_batch_last_error(self.h) or b"").decode())

    def encode_ptrs(self, frame_ptrs, w: int, h: int, out_ptrs, caps, maxval: int = 255, device_frames: bool = False):
        """raw-pointer form (pinned host or device frames); out_ptrs may be None for device frames -> sizes only"""
        n = len(frame_ptrs)
        frames = (C.c_void_p * n)(*frame_ptrs)
        sizes = (C.c_uint64 * n)()
        outs = (C.c_void_p * n)(*out_ptrs) if out_ptrs is not None else None
        capv = (C.c_uint64 * n)(*caps) if caps is not None else None
        fn = self.lib.jpgenc_batch_encode_device if device_frames else self.lib.jpgenc_batch_encode
        self._check(fn(self.h, n, frames, w, h, maxval, outs, capv, sizes))
        return [int(x) for x in sizes]

    def encode(self, frames, maxval: int = 255):
        """list of HxWx3 uint8 arrays of one size -> list of JPEG byte strings"""
        frames = [np.ascontiguousarray(f, np.uint8) for f in frames]
        h, w, _ = frames[0].shape
        cap = max(4096, frames[0].size + 4096)
        outs = [np.empty(cap, np.uint8) for _ in frames]
        sizes = self.encode_ptrs([f.ctypes.data for f in frames], w, h, [o.ctypes.data for o in outs], [cap] * len(frames), maxval)
        return [o[:n].tobytes() for o, n in zip(outs, sizes)]


def bind_host_to_device_numa(device: int):
    """-> (numa node or -1, CPUs in the new affinity mask); see jpgenc_bind_host_to_device_numa"""
    node, cpus = C.c_int(-1), C.c_int(0)
    load_library().jpgenc_bind_host_to_device_numa(device, C.byref(node), C.byref(cpus))
    return node.value, cpus.value


def pinned_empty(nbytes: int):
    """(numpy view, raw pointer) over freshly allocated page-locked host memory."""
    lib = load_library()
    p = C.c_void_p()
    if lib.jpgenc_host_alloc_pinned(nbytes, C.byref(p)) != OK:
        raise MemoryError("cudaMallocHost failed")
    buf = (C.c_uint8 * nbytes).from_address(p.value)
    return np.frombuffer(buf, np.uint8), p.value


def pinned_free(ptr: int):
    load_library().jpgenc_host_free_pinned(ptr)
