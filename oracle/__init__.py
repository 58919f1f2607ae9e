"""ctypes binding of the CPU oracle (oracle/jpeg_oracle.c).

TEST INFRASTRUCTURE, NOT PRODUCT CODE: only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / reference leg may import this module. The product path
(nvjpeg_imagecompressor_b200) never does and fails loudly without its CUDA library.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "liborc.so")

CSS = {"444": 0, "422": 1, "440": 2, "420": 3, "411": 4}
CSS_GRAY = 6      # B2J_CSS_GRAY: one component
SCALES = (2, 4, 8)


def build(force=False):
    newest = max(os.path.getmtime(os.path.join(_HERE, f)) for f in ("jpeg_oracle.c", "jpeg_oracle.h"))
    if force or not os.path.exists(_LIB) or os.path.getmtime(_LIB) < newest:
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
    return _LIB


class Geom(C.Structure):
    _fields_ = [("W", C.c_int), ("H", C.c_int), ("css", C.c_int), ("hs", C.c_int), ("vs", C.c_int),
                ("mcux", C.c_int), ("mcuy", C.c_int), ("bpm", C.c_int), ("wib", C.c_int * 3),
                ("hib", C.c_int * 3), ("dw", C.c_int * 3), ("dh", C.c_int * 3), ("nblocks", C.c_longlong)]


class Info(C.Structure):
    _fields_ = [("W", C.c_int), ("H", C.c_int), ("css", C.c_int), ("hs", C.c_int), ("vs", C.c_int),
                ("restart_interval", C.c_int), ("scan_offset", C.c_size_t), ("scan_len", C.c_size_t),
                ("qt", (C.c_uint16 * 64) * 2), ("bits", (C.c_uint8 * 17) * 4), ("vals", (C.c_uint8 * 256) * 4)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB)
        _lib.orc_stuff.restype = C.c_size_t
        _lib.orc_headers.restype = C.c_size_t
        _lib.orc_ssd.restype = C.c_uint64
        _lib.orc_psnr.restype = C.c_double
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def geometry(W, H, css):
    g = Geom()
    rc = lib().orc_geometry(int(W), int(H), int(css), C.byref(g))
    if rc:
        raise ValueError("bad geometry")
    return g


def quant_tables(quality):
    qt = np.zeros((2, 64), np.uint16)
    lib().orc_quant_tables(int(quality), _p(qt))
    return qt


def synth(W, H, seed=0, amp=8, y0=0, rows=None):
    rows = H - y0 if rows is None else rows
    out = np.empty((rows, W, 3), np.uint8)
    lib().orc_synth_rows(int(W), int(H), int(y0), int(rows), C.c_uint32(seed), int(amp), _p(out))
    return out


def forward(img, css, quality):
    img = np.ascontiguousarray(img)
    H, W = img.shape[:2]
    g = geometry(W, H, css)
    coef = np.empty((g.nblocks, 64), np.int16)
    rc = lib().orc_forward(_p(img), C.c_size_t(img.strides[0]), W, H, int(css), int(quality), _p(coef))
    if rc:
        raise RuntimeError(f"orc_forward rc={rc}")
    return coef


def histogram(coef, bpm, pred_in=None):
    coef = np.ascontiguousarray(coef, np.int16)
    hist = np.zeros((4, 257), np.uint32)
    pred = None if pred_in is None else _p(np.ascontiguousarray(pred_in, np.int16))
    lib().orc_histogram(_p(coef), C.c_longlong(coef.shape[0]), int(bpm), pred, _p(hist))
    return hist


def gen_optimal_table(freq):
    freq = np.ascontiguousarray(freq, np.uint32)
    assert freq.shape == (257,)
    bits = np.zeros(17, np.uint8)
    vals = np.zeros(256, np.uint8)
    n = lib().orc_gen_optimal_table(_p(freq), _p(bits), _p(vals))
    if n < 0:
        raise RuntimeError("code length overflow")
    return bits, vals, n


def std_tables():
    bits = np.zeros((4, 17), np.uint8)
    vals = np.zeros((4, 256), np.uint8)
    for t in range(4):
        lib().orc_std_table(t, _p(bits[t]), _p(vals[t]))
    return bits, vals


def derive_codes(bits, vals):
    code = np.zeros(256, np.uint16)
    size = np.zeros(256, np.uint8)
    lib().orc_derive_codes(_p(np.ascontiguousarray(bits, np.uint8)), _p(np.ascontiguousarray(vals, np.uint8)),
                           _p(code), _p(size))
    return code, size


def entropy_bits(coef, bpm, bits, vals, pred_in=None):
    coef = np.ascontiguousarray(coef, np.int16)
    bits = np.ascontiguousarray(bits, np.uint8)
    vals = np.ascontiguousarray(vals, np.uint8)
    cap = coef.shape[0] * 208 + 16
    out = np.zeros(cap, np.uint8)
    nbits = C.c_uint64(0)
    pred = None if pred_in is None else _p(np.ascontiguousarray(pred_in, np.int16))
    rc = lib().orc_entropy_bits(_p(coef), C.c_longlong(coef.shape[0]), int(bpm), pred, _p(bits), _p(vals),
                                _p(out), C.c_size_t(cap), C.byref(nbits))
    if rc:
        raise RuntimeError("entropy overflow")
    return out[: (nbits.value + 7) // 8].copy(), nbits.value


def stuff(raw, nbits):
    raw = np.ascontiguousarray(raw, np.uint8)
    cap = raw.size * 2 + 8
    out = np.zeros(cap, np.uint8)
    n = lib().orc_stuff(_p(raw), C.c_uint64(nbits), _p(out), C.c_size_t(cap))
    return out[:n].copy()


def headers(W, H, css, qt, bits, vals):
    out = np.zeros(2048, np.uint8)
    n = lib().orc_headers(int(W), int(H), int(css), _p(np.ascontiguousarray(qt, np.uint16)),
                          _p(np.ascontiguousarray(bits, np.uint8)), _p(np.ascontiguousarray(vals, np.uint8)),
                          _p(out), C.c_size_t(2048))
    return out[:n].copy()


def encode(img, css, quality, optimize, restart_interval=0):
    """restart_interval: MCUs between RSTn markers (0 = none), as cv2's IMWRITE_JPEG_RST_INTERVAL."""
    img = np.ascontiguousarray(img)
    H, W = img.shape[:2]
    cap = W * H * 3 * 4 + 4096 + (2 * W * H // 64 if restart_interval else 0)
    out = np.empty(cap, np.uint8)
    n = C.c_size_t(0)
    rc = lib().orc_encode_rst(_p(img), C.c_size_t(img.strides[0]), W, H, int(css), int(quality), int(bool(optimize)),
                              int(restart_interval), _p(out), C.c_size_t(cap), C.byref(n))
    if rc:
        raise RuntimeError(f"orc_encode rc={rc}")
    return out[: n.value].copy()


def encode_gray(img, quality, optimize, restart_interval=0):
    """cv2.imencode(".jpg", gray, [QUALITY, OPTIMIZE(, RST_INTERVAL)]) of an (H, W) or (H, W, 1) uint8 image restated;
    restart_interval in blocks (MCUs of the one-component scan)."""
    img = np.asarray(img)
    if img.ndim == 3 and img.shape[2] == 1:
        img = img[:, :, 0]
    if img.ndim != 2 or img.dtype != np.uint8 or img.strides[1] != 1:
        img = np.ascontiguousarray(img, np.uint8)
    H, W = img.shape
    cap = W * H * 4 + 4096 + (2 * W * H // 64 if restart_interval else 0)
    out = np.empty(cap, np.uint8)
    n = C.c_size_t(0)
    rc = lib().orc_encode_rst(_p(img), C.c_size_t(img.strides[0]), W, H, CSS_GRAY, int(quality), int(bool(optimize)),
                              int(restart_interval), _p(out), C.c_size_t(cap), C.byref(n))
    if rc:
        raise RuntimeError(f"orc_encode_rst rc={rc}")
    return out[: n.value].copy()


def encode_progressive(img, css, quality):
    """cv2.imencode(..., IMWRITE_JPEG_PROGRESSIVE=1) restated (progressive mode always optimises its tables)."""
    img = np.ascontiguousarray(img)
    H, W = img.shape[:2]
    cap = W * H * 3 * 4 + 8192
    out = np.empty(cap, np.uint8)
    n = C.c_size_t(0)
    rc = lib().orc_encode_progressive(_p(img), C.c_size_t(img.strides[0]), W, H, int(css), int(quality), _p(out),
                                      C.c_size_t(cap), C.byref(n))
    if rc:
        raise RuntimeError(f"orc_encode_progressive rc={rc}")
    return out[: n.value].copy()


def parse(jpg):
    jpg = np.ascontiguousarray(jpg, np.uint8)
    info = Info()
    rc = lib().orc_parse(_p(jpg), C.c_size_t(jpg.size), C.byref(info))
    if rc:
        raise RuntimeError(f"orc_parse rc={rc}")
    return info


def decode_coefs(jpg):
    jpg = np.ascontiguousarray(jpg, np.uint8)
    info = parse(jpg)
    g = geometry(info.W, info.H, info.css)
    coef = np.empty((g.nblocks, 64), np.int16)
    rc = lib().orc_decode_coefs(_p(jpg), C.c_size_t(jpg.size), C.byref(info), _p(coef))
    if rc:
        raise RuntimeError(f"orc_decode_coefs rc={rc}")
    return coef, info


def reduced_size(W, H, denom):
    """(W', H') of a decode at 1/denom: libjpeg's jdiv_round_up(W, denom)."""
    return (W + denom - 1) // denom, (H + denom - 1) // denom


def _decode(name, jpg, gray, *args):
    """name(jpg, len, *args, out, step, &W, &H): first the output size, then the pixels"""
    fn = getattr(lib(), name)
    jpg = np.ascontiguousarray(jpg, np.uint8)
    W, H = C.c_int(0), C.c_int(0)
    rc = fn(_p(jpg), C.c_size_t(jpg.size), *args, None, C.c_size_t(0), C.byref(W), C.byref(H))
    if not rc:
        out = np.empty((H.value, W.value) + (() if gray else (3,)), np.uint8)
        rc = fn(_p(jpg), C.c_size_t(jpg.size), *args, _p(out), C.c_size_t(out.strides[0]), C.byref(W), C.byref(H))
    if rc:
        raise RuntimeError(f"{name} rc={rc}")
    return out


def decode(jpg):
    """cv2.imdecode(jpg, IMREAD_COLOR) as (H, W, 3) BGR"""
    return _decode("orc_decode", jpg, False)


def decode_gray(jpg):
    """(H, W) uint8: cv2.imdecode(IMREAD_UNCHANGED) of a one-component file, IMREAD_GRAYSCALE (the Y plane) of a
    three-component one."""
    return _decode("orc_decode_output", jpg, True, 1, 1)


def decode_scaled(jpg, denom, gray=False):
    """cv2.imdecode(jpg, IMREAD_REDUCED_COLOR_denom) as (H', W', 3) BGR, or IMREAD_REDUCED_GRAYSCALE_denom as (H', W')
    with gray=True (denom 1: IMREAD_COLOR / IMREAD_GRAYSCALE)."""
    return _decode("orc_decode_output", jpg, gray, int(denom), int(bool(gray)))


def diff(a, b, mode=0):
    a = np.ascontiguousarray(a, np.uint8)
    b = np.ascontiguousarray(b, np.uint8)
    out = np.empty_like(a)
    lib().orc_diff(_p(a), _p(b), C.c_size_t(a.size), int(mode), _p(out))
    return out


def ssd(a, b):
    a = np.ascontiguousarray(a, np.uint8)
    b = np.ascontiguousarray(b, np.uint8)
    return int(lib().orc_ssd(_p(a), _p(b), C.c_size_t(a.size)))


def psnr(a, b):
    a = np.ascontiguousarray(a, np.uint8)
    b = np.ascontiguousarray(b, np.uint8)
    return float(lib().orc_psnr(_p(a), _p(b), C.c_size_t(a.size)))
