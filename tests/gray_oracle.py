"""ctypes binding of the grayscale CPU checker (tests/cpp/gray_oracle.c, which reuses oracle/jpeg_oracle.c).

TEST INFRASTRUCTURE, NOT PRODUCT CODE. The shared library is compiled with gcc into a temporary directory on first use
(the repository tree may be read-only) and removed when the process exits.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "gray_oracle.c")
CSS_GRAY = 6   # B2J_CSS_GRAY

_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="gray_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libgray_oracle.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-std=c11", "-o", so, SRC, "-lm"])
        _lib = C.CDLL(so)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


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
    rc = lib().orc_encode_gray(_p(img), C.c_size_t(img.strides[0]), W, H, int(quality), int(bool(optimize)),
                               int(restart_interval), _p(out), C.c_size_t(cap), C.byref(n))
    if rc:
        raise RuntimeError(f"orc_encode_gray rc={rc}")
    return out[: n.value].copy()


def decode_gray(jpg):
    """(H, W) uint8: cv2.imdecode(IMREAD_UNCHANGED) of a one-component file, IMREAD_GRAYSCALE (the Y plane) of a
    three-component one."""
    jpg = np.ascontiguousarray(jpg, np.uint8)
    W, H = C.c_int(0), C.c_int(0)
    rc = lib().orc_decode_gray(_p(jpg), C.c_size_t(jpg.size), None, C.c_size_t(0), C.byref(W), C.byref(H))
    if rc:
        raise RuntimeError(f"orc_decode_gray rc={rc}")
    out = np.empty((H.value, W.value), np.uint8)
    rc = lib().orc_decode_gray(_p(jpg), C.c_size_t(jpg.size), _p(out), C.c_size_t(W.value), C.byref(W), C.byref(H))
    if rc:
        raise RuntimeError(f"orc_decode_gray rc={rc}")
    return out
