"""ctypes binding of the reduced-size decode of the CPU checker (tests/cpp/scaled_oracle.c, which reuses
tests/cpp/gray_oracle.c and oracle/jpeg_oracle.c).

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
SRC = os.path.join(ROOT, "tests", "cpp", "scaled_oracle.c")
SCALES = (2, 4, 8)

_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="scaled_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libscaled_oracle.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-std=c11", "-o", so, SRC, "-lm"])
        _lib = C.CDLL(so)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def reduced_size(W, H, denom):
    """(W', H') of a decode at 1/denom: libjpeg's jdiv_round_up(W, denom)."""
    return (W + denom - 1) // denom, (H + denom - 1) // denom


def decode_scaled(jpg, denom, gray=False):
    """cv2.imdecode(jpg, IMREAD_REDUCED_COLOR_denom) as (H', W', 3) BGR, or IMREAD_REDUCED_GRAYSCALE_denom as (H', W')
    with gray=True (denom 1: IMREAD_COLOR / IMREAD_GRAYSCALE)."""
    jpg = np.ascontiguousarray(jpg, np.uint8)
    W, H = C.c_int(0), C.c_int(0)
    rc = lib().orc_decode_scaled(_p(jpg), C.c_size_t(jpg.size), int(denom), int(gray), None, C.c_size_t(0),
                                 C.byref(W), C.byref(H))
    if rc:
        raise RuntimeError(f"orc_decode_scaled rc={rc}")
    ch = 1 if gray else 3
    out = np.empty((H.value, W.value) + (() if gray else (3,)), np.uint8)
    rc = lib().orc_decode_scaled(_p(jpg), C.c_size_t(jpg.size), int(denom), int(gray), _p(out),
                                 C.c_size_t(W.value * ch), C.byref(W), C.byref(H))
    if rc:
        raise RuntimeError(f"orc_decode_scaled rc={rc}")
    return out
