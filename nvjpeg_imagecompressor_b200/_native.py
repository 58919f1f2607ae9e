"""ctypes binding of libb2jpeg.so (include/b2jpeg.h). There is no CPU fallback: a missing library or a missing
CUDA device is an error."""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
LIB_PATH = os.environ.get("B2J_LIB") or os.path.join(_HERE, "libb2jpeg.so")   # B2J_LIB: development builds of the same library

CSS = {"444": 0, "422": 1, "440": 2, "420": 3, "411": 4, "gray": 6, "400": 6}   # 6: B2J_CSS_GRAY (NVJPEG_CSS_GRAY)
CSS_GRAY = 6
ERRORS = {0: "OK", -1: "EINVAL", -2: "ECUDA", -3: "ENOMEM", -4: "ECAPACITY", -5: "EFORMAT", -6: "EINTERNAL", -7: "ESIZE"}

FLAG_NO_PINNED, FLAG_ENCODE, FLAG_DECODE = 1, 2, 4
DBG_COEF, DBG_HIST, DBG_TABLES, DBG_TILE_BITS, DBG_DEC_COEF, DBG_TOKEN_COUNT, DBG_TOKENS, DBG_TILE_RECS, DBG_SLOTS = 0, 1, 2, 3, 4, 5, 6, 7, 8


class Params(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("quality", C.c_int), ("optimize", C.c_int),
                ("css", C.c_int), ("device", C.c_int), ("flags", C.c_int)]


class StripState(C.Structure):
    _fields_ = [("d_hist", C.c_void_p), ("d_last_dc", C.c_void_p), ("d_pred_in", C.c_void_p),
                ("d_strip_bits", C.c_void_p), ("d_out_len", C.c_void_p), ("d_out", C.c_void_p),
                ("d_record", C.c_void_p)]


class ReconPlanes(C.Structure):
    _fields_ = [("row_bytes", C.c_size_t)] + [(n, C.c_void_p) for n in ("cb_first", "cr_first", "cb_last", "cr_last", "cb_halo_top",
                                                                         "cr_halo_top", "cb_halo_bottom", "cr_halo_bottom")]


STRIP_RECORD_BYTES = 4176


class Timings(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("h2d", "fdct", "hist_edge", "tables", "pack", "scan", "stuff", "d2h", "total",
                                         "dec_parse", "dec_sync", "dec_write", "dec_idct", "dec_color")]


class HuffDev(C.Structure):
    _fields_ = [("enc", (C.c_uint32 * 256) * 4), ("bits", (C.c_uint8 * 17) * 4), ("vals", (C.c_uint8 * 256) * 4),
                ("nsym", C.c_uint32 * 4), ("hdr_len", C.c_uint32), ("err", C.c_uint32)]


# every symbol include/b2jpeg.h declares (tests/test_abi.py checks the list against the header)
SYMBOLS = ["b2j_default_params", "b2j_create", "b2j_destroy", "b2j_last_error", "b2j_version", "b2j_set_stream",
           "b2j_encode_bound", "b2j_encode", "b2j_encode_device", "b2j_encode_finish", "b2j_peek", "b2j_decode",
           "b2j_decode_device", "b2j_decode_finish", "b2j_decode_scan_device", "b2j_diff", "b2j_psnr", "b2j_diff_psnr_device", "b2j_secondary",
           "b2j_reconstruct_device", "b2j_reconstruct_planes", "b2j_reconstruct_color", "b2j_secondary_device", "b2j_secondary_finish", "b2j_secondary_fetch", "b2j_encode_begin", "b2j_encode_fetch",
           "b2j_multi_create", "b2j_multi_destroy", "b2j_multi_encode", "b2j_multi_encode_begin", "b2j_multi_encode_fetch",
           "b2j_multi_last_error",
           "b2j_strip_state_get", "b2j_strip_phase1", "b2j_strip_phase1b", "b2j_strip_phase2", "b2j_strip_phase3", "b2j_strip_phase3_dev", "b2j_strip_phase1x", "b2j_strip_phase2x", "b2j_peer_export", "b2j_peer_open", "b2j_peer_connect", "b2j_set_restart_rows",
           "b2j_set_decode_scale",
           "b2j_debug_read", "b2j_set_debug", "b2j_last_timings", "b2j_enable_timing", "b2j_launch_count", "b2j_host_alloc",
           "b2j_host_free"]


def build(force=False):
    """Compile libb2jpeg.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    srcs = [os.path.join(_HERE, "csrc", f) for f in os.listdir(os.path.join(_HERE, "csrc"))]
    srcs.append(os.path.join(ROOT, "include", "b2jpeg.h"))
    stale = (not os.path.exists(LIB_PATH)) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if force or stale:
        subprocess.check_call(["make", "-C", ROOT, "-s", "-j8", os.path.relpath(LIB_PATH, ROOT)] + (["-B"] if force else []))
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with `make` (nvcc, sm_100a). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, sz, i, u8p = C.c_void_p, C.c_size_t, C.c_int, C.c_void_p
    L.b2j_default_params.argtypes = [C.POINTER(Params)]
    L.b2j_default_params.restype = None
    L.b2j_create.argtypes = [C.POINTER(Params), C.POINTER(vp)]
    L.b2j_destroy.argtypes = [vp]
    L.b2j_destroy.restype = None
    L.b2j_last_error.argtypes = [vp]
    L.b2j_last_error.restype = C.c_char_p
    L.b2j_version.restype = C.c_char_p
    L.b2j_set_stream.argtypes = [vp, vp]
    L.b2j_encode_bound.argtypes = [vp]
    L.b2j_encode_bound.restype = sz
    L.b2j_encode.argtypes = [vp, u8p, sz, i, i, u8p, sz, C.POINTER(sz)]
    L.b2j_encode_device.argtypes = [vp, u8p, sz, i, i, C.POINTER(vp), C.POINTER(vp)]
    L.b2j_encode_finish.argtypes = [vp, C.POINTER(sz)]
    L.b2j_peek.argtypes = [u8p, sz, C.POINTER(i), C.POINTER(i), C.POINTER(i)]
    L.b2j_decode.argtypes = [vp, u8p, sz, u8p, sz, C.POINTER(i), C.POINTER(i)]
    L.b2j_decode_device.argtypes = [vp, u8p, sz, u8p, sz, C.POINTER(i), C.POINTER(i)]
    L.b2j_decode_finish.argtypes = [vp]
    L.b2j_diff.argtypes = [vp, u8p, u8p, sz, i, u8p]
    L.b2j_psnr.argtypes = [vp, u8p, u8p, sz, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    L.b2j_diff_psnr_device.argtypes = [vp, u8p, u8p, sz, i, u8p, C.POINTER(vp)]
    L.b2j_secondary.argtypes = [vp, u8p, sz, i, i, i, u8p, sz, C.POINTER(sz), u8p, sz, C.POINTER(sz), u8p, sz,
                                C.POINTER(C.c_double)]
    L.b2j_encode_begin.argtypes = [vp, u8p, sz, i, i, C.POINTER(sz)]
    L.b2j_encode_fetch.argtypes = [vp, u8p, sz]
    L.b2j_multi_create.argtypes = [C.POINTER(Params), i, C.POINTER(C.c_int), C.POINTER(vp)]
    L.b2j_multi_destroy.argtypes = [vp]
    L.b2j_multi_destroy.restype = None
    L.b2j_multi_encode.argtypes = [vp, u8p, sz, i, i, u8p, sz, C.POINTER(sz)]
    L.b2j_multi_last_error.argtypes = [vp]
    L.b2j_multi_last_error.restype = C.c_char_p
    L.b2j_decode_scan_device.argtypes = [vp, u8p, sz, vp, sz, i, vp, sz, C.POINTER(i), C.POINTER(i)]
    L.b2j_secondary_fetch.argtypes = [vp, u8p, sz, u8p, sz, u8p, sz]
    L.b2j_reconstruct_device.argtypes = [vp, vp, sz]
    L.b2j_reconstruct_planes.argtypes = [vp, C.POINTER(ReconPlanes)]
    L.b2j_reconstruct_color.argtypes = [vp, vp, sz, i, i]
    L.b2j_secondary_device.argtypes = [vp, vp, sz, i, i, i, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    L.b2j_secondary_finish.argtypes = [vp, C.POINTER(sz), C.POINTER(sz), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    L.b2j_strip_state_get.argtypes = [vp, C.POINTER(StripState)]
    L.b2j_strip_phase1.argtypes = [vp, u8p, sz, i, i]
    L.b2j_strip_phase1b.argtypes = [vp]
    L.b2j_strip_phase2.argtypes = [vp, i, i]
    L.b2j_strip_phase3.argtypes = [vp, i, i, i]
    L.b2j_strip_phase3_dev.argtypes = [vp, vp, i, i, i]
    L.b2j_strip_phase1x.argtypes = [vp, u8p, sz, i, i]
    L.b2j_strip_phase2x.argtypes = [vp, vp, i, i, i, i, i]
    L.b2j_peer_export.argtypes = [vp, vp, C.POINTER(vp)]
    L.b2j_peer_open.argtypes = [vp, vp, C.POINTER(vp)]
    L.b2j_peer_connect.argtypes = [vp, i, i, C.POINTER(vp)]
    L.b2j_set_restart_rows.argtypes = [vp, i]
    L.b2j_set_decode_scale.argtypes = [vp, i]
    L.b2j_debug_read.argtypes = [vp, i, vp, sz, C.POINTER(sz)]
    L.b2j_set_debug.argtypes = [vp, i]
    L.b2j_last_timings.argtypes = [vp, C.POINTER(Timings)]
    L.b2j_enable_timing.argtypes = [vp, i]
    L.b2j_launch_count.argtypes = [vp]
    L.b2j_launch_count.restype = C.c_uint64
    L.b2j_host_alloc.argtypes = [sz]
    L.b2j_host_alloc.restype = vp
    L.b2j_host_free.argtypes = [vp]
    L.b2j_host_free.restype = None
    _lib = L
    return L
