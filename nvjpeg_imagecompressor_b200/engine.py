"""Engine: thin Python owner of one b2j_ctx (one encoder/decoder state on one GPU)."""
import ctypes as C

import numpy as np

from . import _native as N


class B2JError(RuntimeError):
    def __init__(self, rc, msg):
        super().__init__(f"b2jpeg error {rc} ({N.ERRORS.get(rc, '?')}): {msg}")
        self.rc = rc


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


def css_id(css):
    return N.CSS[css] if isinstance(css, str) else int(css)


class Engine:
    """width/height: the largest image this context will see (buffers are sized once, like the reference's
    initCompressEnv, ImageCompressorImpl.cu:33-37). css "gray" (or "400", 6): images are (H, W) uint8, one byte per
    pixel -- encode takes (H, W) or (H, W, 1), decode returns (H, W) for one-component files and the Y plane of colour
    ones; the strip, reconstruction and secondary-compression entry points refuse such a context."""

    def __init__(self, width=8320, height=40000, quality=95, optimize=True, css="422", device=-1, flags=0):
        self._L = N.lib()
        p = N.Params(int(width), int(height), int(quality), int(bool(optimize)), css_id(css), int(device), int(flags))
        self.params = p
        self.channels = 1 if p.css == N.CSS_GRAY else 3
        h = C.c_void_p()
        rc = self._L.b2j_create(C.byref(p), C.byref(h))
        if rc:
            raise B2JError(rc, "b2j_create failed (is a CUDA device visible? there is no CPU fallback)")
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._L.b2j_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc:
            raise B2JError(rc, self._L.b2j_last_error(self._h).decode())

    # ---------------------------------------------------------------- host API
    def encode(self, img, out=None):
        img = np.asarray(img)
        if self.channels == 1:
            if img.ndim == 3 and img.shape[2] == 1:
                img = img[:, :, 0]
            assert img.dtype == np.uint8 and img.ndim == 2 and (img.strides[1] == 1 or img.shape[1] == 1), \
                "a gray context encodes (H, W) uint8 rows"
        else:
            assert img.dtype == np.uint8 and img.ndim == 3 and img.shape[2] == 3 and img.strides[2] == 1 and img.strides[1] == 3
        H, W = img.shape[:2]
        if out is None:
            out = np.empty(min(self._L.b2j_encode_bound(self._h), W * H * 3 * 2 + 65536), np.uint8)
        n = C.c_size_t(0)
        self._ck(self._L.b2j_encode(self._h, _ptr(img), img.strides[0], W, H, _ptr(out), out.size, C.byref(n)))
        return out[: n.value]

    def encode_ptr(self, ptr, step, W, H, out_ptr, cap):
        n = C.c_size_t(0)
        self._ck(self._L.b2j_encode(self._h, C.c_void_p(ptr), step, W, H, C.c_void_p(out_ptr), cap, C.byref(n)))
        return n.value

    def decode(self, jpg):
        jpg = np.ascontiguousarray(jpg, np.uint8)
        W, H = C.c_int(0), C.c_int(0)
        self._ck(self._L.b2j_decode(self._h, _ptr(jpg), jpg.size, None, 0, C.byref(W), C.byref(H)))
        shape = (H.value, W.value) if self.channels == 1 else (H.value, W.value, 3)
        out = np.empty(shape, np.uint8)
        self._ck(self._L.b2j_decode(self._h, _ptr(jpg), jpg.size, _ptr(out), W.value * self.channels, C.byref(W), C.byref(H)))
        return out

    def decode_ptr(self, jpg, out_ptr, step):
        W, H = C.c_int(0), C.c_int(0)
        self._ck(self._L.b2j_decode(self._h, _ptr(jpg), jpg.size, C.c_void_p(out_ptr), step, C.byref(W), C.byref(H)))
        return W.value, H.value

    @staticmethod
    def peek(jpg):
        jpg = np.ascontiguousarray(jpg, np.uint8)
        W, H, css = C.c_int(0), C.c_int(0), C.c_int(0)
        rc = N.lib().b2j_peek(_ptr(jpg), jpg.size, C.byref(W), C.byref(H), C.byref(css))
        if rc:
            raise B2JError(rc, "b2j_peek")
        return W.value, H.value, css.value

    def diff(self, a, b, mode=0):
        a = np.ascontiguousarray(a, np.uint8)
        b = np.ascontiguousarray(b, np.uint8)
        out = np.empty_like(a)
        self._ck(self._L.b2j_diff(self._h, _ptr(a), _ptr(b), a.size, int(mode), _ptr(out)))
        return out

    def psnr(self, a, b):
        a = np.ascontiguousarray(a, np.uint8)
        b = np.ascontiguousarray(b, np.uint8)
        ps, ssd = C.c_double(0), C.c_uint64(0)
        self._ck(self._L.b2j_psnr(self._h, _ptr(a), _ptr(b), a.size, C.byref(ps), C.byref(ssd)))
        return ps.value, ssd.value

    def secondary(self, img, diff_mode=1, want_recon=True):
        img = np.asarray(img)
        H, W = img.shape[:2]
        cap = min(self._L.b2j_encode_bound(self._h), W * H * 3 + 65536)
        j1, j2 = np.empty(cap, np.uint8), np.empty(cap, np.uint8)
        n1, n2, ps = C.c_size_t(0), C.c_size_t(0), C.c_double(0)
        recon = np.empty((H, W, 3), np.uint8) if want_recon else None
        self._ck(self._L.b2j_secondary(self._h, _ptr(img), img.strides[0], W, H, int(diff_mode), _ptr(j1), cap,
                                       C.byref(n1), _ptr(j2), cap, C.byref(n2),
                                       _ptr(recon) if want_recon else None, W * 3, C.byref(ps)))
        return j1[: n1.value], j2[: n2.value], recon, ps.value

    def set_restart_rows(self, rows):
        """Restart markers every `rows` MCU rows (0 = none); the stream equals cv2's with RST_INTERVAL = rows * mcux."""
        self._ck(self._L.b2j_set_restart_rows(self._h, int(rows)))

    def set_decode_scale(self, denom):
        """Decode at 1/denom (1, 2, 4 or 8; 1 = full size, the default): libjpeg's DCT scaling, the pixels of
        cv2.imdecode(IMREAD_REDUCED_COLOR_denom) / IMREAD_REDUCED_GRAYSCALE_denom on a gray context. decode returns and
        decode_device / decode_scan_device write and report the reduced size ceil(W / denom) x ceil(H / denom)."""
        self._ck(self._L.b2j_set_decode_scale(self._h, int(denom)))

    def set_decode_region(self, x, y=None, w=None, h=None):
        """Decode only columns x .. x + w - 1 and rows y .. y + h - 1 of the output (after the decode scale): decode
        returns and decode_device / decode_scan_device write and report that (h, w) rectangle of what they would return
        without it. set_decode_region(None) (or 0, 0, 0, 0) is the whole image. A region outside a file's output size
        makes its decode fail before anything is written."""
        if x is None:
            x = y = w = h = 0
        self._ck(self._L.b2j_set_decode_region(self._h, int(x), int(y), int(w), int(h)))

    # ---------------------------------------------------------------- device API (pointers from torch tensors)
    def decode_scan_device(self, hdr, d_scan_ptr, scan_len, d_bgr_ptr, step, height_override=0):
        """Baseline JPEG with its scan bytes already in device memory (hdr: host bytes SOI .. SOS header) -> (W, H)."""
        hdr = np.ascontiguousarray(hdr, np.uint8)
        W, H = C.c_int(0), C.c_int(0)
        self._ck(self._L.b2j_decode_scan_device(self._h, _ptr(hdr), hdr.size, C.c_void_p(d_scan_ptr), int(scan_len), int(height_override),
                                                C.c_void_p(d_bgr_ptr), step, C.byref(W), C.byref(H)))
        return W.value, H.value

    def reconstruct_device(self, d_bgr_ptr, step):
        """Pixels of the last encode (made with set_debug(1)) from its quantised coefficients; asynchronous."""
        self._ck(self._L.b2j_reconstruct_device(self._h, C.c_void_p(d_bgr_ptr), step))

    def reconstruct_planes(self):
        """First half of reconstruct_device (de-quantise + IDCT); -> N.ReconPlanes (device pointers of the edge / halo rows)."""
        rp = N.ReconPlanes()
        self._ck(self._L.b2j_reconstruct_planes(self._h, C.byref(rp)))
        return rp

    def reconstruct_color(self, d_bgr_ptr, step, halo_top=False, halo_bottom=False):
        self._ck(self._L.b2j_reconstruct_color(self._h, C.c_void_p(d_bgr_ptr), step, int(halo_top), int(halo_bottom)))

    def secondary_device(self, d_ptr, step, W, H, diff_mode=1):
        """Device-resident secondary compression, asynchronous -> device pointers (jpg1, jpg2, recon, diff)."""
        p = [C.c_void_p() for _ in range(4)]
        self._ck(self._L.b2j_secondary_device(self._h, C.c_void_p(d_ptr), step, W, H, int(diff_mode), *[C.byref(x) for x in p]))
        return tuple(x.value for x in p)

    def secondary_finish(self):
        """-> (len1, len2, psnr, ssd) of the last secondary_device"""
        n1, n2, ps, ssd = C.c_size_t(0), C.c_size_t(0), C.c_double(0), C.c_uint64(0)
        self._ck(self._L.b2j_secondary_finish(self._h, C.byref(n1), C.byref(n2), C.byref(ps), C.byref(ssd)))
        return n1.value, n2.value, ps.value, ssd.value

    def set_stream(self, cuda_stream_ptr):
        self._ck(self._L.b2j_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def encode_device(self, d_ptr, step, W, H):
        """Asynchronous; returns (device pointer of the JPEG, device pointer of its uint64 length)."""
        o, l = C.c_void_p(), C.c_void_p()
        self._ck(self._L.b2j_encode_device(self._h, C.c_void_p(d_ptr), step, W, H, C.byref(o), C.byref(l)))
        return o.value, l.value

    def encode_finish(self):
        n = C.c_size_t(0)
        self._ck(self._L.b2j_encode_finish(self._h, C.byref(n)))
        return n.value

    def decode_device(self, jpg, d_ptr, step):
        """Asynchronous; call decode_finish() before using the pixels (it validates the decode and keeps `jpg` alive)."""
        jpg = np.ascontiguousarray(jpg, np.uint8)
        self._pending_jpg = jpg
        W, H = C.c_int(0), C.c_int(0)
        self._ck(self._L.b2j_decode_device(self._h, _ptr(jpg), jpg.size, C.c_void_p(d_ptr), step, C.byref(W), C.byref(H)))
        return W.value, H.value

    def decode_finish(self):
        self._ck(self._L.b2j_decode_finish(self._h))
        self._pending_jpg = None

    def diff_psnr_device(self, a_ptr, b_ptr, n, mode, out_ptr):
        s = C.c_void_p()
        self._ck(self._L.b2j_diff_psnr_device(self._h, C.c_void_p(a_ptr), C.c_void_p(b_ptr), n, mode,
                                              C.c_void_p(out_ptr) if out_ptr else None, C.byref(s)))
        return s.value

    # staged strip interface
    def strip_state(self):
        st = N.StripState()
        self._ck(self._L.b2j_strip_state_get(self._h, C.byref(st)))
        return st

    def strip_phase1(self, d_ptr, step, W, rows):
        self._ck(self._L.b2j_strip_phase1(self._h, C.c_void_p(d_ptr), step, W, rows))

    def strip_phase1b(self):
        self._ck(self._L.b2j_strip_phase1b(self._h))

    def strip_phase2(self, full_w, full_h):
        self._ck(self._L.b2j_strip_phase2(self._h, full_w, full_h))

    def strip_phase3(self, skip_bits, ext_byte, flags):
        self._ck(self._L.b2j_strip_phase3(self._h, skip_bits, ext_byte, flags))

    def strip_phase3_dev(self, d_bits_all, rank, world, flags):
        self._ck(self._L.b2j_strip_phase3_dev(self._h, C.c_void_p(d_bits_all), rank, world, flags))

    def strip_phase1x(self, d_ptr, step, W, rows):
        self._ck(self._L.b2j_strip_phase1x(self._h, C.c_void_p(d_ptr), step, W, rows))

    def strip_phase2x(self, d_records_all, rank, world, full_w, full_h, flags):
        """d_records_all = None: peer-memory exchange (after peer_connect)."""
        self._ck(self._L.b2j_strip_phase2x(self._h, C.c_void_p(d_records_all), rank, world, full_w, full_h, flags))

    # peer-memory exchange set-up
    def peer_export(self):
        """-> (64-byte IPC handle, raw device pointer of this context's arena)."""
        h = C.create_string_buffer(64)
        p = C.c_void_p(0)
        self._ck(self._L.b2j_peer_export(self._h, h, C.byref(p)))
        return h.raw, p.value

    def peer_open(self, handle):
        p = C.c_void_p(0)
        self._ck(self._L.b2j_peer_open(self._h, C.create_string_buffer(handle, 64), C.byref(p)))
        return p.value

    def peer_connect(self, rank, world, arenas):
        arr = (C.c_void_p * world)(*[C.c_void_p(a or 0) for a in arenas])
        self._ck(self._L.b2j_peer_connect(self._h, rank, world, arr))

    # introspection
    def debug_read(self, what, dtype, count_hint=None):
        n = C.c_size_t(0)
        rc = self._L.b2j_debug_read(self._h, what, C.c_void_p(C.addressof(C.c_char())), 0, C.byref(n))
        if rc not in (0, -4):
            self._ck(rc)
        buf = np.empty(max(1, n.value), np.uint8)
        self._ck(self._L.b2j_debug_read(self._h, what, _ptr(buf), buf.size, C.byref(n)))
        return buf[: n.value].view(dtype)

    def set_debug(self, flags=1):
        self._ck(self._L.b2j_set_debug(self._h, int(flags)))

    def tables(self):
        raw = self.debug_read(N.DBG_TABLES, np.uint8)
        return N.HuffDev.from_buffer_copy(raw.tobytes())

    def enable_timing(self, on=True):
        self._ck(self._L.b2j_enable_timing(self._h, int(on)))

    def timings(self):
        t = N.Timings()
        self._ck(self._L.b2j_last_timings(self._h, C.byref(t)))
        return {n: getattr(t, n) for n, _ in N.Timings._fields_}

    def launch_count(self):
        return int(self._L.b2j_launch_count(self._h))


class MultiEngine:
    """One image over several GPUs from ONE process (b2j_multi_*): MCU-row strips, records exchanged through peer
    memory, every strip uploaded over its own GPU's link. encode() returns the single-GPU stream byte for byte."""

    def __init__(self, width, height, quality=95, optimize=True, css="422", devices=(0,)):
        self._L = N.lib()
        self._h = None
        if css_id(css) == N.CSS_GRAY:
            raise B2JError(-1, "MultiEngine: gray images are encoded on one GPU (Engine); the strips assume three components")
        p = N.Params()
        self._L.b2j_default_params(C.byref(p))
        p.width, p.height, p.quality, p.optimize = int(width), int(height), int(quality), int(bool(optimize))
        p.css = N.CSS[css] if isinstance(css, str) else int(css)
        self._h = C.c_void_p()
        ids = (C.c_int * len(devices))(*[int(d) for d in devices])
        rc = self._L.b2j_multi_create(C.byref(p), len(devices), ids, C.byref(self._h))
        if rc:
            raise B2JError(rc, "b2j_multi_create failed")
        self.W, self.H = int(width), int(height)

    def encode(self, img, out=None):
        img = np.asarray(img)
        H, W = img.shape[:2]
        if out is None:
            out = np.empty(W * H * 3 // 2 + 65536, np.uint8)
        n = C.c_size_t(0)
        rc = self._L.b2j_multi_encode(self._h, _ptr(img), img.strides[0], W, H, _ptr(out), out.size, C.byref(n))
        if rc:
            raise B2JError(rc, self._L.b2j_multi_last_error(self._h).decode())
        return out[: n.value]

    def encode_ptr(self, src_ptr, step, W, H, out_ptr, cap):
        n = C.c_size_t(0)
        rc = self._L.b2j_multi_encode(self._h, C.c_void_p(src_ptr), step, W, H, C.c_void_p(out_ptr), cap, C.byref(n))
        if rc:
            raise B2JError(rc, self._L.b2j_multi_last_error(self._h).decode())
        return n.value

    def close(self):
        if self._h:
            self._L.b2j_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
