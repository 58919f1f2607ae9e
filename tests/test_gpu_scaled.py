"""GPU: reduced-size decode (b2j_set_decode_scale, libjpeg's DCT scaling at 1/2, 1/4, 1/8) against the CPU checker
(oracle/, pinned to libjpeg-turbo by tests/test_oracle_scaled.py) and the committed digests of
tests/golden/golden_scaled.json."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import oracle as O

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
CSS_NAMES = ("444", "422", "440", "420", "411")
SIZES = ((1, 1), (5, 3), (2, 40), (40, 2), (9, 17), (33, 17), (67, 93), (250, 301))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def P():
    import nvjpeg_imagecompressor_b200 as P
    P.lib()
    return P


@pytest.fixture(scope="module")
def golden_scaled():
    with open(os.path.join(HERE, "golden", "golden_scaled.json")) as f:
        return json.load(f)


def pinned_copy(P, a):
    """a in page-locked host memory (b2j_host_alloc): the direct DMA path instead of the staging ring"""
    p = P.lib().b2j_host_alloc(a.nbytes)
    assert p
    buf = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(a.nbytes,)).reshape(a.shape)
    buf[...] = a
    return buf, p


def split_scan(jpg):
    """(header bytes SOI .. SOS header, stuffed scan bytes) of a baseline file"""
    b = jpg.tobytes()
    p = 2
    while b[p + 1] != 0xDA:
        p += 2 + ((b[p + 2] << 8) | b[p + 3])
    hdr_len = p + 2 + ((b[p + 2] << 8) | b[p + 3])
    return jpg[:hdr_len], jpg[hdr_len:-2].copy()


def decode_every_way(P, eng, jpg, want, tag, scan_device=True):
    """host pageable and pinned, decode_device + finish (pitch != width, normal and short synchronisation schedule),
    decode_scan_device; every one must give `want`"""
    import torch
    ch = 1 if want.ndim == 2 else 3
    H, W = want.shape[:2]
    got = eng.decode(jpg)
    assert got.shape == want.shape and np.array_equal(got, want), (tag, "decode")
    buf, p = pinned_copy(P, jpg)
    try:
        assert np.array_equal(eng.decode(buf), want), (tag, "decode pinned")
    finally:
        P.lib().b2j_host_free(p)
    for dbg in (0, 4):   # bit 2: the short synchronisation schedule (the checked retry keeps the scale)
        eng.set_debug(dbg)
        out = torch.zeros((H, W * ch + 5), dtype=torch.uint8, device="cuda")   # pitch != width
        assert eng.decode_device(jpg, out.data_ptr(), W * ch + 5) == (W, H), tag
        eng.decode_finish()
        assert np.array_equal(out[:, :W * ch].cpu().numpy().reshape(want.shape), want), (tag, "decode_device", dbg)
    eng.set_debug(0)
    if scan_device:
        hdr, scan = split_scan(jpg)
        d_scan = torch.from_numpy(scan).cuda()
        out = torch.zeros((H, W * ch + 3), dtype=torch.uint8, device="cuda")
        assert eng.decode_scan_device(hdr, d_scan.data_ptr(), d_scan.numel(), out.data_ptr(), W * ch + 3) == (W, H), tag
        assert np.array_equal(out[:, :W * ch].cpu().numpy().reshape(want.shape), want), (tag, "decode_scan_device")


@pytest.mark.parametrize("css", range(5))
def test_matrix_every_entry_point(P, oracle, css):
    for (W, H) in SIZES:
        img = oracle.synth(W, H, W * 7 + H, 40)
        mcux = oracle.geometry(W, H, css).mcux
        col = P.Engine(W, H, 95, True, CSS_NAMES[css], device=0)
        # a gray context has room for the blocks of a 4:4:4 file of its size; the MCU padding of the other
        # subsamplings can need more at the tiny sizes, full size and reduced alike
        gray = P.Engine(W + 32, H + 32, 95, True, "gray", device=0)
        for q, rst in ((90, 0), (100, 0), (75, mcux)):
            jpg = oracle.encode(img, css, q, 1, rst)
            for d in O.SCALES:
                col.set_decode_scale(d)
                gray.set_decode_scale(d)
                tag = (W, H, css, q, rst, d)
                decode_every_way(P, col, jpg, O.decode_scaled(jpg, d), tag + ("colour",))
                decode_every_way(P, gray, jpg, O.decode_scaled(jpg, d, gray=True), tag + ("gray",))
        col.close()
        gray.close()


def test_one_component_files(P, golden_scaled):
    """one-component golden files (baseline, restart markers, progressive, SOF sampling 2x2) on a gray context"""
    for f in golden_scaled["files"]:
        if not f["file"].startswith("gray/"):
            continue
        jpg = np.fromfile(os.path.join(HERE, "golden", f["file"]), np.uint8)
        eng = P.Engine(f["W"], f["H"], 95, True, "gray", device=0)
        for d in O.SCALES:
            eng.set_decode_scale(d)
            want = O.decode_scaled(jpg, d, gray=True)
            assert sha(want)[:32] == f["g%d" % d], (f["file"], d)
            decode_every_way(P, eng, jpg, want, (f["file"], d), scan_device="prog" not in f["file"])
        eng.close()


def test_progressive_and_nvjpeg_files(P, golden_scaled):
    import torch
    for f in golden_scaled["files"]:
        if f["file"].startswith("gray/"):
            continue
        jpg = np.fromfile(os.path.join(HERE, "golden", f["file"]), np.uint8)
        css = P.Engine.peek(jpg)[2]
        col = P.Engine(f["W"], f["H"], 95, True, CSS_NAMES[css], device=0)
        gray = P.Engine(f["W"], f["H"], 95, True, "gray", device=0)
        for d in O.SCALES:
            col.set_decode_scale(d)
            gray.set_decode_scale(d)
            W, H = O.reduced_size(f["W"], f["H"], d)
            out = col.decode(jpg)
            assert out.shape == (H, W, 3) and sha(out)[:32] == f["c%d" % d], (f["file"], d, "colour")
            assert sha(gray.decode(jpg))[:32] == f["g%d" % d], (f["file"], d, "gray")
            dev = torch.zeros((H, W * 3 + 7), dtype=torch.uint8, device="cuda")
            assert col.decode_device(jpg, dev.data_ptr(), W * 3 + 7) == (W, H)
            col.decode_finish()
            assert sha(dev[:, :W * 3].cpu().numpy())[:32] == f["c%d" % d], (f["file"], d, "decode_device")
        col.close()
        gray.close()


def test_scale_one_equals_default(P, oracle):
    W, H = 121, 135
    img = oracle.synth(W, H, 9, 8)
    for css in range(5):
        jpg = oracle.encode(img, css, 90, 1, oracle.geometry(W, H, css).mcux)
        plain = P.Engine(W, H, 95, True, CSS_NAMES[css], device=0)
        scaled = P.Engine(W, H, 95, True, CSS_NAMES[css], device=0)
        scaled.set_decode_scale(8)
        assert scaled.decode(jpg).shape == (17, 16, 3)
        scaled.set_decode_scale(1)
        full = plain.decode(jpg)
        assert full.shape == (H, W, 3) and np.array_equal(scaled.decode(jpg), full), css
        assert np.array_equal(full, oracle.decode(jpg)), css


def test_invalid_scales_leave_setting(P, oracle):
    W, H = 64, 48
    jpg = oracle.encode(oracle.synth(W, H, 2, 8), 1, 90, 1)
    eng = P.Engine(W, H, 95, True, "422", device=0)
    eng.set_decode_scale(4)
    L = P.lib()
    for bad in (0, 3, 16, -1):
        assert L.b2j_set_decode_scale(eng._h, bad) == -1, bad
        with pytest.raises(P.B2JError):
            eng.set_decode_scale(bad)
    assert L.b2j_set_decode_scale(None, 2) == -1
    out = eng.decode(jpg)
    assert out.shape == (12, 16, 3) and np.array_equal(out, O.decode_scaled(jpg, 4))
    assert P.Engine.peek(jpg) == (W, H, 1)   # peek reports the file's size
    # a step that fits the reduced width but not the full one is accepted; one below the reduced width is not
    dst = np.empty((12, 16 * 3), np.uint8)
    assert eng.decode_ptr(jpg, dst.ctypes.data, 16 * 3) == (16, 12)
    with pytest.raises(P.B2JError):
        eng.decode_ptr(jpg, dst.ctypes.data, 16 * 3 - 1)


def test_timings_filled(P, oracle):
    W, H = 640, 480
    jpg = oracle.encode(oracle.synth(W, H, 4, 8), 1, 90, 1)
    eng = P.Engine(W, H, 95, True, "422", device=0)
    eng.enable_timing(True)
    for d in O.SCALES:
        eng.set_decode_scale(d)
        assert np.array_equal(eng.decode(jpg), O.decode_scaled(jpg, d))
        t = eng.timings()
        assert t["dec_idct"] > 0 and t["dec_color"] > 0, d


def test_headline_reduced_digests(P, oracle, golden_scaled):
    import torch
    h = golden_scaled["headline"]
    W, H = h["W"], h["H"]
    img = torch.empty((H, W, 3), dtype=torch.uint8)
    step = 2000
    for y0 in range(0, H, step):
        img[y0:y0 + step] = torch.from_numpy(oracle.synth(W, H, h["seed"], h["amp"], y0=y0, rows=min(step, H - y0)))
    d = img.cuda()
    del img
    eng = P.Engine(W, H, h["quality"], True, CSS_NAMES[h["css"]], device=0)
    eng.encode_device(d.data_ptr(), W * 3, W, H)
    n = eng.encode_finish()
    del d
    assert n == h["jpeg_len"]
    buf = torch.empty(n, dtype=torch.uint8)
    eng._ck(P.lib().b2j_encode_fetch(eng._h, C.c_void_p(buf.data_ptr()), n))
    jpg = buf.numpy()
    assert sha(jpg) == h["jpeg_sha256"]
    gray = P.Engine(W, H, h["quality"], True, "gray", device=0)
    for dn in O.SCALES:
        ow, oh = O.reduced_size(W, H, dn)
        eng.set_decode_scale(dn)
        gray.set_decode_scale(dn)
        out = torch.empty((oh, ow * 3), dtype=torch.uint8, device="cuda")
        assert eng.decode_device(jpg, out.data_ptr(), ow * 3) == (ow, oh)
        eng.decode_finish()
        assert sha(out.cpu().numpy()) == h["c%d" % dn], dn
        assert sha(eng.decode(jpg)) == h["c%d" % dn], dn
        assert sha(gray.decode(jpg)) == h["g%d" % dn], dn
