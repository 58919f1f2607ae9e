"""GPU: gray (B2J_CSS_GRAY, one byte per pixel) contexts against the grayscale CPU checker (oracle/,
pinned to libjpeg-turbo by tests/test_oracle_gray.py) and the committed digests of tests/golden/golden_gray.json."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import oracle as O

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
SIZES = ((1, 1), (2, 2), (8, 8), (17, 33), (33, 17), (135, 121), (257, 63), (640, 360))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def P():
    import nvjpeg_imagecompressor_b200 as P
    P.lib()
    return P


@pytest.fixture(scope="module")
def golden_gray():
    with open(os.path.join(HERE, "golden", "golden_gray.json")) as f:
        return json.load(f)


def gray_img(oracle, W, H, seed):
    return np.ascontiguousarray(oracle.synth(W, H, seed, 8)[..., 1])


def pinned_copy(P, img):
    """img in page-locked host memory (b2j_host_alloc): the direct DMA path instead of the staging ring"""
    L = P.lib()
    p = L.b2j_host_alloc(img.nbytes)
    assert p
    buf = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(img.nbytes,)).reshape(img.shape)
    buf[...] = img
    return buf, p


def test_encode_matrix_vs_checker_and_golden(P, oracle, golden_gray):
    engines = {}
    for c in golden_gray["encode"]:
        W, H = c["W"], c["H"]
        key = (W, H, c["quality"], c["optimize"])
        if key not in engines:
            engines.clear()
            engines[key] = P.Engine(W, H, c["quality"], bool(c["optimize"]), "gray", device=0)
        eng = engines[key]
        mcux = (W + 7) // 8
        if c["restart_interval"] % mcux:
            continue   # b2j_set_restart_rows: whole rows of blocks
        eng.set_restart_rows(c["restart_interval"] // mcux)
        img = gray_img(oracle, W, H, c["seed"])
        jpg = eng.encode(img)
        assert jpg.size == c["jpeg_len"] and sha(jpg)[:32] == c["jpeg_sha256_128"], c
        assert np.array_equal(jpg, O.encode_gray(img, c["quality"], c["optimize"], c["restart_interval"])), c


@pytest.mark.parametrize("W,H", SIZES)
def test_encode_pinned_pitch_and_shapes(P, oracle, W, H):
    big = gray_img(oracle, W + 21, H, W * 5 + H)
    img = big[:, 5:5 + W]   # pitch != width
    for q, opt, rows in ((95, 1, 0), (75, 0, 1), (100, 1, 2)):
        eng = P.Engine(W, H, q, bool(opt), "400", device=0)
        eng.set_restart_rows(rows)
        want = O.encode_gray(img, q, opt, rows * ((W + 7) // 8))
        assert np.array_equal(eng.encode(img), want), (W, H, q, opt, rows, "pageable, pitch")
        assert np.array_equal(eng.encode(np.ascontiguousarray(img)[:, :, None]), want), (W, H, q, opt, rows, "(H, W, 1)")
        buf, p = pinned_copy(P, np.ascontiguousarray(img))
        try:
            assert np.array_equal(eng.encode(buf), want), (W, H, q, opt, rows, "pinned")
        finally:
            P.lib().b2j_host_free(p)
        eng.close()


def test_special_images(P, oracle):
    H, W = 45, 70
    rng = np.random.default_rng(5)
    imgs = [np.full((H, W), 77, np.uint8), np.where(rng.random((H, W)) < 0.5, 0, 255).astype(np.uint8),
            ((np.indices((H, W)).sum(0) & 1) * 255).astype(np.uint8)]
    for q, opt in ((100, 1), (95, 0), (40, 1)):
        eng = P.Engine(W, H, q, bool(opt), "gray", device=0)
        for img in imgs:
            assert np.array_equal(eng.encode(img), O.encode_gray(img, q, opt)), (q, opt)


def test_device_entry_points(P, oracle):
    import torch
    W, H = 1000, 300   # several fdct tiles per row, an odd last tile
    img = gray_img(oracle, W, H, 3)
    mcux = (W + 7) // 8
    for opt in (1, 0):
        for rows in (0, 1, 3):
            for dbg in (0, 2):   # bit 1: small pack buffers (the entropy coder's overflow path)
                eng = P.Engine(W, H, 90, bool(opt), "gray", device=0)
                eng.set_restart_rows(rows)
                eng.set_debug(dbg)
                want = O.encode_gray(img, 90, opt, rows * mcux)
                d = torch.from_numpy(img).cuda()
                o, _ = eng.encode_device(d.data_ptr(), W, W, H)
                n = eng.encode_finish()
                got = np.empty(n, np.uint8)
                P.lib().b2j_encode_fetch(eng._h, got.ctypes.data_as(C.c_void_p), n)
                assert np.array_equal(got, want), (opt, rows, dbg, "encode_device")
                ln = C.c_size_t(0)
                eng._ck(P.lib().b2j_encode_begin(eng._h, img.ctypes.data_as(C.c_void_p), W, W, H, C.byref(ln)))
                got = np.empty(ln.value, np.uint8)
                eng._ck(P.lib().b2j_encode_fetch(eng._h, got.ctypes.data_as(C.c_void_p), got.size))
                assert np.array_equal(got, want), (opt, rows, dbg, "encode_begin/fetch")
                eng.close()


def _decode_all_ways(P, eng, jpg, want, tag):
    import torch
    assert np.array_equal(eng.decode(jpg), want), (tag, "decode")
    H, W = want.shape
    for dbg in (0, 4):   # bit 2: the short synchronisation schedule (validated retry)
        eng.set_debug(dbg)
        out = torch.zeros((H, W + 3), dtype=torch.uint8, device="cuda")   # pitch W + 3
        eng.decode_device(jpg, out.data_ptr(), W + 3)
        eng.decode_finish()
        assert np.array_equal(out[:, :W].cpu().numpy(), want), (tag, "decode_device", dbg)
    eng.set_debug(0)


def test_decode_gray_files_and_matrix(P, oracle, golden_gray):
    for f in golden_gray["files"]:
        jpg = np.fromfile(os.path.join(HERE, "golden", f["file"]), np.uint8)
        eng = P.Engine(f["W"], f["H"], 95, True, "gray", device=0)
        want = O.decode_gray(jpg)
        assert sha(want) == f["decoded_sha256"]
        _decode_all_ways(P, eng, jpg, want, f["file"])
    for (W, H) in SIZES:
        img = gray_img(oracle, W, H, W + 3 * H)
        eng = P.Engine(W, H, 95, True, "gray", device=0)
        for q, opt, ri in ((95, 1, 0), (75, 0, 1), (90, 1, (W + 7) // 8)):
            jpg = O.encode_gray(img, q, opt, ri)
            _decode_all_ways(P, eng, jpg, O.decode_gray(jpg), (W, H, q, opt, ri))


def test_decode_y_plane_of_colour_files(P, oracle, golden_gray):
    engines = {}
    for c in golden_gray["ydecode"]:
        img = oracle.synth(c["W"], c["H"], c["seed"], 8)
        if c["kind"] == "prog":
            jpg = oracle.encode_progressive(img, c["css"], c["quality"])
        else:
            jpg = oracle.encode(img, c["css"], c["quality"], c["optimize"], c["restart_interval"])
        key = (c["W"], c["H"])
        if key not in engines:
            engines[key] = P.Engine(c["W"], c["H"], 95, True, "gray", device=0)
        want = O.decode_gray(jpg)
        assert sha(want)[:32] == c["gray_sha256_128"], c
        _decode_all_ways(P, engines[key], jpg, want, c)


def test_decode_scan_device_restart_file(P, oracle):
    import torch
    W, H = 257, 63
    img = gray_img(oracle, W, H, 17)
    mcux = (W + 7) // 8
    jpg = O.encode_gray(img, 90, 1, 2 * mcux)
    b = jpg.tobytes()
    p = 2
    while b[p + 1] != 0xDA:
        p += 2 + ((b[p + 2] << 8) | b[p + 3])
    hdr_len = p + 2 + ((b[p + 2] << 8) | b[p + 3])
    scan = torch.from_numpy(jpg[hdr_len:-2].copy()).cuda()
    out = torch.zeros((H, W), dtype=torch.uint8, device="cuda")
    eng = P.Engine(W, H, 90, True, "gray", device=0)
    assert eng.decode_scan_device(jpg[:hdr_len], scan.data_ptr(), scan.numel(), out.data_ptr(), W) == (W, H)
    assert np.array_equal(out.cpu().numpy(), O.decode_gray(jpg))


def test_colour_gray_cross(P, oracle):
    W, H = 135, 121
    gray_file = O.encode_gray(gray_img(oracle, W, H, 1), 90, 1)
    colour_file = oracle.encode(oracle.synth(W, H, 1, 8), 1, 90, 1)
    g = P.Engine(W, H, 90, True, "gray", device=0)
    assert np.array_equal(g.decode(colour_file), O.decode_gray(colour_file))
    c = P.Engine(W, H, 90, True, "422", device=0)
    for f in (gray_file, cv2_progressive_gray(gray_img(oracle, W, H, 1))):
        if f is None:
            continue
        with pytest.raises(P.B2JError) as e:
            c.decode(f)
        assert e.value.rc == -5
    assert P.Engine.peek(gray_file) == (W, H, 6)


def cv2_progressive_gray(img):
    try:
        import cv2
    except ImportError:
        return None
    return cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].ravel()


def test_gray_refusals(P, oracle):
    import torch
    from nvjpeg_imagecompressor_b200 import _native as N
    L = P.lib()
    W, H = 64, 48
    eng = P.Engine(W, H, 90, True, "gray", device=0)
    d = torch.zeros((H, W * 3), dtype=torch.uint8, device="cuda")
    vp = C.c_void_p
    st = N.StripState()
    rp = N.ReconPlanes()
    calls = {
        "b2j_strip_state_get": lambda: L.b2j_strip_state_get(eng._h, C.byref(st)),
        "b2j_strip_phase1": lambda: L.b2j_strip_phase1(eng._h, vp(d.data_ptr()), W, W, H),
        "b2j_strip_phase1b": lambda: L.b2j_strip_phase1b(eng._h),
        "b2j_strip_phase2": lambda: L.b2j_strip_phase2(eng._h, W, H),
        "b2j_strip_phase3": lambda: L.b2j_strip_phase3(eng._h, 0, 0xFF, 3),
        "b2j_strip_phase1x": lambda: L.b2j_strip_phase1x(eng._h, vp(d.data_ptr()), W, W, H),
        "b2j_peer_export": lambda: L.b2j_peer_export(eng._h, None, C.byref(vp())),
        "b2j_reconstruct_device": lambda: L.b2j_reconstruct_device(eng._h, vp(d.data_ptr()), W),
        "b2j_reconstruct_planes": lambda: L.b2j_reconstruct_planes(eng._h, C.byref(rp)),
        "b2j_reconstruct_color": lambda: L.b2j_reconstruct_color(eng._h, vp(d.data_ptr()), W, 0, 0),
        "b2j_secondary_device": lambda: L.b2j_secondary_device(eng._h, vp(d.data_ptr()), W, W, H, 1, None, None, None, None),
        "b2j_secondary_finish": lambda: L.b2j_secondary_finish(eng._h, None, None, None, None),
        "b2j_secondary_fetch": lambda: L.b2j_secondary_fetch(eng._h, None, 0, None, 0, None, 0),
    }
    for name, call in calls.items():
        assert call() == -1, name
        assert "gray" in L.b2j_last_error(eng._h).decode(), name
    img = np.zeros((H, W), np.uint8)
    jbuf = np.empty(W * H * 4 + 4096, np.uint8)
    rc = L.b2j_secondary(eng._h, img.ctypes.data_as(vp), W, W, H, 1, jbuf.ctypes.data_as(vp), jbuf.size, None, None, 0, None,
                         None, 0, None)
    assert rc == -1
    p = N.Params(W, H, 90, 1, 6, 0, 0)
    h = vp()
    assert L.b2j_multi_create(C.byref(p), 1, None, C.byref(h)) == -1
    with pytest.raises(P.B2JError):
        P.MultiEngine(W, H, 90, True, "gray", devices=(0,))
    from nvjpeg_imagecompressor_b200.strips import StripEncoder
    with pytest.raises(P.B2JError):
        StripEncoder(W, H, 90, True, "gray", rank=0, world=1)
    p5 = N.Params(W, H, 90, 1, 5, 0, 0)
    assert L.b2j_create(C.byref(p5), C.byref(vp())) == -1   # 5 stays invalid
    # the byte-wise helpers work on gray contexts
    a, b = np.arange(W * H, dtype=np.uint8), np.zeros(W * H, np.uint8)
    assert np.array_equal(eng.diff(a, b, 0), oracle.diff(a, b, 0))


def test_headline_gray_digests(P, oracle, golden_gray):
    import torch
    h = golden_gray["headline"]
    W, H = h["W"], h["H"]
    img = torch.empty((H, W), dtype=torch.uint8)
    step = 2000
    for y0 in range(0, H, step):
        img[y0:y0 + step] = torch.from_numpy(oracle.synth(W, H, 0, 8, y0=y0, rows=min(step, H - y0))[..., 1])
    d = img.cuda()
    jpg1 = None
    for opt in (1, 0):
        eng = P.Engine(W, H, h["quality"], bool(opt), "gray", device=0)
        o, _ = eng.encode_device(d.data_ptr(), W, W, H)
        n = eng.encode_finish()
        assert n == h["jpeg_len_opt%d" % opt]
        buf = torch.empty(n, dtype=torch.uint8)
        eng._ck(P.lib().b2j_encode_fetch(eng._h, C.c_void_p(buf.data_ptr()), n))
        jpg = buf.numpy()
        assert sha(jpg) == h["jpeg_sha256_opt%d" % opt], opt
        if opt:
            jpg1 = (eng, jpg)
        else:
            eng.close()
    eng, jpg = jpg1
    del d
    out = torch.empty((H, W), dtype=torch.uint8, device="cuda")
    eng.decode_device(jpg, out.data_ptr(), W)
    eng.decode_finish()
    assert sha(out.cpu().numpy()) == h["decoded_sha256"]
