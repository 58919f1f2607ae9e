"""GPU: region decode (b2j_set_decode_region): every decode entry point returns exactly the crop of what it returns
without a region, i.e. of the CPU checker's output (oracle.decode / decode_gray / decode_scaled, pinned to libjpeg-turbo
by the oracle tests), at every scale, for baseline, restart-marker and progressive files, on colour and gray contexts.
Not one byte outside the rectangle of the caller's buffer (pitch padding included) is written; restart intervals away
from the region are not decoded at all."""
import ctypes as C

import numpy as np
import pytest

import oracle as O

pytestmark = pytest.mark.gpu
CSS_NAMES = ("444", "422", "440", "420", "411")
SIZES = ((1, 1), (5, 3), (2, 40), (40, 2), (9, 17), (33, 17), (67, 93), (250, 301))
SCALES = (1, 2, 4, 8)
SENT = 0xA5   # sentinel the output buffers are filled with


@pytest.fixture(scope="module")
def P():
    import nvjpeg_imagecompressor_b200 as P
    P.lib()
    return P


def reference(jpg, d, gray):
    """the CPU checker's whole output at 1 / d"""
    if d == 1:
        return O.decode_gray(jpg) if gray else O.decode(jpg)
    return O.decode_scaled(jpg, d, gray=gray)


def split_scan(jpg):
    """(header bytes SOI .. SOS header, stuffed scan bytes) of a baseline file"""
    b = jpg.tobytes()
    p = 2
    while b[p + 1] != 0xDA:
        p += 2 + ((b[p + 2] << 8) | b[p + 3])
    hdr_len = p + 2 + ((b[p + 2] << 8) | b[p + 3])
    return jpg[:hdr_len], jpg[hdr_len:-2].copy()


def regions(OW, OH, mw, mh, rng):
    """(x, y, w, h) inside an OW x OH output whose MCUs are mw x mh output pixels: the whole image, one row, one column,
    rectangles touching each edge, on and off MCU and chroma-sample boundaries"""
    def rnd(n):
        return int(rng.integers(0, n)) if n > 0 else 0
    out = [(0, 0, OW, OH)]
    y = rnd(OH)
    out.append((rnd(OW), y, 0, 1))
    x = rnd(OW)
    out.append((x, rnd(OH), 1, 0))
    w, h = 1 + rnd(OW), 1 + rnd(OH)
    out += [(0, rnd(OH - h + 1), w, h), (rnd(OW - w + 1), 0, w, h), (OW - w, rnd(OH - h + 1), w, h), (rnd(OW - w + 1), OH - h, w, h)]
    # on MCU boundaries, and one chroma sample / one pixel off them
    for off in (0, 1, mw // 2 + 1):
        x0 = min(OW - 1, (rnd(OW) // mw) * mw + off)
        y0 = min(OH - 1, (rnd(OH) // mh) * mh + off % max(1, mh))
        w = min(OW - x0, max(1, (rnd(OW) // mw) * mw - off % 2))
        h = min(OH - y0, max(1, (rnd(OH) // mh) * mh + off % 2))
        out.append((x0, y0, w, h))
    res = []
    for x, y, w, h in out:
        w = w or OW - x
        h = h or OH - y
        res.append((x, y, min(w, OW - x), min(h, OH - y)))
    return res


def check_region(P, eng, jpg, full, rect, tag, scan_device=True):
    """host decode into a pitched buffer, decode_device (pitch != w, normal and short synchronisation schedule) and
    decode_scan_device: each gives full[y:y+h, x:x+w] and leaves every other byte of its buffer alone"""
    import torch
    x, y, w, h = rect
    ch = 1 if full.ndim == 2 else 3
    want = full[y:y + h, x:x + w]
    eng.set_decode_region(x, y, w, h)
    got = eng.decode(jpg)
    assert got.shape == want.shape and np.array_equal(got, want), (tag, rect, "decode")
    pitch = w * ch + 7
    host = np.full((h + 1, pitch), SENT, np.uint8)
    assert eng.decode_ptr(jpg, host.ctypes.data, pitch) == (w, h)
    assert np.array_equal(host[:h, :w * ch].reshape(want.shape), want), (tag, rect, "decode pitched")
    assert (host[:h, w * ch:] == SENT).all() and (host[h:] == SENT).all(), (tag, rect, "decode wrote outside")
    for dbg in (0, 4):   # bit 2: the short synchronisation schedule (its checked retry keeps the region)
        eng.set_debug(dbg)
        out = torch.full((h + 1, w * ch + 5), SENT, dtype=torch.uint8, device="cuda")
        assert eng.decode_device(jpg, out.data_ptr(), w * ch + 5) == (w, h), tag
        eng.decode_finish()
        o = out.cpu().numpy()
        assert np.array_equal(o[:h, :w * ch].reshape(want.shape), want), (tag, rect, "decode_device", dbg)
        assert (o[:h, w * ch:] == SENT).all() and (o[h:] == SENT).all(), (tag, rect, "decode_device wrote outside", dbg)
    eng.set_debug(0)
    if scan_device:
        hdr, scan = split_scan(jpg)
        d_scan = torch.from_numpy(scan).cuda()
        out = torch.full((h + 1, w * ch + 3), SENT, dtype=torch.uint8, device="cuda")
        assert eng.decode_scan_device(hdr, d_scan.data_ptr(), d_scan.numel(), out.data_ptr(), w * ch + 3) == (w, h), tag
        o = out.cpu().numpy()
        assert np.array_equal(o[:h, :w * ch].reshape(want.shape), want), (tag, rect, "decode_scan_device")
        assert (o[:h, w * ch:] == SENT).all() and (o[h:] == SENT).all(), (tag, rect, "decode_scan_device wrote outside")


def mcu_out(css, d, gray_file=False):
    """MCU size in output pixels at 1 / d"""
    if gray_file:
        return max(1, 8 // d), max(1, 8 // d)
    hs, vs = {0: (1, 1), 1: (2, 1), 2: (1, 2), 3: (2, 2), 4: (4, 1)}[css]
    return hs * 8 // d, vs * 8 // d


@pytest.mark.parametrize("css", range(5))
def test_matrix_every_entry_point(P, oracle, css):
    rng = np.random.default_rng(100 + css)
    for (W, H) in SIZES:
        img = oracle.synth(W, H, W * 7 + H, 40)
        mcux = oracle.geometry(W, H, css).mcux
        col = P.Engine(W, H, 95, True, CSS_NAMES[css], device=0)
        gray = P.Engine(W + 32, H + 32, 95, True, "gray", device=0)   # room for the blocks of a 4:4:4 file (the padding)
        for rst in (0, mcux, 7):   # none, one MCU row, 7 MCUs (not whole rows)
            jpg = oracle.encode(img, css, 90, 1, rst)
            for d in SCALES:
                col.set_decode_scale(d)
                gray.set_decode_scale(d)
                fc, fg = reference(jpg, d, False), reference(jpg, d, True)
                OH, OW = fc.shape[:2]
                for rect in regions(OW, OH, *mcu_out(css, d), rng):
                    tag = (W, H, css, rst, d)
                    check_region(P, col, jpg, fc, rect, tag + ("colour",))
                    check_region(P, gray, jpg, fg, rect, tag + ("gray",))
        col.close()
        gray.close()


def test_gray_files(P, oracle):
    rng = np.random.default_rng(7)
    for (W, H) in SIZES:
        img = np.ascontiguousarray(oracle.synth(W, H, W + 3 * H, 40)[..., 1])
        eng = P.Engine(W, H, 95, True, "gray", device=0)
        for rst in (0, (W + 7) // 8, 7):
            jpg = oracle.encode_gray(img, 90, 1, rst)
            for d in SCALES:
                eng.set_decode_scale(d)
                full = reference(jpg, d, True)
                OH, OW = full.shape
                for rect in regions(OW, OH, *mcu_out(0, d, True), rng):
                    check_region(P, eng, jpg, full, rect, (W, H, rst, d, "gray file"))
        eng.close()


def test_every_pixel_of_a_small_image(P, oracle):
    """every 1 x 1 region of a 33 x 17 image at full size, every sampling, with and without restart intervals"""
    W, H = 33, 17
    img = oracle.synth(W, H, 5, 40)
    for css in range(5):
        eng = P.Engine(W, H, 95, True, CSS_NAMES[css], device=0)
        for rst in (0, 1):
            jpg = oracle.encode(img, css, 90, 1, rst)
            full = O.decode(jpg)
            for y in range(H):
                for x in range(W):
                    eng.set_decode_region(x, y, 1, 1)
                    assert np.array_equal(eng.decode(jpg), full[y:y + 1, x:x + 1]), (css, rst, x, y)
        eng.close()


def test_progressive_golden_files(P):
    import os
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    names = sorted(f for f in os.listdir(here) if f.endswith(".jpg") and "prog" in f)
    names += sorted("gray/" + f for f in os.listdir(os.path.join(here, "gray")) if "prog" in f)
    assert len(names) >= 9
    rng = np.random.default_rng(3)
    for name in names:
        jpg = np.fromfile(os.path.join(here, name), np.uint8)
        W, H, css = P.Engine.peek(jpg)
        gfile = css == O.CSS_GRAY
        col = None if gfile else P.Engine(W, H, 95, True, CSS_NAMES[css], device=0)
        gray = P.Engine(W + 32, H + 32, 95, True, "gray", device=0)
        for d in (1, 4):
            for eng, g in ((col, False), (gray, True)):
                if eng is None:
                    continue
                eng.set_decode_scale(d)
                full = reference(jpg, d, g)
                OH, OW = full.shape[:2]
                for rect in regions(OW, OH, *mcu_out(0 if gfile else css, d, gfile), rng)[:6]:
                    check_region(P, eng, jpg, full, rect, (name, d, g), scan_device=False)
        for e in (col, gray):
            if e is not None:
                e.close()


def test_progressive_catalogue_with_restarts(P, oracle):
    import prog_streams as PS
    rng = np.random.default_rng(4)
    picked = [e for e in PS.catalogue(oracle, big=False) if "restart_interval" in e[0]][:6]
    assert len(picked) == 6
    for tag, jpg, ncomp in picked:
        W, H, css = P.Engine.peek(jpg)
        col = None if ncomp == 1 else P.Engine(W, H, 95, True, "444", device=0)
        gray = P.Engine(W + 32, H + 32, 95, True, "gray", device=0)
        for d in (1, 2):
            for eng, g in ((col, False), (gray, True)):
                if eng is None:
                    continue
                eng.set_decode_scale(d)
                full = reference(jpg, d, g)
                OH, OW = full.shape[:2]
                for rect in regions(OW, OH, 8, 8, rng)[:5]:
                    check_region(P, eng, jpg, full, rect, (tag, d, g), scan_device=False)
        for e in (col, gray):
            if e is not None:
                e.close()


def test_other_writers(P, oracle):
    """fill bytes before RSTn, odd restart intervals, long-code tables"""
    import jpeg_streams as J
    rng = np.random.default_rng(5)
    keep = ("fill2_every_marker", "ri7", "ri_row_plus_1", "long_codes", "long_codes_ri5", "skewed_shared_fill1", "fill2_rst_eoi")
    for css in (1, 3, 4):
        src, streams = J.writer_streams(oracle, css)
        W, H, _ = P.Engine.peek(src)
        col = P.Engine(W, H, 95, True, CSS_NAMES[css], device=0)
        gray = P.Engine(W + 32, H + 32, 95, True, "gray", device=0)
        n = 0
        for name, jpg in streams:
            if name not in keep:
                continue
            n += 1
            jpg = np.asarray(jpg, np.uint8)
            for d in (1, 4):
                col.set_decode_scale(d)
                gray.set_decode_scale(d)
                fc, fg = reference(src, d, False), reference(src, d, True)
                OH, OW = fc.shape[:2]
                for rect in regions(OW, OH, *mcu_out(css, d), rng)[:5]:
                    check_region(P, col, jpg, fc, rect, (css, name, d), scan_device=False)
                    check_region(P, gray, jpg, fg, rect, (css, name, d, "gray"), scan_device=False)
        assert n == len(keep)
        col.close()
        gray.close()


def damage_intervals(jpg, rows_to_damage):
    """jpg with the entropy bytes of the given restart intervals replaced by x ^ 0x55 (a resulting 0xFF becomes 0xFE);
    the markers stay"""
    hdr, scan = split_scan(jpg)
    b = scan.tobytes()
    parts, cur, i = [], bytearray(), 0
    while i < len(b):   # split at RSTn, unstuff
        if b[i] == 0xFF and i + 1 < len(b) and 0xD0 <= b[i + 1] <= 0xD7:
            parts.append((cur, b[i:i + 2]))
            cur, i = bytearray(), i + 2
            continue
        cur.append(b[i])
        i += 2 if (b[i] == 0xFF and i + 1 < len(b) and b[i + 1] == 0) else 1
    parts.append((cur, b""))
    out = bytearray()
    for j, (data, mk) in enumerate(parts):
        if j in rows_to_damage:
            data = bytearray(0xFE if (x ^ 0x55) == 0xFF else x ^ 0x55 for x in data)
        for x in data:
            out.append(x)
            if x == 0xFF:
                out.append(0)
        out += mk
    return np.concatenate([hdr, np.frombuffer(bytes(out), np.uint8), np.array([0xFF, 0xD9], np.uint8)])


@pytest.mark.parametrize("css", (1, 3))
def test_intervals_outside_the_region_are_not_decoded(P, oracle, css):
    W, H = 160, 240
    g = oracle.geometry(W, H, css)
    jpg = oracle.encode(oracle.synth(W, H, 21, 40), css, 90, 1, g.mcux)   # one MCU row per interval
    mh = 8 * (2 if css == 3 else 1)
    full = O.decode(jpg)
    eng = P.Engine(W, H, 95, True, CSS_NAMES[css], device=0)
    for (x, y, w, h) in ((10, 100, 50, 30), (0, 0, W, 20), (3, H - 9, 41, 9)):
        r0, r1 = y // mh, (y + h - 1) // mh
        bad = {j for j in range(g.mcuy) if j <= r0 - 2 or j >= r1 + 2}
        assert bad
        dmg = damage_intervals(jpg, bad)
        assert not np.array_equal(O.decode(dmg), full)   # the damage is visible in a whole decode
        check_region(P, eng, dmg, full, (x, y, w, h), (css, x, y, w, h))
    eng.close()


def test_setting_semantics(P, oracle):
    import torch
    W, H = 120, 88
    img = oracle.synth(W, H, 2, 30)
    jpg = oracle.encode(img, 1, 90, 1, 3)
    full = O.decode(jpg)
    L = P.lib()
    eng = P.Engine(W, H, 95, True, "422", device=0)
    eng.set_decode_region(1, 2, 3, 4)
    for bad in ((-1, 0, 4, 4), (0, -1, 4, 4), (0, 0, -4, 4), (0, 0, 4, -4), (0, 0, 5, 0), (0, 0, 0, 5), (1, 0, 0, 0), (0, 1, 0, 0)):
        assert L.b2j_set_decode_region(eng._h, *bad) == -1, bad
    assert L.b2j_set_decode_region(None, 0, 0, 0, 0) == -1
    assert np.array_equal(eng.decode(jpg), full[2:6, 1:4])   # the refusals left the setting alone
    # the size query with a NULL image reports w x h
    Wq, Hq = C.c_int(0), C.c_int(0)
    assert L.b2j_decode(eng._h, jpg.ctypes.data, jpg.size, None, 0, C.byref(Wq), C.byref(Hq)) == 0
    assert (Wq.value, Hq.value) == (3, 4)
    # a region outside the image: -1 naming both sizes, nothing written on any path
    for rect in ((W - 3, 0, 4, 4), (0, H - 1, 1, 2), (W, H, 1, 1)):
        eng.set_decode_region(*rect)
        host = np.full((8, 64), SENT, np.uint8)
        assert L.b2j_decode(eng._h, jpg.ctypes.data, jpg.size, host.ctypes.data, 64, C.byref(Wq), C.byref(Hq)) == -1
        msg = L.b2j_last_error(eng._h).decode()
        assert f"{W}x{H}" in msg and f"{rect[2]}x{rect[3]}" in msg, msg
        assert (host == SENT).all()
        dev = torch.full((8, 64), SENT, dtype=torch.uint8, device="cuda")
        with pytest.raises(P.B2JError):
            eng.decode_device(jpg, dev.data_ptr(), 64)
        eng.decode_finish()
        hdr, scan = split_scan(jpg)
        d_scan = torch.from_numpy(scan).cuda()
        with pytest.raises(P.B2JError):
            eng.decode_scan_device(hdr, d_scan.data_ptr(), d_scan.numel(), dev.data_ptr(), 64)
        torch.cuda.synchronize()
        assert (dev.cpu().numpy() == SENT).all()
    # at a scale the region is checked against the reduced size
    eng.set_decode_scale(8)
    eng.set_decode_region(0, 0, 15, 11)
    assert np.array_equal(eng.decode(jpg), O.decode_scaled(jpg, 8))
    eng.set_decode_region(0, 0, 16, 11)
    with pytest.raises(P.B2JError):
        eng.decode(jpg)
    eng.set_decode_scale(1)
    # (0, 0, 0, 0) and None: a decode equal to that of a context that never had a region
    fresh = P.Engine(W, H, 95, True, "422", device=0)
    for reset in ((0, 0, 0, 0), (None,)):
        eng.set_decode_region(*reset)
        assert np.array_equal(eng.decode(jpg), fresh.decode(jpg)) and np.array_equal(eng.decode(jpg), full)
    fresh.close()
    eng.close()
    # a decode_device keeps the region it was issued with until decode_finish, also on the checked retry: debug flag 4
    # (one scheduled synchronisation launch) makes b2j_decode_finish decode again, which the launch count shows
    W, H = 640, 480
    jpg = oracle.encode(oracle.synth(W, H, 12, 40), 1, 90, 1)
    full = O.decode(jpg)
    eng = P.Engine(W, H, 95, True, "422", device=0)
    launches = {}
    for dbg in (0, 4):
        eng.set_debug(dbg)
        eng.set_decode_region(5, 7, 30, 20)
        out = torch.full((20, 90), SENT, dtype=torch.uint8, device="cuda")
        n0 = eng.launch_count()
        assert eng.decode_device(jpg, out.data_ptr(), 90) == (30, 20)
        eng.set_decode_region(0, 0, W, H)
        eng.set_decode_scale(2)
        eng.decode_finish()
        launches[dbg] = eng.launch_count() - n0
        eng.set_decode_scale(1)
        assert np.array_equal(out.cpu().numpy().reshape(20, 30, 3), full[7:27, 5:35]), dbg
    # without the retry the short schedule would issue two launches fewer than the default one
    assert launches[4] > launches[0], launches
    eng.close()


def test_encode_reconstruct_secondary_ignore_region(P, oracle):
    import torch
    W, H = 96, 64
    img = oracle.synth(W, H, 8, 30)
    a = P.Engine(W, H, 90, True, "420", device=0)
    b = P.Engine(W, H, 90, True, "420", device=0)
    b.set_decode_region(3, 5, 7, 9)
    assert np.array_equal(a.encode(img), b.encode(img))
    ra, rb = a.secondary(img), b.secondary(img)
    for x, y in zip(ra[:3], rb[:3]):
        assert np.array_equal(x, y)
    assert ra[3] == rb[3]
    outs = []
    for e in (a, b):
        e.set_debug(1)
        d = torch.from_numpy(img).cuda()
        e.encode_device(d.data_ptr(), W * 3, W, H)
        e.encode_finish()
        out = torch.full((H, W * 3), SENT, dtype=torch.uint8, device="cuda")
        e.reconstruct_device(out.data_ptr(), W * 3)
        torch.cuda.synchronize()
        outs.append(out.cpu().numpy())
    assert np.array_equal(outs[0], outs[1]) and not (outs[1] == SENT).all()
    a.close()
    b.close()


@pytest.fixture(scope="module")
def headline(oracle):
    """the 8320 x 40000 headline image in device memory"""
    import torch
    W, H = 8320, 40000
    img = torch.empty((H, W, 3), dtype=torch.uint8)
    step = 2000
    for y0 in range(0, H, step):
        img[y0:y0 + step] = torch.from_numpy(oracle.synth(W, H, 1, 8, y0=y0, rows=min(step, H - y0)))
    yield img.cuda()


@pytest.mark.parametrize("rst_rows", (1, 0))
def test_headline_stream(P, headline, rst_rows):
    """8320 x 40000 q95 4:2:2, optimised, with one restart interval per MCU row and with none: four regions at scale 1
    and 8 through decode_scan_device and decode_device equal the crop of the same engine's whole decode"""
    import torch
    H, W = headline.shape[:2]
    eng = P.Engine(W, H, 95, True, "422", device=0)
    eng.set_restart_rows(rst_rows)
    eng.encode_device(headline.data_ptr(), W * 3, W, H)
    n = eng.encode_finish()
    buf = torch.empty(n, dtype=torch.uint8)
    eng._ck(P.lib().b2j_encode_fetch(eng._h, C.c_void_p(buf.data_ptr()), n))
    jpg = buf.numpy()
    hdr, scan = split_scan(jpg)
    d_scan = torch.from_numpy(scan).cuda()
    for dn in (1, 8):
        eng.set_decode_scale(dn)
        eng.set_decode_region(None)
        OW, OH = O.reduced_size(W, H, dn)
        full = torch.empty((OH, OW * 3), dtype=torch.uint8, device="cuda")
        assert eng.decode_scan_device(hdr, d_scan.data_ptr(), d_scan.numel(), full.data_ptr(), OW * 3) == (OW, OH)
        rw, rh = min(1920, OW), min(1080, OH)
        for (x, y, w, h) in ((0, 0, rw, rh), ((OW - rw) // 2, (OH - rh) // 2, rw, rh), (OW - 257, OH - 131, 257, 131),
                             (0, OH // 2 + 1, OW, 17)):
            want = full[y:y + h, 3 * x:3 * (x + w)]
            eng.set_decode_region(x, y, w, h)
            out = torch.full((h, w * 3 + 16), SENT, dtype=torch.uint8, device="cuda")
            assert eng.decode_scan_device(hdr, d_scan.data_ptr(), d_scan.numel(), out.data_ptr(), w * 3 + 16) == (w, h)
            assert torch.equal(out[:, :w * 3], want), (rst_rows, dn, x, y, w, h, "decode_scan_device")
            assert (out[:, w * 3:] == SENT).all()
            out.fill_(SENT)
            assert eng.decode_device(jpg, out.data_ptr(), w * 3 + 16) == (w, h)
            eng.decode_finish()
            assert torch.equal(out[:, :w * 3], want), (rst_rows, dn, x, y, w, h, "decode_device")
            assert (out[:, w * 3:] == SENT).all()
        del full
    eng.close()
