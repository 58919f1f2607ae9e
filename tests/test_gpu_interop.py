"""GPU: JPEG files from other writers (tests/jpeg_streams.py corpus: table slots, SOF1 and 16-bit tables, ids, fill
bytes, split tables, APPn/COM, no EOI, restart intervals of any length, long-code and skewed tables, Pillow files)
decode to exactly cv2's pixels on every decode path, colour, gray and reduced; the files libjpeg decodes as RGB, or
that name a quantisation slot above 3, are refused on every path. Frames at the format's size limits encode to
libjpeg's bytes and decode to its pixels."""
import cv2
import numpy as np
import pytest

import oracle as O
import jpeg_streams as J

pytestmark = pytest.mark.gpu
CSS_NAMES = ("444", "422", "440", "420", "411")
REDUCED = {2: (cv2.IMREAD_REDUCED_COLOR_2, cv2.IMREAD_REDUCED_GRAYSCALE_2),
           4: (cv2.IMREAD_REDUCED_COLOR_4, cv2.IMREAD_REDUCED_GRAYSCALE_4),
           8: (cv2.IMREAD_REDUCED_COLOR_8, cv2.IMREAD_REDUCED_GRAYSCALE_8)}


@pytest.fixture(scope="module")
def P():
    import nvjpeg_imagecompressor_b200 as P
    P.lib()
    return P


@pytest.fixture(scope="module")
def corpus(oracle):
    return J.corpus(oracle)


@pytest.fixture(scope="module")
def engines(P):
    col = P.Engine(96, 96, 95, True, "444", device=0)
    gray = P.Engine(128, 128, 95, True, "gray", device=0)
    yield col, gray
    col.close()
    gray.close()


def dec(jpg, flag):
    out = cv2.imdecode(np.asarray(jpg, np.uint8), flag)
    assert out is not None
    return out


def device_decode(eng, jpg, want_shape, ch, dbg):
    import torch
    H, W = want_shape[:2]
    eng.set_debug(dbg)
    try:
        out = torch.zeros((H, W * ch + 5), dtype=torch.uint8, device="cuda")   # pitch != width
        assert eng.decode_device(jpg, out.data_ptr(), W * ch + 5) == (W, H)
        eng.decode_finish()
        return out[:, :W * ch].cpu().numpy().reshape(want_shape)
    finally:
        eng.set_debug(0)


def test_accepted_streams_decode_like_cv2(engines, corpus):
    col, gray = engines
    n = 0
    for e in corpus:
        if not e["accept"]:
            continue
        jpg, tag = e["jpg"], e["name"]
        for d in (1, 2, 4, 8):
            col.set_decode_scale(d)
            gray.set_decode_scale(d)
            fc, fg = (cv2.IMREAD_COLOR, cv2.IMREAD_GRAYSCALE) if d == 1 else REDUCED[d]
            want, want_g = dec(e["ref"], fc), dec(e["ref"], fg)
            got = col.decode(jpg)
            assert got.shape == want.shape and np.array_equal(got, want), (tag, d, "decode")
            got_g = gray.decode(jpg)
            assert got_g.shape == want_g.shape and np.array_equal(got_g, want_g), (tag, d, "gray decode")
            for dbg in (0, 4):   # bit 2: the short synchronisation schedule
                assert np.array_equal(device_decode(col, jpg, want.shape, 3, dbg), want), (tag, d, "decode_device", dbg)
            assert np.array_equal(device_decode(gray, jpg, want_g.shape, 1, 0), want_g), (tag, d, "gray decode_device")
        n += 1
    col.set_decode_scale(1)
    gray.set_decode_scale(1)
    assert n == sum(e["accept"] for e in corpus) and n >= 140


def test_refused_streams_on_every_path(P, engines, corpus):
    import torch
    col, gray = engines
    out = torch.zeros((96, 96 * 3), dtype=torch.uint8, device="cuda")
    n = 0
    for e in corpus:
        if e["accept"]:
            continue
        jpg, tag = e["jpg"], e["name"]
        with pytest.raises(P.B2JError) as ex:
            P.Engine.peek(jpg)
        assert ex.value.rc == -5, tag
        for eng in (col, gray):
            for d in (1, 8):
                eng.set_decode_scale(d)
                with pytest.raises(P.B2JError) as ex:
                    eng.decode(jpg)
                assert ex.value.rc == -5 and str(ex.value), (tag, d)
                with pytest.raises(P.B2JError) as ex:
                    eng.decode_device(jpg, out.data_ptr(), 96 * 3)
                    eng.decode_finish()
                assert ex.value.rc == -5, (tag, d)
            eng.set_decode_scale(1)
        n += 1
    assert n == sum(not e["accept"] for e in corpus) and n >= 40


# ------------------------------------------------------------------------------------------- the format's size limits
LIMIT_SHAPES = ((65500, 1), (65500, 8), (65500, 17), (1, 65500), (9, 65500))


@pytest.mark.parametrize("W,H", LIMIT_SHAPES)
def test_size_limit_frames(P, oracle, W, H):
    """at libjpeg's 65500: encode bytes == checker == cv2.imencode, decode == cv2.imdecode, 1/8 == IMREAD_REDUCED_8"""
    img = oracle.synth(W, H, W + H, 24)
    assert img.nbytes <= 3_400_000
    g = np.ascontiguousarray(img[:, :, 1])
    for q in (75, 100):
        for opt in (0, 1):
            for css in list(range(5)) + ["gray"]:
                tag = (W, H, q, opt, css)
                eng = P.Engine(W, H, q, bool(opt), "gray" if css == "gray" else CSS_NAMES[css], device=0)
                try:
                    if css == "gray":
                        jpg = eng.encode(g)
                        want = O.encode_gray(g, q, opt)
                        cv = cv2.imencode(".jpg", g, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, opt])[1].ravel()
                        flags = (cv2.IMREAD_GRAYSCALE, cv2.IMREAD_REDUCED_GRAYSCALE_8)
                    else:
                        jpg = eng.encode(img)
                        want = oracle.encode(img, css, q, opt)
                        flags = (cv2.IMREAD_COLOR, cv2.IMREAD_REDUCED_COLOR_8)
                        cv = None
                        if css in (0, 1, 3):   # the subsamplings cv2.imencode can be asked for
                            s = {0: cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, 1: cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
                                 3: cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420}[css]
                            cv = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, opt,
                                                            cv2.IMWRITE_JPEG_SAMPLING_FACTOR, s])[1].ravel()
                    assert np.array_equal(jpg, want), (tag, "encode vs checker")
                    if cv is not None:
                        assert np.array_equal(want, cv), (tag, "checker vs cv2.imencode")
                    got = eng.decode(jpg)
                    assert np.array_equal(got, dec(jpg, flags[0])), (tag, "decode")
                    eng.set_decode_scale(8)
                    got = eng.decode(jpg)
                    assert np.array_equal(got, dec(jpg, flags[1])), (tag, "decode 1/8")
                finally:
                    eng.close()


@pytest.mark.parametrize("H", (1, 17))
def test_width_65535(P, oracle, H):
    """the product's limit, beyond libjpeg's: encode and decode against the checker, which reads up to 65535"""
    W = 65535
    img = oracle.synth(W, H, H, 24)
    g = np.ascontiguousarray(img[:, :, 1])
    for css in list(range(5)) + ["gray"]:
        eng = P.Engine(W, H, 90, True, "gray" if css == "gray" else CSS_NAMES[css], device=0)
        try:
            if css == "gray":
                jpg = eng.encode(g)
                assert np.array_equal(jpg, O.encode_gray(g, 90, 1)), css
                assert np.array_equal(eng.decode(jpg), O.decode_gray(jpg)), css
            else:
                jpg = eng.encode(img)
                assert np.array_equal(jpg, oracle.encode(img, css, 90, 1)), css
                assert np.array_equal(eng.decode(jpg), oracle.decode(jpg)), css
        finally:
            eng.close()


@pytest.mark.parametrize("W", (65500, 65535))
def test_restart_rows_at_the_dri_limit(P, oracle, W):
    """the largest restart-row count b2j_set_restart_rows takes (rows * mcux <= 65535, DRI is 16 bits) writes the
    checker's bytes; one more is B2J_EINVAL"""
    H = 40
    img = oracle.synth(W, H, 7, 24)
    g = np.ascontiguousarray(img[:, :, 1])
    for css in list(range(5)) + ["gray"]:
        eng = P.Engine(W, H, 90, True, "gray" if css == "gray" else CSS_NAMES[css], device=0)
        try:
            mcux = (W + 7) // 8 if css == "gray" else oracle.geometry(W, H, css).mcux
            rows = 65535 // mcux
            with pytest.raises(P.B2JError) as ex:
                eng.set_restart_rows(rows + 1)
            assert ex.value.rc == -1, css
            eng.set_restart_rows(rows)
            if css == "gray":
                jpg = eng.encode(g)
                assert np.array_equal(jpg, O.encode_gray(g, 90, 1, rows * mcux)), css
                assert np.array_equal(eng.decode(jpg), O.decode_gray(jpg)), css
            else:
                jpg = eng.encode(img)
                assert np.array_equal(jpg, oracle.encode(img, css, 90, 1, rows * mcux)), css
                assert np.array_equal(eng.decode(jpg), oracle.decode(jpg)), css
        finally:
            eng.close()
