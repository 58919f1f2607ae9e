"""GPU: progressive (SOF2) files with any scan script (tests/prog_streams.py catalogue: spectral selection only, DC per
component or over two components, successive approximation down from Al = 3 and Al = 10, refinement bands across bit
31/32 of the history mask, one scan per coefficient, EOB runs of 0x7FFF, long-code / skewed tables, DHT in rotated
slots, restart intervals in interleaved and non-interleaved scans of ragged frames, 640x360 and ~2 MP files) decode to
exactly cv2's pixels on every decode path, colour, gray and reduced. Incomplete files: those libjpeg would block-smooth
are refused on every decode path (b2j_peek still reports their size), the others, including files cut inside a scan,
decode to cv2's pixels."""
import cv2
import numpy as np
import pytest

import prog_streams as PS

pytestmark = pytest.mark.gpu
REDUCED = {2: (cv2.IMREAD_REDUCED_COLOR_2, cv2.IMREAD_REDUCED_GRAYSCALE_2),
           4: (cv2.IMREAD_REDUCED_COLOR_4, cv2.IMREAD_REDUCED_GRAYSCALE_4),
           8: (cv2.IMREAD_REDUCED_COLOR_8, cv2.IMREAD_REDUCED_GRAYSCALE_8)}


@pytest.fixture(scope="module")
def P():
    import nvjpeg_imagecompressor_b200 as P
    P.lib()
    return P


@pytest.fixture(scope="module")
def engines(P, oracle):
    # a context decodes frames of up to its own block count (4:4:4 blocks on a gray context): sized for the largest
    # catalogue frame
    W, H = max((P.Engine.peek(jpg)[:2] for _, jpg, _ in PS.catalogue(oracle)), key=lambda s: s[0] * s[1])
    col = P.Engine(W, H, 95, True, "444", device=0)
    gray = P.Engine(W, H, 95, True, "gray", device=0)
    yield col, gray
    col.set_decode_scale(1)
    gray.set_decode_scale(1)
    col.close()
    gray.close()


def dec(jpg, flag):
    out = cv2.imdecode(np.asarray(jpg, np.uint8), flag)
    assert out is not None
    return out


def device_decode(eng, jpg, shape, ch):
    import torch
    H, W = shape[:2]
    out = torch.zeros((H, W * ch + 5), dtype=torch.uint8, device="cuda")   # pitch != width
    assert eng.decode_device(jpg, out.data_ptr(), W * ch + 5) == (W, H)
    eng.decode_finish()
    return out[:, :W * ch].cpu().numpy().reshape(shape)


def first_bad_scan(eng, jpg, flag):
    """The first scan after which the decode differs from cv2 (the file cut there, with EOI), for a failure message"""
    segs = PS.scan_segments(jpg)
    for k in range(1, len(segs) + 1):
        part = PS.cut(jpg, segs[k - 1][1])
        try:
            got = eng.decode(part)
        except Exception:
            continue   # refused: libjpeg would smooth it
        if not np.array_equal(got, dec(part, flag)):
            return k
    return None


def test_catalogue_decodes_like_cv2(engines, oracle):
    col, gray = engines
    n = 0
    for tag, jpg, ncomp in PS.catalogue(oracle):
        for d in (1, 2, 4, 8):
            col.set_decode_scale(d)
            gray.set_decode_scale(d)
            fc, fg = (cv2.IMREAD_COLOR, cv2.IMREAD_GRAYSCALE) if d == 1 else REDUCED[d]
            want_g = dec(jpg, fg)
            got_g = gray.decode(jpg)
            if not np.array_equal(got_g, want_g):
                pytest.fail(f"{tag} scale {d} gray decode differs from scan {first_bad_scan(gray, jpg, fg)}")
            assert np.array_equal(device_decode(gray, jpg, want_g.shape, 1), want_g), (tag, d, "gray decode_device")
            if ncomp == 1:
                continue
            want = dec(jpg, fc)
            got = col.decode(jpg)
            if not np.array_equal(got, want):
                pytest.fail(f"{tag} scale {d} decode differs from scan {first_bad_scan(col, jpg, fc)}")
            assert np.array_equal(device_decode(col, jpg, want.shape, 3), want), (tag, d, "decode_device")
        n += 1
    col.set_decode_scale(1)
    gray.set_decode_scale(1)
    assert n >= 50


def test_incomplete_files(P, engines, oracle):
    """refused (B2J_EFORMAT) exactly where libjpeg would smooth; otherwise cv2's pixels, on colour and gray contexts"""
    import torch
    col, gray = engines
    n_refused = n_equal = 0
    for tag, jpg, ncomp, received in PS.incomplete(oracle):
        b = bytes(jpg)
        ref = jpg if b.endswith(b"\xff\xd9") else np.frombuffer(b + b"\xff\xd9", np.uint8)   # cv2 refuses a missing EOI
        assert P.Engine.peek(jpg)[:2] == dec(ref, cv2.IMREAD_GRAYSCALE).shape[::-1], tag
        for eng, is_gray in ((col, False), (gray, True)):
            if ncomp == 1 and not is_gray:
                continue
            flag, ch = (cv2.IMREAD_GRAYSCALE, 1) if is_gray else (cv2.IMREAD_COLOR, 3)
            if PS.smoothed(received, ncomp, is_gray):
                with pytest.raises(P.B2JError) as ex:
                    eng.decode(jpg)
                assert ex.value.rc == -5 and "smooth" in str(ex.value), (tag, is_gray)
                out = torch.zeros((8, 8 * ch), dtype=torch.uint8, device="cuda")
                with pytest.raises(P.B2JError) as ex:
                    eng.decode_device(jpg, out.data_ptr(), 8 * ch)
                    eng.decode_finish()
                assert ex.value.rc == -5, (tag, is_gray)
                n_refused += 1
                continue
            want = dec(ref, flag)
            assert np.array_equal(eng.decode(jpg), want), (tag, is_gray, "decode")
            assert np.array_equal(device_decode(eng, jpg, want.shape, ch), want), (tag, is_gray, "decode_device")
            n_equal += 1
    assert n_refused >= 100 and n_equal >= 60


def test_refinement_ah_al_mismatch_refused(P, engines, oracle):
    """a refinement scan must refine by exactly one bit (Al = Ah - 1), as libjpeg requires"""
    col, _ = engines
    script = [((0, 1, 2), 0, 0, 0, 2), ((0, 1, 2), 0, 0, 2, 0)] + [((c,), 1, 63, 0, 0) for c in (0, 1, 2)]
    *_, jpg = PS.entry(oracle, "simple", 40, 24, 0, script=script)
    assert cv2.imdecode(jpg, cv2.IMREAD_COLOR) is None
    with pytest.raises(P.B2JError) as ex:
        col.decode(jpg)
    assert ex.value.rc == -5
