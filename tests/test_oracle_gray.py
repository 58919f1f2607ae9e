"""The grayscale CPU checker (tests/gray_oracle.py: encode_gray / decode_gray) against libjpeg-turbo: live cv2 where it is
importable, and the committed digests of tests/golden/golden_gray.json (tests/golden/make_golden_gray.py) always.
Also b2j_peek on one-component files, which needs no GPU."""
import hashlib
import json
import os

import numpy as np
import pytest

import gray_oracle as G

HERE = os.path.dirname(os.path.abspath(__file__))
SIZES = ((1, 1), (2, 2), (8, 8), (17, 33), (33, 17), (135, 121), (257, 63), (640, 360))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="session")
def golden_gray():
    with open(os.path.join(HERE, "golden", "golden_gray.json")) as f:
        return json.load(f)


def gray_img(oracle, W, H, seed):
    return np.ascontiguousarray(oracle.synth(W, H, seed, 8)[..., 1])


def colour_stream(oracle, c):
    img = oracle.synth(c["W"], c["H"], c["seed"], 8)
    if c["kind"] == "prog":
        return oracle.encode_progressive(img, c["css"], c["quality"])
    return oracle.encode(img, c["css"], c["quality"], c["optimize"], c["restart_interval"])


def test_encode_gray_matches_golden(oracle, golden_gray):
    for c in golden_gray["encode"]:
        img = gray_img(oracle, c["W"], c["H"], c["seed"])
        jpg = G.encode_gray(img, c["quality"], c["optimize"], c["restart_interval"])
        assert jpg.size == c["jpeg_len"] and sha(jpg)[:32] == c["jpeg_sha256_128"], c
        assert sha(G.decode_gray(jpg))[:32] == c["decoded_sha256_128"], c


def test_gray_stream_layout(oracle):
    img = gray_img(oracle, 40, 24, 3)
    jpg = G.encode_gray(img, 90, 1, 5).tobytes()
    markers = []
    p = 2
    while jpg[p + 1] != 0xDA:
        markers.append(jpg[p + 1])
        p += 2 + ((jpg[p + 2] << 8) | jpg[p + 3])
    assert markers == [0xE0, 0xDB, 0xC0, 0xC4, 0xC4, 0xDD]
    sof = jpg.index(b"\xff\xc0")
    assert jpg[sof + 2:sof + 4] == b"\x00\x0b" and jpg[sof + 4:sof + 13] == bytes([8, 0, 24, 0, 40, 1, 1, 0x11, 0])
    assert jpg[p + 2:p + 10] == bytes([0, 8, 1, 1, 0, 0, 0x3F, 0])


def test_decode_gray_of_colour_matches_golden(oracle, golden_gray):
    for c in golden_gray["ydecode"]:
        jpg = colour_stream(oracle, c)
        assert sha(jpg)[:32] == c["jpeg_sha256_128"], c
        assert sha(G.decode_gray(jpg))[:32] == c["gray_sha256_128"], c


def test_decode_gray_files(oracle, golden_gray):
    for f in golden_gray["files"]:
        jpg = np.fromfile(os.path.join(HERE, "golden", f["file"]), np.uint8)
        assert sha(jpg) == f["jpeg_sha256"]
        dec = G.decode_gray(jpg)
        assert dec.shape == (f["H"], f["W"])
        assert sha(dec) == f["decoded_sha256"], f["file"]


def test_colour_functions_still_reject_gray(oracle, golden_gray):
    jpg = np.fromfile(os.path.join(HERE, "golden", golden_gray["files"][0]["file"]), np.uint8)
    with pytest.raises(RuntimeError):
        oracle.decode(jpg)
    with pytest.raises(ValueError):
        oracle.geometry(8, 8, G.CSS_GRAY)


def test_peek_gray_files(golden_gray):
    import nvjpeg_imagecompressor_b200 as P
    if not os.path.exists(P._native.LIB_PATH):
        pytest.skip("libb2jpeg.so not built")
    for f in golden_gray["files"]:
        jpg = np.fromfile(os.path.join(HERE, "golden", f["file"]), np.uint8)
        assert P.Engine.peek(jpg) == (f["W"], f["H"], 6)


# ---- live libjpeg-turbo ------------------------------------------------------------------------------------------
cv2 = pytest.importorskip("cv2")


def cv_gray(img, q, opt, rst=0, prog=0):
    p = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, opt]
    if rst:
        p += [cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    if prog:
        p += [cv2.IMWRITE_JPEG_PROGRESSIVE, 1]
    return cv2.imencode(".jpg", img, p)[1].ravel()


@pytest.mark.parametrize("W,H", SIZES)
def test_encode_gray_vs_cv2(oracle, W, H):
    img = gray_img(oracle, W, H, W * 7 + H)
    mcux = (W + 7) // 8
    for q in (40, 75, 95, 100):
        for opt in (0, 1):
            for rst in sorted({0, 1, 5, mcux, 2 * mcux}):
                ref = cv_gray(img, q, opt, rst)
                jpg = G.encode_gray(img, q, opt, rst)
                assert np.array_equal(jpg, ref), (W, H, q, opt, rst)
                assert np.array_equal(G.decode_gray(jpg), cv2.imdecode(ref, cv2.IMREAD_UNCHANGED)), (W, H, q, opt, rst)


@pytest.mark.parametrize("kind", ["flat", "saturated", "checker"])
def test_encode_gray_special_images_vs_cv2(oracle, kind):
    H, W = 45, 70
    rng = np.random.default_rng(5)
    if kind == "flat":
        img = np.full((H, W), 77, np.uint8)
    elif kind == "saturated":
        img = np.where(rng.random((H, W)) < 0.5, 0, 255).astype(np.uint8)
    else:
        img = ((np.indices((H, W)).sum(0) & 1) * 255).astype(np.uint8)
    for q, opt in ((100, 1), (95, 0), (40, 1)):
        assert np.array_equal(G.encode_gray(img, q, opt), cv_gray(img, q, opt)), (kind, q, opt)


def test_encode_gray_pitch(oracle):
    big = gray_img(oracle, 160, 50, 11)
    img = big[:, 3:140]   # pitch 160 != width 137
    assert np.array_equal(G.encode_gray(img, 90, 1, 3), cv_gray(np.ascontiguousarray(img), 90, 1, 3))


@pytest.mark.parametrize("css", range(5))
def test_decode_gray_of_colour_vs_cv2(oracle, css):
    img = oracle.synth(135, 121, 9, 8)
    mcux = oracle.geometry(135, 121, css).mcux
    for jpg in (oracle.encode(img, css, 90, 1), oracle.encode(img, css, 75, 0, mcux), oracle.encode(img, css, 95, 1, 7),
                oracle.encode_progressive(img, css, 85)):
        assert np.array_equal(G.decode_gray(jpg), cv2.imdecode(jpg, cv2.IMREAD_GRAYSCALE))


def test_decode_gray_progressive_and_patched_vs_cv2(oracle):
    img = gray_img(oracle, 135, 121, 4)
    for rst in (0, 4):
        jpg = cv_gray(img, 85, 1, rst, prog=1)
        assert np.array_equal(G.decode_gray(jpg), cv2.imdecode(jpg, cv2.IMREAD_UNCHANGED))
    for f in ("gray/gray_135x121_q90_sof22.jpg", "gray/gray_135x121_q90_prog.jpg", "gray/gray_135x121_q90_rst5.jpg"):
        jpg = np.fromfile(os.path.join(HERE, "golden", f), np.uint8)
        assert np.array_equal(G.decode_gray(jpg), cv2.imdecode(jpg, cv2.IMREAD_UNCHANGED)), f
