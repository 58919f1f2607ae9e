"""CPU: the reduced-size decode of the checker (oracle/) against libjpeg-turbo's DCT scaling --
live cv2 (IMREAD_REDUCED_COLOR_d / IMREAD_REDUCED_GRAYSCALE_d) when it is installed, and always the committed digests
of tests/golden/golden_scaled.json (tests/golden/make_golden_scaled.py)."""
import hashlib
import json
import os

import numpy as np
import pytest

import oracle as O
import prog_streams as PS

HERE = os.path.dirname(os.path.abspath(__file__))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def golden_scaled():
    with open(os.path.join(HERE, "golden", "golden_scaled.json")) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


def reduced_flag(cv2, d, gray):
    return getattr(cv2, "IMREAD_REDUCED_%s_%d" % ("GRAYSCALE" if gray else "COLOR", d))


def test_matrix_vs_golden(oracle, golden_scaled):
    """the matrix streams re-made by the checker's encoder (byte-identical to cv2's), decoded at 1/2, 1/4, 1/8"""
    for c in golden_scaled["cases"]:
        img = oracle.synth(c["W"], c["H"], c["seed"], c["amp"])
        jpg = oracle.encode(img, c["css"], c["quality"], c["optimize"], c["restart_interval"])
        assert sha(jpg)[:32] == c["jpeg_sha256_128"], c
        for d in O.SCALES:
            assert sha(O.decode_scaled(jpg, d))[:32] == c["c%d" % d], (c, d)
            assert sha(O.decode_scaled(jpg, d, gray=True))[:32] == c["g%d" % d], (c, d)


def test_golden_files_vs_golden(golden_scaled):
    """progressive, nvJPEG and one-component files in gray, and in colour those that have colour digests"""
    for f in golden_scaled["files"]:
        jpg = np.fromfile(os.path.join(HERE, "golden", f["file"]), np.uint8)
        assert sha(jpg) == f["jpeg_sha256"]
        for d in O.SCALES:
            want = O.decode_scaled(jpg, d, gray=True)
            assert want.shape == O.reduced_size(f["W"], f["H"], d)[::-1]
            assert sha(want)[:32] == f["g%d" % d], (f["file"], d)
            if "c%d" % d in f:
                assert sha(O.decode_scaled(jpg, d))[:32] == f["c%d" % d], (f["file"], d)


def test_live_cv2_matrix(cv2, oracle):
    rng = np.random.default_rng(7)
    SF = (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440,
          cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411)
    n = 0
    for (W, H) in ((1, 1), (5, 3), (2, 40), (40, 2), (9, 17), (33, 17), (16, 16), (64, 48), (67, 93), (121, 135), (250, 301)):
        noise = rng.integers(0, 256, (H, W, 3), np.uint8)
        for img in (noise, cv2.GaussianBlur(noise, (0, 0), 3)):
            for css in range(5):
                for q in (50, 90, 100):
                    for rst in ((0, 2) if q == 90 else (0,)):
                        jpg = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SF[css],
                                                         cv2.IMWRITE_JPEG_RST_INTERVAL, rst])[1].ravel()
                        for d in O.SCALES:
                            for gray in (False, True):
                                want = cv2.imdecode(jpg, reduced_flag(cv2, d, gray))
                                got = O.decode_scaled(jpg, d, gray)
                                assert got.shape == want.shape and np.array_equal(got, want), (W, H, css, q, rst, d, gray)
                                n += 1
    assert n == 11 * 2 * 5 * 4 * 3 * 2


def test_live_cv2_one_component_files(cv2, oracle):
    for (W, H) in ((1, 1), (13, 7), (135, 121)):
        img = np.ascontiguousarray(oracle.synth(W, H, W + H, 40)[..., 1])
        for q, opt, ri in ((90, 1, 0), (75, 0, 3)):
            jpg = O.encode_gray(img, q, opt, ri)
            for d in O.SCALES:
                want = cv2.imdecode(jpg, reduced_flag(cv2, d, True))
                assert np.array_equal(O.decode_scaled(jpg, d, gray=True), want), (W, H, q, ri, d)
        prog = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].ravel()
        for d in O.SCALES:
            assert np.array_equal(O.decode_scaled(prog, d, gray=True), cv2.imdecode(prog, reduced_flag(cv2, d, True)))


def test_live_cv2_progressive_catalogue(cv2, oracle):
    """progressive files with any scan script, in colour and gray at every reduced size"""
    n = 0
    for tag, jpg, ncomp in PS.catalogue(oracle, big=False):
        for d in O.SCALES:
            for gray in (False, True) if ncomp == 3 else (True,):
                want = cv2.imdecode(jpg, reduced_flag(cv2, d, gray))
                assert np.array_equal(O.decode_scaled(jpg, d, gray), want), (tag, d, gray)
                n += 1
    assert n >= 200


def test_scale_one_is_the_full_decode(oracle):
    img = oracle.synth(67, 93, 3, 8)
    for css in range(5):
        jpg = oracle.encode(img, css, 90, 1)
        assert np.array_equal(O.decode_scaled(jpg, 1), oracle.decode(jpg))
        assert np.array_equal(O.decode_scaled(jpg, 1, gray=True), O.decode_gray(jpg))


def test_rejections(oracle):
    jpg = oracle.encode(oracle.synth(16, 16, 1, 8), 0, 90, 1)
    for bad in (0, 3, 16, -1):
        with pytest.raises(RuntimeError):
            O.decode_scaled(jpg, bad)
    gray_file = O.encode_gray(np.zeros((8, 8), np.uint8), 90, 1)
    with pytest.raises(RuntimeError):
        O.decode_scaled(gray_file, 2)   # colour output of a one-component file
