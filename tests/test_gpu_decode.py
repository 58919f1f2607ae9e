"""GPU parity: the CUDA decoder (through the C-ABI) against the CPU oracle / libjpeg-turbo digests, plus the
difference-map, PSNR and secondary-compression entry points."""
import hashlib
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def P():
    import nvjpeg_imagecompressor_b200 as P
    P.lib()
    return P


def _check(P, O, eng, jpg, tag):
    from nvjpeg_imagecompressor_b200 import _native as N
    out = eng.decode(jpg)
    want = O.decode(jpg)
    if not np.array_equal(out, want):
        coef = eng.debug_read(N.DBG_DEC_COEF, np.int16).reshape(-1, 64)
        ref, info = O.decode_coefs(jpg)
        coef = coef[: ref.shape[0]]
        bad = np.nonzero((coef != ref).any(axis=1))[0]
        d = np.abs(out.astype(int) - want.astype(int))
        raise AssertionError(f"{tag}: pixels differ (max {d.max()}, {np.count_nonzero(d)} values); coefficient blocks differing: "
                             f"{bad.size} first {bad[:6]}")


def test_golden_files(P, oracle, golden):
    eng = P.Engine(256, 256, 95, True, "422")
    for f in golden["files"]:
        jpg = np.fromfile(os.path.join(HERE, "golden", f["file"]), np.uint8)
        assert P.Engine.peek(jpg) == (f["W"], f["H"], f["css"])
        out = eng.decode(jpg)
        assert sha(out) == f["decoded_sha256"], f
    eng.close()


def test_decode_schedules(P, oracle):
    """The three synchronisation schedules give the same pixels: the unchecked fixed schedule (default), its validated
    retry (forced by cutting the schedule to one launch) and the checked loop (long synchronisation distance: q100),
    through the synchronous call and through decode_device + decode_finish."""
    import torch
    W, H = 1600, 640   # several decoder chunks (256 subsequences of 1024 bits each)
    img = oracle.synth(W, H, 11, 8)
    eng = P.Engine(W, H, 95, True, "444")   # sized for the largest block count of the cases below
    for css, q in ((1, 95), (3, 85), (0, 100)):
        jpg = oracle.encode(img, css, q, 1)
        want = oracle.decode(jpg)
        for dbg in (0, 4):   # 4 = B2J_DEBUG_SHORT_DECODE_SCHEDULE
            eng.set_debug(dbg)
            assert np.array_equal(eng.decode(jpg), want), (css, q, dbg, "decode")
            out = torch.zeros((H, W, 3), dtype=torch.uint8, device="cuda")
            eng.decode_device(jpg, out.data_ptr(), W * 3)
            eng.decode_finish()
            assert np.array_equal(out.cpu().numpy(), want), (css, q, dbg, "decode_device")
    eng.close()


def test_small_sizes_all_modes(P, oracle):
    rng = np.random.default_rng(6)
    sizes = [(64, 96), (48, 64), (50, 70), (17, 33), (135, 121), (8, 8), (1, 1), (257, 63), (33, 17), (2, 2), (3, 5), (5, 3), (4, 4)]
    eng = P.Engine(320, 160, 95, True, "444")
    for css in range(5):
        for q, opt in ((95, 1), (95, 0), (75, 1), (100, 0)):
            for (W, H) in sizes:
                img = oracle.synth(W, H, W * 31 + H, 8)
                _check(P, oracle, eng, oracle.encode(img, css, q, opt), f"synth {W}x{H} css{css} q{q} opt{opt}")
            img = rng.integers(0, 256, (77, 130, 3), dtype=np.uint8)
            _check(P, oracle, eng, oracle.encode(img, css, q, opt), f"random css{css} q{q} opt{opt}")
    eng.close()


def test_golden_case_digests(P, oracle, golden):
    """decoded pixels == cv2.imdecode digests for streams made by the oracle encoder (== cv2.imencode bytes)."""
    eng = P.Engine(1920, 1088, 95, True, "444")
    for c in golden["cases"]:
        if c["quality"] != 95:
            continue
        img = oracle.synth(c["W"], c["H"], c["seed"], c["amp"])
        jpg = oracle.encode(img, c["css"], c["quality"], c["optimize"])
        assert sha(jpg) == c["jpeg_sha256"]
        assert sha(eng.decode(jpg)) == c["decoded_sha256"], c
    eng.close()


def test_degenerate_streams(P, oracle):
    """Flat image (2-4 bit blocks: hundreds of blocks per 1024-bit subsequence), saturated noise (long codes,
    blocks longer than a subsequence), checkerboard."""
    rng = np.random.default_rng(10)
    imgs = {"flat": np.full((512, 768, 3), 128, np.uint8), "noise": rng.integers(0, 256, (256, 384, 3), dtype=np.uint8),
            "checker": (np.indices((128, 192)).sum(0) % 2 * 255).astype(np.uint8)[:, :, None].repeat(3, 2)}
    eng = P.Engine(768, 512, 95, True, "444")
    for css in (0, 1, 3, 4):
        for q, opt in ((100, 1), (95, 0), (40, 1)):
            for name, img in imgs.items():
                _check(P, oracle, eng, oracle.encode(np.ascontiguousarray(img), css, q, opt), f"{name} css{css} q{q} opt{opt}")
    eng.close()


def test_roundtrip_own_encoder_and_metrics(P, oracle):
    img = oracle.synth(640, 360, 3, 8)
    eng = P.Engine(640, 360, 95, True, "422")
    jpg = eng.encode(img)
    rec = eng.decode(jpg)
    assert np.array_equal(rec, oracle.decode(jpg))
    for mode in (0, 1):
        assert np.array_equal(eng.diff(img, rec, mode), oracle.diff(img, rec, mode))
    ps, ssd = eng.psnr(img, rec)
    assert ssd == oracle.ssd(img, rec)
    assert abs(ps - oracle.psnr(img, rec)) < 1e-12
    # odd lengths / unaligned views through the scalar tail
    a = img.reshape(-1)[3:100003]
    b = rec.reshape(-1)[5:100005]
    assert np.array_equal(eng.diff(a, b, 1), oracle.diff(a, b, 1))
    assert eng.psnr(a, b)[1] == oracle.ssd(a, b)
    eng.close()


def test_secondary_compression(P, oracle):
    """encode -> reconstruct -> difference map -> encode(diff) + PSNR (SURVEY.md 8a-12), each step == oracle."""
    img = oracle.synth(333, 222, 8, 8)
    for css, mode in ((1, 1), (3, 0)):
        eng = P.Engine(333, 222, 90, True, css)
        j1, j2, recon, ps = eng.secondary(img, diff_mode=mode)
        w1 = oracle.encode(img, css, 90, 1)
        assert np.array_equal(j1, w1)
        wrec = oracle.decode(w1)
        assert np.array_equal(recon, wrec)
        wdiff = oracle.diff(img, wrec, mode)
        assert np.array_equal(j2, oracle.encode(wdiff, css, 90, 1))
        assert abs(ps - oracle.psnr(img, wrec)) < 1e-12
        eng.close()


def test_reconstruct_from_coefficients_and_device_secondary(P, oracle):
    """b2j_reconstruct_device (de-quantise + IDCT + upsample of the encoder's own coefficients, no entropy decode) gives
    exactly the decoder's pixels for every subsampling and ragged sizes; b2j_secondary_device / _finish == the checker."""
    import torch
    for (W, H) in ((333, 222), (64, 48), (17, 33), (640, 360)):
        img = oracle.synth(W, H, 3, 8)
        d_img = torch.from_numpy(img).cuda()
        for css in range(5):
            eng = P.Engine(W, H, 92, True, css)
            eng.set_debug(1)
            jpg = eng.encode(img)
            rec = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda")
            eng.reconstruct_device(rec.data_ptr(), W * 3)
            torch.cuda.synchronize()
            eng.set_debug(0)
            want = oracle.decode(jpg)
            assert np.array_equal(rec.cpu().numpy(), want), (W, H, css)
            for mode in (0, 1):
                eng.secondary_device(d_img.data_ptr(), W * 3, W, H, mode)
                n1, n2, ps, ssd = eng.secondary_finish()
                assert n1 == jpg.size and ssd == oracle.ssd(img, want), (W, H, css, mode)
                assert abs(ps - oracle.psnr(img, want)) < 1e-12
                assert n2 == oracle.encode(oracle.diff(img, want, mode), css, 92, 1).size
            eng.close()


def test_runner_facade_demo_sequence(P, oracle, tmp_path):
    """The reference demo's call order (src/ImageCompressor/main.cpp:24-78) through the Python facade."""
    r = P.NvjpegCompressRunner(640, 360, 95, True, verbose=False)
    r.buildCompressEnv()
    img1, img2 = oracle.synth(640, 360, 1, 8), oracle.synth(640, 360, 2, 8)
    b1, s1 = r.compress(img1)
    b2, s2 = r.compress(img2)
    assert s1 == 1 and s2 == 1
    r.deleteCompressEnv()
    r.buildDecodeEnv()
    p1, p2 = str(tmp_path / "a.jpeg"), str(tmp_path / "b.jpeg")
    r.save(p1, b1)
    r.save(p2, b2)
    d1, t1 = r.decode(p1)
    d2, t2 = r.decode(p2)
    assert t1 == 1 and t2 == 1
    assert np.array_equal(d1, oracle.decode(oracle.encode(img1, 1, 95, 1)))
    assert np.array_equal(d2, oracle.decode(oracle.encode(img2, 1, 95, 1)))
    bad, st = r.decode(str(tmp_path / "missing.jpeg"))
    assert st == 0 and bad.size == 0
    r.deleteDecodeEnv()


def test_rejects_unsupported(P, oracle):
    cv2 = pytest.importorskip("cv2")
    img = oracle.synth(64, 64, 1, 8)
    ok, gray = cv2.imencode(".jpg", img[:, :, 0])   # one component: outside the three-component interface of the reference
    eng = P.Engine(64, 64)
    with pytest.raises(P.B2JError) as ei:
        eng.decode(gray.ravel())
    assert ei.value.rc == -5
    ok, prog = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])   # progressive files are decoded (row N4)
    assert np.array_equal(eng.decode(prog.ravel()), cv2.imdecode(prog, cv2.IMREAD_COLOR))
    with pytest.raises(P.B2JError):
        eng.decode(np.zeros(1000, np.uint8))
    eng.close()


def test_slab_8320x2000(P, oracle, golden):
    img = oracle.synth(8320, 2000, 0, 8)
    eng = P.Engine(8320, 2000, 95, True, "444")
    for c in golden["slab"]:
        jpg = oracle.encode(img, c["css"], c["quality"], c["optimize"])
        assert sha(jpg) == c["jpeg_sha256"]
        assert sha(eng.decode(jpg)) == c["decoded_sha256"], c
    eng.close()


def test_headline_full_image_decode_digest(P, golden, oracle):
    """8320x40000: encode on the GPU (bytes == cv2.imencode, checked in test_gpu_encode), decode on the GPU, pixels ==
    cv2.imdecode (decoded-BGR SHA-256 from SURVEY.md App. B) and PSNR == the survey's figure."""
    h = golden["headline"]
    W, H = h["image"]["W"], h["image"]["H"]
    img = np.empty((H, W, 3), np.uint8)
    for y0 in range(0, H, 2000):
        img[y0:y0 + 2000] = oracle.synth(W, H, 0, 8, y0=y0, rows=2000)
    for e in h["encodes"][:2]:
        eng = P.Engine(W, H, e["quality"], bool(e["optimize"]), e["css"])
        jpg = eng.encode(img)
        assert sha(jpg)[:32] == e["jpeg_sha256_128"]
        rec = eng.decode(jpg)
        assert sha(rec)[:32] == e["decoded_sha256_128"], e
        eng.close()


def _nvjpeg_golden():
    """What the reference's nvJPEG path wrote (tests/golden/make_golden_nvjpeg.py, which runs the nvJPEG harness
    baseline/ref_nvjpeg.cu = the reference's call sequence): small streams with libjpeg-turbo's pixel digests, and
    nvJPEG's size and PSNR at 4096x3072."""
    import json
    with open(os.path.join(HERE, "golden", "golden_nvjpeg.json")) as f:
        return json.load(f)


def _decode_nvjpeg_files(P, progressive):
    files = [c for c in _nvjpeg_golden()["files"] if c["progressive"] == progressive]
    assert len(files) == 3
    eng = P.Engine(max(c["W"] for c in files), max(c["H"] for c in files), 95, True, "444")
    for c in files:
        jpg = np.fromfile(os.path.join(HERE, "golden", c["file"]), np.uint8)
        assert sha(jpg) == c["jpeg_sha256"], c
        if progressive:
            assert 0xC2 in jpg[:1024].tolist()   # a progressive frame header
        got = eng.decode(jpg)
        assert got.shape == (c["H"], c["W"], 3) and sha(got) == c["decoded_sha256"], c
    eng.close()


def test_decode_nvjpeg_streams(P):
    """BASELINE.json config 5: JPEGs written by the reference's nvJPEG path (baseline sequential, optimised Huffman, no
    restart markers; 4:2:2, 4:4:4 and 4:2:0) decode to exactly the pixels libjpeg-turbo produces from the same bytes."""
    _decode_nvjpeg_files(P, 0)


def test_against_reference_nvjpeg_output(P):
    """North-star target 3: this encoder's output vs the reference's nvJPEG path on the same image and settings
    (4:2:2, q95, optimised Huffman): file size within 2 %, PSNR of the reconstruction not below nvJPEG's by more than
    0.05 dB. (Measured: +1.5 % bytes and +0.39 dB -- the bit-exact libjpeg-turbo arithmetic reconstructs better than
    nvJPEG's, so "within 0.05 dB" can only hold one-sided while the stream is pinned to libjpeg-turbo.)"""
    ref = _nvjpeg_golden()["size_psnr"]
    from nvjpeg_imagecompressor_b200.synth import synth
    W, H = ref["W"], ref["H"]
    img = synth(W, H, ref["seed"], ref["amp"]).cpu().numpy()
    eng = P.Engine(W, H, ref["quality"], bool(ref["optimize"]), ref["css"])
    mine = eng.encode(img)
    psnr_mine = eng.psnr(img, eng.decode(mine))[0]
    eng.close()
    assert abs(mine.size - ref["jpeg_len"]) <= 0.02 * ref["jpeg_len"], (mine.size, ref["jpeg_len"])
    assert psnr_mine >= ref["psnr"] - 0.05, (psnr_mine, ref["psnr"])
    print(f"size {mine.size} vs nvJPEG {ref['jpeg_len']} ({100.0 * (mine.size - ref['jpeg_len']) / ref['jpeg_len']:+.2f} %), "
          f"PSNR {psnr_mine:.3f} vs {ref['psnr']:.3f} dB")


def test_restart_interval_streams(P, oracle, golden_rst):
    """SURVEY.md 8f N2, decoder half: streams with DRI / RSTn markers (every interval is a known synchronisation point;
    DC predictors restart) decode to cv2.imdecode's pixels -- the 200 committed cv2 IMWRITE_JPEG_RST_INTERVAL digests
    (1 MCU, ragged, one and two MCU rows, longer than the image; five subsamplings), regenerated through the checker
    whose byte-identity with cv2 tests/test_oracle_golden.py establishes."""
    eng = P.Engine(640, 360, 95, True, "444")
    n = 0
    for c in golden_rst["cases"]:
        img = oracle.synth(c["W"], c["H"], c["seed"], c["amp"])
        jpg = oracle.encode(img, c["css"], c["quality"], c["optimize"], c["restart_interval"])
        assert jpg.size == c["jpeg_len"] and sha(jpg)[:32] == c["jpeg_sha256_128"], c
        out = eng.decode(jpg)
        assert sha(out)[:32] == c["decoded_sha256_128"], c
        n += 1
    assert n == 200
    eng.close()


def test_restart_round_trip_large(P, oracle):
    """Own restart streams (b2j_set_restart_rows) decode to the same pixels as the stream without markers, over
    several decoder chunks and the three synchronisation schedules; q100 included (long synchronisation distances)."""
    W, H = 1600, 640
    img = oracle.synth(W, H, 5, 8)
    for css, q, rows in ((1, 95, 1), (3, 100, 2), (0, 100, 1)):
        eng = P.Engine(W, H, q, True, css)
        plain = eng.encode(img)
        want = eng.decode(plain)
        eng.set_restart_rows(rows)
        jpg = eng.encode(img)
        assert jpg.size != plain.size
        for dbg in (0, 4):
            eng.set_debug(dbg)
            assert np.array_equal(eng.decode(jpg), want), (css, q, rows, dbg)
        eng.set_debug(0)
        eng.close()


def test_progressive_streams(P, oracle):
    """SURVEY.md 8f N4: progressive (SOF2) files -- the format the reference as shipped writes (ImageCompressorImpl.cu:28)
    -- decode to libjpeg-turbo's pixels: the committed cv2-written files (with and without restart markers) and
    jpeg_simple_progression streams for every subsampling / ragged sizes (the checker's progressive encoder, byte-identical
    to cv2.imencode(IMWRITE_JPEG_PROGRESSIVE): tests/test_oracle_golden.py)."""
    import json
    with open(os.path.join(HERE, "golden", "golden_prog.json")) as f:
        files = json.load(f)["files"]
    eng = P.Engine(640, 360, 95, True, "444")
    for c in files:
        jpg = np.fromfile(os.path.join(HERE, "golden", c["file"]), np.uint8)
        assert P.Engine.peek(jpg) == (c["W"], c["H"], c["css"])
        out = eng.decode(jpg)
        assert out.shape == (c["H"], c["W"], 3) and sha(out) == c["decoded_sha256"], c
    rng = np.random.default_rng(4)
    for (W, H) in ((50, 70), (8, 8), (1, 1), (135, 121), (257, 63), (640, 360)):
        for img in (oracle.synth(W, H, 6, 8), rng.integers(0, 256, (H, W, 3), dtype=np.uint8)):
            for css in range(5):
                for q in (50, 95, 100):
                    jpg = oracle.encode_progressive(img, css, q)
                    assert np.array_equal(eng.decode(jpg), oracle.decode(jpg)), (W, H, css, q)
    eng.close()


def test_decode_reference_progressive_nvjpeg_streams(P):
    """The unmodified reference encodes PROGRESSIVE 4:4:4 (ImageCompressorImpl.cu:28,31): the streams its nvJPEG call
    sequence writes with that setting (4:4:4, 4:2:2 and 4:2:0) decode to cv2.imdecode's pixels."""
    _decode_nvjpeg_files(P, 1)
