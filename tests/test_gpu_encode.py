"""GPU parity: the CUDA encoder (through the C-ABI) against the CPU oracle, stage by stage and end to end."""
import hashlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def P():
    import nvjpeg_imagecompressor_b200 as P
    P.lib()
    return P


def _stage_check(P, O, eng, img, css, q, opt, tag):
    from nvjpeg_imagecompressor_b200 import _native as N
    H, W = img.shape[:2]
    eng.set_debug(1)
    jpg = eng.encode(img)
    g = O.geometry(W, H, css)
    coef = eng.debug_read(N.DBG_COEF, np.int16).reshape(-1, 64)
    ref = O.forward(img, css, q)
    assert coef.shape == ref.shape, tag
    bad = np.nonzero((coef != ref).any(axis=1))[0]
    assert bad.size == 0, f"{tag}: {bad.size} blocks differ, first {bad[:5]} got {coef[bad[0]][:8]} want {ref[bad[0]][:8]}"
    if opt:
        hist = eng.debug_read(N.DBG_HIST, np.uint32).reshape(4, 257)
        assert np.array_equal(hist, O.histogram(ref, g.bpm)), tag
        t = eng.tables()
        for ti in range(4):
            bits, vals, n = O.gen_optimal_table(hist[ti])
            assert list(t.bits[ti]) == bits.tolist(), (tag, ti)
            assert t.nsym[ti] == n and list(t.vals[ti])[:n] == vals[:n].tolist(), (tag, ti)
    want = O.encode(img, css, q, opt)
    assert jpg.size == want.size, f"{tag}: len {jpg.size} vs {want.size}"
    assert np.array_equal(jpg, want), f"{tag}: first diff at {np.nonzero(jpg != want)[0][:4]}"


def test_small_sizes_all_modes(P, oracle):
    rng = np.random.default_rng(5)
    sizes = [(64, 96), (48, 64), (50, 70), (17, 33), (135, 121), (8, 8), (1, 1), (257, 63), (33, 17), (100, 31)]
    for css in range(5):
        for q, opt in ((95, 1), (95, 0), (75, 1), (100, 0), (30, 1)):
            eng = P.Engine(300, 160, q, bool(opt), css)
            for (W, H) in sizes:
                img = oracle.synth(W, H, W * 31 + H, 8)
                _stage_check(P, oracle, eng, img, css, q, opt, f"synth {W}x{H} css{css} q{q} opt{opt}")
            img = rng.integers(0, 256, (77, 130, 3), dtype=np.uint8)
            _stage_check(P, oracle, eng, img, css, q, opt, f"random css{css} q{q} opt{opt}")
            eng.close()


def test_flat_and_extreme_images(P, oracle):
    """Degenerate statistics: constant image (2-bit blocks, many pack tiles per stuff chunk), saturated noise at
    q100 (longest codes, 0xFF-heavy), black/white checker."""
    rng = np.random.default_rng(9)
    imgs = {
        "flat": np.full((512, 768, 3), 128, np.uint8),
        "white": np.full((200, 200, 3), 255, np.uint8),
        "noise": rng.integers(0, 256, (256, 384, 3), dtype=np.uint8),
        "checker": (np.indices((128, 192)).sum(0) % 2 * 255).astype(np.uint8)[:, :, None].repeat(3, 2),
    }
    for css in (0, 1, 3):
        for q, opt in ((100, 1), (95, 0), (50, 1)):
            eng = P.Engine(768, 512, q, bool(opt), css)
            for name, img in imgs.items():
                _stage_check(P, oracle, eng, np.ascontiguousarray(img), css, q, opt, f"{name} css{css} q{q} opt{opt}")
            eng.close()


def test_pack_buffer_regimes(P, oracle):
    """k_pack's three paths: single pass (shares fit the warp buffers), overflow of a warp buffer (long codes, few
    tokens: redone in two passes) and the dense two-pass path (token count above the threshold)."""
    rng = np.random.default_rng(21)
    W, H = 1344, 48
    noise = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    soft = (noise.astype(np.int32) // 8 + oracle.synth(W, H, 5, 8).astype(np.int32) * 7 // 8).astype(np.uint8)
    for css in (0, 1):
        for q in (60, 80, 90, 97, 100):
            for opt in (1, 0):
                eng = P.Engine(W, H, q, bool(opt), css)
                for name, img in (("noise", noise), ("soft", soft)):
                    want = oracle.encode(img, css, q, opt)
                    # 2 = B2J_DEBUG_SMALL_PACK_BUFFERS: every warp buffer overflows -> recovery path
                    for dbg in (0, 2):
                        eng.set_debug(dbg)
                        jpg = eng.encode(img)
                        assert jpg.size == want.size and np.array_equal(jpg, want), f"{name} css{css} q{q} opt{opt} dbg{dbg}"
                eng.close()


def test_tiny_tiles(P, oracle):
    """Flat and narrow images: tiles of one MCU whose codes are 1-2 bits each (a tile shorter than a byte), and
    single-tile images."""
    rng = np.random.default_rng(5)
    for css in range(5):
        for W, H in ((8, 8), (8, 200), (16, 64), (24, 40), (40, 16), (2000, 8)):
            for kind in ("flat", "noise"):
                img = np.full((H, W, 3), 131, np.uint8) if kind == "flat" else rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
                for q, opt in ((95, 1), (50, 0)):
                    eng = P.Engine(W, H, q, bool(opt), css)
                    jpg = eng.encode(img)
                    want = oracle.encode(img, css, q, opt)
                    assert jpg.size == want.size and np.array_equal(jpg, want), (css, W, H, kind, q, opt)
                    eng.close()


def test_golden_cases(P, golden, oracle):
    """End to end against digests written by libjpeg-turbo itself (tests/golden/make_golden.py)."""
    engines = {}
    for c in golden["cases"]:
        key = (c["css"], c["quality"], c["optimize"])
        if key not in engines:
            engines[key] = P.Engine(1920, 1088, c["quality"], bool(c["optimize"]), c["css"])
        img = oracle.synth(c["W"], c["H"], c["seed"], c["amp"])
        jpg = engines[key].encode(img)
        assert jpg.size == c["jpeg_len"] and sha(jpg) == c["jpeg_sha256"], c
    for e in engines.values():
        e.close()


def test_row_pitch_and_unaligned_input(P, oracle):
    """cv::Mat step larger than width*3, and a width whose rows are not 16-byte multiples."""
    img = oracle.synth(203, 99, 4, 8)
    padded = np.zeros((99, 700), np.uint8)
    padded[:, : 203 * 3] = img.reshape(99, -1)
    view = padded[:, : 203 * 3].reshape(99, 203, 3)
    eng = P.Engine(256, 128, 90, True, "420")
    out = np.empty(1 << 20, np.uint8)
    n = eng.encode_ptr(view.ctypes.data, 700, 203, 99, out.ctypes.data, out.size)
    assert np.array_equal(out[:n], oracle.encode(img, 3, 90, 1))
    eng.close()


def test_context_reuse_and_errors(P, oracle):
    eng = P.Engine(128, 128, 95, True, "422")
    a = oracle.synth(128, 128, 1, 8)
    b = oracle.synth(96, 40, 2, 8)
    for img in (a, b, a):
        assert np.array_equal(eng.encode(img), oracle.encode(img, 1, 95, 1))
    with pytest.raises(P.B2JError) as ei:
        eng.encode(oracle.synth(512, 512, 1, 8))  # larger than the context
    assert ei.value.rc == -7
    small = np.empty(100, np.uint8)
    with pytest.raises(P.B2JError) as ei:
        eng.encode(a, out=small)
    assert ei.value.rc == -4
    assert eng.launch_count() > 0
    eng.close()


def test_slab_8320x2000_golden(P, golden, oracle):
    """First 2000 rows of the headline image: bytes == cv2.imencode (digests committed)."""
    img = oracle.synth(8320, 2000, 0, 8)
    for c in golden["slab"]:
        eng = P.Engine(8320, 2000, c["quality"], bool(c["optimize"]), c["css"])
        jpg = eng.encode(img)
        assert jpg.size == c["jpeg_len"], c
        assert sha(jpg) == c["jpeg_sha256"], c
        eng.close()


def test_device_resident_encode_matches_host_encode(P, oracle):
    import torch
    img = oracle.synth(640, 360, 3, 8)
    eng = P.Engine(640, 360, 95, True, "422")
    want = eng.encode(img)
    d = torch.from_numpy(img).cuda()
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    optr, lptr = eng.encode_device(d.data_ptr(), 640 * 3, 640, 360)
    n = eng.encode_finish()
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    import ctypes
    cudart = ctypes.CDLL("libcudart.so")
    assert cudart.cudaMemcpy(ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(optr), ctypes.c_size_t(n), 3) == 0
    assert np.array_equal(out.cpu().numpy(), want)
    eng.close()


def test_headline_full_image_digest(P, golden, oracle):
    """BASELINE.json config 2 at full size: 8320x40000 q95 4:2:2 optimized Huffman, JPEG SHA-256 from SURVEY.md App. B
    (cv2.imencode on the same synthetic image)."""
    h = golden["headline"]
    W, H = h["image"]["W"], h["image"]["H"]
    img = np.empty((H, W, 3), np.uint8)
    for y0 in range(0, H, 2000):
        img[y0:y0 + 2000] = oracle.synth(W, H, 0, 8, y0=y0, rows=2000)
    assert sha(img) == h["image"]["raw_sha256"]
    for e in h["encodes"][:2]:
        eng = P.Engine(W, H, e["quality"], bool(e["optimize"]), e["css"])
        jpg = eng.encode(img)
        assert jpg.size == e["jpeg_len"], e
        assert sha(jpg)[:32] == e["jpeg_sha256_128"], e
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("W,H,css,q,opt,rows", [(256, 320, 1, 95, 1, 1), (200, 333, 3, 90, 1, 2), (129, 200, 0, 75, 0, 1),
                                              (96, 250, 2, 95, 1, 3), (160, 64, 4, 100, 1, 1), (8, 40, 0, 95, 1, 1),
                                              (1040, 600, 1, 95, 1, 5)])
def test_restart_rows(P, oracle, W, H, css, q, opt, rows):
    """SURVEY.md 8f N2, encoder half: RSTn every `rows` MCU rows == libjpeg-turbo with restart_interval = rows * mcux."""
    img = oracle.synth(W, H, 21, 8)
    g = oracle.geometry(W, H, css)
    want = oracle.encode(img, css, q, opt, rows * g.mcux)
    eng = P.Engine(W, H, q, bool(opt), css)
    eng.set_restart_rows(rows)
    got = eng.encode(img)
    assert got.size == want.size and np.array_equal(got, want)
    eng.set_restart_rows(0)
    assert np.array_equal(eng.encode(img), oracle.encode(img, css, q, opt))
    eng.close()


def test_restart_rows_golden_digests(P, oracle, golden_rst):
    """Row-aligned intervals of the committed cv2 IMWRITE_JPEG_RST_INTERVAL digests (all five subsamplings)."""
    n = 0
    for c in golden_rst["cases"]:
        g = oracle.geometry(c["W"], c["H"], c["css"])
        ri = c["restart_interval"]
        if ri % g.mcux or ri // g.mcux == 0 or ri > 65535:
            continue
        img = oracle.synth(c["W"], c["H"], c["seed"], c["amp"])
        eng = P.Engine(c["W"], c["H"], c["quality"], bool(c["optimize"]), c["css"])
        eng.set_restart_rows(ri // g.mcux)
        jpg = eng.encode(img)
        assert jpg.size == c["jpeg_len"] and sha(jpg)[:32] == c["jpeg_sha256_128"], c
        eng.close()
        n += 1
    assert n >= 40
