"""GPU: k_fdct's persistent CTAs against the CPU checker, byte for byte.

k_fdct launches min(tiles, 3 x SM count) CTAs; each codes one tile, then the tiles its tickets name. While a tile is
coded, the next tile's pixel rows are copied in: before stage C when the tile's token run stays below the staged-row
region (OFF_RAW / 4 tokens), else after stage C ("late" copies, over the region the run has just used).

- test_device_launch_walks_many_tiles: one launch (b2j_encode_device) of 1,600-2,800 tiles, every tile interior,
  bands of q100 noise rows between flat / smooth ones. The tile records prove that hundreds of late-path tiles are
  followed by another tile of the same CTA, i.e. that late copies are really issued. Checked: stream bytes, the
  kept coefficients (DUMP), the per-CTA histogram flush, and restart rows on the same launch shape.
- test_row_groups_walk_many_tiles: the host path uploads in MCU-row groups, one launch each; these images have two
  groups of more than 444 tiles, so the second launch (my0 > 0) also walks several tiles per CTA, late path included.
- test_edges_and_remainders: widths whose remainder tile is odd, or an edge tile, or both, and cut bottom rows
  (few tickets per launch; this covers the tile geometry, not the walk)."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOK_BYTES = 64 * 256 * 4 + 256
TILE_REC = np.dtype([("base", "<u4"), ("count", "<u4"), ("first_dc", "<i2", 3), ("last_dc", "<i2", 3),
                     ("pos_cb", "<u2"), ("pos_cr", "<u2")])
HV = {0: (1, 1), 1: (2, 1), 2: (1, 2), 3: (2, 2), 4: (4, 1), "gray": (1, 1)}


@pytest.fixture(scope="module")
def P():
    import nvjpeg_imagecompressor_b200 as P
    P.lib()
    return P


def resident_ctas():
    import torch
    return 3 * torch.cuda.get_device_properties(0).multi_processor_count


def late_threshold(css):
    """Token count above which a tile's run reaches the staged rows (enc_fdct.cu K1::OFF_RAW / 4)."""
    hs, vs = HV[css]
    nc = 1 if css == "gray" else 3
    bpm = 1 if nc == 1 else hs * vs + 2
    tm = (256 // bpm) & ~1
    return (TOK_BYTES - tm * 8 * hs * nc * 8 * vs) // 4


def banded_image(oracle, W, H, gray, seed, band_rows):
    """Rows in bands of `band_rows`: two bands of noise across the whole width (q100 runs reach the staged rows), then
    one band of flat / smooth / noise columns."""
    rng = np.random.default_rng(seed)
    img = oracle.synth(W, H, seed, 8)
    noise = rng.integers(0, 256, img.shape, dtype=np.uint8)
    band = (np.arange(H) // band_rows) % 3
    cols = (np.arange(W) // 200) % 3
    img[band < 2] = noise[band < 2]
    img[np.ix_(band == 2, cols == 0)] = 77
    m = np.ix_(band == 2, cols == 2)
    img[m] = noise[m]
    return np.ascontiguousarray(img[:, :, 1]) if gray else img


def want_of(oracle, img, css, q, opt, interval=0):
    if css == "gray":
        return oracle.encode_gray(img, q, opt, interval)
    return oracle.encode(img, css, q, opt, interval)


def device_encode(eng, d, W, H, ch):
    import torch
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    optr, _ = eng.encode_device(d.data_ptr(), W * ch, W, H)
    n = eng.encode_finish()
    out = np.empty(n, np.uint8)
    cudart = ctypes.CDLL("libcudart.so")
    assert cudart.cudaMemcpy(ctypes.c_void_p(out.ctypes.data), ctypes.c_void_p(optr), ctypes.c_size_t(n), 2) == 0
    return out


def late_followed(recs, thr, grid):
    """Late-path tiles that were not the last tile of their CTA (at most `grid` tiles are last)."""
    return int((recs["count"] > thr).sum()) - grid


# every tile interior (W, H multiples of the MCU; an odd remainder only where its rows stay 16-byte multiples)
MANY = [
    (672, 20000, 0),      # 1 tile of 84 MCUs per row, 2,500 tiles
    (1168, 11200, 1),     # 64 + 9 MCUs per row, 2,800 tiles
    (528, 20000, 2),      # 64 + 2, 2,500 tiles
    (672, 25600, 3),      # 42, 1,600 tiles
    (1344, 12800, 4),     # 42, 1,600 tiles
    (2064, 8000, "gray"),  # 256 + 2, 2,000 tiles
]


@pytest.mark.parametrize("W,H,css", MANY)
def test_device_launch_walks_many_tiles(P, oracle, W, H, css):
    import torch
    from nvjpeg_imagecompressor_b200 import _native as N
    gray = css == "gray"
    ch = 1 if gray else 3
    vs = HV[css][1]
    img = banded_image(oracle, W, H, gray, W + H, 24 * vs)
    d = torch.from_numpy(img).cuda()
    eng = P.Engine(W, H, 100, True, css, device=0)
    ntiles = None
    for rows in (0, 3):
        eng.set_restart_rows(rows)
        eng.set_debug(1 if rows == 0 else 0)
        got = device_encode(eng, d, W, H, ch)
        recs = eng.debug_read(N.DBG_TILE_RECS, np.uint8).view(TILE_REC)
        ntiles = recs.size
        grid = min(ntiles, resident_ctas())
        assert ntiles >= 3 * grid, (ntiles, grid)
        assert late_followed(recs, late_threshold(css), grid) >= 200, (css, rows)
        mcux = (W + 7) // 8 if gray else oracle.geometry(W, H, css).mcux
        want = want_of(oracle, img, css, 100, 1, rows * mcux)
        assert got.size == want.size and np.array_equal(got, want), (css, rows)
        if rows == 0 and not gray:
            coef = eng.debug_read(N.DBG_COEF, np.int16).reshape(-1, 64)
            ref = oracle.forward(img, css, 100)
            assert coef.shape == ref.shape and np.array_equal(coef, ref), css
            hist = eng.debug_read(N.DBG_HIST, np.uint32).reshape(4, 257)
            assert np.array_equal(hist, oracle.histogram(ref, oracle.geometry(W, H, css).bpm)), css
    eng.close()


# mcuy = 128: two upload groups of 64 MCU rows, each more than 444 tiles
@pytest.mark.parametrize("W,H,css", [(13440, 1024, 0), (30720, 1024, "gray")])
def test_row_groups_walk_many_tiles(P, oracle, W, H, css):
    from nvjpeg_imagecompressor_b200 import _native as N
    gray = css == "gray"
    img = banded_image(oracle, W, H, gray, 5, 24)
    eng = P.Engine(W, H, 100, True, css, device=0)
    mcux = (W + 7) // 8
    for rows in (0, 5):
        eng.set_restart_rows(rows)
        got = eng.encode(img)
        recs = eng.debug_read(N.DBG_TILE_RECS, np.uint8).view(TILE_REC).reshape(128, -1)
        grid = resident_ctas()
        for grp in (recs[:64], recs[64:]):
            assert grp.size >= 2 * grid
            assert late_followed(grp.ravel(), late_threshold(css), grid) >= 100, (css, rows)
        want = want_of(oracle, img, css, 100, 1, rows * mcux)
        assert got.size == want.size and np.array_equal(got, want), (css, rows)
    eng.close()


# (W, H, css): TM_MAX is 84 MCUs (4:4:4), 64 (4:2:2, 4:4:0), 42 (4:2:0, 4:1:1), 256 (gray)
EDGES = [
    (709, 2400, 0),     # mcux 89 = 84 + 5, the remainder tile is an edge tile
    (712, 2400, 0),     # mcux 89, W a multiple of 8: the odd remainder is interior, no bulk copies
    (1547, 2000, 1),    # mcux 97 = 64 + 33
    (568, 3997, 2),     # mcux 71 = 64 + 7, last MCU row cut
    (1488, 2560, 3),    # mcux 93 = 42 + 42 + 9
    (1433, 2400, 4),    # mcux 45 = 42 + 3
    (2343, 2000, "gray"),   # mcux 293 = 256 + 37, edge remainder
    (2344, 2000, "gray"),   # interior odd remainder: no bulk copies
]


@pytest.mark.parametrize("W,H,css", EDGES)
def test_edges_and_remainders(P, oracle, W, H, css):
    import torch
    gray = css == "gray"
    img = banded_image(oracle, W, H, gray, W + H, 40)
    d = torch.from_numpy(img).cuda()
    for q, opt in ((100, 1), (90, 0)):
        eng = P.Engine(W, H, q, bool(opt), css, device=0)
        want = want_of(oracle, img, css, q, opt)
        got = eng.encode(img)
        assert got.size == want.size and np.array_equal(got, want), (W, H, css, q, opt, "host")
        got = device_encode(eng, d, W, H, 1 if gray else 3)
        assert got.size == want.size and np.array_equal(got, want), (W, H, css, q, opt, "device")
        eng.close()
