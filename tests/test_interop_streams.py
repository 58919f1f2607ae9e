"""JPEG files from other writers (tests/jpeg_streams.py and Pillow) on the CPU: the writer's own check against live
cv2, the colour-space rule of live libjpeg, and the verdict of the product's header parser (csrc/dec_parse.cpp) on
every stream. tests/test_gpu_interop.py decodes the accepted ones on the GPU."""
import os
import shutil
import subprocess

import cv2
import numpy as np
import pytest

import jpeg_streams as J

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dec(jpg, flag=cv2.IMREAD_COLOR):
    return cv2.imdecode(np.asarray(jpg, np.uint8), flag)


@pytest.mark.parametrize("css", range(5))
@pytest.mark.parametrize("quality", (50, 95, 100))
def test_writer_matches_its_source(oracle, css, quality):
    """every layout the writer makes holds the source's coefficients and tables: cv2 decodes it to the source's pixels"""
    for size in (J.SIZES[css], (1, 1), (9, 17), (33, 5)):
        src, streams = J.writer_streams(oracle, css, quality, size)
        want = dec(src)
        assert want is not None
        for name, jpg in streams:
            got = dec(jpg)
            if name.startswith("no_eoi"):   # libjpeg decodes it with a warning, which cv2 turns into a refusal
                assert got is None or np.array_equal(got, want), (css, quality, size, name)
                continue
            assert got is not None and np.array_equal(got, want), (css, quality, size, name)


def test_table_makers(oracle):
    h = J.std_huff(oracle)
    bits, vals = J.long_code_table(h[(1, 0)][1])
    assert bits[1:11].sum() == 0 and bits[11:].sum() == 162 and sorted(vals) == sorted(h[(1, 0)][1])
    freq = np.zeros(257, np.int64)
    freq[0x00] = 100
    bits, vals = J.skewed_table(freq, h[(1, 0)][1])
    assert bits[1] == 1 and vals[0] == 0x00 and bits[1:].sum() == 162


def test_colour_space_rule_live_cv2(oracle):
    """libjpeg's colour space for three components (jdapimin.c default_decompress_parms) as live cv2 applies it: JFIF
    -> YCbCr; else Adobe transform 0 -> RGB, other transforms -> YCbCr; else ids 'R','G','B' -> RGB; else YCbCr.
    RGB means the planes themselves (each decoded on its own as a one-component stream), YCbCr their transform."""
    img = oracle.synth(40, 24, 3, 40)
    src = oracle.encode(img, 0, 90, 1)
    coef, qt, W, H, _, _ = J.source(src, oracle)
    planes = [dec(J.write_baseline(np.ascontiguousarray(coef[c::3]), qt, W, H, 0, ncomp=1, hsel=((c > 0, c > 0),) * 3,
                                   qsel=(int(c > 0),) * 3, oracle=oracle), cv2.IMREAD_GRAYSCALE) for c in range(3)]
    as_rgb = np.dstack([planes[2], planes[1], planes[0]])
    as_ycc = dec(src)
    assert not np.array_equal(as_rgb, as_ycc)
    variants = {"jfif_ids_123": (dict(), "ycc"), "jfif_ids_RGB": (dict(ids=(82, 71, 66)), "ycc"),
                "adobe0": (dict(jfif=False, adobe=0), "rgb"), "adobe1": (dict(jfif=False, adobe=1), "ycc"),
                "adobe1_ids_RGB": (dict(jfif=False, adobe=1, ids=(82, 71, 66)), "ycc"),
                "none_ids_RGB": (dict(jfif=False, ids=(82, 71, 66)), "rgb"), "none_ids_012": (dict(jfif=False, ids=(0, 1, 2)), "ycc")}
    for name, (kw, want) in variants.items():
        got = dec(J.write_baseline(coef, qt, W, H, 0, oracle=oracle, **kw))
        verdict = "ycc" if np.array_equal(got, as_ycc) else "rgb" if np.array_equal(got, as_rgb) else "neither"
        assert verdict == want, name


@pytest.fixture(scope="module")
def corpus(oracle):
    return J.corpus(oracle)


def test_corpus_decodes_in_cv2(corpus):
    """every accepted stream decodes in cv2 to the pixels of its reference stream"""
    for e in corpus:
        if e["accept"]:
            want = dec(e["ref"])
            got = dec(e["jpg"])
            assert want is not None, e["name"]
            assert got is None and e["name"].split("/")[1].startswith("no_eoi") or np.array_equal(got, want), e["name"]


def test_pillow_corpus_present(corpus):
    pytest.importorskip("PIL")
    names = [e["name"] for e in corpus if e["name"].startswith("pillow/")]
    assert len(names) == 20
    keep = [e for e in corpus if e["name"] == "pillow/keep_rgb"][0]["jpg"].tobytes()
    assert b"Adobe" in keep[:64]   # Pillow marks its RGB files with an Adobe APP14, transform 0
    big = [e for e in corpus if e["name"] == "pillow/q_16bit"][0]["jpg"].tobytes()
    assert b"\xff\xc1" in big   # SOF1: extended sequential, 16-bit tables


@pytest.fixture(scope="module")
def parse_verdict(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    exe = str(tmp_path_factory.mktemp("pv") / "parse_verdict")
    r = subprocess.run([nvcc, "-x", "cu", "-std=c++17", "-O1", "-arch=sm_100a", "--expt-relaxed-constexpr",
                        os.path.join(ROOT, "tests/cpp/parse_verdict.cpp"),
                        os.path.join(ROOT, "nvjpeg_imagecompressor_b200/csrc/dec_parse.cpp"), "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    return exe


def test_parser_verdicts(corpus, parse_verdict, tmp_path):
    """the product's parser accepts exactly the streams of the contract and refuses the others with B2J_EFORMAT"""
    paths = []
    for i, e in enumerate(corpus):
        p = str(tmp_path / f"{i}.jpg")
        e["jpg"].tofile(p)
        paths.append(p)
    r = subprocess.run([parse_verdict] + paths, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.split("\n")
    for e, line in zip(corpus, lines):
        rc, progressive, css = (int(x) for x in line.split())
        if e["accept"]:
            assert rc == 0 and progressive == int(e["progressive"]) and 0 <= css <= 4, (e["name"], line)
        else:
            assert rc == -5, (e["name"], line)
