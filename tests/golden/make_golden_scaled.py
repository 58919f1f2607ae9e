#!/usr/bin/env python
"""Generates tests/golden/golden_scaled.json from libjpeg-turbo through cv2: reduced-size decodes
(cv2.IMREAD_REDUCED_COLOR_d / IMREAD_REDUCED_GRAYSCALE_d, d = 2, 4, 8: libjpeg's DCT scaling).
- matrix: streams of cv2.imencode over sizes x content (synthetic generator with small and large noise) x the five
  subsamplings x qualities, plus restart-marker streams at q90; per stream the 128-bit digests of its colour and gray
  decodes at 1/2, 1/4, 1/8;
- files: the same digests of every committed progressive (golden_prog.json), nvJPEG-written (golden_nvjpeg.json) and
  gray (golden_gray.json) golden file;
- headline: the 8320x40000 4:2:2 q95 optimised stream of the synthetic image (seed 0, amp 8), colour and gray.
Run from the repo root:
    python tests/golden/make_golden_scaled.py
"""
import json
import os
import sys

import cv2
import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
import oracle as O  # noqa: E402
from make_golden import cv_encode, sha  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
SIZES = ((1, 1), (5, 3), (2, 40), (40, 2), (9, 17), (33, 17), (16, 16), (64, 48), (67, 93), (121, 135), (250, 301))
AMPS = (8, 120)       # content: smooth-ish / noisy
QUALITIES = (50, 90, 100)
SCALES = (2, 4, 8)
FLAGS = {2: (cv2.IMREAD_REDUCED_COLOR_2, cv2.IMREAD_REDUCED_GRAYSCALE_2),
         4: (cv2.IMREAD_REDUCED_COLOR_4, cv2.IMREAD_REDUCED_GRAYSCALE_4),
         8: (cv2.IMREAD_REDUCED_COLOR_8, cv2.IMREAD_REDUCED_GRAYSCALE_8)}


def reduced(jpg, colour=True):
    """{"c2": .., "g2": .., ...}: 128-bit digests of the reduced decodes (colour only for three-component files)"""
    out = {}
    for d in SCALES:
        if colour:
            out["c%d" % d] = sha(cv2.imdecode(jpg, FLAGS[d][0]))[:32]
        out["g%d" % d] = sha(cv2.imdecode(jpg, FLAGS[d][1]))[:32]
    return out


def matrix_cases():
    """(W, H, seed, amp, css, quality, restart_interval in MCUs) of the matrix, in file order"""
    for (W, H) in SIZES:
        for amp in AMPS:
            seed = W * 131 + H + amp
            for css in range(5):
                for q in QUALITIES:
                    yield W, H, seed, amp, css, q, 0
                mcux = O.geometry(W, H, css).mcux
                yield W, H, seed, amp, css, 90, mcux if mcux > 1 else 1


def main():
    cv2.setNumThreads(1)
    cases = []
    for (W, H, seed, amp, css, q, rst) in matrix_cases():
        img = O.synth(W, H, seed=seed, amp=amp)
        jpg = cv_encode(img, css, q, 1, rst)
        cases.append(dict(W=W, H=H, seed=seed, amp=amp, css=css, quality=q, optimize=1, restart_interval=rst,
                          jpeg_sha256_128=sha(jpg)[:32], **reduced(jpg)))
    files = []
    for name, colour in (("golden_prog.json", True), ("golden_nvjpeg.json", True), ("golden_gray.json", False)):
        with open(os.path.join(HERE, name)) as f:
            for e in json.load(f)["files"]:
                jpg = np.fromfile(os.path.join(HERE, e["file"]), np.uint8)
                files.append(dict(file=e["file"], W=e["W"], H=e["H"], jpeg_sha256=sha(jpg), **reduced(jpg, colour)))
    big = O.synth(8320, 40000, seed=0, amp=8)
    jpg = cv_encode(big, 1, 95, 1)
    del big
    headline = dict(W=8320, H=40000, seed=0, amp=8, css=1, quality=95, optimize=1, jpeg_len=int(jpg.size),
                    jpeg_sha256=sha(jpg), **{k: sha(cv2.imdecode(jpg, FLAGS[int(k[1])][k[0] == "g"]))
                                             for k in ("c2", "c4", "c8", "g2", "g4", "g8")})
    with open(os.path.join(HERE, "golden_scaled.json"), "w") as f:
        json.dump(dict(generator="tests/golden/make_golden_scaled.py, cv2 %s" % cv2.__version__, cases=cases, files=files,
                       headline=headline), f, separators=(",", ":"))
    print(len(cases), "matrix streams,", len(files), "files;", headline)


if __name__ == "__main__":
    main()
