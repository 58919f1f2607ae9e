#!/usr/bin/env python
"""Generates tests/golden/golden_gray.json and the small gray files next to it, from libjpeg-turbo through cv2:
- digests of cv2.imencode streams of one-channel images (sizes x qualities x Huffman modes x restart intervals, the
  interval counted in blocks = MCUs of the one-component scan) and of their cv2.imdecode(IMREAD_UNCHANGED) pixels;
- IMREAD_GRAYSCALE digests (libjpeg's JCS_GRAYSCALE output: the Y plane) of colour streams in all five subsamplings,
  baseline, with restart markers and progressive;
- the headline gray image (channel 1 of the 8320x40000 synthetic image) at q95 in both Huffman modes;
- gray/gray_*.jpg: a baseline file, one with restart markers, a progressive one and one whose SOF declares sampling 0x22.
Images are channel 1 of the synthetic generator (oracle.synth(W, H, seed, 8)[..., 1]). Run from the repo root:
    python tests/golden/make_golden_gray.py
"""
import json
import os
import sys

import cv2
import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
import oracle as O  # noqa: E402
from make_golden import SF, cv_encode, sha  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
SIZES = ((1, 1), (2, 2), (8, 8), (17, 33), (33, 17), (135, 121), (257, 63), (640, 360))


def gray_img(W, H, seed):
    return np.ascontiguousarray(O.synth(W, H, seed=seed, amp=8)[..., 1])


def cv_gray(img, q, opt, rst=0, prog=0):
    p = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, opt]
    if rst:
        p += [cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    if prog:
        p += [cv2.IMWRITE_JPEG_PROGRESSIVE, 1]
    ok, jpg = cv2.imencode(".jpg", img, p)
    assert ok
    return jpg.ravel()


def patch_sampling(jpg, hv):
    """the one component's sampling factor byte in SOF0 / SOF2 replaced (cv2 decodes it as 1x1 regardless)"""
    b = bytearray(jpg.tobytes())
    i = 2
    while b[i + 1] not in (0xC0, 0xC2):
        i += 2 + ((b[i + 2] << 8) | b[i + 3])
    b[i + 11] = hv
    return np.frombuffer(bytes(b), np.uint8)


def main():
    cv2.setNumThreads(1)
    enc = []
    for (W, H) in SIZES:
        seed = W * 31 + H
        img = gray_img(W, H, seed)
        mcux = (W + 7) // 8
        for q in (40, 75, 95, 100):
            for opt in (0, 1):
                for rst in sorted({0, 1, 5, mcux, 2 * mcux}):
                    jpg = cv_gray(img, q, opt, rst)
                    dec = cv2.imdecode(jpg, cv2.IMREAD_UNCHANGED)
                    enc.append(dict(W=W, H=H, seed=seed, quality=q, optimize=opt, restart_interval=int(rst), jpeg_len=int(jpg.size),
                                    jpeg_sha256_128=sha(jpg)[:32], decoded_sha256_128=sha(dec)[:32]))
    ydec = []
    for (W, H) in ((17, 33), (135, 121), (640, 360)):
        seed = W * 31 + H
        img = O.synth(W, H, seed=seed, amp=8)
        for css in range(5):
            mcux = O.geometry(W, H, css).mcux
            for kind, rst in (("base", 0), ("rst", mcux), ("prog", 0)):
                if kind == "prog":
                    jpg = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SF[css],
                                                     cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].ravel()
                else:
                    jpg = cv_encode(img, css, 90, 1, rst)
                dec = cv2.imdecode(jpg, cv2.IMREAD_GRAYSCALE)
                ydec.append(dict(W=W, H=H, seed=seed, css=css, quality=90, optimize=1, kind=kind, restart_interval=int(rst),
                                 jpeg_sha256_128=sha(jpg)[:32], gray_sha256_128=sha(dec)[:32]))
    files = []
    img = gray_img(135, 121, 7)
    variants = (("gray_135x121_q90_base.jpg", cv_gray(img, 90, 1)),
                ("gray_135x121_q90_rst5.jpg", cv_gray(img, 90, 0, 5)),
                ("gray_135x121_q90_prog.jpg", cv_gray(img, 90, 1, prog=1)),
                ("gray_135x121_q90_sof22.jpg", patch_sampling(cv_gray(img, 90, 1), 0x22)))
    for name, jpg in variants:
        os.makedirs(os.path.join(HERE, "gray"), exist_ok=True)
        jpg.tofile(os.path.join(HERE, "gray", name))
        dec = cv2.imdecode(jpg, cv2.IMREAD_UNCHANGED)
        files.append(dict(file="gray/" + name, W=135, H=121, jpeg_sha256=sha(jpg), decoded_sha256=sha(dec)))
    big = np.ascontiguousarray(O.synth(8320, 40000, seed=0, amp=8)[..., 1])
    headline = dict(W=8320, H=40000, seed=0, quality=95)
    for opt in (1, 0):
        jpg = cv_gray(big, 95, opt)
        headline["jpeg_len_opt%d" % opt] = int(jpg.size)
        headline["jpeg_sha256_opt%d" % opt] = sha(jpg)
        if opt:
            headline["decoded_sha256"] = sha(cv2.imdecode(jpg, cv2.IMREAD_UNCHANGED))
    with open(os.path.join(HERE, "golden_gray.json"), "w") as f:
        json.dump(dict(generator="tests/golden/make_golden_gray.py, cv2 %s" % cv2.__version__, encode=enc, ydecode=ydec,
                       files=files, headline=headline), f, separators=(",", ":"))
    print(len(enc), "encode cases,", len(ydec), "Y-plane decodes,", len(files), "files;", headline)


if __name__ == "__main__":
    main()
