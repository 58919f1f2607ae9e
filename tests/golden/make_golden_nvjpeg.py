#!/usr/bin/env python
"""Generates tests/golden/nvjpeg_*.jpg + golden_nvjpeg.json: what the reference's nvJPEG path writes, so that the
GPU suite compares against it without nvJPEG. Needs a CUDA device, the nvJPEG harness (baseline/ref_nvjpeg.cu = the
reference's call sequence, built by `make -C baseline`) and cv2 for libjpeg-turbo's pixels of every stream.

  files      small streams written by nvJPEG (baseline sequential and progressive, optimised Huffman, no restart
             markers) with the digests of cv2.imdecode's pixels
  size_psnr  nvJPEG's byte count and reconstruction PSNR at 4096x3072, 4:2:2, q95 (too large to store the stream)

Run from the repo root:  python tests/golden/make_golden_nvjpeg.py [output directory, default tests/golden]
"""
import ctypes as C
import json
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.join(HERE, "..", "..")
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
import oracle as O  # noqa: E402
from make_golden import sha  # noqa: E402

# (W, H, seed, quality, progressive, css list); css numbering as the library's (444, 422, 440, 420, 411)
STREAMS = ((384, 288, 3, 90, 0, (1, 0, 3)), (256, 192, 3, 95, 1, (0, 1, 3)))
SIZE_PSNR = dict(W=4096, H=3072, seed=0, amp=8, css=1, quality=95, optimize=1)


def nvjpeg_encode(L, img, css, quality, progressive):
    H, W = img.shape[:2]
    h = C.c_void_p()
    assert L.ref_create(W, H, quality, 1, css, progressive, C.byref(h)) == 0
    assert L.ref_build_compress_env(h) == 0, "nvJPEG env setup failed"
    out = np.empty(W * H * 3, np.uint8)
    n = C.c_size_t(0)
    rc = L.ref_compress(h, C.c_void_p(img.ctypes.data), C.c_size_t(W * 3), C.c_void_p(out.ctypes.data), C.c_size_t(out.size),
                        C.byref(n))
    L.ref_destroy(h)
    assert rc == 0, f"ref_compress rc={rc}"
    return out[: n.value].copy()


def nvjpeg_version():
    v = [C.c_int(0) for _ in range(3)]
    nj = C.CDLL("libnvjpeg.so.12")
    for k in range(3):   # MAJOR_VERSION, MINOR_VERSION, PATCH_LEVEL
        nj.nvjpegGetProperty(k, C.byref(v[k]))
    return ".".join(str(x.value) for x in v)


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else HERE
    os.makedirs(out_dir, exist_ok=True)
    cv2.setNumThreads(1)
    L = C.CDLL(os.path.join(ROOT, "baseline", "_ref", "libref_nvjpeg.so"))
    files = []
    for (W, H, seed, q, prog, csss) in STREAMS:
        img = O.synth(W, H, seed, 8)
        for css in csss:
            jpg = nvjpeg_encode(L, img, css, q, prog)
            dec = cv2.imdecode(jpg, cv2.IMREAD_COLOR)
            assert dec is not None and dec.shape == (H, W, 3)
            assert np.array_equal(O.decode(jpg), dec)
            name = f"nvjpeg_{W}x{H}_css{css}_q{q}_{'prog' if prog else 'base'}.jpg"
            jpg.tofile(os.path.join(out_dir, name))
            files.append(dict(file=name, W=W, H=H, seed=seed, amp=8, css=css, quality=q, optimize=1, progressive=prog,
                              jpeg_sha256=sha(jpg), decoded_sha256=sha(dec)))
    s = SIZE_PSNR
    img = O.synth(s["W"], s["H"], s["seed"], s["amp"])
    jpg = nvjpeg_encode(L, img, s["css"], s["quality"], 0)
    dec = cv2.imdecode(jpg, cv2.IMREAD_COLOR)
    assert np.array_equal(O.decode(jpg), dec)
    size_psnr = dict(s, jpeg_len=int(jpg.size), psnr=O.psnr(img, dec))
    import torch
    gen = "tests/golden/make_golden_nvjpeg.py, nvJPEG %s on %s, cv2 %s" % (nvjpeg_version(), torch.cuda.get_device_name(0),
                                                                          cv2.__version__)
    with open(os.path.join(out_dir, "golden_nvjpeg.json"), "w") as f:
        json.dump(dict(generator=gen, files=files, size_psnr=size_psnr), f, indent=1)
    print(gen, len(files), "files", size_psnr)


if __name__ == "__main__":
    main()
