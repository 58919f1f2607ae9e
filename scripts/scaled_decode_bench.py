#!/usr/bin/env python
"""Reduced-size decode (b2j_set_decode_scale) of the headline stream at 1/1, 1/2, 1/4 and 1/8, in one run on one GPU.

The stream is the 8320x40000 4:2:2 q95 optimised JPEG of the synthetic headline image (seed 0, amp 8), encoded on the
GPU; its digest and the reduced decodes' digests are checked against tests/golden/golden_scaled.json (libjpeg-turbo
through cv2). Three legs per scale, CUDA events on the library's stream, the scales alternated round by round so that
drift hits all of them alike; median and best of --reps rounds after --warmup rounds:
  hbm   JPEG already in HBM -> pixels in HBM (b2j_decode_scan_device)
  h2d   host JPEG (pinned) -> pixels in HBM (b2j_decode_device + b2j_decode_finish)
  h2h   host JPEG (pinned) -> host pixels (pageable, b2j_decode)
A last pass with b2j_enable_timing gives the decoder's per-stage device times (dec_idct, dec_color) per scale.
Prints one JSON line with the GPU name and power limit; --out appends it to a file.
    python scripts/scaled_decode_bench.py [--reps 10] [--warmup 2] [--out profiles/scaled_decode.jsonl]
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import nvjpeg_imagecompressor_b200 as P  # noqa: E402
import oracle as O  # noqa: E402

W, H, Q = 8320, 40000, 95
SCALES = (1, 2, 4, 8)


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip()
    except Exception as e:   # informational only
        return f"unavailable: {e}"


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def split_scan(jpg):
    b = jpg.tobytes()
    p = 2
    while b[p + 1] != 0xDA:
        p += 2 + ((b[p + 2] << 8) | b[p + 3])
    hdr_len = p + 2 + ((b[p + 2] << 8) | b[p + 3])
    return jpg[:hdr_len].copy(), jpg[hdr_len:-2].copy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out")
    a = ap.parse_args()
    with open(os.path.join(ROOT, "tests", "golden", "golden_scaled.json")) as f:
        gold = json.load(f)["headline"]
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    img = torch.empty((H, W, 3), dtype=torch.uint8)
    for y0 in range(0, H, 2000):
        img[y0:y0 + 2000] = torch.from_numpy(O.synth(W, H, 0, 8, y0=y0, rows=min(2000, H - y0)))
    d_img = img.cuda()
    del img
    eng = P.Engine(W, H, Q, True, "422", device=0)
    eng.set_stream(stream.cuda_stream)
    eng.encode_device(d_img.data_ptr(), W * 3, W, H)
    n = eng.encode_finish()
    del d_img
    jpg_t = torch.empty(n, dtype=torch.uint8).pin_memory()
    eng._ck(P.lib().b2j_encode_fetch(eng._h, C.c_void_p(jpg_t.data_ptr()), n))
    jpg = jpg_t.numpy()
    assert sha(jpg) == gold["jpeg_sha256"], "headline stream differs from libjpeg-turbo's"
    hdr, scan = split_scan(jpg)
    d_scan = torch.from_numpy(scan).cuda()
    outs = {d: torch.empty(((H + d - 1) // d, ((W + d - 1) // d) * 3), dtype=torch.uint8, device="cuda") for d in SCALES}
    hosts = {d: np.empty(((H + d - 1) // d, (W + d - 1) // d, 3), np.uint8) for d in SCALES}

    def leg(kind, d):
        eng.set_decode_scale(d)
        o = outs[d]
        step = o.shape[1]
        if kind == "hbm":
            eng.decode_scan_device(hdr, d_scan.data_ptr(), d_scan.numel(), o.data_ptr(), step)
        elif kind == "h2d":
            eng.decode_device(jpg, o.data_ptr(), step)
            eng.decode_finish()
        else:
            eng.decode_ptr(jpg, hosts[d].ctypes.data, hosts[d].shape[1] * 3)

    kinds = ("hbm", "h2d", "h2h")
    times = {(k, d): [] for k in kinds for d in SCALES}
    for r in range(a.warmup + a.reps):
        for k in kinds:
            for d in SCALES:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                leg(k, d)
                e1.record(stream)
                e1.synchronize()
                if r >= a.warmup:
                    times[(k, d)].append(e0.elapsed_time(e1))
    digests = {}
    for d in SCALES:
        if d > 1:
            digests["c%d" % d] = sha(outs[d].cpu().numpy()) == gold["c%d" % d] and sha(hosts[d]) == gold["c%d" % d]
    assert all(digests.values()), digests
    stages = {}
    eng.enable_timing(True)
    for d in SCALES:
        leg("hbm", d)
        t = eng.timings()
        stages[d] = {k: round(t[k], 4) for k in ("dec_parse", "dec_sync", "dec_write", "dec_idct", "dec_color")}
    eng.enable_timing(False)
    res = dict(bench="scaled_decode", gpu=gpu_info(), image=f"{W}x{H} 4:2:2 q{Q} optimised", jpeg_bytes=int(n),
               reps=a.reps, warmup=a.warmup, digests_match=True,
               ms={f"{k}_d{d}": dict(median=round(float(np.median(times[(k, d)])), 4), best=round(float(min(times[(k, d)])), 4))
                   for k in kinds for d in SCALES},
               out_bytes={f"d{d}": int(outs[d].numel()) for d in SCALES},
               stages_ms={f"d{d}": stages[d] for d in SCALES})
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
