#!/usr/bin/env python
"""Gray (B2J_CSS_GRAY) encode and decode of the headline size next to the 4:2:2 headline encode, in one run on one GPU.

The gray image is channel 1 of the synthetic headline image (8320x40000, seed 0, amp 8), the 4:2:2 image the headline
image itself. Device-resident timing as bench.py: input and output in HBM, the library on its own CUDA stream, CUDA
events on that stream around each call, warm-up runs, then the median of --reps runs; a second pass with
b2j_enable_timing gives the per-stage device times. The gray decode is timed twice: JPEG already in HBM
(b2j_decode_scan_device) and host JPEG (pinned) -> pixels in HBM (b2j_decode_device + _finish). The stream
digests are checked against tests/golden/golden_gray.json (libjpeg-turbo through cv2) and golden.json's headline.
Prints one JSON line; --out appends it to a file.
    python scripts/gray_bench.py [--reps 10] [--warmup 3] [--out profiles/gray_bench.jsonl]
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


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip()
    except Exception as e:   # informational only
        return f"unavailable: {e}"


def synth_rows(channel):
    out = torch.empty((H, W) if channel is not None else (H, W, 3), dtype=torch.uint8)
    for y0 in range(0, H, 2000):
        a = O.synth(W, H, 0, 8, y0=y0, rows=min(2000, H - y0))
        out[y0:y0 + a.shape[0]] = torch.from_numpy(np.ascontiguousarray(a[..., channel]) if channel is not None else a)
    return out.cuda()


STREAM = None   # a non-default stream: b2j_set_stream(NULL) would mean the context's own stream


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(STREAM)
        fn()
        e1.record(STREAM)
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(min(ts))


def encode_leg(css, opt, d, step, reps, warmup):
    eng = P.Engine(W, H, Q, bool(opt), css, device=0)
    eng.set_stream(STREAM.cuda_stream)

    def run():
        eng.encode_device(d.data_ptr(), step, W, H)
    med, best = timed(run, reps, warmup)
    n = eng.encode_finish()
    buf = torch.empty(n, dtype=torch.uint8)
    eng._ck(P.lib().b2j_encode_fetch(eng._h, C.c_void_p(buf.data_ptr()), n))
    eng.enable_timing(True)
    eng.encode_device(d.data_ptr(), step, W, H)
    eng.encode_finish()
    t = eng.timings()
    stages = {k: round(t[k], 4) for k in ("fdct", "hist_edge", "tables", "pack", "scan", "stuff", "total")}
    eng.close()
    return dict(css=css, optimize=opt, ms_median=round(med, 4), ms_min=round(best, 4), gpix_s=round(W * H / med / 1e6, 2), bytes=n,
                sha256=hashlib.sha256(buf.numpy().tobytes()).hexdigest(), stages_ms=stages), buf.numpy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    global STREAM
    torch.cuda.set_device(0)
    STREAM = torch.cuda.Stream()
    with open(os.path.join(ROOT, "tests", "golden", "golden_gray.json")) as f:
        gg = json.load(f)["headline"]
    with open(os.path.join(ROOT, "tests", "golden", "golden.json")) as f:
        g = json.load(f)
    want422 = [c for c in g["headline"]["encodes"] if (c["css"], c["quality"], c["optimize"]) == (1, Q, 1)]
    res = dict(what="gray vs 4:2:2, 8320x40000 q95, device resident", gpu=gpu_info(), reps=a.reps, warmup=a.warmup, legs=[])
    dg = synth_rows(1)
    jpg_opt = None
    for opt in (1, 0):
        leg, jpg = encode_leg("gray", opt, dg, W, a.reps, a.warmup)
        leg["golden_ok"] = leg["bytes"] == gg["jpeg_len_opt%d" % opt] and leg["sha256"] == gg["jpeg_sha256_opt%d" % opt]
        res["legs"].append(leg)
        if opt:
            jpg_opt = jpg
    # decodes of the optimised gray stream: JPEG in HBM -> pixels in HBM, and host JPEG (pinned) -> pixels in HBM
    eng = P.Engine(W, H, Q, True, "gray", device=0)
    eng.set_stream(STREAM.cuda_stream)
    out = torch.empty((H, W), dtype=torch.uint8, device="cuda")
    pin = torch.from_numpy(jpg_opt).pin_memory().numpy()
    b = jpg_opt.tobytes()
    p = 2
    while b[p + 1] != 0xDA:
        p += 2 + ((b[p + 2] << 8) | b[p + 3])
    hdr_len = p + 2 + ((b[p + 2] << 8) | b[p + 3])
    d_scan = torch.from_numpy(jpg_opt[hdr_len:-2].copy()).cuda()
    hdr = jpg_opt[:hdr_len].copy()

    def dec_hbm():
        eng.decode_scan_device(hdr, d_scan.data_ptr(), d_scan.numel(), out.data_ptr(), W)

    def dec_host():
        eng.decode_device(pin, out.data_ptr(), W)
        eng.decode_finish()
    for op, fn in (("decode, JPEG in HBM", dec_hbm), ("decode, pinned host JPEG", dec_host)):
        out.zero_()
        med, best = timed(fn, a.reps, a.warmup)
        eng.enable_timing(True)
        fn()
        eng.enable_timing(False)
        t = eng.timings()
        ok = hashlib.sha256(out.cpu().numpy().tobytes()).hexdigest() == gg["decoded_sha256"]
        res["legs"].append(dict(css="gray", op=op, ms_median=round(med, 4), ms_min=round(best, 4), gpix_s=round(W * H / med / 1e6, 2),
                                stages_ms={k: round(t[k], 4) for k in ("dec_parse", "dec_sync", "dec_write", "dec_idct", "dec_color", "total")},
                                golden_ok=ok))
    eng.close()
    del dg, out
    d3 = synth_rows(None)
    leg, _ = encode_leg("422", 1, d3, W * 3, a.reps, a.warmup)
    leg["golden_ok"] = bool(want422) and leg["bytes"] == want422[0]["jpeg_len"] and leg["sha256"][:32] == want422[0]["jpeg_sha256_128"]
    res["legs"].append(leg)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
