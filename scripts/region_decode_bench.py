#!/usr/bin/env python
"""Region decode (b2j_set_decode_region) of the headline stream, with one restart interval per MCU row and without
restart markers, in one run on one GPU.

The stream is the 8320x40000 4:2:2 q95 optimised JPEG of the synthetic headline image (seed 0, amp 8), encoded on the
GPU twice: restart rows 1 and 0. Regions: the whole image; 1920x1080 at the top, middle and bottom; 256x256 in the
middle; a full-width band of 64 rows. Two legs, CUDA events on the library's stream, the regions (full decode
included) alternated round by round so that drift hits all of them alike; median and best of --reps rounds after
--warmup rounds:
  hbm   JPEG already in HBM -> region in HBM (b2j_decode_scan_device)
  h2d   host JPEG (pinned) -> region in HBM (b2j_decode_device + b2j_decode_finish)
Every region is checked against the crop of the whole decode. A last pass with b2j_enable_timing gives the decoder's
per-stage device times per region. Prints one JSON line with the GPU name and power limit; --out appends it to a file.
    python scripts/region_decode_bench.py [--reps 10] [--warmup 2] [--out profiles/region_decode.jsonl]
"""
import argparse
import ctypes as C
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
REGIONS = {"full": None, "1080p_top": (0, 0, 1920, 1080), "1080p_mid": ((W - 1920) // 2, (H - 1080) // 2, 1920, 1080),
           "1080p_bottom": (W - 1920, H - 1080, 1920, 1080), "256_mid": ((W - 256) // 2, (H - 256) // 2, 256, 256),
           "band64": (0, H // 2, W, 64)}


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip()
    except Exception as e:   # informational only
        return f"unavailable: {e}"


def split_scan(jpg):
    b = jpg.tobytes()
    p = 2
    while b[p + 1] != 0xDA:
        p += 2 + ((b[p + 2] << 8) | b[p + 3])
    hdr_len = p + 2 + ((b[p + 2] << 8) | b[p + 3])
    return jpg[:hdr_len].copy(), jpg[hdr_len:-2].copy()


def run_stream(eng, stream, jpg, reps, warmup):
    hdr, scan = split_scan(jpg)
    d_scan = torch.from_numpy(scan).cuda()
    outs = {k: torch.empty(((r or (0, 0, W, H))[3], (r or (0, 0, W, H))[2] * 3), dtype=torch.uint8, device="cuda")
            for k, r in REGIONS.items()}

    def leg(kind, k):
        eng.set_decode_region(*(REGIONS[k] or (None,)))
        o = outs[k]
        if kind == "hbm":
            eng.decode_scan_device(hdr, d_scan.data_ptr(), d_scan.numel(), o.data_ptr(), o.shape[1])
        else:
            eng.decode_device(jpg, o.data_ptr(), o.shape[1])
            eng.decode_finish()

    kinds = ("hbm", "h2d")
    times = {(kind, k): [] for kind in kinds for k in REGIONS}
    for r in range(warmup + reps):
        for kind in kinds:
            for k in REGIONS:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                leg(kind, k)
                e1.record(stream)
                e1.synchronize()
                if r >= warmup:
                    times[(kind, k)].append(e0.elapsed_time(e1))
    full = outs["full"]
    for k, reg in REGIONS.items():
        if reg:
            x, y, w, h = reg
            assert torch.equal(outs[k], full[y:y + h, 3 * x:3 * (x + w)]), k
    stages = {}
    eng.enable_timing(True)
    for k in REGIONS:
        leg("hbm", k)
        t = eng.timings()
        stages[k] = {n: round(t[n], 4) for n in ("dec_parse", "dec_sync", "dec_write", "dec_idct", "dec_color", "total")}
    eng.enable_timing(False)
    eng.set_decode_region(None)
    return ({f"{kind}_{k}": dict(median=round(float(np.median(times[(kind, k)])), 4), best=round(float(min(times[(kind, k)])), 4))
             for kind in kinds for k in REGIONS}, stages)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out")
    a = ap.parse_args()
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    img = torch.empty((H, W, 3), dtype=torch.uint8)
    for y0 in range(0, H, 2000):
        img[y0:y0 + 2000] = torch.from_numpy(O.synth(W, H, 0, 8, y0=y0, rows=min(2000, H - y0)))
    d_img = img.cuda()
    del img
    eng = P.Engine(W, H, Q, True, "422", device=0)
    eng.set_stream(stream.cuda_stream)
    res = dict(bench="region_decode", gpu=gpu_info(), image=f"{W}x{H} 4:2:2 q{Q} optimised", reps=a.reps, warmup=a.warmup,
               regions={k: r for k, r in REGIONS.items()}, crops_match=True, streams={})
    for rows in (1, 0):
        eng.set_restart_rows(rows)
        eng.encode_device(d_img.data_ptr(), W * 3, W, H)
        n = eng.encode_finish()
        jpg_t = torch.empty(n, dtype=torch.uint8).pin_memory()
        eng._ck(P.lib().b2j_encode_fetch(eng._h, C.c_void_p(jpg_t.data_ptr()), n))
        ms, stages = run_stream(eng, stream, jpg_t.numpy(), a.reps, a.warmup)
        res["streams"][f"restart_rows_{rows}"] = dict(jpeg_bytes=int(n), ms=ms, stages_ms=stages)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
