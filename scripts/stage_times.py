#!/usr/bin/env python
"""Per-stage device times of one encode configuration (CUDA events inside the library)."""
import argparse, json, sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import nvjpeg_imagecompressor_b200 as P
from nvjpeg_imagecompressor_b200.synth import synth

ap = argparse.ArgumentParser()
ap.add_argument("--width", type=int, default=8320)
ap.add_argument("--height", type=int, default=40000)
ap.add_argument("--css", default="422")
ap.add_argument("--quality", type=int, default=95)
ap.add_argument("--optimize", type=int, default=1)
ap.add_argument("--iters", type=int, default=5)
ap.add_argument("--debug", type=int, default=0, help="b2j_set_debug flags (include/b2jpeg.h)")
a = ap.parse_args()
img = synth(a.width, a.height)
torch.cuda.synchronize()
eng = P.Engine(a.width, a.height, a.quality, bool(a.optimize), a.css)
eng.enable_timing(True)
eng.set_debug(a.debug)
eng.set_stream(torch.cuda.current_stream().cuda_stream)
for i in range(a.iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.encode_device(img.data_ptr(), a.width * 3, a.width, a.height)
    e1.record()
    n = eng.encode_finish()
    t = eng.timings()
    ms = e0.elapsed_time(e1)
    print(json.dumps(dict(iter=i, debug=a.debug, bytes=n, ms=round(ms, 3), mpix_s=round(a.width * a.height / ms / 1e3, 1),
                          **{k: round(v, 3) for k, v in t.items() if k in ("fdct", "hist_edge", "tables", "pack", "scan", "stuff", "total")})))
