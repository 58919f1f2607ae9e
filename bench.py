#!/usr/bin/env python
"""bench.py -- BASELINE.json's headline metric on B200: encode Mpix/s of one synthetic 8320x40000 BGR image,
quality 95, 4:2:2, optimized Huffman (config 2), bit-exact with libjpeg-turbo.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

N=1 : the whole image on one GPU.  N>1 (torchrun, one rank per GPU): the image is cut into MCU-row strips, one per
      GPU, stitched through a 4 KB per-strip record exchanged over peer memory (NCCL all_gather as the fallback).
One "step" = one complete encode of the image (device-resident input -> complete JPEG bytes in HBM).
Prints ONE JSON line (rank 0). `value` is device-resident throughput, `e2e` is the same metric through the C-ABI with
pinned HOST buffers (H2D of the pixels and D2H of the JPEG inside the timed region).

--impl reference: the reference's nvJPEG path (baseline/ref_nvjpeg.cu = its exact call sequence, see that file) on
      the same GPU, else -- if nvJPEG cannot run -- libjpeg-turbo (cv2.imencode) on the host cores.
--dump-outputs DIR: the JPEG of the last timed step as .npy arrays (see dump_outputs), so that two builds can be
      compared output for output; the input image is the same on every run.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only: leave no __pycache__ in it

W, H, QUALITY, CSS, OPT = 8320, 40000, 95, "422", 1
WORKLOAD = "8320x40000 BGR synth(seed=0,amp=8), q95, 4:2:2, optimized Huffman (BASELINE.json configs[1])"
PEAKS_FALLBACK_GBS = 6650.0
PUBLISHED_MPIX_S = 1652.0   # BASELINE.md section 1 (reference README.md:48): 332.8 Mpix / 201.45 ms, RTX 3060


def kernel_source_digest():
    """sha256 over the CUDA sources of the ENCODE kernels (the ones profiles/traffic.json holds): the file carries the
    digest of the code it was captured on (scripts/ncu_export.py); a capture of other code is not reported as this run's
    traffic. Decoder-only sources do not count."""
    import hashlib
    h = hashlib.sha256()
    for f in [os.path.join(ROOT, "nvjpeg_imagecompressor_b200", "csrc", n) for n in ("common.cuh", "enc_fdct.cu", "enc_huff.cu")]:
        with open(f, "rb") as fh:
            h.update(os.path.basename(f).encode() + b"\0" + fh.read())
    return h.hexdigest()[:16]


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return PEAKS_FALLBACK_GBS, "fallback"


DUMP_SAMPLE = 1 << 22


def dump_outputs(d, jpg):
    """Writes the JPEG bytes `jpg` as float arrays: jpeg_length.npy, jpeg_sha256.npy (the 32 digest bytes of the whole
    stream), jpeg_index.npy and jpeg_bytes.npy (the bytes at those positions: all of them up to DUMP_SAMPLE bytes, else
    a sorted sample of positions drawn with seed 0, so that the directory stays below 64 MB)."""
    os.makedirs(d, exist_ok=True)
    n = int(jpg.size)
    idx = np.arange(n) if n <= DUMP_SAMPLE else np.unique(np.random.default_rng(0).integers(0, n, DUMP_SAMPLE))
    np.save(os.path.join(d, "jpeg_length.npy"), np.array([n], np.float64))
    np.save(os.path.join(d, "jpeg_sha256.npy"), np.frombuffer(hashlib.sha256(jpg.tobytes()).digest(), np.uint8).astype(np.float32))
    np.save(os.path.join(d, "jpeg_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(d, "jpeg_bytes.npy"), jpg[idx].astype(np.float32))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], False, None
        self.t_lo, self.t_hi = 0.0, float("inf")

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([time.time()] + [x.strip() for x in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                mx = max(mx, float(r[2]))
                if not (self.t_lo <= r[0] <= self.t_hi):
                    continue
                sm.append(float(r[1]))
                for i, n in enumerate(names):
                    if r[4 + i].lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "window": "timed device-resident steps + timed end-to-end steps (GPU busy throughout)"}


# ------------------------------------------------------------------------------------------------ CPU baseline
def _cv_worker(args):
    import cv2
    cv2.setNumThreads(1)
    arr, y0, y1, css, q, opt, reps = args
    sf = {"444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
          "440": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, "420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420,
          "411": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411}[css]
    n = 0
    for _ in range(reps):
        ok, b = cv2.imencode(".jpg", arr[y0:y1], [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, opt,
                                                  cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sf])
        n += b.size
    return n


_SHARED = {}


def _cv_worker_shared(args):
    y0, y1, css, q, opt, reps = args
    return _cv_worker((_SHARED["img"], y0, y1, css, q, opt, reps))


def cpu_baseline(sample_rows=8000, reps=10):
    """libjpeg-turbo 3.1.2 (cv2.imencode, the north-star's bit-exactness oracle) on all host cores: the first
    `sample_rows` rows of the workload cut into one MCU-row-aligned strip per core, one process per core."""
    import multiprocessing as mp
    import oracle as O
    cores = os.cpu_count() or 1
    rows = min(H, sample_rows)
    img = O.synth(W, H, 0, 8, y0=0, rows=rows)
    _SHARED["img"] = img
    per = max(8, (rows // cores) // 8 * 8)
    jobs = [(y, min(rows, y + per), CSS, QUALITY, OPT, reps) for y in range(0, rows, per)]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_cv_worker_shared, [(0, 8, CSS, QUALITY, OPT, 1)] * cores)  # warm the workers
        t0 = time.perf_counter()
        pool.map(_cv_worker_shared, jobs)
        dt = time.perf_counter() - t0
    mpix = W * rows * reps / 1e6
    return {"value": round(mpix / dt, 2), "unit": "Mpix/s", "cores": cores, "kind": "port",
            "sample": f"cv2.imencode (libjpeg-turbo 3.1.2, the bit-exactness oracle itself) on the first {rows} rows of the "
                      f"workload, {len(jobs)} MCU-row strips, one process per core, {dt:.2f} s"}


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args, rank, world):
    if rank != 0:
        return None
    import oracle as O
    line = {"impl": "reference", "metric": "encode_mpix_per_s", "unit": "Mpix/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": {"workload": WORKLOAD}}
    lib = os.path.join(ROOT, "baseline", "_ref", "libref_nvjpeg.so")
    err = None
    if args.ref_kind in ("auto", "nvjpeg") and os.path.exists(lib):
        try:
            import torch
            if not torch.cuda.is_available():
                raise RuntimeError("no CUDA device")
            L = C.CDLL(lib)
            h = C.c_void_p()
            assert L.ref_create(W, H, QUALITY, OPT, 1, int(args.ref_progressive), C.byref(h)) == 0
            if L.ref_build_compress_env(h) != 0:
                raise RuntimeError("nvJPEG env setup failed")
            img = np.empty((H, W, 3), np.uint8)
            for y0 in range(0, H, 2000):
                img[y0:y0 + 2000] = O.synth(W, H, 0, 8, y0=y0, rows=2000)
            out = np.empty(W * H * 3, np.uint8)
            n = C.c_size_t(0)
            gpu_ms, e2e_ms = [], []
            tt = [C.c_float(0) for _ in range(4)]
            for i in range(args.warmup + args.steps):
                t0 = time.perf_counter()
                rc = L.ref_compress(h, C.c_void_p(img.ctypes.data), C.c_size_t(W * 3), C.c_void_p(out.ctypes.data),
                                    C.c_size_t(out.size), C.byref(n))
                dt = (time.perf_counter() - t0) * 1e3
                if rc != 0:
                    raise RuntimeError(f"ref_compress rc={rc}")
                L.ref_last_times(h, *[C.byref(t) for t in tt])
                if i >= args.warmup:
                    e2e_ms.append(dt)
            # device-resident bracket (planes already uploaded): the reference's own bracket ImageCompressorImpl.cu:279-281
            # (events around nvjpegEncodeImage only: `strict`) and the same with the size query inside, i.e. until the
            # bitstream is complete on the device (`value`, as in round 1)
            strict_ms = []
            L.ref_encode_resident2.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_size_t)]
            for strict in (1, 0):
                for i in range(args.warmup + args.steps):
                    ms = C.c_float(0)
                    if L.ref_encode_resident2(h, strict, C.byref(ms), C.byref(n)) != 0:
                        raise RuntimeError("ref_encode_resident failed")
                    if i >= args.warmup:
                        (strict_ms if strict else gpu_ms).append(ms.value)
            # the reference's decode of the JPEG it just wrote (DecodeWorker + getCVImageOnCPU: ImageCompressorImpl.cu:311-385,
            # :184-232): device phase (host JPEG -> planar BGR in HBM, cudaEvent bracket) and the whole call (3 x D2H + CPU
            # interleave into a host BGR image)
            ref_decode = None
            try:
                if L.ref_build_decode_env(h) == 0:
                    jpg = out[: n.value].copy()
                    rec = np.empty((H, W, 3), np.uint8)
                    w_, h_, gms = C.c_int(0), C.c_int(0), C.c_float(0)
                    dev_ms, wall_ms = [], []
                    for i in range(3):
                        t0 = time.perf_counter()
                        rc = L.ref_decode(h, C.c_void_p(jpg.ctypes.data), C.c_size_t(jpg.size), C.c_void_p(rec.ctypes.data),
                                          C.c_size_t(W * 3), C.byref(w_), C.byref(h_), C.byref(gms))
                        if rc != 0:
                            raise RuntimeError(f"ref_decode rc={rc}")
                        if i:
                            dev_ms.append(gms.value)
                            wall_ms.append((time.perf_counter() - t0) * 1e3)
                    ref_decode = {"metric": "decode_mpix_per_s", "value": round(W * H / float(np.mean(dev_ms)) / 1e3, 1), "unit": "Mpix/s",
                                  "ms_per_step": round(float(np.mean(dev_ms)), 2),
                                  "e2e": {"value": round(W * H / float(np.mean(wall_ms)) / 1e3, 1), "unit": "Mpix/s",
                                          "ms_per_step": round(float(np.mean(wall_ms)), 1)}}
            except Exception as e:
                ref_decode = {"error": f"{type(e).__name__}: {e}"}
            L.ref_destroy(h)
            ms = float(np.mean(gpu_ms))
            e2e = float(np.mean(e2e_ms))
            line.update({"value": round(W * H / ms / 1e3, 1), "ms_per_step": round(ms, 3), "gpu_launches": None,
                         "e2e": {"value": round(W * H / e2e / 1e3, 1), "unit": "Mpix/s", "ms_per_step": round(e2e, 2),
                                 "h2d_bytes_per_step": W * H * 3, "d2h_bytes_per_step": int(n.value),
                                 "split_ms": round(tt[1].value, 1), "h2d_ms": round(tt[2].value, 1),
                                 "split": "SSSE3 byte shuffles, one thread (a stand-in for cv::split's SIMD path)",
                                 "device_ms_with_size_query": round(ms, 3),
                                 "device_ms_strict_bracket": round(float(np.mean(strict_ms)), 3),
                                 "device_mpix_s_strict_bracket": round(W * H / float(np.mean(strict_ms)) / 1e3, 1)},
                         "reference_kind": "nvjpeg call sequence of ImageCompressorImpl.cu:19-45,269-294 "
                                           f"({'progressive as shipped' if args.ref_progressive else 'baseline sequential'}, "
                                           "4:2:2, q95, optimized Huffman) on this GPU; n_gpus ignored (single-GPU library)",
                         "jpeg_bytes": int(n.value)})
            line["vs_baseline"] = round(line["value"] / PUBLISHED_MPIX_S, 2)
            if ref_decode is not None:
                line["decode"] = ref_decode
                line["e2e"]["decode"] = ref_decode
            line["cpu_baseline"] = cpu_baseline()
            return line
        except Exception as e:  # fall through to the CPU arm
            err = f"{type(e).__name__}: {e}"
    cb = cpu_baseline(sample_rows=8000, reps=max(1, args.steps // 4))
    line.update({"value": cb["value"], "ms_per_step": round(W * H / 1e3 / cb["value"], 2), "cpu_baseline": cb,
                 "e2e": {"value": cb["value"], "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                 "vs_baseline": round(cb["value"] / PUBLISHED_MPIX_S, 2),
                 "reference_kind": "libjpeg-turbo on host cores (nvJPEG harness unavailable: %s)" % err})
    return line


# ------------------------------------------------------------------------------------------------ own arm
def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import nvjpeg_imagecompressor_b200 as P
    from nvjpeg_imagecompressor_b200.strips import StripEncoder, _view, strip_rows
    from nvjpeg_imagecompressor_b200.synth import synth_rows
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    P.lib()
    css_i = P.CSS[CSS]
    rows = strip_rows(H, css_i, world)
    y0, y1 = rows[rank]
    nrows = y1 - y0
    img = torch.empty((nrows, W, 3), dtype=torch.uint8, device=dev)
    for r0 in range(0, nrows, 500):
        n = min(500, nrows - r0)
        img[r0:r0 + n] = synth_rows(W, H, y0 + r0, n, 0, 8, dev)
    stream = torch.cuda.Stream(device=dev)
    sampler = ClockSampler(local_rank) if rank == 0 else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    stage_acc, launches0 = {}, 0
    if world == 1:
        eng = P.Engine(W, H, QUALITY, bool(OPT), CSS, device=local_rank)
        eng.set_stream(stream.cuda_stream)

        def step():   # asynchronous, like the strip step: the length word stays in HBM next to the bytes
            return eng.encode_device(img.data_ptr(), W * 3, W, H)[0]
    else:
        enc = StripEncoder(W, H, QUALITY, bool(OPT), CSS, device=local_rank)
        exchange = {"peer memory": "NVLink stores into the peers' memory + flags (no collective)",
                    "one all_gather": "one NCCL all_gather"}.get(enc.exchange, enc.exchange)
        eng = enc.b.eng
        eng.set_stream(stream.cuda_stream)

        def step():
            enc.encode_strip(img.data_ptr(), W * 3)

    if sampler:
        sampler.start()
    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step()
        barrier()
        if sampler:
            sampler.t_lo = time.time()
        launches0 = eng.launch_count()
        # the timed steps run without the library's per-stage CUDA events (8 event records cost ~20 us per image);
        # the stage times come from a separate, untimed pass below
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            out_ptr = step()
        e1.record(stream)
        barrier()
        ms_total = e0.elapsed_time(e1)
        launches = eng.launch_count() - launches0
        nbytes = eng.encode_finish()   # device-side checks of the last encode + its length (N>1: this rank's strip)
        last_jpeg = None   # host copy of the last timed step's JPEG, taken before any later step overwrites it
        if args.dump_outputs:
            if world == 1:
                last_jpeg = _view(out_ptr, (nbytes,), "|u1", dev).cpu().numpy()
            else:
                whole = enc.gather_jpeg(0)
                last_jpeg = whole.cpu().numpy() if rank == 0 else None
        eng.enable_timing(True)
        ks = args.steps if world == 1 else max(1, min(args.steps, 5))
        for _ in range(ks):
            step()
            eng.encode_finish()
            for k, v in eng.timings().items():
                stage_acc[k] = stage_acc.get(k, 0.0) + v * args.steps / ks
        eng.enable_timing(False)
        if world > 1:
            t = torch.tensor([ms_total], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_total = float(t.item())
            lens = enc.gather_lengths()
            nbytes = int(lens.sum())
            lt = torch.tensor([launches], device=dev, dtype=torch.int64)
            dist.all_reduce(lt)
            launches = int(lt.item())
    ms = ms_total / args.steps

    # ---- end to end through the C-ABI with pinned host buffers (N=1: b2j_encode; N>1: per-rank upload + strip encode
    #      + per-rank download of its strip's bytes)
    e2e = None
    k2 = max(3, min(args.steps, 10))
    h_img = torch.empty((nrows, W, 3), dtype=torch.uint8, pin_memory=True)
    h_img.copy_(img)
    h_out = torch.empty(int(nbytes) + (1 << 20), dtype=torch.uint8, pin_memory=True)
    torch.cuda.synchronize()
    if world == 1:
        def e2e_step():
            return eng.encode_ptr(h_img.data_ptr(), W * 3, W, H, h_out.data_ptr(), h_out.numel())
    else:
        def e2e_step():
            with torch.cuda.stream(stream):
                img.copy_(h_img, non_blocking=True)
                ol = enc.encode_strip(img.data_ptr(), W * 3)
                n = int(ol.item())
                h_out[:n].copy_(enc.b.out_view(n), non_blocking=True)
                stream.synchronize()
            return n
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(k2):
        n2 = e2e_step()
    barrier()
    dt = (time.perf_counter() - t0) / k2
    if world > 1:
        t = torch.tensor([dt], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    e2e = {"value": round(W * H / dt / 1e6, 1), "unit": "Mpix/s", "ms_per_step": round(dt * 1e3, 2),
           "h2d_bytes_per_step": W * H * 3, "d2h_bytes_per_step": int(nbytes),
           "api": "b2j_encode (host BGR -> host JPEG), pinned buffers" if world == 1 else
                  "per rank: pinned H2D of its strip + b2j_strip_phase1..3 + pinned D2H of its bytes"}
    # ---- the same call on PAGEABLE host memory (what the reference's cv::Mat / std::vector hand over): the library
    #      stages row groups through pinned buffers with its own copy threads (hostpipe.h)
    e2e_pageable = None
    if world == 1:
        try:
            p_img = np.array(h_img.numpy(), copy=True)
            p_out = np.empty(int(nbytes) + (1 << 20), np.uint8)
            p_out[:] = 0   # touch the pages: the timed calls measure the codec, not the kernel's page faults
            eng.encode(p_img, out=p_out)
            kp = 3
            t0 = time.perf_counter()
            for _ in range(kp):
                eng.encode(p_img, out=p_out)
            dtp = (time.perf_counter() - t0) / kp
            e2e_pageable = {"value": round(W * H / dtp / 1e6, 1), "unit": "Mpix/s", "ms_per_step": round(dtp * 1e3, 2),
                            "api": "b2j_encode (pageable host BGR -> pageable host JPEG)"}
            del p_img, p_out
        except Exception as e:
            e2e_pageable = {"error": f"{type(e).__name__}: {e}"}

    # ---- the metric's second half (BASELINE.json: "...; decode Mpix/s"): the JPEG just produced, host bytes ->
    #      device BGR (b2j_decode_device, includes the H2D of the scan) and host bytes -> pinned host BGR (b2j_decode)
    decode = None
    if world == 1:
        try:
            jpg = h_out[:int(n2)].numpy()
            d_rec = torch.empty((H, W, 3), dtype=torch.uint8, device=dev)
            kd = max(2, min(args.steps, 5))
            with torch.cuda.stream(stream):
                eng.decode_device(jpg, d_rec.data_ptr(), W * 3)
                eng.decode_finish()
                d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                d0.record(stream)
                for _ in range(kd):
                    eng.decode_device(jpg, d_rec.data_ptr(), W * 3)
                    eng.decode_finish()
                d1.record(stream)
                stream.synchronize()
            dec_ms = d0.elapsed_time(d1) / kd
            # the same with the JPEG bytes already in HBM when the timed region starts (b2j_decode_scan_device)
            from nvjpeg_imagecompressor_b200.strips import parse_baseline_header
            hd = parse_baseline_header(jpg)
            d_jpg = torch.from_numpy(jpg).to(dev)
            scan_len = hd["scan_end"] - hd["scan_off"]
            with torch.cuda.stream(stream):
                eng.decode_scan_device(jpg[:hd["scan_off"]], d_jpg.data_ptr() + hd["scan_off"], scan_len, d_rec.data_ptr(), W * 3)
                d0.record(stream)
                for _ in range(kd):
                    eng.decode_scan_device(jpg[:hd["scan_off"]], d_jpg.data_ptr() + hd["scan_off"], scan_len, d_rec.data_ptr(), W * 3)
                d1.record(stream)
                stream.synchronize()
            dec_res_ms = d0.elapsed_time(d1) / kd
            del d_jpg
            h_rec = torch.empty((H, W, 3), dtype=torch.uint8, pin_memory=True)
            eng.decode_ptr(jpg, h_rec.data_ptr(), W * 3)
            t0 = time.perf_counter()
            for _ in range(kd):
                eng.decode_ptr(jpg, h_rec.data_ptr(), W * 3)
            dth = (time.perf_counter() - t0) / kd
            eng.enable_timing(True)   # per-stage CUDA events inside the library: one extra, untimed decode
            with torch.cuda.stream(stream):
                eng.decode_device(jpg, d_rec.data_ptr(), W * 3)
                eng.decode_finish()
            dt_st = {k: round(v, 3) for k, v in eng.timings().items() if k.startswith("dec_")}
            eng.enable_timing(False)
            decode = {"metric": "decode_mpix_per_s", "value": round(W * H / dec_res_ms / 1e3, 1), "unit": "Mpix/s",
                      "ms_per_step": round(dec_res_ms, 3), "input": "this run's JPEG, bytes resident in HBM (b2j_decode_scan_device), output BGR in HBM",
                      "from_host_bytes": {"value": round(W * H / dec_ms / 1e3, 1), "unit": "Mpix/s", "ms_per_step": round(dec_ms, 3),
                                          "api": "b2j_decode_device + b2j_decode_finish (pinned host JPEG -> BGR in HBM, upload inside)"},
                      "e2e": {"value": round(W * H / dth / 1e6, 1), "unit": "Mpix/s", "ms_per_step": round(dth * 1e3, 2),
                              "h2d_bytes_per_step": int(n2), "d2h_bytes_per_step": W * H * 3,
                              "api": "b2j_decode (host JPEG -> host BGR), pinned output"},
                      "stages_ms": dt_st}
            del d_rec, h_rec
        except Exception as e:  # the encode line must survive a decode problem
            decode = {"error": f"{type(e).__name__}: {e}"}
    # ---- BASELINE.json's other configurations at size, one short leg each (N = 1): what the driver's own run records
    #      for them. Not the headline; every leg is device resident and timed with CUDA events on the stream.
    other = None
    if world == 1:
        other = {}
        import hashlib as _hl
        ko = max(2, min(args.steps, 5))

        def timed(fn, k=ko):
            with torch.cuda.stream(stream):
                fn()
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record(stream)
                for _ in range(k):
                    fn()
                a1.record(stream)
                stream.synchronize()
            return a0.elapsed_time(a1) / k
        try:   # config 1: the same image, 4:2:0 q95 standard Huffman tables; bytes against libjpeg-turbo's digest
            e1c = P.Engine(W, H, 95, False, "420", device=local_rank)
            e1c.set_stream(stream.cuda_stream)
            t1 = timed(lambda: e1c.encode_device(img.data_ptr(), W * 3, W, H))
            o1, _ = e1c.encode_device(img.data_ptr(), W * 3, W, H)
            n1 = e1c.encode_finish()
            from nvjpeg_imagecompressor_b200.strips import _view
            dg = _hl.sha256(_view(o1, (n1,), "|u1", dev).cpu().numpy().tobytes()).hexdigest()
            ok1 = None
            with open(os.path.join(ROOT, "tests", "golden", "golden.json")) as f:
                for c in json.load(f)["headline"]["encodes"]:
                    if (c["css"], c["quality"], c["optimize"]) == (3, 95, 0):
                        ok1 = bool(c["jpeg_len"] == n1 and dg[:32] == c["jpeg_sha256_128"])
            other["config1_420_q95_std_huffman"] = {"ms_per_step": round(t1, 3), "mpix_s": round(W * H / t1 / 1e3, 1), "jpeg_bytes": int(n1),
                                                    "bit_exact_vs_libjpeg_turbo": ok1}
            e1c.close()
        except Exception as e:
            other["config1_420_q95_std_huffman"] = {"error": f"{type(e).__name__}: {e}"}
        try:   # config 4: secondary compression round trip, device resident (b2j_secondary_device)
            t4 = timed(lambda: eng.secondary_device(img.data_ptr(), W * 3, W, H, 1))
            l1, l2, ps, _ = eng.secondary_finish()
            other["config4_secondary_round_trip"] = {"ms_per_step": round(t4, 3), "mpix_s": round(W * H / t4 / 1e3, 1), "jpeg1_bytes": int(l1),
                                                     "jpeg2_bytes": int(l2), "psnr_db": round(ps, 4),
                                                     "api": "b2j_secondary_device: encode -> reconstruct from the kept coefficients -> difference map + SSD -> encode(difference)"}
        except Exception as e:
            other["config4_secondary_round_trip"] = {"error": f"{type(e).__name__}: {e}"}
        try:   # config 5 (batch half): 1920x1080 images, 4:2:0 q95 optimised, 8 engines on 8 streams, 256 encodes + 256 decodes
            BW, BH, NB, NE = 1920, 1080, 256, 8
            bimgs = [synth_rows(BW, BH, 0, BH, sd, 8, dev) for sd in range(NE)]
            engs = [P.Engine(BW, BH, 95, True, "420", device=local_rank) for _ in range(NE)]
            sts = [torch.cuda.Stream(device=dev) for _ in range(NE)]
            for e_, s_ in zip(engs, sts):
                e_.set_stream(s_.cuda_stream)
            jp = []
            for e_, im in zip(engs, bimgs):
                jp.append(np.array(e_.encode(im.cpu().numpy()), copy=True))
            recs = [torch.empty((BH, BW, 3), dtype=torch.uint8, device=dev) for _ in range(NE)]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(NB):
                engs[i % NE].encode_device(bimgs[i % NE].data_ptr(), BW * 3, BW, BH)
            torch.cuda.synchronize()
            tb_e = time.perf_counter() - t0
            for e_, j_, r_ in zip(engs, jp, recs):
                e_.decode_device(j_, r_.data_ptr(), BW * 3); e_.decode_finish()
            t0 = time.perf_counter()
            for i in range(NB):
                engs[i % NE].decode_device(jp[i % NE], recs[i % NE].data_ptr(), BW * 3)
                if i >= NE - 1:
                    engs[(i + 1) % NE].decode_finish()
            for e_ in engs:
                e_.decode_finish()
            torch.cuda.synchronize()
            tb_d = time.perf_counter() - t0
            other["config5_batch_1080p"] = {"images": NB, "engines": NE, "encode_images_s": round(NB / tb_e, 1), "encode_mpix_s": round(NB * BW * BH / tb_e / 1e6, 1),
                                            "decode_images_s": round(NB / tb_d, 1), "decode_mpix_s": round(NB * BW * BH / tb_d / 1e6, 1),
                                            "note": "device-resident images / pinned JPEG bytes in, BGR in HBM out; wall clock over the batch, one host thread"}
            for e_ in engs:
                e_.close()
            del bimgs, recs
        except Exception as e:
            other["config5_batch_1080p"] = {"error": f"{type(e).__name__}: {e}"}
    if sampler:
        sampler.t_hi = time.time()
    clocks = sampler.finish() if sampler else None
    # the bytes themselves: one digest for every N (N>1: the strips' bytes concatenated on rank 0) -- same image, same stream
    import hashlib
    if world == 1:
        digest = hashlib.sha256(h_out[:int(n2)].numpy().tobytes()).hexdigest()
    else:
        with torch.cuda.stream(stream):
            whole = enc.gather_jpeg(0)
            stream.synchronize()
        digest = hashlib.sha256(whole.cpu().numpy().tobytes()).hexdigest() if rank == 0 else None
    if rank != 0:
        return None
    if last_jpeg is not None:
        dump_outputs(args.dump_outputs, last_jpeg)
    bit_exact = None
    try:   # libjpeg-turbo's digest of this very encode (tests/golden/make_golden.py, cv2.imencode in the build container)
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests", "golden", "golden.json")) as f:
            for c in json.load(f)["headline"]["encodes"]:
                if (c["css"], c["quality"], c["optimize"]) == ({"444": 0, "422": 1, "440": 2, "420": 3, "411": 4}[CSS], QUALITY, int(OPT)):
                    bit_exact = bool(c["jpeg_len"] == int(nbytes) and digest[:32] == c["jpeg_sha256_128"])
    except Exception:
        pass

    peak, which = measured_peak()
    line = {"metric": "encode_mpix_per_s", "value": round(W * H / ms / 1e3, 1), "unit": "Mpix/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 4), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": round(W * H / ms / 1e3 / PUBLISHED_MPIX_S, 2), "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks}
    # what the stream is (kept inside `e2e`, which the driver records whole; `config` is the workload alone so that
    # both arms carry the same one)
    e2e.update({"jpeg_bytes": int(nbytes), "jpeg_sha256": digest, "bit_exact_vs_libjpeg_turbo": bit_exact,
                "vs_baseline_basis": "BASELINE.md section 1: the reference README's 201.45 ms = 1652 Mpix/s for this configuration "
                                     "(8320x40000, 4:2:2, q95, optimised Huffman) on an RTX 3060, its own images",
                "l2": "inputs (998 MB image, ~0.8 GB token pool) exceed the 126 MB L2; no flush between steps",
                "parallelism": "single GPU" if world == 1 else
                f"{world} MCU-row strips; per image every strip shares a 4 KB record (symbol counts, edge DCs, first tokens) by {exchange}"})
    if world > 1 and stage_acc:
        st = {k: v / args.steps for k, v in stage_acc.items()}
        ksum = sum(st.get(k, 0.0) for k in ("fdct", "hist_edge", "tables", "pack", "scan", "stuff"))
        line["stages_ms_rank0"] = {k: round(st[k], 4) for k in ("fdct", "hist_edge", "tables", "pack", "scan", "stuff") if k in st}
        line["stages_ms_rank0"]["kernels"] = round(ksum, 4)
        line["stages_ms_rank0"]["collectives_and_gaps"] = round(ms - ksum, 4)
    if e2e_pageable is not None:
        line["e2e_pageable"] = e2e_pageable
    if decode is not None:
        line["decode"] = decode
        e2e["decode"] = decode   # inside a recorded object: the decode half of BASELINE.json's metric
    if other:
        line["other_configs"] = other
        e2e["other_configs"] = other
    if world == 1:
        from nvjpeg_imagecompressor_b200 import _native as NAT
        st = {k: v / args.steps for k, v in stage_acc.items()}
        # Algorithmic bytes per launch (DESIGN.md section 4): k_fdct reads every pixel once (3 B/px) and writes one
        # 4-byte run-length token per Huffman symbol; k_pack reads the tokens and writes the entropy bits; k_stuff reads
        # them and writes the stuffed bytes. Token count and byte count are read back from the encoder itself.
        ntok = int(eng.debug_read(NAT.DBG_TOKEN_COUNT, np.uint32)[0])
        algo = {"fdct": W * H * 3 + 4 * ntok, "pack": 4 * ntok + int(nbytes), "stuff": 2 * int(nbytes)}
        names = {"fdct": "k_fdct<2,1>", "pack": "k_pack", "stuff": "k_stuff"}
        top = max(("fdct", "pack", "stuff"), key=lambda k: st.get(k, 0))
        # roofline (BASELINE.md section 3 / SURVEY.md 8d): the path's algorithmic bytes are 3 B per pixel read + the JPEG bytes
        # written (3.445 B/px here); `achieved` = those bytes over the dominant kernel's launch duration (CUDA events on
        # the launching stream, recorded inside the library). `own_traffic_model` is that kernel's own minimal traffic
        # (it also writes the 4-byte tokens the second pass reads): that is what `traffic` (ncu DRAM bytes) must match.
        path_bytes = W * H * 3 + int(nbytes)
        ach = path_bytes / (st[top] * 1e-3) / 1e9
        traffic = None
        traffic_note = None
        try:   # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tj = json.load(f)
            if tj.get("source_digest") == kernel_source_digest():
                traffic = tj["kernels"].get(names[top], {}).get("dram_bytes")
            else:
                traffic_note = ("profiles/traffic.json was captured on other kernel sources (digest %s, this tree %s): not reported"
                                % (tj.get("source_digest"), kernel_source_digest()))
        except Exception:
            pass
        line["roofline"] = {"bound": "hbm", "kernel": names[top],
                            "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                            "traffic": traffic, "traffic_note": traffic_note, "peak_source": which,
                            "algorithmic_bytes_per_launch": int(path_bytes), "bytes_per_pixel": round(path_bytes / (W * H), 4),
                            "kernel_ms": round(st[top], 4), "tokens": ntok,
                            "kernel_timing": f"CUDA events around every kernel on the launching stream, averaged over a second pass of "
                                             f"{args.steps} steps right after the timed steps (the events cost ~20 us per image, so "
                                             f"the `value` steps run without them)",
                            "note": "k_fdct is bound by integer issue (ALU and FMA pipes ~65 % busy each, profiles/), not by HBM; "
                                    "its DRAM traffic equals its own minimal traffic (pixels read once + tokens written once)",
                            "own_traffic_model": {names[k]: {"ms": round(st[k], 4), "bytes": int(algo[k]),
                                                             "achieved_gbs": round(algo[k] / (st[k] * 1e-3) / 1e9, 1),
                                                             "frac": round(algo[k] / (st[k] * 1e-3) / 1e9 / peak, 4)}
                                                  for k in ("fdct", "pack", "stuff")},
                            "whole_encode": {"algorithmic_bytes": int(path_bytes),
                                             "achieved": round(path_bytes / (ms * 1e-3) / 1e9, 1),
                                             "frac": round(path_bytes / (ms * 1e-3) / 1e9 / peak, 4)}}
        line["stages_ms"] = {k: round(v, 4) for k, v in st.items() if k in ("fdct", "hist_edge", "tables", "pack", "scan", "stuff", "total")}
        line["roofline"]["stages_ms"] = line["stages_ms"]
        if decode and "ms_per_step" in decode:   # decode: JPEG bytes read once + 3 B per pixel written once
            line["roofline"]["decode"] = {"algorithmic_bytes": int(path_bytes), "ms": decode["ms_per_step"],
                                          "achieved": round(path_bytes / (decode["ms_per_step"] * 1e-3) / 1e9, 1),
                                          "frac": round(path_bytes / (decode["ms_per_step"] * 1e-3) / 1e9 / peak, 4),
                                          "stages_ms": decode.get("stages_ms")}
        try:
            line["cpu_baseline"] = cpu_baseline()
        except Exception as e:
            line["cpu_baseline"] = {"value": None, "unit": "Mpix/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-kind", default="auto", choices=["auto", "nvjpeg", "cpu"])
    ap.add_argument("--ref-progressive", type=int, default=0,
                    help="1 = nvJPEG progressive encoding as the reference ships it (ImageCompressorImpl.cu:28); default is "
                         "baseline sequential, the stream type this engine and the north-star target")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the JPEG of the last timed step to DIR as .npy arrays (--impl b200)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    args.warmup = max(3, args.warmup) if args.impl == "b200" else max(1, args.warmup)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        line = run_reference(args, rank, world)
        if line is not None:
            print(json.dumps(line), flush=True)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    line = run_b200(args, rank, world, local_rank)
    if line is not None:
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
