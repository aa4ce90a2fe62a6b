"""Timing study of the channelizer and the scan (csrc/channelizer.cu, DESIGN.md section 5.7).

1. The channelizer alone at K in {8, 64, 256} x Q in {8, 16}, complex and magnitude output, over 512 MB of float32 IQ (more than
   the 126 MB L2, so every pass reads HBM), CUDA events over windows of at least 0.5 s after a warm-up.  Per point: input GS/s,
   and the share of the larger of two bounds per input pair: HBM (8 B in, 8 B of magnitudes or 16 B of pairs out, at 7.7 TB/s)
   and FP32 (8Q flops of FIR + 10 log2 K of FFT + 10 for magnitudes, at SM count x 128 FMA/clk x 2 x the SM clock read in this run).
2. The whole scan (channelizer, captures, batched autocorrelations, running means, scores) at fs = 100 MS/s, K in {8, 64}, fed in
   blocks of 4 Mi pairs; host clock around work that ends in the scan's synchronising results() call.
3. What a scan (K = 8) adds to a pipeline fed a 100 MS/s capture and tuned to cfg2's 25 MS/s geometry (1125 lines, 60 Hz): wall
   time per delivered frame with and without the scan, the two runs alternated twice.
The card's name, power limit and SM clock are read in the same run.

    python profiles/studies/scan_timing.py [--out profiles/studies/scan_timing_<tag>.json]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from tempestsdr_b200 import api, pipeline  # noqa: E402

HBM_BPS = 7.7e12


def nvsmi(q):
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # the numbers are still measured; the card description is then missing
        return f"unavailable ({e})"


def time_events(fn, min_s=0.5):
    """Mean seconds per fn() call, CUDA events, window >= min_s."""
    n = 1
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        b.synchronize()
        el = a.elapsed_time(b) / 1e3
        if el >= min_s:
            return el / n
        n = max(n * 2, int(n * min_s / max(el, 1e-6)) + 1)


def channelizer_points(ctx, x, pairs, fp32_peak, fs):
    points = []
    for K in (8, 64, 256):
        for Q in (8, 16):
            ch = ctx.channelizer()
            ch.configure(fs, K, Q)
            M = pairs // (K // 2) + 2
            for mag in (False, True):
                out = torch.empty(K * M * (1 if mag else 2), dtype=torch.float32, device="cuda")
                o, od = api.C.c_uint64(0), api.C.c_uint64(0)

                def run():
                    ch.reset()
                    ctx.chk(ctx._lib.tsdrgpu_channelizer_run(ch._h, ctx.stream, x.data_ptr(), pairs, 0, int(mag), out.data_ptr(), M,
                                                             api.C.byref(o), api.C.byref(od)))
                run(); torch.cuda.synchronize()                                        # warm-up
                t = time_events(run)
                bytes_ = pairs * (16 if mag else 24)
                flops = pairs * (8 * Q + 10 * math.log2(K) + (10 if mag else 0))
                t_hbm, t_fp = bytes_ / HBM_BPS, flops / fp32_peak
                points.append({"K": K, "Q": Q, "mode": "magnitude" if mag else "complex", "ms": t * 1e3, "gsps_in": pairs / t / 1e9,
                               "bound": "HBM" if t_hbm >= t_fp else "FP32", "bound_gsps": pairs / max(t_hbm, t_fp) / 1e9,
                               "share_of_bound": max(t_hbm, t_fp) / t})
                print(json.dumps(points[-1]), flush=True)
                del out
            del ch
    return points


def scan_points(ctx, x, pairs, fs):
    res = []
    block = 4 << 20
    for K in (8, 64):
        sc = ctx.scan()
        sc.configure(fs, K, 16)
        for k in range(0, pairs, block):                                           # warm-up: every shape once
            sc.run(x[2 * k:2 * min(k + block, pairs)], 0)
        sc.records()
        sc.reset()
        torch.cuda.synchronize()
        fed, t0 = 0, time.perf_counter()
        while True:                                                                # whole passes over the buffer, >= 0.5 s
            for k in range(0, pairs, block):
                sc.run(x[2 * k:2 * min(k + block, pairs)], 0)
            fed += pairs
            recs = sc.records()
            t = time.perf_counter() - t0
            if t >= 0.5:
                break
        res.append({"K": K, "Q": 16, "fs": fs, "input_pairs": fed, "rounds": int(recs[0].captures), "s": t, "gsps_in": fed / t / 1e9,
                    "channel_samples_per_s": 2 * fed / t})
        print(json.dumps(res[-1]), flush=True)
        del sc
    return res


def pipeline_cost(fs=100_000_000, K=8, secs=2.0):
    h, fv, items = 1125, 60.0, 1 << 22
    rng = np.random.default_rng(1)
    blocks = [(rng.standard_normal(items) * 0.3).astype(np.float32) for _ in range(4)]
    nblk = int(fs * secs * 2 // items)
    out = {}
    for rep in range(2):
        for scan in (False, True):
            frames = []
            p = pipeline.Pipeline(samplerate=fs, height=h, refreshrate=fv, batch_frames=1, block_when_busy=True,
                                  on_frame=lambda f, w, hh: frames.append(w))
            p.set_tuner(-20_000_000.0, 25_000_000, 4)
            if scan:
                p.set_scan(K)
            for k in range(8):                                                     # warm-up
                p.process(blocks[k % 4], 0)
            p.flush()
            n0 = len(frames)
            t0 = time.perf_counter()
            for k in range(nblk):
                p.process(blocks[k % 4], 0)
            p.flush()
            if scan:
                p.scan_results()                                                   # the scan's own stream has finished too
            t = time.perf_counter() - t0
            nf = len(frames) - n0
            out.setdefault("scan" if scan else "no_scan", []).append({"s": t, "frames": nf, "ms_per_frame": 1e3 * t / max(nf, 1)})
            p.close()
    mean = {k: float(np.mean([r["ms_per_frame"] for r in v])) for k, v in out.items()}
    return {"fs": fs, "K": K, "tuner": "-20 MHz, 25 MHz, D=4 (cfg2's 25 MS/s, 1125 lines, 60 Hz)", "runs": out,
            "ms_per_frame": mean, "added_ms_per_frame": mean["scan"] - mean["no_scan"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--mbytes", type=int, default=512)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the timing study needs the GPU"
    ctx = api.Context(0)
    props = torch.cuda.get_device_properties(0)
    sm_max_mhz = float(nvsmi("clocks.max.sm"))
    fp32_peak = props.multi_processor_count * 128 * 2 * sm_max_mhz * 1e6
    pairs = args.mbytes * (1 << 20) // 8
    x = torch.randn(2 * pairs, dtype=torch.float32, device="cuda")
    fs = 100_000_000
    points = channelizer_points(ctx, x, pairs, fp32_peak, fs)
    clk = nvsmi("clocks.sm")
    sm_clock_mhz = float(clk) if clk.replace(".", "").isdigit() else float("nan")      # right after the timed windows
    scans = scan_points(ctx, x, pairs, fs)
    del x
    torch.cuda.empty_cache()
    pl = pipeline_cost()
    print(json.dumps(pl), flush=True)
    res = {"gpu": props.name, "sm_count": props.multi_processor_count, "power_limit_w": nvsmi("power.limit"),
           "sm_clock_mhz_during_run": sm_clock_mhz, "sm_clock_max_mhz": sm_max_mhz,
           "fp32_bound_tflops": fp32_peak / 1e12, "hbm_bound_tbps": HBM_BPS / 1e12, "input_mbytes": args.mbytes,
           "channelizer": points, "scan": scans, "pipeline_cfg2_100MSps": pl}
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
