"""Timing study of the notch filter and the power spectrum (csrc/notch.cu, DESIGN.md section 5.8).

Notch: L in {1025, 4097, 8193} over 512 MB of float32 IQ (more than the 126 MB L2, so every pass reads HBM), timed with CUDA
events over windows of at least 0.5 s after a warm-up.  Spectrum: nfft 4096 over the same buffer.  Per point: input GS/s and the
share of the larger of two bounds, HBM bytes / 7.7 TB/s (8 N / hop bytes in and 8 out per pair for the notch, 8 N / hop in
per pair for the spectrum, 16 at its hop of N / 2) and FP32 FLOPs / (SM count x 128 FMA/clk x 2 x the SM clock read in this run) (2 x 5 N log2 N / hop per pair plus the
spectral product, 6 N / hop).  Also the notch's cost per cfg2 frame (1/60 s of a 100 MS/s capture, 4 notches, the tuner at D = 4
behind it), and the card's name, power limit and SM clock.

    python profiles/studies/notch_timing.py [--out profiles/studies/notch_timing_<tag>.json]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from tempestsdr_b200 import api  # noqa: E402

HBM_BPS = 7.7e12


def nvsmi(q):
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # the numbers are still measured; the card description is then missing
        return f"unavailable ({e})"


def time_runs(fn, min_s=0.5):
    """Mean seconds per call of fn, CUDA events, window >= min_s."""
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--mbytes", type=int, default=512)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the timing study needs the GPU"
    ctx = api.Context(0)
    props = torch.cuda.get_device_properties(0)
    sm_max_mhz = float(nvsmi("clocks.max.sm"))
    pairs = args.mbytes * (1 << 20) // 8
    x = torch.randn(2 * pairs, dtype=torch.float32, device="cuda")
    fs = 100_000_000
    rows = []
    for L in (1025, 4097, 8193):
        nt = ctx.notch()
        nt.configure(fs, [-31e6, -5e6, 12e6, 40e6], [3e6, 1e6, 2e6, 4e6], L)
        N = nt.nfft
        hop = N - (L - 1)
        out = torch.empty_like(x)
        run = lambda: ctx._lib.tsdrgpu_notch_run(nt._h, ctx.stream, x.data_ptr(), pairs, 0, out.data_ptr(), None, None)
        run(); torch.cuda.synchronize()                                              # warm-up
        t = time_runs(run)
        rows.append({"stage": "notch", "L": L, "N": N, "hop": hop, "ms": t * 1e3, "gsps_in": pairs / t / 1e9,
                     "bytes_per_pair": 8 * N / hop + 8, "flops_per_pair": (10 * N * math.log2(N) + 6 * N) / hop})
        del nt, out
    sp = ctx.spectrum()
    sp.configure(fs, 4096)
    run = lambda: sp.run(x, 0)
    run(); torch.cuda.synchronize()
    t = time_runs(run)
    rows.append({"stage": "spectrum", "nfft": 4096, "ms": t * 1e3, "gsps_in": pairs / t / 1e9,
                 "bytes_per_pair": 8.0 * 4096 / 2048, "flops_per_pair": (10 * 4096 * 12 + 6 * 4096) / 2048})
    # cfg2 after the notch: one frame (1/60 s) of a 100 MS/s capture through 4 notches (default L), the tuner at D = 4 behind it
    nt = ctx.notch()
    nt.configure(fs, [-7e6, -2e6, 3e6, 9e6], [400e3, 200e3, 300e3, 600e3], 0)
    frame_pairs = int(fs / 60.0)
    xf = torch.randn(2 * frame_pairs, dtype=torch.float32, device="cuda")
    outf = torch.empty_like(xf)
    runf = lambda: ctx._lib.tsdrgpu_notch_run(nt._h, ctx.stream, xf.data_ptr(), frame_pairs, 0, outf.data_ptr(), None, None)
    runf(); torch.cuda.synchronize()
    t_frame = time_runs(runf)
    clk = nvsmi("clocks.sm")
    sm_clock_mhz = float(clk) if clk.replace(".", "").isdigit() else float("nan")      # right after the timed windows
    fp32_peak = props.multi_processor_count * 128 * 2 * (sm_clock_mhz if sm_clock_mhz == sm_clock_mhz else sm_max_mhz) * 1e6
    for r in rows:
        t_hbm, t_fp = r["bytes_per_pair"] / HBM_BPS, r["flops_per_pair"] / fp32_peak       # seconds per pair at each bound
        r["bound"] = "HBM" if t_hbm >= t_fp else "FP32"
        r["share_of_bound"] = max(t_hbm, t_fp) * r["gsps_in"] * 1e9
        print(json.dumps(r), flush=True)
    res = {"gpu": props.name, "sm_count": props.multi_processor_count, "power_limit_w": nvsmi("power.limit"),
           "sm_clock_mhz_during_run": sm_clock_mhz, "sm_clock_max_mhz": sm_max_mhz,
           "fp32_bound_tflops": fp32_peak / 1e12, "hbm_bound_tbps": HBM_BPS / 1e12, "input_mbytes": args.mbytes,
           "points": rows,
           "cfg2_frame": {"input_pairs": frame_pairs, "taps": int(nt.taps().size), "nfft": nt.nfft, "ms_per_frame": t_frame * 1e3,
                          "note": "notch stage alone on one frame (1/60 s) of a 100 MS/s float32 capture, 4 notches, default L; "
                                  "it runs on the ingest stream ahead of the tuner (D = 4 to cfg2's 25 MS/s)"}}
    print(json.dumps({k: v for k, v in res.items() if k != "points"}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
