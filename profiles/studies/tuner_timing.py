"""Timing study of the tuner kernel (csrc/tuner.cu, DESIGN.md section 5.6).

Sweeps ntaps in {17, 65, 257} x D in {1, 2, 4, 8} over 512 MB of float32 IQ (more than the 126 MB L2, so every pass reads
HBM), timed with CUDA events over windows of at least 0.5 s after a warm-up.  Per point: input GS/s, achieved GB/s and
FLOP/s, and the share of the larger of the two bounds (HBM bytes / 7.7 TB/s, FP32 FLOPs / (SM count x 128 FMA/clk x 2 x SM
clock read in this run)).  Also the cost the tuner adds to one cfg2 batch (25 MS/s geometry, 1125 lines, 60 Hz, 10
decimator blocks = one frame) when a 100 MS/s capture is decimated by 4, and the card's name and power limit.

    python profiles/studies/tuner_timing.py [--out profiles/studies/tuner_timing_<tag>.json]
"""
from __future__ import annotations

import argparse
import json
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


def time_runs(tn, x, min_s=0.5):
    """Mean seconds per tuner run over the whole buffer, CUDA events, window >= min_s."""
    n = 1
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            tn.run(x, 0)
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
    fp32_peak = props.multi_processor_count * 128 * 2 * sm_max_mhz * 1e6          # FLOP/s at the card's top SM clock (read now)
    pairs = args.mbytes * (1 << 20) // 8
    x = torch.randn(2 * pairs, dtype=torch.float32, device="cuda")
    fs = 100_000_000
    points = []
    for ntaps in (17, 65, 257):
        for D in (1, 2, 4, 8):
            tn = ctx.tuner()
            tn.configure(fs, 12_500_000.0, fs // D if D > 1 else 40_000_000, D, ntaps)
            tn.run(x, 0); torch.cuda.synchronize()                                 # warm-up
            t = time_runs(tn, x)
            bytes_ = pairs * 8 + (pairs // D) * 8
            flops = pairs // D * ntaps * 4 + pairs * 6                             # 2 FMA per tap per output + one rotation (6 FLOP) per input
            t_hbm, t_fp = bytes_ / HBM_BPS, flops / fp32_peak
            bound = "HBM" if t_hbm >= t_fp else "FP32"
            points.append({"ntaps": ntaps, "D": D, "ms": t * 1e3, "gsps_in": pairs / t / 1e9, "gbps": bytes_ / t / 1e9,
                           "tflops": flops / t / 1e12, "bound": bound, "share_of_bound": max(t_hbm, t_fp) / t,
                           "default_filter": ntaps == 16 * D + 1 or (D == 1 and ntaps == 17)})
            print(json.dumps(points[-1]), flush=True)
            del tn
    # cfg2 after a 100 MS/s -> 25 MS/s tuner: one batch of 10 decimator blocks = one frame of 1/60 s at 25 MS/s = 4x input pairs
    tn = ctx.tuner()
    tn.configure(100_000_000, -20_000_000.0, 25_000_000, 4, 0)
    batch_pairs = 4 * 10 * int(0.1 * 25_000_000 / 60.0)
    xb = torch.randn(2 * batch_pairs, dtype=torch.float32, device="cuda")
    tn.run(xb, 0); torch.cuda.synchronize()
    t_batch = time_runs(tn, xb)
    clk = nvsmi("clocks.sm")
    sm_clock_mhz = float(clk) if clk.replace(".", "").isdigit() else float("nan")      # right after the timed windows
    res = {"gpu": props.name, "sm_count": props.multi_processor_count, "power_limit_w": nvsmi("power.limit"),
           "sm_clock_mhz_during_run": sm_clock_mhz, "sm_clock_max_mhz": sm_max_mhz,
           "fp32_bound_tflops": fp32_peak / 1e12, "hbm_bound_tbps": HBM_BPS / 1e12, "input_mbytes": args.mbytes,
           "points": points,
           "cfg2_batch": {"input_pairs": batch_pairs, "taps": len(tn.taps), "ms_per_batch": t_batch * 1e3,
                          "note": "tuner alone, 100 MS/s float32 -> D=4 -> cfg2's 25 MS/s geometry; one batch = 10 decimator blocks = 1 frame"}}
    print(json.dumps({k: v for k, v in res.items() if k != "points"}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
