#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config, one JSON line on stdout (rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Workload (config.workload): BASELINE configs[1] -- 1080p60 geometry (1125 total lines, the GUI's convention;
W = 740), 25 MS/s float32 IQ.  One BATCH = 64 frames' worth of synthetic IQ (640 decimator blocks of 41666 pairs = 26.7 M
pairs = 213 MB, larger than L2) through the whole hot path:
    fused demod+resample -> pixel stream -> frame stage (auto-gain, temporal IIR, collapse, sync search, re-centre)
    and, beside it (on the detector's own stream), the frame-rate detector: every capture of 3.1*fs/55 samples is
    autocorrelated (2^20-point FFT + IFFT at half size) and accumulated into the two lag plots.
One STEP = 80 batches (~57 ms of device time), so that the default 20 steps time more than a second.
`value`   MS/s with the IQ already resident in HBM (CUDA events around exactly K steps, max over ranks).
`e2e`     the same metric through the reference-facing API end to end: this repo's libTSDRLibrary.so driven by the reference's
          UNMODIFIED RawFile plugin through tsdr_init / tsdr_loadplugin / tsdr_readasync (pageable 2 MiB blocks, pacing off),
          H2D of every block and D2H of every finished frame inside the timed region, frames counted in the host's callback --
          the way the reference arm is measured.  `e2e.pinned_process` beside it: tsdrgpu_pipeline_process_raw_async() on
          page-locked host IQ (a front end that owns page-locked buffers), `e2e_int8_transport`: the same with 8-bit samples.
N > 1     N independent streams, one per GPU (the path has no cross-stream exchange: replicas, weak scaling).
--dump-outputs DIR  after the timed steps, rank 0 writes what the last of them handed out, so that two builds can be compared
          output for output (the inputs are seeded): DIR/frames.npy, the last frames of the last batch (float32, at most
          48 MB of them, one row per frame), and DIR/frame_plot.npy, DIR/line_plot.npy, the frame-rate detector's two lag
          plots (float64).
--impl reference   the reference's own threaded CPU pipeline (oracle/_ref: libTSDRLibrary.so + its RawFile plugin
          with pacing off) on this box's host cores, same geometry; falls back to the pinned C port when the
          reference binary is absent.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# The headline workload is BASELINE configs[1] ("cfg2" in SURVEY section 8).  BENCH_SHAPE=cfg5 / cfg1 re-runs the device-resident
# step on configs[4]'s per-GPU shape (50 MS/s, 1481x1125) or configs[0]'s (8 MS/s, 507x525): child processes of the default N=1 run,
# reported under "other_shapes", never as the headline.
SHAPES = {"cfg2": (25_000_000, 1125, 2576), "cfg5": (50_000_000, 1125, 2576), "cfg1": (8_000_000, 525, 800)}
SHAPE = os.environ.get("BENCH_SHAPE", "cfg2")
FS, HEIGHT, RASTER_W = SHAPES[SHAPE]
FV = 60.0
FRAMES_PER_BATCH = 256 if SHAPE == "cfg1" else 64         # frames per launch group (one pass over the resident 213 MB of IQ; cfg1's small frames: 256 -> 273 MB, still > L2)
BATCHES_PER_STEP = int(os.environ.get("BENCH_BATCHES_PER_STEP", "80"))   # one step = 80 such passes = 5120 frames = 2.13 G IQ pairs (~57 ms): 20 steps time > 1 s
FRAMES_PER_STEP = FRAMES_PER_BATCH * BATCHES_PER_STEP
METRIC = "IQ MS/s ingested -> 1080p60 frames (demod+resample+frame stage+autocorrelation), whole job"


def geometry():
    """set_internal_samplerate's width (TSDRLibrary.c:540-550), restated in Python so that the reference arm loads none of
    this repo's native code."""
    return int(2 * (FS / (FV * HEIGHT)))


def make_iq(pairs: int, seed: int) -> np.ndarray:
    """Video-like synthetic IQ, generated for one frame period and tiled (cheap, deterministic)."""
    from tempestsdr_b200 import synth
    per_frame = int(FS / FV)
    base = synth.video_like_iq(4 * per_frame, FS, RASTER_W, HEIGHT, FV, seed=seed, snr_db=25.0)
    reps = (2 * pairs + base.size - 1) // base.size
    return np.ascontiguousarray(np.tile(base, reps)[: 2 * pairs])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        """index: one GPU index, or a comma-separated list (then `per_gpu` in the result tells the GPUs apart)."""
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile(prefix="clocks_", suffix=".csv", delete=False)
            self.path = f.name
            q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, per = [], [], set(), {}
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                sm.append(float(p[1])); mx.append(float(p[2]))
                per.setdefault(p[0], []).append(float(p[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
            if len(per) > 1:
                out["per_gpu"] = {k: statistics.median(v) for k, v in sorted(per.items())}
        return out


# --------------------------------------------------------------------------------------------------- our arm
class DeviceStep:
    """One step of the hot path with the IQ resident in HBM."""

    def __init__(self, gpu, iq_dev, w):
        import torch
        from tempestsdr_b200.api import FrameRateDetector, PostProcessFlags
        self.torch, self.gpu, self.iq, self.w = torch, gpu, iq_dev, w
        self.block = int(0.1 * FS / FV)
        self.nblocks = FRAMES_PER_BATCH * 10
        self.n = w * HEIGHT
        self.up = w * HEIGHT * FV
        self.rs = gpu.resampler()
        self.pp = gpu.post_processor()
        self.pp.set_overlap(not os.environ.get("BENCH_NO_OVERLAP"))   # sync search + re-centring of batch k under the kernels of batch k+1
        self.frd = gpu.framerate_detector()
        self.flags = PostProcessFlags(autoshift=True, lowpass_before_sync=True)     # the GUI's defaults
        self.cap = FrameRateDetector.capture_size(FS)
        max_pix = int(self.rs.plan((self.block, self.nblocks), self.up, float(FS))) + 1024
        self.pix = torch.empty(max_pix + self.n + 1024, dtype=torch.float32, device=iq_dev.device)
        self.pix_fill = 0
        self.frames_out = [torch.empty((FRAMES_PER_BATCH + 2) * self.n, dtype=torch.float32, device=iq_dev.device) for _ in range(2)]
        self.pairs = self.block * self.nblocks
        # demodulated stream, capture-aligned; two buffers: the transforms of step k (on the detector's own stream) read one
        # while the resampler of step k+1 already fills the other
        self.frd_overlap = not os.environ.get("BENCH_NO_FRD_OVERLAP")
        self.frd.set_overlap(self.frd_overlap)
        self.mags = [torch.empty(self.cap + self.pairs, dtype=torch.float32, device=iq_dev.device) for _ in range(2 if self.frd_overlap else 1)]
        self.mag_sel = 0
        self.mag = self.mags[0]
        self.mag_fill = 0
        self.frames = 0
        self.last_frames = 0                                # frames the last batch wrote to frames_out[(k - 1) & 1]
        self.captures = 0
        self.k = 0
        self.chunk = int(os.environ.get("BENCH_FRAME_CHUNK", "0"))
        self.l2_frames = int(os.environ.get("BENCH_L2_FRAMES", "0"))

    def __call__(self):
        gpu = self.gpu
        # samples -> pixels (fused demod + resample), appended behind the pixels left over from the last step
        # (the same pass also leaves the magnitudes for the frame-rate detector: one demodulation feeds both consumers,
        # as am_demod does in the reference's process(), TSDRLibrary.c:286-292)
        fused_mag = not os.environ.get("BENCH_SEPARATE_DEMOD")
        # The batch goes through resampler + frame stage in sub-batches of `self.l2_frames` frames (BENCH_L2_FRAMES; default: the
        # whole batch at once): with sub-batches of 16 frames the pixels a resampler launch writes (53 MB), the frames the frame
        # stage hands from kernel to kernel and its output stay inside the 126 MB L2 from one kernel to the next, and the same
        # pixel buffer is written again before most of it was ever evicted.  This is what tsdrgpu_pipeline_* does with
        # batch_frames = 16 (the e2e path); here it is a knob of the device-resident step.
        cf = self.l2_frames if self.l2_frames > 0 else FRAMES_PER_BATCH
        fo = self.frames_out[self.k & 1]
        done = 0
        for b0 in range(0, self.nblocks, 10 * cf):
            nb = min(10 * cf, self.nblocks - b0)
            out = self.rs.process(self.iq[2 * self.block * b0: 2 * self.block * (b0 + nb)], (self.block, nb), self.up, float(FS), in_is_iq=True,
                                  out=self.pix[self.pix_fill:], mag_out=self.mag[self.mag_fill + self.block * b0:] if fused_mag else None)
            self.pix_fill += out.numel()
            nf = min(self.pix_fill // self.n, FRAMES_PER_BATCH + 1 - done)
            chunk = self.chunk if self.chunk > 0 else nf
            for c0 in range(0, nf, chunk):
                c1 = min(nf, c0 + chunk)
                self.pp.process(self.pix[c0 * self.n: c1 * self.n], self.w, HEIGHT, 0.0, 0.1, self.flags, out=fo[(done + c0) * self.n: (done + c1) * self.n], want_results=False)
            left = self.pix_fill - nf * self.n
            if left and nf:                                                      # left << nf*n: the ranges do not overlap
                gpu.chk(gpu._lib.tsdrgpu_memcpy_d2d(gpu._h, gpu.stream, self.pix.data_ptr(), self.pix.data_ptr() + 4 * nf * self.n, 4 * left))
            self.pix_fill = left
            done += nf
        self.k += 1
        self.frames += done
        self.last_frames = done
        # frame-rate detector: the whole stream is demodulated once; every complete capture of 3.1*fs/55 samples is
        # autocorrelated (batched FFTs) and accumulated in order
        if not fused_mag:
            gpu.chk(gpu._lib.tsdrgpu_am_demod(gpu._h, gpu.stream, self.iq.data_ptr(), self.pairs, self.mag.data_ptr() + 4 * self.mag_fill))
        self.mag_fill += self.pairs
        ncap = self.mag_fill // self.cap
        if ncap:
            rest = self.mag_fill - ncap * self.cap
            if self.frd_overlap:
                # the samples behind the last complete capture move to the head of the OTHER buffer (once the transforms that
                # last read it are done: they had a whole step), then this buffer's captures go to the detector's stream
                other = self.mags[self.mag_sel ^ 1]
                self.frd.join()
                if rest:
                    gpu.chk(gpu._lib.tsdrgpu_memcpy_d2d(gpu._h, gpu.stream, other.data_ptr(), self.mag.data_ptr() + 4 * ncap * self.cap, 4 * rest))
                self.frd.run_batch(FS, self.mag, self.cap, ncap, self.cap)
                self.mag_sel ^= 1
                self.mag = other
            else:
                self.frd.run_batch(FS, self.mag, self.cap, ncap, self.cap)
                if rest:
                    gpu.chk(gpu._lib.tsdrgpu_memcpy_d2d(gpu._h, gpu.stream, self.mag.data_ptr(), self.mag.data_ptr() + 4 * ncap * self.cap, 4 * rest))
            self.mag_fill = rest
            self.captures += ncap

    def join(self):
        self.pp.join()
        self.frd.join()

    def dump_outputs(self, path):
        """The frames of the last batch (the last ones, at most 48 MB) and the detector's lag plots as .npy files; call after join()."""
        os.makedirs(path, exist_ok=True)
        keep = max(1, min(self.last_frames, (48 << 20) // (4 * self.n)))
        frames = self.frames_out[(self.k - 1) & 1][(self.last_frames - keep) * self.n: self.last_frames * self.n]
        np.save(os.path.join(path, "frames.npy"), frames.view(keep, self.n).cpu().numpy())
        (_, frame_plot), (_, line_plot) = self.frd.plots(FS)
        np.save(os.path.join(path, "frame_plot.npy"), frame_plot)
        np.save(os.path.join(path, "line_plot.npy"), line_plot)


def collect_profile(gpu):
    names = C.create_string_buffer(48 * 48)
    tot = (C.c_double * 48)(); cnt = (C.c_uint64 * 48)(); n = C.c_int(0)
    gpu.chk(gpu._lib.tsdrgpu_profile_collect(gpu._h, names, tot, cnt, 48, C.byref(n)))
    out = {}
    for i in range(n.value):
        nm = names.raw[48 * i: 48 * (i + 1)].split(b"\0")[0].decode()
        out[nm] = (tot[i], cnt[i])
    return out


def cpu_baseline(w, seconds_budget=25.0):
    """The same work as one GPU step on ONE host core: the compiled reference's stage functions driven serially
    (oracle/_ref when present, else the pinned C port).  Bounded sample: 8 frames of IQ + 2 autocorrelation captures."""
    from oracle import oracle as orc
    O = orc.best()
    block = int(0.1 * FS / FV)
    nframes = 8
    pairs = block * 10 * nframes
    iq = make_iq(pairs, seed=77)
    cap = int(3.1 * FS / 55.0)
    t0 = time.perf_counter()
    mag = O.am_demod(iq)
    rs = O.resampler()
    pix = np.concatenate([rs.run(mag[k * block:(k + 1) * block], w * HEIGHT * FV, float(FS)) for k in range(10 * nframes)])
    pp = O.postprocessor(FS, HEIGHT, FV, 1, 0)
    n = w * HEIGHT
    for k in range(pix.size // n):
        pp.run(pix[k * n:(k + 1) * n], w, HEIGHT, 0.0, 0.1, 1, 0)
    t_stream = time.perf_counter() - t0
    det = O.framerate_detector()
    ncap = 2
    capdata = np.tile(mag, (ncap * cap + mag.size - 1) // mag.size)[: ncap * cap]
    t1 = time.perf_counter()
    for c in range(ncap):
        det.run(FS, capdata[c * cap:(c + 1) * cap])
    t_cap = (time.perf_counter() - t1) / ncap
    # one GPU step does pairs_step samples of the stream path and pairs_step/cap captures
    per_sample = t_stream / pairs + t_cap / cap
    return {"value": 1e-6 / per_sample, "unit": "MS/s", "cores": 1, "kind": "reference" if O.kind == "reference" else "port",
            "sample": f"{nframes} frames ({pairs} IQ pairs) through demod+resample+frame stage: {t_stream:.2f} s; "
                      f"{ncap} captures of {cap} samples autocorrelated: {t_cap:.2f} s each; stages driven serially on one thread"}


def _load_tsdr(path):
    lib = C.CDLL(path)
    lib.tsdr_init.argtypes = [C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p, C.c_void_p]
    lib.tsdr_setresolution.argtypes = [C.c_void_p, C.c_int, C.c_double]
    lib.tsdr_motionblur.argtypes = [C.c_void_p, C.c_float]
    lib.tsdr_setgain.argtypes = [C.c_void_p, C.c_float]
    lib.tsdr_setparameter_int.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
    lib.tsdr_loadplugin.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
    lib.tsdr_readasync.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.tsdr_stop.argtypes = [C.c_void_p]
    lib.tsdr_free.argtypes = [C.POINTER(C.c_void_p)]
    lib.tsdr_getlasterrortext.argtypes = [C.c_void_p]
    lib.tsdr_getlasterrortext.restype = C.c_char_p
    return lib


def e2e_through_tsdr_api(local: int, rank: int, w: int, seconds: float, barrier):
    """The drop-in boundary end to end, measured the way the reference arm is measured: this repo's libTSDRLibrary.so driven
    through tsdr_init / tsdr_loadplugin / tsdr_readasync with an UNMODIFIED front-end plugin -- the reference's own
    TSDRPlugin_RawFile (pacing off: its PERFORMANCE_BENCHMARK switch) reading float32 IQ from a file and calling process() with
    its pageable 2 MiB malloc'd buffer -- and counting the frames the frame callback receives.  The plugin binary is a data
    source, not an oracle; when it did not travel with the snapshot this repo's own file plugin plays the same role (host
    conversion, float callback, no raw sink)."""
    FRAME_CB = C.CFUNCTYPE(None, C.POINTER(C.c_float), C.c_int, C.c_int, C.c_void_p)
    VALUE_CB = C.CFUNCTYPE(None, C.c_int, C.c_double, C.c_double, C.c_void_p)
    PLOT_CB = C.CFUNCTYPE(None, C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_uint32, C.c_void_p)
    ref_plugin = os.path.join(ROOT, "oracle", "_ref", "libTSDRPlugin_RawFile_nopace.so")
    own_plugin = os.path.join(ROOT, "tempestsdr_b200", "lib", "TSDRPlugin_RawFileGPU.so")
    per_frame = int(FS / FV)
    shm = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    tmp = tempfile.NamedTemporaryFile(prefix=f"tsdr_iq_r{rank}_", suffix=".raw", delete=False, dir=shm)
    make_iq(16 * per_frame, seed=1000 + rank).tofile(tmp); tmp.close()
    os.environ["TSDR_CUDA_DEVICE"] = str(local); os.environ["TSDR_BATCH_FRAMES"] = "16"; os.environ["TSDR_NO_DROP"] = "1"
    stats_file = tmp.name + ".stats"
    os.environ["TSDR_STATS_FILE"] = stats_file      # the library's own clock around its data callback: plugin time vs. library time per block
    if os.path.exists(ref_plugin):
        plugin, params, which = ref_plugin, f'"{tmp.name}" {FS} float', "reference TSDRPlugin_RawFile (unmodified source, pacing switch off)"
    else:
        os.environ["TSDR_NO_RAW_SINK"] = "1"
        plugin, params, which = own_plugin, f'"{tmp.name}" {FS} float nopace', "this repo's TSDRPlugin_RawFileGPU in plain ten-symbol mode (reference plugin binary absent)"
    lib = _load_tsdr(os.path.join(ROOT, "tempestsdr_b200", "lib", "libTSDRLibrary.so"))
    count = {"frames": 0, "w": 0, "h": 0}

    def on_frame(buf, ww, hh, ctx):
        count["frames"] += 1; count["w"] = ww; count["h"] = hh
    fcb, vcb, pcb = FRAME_CB(on_frame), VALUE_CB(lambda *a: None), PLOT_CB(lambda *a: None)
    t = C.c_void_p()
    lib.tsdr_init(C.byref(t), C.cast(vcb, C.c_void_p), C.cast(pcb, C.c_void_p), None)
    lib.tsdr_setresolution(t, HEIGHT, FV); lib.tsdr_motionblur(t, 0.0); lib.tsdr_setgain(t, 0.5)
    for pid, v in ((0, 1), (1, 0), (6, 1)):          # AUTOSHIFT=1, PLL=0, LOW_PASS_BEFORE_SYNC=1: the reference arm's settings
        lib.tsdr_setparameter_int(t, pid, v)
    out = {"unavailable": None}
    barriers = 0
    try:
        rc = lib.tsdr_loadplugin(t, plugin.encode(), params.encode())
        if rc != 0:
            raise RuntimeError(f"tsdr_loadplugin rc={rc}: {lib.tsdr_getlasterrortext(t)}")
        rcs = []
        th = threading.Thread(target=lambda: rcs.append(lib.tsdr_readasync(t, C.cast(fcb, C.c_void_p), None)), daemon=True)
        th.start()
        deadline = time.perf_counter() + 30.0
        while count["frames"] < 64 and th.is_alive() and time.perf_counter() < deadline:     # warm-up: buffers grow, plugin buffer gets registered
            time.sleep(0.02)
        if not th.is_alive() or count["frames"] < 64:
            raise RuntimeError(f"no frames from tsdr_readasync (rc={rcs}): {lib.tsdr_getlasterrortext(t)}")
        barrier(); barriers += 1
        f0, t0, m0 = count["frames"], time.perf_counter(), time.monotonic()
        time.sleep(seconds)
        f1, t1, m1 = count["frames"], time.perf_counter(), time.monotonic()
        barrier(); barriers += 1
        lib.tsdr_stop(t)
        th.join(timeout=30)
        fps = (f1 - f0) / (t1 - t0)
        out = {"value_per_rank": fps * per_frame / 1e6, "frames_per_s": fps, "seconds": t1 - t0, "frames_delivered": f1 - f0,
               "frame": [count["w"], count["h"]], "plugin": which, "readasync_rc": rcs[0] if rcs else None,
               "h2d_bytes_per_frame": 8 * per_frame, "d2h_bytes_per_frame": 4 * count["w"] * count["h"]}
        try:
            st = json.load(open(stats_file))
            log = [e for e in st.get("log", []) if m0 <= e[0] <= m1]           # cumulative samples inside the timed window (CLOCK_MONOTONIC)
            if len(log) >= 2:
                n = max(1, log[-1][3] - log[0][3]); ins = log[-1][1] - log[0][1]; outs = log[-1][2] - log[0][2]; scope = "timed window"
            else:
                n = max(1, st["callbacks"]); ins = st["inside_callback_s"]; outs = st["between_callbacks_s"]; scope = "whole run, warm-up included"
            out["plugin_thread_per_block_us"] = {"inside_the_library_callback": 1e6 * ins / n, "in_the_plugin_between_callbacks": 1e6 * outs / n, "blocks": int(n),
                                                 "note": "the plugin's one thread alternates fread + memcpy of a 2 MiB block (its own code) with the callback "
                                                         "(this library: H2D of the block, waited for, + enqueueing the kernels); " + scope}
        except Exception:
            pass
    except Exception as e:
        out = {"unavailable": repr(e)[:300]}
    finally:
        while barriers < 2:                               # a rank whose run failed still meets the others at both barriers
            barrier(); barriers += 1
        try:
            lib.tsdr_free(C.byref(t))
        except Exception:
            pass
        os.unlink(tmp.name)
        if os.path.exists(stats_file):
            os.unlink(stats_file)
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from tempestsdr_b200 import api, pipeline

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"            # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line
    torch.cuda.set_device(local)
    gpu = api.Context(local)
    # this rank's threads and page-locked buffers on the socket its GPU hangs off (8 ranks on a two-socket box)
    numa_node = gpu._lib.tsdrgpu_device_numa_node(gpu._h)
    numa_bound = gpu._lib.tsdrgpu_bind_thread_near_device(gpu._h) == 0
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    w = geometry()
    block = int(0.1 * FS / FV)
    pairs = block * 10 * FRAMES_PER_BATCH                 # IQ pairs per batch (one pass over the resident buffer)
    pairs_step = pairs * BATCHES_PER_STEP
    iq_host = make_iq(pairs, seed=1000 + rank)
    iq_pinned = torch.from_numpy(iq_host).pin_memory()
    iq_dev = iq_pinned.cuda(non_blocking=True)
    # The pixel path is the critical chain of a batch (resampler -> auto-gain -> IIR -> collapse, then the sync search on the frame
    # stage's own high-priority stream); the frame-rate detector's transforms are background work on a lowest-priority stream.
    # BENCH_MAIN_STREAM_PRIO=<n> runs the step on a torch stream of that priority instead of the default stream (study knob).
    if os.environ.get("BENCH_MAIN_STREAM_PRIO"):
        torch.cuda.synchronize()                         # the resident IQ was copied on the default stream
        torch.cuda.set_stream(torch.cuda.Stream(priority=int(os.environ["BENCH_MAIN_STREAM_PRIO"])))
    batch = DeviceStep(gpu, iq_dev, w)

    def step():
        for _ in range(BATCHES_PER_STEP):
            batch()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cpu_group = None
    if world > 1:
        try:
            cpu_group = dist.new_group(backend="gloo")    # a barrier that parks the ranks on the HOST (no kernel on any GPU)
        except Exception:
            cpu_group = None

    def host_barrier():
        torch.cuda.synchronize()
        if world > 1:
            if cpu_group is not None:
                dist.barrier(group=cpu_group)
            else:
                dist.barrier()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    launches0 = gpu.launches
    frames0, caps0 = batch.frames, batch.captures
    sampler = ClockSampler(local)
    sampler_all = ClockSampler(",".join(str(i) for i in range(world))) if world > 1 else None     # every GPU of the job, informational
    if rank == 0:
        sampler.start()
        if sampler_all:
            sampler_all.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    t_host0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / (args.steps * BATCHES_PER_STEP)   # host time to ENQUEUE one batch (throttled by the 4-slot descriptor ring)
    batch.join()                                  # the side stream's tail (last sync search + re-centring) is inside the timed region
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and sampler_all:
        allg = sampler_all.stop()
        if allg.get("sm_mhz") is not None:
            clocks["all_gpus"] = allg                 # the headline keys above stay rank 0's GPU, as at N = 1
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = ms.item()
    launches = gpu.launches - launches0
    frames_done, caps_done = batch.frames - frames0, batch.captures - caps0
    value = world * args.steps * pairs_step / (ms_total * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:
        batch.dump_outputs(args.dump_outputs)

    if os.environ.get("BENCH_QUICK"):                 # used under ncu and for the opt-in variants: the timed steps only
        if rank == 0:
            q = {"quick": True, "value": value, "unit": "MS/s", "ms_per_step": ms_total / args.steps, "ms_per_batch": ms_total / (args.steps * BATCHES_PER_STEP),
                 "shape": SHAPE, "samplerate": FS, "frame": [w, HEIGHT], "frames_per_s": frames_done / (ms_total * 1e-3),
                 "captures_per_batch": caps_done / (args.steps * BATCHES_PER_STEP)}
            if os.environ.get("BENCH_SHAPE_CPU"):
                q["cpu_baseline"] = cpu_baseline(w)
            emit(q)
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- per-kernel timing pass (separate from the timed region above): CUDA events on the launching stream.
    # The side stream is switched off for this pass so that every kernel's event pair measures that kernel alone
    # (with it on, intervals on the main stream also contain the slowdown from sharing the chip with the sync search).
    batch.join(); torch.cuda.synchronize()
    batch.pp.set_overlap(False)
    batch.frd.set_overlap(False)                          # (the two-buffer bookkeeping of DeviceStep stays; the runs are just not forked)
    gpu.chk(gpu._lib.tsdrgpu_profile_enable(gpu._h, 1))
    collect_profile(gpu)
    prof_batches = 3
    caps_before_prof = batch.captures
    for _ in range(prof_batches):
        batch()
    prof = collect_profile(gpu)
    gpu.chk(gpu._lib.tsdrgpu_profile_enable(gpu._h, 0))
    batch.pp.set_overlap(not os.environ.get("BENCH_NO_OVERLAP"))
    batch.frd.set_overlap(batch.frd_overlap)
    prof_caps = (batch.captures - caps_before_prof) / prof_batches          # captures autocorrelated per profiled batch
    # rank 0 alone (allocations, first launches of other transform sizes): the other ranks wait on the host, their GPUs idle
    host_barrier()
    acs = autocorr_sweep(gpu, torch) if (rank == 0 and not os.environ.get("BENCH_NO_SWEEP")) else None
    host_barrier()

    # ---- e2e (headline): the reference-facing API end to end with an unmodified plugin, as the reference arm is measured
    e2e_seconds = float(os.environ.get("BENCH_E2E_SECONDS", "3.0"))
    api_run = e2e_through_tsdr_api(local, rank, w, e2e_seconds, barrier)
    if world > 1:
        tot = torch.tensor([api_run.get("value_per_rank", 0.0), 1.0 if "value_per_rank" in api_run else 0.0], device="cuda", dtype=torch.float64)
        dist.all_reduce(tot)
        api_total, api_ok = tot[0].item(), int(tot[1].item())
    else:
        api_total, api_ok = api_run.get("value_per_rank", 0.0), int("value_per_rank" in api_run)

    # ---- beside it: tsdrgpu_pipeline_process() fed from PINNED host memory in 16 MiB calls (what a GPU-aware front end can do)
    chunk = 512 * 1024 * 8                     # floats per process() call (8x the RawFile plugin's block)
    pl = pipeline.Pipeline(samplerate=FS, height=HEIGHT, refreshrate=FV, batch_frames=16, batch_blocks=160, block_when_busy=True,
                           device=local, params={"autoshift": 1, "lowpass_before_sync": 1})
    host = iq_pinned.numpy()
    base_ptr = iq_pinned.data_ptr()

    def feed_once():
        # the pinned source is never modified, so its blocks may be handed over without waiting for each copy (what a front end
        # with a ring of page-locked buffers does: tsdrgpu_pipeline_process_raw_async + tsdrgpu_pipeline_sync_input)
        pos = 0
        while pos < host.size:
            n = min(chunk, host.size - pos)
            pl.process_raw_ptr_async(base_ptr + 4 * pos, 0, n, 0)
            pos += n

    # the link under the e2e number: pinned H2D and D2H of one batch's bytes, alone and together (context, not a claim)
    def link_gbs():
        d_in = torch.empty_like(iq_dev); h_out = torch.empty(FRAMES_PER_BATCH * batch.n, dtype=torch.float32).pin_memory()
        d_out = batch.frames_out[0][: FRAMES_PER_BATCH * batch.n]
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        res = {}
        reps = 4
        for name, both in (("h2d", (True, False)), ("d2h", (False, True)), ("duplex", (True, True))):
            for timed in (False, True):                      # one untimed pass first (first touch of the pinned pages, stream creation)
                torch.cuda.synchronize(); t0 = time.perf_counter()
                for _ in range(reps if timed else 1):
                    if both[0]:
                        with torch.cuda.stream(s1):
                            d_in.copy_(iq_pinned, non_blocking=True)
                    if both[1]:
                        with torch.cuda.stream(s2):
                            h_out.copy_(d_out, non_blocking=True)
                torch.cuda.synchronize(); dt = (time.perf_counter() - t0) / reps
            nbytes = (iq_pinned.numel() * 4 if both[0] else 0) + (h_out.numel() * 4 if both[1] else 0)
            res[name + "_gbs"] = nbytes / dt / 1e9
        return res
    link = link_gbs()
    feed_once(); pl.flush()
    barrier()
    s0 = pl.stats()
    t0 = time.perf_counter()
    e2e_passes = 0
    while True:                                   # at least 2 s of wall clock, the same number of passes on every rank
        feed_once(); e2e_passes += 1
        go = torch.tensor([1.0 if time.perf_counter() - t0 < 2.0 else 0.0], device="cuda")
        if world > 1:
            dist.all_reduce(go, op=dist.ReduceOp.MAX)
        if go.item() == 0.0 or e2e_passes >= 400:
            break
    pl.flush()
    torch.cuda.synchronize()
    t_e2e = torch.tensor([time.perf_counter() - t0], device="cuda")
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    s1 = pl.stats()
    pinned_val = world * e2e_passes * pairs / t_e2e.item() / 1e6
    pinned = {"value": pinned_val, "unit": "MS/s", "seconds": t_e2e.item(), "passes": e2e_passes,
              "h2d_bytes_per_pass": int((s1.h2d_bytes - s0.h2d_bytes) // e2e_passes), "d2h_bytes_per_pass": int((s1.d2h_bytes - s0.d2h_bytes) // e2e_passes),
              "frames_delivered": int(s1.frames_delivered - s0.frames_delivered), "pcie_link_measured": link,
              # bytes per sample over the link: 8 in + 4*pixels-per-sample out; bound by each direction alone and by both together
              "link_bound_MS_per_s": min(link["h2d_gbs"] / 8.0, link["d2h_gbs"] / (4.0 * batch.n * FRAMES_PER_BATCH / pairs),
                                         link["duplex_gbs"] / (8.0 + 4.0 * batch.n * FRAMES_PER_BATCH / pairs)) * 1e3,
              "how": "tsdrgpu_pipeline_process_raw_async() on PINNED host IQ in 16 MiB calls (buffers handed over without a wait per copy), frames copied back to pinned host slots; "
                     "host wall clock between device synchronisations"}
    pinned["of_link_bound"] = pinned_val / world / pinned["link_bound_MS_per_s"]
    pl.close()

    # ---- the same with the samples crossing PCIe as int8 (SURVEY 8f-1: raw sink / tsdrgpu_pipeline_process_raw):
    # reported beside the headline, never instead of it (the reference arm reads float32)
    e2e_int8 = None
    if world == 1 and not os.environ.get("BENCH_NO_INT8"):
        q8 = torch.clamp(torch.round(iq_pinned * (100.0 / float(iq_pinned.abs().max()))), -127, 127).to(torch.int8).pin_memory()
        pl8 = pipeline.Pipeline(samplerate=FS, height=HEIGHT, refreshrate=FV, batch_frames=16, batch_blocks=160, block_when_busy=True,
                                device=local, params={"autoshift": 1, "lowpass_before_sync": 1})
        ptr8, n8 = q8.data_ptr(), q8.numel()

        def feed8():
            pos = 0
            while pos < n8:
                n = min(chunk, n8 - pos)
                pl8.process_raw_ptr(ptr8 + pos, 1, n, 0)
                pos += n
        feed8(); pl8.flush()
        a0 = pl8.stats(); t8 = time.perf_counter(); n8p = 0
        while time.perf_counter() - t8 < 1.0:
            feed8(); n8p += 1
        pl8.flush(); torch.cuda.synchronize()
        t8 = time.perf_counter() - t8
        a1 = pl8.stats()
        e2e_int8 = {"value": n8p * pairs / t8 / 1e6, "unit": "MS/s", "h2d_bytes_per_pass": int((a1.h2d_bytes - a0.h2d_bytes) // n8p),
                    "d2h_bytes_per_pass": int((a1.d2h_bytes - a0.d2h_bytes) // n8p), "frames_delivered": int(a1.frames_delivered - a0.frames_delivered),
                    "how": "tsdrgpu_pipeline_process_raw(int8) on pinned host samples, converted on the device (TSDRPlugin_RawFile.c:247 values); "
                           "float32 frames copied back as in e2e"}
        pl8.close()

    # ---- the other BASELINE shapes (device-resident step only; child processes so that this process's state is untouched)
    other_shapes = None
    if world == 1 and rank == 0 and SHAPE == "cfg2" and not os.environ.get("BENCH_NO_SHAPES"):
        other_shapes = {}
        for name, cpu in (("cfg5", False), ("cfg1", True)):
            env = dict(os.environ, BENCH_SHAPE=name, BENCH_QUICK="1", BENCH_BATCHES_PER_STEP="8")
            if cpu:
                env["BENCH_SHAPE_CPU"] = "1"
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--steps", "10", "--warmup", "3"], env=env, capture_output=True, text=True, timeout=240)
                other_shapes[name] = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
            except Exception as e:
                other_shapes[name] = {"error": repr(e)[:200]}
    # ---- N > 1 only: the path's one real exchange, the superbandwidth stitch with one hop per GPU (configs[3])
    superb = None
    if world > 1:
        try:
            superb = superband_bench(gpu, torch, dist, iq_dev, world, rank, barrier, host_barrier)
        except Exception as e:                            # never lose the headline line to the informational section
            superb = {"error": repr(e)[:300]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel (by total device time in the profiled batches)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak, peak_src = (peaks.get("hbm_gbs"), "measured (MEASURED_PEAKS.json hbm_gbs)") if peaks.get("hbm_gbs") else (6650.0, "fallback (B200_PROFILING.md)")
    ratio = w * HEIGHT * FV / FS
    n_pix = batch.n * FRAMES_PER_BATCH
    NFFT = 1 << (int(3.1 * FS / 55.0).bit_length() - 1)   # the capture's transform size (fft_getrealsize): cfg2 capture 1 409 090 -> N = 2^20
    # ALGORITHMIC bytes per launch (DESIGN.md section 5).  The autocorrelation of one capture runs at half size (N/2 complex
    # points per transform): per capture the fused passes move  fwd A: read 8*(N/2) write 8*(N/2);  fwd B (+ finish, |X|/N):
    # read 8*(N/2) write 4*N;  inv A: read 4*N write 8*(N/2);  inv B (+ finish): read 8*(N/2) write 8*N  = 40*N bytes in all
    # (SURVEY 8d's single-pass ideal is 28*N); a launch covers every capture of the batch (grid.y).
    alg = {
        "rs_main": pairs * (8 + 4 * ratio + (0 if os.environ.get("BENCH_SEPARATE_DEMOD") else 4)),   # 8 B per IQ pair in + 4 B per pixel out (+ 4 B magnitude out)
        "fs_minmax": 4 * n_pix, "fs_normalise": 8 * n_pix, "fs_timelowpass": 8 * n_pix, "fs_norm_lowpass": 8 * n_pix,
        "fs_collapse": 4 * n_pix, "fs_shift": 8 * n_pix, "demod_kernel": 12 * pairs,
        "fft_pass_kernel": FFT_BYTES_PER_CAPTURE(NFFT) * prof_caps / max(1.0, prof.get("fft_pass_kernel", (0, 4 * prof_batches))[1] / prof_batches),
    }
    alg.update({k: v * prof_caps for k, v in FINISH_BYTES(NFFT, int(FS / 55.0) - int(FS / 87.0) + int(FS / (590 * 55.0)) - int(FS / (1500 * 87.0))).items()})
    label = {"rs_main": "rs_main<IQ> (fused demod+resample)", "fft_pass_kernel": "fft_pass_kernel (one pass over every capture of the batch)"}
    total_prof = sum(t for t, _ in prof.values()) or 1.0
    kernels = {k: {"ms_per_batch": t / prof_batches, "launches_per_batch": c / prof_batches, "share": t / total_prof} for k, (t, c) in sorted(prof.items(), key=lambda kv: -kv[1][0])}
    dom = next(iter(kernels))
    # the roofline object is for the dominant kernel of the step among the bandwidth kernels; fs_sync (clusters of CTAs walking
    # the frames in order, FP64-latency bound by construction) is listed in per_kernel but has no bandwidth roofline
    roof_k = next((k for k in kernels if alg.get(k)), "rs_main")
    t_k, c_k = prof.get(roof_k, (0.0, 0))
    achieved = alg[roof_k] / (t_k / c_k * 1e-3) / 1e9 if c_k else None
    roofline = {"kernel": label.get(roof_k, roof_k), "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg[roof_k], "avg_launch_ms": (t_k / c_k) if c_k else None,
                "dominant_kernel_by_time": dom,
                # the whole batch against SURVEY 8d's algorithmic bytes: 16 B per sample + 16 B per pixel + 28 N per capture
                "whole_step": {"algorithmic_bytes_per_batch": 16 * pairs + 16 * n_pix + 28 * NFFT * (caps_done / (args.steps * BATCHES_PER_STEP)),
                               "ms_per_batch": ms_total / (args.steps * BATCHES_PER_STEP)},
                "per_kernel": {k: dict(v, **({"achieved_gbs": alg[k] * v["launches_per_batch"] / (v["ms_per_batch"] * 1e-3) / 1e9,
                                              "frac": alg[k] * v["launches_per_batch"] / (v["ms_per_batch"] * 1e-3) / 1e9 / peak} if alg.get(k) else {})) for k, v in kernels.items()}}
    ws = roofline["whole_step"]
    ws["achieved_gbs"] = ws["algorithmic_bytes_per_batch"] / (ws["ms_per_batch"] * 1e-3) / 1e9
    ws["frac"] = ws["achieved_gbs"] / peak
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic_latest.json")))
        roofline["traffic"] = tr.get(roof_k, {}).get("dram_bytes_per_launch")
        roofline["traffic_source"] = tr.get(roof_k, {}).get("source")
    except Exception:
        pass
    cpu = cpu_baseline(w)
    if api_ok == world:
        e2e = {"value": api_total, "unit": "MS/s",
               "h2d_bytes_per_step": int(api_run["h2d_bytes_per_frame"] * FRAMES_PER_STEP), "d2h_bytes_per_step": int(api_run["d2h_bytes_per_frame"] * FRAMES_PER_STEP),
               "seconds": api_run["seconds"], "frames_per_s_rank0": api_run["frames_per_s"], "plugin": api_run["plugin"],
               "plugin_thread_per_block_us": api_run.get("plugin_thread_per_block_us"),
               "how": "this repo's libTSDRLibrary.so through tsdr_init/tsdr_loadplugin/tsdr_readasync with an unmodified file plugin handing over "
                      "its pageable 2 MiB malloc'd float32 buffer (page-locked in place after it came back 3 times), 16 frames per launch group, "
                      "frames delivered to the tsdr_readasync_function counted x samples per frame -- the reference arm's own method; the plugin's "
                      "single thread (fread + memcpy per block) is inside the timed region",
               "pinned_process": pinned}
    else:                                          # the API run failed on some rank: the pinned figure stands, and says so
        e2e = {"value": pinned_val, "unit": "MS/s", "h2d_bytes_per_step": pinned["h2d_bytes_per_pass"] * BATCHES_PER_STEP,
               "d2h_bytes_per_step": pinned["d2h_bytes_per_pass"] * BATCHES_PER_STEP, "how": pinned["how"], "tsdr_api_run": api_run, "pinned_process": pinned}
    line = {
        "metric": METRIC, "value": value, "unit": "MS/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (f64 accumulators where the reference uses them)", "data": "synthetic",
        "config": {"workload": "BASELINE configs[1]: 1080p60 geometry (1125 total lines -> 740x1125 px frames), 25 MS/s float32 IQ; one step = "
                               f"{BATCHES_PER_STEP} passes over {pairs} resident IQ pairs ({8 * pairs / 1e6:.0f} MB > L2, so no L2 flush is needed) = "
                               f"{FRAMES_PER_STEP} frames, {pairs_step} IQ pairs",
                   "frames_per_step": frames_done / args.steps, "autocorr_captures_per_step": caps_done / args.steps,
                   "frames_per_s": world * frames_done / (ms_total * 1e-3), "parallelism": f"replicas x{world}" if world > 1 else "single stream",
                   "host_enqueue_ms_per_batch": host_enqueue_ms, "numa": {"device_node": numa_node, "rank_bound_to_node": numa_bound},
                   "flags": "AUTOSHIFT=1, LOW_PASS_BEFORE_SYNC=1, AUTOGAIN_AFTER=0, motionblur 0 (GUI defaults), PLL write-back off"},
        "gpu_launches": int(launches),
        "e2e": e2e, "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
    }
    if acs:
        line["autocorr_sweep"] = acs
    if superb:
        line["superbandwidth"] = superb
    if e2e_int8:
        line["e2e_int8_transport"] = e2e_int8
    if other_shapes:
        line["other_shapes"] = other_shapes
    emit(line)
    if world > 1:
        dist.destroy_process_group()


FFT_FUSED_FINISH = False          # flips when k_real_*_finish move into the pass epilogues (then 40 N per capture instead of 52 N)


def FFT_BYTES_PER_CAPTURE(n, passes=2):
    """bytes the FFT PASS kernels of one half-size autocorrelation move: `passes` global passes per N/2-point transform, each
    reading and writing N/2 complex points (8 N bytes per pass); with the finish steps fused into the passes the forward's last
    pass writes N reals (4 N), the inverse's first reads them and its last writes N complex (8 N): 40 N at 2 passes."""
    if FFT_FUSED_FINISH:
        return (2 * passes - 2) * 8 * n + (4 + 4) * n + (4 + 4) * n + (4 + 8) * n - 8 * n if passes == 2 else (2 * passes) * 8 * n + 8 * n
    return 2 * passes * 8 * n


def FINISH_BYTES(n, window_lags=None):
    """forward finish: N/2 complex in, N reals out; inverse finish: z[k], z[N/2-k] and one table entry in, y[k] out -- for every
    lag (12 N), or only for the lags of the frame-rate detector's two windows"""
    return {"k_real_fwd_finish": 8 * n, "k_real_inv_finish": 12 * n if window_lags is None else 32 * window_lags}


def autocorr_sweep(gpu, torch):
    """BASELINE configs[2]: autocorrelation (fft.c:49-64) of windows of 2^16 .. 2^24 real samples on one B200.  Per size: the device
    time of one autocorrelation (CUDA events around `reps` back-to-back calls on inputs that together exceed L2 at the small
    sizes), GB/s against the bytes the passes actually move and against SURVEY 8d's 28*N single-pass ideal."""
    peak = None
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs")
    except Exception:
        pass
    peak = peak or 6650.0
    out = {}
    lib = gpu._lib
    for logn in range(16, 25):
        n = 1 << logn
        batch = max(1, min(64, (1 << 26) // n))           # >= 256 MB of answers per launch at every size: larger than L2
        x = torch.rand(batch * n, device="cuda") + 0.25
        ans = torch.empty(batch * 2 * n, device="cuda")
        run = lambda: gpu.chk(lib.tsdrgpu_autocorrelation_batch(gpu._h, gpu.stream, ans.data_ptr(), x.data_ptr(), n, batch, n))
        for _ in range(3):
            run()
        reps = 10
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for _ in range(reps):
            run()
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps / batch
        passes = 1 if logn - 1 <= 11 else (2 if logn - 1 <= 20 else 3)     # global passes per half-size transform (fft_run's factorisation)
        moved = FFT_BYTES_PER_CAPTURE(n, passes) + (0 if FFT_FUSED_FINISH else sum(FINISH_BYTES(n).values()))
        out[f"2^{logn}"] = {"us_per_autocorrelation": ms * 1e3, "batch": batch, "passes_per_transform": passes,
                            "gbs_vs_bytes_moved": moved / (ms * 1e-3) / 1e9, "frac_vs_bytes_moved": moved / (ms * 1e-3) / 1e9 / peak,
                            "gbs_vs_28N": 28 * n / (ms * 1e-3) / 1e9, "frac_vs_28N": 28 * n / (ms * 1e-3) / 1e9 / peak}
        del x, ans
    return out


def superband_bench(gpu, torch, dist, iq_dev, world, rank, barrier, host_barrier):
    """BASELINE configs[3] / the path's one sharded row (SURVEY 8e): superbandwidth with one hop per GPU, H = world hops of
    10 frames of 25 MS/s IQ each (N = 2^21 per hop).  Reports, all with an L2 flush between repetitions (a stitch runs once per
    H x 0.67 s of signal in production: cold caches are the honest state):
      ms_per_stitch       hops resident on their GPUs -> time-contiguous magnitude stream resident on the root (max over ranks)
      one_gpu_ms          the same H hops through the one-GPU stitch (tsdrgpu_superb_stitch) on rank 0's GPU, its IQ output
      speedup             one_gpu_ms / ms_per_stitch
      frames_per_s        root: stitch + resample + frame stage of the stitched stream, frames of the H x rate geometry per second
      parity              sharded magnitudes vs |one-GPU stitch| (max error / peak), lags equal
      nccl_allgather_baseline_ms   round 1's formulation (one NCCL all-gather of raw spectra, every rank derives every lag)
    Order of the section: everything rank 0 does ALONE (the one-GPU reference, first launches and allocations of the H x rate
    geometry) comes first, before the group's peer-memory windows exist and with the other ranks parked in a HOST barrier (gloo):
    at 8 GPUs the same work done while seven GPUs sat in flag-waiting kernels once took longer than those kernels' patience."""
    from tempestsdr_b200 import superband
    from tempestsdr_b200.api import PostProcessFlags
    H = world
    sif = int(FS / FV)
    hop_pairs = 10 * sif                                  # SUPER_SAMPLES_TO_RECORD frames per hop -> N = 2^21
    src = torch.from_numpy(make_iq(hop_pairs + 16 * 1000, seed=4242)).cuda()       # the same on every rank: rank 0 can rebuild every hop
    offs = [0] + [131 + 977 * q for q in range(1, H)]
    hop_of = lambda q: src[2 * offs[q]: 2 * (offs[q] + hop_pairs)].contiguous()
    hop = hop_of(rank)
    hop0 = hop_of(0)                                      # the alignment reference, kept on every device (the pipeline copies hop 0 to all GPUs at ingest)
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")            # 256 MB > L2
    n_fft = gpu.fft_getrealsize(hop_pairs)
    # the root consumes the stream where the last phase leaves it (its window; tsdrgpu_superb_mgpu_stream_window): no copy out
    stitch = lambda: grp.stitch(hop, sif, hop0=hop0, in_place=True)
    flags = PostProcessFlags(autoshift=True, lowpass_before_sync=True, superresolution=True)
    # ---- rank 0 alone: the same hops on one GPU (timing + the parity reference), buffers and first launches of the frames path
    solo = torch.zeros(2, device="cuda", dtype=torch.float64)                      # [ok, one_gpu_ms]
    r0 = {}
    if rank == 0:
        try:
            hops = [hop_of(q) for q in range(H)]
            for _ in range(2):
                one_iq, one_offs = gpu.superb_stitch(hops, sif)
            t1 = []
            for _ in range(5):
                flush.zero_(); torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); one_iq, one_offs = gpu.superb_stitch(hops, sif); b.record(); torch.cuda.synchronize()
                t1.append(a.elapsed_time(b))
            ref_mag = gpu.am_demod(one_iq)
            r0["ref_mag"], r0["ref_peak"], r0["one_offs"] = ref_mag, float(ref_mag.abs().max()), list(one_offs)
            r0["diff"] = torch.empty_like(ref_mag)
            del one_iq, hops
            # frames from the stitched stream: H x the rate, same lines
            wH = int(2 * (H * FS / (FV * HEIGHT)))
            blockH = int(0.1 * H * FS / FV)
            nblk = (H * n_fft) // blockH
            rs, pp = gpu.resampler(), gpu.post_processor()
            upH = float(wH * HEIGHT) * FV
            pix = torch.empty(int(rs.plan((blockH, nblk), upH, float(H * FS))) + 1024, dtype=torch.float32, device="cuda")
            nH = wH * HEIGHT
            frames_out = torch.empty(((pix.numel() // nH) + 1) * nH, dtype=torch.float32, device="cuda")

            def frames_of(stream_mag):
                px = rs.process(stream_mag, (blockH, nblk), upH, float(H * FS), in_is_iq=False, out=pix)
                nf = px.numel() // nH
                pp.process(px[: nf * nH], wH, HEIGHT, 0.0, 0.1, flags, out=frames_out[: nf * nH], want_results=False)
                return nf
            frames_of(ref_mag)                            # first launches and allocations happen here
            pp.join(); torch.cuda.synchronize()
            r0["frames_of"], r0["geometry"] = frames_of, [wH, HEIGHT]
            solo[0], solo[1] = 1.0, sum(t1) / len(t1)
        except Exception as e:
            r0["error"] = repr(e)[:300]
    host_barrier()
    dist.all_reduce(solo)
    if solo[0].item() != 1.0:
        return {"hops": H, "n_per_hop": n_fft, "error": "rank 0's one-GPU reference failed: " + str(r0.get("error"))}
    one_ms = solo[1].item()
    # ---- the group: windows mapped into every rank (CUDA IPC); a flag wait gives up after 10 s here (a lost rank then costs the
    # section at most a few tens of seconds before every rank leaves it together)
    os.environ.setdefault("TSDRGPU_SBM_TIMEOUT_MS", "10000")
    host_barrier()
    grp = superband.SuperbGroup.for_process_group(gpu, hop_pairs)

    def group_ok():
        """Collective: did any rank's flag wait time out (the status word is sticky)?  Every rank gets the same answer, so the ranks
        leave the section together instead of one raising while the others walk into the next collective."""
        bad = 0
        try:
            grp.lags()
        except Exception:
            bad = 1
        t = torch.tensor([bad], device="cuda", dtype=torch.int32)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return int(t.item()) == 0

    def give_up(where, partial):
        partial["error"] = f"a flag wait of the sharded stitch timed out {where}; the remaining superbandwidth measurements were skipped"
        try:
            grp.close()
        except Exception:
            pass
        return partial

    for k in range(3):
        stitch()
        if k == 0 and not group_ok():                     # the first stitch (tables, first launches) is where ranks can drift apart: check at once
            return give_up("in the first warm-up stitch", {"hops": H, "n_per_hop": n_fft, "one_gpu_ms": one_ms})
    if not group_ok():
        return give_up("in the warm-up stitches", {"hops": H, "n_per_hop": n_fft, "one_gpu_ms": one_ms})
    lags = grp.lags()
    barrier()
    reps = 10
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in evs:
        flush.zero_()
        a.record(); out = stitch(); b.record()
    barrier()
    tms = torch.tensor([sum(a.elapsed_time(b) for a, b in evs) / reps], device="cuda")
    dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    res = {"hops": H, "n_per_hop": n_fft, "ms_per_stitch": tms.item(), "stitched_MS_per_s": H * n_fft / (tms.item() * 1e-3) / 1e6,
           "one_gpu_ms": one_ms, "speedup_vs_one_gpu": one_ms / tms.item(),
           "lags": lags, "l2_flushed_between_repetitions": True,
           "resident_before_the_timed_region": "hop q on GPU q, plus a copy of hop 0 (the alignment reference) on every GPU, as the pipeline leaves them",
           "stream_lands": "in the root's window of the group (consumed in place by the resampler; no device-to-device copy)",
           "exchange": "peer-memory windows (CUDA IPC over NVLink), flags in peer memory; no collective library on the data path",
           "nvlink_bytes_received_per_rank": int(8 * (n_fft // 2) * (1 if rank else 0) + 2 * 8 * n_fft * (H - 1) // H),
           "nvlink_bytes_received_by_root_for_stream": int(4 * n_fft * (H - 1))}
    if not group_ok():
        return give_up("in the timed stitches", res)
    # ---- parity of the sharded stream against the one-GPU path (rank 0; no new allocations while the windows are mapped)
    if rank == 0:
        torch.sub(out, r0["ref_mag"], out=r0["diff"])
        err = float(r0["diff"].abs_().max()) / r0["ref_peak"]
        res["parity_vs_one_gpu_path"] = {"max_err_over_peak": err, "lags_equal": [2 * l for l in lags] == r0["one_offs"], "bound": 1e-5}
    # ---- frames: stitch + resample + frame stage of the stitched stream on the root; every rank takes part in the stitch
    def round_trip():
        so = stitch()
        return r0["frames_of"](so) if rank == 0 else 0
    host_barrier()
    nf = 0
    for _ in range(2):
        nf = round_trip()
    barrier()
    fe = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(5)]
    for a, b in fe:
        flush.zero_()
        a.record(); nf = round_trip(); b.record()
    barrier()
    ft = torch.tensor([sum(a.elapsed_time(b) for a, b in fe) / len(fe)], device="cuda")
    dist.all_reduce(ft, op=dist.ReduceOp.MAX)
    res["frames"] = {"frames_per_round": int(nf) if rank == 0 else None, "ms_per_round_stitch_plus_frames": ft.item(),
                     "frames_per_s": (nf / (ft.item() * 1e-3)) if rank == 0 else None, "geometry": r0.get("geometry")}
    if not group_ok():
        return give_up("in the stitch + frames rounds", res)
    # ---- where one stitch spends its time: CUDA events around every launch of 3 stitches on every rank (a flag-waiting kernel's
    # time is the wait for the slowest peer); informational, outside every timed region above
    try:
        collect_profile(gpu)
        gpu.chk(gpu._lib.tsdrgpu_profile_enable(gpu._h, 1))
        for _ in range(3):
            flush.zero_()
            stitch()
        torch.cuda.synchronize()
        gpu.chk(gpu._lib.tsdrgpu_profile_enable(gpu._h, 0))
        mine = {k: round(1e3 * t / 3, 2) for k, (t, c) in collect_profile(gpu).items()}
    except Exception as e:
        mine = {"error": repr(e)[:160]}
    everyone = [None] * world
    dist.all_gather_object(everyone, mine)
    res["per_kernel_us_per_stitch"] = {"rank0_root": everyone[0], "rank1": everyone[1], "last_rank": everyone[-1]}
    barrier()
    if not group_ok():
        return give_up("in the profiled stitches", res)
    # ---- round 1's formulation as the baseline: one NCCL all-gather of the raw spectra, every rank derives every lag
    try:
        for _ in range(2):
            superband.stitch_distributed(gpu, hop, sif)
        barrier()
        ne = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(5)]
        for a, b in ne:
            flush.zero_()
            a.record(); superband.stitch_distributed(gpu, hop, sif); b.record()
        barrier()
        nt = torch.tensor([sum(a.elapsed_time(b) for a, b in ne) / len(ne)], device="cuda")
        dist.all_reduce(nt, op=dist.ReduceOp.MAX)
        res["nccl_allgather_baseline_ms"] = nt.item()
    except Exception as e:
        res["nccl_allgather_baseline_ms"] = None; res["nccl_allgather_baseline_error"] = repr(e)[:160]
    grp.close()
    return res


# --------------------------------------------------------------------------------------------------- reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    w = geometry()
    ncores = os.cpu_count() or 1
    if not orc.have_ref():
        cpu = cpu_baseline(w)
        cpu["sample"] = "reference binary absent: pinned C port, " + cpu["sample"]
        emit(({"impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": "MS/s", "n_gpus": args.gpus, "steps": args.steps,
                          "warmup": args.warmup, "higher_is_better": True, "data": "synthetic", "cpu_baseline": cpu,
                          "config": {"workload": "BASELINE configs[1] geometry, C port of the reference stages, one thread"},
                          "e2e": {"value": cpu["value"], "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    # The reference's own threaded pipeline is measured in a CHILD process: its worker threads race on shared state (SURVEY F9;
    # TSDRLibrary.c:62-94 leaves fields uninitialised) and now and then the unmodified library segfaults during start-up.
    # A crash must not cost the round its reference number: retry, and only then fall back to the stage-driven figure.
    child = None
    per_frame = int(FS / FV)
    tmp = tempfile.NamedTemporaryFile(prefix="tsdr_iq_", suffix=".raw", delete=False)     # one recording for every attempt
    make_iq(16 * per_frame, seed=1000).tofile(tmp); tmp.close()
    tries = 10
    try:
        for attempt in range(tries):
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference_child", "--gpus", str(args.gpus),
                                "--steps", str(args.steps), "--warmup", str(args.warmup)], capture_output=True, text=True,
                               env=dict(os.environ, BENCH_REF_IQ_FILE=tmp.name))
            lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
            if lines:                                   # the measurement was printed; how the reference's shutdown went afterwards does not matter
                child = json.loads(lines[-1]); child["attempts"] = attempt + 1
                break
            sys.stderr.write(f"[bench] reference pipeline attempt {attempt + 1} ended with rc={r.returncode} (the unmodified library crashed); retrying\n")
            time.sleep(0.2 * (attempt + 1))
    finally:
        os.unlink(tmp.name)
    if child is None:
        cpu = cpu_baseline(w)
        cpu["sample"] = f"the reference's threaded pipeline crashed {tries} times in a row; its stage functions driven serially instead: " + cpu["sample"]
        emit(({"impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": "MS/s", "n_gpus": args.gpus, "steps": args.steps,
               "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "cpu_baseline": cpu, "config": {"workload": "BASELINE configs[1] geometry, the compiled reference's stage functions, one thread"},
               "e2e": {"value": cpu["value"], "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    fps, caps, seconds, per_frame = child["fps"], child["caps"], child["seconds"], child["per_frame"]
    native_maps = child.get("native_libraries_mapped")
    value = fps * per_frame / 1e6
    cpu = {"value": value, "unit": "MS/s", "cores": min(ncores, 6), "kind": "reference",
           "sample": f"the reference's own threaded pipeline (plugin + decimate + post-process + video + autocorr threads) for "
                     f"{args.steps} x {seconds:.0f} s on {ncores} host cores; counts FRAMES DELIVERED x samples per frame "
                     f"(it drops whole blocks when a ring is full); {fps:.1f} frames/s, {caps:.2f} autocorrelation captures/s"
                     + (f"; attempt {child['attempts']} (earlier ones crashed inside the reference library)" if child["attempts"] > 1 else "")}
    emit(({"impl": "reference", "metric": METRIC, "value": value, "unit": "MS/s", "n_gpus": args.gpus, "steps": args.steps,
                      "warmup": args.warmup, "ms_per_step": seconds * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": "f32", "data": "synthetic", "cpu_baseline": cpu,
                      "config": {"workload": "BASELINE configs[1]: 1080p60 geometry (1125 lines), 25 MS/s float32 IQ from a file through "
                                             "TSDRPlugin_RawFile (pacing off) and the unmodified reference library", "frames_per_s": fps,
                                 "native_libraries_mapped_by_the_measuring_process": native_maps},
                      "e2e": {"value": value, "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_reference_child(args):
    """One attempt at driving the unmodified reference library (see run_reference); prints {"fps", "caps", ...} as JSON."""
    from oracle import oracle as orc
    lib = C.CDLL(orc.REF_LIB_SO)
    per_frame = int(FS / FV)
    iq_file = os.environ["BENCH_REF_IQ_FILE"]              # written (and removed) by the parent
    FRAME_CB = C.CFUNCTYPE(None, C.POINTER(C.c_float), C.c_int, C.c_int, C.c_void_p)
    VALUE_CB = C.CFUNCTYPE(None, C.c_int, C.c_double, C.c_double, C.c_void_p)
    PLOT_CB = C.CFUNCTYPE(None, C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_uint32, C.c_void_p)
    count = {"frames": 0, "plots": 0}
    fcb = FRAME_CB(lambda b, ww, hh, c: count.__setitem__("frames", count["frames"] + 1))
    vcb = VALUE_CB(lambda i, a, b, c: None)
    pcb = PLOT_CB(lambda p, o, v, s, sr, c: count.__setitem__("plots", count["plots"] + 1))
    t = C.c_void_p()
    lib.tsdr_init(C.byref(t), vcb, pcb, None)
    lib.tsdr_setresolution.argtypes = [C.c_void_p, C.c_int, C.c_double]
    lib.tsdr_motionblur.argtypes = [C.c_void_p, C.c_float]
    lib.tsdr_setgain.argtypes = [C.c_void_p, C.c_float]
    lib.tsdr_setparameter_int.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
    lib.tsdr_loadplugin.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
    lib.tsdr_readasync.argtypes = [C.c_void_p, FRAME_CB, C.c_void_p]
    lib.tsdr_stop.argtypes = [C.c_void_p]
    lib.tsdr_setresolution(t, HEIGHT, FV); lib.tsdr_motionblur(t, 0.0); lib.tsdr_setgain(t, 0.5)
    for pid, v in ((0, 1), (1, 0), (6, 1)):          # AUTOSHIFT=1, PLL=0, LOW_PASS_BEFORE_SYNC=1
        lib.tsdr_setparameter_int(t, pid, v)
    rc = lib.tsdr_loadplugin(t, orc.REF_RAWFILE_NOPACE_SO.encode(), f'"{iq_file}" {FS} float'.encode())
    assert rc == 0, f"tsdr_loadplugin rc={rc}"
    th = threading.Thread(target=lambda: lib.tsdr_readasync(t, fcb, None), daemon=True)
    th.start()
    seconds = 4.0
    time.sleep(1.0)                                  # warm-up: rings grow, first frames arrive
    results = []
    for s in range(args.warmup + args.steps):
        f0, p0, t0 = count["frames"], count["plots"], time.perf_counter()
        time.sleep(seconds)
        dt = time.perf_counter() - t0
        if s >= args.warmup:
            results.append(((count["frames"] - f0) / dt, (count["plots"] - p0) / 2 / dt))
    fps = statistics.mean(r[0] for r in results)
    caps = statistics.mean(r[1] for r in results)
    try:                                             # which native libraries this child had mapped (the reference's, none of this repo's)
        maps = sorted({l.split()[-1] for l in open("/proc/self/maps") if l.rstrip().endswith(".so") and ("/oracle/" in l or "tempestsdr_b200" in l)})
    except Exception:
        maps = []
    emit({"fps": fps, "caps": caps, "seconds": seconds, "per_frame": per_frame, "native_libraries_mapped": maps})
    sys.stdout.flush(); sys.stderr.flush()
    # End the run the way a host would: tsdr_stop from this thread, then a normal interpreter exit so that exit hooks (the
    # driver's library recorder among them) run.  The reference's shutdown path races now and then (SURVEY F9): a watchdog
    # ends the process if it hangs -- the measurement is already on stdout by then.
    wd = threading.Timer(10.0, lambda: os._exit(0)); wd.daemon = True; wd.start()
    try:
        lib.tsdr_stop(t)
        th.join(timeout=8)
    except Exception:
        pass


_RESULT_OUT = None


def _claim_stdout():
    """Rank 0 must print exactly ONE line on stdout.  Libraries write there too (NCCL's version banner goes to fd 1 whatever
    NCCL_DEBUG says once it is at least VERSION), so the real stdout is set aside for the result line and fd 1 is pointed at
    stderr for everything else."""
    global _RESULT_OUT
    if _RESULT_OUT is None:
        sys.stdout.flush()
        _RESULT_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict) -> None:
    out = _RESULT_OUT if _RESULT_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference_child"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR as .npy files")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "reference_child":
        run_reference_child(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
