"""Host-side mirror of the reference's stage interface, on top of the C-ABI (include/tsdrgpu.h).

Names and argument meaning follow the reference (TempestSDR/src): ``am_demod``, ``dsp_resample_process`` ->
:class:`Resampler`, ``dsp_post_process`` -> :class:`PostProcessor`, ``fft_perform`` / ``fft_autocorrelation`` /
``fft_crosscorrelation``, ``frameratedetector_runontodata`` -> :class:`FrameRateDetector`, ``superb_ondataready`` ->
:func:`superb_stitch`.  torch is used for device memory and streams only; every computation happens in the
hand-written sm_100a kernels of libtsdrgpu.so.  No CPU fallback exists: without the library or a GPU, calls raise.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as N
from ._native import FrameResult, TsdrGpuError  # noqa: F401


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _f32(t: torch.Tensor) -> torch.Tensor:
    assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous(), "expected a contiguous float32 CUDA tensor"
    return t


class Context:
    """One tsdrgpu_ctx_t bound to one CUDA device (one per process/rank)."""

    def __init__(self, device: int | torch.device | None = None):
        if not torch.cuda.is_available():
            raise TsdrGpuError("no CUDA device: tempestsdr_b200 has no CPU fallback")
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device("cuda", device if isinstance(device, int) else device.index)
        self._lib = N.lib()
        h = C.c_void_p()
        N.check(self._lib.tsdrgpu_create(C.byref(h), self.device.index))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._lib.tsdrgpu_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def chk(self, rc: int):
        N.check(rc, self._h)

    @property
    def stream(self) -> int:
        return _stream_ptr(self.device)

    @property
    def sm_count(self) -> int:
        return self._lib.tsdrgpu_sm_count(self._h)

    @property
    def launches(self) -> int:
        return self._lib.tsdrgpu_launch_count(self._h)

    # ------------------------------------------------------------------ a2
    def am_demod(self, iq: torch.Tensor) -> torch.Tensor:
        """TSDRLibrary.c:244-262 -- interleaved I,Q float32 -> magnitudes."""
        _f32(iq)
        out = torch.empty(iq.numel() // 2, dtype=torch.float32, device=iq.device)
        self.chk(self._lib.tsdrgpu_am_demod(self._h, self.stream, iq.data_ptr(), iq.numel() // 2, out.data_ptr()))
        return out

    def convert_samples(self, raw: torch.Tensor) -> torch.Tensor:
        """TSDRPlugin_RawFile.c:241-261 on the device: int8 / uint8 / int16 / uint16 (or float32) samples -> float32."""
        fmt = {torch.float32: 0, torch.int8: 1, torch.int16: 2, torch.uint8: 3, torch.uint16: 4}[raw.dtype]
        out = torch.empty(raw.numel(), dtype=torch.float32, device=raw.device)
        self.chk(self._lib.tsdrgpu_convert_samples(self._h, self.stream, raw.data_ptr(), fmt, raw.numel(), out.data_ptr()))
        return out

    # ------------------------------------------------------------------ a8-a10, a14 (stage level)
    def dsp_autogain_run(self, state: List[float], frame: torch.Tensor, norm: float, snr: bool = True) -> torch.Tensor:
        """dsp.c:41-94.  state = [lastmax, lastmin, snr] is updated in place."""
        _f32(frame)
        out = torch.empty_like(frame)
        a, b, c = C.c_float(state[0]), C.c_float(state[1]), C.c_float(state[2])
        self.chk(self._lib.tsdrgpu_autogain(self._h, self.stream, C.byref(a), C.byref(b), C.byref(c) if snr else None,
                                            frame.numel(), frame.data_ptr(), out.data_ptr(), norm))
        state[0], state[1], state[2] = a.value, b.value, c.value
        return out

    def dsp_timelowpass_run(self, coeff: float, frame: torch.Tensor, screen: torch.Tensor) -> None:
        """dsp.c:22-33, screen updated in place."""
        self.chk(self._lib.tsdrgpu_timelowpass(self._h, self.stream, coeff, frame.numel(), _f32(frame).data_ptr(), _f32(screen).data_ptr()))

    def dsp_average_v_h(self, frame: torch.Tensor, width: int, height: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """dsp.c:96-110 -> (widthcollapsebuffer, heightcollapsebuffer)."""
        wb = torch.empty(width, dtype=torch.float32, device=frame.device)
        hb = torch.empty(height, dtype=torch.float32, device=frame.device)
        self.chk(self._lib.tsdrgpu_average_v_h(self._h, self.stream, width, height, _f32(frame).data_ptr(), wb.data_ptr(), hb.data_ptr()))
        return wb, hb

    def gaussianblur(self, strip: torch.Tensor) -> torch.Tensor:
        """gaussian.c:18-79 (returns a blurred copy)."""
        s = _f32(strip).clone()
        self.chk(self._lib.tsdrgpu_gaussianblur(self._h, self.stream, s.data_ptr(), s.numel()))
        return s

    def pixels_argb(self, frame: torch.Tensor, inverted: bool = False, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """JavaGUI/jni/TSDRLibraryNDK.c:222-283 float -> ARGB int32."""
        if out is None:
            out = torch.zeros(frame.numel(), dtype=torch.int32, device=frame.device)
        self.chk(self._lib.tsdrgpu_pixels_argb(self._h, self.stream, _f32(frame).data_ptr(), frame.numel(), int(inverted), out.data_ptr()))
        return out

    # ------------------------------------------------------------------ a19, a20
    def fft_getrealsize(self, size: int) -> int:
        return self._lib.tsdrgpu_fft_getrealsize(size)

    def fft_perform(self, iq: torch.Tensor, size: int, inverse: bool) -> None:
        """fft.c:96-176, in place on the first 2^floor(log2 size) complex samples."""
        self.chk(self._lib.tsdrgpu_fft(self._h, self.stream, _f32(iq).data_ptr(), size, int(inverse)))

    def fft_autocorrelation(self, real: torch.Tensor) -> torch.Tensor:
        """fft.c:49-64 -> 2*size floats."""
        ans = torch.empty(2 * real.numel(), dtype=torch.float32, device=real.device)
        self.chk(self._lib.tsdrgpu_autocorrelation(self._h, self.stream, ans.data_ptr(), _f32(real).data_ptr(), real.numel()))
        return ans

    def fft_crosscorrelation(self, a: torch.Tensor, b: torch.Tensor, samples: int) -> None:
        """fft.c:69-93, result in `a`, `b` is clobbered."""
        self.chk(self._lib.tsdrgpu_crosscorrelation(self._h, self.stream, _f32(a).data_ptr(), _f32(b).data_ptr(), samples))

    def accummulate(self, out: torch.Tensor, calls: int, ac: torch.Tensor, startid: int, length: int) -> None:
        """frameratedetector.c:34-62 (the reference's spelling), out: float64 running means."""
        assert out.dtype == torch.float64 and out.is_cuda
        self.chk(self._lib.tsdrgpu_accumulate(self._h, self.stream, out.data_ptr(), calls, _f32(ac).data_ptr(), startid, length))

    # ------------------------------------------------------------------ a22
    def complex_to_abs_diff(self, iq: torch.Tensor) -> None:
        self.chk(self._lib.tsdrgpu_complex_to_abs_diff(self._h, self.stream, _f32(iq).data_ptr(), iq.numel()))

    def superb_bestfit(self, hop0: torch.Tensor, hopi: torch.Tensor, size_floats: int, samples_in_frame: int) -> int:
        r = C.c_int(0)
        self.chk(self._lib.tsdrgpu_superb_bestfit(self._h, self.stream, _f32(hop0).data_ptr(), _f32(hopi).data_ptr(), size_floats, samples_in_frame, C.byref(r)))
        return r.value

    def superb_stitch(self, hops: Sequence[torch.Tensor], samples_in_frame: int) -> Tuple[torch.Tensor, List[int]]:
        """superb_ondataready (superbandwidth.c:121-152) on one GPU."""
        pairs = hops[0].numel() // 2
        n = self.fft_getrealsize(pairs)
        out = torch.empty(len(hops) * n * 2, dtype=torch.float32, device=hops[0].device)
        ptrs = (C.c_void_p * len(hops))(*[_f32(h).data_ptr() for h in hops])
        offs = (C.c_int * len(hops))()
        total = C.c_int(0)
        self.chk(self._lib.tsdrgpu_superb_stitch(self._h, self.stream, ptrs, len(hops), pairs, samples_in_frame, out.data_ptr(), offs, C.byref(total)))
        return out[: 2 * total.value], list(offs)

    def superb_hop_spectrum(self, hop: torch.Tensor, best_offset_floats: int) -> torch.Tensor:
        pairs = hop.numel() // 2
        n = self.fft_getrealsize(pairs)
        spec = torch.empty(2 * n, dtype=torch.float32, device=hop.device)
        self.chk(self._lib.tsdrgpu_superb_hop_spectrum(self._h, self.stream, _f32(hop).data_ptr(), pairs, best_offset_floats, spec.data_ptr()))
        return spec

    def superb_residue_ifft(self, gathered: torch.Tensor, nhops: int, n: int, residue: int) -> torch.Tensor:
        out = torch.empty(2 * n, dtype=torch.float32, device=gathered.device)
        self.chk(self._lib.tsdrgpu_superb_residue_ifft(self._h, self.stream, _f32(gathered).data_ptr(), nhops, n, residue, out.data_ptr()))
        return out

    # ------------------------------------------------------------------ factories
    def resampler(self) -> "Resampler":
        return Resampler(self)

    def post_processor(self) -> "PostProcessor":
        return PostProcessor(self)

    def framerate_detector(self) -> "FrameRateDetector":
        return FrameRateDetector(self)

    def tuner(self) -> "Tuner":
        return Tuner(self)

    def channelizer(self) -> "Channelizer":
        return Channelizer(self)

    def scan(self) -> "Scan":
        return Scan(self)

    def notch(self) -> "Notch":
        return Notch(self)

    def spectrum(self) -> "Spectrum":
        return Spectrum(self)


def tuner_design(fs: int, offset_hz: float, bandwidth_hz: float, decimation: int = 1, ntaps: int = 0) -> Tuple[np.ndarray, int]:
    """tsdrgpu_tuner_design (host only): the float32 taps and the 64-bit phase increment round(offset / fs * 2^64) (as an
    unsigned integer) the tuner uses for this configuration.  Raises TsdrGpuError naming the violated rule."""
    taps = np.zeros(1023, np.float32)
    n, inc = C.c_int(0), C.c_uint64(0)
    N.check(N.lib().tsdrgpu_tuner_design(int(fs), float(offset_hz), float(bandwidth_hz), int(decimation), int(ntaps),
                                         taps.ctypes.data_as(C.c_void_p), taps.size, C.byref(n), C.byref(inc)))
    return taps[: n.value].copy(), inc.value


def tuner_out_pairs(position: int, pairs: int, dropped: int, decimation: int) -> Tuple[int, int]:
    """tsdrgpu_tuner_out_pairs (host only): (output pairs, output drop count) of a block."""
    o, od = C.c_uint64(0), C.c_uint64(0)
    N.check(N.lib().tsdrgpu_tuner_out_pairs(position, pairs, dropped, decimation, C.byref(o), C.byref(od)))
    return o.value, od.value


class Tuner:
    """The digital down-converter (tsdrgpu_tuner_*): shift by offset_hz, low-pass to bandwidth_hz, decimate by D."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        h = C.c_void_p()
        ctx.chk(ctx._lib.tsdrgpu_tuner_create(ctx._h, C.byref(h)))
        self._h = h
        self.config = None

    def __del__(self):
        try:
            if self._h:
                self.ctx._lib.tsdrgpu_tuner_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def configure(self, fs: int, offset_hz: float, bandwidth_hz: float, decimation: int = 1, ntaps: int = 0) -> None:
        """Design the filter for this configuration and reset (position 0, history zero)."""
        self.ctx.chk(self.ctx._lib.tsdrgpu_tuner_configure(self._h, int(fs), float(offset_hz), float(bandwidth_hz), int(decimation), int(ntaps)))
        self.config = (int(fs), float(offset_hz), float(bandwidth_hz), int(decimation), int(ntaps))

    @property
    def taps(self) -> np.ndarray:
        assert self.config is not None, "configure() first"
        return tuner_design(*self.config)[0]

    @property
    def phase_inc(self) -> int:
        assert self.config is not None, "configure() first"
        return tuner_design(*self.config)[1]

    def reset(self) -> None:
        self.ctx.chk(self.ctx._lib.tsdrgpu_tuner_reset(self._h, self.ctx.stream))

    def run(self, x: torch.Tensor, dropped: int = 0) -> Tuple[torch.Tensor, int]:
        """x: interleaved I,Q float32 on the device (the next block of the stream), preceded by `dropped` lost pairs.
        Returns (output I,Q pairs as a float32 tensor, output drop count)."""
        pairs = x.numel() // 2
        D = self.config[3]
        out = torch.empty(2 * (pairs // D + 2), dtype=torch.float32, device=self.ctx.device)
        o, od = C.c_uint64(0), C.c_uint64(0)
        self.ctx.chk(self.ctx._lib.tsdrgpu_tuner_run(self._h, self.ctx.stream, _f32(x).data_ptr() if pairs else None, pairs, int(dropped),
                                                     out.data_ptr(), C.byref(o), C.byref(od)))
        return out[: 2 * o.value], od.value


def channelizer_design(fs: int, channels: int, taps_per_channel: int = 0) -> np.ndarray:
    """tsdrgpu_channelizer_design (host only): the float32 prototype taps (Q*K - 1 of them).  Raises TsdrGpuError naming the
    violated rule."""
    taps = np.zeros(32 * 256, np.float32)
    n = C.c_int(0)
    N.check(N.lib().tsdrgpu_channelizer_design(int(fs), int(channels), int(taps_per_channel), taps.ctypes.data_as(C.c_void_p), taps.size,
                                               C.byref(n)))
    return taps[: n.value].copy()


def channelizer_out_pairs(position: int, pairs: int, dropped: int, channels: int) -> Tuple[int, int]:
    """tsdrgpu_channelizer_out_pairs (host only): (outputs per channel, output drop count) of a block."""
    o, od = C.c_uint64(0), C.c_uint64(0)
    N.check(N.lib().tsdrgpu_channelizer_out_pairs(position, pairs, dropped, channels, C.byref(o), C.byref(od)))
    return o.value, od.value


def channel_offsets(fs: int, channels: int) -> np.ndarray:
    """Centre of every channel in Hz: c fs / K for c < K/2, (c - K) fs / K otherwise."""
    c = np.arange(channels)
    return np.where(c < channels // 2, c, c - channels) * (fs / channels)


class Channelizer:
    """The polyphase filter bank (tsdrgpu_channelizer_*): K channels at offsets c fs / K, each decimated by K/2."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        h = C.c_void_p()
        ctx.chk(ctx._lib.tsdrgpu_channelizer_create(ctx._h, C.byref(h)))
        self._h = h
        self.config = None

    def __del__(self):
        try:
            if self._h:
                self.ctx._lib.tsdrgpu_channelizer_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def configure(self, fs: int, channels: int, taps_per_channel: int = 0) -> None:
        self.ctx.chk(self.ctx._lib.tsdrgpu_channelizer_configure(self._h, int(fs), int(channels), int(taps_per_channel)))
        self.config = (int(fs), int(channels), int(taps_per_channel))

    def reset(self) -> None:
        self.ctx.chk(self.ctx._lib.tsdrgpu_channelizer_reset(self._h, self.ctx.stream))

    def run(self, x: torch.Tensor, dropped: int = 0, magnitude: bool = False) -> Tuple[torch.Tensor, int]:
        """x: interleaved I,Q float32 on the device, preceded by `dropped` lost pairs.  Returns (outputs, output drop count): a
        [K, M, 2] float32 tensor of I,Q pairs, or [K, M] magnitudes."""
        pairs = x.numel() // 2
        K = self.config[1]
        stride = pairs // (K // 2) + 2
        out = torch.empty((K, stride, 1 if magnitude else 2), dtype=torch.float32, device=self.ctx.device)
        o, od = C.c_uint64(0), C.c_uint64(0)
        self.ctx.chk(self.ctx._lib.tsdrgpu_channelizer_run(self._h, self.ctx.stream, _f32(x).data_ptr() if pairs else None, pairs, int(dropped),
                                                           int(magnitude), out.data_ptr(), stride, C.byref(o), C.byref(od)))
        out = out[:, : o.value]
        return (out[..., 0] if magnitude else out), od.value


def scan_table(records, n: int):
    """tsdrgpu_scan_channel_t records -> list of dicts (with the channel number), sorted by frame_score, highest first."""
    rows = []
    for c in range(n):
        r = records[c]
        rows.append({"channel": c, **{f: getattr(r, f) for f, _ in N.ScanChannel._fields_}})
    return sorted(rows, key=lambda d: -d["frame_score"])


class Scan:
    """A frame-rate detector on every channel of a channelizer (tsdrgpu_scan_*): which sub-bands hold a raster, in which mode."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        h = C.c_void_p()
        ctx.chk(ctx._lib.tsdrgpu_scan_create(ctx._h, C.byref(h)))
        self._h = h
        self.channels = 0

    def __del__(self):
        try:
            if self._h:
                self.ctx._lib.tsdrgpu_scan_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def configure(self, fs: int, channels: int, taps_per_channel: int = 0) -> None:
        self.ctx.chk(self.ctx._lib.tsdrgpu_scan_configure(self._h, int(fs), int(channels), int(taps_per_channel)))
        self.channels = int(channels)

    def reset(self) -> None:
        self.ctx.chk(self.ctx._lib.tsdrgpu_scan_reset(self._h, self.ctx.stream))

    def run(self, x: torch.Tensor, dropped: int = 0) -> None:
        pairs = x.numel() // 2
        self.ctx.chk(self.ctx._lib.tsdrgpu_scan_run(self._h, self.ctx.stream, _f32(x).data_ptr() if pairs else None, pairs, int(dropped)))

    def records(self):
        """The raw table, channel order (ScanChannel structures)."""
        recs = (N.ScanChannel * self.channels)()
        self.ctx.chk(self.ctx._lib.tsdrgpu_scan_results(self._h, self.ctx.stream, recs, self.channels))
        return recs

    def results(self):
        """One dict per channel, sorted by frame_score, highest first."""
        return scan_table(self.records(), self.channels)

    def plots(self) -> Tuple[np.ndarray, int, int]:
        """The running means, [K, frame_len + line_len] float64, and the two window lengths."""
        fl, ll = C.c_int(0), C.c_int(0)
        self.ctx.chk(self.ctx._lib.tsdrgpu_scan_plots(self._h, self.ctx.stream, None, 0, C.byref(fl), C.byref(ll)))
        out = np.zeros((self.channels, fl.value + ll.value), np.float64)
        self.ctx.chk(self.ctx._lib.tsdrgpu_scan_plots(self._h, self.ctx.stream, out.ctypes.data_as(C.c_void_p), out.size, None, None))
        return out, fl.value, ll.value


class Resampler:
    """dsp_resample_t + dsp_resample_process (dsp.c:250-307), optionally fused with am_demod."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        h = C.c_void_p()
        ctx.chk(ctx._lib.tsdrgpu_resampler_create(ctx._h, C.byref(h)))
        self._h = h

    def __del__(self):
        try:
            if self._h:
                self.ctx._lib.tsdrgpu_resampler_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def reset(self):
        self.ctx.chk(self.ctx._lib.tsdrgpu_resampler_reset(self._h, self.ctx.stream))

    @property
    def state(self) -> Tuple[float, float]:
        c, o = C.c_double(0), C.c_double(0)
        self.ctx.chk(self.ctx._lib.tsdrgpu_resampler_get_state(self._h, self.ctx.stream, C.byref(c), C.byref(o)))
        return c.value, o.value

    @state.setter
    def state(self, co):
        self.ctx.chk(self.ctx._lib.tsdrgpu_resampler_set_state(self._h, self.ctx.stream, co[0], co[1]))

    @staticmethod
    def _blocks(block_sizes):
        if isinstance(block_sizes, tuple):           # (uniform_block, nblocks)
            return None, int(block_sizes[0]), int(block_sizes[1]), None
        arr = np.ascontiguousarray(block_sizes, dtype=np.uint32)
        return arr.ctypes.data_as(C.c_void_p), 0, int(arr.size), arr

    def plan(self, block_sizes, upsample_by: float, downsample_by: float) -> int:
        p, u, n, keep = self._blocks(block_sizes)
        return self.ctx._lib.tsdrgpu_resampler_plan(self._h, p, u, n, upsample_by, downsample_by)

    def process(self, x: torch.Tensor, block_sizes, upsample_by: float, downsample_by: float, nearest: bool = False,
                in_is_iq: bool = False, out: Optional[torch.Tensor] = None, mag_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Run consecutive decimator blocks.  block_sizes: sequence of sizes, or (uniform_block, nblocks).
        mag_out (IQ input only): also receives |x| of every input sample (am_demod's output for the frame-rate detector)."""
        p, u, n, keep = self._blocks(block_sizes)
        if mag_out is not None:
            self.ctx.chk(self.ctx._lib.tsdrgpu_resampler_set_mag_out(self._h, _f32(mag_out).data_ptr()))
        need = self.ctx._lib.tsdrgpu_resampler_plan(self._h, p, u, n, upsample_by, downsample_by)
        if out is None:
            out = torch.empty(max(int(need), 1), dtype=torch.float32, device=x.device)
        n_out = C.c_uint64(0)
        self.ctx.chk(self.ctx._lib.tsdrgpu_resampler_run(self._h, self.ctx.stream, _f32(x).data_ptr(), int(in_is_iq), p, u, n,
                                                         upsample_by, downsample_by, int(nearest), out.data_ptr(), out.numel(), C.byref(n_out)))
        return out[: n_out.value]


@dataclass
class PostProcessFlags:
    autoshift: bool = True            # PARAM_INT_AUTOSHIFT
    lowpass_before_sync: bool = True  # PARAM_LOW_PASS_BEFORE_SYNC
    autogain_after_proc: bool = False # PARAM_AUTOGAIN_AFTER_PROCESSING
    superresolution: bool = False     # PARAM_AUTOCORR_SUPERRESOLUTION
    compute_snr: bool = False

    def bits(self) -> int:
        return (N.FS_AUTOSHIFT * self.autoshift | N.FS_LOWPASS_BEFORE_SYNC * self.lowpass_before_sync |
                N.FS_AUTOGAIN_AFTER_PROC * self.autogain_after_proc | N.FS_SUPERRESOLUTION * self.superresolution |
                N.FS_COMPUTE_SNR * self.compute_snr)


class PostProcessor:
    """dsp_postprocess_t + dsp_post_process (dsp.c:112-239) for batches of frames."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        h = C.c_void_p()
        ctx.chk(ctx._lib.tsdrgpu_framestage_create(ctx._h, C.byref(h)))
        self._h = h

    def __del__(self):
        try:
            if self._h:
                self.ctx._lib.tsdrgpu_framestage_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def reset(self):
        self.ctx.chk(self.ctx._lib.tsdrgpu_framestage_reset(self._h, self.ctx.stream))

    def set_overlap(self, on: bool):
        """Run the sync search + re-centring of batch k on a side stream under batch k+1 (see tsdrgpu.h); outputs are
        valid after :meth:`join`."""
        self.ctx.chk(self.ctx._lib.tsdrgpu_framestage_set_overlap(self._h, int(on)))

    def join(self):
        self.ctx.chk(self.ctx._lib.tsdrgpu_framestage_join(self._h, self.ctx.stream))

    def process(self, frames: torch.Tensor, width: int, height: int, motionblur: float = 0.0, lowpasscoeff: float = 0.1,
                flags: PostProcessFlags = PostProcessFlags(), out: Optional[torch.Tensor] = None, want_results: bool = True):
        """frames: nframes*width*height float32, frames back to back.  Returns (frames_out, [FrameResult])."""
        nframes = frames.numel() // (width * height)
        assert nframes * width * height == frames.numel()
        if out is None:
            out = torch.empty_like(frames)
        res = (FrameResult * nframes)() if want_results else None
        self.ctx.chk(self.ctx._lib.tsdrgpu_framestage_run(self._h, self.ctx.stream, _f32(frames).data_ptr(), nframes, width, height,
                                                          motionblur, lowpasscoeff, flags.bits(), out.data_ptr(), res))
        return out, (list(res) if want_results else None)


class FrameRateDetector:
    """frameratedetector_runontodata + the two running-mean plots (frameratedetector.c:87-126)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        h = C.c_void_p()
        ctx.chk(ctx._lib.tsdrgpu_frd_create(ctx._h, C.byref(h)))
        self._h = h

    def __del__(self):
        try:
            if self._h:
                self.ctx._lib.tsdrgpu_frd_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def reset(self):
        self.ctx._lib.tsdrgpu_frd_reset(self._h)

    def set_overlap(self, on: bool) -> None:
        """Runs go to the detector's own stream and work buffers (tsdrgpu_frd_set_overlap); see :meth:`join`."""
        self.ctx.chk(self.ctx._lib.tsdrgpu_frd_set_overlap(self._h, 1 if on else 0))

    def join(self) -> None:
        """The context's stream waits (on the device) for the last overlapped run: call before the capture memory is reused."""
        self.ctx.chk(self.ctx._lib.tsdrgpu_frd_join(self._h, self.ctx.stream))

    @staticmethod
    def capture_size(samplerate: int) -> int:
        return N.lib().tsdrgpu_frd_capture_size(samplerate)

    @staticmethod
    def windows(samplerate: int) -> Tuple[int, int, int, int]:
        v = [C.c_int(0) for _ in range(4)]
        N.lib().tsdrgpu_frd_windows(samplerate, *[C.byref(x) for x in v])
        return tuple(x.value for x in v)

    def run_batch(self, samplerate: int, captures: torch.Tensor, size: int, batch: int, stride: Optional[int] = None) -> int:
        """`batch` consecutive captures of `size` samples (capture b at captures[b*stride:]) accumulated in order;
        asynchronous, the plots stay on the device (see :meth:`plots`)."""
        calls = C.c_uint64(0)
        self.ctx.chk(self.ctx._lib.tsdrgpu_frd_run_batch(self._h, self.ctx.stream, samplerate, _f32(captures).data_ptr(), size, batch,
                                                         stride if stride is not None else size, C.byref(calls)))
        return calls.value

    def dump_csv(self, samplerate: int, capture: torch.Tensor, path: str) -> None:
        """dump_autocorrect (frameratedetector.c:64-85) of one capture."""
        self.ctx.chk(self.ctx._lib.tsdrgpu_frd_dump_csv(self._h, self.ctx.stream, samplerate, _f32(capture).data_ptr(), capture.numel(), path.encode()))

    def plots(self, samplerate: int):
        fmin, fmax, lmin, lmax = self.windows(samplerate)
        fp, lp = np.zeros(fmax - fmin), np.zeros(lmax - lmin)
        self.ctx.chk(self.ctx._lib.tsdrgpu_frd_get_plots(self._h, self.ctx.stream, samplerate, fp.ctypes.data_as(C.c_void_p), fp.size,
                                                         lp.ctypes.data_as(C.c_void_p), lp.size))
        return (fmin, fp), (lmin, lp)

    def run(self, samplerate: int, capture: torch.Tensor, copy_out: bool = True):
        fmin, fmax, lmin, lmax = self.windows(samplerate)
        fp = np.zeros(fmax - fmin) if copy_out else None
        lp = np.zeros(lmax - lmin) if copy_out else None
        calls = C.c_uint64(0)
        self.ctx.chk(self.ctx._lib.tsdrgpu_frd_run(self._h, self.ctx.stream, samplerate, _f32(capture).data_ptr(), capture.numel(),
                                                   fp.ctypes.data_as(C.c_void_p) if copy_out else None, fmax - fmin,
                                                   lp.ctypes.data_as(C.c_void_p) if copy_out else None, lmax - lmin, C.byref(calls)))
        return (fmin, fp), (lmin, lp), calls.value


def _bands(centers: Sequence[float], widths: Sequence[float]):
    c = np.ascontiguousarray(centers, dtype=np.float64)
    w = np.ascontiguousarray(widths, dtype=np.float64)
    assert c.shape == w.shape and c.ndim == 1, "one width per center"
    return c, w


def notch_design(fs: int, centers: Sequence[float], widths: Sequence[float], ntaps: int = 0) -> Tuple[np.ndarray, int]:
    """tsdrgpu_notch_design (host only): the complex64 taps of the notch filter and its FFT size N.  Raises TsdrGpuError naming
    the violated rule."""
    c, w = _bands(centers, widths)
    n, nfft = C.c_int(0), C.c_int(0)
    N.check(N.lib().tsdrgpu_notch_design(int(fs), c.size, c.ctypes.data_as(C.c_void_p), w.ctypes.data_as(C.c_void_p), int(ntaps),
                                         None, 0, C.byref(n), C.byref(nfft)))
    taps = np.zeros(2 * n.value, np.float32)
    N.check(N.lib().tsdrgpu_notch_design(int(fs), c.size, c.ctypes.data_as(C.c_void_p), w.ctypes.data_as(C.c_void_p), int(ntaps),
                                         taps.ctypes.data_as(C.c_void_p), n.value, None, None))
    return taps.view(np.complex64).copy(), nfft.value


class Notch:
    """The notch filter (tsdrgpu_notch_*): removes the stopbands (center, width) from the stream, one output per input pair."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        h = C.c_void_p()
        ctx.chk(ctx._lib.tsdrgpu_notch_create(ctx._h, C.byref(h)))
        self._h = h
        self.config = None

    def __del__(self):
        try:
            if self._h:
                self.ctx._lib.tsdrgpu_notch_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def configure(self, fs: int, centers: Sequence[float], widths: Sequence[float], ntaps: int = 0) -> None:
        """Design the filter for these stopbands and reset (position 0, history zero)."""
        c, w = _bands(centers, widths)
        self.ctx.chk(self.ctx._lib.tsdrgpu_notch_configure(self._h, int(fs), c.size, c.ctypes.data_as(C.c_void_p), w.ctypes.data_as(C.c_void_p),
                                                           int(ntaps)))
        self.config = (int(fs), c.copy(), w.copy(), int(ntaps))

    def taps(self) -> np.ndarray:
        """The complex64 taps in use."""
        assert self.config is not None, "configure() first"
        return notch_design(*self.config)[0]

    @property
    def nfft(self) -> int:
        assert self.config is not None, "configure() first"
        return notch_design(*self.config)[1]

    def reset(self) -> None:
        self.ctx.chk(self.ctx._lib.tsdrgpu_notch_reset(self._h, self.ctx.stream))

    def run(self, x: torch.Tensor, dropped: int = 0) -> Tuple[torch.Tensor, int]:
        """x: interleaved I,Q float32 on the device (the next block of the stream), preceded by `dropped` lost pairs.
        Returns (the filtered I,Q pairs, as many as x holds, and the drop count, unchanged)."""
        pairs = x.numel() // 2
        out = torch.empty(2 * pairs, dtype=torch.float32, device=self.ctx.device)
        o, od = C.c_uint64(0), C.c_uint64(0)
        self.ctx.chk(self.ctx._lib.tsdrgpu_notch_run(self._h, self.ctx.stream, _f32(x).data_ptr() if pairs else None, pairs, int(dropped),
                                                     out.data_ptr() if pairs else None, C.byref(o), C.byref(od)))
        return out[: 2 * o.value], od.value


def spectrum_freqs(fs: int, nfft: int) -> np.ndarray:
    """The frequencies of the spectrum's bins, fft-shifted: -fs/2 .. fs/2 - fs/nfft."""
    return (np.arange(nfft) - nfft // 2) * (fs / max(nfft, 1))


class Spectrum:
    """Welch's power spectral density of the stream (tsdrgpu_spectrum_*): Hann window, half-overlapping segments, drops skipped."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        h = C.c_void_p()
        ctx.chk(ctx._lib.tsdrgpu_spectrum_create(ctx._h, C.byref(h)))
        self._h = h
        self.config = None

    def __del__(self):
        try:
            if self._h:
                self.ctx._lib.tsdrgpu_spectrum_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def configure(self, fs: int, nfft: int = 4096) -> None:
        self.ctx.chk(self.ctx._lib.tsdrgpu_spectrum_configure(self._h, int(fs), int(nfft)))
        self.config = (int(fs), int(nfft))

    def reset(self) -> None:
        self.ctx.chk(self.ctx._lib.tsdrgpu_spectrum_reset(self._h, self.ctx.stream))

    def run(self, x: torch.Tensor, dropped: int = 0) -> None:
        pairs = x.numel() // 2
        self.ctx.chk(self.ctx._lib.tsdrgpu_spectrum_run(self._h, self.ctx.stream, _f32(x).data_ptr() if pairs else None, pairs, int(dropped)))

    def result(self) -> Tuple[np.ndarray, np.ndarray, int]:
        """(frequencies in Hz, density per Hz, segments averaged), fft-shifted."""
        assert self.config is not None, "configure() first"
        fs, nfft = self.config
        psd = np.zeros(nfft, np.float64)
        segs = C.c_uint64(0)
        self.ctx.chk(self.ctx._lib.tsdrgpu_spectrum_results(self._h, self.ctx.stream, psd.ctypes.data_as(C.c_void_p), nfft, C.byref(segs)))
        return spectrum_freqs(fs, nfft), psd, segs.value
