"""Python face of the streaming pipeline (tsdrgpu_pipeline_*): host IQ blocks in, host frames / plots out.

Mirrors what a host of the reference sees: ``process(buf, samples_dropped)`` is the plugin callback
(TSDRPlugin.h:49), ``on_frame`` is tsdr_readasync_function, ``on_value`` / ``on_plot`` are the two tsdr_init
callbacks (TSDRLibrary.h:57-59).  Callbacks run on the library's delivery thread.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Dict, Optional

import numpy as np

from . import _native as N

RAW_FORMATS = {"float32": 0, "int8": 1, "int16": 2, "uint8": 3, "uint16": 4}     # TSDRPlugin_RawFile.c:29-33
PARAM_IDS = {"autoshift": 0, "framerate_pll": 1, "autocorr_plots_reset": 2, "autocorr_plots_off": 3,
             "superresolution": 4, "nearest_neighbour_resampling": 5, "lowpass_before_sync": 6,
             "autogain_after_processing": 7, "autocorr_dump": 8}


class Pipeline:
    def __init__(self, samplerate: int, height: int, refreshrate: float, motionblur: float = 0.0,
                 params: Optional[Dict[str, int]] = None, batch_frames: int = 1, batch_blocks: int = 10,
                 block_when_busy: bool = False, device: int = 0,
                 on_frame: Optional[Callable] = None, on_value: Optional[Callable] = None, on_plot: Optional[Callable] = None,
                 on_retune: Optional[Callable] = None):
        self._lib = N.lib()
        self._samplerate = int(samplerate)
        ctx = C.c_void_p()
        N.check(self._lib.tsdrgpu_create(C.byref(ctx), device))
        self._ctx = ctx
        cfg = N.PipelineConfig()
        cfg.samplerate, cfg.height, cfg.refreshrate, cfg.motionblur = samplerate, height, refreshrate, motionblur
        for k, v in (params or {}).items():
            cfg.params_int[PARAM_IDS[k]] = int(v)
        cfg.batch_frames, cfg.batch_blocks, cfg.block_when_busy = batch_frames, batch_blocks, int(block_when_busy)
        self.errors = []

        def _frame(buf, w, h, _):
            try:
                if on_frame:
                    on_frame(np.ctypeslib.as_array(buf, shape=(w * h,)), w, h)
            except Exception as e:      # never let an exception cross the C boundary
                self.errors.append(e)

        def _value(vid, a, b, _):
            try:
                if on_value:
                    on_value(vid, a, b)
            except Exception as e:
                self.errors.append(e)

        def _plot(pid, off, vals, size, sr, _):
            try:
                if on_plot:
                    on_plot(pid, off, np.ctypeslib.as_array(vals, shape=(size,)), sr)
            except Exception as e:
                self.errors.append(e)

        self._cbs = (N.FRAME_CB(_frame), N.VALUE_CB(_value), N.PLOT_CB(_plot))    # keep alive
        h = C.c_void_p()
        N.check(self._lib.tsdrgpu_pipeline_create(ctx, C.byref(cfg), *self._cbs, None, C.byref(h)), ctx)
        self._h = h
        if on_retune:
            def _retune(off, _):
                try:
                    on_retune(off)
                except Exception as e:
                    self.errors.append(e)
            self._retune_cb = N.RETUNE_CB(_retune)
            N.check(self._lib.tsdrgpu_pipeline_set_retune(h, self._retune_cb), ctx)

    def process(self, iq: np.ndarray, samples_dropped: int = 0) -> None:
        """iq: interleaved float32 I,Q on the HOST (numpy, or a pinned torch tensor's .numpy())."""
        assert iq.dtype == np.float32 and iq.flags.c_contiguous
        N.check(self._lib.tsdrgpu_pipeline_process(self._h, iq.ctypes.data_as(C.c_void_p), iq.size, samples_dropped), self._ctx)

    def process_ptr(self, ptr: int, items: int, samples_dropped: int = 0) -> None:
        N.check(self._lib.tsdrgpu_pipeline_process(self._h, C.c_void_p(ptr), items, samples_dropped), self._ctx)

    def process_raw(self, samples: np.ndarray, samples_dropped: int = 0) -> None:
        """samples: interleaved I,Q on the HOST still in the front end's wire format (int8 / uint8 / int16 / uint16 /
        float32); converted on the device to the floats TSDRPlugin_RawFile.c:241-261 produces on the host."""
        fmt = RAW_FORMATS[samples.dtype.name]
        assert samples.flags.c_contiguous
        N.check(self._lib.tsdrgpu_pipeline_process_raw(self._h, samples.ctypes.data_as(C.c_void_p), fmt, samples.size, samples_dropped), self._ctx)

    def process_raw_ptr(self, ptr: int, fmt: int, items: int, samples_dropped: int = 0) -> None:
        N.check(self._lib.tsdrgpu_pipeline_process_raw(self._h, C.c_void_p(ptr), fmt, items, samples_dropped), self._ctx)

    def process_raw_ptr_async(self, ptr: int, fmt: int, items: int, samples_dropped: int = 0) -> None:
        """Page-locked buffers only: returns once enqueued; the buffer must stay untouched until sync_input()."""
        N.check(self._lib.tsdrgpu_pipeline_process_raw_async(self._h, C.c_void_p(ptr), fmt, items, samples_dropped), self._ctx)

    def sync_input(self) -> None:
        N.check(self._lib.tsdrgpu_pipeline_sync_input(self._h), self._ctx)

    def flush(self) -> None:
        N.check(self._lib.tsdrgpu_pipeline_flush(self._h), self._ctx)
        if self.errors:
            raise self.errors[0]

    def set_output_argb(self, on: bool, inverted: bool = False) -> None:
        """Deliver the JNI glue's int32 pixels (TSDRLibraryNDK.c:222-283) instead of floats; on_frame then receives the
        same float32 array object whose bytes are int32 pixels: use frame.view(np.int32)."""
        N.check(self._lib.tsdrgpu_pipeline_set_output_argb(self._h, int(on), int(inverted)), self._ctx)

    def set_reports(self, snr: bool = False, detect_mode: bool = False) -> None:
        """on_value then also receives (4, snr, 0) beside every auto-gain report and (100, fps, height) after every pair of plots."""
        N.check(self._lib.tsdrgpu_pipeline_set_reports(self._h, int(snr), int(detect_mode)), self._ctx)

    def set_param(self, name: str, value: int) -> None:
        N.check(self._lib.tsdrgpu_pipeline_set_param_int(self._h, PARAM_IDS[name], value), self._ctx)

    def set_resolution(self, height: int, refreshrate: float) -> None:
        N.check(self._lib.tsdrgpu_pipeline_set_resolution(self._h, height, refreshrate), self._ctx)

    def set_tuner(self, offset_hz: float, bandwidth_hz: float, decimation: int = 1, ntaps: int = 0) -> None:
        """Demodulate only the sub-band of `bandwidth_hz` around `offset_hz`, decimated by `decimation` (the pipeline then runs
        at samplerate / decimation); bandwidth_hz <= 0 switches the tuner off.  Takes effect at the next process() call."""
        N.check(self._lib.tsdrgpu_pipeline_set_tuner(self._h, float(offset_hz), float(bandwidth_hz), int(decimation), int(ntaps)), self._ctx)

    def set_scan(self, channels: int, taps_per_channel: int = 0) -> None:
        """Run a frame-rate detector on each of `channels` sub-bands of the wideband blocks (0 switches it off).  Takes effect,
        reset, at the next process() call; the pixel path is not affected."""
        N.check(self._lib.tsdrgpu_pipeline_set_scan(self._h, int(channels), int(taps_per_channel)), self._ctx)

    def scan_results(self):
        """The scan's table: one dict per channel, sorted by frame_score, highest first (empty while no scan runs)."""
        from .api import scan_table
        recs = (N.ScanChannel * 256)()
        n = C.c_int(0)
        N.check(self._lib.tsdrgpu_pipeline_scan_results(self._h, recs, 256, C.byref(n)), self._ctx)
        return scan_table(recs, n.value)

    def set_notches(self, centers, widths, ntaps: int = 0) -> None:
        """Remove the stopbands (centers[j], widths[j]) in Hz from every block before anything else reads it (empty lists switch
        the notch off).  Takes effect at the next process() call, which starts the stream over behind the notch."""
        c = np.ascontiguousarray(centers, dtype=np.float64)
        w = np.ascontiguousarray(widths, dtype=np.float64)
        assert c.shape == w.shape and c.ndim == 1, "one width per center"
        N.check(self._lib.tsdrgpu_pipeline_set_notches(self._h, c.size, c.ctypes.data_as(C.c_void_p), w.ctypes.data_as(C.c_void_p),
                                                       int(ntaps)), self._ctx)

    def set_spectrum(self, nfft: int) -> None:
        """Accumulate the power spectrum of the blocks as received, with nfft bins (0 switches it off).  Takes effect, reset, at the
        next process() call; the pixel path is not affected."""
        N.check(self._lib.tsdrgpu_pipeline_set_spectrum(self._h, int(nfft)), self._ctx)

    def spectrum(self):
        """(frequencies in Hz, density per Hz, segments averaged), fft-shifted; empty arrays while no spectrum runs."""
        from .api import spectrum_freqs
        nfft = 16384
        psd = np.zeros(nfft, np.float64)
        n, segs = C.c_int(0), C.c_uint64(0)
        N.check(self._lib.tsdrgpu_pipeline_spectrum(self._h, psd.ctypes.data_as(C.c_void_p), nfft, C.byref(n), C.byref(segs)), self._ctx)
        fs = self._samplerate
        return spectrum_freqs(fs, n.value), psd[: n.value].copy(), segs.value

    def set_samplerate(self, samplerate: int) -> None:
        N.check(self._lib.tsdrgpu_pipeline_set_samplerate(self._h, int(samplerate)), self._ctx)
        self._samplerate = int(samplerate)

    def set_superb_devices(self, devices) -> None:
        """Superbandwidth mode with one hop per GPU: devices[0] is this pipeline's device, len(devices) in {2, 4, 8} = hops."""
        arr = (C.c_int * len(devices))(*devices)
        N.check(self._lib.tsdrgpu_pipeline_set_superb_devices(self._h, arr, len(devices)), self._ctx)

    def set_motionblur(self, coeff: float) -> None:
        N.check(self._lib.tsdrgpu_pipeline_set_motionblur(self._h, coeff), self._ctx)

    def sync(self, pixels: int) -> None:
        N.check(self._lib.tsdrgpu_pipeline_sync(self._h, pixels), self._ctx)

    def geometry(self):
        w, h, fv = C.c_int(0), C.c_int(0), C.c_double(0)
        N.check(self._lib.tsdrgpu_pipeline_get_geometry(self._h, C.byref(w), C.byref(h), C.byref(fv)), self._ctx)
        return w.value, h.value, fv.value

    def stats(self) -> N.PipelineStats:
        s = N.PipelineStats()
        N.check(self._lib.tsdrgpu_pipeline_stats(self._h, C.byref(s)), self._ctx)
        return s

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.tsdrgpu_pipeline_destroy(self._h)
            self._h = None
            self._lib.tsdrgpu_destroy(self._ctx)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
