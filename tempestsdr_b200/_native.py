"""ctypes loader of tempestsdr_b200/lib/libtsdrgpu.so (the C-ABI of include/tsdrgpu.h).

There is no fallback of any kind: a missing library or a missing CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libtsdrgpu.so")

OK = 0


class FrameResult(C.Structure):
    """tsdrgpu_frame_result_t"""
    _fields_ = [("x_dx", C.c_int32), ("x_vx", C.c_int32), ("x_absvx", C.c_int32), ("x_stripsize", C.c_int32),
                ("y_dx", C.c_int32), ("y_vx", C.c_int32), ("y_absvx", C.c_int32), ("y_stripsize", C.c_int32),
                ("avg_speed", C.c_double), ("pll_state", C.c_int32),
                ("lastmax", C.c_float), ("lastmin", C.c_float), ("snr", C.c_float),
                ("autogain_report", C.c_int32), ("reserved", C.c_int32)]


class PipelineConfig(C.Structure):
    """tsdrgpu_pipeline_config_t"""
    _fields_ = [("samplerate", C.c_uint32), ("height", C.c_int), ("refreshrate", C.c_double), ("motionblur", C.c_float),
                ("params_int", C.c_uint32 * 9), ("batch_frames", C.c_int), ("batch_blocks", C.c_int), ("block_when_busy", C.c_int)]


class PipelineStats(C.Structure):
    """tsdrgpu_pipeline_stats_t"""
    _fields_ = [(n, C.c_uint64) for n in ("samples_in", "samples_dropped_upstream", "samples_resampled", "frames_processed",
                                          "frames_delivered", "frames_dropped", "captures", "plots_delivered",
                                          "h2d_bytes", "d2h_bytes", "gpu_launches", "stitches", "host_buffers_registered")]


class ScanChannel(C.Structure):
    """tsdrgpu_scan_channel_t"""
    _fields_ = [("offset_hz", C.c_double), ("rate", C.c_uint32), ("captures", C.c_uint64), ("frame_index", C.c_int32),
                ("line_index", C.c_int32), ("fps", C.c_double), ("height", C.c_int32), ("frame_score", C.c_double),
                ("line_score", C.c_double)]


FRAME_CB = C.CFUNCTYPE(None, C.POINTER(C.c_float), C.c_int, C.c_int, C.c_void_p)
VALUE_CB = C.CFUNCTYPE(None, C.c_int, C.c_double, C.c_double, C.c_void_p)
PLOT_CB = C.CFUNCTYPE(None, C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_uint32, C.c_void_p)
RETUNE_CB = C.CFUNCTYPE(None, C.c_int32, C.c_void_p)

FS_AUTOSHIFT, FS_LOWPASS_BEFORE_SYNC, FS_AUTOGAIN_AFTER_PROC, FS_SUPERRESOLUTION, FS_COMPUTE_SNR = 1, 2, 4, 8, 16

_SIGS = {
    "tsdrgpu_device_count": (C.c_int, []),
    "tsdrgpu_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "tsdrgpu_destroy": (None, [C.c_void_p]),
    "tsdrgpu_last_error": (C.c_char_p, [C.c_void_p]),
    "tsdrgpu_sm_count": (C.c_int, [C.c_void_p]),
    "tsdrgpu_launch_count": (C.c_uint64, [C.c_void_p]),
    "tsdrgpu_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "tsdrgpu_profile_collect": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.c_int, C.POINTER(C.c_int)]),
    "tsdrgpu_malloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "tsdrgpu_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_malloc_host": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "tsdrgpu_free_host": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tsdrgpu_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tsdrgpu_memcpy_d2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tsdrgpu_device_numa_node": (C.c_int, [C.c_void_p]),
    "tsdrgpu_bind_thread_near_device": (C.c_int, [C.c_void_p]),
    "tsdrgpu_memset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_size_t]),
    "tsdrgpu_stream_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "tsdrgpu_stream_destroy": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_stream_sync": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_geometry": (None, [C.c_uint32, C.c_int, C.c_double, C.POINTER(C.c_int), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "tsdrgpu_plan_resample": (C.c_uint64, [C.POINTER(C.c_double), C.c_void_p, C.c_uint32, C.c_uint32, C.c_double, C.c_double, C.c_void_p]),
    "tsdrgpu_fft_reference_eps": (None, [C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "tsdrgpu_gauss_taps": (None, [C.POINTER(C.c_float * 5)]),
    "tsdrgpu_pll_step": (C.c_int, [C.POINTER(C.c_double), C.c_int32, C.c_int32, C.c_double]),
    "tsdrgpu_am_demod": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "tsdrgpu_resampler_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "tsdrgpu_resampler_destroy": (None, [C.c_void_p]),
    "tsdrgpu_resampler_reset": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_resampler_get_state": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "tsdrgpu_resampler_set_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_double, C.c_double]),
    "tsdrgpu_resampler_plan": (C.c_uint64, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_double, C.c_double]),
    "tsdrgpu_resampler_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_uint32, C.c_uint32,
                                        C.c_double, C.c_double, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "tsdrgpu_resampler_set_mag_out": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_framestage_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "tsdrgpu_framestage_destroy": (None, [C.c_void_p]),
    "tsdrgpu_framestage_reset": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_framestage_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float,
                                         C.c_uint, C.c_void_p, C.POINTER(FrameResult)]),
    "tsdrgpu_framestage_run_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float,
                                               C.c_uint, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tsdrgpu_framestage_set_overlap": (C.c_int, [C.c_void_p, C.c_int]),
    "tsdrgpu_framestage_join": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_autogain": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float),
                                   C.c_int, C.c_void_p, C.c_void_p, C.c_float]),
    "tsdrgpu_timelowpass": (C.c_int, [C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_void_p]),
    "tsdrgpu_average_v_h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tsdrgpu_gaussianblur": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "tsdrgpu_pixels_argb": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "tsdrgpu_fft_getrealsize": (C.c_uint32, [C.c_uint32]),
    "tsdrgpu_fft": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int]),
    "tsdrgpu_autocorrelation": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]),
    "tsdrgpu_autocorrelation_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64]),
    "tsdrgpu_crosscorrelation": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]),
    "tsdrgpu_frd_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "tsdrgpu_frd_destroy": (None, [C.c_void_p]),
    "tsdrgpu_frd_reset": (C.c_int, [C.c_void_p]),
    "tsdrgpu_frd_set_overlap": (C.c_int, [C.c_void_p, C.c_int]),
    "tsdrgpu_frd_join": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_frd_capture_size": (C.c_uint32, [C.c_uint32]),
    "tsdrgpu_frd_windows": (None, [C.c_uint32] + [C.POINTER(C.c_int)] * 4),
    "tsdrgpu_frd_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_int,
                                  C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]),
    "tsdrgpu_frd_run_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_int,
                                        C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]),
    "tsdrgpu_frd_run_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(C.c_uint64)]),
    "tsdrgpu_frd_dump_csv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_char_p]),
    "tsdrgpu_frd_get_plots": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "tsdrgpu_frd_peaks": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int32)]),
    "tsdrgpu_plot_peaks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int32)]),
    "tsdrgpu_frd_peaks_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "tsdrgpu_videomode_from_peaks": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "tsdrgpu_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int, C.c_int]),
    "tsdrgpu_complex_to_abs_diff": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "tsdrgpu_superb_bestfit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "tsdrgpu_superb_stitch": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_void_p,
                                        C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "tsdrgpu_superb_hop_spectrum": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "tsdrgpu_superb_local_spectra": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "tsdrgpu_superb_lags": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_int)]),
    "tsdrgpu_superb_residue_ifft_lag": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_uint32, C.c_int, C.POINTER(C.c_int), C.c_void_p]),
    "tsdrgpu_superb_residue_ifft": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint32, C.c_int, C.c_void_p]),
    "tsdrgpu_superb_mgpu_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.POINTER(C.c_void_p)]),
    "tsdrgpu_superb_mgpu_destroy": (None, [C.c_void_p]),
    "tsdrgpu_superb_mgpu_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_superb_mgpu_connect_ipc": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_superb_mgpu_connect_local": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "tsdrgpu_superb_mgpu_disconnect": (C.c_int, [C.c_void_p]),
    "tsdrgpu_superb_mgpu_stitch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_uint32)]),
    "tsdrgpu_superb_mgpu_stream_window": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "tsdrgpu_superb_mgpu_lags": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_uint32)]),
    "tsdrgpu_pipeline_create": (C.c_int, [C.c_void_p, C.POINTER(PipelineConfig), FRAME_CB, VALUE_CB, PLOT_CB, C.c_void_p, C.POINTER(C.c_void_p)]),
    "tsdrgpu_pipeline_destroy": (None, [C.c_void_p]),
    "tsdrgpu_pipeline_process": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int64]),
    "tsdrgpu_convert_samples": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_void_p]),
    "tsdrgpu_pipeline_process_raw": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_int64]),
    "tsdrgpu_pipeline_process_raw_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_int64]),
    "tsdrgpu_pipeline_sync_input": (C.c_int, [C.c_void_p]),
    "tsdrgpu_pipeline_flush": (C.c_int, [C.c_void_p]),
    "tsdrgpu_pipeline_set_param_int": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32]),
    "tsdrgpu_pipeline_set_resolution": (C.c_int, [C.c_void_p, C.c_int, C.c_double]),
    "tsdrgpu_pipeline_set_samplerate": (C.c_int, [C.c_void_p, C.c_uint32]),
    "tsdrgpu_pipeline_set_tuner": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_int, C.c_int]),
    "tsdrgpu_tuner_design": (C.c_int, [C.c_uint32, C.c_double, C.c_double, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                       C.POINTER(C.c_int), C.POINTER(C.c_uint64)]),
    "tsdrgpu_tuner_out_pairs": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "tsdrgpu_tuner_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "tsdrgpu_tuner_destroy": (None, [C.c_void_p]),
    "tsdrgpu_tuner_configure": (C.c_int, [C.c_void_p, C.c_uint32, C.c_double, C.c_double, C.c_int, C.c_int]),
    "tsdrgpu_tuner_reset": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_tuner_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p,
                                    C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "tsdrgpu_channelizer_design": (C.c_int, [C.c_uint32, C.c_int, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "tsdrgpu_channelizer_out_pairs": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "tsdrgpu_channelizer_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "tsdrgpu_channelizer_destroy": (None, [C.c_void_p]),
    "tsdrgpu_channelizer_configure": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, C.c_int]),
    "tsdrgpu_channelizer_reset": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_channelizer_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64,
                                          C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "tsdrgpu_scan_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "tsdrgpu_scan_destroy": (None, [C.c_void_p]),
    "tsdrgpu_scan_configure": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, C.c_int]),
    "tsdrgpu_scan_reset": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_scan_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]),
    "tsdrgpu_scan_results": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(ScanChannel), C.c_int]),
    "tsdrgpu_scan_plots": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "tsdrgpu_pipeline_set_scan": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "tsdrgpu_pipeline_scan_results": (C.c_int, [C.c_void_p, C.POINTER(ScanChannel), C.c_int, C.POINTER(C.c_int)]),
    "tsdrgpu_notch_design": (C.c_int, [C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int),
                                       C.POINTER(C.c_int)]),
    "tsdrgpu_notch_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "tsdrgpu_notch_destroy": (None, [C.c_void_p]),
    "tsdrgpu_notch_configure": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "tsdrgpu_notch_reset": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_notch_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p,
                                    C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "tsdrgpu_spectrum_check": (C.c_int, [C.c_uint32, C.c_int]),
    "tsdrgpu_spectrum_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "tsdrgpu_spectrum_destroy": (None, [C.c_void_p]),
    "tsdrgpu_spectrum_configure": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int]),
    "tsdrgpu_spectrum_reset": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_spectrum_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]),
    "tsdrgpu_spectrum_results": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]),
    "tsdrgpu_pipeline_set_notches": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "tsdrgpu_pipeline_set_spectrum": (C.c_int, [C.c_void_p, C.c_int]),
    "tsdrgpu_pipeline_spectrum": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_uint64)]),
    "tsdrgpu_pipeline_set_retune": (C.c_int, [C.c_void_p, RETUNE_CB]),
    "tsdrgpu_pipeline_set_motionblur": (C.c_int, [C.c_void_p, C.c_float]),
    "tsdrgpu_pipeline_set_host_registration": (C.c_int, [C.c_void_p, C.c_int]),
    "tsdrgpu_pipeline_set_superb_devices": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.c_int]),
    "tsdrgpu_ipc_export": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "tsdrgpu_ipc_import": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "tsdrgpu_ipc_release": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsdrgpu_superb_local_spectra_scatter": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.c_int, C.c_int,
                                                       C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "tsdrgpu_pipeline_set_reports": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "tsdrgpu_detect_videomode": (C.c_int, [C.POINTER(C.c_double), C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_int, C.c_uint32,
                                           C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "tsdrgpu_pipeline_set_output_argb": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "tsdrgpu_pixels_argb_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_void_p]),
    "tsdrgpu_pipeline_sync": (C.c_int, [C.c_void_p, C.c_int]),
    "tsdrgpu_pipeline_get_geometry": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_double)]),
    "tsdrgpu_pipeline_stats": (C.c_int, [C.c_void_p, C.POINTER(PipelineStats)]),
}

#: every symbol include/tsdrgpu.h declares (tests check the built library exports all of them)
DECLARED_SYMBOLS = tuple(_SIGS)

_lib = None


def lib() -> C.CDLL:
    """The loaded libtsdrgpu.so.  Raises if it has not been built (python -c 'import __graft_entry__ as g; g.build()')."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `make -C tempestsdr_b200/csrc` "
                               "(or __graft_entry__.build()).  There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class TsdrGpuError(RuntimeError):
    pass


def check(rc: int, ctx=None) -> None:
    if rc != OK:
        msg = lib().tsdrgpu_last_error(ctx)
        raise TsdrGpuError(f"libtsdrgpu error {rc}: {msg.decode() if msg else '?'}")
