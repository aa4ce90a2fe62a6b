/*
 * tsdrgpu.h -- C-ABI of the B200 (sm_100a) implementation of TempestSDR's IQ->raster DSP path.
 *
 * This is the drop-in boundary below the reference's own C host code: plain C, plain pointers and sizes, no
 * C++ or torch types.  Every entry point names the reference function(s) it replaces
 * (paths relative to /root/reference/TempestSDR/src).  The tsdr_* / tsdrplugin_* ABI above it is declared
 * unchanged in TSDRLibrary.h / TSDRPlugin.h / TSDRCodes.h beside this file.
 *
 * Conventions
 *   - every function returns TSDRGPU_OK (0) or a negative TSDRGPU_E* code; tsdrgpu_last_error() gives text;
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream); calls are asynchronous on
 *     that stream unless the comment says "synchronises";
 *   - pointers named d_* are device pointers on the context's device, h_* are host pointers;
 *   - there is NO CPU fallback: without a CUDA device every call fails with TSDRGPU_ENODEVICE.
 */
#ifndef TSDRGPU_H_
#define TSDRGPU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define TSDRGPU_API __attribute__((visibility("default")))
#else
#define TSDRGPU_API
#endif

enum {
	TSDRGPU_OK        = 0,
	TSDRGPU_ENODEVICE = -1,   /* no usable CUDA device / wrong architecture */
	TSDRGPU_ECUDA     = -2,   /* a CUDA runtime call failed (text in tsdrgpu_last_error) */
	TSDRGPU_EINVAL    = -3,   /* bad argument */
	TSDRGPU_ENOMEM    = -4,
	TSDRGPU_ECAPACITY = -5    /* caller's output buffer too small */
};

typedef struct tsdrgpu_ctx tsdrgpu_ctx_t;

/* ------------------------------------------------------------------------------------------------ context */
TSDRGPU_API int         tsdrgpu_device_count(void);
TSDRGPU_API int         tsdrgpu_create(tsdrgpu_ctx_t **ctx, int device);
TSDRGPU_API void        tsdrgpu_destroy(tsdrgpu_ctx_t *ctx);
TSDRGPU_API const char *tsdrgpu_last_error(tsdrgpu_ctx_t *ctx);      /* ctx may be NULL (creation errors) */
TSDRGPU_API int         tsdrgpu_sm_count(tsdrgpu_ctx_t *ctx);
/* number of kernels this library has launched through ctx since creation (bench.py's gpu_launches) */
TSDRGPU_API uint64_t    tsdrgpu_launch_count(tsdrgpu_ctx_t *ctx);

/* per-kernel timing for roofline reporting: when enabled, the library brackets its main kernel launches with CUDA
 * events on the launching stream.  collect() synchronises the device, returns per-name totals (names: cap x 48
 * chars) and resets.  Not for production paths (adds two event records per launch). */
TSDRGPU_API int tsdrgpu_profile_enable(tsdrgpu_ctx_t *ctx, int on);
TSDRGPU_API int tsdrgpu_profile_collect(tsdrgpu_ctx_t *ctx, char *names, double *total_ms, uint64_t *counts, int cap, int *n);

/* plumbing for C hosts that do not bring their own allocator (Python callers use torch tensors instead) */
TSDRGPU_API int tsdrgpu_malloc(tsdrgpu_ctx_t *ctx, size_t bytes, void **d_ptr);
TSDRGPU_API int tsdrgpu_free(tsdrgpu_ctx_t *ctx, void *d_ptr);
/* one process per GPU on one node: map another rank's tsdrgpu_malloc'd buffer into this process (CUDA IPC, NVLink peer
 * access); the 64-byte handle travels by whatever means the ranks already have (torch.distributed all_gather_object) */
TSDRGPU_API int tsdrgpu_ipc_export(tsdrgpu_ctx_t *ctx, void *d_ptr, uint8_t handle[64]);
TSDRGPU_API int tsdrgpu_ipc_import(tsdrgpu_ctx_t *ctx, const uint8_t handle[64], void **d_ptr);
TSDRGPU_API int tsdrgpu_ipc_release(tsdrgpu_ctx_t *ctx, void *d_ptr);
TSDRGPU_API int tsdrgpu_malloc_host(tsdrgpu_ctx_t *ctx, size_t bytes, void **h_ptr);   /* pinned, on the device's NUMA node when known */
/* NUMA node the device hangs off (sysfs), -1 when unknown; pin the calling thread to that node's cores (0 = done).
 * TSDRGPU_NO_NUMA=1 switches both off. */
TSDRGPU_API int tsdrgpu_device_numa_node(tsdrgpu_ctx_t *ctx);
TSDRGPU_API int tsdrgpu_bind_thread_near_device(tsdrgpu_ctx_t *ctx);
TSDRGPU_API int tsdrgpu_free_host(tsdrgpu_ctx_t *ctx, void *h_ptr);
TSDRGPU_API int tsdrgpu_memcpy_h2d(tsdrgpu_ctx_t *ctx, void *stream, void *d_dst, const void *h_src, size_t bytes);
TSDRGPU_API int tsdrgpu_memcpy_d2h(tsdrgpu_ctx_t *ctx, void *stream, void *h_dst, const void *d_src, size_t bytes);
TSDRGPU_API int tsdrgpu_memcpy_d2d(tsdrgpu_ctx_t *ctx, void *stream, void *d_dst, const void *d_src, size_t bytes);
TSDRGPU_API int tsdrgpu_memset(tsdrgpu_ctx_t *ctx, void *stream, void *d_dst, int value, size_t bytes);
TSDRGPU_API int tsdrgpu_stream_create(tsdrgpu_ctx_t *ctx, void **stream);
TSDRGPU_API int tsdrgpu_stream_destroy(tsdrgpu_ctx_t *ctx, void *stream);
TSDRGPU_API int tsdrgpu_stream_sync(tsdrgpu_ctx_t *ctx, void *stream);                 /* synchronises */

/* ---------------------------------------------------------------------------- host-only scalar helpers (no GPU needed)
 * a4: set_internal_samplerate's geometry (TSDRLibrary.c:540-550). */
TSDRGPU_API void tsdrgpu_geometry(uint32_t samplerate, int height, double refreshrate, int *width, double *pixelrate,
                                  double *pixeltimeoversampletime);
/* one decimator block as the device sees it (40 bytes, no padding) */
typedef struct {
	uint64_t in_start;    /* first sample of the block in the input stream (sample index, not float index) */
	uint64_t out_start;   /* first pixel of the block in the output stream */
	uint32_t size;        /* samples in the block                            (dsp.c:261) */
	uint32_t n_out;       /* output_samples                                  (dsp.c:262) */
	double   r;           /* sampletimeoverpixel = upsample_by/downsample_by (dsp.c:258) */
	double   phase;       /* offset_sample = -offset * r                     (dsp.c:272) */
} tsdrgpu_rs_block_t;
/* the per-call phase recurrence of dsp_resample_process (dsp.c:258-262,272,306) for nblocks consecutive calls:
 * advances *offset, returns the total of the reference's output_samples (UINT64_MAX if a block yields none:
 * the reference asserts there, extbuffer.c:48).  `blocks` may be NULL (count only). */
TSDRGPU_API uint64_t tsdrgpu_plan_resample(double *offset, const uint32_t *sizes, uint32_t uniform, uint32_t nblocks,
                                           double upsample_by, double downsample_by, tsdrgpu_rs_block_t *blocks);
/* relative angle errors eps[l] of the reference FFT's stage twiddles (half-angle recurrence, fft.c:132-165): stage l
 * rotates by (pi/2^l)(1+eps[l]) instead of pi/2^l.  Used by tsdrgpu_fft to track the reference at large N. */
TSDRGPU_API void tsdrgpu_fft_reference_eps(int stages, int inverse, double *eps);
/* host-only: the GUI's auto-resolution arithmetic on the two autocorrelation plots (JavaGUI .../PlotVisualizer.java:203-236,
 * Main.java:1233-1253,1301-1303,1346-1350): first strict maximum of each plot -> fps, height.  Optional outputs may be NULL. */
TSDRGPU_API int tsdrgpu_detect_videomode(const double *frame_plot, int frame_offset, int frame_len, const double *line_plot, int line_offset,
                                         int line_len, uint32_t samplerate, double *fps, int *height, int *frame_index, int *line_index);
/* frameratepll's write-back (syncdetector.c:141-152) for one frame, from the frame stage's per-frame result: returns 1 and
 * moves *refreshrate when the reference would (PLL on is the caller's condition; x_vx != 0 is checked here), else 0. */
TSDRGPU_API int tsdrgpu_pll_step(double *refreshrate, int32_t x_vx, int32_t pll_state, double avg_speed);
/* the same arithmetic from peak indices picked elsewhere (tsdrgpu_frd_peaks: on the device) */
TSDRGPU_API int tsdrgpu_videomode_from_peaks(int frame_offset, int frame_index, int line_offset, int line_index, uint32_t samplerate, double *fps, int *height);
/* the normalised 5-tap Gaussian of gaussian.c:16-30 */
TSDRGPU_API void tsdrgpu_gauss_taps(float taps[5]);

/* ---------------------------------------------------------------------------- a2  AM demodulation
 * replaces am_demod (TSDRLibrary.c:244-262): out[k] = sqrtf(I*I + Q*Q), bit-exact (no FMA, IEEE sqrt). */
TSDRGPU_API int tsdrgpu_am_demod(tsdrgpu_ctx_t *ctx, void *stream, const float *d_iq, uint64_t pairs, float *d_out);

/* ---------------------------------------------------------------------------- a6  resampler (+ fused a2)
 * replaces dsp_resample_init / dsp_resample_process / dsp_resample_t (dsp.c:250-307, dsp.h:79-82), optionally
 * fused with am_demod.  The object carries the reference's {contrib, offset} across calls; `offset` lives on
 * the host (it depends only on sizes and rates), `contrib` on the device (it depends on the data).
 *
 * One run processes `nblocks` CONSECUTIVE decimator blocks (the reference's decimatingthread calls
 * dsp_resample_process once per 0.1 frame, TSDRLibrary.c:335-340); the per-block phase recurrence
 * (dsp.c:262,272,306) is replayed on the host in C, the pixels are computed on the GPU, bit-exact.
 * Deviation: a slot the reference leaves stale because its loop writes one pixel fewer than output_samples
 * (exact-integer landings, e.g. r == 2.0) is written as 0.0f.
 */
typedef struct tsdrgpu_resampler tsdrgpu_resampler_t;
TSDRGPU_API int  tsdrgpu_resampler_create(tsdrgpu_ctx_t *ctx, tsdrgpu_resampler_t **r);
TSDRGPU_API void tsdrgpu_resampler_destroy(tsdrgpu_resampler_t *r);
TSDRGPU_API int  tsdrgpu_resampler_reset(tsdrgpu_resampler_t *r, void *stream);                 /* dsp_resample_init */
TSDRGPU_API int  tsdrgpu_resampler_get_state(tsdrgpu_resampler_t *r, void *stream, double *contrib, double *offset); /* synchronises */
TSDRGPU_API int  tsdrgpu_resampler_set_state(tsdrgpu_resampler_t *r, void *stream, double contrib, double offset);
/* host-only: pixels the next run would produce (sum of the reference's output_samples), state untouched.
 * block_sizes may be NULL: then every block has `uniform_block` samples. */
TSDRGPU_API uint64_t tsdrgpu_resampler_plan(tsdrgpu_resampler_t *r, const uint32_t *block_sizes, uint32_t uniform_block,
                                            uint32_t nblocks, double upsample_by, double downsample_by);
/* d_in: IQ pairs (in_is_iq != 0, 2 floats per sample) or magnitudes (1 float per sample), blocks back to back.
 * Writes *h_n_out pixels to d_out (blocks back to back) and advances the state. */
TSDRGPU_API int  tsdrgpu_resampler_run(tsdrgpu_resampler_t *r, void *stream, const float *d_in, int in_is_iq,
                                       const uint32_t *block_sizes, uint32_t uniform_block, uint32_t nblocks,
                                       double upsample_by, double downsample_by, int nearest_neighbour,
                                       float *d_out, uint64_t out_capacity, uint64_t *h_n_out);

/* One-shot: the NEXT tsdrgpu_resampler_run with IQ input also writes |x| of every input sample to d_mag (one float per
 * sample, blocks back to back like d_in) -- am_demod's output for the frame-rate detector (TSDRLibrary.c:286-292 feeds both
 * consumers from one demodulated buffer) without a second pass over the IQ. */
TSDRGPU_API int  tsdrgpu_resampler_set_mag_out(tsdrgpu_resampler_t *r, float *d_mag);

/* ---------------------------------------------------------------------------- a7-a15  frame stage
 * replaces dsp_post_process + dsp_postprocess_t (dsp.c:112-239), dsp_autogain_run (:41-94),
 * dsp_timelowpass_run (:22-33), dsp_average_v_h (:96-110), syncdetector_run / findthesweetspot / findbestfit /
 * frameratepll state (syncdetector.c:26-226) and gaussianblur (gaussian.c:18-79), for a BATCH of consecutive
 * frames.  Pixel outputs and all integer sync results are bit-exact; `snr` (never announced by the reference,
 * dsp.c:234) is computed with parallel double sums, ~1e-12 relative.
 * The PLL's write-back to refreshrate (syncdetector.c:141-152) is the HOST's job: the per-frame results carry
 * vx / avg_speed / state so the caller applies it between batches (geometry is constant inside one batch).
 */
typedef struct tsdrgpu_framestage tsdrgpu_framestage_t;

typedef struct {
	int32_t x_dx, x_vx, x_absvx, x_stripsize;     /* sweetspot_data_t db_x (syncdetector.h:16-22) */
	int32_t y_dx, y_vx, y_absvx, y_stripsize;     /* db_y */
	double  avg_speed;                            /* syncdetector_t.avg_speed after this frame */
	int32_t pll_state;                            /* 1 = locked */
	float   lastmax, lastmin, snr;                /* dsp_autogain_t after this frame */
	int32_t autogain_report;                      /* 1 when dsp.c:231-235 would announce min/max */
	int32_t reserved;
} tsdrgpu_frame_result_t;

enum {                                            /* flags for tsdrgpu_framestage_run */
	TSDRGPU_FS_AUTOSHIFT            = 1,          /* PARAM_INT_AUTOSHIFT */
	TSDRGPU_FS_LOWPASS_BEFORE_SYNC  = 2,          /* PARAM_LOW_PASS_BEFORE_SYNC */
	TSDRGPU_FS_AUTOGAIN_AFTER_PROC  = 4,          /* PARAM_AUTOGAIN_AFTER_PROCESSING */
	TSDRGPU_FS_SUPERRESOLUTION      = 8,          /* PARAM_AUTOCORR_SUPERRESOLUTION (suppresses the green lines) */
	TSDRGPU_FS_COMPUTE_SNR          = 16          /* also fill .snr (costs one more reduction) */
};

TSDRGPU_API int  tsdrgpu_framestage_create(tsdrgpu_ctx_t *ctx, tsdrgpu_framestage_t **fs);
TSDRGPU_API void tsdrgpu_framestage_destroy(tsdrgpu_framestage_t *fs);
TSDRGPU_API int  tsdrgpu_framestage_reset(tsdrgpu_framestage_t *fs, void *stream);          /* dsp_post_process_init */
/* d_frames_in / d_frames_out: nframes * width * height floats, frames back to back (in != out).
 * h_results (nframes entries, may be NULL) is filled when the call returns: this call synchronises `stream`
 * only if h_results != NULL. */
TSDRGPU_API int  tsdrgpu_framestage_run(tsdrgpu_framestage_t *fs, void *stream, const float *d_frames_in, int nframes,
                                        int width, int height, float motionblur, float lowpasscoeff, unsigned flags,
                                        float *d_frames_out, tsdrgpu_frame_result_t *h_results);

/* same, but never synchronises: h_results_pinned (page-locked, nframes entries, may be NULL) is valid once the
 * stream has passed this call; h_autogain_report (nframes ints, may be NULL) is filled on return. */
TSDRGPU_API int  tsdrgpu_framestage_run_async(tsdrgpu_framestage_t *fs, void *stream, const float *d_frames_in, int nframes,
                                              int width, int height, float motionblur, float lowpasscoeff, unsigned flags,
                                              float *d_frames_out, tsdrgpu_frame_result_t *h_results_pinned,
                                              int32_t *h_autogain_report);

/* Overlap mode (off by default).  When on, and for the default stage order (LOWPASS_BEFORE_SYNC set,
 * AUTOGAIN_AFTER_PROC clear), the latency-bound sync search and the re-centring of batch k run on an internal side
 * stream while `stream` already works on batch k+1.  d_frames_out / h_results_pinned of a run are then valid only
 * after tsdrgpu_framestage_join(fs, s) has made stream `s` wait for the side stream (or after a device sync). */
TSDRGPU_API int  tsdrgpu_framestage_set_overlap(tsdrgpu_framestage_t *fs, int on);
TSDRGPU_API int  tsdrgpu_framestage_join(tsdrgpu_framestage_t *fs, void *stream);

/* stage-level entry points (same arithmetic as the kernels inside tsdrgpu_framestage_run) */
TSDRGPU_API int tsdrgpu_autogain(tsdrgpu_ctx_t *ctx, void *stream, float *h_lastmax, float *h_lastmin, float *h_snr,
                                 int n, const float *d_in, float *d_out, float norm);        /* synchronises */
TSDRGPU_API int tsdrgpu_timelowpass(tsdrgpu_ctx_t *ctx, void *stream, float coeff, int n, const float *d_in, float *d_screen);
TSDRGPU_API int tsdrgpu_average_v_h(tsdrgpu_ctx_t *ctx, void *stream, int width, int height, const float *d_in,
                                    float *d_wbuf, float *d_hbuf);
TSDRGPU_API int tsdrgpu_gaussianblur(tsdrgpu_ctx_t *ctx, void *stream, float *d_data, int n);

/* ---------------------------------------------------------------------------- a16 host pixel rule (next-row item)
 * the JNI glue's float->ARGB mapping (JavaGUI/jni/TSDRLibraryNDK.c:222-283), bit-exact; transparent (2048.0f)
 * pixels keep the previous content of d_argb. */
TSDRGPU_API int tsdrgpu_pixels_argb(tsdrgpu_ctx_t *ctx, void *stream, const float *d_frame, int n, int inverted, int32_t *d_argb);
/* a batch of frames converted IN PLACE (float frame f becomes its n int32 pixels); d_last (n int32, caller-zeroed at start)
 * is the host's persistent pixel buffer carried across frames and calls, so transparent samples behave as in the GUI */
TSDRGPU_API int tsdrgpu_pixels_argb_batch(tsdrgpu_ctx_t *ctx, void *stream, float *d_frames_inout, uint64_t n, int nframes, int inverted, int32_t *d_last);

/* ---------------------------------------------------------------------------- a19/a20  FFT and correlations
 * replace fft_perform, fft_autocorrelation, fft_crosscorrelation (fft.c:49-176).  Same definitions as the
 * reference (forward divides by N, inverse does not; N = largest power of two <= size; "autocorrelation" is
 * IFFT(|FFT(x)|/N)), computed by a float32 Stockham FFT with double-derived twiddles: results agree with the
 * reference's float-storage/double-arithmetic radix-2 code to ~1e-6 of the spectrum's peak (tolerance-based).
 */
TSDRGPU_API uint32_t tsdrgpu_fft_getrealsize(uint32_t size);                                   /* fft.c:5-11 */
TSDRGPU_API int tsdrgpu_fft(tsdrgpu_ctx_t *ctx, void *stream, float *d_iq, uint32_t size, int inverse);   /* in place */
TSDRGPU_API int tsdrgpu_autocorrelation(tsdrgpu_ctx_t *ctx, void *stream, float *d_answer, const float *d_real, uint32_t size);
/* `batch` independent autocorrelations in one set of launches: input b at d_reals + b*real_stride (floats), output b at
 * d_answers + b*2*size (floats).  size must be even. */
TSDRGPU_API int tsdrgpu_autocorrelation_batch(tsdrgpu_ctx_t *ctx, void *stream, float *d_answers, const float *d_reals, uint32_t size,
                                              uint32_t batch, uint64_t real_stride);
TSDRGPU_API int tsdrgpu_crosscorrelation(tsdrgpu_ctx_t *ctx, void *stream, float *d_a_out, float *d_b_tmp, uint32_t samples);

/* ---------------------------------------------------------------------------- a17/a18  frame-rate detector
 * replaces frameratedetector_runontodata / accummulate (frameratedetector.c:34-126) and the two extbuffer
 * running means: one capture in, the two lag-window plots out. */
typedef struct tsdrgpu_frd tsdrgpu_frd_t;
TSDRGPU_API int  tsdrgpu_frd_create(tsdrgpu_ctx_t *ctx, tsdrgpu_frd_t **frd);
TSDRGPU_API void tsdrgpu_frd_destroy(tsdrgpu_frd_t *frd);
/* Overlapped mode: a run's kernels go to an internal stream (behind what `stream` held at the call) with work buffers of the
 * detector's own, so the transforms share the chip with what the caller enqueues next; the capture must stay untouched until
 * tsdrgpu_frd_join(frd, s) has put stream s behind the run (plots / peaks readers join by themselves). */
TSDRGPU_API int  tsdrgpu_frd_set_overlap(tsdrgpu_frd_t *frd, int on);
TSDRGPU_API int  tsdrgpu_frd_join(tsdrgpu_frd_t *frd, void *stream);
TSDRGPU_API int  tsdrgpu_frd_reset(tsdrgpu_frd_t *frd);                      /* extbuffer_cleartozero on all three */
TSDRGPU_API uint32_t tsdrgpu_frd_capture_size(uint32_t samplerate);          /* frameratedetector.c:160 */
TSDRGPU_API void tsdrgpu_frd_windows(uint32_t samplerate, int *frame_min, int *frame_max, int *line_min, int *line_max);
/* d_capture: `size` demodulated samples.  The running means stay on the device; pass h_* (may be NULL) to copy
 * them out (then the call synchronises).  *calls = captures accumulated so far. */
TSDRGPU_API int  tsdrgpu_frd_run(tsdrgpu_frd_t *frd, void *stream, uint32_t samplerate, const float *d_capture, uint32_t size,
                                 double *h_frame_plot, int frame_cap, double *h_line_plot, int line_cap, uint64_t *calls);
/* same without the final synchronisation; the h_* buffers must be page-locked */
TSDRGPU_API int  tsdrgpu_frd_run_async(tsdrgpu_frd_t *frd, void *stream, uint32_t samplerate, const float *d_capture, uint32_t size,
                                       double *h_frame_plot_pinned, int frame_cap, double *h_line_plot_pinned, int line_cap, uint64_t *calls);
/* `batch` consecutive captures (capture b at d_captures + b*capture_stride floats) accumulated in order, as if
 * tsdrgpu_frd_run had been called batch times; asynchronous, plots stay on the device. */
TSDRGPU_API int  tsdrgpu_frd_run_batch(tsdrgpu_frd_t *frd, void *stream, uint32_t samplerate, const float *d_captures, uint32_t size,
                                       uint32_t batch, uint64_t capture_stride, uint64_t *calls);
/* copies the current running means (device-resident) to host buffers; synchronises */
/* dump_autocorrect (frameratedetector.c:64-85): CSV of (lag in ms, 10 log10 |r|) of one capture's autocorrelation; synchronises */
TSDRGPU_API int  tsdrgpu_frd_dump_csv(tsdrgpu_frd_t *frd, void *stream, uint32_t samplerate, const float *d_capture, uint32_t size, const char *path);
TSDRGPU_API int  tsdrgpu_frd_get_plots(tsdrgpu_frd_t *frd, void *stream, uint32_t samplerate, double *h_frame_plot, int frame_cap,
                                       double *h_line_plot, int line_cap);
/* SURVEY 8f-3 on the device: index of the first strict maximum of each plot (PlotVisualizer.java:203-236), reduced on the GPU
 * right behind the running means of every run.  h_peaks[0] = frame plot, [1] = line plot.  _async: page-locked destination. */
TSDRGPU_API int  tsdrgpu_frd_peaks(tsdrgpu_frd_t *frd, void *stream, int32_t *h_peaks);                  /* synchronises */
TSDRGPU_API int  tsdrgpu_plot_peaks(tsdrgpu_ctx_t *ctx, void *stream, const double *d_frame_plot, int frame_len, const double *d_line_plot, int line_len,
                                    int32_t *h_peaks);                                                     /* synchronises */
TSDRGPU_API int  tsdrgpu_frd_peaks_async(tsdrgpu_frd_t *frd, void *stream, int32_t *h_peaks_pinned);
TSDRGPU_API int  tsdrgpu_accumulate(tsdrgpu_ctx_t *ctx, void *stream, double *d_out, uint64_t calls,
                                    const float *d_in_complex, int startid, int length);

/* ---------------------------------------------------------------------------- a22  superbandwidth
 * replace complex_to_abs_diff, superb_bestfit, superb_ondataready (superbandwidth.c:67-152). */
TSDRGPU_API int tsdrgpu_complex_to_abs_diff(tsdrgpu_ctx_t *ctx, void *stream, float *d_data, int size_floats);
/* alignment lag in floats (2 * argmax over the first half of |xcorr|), exact integer.  synchronises */
TSDRGPU_API int tsdrgpu_superb_bestfit(tsdrgpu_ctx_t *ctx, void *stream, const float *d_hop0, const float *d_hopi,
                                       int size_floats, int samples_in_frame, int *h_best_offset);
/* single-GPU stitch of nhops hops (each count_pairs IQ pairs, d_hops[i] device pointers in a HOST array);
 * d_out holds nhops * N * 2 floats, N = fft_getrealsize(count_pairs).  synchronises (lags are read back). */
TSDRGPU_API int tsdrgpu_superb_stitch(tsdrgpu_ctx_t *ctx, void *stream, float *const *d_hops, int nhops, int count_pairs,
                                      int samples_in_frame, float *d_out, int *h_best_offsets, int *h_total_samples);
/* multi-GPU building blocks (one hop per rank; the all-gather between them is the caller's NCCL call):
 *   rotate hop by best_offset floats and forward-FFT it into d_spectrum (N complex);
 *   then, given the gathered [X0..X_{H-1}] (H*N complex), produce this rank's share of the H*N-point inverse:
 *   the strided residue s of the output (y[H*p + s], p < N) -- see DESIGN.md "superbandwidth decomposition". */
TSDRGPU_API int tsdrgpu_superb_hop_spectrum(tsdrgpu_ctx_t *ctx, void *stream, const float *d_hop, int count_pairs,
                                            int best_offset_floats, float *d_spectrum);
/* tsdrgpu_superb_local_spectra with the all-gather fused into the transforms: the last pass of each FFT stores its result
 * into the gather buffer of every rank (d_peer_bufs[p], host array of nhops device pointers; the peers' buffers mapped with
 * tsdrgpu_ipc_import) at slot `rank` ([X | D] at complex offset rank*block_stride_complex).  The caller then only needs a
 * barrier across the ranks before reading its own buffer. */
TSDRGPU_API int tsdrgpu_superb_local_spectra_scatter(tsdrgpu_ctx_t *ctx, void *stream, const float *d_hop, int count_pairs, int samples_in_frame,
                                                     float *const *d_peer_bufs, int nhops, int rank, uint64_t block_stride_complex,
                                                     uint32_t *h_n, uint32_t *h_nd);
/* the same with ONE exchange in total (DESIGN.md section 6): every rank sends [FFT_N(raw hop) | FFT_nd(first
 * difference of |hop|)] (n + nd complex, returned in *h_n / *h_nd), one all-gather, then every rank derives the
 * integer alignment lags itself (tsdrgpu_superb_lags, exact) and applies them as spectral phase ramps while mixing. */
TSDRGPU_API int tsdrgpu_superb_local_spectra(tsdrgpu_ctx_t *ctx, void *stream, const float *d_hop, int count_pairs, int samples_in_frame,
                                             float *d_block, uint32_t *h_n, uint32_t *h_nd);
TSDRGPU_API int tsdrgpu_superb_lags(tsdrgpu_ctx_t *ctx, void *stream, const float *d_gathered, int nhops, uint64_t block_stride_complex,
                                    uint32_t n, uint32_t nd, int *h_lags);
TSDRGPU_API int tsdrgpu_superb_residue_ifft_lag(tsdrgpu_ctx_t *ctx, void *stream, const float *d_gathered, int nhops,
                                                uint64_t block_stride_complex, uint32_t n, int residue, const int *h_lags, float *d_out_residue);
TSDRGPU_API int tsdrgpu_superb_residue_ifft(tsdrgpu_ctx_t *ctx, void *stream, const float *d_gathered, int nhops, uint32_t n,
                                            int residue, float *d_out_residue);

/* ---- one hop per GPU, behind the C-ABI (SURVEY section 8e, DESIGN.md section 6; csrc/superb_mgpu.cu) ----------------------
 * superb_ondataready sharded over the GPUs of one node: rank q owns hop q.  Local spectra -> this rank's alignment lag (hop 0's
 * difference spectrum read from rank 0 over NVLink) -> an all-to-all mix (bins pulled from the peers, residues pushed to
 * them) -> one N-point inverse per rank -> |.| pushed into the root's window -> the root interleaves the time-contiguous
 * MAGNITUDE stream (what am_demod makes of superb_run's output, TSDRLibrary.c:271-274).  No host synchronisation, no
 * collective library: flags in peer memory order the phases.  A group object exists once per rank; the windows are tied
 * together either through CUDA IPC handles (one process per GPU: export -> exchange by any means -> connect_ipc) or directly
 * (all ranks in one process: connect_local).  nranks in {2, 4, 8, 16}. */
typedef struct tsdrgpu_superb_mgpu tsdrgpu_superb_mgpu_t;
TSDRGPU_API int  tsdrgpu_superb_mgpu_create(tsdrgpu_ctx_t *ctx, int nranks, int rank, int root, uint32_t max_pairs_per_hop, tsdrgpu_superb_mgpu_t **g);
TSDRGPU_API void tsdrgpu_superb_mgpu_destroy(tsdrgpu_superb_mgpu_t *g);
TSDRGPU_API int  tsdrgpu_superb_mgpu_export(tsdrgpu_superb_mgpu_t *g, uint8_t handle[64]);
TSDRGPU_API int  tsdrgpu_superb_mgpu_connect_ipc(tsdrgpu_superb_mgpu_t *g, const uint8_t *handles /* nranks x 64 bytes, rank-major */);
TSDRGPU_API int  tsdrgpu_superb_mgpu_connect_local(tsdrgpu_superb_mgpu_t *const *all_ranks, int nranks);
/* unmap the peers' windows; with one process per GPU: all ranks disconnect, synchronise among themselves, then destroy */
TSDRGPU_API int  tsdrgpu_superb_mgpu_disconnect(tsdrgpu_superb_mgpu_t *g);
/* every rank calls this once per stitch (same count_pairs / samples_in_frame), each on a stream of its own device; asynchronous.
 * d_hop: this rank's hop.  d_hop0: a copy of hop 0 (the alignment reference, superbandwidth.c:133) on THIS device, or NULL --
 * then its difference spectrum is read from rank 0 over NVLink after one more barrier; either all ranks pass it or none.
 * The root's d_stream_out receives nranks * N magnitudes, N = fft_getrealsize(count_pairs) returned in *h_n. */
TSDRGPU_API int  tsdrgpu_superb_mgpu_stitch(tsdrgpu_superb_mgpu_t *g, void *stream, const float *d_hop, const float *d_hop0, int count_pairs,
                                            int samples_in_frame, float *d_stream_out, uint32_t *h_n);
/* lags (complex samples) of the last stitch as every rank published them, and the status word (0 = fine); synchronises `stream` */
/* the root's stream inside its window: valid after a stitch called with d_stream_out = NULL, until the root's next stitch */
TSDRGPU_API int  tsdrgpu_superb_mgpu_stream_window(tsdrgpu_superb_mgpu_t *g, float **d_stream);
TSDRGPU_API int  tsdrgpu_superb_mgpu_lags(tsdrgpu_superb_mgpu_t *g, void *stream, int *h_lags, uint32_t *h_status);

/* ---------------------------------------------------------------------------- tuner (digital down-converter)
 * Not in the reference: picks one sub-band out of a wideband capture ahead of the pixel path (DESIGN.md section 5.6).  Input
 * pair n (absolute index since the last reset, dropped pairs counted) is mixed by e^{-2 pi i offset n / fs} with the integer
 * phase n * phase_inc mod 2^64, low-passed by a real linear-phase FIR and decimated by D: output m is
 * z[m] = sum_k h[k] x~[mD - k], x~ = the mixed input with zeros before the first sample and over every drop, produced for every
 * m with mD inside a block (outputs whose mD falls into a drop are withheld and counted as the output drop count).
 * Configuration rules: decimation in 1..64, ntaps odd in 3..1023 (0 = 16 * ceil(fs / bandwidth) + 1, at most 1023),
 * fs % decimation == 0, 0 < bandwidth_hz <= fs / decimation, |offset_hz| + bandwidth_hz / 2 <= fs / 2; anything else is
 * TSDRGPU_EINVAL with a text naming the rule.  Filter: scipy.signal.firwin(ntaps, bandwidth_hz / 2, window=('kaiser', 7.857),
 * fs=fs) designed in double, stored as float32. */
typedef struct tsdrgpu_tuner tsdrgpu_tuner_t;
/* host-only: validates and returns the float32 taps (cap entries at least) and the phase increment round(offset / fs * 2^64)
 * (two's complement).  taps / ntaps_out / phase_inc may be NULL (validation only). */
TSDRGPU_API int tsdrgpu_tuner_design(uint32_t fs, double offset_hz, double bandwidth_hz, int decimation, int ntaps, float *taps, int cap,
                                     int *ntaps_out, uint64_t *phase_inc);
/* host-only: outputs of a block of `pairs` input pairs preceded by `dropped` lost pairs, the stream being at absolute index
 * `position` before the loss: *out_dropped = ceil((position + dropped) / D) - ceil(position / D),
 * *out_pairs = ceil((position + dropped + pairs) / D) - ceil((position + dropped) / D). */
TSDRGPU_API int tsdrgpu_tuner_out_pairs(uint64_t position, uint64_t pairs, uint64_t dropped, int decimation, uint64_t *out_pairs,
                                        uint64_t *out_dropped);
TSDRGPU_API int  tsdrgpu_tuner_create(tsdrgpu_ctx_t *ctx, tsdrgpu_tuner_t **t);
TSDRGPU_API void tsdrgpu_tuner_destroy(tsdrgpu_tuner_t *t);
/* (re)design the filter and reset; synchronises the device */
TSDRGPU_API int  tsdrgpu_tuner_configure(tsdrgpu_tuner_t *t, uint32_t fs, double offset_hz, double bandwidth_hz, int decimation, int ntaps);
TSDRGPU_API int  tsdrgpu_tuner_reset(tsdrgpu_tuner_t *t, void *stream);      /* position 0, history zero */
/* d_iq: `pairs` interleaved I,Q pairs; d_out receives *out_pairs pairs (at most ceil(pairs / D) + 1).  Asynchronous: the counts
 * come from host state (tsdrgpu_tuner_out_pairs), the device history of the last ntaps - 1 mixed samples is updated in stream order. */
TSDRGPU_API int  tsdrgpu_tuner_run(tsdrgpu_tuner_t *t, void *stream, const float *d_iq, uint64_t pairs, uint64_t dropped_before, float *d_out,
                                   uint64_t *out_pairs, uint64_t *out_dropped);

/* ---------------------------------------------------------------------------- channelizer (polyphase filter bank)
 * Not in the reference: splits a capture into K sub-bands at once (DESIGN.md section 5.7).  K is a power of two in 2..256, the
 * decimation is D = K/2 (oversampled by 2), Q taps per channel in 4..32 (0 = 16).  The prototype h is the tuner's design
 * tsdrgpu_tuner_design(fs, 0, fs / K, K / 2, Q * K - 1).  Channel c has offset c * fs / K for c < K/2 and (c - K) * fs / K otherwise
 * (channel K/2 reads -fs/2) and output
 *   y_c[m] = sum_k h[k] x[mD - k] e^{-2 pi i off_c (mD - k) / fs},
 * x with zeros before the stream and over every drop, n counted since the last reset: the tuner at off_c with the same taps and
 * decimation.  Output m exists for every mD inside a block, so the counts are tsdrgpu_channelizer_out_pairs's.
 * Configuration rules: K a power of two in 2..256, Q in 4..32 (0 = default), fs % (K/2) == 0, 2 fs / K >= 130500 (the channel
 * rate keeps the frame-rate detector's line window off lag 0), Q*K - 1 taps fit the shared-memory tile; anything else is
 * TSDRGPU_EINVAL with a text naming the rule. */
typedef struct tsdrgpu_channelizer tsdrgpu_channelizer_t;
enum { TSDRGPU_CHANNELIZER_COMPLEX = 0, TSDRGPU_CHANNELIZER_MAGNITUDE = 1 };
/* host-only: validates and returns the Q*K - 1 float32 prototype taps (taps may be NULL: validation only) */
TSDRGPU_API int tsdrgpu_channelizer_design(uint32_t fs, int channels, int taps_per_channel, float *taps, int cap, int *ntaps_out);
/* host-only: the tuner's count arithmetic (tsdrgpu_tuner_out_pairs) at D = channels / 2, outputs per channel */
TSDRGPU_API int tsdrgpu_channelizer_out_pairs(uint64_t position, uint64_t pairs, uint64_t dropped, int channels, uint64_t *out_pairs,
                                              uint64_t *out_dropped);
TSDRGPU_API int  tsdrgpu_channelizer_create(tsdrgpu_ctx_t *ctx, tsdrgpu_channelizer_t **c);
TSDRGPU_API void tsdrgpu_channelizer_destroy(tsdrgpu_channelizer_t *c);
TSDRGPU_API int  tsdrgpu_channelizer_configure(tsdrgpu_channelizer_t *c, uint32_t fs, int channels, int taps_per_channel);   /* synchronises */
TSDRGPU_API int  tsdrgpu_channelizer_reset(tsdrgpu_channelizer_t *c, void *stream);       /* position 0, history zero */
/* mode TSDRGPU_CHANNELIZER_COMPLEX: channel c's *out_pairs I,Q pairs at d_out + 2 * c * channel_stride floats;
 * TSDRGPU_CHANNELIZER_MAGNITUDE: sqrtf(I*I + Q*Q) (tsdrgpu_am_demod's arithmetic) at d_out + c * channel_stride floats.
 * channel_stride (in outputs) >= *out_pairs.  Asynchronous; the history of the last Q*K - 2 input pairs is carried on the device. */
TSDRGPU_API int  tsdrgpu_channelizer_run(tsdrgpu_channelizer_t *c, void *stream, const float *d_iq, uint64_t pairs, uint64_t dropped_before,
                                         int mode, float *d_out, uint64_t channel_stride, uint64_t *out_pairs, uint64_t *out_dropped);

/* ---------------------------------------------------------------------------- scan (a frame-rate detector per channel)
 * A channelizer in magnitude mode; each channel's stream is cut into consecutive captures of tsdrgpu_frd_capture_size(rate)
 * samples, rate = 2 fs / K (a drop discards every channel's partial capture).  Every complete round of K captures goes through the
 * batched autocorrelation and updates K pairs of running means over tsdrgpu_frd_windows(rate), on an internal stream behind the
 * caller's.  Per channel the table reports the first strict maximum of each plot, the video mode they imply
 * (tsdrgpu_videomode_from_peaks) and score = (max - mean) / std of each plot. */
typedef struct {
	double   offset_hz;                  /* the channel's centre, in the frame of tsdrgpu_pipeline_set_tuner's offset_hz */
	uint32_t rate;                       /* 2 fs / K */
	uint64_t captures;                   /* rounds accumulated since the last reset */
	int32_t  frame_index, line_index;    /* first strict maximum of each plot (indices into the windows) */
	double   fps; int32_t height;        /* tsdrgpu_videomode_from_peaks at `rate` (0 before the first round) */
	double   frame_score, line_score;
} tsdrgpu_scan_channel_t;
typedef struct tsdrgpu_scan tsdrgpu_scan_t;
TSDRGPU_API int  tsdrgpu_scan_create(tsdrgpu_ctx_t *ctx, tsdrgpu_scan_t **s);
TSDRGPU_API void tsdrgpu_scan_destroy(tsdrgpu_scan_t *s);
TSDRGPU_API int  tsdrgpu_scan_configure(tsdrgpu_scan_t *s, uint32_t fs, int channels, int taps_per_channel);            /* synchronises */
TSDRGPU_API int  tsdrgpu_scan_reset(tsdrgpu_scan_t *s, void *stream);
TSDRGPU_API int  tsdrgpu_scan_run(tsdrgpu_scan_t *s, void *stream, const float *d_iq, uint64_t pairs, uint64_t dropped_before);
/* min(cap, K) records, channel order; synchronises */
TSDRGPU_API int  tsdrgpu_scan_results(tsdrgpu_scan_t *s, void *stream, tsdrgpu_scan_channel_t *h_out, int cap);
/* the running means, channel-major: channel c's frame plot at h_plots[c * (frame_len + line_len)], its line plot right behind;
 * synchronises */
TSDRGPU_API int  tsdrgpu_scan_plots(tsdrgpu_scan_t *s, void *stream, double *h_plots, uint64_t cap, int *frame_len, int *line_len);

/* ---------------------------------------------------------------------------- notch filter (stopbands ahead of the pixel path)
 * Not in the reference: removes narrowband carriers from every block (DESIGN.md section 5.8).  Stopbands (f_j, w_j), j < n <= 32,
 * in Hz in the capture's frame (that of tsdrgpu_pipeline_set_tuner's offset_hz and of the scan's table); L taps, L odd;
 * delta(L) = (80 - 7.95) / (2.285 * 2 pi * (L - 1)) * fs, the transition width of the 80 dB Kaiser design.  The complex FIR is
 *   h[m] = delta[m - (L-1)/2] - sum_j g_j[m] e^{2 pi i f_j (m - (L-1)/2) / fs},   g_j = the tuner's low-pass design at bandwidth w_j
 * (scipy.signal.firwin(L, w_j / 2, window=('kaiser', 7.857), fs=fs)), designed in double, stored as float32.  Output
 * y[n] = sum_k h[k] x~[n - k], x~ = the input with zeros before the stream and over every drop, n counted since the last reset:
 * one output per input pair, the drop count passes through unchanged, the group delay is (L - 1) / 2 pairs.
 * Configuration rules: 1 <= n <= 32, w_j > 0, |f_j| + w_j / 2 <= fs / 2, w_j >= 2 delta(L), neighbouring bands (sorted by
 * frequency, also across +-fs/2) at least delta(L) apart edge to edge, L odd in 65..8193 (0 = the smallest odd L >= 65 that meets
 * the width rule for the narrowest notch); anything else is TSDRGPU_EINVAL with a text naming the rule.
 * Kernel: overlap-save with an FFT of N = the smallest power of two >= 2 (L - 1) in 1024..16384 points, hop N - (L - 1), segments at
 * every multiple of the hop.  Cutting the stream at multiples of the hop gives bit-identical outputs; other cuts differ by FFT
 * round-off in the segments a block boundary falls into. */
typedef struct tsdrgpu_notch tsdrgpu_notch_t;
/* host-only: validates; taps (NULL: validation only) receives the L complex float32 taps as interleaved re, im (cap >= L complex
 * taps); *ntaps_out = L, *nfft_out = N (either may be NULL) */
TSDRGPU_API int tsdrgpu_notch_design(uint32_t fs, int n, const double *centers, const double *widths, int ntaps, float *taps, int cap,
                                     int *ntaps_out, int *nfft_out);
TSDRGPU_API int  tsdrgpu_notch_create(tsdrgpu_ctx_t *ctx, tsdrgpu_notch_t **t);
TSDRGPU_API void tsdrgpu_notch_destroy(tsdrgpu_notch_t *t);
/* (re)design the filter and reset; synchronises the device */
TSDRGPU_API int  tsdrgpu_notch_configure(tsdrgpu_notch_t *t, uint32_t fs, int n, const double *centers, const double *widths, int ntaps);
TSDRGPU_API int  tsdrgpu_notch_reset(tsdrgpu_notch_t *t, void *stream);      /* position 0, history zero */
/* d_iq: `pairs` interleaved I,Q pairs; d_out (not d_iq) receives *out_pairs = pairs pairs; *out_dropped = dropped_before.
 * Asynchronous; the history of the last (L - 1) + (position mod hop) pairs is carried on the device. */
TSDRGPU_API int  tsdrgpu_notch_run(tsdrgpu_notch_t *t, void *stream, const float *d_iq, uint64_t pairs, uint64_t dropped_before, float *d_out,
                                   uint64_t *out_pairs, uint64_t *out_dropped);

/* ---------------------------------------------------------------------------- power spectrum (Welch) of the capture
 * Periodic Hann window of nfft points (a power of two in 64..16384), hop nfft / 2: segment s covers the absolute positions
 * [s nfft/2, s nfft/2 + nfft) since the reset.  A segment that touches a dropped position is skipped; every complete segment's
 * |X|^2 is added to per-bin double sums in segment order, so the result does not depend on how the stream is cut into blocks.
 * Density = sum / (segments * fs * sum(w^2)), reported fft-shifted from -fs/2 to fs/2 - fs/nfft: with no drops,
 * scipy.signal.welch(x, fs, window='hann', nperseg=nfft, noverlap=nfft/2, detrend=False, return_onesided=False,
 * scaling='density'). */
typedef struct tsdrgpu_spectrum tsdrgpu_spectrum_t;
/* host-only: TSDRGPU_OK, or TSDRGPU_EINVAL with a text naming the rule */
TSDRGPU_API int  tsdrgpu_spectrum_check(uint32_t fs, int nfft);
TSDRGPU_API int  tsdrgpu_spectrum_create(tsdrgpu_ctx_t *ctx, tsdrgpu_spectrum_t **s);
TSDRGPU_API void tsdrgpu_spectrum_destroy(tsdrgpu_spectrum_t *s);
TSDRGPU_API int  tsdrgpu_spectrum_configure(tsdrgpu_spectrum_t *s, uint32_t fs, int nfft);      /* resets; synchronises */
TSDRGPU_API int  tsdrgpu_spectrum_reset(tsdrgpu_spectrum_t *s, void *stream);
TSDRGPU_API int  tsdrgpu_spectrum_run(tsdrgpu_spectrum_t *s, void *stream, const float *d_iq, uint64_t pairs, uint64_t dropped_before);
/* min(cap, nfft) density values (fft-shifted) and the number of segments averaged; synchronises `stream` */
TSDRGPU_API int  tsdrgpu_spectrum_results(tsdrgpu_spectrum_t *s, void *stream, double *h_psd, int cap, uint64_t *segments);

/* ---------------------------------------------------------------------------- a1, a3, a5, a16, a17  streaming pipeline
 * replaces the body of process() (TSDRLibrary.c:264-298), decimatingthread / postprocessingthread /
 * videodecodingthread (TSDRLibrary.c:300-418) with their three rings (circbuff.c), dsp_dropped_compensation_*
 * (dsp.c:313-368) and the frame-rate detector's capture loop (frameratedetector.c:128-187, 215-230).
 * HOST buffers in (the plugin's), HOST frame / plot buffers out (valid during the callback only), callbacks on an
 * internal delivery thread.  The C host library (tempestsdr_b200/host) forwards the reference's process() here.
 */
typedef struct tsdrgpu_pipeline tsdrgpu_pipeline_t;

enum {                                   /* indices of params_int: TSDRLibrary.h:32-41 */
	TSDRGPU_PARAM_INT_AUTOSHIFT = 0, TSDRGPU_PARAM_INT_FRAMERATE_PLL = 1, TSDRGPU_PARAM_AUTOCORR_PLOTS_RESET = 2,
	TSDRGPU_PARAM_AUTOCORR_PLOTS_OFF = 3, TSDRGPU_PARAM_AUTOCORR_SUPERRESOLUTION = 4,
	TSDRGPU_PARAM_NEAREST_NEIGHBOUR_RESAMPLING = 5, TSDRGPU_PARAM_LOW_PASS_BEFORE_SYNC = 6,
	TSDRGPU_PARAM_AUTOGAIN_AFTER_PROCESSING = 7, TSDRGPU_PARAM_AUTOCORR_DUMP = 8
};

typedef struct {
	uint32_t samplerate;                 /* tsdrplugin_getsamplerate() */
	int      height;                     /* tsdr_setresolution */
	double   refreshrate;
	float    motionblur;                 /* tsdr_motionblur */
	uint32_t params_int[9];              /* tsdr_setparameter_int */
	int      batch_frames;               /* frames per frame-stage launch (>= 1; 1 = lowest latency) */
	int      batch_blocks;               /* decimator blocks (0.1 frame each) per resampler launch (>= 1; default 10) */
	int      block_when_busy;            /* 1: wait for the frame callback instead of dropping a batch */
} tsdrgpu_pipeline_config_t;

typedef struct {
	uint64_t samples_in, samples_dropped_upstream, samples_resampled;
	uint64_t frames_processed, frames_delivered, frames_dropped, captures, plots_delivered;
	uint64_t h2d_bytes, d2h_bytes, gpu_launches, stitches;
	uint64_t host_buffers_registered;   /* plugin buffers page-locked in place (cudaHostRegister) after they kept coming back */
} tsdrgpu_pipeline_stats_t;

typedef void (*tsdrgpu_frame_cb)(float *buf, int width, int height, void *user);                  /* tsdr_readasync_function */
typedef void (*tsdrgpu_value_cb)(int value_id, double arg0, double arg1, void *user);             /* tsdr_value_changed_callback */
typedef void (*tsdrgpu_plot_cb)(int plot_id, int offset, double *values, int size, uint32_t samplerate, void *user);
typedef void (*tsdrgpu_retune_cb)(int32_t offset_hz, void *user);        /* shiftfreq (TSDRLibrary.c:208): tune to centre + offset */

TSDRGPU_API int  tsdrgpu_pipeline_create(tsdrgpu_ctx_t *ctx, const tsdrgpu_pipeline_config_t *cfg, tsdrgpu_frame_cb frame_cb,
                                         tsdrgpu_value_cb value_cb, tsdrgpu_plot_cb plot_cb, void *user, tsdrgpu_pipeline_t **p);
TSDRGPU_API void tsdrgpu_pipeline_destroy(tsdrgpu_pipeline_t *p);
/* == process(buf, items_count, ctx, samples_dropped): returns once h_iq has been read (it may then be reused) */
TSDRGPU_API int  tsdrgpu_pipeline_process(tsdrgpu_pipeline_t *p, const float *h_iq, uint64_t items_count, int64_t samples_dropped);
/* The same with the samples still in the front end's wire format (SURVEY section 8f-1): the block crosses PCIe as 1 or 2
 * bytes per component and is converted on the device to exactly the floats TSDRPlugin_RawFile.c:241-261 would have
 * produced on the host.  fmt uses the RawFile plugin's own numbering (TSDRPlugin_RawFile.c:29-33). */
enum { TSDRGPU_FMT_FLOAT = 0, TSDRGPU_FMT_INT8 = 1, TSDRGPU_FMT_INT16 = 2, TSDRGPU_FMT_UINT8 = 3, TSDRGPU_FMT_UINT16 = 4 };
/* the conversion alone, device to device (d_raw: items_count samples of `fmt`; d_out: items_count floats) */
TSDRGPU_API int  tsdrgpu_convert_samples(tsdrgpu_ctx_t *ctx, void *stream, const void *d_raw, int fmt, uint64_t items_count, float *d_out);
TSDRGPU_API int  tsdrgpu_pipeline_process_raw(tsdrgpu_pipeline_t *p, const void *h_samples, int fmt, uint64_t items_count, int64_t samples_dropped);
/* For a front end with a ring of page-locked buffers: returns once everything is enqueued; the buffer must stay untouched until
 * tsdrgpu_pipeline_sync_input() returns.  Consecutive blocks then cross the link back to back. */
TSDRGPU_API int  tsdrgpu_pipeline_process_raw_async(tsdrgpu_pipeline_t *p, const void *h_pinned_samples, int fmt, uint64_t items_count, int64_t samples_dropped);
TSDRGPU_API int  tsdrgpu_pipeline_sync_input(tsdrgpu_pipeline_t *p);
TSDRGPU_API int  tsdrgpu_pipeline_flush(tsdrgpu_pipeline_t *p);            /* waits for the GPU and for every pending callback */
TSDRGPU_API int  tsdrgpu_pipeline_set_param_int(tsdrgpu_pipeline_t *p, int id, uint32_t value);
TSDRGPU_API int  tsdrgpu_pipeline_set_resolution(tsdrgpu_pipeline_t *p, int height, double refreshrate);
TSDRGPU_API int  tsdrgpu_pipeline_set_samplerate(tsdrgpu_pipeline_t *p, uint32_t samplerate);
/* The tuner ahead of the pixel path (see tsdrgpu_tuner_*): every block is shifted by offset_hz, low-passed and decimated by
 * `decimation` right after it reaches the device (any ingest format), and the rest of the pipeline runs at samplerate /
 * decimation (geometry, decimator blocks, frame-rate detector, plots).  bandwidth_hz <= 0 switches it off (the default).
 * Checked against the current rate at once (TSDRGPU_EINVAL + text); takes effect at the next process() call, which then starts
 * over: tuner at position 0 with a zero history, samples and pixels waiting at the old rate discarded, resampler, frame stage
 * and frame-rate detector reset.  Superbandwidth mode bypasses the tuner and resumes it, reset, when it ends.
 * set_samplerate re-designs the taps for the new rate and rejects a rate the current tuning cannot take. */
TSDRGPU_API int  tsdrgpu_pipeline_set_tuner(tsdrgpu_pipeline_t *p, double offset_hz, double bandwidth_hz, int decimation, int ntaps);
/* The scan (see tsdrgpu_scan_*) over the wideband blocks: every non-empty block after it reaches the device, ahead of the tuner, so
 * its offsets are in the tuner's frame.  channels = 0 switches it off (the default).  Checked against the current rate at once;
 * takes effect, reset, at the next process() call.  It changes nothing the pixel path produces; its heavy part runs on a stream of
 * its own.  Superbandwidth mode pauses it; it resumes, reset, when that mode ends.  set_samplerate re-validates it. */
TSDRGPU_API int  tsdrgpu_pipeline_set_scan(tsdrgpu_pipeline_t *p, int channels, int taps_per_channel);
/* the scan's table (tsdrgpu_scan_results): *n = records written (0 while no scan runs); synchronises */
TSDRGPU_API int  tsdrgpu_pipeline_scan_results(tsdrgpu_pipeline_t *p, tsdrgpu_scan_channel_t *out, int cap, int *n);
/* The notch filter (see tsdrgpu_notch_*) on every non-empty block right after it reaches the device (any ingest format), after the
 * spectrum and ahead of the scan and the tuner.  n = 0 switches it off (the default).  Checked against the current rate at once
 * (TSDRGPU_EINVAL + text); takes effect at the next process() call, which then starts over behind it: notch, tuner and scan at
 * position 0, samples and pixels waiting discarded, resampler, frame stage and frame-rate detector reset.  Superbandwidth mode
 * bypasses it and resumes it, reset, when it ends.  set_samplerate re-designs the filter or rejects the rate. */
TSDRGPU_API int  tsdrgpu_pipeline_set_notches(tsdrgpu_pipeline_t *p, int n, const double *centers, const double *widths, int ntaps);
/* The power spectrum (see tsdrgpu_spectrum_*) of every non-empty block as received, at the capture's rate.  nfft = 0 switches it
 * off (the default).  Takes effect, reset, at the next process() call; the pixel path is not affected.  Superbandwidth mode
 * pauses it; it resumes, reset, when that mode ends. */
TSDRGPU_API int  tsdrgpu_pipeline_set_spectrum(tsdrgpu_pipeline_t *p, int nfft);
/* the spectrum (tsdrgpu_spectrum_results): *n = values written (0 while no spectrum runs), *segments averaged; synchronises */
TSDRGPU_API int  tsdrgpu_pipeline_spectrum(tsdrgpu_pipeline_t *p, double *out, int cap, int *n, uint64_t *segments);
/* superbandwidth mode (PARAM_AUTOCORR_SUPERRESOLUTION = 1; superb_run, superbandwidth.c:179-254) retunes the front end
 * between hops through this callback; without it the hops are recorded at one frequency */
TSDRGPU_API int  tsdrgpu_pipeline_set_retune(tsdrgpu_pipeline_t *p, tsdrgpu_retune_cb cb);
/* superbandwidth with ONE HOP PER GPU (tsdrgpu_superb_mgpu_*): devices[0] = the pipeline's own device, n in {2, 4, 8} hops =
 * devices of this node with peer access; hop i is recorded into device i's memory and transformed there, device 0 receives the
 * stitched magnitude stream and makes the frames.  n <= 1: back to 4 hops on one GPU (the reference's SUPER_HOPS_TO_MAKE). */
TSDRGPU_API int  tsdrgpu_pipeline_set_superb_devices(tsdrgpu_pipeline_t *p, const int *devices, int n);
/* Page-lock the caller's sample buffers in place (cudaHostRegister) once the same buffer has been handed to process() three
 * times, so that pageable plugin memory crosses PCIe by direct DMA.  Off by default: only for callers that keep their buffer
 * mapped for the whole run (the reference's plugins malloc once per tsdrplugin_readasync); released at destroy. */
TSDRGPU_API int  tsdrgpu_pipeline_set_host_registration(tsdrgpu_pipeline_t *p, int on);
TSDRGPU_API int  tsdrgpu_pipeline_set_motionblur(tsdrgpu_pipeline_t *p, float coeff);
/* SURVEY section 8f-2: deliver final pixels.  mode 1: the frame callback's buffer holds w*h int32 pixels of the JNI glue's
 * float->ARGB rule (TSDRLibraryNDK.c:222-283) instead of floats (same size, so the callback type is unchanged: cast it);
 * inverted as the GUI's "inverted colours".  mode 0 (default): floats, as the reference. */
TSDRGPU_API int  tsdrgpu_pipeline_set_output_argb(tsdrgpu_pipeline_t *p, int mode, int inverted);
/* SURVEY section 8f-4 / 8f-3, both off by default because the reference announces neither:
 *  report_snr:  value callback id 4 (VALUE_ID_SNR, TSDRLibrary.h:52) with dsp_autogain_t.snr next to every auto-gain report
 *               (the announce dsp.c:234 leaves commented out);
 *  detect_mode: after every pair of plots, value callback id TSDRGPU_VALUE_ID_DETECTED_MODE with (fps, height) computed
 *               like the GUI's auto-resolution (tsdrgpu_detect_videomode). */
#define TSDRGPU_VALUE_ID_DETECTED_MODE 100
TSDRGPU_API int  tsdrgpu_pipeline_set_reports(tsdrgpu_pipeline_t *p, int report_snr, int detect_mode);
TSDRGPU_API int  tsdrgpu_pipeline_sync(tsdrgpu_pipeline_t *p, int pixels);   /* tsdr_sync: syncoffset += pixels */
TSDRGPU_API int  tsdrgpu_pipeline_get_geometry(tsdrgpu_pipeline_t *p, int *width, int *height, double *refreshrate);
TSDRGPU_API int  tsdrgpu_pipeline_stats(tsdrgpu_pipeline_t *p, tsdrgpu_pipeline_stats_t *out);

#ifdef __cplusplus
}
#endif
#endif
