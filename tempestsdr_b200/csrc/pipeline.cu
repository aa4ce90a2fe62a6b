// pipeline.cu -- a1, a3, a5, a16, a17: the streaming glue between the plugin callback and the frame callback.
//
// Replaces the body of process() (TSDRLibrary.c:264-298), decimatingthread / postprocessingthread /
// videodecodingthread (TSDRLibrary.c:300-418), the three CircBuff rings between them (circbuff.c) and the
// frame-rate detector thread's capture loop (frameratedetector.c:128-187, 215-230).  Host buffers in, host frame
// and plot buffers out: this is the object the C host library (tempestsdr_b200/host/TSDRLibrary.c) drives from
// the reference's own process() callback, and the one bench.py times end to end.
//
// Data movement per IQ block: one H2D copy of the plugin's buffer (float32, or the front end's 8/16-bit wire format
// converted on the device: tsdrgpu_pipeline_process_raw),
// everything else stays in HBM: IQ -> (fused demod+resample) -> pixel stream -> (frame stage, batches of frames)
// -> one D2H copy of the finished frames into page-locked slots -> frame callback on the delivery thread.
// The reference's rings, which copy every sample 2x per stage under a mutex, do not exist here; what is kept
// is their observable behaviour: whole-block dropping with frame-aligned resynchronisation (dsp.c:313-368),
// purge of the autocorrelation capture on any drop (frameratedetector.c:221-224).
//
// Ordering differences to the (timing-dependent, SURVEY.md F9) threaded reference, both deterministic here:
//   * geometry changes made by the PLL take effect at the next batch boundary;
//   * tsdr_sync offsets are applied between batches of decimator blocks rather than between single blocks.
#include "common.cuh"
#include <math.h>
#include <pthread.h>
#include <deque>
#include <vector>

struct tsdrgpu_frd;
struct tsdrgpu_resampler;
struct tsdrgpu_framestage;
struct tsdrgpu_tuner;

namespace {

constexpr int PL_SLOTS = 4;

struct FrameJob {
	int kind;                 // 0 = frames, 1 = plots, 2 = barrier
	int slot, nframes, w, h;
	cudaEvent_t ev;
	uint32_t samplerate;      // plots
	int foff, flen, loff, llen; uint64_t calls; int reset_announce, dump_announce;
	int snr_valid;            // frames: results carry an SNR to announce
	int pll_valid;            // frames: h_pll_rr holds the refresh rates the PLL set
};

// block-aligned dropping, dsp.c:313-368 (integer bookkeeping, host side)
struct DropComp {
	int64_t difference = 0;
	static uint64_t debt(int block, int dropped) { const uint64_t whole = (uint64_t) (dropped / block); return ((whole + 1) * block - dropped) % block; }
	void shift_with(uint32_t block, int64_t syncoffset) {
		if (syncoffset >= 0) difference -= syncoffset % block; else difference -= block + syncoffset % block;
		if (difference < 0) difference = (int64_t) debt((int) block, (int) -difference);
	}
	bool will_drop_all(uint32_t size) const { return size <= difference; }
	// returns elements forwarded; *skip = leading elements discarded.  accepted = downstream took the block
	uint32_t add(uint32_t size, uint32_t block, bool accepted, uint32_t *skip) {
		*skip = 0;
		if (size <= difference) { difference -= size; *skip = size; return 0; }
		if (accepted) { const uint32_t lead = (uint32_t) difference; difference = 0; *skip = lead; return size - lead; }
		difference -= size % block;
		if (difference < 0) difference = (int64_t) debt((int) block, (int) -difference);
		return 0;
	}
};

__global__ void pl_copy_f32(const float *__restrict__ src, float *__restrict__ dst, size_t n) {
	for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) dst[i] = src[i];
}

// Raw sample formats of the RawFile front end converted on the device (SURVEY section 8f-1): the same values as the plugin's
// host loop (TSDRPlugin_RawFile.c:241-261) -- int8 v/128.0, uint8 (v-128)/128.0 (exact in float), int16 v/32767.0 and
// uint16 (v-32767)/32767.0 (double quotient rounded to float, exactly as the C expression).
__device__ __forceinline__ float raw_to_float(int v, int fmt) {
	switch (fmt) {
	case TSDRGPU_FMT_INT8:   return (float) v * 0.0078125f;
	case TSDRGPU_FMT_UINT8:  return (float) (v - 128) * 0.0078125f;
	case TSDRGPU_FMT_INT16:  return __double2float_rn(__ddiv_rn((double) v, 32767.0));
	default:                 return __double2float_rn(__ddiv_rn((double) (v - 32767), 32767.0));
	}
}
__global__ void __launch_bounds__(256) pl_convert(const void *__restrict__ raw, float *__restrict__ dst, size_t items, int fmt) {
	const size_t stride = (size_t) gridDim.x * blockDim.x, t0 = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
	if (fmt == TSDRGPU_FMT_INT8 || fmt == TSDRGPU_FMT_UINT8) {
		// 4 samples per thread only where both sides allow it (the superbandwidth gather appends at odd pair counts: dst is then
		// only 8-byte aligned); otherwise everything goes through the scalar tail loop
		const bool vec = ((reinterpret_cast<unsigned long long>(dst) & 15ull) == 0) && ((reinterpret_cast<unsigned long long>(raw) & 3ull) == 0);
		const size_t n4 = vec ? (items >> 2) : 0;
		for (size_t i = t0; i < n4; i += stride) {           // 4 samples per thread
			const uchar4 q = __ldg(reinterpret_cast<const uchar4 *>(raw) + i);
			float4 o;
			if (fmt == TSDRGPU_FMT_INT8) { o.x = raw_to_float((signed char) q.x, fmt); o.y = raw_to_float((signed char) q.y, fmt); o.z = raw_to_float((signed char) q.z, fmt); o.w = raw_to_float((signed char) q.w, fmt); }
			else { o.x = raw_to_float(q.x, fmt); o.y = raw_to_float(q.y, fmt); o.z = raw_to_float(q.z, fmt); o.w = raw_to_float(q.w, fmt); }
			reinterpret_cast<float4 *>(dst)[i] = o;
		}
		for (size_t i = (n4 << 2) + t0; i < items; i += stride) {
			const unsigned char b = reinterpret_cast<const unsigned char *>(raw)[i];
			dst[i] = raw_to_float(fmt == TSDRGPU_FMT_INT8 ? (int) (signed char) b : (int) b, fmt);
		}
		return;
	}
	for (size_t i = t0; i < items; i += stride) {                 // 16-bit formats: scalar (2-byte alignment is the format's own)
		const unsigned short u = __ldg(reinterpret_cast<const unsigned short *>(raw) + i);
		dst[i] = raw_to_float(fmt == TSDRGPU_FMT_INT16 ? (int) (short) u : (int) u, fmt);
	}
}
static inline size_t fmt_bytes(int fmt) { return fmt == TSDRGPU_FMT_FLOAT ? 4 : ((fmt == TSDRGPU_FMT_INT8 || fmt == TSDRGPU_FMT_UINT8) ? 1 : 2); }

}  // namespace

struct tsdrgpu_pipeline {
	tsdrgpu_ctx_t *ctx;
	tsdrgpu_pipeline_config_t cfg;
	tsdrgpu_frame_cb frame_cb; tsdrgpu_value_cb value_cb; tsdrgpu_plot_cb plot_cb; void *user;
	cudaStream_t s_main, s_copy, s_out, s_ingest;      // heavy kernels | H2D | D2H | light per-block kernels
	cudaEvent_t ev_ingest, ev_decim, ev_cap_used[2];
	cudaEvent_t ev_out[2], ev_main; int out_phase;
	cudaEvent_t ev_h2d[4], ev_used[4]; int stage_slot;

	// live geometry (set_internal_samplerate)
	pthread_mutex_t geo_mu;
	uint32_t samplerate; int height, width; double refreshrate, pixelrate, ptos;
	float motionblur; volatile int syncoffset;
	volatile int report_snr, detect_mode;              // 8f-4 / 8f-3, both off by default (the reference announces neither)
	volatile int argb_mode, argb_inverted; int32_t *d_argb_last; size_t argb_cap;      // 8f-2: final pixels instead of floats
	uint32_t params[9];

	// stage 0: H2D staging of the plugin's buffer
	float *d_stage[4]; size_t stage_cap[4];           // floats; 4 slots so H2D runs ahead of the kernels
	void *d_raw[4]; size_t raw_cap[4];                // bytes; raw-format blocks land here and are converted into d_stage
	// plugin buffers seen on process(): page-locked in place (cudaHostRegister) once the same buffer keeps coming back, so that
	// an unmodified plugin's malloc'd block crosses PCIe by direct DMA instead of through the driver's staging copy
	struct HostBuf { const void *base; size_t bytes; int seen; int state; };      // state: 0 candidate, 1 registered here, 2 pinned by its owner, 3 refused
	std::vector<HostBuf> hostbufs; int host_register;
	// stage 1: decimator input (IQ pairs waiting for whole blocks)
	// samples waiting for whole decimator blocks: [decim_read, decim_read + decim_fill) samples of decim_elem floats each
	// (2 = interleaved I,Q, demodulated inside rs_main; 1 = magnitudes, what the multi-GPU superbandwidth stitch delivers).
	// Consumed from the front by moving decim_read; compacted only when the hole in front is at least as large as what is
	// left, so source and destination of the move never overlap.
	float *d_decim; size_t decim_cap /* floats */, decim_fill, decim_read; int decim_elem;
	DropComp dev_drop;
	// stage 2: pixels waiting for whole frames
	tsdrgpu_resampler *rs;
	float *d_pix; size_t pix_cap, pix_read, pix_fill;
	DropComp pix_drop;
	// stage 3: frames
	tsdrgpu_framestage *fs;
	float *d_frames[2]; size_t frames_cap[2];          // double-buffered: D2H of batch k overlaps the kernels of batch k+1
	float *h_frames[PL_SLOTS]; tsdrgpu_frame_result_t *h_results[PL_SLOTS]; int32_t *h_report[PL_SLOTS]; size_t slot_cap;
	double *h_pll_rr[PL_SLOTS];                        // refresh rate after frame f when the PLL moved it there (NaN: it did not)
	cudaEvent_t ev_res;                                // the batch's sync results have reached the host (PLL write-back needs them)
	int slot_busy[PL_SLOTS];
	// autocorrelation side path
	tsdrgpu_frd *frd; float *d_capture[2]; size_t cap_size[2], cap_fill; int cap_phase; uint32_t cap_rate;
	double *h_plot_frame[2], *h_plot_line[2]; size_t plot_cap; int plot_slot; int plot_busy[2];
	int32_t *h_peaks[2];                               // where the two plots peak, picked on the device (8f-3)
	// superbandwidth (superb_run's state machine, superbandwidth.c:179-264)
	struct {
		int state; int buffid; long long to_gather, gathered, in_frame, to_pause; uint32_t rate;
		int nhops;                                    // SUPER_HOPS_TO_MAKE (superbandwidth.c:22): 4, or the number of devices when the hops are sharded
		float *d_hops[16]; size_t hop_cap; float *d_out; size_t out_cap; cudaEvent_t ev;
		// one hop per GPU (tsdrgpu_pipeline_set_superb_devices): rank i records hop i on device dev[i]; rank 0 is this pipeline's device
		int ndev; int dev[16]; tsdrgpu_ctx_t *rctx[16]; tsdrgpu_superb_mgpu_t *grp[16]; cudaStream_t rstream[16], rcopy[16]; cudaEvent_t rev[16];
		void *rraw[16]; size_t rraw_cap[16]; uint32_t grp_pairs;
		float *d_hop0[16];                            // every device's copy of hop 0, the alignment reference (filled when hop 0 is complete)
	} sb;
	uint32_t samplerate_real;
	tsdrgpu_retune_cb retune_cb;
	// tuner (tsdrgpu_pipeline_set_tuner): tn_cfg is the latest request (geo_mu), applied by the next process() call
	struct { double offset, bw; int D, ntaps; } tn_cfg; int tn_dirty;
	tsdrgpu_tuner *tuner; int tn_on, tn_D; uint64_t tn_pos;           // what runs; tn_pos mirrors the tuner's input position
	float *d_tout[4]; size_t tout_cap[4];                               // the tuner's output per staging slot (floats)
	// scan (tsdrgpu_pipeline_set_scan): sc_cfg is the latest request (geo_mu), applied by the next process() call
	struct { int K, Q; } sc_cfg; int sc_dirty;
	tsdrgpu_scan_t *scan; int sc_on;
	// notch filter (tsdrgpu_pipeline_set_notches): nt_cfg is the latest request (geo_mu), applied by the next process() call
	struct { int n, ntaps; double centers[32], widths[32]; } nt_cfg; int nt_dirty;
	tsdrgpu_notch_t *notch; int nt_on;
	float *d_nout[4]; size_t nout_cap[4];                               // the notch's output per staging slot (floats)
	// spectrum (tsdrgpu_pipeline_set_spectrum): sp_nfft is the latest request (geo_mu), applied by the next process() call
	int sp_nfft, sp_dirty;
	tsdrgpu_spectrum_t *spectrum; int sp_on;
	// delivery
	pthread_t thread; pthread_mutex_t mu; pthread_cond_t cv_job, cv_done;
	std::deque<FrameJob> jobs; int stop; uint64_t submitted, delivered;
	tsdrgpu_pipeline_stats_t stats;
	int last_w, last_h;
};

extern "C" {
int tsdrgpu_resampler_create(tsdrgpu_ctx_t *, tsdrgpu_resampler **);
}
enum { SB_STOPPED = 0, SB_STARTING, SB_GATHERING, SB_PAUSE };

static void geometry_locked(tsdrgpu_pipeline *p) {      // set_internal_samplerate, TSDRLibrary.c:540-550
	double pr, pt; int w;
	tsdrgpu_geometry(p->samplerate, p->height, p->refreshrate, &w, &pr, &pt);
	p->width = w; p->pixelrate = pr;
	if (p->samplerate != 0 && pr != 0) p->ptos = pt;
}

static void *delivery_main(void *arg) {
	tsdrgpu_pipeline *p = (tsdrgpu_pipeline *) arg;
	cudaSetDevice(p->ctx->device);
	tsdrgpu_bind_thread_near_device(p->ctx);          // the frames it hands out live in page-locked memory on the device's node
	for (;;) {
		pthread_mutex_lock(&p->mu);
		while (p->jobs.empty() && !p->stop) pthread_cond_wait(&p->cv_job, &p->mu);
		if (p->jobs.empty() && p->stop) { pthread_mutex_unlock(&p->mu); break; }
		FrameJob j = p->jobs.front(); p->jobs.pop_front();
		pthread_mutex_unlock(&p->mu);
		cudaEventSynchronize(j.ev);
		if (j.kind == 0) {
			const size_t n = (size_t) j.w * j.h;
			for (int f = 0; f < j.nframes; f++) {
				const tsdrgpu_frame_result_t &r = p->h_results[j.slot][f];
				// frameratepll's announce (syncdetector.c:151): the write-back itself happened in drain_frames, in stream order
				if (j.pll_valid && p->h_pll_rr[j.slot][f] == p->h_pll_rr[j.slot][f] && p->value_cb)
					p->value_cb(0 /* VALUE_ID_PLL_FRAMERATE */, p->h_pll_rr[j.slot][f], 0, p->user);
				if (p->h_report[j.slot][f] && p->value_cb) p->value_cb(3 /* VALUE_ID_AUTOGAIN_VALUES */, r.lastmin, r.lastmax, p->user);
				if (p->h_report[j.slot][f] && p->value_cb && j.snr_valid) p->value_cb(4 /* VALUE_ID_SNR: the announce dsp.c:234 leaves commented out */, r.snr, 0, p->user);
				if (p->frame_cb) p->frame_cb(p->h_frames[j.slot] + f * n, j.w, j.h, p->user);
			}
			pthread_mutex_lock(&p->mu);
			p->slot_busy[j.slot] = 0; p->stats.frames_delivered += j.nframes;
			pthread_mutex_unlock(&p->mu);
		} else if (j.kind == 1) {
			if (j.reset_announce && p->value_cb) p->value_cb(1 /* VALUE_ID_AUTOCORRECT_RESET */, 0, 0, p->user);
			if (j.dump_announce && p->value_cb) p->value_cb(5 /* VALUE_ID_AUTOCORRECT_DUMPED, frameratedetector.c:115 */, 0, 0, p->user);
			if (p->plot_cb) {
				p->plot_cb(0 /* PLOT_ID_FRAME */, j.foff, p->h_plot_frame[j.slot], j.flen, j.samplerate, p->user);
				p->plot_cb(1 /* PLOT_ID_LINE */, j.loff, p->h_plot_line[j.slot], j.llen, j.samplerate, p->user);
			}
			if (p->value_cb) p->value_cb(2 /* VALUE_ID_AUTOCORRECT_FRAMES_COUNT */, 0, (double) j.calls, p->user);
			if (p->detect_mode && p->value_cb && j.flen > 0 && j.llen > 0) {
				double fps = 0; int height = 0;
				tsdrgpu_detect_videomode(p->h_plot_frame[j.slot], j.foff, j.flen, p->h_plot_line[j.slot], j.loff, j.llen, j.samplerate, &fps, &height, NULL, NULL);
				p->value_cb(TSDRGPU_VALUE_ID_DETECTED_MODE, fps, (double) height, p->user);
			}
			pthread_mutex_lock(&p->mu);
			p->plot_busy[j.slot] = 0; p->stats.plots_delivered++;
			pthread_mutex_unlock(&p->mu);
		}
		cudaEventDestroy(j.ev);
		pthread_mutex_lock(&p->mu);
		p->delivered++;
		pthread_cond_broadcast(&p->cv_done);
		pthread_mutex_unlock(&p->mu);
	}
	return NULL;
}

static int submit(tsdrgpu_pipeline *p, FrameJob &j, cudaStream_t on) {
	tsdrgpu_ctx_t *ctx = p->ctx;
	CU_TRY(ctx, cudaEventCreateWithFlags(&j.ev, cudaEventDisableTiming));
	CU_TRY(ctx, cudaEventRecord(j.ev, on));
	pthread_mutex_lock(&p->mu);
	p->jobs.push_back(j); p->submitted++;
	pthread_cond_signal(&p->cv_job);
	pthread_mutex_unlock(&p->mu);
	return TSDRGPU_OK;
}

static int grow(tsdrgpu_ctx_t *ctx, cudaStream_t s, float **buf, size_t *cap, size_t need, size_t keep_floats) {
	if (*cap >= need) return TSDRGPU_OK;
	float *nb;
	const size_t ncap = need + need / 2 + 1024;
	CU_TRY(ctx, cudaMalloc(&nb, sizeof(float) * ncap));
	if (*buf && keep_floats) CU_TRY(ctx, cudaMemcpyAsync(nb, *buf, sizeof(float) * keep_floats, cudaMemcpyDeviceToDevice, s));
	CU_TRY(ctx, cudaStreamSynchronize(s));
	if (*buf) CU_TRY(ctx, cudaFree(*buf));
	*buf = nb; *cap = ncap;
	return TSDRGPU_OK;
}

// room for `more` samples behind the ones waiting in the decimator input (contents kept); returns where they go
static int decim_reserve(tsdrgpu_pipeline *p, size_t more, float **where) {
	const size_t E = (size_t) p->decim_elem, used = E * (p->decim_read + p->decim_fill);
	int rc = grow(p->ctx, p->s_main, &p->d_decim, &p->decim_cap, used + E * more, used);
	if (rc) return rc;
	*where = p->d_decim + used;
	return TSDRGPU_OK;
}
// the decimator input switches between I,Q pairs and magnitudes: what is still waiting is converted (rare: at most a few
// blocks, when superbandwidth mode with one hop per GPU starts or ends)
static int decim_set_elem(tsdrgpu_pipeline *p, int elem) {
	tsdrgpu_ctx_t *ctx = p->ctx;
	if (p->decim_elem == elem) return TSDRGPU_OK;
	CU_TRY(ctx, cudaStreamSynchronize(p->s_ingest));
	const size_t n = p->decim_fill;
	int rc;
	if (n) {
		void *tmp;
		float *src = p->d_decim + (size_t) p->decim_elem * p->decim_read;
		if ((rc = tsdrgpu_scratch(ctx, 3, sizeof(float) * 2 * n, &tmp))) return rc;
		if (elem == 1) {                                  // pairs -> magnitudes (am_demod, TSDRLibrary.c:244-262)
			if ((rc = tsdrgpu_am_demod(ctx, p->s_main, src, n, (float *) tmp))) return rc;
			CU_TRY(ctx, cudaMemcpyAsync(p->d_decim, tmp, sizeof(float) * n, cudaMemcpyDeviceToDevice, p->s_main));
		} else {                                          // magnitudes -> pairs (m, 0): |(m, 0)| == m
			CU_TRY(ctx, cudaMemsetAsync(tmp, 0, sizeof(float) * 2 * n, p->s_main));
			CU_TRY(ctx, cudaMemcpy2DAsync(tmp, 2 * sizeof(float), src, sizeof(float), sizeof(float), n, cudaMemcpyDeviceToDevice, p->s_main));
			if ((rc = grow(ctx, p->s_main, &p->d_decim, &p->decim_cap, 2 * n, 0))) return rc;
			CU_TRY(ctx, cudaMemcpyAsync(p->d_decim, tmp, sizeof(float) * 2 * n, cudaMemcpyDeviceToDevice, p->s_main));
		}
		CU_TRY(ctx, cudaEventRecord(p->ev_decim, p->s_main));
	}
	p->decim_read = 0; p->decim_elem = elem;
	return TSDRGPU_OK;
}

// A plugin hands over the same malloc'd buffer call after call (TSDRPlugin_RawFile.c:212, Mirics, SDRplay).  From pageable memory
// cudaMemcpyAsync goes through the driver's staging buffer at a fraction of the link rate; once a buffer has come back
// REG_AFTER times it is page-locked in place.  Buffers are released again when the run ends (tsdrgpu_pipeline_destroy).
// OPT-IN (tsdrgpu_pipeline_set_host_registration): a registration pins the PHYSICAL pages behind an address range, so it is
// only safe for a caller that keeps its buffer mapped for the whole run, as the reference's plugins do (one malloc per
// tsdrplugin_readasync).  A caller that frees and re-allocates a buffer per call (numpy temporaries land on the same address
// again and again) would be read through the stale mapping -- measured: wrong frames, then cudaErrorInvalidValue.  The C host
// library switches it on for the plugins it loads (TSDR_NO_HOST_REGISTER=1 keeps it off).
static const void *host_source(tsdrgpu_pipeline *p, const void *h, size_t bytes) {
	constexpr int REG_AFTER = 3;
	if (!p->host_register || bytes < 65536 || h == NULL) return h;
	for (auto &b : p->hostbufs) {
		if (b.base != h) continue;
		if (b.state == 1 && bytes > b.bytes) { cudaHostUnregister(const_cast<void *>(b.base)); cudaGetLastError(); b.state = 0; b.seen = REG_AFTER - 1; }
		if (b.state != 0) return h;
		if (++b.seen < REG_AFTER) return h;
		cudaPointerAttributes a;
		if (cudaPointerGetAttributes(&a, h) == cudaSuccess && a.type != cudaMemoryTypeUnregistered) { b.state = 2; return h; }
		cudaGetLastError();
		if (cudaHostRegister(const_cast<void *>(h), bytes, cudaHostRegisterDefault) == cudaSuccess) { b.state = 1; b.bytes = bytes; p->stats.host_buffers_registered++; }
		else { cudaGetLastError(); b.state = 3; }
		return h;
	}
	if (p->hostbufs.size() >= 8) {
		if (p->hostbufs.front().state == 1) { cudaHostUnregister(const_cast<void *>(p->hostbufs.front().base)); cudaGetLastError(); }
		p->hostbufs.erase(p->hostbufs.begin());
	}
	p->hostbufs.push_back({h, bytes, 1, 0});
	return h;
}

// ---- autocorrelation side path: append demodulated samples, fire a capture when full (frameratedetector.c:128-230)
static int feed_capture(tsdrgpu_pipeline *p, const float *d_iq, uint64_t pairs, bool dropped) {
	tsdrgpu_ctx_t *ctx = p->ctx;
	if (p->params[TSDRGPU_PARAM_AUTOCORR_PLOTS_OFF]) return TSDRGPU_OK;
	if (dropped) { p->cap_fill = 0; return TSDRGPU_OK; }              // cb_purge on any drop
	if (p->cap_rate != p->samplerate) { p->cap_rate = p->samplerate; p->cap_fill = 0; }
	const size_t want = tsdrgpu_frd_capture_size(p->samplerate);
	if (want == 0) return TSDRGPU_OK;
	int rc;
	for (int i = 0; i < 2; i++) if (p->cap_size[i] < want) {
		CU_TRY(ctx, cudaStreamSynchronize(p->s_ingest));
		if ((rc = grow(ctx, p->s_main, &p->d_capture[i], &p->cap_size[i], want, (i == p->cap_phase) ? p->cap_fill : 0))) return rc;
	}
	uint64_t done = 0;
	while (done < pairs) {
		const uint64_t take = (want - p->cap_fill) < (pairs - done) ? (want - p->cap_fill) : (pairs - done);
		float *cap = p->d_capture[p->cap_phase];
		if (p->cap_fill == 0) CU_TRY(ctx, cudaStreamWaitEvent(p->s_ingest, p->ev_cap_used[p->cap_phase], 0));   // the FFT that last read it is done
		if ((rc = tsdrgpu_am_demod(ctx, p->s_ingest, d_iq + 2 * done, take, cap + p->cap_fill))) return rc;
		p->cap_fill += take; done += take;
		if (p->cap_fill == want) {
			p->cap_fill = 0;
			const int cph = p->cap_phase; p->cap_phase ^= 1;
			CU_TRY(ctx, cudaEventRecord(p->ev_ingest, p->s_ingest));
			CU_TRY(ctx, cudaStreamWaitEvent(p->s_main, p->ev_ingest, 0));
			int reset_announce = 0;
			if (p->params[TSDRGPU_PARAM_AUTOCORR_PLOTS_RESET]) {          // frameratedetector.c:97-104
				reset_announce = (p->params[TSDRGPU_PARAM_AUTOCORR_PLOTS_RESET] == 1);
				p->params[TSDRGPU_PARAM_AUTOCORR_PLOTS_RESET] = 0;
				tsdrgpu_frd_reset(p->frd);
			}
			int fmin, fmax, lmin, lmax;
			tsdrgpu_frd_windows(p->samplerate, &fmin, &fmax, &lmin, &lmax);
			const size_t need = (size_t) (fmax - fmin) + 8;
			// pick a free plot slot; when the host is slower than the GPU the capture is still accumulated on
			// the device, only this particular plot delivery is skipped
			pthread_mutex_lock(&p->mu);
			int slot = -1;
			for (int s = 0; s < 2; s++) if (!p->plot_busy[s]) { slot = s; break; }
			if (slot >= 0) p->plot_busy[slot] = 1;
			pthread_mutex_unlock(&p->mu);
			if (p->plot_cap < need) {
				CU_TRY(ctx, cudaStreamSynchronize(p->s_main));
				pthread_mutex_lock(&p->mu);
				while (p->delivered < p->submitted) pthread_cond_wait(&p->cv_done, &p->mu);
				pthread_mutex_unlock(&p->mu);
				for (int s = 0; s < 2; s++) {
					if (p->h_plot_frame[s]) { cudaFreeHost(p->h_plot_frame[s]); cudaFreeHost(p->h_plot_line[s]); cudaFreeHost(p->h_peaks[s]); }
					if ((rc = tsdrgpu_malloc_host(ctx, 64, (void **) &p->h_peaks[s]))) return rc;
					if ((rc = tsdrgpu_malloc_host(ctx, sizeof(double) * need, (void **) &p->h_plot_frame[s]))) return rc;
					if ((rc = tsdrgpu_malloc_host(ctx, sizeof(double) * need, (void **) &p->h_plot_line[s]))) return rc;
				}
				p->plot_cap = need;
			}
			int dump_announce = 0;
			if (p->params[TSDRGPU_PARAM_AUTOCORR_DUMP]) {                    // frameratedetector.c:110-116: "autocorr.csv" in the working directory
				p->params[TSDRGPU_PARAM_AUTOCORR_DUMP] = 0;
				if ((rc = tsdrgpu_frd_dump_csv(p->frd, p->s_main, p->samplerate, cap, (uint32_t) want, "autocorr.csv"))) return rc;
				dump_announce = 1;
			}
			uint64_t calls = 0;
			if ((rc = tsdrgpu_frd_run_async(p->frd, p->s_main, p->samplerate, cap, (uint32_t) want,
			                                slot >= 0 ? p->h_plot_frame[slot] : NULL, fmax - fmin,
			                                slot >= 0 ? p->h_plot_line[slot] : NULL, lmax - lmin, &calls))) return rc;
			if (slot >= 0 && (rc = tsdrgpu_frd_peaks_async(p->frd, p->s_main, p->h_peaks[slot]))) return rc;
			CU_TRY(ctx, cudaEventRecord(p->ev_cap_used[cph], p->s_main));
			p->stats.captures++;
			if (slot >= 0) {
				FrameJob j; memset(&j, 0, sizeof j);
				j.kind = 1; j.slot = slot; j.samplerate = p->samplerate; j.foff = fmin; j.flen = fmax - fmin; j.loff = lmin; j.llen = lmax - lmin;
				j.calls = calls; j.reset_announce = reset_announce; j.dump_announce = dump_announce;
				if ((rc = submit(p, j, p->s_main))) return rc;
			}
		}
	}
	return TSDRGPU_OK;
}

// ---- pixels -> frames (postprocessingthread + videodecodingthread)
static int drain_frames(tsdrgpu_pipeline *p, int w, int h) {
	tsdrgpu_ctx_t *ctx = p->ctx;
	const size_t n = (size_t) w * h;
	int rc;
	const int batch = p->cfg.batch_frames > 0 ? p->cfg.batch_frames : 1;
	while (p->pix_fill - p->pix_read >= n * (size_t) batch) {
		const int nf = batch;
		// a free delivery slot, or the batch is dropped whole (frames stay aligned), as a full ring would (circbuff.c:95-104)
		pthread_mutex_lock(&p->mu);
		int slot = -1;
		for (int s = 0; s < PL_SLOTS; s++) if (!p->slot_busy[s]) { slot = s; break; }
		if (slot >= 0) p->slot_busy[slot] = 1;
		pthread_mutex_unlock(&p->mu);
		if (slot < 0 && p->cfg.block_when_busy) {
			pthread_mutex_lock(&p->mu);
			while (slot < 0) {
				for (int s = 0; s < PL_SLOTS; s++) if (!p->slot_busy[s]) { slot = s; break; }
				if (slot < 0) pthread_cond_wait(&p->cv_done, &p->mu);
			}
			p->slot_busy[slot] = 1;
			pthread_mutex_unlock(&p->mu);
		}
		if (slot < 0) { p->pix_read += n * nf; p->stats.frames_dropped += nf; continue; }
		if (p->slot_cap < n * nf) {
			CU_TRY(ctx, cudaStreamSynchronize(p->s_main));
			pthread_mutex_lock(&p->mu);
			while (p->delivered < p->submitted) pthread_cond_wait(&p->cv_done, &p->mu);
			pthread_mutex_unlock(&p->mu);
			for (int s = 0; s < PL_SLOTS; s++) {
				if (p->h_frames[s]) { cudaFreeHost(p->h_frames[s]); cudaFreeHost(p->h_results[s]); cudaFreeHost(p->h_report[s]); free(p->h_pll_rr[s]); }
				p->h_pll_rr[s] = (double *) malloc(sizeof(double) * nf);
				if ((rc = tsdrgpu_malloc_host(ctx, sizeof(float) * n * nf, (void **) &p->h_frames[s]))) return rc;
				if ((rc = tsdrgpu_malloc_host(ctx, sizeof(tsdrgpu_frame_result_t) * nf, (void **) &p->h_results[s]))) return rc;
				if ((rc = tsdrgpu_malloc_host(ctx, sizeof(int32_t) * nf, (void **) &p->h_report[s]))) return rc;
			}
			p->slot_cap = n * nf;
		}
		const int op = p->out_phase; p->out_phase ^= 1;
		if ((rc = grow(ctx, p->s_main, &p->d_frames[op], &p->frames_cap[op], n * nf, 0))) return rc;
		CU_TRY(ctx, cudaStreamWaitEvent(p->s_main, p->ev_out[op], 0));       // the D2H that last read this buffer is done
		unsigned flags = 0;
		if (p->params[TSDRGPU_PARAM_INT_AUTOSHIFT]) flags |= TSDRGPU_FS_AUTOSHIFT;
		if (p->params[TSDRGPU_PARAM_LOW_PASS_BEFORE_SYNC]) flags |= TSDRGPU_FS_LOWPASS_BEFORE_SYNC;
		if (p->params[TSDRGPU_PARAM_AUTOGAIN_AFTER_PROCESSING]) flags |= TSDRGPU_FS_AUTOGAIN_AFTER_PROC;
		if (p->params[TSDRGPU_PARAM_AUTOCORR_SUPERRESOLUTION]) flags |= TSDRGPU_FS_SUPERRESOLUTION;
		const int want_snr = p->report_snr;
		if (want_snr) flags |= TSDRGPU_FS_COMPUTE_SNR;
		if ((rc = tsdrgpu_framestage_run_async(p->fs, p->s_main, p->d_pix + p->pix_read, nf, w, h, p->motionblur,
		                                       0.1f /* NORMALISATION_LOWPASS_COEFF, TSDRLibrary.c:37 */, flags, p->d_frames[op],
		                                       p->h_results[slot], p->h_report[slot]))) return rc;
		// the frames become valid on the frame stage's side stream: copy them out on the output stream behind it
		CU_TRY(ctx, cudaEventRecord(p->ev_main, p->s_main));
		CU_TRY(ctx, cudaStreamWaitEvent(p->s_out, p->ev_main, 0));             // serial stage orders finish on the main stream
		if ((rc = tsdrgpu_framestage_join(p->fs, p->s_out))) return rc;        // the overlapped order finishes on the side stream
		const bool pll_on = p->params[TSDRGPU_PARAM_INT_FRAMERATE_PLL] != 0;
		if (pll_on) CU_TRY(ctx, cudaEventRecord(p->ev_res, p->s_out));          // the batch's results are on the host behind this
		if (p->argb_mode) {                                                    // float frames -> the host's int32 pixels, in place
			if (p->argb_cap != n) {
				if (p->d_argb_last) CU_TRY(ctx, cudaFree(p->d_argb_last));
				CU_TRY(ctx, cudaMalloc(&p->d_argb_last, sizeof(int32_t) * n));
				CU_TRY(ctx, cudaMemsetAsync(p->d_argb_last, 0, sizeof(int32_t) * n, p->s_out));
				p->argb_cap = n;
			}
			if ((rc = tsdrgpu_pixels_argb_batch(ctx, p->s_out, p->d_frames[op], n, nf, p->argb_inverted, p->d_argb_last))) return rc;
		}
		CU_TRY(ctx, cudaMemcpyAsync(p->h_frames[slot], p->d_frames[op], sizeof(float) * n * nf, cudaMemcpyDeviceToHost, p->s_out));
		CU_TRY(ctx, cudaEventRecord(p->ev_out[op], p->s_out));
		p->stats.d2h_bytes += sizeof(float) * n * nf;
		p->pix_read += n * nf;
		p->stats.frames_processed += nf;
		FrameJob j; memset(&j, 0, sizeof j);
		j.kind = 0; j.slot = slot; j.nframes = nf; j.w = w; j.h = h; j.snr_valid = want_snr; j.pll_valid = pll_on;
		if (pll_on) {
			// frameratepll's write-back (syncdetector.c:141-152).  The reference does it from its post-processing thread while the
			// decimating thread reads refreshrate unlocked (SURVEY F9); here it is applied in stream order: the results of this
			// batch move the refresh rate before the decimator plans its next group of blocks, frame by frame in order.  The
			// price is one host wait per batch, paid only while the PLL is switched on (the frames' D2H is already queued).
			CU_TRY(ctx, cudaEventSynchronize(p->ev_res));
			for (int f = 0; f < nf; f++) {
				const tsdrgpu_frame_result_t &r = p->h_results[slot][f];
				pthread_mutex_lock(&p->geo_mu);
				double rr = p->refreshrate;
				const int moved = tsdrgpu_pll_step(&rr, r.x_vx, r.pll_state, r.avg_speed);
				if (moved) { p->refreshrate = rr; geometry_locked(p); }
				pthread_mutex_unlock(&p->geo_mu);
				p->h_pll_rr[slot][f] = moved ? rr : nan("");
			}
		}
		if ((rc = submit(p, j, p->s_out))) return rc;
	}
	// compact the pixel buffer when the consumed prefix is large
	if (p->pix_read > 0 && p->pix_read >= (p->pix_fill - p->pix_read)) {
		const size_t left = p->pix_fill - p->pix_read;
		if (left) {
			pl_copy_f32<<<(unsigned) ((left + 255) / 256 < 1024 ? (left + 255) / 256 : 1024), 256, 0, p->s_main>>>(p->d_pix + p->pix_read, p->d_pix, left);
			LAUNCH_CHECK(ctx);
		}
		p->pix_read = 0; p->pix_fill = left;
	}
	return TSDRGPU_OK;
}

// ---- samples -> pixels (decimatingthread)
static int drain_blocks(tsdrgpu_pipeline *p) {
	tsdrgpu_ctx_t *ctx = p->ctx;
	int rc;
	for (;;) {
		// the live geometry, read again for every group of blocks: the PLL (drain_frames) or the host may have moved it
		pthread_mutex_lock(&p->geo_mu);
		const int w = p->width, h = p->height; const double fv = p->refreshrate; const uint32_t fs_ = p->samplerate;
		pthread_mutex_unlock(&p->geo_mu);
		if (w <= 0 || h <= 0) return TSDRGPU_OK;
		p->last_w = w; p->last_h = h;
		const uint32_t block = (uint32_t) (0.1 * fs_ / fv);                 // FRAMES_TO_POLL, TSDRLibrary.c:41,335
		if (block == 0) return TSDRGPU_OK;
		const uint32_t min_blocks = p->cfg.batch_blocks > 0 ? (uint32_t) p->cfg.batch_blocks : 10;
		if (p->decim_fill / block < min_blocks) return TSDRGPU_OK;
		// whole multiples of the batch size, so the grouping (and with it every result) does not depend on how the
		// plugin happened to cut the stream into process() calls; with the PLL on exactly one group at a time, because the
		// frames it completes may move the refresh rate the next group is resampled with
		uint32_t nb = (uint32_t) ((p->decim_fill / block / min_blocks) * min_blocks);
		if (nb > 4000) nb = (4000 / min_blocks) * min_blocks;
		if (nb == 0 || p->params[TSDRGPU_PARAM_INT_FRAMERATE_PLL]) nb = min_blocks;
		const double up = (double) (w * h) * fv;        // width*height*refreshrate, TSDRLibrary.c:340
		const uint64_t npix = tsdrgpu_resampler_plan(p->rs, NULL, block, nb, up, (double) fs_);
		if (npix == 0) return tsdrgpu_fail(ctx, TSDRGPU_EINVAL, "resampler plan produced no pixels", cudaSuccess, __FILE__, __LINE__);
		if ((rc = grow(ctx, p->s_main, &p->d_pix, &p->pix_cap, p->pix_fill + npix + 64, p->pix_fill))) return rc;
		uint64_t n_out = 0;
		if ((rc = tsdrgpu_resampler_run(p->rs, p->s_main, p->d_decim + (size_t) p->decim_elem * p->decim_read, p->decim_elem == 2, NULL, block, nb, up, (double) fs_,
		                                (int) p->params[TSDRGPU_PARAM_NEAREST_NEIGHBOUR_RESAMPLING], p->d_pix + p->pix_fill,
		                                p->pix_cap - p->pix_fill, &n_out))) return rc;
		// pixel-level alignment (dsp.c:326-346 on the pixel ring) and manual sync (TSDRLibrary.c:344-346)
		const uint32_t totalpixels = (uint32_t) (w * h);
		uint32_t skip = 0;
		const uint32_t fwd = p->pix_drop.add((uint32_t) n_out, totalpixels, true, &skip);
		if (skip && fwd) {                               // rare (after drops / manual sync): shift through scratch, ranges overlap
			void *tmp;
			if ((rc = tsdrgpu_scratch(ctx, 3, sizeof(float) * fwd, &tmp))) return rc;
			const unsigned g = (unsigned) ((fwd + 255) / 256 < 1024 ? (fwd + 255) / 256 : 1024);
			pl_copy_f32<<<g, 256, 0, p->s_main>>>(p->d_pix + p->pix_fill + skip, (float *) tmp, fwd); LAUNCH_CHECK(ctx);
			pl_copy_f32<<<g, 256, 0, p->s_main>>>((const float *) tmp, p->d_pix + p->pix_fill, fwd); LAUNCH_CHECK(ctx);
		}
		p->pix_fill += fwd;
		const int so = p->syncoffset; p->syncoffset = 0;
		p->pix_drop.shift_with(totalpixels, -(int64_t) so);
		// consume the blocks; move what is left to the front once the hole there is big enough for a non-overlapping move
		const size_t used = (size_t) nb * block, left = p->decim_fill - used, E = (size_t) p->decim_elem;
		p->decim_read += used; p->decim_fill = left;
		if (left == 0) p->decim_read = 0;
		else if (p->decim_read >= left) {
			pl_copy_f32<<<(unsigned) ((E * left + 255) / 256 < 1024 ? (E * left + 255) / 256 : 1024), 256, 0, p->s_main>>>(p->d_decim + E * p->decim_read, p->d_decim, E * left); LAUNCH_CHECK(ctx);
			p->decim_read = 0;
		}
		CU_TRY(ctx, cudaEventRecord(p->ev_decim, p->s_main));                // later appends (ingest stream) must come after this
		p->stats.samples_resampled += used;
		if ((rc = drain_frames(p, w, h))) return rc;
	}
}

extern "C" {

static void superb_release_devices(tsdrgpu_pipeline *p);

int tsdrgpu_pipeline_create(tsdrgpu_ctx_t *ctx, const tsdrgpu_pipeline_config_t *cfg, tsdrgpu_frame_cb frame_cb,
                            tsdrgpu_value_cb value_cb, tsdrgpu_plot_cb plot_cb, void *user, tsdrgpu_pipeline_t **out) {
	BIND(ctx); ARG_TRY(ctx, cfg != NULL && out != NULL);
	ARG_TRY(ctx, cfg->samplerate > 0 && cfg->height > 0 && cfg->refreshrate > 0);
	tsdrgpu_pipeline *p = new tsdrgpu_pipeline();
	p->ctx = ctx; p->cfg = *cfg; p->frame_cb = frame_cb; p->value_cb = value_cb; p->plot_cb = plot_cb; p->user = user;
	p->samplerate = cfg->samplerate; p->height = cfg->height; p->refreshrate = cfg->refreshrate; p->motionblur = cfg->motionblur;
	p->width = 0; p->pixelrate = 0; p->ptos = 0; p->syncoffset = 0;
	for (int i = 0; i < 9; i++) p->params[i] = cfg->params_int[i];
	pthread_mutex_init(&p->geo_mu, NULL); pthread_mutex_init(&p->mu, NULL);
	pthread_cond_init(&p->cv_job, NULL); pthread_cond_init(&p->cv_done, NULL);
	geometry_locked(p);
	for (int i = 0; i < 4; i++) { p->d_stage[i] = NULL; p->stage_cap[i] = 0; p->d_raw[i] = NULL; p->raw_cap[i] = 0; } p->argb_mode = 0; p->argb_inverted = 0; p->report_snr = 0; p->detect_mode = 0; p->d_argb_last = NULL; p->argb_cap = 0; p->stage_slot = 0; p->d_decim = NULL; p->decim_cap = 0; p->decim_fill = 0; p->decim_read = 0; p->decim_elem = 2;
	p->d_pix = NULL; p->pix_cap = 0; p->pix_read = 0; p->pix_fill = 0; p->d_frames[0] = p->d_frames[1] = NULL; p->frames_cap[0] = p->frames_cap[1] = 0; p->out_phase = 0;
	p->slot_cap = 0; p->d_capture[0] = p->d_capture[1] = NULL; p->cap_size[0] = p->cap_size[1] = 0; p->cap_fill = 0; p->cap_phase = 0; p->cap_rate = 0; p->plot_cap = 0; p->plot_slot = 0;
	for (int s = 0; s < PL_SLOTS; s++) { p->h_frames[s] = NULL; p->h_results[s] = NULL; p->h_report[s] = NULL; p->h_pll_rr[s] = NULL; p->slot_busy[s] = 0; }
	p->host_register = 0;                               // opt-in: tsdrgpu_pipeline_set_host_registration
	CU_TRY(ctx, cudaEventCreateWithFlags(&p->ev_res, cudaEventDisableTiming));
	for (int s = 0; s < 2; s++) { p->h_plot_frame[s] = NULL; p->h_plot_line[s] = NULL; p->plot_busy[s] = 0; p->h_peaks[s] = NULL; }
	p->stop = 0; p->submitted = 0; p->delivered = 0; p->last_w = 0; p->last_h = 0;
	memset(&p->sb, 0, sizeof p->sb); p->samplerate_real = cfg->samplerate; p->retune_cb = NULL;
	p->tn_cfg.offset = 0; p->tn_cfg.bw = 0; p->tn_cfg.D = 1; p->tn_cfg.ntaps = 0; p->tn_dirty = 0;
	p->tuner = NULL; p->tn_on = 0; p->tn_D = 1; p->tn_pos = 0;
	for (int i = 0; i < 4; i++) { p->d_tout[i] = NULL; p->tout_cap[i] = 0; }
	p->sc_cfg.K = 0; p->sc_cfg.Q = 0; p->sc_dirty = 0; p->scan = NULL; p->sc_on = 0;
	memset(&p->nt_cfg, 0, sizeof p->nt_cfg); p->nt_dirty = 0; p->notch = NULL; p->nt_on = 0;
	for (int i = 0; i < 4; i++) { p->d_nout[i] = NULL; p->nout_cap[i] = 0; }
	p->sp_nfft = 0; p->sp_dirty = 0; p->spectrum = NULL; p->sp_on = 0;
	CU_TRY(ctx, cudaEventCreateWithFlags(&p->sb.ev, cudaEventDisableTiming));
	memset(&p->stats, 0, sizeof p->stats);
	CU_TRY(ctx, cudaStreamCreateWithFlags(&p->s_main, cudaStreamNonBlocking));
	CU_TRY(ctx, cudaStreamCreateWithFlags(&p->s_copy, cudaStreamNonBlocking));
	CU_TRY(ctx, cudaStreamCreateWithFlags(&p->s_out, cudaStreamNonBlocking));
	for (int i = 0; i < 2; i++) CU_TRY(ctx, cudaEventCreateWithFlags(&p->ev_out[i], cudaEventDisableTiming));
	CU_TRY(ctx, cudaEventCreateWithFlags(&p->ev_main, cudaEventDisableTiming));
	CU_TRY(ctx, cudaStreamCreateWithFlags(&p->s_ingest, cudaStreamNonBlocking));
	for (int i = 0; i < 4; i++) {
		CU_TRY(ctx, cudaEventCreateWithFlags(&p->ev_h2d[i], cudaEventDisableTiming));
		CU_TRY(ctx, cudaEventCreateWithFlags(&p->ev_used[i], cudaEventDisableTiming));
	}
	CU_TRY(ctx, cudaEventCreateWithFlags(&p->ev_ingest, cudaEventDisableTiming));
	CU_TRY(ctx, cudaEventCreateWithFlags(&p->ev_decim, cudaEventDisableTiming));
	for (int i = 0; i < 2; i++) CU_TRY(ctx, cudaEventCreateWithFlags(&p->ev_cap_used[i], cudaEventDisableTiming));
	int rc;
	if ((rc = tsdrgpu_resampler_create(ctx, &p->rs))) return rc;
	if ((rc = tsdrgpu_framestage_create(ctx, &p->fs))) return rc;
	tsdrgpu_framestage_set_overlap(p->fs, 1);
	if ((rc = tsdrgpu_frd_create(ctx, &p->frd))) return rc;
	pthread_create(&p->thread, NULL, delivery_main, p);
	*out = p;
	return TSDRGPU_OK;
}

int tsdrgpu_pipeline_flush(tsdrgpu_pipeline_t *p) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, p != NULL);
	BIND(p->ctx);
	CU_TRY(p->ctx, cudaStreamSynchronize(p->s_copy));
	CU_TRY(p->ctx, cudaStreamSynchronize(p->s_ingest));
	CU_TRY(p->ctx, cudaStreamSynchronize(p->s_main));
	CU_TRY(p->ctx, cudaStreamSynchronize(p->s_out));
	pthread_mutex_lock(&p->mu);
	while (p->delivered < p->submitted) pthread_cond_wait(&p->cv_done, &p->mu);
	pthread_mutex_unlock(&p->mu);
	return TSDRGPU_OK;
}

void tsdrgpu_pipeline_destroy(tsdrgpu_pipeline_t *p) {
	if (!p) return;
	tsdrgpu_pipeline_flush(p);
	pthread_mutex_lock(&p->mu); p->stop = 1; pthread_cond_broadcast(&p->cv_job); pthread_mutex_unlock(&p->mu);
	pthread_join(p->thread, NULL);
	cudaSetDevice(p->ctx->device);
	tsdrgpu_resampler_destroy(p->rs); tsdrgpu_framestage_destroy(p->fs); tsdrgpu_frd_destroy(p->frd);
	for (auto &b : p->hostbufs) if (b.state == 1) { cudaHostUnregister(const_cast<void *>(b.base)); cudaGetLastError(); }
	superb_release_devices(p);
	if (p->sb.d_out) cudaFree(p->sb.d_out);
	cudaEventDestroy(p->sb.ev);
	float *dev[] = {p->d_stage[0], p->d_stage[1], p->d_stage[2], p->d_stage[3], p->d_decim, p->d_pix, p->d_frames[0], p->d_frames[1], p->d_capture[0], p->d_capture[1]};
	for (float *d : dev) if (d) cudaFree(d);
	for (int i = 0; i < 4; i++) if (p->d_raw[i]) cudaFree(p->d_raw[i]);
	for (int i = 0; i < 4; i++) if (p->d_tout[i]) cudaFree(p->d_tout[i]);
	tsdrgpu_tuner_destroy(p->tuner);
	tsdrgpu_scan_destroy(p->scan);
	for (int i = 0; i < 4; i++) if (p->d_nout[i]) cudaFree(p->d_nout[i]);
	tsdrgpu_notch_destroy(p->notch);
	tsdrgpu_spectrum_destroy(p->spectrum);
	if (p->d_argb_last) cudaFree(p->d_argb_last);
	for (int s = 0; s < PL_SLOTS; s++) if (p->h_frames[s]) { cudaFreeHost(p->h_frames[s]); cudaFreeHost(p->h_results[s]); cudaFreeHost(p->h_report[s]); free(p->h_pll_rr[s]); }
	cudaEventDestroy(p->ev_res);
	for (int s = 0; s < 2; s++) if (p->h_plot_frame[s]) { cudaFreeHost(p->h_plot_frame[s]); cudaFreeHost(p->h_plot_line[s]); cudaFreeHost(p->h_peaks[s]); }
	cudaStreamDestroy(p->s_main); cudaStreamDestroy(p->s_copy); cudaStreamDestroy(p->s_out);
	for (int i = 0; i < 2; i++) cudaEventDestroy(p->ev_out[i]);
	cudaEventDestroy(p->ev_main);
	for (int i = 0; i < 4; i++) { cudaEventDestroy(p->ev_h2d[i]); cudaEventDestroy(p->ev_used[i]); }
	cudaEventDestroy(p->ev_ingest); cudaEventDestroy(p->ev_decim); cudaEventDestroy(p->ev_cap_used[0]); cudaEventDestroy(p->ev_cap_used[1]); cudaStreamDestroy(p->s_ingest);
	pthread_mutex_destroy(&p->mu); pthread_mutex_destroy(&p->geo_mu); pthread_cond_destroy(&p->cv_job); pthread_cond_destroy(&p->cv_done);
	delete p;
}

int tsdrgpu_pipeline_set_param_int(tsdrgpu_pipeline_t *p, int id, uint32_t value) {
	if (!p || id < 0 || id >= 9) return TSDRGPU_EINVAL;
	p->params[id] = value;
	return TSDRGPU_OK;
}
int tsdrgpu_pipeline_set_resolution(tsdrgpu_pipeline_t *p, int height, double refreshrate) {
	if (!p || height <= 0 || refreshrate <= 0) return TSDRGPU_EINVAL;
	pthread_mutex_lock(&p->geo_mu);
	p->height = height; p->refreshrate = refreshrate;
	geometry_locked(p);
	pthread_mutex_unlock(&p->geo_mu);
	return TSDRGPU_OK;
}
int tsdrgpu_pipeline_set_samplerate(tsdrgpu_pipeline_t *p, uint32_t samplerate) {
	if (!p || samplerate == 0) return TSDRGPU_EINVAL;
	pthread_mutex_lock(&p->geo_mu);
	if (p->tn_cfg.bw > 0) {                              // tuned: the taps are re-designed for the new rate (next process() call)
		const int rc = tsdrgpu_tuner_design(samplerate, p->tn_cfg.offset, p->tn_cfg.bw, p->tn_cfg.D, p->tn_cfg.ntaps, NULL, 0, NULL, NULL);
		if (rc) { pthread_mutex_unlock(&p->geo_mu); snprintf(p->ctx->err, sizeof p->ctx->err, "%s", tsdrgpu_last_error(NULL)); return rc; }
		p->tn_dirty = 1;
	}
	if (p->sc_cfg.K > 0) {                               // scanning: the filter bank is re-designed for the new rate (next process() call)
		const int rc = tsdrgpu_channelizer_design(samplerate, p->sc_cfg.K, p->sc_cfg.Q, NULL, 0, NULL);
		if (rc) { pthread_mutex_unlock(&p->geo_mu); snprintf(p->ctx->err, sizeof p->ctx->err, "%s", tsdrgpu_last_error(NULL)); return rc; }
		p->sc_dirty = 1;
	}
	if (p->nt_cfg.n > 0) {                               // notched: the filter is re-designed for the new rate (next process() call)
		const int rc = tsdrgpu_notch_design(samplerate, p->nt_cfg.n, p->nt_cfg.centers, p->nt_cfg.widths, p->nt_cfg.ntaps, NULL, 0, NULL, NULL);
		if (rc) { pthread_mutex_unlock(&p->geo_mu); snprintf(p->ctx->err, sizeof p->ctx->err, "%s", tsdrgpu_last_error(NULL)); return rc; }
		p->nt_dirty = 1;
	}
	if (p->sp_nfft > 0) p->sp_dirty = 1;                 // the spectrum starts over at the new rate
	p->samplerate = p->tn_cfg.bw > 0 ? samplerate / (uint32_t) p->tn_cfg.D : samplerate; p->samplerate_real = samplerate;
	geometry_locked(p);
	pthread_mutex_unlock(&p->geo_mu);
	return TSDRGPU_OK;
}
int tsdrgpu_pipeline_set_tuner(tsdrgpu_pipeline_t *p, double offset_hz, double bandwidth_hz, int decimation, int ntaps) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, p != NULL);
	pthread_mutex_lock(&p->geo_mu);
	if (bandwidth_hz > 0) {
		const int rc = tsdrgpu_tuner_design(p->samplerate_real, offset_hz, bandwidth_hz, decimation, ntaps, NULL, 0, NULL, NULL);
		if (rc) { pthread_mutex_unlock(&p->geo_mu); snprintf(p->ctx->err, sizeof p->ctx->err, "%s", tsdrgpu_last_error(NULL)); return rc; }
	}
	p->tn_cfg.offset = offset_hz; p->tn_cfg.bw = bandwidth_hz > 0 ? bandwidth_hz : 0; p->tn_cfg.D = bandwidth_hz > 0 ? decimation : 1; p->tn_cfg.ntaps = ntaps;
	p->tn_dirty = 1;
	pthread_mutex_unlock(&p->geo_mu);
	return TSDRGPU_OK;
}
int tsdrgpu_pipeline_set_scan(tsdrgpu_pipeline_t *p, int channels, int taps_per_channel) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, p != NULL);
	pthread_mutex_lock(&p->geo_mu);
	if (channels != 0) {
		const int rc = tsdrgpu_channelizer_design(p->samplerate_real, channels, taps_per_channel, NULL, 0, NULL);
		if (rc) { pthread_mutex_unlock(&p->geo_mu); snprintf(p->ctx->err, sizeof p->ctx->err, "%s", tsdrgpu_last_error(NULL)); return rc; }
	}
	p->sc_cfg.K = channels; p->sc_cfg.Q = taps_per_channel;
	p->sc_dirty = 1;
	pthread_mutex_unlock(&p->geo_mu);
	return TSDRGPU_OK;
}
int tsdrgpu_pipeline_scan_results(tsdrgpu_pipeline_t *p, tsdrgpu_scan_channel_t *out, int cap, int *n) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, p != NULL);
	if (n) *n = 0;
	if (!p->sc_on) return TSDRGPU_OK;
	const int rc = tsdrgpu_scan_results(p->scan, p->s_ingest, out, cap);
	if (rc) return rc;
	if (n) *n = cap < p->sc_cfg.K ? cap : p->sc_cfg.K;
	return TSDRGPU_OK;
}
int tsdrgpu_pipeline_set_notches(tsdrgpu_pipeline_t *p, int n, const double *centers, const double *widths, int ntaps) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, p != NULL);
	pthread_mutex_lock(&p->geo_mu);
	if (n != 0) {
		const int rc = tsdrgpu_notch_design(p->samplerate_real, n, centers, widths, ntaps, NULL, 0, NULL, NULL);
		if (rc) { pthread_mutex_unlock(&p->geo_mu); snprintf(p->ctx->err, sizeof p->ctx->err, "%s", tsdrgpu_last_error(NULL)); return rc; }
		for (int j = 0; j < n; j++) { p->nt_cfg.centers[j] = centers[j]; p->nt_cfg.widths[j] = widths[j]; }
	}
	p->nt_cfg.n = n; p->nt_cfg.ntaps = ntaps;
	p->nt_dirty = 1;
	pthread_mutex_unlock(&p->geo_mu);
	return TSDRGPU_OK;
}
int tsdrgpu_pipeline_set_spectrum(tsdrgpu_pipeline_t *p, int nfft) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, p != NULL);
	pthread_mutex_lock(&p->geo_mu);
	if (nfft != 0) {
		const int rc = tsdrgpu_spectrum_check(p->samplerate_real, nfft);
		if (rc) { pthread_mutex_unlock(&p->geo_mu); snprintf(p->ctx->err, sizeof p->ctx->err, "%s", tsdrgpu_last_error(NULL)); return rc; }
	}
	p->sp_nfft = nfft; p->sp_dirty = 1;
	pthread_mutex_unlock(&p->geo_mu);
	return TSDRGPU_OK;
}
int tsdrgpu_pipeline_spectrum(tsdrgpu_pipeline_t *p, double *out, int cap, int *n, uint64_t *segments) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, p != NULL);
	if (n) *n = 0;
	if (segments) *segments = 0;
	if (!p->sp_on) return TSDRGPU_OK;
	const int rc = tsdrgpu_spectrum_results(p->spectrum, p->s_ingest, out, cap, segments);
	if (rc) return rc;
	if (n) *n = cap < p->sp_nfft ? cap : p->sp_nfft;
	return TSDRGPU_OK;
}
// superbandwidth with one hop per GPU: devices[0] must be the pipeline's own device; n in {2, 4, 8} = number of hops.  n <= 1
// returns to the one-GPU mode (4 hops).  Call while no superbandwidth round is in flight (before PARAM_AUTOCORR_SUPERRESOLUTION
// is switched on).  The same device may be listed more than once (test set-ups on a single GPU).
int tsdrgpu_pipeline_set_superb_devices(tsdrgpu_pipeline_t *p, const int *devices, int n) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, p != NULL);
	tsdrgpu_ctx_t *ctx = p->ctx;
	BIND(ctx);
	CU_TRY(ctx, cudaStreamSynchronize(p->s_main));
	superb_release_devices(p);
	p->sb.state = SB_STOPPED;
	if (n <= 1) return TSDRGPU_OK;
	ARG_TRY(ctx, devices != NULL && (n == 2 || n == 4 || n == 8) && devices[0] == ctx->device);
	p->sb.rctx[0] = ctx; p->sb.dev[0] = ctx->device; p->sb.rstream[0] = p->s_main; p->sb.rcopy[0] = p->s_copy;
	for (int i = 1; i < n; i++) {
		int rc = tsdrgpu_create(&p->sb.rctx[i], devices[i]);
		if (rc) { snprintf(ctx->err, sizeof ctx->err, "%s", tsdrgpu_last_error(NULL)); p->sb.ndev = i; superb_release_devices(p); return rc; }
		p->sb.dev[i] = devices[i];
		cudaSetDevice(devices[i]);
		cudaStreamCreateWithFlags(&p->sb.rstream[i], cudaStreamNonBlocking);
		cudaStreamCreateWithFlags(&p->sb.rcopy[i], cudaStreamNonBlocking);
		cudaEventCreateWithFlags(&p->sb.rev[i], cudaEventDisableTiming);
	}
	p->sb.ndev = n;
	CU_TRY(ctx, cudaSetDevice(ctx->device));
	return TSDRGPU_OK;
}
int tsdrgpu_pipeline_set_host_registration(tsdrgpu_pipeline_t *p, int on) { if (!p) return TSDRGPU_EINVAL; p->host_register = on != 0; return TSDRGPU_OK; }
int tsdrgpu_pipeline_set_retune(tsdrgpu_pipeline_t *p, tsdrgpu_retune_cb cb) { if (!p) return TSDRGPU_EINVAL; p->retune_cb = cb; return TSDRGPU_OK; }
int tsdrgpu_pipeline_set_motionblur(tsdrgpu_pipeline_t *p, float coeff) { if (!p) return TSDRGPU_EINVAL; p->motionblur = coeff; return TSDRGPU_OK; }
int tsdrgpu_pipeline_set_output_argb(tsdrgpu_pipeline_t *p, int mode, int inverted) { if (!p) return TSDRGPU_EINVAL; p->argb_mode = mode != 0; p->argb_inverted = inverted != 0; return TSDRGPU_OK; }
int tsdrgpu_pipeline_set_reports(tsdrgpu_pipeline_t *p, int report_snr, int detect_mode) { if (!p) return TSDRGPU_EINVAL; p->report_snr = report_snr != 0; p->detect_mode = detect_mode != 0; return TSDRGPU_OK; }
int tsdrgpu_pipeline_sync(tsdrgpu_pipeline_t *p, int pixels) { if (!p) return TSDRGPU_EINVAL; p->syncoffset += pixels; return TSDRGPU_OK; }
int tsdrgpu_pipeline_get_geometry(tsdrgpu_pipeline_t *p, int *width, int *height, double *refreshrate) {
	if (!p) return TSDRGPU_EINVAL;
	pthread_mutex_lock(&p->geo_mu);
	if (width) *width = p->width; if (height) *height = p->height; if (refreshrate) *refreshrate = p->refreshrate;
	pthread_mutex_unlock(&p->geo_mu);
	return TSDRGPU_OK;
}
int tsdrgpu_pipeline_stats(tsdrgpu_pipeline_t *p, tsdrgpu_pipeline_stats_t *out) {
	if (!p || !out) return TSDRGPU_EINVAL;
	pthread_mutex_lock(&p->mu); *out = p->stats; pthread_mutex_unlock(&p->mu);
	out->gpu_launches = p->ctx->launches;
	return TSDRGPU_OK;
}

// ---- superbandwidth mode: superb_run (superbandwidth.c:179-254) + superb_ondataready (:121-152) -------------------
// Four hops of 10 frames each are recorded at centre frequencies fc + (hop-2)*fs (0.5 s settling pause after every
// retune), aligned, and stitched into one 4x-rate signal that then flows through the normal decimator / frame stages.
// The reference does the stitch on a helper thread (~3 s of CPU FFTs); here it runs on the GPU inside the call that
// completes the last hop (a few ms), so its output appears one process() call earlier.  Everything else is the same.
static void superb_stop(tsdrgpu_pipeline *p) {                  // superbandwidth.c:256-264
	if (p->sb.state == SB_STOPPED) return;
	p->sb.state = SB_STOPPED;
	if (p->retune_cb) p->retune_cb(0, p->user);
	pthread_mutex_lock(&p->geo_mu);
	p->samplerate = p->samplerate_real / (uint32_t) p->tn_D;
	geometry_locked(p);
	pthread_mutex_unlock(&p->geo_mu);
	if (p->tn_on) { p->tn_pos = 0; tsdrgpu_tuner_reset(p->tuner, p->s_ingest); }     // the tuner resumes from a clean start
	if (p->sc_on) tsdrgpu_scan_reset(p->scan, p->s_ingest);                          // and so does the scan
	if (p->nt_on) tsdrgpu_notch_reset(p->notch, p->s_ingest);                        // and the notch
	if (p->sp_on) tsdrgpu_spectrum_reset(p->spectrum, p->s_ingest);                  // and the spectrum
}

// a spectrum (re)configuration, at the start of a process() call: the spectrum starts over; the pixel path does not notice
static int spectrum_apply(tsdrgpu_pipeline *p) {
	tsdrgpu_ctx_t *ctx = p->ctx;
	int rc;
	pthread_mutex_lock(&p->geo_mu);
	const int dirty = p->sp_dirty, nfft = p->sp_nfft;
	const uint32_t fs = p->samplerate_real;
	p->sp_dirty = 0;
	pthread_mutex_unlock(&p->geo_mu);
	if (!dirty) return TSDRGPU_OK;
	CU_TRY(ctx, cudaStreamSynchronize(p->s_ingest));
	if (nfft > 0) {
		if (!p->spectrum && (rc = tsdrgpu_spectrum_create(ctx, &p->spectrum))) return rc;
		if ((rc = tsdrgpu_spectrum_configure(p->spectrum, fs, nfft))) return rc;      // resets
		p->sp_on = 1;
	} else p->sp_on = 0;
	return TSDRGPU_OK;
}

// a notch (re)configuration, at the start of a process() call: the stream starts over behind the notch as a new pipeline would
static int notch_apply(tsdrgpu_pipeline *p) {
	tsdrgpu_ctx_t *ctx = p->ctx;
	int rc;
	pthread_mutex_lock(&p->geo_mu);
	const int dirty = p->nt_dirty, n = p->nt_cfg.n, ntaps = p->nt_cfg.ntaps;
	double centers[32], widths[32];
	for (int j = 0; j < n; j++) { centers[j] = p->nt_cfg.centers[j]; widths[j] = p->nt_cfg.widths[j]; }
	const uint32_t fs = p->samplerate_real;
	p->nt_dirty = 0;
	pthread_mutex_unlock(&p->geo_mu);
	if (!dirty) return TSDRGPU_OK;
	if ((rc = tsdrgpu_framestage_join(p->fs, p->s_main))) return rc;
	CU_TRY(ctx, cudaStreamSynchronize(p->s_copy)); CU_TRY(ctx, cudaStreamSynchronize(p->s_ingest));
	CU_TRY(ctx, cudaStreamSynchronize(p->s_main)); CU_TRY(ctx, cudaStreamSynchronize(p->s_out));
	if (n > 0) {
		if (!p->notch && (rc = tsdrgpu_notch_create(ctx, &p->notch))) return rc;
		if ((rc = tsdrgpu_notch_configure(p->notch, fs, n, centers, widths, ntaps))) return rc;      // resets
		p->nt_on = 1;
	} else p->nt_on = 0;
	if (p->tn_on) { p->tn_pos = 0; if ((rc = tsdrgpu_tuner_reset(p->tuner, p->s_ingest))) return rc; }
	if (p->sc_on && (rc = tsdrgpu_scan_reset(p->scan, p->s_ingest))) return rc;
	p->decim_fill = 0; p->decim_read = 0; p->decim_elem = 2; p->pix_fill = 0; p->pix_read = 0; p->cap_fill = 0;
	p->dev_drop = DropComp(); p->pix_drop = DropComp();
	if ((rc = tsdrgpu_resampler_reset(p->rs, p->s_main))) return rc;
	if ((rc = tsdrgpu_framestage_reset(p->fs, p->s_main))) return rc;
	if ((rc = tsdrgpu_frd_reset(p->frd))) return rc;
	CU_TRY(ctx, cudaStreamSynchronize(p->s_main));
	CU_TRY(ctx, cudaStreamSynchronize(p->s_ingest));
	return TSDRGPU_OK;
}

// a scan (re)configuration, at the start of a process() call: the scan starts over; the pixel path does not notice
static int scan_apply(tsdrgpu_pipeline *p) {
	tsdrgpu_ctx_t *ctx = p->ctx;
	int rc;
	pthread_mutex_lock(&p->geo_mu);
	const int dirty = p->sc_dirty, K = p->sc_cfg.K, Q = p->sc_cfg.Q;
	const uint32_t fs = p->samplerate_real;
	p->sc_dirty = 0;
	pthread_mutex_unlock(&p->geo_mu);
	if (!dirty) return TSDRGPU_OK;
	CU_TRY(ctx, cudaStreamSynchronize(p->s_ingest));
	if (K > 0) {
		if (!p->scan && (rc = tsdrgpu_scan_create(ctx, &p->scan))) return rc;
		if ((rc = tsdrgpu_scan_configure(p->scan, fs, K, Q))) return rc;      // resets
		p->sc_on = 1;
	} else p->sc_on = 0;
	return TSDRGPU_OK;
}

// a tuner (re)configuration, at the start of a process() call: the stream starts over at the new internal rate
static int tuner_apply(tsdrgpu_pipeline *p) {
	tsdrgpu_ctx_t *ctx = p->ctx;
	int rc;
	pthread_mutex_lock(&p->geo_mu);
	const int dirty = p->tn_dirty; const double offset = p->tn_cfg.offset, bw = p->tn_cfg.bw; const int D = p->tn_cfg.D, ntaps = p->tn_cfg.ntaps;
	const uint32_t fs = p->samplerate_real;
	p->tn_dirty = 0;
	pthread_mutex_unlock(&p->geo_mu);
	if (!dirty) return TSDRGPU_OK;
	if ((rc = tsdrgpu_framestage_join(p->fs, p->s_main))) return rc;
	CU_TRY(ctx, cudaStreamSynchronize(p->s_copy)); CU_TRY(ctx, cudaStreamSynchronize(p->s_ingest));
	CU_TRY(ctx, cudaStreamSynchronize(p->s_main)); CU_TRY(ctx, cudaStreamSynchronize(p->s_out));
	if (bw > 0) {
		if (!p->tuner && (rc = tsdrgpu_tuner_create(ctx, &p->tuner))) return rc;
		if ((rc = tsdrgpu_tuner_configure(p->tuner, fs, offset, bw, D, ntaps))) return rc;
		p->tn_on = 1; p->tn_D = D;
	} else { p->tn_on = 0; p->tn_D = 1; }
	p->tn_pos = 0;
	// what waits at the old rate is meaningless at the new one: start over behind the tuner as a new pipeline would
	p->decim_fill = 0; p->decim_read = 0; p->decim_elem = 2; p->pix_fill = 0; p->pix_read = 0; p->cap_fill = 0;
	p->dev_drop = DropComp(); p->pix_drop = DropComp();
	if ((rc = tsdrgpu_resampler_reset(p->rs, p->s_main))) return rc;
	if ((rc = tsdrgpu_framestage_reset(p->fs, p->s_main))) return rc;
	if ((rc = tsdrgpu_frd_reset(p->frd))) return rc;
	CU_TRY(ctx, cudaStreamSynchronize(p->s_main));
	pthread_mutex_lock(&p->geo_mu);
	if (p->sb.state == SB_STOPPED) { p->samplerate = p->samplerate_real / (uint32_t) p->tn_D; geometry_locked(p); }
	pthread_mutex_unlock(&p->geo_mu);
	return TSDRGPU_OK;
}
// make room for `bytes` of raw samples in slot ss (contents are not preserved)
static int raw_reserve(tsdrgpu_pipeline *p, int ss, size_t bytes) {
	tsdrgpu_ctx_t *ctx = p->ctx;
	if (p->raw_cap[ss] >= bytes) return TSDRGPU_OK;
	CU_TRY(ctx, cudaStreamSynchronize(p->s_ingest)); CU_TRY(ctx, cudaStreamSynchronize(p->s_copy));
	if (p->d_raw[ss]) CU_TRY(ctx, cudaFree(p->d_raw[ss]));
	const size_t cap = bytes + bytes / 2;
	CU_TRY(ctx, cudaMalloc(&p->d_raw[ss], cap));
	p->raw_cap[ss] = cap;
	return TSDRGPU_OK;
}

// the devices of the sharded mode own contexts, streams and (once the hop size is known) the superbandwidth group
static void superb_release_devices(tsdrgpu_pipeline *p) {
	for (int i = 0; i < p->sb.ndev; i++) {
		if (p->sb.grp[i]) { tsdrgpu_superb_mgpu_destroy(p->sb.grp[i]); p->sb.grp[i] = NULL; }
	}
	for (int i = 0; i < 16; i++) {
		if (p->sb.d_hops[i]) { cudaSetDevice(i < p->sb.ndev ? p->sb.dev[i] : p->ctx->device); cudaFree(p->sb.d_hops[i]); p->sb.d_hops[i] = NULL; }
		if (p->sb.rraw[i]) { cudaSetDevice(p->sb.dev[i]); cudaFree(p->sb.rraw[i]); p->sb.rraw[i] = NULL; p->sb.rraw_cap[i] = 0; }
		if (p->sb.d_hop0[i]) { cudaSetDevice(p->sb.dev[i]); cudaFree(p->sb.d_hop0[i]); p->sb.d_hop0[i] = NULL; }
	}
	for (int i = 1; i < p->sb.ndev; i++) {
		cudaSetDevice(p->sb.dev[i]);
		if (p->sb.rstream[i]) cudaStreamDestroy(p->sb.rstream[i]);
		if (p->sb.rcopy[i]) cudaStreamDestroy(p->sb.rcopy[i]);
		if (p->sb.rev[i]) cudaEventDestroy(p->sb.rev[i]);
		if (p->sb.rctx[i]) tsdrgpu_destroy(p->sb.rctx[i]);
		p->sb.rstream[i] = NULL; p->sb.rcopy[i] = NULL; p->sb.rev[i] = NULL; p->sb.rctx[i] = NULL;
	}
	p->sb.ndev = 0; p->sb.rate = 0;
	cudaSetDevice(p->ctx->device);
}

static int superb_step(tsdrgpu_pipeline *p, const void *h_iq, int fmt, uint64_t items_count, int64_t dropped) {
	tsdrgpu_ctx_t *ctx = p->ctx;
	int rc;
	const int H = p->sb.ndev > 1 ? p->sb.ndev : 4;                    // SUPER_HOPS_TO_MAKE
	const bool sharded = p->sb.ndev > 1;
	if (p->sb.state == SB_STOPPED) p->sb.state = SB_STARTING;
	if (p->sb.state == SB_STARTING) {
		p->sb.buffid = 0; p->sb.gathered = 0;
		if (p->samplerate_real != p->sb.rate || p->sb.nhops != H) {
			p->sb.rate = p->samplerate_real; p->sb.nhops = H;
			pthread_mutex_lock(&p->geo_mu); const double fv = p->refreshrate; pthread_mutex_unlock(&p->geo_mu);
			p->sb.in_frame = (long long) (p->samplerate_real / fv);
			p->sb.to_gather = 10 * p->sb.in_frame;                    // SUPER_SAMPLES_TO_RECORD
			p->sb.to_pause = (long long) (0.5 * p->samplerate_real);   // SUPER_SECS_TO_PAUSE
			CU_TRY(ctx, cudaStreamSynchronize(p->s_main));
			for (int i = 0; i < 16; i++) if (p->sb.d_hops[i]) { CU_TRY(ctx, cudaSetDevice(sharded && i < H ? p->sb.dev[i] : ctx->device)); CU_TRY(ctx, cudaFree(p->sb.d_hops[i])); p->sb.d_hops[i] = NULL; }
			for (int i = 0; i < H; i++) {
				CU_TRY(ctx, cudaSetDevice(sharded ? p->sb.dev[i] : ctx->device));
				CU_TRY(ctx, cudaMalloc(&p->sb.d_hops[i], sizeof(float) * 2 * (size_t) p->sb.to_gather));
				if (p->sb.d_hop0[i]) { CU_TRY(ctx, cudaFree(p->sb.d_hop0[i])); p->sb.d_hop0[i] = NULL; }
				if (sharded && i > 0) CU_TRY(ctx, cudaMalloc(&p->sb.d_hop0[i], sizeof(float) * 2 * (size_t) p->sb.to_gather));
			}
			CU_TRY(ctx, cudaSetDevice(ctx->device));
			if (sharded) {                                            // (re)build the group for this hop size
				for (int i = 0; i < H; i++) if (p->sb.grp[i]) { tsdrgpu_superb_mgpu_destroy(p->sb.grp[i]); p->sb.grp[i] = NULL; }
				for (int i = 0; i < H; i++)
					if ((rc = tsdrgpu_superb_mgpu_create(p->sb.rctx[i], H, i, 0, (uint32_t) p->sb.to_gather, &p->sb.grp[i]))) { snprintf(ctx->err, sizeof ctx->err, "%s", tsdrgpu_last_error(p->sb.rctx[i])); return rc; }
				if ((rc = tsdrgpu_superb_mgpu_connect_local(p->sb.grp, H))) { snprintf(ctx->err, sizeof ctx->err, "%s", tsdrgpu_last_error(p->sb.rctx[0])); return rc; }
				CU_TRY(ctx, cudaSetDevice(ctx->device));
			}
		}
		p->sb.state = SB_GATHERING;
	}
	if (p->sb.state == SB_PAUSE) {
		p->sb.gathered += (long long) (items_count / 2);
		if (p->sb.gathered > p->sb.to_pause) { p->sb.gathered = 0; p->sb.state = SB_GATHERING; }
	}
	if (p->sb.state != SB_GATHERING) return TSDRGPU_OK;
	if (dropped) { p->sb.gathered = 0; return TSDRGPU_OK; }
	const long long now = (long long) (items_count / 2);
	const long long take = (p->sb.gathered + now < p->sb.to_gather) ? now : (p->sb.to_gather - p->sb.gathered);
	if (take > 0) {
		const int b = p->sb.buffid;
		float *hop = p->sb.d_hops[b] + 2 * p->sb.gathered;
		const size_t bytes = fmt_bytes(fmt) * 2 * (size_t) take;
		// hop b lives on the device that will transform it: the block goes there straight from the host
		cudaStream_t cs = (sharded && b > 0) ? p->sb.rcopy[b] : p->s_copy;
		if (sharded && b > 0) CU_TRY(ctx, cudaSetDevice(p->sb.dev[b]));
		cudaError_t e = cudaStreamWaitEvent(cs, (sharded && b > 0) ? p->sb.rev[b] : p->sb.ev, 0);     // the last stitch has finished reading the hop buffer
		if (e == cudaSuccess) {
			if (fmt == TSDRGPU_FMT_FLOAT) e = cudaMemcpyAsync(hop, h_iq, bytes, cudaMemcpyHostToDevice, cs);
			else {
				void **raw = (sharded && b > 0) ? &p->sb.rraw[b] : &p->d_raw[0];
				size_t *cap = (sharded && b > 0) ? &p->sb.rraw_cap[b] : &p->raw_cap[0];
				if (*cap < bytes) { cudaStreamSynchronize(cs); if (*raw) cudaFree(*raw); *raw = NULL; e = cudaMalloc(raw, bytes + bytes / 2); *cap = (e == cudaSuccess) ? bytes + bytes / 2 : 0; }
				if (e == cudaSuccess) e = cudaMemcpyAsync(*raw, h_iq, bytes, cudaMemcpyHostToDevice, cs);
				if (e == cudaSuccess) { pl_convert<<<1024, 256, 0, cs>>>(*raw, hop, 2 * (size_t) take, fmt); ctx->launches++; e = cudaGetLastError(); }
			}
		}
		const cudaError_t e2 = cudaStreamSynchronize(cs);            // the plugin's buffer has been read, whatever happened
		cudaSetDevice(ctx->device);
		if (e != cudaSuccess || e2 != cudaSuccess) return tsdrgpu_fail(ctx, TSDRGPU_ECUDA, "H2D of a superbandwidth hop block", e != cudaSuccess ? e : e2, __FILE__, __LINE__);
		p->stats.h2d_bytes += bytes;
	}
	p->sb.gathered += take;
	if (p->sb.gathered < p->sb.to_gather) return TSDRGPU_OK;
	const long long count_pairs = p->sb.gathered;
	p->sb.buffid++; p->sb.gathered = 0;
	if (sharded && p->sb.buffid == 1) {
		// hop 0 is complete: every other device gets its copy now (NVLink peer copy, seconds before the stitch needs it), so that
		// each rank derives its alignment lag from local data (superb_mgpu.cu phase 2)
		for (int i = 1; i < H; i++) {
			cudaSetDevice(p->sb.dev[i]);
			cudaError_t e = cudaStreamWaitEvent(p->sb.rcopy[i], p->sb.rev[i], 0);
			if (e == cudaSuccess) e = cudaMemcpyPeerAsync(p->sb.d_hop0[i], p->sb.dev[i], p->sb.d_hops[0], p->sb.dev[0], sizeof(float) * 2 * (size_t) count_pairs, p->sb.rcopy[i]);
			if (e == cudaSuccess) e = cudaStreamSynchronize(p->sb.rcopy[i]);
			if (e != cudaSuccess) { cudaSetDevice(ctx->device); return tsdrgpu_fail(ctx, TSDRGPU_ECUDA, "peer copy of the alignment reference (hop 0)", e, __FILE__, __LINE__); }
		}
		cudaSetDevice(ctx->device);
	}
	if (p->sb.buffid < H) {
		if (p->retune_cb) p->retune_cb((int32_t) ((p->sb.buffid - H / 2) * (long long) p->sb.rate), p->user);    // shiftfreq, superbandwidth.c:241
		p->sb.state = SB_PAUSE;
		return TSDRGPU_OK;
	}
	// all hops recorded: align + stitch (superb_ondataready) and hand the H-times-rate signal to the decimator
	const unsigned long long N = tsdrgpu_fft_getrealsize((uint32_t) count_pairs);
	size_t total_samples = 0;
	CU_TRY(ctx, cudaStreamSynchronize(p->s_ingest));
	if (!sharded) {
		if (p->sb.out_cap < 2 * (size_t) H * N) { CU_TRY(ctx, cudaStreamSynchronize(p->s_main)); if (p->sb.d_out) CU_TRY(ctx, cudaFree(p->sb.d_out)); CU_TRY(ctx, cudaMalloc(&p->sb.d_out, sizeof(float) * 2 * (size_t) H * N)); p->sb.out_cap = 2 * (size_t) H * N; }
		int offs[16], total = 0;
		if ((rc = tsdrgpu_superb_stitch(ctx, p->s_main, p->sb.d_hops, H, (int) count_pairs, (int) p->sb.in_frame, p->sb.d_out, offs, &total))) return rc;
		CU_TRY(ctx, cudaEventRecord(p->sb.ev, p->s_main));
		float *where;
		if ((rc = decim_set_elem(p, 2))) return rc;
		if ((rc = decim_reserve(p, (size_t) total, &where))) return rc;
		pl_copy_f32<<<2048, 256, 0, p->s_main>>>(p->sb.d_out, where, 2ull * (size_t) total);
		LAUNCH_CHECK(ctx);
		total_samples = (size_t) total;
	} else {
		// one hop per GPU: every rank runs its share on its own device; rank 0 (this pipeline's device, the main stream) receives
		// the time-contiguous MAGNITUDE stream straight into the decimator input (superb_mgpu.cu)
		float *where;
		if ((rc = decim_set_elem(p, 1))) return rc;
		if ((rc = decim_reserve(p, (size_t) H * N, &where))) return rc;
		for (int r = 0; r < H; r++) {
			uint32_t n = 0;
			rc = tsdrgpu_superb_mgpu_stitch(p->sb.grp[r], r == 0 ? p->s_main : p->sb.rstream[r], p->sb.d_hops[r], r == 0 ? p->sb.d_hops[0] : p->sb.d_hop0[r], (int) count_pairs, (int) p->sb.in_frame, r == 0 ? where : NULL, &n);
			if (rc) { snprintf(ctx->err, sizeof ctx->err, "%s", tsdrgpu_last_error(p->sb.rctx[r])); cudaSetDevice(ctx->device); return rc; }
			if (r > 0) { cudaSetDevice(p->sb.dev[r]); cudaEventRecord(p->sb.rev[r], p->sb.rstream[r]); }
		}
		CU_TRY(ctx, cudaSetDevice(ctx->device));
		CU_TRY(ctx, cudaEventRecord(p->sb.ev, p->s_main));
		ctx->launches += 0;
		total_samples = (size_t) H * N;
	}
	p->stats.stitches++;
	pthread_mutex_lock(&p->geo_mu);
	p->samplerate = (uint32_t) H * p->sb.rate;                        // set_internal_samplerate(tsdr, buffscount*samplerate)
	geometry_locked(p);
	pthread_mutex_unlock(&p->geo_mu);
	p->decim_fill += total_samples;
	p->sb.state = SB_STARTING;
	return drain_blocks(p);
}

// the body of the reference's process() (TSDRLibrary.c:264-298)
int tsdrgpu_convert_samples(tsdrgpu_ctx_t *ctx, void *stream, const void *d_raw, int fmt, uint64_t items_count, float *d_out) {
	BIND(ctx);
	ARG_TRY(ctx, fmt >= TSDRGPU_FMT_FLOAT && fmt <= TSDRGPU_FMT_UINT16);
	if (items_count == 0) return TSDRGPU_OK;
	ARG_TRY(ctx, d_raw != NULL && d_out != NULL);
	if (fmt == TSDRGPU_FMT_FLOAT) { CU_TRY(ctx, cudaMemcpyAsync(d_out, d_raw, sizeof(float) * items_count, cudaMemcpyDeviceToDevice, (cudaStream_t) stream)); return TSDRGPU_OK; }
	const size_t want = (items_count / 4 + 255) / 256;
	KL(ctx, "pl_convert", (cudaStream_t) stream, pl_convert<<<(unsigned) (want < 2048 ? (want ? want : 1) : 2048), 256, 0, (cudaStream_t) stream>>>(d_raw, d_out, items_count, fmt));
	return TSDRGPU_OK;
}

static int process_impl(tsdrgpu_pipeline_t *p, const void *h_iq, int fmt, uint64_t items_count, int64_t samples_dropped, bool wait_for_copy);

int tsdrgpu_pipeline_process(tsdrgpu_pipeline_t *p, const float *h_iq, uint64_t items_count, int64_t samples_dropped) {
	return process_impl(p, h_iq, TSDRGPU_FMT_FLOAT, items_count, samples_dropped, true);
}
int tsdrgpu_pipeline_process_raw(tsdrgpu_pipeline_t *p, const void *h_iq, int fmt, uint64_t items_count, int64_t samples_dropped) {
	return process_impl(p, h_iq, fmt, items_count, samples_dropped, true);
}
// For a front end that owns a ring of PAGE-LOCKED buffers: the call returns as soon as everything is enqueued, the buffer must
// stay untouched until tsdrgpu_pipeline_sync_input() has returned (or the buffer three calls later has been accepted: there are
// four staging slots).  Copies of consecutive blocks then run back to back on the link instead of waiting for the host's
// enqueue work in between.  Not for pageable memory (a pageable cudaMemcpyAsync is synchronous anyway).
int tsdrgpu_pipeline_process_raw_async(tsdrgpu_pipeline_t *p, const void *h_pinned, int fmt, uint64_t items_count, int64_t samples_dropped) {
	return process_impl(p, h_pinned, fmt, items_count, samples_dropped, false);
}
int tsdrgpu_pipeline_sync_input(tsdrgpu_pipeline_t *p) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, p != NULL);
	BIND(p->ctx);
	CU_TRY(p->ctx, cudaStreamSynchronize(p->s_copy));
	return TSDRGPU_OK;
}

static int process_impl(tsdrgpu_pipeline_t *p, const void *h_iq, int fmt, uint64_t items_count, int64_t samples_dropped, bool wait_for_copy) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, p != NULL);
	tsdrgpu_ctx_t *ctx = p->ctx;
	BIND(ctx);
	ARG_TRY(ctx, fmt >= TSDRGPU_FMT_FLOAT && fmt <= TSDRGPU_FMT_UINT16);
	ARG_TRY(ctx, (items_count & 1) == 0);                     // assert at TSDRLibrary.c:265
	const uint64_t size2 = items_count >> 1;
	int rc = tuner_apply(p);
	if (rc) return rc;
	if ((rc = scan_apply(p))) return rc;
	if ((rc = notch_apply(p))) return rc;
	if ((rc = spectrum_apply(p))) return rc;
	pthread_mutex_lock(&p->geo_mu);
	const int w = p->width, h = p->height; const double ptos = p->ptos;
	pthread_mutex_unlock(&p->geo_mu);
	p->stats.samples_in += size2;
	if (samples_dropped > 0) p->stats.samples_dropped_upstream += (uint64_t) samples_dropped;
	if (p->params[TSDRGPU_PARAM_AUTOCORR_SUPERRESOLUTION]) return superb_step(p, h_iq, fmt, items_count, samples_dropped);
	superb_stop(p);
	const int block = (int) round((double) ((w * h) << 1) * ptos);           // TSDRLibrary.c:284
	if (block <= 0) return TSDRGPU_OK;
	// what the stages behind the tuner see: its output pairs and output drop count (the block itself when there is no tuner)
	const bool tuned = p->tn_on != 0;
	const uint64_t gap = samples_dropped > 0 ? (uint64_t) samples_dropped : 0;
	uint64_t n2 = size2; int64_t dropped = samples_dropped;
	if (tuned) {
		uint64_t o = 0, od = 0;
		tsdrgpu_tuner_out_pairs(p->tn_pos, size2, gap, p->tn_D, &o, &od);
		n2 = o; dropped = (int64_t) od;
	}
	p->dev_drop.shift_with((uint32_t) block, dropped);
	const bool drop_all = p->dev_drop.will_drop_all((uint32_t) n2);
	const bool plots_on = !p->params[TSDRGPU_PARAM_AUTOCORR_PLOTS_OFF];
	const bool need_data = n2 > 0 && (!drop_all || (plots_on && dropped != 0));
	// the tuner and the scan see every non-empty block, also one the drop compensation discards whole: their history and position
	// stay continuous
	const bool scanning = p->sc_on != 0, notched = p->nt_on != 0, spectrum = p->sp_on != 0;
	const bool need_copy = (tuned || scanning || notched || spectrum) ? size2 > 0 : need_data;
	const int ss = p->stage_slot;
	float *stage = NULL, *d_in = NULL;
	bool copy_issued = false;
	// Every path out of this block -- success or failure -- passes the synchronisation of the copy stream below: the header's
	// contract is that the caller's buffer is read during the call only.
	do {
		if (need_copy) {
			if (h_iq == NULL) { rc = tsdrgpu_fail(ctx, TSDRGPU_EINVAL, "invalid argument: h_iq != NULL", cudaSuccess, __FILE__, __LINE__); break; }
			p->stage_slot = (p->stage_slot + 1) & 3;
			if (p->stage_cap[ss] < items_count) { cudaStreamSynchronize(p->s_ingest); cudaStreamSynchronize(p->s_copy); }
			if ((rc = grow(ctx, p->s_main, &p->d_stage[ss], &p->stage_cap[ss], items_count, 0))) break;
			stage = p->d_stage[ss];
			// The plugin's buffer is only valid during this call: copy it on the copy stream into one of four staging slots
			// (after the ingest kernels that read the slot four calls ago) and return once the host buffer has been read.
			// The light per-block kernels (capture demod, append to the decimator input) run on their own stream, so the
			// copy of block k+1..k+3 never waits behind the heavy resample / frame / FFT kernels of earlier blocks.
			const size_t bytes = fmt_bytes(fmt) * items_count;
			if (fmt != TSDRGPU_FMT_FLOAT && (rc = raw_reserve(p, ss, bytes))) break;
			const void *src = host_source(p, h_iq, bytes);
			cudaError_t e = cudaStreamWaitEvent(p->s_copy, p->ev_used[ss], 0);
			if (e == cudaSuccess) { e = cudaMemcpyAsync(fmt == TSDRGPU_FMT_FLOAT ? (void *) stage : p->d_raw[ss], src, bytes, cudaMemcpyHostToDevice, p->s_copy); copy_issued = true; }
			if (e == cudaSuccess) e = cudaEventRecord(p->ev_h2d[ss], p->s_copy);
			if (e == cudaSuccess) e = cudaStreamWaitEvent(p->s_ingest, p->ev_h2d[ss], 0);
			if (e != cudaSuccess) { rc = tsdrgpu_fail(ctx, TSDRGPU_ECUDA, "H2D of the plugin's block", e, __FILE__, __LINE__); break; }
			if (fmt != TSDRGPU_FMT_FLOAT) {                                    // raw samples -> float IQ, on the device
				const size_t want = (items_count / 4 + 255) / 256;
				pl_convert<<<(unsigned) (want < 2048 ? (want ? want : 1) : 2048), 256, 0, p->s_ingest>>>(p->d_raw[ss], stage, items_count, fmt);
				ctx->launches++;
				if ((e = cudaGetLastError()) != cudaSuccess) { rc = tsdrgpu_fail(ctx, TSDRGPU_ECUDA, "kernel launch", e, __FILE__, __LINE__); break; }
			}
			p->stats.h2d_bytes += bytes;
			// the spectrum reads the block as received, on this stream (covered by ev_used)
			if (spectrum && (rc = tsdrgpu_spectrum_run(p->spectrum, p->s_ingest, stage, size2, gap))) break;
			float *wide = stage;                                               // what the scan and the tuner read
			if (notched) {                                                     // the stopbands removed (notch.cu)
				if (p->nout_cap[ss] < 2 * size2) cudaStreamSynchronize(p->s_ingest);
				if ((rc = grow(ctx, p->s_ingest, &p->d_nout[ss], &p->nout_cap[ss], 2 * size2, 0))) break;
				if ((rc = tsdrgpu_notch_run(p->notch, p->s_ingest, stage, size2, gap, p->d_nout[ss], NULL, NULL))) break;
				wide = p->d_nout[ss];
			}
			d_in = wide;
			// the scan reads the wideband block on this stream (covered by ev_used); its heavy part runs on a stream of its own
			if (scanning && (rc = tsdrgpu_scan_run(p->scan, p->s_ingest, wide, size2, gap))) break;
			if (tuned) {                                                       // shift, low-pass, decimate (tuner.cu)
				if (p->tout_cap[ss] < 2 * n2 + 2) cudaStreamSynchronize(p->s_ingest);
				if ((rc = grow(ctx, p->s_ingest, &p->d_tout[ss], &p->tout_cap[ss], 2 * n2 + 2, 0))) break;
				if ((rc = tsdrgpu_tuner_run(p->tuner, p->s_ingest, wide, size2, gap, p->d_tout[ss], NULL, NULL))) break;
				p->tn_pos += gap + size2;
				d_in = p->d_tout[ss];
			}
			if (need_data) { if ((rc = feed_capture(p, d_in, n2, dropped != 0))) break; }
			else if (plots_on && dropped != 0) p->cap_fill = 0;
		} else {
			if (spectrum && gap > 0 && (rc = tsdrgpu_spectrum_run(p->spectrum, p->s_ingest, NULL, 0, gap))) break;
			if (notched && gap > 0 && (rc = tsdrgpu_notch_run(p->notch, p->s_ingest, NULL, 0, gap, NULL, NULL, NULL))) break;
			if (scanning && gap > 0 && (rc = tsdrgpu_scan_run(p->scan, p->s_ingest, NULL, 0, gap))) break;
			if (tuned && gap > 0) {                                            // an empty block that only reports a loss
				if ((rc = tsdrgpu_tuner_run(p->tuner, p->s_ingest, NULL, 0, gap, NULL, NULL, NULL))) break;
				p->tn_pos += gap;
			}
			if (plots_on && dropped != 0) p->cap_fill = 0;
		}
		uint32_t skip = 0;
		const uint32_t fwd = p->dev_drop.add((uint32_t) n2, (uint32_t) block, true, &skip);
		if (fwd) {
			float *where;
			if ((rc = decim_set_elem(p, 2))) break;
			if (p->decim_cap < 2 * (p->decim_read + p->decim_fill + fwd)) cudaStreamSynchronize(p->s_ingest);
			if ((rc = decim_reserve(p, fwd, &where))) break;
			cudaError_t e = cudaStreamWaitEvent(p->s_ingest, p->ev_decim, 0);  // the last compaction of the decimator input is done
			if (e == cudaSuccess) {
				pl_copy_f32<<<(unsigned) ((2ull * fwd + 255) / 256 < 2048 ? (2ull * fwd + 255) / 256 : 2048), 256, 0, p->s_ingest>>>(d_in + 2ull * skip, where, 2ull * fwd);
				ctx->launches++;
				e = cudaGetLastError();
			}
			if (e != cudaSuccess) { rc = tsdrgpu_fail(ctx, TSDRGPU_ECUDA, "append to the decimator input", e, __FILE__, __LINE__); break; }
			p->decim_fill += fwd;
		}
		{
			cudaError_t e = cudaSuccess;
			if (need_copy) e = cudaEventRecord(p->ev_used[ss], p->s_ingest);  // the slot may be overwritten after this point
			if (e == cudaSuccess) e = cudaEventRecord(p->ev_ingest, p->s_ingest);
			if (e == cudaSuccess) e = cudaStreamWaitEvent(p->s_main, p->ev_ingest, 0);      // the resampler may read what was appended
			if (e != cudaSuccess) { rc = tsdrgpu_fail(ctx, TSDRGPU_ECUDA, "stream ordering", e, __FILE__, __LINE__); break; }
		}
		// Everything above and the launches below are only ENQUEUED (ordered on the device by events), so the host's launch
		// work for the heavy kernels runs while this block's H2D copy is still in flight; the copy is waited for last.
		rc = drain_blocks(p);
	} while (0);
	if (copy_issued && (wait_for_copy || rc != TSDRGPU_OK)) {
		const cudaError_t e = cudaStreamSynchronize(p->s_copy);             // the host buffer has been read
		if (e != cudaSuccess && rc == TSDRGPU_OK) return tsdrgpu_fail(ctx, TSDRGPU_ECUDA, "cudaStreamSynchronize(s_copy)", e, __FILE__, __LINE__);
	}
	return rc;
}

}  // extern "C"
