/*
 * TSDRLibrary.c -- the tsdr_* host library (plain C) on top of the sm_100a kernels behind include/tsdrgpu.h.
 *
 * Drop-in for the reference's TempestSDR/src/TSDRLibrary.c + TSDRPluginLoader.c: same exported symbols, same
 * status codes and error-text ownership, same callback types and threading contract (include/TSDRLibrary.h), same
 * ten-symbol plugin ABI (include/TSDRPlugin.h).  What differs is everything underneath process(): instead of three
 * worker threads joined by mutex-guarded float rings, the plugin's buffer goes to the GPU once
 * (tsdrgpu_pipeline_process) and finished frames / plots come back on the pipeline's delivery thread.
 *
 * There is no CPU fallback: if the CUDA library cannot create a context, tsdr_readasync fails with
 * TSDR_CANNOT_OPEN_DEVICE and the reason in tsdr_getlasterrortext().
 */
#include "../../include/TSDRLibrary.h"
#include "../../include/TSDRCodes.h"
#include "../../include/TSDRPlugin.h"
#include "../../include/TSDRPluginX.h"
#include "../../include/tsdrgpu.h"

#include <dlfcn.h>
#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define MAX_PIXELS (4000 * 4000)          /* MAX_ARR_SIZE, TSDRLibrary.c:31 */
#define MAX_SAMPLE_RATE (500e6)           /* TSDRLibrary.c:32,186 */

typedef struct {
	void *handle;
	int      (*init)(const char *);
	void     (*getName)(char *);
	uint32_t (*setsamplerate)(uint32_t);
	uint32_t (*getsamplerate)(void);
	int      (*setbasefreq)(uint32_t);
	int      (*stop)(void);
	int      (*setgain)(float);
	int      (*readasync)(tsdrplugin_readasync_function, void *);
	char *   (*getlasterrortext)(void);
	void     (*cleanup)(void);
	tsdrpluginx_set_raw_sink_fn set_raw_sink;       /* optional 11th symbol (include/TSDRPluginX.h), NULL for ordinary plugins */
	volatile int initialized;
} plugin_t;

struct tsdr_lib {
	plugin_t plugin;
	volatile int running, nativerunning;
	uint32_t samplerate, samplerate_real;
	int width, height;
	double pixelrate, refreshrate, pixeltimeoversampletime;
	uint32_t centfreq;
	float gain, motionblur;
	char *errormsg, *errormsg_old; int errormsg_code;
	uint32_t params_int[COUNT_PARAM_INT];
	double params_double[COUNT_PARAM_DOUBLE];
	tsdr_value_changed_callback callback;
	tsdr_on_plot_ready_callback plotready_callback;
	void *callbackctx;
	/* run state */
	tsdr_readasync_function frame_cb; void *frame_ctx;
	tsdrgpu_ctx_t *gpu; tsdrgpu_pipeline_t *pipe;
	int gpu_failed;
	pthread_mutex_t mu; pthread_cond_t finished;
	/* t->pipe lives from tsdr_readasync's set-up to its tear-down while setters arrive from other threads: readers (the
	 * setters, the plugin's data callback) hold pipe_lock shared, the tear-down takes it exclusively before the object dies */
	pthread_rwlock_t pipe_lock;
	pthread_mutex_t err_mu;              /* errormsg is replaced from the plugin's thread too (GPU failures) */
	/* optional timing of the data callback (TSDR_STATS_FILE=<path>): where a run's wall time goes, per block */
	int stats_on; uint64_t cb_count; double cb_inside_s, cb_outside_s, cb_last_exit;
	struct { double t, inside, outside; uint64_t n; } cb_log[1024]; int cb_nlog;   /* cumulative values every 128 callbacks (CLOCK_MONOTONIC) */
	/* TSDR_TUNER=<offset_hz>,<bandwidth_hz>[,<decimation>[,<ntaps>]] (read by tsdr_readasync): the run demodulates that sub-band
	 * only, at samplerate_real / tuner_d (1 = no tuner) */
	double tn_offset, tn_bw; int tuner_d, tn_ntaps;
	/* TSDR_SCAN=<channels>[,<taps_per_channel>] with TSDR_SCAN_FILE=<path> (read by tsdr_readasync): a frame-rate detector on every
	 * sub-band of the capture; its table is written to the file as CSV when the run ends */
	int sc_k, sc_q; const char *sc_file;
	/* TSDR_NOTCH=<center_hz>:<width_hz>[,<center_hz>:<width_hz>...] with an optional TSDR_NOTCH_TAPS=<ntaps> (read by
	 * tsdr_readasync): those stopbands are removed from every block before anything else reads it */
	int nt_n, nt_taps; double nt_centers[32], nt_widths[32];
	/* TSDR_SPECTRUM=<nfft> with TSDR_SPECTRUM_FILE=<path> (read by tsdr_readasync): the capture's power spectrum, written to the file
	 * as CSV when the run ends */
	int sp_nfft; const char *sp_file;
};

/* ---- error text: library-owned, NULL after a successful call (TSDRLibrary.c:136-159) ---------------------- */
static int fail(tsdr_lib_t *t, const char *msg, int status) {
	if (status == TSDR_OK) { t->errormsg_code = status; return status; }
	if (!msg) msg = "An exception with no detailed explanation cause has occurred. This could as well be a bug in the TSDRlibrary or in one of its plugins.";
	/* the previous text is kept alive until the NEXT failure replaces it (a reader that fetched the pointer just before an
	 * update still sees valid memory, as with the reference's realloc'd buffer nobody frees in between) */
	pthread_mutex_lock(&t->err_mu);
	free(t->errormsg_old);
	t->errormsg_old = t->errormsg;
	t->errormsg = strdup(msg);
	t->errormsg_code = status;
	pthread_mutex_unlock(&t->err_mu);
	return status;
}
static int ok(tsdr_lib_t *t) { t->errormsg_code = TSDR_OK; return TSDR_OK; }
static int plugin_result(tsdr_lib_t *t, int status) {
	return status == TSDR_OK ? ok(t) : fail(t, t->plugin.getlasterrortext ? t->plugin.getlasterrortext() : NULL, status);
}

char *tsdr_getlasterrortext(tsdr_lib_t *t) {
	pthread_mutex_lock(&t->err_mu);
	char *text = t->errormsg_code == TSDR_OK ? NULL : t->errormsg;
	pthread_mutex_unlock(&t->err_mu);
	return text;
}

/* run `call` on the live pipeline, if there is one, with the object pinned against the run's tear-down */
#define WITH_PIPE(t, call) do { pthread_rwlock_rdlock(&(t)->pipe_lock); if ((t)->pipe) { call; } pthread_rwlock_unlock(&(t)->pipe_lock); } while (0)

/* ---- geometry (set_internal_samplerate, TSDRLibrary.c:540-550) ------------------------------------------- */
static void set_internal_samplerate(tsdr_lib_t *t, uint32_t samplerate) {
	int w; double pr, pt;
	t->samplerate = samplerate;
	tsdrgpu_geometry(samplerate, t->height, t->refreshrate, &w, &pr, &pt);
	t->width = w; t->pixelrate = pr;
	if (t->samplerate != 0 && t->pixelrate != 0) t->pixeltimeoversampletime = pt;
}

/* ---- plugin loader: dlopen(RTLD_NOW) + exactly these ten symbols (TSDRPluginLoader.c:33-72) --------------- */
static void plugin_close(plugin_t *p) {
	if (p->initialized && p->set_raw_sink) p->set_raw_sink(NULL);
	if (p->initialized && p->cleanup) p->cleanup();
	p->initialized = 0;
	if (p->handle) { dlclose(p->handle); p->handle = NULL; }
}
static int plugin_load(plugin_t *p, const char *path) {
	memset(p, 0, sizeof *p);
	p->handle = dlopen(path, RTLD_NOW);
	if (!p->handle) { fprintf(stderr, "Library %s load exception: %s\n", path, dlerror()); return TSDR_INCOMPATIBLE_PLUGIN; }
#define SYM(field, name) do { *(void **) (&p->field) = dlsym(p->handle, name); if (!p->field) return TSDR_ERR_PLUGIN; } while (0)
	SYM(init, "tsdrplugin_init"); SYM(getsamplerate, "tsdrplugin_getsamplerate"); SYM(getName, "tsdrplugin_getName");
	SYM(setsamplerate, "tsdrplugin_setsamplerate"); SYM(setbasefreq, "tsdrplugin_setbasefreq"); SYM(stop, "tsdrplugin_stop");
	SYM(setgain, "tsdrplugin_setgain"); SYM(readasync, "tsdrplugin_readasync"); SYM(getlasterrortext, "tsdrplugin_getlasterrortext");
	SYM(cleanup, "tsdrplugin_cleanup");
#undef SYM
	*(void **) (&p->set_raw_sink) = dlsym(p->handle, "tsdrpluginx_set_raw_sink");      /* optional */
	p->initialized = 1;
	return TSDR_OK;
}

/* ---- lifecycle -------------------------------------------------------------------------------------------- */
void tsdr_init(tsdr_lib_t **out, tsdr_value_changed_callback callback, tsdr_on_plot_ready_callback plotready_callback, void *ctx) {
	tsdr_lib_t *t = (tsdr_lib_t *) calloc(1, sizeof(tsdr_lib_t));   /* every field defined, unlike TSDRLibrary.c:62-94 */
	t->callback = callback; t->plotready_callback = plotready_callback; t->callbackctx = ctx;
	pthread_mutex_init(&t->mu, NULL); pthread_cond_init(&t->finished, NULL);
	pthread_rwlock_init(&t->pipe_lock, NULL); pthread_mutex_init(&t->err_mu, NULL);
	*out = t;
}

void tsdr_free(tsdr_lib_t **pt) {
	tsdr_lib_t *t = *pt;
	if (!t) return;
	t->callback = NULL; t->plotready_callback = NULL;
	plugin_close(&t->plugin);
	if (t->gpu) tsdrgpu_destroy(t->gpu);
	free(t->errormsg); free(t->errormsg_old);
	pthread_mutex_destroy(&t->mu); pthread_cond_destroy(&t->finished);
	pthread_rwlock_destroy(&t->pipe_lock); pthread_mutex_destroy(&t->err_mu);
	free(t);
	*pt = NULL;
}

void tsdr_reset(tsdr_lib_t *t) { (void) t; /* per-run DSP state lives in the pipeline object created by tsdr_readasync */ }
void *tsdr_getctx(tsdr_lib_t *t) { return t->callbackctx; }
int tsdr_isrunning(tsdr_lib_t *t) { return t->nativerunning; }

int tsdr_getsamplerate(tsdr_lib_t *t) {
	if (!t->plugin.initialized) return fail(t, "Cannot change sample rate. Plugin not loaded yet.", TSDR_ERR_PLUGIN);
	t->samplerate_real = t->plugin.getsamplerate();
	if (t->samplerate_real == 0 || t->samplerate_real > MAX_SAMPLE_RATE) return fail(t, "Invalid/unsupported value for sample rate.", TSDR_SAMPLE_RATE_WRONG);
	set_internal_samplerate(t, t->samplerate_real / (uint32_t) (t->tuner_d > 1 ? t->tuner_d : 1));
	return ok(t);
}

/* TSDR_TUNER: numbers separated by commas, all of them consumed; checked against the plugin's rate by the tuner's own rules */
static int parse_tuner(tsdr_lib_t *t, const char *text) {
	double v[4] = {0.0, 0.0, 1.0, 0.0};
	int n = 0;
	const char *c = text;
	for (;;) {
		char *e;
		const double x = strtod(c, &e);
		if (e == c || n == 4) { n = -1; break; }
		v[n++] = x; c = e;
		while (*c == ' ') c++;
		if (*c != ',') break;
		c++;
	}
	if (n < 2 || *c != '\0' || !(v[2] >= 1.0 && v[2] <= 1024.0 && v[2] == (double) (int) v[2]) || !(v[3] >= 0.0 && v[3] <= 65536.0 && v[3] == (double) (int) v[3]))
		return fail(t, "TSDR_TUNER: expected <offset_hz>,<bandwidth_hz>[,<decimation>[,<ntaps>]] with an integer decimation and ntaps", TSDR_INVALID_PARAMETER_VALUE);
	if (tsdrgpu_tuner_design(t->samplerate_real, v[0], v[1], (int) v[2], (int) v[3], NULL, 0, NULL, NULL) != TSDRGPU_OK)
		return fail(t, tsdrgpu_last_error(NULL), TSDR_INVALID_PARAMETER_VALUE);
	t->tn_offset = v[0]; t->tn_bw = v[1]; t->tuner_d = (int) v[2]; t->tn_ntaps = (int) v[3];
	return TSDR_OK;
}

/* TSDR_SCAN: one or two integers separated by a comma, all of it consumed; checked against the plugin's rate by the channelizer's
 * own rules, and only together with TSDR_SCAN_FILE */
static int parse_scan(tsdr_lib_t *t, const char *text, const char *file) {
	long v[2] = {0, 0};
	int n = 0;
	const char *c = text;
	for (;;) {
		char *e;
		const long x = strtol(c, &e, 10);
		if (e == c || n == 2) { n = -1; break; }
		v[n++] = x; c = e;
		while (*c == ' ') c++;
		if (*c != ',') break;
		c++;
	}
	if (n < 1 || *c != '\0' || v[0] < 1 || v[0] > 4096 || v[1] < 0 || v[1] > 4096)
		return fail(t, "TSDR_SCAN: expected <channels>[,<taps_per_channel>] with integer values", TSDR_INVALID_PARAMETER_VALUE);
	if (!file || !file[0]) return fail(t, "TSDR_SCAN: needs TSDR_SCAN_FILE=<path> for the table", TSDR_INVALID_PARAMETER_VALUE);
	if (tsdrgpu_channelizer_design(t->samplerate_real, (int) v[0], (int) v[1], NULL, 0, NULL) != TSDRGPU_OK)
		return fail(t, tsdrgpu_last_error(NULL), TSDR_INVALID_PARAMETER_VALUE);
	t->sc_k = (int) v[0]; t->sc_q = (int) v[1]; t->sc_file = file;
	return TSDR_OK;
}

/* TSDR_NOTCH: center:width pairs separated by commas, all of it consumed; TSDR_NOTCH_TAPS: one integer.  Checked against the
 * plugin's rate by the notch's own rules */
static int parse_notch(tsdr_lib_t *t, const char *text, const char *taps) {
	int n = 0;
	const char *c = text;
	for (;;) {
		char *e;
		if (n == 32) return fail(t, "TSDR_NOTCH: at most 32 notches", TSDR_INVALID_PARAMETER_VALUE);
		const double f = strtod(c, &e);
		if (e == c || *e != ':') { n = -1; break; }
		c = e + 1;
		const double w = strtod(c, &e);
		if (e == c) { n = -1; break; }
		t->nt_centers[n] = f; t->nt_widths[n] = w; n++; c = e;
		while (*c == ' ') c++;
		if (*c != ',') break;
		c++;
	}
	if (n < 1 || *c != '\0') return fail(t, "TSDR_NOTCH: expected <center_hz>:<width_hz>[,<center_hz>:<width_hz>...]", TSDR_INVALID_PARAMETER_VALUE);
	long L = 0;
	if (taps && taps[0]) {
		char *e;
		L = strtol(taps, &e, 10);
		if (e == taps || *e != '\0' || L < 1 || L > 1000000) return fail(t, "TSDR_NOTCH_TAPS: expected an odd integer ntaps", TSDR_INVALID_PARAMETER_VALUE);
	}
	if (tsdrgpu_notch_design(t->samplerate_real, n, t->nt_centers, t->nt_widths, (int) L, NULL, 0, NULL, NULL) != TSDRGPU_OK)
		return fail(t, tsdrgpu_last_error(NULL), TSDR_INVALID_PARAMETER_VALUE);
	t->nt_n = n; t->nt_taps = (int) L;
	return TSDR_OK;
}

/* TSDR_SPECTRUM: one integer, only together with TSDR_SPECTRUM_FILE */
static int parse_spectrum(tsdr_lib_t *t, const char *text, const char *file) {
	char *e;
	const long v = strtol(text, &e, 10);
	if (e == text || *e != '\0' || v < 1 || v > 1000000) return fail(t, "TSDR_SPECTRUM: expected <nfft>, an integer", TSDR_INVALID_PARAMETER_VALUE);
	if (!file || !file[0]) return fail(t, "TSDR_SPECTRUM: needs TSDR_SPECTRUM_FILE=<path> for the spectrum", TSDR_INVALID_PARAMETER_VALUE);
	if (tsdrgpu_spectrum_check(t->samplerate_real, (int) v) != TSDRGPU_OK) return fail(t, tsdrgpu_last_error(NULL), TSDR_INVALID_PARAMETER_VALUE);
	t->sp_nfft = (int) v; t->sp_file = file;
	return TSDR_OK;
}

/* the spectrum as CSV, frequency ascending, density in dB per Hz */
static void write_spectrum(tsdr_lib_t *t, tsdrgpu_pipeline_t *p) {
	static double psd[16384];
	int n = 0; uint64_t segs = 0;
	if (tsdrgpu_pipeline_spectrum(p, psd, 16384, &n, &segs) != TSDRGPU_OK) return;
	FILE *f = fopen(t->sp_file, "w");
	if (!f) return;
	fprintf(f, "frequency_hz,psd_db_per_hz\n");
	for (int i = 0; i < n; i++)
		fprintf(f, "%.3f,%.6f\n", ((double) i - n / 2) * (double) t->samplerate_real / n, psd[i] > 0.0 ? 10.0 * log10(psd[i]) : -400.0);
	fclose(f);
}

/* the scan's table as CSV, one row per channel, highest frame_score first (ties: lower channel first) */
struct scan_row { int channel; tsdrgpu_scan_channel_t r; };
static int scan_cmp(const void *a, const void *b) {
	const struct scan_row *x = (const struct scan_row *) a, *y = (const struct scan_row *) b;
	if (x->r.frame_score != y->r.frame_score) return x->r.frame_score < y->r.frame_score ? 1 : -1;
	return x->channel - y->channel;
}
static void write_scan(tsdr_lib_t *t, tsdrgpu_pipeline_t *p) {
	tsdrgpu_scan_channel_t rec[256];
	struct scan_row rows[256];
	int n = 0;
	if (tsdrgpu_pipeline_scan_results(p, rec, 256, &n) != TSDRGPU_OK) return;
	for (int c = 0; c < n; c++) { rows[c].channel = c; rows[c].r = rec[c]; }
	qsort(rows, (size_t) n, sizeof rows[0], scan_cmp);
	FILE *f = fopen(t->sc_file, "w");
	if (!f) return;
	fprintf(f, "channel,offset_hz,rate,captures,fps,height,frame_score,line_score\n");
	for (int i = 0; i < n; i++)
		fprintf(f, "%d,%.3f,%u,%llu,%.6f,%d,%.6f,%.6f\n", rows[i].channel, rows[i].r.offset_hz, rows[i].r.rate, (unsigned long long) rows[i].r.captures,
		        rows[i].r.fps, rows[i].r.height, rows[i].r.frame_score, rows[i].r.line_score);
	fclose(f);
}

int tsdr_setbasefreq(tsdr_lib_t *t, uint32_t freq) {
	t->centfreq = freq;
	if (!t->plugin.initialized) return ok(t);
	t->params_int[PARAM_AUTOCORR_PLOTS_RESET] = 2;            /* frameratedetector_flushcachedestimation */
	WITH_PIPE(t, tsdrgpu_pipeline_set_param_int(t->pipe, PARAM_AUTOCORR_PLOTS_RESET, 2));
	return plugin_result(t, t->plugin.setbasefreq(t->centfreq));
}

int tsdr_setgain(tsdr_lib_t *t, float gain) {
	t->gain = gain;
	if (!t->plugin.initialized) return ok(t);
	return plugin_result(t, t->plugin.setgain(gain));
}

int tsdr_unloadplugin(tsdr_lib_t *t) {
	if (!t->plugin.initialized) return fail(t, "No plugin has been loaded so it can't be unloaded", TSDR_ERR_PLUGIN);
	if (t->nativerunning || t->running) return fail(t, "The library is already running in async mode. Stop it first!", TSDR_ALREADY_RUNNING);
	plugin_close(&t->plugin);
	return ok(t);
}

static const tsdrx_raw_sink_t g_raw_sink;          /* defined beside tsdr_readasync */

int tsdr_loadplugin(tsdr_lib_t *t, const char *path, const char *params) {
	if (t->nativerunning || t->running) return fail(t, "The library is already running in async mode. Stop it first!", TSDR_ALREADY_RUNNING);
	plugin_close(&t->plugin);
	int status = plugin_load(&t->plugin, path);
	if (status == TSDR_INCOMPATIBLE_PLUGIN)
		return fail(t, "The plugin cannot be loaded. It is incompatible or there are depending libraries missing. Please check the readme file that comes with the plugin.", status);
	if (status != TSDR_OK) { plugin_close(&t->plugin); return fail(t, "The selected library is not a valid TSDR plugin!", status); }
	char name[256];
	t->plugin.getName(name);
	if (t->plugin.set_raw_sink && !getenv("TSDR_NO_RAW_SINK")) t->plugin.set_raw_sink(&g_raw_sink);
	char *mutable_params = strdup(params ? params : "");    /* RawFile's tokenizer writes into the string it is given */
	status = t->plugin.init(mutable_params);
	free(mutable_params);
	if (status != TSDR_OK) { fail(t, t->plugin.getlasterrortext(), status); plugin_close(&t->plugin); return status; }
	return ok(t);
}

int tsdr_setresolution(tsdr_lib_t *t, int height, double refreshrate) {
	if (height <= 0 || refreshrate <= 0) return fail(t, "The supplied height is invalid or refreshrate is negative!", TSDR_WRONG_VIDEOPARAMS);
	t->height = height; t->refreshrate = refreshrate;
	if (t->plugin.initialized) set_internal_samplerate(t, t->samplerate);
	WITH_PIPE(t, tsdrgpu_pipeline_set_resolution(t->pipe, height, refreshrate));
	return ok(t);
}

int tsdr_motionblur(tsdr_lib_t *t, float coeff) {
	if (coeff < 0.0f || coeff > 1.0f) return TSDR_WRONG_VIDEOPARAMS;
	t->motionblur = coeff;
	WITH_PIPE(t, tsdrgpu_pipeline_set_motionblur(t->pipe, coeff));
	return ok(t);
}

int tsdr_sync(tsdr_lib_t *t, int pixels, int direction) {      /* TSDRLibrary.c:576-602 */
	if (pixels == 0) return TSDR_OK;
	int delta = 0;
	/* the geometry the frames are produced with right now: in superbandwidth mode the pipeline runs at 4x the plugin's rate
	 * (superb_ondataready calls set_internal_samplerate(4 fs), superbandwidth.c:151, so tsdr->width follows there too) */
	int width = t->width, height = t->height;
	WITH_PIPE(t, tsdrgpu_pipeline_get_geometry(t->pipe, &width, &height, NULL));
	switch (direction) {
	case DIRECTION_CUSTOM: delta = pixels; break;
	case DIRECTION_UP:
		if (pixels > height || pixels < 0) return fail(t, "Cannot shift up with more pixels than the height of the image or shift is negative!", TSDR_WRONG_VIDEOPARAMS);
		delta = pixels * width; break;
	case DIRECTION_DOWN:
		if (pixels > height || pixels < 0) return fail(t, "Cannot shift down with more pixels than the height of the image or shift is negative!", TSDR_WRONG_VIDEOPARAMS);
		delta = -pixels * width; break;
	case DIRECTION_LEFT:
		if (pixels > width || pixels < 0) return fail(t, "Cannot shift to the left with more pixels than the width of the image or shift is negative!", TSDR_WRONG_VIDEOPARAMS);
		delta = pixels; break;
	case DIRECTION_RIGHT:
		if (pixels > width || pixels < 0) return fail(t, "Cannot shift to the right with more pixels than the width of the image or shift is negative!", TSDR_WRONG_VIDEOPARAMS);
		delta = -pixels; break;
	}
	if (delta) WITH_PIPE(t, tsdrgpu_pipeline_sync(t->pipe, delta));
	return ok(t);
}

int tsdr_setparameter_int(tsdr_lib_t *t, int parameter, uint32_t value) {
	if (parameter < 0 || parameter >= COUNT_PARAM_INT) return fail(t, "Invalid integer parameter id", TSDR_INVALID_PARAMETER);
	t->params_int[parameter] = value;
	WITH_PIPE(t, tsdrgpu_pipeline_set_param_int(t->pipe, parameter, value));
	return ok(t);
}

int tsdr_setparameter_double(tsdr_lib_t *t, int parameter, double value) {
	if (parameter < 0 || parameter >= COUNT_PARAM_DOUBLE) return fail(t, "Invalid double floating point parameter id", TSDR_INVALID_PARAMETER);
	printf("Parameter %d to double value %f\n", parameter, value); fflush(stdout);   /* TSDRLibrary.c:616 */
	return ok(t);
}

/* ---- the run loop ----------------------------------------------------------------------------------------- */
static void on_frame(float *buf, int w, int h, void *user) {
	tsdr_lib_t *t = (tsdr_lib_t *) user;
	if (t->frame_cb) t->frame_cb(buf, w, h, t->frame_ctx);
}
static void on_value(int id, double a0, double a1, void *user) {
	tsdr_lib_t *t = (tsdr_lib_t *) user;
	if (id == VALUE_ID_PLL_FRAMERATE) {       /* the PLL moved the refresh rate: mirror it (syncdetector.c:149-150) */
		t->refreshrate = a0;
		set_internal_samplerate(t, t->samplerate);
	}
	if (t->callback) t->callback(id, a0, a1, t->callbackctx);
}
static void on_plot(int plot_id, int offset, double *values, int size, uint32_t samplerate, void *user) {
	tsdr_lib_t *t = (tsdr_lib_t *) user;
	if (t->plotready_callback) t->plotready_callback(plot_id, offset, values, size, samplerate, t->callbackctx);
}

/* shiftfreq (TSDRLibrary.c:208-211): the superbandwidth mode retunes the front end between hops */
static void on_retune(int32_t offset_hz, void *user) {
	tsdr_lib_t *t = (tsdr_lib_t *) user;
	if (t->plugin.initialized) t->plugin.setbasefreq(t->centfreq + offset_hz);
}

/* the plugin's data callback == the reference's process() (TSDRLibrary.c:264-298), on the plugin's thread */
static double now_s(void) { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return (double) ts.tv_sec + 1e-9 * (double) ts.tv_nsec; }
static void process(float *buf, uint64_t items_count, void *ctx, int64_t samples_dropped) {
	tsdr_lib_t *t = (tsdr_lib_t *) ctx;
	if (t->gpu_failed) return;
	int rc = TSDRGPU_OK;
	double t_in = 0.0;
	if (t->stats_on) { t_in = now_s(); if (t->cb_count) t->cb_outside_s += t_in - t->cb_last_exit; }
	WITH_PIPE(t, rc = tsdrgpu_pipeline_process(t->pipe, buf, items_count, samples_dropped));
	if (t->stats_on) {
		t->cb_last_exit = now_s(); t->cb_inside_s += t->cb_last_exit - t_in; t->cb_count++;
		if ((t->cb_count & 127u) == 0 && t->cb_nlog < 1024) {
			t->cb_log[t->cb_nlog].t = t->cb_last_exit; t->cb_log[t->cb_nlog].inside = t->cb_inside_s;
			t->cb_log[t->cb_nlog].outside = t->cb_outside_s; t->cb_log[t->cb_nlog].n = t->cb_count; t->cb_nlog++;
		}
	}
	if (rc != TSDRGPU_OK) {
		t->gpu_failed = 1;
		fail(t, tsdrgpu_last_error(t->gpu), TSDR_CANNOT_OPEN_DEVICE);
		t->plugin.stop();
	}
}

/* ---- optional raw sink (include/TSDRPluginX.h): the plugin keeps its samples in wire format, the GPU converts ---- */
static int raw_ingest(const void *samples, int fmt, uint64_t items_count, void *ctx, int64_t samples_dropped) {
	tsdr_lib_t *t = (tsdr_lib_t *) ctx;
	if (t->gpu_failed) return 1;
	int rc = TSDRGPU_OK, live = 0;
	WITH_PIPE(t, (live = 1, rc = tsdrgpu_pipeline_process_raw(t->pipe, samples, fmt, items_count, samples_dropped)));
	if (!live) return 1;
	if (rc != TSDRGPU_OK) {
		t->gpu_failed = 1;
		fail(t, tsdrgpu_last_error(t->gpu), TSDR_CANNOT_OPEN_DEVICE);
		t->plugin.stop();
		return 1;
	}
	return 0;
}
static void *raw_alloc_host(size_t bytes, void *ctx) {
	tsdr_lib_t *t = (tsdr_lib_t *) ctx;
	void *p = NULL;
	return (t && t->gpu && tsdrgpu_malloc_host(t->gpu, bytes, &p) == TSDRGPU_OK) ? p : NULL;
}
static void raw_free_host(void *p, void *ctx) { tsdr_lib_t *t = (tsdr_lib_t *) ctx; if (t && t->gpu) tsdrgpu_free_host(t->gpu, p); }
static const tsdrx_raw_sink_t g_raw_sink = { 1, raw_ingest, raw_alloc_host, raw_free_host };

int tsdr_readasync(tsdr_lib_t *t, tsdr_readasync_function cb, void *ctx) {
	if (t->nativerunning || t->running) return fail(t, "The library is already running in async mode. Stop it first!", TSDR_ALREADY_RUNNING);
	if (!t->plugin.initialized) return fail(t, "Please load a working plugin first!", TSDR_ERR_PLUGIN);
	tsdr_reset(t);
	t->nativerunning = 1; t->running = 1; t->gpu_failed = 0;
	int status, pluginsfault = 0;
	t->tuner_d = 1; t->tn_bw = 0.0; t->sc_k = 0; t->nt_n = 0; t->sp_nfft = 0;
	if ((status = tsdr_getsamplerate(t)) != TSDR_OK) goto end;
	{
		const char *tuner = getenv("TSDR_TUNER");
		if (tuner && tuner[0]) {
			if ((status = parse_tuner(t, tuner)) != TSDR_OK) goto end;
			set_internal_samplerate(t, t->samplerate_real / (uint32_t) t->tuner_d);     /* the geometry of the tuned sub-band */
		}
		const char *scan = getenv("TSDR_SCAN");
		if (scan && scan[0] && (status = parse_scan(t, scan, getenv("TSDR_SCAN_FILE"))) != TSDR_OK) goto end;
		const char *notch = getenv("TSDR_NOTCH");
		if (notch && notch[0] && (status = parse_notch(t, notch, getenv("TSDR_NOTCH_TAPS"))) != TSDR_OK) goto end;
		const char *spec = getenv("TSDR_SPECTRUM");
		if (spec && spec[0] && (status = parse_spectrum(t, spec, getenv("TSDR_SPECTRUM_FILE"))) != TSDR_OK) goto end;
	}
	if (t->width <= 0 || t->height <= 0 || (long long) t->width * t->height > MAX_PIXELS) {
		status = fail(t, "The supplied height and the width are invalid!", TSDR_WRONG_VIDEOPARAMS);
		goto end;
	}
	if ((status = tsdr_setbasefreq(t, t->centfreq)) != TSDR_OK) goto end;
	if ((status = tsdr_setgain(t, t->gain)) != TSDR_OK) goto end;
	if (t->pixeltimeoversampletime <= 0) goto end;

	/* TSDR_CUDA_DEVICES="0,1,2,3": superbandwidth mode records one hop per listed GPU and shards the stitch over them
	 * (tsdrgpu_pipeline_set_superb_devices); the first entry is the device everything else runs on.  TSDR_CUDA_DEVICE=n: one GPU. */
	int devlist[16], ndev = 0;
	{
		const char *list = getenv("TSDR_CUDA_DEVICES");
		if (list) {
			char *copy = strdup(list), *save = NULL;
			for (char *tok = strtok_r(copy, ", ", &save); tok && ndev < 16; tok = strtok_r(NULL, ", ", &save)) devlist[ndev++] = atoi(tok);
			free(copy);
		}
	}
	if (!t->gpu) {
		const char *dev = getenv("TSDR_CUDA_DEVICE");
		if (tsdrgpu_create(&t->gpu, ndev > 0 ? devlist[0] : (dev ? atoi(dev) : 0)) != TSDRGPU_OK) {
			status = fail(t, tsdrgpu_last_error(NULL), TSDR_CANNOT_OPEN_DEVICE);
			t->gpu = NULL;
			goto end;
		}
	}
	{
		tsdrgpu_pipeline_config_t cfg;
		memset(&cfg, 0, sizeof cfg);
		cfg.samplerate = t->samplerate_real; cfg.height = t->height; cfg.refreshrate = t->refreshrate; cfg.motionblur = t->motionblur;
		memcpy(cfg.params_int, t->params_int, sizeof cfg.params_int);
		const char *bf = getenv("TSDR_BATCH_FRAMES");
		cfg.batch_frames = bf ? atoi(bf) : 1;               /* 1 frame per launch: lowest latency for an interactive host */
		cfg.batch_blocks = 10 * (cfg.batch_frames > 0 ? cfg.batch_frames : 1);
		cfg.block_when_busy = getenv("TSDR_NO_DROP") ? 1 : 0;
		t->frame_cb = cb; t->frame_ctx = ctx;
		tsdrgpu_pipeline_t *np = NULL;
		if (tsdrgpu_pipeline_create(t->gpu, &cfg, on_frame, on_value, on_plot, t, &np) != TSDRGPU_OK) {
			status = fail(t, tsdrgpu_last_error(t->gpu), TSDR_CANNOT_OPEN_DEVICE);
			goto end;
		}
		tsdrgpu_pipeline_set_retune(np, on_retune);
		/* a plugin keeps its buffer for the whole tsdrplugin_readasync (TSDRPlugin_RawFile.c:212, 263): page-lock it in place */
		tsdrgpu_pipeline_set_host_registration(np, getenv("TSDR_NO_HOST_REGISTER") ? 0 : 1);
		if (t->tn_bw > 0 && tsdrgpu_pipeline_set_tuner(np, t->tn_offset, t->tn_bw, t->tuner_d, t->tn_ntaps) != TSDRGPU_OK) {
			status = fail(t, tsdrgpu_last_error(t->gpu), TSDR_INVALID_PARAMETER_VALUE);
			tsdrgpu_pipeline_destroy(np);
			goto end;
		}
		if (t->sc_k > 0 && tsdrgpu_pipeline_set_scan(np, t->sc_k, t->sc_q) != TSDRGPU_OK) {
			status = fail(t, tsdrgpu_last_error(t->gpu), TSDR_INVALID_PARAMETER_VALUE);
			tsdrgpu_pipeline_destroy(np);
			goto end;
		}
		if ((t->nt_n > 0 && tsdrgpu_pipeline_set_notches(np, t->nt_n, t->nt_centers, t->nt_widths, t->nt_taps) != TSDRGPU_OK) ||
		    (t->sp_nfft > 0 && tsdrgpu_pipeline_set_spectrum(np, t->sp_nfft) != TSDRGPU_OK)) {
			status = fail(t, tsdrgpu_last_error(t->gpu), TSDR_INVALID_PARAMETER_VALUE);
			tsdrgpu_pipeline_destroy(np);
			goto end;
		}
		if (ndev > 1 && tsdrgpu_pipeline_set_superb_devices(np, devlist, ndev) != TSDRGPU_OK) {
			status = fail(t, tsdrgpu_last_error(t->gpu), TSDR_CANNOT_OPEN_DEVICE);
			tsdrgpu_pipeline_destroy(np);
			goto end;
		}
		/* opt-in extras (SURVEY section 8f), all off by default so that an unchanged host sees exactly the reference's callbacks */
		{
			const char *snr = getenv("TSDR_REPORT_SNR"), *mode = getenv("TSDR_DETECT_MODE"), *argb = getenv("TSDR_OUTPUT_ARGB");
			if ((snr && atoi(snr)) || (mode && atoi(mode))) tsdrgpu_pipeline_set_reports(np, snr && atoi(snr), mode && atoi(mode));
			if (argb && argb[0] && argb[0] != '0') tsdrgpu_pipeline_set_output_argb(np, 1, strcmp(argb, "inverted") == 0);
		}
		pthread_rwlock_wrlock(&t->pipe_lock);
		t->pipe = np;                                 /* published: setters on other threads reach the run from here on */
		pthread_rwlock_unlock(&t->pipe_lock);
	}
	t->stats_on = getenv("TSDR_STATS_FILE") != NULL; t->cb_count = 0; t->cb_inside_s = t->cb_outside_s = 0.0; t->cb_nlog = 0;
	status = t->plugin.readasync(process, t);                 /* blocks until tsdr_stop or a plugin error */
	if (status != TSDR_OK) pluginsfault = 1;
	if (t->stats_on) {                                         /* seconds inside process() vs. between two calls (= the plugin's own work) */
		FILE *sf = fopen(getenv("TSDR_STATS_FILE"), "w");
		if (sf) {
			fprintf(sf, "{\"callbacks\": %llu, \"inside_callback_s\": %.6f, \"between_callbacks_s\": %.6f, \"log\": [",
			        (unsigned long long) t->cb_count, t->cb_inside_s, t->cb_outside_s);
			for (int i = 0; i < t->cb_nlog; i++)
				fprintf(sf, "%s[%.6f, %.6f, %.6f, %llu]", i ? ", " : "", t->cb_log[i].t, t->cb_log[i].inside, t->cb_log[i].outside, (unsigned long long) t->cb_log[i].n);
			fprintf(sf, "]}\n");
			fclose(sf);
		}
	}
	tsdrgpu_pipeline_flush(t->pipe);
	if (t->sc_k > 0) write_scan(t, t->pipe);
	if (t->sp_nfft > 0) write_spectrum(t, t->pipe);
	{
		pthread_rwlock_wrlock(&t->pipe_lock);        /* no setter is inside the object any more, none can enter */
		tsdrgpu_pipeline_t *p = t->pipe;
		t->pipe = NULL;
		pthread_rwlock_unlock(&t->pipe_lock);
		tsdrgpu_pipeline_destroy(p);
	}
	if (t->gpu_failed) status = TSDR_CANNOT_OPEN_DEVICE;
end:
	t->tuner_d = 1;
	if (pluginsfault) fail(t, t->plugin.getlasterrortext(), status);
	pthread_mutex_lock(&t->mu);
	t->running = 0; t->nativerunning = 0;
	pthread_cond_broadcast(&t->finished);
	pthread_mutex_unlock(&t->mu);
	return status;
}

int tsdr_stop(tsdr_lib_t *t) {
	if (!t->running) return ok(t);
	const int status = t->plugin.stop();
	pthread_mutex_lock(&t->mu);
	while (t->running) pthread_cond_wait(&t->finished, &t->mu);   /* the reference waits for its workers here too */
	pthread_mutex_unlock(&t->mu);
	return plugin_result(t, status);
}
