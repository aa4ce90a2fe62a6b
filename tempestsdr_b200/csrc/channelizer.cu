// channelizer.cu -- polyphase filter bank ("channelizer") and the scan built on it: split the capture into K sub-bands at once and
// run the frame-rate detector on every one of them, to find where in a wideband capture the video emitters sit.  Nothing in the
// reference does this, so this file is tolerance-based like tuner.cu: FMA contraction is allowed, and every sum runs in one fixed
// order so that the bits do not depend on how the stream is cut into blocks.
//
// Definition (DESIGN.md section 5.7).  K channels, D = K/2, prototype h[0 .. QK-2] (the tuner's design at bandwidth fs/K).
// Channel c's output m is y_c[m] = sum_k h[k] x[mD - k] e^{-2 pi i c (mD - k) / K}.  With k = qK + rho this is
//   y_c[m] = (-1)^{c m} sum_rho e^{+2 pi i c rho / K} v_rho[m],   v_rho[m] = sum_q h[qK + rho] x[mD - qK - rho],
// K branch sums and one K-point DFT with a positive exponent per output; the mixer (-1)^{cm} is exact (2D = K), so unlike the
// tuner there is no per-sample sincospif.
//
// Kernel shape: one CTA per tile of T consecutive outputs.  The tile's input span (the last QK-2 pairs of earlier blocks come from a
// device-side history) is read from HBM once and staged in shared memory de-interleaved by K: row r holds the span samples i == r
// (mod K), with an odd row pitch.  Thread (rho, parity, g) owns R outputs of one parity: output m + 2 reads, for tap q, the sample
// output m read for tap q - 1, so a register window of R samples slides down the row by one shared-memory load per tap and feeds
// 2R FMAs (the tuner's scheme with stride K).  Lanes take consecutive rho, i.e. consecutive rows at the odd pitch: conflict-free.
// The branch sums go to shared memory, rows of K + 1 pairs, and a radix-2 decimation-in-frequency FFT (natural order in,
// bit-reversed out, twiddles from a table made in double on the host) turns each row into the K channels; the output pass reads
// the rows bit-reversed and writes channel-major, consecutive outputs on consecutive lanes.
//
// No tensor cores: the K-point DFT is a matrix product, but as one it costs 8K^2 flops per output against about 5K log2 K for the
// FFT, and TF32 does not hold the 1e-5 accuracy without a three-way split.
#include "common.cuh"
#include <math.h>

namespace {

constexpr int CH_R = 8;                                // outputs per thread and pass (the register window)
constexpr int CH_MIN_K = 2, CH_MAX_K = 256, CH_MIN_Q = 4, CH_MAX_Q = 32, CH_DEFAULT_Q = 16;
constexpr uint32_t CH_MIN_RATE = 130500;               // 1500 lines x 87 Hz: below it the line window starts at lag 0
constexpr size_t CH_SMEM_MAX = 227 * 1024;             // dynamic shared memory of one CTA on sm_100
constexpr size_t CH_SMEM_TARGET = 113 * 1024;          // two CTAs per SM

struct ChArgs {
	const float2 *in;          // this block's k input pairs
	const float2 *hist;        // x[p - L .. p - 1]
	void *out;
	const float *taps;         // taps[q * K + rho] = h[qK + rho], zero from QK - 1 on, Qp rows
	const float2 *tw;          // e^{+2 pi i j / K}, j < K/2
	long long p, g, k;         // position before the gap, gap, pairs in the block
	long long m_first, M, stride;
	int K, logK, D, L, Q, Qp, NP, U, P, mag;
};

struct ChGeom { int NT, Qp, NP, U, P, O; size_t smem; };

inline ChGeom ch_geometry(int K, int Q, int NP) {
	ChGeom g;
	g.NT = 2 * K > 256 ? 2 * K : 256;
	g.Qp = (Q + CH_R - 1) / CH_R * CH_R;
	g.NP = NP;
	g.O = CH_R * g.NT / K;                             // outputs per pass
	const int G = NP * (g.NT / (2 * K));               // thread groups along the tile
	g.U = G * CH_R + Q;                                // span columns
	g.P = g.U | 1;                                     // odd row pitch
	g.smem = sizeof(float) * (size_t) g.Qp * K + sizeof(float2) * ((size_t) K / 2 + (size_t) g.O * (K + 1) + (size_t) K * g.P);
	return g;
}
// passes per tile: enough that the new input outweighs the Q K halo four times, at most 8, halved until two CTAs fit an SM
inline ChGeom ch_pick(int K, int Q) {
	const int Qp = (Q + CH_R - 1) / CH_R * CH_R, per_pass = (2 * K > 256 ? 2 * K : 256) / (2 * K) * CH_R;
	int NP = 1;
	while (NP < 8 && NP * per_pass < 4 * Qp) NP *= 2;
	ChGeom g = ch_geometry(K, Q, NP);
	while (g.NP > 1 && g.smem > CH_SMEM_TARGET) g = ch_geometry(K, Q, g.NP / 2);
	return g;
}

// x[n]: the block's samples, zeros over the gap, before the stream and past the block's end, older samples from the history
__device__ __forceinline__ float2 ch_load(const ChArgs &a, long long n) {
	const long long b0 = a.p + a.g;
	if (n >= b0) return n - b0 < a.k ? ldg_stream_f2(a.in + (n - b0)) : make_float2(0.f, 0.f);
	if (n >= a.p || n < a.p - a.L) return make_float2(0.f, 0.f);
	return a.hist[n - (a.p - a.L)];
}

__global__ void __launch_bounds__(512) channelizer_pfb(ChArgs a) {
	extern __shared__ __align__(16) float ch_smem[];
	const int K = a.K, logK = a.logK, NT = blockDim.x, tid = threadIdx.x;
	const int O = CH_R * NT / K;
	float *s_taps = ch_smem;
	float2 *s_tw = reinterpret_cast<float2 *>(ch_smem + a.Qp * K);   // Qp * K is a multiple of 8
	float2 *s_v = s_tw + K / 2;
	float2 *s_x = s_v + O * (K + 1);
	const long long t0 = (long long) blockIdx.x * a.NP * O;          // the tile's first output, relative to m_first
	const long long base = (a.m_first + t0) * a.D - (long long) a.Q * K;   // absolute index of span sample 0
	for (int i = tid; i < a.Qp * K; i += NT) s_taps[i] = a.taps[i];
	for (int i = tid; i < K / 2; i += NT) s_tw[i] = a.tw[i];
	const int S = K * a.U;
	for (int i0 = tid; i0 < S; i0 += 4 * NT) {                      // four independent loads in flight per thread
		float2 v[4];
		#pragma unroll
		for (int j = 0; j < 4; j++) { const int i = i0 + j * NT; v[j] = i < S ? ch_load(a, base + i) : make_float2(0.f, 0.f); }
		#pragma unroll
		for (int j = 0; j < 4; j++) { const int i = i0 + j * NT; if (i < S) s_x[(i & (K - 1)) * a.P + (i >> logK)] = v[j]; }
	}
	__syncthreads();
	const int rho = tid & (K - 1), par = (tid >> logK) & 1, gl = tid >> (logK + 1), GP = NT / (2 * K);
	// output t (relative to the tile) of parity par reads span sample par D - rho + K (t / 2 - q + Q) for tap qK + rho
	const int c = par * a.D - rho;
	const float2 *row = s_x + (c & (K - 1)) * a.P;
	const float *hp = s_taps + rho;
	for (int pass = 0; pass < a.NP; pass++) {
		const int u0 = (pass * GP + gl) * CH_R + a.Q + (c < 0 ? -1 : 0);   // column of this thread's first output for q = 0
		float2 acc[CH_R], w[CH_R];
		#pragma unroll
		for (int r = 0; r < CH_R; r++) { acc[r] = make_float2(0.f, 0.f); w[r] = row[u0 + r]; }
		int nxt = u0 - 1;
		for (int q0 = 0; q0 < a.Qp; q0 += CH_R) {
			#pragma unroll
			for (int u = 0; u < CH_R; u++) {
				const float t = hp[(q0 + u) * K];
				#pragma unroll
				for (int r = 0; r < CH_R; r++) {
					const float2 v = w[(r - u + CH_R) % CH_R];
					acc[r].x = __fmaf_rn(t, v.x, acc[r].x);
					acc[r].y = __fmaf_rn(t, v.y, acc[r].y);
				}
				w[(2 * CH_R - 1 - u) % CH_R] = row[max(nxt, 0)];     // the window slides by one output; past column 0 only zero taps follow
				nxt--;
			}
		}
		#pragma unroll
		for (int r = 0; r < CH_R; r++) s_v[(2 * (gl * CH_R + r) + par) * (K + 1) + rho] = acc[r];
		__syncthreads();
		// K-point DFT of every row, positive exponent: radix-2 decimation in frequency, result in bit-reversed order
		for (int lh = logK - 1; lh >= 0; lh--) {
			const int half = 1 << lh;
			#pragma unroll
			for (int j = 0; j < CH_R / 2; j++) {
				const int b = tid + j * NT, o = b >> (logK - 1), bb = b & (K / 2 - 1);
				const int k = bb & (half - 1), i0 = o * (K + 1) + ((bb >> lh) << (lh + 1)) + k;
				const float2 x0 = s_v[i0], x1 = s_v[i0 + half], tw = s_tw[k << (logK - 1 - lh)];
				const float dx = x0.x - x1.x, dy = x0.y - x1.y;
				s_v[i0] = make_float2(x0.x + x1.x, x0.y + x1.y);
				s_v[i0 + half] = make_float2(__fmaf_rn(dx, tw.x, -__fmul_rn(dy, tw.y)), __fmaf_rn(dx, tw.y, __fmul_rn(dy, tw.x)));
			}
			__syncthreads();
		}
		#pragma unroll
		for (int j = 0; j < CH_R; j++) {
			const int e = tid + j * NT, o = e & (O - 1), ch = e / O;
			const long long tl = t0 + (long long) pass * O + o;
			if (tl < a.M) {
				float2 y = s_v[o * (K + 1) + (int) (__brev((unsigned) ch) >> (32 - logK))];
				if (ch & (int) ((a.m_first + tl) & 1)) { y.x = -y.x; y.y = -y.y; }          // (-1)^{c m}
				if (a.mag) reinterpret_cast<float *>(a.out)[ch * a.stride + tl] = mag_exact(y.x, y.y);
				else reinterpret_cast<float2 *>(a.out)[ch * a.stride + tl] = y;
			}
		}
		__syncthreads();
	}
}

// the history after this block: x[p + g + k - L .. p + g + k - 1], from the old history, the gap's zeros and the block
__global__ void __launch_bounds__(256) channelizer_history(ChArgs a, float2 *hist_new) {
	const int j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= a.L) return;
	hist_new[j] = ch_load(a, a.p + a.g + a.k - a.L + j);
}

inline int ch_bad(tsdrgpu_ctx_t *ctx, const char *what) { return tsdrgpu_fail(ctx, TSDRGPU_EINVAL, what, cudaSuccess, __FILE__, __LINE__); }

int ch_validate(tsdrgpu_ctx_t *ctx, uint32_t fs, int K, int Q, int *Q_out) {
	if (K < CH_MIN_K || K > CH_MAX_K || (K & (K - 1)) != 0) return ch_bad(ctx, "channelizer: channels must be a power of two in 2..256");
	if (Q != 0 && (Q < CH_MIN_Q || Q > CH_MAX_Q)) return ch_bad(ctx, "channelizer: taps_per_channel must be in 4..32 (0 = default)");
	if (Q == 0) Q = CH_DEFAULT_Q;
	if (fs == 0 || fs % (uint32_t) (K / 2) != 0) return ch_bad(ctx, "channelizer: the sample rate must be a multiple of channels / 2 (fs % (K/2) == 0)");
	if (2.0 * (double) fs / K < (double) CH_MIN_RATE) return ch_bad(ctx, "channelizer: the channel rate 2 fs / K must be at least 130500");
	if (ch_geometry(K, Q, 1).smem > CH_SMEM_MAX) return ch_bad(ctx, "channelizer: Q*K - 1 taps do not fit the shared-memory tile");
	*Q_out = Q;
	return TSDRGPU_OK;
}

inline uint64_t ceil_div(uint64_t a, uint64_t b) { return a / b + (a % b != 0); }

}  // namespace

struct tsdrgpu_channelizer {
	tsdrgpu_ctx_t *ctx;
	int configured;
	int K, Q, D, L;
	ChGeom geo;
	uint64_t pos;                             // absolute index of the next input pair
	float *d_taps; float2 *d_tw;
	float2 *d_hist[2]; int cur;
};

struct tsdrgpu_scan {
	tsdrgpu_ctx_t *ctx;
	tsdrgpu_channelizer *ch;
	int configured, K;
	uint32_t fs, rate, size;                  // channel rate, capture size
	int flen, llen;
	// the channels' magnitudes land in d_buf[cur] ([K][width]); a complete round is handed to the heavy stream there, and the rest
	// moves to the other buffer, which the heavy stream has finished with (ev_done)
	float *d_buf[2]; uint64_t width; int cur; uint64_t fill;
	uint64_t rounds;
	float *d_big; float2 *w0, *w1; double *d_plots; TsdrScanPeak *d_res;
	cudaStream_t s_heavy; cudaEvent_t ev_in, ev_done[2]; int pending[2];
};

extern "C" {

int tsdrgpu_channelizer_design(uint32_t fs, int channels, int taps_per_channel, float *taps, int cap, int *ntaps_out) {
	int Q = 0;
	int rc = ch_validate(NULL, fs, channels, taps_per_channel, &Q);
	if (rc) return rc;
	const int n = Q * channels - 1;
	if (ntaps_out) *ntaps_out = n;
	if (taps) {
		if (cap < n) return tsdrgpu_fail(NULL, TSDRGPU_ECAPACITY, "channelizer: the taps buffer is smaller than Q*K - 1", cudaSuccess, __FILE__, __LINE__);
		tsdrgpu_kaiser_lowpass_internal(fs, (double) fs / channels, n, taps);
	}
	return TSDRGPU_OK;
}

int tsdrgpu_channelizer_out_pairs(uint64_t position, uint64_t pairs, uint64_t dropped, int channels, uint64_t *out_pairs, uint64_t *out_dropped) {
	if (channels < CH_MIN_K || channels > CH_MAX_K || (channels & (channels - 1)) != 0) return ch_bad(NULL, "channelizer: channels must be a power of two in 2..256");
	const uint64_t D = (uint64_t) channels / 2, b0 = position + dropped;
	if (out_dropped) *out_dropped = ceil_div(b0, D) - ceil_div(position, D);
	if (out_pairs) *out_pairs = ceil_div(b0 + pairs, D) - ceil_div(b0, D);
	return TSDRGPU_OK;
}

int tsdrgpu_channelizer_create(tsdrgpu_ctx_t *ctx, tsdrgpu_channelizer_t **out) {
	BIND(ctx); ARG_TRY(ctx, out != NULL);
	tsdrgpu_channelizer *c = new tsdrgpu_channelizer();
	memset(c, 0, sizeof *c);
	c->ctx = ctx;
	*out = c;
	return TSDRGPU_OK;
}

void tsdrgpu_channelizer_destroy(tsdrgpu_channelizer_t *c) {
	if (!c) return;
	cudaSetDevice(c->ctx->device);
	if (c->d_taps) cudaFree(c->d_taps);
	if (c->d_tw) cudaFree(c->d_tw);
	for (int i = 0; i < 2; i++) if (c->d_hist[i]) cudaFree(c->d_hist[i]);
	delete c;
}

int tsdrgpu_channelizer_reset(tsdrgpu_channelizer_t *c, void *stream) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, c != NULL);
	tsdrgpu_ctx_t *ctx = c->ctx;
	BIND(ctx);
	ARG_TRY(ctx, c->configured);
	c->pos = 0; c->cur = 0;
	CU_TRY(ctx, cudaMemsetAsync(c->d_hist[0], 0, sizeof(float2) * (size_t) c->L, (cudaStream_t) stream));
	return TSDRGPU_OK;
}

int tsdrgpu_channelizer_configure(tsdrgpu_channelizer_t *c, uint32_t fs, int channels, int taps_per_channel) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, c != NULL);
	tsdrgpu_ctx_t *ctx = c->ctx;
	BIND(ctx);
	int Q = 0;
	int rc = ch_validate(ctx, fs, channels, taps_per_channel, &Q);
	if (rc) return rc;
	const int K = channels, n = Q * K - 1;
	const ChGeom g = ch_pick(K, Q);
	std::vector<float> h((size_t) n), poly((size_t) g.Qp * K, 0.0f);
	tsdrgpu_kaiser_lowpass_internal(fs, (double) fs / K, n, h.data());
	for (int i = 0; i < n; i++) poly[i] = h[i];                   // taps[q K + rho] = h[q K + rho]: the natural order
	std::vector<float2> tw((size_t) K / 2);
	for (int j = 0; j < K / 2; j++) { const double a = 2.0 * M_PI * j / K; tw[j] = make_float2((float) cos(a), (float) sin(a)); }
	CU_TRY(ctx, cudaDeviceSynchronize());                          // a reconfiguration is not on the hot path
	if (c->d_taps) { CU_TRY(ctx, cudaFree(c->d_taps)); c->d_taps = NULL; }
	if (c->d_tw) { CU_TRY(ctx, cudaFree(c->d_tw)); c->d_tw = NULL; }
	for (int i = 0; i < 2; i++) if (c->d_hist[i]) { CU_TRY(ctx, cudaFree(c->d_hist[i])); c->d_hist[i] = NULL; }
	CU_TRY(ctx, cudaMalloc(&c->d_taps, sizeof(float) * poly.size()));
	CU_TRY(ctx, cudaMemcpy(c->d_taps, poly.data(), sizeof(float) * poly.size(), cudaMemcpyHostToDevice));
	CU_TRY(ctx, cudaMalloc(&c->d_tw, sizeof(float2) * tw.size()));
	CU_TRY(ctx, cudaMemcpy(c->d_tw, tw.data(), sizeof(float2) * tw.size(), cudaMemcpyHostToDevice));
	c->K = K; c->Q = Q; c->D = K / 2; c->L = Q * K - 2; c->geo = g;
	for (int i = 0; i < 2; i++) CU_TRY(ctx, cudaMalloc(&c->d_hist[i], sizeof(float2) * (size_t) c->L));
	CU_TRY(ctx, cudaFuncSetAttribute(channelizer_pfb, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) CH_SMEM_MAX));
	c->configured = 1;
	return tsdrgpu_channelizer_reset(c, NULL) == TSDRGPU_OK ? (cudaDeviceSynchronize() == cudaSuccess ? TSDRGPU_OK : TSDRGPU_ECUDA) : TSDRGPU_ECUDA;
}

int tsdrgpu_channelizer_run(tsdrgpu_channelizer_t *c, void *stream, const float *d_iq, uint64_t pairs, uint64_t dropped_before, int mode,
                            float *d_out, uint64_t channel_stride, uint64_t *out_pairs, uint64_t *out_dropped) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, c != NULL);
	tsdrgpu_ctx_t *ctx = c->ctx;
	BIND(ctx);
	ARG_TRY(ctx, c->configured);
	ARG_TRY(ctx, mode == TSDRGPU_CHANNELIZER_COMPLEX || mode == TSDRGPU_CHANNELIZER_MAGNITUDE);
	ARG_TRY(ctx, pairs == 0 || d_iq != NULL);
	uint64_t M = 0, Md = 0;
	tsdrgpu_channelizer_out_pairs(c->pos, pairs, dropped_before, c->K, &M, &Md);
	ARG_TRY(ctx, M == 0 || (d_out != NULL && channel_stride >= M));
	cudaStream_t s = (cudaStream_t) stream;
	ChArgs a;
	a.in = reinterpret_cast<const float2 *>(d_iq); a.hist = c->d_hist[c->cur]; a.out = d_out; a.taps = c->d_taps; a.tw = c->d_tw;
	a.p = (long long) c->pos; a.g = (long long) dropped_before; a.k = (long long) pairs;
	a.m_first = (long long) ceil_div(c->pos + dropped_before, (uint64_t) c->D); a.M = (long long) M; a.stride = (long long) channel_stride;
	a.K = c->K; a.logK = __builtin_ctz((unsigned) c->K); a.D = c->D; a.L = c->L; a.Q = c->Q; a.Qp = c->geo.Qp; a.NP = c->geo.NP;
	a.U = c->geo.U; a.P = c->geo.P; a.mag = mode == TSDRGPU_CHANNELIZER_MAGNITUDE;
	if (M > 0) {
		const uint64_t T = (uint64_t) c->geo.NP * c->geo.O;
		const unsigned long long grid = (M + T - 1) / T;
		ARG_TRY(ctx, grid < (1ull << 31));
		KL(ctx, "channelizer_pfb", s, channelizer_pfb<<<(unsigned) grid, c->geo.NT, c->geo.smem, s>>>(a));
	}
	if (pairs > 0 || dropped_before > 0) {                           // the history moves on, also over an empty block's gap
		KL(ctx, "channelizer_history", s, channelizer_history<<<(unsigned) ((c->L + 255) / 256), 256, 0, s>>>(a, c->d_hist[c->cur ^ 1]));
		c->cur ^= 1;
	}
	c->pos += dropped_before + pairs;
	if (out_pairs) *out_pairs = M;
	if (out_dropped) *out_dropped = Md;
	return TSDRGPU_OK;
}

// ---- scan ------------------------------------------------------------------------------------------------------------
static void scan_free(tsdrgpu_scan *s) {
	for (int i = 0; i < 2; i++) if (s->d_buf[i]) { cudaFree(s->d_buf[i]); s->d_buf[i] = NULL; }
	void *bufs[] = {s->d_big, s->w0, s->w1, s->d_plots, s->d_res};
	for (void *b : bufs) if (b) cudaFree(b);
	s->d_big = NULL; s->w0 = s->w1 = NULL; s->d_plots = NULL; s->d_res = NULL; s->width = 0;
}

int tsdrgpu_scan_create(tsdrgpu_ctx_t *ctx, tsdrgpu_scan_t **out) {
	BIND(ctx); ARG_TRY(ctx, out != NULL);
	tsdrgpu_scan *s = new tsdrgpu_scan();
	memset(s, 0, sizeof *s);
	s->ctx = ctx;
	int rc = tsdrgpu_channelizer_create(ctx, &s->ch);
	if (rc) { delete s; return rc; }
	// background work like the frame-rate detector's: lowest priority, so the pixel path gets free SM resources first
	int lo = 0, hi = 0;
	CU_TRY(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));
	CU_TRY(ctx, cudaStreamCreateWithPriority(&s->s_heavy, cudaStreamNonBlocking, lo));
	CU_TRY(ctx, cudaEventCreateWithFlags(&s->ev_in, cudaEventDisableTiming));
	for (int i = 0; i < 2; i++) CU_TRY(ctx, cudaEventCreateWithFlags(&s->ev_done[i], cudaEventDisableTiming));
	*out = s;
	return TSDRGPU_OK;
}

void tsdrgpu_scan_destroy(tsdrgpu_scan_t *s) {
	if (!s) return;
	cudaSetDevice(s->ctx->device);
	cudaStreamSynchronize(s->s_heavy);
	scan_free(s);
	tsdrgpu_channelizer_destroy(s->ch);
	cudaStreamDestroy(s->s_heavy); cudaEventDestroy(s->ev_in); cudaEventDestroy(s->ev_done[0]); cudaEventDestroy(s->ev_done[1]);
	delete s;
}

int tsdrgpu_scan_reset(tsdrgpu_scan_t *s, void *stream) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, s != NULL);
	tsdrgpu_ctx_t *ctx = s->ctx;
	BIND(ctx);
	ARG_TRY(ctx, s->configured);
	cudaStream_t st = (cudaStream_t) stream;
	CU_TRY(ctx, cudaStreamSynchronize(s->s_heavy));
	s->pending[0] = s->pending[1] = 0; s->cur = 0; s->fill = 0; s->rounds = 0;
	int rc = tsdrgpu_channelizer_reset(s->ch, stream);
	if (rc) return rc;
	CU_TRY(ctx, cudaMemsetAsync(s->d_plots, 0, sizeof(double) * (size_t) s->K * (size_t) (s->flen + s->llen), st));
	CU_TRY(ctx, cudaMemsetAsync(s->d_res, 0, sizeof(TsdrScanPeak) * 2 * (size_t) s->K, st));
	return TSDRGPU_OK;
}

int tsdrgpu_scan_configure(tsdrgpu_scan_t *s, uint32_t fs, int channels, int taps_per_channel) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, s != NULL);
	tsdrgpu_ctx_t *ctx = s->ctx;
	BIND(ctx);
	int rc = tsdrgpu_channelizer_configure(s->ch, fs, channels, taps_per_channel);
	if (rc) return rc;
	CU_TRY(ctx, cudaStreamSynchronize(s->s_heavy));
	scan_free(s);
	const int K = channels;
	s->K = K; s->fs = fs; s->rate = (uint32_t) (2ull * fs / (uint64_t) K); s->size = tsdrgpu_frd_capture_size(s->rate);
	int fmin, fmax, lmin, lmax;
	tsdrgpu_frd_windows(s->rate, &fmin, &fmax, &lmin, &lmax);
	s->flen = fmax - fmin; s->llen = lmax - lmin;
	const size_t N = tsdrgpu_fft_getrealsize(s->size);
	CU_TRY(ctx, cudaMalloc(&s->d_big, sizeof(float) * 2 * (size_t) s->size * K));
	CU_TRY(ctx, cudaMalloc(&s->w0, sizeof(float2) * N * K));                 // the work buffers of the batched autocorrelation
	CU_TRY(ctx, cudaMalloc(&s->w1, sizeof(float2) * ((N / 2) * K + 16)));
	CU_TRY(ctx, cudaMalloc(&s->d_plots, sizeof(double) * (size_t) K * (size_t) (s->flen + s->llen)));
	CU_TRY(ctx, cudaMalloc(&s->d_res, sizeof(TsdrScanPeak) * 2 * (size_t) K));
	s->configured = 1;
	if ((rc = tsdrgpu_scan_reset(s, NULL))) return rc;
	CU_TRY(ctx, cudaDeviceSynchronize());
	return TSDRGPU_OK;
}

int tsdrgpu_scan_run(tsdrgpu_scan_t *s, void *stream, const float *d_iq, uint64_t pairs, uint64_t dropped_before) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, s != NULL);
	tsdrgpu_ctx_t *ctx = s->ctx;
	BIND(ctx);
	ARG_TRY(ctx, s->configured);
	cudaStream_t st = (cudaStream_t) stream;
	const int K = s->K;
	uint64_t M = 0;
	tsdrgpu_channelizer_out_pairs(s->ch->pos, pairs, dropped_before, K, &M, NULL);
	if (dropped_before > 0) s->fill = 0;                           // a drop discards every channel's partial capture
	if (s->width < s->fill + M) {                                  // grow both buffers, keeping what the current one holds
		const uint64_t wnew = (s->fill + M > s->size ? s->fill + M : s->size) * 3 / 2 + 16;
		CU_TRY(ctx, cudaStreamSynchronize(st)); CU_TRY(ctx, cudaStreamSynchronize(s->s_heavy));
		s->pending[0] = s->pending[1] = 0;
		float *nb[2] = {NULL, NULL};
		for (int i = 0; i < 2; i++) CU_TRY(ctx, cudaMalloc(&nb[i], sizeof(float) * (size_t) wnew * K));
		if (s->fill) CU_TRY(ctx, cudaMemcpy2D(nb[s->cur], sizeof(float) * wnew, s->d_buf[s->cur], sizeof(float) * s->width, sizeof(float) * s->fill, K, cudaMemcpyDeviceToDevice));
		for (int i = 0; i < 2; i++) { if (s->d_buf[i]) CU_TRY(ctx, cudaFree(s->d_buf[i])); s->d_buf[i] = nb[i]; }
		s->width = wnew;
	}
	if (s->pending[s->cur]) CU_TRY(ctx, cudaStreamWaitEvent(st, s->ev_done[s->cur], 0));   // the heavy stream is done with this buffer
	int rc = tsdrgpu_channelizer_run(s->ch, stream, d_iq, pairs, dropped_before, TSDRGPU_CHANNELIZER_MAGNITUDE, s->d_buf[s->cur] + s->fill,
	                                 s->width, NULL, NULL);
	if (rc) return rc;
	s->fill += M;
	if (s->fill < s->size) return TSDRGPU_OK;
	// complete rounds: the autocorrelations and running means go to the heavy stream, behind what `stream` holds now
	const uint64_t nr = s->fill / s->size, rest = s->fill - nr * s->size;
	float *buf = s->d_buf[s->cur];
	CU_TRY(ctx, cudaEventRecord(s->ev_in, st));
	CU_TRY(ctx, cudaStreamWaitEvent(s->s_heavy, s->ev_in, 0));
	for (uint64_t r = 0; r < nr; r++) {
		s->rounds++;
		if ((rc = tsdrgpu_scan_round_internal(ctx, s->s_heavy, buf + r * s->size, s->width, s->size, (unsigned) K, s->rate, s->d_big, s->w0, s->w1,
		                                      s->d_plots, s->rounds, s->d_res))) return rc;
	}
	CU_TRY(ctx, cudaEventRecord(s->ev_done[s->cur], s->s_heavy));
	s->pending[s->cur] = 1;
	const int nxt = s->cur ^ 1;
	if (rest) {
		if (s->pending[nxt]) CU_TRY(ctx, cudaStreamWaitEvent(st, s->ev_done[nxt], 0));
		CU_TRY(ctx, cudaMemcpy2DAsync(s->d_buf[nxt], sizeof(float) * s->width, buf + nr * s->size, sizeof(float) * s->width, sizeof(float) * rest, K,
		                              cudaMemcpyDeviceToDevice, st));
	}
	s->cur = nxt; s->fill = rest;
	return TSDRGPU_OK;
}

int tsdrgpu_scan_results(tsdrgpu_scan_t *s, void *stream, tsdrgpu_scan_channel_t *h_out, int cap) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, s != NULL);
	tsdrgpu_ctx_t *ctx = s->ctx;
	BIND(ctx);
	ARG_TRY(ctx, s->configured && (h_out != NULL || cap <= 0));
	const int K = s->K;
	std::vector<TsdrScanPeak> r((size_t) 2 * K);
	CU_TRY(ctx, cudaStreamSynchronize((cudaStream_t) stream));
	CU_TRY(ctx, cudaStreamSynchronize(s->s_heavy));
	CU_TRY(ctx, cudaMemcpy(r.data(), s->d_res, sizeof(TsdrScanPeak) * r.size(), cudaMemcpyDeviceToHost));
	int fmin, fmax, lmin, lmax;
	tsdrgpu_frd_windows(s->rate, &fmin, &fmax, &lmin, &lmax);
	for (int c = 0; c < K && c < cap; c++) {
		tsdrgpu_scan_channel_t &o = h_out[c];
		memset(&o, 0, sizeof o);
		o.offset_hz = (double) (c < K / 2 ? c : c - K) * (double) s->fs / K;
		o.rate = s->rate; o.captures = s->rounds;
		o.frame_index = r[2 * c].index; o.line_index = r[2 * c + 1].index;
		o.frame_score = r[2 * c].score; o.line_score = r[2 * c + 1].score;
		if (s->rounds) tsdrgpu_videomode_from_peaks(fmin, o.frame_index, lmin, o.line_index, s->rate, &o.fps, &o.height);
	}
	return TSDRGPU_OK;
}

int tsdrgpu_scan_plots(tsdrgpu_scan_t *s, void *stream, double *h_plots, uint64_t cap, int *frame_len, int *line_len) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, s != NULL);
	tsdrgpu_ctx_t *ctx = s->ctx;
	BIND(ctx);
	ARG_TRY(ctx, s->configured);
	if (frame_len) *frame_len = s->flen;
	if (line_len) *line_len = s->llen;
	const uint64_t n = (uint64_t) s->K * (uint64_t) (s->flen + s->llen);
	CU_TRY(ctx, cudaStreamSynchronize((cudaStream_t) stream));
	CU_TRY(ctx, cudaStreamSynchronize(s->s_heavy));
	if (h_plots) CU_TRY(ctx, cudaMemcpy(h_plots, s->d_plots, sizeof(double) * (size_t) (n < cap ? n : cap), cudaMemcpyDeviceToHost));
	return TSDRGPU_OK;
}

}  // extern "C"
