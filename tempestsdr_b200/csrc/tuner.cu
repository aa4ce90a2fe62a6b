// tuner.cu -- digital down-converter (the "tuner") ahead of the pixel path: shift a sub-band of the capture to 0 Hz,
// low-pass it and keep every D-th sample.  Nothing in the reference does this (it demodulates the whole band the front end
// delivers), so this file is tolerance-based like fft.cu: FMA contraction is allowed, every sum is written with explicit
// __fmaf_rn in one fixed order so that the bits do not depend on how the stream is cut into blocks.
//
// Definition (DESIGN.md section 5.6).  Input pair n (absolute index since the last reset, dropped pairs counted) is mixed by
// e^{-2 pi i offset n / fs}; the phase is the 64-bit integer n * inc mod 2^64, inc = round(offset / fs * 2^64), so a sample's
// rotation depends on its index only.  Output m is z[m] = sum_k h[k] x~[mD - k] with x~ the mixed input, zeros before the first
// sample and over every drop.  One output per absolute index n == 0 (mod D) that is inside a block.
//
// Kernel shape: one CTA per tile of T consecutive outputs.  The tile's input span ((T-1) D + ntaps pairs: the previous blocks'
// last ntaps-1 mixed samples come from a device-side history) is loaded from HBM, rotated, and written to shared memory
// de-interleaved by D (row r holds span samples i == r mod D), each row padded by one pair every R columns.  A thread owns R
// consecutive outputs and runs the polyphase form of the FIR: for every phase rho, the outputs' samples for tap q + 1 are the
// samples for tap q shifted by one output, so a register window of R samples slides down the row by one shared-memory load per
// tap, and every tap (a broadcast) and every sample feed 2R FMAs.  The padding makes the lanes' addresses (R+1 pairs apart)
// conflict-free.  No tensor cores: a real FIR against complex data is 2 FMAs per tap and sample, there is no matrix product
// to map onto them.
#include "common.cuh"
#include <math.h>

namespace {

constexpr int TN_THREADS = 256;
constexpr int TN_SPAN_MAX = 12288;                 // staged input pairs per CTA at most (96 KB before padding)
constexpr int TN_MAX_TAPS = 1023, TN_MAX_D = 64;
constexpr double TN_KAISER_BETA = 0.1102 * (80.0 - 8.7);   // Kaiser's rule for 80 dB stop-band attenuation

struct TnArgs {
	const float2 *in;          // this block's k input pairs
	const float2 *hist;        // x~[p - L .. p - 1]
	float2 *out;
	const float *taps;         // polyphase: taps[rho * Qp + q] = h[q D + rho], zero past ntaps
	long long p, g, k;         // position before the gap, gap, pairs in the block
	long long m_first, M;      // first output index, outputs of this run
	unsigned long long inc;
	int D, L, Qp, T, nrho;     // L = ntaps - 1; nrho = min(D, ntaps) phases that have taps
	int U, P;                  // columns per de-interleaved row, row pitch (pairs, padding included)
	float invD;
};

// v * e^{-i pi x}, x = phase / 2^63 from the top 32 bits of the phase (half-turns in [-1, 1))
__device__ __forceinline__ float2 tn_rotate(float2 v, long long n, unsigned long long inc) {
	const unsigned long long ph = (unsigned long long) n * inc;
	const float x = (float) (int) (unsigned) (ph >> 32) * 4.656612873077393e-10f;      // * 2^-31, exact
	float s, c;
	sincospif(x, &s, &c);
	return make_float2(__fmaf_rn(v.x, c, __fmul_rn(v.y, s)), __fmaf_rn(v.y, c, -__fmul_rn(v.x, s)));
}

// x~[n] before rotation: block samples raw (the caller rotates them), the gap and the time before the stream as zeros,
// older samples from the history (already mixed)
__device__ __forceinline__ float2 tn_load(const TnArgs &a, long long n) {
	const long long b0 = a.p + a.g;
	if (n >= b0) return ldg_stream_f2(a.in + (n - b0));
	if (n >= a.p || n < a.p - a.L) return make_float2(0.f, 0.f);
	return a.hist[n - (a.p - a.L)];
}

template <int R>
__device__ __forceinline__ int tn_col(int u) { return R >= 2 ? u + u / R : u; }      // padded column (R is a power of two)

template <int R>
__global__ void __launch_bounds__(TN_THREADS) tuner_fir(TnArgs a) {
	extern __shared__ __align__(16) float tn_smem[];
	const int ntp = a.D * a.Qp;
	float *s_taps = tn_smem;
	float2 *s_x = reinterpret_cast<float2 *>(tn_smem + ((ntp + 3) & ~3));
	const int tid = threadIdx.x;
	const long long t0 = (long long) blockIdx.x * a.T;                // the tile's first output, relative to m_first
	const int T = (int) ((a.M - t0) < a.T ? (a.M - t0) : a.T);
	const int S = (T - 1) * a.D + a.L + 1;
	const long long base = (a.m_first + t0) * a.D - a.L;              // absolute index of span sample 0
	const long long b0 = a.p + a.g;
	for (int i = tid; i < ntp; i += TN_THREADS) s_taps[i] = a.taps[i];
	// stage the span: four independent loads in flight per thread, then rotate and scatter into the de-interleaved rows
	for (int i0 = tid; i0 < S; i0 += 4 * TN_THREADS) {
		float2 v[4];
		#pragma unroll
		for (int j = 0; j < 4; j++) { const int i = i0 + j * TN_THREADS; v[j] = i < S ? tn_load(a, base + i) : make_float2(0.f, 0.f); }
		#pragma unroll
		for (int j = 0; j < 4; j++) {
			const int i = i0 + j * TN_THREADS;
			if (i >= S) break;
			const long long n = base + i;
			const float2 w = n >= b0 ? tn_rotate(v[j], n, a.inc) : v[j];
			const int u = (int) (((float) i + 0.5f) * a.invD), r = i - u * a.D;      // exact: S <= TN_SPAN_MAX keeps the float error below 0.5 / D
			s_x[r * a.P + tn_col<R>(u)] = w;
		}
	}
	__syncthreads();
	const int ml0 = tid * R;
	if (ml0 >= T) return;
	float2 acc[R];
	#pragma unroll
	for (int r = 0; r < R; r++) acc[r] = make_float2(0.f, 0.f);
	for (int rho = 0; rho < a.nrho; rho++) {
		const float *hp = s_taps + rho * a.Qp;
		const int c = a.L - rho;                                      // >= 0: phases past ntaps - 1 have no taps
		const float2 *row = s_x + (c % a.D) * a.P;
		const int u0 = ml0 + c / a.D;                                 // column of output ml0's sample for tap q = 0
		float2 w[R];
		#pragma unroll
		for (int r = 0; r < R; r++) w[r] = row[tn_col<R>(min(u0 + r, a.U - 1))];     // clamped: only outputs past T read there
		int nxt = u0 - 1;
		for (int q0 = 0; q0 < a.Qp; q0 += R) {
			#pragma unroll
			for (int u = 0; u < R; u++) {
				const float t = hp[q0 + u];
				#pragma unroll
				for (int r = 0; r < R; r++) {
					const float2 v = w[(r - u + R) % R];
					acc[r].x = __fmaf_rn(t, v.x, acc[r].x);
					acc[r].y = __fmaf_rn(t, v.y, acc[r].y);
				}
				w[(2 * R - 1 - u) % R] = row[tn_col<R>(max(nxt, 0))];   // the window slides by one output; past column 0 only zero taps follow
				nxt--;
			}
		}
	}
	float2 *o = a.out + t0 + ml0;
	#pragma unroll
	for (int r = 0; r < R; r++) if (ml0 + r < T) o[r] = acc[r];
}

// the history after this block: x~[p + g + k - L .. p + g + k - 1], from the old history, the gap's zeros and the block
__global__ void __launch_bounds__(256) tuner_history(TnArgs a, float2 *hist_new) {
	const int j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= a.L) return;
	const long long n = a.p + a.g + a.k - a.L + j;
	const float2 v = tn_load(a, n);
	hist_new[j] = n >= a.p + a.g ? tn_rotate(v, n, a.inc) : v;
}

inline int tn_bad(tsdrgpu_ctx_t *ctx, const char *what) { return tsdrgpu_fail(ctx, TSDRGPU_EINVAL, what, cudaSuccess, __FILE__, __LINE__); }

double bessel_i0(double x) {                                          // power series, converges fast for the betas used here
	double sum = 1.0, term = 1.0;
	const double q = 0.25 * x * x;
	for (int k = 1; k < 500; k++) {
		term *= q / ((double) k * (double) k);
		sum += term;
		if (term < 1e-17 * sum) break;
	}
	return sum;
}

}  // namespace

// scipy.signal.firwin(n, bandwidth / 2, window=('kaiser', beta), fs=fs): windowed sinc for 80 dB, designed in double and scaled to
// unit DC gain.  The tuner and the channelizer store it as float32 (tsdrgpu_kaiser_lowpass_internal), the notch builds on the
// doubles; each checks its own limits on n.
void tsdrgpu_kaiser_lowpass_double_internal(uint32_t fs, double bandwidth_hz, int n, double *taps) {
	const double cut = bandwidth_hz / (double) fs, alpha = 0.5 * (double) (n - 1), i0b = bessel_i0(TN_KAISER_BETA);
	double sum = 0.0;
	for (int i = 0; i < n; i++) {
		const double m = (double) i - alpha, xm = cut * m;
		const double sinc = xm == 0.0 ? 1.0 : sin(M_PI * xm) / (M_PI * xm);
		const double rr = m / alpha, win = bessel_i0(TN_KAISER_BETA * sqrt(fmax(0.0, 1.0 - rr * rr))) / i0b;
		taps[i] = cut * sinc * win;
		sum += taps[i];
	}
	for (int i = 0; i < n; i++) taps[i] /= sum;
}

void tsdrgpu_kaiser_lowpass_internal(uint32_t fs, double bandwidth_hz, int n, float *taps) {
	std::vector<double> h((size_t) n);
	tsdrgpu_kaiser_lowpass_double_internal(fs, bandwidth_hz, n, h.data());
	for (int i = 0; i < n; i++) taps[i] = (float) h[i];
}

namespace {

// validation + filter design shared by tsdrgpu_tuner_design and the tuner object (errors into ctx, or the thread's text)
int tn_design(tsdrgpu_ctx_t *ctx, uint32_t fs, double offset_hz, double bandwidth_hz, int decimation, int ntaps, float *taps, int cap,
              int *ntaps_out, uint64_t *phase_inc) {
	if (decimation < 1 || decimation > TN_MAX_D) return tn_bad(ctx, "tuner: decimation must be an integer in 1..64");
	if (ntaps != 0 && (ntaps < 3 || ntaps > TN_MAX_TAPS || (ntaps & 1) == 0)) return tn_bad(ctx, "tuner: ntaps must be odd, in 3..1023 (0 = default)");
	if (fs == 0) return tn_bad(ctx, "tuner: the sample rate must be > 0");
	if (!(bandwidth_hz > 0.0) || !isfinite(bandwidth_hz)) return tn_bad(ctx, "tuner: bandwidth_hz must be > 0");
	if (!isfinite(offset_hz)) return tn_bad(ctx, "tuner: offset_hz must be finite");
	if (fs % (uint32_t) decimation != 0) return tn_bad(ctx, "tuner: the sample rate must be a multiple of the decimation (fs % D == 0)");
	if (bandwidth_hz > (double) (fs / (uint32_t) decimation)) return tn_bad(ctx, "tuner: bandwidth_hz must not exceed the decimated rate (bandwidth <= fs / D)");
	if (fabs(offset_hz) + 0.5 * bandwidth_hz > 0.5 * (double) fs) return tn_bad(ctx, "tuner: the band must lie inside the capture (|offset| + bandwidth / 2 <= fs / 2)");
	int n = ntaps;
	if (n == 0) {                                                     // 16 taps per unit of fs / bandwidth, plus the centre tap
		const double r = ceil((double) fs / bandwidth_hz);
		n = r >= 63.0 ? TN_MAX_TAPS : 16 * (int) r + 1;
	}
	if (ntaps_out) *ntaps_out = n;
	if (taps) {
		if (cap < n) return tsdrgpu_fail(ctx, TSDRGPU_ECAPACITY, "tuner: the taps buffer is smaller than ntaps", cudaSuccess, __FILE__, __LINE__);
		tsdrgpu_kaiser_lowpass_internal(fs, bandwidth_hz, n, taps);
	}
	if (phase_inc) {                                                  // round(offset / fs * 2^64), two's complement
		long double v = rintl((long double) offset_hz * 18446744073709551616.0L / (long double) fs);
		if (v >= 9223372036854775808.0L) v -= 18446744073709551616.0L;
		*phase_inc = (uint64_t) (int64_t) v;
	}
	return TSDRGPU_OK;
}

}  // namespace

struct tsdrgpu_tuner {
	tsdrgpu_ctx_t *ctx;
	int configured;
	int D, ntaps, L, R, Qp, T, U, P, nrho;
	size_t smem;
	uint64_t inc, pos;                        // pos: absolute index of the next input pair
	float *d_taps;                            // polyphase layout (TnArgs::taps)
	float2 *d_hist[2]; int cur;
};

extern "C" {

int tsdrgpu_tuner_design(uint32_t fs, double offset_hz, double bandwidth_hz, int decimation, int ntaps, float *taps, int cap,
                         int *ntaps_out, uint64_t *phase_inc) {
	return tn_design(NULL, fs, offset_hz, bandwidth_hz, decimation, ntaps, taps, cap, ntaps_out, phase_inc);
}

static inline uint64_t ceil_div(uint64_t a, uint64_t b) { return a / b + (a % b != 0); }

int tsdrgpu_tuner_out_pairs(uint64_t position, uint64_t pairs, uint64_t dropped, int decimation, uint64_t *out_pairs, uint64_t *out_dropped) {
	if (decimation < 1 || decimation > TN_MAX_D) return tn_bad(NULL, "tuner: decimation must be an integer in 1..64");
	const uint64_t D = (uint64_t) decimation, b0 = position + dropped;
	if (out_dropped) *out_dropped = ceil_div(b0, D) - ceil_div(position, D);
	if (out_pairs) *out_pairs = ceil_div(b0 + pairs, D) - ceil_div(b0, D);
	return TSDRGPU_OK;
}

int tsdrgpu_tuner_create(tsdrgpu_ctx_t *ctx, tsdrgpu_tuner_t **out) {
	BIND(ctx); ARG_TRY(ctx, out != NULL);
	tsdrgpu_tuner *t = new tsdrgpu_tuner();
	memset(t, 0, sizeof *t);
	t->ctx = ctx;
	*out = t;
	return TSDRGPU_OK;
}

void tsdrgpu_tuner_destroy(tsdrgpu_tuner_t *t) {
	if (!t) return;
	cudaSetDevice(t->ctx->device);
	if (t->d_taps) cudaFree(t->d_taps);
	for (int i = 0; i < 2; i++) if (t->d_hist[i]) cudaFree(t->d_hist[i]);
	delete t;
}

int tsdrgpu_tuner_reset(tsdrgpu_tuner_t *t, void *stream) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, t != NULL);
	tsdrgpu_ctx_t *ctx = t->ctx;
	BIND(ctx);
	ARG_TRY(ctx, t->configured);
	t->pos = 0; t->cur = 0;
	CU_TRY(ctx, cudaMemsetAsync(t->d_hist[0], 0, sizeof(float2) * (size_t) t->L, (cudaStream_t) stream));
	return TSDRGPU_OK;
}

int tsdrgpu_tuner_configure(tsdrgpu_tuner_t *t, uint32_t fs, double offset_hz, double bandwidth_hz, int decimation, int ntaps) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, t != NULL);
	tsdrgpu_ctx_t *ctx = t->ctx;
	BIND(ctx);
	float h[TN_MAX_TAPS];
	int n = 0; uint64_t inc = 0;
	int rc = tn_design(ctx, fs, offset_hz, bandwidth_hz, decimation, ntaps, h, TN_MAX_TAPS, &n, &inc);
	if (rc) return rc;
	const int D = decimation, L = n - 1;
	// tile: as many outputs as fit TN_SPAN_MAX staged pairs, at most 256 threads x R outputs; R as large as the tile allows
	const int Tfit = (TN_SPAN_MAX - L - 1) / D + 1;
	const int R = Tfit >= 1024 ? 8 : (Tfit >= 512 ? 4 : (Tfit >= 256 ? 2 : 1));
	const int T = Tfit < TN_THREADS * R ? Tfit : TN_THREADS * R;
	const int S = (T - 1) * D + L + 1;
	const int U = (S + D - 1) / D;
	const int P = U + (R >= 2 ? U / R : 0) + 1;
	const int Q = (n + D - 1) / D, Qp = (Q + R - 1) / R * R;
	const int nrho = D < n ? D : n;
	std::vector<float> poly((size_t) D * Qp, 0.0f);
	for (int rho = 0; rho < D; rho++)
		for (int q = 0; q < Qp; q++) if (q * D + rho < n) poly[(size_t) rho * Qp + q] = h[q * D + rho];
	CU_TRY(ctx, cudaDeviceSynchronize());                                  // a reconfiguration is not on the hot path
	if (t->d_taps) { CU_TRY(ctx, cudaFree(t->d_taps)); t->d_taps = NULL; }
	for (int i = 0; i < 2; i++) if (t->d_hist[i]) { CU_TRY(ctx, cudaFree(t->d_hist[i])); t->d_hist[i] = NULL; }
	CU_TRY(ctx, cudaMalloc(&t->d_taps, sizeof(float) * poly.size()));
	CU_TRY(ctx, cudaMemcpy(t->d_taps, poly.data(), sizeof(float) * poly.size(), cudaMemcpyHostToDevice));
	for (int i = 0; i < 2; i++) CU_TRY(ctx, cudaMalloc(&t->d_hist[i], sizeof(float2) * (size_t) L));
	t->D = D; t->ntaps = n; t->L = L; t->R = R; t->Qp = Qp; t->T = T; t->U = U; t->P = P; t->nrho = nrho; t->inc = inc;
	t->smem = sizeof(float) * (size_t) ((D * Qp + 3) & ~3) + sizeof(float2) * (size_t) D * P;
	static const size_t attr = 200 * 1024;
	CU_TRY(ctx, cudaFuncSetAttribute(tuner_fir<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) attr));
	CU_TRY(ctx, cudaFuncSetAttribute(tuner_fir<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) attr));
	CU_TRY(ctx, cudaFuncSetAttribute(tuner_fir<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) attr));
	CU_TRY(ctx, cudaFuncSetAttribute(tuner_fir<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) attr));
	if (t->smem > attr) return tsdrgpu_fail(ctx, TSDRGPU_EINVAL, "tuner: tile does not fit shared memory", cudaSuccess, __FILE__, __LINE__);
	t->configured = 1;
	return tsdrgpu_tuner_reset(t, NULL) == TSDRGPU_OK ? (cudaDeviceSynchronize() == cudaSuccess ? TSDRGPU_OK : TSDRGPU_ECUDA) : TSDRGPU_ECUDA;
}

int tsdrgpu_tuner_run(tsdrgpu_tuner_t *t, void *stream, const float *d_iq, uint64_t pairs, uint64_t dropped_before, float *d_out,
                      uint64_t *out_pairs, uint64_t *out_dropped) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, t != NULL);
	tsdrgpu_ctx_t *ctx = t->ctx;
	BIND(ctx);
	ARG_TRY(ctx, t->configured);
	ARG_TRY(ctx, pairs == 0 || d_iq != NULL);
	uint64_t M = 0, Md = 0;
	tsdrgpu_tuner_out_pairs(t->pos, pairs, dropped_before, t->D, &M, &Md);
	ARG_TRY(ctx, M == 0 || d_out != NULL);
	cudaStream_t s = (cudaStream_t) stream;
	TnArgs a;
	a.in = reinterpret_cast<const float2 *>(d_iq); a.hist = t->d_hist[t->cur]; a.out = reinterpret_cast<float2 *>(d_out); a.taps = t->d_taps;
	a.p = (long long) t->pos; a.g = (long long) dropped_before; a.k = (long long) pairs;
	a.m_first = (long long) ceil_div(t->pos + dropped_before, (uint64_t) t->D); a.M = (long long) M; a.inc = t->inc;
	a.D = t->D; a.L = t->L; a.Qp = t->Qp; a.T = t->T; a.nrho = t->nrho; a.U = t->U; a.P = t->P; a.invD = 1.0f / (float) t->D;
	if (M > 0) {
		const unsigned long long grid = (M + (uint64_t) t->T - 1) / (uint64_t) t->T;
		ARG_TRY(ctx, grid < (1ull << 31));
		switch (t->R) {
		case 8: KL(ctx, "tuner_fir", s, tuner_fir<8><<<(unsigned) grid, TN_THREADS, t->smem, s>>>(a)); break;
		case 4: KL(ctx, "tuner_fir", s, tuner_fir<4><<<(unsigned) grid, TN_THREADS, t->smem, s>>>(a)); break;
		case 2: KL(ctx, "tuner_fir", s, tuner_fir<2><<<(unsigned) grid, TN_THREADS, t->smem, s>>>(a)); break;
		default: KL(ctx, "tuner_fir", s, tuner_fir<1><<<(unsigned) grid, TN_THREADS, t->smem, s>>>(a)); break;
		}
	}
	if (pairs > 0 || dropped_before > 0) {                           // the history moves on, also over an empty block's gap
		KL(ctx, "tuner_history", s, tuner_history<<<(unsigned) ((t->L + 255) / 256), 256, 0, s>>>(a, t->d_hist[t->cur ^ 1]));
		t->cur ^= 1;
	}
	t->pos += dropped_before + pairs;
	if (out_pairs) *out_pairs = M;
	if (out_dropped) *out_dropped = Md;
	return TSDRGPU_OK;
}

}  // extern "C"
