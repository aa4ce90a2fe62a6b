// notch.cu -- notch filter (a list of stopbands removed from every block ahead of the pixel path) and the Welch power spectrum of
// the capture that shows where to put them.  Nothing in the reference does either, so this file is tolerance-based like tuner.cu:
// FMA contraction is allowed, and every result is computed by one fixed sequence of operations per output so that repeated runs
// give the same bits.
//
// Definition (DESIGN.md section 5.8).  Stopbands (f_j, w_j), j < J <= 32, L taps (odd),
//   h[n] = delta[n - (L-1)/2] - sum_j g_j[n] e^{2 pi i f_j (n - (L-1)/2) / fs},   g_j = firwin(L, w_j / 2, kaiser 7.857, fs)
// (the tuner's low-pass design), designed in double, stored as float32.  Output y[n] = sum_k h[k] x~[n - k] for every input pair n
// of a block, x~ = the input with zeros before the stream and over every drop, n counted since the last reset.
//
// Notch kernel: overlap-save with an N-point FFT, N = the smallest power of two >= 2 (L - 1) in 1024..16384, hop = N - (L - 1).
// Segment s produces outputs [s hop, (s+1) hop) from inputs [s hop - (L-1), (s+1) hop): one CTA loads those N pairs into shared
// memory (a device history supplies what earlier blocks held, zeros stand for drops, the time before the stream and everything past
// the block's end), runs a forward FFT, multiplies by H = FFT_N(h) / N and runs the inverse.  A block that ends inside a segment
// emits the outputs it has; the next block recomputes that segment and emits the rest.
//
// The FFT (nt_fft_dif / nt_fft_dit) is one in-place radix-2 transform of up to 16384 points in shared memory, twiddles from a table
// made in double on the host.  The forward transform is decimation in frequency (natural order in, bit-reversed out) and the
// inverse decimation in time (bit-reversed in, natural order out), so no pass reorders the data: H is stored bit-reversed, and the
// spectrum reads its bins through __brev.
#include "common.cuh"
#include <math.h>
#include <algorithm>
#include <complex>

namespace {

constexpr int NT_MAX_J = 32, NT_MIN_TAPS = 65, NT_MAX_TAPS = 8193, NT_MIN_N = 1024, NT_MAX_N = 16384;
constexpr int SP_MIN_N = 64, SP_MAX_N = 16384, SP_CHUNK = 1 << 22;    // spectrum: |X|^2 of at most SP_CHUNK bins per launch pair
constexpr double NT_DELTA_K = (80.0 - 7.95) / (2.285 * 2.0 * M_PI);  // Kaiser's transition width of the 80 dB design, per fs / (L - 1)

__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }

// forward transform, e^{-2 pi i jk / N}: natural order in, s[i] = X[brev(i)] out.  Ends with a barrier.
__device__ void nt_fft_dif(float2 *s, int logN, const float2 *__restrict__ tw) {
	const int half_n = 1 << (logN - 1);
	for (int lh = logN - 1; lh >= 0; lh--) {
		const int half = 1 << lh;
		for (int b = threadIdx.x; b < half_n; b += blockDim.x) {
			const int k = b & (half - 1), i0 = ((b >> lh) << (lh + 1)) + k;
			const float2 x0 = s[i0], x1 = s[i0 + half], w = __ldg(tw + (k << (logN - 1 - lh)));
			s[i0] = make_float2(x0.x + x1.x, x0.y + x1.y);
			s[i0 + half] = cmul(make_float2(x0.x - x1.x, x0.y - x1.y), w);
		}
		__syncthreads();
	}
}

// inverse transform without the 1/N, e^{+2 pi i jk / N}: s[i] = X[brev(i)] in, natural order out.  Ends with a barrier.
__device__ void nt_fft_dit(float2 *s, int logN, const float2 *__restrict__ tw) {
	const int half_n = 1 << (logN - 1);
	for (int lh = 0; lh < logN; lh++) {
		const int half = 1 << lh;
		for (int b = threadIdx.x; b < half_n; b += blockDim.x) {
			const int k = b & (half - 1), i0 = ((b >> lh) << (lh + 1)) + k;
			const float2 w = __ldg(tw + (k << (logN - 1 - lh)));
			const float2 x0 = s[i0], x1 = cmul(s[i0 + half], make_float2(w.x, -w.y));
			s[i0] = make_float2(x0.x + x1.x, x0.y + x1.y);
			s[i0 + half] = make_float2(x0.x - x1.x, x0.y - x1.y);
		}
		__syncthreads();
	}
}

// x~[n]: the block's samples, zeros over the gap, past the block's end and before the history, older samples from the history
struct StreamView {
	const float2 *in, *hist;
	long long p, g, k, hstart;          // position before the gap, gap, pairs in the block, absolute index of hist[0]
};
__device__ __forceinline__ float2 sv_load(const StreamView &v, long long n) {
	const long long b0 = v.p + v.g;
	if (n >= b0) return n - b0 < v.k ? ldg_stream_f2(v.in + (n - b0)) : make_float2(0.f, 0.f);
	if (n >= v.p || n < v.hstart) return make_float2(0.f, 0.f);
	return v.hist[n - v.hstart];
}

struct NtArgs {
	StreamView v;
	float2 *out;
	const float2 *H;                    // FFT_N(h) / N, bit-reversed order
	const float2 *tw;                   // e^{-2 pi i j / N}, j < N/2
	long long s0;                       // first segment of this run
	int logN, L1, hop;                  // L1 = L - 1
};

__global__ void __launch_bounds__(1024) notch_ols(NtArgs a) {
	extern __shared__ __align__(16) float2 nt_smem[];
	float2 *s = nt_smem;
	const int N = 1 << a.logN, NT = blockDim.x, tid = threadIdx.x;
	const long long seg = a.s0 + blockIdx.x, base = seg * a.hop - a.L1;
	for (int i0 = tid; i0 < N; i0 += 4 * NT) {                          // four independent loads in flight per thread
		float2 x[4];
		#pragma unroll
		for (int j = 0; j < 4; j++) { const int i = i0 + j * NT; x[j] = i < N ? sv_load(a.v, base + i) : make_float2(0.f, 0.f); }
		#pragma unroll
		for (int j = 0; j < 4; j++) { const int i = i0 + j * NT; if (i < N) s[i] = x[j]; }
	}
	__syncthreads();
	nt_fft_dif(s, a.logN, a.tw);
	for (int i = tid; i < N; i += NT) s[i] = cmul(s[i], __ldg(a.H + i));
	__syncthreads();
	nt_fft_dit(s, a.logN, a.tw);
	const long long b0 = a.v.p + a.v.g, lo = max(b0, seg * a.hop), hi = min(b0 + a.v.k, (seg + 1) * a.hop);
	for (long long n = lo + tid; n < hi; n += NT) a.out[n - b0] = s[n - base];
}

// the history after a block: x~[hstart_new .. hstart_new + len - 1]
__global__ void __launch_bounds__(256) stream_history(StreamView v, float2 *hist_new, long long hstart_new, int len) {
	const int j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j < len) hist_new[j] = sv_load(v, hstart_new + j);
}

// Welch: segment s_first + blockIdx.x covers [s nfft/2, s nfft/2 + nfft); its Hann-windowed transform's |X|^2 goes to row blockIdx.x
// of pw, bin order
__global__ void __launch_bounds__(1024) spectrum_segments(StreamView v, const float *__restrict__ win, const float2 *__restrict__ tw,
                                                          long long s_first, int logN, double *pw) {
	extern __shared__ __align__(16) float2 sp_smem[];
	float2 *s = sp_smem;
	const int N = 1 << logN, NT = blockDim.x, tid = threadIdx.x;
	const long long base = (s_first + blockIdx.x) * (long long) (N / 2);
	for (int i = tid; i < N; i += NT) {
		const float2 x = sv_load(v, base + i);
		const float w = __ldg(win + i);
		s[i] = make_float2(x.x * w, x.y * w);
	}
	__syncthreads();
	nt_fft_dif(s, logN, tw);
	double *row = pw + (size_t) blockIdx.x * N;
	for (int i = tid; i < N; i += NT) {
		const float2 X = s[i];
		row[__brev((unsigned) i) >> (32 - logN)] = __dadd_rn(__dmul_rn((double) X.x, (double) X.x), __dmul_rn((double) X.y, (double) X.y));
	}
}

// per-bin sums over the rows, in segment order (so the result does not depend on how the segments were grouped into launches)
__global__ void __launch_bounds__(256) spectrum_accumulate(const double *__restrict__ pw, int rows, int N, double *sum) {
	const int bin = blockIdx.x * blockDim.x + threadIdx.x;
	if (bin >= N) return;
	double acc = sum[bin];
	for (int r = 0; r < rows; r++) acc = __dadd_rn(acc, pw[(size_t) r * N + bin]);
	sum[bin] = acc;
}

inline int nt_bad(tsdrgpu_ctx_t *ctx, const char *what) { return tsdrgpu_fail(ctx, TSDRGPU_EINVAL, what, cudaSuccess, __FILE__, __LINE__); }
inline double nt_delta(uint32_t fs, int L) { return NT_DELTA_K * (double) fs / (double) (L - 1); }
inline int ilog2(int n) { return 31 - __builtin_clz((unsigned) n); }

int nt_fft_size(int L) {
	int N = NT_MIN_N;
	while (N < 2 * (L - 1)) N *= 2;
	return N;
}

// validation and the choice of L shared by tsdrgpu_notch_design and the notch object (errors into ctx, or the thread's text)
int nt_validate(tsdrgpu_ctx_t *ctx, uint32_t fs, int n, const double *centers, const double *widths, int ntaps, int *L_out) {
	if (n < 1 || n > NT_MAX_J) return nt_bad(ctx, "notch: the number of notches must be in 1..32");
	if (!centers || !widths) return nt_bad(ctx, "notch: centers and widths must not be NULL");
	if (fs == 0) return nt_bad(ctx, "notch: the sample rate must be > 0");
	if (ntaps != 0 && (ntaps < NT_MIN_TAPS || ntaps > NT_MAX_TAPS || (ntaps & 1) == 0)) return nt_bad(ctx, "notch: ntaps must be odd, in 65..8193 (0 = default)");
	double wmin = INFINITY;
	for (int j = 0; j < n; j++) {
		if (!isfinite(centers[j])) return nt_bad(ctx, "notch: every center must be finite");
		if (!(widths[j] > 0.0) || !isfinite(widths[j])) return nt_bad(ctx, "notch: every width must be > 0");
		if (fabs(centers[j]) + 0.5 * widths[j] > 0.5 * (double) fs) return nt_bad(ctx, "notch: every band must lie inside the capture (|center| + width / 2 <= fs / 2)");
		wmin = fmin(wmin, widths[j]);
	}
	int L = ntaps;
	if (L == 0) {                                                     // the smallest odd L with wmin >= 2 delta(L)
		const double need = 1.0 + 2.0 * NT_DELTA_K * (double) fs / wmin;
		if (need > (double) NT_MAX_TAPS) return nt_bad(ctx, "notch: the narrowest notch needs more than 8193 taps (width >= 2 delta(L)): widen it");
		L = std::max(NT_MIN_TAPS, (int) ceil(need) | 1);
		while (L <= NT_MAX_TAPS && wmin < 2.0 * nt_delta(fs, L)) L += 2;
		if (L > NT_MAX_TAPS) return nt_bad(ctx, "notch: the narrowest notch needs more than 8193 taps (width >= 2 delta(L)): widen it");
	}
	const double d = nt_delta(fs, L);
	for (int j = 0; j < n; j++)
		if (widths[j] < 2.0 * d) return nt_bad(ctx, "notch: every width must be at least twice the transition width (width >= 2 delta(L), delta(L) = (80 - 7.95) / (2.285 * 2 pi * (L - 1)) * fs)");
	if (n > 1) {
		std::vector<int> o((size_t) n);
		for (int j = 0; j < n; j++) o[j] = j;
		std::sort(o.begin(), o.end(), [&](int x, int y) { return centers[x] < centers[y]; });
		for (int i = 0; i < n; i++) {                                 // the last band's neighbour is the first one, across +-fs/2
			const int a = o[i], b = o[(i + 1) % n];
			const double upper = centers[a] + 0.5 * widths[a], lower = centers[b] - 0.5 * widths[b] + (i + 1 == n ? (double) fs : 0.0);
			if (lower - upper < d)
				return nt_bad(ctx, "notch: neighbouring notches must leave at least delta(L) between their edges (overlapping notches would remove more than the signal: merge them into one)");
		}
	}
	*L_out = L;
	return TSDRGPU_OK;
}

// h in double (L complex taps)
void nt_taps(uint32_t fs, int n, const double *centers, const double *widths, int L, std::vector<std::complex<double>> &h) {
	const int c = (L - 1) / 2;
	std::vector<double> g((size_t) L);
	h.assign((size_t) L, std::complex<double>(0.0, 0.0));
	h[c] = 1.0;
	for (int j = 0; j < n; j++) {
		tsdrgpu_kaiser_lowpass_double_internal(fs, widths[j], L, g.data());
		for (int i = 0; i < L; i++) {
			const double cyc = centers[j] * (double) (i - c) / (double) fs, ph = 2.0 * M_PI * (cyc - rint(cyc));
			h[i] -= g[i] * std::complex<double>(cos(ph), sin(ph));
		}
	}
}

// in-place forward DFT in double (radix 2, natural order in and out), for H on the host
void host_fft(std::vector<std::complex<double>> &x) {
	const size_t N = x.size();
	for (size_t i = 1, j = 0; i < N; i++) {
		size_t bit = N >> 1;
		for (; j & bit; bit >>= 1) j ^= bit;
		j ^= bit;
		if (i < j) std::swap(x[i], x[j]);
	}
	for (size_t m = 2; m <= N; m <<= 1)
		for (size_t i = 0; i < N; i += m)
			for (size_t k = 0; k < m / 2; k++) {
				const double a = -2.0 * M_PI * (double) k / (double) m;
				const std::complex<double> t = std::complex<double>(cos(a), sin(a)) * x[i + k + m / 2];
				x[i + k + m / 2] = x[i + k] - t;
				x[i + k] += t;
			}
}

std::vector<float2> twiddles(int N) {
	std::vector<float2> tw((size_t) N / 2);
	for (int j = 0; j < N / 2; j++) { const double a = -2.0 * M_PI * j / N; tw[j] = make_float2((float) cos(a), (float) sin(a)); }
	return tw;
}

inline unsigned brev_n(unsigned i, int logN) {
	unsigned r = 0;
	for (int b = 0; b < logN; b++) r |= ((i >> b) & 1u) << (logN - 1 - b);
	return r;
}

}  // namespace

struct tsdrgpu_notch {
	tsdrgpu_ctx_t *ctx;
	int configured;
	int L, N, logN, hop, NT;
	size_t smem;
	uint64_t pos;                             // absolute index of the next input pair
	long long hstart;                         // absolute index of the history's first pair
	float2 *d_H, *d_tw;
	float2 *d_hist[2]; int cur;
};

struct tsdrgpu_spectrum {
	tsdrgpu_ctx_t *ctx;
	int configured;
	uint32_t fs; int N, logN, NT;
	double wsum2;                             // sum of the window's squares
	uint64_t pos, seg_next, drop_end, segments;
	float *d_win; float2 *d_tw; double *d_sum, *d_pw;
	float2 *d_hist[2]; int cur;
};

extern "C" {

int tsdrgpu_notch_design(uint32_t fs, int n, const double *centers, const double *widths, int ntaps, float *taps, int cap, int *ntaps_out,
                         int *nfft_out) {
	int L = 0;
	int rc = nt_validate(NULL, fs, n, centers, widths, ntaps, &L);
	if (rc) return rc;
	if (ntaps_out) *ntaps_out = L;
	if (nfft_out) *nfft_out = nt_fft_size(L);
	if (taps) {
		if (cap < L) return tsdrgpu_fail(NULL, TSDRGPU_ECAPACITY, "notch: the taps buffer is smaller than ntaps", cudaSuccess, __FILE__, __LINE__);
		std::vector<std::complex<double>> h;
		nt_taps(fs, n, centers, widths, L, h);
		for (int i = 0; i < L; i++) { taps[2 * i] = (float) h[i].real(); taps[2 * i + 1] = (float) h[i].imag(); }
	}
	return TSDRGPU_OK;
}

int tsdrgpu_notch_create(tsdrgpu_ctx_t *ctx, tsdrgpu_notch_t **out) {
	BIND(ctx); ARG_TRY(ctx, out != NULL);
	tsdrgpu_notch *t = new tsdrgpu_notch();
	memset(t, 0, sizeof *t);
	t->ctx = ctx;
	*out = t;
	return TSDRGPU_OK;
}

void tsdrgpu_notch_destroy(tsdrgpu_notch_t *t) {
	if (!t) return;
	cudaSetDevice(t->ctx->device);
	if (t->d_H) cudaFree(t->d_H);
	if (t->d_tw) cudaFree(t->d_tw);
	for (int i = 0; i < 2; i++) if (t->d_hist[i]) cudaFree(t->d_hist[i]);
	delete t;
}

int tsdrgpu_notch_reset(tsdrgpu_notch_t *t, void *stream) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, t != NULL);
	tsdrgpu_ctx_t *ctx = t->ctx;
	BIND(ctx);
	ARG_TRY(ctx, t->configured);
	t->pos = 0; t->cur = 0; t->hstart = -(long long) (t->L - 1);
	CU_TRY(ctx, cudaMemsetAsync(t->d_hist[0], 0, sizeof(float2) * (size_t) t->N, (cudaStream_t) stream));
	return TSDRGPU_OK;
}

int tsdrgpu_notch_configure(tsdrgpu_notch_t *t, uint32_t fs, int n, const double *centers, const double *widths, int ntaps) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, t != NULL);
	tsdrgpu_ctx_t *ctx = t->ctx;
	BIND(ctx);
	int L = 0;
	int rc = nt_validate(ctx, fs, n, centers, widths, ntaps, &L);
	if (rc) return rc;
	const int N = nt_fft_size(L), logN = ilog2(N);
	std::vector<std::complex<double>> h, X((size_t) N, std::complex<double>(0.0, 0.0));
	nt_taps(fs, n, centers, widths, L, h);
	for (int i = 0; i < L; i++) X[i] = std::complex<double>((double) (float) h[i].real(), (double) (float) h[i].imag());   // the float32 taps
	host_fft(X);
	std::vector<float2> H((size_t) N);
	for (int i = 0; i < N; i++) { const std::complex<double> v = X[brev_n((unsigned) i, logN)] / (double) N; H[i] = make_float2((float) v.real(), (float) v.imag()); }
	const std::vector<float2> tw = twiddles(N);
	CU_TRY(ctx, cudaDeviceSynchronize());                                  // a reconfiguration is not on the hot path
	if (t->d_H) { CU_TRY(ctx, cudaFree(t->d_H)); t->d_H = NULL; }
	if (t->d_tw) { CU_TRY(ctx, cudaFree(t->d_tw)); t->d_tw = NULL; }
	for (int i = 0; i < 2; i++) if (t->d_hist[i]) { CU_TRY(ctx, cudaFree(t->d_hist[i])); t->d_hist[i] = NULL; }
	CU_TRY(ctx, cudaMalloc(&t->d_H, sizeof(float2) * H.size()));
	CU_TRY(ctx, cudaMemcpy(t->d_H, H.data(), sizeof(float2) * H.size(), cudaMemcpyHostToDevice));
	CU_TRY(ctx, cudaMalloc(&t->d_tw, sizeof(float2) * tw.size()));
	CU_TRY(ctx, cudaMemcpy(t->d_tw, tw.data(), sizeof(float2) * tw.size(), cudaMemcpyHostToDevice));
	for (int i = 0; i < 2; i++) CU_TRY(ctx, cudaMalloc(&t->d_hist[i], sizeof(float2) * (size_t) N));   // (L - 1) + (pos mod hop) < N pairs
	t->L = L; t->N = N; t->logN = logN; t->hop = N - (L - 1); t->NT = N / 2 < 1024 ? N / 2 : 1024;
	t->smem = sizeof(float2) * (size_t) N;
	CU_TRY(ctx, cudaFuncSetAttribute(notch_ols, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) (sizeof(float2) * NT_MAX_N)));
	t->configured = 1;
	return tsdrgpu_notch_reset(t, NULL) == TSDRGPU_OK ? (cudaDeviceSynchronize() == cudaSuccess ? TSDRGPU_OK : TSDRGPU_ECUDA) : TSDRGPU_ECUDA;
}

int tsdrgpu_notch_run(tsdrgpu_notch_t *t, void *stream, const float *d_iq, uint64_t pairs, uint64_t dropped_before, float *d_out,
                      uint64_t *out_pairs, uint64_t *out_dropped) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, t != NULL);
	tsdrgpu_ctx_t *ctx = t->ctx;
	BIND(ctx);
	ARG_TRY(ctx, t->configured);
	ARG_TRY(ctx, pairs == 0 || (d_iq != NULL && d_out != NULL));
	cudaStream_t s = (cudaStream_t) stream;
	NtArgs a;
	a.v.in = reinterpret_cast<const float2 *>(d_iq); a.v.hist = t->d_hist[t->cur];
	a.v.p = (long long) t->pos; a.v.g = (long long) dropped_before; a.v.k = (long long) pairs; a.v.hstart = t->hstart;
	a.out = reinterpret_cast<float2 *>(d_out); a.H = t->d_H; a.tw = t->d_tw;
	a.logN = t->logN; a.L1 = t->L - 1; a.hop = t->hop;
	const long long b0 = a.v.p + a.v.g, end = b0 + a.v.k;
	if (pairs > 0) {
		a.s0 = b0 / t->hop;
		const unsigned long long grid = (unsigned long long) ((end - 1) / t->hop - a.s0 + 1);
		ARG_TRY(ctx, grid < (1ull << 31));
		KL(ctx, "notch_ols", s, notch_ols<<<(unsigned) grid, t->NT, t->smem, s>>>(a));
	}
	if (pairs > 0 || dropped_before > 0) {                           // the history moves on, also over an empty block's gap
		const long long hs = end / t->hop * t->hop - (t->L - 1);
		const int len = (int) (end - hs);
		KL(ctx, "notch_history", s, stream_history<<<(unsigned) ((len + 255) / 256), 256, 0, s>>>(a.v, t->d_hist[t->cur ^ 1], hs, len));
		t->cur ^= 1; t->hstart = hs;
	}
	t->pos = (uint64_t) end;
	if (out_pairs) *out_pairs = pairs;
	if (out_dropped) *out_dropped = dropped_before;
	return TSDRGPU_OK;
}

// ---- spectrum --------------------------------------------------------------------------------------------------------
int tsdrgpu_spectrum_check(uint32_t fs, int nfft) {
	if (fs == 0) return nt_bad(NULL, "spectrum: the sample rate must be > 0");
	if (nfft < SP_MIN_N || nfft > SP_MAX_N || (nfft & (nfft - 1)) != 0) return nt_bad(NULL, "spectrum: nfft must be a power of two in 64..16384");
	return TSDRGPU_OK;
}

int tsdrgpu_spectrum_create(tsdrgpu_ctx_t *ctx, tsdrgpu_spectrum_t **out) {
	BIND(ctx); ARG_TRY(ctx, out != NULL);
	tsdrgpu_spectrum *s = new tsdrgpu_spectrum();
	memset(s, 0, sizeof *s);
	s->ctx = ctx;
	*out = s;
	return TSDRGPU_OK;
}

void tsdrgpu_spectrum_destroy(tsdrgpu_spectrum_t *s) {
	if (!s) return;
	cudaSetDevice(s->ctx->device);
	void *bufs[] = {s->d_win, s->d_tw, s->d_sum, s->d_pw, s->d_hist[0], s->d_hist[1]};
	for (void *b : bufs) if (b) cudaFree(b);
	delete s;
}

int tsdrgpu_spectrum_reset(tsdrgpu_spectrum_t *s, void *stream) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, s != NULL);
	tsdrgpu_ctx_t *ctx = s->ctx;
	BIND(ctx);
	ARG_TRY(ctx, s->configured);
	s->pos = 0; s->seg_next = 0; s->drop_end = 0; s->segments = 0; s->cur = 0;
	CU_TRY(ctx, cudaMemsetAsync(s->d_hist[0], 0, sizeof(float2) * (size_t) s->N, (cudaStream_t) stream));
	CU_TRY(ctx, cudaMemsetAsync(s->d_sum, 0, sizeof(double) * (size_t) s->N, (cudaStream_t) stream));
	return TSDRGPU_OK;
}

int tsdrgpu_spectrum_configure(tsdrgpu_spectrum_t *s, uint32_t fs, int nfft) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, s != NULL);
	tsdrgpu_ctx_t *ctx = s->ctx;
	BIND(ctx);
	if (tsdrgpu_spectrum_check(fs, nfft)) { snprintf(ctx->err, sizeof ctx->err, "%s", tsdrgpu_last_error(NULL)); return TSDRGPU_EINVAL; }
	const int N = nfft;
	std::vector<float> win((size_t) N);
	double w2 = 0.0;
	for (int i = 0; i < N; i++) {                                   // periodic Hann (scipy.signal.get_window('hann', N))
		const double w = 0.5 - 0.5 * cos(2.0 * M_PI * i / N);
		win[i] = (float) w; w2 += w * w;
	}
	const std::vector<float2> tw = twiddles(N);
	CU_TRY(ctx, cudaDeviceSynchronize());
	void *bufs[] = {s->d_win, s->d_tw, s->d_sum, s->d_pw, s->d_hist[0], s->d_hist[1]};
	for (void *b : bufs) if (b) CU_TRY(ctx, cudaFree(b));
	s->d_win = NULL; s->d_tw = NULL; s->d_sum = NULL; s->d_pw = NULL; s->d_hist[0] = s->d_hist[1] = NULL;
	CU_TRY(ctx, cudaMalloc(&s->d_win, sizeof(float) * N));
	CU_TRY(ctx, cudaMemcpy(s->d_win, win.data(), sizeof(float) * N, cudaMemcpyHostToDevice));
	CU_TRY(ctx, cudaMalloc(&s->d_tw, sizeof(float2) * tw.size()));
	CU_TRY(ctx, cudaMemcpy(s->d_tw, tw.data(), sizeof(float2) * tw.size(), cudaMemcpyHostToDevice));
	CU_TRY(ctx, cudaMalloc(&s->d_sum, sizeof(double) * N));
	CU_TRY(ctx, cudaMalloc(&s->d_pw, sizeof(double) * (size_t) SP_CHUNK));
	for (int i = 0; i < 2; i++) CU_TRY(ctx, cudaMalloc(&s->d_hist[i], sizeof(float2) * N));
	CU_TRY(ctx, cudaFuncSetAttribute(spectrum_segments, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) (sizeof(float2) * SP_MAX_N)));
	s->fs = fs; s->N = N; s->logN = ilog2(N); s->NT = N / 2 < 1024 ? N / 2 : 1024; s->wsum2 = w2;
	s->configured = 1;
	int rc = tsdrgpu_spectrum_reset(s, NULL);
	if (rc) return rc;
	CU_TRY(ctx, cudaDeviceSynchronize());
	return TSDRGPU_OK;
}

int tsdrgpu_spectrum_run(tsdrgpu_spectrum_t *s, void *stream, const float *d_iq, uint64_t pairs, uint64_t dropped_before) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, s != NULL);
	tsdrgpu_ctx_t *ctx = s->ctx;
	BIND(ctx);
	ARG_TRY(ctx, s->configured);
	ARG_TRY(ctx, pairs == 0 || d_iq != NULL);
	cudaStream_t st = (cudaStream_t) stream;
	const uint64_t N = (uint64_t) s->N, h2 = N / 2, b0 = s->pos + dropped_before, end = b0 + pairs;
	StreamView v;
	v.in = reinterpret_cast<const float2 *>(d_iq); v.hist = s->d_hist[s->cur];
	v.p = (long long) s->pos; v.g = (long long) dropped_before; v.k = (long long) pairs; v.hstart = (long long) s->pos - (long long) N;
	if (dropped_before > 0) s->drop_end = b0;                      // a segment that starts before drop_end touches a drop: skipped
	const uint64_t s_end = end >= N ? (end - N) / h2 + 1 : 0;      // segments complete with this block: s < s_end
	uint64_t s_lo = std::max(s->seg_next, (s->drop_end + h2 - 1) / h2);
	const uint64_t rows_max = (uint64_t) SP_CHUNK / N;
	while (s_lo < s_end) {
		const uint64_t rows = std::min(rows_max, s_end - s_lo);
		KL(ctx, "spectrum_segments", st, spectrum_segments<<<(unsigned) rows, s->NT, sizeof(float2) * N, st>>>(v, s->d_win, s->d_tw, (long long) s_lo,
		                                                                                                       s->logN, s->d_pw));
		KL(ctx, "spectrum_accumulate", st, spectrum_accumulate<<<(unsigned) ((N + 255) / 256), 256, 0, st>>>(s->d_pw, (int) rows, (int) N, s->d_sum));
		s->segments += rows; s_lo += rows;
	}
	s->seg_next = std::max(s->seg_next, s_end);
	if (pairs > 0 || dropped_before > 0) {                         // the history: the last N positions
		KL(ctx, "spectrum_history", st, stream_history<<<(unsigned) ((N + 255) / 256), 256, 0, st>>>(v, s->d_hist[s->cur ^ 1], (long long) end - (long long) N, (int) N));
		s->cur ^= 1;
	}
	s->pos = end;
	return TSDRGPU_OK;
}

int tsdrgpu_spectrum_results(tsdrgpu_spectrum_t *s, void *stream, double *h_psd, int cap, uint64_t *segments) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, s != NULL);
	tsdrgpu_ctx_t *ctx = s->ctx;
	BIND(ctx);
	ARG_TRY(ctx, s->configured && (h_psd != NULL || cap <= 0));
	std::vector<double> sum((size_t) s->N);
	CU_TRY(ctx, cudaStreamSynchronize((cudaStream_t) stream));
	CU_TRY(ctx, cudaMemcpy(sum.data(), s->d_sum, sizeof(double) * sum.size(), cudaMemcpyDeviceToHost));
	const double scale = s->segments ? 1.0 / ((double) s->segments * (double) s->fs * s->wsum2) : 0.0;
	for (int i = 0; i < s->N && i < cap; i++) h_psd[i] = sum[(size_t) ((i + s->N / 2) % s->N)] * scale;    // fft-shifted: -fs/2 first
	if (segments) *segments = s->segments;
	return TSDRGPU_OK;
}

}  // extern "C"
