// fft.cu -- a18..a20, a22: FFT, "autocorrelation", cross-correlation, the frame-rate detector's running means and
// the superbandwidth stitch.
//
// Replaces fft_perform / fft_autocorrelation / fft_crosscorrelation (fft.c:49-176), accummulate and
// frameratedetector_runontodata (frameratedetector.c:34-126), complex_to_abs_diff / superb_bestfit /
// superb_ondataready (superbandwidth.c:67-152).
//
// FFT design (no tensor cores: nothing here is a dense contraction; the bound is HBM bandwidth and issue slots):
//   N = 2^m is factored into 1, 2 or 3 line lengths (Cooley-Tukey index maps; 2 passes up to 2^20, 3 above).  One CTA
//   transforms a BUNDLE of C adjacent lines (4096 points, 512 threads): radix-8 Stockham stages written as their radix-2
//   layers, the first fed from global memory, the last storing to global memory through the epilogue (inter-pass twiddle,
//   scale, |.|), the ones between through XOR-swizzled shared memory.  Bundling makes every global access a run of >= C
//   consecutive complex values even on the strided passes, so each pass is one coalesced read + one coalesced write of
//   the array: 16 N bytes per pass.  The transposing last pass writes to the other buffer, so no copy pass exists.
//   Real->complex widening and |X|/N are fused into the first / last pass of the autocorrelation's forward transform;
//   a FAN variant of the last pass stores into the gather buffers of all ranks (superbandwidth, one hop per GPU).
// Numerics: float32 data.  Layer twiddles come from host-built double-precision tables that carry the REFERENCE'S stage
// angles (its half-angle recurrence, fft.c:161, is off by up to 5e-5 relative at the largest stages: see
// tsdrgpu_fft_reference_eps), inter-pass twiddles from sincospif of an exactly reduced argument times a host-built step
// table.  The reference keeps float32 storage between its radix-2 stages too (fft.c:150-155); results agree to <= 1e-6 of
// the spectrum's peak up to 2^22 (not bit-exact).
#include "common.cuh"
#include <math.h>
#include <stdlib.h>
#include <vector>
#include <mutex>

namespace {

constexpr int FFT_MAX_LOG2L = 11;            // longest line transformed inside one CTA: 2048
constexpr int FFT_TABLE = 1 << FFT_MAX_LOG2L;
constexpr int FFT_MAX_ELEMS = 4096;          // complex elements per CTA bundle: 512 threads x 8 (35 KB of shared memory, >= 3 CTAs/SM)

struct FftPass {
	int log2L, C, log2C, c_fast_in, c_fast_out;
	long long in_bs, out_bs;                            // batch strides (blockIdx.y), in elements of the in / out type
	unsigned G_lo;
	long long in_hi, in_lo, in_cs, in_js;
	long long out_hi, out_lo, out_cs, out_ks;
	unsigned long long tw_M; long long tw_lo, tw_cs;    // column index = g_lo*tw_lo + c*tw_cs ; tw_M == 0: none
	float scale;
	int in_real, out_abs;                               // in_real: 1 = real input widened to (x, 0); 2 = complex input given as PAIRS OF FLOATS that are only 4-byte aligned (in_bs then counts floats)
	const float2 *tw_step;                              // host-built W_M^(col (L/8) j), [col][8]; NULL: compute every twiddle
	float2 *fan[16]; int nfan;                          // FAN kernels: the last stage stores to every fan[p] + offset instead of `out`
	int exact0;                                         // the first three layers of this pass have eps = 0: plain DFT-8
	int conj_in, conj_out;                              // inverse transforms: conjugate on load (first pass) / on store (last pass)
	float *abs_real;                                    // with out_abs: |.| goes here as float32 (same element index) instead of (|.|, 0) to `out` -- may be peer memory
	int dbg;                                            // timing experiments only (TSDRGPU_FFT_DBG): 1 = no global loads, 2 = no global stores; results are garbage
};

__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }

// ---- in-register small DFTs (natural order in, natural order out) -------------------------------------------------
// Packed single precision (sm_100: add/mul/fma.rn.f32x2 -> SASS FADD2 / FMUL2 / FFMA2): one instruction works on both halves of
// a complex value held in an aligned register pair.  The pass kernel is bound by issue slots, not by the FP pipes, so halving
// the arithmetic instruction count is what counts: a complex add is 1 instruction instead of 2, a complex multiply by a
// twiddle kept in both forms (c, s) and (-s, c) is 2 instead of 4 (the scalar broadcast of x.x / x.y is an operand modifier).
__device__ __forceinline__ unsigned long long pk2(float2 a) { unsigned long long r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a.x), "f"(a.y)); return r; }
__device__ __forceinline__ float2 up2(unsigned long long r) { float2 a; asm("mov.b64 {%0, %1}, %2;" : "=f"(a.x), "=f"(a.y) : "l"(r)); return a; }
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { unsigned long long r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk2(a)), "l"(pk2(b))); return up2(r); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) {      // a - b = b * (-1, -1) + a
	unsigned long long r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(pk2(b)), "l"(pk2(make_float2(-1.0f, -1.0f))), "l"(pk2(a))); return up2(r);
}
// x * w with w given as (c, s) and its quarter turn (-s, c):  (x.x c - x.y s, x.x s + x.y c)
__device__ __forceinline__ float2 cmulp(float2 x, float4 w) {
	unsigned long long t, r;
	asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(t) : "l"(pk2(make_float2(x.y, x.y))), "l"(pk2(make_float2(w.z, w.w))));
	asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(pk2(make_float2(x.x, x.x))), "l"(pk2(make_float2(w.x, w.y))), "l"(t));
	return up2(r);
}
__device__ __forceinline__ float4 twform(float2 w) { return make_float4(w.x, w.y, -w.y, w.x); }
__device__ __forceinline__ float2 cscale(float2 a, float s) { unsigned long long r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk2(a)), "l"(pk2(make_float2(s, s)))); return up2(r); }
// multiply by -i (forward) or +i (inverse)
__device__ __forceinline__ float2 rot90(float2 a, bool inverse) { return inverse ? make_float2(-a.y, a.x) : make_float2(a.y, -a.x); }

__device__ __forceinline__ void dft2(float2 &a, float2 &b) { const float2 t = a; a = cadd(t, b); b = csub(t, b); }
__device__ __forceinline__ void dft4(float2 &v0, float2 &v1, float2 &v2, float2 &v3, bool inverse) {
	const float2 a0 = cadd(v0, v2), a1 = csub(v0, v2), a2 = cadd(v1, v3), a3 = rot90(csub(v1, v3), inverse);
	v0 = cadd(a0, a2); v1 = cadd(a1, a3); v2 = csub(a0, a2); v3 = csub(a1, a3);
}
__device__ __forceinline__ void dft8(float2 (&v)[8], bool inverse) {
	// even / odd halves as two 4-point DFTs, then the W8^k twiddles
	dft4(v[0], v[2], v[4], v[6], inverse);
	dft4(v[1], v[3], v[5], v[7], inverse);
	const float h = 0.70710678118654752440f;
	const float2 o0 = v[1];
	const float2 t1 = v[3];            // * W8^1 = (1 -+ i)/sqrt2
	const float2 o1 = inverse ? make_float2(h * (t1.x - t1.y), h * (t1.x + t1.y)) : make_float2(h * (t1.x + t1.y), h * (t1.y - t1.x));
	const float2 o2 = rot90(v[5], inverse);
	const float2 t3 = v[7];            // * W8^3 = (-1 -+ i)/sqrt2
	const float2 o3 = inverse ? make_float2(-h * (t3.x + t3.y), h * (t3.x - t3.y)) : make_float2(h * (t3.y - t3.x), -h * (t3.x + t3.y));
	const float2 e0 = v[0], e1 = v[2], e2 = v[4], e3 = v[6];
	v[0] = cadd(e0, o0); v[1] = cadd(e1, o1); v[2] = cadd(e2, o2); v[3] = cadd(e3, o3);
	v[4] = csub(e0, o0); v[5] = csub(e1, o1); v[6] = csub(e2, o2); v[7] = csub(e3, o3);
}

// transforms of 2 or 4 points (whole transforms only: passes of longer ones have lines of >= 64): one thread each, exact
// twiddles (the reference's first two stages have no angle error), the same load / store conventions as the pass kernel
template <int LOG2L>
__global__ void __launch_bounds__(32) fft_tiny_kernel(const float2 *in, float2 *out, FftPass P) {
	if (threadIdx.x != 0) return;
	constexpr int L = 1 << LOG2L;
	const long long ib = (long long) blockIdx.y * P.in_bs, ob = (long long) blockIdx.y * P.out_bs;
	float2 v[L];
	#pragma unroll
	for (int j = 0; j < L; j++) {
		if (P.in_real == 2) { const float *pr = reinterpret_cast<const float *>(in) + ib + 2 * j; v[j] = make_float2(pr[0], pr[1]); }
		else v[j] = P.in_real ? make_float2(reinterpret_cast<const float *>(in)[ib + j], 0.0f) : in[ib + j];
		if (P.conj_in) v[j].y = -v[j].y;
	}
	if (L == 2) dft2(v[0], v[1]); else dft4(v[0], v[1], v[2], v[3], false);
	#pragma unroll
	for (int k = 0; k < L; k++) {
		float2 r = make_float2(v[k].x * P.scale, v[k].y * (P.conj_out ? -P.scale : P.scale));
		if (P.out_abs) r = make_float2(__fsqrt_rn(__fadd_rn(__fmul_rn(r.x, r.x), __fmul_rn(r.y, r.y))), 0.0f);
		out[ob + k] = r;
	}
}

// ---- the pass kernel for lines of length L >= 8 --------------------------------------------------------------------
// Each thread owns 8 points per stage.  The first radix-8 butterfly is fed straight from global memory and the last
// butterfly (radix 8, 4 or 2) stores straight to global memory (through the inter-pass twiddle / scale / |.| epilogue),
// so a 1024-point line makes 3 trips through shared memory instead of 5 + load + store, with one barrier each
// (ping-pong buffers).  Thread -> (line, butterfly) maps are chosen per pass so that the global accesses of a warp are
// runs of consecutive complex values: line-fastest on strided passes, butterfly-fastest on contiguous lines.
//
// Butterflies are written as their radix-2 layers (a radix-8 Stockham step with block size p = layers with blocks p, 2p,
// 4p): layer t multiplies the upper input by T_t[K], K = k + p q0 (+ 2p q1).  The layer twiddles come from a per-pass
// table built on the host in double precision, T_s[K] = exp(-i pi K / 2^s (1 + eps_s)), stored layer after layer
// (layer s at offset 2^s - 1), so the seven twiddles of a radix-8 butterfly are table[k + j p - 1], j = 1..7.
// eps_s is the relative angle error of the reference's stage l_base + s (tsdrgpu_fft_reference_eps; fft.c:161 derives
// its twiddles by a half-angle recurrence that loses accuracy for small angles) or 0 for the mathematically exact DFT:
// same kernel, same operation count (12 complex multiplications + 24 additions per 8 points) either way.
//
// Shared memory is unpadded; a line's point q lives at slot (q ^ swz(q)) ^ xc(line): swz permutes inside aligned groups
// of 16 so that the stride-8 stores of stage 0 and the stride-p stores of the p = 8 stage hit 16 distinct bank pairs per
// half-warp, and xc (a per-line constant < 16) does the same for the line-fastest thread maps of strided passes.
// swz is linear over GF(2): swz(a ^ b) = swz(a) ^ swz(b).  Every index the kernel forms is a sum of two terms with
// disjoint bits (i + m L/8, 8 i + m, j + m p), so slot = swz(thread part) ^ swz(m part) and the m part is a compile-time
// constant: one XOR and one add per access on 32-bit shared addresses.
__host__ __device__ constexpr int swz(int q) { return q ^ ((q >> 4) & 7) ^ (((q >> 6) & 1) << 3); }
__device__ __forceinline__ unsigned smem_addr(const void *p) { return (unsigned) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void sts2(unsigned addr, float2 v) { asm volatile("st.shared.v2.f32 [%0], {%1, %2};" :: "r"(addr), "f"(v.x), "f"(v.y) : "memory"); }
__device__ __forceinline__ float2 lds2(unsigned addr) { float2 v; asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr) : "memory"); return v; }

// Butterflies exist in the FORWARD direction only.  An inverse transform is the conjugate of the forward transform of the
// conjugated input -- conj(x conj(w)) = conj(x) w, and IEEE arithmetic is sign-symmetric -- so an inverse pass conjugates what it
// loads from global memory in its first pass and what it stores in its last one (FftPass.conj_in / conj_out) and is otherwise
// the same code.  Layer twiddles are loaded as (c, s) and turned into cmulp's (c, s, -s, c) in registers: 16-byte table entries
// were measured slower (twice the L1 wavefronts on a kernel whose first stall reason is the memory-instruction queue).
__device__ __forceinline__ void bf8(float2 *v, const float2 *__restrict__ tw /* = table + k - 1 */, int p) {
	float2 a[4][2], b[2][2][2];
	const float4 TA = twform(__ldg(tw + p)), TB0 = twform(__ldg(tw + 2 * p)), TB1 = twform(__ldg(tw + 3 * p));
	const float4 TC00 = twform(__ldg(tw + 4 * p)), TC10 = twform(__ldg(tw + 5 * p)), TC01 = twform(__ldg(tw + 6 * p)), TC11 = twform(__ldg(tw + 7 * p));
	#pragma unroll
	for (int r = 0; r < 4; r++) { const float2 hi = cmulp(v[r + 4], TA); a[r][0] = cadd(v[r], hi); a[r][1] = csub(v[r], hi); }
	#pragma unroll
	for (int q0 = 0; q0 < 2; q0++) {
		const float4 TB = q0 ? TB1 : TB0;
		#pragma unroll
		for (int m0 = 0; m0 < 2; m0++) { const float2 hi = cmulp(a[m0 + 2][q0], TB); b[m0][q0][0] = cadd(a[m0][q0], hi); b[m0][q0][1] = csub(a[m0][q0], hi); }
	}
	#pragma unroll
	for (int q0 = 0; q0 < 2; q0++) {
		#pragma unroll
		for (int q1 = 0; q1 < 2; q1++) {
			const float4 TC = q1 ? (q0 ? TC11 : TC01) : (q0 ? TC10 : TC00);
			const float2 hi = cmulp(b[1][q0][q1], TC);
			v[q0 + 2 * q1] = cadd(b[0][q0][q1], hi); v[q0 + 2 * q1 + 4] = csub(b[0][q0][q1], hi);
		}
	}
}
__device__ __forceinline__ void bf4(float2 *v, const float2 *__restrict__ tw, int p) {
	float2 a[2][2];
	const float4 TA = twform(__ldg(tw + p)), TB0 = twform(__ldg(tw + 2 * p)), TB1 = twform(__ldg(tw + 3 * p));
	#pragma unroll
	for (int r = 0; r < 2; r++) { const float2 hi = cmulp(v[r + 2], TA); a[r][0] = cadd(v[r], hi); a[r][1] = csub(v[r], hi); }
	#pragma unroll
	for (int q0 = 0; q0 < 2; q0++) {
		const float2 hi = cmulp(a[1][q0], q0 ? TB1 : TB0);
		v[q0] = cadd(a[0][q0], hi); v[q0 + 2] = csub(a[0][q0], hi);
	}
}
__device__ __forceinline__ void bf2(float2 *v, const float2 *__restrict__ tw, int p) {
	const float2 hi = cmulp(v[1], twform(__ldg(tw + p)));
	const float2 lo = v[0];
	v[0] = cadd(lo, hi); v[1] = csub(lo, hi);
}

// ---- TMA: a pass whose lines are contiguous in memory (the second pass of a two-pass plan, the third of a three-pass plan,
// a single-pass transform) gets its whole bundle with bulk copies (cp.async.bulk.shared::cluster.global, SASS UBLKCP) issued
// by one thread and counted in bytes on an mbarrier: C copies of one line each -- or ONE copy of C L complex values when the
// lines of the bundle are adjacent, as in two-pass plans -- land linearly in the half of the ping-pong buffer the first
// butterfly does not write; the threads wait on the barrier and read their eight inputs from shared memory (consecutive
// lanes read consecutive values: conflict-free without a swizzle).  The eight dependent global loads per thread, their address
// arithmetic and their scoreboard stalls are gone from the instruction stream.
__device__ __forceinline__ void fft_mbar_init(unsigned bar, unsigned count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void fft_mbar_expect_tx(unsigned bar, unsigned bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory"); }
__device__ __forceinline__ void fft_mbar_wait(unsigned bar, unsigned parity) {
	asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}"
	             :: "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void fft_bulk_g2s(unsigned dst_smem, const void *src, unsigned bytes, unsigned bar) {
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
	             :: "r"(dst_smem), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

template <int LOG2L, bool FAN = false, bool TMA = false>
__global__ void __launch_bounds__(512, 3) fft_pass_kernel(const float2 *in, float2 *out, FftPass P, const float2 *__restrict__ stw) {
	extern __shared__ __align__(128) float2 s[];
	constexpr int L = 1 << LOG2L, NST8 = LOG2L / 3, RL = LOG2L % 3;
	constexpr int RLAST = (RL == 0) ? 8 : ((RL == 1) ? 2 : 4);
	constexpr int NSTAGES = NST8 + (RL ? 1 : 0);
	constexpr int NMID = NSTAGES - 2;                    // radix-8 stages between the first and the last one
	constexpr int L8 = L / 8, LOG2L8 = LOG2L - 3;
	const int C = P.C, log2C = P.log2C;
	const int tid = threadIdx.x;
	const unsigned g = blockIdx.x, g_hi = g / P.G_lo, g_lo = g - g_hi * P.G_lo;
	const long long in_base = (long long) g_hi * P.in_hi + (long long) g_lo * P.in_lo + (P.in_real == 2 ? 0ll : (long long) blockIdx.y * P.in_bs);
	float2 *gout = out + ((long long) g_hi * P.out_hi + (long long) g_lo * P.out_lo + (long long) blockIdx.y * P.out_bs);
	const bool active = tid < C * L8;                    // tiny bundles leave part of the last warp idle
	// per-line slot constants (see above): xa for the buffer stage 0 writes, xb for the buffer the last stage reads
	const int sha = (log2C >= 4) ? 0 : 3 - log2C, shb = (NSTAGES == 2 || log2C >= 4) ? sha : 4 - log2C;
	const unsigned sbase = smem_addr(s);
	float2 v[8];
	// Inter-pass twiddles W_M^(col k): a thread's eight outputs are k = i0 + (L/8) j, j = 0..7, of ONE column, so
	// W^(col k) = W^(col i0) * W^(col (L/8) j): one sincospif per thread for the first factor (exactly reduced argument),
	// the second from a host-built table of 8 values per column (double precision; P.tw_step[col * 8 + j]).
	const bool tw_fast = P.tw_step != NULL && P.c_fast_out && (int) blockDim.x == C * L8;

	// ---- stage 0: radix 8, p = 1, inputs x[i + m L/8] from global memory (or, TMA, from the bundle the bulk copies landed)
	{
		int c, i;
		if (P.c_fast_in) { c = tid & (C - 1); i = tid >> log2C; } else { i = tid & (L8 - 1); c = tid >> LOG2L8; }
		if (P.dbg & 1) {
			#pragma unroll
			for (int m = 0; m < 8; m++) v[m] = make_float2((float) tid, (float) m);
		} else if (TMA) {
			__shared__ __align__(8) unsigned long long bar_mem;
			const unsigned bar = smem_addr(&bar_mem);
			const unsigned landing = sbase + ((NSTAGES > 1) ? (unsigned) (C * L) * 8u : 0u);      // the half stage 0 does not write
			if (tid == 0) { fft_mbar_init(bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
			__syncthreads();
			if (tid == 0) {
				const unsigned line_bytes = (unsigned) L * 8u;
				fft_mbar_expect_tx(bar, (unsigned) C * line_bytes);
				const float2 *g0 = in + in_base;
				if ((int) P.in_cs == L) fft_bulk_g2s(landing, g0, (unsigned) C * line_bytes, bar);          // adjacent lines: one copy
				else for (int cc = 0; cc < C; cc++) fft_bulk_g2s(landing + (unsigned) cc * line_bytes, g0 + (long long) cc * P.in_cs, line_bytes, bar);
			}
			fft_mbar_wait(bar, 0);
			if (active) {
				const unsigned lr = landing + (unsigned) (c * L + i) * 8u;
				#pragma unroll
				for (int m = 0; m < 8; m++) v[m] = lds2(lr + (unsigned) (m * L8) * 8u);
				if (P.conj_in) {
					#pragma unroll
					for (int m = 0; m < 8; m++) v[m].y = -v[m].y;
				}
			}
		} else if (active) {
			const int off = c * (int) P.in_cs + i * (int) P.in_js, step = L8 * (int) P.in_js;
			if (P.in_real == 2) {                             // pairs of floats, 4-byte aligned (a capture that starts on an odd sample)
				const float *gr = reinterpret_cast<const float *>(in) + (long long) blockIdx.y * P.in_bs + 2 * (in_base + off);
				#pragma unroll
				for (int m = 0; m < 8; m++) v[m] = make_float2(__ldg(gr + 2 * m * step), __ldg(gr + 2 * m * step + 1));
				if (P.conj_in) {
					#pragma unroll
					for (int m = 0; m < 8; m++) v[m].y = -v[m].y;
				}
			} else if (P.in_real) {
				const float *gr = reinterpret_cast<const float *>(in) + in_base + off;
				#pragma unroll
				for (int m = 0; m < 8; m++) v[m] = make_float2(__ldg(gr + m * step), 0.0f);
			} else {
				const float2 *gc = in + in_base + off;
				#pragma unroll
				for (int m = 0; m < 8; m++) v[m] = __ldg(gc + m * step);
				if (P.conj_in) {
					#pragma unroll
					for (int m = 0; m < 8; m++) v[m].y = -v[m].y;
				}
			}
		}
		if (active) {
			if (P.exact0) { float2 (&u)[8] = *reinterpret_cast<float2 (*)[8]>(&v[0]); dft8(u, false); }     // layers with eps = 0: plain DFT-8
			else bf8(v, stw - 1, 1);
		}
		if (NSTAGES > 1) {
			if (active) {
				const unsigned la = sbase + (unsigned) (c * L) * 8u, rb = (unsigned) (swz(8 * i) ^ ((c << sha) & 15)) * 8u;
				#pragma unroll
				for (int m = 0; m < 8; m++) sts2(la + (rb ^ (unsigned) (m * 8)), v[m]);
			}
			__syncthreads();
		}
	}
	unsigned src = sbase, dst = sbase + (unsigned) (C * L) * 8u;
	// ---- middle radix-8 stages (shared -> shared, ping-pong)
	#pragma unroll
	for (int st = 0; st < (NMID > 0 ? NMID : 0); st++) {
		const int p = 8 << (3 * st);
		const int i = tid & (L8 - 1), c = tid >> LOG2L8;
		if (active) {
			const int xa = (c << sha) & 15, xw = (st == NMID - 1) ? ((c << shb) & 15) : xa;
			const unsigned lr = src + (unsigned) (c * L) * 8u, rb = (unsigned) (swz(i) ^ xa) * 8u;
			#pragma unroll
			for (int m = 0; m < 8; m++) v[m] = lds2(lr + (rb ^ (unsigned) (swz(m * L8) * 8)));
			const int k = i & (p - 1);
			bf8(v, stw + k - 1, p);
			const int j = ((i - k) << 3) + k;
			const unsigned lw = dst + (unsigned) (c * L) * 8u, wb = (unsigned) (swz(j) ^ xw) * 8u;
			#pragma unroll
			for (int m = 0; m < 8; m++) sts2(lw + (wb ^ (unsigned) (swz(m * p) * 8)), v[m]);
		}
		__syncthreads();
		const unsigned t = src; src = dst; dst = t;
	}
	// ---- last stage: radix RLAST with p = L / RLAST, results X[i + m p] go to global memory
	constexpr int NB = 8 / RLAST, PL = L / RLAST, LOG2PL = LOG2L - (RLAST == 8 ? 3 : (RLAST == 4 ? 2 : 1));
	const int T = blockDim.x;
	const unsigned twmask = (unsigned) (P.tw_M - 1);
	const float inv_M = P.tw_M ? 1.0f / (float) P.tw_M : 0.0f;       // a power of two: exact
	float4 tw_base4 = make_float4(1.0f, 0.0f, -0.0f, 1.0f);
	#pragma unroll
	for (int it = 0; it < NB; it++) {
		const int widx = tid + it * T;
		if (widx >= C * PL) continue;
		int c, i;
		if (P.c_fast_out) { c = widx & (C - 1); i = widx >> log2C; } else { i = widx & (PL - 1); c = widx >> LOG2PL; }
		float2 *w = v + it * RLAST;
		if (NSTAGES > 1) {
			const unsigned lr = src + (unsigned) (c * L) * 8u, rb = (unsigned) (swz(i) ^ ((c << shb) & 15)) * 8u;
			#pragma unroll
			for (int m = 0; m < RLAST; m++) w[m] = lds2(lr + (rb ^ (unsigned) (swz(m * PL) * 8)));
			if (RLAST == 8) bf8(w, stw + i - 1, PL);
			else if (RLAST == 4) bf4(w, stw + i - 1, PL);
			else bf2(w, stw + i - 1, PL);
		}
		float2 *o = gout + c * (int) P.out_cs;
		const int ks = (int) P.out_ks;
		if (P.tw_M) {
			// inter-pass twiddle W_M^(col k): the argument is reduced exactly in integers, sincospif sees an exact float
			const unsigned col = (unsigned) ((int) g_lo * (int) P.tw_lo + c * (int) P.tw_cs);
			if (tw_fast) {
				if (it == 0) {
					const unsigned e = (col * (unsigned) i) & twmask;            // i == i0 in the first round
					float sn, cs;
					sincospif(-2.0f * ((float) e * inv_M), &sn, &cs);
					tw_base4 = make_float4(cs, sn, -sn, cs);
				}
				#pragma unroll
				for (int m = 0; m < RLAST; m++) {
					const float2 st = __ldg(P.tw_step + col * 8u + (unsigned) (it + NB * m));
					w[m] = cmulp(w[m], twform(cmulp(st, tw_base4)));
				}
			} else if (P.tw_M <= (1ull << 24)) {
				#pragma unroll
				for (int m = 0; m < RLAST; m++) {
					const int k = i + m * PL;
					const unsigned e = (col * (unsigned) k) & twmask;
					float sn, cs;
					sincospif(-2.0f * ((float) e * inv_M), &sn, &cs);
					w[m] = cmulp(w[m], make_float4(cs, sn, -sn, cs));
				}
			} else {
				#pragma unroll
				for (int m = 0; m < RLAST; m++) {
					const int k = i + m * PL;
					const unsigned long long e = ((unsigned long long) col * (unsigned long long) k) & (P.tw_M - 1);
					double dsn, dcs;
					sincospi(-2.0 * ((double) e / (double) P.tw_M), &dsn, &dcs);
					w[m] = cmulp(w[m], make_float4((float) dcs, (float) dsn, -(float) dsn, (float) dcs));
				}
			}
		}
		if (FAN) {
			// fused "transform + all-gather": the result goes straight into every peer's gather buffer (NVLink peer stores;
			// fan[own rank] is local memory), so the exchange overlaps the transform instead of following it
			const long long ob = (gout - out) + (long long) c * (int) P.out_cs;
			#pragma unroll
			for (int m = 0; m < RLAST; m++) {
				const float2 val = make_float2(w[m].x * P.scale, w[m].y * P.scale);
				const long long idx = ob + (long long) (i + m * PL) * ks;
				for (int pr = 0; pr < P.nfan; pr++) P.fan[pr][idx] = val;
			}
		} else if (P.out_abs) {
			#pragma unroll
			for (int m = 0; m < RLAST; m++) {
				const float x = w[m].x * P.scale, y = w[m].y * P.scale;
				const float mag = __fsqrt_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)));
				if (P.abs_real) P.abs_real[(gout - out) + (long long) c * (int) P.out_cs + (long long) (i + m * PL) * ks] = mag;
				else o[(i + m * PL) * ks] = make_float2(mag, 0.0f);
			}
		} else {
			const float sy = P.conj_out ? -P.scale : P.scale;      // inverse transforms: the conjugate on the way out (see bf8)
			#pragma unroll
			for (int m = 0; m < RLAST; m++) if (!(P.dbg & 2) || w[m].x == 1.2345e30f) o[(i + m * PL) * ks] = make_float2(w[m].x * P.scale, w[m].y * sy);
		}
	}
}

// ---- small elementwise helpers -----------------------------------------------------------------------------
__global__ void k_scale(float2 *d, unsigned long long n, float scale) {
	for (unsigned long long i = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long) gridDim.x * blockDim.x) {
		float2 v = d[i]; v.x *= scale; v.y *= scale; d[i] = v;
	}
}
// answer[2i] = real[i], answer[2i+1] = 0 for i in [from, to)          (fft.c:14-22)
__global__ void k_real_to_complex(float2 *answer, const float *real, unsigned long long from, unsigned long long to) {
	for (unsigned long long i = from + (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x; i < to; i += (unsigned long long) gridDim.x * blockDim.x)
		answer[i] = make_float2(real[i], 0.0f);
}
// answer[i] = (|answer[i]|, 0)                                          (fft.c:34-45)
__global__ void k_abs(float2 *answer, unsigned long long from, unsigned long long to) {
	for (unsigned long long i = from + (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x; i < to; i += (unsigned long long) gridDim.x * blockDim.x) {
		const float2 v = answer[i];
		answer[i] = make_float2(mag_exact(v.x, v.y), 0.0f);
	}
}
// ---- real-input transforms at half size (opt-in, see autocorrelation_batch) ------------------------------------------------
// z[j] = x[2j] + i x[2j+1] has been transformed (N/2 points, unscaled) into Z.  With E, O the transforms of the even and odd
// samples, E = (Z[k] + conj Z[-k]) / 2, O = (Z[k] - conj Z[-k]) / 2i, and the reference's LAST radix-2 stage (its perturbed
// angle: last[k] = exp(-i pi k / (N/2) (1 + eps_{m-1})), host-built) gives X[k] = E + last[k] O, X[k + N/2] = E - last[k] O.
__device__ __forceinline__ void real_split(float2 zk, float2 zm, float2 w, float2 &x0, float2 &x1) {
	const float2 e = make_float2(0.5f * (zk.x + zm.x), 0.5f * (zk.y - zm.y));
	const float2 o = make_float2(0.5f * (zk.y + zm.y), -0.5f * (zk.x - zm.x));
	const float2 t = make_float2(w.x * o.x - w.y * o.y, w.x * o.y + w.y * o.x);
	x0 = make_float2(e.x + t.x, e.y + t.y); x1 = make_float2(e.x - t.x, e.y - t.y);
}
// forward: R[k] = |X[k]| / N for all N outputs, as REAL numbers (they are the next transform's real input); grid.y = batch
__global__ void __launch_bounds__(256) k_real_fwd_finish(const float2 *__restrict__ Z, long long z_bs, const float2 *__restrict__ last,
                                                         unsigned half, float inv_n, float *__restrict__ R, long long r_bs) {
	const float2 *z = Z + (long long) blockIdx.y * z_bs;
	float *r = R + (long long) blockIdx.y * r_bs;
	for (unsigned k = blockIdx.x * blockDim.x + threadIdx.x; k < half; k += gridDim.x * blockDim.x) {
		float2 x0, x1;
		real_split(z[k], z[(half - k) & (half - 1)], __ldg(last + k), x0, x1);
		r[k] = mag_exact(x0.x * inv_n, x0.y * inv_n);
		r[k + half] = mag_exact(x1.x * inv_n, x1.y * inv_n);
	}
}
// inverse (no scaling, conjugate twiddle): the N complex outputs
__global__ void __launch_bounds__(256) k_real_inv_finish(const float2 *__restrict__ Z, long long z_bs, const float2 *__restrict__ last,
                                                         unsigned half, float2 *__restrict__ Y, long long y_bs) {
	const float2 *z = Z + (long long) blockIdx.y * z_bs;
	float2 *y = Y + (long long) blockIdx.y * y_bs;
	for (unsigned k = blockIdx.x * blockDim.x + threadIdx.x; k < half; k += gridDim.x * blockDim.x) {
		const float2 w = __ldg(last + k);
		float2 x0, x1;
		real_split(z[k], z[(half - k) & (half - 1)], make_float2(w.x, -w.y), x0, x1);
		y[k] = x0; y[k + half] = x1;
	}
}

// the same, but only the lags a caller will read: lags [lo0, hi0) and [lo1, hi1), all below `half` (the frame-rate detector's
// two windows, frameratedetector.c:91-95): the kernel touches (hi0-lo0)+(hi1-lo1) lags instead of N
__global__ void __launch_bounds__(256) k_real_inv_finish_win(const float2 *__restrict__ Z, long long z_bs, const float2 *__restrict__ last,
                                                             unsigned half, float2 *__restrict__ Y, long long y_bs, unsigned lo0, unsigned hi0, unsigned lo1, unsigned hi1) {
	const float2 *z = Z + (long long) blockIdx.y * z_bs;
	float2 *y = Y + (long long) blockIdx.y * y_bs;
	const unsigned n0 = hi0 - lo0, total = n0 + (hi1 - lo1);
	for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
		const unsigned k = (t < n0) ? (lo0 + t) : (lo1 + (t - n0));
		const float2 w = __ldg(last + k);
		float2 x0, x1;
		real_split(z[k], z[(half - k) & (half - 1)], make_float2(w.x, -w.y), x0, x1);
		y[k] = x0;
	}
}

// a = (aI*bI + aQ*bQ, aI*bQ - aQ*bI)                                   (fft.c:80-89)
__global__ void k_conj_mul(float2 *a, const float2 *b, unsigned long long n) {
	for (unsigned long long i = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long) gridDim.x * blockDim.x) {
		const float2 x = a[i], y = b[i];
		a[i] = make_float2(__fadd_rn(__fmul_rn(x.x, y.x), __fmul_rn(x.y, y.y)), __fsub_rn(__fmul_rn(x.x, y.y), __fmul_rn(x.y, y.x)));
	}
}
// running mean of lag magnitudes in double                             (frameratedetector.c:34-62)
__global__ void k_accumulate(double *out, unsigned long long calls, const float2 *in, int startid, int length) {
	const double now_n = (double) calls, before_n = (double) (calls - 1);
	for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < length; i += gridDim.x * blockDim.x) {
		const float2 v = in[(size_t) startid + i];
		const double re = (double) v.x, im = (double) v.y;
		const double mag = __dsqrt_rn(__dadd_rn(__dmul_rn(re, re), __dmul_rn(im, im)));
		out[i] = (calls == 0) ? mag : __ddiv_rn(__dadd_rn(__dmul_rn(out[i], before_n), mag), now_n);
	}
}
// the same running mean for `batch` consecutive captures in order (one launch instead of `batch`)
__global__ void k_accumulate_batch(double *out, unsigned long long first_calls, const float2 *in, long long in_stride, unsigned batch,
                                   int startid, int length) {
	for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < length; i += gridDim.x * blockDim.x) {
		double acc = out[i];
		for (unsigned b = 0; b < batch; b++) {
			const unsigned long long calls = first_calls + b;
			const float2 v = in[(size_t) b * in_stride + startid + i];
			const double re = (double) v.x, im = (double) v.y;
			const double mag = __dsqrt_rn(__dadd_rn(__dmul_rn(re, re), __dmul_rn(im, im)));
			acc = (calls == 0) ? mag : __ddiv_rn(__dadd_rn(__dmul_rn(acc, (double) (calls - 1)), mag), (double) calls);
		}
		out[i] = acc;
	}
}
// SURVEY 8f-3 on the device: the index of the first strict maximum of each running-mean plot, the pick the GUI makes on the
// host (PlotVisualizer.java:203-236: start from element 0, move on a strict '>').  One CTA per plot; NaN never wins, a NaN in
// element 0 keeps index 0 (nothing compares greater than it), equal values keep the smallest index.
__global__ void __launch_bounds__(1024) k_plot_peaks(const double *p0, int n0, const double *p1, int n1, int *peaks) {
	__shared__ double s_v[32]; __shared__ int s_i[32];
	const double *v = blockIdx.x ? p1 : p0;
	const int n = blockIdx.x ? n1 : n0;
	double best = -INFINITY; int bi = 0x7fffffff;
	for (int i0 = threadIdx.x; i0 < n; i0 += 8 * (int) blockDim.x) {      // eight loads in flight per thread, folded in index order
		double x[8];
		#pragma unroll
		for (int u = 0; u < 8; u++) { const int i = i0 + u * (int) blockDim.x; x[u] = (i < n) ? v[i] : -INFINITY; }
		#pragma unroll
		for (int u = 0; u < 8; u++) { const int i = i0 + u * (int) blockDim.x; if (i < n && (x[u] > best || (x[u] == best && i < bi))) { best = x[u]; bi = i; } }
	}
	for (int o = 16; o > 0; o >>= 1) {
		const double ov = __shfl_xor_sync(0xffffffffu, best, o); const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
		if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
	}
	if ((threadIdx.x & 31) == 0) { s_v[threadIdx.x >> 5] = best; s_i[threadIdx.x >> 5] = bi; }
	__syncthreads();
	if (threadIdx.x == 0) {
		for (int w = 1; w < (int) (blockDim.x >> 5); w++) if (s_v[w] > best || (s_v[w] == best && s_i[w] < bi)) { best = s_v[w]; bi = s_i[w]; }
		const double first = n > 0 ? v[0] : 0.0;
		peaks[blockIdx.x] = (n <= 0 || first != first || bi == 0x7fffffff) ? 0 : bi;
	}
}
// the scan (channelizer.cu): the running means of K channels at once, one capture each.  Channel y's answer starts at
// in + y * in_stride, its plots at out + y * out_stride ([frame window | line window]); the same arithmetic as k_accumulate_batch
// with batch = 1.
__global__ void k_accumulate_channels(double *out, long long out_stride, unsigned long long calls, const float2 *in, long long in_stride,
                                      int fmin, int flen, int lmin, int llen) {
	double *o = out + (long long) blockIdx.y * out_stride;
	const float2 *a = in + (long long) blockIdx.y * in_stride;
	for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < flen + llen; i += gridDim.x * blockDim.x) {
		const float2 v = a[i < flen ? fmin + i : lmin + (i - flen)];
		const double re = (double) v.x, im = (double) v.y;
		const double mag = __dsqrt_rn(__dadd_rn(__dmul_rn(re, re), __dmul_rn(im, im)));
		o[i] = (calls == 0) ? mag : __ddiv_rn(__dadd_rn(__dmul_rn(o[i], (double) (calls - 1)), mag), (double) calls);
	}
}
// One CTA per plot of every channel (CTA b: channel b / 2, frame plot for even b, line plot for odd b): the first strict maximum
// with k_plot_peaks's rule, and score = (max - mean) / std over the plot (population std; 0 when std is 0), sums in double.
__global__ void __launch_bounds__(1024) k_plot_scores(const double *plots, long long stride, int flen, int llen, TsdrScanPeak *res) {
	__shared__ double s_v[32], s_s[32], s_q[32]; __shared__ int s_i[32];
	const double *v = plots + (long long) (blockIdx.x >> 1) * stride + ((blockIdx.x & 1) ? flen : 0);
	const int n = (blockIdx.x & 1) ? llen : flen;
	double best = -INFINITY, sum = 0.0, sq = 0.0; int bi = 0x7fffffff;
	for (int i = threadIdx.x; i < n; i += blockDim.x) {
		const double x = v[i];
		if (x > best) { best = x; bi = i; }                      // i grows within a thread: '>' keeps the smallest index of a tie
		sum += x; sq = fma(x, x, sq);
	}
	for (int o = 16; o > 0; o >>= 1) {
		const double ov = __shfl_xor_sync(0xffffffffu, best, o); const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
		if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
		sum += __shfl_xor_sync(0xffffffffu, sum, o); sq += __shfl_xor_sync(0xffffffffu, sq, o);
	}
	if ((threadIdx.x & 31) == 0) { s_v[threadIdx.x >> 5] = best; s_i[threadIdx.x >> 5] = bi; s_s[threadIdx.x >> 5] = sum; s_q[threadIdx.x >> 5] = sq; }
	__syncthreads();
	if (threadIdx.x == 0) {
		for (int w = 1; w < (int) (blockDim.x >> 5); w++) {
			if (s_v[w] > best || (s_v[w] == best && s_i[w] < bi)) { best = s_v[w]; bi = s_i[w]; }
			sum += s_s[w]; sq += s_q[w];
		}
		const double first = n > 0 ? v[0] : 0.0;
		const int idx = (n <= 0 || first != first || bi == 0x7fffffff) ? 0 : bi;
		double score = 0.0;
		if (n > 0) {
			const double mean = sum / n, var = sq / n - mean * mean, sd = var > 0.0 ? sqrt(var) : 0.0;
			score = sd > 0.0 ? (v[idx] - mean) / sd : 0.0;
		}
		res[blockIdx.x].score = score; res[blockIdx.x].index = idx;
	}
}
// first difference of magnitudes, out of place                          (superbandwidth.c:67-81)
__global__ void k_abs_diff(const float2 *src, float2 *dst, unsigned long long pairs) {
	for (unsigned long long i = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x; i < pairs; i += (unsigned long long) gridDim.x * blockDim.x) {
		const float2 v = src[i];
		const float cur = mag_exact(v.x, v.y);
		float prev;
		if (i == 0) prev = __fadd_rn(__fmul_rn(v.x, v.x), __fmul_rn(v.y, v.y));    // seed without the square root
		else { const float2 u = src[i - 1]; prev = mag_exact(u.x, u.y); }
		dst[i] = make_float2(__fsub_rn(cur, prev), 0.0f);
	}
}
// rotate left by `shift` complex elements
__global__ void k_rotate(const float2 *src, float2 *dst, unsigned long long n, unsigned long long shift) {
	for (unsigned long long i = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long) gridDim.x * blockDim.x) {
		unsigned long long s = i + shift; if (s >= n) s -= n;
		dst[i] = src[s];
	}
}
// argmax of |x| over [0, n): first maximum wins                         (superbandwidth.c:100-116)
// Two steps over the whole chip instead of one CTA: every CTA reduces a contiguous chunk to (value, index), the last step
// (one CTA) reduces the partials.  "First maximum" = smallest index among equal values, so the result does not depend on
// how the range is cut; the reference starts from element 0 and only moves on a strict '>' (NaN never wins).
__device__ __forceinline__ void argmax_merge(float &best, unsigned &bi, float ov, unsigned oi) {
	if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
}
__device__ __forceinline__ void argmax_block_reduce(float &best, unsigned &bi, float *s_v, unsigned *s_i) {
	for (int o = 16; o > 0; o >>= 1) argmax_merge(best, bi, __shfl_xor_sync(0xffffffffu, best, o), __shfl_xor_sync(0xffffffffu, bi, o));
	if ((threadIdx.x & 31) == 0) { s_v[threadIdx.x >> 5] = best; s_i[threadIdx.x >> 5] = bi; }
	__syncthreads();
	if (threadIdx.x == 0) for (int w = 1; w < (int) (blockDim.x >> 5); w++) argmax_merge(best, bi, s_v[w], s_i[w]);
}
__global__ void __launch_bounds__(256) k_argmax_partial(const float2 *__restrict__ x, unsigned n, float *__restrict__ pv, unsigned *__restrict__ pi) {
	__shared__ float s_v[8]; __shared__ unsigned s_i[8];
	const unsigned per = (n + gridDim.x - 1) / gridDim.x, lo = blockIdx.x * per, hi = min(n, lo + per);
	float best = -1.0f; unsigned bi = 0xffffffffu;
	for (unsigned i = lo + threadIdx.x; i < hi; i += blockDim.x) {
		const float2 v = __ldg(x + i);
		const float m = mag_exact(v.x, v.y);
		if (m > best) { best = m; bi = i; }              // a thread walks upwards: the first of equal values stays
	}
	argmax_block_reduce(best, bi, s_v, s_i);
	if (threadIdx.x == 0) { pv[blockIdx.x] = best; pi[blockIdx.x] = bi; }
}
__global__ void __launch_bounds__(256) k_argmax_final(const float *__restrict__ pv, const unsigned *__restrict__ pi, unsigned parts, int *result) {
	__shared__ float s_v[8]; __shared__ unsigned s_i[8];
	float best = -1.0f; unsigned bi = 0xffffffffu;
	for (unsigned i = threadIdx.x; i < parts; i += blockDim.x) argmax_merge(best, bi, pv[i], pi[i]);
	argmax_block_reduce(best, bi, s_v, s_i);
	if (threadIdx.x == 0) *result = (bi == 0xffffffffu) ? 0 : (int) bi;
}
// rotate left by *shift complex elements, the shift read from device memory (the lag the kernels before produced)
__global__ void k_rotate_dev(const float2 *src, float2 *dst, unsigned long long n, const int *shift_) {
	const unsigned long long shift = (unsigned long long) *shift_;
	for (unsigned long long i = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long) gridDim.x * blockDim.x) {
		unsigned long long s = i + shift; if (s >= n) s -= n;
		dst[i] = src[s];
	}
}
// U_s[m] = e^{+2 pi i m s/(H N)} * sum_q e^{+2 pi i q s / H} X_q[m]     (DESIGN.md, superbandwidth decomposition)
__global__ void k_residue_mix(const float2 *gathered, int H, unsigned n, int s, float2 *dst) {
	for (unsigned m = blockIdx.x * blockDim.x + threadIdx.x; m < n; m += gridDim.x * blockDim.x) {
		double accr = 0.0, acci = 0.0;
		for (int q = 0; q < H; q++) {
			double sn, cs;
			sincospi(2.0 * (double) ((q * s) % H) / (double) H, &sn, &cs);
			const float2 v = gathered[(size_t) q * n + m];
			accr += cs * v.x - sn * v.y; acci += cs * v.y + sn * v.x;
		}
		double sn, cs;
		sincospi(2.0 * ((double) m * (double) s) / ((double) H * (double) n), &sn, &cs);
		dst[m] = make_float2((float) (accr * cs - acci * sn), (float) (accr * sn + acci * cs));
	}
}

// multi-GPU stitch with the alignment folded into the spectrum: rotating hop q left by lag_q samples multiplies its
// spectrum by e^{+2 pi i m lag_q / N}, so ranks exchange RAW spectra and apply the ramp after the gather:
// U_s[m] = e^{+2 pi i m s/(H N)} * sum_q e^{+2 pi i (q s / H + m lag_q / N)} X_q[m]
struct LagSet { int lag[16]; };
__global__ void k_residue_mix_lag(const float2 *gathered, long long block_stride, int H, unsigned n, int s, LagSet lags, float2 *dst) {
	for (unsigned m = blockIdx.x * blockDim.x + threadIdx.x; m < n; m += gridDim.x * blockDim.x) {
		float accr = 0.0f, acci = 0.0f;
		for (int q = 0; q < H; q++) {
			// phase = 2 pi (q s / H + m lag / N): both terms reduced exactly in integers before the division
			const unsigned long long e = ((unsigned long long) m * (unsigned long long) lags.lag[q]) & (unsigned long long) (n - 1);
			const double frac = (double) e / (double) n + (double) ((q * s) % H) / (double) H;
			float sn, cs;
			sincospif((float) (2.0 * (frac - floor(frac))), &sn, &cs);
			const float2 v = gathered[(size_t) q * block_stride + m];
			accr += cs * v.x - sn * v.y; acci += cs * v.y + sn * v.x;
		}
		double dsn, dcs;
		sincospi(2.0 * ((double) m * (double) s) / ((double) H * (double) n), &dsn, &dcs);
		const float sn = (float) dsn, cs = (float) dcs;
		dst[m] = make_float2(accr * cs - acci * sn, accr * sn + acci * cs);
	}
}

inline unsigned grid1d(unsigned long long n, int sm_count) {
	const unsigned long long want = (n + 255) / 256, cap = (unsigned long long) sm_count * 8;
	return (unsigned) (want < cap ? (want ? want : 1) : cap);
}

bool g_attr_set[64] = {false};      // per device: the pass kernels' dynamic shared-memory limit has been raised
// per-pass layer-twiddle tables (see fft_pass_kernel), built on the host in double precision and cached
struct StageTab { int device, log2L, l_base, pert; float2 *d; };
std::vector<StageTab> g_stage_tabs;
std::mutex g_tw_mu;

int stage_table(tsdrgpu_ctx_t *ctx, int log2L, int l_base, const double *eps_all, const float2 **out) {
	static const bool exact_dft = getenv("TSDRGPU_FFT_TRUE_DFT") != NULL;      // opt out: the mathematically exact DFT
	double eps[FFT_MAX_LOG2L + 1];
	int pert = 0;
	for (int sidx = 0; sidx < log2L; sidx++) {
		eps[sidx] = (!exact_dft && eps_all && l_base + sidx < 40) ? eps_all[l_base + sidx] : 0.0;
		if (eps[sidx] != 0.0) pert = 1;
	}
	std::lock_guard<std::mutex> lock(g_tw_mu);
	for (auto &t : g_stage_tabs) if (t.device == ctx->device && t.log2L == log2L && t.l_base == (pert ? l_base : -1) && t.pert == pert) { *out = t.d; return TSDRGPU_OK; }
	const int L = 1 << log2L;
	std::vector<float2> h((size_t) L);
	for (int sidx = 0; sidx < log2L; sidx++) {
		const int blk = 1 << sidx;
		for (int K = 0; K < blk; K++) {
			const double ang = -3.14159265358979323846 * ((double) K / (double) blk) * (1.0 + eps[sidx]);
			h[(size_t) blk - 1 + K] = make_float2((float) cos(ang), (float) sin(ang));
		}
	}
	h[(size_t) L - 1] = make_float2(1.0f, 0.0f);
	StageTab t; t.device = ctx->device; t.log2L = log2L; t.l_base = pert ? l_base : -1; t.pert = pert;
	CU_TRY(ctx, cudaMalloc(&t.d, sizeof(float2) * L));
	CU_TRY(ctx, cudaMemcpy(t.d, h.data(), sizeof(float2) * L, cudaMemcpyHostToDevice));
	g_stage_tabs.push_back(t);
	*out = t.d;
	return TSDRGPU_OK;
}

// W_M^(col * L8 * j) for every column of a pass and j = 0..7 (see fft_pass_kernel), built on the host, cached
struct StepTab { int device; unsigned long long M; unsigned ncols, L8; float2 *d; };
std::vector<StepTab> g_step_tabs;
int step_table(tsdrgpu_ctx_t *ctx, unsigned long long M, unsigned ncols, unsigned L8, const float2 **out) {
	std::lock_guard<std::mutex> lock(g_tw_mu);
	for (auto &t : g_step_tabs) if (t.device == ctx->device && t.M == M && t.ncols == ncols && t.L8 == L8) { *out = t.d; return TSDRGPU_OK; }
	std::vector<float2> h((size_t) ncols * 8);
	for (unsigned col = 0; col < ncols; col++)
		for (unsigned j = 0; j < 8; j++) {
			const unsigned long long e = ((unsigned long long) col * (unsigned long long) (L8 * j)) & (M - 1);
			const double ang = -2.0 * 3.14159265358979323846 * ((double) e / (double) M);
			h[(size_t) col * 8 + j] = make_float2((float) cos(ang), (float) sin(ang));
		}
	StepTab t; t.device = ctx->device; t.M = M; t.ncols = ncols; t.L8 = L8;
	CU_TRY(ctx, cudaMalloc(&t.d, sizeof(float2) * h.size()));
	CU_TRY(ctx, cudaMemcpy(t.d, h.data(), sizeof(float2) * h.size(), cudaMemcpyHostToDevice));
	g_step_tabs.push_back(t);
	*out = t.d;
	return TSDRGPU_OK;
}

int ensure_table(tsdrgpu_ctx_t *ctx, cudaStream_t stream) {
	(void) stream;
	if (g_attr_set[ctx->device]) return TSDRGPU_OK;
	const int max_smem = (int) (2 * sizeof(float2) * FFT_MAX_ELEMS);     // ping-pong
#define SET_ATTR(l) CU_TRY(ctx, cudaFuncSetAttribute(fft_pass_kernel<l, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem)); \
	CU_TRY(ctx, cudaFuncSetAttribute(fft_pass_kernel<l, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem)); \
	CU_TRY(ctx, cudaFuncSetAttribute(fft_pass_kernel<l, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem))
	SET_ATTR(3); SET_ATTR(4); SET_ATTR(5); SET_ATTR(6); SET_ATTR(7); SET_ATTR(8); SET_ATTR(9); SET_ATTR(10); SET_ATTR(11);
#undef SET_ATTR
	g_attr_set[ctx->device] = true;
	return TSDRGPU_OK;
}

int bundle_for(int log2L, unsigned long long lines, bool contiguous_lines = false) {
	const int L = 1 << log2L;
	int C = 4096 / L; if (C < 8) C = 8;
	while ((long long) C * L > FFT_MAX_ELEMS) C >>= 1;
	// experiment knob: smaller bundles (more, smaller CTAs per SM) on passes whose lines are contiguous in memory
	static const int small = getenv("TSDRGPU_FFT_SMALL_BUNDLE") ? atoi(getenv("TSDRGPU_FFT_SMALL_BUNDLE")) : 0;
	if (contiguous_lines && small >= 512) while ((long long) C * L > small && C > 1) C >>= 1;
	while ((unsigned long long) C > lines) C >>= 1;
	return C < 1 ? 1 : C;
}

int launch_pass(tsdrgpu_ctx_t *ctx, cudaStream_t stream, const float2 *in, float2 *out, FftPass P, unsigned bundles, int inverse,
                unsigned batch, long long in_bs, long long out_bs, const double *eps_all = NULL, int l_base = 0) {
	P.in_bs = in_bs; P.out_bs = out_bs;
	P.log2C = 0; while ((1 << P.log2C) < P.C) P.log2C++;
	const int L = 1 << P.log2L, total = P.C * L;
	int threads = (total / 8 + 31) / 32 * 32;            // one radix-8 butterfly (8 elements) per thread and stage
	if (threads < 32) threads = 32;
	if (threads > 512) return tsdrgpu_fail(ctx, TSDRGPU_EINVAL, "FFT bundle too large", cudaSuccess, __FILE__, __LINE__);
	const int nstages = P.log2L / 3 + ((P.log2L % 3) ? 1 : 0);
	const dim3 grid(bundles, batch);
	if (P.log2L <= 2) {
		if (P.log2L == 1) KL(ctx, "fft_pass_kernel", stream, fft_tiny_kernel<1><<<dim3(1, batch), 32, 0, stream>>>(in, out, P));
		else KL(ctx, "fft_pass_kernel", stream, fft_tiny_kernel<2><<<dim3(1, batch), 32, 0, stream>>>(in, out, P));
		return TSDRGPU_OK;
	}
	const float2 *stw;
	{ int rc = stage_table(ctx, P.log2L, l_base, eps_all, &stw); if (rc) return rc; }
	P.tw_step = NULL;
	if (P.tw_M && P.tw_M <= (1ull << 24) && P.c_fast_out && P.log2L >= 3 && P.tw_lo == P.C && P.tw_cs == 1) {
		// columns of this pass: col = g_lo * C + c, g_lo < G_lo
		const unsigned ncols = P.G_lo * (unsigned) P.C;
		if (ncols <= (1u << 20)) { int rc = step_table(ctx, P.tw_M, ncols, (unsigned) (L >> 3), &P.tw_step); if (rc) return rc; }
	}
	P.dbg = getenv("TSDRGPU_FFT_DBG") ? atoi(getenv("TSDRGPU_FFT_DBG")) : 0;
	P.exact0 = 1;
	for (int sidx = 0; sidx < 3 && sidx < P.log2L; sidx++) if (eps_all && l_base + sidx < 40 && fabs(eps_all[l_base + sidx]) > 1e-10) P.exact0 = 0;
	// bulk copies (TMA) feed the passes whose lines are contiguous and 16-byte aligned; TSDRGPU_FFT_NO_TMA=1 keeps the plain loads
	static const bool no_tma = getenv("TSDRGPU_FFT_NO_TMA") != NULL;
	const bool tma = !no_tma && !P.c_fast_in && !P.in_real && P.in_js == 1 && P.nfan == 0 && total * 8 == threads * 64
	                 && ((reinterpret_cast<unsigned long long>(in) | ((unsigned long long) in_bs * 8ull)) & 15ull) == 0;
	const size_t smem = sizeof(float2) * (size_t) total * ((nstages >= 3 || (tma && nstages == 2)) ? 2 : 1);
	switch (P.log2L) {
#define CASE(l) case l: if (P.nfan > 0) KL(ctx, "fft_pass_kernel", stream, fft_pass_kernel<l, true, false><<<grid, threads, smem, stream>>>(in, out, P, stw)); \
	                else if (tma) KL(ctx, "fft_pass_kernel", stream, fft_pass_kernel<l, false, true><<<grid, threads, smem, stream>>>(in, out, P, stw)); \
	                else KL(ctx, "fft_pass_kernel", stream, fft_pass_kernel<l, false, false><<<grid, threads, smem, stream>>>(in, out, P, stw)); break
	CASE(3); CASE(4); CASE(5); CASE(6); CASE(7); CASE(8); CASE(9); CASE(10); CASE(11);
#undef CASE
	default: return tsdrgpu_fail(ctx, TSDRGPU_EINVAL, "unsupported FFT line length", cudaSuccess, __FILE__, __LINE__);
	}
	return TSDRGPU_OK;
}

struct FftOpts {
	const float *real_in; bool out_abs; float scale;
	unsigned batch;                 // independent transforms (grid.y)
	long long data_bs, scratch_bs, real_bs;   // distance between consecutive transforms in data (complex), scratch (complex), real_in (floats)
	float2 *const *fan; int nfan;             // forward only: the final pass stores the result to every fan[p] (same layout as `data`) instead of `data`
	const float2 *cplx_in; long long cplx_bs; // the first pass reads its (complex) input from here instead of `data` (which is then output only)
	const float *pair_in; long long pair_bs;  // the same, but the input is pairs of floats with 4-byte alignment only; pair_bs in FLOATS
	float *abs_real;                          // with out_abs (batch 1): the final pass stores |.| as float32 here (peer memory allowed) and leaves `data` alone
};

// N-point transform of `data` (complex, natural order) through `scratch`; result lands in `data`.
// With opts.real_in the input is read from a real array instead (data is output only).
int fft_run(tsdrgpu_ctx_t *ctx, cudaStream_t stream, float2 *data, float2 *scratch, unsigned log2N, int inverse, FftOpts o) {
	const unsigned long long N = 1ull << log2N;
	const float2 *src0 = o.real_in ? reinterpret_cast<const float2 *>(o.real_in) : (o.pair_in ? reinterpret_cast<const float2 *>(o.pair_in) : (o.cplx_in ? o.cplx_in : data));
	const long long in0_bs = o.real_in ? o.real_bs : (o.pair_in ? o.pair_bs : (o.cplx_in ? o.cplx_bs : o.data_bs));
	const int in_mode = o.real_in ? 1 : (o.pair_in ? 2 : 0);
	double eps_all[40];
	tsdrgpu_fft_reference_eps((int) log2N < 40 ? (int) log2N : 40, inverse, eps_all);
	FftPass P; memset(&P, 0, sizeof P);
	auto with_fan = [&](FftPass &F) {                   // the pass that produces the final result
		F.nfan = 0;
		if (o.fan && o.nfan > 0 && !inverse) { F.nfan = o.nfan < 16 ? o.nfan : 16; for (int q = 0; q < F.nfan; q++) F.fan[q] = o.fan[q]; }
	};
	if (log2N <= FFT_MAX_LOG2L) {                       // one pass, one CTA
		P.log2L = (int) log2N; P.C = 1; P.G_lo = 1; P.in_js = 1; P.out_ks = 1; P.scale = o.scale;
		P.in_real = in_mode; P.out_abs = o.out_abs; P.abs_real = o.out_abs ? o.abs_real : NULL;
		with_fan(P);
		P.conj_in = P.conj_out = inverse ? 1 : 0;
		return launch_pass(ctx, stream, src0, data, P, 1, inverse, o.batch, in0_bs, o.data_bs, eps_all, 0);
	}
	int rc;
	// two passes up to 2^21 (1024 x 2048: the 2048-point lines go to the contiguous pass, one TMA bulk copy per 2-line bundle);
	// TSDRGPU_FFT_2PASS_MAX=20 restores three passes at 2^21 for comparison
	static const unsigned two_pass_max = getenv("TSDRGPU_FFT_2PASS_MAX") ? (unsigned) atoi(getenv("TSDRGPU_FFT_2PASS_MAX")) : 21u;
	if (log2N <= two_pass_max && log2N <= 22) {         // N = N1 * N2 ; n = N2*n1 + n2 ; k = k1 + N1*k2
		// odd log2 N: the SHORTER line goes to the strided pass (bundle of 8 columns = 64-byte runs instead of 4 = 32-byte runs on
		// both its loads and its stores); TSDRGPU_FFT_SPLIT=ceil restores the other split for comparison
		static const bool split_ceil = getenv("TSDRGPU_FFT_SPLIT") && !strcmp(getenv("TSDRGPU_FFT_SPLIT"), "ceil");
		const unsigned l1 = split_ceil ? (log2N + 1) / 2 : log2N / 2, l2 = log2N - l1;
		const unsigned long long N1 = 1ull << l1, N2 = 1ull << l2;
		P.log2L = (int) l1; P.C = bundle_for((int) l1, N2); P.c_fast_in = P.c_fast_out = 1;
		P.G_lo = (unsigned) (N2 / P.C);
		P.in_lo = P.C; P.in_cs = 1; P.in_js = (long long) N2;
		P.out_lo = P.C; P.out_cs = 1; P.out_ks = (long long) N2;
		P.tw_M = N; P.tw_lo = P.C; P.tw_cs = 1; P.scale = 1.0f; P.in_real = in_mode;
		P.conj_in = inverse ? 1 : 0;
		if ((rc = launch_pass(ctx, stream, src0, scratch, P, P.G_lo, inverse, o.batch, in0_bs, o.scratch_bs, eps_all, 0))) return rc;
		FftPass Q; memset(&Q, 0, sizeof Q);
		Q.log2L = (int) l2; Q.C = bundle_for((int) l2, N1, true); Q.c_fast_in = 0; Q.c_fast_out = 1;
		Q.G_lo = (unsigned) (N1 / Q.C);
		Q.in_lo = (long long) Q.C * (long long) N2; Q.in_cs = (long long) N2; Q.in_js = 1;
		Q.out_lo = Q.C; Q.out_cs = 1; Q.out_ks = (long long) N1;
		Q.scale = o.scale; Q.out_abs = o.out_abs; Q.abs_real = o.out_abs ? o.abs_real : NULL;
		with_fan(Q);
		Q.conj_out = inverse ? 1 : 0;
		return launch_pass(ctx, stream, scratch, data, Q, Q.G_lo, inverse, o.batch, o.scratch_bs, o.data_bs, eps_all, (int) l1);
	}
	// N = N1*N2*N3 ; n = N2N3 n1 + N3 n2 + n3 ; k = k1 + N1 k2 + N1N2 k3
	const unsigned l1 = (log2N + 2) / 3, l2 = (log2N - l1 + 1) / 2, l3 = log2N - l1 - l2;
	if (l1 > (unsigned) FFT_MAX_LOG2L) return tsdrgpu_fail(ctx, TSDRGPU_EINVAL, "FFT too long", cudaSuccess, __FILE__, __LINE__);
	const unsigned long long N1 = 1ull << l1, N2 = 1ull << l2, N3 = 1ull << l3, N23 = N2 * N3;
	{   // pass A: length N1 along stride N2N3, bundle over adjacent columns m
		P.log2L = (int) l1; P.C = bundle_for((int) l1, N23); P.c_fast_in = P.c_fast_out = 1;
		P.G_lo = (unsigned) (N23 / P.C);
		P.in_lo = P.C; P.in_cs = 1; P.in_js = (long long) N23;
		P.out_lo = P.C; P.out_cs = 1; P.out_ks = (long long) N23;
		P.tw_M = N; P.tw_lo = P.C; P.tw_cs = 1; P.scale = 1.0f; P.in_real = in_mode;
		P.conj_in = inverse ? 1 : 0;
		if ((rc = launch_pass(ctx, stream, src0, scratch, P, P.G_lo, inverse, o.batch, in0_bs, o.scratch_bs, eps_all, 0))) return rc;
	}
	{   // pass B: for every k1, length N2 along stride N3, bundle over adjacent n3 (in place in scratch)
		FftPass B; memset(&B, 0, sizeof B);
		B.log2L = (int) l2; B.C = bundle_for((int) l2, N3); B.c_fast_in = B.c_fast_out = 1;
		B.G_lo = (unsigned) (N3 / B.C);
		B.in_hi = (long long) N23; B.in_lo = B.C; B.in_cs = 1; B.in_js = (long long) N3;
		B.out_hi = (long long) N23; B.out_lo = B.C; B.out_cs = 1; B.out_ks = (long long) N3;
		B.tw_M = N23; B.tw_lo = B.C; B.tw_cs = 1; B.scale = 1.0f;
		if ((rc = launch_pass(ctx, stream, scratch, scratch, B, (unsigned) (N1 * B.G_lo), inverse, o.batch, o.scratch_bs, o.scratch_bs, eps_all, (int) l1))) return rc;
	}
	{   // pass C: contiguous lines of N3 at (k1,k2); bundle over adjacent k1; output k1 + N1 k2 + N1N2 k3
		FftPass Cc; memset(&Cc, 0, sizeof Cc);
		Cc.log2L = (int) l3; Cc.C = bundle_for((int) l3, N1, true); Cc.c_fast_in = 0; Cc.c_fast_out = 1;
		Cc.G_lo = (unsigned) (N1 / Cc.C);                // g = k2 * G_lo + (k1 / C)
		Cc.in_hi = (long long) N3; Cc.in_lo = (long long) Cc.C * (long long) N23; Cc.in_cs = (long long) N23; Cc.in_js = 1;
		Cc.out_hi = (long long) N1; Cc.out_lo = Cc.C; Cc.out_cs = 1; Cc.out_ks = (long long) (N1 * N2);
		Cc.scale = o.scale; Cc.out_abs = o.out_abs; Cc.abs_real = o.out_abs ? o.abs_real : NULL;
		with_fan(Cc);
		Cc.conj_out = inverse ? 1 : 0;
		return launch_pass(ctx, stream, scratch, data, Cc, (unsigned) (N2 * Cc.G_lo), inverse, o.batch, o.scratch_bs, o.data_bs, eps_all, (int) (l1 + l2));
	}
}

unsigned ilog2(unsigned long long n) { unsigned m = 0; while ((n >>= 1) != 0) m++; return m; }

}  // namespace

// internal entry used by other translation units
int tsdrgpu_fft_internal(tsdrgpu_ctx_t *ctx, cudaStream_t stream, float2 *data, unsigned long long n_pow2, int inverse) {
	int rc = ensure_table(ctx, stream);
	if (rc) return rc;
	if (n_pow2 <= 1) return TSDRGPU_OK;
	void *scratch;
	if ((rc = tsdrgpu_scratch(ctx, 0, sizeof(float2) * n_pow2, &scratch))) return rc;
	FftOpts o; memset(&o, 0, sizeof o); o.batch = 1; o.scale = inverse ? 1.0f : 1.0f / (float) n_pow2;
	return fft_run(ctx, stream, data, (float2 *) scratch, ilog2(n_pow2), inverse, o);
}

// out of place: out = FFT(in), both n_pow2 complex, `in` untouched
int tsdrgpu_fft_oop_internal(tsdrgpu_ctx_t *ctx, cudaStream_t stream, const float2 *in, float2 *out, unsigned long long n_pow2, int inverse) {
	int rc = ensure_table(ctx, stream);
	if (rc) return rc;
	if (n_pow2 <= 1) { if (n_pow2 == 1) CU_TRY(ctx, cudaMemcpyAsync(out, in, sizeof(float2), cudaMemcpyDeviceToDevice, stream)); return TSDRGPU_OK; }
	void *scratch;
	if ((rc = tsdrgpu_scratch(ctx, 0, sizeof(float2) * n_pow2, &scratch))) return rc;
	FftOpts o; memset(&o, 0, sizeof o); o.batch = 1; o.scale = inverse ? 1.0f : 1.0f / (float) n_pow2;
	o.cplx_in = in; o.cplx_bs = 0;
	return fft_run(ctx, stream, out, (float2 *) scratch, ilog2(n_pow2), inverse, o);
}
// `batch` independent out-of-place transforms (transform b reads in + b*in_bs, writes out + b*out_bs) through a scratch area the
// CALLER owns (batch * n_pow2 complex; NULL: the context's scratch slot 0) -- for callers that run transforms on two streams at once
int tsdrgpu_fft_batch_internal(tsdrgpu_ctx_t *ctx, cudaStream_t stream, const float2 *in, long long in_bs, float2 *out, long long out_bs,
                               float2 *scratch, unsigned long long n_pow2, unsigned batch, int inverse) {
	int rc = ensure_table(ctx, stream);
	if (rc) return rc;
	ARG_TRY(ctx, n_pow2 >= 2 && batch >= 1);
	if (!scratch) {
		void *sc;
		if ((rc = tsdrgpu_scratch(ctx, 0, sizeof(float2) * n_pow2 * batch, &sc))) return rc;
		scratch = (float2 *) sc;
	}
	FftOpts o; memset(&o, 0, sizeof o); o.batch = batch; o.scale = inverse ? 1.0f : 1.0f / (float) n_pow2;
	o.cplx_in = in; o.cplx_bs = in_bs; o.data_bs = out_bs; o.scratch_bs = (long long) n_pow2;
	return fft_run(ctx, stream, out, scratch, ilog2(n_pow2), inverse, o);
}
// inverse transform of `data` (n_pow2 complex, clobbered) whose final pass stores |y| as float32 straight into real_out (n_pow2
// floats; peer memory allowed: the stores of the last butterflies ARE the transfer)
int tsdrgpu_ifft_abs_internal(tsdrgpu_ctx_t *ctx, cudaStream_t stream, float2 *data, float *real_out, unsigned long long n_pow2) {
	int rc = ensure_table(ctx, stream);
	if (rc) return rc;
	ARG_TRY(ctx, n_pow2 >= 8);
	void *scratch;
	if ((rc = tsdrgpu_scratch(ctx, 0, sizeof(float2) * n_pow2, &scratch))) return rc;
	FftOpts o; memset(&o, 0, sizeof o); o.batch = 1; o.scale = 1.0f; o.out_abs = true; o.abs_real = real_out;
	return fft_run(ctx, stream, data, (float2 *) scratch, ilog2(n_pow2), 1, o);
}
// *d_result = index of the first maximum of |x[0..n)|; d_part: room for 2 * TSDRGPU_ARGMAX_PARTS 32-bit words
int tsdrgpu_argmax_mag_internal(tsdrgpu_ctx_t *ctx, cudaStream_t stream, const float2 *x, unsigned n, void *d_part, int *d_result) {
	unsigned parts = (n + 4095) / 4096; if (parts > TSDRGPU_ARGMAX_PARTS) parts = TSDRGPU_ARGMAX_PARTS; if (parts < 1) parts = 1;
	float *pv = (float *) d_part; unsigned *pi = (unsigned *) d_part + TSDRGPU_ARGMAX_PARTS;
	KL(ctx, "k_argmax", stream, k_argmax_partial<<<parts, 256, 0, stream>>>(x, n, pv, pi));
	KL(ctx, "k_argmax", stream, k_argmax_final<<<1, 256, 0, stream>>>(pv, pi, parts, d_result));
	return TSDRGPU_OK;
}

struct tsdrgpu_frd {
	tsdrgpu_ctx_t *ctx;
	float *d_big; size_t big_cap;                 // extbuff (2*size floats)
	double *d_p1, *d_p2; size_t p1_cap, p2_cap;   // the two running means
	uint64_t calls; int fresh;
	int *d_peaks;                                 // first strict maximum of each plot (k_plot_peaks), refreshed with every run
	// overlapped mode (tsdrgpu_frd_set_overlap): everything a run launches goes to an internal stream, behind what the caller's
	// stream held at the call, with work buffers of its own -- the transforms then share the chip with whatever the caller
	// enqueues next (the pass kernels are bound by issue slots, the resampler and the frame stage by other things)
	int overlap, pending;
	cudaStream_t s_side; cudaEvent_t ev_in, ev_done;
	float2 *w0, *w1; size_t w0_cap, w1_cap;
};

extern "C" {

uint32_t tsdrgpu_fft_getrealsize(uint32_t size) {          // fft.c:5-11
	uint32_t m = 0;
	while ((size /= 2) != 0) m++;
	return 1u << m;
}

int tsdrgpu_fft(tsdrgpu_ctx_t *ctx, void *stream, float *d_iq, uint32_t size, int inverse) {
	BIND(ctx); ARG_TRY(ctx, d_iq != NULL);
	if (size == 0) return TSDRGPU_OK;
	return tsdrgpu_fft_internal(ctx, (cudaStream_t) stream, reinterpret_cast<float2 *>(d_iq), tsdrgpu_fft_getrealsize(size), inverse);
}

// batch of independent autocorrelations: transform b reads d_real + b*real_stride (floats) and writes
// d_answer + b*answer_stride (floats, 2*size each).  skip_tail leaves answer[2N .. 2*size) untouched (the
// frame-rate detector never reads lags >= N).
// last[k] = exp(-i pi k / half (1 + eps)), k < half: the reference's final radix-2 stage of an (2 half)-point transform
struct LastTab { int device; unsigned half; double eps; float2 *d; };
static std::vector<LastTab> g_last_tabs;
static int last_stage_table(tsdrgpu_ctx_t *ctx, unsigned half, double eps, const float2 **out) {
	std::lock_guard<std::mutex> lock(g_tw_mu);
	for (auto &t : g_last_tabs) if (t.device == ctx->device && t.half == half && t.eps == eps) { *out = t.d; return TSDRGPU_OK; }
	std::vector<float2> h(half);
	for (unsigned k = 0; k < half; k++) {
		const double ang = -3.14159265358979323846 * ((double) k / (double) half) * (1.0 + eps);
		h[k] = make_float2((float) cos(ang), (float) sin(ang));
	}
	LastTab t; t.device = ctx->device; t.half = half; t.eps = eps;
	CU_TRY(ctx, cudaMalloc(&t.d, sizeof(float2) * half));
	CU_TRY(ctx, cudaMemcpy(t.d, h.data(), sizeof(float2) * half, cudaMemcpyHostToDevice));
	g_last_tabs.push_back(t);
	*out = t.d;
	return TSDRGPU_OK;
}

// Default path (measured +15.6 % on the whole step in round 1; TSDRGPU_AUTOCORR_FULL=1 opts out): both transforms of the
// autocorrelation at half size.  The capture and |X|/N are
// real; a real sequence of length N is a complex one of length N/2, one N/2-point transform + the reference's last radix-2
// stage (k_real_*_finish) gives the N-point result.  profiles/studies/real_input_autocorr_study.py measures the only
// approximation (the mirror identity under perturbed stage angles): 6.6e-10 of the zero-lag peak at 2^20, 7.9e-9 at 2^22.
struct LagWindows { unsigned lo0, hi0, lo1, hi1; };      // only these lags of every answer are needed (all zero: every lag)

// How many captures share one pair of work buffers (TSDRGPU_AUTOCORR_GROUP; default: the whole batch).  Small groups would keep
// the intermediates of the four passes inside the 126 MB L2 instead of streaming them through HBM; measured on the B200
// (profiles/studies/autocorr_group_sweep.py, 19 captures of 2^20): 41.6 / 22.4 / 20.4 / 17.4 / 17.1 us per capture at groups of
// 1 / 4 / 6 / 10 / 19 -- the pass kernel is bound by issue slots and shared-memory traffic, not by HBM, so what small groups buy
// in L2 hits they lose twice over in partial waves (128 CTAs per capture on 444 resident slots).  The knob stays for studies.
static unsigned autocorr_group(unsigned long long N, unsigned batch) {
	(void) N;
	const int forced = getenv("TSDRGPU_AUTOCORR_GROUP") ? atoi(getenv("TSDRGPU_AUTOCORR_GROUP")) : 0;       // read per call
	if (forced > 0 && (unsigned) forced < batch) return (unsigned) forced;
	return batch;
}

struct WorkBufs { float2 *w0, *w1; };                     // caller-owned work buffers (NULL: the context's scratch slots 0 and 1)
static int autocorrelation_batch_half(tsdrgpu_ctx_t *ctx, cudaStream_t stream, float2 *ans, long long ans_bs, const float *d_real,
                                      long long real_stride, unsigned long long N, unsigned batch, LagWindows win, WorkBufs wb) {
	const unsigned log2N = ilog2(N), half = (unsigned) (N >> 1);
	double eps_all[40];
	tsdrgpu_fft_reference_eps((int) log2N, 0, eps_all);
	static const bool exact_dft = getenv("TSDRGPU_FFT_TRUE_DFT") != NULL;
	const float2 *last;
	int rc = last_stage_table(ctx, half, exact_dft ? 0.0 : eps_all[log2N - 1], &last);
	if (rc) return rc;
	const unsigned G = autocorr_group(N, batch);
	void *w0_ = wb.w0, *w1_ = wb.w1;
	if (!w0_ && (rc = tsdrgpu_scratch(ctx, 0, sizeof(float2) * half * G, &w0_))) return rc;
	if (!w1_ && (rc = tsdrgpu_scratch(ctx, 1, sizeof(float2) * half * G, &w1_))) return rc;
	float2 *W0 = (float2 *) w0_, *W1 = (float2 *) w1_;
	const bool windowed = win.hi0 > win.lo0 || win.hi1 > win.lo1;
	for (unsigned g0 = 0; g0 < batch; g0 += G) {
		const unsigned gb = (batch - g0 < G) ? (batch - g0) : G;
		const dim3 grid(grid1d(half, ctx->sm_count), gb);
		// forward: Z = FFT_{N/2}(capture viewed as complex pairs), unscaled: capture -> W0 -> W1
		FftOpts f; memset(&f, 0, sizeof f);
		f.scale = 1.0f; f.batch = gb; f.data_bs = (long long) half; f.scratch_bs = (long long) half;
		const float *cap0 = d_real + (long long) g0 * real_stride;
		if ((real_stride & 1) || (reinterpret_cast<unsigned long long>(cap0) & 7ull)) { f.pair_in = cap0; f.pair_bs = real_stride; }   // odd capture sizes: every other capture starts on an odd sample
		else { f.cplx_in = reinterpret_cast<const float2 *>(cap0); f.cplx_bs = real_stride / 2; }
		if ((rc = fft_run(ctx, stream, W1, W0, log2N - 1, 0, f))) return rc;
		// R = |X| / N as N reals = N/2 complex: W1 -> W0
		KL(ctx, "k_real_fwd_finish", stream, k_real_fwd_finish<<<grid, 256, 0, stream>>>(W1, (long long) half, last, half, 1.0f / (float) N,
		                                                                                  reinterpret_cast<float *>(W0), (long long) N));
		// inverse: Z' = IFFT_{N/2}(R viewed as complex pairs): W0 -> W1 -> W0
		FftOpts gopt; memset(&gopt, 0, sizeof gopt);
		gopt.scale = 1.0f; gopt.batch = gb; gopt.data_bs = (long long) half; gopt.scratch_bs = (long long) half;
		if ((rc = fft_run(ctx, stream, W0, W1, log2N - 1, 1, gopt))) return rc;
		float2 *out = ans + (long long) g0 * ans_bs;
		if (windowed) {
			const unsigned total = (win.hi0 - win.lo0) + (win.hi1 - win.lo1);
			KL(ctx, "k_real_inv_finish", stream, k_real_inv_finish_win<<<dim3(grid1d(total, ctx->sm_count), gb), 256, 0, stream>>>(W0, (long long) half, last, half, out, ans_bs,
				win.lo0, win.hi0, win.lo1, win.hi1));
		} else KL(ctx, "k_real_inv_finish", stream, k_real_inv_finish<<<grid, 256, 0, stream>>>(W0, (long long) half, last, half, out, ans_bs));
	}
	return TSDRGPU_OK;
}

static int autocorrelation_batch(tsdrgpu_ctx_t *ctx, cudaStream_t stream, float *d_answer, long long answer_stride,
                                 const float *d_real, long long real_stride, uint32_t size, unsigned batch, bool skip_tail, LagWindows win = LagWindows{0, 0, 0, 0},
                                 WorkBufs wb = WorkBufs{NULL, NULL}) {
	int rc = ensure_table(ctx, stream);
	if (rc) return rc;
	const unsigned long long N = tsdrgpu_fft_getrealsize(size);
	float2 *ans = reinterpret_cast<float2 *>(d_answer);
	if (N == 1 || !skip_tail) {
		for (unsigned b = 0; b < batch; b++) {       // the part that never enters a transform (fft.c:52-60): (|x|, 0)
			const unsigned long long from = (N == 1) ? 0 : N;
			if (from >= size) break;
			float2 *a = reinterpret_cast<float2 *>(d_answer + (long long) b * answer_stride);
			KL(ctx, "k_real_to_complex", stream, k_real_to_complex<<<grid1d(size - from, ctx->sm_count), 256, 0, stream>>>(a, d_real + (long long) b * real_stride, from, size));
			KL(ctx, "k_abs", stream, k_abs<<<grid1d(size - from, ctx->sm_count), 256, 0, stream>>>(a, from, size));
		}
		if (N == 1) return TSDRGPU_OK;
	}
	// default: both transforms at half size (autocorrelation_batch_half); TSDRGPU_AUTOCORR_FULL=1 keeps the N-point transforms
	const bool full_size = getenv("TSDRGPU_AUTOCORR_FULL") != NULL;     // read per call: the tests flip it inside one process
	if (!full_size && N >= 16 && (answer_stride & 1) == 0) {
		if (win.hi0 > (unsigned) (N >> 1) || win.hi1 > (unsigned) (N >> 1)) win = LagWindows{0, 0, 0, 0};      // a window beyond N/2: produce every lag
		return autocorrelation_batch_half(ctx, stream, ans, answer_stride / 2, d_real, real_stride, N, batch, win, wb);
	}
	void *scratch = wb.w0;                              // (sized for N * batch by the overlapped detector)
	if (!scratch && (rc = tsdrgpu_scratch(ctx, 0, sizeof(float2) * N * batch, &scratch))) return rc;
	// forward transform of the first N samples, real input widened on load, |X|/N on store
	FftOpts f; memset(&f, 0, sizeof f);
	f.real_in = d_real; f.out_abs = true; f.scale = 1.0f / (float) N; f.batch = batch;
	f.data_bs = answer_stride / 2; f.scratch_bs = (long long) N; f.real_bs = real_stride;
	if ((rc = fft_run(ctx, stream, ans, (float2 *) scratch, ilog2(N), 0, f))) return rc;
	FftOpts g; memset(&g, 0, sizeof g);
	g.scale = 1.0f; g.batch = batch; g.data_bs = answer_stride / 2; g.scratch_bs = (long long) N;
	return fft_run(ctx, stream, ans, (float2 *) scratch, ilog2(N), 1, g);
}

int tsdrgpu_autocorrelation(tsdrgpu_ctx_t *ctx, void *stream, float *d_answer, const float *d_real, uint32_t size) {
	BIND(ctx); ARG_TRY(ctx, d_answer != NULL && d_real != NULL);
	if (size == 0) return TSDRGPU_OK;
	return autocorrelation_batch(ctx, (cudaStream_t) stream, d_answer, 2ll * size, d_real, size, size, 1, false);
}

int tsdrgpu_autocorrelation_batch(tsdrgpu_ctx_t *ctx, void *stream, float *d_answers, const float *d_reals, uint32_t size,
                                  uint32_t batch, uint64_t real_stride) {
	BIND(ctx); ARG_TRY(ctx, d_answers != NULL && d_reals != NULL && (size & 1) == 0);
	if (size == 0 || batch == 0) return TSDRGPU_OK;
	return autocorrelation_batch(ctx, (cudaStream_t) stream, d_answers, 2ll * size, d_reals, (long long) real_stride, size, batch, false);
}

int tsdrgpu_crosscorrelation(tsdrgpu_ctx_t *ctx, void *stream_, float *d_a, float *d_b, uint32_t samples) {
	BIND(ctx); ARG_TRY(ctx, d_a != NULL && d_b != NULL);
	if (samples == 0) return TSDRGPU_OK;
	cudaStream_t stream = (cudaStream_t) stream_;
	const unsigned long long N = tsdrgpu_fft_getrealsize(samples);
	int rc;
	if ((rc = tsdrgpu_fft_internal(ctx, stream, reinterpret_cast<float2 *>(d_a), N, 0))) return rc;
	if ((rc = tsdrgpu_fft_internal(ctx, stream, reinterpret_cast<float2 *>(d_b), N, 0))) return rc;
	KL(ctx, "k_conj_mul", stream, k_conj_mul<<<grid1d(N, ctx->sm_count), 256, 0, stream>>>(reinterpret_cast<float2 *>(d_a), reinterpret_cast<const float2 *>(d_b), N));
	return tsdrgpu_fft_internal(ctx, stream, reinterpret_cast<float2 *>(d_a), N, 1);
}

}  // extern "C"

// one capture round of the scan (channelizer.cu): K captures of `size` magnitudes (capture c at d_caps + c * cap_stride) through the
// batched autocorrelation (only the detector's two lag windows), the running means of every channel, then the peaks and scores
int tsdrgpu_scan_round_internal(tsdrgpu_ctx_t *ctx, cudaStream_t stream, const float *d_caps, uint64_t cap_stride, uint32_t size,
                                unsigned K, uint32_t rate, float *d_big, float2 *w0, float2 *w1, double *d_plots, uint64_t calls,
                                TsdrScanPeak *d_res) {
	int fmin, fmax, lmin, lmax;
	tsdrgpu_frd_windows(rate, &fmin, &fmax, &lmin, &lmax);
	const int flen = fmax - fmin, llen = lmax - lmin;
	const uint32_t N = tsdrgpu_fft_getrealsize(size);
	const bool skip_tail = (uint32_t) fmax <= N;
	LagWindows win = LagWindows{0, 0, 0, 0};
	if (skip_tail) win = LagWindows{(unsigned) fmin, (unsigned) fmax, (unsigned) lmin, (unsigned) lmax};
	int rc = autocorrelation_batch(ctx, stream, d_big, 2ll * size, d_caps, (long long) cap_stride, size, K, skip_tail, win, WorkBufs{w0, w1});
	if (rc) return rc;
	KL(ctx, "k_accumulate_channels", stream, k_accumulate_channels<<<dim3(grid1d((unsigned long long) (flen + llen), ctx->sm_count), K), 256, 0, stream>>>(
		d_plots, (long long) (flen + llen), (unsigned long long) calls, reinterpret_cast<const float2 *>(d_big), (long long) size, fmin, flen, lmin, llen));
	KL(ctx, "k_plot_scores", stream, k_plot_scores<<<2 * K, 1024, 0, stream>>>(d_plots, (long long) (flen + llen), flen, llen, d_res));
	return TSDRGPU_OK;
}

extern "C" {

int tsdrgpu_accumulate(tsdrgpu_ctx_t *ctx, void *stream, double *d_out, uint64_t calls, const float *d_in, int startid, int length) {
	BIND(ctx); ARG_TRY(ctx, d_out != NULL && d_in != NULL && length >= 0 && startid >= 0);
	if (length == 0) return TSDRGPU_OK;
	KL(ctx, "k_accumulate", (cudaStream_t) stream, k_accumulate<<<grid1d((unsigned long long) length, ctx->sm_count), 256, 0, (cudaStream_t) stream>>>(d_out, calls, reinterpret_cast<const float2 *>(d_in), startid, length));
	return TSDRGPU_OK;
}

// ---- frame-rate detector ---------------------------------------------------------------------------------------
int tsdrgpu_frd_create(tsdrgpu_ctx_t *ctx, tsdrgpu_frd_t **out) {
	BIND(ctx); ARG_TRY(ctx, out != NULL);
	tsdrgpu_frd *f = new tsdrgpu_frd();
	memset(f, 0, sizeof *f);
	f->ctx = ctx; f->fresh = 1;
	CU_TRY(ctx, cudaMalloc(&f->d_peaks, 256));
	CU_TRY(ctx, cudaMemset(f->d_peaks, 0, 256));
	*out = f;
	return TSDRGPU_OK;
}
// overlapped mode on/off (see struct tsdrgpu_frd).  While it is on, a capture handed to tsdrgpu_frd_run* must stay untouched
// until tsdrgpu_frd_join (or the next synchronising call) has put the caller's stream behind the run.
int tsdrgpu_frd_set_overlap(tsdrgpu_frd_t *f, int on) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, f != NULL);
	tsdrgpu_ctx_t *ctx = f->ctx;
	BIND(ctx);
	if (on && !f->s_side) {
		// the detector's work is background work (a plot every few frames): lowest priority, so that the block scheduler hands free
		// SM resources to the pixel path first and lets the transforms fill what is left (TSDRGPU_FRD_PRIO=high|default for studies)
		int lo = 0, hi = 0;
		CU_TRY(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));
		const char *pr = getenv("TSDRGPU_FRD_PRIO");
		const int prio = (pr && !strcmp(pr, "high")) ? hi : ((pr && !strcmp(pr, "default")) ? 0 : lo);
		CU_TRY(ctx, cudaStreamCreateWithPriority(&f->s_side, cudaStreamNonBlocking, prio));
		CU_TRY(ctx, cudaEventCreateWithFlags(&f->ev_in, cudaEventDisableTiming));
		CU_TRY(ctx, cudaEventCreateWithFlags(&f->ev_done, cudaEventDisableTiming));
	}
	if (!on && f->pending) { CU_TRY(ctx, cudaStreamSynchronize(f->s_side)); f->pending = 0; }
	f->overlap = on ? 1 : 0;
	return TSDRGPU_OK;
}
// `stream` waits (on the device) for the detector's last overlapped run; a no-op otherwise
int tsdrgpu_frd_join(tsdrgpu_frd_t *f, void *stream) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, f != NULL);
	BIND(f->ctx);
	if (f->pending) CU_TRY(f->ctx, cudaStreamWaitEvent((cudaStream_t) stream, f->ev_done, 0));
	return TSDRGPU_OK;
}
void tsdrgpu_frd_destroy(tsdrgpu_frd_t *f) {
	if (!f) return;
	cudaSetDevice(f->ctx->device); cudaDeviceSynchronize();
	if (f->d_big) cudaFree(f->d_big);
	if (f->d_p1) cudaFree(f->d_p1);
	if (f->d_p2) cudaFree(f->d_p2);
	if (f->d_peaks) cudaFree(f->d_peaks);
	if (f->w0) cudaFree(f->w0);
	if (f->w1) cudaFree(f->w1);
	if (f->s_side) { cudaStreamDestroy(f->s_side); cudaEventDestroy(f->ev_in); cudaEventDestroy(f->ev_done); }
	delete f;
}
int tsdrgpu_frd_reset(tsdrgpu_frd_t *f) { if (!f) return TSDRGPU_EINVAL; f->fresh = 1; return TSDRGPU_OK; }

uint32_t tsdrgpu_frd_capture_size(uint32_t samplerate) { return (uint32_t) (3.1 * samplerate / (double) (55)); }   // frameratedetector.c:160
void tsdrgpu_frd_windows(uint32_t samplerate, int *frame_min, int *frame_max, int *line_min, int *line_max) {
	*frame_max = (int) (samplerate / (double) (55));               // frameratedetector.c:91-95
	*frame_min = (int) (samplerate / (double) (87));
	*line_max = (int) (samplerate / (double) (590 * 55));
	*line_min = (int) (samplerate / (double) (1500 * 87));
}

static int frd_run_impl(tsdrgpu_frd_t *f, void *stream_, uint32_t samplerate, const float *d_capture, uint32_t size,
                        uint32_t batch, uint64_t capture_stride,
                        double *h_frame_plot, int frame_cap, double *h_line_plot, int line_cap, uint64_t *calls, bool synchronise) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, f != NULL);
	tsdrgpu_ctx_t *ctx = f->ctx;
	BIND(ctx); ARG_TRY(ctx, d_capture != NULL && size > 0 && batch > 0);
	cudaStream_t caller = (cudaStream_t) stream_, stream = caller;
	int fmin, fmax, lmin, lmax;
	tsdrgpu_frd_windows(samplerate, &fmin, &fmax, &lmin, &lmax);
	const int flen = fmax - fmin, llen = lmax - lmin;
	const uint32_t N = tsdrgpu_fft_getrealsize(size);
	ARG_TRY(ctx, (uint64_t) fmax <= (uint64_t) size && flen >= 0 && llen >= 0);
	const bool skip_tail = (uint32_t) fmax <= N;               // always true for the detector's own capture size
	const size_t big_need = 2ull * size * batch;
	WorkBufs wb = WorkBufs{NULL, NULL};
	if (f->overlap) {
		// the internal stream picks up behind everything the caller's stream holds now (the capture is complete there)
		stream = f->s_side;
		const size_t need0 = (size_t) N * batch, need1 = (size_t) (N / 2) * batch + 16;
		if (f->w0_cap < need0 || f->w1_cap < need1) {
			CU_TRY(ctx, cudaStreamSynchronize(f->s_side));
			if (f->w0) CU_TRY(ctx, cudaFree(f->w0));
			if (f->w1) CU_TRY(ctx, cudaFree(f->w1));
			f->w0 = f->w1 = NULL; f->w0_cap = f->w1_cap = 0;
			CU_TRY(ctx, cudaMalloc(&f->w0, sizeof(float2) * need0)); f->w0_cap = need0;
			CU_TRY(ctx, cudaMalloc(&f->w1, sizeof(float2) * need1)); f->w1_cap = need1;
		}
		wb = WorkBufs{f->w0, f->w1};
		CU_TRY(ctx, cudaEventRecord(f->ev_in, caller));
		CU_TRY(ctx, cudaStreamWaitEvent(f->s_side, f->ev_in, 0));
	}
	if (f->big_cap < big_need) {
		CU_TRY(ctx, cudaStreamSynchronize(stream));
		if (f->d_big) CU_TRY(ctx, cudaFree(f->d_big));
		CU_TRY(ctx, cudaMalloc(&f->d_big, sizeof(float) * big_need)); f->big_cap = big_need;
	}
	if (f->p1_cap < (size_t) flen || f->fresh) {
		if (f->p1_cap < (size_t) flen) { CU_TRY(ctx, cudaStreamSynchronize(stream)); if (f->d_p1) CU_TRY(ctx, cudaFree(f->d_p1)); CU_TRY(ctx, cudaMalloc(&f->d_p1, sizeof(double) * (flen + 1))); f->p1_cap = flen; }
		CU_TRY(ctx, cudaMemsetAsync(f->d_p1, 0, sizeof(double) * (flen + 1), stream));
	}
	if (f->p2_cap < (size_t) llen || f->fresh) {
		if (f->p2_cap < (size_t) llen) { CU_TRY(ctx, cudaStreamSynchronize(stream)); if (f->d_p2) CU_TRY(ctx, cudaFree(f->d_p2)); CU_TRY(ctx, cudaMalloc(&f->d_p2, sizeof(double) * (llen + 1))); f->p2_cap = llen; }
		CU_TRY(ctx, cudaMemsetAsync(f->d_p2, 0, sizeof(double) * (llen + 1), stream));
	}
	if (f->fresh) { f->calls = 0; f->fresh = 0; }
	const uint64_t first_calls = f->calls + 1;                  // extbuffer.c:81, one prepare per capture
	f->calls += batch;
	int rc;
	// only the two lag windows are ever read (frameratedetector.c:106-109): the last step writes nothing else
	LagWindows win = LagWindows{0, 0, 0, 0};
	if (skip_tail && !getenv("TSDRGPU_AUTOCORR_ALL_LAGS")) win = LagWindows{(unsigned) fmin, (unsigned) fmax, (unsigned) lmin, (unsigned) lmax};
	if ((rc = autocorrelation_batch(ctx, stream, f->d_big, 2ll * size, d_capture, (long long) capture_stride, size, batch, skip_tail, win, wb))) return rc;
	if (flen) KL(ctx, "k_accumulate", stream, k_accumulate_batch<<<grid1d((unsigned long long) flen, ctx->sm_count), 256, 0, stream>>>(f->d_p1, first_calls, reinterpret_cast<const float2 *>(f->d_big), (long long) size, batch, fmin, flen));
	if (llen) KL(ctx, "k_accumulate", stream, k_accumulate_batch<<<grid1d((unsigned long long) llen, ctx->sm_count), 256, 0, stream>>>(f->d_p2, first_calls, reinterpret_cast<const float2 *>(f->d_big), (long long) size, batch, lmin, llen));
	KL(ctx, "k_plot_peaks", stream, k_plot_peaks<<<2, 1024, 0, stream>>>(f->d_p1, flen, f->d_p2, llen, f->d_peaks));
	if (calls) *calls = f->calls;
	if (h_frame_plot || h_line_plot) {
		if (h_frame_plot) CU_TRY(ctx, cudaMemcpyAsync(h_frame_plot, f->d_p1, sizeof(double) * (size_t) (flen < frame_cap ? flen : frame_cap), cudaMemcpyDeviceToHost, stream));
		if (h_line_plot) CU_TRY(ctx, cudaMemcpyAsync(h_line_plot, f->d_p2, sizeof(double) * (size_t) (llen < line_cap ? llen : line_cap), cudaMemcpyDeviceToHost, stream));
		if (synchronise) CU_TRY(ctx, cudaStreamSynchronize(stream));
	}
	if (f->overlap) { CU_TRY(ctx, cudaEventRecord(f->ev_done, f->s_side)); f->pending = 1; }
	return TSDRGPU_OK;
}

int tsdrgpu_frd_run(tsdrgpu_frd_t *f, void *stream, uint32_t samplerate, const float *d_capture, uint32_t size,
                    double *h_frame_plot, int frame_cap, double *h_line_plot, int line_cap, uint64_t *calls) {
	return frd_run_impl(f, stream, samplerate, d_capture, size, 1, size, h_frame_plot, frame_cap, h_line_plot, line_cap, calls, true);
}
int tsdrgpu_frd_run_batch(tsdrgpu_frd_t *f, void *stream, uint32_t samplerate, const float *d_captures, uint32_t size, uint32_t batch,
                          uint64_t capture_stride, uint64_t *calls) {
	return frd_run_impl(f, stream, samplerate, d_captures, size, batch, capture_stride, NULL, 0, NULL, 0, calls, false);
}
int tsdrgpu_frd_run_async(tsdrgpu_frd_t *f, void *stream, uint32_t samplerate, const float *d_capture, uint32_t size,
                          double *h_frame_plot_pinned, int frame_cap, double *h_line_plot_pinned, int line_cap, uint64_t *calls) {
	return frd_run_impl(f, stream, samplerate, d_capture, size, 1, size, h_frame_plot_pinned, frame_cap, h_line_plot_pinned, line_cap, calls, false);
}

// dump_autocorrect (frameratedetector.c:64-85): the autocorrelation of ONE capture as a CSV of (lag in ms, 10 log10 |r|) for the
// lags the reference writes (i < fft_getrealsize(2 size) / 2 floats, i.e. the first half of the transformed lags), same header and
// "%f, %f" rows.  A debugging aid of the GUI (PARAM_AUTOCORR_DUMP): one extra autocorrelation with every lag produced, a device-to-
// host copy and a synchronisation, only when asked for.  Does not touch the running means.
int tsdrgpu_frd_dump_csv(tsdrgpu_frd_t *f, void *stream_, uint32_t samplerate, const float *d_capture, uint32_t size, const char *path) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, f != NULL);
	tsdrgpu_ctx_t *ctx = f->ctx;
	BIND(ctx); ARG_TRY(ctx, d_capture != NULL && size > 0 && path != NULL && samplerate > 0);
	cudaStream_t stream = (cudaStream_t) stream_;
	const uint32_t maxels = tsdrgpu_fft_getrealsize(2u * size) / 2u;           // floats of the answer the reference walks
	float *d_ans = NULL;
	CU_TRY(ctx, cudaMalloc(&d_ans, sizeof(float) * 2ull * size));
	int rc = autocorrelation_batch(ctx, stream, d_ans, 2ll * size, d_capture, (long long) size, size, 1, false);
	std::vector<float> h(maxels);
	if (rc == TSDRGPU_OK) {
		const cudaError_t e1 = cudaMemcpyAsync(h.data(), d_ans, sizeof(float) * maxels, cudaMemcpyDeviceToHost, stream);
		const cudaError_t e2 = (e1 == cudaSuccess) ? cudaStreamSynchronize(stream) : e1;
		if (e2 != cudaSuccess) rc = tsdrgpu_fail(ctx, TSDRGPU_ECUDA, "autocorrelation dump: copy", e2, __FILE__, __LINE__);
	} else cudaStreamSynchronize(stream);
	cudaFree(d_ans);
	if (rc != TSDRGPU_OK) return rc;
	FILE *fp = fopen(path, "w");
	if (!fp) return tsdrgpu_fail(ctx, TSDRGPU_EINVAL, "autocorrelation dump: cannot open the file", cudaSuccess, __FILE__, __LINE__);
	fprintf(fp, "%s, %s\n", "ms", "dB");
	for (uint32_t i = 0; i < maxels; i += 2) {
		const double I = (double) h[i], Q = (i + 1 < maxels) ? (double) h[i + 1] : 0.0;
		const double db = 10.0 * log10(sqrt(I * I + Q * Q));
		const double t = 1000.0 * (double) (i / 2) / (double) samplerate;
		fprintf(fp, "%f, %f\n", t, db);
	}
	fclose(fp);
	return TSDRGPU_OK;
}

int tsdrgpu_frd_get_plots(tsdrgpu_frd_t *f, void *stream_, uint32_t samplerate, double *h_frame_plot, int frame_cap,
                          double *h_line_plot, int line_cap) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, f != NULL);
	tsdrgpu_ctx_t *ctx = f->ctx;
	BIND(ctx);
	cudaStream_t stream = (cudaStream_t) stream_;
	int fmin, fmax, lmin, lmax;
	tsdrgpu_frd_windows(samplerate, &fmin, &fmax, &lmin, &lmax);
	const int flen = fmax - fmin, llen = lmax - lmin;
	ARG_TRY(ctx, f->p1_cap >= (size_t) flen && f->p2_cap >= (size_t) llen);
	if (f->pending) CU_TRY(ctx, cudaStreamWaitEvent(stream, f->ev_done, 0));
	if (h_frame_plot) CU_TRY(ctx, cudaMemcpyAsync(h_frame_plot, f->d_p1, sizeof(double) * (size_t) (flen < frame_cap ? flen : frame_cap), cudaMemcpyDeviceToHost, stream));
	if (h_line_plot) CU_TRY(ctx, cudaMemcpyAsync(h_line_plot, f->d_p2, sizeof(double) * (size_t) (llen < line_cap ? llen : line_cap), cudaMemcpyDeviceToHost, stream));
	CU_TRY(ctx, cudaStreamSynchronize(stream));
	return TSDRGPU_OK;
}

// SURVEY 8f-3: where the two plots peak, picked on the device right after the running means were updated.
// h_peaks[0] = frame plot, [1] = line plot (indices into the plots; add the window offsets for lags).  tsdrgpu_frd_peaks
// synchronises; the _async form needs page-locked memory and is valid once the stream has passed it.
// stage-level entry: the same reduction on any two device-resident plots (synchronises)
int tsdrgpu_plot_peaks(tsdrgpu_ctx_t *ctx, void *stream_, const double *d_frame_plot, int frame_len, const double *d_line_plot, int line_len, int32_t *h_peaks) {
	BIND(ctx); ARG_TRY(ctx, d_frame_plot && d_line_plot && frame_len >= 0 && line_len >= 0 && h_peaks);
	cudaStream_t stream = (cudaStream_t) stream_;
	void *d;
	int rc = tsdrgpu_scratch(ctx, 3, 256, &d);
	if (rc) return rc;
	KL(ctx, "k_plot_peaks", stream, k_plot_peaks<<<2, 1024, 0, stream>>>(d_frame_plot, frame_len, d_line_plot, line_len, (int *) d));
	CU_TRY(ctx, cudaMemcpyAsync(h_peaks, d, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
	CU_TRY(ctx, cudaStreamSynchronize(stream));
	return TSDRGPU_OK;
}
int tsdrgpu_frd_peaks_async(tsdrgpu_frd_t *f, void *stream, int32_t *h_peaks_pinned) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, f != NULL && h_peaks_pinned != NULL);
	BIND(f->ctx);
	if (f->pending) CU_TRY(f->ctx, cudaStreamWaitEvent((cudaStream_t) stream, f->ev_done, 0));
	CU_TRY(f->ctx, cudaMemcpyAsync(h_peaks_pinned, f->d_peaks, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, (cudaStream_t) stream));
	return TSDRGPU_OK;
}
int tsdrgpu_frd_peaks(tsdrgpu_frd_t *f, void *stream, int32_t *h_peaks) {
	ARG_TRY((tsdrgpu_ctx_t *) NULL, f != NULL && h_peaks != NULL);
	BIND(f->ctx);
	if (f->pending) CU_TRY(f->ctx, cudaStreamWaitEvent((cudaStream_t) stream, f->ev_done, 0));
	CU_TRY(f->ctx, cudaMemcpyAsync(h_peaks, f->d_peaks, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, (cudaStream_t) stream));
	CU_TRY(f->ctx, cudaStreamSynchronize((cudaStream_t) stream));
	return TSDRGPU_OK;
}

// ---- superbandwidth ----------------------------------------------------------------------------------------------
int tsdrgpu_complex_to_abs_diff(tsdrgpu_ctx_t *ctx, void *stream_, float *d_data, int size_floats) {
	BIND(ctx); ARG_TRY(ctx, d_data != NULL && size_floats >= 0 && (size_floats & 1) == 0);
	if (size_floats == 0) return TSDRGPU_OK;
	cudaStream_t stream = (cudaStream_t) stream_;
	const unsigned long long pairs = (unsigned long long) size_floats / 2;
	void *tmp; int rc;
	if ((rc = tsdrgpu_scratch(ctx, 1, sizeof(float2) * pairs, &tmp))) return rc;
	KL(ctx, "k_abs_diff", stream, k_abs_diff<<<grid1d(pairs, ctx->sm_count), 256, 0, stream>>>(reinterpret_cast<const float2 *>(d_data), (float2 *) tmp, pairs));
	CU_TRY(ctx, cudaMemcpyAsync(d_data, tmp, sizeof(float2) * pairs, cudaMemcpyDeviceToDevice, stream));
	return TSDRGPU_OK;
}

// the lag (in complex samples) of hop i against hop 0, left in device memory at d_lag -- no host round trip
static int superb_bestfit_dev(tsdrgpu_ctx_t *ctx, cudaStream_t stream, const float *d_hop0, const float *d_hopi, int size_floats,
                              int samples_in_frame, int *d_lag) {
	int size = (size_floats / samples_in_frame) * samples_in_frame;      // superbandwidth.c:84-86
	ARG_TRY(ctx, size >= 2);
	size = (int) tsdrgpu_fft_getrealsize((uint32_t) size);
	const unsigned long long pairs = (unsigned long long) size / 2;
	void *wa, *wb, *part; int rc;
	if ((rc = tsdrgpu_scratch(ctx, 1, sizeof(float2) * pairs + 256, &wa))) return rc;
	if ((rc = tsdrgpu_scratch(ctx, 2, sizeof(float2) * pairs + 8 * TSDRGPU_ARGMAX_PARTS + 256, &wb))) return rc;
	KL(ctx, "k_abs_diff", stream, k_abs_diff<<<grid1d(pairs, ctx->sm_count), 256, 0, stream>>>(reinterpret_cast<const float2 *>(d_hop0), (float2 *) wa, pairs));
	KL(ctx, "k_abs_diff", stream, k_abs_diff<<<grid1d(pairs, ctx->sm_count), 256, 0, stream>>>(reinterpret_cast<const float2 *>(d_hopi), (float2 *) wb, pairs));
	if ((rc = tsdrgpu_crosscorrelation(ctx, stream, (float *) wa, (float *) wb, (uint32_t) pairs))) return rc;
	part = wb;                                            // wb is free again after the cross-correlation
	return tsdrgpu_argmax_mag_internal(ctx, stream, (const float2 *) wa, (unsigned) pairs, part, d_lag);
}

int tsdrgpu_superb_bestfit(tsdrgpu_ctx_t *ctx, void *stream_, const float *d_hop0, const float *d_hopi, int size_floats,
                           int samples_in_frame, int *h_best_offset) {
	BIND(ctx); ARG_TRY(ctx, d_hop0 && d_hopi && h_best_offset && size_floats > 0 && samples_in_frame > 0);
	cudaStream_t stream = (cudaStream_t) stream_;
	void *res; int rc;
	if ((rc = tsdrgpu_scratch(ctx, 3, 256, &res))) return rc;
	if ((rc = superb_bestfit_dev(ctx, stream, d_hop0, d_hopi, size_floats, samples_in_frame, (int *) res))) return rc;
	int lag = 0;
	CU_TRY(ctx, cudaMemcpyAsync(&lag, res, sizeof(int), cudaMemcpyDeviceToHost, stream));
	CU_TRY(ctx, cudaStreamSynchronize(stream));
	*h_best_offset = 2 * lag;
	return TSDRGPU_OK;
}

int tsdrgpu_superb_hop_spectrum(tsdrgpu_ctx_t *ctx, void *stream_, const float *d_hop, int count_pairs, int best_offset_floats, float *d_spectrum) {
	BIND(ctx); ARG_TRY(ctx, d_hop && d_spectrum && count_pairs > 0 && best_offset_floats >= 0 && (best_offset_floats & 1) == 0);
	cudaStream_t stream = (cudaStream_t) stream_;
	const unsigned long long N = tsdrgpu_fft_getrealsize((uint32_t) count_pairs);
	ARG_TRY(ctx, (unsigned long long) best_offset_floats / 2 < N);
	KL(ctx, "k_rotate", stream, k_rotate<<<grid1d(N, ctx->sm_count), 256, 0, stream>>>(reinterpret_cast<const float2 *>(d_hop), reinterpret_cast<float2 *>(d_spectrum), N, (unsigned long long) best_offset_floats / 2));
	return tsdrgpu_fft_internal(ctx, stream, reinterpret_cast<float2 *>(d_spectrum), N, 0);
}

// superb_ondataready (superbandwidth.c:121-152) on one GPU.  Everything stays on the device: the H-1 alignment lags are left
// in device memory by the grid argmax, the rotations read them from there, and the host sees them once, at the end (one
// synchronisation per stitch instead of one per hop).
int tsdrgpu_superb_stitch(tsdrgpu_ctx_t *ctx, void *stream_, float *const *d_hops, int nhops, int count_pairs, int samples_in_frame,
                          float *d_out, int *h_best_offsets, int *h_total_samples) {
	BIND(ctx); ARG_TRY(ctx, d_hops && nhops > 0 && nhops <= 16 && count_pairs > 0 && d_out && h_best_offsets);
	cudaStream_t stream = (cudaStream_t) stream_;
	const unsigned long long N = tsdrgpu_fft_getrealsize((uint32_t) count_pairs);
	int rc;
	void *lags_;
	if ((rc = tsdrgpu_scratch(ctx, 3, 256, &lags_))) return rc;
	int *d_lags = (int *) lags_;
	CU_TRY(ctx, cudaMemsetAsync(d_lags, 0, sizeof(int) * 16, stream));
	for (int i = 1; i < nhops; i++)
		if ((rc = superb_bestfit_dev(ctx, stream, d_hops[0], d_hops[i], (int) (2 * N), samples_in_frame, d_lags + i))) return rc;
	for (int i = 0; i < nhops; i++) {
		float2 *spec = reinterpret_cast<float2 *>(d_out) + (size_t) i * N;
		KL(ctx, "k_rotate", stream, k_rotate_dev<<<grid1d(N, ctx->sm_count), 256, 0, stream>>>(reinterpret_cast<const float2 *>(d_hops[i]), spec, N, d_lags + i));
		if ((rc = tsdrgpu_fft_internal(ctx, stream, spec, N, 0))) return rc;
	}
	const unsigned long long total = N * (unsigned long long) nhops;
	const unsigned long long tp = 1ull << ilog2(total);            // fft_perform transforms the largest power of two (fft.c:101-105)
	if ((rc = tsdrgpu_fft_internal(ctx, stream, reinterpret_cast<float2 *>(d_out), tp, 1))) return rc;
	int lags[16];
	CU_TRY(ctx, cudaMemcpyAsync(lags, d_lags, sizeof(int) * 16, cudaMemcpyDeviceToHost, stream));
	CU_TRY(ctx, cudaStreamSynchronize(stream));
	for (int i = 0; i < nhops; i++) h_best_offsets[i] = 2 * lags[i];
	if (h_total_samples) *h_total_samples = (int) total;
	return TSDRGPU_OK;
}

// ---- one hop per GPU -------------------------------------------------------------------------------------------------
// what a rank contributes to the single all-gather: [ X = FFT_N(raw hop) | D = FFT_nd(first difference of |hop|) ]
int tsdrgpu_superb_local_spectra(tsdrgpu_ctx_t *ctx, void *stream_, const float *d_hop, int count_pairs, int samples_in_frame,
                                 float *d_block, uint32_t *h_n, uint32_t *h_nd) {
	BIND(ctx); ARG_TRY(ctx, d_hop && d_block && count_pairs > 0 && samples_in_frame > 0 && h_n && h_nd);
	cudaStream_t stream = (cudaStream_t) stream_;
	const unsigned long long N = tsdrgpu_fft_getrealsize((uint32_t) count_pairs);
	int size = (int) ((2 * N / samples_in_frame) * samples_in_frame);          // superbandwidth.c:84-86 with bufsize = 2N floats
	ARG_TRY(ctx, size >= 2);
	size = (int) tsdrgpu_fft_getrealsize((uint32_t) size);
	const unsigned long long nd = (unsigned long long) size / 2;
	float2 *X = reinterpret_cast<float2 *>(d_block), *D = X + N;
	CU_TRY(ctx, cudaMemcpyAsync(X, d_hop, sizeof(float2) * N, cudaMemcpyDeviceToDevice, stream));
	int rc;
	if ((rc = tsdrgpu_fft_internal(ctx, stream, X, N, 0))) return rc;
	KL(ctx, "k_abs_diff", stream, k_abs_diff<<<grid1d(nd, ctx->sm_count), 256, 0, stream>>>(reinterpret_cast<const float2 *>(d_hop), D, nd));
	if ((rc = tsdrgpu_fft_internal(ctx, stream, D, nd, 0))) return rc;
	*h_n = (uint32_t) N; *h_nd = (uint32_t) nd;
	return TSDRGPU_OK;
}

// The same contribution, but delivered: the final pass of each of the two transforms stores its result straight into the
// gather buffer of EVERY rank (d_peer_bufs[p] = rank p's buffer, mapped here through CUDA IPC; the own entry is local memory)
// at this rank's slot, so the all-gather happens inside the transform's epilogue, over NVLink, while the transform runs.
// What remains for the caller is a barrier (all ranks have finished storing) before anybody reads its buffer.
int tsdrgpu_superb_local_spectra_scatter(tsdrgpu_ctx_t *ctx, void *stream_, const float *d_hop, int count_pairs, int samples_in_frame,
                                         float *const *d_peer_bufs, int nhops, int rank, uint64_t block_stride_complex,
                                         uint32_t *h_n, uint32_t *h_nd) {
	BIND(ctx); ARG_TRY(ctx, d_hop && d_peer_bufs && count_pairs > 0 && samples_in_frame > 0 && h_n && h_nd);
	ARG_TRY(ctx, nhops > 0 && nhops <= 16 && rank >= 0 && rank < nhops);
	cudaStream_t stream = (cudaStream_t) stream_;
	const unsigned long long N = tsdrgpu_fft_getrealsize((uint32_t) count_pairs);
	int size = (int) ((2 * N / samples_in_frame) * samples_in_frame);          // superbandwidth.c:84-86 with bufsize = 2N floats
	ARG_TRY(ctx, size >= 2);
	size = (int) tsdrgpu_fft_getrealsize((uint32_t) size);
	const unsigned long long nd = (unsigned long long) size / 2;
	ARG_TRY(ctx, N + nd <= block_stride_complex && N > 4 && nd > 4);
	int rc = ensure_table(ctx, stream);
	if (rc) return rc;
	void *work, *scratch;
	if ((rc = tsdrgpu_scratch(ctx, 1, sizeof(float2) * N, &work))) return rc;
	if ((rc = tsdrgpu_scratch(ctx, 0, sizeof(float2) * N, &scratch))) return rc;
	float2 *fanX[16], *fanD[16];
	for (int q = 0; q < nhops; q++) {
		ARG_TRY(ctx, d_peer_bufs[q] != NULL);
		fanX[q] = reinterpret_cast<float2 *>(d_peer_bufs[q]) + (size_t) rank * block_stride_complex;
		fanD[q] = fanX[q] + N;
	}
	FftOpts o; memset(&o, 0, sizeof o); o.batch = 1;
	// X = FFT_N(raw hop)
	CU_TRY(ctx, cudaMemcpyAsync(work, d_hop, sizeof(float2) * N, cudaMemcpyDeviceToDevice, stream));
	o.scale = 1.0f / (float) N; o.fan = fanX; o.nfan = nhops;
	if ((rc = fft_run(ctx, stream, (float2 *) work, (float2 *) scratch, ilog2(N), 0, o))) return rc;
	// D = FFT_nd(first difference of |hop|)
	KL(ctx, "k_abs_diff", stream, k_abs_diff<<<grid1d(nd, ctx->sm_count), 256, 0, stream>>>(reinterpret_cast<const float2 *>(d_hop), (float2 *) work, nd));
	o.scale = 1.0f / (float) nd; o.fan = fanD;
	if ((rc = fft_run(ctx, stream, (float2 *) work, (float2 *) scratch, ilog2(nd), 0, o))) return rc;
	*h_n = (uint32_t) N; *h_nd = (uint32_t) nd;
	return TSDRGPU_OK;
}

// after the all-gather: the alignment lag of every hop against hop 0 (pairs), exact integers.  synchronises
int tsdrgpu_superb_lags(tsdrgpu_ctx_t *ctx, void *stream_, const float *d_gathered, int nhops, uint64_t block_stride_complex,
                        uint32_t n, uint32_t nd, int *h_lags) {
	BIND(ctx); ARG_TRY(ctx, d_gathered && nhops > 0 && nhops <= 16 && h_lags && nd > 0 && (nd & (nd - 1)) == 0);
	cudaStream_t stream = (cudaStream_t) stream_;
	const float2 *G = reinterpret_cast<const float2 *>(d_gathered);
	void *wa, *res; int rc;
	if ((rc = tsdrgpu_scratch(ctx, 1, sizeof(float2) * nd + 256, &wa))) return rc;
	if ((rc = tsdrgpu_scratch(ctx, 2, 256 + 8 * TSDRGPU_ARGMAX_PARTS + 256, &res))) return rc;
	h_lags[0] = 0;
	for (int q = 1; q < nhops; q++) {
		CU_TRY(ctx, cudaMemcpyAsync(wa, G + n, sizeof(float2) * nd, cudaMemcpyDeviceToDevice, stream));            // D_0
		KL(ctx, "k_conj_mul", stream, k_conj_mul<<<grid1d(nd, ctx->sm_count), 256, 0, stream>>>((float2 *) wa, G + (size_t) q * block_stride_complex + n, nd));
		if ((rc = tsdrgpu_fft_internal(ctx, stream, (float2 *) wa, nd, 1))) return rc;
		if ((rc = tsdrgpu_argmax_mag_internal(ctx, stream, (const float2 *) wa, nd, (char *) res + 256, (int *) res + q))) return rc;
	}
	CU_TRY(ctx, cudaMemcpyAsync(h_lags + 1, (int *) res + 1, sizeof(int) * (nhops - 1), cudaMemcpyDeviceToHost, stream));
	CU_TRY(ctx, cudaStreamSynchronize(stream));
	return TSDRGPU_OK;
}

// this rank's strided residue of the H*N-point inverse, from the gathered RAW spectra and the lags
int tsdrgpu_superb_residue_ifft_lag(tsdrgpu_ctx_t *ctx, void *stream_, const float *d_gathered, int nhops, uint64_t block_stride_complex,
                                    uint32_t n, int residue, const int *h_lags, float *d_out) {
	BIND(ctx); ARG_TRY(ctx, d_gathered && d_out && h_lags && nhops > 0 && nhops <= 16 && n > 0 && residue >= 0 && residue < nhops && (n & (n - 1)) == 0);
	cudaStream_t stream = (cudaStream_t) stream_;
	LagSet ls; for (int q = 0; q < 16; q++) ls.lag[q] = q < nhops ? h_lags[q] : 0;
	KL(ctx, "k_residue_mix", stream, k_residue_mix_lag<<<grid1d(n, ctx->sm_count), 256, 0, stream>>>(reinterpret_cast<const float2 *>(d_gathered), (long long) block_stride_complex, nhops, n, residue, ls, reinterpret_cast<float2 *>(d_out)));
	return tsdrgpu_fft_internal(ctx, stream, reinterpret_cast<float2 *>(d_out), n, 1);
}

int tsdrgpu_superb_residue_ifft(tsdrgpu_ctx_t *ctx, void *stream_, const float *d_gathered, int nhops, uint32_t n, int residue, float *d_out) {
	BIND(ctx); ARG_TRY(ctx, d_gathered && d_out && nhops > 0 && n > 0 && residue >= 0 && residue < nhops && (n & (n - 1)) == 0);
	cudaStream_t stream = (cudaStream_t) stream_;
	KL(ctx, "k_residue_mix", stream, k_residue_mix<<<grid1d(n, ctx->sm_count), 256, 0, stream>>>(reinterpret_cast<const float2 *>(d_gathered), nhops, n, residue, reinterpret_cast<float2 *>(d_out)));
	return tsdrgpu_fft_internal(ctx, stream, reinterpret_cast<float2 *>(d_out), n, 1);
}

}  // extern "C"
