// common.cuh -- shared plumbing of libtsdrgpu (context, error handling, exact-arithmetic helpers).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <mutex>
#include <vector>

#include "../../include/tsdrgpu.h"

struct tsdrgpu_ctx {
	int device;
	int sm_count;
	char err[512];
	uint64_t launches;
	// scratch owned by the context (grown on demand, reused across calls on the same stream)
	void *scratch[4];
	size_t scratch_bytes[4];
	void *pinned;            // small pinned staging area for descriptor uploads / scalar read-backs
	size_t pinned_bytes;
	std::mutex mu;
	// optional per-kernel timing (bench.py's roofline): CUDA events on the launching stream around named launches
	bool profiling;
	struct ProfRec { int id; cudaEvent_t a, b; };
	std::vector<ProfRec> prof_recs;
	std::vector<cudaEvent_t> prof_pool;
	char prof_names[48][48];
	int prof_nnames;
};

void tsdrgpu_prof_begin(tsdrgpu_ctx_t *ctx, const char *name, cudaStream_t stream);
void tsdrgpu_prof_end(tsdrgpu_ctx_t *ctx, cudaStream_t stream);
// wrap a kernel launch: KL(ctx, "name", stream, kernel<<<...>>>(...));
#define KL(ctx, name, stream, ...) do { if ((ctx)->profiling) tsdrgpu_prof_begin((ctx), (name), (stream)); __VA_ARGS__; \
	if ((ctx)->profiling) tsdrgpu_prof_end((ctx), (stream)); LAUNCH_CHECK(ctx); } while (0)

extern thread_local char g_tsdrgpu_err[512];

static inline int tsdrgpu_fail(tsdrgpu_ctx_t *ctx, int code, const char *what, cudaError_t e, const char *file, int line) {
	char *dst = ctx ? ctx->err : g_tsdrgpu_err;
	if (e != cudaSuccess) { snprintf(dst, 512, "%s: %s (%s:%d)", what, cudaGetErrorString(e), file, line); cudaGetLastError(); /* reported here: do not let it resurface at the next launch check */ }
	else snprintf(dst, 512, "%s (%s:%d)", what, file, line);
	return code;
}

#define CU_TRY(ctx, expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) \
	return tsdrgpu_fail((ctx), TSDRGPU_ECUDA, #expr, e_, __FILE__, __LINE__); } while (0)
#define ARG_TRY(ctx, cond) do { if (!(cond)) \
	return tsdrgpu_fail((ctx), TSDRGPU_EINVAL, "invalid argument: " #cond, cudaSuccess, __FILE__, __LINE__); } while (0)
#define LAUNCH_CHECK(ctx) do { (ctx)->launches++; cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) \
	return tsdrgpu_fail((ctx), TSDRGPU_ECUDA, "kernel launch", e_, __FILE__, __LINE__); } while (0)

static inline int tsdrgpu_bind(tsdrgpu_ctx_t *ctx) {
	if (!ctx) return tsdrgpu_fail(NULL, TSDRGPU_EINVAL, "null context", cudaSuccess, __FILE__, __LINE__);
	CU_TRY(ctx, cudaSetDevice(ctx->device));
	return TSDRGPU_OK;
}
#define BIND(ctx) do { int rc_ = tsdrgpu_bind(ctx); if (rc_ != TSDRGPU_OK) return rc_; } while (0)

// grow-only scratch slot
int tsdrgpu_scratch(tsdrgpu_ctx_t *ctx, int slot, size_t bytes, void **out);
int tsdrgpu_pinned(tsdrgpu_ctx_t *ctx, size_t bytes, void **out);

// ---- exact single-precision magnitude: fl(sqrt(fl(fl(I*I) + fl(Q*Q)))), no contraction (TSDRLibrary.c:260)
__device__ __forceinline__ float mag_exact(float i, float q) {
	return __fsqrt_rn(__fadd_rn(__fmul_rn(i, i), __fmul_rn(q, q)));
}

__device__ __forceinline__ float2 ldg_stream_f2(const float2 *p) {
	float2 v;
	asm("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
	return v;
}
__device__ __forceinline__ float4 ldg_stream_f4(const float4 *p) {
	float4 v;
	asm("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
	             : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
	return v;
}
__device__ __forceinline__ float ldg_stream_f1(const float *p) {
	float v;
	asm("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
	return v;
}

// ---- internal entry points shared between translation units (fft.cu owns the transforms)
constexpr unsigned TSDRGPU_ARGMAX_PARTS = 1024;
int tsdrgpu_fft_internal(tsdrgpu_ctx_t *ctx, cudaStream_t stream, float2 *data, unsigned long long n_pow2, int inverse);
int tsdrgpu_fft_oop_internal(tsdrgpu_ctx_t *ctx, cudaStream_t stream, const float2 *in, float2 *out, unsigned long long n_pow2, int inverse);
int tsdrgpu_fft_batch_internal(tsdrgpu_ctx_t *ctx, cudaStream_t stream, const float2 *in, long long in_bs, float2 *out, long long out_bs,
                               float2 *scratch, unsigned long long n_pow2, unsigned batch, int inverse);
int tsdrgpu_ifft_abs_internal(tsdrgpu_ctx_t *ctx, cudaStream_t stream, float2 *data, float *real_out, unsigned long long n_pow2);
int tsdrgpu_argmax_mag_internal(tsdrgpu_ctx_t *ctx, cudaStream_t stream, const float2 *x, unsigned n, void *d_part, int *d_result);
// the tuner's filter designer (tuner.cu), shared with the channelizer: n float32 taps of a Kaiser-windowed sinc low-pass
void tsdrgpu_kaiser_lowpass_internal(uint32_t fs, double bandwidth_hz, int n, float *taps);
// the same design before the rounding to float32 (the notch filter's low-pass prototypes)
void tsdrgpu_kaiser_lowpass_double_internal(uint32_t fs, double bandwidth_hz, int n, double *taps);
// the scan's per-plot result (fft.cu's k_plot_scores): first strict maximum and (max - mean) / std
struct TsdrScanPeak { double score; int32_t index, pad; };
int tsdrgpu_scan_round_internal(tsdrgpu_ctx_t *ctx, cudaStream_t stream, const float *d_caps, uint64_t cap_stride, uint32_t size,
                                unsigned K, uint32_t rate, float *d_big, float2 *w0, float2 *w1, double *d_plots, uint64_t calls,
                                TsdrScanPeak *d_res);
