// Streaming reductions and element-wise helpers: sum of squares (Frobenius norm,
// core/ndmps.py:61), per-core [min, max] (boundary_list, core/ndmps.py:75,82),
// PSNR terms (utils/metrics.py:143-146), min-max quantisation
// (utils/filetools.py:20-39).  All accumulate in float64; two-stage
// (per-block partials, then one block) so results are run-to-run deterministic.
#include "common.cuh"

namespace ndmps {

static inline int reduce_grid(const ndmps_ctx* ctx, int64_t n, int per_thread) {
    int64_t want = (n + 256 * (int64_t)per_thread - 1) / (256 * (int64_t)per_thread);
    int64_t cap = (int64_t)ctx->sm_count * 8;
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

// mode 0: sum x^2        -> out[0]
// mode 1: min, max       -> out[0], out[1]
// mode 2: sum (a-b)^2, max a -> out[0], out[1]
template <class T, int MODE>
__global__ void __launch_bounds__(256) reduce_stage1(const T* __restrict__ a, const T* __restrict__ b, int64_t n,
                                                      double* __restrict__ partial) {
    __shared__ double scratch[32];
    double acc0 = MODE == 1 ? INFINITY : 0.0;
    double acc1 = -INFINITY;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t done = 0;
    if (sizeof(T) == 4 && (reinterpret_cast<uintptr_t>(a) & 15) == 0 && (MODE != 2 || (reinterpret_cast<uintptr_t>(b) & 15) == 0)) {
        // float32: 16-byte loads, two of them in flight per array and thread; sums in two independent float64 chains
        const int64_t n4 = n >> 2;
        const float4* a4 = reinterpret_cast<const float4*>(a);
        const float4* b4 = reinterpret_cast<const float4*>(b);
        double accb = 0.0;
        auto take = [&](const float4& va, const float4& vb, double& sum) {
            const float xs[4] = {va.x, va.y, va.z, va.w}, ys[4] = {vb.x, vb.y, vb.z, vb.w};
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const double x = (double)xs[q];
                if (MODE == 0) {
                    sum = fma(x, x, sum);
                } else if (MODE == 1) {
                    acc0 = fmin(acc0, x);
                    acc1 = fmax(acc1, x);
                } else {
                    const double d = x - (double)ys[q];
                    sum = fma(d, d, sum);
                    acc1 = fmax(acc1, x);
                }
            }
        };
        int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        for (; i + stride < n4; i += 2 * stride) {
            const float4 va0 = __ldcs(a4 + i), va1 = __ldcs(a4 + i + stride);
            float4 vb0 = va0, vb1 = va1;
            if (MODE == 2) { vb0 = __ldcs(b4 + i); vb1 = __ldcs(b4 + i + stride); }
            if (MODE == 1) { take(va0, vb0, accb); take(va1, vb1, accb); }
            else { take(va0, vb0, acc0); take(va1, vb1, accb); }
        }
        for (; i < n4; i += stride) {
            const float4 va0 = __ldcs(a4 + i);
            float4 vb0 = va0;
            if (MODE == 2) vb0 = __ldcs(b4 + i);
            if (MODE == 1) take(va0, vb0, accb); else take(va0, vb0, acc0);
        }
        if (MODE != 1) acc0 += accb;
        done = n4 << 2;
    }
    for (int64_t i = done + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        double x = (double)a[i];
        if (MODE == 0) {
            acc0 += x * x;
        } else if (MODE == 1) {
            acc0 = fmin(acc0, x);
            acc1 = fmax(acc1, x);
        } else {
            double d = x - (double)b[i];
            acc0 += d * d;
            acc1 = fmax(acc1, x);
        }
    }
    double r0 = MODE == 1 ? block_min(acc0, scratch) : block_sum(acc0, scratch);
    double r1 = MODE == 0 ? 0.0 : block_max(acc1, scratch);
    if (threadIdx.x == 0) {
        partial[2 * blockIdx.x] = r0;
        partial[2 * blockIdx.x + 1] = r1;
    }
}

template <int MODE>
__global__ void __launch_bounds__(256) reduce_stage2(const double* __restrict__ partial, int nblocks,
                                                      double* __restrict__ out) {
    __shared__ double scratch[32];
    double acc0 = MODE == 1 ? INFINITY : 0.0;
    double acc1 = -INFINITY;
    for (int i = threadIdx.x; i < nblocks; i += blockDim.x) {
        double p0 = partial[2 * i], p1 = partial[2 * i + 1];
        if (MODE == 1) acc0 = fmin(acc0, p0); else acc0 += p0;
        acc1 = fmax(acc1, p1);
    }
    double r0 = MODE == 1 ? block_min(acc0, scratch) : block_sum(acc0, scratch);
    double r1 = block_max(acc1, scratch);
    if (threadIdx.x == 0) {
        out[0] = r0;
        out[1] = r1;
    }
}

template <class T, int MODE>
static int reduce_to_device(ndmps_ctx* ctx, const T* a, const T* b, int64_t n, double* out_dev2) {
    int grid = reduce_grid(ctx, n, 8);
    double* partial = nullptr;
    NDMPS_TRY(ctx->ws.get<double>(2 * (size_t)grid, &partial));
    reduce_stage1<T, MODE><<<grid, 256, 0, ctx->stream>>>(a, b, n, partial);
    NDMPS_LAUNCH_CHECK(ctx);
    reduce_stage2<MODE><<<1, 256, 0, ctx->stream>>>(partial, grid, out_dev2);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

template <int MODE>
static int reduce_dispatch(ndmps_ctx* ctx, const void* a, const void* b, int64_t n, int dtype, double* out_dev2) {
    if (dtype == NDMPS_F32) return reduce_to_device<float, MODE>(ctx, (const float*)a, (const float*)b, n, out_dev2);
    return reduce_to_device<double, MODE>(ctx, (const double*)a, (const double*)b, n, out_dev2);
}

// ---- quantisation -------------------------------------------------------------
template <class T, class Q>
__global__ void __launch_bounds__(256) quantize_kernel(const T* __restrict__ x, int64_t n, double lo, double span,
                                                        double qmax, Q* __restrict__ q) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        // filetools.py:24-26: (x - min) / max(x - min) * iinfo.max, cast truncates toward zero
        // every step rounded separately (no FMA contraction) so the bytes match numpy's
        double u = __ddiv_rn(__dsub_rn((double)x[i], lo), span);
        double v = __dmul_rn(u, qmax);
        // NaN (0 / 0: a constant array, lo == hi) gives 0 for every type; the conversion alone gives 0x80...0 for the
        // 32- and 64-bit ones.  Values past the type's range (the top code of the 64-bit types, 2^64 or 2^63 in
        // float64) saturate in the conversion
        q[i] = isnan(v) ? (Q)0 : (Q)v;
    }
}

template <class T, class Q>
__global__ void __launch_bounds__(256) dequantize_kernel(const Q* __restrict__ q, int64_t n, double lo, double hi,
                                                          double qmax, T* __restrict__ x) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        // filetools.py:38-39: q / iinfo.max * (max - min) + min
        double u = __ddiv_rn((double)q[i], qmax);
        x[i] = (T)__dadd_rn(__dmul_rn(u, __dsub_rn(hi, lo)), lo);
    }
}

// {min, max} of one device array into out_dev2 (device), for callers inside the library
int minmax_device(ndmps_ctx* ctx, const void* x, int64_t n, int dtype, double* out_dev2) {
    return reduce_dispatch<1>(ctx, x, nullptr, n, dtype, out_dev2);
}

}  // namespace ndmps

using namespace ndmps;

// integer codes of the quantised type: +8/+16/+32/+64 unsigned, -8/-16/-32/-64 signed (numpy iinfo dtypes)
static bool qcode_ok(int code) { int a = code < 0 ? -code : code; return a == 8 || a == 16 || a == 32 || a == 64; }
static double qcode_max(int code) {
    switch (code) {
        case 8: return 255.0; case 16: return 65535.0; case 32: return 4294967295.0; case 64: return 18446744073709551615.0;
        case -8: return 127.0; case -16: return 32767.0; case -32: return 2147483647.0; default: return 9223372036854775807.0;
    }
}

template <class T>
static void launch_quantize(ndmps_ctx* ctx, int grid, const T* x, int64_t n, double lo, double span, double qmax, int code, void* q) {
#define NDMPS_Q(CODE, Q) case CODE: quantize_kernel<T, Q><<<grid, 256, 0, ctx->stream>>>(x, n, lo, span, qmax, (Q*)q); break
    switch (code) {
        NDMPS_Q(8, uint8_t); NDMPS_Q(16, uint16_t); NDMPS_Q(32, uint32_t); NDMPS_Q(64, uint64_t);
        NDMPS_Q(-8, int8_t); NDMPS_Q(-16, int16_t); NDMPS_Q(-32, int32_t); NDMPS_Q(-64, int64_t);
    }
#undef NDMPS_Q
}

template <class T>
static void launch_dequantize(ndmps_ctx* ctx, int grid, const void* q, int64_t n, double lo, double hi, double qmax, int code, T* x) {
#define NDMPS_Q(CODE, Q) case CODE: dequantize_kernel<T, Q><<<grid, 256, 0, ctx->stream>>>((const Q*)q, n, lo, hi, qmax, x); break
    switch (code) {
        NDMPS_Q(8, uint8_t); NDMPS_Q(16, uint16_t); NDMPS_Q(32, uint32_t); NDMPS_Q(64, uint64_t);
        NDMPS_Q(-8, int8_t); NDMPS_Q(-16, int16_t); NDMPS_Q(-32, int32_t); NDMPS_Q(-64, int64_t);
    }
#undef NDMPS_Q
}

extern "C" {

int ndmps_sumsq(ndmps_ctx_t* ctx, const void* x, int64_t n, int dtype, double* out_host) {
    NDMPS_REQUIRE(ctx && (x || n == 0) && out_host, "ndmps_sumsq: NULL argument");   // an empty tensor may have no storage
    NDMPS_REQUIRE(dtype_ok(dtype) && n >= 0, "ndmps_sumsq: bad dtype or size");
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    NDMPS_TRY(ensure_pinned(ctx, 2));
    double* out_dev = nullptr;
    NDMPS_TRY(ctx->ws.get<double>(2, &out_dev));
    NDMPS_TRY(reduce_dispatch<0>(ctx, x, nullptr, n, dtype, out_dev));
    NDMPS_TRY(readback(ctx, ctx->pinned, out_dev, 2 * sizeof(double)));
    NDMPS_CUDA_TRY(stream_wait(ctx));
    out_host[0] = ctx->pinned[0];
    return NDMPS_OK;
}

int ndmps_minmax(ndmps_ctx_t* ctx, const void* const* arrays, const int64_t* sizes, int count, int dtype,
                 double* out_host) {
    NDMPS_REQUIRE(ctx && arrays && sizes && out_host, "ndmps_minmax: NULL argument");
    NDMPS_REQUIRE(dtype_ok(dtype) && count >= 0, "ndmps_minmax: bad dtype or count");
    if (count == 0) return NDMPS_OK;
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    NDMPS_TRY(ensure_pinned(ctx, 2 * (size_t)count));
    double* out_dev = nullptr;
    NDMPS_TRY(ctx->ws.get<double>(2 * (size_t)count, &out_dev));
    for (int i = 0; i < count; i++) {
        NDMPS_REQUIRE(arrays[i] && sizes[i] > 0, "ndmps_minmax: array %d is empty", i);
        NDMPS_TRY(reduce_dispatch<1>(ctx, arrays[i], nullptr, sizes[i], dtype, out_dev + 2 * i));
    }
    NDMPS_TRY(readback(ctx, ctx->pinned, out_dev, 2 * (size_t)count * sizeof(double)));
    NDMPS_CUDA_TRY(stream_wait(ctx));
    memcpy(out_host, ctx->pinned, 2 * (size_t)count * sizeof(double));
    return NDMPS_OK;
}

int ndmps_psnr_terms(ndmps_ctx_t* ctx, const void* a, const void* b, int64_t n, int dtype, double* out_host) {
    NDMPS_REQUIRE(ctx && a && b && out_host, "ndmps_psnr_terms: NULL argument");
    NDMPS_REQUIRE(dtype_ok(dtype) && n > 0, "ndmps_psnr_terms: bad dtype or size");
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    NDMPS_TRY(ensure_pinned(ctx, 2));
    double* out_dev = nullptr;
    NDMPS_TRY(ctx->ws.get<double>(2, &out_dev));
    { StageScope sc(ctx, ST_METRIC); NDMPS_TRY(reduce_dispatch<2>(ctx, a, b, n, dtype, out_dev)); }
    NDMPS_TRY(readback(ctx, ctx->pinned, out_dev, 2 * sizeof(double)));
    NDMPS_CUDA_TRY(stream_wait(ctx));
    out_host[0] = ctx->pinned[0];
    out_host[1] = ctx->pinned[1];
    return NDMPS_OK;
}

int ndmps_quantize(ndmps_ctx_t* ctx, const void* x, int64_t n, int dtype, double lo, double hi, int bits, void* q_out) {
    NDMPS_REQUIRE(ctx && x && q_out, "ndmps_quantize: NULL argument");
    NDMPS_REQUIRE(dtype_ok(dtype) && n >= 0, "ndmps_quantize: bad dtype or size");
    NDMPS_REQUIRE(qcode_ok(bits), "ndmps_quantize: bits must be +-8, +-16, +-32 or +-64 (negative: signed), got %d", bits);
    if (n == 0) return NDMPS_OK;
    int grid = reduce_grid(ctx, n, 4);
    const double span = hi - lo, qmax = qcode_max(bits);
    if (dtype == NDMPS_F32) launch_quantize<float>(ctx, grid, (const float*)x, n, lo, span, qmax, bits, q_out);
    else launch_quantize<double>(ctx, grid, (const double*)x, n, lo, span, qmax, bits, q_out);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

int ndmps_dequantize(ndmps_ctx_t* ctx, const void* q, int64_t n, int bits, double lo, double hi, int dtype, void* x_out) {
    NDMPS_REQUIRE(ctx && q && x_out, "ndmps_dequantize: NULL argument");
    NDMPS_REQUIRE(dtype_ok(dtype) && n >= 0, "ndmps_dequantize: bad dtype or size");
    NDMPS_REQUIRE(qcode_ok(bits), "ndmps_dequantize: bits must be +-8, +-16, +-32 or +-64 (negative: signed), got %d", bits);
    if (n == 0) return NDMPS_OK;
    int grid = reduce_grid(ctx, n, 4);
    const double qmax = qcode_max(bits);
    if (dtype == NDMPS_F32) launch_dequantize<float>(ctx, grid, q, n, lo, hi, qmax, bits, (float*)x_out);
    else launch_dequantize<double>(ctx, grid, q, n, lo, hi, qmax, bits, (double*)x_out);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

}  // extern "C"
