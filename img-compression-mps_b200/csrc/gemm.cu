// Generic strided GEMM with float64 accumulation (SIMT, DFMA pipe).
//
// This is the *exact* arithmetic path of the sweep: Gram matrices of float32
// unfoldings are accumulated in float64 (products of float32 values are exact in
// float64), and all bond-sized glue (r x r, <= a few thousand) runs through it.
// B200 keeps a full-rate FP64 pipe (about half the FP32 SIMT rate), so this path is
// not the bottleneck for bond-sized problems; the long-K Gram of the first
// unfoldings of a capped float32 sweep goes to tcgen05 on split planes (tc_gemm.cu).
//
// C (m x n, row-major, ldc) = alpha * A (m x k) * B (k x n); A and B are addressed
// as a[i*rs + j*cs], so transposes and K-major / MN-major operands need no copies.
// Tiles 64 x 64 x 16, 256 threads, 4 x 4 outputs per thread, register-staged
// double buffering, optional split-K with float64 partials reduced in a fixed order
// (deterministic).
#include "common.cuh"

namespace ndmps {

constexpr int BM = 64, BN = 64, BK = 16;

template <class T>
__device__ __forceinline__ void load_tile(const T* __restrict__ p, int64_t rs, int64_t cs, int64_t r0, int64_t k0,
                                          int64_t rmax, int64_t kmax, bool k_fast, int tid, double (&reg)[4]) {
    // tile element (r, kk): r in [0,64) is the M (or N) index, kk in [0,16) the K index
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int e = tid + 256 * i;
        int r = k_fast ? (e >> 4) : (e & 63);
        int kk = k_fast ? (e & 15) : (e >> 6);
        int64_t gr = r0 + r, gk = k0 + kk;
        reg[i] = (gr < rmax && gk < kmax) ? (double)p[gr * rs + gk * cs] : 0.0;
    }
}

__device__ __forceinline__ void store_tile(double (*s)[BM + 2], bool k_fast, int tid, const double (&reg)[4]) {
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int e = tid + 256 * i;
        int r = k_fast ? (e >> 4) : (e & 63);
        int kk = k_fast ? (e & 15) : (e >> 6);
        s[kk][r] = reg[i];
    }
}

template <class TA, class TB>
__global__ void __launch_bounds__(256)
gemm_f64acc_kernel(int64_t M, int64_t N, int64_t K, const TA* __restrict__ A, int64_t a_rs, int64_t a_cs,
                   const TB* __restrict__ B, int64_t b_rs, int64_t b_cs, double* __restrict__ partial,
                   void* __restrict__ C, int dtype_c, int64_t ldc, double alpha, int64_t k_per_split,
                   int64_t tiles_n) {
    __shared__ double As[BK][BM + 2];
    __shared__ double Bs[BK][BN + 2];
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int64_t tile_m = (int64_t)blockIdx.x / tiles_n, tile_n = (int64_t)blockIdx.x - tile_m * tiles_n;
    const int64_t m0 = tile_m * BM, n0 = tile_n * BN;
    const int64_t kbeg = (int64_t)blockIdx.y * k_per_split;
    const int64_t kend = kbeg + k_per_split < K ? kbeg + k_per_split : K;
    // the K index runs fastest across threads when it is the operand's smaller stride
    const bool a_kfast = a_cs <= a_rs;
    const bool b_kfast = b_rs <= b_cs;

    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = 0.0;

    double ra[4], rb[4];
    if (kbeg < kend) {
        load_tile<TA>(A, a_rs, a_cs, m0, kbeg, M, kend, a_kfast, tid, ra);
        load_tile<TB>(B, b_cs, b_rs, n0, kbeg, N, kend, b_kfast, tid, rb);
    }
    for (int64_t k0 = kbeg; k0 < kend; k0 += BK) {
        store_tile(As, a_kfast, tid, ra);
        store_tile(Bs, b_kfast, tid, rb);
        __syncthreads();
        if (k0 + BK < kend) {
            load_tile<TA>(A, a_rs, a_cs, m0, k0 + BK, M, kend, a_kfast, tid, ra);
            load_tile<TB>(B, b_cs, b_rs, n0, k0 + BK, N, kend, b_kfast, tid, rb);
        }
#pragma unroll
        for (int kk = 0; kk < BK; kk++) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; i++) a[i] = As[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; j++) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) acc[i][j] = fma(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }

    if (partial != nullptr) {
        double* dst = partial + (int64_t)blockIdx.y * M * N;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            int64_t r = m0 + ty * 4 + i;
            if (r >= M) continue;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                int64_t c = n0 + tx * 4 + j;
                if (c < N) dst[r * N + c] = acc[i][j];
            }
        }
    } else {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            int64_t r = m0 + ty * 4 + i;
            if (r >= M) continue;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                int64_t c = n0 + tx * 4 + j;
                if (c >= N) continue;
                double v = alpha * acc[i][j];
                if (dtype_c == NDMPS_F32) ((float*)C)[r * ldc + c] = (float)v;
                else ((double*)C)[r * ldc + c] = v;
            }
        }
    }
}

__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const double* __restrict__ partial, int splits, int64_t M, int64_t N, void* __restrict__ C,
                     int dtype_c, int64_t ldc, double alpha) {
    int64_t total = M * N;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        double s = 0.0;
        for (int z = 0; z < splits; z++) s += partial[(int64_t)z * total + i];
        s *= alpha;
        int64_t r = i / N, c = i - r * N;
        if (dtype_c == NDMPS_F32) ((float*)C)[r * ldc + c] = (float)s;
        else ((double*)C)[r * ldc + c] = s;
    }
}

int gemm(ndmps_ctx* ctx, int64_t m, int64_t n, int64_t k, double alpha,
         const void* a, int dtype_a, int64_t a_rs, int64_t a_cs,
         const void* b, int dtype_b, int64_t b_rs, int64_t b_cs,
         void* c, int dtype_c, int64_t ldc) {
    NDMPS_REQUIRE(m >= 0 && n >= 0 && k >= 0, "gemm: negative size");
    NDMPS_REQUIRE(dtype_ok(dtype_a) && dtype_ok(dtype_b) && dtype_ok(dtype_c), "gemm: bad dtype");
    if (m == 0 || n == 0) return NDMPS_OK;
    if (ctx->opt_gemm_path == 3) {
        // tcgen05 on bf16x3 planes (tc_gemm.cu): float32-class products of the capped sweep and the reconstruction
        bool done = false;
        NDMPS_TRY(gemm_tc(ctx, m, n, k, alpha, a, dtype_a, a_rs, a_cs, b, dtype_b, b_rs, b_cs, c, dtype_c, ldc,
                          ctx->opt_gemm_out_t != 0, &done));
        if (done) return NDMPS_OK;
        NDMPS_REQUIRE(ctx->opt_gemm_out_t == 0, "gemm: transposed output needs the tcgen05 path (shape not eligible)");
    }
    if (ctx->opt_gemm_path != 2) {   // large row-major products go to the FP64 tensor pipe (gemm_dmma.cu)
        bool done = false;
        NDMPS_TRY(gemm_dmma(ctx, m, n, k, alpha, a, dtype_a, a_rs, a_cs, b, dtype_b, b_rs, b_cs, c, dtype_c, ldc, &done));
        if (done) return NDMPS_OK;
    }
    int64_t tiles_m = (m + BM - 1) / BM, tiles_n = (n + BN - 1) / BN;
    int64_t tiles = tiles_m * tiles_n;
    NDMPS_REQUIRE(tiles < (int64_t(1) << 31), "gemm: %lld x %lld output too large for one launch", (long long)m, (long long)n);
    int64_t target = 2 * (int64_t)ctx->sm_count;
    int64_t splits = 1;
    if (tiles < target && k >= 128) {                        // few output tiles: spread K over CTAs (bond-sized products)
        splits = (target + tiles - 1) / tiles;
        int64_t max_splits = (k + 63) / 64;
        if (splits > max_splits) splits = max_splits;
        if (splits > 2048) splits = 2048;
        // keep the float64 partial buffer modest
        while (splits > 1 && splits * m * n * 8 > (int64_t(256) << 20)) splits = (splits + 1) / 2;
    }
    int64_t k_per = (k + splits - 1) / splits;
    k_per = ((k_per + BK - 1) / BK) * BK;
    if (k_per == 0) k_per = BK;
    splits = k > 0 ? (k + k_per - 1) / k_per : 1;
    double* partial = nullptr;
    if (splits > 1) NDMPS_TRY(ctx->ws.get<double>((size_t)(splits * m * n), &partial));
    dim3 grid((unsigned)tiles, (unsigned)splits, 1);
#define NDMPS_GEMM_LAUNCH(TA, TB)                                                                               \
    gemm_f64acc_kernel<TA, TB><<<grid, 256, 0, ctx->stream>>>(m, n, k, (const TA*)a, a_rs, a_cs, (const TB*)b,  \
                                                              b_rs, b_cs, partial, c, dtype_c, ldc, alpha, k_per, tiles_n)
    if (dtype_a == NDMPS_F32 && dtype_b == NDMPS_F32) NDMPS_GEMM_LAUNCH(float, float);
    else if (dtype_a == NDMPS_F32) NDMPS_GEMM_LAUNCH(float, double);
    else if (dtype_b == NDMPS_F32) NDMPS_GEMM_LAUNCH(double, float);
    else NDMPS_GEMM_LAUNCH(double, double);
#undef NDMPS_GEMM_LAUNCH
    NDMPS_LAUNCH_CHECK(ctx);
    if (splits > 1) {
        int64_t total = m * n;
        int64_t want = (total + 255) / 256, cap = (int64_t)ctx->sm_count * 8;
        int g = (int)(want < cap ? want : cap);
        splitk_reduce_kernel<<<g, 256, 0, ctx->stream>>>(partial, (int)splits, m, n, c, dtype_c, ldc, alpha);
        NDMPS_LAUNCH_CHECK(ctx);
    }
    return NDMPS_OK;
}

// float32 payloads from 2^20 elements on: the product on tcgen05 (bf16x3 planes, tc_gemm.cu)
int payload_gemm(ndmps_ctx* ctx, int64_t payload, int64_t m, int64_t n, int64_t k,
                 const void* a, int dtype_a, int64_t a_rs, int64_t a_cs,
                 const void* b, int dtype_b, int64_t b_rs, int64_t b_cs,
                 void* c, int dtype_c, int64_t ldc) {
    if (ctx->opt_tc && dtype_c == NDMPS_F32 && payload >= (int64_t(1) << 20)) {
        bool done = false;
        NDMPS_TRY(gemm_tc(ctx, m, n, k, 1.0, a, dtype_a, a_rs, a_cs, b, dtype_b, b_rs, b_cs, c, dtype_c, ldc, false, &done));
        if (done) return NDMPS_OK;
    }
    return gemm(ctx, m, n, k, 1.0, a, dtype_a, a_rs, a_cs, b, dtype_b, b_rs, b_cs, c, dtype_c, ldc);
}

int gram(ndmps_ctx* ctx, const void* mat, int64_t rows, int64_t cols, int64_t ld, int dtype, int side, double* g_dev, TcDigits* tc) {
    if (side == 0 && (ctx->opt_gram_path == 3 || (ctx->opt_gram_path == 0 && tc != nullptr))) {
        // sliced-integer Gram on tcgen05 kind::i8 (tc_gemm.cu): float32 unfoldings of a capped sweep.  Exact accumulation,
        // five 7-bit digits; rows too heavy-tailed for five digits go to the FP64-pipe kernel through a device-side flag
        TcDigits dropped;
        bool done = false;
        NDMPS_TRY(gram_tc(ctx, mat, rows, cols, ld, dtype, g_dev, tc ? tc : &dropped, &done));
        if (done) return NDMPS_OK;
    }
    if (side == 0 && ctx->opt_gram_path != 2) {   // FP64 tensor-pipe path when the shape allows (gram_dmma.cu)
        bool done = false;
        NDMPS_TRY(gram_dmma(ctx, mat, rows, cols, ld, dtype, g_dev, &done));
        if (done) return NDMPS_OK;
    }
    if (side == 0)  // G = M M^T : A = M (rows x cols), B = M^T
        return gemm(ctx, rows, rows, cols, 1.0, mat, dtype, ld, 1, mat, dtype, 1, ld, g_dev, NDMPS_F64, rows);
    // G = M^T M : A = M^T (cols x rows), B = M
    return gemm(ctx, cols, cols, rows, 1.0, mat, dtype, 1, ld, mat, dtype, ld, 1, g_dev, NDMPS_F64, cols);
}

}  // namespace ndmps

using namespace ndmps;

extern "C" {

int ndmps_gemm(ndmps_ctx_t* ctx, int64_t m, int64_t n, int64_t k, double alpha,
               const void* a, int dtype_a, int64_t a_rs, int64_t a_cs,
               const void* b, int dtype_b, int64_t b_rs, int64_t b_cs,
               void* c, int dtype_c, int64_t ldc) {
    NDMPS_REQUIRE(ctx && a && b && c, "ndmps_gemm: NULL argument");
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    return gemm(ctx, m, n, k, alpha, a, dtype_a, a_rs, a_cs, b, dtype_b, b_rs, b_cs, c, dtype_c, ldc);
}

int ndmps_gram(ndmps_ctx_t* ctx, const void* m, int64_t rows, int64_t cols, int64_t ld, int dtype, int side,
               double* g_dev) {
    NDMPS_REQUIRE(ctx && m && g_dev, "ndmps_gram: NULL argument");
    NDMPS_REQUIRE(dtype_ok(dtype) && rows > 0 && cols > 0 && ld >= cols, "ndmps_gram: bad shape or dtype");
    NDMPS_REQUIRE(side == 0 || side == 1, "ndmps_gram: side must be 0 or 1");
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    return gram(ctx, m, rows, cols, ld, dtype, side, g_dev);
}

}  // extern "C"
