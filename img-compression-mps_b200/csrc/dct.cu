// K11: orthonormal DCT-II / DCT-III along the last axis
// (scipy.fftpack.dct(x, norm="ortho") / idct at core/ndmps.py:63,153; SURVEY A.6).
//
// Matrix form: y = x C^T with C[k, i] = sqrt(2/n) cos(pi (2i+1) k / (2n)), row 0
// scaled by 1/sqrt(2).  C is orthogonal, so the inverse is x = y C.  The lines are
// the GEMM's M dimension; accumulation is float64, any n.
#include "common.cuh"

namespace ndmps {

// C (row-major, C[k][i]) when transposed == 0, C^T (Ct[i][k]) otherwise: both products of the transform then read
// their small operand along its rows, which is what the FP64 tensor-pipe GEMM wants
__global__ void __launch_bounds__(256) dct_matrix_kernel(double* __restrict__ C, int64_t n, int transposed) {
    int64_t total = n * n, stride = (int64_t)gridDim.x * blockDim.x;
    const double scale = sqrt(2.0 / (double)n);
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        int64_t k = e / n, i = e - k * n;
        // reduce (2i+1) k modulo 4n exactly so cospi sees a small argument
        int64_t q = ((2 * i + 1) * k) % (4 * n);
        double v = scale * cospi((double)q / (double)(2 * n));
        if (k == 0) v *= 0.70710678118654752440;
        C[transposed ? i * n + k : e] = v;
    }
}

// B[k][j] = (1/block) sum_{t in block j} C[k][t] (n x n/block): the DCT-III matrix averaged over column blocks, so that
// y B is the block mean of the inverse transform y C
__global__ void __launch_bounds__(256) dct_block_mean_matrix_kernel(double* __restrict__ B, int64_t n, int64_t block) {
    const int64_t m = n / block, total = n * m, stride = (int64_t)gridDim.x * blockDim.x;
    const double scale = sqrt(2.0 / (double)n) / (double)block;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        const int64_t k = e / m, j = e - k * m;
        double s = 0.0;
        for (int64_t t = j * block; t < (j + 1) * block; t++) s += cospi((double)(((2 * t + 1) * k) % (4 * n)) / (double)(2 * n));
        B[e] = (k == 0 ? 0.70710678118654752440 : 1.0) * scale * s;
    }
}

int dct_matrix(ndmps_ctx* ctx, int64_t n, int inverse, double** C_out) {
    double* C = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)(n * n), &C));
    int64_t want = (n * n + 255) / 256, cap = (int64_t)ctx->sm_count * 8;
    dct_matrix_kernel<<<(int)(want < cap ? want : cap), 256, 0, ctx->stream>>>(C, n, inverse ? 0 : 1);
    NDMPS_LAUNCH_CHECK(ctx);
    *C_out = C;
    return NDMPS_OK;
}

// forward: y[l, k] = sum_i x[l, i] C[k, i] = sum_i x[l, i] Ct[i, k]; inverse: x[l, i] = sum_k y[l, k] C[k, i].  Both are
// dst = src . C with the matrix dct_matrix built for the direction.
int dct_lines(ndmps_ctx* ctx, const void* src, void* dst, int64_t lines, int64_t n, int dtype, const double* C) {
    return payload_gemm(ctx, lines * n, lines, n, n, src, dtype, n, 1, C, NDMPS_F64, n, 1, dst, dtype, n);
}

}  // namespace ndmps

using namespace ndmps;

extern "C" {

int ndmps_dct_last_axis(ndmps_ctx_t* ctx, const void* src, void* dst, int64_t lines, int64_t n, int inverse, int dtype) {
    NDMPS_REQUIRE(ctx && src && dst, "ndmps_dct_last_axis: NULL argument");
    NDMPS_REQUIRE(dtype_ok(dtype) && lines >= 0 && n >= 1, "ndmps_dct_last_axis: bad shape or dtype");
    NDMPS_REQUIRE(src != dst, "ndmps_dct_last_axis: in-place transform is not supported");
    if (lines == 0) return NDMPS_OK;
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    StageScope sc(ctx, ST_DCT);
    double* C = nullptr;
    NDMPS_TRY(dct_matrix(ctx, n, inverse, &C));
    return dct_lines(ctx, src, dst, lines, n, dtype, C);
}

int ndmps_idct_block_mean_last_axis(ndmps_ctx_t* ctx, const void* src, void* dst, int64_t lines, int64_t n, int64_t block, int dtype) {
    NDMPS_REQUIRE(ctx && src && dst, "ndmps_idct_block_mean_last_axis: NULL argument");
    NDMPS_REQUIRE(dtype_ok(dtype) && lines >= 0 && n >= 1, "ndmps_idct_block_mean_last_axis: bad shape or dtype");
    NDMPS_REQUIRE(block >= 1 && n % block == 0, "ndmps_idct_block_mean_last_axis: block %lld does not divide n = %lld",
                  (long long)block, (long long)n);
    NDMPS_REQUIRE(src != dst, "ndmps_idct_block_mean_last_axis: in-place transform is not supported");
    if (lines == 0) return NDMPS_OK;
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    StageScope sc(ctx, ST_DCT);
    const int64_t m = n / block;
    double* B = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)(n * m), &B));
    int64_t want = (n * m + 255) / 256, cap = (int64_t)ctx->sm_count * 8;
    dct_block_mean_matrix_kernel<<<(int)(want < cap ? want : cap), 256, 0, ctx->stream>>>(B, n, block);
    NDMPS_LAUNCH_CHECK(ctx);
    // the payload is the input (lines x n), as for ndmps_dct_last_axis
    return payload_gemm(ctx, lines * n, lines, m, n, src, dtype, n, 1, B, NDMPS_F64, m, 1, dst, dtype, m);
}

}  // extern "C"
