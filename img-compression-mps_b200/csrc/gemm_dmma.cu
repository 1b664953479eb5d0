// General C = alpha * A * B on the FP64 tensor pipe (mma.sync m8n8k4 f64), exact float64
// accumulation of float32 / float64 operands.
//
// Used for the two big products of the path: the projection T = P^T M of the sweep
// (core/ndmps.py:74) and the final product of the reconstruction (core/ndmps.py:140).
// A is M x K with K contiguous (row-major, lda), B is K x N with N contiguous (row-major,
// ldb), C is M x N row-major (ldc).  CTA tile BM x 128 (BM = 64 or 128), BK = 16, one warp per
// 32 x 32 sub-tile; operands are converted to float64 when they are staged into shared
// memory (register-prefetched double buffering).  No split-K: callers use it when M*N is large.
#include "common.cuh"

namespace ndmps {

namespace gdm {

constexpr int BN = 128, BK = 16, LDA = BK + 4, LDB = BN + 4;   // strides chosen so the fragment reads are bank-conflict free

template <int BM, class TA, class TB, class TC>
__global__ void __launch_bounds__(BM * 4, BM == 64 ? 2 : 1)
gemm_dmma_kernel(int64_t M, int64_t N, int64_t K, const TA* __restrict__ A, int64_t lda, const TB* __restrict__ B, int64_t ldb,
                 TC* __restrict__ C, int64_t ldc, double alpha, int64_t tiles_n) {
    constexpr int THREADS = BM * 4;                     // one warp per 32 x 32 sub-tile
    constexpr int A_PER = BM * BK / THREADS;            // 4
    constexpr int B_PER = BK * BN / THREADS;            // 8 (BM = 64) or 4 (BM = 128)
    __shared__ double As[BM][LDA];
    __shared__ double Bs[BK][LDB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t tile_m = (int64_t)blockIdx.x / tiles_n, tile_n = (int64_t)blockIdx.x - tile_m * tiles_n;
    const int64_t m0 = tile_m * BM, n0 = tile_n * BN;
    const int wm = (warp >> 2) * 32, wn = (warp & 3) * 32;
    const int fr = lane >> 2, fc = lane & 3;

    double ra[A_PER], rb[B_PER];
    auto load_regs = [&](int64_t k0) {
#pragma unroll
        for (int i = 0; i < A_PER; i++) {
            const int e = tid + i * THREADS;            // BM x 16, k fastest
            const int r = e >> 4, kk = e & 15;
            const int64_t gr = m0 + r, gk = k0 + kk;
            ra[i] = (gr < M && gk < K) ? (double)A[gr * lda + gk] : 0.0;
        }
#pragma unroll
        for (int i = 0; i < B_PER; i++) {
            const int e = tid + i * THREADS;            // 16 x 128, n fastest
            const int kk = e >> 7, c = e & 127;
            const int64_t gk = k0 + kk, gc = n0 + c;
            rb[i] = (gk < K && gc < N) ? (double)B[gk * ldb + gc] : 0.0;
        }
    };
    auto store_smem = [&]() {
#pragma unroll
        for (int i = 0; i < A_PER; i++) {
            const int e = tid + i * THREADS;
            As[e >> 4][e & 15] = ra[i];
        }
#pragma unroll
        for (int i = 0; i < B_PER; i++) {
            const int e = tid + i * THREADS;
            Bs[e >> 7][e & 127] = rb[i];
        }
    };

    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

    load_regs(0);
    for (int64_t k0 = 0; k0 < K; k0 += BK) {
        store_smem();
        __syncthreads();
        if (k0 + BK < K) load_regs(k0 + BK);
#pragma unroll
        for (int k4 = 0; k4 < BK / 4; k4++) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; i++) a[i] = As[wm + i * 8 + fr][k4 * 4 + fc];
#pragma unroll
            for (int j = 0; j < 4; j++) b[j] = Bs[k4 * 4 + fc][wn + j * 8 + fr];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) mma_f64(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int64_t r = m0 + wm + i * 8 + fr;
        if (r >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int64_t c = n0 + wn + j * 8 + 2 * fc;
            if (c < N) C[r * ldc + c] = (TC)(alpha * acc[i][j][0]);
            if (c + 1 < N) C[r * ldc + c + 1] = (TC)(alpha * acc[i][j][1]);
        }
    }
}

template <int BM, class TA, class TB, class TC>
static int launch(ndmps_ctx* ctx, int64_t M, int64_t N, int64_t K, double alpha, const void* a, int64_t lda, const void* b,
                  int64_t ldb, void* c, int64_t ldc) {
    const int64_t tiles_m = (M + BM - 1) / BM, tiles_n = (N + BN - 1) / BN;
    gemm_dmma_kernel<BM, TA, TB, TC><<<(unsigned)(tiles_m * tiles_n), BM * 4, 0, ctx->stream>>>(
        M, N, K, (const TA*)a, lda, (const TB*)b, ldb, (TC*)c, ldc, alpha, tiles_n);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

template <int BM>
static int dispatch(ndmps_ctx* ctx, int64_t M, int64_t N, int64_t K, double alpha, const void* a, int da, int64_t lda,
                    const void* b, int db, int64_t ldb, void* c, int dc, int64_t ldc) {
    const int key = (da == NDMPS_F64) * 4 + (db == NDMPS_F64) * 2 + (dc == NDMPS_F64);
    switch (key) {
        case 0: return launch<BM, float, float, float>(ctx, M, N, K, alpha, a, lda, b, ldb, c, ldc);
        case 1: return launch<BM, float, float, double>(ctx, M, N, K, alpha, a, lda, b, ldb, c, ldc);
        case 2: return launch<BM, float, double, float>(ctx, M, N, K, alpha, a, lda, b, ldb, c, ldc);
        case 3: return launch<BM, float, double, double>(ctx, M, N, K, alpha, a, lda, b, ldb, c, ldc);
        case 4: return launch<BM, double, float, float>(ctx, M, N, K, alpha, a, lda, b, ldb, c, ldc);
        case 5: return launch<BM, double, float, double>(ctx, M, N, K, alpha, a, lda, b, ldb, c, ldc);
        case 6: return launch<BM, double, double, float>(ctx, M, N, K, alpha, a, lda, b, ldb, c, ldc);
        default: return launch<BM, double, double, double>(ctx, M, N, K, alpha, a, lda, b, ldb, c, ldc);
    }
}

}  // namespace gdm

// Takes the product when A is K-contiguous, B is N-contiguous and the output is large enough to
// fill the machine without split-K; otherwise leaves *done = false for the SIMT kernel.
int gemm_dmma(ndmps_ctx* ctx, int64_t m, int64_t n, int64_t k, double alpha, const void* a, int dtype_a, int64_t a_rs,
              int64_t a_cs, const void* b, int dtype_b, int64_t b_rs, int64_t b_cs, void* c, int dtype_c, int64_t ldc,
              bool* done) {
    *done = false;
    if (a_cs != 1 || b_cs != 1 || m < 48 || n < 64 || k < 4) return NDMPS_OK;   // n = 64: half of the 128-wide tile idles, still ahead of SIMT
    const int64_t tiles64 = ((m + 63) / 64) * ((n + gdm::BN - 1) / gdm::BN);
    if (tiles64 < ctx->sm_count) return NDMPS_OK;          // would need split-K: SIMT path has it
    if (tiles64 >= (int64_t(1) << 31)) return NDMPS_OK;
    // BM = 64 when M is a small multiple of 64 (the projection), else 128
    const bool small_m = m <= 64 || (m % 128 != 0 && m % 128 <= 64 && m < 512);
    if (small_m) NDMPS_TRY(gdm::dispatch<64>(ctx, m, n, k, alpha, a, dtype_a, a_rs, b, dtype_b, b_rs, c, dtype_c, ldc));
    else NDMPS_TRY(gdm::dispatch<128>(ctx, m, n, k, alpha, a, dtype_a, a_rs, b, dtype_b, b_rs, c, dtype_c, ldc));
    *done = true;
    return NDMPS_OK;
}

}  // namespace ndmps
