// K2 fast path: G = M M^T on the FP64 tensor pipe (mma.sync m8n8k4 f64), exact.
//
// The Gram matrix of a float32 unfolding must be accumulated in float64 (DESIGN.md section 4:
// rank decisions sit at lambda/lambda_max ~ 1e-10, and products of float32 values are exact in
// float64).  tcgen05 has no float64 kind, so the tensor-core route for this contraction is the
// DMMA instruction: float32 tiles are staged global -> shared with cp.async (16-byte chunks,
// 3 stages), converted to float64 when the fragments are read, and multiplied 8x8x4 at a time.
//
// M: m x K row-major float32 (K contiguous, leading dimension ld, ld % 4 == 0, 16-byte aligned).
// CTA tile 128 x 128, 16 warps of 32 x 32, BK = 32.  Only tiles on or above the diagonal are
// computed; split-K partials go to a float64 buffer and a fixed-order reduction writes both
// triangles (deterministic, bitwise symmetric).
#include "common.cuh"

namespace ndmps {

namespace dmma {

constexpr int TM = 128, BK = 32, LDS = BK + 4, STAGES = 3, THREADS = 512;

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, int src_bytes) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__global__ void __launch_bounds__(THREADS, 1)
gram_dmma_kernel(const float* __restrict__ M, int m, int64_t K, int64_t ld, int nt, int64_t k_per, double* __restrict__ partial,
                 const int* __restrict__ run_flag) {
    if (run_flag != nullptr && run_flag[0] == 0) return;     // the tensor-core Gram took this matrix (tc_gemm.cu)
    extern __shared__ float smem[];
    float* As = smem;                                   // STAGES x TM x LDS
    float* Bs = smem + (size_t)STAGES * TM * LDS;       // STAGES x TM x LDS
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int ti, tj;
    upper_tile(blockIdx.x, nt, ti, tj);
    const int split = blockIdx.y;
    const int64_t kbeg = (int64_t)split * k_per;
    const int64_t kend = kbeg + k_per < K ? kbeg + k_per : K;
    const int nk = (int)((kend - kbeg + BK - 1) / BK);
    const int row_a0 = ti * TM, row_b0 = tj * TM;

    auto load_stage = [&](int stage, int kt) {
        const int64_t k0 = kbeg + (int64_t)kt * BK;
        // 128 rows x 8 chunks of 4 floats per operand; 512 threads -> 2 chunks each per operand
#pragma unroll
        for (int it = 0; it < 2; it++) {
            const int c = tid + it * THREADS;           // 0..1023
            const int r = c >> 3, ch = c & 7;
            const int64_t k = k0 + ch * 4;
            int bytes = 0;
            if (k < kend) { int64_t rem = kend - k; bytes = rem >= 4 ? 16 : (int)rem * 4; }
            {
                const int gr = row_a0 + r;
                const bool ok = gr < m && bytes > 0;
                const float* src = M + (ok ? (int64_t)gr * ld + k : 0);
                cp_async16(As + ((size_t)stage * TM + r) * LDS + ch * 4, src, ok ? bytes : 0);
            }
            {
                const int gr = row_b0 + r;
                const bool ok = gr < m && bytes > 0;
                const float* src = M + (ok ? (int64_t)gr * ld + k : 0);
                cp_async16(Bs + ((size_t)stage * TM + r) * LDS + ch * 4, src, ok ? bytes : 0);
            }
        }
    };

    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

    for (int s = 0; s < STAGES - 1; s++) {
        if (s < nk) load_stage(s, s);
        cp_async_commit();
    }
    const int wm = (warp >> 2) * 32, wn = (warp & 3) * 32;
    const int fr = lane >> 2, fc = lane & 3;            // fragment row (0..7) and k column (0..3)
    for (int kt = 0; kt < nk; kt++) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        const int nxt = kt + STAGES - 1;
        if (nxt < nk) load_stage(nxt % STAGES, nxt);
        cp_async_commit();
        const float* a_s = As + (size_t)(kt % STAGES) * TM * LDS;
        const float* b_s = Bs + (size_t)(kt % STAGES) * TM * LDS;
#pragma unroll
        for (int k4 = 0; k4 < BK / 4; k4++) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; i++) a[i] = (double)a_s[(size_t)(wm + i * 8 + fr) * LDS + k4 * 4 + fc];
#pragma unroll
            for (int j = 0; j < 4; j++) b[j] = (double)b_s[(size_t)(wn + j * 8 + fr) * LDS + k4 * 4 + fc];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) mma_f64(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
    }
    cp_async_wait<0>();
    // partial[split][tile][128][128]
    double* out = partial + ((size_t)split * gridDim.x + blockIdx.x) * TM * TM;
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int r = wm + i * 8 + fr, c = wn + j * 8 + 2 * fc;
            *reinterpret_cast<double2*>(out + (size_t)r * TM + c) = make_double2(acc[i][j][0], acc[i][j][1]);
        }
}

// G[i][j] = G[j][i] = sum over splits, in split order
__global__ void __launch_bounds__(256)
gram_dmma_reduce_kernel(const double* __restrict__ partial, int m, int nt, int ntiles, int splits, double* __restrict__ G,
                        const int* __restrict__ run_flag) {
    if (run_flag != nullptr && run_flag[0] == 0) return;
    const int tile = blockIdx.y;
    int ti, tj;
    upper_tile(tile, nt, ti, tj);
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < TM * TM; e += gridDim.x * blockDim.x) {
        const int r = e / TM, c = e - r * TM;
        const int gi = ti * TM + r, gj = tj * TM + c;
        if (gi >= m || gj >= m) continue;
        if (ti == tj && gj < gi) continue;               // lower half of a diagonal tile: mirrored below
        double s = 0.0;
        for (int z = 0; z < splits; z++) s += partial[((size_t)z * ntiles + tile) * TM * TM + e];
        G[(size_t)gi * m + gj] = s;
        G[(size_t)gj * m + gi] = s;
    }
}

}  // namespace dmma

// returns NDMPS_OK and sets *done = true when the fast path ran
int gram_dmma(ndmps_ctx* ctx, const void* mat, int64_t rows, int64_t cols, int64_t ld, int dtype, double* g_dev, bool* done,
              const int* run_flag) {
    using namespace dmma;
    *done = false;
    if (dtype != NDMPS_F32 || rows < 48 || rows > 4096 || cols < 4 * BK) return NDMPS_OK;
    if ((ld & 3) != 0 || (reinterpret_cast<uintptr_t>(mat) & 15) != 0) return NDMPS_OK;
    const int m = (int)rows;
    const int nt = (m + TM - 1) / TM;
    const int ntiles = nt * (nt + 1) / 2;
    // one CTA per SM is resident (111 registers x 512 threads): fill whole waves, 2 x sm_count CTAs at most
    int64_t splits = (2 * (int64_t)ctx->sm_count) / ntiles;
    const int64_t max_splits = (cols + 4 * BK - 1) / (4 * BK);
    if (splits > max_splits) splits = max_splits;
    if (splits < 1) splits = 1;
    int64_t k_per = (cols + splits - 1) / splits;
    k_per = ((k_per + BK - 1) / BK) * BK;
    splits = (cols + k_per - 1) / k_per;
    double* partial = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)splits * ntiles * TM * TM, &partial));
    const size_t smem = (size_t)2 * STAGES * TM * LDS * sizeof(float);
    NDMPS_TRY(raise_dynamic_smem((const void*)gram_dmma_kernel, ctx->device, (int)smem));
    dim3 grid((unsigned)ntiles, (unsigned)splits);
    gram_dmma_kernel<<<grid, THREADS, smem, ctx->stream>>>((const float*)mat, m, cols, ld, nt, k_per, partial, run_flag);
    NDMPS_LAUNCH_CHECK(ctx);
    dim3 rgrid(16, (unsigned)ntiles);
    gram_dmma_reduce_kernel<<<rgrid, 256, 0, ctx->stream>>>(partial, m, nt, ntiles, (int)splits, g_dev, run_flag);
    NDMPS_LAUNCH_CHECK(ctx);
    *done = true;
    return NDMPS_OK;
}

}  // namespace ndmps
