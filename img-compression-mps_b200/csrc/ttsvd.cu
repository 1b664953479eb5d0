// K2-K8 drivers: left -> right TT-SVD sweep, pairwise bond truncation, MPS -> dense
// contraction and MPS overlap, built from gram / eigh / gemm.
//
// Sweep (qtn.MatrixProductState.from_dense at core/ndmps.py:74; SURVEY Appendix A.1):
// step i factorises the unfolding M_i ((r_{i-1} d_i) x C_i).  Here:
//
//   * left factor from the Gram matrix G = M M^T (float64 accumulation) and a
//     float64 Jacobi eigensolve: U = eigenvectors, s = sqrt(lambda); the remainder
//     is T = U_r^T M (= diag(s) V^T, weight absorbed right as quimb does).
//   * FRONT MERGING: consecutive sites whose fused row count stays <= MERGE_CAP (512)
//     share ONE Gram pass and ONE projection pass over the big unfolding.  With
//     rows (a, s_i, .., s_{i+k-1}) fused, the Gram of sub-step j is
//         G_j = (P_j (x) I)^T  Tr_rest(G)  (P_j (x) I)
//     where P_j is the accumulated isometry of the earlier sub-steps and Tr_rest the
//     partial trace over the not-yet-split row digits, so every core of the group
//     comes from small float64 algebra on G and the data is read twice in total.
//     This is exactly the sequential algorithm (truncation and renorm included).
//   * when an unfolding has more rows than columns (late steps) the Gram is taken
//     on the column side: G' = M^T M = V s^2 V^T, U = M V / s.
#include <math.h>

#include "common.cuh"

namespace ndmps {

constexpr int64_t MERGE_CAP = 512;   // largest fused row count of a front-merged group of sites

// ---------------------------------------------------------------------------------
// small float64 glue kernels
// ---------------------------------------------------------------------------------
// Gt[x, y] = sum_t G[(x*rest + t), (y*rest + t)]     G: D x D, D = X*rest
__global__ void __launch_bounds__(256) partial_trace_kernel(const double* __restrict__ G, int64_t D, int64_t X, int64_t rest,
                                                             double* __restrict__ Gt) {
    int64_t total = X * X, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        int64_t x = i / X, y = i - x * X;
        double s = 0.0;
        for (int64_t t = 0; t < rest; t++) s += G[(x * rest + t) * D + (y * rest + t)];
        Gt[i] = s;
    }
}

// K = P (x) I_d : K[(p*d + s), (b*d + s')] = P[p, b] * delta(s, s');  P: pd x r
__global__ void __launch_bounds__(256) kron_identity_kernel(const double* __restrict__ P, int64_t pd, int64_t r, int64_t d,
                                                             double* __restrict__ K) {
    int64_t rows = pd * d, cols = r * d, total = rows * cols, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        int64_t row = i / cols, col = i - row * cols;
        int64_t p = row / d, s = row - p * d, b = col / d, s2 = col - b * d;
        K[i] = s == s2 ? P[p * r + b] : 0.0;
    }
}

// per-column scale vector from eigenvalues:  out[j] = f(lambda_j)
//   mode 0: sqrt(l)   mode 1: 1/sqrt(l)   mode 2: l^(-1/4)   mode 3: l^(-3/4)
// times `factor`; entries whose sqrt(l) <= floor_rel * sqrt(l_0) give 0 for the inverse modes.
__global__ void col_scale_kernel(const double* __restrict__ evals, int64_t n, int mode, double factor, double floor_rel,
                                 double* __restrict__ out) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    double l0 = evals[0] > 0.0 ? evals[0] : 0.0;
    double l = evals[j] > 0.0 ? evals[j] : 0.0;
    double s = sqrt(l), s0 = sqrt(l0);
    double v;
    if (mode == 0) v = s;
    else if (s <= floor_rel * s0 || s == 0.0) v = 0.0;
    else if (mode == 1) v = 1.0 / s;
    else if (mode == 2) v = 1.0 / sqrt(s);
    else v = 1.0 / (s * sqrt(s));
    out[j] = v * factor;
}

// dst[i, j] = src[i*ld_src + j] * (colscale ? colscale[j] : 1) * (rowscale ? rowscale[i] : 1) * alpha, converted
template <class T>
__global__ void __launch_bounds__(256)
scale_convert_kernel(const double* __restrict__ src, int64_t rows, int64_t cols, int64_t ld_src,
                     const double* __restrict__ rowscale, const double* __restrict__ colscale, double alpha,
                     T* __restrict__ dst, int64_t ld_dst) {
    int64_t total = rows * cols, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        int64_t r = i / cols, c = i - r * cols;
        double v = src[r * ld_src + c] * alpha;
        if (rowscale) v *= rowscale[r];
        if (colscale) v *= colscale[c];
        dst[r * ld_dst + c] = (T)v;
    }
}

// dst[j, c] = src[c*ld_src + j] * rowscale[j] * alpha   (j < n rows of dst, c < cols)
template <class T>
__global__ void __launch_bounds__(256)
scaled_transpose_kernel(const double* __restrict__ src, int64_t n, int64_t cols, int64_t ld_src,
                        const double* __restrict__ rowscale, double alpha, T* __restrict__ dst) {
    int64_t total = n * cols, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        int64_t j = i / cols, c = i - j * cols;
        dst[i] = (T)(src[c * ld_src + j] * (rowscale ? rowscale[j] : 1.0) * alpha);
    }
}

template <class TA, class TB>
__global__ void __launch_bounds__(256) dot_kernel(const TA* __restrict__ a, const TB* __restrict__ b, int64_t n,
                                                   double* __restrict__ out) {
    __shared__ double scratch[32];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) s = fma((double)a[i], (double)b[i], s);
    s = block_sum(s, scratch);
    if (threadIdx.x == 0) out[0] = s;
}

static inline int ew_grid(const ndmps_ctx* ctx, int64_t total) {
    int64_t want = (total + 255) / 256, cap = (int64_t)ctx->sm_count * 8;
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

static int scale_convert(ndmps_ctx* ctx, const double* src, int64_t rows, int64_t cols, int64_t ld_src,
                         const double* rowscale, const double* colscale, double alpha, void* dst, int dtype, int64_t ld_dst) {
    if (rows * cols == 0) return NDMPS_OK;
    int g = ew_grid(ctx, rows * cols);
    if (dtype == NDMPS_F32)
        scale_convert_kernel<float><<<g, 256, 0, ctx->stream>>>(src, rows, cols, ld_src, rowscale, colscale, alpha, (float*)dst, ld_dst);
    else
        scale_convert_kernel<double><<<g, 256, 0, ctx->stream>>>(src, rows, cols, ld_src, rowscale, colscale, alpha, (double*)dst, ld_dst);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

static int scaled_transpose(ndmps_ctx* ctx, const double* src, int64_t n, int64_t cols, int64_t ld_src,
                            const double* rowscale, double alpha, void* dst, int dtype) {
    if (n * cols == 0) return NDMPS_OK;
    int g = ew_grid(ctx, n * cols);
    if (dtype == NDMPS_F32)
        scaled_transpose_kernel<float><<<g, 256, 0, ctx->stream>>>(src, n, cols, ld_src, rowscale, alpha, (float*)dst);
    else
        scaled_transpose_kernel<double><<<g, 256, 0, ctx->stream>>>(src, n, cols, ld_src, rowscale, alpha, (double*)dst);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

static int col_scale(ndmps_ctx* ctx, const double* evals, int64_t n, int mode, double factor, double floor_rel, double* out) {
    col_scale_kernel<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(evals, n, mode, factor, floor_rel, out);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

// ---------------------------------------------------------------------------------
// singular-value trimming on the host (quimb.tensor.decomp semantics, Appendix A.1/A.2)
// ---------------------------------------------------------------------------------
static int64_t n_keep(const double* s, int64_t n, double cutoff, int mode, int64_t max_bond) {
    int64_t keep = n;
    if (cutoff > 0.0) {
        if (mode == NDMPS_CUT_ABS) {
            keep = 0;
            for (int64_t i = 0; i < n; i++) keep += s[i] > cutoff;
        } else if (mode == NDMPS_CUT_REL) {
            keep = 0;
            for (int64_t i = 0; i < n; i++) keep += s[i] > cutoff * s[0];
        } else {
            int pw = (mode == NDMPS_CUT_SUM2 || mode == NDMPS_CUT_RSUM2) ? 2 : 1;
            bool rel = (mode == NDMPS_CUT_RSUM2 || mode == NDMPS_CUT_RSUM1);
            double target = cutoff;
            if (rel) {
                double tot = 0.0;
                for (int64_t i = 0; i < n; i++) tot += pw == 2 ? s[i] * s[i] : s[i];
                target *= tot;
            }
            double run = 0.0;
            keep = n;
            for (int64_t i = n - 1; i >= 0; i--) {
                run += pw == 2 ? s[i] * s[i] : s[i];
                if (run > target) break;
                keep--;
            }
        }
        if (keep < 1) keep = 1;
    }
    if (max_bond > 0 && keep > max_bond) keep = max_bond;
    return keep;
}

static double renorm_factor(const double* s, int64_t n, int64_t keep, int power) {
    if (keep >= n || power <= 0) return 1.0;
    double k = 0.0, l = 0.0;
    for (int64_t i = 0; i < n; i++) {
        double v = power == 2 ? s[i] * s[i] : (power == 1 ? s[i] : pow(s[i], power));
        if (i < keep) k += v; else l += v;
    }
    if (!(k > 0.0)) return 1.0;
    return pow((k + l) / k, 1.0 / power);
}

// The tcgen05 Gram decides ON THE DEVICE whether its digits are exact enough (tc_gemm.cu); the projection needs that
// answer on the host to pick its kernel.  It rides along with the eigenvalue readback every sweep step does anyway:
// the 4-byte flag is copied into an unused slot of the pinned scratch before the same synchronisation.
static int fetch_exact_flag(ndmps_ctx* ctx, size_t slot) {
    auto& dg = ctx->tc_digits;
    if (dg.use_exact == nullptr || dg.gen != ctx->ws.generation || dg.exact_host >= 0) return NDMPS_OK;
    NDMPS_TRY(readback(ctx, ctx->pinned + slot, dg.use_exact, sizeof(int)));
    dg.exact_host = -2;                                  // in flight
    return NDMPS_OK;
}
static void note_exact_flag(ndmps_ctx* ctx, size_t slot) {
    auto& dg = ctx->tc_digits;
    if (dg.exact_host == -2) dg.exact_host = *reinterpret_cast<const int*>(ctx->pinned + slot) != 0 ? 1 : 0;
}

// copy n eigenvalues to the host, return sqrt(max(l, 0)) in sv (host vector)
static int fetch_svals(ndmps_ctx* ctx, const double* evals_dev, int64_t n, std::vector<double>& sv) {
    NDMPS_TRY(ensure_pinned(ctx, (size_t)n + 64));
    NDMPS_TRY(readback(ctx, ctx->pinned, evals_dev, (size_t)n * sizeof(double)));
    NDMPS_TRY(fetch_exact_flag(ctx, (size_t)n + 8));
    NDMPS_CUDA_TRY(stream_wait(ctx));
    note_exact_flag(ctx, (size_t)n + 8);
    sv.resize((size_t)n);
    for (int64_t i = 0; i < n; i++) sv[i] = ctx->pinned[i] > 0.0 ? sqrt(ctx->pinned[i]) : 0.0;
    return NDMPS_OK;
}

// ---------------------------------------------------------------------------------
// the sweep
// ---------------------------------------------------------------------------------
struct TrimOpts {
    double cutoff;
    int mode;
    int64_t max_bond;
    int renorm;
};

// Bond cap set and the matrix much larger than the cap: try the leading-eigenpair solver
// (eig_topk.cu).  It is used only when the host can PROVE from its output that the trimming rule
// (n_keep above) lands on the cap: the weight outside the k leading eigenvalues, trace(G) minus
// their sum, must exceed the cutoff target with a margin far above the rounding error of that
// difference, and lambda_k must be well above the absolute error floor of the tridiagonal
// reduction (~ n eps lambda_1).  Anything else: *capped = false and the caller runs the full
// solver, so ranks never depend on which solver ran.  U: mj x mj buffer, eigenvector t in column t.
static int capped_eigh(ndmps_ctx* ctx, const double* Gj, int64_t mj, int64_t nmax, const TrimOpts& opt, double* evals_dev,
                       double* U, std::vector<double>& sv, int64_t* n_out, double* f_out, bool* capped) {
    *capped = false;
    const int64_t k = opt.max_bond;
    if (!ctx->opt_eig_topk || k <= 0 || mj < 4 * k || mj < 96 || nmax <= k) return NDMPS_OK;
    const bool sum2 = opt.mode == NDMPS_CUT_SUM2 || opt.mode == NDMPS_CUT_RSUM2;
    if (opt.cutoff > 0.0 && !sum2) return NDMPS_OK;
    if (opt.renorm != 0 && opt.renorm != 2) return NDMPS_OK;
    double* out = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)k + 2, &out));
    bool done = false;
    { StageScope sc(ctx, ST_EIG); NDMPS_TRY(eigh_topk(ctx, Gj, mj, k, out, U, mj, &done)); }
    if (!done) return NDMPS_OK;
    NDMPS_TRY(ensure_pinned(ctx, (size_t)k + 64));
    NDMPS_TRY(readback(ctx, ctx->pinned, out, (size_t)(k + 2) * sizeof(double)));
    NDMPS_TRY(fetch_exact_flag(ctx, (size_t)k + 8));
    NDMPS_CUDA_TRY(stream_wait(ctx));
    note_exact_flag(ctx, (size_t)k + 8);
    const double* ev = ctx->pinned;
    const double trace = ev[k], rank_loss = ev[k + 1];
    double kept = 0.0;
    for (int64_t i = 0; i < k; i++) kept += ev[i];
    const double tail = trace - kept;
    const double target = opt.cutoff > 0.0 ? opt.cutoff * (opt.mode == NDMPS_CUT_RSUM2 ? trace : 1.0) : 0.0;
    bool ok = rank_loss == 0.0 && trace > 0.0 && ev[0] > 0.0 && ev[k - 1] > 1e-9 * ev[0];
    ok = ok && tail > 2.0 * target + 1e-11 * trace;
    for (int64_t i = 1; ok && i < k; i++) ok = ev[i] <= ev[i - 1];
    if (ctx->opt_verbose)
        fprintf(stderr, "[ndmps] capped eigh n = %lld, k = %lld: lambda_k / lambda_1 = %.3e, discarded weight %.3e of trace -> %s\n",
                (long long)mj, (long long)k, ev[0] > 0.0 ? ev[k - 1] / ev[0] : 0.0, trace > 0.0 ? tail / trace : 0.0,
                ok ? "cap binds" : "full solver");
    if (!ok) return NDMPS_OK;
    sv.assign((size_t)mj, 0.0);
    for (int64_t i = 0; i < k; i++) sv[(size_t)i] = sqrt(ev[i]);
    *n_out = k;
    *f_out = opt.renorm == 2 ? sqrt(trace / kept) : 1.0;
    // the kept eigenvalues also on the device, where the column-side branch scales by them
    NDMPS_TRY(copy_small(ctx, evals_dev, out, (size_t)k * sizeof(double)));
    *capped = true;
    return NDMPS_OK;
}

// Column-sharded sweep (SURVEY section 8e, row 2): this rank holds the slice of the dense site array
// with the last site index in its block, i.e. a column block of every unfolding.  The left factor
// of a step depends only on G = M M^T, a SUM over column blocks: local Gram, allreduce through the
// caller's hook (NCCL on the launching stream), then the identical small eigenproblem on every rank
// and a local projection.  The sweep stops being sharded (stop_site) once the remainder is small.
struct ShardCtl {
    int world = 1;
    ndmps_allreduce_fn allreduce = nullptr;
    void* user = nullptr;
    int64_t stop_bytes = 0;        // hand back once the GLOBAL remainder is at most this many bytes
    int sites_done = 0;            // out
    const void* remainder = nullptr;   // out: (r_prev x remaining_local), in the workspace
    int64_t remainder_rows = 1, remainder_cols = 0;
};

static int ttsvd(ndmps_ctx* ctx, const void* dense, int dtype, int L, const int64_t* dims, const TrimOpts& opt,
                 void* const* cores_out, const int64_t* core_cap, int64_t* ranks_out, double* svals_out,
                 int64_t svals_stride, ShardCtl* sh = nullptr) {
    const size_t esz = dtype_size(dtype);
    // cores stored in float32 need eigenvectors orthogonal to ~1e-8, not 1e-15: one sweep less
    const double eig_tol = dtype == NDMPS_F32 ? 1e-10 : 0.0;
    int64_t total = 1;
    for (int i = 0; i < L; i++) total *= dims[i];
    if (svals_out)
        for (int64_t i = 0; i < (int64_t)(L - 1) * svals_stride; i++) svals_out[i] = 0.0;
    if (L == 1) {
        NDMPS_REQUIRE(core_cap[0] >= total, "ttsvd: core 0 capacity too small");
        NDMPS_CUDA_TRY(cudaMemcpyAsync(cores_out[0], dense, (size_t)total * esz, cudaMemcpyDeviceToDevice, ctx->stream));
        return NDMPS_OK;
    }
    // float32 payload with a bond cap: the long Gram and projection passes run on tcgen05 (tc_gemm.cu); the rank
    // decisions of an UNCAPPED sweep sit at lambda / lambda_1 ~ 1e-10 and keep the exact FP64-pipe path
    struct TcScope { ndmps_ctx* c; ~TcScope() { c->tc_sweep = false; } } tc_scope{ctx};
    ctx->tc_sweep = ctx->opt_tc && dtype == NDMPS_F32 && opt.max_bond > 0;
    const void* M = dense;         // current remainder, (r_prev * remaining) elements
    int64_t r_prev = 1;
    int64_t remaining = total;     // elements of the remainder divided by r_prev
    std::vector<double> sv;
    int site = 0;
    while (site < L - 1) {
        // ---- choose the group of sites sharing one Gram pass ----
        int64_t D = r_prev * dims[site];
        int64_t C = remaining / dims[site];
        int k = 1;
        while (site + k < L - 1) {
            int64_t Dn = D * dims[site + k], Cn = C / dims[site + k];
            if (Dn <= MERGE_CAP && Dn <= Cn) { D = Dn; C = Cn; k++; } else break;
        }
        if (sh) {
            // sharded phase ends when the global remainder is small or the local block gets wider than long
            const int64_t glob_bytes = r_prev * remaining * (int64_t)sh->world * (int64_t)esz;
            if (glob_bytes <= sh->stop_bytes || D > C || site + k >= L - 1) {
                sh->sites_done = site;
                sh->remainder = M;
                sh->remainder_rows = r_prev;
                sh->remainder_cols = remaining;
                return NDMPS_OK;
            }
        }
        if (ctx->opt_verbose)
            fprintf(stderr, "[ndmps] sweep site %d: group of %d, unfolding %lld x %lld (%s Gram)%s\n", site, k,
                    (long long)D, (long long)C, D <= C ? "row" : "column", sh ? " [column shard]" : "");
        int64_t r_out = 0;
        void* T = nullptr;
        if (D <= C) {
            double* G = nullptr;
            NDMPS_TRY(ctx->ws.get<double>((size_t)(D * D), &G));
            { StageScope sc(ctx, ST_GRAM); NDMPS_TRY(gram(ctx, M, D, C, C, dtype, 0, G)); }
            if (sh && sh->world > 1) {
                const int rc_hook = sh->allreduce(sh->user, G, D * D, (void*)ctx->stream);
                if (rc_hook != 0) { set_error("ttsvd: the allreduce hook failed (%d)", rc_hook); return NDMPS_ERR_CUDA; }
            }
            double* P = nullptr;       // (pd x rc) accumulated isometry (times renorm factors); nullptr = identity
            int64_t pd = r_prev, rc = r_prev;
            for (int j = 0; j < k; j++) {
                const int64_t d = dims[site + j];
                const int64_t X = pd * d, rest = D / X, mj = rc * d;
                double* Gt = G;
                if (rest > 1) {
                    NDMPS_TRY(ctx->ws.get<double>((size_t)(X * X), &Gt));
                    partial_trace_kernel<<<ew_grid(ctx, X * X), 256, 0, ctx->stream>>>(G, D, X, rest, Gt);
                    NDMPS_LAUNCH_CHECK(ctx);
                }
                double* Gj = Gt;
                double* K = nullptr;
                if (P != nullptr) {
                    NDMPS_TRY(ctx->ws.get<double>((size_t)(X * mj), &K));
                    kron_identity_kernel<<<ew_grid(ctx, X * mj), 256, 0, ctx->stream>>>(P, pd, rc, d, K);
                    NDMPS_LAUNCH_CHECK(ctx);
                    double* tmp = nullptr;
                    NDMPS_TRY(ctx->ws.get<double>((size_t)(X * mj), &tmp));
                    NDMPS_TRY(gemm(ctx, X, mj, X, 1.0, Gt, NDMPS_F64, X, 1, K, NDMPS_F64, mj, 1, tmp, NDMPS_F64, mj));
                    NDMPS_TRY(ctx->ws.get<double>((size_t)(mj * mj), &Gj));
                    NDMPS_TRY(gemm(ctx, mj, mj, X, 1.0, K, NDMPS_F64, 1, mj, tmp, NDMPS_F64, mj, 1, Gj, NDMPS_F64, mj));
                }
                double *evals = nullptr, *U = nullptr;
                NDMPS_TRY(ctx->ws.get<double>((size_t)mj, &evals));
                NDMPS_TRY(ctx->ws.get<double>((size_t)(mj * mj), &U));
                // rank of this unfolding is at most min(rows, cols)
                int64_t cols_j = C * rest * (sh ? sh->world : 1);
                int64_t nmax = mj < cols_j ? mj : cols_j;
                int64_t n = 0;
                double f = 1.0;
                bool capped = false;
                NDMPS_TRY(capped_eigh(ctx, Gj, mj, nmax, opt, evals, U, sv, &n, &f, &capped));
                if (!capped) {
                    { StageScope sc(ctx, ST_EIG); NDMPS_TRY(eigh(ctx, Gj, mj, evals, U, eig_tol)); }
                    NDMPS_TRY(fetch_svals(ctx, evals, mj, sv));
                    n = n_keep(sv.data(), nmax, opt.cutoff, opt.mode, opt.max_bond);
                    f = renorm_factor(sv.data(), nmax, n, opt.renorm);
                }
                const int s_idx = site + j;
                ranks_out[s_idx] = n;
                if (svals_out)
                    for (int64_t t = 0; t < n && t < svals_stride; t++) svals_out[(int64_t)s_idx * svals_stride + t] = sv[t] * f;
                if (core_cap[s_idx] < mj * n) {
                    set_error("ttsvd: core %d needs %lld elements, capacity %lld", s_idx, (long long)(mj * n), (long long)core_cap[s_idx]);
                    return NDMPS_ERR_CAPACITY;
                }
                NDMPS_TRY(scale_convert(ctx, U, mj, n, mj, nullptr, nullptr, 1.0, cores_out[s_idx], dtype, n));
                // P_next = f * K * U[:, :n]   (X x n)
                double* Pn = nullptr;
                NDMPS_TRY(ctx->ws.get<double>((size_t)(X * n), &Pn));
                if (K == nullptr) NDMPS_TRY(scale_convert(ctx, U, X, n, mj, nullptr, nullptr, f, Pn, NDMPS_F64, n));
                else NDMPS_TRY(gemm(ctx, X, n, mj, f, K, NDMPS_F64, mj, 1, U, NDMPS_F64, mj, 1, Pn, NDMPS_F64, n));
                P = Pn;
                pd = X;
                rc = n;
            }
            // T = P^T M   (rc x C)
            r_out = rc;
            NDMPS_TRY(ctx->ws.alloc((size_t)(r_out * C) * esz, &T));
            {
                StageScope sc(ctx, ST_PROJECT);
                bool on_tc = false;
                if (ctx->tc_sweep && C >= 2048) {
                    // the digits the Gram of this step sliced, when it ran on the integer tensor cores (exact accumulation) ...
                    NDMPS_TRY(proj_tc_digits(ctx, M, D, C, C, P, r_out, T, dtype, C, &on_tc));
                    // ... else T^T = M^T P on bf16x3 planes: the unfolding is the MN-major operand, T leaves transposed
                    if (!on_tc) NDMPS_TRY(gemm_tc(ctx, C, r_out, D, 1.0, M, dtype, 1, C, P, NDMPS_F64, r_out, 1, T, dtype, C, true, &on_tc));
                }
                if (!on_tc) {
                    // P^T made explicit (r x D, tiny) so the big product reads both operands along their rows
                    double* Pt = nullptr;
                    NDMPS_TRY(ctx->ws.get<double>((size_t)(r_out * D), &Pt));
                    NDMPS_TRY(scaled_transpose(ctx, P, r_out, D, r_out, nullptr, 1.0, Pt, NDMPS_F64));
                    NDMPS_TRY(gemm(ctx, r_out, C, D, 1.0, Pt, NDMPS_F64, D, 1, M, dtype, C, 1, T, dtype, C));
                }
            }
        } else {
            // more rows than columns: Gram on the column side, G' = M^T M = V s^2 V^T
            double *G = nullptr, *evals = nullptr, *V = nullptr;
            NDMPS_TRY(ctx->ws.get<double>((size_t)(C * C), &G));
            { StageScope sc(ctx, ST_GRAM); NDMPS_TRY(gram(ctx, M, D, C, C, dtype, 1, G)); }
            NDMPS_TRY(ctx->ws.get<double>((size_t)C, &evals));
            NDMPS_TRY(ctx->ws.get<double>((size_t)(C * C), &V));
            int64_t n = 0;
            double f = 1.0;
            bool capped = false;
            NDMPS_CUDA_TRY(cudaMemsetAsync(evals, 0, (size_t)C * sizeof(double), ctx->stream));
            if (!sh) NDMPS_TRY(capped_eigh(ctx, G, C, C < D ? C : D, opt, evals, V, sv, &n, &f, &capped));
            if (!capped) {
                { StageScope sc(ctx, ST_EIG); NDMPS_TRY(eigh(ctx, G, C, evals, V, eig_tol)); }
                NDMPS_TRY(fetch_svals(ctx, evals, C, sv));
                n = n_keep(sv.data(), C, opt.cutoff, opt.mode, opt.max_bond);
                f = renorm_factor(sv.data(), C, n, opt.renorm);
            }
            ranks_out[site] = n;
            if (svals_out)
                for (int64_t t = 0; t < n && t < svals_stride; t++) svals_out[(int64_t)site * svals_stride + t] = sv[t] * f;
            if (core_cap[site] < D * n) {
                set_error("ttsvd: core %d needs %lld elements, capacity %lld", site, (long long)(D * n), (long long)core_cap[site]);
                return NDMPS_ERR_CAPACITY;
            }
            double *inv_s = nullptr, *s_f = nullptr, *MV = nullptr;
            NDMPS_TRY(ctx->ws.get<double>((size_t)C, &inv_s));
            NDMPS_TRY(ctx->ws.get<double>((size_t)C, &s_f));
            NDMPS_TRY(col_scale(ctx, evals, C, 1, 1.0, 1e-14, inv_s));
            NDMPS_TRY(col_scale(ctx, evals, C, 0, f, 0.0, s_f));
            // U = M V[:, :n] / s   (D x n)
            NDMPS_TRY(ctx->ws.get<double>((size_t)(D * n), &MV));
            NDMPS_TRY(gemm(ctx, D, n, C, 1.0, M, dtype, C, 1, V, NDMPS_F64, C, 1, MV, NDMPS_F64, n));
            NDMPS_TRY(scale_convert(ctx, MV, D, n, n, nullptr, inv_s, 1.0, cores_out[site], dtype, n));
            // T = f diag(s) V[:, :n]^T   (n x C)
            r_out = n;
            NDMPS_TRY(ctx->ws.alloc((size_t)(r_out * C) * esz, &T));
            NDMPS_TRY(scaled_transpose(ctx, V, n, C, C, s_f, 1.0, T, dtype));
        }
        M = T;
        r_prev = r_out;
        remaining = C;
        site += k;
    }
    if (sh) {   // not reached: the sharded phase always hands back before the last site
        set_error("ttsvd: sharded sweep ran to the last site");
        return NDMPS_ERR_INVALID;
    }
    // last core = final remainder (r_{L-2} x d_{L-1})
    int64_t last = r_prev * dims[L - 1];
    if (core_cap[L - 1] < last) {
        set_error("ttsvd: last core needs %lld elements, capacity %lld", (long long)last, (long long)core_cap[L - 1]);
        return NDMPS_ERR_CAPACITY;
    }
    NDMPS_TRY(copy_small(ctx, cores_out[L - 1], M, (size_t)last * esz));
    return NDMPS_OK;
}

// ---------------------------------------------------------------------------------
// pairwise bond truncation (tensor_compress_bond, Appendix A.2) without QR:
//   G1 = T1^T T1 = X L X^T,  S1 = L^(1/2) X^T  (so T1 = Q1 S1 with Q1 an isometry)
//   H  = S1 (T2 T2^T) S1^T = U' s^2 U'^T       (left Gram of S1 T2, same s as R.L)
//   Y  = S1^T U'[:, :n]
//   T2' = s^(-1/2) Y^T T2,   T1' = T1 (T2 T2^T) Y s^(-3/2)
// Only kept singular values are inverted; values below 1e-13 s_0 give zero rows/columns.
// ---------------------------------------------------------------------------------
static int compress_bond(ndmps_ctx* ctx, const void* t1, const void* t2, int dtype, int64_t a, int64_t r, int64_t b,
                         const TrimOpts& opt, void* t1_out, void* t2_out, int64_t* new_rank, double* svals_out) {
    double *G1 = nullptr, *l1 = nullptr, *X = nullptr, *S1 = nullptr, *G2 = nullptr, *tmp = nullptr, *H = nullptr;
    double *sig2 = nullptr, *Up = nullptr, *Y = nullptr, *Z = nullptr, *sc = nullptr, *root1 = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)(r * r), &G1));
    NDMPS_TRY(ctx->ws.get<double>((size_t)r, &l1));
    NDMPS_TRY(ctx->ws.get<double>((size_t)(r * r), &X));
    NDMPS_TRY(ctx->ws.get<double>((size_t)(r * r), &S1));
    NDMPS_TRY(ctx->ws.get<double>((size_t)(r * r), &G2));
    NDMPS_TRY(ctx->ws.get<double>((size_t)(r * r), &tmp));
    NDMPS_TRY(ctx->ws.get<double>((size_t)(r * r), &H));
    NDMPS_TRY(ctx->ws.get<double>((size_t)r, &sig2));
    NDMPS_TRY(ctx->ws.get<double>((size_t)(r * r), &Up));
    NDMPS_TRY(ctx->ws.get<double>((size_t)r, &sc));
    NDMPS_TRY(ctx->ws.get<double>((size_t)r, &root1));
    NDMPS_TRY(gram(ctx, t1, a, r, r, dtype, 1, G1));
    NDMPS_TRY(eigh(ctx, G1, r, l1, X));
    NDMPS_TRY(col_scale(ctx, l1, r, 0, 1.0, 0.0, root1));
    NDMPS_TRY(scaled_transpose(ctx, X, r, r, r, root1, 1.0, S1, NDMPS_F64));          // S1[i, :] = sqrt(l_i) X[:, i]
    NDMPS_TRY(gram(ctx, t2, r, b, b, dtype, 0, G2));
    NDMPS_TRY(gemm(ctx, r, r, r, 1.0, S1, NDMPS_F64, r, 1, G2, NDMPS_F64, r, 1, tmp, NDMPS_F64, r));
    NDMPS_TRY(gemm(ctx, r, r, r, 1.0, tmp, NDMPS_F64, r, 1, S1, NDMPS_F64, 1, r, H, NDMPS_F64, r));
    NDMPS_TRY(eigh(ctx, H, r, sig2, Up));
    std::vector<double> sv;
    NDMPS_TRY(fetch_svals(ctx, sig2, r, sv));
    int64_t nmax = r < a ? r : a;
    if (b < nmax) nmax = b;
    int64_t n = n_keep(sv.data(), nmax, opt.cutoff, opt.mode, opt.max_bond);
    double f = renorm_factor(sv.data(), nmax, n, opt.renorm);
    *new_rank = n;
    if (svals_out)
        for (int64_t t = 0; t < r; t++) svals_out[t] = t < n ? sv[t] * f : 0.0;
    const double rf = sqrt(f);
    // Y = S1^T U'[:, :n]   (r x n)
    NDMPS_TRY(ctx->ws.get<double>((size_t)(r * n), &Y));
    NDMPS_TRY(gemm(ctx, r, n, r, 1.0, S1, NDMPS_F64, 1, r, Up, NDMPS_F64, r, 1, Y, NDMPS_F64, n));
    // Z = G2 Y s^(-3/2) sqrt(f)   (r x n), computed before T2 is overwritten
    NDMPS_TRY(ctx->ws.get<double>((size_t)(r * n), &Z));
    NDMPS_TRY(gemm(ctx, r, n, r, 1.0, G2, NDMPS_F64, r, 1, Y, NDMPS_F64, n, 1, tmp, NDMPS_F64, n));
    NDMPS_TRY(col_scale(ctx, sig2, r, 3, rf, 1e-8, sc));
    NDMPS_TRY(scale_convert(ctx, tmp, r, n, n, nullptr, sc, 1.0, Z, NDMPS_F64, n));
    // T2' = s^(-1/2) sqrt(f) Y^T T2   (n x b)
    double* t2tmp = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)(n * b), &t2tmp));
    NDMPS_TRY(gemm(ctx, n, b, r, 1.0, Y, NDMPS_F64, 1, n, t2, dtype, b, 1, t2tmp, NDMPS_F64, b));
    // T1' = T1 Z   (a x n)
    void* t1tmp = nullptr;
    NDMPS_TRY(ctx->ws.alloc((size_t)(a * n) * dtype_size(dtype), &t1tmp));
    NDMPS_TRY(gemm(ctx, a, n, r, 1.0, t1, dtype, r, 1, Z, NDMPS_F64, n, 1, t1tmp, dtype, n));
    NDMPS_TRY(col_scale(ctx, sig2, r, 2, rf, 1e-8, sc));
    NDMPS_TRY(scale_convert(ctx, t2tmp, n, b, b, sc, nullptr, 1.0, t2_out, dtype, b));
    NDMPS_TRY(copy_small(ctx, t1_out, t1tmp, (size_t)(a * n) * dtype_size(dtype)));
    return NDMPS_OK;
}

// ---------------------------------------------------------------------------------
// MPS -> dense (cumulative left -> right, Appendix A.3)
// ---------------------------------------------------------------------------------
static int contract_dense(ndmps_ctx* ctx, const void* const* cores, int dtype, int L, const int64_t* dims,
                          const int64_t* ranks, void* dense_out) {
    // Meet in the middle: X = product of the cores left of a split site s (P_s x r), W = product of
    // the cores from s on (r x Q_s), dense = X W in ONE large product that writes every voxel once.
    // Left and right chains are small; total flops ~ 2 N r instead of sum_k 2 P_k r d r.
    const size_t esz = dtype_size(dtype);
    if (L == 1) {
        NDMPS_CUDA_TRY(cudaMemcpyAsync(dense_out, cores[0], (size_t)dims[0] * esz, cudaMemcpyDeviceToDevice, ctx->stream));
        return NDMPS_OK;
    }
    StageScope sc(ctx, ST_CONTRACT);
    // split site: first s with P_s = prod_{k<s} d_k >= sqrt(N) (balanced), 1 <= s <= L-1
    double logn = 0.0;
    for (int k = 0; k < L; k++) logn += log((double)dims[k]);
    int s = 1;
    {
        double acc = log((double)dims[0]);
        while (s < L - 1 && acc < 0.5 * logn) { acc += log((double)dims[s]); s++; }
    }
    // left chain: X (rows x ranks[s-1])
    const void* X = cores[0];
    int64_t rows = dims[0];
    for (int k = 1; k < s; k++) {
        int64_t rin = ranks[k - 1], rout = ranks[k], ncols = dims[k] * rout;
        void* out = nullptr;
        NDMPS_TRY(ctx->ws.alloc((size_t)(rows * ncols) * esz, &out));
        NDMPS_TRY(gemm(ctx, rows, ncols, rin, 1.0, X, dtype, rin, 1, cores[k], dtype, ncols, 1, out, dtype, ncols));
        X = out;
        rows *= dims[k];
    }
    // right chain: W (ranks[s-1] x cols), built from the last core backwards
    const void* W = cores[L - 1];                 // (r_{L-2} x d_{L-1})
    int64_t cols = dims[L - 1];
    for (int k = L - 2; k >= s; k--) {
        int64_t rl = ranks[k - 1], rr = ranks[k];  // core k: (rl, d_k, rr) = (rl*d_k) x rr
        void* out = nullptr;
        NDMPS_TRY(ctx->ws.alloc((size_t)(rl * dims[k] * cols) * esz, &out));
        NDMPS_TRY(gemm(ctx, rl * dims[k], cols, rr, 1.0, cores[k], dtype, rr, 1, W, dtype, cols, 1, out, dtype, cols));
        W = out;
        cols *= dims[k];
    }
    const int64_t r = ranks[s - 1];
    if (ctx->opt_tc && dtype == NDMPS_F32 && rows * cols >= (int64_t(1) << 20)) {   // float32 payload: the one big product on tcgen05
        bool on_tc = false;
        NDMPS_TRY(gemm_tc(ctx, rows, cols, r, 1.0, X, dtype, r, 1, W, dtype, cols, 1, dense_out, dtype, cols, false, &on_tc));
        if (on_tc) return NDMPS_OK;
    }
    return gemm(ctx, rows, cols, r, 1.0, X, dtype, r, 1, W, dtype, cols, 1, dense_out, dtype, cols);
}

// ---------------------------------------------------------------------------------
// <a|b> by transfer matrices (float64)
// ---------------------------------------------------------------------------------
static int overlap(ndmps_ctx* ctx, const void* const* ca, const int64_t* ra, int da, const void* const* cb,
                   const int64_t* rb, int db, int L, const int64_t* dims, double* out_dev) {
    auto dot = [&](const void* x, int dx, const void* y, int dy, int64_t n) -> int {
        if (dx == NDMPS_F32 && dy == NDMPS_F32) dot_kernel<float, float><<<1, 256, 0, ctx->stream>>>((const float*)x, (const float*)y, n, out_dev);
        else if (dx == NDMPS_F32) dot_kernel<float, double><<<1, 256, 0, ctx->stream>>>((const float*)x, (const double*)y, n, out_dev);
        else if (dy == NDMPS_F32) dot_kernel<double, float><<<1, 256, 0, ctx->stream>>>((const double*)x, (const float*)y, n, out_dev);
        else dot_kernel<double, double><<<1, 256, 0, ctx->stream>>>((const double*)x, (const double*)y, n, out_dev);
        NDMPS_LAUNCH_CHECK(ctx);
        return NDMPS_OK;
    };
    if (L == 1) return dot(ca[0], da, cb[0], db, dims[0]);
    // E0 = A0^T B0   (ra0 x rb0)
    double* E = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)(ra[0] * rb[0]), &E));
    NDMPS_TRY(gemm(ctx, ra[0], rb[0], dims[0], 1.0, ca[0], da, 1, ra[0], cb[0], db, rb[0], 1, E, NDMPS_F64, rb[0]));
    for (int k = 1; k < L - 1; k++) {
        int64_t al = ra[k - 1], ar = ra[k], bl = rb[k - 1], br = rb[k], d = dims[k];
        double *T1 = nullptr, *E2 = nullptr;
        NDMPS_TRY(ctx->ws.get<double>((size_t)(al * d * br), &T1));
        // T1 = E (al x bl) . B_k (bl x d*br)
        NDMPS_TRY(gemm(ctx, al, d * br, bl, 1.0, E, NDMPS_F64, bl, 1, cb[k], db, d * br, 1, T1, NDMPS_F64, d * br));
        // E' = A_k^T (ar x al*d) . T1 (al*d x br)
        NDMPS_TRY(ctx->ws.get<double>((size_t)(ar * br), &E2));
        NDMPS_TRY(gemm(ctx, ar, br, al * d, 1.0, ca[k], da, 1, ar, T1, NDMPS_F64, br, 1, E2, NDMPS_F64, br));
        E = E2;
    }
    // result = sum (E . B_last) o A_last
    int64_t al = ra[L - 2], bl = rb[L - 2], d = dims[L - 1];
    double* F = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)(al * d), &F));
    NDMPS_TRY(gemm(ctx, al, d, bl, 1.0, E, NDMPS_F64, bl, 1, cb[L - 1], db, d, 1, F, NDMPS_F64, d));
    return dot(ca[L - 1], da, F, NDMPS_F64, al * d);
}

// out[r][c][g][t] = gathered[g][r][c][t]: the column blocks of `world` ranks put back in site order
template <class T>
__global__ void __launch_bounds__(256)
interleave_shards_kernel(const T* __restrict__ gathered, int world, int64_t rows, int64_t cmid, int64_t dl, T* __restrict__ out) {
    const int64_t total = (int64_t)world * rows * cmid * dl;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (int64_t)gridDim.x * 256) {
        const int64_t t = i % dl, g = (i / dl) % world, c = (i / (dl * world)) % cmid, r = i / (dl * world * cmid);
        out[i] = gathered[((g * rows + r) * cmid + c) * dl + t];
    }
}

}  // namespace ndmps

using namespace ndmps;

extern "C" {

int ndmps_ttsvd(ndmps_ctx_t* ctx, const void* dense, int dtype, int levels, const int64_t* dims,
                double cutoff, int cutoff_mode, int64_t max_bond, int renorm,
                void* const* cores_out, const int64_t* core_cap, int64_t* ranks_out_host,
                double* svals_out_host, int64_t svals_stride) {
    NDMPS_REQUIRE(ctx && dense && dims && cores_out && core_cap, "ndmps_ttsvd: NULL argument");
    NDMPS_REQUIRE(levels >= 1 && dtype_ok(dtype), "ndmps_ttsvd: bad levels or dtype");
    NDMPS_REQUIRE(levels == 1 || ranks_out_host, "ndmps_ttsvd: ranks_out_host is NULL");
    NDMPS_REQUIRE(cutoff_mode >= NDMPS_CUT_ABS && cutoff_mode <= NDMPS_CUT_RSUM1, "ndmps_ttsvd: bad cutoff_mode %d", cutoff_mode);
    for (int i = 0; i < levels; i++) NDMPS_REQUIRE(dims[i] >= 1 && cores_out[i], "ndmps_ttsvd: bad dims or core pointer at %d", i);
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    TrimOpts opt{cutoff, cutoff_mode, max_bond, renorm};
    NDMPS_TRY(ttsvd(ctx, dense, dtype, levels, dims, opt, cores_out, core_cap, ranks_out_host, svals_out_host, svals_stride));
    NDMPS_CUDA_TRY(stream_wait(ctx));
    return NDMPS_OK;
}

int ndmps_ttsvd_sharded(ndmps_ctx_t* ctx, const void* dense_local, int dtype, int levels, const int64_t* dims_local,
                        int world, ndmps_allreduce_fn allreduce, void* user, int64_t stop_bytes,
                        double cutoff, int cutoff_mode, int64_t max_bond, int renorm,
                        void* const* cores_out, const int64_t* core_cap, int64_t* ranks_out_host,
                        double* svals_out_host, int64_t svals_stride,
                        int* sites_done_host, void* remainder_out, int64_t remainder_cap, int64_t* remainder_shape_host) {
    NDMPS_REQUIRE(ctx && dense_local && dims_local && cores_out && core_cap && ranks_out_host, "ndmps_ttsvd_sharded: NULL argument");
    NDMPS_REQUIRE(sites_done_host && remainder_out && remainder_shape_host, "ndmps_ttsvd_sharded: NULL output");
    NDMPS_REQUIRE(levels >= 2 && dtype_ok(dtype), "ndmps_ttsvd_sharded: bad levels or dtype");
    NDMPS_REQUIRE(world >= 1 && (world == 1 || allreduce), "ndmps_ttsvd_sharded: world %d needs an allreduce hook", world);
    NDMPS_REQUIRE(cutoff_mode >= NDMPS_CUT_ABS && cutoff_mode <= NDMPS_CUT_RSUM1, "ndmps_ttsvd_sharded: bad cutoff_mode %d", cutoff_mode);
    for (int i = 0; i < levels; i++) NDMPS_REQUIRE(dims_local[i] >= 1, "ndmps_ttsvd_sharded: bad dims at %d", i);
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    TrimOpts opt{cutoff, cutoff_mode, max_bond, renorm};
    ShardCtl sh;
    sh.world = world;
    sh.allreduce = allreduce;
    sh.user = user;
    sh.stop_bytes = stop_bytes;
    NDMPS_TRY(ttsvd(ctx, dense_local, dtype, levels, dims_local, opt, cores_out, core_cap, ranks_out_host, svals_out_host,
                    svals_stride, &sh));
    const int64_t count = sh.remainder_rows * sh.remainder_cols;
    NDMPS_REQUIRE(count <= remainder_cap, "ndmps_ttsvd_sharded: remainder needs %lld elements, capacity %lld", (long long)count,
                  (long long)remainder_cap);
    NDMPS_CUDA_TRY(cudaMemcpyAsync(remainder_out, sh.remainder, (size_t)count * dtype_size(dtype), cudaMemcpyDeviceToDevice, ctx->stream));
    NDMPS_CUDA_TRY(stream_wait(ctx));
    *sites_done_host = sh.sites_done;
    remainder_shape_host[0] = sh.remainder_rows;
    remainder_shape_host[1] = sh.remainder_cols;
    return NDMPS_OK;
}

int ndmps_interleave_shards(ndmps_ctx_t* ctx, const void* gathered, int dtype, int world, int64_t rows, int64_t cmid, int64_t dl,
                            void* out) {
    NDMPS_REQUIRE(ctx && gathered && out && gathered != out, "ndmps_interleave_shards: NULL or aliased argument");
    NDMPS_REQUIRE(dtype_ok(dtype) && world >= 1 && rows >= 1 && cmid >= 1 && dl >= 1, "ndmps_interleave_shards: bad shape or dtype");
    const int64_t total = (int64_t)world * rows * cmid * dl;
    const int g = ew_grid(ctx, total);
    if (dtype == NDMPS_F32)
        interleave_shards_kernel<float><<<g, 256, 0, ctx->stream>>>((const float*)gathered, world, rows, cmid, dl, (float*)out);
    else
        interleave_shards_kernel<double><<<g, 256, 0, ctx->stream>>>((const double*)gathered, world, rows, cmid, dl, (double*)out);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

int ndmps_compress_bond(ndmps_ctx_t* ctx, const void* t1, const void* t2, int dtype, int64_t a, int64_t r, int64_t b,
                        double cutoff, int cutoff_mode, int64_t max_bond, int renorm,
                        void* t1_out, void* t2_out, int64_t* new_rank_host, double* svals_out_host) {
    NDMPS_REQUIRE(ctx && t1 && t2 && t1_out && t2_out && new_rank_host, "ndmps_compress_bond: NULL argument");
    NDMPS_REQUIRE(dtype_ok(dtype) && a >= 1 && r >= 1 && b >= 1, "ndmps_compress_bond: bad shape or dtype");
    NDMPS_REQUIRE(cutoff_mode >= NDMPS_CUT_ABS && cutoff_mode <= NDMPS_CUT_RSUM1, "ndmps_compress_bond: bad cutoff_mode %d", cutoff_mode);
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    TrimOpts opt{cutoff, cutoff_mode, max_bond, renorm};
    NDMPS_TRY(compress_bond(ctx, t1, t2, dtype, a, r, b, opt, t1_out, t2_out, new_rank_host, svals_out_host));
    NDMPS_CUDA_TRY(stream_wait(ctx));
    return NDMPS_OK;
}

int ndmps_contract_dense(ndmps_ctx_t* ctx, const void* const* cores, int dtype, int levels, const int64_t* dims,
                         const int64_t* ranks, void* dense_out) {
    NDMPS_REQUIRE(ctx && cores && dims && dense_out, "ndmps_contract_dense: NULL argument");
    NDMPS_REQUIRE(levels >= 1 && dtype_ok(dtype), "ndmps_contract_dense: bad levels or dtype");
    NDMPS_REQUIRE(levels == 1 || ranks, "ndmps_contract_dense: ranks is NULL");
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    return contract_dense(ctx, cores, dtype, levels, dims, ranks, dense_out);
}

int ndmps_overlap(ndmps_ctx_t* ctx, const void* const* cores_a, const int64_t* ranks_a, int dtype_a,
                  const void* const* cores_b, const int64_t* ranks_b, int dtype_b, int levels, const int64_t* dims,
                  double* out_host) {
    NDMPS_REQUIRE(ctx && cores_a && cores_b && dims && out_host, "ndmps_overlap: NULL argument");
    NDMPS_REQUIRE(levels >= 1 && dtype_ok(dtype_a) && dtype_ok(dtype_b), "ndmps_overlap: bad levels or dtype");
    NDMPS_REQUIRE(levels == 1 || (ranks_a && ranks_b), "ndmps_overlap: ranks is NULL");
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    NDMPS_TRY(ensure_pinned(ctx, 2));
    double* out_dev = nullptr;
    NDMPS_TRY(ctx->ws.get<double>(2, &out_dev));
    NDMPS_TRY(overlap(ctx, cores_a, ranks_a, dtype_a, cores_b, ranks_b, dtype_b, levels, dims, out_dev));
    NDMPS_TRY(readback(ctx, ctx->pinned, out_dev, sizeof(double)));
    NDMPS_CUDA_TRY(stream_wait(ctx));
    out_host[0] = ctx->pinned[0];
    return NDMPS_OK;
}

int ndmps_roundtrip_host(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* src_host, void* dst_host, int dtype,
                         double cutoff, int cutoff_mode, int64_t max_bond, int renorm, int64_t* ranks_out_host,
                         double* norm_out_host, double* boundaries_out_host) {
    NDMPS_REQUIRE(ctx && plan && src_host && dst_host, "ndmps_roundtrip_host: NULL argument");
    NDMPS_REQUIRE(dtype_ok(dtype), "ndmps_roundtrip_host: bad dtype");
    NDMPS_REQUIRE(cutoff_mode >= NDMPS_CUT_ABS && cutoff_mode <= NDMPS_CUT_RSUM1, "ndmps_roundtrip_host: bad cutoff_mode %d", cutoff_mode);
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    const int L = plan->levels;
    const int64_t N = plan->total;
    const size_t esz = dtype_size(dtype);
    void *vol = nullptr, *dense = nullptr;
    NDMPS_TRY(ctx->ws.alloc((size_t)N * esz, &vol));
    NDMPS_TRY(ctx->ws.alloc((size_t)N * esz, &dense));
    NDMPS_CUDA_TRY(cudaMemcpyAsync(vol, src_host, (size_t)N * esz, cudaMemcpyDefault, ctx->stream));
    NDMPS_TRY(permute(ctx, plan, false, vol, dense, dtype, 1.0));
    // core capacities from the bond bounds min(max_bond, prod left, prod right)
    std::vector<int64_t> bound((size_t)(L > 1 ? L - 1 : 0)), cap((size_t)L), ranks((size_t)(L > 1 ? L - 1 : 1));
    std::vector<void*> cores((size_t)L);
    {
        double left = 1.0;
        for (int i = 0; i < L - 1; i++) {
            left *= (double)plan->site_dims[i];
            double right = 1.0;
            for (int j = i + 1; j < L; j++) right *= (double)plan->site_dims[j];
            double bd = left < right ? left : right;
            if (max_bond > 0 && (double)max_bond < bd) bd = (double)max_bond;
            bound[(size_t)i] = (int64_t)bd;
        }
        for (int i = 0; i < L; i++) {
            int64_t l = i == 0 ? 1 : bound[(size_t)i - 1], r = i == L - 1 ? 1 : bound[(size_t)i];
            // a bond can never exceed (left bond * d): tighten so lossless capacities stay finite
            cap[(size_t)i] = l * plan->site_dims[i] * r;
            NDMPS_TRY(ctx->ws.alloc((size_t)cap[(size_t)i] * esz, &cores[(size_t)i]));
        }
    }
    TrimOpts opt{cutoff, cutoff_mode, max_bond, renorm};
    NDMPS_TRY(ttsvd(ctx, dense, dtype, L, plan->site_dims, opt, cores.data(), cap.data(), ranks.data(), nullptr, 0));
    if (ranks_out_host)
        for (int i = 0; i < L - 1; i++) ranks_out_host[i] = ranks[(size_t)i];
    // boundary list and norm of the MPS, as from_tensor keeps them (core/ndmps.py:75-76, 80-86)
    double* extras = nullptr;
    NDMPS_TRY(ctx->ws.get<double>(2 * (size_t)L + 2, &extras));
    {
        StageScope sc(ctx, ST_GLUE);
        for (int i = 0; i < L; i++) {
            const int64_t l = i == 0 ? 1 : ranks[(size_t)i - 1], r = i == L - 1 ? 1 : ranks[(size_t)i];
            NDMPS_TRY(minmax_device(ctx, cores[(size_t)i], l * plan->site_dims[i] * r, dtype, extras + 2 * i));
        }
        NDMPS_TRY(overlap(ctx, (const void* const*)cores.data(), ranks.data(), dtype, (const void* const*)cores.data(), ranks.data(),
                          dtype, L, plan->site_dims, extras + 2 * L));
    }
    NDMPS_TRY(contract_dense(ctx, (const void* const*)cores.data(), dtype, L, plan->site_dims, ranks.data(), dense));
    NDMPS_TRY(permute(ctx, plan, true, dense, vol, dtype, 1.0));
    NDMPS_CUDA_TRY(cudaMemcpyAsync(dst_host, vol, (size_t)N * esz, cudaMemcpyDefault, ctx->stream));
    NDMPS_TRY(ensure_pinned(ctx, 2 * (size_t)L + 2));
    NDMPS_TRY(readback(ctx, ctx->pinned, extras, (2 * (size_t)L + 2) * sizeof(double)));
    NDMPS_CUDA_TRY(stream_wait(ctx));
    if (boundaries_out_host)
        for (int i = 0; i < 2 * L; i++) boundaries_out_host[i] = ctx->pinned[i];
    if (norm_out_host) *norm_out_host = ctx->pinned[2 * L] > 0.0 ? sqrt(ctx->pinned[2 * L]) : 0.0;
    return NDMPS_OK;
}

}  // extern "C"
