// K3: symmetric eigen-decomposition of bond-sized Gram matrices, float64,
// by parallel one-sided (Hestenes) Jacobi.
//
// Replaces the LAPACK gesdd call quimb makes under from_dense / tensor_compress_bond
// (core/ndmps.py:74,106) for the small matrix of each sweep step: with
// G = M M^T symmetric positive semi-definite, orthogonalising the columns of G by
// plane rotations gives G V = W with W's columns mutually orthogonal, so
// lambda_j = |w_j| and u_j = w_j / |w_j|.  Everything is float64 (B200's FP64 pipe),
// because the sweep's rank decisions sit at lambda/lambda_max ~ 1e-10.
//
// Parallel scheme: the n columns are split into nb blocks of b columns.  A sweep is a
// round-robin tournament over blocks (nb-1 rounds); in a round every CTA owns one block
// pair in shared memory and one warp owns one column pair at a time.  Round 0 of a
// sweep runs the full tournament inside the 2b columns (this covers the within-block
// pairs); later rounds only rotate cross pairs.  The whole solve is ONE persistent
// cooperative launch: CTAs exchange column blocks through L2 (ld.cg / st.cg) and meet
// at a counter barrier after every round; convergence is a per-sweep flag.  Matrices
// with n <= 64 are solved whole by one CTA (eigh_small_kernel).
//
// Per rotation the latency chain is what matters (the FP64 work is tiny), so:
//   * the three reductions of a pair (|x|^2, |y|^2, x.y) run as interleaved butterflies;
//   * short columns (n <= 128) use 8 lanes per pair, four pairs per warp;
//   * in the cross rounds of a block pair the P column stays in registers and only the Q
//     columns stream through shared memory (the long-column case is smem-bandwidth bound);
//   * tangent / cosine come from MUFU rcp / rsqrt seeds plus Newton steps (full float64
//     accuracy) instead of the IEEE division / square-root instruction sequences;
// (de Rijk's dynamic column swaps were tried and dropped: in a parallel tournament they break
// the once-per-sweep pair coverage and the sweep count explodes.)
#include "common.cuh"

namespace ndmps {

// rotation threshold |x.y| <= tol |x||y| with tol = sqrt(n) * 2 eps (LAPACK dgesvj uses sqrt(n) eps)
static inline double jacobi_tol(int n) { return sqrt((double)n) * 4.4408920985006262e-16; }

constexpr int JACOBI_MAX_SWEEPS = 40;

__device__ __forceinline__ double rsqrt_refined(double x) {   // x in the normal range
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x * r, r, 1.0);
    r = fma(0.5 * r, e, r);
    e = fma(-x * r, r, 1.0);
    r = fma(0.5 * r, e, r);
    return r;
}

__device__ __forceinline__ double rcp_approx(double x) {      // ~20 bits, full exponent range
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    return r;
}

__device__ __forceinline__ double rcp_refined(double x) {     // full float64 accuracy
    double r = rcp_approx(x);
    r = fma(r, fma(-x, r, 1.0), r);
    r = fma(r, fma(-x, r, 1.0), r);
    return r;
}

// cos / sin / tan of the Jacobi rotation that orthogonalises two columns with squared
// norms alpha, beta and inner product gamma (gamma != 0): t is the smaller root of
// t^2 + 2 zeta t - 1 = 0.  MUFU seeds + Newton steps instead of the IEEE div / sqrt sequences;
// all results are float64-accurate (the cached-norm identities below rely on an exact t).
__device__ __forceinline__ void rotation(double alpha, double beta, double gamma, double& c, double& s, double& t) {
    const double zeta = (beta - alpha) * rcp_refined(2.0 * gamma);
    const double az = fabs(zeta);
    if (az > 1e150) {
        t = 0.5 * rcp_refined(zeta);
    } else {
        const double w = fma(az, az, 1.0);
        const double sq = w * rsqrt_refined(w);
        t = copysign(rcp_refined(az + sq), zeta);
    }
    c = rsqrt_refined(fma(t, t, 1.0));
    s = c * t;
}

// The same rotation from cos 2theta = |beta - alpha| / h, h = hypot(beta - alpha, 2 gamma):
// c = sqrt((1 + cos 2theta) / 2), s = sign(beta - alpha) 2 gamma / (2 h c).  Two reciprocal square roots in the
// dependent chain instead of two reciprocals and two square roots; no cancellation anywhere (c^2 + s^2 = 1 to rounding).
__device__ __forceinline__ void rotation_cs(double alpha, double beta, double gamma, double& c, double& s) {
    const double d = beta - alpha, g2 = 2.0 * gamma;
    const double r = rsqrt_refined(fma(d, d, g2 * g2));       // 1 / h
    const double c2 = fma(0.5 * fabs(d), r, 0.5);
    const double rc = rsqrt_refined(c2);
    c = c2 * rc;
    s = copysign(0.5, d) * g2 * r * rc;
}

// Orthogonalise columns x, y (length n, shared memory) with a group of LP lanes (LP = 32: one
// pair per warp; LP = 8: four pairs per warp, for short columns where the butterfly
// reductions and the redundant per-lane rotation math would otherwise dominate).
// li: lane index inside the group.  Every lane of the warp must call this (the shuffles
// use the full mask); `valid` masks out groups without a pair.  Squared norms are
// recomputed at every visit: three interleaved butterflies.
template <int NR, int LP>
__device__ __forceinline__ bool rotate_group(double* x, double* y, int n, int li, bool valid, double tol2, double floor2,
                                             float& relmax) {
    double xr[NR], yr[NR];
    double alpha = 0.0, beta = 0.0, gamma = 0.0;
#pragma unroll
    for (int t = 0; t < NR; t++) {
        const int i = li + LP * t;
        const bool in = valid && i < n;
        xr[t] = in ? x[i] : 0.0;
        yr[t] = in ? y[i] : 0.0;
        alpha = fma(xr[t], xr[t], alpha);
        beta = fma(yr[t], yr[t], beta);
        gamma = fma(xr[t], yr[t], gamma);
    }
#pragma unroll
    for (int o = LP / 2; o > 0; o >>= 1) {
        alpha += __shfl_xor_sync(0xffffffffu, alpha, o);
        beta += __shfl_xor_sync(0xffffffffu, beta, o);
        gamma += __shfl_xor_sync(0xffffffffu, gamma, o);
    }
    // columns whose norm is below n*eps*|G| are numerically null: rotating them only churns
    // round-off and would keep the sweep from ever reporting convergence
    if (!valid || !(alpha > floor2) || !(beta > floor2)) return false;
    if (!(gamma * gamma > tol2 * alpha * beta)) return false;
    relmax = fmaxf(relmax, (float)(gamma * gamma * rcp_approx(alpha * beta)));
    double c, s;
    rotation_cs(alpha, beta, gamma, c, s);
#pragma unroll
    for (int tt = 0; tt < NR; tt++) {
        const int i = li + LP * tt;
        if (i < n) {
            x[i] = c * xr[tt] - s * yr[tt];
            y[i] = s * xr[tt] + c * yr[tt];
        }
    }
    return true;
}

// same for columns of any length (n > 512): one pair per warp, two passes over shared memory
__device__ __forceinline__ bool rotate_generic(double* x, double* y, int n, int lane, bool valid, double tol2, double floor2,
                                               float& relmax) {
    double alpha = 0.0, beta = 0.0, gamma = 0.0;
    if (valid) {
        for (int i = lane; i < n; i += 32) {
            double a = x[i], b = y[i];
            alpha = fma(a, a, alpha);
            beta = fma(b, b, beta);
            gamma = fma(a, b, gamma);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        alpha += __shfl_xor_sync(0xffffffffu, alpha, o);
        beta += __shfl_xor_sync(0xffffffffu, beta, o);
        gamma += __shfl_xor_sync(0xffffffffu, gamma, o);
    }
    if (!valid || !(alpha > floor2) || !(beta > floor2)) return false;
    if (!(gamma * gamma > tol2 * alpha * beta)) return false;
    relmax = fmaxf(relmax, (float)(gamma * gamma * rcp_approx(alpha * beta)));
    double c, s, t;
    rotation(alpha, beta, gamma, c, s, t);
    for (int i = lane; i < n; i += 32) {
        double xv = x[i], yv = y[i];
        x[i] = c * xv - s * yv;
        y[i] = s * xv + c * yv;
    }
    return true;
}

template <int NR>
__device__ __forceinline__ bool rotate_warp(double* x, double* y, int n, int lane, bool valid, double tol2, double floor2,
                                            float& relmax) {
    if constexpr (NR > 0) return rotate_group<NR, 32>(x, y, n, lane, valid, tol2, floor2, relmax);
    else return rotate_generic(x, y, n, lane, valid, tol2, floor2, relmax);
}

// The b cross rounds of one block pair with the P column held in REGISTERS: warp w keeps
// column P_w for all b rounds and only the Q columns stream through shared memory, which
// halves the shared-memory traffic that bounds the long-column case.  Squared norms are
// cached for the duration of the block pair (<= b rotations per column) and updated by the
// exact identities a' = a - t g, b' = b + t g; they are recomputed from the data whenever a
// column collapses (catastrophic cancellation) and at every block load.
template <int NR>
__device__ __forceinline__ bool cross_rounds_stationary(double* S, double* norm2, int n, int b, int cntp, int cntq,
                                                        int warp, int lane, double tol2, double floor2, float& relmax) {
    double xr[NR];
    double* x = S + (size_t)warp * n;
    const bool have_x = warp < cntp;
#pragma unroll
    for (int t = 0; t < NR; t++) {
        const int i = lane + 32 * t;
        xr[t] = (have_x && i < n) ? x[i] : 0.0;
    }
    double alpha = have_x ? norm2[warp] : 0.0;
    bool any = false;
    for (int k = 0; k < b; k++) {
        int j = warp + k;
        j = j >= b ? j - b : j;
        const bool valid = have_x && j < cntq;
        double* y = S + (size_t)(b + j) * n;
        double yr[NR];
        double g4[4] = {0.0, 0.0, 0.0, 0.0};                 // four chains: the dot is latency-, not throughput-bound
#pragma unroll
        for (int t = 0; t < NR; t++) {
            const int i = lane + 32 * t;
            yr[t] = (valid && i < n) ? y[i] : 0.0;
            g4[t & 3] = fma(xr[t], yr[t], g4[t & 3]);
        }
        double gamma = warp_sum((g4[0] + g4[1]) + (g4[2] + g4[3]));
        const double beta = valid ? norm2[b + j] : 0.0;
        if (valid && alpha > floor2 && beta > floor2 && gamma * gamma > tol2 * alpha * beta) {
            relmax = fmaxf(relmax, (float)(gamma * gamma * rcp_approx(alpha * beta)));
            double c, s, t;
            rotation(alpha, beta, gamma, c, s, t);
            double ra = 0.0, rb = 0.0;
#pragma unroll
            for (int tt = 0; tt < NR; tt++) {
                const int i = lane + 32 * tt;
                const double xn = c * xr[tt] - s * yr[tt];
                const double yn = s * xr[tt] + c * yr[tt];
                xr[tt] = xn;
                if (i < n) y[i] = yn;
                yr[tt] = yn;
            }
            double na = alpha - t * gamma, nb = beta + t * gamma;
            if (na < 0.01 * alpha || nb < 0.01 * beta) {      // warp-uniform
#pragma unroll
                for (int tt = 0; tt < NR; tt++) {
                    ra = fma(xr[tt], xr[tt], ra);
                    rb = fma(yr[tt], yr[tt], rb);
                }
                na = warp_sum(ra);
                nb = warp_sum(rb);
            }
            alpha = na;
            if (lane == 0) norm2[b + j] = nb;
            any = true;
        }
        __syncthreads();
    }
    if (any) {
#pragma unroll
        for (int t = 0; t < NR; t++) {
            const int i = lane + 32 * t;
            if (i < n) x[i] = xr[t];
        }
    }
    return any;
}

// slot pair of a round-robin tournament over P (even) players, match `w` of round `lr`
__device__ __forceinline__ void tournament_pair(int P, int lr, int w, int& s1, int& s2) {
    int m = P - 1;
    if (w == 0) {
        s1 = m;
        s2 = lr;
    } else {
        s1 = lr + w;                 // lr, w < m: no integer division (it cost ~450 cycles per round of the n <= 64 solver)
        s1 = s1 >= m ? s1 - m : s1;
        s2 = lr - w;
        s2 = s2 < 0 ? s2 + m : s2;
    }
}

__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1u);
        while (*((volatile unsigned*)counter) < target) {
        }
        __threadfence();
    }
    __syncthreads();
}

// One CTA, one block pair (p, q) of one tournament round: load both column blocks from
// L2, rotate, store back.  S: 2*b*n doubles followed by 2*b cached squared norms.
template <int NR>
__device__ __forceinline__ bool process_block_pair(double* A, int n, int ncols, int b, int nb, int round, int cta,
                                                   double* S, double tol2, double floor2, float& relmax) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* norm2 = S + (size_t)2 * b * n;
    int p, q;
    tournament_pair(nb, round, cta, p, q);
    const int colp0 = p * b, colq0 = q * b;
    int cntp = ncols - colp0; cntp = cntp < 0 ? 0 : (cntp > b ? b : cntp);
    int cntq = ncols - colq0; cntq = cntq < 0 ? 0 : (cntq > b ? b : cntq);
    if constexpr (NR > 0) {
        // both columns of this warp are fetched with all loads in flight before anything is stored:
        // a load -> store loop would serialise 2*NR L2 round trips per global round
        double vp[NR], vq[NR];
        const bool hp = warp < cntp, hq = warp < cntq;
        const double* sp = A + (size_t)(colp0 + warp) * n;
        const double* sq = A + (size_t)(colq0 + warp) * n;
#pragma unroll
        for (int t = 0; t < NR; t++) {
            const int i = lane + 32 * t;
            vp[t] = (hp && i < n) ? __ldcg(sp + i) : 0.0;
            vq[t] = (hq && i < n) ? __ldcg(sq + i) : 0.0;
        }
        double ap = 0.0, aq = 0.0;
        double* dp = S + (size_t)warp * n;
        double* dq = S + (size_t)(b + warp) * n;
#pragma unroll
        for (int t = 0; t < NR; t++) {
            const int i = lane + 32 * t;
            if (i < n) {
                if (hp) dp[i] = vp[t];
                if (hq) dq[i] = vq[t];
            }
            ap = fma(vp[t], vp[t], ap);
            aq = fma(vq[t], vq[t], aq);
        }
        ap = warp_sum(ap);
        aq = warp_sum(aq);
        if (lane == 0) { norm2[warp] = ap; norm2[b + warp] = aq; }
    } else {
        for (int lc = warp; lc < 2 * b; lc += b) {
            const bool isq = lc >= b;
            const int l = isq ? lc - b : lc;
            double acc = 0.0;
            if (l < (isq ? cntq : cntp)) {
                const double* src = A + (size_t)((isq ? colq0 : colp0) + l) * n;
                double* dst = S + (size_t)lc * n;
                for (int i = lane; i < n; i += 32) {
                    double v = __ldcg(src + i);
                    dst[i] = v;
                    acc = fma(v, v, acc);
                }
            }
            acc = warp_sum(acc);
            if (lane == 0) norm2[lc] = acc;
        }
    }
    __syncthreads();
    bool any = false;
    if (round == 0) {
        const int P = 2 * b;
        for (int lr = 0; lr < P - 1; lr++) {
            int s1, s2;
            tournament_pair(P, lr, warp, s1, s2);
            const bool v1 = s1 < b ? s1 < cntp : (s1 - b) < cntq;
            const bool v2 = s2 < b ? s2 < cntp : (s2 - b) < cntq;
            any |= rotate_warp<NR>(S + (size_t)s1 * n, S + (size_t)s2 * n, n, lane, v1 && v2, tol2, floor2, relmax);
            __syncthreads();
        }
    } else if constexpr (NR > 0) {
        any = cross_rounds_stationary<NR>(S, norm2, n, b, cntp, cntq, warp, lane, tol2, floor2, relmax);
        __syncthreads();
    } else {
        for (int k = 0; k < b; k++) {
            int j = warp + k;
            j = j >= b ? j - b : j;
            any |= rotate_warp<0>(S + (size_t)warp * n, S + (size_t)(b + j) * n, n, lane, warp < cntp && j < cntq, tol2, floor2, relmax);
            __syncthreads();
        }
    }
    if constexpr (NR > 0) {
        const bool hp = warp < cntp, hq = warp < cntq;
        double* gp = A + (size_t)(colp0 + warp) * n;
        double* gq = A + (size_t)(colq0 + warp) * n;
        const double* sp = S + (size_t)warp * n;
        const double* sq = S + (size_t)(b + warp) * n;
        double vp[NR], vq[NR];
#pragma unroll
        for (int t = 0; t < NR; t++) {
            const int i = lane + 32 * t;
            vp[t] = (hp && i < n) ? sp[i] : 0.0;
            vq[t] = (hq && i < n) ? sq[i] : 0.0;
        }
#pragma unroll
        for (int t = 0; t < NR; t++) {
            const int i = lane + 32 * t;
            if (i < n) {
                if (hp) __stcg(gp + i, vp[t]);
                if (hq) __stcg(gq + i, vq[t]);
            }
        }
    } else {
        for (int lc = warp; lc < 2 * b; lc += b) {
            const bool isq = lc >= b;
            const int l = isq ? lc - b : lc;
            if (l < (isq ? cntq : cntp)) {
                double* dst = A + (size_t)((isq ? colq0 : colp0) + l) * n;
                const double* src = S + (size_t)lc * n;
                for (int i = lane; i < n; i += 32) __stcg(dst + i, src[i]);
            }
        }
    }
    return any;
}

// Persistent solve of an n x ncols column set (column j at A + j*n): grid = nb/2 CTAs
// (cooperative launch), block = 32*b threads.
// ctrl[0]: barrier counter, ctrl[1]: sweeps used (negative = not converged), ctrl[2+s]: sweep flags.
template <int NR>
__global__ void __launch_bounds__(512)
jacobi_persistent_kernel(double* A, int n, int ncols, int b, int nb, int max_sweeps, unsigned* ctrl, double tol2,
                         const double* floor2_ptr, unsigned* stamps, float quad_stop2) {
    extern __shared__ double S[];
    __shared__ int s_skip;
    const double floor2 = *floor2_ptr;
    // stamps[0..nb): time a block was last modified; stamps[nb + p*nb + q]: time the pair (p, q) was
    // last found orthogonal.  A pair verified after both blocks' last modification is still
    // orthogonal and is skipped entirely - the late sweeps, where almost nothing rotates, and the
    // final verification sweep then cost little more than their barriers.
    unsigned* mod = stamps;
    unsigned* okt = stamps + nb;
    unsigned epoch = 0;
    int sweep = 0;
    bool converged = false;
    while (sweep < max_sweeps) {
        for (int round = 0; round < nb - 1; round++) {
            int bp, bq;
            tournament_pair(nb, round, blockIdx.x, bp, bq);
            if (bp > bq) { int t = bp; bp = bq; bq = t; }
            if (threadIdx.x == 0) {
                const unsigned ok = __ldcg(okt + (size_t)bp * nb + bq);
                s_skip = ok != 0 && ok >= __ldcg(mod + bp) && ok >= __ldcg(mod + bq);
            }
            __syncthreads();
            const bool skip = s_skip != 0;
            epoch++;
            if (!skip) {
                float relmax = 0.f;
                bool any = process_block_pair<NR>(A, n, ncols, b, nb, round, blockIdx.x, S, tol2, floor2, relmax);
                any = __syncthreads_or(any ? 1 : 0) != 0;
                // largest squared relative off-diagonal rotated away in this sweep (positive floats order as uints)
                if (relmax > 0.f && (threadIdx.x & 31) == 0) atomicMax(ctrl + 2 + sweep, __float_as_uint(relmax));
                if (threadIdx.x == 0) {
                    if (any) {
                        __stcg(mod + bp, epoch);
                        __stcg(mod + bq, epoch);
                    } else {
                        __stcg(okt + (size_t)bp * nb + bq, epoch);
                    }
                }
            }
            grid_barrier(ctrl, epoch * gridDim.x);
        }
        unsigned flag = __ldcg(ctrl + 2 + sweep);
        sweep++;
        // no rotation at all, or every rotated pair was already so close to orthogonal that - Jacobi
        // converging quadratically - what is left is below the threshold: skip the verification sweep
        if (flag == 0 || __uint_as_float(flag) < quad_stop2) { converged = true; break; }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) ((int*)ctrl)[1] = converged ? sweep : -sweep;
}

// Same work as one round of the persistent kernel, for matrices whose block count exceeds the
// number of co-resident CTAs (n > ~4700): one launch per round.
template <int NR>
__global__ void __launch_bounds__(512)
jacobi_round_kernel(double* A, int n, int ncols, int b, int nb, int round, unsigned* flag, double tol2,
                    const double* floor2_ptr) {
    extern __shared__ double S[];
    float relmax = 0.f;
    bool any = process_block_pair<NR>(A, n, ncols, b, nb, round, blockIdx.x, S, tol2, *floor2_ptr, relmax);
    if (any && (threadIdx.x & 31) == 0) atomicOr(flag, 1u);
}

// |column j| for j < ncols (columns of length n), one warp per column
__global__ void __launch_bounds__(256)
column_norms_kernel(const double* __restrict__ A, int n, int ncols, double* __restrict__ norms) {
    int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= ncols) return;
    const double* col = A + (size_t)warp * n;
    double s = 0.0;
    for (int i = lane; i < n; i += 32) s = fma(col[i], col[i], s);
    s = warp_sum(s);
    if (lane == 0) norms[warp] = sqrt(s);
}

// floor2 = (n * eps * max_j |column j|)^2 : squared norm below which a column counts as null
__global__ void __launch_bounds__(256)
null_floor_kernel(const double* __restrict__ norms, int n, int ncols, double* __restrict__ floor2) {
    __shared__ double scratch[32];
    double m = 0.0;
    for (int i = threadIdx.x; i < ncols; i += blockDim.x) m = fmax(m, norms[i]);
    m = block_max(m, scratch);
    if (threadIdx.x == 0) {
        double f = (double)n * 2.220446049250313e-16 * m;
        floor2[0] = f * f;
    }
}

// descending rank of every column by counting (ties broken by index), then write
// evals[rank] (the norm, or its square when the columns are those of a Cholesky factor) and
// the normalised column into evecs[:, rank] (row-major n x n).  Ranks >= ncols are zero-filled.
__global__ void __launch_bounds__(256)
sort_extract_kernel(const double* __restrict__ A, const double* __restrict__ norms, int n, int ncols, int square,
                    double* __restrict__ evals, double* __restrict__ evecs) {
    int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= n) return;
    if (warp >= ncols) {                                     // rank-deficient tail
        if (lane == 0) evals[warp] = 0.0;
        for (int i = lane; i < n; i += 32) evecs[(size_t)i * n + warp] = 0.0;
        return;
    }
    double mine = norms[warp];
    int cnt = 0;
    for (int k = lane; k < ncols; k += 32) {
        double o = norms[k];
        cnt += (o > mine || (o == mine && k < warp)) ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    int rank = cnt;
    if (lane == 0) evals[rank] = square ? mine * mine : mine;
    double inv = mine > 0.0 ? 1.0 / mine : 0.0;
    const double* col = A + (size_t)warp * n;
    for (int i = lane; i < n; i += 32) evecs[(size_t)i * n + rank] = col[i] * inv;
}

// ---------------------------------------------------------------------------------------------
// Pivoted Cholesky G = L L^T (diagonal pivoting, rank revealing), the preconditioner of the
// Jacobi solve: one-sided Jacobi on the columns of L works on sqrt(lambda) instead of lambda,
// on rank(G) columns instead of n, and L's columns are graded and nearly orthogonal - on the
// bond Gram matrices of real volumes this halves the sweep count (profiles/r01_jacobi_sweeps.md).
//
// Persistent cooperative kernel, rows distributed over CTAs (each keeps its rows of the running
// Schur complement in shared memory), CHB pivots per pair of grid barriers.  Per block step every
// CTA (1) publishes the diagonal of its live rows, (2) picks the same CHB largest candidates, whose
// owners publish those rows, (3) factors the block redundantly with pivoting INSIDE the block (a
// candidate that turns out to depend on the ones already taken is left for a later step), (4)
// writes its rows of the new L columns and applies the rank-CHB update to its slab.  L is produced
// column-major in the ORIGINAL row order (no permutation to undo: G = sum_k l_k l_k^T).  A
// one-pivot-per-barrier kernel gave the same factor quality for preconditioning at ~4x the time.
// ---------------------------------------------------------------------------------------------
constexpr int CHB = 8;

__global__ void __launch_bounds__(256)
pivoted_cholesky_blocked_kernel(const double* __restrict__ G, int n, int rows_per, double* __restrict__ Lcol,
                                double* diag_g, double* rows_g, unsigned* ctrl, double stop_rel) {
    extern __shared__ double sm[];
    double* slab = sm;                                   // rows_per x n
    double* Lc = slab + (size_t)rows_per * n;            // n x CHB   (row c: Lc[c*CHB + j])
    double* rowsB = Lc + (size_t)n * CHB;                // CHB x n
    double* dall = rowsB + (size_t)CHB * n;              // n
    int* dead = reinterpret_cast<int*>(dall + n);        // n
    __shared__ int sel[CHB];
    __shared__ int s_nsel, s_q;
    __shared__ double s_root;
    __shared__ double dd[CHB];
    __shared__ int taken[CHB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, cta = blockIdx.x, ncta = gridDim.x;
    const int row0 = cta * rows_per;
    int nrows = n - row0;
    nrows = nrows < 0 ? 0 : (nrows > rows_per ? rows_per : nrows);
    for (int idx = tid; idx < nrows * n; idx += blockDim.x) slab[idx] = G[(size_t)row0 * n + idx];
    for (int c = tid; c < n; c += blockDim.x) dead[c] = 0;
    __syncthreads();
    double p0 = 0.0;
    int k = 0, rank = n;
    unsigned epoch = 0;
    for (int step = 0; k < n; step++) {
        const int par = step & 1;
        // ---- (1) publish the diagonal of our live rows ----
        if (tid < nrows) __stcg(diag_g + (size_t)par * n + row0 + tid, dead[row0 + tid] ? -1.0 : slab[(size_t)tid * n + row0 + tid]);
        epoch++;
        grid_barrier(ctrl, epoch * ncta);
        // ---- (2) every CTA picks the same CHB largest live diagonals ----
        for (int c = tid; c < n; c += blockDim.x) dall[c] = __ldcg(diag_g + (size_t)par * n + c);
        __syncthreads();
        if (warp == 0) {
            int nsel = 0;
            for (int m = 0; m < CHB; m++) {
                double best = -1.0;
                int bi = -1;
                for (int c = lane; c < n; c += 32) {
                    double d = dall[c];
                    if (d > best) { best = d; bi = c; }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    double ob = __shfl_xor_sync(0xffffffffu, best, o);
                    int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                    if (oi >= 0 && (ob > best || (ob == best && (bi < 0 || oi < bi)))) { best = ob; bi = oi; }
                }
                if (step == 0 && m == 0) p0 = best;                       // same in every lane / CTA
                if (bi < 0 || !(best > stop_rel * p0) || !(best > 0.0)) break;
                if (lane == 0) { sel[m] = bi; dall[bi] = -2.0; }
                nsel++;
                __syncwarp();
            }
            if (lane == 0) s_nsel = nsel;
            if (step == 0) dd[0] = p0;                                   // hand p0 to the other warps
        }
        __syncthreads();
        if (step == 0) p0 = dd[0];
        const int nsel = s_nsel;
        if (nsel == 0) { rank = k; break; }                              // uniform across the grid
        // ---- (3) owners publish the selected rows ----
        for (int m = 0; m < nsel; m++) {
            const int r = sel[m] - row0;
            if (r >= 0 && r < nrows) {
                double* dst = rows_g + ((size_t)par * CHB + m) * n;
                for (int c = tid; c < n; c += blockDim.x) __stcg(dst + c, slab[(size_t)r * n + c]);
            }
        }
        epoch++;
        grid_barrier(ctrl, epoch * ncta);
        {   // all loads in flight before the first store (a load -> store loop serialises L2 round trips)
            const double* src = rows_g + (size_t)par * CHB * n;
            const int total = nsel * n;
            for (int base = 0; base < total; base += 8 * 256) {
                double v[8];
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int idx = base + u * 256 + tid;
                    v[u] = idx < total ? __ldcg(src + idx) : 0.0;
                }
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int idx = base + u * 256 + tid;
                    if (idx < total) rowsB[idx] = v[u];
                }
            }
        }
        if (tid < CHB) { taken[tid] = 0; dd[tid] = 0.0; }
        __syncthreads();
        // ---- (4) factor the block, pivoting among the candidates ----
        int bused = 0;
        for (int j = 0; j < nsel; j++) {
            if (tid < nsel && !taken[tid]) {                             // updated diagonal of candidate tid
                const int rq = sel[tid];
                double d = rowsB[(size_t)tid * n + rq];
                for (int m2 = 0; m2 < j; m2++) d = fma(-Lc[(size_t)rq * CHB + m2], Lc[(size_t)rq * CHB + m2], d);
                dd[tid] = d;
            }
            __syncthreads();
            if (tid == 0) {
                int q = -1;
                for (int t = 0; t < nsel; t++)
                    if (!taken[t] && (q < 0 || dd[t] > dd[q])) q = t;
                if (q >= 0 && dd[q] > stop_rel * p0 && dd[q] > 0.0) { s_q = q; s_root = sqrt(dd[q]); }
                else s_q = -1;
            }
            __syncthreads();
            const int q = s_q;
            if (q < 0) break;                                            // the remaining candidates depend on the taken ones
            const int rq = sel[q];
            const double root = s_root, inv = 1.0 / root;
            for (int c = tid; c < n; c += blockDim.x) {
                double v = 0.0;
                if (c == rq) v = root;
                else if (!dead[c]) {
                    v = rowsB[(size_t)q * n + c];
                    for (int m2 = 0; m2 < j; m2++) v = fma(-Lc[(size_t)c * CHB + m2], Lc[(size_t)rq * CHB + m2], v);
                    v *= inv;
                }
                Lc[(size_t)c * CHB + j] = v;
            }
            __syncthreads();
            if (tid == 0) { dead[rq] = 1; taken[q] = 1; }
            bused = j + 1;
            __syncthreads();
        }
        if (bused == 0) { rank = k; break; }                             // uniform: nothing usable left
        // ---- (5) our rows of the new columns of L, rank-bused update of our live rows ----
        for (int idx = tid; idx < nrows * bused; idx += blockDim.x) {
            const int r = idx / bused, j = idx - r * bused;
            __stcg(Lcol + (size_t)(k + j) * n + row0 + r, Lc[(size_t)(row0 + r) * CHB + j]);
        }
        for (int idx = tid; idx < nrows * n; idx += blockDim.x) {
            const int r = idx / n, c = idx - r * n;
            if (dead[row0 + r]) continue;
            double v = slab[idx];
            for (int j = 0; j < bused; j++) v = fma(-Lc[(size_t)(row0 + r) * CHB + j], Lc[(size_t)c * CHB + j], v);
            slab[idx] = v;
        }
        k += bused;
        __syncthreads();
    }
    if (cta == 0 && tid == 0) ((int*)ctrl)[1] = rank < k ? rank : k;
}

// ---------------------------------------------------------------------------------------------
// All-in-one solver for n <= 64 (beyond that one SM's shared-memory bandwidth is the limit): pivoted Cholesky, Jacobi on the factor's columns, sort and
// eigenvector extraction in ONE CTA and ONE launch (no grid barrier, no host round trip).
//
// Shared memory holds the n x n working matrix column-major.  The Cholesky is right-looking on
// the full symmetric Schur complement with a "dead" mask instead of row/column swaps; column k
// of L is written into the storage of the column that step k eliminates (slot piv[k]), so the
// factorisation is in place.  The Jacobi phase then sweeps the rank columns piv[0..rank) with
// eight lanes per column pair.
// ---------------------------------------------------------------------------------------------
template <int NR>
__global__ void __launch_bounds__(512)
eigh_small_kernel(const double* __restrict__ G, int n, int max_sweeps, double tol2, double stop_rel, float quad_stop2,
                  double diag_tol, double* __restrict__ evals, double* __restrict__ evecs, int* __restrict__ info) {
    extern __shared__ double S[];                    // n columns of stride ld = n + 2 (the pad spreads columns over banks)
    const int ld = n + 2;
    __shared__ int piv[128];                         // piv[k] = original index eliminated at step k = slot of L's column k
    __shared__ int dead[128];
    __shared__ double lcol[128];
    __shared__ double red_val[16];
    __shared__ int red_idx[16];
    __shared__ double s_pval;
    __shared__ int s_prow;
    __shared__ double cnorm[128];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, W = blockDim.x >> 5;
    // ---- already diagonal?  (Rayleigh-Ritz block of converged Ritz vectors, eig_topk.cu): every off-diagonal entry
    // below diag_tol x the largest diagonal entry -> eigenvalues are the diagonal, eigenvectors a permutation.  The
    // caller checks the residuals of what comes out, so a block that only looks diagonal cannot slip through. ----
    if (diag_tol > 0.0) {
        double off = 0.0, dg = 0.0;
        for (int i = tid; i < n * n; i += blockDim.x) {
            const int c = i / n, r = i - c * n;
            const double v = fabs(G[i]);
            if (c == r) dg = fmax(dg, v); else off = fmax(off, v);
        }
        off = warp_max(off);
        dg = warp_max(dg);
        if (lane == 0) { red_val[warp] = off; lcol[warp] = dg; }
        __syncthreads();
        off = 0.0; dg = 0.0;
        for (int w = 0; w < W; w++) { off = fmax(off, red_val[w]); dg = fmax(dg, lcol[w]); }
        __syncthreads();
        if (off <= diag_tol * dg) {                      // uniform over the CTA
            for (int c = warp; c < n; c += W) {
                const double mine = G[(size_t)c * n + c];
                int cnt = 0;
                for (int k = lane; k < n; k += 32) {
                    const double o = G[(size_t)k * n + k];
                    cnt += (o > mine || (o == mine && k < c)) ? 1 : 0;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
                if (lane == 0) evals[cnt] = mine;
                for (int i = lane; i < n; i += 32) evecs[(size_t)i * n + cnt] = i == c ? 1.0 : 0.0;
            }
            if (tid == 0) { info[0] = 0; info[1] = n; }
            return;
        }
    }
    for (int i = tid; i < n * n; i += blockDim.x) { const int c = i / n, r = i - c * n; S[(size_t)c * ld + r] = G[i]; }
    if (tid < n) dead[tid] = 0;
    __syncthreads();
    // ---- pivoted Cholesky ----
    double p0 = 0.0;
    int rank = n;
    for (int k = 0; k < n; k++) {
        double best = -1.0;
        int bi = -1;
        if (tid < n && !dead[tid]) { best = S[(size_t)tid * ld + tid]; bi = tid; }
        if (warp < 4) {                              // n <= 128: candidates live in the first four warps
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                double ob = __shfl_xor_sync(0xffffffffu, best, o);
                int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (oi >= 0 && (ob > best || (ob == best && (bi < 0 || oi < bi)))) { best = ob; bi = oi; }
            }
            if (lane == 0) { red_val[warp] = best; red_idx[warp] = bi; }
        }
        __syncthreads();
        if (tid == 0) {
            double b = -1.0;
            int bj = -1;
            for (int w = 0; w < 4; w++)
                if (red_idx[w] >= 0 && (red_val[w] > b || (red_val[w] == b && (bj < 0 || red_idx[w] < bj)))) { b = red_val[w]; bj = red_idx[w]; }
            s_pval = b;
            s_prow = bj;
        }
        __syncthreads();
        const double pval = s_pval;
        const int prow = s_prow;
        if (k == 0) p0 = pval;
        if (prow < 0 || !(pval > stop_rel * p0) || !(pval > 0.0)) { rank = k; break; }
        const double root = sqrt(pval), inv = 1.0 / root;
        if (tid < n) {
            double l = 0.0;
            if (tid == prow) l = root;
            else if (!dead[tid]) l = S[(size_t)prow * ld + tid] * inv;     // column prow = row prow (symmetric)
            lcol[tid] = l;
        }
        __syncthreads();
        // Schur complement update of the live part; column prow is dead from now on
        for (int idx = tid; idx < n * n; idx += blockDim.x) {
            const int c = idx / n, r = idx - c * n;
            if (c == prow) continue;
            if (!dead[c] && !dead[r] && r != prow) S[(size_t)c * ld + r] = fma(-lcol[r], lcol[c], S[(size_t)c * ld + r]);
        }
        __syncthreads();
        if (tid < n) S[(size_t)prow * ld + tid] = lcol[tid];               // L's column k takes the dead slot
        if (tid == 0) { dead[prow] = 1; piv[k] = prow; }
        __syncthreads();
    }
    // ---- Jacobi on the rank columns (slots piv[0..rank)) ----
    const double floor2 = (double)n * 2.220446049250313e-16 * (double)n * 2.220446049250313e-16 * p0;
    const int grp = lane >> 3, li = lane & 7;
    const int P = (rank + 1) & ~1;
    const int matches = P / 2;
    int sweep = 0;
    int done = rank < 2 ? 1 : 0;
    float relmax = 0.f;
    while (!done && sweep < max_sweeps) {
        bool any = false;
        for (int lr = 0; lr < P - 1; lr++) {
            for (int m0 = warp * 4; m0 < matches; m0 += W * 4) {      // warp-uniform trip count
                const int m = m0 + grp;
                int s1 = 0, s2 = 0;
                if (m < matches) tournament_pair(P, lr, m, s1, s2);
                const bool valid = m < matches && s1 < rank && s2 < rank;
                const int c1 = valid ? piv[s1] : 0, c2 = valid ? piv[s2] : 0;
                any |= rotate_group<NR, 8>(S + (size_t)c1 * ld, S + (size_t)c2 * ld, n, li, valid, tol2, floor2, relmax);
            }
            __syncthreads();
        }
        sweep++;
        done = !__syncthreads_or(any ? 1 : 0);
        // quadratic convergence: a sweep whose largest rotated off-diagonal was below sqrt(quad_stop2)
        // relative leaves less than quad_stop2 behind
        if (quad_stop2 > 0.f && !__syncthreads_or(relmax >= quad_stop2 ? 1 : 0)) done = 1;
        relmax = 0.f;
    }
    // ---- eigenvalues (squared column norms), descending order, eigenvectors ----
    for (int c = warp; c < rank; c += W) {
        const double* col = S + (size_t)piv[c] * ld;
        double s = 0.0;
        for (int i = lane; i < n; i += 32) s = fma(col[i], col[i], s);
        s = warp_sum(s);
        if (lane == 0) cnorm[c] = sqrt(s);
    }
    __syncthreads();
    for (int c = warp; c < n; c += W) {
        if (c >= rank) {                                             // rank-deficient tail
            if (lane == 0) evals[c] = 0.0;
            for (int i = lane; i < n; i += 32) evecs[(size_t)i * n + c] = 0.0;
            continue;
        }
        const double mine = cnorm[c];
        int cnt = 0;
        for (int k = lane; k < rank; k += 32) {
            double o = cnorm[k];
            cnt += (o > mine || (o == mine && k < c)) ? 1 : 0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        if (lane == 0) evals[cnt] = mine * mine;
        const double invn = mine > 0.0 ? 1.0 / mine : 0.0;
        const double* col = S + (size_t)piv[c] * ld;
        for (int i = lane; i < n; i += 32) evecs[(size_t)i * n + cnt] = col[i] * invn;
    }
    if (tid == 0) { info[0] = done ? sweep : -(sweep + 1); info[1] = rank; }
}

template <class K>
static int raise_smem_minus(K kernel, const ndmps_ctx* ctx, int reserve) {
    return raise_dynamic_smem((const void*)kernel, ctx->device, (int)ctx->smem_optin - reserve);
}

template <class K>
static int raise_smem(K kernel, const ndmps_ctx* ctx) {
    // leave room for the kernels' few bytes of static shared memory
    return raise_dynamic_smem((const void*)kernel, ctx->device, (int)ctx->smem_optin - 1024);
}

template <int NR>
static int run_persistent(ndmps_ctx* ctx, double* A, int n, int ncols, int b, int nb, int max_sweeps, unsigned* ctrl,
                          double tol2, const double* floor2, size_t smem, float quad_stop2) {
    NDMPS_TRY(raise_smem(jacobi_persistent_kernel<NR>, ctx));
    unsigned* stamps = nullptr;
    NDMPS_TRY(ctx->ws.get<unsigned>((size_t)nb * nb + nb, &stamps));
    NDMPS_CUDA_TRY(cudaMemsetAsync(stamps, 0, ((size_t)nb * nb + nb) * sizeof(unsigned), ctx->stream));
    void* args[] = {&A, &n, &ncols, &b, &nb, &max_sweeps, &ctrl, &tol2, &floor2, &stamps, &quad_stop2};
    NDMPS_TRY(coop_launch(ctx, (const void*)jacobi_persistent_kernel<NR>, dim3(nb / 2), dim3(32 * b), args, smem));
    return NDMPS_OK;
}

template <int NR>
static int run_round(ndmps_ctx* ctx, double* A, int n, int ncols, int b, int nb, int round, unsigned* flag, double tol2,
                     const double* floor2, size_t smem) {
    NDMPS_TRY(raise_smem(jacobi_round_kernel<NR>, ctx));
    jacobi_round_kernel<NR><<<nb / 2, 32 * b, smem, ctx->stream>>>(A, n, ncols, b, nb, round, flag, tol2, floor2);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

// Jacobi sweeps over the ncols columns (length n) stored at A + j*n, block path.
static int jacobi_columns(ndmps_ctx* ctx, double* A, int n, int ncols, double tol2, const double* floor2, int* sweeps_used,
                          float quad_stop2) {
    const int max_sweeps = JACOBI_MAX_SWEEPS;
    const size_t smem_cap = ctx->smem_optin > 4096 ? ctx->smem_optin - 2048 : 0;
    unsigned* ctrl = nullptr;   // [0] barrier counter, [1] sweeps used, [2..] per-sweep rotation flags
    NDMPS_TRY(ctx->ws.get<unsigned>((size_t)max_sweeps + 4, &ctrl));
    NDMPS_CUDA_TRY(cudaMemsetAsync(ctrl, 0, ((size_t)max_sweeps + 4) * sizeof(unsigned), ctx->stream));
    int* host_flag = reinterpret_cast<int*>(ctx->pinned);
    const int nr = n <= 256 ? 8 : n <= 512 ? 16 : 0;      // rows per lane of the block kernels
    // block size: as many columns as shared memory allows, at most 8 (measured best: more CTAs, cheaper rounds)
    int b = (int)((smem_cap - 512) / (16 * (size_t)n));
    if (b > 8) b = 8;
    NDMPS_REQUIRE(b >= 1, "eigh: n = %d does not fit a column pair in shared memory", n);
    while (b > 1 && (ncols + b - 1) / b < 2) b /= 2;      // at least two blocks
    int nb = (ncols + b - 1) / b;
    if (nb & 1) nb++;
    if (nb < 2) nb = 2;
    const size_t smem = ((size_t)2 * b * n + 2 * b) * sizeof(double);
    if (nb / 2 <= ctx->sm_count) {
        switch (nr) {
            case 8: NDMPS_TRY(run_persistent<8>(ctx, A, n, ncols, b, nb, max_sweeps, ctrl, tol2, floor2, smem, quad_stop2)); break;
            case 16: NDMPS_TRY(run_persistent<16>(ctx, A, n, ncols, b, nb, max_sweeps, ctrl, tol2, floor2, smem, quad_stop2)); break;
            default: NDMPS_TRY(run_persistent<0>(ctx, A, n, ncols, b, nb, max_sweeps, ctrl, tol2, floor2, smem, quad_stop2)); break;
        }
        NDMPS_TRY(readback(ctx, host_flag, ctrl + 1, sizeof(int)));
        NDMPS_CUDA_TRY(stream_wait(ctx));
        if (host_flag[0] <= 0) {
            set_error("eigh: Jacobi did not converge in %d sweeps (n = %d, cols = %d, b = %d)", max_sweeps, n, ncols, b);
            return NDMPS_ERR_NOCONV;
        }
        *sweeps_used = host_flag[0];
        return NDMPS_OK;
    }
    bool converged = false;
    for (int s = 0; s < max_sweeps && !converged; s++) {
        unsigned* flag = ctrl + 2 + s;
        for (int round = 0; round < nb - 1; round++)
            NDMPS_TRY(run_round<0>(ctx, A, n, ncols, b, nb, round, flag, tol2, floor2, smem));
        *sweeps_used = s + 1;
        if (s >= 3) {
            NDMPS_TRY(readback(ctx, host_flag, flag, sizeof(int)));
            NDMPS_CUDA_TRY(stream_wait(ctx));
            converged = host_flag[0] == 0;
        }
    }
    if (!converged) {
        set_error("eigh: Jacobi did not converge in %d sweeps (n = %d, cols = %d, b = %d)", max_sweeps, n, ncols, b);
        return NDMPS_ERR_NOCONV;
    }
    return NDMPS_OK;
}

// G = L L^T with diagonal pivoting; returns the numerical rank (host) and L column-major.
static int pivoted_cholesky(ndmps_ctx* ctx, const double* G, int n, double* Lcol, int* rank_out) {
    int rows_per = (n + 127) / 128;                          // many small slabs: the per-step update is the critical path
    int ncta = (n + rows_per - 1) / rows_per;
    while (ncta > ctx->sm_count) { rows_per++; ncta = (n + rows_per - 1) / rows_per; }
    const size_t smem = ((size_t)rows_per * n + (size_t)n * CHB + (size_t)CHB * n + n) * sizeof(double) + (size_t)n * sizeof(int) + 16;
    NDMPS_REQUIRE(smem <= ctx->smem_optin - 4096, "pivoted_cholesky: n = %d does not fit shared memory", n);
    // the kernel also has static shared memory: static + dynamic must stay within the opt-in limit
    NDMPS_TRY(raise_smem_minus(pivoted_cholesky_blocked_kernel, ctx, 4096));
    double *diag_g = nullptr, *rows_g = nullptr;
    unsigned* ctrl = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)2 * n, &diag_g));
    NDMPS_TRY(ctx->ws.get<double>((size_t)2 * CHB * n, &rows_g));
    NDMPS_TRY(ctx->ws.get<unsigned>(4, &ctrl));
    NDMPS_CUDA_TRY(cudaMemsetAsync(ctrl, 0, 4 * sizeof(unsigned), ctx->stream));
    double stop_rel = 2.220446049250313e-16;
    void* args[] = {&G, &n, &rows_per, &Lcol, &diag_g, &rows_g, &ctrl, &stop_rel};
    NDMPS_TRY(coop_launch(ctx, (const void*)pivoted_cholesky_blocked_kernel, dim3(ncta), dim3(256), args, smem));
    int* host_flag = reinterpret_cast<int*>(ctx->pinned);
    NDMPS_TRY(readback(ctx, host_flag, ctrl + 1, sizeof(int)));
    NDMPS_CUDA_TRY(stream_wait(ctx));
    *rank_out = host_flag[0];
    return NDMPS_OK;
}

// Single-CTA solver for 2 <= n <= 64, no host synchronisation: *info_dev points at {sweeps (negative:
// not converged), rank} on the device.  quad_stop2 > 0: also stop after a sweep whose largest rotated
// off-diagonal, squared and relative, was below it.
int eigh_small_async(ndmps_ctx* ctx, double* a_in, int n, double* evals_dev, double* evecs_dev, float quad_stop2, int** info_dev,
                     double diag_tol) {
    NDMPS_REQUIRE(n >= 2 && n <= 64, "eigh_small_async: n = %d outside 2..64", n);
    const int max_sweeps = JACOBI_MAX_SWEEPS;
    const double tol = jacobi_tol(n);
    const double tol2 = tol * tol;
    int* info = nullptr;
    NDMPS_TRY(ctx->ws.get<int>(4, &info));
    const size_t smem = (size_t)n * (n + 2) * sizeof(double);
    const double stop_rel = 2.220446049250313e-16;
#define NDMPS_SMALL(NRV)                                                                                              \
    do {                                                                                                            \
        NDMPS_TRY(raise_smem_minus(eigh_small_kernel<NRV>, ctx, 8192));                                           \
        eigh_small_kernel<NRV><<<1, 512, smem, ctx->stream>>>(a_in, n, max_sweeps, tol2, stop_rel, quad_stop2, diag_tol, evals_dev, evecs_dev, info); \
    } while (0)
    if (n <= 32) NDMPS_SMALL(4);
    else NDMPS_SMALL(8);
#undef NDMPS_SMALL
    NDMPS_LAUNCH_CHECK(ctx);
    *info_dev = info;
    return NDMPS_OK;
}

int eigh(ndmps_ctx* ctx, double* a_in, int64_t n64, double* evals_dev, double* evecs_dev, double tol_override) {
    NDMPS_REQUIRE(n64 >= 1 && n64 <= 16384, "eigh: n = %lld outside 1..16384", (long long)n64);
    const int n = (int)n64;
    NDMPS_TRY(ensure_pinned(ctx, 64));
    int sweeps_used = 0;
    double* norms = nullptr;
    double* floor2 = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)n, &norms));
    NDMPS_TRY(ctx->ws.get<double>(1, &floor2));
    const int ngrid = (n * 32 + 255) / 256;
    double tol = jacobi_tol(n);
    if (tol_override > tol) tol = tol_override;
    const double tol2 = tol * tol;

    if (n >= 2 && n <= 64) {
        // one launch; the convergence code is read back here because the eigenvalues are needed on the host next
        int* info = nullptr;
        NDMPS_TRY(eigh_small_async(ctx, a_in, n, evals_dev, evecs_dev, tol_override > 0.0 ? 1e-14f : 0.f, &info));
        int* host_flag = reinterpret_cast<int*>(ctx->pinned);
        NDMPS_TRY(readback(ctx, host_flag, info, 2 * sizeof(int)));
        NDMPS_CUDA_TRY(stream_wait(ctx));
        if (host_flag[0] < 0) {
            set_error("eigh: Jacobi did not converge in %d sweeps (n = %d, single-CTA solver)", JACOBI_MAX_SWEEPS, n);
            return NDMPS_ERR_NOCONV;
        }
        ctx->last_eig_sweeps = host_flag[0];
        ctx->eig_calls++;
        ctx->eig_flops += 7.0 * n * 0.5 * host_flag[1] * (host_flag[1] - 1.0) * host_flag[0] + (double)n * host_flag[1] * host_flag[1];
        if (ctx->opt_verbose) fprintf(stderr, "[ndmps] eigh n = %d: %d columns, %d sweeps (single CTA)\n", n, host_flag[1], host_flag[0]);
        return NDMPS_OK;
    }
    double* cols = a_in;      // the column set Jacobi works on
    int ncols = n;
    int square = 0;           // eigenvalue = column norm (Jacobi on G) or its square (Jacobi on L)
    const bool use_chol = n > 64 && n <= 1024;      // n = 1 takes neither the Cholesky nor a sweep
    if (use_chol) {
        double* Lcol = nullptr;
        NDMPS_TRY(ctx->ws.get<double>((size_t)n * n, &Lcol));
        int rank = 0;
        NDMPS_TRY(pivoted_cholesky(ctx, a_in, n, Lcol, &rank));
        cols = Lcol;
        ncols = rank;
        square = 1;
    }
    if (ncols >= 1) {
        column_norms_kernel<<<ngrid, 256, 0, ctx->stream>>>(cols, n, ncols, norms);
        NDMPS_LAUNCH_CHECK(ctx);
        null_floor_kernel<<<1, 256, 0, ctx->stream>>>(norms, n, ncols, floor2);
        NDMPS_LAUNCH_CHECK(ctx);
    }
    if (ncols >= 2) {
        // float32 payloads (loosened tolerance): a sweep whose largest rotated off-diagonal was below
        // 1e-7 relative leaves less than the tolerance behind (quadratic convergence), so it is the last
        const float quad_stop2 = tol_override > 0.0 ? 1e-14f : 0.f;
        NDMPS_TRY(jacobi_columns(ctx, cols, n, ncols, tol2, floor2, &sweeps_used, quad_stop2));
    }
    ctx->last_eig_sweeps = sweeps_used;
    ctx->eig_calls++;
    ctx->eig_flops += 7.0 * n * 0.5 * ncols * (ncols - 1.0) * sweeps_used + (use_chol ? (double)n * ncols * ncols : 0.0);
    if (ctx->opt_verbose)
        fprintf(stderr, "[ndmps] eigh n = %d: %d columns, %d sweeps%s\n", n, ncols, sweeps_used, use_chol ? " (pivoted Cholesky)" : "");
    if (ncols >= 1) {
        column_norms_kernel<<<ngrid, 256, 0, ctx->stream>>>(cols, n, ncols, norms);
        NDMPS_LAUNCH_CHECK(ctx);
    }
    sort_extract_kernel<<<ngrid, 256, 0, ctx->stream>>>(cols, norms, n, ncols, square, evals_dev, evecs_dev);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

}  // namespace ndmps

using namespace ndmps;

extern "C" {

int ndmps_eigh(ndmps_ctx_t* ctx, double* a_dev, int64_t n, double* evals_dev, double* evecs_dev, int* sweeps_out_host) {
    NDMPS_REQUIRE(ctx && a_dev && evals_dev && evecs_dev, "ndmps_eigh: NULL argument");
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    NDMPS_TRY(eigh(ctx, a_dev, n, evals_dev, evecs_dev, 0.0));
    if (sweeps_out_host) *sweeps_out_host = ctx->last_eig_sweeps;
    return NDMPS_OK;
}

}  // extern "C"
