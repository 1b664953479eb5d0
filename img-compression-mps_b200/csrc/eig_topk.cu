// K3b: the leading k eigenpairs of a bond-sized Gram matrix, float64.
//
// When from_dense / compress run with a bond cap (core/ndmps.py:74 via quimb's max_bond; the
// reference benchmark's chi = 64 on (chi d) x (chi d) = 512 x 512 Gram matrices), only the k
// largest singular triplets of an unfolding are kept, and the trimming rule
// (quimb.tensor.decomp, Appendix A.1 of SURVEY.md) needs nothing else from the discarded part than its
// total weight, which is trace(G) minus the kept eigenvalues.  So instead of diagonalising
// the whole matrix (eig.cu: ~n sequential rounds per sweep, ~11 sweeps) this path does
//
//   1. G = Q T Q^T          Householder tridiagonalisation, ONE persistent cooperative launch,
//                           one grid barrier per column (tridiag_kernel);
//   2. k shifts             bisection on T, 129-section per pass (bisect_kernel);
//   3. k vectors of T       inverse iteration (pivoted tridiagonal LU, one CTA per shift),
//                           the block re-orthonormalised by Cholesky-QR between iterations so
//                           unresolved clusters keep spanning their invariant subspace;
//   4. Rayleigh-Ritz        H = Q_k^T T Q_k (k x k) through the Jacobi solver of eig.cu: the
//                           returned eigenvalues are second-order accurate Ritz values and the
//                           basis is rotated inside clusters;
//   5. U = Q Z              the Householder reflectors applied to the k Ritz vectors.
//
// n - 2 sequential steps instead of ~11 n, and everything after step 1 works on k vectors.
// The caller (ttsvd.cu) checks on the host that the cap really binds (discarded weight well
// above the cutoff target, lambda_k well above the rounding floor of T) and otherwise falls
// back to the full solver, so rank decisions stay identical to the oracle's.
#include <mutex>

#include "common.cuh"

namespace ndmps {

namespace topk {

// threads per CTA of the tridiagonalisation.  512 = 16 rows per CTA: alone it is ~3 % slower than 256, but a
// reduction then sits on half as many SMs, which leaves room for the register-hungry Gram / GEMM CTAs of the
// other volumes in flight (batch throughput +8 %)
constexpr int TDT = 512;
constexpr int MID_NT = 352;   // threads per CTA of the 1024 < n <= 1536 register-resident reduction
constexpr int NMAX = 4096; // largest matrix of this path (registers up to 1024, L2-resident working copy beyond)
constexpr int BIS = 128;   // shifts per pass and eigenvalue in the bisection

__device__ __forceinline__ double rcp_fast(double x) {      // MUFU seed + 2 Newton steps, normal range
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(r, fma(-x, r, 1.0), r);
    r = fma(r, fma(-x, r, 1.0), r);
    return r;
}

__device__ __forceinline__ double rsqrt_fast(double x) {    // MUFU seed + 2 Newton steps, normal range
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x * r, r, 1.0);
    r = fma(0.5 * r, e, r);
    e = fma(-x * r, r, 1.0);
    r = fma(0.5 * r, e, r);
    return r;
}

// arrive: fence + relaxed add; wait: acquire loads.  Everything read after it goes through L2 (ld.cg).
__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1u);
        unsigned seen;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counter) : "memory");
        } while (seen < target);
    }
    __syncthreads();
}

// all threads of all CTAs of the cluster; release / acquire at cluster scope orders the remote shared-memory stores
__device__ __forceinline__ void cluster_barrier() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// sum over the CTA's NW warps, same value (bitwise) in every thread; one __syncthreads; the partial sums are added
// as a tree (4 dependent adds)
template <int NW = TDT / 32>
__device__ __forceinline__ double block_sum_all(double v, double* scratch) {
    static_assert(NW <= 16, "at most 16 warps");
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
    __syncthreads();
    double s[16];
#pragma unroll
    for (int w = 0; w < 16; w++) s[w] = w < NW ? scratch[w] : 0.0;
#pragma unroll
    for (int o = 8; o > 0; o >>= 1)
#pragma unroll
        for (int w = 0; w < o; w++) s[w] += s[w + o];
    return s[0];
}

// The inner pass of the tridiagonalisation for the chunks Q0 .. NEQ-1 of a warp's RPW rows: A -= u w^T + w u^T on
// these columns, acc += A u'.  No predicates and no branches: the loads of u, w, u' are hoisted ahead of the
// dependent DFMA pairs by the compiler, which a per-chunk `if` prevented (each chunk then cost a full
// shared-memory latency).
template <int NEQ, int RPW, int Q0>
__device__ __forceinline__ void fused_pass(double (&a)[RPW][NEQ], const double* __restrict__ u, const double* __restrict__ wv,
                                           const double* __restrict__ un, int lane, const double (&ui)[RPW],
                                           const double (&wi)[RPW], double (&acc)[RPW]) {
    double acc1[RPW];
#pragma unroll
    for (int t = 0; t < RPW; t++) acc1[t] = 0.0;
#pragma unroll
    for (int q = Q0; q < NEQ; q++) {
        const int k = lane + 32 * q;
        const double wk = wv[k], uk = u[k], nk = un[k];
#pragma unroll
        for (int t = 0; t < RPW; t++) {
            double v = a[t][q];
            v = fma(-ui[t], wk, v);
            v = fma(-wi[t], uk, v);
            a[t][q] = v;
            if (q & 1) acc1[t] = fma(v, nk, acc1[t]); else acc[t] = fma(v, nk, acc[t]);
        }
    }
#pragma unroll
    for (int t = 0; t < RPW; t++) acc[t] += acc1[t];
}

// ---------------------------------------------------------------------------------------------
// 1. Householder tridiagonalisation.  Rows are dealt cyclically to the CTAs and then to their warps,
// RPW rows per warp, in REGISTERS (full rows: the symmetric half is not exploited, the 2x flops are
// free next to the barrier).  RPW = 2 up to n = 512: 16 CTAs x 512 threads x 128 registers, so a
// reduction owns its SMs outright and leaves all the others to the kernels of the volumes running
// beside it (see profiles/r01_summary.md, "Interference between volumes in flight").  Per column jn every CTA redundantly derives, from the partial
// products p = A u and the pivot row that were published before the barrier, the vector w of
// the rank-2 update of the PREVIOUS reflector and the NEXT reflector u'; then one fused pass
// over its rows applies A -= u w^T + w u^T and accumulates p' = A u', publishes p' and the next
// pivot row, and meets the others at the barrier.  One barrier per column.
// V row j = reflector j (unit at j+1, zero before), H_j = I - tau_j v_j v_j^T.
// ---------------------------------------------------------------------------------------------
//
// CL = true (n <= 512, two rows per warp): the <= 16 CTAs are ONE thread-block cluster and the per-column exchange
// never leaves the SMs.  Every owner pushes (p_i, A[i][jn+1]) of its rows into the shared memory of all CTAs of
// the cluster (st.shared::cluster; the pivot ROW of the global-memory variant is read as the pivot COLUMN, which
// by symmetry each CTA already holds for its own rows) and the column ends in the hardware cluster barrier
// instead of an L2 atomic + poll + reload.  Measured: 2.50 -> 2.28 ms per n = 512 problem (profiles/r02_summary.md
// has the per-phase cycle counts and the two restructurings that did NOT pay).
// NT threads per CTA: 512 up to n = 1024; 352 (11 warps, one 48-chunk row each, up to 186 registers) for
// 1024 < n <= 1536, where ceil(n / 11) <= 140 CTAs put the whole matrix into the register files of the chip.
template <int NEQ, int RPW, bool CL, int NT>
__global__ void __launch_bounds__(NT)
tridiag_kernel(const double* __restrict__ G, int n, int ldv, double* __restrict__ V, double* __restrict__ tau_g,
               double* __restrict__ d_g, double* __restrict__ e_g, double* pbuf, double* rowbuf, unsigned* ctrl) {
    __shared__ double ub0[32 * NEQ], ub1[32 * NEQ], wv[32 * NEQ];
    __shared__ double red0[NT / 32], red1[NT / 32];
    __shared__ double s_alpha;
    __shared__ double2 pcol[CL ? 2 * 32 * NEQ : 1];                                  // (p_k, A[k][pivot]) of both parities
    constexpr int KM = (32 * NEQ + NT - 1) / NT;                 // vector elements per thread
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, cta = blockIdx.x, C = gridDim.x;
    // this warp's RPW rows, held in registers: lane l has columns l + 32 q.  Row t of the warp is row
    // (t * warps + warp) * C + cta of the matrix (cyclic over CTAs first, so live rows stay spread to the end)
    int gi[RPW];
    double a[RPW][NEQ];
#pragma unroll
    for (int t = 0; t < RPW; t++) {
        gi[t] = (t * (NT / 32) + warp) * C + cta;
#pragma unroll
        for (int q = 0; q < NEQ; q++) {
            const int k = lane + 32 * q;
            a[t][q] = (gi[t] < n && k < n) ? G[(size_t)gi[t] * n + k] : 0.0;
        }
    }
    for (int c = tid; c < 32 * NEQ; c += NT) { ub0[c] = 0.0; ub1[c] = 0.0; wv[c] = 0.0; }
    double* u = ub0;
    double* un = ub1;
    double tau = 0.0;
    unsigned epoch = 0;
    __syncthreads();
    if constexpr (CL) cluster_barrier();                 // every CTA of the cluster is resident before the first remote store
    for (int jn = 0; jn <= n - 2; jn++) {
        const int par = jn & 1;
        double r[KM];                                    // row jn of the current matrix, columns >= jn
        if (jn == 0) {
#pragma unroll
            for (int m = 0; m < KM; m++) {
                const int k = tid + m * NT;
                r[m] = k < n ? G[k] : 0.0;
            }
        } else {
            double pf[KM], rj[KM];
            double pj;
            if constexpr (CL) {
                const double2* pc = pcol + (par ^ 1) * 32 * NEQ;
#pragma unroll
                for (int m = 0; m < KM; m++) {
                    const int k = tid + m * NT;
                    const bool on = k >= jn && k < n;
                    const double2 v = on ? pc[k] : make_double2(0.0, 0.0);
                    pf[m] = v.x;
                    rj[m] = v.y;
                }
                pj = pc[jn].x;
            } else {
                const double* pb = pbuf + (size_t)(par ^ 1) * n;
                const double* rb = rowbuf + (size_t)(par ^ 1) * n;
#pragma unroll
                for (int m = 0; m < KM; m++) {
                    const int k = tid + m * NT;
                    const bool on = k >= jn && k < n;
                    pf[m] = on ? __ldcg(pb + k) : 0.0;
                    rj[m] = on ? __ldcg(rb + k) : 0.0;
                }
                pj = __ldcg(pb + jn);
            }
            double part = 0.0;
#pragma unroll
            for (int m = 0; m < KM; m++) part = fma(pf[m], u[tid + m * NT], part);
            const double s = block_sum_all<NT / 32>(part, red0);
            const double K = -0.5 * tau * tau * s;
            const double wj = fma(tau, pj, K);           // u[jn] = 1
#pragma unroll
            for (int m = 0; m < KM; m++) {
                const int k = tid + m * NT;
                r[m] = 0.0;
                if (k >= jn && k < n) {
                    const double uk = u[k];
                    const double wk = fma(tau, pf[m], K * uk);
                    wv[k] = wk;
                    r[m] = rj[m] - wk - wj * uk;
                }
            }
        }
#pragma unroll
        for (int m = 0; m < KM; m++) {
            const int k = tid + m * NT;
            if (k == jn && cta == 0) d_g[jn] = r[m];
            if (k == jn + 1) s_alpha = r[m];
        }
        if (jn == n - 2) {                               // last 2 x 2 block: no reflector left
            __syncthreads();
            if (cta == 0 && tid == 0) { e_g[jn] = s_alpha; tau_g[jn] = 0.0; }
#pragma unroll
            for (int t = 0; t < RPW; t++) {
                if (gi[t] == n - 1) {
#pragma unroll
                    for (int q = 0; q < NEQ; q++)
                        if (lane + 32 * q == n - 1) d_g[n - 1] = a[t][q] - (jn > 0 ? 2.0 * u[n - 1] * wv[n - 1] : 0.0);
                }
            }
            break;
        }
        double part = 0.0;
#pragma unroll
        for (int m = 0; m < KM; m++) {
            const int k = tid + m * NT;
            if (k >= jn + 2 && k < n) part = fma(r[m], r[m], part);
        }
        const double sigma = block_sum_all<NT / 32>(part, red1);  // the barrier inside also publishes s_alpha and wv
        const double alpha = s_alpha;
        double beta = alpha, taun = 0.0, scal = 0.0;
        if (sigma > 1e-280) {
            const double h2 = fma(alpha, alpha, sigma);
            beta = -copysign(h2 * rsqrt_fast(h2), alpha);
            taun = (beta - alpha) * rcp_fast(beta);
            scal = rcp_fast(alpha - beta);
        }
#pragma unroll
        for (int m = 0; m < KM; m++) {
            const int k = tid + m * NT;
            const double v = k == jn + 1 ? 1.0 : ((k >= jn + 2 && k < n) ? r[m] * scal : 0.0);
            if (k < 32 * NEQ) un[k] = v;
            if (cta == jn % C && k < ldv) V[(size_t)jn * ldv + k] = v;   // the pad element of an odd n too: rows are read in 16-byte chunks
        }
        if (cta == 0 && tid == 0) { e_g[jn] = beta; tau_g[jn] = taun; }
        __syncthreads();
        // fused rank-2 update (reflector jn-1) + product with reflector jn, this warp's rows, column chunks >= jn+1.
        // Straight-line code from the first live quarter of the chunks on (fused_pass): dead columns and dead rows
        // are updated with whatever finite values the vectors hold there and multiply u'[k] = 0.
        {
            double* pw = pbuf + (size_t)par * n;
            double* rw = rowbuf + (size_t)par * n;
            const int q0 = (jn + 1) >> 5;
            double acc[RPW], colv[RPW], ui[RPW], wi[RPW];
            bool live[RPW];
            bool any = false;
#pragma unroll
            for (int t = 0; t < RPW; t++) {
                live[t] = gi[t] >= jn + 1 && gi[t] < n;
                any = any || live[t];
                acc[t] = 0.0;
                colv[t] = 0.0;
                ui[t] = live[t] ? u[gi[t]] : 0.0;        // zero while jn == 0
                wi[t] = live[t] ? wv[gi[t]] : 0.0;
            }
            if (any) {
                constexpr int QG = NEQ / 4;
                switch (q0 / QG) {
                    case 0: fused_pass<NEQ, RPW, 0>(a, u, wv, un, lane, ui, wi, acc); break;
                    case 1: fused_pass<NEQ, RPW, QG>(a, u, wv, un, lane, ui, wi, acc); break;
                    case 2: fused_pass<NEQ, RPW, 2 * QG>(a, u, wv, un, lane, ui, wi, acc); break;
                    default: fused_pass<NEQ, RPW, 3 * QG>(a, u, wv, un, lane, ui, wi, acc); break;
                }
                if constexpr (CL) {
                    // the pivot column jn+1 sits in chunk q0, lane (jn+1) % 32
#pragma unroll
                    for (int t = 0; t < RPW; t++) {
#pragma unroll
                        for (int q = 0; q < NEQ; q++)
                            if (q == q0) colv[t] = a[t][q];
                        colv[t] = __shfl_sync(0xffffffffu, colv[t], (jn + 1) & 31);
                    }
                } else {
#pragma unroll
                    for (int t = 0; t < RPW; t++) {
                        if (gi[t] == jn + 1) {
#pragma unroll
                            for (int q = 0; q < NEQ; q++) {
                                const int k = lane + 32 * q;
                                if (q >= q0 && k >= jn + 1 && k < n) __stcg(rw + k, a[t][q]);
                            }
                        }
                    }
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1)              // the RPW reductions interleaved
#pragma unroll
                for (int t = 0; t < RPW; t++) acc[t] += __shfl_xor_sync(0xffffffffu, acc[t], o);
            if constexpr (CL) {
                // lane l hands this warp's rows to CTA l of the cluster
                const unsigned base = (unsigned)__cvta_generic_to_shared(pcol + par * 32 * NEQ);
#pragma unroll
                for (int t = 0; t < RPW; t++)
                    if (live[t] && lane < C) {
                        unsigned remote;
                        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(base + (unsigned)gi[t] * 16u), "r"(lane));
                        asm volatile("st.shared::cluster.v2.f64 [%0], {%1, %2};" ::"r"(remote), "d"(acc[t]), "d"(colv[t]) : "memory");
                    }
            } else {
#pragma unroll
                for (int t = 0; t < RPW; t++)
                    if (live[t] && lane == 0) __stcg(pw + gi[t], acc[t]);
            }
        }
        if constexpr (CL) {
            cluster_barrier();
        } else {
            epoch++;
            grid_barrier(ctrl, epoch * C);
        }
        double* t = u; u = un; un = t;
        tau = taun;
    }
}

// ---------------------------------------------------------------------------------------------
// 1c. n > 1024 (bond x wide site, e.g. 64 x 40 rows): the matrix no longer fits the register files,
// so the working copy stays in global memory (L2-resident up to ~3500^2) and the fused pass streams
// the live part of every row through the SMs once per column: same algorithm, same one barrier per
// column, rows dealt cyclically to the warps of a grid of one CTA per SM.  The three n-vectors
// live in dynamic shared memory.  Traffic 16 n^3 / 3 bytes through L2 in total.
// ---------------------------------------------------------------------------------------------
constexpr int KMAX_BIG = 16;    // vector elements per thread -> n <= 4096

__global__ void __launch_bounds__(TDT)
tridiag_big_kernel(double* __restrict__ A, int n, int ldv, double* __restrict__ V, double* __restrict__ tau_g,
                   double* __restrict__ d_g, double* __restrict__ e_g, double* pbuf, double* rowbuf, unsigned* ctrl) {
    extern __shared__ double sm[];
    double* ub0 = sm;
    double* ub1 = sm + n;
    double* wv = sm + 2 * (size_t)n;
    __shared__ double red0[TDT / 32], red1[TDT / 32];
    __shared__ double s_alpha;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, cta = blockIdx.x, C = gridDim.x;
    const int gw = warp * C + cta, nw = (TDT / 32) * C;  // this warp owns rows gw, gw + nw, ...
    for (int c = tid; c < n; c += TDT) { ub0[c] = 0.0; ub1[c] = 0.0; wv[c] = 0.0; }
    double* u = ub0;
    double* un = ub1;
    double tau = 0.0;
    unsigned epoch = 0;
    __syncthreads();
    for (int jn = 0; jn <= n - 2; jn++) {
        const int par = jn & 1;
        double r[KMAX_BIG];
        if (jn == 0) {
#pragma unroll
            for (int m = 0; m < KMAX_BIG; m++) {
                const int k = tid + m * TDT;
                r[m] = k < n ? A[k] : 0.0;
            }
        } else {
            const double* pb = pbuf + (size_t)(par ^ 1) * n;
            const double* rb = rowbuf + (size_t)(par ^ 1) * n;
            double pf[KMAX_BIG];
#pragma unroll
            for (int m = 0; m < KMAX_BIG; m++) {
                const int k = tid + m * TDT;
                const bool on = k >= jn && k < n;
                pf[m] = on ? __ldcg(pb + k) : 0.0;
                r[m] = on ? __ldcg(rb + k) : 0.0;
            }
            const double pj = __ldcg(pb + jn);
            double part = 0.0;
#pragma unroll
            for (int m = 0; m < KMAX_BIG; m++) {
                const int k = tid + m * TDT;
                if (k < n) part = fma(pf[m], u[k], part);
            }
            const double s = block_sum_all(part, red0);
            const double K = -0.5 * tau * tau * s;
            const double wj = fma(tau, pj, K);
#pragma unroll
            for (int m = 0; m < KMAX_BIG; m++) {
                const int k = tid + m * TDT;
                if (k >= jn && k < n) {
                    const double uk = u[k];
                    const double wk = fma(tau, pf[m], K * uk);
                    wv[k] = wk;
                    r[m] = r[m] - wk - wj * uk;
                } else {
                    r[m] = 0.0;
                }
            }
        }
#pragma unroll
        for (int m = 0; m < KMAX_BIG; m++) {
            const int k = tid + m * TDT;
            if (k == jn && cta == 0) d_g[jn] = r[m];
            if (k == jn + 1) s_alpha = r[m];
        }
        if (jn == n - 2) {
            __syncthreads();
            if (cta == 0 && tid == 0) { e_g[jn] = s_alpha; tau_g[jn] = 0.0; }
            if ((n - 1) % nw == gw && lane == 0)
                d_g[n - 1] = __ldcg(A + (size_t)(n - 1) * n + (n - 1)) - (jn > 0 ? 2.0 * u[n - 1] * wv[n - 1] : 0.0);
            break;
        }
        double part = 0.0;
#pragma unroll
        for (int m = 0; m < KMAX_BIG; m++) {
            const int k = tid + m * TDT;
            if (k >= jn + 2 && k < n) part = fma(r[m], r[m], part);
        }
        const double sigma = block_sum_all(part, red1);
        const double alpha = s_alpha;
        double beta = alpha, taun = 0.0, scal = 0.0;
        if (sigma > 1e-280) {
            const double h2 = fma(alpha, alpha, sigma);
            beta = -copysign(h2 * rsqrt_fast(h2), alpha);
            taun = (beta - alpha) * rcp_fast(beta);
            scal = rcp_fast(alpha - beta);
        }
#pragma unroll
        for (int m = 0; m < KMAX_BIG; m++) {
            const int k = tid + m * TDT;
            if (k < n) {
                const double v = k == jn + 1 ? 1.0 : (k >= jn + 2 ? r[m] * scal : 0.0);
                un[k] = v;
                if (cta == jn % C) V[(size_t)jn * ldv + k] = v;
            }
        }
        if (cta == 0 && tid == 0) { e_g[jn] = beta; tau_g[jn] = taun; }
        __syncthreads();
        // fused rank-2 update (reflector jn-1) + product with reflector jn over this warp's live rows
        double* pw = pbuf + (size_t)par * n;
        double* rw = rowbuf + (size_t)par * n;
        const int kbase = (jn + 1) & ~31;
        int first = gw;
        if (first < jn + 1) first += ((jn + 1 - first + nw - 1) / nw) * nw;
        for (int gi = first; gi < n; gi += nw) {
            double* Ar = A + (size_t)gi * n;
            const bool pub = gi == jn + 1;
            const double ui = u[gi], wi = wv[gi];          // zero while jn == 0
            double acc0 = 0.0, acc1 = 0.0;
            int k = kbase + lane;
            for (; k + 224 < n; k += 256) {                 // eight independent 256-byte row segments in flight per warp
                double a[8];
#pragma unroll
                for (int q = 0; q < 8; q++) a[q] = __ldcg(Ar + k + 32 * q);
#pragma unroll
                for (int q = 0; q < 8; q++) {
                    const int kk = k + 32 * q;
                    if (q > 0 || kk >= jn + 1) {            // only the first segment can straddle the pivot column
                        const double v = fma(-wi, u[kk], fma(-ui, wv[kk], a[q]));
                        __stcg(Ar + kk, v);
                        if (q & 1) acc1 = fma(v, un[kk], acc1); else acc0 = fma(v, un[kk], acc0);
                        if (pub) __stcg(rw + kk, v);
                    }
                }
            }
            for (; k < n; k += 32) {
                if (k >= jn + 1) {
                    double a0 = __ldcg(Ar + k);
                    a0 = fma(-wi, u[k], fma(-ui, wv[k], a0));
                    __stcg(Ar + k, a0);
                    acc0 = fma(a0, un[k], acc0);
                    if (pub) __stcg(rw + k, a0);
                }
            }
            const double p = warp_sum(acc0 + acc1);
            if (lane == 0) __stcg(pw + gi, p);
        }
        epoch++;
        grid_barrier(ctrl, epoch * C);
        double* t = u; u = un; un = t;
        tau = taun;
    }
}

// ---------------------------------------------------------------------------------------------
// 2. Bisection: CTA t finds the t-th largest eigenvalue of T.  Every pass evaluates the Sturm
// count at 128 interior points of the bracket (one per thread), so a pass divides the bracket
// by 129.  The count is the number of sign changes of the leading principal minors
// p_i = (d_i - x) p_{i-1} - e_{i-1}^2 p_{i-2}: one dependent FMA per row instead of the
// reciprocal of the usual pivot recurrence.  T is scaled to unit size and the pair (p_i, p_{i-1})
// is renormalised by a power of two every four rows, so nothing overflows or dies out.
// bounds[0] = max |Gershgorin bound| (scale of T) for the later kernels.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BIS)
bisect_kernel(const double* __restrict__ d_g, const double* __restrict__ e_g, int n, int passes, double* __restrict__ lam,
              double* __restrict__ bounds) {
    extern __shared__ double sm[];
    double* d = sm;            // n, scaled
    double* e2 = sm + n;       // n, scaled (e2[n-1] = 0)
    __shared__ double scratch[32];
    __shared__ double s_lo, s_hi;
    const int tid = threadIdx.x;
    double gl = INFINITY, gu = -INFINITY;
    for (int i = tid; i < n; i += BIS) {
        const double di = d_g[i];
        const double el = i > 0 ? fabs(e_g[i - 1]) : 0.0, er = i < n - 1 ? fabs(e_g[i]) : 0.0;
        gl = fmin(gl, di - el - er);
        gu = fmax(gu, di + el + er);
    }
    gl = block_min(gl, scratch);
    if (tid == 0) s_lo = gl;
    gu = block_max(gu, scratch);
    if (tid == 0) s_hi = gu;
    __syncthreads();
    const double scale = fmax(fmax(fabs(s_lo), fabs(s_hi)), 1e-300);
    const double inv_scale = 1.0 / scale;
    for (int i = tid; i < n; i += BIS) {
        d[i] = d_g[i] * inv_scale;
        const double er = i < n - 1 ? e_g[i] * inv_scale : 0.0;
        e2[i] = er * er;
    }
    __syncthreads();
    const double pad = 2.220446049250313e-16 * n;
    double lo = s_lo * inv_scale - pad, hi = s_hi * inv_scale + pad;
    const int idx = n - 1 - (int)blockIdx.x;             // ascending index of the wanted eigenvalue
    for (int pass = 0; pass < passes; pass++) {
        const double step = (hi - lo) * (1.0 / (BIS + 1));
        const double x = fma(step, (double)(tid + 1), lo);
        double pp = 1.0, pc = d[0] - x;
        bool neg = pc < 0.0 || pc == 0.0;                // an exact zero counts as a change (pivot -> -0)
        int cnt = neg ? 1 : 0;
        for (int i = 1; i < n; i++) {
            const double pn = fma(d[i] - x, pc, -e2[i - 1] * pp);
            const bool nneg = pn < 0.0 ? true : (pn > 0.0 ? false : !neg);
            cnt += nneg != neg;
            neg = nneg;
            pp = pc;
            pc = pn;
            if ((i & 3) == 3) {
                const double mx = fmax(fabs(pp), fabs(pc));
                const int ex = (__double2hiint(mx) >> 20) & 0x7ff;
                if (ex > 0 && ex < 2046) {
                    const double f = __hiloint2double((2046 - ex) << 20, 0);   // 2^(1023 - ex)
                    pp *= f;
                    pc *= f;
                }
            }
        }
        const int L = __syncthreads_count(cnt <= idx);   // points still at or below the eigenvalue
        const double nlo = L > 0 ? fma(step, (double)L, lo) : lo;
        const double nhi = L < BIS ? fma(step, (double)(L + 1), lo) : hi;
        lo = nlo;
        hi = nhi;
    }
    if (tid == 0) {
        lam[blockIdx.x] = 0.5 * (lo + hi) * scale;
        if (blockIdx.x == 0) bounds[0] = scale;
    }
}

// ---------------------------------------------------------------------------------------------
// 3. One step of inverse iteration for shift t: x = (T - lam_t I)^-1 b, normalised.  Pivoted
// LU of the shifted tridiagonal (row interchanges as LAPACK's gttrf), b = row t of Bt or a
// fixed pseudo-random vector.  The recurrences are sequential: lane 0 runs them out of shared
// memory, the warp loads, normalises and stores.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double hash_unit(unsigned a, unsigned b) {
    unsigned h = a * 0x9E3779B1u ^ (b + 0x7F4A7C15u) * 0x85EBCA77u;
    h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12; h *= 0x297A2D39u; h ^= h >> 15;
    return ((double)(h >> 8) + 0.5) * (2.0 / 16777216.0) - 1.0;   // (-1, 1), never 0
}

__global__ void __launch_bounds__(32)
invit_kernel(const double* __restrict__ d_g, const double* __restrict__ e_g, int n, const double* __restrict__ lam,
             const double* __restrict__ bounds, const double* __restrict__ Bt, double* __restrict__ Xt,
             double* __restrict__ factors, int reuse) {
    extern __shared__ double sm[];
    double* dd = sm;               // d - mu, later the reciprocal pivots
    double* ee = dd + n;           // off-diagonal
    double* L = ee + n;            // multipliers
    double* U1 = L + n;            // first super-diagonal of U
    double* U2 = U1 + n;           // second super-diagonal of U
    double* x = U2 + n;            // right-hand side / solution
    unsigned char* piv = reinterpret_cast<unsigned char*>(x + n);
    const int lane = threadIdx.x, t = blockIdx.x;
    const double mu = lam[t];
    const double tiny = fmax(bounds[0] * 2.220446049250313e-16, 1e-290);
    // factors of shift t: L, reciprocal pivots, U1, U2 (n doubles each) then n pivot bytes (padded to 8)
    double* fac = factors + (size_t)t * (4 * (size_t)n + ((size_t)n + 7) / 8);
    for (int i = lane; i < n; i += 32) {
        if (reuse) {
            L[i] = fac[i]; dd[i] = fac[n + i]; U1[i] = fac[2 * (size_t)n + i]; U2[i] = fac[3 * (size_t)n + i];
            piv[i] = reinterpret_cast<const unsigned char*>(fac + 4 * (size_t)n)[i];
        } else {
            dd[i] = d_g[i] - mu;
            ee[i] = i < n - 1 ? e_g[i] : 0.0;
        }
        x[i] = Bt ? Bt[(size_t)t * n + i] : hash_unit((unsigned)t, (unsigned)i);
    }
    __syncwarp();
    if (lane == 0 && !reuse) {
        double dcur = dd[0], ucur = ee[0];
        for (int i = 0; i < n - 1; i++) {
            const double sub = ee[i], dnext = dd[i + 1], unext = ee[i + 1];   // ee[n-1] = 0
            if (fabs(dcur) >= fabs(sub) || fabs(sub) < tiny) {
                if (fabs(dcur) < tiny) dcur = dcur < 0.0 ? -tiny : tiny;
                const double inv = rcp_fast(dcur), f = sub * inv;
                L[i] = f; piv[i] = 0; dd[i] = inv; U1[i] = ucur; U2[i] = 0.0;
                dcur = fma(-f, ucur, dnext);
                ucur = unext;
            } else {
                const double inv = rcp_fast(sub), f = dcur * inv;
                L[i] = f; piv[i] = 1; dd[i] = inv; U1[i] = dnext; U2[i] = unext;
                dcur = fma(-f, dnext, ucur);
                ucur = -f * unext;
            }
        }
        if (fabs(dcur) < tiny) dcur = dcur < 0.0 ? -tiny : tiny;
        dd[n - 1] = rcp_fast(dcur);
        L[n - 1] = 0.0; U1[n - 1] = 0.0; U2[n - 1] = 0.0; piv[n - 1] = 0;
    }
    __syncwarp();
    if (!reuse) {
        for (int i = lane; i < n; i += 32) {
            fac[i] = L[i]; fac[n + i] = dd[i]; fac[2 * (size_t)n + i] = U1[i]; fac[3 * (size_t)n + i] = U2[i];
            reinterpret_cast<unsigned char*>(fac + 4 * (size_t)n)[i] = piv[i];
        }
    }
    if (lane == 0) {
        // forward substitution with the interchanges
        double cur = x[0];
        for (int i = 0; i < n - 1; i++) {
            const double nxt = x[i + 1];
            if (!piv[i]) { x[i] = cur; cur = fma(-L[i], cur, nxt); }
            else { x[i] = nxt; cur = fma(-L[i], nxt, cur); }
        }
        // back substitution
        double x1 = cur * dd[n - 1], x2 = 0.0;
        x[n - 1] = x1;
        for (int i = n - 2; i >= 0; i--) {
            double v = x[i];
            v = fma(-U1[i], x1, v);
            v = fma(-U2[i], x2, v);
            v *= dd[i];
            x[i] = v;
            x2 = x1;
            x1 = v;
        }
    }
    __syncwarp();
    double big = 0.0;
    for (int i = lane; i < n; i += 32) big = fmax(big, fabs(x[i]));
    big = warp_max(big);
    const double sc = big > 0.0 ? 1.0 / big : 1.0;       // scale first: |x| can be ~1e16 / |T|
    double ss = 0.0;
    for (int i = lane; i < n; i += 32) { const double v = x[i] * sc; ss = fma(v, v, ss); }
    ss = warp_sum(ss);
    const double nrm = ss > 0.0 ? sc / sqrt(ss) : 0.0;
    for (int i = lane; i < n; i += 32) Xt[(size_t)t * n + i] = x[i] * nrm;
}

// out[a][b] = sum_i A[a][i] B[b][i]   (A: ma x n, B: mb x n, both row-major); one CTA per row a
__global__ void __launch_bounds__(256)
rows_dot_kernel(const double* __restrict__ A, const double* __restrict__ B, int mb, int n, double* __restrict__ out) {
    extern __shared__ double sm[];
    const int a = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < n; i += 256) sm[i] = A[(size_t)a * n + i];
    __syncthreads();
    for (int b = warp; b < mb; b += 8) {
        const double* row = B + (size_t)b * n;
        double acc = 0.0;
        for (int i = lane; i < n; i += 32) acc = fma(sm[i], row[i], acc);
        acc = warp_sum(acc);
        if (lane == 0) out[(size_t)a * mb + b] = acc;
    }
}

// out[c][i] = sum_r coef(c, r) X[r][i],  coef(c, r) = Cf[c * crs + r * ccs];  m <= 128
// grid (ceil(n / 128), ceil(m / 8)), 128 threads: a thread owns one i and 8 consecutive c
__global__ void __launch_bounds__(128)
combine_rows_kernel(const double* __restrict__ Cf, int64_t crs, int64_t ccs, const double* __restrict__ X, int m, int n,
                    double* __restrict__ out) {
    __shared__ double cf[8][128];
    const int c0 = blockIdx.y * 8, i = blockIdx.x * 128 + threadIdx.x;
    for (int e = threadIdx.x; e < 8 * m; e += 128) {
        const int cc = e / m, r = e - cc * m;
        cf[cc][r] = c0 + cc < m ? Cf[(size_t)(c0 + cc) * crs + (size_t)r * ccs] : 0.0;
    }
    __syncthreads();
    if (i >= n) return;
    double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int r = 0; r < m; r++) {
        const double xv = X[(size_t)r * n + i];
#pragma unroll
        for (int cc = 0; cc < 8; cc++) acc[cc] = fma(cf[cc][r], xv, acc[cc]);
    }
#pragma unroll
    for (int cc = 0; cc < 8; cc++)
        if (c0 + cc < m) out[(size_t)(c0 + cc) * n + i] = acc[cc];
}

// S = L L^T (m <= 128, one CTA), Linv = L^-1 (lower triangular, row-major).  Left-looking by
// columns: thread r owns row r; column j needs one barrier (the pivot and the dot products of
// all rows with row j read only finished columns).  A pivot that drops below m eps of its
// original diagonal means the block lost rank numerically: counted in info[0] (the caller falls
// back to the full solver) and regularised so the kernel terminates.  The inverse is then one
// forward substitution per column, four accumulators deep.
__global__ void __launch_bounds__(128)
chol_inverse_kernel(const double* __restrict__ S, int m, double* __restrict__ Linv, int* __restrict__ info, double* __restrict__ Yg) {
    // Yg == nullptr: both m x (m + 1) matrices live in shared memory (m <= ~118).  Otherwise (m up to 128) only Lm does:
    // the series path keeps E^2 in the global scratch Yg (m x m; independent loads), the Cholesky path inverts L in place.
    extern __shared__ double sm[];
    double* Lm = sm;                         // m x (m + 1), lower triangle = L
    double* Y = Yg ? Yg : sm + (size_t)m * (m + 1);
    const int ldy = Yg ? m : m + 1;
    __shared__ int s_bad;
    __shared__ double diag0[128];
    __shared__ double s_piv;
    const int tid = threadIdx.x, ld = m + 1;
    if (tid == 0) s_bad = 0;
    double dev = 0.0;                                    // max |S - I|
    for (int e = tid; e < m * m; e += 128) {
        const int r = e / m, c = e - r * m;
        const double v = 0.5 * (S[(size_t)r * m + c] + S[(size_t)c * m + r]);
        Lm[r * ld + c] = v;
        dev = fmax(dev, fabs(v - (r == c ? 1.0 : 0.0)));
    }
    const int far = __syncthreads_or(dev > 4.0 * 2.220446049250313e-16 * m ? 1 : 0);
    if (!far) {                                          // already orthonormal to rounding: L = I
        for (int e = tid; e < m * m; e += 128) Linv[e] = (e / m == e % m) ? 1.0 : 0.0;
        return;
    }
    const int big = __syncthreads_or(dev > 1e-5 ? 1 : 0);
    if (!big) {
        // nearly orthonormal (the usual case: well separated eigenvalues): symmetric orthogonalisation by the
        // series S^-1/2 = I - E/2 + 3/8 E^2 - 5/16 E^3 + O(E^4), E = S - I, |E| <= 1e-5 -> error ~1e-20.
        // No sequential factorisation; any orthonormal basis of the span serves the Rayleigh-Ritz step.
        for (int e = tid; e < m * m; e += 128) {
            const int r = e / m, c = e - r * m;
            if (r == c) Lm[r * ld + c] -= 1.0;           // Lm = E
        }
        __syncthreads();
        for (int e = tid; e < m * m; e += 128) {          // Y = E^2
            const int r = e / m, c = e - r * m;
            double acc = 0.0;
            for (int q = 0; q < m; q++) acc = fma(Lm[r * ld + q], Lm[q * ld + c], acc);
            Y[r * ldy + c] = acc;
        }
        __syncthreads();
        for (int e = tid; e < m * m; e += 128) {          // Linv = I - E/2 + 3/8 E^2 - 5/16 E E^2
            const int r = e / m, c = e - r * m;
            double acc = 0.0;
            for (int q = 0; q < m; q++) acc = fma(Lm[r * ld + q], Y[q * ldy + c], acc);
            Linv[e] = (r == c ? 1.0 : 0.0) - 0.5 * Lm[r * ld + c] + 0.375 * Y[r * ldy + c] - 0.3125 * acc;
        }
        return;
    }
    for (int j = tid; j < m; j += 128) diag0[j] = fabs(Lm[j * ld + j]);
    __syncthreads();
    const int r = tid;
    for (int j = 0; j < m; j++) {
        // v = S[r][j] - sum_{q<j} L[r][q] L[j][q]   (row j's finished part is broadcast-read)
        double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
        if (r >= j && r < m) {
            const double* lr = Lm + r * ld;
            const double* lj = Lm + j * ld;
            int q = 0;
#pragma unroll 4
            for (; q + 3 < j; q += 4) {
                v0 = fma(lr[q], lj[q], v0);
                v1 = fma(lr[q + 1], lj[q + 1], v1);
                v2 = fma(lr[q + 2], lj[q + 2], v2);
                v3 = fma(lr[q + 3], lj[q + 3], v3);
            }
            for (; q < j; q++) v0 = fma(lr[q], lj[q], v0);
        }
        const double mine = (r >= j && r < m) ? Lm[r * ld + j] - ((v0 + v1) + (v2 + v3)) : 0.0;
        if (r == j) s_piv = mine;                         // pivot candidate
        __syncthreads();
        double piv = s_piv;
        const double floor_j = 2.220446049250313e-16 * m * diag0[j];
        if (!(piv > floor_j)) {
            if (tid == 0) s_bad++;
            piv = floor_j > 0.0 ? floor_j : 1e-300;
        }
        const double inv_root = rsqrt_fast(piv);
        if (r == j) Lm[r * ld + j] = piv * inv_root;
        else if (r > j && r < m) Lm[r * ld + j] = mine * inv_root;
        __syncthreads();
    }
    if (Yg) {
        // in place, row by row: X[i][j] = -(1 / L[i][i]) sum_{q = j}^{i - 1} L[i][q] X[q][j]; rows above i already hold X,
        // row i still holds L.  Thread j owns column j (conflict-free column reads, broadcast row reads).
        for (int i = 0; i < m; i++) {
            const double inv_ii = rcp_fast(Lm[i * ld + i]);
            double x = 0.0;
            if (tid < i) {
                double a0 = 0.0, a1 = 0.0;
                const double* li = Lm + i * ld;
                int q = tid;
                for (; q + 1 < i; q += 2) {
                    a0 = fma(li[q], Lm[q * ld + tid], a0);
                    a1 = fma(li[q + 1], Lm[(q + 1) * ld + tid], a1);
                }
                if (q < i) a0 = fma(li[q], Lm[q * ld + tid], a0);
                x = -(a0 + a1) * inv_ii;
            } else if (tid == i) {
                x = inv_ii;
            }
            __syncthreads();
            if (tid <= i) Lm[i * ld + tid] = x;
            __syncthreads();
        }
        for (int e = tid; e < m * m; e += 128) {
            const int rr = e / m, c = e - rr * m;
            Linv[e] = c <= rr ? Lm[rr * ld + c] : 0.0;
        }
        if (tid == 0) atomicAdd(info, s_bad);
        return;
    }
    // column c of Y = L^-1 e_c by forward substitution, one thread per column
    if (tid < m) {
        const int c = tid;
        for (int rr = 0; rr < m; rr++) {
            if (rr < c) { Y[rr * ld + c] = 0.0; continue; }
            double a0 = rr == c ? 1.0 : 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
            const double* lr = Lm + rr * ld;
            int q = c;
#pragma unroll 4
            for (; q + 3 < rr; q += 4) {
                a0 = fma(-lr[q], Y[q * ld + c], a0);
                a1 = fma(-lr[q + 1], Y[(q + 1) * ld + c], a1);
                a2 = fma(-lr[q + 2], Y[(q + 2) * ld + c], a2);
                a3 = fma(-lr[q + 3], Y[(q + 3) * ld + c], a3);
            }
            for (; q < rr; q++) a0 = fma(-lr[q], Y[q * ld + c], a0);
            Y[rr * ld + c] = ((a0 + a1) + (a2 + a3)) * rcp_fast(lr[rr]);
        }
    }
    __syncthreads();
    for (int e = tid; e < m * m; e += 128) {
        const int rr = e / m, c = e - rr * m;
        Linv[e] = Y[rr * ld + c];
    }
    if (tid == 0) atomicAdd(info, s_bad);
}

// Y[t][i] = (T X[t])_i
__global__ void __launch_bounds__(256)
tridiag_apply_kernel(const double* __restrict__ d, const double* __restrict__ e, const double* __restrict__ X, int m, int n,
                     double* __restrict__ Y) {
    const int64_t total = (int64_t)m * n;
    for (int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * 256) {
        const int i = (int)(idx % n);
        double v = d[i] * X[idx];
        if (i > 0) v = fma(e[i - 1], X[idx - 1], v);
        if (i < n - 1) v = fma(e[i], X[idx + 1], v);
        Y[idx] = v;
    }
}

// Rayleigh-Ritz block already diagonal (every off-diagonal entry <= tol x the largest diagonal entry)?  Then the
// eigenvalues are the sorted diagonal and the eigenvectors a permutation: written here, flag[0] = 1.  One CTA.
// (The n <= 64 solver has this test built in; this is for blocks of 65 .. 128 Ritz vectors, where the general solver
// costs 1.6 ms.)
__global__ void __launch_bounds__(512) rr_passthrough_kernel(const double* __restrict__ H, int m, double tol, double* __restrict__ evals,
                                                             double* __restrict__ evecs, int* __restrict__ flag) {
    __shared__ double s_off[16], s_dg[16];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double off = 0.0, dg = 0.0;
    for (int i = tid; i < m * m; i += 512) {
        const int c = i / m, r = i - c * m;
        const double v = fabs(H[i]);
        if (c == r) dg = fmax(dg, v); else off = fmax(off, v);
    }
    off = warp_max(off);
    dg = warp_max(dg);
    if (lane == 0) { s_off[warp] = off; s_dg[warp] = dg; }
    __syncthreads();
    off = 0.0; dg = 0.0;
    for (int w = 0; w < 16; w++) { off = fmax(off, s_off[w]); dg = fmax(dg, s_dg[w]); }
    const bool diagonal = off <= tol * dg;               // uniform over the CTA
    if (tid == 0) flag[0] = diagonal ? 1 : 0;
    if (!diagonal) return;
    for (int c = warp; c < m; c += 16) {
        const double mine = H[(size_t)c * m + c];
        int cnt = 0;
        for (int k = lane; k < m; k += 32) {
            const double o = H[(size_t)k * m + k];
            cnt += (o > mine || (o == mine && k < c)) ? 1 : 0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        if (lane == 0) evals[cnt] = mine;
        for (int i = lane; i < m; i += 32) evecs[(size_t)i * m + cnt] = i == c ? 1.0 : 0.0;
    }
}

__global__ void __launch_bounds__(256) symmetrise_kernel(double* H, int m) {
    for (int e = blockIdx.x * 256 + threadIdx.x; e < m * m; e += gridDim.x * 256) {
        const int r = e / m, c = e - r * m;
        if (c > r) {
            const double v = 0.5 * (H[e] + H[(size_t)c * m + r]);
            H[e] = v;
            H[(size_t)c * m + r] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// 5. Back-transformation, n <= 1024: one warp (one CTA) per Ritz vector, TWO reflectors per dependent
// reduction.  With d = v_j.z, e = v_{j-1}.z and g = v_{j-1}.v_j (three dot products of one pass, reduced by
// interleaved butterflies),  H_{j-1} H_j z = z - tau_j d v_j - tau_{j-1} (e - tau_j d g) v_{j-1}:
// (n - 2) / 2 reduction latencies instead of n - 2 (the one-reflector form took about twice as long).  The reflector rows arrive through a cp.async ring of
// PAIRS_AHEAD pairs in shared memory (only the 16-byte chunks right of the zero part), so the L2 latency of a row
// is paid PAIRS_AHEAD pairs before it is used.  U[i * ldu + t] = z_i.
// ---------------------------------------------------------------------------------------------
constexpr int PAIRS_AHEAD = 4;

__device__ __forceinline__ void bt_cp_async16(void* smem, const void* gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem));
}

template <int NE>
__global__ void __launch_bounds__(32)
backtransform_pair_kernel(const double* __restrict__ V, int ldv, const double* __restrict__ tau_g, int n,
                          const double* __restrict__ Zt, double* __restrict__ U, int64_t ldu) {
    extern __shared__ __align__(16) double bt_ring[];    // [PAIRS_AHEAD][2][32 * NE], then tau[32 * NE]
    constexpr int NV = 32 * NE;
    double* tau_s = bt_ring + PAIRS_AHEAD * 2 * NV;
    const int lane = threadIdx.x, t = blockIdx.x;
    double z[NE];
#pragma unroll
    for (int q = 0; q < NE; q++) {
        const int k = lane + 32 * q;
        z[q] = k < n ? Zt[(size_t)t * n + k] : 0.0;
    }
    for (int c = lane; c < PAIRS_AHEAD * 2 * NV; c += 32) bt_ring[c] = 0.0;
    for (int c = lane; c < NV; c += 32) tau_s[c] = c < n - 2 ? tau_g[c] : 0.0;   // a global load per pair would sit in the dependent chain
    __syncwarp();
    const int pairs = (n - 1) / 2;                       // reflectors n-3 .. 0, the last pair may be single
    const int chunks = (n + 1) / 2;                      // 16-byte chunks of a row (ldv is even, rows start 16-byte aligned)
    auto issue = [&](int p) {
        if (p < pairs) {
            const int ja = n - 3 - 2 * p, jb = ja - 1;
            double* slot = bt_ring + (size_t)(p % PAIRS_AHEAD) * 2 * NV;
            const int c0 = (jb < 0 ? ja : jb) / 2;       // both rows are zero left of column jb + 1 >= 2 c0
            for (int c = c0 + lane; c < chunks; c += 32) {
                bt_cp_async16(slot + 2 * c, V + (size_t)ja * ldv + 2 * c);
                if (jb >= 0) bt_cp_async16(slot + NV + 2 * c, V + (size_t)jb * ldv + 2 * c);
            }
        }
        asm volatile("cp.async.commit_group;\n" ::);
    };
    for (int p = 0; p < PAIRS_AHEAD - 1; p++) issue(p);
    for (int p = 0; p < pairs; p++) {
        issue(p + PAIRS_AHEAD - 1);
        asm volatile("cp.async.wait_group %0;\n" ::"n"(PAIRS_AHEAD - 1));
        __syncwarp();
        const int ja = n - 3 - 2 * p, jb = ja - 1;
        const double* va = bt_ring + (size_t)(p % PAIRS_AHEAD) * 2 * NV;
        const double* vb = va + NV;
        const double ta = tau_s[ja], tb = jb >= 0 ? tau_s[jb] : 0.0;
        // no predicates: left of the copied chunks the ring still holds its initial zeros, the copied chunks hold the
        // rows' own zeros up to the unit element, and an odd n reads the (zero) first element of the next row
        double a[NE], b[NE];
        double d0 = 0.0, d1 = 0.0, e0 = 0.0, e1 = 0.0, g0 = 0.0, g1 = 0.0;
#pragma unroll
        for (int q = 0; q < NE; q++) {
            a[q] = va[lane + 32 * q];
            b[q] = vb[lane + 32 * q];
        }
#pragma unroll
        for (int q = 0; q < NE; q++) {
            if (q & 1) { d1 = fma(a[q], z[q], d1); e1 = fma(b[q], z[q], e1); g1 = fma(a[q], b[q], g1); }
            else { d0 = fma(a[q], z[q], d0); e0 = fma(b[q], z[q], e0); g0 = fma(a[q], b[q], g0); }
        }
        double d = d0 + d1, e = e0 + e1, g = g0 + g1;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            d += __shfl_xor_sync(0xffffffffu, d, o);
            e += __shfl_xor_sync(0xffffffffu, e, o);
            g += __shfl_xor_sync(0xffffffffu, g, o);
        }
        const double ca = ta * d;
        const double cb = tb * fma(-ca, g, e);
#pragma unroll
        for (int q = 0; q < NE; q++) z[q] = fma(-cb, b[q], fma(-ca, a[q], z[q]));
        __syncwarp();                                    // the slot is refilled PAIRS_AHEAD - 1 pairs from now
    }
#pragma unroll
    for (int q = 0; q < NE; q++) {
        const int k = lane + 32 * q;
        if (k < n) U[(size_t)k * ldu + t] = z[q];
    }
}

// Back-transformation for n > 1024: one CTA per Ritz vector, KMAX_BIG elements per thread.
__global__ void __launch_bounds__(TDT)
backtransform_big_kernel(const double* __restrict__ V, int ldv, const double* __restrict__ tau_g, int n, const double* __restrict__ Zt,
                         double* __restrict__ U, int64_t ldu) {
    __shared__ double red[2][TDT / 32];
    const int tid = threadIdx.x, t = blockIdx.x;
    double z[KMAX_BIG];
#pragma unroll
    for (int m = 0; m < KMAX_BIG; m++) {
        const int k = tid + m * TDT;
        z[m] = k < n ? Zt[(size_t)t * n + k] : 0.0;
    }
    for (int j = n - 3; j >= 0; j--) {
        const double tau = tau_g[j];
        if (tau == 0.0) continue;                        // uniform
        const double* v = V + (size_t)j * ldv;
        double vv[KMAX_BIG];
        double dot = 0.0;
#pragma unroll
        for (int m = 0; m < KMAX_BIG; m++) {
            const int k = tid + m * TDT;
            vv[m] = (k > j && k < n) ? __ldg(v + k) : 0.0;
            dot = fma(vv[m], z[m], dot);
        }
        dot = block_sum_all(dot, red[j & 1]) * tau;
#pragma unroll
        for (int m = 0; m < KMAX_BIG; m++) z[m] = fma(-dot, vv[m], z[m]);
    }
#pragma unroll
    for (int m = 0; m < KMAX_BIG; m++) {
        const int k = tid + m * TDT;
        if (k < n) U[(size_t)k * ldu + t] = z[m];
    }
}

// res[t] = | T z_t - theta_t z_t |  for the Ritz pairs (rows of Z): the one check that does not depend on
// how the vectors were obtained
__global__ void __launch_bounds__(128)
ritz_residual_kernel(const double* __restrict__ d, const double* __restrict__ e, const double* __restrict__ Z, const double* __restrict__ theta,
                     int n, double* __restrict__ res) {
    __shared__ double scratch[32];
    const int t = blockIdx.x;
    const double* z = Z + (size_t)t * n;
    const double th = theta[t];
    double acc = 0.0;
    for (int i = threadIdx.x; i < n; i += 128) {
        double v = (d[i] - th) * z[i];
        if (i > 0) v = fma(e[i - 1], z[i - 1], v);
        if (i < n - 1) v = fma(e[i], z[i + 1], v);
        acc = fma(v, v, acc);
    }
    acc = block_sum(acc, scratch);
    if (threadIdx.x == 0) res[t] = sqrt(acc);
}

// out[0..k-1] = Ritz values (descending), out[k] = trace(G), out[k+1] = health: rank-loss count of the
// Cholesky-QR steps + 1e3 if a Ritz residual exceeds 1e-11 |T| + 1e6 if the Rayleigh-Ritz solve did not
// converge (0 when healthy; the caller falls back to the full solver otherwise)
__global__ void __launch_bounds__(256)
finish_kernel(const double* __restrict__ G, int n, const double* __restrict__ hev, int k, const int* __restrict__ info,
              const int* __restrict__ rr_info, const double* __restrict__ res, const double* __restrict__ bounds,
              double* __restrict__ out) {
    __shared__ double scratch[32];
    double tr = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) tr += G[(size_t)i * n + i];
    tr = block_sum(tr, scratch);
    for (int i = threadIdx.x; i < k; i += 256) out[i] = hev[i];
    if (threadIdx.x == 0) {
        double worst = 0.0;                               // largest Ritz residual relative to the scale of T
        for (int i = 0; i < k; i++) worst = fmax(worst, res[i]);
        const bool bad_res = !(worst <= 1e-11 * bounds[0]);
        out[k] = tr;
        out[k + 1] = (double)info[0] + ((rr_info && rr_info[0] < 0) ? 1e6 : 0.0) + (bad_res ? 1e3 : 0.0);
    }
}

// two m x (m + 1) float64 matrices in shared memory while they fit; beyond that one, with a global scratch (chol_inverse_kernel)
static inline bool chol_two_buffers(const ndmps_ctx* ctx, int m) { return (size_t)2 * m * (m + 1) * sizeof(double) + 4096 <= ctx->smem_optin; }

static int orthonormalise(ndmps_ctx* ctx, const double* Xin, int m, int n, double* S, double* Linv, int* info, double* Xout, double* Yg) {
    rows_dot_kernel<<<m, 256, (size_t)n * sizeof(double), ctx->stream>>>(Xin, Xin, m, n, S);
    NDMPS_LAUNCH_CHECK(ctx);
    const bool two = chol_two_buffers(ctx, m);
    chol_inverse_kernel<<<1, 128, (size_t)(two ? 2 : 1) * m * (m + 1) * sizeof(double), ctx->stream>>>(S, m, Linv, info, two ? nullptr : Yg);
    NDMPS_LAUNCH_CHECK(ctx);
    combine_rows_kernel<<<dim3((unsigned)((n + 127) / 128), (unsigned)((m + 7) / 8)), 128, 0, ctx->stream>>>(Linv, m, 1, Xin, m, n, Xout);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

}  // namespace topk

// Leading k eigenpairs of the symmetric positive semi-definite G (n x n, float64, device; not
// modified).  out_dev: k + 2 doubles (see finish_kernel); U: eigenvector t in column t, leading
// dimension ldu >= k.  *done = false (nothing computed) when the shape is outside what this
// path supports.
int eigh_topk(ndmps_ctx* ctx, const double* G, int64_t n64, int64_t k64, double* out_dev, double* U, int64_t ldu, bool* done) {
    using namespace topk;
    *done = false;
    if (n64 < 96 || n64 > NMAX || k64 < 1 || k64 > 128 || 2 * k64 > n64) return NDMPS_OK;
    const int n = (int)n64, m = (int)k64;
    // 1024 < n <= 1536: still register-resident, 11 warps x one row per CTA, if that many CTAs fit the device
    const bool mid = n > 1024 && n <= 1536 && (n + MID_NT / 32 - 1) / (MID_NT / 32) <= ctx->sm_count;
    const bool big = n > 1024 && !mid;
    // register route: RPW rows per warp.  Two rows per warp up to n = 512 (the row pair still fits the register
    // file) halve the SMs a reduction sits on, which is what the other volumes in flight need
    const int rpw = n <= 512 ? 2 : 1;
    const int C = big ? ctx->sm_count : (mid ? (n + MID_NT / 32 - 1) / (MID_NT / 32) : (n + rpw * (TDT / 32) - 1) / (rpw * (TDT / 32)));
    const size_t smem_iv = (size_t)6 * n * sizeof(double) + (size_t)n + 16;
    const size_t smem_ch = (size_t)(chol_two_buffers(ctx, m) ? 2 : 1) * m * (m + 1) * sizeof(double);
    if (smem_ch + 2048 > ctx->smem_optin) return NDMPS_OK;
    {   // fixed ceilings, set once per device: contexts on several host threads share these function attributes
        const int ceiling = (int)ctx->smem_optin - 2048;
        NDMPS_TRY(raise_dynamic_smem((const void*)invit_kernel, ctx->device, ceiling));
        NDMPS_TRY(raise_dynamic_smem((const void*)chol_inverse_kernel, ctx->device, ceiling));
        if (smem_iv > (size_t)ceiling) return NDMPS_OK;
    }
    double *V, *tau, *d, *e, *pbuf, *rowbuf, *lam, *bounds, *Xa, *Xb, *S, *Linv, *TQ, *H, *hev, *W, *factors;
    unsigned* ctrl;
    int* info;
    const int ldv = (n + 1) & ~1;                        // even: 16-byte row starts for the cp.async ring
    NDMPS_TRY(ctx->ws.get<double>((size_t)n * ldv, &V));
    NDMPS_TRY(ctx->ws.get<double>((size_t)n, &tau));
    NDMPS_TRY(ctx->ws.get<double>((size_t)n, &d));
    NDMPS_TRY(ctx->ws.get<double>((size_t)n, &e));
    NDMPS_TRY(ctx->ws.get<double>((size_t)2 * n, &pbuf));
    NDMPS_TRY(ctx->ws.get<double>((size_t)2 * n, &rowbuf));
    NDMPS_TRY(ctx->ws.get<double>((size_t)m, &lam));
    NDMPS_TRY(ctx->ws.get<double>(4, &bounds));
    NDMPS_TRY(ctx->ws.get<double>((size_t)m * n, &Xa));
    NDMPS_TRY(ctx->ws.get<double>((size_t)m * n, &Xb));
    NDMPS_TRY(ctx->ws.get<double>((size_t)m * m, &S));
    NDMPS_TRY(ctx->ws.get<double>((size_t)m * m, &Linv));
    double* Yg = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)m * m, &Yg));
    NDMPS_TRY(ctx->ws.get<double>((size_t)m * n, &TQ));
    NDMPS_TRY(ctx->ws.get<double>((size_t)m * m, &H));
    NDMPS_TRY(ctx->ws.get<double>((size_t)m, &hev));
    NDMPS_TRY(ctx->ws.get<double>((size_t)m * m, &W));
    NDMPS_TRY(ctx->ws.get<double>((size_t)m * (4 * (size_t)n + ((size_t)n + 7) / 8), &factors));
    NDMPS_TRY(ctx->ws.get<unsigned>(8, &ctrl));
    info = reinterpret_cast<int*>(ctrl + 4);
    NDMPS_CUDA_TRY(cudaMemsetAsync(ctrl, 0, 8 * sizeof(unsigned), ctx->stream));

    // 1. tridiagonalise
    if (big) {
        double* Awork = nullptr;                         // the reduction overwrites its matrix; G stays intact
        NDMPS_TRY(ctx->ws.get<double>((size_t)n * n, &Awork));
        NDMPS_CUDA_TRY(cudaMemcpyAsync(Awork, G, (size_t)n * n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        const size_t smem_big = (size_t)3 * n * sizeof(double);
        NDMPS_TRY(raise_dynamic_smem((const void*)tridiag_big_kernel, ctx->device, (int)(3 * NMAX * sizeof(double))));
        NDMPS_TRY(raise_dynamic_smem((const void*)bisect_kernel, ctx->device, (int)(2 * NMAX * sizeof(double))));
        int n_arg = n, ldv_arg = ldv;
        // the fused pass is bound by L2 latency per warp: as many resident warps as fit (up to 3 CTAs per SM)
        int per_sm = 1;
        NDMPS_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tridiag_big_kernel, TDT, smem_big));
        per_sm = per_sm < 1 ? 1 : (per_sm > 3 ? 3 : per_sm);
        void* args[] = {&Awork, &n_arg, &ldv_arg, &V, &tau, &d, &e, &pbuf, &rowbuf, &ctrl};
        NDMPS_TRY(coop_launch(ctx, (const void*)tridiag_big_kernel, dim3(C * per_sm), dim3(TDT), args, smem_big));
    } else {
        int n_arg = n, ldv_arg = ldv;
        void* args[] = {(void*)&G, &n_arg, &ldv_arg, &V, &tau, &d, &e, &pbuf, &rowbuf, &ctrl};
        bool clustered = false;
        if (rpw == 2 && ctx->opt_topk_cluster) {
            // one cluster of 2^x CTAs (CTAs past the last row only take part in the barriers)
            int cc = 1;
            while (cc < C) cc *= 2;
            const void* cfn = (const void*)tridiag_kernel<16, 2, true, TDT>;
            bool fits = false;
            NDMPS_TRY(cluster_fits(cfn, ctx->device, cc, TDT, &fits));
            if (fits) {
                cudaLaunchConfig_t cfg = {};
                cfg.gridDim = dim3((unsigned)cc);
                cfg.blockDim = dim3(TDT);
                cfg.stream = ctx->stream;
                cudaLaunchAttribute at[1];
                at[0].id = cudaLaunchAttributeClusterDimension;
                at[0].val.clusterDim.x = (unsigned)cc;
                at[0].val.clusterDim.y = 1;
                at[0].val.clusterDim.z = 1;
                cfg.attrs = at;
                cfg.numAttrs = 1;
                NDMPS_CUDA_TRY(cudaLaunchKernelExC(&cfg, cfn, args));
                clustered = true;
                ctx->cluster_launches++;
            }
        }
        if (!clustered) {
            if (n > 1024) {
                NDMPS_TRY(coop_launch(ctx, (const void*)tridiag_kernel<48, 1, false, MID_NT>, dim3(C), dim3(MID_NT), args, 0));
            } else {
                void* fn = n <= 512 ? (void*)tridiag_kernel<16, 2, false, TDT> : (void*)tridiag_kernel<32, 1, false, TDT>;
                NDMPS_TRY(coop_launch(ctx, fn, dim3(C), dim3(TDT), args, 0));
            }
        }
    }
    // 2. shifts
    const int passes = 8;
    bisect_kernel<<<m, BIS, (size_t)2 * n * sizeof(double), ctx->stream>>>(d, e, n, passes, lam, bounds);
    NDMPS_LAUNCH_CHECK(ctx);
    // 3. inverse iteration (the LU factors of step 1 are reused), re-orthonormalised between steps;
    //    the last basis is orthonormalised twice
    const int iters = 2;                                 // the Ritz residuals are checked below
    const double* rhs = nullptr;
    for (int it = 0; it < iters; it++) {
        invit_kernel<<<m, 32, smem_iv, ctx->stream>>>(d, e, n, lam, bounds, rhs, Xa, factors, it > 0 ? 1 : 0);
        NDMPS_LAUNCH_CHECK(ctx);
        NDMPS_TRY(orthonormalise(ctx, Xa, m, n, S, Linv, info, Xb, Yg));
        rhs = Xb;
    }
    NDMPS_TRY(orthonormalise(ctx, Xb, m, n, S, Linv, info, Xa, Yg));       // Q = Xa
    // 4. Rayleigh-Ritz on span(Q)
    tridiag_apply_kernel<<<(unsigned)(((int64_t)m * n + 255) / 256), 256, 0, ctx->stream>>>(d, e, Xa, m, n, TQ);
    NDMPS_LAUNCH_CHECK(ctx);
    rows_dot_kernel<<<m, 256, (size_t)n * sizeof(double), ctx->stream>>>(Xa, TQ, m, n, H);
    NDMPS_LAUNCH_CHECK(ctx);
    symmetrise_kernel<<<(unsigned)((m * m + 255) / 256), 256, 0, ctx->stream>>>(H, m);
    NDMPS_LAUNCH_CHECK(ctx);
    int* rr_info = nullptr;
    // no host round trip.  Converged Ritz vectors of separated eigenvalues give a diagonal H (off-diagonals at the
    // residual level): then the block is passed through; clusters keep the Jacobi rotation.  Either way the residual
    // check below decides whether the result is used.
    if (m >= 2 && m <= 64) NDMPS_TRY(eigh_small_async(ctx, H, m, hev, W, 1e-16f, &rr_info, 1e-13));
    else {                                               // one short host round trip against 1.6 ms of the general solver
        int* flag = info + 2;
        rr_passthrough_kernel<<<1, 512, 0, ctx->stream>>>(H, m, 1e-13, hev, W, flag);
        NDMPS_LAUNCH_CHECK(ctx);
        NDMPS_TRY(ensure_pinned(ctx, 64));
        NDMPS_TRY(readback(ctx, ctx->pinned, flag, sizeof(int)));
        NDMPS_CUDA_TRY(stream_wait(ctx));
        if (*reinterpret_cast<const int*>(ctx->pinned) != 1) NDMPS_TRY(eigh(ctx, H, m, hev, W, 0.0));
    }
    // Zt[c] = sum_r W[r][c] Q[r]
    combine_rows_kernel<<<dim3((unsigned)((n + 127) / 128), (unsigned)((m + 7) / 8)), 128, 0, ctx->stream>>>(W, 1, m, Xa, m, n, Xb);
    NDMPS_LAUNCH_CHECK(ctx);
    double* res = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)m, &res));
    ritz_residual_kernel<<<m, 128, 0, ctx->stream>>>(d, e, Xb, hev, n, res);
    NDMPS_LAUNCH_CHECK(ctx);
    // 5. back-transform
    if (n <= 1024) {
        const size_t ring = (size_t)(PAIRS_AHEAD * 2 + 1) * (n <= 512 ? 512 : 1024) * sizeof(double);
        if (n <= 512) {
            NDMPS_TRY(raise_dynamic_smem((const void*)backtransform_pair_kernel<16>, ctx->device, (int)ring));
            backtransform_pair_kernel<16><<<(unsigned)m, 32, ring, ctx->stream>>>(V, ldv, tau, n, Xb, U, ldu);
        } else {
            NDMPS_TRY(raise_dynamic_smem((const void*)backtransform_pair_kernel<32>, ctx->device, (int)ring));
            backtransform_pair_kernel<32><<<(unsigned)m, 32, ring, ctx->stream>>>(V, ldv, tau, n, Xb, U, ldu);
        }
    } else backtransform_big_kernel<<<m, TDT, 0, ctx->stream>>>(V, ldv, tau, n, Xb, U, ldu);
    NDMPS_LAUNCH_CHECK(ctx);
    finish_kernel<<<1, 256, 0, ctx->stream>>>(G, n, hev, m, info, rr_info, res, bounds, out_dev);
    NDMPS_LAUNCH_CHECK(ctx);
    if (ctx->opt_verbose) fprintf(stderr, "[ndmps] eigh_topk n = %d, k = %d: %d CTAs\n", n, m, C);
    ctx->eig_calls++;
    ctx->eig_flops += 2.0 * n * (double)n * n + 4.0 * (double)n * n * m;   // full-matrix rank-2 updates + products; back-transformation
    *done = true;
    return NDMPS_OK;
}

}  // namespace ndmps

using namespace ndmps;

extern "C" {

int ndmps_eigh_topk(ndmps_ctx_t* ctx, const double* a_dev, int64_t n, int64_t k, double* evals_dev, double* evecs_dev) {
    NDMPS_REQUIRE(ctx && a_dev && evals_dev && evecs_dev, "ndmps_eigh_topk: NULL argument");
    NDMPS_REQUIRE(n >= 1 && k >= 1 && k <= n, "ndmps_eigh_topk: need 1 <= k <= n");
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    bool done = false;
    NDMPS_TRY(eigh_topk(ctx, a_dev, n, k, evals_dev, evecs_dev, k, &done));
    if (!done) {
        set_error("ndmps_eigh_topk: shape n = %lld, k = %lld is outside the leading-eigenpair path (96 <= n <= 4096, 2k <= n, k <= 128)",
                  (long long)n, (long long)k);
        return NDMPS_ERR_INVALID;
    }
    return NDMPS_OK;
}

}  // extern "C"
