// Box decode and point evaluation of an MPS without reconstructing the whole tensor.
//
// Digits.  Axis a of the volume has mixed-radix digits with factors[l, a], level 0 most significant, and the site
// index at level l is the C-order ravel of the axis digits of that level.  With pw[l][a] = prod_{l' >= l} factors[l', a]
// the row of a voxel at the split s of contract_dense (sites 0..s-1) depends on axis a only through the high part
// x_a / pw[s][a], and the column (sites s..L-1) only through the low part x_a mod pw[s][a]:
//     row(x) = sum_a R_a[x_a / pw[s][a]],   col(x) = sum_a C_a[x_a mod pw[s][a]].
// For a box [lo, hi) the rows needed are the product over axes of contiguous ranges of high parts (the set H) and
// the columns the product over axes of sets of low parts (the set C: a range that wraps modulo pw[s][a] when the
// box is narrower than a block, so it is kept as a per-axis table).  |H| |C| <= 3^ndim |box|, with equality to
// |box| for slices and for block-aligned or full-axis ranges.
//
// Region path (ndmps_contract_region):
//   1. restricted chains: the left chain of contract_dense keeps, after each level's product, only the
//      (parent, digit) rows whose prefix the box touches (X_H, |H| x r); the right chain keeps only the columns
//      the box touches (W_C, r x |C|).  Each keep is one gather_sum with per-axis tables.
//   2. T = X_H W_C (|H| x |C|) through the product contract_dense uses (tcgen05 for large float32 products).
//   3. out[x] = T[iH(x), iC(x)] in volume order, one more gather_sum.
// The workspace holds T, the restricted chains and the tables - nothing of the size of the volume.
//
// Point path (ndmps_evaluate_points, ndmps_sample_points, ndmps_sample_grid): one kernel over three coordinate sources
// (integer points, a list of real coordinates, an affine grid) on the full chains X (P_s x r) and W (r x Q_s) of
// contract_dense, W transposed so that the column of a point is one contiguous bond vector; a warp works out the
// indices of 32 points (one per lane) and then runs their length-r dot products.  A real coordinate is clamped to
// [0, n - 1] per axis and contributes its floor and floor + 1 (clamped) digits, so a sample is the weighted sum of the
// dot products of its 2^ndim corners (corners of weight 0 are skipped); an integer point is its one corner, weight 1.
#include <math.h>

#include <type_traits>

#include "common.cuh"

namespace ndmps {

// ---------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------
// one warp per line of the innermost axis: the line's prefix offset is summed once, its ext[n-1] * row elements are
// written contiguously
template <class T>
__global__ void __launch_bounds__(256)
gather_sum_kernel(const T* __restrict__ src, T* __restrict__ dst, GatherArgs g, int64_t lines) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    int64_t inner = 1;
    const int64_t* tin = nullptr;
#pragma unroll
    for (int a = 0; a < NDMPS_GATHER_AXES; a++)
        if (a == g.n - 1) { inner = g.ext[a]; tin = g.tab[a]; }
    for (int64_t line = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; line < lines; line += nwarps) {
        int64_t rem = line, base = 0;
#pragma unroll
        for (int a = NDMPS_GATHER_AXES - 2; a >= 0; a--)
            if (a < g.n - 1) {
                const int64_t q = rem / g.ext[a];
                base += g.tab[a][rem - q * g.ext[a]];
                rem = q;
            }
        T* out = dst + line * inner * g.row;
        if (g.row == 1) {
            for (int64_t t = lane; t < inner; t += 32) out[t] = src[base + tin[t]];
        } else {
            const int64_t len = inner * g.row;
            for (int64_t t = lane; t < len; t += 32) {
                const int64_t i = t / g.row;
                out[t] = src[(base + tin[i]) * g.row + (t - i * g.row)];
            }
        }
    }
}

struct PointArgs {
    int n = 0;
    int idct = 0;                      // 1: the last axis holds DCT-II coefficients, evaluate the orthonormal inverse
    int64_t r = 1;                     // bond at the split
    int64_t shape[8] = {0};
    int64_t gran[8] = {0};             // pw[s][a]
    const int64_t* rtab[8] = {nullptr};   // high part -> contribution to the row of X
    const int64_t* ctab[8] = {nullptr};   // low part -> contribution to the row of W^T
};

template <class T>
__device__ __forceinline__ double bond_dot(const T* __restrict__ x, const T* __restrict__ w, int64_t r, int lane) {
    double s = 0.0;
    for (int64_t j = lane; j < r; j += 32) s = fma((double)x[j], w ? (double)w[j] : 1.0, s);
    return s;
}

// C[k, t] of the orthonormal inverse DCT-II of length n: x[t] = sum_k y[k] C[k, t],
// C[k, t] = sqrt(2/n) cos(pi (2t+1) k / (2n)), row k = 0 scaled by 1/sqrt(2); q = (2t+1) k mod 4n
__device__ __forceinline__ double idct_basis(int64_t q, int64_t k, int64_t n) {
    double c = sqrt(2.0 / (double)n) * cospi((double)q / (double)(2 * n));
    if (k == 0) c *= 0.70710678118654752440;
    return c;
}

// Coordinate sources of sample_points_kernel.  `interpolates` is false for integer points: their one corner is the point
// itself, so the kernel stages no neighbours for them (PointStage below) and walks no corners.  `warps` (a block) and
// `min_blocks` (resident blocks asked of ptxas, 0: none) follow the size of the staging record.
struct IntPoints {                     // (count x n) int64, C order; negatives count from the end
    // PointStage of 32 points per warp: 8 KB a block; the kernel fits 64 registers without asking
    static constexpr bool interpolates = false;
    static constexpr int warps = 8, min_blocks = 0;
    const int64_t* c = nullptr;
};

struct Interpolated {
    // SampleStage of 32 samples per warp: 30 KB of shared memory a block.  The kernel asks for 4 resident blocks (up to
    // 128 registers a thread): left to the shared-memory occupancy of 7 blocks, ptxas caps it at 72 registers and spills.
    static constexpr bool interpolates = true;
    static constexpr int warps = 4, min_blocks = 4;
};

// real sources: at(p, n, x) writes the n coordinates of sample p
struct CoordList : Interpolated {      // (count x n) float64, C order
    const double* c = nullptr;
    __device__ __forceinline__ void at(int64_t p, int n, double (&x)[8]) const {
#pragma unroll
        for (int a = 0; a < 8; a++) x[a] = a < n ? c[p * n + a] : 0.0;
    }
};

struct AffineGrid : Interpolated {     // sample p = C-order index (i_0, .., i_{m-1}) over shape: origin + sum_j i_j steps[j]
    int m = 0;
    int64_t shape[8] = {0};
    double origin[8] = {0};
    double steps[8][8] = {{0}};
    __device__ __forceinline__ void at(int64_t p, int n, double (&x)[8]) const {
#pragma unroll
        for (int a = 0; a < 8; a++) x[a] = origin[a];
        int64_t rem = p;
#pragma unroll
        for (int j = 7; j >= 0; j--)
            if (j < m) {
                const int64_t q = rem / shape[j];
                const double i = (double)(rem - q * shape[j]);
                rem = q;
#pragma unroll
                for (int a = 0; a < 8; a++)
                    if (a < n) x[a] = fma(i, steps[j][a], x[a]);
            }
    }
};

struct PointStage {                    // one point as its warp reads it
    int64_t row, col;                  // the corner at the floor of every axis (an integer point: the point)
    int64_t t0;                        // DCT mode: the (lower) position on the last axis
    int ok;
};

struct SampleStage : PointStage {      // an interpolated sample adds its upper neighbours
    int64_t drow[8], dcol[8];          // change of row / column when axis a moves to its upper neighbour
    double f[8];                       // weight of the upper neighbour (1 - f of the floor)
    int64_t t1;                        // DCT mode: the upper position on the last axis
};

// out[p] = the volume at src's point p: X[row, :] . Wt[col, :] at an integer point, NaN for one outside
// [-shape, shape); for a real one the multilinear interpolation, each coordinate clamped to [0, n - 1] first, NaN for a
// non-finite coordinate.  A NaN point reads no core (the host refuses such input first).  A warp takes 32 points: each
// lane works out the row and column of its own point (the integer divisions are most of a point's instructions) and,
// for a real one, those of its upper neighbours into shared memory; then the warp walks the 32 points, accumulating
// w_c * (its lanes' share of the dot product of corner c) over the corners, so one warp sum per point, and the 32
// results leave in one coalesced store.  In DCT mode the last axis holds coefficients: every coefficient k is summed
// with the basis row C[k, t] (for a real t, c(k) = (1 - f) C[k, t0] + f C[k, t1]), over the corners of the other axes.
template <class T, class Src>
__global__ void __launch_bounds__(Src::warps * 32, Src::min_blocks)
sample_points_kernel(const T* __restrict__ X, const T* __restrict__ Wt, Src src, int64_t count, PointArgs pa,
                     T* __restrict__ out) {
    using Stage = std::conditional_t<Src::interpolates, SampleStage, PointStage>;
    __shared__ Stage smem[Src::warps][32];
    const int lane = threadIdx.x & 31;
    Stage* sc = smem[threadIdx.x >> 5];
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int nc = pa.n - pa.idct;     // axes that contribute a row and a column (the others: the DCT axis)
    int64_t nl = 1, gl = 1;
    const int64_t *rl = nullptr, *cl = nullptr;
#pragma unroll
    for (int a = 0; a < 8; a++)
        if (a == pa.n - 1) { nl = pa.shape[a]; gl = pa.gran[a]; rl = pa.rtab[a]; cl = pa.ctab[a]; }
    for (int64_t first = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32; first < count; first += nwarps * 32) {
        const int64_t p = first + lane;
        Stage& s = sc[lane];
        int ok = p < count;
        if (ok) {
            int64_t row = 0, col = 0;
            if constexpr (Src::interpolates) {
                double x[8];
                src.at(p, pa.n, x);
#pragma unroll
                for (int a = 0; a < 8; a++) {
                    if (a >= pa.n) continue;
                    if (!isfinite(x[a])) ok = 0;     // clamped below like any other value, so every table read stays in bounds
                    const double v = fmin(fmax(x[a], 0.0), (double)(pa.shape[a] - 1));
                    const double fl = floor(v);
                    const int64_t i0 = (int64_t)fl, i1 = i0 + 1 < pa.shape[a] ? i0 + 1 : i0;
                    s.f[a] = v - fl;
                    if (a >= nc) {
                        s.t0 = i0;
                        s.t1 = i1;
                    } else {
                        const int64_t r0 = pa.rtab[a][i0 / pa.gran[a]], c0 = pa.ctab[a][i0 % pa.gran[a]];
                        row += r0;
                        col += c0;
                        s.drow[a] = pa.rtab[a][i1 / pa.gran[a]] - r0;
                        s.dcol[a] = pa.ctab[a][i1 % pa.gran[a]] - c0;
                    }
                }
            } else {
#pragma unroll
                for (int a = 0; a < 8; a++) {
                    if (a >= pa.n) break;
                    int64_t x = src.c[p * pa.n + a];
                    if (x < 0) x += pa.shape[a];
                    if (x < 0 || x >= pa.shape[a]) { ok = 0; x = 0; }   // x = 0 keeps the table reads in bounds
                    if (a >= nc) { s.t0 = x; continue; }
                    row += pa.rtab[a][x / pa.gran[a]];
                    col += pa.ctab[a][x % pa.gran[a]];
                }
            }
            s.row = row;
            s.col = col;
        }
        s.ok = ok;
        __syncwarp();
        const int m = count - first < 32 ? (int)(count - first) : 32;
        double mine = 0.0;
        for (int j = 0; j < m; j++) {                 // uniform over the warp
            const Stage& sj = sc[j];
            if (!sj.ok) continue;
            double acc = 0.0;
            const int64_t kn = pa.idct ? nl : 1;
            double ft = 0.0;
            if constexpr (Src::interpolates) ft = pa.idct ? sj.f[pa.n - 1] : 0.0;
            // DCT mode: (2t+1) k mod 4n of both positions and the digits k / gl, k mod gl, stepped with k
            int64_t q0 = 0, q1 = 0, kh = 0, kl = 0;
            for (int64_t k = 0; k < kn; k++) {
                double ck = 1.0;
                int64_t rk = sj.row, ckol = sj.col;
                if (pa.idct) {
                    ck = idct_basis(q0, k, nl);
                    rk += rl[kh];
                    ckol += cl[kl];
                    q0 += 2 * sj.t0 + 1;
                    q0 -= q0 >= 4 * nl ? 4 * nl : 0;
                    if constexpr (Src::interpolates) {
                        if (ft != 0.0) ck = fma(ft, idct_basis(q1, k, nl) - ck, ck);
                        q1 += 2 * sj.t1 + 1;
                        q1 -= q1 >= 4 * nl ? 4 * nl : 0;
                    }
                    if (++kl == gl) { kl = 0; kh++; }
                }
                for (int c = 0; c < (Src::interpolates ? 1 << nc : 1); c++) {
                    double w = ck;
                    int64_t rc = rk, cc = ckol;
                    if constexpr (Src::interpolates) {
#pragma unroll
                        for (int a = 0; a < 8; a++)
                            if (a < nc) {
                                if ((c >> a) & 1) { w *= sj.f[a]; rc += sj.drow[a]; cc += sj.dcol[a]; }
                                else w *= 1.0 - sj.f[a];
                            }
                        if (w == 0.0) continue;
                    }
                    acc = fma(w, bond_dot(X + rc * pa.r, Wt ? Wt + cc * pa.r : nullptr, pa.r, lane), acc);
                }
            }
            acc = warp_sum(acc);
            if (lane == j) mine = acc;
        }
        if (p < count) out[p] = ok ? (T)mine : (T)NAN;
        __syncwarp();                                 // sc is rewritten by the next round
    }
}

static int warp_grid(const ndmps_ctx* ctx, int64_t warps, int warps_per_block = 8) {
    int64_t want = (warps + warps_per_block - 1) / warps_per_block, cap = (int64_t)ctx->sm_count * 16 * (8 / warps_per_block);
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

int gather_sum(ndmps_ctx* ctx, const void* src, void* dst, int dtype, const GatherArgs& g) {
    int64_t lines = 1;
    for (int a = 0; a + 1 < g.n; a++) lines *= g.ext[a];
    if (lines * g.ext[g.n - 1] == 0) return NDMPS_OK;
    const int grid = warp_grid(ctx, lines);
    if (dtype == NDMPS_F32)
        gather_sum_kernel<float><<<grid, 256, 0, ctx->stream>>>((const float*)src, (float*)dst, g, lines);
    else
        gather_sum_kernel<double><<<grid, 256, 0, ctx->stream>>>((const double*)src, (double*)dst, g, lines);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

// ---------------------------------------------------------------------------------
// host planning of a box
// ---------------------------------------------------------------------------------
namespace {

struct Level {                         // one gather: n axes, table of axis a at RegionPlan::tabs[off[a]]
    int n = 0;
    int64_t ext[8] = {0};
    int64_t off[8] = {0};
    int64_t count() const {
        int64_t c = 1;
        for (int a = 0; a < n; a++) c *= ext[a];
        return c;
    }
};

struct RegionPlan {
    int s = 1;                         // split site (1 when L = 1: the single core is the volume in C order)
    int64_t H = 0, C = 0;              // |H| rows and |C| columns of T
    std::vector<int64_t> tabs;         // every table, uploaded in one copy
    std::vector<Level> left;           // level l < s: prefix rows kept, as rows (parent, digit) of X_{l-1} core_l
    std::vector<Level> right;          // level k >= s: suffix columns kept, as columns (digit, child) of core_k W_{k+1}
    std::vector<int64_t> m;            // m[k]: columns kept at level k, m[L] = 1
    Level box;                         // box voxel -> iH |C| + iC
};

Level add_level(RegionPlan& rp, int n, const int64_t* ext) {
    Level lv;
    lv.n = n;
    for (int a = 0; a < n; a++) {
        lv.ext[a] = ext[a];
        lv.off[a] = (int64_t)rp.tabs.size();
        rp.tabs.resize(rp.tabs.size() + (size_t)ext[a]);
    }
    return lv;
}

// visit every compact index j of a level (C order) with the sum q of its table entries
template <class F>
void walk(const RegionPlan& rp, const Level& lv, F fn) {
    const int64_t total = lv.count();
    for (int64_t j = 0; j < total; j++) {
        int64_t rem = j, q = 0;
        for (int a = lv.n - 1; a >= 0; a--) {
            q += rp.tabs[(size_t)(lv.off[a] + rem % lv.ext[a])];
            rem /= lv.ext[a];
        }
        fn(j, q);
    }
}

int64_t pos_mod(int64_t v, int64_t m) { return ((v % m) + m) % m; }

// pw[l * n + a] = prod_{l' >= l} factors[l', a] (l <= L);  fs[l * n + a] = prod_{a' > a} factors[l, a']
void digit_products(const ndmps_plan* p, std::vector<int64_t>& pw, std::vector<int64_t>& fs) {
    const int n = p->ndim, L = p->levels;
    pw.assign((size_t)(L + 1) * n, 1);
    fs.assign((size_t)L * n, 1);
    for (int a = 0; a < n; a++)
        for (int l = L - 1; l >= 0; l--) pw[(size_t)(l * n + a)] = pw[(size_t)((l + 1) * n + a)] * p->factors[l * n + a];
    for (int l = 0; l < L; l++) {
        int64_t st = 1;
        for (int a = n - 1; a >= 0; a--) { fs[(size_t)(l * n + a)] = st; st *= p->factors[l * n + a]; }
    }
}

int split_of(const ndmps_plan* p) { return p->levels == 1 ? 1 : split_site(p->levels, p->site_dims); }

// tables of a non-empty box [lo, hi)
void plan_region(const ndmps_plan* p, const int64_t* lo, const int64_t* hi, RegionPlan& rp) {
    const int n = p->ndim, L = p->levels;
    std::vector<int64_t> pw, fs;
    digit_products(p, pw, fs);
    rp.s = split_of(p);
    const int s = rp.s;
    // left: level l keeps the high parts x_a / pw[l+1][a] of the box (a contiguous range per axis)
    std::vector<int64_t> plo((size_t)n, 0), pcnt((size_t)n, 1), hlo((size_t)n), cnt((size_t)n);
    rp.left.resize((size_t)s);
    for (int l = 0; l < s; l++) {
        for (int a = 0; a < n; a++) {
            const int64_t g = pw[(size_t)((l + 1) * n + a)];
            hlo[(size_t)a] = lo[a] / g;
            cnt[(size_t)a] = (hi[a] - 1) / g - hlo[(size_t)a] + 1;
        }
        Level lv = add_level(rp, n, cnt.data());
        int64_t pstride = 1;                           // compact stride of axis a in the parent level
        for (int a = n - 1; a >= 0; a--) {
            const int64_t f = p->factors[l * n + a];
            int64_t* t = rp.tabs.data() + lv.off[a];
            for (int64_t i = 0; i < cnt[(size_t)a]; i++) {
                const int64_t h = hlo[(size_t)a] + i;  // parent h / f, digit h % f
                t[i] = (h / f - plo[(size_t)a]) * pstride * p->site_dims[l] + (h % f) * fs[(size_t)(l * n + a)];
            }
            pstride *= pcnt[(size_t)a];
        }
        rp.left[(size_t)l] = lv;
        plo = hlo;
        pcnt = cnt;
    }
    rp.H = 1;
    for (int a = 0; a < n; a++) rp.H *= pcnt[(size_t)a];
    // right: level k keeps the low parts x_a mod pw[k][a]: st, st+1, ... (mod pw[k][a]), min(box, pw[k][a]) of them
    std::vector<int64_t> cst((size_t)n, 0), ce((size_t)n, 1), st((size_t)n), e((size_t)n);
    rp.m.assign((size_t)L + 1, 1);
    rp.right.resize((size_t)L);
    for (int k = L - 1; k >= s; k--) {
        for (int a = 0; a < n; a++) {
            const int64_t P = pw[(size_t)(k * n + a)], nb = hi[a] - lo[a];
            e[(size_t)a] = nb < P ? nb : P;
            st[(size_t)a] = nb >= P ? 0 : lo[a] % P;
        }
        Level lv = add_level(rp, n, e.data());
        int64_t cstride = 1;                           // compact stride of axis a in the child level
        for (int a = n - 1; a >= 0; a--) {
            const int64_t P = pw[(size_t)(k * n + a)], Pc = pw[(size_t)((k + 1) * n + a)];
            int64_t* t = rp.tabs.data() + lv.off[a];
            for (int64_t j = 0; j < e[(size_t)a]; j++) {
                const int64_t u = (st[(size_t)a] + j) % P;   // digit u / Pc, child u mod Pc
                t[j] = (u / Pc) * fs[(size_t)(k * n + a)] * rp.m[(size_t)k + 1] + pos_mod(u % Pc - cst[(size_t)a], Pc) * cstride;
            }
            cstride *= ce[(size_t)a];
        }
        rp.right[(size_t)k] = lv;
        rp.m[(size_t)k] = lv.count();
        cst = st;
        ce = e;
    }
    rp.C = rp.m[(size_t)s];
    // box: voxel x -> (x / pw[s] - hlo) in H, (x mod pw[s] - st) mod pw[s] in C
    std::vector<int64_t> nb((size_t)n);
    for (int a = 0; a < n; a++) nb[(size_t)a] = hi[a] - lo[a];
    rp.box = add_level(rp, n, nb.data());
    int64_t hstride = 1, cstride = 1;
    for (int a = n - 1; a >= 0; a--) {
        const int64_t P = pw[(size_t)(s * n + a)];
        int64_t* t = rp.tabs.data() + rp.box.off[a];
        for (int64_t i = 0; i < nb[(size_t)a]; i++) {
            const int64_t x = lo[a] + i;
            t[i] = (x / P - plo[(size_t)a]) * hstride * rp.C + pos_mod(x % P - cst[(size_t)a], P) * cstride;
        }
        hstride *= pcnt[(size_t)a];
        cstride *= ce[(size_t)a];
    }
}

int check_box(const ndmps_plan* p, const int64_t* lo, const int64_t* hi, bool* empty) {
    *empty = false;
    for (int a = 0; a < p->ndim; a++) {
        NDMPS_REQUIRE(lo[a] >= 0 && lo[a] <= hi[a] && hi[a] <= p->shape[a], "box axis %d: [%lld, %lld) is not inside [0, %lld)", a,
                      (long long)lo[a], (long long)hi[a], (long long)p->shape[a]);
        if (lo[a] == hi[a]) *empty = true;
    }
    return NDMPS_OK;
}

GatherArgs level_args(const Level& lv, const int64_t* tabs_dev, int64_t row) {
    GatherArgs g;
    g.n = lv.n;
    for (int a = 0; a < lv.n; a++) { g.ext[a] = lv.ext[a]; g.tab[a] = tabs_dev + lv.off[a]; }
    g.row = row;
    return g;
}

}  // namespace

int upload_tables(ndmps_ctx* ctx, const std::vector<int64_t>& tabs, int64_t** out) {
    NDMPS_TRY(ctx->ws.get<int64_t>(tabs.size(), out));
    // pageable source: staged before the call returns, so the host vector may go right after
    NDMPS_CUDA_TRY(cudaMemcpyAsync(*out, tabs.data(), tabs.size() * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    return NDMPS_OK;
}

int check_mps(const char* fn, const ndmps_plan* plan, const void* const* cores, int dtype, const int64_t* ranks) {
    NDMPS_REQUIRE(dtype_ok(dtype), "%s: bad dtype %d", fn, dtype);
    NDMPS_REQUIRE(plan->levels == 1 || ranks, "%s: ranks is NULL", fn);
    for (int i = 0; i < plan->levels; i++) NDMPS_REQUIRE(cores[i], "%s: core %d is NULL", fn, i);
    for (int i = 0; i + 1 < plan->levels; i++) NDMPS_REQUIRE(ranks[i] >= 1, "%s: bond %d is %lld", fn, i, (long long)ranks[i]);
    return NDMPS_OK;
}

static int contract_region(ndmps_ctx* ctx, const ndmps_plan* p, const void* const* cores, int dtype, const int64_t* ranks,
                           const int64_t* lo, const int64_t* hi, void* out) {
    const int L = p->levels, n = p->ndim;
    const size_t esz = dtype_size(dtype);
    RegionPlan rp;
    plan_region(p, lo, hi, rp);
    // the left bond of every right-chain level as the gather's outer axis: a -> a * (d_k * m[k+1])
    std::vector<int64_t> bond_off((size_t)L, 0);
    for (int k = rp.s; k < L; k++) {
        bond_off[(size_t)k] = (int64_t)rp.tabs.size();
        for (int64_t a = 0; a < ranks[k - 1]; a++) rp.tabs.push_back(a * p->site_dims[k] * rp.m[(size_t)k + 1]);
    }
    int64_t* tabs = nullptr;
    NDMPS_TRY(upload_tables(ctx, rp.tabs, &tabs));
    StageScope sc(ctx, ST_CONTRACT);
    if (L == 1)   // H is the box itself, in C order
        return gather_sum(ctx, cores[0], out, dtype, level_args(rp.left[0], tabs, 1));
    std::vector<GatherArgs> gl((size_t)rp.s), gr((size_t)L);
    for (int l = 0; l < rp.s; l++) gl[(size_t)l] = level_args(rp.left[(size_t)l], tabs, ranks[l]);
    for (int k = rp.s; k < L; k++) {
        const Level& lv = rp.right[(size_t)k];
        GatherArgs& g = gr[(size_t)k];
        g.n = n + 1;
        g.ext[0] = ranks[k - 1];
        g.tab[0] = tabs + bond_off[(size_t)k];
        for (int a = 0; a < n; a++) { g.ext[a + 1] = lv.ext[a]; g.tab[a + 1] = tabs + lv.off[a]; }
    }
    const void *X = nullptr, *W = nullptr;
    int64_t rows = 0, cols = 0;
    NDMPS_TRY(left_chain(ctx, cores, dtype, rp.s, p->site_dims, ranks, gl.data(), &X, &rows));
    NDMPS_TRY(right_chain(ctx, cores, dtype, L, rp.s, p->site_dims, ranks, gr.data(), &W, &cols));
    void* T = nullptr;
    NDMPS_TRY(ctx->ws.alloc((size_t)(rows * cols) * esz, &T));
    NDMPS_TRY(chain_product(ctx, rows, cols, ranks[rp.s - 1], X, W, dtype, T));
    return gather_sum(ctx, T, out, dtype, level_args(rp.box, tabs, 1));
}

// Set-up shared by the point and sampling paths: the per-axis row / column tables (uploaded in one copy), the full
// left chain X (P_s x r) and W^T (Q_s x r), the gather of the full right chain.  L = 1: X is the core and *Wt nullptr.
static int point_setup(ndmps_ctx* ctx, const ndmps_plan* p, const void* const* cores, int dtype, const int64_t* ranks,
                       int idct, PointArgs* pa_out, const void** X_out, const void** Wt_out) {
    const int L = p->levels, n = p->ndim;
    const size_t esz = dtype_size(dtype);
    const int s = split_of(p);
    std::vector<int64_t> pw, fs;
    digit_products(p, pw, fs);
    // per-axis tables of the row of X and the row of W^T (site-order strides of the digits of each part)
    std::vector<int64_t> tabs, roff((size_t)n), coff((size_t)n);
    for (int a = 0; a < n; a++) {
        const int64_t g = pw[(size_t)(s * n + a)];
        roff[(size_t)a] = (int64_t)tabs.size();
        for (int64_t h = 0; h < p->shape[a] / g; h++) {
            int64_t v = 0, below = 1;                  // below: prod of d_l' for l < l' < s
            for (int l = s - 1; l >= 0; l--) {
                v += (h / (pw[(size_t)((l + 1) * n + a)] / g)) % p->factors[l * n + a] * fs[(size_t)(l * n + a)] * below;
                below *= p->site_dims[l];
            }
            tabs.push_back(v);
        }
        coff[(size_t)a] = (int64_t)tabs.size();
        for (int64_t u = 0; u < g; u++) {
            int64_t v = 0, below = 1;                  // below: prod of d_l' for l' > l
            for (int l = L - 1; l >= s; l--) {
                v += (u / pw[(size_t)((l + 1) * n + a)]) % p->factors[l * n + a] * fs[(size_t)(l * n + a)] * below;
                below *= p->site_dims[l];
            }
            tabs.push_back(v);
        }
    }
    // W^T = gather of W (r x Q) with the tables q -> q, a -> a Q
    const int64_t r = L > 1 ? ranks[s - 1] : 1;
    int64_t Q = 1;
    for (int l = s; l < L; l++) Q *= p->site_dims[l];
    const size_t toff = tabs.size();
    if (L > 1) {
        for (int64_t q = 0; q < Q; q++) tabs.push_back(q);
        for (int64_t a = 0; a < r; a++) tabs.push_back(a * Q);
    }
    int64_t* tabs_dev = nullptr;
    NDMPS_TRY(upload_tables(ctx, tabs, &tabs_dev));
    const void* X = cores[0];          // L = 1: the core is the volume and W the scalar 1 (Wt = nullptr)
    void* Wt = nullptr;
    if (L > 1) {
        const void* W = nullptr;
        int64_t rows = 0, cols = 0;
        NDMPS_TRY(left_chain(ctx, cores, dtype, s, p->site_dims, ranks, nullptr, &X, &rows));
        NDMPS_TRY(right_chain(ctx, cores, dtype, L, s, p->site_dims, ranks, nullptr, &W, &cols));
        NDMPS_TRY(ctx->ws.alloc((size_t)(Q * r) * esz, &Wt));
        GatherArgs g;
        g.n = 2;
        g.ext[0] = Q;
        g.ext[1] = r;
        g.tab[0] = tabs_dev + toff;
        g.tab[1] = tabs_dev + toff + Q;
        NDMPS_TRY(gather_sum(ctx, W, Wt, dtype, g));
    }
    PointArgs& pa = *pa_out;
    pa.n = n;
    pa.idct = idct;
    pa.r = r;
    for (int a = 0; a < n; a++) {
        pa.shape[a] = p->shape[a];
        pa.gran[a] = pw[(size_t)(s * n + a)];
        pa.rtab[a] = tabs_dev + roff[(size_t)a];
        pa.ctab[a] = tabs_dev + coff[(size_t)a];
    }
    *X_out = X;
    *Wt_out = Wt;
    return NDMPS_OK;
}

template <class Src>
static int sample_points(ndmps_ctx* ctx, const ndmps_plan* p, const void* const* cores, int dtype, const int64_t* ranks,
                         const Src& src, int64_t count, int idct, void* out) {
    StageScope sc(ctx, ST_CONTRACT);
    PointArgs pa;
    const void *X = nullptr, *Wt = nullptr;
    NDMPS_TRY(point_setup(ctx, p, cores, dtype, ranks, idct, &pa, &X, &Wt));
    const int grid = warp_grid(ctx, (count + 31) / 32, Src::warps);   // a warp per 32 points
    if (dtype == NDMPS_F32)
        sample_points_kernel<float, Src><<<grid, Src::warps * 32, 0, ctx->stream>>>((const float*)X, (const float*)Wt, src, count, pa,
                                                                                  (float*)out);
    else
        sample_points_kernel<double, Src><<<grid, Src::warps * 32, 0, ctx->stream>>>((const double*)X, (const double*)Wt, src, count,
                                                                                   pa, (double*)out);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

}  // namespace ndmps

using namespace ndmps;

extern "C" {

int ndmps_contract_region(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* const* cores, int dtype, const int64_t* ranks,
                          const int64_t* lo, const int64_t* hi, void* out) {
    NDMPS_REQUIRE(ctx && plan && cores && lo && hi, "ndmps_contract_region: NULL argument");
    NDMPS_TRY(check_mps("ndmps_contract_region", plan, cores, dtype, ranks));
    bool empty = false;
    NDMPS_TRY(check_box(plan, lo, hi, &empty));
    // an empty box writes nothing, so its output may be NULL (a zero-size tensor has no storage)
    if (empty) return NDMPS_OK;
    NDMPS_REQUIRE(out, "ndmps_contract_region: out is NULL");
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    return contract_region(ctx, plan, cores, dtype, ranks, lo, hi, out);
}

int ndmps_evaluate_points(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* const* cores, int dtype, const int64_t* ranks,
                          const int64_t* coords_dev, int64_t count, int idct_last_axis, void* out_dev) {
    NDMPS_REQUIRE(ctx && plan && cores && (count == 0 || (coords_dev && out_dev)), "ndmps_evaluate_points: NULL argument");
    NDMPS_REQUIRE(count >= 0, "ndmps_evaluate_points: count %lld", (long long)count);
    NDMPS_TRY(check_mps("ndmps_evaluate_points", plan, cores, dtype, ranks));
    if (count == 0) return NDMPS_OK;
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    IntPoints src;
    src.c = coords_dev;
    return sample_points(ctx, plan, cores, dtype, ranks, src, count, idct_last_axis ? 1 : 0, out_dev);
}

int ndmps_sample_points(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* const* cores, int dtype, const int64_t* ranks,
                        const double* coords_dev, int64_t count, int idct_last_axis, void* out_dev) {
    NDMPS_REQUIRE(ctx && plan && cores && (count == 0 || (coords_dev && out_dev)), "ndmps_sample_points: NULL argument");
    NDMPS_REQUIRE(count >= 0, "ndmps_sample_points: count %lld", (long long)count);
    NDMPS_TRY(check_mps("ndmps_sample_points", plan, cores, dtype, ranks));
    if (count == 0) return NDMPS_OK;
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    CoordList src;
    src.c = coords_dev;
    return sample_points(ctx, plan, cores, dtype, ranks, src, count, idct_last_axis ? 1 : 0, out_dev);
}

int ndmps_sample_grid(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* const* cores, int dtype, const int64_t* ranks,
                      const double* origin, const double* steps, const int64_t* out_shape, int m, int idct_last_axis,
                      void* out_dev) {
    NDMPS_REQUIRE(ctx && plan && cores && origin && steps && out_shape, "ndmps_sample_grid: NULL argument");
    NDMPS_REQUIRE(m >= 1 && m <= 8, "ndmps_sample_grid: m = %d outside 1..8", m);
    NDMPS_TRY(check_mps("ndmps_sample_grid", plan, cores, dtype, ranks));
    const int n = plan->ndim;
    AffineGrid src;
    src.m = m;
    int64_t count = 1;
    for (int j = 0; j < m; j++) {
        NDMPS_REQUIRE(out_shape[j] >= 0, "ndmps_sample_grid: out_shape[%d] = %lld", j, (long long)out_shape[j]);
        src.shape[j] = out_shape[j];
        count *= out_shape[j];
    }
    for (int a = 0; a < n; a++) {
        NDMPS_REQUIRE(std::isfinite(origin[a]), "ndmps_sample_grid: origin[%d] is not finite", a);
        src.origin[a] = origin[a];
        for (int j = 0; j < m; j++) {
            NDMPS_REQUIRE(std::isfinite(steps[j * n + a]), "ndmps_sample_grid: steps[%d][%d] is not finite", j, a);
            src.steps[j][a] = steps[j * n + a];
        }
    }
    // an empty grid writes nothing, so its output may be NULL
    if (count == 0) return NDMPS_OK;
    NDMPS_REQUIRE(out_dev, "ndmps_sample_grid: out_dev is NULL");
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    return sample_points(ctx, plan, cores, dtype, ranks, src, count, idct_last_axis ? 1 : 0, out_dev);
}

int ndmps_region_debug_offsets(const ndmps_plan_t* plan, const int64_t* lo, const int64_t* hi, int64_t* info_out,
                               int64_t* site_offsets_out_host) {
    NDMPS_REQUIRE(plan && lo && hi && info_out, "ndmps_region_debug_offsets: NULL argument");
    bool empty = false;
    NDMPS_TRY(check_box(plan, lo, hi, &empty));
    info_out[0] = split_of(plan);
    info_out[1] = info_out[2] = 0;
    if (empty) return NDMPS_OK;
    NDMPS_REQUIRE(site_offsets_out_host, "ndmps_region_debug_offsets: NULL argument");
    const int L = plan->levels;
    RegionPlan rp;
    plan_region(plan, lo, hi, rp);
    // site-order prefix of every kept row, level by level: row (parent, digit) of the gathered product
    std::vector<int64_t> prev(1, 0), cur;
    for (int l = 0; l < rp.s; l++) {
        const int64_t d = plan->site_dims[l];
        cur.assign((size_t)rp.left[(size_t)l].count(), 0);
        walk(rp, rp.left[(size_t)l], [&](int64_t j, int64_t q) { cur[(size_t)j] = prev[(size_t)(q / d)] * d + q % d; });
        prev.swap(cur);
    }
    const std::vector<int64_t> rowH = prev;
    // site-order suffix of every kept column: column (digit, child) of the gathered product
    prev.assign(1, 0);
    int64_t Q = 1;
    for (int k = L - 1; k >= rp.s; k--) {
        const int64_t mc = rp.m[(size_t)k + 1];
        cur.assign((size_t)rp.m[(size_t)k], 0);
        walk(rp, rp.right[(size_t)k], [&](int64_t j, int64_t q) { cur[(size_t)j] = (q / mc) * Q + prev[(size_t)(q % mc)]; });
        prev.swap(cur);
        Q *= plan->site_dims[k];
    }
    const std::vector<int64_t>& colC = prev;
    const int64_t C = rp.C;
    walk(rp, rp.box, [&](int64_t j, int64_t q) { site_offsets_out_host[j] = rowH[(size_t)(q / C)] * Q + colC[(size_t)(q % C)]; });
    info_out[1] = rp.H;
    info_out[2] = rp.C;
    return NDMPS_OK;
}

}  // extern "C"
