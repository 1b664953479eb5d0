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
// Projection path (ndmps_project_region): steps 1 and 2 of the region path, with T computed in row blocks of at most
// 16 MB (whole axis-0 high parts), each reduced (max / min along one axis) into the output by project_reduce_kernel
// as soon as it is written instead of being gathered into the box; the workspace holds one block at a time.
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

// max / min that propagate NaN as numpy's do (fmax / fmin drop it): a NaN on either side wins
template <int OP, class T>
__device__ __forceinline__ T proj_op(T a, T b) {
    if (OP == NDMPS_PROJ_MAX) return (a != a || a > b) ? a : b;
    return (a != a || a < b) ? a : b;
}

struct ProjectArgs {
    int n = 0;                         // axes of the block
    int ax = 0;                        // the projected one
    int store = 1;                     // 0: combine with what out holds (axis 0 projected, a block after the first)
    int64_t ext[8] = {0};
    const int64_t* tab[8] = {nullptr}; // per-axis source offsets: the element at (i_0, ..) is src[sum_a tab[a][i_a]]
    int64_t count = 0;                 // output elements: the product of ext over every axis but ax
};

// out[o] = OP over i_ax of src[sum_a tab[a][i_a]], o the C-order index over the other axes.  ax below the innermost
// axis: a thread per output element, consecutive threads along the innermost axis; ax the innermost: a warp per output
// element, lanes strided along the line and a shuffle reduction.
template <class T, int OP>
__global__ void __launch_bounds__(256)
project_reduce_kernel(const T* __restrict__ src, T* __restrict__ out, ProjectArgs pa) {
    const T ident = OP == NDMPS_PROJ_MAX ? (T)-INFINITY : (T)INFINITY;
    const int64_t* tp = nullptr;
    int64_t ne = 1;
#pragma unroll
    for (int a = 0; a < 8; a++)
        if (a == pa.ax) { tp = pa.tab[a]; ne = pa.ext[a]; }
    const bool per_warp = pa.ax == pa.n - 1;
    const int lane = threadIdx.x & 31;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t step = per_warp ? ((int64_t)gridDim.x * blockDim.x) >> 5 : (int64_t)gridDim.x * blockDim.x;
    for (int64_t o = per_warp ? gid >> 5 : gid; o < pa.count; o += step) {
        int64_t rem = o, base = 0;
#pragma unroll
        for (int a = 7; a >= 0; a--)
            if (a < pa.n && a != pa.ax) {
                const int64_t q = rem / pa.ext[a];
                base += pa.tab[a][rem - q * pa.ext[a]];
                rem = q;
            }
        T v = ident;
        if (per_warp) {
            for (int64_t j = lane; j < ne; j += 32) v = proj_op<OP>(v, src[base + tp[j]]);
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) v = proj_op<OP>(v, __shfl_xor_sync(0xffffffffu, v, d));
            if (lane != 0) continue;
        } else {
            // four independent chains keep four loads in flight; max and min are exact, so the order is free
            T v1 = ident, v2 = ident, v3 = ident;
            int64_t j = 0;
            for (; j + 4 <= ne; j += 4) {
                v = proj_op<OP>(v, src[base + tp[j]]);
                v1 = proj_op<OP>(v1, src[base + tp[j + 1]]);
                v2 = proj_op<OP>(v2, src[base + tp[j + 2]]);
                v3 = proj_op<OP>(v3, src[base + tp[j + 3]]);
            }
            for (; j < ne; j++) v = proj_op<OP>(v, src[base + tp[j]]);
            v = proj_op<OP>(proj_op<OP>(v, v1), proj_op<OP>(v2, v3));
        }
        out[o] = pa.store ? v : proj_op<OP>(out[o], v);
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

// A projection decodes its box in blocks of T = X_H W_C that stay small (in L2 once written): a block is a range of
// whole axis-0 high parts, i.e. a contiguous range of rows of X_H, and covers a contiguous range of the box's axis-0
// positions.  The block's source is addressed by rp.tabs from one more Level, `src` (the box tables of the region path
// with each axis-0 entry taken relative to its own block; for L = 1 the core offsets of rp.left[0]).  In DCT mode the
// box covers the whole last axis and every block is gathered to volume order, transformed and reduced through the
// Level `vol` (volume-order offsets in the block, the last axis starting at the caller's lo[-1]).
constexpr int64_t PROJECT_BLOCK_BYTES = int64_t(16) << 20;

struct ProjectBlock {
    int64_t row0 = 0, rows = 0;        // rows of X_H
    int64_t i0 = 0, n0 = 0;            // box positions along axis 0
};

struct ProjectPlan {
    RegionPlan rp;                     // of the box widened to the whole last axis in DCT mode
    Level src, vol;
    std::vector<ProjectBlock> blocks;
};

// lo / hi: the caller's non-empty box; block_elems: the bound on the elements of a block of T
void plan_project(const ndmps_plan* p, const int64_t* lo, const int64_t* hi, int idct, int64_t block_elems, ProjectPlan& pp) {
    const int n = p->ndim, L = p->levels;
    std::vector<int64_t> wlo(lo, lo + n), whi(hi, hi + n), nb((size_t)n);
    if (idct) { wlo[(size_t)n - 1] = 0; whi[(size_t)n - 1] = p->shape[n - 1]; }
    for (int a = 0; a < n; a++) nb[(size_t)a] = whi[(size_t)a] - wlo[(size_t)a];
    RegionPlan& rp = pp.rp;
    plan_region(p, wlo.data(), whi.data(), rp);
    // blocks: high parts of axis 0 at the split (whole lines when axis 0 is the DCT axis, and the one core for L = 1)
    std::vector<int64_t> pw, fs;
    digit_products(p, pw, fs);
    const int64_t g0 = pw[(size_t)(rp.s * n)], h_lo = wlo[0] / g0, nh = (whi[0] - 1) / g0 - h_lo + 1;
    const int64_t per_h = rp.H / nh;   // rows of X_H in one axis-0 high part
    int64_t hb = block_elems / (per_h * rp.C);
    if (hb < 1) hb = 1;
    if (L == 1 || (idct && n == 1)) hb = nh;
    for (int64_t h = 0; h < nh; h += hb) {
        ProjectBlock b;
        const int64_t h1 = h + hb < nh ? h + hb : nh;
        b.row0 = h * per_h;
        b.rows = (h1 - h) * per_h;
        const int64_t x0 = (h_lo + h) * g0 > wlo[0] ? (h_lo + h) * g0 : wlo[0], x1 = (h_lo + h1) * g0 < whi[0] ? (h_lo + h1) * g0 : whi[0];
        b.i0 = x0 - wlo[0];
        b.n0 = x1 - x0;
        pp.blocks.push_back(b);
    }
    // src: the region path's box tables, or the core offsets of a single core; axis 0 relative to its block
    const Level& from = L == 1 ? rp.left[0] : rp.box;
    pp.src = add_level(rp, n, nb.data());
    for (int a = 0; a < n; a++)
        for (int64_t i = 0; i < nb[(size_t)a]; i++) rp.tabs[(size_t)(pp.src.off[a] + i)] = rp.tabs[(size_t)(from.off[a] + i)];
    for (const ProjectBlock& b : pp.blocks)
        for (int64_t i = b.i0; i < b.i0 + b.n0; i++) rp.tabs[(size_t)(pp.src.off[0] + i)] -= b.row0 * rp.C;
    if (!idct) return;
    // vol: volume order in the block's gathered lines (extents nb, axis 0 the block's), the caller's box on the last axis
    std::vector<int64_t> ob((size_t)n);
    for (int a = 0; a < n; a++) ob[(size_t)a] = hi[a] - lo[a];
    pp.vol = add_level(rp, n, ob.data());
    int64_t stride = 1;
    for (int a = n - 1; a >= 0; a--) {
        int64_t* t = rp.tabs.data() + pp.vol.off[a];
        for (int64_t i = 0; i < ob[(size_t)a]; i++) t[i] = (a == n - 1 ? lo[a] - wlo[(size_t)a] + i : i) * stride;
        stride *= nb[(size_t)a];
    }
    if (n == 1) return;                // one block, the whole line
    for (const ProjectBlock& b : pp.blocks)
        for (int64_t i = b.i0; i < b.i0 + b.n0; i++) rp.tabs[(size_t)(pp.vol.off[0] + i)] -= b.i0 * (stride / nb[0]);
}

// site-order prefix of every kept row (rowH) and suffix of every kept column (colC) of T, and Q = Q_s, the columns of
// the full product: the flat site-order index of T[i, c] is rowH[i] * Q + colC[c]
void region_sites(const ndmps_plan* plan, const RegionPlan& rp, std::vector<int64_t>& rowH, std::vector<int64_t>& colC,
                  int64_t* Q_out) {
    // level by level: row (parent, digit) of the gathered product
    std::vector<int64_t> prev(1, 0), cur;
    for (int l = 0; l < rp.s; l++) {
        const int64_t d = plan->site_dims[l];
        cur.assign((size_t)rp.left[(size_t)l].count(), 0);
        walk(rp, rp.left[(size_t)l], [&](int64_t j, int64_t q) { cur[(size_t)j] = prev[(size_t)(q / d)] * d + q % d; });
        prev.swap(cur);
    }
    rowH = prev;
    // column (digit, child) of the gathered product
    prev.assign(1, 0);
    int64_t Q = 1;
    for (int k = plan->levels - 1; k >= rp.s; k--) {
        const int64_t mc = rp.m[(size_t)k + 1];
        cur.assign((size_t)rp.m[(size_t)k], 0);
        walk(rp, rp.right[(size_t)k], [&](int64_t j, int64_t q) { cur[(size_t)j] = (q / mc) * Q + prev[(size_t)(q % mc)]; });
        prev.swap(cur);
        Q *= plan->site_dims[k];
    }
    colC = prev;
    *Q_out = Q;
}

// a Level restricted to one block: axis 0 is the block's range of positions
Level block_level(const Level& lv, const ProjectBlock& b) {
    Level r = lv;
    r.ext[0] = b.n0;
    r.off[0] += b.i0;
    return r;
}

// the source of block b's reduction, the level the device path and ndmps_project_debug_offsets both read: src restricted
// to the block, or in DCT mode vol restricted to it - except for a 1-D box, whose one block is the whole widened line
// while vol is the caller's range of it, so vol is read as it stands
Level reduce_level(const ProjectPlan& pp, int idct, const ProjectBlock& b) {
    if (!idct) return block_level(pp.src, b);
    return pp.vol.n == 1 ? pp.vol : block_level(pp.vol, b);
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

// the left bond of every right-chain level as the gather's outer axis, a -> a * (d_k * m[k+1]), appended to rp.tabs:
// bond_off[k] (k >= s) is where level k's table starts
static std::vector<int64_t> add_bond_tables(const ndmps_plan* p, const int64_t* ranks, RegionPlan& rp) {
    std::vector<int64_t> bond_off((size_t)p->levels, 0);
    for (int k = rp.s; k < p->levels; k++) {
        bond_off[(size_t)k] = (int64_t)rp.tabs.size();
        for (int64_t a = 0; a < ranks[k - 1]; a++) rp.tabs.push_back(a * p->site_dims[k] * rp.m[(size_t)k + 1]);
    }
    return bond_off;
}

// X_H (|H| x r) and W_C (r x |C|) of a planned box (L > 1), its tables uploaded to `tabs`
static int region_chains(ndmps_ctx* ctx, const ndmps_plan* p, const void* const* cores, int dtype, const int64_t* ranks,
                         const RegionPlan& rp, const int64_t* tabs, const std::vector<int64_t>& bond_off, const void** X,
                         const void** W) {
    const int L = p->levels, n = p->ndim;
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
    int64_t rows = 0, cols = 0;
    NDMPS_TRY(left_chain(ctx, cores, dtype, rp.s, p->site_dims, ranks, gl.data(), X, &rows));
    return right_chain(ctx, cores, dtype, L, rp.s, p->site_dims, ranks, gr.data(), W, &cols);
}

static int contract_region(ndmps_ctx* ctx, const ndmps_plan* p, const void* const* cores, int dtype, const int64_t* ranks,
                           const int64_t* lo, const int64_t* hi, void* out) {
    const int L = p->levels;
    const size_t esz = dtype_size(dtype);
    RegionPlan rp;
    plan_region(p, lo, hi, rp);
    const std::vector<int64_t> bond_off = add_bond_tables(p, ranks, rp);
    int64_t* tabs = nullptr;
    NDMPS_TRY(upload_tables(ctx, rp.tabs, &tabs));
    StageScope sc(ctx, ST_CONTRACT);
    if (L == 1)   // H is the box itself, in C order
        return gather_sum(ctx, cores[0], out, dtype, level_args(rp.left[0], tabs, 1));
    const void *X = nullptr, *W = nullptr;
    NDMPS_TRY(region_chains(ctx, p, cores, dtype, ranks, rp, tabs, bond_off, &X, &W));
    void* T = nullptr;
    NDMPS_TRY(ctx->ws.alloc((size_t)(rp.H * rp.C) * esz, &T));
    NDMPS_TRY(chain_product(ctx, rp.H, rp.C, ranks[rp.s - 1], X, W, dtype, T));
    return gather_sum(ctx, T, out, dtype, level_args(rp.box, tabs, 1));
}

template <class T>
static int launch_project(ndmps_ctx* ctx, const void* src, void* out, const GatherArgs& g, int ax, int op, int store) {
    ProjectArgs pa;
    pa.n = g.n;
    pa.ax = ax;
    pa.store = store;
    pa.count = 1;
    for (int a = 0; a < g.n; a++) {
        pa.ext[a] = g.ext[a];
        pa.tab[a] = g.tab[a];
        if (a != ax) pa.count *= g.ext[a];
    }
    const int grid = ax == g.n - 1 ? warp_grid(ctx, pa.count) : warp_grid(ctx, (pa.count + 31) / 32);
    if (op == NDMPS_PROJ_MAX)
        project_reduce_kernel<T, NDMPS_PROJ_MAX><<<grid, 256, 0, ctx->stream>>>((const T*)src, (T*)out, pa);
    else
        project_reduce_kernel<T, NDMPS_PROJ_MIN><<<grid, 256, 0, ctx->stream>>>((const T*)src, (T*)out, pa);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

// op over volume axis `ax` of the box [lo, hi) into out (C order over the other axes), a block of T at a time
static int project_region(ndmps_ctx* ctx, const ndmps_plan* p, const void* const* cores, int dtype, const int64_t* ranks,
                          const int64_t* lo, const int64_t* hi, int ax, int op, int idct, void* out) {
    const int L = p->levels, n = p->ndim;
    const size_t esz = dtype_size(dtype);
    ProjectPlan pp;
    plan_project(p, lo, hi, idct, PROJECT_BLOCK_BYTES / (int64_t)esz, pp);
    const RegionPlan& rp = pp.rp;
    const std::vector<int64_t> bond_off = add_bond_tables(p, ranks, pp.rp);
    int64_t* tabs = nullptr;
    NDMPS_TRY(upload_tables(ctx, rp.tabs, &tabs));
    StageScope sc(ctx, ST_CONTRACT);
    const void *X = nullptr, *W = nullptr;
    if (L > 1) NDMPS_TRY(region_chains(ctx, p, cores, dtype, ranks, rp, tabs, bond_off, &X, &W));
    const int64_t nl = p->shape[n - 1];
    double* C = nullptr;
    if (idct) NDMPS_TRY(dct_matrix(ctx, nl, 1, &C));
    // output elements before a block's first axis-0 position (axis 0 projected: every block reduces into all of out)
    int64_t out_per_i0 = 1;
    for (int a = 1; a < n; a++)
        if (a != ax) out_per_i0 *= hi[a] - lo[a];
    const Arena::Mark mk = ctx->ws.mark();
    for (size_t k = 0; k < pp.blocks.size(); k++) {
        const ProjectBlock& b = pp.blocks[k];
        const void* S = cores[0];      // L = 1: the core is the volume in C order
        if (L > 1) {
            void* T = nullptr;
            NDMPS_TRY(ctx->ws.alloc((size_t)(b.rows * rp.C) * esz, &T));
            NDMPS_TRY(chain_product(ctx, b.rows, rp.C, ranks[rp.s - 1], (const char*)X + (size_t)(b.row0 * ranks[rp.s - 1]) * esz, W,
                                    dtype, T));
            S = T;
        }
        if (idct) {                    // whole lines to volume order, inverse DCT, then reduced through vol
            const GatherArgs g = level_args(block_level(pp.src, b), tabs, 1);
            int64_t count = 1;
            for (int a = 0; a < n; a++) count *= g.ext[a];
            void *V = nullptr, *Y = nullptr;
            NDMPS_TRY(ctx->ws.alloc((size_t)count * esz, &V));
            NDMPS_TRY(ctx->ws.alloc((size_t)count * esz, &Y));
            NDMPS_TRY(gather_sum(ctx, S, V, dtype, g));
            NDMPS_TRY(dct_lines(ctx, V, Y, count / nl, nl, dtype, C));
            S = Y;
        }
        const GatherArgs r = level_args(reduce_level(pp, idct, b), tabs, 1);
        void* o = ax == 0 ? out : (char*)out + (size_t)(b.i0 * out_per_i0) * esz;
        const int store = ax != 0 || k == 0;
        if (dtype == NDMPS_F32) NDMPS_TRY(launch_project<float>(ctx, S, o, r, ax, op, store));
        else NDMPS_TRY(launch_project<double>(ctx, S, o, r, ax, op, store));
        ctx->ws.rewind(mk);
    }
    return NDMPS_OK;
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

// the checks ndmps_project_region and its debug twin share; *empty: an empty extent on an axis other than `axis`
static int check_projection(const char* fn, const ndmps_plan* plan, const int64_t* lo, const int64_t* hi, int axis, bool* empty) {
    NDMPS_TRY(check_box(plan, lo, hi, empty));
    NDMPS_REQUIRE(axis >= 0 && axis < plan->ndim, "%s: axis %d outside 0..%d", fn, axis, plan->ndim - 1);
    NDMPS_REQUIRE(hi[axis] > lo[axis], "%s: the box is empty along the projected axis %d", fn, axis);
    return NDMPS_OK;
}

int ndmps_project_region(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* const* cores, int dtype, const int64_t* ranks,
                         const int64_t* lo, const int64_t* hi, int axis, int op, int idct_last_axis, void* out) {
    NDMPS_REQUIRE(ctx && plan && cores && lo && hi, "ndmps_project_region: NULL argument");
    NDMPS_TRY(check_mps("ndmps_project_region", plan, cores, dtype, ranks));
    NDMPS_REQUIRE(op == NDMPS_PROJ_MAX || op == NDMPS_PROJ_MIN, "ndmps_project_region: op %d is not max or min", op);
    bool empty = false;
    NDMPS_TRY(check_projection("ndmps_project_region", plan, lo, hi, axis, &empty));
    if (empty) return NDMPS_OK;
    NDMPS_REQUIRE(out, "ndmps_project_region: out is NULL");
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    return project_region(ctx, plan, cores, dtype, ranks, lo, hi, axis, op, idct_last_axis ? 1 : 0, out);
}

int ndmps_project_debug_offsets(const ndmps_plan_t* plan, const int64_t* lo, const int64_t* hi, int axis, int64_t block_elems,
                                int64_t* info_out, int64_t* offsets_out_host) {
    NDMPS_REQUIRE(plan && lo && hi && info_out, "ndmps_project_debug_offsets: NULL argument");
    NDMPS_REQUIRE(block_elems >= 1, "ndmps_project_debug_offsets: block_elems %lld", (long long)block_elems);
    bool empty = false;
    NDMPS_TRY(check_projection("ndmps_project_debug_offsets", plan, lo, hi, axis, &empty));
    info_out[0] = split_of(plan);
    info_out[1] = info_out[2] = info_out[3] = 0;
    if (empty) return NDMPS_OK;
    NDMPS_REQUIRE(offsets_out_host, "ndmps_project_debug_offsets: NULL argument");
    const int n = plan->ndim;
    ProjectPlan pp;
    plan_project(plan, lo, hi, 0, block_elems, pp);
    const RegionPlan& rp = pp.rp;
    // compact row / column of T -> site-order prefix / suffix, as ndmps_region_debug_offsets derives them
    std::vector<int64_t> rowH, colC;
    int64_t Q = 1;
    region_sites(plan, rp, rowH, colC, &Q);
    const int64_t e = hi[axis] - lo[axis];
    int64_t count = 1;
    for (int a = 0; a < n; a++)
        if (a != axis) count *= hi[a] - lo[a];
    int64_t* block_of = offsets_out_host + count * e;   // -1: read by no block, -2: by more than one
    for (int64_t i = 0; i < count * e; i++) block_of[i] = -1;
    for (size_t k = 0; k < pp.blocks.size(); k++) {
        const ProjectBlock& b = pp.blocks[k];
        const Level lv = reduce_level(pp, 0, b);
        int64_t per_i0 = 1;            // output elements and positions before the block's first axis-0 position
        for (int a = 1; a < n; a++) per_i0 *= hi[a] - lo[a];
        walk(rp, lv, [&](int64_t j, int64_t q) {
            // j: C-order index in the block -> (output element, position along axis) of the whole box
            int64_t rem = j + b.i0 * per_i0, o = 0, ostride = 1, pos = 0;
            for (int a = n - 1; a >= 0; a--) {
                const int64_t ext = hi[a] - lo[a], i = rem % ext;
                rem /= ext;
                if (a == axis) pos = i;
                else { o += i * ostride; ostride *= ext; }
            }
            const int64_t t = b.row0 * rp.C + q;   // the element of the whole T the block's element is
            offsets_out_host[o * e + pos] = plan->levels == 1 ? q : rowH[(size_t)(t / rp.C)] * Q + colC[(size_t)(t % rp.C)];
            block_of[o * e + pos] = block_of[o * e + pos] == -1 ? (int64_t)k : -2;
        });
    }
    info_out[1] = rp.H;
    info_out[2] = rp.C;
    info_out[3] = (int64_t)pp.blocks.size();
    return NDMPS_OK;
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
    RegionPlan rp;
    plan_region(plan, lo, hi, rp);
    std::vector<int64_t> rowH, colC;
    int64_t Q = 1;
    region_sites(plan, rp, rowH, colC, &Q);
    const int64_t C = rp.C;
    walk(rp, rp.box, [&](int64_t j, int64_t q) { site_offsets_out_host[j] = rowH[(size_t)(q / C)] * Q + colC[(size_t)(q % C)]; });
    info_out[1] = rp.H;
    info_out[2] = rp.C;
    return NDMPS_OK;
}

}  // extern "C"
