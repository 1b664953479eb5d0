// Block-mean (coarse) decode of an MPS: the cores of the tensor whose voxels are the means of non-overlapping blocks
// of the volume, without the full-resolution tensor.
//
// Axis a has mixed-radix digits with factors[l, a], level 0 most significant, and site l is the C-order ravel of the
// level-l digits of every axis.  Averaging the finest k_a digits of axis a (levels l >= L - k_a) is the mean over
// blocks of b_a = prod_{l >= L - k_a} factors[l, a] voxels, and since every digit lives at exactly one site that mean
// factorises: core l becomes its mean over the averaged digits of site l, (r, d_l, r') -> (r, d'_l, r').
//
// Layout of the result (ndmps_plan_coarse, the one place that decides it): factors[l, a] -> 1 wherever the digit is
// averaged; the trailing levels in which every axis is averaged (l >= L - min_a k_a) are removed, keeping at least one.
// Their reduced cores are bond matrices M_l (float64); they fold into one right boundary vector
// v = M_{L'} ... M_{L-1} (r_{L'-1}), which the last kept core absorbs through gemm.  No N-element array is involved:
// the work is sum r d r' over the sites.
#include "common.cuh"

namespace ndmps {

// out[i, j, k] = scale * sum_t in[i, keep[j] + avg[t], k]  for a core (rl, d, rr) -> (rl, dk, rr); float64 sums
template <class Tin, class Tout>
__global__ void __launch_bounds__(256)
marginalize_site_kernel(const Tin* __restrict__ in, Tout* __restrict__ out, int64_t rl, int64_t d, int64_t dk, int64_t rr,
                        const int64_t* __restrict__ keep, const int64_t* __restrict__ avg, int64_t nb, double scale) {
    const int64_t total = rl * dk * rr, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        const int64_t k = e % rr, ij = e / rr, j = ij % dk, i = ij / dk;
        const Tin* src = in + (i * d + keep[j]) * rr + k;
        double s = 0.0;
        for (int64_t t = 0; t < nb; t++) s += (double)src[avg[t] * rr];
        out[e] = (Tout)(s * scale);
    }
}

namespace {

// the factor table of the block-mean tensor: levels kept and factors (kept levels x ndim)
void coarse_layout(const ndmps_plan* p, const int64_t* drop, int* levels_out, std::vector<int64_t>& factors) {
    const int n = p->ndim, L = p->levels;
    int64_t kmin = L;
    for (int a = 0; a < n; a++) kmin = drop[a] < kmin ? drop[a] : kmin;
    const int Lk = L - (int)kmin > 1 ? L - (int)kmin : 1;
    factors.assign((size_t)Lk * n, 1);
    for (int l = 0; l < Lk; l++)
        for (int a = 0; a < n; a++)
            if (l < L - drop[a]) factors[(size_t)(l * n + a)] = p->factors[l * n + a];
    *levels_out = Lk;
}

int check_drop(const ndmps_plan* p, const int64_t* drop, const char* who) {
    NDMPS_REQUIRE(drop, "%s: drop_levels is NULL", who);
    for (int a = 0; a < p->ndim; a++)
        NDMPS_REQUIRE(drop[a] >= 0 && drop[a] <= p->levels, "%s: drop_levels[%d] = %lld outside 0..%d", who, a,
                      (long long)drop[a], p->levels);
    return NDMPS_OK;
}

// offsets inside site l of the kept digits (C order over the kept axes: the coarse site index) and of the averaged ones
void site_offsets(const ndmps_plan* p, const int64_t* drop, int l, std::vector<int64_t>& keep, std::vector<int64_t>& avg) {
    const int n = p->ndim, L = p->levels;
    keep.assign(1, 0);
    avg.assign(1, 0);
    int64_t st = 1;
    std::vector<int64_t> fs((size_t)n);
    for (int a = n - 1; a >= 0; a--) { fs[(size_t)a] = st; st *= p->factors[l * n + a]; }
    for (int a = 0; a < n; a++) {
        std::vector<int64_t>& v = l >= L - drop[a] ? avg : keep;
        const int64_t f = p->factors[l * n + a];
        std::vector<int64_t> next;
        next.reserve(v.size() * (size_t)f);
        for (int64_t base : v)
            for (int64_t u = 0; u < f; u++) next.push_back(base + u * fs[(size_t)a]);
        v.swap(next);
    }
}

template <class Tin, class Tout>
int launch_site(ndmps_ctx* ctx, const void* in, void* out, int64_t rl, int64_t d, int64_t dk, int64_t rr, const int64_t* keep,
                const int64_t* avg, int64_t nb) {
    const int64_t total = rl * dk * rr, cap = (int64_t)ctx->sm_count * 8;
    const int64_t want = (total + 255) / 256;
    marginalize_site_kernel<Tin, Tout><<<(int)(want < cap ? want : cap), 256, 0, ctx->stream>>>(
        (const Tin*)in, (Tout*)out, rl, d, dk, rr, keep, avg, nb, 1.0 / (double)nb);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

// reduce core l into `out` (payload dtype, or float64 when to_f64)
int reduce_site(ndmps_ctx* ctx, const void* in, void* out, int dtype, bool to_f64, int64_t rl, int64_t d, int64_t dk, int64_t rr,
                const int64_t* keep, const int64_t* avg, int64_t nb) {
    if (dtype == NDMPS_F64) return launch_site<double, double>(ctx, in, out, rl, d, dk, rr, keep, avg, nb);
    if (to_f64) return launch_site<float, double>(ctx, in, out, rl, d, dk, rr, keep, avg, nb);
    return launch_site<float, float>(ctx, in, out, rl, d, dk, rr, keep, avg, nb);
}

}  // namespace

static int marginalize(ndmps_ctx* ctx, const ndmps_plan* p, const void* const* cores, int dtype, const int64_t* ranks,
                       const int64_t* drop, void* const* cores_out, const int64_t* core_cap) {
    const int L = p->levels;
    int Lk = 1;
    std::vector<int64_t> cf;
    coarse_layout(p, drop, &Lk, cf);
    const bool fold = Lk < L;                      // levels Lk..L-1 are averaged on every axis
    auto rl_of = [&](int l) -> int64_t { return l == 0 ? 1 : ranks[l - 1]; };
    auto rr_of = [&](int l) -> int64_t { return l == L - 1 ? 1 : ranks[l]; };
    // tables of every site, uploaded in one copy; output sizes checked before anything is enqueued
    std::vector<int64_t> tabs, koff((size_t)L), aoff((size_t)L), dk((size_t)L), nb((size_t)L), keep, avg;
    for (int l = 0; l < L; l++) {
        site_offsets(p, drop, l, keep, avg);
        koff[(size_t)l] = (int64_t)tabs.size();
        tabs.insert(tabs.end(), keep.begin(), keep.end());
        aoff[(size_t)l] = (int64_t)tabs.size();
        tabs.insert(tabs.end(), avg.begin(), avg.end());
        dk[(size_t)l] = (int64_t)keep.size();
        nb[(size_t)l] = (int64_t)avg.size();
    }
    for (int l = 0; l < Lk; l++) {
        const int64_t need = rl_of(l) * dk[(size_t)l] * (l == Lk - 1 ? 1 : rr_of(l));
        if (core_cap[l] < need) {
            set_error("ndmps_marginalize: core %d needs %lld elements, capacity is %lld", l, (long long)need,
                      (long long)core_cap[l]);
            return NDMPS_ERR_CAPACITY;
        }
    }
    NDMPS_TRY(ctx->ws.reset(ctx->stream));
    int64_t* tabs_dev = nullptr;
    NDMPS_TRY(upload_tables(ctx, tabs, &tabs_dev));
    StageScope sc(ctx, ST_CONTRACT);
    auto reduce = [&](int l, void* out, bool to_f64) {
        return reduce_site(ctx, cores[l], out, dtype, to_f64, rl_of(l), p->site_dims[l], dk[(size_t)l], rr_of(l),
                           tabs_dev + koff[(size_t)l], tabs_dev + aoff[(size_t)l], nb[(size_t)l]);
    };
    for (int l = 0; l < Lk - (fold ? 1 : 0); l++) NDMPS_TRY(reduce(l, cores_out[l], false));
    if (!fold) return NDMPS_OK;
    // v = M_{Lk} ... M_{L-1}, from the last core backwards (float64)
    double* v = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)rl_of(L - 1), &v));
    NDMPS_TRY(reduce(L - 1, v, true));
    for (int l = L - 2; l >= Lk; l--) {
        double *M = nullptr, *nv = nullptr;
        NDMPS_TRY(ctx->ws.get<double>((size_t)(rl_of(l) * rr_of(l)), &M));
        NDMPS_TRY(ctx->ws.get<double>((size_t)rl_of(l), &nv));
        NDMPS_TRY(reduce(l, M, true));
        NDMPS_TRY(gemm(ctx, rl_of(l), 1, rr_of(l), 1.0, M, NDMPS_F64, rr_of(l), 1, v, NDMPS_F64, 1, 1, nv, NDMPS_F64, 1));
        v = nv;
    }
    // the last kept core absorbs v: (rl d', r) . v -> (rl, d') in the payload dtype
    const int l = Lk - 1;
    const int64_t rows = rl_of(l) * dk[(size_t)l], r = rr_of(l);
    double* last = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)(rows * r), &last));
    NDMPS_TRY(reduce(l, last, true));
    return gemm(ctx, rows, 1, r, 1.0, last, NDMPS_F64, r, 1, v, NDMPS_F64, 1, 1, cores_out[l], dtype, 1);
}

}  // namespace ndmps

using namespace ndmps;

extern "C" {

int ndmps_plan_coarse(const ndmps_plan_t* plan, const int64_t* drop_levels, ndmps_plan_t** out) {
    NDMPS_REQUIRE(plan && out, "ndmps_plan_coarse: NULL argument");
    NDMPS_TRY(check_drop(plan, drop_levels, "ndmps_plan_coarse"));
    int Lk = 1;
    std::vector<int64_t> cf;
    coarse_layout(plan, drop_levels, &Lk, cf);
    int64_t shape[8];
    for (int a = 0; a < plan->ndim; a++) {
        shape[a] = 1;
        for (int l = 0; l < Lk; l++) shape[a] *= cf[(size_t)(l * plan->ndim + a)];
    }
    return ndmps_plan_create(plan->ndim, shape, Lk, cf.data(), out);
}

int ndmps_plan_layout(const ndmps_plan_t* plan, int* ndim_out, int* levels_out, int64_t* shape_out, int64_t* factors_out) {
    NDMPS_REQUIRE(plan && ndim_out && levels_out, "ndmps_plan_layout: NULL argument");
    *ndim_out = plan->ndim;
    *levels_out = plan->levels;
    if (shape_out)
        for (int a = 0; a < plan->ndim; a++) shape_out[a] = plan->shape[a];
    if (factors_out)
        for (int i = 0; i < plan->levels * plan->ndim; i++) factors_out[i] = plan->factors[i];
    return NDMPS_OK;
}

int ndmps_marginalize(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* const* cores, int dtype, const int64_t* ranks,
                      const int64_t* drop_levels, void* const* cores_out, const int64_t* core_cap) {
    NDMPS_REQUIRE(ctx && plan && cores && cores_out && core_cap, "ndmps_marginalize: NULL argument");
    NDMPS_TRY(check_mps("ndmps_marginalize", plan, cores, dtype, ranks));
    NDMPS_TRY(check_drop(plan, drop_levels, "ndmps_marginalize"));
    int Lk = 1;
    std::vector<int64_t> cf;
    coarse_layout(plan, drop_levels, &Lk, cf);
    for (int i = 0; i < Lk; i++) NDMPS_REQUIRE(cores_out[i], "ndmps_marginalize: output core %d is NULL", i);
    return marginalize(ctx, plan, cores, dtype, ranks, drop_levels, cores_out, core_cap);
}

}  // extern "C"
