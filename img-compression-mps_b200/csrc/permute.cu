// K1: N-D volume <-> interleaved MPS site order.
//
// The reference builds an int64 map (utils/core.py:6-35,129-168) and scatters /
// gathers through it (core/ndmps.py:66-71,144-148).  The map is a pure
// permutation: axis a of the volume splits into per-level digits f[l][a]
// (most significant first), and site l is the C-order fusion of the level-l
// digits of all axes.  So   dst_digits(l, a)  <->  src_digits(a, l).
//
// Here the plan stores, for each direction, the destination's digit extents (in
// C order) and the source stride of every digit.  Three kernels, chosen per shape:
//   permute_bits_kernel    every factor a power of two (256^3, 512^3, 2^k images), float32: the map permutes the BITS
//                          of the offset; two 16-byte loads, a register transposition, two 16-byte stores per thread
//   permute_tiled_kernel   every other shape that tiles: contiguous runs on both sides through shared memory
//   permute_gather_kernel  the rest: walk destination offsets (coalesced writes), gather the source
#include <algorithm>
#include <type_traits>

#include <mutex>

#include "common.cuh"

namespace ndmps {

static void push_digit(DigitList& d, uint32_t extent, int64_t stride) {
    if (extent == 1) return;
    if (d.n > 0 && d.stride[d.n - 1] == stride * (int64_t)extent &&
        (uint64_t)d.extent[d.n - 1] * extent < (1ull << 31)) {
        // previous (outer) digit is contiguous with this one in the source: fuse
        d.extent[d.n - 1] *= extent;
        d.stride[d.n - 1] = stride;
    } else {
        d.extent[d.n] = extent;
        d.stride[d.n] = stride;
        d.n++;
    }
}

static void finish(DigitList& d) {
    if (d.n == 0) { d.extent[0] = 1; d.stride[0] = 0; d.n = 1; }
    for (int i = 0; i < d.n; i++) {
        uint32_t e = d.extent[i];
        d.shift[i] = (e & (e - 1)) == 0 ? __builtin_ctz(e) : -1;
    }
}

// source offset of destination element `o`: peel destination digits from the
// innermost outwards (shared by the kernels and the host-side plan check)
template <class idx_t>
__host__ __device__ __forceinline__ int64_t digit_offset(const DigitList& dl, idx_t rem) {
    int64_t off = 0;
#pragma unroll 1
    for (int j = dl.n - 1; j > 0; j--) {
        idx_t q, d;
        if (dl.shift[j] >= 0) {
            q = rem >> dl.shift[j];
            d = rem & (idx_t)(dl.extent[j] - 1);
        } else {
            q = rem / dl.extent[j];
            d = rem - q * dl.extent[j];
        }
        off += (int64_t)d * dl.stride[j];
        rem = q;
    }
    return off + (int64_t)rem * dl.stride[0];
}

template <class T, bool SMALL>
__global__ void __launch_bounds__(256) permute_gather_kernel(const T* __restrict__ src, T* __restrict__ dst,
                                                              const DigitList dl, int64_t total, double scale,
                                                              bool do_scale) {
    using idx_t = typename std::conditional<SMALL, uint32_t, uint64_t>::type;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += stride) {
        int64_t off = digit_offset<idx_t>(dl, (idx_t)o);
        T v = src[off];
        if (do_scale) v = (T)((double)v * scale);
        dst[o] = v;
    }
}

template <class T>
__global__ void __launch_bounds__(256) copy_scale_kernel(const T* __restrict__ src, T* __restrict__ dst,
                                                          int64_t total, double scale, bool do_scale) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += stride) {
        T v = src[o];
        if (do_scale) v = (T)((double)v * scale);
        dst[o] = v;
    }
}

// ---------------------------------------------------------------------------------------------
// Tiled permutation.  Each CTA moves tiles through shared memory: it reads contiguous SOURCE runs
// (pb elements, coalesced), scatters them into the tile's destination order in shared memory
// (slot table from the plan, skewed against bank conflicts), then writes contiguous
// DESTINATION runs (pa elements, coalesced).  Index arithmetic per element is one table
// lookup; per tile a handful of divisions for the outer digits.
// ---------------------------------------------------------------------------------------------
constexpr int PERM_THREADS = 256;

__host__ __device__ __forceinline__ int skew_slot(int w) { return w + (w >> 5); }

struct TileArgs {
    int tile, pa, pb, n_outer;
    int64_t n_tiles;
    uint32_t outer_extent[NDMPS_MAX_DIGITS];
    int64_t outer_dst[NDMPS_MAX_DIGITS];
    int64_t outer_src[NDMPS_MAX_DIGITS];
    const int64_t* hi_src;
    const int64_t* hi_dst;
    const uint16_t* pos;
};

template <class T, int VEC>
__global__ void __launch_bounds__(PERM_THREADS)
permute_tiled_kernel(const T* __restrict__ src, T* __restrict__ dst, const TileArgs ta, double scale, bool do_scale) {
    extern __shared__ unsigned char perm_smem[];
    T* buf = reinterpret_cast<T*>(perm_smem);
    const int tid = threadIdx.x;
    for (int64_t tile = blockIdx.x; tile < ta.n_tiles; tile += gridDim.x) {
        int64_t rem = tile, base_dst = 0, base_src = 0;
        for (int j = ta.n_outer - 1; j >= 0; j--) {
            int64_t q = rem / ta.outer_extent[j];
            int64_t d = rem - q * ta.outer_extent[j];
            base_dst += d * ta.outer_dst[j];
            base_src += d * ta.outer_src[j];
            rem = q;
        }
        // ---- source runs -> shared memory (destination order) ----
        if (VEC == 4) {
            const int nvec = ta.tile >> 2, pbv = ta.pb >> 2;
            // four independent 16-byte loads in flight per thread before anything is stored
            for (int v0 = tid; v0 < nvec; v0 += 4 * PERM_THREADS) {
                float4 val[4];
                int rr[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int v = v0 + u * PERM_THREADS;
                    rr[u] = -1;
                    if (v < nvec) {
                        const int hi = v / pbv, lo = (v - hi * pbv) << 2;
                        val[u] = __ldcs(reinterpret_cast<const float4*>(src + base_src + ta.hi_src[hi] + lo));
                        rr[u] = hi * ta.pb + lo;
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    if (rr[u] >= 0) {
                        const ushort4 p4 = *reinterpret_cast<const ushort4*>(ta.pos + rr[u]);
                        buf[p4.x] = (T)val[u].x; buf[p4.y] = (T)val[u].y; buf[p4.z] = (T)val[u].z; buf[p4.w] = (T)val[u].w;
                    }
                }
            }
        } else {
            for (int r = tid; r < ta.tile; r += PERM_THREADS) {
                const int hi = r / ta.pb, lo = r - hi * ta.pb;
                buf[ta.pos[r]] = src[base_src + ta.hi_src[hi] + lo];
            }
        }
        __syncthreads();
        // ---- shared memory -> destination runs ----
        if (VEC == 4) {
            const int nvec = ta.tile >> 2, pav = ta.pa >> 2;
            for (int v = tid; v < nvec; v += PERM_THREADS) {
                const int hi = v / pav, lo = (v - hi * pav) << 2;
                const int w = hi * ta.pa + lo;
                const int s = skew_slot(w);                 // 4 consecutive slots: w % 4 == 0 keeps them inside one 32-group
                float4 val = make_float4((float)buf[s], (float)buf[s + 1], (float)buf[s + 2], (float)buf[s + 3]);
                if (do_scale) { val.x *= (float)scale; val.y *= (float)scale; val.z *= (float)scale; val.w *= (float)scale; }
                __stcs(reinterpret_cast<float4*>(dst + base_dst + ta.hi_dst[hi] + lo), val);
            }
        } else {
            for (int w = tid; w < ta.tile; w += PERM_THREADS) {
                const int hi = w / ta.pa, lo = w - hi * ta.pa;
                T val = buf[skew_slot(w)];
                if (do_scale) val = (T)((double)val * scale);
                dst[base_dst + ta.hi_dst[hi] + lo] = val;
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// Register-only permutation for power-of-two shapes (256^3, 512^3, 2^k images): every factor is a power of two, so
// the voxel -> site map permutes the BITS of the element offset (a Morton-style interleave).  No shared memory, no
// tables, no barrier.  In both directions destination bit 0 is source bit 0 (the last axis' lowest digit); a thread
// owns the 8 elements spanned by destination bits {0, 1, pair}, where `pair` is the destination bit that holds source
// bit 1: it reads two 16-byte vectors (source bits {0, 1}, rows selected by destination bit 1) and writes two 16-byte
// vectors (destination bits {0, 1}, selected by `pair`) - a 2 x 2 transposition of 8-byte pairs in registers.  Lanes take
// the bits that complete the 128-byte lines on both sides, warps / unrolled steps / CTAs the following ones (alternately
// the next source and the next destination bit), so one CTA moves 8192 elements in KB-sized runs on both sides.
// ---------------------------------------------------------------------------------------------
constexpr int BITS_THREADS = 256;      // 5 lane bits + 3 warp bits
constexpr int BITS_UNROLL = 4;         // 2 bits: independent load pairs in flight per thread
constexpr int BITS_FIXED_IDX = 10;     // lane + warp + unroll index bits; the others select the CTA

struct BitArgs {
    int row_shift, pair_shift, n_cta;
    int8_t tdst[8], tsrc[8];           // thread index bits
    int8_t cdst[40], csrc[40];         // CTA index bits
    int64_t u_src[BITS_UNROLL], u_dst[BITS_UNROLL];
};

// element offsets (source, destination) of the first of the eight elements thread `tid` of CTA `block` moves in
// unrolled step 0; shared by the kernel and by the host-side walk of the plan (ndmps_plan_debug_apply_bits)
__host__ __device__ __forceinline__ void bits_offsets(const BitArgs& ba, unsigned tid, unsigned block, int64_t& so, int64_t& dofs_out) {
    int64_t s = 0, d = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const int64_t on = (tid >> k) & 1u;
        s += on << ba.tsrc[k];
        d += on << ba.tdst[k];
    }
    for (int k = 0; k < ba.n_cta; k++) {
        const int64_t on = (block >> k) & 1u;
        s += on << ba.csrc[k];
        d += on << ba.cdst[k];
    }
    so = s;
    dofs_out = d;
}

__global__ void __launch_bounds__(BITS_THREADS, 4)
permute_bits_kernel(const float* __restrict__ src, float* __restrict__ dst, const BitArgs ba, float scale, bool do_scale) {
    int64_t so, dofs;
    bits_offsets(ba, threadIdx.x, blockIdx.x, so, dofs);
    const int64_t row = int64_t(1) << ba.row_shift, pair = int64_t(1) << ba.pair_shift;
    float4 lo[BITS_UNROLL], hi[BITS_UNROLL];
#pragma unroll
    for (int u = 0; u < BITS_UNROLL; u++) {
        const float* p = src + so + ba.u_src[u];
        lo[u] = __ldcs(reinterpret_cast<const float4*>(p));
        hi[u] = __ldcs(reinterpret_cast<const float4*>(p + row));
    }
#pragma unroll
    for (int u = 0; u < BITS_UNROLL; u++) {
        float4 a = make_float4(lo[u].x, lo[u].y, hi[u].x, hi[u].y);
        float4 b = make_float4(lo[u].z, lo[u].w, hi[u].z, hi[u].w);
        if (do_scale) {
            a.x *= scale; a.y *= scale; a.z *= scale; a.w *= scale;
            b.x *= scale; b.y *= scale; b.z *= scale; b.w *= scale;
        }
        float* q = dst + dofs + ba.u_dst[u];
        __stcs(reinterpret_cast<float4*>(q), a);
        __stcs(reinterpret_cast<float4*>(q + pair), b);
    }
}

static void fill_bit_args(const BitPlan& bp, BitArgs& ba) {
    ba.row_shift = bp.row_shift;
    ba.pair_shift = bp.pair_shift;
    ba.n_cta = bp.n_idx - BITS_FIXED_IDX;
    for (int k = 0; k < 5; k++) { ba.tdst[k] = bp.dst_bit[k]; ba.tsrc[k] = bp.src_bit[k]; }
    for (int k = 0; k < 3; k++) { ba.tdst[5 + k] = bp.dst_bit[5 + k]; ba.tsrc[5 + k] = bp.src_bit[5 + k]; }
    for (int u = 0; u < BITS_UNROLL; u++) {
        ba.u_src[u] = ba.u_dst[u] = 0;
        for (int k = 0; k < 2; k++)
            if ((u >> k) & 1) {
                ba.u_src[u] += int64_t(1) << bp.src_bit[8 + k];
                ba.u_dst[u] += int64_t(1) << bp.dst_bit[8 + k];
            }
    }
    for (int k = 0; k < ba.n_cta; k++) { ba.cdst[k] = bp.dst_bit[BITS_FIXED_IDX + k]; ba.csrc[k] = bp.src_bit[BITS_FIXED_IDX + k]; }
}

// Bit form of a digit list (host).  ok = false unless every extent and stride is a power of two, the volume has at
// least 2^13 elements, and the low bits have the pattern the kernel's register transposition assumes.
static void build_bit_plan(const DigitList& dl, int64_t total, BitPlan& bp) {
    bp.ok = false;
    int sigma[64];                       // destination bit -> source bit
    int n = 0;
    for (int j = dl.n - 1; j >= 0; j--) {
        if (dl.shift[j] < 0) return;
        const int64_t st = dl.stride[j];
        if (dl.shift[j] > 0 && (st <= 0 || (st & (st - 1)) != 0)) return;
        for (int b = 0; b < dl.shift[j]; b++) {
            if (n >= 40 + 3) return;
            sigma[n++] = __builtin_ctzll((unsigned long long)st) + b;
        }
    }
    if (n < BITS_FIXED_IDX + 3 || (int64_t(1) << n) != total) return;
    int inv[64];
    for (int k = 0; k < n; k++) inv[k] = -1;
    for (int k = 0; k < n; k++) {
        if (sigma[k] < 0 || sigma[k] >= n || inv[sigma[k]] >= 0) return;     // not a permutation of the bits
        inv[sigma[k]] = k;
    }
    if (sigma[0] != 0 || sigma[1] < 2) return;
    const int pair = inv[1];
    if (pair < 2) return;
    bool used[64] = {false};
    used[0] = used[1] = used[pair] = true;
    int order[64], cnt = 0;
    // lane bits: alternately the lowest free source bit and the lowest free destination bit (128-byte lines on both
    // sides of a warp); warp and unroll bits: whichever side has the shorter contiguous run so far (source on a tie),
    // as the tile planner does - long runs on BOTH sides keep DRAM pages open
    int ps = 2, pd = 2;
    bool src_turn = true;
    while (cnt < BITS_FIXED_IDX) {
        while (ps < n && used[inv[ps]]) ps++;     // lowest source bit not covered = log2 of the source run
        while (pd < n && used[pd]) pd++;          // same on the destination side
        if (ps >= n && pd >= n) return;
        if (cnt >= 5) src_turn = ps <= pd;
        int pick = (src_turn && ps < n) || pd >= n ? inv[ps] : pd;
        used[pick] = true;
        order[cnt++] = pick;
        src_turn = !src_turn;
    }
    for (int k = 0; k < n; k++) if (!used[k]) order[cnt++] = k;               // CTA bits, ascending destination order
    if (cnt != n - 3 || cnt - BITS_FIXED_IDX > 31) return;
    bp.nbits = n;
    bp.row_shift = sigma[1];
    bp.pair_shift = pair;
    bp.n_idx = cnt;
    for (int t = 0; t < cnt; t++) { bp.dst_bit[t] = (int8_t)order[t]; bp.src_bit[t] = (int8_t)sigma[order[t]]; }
    bp.ok = true;
}

// Build the tiled form of a digit list (host).  Returns ok = false when the shape does not tile
// (no unit-stride source digit, or the united digit set is too large): the gather kernel is used.
static void build_tile_plan(const DigitList& dl, TilePlan& tp) {
    const int J = dl.n;
    int MAX_TILE = 8192;
    const int TARGET = 32;
    if (const char* env = getenv("NDMPS_PERM_TILE")) {      // development knob
        int v = atoi(env);
        if (v >= 64 && v <= 16384) MAX_TILE = v;
    }
    tp.ok = false;
    if (J < 2) return;
    std::vector<int64_t> dst_stride(J);
    int64_t s = 1;
    for (int j = J - 1; j >= 0; j--) { dst_stride[j] = s; s *= dl.extent[j]; }
    std::vector<char> in_a(J, 0), in_b(J, 0);
    auto tile_size = [&]() { int64_t t = 1; for (int j = 0; j < J; j++) if (in_a[j] || in_b[j]) t *= dl.extent[j]; return t; };
    // next digit that would extend the source chain (stride == current run length), or -1
    int64_t pa = 1, pb = 1;
    auto next_b = [&]() { for (int j = 0; j < J; j++) if (!in_b[j] && dl.stride[j] == pb) return j; return -1; };
    auto next_a = [&]() { for (int j = J - 1; j >= 0; j--) if (!in_a[j]) return j; return -1; };
    // A: innermost destination digits, B: chain of smallest source strides, both to >= TARGET
    while (pa < TARGET) { int j = next_a(); if (j < 0) break; in_a[j] = 1; pa *= dl.extent[j]; }
    while (pb < TARGET) { int j = next_b(); if (j < 0) break; in_b[j] = 1; pb *= dl.extent[j]; }
    if (pb < 2) return;
    if (tile_size() > MAX_TILE) return;
    // grow the shorter run first while the tile fits: long runs on BOTH sides keep DRAM pages open
    for (;;) {
        int ja = next_a(), jb = next_b();
        int64_t ta = ja >= 0 ? tile_size() * (in_b[ja] ? 1 : dl.extent[ja]) : MAX_TILE + 1;
        int64_t tb = jb >= 0 ? tile_size() * (in_a[jb] ? 1 : dl.extent[jb]) : MAX_TILE + 1;
        bool can_a = ta <= MAX_TILE, can_b = tb <= MAX_TILE;
        if (!can_a && !can_b) break;
        bool pick_b = can_b && (!can_a || pb <= pa);
        if (pick_b) { in_b[jb] = 1; pb *= dl.extent[jb]; }
        else { in_a[ja] = 1; pa *= dl.extent[ja]; }
    }
    const int64_t tile = tile_size();
    if (tile > MAX_TILE || tile < 2) return;
    // digit orders inside the tile
    std::vector<int> wdig, rdig;           // write order (outer -> inner), read order (outer -> inner)
    for (int j = 0; j < J; j++) if ((in_a[j] || in_b[j]) && !in_a[j]) wdig.push_back(j);   // B \ A: outer part of the write order
    for (int j = 0; j < J; j++) if (in_a[j]) wdig.push_back(j);                              // A: inner, destination-contiguous
    std::vector<int> bchain, arest;
    for (int j = 0; j < J; j++) if (in_b[j]) bchain.push_back(j);
    std::sort(bchain.begin(), bchain.end(), [&](int x, int y) { return dl.stride[x] > dl.stride[y]; });   // outer -> inner
    for (int j = 0; j < J; j++) if (in_a[j] && !in_b[j]) arest.push_back(j);
    std::sort(arest.begin(), arest.end(), [&](int x, int y) { return dl.stride[x] > dl.stride[y]; });
    rdig = arest;
    rdig.insert(rdig.end(), bchain.begin(), bchain.end());
    tp.tile = (int)tile;
    tp.pa = (int)pa;
    tp.pb = (int)pb;
    tp.hi_src.assign((size_t)(tile / pb), 0);
    tp.hi_dst.assign((size_t)(tile / pa), 0);
    tp.pos.assign((size_t)tile, 0);
    std::vector<int> digit(J, 0);
    for (int64_t r = 0; r < tile; r++) {
        // decode read index r into digits (rdig, innermost last)
        int64_t rem = r, soff = 0;
        for (int k = (int)rdig.size() - 1; k >= 0; k--) {
            int j = rdig[k];
            digit[j] = (int)(rem % dl.extent[j]);
            rem /= dl.extent[j];
            soff += (int64_t)digit[j] * dl.stride[j];
        }
        if (r % pb == 0) tp.hi_src[(size_t)(r / pb)] = soff;
        // write index of the same element
        int64_t w = 0, doff = 0;
        for (size_t k = 0; k < wdig.size(); k++) {
            int j = wdig[k];
            w = w * dl.extent[j] + digit[j];
            doff += (int64_t)digit[j] * dst_stride[j];
        }
        if (w % pa == 0) tp.hi_dst[(size_t)(w / pa)] = doff;
        tp.pos[(size_t)r] = (uint16_t)skew_slot((int)w);
    }
    // outer digits in destination order
    tp.n_outer = 0;
    tp.n_tiles = 1;
    for (int j = 0; j < J; j++) {
        if (in_a[j] || in_b[j]) continue;
        tp.outer_extent[tp.n_outer] = dl.extent[j];
        tp.outer_dst[tp.n_outer] = dst_stride[j];
        tp.outer_src[tp.n_outer] = dl.stride[j];
        tp.n_outer++;
        tp.n_tiles *= dl.extent[j];
    }
    // worst bank-conflict degree of the scatter (32 consecutive read indices, 4-byte words)
    int worst = 1;
    for (int64_t r0 = 0; r0 + 32 <= tile; r0 += 32) {
        int cnt[32] = {0};
        for (int k = 0; k < 32; k++) cnt[tp.pos[(size_t)(r0 + k)] & 31]++;
        for (int k = 0; k < 32; k++) worst = cnt[k] > worst ? cnt[k] : worst;
    }
    tp.conflict = worst;
    tp.ok = true;
}

static std::mutex g_upload_mutex;   // plans are shared between host threads (batch.py); the upload happens once

// Returns (a copy of) the table pointers of `device`, uploading them on first use.  The copy is taken under the
// lock, so host threads driving different GPUs with one shared plan never see each other's pointers.
static int upload_tile_plan(TilePlan& tp, int device, TilePlan::DevTables* out) {
    std::lock_guard<std::mutex> lock(g_upload_mutex);
    for (const auto& d : tp.dev)
        if (d.device == device) { *out = d; return NDMPS_OK; }
    TilePlan::DevTables d;
    d.device = device;
    NDMPS_CUDA_TRY(cudaMalloc(&d.hi_src, tp.hi_src.size() * sizeof(int64_t)));
    NDMPS_CUDA_TRY(cudaMalloc(&d.hi_dst, tp.hi_dst.size() * sizeof(int64_t)));
    NDMPS_CUDA_TRY(cudaMalloc(&d.pos, tp.pos.size() * sizeof(uint16_t)));
    NDMPS_CUDA_TRY(cudaMemcpy(d.hi_src, tp.hi_src.data(), tp.hi_src.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
    NDMPS_CUDA_TRY(cudaMemcpy(d.hi_dst, tp.hi_dst.data(), tp.hi_dst.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
    NDMPS_CUDA_TRY(cudaMemcpy(d.pos, tp.pos.data(), tp.pos.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
    tp.dev.push_back(d);
    *out = d;
    return NDMPS_OK;
}

template <class T>
static int permute_tiled(ndmps_ctx* ctx, TilePlan& tp, const T* src, T* dst, double scale, bool do_scale) {
    TilePlan::DevTables dt;
    NDMPS_TRY(upload_tile_plan(tp, ctx->device, &dt));
    TileArgs ta;
    ta.tile = tp.tile; ta.pa = tp.pa; ta.pb = tp.pb; ta.n_outer = tp.n_outer; ta.n_tiles = tp.n_tiles;
    for (int j = 0; j < tp.n_outer; j++) {
        ta.outer_extent[j] = tp.outer_extent[j];
        ta.outer_dst[j] = tp.outer_dst[j];
        ta.outer_src[j] = tp.outer_src[j];
    }
    ta.hi_src = dt.hi_src; ta.hi_dst = dt.hi_dst; ta.pos = dt.pos;
    const size_t smem = (size_t)(skew_slot(tp.tile) + 8) * sizeof(T);
    {
        // float64 tiles exceed the 48 KB default
        NDMPS_TRY(raise_dynamic_smem((const void*)permute_tiled_kernel<T, 4>, ctx->device, 96 * 1024));
        NDMPS_TRY(raise_dynamic_smem((const void*)permute_tiled_kernel<T, 1>, ctx->device, 96 * 1024));
    }
    int64_t grid = tp.n_tiles;
    // measured: the fewer tiles a CTA walks the better (the hardware scheduler balances the tail); 64 CTAs
    // per SM in the grid means one tile per CTA up to 512^3 and a grid-stride loop beyond
    int64_t cap = (int64_t)ctx->sm_count * 64;
    if (grid > cap) grid = cap;
    // 16-byte accesses when every run and every run offset is a multiple of 4 elements (float32 only)
    bool vec4 = sizeof(T) == 4 && (tp.pa % 4 == 0) && (tp.pb % 4 == 0) &&
                (reinterpret_cast<uintptr_t>(src) % 16 == 0) && (reinterpret_cast<uintptr_t>(dst) % 16 == 0);
    if (vec4) {
        for (size_t k = 0; k < tp.hi_src.size() && vec4; k++) vec4 = tp.hi_src[k] % 4 == 0;
        for (size_t k = 0; k < tp.hi_dst.size() && vec4; k++) vec4 = tp.hi_dst[k] % 4 == 0;
        for (int j = 0; j < tp.n_outer && vec4; j++) vec4 = tp.outer_dst[j] % 4 == 0 && tp.outer_src[j] % 4 == 0;
    }
    if (vec4) permute_tiled_kernel<T, 4><<<(unsigned)grid, PERM_THREADS, smem, ctx->stream>>>(src, dst, ta, scale, do_scale);
    else permute_tiled_kernel<T, 1><<<(unsigned)grid, PERM_THREADS, smem, ctx->stream>>>(src, dst, ta, scale, do_scale);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

template <class T>
static int permute_typed(ndmps_ctx* ctx, const ndmps_plan* plan, bool inverse, const T* src, T* dst, double scale) {
    int64_t total = plan->total;
    if (total == 0) return NDMPS_OK;
    bool do_scale = scale != 1.0;
    int64_t want = (total + 255) / 256;
    int64_t cap = (int64_t)ctx->sm_count * 32;
    int grid = (int)(want < cap ? want : cap);
    if (plan->identity) {
        if (src == dst && !do_scale) return NDMPS_OK;
        copy_scale_kernel<T><<<grid, 256, 0, ctx->stream>>>(src, dst, total, scale, do_scale);
        NDMPS_LAUNCH_CHECK(ctx);
        return NDMPS_OK;
    }
    NDMPS_REQUIRE(src != dst, "ndmps permute: in-place permutation is not supported");
    if (std::is_same<T, float>::value && ctx->opt_permute_path == 0) {
        const BitPlan& bp = inverse ? plan->dec_bits : plan->enc_bits;
        if (bp.ok && reinterpret_cast<uintptr_t>(src) % 16 == 0 && reinterpret_cast<uintptr_t>(dst) % 16 == 0) {
            BitArgs ba;
            fill_bit_args(bp, ba);
            permute_bits_kernel<<<1u << ba.n_cta, BITS_THREADS, 0, ctx->stream>>>((const float*)src, (float*)dst, ba, (float)scale,
                                                                                 do_scale);
            NDMPS_LAUNCH_CHECK(ctx);
            return NDMPS_OK;
        }
    }
    TilePlan& tp = const_cast<TilePlan&>(inverse ? plan->dec_tile : plan->enc_tile);
    if (tp.ok && ctx->opt_permute_path != 2) return permute_tiled<T>(ctx, tp, src, dst, scale, do_scale);
    const DigitList& dl = inverse ? plan->dec : plan->enc;
    if (total < (int64_t(1) << 32))
        permute_gather_kernel<T, true><<<grid, 256, 0, ctx->stream>>>(src, dst, dl, total, scale, do_scale);
    else
        permute_gather_kernel<T, false><<<grid, 256, 0, ctx->stream>>>(src, dst, dl, total, scale, do_scale);
    NDMPS_LAUNCH_CHECK(ctx);
    return NDMPS_OK;
}

int permute(ndmps_ctx* ctx, const ndmps_plan* plan, bool inverse, const void* src, void* dst, int dtype, double scale) {
    StageScope sc(ctx, ST_PERMUTE);
    if (dtype == NDMPS_F32) return permute_typed<float>(ctx, plan, inverse, (const float*)src, (float*)dst, scale);
    return permute_typed<double>(ctx, plan, inverse, (const double*)src, (double*)dst, scale);
}

}  // namespace ndmps

using namespace ndmps;

extern "C" {

int ndmps_plan_create(int ndim, const int64_t* shape, int levels, const int64_t* factors, ndmps_plan_t** out) {
    NDMPS_REQUIRE(out && shape && factors, "ndmps_plan_create: NULL argument");
    NDMPS_REQUIRE(ndim >= 1 && ndim <= 8, "ndmps_plan_create: ndim %d outside 1..8", ndim);
    NDMPS_REQUIRE(levels >= 1 && levels * ndim <= NDMPS_MAX_DIGITS,
                  "ndmps_plan_create: levels*ndim = %d exceeds %d", levels * ndim, NDMPS_MAX_DIGITS);
    ndmps_plan* p = new ndmps_plan();
    p->ndim = ndim;
    p->levels = levels;
    p->total = 1;
    for (int a = 0; a < ndim; a++) {
        if (shape[a] <= 0) { delete p; set_error("ndmps_plan_create: non-positive extent"); return NDMPS_ERR_INVALID; }
        p->shape[a] = shape[a];
        p->total *= shape[a];
        int64_t prod = 1;
        for (int l = 0; l < levels; l++) {
            int64_t f = factors[l * ndim + a];
            if (f <= 0) { delete p; set_error("ndmps_plan_create: non-positive factor"); return NDMPS_ERR_INVALID; }
            p->factors[l * ndim + a] = f;
            prod *= f;
        }
        if (prod != shape[a]) {
            delete p;
            set_error("ndmps_plan_create: factors of axis %d multiply to %lld, extent is %lld", a, (long long)prod,
                      (long long)shape[a]);
            return NDMPS_ERR_INVALID;
        }
    }
    for (int l = 0; l < levels; l++) {
        int64_t d = 1;
        for (int a = 0; a < ndim; a++) d *= factors[l * ndim + a];
        p->site_dims[l] = d;
    }
    // strides of digit (l, a) in the volume (C order over axes, then over the axis' own digits)
    // and in the site-ordered array (C order over levels, then over axes inside a level)
    std::vector<int64_t> vol_stride(levels * ndim), site_stride(levels * ndim);
    int64_t axis_stride = 1;
    for (int a = ndim - 1; a >= 0; a--) {
        int64_t s = axis_stride;
        for (int l = levels - 1; l >= 0; l--) { vol_stride[l * ndim + a] = s; s *= factors[l * ndim + a]; }
        axis_stride *= shape[a];
    }
    int64_t s = 1;
    for (int l = levels - 1; l >= 0; l--)
        for (int a = ndim - 1; a >= 0; a--) { site_stride[l * ndim + a] = s; s *= factors[l * ndim + a]; }
    // encode: destination walks (l, a) in C order, gathers from the volume
    for (int l = 0; l < levels; l++)
        for (int a = 0; a < ndim; a++) push_digit(p->enc, (uint32_t)factors[l * ndim + a], vol_stride[l * ndim + a]);
    // decode: destination walks (a, l) in C order, gathers from the site-ordered array
    for (int a = 0; a < ndim; a++)
        for (int l = 0; l < levels; l++) push_digit(p->dec, (uint32_t)factors[l * ndim + a], site_stride[l * ndim + a]);
    finish(p->enc);
    finish(p->dec);
    p->identity = (p->enc.n == 1 && p->enc.stride[0] <= 1);
    if (!p->identity) {
        build_tile_plan(p->enc, p->enc_tile);
        build_tile_plan(p->dec, p->dec_tile);
        build_bit_plan(p->enc, p->total, p->enc_bits);
        build_bit_plan(p->dec, p->total, p->dec_bits);
    }
    *out = p;
    return NDMPS_OK;
}

int ndmps_plan_destroy(ndmps_plan_t* plan) {
    if (plan) {
        int cur = -1;
        cudaGetDevice(&cur);
        for (TilePlan* tp : {&plan->enc_tile, &plan->dec_tile}) {
            for (auto& d : tp->dev) {
                if (d.device != cur) cudaSetDevice(d.device);
                cudaFree(d.hi_src);
                cudaFree(d.hi_dst);
                cudaFree(d.pos);
                if (d.device != cur) cudaSetDevice(cur);
            }
            tp->dev.clear();
        }
    }
    delete plan;
    return NDMPS_OK;
}

int ndmps_plan_site_dims(const ndmps_plan_t* plan, int64_t* dims_out) {
    NDMPS_REQUIRE(plan && dims_out, "ndmps_plan_site_dims: NULL argument");
    for (int l = 0; l < plan->levels; l++) dims_out[l] = plan->site_dims[l];
    return NDMPS_OK;
}

int ndmps_plan_debug_offsets(const ndmps_plan_t* plan, int inverse, int64_t first, int64_t count, int64_t* out_host) {
    NDMPS_REQUIRE(plan && out_host, "ndmps_plan_debug_offsets: NULL argument");
    NDMPS_REQUIRE(first >= 0 && count >= 0 && first + count <= plan->total, "ndmps_plan_debug_offsets: range outside the volume");
    const DigitList& dl = inverse ? plan->dec : plan->enc;
    for (int64_t i = 0; i < count; i++)
        out_host[i] = plan->identity ? first + i : digit_offset<uint64_t>(dl, (uint64_t)(first + i));
    return NDMPS_OK;
}

int ndmps_plan_debug_tile_info(const ndmps_plan_t* plan, int inverse, int64_t* info_out) {
    NDMPS_REQUIRE(plan && info_out, "ndmps_plan_debug_tile_info: NULL argument");
    const TilePlan& tp = inverse ? plan->dec_tile : plan->enc_tile;
    info_out[0] = tp.ok ? 1 : 0;
    info_out[1] = tp.tile;
    info_out[2] = tp.pa;
    info_out[3] = tp.pb;
    info_out[4] = tp.n_tiles;
    info_out[5] = tp.conflict;
    return NDMPS_OK;
}

int ndmps_plan_debug_apply_tiled(const ndmps_plan_t* plan, int inverse, const int32_t* src_host, int32_t* dst_host) {
    NDMPS_REQUIRE(plan && src_host && dst_host, "ndmps_plan_debug_apply_tiled: NULL argument");
    const TilePlan& tp = inverse ? plan->dec_tile : plan->enc_tile;
    NDMPS_REQUIRE(tp.ok, "ndmps_plan_debug_apply_tiled: this shape does not tile");
    std::vector<int32_t> buf((size_t)skew_slot(tp.tile) + 8);
    const bool vec4 = tp.pa % 4 == 0 && tp.pb % 4 == 0;
    for (int64_t tile = 0; tile < tp.n_tiles; tile++) {
        int64_t rem = tile, base_dst = 0, base_src = 0;
        for (int j = tp.n_outer - 1; j >= 0; j--) {
            int64_t q = rem / tp.outer_extent[j], d = rem - q * tp.outer_extent[j];
            base_dst += d * tp.outer_dst[j];
            base_src += d * tp.outer_src[j];
            rem = q;
        }
        if (vec4) {   // same grouping as the 16-byte kernel path
            const int nvec = tp.tile >> 2, pbv = tp.pb >> 2, pav = tp.pa >> 2;
            for (int v = 0; v < nvec; v++) {
                const int hi = v / pbv, lo = (v - hi * pbv) << 2;
                for (int e = 0; e < 4; e++) buf[tp.pos[(size_t)(hi * tp.pb + lo + e)]] = src_host[base_src + tp.hi_src[(size_t)hi] + lo + e];
            }
            for (int v = 0; v < nvec; v++) {
                const int hi = v / pav, lo = (v - hi * pav) << 2;
                const int s = skew_slot(hi * tp.pa + lo);
                for (int e = 0; e < 4; e++) dst_host[base_dst + tp.hi_dst[(size_t)hi] + lo + e] = buf[(size_t)s + e];
            }
        } else {
            for (int r = 0; r < tp.tile; r++) {
                const int hi = r / tp.pb, lo = r - hi * tp.pb;
                buf[tp.pos[(size_t)r]] = src_host[base_src + tp.hi_src[(size_t)hi] + lo];
            }
            for (int w = 0; w < tp.tile; w++) {
                const int hi = w / tp.pa, lo = w - hi * tp.pa;
                dst_host[base_dst + tp.hi_dst[(size_t)hi] + lo] = buf[(size_t)skew_slot(w)];
            }
        }
    }
    return NDMPS_OK;
}

int ndmps_plan_debug_bit_info(const ndmps_plan_t* plan, int inverse, int64_t* info_out) {
    NDMPS_REQUIRE(plan && info_out, "ndmps_plan_debug_bit_info: NULL argument");
    const BitPlan& bp = inverse ? plan->dec_bits : plan->enc_bits;
    info_out[0] = bp.ok ? 1 : 0;
    info_out[1] = bp.nbits;
    info_out[2] = bp.row_shift;
    info_out[3] = bp.pair_shift;
    info_out[4] = bp.ok ? (int64_t(1) << (bp.n_idx - BITS_FIXED_IDX)) : 0;
    // contiguous run (elements) one CTA covers on the destination / source side
    int64_t run[2] = {0, 0};
    if (bp.ok) {
        for (int side = 0; side < 2; side++) {
            bool have[64] = {false};
            have[0] = have[1] = true;
            have[side == 0 ? bp.pair_shift : bp.row_shift] = true;
            for (int t = 0; t < BITS_FIXED_IDX; t++) have[side == 0 ? bp.dst_bit[t] : bp.src_bit[t]] = true;
            int k = 0;
            while (k < bp.nbits && have[k]) k++;
            run[side] = int64_t(1) << k;
        }
    }
    info_out[5] = run[0];
    info_out[6] = run[1];
    return NDMPS_OK;
}

int ndmps_plan_debug_apply_bits(const ndmps_plan_t* plan, int inverse, const int32_t* src_host, int32_t* dst_host) {
    NDMPS_REQUIRE(plan && src_host && dst_host, "ndmps_plan_debug_apply_bits: NULL argument");
    const BitPlan& bp = inverse ? plan->dec_bits : plan->enc_bits;
    NDMPS_REQUIRE(bp.ok, "ndmps_plan_debug_apply_bits: this shape has no bit plan");
    BitArgs ba;
    fill_bit_args(bp, ba);
    const int64_t row = int64_t(1) << ba.row_shift, pair = int64_t(1) << ba.pair_shift;
    for (unsigned block = 0; block < (1u << ba.n_cta); block++)
        for (unsigned tid = 0; tid < (unsigned)BITS_THREADS; tid++) {
            int64_t so, d0;
            bits_offsets(ba, tid, block, so, d0);
            for (int u = 0; u < BITS_UNROLL; u++) {
                const int32_t* lo = src_host + so + ba.u_src[u];
                const int32_t* hi = lo + row;
                int32_t* q = dst_host + d0 + ba.u_dst[u];
                q[0] = lo[0]; q[1] = lo[1]; q[2] = hi[0]; q[3] = hi[1];
                q[pair] = lo[2]; q[pair + 1] = lo[3]; q[pair + 2] = hi[2]; q[pair + 3] = hi[3];
            }
        }
    return NDMPS_OK;
}

int ndmps_encode(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* src, void* dst, int dtype, double scale) {
    NDMPS_REQUIRE(ctx && plan && src && dst, "ndmps_encode: NULL argument");
    NDMPS_REQUIRE(dtype_ok(dtype), "ndmps_encode: bad dtype %d", dtype);
    return permute(ctx, plan, false, src, dst, dtype, scale);
}

int ndmps_decode(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* src, void* dst, int dtype) {
    NDMPS_REQUIRE(ctx && plan && src && dst, "ndmps_decode: NULL argument");
    NDMPS_REQUIRE(dtype_ok(dtype), "ndmps_decode: bad dtype %d", dtype);
    return permute(ctx, plan, true, src, dst, dtype, 1.0);
}

}  // extern "C"
