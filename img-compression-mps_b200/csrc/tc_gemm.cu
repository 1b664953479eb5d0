// K2 / K5 / K7 on the 5th-generation tensor cores: tcgen05.mma on bf16x3 split planes.
//
// The capped (max_bond) float32 sweep of `MatrixProductState.from_dense` (core/ndmps.py:74) and
// the contraction of `to_tensor` (core/ndmps.py:140) need float32-class products with
// better-than-float32 accumulation; tcgen05 has no float32/float64 kind.  A float32 value splits
// EXACTLY into three bfloat16 values (8 + 8 + 8 significand bits, round to nearest at every step:
// x = h + m + l), so
//
//     a . b  =  h.h + (h.m + m.h) + (h.l + l.h + m.m)  +  O(2^-26 |a||b|)
//
// is six kind::f16 MMAs with float32 accumulation in TMEM.  The operands live in HBM as "split
// planes" (bf16[3][rows][ld]); tiles arrive in shared memory by TMA (cp.async.bulk.tensor, 128-byte
// swizzle, out-of-range rows/columns zero-filled), one elected thread issues the MMAs, the
// accumulators stay in tensor memory and come back with tcgen05.ld.
//
//   * gram_tc_kernel : G = M M^T.  K = C is long (2^15 .. 2^18): the TMEM accumulators are drained
//     into float64 registers (double-buffered, so draining overlaps the MMAs) - the truncating
//     float32 accumulation of the tensor core then acts on short chains only (see "Accumulation
//     discipline" below).  Upper-triangle tiles, split-K partials reduced in fixed order
//     (deterministic, symmetric).
//   * gemm_tc_kernel : C = A B for the projection T = P^T M and the final contraction
//     dense = X W: K is bond-sized, the whole K loop accumulates in TMEM.  Either operand may be
//     K-major or MN-major (the big unfolding is MN-major for the projection); the output is written
//     row-major or transposed.
//
// Warp roles (one CTA per SM: the stages fill its shared memory): warp 0 TMA producer, warp 1 MMA
// issuer, warp 2 TMEM allocator, warps 4-11 epilogue (TMEM lane quadrant = warp % 4).
#include <cuda.h>
#include <cuda_bf16.h>

#include <mutex>

#include <type_traits>

#include "common.cuh"

namespace ndmps {
namespace tc {

constexpr int TILE = 128;                 // MMA M (rows of A per CTA) and the Gram's N
constexpr int BK = 64;                    // bf16 elements per k-tile: one 128-byte swizzled row
constexpr int UK = 16;                    // K of one tcgen05.mma.kind::f16
constexpr int PLANE_TILE = TILE * BK * 2; // bytes of one 128 x 64 bf16 tile
constexpr int CTRL_THREADS = 128, EPI_THREADS = 256, THREADS = CTRL_THREADS + EPI_THREADS;
constexpr unsigned long long SPIN_LIMIT = 4000000000ull;   // ~2 s of SM clocks: a protocol bug traps instead of hanging the GPU

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const unsigned long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if ((unsigned long long)clock64() - t0 > SPIN_LIMIT) __trap();
    }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, float32 accumulate
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on `bar` when every tcgen05 operation this thread issued so far has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 32 consecutive float32 columns: thread t of the warp gets lane (quadrant base + t)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Shared-memory matrix descriptor, 128-byte swizzle, descriptor version 1 (sm_100).
//   K-major  tile (rows x 64 bf16, 128-byte rows, 8-row groups 1024 B apart): lbo = 1 (unused), sbo = 1024 B;
//            the k-step inside the swizzled row advances the start address by 32 B.
//   MN-major tile (64 k-rows x 64 bf16 per TMA box, boxes 8192 B apart along MN): lbo = 8192 B, sbo = 1024 B
//            (8 k-rows); a k-step of 16 rows advances the start address by 2048 B.
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    const uint32_t lo = ((addr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
    const uint32_t hi = ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | (2u << 29);
    return ((uint64_t)hi << 32) | lo;
}
// kind::f16 instruction descriptor: D float32, A and B bfloat16, M x N, majors (0 = K, 1 = MN)
__host__ __device__ constexpr uint32_t instr_desc(int m, int n, int a_mn, int b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(n >> 3) << 17) |
           ((uint32_t)(m >> 4) << 24);
}

// ---------------------------------------------------------------------------------------------
// float32 / float64 -> three bfloat16 planes (x = h + m + l, every step round-to-nearest)
// ---------------------------------------------------------------------------------------------
template <class T>
__device__ __forceinline__ void split3(T x, __nv_bfloat16& h, __nv_bfloat16& m, __nv_bfloat16& l) {
    h = __float2bfloat16_rn((float)x);
    T r = x - (T)__bfloat162float(h);
    m = __float2bfloat16_rn((float)r);
    r = r - (T)__bfloat162float(m);
    l = __float2bfloat16_rn((float)r);
}

// src: rows x cols (row stride ld_src); dst: bf16[3][rows][ldp], columns cols..ldp-1 zeroed.  Eight elements per thread
// (16-byte stores).
template <class T>
__global__ void __launch_bounds__(256)
split_planes_kernel(const T* __restrict__ src, int64_t rows, int64_t cols, int64_t ld_src, double alpha,
                    __nv_bfloat16* __restrict__ dst, int64_t ldp, int64_t plane_stride) {
    const int64_t groups = ldp >> 3, total = rows * groups, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t r = i / groups, c0 = (i - r * groups) << 3;
        __align__(16) __nv_bfloat16 h[8], m[8], l[8];
        T v[8];
        const T* p = src + r * ld_src + c0;
        if (sizeof(T) == 4 && c0 + 8 <= cols && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) {
            const float4 a = __ldcs(reinterpret_cast<const float4*>(p)), b = __ldcs(reinterpret_cast<const float4*>(p) + 1);
            v[0] = (T)a.x; v[1] = (T)a.y; v[2] = (T)a.z; v[3] = (T)a.w; v[4] = (T)b.x; v[5] = (T)b.y; v[6] = (T)b.z; v[7] = (T)b.w;
        } else {
#pragma unroll
            for (int j = 0; j < 8; j++) v[j] = c0 + j < cols ? p[j] : (T)0;
        }
#pragma unroll
        for (int j = 0; j < 8; j++) split3<T>(v[j] * (T)alpha, h[j], m[j], l[j]);
        __nv_bfloat16* o = dst + r * ldp + c0;
        *reinterpret_cast<uint4*>(o) = *reinterpret_cast<const uint4*>(h);
        *reinterpret_cast<uint4*>(o + plane_stride) = *reinterpret_cast<const uint4*>(m);
        *reinterpret_cast<uint4*>(o + 2 * plane_stride) = *reinterpret_cast<const uint4*>(l);
    }
}

// ---------------------------------------------------------------------------------------------
// Accumulation discipline (measured on B200, tools/tc_probe.py): the tensor core adds into its float32
// TMEM accumulator with TRUNCATION, a relative bias of about -3e-8 of the accumulator per MMA.  So:
//   * the leading products h.h (16 significant bits each) go to their OWN accumulator, restarted
//     every k-tile (4 MMAs of K = 16): 64 products per chain, then the chain is drained by the
//     epilogue warps and summed on the CUDA cores (round to nearest, unbiased; float64 for the Gram);
//   * the five correction products (2^-8 and 2^-16 of the result) share a second accumulator with
//     long chains: the same relative bias there is 2^-8 smaller in the result.
// Both accumulators are double-buffered so the drains overlap the MMAs of the next k-tile.
// ---------------------------------------------------------------------------------------------
// correction products, smallest first: (plane of A, plane of B)
__device__ __constant__ int8_t REST_A[5] = {1, 2, 0, 1, 0};
__device__ __constant__ int8_t REST_B[5] = {1, 0, 2, 0, 1};

// ---------------------------------------------------------------------------------------------
// Gram on the INTEGER tensor cores (kind::i8, int32 accumulators): error-free accumulation.
//
// The left factor of a sweep step is decided by the trailing kept eigenvalues of G = M M^T, which sit at
// lambda_chi / lambda_1 ~ 1e-6 with gaps of a few percent of that.  Measured (profiles/r02_summary.md): a Gram
// accumulated in float32 on the tensor cores (bf16x3 planes: 1e-7 .. 3e-7 normwise, the accumulator truncates)
// rotates those eigenvectors - reconstructions 2e-4 off on the DCT video chunk.  So the tensor-core Gram uses
// sliced integers (Ozaki scheme): row i is scaled by a power of two, y = x 2^-sc_i in (-1/2, 1/2), and written
// as five signed 7-bit digits, y = sum_p a_p 2^(-7 (p + 1)) + O(2^-36), |a_p| <= 64 (round to nearest at every
// digit, exact in float32).  Digit products are exact in the int32 accumulators:
//     y_i . y_j = sum_s 2^(-7 (s + 2)) ACC_s,    ACC_s = sum_k sum_{p + q = s} a_p b_q,   s = 0 .. 4
// fifteen MMAs per k-step of 32, five accumulators of 64 columns (tiles are 128 x 64), NO drains inside a chain
// (|ACC_4| <= 5 * 4096 K: chains of 2^16 columns), one exact int32 -> float64 combination per chain.
// What is dropped: products with p + q >= 5.  Those with p + q = 5 are zero-mean (independent digits); the
// first systematic term is the digit-3 square at 2^-56, i.e. a relative error of 8e-14 rho_i^2 on G_ii with
// rho_i = max|row| / rms(row) (with FOUR digits the same term sits at 2^-42: 1.2e-9 rho^2, measured, and
// breaks fMRI and DCT rows with rho ~ 25; exact zeros have all-zero digits, so rho runs over the nonzero
// elements).  rho is known before the products run (the scaling pass measures max, sum of squares and nonzero
// count of every row): if 8e-14 max rho^2 exceeds 3e-10 a device-side flag hands the matrix to the exact
// FP64-pipe kernel instead (gram_dmma.cu), without a host round trip.
// ---------------------------------------------------------------------------------------------
constexpr int I8_PLANES = 5;
constexpr int I8_TN = 64;                        // columns of a Gram tile (five accumulators of 64 columns)
constexpr int I8_BK = 64;                        // int8 elements per k-tile: 64-byte rows (SWIZZLE_64B)
constexpr int I8_UK = 32;                        // K of one tcgen05.mma.kind::i8
constexpr int I8_BOX_BYTES = 64 * I8_BK;         // 4 KB: one TMA box of 64 rows x 64 digits
constexpr int I8_MAX_CHAIN_TILES = 1024;         // 2^16 columns per accumulator chain: |ACC_4| <= 5 * 4096 * 2^16 < 2^31
constexpr double I8_RHO2_LIMIT = 4096.0;         // 8e-14 * 4096 = 3.3e-10 relative on the worst diagonal entry

struct GramI8Smem {
    static constexpr int STAGES = 3;
    static constexpr int A_BYTES = I8_PLANES * 2 * I8_BOX_BYTES;       // 128 rows per digit plane
    static constexpr int STAGE_BYTES = A_BYTES + I8_PLANES * I8_BOX_BYTES;   // + 64 rows per digit plane = 60 KB
    static constexpr int BARRIER_OFF = STAGES * STAGE_BYTES;
    static constexpr int TOTAL = BARRIER_OFF + 256 + 1024;
};

// 64-byte swizzle, K-major: 8-row groups are 512 B apart, a k-step of 32 int8 advances the start address by 32 B
__device__ __forceinline__ uint64_t smem_desc_sw64(uint32_t addr) {
    const uint32_t lo = ((addr >> 4) & 0x3FFFu) | (1u << 16);
    const uint32_t hi = (512u >> 4) | (1u << 14) | (4u << 29);
    return ((uint64_t)hi << 32) | lo;
}
// kind::i8 instruction descriptor: D int32, A and B signed int8, K-major both
__host__ __device__ constexpr uint32_t instr_desc_i8(int m, int n) {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// The digit products of one k-step.  A_p . B_q^T belongs to accumulator p + q, the accumulators are consecutive blocks of
// 64 TMEM columns and the B digit planes are consecutive 64-row blocks of shared memory, so for a fixed p the products
// with q = 0 .. 4 - p are ONE MMA of N = 64 (5 - p) on the stacked planes into columns [64 p, 320): six instructions
// instead of fifteen (N <= 256 splits p = 0 in two), and every A plane is fetched from shared memory once or twice instead
// of 5 - p times - the operand fetch, not the arithmetic, bounded the 15-instruction form (tensor pipe 50 % active).
// `first` = these are the first products of an accumulator chain (p = 0 writes every accumulator first).
template <class DescA>
__device__ __forceinline__ void digit_products(uint32_t tmem_base, DescA desc_a, uint32_t b_planes, int ks, uint32_t idesc_flags, bool first) {
    const uint32_t i64 = instr_desc_i8(TILE, 64) | idesc_flags, i128 = instr_desc_i8(TILE, 128) | idesc_flags;
    const uint32_t i192 = instr_desc_i8(TILE, 192) | idesc_flags, i256 = instr_desc_i8(TILE, 256) | idesc_flags;
    const uint64_t b0 = smem_desc_sw64(b_planes + ks * 32);                        // planes 0 .. (N / 64 - 1)
    const uint64_t b4 = smem_desc_sw64(b_planes + 4 * I8_BOX_BYTES + ks * 32);     // plane 4 alone
    umma_i8(tmem_base, desc_a(0), b0, i256, first ? 0u : 1u);                      // s = 0 .. 3
    umma_i8(tmem_base + 4 * I8_TN, desc_a(0), b4, i64, first ? 0u : 1u);           // s = 4
    umma_i8(tmem_base + 1 * I8_TN, desc_a(1), b0, i256, 1u);                       // s = 1 .. 4
    umma_i8(tmem_base + 2 * I8_TN, desc_a(2), b0, i192, 1u);                       // s = 2 .. 4
    umma_i8(tmem_base + 3 * I8_TN, desc_a(3), b0, i128, 1u);                       // s = 3, 4
    umma_i8(tmem_base + 4 * I8_TN, desc_a(4), b0, i64, 1u);                        // s = 4
}

// tile t -> (row tile of 128, column tile of 64) over the tiles that touch the upper triangle: tj >= 2 ti
__device__ __forceinline__ void upper_tile_i8(int t, int ntc, int& ti, int& tj) {
    int row = 0, left = t;
    while (left >= ntc - 2 * row) { left -= ntc - 2 * row; row++; }
    ti = row;
    tj = 2 * row + left;
}

// stats[(r * chunks + c) * 3 + {0, 1, 2}] = max |x|, sum x^2 (float64), number of nonzero elements of columns chunk c of row r
__global__ void __launch_bounds__(256)
row_stats_kernel(const float* __restrict__ x, int64_t cols, int64_t ld, int64_t cols_per_cta, double* __restrict__ stats) {
    __shared__ double red[3][8];
    const int64_t r = blockIdx.x;
    const int64_t c0 = (int64_t)blockIdx.y * cols_per_cta, c1 = c0 + cols_per_cta < cols ? c0 + cols_per_cta : cols;
    const float* p = x + r * ld;
    float m = 0.f;
    double sq = 0.0;
    int nz = 0;
    if ((ld & 3) == 0 && (c0 & 3) == 0 && ((reinterpret_cast<uintptr_t>(x) & 15) == 0)) {
        const int64_t v1 = c0 + ((c1 - c0) & ~int64_t(3));
        for (int64_t c = c0 + 4 * threadIdx.x; c < v1; c += 1024) {
            const float4 v = *reinterpret_cast<const float4*>(p + c);
            m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
            sq += (double)(v.x * v.x + v.y * v.y) + (double)(v.z * v.z + v.w * v.w);
            nz += (v.x != 0.f) + (v.y != 0.f) + (v.z != 0.f) + (v.w != 0.f);
        }
        for (int64_t c = v1 + threadIdx.x; c < c1; c += 256) { m = fmaxf(m, fabsf(p[c])); sq += (double)p[c] * p[c]; nz += p[c] != 0.f; }
    } else {
        for (int64_t c = c0 + threadIdx.x; c < c1; c += 256) { m = fmaxf(m, fabsf(p[c])); sq += (double)p[c] * p[c]; nz += p[c] != 0.f; }
    }
    double md = (double)m, cnt = (double)nz;
    md = warp_max(md);
    sq = warp_sum(sq);
    cnt = warp_sum(cnt);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = md; red[1][threadIdx.x >> 5] = sq; red[2][threadIdx.x >> 5] = cnt; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++) { md = fmax(md, red[0][w]); sq += red[1][w]; cnt += red[2][w]; }
        double* o = stats + ((size_t)r * gridDim.y + blockIdx.y) * 3;
        o[0] = md; o[1] = sq; o[2] = cnt;
    }
}

// sc[r]: y = x 2^-sc[r] lies in (-1/2, 1/2).  use_exact[0] = 1 when a row is too heavy-tailed for five digits
// (or not finite): the FP64-pipe kernel computes this Gram instead.  One CTA, fixed summation order.
__global__ void __launch_bounds__(256)
row_scale_kernel(const double* __restrict__ stats, int64_t rows, int chunks, int* __restrict__ sc, int* __restrict__ use_exact) {
    __shared__ int bad;
    if (threadIdx.x == 0) bad = 0;
    __syncthreads();
    for (int64_t r = threadIdx.x; r < rows; r += 256) {
        double mx = 0.0, sq = 0.0, nz = 0.0;
        for (int c = 0; c < chunks; c++) {
            const double* st = stats + (r * chunks + c) * 3;
            mx = fmax(mx, st[0]); sq += st[1]; nz += st[2];
        }
        int e = 0;
        if (mx > 0.0) frexp(mx, &e);                  // mx = f 2^e, f in [1/2, 1)
        sc[r] = e + 1;
        const bool finite = mx < INFINITY && sq < INFINITY && sq == sq;
        // rho^2 over the NONZERO elements: an exact zero has all-zero digits and contributes nothing to the dropped products
        if (!finite || (sq > 0.0 && mx * mx * nz > I8_RHO2_LIMIT * sq)) atomicOr(&bad, 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) use_exact[0] = bad;
}

// digits[p][r][c] = digit p of y = x 2^-sc[r].  16 elements per thread (16-byte stores).
__global__ void __launch_bounds__(256)
split_i8_kernel(const float* __restrict__ x, int64_t rows, int64_t cols, int64_t ld, const int* __restrict__ sc,
                const int* __restrict__ use_exact, int8_t* __restrict__ digits, int64_t ldp, int64_t plane_stride) {
    if (use_exact[0]) return;
    const int64_t groups = ldp >> 4, total = rows * groups, stride = (int64_t)gridDim.x * blockDim.x;
    const bool vec = (ld & 3) == 0 && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t r = i / groups, c0 = (i - r * groups) << 4;
        const float down = ldexpf(1.f, 7 - sc[r]);     // y * 128
        __align__(16) float v[16];
        const float* p = x + r * ld + c0;
        if (vec && c0 + 16 <= cols) {
#pragma unroll
            for (int j = 0; j < 4; j++) *reinterpret_cast<float4*>(v + 4 * j) = __ldcs(reinterpret_cast<const float4*>(p) + j);
        } else {
#pragma unroll
            for (int j = 0; j < 16; j++) v[j] = c0 + j < cols ? p[j] : 0.f;
        }
        // digit = rint(t), |t| <= 64, without the conversion pipe (FRND + F2I run at a quarter of the FP32 rate and were
        // the bound of this kernel: SM 91 % busy at 47 % of the DRAM peak): t + 1.5 * 2^23 rounds to nearest-even in the
        // adder, the low byte of its bit pattern IS the two's-complement digit, and subtracting the constant gives rint(t)
        constexpr float MAGIC = 12582912.f;
        uint32_t w[I8_PLANES][4];
#pragma unroll
        for (int j4 = 0; j4 < 4; j4++) {
            uint32_t b[I8_PLANES][4];
#pragma unroll
            for (int jj = 0; jj < 4; jj++) {
                float t = v[4 * j4 + jj] * down;
#pragma unroll
                for (int q = 0; q < I8_PLANES; q++) {
                    const float sft = t + MAGIC;
                    b[q][jj] = __float_as_uint(sft);
                    t = (t - (sft - MAGIC)) * 128.f;  // exact: |t - rint(t)| <= 1/2 has fewer significant bits than t
                }
            }
#pragma unroll
            for (int q = 0; q < I8_PLANES; q++)
                w[q][j4] = __byte_perm(__byte_perm(b[q][0], b[q][1], 0x0040), __byte_perm(b[q][2], b[q][3], 0x0040), 0x5410);
        }
        int8_t* o = digits + r * ldp + c0;
#pragma unroll
        for (int q = 0; q < I8_PLANES; q++) *reinterpret_cast<uint4*>(o + q * plane_stride) = make_uint4(w[q][0], w[q][1], w[q][2], w[q][3]);
    }
}

// TMEM columns: accumulator s at [64 s, 64 s + 64), s = p + q = 0 .. 4.  partial[split][tile]: 128 x 64 float64.
__global__ void __launch_bounds__(THREADS, 1)
gram_i8_kernel(const __grid_constant__ CUtensorMap map, int ntc, int m, int64_t K, int64_t k_per, const int* __restrict__ sc,
               const int* __restrict__ use_exact, double* __restrict__ partial) {
    if (use_exact[0]) return;                         // uniform over the grid: the FP64-pipe kernel takes this matrix
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + GramI8Smem::BARRIER_OFF);
    uint64_t* empty = full + GramI8Smem::STAGES;
    uint64_t* acc_full = empty + GramI8Smem::STAGES;     // [1]
    uint64_t* acc_empty = acc_full + 1;                  // [1]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int ti, tj;
    upper_tile_i8(blockIdx.x, ntc, ti, tj);
    const int64_t kbeg = (int64_t)blockIdx.y * k_per;
    const int64_t kend = kbeg + k_per < K ? kbeg + k_per : K;
    const int nk = (int)((kend - kbeg + I8_BK - 1) / I8_BK);
    const int n_chains = (nk + I8_MAX_CHAIN_TILES - 1) / I8_MAX_CHAIN_TILES;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&map);
        for (int s = 0; s < GramI8Smem::STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(acc_full, 1);
        mbar_init(acc_empty, EPI_THREADS / 32);
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0 && lane == 0) {
        // ---- TMA producer: per digit plane two boxes of 64 rows for A, one for B ----
        for (int kt = 0; kt < nk; kt++) {
            const int s = kt % GramI8Smem::STAGES;
            mbar_wait(&empty[s], ((kt / GramI8Smem::STAGES) & 1) ^ 1);
            mbar_expect_tx(&full[s], GramI8Smem::STAGE_BYTES);
            uint8_t* st = smem + s * GramI8Smem::STAGE_BYTES;
            const int kc = (int)(kbeg + (int64_t)kt * I8_BK);
#pragma unroll
            for (int p = 0; p < I8_PLANES; p++) {
                tma_load_3d(st + (2 * p) * I8_BOX_BYTES, &map, &full[s], kc, ti * TILE, p);
                tma_load_3d(st + (2 * p + 1) * I8_BOX_BYTES, &map, &full[s], kc, ti * TILE + 64, p);
                tma_load_3d(st + GramI8Smem::A_BYTES + p * I8_BOX_BYTES, &map, &full[s], kc, tj * I8_TN, p);
            }
        }
    } else if (warp == 1 && lane == 0) {
        // ---- MMA issuer ----
        for (int kt = 0; kt < nk; kt++) {
            const int s = kt % GramI8Smem::STAGES;
            const int chain = kt / I8_MAX_CHAIN_TILES, within = kt - chain * I8_MAX_CHAIN_TILES;
            if (within == 0 && chain > 0) {           // the epilogue has read the previous chain out of tensor memory
                mbar_wait(acc_empty, (chain - 1) & 1);
                tc_fence_after();
            }
            mbar_wait(&full[s], (kt / GramI8Smem::STAGES) & 1);
            tc_fence_after();
            const uint32_t st = smem_u32(smem + s * GramI8Smem::STAGE_BYTES);
#pragma unroll
            for (int ks = 0; ks < I8_BK / I8_UK; ks++)
                digit_products(tmem_base, [&](int p) { return smem_desc_sw64(st + (2 * p) * I8_BOX_BYTES + ks * 32); },
                               st + GramI8Smem::A_BYTES, ks, 0u, within == 0 && ks == 0);
            umma_commit(&empty[s]);
            if (within == I8_MAX_CHAIN_TILES - 1 || kt == nk - 1) umma_commit(acc_full);
        }
    } else if (warp >= 4) {
        // ---- epilogue: exact int32 -> float64 combination of the five digit-sum accumulators ----
        const int q4 = warp & 3, half = (warp - 4) >> 2;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(half * 32);
        double acc[32];
#pragma unroll
        for (int i = 0; i < 32; i++) acc[i] = 0.0;
        for (int chain = 0; chain < n_chains; chain++) {
            mbar_wait(acc_full, chain & 1);
            tc_fence_after();
#pragma unroll
            for (int s = 0; s < I8_PLANES; s++) {
                const double w = s == 0 ? 0x1p-14 : (s == 1 ? 0x1p-21 : (s == 2 ? 0x1p-28 : (s == 3 ? 0x1p-35 : 0x1p-42)));
                uint32_t v[32];
                tmem_ld32(lane_base + (uint32_t)(s * I8_TN), v);
#pragma unroll
                for (int i = 0; i < 32; i++) acc[i] = fma((double)(int)v[i], w, acc[i]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty);
        }
        // undo the row scalings: G_ij = 2^(sc_i + sc_j) y_i . y_j
        const int gi = ti * TILE + q4 * 32 + lane;
        const int sci = gi < m ? sc[gi] : 0;
        double* out = partial + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * TILE * I8_TN + (size_t)(q4 * 32 + lane) * I8_TN + half * 32;
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
            const int gj = tj * I8_TN + half * 32 + i;
            const double s0 = ldexp(acc[i], sci + (gj < m ? sc[gj] : 0));
            const double s1 = ldexp(acc[i + 1], sci + (gj + 1 < m ? sc[gj + 1] : 0));
            *reinterpret_cast<double2*>(out + i) = make_double2(s0, s1);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ---------------------------------------------------------------------------------------------
// Projection T = P^T M on the digits the Gram already made (no second pass over the unfolding):
//     T[i, c] = sum_k P[k, i] M[k, c] = 2^tc_i sum_k b(k, i) y(k, c),   b = P[k, i] 2^(sc_k - tc_i),  y = M 2^-sc_k
// y are the Gram's digit planes ([digit][k][c]: the MN-major A operand, 128-byte swizzle); b is sliced the same way
// per output row i (K-major B operand, [digit][i][k]).  Fifteen digit products into five int32 accumulators
// (tile: 128 columns c x 64 rows i), one chain over all of k (k <= 4096: |ACC_4| <= 5 * 4096 * 4096), exact.
// ---------------------------------------------------------------------------------------------
struct ProjI8Smem {
    static constexpr int STAGES = 3;
    static constexpr int A_PLANE = I8_BK * TILE;                 // 64 k-rows x 128 bytes of c = 8 KB
    static constexpr int A_BYTES = I8_PLANES * A_PLANE;
    static constexpr int STAGE_BYTES = A_BYTES + I8_PLANES * I8_BOX_BYTES;   // + 64 rows i x 64 digits of k per plane = 60 KB
    static constexpr int BARRIER_OFF = STAGES * STAGE_BYTES;
    static constexpr int TOTAL = BARRIER_OFF + 256 + 1024;
};

// bdig[p][i][k] = digit p of P[k, i] 2^(sc_k - tc_i); tc[i] chosen so that the scaled column lies in (-1/2, 1/2).
// One CTA per output row i (column of P).  P: D x r row-major (float64).
__global__ void __launch_bounds__(256)
split_i8_proj_kernel(const double* __restrict__ P, int64_t D, int64_t r, const int* __restrict__ sc, int8_t* __restrict__ bdig,
                     int64_t ldk, int64_t plane_stride, int* __restrict__ tc_out) {
    __shared__ double red[8];
    __shared__ int s_tc;
    const int64_t i = blockIdx.x;
    double mx = 0.0;
    for (int64_t k = threadIdx.x; k < D; k += 256) mx = fmax(mx, fabs(ldexp(P[k * r + i], sc[k])));
    mx = warp_max(mx);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++) mx = fmax(mx, red[w]);
        int e = 0;
        if (mx > 0.0 && mx < INFINITY) frexp(mx, &e);
        s_tc = e + 1;
        tc_out[i] = e + 1;
    }
    __syncthreads();
    const int tcv = s_tc;
    for (int64_t k = threadIdx.x; k < ldk; k += 256) {
        double t = k < D ? ldexp(P[k * r + i], sc[k] - tcv + 7) : 0.0;      // b * 128
#pragma unroll
        for (int p = 0; p < I8_PLANES; p++) {
            const double a = rint(t);
            bdig[p * plane_stride + i * ldk + k] = (int8_t)(int)a;
            t = (t - a) * 128.0;
        }
    }
}

// TMEM columns: accumulator s at [64 s, 64 s + 64).  T: r x C row-major (ldt), written transposed from the accumulator.
template <class TT>
__global__ void __launch_bounds__(THREADS, 1)
proj_i8_kernel(const __grid_constant__ CUtensorMap map_y, const __grid_constant__ CUtensorMap map_b, int64_t C, int64_t r, int64_t D,
               const int* __restrict__ tc, TT* __restrict__ T, int64_t ldt) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + ProjI8Smem::BARRIER_OFF);
    uint64_t* empty = full + ProjI8Smem::STAGES;
    uint64_t* acc_full = empty + ProjI8Smem::STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t c0 = (int64_t)blockIdx.x * TILE, i0 = (int64_t)blockIdx.y * I8_TN;
    const int nk = (int)((D + I8_BK - 1) / I8_BK);

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&map_y);
        tma_prefetch_desc(&map_b);
        for (int s = 0; s < ProjI8Smem::STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(acc_full, 1);
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0 && lane == 0) {
        for (int kt = 0; kt < nk; kt++) {
            const int s = kt % ProjI8Smem::STAGES;
            mbar_wait(&empty[s], ((kt / ProjI8Smem::STAGES) & 1) ^ 1);
            mbar_expect_tx(&full[s], ProjI8Smem::STAGE_BYTES);
            uint8_t* st = smem + s * ProjI8Smem::STAGE_BYTES;
            const int k0 = kt * I8_BK;
#pragma unroll
            for (int p = 0; p < I8_PLANES; p++) {
                tma_load_3d(st + p * ProjI8Smem::A_PLANE, &map_y, &full[s], (int)c0, k0, p);                       // 64 k-rows x 128 c
                tma_load_3d(st + ProjI8Smem::A_BYTES + p * I8_BOX_BYTES, &map_b, &full[s], k0, (int)i0, p);        // 64 rows i x 64 k
            }
        }
    } else if (warp == 1 && lane == 0) {
        for (int kt = 0; kt < nk; kt++) {                                           // A is MN-major: bit 15 of the descriptor
            const int s = kt % ProjI8Smem::STAGES;
            mbar_wait(&full[s], (kt / ProjI8Smem::STAGES) & 1);
            tc_fence_after();
            const uint32_t st = smem_u32(smem + s * ProjI8Smem::STAGE_BYTES);
#pragma unroll
            for (int ks = 0; ks < I8_BK / I8_UK; ks++)
                // A: 32 k-rows of 128 bytes per k-step (4096 B), 8-row groups 1024 B apart, one 128-byte atom along c
                digit_products(tmem_base, [&](int p) { return smem_desc(st + p * ProjI8Smem::A_PLANE + ks * 4096, 8192, 1024); },
                               st + ProjI8Smem::A_BYTES, ks, 1u << 15, kt == 0 && ks == 0);
            umma_commit(&empty[s]);
            if (kt == nk - 1) umma_commit(acc_full);
        }
    } else if (warp >= 4) {
        const int q4 = warp & 3, half = (warp - 4) >> 2;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(half * 32);
        double acc[32];
#pragma unroll
        for (int j = 0; j < 32; j++) acc[j] = 0.0;
        mbar_wait(acc_full, 0);
        tc_fence_after();
#pragma unroll
        for (int s = 0; s < I8_PLANES; s++) {
            const double w = s == 0 ? 0x1p-14 : (s == 1 ? 0x1p-21 : (s == 2 ? 0x1p-28 : (s == 3 ? 0x1p-35 : 0x1p-42)));
            uint32_t v[32];
            tmem_ld32(lane_base + (uint32_t)(s * I8_TN), v);
#pragma unroll
            for (int j = 0; j < 32; j++) acc[j] = fma((double)(int)v[j], w, acc[j]);
        }
        const int64_t c = c0 + q4 * 32 + lane;
        if (c < C) {
#pragma unroll
            for (int j = 0; j < 32; j++) {
                const int64_t i = i0 + half * 32 + j;
                if (i < r) T[i * ldt + c] = (TT)ldexp(acc[j], tc[i]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// G[i][j] = G[j][i] = sum over splits, in split order
__global__ void __launch_bounds__(256)
gram_i8_reduce_kernel(const double* __restrict__ partial, int m, int ntc, int ntiles, int splits, const int* __restrict__ use_exact,
                      double* __restrict__ G) {
    if (use_exact[0]) return;
    int ti, tj;
    upper_tile_i8(blockIdx.y, ntc, ti, tj);
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < TILE * I8_TN; e += gridDim.x * blockDim.x) {
        const int r = e / I8_TN, c = e - r * I8_TN;
        const int gi = ti * TILE + r, gj = tj * I8_TN + c;
        if (gi >= m || gj >= m || gj < gi) continue;
        double s = 0.0;
        for (int z = 0; z < splits; z++) s += partial[((size_t)z * ntiles + blockIdx.y) * TILE * I8_TN + e];
        G[(size_t)gi * m + gj] = s;
        G[(size_t)gj * m + gi] = s;
    }
}

// ---------------------------------------------------------------------------------------------
// C (m x n) = A (m x k) . B (k x n), bond-sized k, one CTA per 128 x BN output tile
// ---------------------------------------------------------------------------------------------
template <int BN, int STAGES>
struct GemmSmem {
    static constexpr int A_BYTES = 3 * PLANE_TILE;
    static constexpr int B_PLANE = BN * BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + 3 * B_PLANE;
    static constexpr int XPOSE_OFF = STAGES * STAGE_BYTES;              // per-warp 32 x 32 float transposes (row-major output),
    static constexpr int XPOSE_BYTES = (EPI_THREADS / 32) * 32 * 32 * 4;  // 16-byte chunks XOR-swizzled by the row
    static constexpr int BARRIER_OFF = XPOSE_OFF + XPOSE_BYTES;
    static constexpr int TOTAL = BARRIER_OFF + 256 + 1024;
};

// A_MN / B_MN: operand stored MN-major (planes are [k][mn]) instead of K-major ([mn][k]).
// OUT_T: write C transposed (C[n][m], lanes = consecutive m: coalesced) instead of row-major (through a
// per-warp shared-memory transpose so that rows leave in 128-byte lines).
template <int BN, int STAGES, bool A_MN, bool B_MN, bool OUT_T, class TC>
__global__ void __launch_bounds__(THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, int64_t m, int64_t n,
               int64_t k, TC* __restrict__ C, int64_t ldc) {
    // PERSISTENT: a CTA walks tiles blockIdx.x, blockIdx.x + gridDim.x, ... (n-tile fastest, so the CTAs running at
    // the same time share an A row block through L2 and write neighbouring column blocks of the same rows).  The stage
    // ring, the h.h ping-pong and the two correction accumulators run on through the tile boundaries: while the drain
    // warps write tile i, the copy thread is loading tile i + 1 / i + 2 and the MMA thread is up to two k-tiles ahead.
    // TMEM columns: [0, BN) h.h buffer 0, [BN, 2 BN) h.h buffer 1, [2 BN, 3 BN) / [3 BN, 4 BN) corrections of even / odd tiles.
    using S = GemmSmem<BN, STAGES>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + S::BARRIER_OFF);
    uint64_t* empty = full + STAGES;
    uint64_t* hh_full = empty + STAGES;        // [2]
    uint64_t* hh_empty = hh_full + 2;          // [2]
    uint64_t* rest_full = hh_empty + 2;        // [2]
    uint64_t* rest_empty = rest_full + 2;      // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rest_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nk = (int)((k + BK - 1) / BK);
    const int64_t ntn = (n + BN - 1) / BN, n_tiles = ((m + TILE - 1) / TILE) * ntn;
    constexpr uint32_t TMEM_COLS = 4 * BN;     // 256 or 512

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&map_a);
        tma_prefetch_desc(&map_b);
        for (int s = 0; s < STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < 2; b++) {
            mbar_init(&hh_full[b], 1);
            mbar_init(&hh_empty[b], EPI_THREADS / 32);
            mbar_init(&rest_full[b], 1);
            mbar_init(&rest_empty[b], EPI_THREADS / 32);
        }
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0 && lane == 0) {
        int g = 0;                                   // k-tiles issued so far (all tiles)
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int64_t m0 = (tile / ntn) * TILE, n0 = (tile % ntn) * BN;
            for (int kt = 0; kt < nk; kt++, g++) {
                const int s = g % STAGES;
                mbar_wait(&empty[s], ((g / STAGES) & 1) ^ 1);
                mbar_expect_tx(&full[s], S::STAGE_BYTES);
                uint8_t* st = smem + s * S::STAGE_BYTES;
                const int k0 = kt * BK;
#pragma unroll
                for (int p = 0; p < 3; p++) {
                    uint8_t* a = st + p * PLANE_TILE;
                    if constexpr (A_MN) {      // two boxes of 64 k-rows x 64 mn-columns
                        tma_load_3d(a, &map_a, &full[s], (int)m0, k0, p);
                        tma_load_3d(a + PLANE_TILE / 2, &map_a, &full[s], (int)m0 + 64, k0, p);
                    } else {                   // one box of 128 mn-rows x 64 k-columns
                        tma_load_3d(a, &map_a, &full[s], k0, (int)m0, p);
                    }
                    uint8_t* b = st + S::A_BYTES + p * S::B_PLANE;
                    if constexpr (B_MN) {
#pragma unroll
                        for (int h = 0; h < BN / 64; h++) tma_load_3d(b + h * 8192, &map_b, &full[s], (int)n0 + 64 * h, k0, p);
                    } else {
                        tma_load_3d(b, &map_b, &full[s], k0, (int)n0, p);
                    }
                }
            }
        }
    } else if (warp == 1 && lane == 0) {
        constexpr uint32_t idesc = instr_desc(TILE, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
        constexpr uint32_t A_STEP = A_MN ? 2048 : 32, B_STEP = B_MN ? 2048 : 32;
        constexpr uint32_t A_LBO = A_MN ? 8192 : 16, B_LBO = B_MN ? 8192 : 16;
        int g = 0, t_local = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, t_local++) {
            const int rb = t_local & 1;
            mbar_wait(&rest_empty[rb], ((t_local >> 1) & 1) ^ 1);
            for (int kt = 0; kt < nk; kt++, g++) {
                const int s = g % STAGES, hb = g & 1;
                mbar_wait(&hh_empty[hb], ((g >> 1) & 1) ^ 1);
                mbar_wait(&full[s], (g / STAGES) & 1);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + s * S::STAGE_BYTES), sb = sa + S::A_BYTES;
                const uint32_t d_hh = tmem_base + (uint32_t)hb * BN, d_rest = tmem_base + (uint32_t)(2 + rb) * BN;
#pragma unroll
                for (int ks = 0; ks < BK / UK; ks++)
                    umma_bf16(d_hh, smem_desc(sa + ks * A_STEP, A_LBO, 1024), smem_desc(sb + ks * B_STEP, B_LBO, 1024), idesc, ks != 0);
                umma_commit(&hh_full[hb]);
#pragma unroll
                for (int t = 0; t < 5; t++) {
#pragma unroll
                    for (int ks = 0; ks < BK / UK; ks++) {
                        const uint64_t da = smem_desc(sa + REST_A[t] * PLANE_TILE + ks * A_STEP, A_LBO, 1024);
                        const uint64_t db = smem_desc(sb + REST_B[t] * S::B_PLANE + ks * B_STEP, B_LBO, 1024);
                        umma_bf16(d_rest, da, db, idesc, (kt | t | ks) != 0);
                    }
                }
                umma_commit(&empty[s]);
                if (kt == nk - 1) umma_commit(&rest_full[rb]);
            }
        }
    } else if (warp >= 4) {
        const int q = warp & 3, half = (warp - 4) >> 2;
        constexpr int CPW = BN / 2;                       // columns per warp (the two halves split N)
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * CPW);
        // pointer arithmetic on the __shared__ array itself, so that the compiler keeps the address space (LDS / STS)
        const uint32_t raw_addr = smem_u32(smem_raw);
        float* xpose = reinterpret_cast<float*>(smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr) + S::XPOSE_OFF) + (warp - 4) * 32 * 32;
        float4* xpose4 = reinterpret_cast<float4*>(xpose);
        int g = 0, t_local = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, t_local++) {
            const int64_t m0 = (tile / ntn) * TILE, n0 = (tile % ntn) * BN;
            const int rb = t_local & 1;
            float acc[CPW];
#pragma unroll
            for (int i = 0; i < CPW; i++) acc[i] = 0.f;
            for (int kt = 0; kt < nk; kt++, g++) {
                const int hb = g & 1;
                mbar_wait(&hh_full[hb], (g >> 1) & 1);
                tc_fence_after();
#pragma unroll
                for (int gg = 0; gg < CPW / 32; gg++) {
                    uint32_t v[32];
                    tmem_ld32(lane_base + (uint32_t)(hb * BN + gg * 32), v);
#pragma unroll
                    for (int i = 0; i < 32; i++) acc[gg * 32 + i] += __uint_as_float(v[i]);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&hh_empty[hb]);
            }
            mbar_wait(&rest_full[rb], (t_local >> 1) & 1);
            tc_fence_after();
#pragma unroll
            for (int gg = 0; gg < CPW / 32; gg++) {
                uint32_t v[32];
                tmem_ld32(lane_base + (uint32_t)((2 + rb) * BN + gg * 32), v);
#pragma unroll
                for (int i = 0; i < 32; i++) acc[gg * 32 + i] += __uint_as_float(v[i]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&rest_empty[rb]);     // the accumulator is in registers: the MMA thread may reuse it
            const int64_t row = m0 + q * 32 + lane;
#pragma unroll
            for (int gg = 0; gg < CPW / 32; gg++) {
                const int col0 = half * CPW + gg * 32;
                if constexpr (OUT_T) {
                    if (row < m) {
#pragma unroll
                        for (int i = 0; i < 32; i++) {
                            const int64_t cn = n0 + col0 + i;
                            if (cn < n) C[cn * ldc + row] = (TC)acc[gg * 32 + i];
                        }
                    }
                } else {
                    // lane = row writes its 32 columns as eight 16-byte chunks, chunk j at slot j ^ (row & 7): conflict-free
                    // both for these stores and for the row-segment loads below
#pragma unroll
                    for (int j = 0; j < 8; j++)
                        xpose4[lane * 8 + (j ^ (lane & 7))] =
                            make_float4(acc[gg * 32 + 4 * j], acc[gg * 32 + 4 * j + 1], acc[gg * 32 + 4 * j + 2], acc[gg * 32 + 4 * j + 3]);
                    __syncwarp();
                    const bool interior = m0 + TILE <= m && n0 + BN <= n;
                    if (std::is_same<TC, float>::value && interior && (ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(C) & 15) == 0) {
                        // a quarter-warp writes one 128-byte row segment, the warp four rows per instruction
                        const int c4 = lane & 7;
                        float* crow = reinterpret_cast<float*>(C) + (m0 + q * 32 + (lane >> 3)) * ldc + n0 + col0 + 4 * c4;
#pragma unroll
                        for (int jj = 0; jj < 8; jj++) {
                            const int r = jj * 4 + (lane >> 3);
                            const float4 v = xpose4[r * 8 + (c4 ^ (r & 7))];
                            __stcs(reinterpret_cast<float4*>(crow), v);
                            crow += 4 * ldc;
                        }
                    } else {
                        const int64_t cn = n0 + col0 + lane;
                        const int chunk = lane >> 2, within = lane & 3;
#pragma unroll 4
                        for (int r = 0; r < 32; r++) {
                            const int64_t rr = m0 + q * 32 + r;
                            if (rr < m && cn < n) C[rr * ldc + cn] = (TC)xpose[r * 32 + ((chunk ^ (r & 7)) << 2) + within];
                        }
                    }
                    __syncwarp();
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

// 3-d tensor map of a stack of planes: dims {cols, rows, planes}, strides {row, plane} in bytes, zero fill outside.
// `what` names the operand in the error text.
static int encode_map(CUtensorMap* map, CUtensorMapDataType type, const void* base, const cuuint64_t (&dims)[3],
                      const cuuint64_t (&strides)[2], const cuuint32_t (&box)[3], CUtensorMapSwizzle swizzle, const char* what) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) { set_error("tc: cuTensorMapEncodeTiled is not available from the driver"); return NDMPS_ERR_CUDA; }
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(map, type, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("tc: cuTensorMapEncodeTiled (%s) failed (%d): %llu x %llu x %llu, row pitch %llu B", what, (int)r,
                  (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)dims[2], (unsigned long long)strides[0]);
        return NDMPS_ERR_CUDA;
    }
    return NDMPS_OK;
}

// planes: bf16[3][rows][ldp]; box = 64 columns x box_rows rows x 1 plane, 128-byte swizzle
static int make_plane_map(CUtensorMap* map, const void* planes, int64_t rows, int64_t cols, int64_t ldp, int64_t plane_stride,
                          int box_rows) {
    return encode_map(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, planes, {(cuuint64_t)cols, (cuuint64_t)rows, 3},
                      {(cuuint64_t)ldp * 2, (cuuint64_t)plane_stride * 2}, {64, (cuuint32_t)box_rows, 1}, CU_TENSOR_MAP_SWIZZLE_128B,
                      "bf16x3 planes");
}

static inline int64_t round8(int64_t x) { return (x + 7) & ~int64_t(7); }

}  // namespace tc

// Split `src` (rows x cols, row stride ld_src) into planes in the workspace.
int tc_split(ndmps_ctx* ctx, const void* src, int dtype, int64_t rows, int64_t cols, int64_t ld_src, double alpha,
             __nv_bfloat16** planes_out, int64_t* ldp_out, int64_t* plane_stride_out) {
    using namespace tc;
    const int64_t ldp = round8(cols), pstride = rows * ldp;
    __nv_bfloat16* planes = nullptr;
    NDMPS_TRY(ctx->ws.get<__nv_bfloat16>((size_t)(3 * pstride), &planes));
    const int64_t total = rows * (ldp >> 3);
    int64_t want = (total + 255) / 256, cap = (int64_t)ctx->sm_count * 16;
    const int g = (int)(want < 1 ? 1 : (want < cap ? want : cap));
    if (dtype == NDMPS_F32)
        split_planes_kernel<float><<<g, 256, 0, ctx->stream>>>((const float*)src, rows, cols, ld_src, alpha, planes, ldp, pstride);
    else
        split_planes_kernel<double><<<g, 256, 0, ctx->stream>>>((const double*)src, rows, cols, ld_src, alpha, planes, ldp, pstride);
    NDMPS_LAUNCH_CHECK(ctx);
    *planes_out = planes;
    *ldp_out = ldp;
    *plane_stride_out = pstride;
    return NDMPS_OK;
}

// G = M M^T from the float32 unfolding `mat` (rows x cols, row stride ld).  *done = false: shape not eligible.
// Launches BOTH the sliced-integer tensor-core Gram and the exact FP64-pipe Gram; a device-side flag set by the
// row-scaling pass lets exactly one of them run (the other returns at once), so no host round trip is needed.
// *dg receives the digits and the flag, for a projection of the same unfolding (proj_tc_digits).
int gram_tc(ndmps_ctx* ctx, const void* mat, int64_t rows, int64_t cols, int64_t ld, int dtype, double* g_dev, TcDigits* dg,
            bool* done) {
    using namespace tc;
    *done = false;
    if (dtype != NDMPS_F32 || rows < 64 || rows > 4096 || cols < 2048) return NDMPS_OK;
    if ((ld & 3) != 0 || (reinterpret_cast<uintptr_t>(mat) & 15) != 0) return NDMPS_OK;      // the FP64-pipe fallback needs it
    // 1. row statistics -> power-of-two row scales + the exactness flag
    int64_t chunks = ((int64_t)ctx->sm_count * 8 + rows - 1) / rows;
    {
        const int64_t max_chunks = (cols + 4095) / 4096;
        if (chunks > max_chunks) chunks = max_chunks;
        if (chunks < 1) chunks = 1;
    }
    int64_t per = (cols + chunks - 1) / chunks;
    per = (per + 3) & ~int64_t(3);
    chunks = (cols + per - 1) / per;
    double* stats = nullptr;
    int *sc = nullptr, *use_exact = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)(3 * rows * chunks), &stats));
    NDMPS_TRY(ctx->ws.get<int>((size_t)rows, &sc));
    NDMPS_TRY(ctx->ws.get<int>(4, &use_exact));
    row_stats_kernel<<<dim3((unsigned)rows, (unsigned)chunks), 256, 0, ctx->stream>>>((const float*)mat, cols, ld, per, stats);
    NDMPS_LAUNCH_CHECK(ctx);
    row_scale_kernel<<<1, 256, 0, ctx->stream>>>(stats, rows, (int)chunks, sc, use_exact);
    NDMPS_LAUNCH_CHECK(ctx);
    // 2. five int8 digit planes
    const int64_t ldp = (cols + 15) & ~int64_t(15), pstride = rows * ldp;
    int8_t* digits = nullptr;
    NDMPS_TRY(ctx->ws.get<int8_t>((size_t)(I8_PLANES * pstride), &digits));
    {
        const int64_t total = rows * (ldp >> 4);
        int64_t want = (total + 255) / 256, cap = (int64_t)ctx->sm_count * 16;
        split_i8_kernel<<<(int)(want < 1 ? 1 : (want < cap ? want : cap)), 256, 0, ctx->stream>>>((const float*)mat, rows, cols, ld, sc, use_exact,
                                                                                                digits, ldp, pstride);
        NDMPS_LAUNCH_CHECK(ctx);
    }
    // 3. digit products on the integer tensor cores
    CUtensorMap map;
    NDMPS_TRY(encode_map(&map, CU_TENSOR_MAP_DATA_TYPE_UINT8, digits, {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)I8_PLANES},
                         {(cuuint64_t)ldp, (cuuint64_t)pstride}, {(cuuint32_t)I8_BK, 64, 1}, CU_TENSOR_MAP_SWIZZLE_64B, "int8 digits"));
    const int m = (int)rows, ntr = (m + TILE - 1) / TILE, ntc = (m + I8_TN - 1) / I8_TN;
    int ntiles = 0;
    for (int ti = 0; ti < ntr; ti++) ntiles += ntc - 2 * ti > 0 ? ntc - 2 * ti : 0;
    // one CTA per SM and wave; more than one wave of shorter CTAs packs better beside the eigen-solver CTAs of the other
    // volumes in flight (option tc_waves)
    int64_t splits = (int64_t)ctx->sm_count * (ctx->opt_tc_waves > 0 ? ctx->opt_tc_waves : 1) / ntiles;
    if (splits < 1) splits = 1;
    int64_t k_per = (cols + splits - 1) / splits;
    k_per = ((k_per + I8_BK - 1) / I8_BK) * I8_BK;
    splits = (cols + k_per - 1) / k_per;
    double* partial = nullptr;
    NDMPS_TRY(ctx->ws.get<double>((size_t)splits * ntiles * TILE * I8_TN, &partial));
    NDMPS_TRY(raise_dynamic_smem((const void*)gram_i8_kernel, ctx->device, GramI8Smem::TOTAL));
    dim3 grid((unsigned)ntiles, (unsigned)splits);
    gram_i8_kernel<<<grid, THREADS, GramI8Smem::TOTAL, ctx->stream>>>(map, ntc, m, cols, k_per, sc, use_exact, partial);
    NDMPS_LAUNCH_CHECK(ctx);
    ctx->tc_launches++;
    dim3 rgrid(8, (unsigned)ntiles);
    gram_i8_reduce_kernel<<<rgrid, 256, 0, ctx->stream>>>(partial, m, ntc, ntiles, (int)splits, use_exact, g_dev);
    NDMPS_LAUNCH_CHECK(ctx);
    *dg = {digits, sc, use_exact, ldp, pstride, rows, cols};
    // 4. the exact kernel: runs only when the flag is set
    bool exact_ok = false;
    NDMPS_TRY(gram_dmma(ctx, mat, rows, cols, ld, dtype, g_dev, &exact_ok, use_exact));
    NDMPS_REQUIRE(exact_ok, "gram_tc: the FP64-pipe fallback declined a %lld x %lld unfolding", (long long)rows, (long long)cols);
    *done = true;
    return NDMPS_OK;
}

// T (r x C, row-major ldt) = P^T M on the digit planes gram_tc made of M (rows D x cols C), P: D x r float64 row-major.
// *done = false: the digits are not known to be exact (the Gram fell back to the FP64 pipe, or did not slice M) - the
// caller takes the bf16x3 route.  The exactness flag must have reached the host (ttsvd copies it beside the eigenvalues).
int proj_tc_digits(ndmps_ctx* ctx, const TcDigits& dg, const double* P, int64_t r, void* T, int dtype_t, int64_t ldt, bool* done) {
    using namespace tc;
    *done = false;
    const int64_t D = dg.rows, C = dg.cols;
    if (dg.exact_host != 0 || D > 4096 || r < 1 || C < TILE) return NDMPS_OK;
    // digits of the scaled columns of P: [digit][i][k], k padded to 16
    const int64_t ldk = (D + 15) & ~int64_t(15), bstride = r * ldk;
    int8_t* bdig = nullptr;
    int* tcs = nullptr;
    NDMPS_TRY(ctx->ws.get<int8_t>((size_t)(I8_PLANES * bstride), &bdig));
    NDMPS_TRY(ctx->ws.get<int>((size_t)r, &tcs));
    split_i8_proj_kernel<<<(unsigned)r, 256, 0, ctx->stream>>>(P, D, r, dg.sc, bdig, ldk, bstride, tcs);
    NDMPS_LAUNCH_CHECK(ctx);
    CUtensorMap map_y, map_b;
    NDMPS_TRY(encode_map(&map_y, CU_TENSOR_MAP_DATA_TYPE_UINT8, dg.digits, {(cuuint64_t)C, (cuuint64_t)D, (cuuint64_t)I8_PLANES},
                         {(cuuint64_t)dg.ldp, (cuuint64_t)dg.pstride}, {(cuuint32_t)TILE, (cuuint32_t)I8_BK, 1}, CU_TENSOR_MAP_SWIZZLE_128B,
                         "projection digits"));
    NDMPS_TRY(encode_map(&map_b, CU_TENSOR_MAP_DATA_TYPE_UINT8, bdig, {(cuuint64_t)D, (cuuint64_t)r, (cuuint64_t)I8_PLANES},
                         {(cuuint64_t)ldk, (cuuint64_t)bstride}, {(cuuint32_t)I8_BK, 64, 1}, CU_TENSOR_MAP_SWIZZLE_64B, "projector digits"));
    dim3 grid((unsigned)((C + TILE - 1) / TILE), (unsigned)((r + I8_TN - 1) / I8_TN));
    if (dtype_t == NDMPS_F32) {
        NDMPS_TRY(raise_dynamic_smem((const void*)proj_i8_kernel<float>, ctx->device, ProjI8Smem::TOTAL));
        proj_i8_kernel<float><<<grid, THREADS, ProjI8Smem::TOTAL, ctx->stream>>>(map_y, map_b, C, r, D, tcs, (float*)T, ldt);
    } else {
        NDMPS_TRY(raise_dynamic_smem((const void*)proj_i8_kernel<double>, ctx->device, ProjI8Smem::TOTAL));
        proj_i8_kernel<double><<<grid, THREADS, ProjI8Smem::TOTAL, ctx->stream>>>(map_y, map_b, C, r, D, tcs, (double*)T, ldt);
    }
    NDMPS_LAUNCH_CHECK(ctx);
    ctx->tc_launches++;
    *done = true;
    return NDMPS_OK;
}

namespace tc {

template <int BN, int STAGES, bool A_MN, bool B_MN, bool OUT_T, class TC>
static int launch_gemm(ndmps_ctx* ctx, const CUtensorMap& ma, const CUtensorMap& mb, int64_t m, int64_t n, int64_t k, TC* c, int64_t ldc) {
    using S = GemmSmem<BN, STAGES>;
    auto kern = gemm_tc_kernel<BN, STAGES, A_MN, B_MN, OUT_T, TC>;
    NDMPS_TRY(raise_dynamic_smem((const void*)kern, ctx->device, S::TOTAL));
    const int64_t tiles = ((m + TILE - 1) / TILE) * ((n + BN - 1) / BN);
    const unsigned grid = (unsigned)(tiles < ctx->sm_count ? tiles : ctx->sm_count);      // one persistent CTA per SM
    kern<<<grid, THREADS, S::TOTAL, ctx->stream>>>(ma, mb, m, n, k, c, ldc);
    NDMPS_LAUNCH_CHECK(ctx);
    ctx->tc_launches++;
    return NDMPS_OK;
}

}  // namespace tc

// C (m x n, row-major ldc; or n x m when out_t) = A . B on the tensor cores.
//   a: m x k with strides (a_rs, a_cs); b: k x n with strides (b_rs, b_cs); one stride of each must be 1.
// Operands are split into planes here (the big one costs a pass; bond-sized ones are negligible).
int gemm_tc(ndmps_ctx* ctx, int64_t m, int64_t n, int64_t k, double alpha, const void* a, int dtype_a, int64_t a_rs, int64_t a_cs,
            const void* b, int dtype_b, int64_t b_rs, int64_t b_cs, void* c, int dtype_c, int64_t ldc, bool out_t, bool* done) {
    using namespace tc;
    *done = false;
    if (m < 128 || n < 8 || k < 8 || (a_cs != 1 && a_rs != 1) || (b_cs != 1 && b_rs != 1)) return NDMPS_OK;
    if (m >= (int64_t(1) << 31) || n >= (int64_t(1) << 31) || k >= (int64_t(1) << 31)) return NDMPS_OK;
    const bool a_mn = a_cs != 1;                 // a[i * a_rs + j]: K contiguous -> K-major; else M contiguous -> MN-major
    const bool b_mn = b_cs == 1 && b_rs != 1;    // b[j * b_rs + l]: N contiguous -> MN-major; K contiguous (b_rs == 1) -> K-major
    // plane matrices as stored: K-major A planes are [m][k]; MN-major A planes are [k][m]; same for B with n
    __nv_bfloat16 *pa = nullptr, *pb = nullptr;
    int64_t lda = 0, sa = 0, ldb = 0, sb = 0;
    if (a_mn) NDMPS_TRY(tc_split(ctx, a, dtype_a, k, m, a_cs, alpha, &pa, &lda, &sa));
    else NDMPS_TRY(tc_split(ctx, a, dtype_a, m, k, a_rs, alpha, &pa, &lda, &sa));
    if (b_mn) NDMPS_TRY(tc_split(ctx, b, dtype_b, k, n, b_rs, 1.0, &pb, &ldb, &sb));
    else NDMPS_TRY(tc_split(ctx, b, dtype_b, n, k, b_cs, 1.0, &pb, &ldb, &sb));
    CUtensorMap ma, mb;
    if (a_mn) NDMPS_TRY(make_plane_map(&ma, pa, k, m, lda, sa, 64));
    else NDMPS_TRY(make_plane_map(&ma, pa, m, k, lda, sa, TILE));
    const int bn = n <= 64 ? 64 : 128;
    if (b_mn) NDMPS_TRY(make_plane_map(&mb, pb, k, n, ldb, sb, 64));
    else NDMPS_TRY(make_plane_map(&mb, pb, n, k, ldb, sb, bn));
#define NDMPS_TC_GO(BN, ST, AMN, BMN)                                                                                          \
    do {                                                                                                                       \
        if (dtype_c == NDMPS_F32) {                                                                                            \
            if (out_t) NDMPS_TRY((launch_gemm<BN, ST, AMN, BMN, true, float>(ctx, ma, mb, m, n, k, (float*)c, ldc)));          \
            else NDMPS_TRY((launch_gemm<BN, ST, AMN, BMN, false, float>(ctx, ma, mb, m, n, k, (float*)c, ldc)));               \
        } else {                                                                                                               \
            if (out_t) NDMPS_TRY((launch_gemm<BN, ST, AMN, BMN, true, double>(ctx, ma, mb, m, n, k, (double*)c, ldc)));        \
            else NDMPS_TRY((launch_gemm<BN, ST, AMN, BMN, false, double>(ctx, ma, mb, m, n, k, (double*)c, ldc)));             \
        }                                                                                                                      \
    } while (0)
    if (bn == 64) {
        if (a_mn && !b_mn) NDMPS_TC_GO(64, 2, true, false);
        else if (!a_mn && b_mn) NDMPS_TC_GO(64, 2, false, true);
        else if (!a_mn && !b_mn) NDMPS_TC_GO(64, 2, false, false);
        else NDMPS_TC_GO(64, 2, true, true);
    } else {
        if (a_mn && !b_mn) NDMPS_TC_GO(128, 2, true, false);
        else if (!a_mn && b_mn) NDMPS_TC_GO(128, 2, false, true);
        else if (!a_mn && !b_mn) NDMPS_TC_GO(128, 2, false, false);
        else NDMPS_TC_GO(128, 2, true, true);
    }
#undef NDMPS_TC_GO
    *done = true;
    return NDMPS_OK;
}

}  // namespace ndmps
