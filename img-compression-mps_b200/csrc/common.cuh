// Shared host/device plumbing of libndmps_sm100.so (context, workspace arena,
// error reporting, warp/block reductions).  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>

#include "../../include/ndmps.h"

#define NDMPS_MAX_DIGITS 40

struct DigitList {
    int n;                              // number of digits (after dropping extent-1 and merging)
    uint32_t extent[NDMPS_MAX_DIGITS];  // destination extents, outermost first
    int64_t stride[NDMPS_MAX_DIGITS];   // source stride (elements) of each digit
    int32_t shift[NDMPS_MAX_DIGITS];    // log2(extent) if power of two else -1
};

// Tiled form of one permutation direction (permute.cu): a tile is the set of digits A (the
// innermost destination digits: a contiguous destination run of `pa` elements) united with B
// (the smallest-stride source digits: a contiguous source run of `pb` elements).
struct TilePlan {
    bool ok = false;
    int tile = 0;                        // elements per tile
    int pa = 0, pb = 0;                  // contiguous run lengths on the destination / source side
    int n_outer = 0;                     // digits outside the tile
    uint32_t outer_extent[NDMPS_MAX_DIGITS];
    int64_t outer_dst[NDMPS_MAX_DIGITS];
    int64_t outer_src[NDMPS_MAX_DIGITS];
    int64_t n_tiles = 0;
    int conflict = 0;                    // worst shared-memory bank conflict degree of the scatter
    std::vector<int64_t> hi_src;         // tile/pb source offsets of the source runs (read order)
    std::vector<int64_t> hi_dst;         // tile/pa destination offsets of the destination runs (write order)
    std::vector<uint16_t> pos;           // read index -> (skewed) shared-memory slot
    // device copies, uploaded on first use PER DEVICE (a plan is shared by host threads that may drive different GPUs)
    struct DevTables {
        int device = -1;
        int64_t* hi_src = nullptr;
        int64_t* hi_dst = nullptr;
        uint16_t* pos = nullptr;
    };
    std::vector<DevTables> dev;          // guarded by the upload mutex in permute.cu; read through upload_tile_plan only
};

// Register-only form of one permutation direction for shapes whose every factor is a power of two (permute.cu):
// the permutation is then a permutation of the BITS of the element offset.  A thread owns the eight elements spanned by
// destination bits {0, 1, pair}: two 16-byte loads (source rows 1 << row_shift apart), two 16-byte stores
// (1 << pair_shift apart).  The other bits index the thread: [0,5) lane, [5,8) warp, [8,10) unrolled steps, the rest CTA.
struct BitPlan {
    bool ok = false;
    int nbits = 0;                       // log2(elements)
    int row_shift = 0;                   // source bit of destination bit 1
    int pair_shift = 0;                  // destination bit that holds source bit 1
    int n_idx = 0;                       // nbits - 3
    int8_t dst_bit[48] = {0};            // index bit t -> destination bit
    int8_t src_bit[48] = {0};            // index bit t -> source bit
};

struct ndmps_plan {
    int ndim = 0, levels = 0;
    int64_t shape[8] = {0};
    int64_t factors[NDMPS_MAX_DIGITS] = {0};  // (levels, ndim)
    int64_t site_dims[NDMPS_MAX_DIGITS] = {0};
    int64_t total = 0;
    DigitList enc = {};                 // destination = site order, source = volume
    DigitList dec = {};                 // destination = volume, source = site order
    bool identity = false;
    TilePlan enc_tile, dec_tile;
    BitPlan enc_bits, dec_bits;
};

namespace ndmps {

void set_error(const char* fmt, ...);

#define NDMPS_CUDA_TRY(expr)                                                                 \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            ::ndmps::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return NDMPS_ERR_CUDA;                                                           \
        }                                                                                    \
    } while (0)

#define NDMPS_TRY(expr)                 \
    do {                                \
        int _rc = (expr);               \
        if (_rc != NDMPS_OK) return _rc; \
    } while (0)

#define NDMPS_REQUIRE(cond, ...)                    \
    do {                                            \
        if (!(cond)) {                              \
            ::ndmps::set_error(__VA_ARGS__);        \
            return NDMPS_ERR_INVALID;               \
        }                                           \
    } while (0)

// check the launch that was just issued
#define NDMPS_LAUNCH_CHECK(ctx)                                                              \
    do {                                                                                     \
        (ctx)->launches++;                                                                   \
        cudaError_t _e = cudaGetLastError();                                                 \
        if (_e != cudaSuccess) {                                                             \
            ::ndmps::set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return NDMPS_ERR_CUDA;                                                           \
        }                                                                                    \
    } while (0)

// Grow-only device arena.  alloc() is a bump pointer; when a chunk runs out a new
// one is added (cudaMalloc) and on the next reset() the chunks are merged into
// one allocation of the total size, so steady state never allocates.
struct Arena {
    struct Chunk { char* base; size_t cap; size_t used; };
    std::vector<Chunk> chunks;
    size_t high_water = 0;
    size_t cur_total = 0;
    uint64_t generation = 0;            // bumped by reset(): cached workspace pointers of an older generation are dead

    int reset(cudaStream_t stream);
    int alloc(size_t bytes, void** out);
    void release();
    template <class T> int get(size_t count, T** out) {
        void* p = nullptr;
        int rc = alloc(count * sizeof(T), &p);
        *out = static_cast<T*>(p);
        return rc;
    }
};

}  // namespace ndmps

// ---- per-stage device timing (CUDA events on the launching stream; off by default) ----
enum NdmpsStage { ST_PERMUTE = 0, ST_GRAM, ST_EIG, ST_PROJECT, ST_GLUE, ST_CONTRACT, ST_DCT, ST_METRIC, ST_COUNT };

struct ndmps_ctx {
    cudaStream_t stream = nullptr;
    ndmps::Arena ws;
    int device = 0;
    int sm_count = 148;
    size_t smem_optin = 0;
    int64_t launches = 0;
    // pinned host scratch for small D2H readbacks (eigenvalues, flags, scalars)
    double* pinned = nullptr;
    size_t pinned_doubles = 0;
    // options: ndmps_ctx_set_option in ndmps.h lists names, defaults and values
    int64_t opt_gram_path = 0;      // 0 auto, 2 SIMT, 3 tcgen05
    int64_t opt_tc = 1;             // tcgen05 contractions for float32 payloads
    int64_t opt_gemm_out_t = 0;     // test hook: ndmps_gemm writes C transposed
    // int8 digit planes of the unfolding the tcgen05 Gram sliced last (workspace memory: valid until the next ws.reset);
    // the projection of the same sweep step multiplies the same digits.  exact_host: the device-side "use the FP64 pipe"
    // flag once it has been copied to the host beside the eigenvalues (-1: not yet known)
    struct {
        const void* src = nullptr; int64_t rows = 0, cols = 0, ld = 0; void* digits = nullptr; int64_t ldp = 0, pstride = 0;
        const int* sc = nullptr; const int* use_exact = nullptr; uint64_t gen = 0; int exact_host = -1;
    } tc_digits;
    bool tc_sweep = false;          // set by the sweep while the tcgen05 Gram / projection are admissible (float32, bond cap)
    int64_t opt_gemm_path = 0;      // 0 auto, 2 SIMT
    int64_t opt_permute_path = 0;   // 0 auto, 1 tiles, 2 gather
    int64_t opt_eig_topk = 1;             // leading-eigenpair solver for capped bonds
    int64_t opt_topk_cluster = 1;         // cluster tridiagonalisation for n <= 512
    int64_t cluster_launches = 0;
    int64_t opt_tc_waves = 1;             // waves of gram_i8 CTAs
    int64_t opt_ssim_exact = 0;           // float64 SSIM for float32 inputs
    int64_t opt_blocking_sync = 0;        // host waits: 0 spin, 3 watch a pinned word
    int64_t opt_verbose = 0;
    volatile unsigned* wait_flag = nullptr;   // pinned word the stream writes its sequence numbers into (wait mode 3)
    unsigned wait_seq = 0;
    // stats of the last eigensolve / sweep (for tests and profiling)
    int last_eig_sweeps = 0;
    double eig_flops = 0.0;        // 7 n per rotation x pairs x sweeps (+ n r^2 for the Cholesky), accumulated
    int64_t eig_calls = 0;
    int64_t tc_launches = 0;       // tcgen05 kernels launched (tc_gemm.cu)
    // stage profiler
    bool profile = false;
    struct Pending { int stage; cudaEvent_t beg, end; };
    std::vector<Pending> pending;
    double stage_ms[ST_COUNT] = {0};
    int64_t stage_calls[ST_COUNT] = {0};
};

namespace ndmps {

int ensure_pinned(ndmps_ctx* ctx, size_t doubles);
// small device -> host copy into the pinned scratch, enqueued on the context's stream (api.cu: SM stores, not the copy engine)
int readback(ndmps_ctx* ctx, void* pinned_dst, const void* dev_src, size_t bytes);
int copy_small(ndmps_ctx* ctx, void* dev_dst, const void* dev_src, size_t bytes);
// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute of a kernel: raise it to `bytes` once per
// (kernel, device), from any host thread (the largest value set so far is remembered under a mutex).
int raise_dynamic_smem(const void* kernel, int device, int bytes);
// wait for everything enqueued on the context's stream (spinning cudaStreamSynchronize, or watching a pinned word)
cudaError_t stream_wait(ndmps_ctx* ctx);

// RAII stage marker: records an event pair around a leaf stage when profiling is on
struct StageScope {
    ndmps_ctx* ctx;
    cudaEvent_t beg = nullptr, end = nullptr;
    int stage;
    StageScope(ndmps_ctx* c, int st) : ctx(c), stage(st) {
        if (!ctx->profile) return;
        cudaEventCreate(&beg);
        cudaEventCreate(&end);
        cudaEventRecord(beg, ctx->stream);
    }
    ~StageScope() {
        if (!beg) return;
        cudaEventRecord(end, ctx->stream);
        ctx->pending.push_back({stage, beg, end});
    }
};
int profile_collect(ndmps_ctx* ctx);

static inline size_t dtype_size(int dtype) { return dtype == NDMPS_F64 ? 8 : 4; }
static inline bool dtype_ok(int dtype) { return dtype == NDMPS_F32 || dtype == NDMPS_F64; }

// ---- internal entry points shared between translation units -------------------
// generic strided GEMM, float64 accumulation; C row-major with ldc.
int gemm(ndmps_ctx* ctx, int64_t m, int64_t n, int64_t k, double alpha,
         const void* a, int dtype_a, int64_t a_rs, int64_t a_cs,
         const void* b, int dtype_b, int64_t b_rs, int64_t b_cs,
         void* c, int dtype_c, int64_t ldc);
int gram(ndmps_ctx* ctx, const void* m, int64_t rows, int64_t cols, int64_t ld, int dtype, int side, double* g_dev);
// tcgen05 paths (tc_gemm.cu); *done = false when the shape is not eligible
int gram_tc(ndmps_ctx* ctx, const void* mat, int64_t rows, int64_t cols, int64_t ld, int dtype, double* g_dev, bool* done);
int proj_tc_digits(ndmps_ctx* ctx, const void* mat, int64_t D, int64_t C, int64_t ld, const double* P, int64_t r, void* T, int dtype_t,
                   int64_t ldt, bool* done);
int gemm_tc(ndmps_ctx* ctx, int64_t m, int64_t n, int64_t k, double alpha, const void* a, int dtype_a, int64_t a_rs, int64_t a_cs,
            const void* b, int dtype_b, int64_t b_rs, int64_t b_cs, void* c, int dtype_c, int64_t ldc, bool out_t, bool* done);
// tol_override > 0 loosens the relative off-diagonal threshold (float32 payloads do not need 1e-15)
int eigh(ndmps_ctx* ctx, double* a_dev, int64_t n, double* evals_dev, double* evecs_dev, double tol_override = 0.0);
// diag_tol > 0: a matrix whose off-diagonal entries are all below diag_tol x max |diagonal| is taken as diagonal
int eigh_small_async(ndmps_ctx* ctx, double* a_dev, int n, double* evals_dev, double* evecs_dev, float quad_stop2, int** info_dev,
                     double diag_tol = 0.0);
// leading k eigenpairs (eig_topk.cu); out_dev: k Ritz values, trace(G), rank-loss count
int eigh_topk(ndmps_ctx* ctx, const double* g_dev, int64_t n, int64_t k, double* out_dev, double* evecs_dev, int64_t ldu, bool* done);
// Cooperative (grid-barrier) kernels of several contexts may be in flight at once (batch.py).  Their
// CTAs spin at barriers, so the sum of what is launched must fit the machine: a launch books the SMs
// its grid needs (grid / resident CTAs per SM) in a process-wide gate and gives them back from a
// stream callback when the kernel has finished; a launch that does not fit waits on the host.
int cluster_fits(const void* kernel, int device, int cluster_ctas, int threads, bool* fits);
int coop_launch(ndmps_ctx* ctx, const void* fn, dim3 grid, dim3 block, void** args, size_t smem);
int minmax_device(ndmps_ctx* ctx, const void* x, int64_t n, int dtype, double* out_dev2);
int permute(ndmps_ctx* ctx, const ndmps_plan* plan, bool inverse, const void* src, void* dst, int dtype, double scale);

#ifdef __CUDACC__
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// block reductions; `scratch` must hold 32 doubles; result valid in thread 0
__device__ __forceinline__ double block_sum(double v, double* scratch) {
    v = warp_sum(v);
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane == 0) scratch[w] = v;
    __syncthreads();
    if (w == 0) {
        v = lane < nw ? scratch[lane] : 0.0;
        v = warp_sum(v);
    }
    return v;
}
__device__ __forceinline__ double block_max(double v, double* scratch) {
    v = warp_max(v);
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane == 0) scratch[w] = v;
    __syncthreads();
    if (w == 0) {
        v = lane < nw ? scratch[lane] : -INFINITY;
        v = warp_max(v);
    }
    return v;
}
__device__ __forceinline__ double block_min(double v, double* scratch) {
    v = warp_min(v);
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane == 0) scratch[w] = v;
    __syncthreads();
    if (w == 0) {
        v = lane < nw ? scratch[lane] : INFINITY;
        v = warp_min(v);
    }
    return v;
}
#endif

}  // namespace ndmps
