/*
 * ndmps.h - C ABI of libndmps_sm100.so, the B200 (sm_100a) device path under the
 * reference's NDMPS encode / compress / reconstruct API.
 *
 * The reference (Alandroid/img-compression-mps) is pure Python and has no FFI of
 * its own; the boundary it offers is the NDMPS class and the utils modules.  Every
 * entry point below therefore replaces one *step* of that Python path, cited as
 * file:line under src/imgcompressionmps/ of the reference.  The Python package in
 * img-compression-mps_b200/imgcompressionmps binds these with ctypes (see
 * INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - plain C types only: device pointers are `void*` / `double*`, sizes are
 *     int64_t, the CUDA stream is a `void*` holding a cudaStream_t.
 *   - every function returns 0 on success and a negative NDMPS_ERR_* code on
 *     failure; ndmps_last_error() returns a thread-local message.
 *   - the caller owns every buffer.  A context owns only a grow-only device
 *     workspace and the stream it launches on.  One context per host thread.
 *   - `dtype`: NDMPS_F32 or NDMPS_F64 for the payload (volumes, cores).  Small
 *     bond matrices (Gram, eigenvectors, transfer matrices) are always float64.
 *   - pointers named *_host are host memory and are written synchronously (the
 *     call synchronises the context's stream before returning).
 *   - array layouts are C order.  Cores are (left bond, physical, right bond).
 */
#ifndef NDMPS_H
#define NDMPS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NDMPS_F32 0
#define NDMPS_F64 1

#define NDMPS_OK               0
#define NDMPS_ERR_INVALID     -1   /* bad argument */
#define NDMPS_ERR_CUDA        -2   /* CUDA runtime error (message has the string) */
#define NDMPS_ERR_NOMEM       -3
#define NDMPS_ERR_CAPACITY    -4   /* caller-provided output buffer too small */
#define NDMPS_ERR_NOCONV      -5   /* Jacobi eigensolver did not converge */

/* cutoff modes of the singular-value trim (quimb names; the reference uses
 * "rsum2" implicitly at core/ndmps.py:74 and "rel" at core/ndmps.py:106) */
#define NDMPS_CUT_ABS   1
#define NDMPS_CUT_REL   2
#define NDMPS_CUT_SUM2  3
#define NDMPS_CUT_RSUM2 4
#define NDMPS_CUT_SUM1  5
#define NDMPS_CUT_RSUM1 6

typedef struct ndmps_ctx  ndmps_ctx_t;
typedef struct ndmps_plan ndmps_plan_t;

/* ---- library / context -------------------------------------------------- */
int         ndmps_version(void);
const char* ndmps_last_error(void);
int ndmps_ctx_create(ndmps_ctx_t** out);
int ndmps_ctx_destroy(ndmps_ctx_t* ctx);
/* One context = one stream at a time = one workspace arena reused in stream order.  Changing the stream makes the new
 * one wait (event) for everything already queued on the old one. */
int ndmps_ctx_set_stream(ndmps_ctx_t* ctx, void* cuda_stream);
int ndmps_ctx_sync(ndmps_ctx_t* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int64_t ndmps_ctx_launch_count(const ndmps_ctx_t* ctx);
/* per-stage device time (CUDA events on the context's stream).  profile(1) turns the
 * event pairs on; stage_times() synchronises and returns accumulated ms / call counts
 * for the ndmps_stage_count() stages named by ndmps_stage_name(). */
int ndmps_ctx_profile(ndmps_ctx_t* ctx, int enable);
int ndmps_stage_count(void);
const char* ndmps_stage_name(int stage);
int ndmps_ctx_stage_times(ndmps_ctx_t* ctx, double* ms_out, int64_t* calls_out, int reset);
/* counters: "eig_flops" (rotation + factorisation flops of the bond eigensolves), "eig_calls",
 * "workspace_bytes" (arena high-water mark). */
int ndmps_ctx_get_stat(ndmps_ctx_t* ctx, const char* name, double* value_out, int reset);
/* options: name (default) values - what the option is for.  An unknown name, or a value outside the listed set of
 * permute_path / blocking_sync, returns NDMPS_ERR_INVALID.
 *   "gram_path" (0)      0 auto (tcgen05 in a capped float32 sweep, else the FP64 tensor pipe when the shape allows),
 *                        2 SIMT kernel, 3 tcgen05 - lets tests compare the Gram routes
 *   "gemm_path" (0)      0 FP64 tensor pipe when the shape allows, 2 SIMT only, 3 tcgen05 - lets tests compare the routes
 *   "gemm_out_t" (0)     1: ndmps_gemm writes C transposed through the tcgen05 epilogue - test hook
 *   "tc" (1)             0/1: tcgen05 contractions on bf16x3 planes for float32 payloads of a capped sweep / reconstruction
 *   "tc_waves" (1)       waves of integer-Gram CTAs (split-K factor = waves x SMs / tiles) - tests check it is the same bound
 *   "permute_path" (0)   0 register bit-permutation when the shape allows, else shared-memory tiles; 1 tiles always;
 *                        2 gather kernel - 1 and 2 are the references of the permutation tests
 *   "eig_topk" (1)       0/1: leading-eigenpair solver when a bond cap provably binds - 0, the full solver, is its reference
 *   "topk_cluster" (1)   0/1: n <= 512 tridiagonalisation as one thread-block cluster - 0 forces the grid-barrier kernel
 *                        that runs when the cluster does not fit the device
 *   "ssim_exact" (0)     0/1: float64 SSIM arithmetic for float32 inputs too - the reference of the SSIM tests
 *   "blocking_sync" (0)  host waits: 0 spin in cudaStreamSynchronize, 3 watch a pinned word the stream writes and yield
 *                        (more waiting host threads than cores: batch.VolumePipeline picks)
 *   "verbose" (0)        0/1: one line per eigensolve / sweep step on stderr - diagnostics
 * A context belongs to one host thread; several contexts (one per thread, each with its own stream) may run concurrently. */
int ndmps_ctx_set_option(ndmps_ctx_t* ctx, const char* name, int64_t value);

/* ---- K1: N-D volume <-> interleaved MPS site order ----------------------
 * Replaces utils/core.py:6-35,129-168 (gen_encoding_map +
 * hierarchical_block_indexing) and the fancy-index scatter / gather at
 * core/ndmps.py:66-71 and core/ndmps.py:144-148.  `factors` is the (levels, ndim)
 * array get_factorlist returns (utils/core.py:79-126), row-major.  The int64
 * encoding map is never materialised on the device. */
int ndmps_plan_create(int ndim, const int64_t* shape, int levels, const int64_t* factors,
                      ndmps_plan_t** out);
int ndmps_plan_destroy(ndmps_plan_t* plan);
int ndmps_plan_site_dims(const ndmps_plan_t* plan, int64_t* dims_out);
/* ndim, levels, shape (ndim values) and factor table (levels x ndim, row-major) of a plan; shape_out and factors_out
 * may be NULL, so a caller can read ndim and levels first (plans from ndmps_plan_coarse). */
int ndmps_plan_layout(const ndmps_plan_t* plan, int* ndim_out, int* levels_out, int64_t* shape_out, int64_t* factors_out);
/* host-only index check (no device work): source offsets the kernels read for
 * destination elements [first, first+count); inverse=0 encode, 1 decode. */
int ndmps_plan_debug_offsets(const ndmps_plan_t* plan, int inverse, int64_t first, int64_t count, int64_t* out_host);
/* host-only checks of the shared-memory tiling of the permutation (no device work):
 * info_out[6] = {tiled?, tile elements, destination run, source run, tiles, worst bank conflict};
 * apply_tiled walks the tile tables on int32 host arrays exactly as the kernel does. */
int ndmps_plan_debug_tile_info(const ndmps_plan_t* plan, int inverse, int64_t* info_out);
int ndmps_plan_debug_apply_tiled(const ndmps_plan_t* plan, int inverse, const int32_t* src_host, int32_t* dst_host);
/* host-only checks of the register bit-permutation used for power-of-two shapes (no device work):
 * info_out[7] = {has a bit plan?, log2(elements), source bit of destination bit 1, destination bit of source bit 1, CTAs,
 * contiguous destination run per CTA, contiguous source run per CTA}; apply_bits moves int32 host arrays with the
 * kernel's own thread -> offset function and register shuffle. */
int ndmps_plan_debug_bit_info(const ndmps_plan_t* plan, int inverse, int64_t* info_out);
int ndmps_plan_debug_apply_bits(const ndmps_plan_t* plan, int inverse, const int32_t* src_host, int32_t* dst_host);
/* dst[site order] = scale * src[volume order]   (scale folds the 1/||x|| of core/ndmps.py:60-61) */
int ndmps_encode(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* src, void* dst, int dtype, double scale);
/* dst[volume order] = src[site order] */
int ndmps_decode(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* src, void* dst, int dtype);

/* ---- reductions ---------------------------------------------------------- */
/* sum of squares (np.linalg.norm at core/ndmps.py:61 is its square root); n = 0 gives 0 and x may then be NULL */
int ndmps_sumsq(ndmps_ctx_t* ctx, const void* x, int64_t n, int dtype, double* out_host);
/* K12: [min, max] of each of `count` arrays (boundary_list, core/ndmps.py:75,82) */
int ndmps_minmax(ndmps_ctx_t* ctx, const void* const* arrays, const int64_t* sizes, int count, int dtype,
                 double* out_host /* 2*count */);
/* K10: out = [sum (a-b)^2, max(a)]  (utils/metrics.py:143-146) */
int ndmps_psnr_terms(ndmps_ctx_t* ctx, const void* a, const void* b, int64_t n, int dtype, double* out_host);

/* ---- K11: orthonormal DCT-II / DCT-III along the last axis ----------------
 * scipy.fftpack.dct(x, norm="ortho") / idct at core/ndmps.py:63,153. */
int ndmps_dct_last_axis(ndmps_ctx_t* ctx, const void* src, void* dst, int64_t lines, int64_t n, int inverse, int dtype);
/* Block mean of the inverse transform, without the n-element lines: dst (lines x n/block) = src (lines x n) . B with
 * B[k, j] = (1/block) sum_{t in block j} C[k, t], C the orthonormal DCT-III matrix (built on the device in float64).
 * tcgen05 (bf16x3) for float32 when lines * n >= 2^20, as ndmps_dct_last_axis.  block must be >= 1 and divide n,
 * otherwise NDMPS_ERR_INVALID.  block = 1 is ndmps_dct_last_axis(inverse = 1). */
int ndmps_idct_block_mean_last_axis(ndmps_ctx_t* ctx, const void* src, void* dst, int64_t lines, int64_t n, int64_t block,
                                    int dtype);

/* ---- building blocks of the sweep (exported for tests and profiling) ------ */
/* G (float64, device) = M M^T (side 0, rows x rows) or M^T M (side 1, cols x cols);
 * M is rows x cols, row-major with leading dimension ld. */
int ndmps_gram(ndmps_ctx_t* ctx, const void* m, int64_t rows, int64_t cols, int64_t ld, int dtype, int side,
               double* g_dev);
/* symmetric eigen-decomposition by parallel one-sided Jacobi, float64.
 * a_dev (n x n) is destroyed.  evals_dev: n values, descending.  evecs_dev:
 * n x n row-major, column j is the j-th eigenvector. */
int ndmps_eigh(ndmps_ctx_t* ctx, double* a_dev, int64_t n, double* evals_dev, double* evecs_dev, int* sweeps_out_host);
/* Leading k eigenpairs of a symmetric positive semi-definite matrix (what a capped bond needs:
 * quimb's max_bond at core/ndmps.py:74,104-106 keeps the k largest singular triplets and only the
 * total weight of the rest).  a_dev (n x n) is NOT modified.  evals_dev: k + 2 values = k
 * eigenvalues descending, trace(a), and a health flag (0 = ok).  evecs_dev: n x k row-major,
 * column j is the j-th eigenvector.  Supported: 96 <= n <= 4096, 2k <= n, k <= ~100;
 * other shapes return NDMPS_ERR_INVALID (use ndmps_eigh). */
int ndmps_eigh_topk(ndmps_ctx_t* ctx, const double* a_dev, int64_t n, int64_t k, double* evals_dev, double* evecs_dev);
/* C (m x n, ldc) = alpha * A(m x k) * B(k x n) with arbitrary element strides, float64 accumulation. */
int ndmps_gemm(ndmps_ctx_t* ctx, int64_t m, int64_t n, int64_t k, double alpha,
               const void* a, int dtype_a, int64_t a_rs, int64_t a_cs,
               const void* b, int dtype_b, int64_t b_rs, int64_t b_cs,
               void* c, int dtype_c, int64_t ldc);

/* ---- K2-K5: left -> right TT-SVD sweep ------------------------------------
 * qtn.MatrixProductState.from_dense(dense, dims) at core/ndmps.py:74 (quimb
 * 1.9.0 defaults: cutoff 1e-10, NDMPS_CUT_RSUM2, renorm 2, weight absorbed to
 * the right).  dense: prod(dims) elements in site order (read only).
 * cores_out[i]: device buffer of core_cap[i] elements; core i is written
 * compactly as (r_{i-1}, d_i, r_i).  ranks_out_host: L-1 bond dimensions.
 * svals_out_host: (L-1) x svals_stride, kept singular values per bond (after
 * renorm), rest zero-filled; may be NULL.  max_bond <= 0 means unlimited. */
int ndmps_ttsvd(ndmps_ctx_t* ctx, const void* dense, int dtype, int levels, const int64_t* dims,
                double cutoff, int cutoff_mode, int64_t max_bond, int renorm,
                void* const* cores_out, const int64_t* core_cap, int64_t* ranks_out_host,
                double* svals_out_host, int64_t svals_stride);

/* ---- column-sharded sweep over several GPUs (one process per GPU) -------------
 * The same from_dense sweep (core/ndmps.py:74) when ONE tensor is spread over `world` ranks: rank g
 * holds the slice of the dense site array whose LAST site index lies in block g
 * (dims_local = dims with the last entry divided by world), i.e. a column block of every unfolding.
 * Per step: local Gram, `allreduce` (sum, float64, in place, `count` doubles at buf_dev, enqueued on
 * `stream`; return 0 on success - the binding calls ncclAllReduce / torch.distributed.all_reduce),
 * the same bond eigenproblem on every rank, local projection.  The sharded phase stops before the
 * step at which the GLOBAL remainder is <= stop_bytes (or the local block stops being wide): cores
 * 0 .. *sites_done_host-1 (identical on every rank) are written, and the local remainder
 * (remainder_shape_host[0] x remainder_shape_host[1], row-major) is copied to remainder_out.  The
 * caller gathers the remainders, restores site order with ndmps_interleave_shards and finishes with
 * ndmps_ttsvd on dims (rows * d_s, d_{s+1}, ...). */
typedef int (*ndmps_allreduce_fn)(void* user, double* buf_dev, int64_t count, void* stream);
int ndmps_ttsvd_sharded(ndmps_ctx_t* ctx, const void* dense_local, int dtype, int levels, const int64_t* dims_local,
                        int world, ndmps_allreduce_fn allreduce, void* user, int64_t stop_bytes,
                        double cutoff, int cutoff_mode, int64_t max_bond, int renorm,
                        void* const* cores_out, const int64_t* core_cap, int64_t* ranks_out_host,
                        double* svals_out_host, int64_t svals_stride,
                        int* sites_done_host, void* remainder_out, int64_t remainder_cap, int64_t* remainder_shape_host);
/* out[r][c][g][t] = gathered[g][r][c][t]  (g < world, r < rows, c < cmid, t < dl): column blocks of
 * the ranks (as all-gathered, rank-major) back into the site order of the unsharded remainder. */
int ndmps_interleave_shards(ndmps_ctx_t* ctx, const void* gathered, int dtype, int world, int64_t rows, int64_t cmid, int64_t dl,
                            void* out);

/* ---- K6: pairwise bond truncation -----------------------------------------
 * qtn.tensor_compress_bond(T1, T2, cutoff, cutoff_mode="rel") at
 * core/ndmps.py:104-106 (absorb="both", no renorm).  t1: a x r, t2: r x b
 * (row-major matricisations of the two cores).  Outputs a x n and n x b written
 * compactly; t1_out/t2_out must not alias t1/t2.  svals_out_host: r values
 * (kept ones, rest zero).  Kept singular values below 1e-8 of the largest are
 * below the resolution of the Gram route and give zero columns / rows. */
int ndmps_compress_bond(ndmps_ctx_t* ctx, const void* t1, const void* t2, int dtype,
                        int64_t a, int64_t r, int64_t b,
                        double cutoff, int cutoff_mode, int64_t max_bond, int renorm,
                        void* t1_out, void* t2_out, int64_t* new_rank_host, double* svals_out_host);

/* ---- K7: MPS -> dense ------------------------------------------------------
 * `mps ^ ...` + moveindex at core/ndmps.py:140-142.  ranks: L-1 bond dims.
 * dense_out: prod(dims) elements, site order. */
int ndmps_contract_dense(ndmps_ctx_t* ctx, const void* const* cores, int dtype, int levels,
                         const int64_t* dims, const int64_t* ranks, void* dense_out);

/* ---- K7b: part of the MPS -> volume, without the whole tensor ----------------
 * An extension beyond the reference: to_tensor()[box] and to_tensor()[points] at core/ndmps.py:131-153 without
 * the N-element reconstruction.  `plan` is the volume's (ndmps_plan_create); cores / ranks as for
 * ndmps_contract_dense with levels = the plan's levels.
 * ndmps_contract_region: out = the box [lo, hi) (ndim values each) of the volume, in volume axis order,
 * C-contiguous, written on the context's stream without a host synchronisation.  The workspace is bounded by a
 * small multiple of the box (at most 3^ndim times it) plus the two chains restricted to the digits the box
 * touches.  A box outside the volume returns NDMPS_ERR_INVALID; an empty box is a no-op (out may then be NULL). */
int ndmps_contract_region(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* const* cores, int dtype,
                          const int64_t* ranks, const int64_t* lo, const int64_t* hi, void* out);
/* out_dev[i] = volume[coords_dev[i, :]] for `count` points; coords_dev: int64 device array (count x ndim),
 * negative coordinates count from the end as in numpy.  idct_last_axis = 1: the cores hold the DCT-II of the
 * volume along its last axis (mode "DCT"), the value is the orthonormal inverse DCT of that line evaluated at
 * the point (n = last extent dot products per point instead of 1).  A coordinate outside [-extent, extent) gives NaN;
 * no core is ever read outside its bounds.  No host synchronisation. */
int ndmps_evaluate_points(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* const* cores, int dtype,
                          const int64_t* ranks, const int64_t* coords_dev, int64_t count, int idct_last_axis,
                          void* out_dev);
/* Multilinear interpolation of the volume at real-valued coordinates: scipy.ndimage.map_coordinates(volume, coords.T,
 * order=1, mode="nearest"), i.e. each coordinate clamped to [0, extent - 1], then the 2^ndim corners around it weighted
 * by prod_a (1 - f_a or f_a) (corners of weight 0 are skipped).  Same chains as ndmps_evaluate_points, float64
 * accumulation, result in the cores' dtype.  idct_last_axis = 1 (mode "DCT"): the inverse-DCT basis row is interpolated
 * along the last axis instead, n * 2^(ndim-1) dot products per sample.  A non-finite coordinate gives NaN and reads no
 * core.  No host synchronisation.
 * ndmps_sample_points: coords_dev: float64 device array (count x ndim).  count 0 is a no-op (NULLs allowed). */
int ndmps_sample_points(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* const* cores, int dtype,
                        const int64_t* ranks, const double* coords_dev, int64_t count, int idct_last_axis, void* out_dev);
/* ndmps_sample_grid: the coordinates of an affine grid, computed in the kernel (nothing of the output's size is
 * uploaded): out_dev (C order over out_shape, m axes, 1 <= m <= 8) at index (i_0, .., i_{m-1}) is the sample at
 * origin + sum_j i_j steps[j].  origin (ndim), steps (m x ndim, row-major) and out_shape (m) are host arrays; origin
 * and steps must be finite, out_shape non-negative.  A grid with a zero extent is a no-op (out_dev may be NULL). */
int ndmps_sample_grid(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* const* cores, int dtype,
                      const int64_t* ranks, const double* origin, const double* steps, const int64_t* out_shape, int m,
                      int idct_last_axis, void* out_dev);
/* host-only index check of ndmps_contract_region (no device work): info_out[3] = {split site s, |H| kept rows,
 * |C| kept columns}; site_offsets_out_host (one value per box voxel, C order) = the flat site-order index
 * (row * Q_s + column) the region path reads for the voxel, mapped back from its compact row and column sets.
 * An empty box writes {s, 0, 0} and no offsets. */
int ndmps_region_debug_offsets(const ndmps_plan_t* plan, const int64_t* lo, const int64_t* hi, int64_t* info_out,
                               int64_t* site_offsets_out_host);

/* ---- K7d: maximum / minimum intensity projection of a box, without the box ------
 * An extension beyond the reference: op(to_tensor()[box], axis) (numpy's max / min, NaN propagating) from the cores.
 * out = op over volume axis `axis` of the box [lo, hi), C order over the other axes, in the cores' dtype.  The box is
 * decoded as in ndmps_contract_region, but the product T = X_H W_C runs in row blocks of whole axis-0 high parts of at
 * most 16 MB each, and every block is reduced into out as soon as it is written, so the workspace holds the two
 * restricted chains and one block, never the box.  idct_last_axis = 1 (mode "DCT"): the box is widened to the whole
 * last axis, and every block is gathered to volume order and inverse-transformed along it before the reduction.
 * On the context's stream, no host synchronisation.  A box outside the volume, an axis outside 0..ndim-1, an op other
 * than NDMPS_PROJ_MAX / NDMPS_PROJ_MIN, or an empty extent along `axis` return NDMPS_ERR_INVALID; an empty extent on
 * another axis is a no-op (out may then be NULL). */
#define NDMPS_PROJ_MAX 1
#define NDMPS_PROJ_MIN 2
int ndmps_project_region(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* const* cores, int dtype,
                         const int64_t* ranks, const int64_t* lo, const int64_t* hi, int axis, int op,
                         int idct_last_axis, void* out);
/* host-only index check of ndmps_project_region in Std mode (no device work), with the block bound `block_elems`
 * (elements of T; the device path uses 16 MB): info_out[4] = {split site s, |H|, |C|, blocks}; for every output
 * element o (C order over the box without `axis`) and position j along `axis`, offsets_out_host[o * e + j] (e = the
 * box's extent along `axis`) = the flat site-order index (row * Q_s + column) the reduction reads, and
 * offsets_out_host[count * e + o * e + j] (count = the output elements) = the block that reads it (-1: none, -2: more
 * than one).  The arguments are
 * checked as ndmps_project_region checks them; an empty box writes {s, 0, 0, 0} and nothing else. */
int ndmps_project_debug_offsets(const ndmps_plan_t* plan, const int64_t* lo, const int64_t* hi, int axis,
                                int64_t block_elems, int64_t* info_out, int64_t* offsets_out_host);

/* ---- K7c: block-mean (coarse) MPS, without the whole tensor -------------------
 * An extension beyond the reference: the mean of to_tensor() over non-overlapping blocks, from the cores.
 * drop_levels (ndim values, 0 <= k_a <= levels): axis a is averaged over its finest k_a digits, i.e. over blocks of
 * b_a = prod_{l >= levels - k_a} factors[l, a] voxels.
 * ndmps_plan_coarse (host only): *out = the plan of the block-mean tensor, shape[a] / b_a, with factors[l, a] = 1
 * wherever the digit is averaged and the trailing levels averaged on every axis removed (at least one level stays).
 * The result is an ordinary plan (ndmps_plan_layout reads it, ndmps_plan_destroy frees it).  This is the one place
 * that decides the coarse site layout. */
int ndmps_plan_coarse(const ndmps_plan_t* plan, const int64_t* drop_levels, ndmps_plan_t** out);
/* cores_out[i] (i < the coarse plan's levels, core_cap[i] elements each): the cores of the block-mean tensor in the
 * layout of ndmps_plan_coarse; cores / ranks as for ndmps_contract_region.  A partly averaged site maps (r, d, r') to
 * (r, d', r'), the mean over the averaged digits of the fused site index (float64 sums, stored in the payload dtype);
 * the removed sites fold, in float64, into one right boundary vector that the last kept core absorbs.  Output ranks:
 * the kept bonds (ranks[0 .. levels'-2]); the last kept core has no right bond.  On the context's stream, no host
 * synchronisation.  Bad drop_levels: NDMPS_ERR_INVALID; a core_cap below a core's size: NDMPS_ERR_CAPACITY, before
 * anything is enqueued. */
int ndmps_marginalize(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* const* cores, int dtype, const int64_t* ranks,
                      const int64_t* drop_levels, void* const* cores_out, const int64_t* core_cap);

/* ---- K8: <a|b> --------------------------------------------------------------
 * `mps @ mps` at core/ndmps.py:76,86 and utils/metrics.py:160 (no conjugation). */
int ndmps_overlap(ndmps_ctx_t* ctx, const void* const* cores_a, const int64_t* ranks_a, int dtype_a,
                  const void* const* cores_b, const int64_t* ranks_b, int dtype_b,
                  int levels, const int64_t* dims, double* out_host);

/* ---- K12: min-max quantisation ----------------------------------------------
 * utils/filetools.py:20-26 (scale_to_dtype, truncating cast) and :29-39
 * (scale_back), used by core/ndmps.py:200-204.  `bits` names the integer type like numpy's iinfo
 * dtypes: 8 / 16 / 32 / 64 unsigned, -8 / -16 / -32 / -64 signed; iinfo(dtype).max is the scale.
 * Where numpy's cast is undefined the result is defined here: NaN (every element of a constant array,
 * lo == hi) gives 0, and values past the type's range (the top code of the 64-bit types) saturate. */
int ndmps_quantize(ndmps_ctx_t* ctx, const void* x, int64_t n, int dtype, double lo, double hi, int bits, void* q_out);
int ndmps_dequantize(ndmps_ctx_t* ctx, const void* q, int64_t n, int bits, double lo, double hi, int dtype, void* x_out);

/* ---- K9: SSIM -----------------------------------------------------------------
 * compute_ssim_by_dim at utils/metrics.py:108-129 (2-D: :11-32, 3-D: :35-85,
 * 4-D: :88-105) with skimage's uniform-window structural_similarity.  `b` is the
 * argument the reference clips at 0.  ndim in {2,3,4}. */
int ndmps_ssim(ndmps_ctx_t* ctx, const void* a, const void* b, int dtype, int ndim, const int64_t* shape,
               double* out_host);

/* per-slice scores of ssim_3d_axis (utils/metrics.py:35-65): a, b are 3-D, axis in
 * {0,1,2}; scores_out_host receives shape[axis] values. */
int ndmps_ssim_slices(ndmps_ctx_t* ctx, const void* a, const void* b, int dtype, const int64_t* shape, int axis,
                      double* scores_out_host);

/* ---- whole path on HOST buffers (the e2e measurement entry) --------------------
 * NDMPS.from_tensor(x).to_tensor() with the max_bond / cutoff extension (core/ndmps.py:36-78, 131-153):
 * H2D copy, encode, sweep, boundary list + norm of the MPS (core/ndmps.py:75-76), contract, decode,
 * D2H copy.  ranks_out_host: L-1 values.  Optional: norm_out_host (1 value, sqrt(<mps|mps>)),
 * boundaries_out_host (2 L values: min, max of every core).  src / dst may also be device pointers. */
int ndmps_roundtrip_host(ndmps_ctx_t* ctx, const ndmps_plan_t* plan, const void* src_host, void* dst_host, int dtype,
                         double cutoff, int cutoff_mode, int64_t max_bond, int renorm, int64_t* ranks_out_host,
                         double* norm_out_host, double* boundaries_out_host);

#ifdef __cplusplus
}
#endif
#endif /* NDMPS_H */
