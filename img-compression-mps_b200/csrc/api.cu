// Context, workspace arena and error plumbing of libndmps_sm100.so.
#include <stdarg.h>

#include <chrono>
#include <map>
#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"

namespace ndmps {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

void Arena::release() {
    for (auto& c : chunks) cudaFree(c.base);
    chunks.clear();
}

int Arena::reset(cudaStream_t stream) {
    generation++;
    if (cur_total > high_water) high_water = cur_total;
    cur_total = 0;
    if (chunks.size() > 1) {
        // merge: everything issued against the old chunks must have finished first
        NDMPS_CUDA_TRY(cudaStreamSynchronize(stream));
        size_t total = 0;
        for (auto& c : chunks) total += c.cap;
        release();
        char* p = nullptr;
        NDMPS_CUDA_TRY(cudaMalloc(&p, total));
        chunks.push_back({p, total, 0});
    }
    for (auto& c : chunks) c.used = 0;
    return NDMPS_OK;
}

int Arena::alloc(size_t bytes, void** out) {
    bytes = (bytes + 255) & ~size_t(255);
    if (bytes == 0) bytes = 256;
    for (auto& c : chunks) {
        if (c.cap - c.used >= bytes) {
            *out = c.base + c.used;
            c.used += bytes;
            cur_total += bytes;
            return NDMPS_OK;
        }
    }
    size_t cap = bytes < (size_t(64) << 20) ? (size_t(64) << 20) : bytes;
    char* p = nullptr;
    cudaError_t e = cudaMalloc(&p, cap);
    if (e != cudaSuccess) {
        set_error("workspace cudaMalloc(%zu) failed: %s", cap, cudaGetErrorString(e));
        return NDMPS_ERR_NOMEM;
    }
    chunks.push_back({p, cap, bytes});
    cur_total += bytes;
    *out = p;
    return NDMPS_OK;
}

int raise_dynamic_smem(const void* kernel, int device, int bytes) {
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, int> raised;
    std::lock_guard<std::mutex> lock(mu);
    auto key = std::make_pair(kernel, device);
    auto it = raised.find(key);
    if (it != raised.end() && it->second >= bytes) return NDMPS_OK;
    int cur = -1;
    NDMPS_CUDA_TRY(cudaGetDevice(&cur));
    if (cur != device) NDMPS_CUDA_TRY(cudaSetDevice(device));
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (cur != device) cudaSetDevice(cur);
    NDMPS_CUDA_TRY(e);
    raised[key] = bytes;
    return NDMPS_OK;
}

// Can one cluster of `cluster_ctas` CTAs of `kernel` be resident on `device`?  Sizes above the portable 8 need the
// kernel's opt-in first.  Answer cached per (kernel, device, size).
int cluster_fits(const void* kernel, int device, int cluster_ctas, int threads, bool* fits) {
    static std::mutex mu;
    static std::map<std::pair<const void*, std::pair<int, int>>, bool> known;
    std::lock_guard<std::mutex> lock(mu);
    auto key = std::make_pair(kernel, std::make_pair(device, cluster_ctas));
    auto it = known.find(key);
    if (it != known.end()) { *fits = it->second; return NDMPS_OK; }
    int cur = -1;
    NDMPS_CUDA_TRY(cudaGetDevice(&cur));
    if (cur != device) NDMPS_CUDA_TRY(cudaSetDevice(device));
    bool ok = cluster_ctas <= 16;
    if (ok && cluster_ctas > 8) ok = cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess;
    if (ok) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)cluster_ctas);
        cfg.blockDim = dim3((unsigned)threads);
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = (unsigned)cluster_ctas;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        int clusters = 0;
        ok = cudaOccupancyMaxActiveClusters(&clusters, kernel, &cfg) == cudaSuccess && clusters >= 1;
    }
    cudaGetLastError();                                  // a refused size is an answer, not an error of the context
    if (cur != device) cudaSetDevice(cur);
    known[key] = ok;
    *fits = ok;
    return NDMPS_OK;
}

int ensure_pinned(ndmps_ctx* ctx, size_t doubles) {
    if (ctx->pinned_doubles >= doubles) return NDMPS_OK;
    if (ctx->pinned) {
        NDMPS_CUDA_TRY(stream_wait(ctx));
        cudaFreeHost(ctx->pinned);
        ctx->pinned = nullptr;
        ctx->pinned_doubles = 0;
    }
    size_t want = doubles < 16384 ? 16384 : doubles;
    // mapped: the read-back kernel below stores into it from the SMs (same pointer on both sides under unified addressing)
    NDMPS_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&ctx->pinned), want * sizeof(double), cudaHostAllocMapped));
    ctx->pinned_doubles = want;
    return NDMPS_OK;
}

// Small device -> host read-backs (eigenvalues, flags, scalars: 4 bytes ... a few hundred KB) leave through the SMs, not
// through the copy engine: a cudaMemcpyAsync queues behind whatever the device-to-host engine is moving for ANOTHER
// stream, and with volumes in flight through host buffers that is a 537 MB reconstruction (10 ms) - every one of the
// eight waits of a sweep stood behind one.  A few warps storing into mapped pinned memory do not queue behind anything.
__global__ void __launch_bounds__(256) readback_kernel(const unsigned* __restrict__ src, unsigned* dst_host, int64_t words) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < words; i += (int64_t)gridDim.x * blockDim.x)
        dst_host[i] = src[i];
    __threadfence_system();
}

// device -> device copies of bond-sized data: the same few warps instead of a copy-engine descriptor (which shares its
// engine's queue with the other streams' transfers)
int copy_small(ndmps_ctx* ctx, void* dev_dst, const void* dev_src, size_t bytes) {
    if (bytes == 0) return NDMPS_OK;
    const bool words = bytes % 4 == 0 && reinterpret_cast<uintptr_t>(dev_dst) % 4 == 0 && reinterpret_cast<uintptr_t>(dev_src) % 4 == 0;
    if (words && bytes <= (size_t(8) << 20)) {
        const int64_t n = (int64_t)(bytes / 4);
        int64_t grid = (n + 1023) / 1024;
        if (grid > 64) grid = 64;
        readback_kernel<<<(unsigned)grid, 256, 0, ctx->stream>>>((const unsigned*)dev_src, (unsigned*)dev_dst, n);
        NDMPS_LAUNCH_CHECK(ctx);
        return NDMPS_OK;
    }
    NDMPS_CUDA_TRY(cudaMemcpyAsync(dev_dst, dev_src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return NDMPS_OK;
}

int readback(ndmps_ctx* ctx, void* pinned_dst, const void* dev_src, size_t bytes) {
    if (bytes == 0) return NDMPS_OK;
    const bool in_scratch = ctx->pinned && (const char*)pinned_dst >= (const char*)ctx->pinned &&
                            (const char*)pinned_dst + bytes <= (const char*)(ctx->pinned + ctx->pinned_doubles);
    const bool words = bytes % 4 == 0 && reinterpret_cast<uintptr_t>(pinned_dst) % 4 == 0 && reinterpret_cast<uintptr_t>(dev_src) % 4 == 0;
    if (in_scratch && words && bytes <= (size_t(8) << 20)) {
        const int64_t n = (int64_t)(bytes / 4);
        int64_t grid = (n + 1023) / 1024;
        if (grid > 32) grid = 32;
        readback_kernel<<<(unsigned)grid, 256, 0, ctx->stream>>>((const unsigned*)dev_src, (unsigned*)pinned_dst, n);
        NDMPS_LAUNCH_CHECK(ctx);
        return NDMPS_OK;
    }
    NDMPS_CUDA_TRY(cudaMemcpyAsync(pinned_dst, dev_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return NDMPS_OK;
}

int profile_collect(ndmps_ctx* ctx) {
    if (ctx->pending.empty()) return NDMPS_OK;
    NDMPS_CUDA_TRY(stream_wait(ctx));
    for (auto& p : ctx->pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.beg, p.end) == cudaSuccess) {
            ctx->stage_ms[p.stage] += ms;
            ctx->stage_calls[p.stage] += 1;
        }
        cudaEventDestroy(p.beg);
        cudaEventDestroy(p.end);
    }
    ctx->pending.clear();
    return NDMPS_OK;
}


// mode 3: the stream writes a sequence number into pinned host memory (one-thread kernel, system-scope store) and the
// host watches that word: no driver call - and so no driver lock shared with the threads that are launching - while
// waiting.  Yields between looks; asks the driver now and then so that a faulted stream cannot hang the wait.
__global__ void wait_flag_kernel(volatile unsigned* flag, unsigned seq) {
    *flag = seq;
    __threadfence_system();
}

static cudaError_t flag_wait(ndmps_ctx* ctx) {
    if (!ctx->wait_flag) {
        cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(const_cast<unsigned**>(&ctx->wait_flag)), 64, cudaHostAllocMapped);
        if (e != cudaSuccess) return e;
        *ctx->wait_flag = 0;
    }
    const unsigned seq = ++ctx->wait_seq;
    wait_flag_kernel<<<1, 1, 0, ctx->stream>>>(ctx->wait_flag, seq);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    for (unsigned looks = 1;; looks++) {
        if (*ctx->wait_flag == seq) return cudaSuccess;
        if ((looks & 15) == 0) std::this_thread::yield();
        if ((looks & 0xFFFFF) == 0) {
            e = cudaStreamQuery(ctx->stream);
            if (e != cudaSuccess && e != cudaErrorNotReady) return e;
        }
    }
}

cudaError_t stream_wait(ndmps_ctx* ctx) {
    if (ctx->opt_blocking_sync == 3) return flag_wait(ctx);
    return cudaStreamSynchronize(ctx->stream);
}

// ---- gate for concurrent cooperative launches (see common.cuh) ---------------------------------
namespace {
struct CoopTicket { cudaEvent_t done; int sms; };
struct CoopGate {
    std::mutex m;
    int in_use = 0;                        // SMs booked by cooperative kernels in flight
    std::vector<CoopTicket> inflight;
    std::vector<cudaEvent_t> pool;
    void reap() {                          // give back what has finished (called with m held)
        for (size_t i = 0; i < inflight.size();) {
            if (cudaEventQuery(inflight[i].done) != cudaErrorNotReady) {
                in_use -= inflight[i].sms;
                pool.push_back(inflight[i].done);
                inflight[i] = inflight.back();
                inflight.pop_back();
            } else {
                i++;
            }
        }
    }
};
CoopGate g_gate;
}  // namespace

int coop_launch(ndmps_ctx* ctx, const void* fn, dim3 grid, dim3 block, void** args, size_t smem) {
    int per_sm = 0;
    NDMPS_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, (int)(block.x * block.y * block.z), smem));
    if (per_sm < 1) per_sm = 1;
    const int ctas = (int)(grid.x * grid.y * grid.z);
    int sms = (ctas + per_sm - 1) / per_sm;
    const int budget = ctx->sm_count;
    if (sms > budget) sms = budget;
    cudaEvent_t ev = nullptr;
    for (;;) {
        {
            std::lock_guard<std::mutex> lock(g_gate.m);
            g_gate.reap();
            if (g_gate.in_use == 0 || g_gate.in_use + sms <= budget) {
                g_gate.in_use += sms;
                if (!g_gate.pool.empty()) { ev = g_gate.pool.back(); g_gate.pool.pop_back(); }
                break;
            }
        }
        std::this_thread::sleep_for(std::chrono::microseconds(20));
    }
    cudaError_t e = cudaSuccess;
    if (!ev) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaLaunchCooperativeKernel(fn, grid, block, args, smem, ctx->stream);
    if (e == cudaSuccess) e = cudaEventRecord(ev, ctx->stream);
    {
        std::lock_guard<std::mutex> lock(g_gate.m);
        if (e == cudaSuccess) g_gate.inflight.push_back({ev, sms});
        else g_gate.in_use -= sms;
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("%s:%d: cooperative launch -> %s", __FILE__, __LINE__, cudaGetErrorString(e));
        return NDMPS_ERR_CUDA;
    }
    ctx->launches++;
    return NDMPS_OK;
}

}  // namespace ndmps

using namespace ndmps;

extern "C" {

int ndmps_version(void) { return 100; }

const char* ndmps_last_error(void) { return g_err; }

int ndmps_ctx_create(ndmps_ctx_t** out) {
    NDMPS_REQUIRE(out != nullptr, "ndmps_ctx_create: out is NULL");
    int dev = 0;
    NDMPS_CUDA_TRY(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    NDMPS_CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    if (prop.major != 10) {
        set_error("libndmps_sm100 needs a compute capability 10.x device (B200); found %d.%d (%s)", prop.major,
                  prop.minor, prop.name);
        return NDMPS_ERR_CUDA;
    }
    ndmps_ctx* ctx = new ndmps_ctx();
    ctx->device = dev;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    *out = ctx;
    return NDMPS_OK;
}

int ndmps_ctx_destroy(ndmps_ctx_t* ctx) {
    if (!ctx) return NDMPS_OK;
    stream_wait(ctx);
    ctx->ws.release();
    if (ctx->wait_flag) cudaFreeHost(const_cast<unsigned*>(ctx->wait_flag));
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    delete ctx;
    return NDMPS_OK;
}

int ndmps_ctx_set_stream(ndmps_ctx_t* ctx, void* cuda_stream) {
    NDMPS_REQUIRE(ctx != nullptr, "ndmps_ctx_set_stream: ctx is NULL");
    cudaStream_t next = static_cast<cudaStream_t>(cuda_stream);
    if (next != ctx->stream) {
        // one context = one workspace arena, reused call after call in stream order: work still queued on the old stream
        // may be reading it, so the new stream starts behind everything the old one has been given
        cudaEvent_t ev = nullptr;
        NDMPS_CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        if (cudaEventRecord(ev, ctx->stream) == cudaSuccess) {
            cudaError_t e = cudaStreamWaitEvent(next, ev, 0);
            cudaEventDestroy(ev);
            NDMPS_CUDA_TRY(e);
        } else {                                         // the old stream no longer exists: nothing of it can be pending
            cudaGetLastError();
            cudaEventDestroy(ev);
        }
        ctx->stream = next;
    }
    return NDMPS_OK;
}

int ndmps_ctx_sync(ndmps_ctx_t* ctx) {
    NDMPS_REQUIRE(ctx != nullptr, "ndmps_ctx_sync: ctx is NULL");
    NDMPS_CUDA_TRY(stream_wait(ctx));
    return NDMPS_OK;
}

int64_t ndmps_ctx_launch_count(const ndmps_ctx_t* ctx) { return ctx ? ctx->launches : 0; }

static const char* kStageNames[ST_COUNT] = {"permute", "gram", "eig", "project", "glue", "contract", "dct", "metric"};

int ndmps_ctx_profile(ndmps_ctx_t* ctx, int enable) {
    NDMPS_REQUIRE(ctx != nullptr, "ndmps_ctx_profile: ctx is NULL");
    NDMPS_TRY(profile_collect(ctx));
    ctx->profile = enable != 0;
    return NDMPS_OK;
}

int ndmps_stage_count(void) { return ST_COUNT; }

const char* ndmps_stage_name(int stage) { return stage >= 0 && stage < ST_COUNT ? kStageNames[stage] : ""; }

int ndmps_ctx_stage_times(ndmps_ctx_t* ctx, double* ms_out, int64_t* calls_out, int reset) {
    NDMPS_REQUIRE(ctx && ms_out && calls_out, "ndmps_ctx_stage_times: NULL argument");
    NDMPS_TRY(profile_collect(ctx));
    for (int i = 0; i < ST_COUNT; i++) {
        ms_out[i] = ctx->stage_ms[i];
        calls_out[i] = ctx->stage_calls[i];
        if (reset) { ctx->stage_ms[i] = 0.0; ctx->stage_calls[i] = 0; }
    }
    return NDMPS_OK;
}

int ndmps_ctx_get_stat(ndmps_ctx_t* ctx, const char* name, double* value_out, int reset) {
    NDMPS_REQUIRE(ctx && name && value_out, "ndmps_ctx_get_stat: NULL argument");
    if (!strcmp(name, "eig_flops")) { *value_out = ctx->eig_flops; if (reset) ctx->eig_flops = 0.0; }
    else if (!strcmp(name, "eig_calls")) { *value_out = (double)ctx->eig_calls; if (reset) ctx->eig_calls = 0; }
    else if (!strcmp(name, "workspace_bytes")) { *value_out = (double)ctx->ws.high_water; }
    else if (!strcmp(name, "cluster_launches")) { *value_out = (double)ctx->cluster_launches; if (reset) ctx->cluster_launches = 0; }
    else if (!strcmp(name, "tc_launches")) { *value_out = (double)ctx->tc_launches; if (reset) ctx->tc_launches = 0; }
    else {
        set_error("ndmps_ctx_get_stat: unknown statistic '%s'", name);
        return NDMPS_ERR_INVALID;
    }
    return NDMPS_OK;
}

int ndmps_ctx_set_option(ndmps_ctx_t* ctx, const char* name, int64_t value) {
    NDMPS_REQUIRE(ctx != nullptr && name != nullptr, "ndmps_ctx_set_option: NULL argument");
    if (!strcmp(name, "gram_path")) ctx->opt_gram_path = value;
    else if (!strcmp(name, "gemm_path")) ctx->opt_gemm_path = value;
    else if (!strcmp(name, "gemm_out_t")) ctx->opt_gemm_out_t = value;
    else if (!strcmp(name, "tc")) ctx->opt_tc = value;
    else if (!strcmp(name, "tc_waves")) ctx->opt_tc_waves = value;
    else if (!strcmp(name, "permute_path")) {
        NDMPS_REQUIRE(value >= 0 && value <= 2, "ndmps_ctx_set_option: permute_path must be 0, 1 or 2 (got %lld)", (long long)value);
        ctx->opt_permute_path = value;
    }
    else if (!strcmp(name, "eig_topk")) ctx->opt_eig_topk = value;
    else if (!strcmp(name, "topk_cluster")) ctx->opt_topk_cluster = value;
    else if (!strcmp(name, "ssim_exact")) ctx->opt_ssim_exact = value;
    else if (!strcmp(name, "blocking_sync")) {
        NDMPS_REQUIRE(value == 0 || value == 3, "ndmps_ctx_set_option: blocking_sync must be 0 or 3 (got %lld)", (long long)value);
        ctx->opt_blocking_sync = value;
    }
    else if (!strcmp(name, "verbose")) ctx->opt_verbose = value;
    else {
        set_error("ndmps_ctx_set_option: unknown option '%s'", name);
        return NDMPS_ERR_INVALID;
    }
    return NDMPS_OK;
}

}  // extern "C"
