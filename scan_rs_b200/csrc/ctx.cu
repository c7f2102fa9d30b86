// ctx.cu -- context, errors, communicator, timers and per-phase accounting.
#include <dlfcn.h>

#include <chrono>
#include <cstdlib>
#include <map>
#include <mutex>
#include <unordered_map>
#include <set>

#include "common.cuh"

static thread_local char g_err[1024] = "";
static thread_local cudaStream_t g_alloc_stream = nullptr;
static thread_local cudaMemPool_t g_alloc_pool = nullptr;
cudaStream_t sb_alloc_stream() { return g_alloc_stream; }
cudaMemPool_t sb_alloc_pool() { return g_alloc_pool; }
void sb_set_alloc_stream(cudaStream_t s, cudaMemPool_t pool) {
    g_alloc_stream = s;
    g_alloc_pool = pool;
}

static std::mutex g_streams_mu;
static std::set<cudaStream_t> g_streams;
bool sb_stream_alive(cudaStream_t s) {
    std::lock_guard<std::mutex> lk(g_streams_mu);
    return g_streams.count(s) != 0;
}
void sb_stream_register(cudaStream_t s, bool alive) {
    std::lock_guard<std::mutex> lk(g_streams_mu);
    if (alive) g_streams.insert(s);
    else g_streams.erase(s);
}

// ---------------------------------------------------------------- exact-size block cache (common.cuh), one per context stream
struct BlockCache {
    std::unordered_map<size_t, std::vector<void *>> by_size;
    size_t bytes = 0, cap = 0;
};
static std::map<cudaStream_t, BlockCache> g_caches;  // under g_streams_mu
static void cache_flush_locked(cudaStream_t st, BlockCache &c) {
    for (auto &kv : c.by_size)
        for (void *p : kv.second) cudaFreeAsync(p, st);
    c.by_size.clear();
    c.bytes = 0;
}
void *sb_cache_take(cudaStream_t st, size_t bytes) {
    std::lock_guard<std::mutex> lk(g_streams_mu);
    auto it = g_caches.find(st);
    if (it == g_caches.end()) return nullptr;
    auto b = it->second.by_size.find(bytes);
    if (b == it->second.by_size.end() || b->second.empty()) return nullptr;
    void *p = b->second.back();
    b->second.pop_back();
    it->second.bytes -= bytes;
    return p;
}
bool sb_cache_give(cudaStream_t st, void *p, size_t bytes) {
    std::lock_guard<std::mutex> lk(g_streams_mu);
    auto it = g_caches.find(st);
    if (it == g_caches.end() || bytes > it->second.cap) return false;
    BlockCache &c = it->second;
    if (c.bytes + bytes > c.cap) cache_flush_locked(st, c);  // a changing workload: start over rather than hoard
    c.by_size[bytes].push_back(p);
    c.bytes += bytes;
    return true;
}
void sb_cache_flush(cudaStream_t st) {
    std::lock_guard<std::mutex> lk(g_streams_mu);
    auto it = g_caches.find(st);
    if (it != g_caches.end()) cache_flush_locked(st, it->second);
}
void sb_cache_configure(cudaStream_t st, size_t cap_bytes) {
    std::lock_guard<std::mutex> lk(g_streams_mu);
    if (cap_bytes == (size_t)-1) {  // the context is going away
        auto it = g_caches.find(st);
        if (it != g_caches.end()) {
            cache_flush_locked(st, it->second);
            g_caches.erase(it);
        }
        return;
    }
    BlockCache &c = g_caches[st];
    c.cap = cap_bytes;
    if (c.bytes > c.cap) cache_flush_locked(st, c);
}

void sb_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int sb_fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

// SCANB200_TRACE=1: synchronising stage trace, uploads take the unpipelined path; =2: same trace, pipelined uploads kept
int TraceScope::level() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("SCANB200_TRACE");
        v = (e && *e && *e != '0') ? (*e == '2' ? 2 : 1) : 0;
    }
    return v;
}
bool TraceScope::on() {
    return level() > 0;
}
double TraceScope::now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

extern "C" const char *sb_last_error(void) { return g_err; }
extern "C" int sb_version(void) { return SB_VERSION; }

extern "C" int sb_init(int device, sb_ctx **out) {
    if (!out) return sb_fail(SB_ERR_INVALID_ARG, "sb_init: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return sb_fail(SB_ERR_CUDA, "sb_init: no CUDA device (%s); this library has no CPU fallback",
                       e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0 || device >= ndev) return sb_fail(SB_ERR_INVALID_ARG, "sb_init: device %d of %d", device, ndev);
    SB_CUDA(cudaSetDevice(device));
    sb_ctx *ctx = new sb_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    SB_CUDA(cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    ctx->l2_bytes = (size_t)prop.l2CacheSize;
    SB_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    sb_stream_register(ctx->stream, true);
    {
        // a private pool: the release threshold ("never give memory back between calls") and the trim at shutdown are this context's
        // business and must not touch the default pool other CUDA users of the process (PyTorch, another library) allocate from
        const char *dp = getenv("SCANB200_DEFAULT_POOL");  // diagnostics: 1 = allocate from the device's default pool instead
        if (dp && *dp == '1') {
            cudaMemPool_t pool;
            SB_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
            uint64_t never0 = UINT64_MAX;
            SB_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &never0));
        } else {
        cudaMemPoolProps props;
        memset(&props, 0, sizeof(props));
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        SB_CUDA(cudaMemPoolCreate(&ctx->pool, &props));
        uint64_t never = UINT64_MAX;
        SB_CUDA(cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &never));
        }
    }
    sb_set_alloc_stream(ctx->stream, ctx->pool);
    {
        size_t free_b = 0, total_b = 0;
        SB_CUDA(cudaMemGetInfo(&free_b, &total_b));
        sb_cache_configure(ctx->stream, total_b / 2);  // option block_cache_gb
    }
    SB_CUBLAS(cublasCreate(&ctx->cublas));
    SB_CUBLAS(cublasSetStream(ctx->cublas, ctx->stream));
    SB_CUSOLVER(cusolverDnCreate(&ctx->cusolver));
    SB_CUSOLVER(cusolverDnSetStream(ctx->cusolver, ctx->stream));
    SB_CUDA(cudaEventCreate(&ctx->t0));
    SB_CUDA(cudaEventCreate(&ctx->t1));
    SB_CUDA(cudaMallocHost(&ctx->pinned, 4096));
    memset(&ctx->prof, 0, sizeof(ctx->prof));
    *out = ctx;
    return SB_OK;
}

extern "C" void sb_shutdown(sb_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    sb_set_alloc_stream(ctx->stream, ctx->pool);
    cudaStreamSynchronize(ctx->stream);
    prof_collect(ctx);
    for (auto ev : ctx->event_pool) cudaEventDestroy(ev);
    if (ctx->comm) ncclCommDestroy(ctx->comm);
    if (ctx->cusolver) cusolverDnDestroy(ctx->cusolver);
    if (ctx->cublas) cublasDestroy(ctx->cublas);
    if (ctx->t0) cudaEventDestroy(ctx->t0);
    if (ctx->t1) cudaEventDestroy(ctx->t1);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    if (ctx->eig_pinned) cudaFreeHost(ctx->eig_pinned);
    // every device buffer the context owns goes back to the pool while its stream still exists (a DevBuf released by `delete ctx`
    // below would hand cudaFreeAsync a destroyed stream: a crash at shutdown, seen with the cached start block)
    ctx->flush_buf.release();
    ctx->scratch.release();
    ctx->omega_dev.release();
    ctx->syrk_parts.release();
    sb_cache_configure(ctx->stream, (size_t)-1);  // cached blocks back to the pool, cache gone
    cudaStreamSynchronize(ctx->stream);

    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream) {
        sb_stream_register(ctx->stream, false);
        cudaStreamDestroy(ctx->stream);
    }
    if (ctx->pool) cudaMemPoolDestroy(ctx->pool);  // returns whatever handles created on this context still hold
    sb_set_alloc_stream(nullptr, nullptr);
    delete ctx;
}

extern "C" int sb_host_alloc(size_t bytes, void **out) {
    if (!out) return sb_fail(SB_ERR_INVALID_ARG, "sb_host_alloc: out is NULL");
    SB_CUDA(cudaMallocHost(out, bytes ? bytes : 1));
    return SB_OK;
}

extern "C" void sb_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

extern "C" int sb_set_option(sb_ctx *ctx, const char *name, double value) {
    if (!ctx || !name) return sb_fail(SB_ERR_INVALID_ARG, "sb_set_option: NULL argument");
    if (!strcmp(name, "direct_projection")) {
        ctx->direct_projection = value != 0.0;
        return SB_OK;
    }
    if (!strcmp(name, "verify_projection")) {
        ctx->verify_projection = value != 0.0;
        return SB_OK;
    }
    if (!strcmp(name, "own_dense")) {  // 1 (default): dense_own.cu kernels; 0: cuSOLVER / cuBLAS
        ctx->own_dense = value != 0.0;
        return SB_OK;
    }
    if (!strcmp(name, "upload_sync")) {
        ctx->upload_sync = value != 0.0;
        return SB_OK;
    }
    if (!strcmp(name, "gather")) {  // 1 (default): panelled gather kernels; 0: first-generation sparse kernels
        ctx->use_gather = value != 0.0;
        return SB_OK;
    }
    if (!strcmp(name, "gather_items_per_cta")) {  // applies to matrices built afterwards
        if (value < 1 || value > 64) return sb_fail(SB_ERR_INVALID_ARG, "sb_set_option: gather_items_per_cta must be 1..64");
        ctx->gather_items_per_cta = (int)value;
        return SB_OK;
    }
    if (!strcmp(name, "eig_jacobi")) {
        ctx->eig_jacobi = value != 0.0;
        return SB_OK;
    }
    if (!strcmp(name, "block_cache_gb")) {  // capacity of the exact-size block cache in front of the memory pool (0 = off)
        if (!(value >= 0.0 && value <= 1.0e6)) return sb_fail(SB_ERR_INVALID_ARG, "sb_set_option: block_cache_gb must be in [0, 1e6]");
        sb_cache_configure(ctx->stream, (size_t)(value * 1.0e9));
        return SB_OK;
    }
    if (!strcmp(name, "gemm_skinny")) {
        ctx->gemm_skinny = value != 0.0;
        return SB_OK;
    }
    if (!strcmp(name, "eig_host")) {
        ctx->eig_host = value != 0.0;
        return SB_OK;
    }
    if (!strcmp(name, "upload_chunks")) {
        if (!(value >= 1.0 && value <= 256.0)) return sb_fail(SB_ERR_INVALID_ARG, "sb_set_option: upload_chunks must be in [1, 256]");
        ctx->upload_chunks = (int)value;
        return SB_OK;
    }
    if (!strcmp(name, "gather_defer")) {
        ctx->gather_defer = value != 0.0;
        return SB_OK;
    }
    if (!strcmp(name, "gather_calibrate")) {
        ctx->gather_calibrate = value <= 0.0 ? 0 : (value > 8.0 ? 8 : (int)value);
        return SB_OK;
    }
    if (!strcmp(name, "gather_seg_cost")) {  // applies to matrices built afterwards
        if (!(value >= 0.0 && value <= 1.0e7)) return sb_fail(SB_ERR_INVALID_ARG, "sb_set_option: gather_seg_cost must be in [0, 1e7]");
        ctx->gather_seg_cost = value;
        return SB_OK;
    }
    if (!strcmp(name, "gather_flush_cost")) {  // applies to matrices built afterwards
        if (!(value >= 0.0 && value <= 1000.0)) return sb_fail(SB_ERR_INVALID_ARG, "sb_set_option: gather_flush_cost must be in [0, 1000]");
        ctx->gather_flush_cost = value;
        return SB_OK;
    }
    if (!strcmp(name, "plane_items_per_cta")) {  // applies to matrices built afterwards
        if (value < 1 || value > 256) return sb_fail(SB_ERR_INVALID_ARG, "sb_set_option: plane_items_per_cta must be 1..256");
        ctx->plane_items_per_cta = (int)value;
        return SB_OK;
    }
    if (!strcmp(name, "plane_cap")) {  // applies to matrices built afterwards; < 128: no planes
        ctx->plane_cap = value < 0 ? 0 : (int)value;
        return SB_OK;
    }
    if (!strcmp(name, "plane_levels")) {
        if (value < 1 || value > PL_MAX_LEVELS) return sb_fail(SB_ERR_INVALID_ARG, "sb_set_option: plane_levels must be 1..%d", PL_MAX_LEVELS);
        ctx->plane_levels = (int)value;
        return SB_OK;
    }
    if (!strcmp(name, "plane_min_density")) {
        ctx->plane_min_density = value;
        return SB_OK;
    }
    return sb_fail(SB_ERR_INVALID_ARG, "sb_set_option: unknown option %s", name);
}

extern "C" int sb_sync(sb_ctx *ctx) {
    if (!ctx) return sb_fail(SB_ERR_INVALID_ARG, "sb_sync: ctx is NULL");
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// ---------------------------------------------------------------- communicator
#undef ncclGetUniqueId
#undef ncclCommInitRank
#undef ncclCommDestroy
#undef ncclAllReduce
#undef ncclAllGather
#undef ncclBroadcast
#undef ncclGroupStart
#undef ncclGroupEnd
#undef ncclGetErrorString
const NcclApi *sb_nccl() {
    static NcclApi api;
    static int state = 0;  // 0 untried, 1 ok, -1 failed
    if (state == 1) return &api;
    if (state == -1) return nullptr;
    void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
        sb_set_error("cannot load libnccl.so.2: %s", dlerror());
        state = -1;
        return nullptr;
    }
    bool ok = true;
    auto sym = [&](const char *name) {
        void *p = dlsym(h, name);
        if (!p) ok = false;
        return p;
    };
    api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
    api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
    api.AllReduce = (decltype(api.AllReduce))sym("ncclAllReduce");
    api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
    api.Broadcast = (decltype(api.Broadcast))sym("ncclBroadcast");
    api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
    api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
    api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
    if (!ok) {
        sb_set_error("libnccl.so.2 lacks a required symbol");
        state = -1;
        return nullptr;
    }
    state = 1;
    return &api;
}
#define ncclGetUniqueId sb_nccl()->GetUniqueId
#define ncclCommInitRank sb_nccl()->CommInitRank
#define ncclCommDestroy sb_nccl()->CommDestroy
#define ncclAllReduce sb_nccl()->AllReduce
#define ncclAllGather sb_nccl()->AllGather
#define ncclBroadcast sb_nccl()->Broadcast
#define ncclGroupStart sb_nccl()->GroupStart
#define ncclGroupEnd sb_nccl()->GroupEnd
#define ncclGetErrorString sb_nccl()->GetErrorString
extern "C" int sb_comm_unique_id(char id[128]) {
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
    ncclUniqueId uid;
    if (!sb_nccl()) return SB_ERR_NCCL;
    SB_NCCL(ncclGetUniqueId(&uid));
    memcpy(id, &uid, 128);
    return SB_OK;
}

extern "C" int sb_comm_init(sb_ctx *ctx, int nranks, int rank, const char id[128]) {
    if (!ctx || nranks < 1 || rank < 0 || rank >= nranks) return sb_fail(SB_ERR_INVALID_ARG, "sb_comm_init: bad arguments");
    if (ctx->comm) return sb_fail(SB_ERR_INVALID_ARG, "sb_comm_init: communicator already initialised");
    SB_CUDA(cudaSetDevice(ctx->device));
    if (nranks == 1) return SB_OK;
    ncclUniqueId uid;
    if (!sb_nccl()) return SB_ERR_NCCL;
    memcpy(&uid, id, 128);
    SB_NCCL(ncclCommInitRank(&ctx->comm, nranks, uid, rank));
    ctx->nranks = nranks;
    ctx->rank = rank;
    return SB_OK;
}

int ctx_scratch(sb_ctx *ctx, size_t bytes, void **out) {
    SB_TRY(ctx->scratch.ensure(bytes));
    *out = ctx->scratch.p;
    return SB_OK;
}

int comm_allreduce_f64(sb_ctx *ctx, double *buf, size_t count) {
    if (ctx->nranks == 1 || count == 0) return SB_OK;
    ProfScope ps(ctx, PH_COMM);
    SB_NCCL(ncclAllReduce(buf, buf, count, ncclDouble, ncclSum, ctx->comm, ctx->stream));
    count_launch(ctx, false);
    return SB_OK;
}

int comm_allreduce_u64(sb_ctx *ctx, u64 *buf, size_t count) {
    if (ctx->nranks == 1 || count == 0) return SB_OK;
    ProfScope ps(ctx, PH_COMM);
    SB_NCCL(ncclAllReduce(buf, buf, count, ncclUint64, ncclSum, ctx->comm, ctx->stream));
    count_launch(ctx, false);
    return SB_OK;
}

int comm_allreduce_max_i32(sb_ctx *ctx, int *host_val) {
    if (ctx->nranks == 1) return SB_OK;
    void *d;
    SB_TRY(ctx_scratch(ctx, 256, &d));
    SB_CUDA(cudaMemcpyAsync(d, host_val, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    SB_NCCL(ncclAllReduce(d, d, 1, ncclInt32, ncclMax, ctx->comm, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(host_val, d, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

int comm_allgather_u64_host(sb_ctx *ctx, u64 mine, std::vector<u64> &all) {
    all.assign(ctx->nranks, 0);
    if (ctx->nranks == 1) {
        all[0] = mine;
        return SB_OK;
    }
    void *d;
    SB_TRY(ctx_scratch(ctx, sizeof(u64) * (ctx->nranks + 1), &d));
    u64 *dv = (u64 *)d;
    SB_CUDA(cudaMemcpyAsync(dv + ctx->nranks, &mine, sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
    SB_NCCL(ncclAllGather(dv + ctx->nranks, dv, 1, ncclUint64, ctx->comm, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(all.data(), dv, sizeof(u64) * ctx->nranks, cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// ---------------------------------------------------------------- profiling
static cudaEvent_t get_event(sb_ctx *ctx) {
    if (!ctx->event_pool.empty()) {
        cudaEvent_t e = ctx->event_pool.back();
        ctx->event_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

void prof_begin(sb_ctx *ctx, int phase) {
    if (!ctx->profile_on) return;
    cudaEvent_t a = get_event(ctx), b = get_event(ctx);
    cudaEventRecord(a, ctx->stream);
    ctx->pending.push_back({phase, {a, b}});
}

void prof_end(sb_ctx *ctx, int phase) {
    if (!ctx->profile_on) return;
    for (int i = (int)ctx->pending.size() - 1; i >= 0; i--)
        if (ctx->pending[i].first == phase) {
            cudaEventRecord(ctx->pending[i].second.second, ctx->stream);
            ctx->pending[i].first = phase + 100;  // closed
            return;
        }
}

void prof_collect(sb_ctx *ctx) {
    if (ctx->pending.empty()) return;
    cudaStreamSynchronize(ctx->stream);
    for (auto &p : ctx->pending) {
        float ms = 0.f;
        if (p.first >= 100) {
            cudaEventElapsedTime(&ms, p.second.first, p.second.second);
            switch (p.first - 100) {
            case PH_SPMM_T: ctx->prof.spmm_t_ms += ms; break;
            case PH_SPMM_N: ctx->prof.spmm_n_ms += ms; break;
            case PH_MOMENTS: ctx->prof.moments_ms += ms; break;
            case PH_REDUCE: ctx->prof.reduce_ms += ms; break;
            case PH_DENSE: ctx->prof.dense_ms += ms; break;
            case PH_COMM: ctx->prof.comm_ms += ms; break;
            case PH_UPLOAD: ctx->prof.upload_ms += ms; break;
            case PH_BUILD: ctx->prof.build_ms += ms; break;
            case PH_OUTPUT: ctx->prof.output_ms += ms; break;
            }
        }
        ctx->event_pool.push_back(p.second.first);
        ctx->event_pool.push_back(p.second.second);
    }
    ctx->pending.clear();
}

extern "C" int sb_profile_enable(sb_ctx *ctx, int on) {
    if (!ctx) return sb_fail(SB_ERR_INVALID_ARG, "ctx is NULL");
    prof_collect(ctx);
    ctx->profile_on = on != 0;
    return SB_OK;
}

extern "C" int sb_profile_reset(sb_ctx *ctx) {
    if (!ctx) return sb_fail(SB_ERR_INVALID_ARG, "ctx is NULL");
    prof_collect(ctx);
    memset(&ctx->prof, 0, sizeof(ctx->prof));
    return SB_OK;
}

extern "C" int sb_profile_get(sb_ctx *ctx, sb_profile *out) {
    if (!ctx || !out) return sb_fail(SB_ERR_INVALID_ARG, "NULL argument");
    prof_collect(ctx);
    *out = ctx->prof;
    return SB_OK;
}

extern "C" int sb_timer_begin(sb_ctx *ctx) {
    if (!ctx) return sb_fail(SB_ERR_INVALID_ARG, "ctx is NULL");
    SB_ENTER(ctx);
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    SB_CUDA(cudaEventRecord(ctx->t0, ctx->stream));
    return SB_OK;
}

extern "C" int sb_timer_end(sb_ctx *ctx, float *ms) {
    if (!ctx || !ms) return sb_fail(SB_ERR_INVALID_ARG, "NULL argument");
    SB_CUDA(cudaEventRecord(ctx->t1, ctx->stream));
    SB_CUDA(cudaEventSynchronize(ctx->t1));
    SB_CUDA(cudaEventElapsedTime(ms, ctx->t0, ctx->t1));
    return SB_OK;
}

extern "C" int sb_flush_l2(sb_ctx *ctx) {
    if (!ctx) return sb_fail(SB_ERR_INVALID_ARG, "ctx is NULL");
    SB_ENTER(ctx);
    size_t bytes = ctx->l2_bytes ? ctx->l2_bytes * 2 : ((size_t)256 << 20);
    SB_TRY(ctx->flush_buf.ensure(bytes));
    SB_CUDA(cudaMemsetAsync(ctx->flush_buf.p, 1, bytes, ctx->stream));
    count_launch(ctx, false);
    return SB_OK;
}
