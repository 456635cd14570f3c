// api.cu -- the extern "C" boundary (include/pcr_b200.h): argument checks, the reference's
// degenerate-input rules, host<->device staging, and nothing else.  Every entry point catches
// everything: no exception and no sticky CUDA error crosses the ABI.
#include "pcr_internal.cuh"

#include <stdarg.h>

#include <atomic>
#include <chrono>
#include <cstring>
#include <utility>
#include <vector>
#include <algorithm>
#include <new>

namespace pcr {

static thread_local std::string g_thread_error = "no error";
static thread_local uint64_t g_thread_err_seq = 0;
static std::atomic<uint64_t> g_err_seq{0};

void set_thread_error(const char *msg) {
    g_thread_error = msg ? msg : "unknown error";
    g_thread_err_seq = ++g_err_seq;
}

int fail(Ctx *ctx, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_thread_error = buf;
    g_thread_err_seq = ++g_err_seq;
    if (ctx) {
        ctx->err = buf;
        ctx->err_seq = g_thread_err_seq;
    }
    return code;
}

TimeScope::TimeScope(Ctx *ctx, int tag) : c(ctx) {
    if (!c->timing) return;
    Ctx::TimedSpan sp;
    sp.tag = tag;
    for (cudaEvent_t *e : {&sp.a, &sp.b}) {
        if (!c->event_pool.empty()) {
            *e = c->event_pool.back();
            c->event_pool.pop_back();
        } else if (cudaEventCreate(e) != cudaSuccess) {
            cudaGetLastError();
            return;
        }
    }
    cudaEventRecord(sp.a, c->stream);
    idx = (int)c->spans.size();
    c->spans.push_back(sp);
}
TimeScope::~TimeScope() {
    if (idx >= 0) cudaEventRecord(c->spans[idx].b, c->stream);
}

bool g_trace_on = getenv("PCR_TRACE") != nullptr;
namespace {
thread_local std::vector<std::pair<const char *, double>> t_trace;
}
static void trace_dump();
// PCR_TRACE_SLOW_US=<t>: keep only the marks of calls that took longer than t (a call = a mark ending in "enter" ... "exit")
static const double g_trace_slow_us = getenv("PCR_TRACE_SLOW_US") ? atof(getenv("PCR_TRACE_SLOW_US")) : 0.0;
void trace_mark(const char *label) {
    const size_t len = strlen(label);
    if (g_trace_slow_us > 0.0 && len >= 5 && !strcmp(label + len - 5, "enter")) t_trace.clear();
    t_trace.emplace_back(label, std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count());
    if (g_trace_slow_us > 0.0 && len >= 4 && !strcmp(label + len - 4, "exit")) {
        if (t_trace.back().second - t_trace.front().second > g_trace_slow_us) trace_dump();
        else t_trace.clear();
    }
}
static void trace_dump() {
    if (!g_trace_on || t_trace.empty()) return;
    const size_t n = t_trace.size(), b = n > 160 ? n - 160 : 0;
    for (size_t i = b; i < n; i++)
        fprintf(stderr, "[trace] %9.1f us  +%6.1f  %s\n", t_trace[i].second - t_trace[b].second, i > b ? t_trace[i].second - t_trace[i - 1].second : 0.0,
                t_trace[i].first);
    t_trace.clear();
}

int ensure(Ctx *ctx, DevBuf &b, size_t bytes) {
    if (bytes <= b.cap) return PCR_OK;
    size_t want = std::max(bytes, b.cap + b.cap / 2);
    want = (want + 255) & ~(size_t)255;
    if (b.p) {
        // the old block may still be in use by work queued on the stream: free it stream-ordered
        PCR_CUDA(ctx, cudaFreeAsync(b.p, ctx->stream));
        b.p = nullptr;
        b.cap = 0;
    }
    PCR_CUDA(ctx, cudaMallocAsync(&b.p, want, ctx->stream));
    b.cap = want;
    return PCR_OK;
}

int ensure_pinned(Ctx *ctx, size_t bytes) {
    if (bytes <= ctx->pinned_cap) return PCR_OK;
    size_t want = std::max<size_t>(bytes, 1 << 16);
    if (ctx->pinned) {
        PCR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFreeHost(ctx->pinned);
        ctx->pinned = nullptr;
        ctx->pinned_cap = 0;
    }
    PCR_CUDA(ctx, cudaHostAlloc(&ctx->pinned, want, cudaHostAllocMapped | cudaHostAllocPortable));
    ctx->pinned_cap = want;
    return PCR_OK;
}

namespace {

void free_buf(Ctx *ctx, DevBuf &b) {
    if (b.p) cudaFreeAsync(b.p, ctx->stream);
    b.p = nullptr;
    b.cap = 0;
}

int ctx_create(int device, void *stream, bool have_stream, Ctx **out) {
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(nullptr, PCR_ERR_NO_DEVICE, "no CUDA device available (%s); this library has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    if (device < 0 || device >= count) return fail(nullptr, PCR_ERR_INVALID_ARG, "device %d out of range [0,%d)", device, count);
    Ctx *ctx = new (std::nothrow) Ctx();
    if (!ctx) return fail(nullptr, PCR_ERR_OOM, "host allocation failed");
    ctx->device = device;
    struct Guard {  // a half-made context: give back what it already owns
        Ctx *c;
        ~Guard() {
            if (!c) return;
            if (c->pinned) cudaFreeHost(c->pinned);
            if (c->owns_stream && c->stream) cudaStreamDestroy(c->stream);
            delete c;
        }
    } g{ctx};
    PCR_CUDA(ctx, cudaSetDevice(device));
    cudaDeviceProp prop;
    PCR_CUDA(ctx, cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(nullptr, PCR_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major,
                    prop.minor);
    ctx->sm_count = prop.multiProcessorCount;
    if (have_stream) {
        ctx->stream = (cudaStream_t)stream;
        ctx->owns_stream = false;
    } else {
        PCR_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->owns_stream = true;
    }
    // keep freed blocks in the stream-ordered pool: index builds allocate and free every call
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    cudaGetLastError();
    PCR_TRY(ensure_pinned(ctx, 1 << 16));
    g.c = nullptr;
    *out = ctx;
    return PCR_OK;
}

struct DevSetter {  // every entry point runs on the context's device
    int prev = -1;
    explicit DevSetter(Ctx *c) {
        cudaGetDevice(&prev);
        if (prev != c->device) cudaSetDevice(c->device);
        else prev = -1;
    }
    ~DevSetter() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// stage three host arrays into one device buffer: returns device pointers
int stage_xyz(Ctx *ctx, DevBuf &buf, const float *x, const float *y, const float *z, size_t n, float **dx, float **dy, float **dz) {
    size_t stride = (n + 63) & ~(size_t)63;  // keeps every array 256 B aligned
    PCR_TRY(ensure(ctx, buf, sizeof(float) * 3 * std::max<size_t>(stride, 64)));
    float *base = (float *)buf.p;
    *dx = base;
    *dy = base + stride;
    *dz = base + 2 * stride;
    if (n) {
        PCR_CUDA(ctx, cudaMemcpyAsync(*dx, x, sizeof(float) * n, cudaMemcpyHostToDevice, ctx->stream));
        PCR_CUDA(ctx, cudaMemcpyAsync(*dy, y, sizeof(float) * n, cudaMemcpyHostToDevice, ctx->stream));
        PCR_CUDA(ctx, cudaMemcpyAsync(*dz, z, sizeof(float) * n, cudaMemcpyHostToDevice, ctx->stream));
    }
    return PCR_OK;
}

#define PCR_API_BEGIN try {
#define PCR_API_END(ctx_expr)                                                         \
    }                                                                                 \
    catch (const std::bad_alloc &) { return pcr::fail((ctx_expr), PCR_ERR_OOM, "host allocation failed"); } \
    catch (...) { return pcr::fail((ctx_expr), PCR_ERR_CUDA, "unexpected C++ exception"); }

}  // namespace
}  // namespace pcr

using namespace pcr;

// struct pcr_ctx / pcr_index: pcr_internal.cuh

extern "C" {

int pcr_version(void) { return PCR_B200_VERSION; }

int pcr_device_count(void) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return count;
}

const char *pcr_last_error(const pcr_ctx *ctx) {
    // the context's message only if it is newer than this thread's last failure (which may have been reported
    // without a context: NULL-argument checks, cloud-handle checks, the NCCL id)
    if (ctx && !ctx->c.err.empty() && ctx->c.err_seq >= g_thread_err_seq) return ctx->c.err.c_str();
    return g_thread_error.c_str();
}

static int create_common(int device, void *stream, bool have, pcr_ctx **out) {
    if (!out) return fail(nullptr, PCR_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    PCR_API_BEGIN
    Ctx *c = nullptr;
    PCR_TRY(ctx_create(device, stream, have, &c));
    pcr_ctx *w = new (std::nothrow) pcr_ctx();
    if (!w) {
        delete c;
        return fail(nullptr, PCR_ERR_OOM, "host allocation failed");
    }
    w->c = *c;  // plain members only
    delete c;
    *out = w;
    return PCR_OK;
    PCR_API_END(nullptr)
}

int pcr_ctx_create(int device, pcr_ctx **out) { return create_common(device, nullptr, false, out); }
int pcr_ctx_create_on_stream(int device, void *cuda_stream, pcr_ctx **out) { return create_common(device, cuda_stream, true, out); }

void pcr_ctx_destroy(pcr_ctx *ctx) {
    if (!ctx) return;
    trace_dump();
    Ctx *c = &ctx->c;
    DevSetter ds(c);
    cudaStreamSynchronize(c->stream);
    comm_destroy(c);
    free_buf(c, c->b_in);
    free_buf(c, c->b_in2);
    free_buf(c, c->b_out);
    free_buf(c, c->b_misc);
    free_buf(c, c->b_misc2);
    free_buf(c, c->b_small);
    free_buf(c, c->b_table);
    free_buf(c, c->b_scan);
    free_buf(c, c->b_fine_misc);
    free_buf(c, c->b_fine_scan);
    free_buf(c, c->b_list);
    free_buf(c, c->b_qoff);
    for (auto &b : c->b_cells) free_buf(c, b);
    for (auto &b : c->b_lsorted) free_buf(c, b);
    for (auto &b : c->b_lgrids) free_buf(c, b);
    cudaStreamSynchronize(c->stream);
    for (auto &sp : c->spans) {
        cudaEventDestroy(sp.a);
        cudaEventDestroy(sp.b);
    }
    for (auto e : c->event_pool) cudaEventDestroy(e);
    if (c->d_knn_stats) cudaFree(c->d_knn_stats);
    for (int i = 0; i < 2; i++) {
        if (c->side[i]) cudaStreamDestroy(c->side[i]);
        if (c->ev_join[i]) cudaEventDestroy(c->ev_join[i]);
    }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_count) cudaEventDestroy(c->ev_count);
    if (c->pinned) cudaFreeHost(c->pinned);
    if (c->owns_stream) cudaStreamDestroy(c->stream);
    cudaGetLastError();
    delete ctx;
}

int pcr_ctx_synchronize(pcr_ctx *ctx) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    DevSetter ds(&ctx->c);
    PCR_CUDA(&ctx->c, cudaStreamSynchronize(ctx->c.stream));
    return PCR_OK;
}

uint64_t pcr_ctx_launch_count(const pcr_ctx *ctx) { return ctx ? ctx->c.launches : 0; }

int pcr_ctx_set_timing(pcr_ctx *ctx, int enable) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    c->timing = enable != 0;
    if (c->timing && !c->d_knn_stats) {  // counters of the level-0 selection kernel (pcr_ctx_get_knn_counters)
        DevSetter ds(c);
        PCR_CUDA(c, cudaMalloc((void **)&c->d_knn_stats, 2 * sizeof(unsigned long long)));
        PCR_CUDA(c, cudaMemsetAsync(c->d_knn_stats, 0, 2 * sizeof(unsigned long long), c->stream));
    }
    return PCR_OK;
}

int pcr_ctx_get_timing(pcr_ctx *ctx, double *ms_per_tag, uint64_t *spans_per_tag) {
    if (!ctx || !ms_per_tag) return fail(nullptr, PCR_ERR_INVALID_ARG, "null pointer");
    Ctx *c = &ctx->c;
    DevSetter ds(c);
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int t = 0; t < PCR_NUM_TIMING_TAGS; t++) {
        ms_per_tag[t] = 0.0;
        if (spans_per_tag) spans_per_tag[t] = 0;
    }
    for (auto &sp : c->spans) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, sp.a, sp.b) == cudaSuccess && sp.tag >= 0 && sp.tag < PCR_NUM_TIMING_TAGS) {
            ms_per_tag[sp.tag] += ms;
            if (spans_per_tag) spans_per_tag[sp.tag]++;
        }
        c->event_pool.push_back(sp.a);
        c->event_pool.push_back(sp.b);
    }
    cudaGetLastError();
    c->spans.clear();
    return PCR_OK;
}

int pcr_ctx_get_knn_counters(pcr_ctx *ctx, uint64_t out[2]) {
    if (!ctx || !out) return fail(ctx ? &ctx->c : nullptr, PCR_ERR_INVALID_ARG, "null pointer");
    Ctx *c = &ctx->c;
    out[0] = out[1] = 0;
    if (!c->d_knn_stats) return PCR_OK;
    DevSetter ds(c);
    unsigned long long h[2] = {0, 0};
    PCR_CUDA(c, cudaMemcpyAsync(h, c->d_knn_stats, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaMemsetAsync(c->d_knn_stats, 0, sizeof(h), c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    out[0] = h[0];
    out[1] = h[1];
    return PCR_OK;
}

int pcr_ctx_set_frame_stream(pcr_ctx *ctx, int enable) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    ctx->c.frame_stream = enable != 0;
    ctx->c.cell_cache.valid = false;
    ctx->c.vox_cache.valid = false;
    return PCR_OK;
}

int pcr_ctx_set_query_sharding(pcr_ctx *ctx, int enable) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    ctx->c.shard_queries = enable != 0;
    return PCR_OK;
}

int pcr_ctx_debug_set_shard(pcr_ctx *ctx, int rank, int world_size) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (world_size < 1 || rank < 0 || rank >= world_size) return fail(c, PCR_ERR_INVALID_ARG, "bad rank/world");
    comm_destroy(c);
    c->rank = rank;
    c->world = world_size;
    c->fake_comm = world_size > 1;
    return PCR_OK;
}

int pcr_ctx_get_hint_stats(pcr_ctx *ctx, uint64_t out[PCR_NUM_HINT_STATS]) {
    if (!ctx || !out) return fail(ctx ? &ctx->c : nullptr, PCR_ERR_INVALID_ARG, "null pointer");
    const Ctx &c = ctx->c;
    const uint64_t v[PCR_NUM_HINT_STATS] = {c.stat_cell_hits, c.stat_cell_misses, c.stat_vox_hits, c.stat_vox_misses, c.stat_spec_hits, c.stat_spec_misses,
                                             c.stat_nowait_hits, c.stat_nowait_misses};
    for (int i = 0; i < PCR_NUM_HINT_STATS; i++) out[i] = v[i];
    return PCR_OK;
}

int pcr_ctx_set_cell_size(pcr_ctx *ctx, float cell_size) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    if (!(cell_size >= 0.f) || !std::isfinite(cell_size)) return fail(&ctx->c, PCR_ERR_INVALID_ARG, "cell_size must be >= 0 and finite");
    ctx->c.forced_cell = cell_size;
    return PCR_OK;
}

int pcr_comm_unique_id(void *out_id) {
    if (!out_id) return fail(nullptr, PCR_ERR_INVALID_ARG, "out_id is NULL");
    PCR_API_BEGIN
    return comm_unique_id(out_id);
    PCR_API_END(nullptr)
}
int pcr_ctx_comm_init(pcr_ctx *ctx, const void *id, int rank, int world_size) {
    if (!ctx || !id) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx/id is NULL");
    PCR_API_BEGIN
    DevSetter ds(&ctx->c);
    return comm_init(&ctx->c, id, rank, world_size);
    PCR_API_END(&ctx->c)
}
int pcr_ctx_comm_rank(const pcr_ctx *ctx) { return ctx ? ctx->c.rank : 0; }
int pcr_ctx_comm_size(const pcr_ctx *ctx) { return ctx ? ctx->c.world : 1; }
int pcr_ctx_comm_kind(const pcr_ctx *ctx) {
    if (!ctx || ctx->c.world <= 1 || ctx->c.fake_comm) return PCR_COMM_NONE;
    return ctx->c.peer_ok ? PCR_COMM_PEER : PCR_COMM_NCCL;
}

/* ---- index ------------------------------------------------------------------------------------ */
static int wrap_index(pcr_ctx *ctx, Index *ix, pcr_index **out) {
    pcr_index *w = new (std::nothrow) pcr_index();
    if (!w) {
        index_free(ix);
        return fail(&ctx->c, PCR_ERR_OOM, "host allocation failed");
    }
    w->ix = ix;
    w->owner = ctx;
    *out = w;
    return PCR_OK;
}

int pcr_index_build_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, size_t n, size_t k_hint,
                        pcr_index **out) {
    if (!ctx || !out) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx/out is NULL");
    *out = nullptr;
    if (n && (!d_x || !d_y || !d_z)) return fail(&ctx->c, PCR_ERR_INVALID_ARG, "x/y/z is NULL");
    PCR_API_BEGIN
    DevSetter ds(&ctx->c);
    BuildOpts bo;
    bo.k_hint = k_hint;
    Index *ix = nullptr;
    PCR_TRY(index_build_dev(&ctx->c, d_x, d_y, d_z, n, bo, &ix));
    return wrap_index(ctx, ix, out);
    PCR_API_END(&ctx->c)
}

int pcr_index_build(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n, size_t k_hint, pcr_index **out) {
    if (!ctx || !out) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx/out is NULL");
    *out = nullptr;
    if (n && (!x || !y || !z)) return fail(&ctx->c, PCR_ERR_INVALID_ARG, "x/y/z is NULL");
    PCR_API_BEGIN
    Ctx *c = &ctx->c;
    DevSetter ds(c);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    BuildOpts bo;
    bo.k_hint = k_hint;
    Index *ix = nullptr;
    PCR_TRY(index_build_dev(c, dx, dy, dz, n, bo, &ix));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return wrap_index(ctx, ix, out);
    PCR_API_END(&ctx->c)
}

void pcr_index_free(pcr_index *index) {
    if (!index) return;
    if (index->ix) {
        DevSetter ds(index->ix->ctx);
        index_free(index->ix);
    }
    delete index;
}

size_t pcr_index_len(const pcr_index *index) { return index && index->ix ? index->ix->n : 0; }

int pcr_index_info(const pcr_index *index, float *cell_size, int32_t dims[3], size_t *n_indexed) {
    if (!index || !index->ix) return fail(nullptr, PCR_ERR_INVALID_ARG, "index is NULL");
    const GridDesc &g = index->ix->grids_h[0];
    if (cell_size) *cell_size = (float)g.h;
    if (dims)
        for (int j = 0; j < 3; j++) dims[g.ax[j]] = g.dims[j];
    if (n_indexed) *n_indexed = index->ix->n_indexed;
    return PCR_OK;
}

// The single-cloud queries would mix the frames of a batch index (pcr_index_build_batch): they name the batch form instead.
static int single_cloud_check(const Index *ix, const char *batch_call) {
    if (ix->n_frames == 1) return PCR_OK;
    return fail(ix->ctx, PCR_ERR_INVALID_ARG, "the index holds %d frames: query it with %s", ix->n_frames, batch_call);
}

int pcr_knn_dev(pcr_index *index, const float *d_qx, const float *d_qy, const float *d_qz, size_t nq, size_t k, uint32_t *d_idx,
                float *d_dist, uint32_t *d_counts) {
    if (!index || !index->ix) return fail(nullptr, PCR_ERR_INVALID_ARG, "index is NULL");
    Ctx *c = index->ix->ctx;
    PCR_TRY(single_cloud_check(index->ix, "pcr_knn_batch_dev"));
    if (nq && k && (!d_qx || !d_qy || !d_qz || !d_idx)) return fail(c, PCR_ERR_INVALID_ARG, "null query/output pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    if (k == 0 && d_counts && nq) PCR_CUDA(c, cudaMemsetAsync(d_counts, 0, sizeof(uint32_t) * nq, c->stream));
    return knn_queries_dev(index->ix, d_qx, d_qy, d_qz, nq, k, d_idx, d_dist, d_counts);
    PCR_API_END(c)
}

int pcr_knn(pcr_index *index, const float *qx, const float *qy, const float *qz, size_t nq, size_t k, uint32_t *idx, float *dist,
            uint32_t *counts) {
    if (!index || !index->ix) return fail(nullptr, PCR_ERR_INVALID_ARG, "index is NULL");
    Ctx *c = index->ix->ctx;
    PCR_TRY(single_cloud_check(index->ix, "pcr_knn_batch"));
    if (nq == 0) return PCR_OK;
    if (!qx || !qy || !qz) return fail(c, PCR_ERR_INVALID_ARG, "null query pointer");
    if (k == 0) {  // kdtree.rs:65
        if (counts) memset(counts, 0, sizeof(uint32_t) * nq);
        return PCR_OK;
    }
    if (!idx) return fail(c, PCR_ERR_INVALID_ARG, "idx is NULL");
    if (k > PCR_MAX_K) return fail(c, PCR_ERR_UNSUPPORTED, "k = %zu exceeds PCR_MAX_K = %d", k, PCR_MAX_K);
    PCR_API_BEGIN
    DevSetter ds(c);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in2, qx, qy, qz, nq, &dx, &dy, &dz));
    size_t rows = nq * k;
    size_t bytes = rows * sizeof(uint32_t) + (dist ? rows * sizeof(float) : 0) + nq * sizeof(uint32_t) + 512;
    PCR_TRY(ensure(c, c->b_out, bytes));
    uint32_t *d_idx = (uint32_t *)c->b_out.p;
    float *d_dist = dist ? (float *)(d_idx + rows) : nullptr;
    uint32_t *d_cnt = (uint32_t *)((char *)c->b_out.p + rows * sizeof(uint32_t) + (dist ? rows * sizeof(float) : 0));
    PCR_TRY(knn_queries_dev(index->ix, dx, dy, dz, nq, k, d_idx, d_dist, d_cnt));
    PCR_CUDA(c, cudaMemcpyAsync(idx, d_idx, rows * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    if (dist) PCR_CUDA(c, cudaMemcpyAsync(dist, d_dist, rows * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    if (counts) PCR_CUDA(c, cudaMemcpyAsync(counts, d_cnt, nq * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_radius_count(pcr_index *index, const float *qx, const float *qy, const float *qz, size_t nq, float radius,
                     uint32_t *counts) {
    if (!index || !index->ix) return fail(nullptr, PCR_ERR_INVALID_ARG, "index is NULL");
    Ctx *c = index->ix->ctx;
    PCR_TRY(single_cloud_check(index->ix, "pcr_radius_count_batch"));
    if (nq == 0) return PCR_OK;
    if (!qx || !qy || !qz || !counts) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in2, qx, qy, qz, nq, &dx, &dy, &dz));
    PCR_TRY(ensure(c, c->b_out, nq * sizeof(uint32_t)));
    PCR_TRY(radius_count_dev(index->ix, dx, dy, dz, nq, radius, (uint32_t *)c->b_out.p));
    PCR_CUDA(c, cudaMemcpyAsync(counts, c->b_out.p, nq * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_radius_search(pcr_index *index, const float *qx, const float *qy, const float *qz, size_t nq, float radius,
                      uint64_t *offsets, uint32_t *idx, size_t cap, size_t *total) {
    if (!index || !index->ix) return fail(nullptr, PCR_ERR_INVALID_ARG, "index is NULL");
    Ctx *c = index->ix->ctx;
    PCR_TRY(single_cloud_check(index->ix, "pcr_radius_search_batch"));
    if (!offsets || !total) return fail(c, PCR_ERR_INVALID_ARG, "offsets/total is NULL");
    *total = 0;
    offsets[0] = 0;
    if (nq == 0) return PCR_OK;
    if (!qx || !qy || !qz) return fail(c, PCR_ERR_INVALID_ARG, "null query pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in2, qx, qy, qz, nq, &dx, &dy, &dz));
    // counts (u32) | offsets (u64, nq+1)
    size_t off_bytes = ((nq * sizeof(uint32_t) + 255) & ~(size_t)255);
    PCR_TRY(ensure(c, c->b_out, off_bytes + (nq + 1) * sizeof(uint64_t)));
    uint32_t *d_cnt = (uint32_t *)c->b_out.p;
    uint64_t *d_off = (uint64_t *)((char *)c->b_out.p + off_bytes);
    PCR_TRY(radius_count_dev(index->ix, dx, dy, dz, nq, radius, d_cnt));
    PCR_TRY(exclusive_scan_u64_from_u32_dev(c, d_cnt, d_off, nq));
    PCR_CUDA(c, cudaMemcpyAsync(offsets, d_off, (nq + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    *total = (size_t)offsets[nq];
    if (*total > cap) return fail(c, PCR_ERR_CAPACITY, "radius_search needs room for %zu indices, cap is %zu", *total, cap);
    if (*total == 0) return PCR_OK;
    if (!idx) return fail(c, PCR_ERR_INVALID_ARG, "idx is NULL");
    PCR_TRY(ensure(c, c->b_misc, *total * sizeof(uint32_t)));
    PCR_TRY(radius_fill_dev(index->ix, dx, dy, dz, nq, radius, d_off, (uint32_t *)c->b_misc.p));
    PCR_CUDA(c, cudaMemcpyAsync(idx, c->b_misc.p, *total * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return PCR_OK;
    PCR_API_END(c)
}

/* ---- SOR -------------------------------------------------------------------------------------- */
// shared by the host- and device-pointer entry points; d_stats: 4 floats, d_kept: 1 u64
static int sor_core(Ctx *c, const float *dx, const float *dy, const float *dz, size_t n, size_t k, float std_mul, uint8_t *d_keep,
                    float *d_mean, float *d_stats, unsigned long long *d_kept) {
    BuildOpts bo;
    bo.k_hint = k + 1;
    bo.self_knn = true;
    bo.transient = true;
    Index *ix = nullptr;
    PCR_TRY(index_build_dev(c, dx, dy, dz, n, bo, &ix));
    const IndexPtr guard(ix);
    // (a query-sharded context: every rank searches its share, the mean distances are merged, and every rank runs the
    // same exact fold over all of them -- the statistics and the mask do not depend on the number of ranks)
    PCR_TRY(sor_mean_dist_dev(ix, k, d_mean, nullptr, c->shard_queries));
    return sor_threshold_mask_dev(c, d_mean, nullptr, 1, n, std_mul, d_keep, d_stats, d_kept);
}

int pcr_sor_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, size_t n, size_t k, float std_mul,
                uint8_t *d_keep, float *d_mean_d) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (n && (!d_x || !d_y || !d_z || !d_keep)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (!std::isfinite(std_mul) || std_mul < 0.f) return fail(c, PCR_ERR_INVALID_ARG, "std_mul must be >= 0 and finite");
    if (k + 1 > PCR_MAX_K) return fail(c, PCR_ERR_UNSUPPORTED, "k = %zu exceeds PCR_MAX_K - 1", k);
    PCR_API_BEGIN
    DevSetter ds(c);
    if (n == 0) return PCR_OK;
    if (k == 0) {  // statistical_outlier.rs:5-7
        PCR_CUDA(c, cudaMemsetAsync(d_keep, 0, n, c->stream));
        return PCR_OK;
    }
    if (n == 1) {  // statistical_outlier.rs:10-12
        PCR_CUDA(c, cudaMemsetAsync(d_keep, 1, 1, c->stream));
        return PCR_OK;
    }
    PCR_TRY(ensure(c, c->b_out, n * sizeof(float) + 1024));
    float *d_mean = d_mean_d ? d_mean_d : (float *)c->b_out.p;
    float *d_stats = (float *)((char *)c->b_out.p + ((n * sizeof(float) + 255) & ~(size_t)255));
    unsigned long long *d_kept = (unsigned long long *)(d_stats + 8);
    return sor_core(c, d_x, d_y, d_z, n, k, std_mul, d_keep, d_mean, d_stats, d_kept);
    PCR_API_END(c)
}

int pcr_sor(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n, size_t k, float std_mul, uint8_t *keep,
            size_t *n_kept, float *mean_d, float *stats) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (n_kept) *n_kept = 0;
    if (n && (!x || !y || !z || !keep)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (!std::isfinite(std_mul) || std_mul < 0.f)  // crates/python/src/filters.rs:42-46
        return fail(c, PCR_ERR_INVALID_ARG, "std_mul must be >= 0 and finite");
    if (k + 1 > PCR_MAX_K) return fail(c, PCR_ERR_UNSUPPORTED, "k = %zu exceeds PCR_MAX_K - 1", k);
    if (stats) stats[0] = stats[1] = stats[2] = NAN;
    if (n == 0) return PCR_OK;
    if (k == 0) {  // statistical_outlier.rs:5-7: empty result
        memset(keep, 0, n);
        if (mean_d) std::fill(mean_d, mean_d + n, INFINITY);
        return PCR_OK;
    }
    if (n == 1) {  // statistical_outlier.rs:10-12: the cloud itself
        keep[0] = 1;
        if (n_kept) *n_kept = 1;
        if (mean_d) mean_d[0] = INFINITY;
        return PCR_OK;
    }
    PCR_API_BEGIN
    DevSetter ds(c);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    // out: mean_d f32[n] | stats f32[8] | kept u64 | keep u8[n]
    size_t o_stats = (n * sizeof(float) + 255) & ~(size_t)255;
    size_t o_keep = o_stats + 256;
    PCR_TRY(ensure(c, c->b_out, o_keep + n));
    float *d_mean = (float *)c->b_out.p;
    float *d_stats = (float *)((char *)c->b_out.p + o_stats);
    unsigned long long *d_kept = (unsigned long long *)(d_stats + 8);
    uint8_t *d_keep = (uint8_t *)c->b_out.p + o_keep;
    PCR_TRY(sor_core(c, dx, dy, dz, n, k, std_mul, d_keep, d_mean, d_stats, d_kept));
    struct {
        float stats[8];
        unsigned long long kept;
    } *mail = (decltype(mail))c->pinned;
    PCR_CUDA(c, cudaMemcpyAsync(keep, d_keep, n, cudaMemcpyDeviceToHost, c->stream));
    if (mean_d) PCR_CUDA(c, cudaMemcpyAsync(mean_d, d_mean, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaMemcpyAsync(mail, d_stats, sizeof(*mail), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    if (n_kept) *n_kept = (size_t)mail->kept;
    if (stats) {
        stats[0] = mail->stats[0];
        stats[1] = mail->stats[1];
        stats[2] = mail->stats[2];
    }
    return PCR_OK;
    PCR_API_END(c)
}

/* ---- radius outlier ------------------------------------------------------------------------------ */
namespace pcr {
__global__ void ror_mask_kernel(const uint32_t *__restrict__ counts, size_t n, uint64_t min_neighbors, uint8_t *__restrict__ keep,
                                unsigned long long *__restrict__ kept) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned k = 0;
    if (i < n) {
        k = (uint64_t)counts[i] >= min_neighbors ? 1 : 0;  // radius_outlier.rs:13
        keep[i] = (uint8_t)k;
    }
    k = __reduce_add_sync(PCR_FULL, k);
    if ((threadIdx.x & 31) == 0 && k) atomicAdd(kept, (unsigned long long)k);
}
}  // namespace pcr

// keep mask + kept count of radius_outlier_removal on device arrays (radius_outlier.rs:4-18).  frame_offsets (host,
// n_frames + 1): a batch of frames back to back, every point counted only within its own frame; a batch never shards.
static int ror_core(Ctx *c, const float *dx, const float *dy, const float *dz, size_t n, float radius, size_t min_neighbors,
                    uint8_t *d_keep, unsigned long long *d_kept, const uint64_t *frame_offsets = nullptr, size_t n_frames = 1) {
    // cell size = radius: the search box spans at most 3 cells per axis
    const float saved = c->forced_cell;
    if (saved == 0.f && radius > 0.f && std::isfinite(radius)) c->forced_cell = radius;
    BuildOpts bo;
    bo.transient = true;
    bo.n_frames = (int)n_frames;
    bo.frame_offsets = frame_offsets;
    Index *ix = nullptr;
    int s = index_build_dev(c, dx, dy, dz, n, bo, &ix);
    c->forced_cell = saved;
    PCR_TRY(s);
    const IndexPtr guard(ix);
    PCR_TRY(ensure(c, c->b_misc, n * sizeof(uint32_t)));
    uint32_t *d_cnt = (uint32_t *)c->b_misc.p;
    if (!frame_offsets && query_sharding_active(c, ix)) {
        // the count kernel takes its queries in input order: this rank counts for the input range [b, e), the counts are
        // merged like every sharded result (zero elsewhere, integer sum over NCCL), the mask is computed by every rank
        const size_t b = n * (size_t)c->rank / (size_t)c->world, e = n * (size_t)(c->rank + 1) / (size_t)c->world;
        PCR_CUDA(c, cudaMemsetAsync(d_cnt, 0, n * sizeof(uint32_t), c->stream));
        PCR_TRY(radius_count_dev(ix, dx + b, dy + b, dz + b, e - b, radius, d_cnt + b));
        PCR_TRY(comm_allreduce_u32(c, d_cnt, n));
    } else {
        PCR_TRY(radius_count_dev(ix, dx, dy, dz, n, radius, d_cnt));
    }
    PCR_CUDA(c, cudaMemsetAsync(d_kept, 0, sizeof(unsigned long long), c->stream));
    ror_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(d_cnt, n, (uint64_t)min_neighbors, d_keep, d_kept);
    PCR_LAUNCH_CHECK(c);
    return PCR_OK;
}

int pcr_radius_outlier_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, size_t n, float radius,
                           size_t min_neighbors, uint8_t *d_keep) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (n && (!d_x || !d_y || !d_z || !d_keep)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (n == 0) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    PCR_TRY(ensure(c, c->b_small, 4096));
    return ror_core(c, d_x, d_y, d_z, n, radius, min_neighbors, d_keep, (unsigned long long *)((char *)c->b_small.p + 1024));
    PCR_API_END(c)
}

int pcr_radius_outlier(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n, float radius, size_t min_neighbors,
                       uint8_t *keep, size_t *n_kept) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (n_kept) *n_kept = 0;
    if (n && (!x || !y || !z || !keep)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (n == 0) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    size_t o_kept = (n + 255) & ~(size_t)255;
    PCR_TRY(ensure(c, c->b_out, o_kept + 64));
    uint8_t *d_keep = (uint8_t *)c->b_out.p;
    unsigned long long *d_kept = (unsigned long long *)((char *)c->b_out.p + o_kept);
    PCR_TRY(ror_core(c, dx, dy, dz, n, radius, min_neighbors, d_keep, d_kept));
    unsigned long long *mail = (unsigned long long *)c->pinned;
    PCR_CUDA(c, cudaMemcpyAsync(keep, d_keep, n, cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaMemcpyAsync(mail, d_kept, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    if (n_kept) *n_kept = (size_t)*mail;
    return PCR_OK;
    PCR_API_END(c)
}

/* ---- voxel grid filter ------------------------------------------------------------------------------ */
int pcr_voxel_downsample_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, size_t n, float voxel_size,
                             float *d_ox, float *d_oy, float *d_oz, size_t *n_out) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (!n_out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *n_out = 0;
    if (!std::isfinite(voxel_size) || !(voxel_size > 0.f)) return fail(c, PCR_ERR_INVALID_ARG, "voxel_size must be > 0 and finite");
    if (n && (!d_x || !d_y || !d_z || !d_ox || !d_oy || !d_oz)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    return voxel_downsample_dev(c, d_x, d_y, d_z, n, voxel_size, d_ox, d_oy, d_oz, n_out);
    PCR_API_END(c)
}

int pcr_voxel_downsample(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n, float voxel_size, float *ox,
                         float *oy, float *oz, size_t *n_out) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (!n_out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *n_out = 0;
    if (!std::isfinite(voxel_size) || !(voxel_size > 0.f)) return fail(c, PCR_ERR_INVALID_ARG, "voxel_size must be > 0 and finite");
    if (n && (!x || !y || !z || !ox || !oy || !oz)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (n == 0) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    const size_t stride = (n + 63) & ~(size_t)63;
    PCR_TRY(ensure(c, c->b_out, sizeof(float) * 3 * stride));
    float *o0 = (float *)c->b_out.p, *o1 = o0 + stride, *o2 = o1 + stride;
    size_t m = 0;
    PCR_TRY(voxel_downsample_dev(c, dx, dy, dz, n, voxel_size, o0, o1, o2, &m));
    if (m) {
        PCR_CUDA(c, cudaMemcpyAsync(ox, o0, m * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaMemcpyAsync(oy, o1, m * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaMemcpyAsync(oz, o2, m * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    *n_out = m;
    return PCR_OK;
    PCR_API_END(c)
}

/* ---- segmentation ---------------------------------------------------------------------------------- */
int pcr_cluster_labels_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, size_t n, float distance_threshold,
                           uint32_t *d_labels) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (n && (!d_x || !d_y || !d_z || !d_labels)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (distance_threshold <= 0.0f) return fail(c, PCR_ERR_INVALID_ARG, "distance_threshold must be > 0");
    if (n == 0) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    return cluster_labels_dev(c, d_x, d_y, d_z, n, distance_threshold, d_labels);
    PCR_API_END(c)
}

int pcr_euclidean_cluster(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n, float distance_threshold,
                          size_t min_size, size_t max_size, uint32_t *offsets, uint32_t *indices, size_t *n_clusters) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (n_clusters) *n_clusters = 0;
    if (!offsets || !n_clusters) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    offsets[0] = 0;
    if (n && (!x || !y || !z || !indices)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (n == 0 || distance_threshold <= 0.0f || min_size == 0) return PCR_OK;  // euclidean_cluster.rs:102-104
    PCR_API_BEGIN
    DevSetter ds(c);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    PCR_TRY(ensure(c, c->b_out, n * sizeof(uint32_t)));
    uint32_t *d_labels = (uint32_t *)c->b_out.p;
    PCR_TRY(cluster_labels_dev(c, dx, dy, dz, n, distance_threshold, d_labels));
    std::vector<uint32_t> labels(n), scratch;
    PCR_CUDA(c, cudaMemcpyAsync(labels.data(), d_labels, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    *n_clusters = clusters_from_labels(labels.data(), n, min_size, max_size, offsets, indices, scratch);
    return PCR_OK;
    PCR_API_END(c)
}

/* ---- normals -------------------------------------------------------------------------------------- */
int pcr_estimate_normals_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, size_t n, size_t k,
                             const float viewpoint[3], float *d_nx, float *d_ny, float *d_nz) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (n == 0 || k == 0) return PCR_OK;  // estimate.rs:25-31
    if (!d_x || !d_y || !d_z || !d_nx || !d_ny || !d_nz || !viewpoint) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (k > PCR_MAX_K) return fail(c, PCR_ERR_UNSUPPORTED, "k = %zu exceeds PCR_MAX_K = %d", k, PCR_MAX_K);
    PCR_API_BEGIN
    DevSetter ds(c);
    BuildOpts bo;
    bo.k_hint = k;
    bo.self_knn = true;
    bo.transient = true;
    Index *ix = nullptr;
    PCR_TRY(index_build_dev(c, d_x, d_y, d_z, n, bo, &ix));
    const IndexPtr guard(ix);
    return normals_dev(ix, k, viewpoint, d_nx, d_ny, d_nz, nullptr, c->shard_queries);
    PCR_API_END(c)
}

int pcr_estimate_normals(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n, size_t k, const float viewpoint[3],
                         float *nx, float *ny, float *nz) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (n == 0 || k == 0) return PCR_OK;  // estimate.rs:25-31: empty normals
    if (!x || !y || !z || !nx || !ny || !nz || !viewpoint) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (k > PCR_MAX_K) return fail(c, PCR_ERR_UNSUPPORTED, "k = %zu exceeds PCR_MAX_K = %d", k, PCR_MAX_K);
    PCR_API_BEGIN
    DevSetter ds(c);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    size_t stride = (n + 63) & ~(size_t)63;
    PCR_TRY(ensure(c, c->b_out, stride * 3 * sizeof(float)));
    float *dnx = (float *)c->b_out.p, *dny = dnx + stride, *dnz = dny + stride;
    BuildOpts bo;
    bo.k_hint = k;
    bo.self_knn = true;
    bo.transient = true;
    Index *ix = nullptr;
    PCR_TRY(index_build_dev(c, dx, dy, dz, n, bo, &ix));
    PCR_TRY(normals_dev(IndexPtr(ix).get(), k, viewpoint, dnx, dny, dnz, nullptr, c->shard_queries));  // (freed before the copies)
    PCR_CUDA(c, cudaMemcpyAsync(nx, dnx, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaMemcpyAsync(ny, dny, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaMemcpyAsync(nz, dnz, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return PCR_OK;
    PCR_API_END(c)
}

/* ---- registration --------------------------------------------------------------------------------- */
int pcr_find_correspondences(pcr_index *target, const float *sx, const float *sy, const float *sz, size_t ns, float max_distance,
                             uint32_t *src_idx, uint32_t *tgt_idx, float *dist, size_t *count) {
    if (!target || !target->ix) return fail(nullptr, PCR_ERR_INVALID_ARG, "target is NULL");
    Ctx *c = target->ix->ctx;
    PCR_TRY(single_cloud_check(target->ix, "pcr_find_correspondences_batch"));
    if (!count) return fail(c, PCR_ERR_INVALID_ARG, "count is NULL");
    *count = 0;
    if (ns == 0) return PCR_OK;
    if (!sx || !sy || !sz || !src_idx || !tgt_idx || !dist) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in2, sx, sy, sz, ns, &dx, &dy, &dz));
    PCR_TRY(ensure(c, c->b_out, ns * 8));
    uint32_t *d_t = (uint32_t *)c->b_out.p;
    float *d_d = (float *)(d_t + ns);
    PCR_TRY(find_correspondences_dev(target->ix, dx, dy, dz, ns, max_distance, d_t, d_d));
    // compact on the host, in source order (correspondence.rs:23-36)
    std::vector<uint32_t> ht(ns);
    std::vector<float> hd(ns);
    PCR_CUDA(c, cudaMemcpyAsync(ht.data(), d_t, ns * 4, cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaMemcpyAsync(hd.data(), d_d, ns * 4, cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    size_t m = 0;
    for (size_t i = 0; i < ns; i++)
        if (ht[i] != 0xffffffffu) {
            src_idx[m] = (uint32_t)i;
            tgt_idx[m] = ht[i];
            dist[m] = hd[i];
            m++;
        }
    *count = m;
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_apply_transform(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n, const float rotation[9],
                        const float translation[3], float *ox, float *oy, float *oz) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (n == 0) return PCR_OK;
    if (!x || !y || !z || !ox || !oy || !oz || !rotation || !translation) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    size_t stride = (n + 63) & ~(size_t)63;
    PCR_TRY(ensure(c, c->b_out, stride * 3 * sizeof(float)));
    float *a = (float *)c->b_out.p, *b = a + stride, *d = b + stride;
    PCR_TRY(apply_transform_dev(c, dx, dy, dz, n, rotation, translation, a, b, d));
    PCR_CUDA(c, cudaMemcpyAsync(ox, a, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaMemcpyAsync(oy, b, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaMemcpyAsync(oz, d, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return PCR_OK;
    PCR_API_END(c)
}

static void icp_identity(pcr_icp_result *r) {
    memset(r, 0, sizeof(*r));
    r->rotation[0] = r->rotation[4] = r->rotation[8] = 1.f;
}

static int icp_common_dev(Ctx *c, const float *dsx, const float *dsy, const float *dsz, size_t ns, const float *dtx, const float *dty,
                          const float *dtz, size_t nt, const float *dnx, const float *dny, const float *dnz,
                          const pcr_icp_params *params, pcr_icp_result *result) {
    IcpArgs a;
    a.d_sx = dsx; a.d_sy = dsy; a.d_sz = dsz; a.ns = ns;
    a.d_tx = dtx; a.d_ty = dty; a.d_tz = dtz; a.nt = nt;
    a.d_nx = dnx; a.d_ny = dny; a.d_nz = dnz;
    a.params = *params;
    return icp_dev(c, a, result);
}

static int icp_check(Ctx *c, const pcr_icp_params *params, pcr_icp_result *result) {
    if (!params || !result) return fail(c, PCR_ERR_INVALID_ARG, "params/result is NULL");
    // crates/python/src/registration.rs:67-72: tolerance must not be NaN / negative
    if (std::isnan(params->tolerance) || params->tolerance < 0.f) return fail(c, PCR_ERR_INVALID_ARG, "tolerance must be >= 0");
    if (std::isnan(params->max_correspondence_distance) || params->max_correspondence_distance < 0.f)
        return fail(c, PCR_ERR_INVALID_ARG, "max_correspondence_distance must be >= 0");
    return PCR_OK;
}

static int icp_entry(pcr_ctx *ctx, bool dev, bool plane, const float *sx, const float *sy, const float *sz, size_t ns, const float *tx,
                     const float *ty, const float *tz, size_t nt, const float *nx, const float *ny, const float *nz, size_t nn,
                     const pcr_icp_params *params, pcr_icp_result *result) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    PCR_TRY(icp_check(c, params, result));
    icp_identity(result);
    if (plane && nn != nt)  // icp_plane.rs:27-32
        return fail(c, PCR_ERR_NORMALS_MISMATCH, "target_normals length (%zu) does not match target cloud length (%zu)", nn, nt);
    if (c->world == 1 && (ns == 0 || nt == 0)) {  // icp.rs:131-139
        result->converged = (ns == 0 && nt == 0) ? 1 : 0;
        return PCR_OK;
    }
    if (nt == 0) {
        result->converged = 0;
        return PCR_OK;
    }
    if ((ns && (!sx || !sy || !sz)) || !tx || !ty || !tz || (plane && (!nx || !ny || !nz))) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    if (dev) return icp_common_dev(c, sx, sy, sz, ns, tx, ty, tz, nt, plane ? nx : nullptr, ny, nz, params, result);
    float *dsx, *dsy, *dsz, *dtx, *dty, *dtz, *dnx = nullptr, *dny = nullptr, *dnz = nullptr;
    PCR_TRY(stage_xyz(c, c->b_in2, sx, sy, sz, ns, &dsx, &dsy, &dsz));
    PCR_TRY(stage_xyz(c, c->b_in, tx, ty, tz, nt, &dtx, &dty, &dtz));
    if (plane) PCR_TRY(stage_xyz(c, c->b_out, nx, ny, nz, nt, &dnx, &dny, &dnz));
    return icp_common_dev(c, dsx, dsy, dsz, ns, dtx, dty, dtz, nt, dnx, dny, dnz, params, result);
    PCR_API_END(c)
}

int pcr_icp_point_to_point(pcr_ctx *ctx, const float *sx, const float *sy, const float *sz, size_t ns, const float *tx,
                           const float *ty, const float *tz, size_t nt, const pcr_icp_params *params, pcr_icp_result *result) {
    return icp_entry(ctx, false, false, sx, sy, sz, ns, tx, ty, tz, nt, nullptr, nullptr, nullptr, nt, params, result);
}
int pcr_icp_point_to_plane(pcr_ctx *ctx, const float *sx, const float *sy, const float *sz, size_t ns, const float *tx,
                           const float *ty, const float *tz, size_t nt, const float *nx, const float *ny, const float *nz,
                           size_t n_normals, const pcr_icp_params *params, pcr_icp_result *result) {
    return icp_entry(ctx, false, true, sx, sy, sz, ns, tx, ty, tz, nt, nx, ny, nz, n_normals, params, result);
}
int pcr_icp_point_to_point_dev(pcr_ctx *ctx, const float *sx, const float *sy, const float *sz, size_t ns, const float *tx,
                               const float *ty, const float *tz, size_t nt, const pcr_icp_params *params, pcr_icp_result *result) {
    return icp_entry(ctx, true, false, sx, sy, sz, ns, tx, ty, tz, nt, nullptr, nullptr, nullptr, nt, params, result);
}
int pcr_icp_point_to_plane_dev(pcr_ctx *ctx, const float *sx, const float *sy, const float *sz, size_t ns, const float *tx,
                               const float *ty, const float *tz, size_t nt, const float *nx, const float *ny, const float *nz,
                               size_t n_normals, const pcr_icp_params *params, pcr_icp_result *result) {
    return icp_entry(ctx, true, true, sx, sy, sz, ns, tx, ty, tz, nt, nx, ny, nz, n_normals, params, result);
}

// Offsets of a batch argument (frame, query, sample or index offsets; `name` names it in the message): frame f = entries
// [offsets[f], offsets[f+1]), starting at 0, never decreasing.
static int offsets_check(Ctx *c, const char *name, const uint64_t *offsets, size_t n_frames) {
    if (!offsets) return fail(c, PCR_ERR_INVALID_ARG, "%s is NULL", name);
    if (offsets[0] != 0) return fail(c, PCR_ERR_INVALID_ARG, "%s must start at 0", name);
    for (size_t f = 0; f < n_frames; f++)
        if (offsets[f + 1] < offsets[f]) return fail(c, PCR_ERR_INVALID_ARG, "%s must be non-decreasing", name);
    return PCR_OK;
}
// ... and the sizes their kernels are built for: u32 point indices, one grid row per frame
static int batch_size_check(Ctx *c, size_t n, size_t n_frames) {
    if (n > 0x7fffffffull) return fail(c, PCR_ERR_UNSUPPORTED, "clouds above 2^31 points are not supported");
    if (n_frames > 65535) return fail(c, PCR_ERR_UNSUPPORTED, "at most 65535 frames per batch");
    return PCR_OK;
}

// Pairs of frames of one buffer: every pair is checked and answered as the single-pair call would (icp_entry).
static int icp_batch_entry(pcr_ctx *ctx, bool dev, bool plane, const float *x, const float *y, const float *z, const uint64_t *frame_offsets,
                           size_t n_frames, const float *nx, const float *ny, const float *nz, size_t n_normals, const uint32_t *pairs,
                           size_t n_pairs, const pcr_icp_params *params, pcr_icp_result *results) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    PCR_TRY(icp_check(c, params, results));
    for (size_t p = 0; p < n_pairs; p++) icp_identity(&results[p]);
    if (n_pairs && !pairs) return fail(c, PCR_ERR_INVALID_ARG, "pairs is NULL");
    PCR_TRY(offsets_check(c, "frame_offsets", frame_offsets, n_frames));
    const size_t n = (size_t)frame_offsets[n_frames];
    if (plane && n_normals != n)  // icp_plane.rs:27-32, for the whole buffer
        return fail(c, PCR_ERR_NORMALS_MISMATCH, "normals length (%zu) does not match the number of points (%zu)", n_normals, n);
    uint64_t src_points = 0;
    for (size_t p = 0; p < n_pairs; p++) {
        const uint32_t s = pairs[2 * p], t = pairs[2 * p + 1];
        if (s >= n_frames || t >= n_frames) return fail(c, PCR_ERR_INVALID_ARG, "pair %zu: frame id out of range (%zu frames)", p, n_frames);
        src_points += frame_offsets[s + 1] - frame_offsets[s];
    }
    if (src_points >= (1ull << 31)) return fail(c, PCR_ERR_UNSUPPORTED, "the source frames of one batch must hold fewer than 2^31 points");
    PCR_TRY(batch_size_check(c, n, n_frames));
    if (n && (!x || !y || !z || (plane && (!nx || !ny || !nz)))) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    IcpBatchArgs a;
    a.d_x = x; a.d_y = y; a.d_z = z; a.n = n;
    a.frame_offsets = frame_offsets; a.n_frames = n_frames;
    a.d_nx = a.d_ny = a.d_nz = nullptr;
    a.pairs = pairs; a.n_pairs = n_pairs;
    a.params = *params;
    if (dev) {
        if (plane) { a.d_nx = nx; a.d_ny = ny; a.d_nz = nz; }
        return icp_batch_dev(c, a, results);
    }
    float *dx, *dy, *dz, *dnx = nullptr, *dny = nullptr, *dnz = nullptr;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    if (plane) PCR_TRY(stage_xyz(c, c->b_out, nx, ny, nz, n, &dnx, &dny, &dnz));
    a.d_x = dx; a.d_y = dy; a.d_z = dz;
    a.d_nx = dnx; a.d_ny = dny; a.d_nz = dnz;
    return icp_batch_dev(c, a, results);
    PCR_API_END(c)
}

int pcr_icp_point_to_point_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z, const uint64_t *frame_offsets, size_t n_frames,
                                 const uint32_t *pairs, size_t n_pairs, const pcr_icp_params *params, pcr_icp_result *results) {
    return icp_batch_entry(ctx, false, false, x, y, z, frame_offsets, n_frames, nullptr, nullptr, nullptr, 0, pairs, n_pairs, params, results);
}
int pcr_icp_point_to_plane_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z, const uint64_t *frame_offsets, size_t n_frames,
                                 const float *nx, const float *ny, const float *nz, size_t n_normals, const uint32_t *pairs, size_t n_pairs,
                                 const pcr_icp_params *params, pcr_icp_result *results) {
    return icp_batch_entry(ctx, false, true, x, y, z, frame_offsets, n_frames, nx, ny, nz, n_normals, pairs, n_pairs, params, results);
}
int pcr_icp_point_to_point_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, const uint64_t *frame_offsets,
                                     size_t n_frames, const uint32_t *pairs, size_t n_pairs, const pcr_icp_params *params,
                                     pcr_icp_result *results) {
    return icp_batch_entry(ctx, true, false, d_x, d_y, d_z, frame_offsets, n_frames, nullptr, nullptr, nullptr, 0, pairs, n_pairs, params, results);
}
int pcr_icp_point_to_plane_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, const uint64_t *frame_offsets,
                                     size_t n_frames, const float *d_nx, const float *d_ny, const float *d_nz, size_t n_normals,
                                     const uint32_t *pairs, size_t n_pairs, const pcr_icp_params *params, pcr_icp_result *results) {
    return icp_batch_entry(ctx, true, true, d_x, d_y, d_z, frame_offsets, n_frames, d_nx, d_ny, d_nz, n_normals, pairs, n_pairs, params,
                           results);
}

/* ---- batched voxel_downsample and estimate_normals --------------------------------------------------- */
// Frames back to back; every frame gets what the single call returns for it alone.  Neither batch communicates or
// shards its queries: on a context with a communicator each rank processes the frames it was given.
static int voxel_batch_entry(pcr_ctx *ctx, bool dev, const float *x, const float *y, const float *z, const uint64_t *frame_offsets,
                             size_t n_frames, float voxel_size, float *ox, float *oy, float *oz, uint64_t *out_offsets) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (!out_offsets) return fail(c, PCR_ERR_INVALID_ARG, "out_offsets is NULL");
    out_offsets[0] = 0;
    PCR_TRY(offsets_check(c, "frame_offsets", frame_offsets, n_frames));
    for (size_t f = 1; f <= n_frames; f++) out_offsets[f] = 0;
    const size_t n = (size_t)frame_offsets[n_frames];
    PCR_TRY(batch_size_check(c, n, n_frames));
    if (!std::isfinite(voxel_size) || !(voxel_size > 0.f)) return fail(c, PCR_ERR_INVALID_ARG, "voxel_size must be > 0 and finite");
    if (n && (!x || !y || !z || !ox || !oy || !oz)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (n == 0) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    if (dev) return voxel_downsample_batch_dev(c, x, y, z, frame_offsets, n_frames, voxel_size, ox, oy, oz, out_offsets);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    const size_t stride = (n + 63) & ~(size_t)63;
    PCR_TRY(ensure(c, c->b_out, sizeof(float) * 3 * stride));
    float *o0 = (float *)c->b_out.p, *o1 = o0 + stride, *o2 = o1 + stride;
    PCR_TRY(voxel_downsample_batch_dev(c, dx, dy, dz, frame_offsets, n_frames, voxel_size, o0, o1, o2, out_offsets));
    const size_t m = (size_t)out_offsets[n_frames];
    if (m) {
        PCR_CUDA(c, cudaMemcpyAsync(ox, o0, m * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaMemcpyAsync(oy, o1, m * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaMemcpyAsync(oz, o2, m * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_voxel_downsample_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z, const uint64_t *frame_offsets, size_t n_frames,
                               float voxel_size, float *ox, float *oy, float *oz, uint64_t *out_offsets) {
    return voxel_batch_entry(ctx, false, x, y, z, frame_offsets, n_frames, voxel_size, ox, oy, oz, out_offsets);
}
int pcr_voxel_downsample_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, const uint64_t *frame_offsets,
                                   size_t n_frames, float voxel_size, float *d_ox, float *d_oy, float *d_oz, uint64_t *out_offsets) {
    return voxel_batch_entry(ctx, true, d_x, d_y, d_z, frame_offsets, n_frames, voxel_size, d_ox, d_oy, d_oz, out_offsets);
}

// One transient index over all frames (each frame searched only within itself), then the normals of every point: the
// non-SOR half of batch_core.
static int normals_batch_core(Ctx *c, const float *dx, const float *dy, const float *dz, const uint64_t *frame_offsets, size_t n_frames,
                              size_t n, size_t k, const float vp[3], float *d_nx, float *d_ny, float *d_nz) {
    BuildOpts bo;
    bo.k_hint = k;
    bo.self_knn = true;
    bo.n_frames = (int)n_frames;
    bo.frame_offsets = frame_offsets;
    bo.transient = true;
    Index *ix = nullptr;
    PCR_TRY(index_build_dev(c, dx, dy, dz, n, bo, &ix));
    const IndexPtr guard(ix);
    return normals_dev(ix, k, vp, d_nx, d_ny, d_nz, nullptr, /*allow_shard=*/false);
}

static int normals_batch_entry(pcr_ctx *ctx, bool dev, const float *x, const float *y, const float *z, const uint64_t *frame_offsets,
                               size_t n_frames, size_t k, const float viewpoint[3], float *nx, float *ny, float *nz) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    PCR_TRY(offsets_check(c, "frame_offsets", frame_offsets, n_frames));
    const size_t n = (size_t)frame_offsets[n_frames];
    PCR_TRY(batch_size_check(c, n, n_frames));
    if (n == 0 || k == 0) return PCR_OK;  // estimate.rs:25-31, as the single call
    if (!x || !y || !z || !nx || !ny || !nz || !viewpoint) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (k > PCR_MAX_K) return fail(c, PCR_ERR_UNSUPPORTED, "k = %zu exceeds PCR_MAX_K = %d", k, PCR_MAX_K);
    PCR_API_BEGIN
    DevSetter ds(c);
    if (dev) return normals_batch_core(c, x, y, z, frame_offsets, n_frames, n, k, viewpoint, nx, ny, nz);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    const size_t stride = (n + 63) & ~(size_t)63;
    PCR_TRY(ensure(c, c->b_out, stride * 3 * sizeof(float)));
    float *dnx = (float *)c->b_out.p, *dny = dnx + stride, *dnz = dny + stride;
    PCR_TRY(normals_batch_core(c, dx, dy, dz, frame_offsets, n_frames, n, k, viewpoint, dnx, dny, dnz));
    PCR_CUDA(c, cudaMemcpyAsync(nx, dnx, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaMemcpyAsync(ny, dny, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaMemcpyAsync(nz, dnz, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_estimate_normals_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z, const uint64_t *frame_offsets, size_t n_frames,
                               size_t k, const float viewpoint[3], float *nx, float *ny, float *nz) {
    return normals_batch_entry(ctx, false, x, y, z, frame_offsets, n_frames, k, viewpoint, nx, ny, nz);
}
int pcr_estimate_normals_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, const uint64_t *frame_offsets,
                                   size_t n_frames, size_t k, const float viewpoint[3], float *d_nx, float *d_ny, float *d_nz) {
    return normals_batch_entry(ctx, true, d_x, d_y, d_z, frame_offsets, n_frames, k, viewpoint, d_nx, d_ny, d_nz);
}

/* ---- batch index: the KdTree queries of many frames per call ----------------------------------------------- */
// A persistent index over frames back to back (it owns every level it builds: no context slot is borrowed), queried with
// frames of queries back to back, query frame f searched in index frame f only, indices frame-local.
static int index_build_batch_entry(pcr_ctx *ctx, bool dev, const float *x, const float *y, const float *z, const uint64_t *frame_offsets,
                                   size_t n_frames, size_t k_hint, pcr_index **out) {
    if (!ctx || !out) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx/out is NULL");
    *out = nullptr;
    Ctx *c = &ctx->c;
    if (n_frames == 0) return fail(c, PCR_ERR_INVALID_ARG, "a batch index holds at least one frame");
    PCR_TRY(offsets_check(c, "frame_offsets", frame_offsets, n_frames));
    const size_t n = (size_t)frame_offsets[n_frames];
    PCR_TRY(batch_size_check(c, n, n_frames));
    if (n && (!x || !y || !z)) return fail(c, PCR_ERR_INVALID_ARG, "x/y/z is NULL");
    PCR_API_BEGIN
    DevSetter ds(c);
    const float *dx = x, *dy = y, *dz = z;
    if (!dev) {
        float *sx, *sy, *sz;
        PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &sx, &sy, &sz));
        dx = sx; dy = sy; dz = sz;
    }
    BuildOpts bo;
    bo.k_hint = k_hint;
    bo.n_frames = (int)n_frames;
    bo.frame_offsets = frame_offsets;
    Index *ix = nullptr;
    PCR_TRY(index_build_dev(c, dx, dy, dz, n, bo, &ix));
    if (!dev) PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return wrap_index(ctx, ix, out);
    PCR_API_END(c)
}

int pcr_index_build_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z, const uint64_t *frame_offsets, size_t n_frames,
                          size_t k_hint, pcr_index **out) {
    return index_build_batch_entry(ctx, false, x, y, z, frame_offsets, n_frames, k_hint, out);
}
int pcr_index_build_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, const uint64_t *frame_offsets,
                              size_t n_frames, size_t k_hint, pcr_index **out) {
    return index_build_batch_entry(ctx, true, d_x, d_y, d_z, frame_offsets, n_frames, k_hint, out);
}

// The query side of a batch call: offsets as offsets_check, as many frames as the index, at most 0xfffffff0 queries.
static int batch_query_check(const Index *ix, const uint64_t *query_offsets, size_t n_frames, size_t *nq) {
    Ctx *c = ix->ctx;
    PCR_TRY(offsets_check(c, "query_offsets", query_offsets, n_frames));
    if (n_frames != (size_t)ix->n_frames)
        return fail(c, PCR_ERR_INVALID_ARG, "%zu query frames for an index of %d frames", n_frames, ix->n_frames);
    *nq = (size_t)query_offsets[n_frames];
    if (*nq > 0xfffffff0ull) return fail(c, PCR_ERR_UNSUPPORTED, "too many queries");
    return PCR_OK;
}

static int knn_batch_entry(pcr_index *index, bool dev, const float *qx, const float *qy, const float *qz, const uint64_t *query_offsets,
                           size_t n_frames, size_t k, uint32_t *idx, float *dist, uint32_t *counts) {
    if (!index || !index->ix) return fail(nullptr, PCR_ERR_INVALID_ARG, "index is NULL");
    Ctx *c = index->ix->ctx;
    size_t nq = 0;
    PCR_TRY(batch_query_check(index->ix, query_offsets, n_frames, &nq));
    if (nq == 0) return PCR_OK;
    if (!qx || !qy || !qz) return fail(c, PCR_ERR_INVALID_ARG, "null query pointer");
    if (k > PCR_MAX_K) return fail(c, PCR_ERR_UNSUPPORTED, "k = %zu exceeds PCR_MAX_K = %d", k, PCR_MAX_K);
    if (k && !idx) return fail(c, PCR_ERR_INVALID_ARG, "idx is NULL");
    PCR_API_BEGIN
    DevSetter ds(c);
    const QueryFrames qf = {query_offsets, n_frames};
    if (k == 0) {  // kdtree.rs:65
        if (counts && dev) PCR_CUDA(c, cudaMemsetAsync(counts, 0, sizeof(uint32_t) * nq, c->stream));
        if (counts && !dev) memset(counts, 0, sizeof(uint32_t) * nq);
        return PCR_OK;
    }
    if (dev) return knn_queries_dev(index->ix, qx, qy, qz, nq, k, idx, dist, counts, &qf);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in2, qx, qy, qz, nq, &dx, &dy, &dz));
    const size_t rows = nq * k;
    PCR_TRY(ensure(c, c->b_out, rows * sizeof(uint32_t) + (dist ? rows * sizeof(float) : 0) + nq * sizeof(uint32_t) + 512));
    uint32_t *d_idx = (uint32_t *)c->b_out.p;
    float *d_dist = dist ? (float *)(d_idx + rows) : nullptr;
    uint32_t *d_cnt = (uint32_t *)((char *)c->b_out.p + rows * sizeof(uint32_t) + (dist ? rows * sizeof(float) : 0));
    PCR_TRY(knn_queries_dev(index->ix, dx, dy, dz, nq, k, d_idx, d_dist, d_cnt, &qf));
    PCR_CUDA(c, cudaMemcpyAsync(idx, d_idx, rows * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    if (dist) PCR_CUDA(c, cudaMemcpyAsync(dist, d_dist, rows * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    if (counts) PCR_CUDA(c, cudaMemcpyAsync(counts, d_cnt, nq * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_knn_batch(pcr_index *index, const float *qx, const float *qy, const float *qz, const uint64_t *query_offsets, size_t n_frames,
                  size_t k, uint32_t *idx, float *dist, uint32_t *counts) {
    return knn_batch_entry(index, false, qx, qy, qz, query_offsets, n_frames, k, idx, dist, counts);
}
int pcr_knn_batch_dev(pcr_index *index, const float *d_qx, const float *d_qy, const float *d_qz, const uint64_t *query_offsets,
                      size_t n_frames, size_t k, uint32_t *d_idx, float *d_dist, uint32_t *d_counts) {
    return knn_batch_entry(index, true, d_qx, d_qy, d_qz, query_offsets, n_frames, k, d_idx, d_dist, d_counts);
}

static int radius_count_batch_entry(pcr_index *index, bool dev, const float *qx, const float *qy, const float *qz,
                                    const uint64_t *query_offsets, size_t n_frames, float radius, uint32_t *counts) {
    if (!index || !index->ix) return fail(nullptr, PCR_ERR_INVALID_ARG, "index is NULL");
    Ctx *c = index->ix->ctx;
    size_t nq = 0;
    PCR_TRY(batch_query_check(index->ix, query_offsets, n_frames, &nq));
    if (nq == 0) return PCR_OK;
    if (!qx || !qy || !qz || !counts) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    const QueryFrames qf = {query_offsets, n_frames};
    if (dev) return radius_count_dev(index->ix, qx, qy, qz, nq, radius, counts, &qf);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in2, qx, qy, qz, nq, &dx, &dy, &dz));
    PCR_TRY(ensure(c, c->b_out, nq * sizeof(uint32_t)));
    PCR_TRY(radius_count_dev(index->ix, dx, dy, dz, nq, radius, (uint32_t *)c->b_out.p, &qf));
    PCR_CUDA(c, cudaMemcpyAsync(counts, c->b_out.p, nq * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_radius_count_batch(pcr_index *index, const float *qx, const float *qy, const float *qz, const uint64_t *query_offsets,
                           size_t n_frames, float radius, uint32_t *counts) {
    return radius_count_batch_entry(index, false, qx, qy, qz, query_offsets, n_frames, radius, counts);
}
int pcr_radius_count_batch_dev(pcr_index *index, const float *d_qx, const float *d_qy, const float *d_qz, const uint64_t *query_offsets,
                               size_t n_frames, float radius, uint32_t *d_counts) {
    return radius_count_batch_entry(index, true, d_qx, d_qy, d_qz, query_offsets, n_frames, radius, d_counts);
}

int pcr_radius_search_batch(pcr_index *index, const float *qx, const float *qy, const float *qz, const uint64_t *query_offsets,
                            size_t n_frames, float radius, uint64_t *offsets, uint32_t *idx, size_t cap, size_t *total) {
    if (!index || !index->ix) return fail(nullptr, PCR_ERR_INVALID_ARG, "index is NULL");
    Ctx *c = index->ix->ctx;
    if (!offsets || !total) return fail(c, PCR_ERR_INVALID_ARG, "offsets/total is NULL");
    *total = 0;
    offsets[0] = 0;
    size_t nq = 0;
    PCR_TRY(batch_query_check(index->ix, query_offsets, n_frames, &nq));
    if (nq == 0) return PCR_OK;
    if (!qx || !qy || !qz) return fail(c, PCR_ERR_INVALID_ARG, "null query pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    const QueryFrames qf = {query_offsets, n_frames};
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in2, qx, qy, qz, nq, &dx, &dy, &dz));
    // counts (u32) | offsets (u64, nq+1), as pcr_radius_search
    size_t off_bytes = ((nq * sizeof(uint32_t) + 255) & ~(size_t)255);
    PCR_TRY(ensure(c, c->b_out, off_bytes + (nq + 1) * sizeof(uint64_t)));
    uint32_t *d_cnt = (uint32_t *)c->b_out.p;
    uint64_t *d_off = (uint64_t *)((char *)c->b_out.p + off_bytes);
    PCR_TRY(radius_count_dev(index->ix, dx, dy, dz, nq, radius, d_cnt, &qf));
    PCR_TRY(exclusive_scan_u64_from_u32_dev(c, d_cnt, d_off, nq));
    PCR_CUDA(c, cudaMemcpyAsync(offsets, d_off, (nq + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    *total = (size_t)offsets[nq];
    if (*total > cap) return fail(c, PCR_ERR_CAPACITY, "radius_search needs room for %zu indices, cap is %zu", *total, cap);
    if (*total == 0) return PCR_OK;
    if (!idx) return fail(c, PCR_ERR_INVALID_ARG, "idx is NULL");
    PCR_TRY(ensure(c, c->b_misc, *total * sizeof(uint32_t)));
    PCR_TRY(radius_fill_dev(index->ix, dx, dy, dz, nq, radius, d_off, (uint32_t *)c->b_misc.p, &qf));
    PCR_CUDA(c, cudaMemcpyAsync(idx, c->b_misc.p, *total * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_find_correspondences_batch(pcr_index *target, const float *sx, const float *sy, const float *sz, const uint64_t *query_offsets,
                                   size_t n_frames, float max_distance, uint32_t *src_idx, uint32_t *tgt_idx, float *dist,
                                   uint64_t *corr_offsets) {
    if (!target || !target->ix) return fail(nullptr, PCR_ERR_INVALID_ARG, "target is NULL");
    Ctx *c = target->ix->ctx;
    if (!corr_offsets) return fail(c, PCR_ERR_INVALID_ARG, "corr_offsets is NULL");
    size_t ns = 0;
    PCR_TRY(batch_query_check(target->ix, query_offsets, n_frames, &ns));
    for (size_t f = 0; f <= n_frames; f++) corr_offsets[f] = 0;
    if (ns == 0) return PCR_OK;
    if (!sx || !sy || !sz || !src_idx || !tgt_idx || !dist) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    const QueryFrames qf = {query_offsets, n_frames};
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in2, sx, sy, sz, ns, &dx, &dy, &dz));
    PCR_TRY(ensure(c, c->b_out, ns * 8));
    uint32_t *d_t = (uint32_t *)c->b_out.p;
    float *d_d = (float *)(d_t + ns);
    PCR_TRY(find_correspondences_dev(target->ix, dx, dy, dz, ns, max_distance, d_t, d_d, &qf));
    // compact on the host, frame by frame in source order (correspondence.rs:23-36); source indices frame-local
    std::vector<uint32_t> ht(ns);
    std::vector<float> hd(ns);
    PCR_CUDA(c, cudaMemcpyAsync(ht.data(), d_t, ns * 4, cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaMemcpyAsync(hd.data(), d_d, ns * 4, cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    size_t m = 0;
    for (size_t f = 0; f < n_frames; f++) {
        corr_offsets[f] = m;
        for (size_t i = (size_t)query_offsets[f]; i < (size_t)query_offsets[f + 1]; i++)
            if (ht[i] != 0xffffffffu) {
                src_idx[m] = (uint32_t)(i - (size_t)query_offsets[f]);
                tgt_idx[m] = ht[i];
                dist[m] = hd[i];
                m++;
            }
    }
    corr_offsets[n_frames] = m;
    return PCR_OK;
    PCR_API_END(c)
}

/* ---- batched RANSAC plane fit and euclidean_cluster ------------------------------------------------- */
// The back end of the obstacle pipeline over many frames; every frame gets what the single call returns for it alone.
// Neither batch communicates: on a context with a communicator each rank processes the frames it was given.
static int ransac_batch_entry(pcr_ctx *ctx, bool dev, const float *x, const float *y, const float *z, const uint64_t *frame_offsets,
                              size_t n_frames, float distance_threshold, const uint32_t *samples, const uint64_t *sample_offsets,
                              float *models, uint32_t *inliers, uint64_t *inlier_offsets) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (!models || !inlier_offsets) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    inlier_offsets[0] = 0;
    PCR_TRY(offsets_check(c, "frame_offsets", frame_offsets, n_frames));
    for (size_t f = 1; f <= n_frames; f++) inlier_offsets[f] = 0;
    const size_t n = (size_t)frame_offsets[n_frames];
    PCR_TRY(batch_size_check(c, n, n_frames));
    if (sample_offsets) {
        PCR_TRY(offsets_check(c, "sample_offsets", sample_offsets, n_frames));
        if (sample_offsets[n_frames] && !samples) return fail(c, PCR_ERR_INVALID_ARG, "samples is NULL");
        if (sample_offsets[n_frames] > 0x7fffffffull) return fail(c, PCR_ERR_UNSUPPORTED, "at most 2^31 - 1 sample triples per batch");
    } else if (samples) {
        return fail(c, PCR_ERR_INVALID_ARG, "sample_offsets is NULL");
    }
    if (n && (!x || !y || !z || !inliers)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    if (dev || n == 0)
        return ransac_plane_samples_batch_dev(c, x, y, z, frame_offsets, n_frames, distance_threshold, samples, sample_offsets, models, inliers,
                                              inlier_offsets);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    PCR_TRY(ensure(c, c->b_out, sizeof(uint32_t) * n));
    uint32_t *d_inl = (uint32_t *)c->b_out.p;
    PCR_TRY(ransac_plane_samples_batch_dev(c, dx, dy, dz, frame_offsets, n_frames, distance_threshold, samples, sample_offsets, models, d_inl,
                                           inlier_offsets));
    const size_t k = (size_t)inlier_offsets[n_frames];
    if (k) {
        PCR_CUDA(c, cudaMemcpyAsync(inliers, d_inl, sizeof(uint32_t) * k, cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_ransac_plane_samples_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z, const uint64_t *frame_offsets, size_t n_frames,
                                   float distance_threshold, const uint32_t *samples, const uint64_t *sample_offsets, float *models,
                                   uint32_t *inliers, uint64_t *inlier_offsets) {
    return ransac_batch_entry(ctx, false, x, y, z, frame_offsets, n_frames, distance_threshold, samples, sample_offsets, models, inliers,
                              inlier_offsets);
}
int pcr_ransac_plane_samples_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, const uint64_t *frame_offsets,
                                       size_t n_frames, float distance_threshold, const uint32_t *samples, const uint64_t *sample_offsets,
                                       float *models, uint32_t *d_inliers, uint64_t *inlier_offsets) {
    return ransac_batch_entry(ctx, true, d_x, d_y, d_z, frame_offsets, n_frames, distance_threshold, samples, sample_offsets, models, d_inliers,
                              inlier_offsets);
}

// in_dev: x, y, z are device pointers; dev: offsets and indices too (in_dev alone: the CSR is downloaded)
static int cluster_batch_entry(pcr_ctx *ctx, bool in_dev, bool dev, const float *x, const float *y, const float *z, const uint64_t *frame_offsets,
                               size_t n_frames, float distance_threshold, size_t min_size, size_t max_size, uint32_t *offsets,
                               uint32_t *indices, uint64_t *cluster_offsets) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (!offsets || !cluster_offsets) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    cluster_offsets[0] = 0;
    if (!dev) offsets[0] = 0;
    PCR_TRY(offsets_check(c, "frame_offsets", frame_offsets, n_frames));
    for (size_t f = 1; f <= n_frames; f++) cluster_offsets[f] = 0;
    const size_t n = (size_t)frame_offsets[n_frames];
    PCR_TRY(batch_size_check(c, n, n_frames));
    if (n && (!x || !y || !z || !indices)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    if (n == 0 || distance_threshold <= 0.0f || min_size == 0) {  // euclidean_cluster.rs:102-104, in every frame
        if (dev) {
            PCR_CUDA(c, cudaMemsetAsync(offsets, 0, sizeof(uint32_t), c->stream));
            PCR_CUDA(c, cudaStreamSynchronize(c->stream));
        }
        return PCR_OK;
    }
    size_t total = 0;
    if (dev)
        return euclidean_cluster_batch_dev(c, x, y, z, frame_offsets, n_frames, distance_threshold, min_size, max_size, offsets, indices,
                                           cluster_offsets, &total);
    const float *dx = x, *dy = y, *dz = z;
    if (!in_dev) {
        float *sx, *sy, *sz;
        PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &sx, &sy, &sz));
        dx = sx, dy = sy, dz = sz;
    }
    PCR_TRY(ensure(c, c->b_out, sizeof(uint32_t) * (2 * n + 1)));
    uint32_t *d_off = (uint32_t *)c->b_out.p, *d_idx = d_off + n + 1;
    PCR_TRY(euclidean_cluster_batch_dev(c, dx, dy, dz, frame_offsets, n_frames, distance_threshold, min_size, max_size, d_off, d_idx,
                                        cluster_offsets, &total));
    const size_t k = (size_t)cluster_offsets[n_frames];
    if (k) {
        PCR_CUDA(c, cudaMemcpyAsync(offsets, d_off, sizeof(uint32_t) * (k + 1), cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaMemcpyAsync(indices, d_idx, sizeof(uint32_t) * total, cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_euclidean_cluster_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z, const uint64_t *frame_offsets, size_t n_frames,
                                float distance_threshold, size_t min_size, size_t max_size, uint32_t *offsets, uint32_t *indices,
                                uint64_t *cluster_offsets) {
    return cluster_batch_entry(ctx, false, false, x, y, z, frame_offsets, n_frames, distance_threshold, min_size, max_size, offsets, indices,
                               cluster_offsets);
}
int pcr_euclidean_cluster_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, const uint64_t *frame_offsets,
                                    size_t n_frames, float distance_threshold, size_t min_size, size_t max_size, uint32_t *d_offsets,
                                    uint32_t *d_indices, uint64_t *cluster_offsets) {
    return cluster_batch_entry(ctx, true, true, d_x, d_y, d_z, frame_offsets, n_frames, distance_threshold, min_size, max_size, d_offsets, d_indices,
                               cluster_offsets);
}

int pcr_cluster_labels_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, const uint64_t *frame_offsets,
                                 size_t n_frames, float distance_threshold, uint32_t *d_labels) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    PCR_TRY(offsets_check(c, "frame_offsets", frame_offsets, n_frames));
    const size_t n = (size_t)frame_offsets[n_frames];
    PCR_TRY(batch_size_check(c, n, n_frames));
    if (n && (!d_x || !d_y || !d_z || !d_labels)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (distance_threshold <= 0.0f) return fail(c, PCR_ERR_INVALID_ARG, "distance_threshold must be > 0");
    if (n == 0) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    return cluster_labels_batch_dev(c, d_x, d_y, d_z, frame_offsets, n_frames, distance_threshold, d_labels);
    PCR_API_END(c)
}

/* ---- batched radius outlier removal ------------------------------------------------------------------ */
// One index over all frames (cell = radius, as for one cloud); every point counts only the points of its own frame.
static int ror_batch_entry(pcr_ctx *ctx, bool dev, const float *x, const float *y, const float *z, const uint64_t *frame_offsets,
                           size_t n_frames, float radius, size_t min_neighbors, uint8_t *keep, uint64_t *n_kept_per_frame) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    PCR_TRY(offsets_check(c, "frame_offsets", frame_offsets, n_frames));
    if (n_kept_per_frame)
        for (size_t f = 0; f < n_frames; f++) n_kept_per_frame[f] = 0;
    const size_t n = (size_t)frame_offsets[n_frames];
    PCR_TRY(batch_size_check(c, n, n_frames));
    if (n && (!x || !y || !z || !keep)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (n == 0) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    if (dev) {
        PCR_TRY(ensure(c, c->b_small, 4096));
        return ror_core(c, x, y, z, n, radius, min_neighbors, keep, (unsigned long long *)((char *)c->b_small.p + 1024), frame_offsets,
                        n_frames);
    }
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    const size_t o_kept = (n + 255) & ~(size_t)255;
    PCR_TRY(ensure(c, c->b_out, o_kept + 64));
    uint8_t *d_keep = (uint8_t *)c->b_out.p;
    PCR_TRY(ror_core(c, dx, dy, dz, n, radius, min_neighbors, d_keep, (unsigned long long *)((char *)c->b_out.p + o_kept), frame_offsets,
                     n_frames));
    PCR_CUDA(c, cudaMemcpyAsync(keep, d_keep, n, cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    if (n_kept_per_frame)
        for (size_t f = 0; f < n_frames; f++)
            for (uint64_t i = frame_offsets[f]; i < frame_offsets[f + 1]; i++) n_kept_per_frame[f] += keep[i];
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_radius_outlier_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z, const uint64_t *frame_offsets, size_t n_frames,
                             float radius, size_t min_neighbors, uint8_t *keep, uint64_t *n_kept_per_frame) {
    return ror_batch_entry(ctx, false, x, y, z, frame_offsets, n_frames, radius, min_neighbors, keep, n_kept_per_frame);
}
int pcr_radius_outlier_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, const uint64_t *frame_offsets,
                                 size_t n_frames, float radius, size_t min_neighbors, uint8_t *d_keep) {
    return ror_batch_entry(ctx, true, d_x, d_y, d_z, frame_offsets, n_frames, radius, min_neighbors, d_keep, nullptr);
}

/* ---- batched apply_transform --------------------------------------------------------------------------- */
// Frame f moved by transform f; the transform values are not checked (pcr_apply_transform does not check them either).
static int apply_transform_batch_entry(pcr_ctx *ctx, bool dev, const float *x, const float *y, const float *z, const uint64_t *frame_offsets,
                                       size_t n_frames, const float *transforms, float *ox, float *oy, float *oz) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    PCR_TRY(offsets_check(c, "frame_offsets", frame_offsets, n_frames));
    const size_t n = (size_t)frame_offsets[n_frames];
    PCR_TRY(batch_size_check(c, n, n_frames));
    if ((n_frames && !transforms) || (n && (!x || !y || !z || !ox || !oy || !oz))) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (n == 0) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    if (dev) return apply_transform_batch_dev(c, x, y, z, frame_offsets, n_frames, nullptr, transforms, ox, oy, oz);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    const size_t stride = (n + 63) & ~(size_t)63;
    PCR_TRY(ensure(c, c->b_out, sizeof(float) * 3 * stride));
    float *o0 = (float *)c->b_out.p, *o1 = o0 + stride, *o2 = o1 + stride;
    PCR_TRY(apply_transform_batch_dev(c, dx, dy, dz, frame_offsets, n_frames, nullptr, transforms, o0, o1, o2));
    PCR_CUDA(c, cudaMemcpyAsync(ox, o0, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaMemcpyAsync(oy, o1, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaMemcpyAsync(oz, o2, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_apply_transform_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z, const uint64_t *frame_offsets, size_t n_frames,
                              const float *transforms, float *ox, float *oy, float *oz) {
    return apply_transform_batch_entry(ctx, false, x, y, z, frame_offsets, n_frames, transforms, ox, oy, oz);
}
int pcr_apply_transform_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, const uint64_t *frame_offsets,
                                  size_t n_frames, const float *transforms, float *d_ox, float *d_oy, float *d_oz) {
    return apply_transform_batch_entry(ctx, true, d_x, d_y, d_z, frame_offsets, n_frames, transforms, d_ox, d_oy, d_oz);
}

// icp.rs:52-73 (RigidTransform::compose), the operation order of icp_step's compose (icp.cu): host code, built with
// -ffp-contract=off (Makefile) so that no product is fused into a sum.
int pcr_transform_compose(const float first[12], const float then[12], float out[12]) {
    if (!first || !then || !out) return fail(nullptr, PCR_ERR_INVALID_ARG, "null pointer");
    const float *A = then, *B = first;  // R = then.R * first.R, t = then.R * first.t + then.t
    float r[12];
    for (int i = 0; i < 3; i++) {
        for (int j = 0; j < 3; j++) r[i * 3 + j] = (A[i * 3 + 0] * B[0 * 3 + j] + A[i * 3 + 1] * B[1 * 3 + j]) + A[i * 3 + 2] * B[2 * 3 + j];
        r[9 + i] = ((A[i * 3 + 0] * B[9] + A[i * 3 + 1] * B[10]) + A[i * 3 + 2] * B[11]) + A[9 + i];
    }
    memcpy(out, r, sizeof(r));  // out may be first or then
    return PCR_OK;
}

/* ---- multi-frame batch ---------------------------------------------------------------------------- */
namespace pcr {
// frames of exactly one point are returned unchanged by the reference (statistical_outlier.rs:10-12)
__global__ void single_point_frames_kernel(const uint32_t *__restrict__ frame_off, int n_frames, size_t n,
                                           uint8_t *__restrict__ keep, unsigned long long *__restrict__ kept) {
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames) return;
    const size_t b = frame_off ? frame_off[f] : 0, e = frame_off ? frame_off[f + 1] : n;
    if (e - b == 1) {
        keep[b] = 1;
        kept[f] = 1;
    }
}
}  // namespace pcr
// One batched index over all frames for SOR, a second one over the kept points for the normals:
// every kernel runs once for the whole batch (frames are an extra axis of the cell table).
static int batch_core(Ctx *c, const float *dx, const float *dy, const float *dz, const uint64_t *frame_offsets, size_t n_frames,
                      size_t n, size_t k_sor, float std_mul, size_t k_normals, const float vp[3], uint8_t *d_keep, float *d_nx,
                      float *d_ny, float *d_nz, unsigned long long *d_kept /* n_frames */,
                      unsigned long long *h_kept0 = nullptr /* single frame: set if the count came back with another round trip */,
                      const CloudStats *known_stats = nullptr /* single frame: its box and finite count, if already measured */,
                      bool allow_nowait = true /* false: the redo of a call whose unawaited deferred counts were not zero */) {
    const int F = (int)n_frames;
    StreamAlloc<float> mean_mem(c->stream), stats_mem(c->stream);
    PCR_CUDA(c, mean_mem.alloc(sizeof(float) * std::max<size_t>(n, 1)));
    PCR_CUDA(c, stats_mem.alloc(sizeof(float) * 4 * F));
    float *d_mean = mean_mem.p, *d_stats = stats_mem.p;

    // ONE index serves both stages: built for the larger k, then the points SOR removes are
    // tombstoned in place (NaN coordinates) and the normals of the kept points run on the same grid.
    // Fused form: the SOR pass searches K = max(k_sor, k_normals) + 1 neighbours once and keeps the lists;
    // the normals of the kept points are computed from them (a kept point's nearest kept neighbours are
    // its nearest neighbours minus the removed ones), and only the queries that lose more neighbours
    // than the margin allows are searched again.  One KNN pass instead of two.
    // The lists are allocated -- and their lengths, the fallback counter and the kept counters initialised -- BEFORE the
    // index build: a memset between two kernels of the chain costs its own 2-3 us and breaks the programmatic launch
    // behind it; up here the device is still waiting for the host.
    const size_t K = std::max(k_sor, k_normals) + 1;
    static const bool no_fuse = getenv("PCR_NO_LIST_REUSE") != nullptr;  // A/B hook
    const bool may_fuse = !no_fuse && k_sor > 0 && k_normals > 0 && K <= 32 && n > 1;
    SorLists sl;
    bool early = false;
    StreamAlloc<uint32_t> list_mem(c->stream);
    if (may_fuse) {
        sl.K = K;
        sl.stride = (n + 63) & ~(size_t)63;  // (>= the indexed points, whose number the build has yet to report)
        const size_t bytes = sizeof(uint32_t) * (K * sl.stride + sl.stride + 64) + sl.stride;
        PCR_CUDA(c, list_mem.alloc(bytes));
        sl.lists = list_mem.p;
        sl.fallback = sl.lists + K * sl.stride;
        sl.cnt = (uint8_t *)(sl.fallback + sl.stride + 64);
        PCR_CUDA(c, cudaMemsetAsync(sl.fallback + sl.stride, 0, 64 * sizeof(uint32_t), c->stream));  // the fallback counter (and its padding)
        PCR_CUDA(c, cudaMemsetAsync(sl.cnt, 0xff, sl.stride, c->stream));                            // "no list yet"
        sl.initialised = true;
        PCR_MARK("core: lists allocated");
    }
    if (k_sor > 0) PCR_CUDA(c, cudaMemsetAsync(d_kept, 0, sizeof(unsigned long long) * F, c->stream));
    BuildOpts bo;
    bo.k_hint = std::max(k_sor + 1, k_normals);
    bo.self_knn = true;
    if (const char *e = getenv("PCR_BATCH_KHINT")) bo.k_hint = (size_t)atoi(e);
    bo.n_frames = F;
    bo.transient = true;
    bo.known_stats = known_stats;
    bo.frame_offsets = frame_offsets;
    Index *ix = nullptr;
    PCR_MARK("core: build begin");
    PCR_TRY(index_build_dev(c, dx, dy, dz, n, bo, &ix));
    PCR_MARK("core: build queued");
    const IndexPtr guard(ix);
    const bool fused = may_fuse && ix->n_indexed > 0;
    struct EarlyJoin {  // an error return between the early normals pass and its join: the lists are freed in stream order
        Ctx *c;
        bool *armed;
        ~EarlyJoin() {
            if (*armed) cudaStreamWaitEvent(c->stream, c->ev_join[0], 0);
        }
    } early_join{c, &early};
    if (k_sor == 0) {  // statistical_outlier.rs:5-7: empty result
        PCR_CUDA(c, cudaMemsetAsync(d_keep, 0, n, c->stream));
        PCR_CUDA(c, cudaMemsetAsync(d_kept, 0, sizeof(unsigned long long) * F, c->stream));
    } else {
        c->spec_request = fused && allow_nowait && F == 1 && k_normals > 0 && !c->shard_queries;
        c->spec_pending = false;
        const int ss = sor_mean_dist_dev(ix, k_sor, d_mean, fused ? &sl : nullptr);
        c->spec_request = false;
        PCR_TRY(ss);
        PCR_MARK("core: sor search done");
        // the normals of every query as if SOR removed nothing, beside the exact fold (which occupies 16 SMs per frame);
        // the pass after the mask only redoes the queries that lost one of their first k neighbours
        if (fused) PCR_TRY(normals_early_fork(c));
        PCR_TRY(sor_threshold_mask_dev(c, d_mean, ix->frame_in_off, F, n, std_mul, d_keep, d_stats, d_kept, true));
        if (fused) PCR_TRY(normals_early_from_lists_dev(ix, k_normals, vp, sl, d_nx, d_ny, d_nz, &early));
        PCR_MARK("core: stats queued");
        if (F > 1 || n == 1) {  // a one-point frame is returned as is, even if the point is not finite
            single_point_frames_kernel<<<(F + 127) / 128, 128, 0, c->stream>>>(ix->frame_in_off, F, n, d_keep, d_kept);
            PCR_LAUNCH_CHECK(c);
        }
    }
    if (k_normals == 0) return PCR_OK;
    if (early) PCR_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_join[0], 0));  // (the early pass reads the coordinates the mask is about to overwrite)
    PCR_TRY(index_apply_mask_dev(ix, d_keep));
    // removed points get 0 and kept non-finite points (0,0,1) inside normals_dev / normals_from_lists_dev
    if (fused) {
        const int sn = normals_from_lists_dev(ix, k_normals, vp, sl, d_keep, d_nx, d_ny, d_nz, F == 1 ? d_kept : nullptr, h_kept0, early);
        if (c->spec_pending) {  // the SOR pass's deferred counts, read by the round trip that just ended
            c->spec_pending = false;
            if (sn == PCR_OK) {
                const uint32_t *m2 = (const uint32_t *)c->pinned + 128;
                const bool zero = m2[0] == 0 && m2[1] == 0;
                c->spec_zero = zero;
                (zero ? c->stat_nowait_hits : c->stat_nowait_misses)++;
                if (!zero)  // queries were left for the coarser levels: everything downstream saw incomplete mean distances
                    return batch_core(c, dx, dy, dz, frame_offsets, (size_t)F, n, k_sor, std_mul, k_normals, vp, d_keep, d_nx, d_ny, d_nz, d_kept,
                                      h_kept0, known_stats, false);
            }
        }
        return sn;
    }
    return normals_dev(ix, k_normals, vp, d_nx, d_ny, d_nz, d_keep);
}

// The parameters the three pcr_sor_normals_batch forms check after their offsets and pointers
static int sor_normals_batch_check(Ctx *c, size_t n, size_t n_frames, size_t k_sor, float std_mul, size_t k_normals) {
    if (!std::isfinite(std_mul) || std_mul < 0.f) return fail(c, PCR_ERR_INVALID_ARG, "std_mul must be >= 0 and finite");
    if (k_sor + 1 > PCR_MAX_K || k_normals > PCR_MAX_K) return fail(c, PCR_ERR_UNSUPPORTED, "k exceeds PCR_MAX_K");
    return batch_size_check(c, n, n_frames);
}

int pcr_sor_normals_batch_dev(pcr_ctx *ctx, const float *d_x, const float *d_y, const float *d_z, const uint64_t *frame_offsets,
                              size_t n_frames, size_t k_sor, float std_mul, size_t k_normals, const float viewpoint[3],
                              uint8_t *d_keep, float *d_nx, float *d_ny, float *d_nz) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (n_frames == 0) return PCR_OK;
    PCR_TRY(offsets_check(c, "frame_offsets", frame_offsets, n_frames));
    const size_t n = (size_t)frame_offsets[n_frames];
    if (n == 0) return PCR_OK;
    if (!d_x || !d_y || !d_z || !d_keep || !viewpoint || (k_normals && (!d_nx || !d_ny || !d_nz)))
        return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_TRY(sor_normals_batch_check(c, n, n_frames, k_sor, std_mul, k_normals));
    PCR_API_BEGIN
    DevSetter ds(c);
    PCR_MARK("batch_dev: enter");
    StreamAlloc<unsigned long long> d_kept(c->stream);
    PCR_CUDA(c, d_kept.alloc(sizeof(unsigned long long) * n_frames));
    const int s = batch_core(c, d_x, d_y, d_z, frame_offsets, n_frames, n, k_sor, std_mul, k_normals, viewpoint, d_keep, d_nx, d_ny, d_nz,
                             d_kept.p);
    if (g_trace_on) {  // (tracing only: the entry point itself is asynchronous)
        cudaStreamSynchronize(c->stream);
        PCR_MARK("batch_dev: synced, exit");
    }
    return s;
    PCR_API_END(c)
}

int pcr_sor_normals_batch(pcr_ctx *ctx, const float *x, const float *y, const float *z, const uint64_t *frame_offsets, size_t n_frames,
                          size_t k_sor, float std_mul, size_t k_normals, const float viewpoint[3], uint8_t *keep, float *nx, float *ny,
                          float *nz, uint64_t *n_kept_per_frame) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (n_frames == 0) return PCR_OK;
    PCR_TRY(offsets_check(c, "frame_offsets", frame_offsets, n_frames));
    const size_t n = (size_t)frame_offsets[n_frames];
    if (n_kept_per_frame) memset(n_kept_per_frame, 0, sizeof(uint64_t) * n_frames);
    if (n == 0) return PCR_OK;
    if (!x || !y || !z || !keep || !viewpoint || (k_normals && (!nx || !ny || !nz))) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_TRY(sor_normals_batch_check(c, n, n_frames, k_sor, std_mul, k_normals));
    PCR_API_BEGIN
    DevSetter ds(c);
    float *dx, *dy, *dz;
    PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    size_t stride = (n + 63) & ~(size_t)63;
    size_t o_keep = stride * 3 * sizeof(float);
    size_t o_kept = o_keep + ((n + 255) & ~(size_t)255);
    PCR_TRY(ensure(c, c->b_out, o_kept + sizeof(unsigned long long) * n_frames));
    float *dnx = (float *)c->b_out.p, *dny = dnx + stride, *dnz = dny + stride;
    uint8_t *d_keep = (uint8_t *)c->b_out.p + o_keep;
    unsigned long long *d_kept = (unsigned long long *)((char *)c->b_out.p + o_kept);
    PCR_TRY(batch_core(c, dx, dy, dz, frame_offsets, n_frames, n, k_sor, std_mul, k_normals, viewpoint, d_keep, dnx, dny, dnz, d_kept));
    PCR_CUDA(c, cudaMemcpyAsync(keep, d_keep, n, cudaMemcpyDeviceToHost, c->stream));
    if (k_normals) {
        PCR_CUDA(c, cudaMemcpyAsync(nx, dnx, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaMemcpyAsync(ny, dny, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaMemcpyAsync(nz, dnz, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    }
    std::vector<unsigned long long> hk(n_frames);
    PCR_CUDA(c, cudaMemcpyAsync(hk.data(), d_kept, sizeof(unsigned long long) * n_frames, cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    if (n_kept_per_frame)
        for (size_t f = 0; f < n_frames; f++) n_kept_per_frame[f] = hk[f];
    return PCR_OK;
    PCR_API_END(c)
}

}  // extern "C"

/* ---- device-resident clouds (SURVEY 8f-3) -------------------------------------------------------------
 * PointCloud (crates/core/src/cloud.rs:4-18) kept in HBM between the steps of a pipeline
 * (voxel -> SOR -> normals -> cluster / ICP): one upload, one download, `select` as a device
 * compaction.  DevPoints is the storage of both handles (pcr_cloud and the frame batch pcr_frames):
 * one allocation, x | y | z | (nx | ny | nz), every array `stride` floats apart and 256 B aligned. */
struct DevPoints {
    pcr_ctx *owner = nullptr;
    size_t n = 0, stride = 0;
    float *base = nullptr;
    bool has_normals = false;
    int arrays() const { return has_normals ? 6 : 3; }
    float *x() const { return base; }
    float *y() const { return base + stride; }
    float *z() const { return base + 2 * stride; }
    float *nx() const { return base + 3 * stride; }
    float *ny() const { return base + 4 * stride; }
    float *nz() const { return base + 5 * stride; }
};

struct pcr_cloud : DevPoints {
    pcr::CloudStats stats;  // bounding box + finite count if the step that wrote the cloud measured them (stats.valid)
};

namespace pcr {
namespace {

// Owning handles: a failed call frees what it built, and `*out = h.release()` is the only place a handle is handed out.
struct HandleFree {
    void operator()(pcr_cloud *h) const { pcr_cloud_free(h); }
    void operator()(pcr_frames *h) const { pcr_frames_free(h); }
};
using CloudPtr = std::unique_ptr<pcr_cloud, HandleFree>;
using FramesPtr = std::unique_ptr<pcr_frames, HandleFree>;

// A new handle of n points on ctx, `tail` more bytes after its arrays (a frame batch keeps its offsets there).
template <class H>
int points_alloc(pcr_ctx *ctx, size_t n, bool normals, std::unique_ptr<H, HandleFree> &out, size_t tail = 0) {
    std::unique_ptr<H, HandleFree> h(new H());
    h->owner = ctx;
    h->n = n;
    h->stride = std::max<size_t>((n + 63) & ~(size_t)63, 64);
    h->has_normals = normals;
    float *base = nullptr;
    PCR_CUDA(&ctx->c, cudaMallocAsync((void **)&base, sizeof(float) * h->stride * h->arrays() + tail, ctx->c.stream));
    h->base = base;
    out = std::move(h);
    return PCR_OK;
}

template <class H>
void handle_free(H *h) {
    if (!h) return;
    if (h->base && h->owner) {
        DevSetter ds(&h->owner->c);
        cudaFreeAsync(h->base, h->owner->c.stream);
    }
    delete h;
}

__global__ void mask_to_u32_kernel(const uint8_t *__restrict__ keep, size_t n, uint32_t *__restrict__ flag) {
    PCR_GRID_DEP_SYNC();
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) flag[i] = (i < n && keep[i]) ? 1u : 0u;
}

// cloud.rs:103-140 as a stream compaction: kept points keep their order, normals travel along.  Rows 0..n_a-1
// come from `a`, rows n_a..n_a+n_b-1 from `b` (normals computed into a scratch block).
__global__ void compact_kernel(const float *__restrict__ a, size_t a_stride, int n_a, const float *__restrict__ b, size_t b_stride, int n_b,
                               size_t n, const uint32_t *__restrict__ pos /* exclusive scan of the flags, n + 1 */,
                               float *__restrict__ dst, size_t dst_stride) {
    PCR_GRID_DEP_SYNC();
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t p = pos[i];
    if (pos[i + 1] == p) return;
    for (int r = 0; r < n_a; r++) dst[(size_t)r * dst_stride + p] = a[(size_t)r * a_stride + i];
    for (int r = 0; r < n_b; r++) dst[(size_t)(n_a + r) * dst_stride + p] = b[(size_t)r * b_stride + i];
}

// (N, 3) rows <-> SoA rows, 256 points per block through shared memory so that both sides are coalesced
__global__ void __launch_bounds__(256) rows_to_soa_kernel(const float *__restrict__ rows, size_t n, float *__restrict__ dst, size_t dst_stride) {
    __shared__ float sh[768];
    const size_t p0 = (size_t)blockIdx.x * 256;
    const size_t m = min((size_t)256, n - p0);
    for (size_t i = threadIdx.x; i < 3 * m; i += 256) sh[i] = rows[3 * p0 + i];
    __syncthreads();
    if (threadIdx.x < m)
        for (int r = 0; r < 3; r++) dst[(size_t)r * dst_stride + p0 + threadIdx.x] = sh[3 * threadIdx.x + r];
}
__global__ void __launch_bounds__(256) soa_to_rows_kernel(const float *__restrict__ src, size_t src_stride, size_t n, float *__restrict__ rows) {
    __shared__ float sh[768];
    const size_t p0 = (size_t)blockIdx.x * 256;
    const size_t m = min((size_t)256, n - p0);
    if (threadIdx.x < m)
        for (int r = 0; r < 3; r++) sh[3 * threadIdx.x + r] = src[(size_t)r * src_stride + p0 + threadIdx.x];
    __syncthreads();
    for (size_t i = threadIdx.x; i < 3 * m; i += 256) rows[3 * p0 + i] = sh[i];
}

__global__ void gather_kernel(const float *__restrict__ src, size_t src_stride, int n_arrays, const uint32_t *__restrict__ idx, size_t m,
                              float *__restrict__ dst, size_t dst_stride) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const uint32_t i = idx[t];
    for (int a = 0; a < n_arrays; a++) dst[(size_t)a * dst_stride + t] = src[(size_t)a * src_stride + i];
}

// The first half of every compaction (a cloud's or a frame batch's): flags of the keep mask and their exclusive scan,
// pos[i] = kept points before point i, pos[n] = kept points.  pos lives in b_list.  Frames are contiguous and the
// compaction keeps the order, so one scan serves every frame of a batch: frame f starts at pos[frame_offsets[f]].
int keep_scan(Ctx *c, const uint8_t *d_keep, size_t n, uint32_t **pos_out) {
    // (measured and dropped: flags -> tile scan -> look-back -> scatter in ONE kernel: 10-13 us against 2.5 + 6.6 + 4.4 for the
    // three launches of a compaction -- 58 tiles of eight items per thread leave the GPU two thirds empty -- and no gain on the step)
    PCR_TRY(ensure(c, c->b_list, sizeof(uint32_t) * (n + 1)));
    uint32_t *pos = (uint32_t *)c->b_list.p;
    PCR_CUDA(c, launch_chained(mask_to_u32_kernel, dim3((unsigned)((n + 1 + 255) / 256)), dim3(256), 0, c->stream, d_keep, n, pos));
    c->launches++;
    PCR_TRY(exclusive_scan_u32_dev(c, pos, n + 1));
    *pos_out = pos;
    return PCR_OK;
}

// The second half of every compaction: the points of `in` whose pos[i + 1] != pos[i] go to row pos[i] of `out`, in order,
// normals along.  `nrm` (optional): normals of the points of `in`, three rows `nrm_stride` apart, for an `in` that
// carries none.
int compact_into(const DevPoints *in, const uint32_t *pos, const float *nrm, size_t nrm_stride, const DevPoints *out) {
    if (!out->n) return PCR_OK;
    Ctx *c = &in->owner->c;
    const int n_a = nrm ? 3 : in->arrays(), n_b = nrm ? 3 : 0;
    c->launches++;
    PCR_CUDA(c, launch_chained(compact_kernel, dim3((unsigned)((in->n + 255) / 256)), dim3(256), 0, c->stream, in->base, in->stride, n_a, nrm,
                               nrm_stride, n_b, in->n, pos, out->base, out->stride));
    return PCR_OK;
}

// new cloud = the points of `in` with keep != 0 (see compact_into).  `known_m`: the number of kept points if the caller
// already has it on the host (saves the round trip), else SIZE_MAX.
int cloud_compact(const pcr_cloud *in, const uint8_t *d_keep, CloudPtr &out, const float *nrm = nullptr, size_t nrm_stride = 0,
                  size_t known_m = SIZE_MAX) {
    Ctx *c = &in->owner->c;
    uint32_t *pos = nullptr;
    PCR_TRY(keep_scan(c, d_keep, in->n, &pos));
    size_t m = known_m;
    if (m == SIZE_MAX) {
        uint32_t *mail = (uint32_t *)c->pinned + 96;
        PCR_CUDA(c, cudaMemcpyAsync(mail, pos + in->n, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaStreamSynchronize(c->stream));
        m = *mail;
    }
    PCR_TRY(points_alloc(in->owner, m, nrm || in->has_normals, out));
    return compact_into(in, pos, nrm, nrm_stride, out.get());
}

// the first `arrays` arrays of dst <- those of src from point `first` on, dst->n points each
int copy_arrays(const DevPoints *src, size_t first, int arrays, const DevPoints *dst) {
    Ctx *c = &src->owner->c;
    for (int a = 0; dst->n && a < arrays; a++)
        PCR_CUDA(c, cudaMemcpyAsync(dst->base + (size_t)a * dst->stride, src->base + (size_t)a * src->stride + first, sizeof(float) * dst->n,
                                    cudaMemcpyDeviceToDevice, c->stream));
    return PCR_OK;
}

// The end of an upload: wait, so that the caller's buffers are free again on return, then report the first error.
int upload_wait(Ctx *c, cudaError_t upload) {
    const cudaError_t sync = cudaStreamSynchronize(c->stream);
    PCR_CUDA(c, upload);
    PCR_CUDA(c, sync);
    return PCR_OK;
}

// host x, y, z (n floats each) into the first three arrays of p
int points_upload(const DevPoints *p, const float *x, const float *y, const float *z) {
    Ctx *c = &p->owner->c;
    const float *src[3] = {x, y, z};
    cudaError_t upload = cudaSuccess;
    for (int a = 0; p->n && a < 3 && upload == cudaSuccess; a++)
        upload = cudaMemcpyAsync(p->base + (size_t)a * p->stride, src[a], sizeof(float) * p->n, cudaMemcpyHostToDevice, c->stream);
    return upload_wait(c, upload);
}

// Row-major (N, 3) in and out (the PyO3 surface's layout): one contiguous transfer, (de)interleaved on the device.
int points_upload_rows(const DevPoints *p, const float *xyz) {
    Ctx *c = &p->owner->c;
    const size_t n = p->n;
    cudaError_t upload = cudaSuccess;
    if (n) {
        PCR_TRY(ensure(c, c->b_in, sizeof(float) * 3 * n));
        upload = cudaMemcpyAsync(c->b_in.p, xyz, sizeof(float) * 3 * n, cudaMemcpyHostToDevice, c->stream);
        if (upload == cudaSuccess) {
            rows_to_soa_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>((const float *)c->b_in.p, n, p->base, p->stride);
            c->launches++;
            upload = cudaGetLastError();
        }
    }
    return upload_wait(c, upload);
}

int points_download_rows(const DevPoints *p, float *xyz, float *normals) {
    Ctx *c = &p->owner->c;
    const size_t n = p->n, row = sizeof(float) * 3 * n;
    PCR_TRY(ensure(c, c->b_out, 2 * row));
    float *d_xyz = (float *)c->b_out.p, *d_nrm = d_xyz + 3 * n;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    if (xyz) {
        soa_to_rows_kernel<<<blocks, 256, 0, c->stream>>>(p->base, p->stride, n, d_xyz);
        PCR_LAUNCH_CHECK(c);
        PCR_CUDA(c, cudaMemcpyAsync(xyz, d_xyz, row, cudaMemcpyDeviceToHost, c->stream));
    }
    if (normals) {
        soa_to_rows_kernel<<<blocks, 256, 0, c->stream>>>(p->nx(), p->stride, n, d_nrm);
        PCR_LAUNCH_CHECK(c);
        PCR_CUDA(c, cudaMemcpyAsync(normals, d_nrm, row, cudaMemcpyDeviceToHost, c->stream));
    }
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return PCR_OK;
}

// any of the six arrays to the host (n floats each): a NULL destination is skipped
int points_download(const DevPoints *p, float *x, float *y, float *z, float *nx, float *ny, float *nz) {
    Ctx *c = &p->owner->c;
    float *const dst[6] = {x, y, z, nx, ny, nz};
    for (int a = 0; a < 6; a++)
        if (dst[a]) PCR_CUDA(c, cudaMemcpyAsync(dst[a], p->base + (size_t)a * p->stride, sizeof(float) * p->n, cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return PCR_OK;
}

void points_device_pointers(const DevPoints *p, const float **d_x, const float **d_y, const float **d_z, const float **d_nx, const float **d_ny,
                            const float **d_nz) {
    const float **const dst[6] = {d_x, d_y, d_z, d_nx, d_ny, d_nz};
    for (int a = 0; a < 6; a++)
        if (dst[a]) *dst[a] = a < p->arrays() ? p->base + (size_t)a * p->stride : nullptr;
}

// a handle argument of a pcr_cloud_* / pcr_frames_* call: `what` names it
int handle_check(const DevPoints *h, const char *what) {
    if (h && h->owner) return PCR_OK;
    return fail(nullptr, PCR_ERR_INVALID_ARG, "%s is NULL", what);
}

}  // namespace
}  // namespace pcr


extern "C" {

int pcr_cloud_upload(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n, pcr_cloud **out) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (!out || (n && (!x || !y || !z))) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    PCR_API_BEGIN
    DevSetter ds(c);
    CloudPtr res;
    PCR_TRY(points_alloc(ctx, n, false, res));
    PCR_TRY(points_upload(res.get(), x, y, z));
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

void pcr_cloud_free(pcr_cloud *cloud) { handle_free(cloud); }

size_t pcr_cloud_len(const pcr_cloud *cloud) { return cloud ? cloud->n : 0; }
int pcr_cloud_has_normals(const pcr_cloud *cloud) { return cloud && cloud->has_normals ? 1 : 0; }

int pcr_cloud_device_pointers(const pcr_cloud *cloud, const float **d_x, const float **d_y, const float **d_z, const float **d_nx,
                              const float **d_ny, const float **d_nz) {
    PCR_TRY(handle_check(cloud, "cloud"));
    points_device_pointers(cloud, d_x, d_y, d_z, d_nx, d_ny, d_nz);
    return PCR_OK;
}

int pcr_cloud_download(const pcr_cloud *cloud, float *x, float *y, float *z) {
    PCR_TRY(handle_check(cloud, "cloud"));
    Ctx *c = &cloud->owner->c;
    if (cloud->n && (!x || !y || !z)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (!cloud->n) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    return points_download(cloud, x, y, z, nullptr, nullptr, nullptr);
    PCR_API_END(c)
}

int pcr_cloud_download_normals(const pcr_cloud *cloud, float *nx, float *ny, float *nz) {
    PCR_TRY(handle_check(cloud, "cloud"));
    Ctx *c = &cloud->owner->c;
    if (!cloud->has_normals) return fail(c, PCR_ERR_INVALID_ARG, "the cloud has no normals");
    if (cloud->n && (!nx || !ny || !nz)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (!cloud->n) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    return points_download(cloud, nullptr, nullptr, nullptr, nx, ny, nz);
    PCR_API_END(c)
}

int pcr_cloud_upload_rows(pcr_ctx *ctx, const float *xyz, size_t n, pcr_cloud **out) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (!out || (n && !xyz)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    PCR_API_BEGIN
    DevSetter ds(c);
    CloudPtr res;
    PCR_TRY(points_alloc(ctx, n, false, res));
    PCR_TRY(points_upload_rows(res.get(), xyz));
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_cloud_download_rows(const pcr_cloud *cloud, float *xyz, float *normals) {
    PCR_TRY(handle_check(cloud, "cloud"));
    Ctx *c = &cloud->owner->c;
    if (normals && !cloud->has_normals) return fail(c, PCR_ERR_INVALID_ARG, "the cloud has no normals");
    if (cloud->n && !xyz && !normals) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (!cloud->n) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    return points_download_rows(cloud, xyz, normals);
    PCR_API_END(c)
}

int pcr_sor_normals_batch_rows(pcr_ctx *ctx, const float *xyz, const uint64_t *frame_offsets, size_t n_frames, size_t k_sor, float std_mul,
                               size_t k_normals, const float viewpoint[3], uint8_t *keep, float *normals, uint64_t *n_kept_per_frame) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (n_frames == 0) return PCR_OK;
    PCR_TRY(offsets_check(c, "frame_offsets", frame_offsets, n_frames));
    const size_t n = (size_t)frame_offsets[n_frames];
    if (n_kept_per_frame) memset(n_kept_per_frame, 0, sizeof(uint64_t) * n_frames);
    if (n == 0) return PCR_OK;
    if (!xyz || !keep || !viewpoint || (k_normals && !normals)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_TRY(sor_normals_batch_check(c, n, n_frames, k_sor, std_mul, k_normals));
    PCR_API_BEGIN
    DevSetter ds(c);
    const size_t stride = (n + 63) & ~(size_t)63;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    // b_in: x | y | z (stride apart) | the rows as uploaded;  b_out: nx | ny | nz | keep | kept | the normals as rows
    PCR_TRY(ensure(c, c->b_in, sizeof(float) * (3 * stride + 3 * n)));
    float *dx = (float *)c->b_in.p, *d_rows = dx + 3 * stride;
    PCR_CUDA(c, cudaMemcpyAsync(d_rows, xyz, sizeof(float) * 3 * n, cudaMemcpyHostToDevice, c->stream));
    rows_to_soa_kernel<<<blocks, 256, 0, c->stream>>>(d_rows, n, dx, stride);
    PCR_LAUNCH_CHECK(c);
    const size_t o_keep = stride * 3 * sizeof(float);
    const size_t o_kept = o_keep + ((n + 255) & ~(size_t)255);
    const size_t o_rows = (o_kept + sizeof(unsigned long long) * n_frames + 255) & ~(size_t)255;
    PCR_TRY(ensure(c, c->b_out, o_rows + sizeof(float) * 3 * n));
    float *dnx = (float *)c->b_out.p, *dny = dnx + stride, *dnz = dny + stride;
    uint8_t *d_keep = (uint8_t *)c->b_out.p + o_keep;
    unsigned long long *d_kept = (unsigned long long *)((char *)c->b_out.p + o_kept);
    float *d_nrows = (float *)((char *)c->b_out.p + o_rows);
    PCR_TRY(batch_core(c, dx, dx + stride, dx + 2 * stride, frame_offsets, n_frames, n, k_sor, std_mul, k_normals, viewpoint, d_keep, dnx, dny, dnz,
                       d_kept));
    PCR_CUDA(c, cudaMemcpyAsync(keep, d_keep, n, cudaMemcpyDeviceToHost, c->stream));
    if (k_normals) {
        soa_to_rows_kernel<<<blocks, 256, 0, c->stream>>>(dnx, stride, n, d_nrows);
        PCR_LAUNCH_CHECK(c);
        PCR_CUDA(c, cudaMemcpyAsync(normals, d_nrows, sizeof(float) * 3 * n, cudaMemcpyDeviceToHost, c->stream));
    }
    std::vector<unsigned long long> hk(n_frames);
    PCR_CUDA(c, cudaMemcpyAsync(hk.data(), d_kept, sizeof(unsigned long long) * n_frames, cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    if (n_kept_per_frame)
        for (size_t f = 0; f < n_frames; f++) n_kept_per_frame[f] = hk[f];
    return PCR_OK;
    PCR_API_END(c)
}

// One strided copy each way for callers that keep their SoA arrays in one block (x | y | z [| nx | ny | nz], `stride`
// floats apart): a single cudaMemcpy2DAsync instead of three or six separate transfers.
static int upload_block(pcr_ctx *ctx, const float *xyz, size_t stride, size_t n, pcr_cloud **out, bool wait);
int pcr_cloud_upload_block(pcr_ctx *ctx, const float *xyz, size_t stride, size_t n, pcr_cloud **out) {
    return upload_block(ctx, xyz, stride, n, out, true);
}
int pcr_cloud_upload_block_nowait(pcr_ctx *ctx, const float *xyz, size_t stride, size_t n, pcr_cloud **out) {
    return upload_block(ctx, xyz, stride, n, out, false);
}
static int upload_block(pcr_ctx *ctx, const float *xyz, size_t stride, size_t n, pcr_cloud **out, bool wait) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (!out || (n && !xyz) || stride < n) return fail(c, PCR_ERR_INVALID_ARG, "null pointer or stride < n");
    *out = nullptr;
    PCR_API_BEGIN
    DevSetter ds(c);
    CloudPtr res;
    PCR_TRY(points_alloc(ctx, n, false, res));
    cudaError_t e = cudaSuccess;
    if (n) e = cudaMemcpy2DAsync(res->base, res->stride * sizeof(float), xyz, stride * sizeof(float), n * sizeof(float), 3, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess && wait) e = cudaStreamSynchronize(c->stream);  // the caller's buffer is free again on return
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(c, PCR_ERR_CUDA, "upload failed: %s", cudaGetErrorString(e));
    }
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_cloud_download_block(const pcr_cloud *cloud, float *dst, size_t stride, int with_normals) {
    PCR_TRY(handle_check(cloud, "cloud"));
    Ctx *c = &cloud->owner->c;
    if (with_normals && !cloud->has_normals) return fail(c, PCR_ERR_INVALID_ARG, "the cloud has no normals");
    if ((cloud->n && !dst) || stride < cloud->n) return fail(c, PCR_ERR_INVALID_ARG, "null pointer or stride < len");
    if (!cloud->n) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    PCR_CUDA(c, cudaMemcpy2DAsync(dst, stride * sizeof(float), cloud->base, cloud->stride * sizeof(float), cloud->n * sizeof(float),
                                  with_normals ? 6 : 3, cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_cloud_select(const pcr_cloud *cloud, const uint32_t *indices, size_t m, pcr_cloud **out) {
    PCR_TRY(handle_check(cloud, "cloud"));
    Ctx *c = &cloud->owner->c;
    if (!out || (m && !indices)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    for (size_t t = 0; t < m; t++)  // cloud.rs:109: select panics on an out-of-bounds index
        if (indices[t] >= cloud->n) return fail(c, PCR_ERR_INVALID_ARG, "index %u out of bounds for cloud with %zu points", indices[t], cloud->n);
    PCR_API_BEGIN
    DevSetter ds(c);
    CloudPtr res;
    PCR_TRY(points_alloc(cloud->owner, m, cloud->has_normals, res));
    if (m) {
        PCR_TRY(ensure(c, c->b_list, sizeof(uint32_t) * m));
        PCR_CUDA(c, cudaMemcpyAsync(c->b_list.p, indices, sizeof(uint32_t) * m, cudaMemcpyHostToDevice, c->stream));
        gather_kernel<<<(unsigned)((m + 255) / 256), 256, 0, c->stream>>>(cloud->base, cloud->stride, cloud->arrays(), (const uint32_t *)c->b_list.p,
                                                                          m, res->base, res->stride);
        PCR_LAUNCH_CHECK(c);
        PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_cloud_voxel_downsample(const pcr_cloud *cloud, float voxel_size, pcr_cloud **out) {
    PCR_TRY(handle_check(cloud, "cloud"));
    Ctx *c = &cloud->owner->c;
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    if (!std::isfinite(voxel_size) || !(voxel_size > 0.f)) return fail(c, PCR_ERR_INVALID_ARG, "voxel_size must be > 0 and finite");
    PCR_API_BEGIN
    DevSetter ds(c);
    PCR_MARK("voxel: enter");
    CloudPtr res;
    PCR_TRY(points_alloc(cloud->owner, cloud->n, false, res));  // voxel_downsample.rs:64: xyz only
    size_t m = 0;
    PCR_TRY(voxel_downsample_dev(c, cloud->x(), cloud->y(), cloud->z(), cloud->n, voxel_size, res->x(), res->y(), res->z(), &m, &res->stats));
    res->n = m;  // (the allocation keeps its original stride)
    *out = res.release();
    PCR_MARK("voxel: exit");
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_cloud_statistical_outlier_removal(const pcr_cloud *cloud, size_t k, float std_mul, pcr_cloud **out) {
    PCR_TRY(handle_check(cloud, "cloud"));
    Ctx *c = &cloud->owner->c;
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    PCR_API_BEGIN
    DevSetter ds(c);
    const size_t n = cloud->n;
    CloudPtr res;
    if (n == 0 || k == 0) {  // statistical_outlier.rs:5-7: PointCloud::new()
        PCR_TRY(points_alloc(cloud->owner, 0, false, res));
    } else {
        PCR_TRY(ensure(c, c->b_in2, n + 256));
        uint8_t *d_keep = (uint8_t *)c->b_in2.p;
        PCR_TRY(pcr_sor_dev(cloud->owner, cloud->x(), cloud->y(), cloud->z(), n, k, std_mul, d_keep, nullptr));
        PCR_TRY(cloud_compact(cloud, d_keep, res));  // :68 select
    }
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_cloud_radius_outlier_removal(const pcr_cloud *cloud, float radius, size_t min_neighbors, pcr_cloud **out) {
    PCR_TRY(handle_check(cloud, "cloud"));
    Ctx *c = &cloud->owner->c;
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    PCR_API_BEGIN
    DevSetter ds(c);
    const size_t n = cloud->n;
    CloudPtr res;
    if (n == 0) {
        PCR_TRY(points_alloc(cloud->owner, 0, cloud->has_normals, res));
    } else {
        PCR_TRY(ensure(c, c->b_in2, n + 256));
        uint8_t *d_keep = (uint8_t *)c->b_in2.p;
        PCR_TRY(pcr_radius_outlier_dev(cloud->owner, cloud->x(), cloud->y(), cloud->z(), n, radius, min_neighbors, d_keep));
        PCR_TRY(cloud_compact(cloud, d_keep, res));
    }
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_cloud_estimate_normals(const pcr_cloud *cloud, size_t k, const float viewpoint[3], pcr_cloud **out) {
    PCR_TRY(handle_check(cloud, "cloud"));
    Ctx *c = &cloud->owner->c;
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    // estimate.rs:25-31 returns EMPTY normals for k == 0, which no consumer accepts (icp_plane.rs:27-32): reported here
    if (k == 0) return fail(c, PCR_ERR_INVALID_ARG, "k must be > 0");
    PCR_API_BEGIN
    DevSetter ds(c);
    CloudPtr res;
    PCR_TRY(points_alloc(cloud->owner, cloud->n, true, res));
    PCR_TRY(copy_arrays(cloud, 0, 3, res.get()));
    const float vp0[3] = {0.f, 0.f, 0.f};  // estimate.rs:13-15
    PCR_TRY(pcr_estimate_normals_dev(cloud->owner, cloud->x(), cloud->y(), cloud->z(), cloud->n, k, viewpoint ? viewpoint : vp0, res->nx(),
                                     res->ny(), res->nz()));
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

// statistical_outlier_removal followed by estimate_normals on the kept points with ONE index (the points
// SOR removes are tombstoned in place, see batch_core): the fused form of the two calls above
int pcr_cloud_sor_normals(const pcr_cloud *cloud, size_t k_sor, float std_mul, size_t k_normals, const float viewpoint[3],
                          pcr_cloud **out) {
    PCR_TRY(handle_check(cloud, "cloud"));
    Ctx *c = &cloud->owner->c;
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    if (k_normals == 0) return fail(c, PCR_ERR_INVALID_ARG, "k_normals must be > 0");
    if (!std::isfinite(std_mul) || std_mul < 0.f) return fail(c, PCR_ERR_INVALID_ARG, "std_mul must be >= 0 and finite");
    if (k_sor + 1 > PCR_MAX_K || k_normals > PCR_MAX_K) return fail(c, PCR_ERR_UNSUPPORTED, "k exceeds PCR_MAX_K");
    PCR_API_BEGIN
    DevSetter ds(c);
    const size_t n = cloud->n;
    CloudPtr res;
    if (n == 0 || k_sor == 0) {  // statistical_outlier.rs:5-7
        PCR_TRY(points_alloc(cloud->owner, 0, true, res));
        *out = res.release();
        return PCR_OK;
    }
    PCR_MARK("sor_normals: enter");
    // normals by original index go to a scratch block; the kept points and their normals are compacted from the
    // input cloud and that block in one pass
    const size_t stride = (n + 63) & ~(size_t)63;
    StreamAlloc<float> nrm_mem(c->stream);
    PCR_CUDA(c, nrm_mem.alloc(sizeof(float) * 3 * stride));
    float *d_nrm = nrm_mem.p;
    PCR_TRY(ensure(c, c->b_in2, n + 512));
    uint8_t *d_keep = (uint8_t *)c->b_in2.p;
    unsigned long long *d_kept = (unsigned long long *)((char *)c->b_in2.p + ((n + 255) & ~(size_t)255));
    const uint64_t offs[2] = {0, n};
    const float vp0[3] = {0.f, 0.f, 0.f};
    unsigned long long h_kept = ~0ull;
    PCR_TRY(batch_core(c, cloud->x(), cloud->y(), cloud->z(), offs, 1, n, k_sor, std_mul, k_normals, viewpoint ? viewpoint : vp0, d_keep,
                       d_nrm, d_nrm + stride, d_nrm + 2 * stride, d_kept, &h_kept, cloud->stats.valid ? &cloud->stats : nullptr));
    PCR_MARK("sor_normals: core done");
    PCR_TRY(cloud_compact(cloud, d_keep, res, d_nrm, stride, h_kept == ~0ull ? SIZE_MAX : (size_t)h_kept));
    PCR_MARK("sor_normals: exit");
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_cloud_euclidean_cluster(const pcr_cloud *cloud, float distance_threshold, size_t min_size, size_t max_size, uint32_t *offsets,
                                uint32_t *indices, size_t *n_clusters) {
    PCR_TRY(handle_check(cloud, "cloud"));
    Ctx *c = &cloud->owner->c;
    if (n_clusters) *n_clusters = 0;
    if (!offsets || !n_clusters) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    offsets[0] = 0;
    const size_t n = cloud->n;
    if (n && !indices) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (n == 0 || distance_threshold <= 0.0f || min_size == 0) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    PCR_TRY(ensure(c, c->b_out, n * sizeof(uint32_t)));
    uint32_t *d_labels = (uint32_t *)c->b_out.p;
    PCR_TRY(cluster_labels_dev(c, cloud->x(), cloud->y(), cloud->z(), n, distance_threshold, d_labels));
    std::vector<uint32_t> labels(n), scratch;
    PCR_CUDA(c, cudaMemcpyAsync(labels.data(), d_labels, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    *n_clusters = clusters_from_labels(labels.data(), n, min_size, max_size, offsets, indices, scratch);
    return PCR_OK;
    PCR_API_END(c)
}

static int ransac_common(Ctx *c, const float *dx, const float *dy, const float *dz, size_t n, float thr, const uint32_t *samples, size_t m,
                         float model[4], uint32_t *inliers, size_t *n_inliers) {
    PCR_TRY(ensure(c, c->b_out, sizeof(uint32_t) * std::max<size_t>(n, 1)));
    uint32_t *d_inl = (uint32_t *)c->b_out.p;
    size_t k = 0;
    PCR_TRY(ransac_plane_samples_dev(c, dx, dy, dz, n, thr, samples, m, model, d_inl, &k));
    if (k) {
        PCR_CUDA(c, cudaMemcpyAsync(inliers, d_inl, sizeof(uint32_t) * k, cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    *n_inliers = k;
    return PCR_OK;
}

int pcr_ransac_plane_samples(pcr_ctx *ctx, const float *x, const float *y, const float *z, size_t n, float distance_threshold,
                             const uint32_t *samples, size_t m, float model[4], uint32_t *inliers, size_t *n_inliers) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    if (!model || !n_inliers || (m && !samples) || (n && (!x || !y || !z || !inliers))) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    float *dx = nullptr, *dy = nullptr, *dz = nullptr;
    if (n >= 3) PCR_TRY(stage_xyz(c, c->b_in, x, y, z, n, &dx, &dy, &dz));
    return ransac_common(c, dx, dy, dz, n, distance_threshold, samples, m, model, inliers, n_inliers);
    PCR_API_END(c)
}

int pcr_cloud_ransac_plane_samples(const pcr_cloud *cloud, float distance_threshold, const uint32_t *samples, size_t m, float model[4],
                                   uint32_t *inliers, size_t *n_inliers) {
    PCR_TRY(handle_check(cloud, "cloud"));
    Ctx *c = &cloud->owner->c;
    if (!model || !n_inliers || (m && !samples) || (cloud->n && !inliers)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    return ransac_common(c, cloud->x(), cloud->y(), cloud->z(), cloud->n, distance_threshold, samples, m, model, inliers, n_inliers);
    PCR_API_END(c)
}

int pcr_cloud_apply_transform(const pcr_cloud *cloud, const float rotation[9], const float translation[3], pcr_cloud **out) {
    PCR_TRY(handle_check(cloud, "cloud"));
    Ctx *c = &cloud->owner->c;
    if (!out || !rotation || !translation) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    PCR_API_BEGIN
    DevSetter ds(c);
    CloudPtr res;
    PCR_TRY(points_alloc(cloud->owner, cloud->n, false, res));  // icp.rs:91: xyz only
    if (cloud->n) PCR_TRY(apply_transform_dev(c, cloud->x(), cloud->y(), cloud->z(), cloud->n, rotation, translation, res->x(), res->y(), res->z()));
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_cloud_icp_point_to_point(const pcr_cloud *source, const pcr_cloud *target, const pcr_icp_params *params, pcr_icp_result *result) {
    PCR_TRY(handle_check(source, "cloud"));
    Ctx *c = &source->owner->c;
    if (!target || target->owner != source->owner) return fail(c, PCR_ERR_INVALID_ARG, "source and target must live on the same context");
    return pcr_icp_point_to_point_dev(source->owner, source->x(), source->y(), source->z(), source->n, target->x(), target->y(), target->z(),
                                      target->n, params, result);
}

int pcr_cloud_icp_point_to_plane(const pcr_cloud *source, const pcr_cloud *target, const pcr_icp_params *params, pcr_icp_result *result) {
    PCR_TRY(handle_check(source, "cloud"));
    Ctx *c = &source->owner->c;
    if (!target || target->owner != source->owner) return fail(c, PCR_ERR_INVALID_ARG, "source and target must live on the same context");
    if (!target->has_normals)  // crates/python/src/registration.rs:80-86
        return fail(c, PCR_ERR_INVALID_ARG, "target cloud must have normals (call estimate_normals first)");
    return pcr_icp_point_to_plane_dev(source->owner, source->x(), source->y(), source->z(), source->n, target->x(), target->y(), target->z(),
                                      target->n, target->nx(), target->ny(), target->nz(), target->n, params, result);
}

}  // extern "C"

/* ---- device-resident frame batches ----------------------------------------------------------------------
 * F clouds back to back in one allocation, laid out like pcr_cloud (x | y | z [| nx | ny | nz], `stride` floats apart),
 * then the frame offsets as the kernels read them (u32[F + 1]); the host keeps them as u64[F + 1].  Every method is a
 * batch core of the raw-pointer calls, and the filters end in ONE compaction for all frames (keep_scan, then the new
 * frame starts read off the scan, then compact_kernel): each frame's result is what the pcr_cloud method returns for it. */
struct pcr_frames : DevPoints {
    uint32_t *d_off = nullptr;
    std::vector<uint64_t> off;
    size_t count() const { return off.size() - 1; }
};

namespace pcr {
namespace {

// host offsets (u64[F + 1]) to the u32 copy the kernels read (pageable source: the copy has taken the bytes when it returns)
int offsets_upload(Ctx *c, const std::vector<uint64_t> &off, uint32_t *d_off) {
    const std::vector<uint32_t> h(off.begin(), off.end());
    PCR_CUDA(c, cudaMemcpyAsync(d_off, h.data(), sizeof(uint32_t) * h.size(), cudaMemcpyHostToDevice, c->stream));
    return PCR_OK;
}

// A new batch of n points with the given frame offsets.  d_off_src: the same offsets as u32 on the device (copied from
// there), else they are uploaded from `off`.
int frames_alloc(pcr_ctx *ctx, size_t n, bool normals, std::vector<uint64_t> off, FramesPtr &out, const uint32_t *d_off_src = nullptr) {
    Ctx *c = &ctx->c;
    FramesPtr fr;
    PCR_TRY(points_alloc(ctx, n, normals, fr, sizeof(uint32_t) * off.size()));
    fr->off = std::move(off);
    fr->d_off = (uint32_t *)(fr->base + fr->stride * fr->arrays());
    if (d_off_src)
        PCR_CUDA(c, cudaMemcpyAsync(fr->d_off, d_off_src, sizeof(uint32_t) * fr->off.size(), cudaMemcpyDeviceToDevice, c->stream));
    else
        PCR_TRY(offsets_upload(c, fr->off, fr->d_off));
    out = std::move(fr);
    return PCR_OK;
}

// the compacted batch's frame f starts where the scan stands at the old start of frame f
__global__ void frame_starts_kernel(const uint32_t *__restrict__ pos, const uint32_t *__restrict__ frame_off, int n_frames,
                                    uint32_t *__restrict__ new_off) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f <= n_frames) new_off[f] = pos[frame_off[f]];
}

// new batch = the points of `in` with keep != 0, frame by frame.  `nrm` (optional): normals of the points of `in`, three
// rows `nrm_stride` apart, for an `in` that carries none.  One round trip: all F + 1 new offsets in one copy.
int frames_compact(const pcr_frames *in, const uint8_t *d_keep, FramesPtr &out, const float *nrm = nullptr, size_t nrm_stride = 0) {
    Ctx *c = &in->owner->c;
    const size_t F = in->count();
    uint32_t *pos = nullptr;
    PCR_TRY(keep_scan(c, d_keep, in->n, &pos));
    StreamAlloc<uint32_t> new_off(c->stream);
    PCR_CUDA(c, new_off.alloc(sizeof(uint32_t) * (F + 1)));
    uint32_t *d_new = new_off.p;
    frame_starts_kernel<<<(unsigned)((F + 1 + 255) / 256), 256, 0, c->stream>>>(pos, in->d_off, (int)F, d_new);
    PCR_LAUNCH_CHECK(c);
    PCR_TRY(ensure_pinned(c, sizeof(uint32_t) * (F + 1)));
    uint32_t *mail = (uint32_t *)c->pinned;
    PCR_CUDA(c, cudaMemcpyAsync(mail, d_new, sizeof(uint32_t) * (F + 1), cudaMemcpyDeviceToHost, c->stream));
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    std::vector<uint64_t> off(F + 1);
    for (size_t f = 0; f <= F; f++) off[f] = mail[f];
    const size_t m = (size_t)off[F];
    PCR_TRY(frames_alloc(in->owner, m, nrm || in->has_normals, std::move(off), out, d_new));
    return compact_into(in, pos, nrm, nrm_stride, out.get());
}

// An empty batch with in's frame count: every frame empty (the SOR rule for k == 0).
int frames_empty(const pcr_frames *in, bool normals, FramesPtr &out) {
    return frames_alloc(in->owner, 0, normals, std::vector<uint64_t>(in->count() + 1, 0), out);
}

// Entry t of the frame-local lists (list f = [list_off[f], list_off[f+1])) names input point frame_off[f] + idx[t].
__device__ __forceinline__ uint32_t list_point(const uint32_t *__restrict__ idx, const uint32_t *__restrict__ list_off,
                                               const uint32_t *__restrict__ frame_off, int n_frames, uint32_t t) {
    return frame_off[frame_of(list_off, n_frames, t)] + idx[t];
}

__global__ void frames_gather_kernel(const float *__restrict__ src, size_t src_stride, int n_arrays, const uint32_t *__restrict__ idx,
                                     const uint32_t *__restrict__ list_off, const uint32_t *__restrict__ frame_off, int n_frames, size_t m,
                                     float *__restrict__ dst, size_t dst_stride) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const uint32_t i = list_point(idx, list_off, frame_off, n_frames, (uint32_t)t);
    for (int a = 0; a < n_arrays; a++) dst[(size_t)a * dst_stride + t] = src[(size_t)a * src_stride + i];
}

// keep[listed point] = 0 (select_inverse: the mask starts all ones)
__global__ void frames_unkeep_kernel(const uint32_t *__restrict__ idx, const uint32_t *__restrict__ list_off,
                                     const uint32_t *__restrict__ frame_off, int n_frames, size_t m, uint8_t *__restrict__ keep) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < m) keep[list_point(idx, list_off, frame_off, n_frames, (uint32_t)t)] = 0;
}

// select_inverse of frame-local DEVICE lists with HOST list offsets (in bounds, checked by the caller or by construction)
int frames_select_inverse_dev(const pcr_frames *in, const uint32_t *d_idx, const std::vector<uint64_t> &list_off, FramesPtr &out) {
    Ctx *c = &in->owner->c;
    const size_t n = in->n, F = in->count(), m = (size_t)list_off[F];
    // keep u8[n] (rounded up to 4 bytes) | list offsets u32[F + 1]
    const size_t o_loff = (n + 3) & ~(size_t)3;
    StreamAlloc<uint8_t> keep_mem(c->stream);
    PCR_CUDA(c, keep_mem.alloc(o_loff + sizeof(uint32_t) * (F + 1)));
    uint8_t *d_keep = keep_mem.p;
    uint32_t *d_loff = (uint32_t *)(d_keep + o_loff);
    if (n) PCR_CUDA(c, cudaMemsetAsync(d_keep, 1, n, c->stream));
    if (m) {
        PCR_TRY(offsets_upload(c, list_off, d_loff));
        frames_unkeep_kernel<<<(unsigned)((m + 255) / 256), 256, 0, c->stream>>>(d_idx, d_loff, in->d_off, (int)F, m, d_keep);
        PCR_LAUNCH_CHECK(c);
    }
    return frames_compact(in, d_keep, out);
}

}  // namespace
}  // namespace pcr

extern "C" {

// offsets, sizes and the output handle of an upload; n receives the point count
static int frames_upload_check(Ctx *c, const uint64_t *frame_offsets, size_t n_frames, pcr_frames **out, size_t *n) {
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    if (n_frames == 0) return fail(c, PCR_ERR_INVALID_ARG, "a batch holds at least one frame");
    PCR_TRY(offsets_check(c, "frame_offsets", frame_offsets, n_frames));
    *n = (size_t)frame_offsets[n_frames];
    return batch_size_check(c, *n, n_frames);
}

int pcr_frames_upload(pcr_ctx *ctx, const float *x, const float *y, const float *z, const uint64_t *frame_offsets, size_t n_frames,
                      pcr_frames **out) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    size_t n = 0;
    PCR_TRY(frames_upload_check(c, frame_offsets, n_frames, out, &n));
    if (n && (!x || !y || !z)) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    FramesPtr res;
    PCR_TRY(frames_alloc(ctx, n, false, std::vector<uint64_t>(frame_offsets, frame_offsets + n_frames + 1), res));
    PCR_TRY(points_upload(res.get(), x, y, z));
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_frames_upload_rows(pcr_ctx *ctx, const float *xyz, const uint64_t *frame_offsets, size_t n_frames, pcr_frames **out) {
    if (!ctx) return fail(nullptr, PCR_ERR_INVALID_ARG, "ctx is NULL");
    Ctx *c = &ctx->c;
    size_t n = 0;
    PCR_TRY(frames_upload_check(c, frame_offsets, n_frames, out, &n));
    if (n && !xyz) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    FramesPtr res;
    PCR_TRY(frames_alloc(ctx, n, false, std::vector<uint64_t>(frame_offsets, frame_offsets + n_frames + 1), res));
    PCR_TRY(points_upload_rows(res.get(), xyz));
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

void pcr_frames_free(pcr_frames *frames) { handle_free(frames); }

size_t pcr_frames_len(const pcr_frames *frames) { return frames ? frames->n : 0; }
size_t pcr_frames_count(const pcr_frames *frames) { return frames ? frames->count() : 0; }
int pcr_frames_has_normals(const pcr_frames *frames) { return frames && frames->has_normals ? 1 : 0; }

int pcr_frames_offsets(const pcr_frames *frames, uint64_t *out) {
    PCR_TRY(handle_check(frames, "frames"));
    if (!out) return fail(&frames->owner->c, PCR_ERR_INVALID_ARG, "null pointer");
    std::copy(frames->off.begin(), frames->off.end(), out);
    return PCR_OK;
}

int pcr_frames_device_pointers(const pcr_frames *frames, const float **d_x, const float **d_y, const float **d_z, const float **d_nx,
                               const float **d_ny, const float **d_nz) {
    PCR_TRY(handle_check(frames, "frames"));
    points_device_pointers(frames, d_x, d_y, d_z, d_nx, d_ny, d_nz);
    return PCR_OK;
}

int pcr_frames_download(const pcr_frames *frames, float *x, float *y, float *z, float *nx, float *ny, float *nz) {
    PCR_TRY(handle_check(frames, "frames"));
    Ctx *c = &frames->owner->c;
    const bool want_n = nx || ny || nz;
    if (want_n && !frames->has_normals) return fail(c, PCR_ERR_INVALID_ARG, "the frames have no normals");
    const size_t n = frames->n;
    if (n && (!x || !y || !z || (want_n && (!nx || !ny || !nz)))) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (!n) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    return points_download(frames, x, y, z, nx, ny, nz);
    PCR_API_END(c)
}

int pcr_frames_download_rows(const pcr_frames *frames, float *xyz, float *normals) {
    PCR_TRY(handle_check(frames, "frames"));
    Ctx *c = &frames->owner->c;
    if (normals && !frames->has_normals) return fail(c, PCR_ERR_INVALID_ARG, "the frames have no normals");
    if (frames->n && !xyz && !normals) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (!frames->n) return PCR_OK;
    PCR_API_BEGIN
    DevSetter ds(c);
    return points_download_rows(frames, xyz, normals);
    PCR_API_END(c)
}

int pcr_frames_frame(const pcr_frames *frames, size_t f, pcr_cloud **out) {
    PCR_TRY(handle_check(frames, "frames"));
    Ctx *c = &frames->owner->c;
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    if (f >= frames->count()) return fail(c, PCR_ERR_INVALID_ARG, "frame %zu out of range (%zu frames)", f, frames->count());
    PCR_API_BEGIN
    DevSetter ds(c);
    CloudPtr res;
    PCR_TRY(points_alloc(frames->owner, (size_t)(frames->off[f + 1] - frames->off[f]), frames->has_normals, res));
    PCR_TRY(copy_arrays(frames, (size_t)frames->off[f], frames->arrays(), res.get()));
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_frames_merge(const pcr_frames *frames, pcr_cloud **out) {
    if (out) *out = nullptr;
    PCR_TRY(handle_check(frames, "frames"));
    Ctx *c = &frames->owner->c;
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    CloudPtr res;  // pcr_frames_frame over all frames: the arrays hold the frames back to back already
    PCR_TRY(points_alloc(frames->owner, frames->n, frames->has_normals, res));
    PCR_TRY(copy_arrays(frames, 0, frames->arrays(), res.get()));
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_frames_apply_transform(const pcr_frames *frames, const float *transforms, pcr_frames **out) {
    if (out) *out = nullptr;
    PCR_TRY(handle_check(frames, "frames"));
    Ctx *c = &frames->owner->c;
    if (!out || !transforms) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    PCR_API_BEGIN
    DevSetter ds(c);
    FramesPtr res;  // icp.rs:91: xyz only; the offsets are the input's
    PCR_TRY(frames_alloc(frames->owner, frames->n, false, frames->off, res, frames->d_off));
    PCR_TRY(apply_transform_batch_dev(c, frames->x(), frames->y(), frames->z(), frames->off.data(), frames->count(), frames->d_off, transforms,
                                      res->x(), res->y(), res->z()));
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_frames_select(const pcr_frames *frames, const uint32_t *indices, const uint64_t *index_offsets, int invert, pcr_frames **out) {
    PCR_TRY(handle_check(frames, "frames"));
    Ctx *c = &frames->owner->c;
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    const size_t F = frames->count();
    PCR_TRY(offsets_check(c, "index_offsets", index_offsets, F));
    const size_t m = (size_t)index_offsets[F];
    if (m && !indices) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    if (m > 0x7fffffffull) return fail(c, PCR_ERR_UNSUPPORTED, "at most 2^31 - 1 listed indices per call");
    for (size_t f = 0; f < F; f++) {  // cloud.rs:109: select panics on an out-of-bounds index
        const uint64_t n_f = frames->off[f + 1] - frames->off[f];
        for (uint64_t t = index_offsets[f]; t < index_offsets[f + 1]; t++)
            if (indices[t] >= n_f)
                return fail(c, PCR_ERR_INVALID_ARG, "frame %zu: index %u out of bounds for a frame with %llu points", f, indices[t],
                            (unsigned long long)n_f);
    }
    PCR_API_BEGIN
    DevSetter ds(c);
    std::vector<uint64_t> loff(index_offsets, index_offsets + F + 1);
    StreamAlloc<uint32_t> d_idx(c->stream);
    PCR_CUDA(c, d_idx.alloc(sizeof(uint32_t) * std::max<size_t>(m, 1)));
    if (m) PCR_CUDA(c, cudaMemcpyAsync(d_idx.p, indices, sizeof(uint32_t) * m, cudaMemcpyHostToDevice, c->stream));
    FramesPtr res;
    if (invert) {
        PCR_TRY(frames_select_inverse_dev(frames, d_idx.p, loff, res));
        *out = res.release();
        return PCR_OK;
    }
    PCR_TRY(frames_alloc(frames->owner, m, frames->has_normals, loff, res));
    if (m) {
        // the gather reads the list offsets as u32: the new batch's own device offsets are exactly those
        frames_gather_kernel<<<(unsigned)((m + 255) / 256), 256, 0, c->stream>>>(frames->base, frames->stride, frames->arrays(), d_idx.p,
                                                                                 res->d_off, frames->d_off, (int)F, m, res->base, res->stride);
        PCR_LAUNCH_CHECK(c);
    }
    // the caller's index array is free again on return (a pinned one is read by the copy while it runs)
    PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_frames_voxel_downsample(const pcr_frames *frames, float voxel_size, pcr_frames **out) {
    PCR_TRY(handle_check(frames, "frames"));
    Ctx *c = &frames->owner->c;
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    if (!std::isfinite(voxel_size) || !(voxel_size > 0.f)) return fail(c, PCR_ERR_INVALID_ARG, "voxel_size must be > 0 and finite");
    PCR_API_BEGIN
    DevSetter ds(c);
    const size_t F = frames->count();
    FramesPtr res;  // voxel_downsample.rs:64: xyz only; sized for the input, then shrunk to the voxels
    PCR_TRY(frames_alloc(frames->owner, frames->n, false, std::vector<uint64_t>(F + 1, 0), res));
    std::vector<uint64_t> out_off(F + 1, 0);
    PCR_TRY(voxel_batch_entry(frames->owner, true, frames->x(), frames->y(), frames->z(), frames->off.data(), F, voxel_size, res->x(), res->y(),
                              res->z(), out_off.data()));
    PCR_TRY(offsets_upload(c, out_off, res->d_off));
    res->n = (size_t)out_off[F];  // (the allocation keeps its original stride)
    res->off = std::move(out_off);
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_frames_statistical_outlier_removal(const pcr_frames *frames, size_t k, float std_mul, pcr_frames **out) {
    PCR_TRY(handle_check(frames, "frames"));
    Ctx *c = &frames->owner->c;
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    if (!std::isfinite(std_mul) || std_mul < 0.f) return fail(c, PCR_ERR_INVALID_ARG, "std_mul must be >= 0 and finite");
    if (k + 1 > PCR_MAX_K) return fail(c, PCR_ERR_UNSUPPORTED, "k = %zu exceeds PCR_MAX_K - 1", k);
    PCR_API_BEGIN
    DevSetter ds(c);
    const size_t n = frames->n;
    FramesPtr res;
    if (n == 0 || k == 0) {  // statistical_outlier.rs:5-7: PointCloud::new()
        PCR_TRY(frames_empty(frames, false, res));
    } else {
        StreamAlloc<uint8_t> d_keep(c->stream);
        PCR_CUDA(c, d_keep.alloc(n));
        const float vp0[3] = {0.f, 0.f, 0.f};
        PCR_TRY(pcr_sor_normals_batch_dev(frames->owner, frames->x(), frames->y(), frames->z(), frames->off.data(), frames->count(), k, std_mul, 0,
                                          vp0, d_keep.p, nullptr, nullptr, nullptr));
        PCR_TRY(frames_compact(frames, d_keep.p, res));  // :68 select
    }
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_frames_radius_outlier_removal(const pcr_frames *frames, float radius, size_t min_neighbors, pcr_frames **out) {
    PCR_TRY(handle_check(frames, "frames"));
    Ctx *c = &frames->owner->c;
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    PCR_API_BEGIN
    DevSetter ds(c);
    const size_t n = frames->n;
    FramesPtr res;
    if (n == 0) {
        PCR_TRY(frames_empty(frames, frames->has_normals, res));
    } else {
        StreamAlloc<uint8_t> d_keep(c->stream);
        PCR_CUDA(c, d_keep.alloc(n));
        PCR_TRY(pcr_radius_outlier_batch_dev(frames->owner, frames->x(), frames->y(), frames->z(), frames->off.data(), frames->count(), radius,
                                             min_neighbors, d_keep.p));
        PCR_TRY(frames_compact(frames, d_keep.p, res));
    }
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_frames_estimate_normals(const pcr_frames *frames, size_t k, const float viewpoint[3], pcr_frames **out) {
    PCR_TRY(handle_check(frames, "frames"));
    Ctx *c = &frames->owner->c;
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    if (k == 0) return fail(c, PCR_ERR_INVALID_ARG, "k must be > 0");  // as pcr_cloud_estimate_normals
    PCR_API_BEGIN
    DevSetter ds(c);
    FramesPtr res;
    PCR_TRY(frames_alloc(frames->owner, frames->n, true, frames->off, res, frames->d_off));
    PCR_TRY(copy_arrays(frames, 0, 3, res.get()));
    const float vp0[3] = {0.f, 0.f, 0.f};  // estimate.rs:13-15
    PCR_TRY(pcr_estimate_normals_batch_dev(frames->owner, frames->x(), frames->y(), frames->z(), frames->off.data(), frames->count(), k,
                                           viewpoint ? viewpoint : vp0, res->nx(), res->ny(), res->nz()));
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_frames_sor_normals(const pcr_frames *frames, size_t k_sor, float std_mul, size_t k_normals, const float viewpoint[3],
                           pcr_frames **out) {
    PCR_TRY(handle_check(frames, "frames"));
    Ctx *c = &frames->owner->c;
    if (!out) return fail(c, PCR_ERR_INVALID_ARG, "null pointer");
    *out = nullptr;
    if (k_normals == 0) return fail(c, PCR_ERR_INVALID_ARG, "k_normals must be > 0");
    if (!std::isfinite(std_mul) || std_mul < 0.f) return fail(c, PCR_ERR_INVALID_ARG, "std_mul must be >= 0 and finite");
    if (k_sor + 1 > PCR_MAX_K || k_normals > PCR_MAX_K) return fail(c, PCR_ERR_UNSUPPORTED, "k exceeds PCR_MAX_K");
    PCR_API_BEGIN
    DevSetter ds(c);
    const size_t n = frames->n;
    FramesPtr res;
    if (n == 0 || k_sor == 0) {  // statistical_outlier.rs:5-7
        PCR_TRY(frames_empty(frames, true, res));
    } else {
        // normals by input index go to a scratch block; the kept points and their normals are compacted together
        const size_t stride = (n + 63) & ~(size_t)63;
        StreamAlloc<float> nrm_mem(c->stream);
        PCR_CUDA(c, nrm_mem.alloc(sizeof(float) * 3 * stride + n));
        float *d_nrm = nrm_mem.p;
        uint8_t *d_keep = (uint8_t *)(d_nrm + 3 * stride);
        const float vp0[3] = {0.f, 0.f, 0.f};
        PCR_TRY(pcr_sor_normals_batch_dev(frames->owner, frames->x(), frames->y(), frames->z(), frames->off.data(), frames->count(), k_sor, std_mul,
                                          k_normals, viewpoint ? viewpoint : vp0, d_keep, d_nrm, d_nrm + stride, d_nrm + 2 * stride));
        PCR_TRY(frames_compact(frames, d_keep, res, d_nrm, stride));
    }
    *out = res.release();
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_frames_ransac_plane_samples(const pcr_frames *frames, float distance_threshold, const uint32_t *samples, const uint64_t *sample_offsets,
                                    float *models, uint32_t *inliers, uint64_t *inlier_offsets, pcr_frames **outliers) {
    PCR_TRY(handle_check(frames, "frames"));
    Ctx *c = &frames->owner->c;
    if (outliers) *outliers = nullptr;
    PCR_API_BEGIN
    DevSetter ds(c);
    const size_t n = frames->n, F = frames->count();
    StreamAlloc<uint32_t> d_inl(c->stream);
    PCR_CUDA(c, d_inl.alloc(sizeof(uint32_t) * std::max<size_t>(n, 1)));
    PCR_TRY(ransac_batch_entry(frames->owner, true, frames->x(), frames->y(), frames->z(), frames->off.data(), F, distance_threshold, samples,
                               sample_offsets, models, d_inl.p, inlier_offsets));
    const size_t k = (size_t)inlier_offsets[F];
    if (inliers && k) {
        PCR_CUDA(c, cudaMemcpyAsync(inliers, d_inl.p, sizeof(uint32_t) * k, cudaMemcpyDeviceToHost, c->stream));
        PCR_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    if (outliers) {  // ransac_plane.rs's inliers are in bounds by construction: straight to the device select_inverse
        FramesPtr res;
        PCR_TRY(frames_select_inverse_dev(frames, d_inl.p, std::vector<uint64_t>(inlier_offsets, inlier_offsets + F + 1), res));
        *outliers = res.release();
    }
    return PCR_OK;
    PCR_API_END(c)
}

int pcr_frames_euclidean_cluster(const pcr_frames *frames, float distance_threshold, size_t min_size, size_t max_size, uint32_t *offsets,
                                 uint32_t *indices, uint64_t *cluster_offsets) {
    PCR_TRY(handle_check(frames, "frames"));
    return cluster_batch_entry(frames->owner, true, false, frames->x(), frames->y(), frames->z(), frames->off.data(), frames->count(),
                               distance_threshold, min_size, max_size, offsets, indices, cluster_offsets);
}

int pcr_frames_icp_point_to_point(const pcr_frames *frames, const uint32_t *pairs, size_t n_pairs, const pcr_icp_params *params,
                                  pcr_icp_result *results) {
    PCR_TRY(handle_check(frames, "frames"));
    return icp_batch_entry(frames->owner, true, false, frames->x(), frames->y(), frames->z(), frames->off.data(), frames->count(), nullptr, nullptr,
                           nullptr, 0, pairs, n_pairs, params, results);
}

int pcr_frames_icp_point_to_plane(const pcr_frames *frames, const uint32_t *pairs, size_t n_pairs, const pcr_icp_params *params,
                                  pcr_icp_result *results) {
    PCR_TRY(handle_check(frames, "frames"));
    if (!frames->has_normals)  // crates/python/src/registration.rs:80-86
        return fail(&frames->owner->c, PCR_ERR_INVALID_ARG, "point-to-plane ICP needs frames with normals (call estimate_normals first)");
    return icp_batch_entry(frames->owner, true, true, frames->x(), frames->y(), frames->z(), frames->off.data(), frames->count(), frames->nx(),
                           frames->ny(), frames->nz(), frames->n, pairs, n_pairs, params, results);
}

}  // extern "C"
