// mbc_api.cu -- context, table and result management of libmbcol.so (C ABI in include/mbcol.h).
//
// Device HBM replaces the reference's buffer pool (bufmgr/BufMgr.java) for this path: whole
// columns stay resident as contiguous arrays, one per Columnarfile column
// (columnar/Columnarfile.java:329-337 opens one heapfile per column instead).
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <algorithm>

#include "mbc_internal.cuh"

namespace mbc {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int32_t dev_alloc(mbc_ctx* ctx, void** p, size_t bytes, bool zero) {
    *p = nullptr;
    if (bytes == 0) bytes = 16;
    MBC_CUDA(cudaMallocAsync(p, bytes, ctx->stream));
    if (zero) MBC_CUDA(cudaMemsetAsync(*p, 0, bytes, ctx->stream));
    return MBC_OK;
}

}  // namespace mbc
static void ctx_destroy(mbc_ctx* ctx) {
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto& b : ctx->pinned_free) cudaFreeHost(b.p);
    for (auto e : ctx->event_free) cudaEventDestroy(e);
    if (ctx->ws) cudaFree(ctx->ws);
    if (ctx->fused_flags) cudaFree(ctx->fused_flags);
    if (ctx->ev_begin) cudaEventDestroy(ctx->ev_begin);
    if (ctx->ev_end) cudaEventDestroy(ctx->ev_end);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->d2h_stream) cudaStreamDestroy(ctx->d2h_stream);
    delete ctx;
}

namespace mbc {

void ctx_retain(mbc_ctx* ctx) { ++ctx->live_objects; }

void ctx_release(mbc_ctx* ctx) {
    if (--ctx->live_objects <= 0 && ctx->shutdown_pending) ctx_destroy(ctx);
}

void dev_free(mbc_ctx* ctx, void* p) {
    if (p) cudaFreeAsync(p, ctx->stream);
}

int32_t pinned_alloc(mbc_ctx* ctx, void** p, size_t bytes, size_t* actual) {
    if (bytes == 0) bytes = 16;
    *actual = bytes;
    // best fit from the recycled blocks (pinning gigabytes costs more than the copy it serves)
    int best = -1;
    for (int i = 0; i < (int)ctx->pinned_free.size(); ++i) {
        if (ctx->pinned_free[i].bytes >= bytes &&
            (best < 0 || ctx->pinned_free[i].bytes < ctx->pinned_free[best].bytes))
            best = i;
    }
    if (best >= 0 && ctx->pinned_free[best].bytes <= 2 * bytes + (1u << 20)) {
        *p = ctx->pinned_free[best].p;
        *actual = ctx->pinned_free[best].bytes;
        ctx->pinned_free.erase(ctx->pinned_free.begin() + best);
        return MBC_OK;
    }
    MBC_CUDA(cudaHostAlloc(p, bytes, cudaHostAllocDefault));
    return MBC_OK;
}

void pinned_release(mbc_ctx* ctx, void* p, size_t bytes) {
    if (!p) return;
    if (ctx->pinned_free.size() >= 64) {
        cudaFreeHost(p);
        return;
    }
    ctx->pinned_free.push_back({p, bytes});
}

int32_t ensure_workspace(mbc_ctx* ctx, size_t bytes) {
    if (ctx->ws_bytes >= bytes) return MBC_OK;
    if (ctx->ws) {
        MBC_CUDA(cudaStreamSynchronize(ctx->stream));
        MBC_CUDA(cudaFree(ctx->ws));
        ctx->ws = nullptr;
        ctx->ws_bytes = 0;
    }
    size_t want = std::max(bytes, (size_t)1 << 20);
    MBC_CUDA(cudaMalloc(&ctx->ws, want));
    ctx->ws_bytes = want;
    return MBC_OK;
}

void begin_timing(mbc_ctx* ctx) {
    if (!ctx->timing_split) ctx->extra_ms = 0.f;
    ctx->timing_split = false;
    cudaEventRecord(ctx->ev_begin, ctx->stream);
}
void end_timing(mbc_ctx* ctx) { cudaEventRecord(ctx->ev_end, ctx->stream); }
cudaEvent_t event_get(mbc_ctx* ctx) {
    if (!ctx->event_free.empty()) {
        cudaEvent_t e = ctx->event_free.back();
        ctx->event_free.pop_back();
        return e;
    }
    cudaEvent_t e = nullptr;
    return cudaEventCreate(&e) == cudaSuccess ? e : nullptr;
}
void event_put(mbc_ctx* ctx, cudaEvent_t e) {
    if (!e) return;
    if (ctx->event_free.size() >= 64) cudaEventDestroy(e);
    else ctx->event_free.push_back(e);
}

void result_phase_times(mbc_result* r) {
    if (!r->ev_t0 || !r->ev_t1 || !r->ev_mid[0] || !r->ev_mid[1] || !r->ev_mid[2]) return;
    cudaEvent_t e[5] = {r->ev_t0, r->ev_mid[0], r->ev_mid[1], r->ev_mid[2], r->ev_t1};
    for (int i = 0; i < 4; ++i)
        if (cudaEventElapsedTime(&r->phase_ms[i], e[i], e[i + 1]) != cudaSuccess) r->phase_ms[i] = -1.f;
}

int32_t result_finalize(mbc_result* r) {
    if (!r->ev_ready) return MBC_OK;
    mbc_ctx* ctx = r->ctx;
    cudaError_t e = cudaEventSynchronize(r->ev_ready);
    event_put(ctx, r->ev_ready);
    r->ev_ready = nullptr;
    if (e != cudaSuccess) MBC_FAIL(MBC_ERR_CUDA, "deferred scan failed: %s", cudaGetErrorString(e));
    r->count = (int64_t)r->h_small[kMaxAgg];
    for (size_t a = 0; a < r->aggs.size(); ++a) {
        mbc_result::Agg& g = r->aggs[a];
        agg_from_raw(g.kind, g.type, r->h_small[a], r->count > 0, &g.i, &g.f, &g.valid);
    }
    if (r->ev_t0 && r->ev_t1 && cudaEventElapsedTime(&r->kernel_ms, r->ev_t0, r->ev_t1) != cudaSuccess) r->kernel_ms = -1.f;
    result_phase_times(r);
    return MBC_OK;
}

void agg_from_raw(int32_t kind, int32_t type, unsigned long long raw, bool nonempty, int64_t* i, double* f, int32_t* valid) {
    if (kind == MBC_AGG_COUNT || type == MBC_ATTR_INTEGER) {
        *i = (int64_t)raw;
        *f = (double)*i;
    } else {
        double d;
        memcpy(&d, &raw, 8);
        *f = d;
        *i = real_agg_as_i64(d);
    }
    *valid = (kind == MBC_AGG_COUNT || kind == MBC_AGG_SUM) ? 1 : nonempty;
    if (!*valid) { *i = 0; *f = 0.0; }
}

void split_timing(mbc_ctx* ctx) {
    cudaEventRecord(ctx->ev_end, ctx->stream);
    float ms = 0.f;
    if (cudaEventSynchronize(ctx->ev_end) == cudaSuccess && cudaEventElapsedTime(&ms, ctx->ev_begin, ctx->ev_end) == cudaSuccess)
        ctx->extra_ms += ms;
    ctx->timing_split = true;
}

}  // namespace mbc

using namespace mbc;

extern "C" {

const char* mbc_last_error(void) { return g_err; }
int32_t mbc_abi_version(void) { return MBC_ABI_VERSION; }

int32_t mbc_init(int32_t device_id, mbc_ctx** out) {
    if (!out) MBC_FAIL(MBC_ERR_ARG, "mbc_init: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        MBC_FAIL(MBC_ERR_NODEVICE, "mbc_init: no CUDA device (%s); this library has no CPU fallback",
                 e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device_id < 0 || device_id >= ndev) MBC_FAIL(MBC_ERR_ARG, "mbc_init: device %d of %d", device_id, ndev);
    cudaDeviceProp prop;
    MBC_CUDA(cudaGetDeviceProperties(&prop, device_id));
    if (prop.major != 10)
        MBC_FAIL(MBC_ERR_NODEVICE, "mbc_init: device %d is sm_%d%d; libmbcol.so carries sm_100a code only",
                 device_id, prop.major, prop.minor);
    MBC_CUDA(cudaSetDevice(device_id));
    if (const char* g = getenv("MBC_L2_FETCH")) {                   // experiment knob: L2 fetch granularity on a miss (32 / 64 / 128)
        cudaError_t le = cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)atoi(g));
        size_t got = 0;
        cudaDeviceGetLimit(&got, cudaLimitMaxL2FetchGranularity);
        fprintf(stderr, "[mbc] L2 fetch granularity: asked %s, set -> %s, now %zu\n", g, cudaGetErrorString(le), got);
        cudaGetLastError();
    }
    mbc_ctx* ctx = new mbc_ctx();
    ctx->device = device_id;
    ctx->sm_count = prop.multiProcessorCount;
    cudaMemPool_t pool;
    uint64_t thr = UINT64_MAX;
    // keep freed device memory in the stream-ordered pool: result buffers are re-used across scans without going back to
    // the driver
    cudaError_t e2 = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking);
    if (e2 == cudaSuccess) e2 = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    if (e2 == cudaSuccess) e2 = cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking);
    ctx->stream = ctx->own_stream;
    if (e2 == cudaSuccess) e2 = cudaEventCreate(&ctx->ev_begin);
    if (e2 == cudaSuccess) e2 = cudaEventCreate(&ctx->ev_end);
    if (e2 == cudaSuccess) e2 = cudaDeviceGetDefaultMemPool(&pool, device_id);
    if (e2 == cudaSuccess) e2 = cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    if (e2 != cudaSuccess) {                   // nothing half-built is left behind
        set_error("mbc_init: %s", cudaGetErrorString(e2));
        ctx->stream = ctx->own_stream ? ctx->own_stream : nullptr;
        if (ctx->stream) ctx_destroy(ctx); else delete ctx;
        return MBC_ERR_CUDA;
    }
    *out = ctx;
    return MBC_OK;
}

void mbc_shutdown(mbc_ctx* ctx) {
    if (!ctx) return;
    if (ctx->live_objects > 0) {               // tables / results are still open: the last one to close destroys the context
        ctx->shutdown_pending = true;
        return;
    }
    ctx_destroy(ctx);
}

int32_t mbc_set_stream(mbc_ctx* ctx, void* cuda_stream) {
    if (!ctx) MBC_FAIL(MBC_ERR_ARG, "mbc_set_stream: ctx is NULL");
    MBC_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return MBC_OK;
}

int32_t mbc_sync(mbc_ctx* ctx) {
    if (!ctx) MBC_FAIL(MBC_ERR_ARG, "mbc_sync: ctx is NULL");
    MBC_CUDA(cudaStreamSynchronize(ctx->stream));
    return MBC_OK;
}

int64_t mbc_kernel_launches(const mbc_ctx* ctx) { return ctx ? ctx->launches : 0; }

int64_t mbc_h2d_bytes(const mbc_ctx* ctx) { return ctx ? ctx->h2d_bytes : 0; }

float mbc_last_kernel_ms(const mbc_ctx* ctx) {
    if (!ctx) return 0.f;
    float ms = 0.f;
    if (cudaEventSynchronize(ctx->ev_end) != cudaSuccess) return 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev_begin, ctx->ev_end) != cudaSuccess) return 0.f;
    return ms + ctx->extra_ms;
}

int32_t mbc_host_alloc(void** p, int64_t bytes) {
    if (!p || bytes < 0) MBC_FAIL(MBC_ERR_ARG, "mbc_host_alloc: bad argument");
    MBC_CUDA(cudaHostAlloc(p, (size_t)std::max<int64_t>(bytes, 16), cudaHostAllocDefault));
    return MBC_OK;
}

void mbc_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

// ---- tables ------------------------------------------------------------------------------

int32_t mbc_table_create(mbc_ctx* ctx, int32_t ncols, const mbc_coldesc* cols, int64_t nrows,
                         int64_t position_base, mbc_table** out) {
    if (!ctx || !cols || !out || ncols <= 0 || nrows < 0)
        MBC_FAIL(MBC_ERR_ARG, "mbc_table_create: bad argument");
    *out = nullptr;
    MBC_CUDA(cudaSetDevice(ctx->device));
    mbc_table* t = new mbc_table();
    t->ctx = ctx;
    ctx_retain(ctx);
    t->nrows = nrows;
    t->nrows_pad = std::max<int64_t>(round_up(nrows, kPadRows), kPadRows);
    t->words_pad = t->nrows_pad / 32;
    t->pos_base = position_base;
    t->cols.resize(ncols);
    t->bm.resize(ncols);
    for (int c = 0; c < ncols; ++c) {
        Column& col = t->cols[c];
        col.type = cols[c].type;
        col.width = cols[c].width;
        if (col.type == MBC_ATTR_INTEGER || col.type == MBC_ATTR_REAL) {
            if (col.width != 4) {
                mbc_table_free(t);
                MBC_FAIL(MBC_ERR_ARG, "mbc_table_create: column %d: int/real width must be 4", c);
            }
            col.stride = 4;
        } else if (col.type == MBC_ATTR_STRING) {
            if (col.width <= 0 || col.width > kMaxStrStride) {
                mbc_table_free(t);
                MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_table_create: column %d: char(%d) outside 1..%d", c,
                         col.width, kMaxStrStride);
            }
            col.stride = str_stride(col.width);
        } else {
            mbc_table_free(t);
            MBC_FAIL(MBC_ERR_ARG, "mbc_table_create: column %d: unknown AttrType %d", c, col.type);
        }
        int32_t s = dev_alloc(ctx, &col.d, (size_t)t->nrows_pad * col.stride, true);
        if (s != MBC_OK) {
            mbc_table_free(t);
            return s;
        }
    }
    *out = t;
    return MBC_OK;
}

void mbc_table_free(mbc_table* t) {
    if (!t) return;
    cudaSetDevice(t->ctx->device);
    for (auto& c : t->cols) dev_free(t->ctx, c.d);
    for (auto& b : t->bm) {
        dev_free(t->ctx, b.d_words);
        dev_free(t->ctx, b.d_ids);
        dev_free(t->ctx, b.d_rows);
        dev_free(t->ctx, b.d_indexed);
    }
    dev_free(t->ctx, t->d_deleted);
    mbc_ctx* ctx = t->ctx;
    delete t;
    ctx_release(ctx);
}

int64_t mbc_table_nrows(const mbc_table* t) { return t ? t->nrows : -1; }
int32_t mbc_table_ncols(const mbc_table* t) { return t ? (int32_t)t->cols.size() : -1; }

int32_t mbc_table_coldesc(const mbc_table* t, int32_t col, mbc_coldesc* out) {
    if (!t || !out || col < 0 || col >= (int)t->cols.size()) MBC_FAIL(MBC_ERR_ARG, "mbc_table_coldesc: bad argument");
    out->type = t->cols[col].type;
    out->width = t->cols[col].width;
    return MBC_OK;
}

int32_t mbc_table_load_column(mbc_table* t, int32_t col, const void* host_packed, int64_t nrows) {
    if (!t || col < 0 || col >= (int)t->cols.size() || nrows != t->nrows || (!host_packed && nrows > 0))
        MBC_FAIL(MBC_ERR_ARG, "mbc_table_load_column: bad argument (col %d, nrows %lld vs table %lld)", col,
                 (long long)nrows, t ? (long long)t->nrows : -1LL);
    if (nrows == 0) return MBC_OK;
    MBC_CUDA(cudaSetDevice(t->ctx->device));
    Column& c = t->cols[col];
    if (c.stride == c.width) {
        MBC_CUDA(cudaMemcpyAsync(c.d, host_packed, (size_t)nrows * c.width, cudaMemcpyHostToDevice, t->ctx->stream));
    } else {
        // host rows are packed at `width`, device rows sit at `stride` with zero padding
        MBC_CUDA(cudaMemcpy2DAsync(c.d, c.stride, host_packed, c.width, c.width, (size_t)nrows,
                                   cudaMemcpyHostToDevice, t->ctx->stream));
    }
    MBC_CUDA(cudaStreamSynchronize(t->ctx->stream));
    return MBC_OK;
}

int32_t mbc_table_read_column(mbc_table* t, int32_t col, void* host_out, int64_t nrows) {
    if (!t || col < 0 || col >= (int)t->cols.size() || nrows != t->nrows || (!host_out && nrows > 0))
        MBC_FAIL(MBC_ERR_ARG, "mbc_table_read_column: bad argument");
    if (nrows == 0) return MBC_OK;
    MBC_CUDA(cudaSetDevice(t->ctx->device));
    Column& c = t->cols[col];
    if (c.stride == c.width) {
        MBC_CUDA(cudaMemcpyAsync(host_out, c.d, (size_t)nrows * c.width, cudaMemcpyDeviceToHost, t->ctx->stream));
    } else {
        MBC_CUDA(cudaMemcpy2DAsync(host_out, c.width, c.d, c.stride, c.width, (size_t)nrows,
                                   cudaMemcpyDeviceToHost, t->ctx->stream));
    }
    MBC_CUDA(cudaStreamSynchronize(t->ctx->stream));
    return MBC_OK;
}

int32_t mbc_table_column_device(mbc_table* t, int32_t col, void** dev_ptr, int32_t* stride_bytes) {
    if (!t || col < 0 || col >= (int)t->cols.size()) MBC_FAIL(MBC_ERR_ARG, "mbc_table_column_device: bad argument");
    if (dev_ptr) *dev_ptr = t->cols[col].d;
    if (stride_bytes) *stride_bytes = t->cols[col].stride;
    return MBC_OK;
}

int32_t mbc_table_set_deleted(mbc_table* t, const uint64_t* bitset_words, int64_t nwords) {
    if (!t || nwords < 0 || (nwords > 0 && !bitset_words)) MBC_FAIL(MBC_ERR_ARG, "mbc_table_set_deleted: bad argument");
    MBC_CUDA(cudaSetDevice(t->ctx->device));
    if (!t->d_deleted) MBC_TRY(dev_alloc(t->ctx, (void**)&t->d_deleted, (size_t)t->words_pad * 4, true));
    else MBC_CUDA(cudaMemsetAsync(t->d_deleted, 0, (size_t)t->words_pad * 4, t->ctx->stream));
    // a little-endian uint64 word is two consecutive uint32 words with the same bit numbering;
    // bits at or beyond nrows are irrelevant (the scan masks rows >= nrows)
    int64_t max_words64 = t->words_pad / 2;
    int64_t n = std::min(nwords, max_words64);
    bool any = false;
    for (int64_t i = 0; i < n && !any; ++i) any = bitset_words[i] != 0;
    if (n > 0)
        MBC_CUDA(cudaMemcpyAsync(t->d_deleted, bitset_words, (size_t)n * 8, cudaMemcpyHostToDevice, t->ctx->stream));
    MBC_CUDA(cudaStreamSynchronize(t->ctx->stream));
    t->has_deleted = any;
    return MBC_OK;
}

// ---- results -----------------------------------------------------------------------------

int64_t mbc_result_count(const mbc_result* r) {
    if (!r) return -1;
    if (result_finalize(const_cast<mbc_result*>(r)) != MBC_OK) return -1;
    return r->count;
}

int32_t mbc_result_phase_ms(const mbc_result* r, float* ms4) {
    if (!r || !ms4) MBC_FAIL(MBC_ERR_ARG, "mbc_result_phase_ms: bad argument");
    MBC_TRY(result_finalize(const_cast<mbc_result*>(r)));
    for (int i = 0; i < 4; ++i) ms4[i] = r->phase_ms[i];
    return MBC_OK;
}

float mbc_result_kernel_ms(const mbc_result* r) {
    if (!r) return -1.f;
    if (result_finalize(const_cast<mbc_result*>(r)) != MBC_OK) return -1.f;
    return r->kernel_ms;
}
const int64_t* mbc_result_positions(const mbc_result* r) { return r ? r->h_pos : nullptr; }
const int64_t* mbc_result_positions2(const mbc_result* r) { return r ? r->h_pos2 : nullptr; }

const void* mbc_result_column(const mbc_result* r, int32_t i, int32_t* width) {
    if (!r || i < 0 || i >= (int)r->cols.size()) return nullptr;
    if (width) *width = r->cols[i].width;
    return r->cols[i].h;
}

const uint8_t* mbc_result_tuples(const mbc_result* r, int32_t* tuple_len) {
    if (!r) return nullptr;
    if (tuple_len) *tuple_len = r->tuple_len;
    return r->h_tuples;
}

int32_t mbc_result_agg(const mbc_result* r, int32_t i, int64_t* as_i64, double* as_f64, int32_t* valid) {
    if (r && r->grouped) MBC_FAIL(MBC_ERR_ARG, "mbc_result_agg: a grouped result has one value per group (mbc_result_group_agg)");
    if (!r || i < 0 || i >= (int)r->aggs.size()) MBC_FAIL(MBC_ERR_ARG, "mbc_result_agg: index %d of %d", i,
                                                          r ? (int)r->aggs.size() : 0);
    MBC_TRY(result_finalize(const_cast<mbc_result*>(r)));
    if (as_i64) *as_i64 = r->aggs[i].i;
    if (as_f64) *as_f64 = r->aggs[i].f;
    if (valid) *valid = r->aggs[i].valid;
    return MBC_OK;
}

int32_t mbc_result_group_agg(const mbc_result* r, int32_t i, const int64_t** as_i64, const double** as_f64) {
    if (!r || !r->grouped) MBC_FAIL(MBC_ERR_ARG, "mbc_result_group_agg: not a result of mbc_group_aggregate");
    if (i < 0 || i >= (int)r->group_aggs.size())
        MBC_FAIL(MBC_ERR_ARG, "mbc_result_group_agg: index %d of %d aggregates on the host (MBC_WANT_AGG | MBC_WANT_HOST)", i,
                 (int)r->group_aggs.size());
    if (as_i64) *as_i64 = r->group_aggs[i].i.data();
    if (as_f64) *as_f64 = r->group_aggs[i].f.data();
    return MBC_OK;
}

const uint64_t* mbc_result_bitmap(const mbc_result* r, int64_t* nwords) {
    if (!r) return nullptr;
    if (nwords) *nwords = (r->nrows + 63) / 64;
    return r->h_bitmap;
}

int32_t mbc_result_device(const mbc_result* r, void** d_positions, void** d_positions2, void** d_bitmap,
                          void** d_aggs) {
    if (!r) MBC_FAIL(MBC_ERR_ARG, "mbc_result_device: r is NULL");
    if (d_positions) *d_positions = r->d_pos;
    if (d_positions2) *d_positions2 = r->d_pos2;
    if (d_bitmap) *d_bitmap = r->d_bitmap;
    if (d_aggs) *d_aggs = r->d_aggs;
    return MBC_OK;
}

int32_t mbc_result_column_device(const mbc_result* r, int32_t i, void** d_ptr, int32_t* stride_bytes) {
    if (!r || i < 0 || i >= (int)r->cols.size()) MBC_FAIL(MBC_ERR_ARG, "mbc_result_column_device: bad argument");
    if (d_ptr) *d_ptr = r->cols[i].d;
    if (stride_bytes) *stride_bytes = r->cols[i].stride;
    return MBC_OK;
}

void mbc_result_free(mbc_result* r) {
    if (!r) return;
    mbc_ctx* ctx = r->ctx;
    cudaSetDevice(ctx->device);
    result_finalize(r);                            // the pinned count/aggregate block must have landed before it is recycled
    event_put(ctx, r->ev_t0);
    event_put(ctx, r->ev_t1);
    event_put(ctx, r->ev_done);
    for (auto& e : r->ev_mid) event_put(ctx, e);
    dev_free(ctx, r->d_pos);
    dev_free(ctx, r->d_pos2);
    for (auto& c : r->cols) dev_free(ctx, c.d);
    dev_free(ctx, r->d_bitmap);
    dev_free(ctx, r->d_aggs);
    dev_free(ctx, r->d_tuples);
    for (auto& b : r->pinned) pinned_release(ctx, b.first, b.second);
    delete r;
    ctx_release(ctx);
}

}  // extern "C"
