// mbc_scan.cu -- host side of K2/K5 (kernels in mbc_scan_kernels.cuh): builds the term program,
// owns the result buffers, launches the fused scan, and implements the two public entry points
// mbc_scan (table resident in HBM) and mbc_scan_host (host-resident columns streamed through HBM).
#include <cstdio>
#include <cstring>
#include <algorithm>

#include "mbc_internal.cuh"
#include "mbc_scan_kernels.cuh"
#include "mbc_scan_fused.cuh"

namespace mbc {

static int32_t fill_operand(const mbc_table* t, const mbc_operand& o, int cmp_type, DevOperand* d, DevTerm* term,
                            int k) {
    memset(d, 0, sizeof(*d));
    d->col = -1;
    d->staged = -1;
    if (o.kind == MBC_OPERAND_LITERAL) {
        d->kind = 0;
        if (cmp_type == MBC_ATTR_STRING) {
            if (o.type != MBC_ATTR_STRING)
                MBC_FAIL(MBC_ERR_UNSUPPORTED, "term %d: string comparison against a non-string literal", k);
            if (o.lit_slen < 0 || o.lit_slen > kMaxLit || (o.lit_slen > 0 && !o.lit_s))
                MBC_FAIL(MBC_ERR_UNSUPPORTED, "term %d: string literal of %d bytes (max %d)", k, o.lit_slen, kMaxLit);
            for (int i = 0; i < o.lit_slen; ++i)
                if (o.lit_s[i] == 0) MBC_FAIL(MBC_ERR_UNSUPPORTED, "term %d: NUL byte in a string literal", k);
            memset(term->lit, 0, sizeof(term->lit));
            if (o.lit_slen) memcpy(term->lit, o.lit_s, o.lit_slen);
            term->lit_words = (o.lit_slen + 3) / 4;
        } else {
            // PredEval builds a one-field tuple of the literal's own type and the compare reads it
            // with the comparison type's getter (PredEval.java:60-78,101-116): the raw 4 bytes are
            // what is compared.
            if (o.type == MBC_ATTR_INTEGER) d->bits = (uint32_t)o.lit_i;
            else if (o.type == MBC_ATTR_REAL) memcpy(&d->bits, &o.lit_f, 4);
            else MBC_FAIL(MBC_ERR_UNSUPPORTED, "term %d: numeric comparison against a string literal", k);
        }
        return MBC_OK;
    }
    if (o.kind != MBC_OPERAND_OUTER) MBC_FAIL(MBC_ERR_ARG, "term %d: a single-table scan only has outer columns", k);
    if (o.col < 0 || o.col >= (int)t->cols.size()) MBC_FAIL(MBC_ERR_ARG, "term %d: column %d out of range", k, o.col);
    const Column& c = t->cols[o.col];
    if ((cmp_type == MBC_ATTR_STRING) != (c.type == MBC_ATTR_STRING))
        MBC_FAIL(MBC_ERR_UNSUPPORTED, "term %d: column %d of type %d compared as type %d", k, o.col, c.type, cmp_type);
    if (cmp_type == MBC_ATTR_STRING && c.stride > kMaxLit)
        MBC_FAIL(MBC_ERR_UNSUPPORTED, "term %d: char(%d) predicate column wider than %d", k, c.width, kMaxLit);
    d->kind = 1;
    d->col = o.col;
    d->ptr = c.d;
    d->stride = c.stride;
    return MBC_OK;
}

int32_t build_terms(const mbc_table* t, const mbc_term* terms, int32_t nterms, DevTerm* out) {
    if (nterms < 0 || nterms > kMaxTerms) MBC_FAIL(MBC_ERR_UNSUPPORTED, "%d predicate terms (max %d)", nterms, kMaxTerms);
    for (int k = 0; k < nterms; ++k) {
        const mbc_term& s = terms[k];
        DevTerm& d = out[k];
        memset(&d, 0, sizeof(d));
        if (k > 0 && s.conj_id < terms[k - 1].conj_id) MBC_FAIL(MBC_ERR_ARG, "terms must be sorted by conj_id");
        d.op = s.op;
        if (s.op < 0 || s.op > MBC_OP_RANGE) MBC_FAIL(MBC_ERR_ARG, "term %d: unknown operator %d", k, s.op);
        // comparison type = type of the lhs (PredEval.java:64,70,77,84,89)
        int cmp_type;
        if (s.lhs.kind == MBC_OPERAND_LITERAL) cmp_type = s.lhs.type;
        else {
            if (s.lhs.col < 0 || s.lhs.col >= (int)t->cols.size())
                MBC_FAIL(MBC_ERR_ARG, "term %d: column %d out of range", k, s.lhs.col);
            cmp_type = t->cols[s.lhs.col].type;
        }
        if (cmp_type != MBC_ATTR_INTEGER && cmp_type != MBC_ATTR_REAL && cmp_type != MBC_ATTR_STRING)
            MBC_FAIL(MBC_ERR_ARG, "term %d: comparison type %d", k, cmp_type);
        if (s.lhs.kind == MBC_OPERAND_LITERAL && s.rhs.kind == MBC_OPERAND_LITERAL && cmp_type == MBC_ATTR_STRING)
            MBC_FAIL(MBC_ERR_UNSUPPORTED, "term %d: literal-vs-literal string comparison (fold it on the host)", k);
        d.cmp_type = cmp_type;
        MBC_TRY(fill_operand(t, s.lhs, cmp_type, &d.lhs, &d, k));
        MBC_TRY(fill_operand(t, s.rhs, cmp_type, &d.rhs, &d, k));
        d.end_conj = (k == nterms - 1 || terms[k + 1].conj_id != s.conj_id) ? 1 : 0;
    }
    return MBC_OK;
}

// Choose which 4-byte predicate columns are staged through the TMA ring of the filter pass, the ring
// depth, the dynamic shared memory size and the persistent grid.
static int32_t plan_staging(mbc_ctx* ctx, ScanParams* p, size_t* smem_bytes, int* grid) {
    p->nstaged = 0;
    auto stage_of = [&](int col) -> int {
        for (int s = 0; s < p->nstaged; ++s) if (p->staged_cols[s] == col) return s;
        if (p->nstaged == kMaxStaged) return -1;
        p->staged_cols[p->nstaged] = col;
        return p->nstaged++;
    };
    for (int k = 0; k < p->nterms; ++k) {
        DevTerm& t = p->terms[k];
        if (t.cmp_type == MBC_ATTR_STRING) continue;
        if (t.lhs.kind == 1) t.lhs.staged = stage_of(t.lhs.col);
        if (t.rhs.kind == 1) t.rhs.staged = stage_of(t.rhs.col);
    }
    // ring depth: as deep as ~100 KB of shared memory allows (two CTAs per SM), at least 2
    p->nstages = p->nstaged == 0 ? 2 : std::max(2, std::min(kMaxStages, (int)(200 * 1024 / MBC_FILTER_CTAS / (p->nstaged * kStageColBytes))));
    *smem_bytes = (size_t)p->nstages * p->nstaged * kStageColBytes;
    if (!ctx->filter_smem_set) {                                  // a function attribute is per device: once per context
        MBC_CUDA(cudaFuncSetAttribute(filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        ctx->filter_smem_set = true;
    }
    int blocks_per_sm = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, filter_kernel, kScanThreads, *smem_bytes) != cudaSuccess || blocks_per_sm < 1)
        blocks_per_sm = 1;
    blocks_per_sm = std::min(blocks_per_sm, 8);
    *grid = std::max(1, ctx->sm_count * blocks_per_sm);
    return MBC_OK;
}

// tuple layout of a projected field list (iterator/TupleUtils.java:295-341 setup_op_tuple)
static int32_t tuple_layout(const std::vector<mbc_result::Col>& cols, TupleParams* tp) {
    int n = (int)cols.size();
    int off = (n + 2) * 2;
    tp->nfields = n;
    for (int i = 0; i < n; ++i) {
        tp->f[i].src = cols[i].d;
        tp->f[i].type = cols[i].type;
        tp->f[i].width = cols[i].width;
        tp->f[i].stride = cols[i].stride;
        tp->f[i].offset = off;
        off += cols[i].type == MBC_ATTR_STRING ? cols[i].width + 2 : 4;
    }
    if (off > 1024) MBC_FAIL(MBC_ERR_UNSUPPORTED, "projected tuple of %d bytes exceeds the reference's 1024-byte Tuple", off);
    tp->tuple_len = off;
    return MBC_OK;
}

int32_t encode_tuples(mbc_result* r) {
    mbc_ctx* ctx = r->ctx;
    TupleParams tp;
    memset(&tp, 0, sizeof(tp));
    MBC_TRY(tuple_layout(r->cols, &tp));
    r->tuple_len = tp.tuple_len;
    if (r->count == 0) return MBC_OK;
    MBC_TRY(dev_alloc(ctx, (void**)&r->d_tuples, (size_t)r->count * tp.tuple_len, false));
    tp.count = r->count;
    tp.out = r->d_tuples;
    int rows = std::max(16, std::min(128, (40 * 1024 / tp.tuple_len) / 16 * 16));
    tp.rows_per_cta = rows;
    int64_t grid = (r->count + rows - 1) / rows;
    size_t smem = (size_t)rows * tp.tuple_len;
    tuple_encode_kernel<<<(unsigned)grid, 128, smem, ctx->stream>>>(tp);
    ctx->launches++;
    MBC_CUDA(cudaGetLastError());
    return MBC_OK;
}

static int32_t pinned_for(mbc_result* r, void** p, size_t bytes) {
    size_t actual = 0;
    MBC_TRY(pinned_alloc(r->ctx, p, bytes, &actual));
    r->pinned.push_back({*p, actual});
    return MBC_OK;
}

int32_t finish_result_host(mbc_result* r) {
    mbc_ctx* ctx = r->ctx;
    if ((r->want & MBC_WANT_TUPLES) && !r->cols.empty()) MBC_TRY(encode_tuples(r));
    if (!(r->want & MBC_WANT_HOST)) return MBC_OK;
    const size_t n = (size_t)r->count;
    if ((r->want & MBC_WANT_POSITIONS) && r->d_pos) {
        MBC_TRY(pinned_for(r, (void**)&r->h_pos, n * 8));
        if (n) MBC_CUDA(cudaMemcpyAsync(r->h_pos, r->d_pos, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
        if (r->d_pos2) {
            MBC_TRY(pinned_for(r, (void**)&r->h_pos2, n * 8));
            if (n) MBC_CUDA(cudaMemcpyAsync(r->h_pos2, r->d_pos2, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
        }
    }
    if (r->want & MBC_WANT_COLUMNS) {
        for (auto& c : r->cols) {
            MBC_TRY(pinned_for(r, &c.h, n * c.width));
            if (!n) continue;
            if (c.stride == c.width)
                MBC_CUDA(cudaMemcpyAsync(c.h, c.d, n * c.width, cudaMemcpyDeviceToHost, ctx->stream));
            else
                MBC_CUDA(cudaMemcpy2DAsync(c.h, c.width, c.d, c.stride, c.width, n, cudaMemcpyDeviceToHost, ctx->stream));
        }
    }
    if ((r->want & MBC_WANT_TUPLES) && !r->cols.empty()) {
        MBC_TRY(pinned_for(r, (void**)&r->h_tuples, n * r->tuple_len));
        if (n) MBC_CUDA(cudaMemcpyAsync(r->h_tuples, r->d_tuples, n * r->tuple_len, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if ((r->want & MBC_WANT_BITMAP) && r->d_bitmap) {
        size_t words64 = (size_t)(r->nrows + 63) / 64;
        MBC_TRY(pinned_for(r, (void**)&r->h_bitmap, words64 * 8 + 8));
        if (words64) MBC_CUDA(cudaMemcpyAsync(r->h_bitmap, r->d_bitmap, words64 * 8, cudaMemcpyDeviceToHost, ctx->stream));
    }
    MBC_CUDA(cudaStreamSynchronize(ctx->stream));
    return MBC_OK;
}

static int32_t build_aggs(const mbc_table* t, const mbc_aggspec* aggs, int32_t nagg, DevAgg* dev) {
    if (nagg < 0 || nagg > kMaxAgg) MBC_FAIL(MBC_ERR_UNSUPPORTED, "%d aggregates (max %d)", nagg, kMaxAgg);
    memset(dev, 0, sizeof(DevAgg) * kMaxAgg);
    for (int a = 0; a < nagg; ++a) {
        DevAgg& d = dev[a];
        d.kind = aggs[a].kind;
        d.col = -1;
        if (d.kind == MBC_AGG_COUNT) { d.type = MBC_ATTR_INTEGER; continue; }
        if (d.kind < 0 || d.kind > MBC_AGG_MAX) MBC_FAIL(MBC_ERR_ARG, "aggregate %d: unknown kind %d", a, d.kind);
        int c = aggs[a].col;
        if (c < 0 || c >= (int)t->cols.size()) MBC_FAIL(MBC_ERR_ARG, "aggregate %d: column %d out of range", a, c);
        if (t->cols[c].type == MBC_ATTR_STRING) MBC_FAIL(MBC_ERR_UNSUPPORTED, "aggregate %d over a string column", a);
        d.type = t->cols[c].type;
        d.col = c;
        d.src = t->cols[c].d;
    }
    return MBC_OK;
}

void decode_aggs(mbc_result* r, const DevAgg* dev, int nagg, const unsigned long long* raw) {
    r->aggs.resize(nagg);
    for (int a = 0; a < nagg; ++a) {
        mbc_result::Agg& g = r->aggs[a];
        g.kind = dev[a].kind;
        g.type = dev[a].type;
        agg_from_raw(g.kind, g.type, raw[a], r->count > 0, &g.i, &g.f, &g.valid);
    }
}

// Workspace layout: [running count: 2 slots i64 @0][write-pass ticket counter u32 @32][agg out: 8 u64 + count @64][tile_counts: launch_tiles u32]
//                   [tile_out: launch_tiles + 1 u64][partials: nagg*total_tiles u64]
struct Workspace {
    long long* count;             // two slots: launch i reads slot i & 1 (not the first) and writes slot (i + 1) & 1
    uint32_t* tile_counts;
    unsigned long long* tile_out;
    unsigned long long* partials;
    unsigned long long* agg_out;  // [kMaxAgg] aggregates, [kMaxAgg] = the count (agg_finish_kernel)
    uint8_t* group_class;         // one byte per group of kGroupTiles tiles
};

static int32_t carve_workspace(mbc_ctx* ctx, int64_t launch_tiles, int64_t part_slots, int nagg, Workspace* w) {
    const size_t head = 64 + round_up((kMaxAgg + 1) * 8, 64);
    size_t counts_bytes = (size_t)round_up(launch_tiles * 4, 64);
    size_t out_bytes = (size_t)round_up((launch_tiles + 1) * 8, 64);
    size_t partial_bytes = (size_t)std::max(nagg, 1) * part_slots * 8;
    size_t class_bytes = (size_t)round_up(launch_tiles / kGroupTiles + 1, 64);
    size_t total = head + counts_bytes + out_bytes + partial_bytes + class_bytes + 64;
    MBC_TRY(ensure_workspace(ctx, total));
    char* b = (char*)ctx->ws;
    w->count = (long long*)b;
    w->agg_out = (unsigned long long*)(b + 64);
    w->tile_counts = (uint32_t*)(b + head);
    w->tile_out = (unsigned long long*)(b + head + counts_bytes);
    w->partials = (unsigned long long*)(b + head + counts_bytes + out_bytes);
    w->group_class = (uint8_t*)(b + head + counts_bytes + out_bytes + partial_bytes);
    return MBC_OK;
}

// A scan job: the parameter block, the result that owns the output buffers, and the workspace.
// `schema` supplies column types/strides; bind_table() points the job at the table whose rows the
// next launch reads (the resident table, or one of the staging tables of mbc_scan_host).
constexpr int kPartScale = kTileRows / kFR;   // partial slots per 4096-row tile: the fused engine's tiles are smaller

struct ScanJob {
    ScanParams p;
    mbc_result* r = nullptr;
    Workspace w;
    int64_t part_slots = 0;       // capacity (= stride) of the per-tile aggregate partials: one slot per tile of either engine
    int64_t part_done = 0;        // slots written by the launches so far
    size_t smem_bytes = 0;
    size_t staged_smem = 0;       // ring of write_staged_kernel
    bool staged_off = false;      // a launch whose projected columns are read in place from host memory gathers them
    bool pdl_tail = false;        // the last thing queued was a kernel of this job launched by launch_job (agg_finish may follow it with PDL)
    int max_grid = 1;
    int launches = 0;             // launches so far: the running count is in slot launches & 1
    // single-residency engine (mbc_scan_fused.cuh): planned once per job, chosen per launch
    bool fused_ok = false;
    bool fused_off = false;       // a launch whose projected columns are read in place from host memory stays two-pass
    FusedParams f;
    size_t fused_smem = 0;
    int fused_ctas_per_sm = 1;
    long long* count_slot() const { return w.count + (launches & 1); }
    int grid_per_tiles(int ntiles) const { return std::max(1, std::min(ntiles, max_grid)); }
};


// Dense groups through write_staged_kernel: every column the write pass reads (projected fields, aggregate sources) gets a
// slice of a ring stage; the ring takes what two CTAs per SM leave of the shared memory.  Off (write_kernel's own dense paths
// take over) when there is nothing to stage, or a stage is so wide that the ring would be shallower than two stages.
static void plan_staged(mbc_ctx* ctx, ScanJob* job) {
    ScanParams& p = job->p;
    p.stg_n = 0;
    p.dense_staged = 0;
    job->staged_smem = 0;
    // groups above this many survivors read their columns whole through write_staged_kernel; measured crossover with the
    // per-tile gather of write_kernel on B200 (profiles/README.md)
    p.stg_min = kGroupRows * 28 / 100;
    if (const char* g = getenv("MBC_STAGED_MIN_PCT")) p.stg_min = (int)((long long)kGroupRows * std::max(0, std::min(100, atoi(g))) / 100);
    p.stg_min = std::max(p.stg_min, kSparseMax);
    const char* e = getenv("MBC_WRITE_STAGED");                    // "0": the gather / streaming paths (tests, profiles)
    if (e && !strcmp(e, "0")) return;
    int n = 0;
    size_t off = 0;
    auto stage_of = [&](int col, int stride) -> int {
        for (int i = 0; i < n; ++i) if (p.stg_col[i] == col) return i;
        p.stg_col[n] = col;
        p.stg_stride[n] = stride;
        p.stg_off[n] = (int32_t)off;
        off += (size_t)stride * kStgRows;
        return n++;
    };
    for (int c = 0; c < p.nproj; ++c) {
        if (p.proj[c].stride & 3) return;
        p.proj_stg[c] = (int8_t)stage_of(p.proj[c].col, p.proj[c].stride);
    }
    for (int a = 0; a < p.nagg; ++a) p.agg_stg[a] = p.aggs[a].kind == MBC_AGG_COUNT ? (int8_t)-1 : (int8_t)stage_of(p.aggs[a].col, 4);
    if (n == 0) return;                                             // positions / counts only: nothing to read but the bitmap
    // per SM: 227 KB less the static arrays (list, barriers, partials) and the 1 KB the driver reserves per CTA, two CTAs
    static size_t budget = 0;
    if (!budget) {
        cudaFuncAttributes fa;
        if (cudaFuncGetAttributes(&fa, write_staged_kernel) != cudaSuccess) { cudaGetLastError(); return; }
        budget = (227 * 1024 - 2 * (fa.sharedSizeBytes + 1024)) / 2 / 128 * 128;
    }
    int stages = (int)std::min<size_t>(kStgMaxStages, budget / off);
    if (const char* m = getenv("MBC_STAGED_STAGES")) stages = std::min(stages, std::max(1, atoi(m)));
    if (stages < 2) return;
    if (!ctx->staged_smem_set) {
        if (cudaFuncSetAttribute(write_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget) != cudaSuccess) {
            cudaGetLastError();
            return;
        }
        ctx->staged_smem_set = true;
    }
    p.stg_n = n;
    p.stg_stages = stages;
    p.stg_bytes = (int32_t)off;
    job->staged_smem = (size_t)stages * off;
}

// Plan the single-residency engine (mbc_scan_fused.cuh) for this job: payload columns, ring depths, shared memory.
// Leaves job->fused_ok false when the scan does not fit it; every launch then takes the two-pass engine.
static void plan_fused(mbc_ctx* ctx, ScanJob* job) {
    job->fused_ok = false;
    // MBC_SCAN_PATH=fused opts in (tests, profiles).  Measured on B200 (profiles/README.md): the two-pass engine with the
    // TMA-staged dense write pass is faster at every selectivity -- the fused kernel's three roles each sit close to
    // the per-tile HBM time (term-program interpretation in the count warps, the ~2 us L2 round trip of the published
    // counts while HBM is saturated, ~800 instructions per tile and warp in the write warps), so it is not the default.
    const char* path = getenv("MBC_SCAN_PATH");
    if (!path || strcmp(path, "fused")) return;
    ScanParams& p = job->p;
    FusedParams& f = job->f;
    memset(&f, 0, sizeof(f));
    bool need_write = p.out_pos || p.nproj > 0;
    for (int a = 0; a < p.nagg; ++a) need_write |= p.aggs[a].kind != MBC_AGG_COUNT;
    if (!need_write) return;                                       // COUNT alone: pass 1 + the offsets kernel is all there is to do
    if (ctx->fused_smem_budget < 0) {                              // once per context: opt in to the large shared memory carve-out
        ctx->fused_smem_budget = 0;
        int reserved = 0, optin = 0, coop = 0;
        cudaFuncAttributes fa;
        if (cudaDeviceGetAttribute(&reserved, cudaDevAttrReservedSharedMemoryPerBlock, ctx->device) == cudaSuccess &&
            cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device) == cudaSuccess &&
            cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, ctx->device) == cudaSuccess && coop &&
            cudaFuncGetAttributes(&fa, fused_scan_kernel) == cudaSuccess) {
            const int budget = (optin - (int)fa.sharedSizeBytes) / 1024 * 1024;   // one CTA per SM: everything the SM has
            if (budget > 0 && cudaFuncSetAttribute(fused_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, budget) == cudaSuccess)
                ctx->fused_smem_budget = budget;
        }
        cudaGetLastError();
    }
    const int budget = ctx->fused_smem_budget;
    if (budget <= 0) return;
    // payload = the distinct projected / aggregated columns, laid out back to back in a payload stage
    int pay_col[kFMaxPay];
    auto pay_of = [&](int col, int stride) -> int {
        for (int k = 0; k < f.npay; ++k) if (pay_col[k] == col) return k;
        if (f.npay == kFMaxPay || (stride & 3)) return -1;
        pay_col[f.npay] = col;
        f.pay_stride[f.npay] = stride;
        f.pay_off[f.npay] = f.pay_stage_bytes;
        f.pay_stage_bytes += stride * kFR;
        return f.npay++;
    };
    for (int c = 0; c < p.nproj; ++c) {
        const int k = pay_of(p.proj[c].col, p.proj[c].stride);
        if (k < 0) return;
        f.proj_pay[c] = (int8_t)k;
    }
    for (int a = 0; a < p.nagg; ++a) {
        f.agg_pay[a] = -1;
        if (p.aggs[a].kind == MBC_AGG_COUNT) continue;
        const int k = pay_of(p.aggs[a].col, 4);
        if (k < 0) return;
        f.agg_pay[a] = (int8_t)k;
    }
    const int pred_stage = p.nstaged * kFPredColBytes, pay_stage = f.pay_stage_bytes;
    // Ring depths.  The payload ring takes 3 stages when they fit (one tile being written, two loading: ~110 KB in flight
    // per SM for the C2 row), the predicate ring the rest; a scan that fetches nothing per row gives it all to the predicates.
    int P = 2, S = 0;
    if (f.npay) {
        S = std::min(3, (budget - 2 * pred_stage) / pay_stage);
        if (S < 2) return;                                         // rows too wide for a double-buffered shared-memory tile
    }
    if (const char* e = getenv("MBC_FUSED_PAY_STAGES")) S = f.npay ? std::max(2, std::min(kFMaxPayStages, atoi(e))) : 0;
    if (pred_stage) P = std::max(2, std::min(kFMaxPredStages, (budget - S * pay_stage) / pred_stage));
    if (const char* e = getenv("MBC_FUSED_PRED_STAGES")) P = std::max(2, std::min(kFMaxPredStages, atoi(e)));
    // every predicate stage belongs to ONE count group (tile i -> stage i % P, group i % kFGroups): a waiter never sees a stage
    // whose previous phase was another group's (mbarrier parity waits cannot tell "two phases behind" from "done")
    P = P / kFGroups * kFGroups;
    if (P < kFGroups || (size_t)P * pred_stage + (size_t)S * pay_stage > (size_t)budget) return;
    f.pred_stages = P;
    f.pay_stages = S;
    f.dense_min = kFR / 16;                                        // below 1 survivor in 16 rows a batched gather moves fewer bytes
    if (const char* e = getenv("MBC_FUSED_DENSE_MIN")) f.dense_min = atoi(e);
    f.dense_min = std::max(1, std::min(f.dense_min, kFPendCap / 2));
    job->fused_smem = (size_t)P * pred_stage + (size_t)S * pay_stage;
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fused_scan_kernel, kFThreads, job->fused_smem) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        return;
    }
    job->fused_ctas_per_sm = 1;
    job->fused_ok = true;
}

// published-count buffer of the fused engine: grown (zero filled) on demand, never cleared between launches
static int32_t fused_flags_for(mbc_ctx* ctx, int64_t ntiles, uint32_t** flags, uint32_t* epoch) {
    ntiles += kFMaxGrid;                                           // the control warps bulk-copy whole waves: one wave of padding
    if (ctx->fused_flags_cap < ntiles) {
        if (ctx->fused_flags) {
            MBC_CUDA(cudaStreamSynchronize(ctx->stream));
            MBC_CUDA(cudaFree(ctx->fused_flags));
            ctx->fused_flags = nullptr;
            ctx->fused_flags_cap = 0;
        }
        const int64_t cap = std::max<int64_t>(round_up(ntiles, 4096), 65536);
        MBC_CUDA(cudaMalloc((void**)&ctx->fused_flags, (size_t)cap * 4));
        MBC_CUDA(cudaMemsetAsync(ctx->fused_flags, 0, (size_t)cap * 4, ctx->stream));
        ctx->fused_flags_cap = cap;
        ctx->fused_epoch = 0;
    }
    if (++ctx->fused_epoch >= (1u << (32 - kFCountBits))) {       // the tag wrapped: stale words could match again
        MBC_CUDA(cudaMemsetAsync(ctx->fused_flags, 0, (size_t)ctx->fused_flags_cap * 4, ctx->stream));
        ctx->fused_epoch = 1;
    }
    *flags = ctx->fused_flags;
    *epoch = ctx->fused_epoch;
    return MBC_OK;
}

static int32_t prepare_job(const mbc_table* schema, const ScanRequest& rq, int64_t capacity_rows, int64_t launch_tiles,
                           int64_t total_tiles, ScanJob* job) {
    mbc_ctx* ctx = schema->ctx;
    if (rq.nproj < 0 || rq.nproj > kMaxProj) MBC_FAIL(MBC_ERR_UNSUPPORTED, "%d projected fields (max %d)", rq.nproj, kMaxProj);
    if ((rq.nterms > 0 && !rq.terms) || (rq.nproj > 0 && !rq.proj_cols) || (rq.nagg > 0 && !rq.aggs))
        MBC_FAIL(MBC_ERR_ARG, "scan: NULL array with a non-zero count");
    if (launch_tiles > INT32_MAX || total_tiles > INT32_MAX) MBC_FAIL(MBC_ERR_UNSUPPORTED, "table too large for one device scan");
    ScanParams& p = job->p;
    memset(&p, 0, sizeof(p));
    MBC_TRY(build_terms(schema, rq.terms, rq.nterms, p.terms));
    p.nterms = rq.nterms;
    p.nagg = (rq.want & MBC_WANT_AGG) ? rq.nagg : 0;
    MBC_TRY(build_aggs(schema, rq.aggs, p.nagg, p.aggs));
    for (int c = 0; c < rq.nproj; ++c)
        if (rq.proj_cols[c] < 0 || rq.proj_cols[c] >= (int)schema->cols.size())
            MBC_FAIL(MBC_ERR_ARG, "projection field %d: column %d out of range", c, rq.proj_cols[c]);

    mbc_result* r = new mbc_result();
    job->r = r;
    r->ctx = ctx;
    ctx_retain(ctx);
    r->want = rq.want;
    r->capacity = capacity_rows;
    const bool want_cols = (rq.want & (MBC_WANT_COLUMNS | MBC_WANT_TUPLES)) != 0 && rq.nproj > 0;
    if (rq.want & MBC_WANT_POSITIONS) MBC_TRY(dev_alloc(ctx, (void**)&r->d_pos, (size_t)capacity_rows * 8, false));
    if (want_cols) {
        for (int c = 0; c < rq.nproj; ++c) {
            const Column& col = schema->cols[rq.proj_cols[c]];
            mbc_result::Col rc{col.type, col.width, col.stride, nullptr, nullptr};
            MBC_TRY(dev_alloc(ctx, &rc.d, (size_t)capacity_rows * col.stride, false));
            r->cols.push_back(rc);
            p.proj[c].dst = rc.d;
            p.proj[c].stride = col.stride;
            p.proj[c].col = rq.proj_cols[c];
        }
        p.nproj = rq.nproj;
    }
    MBC_TRY(dev_alloc(ctx, (void**)&r->d_aggs, (kMaxAgg + 1) * 8, false));
    if (total_tiles * kPartScale > INT32_MAX) MBC_FAIL(MBC_ERR_UNSUPPORTED, "table too large for one device scan");
    job->part_slots = total_tiles * kPartScale;
    MBC_TRY(carve_workspace(ctx, launch_tiles, job->part_slots, p.nagg, &job->w));
    p.total_tiles = (int)job->part_slots;
    p.tile_counts = job->w.tile_counts;
    p.tile_out = job->w.tile_out;
    p.group_class = job->w.group_class;
    p.partials = job->w.partials;
    p.out_pos = r->d_pos;
    p.out_cap = capacity_rows;
    p.ntiles = INT32_MAX;                         // the grid bound comes from the device; bind_table sets the real count
    MBC_TRY(plan_staging(ctx, &p, &job->smem_bytes, &job->max_grid));
    // who loads an aggregate's source values in the gather paths of write_kernel: the projection of the same column if there
    // is one, else the first aggregate of that column on behalf of all of them
    memset(p.proj_aggs, 0, sizeof(p.proj_aggs));
    memset(p.agg_group, 0, sizeof(p.agg_group));
    for (int a = 0; a < p.nagg; ++a) {
        if (p.aggs[a].kind == MBC_AGG_COUNT) continue;
        int owner = -1;
        for (int c = 0; c < p.nproj && owner < 0; ++c)
            if (p.proj[c].col == p.aggs[a].col && p.proj[c].stride == 4) owner = c;
        if (owner >= 0) { p.proj_aggs[owner] |= (uint8_t)(1u << a); continue; }
        int first = a;
        for (int b = 0; b < a; ++b)
            if (p.aggs[b].kind != MBC_AGG_COUNT && p.aggs[b].col == p.aggs[a].col) { first = b; break; }
        p.agg_group[first] |= (uint8_t)(1u << a);
    }
    plan_staged(ctx, job);
    plan_fused(ctx, job);
    return MBC_OK;
}

static void bind_table(ScanJob* job, const mbc_table* t) {
    ScanParams& p = job->p;
    for (int k = 0; k < p.nterms; ++k) {
        if (p.terms[k].lhs.kind == 1) p.terms[k].lhs.ptr = t->cols[p.terms[k].lhs.col].d;
        if (p.terms[k].rhs.kind == 1) p.terms[k].rhs.ptr = t->cols[p.terms[k].rhs.col].d;
    }
    for (int c = 0; c < p.nproj; ++c) p.proj[c].src = t->cols[p.proj[c].col].d;
    for (int s = 0; s < p.nstaged; ++s) p.staged_src[s] = t->cols[p.staged_cols[s]].d;
    for (int i = 0; i < p.stg_n; ++i) p.stg_src[i] = t->cols[p.stg_col[i]].d;
    for (int a = 0; a < p.nagg; ++a)
        if (p.aggs[a].col >= 0) p.aggs[a].src = t->cols[p.aggs[a].col].d;
    p.deleted = t->has_deleted ? t->d_deleted : nullptr;
    p.nrows = t->nrows;
    p.pos_base = t->pos_base;
    p.ntiles = (int)((t->nrows + kTileRows - 1) / kTileRows);
}

// Launch with (or without) programmatic dependent launch: the kernel may be scheduled while its predecessor in the stream
// is still running and blocks in pdl_wait() until that has completed (mbc_scan_kernels.cuh).  Opt-in (MBC_PDL=1): measured on
// B200 it does not pay here -- C2 step 1.769 ms with, 1.761 ms without; C5 1.009 vs 0.985 ms; the 25 % scan 0.84 vs 0.81 ms:
// the early CTAs of a successor sit on registers and shared memory its predecessor's last waves could use.
static bool pdl_enabled() {
    static const int on = [] { const char* e = getenv("MBC_PDL"); return e ? atoi(e) : 0; }();
    return on != 0;
}
template <typename... KArgs, typename... Args>
static cudaError_t launch_after(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// the launches over the bound table; its tiles take the next slots of the partials array
static int32_t launch_job(ScanJob* job, bool first) {
    mbc_ctx* ctx = job->r->ctx;
    ScanParams& p = job->p;
    if (first) { job->launches = 0; job->part_done = 0; }
    p.tile_base = (int)job->part_done;
    if (p.ntiles == 0) return MBC_OK;
    p.count_in = job->launches == 0 ? nullptr : job->count_slot();   // later launches append at the running offset
    p.count_out = job->w.count + ((job->launches + 1) & 1);
    p.work_counter = reinterpret_cast<unsigned int*>(job->w.count + 4);
    if (job->fused_ok && !job->fused_off && !(p.nterms == 0 && p.sel_bitmap)) {
        // single residency: count warps ahead, offsets from the published counts, compaction out of shared memory
        FusedParams& f = job->f;
        const int64_t ntiles = (p.nrows + kFR - 1) / kFR;
        f.ntiles = (int32_t)ntiles;
        MBC_TRY(fused_flags_for(ctx, ntiles, &f.flags, &f.epoch));
        for (int c = 0; c < p.nproj; ++c) f.pay_src[f.proj_pay[c]] = p.proj[c].src;
        for (int a = 0; a < p.nagg; ++a)
            if (f.agg_pay[a] >= 0) f.pay_src[f.agg_pay[a]] = p.aggs[a].src;
        int grid = (int)std::min<int64_t>(ntiles, std::min(ctx->sm_count, kFMaxGrid));
        if (grid >= 4) grid &= ~3;                                  // a wave of published counts is a 16-byte multiple
        const bool prof = getenv("MBC_FUSED_PROF") != nullptr;      // per-role wait cycles of every CTA, averaged, on stderr
        f.prof = nullptr;
        if (prof) MBC_TRY(dev_alloc(ctx, (void**)&f.prof, (size_t)grid * 24 * 8, true));
        f.dbg = nullptr;
#ifdef MBC_FUSED_DEBUG
        static long long* h_dbg = nullptr;                          // host-mapped: survives a faulting kernel
        if (!h_dbg && cudaHostAlloc((void**)&h_dbg, 64, cudaHostAllocMapped) == cudaSuccess) memset(h_dbg, 0, 64);
        if (h_dbg) {
            if (h_dbg[0]) fprintf(stderr, "[fused check] EARLIER launch: line %lld cta %lld thread %lld values %lld %lld %lld %lld\n", h_dbg[0], h_dbg[1],
                                  h_dbg[2], h_dbg[3], h_dbg[4], h_dbg[5], h_dbg[6]);
            cudaHostGetDevicePointer((void**)&f.dbg, h_dbg, 0);
        }
#endif
        void* args[] = {(void*)&p, (void*)&f};
        MBC_CUDA(cudaLaunchCooperativeKernel((const void*)fused_scan_kernel, dim3(grid), dim3(kFThreads), args, job->fused_smem, ctx->stream));
#ifdef MBC_FUSED_DEBUG
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess && h_dbg)
            fprintf(stderr, "[fused check] line %lld cta %lld thread %lld values %lld %lld %lld %lld (grid %d P %d S %d ntiles %lld)\n", h_dbg[0], h_dbg[1], h_dbg[2],
                    h_dbg[3], h_dbg[4], h_dbg[5], h_dbg[6], grid, f.pred_stages, f.pay_stages, (long long)ntiles);
#endif
        if (prof) {
            std::vector<long long> h((size_t)grid * 24);
            MBC_CUDA(cudaMemcpyAsync(h.data(), f.prof, h.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
            MBC_CUDA(cudaStreamSynchronize(ctx->stream));
            dev_free(ctx, f.prof);
            double m[24] = {0};
            for (int c = 0; c < grid; ++c)
                for (int k = 0; k < 24; ++k) m[k] += (double)h[(size_t)c * 24 + k] / grid;
            fprintf(stderr,
                    "[fused prof] tiles/cta %.1f grid %d P %d S %d dense_min %d | control: total %.0f flag-wait %.0f sum+stale %.0f payfree-wait %.0f "
                    "dense %.1f stale waves %.1f | count(g0): total %.0f maskfree-wait %.0f pred-wait %.0f eval %.0f | write: total %.0f "
                    "maskready-wait %.0f ctl-wait %.0f rank %.0f payfull-wait %.0f dense+other %.0f sparse %.0f flush %.0f (cycles, mean over CTAs)\n",
                    (double)ntiles / grid, grid, f.pred_stages, f.pay_stages, f.dense_min, m[0], m[1], m[2], m[3], m[4], m[5], m[8], m[9], m[10],
                    m[11], m[12], m[13], m[14], m[15], m[16], m[17], m[18], m[19]);
        }
        job->launches++;
        ctx->launches++;
        job->part_done += grid;                                     // one aggregate partial per CTA
        for (int i = 0; i < 3; ++i)
            if (job->r->ev_mid[i]) cudaEventRecord(job->r->ev_mid[i], ctx->stream);
        return MBC_OK;
    }
    if (p.nterms == 0 && p.sel_bitmap) {
        const int grid = std::max(1, std::min((p.ntiles + kWarpsPerCta - 1) / kWarpsPerCta, ctx->sm_count * 8));
        select_bitmap_kernel<<<grid, kScanThreads, 0, ctx->stream>>>(p.sel_bitmap, p.deleted, p.nrows, p.ntiles, p.out_bitmap, p.tile_counts);
    } else {
        filter_kernel<<<job->grid_per_tiles(p.ntiles), kScanThreads, job->smem_bytes, ctx->stream>>>(p);
    }
    if (job->r->ev_mid[0]) cudaEventRecord(job->r->ev_mid[0], ctx->stream);
    const bool pdl = pdl_enabled() && !job->r->ev_mid[0];          // events between the launches would serialise them anyway
    // groups above p.stg_min survivors go to write_staged_kernel when their columns fit its ring; write_kernel writes the
    // others (and those too when they do not).  Tables of >= 49 152 tiles take the persistent write_kernel (a sparse scan of
    // 10^5 tiles saves the dispatch of as many idle CTAs: 0.78 vs 0.86 ms on 500 M rows at 0.01 %), whose tile-by-tile gather
    // of mid groups is slow (250 M rows at 25 %: 2.67 ms against 1.93 ms with one CTA per tile) -- there every group above
    // the sparse limit is staged (2.07 ms).
    const bool staged_now = p.stg_n > 0 && !job->staged_off;
    const char* pt = getenv("MBC_WRITE_PERSISTENT_TILES");              // tests force either form
    const bool persistent = p.ntiles >= (pt ? atoi(pt) : 49152);
    const int full_min = (persistent && staged_now && !getenv("MBC_STAGED_MIN_PCT")) ? kSparseMax : p.stg_min;
    launch_after(tile_offsets_kernel, dim3((p.ntiles + kOffsetsPerBlock - 1) / kOffsetsPerBlock), dim3(1024), 0, ctx->stream, pdl,
                 (const uint32_t*)p.tile_counts, p.ntiles, p.tile_out, p.count_in, p.count_out, p.work_counter, p.group_class, (int)kSparseMax,
                 full_min);
    job->launches++;
    ctx->launches += 2;
    job->part_done += p.ntiles;
    if (job->r->ev_mid[1]) cudaEventRecord(job->r->ev_mid[1], ctx->stream);
    bool need_write = p.out_pos || p.nproj > 0;
    for (int a = 0; a < p.nagg; ++a) need_write |= p.aggs[a].kind != MBC_AGG_COUNT;   // COUNT comes from the tile offsets
    if (need_write) {
        p.dense_staged = staged_now ? 1 : 0;
        if (persistent) {
            static int ctas_per_sm = 0;
            if (!ctas_per_sm &&
                (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, write_kernel<true>, kScanThreads, 0) != cudaSuccess || ctas_per_sm < 1))
                ctas_per_sm = 1;
            launch_after(write_kernel<true>, dim3(std::min(p.ntiles, ctx->sm_count * ctas_per_sm)), dim3(kScanThreads), 0, ctx->stream, pdl, p);
        } else {
            launch_after(write_kernel<false>, dim3(p.ntiles), dim3(kScanThreads), 0, ctx->stream, pdl, p);
        }
        ctx->launches++;
        if (staged_now) {
            p.dense_staged = 0;
            launch_after(write_staged_kernel, dim3(std::min(p.ntiles, ctx->sm_count * 2)), dim3(kStgThreads), job->staged_smem, ctx->stream, pdl, p);
            ctx->launches++;
        }
    }
    if (job->r->ev_mid[2]) cudaEventRecord(job->r->ev_mid[2], ctx->stream);
    job->pdl_tail = pdl;
    MBC_CUDA(cudaGetLastError());
    return MBC_OK;
}

// aggregate finish + count/aggregate readback.  Synchronous form: the device work of the job is complete after this.
// Deferred form: everything is queued, the result carries the event and mbc::result_finalize() completes it.
static int32_t finish_job_device(ScanJob* job, bool deferred = false) {
    mbc_ctx* ctx = job->r->ctx;
    ScanParams& p = job->p;
    mbc_result* r = job->r;
    if (job->launches == 0) MBC_CUDA(cudaMemsetAsync(job->w.count, 0, 16, ctx->stream));   // nothing was scanned
    if (p.nagg > 0) {
        bool count_only = true;
        for (int a = 0; a < p.nagg; ++a) count_only &= p.aggs[a].kind == MBC_AGG_COUNT;
        if (count_only) {
            agg_count_only_kernel<<<1, 32, 0, ctx->stream>>>(p.nagg, job->w.agg_out, job->count_slot());
        } else {
            AggList list;
            memcpy(list.g, p.aggs, sizeof(list.g));
            // (after the last launch of a resident scan; a chunked host scan has copies in between: plain launch)
            const bool pdl = pdl_enabled() && job->pdl_tail;
            launch_after(agg_finish_kernel, dim3(p.nagg), dim3(1024), 0, ctx->stream, pdl, (const unsigned long long*)job->w.partials,
                         (int)job->part_slots, (int)job->part_done, list, job->w.agg_out, (const long long*)job->count_slot());
        }
        ctx->launches++;
        MBC_CUDA(cudaGetLastError());
    }
    end_timing(ctx);
    if (r->ev_t1) cudaEventRecord(r->ev_t1, ctx->stream);
    // count + aggregates come back in one small copy
    if (p.nagg > 0) {
        MBC_CUDA(cudaMemcpyAsync(r->d_aggs, job->w.agg_out, (kMaxAgg + 1) * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    } else {
        MBC_CUDA(cudaMemcpyAsync(r->d_aggs + kMaxAgg, job->count_slot(), 8, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    r->ev_done = event_get(ctx);                                   // mbc_shard_gather pushes behind this, not behind later scans
    if (r->ev_done) cudaEventRecord(r->ev_done, ctx->stream);
    if (deferred) {
        r->aggs.resize(p.nagg);
        for (int a = 0; a < p.nagg; ++a) { r->aggs[a].kind = p.aggs[a].kind; r->aggs[a].type = p.aggs[a].type; }
        MBC_TRY(pinned_for(r, (void**)&r->h_small, (kMaxAgg + 1) * 8));
        MBC_CUDA(cudaMemcpyAsync(r->h_small, r->d_aggs, (kMaxAgg + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
        r->ev_ready = event_get(ctx);
        if (!r->ev_ready) MBC_FAIL(MBC_ERR_CUDA, "cudaEventCreate failed");
        MBC_CUDA(cudaEventRecord(r->ev_ready, ctx->stream));
        return MBC_OK;
    }
    unsigned long long host_small[kMaxAgg + 1];
    MBC_CUDA(cudaMemcpyAsync(host_small, r->d_aggs, sizeof(host_small), cudaMemcpyDeviceToHost, ctx->stream));
    MBC_CUDA(cudaStreamSynchronize(ctx->stream));
    r->count = (int64_t)host_small[kMaxAgg];
    decode_aggs(r, p.aggs, p.nagg, host_small);
    if (r->ev_t0 && r->ev_t1 && cudaEventElapsedTime(&r->kernel_ms, r->ev_t0, r->ev_t1) != cudaSuccess) r->kernel_ms = -1.f;
    result_phase_times(r);
    return MBC_OK;
}

static int32_t finish_job(ScanJob* job) {
    MBC_TRY(finish_job_device(job));
    return finish_result_host(job->r);
}

int32_t run_scan(const ScanRequest& rq, mbc_result** out) {
    mbc_table* t = rq.table;
    if (!t || !out) MBC_FAIL(MBC_ERR_ARG, "scan: table/out is NULL");
    *out = nullptr;
    mbc_ctx* ctx = t->ctx;
    MBC_CUDA(cudaSetDevice(ctx->device));
    const int64_t ntiles = (t->nrows + kTileRows - 1) / kTileRows;
    ScanJob job;
    int32_t s = prepare_job(t, rq, t->nrows, std::max<int64_t>(ntiles, 1), std::max<int64_t>(ntiles, 1), &job);
    if (s == MBC_OK) {
        mbc_result* r = job.r;
        r->nrows = t->nrows;
        job.p.sel_bitmap = rq.d_sel_bitmap;
        // the filter pass always leaves the selection as a bitmap; it is the result's bitmap when asked for
        // (the filter writes every word of every tile: only the padding beyond the last tile is zeroed)
        s = dev_alloc(ctx, (void**)&r->d_bitmap, (size_t)t->words_pad * 4, false);
        const int64_t written = ntiles * (kTileRows / 32);
        if (s == MBC_OK && t->words_pad > written &&
            cudaMemsetAsync(r->d_bitmap + written, 0, (size_t)(t->words_pad - written) * 4, ctx->stream) != cudaSuccess) s = MBC_ERR_CUDA;
        r->bitmap_words32 = t->words_pad;
        job.p.out_bitmap = r->d_bitmap;
    }
    if (s == MBC_OK) {
        bind_table(&job, t);
        begin_timing(ctx);
        job.r->ev_t0 = event_get(ctx);
        job.r->ev_t1 = event_get(ctx);
        if (getenv("MBC_PHASE_EVENTS"))                        // per-kernel times of a resident scan (mbc_result_phase_ms): three
            for (auto& e : job.r->ev_mid) e = event_get(ctx);  // more events between the launches, so only on request
        if (job.r->ev_t0) cudaEventRecord(job.r->ev_t0, ctx->stream);
        s = launch_job(&job, true);
    }
    const bool deferred = rq.allow_deferred && !(rq.want & (MBC_WANT_HOST | MBC_WANT_TUPLES)) && !getenv("MBC_SYNC_RESULTS");
    if (s == MBC_OK) s = deferred ? finish_job_device(&job, true) : finish_job(&job);
    if (s != MBC_OK) {
        if (job.r) mbc_result_free(job.r);
        return s;
    }
    *out = job.r;
    return MBC_OK;
}

// Host-resident columns: stream row chunks through two staging tables.  The copy stream uploads
// chunk k+1 while the scan of chunk k runs; every chunk appends to the same result buffers (the
// output offsets of a chunk start from the running count left by the previous one).
static int32_t run_scan_host(mbc_ctx* ctx, int32_t ncols, const mbc_coldesc* cols, const void* const* host_cols,
                             int64_t nrows, int64_t position_base, const ScanRequest& rq_in, mbc_result** out) {
    *out = nullptr;
    MBC_CUDA(cudaSetDevice(ctx->device));
    const int64_t chunk_rows = 4 << 20;                      // 4 Mi rows per chunk (multiple of the tile)
    const int64_t sample_rows = 256 << 10;                   // first chunk of a scan that may materialise late
    const int64_t stage_rows = std::min<int64_t>(chunk_rows, std::max<int64_t>(nrows, 1));

    // Late materialisation: a column that is only projected / aggregated (not compared) need not cross PCIe in full.
    // When its host buffer is pinned (device-addressable) and laid out like the device column, a selective scan uploads
    // the predicate columns alone and the write pass gathers the survivors' values straight from host memory.  The
    // decision is taken from the selectivity of a small first chunk.
    std::vector<char> pred(ncols, 0), late_ok(ncols, 0);
    std::vector<const char*> host_dev(ncols, nullptr);
    for (int k = 0; k < rq_in.nterms; ++k)
        for (const mbc_operand* o : {&rq_in.terms[k].lhs, &rq_in.terms[k].rhs})
            if (o->kind != MBC_OPERAND_LITERAL && o->col >= 0 && o->col < ncols) pred[o->col] = 1;
    bool any_late = false;
    if (nrows > 2 * chunk_rows && !getenv("MBC_NO_LATE")) {
        for (int c = 0; c < ncols; ++c) {
            const bool plain = cols[c].type != MBC_ATTR_STRING || (cols[c].width > 0 && str_stride(cols[c].width) == cols[c].width);
            if (pred[c] || !plain || ((uintptr_t)host_cols[c] & 15u)) continue;
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, host_cols[c]) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) {
                host_dev[c] = (const char*)at.devicePointer;
                late_ok[c] = 1;
                any_late = true;
            } else {
                cudaGetLastError();
            }
        }
    }
    struct Chunk { int64_t row0, n; };
    std::vector<Chunk> chunks;
    {
        int64_t r0 = 0;
        if (any_late) { chunks.push_back({0, sample_rows}); r0 = sample_rows; }
        for (; r0 < nrows; r0 += chunk_rows) chunks.push_back({r0, std::min<int64_t>(chunk_rows, nrows - r0)});
        if (chunks.empty()) chunks.push_back({0, 0});
    }
    const int64_t nchunks = (int64_t)chunks.size();
    int64_t plan_tiles = 0;
    for (const Chunk& ch : chunks) plan_tiles += (ch.n + kTileRows - 1) / kTileRows;
    mbc_table* stage[2] = {nullptr, nullptr};
    cudaEvent_t ev_up[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
    ScanJob job;
    int32_t s = MBC_OK;
    auto cleanup = [&]() {
        for (int b = 0; b < 2; ++b) {
            if (stage[b]) mbc_table_free(stage[b]);
            if (ev_up[b]) cudaEventDestroy(ev_up[b]);
            if (ev_done[b]) cudaEventDestroy(ev_done[b]);
        }
    };
    for (int b = 0; b < 2 && s == MBC_OK; ++b) {
        s = mbc_table_create(ctx, ncols, cols, stage_rows, position_base, &stage[b]);
        if (s == MBC_OK && cudaEventCreateWithFlags(&ev_up[b], cudaEventDisableTiming) != cudaSuccess) s = MBC_ERR_CUDA;
        if (s == MBC_OK && cudaEventCreateWithFlags(&ev_done[b], cudaEventDisableTiming) != cudaSuccess) s = MBC_ERR_CUDA;
    }
    if (s != MBC_OK) { cleanup(); return s; }

    ScanRequest rq = rq_in;
    rq.table = stage[0];
    const int64_t tiles_per_chunk = (stage_rows + kTileRows - 1) / kTileRows;
    s = prepare_job(stage[0], rq, nrows, tiles_per_chunk, std::max<int64_t>(plan_tiles, 1), &job);
    if (s != MBC_OK) { if (job.r) mbc_result_free(job.r); cleanup(); return s; }
    job.r->nrows = nrows;
    // per-chunk selection bitmap of the filter pass (scratch: the chunks reuse it in stream order)
    s = dev_alloc(ctx, (void**)&job.r->d_bitmap, (size_t)stage[0]->words_pad * 4, true);
    if (s != MBC_OK) { mbc_result_free(job.r); cleanup(); return s; }
    job.p.out_bitmap = job.r->d_bitmap;

    // which columns does the query touch?
    std::vector<char> used(ncols, 0);
    for (int k = 0; k < job.p.nterms; ++k) {
        if (job.p.terms[k].lhs.kind == 1) used[job.p.terms[k].lhs.col] = 1;
        if (job.p.terms[k].rhs.kind == 1) used[job.p.terms[k].rhs.col] = 1;
    }
    for (int c = 0; c < job.p.nproj; ++c) used[job.p.proj[c].col] = 1;
    for (int a = 0; a < job.p.nagg; ++a) if (job.p.aggs[a].col >= 0) used[job.p.aggs[a].col] = 1;

    // the staging tables were zero-filled on ctx->stream; the copy stream must not overtake that
    cudaEvent_t ev_init;
    cudaEventCreateWithFlags(&ev_init, cudaEventDisableTiming);
    cudaEventRecord(ev_init, ctx->stream);
    cudaStreamWaitEvent(ctx->copy_stream, ev_init, 0);
    cudaEventDestroy(ev_init);

    // Results stream back while later chunks are still uploading (PCIe is full duplex): after every chunk the running
    // count comes to the host, and the rows that chunk appended are copied out on a third stream.  The pinned result
    // buffers are sized from the first chunk's selectivity (x1.3); if the estimate is exceeded the rest is copied at the end.
    mbc_result* r = job.r;
    const bool stream_out = (rq.want & MBC_WANT_HOST) && (rq.want & (MBC_WANT_POSITIONS | MBC_WANT_COLUMNS)) && nchunks > 2;
    long long* h_counts = nullptr;
    if (stream_out || any_late) {
        s = pinned_for(r, (void**)&h_counts, (size_t)(nchunks + 1) * 8);
        if (s != MBC_OK) { mbc_result_free(job.r); cleanup(); return s; }
    }
    int64_t out_cap = -1, copied = 0;
    bool out_overflow = false;
    auto copy_rows = [&](int64_t from, int64_t to) -> int32_t {          // rows [from, to) of every host-visible buffer
        if (to <= from) return MBC_OK;
        const size_t n = (size_t)(to - from);
        if (r->h_pos) MBC_CUDA(cudaMemcpyAsync(r->h_pos + from, r->d_pos + from, n * 8, cudaMemcpyDeviceToHost, ctx->d2h_stream));
        if (rq.want & MBC_WANT_COLUMNS)
            for (auto& c : r->cols) {
                if (c.stride == c.width)
                    MBC_CUDA(cudaMemcpyAsync((char*)c.h + (size_t)from * c.width, (char*)c.d + (size_t)from * c.stride, n * c.width,
                                             cudaMemcpyDeviceToHost, ctx->d2h_stream));
                else
                    MBC_CUDA(cudaMemcpy2DAsync((char*)c.h + (size_t)from * c.width, c.width, (char*)c.d + (size_t)from * c.stride, c.stride,
                                               c.width, n, cudaMemcpyDeviceToHost, ctx->d2h_stream));
            }
        return MBC_OK;
    };
    auto drain = [&](int64_t k) -> int32_t {                              // chunk k has finished on the device
        MBC_CUDA(cudaEventSynchronize(ev_done[k & 1]));
        const int64_t c = h_counts[k];
        if (out_cap < 0) {
            const int64_t rows_seen = chunks[k].row0 + chunks[k].n;
            out_cap = std::min<int64_t>(nrows, (int64_t)((double)c / (double)rows_seen * (double)nrows * 1.3) + 65536);
            if ((rq.want & MBC_WANT_POSITIONS) && r->d_pos) MBC_TRY(pinned_for(r, (void**)&r->h_pos, (size_t)out_cap * 8));
            if (rq.want & MBC_WANT_COLUMNS)
                for (auto& col : r->cols) MBC_TRY(pinned_for(r, &col.h, (size_t)out_cap * col.width));
        }
        if (out_overflow || c > out_cap) { out_overflow = true; return MBC_OK; }
        MBC_TRY(copy_rows(copied, c));
        copied = c;
        return MBC_OK;
    };

    begin_timing(ctx);
    bool late_mode = false;
    int64_t late_row_bytes = 0;                                           // bytes per survivor read from host memory
    for (int64_t k = 0; k < nchunks && s == MBC_OK; ++k) {
        const int b = (int)(k & 1);
        const int64_t row0 = chunks[k].row0;
        const int64_t n = chunks[k].n;
        if (n <= 0) break;
        mbc_table* st = stage[b];
        if (k >= 2) cudaStreamWaitEvent(ctx->copy_stream, ev_done[b], 0);    // staging buffer is free again
        for (int c = 0; c < ncols && s == MBC_OK; ++c) {
            if (!used[c] || (late_mode && late_ok[c])) continue;
            const Column& col = st->cols[c];
            const char* src = (const char*)host_cols[c] + (size_t)row0 * col.width;
            cudaError_t e = col.stride == col.width
                ? cudaMemcpyAsync(col.d, src, (size_t)n * col.width, cudaMemcpyHostToDevice, ctx->copy_stream)
                : cudaMemcpy2DAsync(col.d, col.stride, src, col.width, col.width, (size_t)n, cudaMemcpyHostToDevice, ctx->copy_stream);
            if (e != cudaSuccess) { set_error("H2D chunk %lld col %d: %s", (long long)k, c, cudaGetErrorString(e)); s = MBC_ERR_CUDA; }
            ctx->h2d_bytes += n * col.width;
        }
        if (s != MBC_OK) break;
        cudaEventRecord(ev_up[b], ctx->copy_stream);
        cudaStreamWaitEvent(ctx->stream, ev_up[b], 0);
        st->nrows = n;
        st->pos_base = position_base + row0;
        bind_table(&job, st);
        job.fused_off = late_mode;
        job.staged_off = late_mode;                                       // whole-tile loads would pull every row over PCIe
        if (late_mode) {                                                  // survivors of these columns come from host memory
            ScanParams& p = job.p;
            for (int c = 0; c < p.nproj; ++c)
                if (late_ok[p.proj[c].col]) p.proj[c].src = host_dev[p.proj[c].col] + (size_t)row0 * p.proj[c].stride;
            for (int a = 0; a < p.nagg; ++a)
                if (p.aggs[a].col >= 0 && late_ok[p.aggs[a].col]) p.aggs[a].src = host_dev[p.aggs[a].col] + (size_t)row0 * 4;
        }
        s = launch_job(&job, k == 0);
        job.pdl_tail = false;                                             // copies and events follow the kernels of a chunk
        if (h_counts && s == MBC_OK &&
            cudaMemcpyAsync(&h_counts[k], job.count_slot(), 8, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) s = MBC_ERR_CUDA;
        cudaEventRecord(ev_done[b], ctx->stream);
        if (k == 0 && any_late && s == MBC_OK) {                          // the sample decides: late when <= 1/5 of the rows qualify
            // (measured on B200 / PCIe 5: 100 M C2 rows take 17.6 / 33.4 / 80 ms late vs 52 / 52 / 57 ms uploaded at 1 / 10 / 50 %)
            if (cudaEventSynchronize(ev_done[0]) != cudaSuccess) { set_error("sample chunk failed"); s = MBC_ERR_CUDA; break; }
            const char* div = getenv("MBC_LATE_DIV");                    // tuning probe
            late_mode = h_counts[0] * (div ? atoll(div) : 5) <= n;
            if (late_mode)
                for (int c = 0; c < ncols; ++c)
                    if (used[c] && late_ok[c]) late_row_bytes += cols[c].width;
        }
        // chunk k is queued; now that the copy engine is busy with it, hand chunk k-1's rows to the D2H stream
        if (stream_out && s == MBC_OK && k >= 1) s = drain(k - 1);
    }
    if (s == MBC_OK && stream_out) {
        s = finish_job_device(&job);
        if (s == MBC_OK) {
            if (out_cap >= 0 && !out_overflow && r->count <= out_cap) {
                s = copy_rows(copied, r->count);                          // the tail, then everything has landed
                if (s == MBC_OK && cudaStreamSynchronize(ctx->d2h_stream) != cudaSuccess) s = MBC_ERR_CUDA;
                if (s == MBC_OK && (rq.want & MBC_WANT_TUPLES)) {
                    const uint32_t keep = r->want;
                    r->want = MBC_WANT_TUPLES | MBC_WANT_HOST;            // only the tuple bytes are still missing
                    s = finish_result_host(r);
                    r->want = keep;
                }
            } else {
                cudaStreamSynchronize(ctx->d2h_stream);
                r->h_pos = nullptr;                                       // estimate exceeded: plain copy of the final result
                for (auto& c : r->cols) c.h = nullptr;
                s = finish_result_host(r);
            }
        }
    } else if (s == MBC_OK) {
        s = finish_job(&job);
    }
    cudaStreamSynchronize(ctx->copy_stream);
    cudaStreamSynchronize(ctx->d2h_stream);
    cudaStreamSynchronize(ctx->stream);
    cleanup();
    if (s != MBC_OK) { if (job.r) mbc_result_free(job.r); return s; }
    if (late_mode) ctx->h2d_bytes += (job.r->count - (h_counts ? h_counts[0] : 0)) * late_row_bytes;   // read in place over PCIe
    *out = job.r;
    return MBC_OK;
}

}  // namespace mbc

using namespace mbc;

extern "C" int32_t mbc_scan(mbc_table* t, const mbc_term* terms, int32_t nterms, const int32_t* proj_cols,
                            int32_t nproj, uint32_t want, const mbc_aggspec* aggs, int32_t nagg, mbc_result** out) {
    ScanRequest rq;
    rq.table = t;
    rq.terms = terms;
    rq.nterms = nterms;
    rq.proj_cols = proj_cols;
    rq.nproj = nproj;
    rq.want = want;
    rq.aggs = aggs;
    rq.nagg = nagg;
    rq.allow_deferred = true;
    return run_scan(rq, out);
}

extern "C" int32_t mbc_scan_host(mbc_ctx* ctx, int32_t ncols, const mbc_coldesc* cols, const void* const* host_cols,
                                 int64_t nrows, int64_t position_base, const mbc_term* terms, int32_t nterms,
                                 const int32_t* proj_cols, int32_t nproj, uint32_t want, const mbc_aggspec* aggs,
                                 int32_t nagg, mbc_result** out) {
    if (!ctx || !cols || !host_cols || !out || ncols <= 0 || nrows < 0) MBC_FAIL(MBC_ERR_ARG, "mbc_scan_host: bad argument");
    if (want & MBC_WANT_BITMAP) MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_scan_host: MBC_WANT_BITMAP needs a resident table");
    ScanRequest rq;
    rq.terms = terms;
    rq.nterms = nterms;
    rq.proj_cols = proj_cols;
    rq.nproj = nproj;
    rq.want = want;
    rq.aggs = aggs;
    rq.nagg = nagg;
    return run_scan_host(ctx, ncols, cols, host_cols, nrows, position_base, rq, out);
}
