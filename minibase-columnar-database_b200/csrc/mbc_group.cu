// mbc_group.cu -- GROUP BY key columns with COUNT / SUM / MIN / MAX per group over a filtered table (mbc_group_aggregate).
//
// Sort-based: the qualifying rows (run_scan) are stably sorted by the key columns with mbc_sort's radix passes, so each
// group is one run of the sorted order and its rows keep ascending position order.  Head flags mark where the key
// tuple changes, an exclusive scan numbers the groups, and a segmented reduction folds each run.
//
// The segmented reduction is deterministic: every CTA owns a fixed 4096-element chunk of the sorted order, each thread
// folds 16 consecutive elements in order, and a segmented scan over the threads (a fixed tree) joins the runs that cross
// thread boundaries.  A run that starts and ends inside the chunk is written directly; a group that crosses a chunk
// boundary leaves two partials per chunk (the chunk's first and last run), which group_straddle_kernel folds in chunk
// order with a fixed tree.  So every association depends on the data and the geometry alone, real SUMs included, and
// neither one giant group nor millions of singletons serialise the work.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include <vector>

#include "mbc_internal.cuh"

namespace mbc {

constexpr int kGroupThreads = 256;
constexpr int kGroupItems = 16;
constexpr int kGroupChunk = kGroupThreads * kGroupItems;     // 4096 sorted elements per CTA

struct GroupKeys {
    const void* d[kMaxTerms];
    int32_t stride[kMaxTerms];
    int32_t type[kMaxTerms];
    int32_t n;
};

struct GroupAggs {
    const void* src[kMaxAgg];
    int32_t kind[kMaxAgg];
    int32_t type[kMaxAgg];     // column type; MBC_ATTR_INTEGER for COUNT
    int32_t n;
    int32_t partials;          // every src holds 8-byte raw aggregates (int64, or double for a real SUM / MIN / MAX)
};

// head[i] = 1 where sorted row rows[i] starts a group: some key differs from that of rows[i-1].  Reals compare as floats,
// so -0.0 and +0.0 (which the sort places next to each other) are one key; ints and strings compare their bytes.
__global__ void __launch_bounds__(256) group_heads_kernel(const uint32_t* __restrict__ rows, int64_t n, GroupKeys keys,
                                                          uint32_t* __restrict__ head) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        uint32_t h = 1;
        if (i > 0) {
            h = 0;
            const uint32_t ra = rows[i], rb = rows[i - 1];
            for (int k = 0; k < keys.n && !h; ++k) {
                const char* base = reinterpret_cast<const char*>(keys.d[k]);
                const uint32_t* a = reinterpret_cast<const uint32_t*>(base + (size_t)ra * keys.stride[k]);
                const uint32_t* b = reinterpret_cast<const uint32_t*>(base + (size_t)rb * keys.stride[k]);
                if (keys.type[k] == MBC_ATTR_REAL) h = __uint_as_float(a[0]) != __uint_as_float(b[0]);
                else
                    for (int w = 0; w < (keys.stride[k] >> 2); ++w) h |= a[w] != b[w];
            }
        }
        head[i] = h;
    }
}

// ---- segmented fold ---------------------------------------------------------------------------------------------
enum { kOpAdd = 0, kOpMin = 1, kOpMax = 2 };
enum { kSrcOne = 0, kSrcInt = 1, kSrcReal = 2, kSrcPartial = 3 };

template <typename T, int OP> __device__ __forceinline__ T fold_identity() {
    using L = std::numeric_limits<T>;
    if (OP == kOpAdd) return (T)0;
    if (OP == kOpMin) return L::has_infinity ? L::infinity() : L::max();
    return L::has_infinity ? -L::infinity() : L::lowest();
}
template <typename T, int OP> __device__ __forceinline__ T fold_op(T a, T b) {
    if (OP == kOpAdd) return a + b;
    if (OP == kOpMin) return b < a ? b : a;
    return b > a ? b : a;
}
template <typename T, int SRC> __device__ __forceinline__ T fold_load(const void* src, uint32_t row) {
    if (SRC == kSrcOne) return (T)1;
    if (SRC == kSrcInt) return (T)__ldg(reinterpret_cast<const int32_t*>(src) + row);
    if (SRC == kSrcPartial) return __ldg(reinterpret_cast<const T*>(src) + row);   // a COUNT partial is an int64 to add
    return (T)__ldg(reinterpret_cast<const float*>(src) + row);
}
template <typename T> __device__ __forceinline__ unsigned long long fold_raw(T v) {
    unsigned long long r;
    memcpy(&r, &v, 8);
    return r;
}
template <typename T> __device__ __forceinline__ T fold_from_raw(unsigned long long r) {
    T v;
    memcpy(&v, &r, 8);
    return v;
}

// The elements one thread of group_fold_kernel owns, loaded once for every aggregate.
struct FoldThread {
    uint32_t rows[kGroupItems];
    uint32_t heads;        // bit j: element base + j starts a group
    int nv;                // valid elements (< kGroupItems only in the last chunk)
    bool next_head;        // the element after the thread's last one starts a group or does not exist
    unsigned long long g0; // group of the thread's first element
};

// One aggregate over one chunk.  out[g] for groups inside the chunk, parts[2 * chunk + {0, 1}] = the chunk's first run
// (when its group started in an earlier chunk) and its last run (when its group goes on into the next chunk).
template <typename T, int OP, int SRC>
__device__ void fold_chunk(const FoldThread& ft, const void* src, unsigned long long* __restrict__ out,
                           unsigned long long* __restrict__ parts, int* s_flag, T* s_val) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // 1. in order over the thread's elements: runs that start and end inside the thread are final
    T acc = fold_identity<T, OP>(), first = acc;
    bool first_closed = false;
    unsigned long long g = ft.g0;
#pragma unroll
    for (int j = 0; j < kGroupItems; ++j) {
        if (j < ft.nv) {
            if (j > 0 && ((ft.heads >> j) & 1u)) {
                if (!first_closed) { first = acc; first_closed = true; }
                else out[g] = fold_raw(acc);
                acc = fold_identity<T, OP>();
                ++g;
            }
            acc = fold_op<T, OP>(acc, fold_load<T, SRC>(src, ft.rows[j]));
        }
    }
    // 2. segmented inclusive scan of (thread has a head, its last run's partial) over the CTA: a fixed tree
    int f = ft.heads != 0;
    T v = acc;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int f2 = __shfl_up_sync(0xFFFFFFFFu, f, d);
        const T v2 = __shfl_up_sync(0xFFFFFFFFu, v, d);
        if (lane >= d) {
            if (!f) v = fold_op<T, OP>(v2, v);
            f |= f2;
        }
    }
    __syncthreads();                                              // the previous aggregate's readers are done
    if (lane == 31) { s_flag[warp] = f; s_val[warp] = v; }
    __syncthreads();
    int wf = 0;
    T wv = fold_identity<T, OP>();
    for (int w = 0; w < warp; ++w) {                              // prefix of the earlier warps, in warp order
        if (s_flag[w]) { wv = s_val[w]; wf = 1; }
        else wv = fold_op<T, OP>(wv, s_val[w]);
    }
    if (!f) v = fold_op<T, OP>(wv, v);
    f |= wf;
    // exclusive value: the inclusive value of the thread before
    int ef = __shfl_up_sync(0xFFFFFFFFu, f, 1);
    T ev = __shfl_up_sync(0xFFFFFFFFu, v, 1);
    if (lane == 0) { ef = wf; ev = wv; }
    if (ft.nv == 0) return;
    const unsigned long long chunk = blockIdx.x;
    // 3. the thread's first run, when it ends inside the thread
    if (first_closed) {
        const bool own_start = ft.heads & 1u;
        const T val = own_start ? first : fold_op<T, OP>(ev, first);
        if (!own_start && !ef) parts[2 * chunk] = fold_raw(val);   // began in an earlier chunk
        else out[ft.g0] = fold_raw(val);
    }
    // 4. the thread's last run, when it ends with the thread (or the chunk)
    if (ft.next_head || tid == kGroupThreads - 1) {
        if (!ft.next_head) parts[2 * chunk + 1] = fold_raw(v);    // goes on into the next chunk
        if (!f) parts[2 * chunk] = fold_raw(v);                   // began in an earlier chunk
        else if (ft.next_head) out[g] = fold_raw(v);
    }
}

template <typename T, int OP, int SRC>
__device__ __forceinline__ void fold_chunk_smem(const FoldThread& ft, const void* src, bool partial, unsigned long long* out,
                                                unsigned long long* parts, int* s_flag, unsigned long long* s_raw) {
    if (partial) fold_chunk<T, OP, kSrcPartial>(ft, src, out, parts, s_flag, reinterpret_cast<T*>(s_raw));
    else fold_chunk<T, OP, SRC>(ft, src, out, parts, s_flag, reinterpret_cast<T*>(s_raw));
}

// aggregate a of the groups: out[a * G + g] raw (int64, or the bits of a double for a real SUM / MIN / MAX)
__global__ void __launch_bounds__(kGroupThreads) group_fold_kernel(const uint32_t* __restrict__ rows, const uint32_t* __restrict__ head,
                                                                   const unsigned long long* __restrict__ group_of, int64_t n,
                                                                   GroupAggs aggs, unsigned long long* __restrict__ out, int64_t G,
                                                                   unsigned long long* __restrict__ parts, int64_t nchunks) {
    __shared__ int s_flag[kGroupThreads / 32];
    __shared__ unsigned long long s_raw[kGroupThreads / 32];
    FoldThread ft;
    const int64_t base = (int64_t)blockIdx.x * kGroupChunk + (int64_t)threadIdx.x * kGroupItems;
    ft.nv = (int)std::max<int64_t>(0, std::min<int64_t>(kGroupItems, n - base));
    ft.heads = 0;
    if (ft.nv == kGroupItems) {
        const uint4* r4 = reinterpret_cast<const uint4*>(rows + base);
        const uint4* h4 = reinterpret_cast<const uint4*>(head + base);
#pragma unroll
        for (int q = 0; q < kGroupItems / 4; ++q) {
            const uint4 r = r4[q], h = h4[q];
            ft.rows[4 * q] = r.x; ft.rows[4 * q + 1] = r.y; ft.rows[4 * q + 2] = r.z; ft.rows[4 * q + 3] = r.w;
            ft.heads |= ((h.x & 1u) | (h.y & 1u) << 1 | (h.z & 1u) << 2 | (h.w & 1u) << 3) << (4 * q);
        }
    } else {
#pragma unroll
        for (int j = 0; j < kGroupItems; ++j) {
            ft.rows[j] = j < ft.nv ? rows[base + j] : 0u;
            if (j < ft.nv && head[base + j]) ft.heads |= 1u << j;
        }
    }
    const int64_t e = base + ft.nv;
    ft.next_head = e >= n || head[e] != 0;
    ft.g0 = ft.nv > 0 ? group_of[base + 1] - 1 : 0;               // heads in [0, base] minus one
    unsigned long long* cparts = parts;
    for (int a = 0; a < aggs.n; ++a) {
        unsigned long long* o = out + (size_t)a * G;
        unsigned long long* p = cparts + (size_t)a * 2 * nchunks;
        const void* src = aggs.src[a];
        const bool real = aggs.type[a] == MBC_ATTR_REAL, pt = aggs.partials != 0;
        switch (aggs.kind[a]) {
            case MBC_AGG_COUNT: fold_chunk_smem<long long, kOpAdd, kSrcOne>(ft, src, pt, o, p, s_flag, s_raw); break;
            case MBC_AGG_SUM:
                if (real) fold_chunk_smem<double, kOpAdd, kSrcReal>(ft, src, pt, o, p, s_flag, s_raw);
                else fold_chunk_smem<long long, kOpAdd, kSrcInt>(ft, src, pt, o, p, s_flag, s_raw);
                break;
            case MBC_AGG_MIN:
                if (real) fold_chunk_smem<double, kOpMin, kSrcReal>(ft, src, pt, o, p, s_flag, s_raw);
                else fold_chunk_smem<long long, kOpMin, kSrcInt>(ft, src, pt, o, p, s_flag, s_raw);
                break;
            default:
                if (real) fold_chunk_smem<double, kOpMax, kSrcReal>(ft, src, pt, o, p, s_flag, s_raw);
                else fold_chunk_smem<long long, kOpMax, kSrcInt>(ft, src, pt, o, p, s_flag, s_raw);
                break;
        }
    }
}

// Fold the partials of a group that crosses chunk boundaries: its last run in chunk ca, then the first runs of chunks
// ca+1 .. cb, in that order.  Thread t folds a contiguous slice, then a fixed tree joins the slices.
template <typename T, int OP>
__device__ void straddle_fold(const unsigned long long* __restrict__ parts, int64_t ca, int64_t m, unsigned long long* out_g,
                              T* s_val) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t per = (m + kGroupThreads - 1) / kGroupThreads;
    T acc = fold_identity<T, OP>();
    for (int64_t k = (int64_t)tid * per; k < std::min<int64_t>(m, (int64_t)(tid + 1) * per); ++k)
        acc = fold_op<T, OP>(acc, fold_from_raw<T>(parts[2 * (ca + k) + (k == 0 ? 1 : 0)]));
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const T o = __shfl_down_sync(0xFFFFFFFFu, acc, d);
        if ((lane & (2 * d - 1)) == 0) acc = fold_op<T, OP>(acc, o);
    }
    __syncthreads();
    if (lane == 0) s_val[warp] = acc;
    __syncthreads();
    if (tid == 0) {
        T r = s_val[0];
        for (int w = 1; w < kGroupThreads / 32; ++w) r = fold_op<T, OP>(r, s_val[w]);
        *out_g = fold_raw(r);
    }
}

// CTA c owns the group that crosses the end of chunk c when that group starts in chunk c
__global__ void __launch_bounds__(kGroupThreads) group_straddle_kernel(const uint32_t* __restrict__ head,
                                                                       const unsigned long long* __restrict__ group_of,
                                                                       const uint32_t* __restrict__ start, int64_t n, GroupAggs aggs,
                                                                       unsigned long long* __restrict__ out, int64_t G,
                                                                       const unsigned long long* __restrict__ parts, int64_t nchunks) {
    __shared__ unsigned long long s_raw[kGroupThreads / 32];
    const int64_t ca = blockIdx.x;
    const int64_t c1 = (ca + 1) * kGroupChunk;
    if (c1 >= n || head[c1]) return;
    const unsigned long long g = group_of[c1] - 1;
    if ((int64_t)start[g] < ca * kGroupChunk) return;            // an earlier chunk owns it
    const int64_t end = g + 1 < (unsigned long long)G ? (int64_t)start[g + 1] : n;
    const int64_t m = (end - 1) / kGroupChunk - ca + 1;           // chunks the group touches
    for (int a = 0; a < aggs.n; ++a) {
        const unsigned long long* p = parts + (size_t)a * 2 * nchunks;
        unsigned long long* o = out + (size_t)a * G + g;
        const bool real = aggs.type[a] == MBC_ATTR_REAL;
        switch (aggs.kind[a]) {
            case MBC_AGG_COUNT: straddle_fold<long long, kOpAdd>(p, ca, m, o, reinterpret_cast<long long*>(s_raw)); break;
            case MBC_AGG_SUM:
                if (real) straddle_fold<double, kOpAdd>(p, ca, m, o, reinterpret_cast<double*>(s_raw));
                else straddle_fold<long long, kOpAdd>(p, ca, m, o, reinterpret_cast<long long*>(s_raw));
                break;
            case MBC_AGG_MIN:
                if (real) straddle_fold<double, kOpMin>(p, ca, m, o, reinterpret_cast<double*>(s_raw));
                else straddle_fold<long long, kOpMin>(p, ca, m, o, reinterpret_cast<long long*>(s_raw));
                break;
            default:
                if (real) straddle_fold<double, kOpMax>(p, ca, m, o, reinterpret_cast<double*>(s_raw));
                else straddle_fold<long long, kOpMax>(p, ca, m, o, reinterpret_cast<long long*>(s_raw));
                break;
        }
    }
}

static int grid_for(const mbc_ctx* ctx, int64_t n) {
    return (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8));
}

int32_t group_rows(mbc_ctx* ctx, uint32_t* rows, int64_t n, const Column* keys, int32_t nkeys, const GroupAggSpec* aggs, int32_t nagg,
                   bool partials, const int64_t* pos, int64_t pos_base, mbc_result* r) {
    const uint32_t want = r->want;
    GroupKeys gk{};
    gk.n = nkeys;
    for (int k = 0; k < nkeys; ++k) {
        gk.d[k] = keys[k].d;
        gk.stride[k] = keys[k].stride;
        gk.type[k] = keys[k].type;
    }
    GroupAggs ga{};
    ga.n = (want & MBC_WANT_AGG) ? nagg : 0;
    ga.partials = partials ? 1 : 0;
    for (int a = 0; a < ga.n; ++a) {
        ga.src[a] = aggs[a].src;
        ga.kind[a] = aggs[a].kind;
        ga.type[a] = aggs[a].type;
    }
    r->kind = mbc_result::kGrouped;
    r->group_nagg = ga.n;
    uint32_t *head = nullptr, *bits = nullptr, *start = nullptr, *head_row = nullptr;
    unsigned long long *group_of = nullptr, *parts = nullptr;
    auto release = [&]() {
        for (void* p : {(void*)head, (void*)bits, (void*)start, (void*)head_row, (void*)group_of, (void*)parts}) dev_free(ctx, p);
    };
    auto fail = [&](int32_t s) {
        release();
        return s;
    };
#define GTRY(x) do { int32_t _s = (x); if (_s != MBC_OK) return fail(_s); } while (0)
#define GCUDA(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) return fail((set_error("group: %s", cudaGetErrorString(_e)), MBC_ERR_CUDA)); } while (0)
    const int grid = grid_for(ctx, n);
    GTRY(dev_alloc(ctx, (void**)&group_of, (size_t)(n + 1) * 8, false));
    if (n > 0) {
        GTRY(dev_alloc(ctx, (void**)&head, (size_t)n * 4, false));            // sort keys, then the head flags
        GTRY(dev_alloc(ctx, (void**)&bits, 8, false));
        for (int k = nkeys - 1; k >= 0; --k) GTRY(sort_rows_by_column(ctx, rows, n, keys[k], false, head, bits));
        group_heads_kernel<<<grid, 256, 0, ctx->stream>>>(rows, n, gk, head);
        ctx->launches++;
    }
    GTRY(exclusive_scan_u32(ctx, head, n, group_of));
    unsigned long long G = 0;
    GCUDA(cudaMemcpyAsync(&G, group_of + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    GCUDA(cudaStreamSynchronize(ctx->stream));
    r->count = (int64_t)G;
    r->capacity = (int64_t)G;
    if (G > 0) {
        GTRY(dev_alloc(ctx, (void**)&start, (size_t)G * 4, false));
        GTRY(dev_alloc(ctx, (void**)&head_row, (size_t)G * 4, false));
        sparse_run_starts_kernel<<<grid, 256, 0, ctx->stream>>>(head, group_of, rows, n, start, head_row);
        ctx->launches++;
    }
    // a group's head row is its first row id: the sort is stable over row ids in position order
    if ((want & MBC_WANT_POSITIONS) && G > 0) {
        GTRY(dev_alloc(ctx, (void**)&r->d_pos, (size_t)G * 8, false));
        if (pos) sort_gather_kernel<<<grid_for(ctx, (int64_t)G), 256, 0, ctx->stream>>>(head_row, (int64_t)G, pos, 8, r->d_pos);
        else sort_positions_kernel<<<grid_for(ctx, (int64_t)G), 256, 0, ctx->stream>>>(head_row, (int64_t)G, pos_base, r->d_pos);
        ctx->launches++;
    }
    if (want & MBC_WANT_COLUMNS) {
        for (int k = 0; k < nkeys; ++k) {
            const Column& col = keys[k];
            mbc_result::Col rc{col.type, col.width, col.stride, nullptr, nullptr};
            GTRY(dev_alloc(ctx, &rc.d, (size_t)std::max<unsigned long long>(G, 1) * col.stride, false));
            r->cols.push_back(rc);
            if (G > 0) {
                sort_gather_kernel<<<grid_for(ctx, (int64_t)G), 256, 0, ctx->stream>>>(head_row, (int64_t)G, col.d, col.stride, rc.d);
                ctx->launches++;
            }
        }
    }
    if (ga.n > 0) {
        const int64_t nchunks = (n + kGroupChunk - 1) / kGroupChunk;
        GTRY(dev_alloc(ctx, (void**)&r->d_aggs, (size_t)std::max<unsigned long long>(G, 1) * ga.n * 8, false));
        if (G > 0) {
            GTRY(dev_alloc(ctx, (void**)&parts, (size_t)nchunks * 2 * ga.n * 8, false));
            group_fold_kernel<<<(unsigned)nchunks, kGroupThreads, 0, ctx->stream>>>(rows, head, group_of, n, ga, (unsigned long long*)r->d_aggs, (int64_t)G,
                                                                                   parts, nchunks);
            ctx->launches++;
            if (nchunks > 1) {
                group_straddle_kernel<<<(unsigned)(nchunks - 1), kGroupThreads, 0, ctx->stream>>>(head, group_of, start, n, ga, (unsigned long long*)r->d_aggs,
                                                                                                  (int64_t)G, parts, nchunks);
                ctx->launches++;
            }
        }
    }
    end_timing(ctx);
    GCUDA(cudaGetLastError());
    GTRY(finish_result_host(r));
    if ((want & MBC_WANT_HOST) && ga.n > 0) {
        std::vector<unsigned long long> raw((size_t)G * ga.n);
        if (G > 0) GCUDA(cudaMemcpyAsync(raw.data(), r->d_aggs, raw.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
        GCUDA(cudaStreamSynchronize(ctx->stream));
        r->group_aggs.resize(ga.n);
        for (int a = 0; a < ga.n; ++a) {
            mbc_result::GroupAgg& ag = r->group_aggs[a];
            ag.i.resize(G);
            ag.f.resize(G);
            for (unsigned long long g = 0; g < G; ++g) {
                int32_t valid;
                agg_from_raw(ga.kind[a], ga.type[a], raw[(size_t)a * G + g], true, &ag.i[g], &ag.f[g], &valid);
            }
        }
    }
    GCUDA(cudaStreamSynchronize(ctx->stream));
#undef GTRY
#undef GCUDA
    release();
    return MBC_OK;
}

}  // namespace mbc

using namespace mbc;

extern "C" int32_t mbc_group_aggregate(mbc_table* t, const mbc_term* terms, int32_t nterms, const int32_t* key_cols, int32_t nkeys,
                                       const mbc_aggspec* aggs, int32_t nagg, uint32_t want, mbc_result** out) {
    if (!t || !out || !key_cols || nkeys <= 0 || (nagg > 0 && !aggs) || nagg < 0)
        MBC_FAIL(MBC_ERR_ARG, "mbc_group_aggregate: bad argument");
    *out = nullptr;
    if (want & (MBC_WANT_TUPLES | MBC_WANT_BITMAP))
        MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_group_aggregate: MBC_WANT_TUPLES / MBC_WANT_BITMAP are not available for groups");
    if (nkeys > kMaxTerms) MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_group_aggregate: %d key columns (max %d)", nkeys, kMaxTerms);
    if (nagg > kMaxAgg) MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_group_aggregate: %d aggregates (max %d)", nagg, kMaxAgg);
    Column keys[kMaxTerms];
    for (int k = 0; k < nkeys; ++k) {
        if (key_cols[k] < 0 || key_cols[k] >= (int)t->cols.size())
            MBC_FAIL(MBC_ERR_ARG, "mbc_group_aggregate: key column %d out of range", key_cols[k]);
        keys[k] = t->cols[key_cols[k]];
    }
    GroupAggSpec specs[kMaxAgg] = {};
    for (int a = 0; a < nagg; ++a) {
        const int kind = aggs[a].kind, col = aggs[a].col;
        if (kind < MBC_AGG_COUNT || kind > MBC_AGG_MAX) MBC_FAIL(MBC_ERR_ARG, "mbc_group_aggregate: aggregate %d: unknown kind %d", a, kind);
        specs[a].kind = kind;
        specs[a].type = MBC_ATTR_INTEGER;
        if (kind == MBC_AGG_COUNT) continue;
        if (col < 0 || col >= (int)t->cols.size()) MBC_FAIL(MBC_ERR_ARG, "mbc_group_aggregate: aggregate %d: column %d out of range", a, col);
        if (t->cols[col].type == MBC_ATTR_STRING) MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_group_aggregate: aggregate %d over a string column", a);
        specs[a].src = t->cols[col].d;
        specs[a].type = t->cols[col].type;
    }
    if (t->nrows > (int64_t)UINT32_MAX) MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_group_aggregate: more than 2^32 rows in one table");
    mbc_ctx* ctx = t->ctx;
    MBC_CUDA(cudaSetDevice(ctx->device));

    // the qualifying rows in position order (the predicate checks its terms)
    mbc_result* sel = nullptr;
    ScanRequest rq;
    rq.table = t;
    rq.terms = terms;
    rq.nterms = nterms;
    rq.want = MBC_WANT_POSITIONS;
    MBC_TRY(run_scan(rq, &sel));
    const int64_t n = sel->count;
    split_timing(ctx);                                      // the scan's kernels count, the host wait in between does not
    begin_timing(ctx);

    mbc_result* r = new mbc_result();
    r->ctx = ctx;
    ctx_retain(ctx);
    r->want = want;
    r->nrows = t->nrows;
    uint32_t* rows = nullptr;
    int32_t s = dev_alloc(ctx, (void**)&rows, (size_t)std::max<int64_t>(n, 1) * 4, false);
    if (s == MBC_OK && n > 0) {
        sort_rows_from_positions_kernel<<<grid_for(ctx, n), 256, 0, ctx->stream>>>(sel->d_pos, n, t->pos_base, rows);
        ctx->launches++;
    }
    if (s == MBC_OK) s = group_rows(ctx, rows, n, keys, nkeys, specs, nagg, false, nullptr, t->pos_base, r);
    dev_free(ctx, rows);
    mbc_result_free(sel);
    if (s != MBC_OK) {
        mbc_result_free(r);
        return s;
    }
    *out = r;
    return MBC_OK;
}
