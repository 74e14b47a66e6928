// mbc_internal.cuh -- shared declarations of libmbcol.so (host side + device helpers).
// Nothing here is part of the ABI; the ABI is include/mbcol.h.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/mbcol.h"

namespace mbc {

// ---- geometry of the scan engine --------------------------------------------------------
// A warp owns 512 consecutive rows = 4 "units" of 128 rows; in unit u lane l owns rows
// u*128 + l*4 + {0..3}, i.e. exactly one 128-bit load of a 4-byte column.  A 256-thread CTA
// (8 warps) owns a 4096-row tile.  Every column allocation is padded to a whole tile so the
// vector loads of the last tile stay in bounds; rows >= nrows are masked off.
#ifndef MBC_WORKER_WARPS
#define MBC_WORKER_WARPS 8
#endif
constexpr int kWarpsPerCta   = MBC_WORKER_WARPS;          // worker warps of a scan CTA (+1 scan warp)
constexpr int kScanThreads   = kWarpsPerCta * 32;
constexpr int kVec           = 4;
constexpr int kUnits         = 4;
constexpr int kRowsPerThread = kVec * kUnits;              // 16
constexpr int kUnitRows      = 32 * kVec;                  // 128
constexpr int kWarpRows      = kUnitRows * kUnits;         // 512
constexpr int kTileRows      = kWarpRows * kWarpsPerCta;   // 4096
constexpr int kPadRows       = 8192;                       // row padding of every column / bitmap

constexpr int kMaxTerms = 16;
constexpr int kMaxProj  = 16;
constexpr int kMaxAgg   = 8;
constexpr int kMaxLit   = 64;     // widest string literal / string column in a predicate
constexpr int kMaxStrStride = 256; // widest device string row

static inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

// as_i64 of a real aggregate, with Java's (long) d semantics: truncated toward zero, saturated to INT64_MIN / INT64_MAX
// out of range (±inf included), 0 for NaN.  A plain (int64_t) cast of such a double (MAX over FLT_MAX) is undefined.
static inline int64_t real_agg_as_i64(double d) {
    if (d != d) return 0;
    if (d >= 9223372036854775808.0) return INT64_MAX;    // 2^63
    if (d < -9223372036854775808.0) return INT64_MIN;
    return (int64_t)d;
}

// device row stride of a char(width) column: multiples of 4 below 16, multiples of 16 above,
// so every row is reachable with aligned 32-bit or 128-bit loads.  Padding bytes are zero.
static inline int str_stride(int width) {
    if (width <= 0) return 4;
    if (width < 16) return (int)round_up(width, 4);
    return (int)round_up(width, 16);
}

void set_error(const char* fmt, ...);

#define MBC_CUDA(call)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (call);                                                             \
        if (_e != cudaSuccess) {                                                             \
            mbc::set_error("CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__,    \
                           __LINE__, cudaGetErrorString(_e));                                \
            return MBC_ERR_CUDA;                                                             \
        }                                                                                    \
    } while (0)

#define MBC_TRY(call)                      \
    do {                                   \
        int32_t _s = (call);               \
        if (_s != MBC_OK) return _s;       \
    } while (0)

#define MBC_FAIL(code, ...)                \
    do {                                   \
        mbc::set_error(__VA_ARGS__);       \
        return (code);                     \
    } while (0)

struct Column {
    int32_t type   = 0;       // MBC_ATTR_*
    int32_t width  = 0;       // payload bytes (4, or strSize)
    int32_t stride = 0;       // device row stride (4, or str_stride(width))
    void*   d      = nullptr; // nrows_pad * stride bytes, zero padded
};

struct BitmapIndex {
    bool     exists = false;
    int64_t  nvalues = 0;
    std::vector<int32_t> ivals;    // sorted distinct values (int columns)
    std::vector<uint8_t> svals;    // sorted distinct values, nvalues*width bytes (string columns)
    // chunk-major storage: [chunk][value][chunk_rows/32] uint32 words (bit p of a value's bitmap = word p/32, bit p%32).
    // A build CTA writes one fully contiguous block per chunk; a scan reads a value's bitmap as chunk_rows/8-byte pieces.
    uint32_t* d_words = nullptr;
    int32_t   chunk_rows = 0;      // rows per chunk (power of two, 1024..8192)
    uint32_t* d_ids   = nullptr;   // per-row dense value id (kept for the join's low-cardinality path)
    // sparse layout (value-sorted position lists), built where the per-value bitsets above cannot be (mbc_bitmap.cu):
    // value v's rows are d_rows[offsets[v] .. offsets[v+1]), ascending.  The offsets stay on the host: every reader (the
    // scan's binary search and row counts, mbc_bitmap_get) needs them there, and no kernel reads them.
    bool      sparse = false;
    uint32_t* d_rows = nullptr;    // n_indexed local row ids ordered by (value id, row)
    uint32_t* d_indexed = nullptr; // words_pad words: the rows that were live when the index was built
    int64_t   n_indexed = 0;
    std::vector<uint32_t> offsets; // nvalues + 1
};

}  // namespace mbc

struct mbc_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;       // where kernels go (own_stream unless mbc_set_stream)
    cudaStream_t copy_stream = nullptr;  // H2D staging of mbc_scan_host
    cudaStream_t d2h_stream = nullptr;   // results of mbc_scan_host streaming back while later chunks upload
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    int64_t launches = 0;
    bool filter_smem_set = false, sort_smem_set = false, staged_smem_set = false;   // per-device opt-in to > 48 KB of dynamic shared memory
    // single-residency scan (mbc_scan_fused.cuh): published tile counts, tagged with the launch epoch so the buffer is
    // never cleared between launches (zeroed when it is allocated and when the 20-bit epoch wraps)
    uint32_t* fused_flags = nullptr;
    int64_t   fused_flags_cap = 0;
    uint32_t  fused_epoch = 0;
    int       fused_smem_budget = -1;    // dynamic shared memory the fused kernel may use (-1: not probed, 0: unusable)
    int64_t h2d_bytes = 0;            // host -> device bytes moved by mbc_scan_host (copies + rows read in place)
    // tables, results and shards alive on this context: mbc_shutdown with live objects only marks the context, the last
    // free destroys it (a handle closed after its context must not touch freed memory)
    int64_t live_objects = 0;
    bool shutdown_pending = false;
    float last_ms = 0.f;
    bool timing_split = false;
    float extra_ms = 0.f;                // device time of earlier timed segments of the same call
    // per-context scan workspace (tile status words, ticket, partials), grown on demand
    void*   ws = nullptr;
    size_t  ws_bytes = 0;
    // pinned host blocks recycled between results
    struct PinnedBlock { void* p; size_t bytes; };
    std::vector<PinnedBlock> pinned_free;
    std::vector<cudaEvent_t> event_free;  // recycled timing / completion events
};

struct mbc_table {
    mbc_ctx* ctx = nullptr;
    int64_t nrows = 0;
    int64_t nrows_pad = 0;      // multiple of kTileRows
    int64_t pos_base = 0;
    int64_t words_pad = 0;      // uint32 words per bitmap (nrows_pad/32)
    std::vector<mbc::Column> cols;
    std::vector<mbc::BitmapIndex> bm;
    uint32_t* d_deleted = nullptr;
    bool has_deleted = false;
};

struct mbc_result {
    // what the buffers hold, set by the call that made the result (mbc_shard_gather carries each kind differently)
    enum Kind : int32_t {
        kUnset = 0,
        kScan,      // mbc_scan / mbc_scan_host / mbc_bitmap_scan: d_aggs = kMaxAgg raw aggregates + the count
        kRows,      // mbc_sort / mbc_topk / mbc_shard_topk: positions + fields in sort order, no d_aggs
        kGrouped,   // mbc_group_aggregate / mbc_shard_group: one row per group, d_aggs = nagg x count raw values
        kJoin,      // mbc_bitmap_join: position pairs
    };
    Kind kind = kUnset;
    mbc_ctx* ctx = nullptr;
    uint32_t want = 0;
    int64_t count = 0;
    int64_t capacity = 0;        // rows the device buffers can hold
    int64_t nrows = 0;           // rows scanned (bitmap length)
    // device
    int64_t* d_pos = nullptr;
    int64_t* d_pos2 = nullptr;
    struct Col { int32_t type, width, stride; void* d; void* h; };
    std::vector<Col> cols;
    uint32_t* d_bitmap = nullptr;
    int64_t   bitmap_words32 = 0;
    uint64_t* d_aggs = nullptr;  // nagg raw 8-byte values followed by the count
    uint8_t*  d_tuples = nullptr;
    int32_t   tuple_len = 0;
    // host (pinned, from the ctx pool)
    int64_t* h_pos = nullptr;
    int64_t* h_pos2 = nullptr;
    uint64_t* h_bitmap = nullptr;
    uint8_t* h_tuples = nullptr;
    std::vector<std::pair<void*, size_t>> pinned;  // blocks to give back
    // aggregates
    struct Agg { int32_t kind, type; int64_t i; double f; int32_t valid; };
    std::vector<Agg> aggs;
    // kGrouped: d_aggs holds group_nagg x count raw values, group_aggs their host decode
    int32_t group_nagg = 0;
    struct GroupAgg { std::vector<int64_t> i; std::vector<double> f; };
    std::vector<GroupAgg> group_aggs;
    // Deferred completion (device-resident results of mbc_scan): the call returns with its kernels and the small
    // count/aggregate copy queued; the first accessor that needs the count waits on ev_ready.  Back-to-back scans
    // then run without host gaps between them.
    cudaEvent_t ev_ready = nullptr;        // non-null while count/aggs are still in flight
    cudaEvent_t ev_done = nullptr;         // the result's device buffers (rows, count, aggregates) are complete (kept until free)
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;   // device time of this result's kernels
    cudaEvent_t ev_mid[3] = {nullptr, nullptr, nullptr};   // resident scans: after pass 1, after the offsets, after the write pass
    float phase_ms[4] = {-1.f, -1.f, -1.f, -1.f};          // pass 1, tile offsets, write pass, aggregate finish
    unsigned long long* h_small = nullptr; // pinned: nagg raw values + count
    float kernel_ms = -1.f;
};

namespace mbc {

// ---- helpers implemented in mbc_api.cu ----------------------------------------------------
void    ctx_retain(mbc_ctx* ctx);            // a table / result / shard now lives on the context
void    ctx_release(mbc_ctx* ctx);           // ... and is gone: destroys the context if mbc_shutdown was called meanwhile
int32_t dev_alloc(mbc_ctx* ctx, void** p, size_t bytes, bool zero);
void    dev_free(mbc_ctx* ctx, void* p);
int32_t pinned_alloc(mbc_ctx* ctx, void** p, size_t bytes, size_t* actual);
void    pinned_release(mbc_ctx* ctx, void* p, size_t bytes);
int32_t ensure_workspace(mbc_ctx* ctx, size_t bytes);
void    begin_timing(mbc_ctx* ctx);
void    end_timing(mbc_ctx* ctx);
void    split_timing(mbc_ctx* ctx);
void    result_phase_times(mbc_result* r);  // fills phase_ms from the events of a completed resident scan
int32_t result_finalize(mbc_result* r);   // wait for a deferred result's count/aggregates (no-op when final)
cudaEvent_t event_get(mbc_ctx* ctx);
// one aggregate from its raw 8 bytes (int64 for COUNT and integer columns, else the bits of a double): exact integers, a
// real's as_i64 through real_agg_as_i64; MIN / MAX over an empty set are invalid and read 0
void    agg_from_raw(int32_t kind, int32_t type, unsigned long long raw, bool nonempty, int64_t* i, double* f, int32_t* valid);
void    event_put(mbc_ctx* ctx, cudaEvent_t e);        // close a timed segment (sync), keep its time, the next begin_timing adds to it

// ---- the select -> compact -> project -> aggregate engine (mbc_scan.cu) ---------------------
struct ScanRequest {
    mbc_table* table = nullptr;
    const mbc_term* terms = nullptr;
    int32_t nterms = 0;
    const uint32_t* d_sel_bitmap = nullptr;   // precomputed selection (bitmap scan / join sides)
    const int32_t* proj_cols = nullptr;
    int32_t nproj = 0;
    uint32_t want = 0;
    const mbc_aggspec* aggs = nullptr;
    int32_t nagg = 0;
    bool allow_deferred = false;              // mbc_scan: device-resident results may complete asynchronously
};
int32_t run_scan(const ScanRequest& rq, mbc_result** out);
int32_t finish_result_host(mbc_result* r);     // tuple encode + D2H according to r->want
// stable LSD radix sort of (key, value) pairs by the low key_bits bits of the keys, in place (mbc_join.cu)
// pass_mask: bit p = run the pass over key bits [8p, 8p+8) (clear it for digits known to be constant)
int32_t radix_sort_pairs(mbc_ctx* ctx, uint32_t* d_keys, uint32_t* d_vals, int64_t n, int key_bits, uint32_t pass_mask = 0xFu);
// exclusive scan of n uint32 counts into n+1 uint64 offsets, total in d_out[n] (mbc_join.cu)
int32_t exclusive_scan_u32(mbc_ctx* ctx, const uint32_t* d_in, int64_t n, unsigned long long* d_out);

// ---- row-id sorting shared by mbc_sort, the sparse bitmap layout and mbc_topk (mbc_sort.cu) ------------------------
// keys[i] = 32-bit word `word` of column row rows[i] as an unsigned key in sort order (ints biased, reals in total order
// with -0.0 as +0.0, string words byte-swapped), complemented when descending
__global__ void __launch_bounds__(256) sort_key_kernel(const uint32_t* __restrict__ rows, int64_t n, const void* col, int stride, int word,
                                                       int type, int descending, uint32_t* __restrict__ keys);
// or_and[0] |= every key, or_and[1] &= every key (preset {0, ~0}): the digits where they agree are constant
__global__ void __launch_bounds__(256) sort_key_bits_kernel(const uint32_t* __restrict__ keys, int64_t n, uint32_t* or_and);
// rows[i] = pos[i] - base
__global__ void __launch_bounds__(256) sort_rows_from_positions_kernel(const int64_t* __restrict__ pos, int64_t n, int64_t base,
                                                                      uint32_t* __restrict__ rows);
// rows[i] = i
__global__ void __launch_bounds__(256) sort_iota_kernel(int64_t n, uint32_t* __restrict__ rows);
// out row i = column row rows[i] (stride bytes, a multiple of 4; stride 8 gathers int64 positions)
__global__ void __launch_bounds__(256) sort_gather_kernel(const uint32_t* __restrict__ rows, int64_t n, const void* src, int stride, void* dst);
// pos[i] = base + rows[i]
__global__ void __launch_bounds__(256) sort_positions_kernel(const uint32_t* __restrict__ rows, int64_t n, int64_t base, int64_t* __restrict__ pos);
// run d = run_of[i] of a head i starts at element i: start[d] = i, head_row[d] = rows[i] (mbc_bitmap.cu)
__global__ void __launch_bounds__(256) sparse_run_starts_kernel(const uint32_t* __restrict__ head, const unsigned long long* __restrict__ run_of,
                                                                const uint32_t* __restrict__ rows, int64_t n, uint32_t* __restrict__ start,
                                                                uint32_t* __restrict__ head_row);
// stable reorder of the row ids `rows` by column c (every 32-bit word of its key, least significant first), so rows
// with equal keys keep their order; keys (n words) and bits (2 words) are scratch
int32_t sort_rows_by_column(mbc_ctx* ctx, uint32_t* rows, int64_t n, const Column& c, bool descending, uint32_t* keys, uint32_t* bits);

// ---- GROUP BY over row ids, shared by mbc_group_aggregate and mbc_shard_group (mbc_group.cu) ------------------------
struct GroupAggSpec {
    int32_t kind;              // MBC_AGG_*
    int32_t type;              // type of the aggregated column (MBC_ATTR_INTEGER for COUNT)
    const void* src;           // per row id: int32 / float32 column values, or 8-byte raw partials when `partials`
};
// Groups the n row ids `rows` (sorted in place) by the key columns, ascending, equal keys in row-id order.  Row id i's
// position is pos[i] when pos is not NULL, else pos_base + i; each group's positions / key values are those of its first
// row id.  `partials`: every source holds raw aggregates of earlier groupings (a COUNT partial is added).  Fills r (ctx,
// want set by the caller): count, d_pos, cols, d_aggs, group_nagg, group_aggs; host copies per r->want.  Ends the caller's
// timed segment (begin_timing) after the kernels, and returns after they have finished.
int32_t group_rows(mbc_ctx* ctx, uint32_t* rows, int64_t n, const Column* keys, int32_t nkeys, const GroupAggSpec* aggs, int32_t nagg,
                   bool partials, const int64_t* pos, int64_t pos_base, mbc_result* r);

}  // namespace mbc
