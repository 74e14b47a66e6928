// mbc_topk.cu -- ORDER BY key columns LIMIT k over a filtered table (mbc_topk), by radix select.
//
// The result is the first min(k, Q) rows of mbc_sort's order over the Q qualifying rows.  When k is a large share of Q
// the qualifying rows are simply sorted with mbc_sort's stable radix passes (a filtered sort).  Otherwise the k rows are
// selected without sorting the rest: the composite key (key 0's 32-bit words, then key 1's, ..., then the row id) is read
// one 8-bit digit at a time, most significant first.  Per digit a histogram over the candidates finds the bucket b that
// holds the k-th key; rows with a digit below b are marked in a selection bitmap, the rows of bucket b stay candidates,
// the rest are dropped.  The row id, the last word, makes the composite key unique (it is never complemented, so equal
// keys rank by ascending position in both directions), so the select ends with exactly k marked rows.  A scan of the
// selection bitmap lists them in position order, and a stable sort of those <= k rows gives mbc_sort's order.
//
// The per-digit choice stays on the device (topk_pick_kernel writes it into a TopkState that the next kernels read), so
// the host waits once per key word: it reads the candidate count to size the next word's launches.
#include <algorithm>
#include <cstddef>
#include <vector>

#include "mbc_internal.cuh"

// Share of the qualifying rows above which a top-k sorts them all instead of selecting (DESIGN.md §5, measured with
// scripts/bench_topk.py).  Overridable at compile time only, to measure both paths at every k.
#ifndef MBC_TOPK_SORT_FRACTION
#define MBC_TOPK_SORT_FRACTION 0.5
#endif

namespace mbc {

constexpr double kTopkSortFraction = MBC_TOPK_SORT_FRACTION;
constexpr int kHistWarps = 8;                    // topk_hist_kernel: one shared histogram per warp

// Candidates live in one of two buffers; a split moves those of bucket b to the other one.  For the row-id word the
// key buffers are the row buffers themselves.
struct TopkBufs {
    uint32_t* rows[2];
    uint32_t* keys[2];
    // buffer i's pointers without indexing the kernel parameter by a runtime value (that would copy it to the stack)
    __device__ __forceinline__ uint32_t* row_buf(uint32_t i) const { return i ? rows[1] : rows[0]; }
    __device__ __forceinline__ uint32_t* key_buf(uint32_t i) const { return i ? keys[1] : keys[0]; }
};

// Select state on the device.  count[] is per buffer, so a split (which reads count[src]) and the kernels after it
// (which read count[cur]) both see the right value without a host round trip.
struct TopkState {
    uint32_t count[2];     // candidates in buffer 0 / 1
    uint32_t need;         // rows still to select among the candidates in buffer cur
    uint32_t cur;          // buffer of the current candidates
    uint32_t src;          // buffer the pending split reads (the other one receives bucket b)
    uint32_t skip;         // the pending split has nothing to do
    uint32_t lo;           // the pending split marks digits < lo
    uint32_t keep;         // ... and keeps digit == keep as the next candidates (256: none)
    uint32_t ticket;       // output slots taken by the pending split
    uint32_t or_and[2];    // sort_key_bits_kernel over the current word's keys: digits where they agree are constant
    uint32_t hist[256];    // digit counts of the current pass (zeroed again by topk_pick_kernel)
};

__device__ __forceinline__ bool topk_digit_constant(const TopkState* st, int shift) {
    return (((st->or_and[0] ^ st->or_and[1]) >> shift) & 0xFFu) == 0u;
}

// hist[d] += candidates whose digit (key >> shift) & 0xFF is d.  Per-warp shared histograms, merged with integer atomics,
// so the counts do not depend on the order of the adds.
__global__ void __launch_bounds__(256) topk_hist_kernel(TopkBufs b, TopkState* st, int shift) {
    __shared__ uint32_t h[kHistWarps][256];
    if (st->need == 0 || topk_digit_constant(st, shift)) return;
    const uint32_t cur = st->cur, n = st->count[cur];
    const uint32_t* __restrict__ keys = b.key_buf(cur);
    for (int i = threadIdx.x; i < kHistWarps * 256; i += blockDim.x) (&h[0][0])[i] = 0u;
    __syncthreads();
    uint32_t* hw = h[(threadIdx.x >> 5) % kHistWarps];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        atomicAdd(hw + ((keys[i] >> shift) & 0xFFu), 1u);
    __syncthreads();
    for (int d = threadIdx.x; d < 256; d += blockDim.x) {
        uint32_t s = 0;
        for (int w = 0; w < kHistWarps; ++w) s += h[w][d];
        if (s) atomicAdd(st->hist + d, s);
    }
}

// One block of 256 threads: the bucket b in which the need-th smallest remaining key falls (a prefix over the counts),
// and what the split does with it.  Zeroes the histogram for the next pass.
__global__ void __launch_bounds__(256) topk_pick_kernel(TopkState* st, int shift) {
    __shared__ uint32_t s_warp[8];
    const int d = threadIdx.x, lane = d & 31, warp = d >> 5;
    if (d == 0) st->ticket = 0u;
    if (st->need == 0 || topk_digit_constant(st, shift)) {
        if (d == 0) st->skip = 1u;
        return;
    }
    const uint32_t need = st->need, cur = st->cur, n = st->count[cur];
    const uint32_t c = st->hist[d];
    st->hist[d] = 0u;
    uint32_t incl = c;                                            // inclusive prefix over the digits
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    for (int w = 0; w < warp; ++w) incl += s_warp[w];
    const uint32_t excl = incl - c;
    if (c == 0u || excl >= need || need > incl) return;          // exactly one digit holds the need-th key
    const uint32_t left = need - excl;                            // rows still needed inside bucket d
    if (left == c) {                                              // the whole bucket: mark digits <= d, done
        st->lo = d + 1;
        st->keep = 256u;
        st->need = 0u;
        st->count[cur ^ 1u] = 0u;
    } else if (c == n) {                                          // every candidate is in bucket d: nothing to split
        st->skip = 1u;
        return;
    } else {
        st->lo = d;
        st->keep = d;
        st->need = left;
        st->count[cur ^ 1u] = c;
    }
    st->src = cur;
    st->cur = cur ^ 1u;
    st->skip = 0u;
}

// The split that topk_pick_kernel chose (mark_all: mark every current candidate).  Marks merge per warp into one
// atomicOr per touched bitmap word, as sparse_scatter_kernel does.  Kept candidates take their output slots through one
// ticket per 4096-candidate tile (a block-wide scan places them inside it): one ticket per warp made a bucket holding most
// of 10^8 candidates wait on millions of atomics to one address.  Their order in the next buffer is arbitrary; the
// composite key is unique, so no later step depends on it.
constexpr int kSplitItems = 16;
constexpr int kSplitTile = 256 * kSplitItems;

__global__ void __launch_bounds__(256) topk_split_kernel(TopkBufs b, TopkState* st, int shift, int mark_all, uint32_t* __restrict__ sel) {
    __shared__ uint32_t s_warp[8];
    __shared__ uint32_t s_base;
    if (!mark_all && st->skip) return;
    const uint32_t src = mark_all ? st->cur : st->src, n = st->count[src];
    const uint32_t lo = mark_all ? 256u : st->lo, keep = mark_all ? 256u : st->keep;
    const uint32_t* __restrict__ rows_in = b.row_buf(src);
    const uint32_t* __restrict__ keys_in = b.key_buf(src);
    uint32_t* rows_out = b.row_buf(src ^ 1u);
    uint32_t* keys_out = b.key_buf(src ^ 1u);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int64_t t0 = (int64_t)blockIdx.x * kSplitTile; t0 < n; t0 += (int64_t)gridDim.x * kSplitTile) {   // block-uniform
        uint32_t kept = 0;                                        // bit j: element t0 + j * 256 + tid stays a candidate
#pragma unroll 4
        for (int j = 0; j < kSplitItems; ++j) {
            const int64_t i = t0 + j * 256 + tid;
            const bool ok = i < n;
            const uint32_t r = ok ? rows_in[i] : 0u;
            const uint32_t digit = ok && !mark_all ? (keys_in[i] >> shift) & 0xFFu : 0u;
            const bool mark = ok && digit < lo;
            const uint32_t word = mark ? r >> 5 : 0xFFFFFFFFu;   // (a row id's word is below 2^27)
            const uint32_t group = __match_any_sync(0xFFFFFFFFu, word);
            const uint32_t bits = __reduce_or_sync(group, mark ? 1u << (r & 31) : 0u);
            if (mark && (group & ((1u << lane) - 1)) == 0) atomicOr(sel + word, bits);
            if (ok && digit == keep) kept |= 1u << j;
        }
        if (__syncthreads_or(kept) == 0) continue;
        // exclusive prefix of the threads' kept counts over the block, one ticket for the tile
        const uint32_t c = __popc(kept);
        uint32_t incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        uint32_t before = 0, total = 0;
        for (int w = 0; w < 8; ++w) {
            if (w < warp) before += s_warp[w];
            total += s_warp[w];
        }
        if (tid == 0) s_base = atomicAdd(&st->ticket, total);
        __syncthreads();
        uint32_t o = s_base + before + incl - c;
        for (int j = 0; kept; ++j, kept >>= 1) {
            if (!(kept & 1u)) continue;
            const int64_t i = t0 + j * 256 + tid;
            rows_out[o] = rows_in[i];
            if (keys_out != rows_out) keys_out[o] = keys_in[i];
            ++o;
        }
        __syncthreads();                                          // s_warp / s_base are reused by the next tile
    }
}

static int grid_for(const mbc_ctx* ctx, int64_t n) {
    return (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8));
}

// Mark the k rows of `rows` (n qualifying row ids, k < n) that come first in key order in sel (words_pad words, zero).
// rows and keys are n-word scratch pairs; rows[0] holds the row ids on entry.
static int32_t topk_select(mbc_ctx* ctx, mbc_table* t, const int32_t* key_cols, int32_t nkeys, bool descending, int64_t n, int64_t k,
                           TopkBufs bufs, TopkState* d_st, uint32_t* sel) {
    TopkState init{};
    init.count[0] = (uint32_t)n;
    init.need = (uint32_t)k;
    MBC_CUDA(cudaMemcpyAsync(d_st, &init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
    const uint32_t preset[2] = {0u, ~0u};
    TopkState st = init;
    // the key words, most significant first, then the row id (key_col = -1)
    std::vector<std::pair<int, int>> words;
    for (int q = 0; q < nkeys; ++q) {
        const Column& c = t->cols[key_cols[q]];
        const int nw = c.type == MBC_ATTR_STRING ? (c.width + 3) / 4 : 1;   // bytes past the width are zero padding
        for (int w = 0; w < nw; ++w) words.push_back({key_cols[q], w});
    }
    words.push_back({-1, 0});
    for (size_t wi = 0; wi <= words.size(); ++wi) {
        if (wi > 0) {                                             // the one host wait per word: the candidates left
            MBC_CUDA(cudaMemcpyAsync(&st, d_st, offsetof(TopkState, or_and), cudaMemcpyDeviceToHost, ctx->stream));
            MBC_CUDA(cudaStreamSynchronize(ctx->stream));
        }
        const uint32_t count = st.count[st.cur];
        if (st.need == 0) return MBC_OK;
        if (st.need == count) {                                   // every candidate is selected
            topk_split_kernel<<<grid_for(ctx, count), 256, 0, ctx->stream>>>(bufs, d_st, 0, 1, sel);
            ctx->launches++;
            return MBC_OK;
        }
        if (wi == words.size()) break;
        const int col = words[wi].first;
        TopkBufs b = bufs;
        if (col >= 0) {
            const Column& c = t->cols[col];
            sort_key_kernel<<<grid_for(ctx, count), 256, 0, ctx->stream>>>(b.rows[st.cur], count, c.d, c.stride, words[wi].second, c.type,
                                                                            descending ? 1 : 0, b.keys[st.cur]);
            ctx->launches++;
        } else {                                                  // the row id is its own key, ascending in both directions
            b.keys[0] = b.rows[0];
            b.keys[1] = b.rows[1];
        }
        MBC_CUDA(cudaMemcpyAsync(d_st->or_and, preset, 8, cudaMemcpyHostToDevice, ctx->stream));
        sort_key_bits_kernel<<<grid_for(ctx, count), 256, 0, ctx->stream>>>(b.keys[st.cur], count, d_st->or_and);
        ctx->launches++;
        for (int shift = 24; shift >= 0; shift -= 8) {
            topk_hist_kernel<<<grid_for(ctx, count), 256, 0, ctx->stream>>>(b, d_st, shift);
            topk_pick_kernel<<<1, 256, 0, ctx->stream>>>(d_st, shift);
            topk_split_kernel<<<grid_for(ctx, count), 256, 0, ctx->stream>>>(b, d_st, shift, 0, sel);
            ctx->launches += 3;
        }
        MBC_CUDA(cudaGetLastError());
    }
    MBC_FAIL(MBC_ERR_CUDA, "mbc_topk: the select ended with %u rows still needed", st.need);
}

}  // namespace mbc

using namespace mbc;

extern "C" int32_t mbc_topk(mbc_table* t, const mbc_term* terms, int32_t nterms, const int32_t* key_cols, int32_t nkeys, int32_t descending,
                            int64_t k, const int32_t* proj_cols, int32_t nproj, uint32_t want, mbc_result** out) {
    if (!t || !out || !key_cols || nkeys <= 0 || (nproj > 0 && !proj_cols) || nproj < 0) MBC_FAIL(MBC_ERR_ARG, "mbc_topk: bad argument");
    *out = nullptr;
    if (k < 0) MBC_FAIL(MBC_ERR_ARG, "mbc_topk: k = %lld is negative", (long long)k);
    if (want & (MBC_WANT_AGG | MBC_WANT_BITMAP))
        MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_topk: MBC_WANT_AGG / MBC_WANT_BITMAP are not available for a top-k");
    if (nkeys > kMaxTerms || nproj > kMaxProj) MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_topk: %d key columns / %d projected fields", nkeys, nproj);
    for (int q = 0; q < nkeys; ++q)
        if (key_cols[q] < 0 || key_cols[q] >= (int)t->cols.size()) MBC_FAIL(MBC_ERR_ARG, "mbc_topk: key column %d out of range", key_cols[q]);
    for (int c = 0; c < nproj; ++c)
        if (proj_cols[c] < 0 || proj_cols[c] >= (int)t->cols.size()) MBC_FAIL(MBC_ERR_ARG, "mbc_topk: projected column %d out of range", proj_cols[c]);
    if (t->nrows > (int64_t)UINT32_MAX) MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_topk: more than 2^32 rows in one table");
    mbc_ctx* ctx = t->ctx;
    MBC_CUDA(cudaSetDevice(ctx->device));

    // the qualifying rows in position order (the predicate checks its terms)
    mbc_result* qual = nullptr;
    ScanRequest rq;
    rq.table = t;
    rq.terms = terms;
    rq.nterms = nterms;
    rq.want = MBC_WANT_POSITIONS;
    MBC_TRY(run_scan(rq, &qual));
    const int64_t n = qual->count;
    const int64_t m = std::min<int64_t>(k, n);
    split_timing(ctx);                                      // the scan's kernels count, the host wait in between does not
    begin_timing(ctx);

    mbc_result* r = new mbc_result();
    r->ctx = ctx;
    ctx_retain(ctx);
    r->want = want;
    r->nrows = t->nrows;
    r->count = m;
    r->capacity = m;
    mbc_result* chosen = nullptr;
    uint32_t *rows = nullptr, *rows2 = nullptr, *keys = nullptr, *keys2 = nullptr, *bits = nullptr, *sel = nullptr;
    TopkState* st = nullptr;
    auto release = [&]() {
        for (void* p : {(void*)rows, (void*)rows2, (void*)keys, (void*)keys2, (void*)bits, (void*)sel, (void*)st}) dev_free(ctx, p);
        mbc_result_free(qual);
        mbc_result_free(chosen);
    };
    auto fail = [&](int32_t s) {
        release();
        mbc_result_free(r);
        return s;
    };
#define KTRY(x) do { int32_t _s = (x); if (_s != MBC_OK) return fail(_s); } while (0)
#define KCUDA(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) return fail((set_error("mbc_topk: %s", cudaGetErrorString(_e)), MBC_ERR_CUDA)); } while (0)
    // `rows` ends up holding the result's m row ids in key order
    if (m > 0) {
        KTRY(dev_alloc(ctx, (void**)&rows, (size_t)n * 4, false));
        KTRY(dev_alloc(ctx, (void**)&keys, (size_t)n * 4, false));
        KTRY(dev_alloc(ctx, (void**)&bits, 8, false));
        sort_rows_from_positions_kernel<<<grid_for(ctx, n), 256, 0, ctx->stream>>>(qual->d_pos, n, t->pos_base, rows);
        ctx->launches++;
        if ((double)k > kTopkSortFraction * (double)n) {
            // filtered sort: every qualifying row, the first m kept
            for (int q = nkeys - 1; q >= 0; --q) KTRY(sort_rows_by_column(ctx, rows, n, t->cols[key_cols[q]], descending != 0, keys, bits));
        } else {
            KTRY(dev_alloc(ctx, (void**)&rows2, (size_t)n * 4, false));
            KTRY(dev_alloc(ctx, (void**)&keys2, (size_t)n * 4, false));
            KTRY(dev_alloc(ctx, (void**)&sel, (size_t)t->words_pad * 4, true));
            KTRY(dev_alloc(ctx, (void**)&st, sizeof(TopkState), false));
            TopkBufs bufs{{rows, rows2}, {keys, keys2}};
            KTRY(topk_select(ctx, t, key_cols, nkeys, descending != 0, n, k, bufs, st, sel));
            // the m selected rows in position order, then stably by the keys
            split_timing(ctx);
            ScanRequest srq;
            srq.table = t;
            srq.d_sel_bitmap = sel;
            srq.want = MBC_WANT_POSITIONS;
            KTRY(run_scan(srq, &chosen));
            split_timing(ctx);
            begin_timing(ctx);
            if (chosen->count != m) {
                set_error("mbc_topk: %lld rows selected, %lld expected", (long long)chosen->count, (long long)m);
                return fail(MBC_ERR_CUDA);
            }
            sort_rows_from_positions_kernel<<<grid_for(ctx, m), 256, 0, ctx->stream>>>(chosen->d_pos, m, t->pos_base, rows);
            ctx->launches++;
            for (int q = nkeys - 1; q >= 0; --q) KTRY(sort_rows_by_column(ctx, rows, m, t->cols[key_cols[q]], descending != 0, keys, bits));
        }
    }
    if ((want & MBC_WANT_POSITIONS) && m > 0) {
        KTRY(dev_alloc(ctx, (void**)&r->d_pos, (size_t)m * 8, false));
        sort_positions_kernel<<<grid_for(ctx, m), 256, 0, ctx->stream>>>(rows, m, t->pos_base, r->d_pos);
        ctx->launches++;
    }
    if ((want & (MBC_WANT_COLUMNS | MBC_WANT_TUPLES)) && nproj > 0) {
        for (int c = 0; c < nproj; ++c) {
            const Column& col = t->cols[proj_cols[c]];
            mbc_result::Col rc{col.type, col.width, col.stride, nullptr, nullptr};
            KTRY(dev_alloc(ctx, &rc.d, (size_t)std::max<int64_t>(m, 1) * col.stride, false));
            r->cols.push_back(rc);
            if (m > 0) {
                sort_gather_kernel<<<grid_for(ctx, m), 256, 0, ctx->stream>>>(rows, m, col.d, col.stride, rc.d);
                ctx->launches++;
            }
        }
    }
    end_timing(ctx);
    KCUDA(cudaGetLastError());
    KTRY(finish_result_host(r));
    KCUDA(cudaStreamSynchronize(ctx->stream));
#undef KTRY
#undef KCUDA
    release();
    *out = r;
    return MBC_OK;
}
