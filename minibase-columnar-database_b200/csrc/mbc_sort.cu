// mbc_sort.cu -- ColumnarSort on the GPU (SURVEY.md 8f rank 4; input/ColumnarSort.java:73-400).
//
// The reference sorts (key columns..., position) records with an external merge sort under a comparator that walks the
// key columns in order: ints numerically, strings by String.compareTo (:163-205); ASC or DSC for all keys at once.  Here
// the row ids are sorted by a stable LSD radix sort, one 32-bit key word at a time from the least significant word of
// the last key column to the most significant word of the first, so equal keys keep ascending position order (the
// Java's merge leaves the order of ties unspecified).  Deleted rows are skipped (it reads through ColumnScan).
#include <algorithm>
#include <vector>

#include "mbc_internal.cuh"

namespace mbc {

// key word of every row id in `rows`: ints biased to unsigned order, reals mapped to their total order, string words
// byte-swapped so that unsigned compare = byte order; complemented for a descending sort
__global__ void __launch_bounds__(256) sort_key_kernel(const uint32_t* __restrict__ rows, int64_t n, const void* col, int stride, int word,
                                                       int type, int descending, uint32_t* __restrict__ keys) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        uint32_t v = reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(col) + (size_t)rows[i] * stride)[word];
        if (type == MBC_ATTR_INTEGER) v ^= 0x80000000u;
        else if (type == MBC_ATTR_REAL) v = (v & 0x80000000u) ? ~v : (v | 0x80000000u);
        else v = __byte_perm(v, 0, 0x0123);
        keys[i] = descending ? ~v : v;
    }
}

// OR and AND of all keys: a byte in which they agree is the same in every key, and its radix pass can be skipped
__global__ void __launch_bounds__(256) sort_key_bits_kernel(const uint32_t* __restrict__ keys, int64_t n, uint32_t* or_and /* [2], preset {0, ~0} */) {
    uint32_t o = 0u, a = ~0u;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t k = keys[i];
        o |= k;
        a &= k;
    }
    o = __reduce_or_sync(0xFFFFFFFFu, o);
    a = __reduce_and_sync(0xFFFFFFFFu, a);
    if ((threadIdx.x & 31) == 0) {
        atomicOr(or_and, o);
        atomicAnd(or_and + 1, a);
    }
}

__global__ void __launch_bounds__(256) sort_rows_from_positions_kernel(const int64_t* __restrict__ pos, int64_t n, int64_t base,
                                                                      uint32_t* __restrict__ rows) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        rows[i] = (uint32_t)(pos[i] - base);
}

__global__ void __launch_bounds__(256) sort_positions_kernel(const uint32_t* __restrict__ rows, int64_t n, int64_t base, int64_t* __restrict__ pos) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        pos[i] = base + rows[i];
}

// out row i = column row rows[i] (stride bytes, a multiple of 4)
__global__ void __launch_bounds__(256) sort_gather_kernel(const uint32_t* __restrict__ rows, int64_t n, const void* src, int stride, void* dst) {
    const int words = stride >> 2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n * words; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / words;
        const int w = (int)(i - r * words);
        reinterpret_cast<uint32_t*>(dst)[i] = reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(src) + (size_t)rows[r] * stride)[w];
    }
}

int32_t sort_rows_by_column(mbc_ctx* ctx, uint32_t* rows, int64_t n, const Column& c, bool descending, uint32_t* keys, uint32_t* bits) {
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8));
    const int words = c.type == MBC_ATTR_STRING ? (c.width + 3) / 4 : 1;      // bytes past the width are zero padding
    for (int w = words - 1; w >= 0; --w) {
        sort_key_kernel<<<grid, 256, 0, ctx->stream>>>(rows, n, c.d, c.stride, w, c.type, descending ? 1 : 0, keys);
        // which of the four digits vary at all (small int domains, zero padding and common prefixes of strings do not)
        const uint32_t preset[2] = {0u, ~0u};
        uint32_t seen[2];
        MBC_CUDA(cudaMemcpyAsync(bits, preset, 8, cudaMemcpyHostToDevice, ctx->stream));
        sort_key_bits_kernel<<<grid, 256, 0, ctx->stream>>>(keys, n, bits);
        ctx->launches += 2;
        MBC_CUDA(cudaMemcpyAsync(seen, bits, 8, cudaMemcpyDeviceToHost, ctx->stream));
        MBC_CUDA(cudaStreamSynchronize(ctx->stream));
        const uint32_t differ = seen[0] ^ seen[1];
        uint32_t pass_mask = 0;
        for (int b = 0; b < 4; ++b)
            if ((differ >> (8 * b)) & 0xFFu) pass_mask |= 1u << b;
        MBC_TRY(radix_sort_pairs(ctx, keys, rows, n, 32, pass_mask));
    }
    return MBC_OK;
}

}  // namespace mbc

using namespace mbc;

extern "C" int32_t mbc_sort(mbc_table* t, const int32_t* key_cols, int32_t nkeys, int32_t descending, const int32_t* proj_cols,
                            int32_t nproj, uint32_t want, mbc_result** out) {
    if (!t || !out || !key_cols || nkeys <= 0 || (nproj > 0 && !proj_cols)) MBC_FAIL(MBC_ERR_ARG, "mbc_sort: bad argument");
    *out = nullptr;
    if (nkeys > kMaxTerms || nproj > kMaxProj) MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_sort: %d key columns / %d projected fields", nkeys, nproj);
    for (int k = 0; k < nkeys; ++k)
        if (key_cols[k] < 0 || key_cols[k] >= (int)t->cols.size()) MBC_FAIL(MBC_ERR_ARG, "mbc_sort: key column %d out of range", key_cols[k]);
    for (int c = 0; c < nproj; ++c)
        if (proj_cols[c] < 0 || proj_cols[c] >= (int)t->cols.size()) MBC_FAIL(MBC_ERR_ARG, "mbc_sort: projected column %d out of range", proj_cols[c]);
    if (t->nrows > (int64_t)UINT32_MAX) MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_sort: more than 2^32 rows in one table");
    mbc_ctx* ctx = t->ctx;
    MBC_CUDA(cudaSetDevice(ctx->device));

    // the rows that exist (not deleted), in position order: a scan with no predicate
    mbc_result* all = nullptr;
    ScanRequest rq;
    rq.table = t;
    rq.want = MBC_WANT_POSITIONS;
    MBC_TRY(run_scan(rq, &all));
    const int64_t n = all->count;

    mbc_result* r = new mbc_result();
    r->ctx = ctx;
    ctx_retain(ctx);
    r->want = want;
    r->nrows = t->nrows;
    r->count = n;
    r->capacity = n;
    uint32_t *rows = nullptr, *keys = nullptr, *bits = nullptr;
    auto fail = [&](int32_t s) {
        dev_free(ctx, rows);
        dev_free(ctx, keys);
        dev_free(ctx, bits);
        mbc_result_free(all);
        mbc_result_free(r);
        return s;
    };
#define STRY(x) do { int32_t _s = (x); if (_s != MBC_OK) return fail(_s); } while (0)
    begin_timing(ctx);
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8));
    if (n > 0) {
        STRY(dev_alloc(ctx, (void**)&rows, (size_t)n * 4, false));
        STRY(dev_alloc(ctx, (void**)&keys, (size_t)n * 4, false));
        STRY(dev_alloc(ctx, (void**)&bits, 8, false));
        sort_rows_from_positions_kernel<<<grid, 256, 0, ctx->stream>>>(all->d_pos, n, t->pos_base, rows);
        ctx->launches++;
        for (int k = nkeys - 1; k >= 0; --k) STRY(sort_rows_by_column(ctx, rows, n, t->cols[key_cols[k]], descending != 0, keys, bits));
    }
    if ((want & MBC_WANT_POSITIONS) && n > 0) {
        STRY(dev_alloc(ctx, (void**)&r->d_pos, (size_t)n * 8, false));
        sort_positions_kernel<<<grid, 256, 0, ctx->stream>>>(rows, n, t->pos_base, r->d_pos);
        ctx->launches++;
    }
    if ((want & (MBC_WANT_COLUMNS | MBC_WANT_TUPLES)) && nproj > 0) {
        for (int c = 0; c < nproj; ++c) {
            const Column& col = t->cols[proj_cols[c]];
            mbc_result::Col rc{col.type, col.width, col.stride, nullptr, nullptr};
            STRY(dev_alloc(ctx, &rc.d, (size_t)std::max<int64_t>(n, 1) * col.stride, false));
            r->cols.push_back(rc);
            if (n > 0) {
                sort_gather_kernel<<<grid, 256, 0, ctx->stream>>>(rows, n, col.d, col.stride, rc.d);
                ctx->launches++;
            }
        }
    }
    end_timing(ctx);
    if (cudaGetLastError() != cudaSuccess) return fail((set_error("mbc_sort: launch failed"), MBC_ERR_CUDA));
    STRY(finish_result_host(r));
#undef STRY
    MBC_CUDA(cudaStreamSynchronize(ctx->stream));
    dev_free(ctx, rows);
    dev_free(ctx, keys);
    dev_free(ctx, bits);
    mbc_result_free(all);
    *out = r;
    return MBC_OK;
}
