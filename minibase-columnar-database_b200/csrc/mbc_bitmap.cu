// mbc_bitmap.cu -- K3 bitmap-index build and K4 bitmap CNF combine.
//
// K3 replaces columnar/Columnarfile.java:698-753 createBitMapIndex(): one UNCOMPRESSED bitset per
// distinct value of a column (bit p set iff column[p] == value and p was not deleted at build time;
// the reference's ColumnScan skips deleted rows, columnar/ColumnScan.java:49-65).  Bit order is
// java.util.BitSet's: bit p lives in byte p/8, bit p%8 (bitmap/BM.java:64-129 persists
// BitSet.toByteArray()), which is also bit p%32 of little-endian uint32 word p/32.
//
// K4 replaces index/ColumnarIndexScan.java:130-181 (OR inside a conjunct, AND across conjuncts) with
// each term resolved as index/ColumnIndexScan.java:656-740 getBitSet(): EQ -> that value's bitmap,
// LT/LE/GT/GE/NE -> OR of the bitmaps of every indexed value that satisfies the operator; rows in
// markedDeleted are dropped (ColumnIndexScan.java:600-624).
//
// Build kernel: a CTA owns a chunk of R rows and an smem matrix [values][R/32] of bitmap words.  A
// warp's 32 rows are exactly one word column; __match_any_sync groups the lanes that hold the same
// value, and the group leader stores the group's lane mask as the finished word -- no atomics, every
// word is written once.  The matrix (zeros included: the index is uncompressed by definition) is
// then streamed out with 128-bit stores, R/8 contiguous bytes per value.  The kernel is bound by
// HBM writes: D*N/8 bytes out for 4*N bytes in.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <numeric>

#include "mbc_internal.cuh"

namespace mbc {

// ---- distinct values: open-addressing hash set in global memory ---------------------------------
// ints   : slot = (1<<32) | (uint32)value
// strings: slot = row index + 1 of a representative row
struct HashTab {
    unsigned long long* slots;
    uint32_t* slot_id;       // dense id per slot, filled by the host after sorting the values
    uint32_t mask;           // capacity - 1
    // direct mode (int column whose value range is small): id = id_of[value - kmin], no hashing
    const uint32_t* id_of;
    long long kmin;
    uint32_t range;
    int32_t direct;
};

constexpr uint32_t kMaxDirectRange = 1u << 16;

__global__ void __launch_bounds__(256) column_minmax_kernel(const int32_t* col, int64_t nrows, const uint32_t* deleted, long long* out) {
    long long mn = INT64_MAX, mx = INT64_MIN;
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (!deleted) {                                                  // 128-bit loads, two in flight (columns are padded to 8192 rows)
        const int64_t nq = nrows >> 2;
        const int4* c4 = reinterpret_cast<const int4*>(col);
        int64_t q = r;
        for (; q + step < nq; q += 2 * step) {
            const int4 a = __ldg(c4 + q), b = __ldg(c4 + q + step);
            int lo = min(min(min(a.x, a.y), min(a.z, a.w)), min(min(b.x, b.y), min(b.z, b.w)));
            int hi = max(max(max(a.x, a.y), max(a.z, a.w)), max(max(b.x, b.y), max(b.z, b.w)));
            mn = min(mn, (long long)lo);
            mx = max(mx, (long long)hi);
        }
        for (; q < nq; q += step) {
            const int4 a = __ldg(c4 + q);
            mn = min(mn, (long long)min(min(a.x, a.y), min(a.z, a.w)));
            mx = max(mx, (long long)max(max(a.x, a.y), max(a.z, a.w)));
        }
        r = (nq << 2) + r;                                           // ragged tail below
        for (; r < nrows; r += step) { mn = min(mn, (long long)col[r]); mx = max(mx, (long long)col[r]); }
    } else {
        for (; r < nrows; r += step) {
            if ((deleted[r >> 5] >> (r & 31)) & 1u) continue;
            long long k = col[r];
            mn = min(mn, k);
            mx = max(mx, k);
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xFFFFFFFFu, mn, o));
        mx = max(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
    }
    if ((threadIdx.x & 31) == 0 && mn <= mx) {                       // (a warp that saw no row keeps mn > mx)
        atomicMin(out, (long long)mn);
        atomicMax(out + 1, (long long)mx);
    }
}

// presence bits of the values of a small-range int column: per-CTA bitmap in shared memory, OR-ed into global
__global__ void __launch_bounds__(256) column_presence_kernel(const int32_t* col, int64_t nrows, const uint32_t* deleted, long long kmin,
                                                              uint32_t range, uint32_t* presence) {
    __shared__ uint32_t sh[kMaxDirectRange / 32];
    const uint32_t words = (range + 31) / 32;
    for (uint32_t i = threadIdx.x; i < words; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (!deleted) {                                                  // 128-bit loads; the bit is almost always already set
        const int64_t nq = nrows >> 2;
        const int4* c4 = reinterpret_cast<const int4*>(col);
        for (int64_t q = r; q < nq; q += step) {
            const int4 a = __ldg(c4 + q);
            const int v[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t k = (uint32_t)((long long)v[j] - kmin);
                const uint32_t bit = 1u << (k & 31);
                if (!(sh[k >> 5] & bit)) atomicOr(&sh[k >> 5], bit);
            }
        }
        r = (nq << 2) + r;
    }
    for (; r < nrows; r += step) {
        if (deleted && ((deleted[r >> 5] >> (r & 31)) & 1u)) continue;
        const uint32_t k = (uint32_t)((long long)col[r] - kmin);
        const uint32_t bit = 1u << (k & 31);
        if (!(sh[k >> 5] & bit)) atomicOr(&sh[k >> 5], bit);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < words; i += blockDim.x)
        if (sh[i]) atomicOr(&presence[i], sh[i]);
}

// min / max AND presence in ONE pass over the column: the presence bitmap is indexed by the value's low 16 bits, which is
// injective for any column whose value range is below 65 536 -- the only case in which the bits are used (the range is
// known only after the pass: a wider column ignores them and takes the hash path).  Saves one of the three column reads of
// a small-range build (C3's G / H: 2 GB each).
__global__ void __launch_bounds__(256) column_range_presence_kernel(const int32_t* col, int64_t nrows, const uint32_t* deleted, long long* out,
                                                                    uint32_t* presence /* kMaxDirectRange bits */) {
    __shared__ uint32_t sh[kMaxDirectRange / 32];
    for (uint32_t i = threadIdx.x; i < kMaxDirectRange / 32; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    int mn = INT32_MAX, mx = INT32_MIN;                              // 32-bit min / max: one instruction each per value
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    auto take = [&](int v) {
        mn = min(mn, v);
        mx = max(mx, v);
        const uint32_t k = (uint32_t)v & (kMaxDirectRange - 1);
        const uint32_t bit = 1u << (k & 31);
        if (!(sh[k >> 5] & bit)) atomicOr(&sh[k >> 5], bit);         // the bit is almost always already set
    };
    if (!deleted) {                                                  // 128-bit loads (columns are padded to 8192 rows)
        const int64_t nq = nrows >> 2;
        const int4* c4 = reinterpret_cast<const int4*>(col);
        for (int64_t q = r; q < nq; q += step) {
            const int4 a = __ldg(c4 + q);
            take(a.x); take(a.y); take(a.z); take(a.w);
        }
        r = (nq << 2) + r;
    }
    for (; r < nrows; r += step) {
        if (deleted && ((deleted[r >> 5] >> (r & 31)) & 1u)) continue;
        take(col[r]);
    }
    for (int o = 16; o > 0; o >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xFFFFFFFFu, mn, o));
        mx = max(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
    }
    if ((threadIdx.x & 31) == 0 && mn <= mx) {
        atomicMin(out, mn);
        atomicMax(out + 1, mx);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < kMaxDirectRange / 32; i += blockDim.x)
        if (sh[i]) atomicOr(&presence[i], sh[i]);
}

__device__ __forceinline__ uint32_t hash32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}

__device__ __forceinline__ uint32_t hash_row(const uint32_t* row, int words) {
    uint32_t h = 0x811C9DC5u;
    for (int w = 0; w < words; ++w) h = hash32(h ^ row[w]);
    return h;
}

__device__ __forceinline__ bool rows_equal(const uint32_t* a, const uint32_t* b, int words) {
    for (int w = 0; w < words; ++w)
        if (a[w] != b[w]) return false;
    return true;
}

// A table is only accepted at load <= 1/2, where probe sequences are a few slots long; the cap keeps a table that fills up
// (a column with more distinct values than slots) from costing every thread a walk over all slots before it can fail.
constexpr uint32_t kMaxProbe = 4096;

// returns the slot of the value of row `r`, inserting it when INSERT; -1 when the table is full
template <bool INSERT>
__device__ __forceinline__ int probe(const HashTab& h, const void* col, int stride, bool is_str, int64_t r) {
    const uint32_t max_n = min(h.mask, kMaxProbe);
    if (!is_str) {
        const uint32_t v = reinterpret_cast<const uint32_t*>(col)[r];
        const unsigned long long key = (1ull << 32) | v;
        uint32_t s = hash32(v) & h.mask;
        for (uint32_t n = 0; n <= max_n; ++n, s = (s + 1) & h.mask) {
            unsigned long long cur = INSERT ? *reinterpret_cast<volatile unsigned long long*>(h.slots + s)
                                            : __ldg(h.slots + s);
            if (cur == key) return (int)s;
            if (cur == 0) {
                if (!INSERT) return -1;
                unsigned long long old = atomicCAS(h.slots + s, 0ull, key);
                if (old == 0 || old == key) return (int)s;
            }
        }
        return -1;
    } else {
        const int words = stride >> 2;
        const uint32_t* row = reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(col) + r * stride);
        uint32_t s = hash_row(row, words) & h.mask;
        for (uint32_t n = 0; n <= max_n; ++n, s = (s + 1) & h.mask) {
            unsigned long long cur = INSERT ? *reinterpret_cast<volatile unsigned long long*>(h.slots + s)
                                            : __ldg(h.slots + s);
            if (cur == 0) {
                if (!INSERT) return -1;
                unsigned long long old = atomicCAS(h.slots + s, 0ull, (unsigned long long)(r + 1));
                if (old == 0) return (int)s;
                cur = old;
            }
            const uint32_t* rep = reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(col) + (int64_t)(cur - 1) * stride);
            if (rows_equal(row, rep, words)) return (int)s;
        }
        return -1;
    }
}

__global__ void distinct_insert_kernel(HashTab h, const void* col, int stride, int is_str, int64_t nrows,
                                       const uint32_t* deleted, int* overflow) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (; i < nrows; i += step) {
        if (deleted && ((deleted[i >> 5] >> (i & 31)) & 1u)) continue;
        if (probe<true>(h, col, stride, is_str != 0, i) < 0) { *overflow = 1; return; }
    }
}

// ---- K3 build -------------------------------------------------------------------------------------

constexpr int kBuildThreads = 512;

struct BuildParams {
    HashTab h;
    const void* col;
    const uint32_t* deleted;
    uint32_t* bitmaps;        // [chunk][nvalues_total][chunk_rows/32]
    int64_t nvalues_total;
    int64_t nrows;
    int64_t words_pad;
    int64_t nchunks;
    int32_t stride, is_str;
    int32_t chunk_rows;       // R (multiple of 1024)
    int32_t npass;            // the values are split into npass slices of nv_per; CTA b builds slice b % npass
    int32_t nv_per;
    int32_t identity;         // direct mode and every value of [kmin, kmax] occurs: id = value - kmin
};

constexpr int kMaxPerThread = 8192 / kBuildThreads;        // rows of one chunk a thread handles (chunk_rows <= 8192)

// Fill of one chunk for <= 32 values (always chunk_rows = 8192): lane v assembles value v's word from one ballot per id
// bit, so the cost does not depend on how many distinct values a warp sees.
template <bool IDENT, bool FULL, int BITS>
__device__ __forceinline__ void fill_few_values(const BuildParams& p, uint32_t* sm, const int32_t* __restrict__ vals, int nv, int v0,
                                                int64_t row0) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inv[BITS];
#pragma unroll
    for (int k = 0; k < BITS; ++k) inv[k] = ((lane >> k) & 1) ? 0u : ~0u;
    uint32_t* mine = sm + lane * (8192 / 32);
    const int sw = (lane & 7) << 2;
    const int base = IDENT ? (int)p.h.kmin + v0 : v0;
#pragma unroll
    for (int q = 0; q < kMaxPerThread; ++q) {
        // rows past the end of the table hold the column's zero padding: the id table is only read for a row of the table
        // whose value lies inside [kmin, kmax] (0 may be far outside it)
        bool ok = FULL || row0 + threadIdx.x + q * kBuildThreads < p.nrows;
        const int32_t val = vals[threadIdx.x + q * kBuildThreads];  // the chunk's values, bulk-copied into shared memory
        int id = -1;
        if (IDENT) {
            id = val - base;
        } else {
            const uint32_t k = (uint32_t)((long long)val - p.h.kmin);
            if (ok && k < (uint32_t)p.h.range) id = (int)__ldg(p.h.id_of + k) - base;
        }
        ok = ok && (unsigned)id < (unsigned)nv;
        uint32_t w = __ballot_sync(0xFFFFFFFFu, ok);
#pragma unroll
        for (int k = 0; k < BITS; ++k) w &= __ballot_sync(0xFFFFFFFFu, (id >> k) & 1) ^ inv[k];
        if (lane < nv) mine[(warp + q * (kBuildThreads / 32)) ^ sw] = w;
    }
}

__global__ void __launch_bounds__(kBuildThreads, 2) bitmap_build_kernel(const __grid_constant__ BuildParams p) {
    extern __shared__ uint4 sm4[];
    uint32_t* sm = reinterpret_cast<uint32_t*>(sm4);
    const int pass = blockIdx.x % p.npass;                // value slices are a grid dimension, not successive launches: the
    const int v0 = pass * p.nv_per;                       // column is read once from HBM (the other slices hit L2) and one
    const int nv = (int)min((int64_t)p.nv_per, p.nvalues_total - v0);   // slice's row work overlaps another's write-out
    const int cta = blockIdx.x / p.npass, nctas = gridDim.x / p.npass;
    const int wpc = p.chunk_rows >> 5;                    // words per value per chunk
    const int total_quads = nv * wpc / 4;
    const int lane = threadIdx.x & 31;
    const int per = p.chunk_rows / kBuildThreads;         // 2..16 rows per thread per chunk
    const bool fast = p.h.direct && !p.deleted;
    const int32_t* col32 = reinterpret_cast<const int32_t*>(p.col);

    for (int i = threadIdx.x; i < total_quads; i += kBuildThreads) sm4[i] = make_uint4(0, 0, 0, 0);

    // chunks are assigned statically (no CTA depends on another); the column values of the NEXT chunk are
    // loaded while the current chunk's matrix streams out, so their HBM latency is off the critical path
    int32_t pv[kMaxPerThread];
    int64_t chunk = cta;
    if (fast && chunk < p.nchunks) {
#pragma unroll
        for (int q = 0; q < kMaxPerThread; ++q)
            if (q < per) pv[q] = col32[chunk * p.chunk_rows + threadIdx.x + q * kBuildThreads];   // columns are padded: in bounds
    }
    __syncthreads();
    // Shared-memory matrix [value][word of the chunk].  Rows are a multiple of 32 words, so the words of one chunk column
    // would all fall into ONE bank: the word index is XOR-swizzled with the value id at 16-byte granularity (8 banks
    // instead of 1; the write-out undoes it quad by quad).
    const int qshift = 31 - __clz(wpc >> 2);              // log2(quads per value row), >= 3
    for (; chunk < p.nchunks; chunk += nctas) {
        const int64_t row0 = chunk * p.chunk_rows;
        const bool full = row0 + p.chunk_rows <= p.nrows;
        if (fast) {
#pragma unroll
            for (int q = 0; q < kMaxPerThread; ++q) {
                if (q < per) {                                              // warp-uniform
                    const int r = threadIdx.x + q * kBuildThreads;          // a warp's 32 rows = one word column
                    int id = -1;
                    if (full || row0 + r < p.nrows) {
                        const uint32_t k = (uint32_t)((long long)pv[q] - p.h.kmin);
                        id = (int)(p.identity ? k : __ldg(p.h.id_of + k)) - v0;
                        if ((unsigned)id >= (unsigned)nv) id = -1;
                    }
                    const uint32_t group = __match_any_sync(0xFFFFFFFFu, id);
                    if (id >= 0 && (group & ((1u << lane) - 1)) == 0) sm[id * wpc + ((r >> 5) ^ ((id & 7) << 2))] = group;   // leader of its value group
                }
            }
        } else {
            for (int r = threadIdx.x; r < p.chunk_rows; r += kBuildThreads) {
                const int64_t row = row0 + r;
                int id = -1;
                if (row < p.nrows && !(p.deleted && ((p.deleted[row >> 5] >> (row & 31)) & 1u))) {
                    if (p.h.direct) {
                        id = (int)__ldg(p.h.id_of + (uint32_t)((long long)col32[row] - p.h.kmin)) - v0;
                    } else {
                        int s = probe<false>(p.h, p.col, p.stride, p.is_str != 0, row);
                        if (s >= 0) id = (int)p.h.slot_id[s] - v0;
                    }
                    if (id < 0 || id >= nv) id = -1;
                }
                const uint32_t group = __match_any_sync(0xFFFFFFFFu, id);
                if (id >= 0 && (group & ((1u << lane) - 1)) == 0) sm[id * wpc + ((r >> 5) ^ ((id & 7) << 2))] = group;
            }
        }
        __syncthreads();
        const int64_t next = chunk + nctas;
        if (fast && next < p.nchunks) {
#pragma unroll
            for (int q = 0; q < kMaxPerThread; ++q)
                if (q < per) pv[q] = col32[next * p.chunk_rows + threadIdx.x + q * kBuildThreads];
        }
        // chunk-major layout: this slice's values of this chunk are ONE contiguous block; the matrix is zeroed for
        // the next chunk in the same sweep
        uint4* dst4 = reinterpret_cast<uint4*>(p.bitmaps + ((int64_t)chunk * p.nvalues_total + v0) * wpc);
        for (int i = threadIdx.x; i < total_quads; i += kBuildThreads) {
            const int v = i >> qshift;
            const int src = (v << qshift) + ((i & ((1 << qshift) - 1)) ^ (v & 7));
            dst4[i] = sm4[src];
            sm4[src] = make_uint4(0, 0, 0, 0);
        }
        __syncthreads();
    }
}

template <int BITS>
__device__ __forceinline__ void fill_few_dispatch(const BuildParams& p, uint32_t* sm, const int32_t* vals, int nv, int64_t row0, bool full) {
    if (p.identity) {
        if (full) fill_few_values<true, true, BITS>(p, sm, vals, nv, 0, row0);
        else fill_few_values<true, false, BITS>(p, sm, vals, nv, 0, row0);
    } else {
        if (full) fill_few_values<false, true, BITS>(p, sm, vals, nv, 0, row0);
        else fill_few_values<false, false, BITS>(p, sm, vals, nv, 0, row0);
    }
}

// <= 32 values, direct map, no deleted rows, 8192-row chunks: the same matrix and write-out, but the column is fed by a
// ring of bulk-TMA copies (cp.async.bulk, 32 KB per chunk, completion on an mbarrier) that runs kFewStages chunks ahead (3: 1.28 -> 1.24 ms for G against 2).  The
// generic kernel prefetches ONE chunk into registers and can only issue that prefetch after the fill that consumes the
// registers, so every chunk exposed most of a DRAM round trip (measured 1.04 ms for the 500 M-row column G: 2.9 TB/s).
constexpr int kFewStages = 3;
constexpr int kFewRows = 8192;
__device__ __forceinline__ uint32_t bm_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bm_mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "BM_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra BM_DONE;\n"
        "bra BM_WAIT;\n"
        "BM_DONE:\n"
        "}" ::"r"(bm_smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bm_issue_chunk(int32_t* dst, const int32_t* src, uint64_t* bar) {
    constexpr uint32_t bytes = kFewRows * 4;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bm_smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(bm_smem_u32(dst)), "l"(src),
                 "r"(bytes), "r"(bm_smem_u32(bar))
                 : "memory");
}

__global__ void __launch_bounds__(kBuildThreads, 2) bitmap_build_few_kernel(const __grid_constant__ BuildParams p) {
    extern __shared__ uint4 sm4[];                        // [nv_per][256 words] matrix, then kFewStages x 8192 column values
    __shared__ __align__(8) uint64_t s_full[kFewStages];
    uint32_t* sm = reinterpret_cast<uint32_t*>(sm4);
    const int nv = (int)p.nvalues_total;                  // one slice: npass == 1
    constexpr int wpc = kFewRows / 32;
    const int total_quads = p.nv_per * wpc / 4;
    int32_t* ring = reinterpret_cast<int32_t*>(sm + (size_t)p.nv_per * wpc);
    const int32_t* col32 = reinterpret_cast<const int32_t*>(p.col);
    const int64_t nctas = gridDim.x;
    for (int i = threadIdx.x; i < total_quads; i += kBuildThreads) sm4[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
        for (int s = 0; s < kFewStages; ++s)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bm_smem_u32(&s_full[s])), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        for (int s = 0; s < kFewStages; ++s) {
            const int64_t c = (int64_t)blockIdx.x + s * nctas;
            if (c < p.nchunks) bm_issue_chunk(ring + (size_t)s * kFewRows, col32 + c * kFewRows, &s_full[s]);   // columns are padded: in bounds
        }
    }
    __syncthreads();
    const int qshift = 31 - __clz(wpc >> 2);
    const int bits = 32 - __clz(max(nv - 1, 1));          // id bits: 1..5
    int slot = 0;
    uint32_t phase = 0;
    for (int64_t chunk = blockIdx.x; chunk < p.nchunks; chunk += nctas) {
        const int64_t row0 = chunk * kFewRows;
        const bool full = row0 + kFewRows <= p.nrows;
        bm_mbar_wait(&s_full[slot], phase);               // this chunk's values have landed
        const int32_t* vals = ring + (size_t)slot * kFewRows;
        switch (bits) {                                   // id bits as a template parameter: straight-line ballots
            case 1: fill_few_dispatch<1>(p, sm, vals, nv, row0, full); break;
            case 2: fill_few_dispatch<2>(p, sm, vals, nv, row0, full); break;
            case 3: fill_few_dispatch<3>(p, sm, vals, nv, row0, full); break;
            case 4: fill_few_dispatch<4>(p, sm, vals, nv, row0, full); break;
            default: fill_few_dispatch<5>(p, sm, vals, nv, row0, full); break;
        }
        __syncthreads();                                  // the matrix is complete and the stage is free
        if (threadIdx.x == 0) {
            const int64_t next = chunk + kFewStages * nctas;
            if (next < p.nchunks) bm_issue_chunk(ring + (size_t)slot * kFewRows, col32 + next * kFewRows, &s_full[slot]);
        }
        uint4* dst4 = reinterpret_cast<uint4*>(p.bitmaps + chunk * p.nvalues_total * wpc);
        for (int i = threadIdx.x; i < total_quads; i += kBuildThreads) {
            const int v = i >> qshift;
            const int src = (v << qshift) + ((i & ((1 << qshift) - 1)) ^ (v & 7));
            if (v < nv) dst4[i] = sm4[src];                // (nv_per is nv rounded up to whole quads of values)
            sm4[src] = make_uint4(0, 0, 0, 0);
        }
        __syncthreads();
        if (++slot == kFewStages) { slot = 0; phase ^= 1u; }
    }
}

// ---- K4 combine -------------------------------------------------------------------------------------

constexpr int kMaxInlineBitmaps = 96;

struct BmRef {                            // one value's bitmap inside a chunk-major index
    const uint4* base;                    // first piece (chunk 0); NULL = empty bitmap (value never indexed)
    uint32_t stride_quads;                // distance between consecutive pieces, in 16-byte units
    uint32_t qshift;                      // log2(quads per piece)
};

struct CnfParams {
    int64_t nquads;                       // words_pad / 4
    uint4* out;
    const uint4* deleted;
    const BmRef* list;                    // device list when there are more than kMaxInlineBitmaps
    int32_t nconj, nbitmaps;
    int32_t conj_end[kMaxTerms];          // exclusive end index of each conjunct in the bitmap list
    BmRef inl[kMaxInlineBitmaps];
};

__global__ void __launch_bounds__(256) bitmap_cnf_kernel(const __grid_constant__ CnfParams p) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    const BmRef* list = p.list ? p.list : p.inl;
    for (; i < p.nquads; i += step) {
        uint4 acc = make_uint4(~0u, ~0u, ~0u, ~0u);
        int j = 0;
        for (int g = 0; g < p.nconj; ++g) {
            uint4 d = make_uint4(0, 0, 0, 0);
            for (; j < p.conj_end[g]; ++j) {
                const BmRef bm = list[j];
                if (bm.base) {
                    const uint4 w = __ldg(bm.base + (i >> bm.qshift) * bm.stride_quads + (i & ((1u << bm.qshift) - 1)));
                    d.x |= w.x; d.y |= w.y; d.z |= w.z; d.w |= w.w;
                }
            }
            acc.x &= d.x; acc.y &= d.y; acc.z &= d.z; acc.w &= d.w;
        }
        if (p.deleted) {
            uint4 w = __ldg(p.deleted + i);
            acc.x &= ~w.x; acc.y &= ~w.y; acc.z &= ~w.z; acc.w &= ~w.w;
        }
        p.out[i] = acc;
    }
}

// ---- sparse layout: value-sorted position lists ---------------------------------------------------------
// The live rows, stably sorted by value (mbc_sort's radix passes), form one run per distinct value.  A term on such a
// column selects at most two contiguous runs of value ids; it is materialised as one flat bitmap of the table and fed
// to bitmap_cnf_kernel like any other bitmap.

// head[i] = 1 where rows[i] starts a run: its full key (4 or stride bytes) differs from that of rows[i-1]
__global__ void __launch_bounds__(256) sparse_run_heads_kernel(const uint32_t* __restrict__ rows, int64_t n, const void* col, int stride,
                                                               uint32_t* __restrict__ head) {
    const char* base = reinterpret_cast<const char*>(col);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        uint32_t h = 1;
        if (i > 0)
            h = !rows_equal(reinterpret_cast<const uint32_t*>(base + (size_t)rows[i] * stride),
                            reinterpret_cast<const uint32_t*>(base + (size_t)rows[i - 1] * stride), stride >> 2);
        head[i] = h;
    }
}

// run d = run_of[i] of a head i starts at element i; its first row carries the value
__global__ void __launch_bounds__(256) sparse_run_starts_kernel(const uint32_t* __restrict__ head, const unsigned long long* __restrict__ run_of,
                                                                const uint32_t* __restrict__ rows, int64_t n, uint32_t* __restrict__ start,
                                                                uint32_t* __restrict__ head_row) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        if (head[i]) {
            const unsigned long long d = run_of[i];
            start[d] = (uint32_t)i;
            head_row[d] = rows[i];
        }
}

// the rows an index built now covers: below nrows and not deleted (exactly the positions of a scan without predicate)
__global__ void __launch_bounds__(256) sparse_indexed_kernel(const uint32_t* __restrict__ deleted, int64_t nrows, int64_t nwords,
                                                             uint32_t* __restrict__ indexed) {
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < nwords; w += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r0 = w * 32;
        uint32_t live = r0 + 32 <= nrows ? ~0u : r0 >= nrows ? 0u : (1u << (nrows - r0)) - 1u;
        if (deleted) live &= ~deleted[w];
        indexed[w] = live;
    }
}

// Scatter form: the bits of rows[s0, s0+n0) and rows[s1, s1+n1) are OR-ed into out (or, with CLEAR, cleared from it).
// Lanes that hit the same word are grouped with __match_any_sync and their bits merged, so a word takes one atomic per
// warp; rows of one value are ascending, so the groups are large where the runs are long.
template <bool CLEAR>
__global__ void __launch_bounds__(256) sparse_scatter_kernel(const uint32_t* __restrict__ rows, int64_t s0, int64_t n0, int64_t s1, int64_t n1,
                                                             uint32_t* out) {
    const int lane = threadIdx.x & 31;
    const int64_t total = n0 + n1;
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x - lane; i0 < total; i0 += step) {   // warp-uniform trip count
        const int64_t i = i0 + lane;
        const bool ok = i < total;
        const uint32_t r = ok ? __ldg(rows + (i < n0 ? s0 + i : s1 + (i - n0))) : 0u;
        const uint32_t word = ok ? r >> 5 : 0xFFFFFFFFu;                     // (a row id's word is below 2^27)
        const uint32_t group = __match_any_sync(0xFFFFFFFFu, word);
        const uint32_t bits = __reduce_or_sync(group, ok ? 1u << (r & 31) : 0u);
        if (ok && (group & ((1u << lane) - 1)) == 0) {
            if (CLEAR) atomicAnd(out + word, ~bits);
            else atomicOr(out + word, bits);
        }
    }
}

// Compare form: row r is selected iff its value lies in one of up to two inclusive ranges [lo, hi] of indexed values.
// Ints compare as int32, strings as stride zero-padded bytes (held here as byte-swapped words: unsigned order = byte
// order).  One warp assembles one 32-row word with a ballot and ANDs it with the rows the index covers.
struct SparseCmp {
    const void* col;
    int32_t stride, is_str, nranges;
    int32_t ilo[2], ihi[2];
    uint32_t slo[2][kMaxStrStride / 4], shi[2][kMaxStrStride / 4];
};

__device__ __forceinline__ int cmp_swapped_words(const uint32_t* row, const uint32_t* bound, int words) {
    for (int w = 0; w < words; ++w) {
        const uint32_t a = __byte_perm(row[w], 0, 0x0123), b = bound[w];
        if (a != b) return a < b ? -1 : 1;
    }
    return 0;
}

__global__ void __launch_bounds__(256) sparse_compare_kernel(const __grid_constant__ SparseCmp p, const uint32_t* __restrict__ indexed,
                                                             int64_t nwords, uint32_t* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (!p.is_str) {
        // 128 rows (4 words) per warp and step: lane l loads rows 4l..4l+3 with one 128-bit load (one 4-byte load per lane
        // and word measured 0.31 ms for 100 M rows, 1.4 TB/s); the 8 lanes of a word OR their nibbles together
        auto in = [&](int v) {
            bool s = false;
            for (int k = 0; k < p.nranges; ++k) s |= v >= p.ilo[k] && v <= p.ihi[k];
            return (uint32_t)s;
        };
        const int4* col4 = reinterpret_cast<const int4*>(p.col);
        for (int64_t q = warp; q < nwords / 4; q += nwarps) {                // nwords = words_pad, a multiple of 256
            const int4 v = __ldg(col4 + q * 32 + lane);
            uint32_t part = (in(v.x) | in(v.y) << 1 | in(v.z) << 2 | in(v.w) << 3) << (4 * (lane & 7));
            part |= __shfl_xor_sync(0xFFFFFFFFu, part, 1);
            part |= __shfl_xor_sync(0xFFFFFFFFu, part, 2);
            part |= __shfl_xor_sync(0xFFFFFFFFu, part, 4);
            const int64_t w = q * 4 + (lane >> 3);
            if ((lane & 7) == 0) out[w] = part & __ldg(indexed + w);
        }
        return;
    }
    const int words = p.stride >> 2;
    for (int64_t w = warp; w < nwords; w += nwarps) {
        const int64_t r = w * 32 + lane;                                      // < nrows_pad: columns are padded
        const uint32_t* row = reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(p.col) + (size_t)r * p.stride);
        bool sel = false;
        for (int k = 0; k < p.nranges; ++k)
            sel |= cmp_swapped_words(row, p.slo[k], words) >= 0 && cmp_swapped_words(row, p.shi[k], words) <= 0;
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, sel);
        if (lane == 0) out[w] = m & __ldg(indexed + w);
    }
}

// ---- host side ----------------------------------------------------------------------------------------

static int cmp_bytes(const uint8_t* a, const uint8_t* b, int n) { return memcmp(a, b, n); }

static int grid_for(const mbc_ctx* ctx, int64_t n) {
    return (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8));
}

// Sparse layout of column `col` (see BitmapIndex): the live rows from a scan without predicate, stably sorted by value,
// cut into runs.  Device time of every step goes into mbc_last_kernel_ms, added to that of any dense attempt before it.
static int32_t build_sparse(mbc_table* t, int col) {
    if (t->nrows > (int64_t)UINT32_MAX) MBC_FAIL(MBC_ERR_UNSUPPORTED, "bitmap index: more than 2^32 rows in one table");
    mbc_ctx* ctx = t->ctx;
    BitmapIndex& bi = t->bm[col];
    const Column& c = t->cols[col];
    mbc_result* all = nullptr;
    uint32_t *rows = nullptr, *keys = nullptr, *bits = nullptr, *start = nullptr, *head_row = nullptr, *indexed = nullptr;
    unsigned long long* run_of = nullptr;
    void* dvals = nullptr;
    auto release = [&]() {
        for (void* p : {(void*)keys, (void*)bits, (void*)start, (void*)head_row, (void*)run_of, dvals}) dev_free(ctx, p);
        if (all) mbc_result_free(all);
    };
    auto fail = [&](int32_t s) {
        dev_free(ctx, rows);
        dev_free(ctx, indexed);
        release();
        return s;
    };
#define SPTRY(x) do { int32_t _s = (x); if (_s != MBC_OK) return fail(_s); } while (0)
#define SPCUDA(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) return fail((set_error("bitmap index (sparse): %s", cudaGetErrorString(_e)), MBC_ERR_CUDA)); } while (0)
    ScanRequest rq;
    rq.table = t;
    rq.want = MBC_WANT_POSITIONS;
    SPTRY(run_scan(rq, &all));
    const int64_t n = all->count;
    split_timing(ctx);                                      // the scan's kernels count, the host wait in between does not
    begin_timing(ctx);
    SPTRY(dev_alloc(ctx, (void**)&rows, (size_t)n * 4, false));
    SPTRY(dev_alloc(ctx, (void**)&keys, (size_t)n * 4, false));           // sort keys, then the head flags
    SPTRY(dev_alloc(ctx, (void**)&bits, 8, false));
    SPTRY(dev_alloc(ctx, (void**)&run_of, (size_t)(n + 1) * 8, false));
    SPTRY(dev_alloc(ctx, (void**)&indexed, (size_t)t->words_pad * 4, false));
    const int grid = grid_for(ctx, n);
    if (n > 0) {
        sort_rows_from_positions_kernel<<<grid, 256, 0, ctx->stream>>>(all->d_pos, n, t->pos_base, rows);
        ctx->launches++;
        SPTRY(sort_rows_by_column(ctx, rows, n, c, false, keys, bits));
        sparse_run_heads_kernel<<<grid, 256, 0, ctx->stream>>>(rows, n, c.d, c.stride, keys);
        ctx->launches++;
    }
    SPTRY(exclusive_scan_u32(ctx, keys, n, run_of));
    unsigned long long D = 0;
    SPCUDA(cudaMemcpyAsync(&D, run_of + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    SPCUDA(cudaStreamSynchronize(ctx->stream));
    SPTRY(dev_alloc(ctx, (void**)&start, (size_t)D * 4, false));
    SPTRY(dev_alloc(ctx, (void**)&head_row, (size_t)D * 4, false));
    SPTRY(dev_alloc(ctx, &dvals, (size_t)D * c.stride, false));
    if (n > 0) {
        sparse_run_starts_kernel<<<grid, 256, 0, ctx->stream>>>(keys, run_of, rows, n, start, head_row);
        sort_gather_kernel<<<grid_for(ctx, (int64_t)D), 256, 0, ctx->stream>>>(head_row, (int64_t)D, c.d, c.stride, dvals);
        ctx->launches += 2;
    }
    sparse_indexed_kernel<<<grid_for(ctx, t->words_pad), 256, 0, ctx->stream>>>(t->has_deleted ? t->d_deleted : nullptr, t->nrows,
                                                                                t->words_pad, indexed);
    ctx->launches++;
    end_timing(ctx);
    SPCUDA(cudaGetLastError());
    std::vector<uint32_t> offsets((size_t)D + 1);
    std::vector<uint8_t> vals((size_t)D * c.stride);
    SPCUDA(cudaMemcpyAsync(offsets.data(), start, (size_t)D * 4, cudaMemcpyDeviceToHost, ctx->stream));
    SPCUDA(cudaMemcpyAsync(vals.data(), dvals, vals.size(), cudaMemcpyDeviceToHost, ctx->stream));
    SPCUDA(cudaStreamSynchronize(ctx->stream));
#undef SPTRY
#undef SPCUDA
    offsets[D] = (uint32_t)n;
    bi.ivals.clear();
    bi.svals.clear();
    if (c.type == MBC_ATTR_STRING) {
        bi.svals.resize((size_t)D * c.width);
        for (size_t k = 0; k < D; ++k) memcpy(bi.svals.data() + k * c.width, vals.data() + k * c.stride, c.width);
    } else {
        bi.ivals.resize(D);
        memcpy(bi.ivals.data(), vals.data(), (size_t)D * 4);
    }
    bi.nvalues = (int64_t)D;
    bi.offsets = std::move(offsets);
    bi.d_rows = rows;
    bi.d_indexed = indexed;
    bi.n_indexed = n;
    bi.sparse = true;
    bi.exists = true;
    release();
    MBC_CUDA(cudaStreamSynchronize(ctx->stream));
    return MBC_OK;
}

// MBC_BM_SPARSE=1: every index takes the sparse layout whenever it is legal (tests, profiling)
static bool sparse_forced() {
    const char* e = getenv("MBC_BM_SPARSE");
    return e && strcmp(e, "1") == 0;
}

}  // namespace mbc

using namespace mbc;

extern "C" int32_t mbc_bitmap_exists(const mbc_table* t, int32_t col) {
    if (!t || col < 0 || col >= (int)t->cols.size()) return 0;
    return t->bm[col].exists ? 1 : 0;
}

extern "C" int32_t mbc_bitmap_build(mbc_table* t, int32_t col) {
    if (!t || col < 0 || col >= (int)t->cols.size()) MBC_FAIL(MBC_ERR_ARG, "mbc_bitmap_build: bad column");
    mbc_ctx* ctx = t->ctx;
    MBC_CUDA(cudaSetDevice(ctx->device));
    BitmapIndex& bi = t->bm[col];
    if (bi.exists) return MBC_OK;                       // Columnarfile.java:699: no-op when it exists
    const Column& c = t->cols[col];
    if (c.type == MBC_ATTR_REAL) MBC_FAIL(MBC_ERR_UNSUPPORTED, "bitmap index on a real column (the reference indexes int and string only)");
    if (sparse_forced()) return build_sparse(t, col);
    const bool is_str = c.type == MBC_ATTR_STRING;
    const uint32_t* deleted = t->has_deleted ? t->d_deleted : nullptr;

    // 1. distinct values
    HashTab h{};
    int* d_overflow = nullptr;
    MBC_TRY(dev_alloc(ctx, (void**)&d_overflow, 4, true));
    std::vector<unsigned long long> slots;
    uint32_t cap = 0;
    bool direct = false;
    std::vector<uint32_t> id_of_host;
    if (!is_str && t->nrows > 0) {
        long long* d_mm = nullptr;
        uint32_t* d_presence = nullptr;
        MBC_TRY(dev_alloc(ctx, (void**)&d_mm, 16, false));
        long long init[2] = {INT64_MAX, INT64_MIN}, mm[2];
        MBC_CUDA(cudaMemcpyAsync(d_mm, init, 16, cudaMemcpyHostToDevice, ctx->stream));
        MBC_TRY(dev_alloc(ctx, (void**)&d_presence, kMaxDirectRange / 8, true));
        begin_timing(ctx);
        const int grid = (int)std::min<int64_t>((t->nrows + 255) / 256, (int64_t)ctx->sm_count * 8);
        column_range_presence_kernel<<<grid, 256, 0, ctx->stream>>>((const int32_t*)c.d, t->nrows, deleted, d_mm, d_presence);
        ctx->launches++;
        split_timing(ctx);
        std::vector<uint32_t> pres_mod(kMaxDirectRange / 32);
        MBC_CUDA(cudaMemcpyAsync(mm, d_mm, 16, cudaMemcpyDeviceToHost, ctx->stream));
        MBC_CUDA(cudaMemcpyAsync(pres_mod.data(), d_presence, kMaxDirectRange / 8, cudaMemcpyDeviceToHost, ctx->stream));
        MBC_CUDA(cudaStreamSynchronize(ctx->stream));
        dev_free(ctx, d_mm);
        dev_free(ctx, d_presence);
        if (mm[0] <= mm[1] && mm[1] - mm[0] < (long long)kMaxDirectRange) {
            direct = true;
            h.direct = 1;
            h.kmin = mm[0];
            h.range = (uint32_t)(mm[1] - mm[0] + 1);
            const uint32_t words = (h.range + 31) / 32;
            std::vector<uint32_t> pres(words, 0u);
            for (uint32_t k = 0; k < h.range; ++k) {                // value kmin + k sits at its low 16 bits in the modular bitmap
                const uint32_t m = (uint32_t)(h.kmin + k) & (kMaxDirectRange - 1);
                if ((pres_mod[m >> 5] >> (m & 31)) & 1u) pres[k >> 5] |= 1u << (k & 31);
            }
            id_of_host.assign(h.range, 0xFFFFFFFFu);
            bi.ivals.clear();
            bi.svals.clear();
            for (uint32_t k = 0; k < h.range; ++k)
                if ((pres[k >> 5] >> (k & 31)) & 1u) {
                    id_of_host[k] = (uint32_t)bi.ivals.size();
                    bi.ivals.push_back((int32_t)(h.kmin + k));
                }
            bi.nvalues = (int64_t)bi.ivals.size();
        }
    }
    for (uint32_t try_cap : {1u << 12, 1u << 16, 1u << 20}) {
        if (direct) break;
        cap = try_cap;
        MBC_TRY(dev_alloc(ctx, (void**)&h.slots, (size_t)cap * 8, true));
        h.mask = cap - 1;
        MBC_CUDA(cudaMemsetAsync(d_overflow, 0, 4, ctx->stream));
        begin_timing(ctx);
        if (t->nrows > 0) {
            int grid = (int)std::min<int64_t>((t->nrows + 255) / 256, (int64_t)ctx->sm_count * 8);
            distinct_insert_kernel<<<grid, 256, 0, ctx->stream>>>(h, c.d, c.stride, is_str, t->nrows, deleted, d_overflow);
            ctx->launches++;
        }
        split_timing(ctx);
        int overflow = 0;
        MBC_CUDA(cudaMemcpyAsync(&overflow, d_overflow, 4, cudaMemcpyDeviceToHost, ctx->stream));
        slots.resize(cap);
        MBC_CUDA(cudaMemcpyAsync(slots.data(), h.slots, (size_t)cap * 8, cudaMemcpyDeviceToHost, ctx->stream));
        MBC_CUDA(cudaStreamSynchronize(ctx->stream));
        size_t used = 0;
        for (auto s : slots) used += s != 0;
        if (!overflow && used <= cap / 2) break;
        dev_free(ctx, h.slots);
        h.slots = nullptr;
        if (try_cap == (1u << 20)) {                    // more than 2^19 distinct values: position lists instead
            dev_free(ctx, d_overflow);
            return build_sparse(t, col);
        }
    }
    dev_free(ctx, d_overflow);

    // 2. sort the values, give every slot its dense id
    uint32_t* d_id_of = nullptr;
    if (direct) {
        MBC_TRY(dev_alloc(ctx, (void**)&d_id_of, (size_t)h.range * 4, false));
        MBC_CUDA(cudaMemcpyAsync(d_id_of, id_of_host.data(), (size_t)h.range * 4, cudaMemcpyHostToDevice, ctx->stream));
        h.id_of = d_id_of;
    }
    std::vector<int> used_slots;
    for (uint32_t s = 0; s < cap; ++s) if (slots[s]) used_slots.push_back((int)s);
    const int64_t D = direct ? bi.nvalues : (int64_t)used_slots.size();
    std::vector<uint8_t> rep_bytes;                      // strings: representative rows
    if (is_str && D > 0) {
        rep_bytes.resize((size_t)D * c.stride);
        for (int64_t k = 0; k < D; ++k) {
            int64_t row = (int64_t)slots[used_slots[k]] - 1;
            MBC_CUDA(cudaMemcpyAsync(rep_bytes.data() + k * c.stride, (const char*)c.d + row * c.stride, c.stride,
                                     cudaMemcpyDeviceToHost, ctx->stream));
        }
        MBC_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    std::vector<int> order(direct ? 0 : D);
    std::iota(order.begin(), order.end(), 0);
    if (is_str) {
        std::sort(order.begin(), order.end(), [&](int a, int b) {
            return cmp_bytes(rep_bytes.data() + (size_t)a * c.stride, rep_bytes.data() + (size_t)b * c.stride, c.stride) < 0;
        });
    } else {
        std::sort(order.begin(), order.end(), [&](int a, int b) {
            return (int32_t)(uint32_t)slots[used_slots[a]] < (int32_t)(uint32_t)slots[used_slots[b]];
        });
    }
    std::vector<uint32_t> slot_id(cap, 0xFFFFFFFFu);
    if (!direct) {
        bi.ivals.clear();
        bi.svals.clear();
    }
    for (int64_t k = 0; k < (direct ? 0 : D); ++k) {
        int src = order[k];
        slot_id[used_slots[src]] = (uint32_t)k;
        if (is_str) bi.svals.insert(bi.svals.end(), rep_bytes.begin() + (size_t)src * c.stride,
                                    rep_bytes.begin() + (size_t)src * c.stride + c.width);
        else bi.ivals.push_back((int32_t)(uint32_t)slots[used_slots[src]]);
    }
    bi.nvalues = D;
    if (!direct) {
        MBC_TRY(dev_alloc(ctx, (void**)&h.slot_id, (size_t)cap * 4, false));
        MBC_CUDA(cudaMemcpyAsync(h.slot_id, slot_id.data(), (size_t)cap * 4, cudaMemcpyHostToDevice, ctx->stream));
    }

    // 3. build
    if (D > 0) {
        size_t free_b = 0, total_b = 0;
        MBC_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const size_t need = (size_t)D * t->words_pad * 4;
        // per-value bitsets larger than the device, or than what it can give now: position lists instead
        // (the stream-ordered pool may already hold reusable memory, so only the allocation itself tells)
        cudaError_t ae = need > total_b ? cudaErrorMemoryAllocation : cudaMallocAsync((void**)&bi.d_words, need, ctx->stream);
        if (ae == cudaErrorMemoryAllocation) {
            cudaGetLastError();
            bi.d_words = nullptr;
            dev_free(ctx, h.slots);
            dev_free(ctx, h.slot_id);
            dev_free(ctx, d_id_of);
            return build_sparse(t, col);
        }
        MBC_CUDA(ae);
        const size_t smem_budget = 100 * 1024;                    // two CTAs per SM: one streams out while the other fills
        // rows per chunk: as many as fit for the values of one pass, power of two in [1024, 8192]
        int R = 8192;
        while (R > 1024 && (size_t)std::min<int64_t>(D, 4096) * (R / 8) > smem_budget) R >>= 1;
        if (const char* e = getenv("MBC_BM_CHUNK_ROWS")) {          // tuning knob: longer per-value segments, more passes
            int v = atoi(e);
            if (v == 1024 || v == 2048 || v == 4096 || v == 8192) R = v;
        }
        const int max_nv = (int)std::min<int64_t>(D, (int64_t)(smem_budget / (R / 8)));
        bi.chunk_rows = R;
        MBC_CUDA(cudaFuncSetAttribute(bitmap_build_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_budget));
        MBC_CUDA(cudaStreamSynchronize(ctx->stream));        // the allocation above is not kernel time
        begin_timing(ctx);
        {
            BuildParams p{};
            p.h = h;
            p.col = c.d;
            p.deleted = deleted;
            p.bitmaps = bi.d_words;
            p.nvalues_total = D;
            p.nrows = t->nrows;
            p.words_pad = t->words_pad;
            p.chunk_rows = R;
            p.nchunks = t->nrows_pad / R;                // nrows_pad is a multiple of kPadRows = 8192 >= R
            p.stride = c.stride;
            p.is_str = is_str;
            p.npass = (int)((D + max_nv - 1) / max_nv);
            p.nv_per = (int)(((D + p.npass - 1) / p.npass + 3) & ~3ll);       // even slices, whole quads
            p.npass = (int)((D + p.nv_per - 1) / p.nv_per);
            p.identity = direct && D == (int64_t)h.range;
            size_t smem = (size_t)p.nv_per * (R / 8);
            const bool few = direct && !deleted && D <= 32 && R == kFewRows && p.npass == 1 && !getenv("MBC_BM_FEW_OFF");
            if (few) {
                // <= 32 values: the column comes through a TMA ring (bitmap_build_few_kernel)
                smem += (size_t)kFewStages * kFewRows * 4;
                MBC_CUDA(cudaFuncSetAttribute(bitmap_build_few_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                int per_sm = 1;
                if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bitmap_build_few_kernel, kBuildThreads, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
                const int64_t grid = std::max<int64_t>(1, std::min<int64_t>(p.nchunks, (int64_t)ctx->sm_count * per_sm));
                bitmap_build_few_kernel<<<(int)grid, kBuildThreads, smem, ctx->stream>>>(p);
            } else {
                int per_sm = 1;
                if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bitmap_build_kernel, kBuildThreads, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
                int64_t grid = std::min<int64_t>(p.nchunks * p.npass, (int64_t)ctx->sm_count * per_sm);
                grid = std::max<int64_t>(grid / p.npass, 1) * p.npass;           // every chunk stride carries all slices
                bitmap_build_kernel<<<(int)grid, kBuildThreads, smem, ctx->stream>>>(p);
            }
            ctx->launches++;
        }
        end_timing(ctx);
    } else {
        begin_timing(ctx);
        end_timing(ctx);
    }
    MBC_CUDA(cudaGetLastError());
    MBC_CUDA(cudaStreamSynchronize(ctx->stream));
    dev_free(ctx, h.slots);
    dev_free(ctx, h.slot_id);
    dev_free(ctx, d_id_of);
    bi.exists = true;
    return MBC_OK;
}

extern "C" int32_t mbc_bitmap_layout(const mbc_table* t, int32_t col, int64_t* device_bytes) {
    if (!t || col < 0 || col >= (int)t->cols.size()) MBC_FAIL(MBC_ERR_ARG, "mbc_bitmap_layout: bad column");
    const BitmapIndex& bi = t->bm[col];
    int64_t bytes = 0;
    int32_t layout = MBC_BITMAP_NONE;
    if (bi.exists && bi.sparse) {
        layout = MBC_BITMAP_SPARSE;
        bytes = std::max<int64_t>(bi.n_indexed, 4) * 4 + t->words_pad * 4;       // (an empty allocation takes 16 bytes)
    } else if (bi.exists) {
        layout = MBC_BITMAP_DENSE;
        bytes = bi.nvalues * t->words_pad * 4;
    }
    if (device_bytes) *device_bytes = bytes;
    return layout;
}

extern "C" int32_t mbc_bitmap_values(mbc_table* t, int32_t col, const void** values, int64_t* n) {
    if (!t || col < 0 || col >= (int)t->cols.size() || !values || !n) MBC_FAIL(MBC_ERR_ARG, "mbc_bitmap_values: bad argument");
    const BitmapIndex& bi = t->bm[col];
    if (!bi.exists) MBC_FAIL(MBC_ERR_NOINDEX, "column %d has no bitmap index", col);
    *n = bi.nvalues;
    *values = t->cols[col].type == MBC_ATTR_STRING ? (const void*)bi.svals.data() : (const void*)bi.ivals.data();
    return MBC_OK;
}

namespace mbc {

// index of `value` among the sorted distinct values, or -1
static int64_t find_value(const mbc_table* t, int col, const void* value) {
    const BitmapIndex& bi = t->bm[col];
    const Column& c = t->cols[col];
    if (c.type == MBC_ATTR_STRING) {
        const uint8_t* v = (const uint8_t*)value;
        int64_t lo = 0, hi = bi.nvalues;
        while (lo < hi) {
            int64_t mid = (lo + hi) / 2;
            int r = memcmp(bi.svals.data() + mid * c.width, v, c.width);
            if (r == 0) return mid;
            if (r < 0) lo = mid + 1; else hi = mid;
        }
        return -1;
    }
    int32_t v = *(const int32_t*)value;
    auto it = std::lower_bound(bi.ivals.begin(), bi.ivals.end(), v);
    if (it == bi.ivals.end() || *it != v) return -1;
    return it - bi.ivals.begin();
}

}  // namespace mbc

extern "C" int32_t mbc_bitmap_get(mbc_table* t, int32_t col, const void* value, uint64_t* out_words, int64_t nwords) {
    if (!t || col < 0 || col >= (int)t->cols.size() || !value || (!out_words && nwords > 0))
        MBC_FAIL(MBC_ERR_ARG, "mbc_bitmap_get: bad argument");
    const BitmapIndex& bi = t->bm[col];
    if (!bi.exists) MBC_FAIL(MBC_ERR_NOINDEX, "column %d has no bitmap index", col);
    MBC_CUDA(cudaSetDevice(t->ctx->device));
    memset(out_words, 0, (size_t)nwords * 8);
    int64_t k = find_value(t, col, value);
    if (k < 0) return MBC_OK;                            // Columnarfile.java:1103-1127: empty BitMapFile
    mbc_ctx* ctx = t->ctx;
    if (bi.sparse) {                                     // the value's run of row ids scattered into a zeroed bitmap
        uint32_t* d = nullptr;
        MBC_TRY(dev_alloc(ctx, (void**)&d, (size_t)t->words_pad * 4, true));
        const int64_t s = bi.offsets[k], len = (int64_t)bi.offsets[k + 1] - s;
        sparse_scatter_kernel<false><<<grid_for(ctx, len), 256, 0, ctx->stream>>>(bi.d_rows, s, len, 0, 0, d);
        ctx->launches++;
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(out_words, d, (size_t)std::min<int64_t>(nwords * 8, t->words_pad * 4), cudaMemcpyDeviceToHost, ctx->stream);
        dev_free(ctx, d);
        MBC_CUDA(e);
        MBC_CUDA(cudaStreamSynchronize(ctx->stream));
        return MBC_OK;
    }
    // the value's bitmap is one chunk_rows/8-byte piece per chunk: a pitched copy gathers them
    const int64_t wpc = bi.chunk_rows / 32;
    const int64_t nchunks = t->nrows_pad / bi.chunk_rows;
    std::vector<uint32_t> tmp((size_t)(nchunks * wpc));
    MBC_CUDA(cudaMemcpy2DAsync(tmp.data(), (size_t)wpc * 4, bi.d_words + k * wpc, (size_t)bi.nvalues * wpc * 4, (size_t)wpc * 4,
                               (size_t)nchunks, cudaMemcpyDeviceToHost, t->ctx->stream));
    MBC_CUDA(cudaStreamSynchronize(t->ctx->stream));
    memcpy(out_words, tmp.data(), (size_t)std::min<int64_t>(nwords * 8, (int64_t)tmp.size() * 4));
    return MBC_OK;
}

namespace mbc {

// ColumnIndexScan.java:656-740: which indexed values does `column op literal` select?
static bool value_selected(int op, int cmp /* sign of compare(indexed value, literal) */) {
    switch (op) {
        case MBC_OP_EQ: return cmp == 0;
        case MBC_OP_LT: return cmp < 0;
        case MBC_OP_LE: return cmp <= 0;
        case MBC_OP_GT: return cmp > 0;
        case MBC_OP_GE: return cmp >= 0;
        case MBC_OP_NE: return cmp != 0;
        default: return false;                           // getBitSet() has no branch for aopNOT/NOP/RANGE: empty set
    }
}

static BmRef bm_ref(const BitmapIndex& bi, int64_t v) {
    BmRef r;
    const uint32_t wpc = (uint32_t)bi.chunk_rows / 32;
    r.base = reinterpret_cast<const uint4*>(bi.d_words + v * wpc);
    r.stride_quads = (uint32_t)(bi.nvalues * wpc / 4);
    r.qshift = 0;
    while ((1u << r.qshift) < wpc / 4) ++r.qshift;
    return r;
}

struct IdRange { int64_t lo, hi; };                     // value ids [lo, hi)

// Bytes of column read that cost as much device time as scattering one row's bit.  Measured on 100 M rows
// (scripts/bench_bitmap_sparse.py, DESIGN.md section 5): a scattered row 23 ps, the compare form 1.45 ps per int row and
// 3.55 ps per char(16) row, i.e. 68 and 106 bytes of column per scattered row; 85 puts the switch at 5 % of the rows for
// ints and 19 % for char(16).
constexpr double kScatterRowBytes = 85.0;

// A term on a sparse column as one flat bitmap of the table (a BmRef of a single piece).  Scatter touches the selected
// rows, or starts from the covered rows and clears the unselected ones when those are fewer; compare reads the whole
// column against the boundary values of the ranges.  Compare is taken when the rows to touch cost more than that read.
// MBC_BM_SPARSE_FORM=scatter|compare forces a form (tests, profiling); MBC_BM_SPARSE_TRACE prints the choice on stderr.
static int32_t sparse_term_bitmap(mbc_table* t, int col, const IdRange* rg, int nr, BmRef* ref, std::vector<void*>* temps) {
    mbc_ctx* ctx = t->ctx;
    const BitmapIndex& bi = t->bm[col];
    const Column& c = t->cols[col];
    int64_t sel = 0;
    for (int k = 0; k < nr; ++k) sel += (int64_t)bi.offsets[rg[k].hi] - bi.offsets[rg[k].lo];
    const int64_t unsel = bi.n_indexed - sel;
    const char* form = "empty";
    *ref = BmRef{nullptr, 0, 0};
    if (sel > 0 && unsel == 0) {
        *ref = BmRef{reinterpret_cast<const uint4*>(bi.d_indexed), 0, 31};
        form = "all indexed rows";
    } else if (sel > 0) {
        const bool complement = unsel < sel;
        const int64_t touch = complement ? unsel : sel;
        bool compare = (double)touch * kScatterRowBytes > (double)t->nrows * (c.stride + 0.25);
        if (const char* f = getenv("MBC_BM_SPARSE_FORM")) {
            if (!strcmp(f, "scatter")) compare = false;
            else if (!strcmp(f, "compare")) compare = true;
        }
        uint32_t* out = nullptr;
        MBC_TRY(dev_alloc(ctx, (void**)&out, (size_t)t->words_pad * 4, false));
        temps->push_back(out);
        if (compare) {
            SparseCmp p{};
            p.col = c.d;
            p.stride = c.stride;
            p.is_str = c.type == MBC_ATTR_STRING;
            p.nranges = nr;
            for (int k = 0; k < nr; ++k) {
                if (!p.is_str) {
                    p.ilo[k] = bi.ivals[rg[k].lo];
                    p.ihi[k] = bi.ivals[rg[k].hi - 1];
                    continue;
                }
                for (int b = 0; b < c.width; ++b) {              // zero padded to the stride, big-endian words
                    const int sh = 8 * (3 - (b & 3));
                    p.slo[k][b >> 2] |= (uint32_t)bi.svals[(size_t)rg[k].lo * c.width + b] << sh;
                    p.shi[k][b >> 2] |= (uint32_t)bi.svals[(size_t)(rg[k].hi - 1) * c.width + b] << sh;
                }
            }
            sparse_compare_kernel<<<grid_for(ctx, t->words_pad * 32), 256, 0, ctx->stream>>>(p, bi.d_indexed, t->words_pad, out);
            form = "compare";
        } else {
            IdRange w[3];                                        // the ranges to scatter: the selected ones or the gaps between them
            int nw = 0;
            if (complement) {
                int64_t prev = 0;
                for (int k = 0; k < nr; ++k) {
                    if (prev < rg[k].lo) w[nw++] = {prev, rg[k].lo};
                    prev = rg[k].hi;
                }
                if (prev < bi.nvalues) w[nw++] = {prev, bi.nvalues};
            } else {
                for (int k = 0; k < nr; ++k) w[nw++] = rg[k];
            }
            // (selections are a prefix, a suffix, one middle run or prefix + suffix: never more than two gaps)
            const int64_t s0 = bi.offsets[w[0].lo], n0 = (int64_t)bi.offsets[w[0].hi] - s0;
            const int64_t s1 = nw > 1 ? bi.offsets[w[1].lo] : 0, n1 = nw > 1 ? (int64_t)bi.offsets[w[1].hi] - s1 : 0;
            if (complement) {
                MBC_CUDA(cudaMemcpyAsync(out, bi.d_indexed, (size_t)t->words_pad * 4, cudaMemcpyDeviceToDevice, ctx->stream));
                sparse_scatter_kernel<true><<<grid_for(ctx, touch), 256, 0, ctx->stream>>>(bi.d_rows, s0, n0, s1, n1, out);
                form = "scatter (clear the complement)";
            } else {
                MBC_CUDA(cudaMemsetAsync(out, 0, (size_t)t->words_pad * 4, ctx->stream));
                sparse_scatter_kernel<false><<<grid_for(ctx, touch), 256, 0, ctx->stream>>>(bi.d_rows, s0, n0, s1, n1, out);
                form = "scatter";
            }
        }
        ctx->launches++;
        MBC_CUDA(cudaGetLastError());
        *ref = BmRef{reinterpret_cast<const uint4*>(out), 0, 31};
    }
    if (getenv("MBC_BM_SPARSE_TRACE"))
        fprintf(stderr, "[mbc] sparse bitmap term on column %d: %lld of %lld indexed rows, %s\n", col, (long long)sel,
                (long long)bi.n_indexed, form);
    return MBC_OK;
}

int32_t resolve_bitmap_terms(mbc_table* t, const mbc_term* terms, int32_t nterms, std::vector<BmRef>* list,
                             std::vector<int>* conj_end, std::vector<void*>* temps) {
    if (nterms <= 0) MBC_FAIL(MBC_ERR_ARG, "bitmap scan needs at least one term (ColumnarIndexScan dereferences selects[0])");
    for (int k = 0; k < nterms; ++k) {
        const mbc_term& s = terms[k];
        if (k > 0 && s.conj_id < terms[k - 1].conj_id) MBC_FAIL(MBC_ERR_ARG, "terms must be sorted by conj_id");
        if (k > 0 && s.conj_id != terms[k - 1].conj_id) conj_end->push_back((int)list->size());
        // ColumnarIndexScan.java:137-142: exactly one side is a column; the literal is operand2
        if (s.lhs.kind != MBC_OPERAND_OUTER || s.rhs.kind != MBC_OPERAND_LITERAL)
            MBC_FAIL(MBC_ERR_ARG, "bitmap term %d must be `column op literal`", k);
        int col = s.lhs.col;
        if (col < 0 || col >= (int)t->cols.size()) MBC_FAIL(MBC_ERR_ARG, "bitmap term %d: column %d out of range", k, col);
        const BitmapIndex& bi = t->bm[col];
        if (!bi.exists) MBC_FAIL(MBC_ERR_NOINDEX, "bitmap term %d: column %d has no bitmap index", k, col);
        const Column& c = t->cols[col];
        std::vector<uint8_t> lit;
        if (c.type == MBC_ATTR_STRING) {
            if (s.rhs.type != MBC_ATTR_STRING) MBC_FAIL(MBC_ERR_ARG, "bitmap term %d: string column needs a string literal", k);
            lit.assign(std::max(c.width, s.rhs.lit_slen), 0);
            if (s.rhs.lit_slen) memcpy(lit.data(), s.rhs.lit_s, s.rhs.lit_slen);
        } else if (s.rhs.type != MBC_ATTR_INTEGER) {
            MBC_FAIL(MBC_ERR_ARG, "bitmap term %d: int column needs an int literal", k);
        }
        // sign of compare(indexed value v, literal): String.compareTo over zero padded bytes, where an over-long literal
        // can only be greater on a tie; ints numerically
        auto value_cmp = [&](int64_t v) {
            if (c.type == MBC_ATTR_STRING) {
                int cmp = memcmp(bi.svals.data() + v * c.width, lit.data(), c.width);
                if (cmp == 0 && s.rhs.lit_slen > c.width) cmp = -1;
                return cmp;
            }
            return bi.ivals[v] < s.rhs.lit_i ? -1 : bi.ivals[v] > s.rhs.lit_i ? 1 : 0;
        };
        if (bi.sparse) {
            // the values are sorted, so value_cmp is monotone: a = first value not below the literal, b = first above it
            auto first_where = [&](auto pred) {
                int64_t lo = 0, hi = bi.nvalues;
                while (lo < hi) {
                    const int64_t m = lo + (hi - lo) / 2;
                    if (pred(m)) hi = m; else lo = m + 1;
                }
                return lo;
            };
            const int64_t a = first_where([&](int64_t v) { return value_cmp(v) >= 0; });
            const int64_t b = first_where([&](int64_t v) { return value_cmp(v) > 0; });
            IdRange rg[2];
            int nr = 0;
            auto take = [&](int64_t lo, int64_t hi) { if (lo < hi) rg[nr++] = {lo, hi}; };
            switch (s.op) {                              // the value ids value_selected() accepts
                case MBC_OP_EQ: take(a, b); break;
                case MBC_OP_LT: take(0, a); break;
                case MBC_OP_LE: take(0, b); break;
                case MBC_OP_GT: take(b, bi.nvalues); break;
                case MBC_OP_GE: take(a, bi.nvalues); break;
                case MBC_OP_NE: take(0, a); take(b, bi.nvalues); break;
                default: break;
            }
            BmRef r;
            MBC_TRY(sparse_term_bitmap(t, col, rg, nr, &r, temps));
            list->push_back(r);
            continue;
        }
        const size_t before = list->size();
        for (int64_t v = 0; v < bi.nvalues; ++v)
            if (value_selected(s.op, value_cmp(v))) list->push_back(bm_ref(bi, v));
        if (list->size() == before) list->push_back(BmRef{nullptr, 0, 0});   // nothing selected: an empty bitset takes the term's place
    }
    conj_end->push_back((int)list->size());
    if ((int)conj_end->size() > kMaxTerms) MBC_FAIL(MBC_ERR_UNSUPPORTED, "%d conjuncts (max %d)", (int)conj_end->size(), kMaxTerms);
    return MBC_OK;
}

// runs K4 into a fresh device bitmap of t->words_pad words
static int32_t run_bitmap_cnf_resolved(mbc_table* t, const std::vector<BmRef>& list, const std::vector<int>& conj_end, uint32_t** d_out);

int32_t run_bitmap_cnf(mbc_table* t, const mbc_term* terms, int32_t nterms, uint32_t** d_out) {
    std::vector<BmRef> list;
    std::vector<int> conj_end;
    std::vector<void*> temps;                             // flat bitmaps of sparse terms, freed behind the combine kernel
    int32_t s = resolve_bitmap_terms(t, terms, nterms, &list, &conj_end, &temps);
    if (s == MBC_OK) s = run_bitmap_cnf_resolved(t, list, conj_end, d_out);
    for (void* p : temps) dev_free(t->ctx, p);
    return s;
}

static int32_t run_bitmap_cnf_resolved(mbc_table* t, const std::vector<BmRef>& list, const std::vector<int>& conj_end, uint32_t** d_out) {
    mbc_ctx* ctx = t->ctx;
    MBC_TRY(dev_alloc(ctx, (void**)d_out, (size_t)t->words_pad * 4, false));
    CnfParams p{};
    p.nquads = t->words_pad / 4;
    p.out = reinterpret_cast<uint4*>(*d_out);
    p.deleted = t->has_deleted ? reinterpret_cast<const uint4*>(t->d_deleted) : nullptr;
    p.nconj = (int)conj_end.size();
    p.nbitmaps = (int)list.size();
    for (int g = 0; g < p.nconj; ++g) p.conj_end[g] = conj_end[g];
    BmRef* d_list = nullptr;
    if ((int)list.size() <= kMaxInlineBitmaps) {
        for (size_t j = 0; j < list.size(); ++j) p.inl[j] = list[j];
    } else {
        MBC_TRY(dev_alloc(ctx, (void**)&d_list, list.size() * sizeof(BmRef), false));
        MBC_CUDA(cudaMemcpyAsync(d_list, list.data(), list.size() * sizeof(BmRef), cudaMemcpyHostToDevice, ctx->stream));
        MBC_CUDA(cudaStreamSynchronize(ctx->stream));    // `list` is pageable host memory
        p.list = d_list;
    }
    int grid = (int)std::max<int64_t>(1, std::min<int64_t>((p.nquads + 255) / 256, (int64_t)ctx->sm_count * 8));
    bitmap_cnf_kernel<<<grid, 256, 0, ctx->stream>>>(p);
    ctx->launches++;
    MBC_CUDA(cudaGetLastError());
    if (d_list) dev_free(ctx, d_list);
    return MBC_OK;
}

}  // namespace mbc

extern "C" int32_t mbc_bitmap_scan(mbc_table* t, const mbc_term* terms, int32_t nterms, const int32_t* proj_cols,
                                   int32_t nproj, uint32_t want, const mbc_aggspec* aggs, int32_t nagg,
                                   mbc_result** out) {
    if (!t || !out) MBC_FAIL(MBC_ERR_ARG, "mbc_bitmap_scan: table/out is NULL");
    if (!terms && nterms > 0) MBC_FAIL(MBC_ERR_ARG, "mbc_bitmap_scan: terms is NULL");
    mbc_ctx* ctx = t->ctx;
    MBC_CUDA(cudaSetDevice(ctx->device));
    uint32_t* d_sel = nullptr;
    cudaEvent_t ev0;
    MBC_CUDA(cudaEventCreate(&ev0));
    cudaEventRecord(ev0, ctx->stream);
    int32_t s = run_bitmap_cnf(t, terms, nterms, &d_sel);
    if (s != MBC_OK) { cudaEventDestroy(ev0); return s; }
    ScanRequest rq;
    rq.table = t;
    rq.d_sel_bitmap = d_sel;
    rq.proj_cols = proj_cols;
    rq.nproj = nproj;
    rq.want = want;
    rq.aggs = aggs;
    rq.nagg = nagg;
    s = run_scan(rq, out);
    // account the combine kernel into the reported device time
    std::swap(ev0, ctx->ev_begin);
    cudaEventDestroy(ev0);
    dev_free(ctx, d_sel);
    return s;
}
