// mbc_join.cu -- K6: the bitmap equi-join of input/BitMapQuery.java:187-305 as a GPU join.
//
// Reference semantics (BitMapQuery.executeJoin): for every outer position o of the outer filter bitset,
// ascending (:227), plug the outer row's join-column values into the join CNF (:307-320), evaluate that
// CNF on the INNER table through its bitmap indexes (ColumnarIndexScan, :244-247), AND with the inner
// filter bitset (:249) and emit one joined tuple per set bit, ascending (:269-294).  The pair set is
//     { (o, i) : o in outerSel, i in innerSel, i not deleted, JOINCNF(outer[o], inner[i]) }
// ordered by (o, i); the projected tuple is Projection.Join of the target columns (:279-280).
//
// Two device strategies produce exactly that set and order:
//   * EQUI  (every conjunct is a single `outerCol = innerCol` term): keys are grouped -- directly
//     addressed when the key is one int column with a compact range (the group table then stays resident
//     in the 126 MB L2), otherwise through an open-addressing hash table on the key bytes.  Aggregates
//     need no pair list: COUNT = sum_i n_outer[g(i)], inner-side sums are weighted by n_outer, outer-side
//     sums by n_inner (three streaming passes, HBM-bound on the inner columns).  The pair list, when it is
//     asked for, comes from a stable radix sort of the matching inner rows by group.
//   * THETA (anything else: <, >, !=, OR-chains): the compacted survivors of both sides are crossed
//     by a tiled nested-loop kernel (count pass, scan, ordered write pass).
#include <algorithm>
#include <cstring>

#include "mbc_internal.cuh"

namespace mbc {

// ---- small device utilities ---------------------------------------------------------------------------

__device__ __forceinline__ bool test_bit(const uint32_t* bm, int64_t r) { return (bm[r >> 5] >> (r & 31)) & 1u; }

// L2 residency hints of the equi-join's counting pass: the per-group tables (n_outer / n_inner, 4 B per key) are hit at
// random by every inner row and must stay in L2 while gigabytes of key / value columns stream past them.  Table accesses
// carry an evict_last policy, the streamed columns are read evict-first (ld.global.cs).
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint32_t ld_keep_u32(const uint32_t* p, uint64_t pol) {
    uint32_t v;
    asm volatile("ld.global.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void red_add_keep_u32(uint32_t* p, uint32_t v, uint64_t pol) {
    asm volatile("red.global.add.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}

__device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}

// exclusive scan of n uint32 counts into uint64 offsets; total in out[n].  Three launches:
// per-block sums, scan of the block sums (one block), per-block scan + add.
constexpr int kScanBlock = 1024;
constexpr int kScanPerThread = 4;
constexpr int kScanChunk = kScanBlock * kScanPerThread;

__global__ void __launch_bounds__(kScanBlock) xscan_reduce_kernel(const uint32_t* in, int64_t n, unsigned long long* block_sums) {
    __shared__ unsigned long long sh[32];
    int64_t base = (int64_t)blockIdx.x * kScanChunk;
    unsigned long long s = 0;
    for (int k = 0; k < kScanPerThread; ++k) {
        int64_t i = base + (int64_t)threadIdx.x * kScanPerThread + k;
        if (i < n) s += in[i];
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        unsigned long long v = sh[threadIdx.x];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
        if (threadIdx.x == 0) block_sums[blockIdx.x] = v;
    }
}

__global__ void __launch_bounds__(1024) xscan_blocks_kernel(unsigned long long* block_sums, int64_t nblocks) {
    // single block: sequential chunks of 1024 with a running carry
    __shared__ unsigned long long sh[1024];
    __shared__ unsigned long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int64_t base = 0; base < nblocks; base += 1024) {
        int64_t i = base + threadIdx.x;
        unsigned long long v = i < nblocks ? block_sums[i] : 0;
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {
            unsigned long long t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
            __syncthreads();
            sh[threadIdx.x] += t;
            __syncthreads();
        }
        if (i < nblocks) block_sums[i] = carry + sh[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 0) carry += sh[1023];
        __syncthreads();
    }
    if (threadIdx.x == 0) block_sums[nblocks] = carry;
}

__global__ void __launch_bounds__(kScanBlock) xscan_apply_kernel(const uint32_t* in, int64_t n, const unsigned long long* block_sums,
                                                                 unsigned long long* out) {
    __shared__ unsigned long long sh[kScanBlock];
    int64_t base = (int64_t)blockIdx.x * kScanChunk + (int64_t)threadIdx.x * kScanPerThread;
    uint32_t v[kScanPerThread];
    unsigned long long s = 0;
    for (int k = 0; k < kScanPerThread; ++k) {
        v[k] = base + k < n ? in[base + k] : 0u;
        s += v[k];
    }
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 1; o < kScanBlock; o <<= 1) {
        unsigned long long t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
        __syncthreads();
        sh[threadIdx.x] += t;
        __syncthreads();
    }
    unsigned long long run = block_sums[blockIdx.x] + sh[threadIdx.x] - s;
    for (int k = 0; k < kScanPerThread; ++k) {
        if (base + k < n) out[base + k] = run;
        run += v[k];
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == kScanBlock - 1) out[n] = block_sums[gridDim.x];
}

int32_t exclusive_scan_u32(mbc_ctx* ctx, const uint32_t* d_in, int64_t n, unsigned long long* d_out /* n+1 */) {
    if (n == 0) {
        MBC_CUDA(cudaMemsetAsync(d_out, 0, 8, ctx->stream));
        return MBC_OK;
    }
    int64_t nblocks = (n + kScanChunk - 1) / kScanChunk;
    unsigned long long* d_sums = nullptr;
    MBC_TRY(dev_alloc(ctx, (void**)&d_sums, (size_t)(nblocks + 1) * 8, false));
    xscan_reduce_kernel<<<(unsigned)nblocks, kScanBlock, 0, ctx->stream>>>(d_in, n, d_sums);
    xscan_blocks_kernel<<<1, 1024, 0, ctx->stream>>>(d_sums, nblocks);
    xscan_apply_kernel<<<(unsigned)nblocks, kScanBlock, 0, ctx->stream>>>(d_in, n, d_sums, d_out);
    ctx->launches += 3;
    MBC_CUDA(cudaGetLastError());
    dev_free(ctx, d_sums);
    return MBC_OK;
}

// ---- stable LSD radix sort of (uint32 key, uint32 value) pairs, 8 bits per pass ---------------------------
constexpr int kSortThreads = 256;
constexpr int kSortWarps = kSortThreads / 32;
constexpr int kSortRounds = 32;                                   // elements per lane
constexpr int kSortChunk = kSortThreads * kSortRounds;            // 8192 elements per block; each warp owns 1024 consecutive ones

__global__ void __launch_bounds__(kSortThreads) rsort_hist_kernel(const uint32_t* keys, int64_t n, int shift, uint32_t* hist /*[256][nblocks]*/) {
    __shared__ uint32_t sh[256];
    sh[threadIdx.x] = 0;
    __syncthreads();
    int64_t base = (int64_t)blockIdx.x * kSortChunk;
    for (int k = threadIdx.x; k < kSortChunk; k += kSortThreads) {
        int64_t i = base + k;
        if (i < n) atomicAdd(&sh[(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    hist[(size_t)threadIdx.x * gridDim.x + blockIdx.x] = sh[threadIdx.x];
}

// lanes of the warp that hold the same digit (d < 0: none): one ballot per digit bit -- constant cost, where
// __match_any_sync's grows with the number of distinct digits in the warp (~32 here)
__device__ __forceinline__ uint32_t same_digit_lanes(int d) {
    uint32_t peers = __ballot_sync(0xFFFFFFFFu, d >= 0);
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        const uint32_t v = __ballot_sync(0xFFFFFFFFu, (d >> b) & 1);
        peers &= ((d >> b) & 1) ? v : ~v;
    }
    return peers;
}

__global__ void __launch_bounds__(kSortThreads) rsort_scatter_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, int64_t n,
                                                                     int shift, const unsigned long long* __restrict__ offsets /*[256][nblocks] scanned*/,
                                                                     uint32_t* __restrict__ out_keys, uint32_t* __restrict__ out_vals) {
    extern __shared__ uint32_t stage[];               // [kSortChunk] keys then [kSortChunk] values, in block-sorted order
    __shared__ uint32_t cnt[kSortWarps][256];         // per-warp digit counts, then running cursors (block-local positions)
    __shared__ uint32_t dstart[256];                  // block-local start of every digit's run
    __shared__ unsigned long long gbase[256];         // global start of every digit's run of this block
    __shared__ uint32_t wsum[kSortWarps];
    uint32_t* s_key = stage;
    uint32_t* s_val = stage + kSortChunk;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int d = lane; d < 256; d += 32) cnt[warp][d] = 0;
    __syncwarp();
    const int64_t bbase = (int64_t)blockIdx.x * kSortChunk;
    const int64_t wbase = bbase + warp * (kSortChunk / kSortWarps);
    const int nblk = (int)min((int64_t)kSortChunk, n - bbase);
    // phase A: the warp's 1024 consecutive keys into registers (all loads in flight at once) and its digit histogram
    uint32_t key[kSortRounds];
#pragma unroll
    for (int r = 0; r < kSortRounds; ++r) {
        const int64_t i = wbase + r * 32 + lane;
        key[r] = i < n ? keys[i] : 0u;
    }
#pragma unroll
    for (int r = 0; r < kSortRounds; ++r)
        if (wbase + r * 32 + lane < n) atomicAdd(&cnt[warp][(key[r] >> shift) & 255u], 1u);
    __syncthreads();
    // phase B: thread d owns digit d: prefix over the warps, then an exclusive scan of the 256 digit totals of the block
    {
        const int d = threadIdx.x;
        uint32_t run = 0;
        for (int w = 0; w < kSortWarps; ++w) {
            const uint32_t c = cnt[w][d];
            cnt[w][d] = run;
            run += c;
        }
        uint32_t incl = run;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t x = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += x;
        }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        uint32_t before = 0;
        for (int w = 0; w < warp; ++w) before += wsum[w];
        dstart[d] = before + incl - run;
        gbase[d] = offsets[(size_t)d * gridDim.x + blockIdx.x];
    }
    __syncthreads();
    // phase C: stable placement in shared memory, round by round (rank within the round = lower lanes with the same digit)
#pragma unroll
    for (int r = 0; r < kSortRounds; ++r) {
        const int64_t i = wbase + r * 32 + lane;
        const int dg = i < n ? (int)((key[r] >> shift) & 255u) : -1;
        const uint32_t grp = same_digit_lanes(dg);
        const uint32_t rank = __popc(grp & ((1u << lane) - 1));
        if (dg >= 0) {
            const uint32_t pos = dstart[dg] + cnt[warp][dg] + rank;
            s_key[pos] = key[r];
            s_val[pos] = vals[i];
        }
        __syncwarp();
        if (dg >= 0 && rank == 0) cnt[warp][dg] += __popc(grp);
        __syncwarp();
    }
    __syncthreads();
    // phase D: copy out in sorted order: consecutive threads write consecutive addresses inside every digit's run
    for (int j = threadIdx.x; j < nblk; j += kSortThreads) {
        const uint32_t k = s_key[j];
        const uint32_t d = (k >> shift) & 255u;
        const unsigned long long dst = gbase[d] + (uint32_t)j - dstart[d];
        out_keys[dst] = k;
        out_vals[dst] = s_val[j];
    }
}

// sorts in place (result ends in keys/vals); tmp buffers of the same size are allocated here
int32_t radix_sort_pairs(mbc_ctx* ctx, uint32_t* d_keys, uint32_t* d_vals, int64_t n, int key_bits, uint32_t pass_mask) {
    if (n <= 1 || pass_mask == 0) return MBC_OK;
    uint32_t *tk = nullptr, *tv = nullptr, *hist = nullptr;
    unsigned long long* offs = nullptr;
    int64_t nblocks = (n + kSortChunk - 1) / kSortChunk;
    MBC_TRY(dev_alloc(ctx, (void**)&tk, (size_t)n * 4, false));
    MBC_TRY(dev_alloc(ctx, (void**)&tv, (size_t)n * 4, false));
    MBC_TRY(dev_alloc(ctx, (void**)&hist, (size_t)256 * nblocks * 4, false));
    MBC_TRY(dev_alloc(ctx, (void**)&offs, ((size_t)256 * nblocks + 1) * 8, false));
    if (!ctx->sort_smem_set) {                                    // a function attribute is per device: once per context
        MBC_CUDA(cudaFuncSetAttribute(rsort_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSortChunk * 8));
        ctx->sort_smem_set = true;
    }
    uint32_t *sk = d_keys, *sv = d_vals, *dk = tk, *dv = tv;
    int passes = std::max(1, (key_bits + 7) / 8);
    for (int p = 0; p < passes; ++p) {
        if (!((pass_mask >> p) & 1u)) continue;                 // this digit is the same in every key: a stable pass would change nothing
        rsort_hist_kernel<<<(unsigned)nblocks, kSortThreads, 0, ctx->stream>>>(sk, n, p * 8, hist);
        ctx->launches++;
        MBC_TRY(exclusive_scan_u32(ctx, hist, 256 * nblocks, offs));
        rsort_scatter_kernel<<<(unsigned)nblocks, kSortThreads, kSortChunk * 8, ctx->stream>>>(sk, sv, n, p * 8, offs, dk, dv);
        ctx->launches++;
        std::swap(sk, dk);
        std::swap(sv, dv);
    }
    if (sk != d_keys) {
        MBC_CUDA(cudaMemcpyAsync(d_keys, sk, (size_t)n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        MBC_CUDA(cudaMemcpyAsync(d_vals, sv, (size_t)n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    MBC_CUDA(cudaGetLastError());
    dev_free(ctx, tk); dev_free(ctx, tv); dev_free(ctx, hist); dev_free(ctx, offs);
    return MBC_OK;
}

// ---- join description shared by the kernels -----------------------------------------------------------------

constexpr int kMaxJoinTerms = 8;
constexpr int kMaxJoinAgg = 8;

struct JoinCol {
    const void* ptr;
    int32_t stride;       // 4 or the string stride
    int32_t is_str;
};

struct JoinTerm {
    JoinCol o, i;
    int32_t op, cmp_type, end_conj, pad;
};

struct JoinSide {
    const uint32_t* sel;        // optional filter bitmap
    const uint32_t* deleted;    // optional markedDeleted
    int64_t nrows;
};

struct GroupMap {
    int32_t mode;               // 0 = direct (single int key, group = key - kmin), 1 = hash
    int32_t nkeys;
    long long kmin, kmax;       // direct mode
    unsigned long long* slots;  // hash mode: representative (side,row)+1
    uint32_t mask;
    uint32_t ngroups;           // direct: range ; hash: capacity
    JoinCol okey[kMaxJoinTerms], ikey[kMaxJoinTerms];
};

__device__ __forceinline__ bool side_selected(const JoinSide& s, int64_t r) {
    if (r >= s.nrows) return false;
    if (s.sel && !test_bit(s.sel, r)) return false;
    if (s.deleted && test_bit(s.deleted, r)) return false;
    return true;
}

// word w of key column c of row r, zero beyond the column's own width (strings of different declared
// widths compare equal when their zero-padded bytes do)
__device__ __forceinline__ uint32_t key_word(const JoinCol& c, int64_t r, int w) {
    if (w >= (c.stride >> 2)) return 0u;
    return reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(c.ptr) + r * c.stride)[w];
}

__device__ __forceinline__ uint32_t key_hash(const JoinCol* cols, int nkeys, const JoinCol* other, int64_t r) {
    uint32_t h = 0x9E3779B9u;
    for (int k = 0; k < nkeys; ++k) {
        int words = max(cols[k].stride, other[k].stride) >> 2;
        for (int w = 0; w < words; ++w) h = mix32(h ^ key_word(cols[k], r, w)) + 0x85EBCA6Bu * (uint32_t)(k + 1);
    }
    return h;
}

__device__ __forceinline__ bool keys_equal(const JoinCol* a, int64_t ra, const JoinCol* b, int64_t rb, int nkeys) {
    for (int k = 0; k < nkeys; ++k) {
        int words = max(a[k].stride, b[k].stride) >> 2;
        for (int w = 0; w < words; ++w)
            if (key_word(a[k], ra, w) != key_word(b[k], rb, w)) return false;
    }
    return true;
}

// group of an OUTER row (inserting in hash mode); -1 on table overflow
__device__ __forceinline__ long long group_of_outer(const GroupMap& g, int64_t o, bool insert) {
    if (g.mode == 0) return (long long)reinterpret_cast<const int32_t*>(g.okey[0].ptr)[o] - g.kmin;
    uint32_t s = key_hash(g.okey, g.nkeys, g.ikey, o) & g.mask;
    for (uint32_t n = 0; n <= g.mask; ++n, s = (s + 1) & g.mask) {
        unsigned long long cur = *reinterpret_cast<volatile unsigned long long*>(g.slots + s);
        if (cur == 0) {
            if (!insert) return -1;
            unsigned long long old = atomicCAS(g.slots + s, 0ull, (unsigned long long)(o + 1));
            if (old == 0) return s;
            cur = old;
        }
        if (keys_equal(g.okey, o, g.okey, (int64_t)(cur - 1), g.nkeys)) return s;
    }
    return -1;
}

// group of an INNER row, -1 when no outer row carries that key
__device__ __forceinline__ long long group_of_inner(const GroupMap& g, int64_t i) {
    if (g.mode == 0) {
        long long k = (long long)__ldcs(reinterpret_cast<const int32_t*>(g.ikey[0].ptr) + i);
        return (k < g.kmin || k > g.kmax) ? -1 : k - g.kmin;
    }
    uint32_t s = key_hash(g.ikey, g.nkeys, g.okey, i) & g.mask;
    for (uint32_t n = 0; n <= g.mask; ++n, s = (s + 1) & g.mask) {
        unsigned long long cur = __ldg(g.slots + s);
        if (cur == 0) return -1;
        if (keys_equal(g.ikey, i, g.okey, (int64_t)(cur - 1), g.nkeys)) return s;
    }
    return -1;
}

// ---- EQUI path: counting passes + weighted aggregates -------------------------------------------------------------

struct JoinAgg {
    const void* src;      // column of the side the aggregate reads
    int32_t kind, type;   // MBC_AGG_*, MBC_ATTR_INTEGER/REAL
    int32_t side;         // 1 outer, 2 inner, 0 COUNT
    int32_t slot;         // unique-key path: word of the group slot that carries this outer-side value (1..3)
};

struct EquiParams {
    GroupMap g;
    JoinSide outer, inner;
    uint32_t* n_outer;
    uint32_t* n_inner;
    uint32_t* inner_match;         // optional bitmap of inner rows that found a partner
    int* overflow;                 // [0] hash table overflow, [1] some key occurs on more than one outer row, [2] selected outer rows
    int32_t nagg, pad;
    int32_t pre[2];                // unique path: the (up to two) inner-side aggregates whose inputs are loaded with the keys, or -1
    JoinAgg aggs[kMaxJoinAgg];
    unsigned long long* partials;  // [nagg][gridDim.x]
};

__global__ void __launch_bounds__(256) join_minmax_kernel(const int32_t* key, JoinSide s, long long* out /* min,max */) {
    long long mn = INT64_MAX, mx = INT64_MIN;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < s.nrows; r += (int64_t)gridDim.x * blockDim.x) {
        if (!side_selected(s, r)) continue;
        long long k = key[r];
        mn = min(mn, k);
        mx = max(mx, k);
    }
    for (int o = 16; o > 0; o >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xFFFFFFFFu, mn, o));
        mx = max(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(out, mn);
        atomicMax(out + 1, mx);
    }
}

// Few groups (a low-cardinality key: C4's secondary variant has 1 000) would put every row's atomic on one of a few hundred
// L2 addresses: the counts are then kept in a per-CTA shared-memory histogram and merged once per CTA and group.
constexpr uint32_t kSmallGroups = 4096;

__global__ void __launch_bounds__(256) join_outer_count_kernel(const __grid_constant__ EquiParams p) {
    __shared__ uint32_t s_hist[kSmallGroups];
    const bool small = p.g.mode == 0 && p.g.ngroups <= kSmallGroups;
    if (small) {
        for (uint32_t i = threadIdx.x; i < p.g.ngroups; i += blockDim.x) s_hist[i] = 0u;
        __syncthreads();
    }
    int selected = 0;
    for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < p.outer.nrows; o += (int64_t)gridDim.x * blockDim.x) {
        if (!side_selected(p.outer, o)) continue;
        long long g = group_of_outer(p.g, o, true);
        if (g < 0) { *p.overflow = 1; break; }
        if (small) atomicAdd(&s_hist[g], 1u);
        else if (atomicAdd(p.n_outer + g, 1u) != 0u) p.overflow[1] = 1;
        ++selected;
    }
    if (small) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < p.g.ngroups; i += blockDim.x) {
            const uint32_t c = s_hist[i];
            if (c && (atomicAdd(p.n_outer + i, c) != 0u || c > 1u)) p.overflow[1] = 1;      // some key on more than one outer row
        }
    }
    // selected outer rows (dense-key test of the unique path): one atomic per warp, not one per row on a single address
    __syncwarp();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) selected += __shfl_xor_sync(0xFFFFFFFFu, selected, o);
    if ((threadIdx.x & 31) == 0 && selected) atomicAdd(p.overflow + 2, selected);
}

__device__ __forceinline__ void agg_fold(const JoinAgg& a, bool integral, long long& ai, double& af, int64_t row, unsigned long long weight) {
    if (a.kind == MBC_AGG_COUNT) { ai += (long long)weight; return; }
    uint32_t bits = __ldcs(reinterpret_cast<const uint32_t*>(a.src) + row);
    if (integral) {
        long long v = (int32_t)bits;
        if (a.kind == MBC_AGG_SUM) ai += v * (long long)weight;
        else if (a.kind == MBC_AGG_MIN) ai = min(ai, v);
        else ai = max(ai, v);
    } else {
        double v = (double)__uint_as_float(bits);
        if (a.kind == MBC_AGG_SUM) af += v * (double)weight;
        else if (a.kind == MBC_AGG_MIN) af = fmin(af, v);
        else af = fmax(af, v);
    }
}

// one pass over `side` rows (2 = inner: counts n_inner, folds COUNT + inner-side aggregates weighted by n_outer;
// 1 = outer: folds outer-side aggregates weighted by n_inner)
template <int SIDE>
__global__ void __launch_bounds__(256) join_agg_pass_kernel(const __grid_constant__ EquiParams p) {
    __shared__ unsigned long long sh[kMaxJoinAgg][8];
    long long ai[kMaxJoinAgg];
    double af[kMaxJoinAgg];
    for (int a = 0; a < p.nagg; ++a) {
        const JoinAgg& g = p.aggs[a];
        ai[a] = (g.kind == MBC_AGG_MIN) ? (long long)INT32_MAX : (g.kind == MBC_AGG_MAX) ? (long long)INT32_MIN : 0ll;
        af[a] = (g.kind == MBC_AGG_MIN) ? (double)INFINITY : (g.kind == MBC_AGG_MAX) ? (double)-INFINITY : 0.0;
    }
    __shared__ uint32_t s_hist[SIDE == 2 ? kSmallGroups : 1];
    const bool small = SIDE == 2 && p.g.mode == 0 && p.g.ngroups <= kSmallGroups;
    if (small) {
        for (uint32_t i = threadIdx.x; i < p.g.ngroups; i += blockDim.x) s_hist[i] = 0u;
        __syncthreads();
    }
    const JoinSide& s = SIDE == 2 ? p.inner : p.outer;
    const uint64_t keep = l2_policy_evict_last();
    const int64_t nrows32 = (s.nrows + 31) & ~31ll;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < nrows32; r += (int64_t)gridDim.x * blockDim.x) {
        unsigned long long weight = 0;
        if (side_selected(s, r)) {
            long long g = SIDE == 2 ? group_of_inner(p.g, r) : group_of_outer(p.g, r, false);
            if (g >= 0) {
                weight = SIDE == 2 ? ld_keep_u32(p.n_outer + g, keep) : p.n_inner[g];
                if (SIDE == 2 && weight) {
                    if (small) atomicAdd(&s_hist[g], 1u);
                    else red_add_keep_u32(p.n_inner + g, 1u, keep);
                }
            }
        }
        if (SIDE == 2 && p.inner_match) {
            uint32_t word = __ballot_sync(0xFFFFFFFFu, weight != 0);
            if ((threadIdx.x & 31) == 0) p.inner_match[r >> 5] = word;
        }
        if (weight) {
            for (int a = 0; a < p.nagg; ++a) {
                const JoinAgg& g = p.aggs[a];
                if ((g.side == 0 && SIDE == 2) || g.side == SIDE)
                    agg_fold(g, g.kind == MBC_AGG_COUNT || g.type == MBC_ATTR_INTEGER, ai[a], af[a], r, weight);
            }
        }
    }
    if (small) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < p.g.ngroups; i += blockDim.x) {
            const uint32_t c = s_hist[i];
            if (c) atomicAdd(p.n_inner + i, c);
        }
    }
    // block reduction, one partial per block per aggregate (fixed order -> reproducible sums)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int a = 0; a < p.nagg; ++a) {
        const JoinAgg& g = p.aggs[a];
        const bool mine = (g.side == 0 && SIDE == 2) || g.side == SIDE;
        if (!mine) continue;
        const bool integral = g.kind == MBC_AGG_COUNT || g.type == MBC_ATTR_INTEGER;
        const bool additive = g.kind == MBC_AGG_COUNT || g.kind == MBC_AGG_SUM;
        long long vi = ai[a];
        double vf = af[a];
        for (int o = 16; o > 0; o >>= 1) {
            long long xi = __shfl_xor_sync(0xFFFFFFFFu, vi, o);
            double xf = __shfl_xor_sync(0xFFFFFFFFu, vf, o);
            vi = additive ? vi + xi : g.kind == MBC_AGG_MIN ? min(vi, xi) : max(vi, xi);
            vf = additive ? vf + xf : g.kind == MBC_AGG_MIN ? fmin(vf, xf) : fmax(vf, xf);
        }
        if (lane == 0) sh[a][warp] = integral ? (unsigned long long)vi : (unsigned long long)__double_as_longlong(vf);
        __syncthreads();
        if (threadIdx.x == 0) {
            long long ri = (long long)sh[a][0];
            double rf = __longlong_as_double((long long)sh[a][0]);
            for (int w = 1; w < 8; ++w) {
                long long xi = (long long)sh[a][w];
                double xf = __longlong_as_double((long long)sh[a][w]);
                ri = additive ? ri + xi : g.kind == MBC_AGG_MIN ? min(ri, xi) : max(ri, xi);
                rf = additive ? rf + xf : g.kind == MBC_AGG_MIN ? fmin(rf, xf) : fmax(rf, xf);
            }
            p.partials[(size_t)a * gridDim.x + blockIdx.x] = integral ? (unsigned long long)ri : (unsigned long long)__double_as_longlong(rf);
        }
        __syncthreads();
    }
}

// ---- unique-key aggregate path (PK-FK joins, aggregates only) ------------------------------------------------------
// When every join key occurs on at most one outer row and no pair list is wanted, a pair is (inner row, THE outer row
// of its key): a 1-bit-per-key presence bitmap plus a slot of the outer-side aggregate inputs per key, and a single
// pass over the inner rows folds every aggregate from one bit test and ONE random slot read per row -- no n_inner
// atomics, no outer pass.  The general path keeps two 4-byte tables per key (a random read and a random atomic per
// inner row); for 10 M keys they do not stay in L2 next to the streamed columns and most accesses go to HBM as 64-byte
// fetches, which is what bounds it.
template <int VALW>      // value words per key: 0, 1, 2 or 4 (three columns are padded to four)
__global__ void __launch_bounds__(256) join_slot_build_kernel(const __grid_constant__ EquiParams p, uint32_t* present, uint32_t* slots,
                                                              const void* c1, const void* c2, const void* c3) {
    const int32_t* key = reinterpret_cast<const int32_t*>(p.g.okey[0].ptr);
    for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < p.outer.nrows; o += (int64_t)gridDim.x * blockDim.x) {
        if (!side_selected(p.outer, o)) continue;
        const long long g = (long long)key[o] - p.g.kmin;
        atomicOr(present + (g >> 5), 1u << (g & 31));
        if (VALW == 1) slots[g] = reinterpret_cast<const uint32_t*>(c1)[o];
        if (VALW == 2) reinterpret_cast<uint2*>(slots)[g] = make_uint2(reinterpret_cast<const uint32_t*>(c1)[o], reinterpret_cast<const uint32_t*>(c2)[o]);
        if (VALW == 4) reinterpret_cast<uint4*>(slots)[g] = make_uint4(reinterpret_cast<const uint32_t*>(c1)[o], reinterpret_cast<const uint32_t*>(c2)[o],
                                                                       reinterpret_cast<const uint32_t*>(c3)[o], 0u);
    }
}

// One 64-bit accumulator per aggregate (an aggregate is either integral or real, never both): half the registers of an
// (int64, double) pair, which is what sets this kernel's occupancy.
__device__ __forceinline__ unsigned long long acc_identity(const JoinAgg& g, bool integral) {
    if (integral) return (unsigned long long)((g.kind == MBC_AGG_MIN) ? (long long)INT32_MAX : (g.kind == MBC_AGG_MAX) ? (long long)INT32_MIN : 0ll);
    return (unsigned long long)__double_as_longlong((g.kind == MBC_AGG_MIN) ? (double)INFINITY : (g.kind == MBC_AGG_MAX) ? (double)-INFINITY : 0.0);
}
__device__ __forceinline__ unsigned long long acc_merge(const JoinAgg& g, bool integral, unsigned long long x, unsigned long long y) {
    const bool additive = g.kind == MBC_AGG_COUNT || g.kind == MBC_AGG_SUM;
    if (integral) {
        const long long a = (long long)x, b = (long long)y;
        return (unsigned long long)(additive ? a + b : g.kind == MBC_AGG_MIN ? min(a, b) : max(a, b));
    }
    const double a = __longlong_as_double((long long)x), b = __longlong_as_double((long long)y);
    return (unsigned long long)__double_as_longlong(additive ? a + b : g.kind == MBC_AGG_MIN ? fmin(a, b) : fmax(a, b));
}
__device__ __forceinline__ unsigned long long acc_fold_bits(const JoinAgg& g, bool integral, unsigned long long acc, uint32_t bits) {
    if (integral) return acc_merge(g, true, acc, (unsigned long long)(long long)(int32_t)bits);
    return acc_merge(g, false, acc, (unsigned long long)__double_as_longlong((double)__uint_as_float(bits)));
}

constexpr int kJoinBatch = 4;      // inner rows a thread has in flight: key -> slot -> value loads are dependent HBM round trips

template <int VALW, bool DENSE>      // DENSE: every key of [kmin, kmax] is on an outer row, no presence test
__global__ void __launch_bounds__(256, 4) join_unique_pass_kernel(const __grid_constant__ EquiParams p, const uint32_t* __restrict__ present,
                                                                  const uint32_t* __restrict__ slots) {
    __shared__ unsigned long long sh[kMaxJoinAgg][8];
    unsigned long long acc[kMaxJoinAgg];
#pragma unroll
    for (int a = 0; a < kMaxJoinAgg; ++a)                 // static indices everywhere: the accumulators live in registers
        acc[a] = acc_identity(p.aggs[a], p.aggs[a].kind == MBC_AGG_COUNT || p.aggs[a].type == MBC_ATTR_INTEGER);
    const uint64_t keep = l2_policy_evict_last();
    const int32_t* fk = reinterpret_cast<const int32_t*>(p.g.ikey[0].ptr);
    const int64_t nrows32 = (p.inner.nrows + 31) & ~31ll;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;               // a multiple of 32: a warp's rows stay consecutive
    const uint32_t* pre_src0 = p.pre[0] >= 0 ? reinterpret_cast<const uint32_t*>(p.aggs[p.pre[0] & (kMaxJoinAgg - 1)].src) : nullptr;
    const uint32_t* pre_src1 = p.pre[1] >= 0 ? reinterpret_cast<const uint32_t*>(p.aggs[p.pre[1] & (kMaxJoinAgg - 1)].src) : nullptr;
    for (int64_t r0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r0 < nrows32; r0 += stride * kJoinBatch) {
        long long k[kJoinBatch];
        uint32_t pre0[kJoinBatch], pre1[kJoinBatch];
#pragma unroll
        for (int b = 0; b < kJoinBatch; ++b) {                            // round trip 1: the keys, and the inputs of the first
            const int64_t r = r0 + b * stride;                            // two inner-side aggregates (they do not depend on the
            const bool sel = side_selected(p.inner, r);                   // key; a row without a partner wastes its 8 bytes)
            k[b] = sel ? (long long)__ldcs(fk + r) : p.g.kmin - 1;
            pre0[b] = (sel && pre_src0) ? __ldcs(pre_src0 + r) : 0u;
            pre1[b] = (sel && pre_src1) ? __ldcs(pre_src1 + r) : 0u;
        }
        uint32_t pw[kJoinBatch], v1[kJoinBatch], v2[kJoinBatch], v3[kJoinBatch];
#pragma unroll
        for (int b = 0; b < kJoinBatch; ++b) {                            // round trip 2: presence word and value slot together
            pw[b] = v1[b] = v2[b] = v3[b] = 0u;
            if (k[b] >= p.g.kmin && k[b] <= p.g.kmax) {
                const long long g = k[b] - p.g.kmin;
                pw[b] = DENSE ? 1u : __ldg(present + (g >> 5)) >> (g & 31);
                if (VALW == 1) v1[b] = ld_keep_u32(slots + g, keep);
                if (VALW == 2) {
                    const uint2 v = __ldg(reinterpret_cast<const uint2*>(slots) + g);
                    v1[b] = v.x; v2[b] = v.y;
                }
                if (VALW == 4) {
                    const uint4 v = __ldg(reinterpret_cast<const uint4*>(slots) + g);
                    v1[b] = v.x; v2[b] = v.y; v3[b] = v.z;
                }
            }
        }
        bool hit[kJoinBatch];
        int nhit = 0;
#pragma unroll
        for (int b = 0; b < kJoinBatch; ++b) {
            hit[b] = pw[b] & 1u;
            nhit += hit[b];
            if (p.inner_match) {
                const int64_t r = r0 + b * stride;
                const uint32_t word = __ballot_sync(0xFFFFFFFFu, hit[b]);
                if ((threadIdx.x & 31) == 0 && r < nrows32) p.inner_match[r >> 5] = word;
            }
        }
#pragma unroll
        for (int a = 0; a < kMaxJoinAgg; ++a) {
            if (a >= p.nagg) break;
            const JoinAgg& g = p.aggs[a];
            const bool integral = g.kind == MBC_AGG_COUNT || g.type == MBC_ATTR_INTEGER;
            if (g.kind == MBC_AGG_COUNT) {
                acc[a] += (unsigned long long)nhit;
            } else if (g.side == 2) {                                     // round trip 3 (per inner-side aggregate): its column
                uint32_t bits[kJoinBatch];
#pragma unroll
                for (int b = 0; b < kJoinBatch; ++b) {
                    if (a == p.pre[0]) bits[b] = pre0[b];
                    else if (a == p.pre[1]) bits[b] = pre1[b];
                    else if (hit[b]) bits[b] = __ldcs(reinterpret_cast<const uint32_t*>(g.src) + r0 + b * stride);
                }
#pragma unroll
                for (int b = 0; b < kJoinBatch; ++b)
                    if (hit[b]) acc[a] = acc_fold_bits(g, integral, acc[a], bits[b]);
            } else {
#pragma unroll
                for (int b = 0; b < kJoinBatch; ++b)
                    if (hit[b]) acc[a] = acc_fold_bits(g, integral, acc[a], g.slot == 1 ? v1[b] : g.slot == 2 ? v2[b] : v3[b]);
            }
        }
    }
    // block reduction, one partial per block per aggregate (fixed order -> reproducible sums)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int a = 0; a < kMaxJoinAgg; ++a) {
        if (a >= p.nagg) break;
        const JoinAgg& g = p.aggs[a];
        const bool integral = g.kind == MBC_AGG_COUNT || g.type == MBC_ATTR_INTEGER;
        unsigned long long v = acc[a];
        for (int o = 16; o > 0; o >>= 1) v = acc_merge(g, integral, v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
        if (lane == 0) sh[a][warp] = v;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long r = sh[a][0];
            for (int w8 = 1; w8 < 8; ++w8) r = acc_merge(g, integral, r, sh[a][w8]);
            p.partials[(size_t)a * gridDim.x + blockIdx.x] = r;
        }
        __syncthreads();
    }
}

__global__ void join_agg_finish_kernel(const unsigned long long* partials, int nblocks, int nagg, const JoinAgg* aggs_unused,
                                       int kind0, unsigned long long* out) {
    (void)aggs_unused; (void)kind0; (void)nagg; (void)partials; (void)nblocks; (void)out;
}

// ---- EQUI path: pair list --------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(256) join_group_keys_kernel(GroupMap g, const int64_t* inner_pos, int64_t n, int64_t inner_base,
                                                              uint32_t* keys, uint32_t* vals) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        int64_t i = inner_pos[k] - inner_base;
        keys[k] = (uint32_t)group_of_inner(g, i);
        vals[k] = (uint32_t)i;
    }
}

__global__ void __launch_bounds__(256) join_outer_counts_kernel(GroupMap g, const int64_t* outer_pos, int64_t n, int64_t outer_base,
                                                                const uint32_t* n_inner, uint32_t* cnt, uint32_t* grp) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        long long gg = group_of_outer(g, outer_pos[k] - outer_base, false);
        grp[k] = (uint32_t)gg;
        cnt[k] = gg >= 0 ? n_inner[gg] : 0u;
    }
}

// pair p belongs to the outer list entry idx with off[idx] <= p < off[idx+1]
__global__ void __launch_bounds__(256) join_fill_pairs_kernel(const unsigned long long* off, int64_t n_outer_list, const int64_t* outer_pos,
                                                              const uint32_t* grp, const unsigned long long* group_start,
                                                              const uint32_t* sorted_inner, int64_t inner_base, int64_t npairs,
                                                              int64_t* out_o, int64_t* out_i) {
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < npairs; p += (int64_t)gridDim.x * blockDim.x) {
        int64_t lo = 0, hi = n_outer_list;            // largest idx with off[idx] <= p
        while (hi - lo > 1) {
            int64_t mid = (lo + hi) >> 1;
            if (off[mid] <= (unsigned long long)p) lo = mid; else hi = mid;
        }
        unsigned long long k = (unsigned long long)p - off[lo];
        out_o[p] = outer_pos[lo];
        out_i[p] = inner_base + sorted_inner[group_start[grp[lo]] + k];
    }
}

// ---- THETA path: tiled nested loop over the compacted survivors ------------------------------------------------------------

struct ThetaParams {
    const int64_t* outer_pos;
    const int64_t* inner_pos;
    int64_t n_outer, n_inner, outer_base, inner_base;
    int32_t nterms, chunks;
    JoinTerm terms[kMaxJoinTerms];
    uint32_t* counts;                       // [n_outer][chunks]
    const unsigned long long* offsets;      // scanned counts
    int64_t* out_o;
    int64_t* out_i;
};

constexpr int kThetaThreads = 256;
constexpr int kThetaChunk = 2048;           // inner survivors per CTA

__device__ __forceinline__ uint32_t bswap(uint32_t x) { return __byte_perm(x, 0, 0x0123); }

__device__ __forceinline__ bool theta_pair(const ThetaParams& p, int64_t o, int64_t i) {
    bool acc = false;
    for (int k = 0; k < p.nterms; ++k) {
        const JoinTerm& t = p.terms[k];
        bool lt = false, eq = true;
        if (t.cmp_type == MBC_ATTR_STRING) {
            int words = max(t.o.stride, t.i.stride) >> 2;
            for (int w = 0; w < words; ++w) {
                uint32_t x = bswap(key_word(t.o, o, w)), y = bswap(key_word(t.i, i, w));
                if (x != y) { lt = x < y; eq = false; break; }
            }
        } else {
            uint32_t a = reinterpret_cast<const uint32_t*>(t.o.ptr)[o], b = reinterpret_cast<const uint32_t*>(t.i.ptr)[i];
            if (t.cmp_type == MBC_ATTR_INTEGER) { lt = (int32_t)a < (int32_t)b; eq = a == b; }
            else { float x = __uint_as_float(a), y = __uint_as_float(b); lt = x < y; eq = x == y; }
        }
        bool r;
        switch (t.op) {
            case MBC_OP_EQ: r = eq; break;
            case MBC_OP_LT: r = lt; break;
            case MBC_OP_GT: r = !(lt || eq); break;
            case MBC_OP_NE: r = !eq; break;
            case MBC_OP_LE: r = lt || eq; break;
            case MBC_OP_GE: r = !lt; break;
            default: r = false;                     // getBitSet has no branch for aopNOT / NOP / RANGE
        }
        acc = acc || r;
        if (t.end_conj) {
            if (!acc) return false;
            acc = false;
        }
    }
    return true;
}

template <bool WRITE>
__global__ void __launch_bounds__(kThetaThreads) join_theta_kernel(const __grid_constant__ ThetaParams p) {
    __shared__ uint32_t warp_tot[kThetaThreads / 32];
    const int64_t oi = blockIdx.x;                  // outer list index
    const int chunk = blockIdx.y;
    const int64_t o = p.outer_pos[oi] - p.outer_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t k0 = (int64_t)chunk * kThetaChunk;
    unsigned long long base = WRITE ? p.offsets[oi * p.chunks + chunk] : 0ull;
    uint32_t block_count = 0;
    // the CTA walks its chunk in order, kThetaThreads inner rows at a time, so writes stay ascending
    for (int r = 0; r < kThetaChunk / kThetaThreads; ++r) {
        int64_t k = k0 + r * kThetaThreads + threadIdx.x;
        bool hit = false;
        int64_t ipos = 0;
        if (k < p.n_inner) {
            ipos = p.inner_pos[k];
            hit = theta_pair(p, o, ipos - p.inner_base);
        }
        uint32_t bal = __ballot_sync(0xFFFFFFFFu, hit);
        if (lane == 0) warp_tot[warp] = __popc(bal);
        __syncthreads();
        uint32_t before = 0, total = 0;
        for (int w = 0; w < kThetaThreads / 32; ++w) {
            if (w < warp) before += warp_tot[w];
            total += warp_tot[w];
        }
        if (WRITE && hit) {
            unsigned long long dst = base + block_count + before + __popc(bal & ((1u << lane) - 1));
            p.out_o[dst] = p.outer_pos[oi];
            p.out_i[dst] = ipos;
        }
        block_count += total;
        __syncthreads();
    }
    if (!WRITE && threadIdx.x == 0) p.counts[oi * p.chunks + chunk] = block_count;
}

// ---- projection of the pair list into result columns ---------------------------------------------------------------------------

struct GatherParams {
    const int64_t* pos;      // positions (global) of the side this field reads
    int64_t base, npairs;
    const void* src;
    void* dst;
    int32_t stride, pad;
};

__global__ void __launch_bounds__(256) join_gather_kernel(const __grid_constant__ GatherParams p) {
    const int words = p.stride >> 2;
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < p.npairs; k += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t* s = reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(p.src) + (p.pos[k] - p.base) * p.stride);
        uint32_t* d = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(p.dst) + k * p.stride);
        for (int w = 0; w < words; ++w) d[w] = s[w];
    }
}

// ---- host side -------------------------------------------------------------------------------------------------------------------------

int32_t finish_result_host(mbc_result* r);
void decode_aggs_join(mbc_result* r, const JoinAgg* aggs, int nagg, const unsigned long long* raw);

static JoinCol join_col(const mbc_table* t, int col) {
    JoinCol c;
    c.ptr = t->cols[col].d;
    c.stride = t->cols[col].stride;
    c.is_str = t->cols[col].type == MBC_ATTR_STRING;
    return c;
}

static int grid_for(mbc_ctx* ctx, int64_t n, int per_sm = 8) {
    return (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * per_sm));
}

// ordered positions of the rows of `t` selected by `sel` (device int64 list, global positions)
static int32_t compact_side(mbc_table* t, const uint32_t* d_sel, mbc_result** out) {
    ScanRequest rq;
    rq.table = t;
    rq.d_sel_bitmap = d_sel;
    rq.want = MBC_WANT_POSITIONS;
    return run_scan(rq, out);
}

}  // namespace mbc

using namespace mbc;

extern "C" int32_t mbc_bitmap_join(mbc_table* outer, mbc_table* inner, const mbc_result* outer_sel, const mbc_result* inner_sel,
                                   const mbc_term* join_terms, int32_t njoin, const mbc_projspec* proj, int32_t nproj,
                                   uint32_t want, const mbc_aggspec* aggs, int32_t nagg, mbc_result** out) {
    if (!outer || !inner || !out || !join_terms || njoin <= 0) MBC_FAIL(MBC_ERR_ARG, "mbc_bitmap_join: bad argument");
    if (outer->ctx != inner->ctx) MBC_FAIL(MBC_ERR_ARG, "mbc_bitmap_join: tables live in different contexts");
    if (njoin > kMaxJoinTerms) MBC_FAIL(MBC_ERR_UNSUPPORTED, "%d join terms (max %d)", njoin, kMaxJoinTerms);
    if (nproj < 0 || nproj > kMaxProj || (nproj > 0 && !proj)) MBC_FAIL(MBC_ERR_ARG, "mbc_bitmap_join: bad projection");
    if (!(want & MBC_WANT_AGG)) nagg = 0;
    if (nagg < 0 || nagg > kMaxJoinAgg || (nagg > 0 && !aggs)) MBC_FAIL(MBC_ERR_UNSUPPORTED, "%d aggregates (max %d)", nagg, kMaxJoinAgg);
    *out = nullptr;
    mbc_ctx* ctx = outer->ctx;
    MBC_CUDA(cudaSetDevice(ctx->device));
    if ((outer_sel && (!outer_sel->d_bitmap || outer_sel->nrows != outer->nrows)) ||
        (inner_sel && (!inner_sel->d_bitmap || inner_sel->nrows != inner->nrows)))
        MBC_FAIL(MBC_ERR_ARG, "mbc_bitmap_join: side selections must carry MBC_WANT_BITMAP of the same table");

    // ---- validate terms; classify -------------------------------------------------------------------
    JoinTerm jt[kMaxJoinTerms];
    bool equi = true;
    for (int k = 0; k < njoin; ++k) {
        const mbc_term& s = join_terms[k];
        if (k > 0 && s.conj_id < join_terms[k - 1].conj_id) MBC_FAIL(MBC_ERR_ARG, "join terms must be sorted by conj_id");
        if (s.lhs.kind != MBC_OPERAND_OUTER || s.rhs.kind != MBC_OPERAND_INNER)
            MBC_FAIL(MBC_ERR_ARG, "join term %d must be `outerCol op innerCol`", k);
        if (s.lhs.col < 0 || s.lhs.col >= (int)outer->cols.size() || s.rhs.col < 0 || s.rhs.col >= (int)inner->cols.size())
            MBC_FAIL(MBC_ERR_ARG, "join term %d: column out of range", k);
        int to = outer->cols[s.lhs.col].type, ti = inner->cols[s.rhs.col].type;
        // BitMapQuery.java:446-449 "Invalid JOIN COLUMN ATTR TYPE NOT MATCH."
        if (to != ti) MBC_FAIL(MBC_ERR_ARG, "join term %d: column types differ (%d vs %d)", k, to, ti);
        jt[k].o = join_col(outer, s.lhs.col);
        jt[k].i = join_col(inner, s.rhs.col);
        jt[k].op = s.op;
        jt[k].cmp_type = to;
        jt[k].end_conj = (k == njoin - 1 || join_terms[k + 1].conj_id != s.conj_id) ? 1 : 0;
        const bool single = (k == 0 || join_terms[k - 1].conj_id != s.conj_id) && jt[k].end_conj;
        if (s.op != MBC_OP_EQ || !single || to == MBC_ATTR_REAL) equi = false;
    }
    for (int f = 0; f < nproj; ++f) {
        const mbc_table* t = proj[f].rel == MBC_OPERAND_OUTER ? outer : proj[f].rel == MBC_OPERAND_INNER ? inner : nullptr;
        if (!t || proj[f].col < 0 || proj[f].col >= (int)t->cols.size()) MBC_FAIL(MBC_ERR_ARG, "join projection field %d is invalid", f);
    }
    JoinAgg ja[kMaxJoinAgg];
    memset(ja, 0, sizeof(ja));
    for (int a = 0; a < nagg; ++a) {
        ja[a].kind = aggs[a].kind;
        if (aggs[a].kind == MBC_AGG_COUNT) { ja[a].type = MBC_ATTR_INTEGER; ja[a].side = 0; continue; }
        if (aggs[a].kind < 0 || aggs[a].kind > MBC_AGG_MAX) MBC_FAIL(MBC_ERR_ARG, "aggregate %d: unknown kind", a);
        if (aggs[a].col < 0 || aggs[a].col >= nproj) MBC_FAIL(MBC_ERR_ARG, "aggregate %d addresses projected field %d of %d", a, aggs[a].col, nproj);
        const mbc_projspec& pf = proj[aggs[a].col];
        const mbc_table* t = pf.rel == MBC_OPERAND_OUTER ? outer : inner;
        if (t->cols[pf.col].type == MBC_ATTR_STRING) MBC_FAIL(MBC_ERR_UNSUPPORTED, "aggregate %d over a string field", a);
        ja[a].type = t->cols[pf.col].type;
        ja[a].side = pf.rel == MBC_OPERAND_OUTER ? 1 : 2;
        ja[a].src = t->cols[pf.col].d;
    }

    JoinSide so{outer_sel ? outer_sel->d_bitmap : nullptr, outer->has_deleted ? outer->d_deleted : nullptr, outer->nrows};
    JoinSide si{inner_sel ? inner_sel->d_bitmap : nullptr, inner->has_deleted ? inner->d_deleted : nullptr, inner->nrows};
    const bool want_pairs = (want & (MBC_WANT_POSITIONS | MBC_WANT_COLUMNS | MBC_WANT_TUPLES)) != 0;

    mbc_result* r = new mbc_result();
    r->kind = mbc_result::kJoin;
    r->ctx = ctx;
    ctx_retain(ctx);
    r->want = want;
    r->nrows = 0;
    std::vector<void*> temps;
    auto fail = [&](int32_t s) {
        for (void* t : temps) dev_free(ctx, t);
        mbc_result_free(r);
        return s;
    };
#define JTRY(x) do { int32_t _s = (x); if (_s != MBC_OK) return fail(_s); } while (0)
#define JCUDA(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) { set_error("CUDA error %s at %s:%d", cudaGetErrorString(_e), __FILE__, __LINE__); return fail(MBC_ERR_CUDA); } } while (0)
    auto talloc = [&](void** p, size_t bytes, bool zero) -> int32_t {
        int32_t s = dev_alloc(ctx, p, bytes, zero);
        if (s == MBC_OK) temps.push_back(*p);
        return s;
    };

    begin_timing(ctx);
    int64_t npairs = 0;
    unsigned long long agg_raw[kMaxJoinAgg] = {0};
    int64_t* d_pair_o = nullptr;
    int64_t* d_pair_i = nullptr;

    if (equi) {
        // ---- group map ---------------------------------------------------------------------------
        EquiParams ep;
        memset(&ep, 0, sizeof(ep));
        GroupMap& g = ep.g;
        int nkeys = 0;
        for (int k = 0; k < njoin; ++k) { g.okey[nkeys] = jt[k].o; g.ikey[nkeys] = jt[k].i; ++nkeys; }
        g.nkeys = nkeys;
        bool direct = false;
        if (nkeys == 1 && !jt[0].o.is_str) {
            long long* d_mm = nullptr;
            JTRY(talloc((void**)&d_mm, 16, false));
            long long init[2] = {INT64_MAX, INT64_MIN}, mm[2];
            JCUDA(cudaMemcpyAsync(d_mm, init, 16, cudaMemcpyHostToDevice, ctx->stream));
            if (outer->nrows > 0) {
                join_minmax_kernel<<<grid_for(ctx, outer->nrows), 256, 0, ctx->stream>>>((const int32_t*)jt[0].o.ptr, so, d_mm);
                ctx->launches++;
            }
            JCUDA(cudaMemcpyAsync(mm, d_mm, 16, cudaMemcpyDeviceToHost, ctx->stream));
            JCUDA(cudaStreamSynchronize(ctx->stream));
            if (mm[0] <= mm[1]) {
                long long range = mm[1] - mm[0] + 1;
                // direct addressing when the table (2 x 4 B per key) is not much larger than a hash table would be
                if (range <= std::max<long long>(4 * outer->nrows, 1 << 20) && range <= (1ll << 30)) {
                    direct = true;
                    g.mode = 0; g.kmin = mm[0]; g.kmax = mm[1]; g.ngroups = (uint32_t)range;
                }
            } else {
                direct = true;               // no outer row selected: empty join
                g.mode = 0; g.kmin = 0; g.kmax = -1; g.ngroups = 1;
            }
        }
        if (!direct) {
            uint64_t cap = 1024;
            while (cap < (uint64_t)std::max<int64_t>(outer->nrows, 1) * 2) cap <<= 1;
            if (cap > (1ull << 31)) return fail((set_error("join: outer side too large for the hash table"), MBC_ERR_UNSUPPORTED));
            g.mode = 1; g.mask = (uint32_t)(cap - 1); g.ngroups = (uint32_t)cap;
            JTRY(talloc((void**)&g.slots, cap * 8, true));
        }
        JTRY(talloc((void**)&ep.n_outer, (size_t)g.ngroups * 4, true));
        JTRY(talloc((void**)&ep.n_inner, (size_t)g.ngroups * 4, true));
        JTRY(talloc((void**)&ep.overflow, 16, true));
        ep.outer = so;
        ep.inner = si;
        ep.nagg = nagg;
        memcpy(ep.aggs, ja, sizeof(ja));
        const int grid_i = grid_for(ctx, inner->nrows, 16), grid_o = grid_for(ctx, outer->nrows, 16);
        const int pgrid = std::max(grid_i, grid_o);
        JTRY(talloc((void**)&ep.partials, (size_t)std::max(nagg, 1) * pgrid * 8, true));
        if (want_pairs) JTRY(talloc((void**)&ep.inner_match, (size_t)inner->words_pad * 4, true));

        if (outer->nrows > 0) {
            join_outer_count_kernel<<<grid_o, 256, 0, ctx->stream>>>(ep);
            ctx->launches++;
        }
        // inner pass: n_inner, COUNT, inner-side aggregates
        std::vector<unsigned long long> part((size_t)std::max(nagg, 1) * pgrid);
        auto fold = [&](int side, int grid) -> int32_t {
            MBC_CUDA(cudaMemcpyAsync(part.data(), ep.partials, part.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
            MBC_CUDA(cudaStreamSynchronize(ctx->stream));
            for (int a = 0; a < nagg; ++a) {
                const bool mine = (ja[a].side == 0 && side == 2) || ja[a].side == side;
                if (!mine) continue;
                const bool integral = ja[a].kind == MBC_AGG_COUNT || ja[a].type == MBC_ATTR_INTEGER;
                const bool additive = ja[a].kind == MBC_AGG_COUNT || ja[a].kind == MBC_AGG_SUM;
                long long ri = additive ? 0 : ja[a].kind == MBC_AGG_MIN ? (long long)INT32_MAX : (long long)INT32_MIN;
                double rf = additive ? 0.0 : ja[a].kind == MBC_AGG_MIN ? INFINITY : -INFINITY;
                for (int b = 0; b < grid; ++b) {
                    unsigned long long raw = part[(size_t)a * grid + b];
                    long long xi = (long long)raw;
                    double xf;
                    memcpy(&xf, &raw, 8);
                    ri = additive ? ri + xi : ja[a].kind == MBC_AGG_MIN ? std::min(ri, xi) : std::max(ri, xi);
                    rf = additive ? rf + xf : ja[a].kind == MBC_AGG_MIN ? std::min(rf, xf) : std::max(rf, xf);
                }
                if (integral) agg_raw[a] = (unsigned long long)ri; else memcpy(&agg_raw[a], &rf, 8);
            }
            return MBC_OK;
        };
        // COUNT is always needed (it sizes the pair list): make sure one COUNT aggregate runs
        int count_slot = -1;
        for (int a = 0; a < nagg; ++a) if (ja[a].kind == MBC_AGG_COUNT) count_slot = a;
        EquiParams ep_inner = ep;
        if (count_slot < 0) {
            if (nagg == kMaxJoinAgg) return fail((set_error("join: add a COUNT aggregate or use fewer aggregates"), MBC_ERR_UNSUPPORTED));
            // run the inner pass with an extra hidden COUNT
            ep_inner.aggs[nagg].kind = MBC_AGG_COUNT; ep_inner.aggs[nagg].type = MBC_ATTR_INTEGER; ep_inner.aggs[nagg].side = 0;
            ep_inner.nagg = nagg + 1;
            dev_free(ctx, ep.partials);
            temps.erase(std::find(temps.begin(), temps.end(), (void*)ep.partials));
            JTRY(talloc((void**)&ep.partials, (size_t)(nagg + 1) * pgrid * 8, true));
            ep_inner.partials = ep.partials;
            part.resize((size_t)(nagg + 1) * pgrid);
        }
        // unique-key aggregate path: direct addressing, aggregates only, every key on at most one outer row, and at most
        // three distinct outer-side aggregate columns (they ride in the key's slot)
        bool unique_fast = false;
        // (an inner side thinned by a selection bitmap keeps the general path: measured 3.1 ms vs 4.5 ms on C4's 10 % run --
        // most lanes of the batched kernel idle there)
        const char* force = getenv("MBC_JOIN_UNIQUE");               // tests: "0" = never, "1" = whenever legal
        const bool allow = force ? atoi(force) != 0 : !si.sel;
        if (direct && !want_pairs && allow && outer->nrows > 0 && inner->nrows > 0 && g.kmin <= g.kmax) {
            const void* slot_cols[3] = {nullptr, nullptr, nullptr};
            int nslot = 0;
            bool fits = true;
            for (int a = 0; a < ep_inner.nagg && fits; ++a) {
                JoinAgg& ga = ep_inner.aggs[a];
                if (ga.side != 1) continue;
                int w = -1;
                for (int c = 0; c < nslot; ++c) if (slot_cols[c] == ga.src) w = c;
                if (w < 0) { if (nslot == 3) { fits = false; break; } slot_cols[nslot] = ga.src; w = nslot++; }
                ga.slot = w + 1;
            }
            const int valw = nslot == 3 ? 4 : nslot;
            ep_inner.pre[0] = ep_inner.pre[1] = -1;
            for (int a = 0, n = 0; a < ep_inner.nagg && n < 2; ++a)
                if (ep_inner.aggs[a].side == 2 && ep_inner.aggs[a].kind != MBC_AGG_COUNT) ep_inner.pre[n++] = a;
            if (fits) {
                int flags[2] = {0, 0};                                    // duplicate flag, selected outer rows
                JCUDA(cudaMemcpyAsync(flags, ep.overflow + 1, 8, cudaMemcpyDeviceToHost, ctx->stream));
                JCUDA(cudaStreamSynchronize(ctx->stream));
                if (!flags[0]) {
                    const bool dense = (uint32_t)flags[1] == g.ngroups;       // unique + as many rows as keys in range
                    uint32_t *present = nullptr, *slots = nullptr;
                    JTRY(talloc((void**)&present, ((size_t)g.ngroups + 31) / 32 * 4, true));
                    if (valw) JTRY(talloc((void**)&slots, (size_t)g.ngroups * valw * 4, false));
#define MBC_UNIQUE(V)                                                                                                          \
    join_slot_build_kernel<V><<<grid_o, 256, 0, ctx->stream>>>(ep_inner, present, slots, slot_cols[0], slot_cols[1], slot_cols[2]); \
    if (dense) join_unique_pass_kernel<V, true><<<grid_i, 256, 0, ctx->stream>>>(ep_inner, present, slots);                      \
    else join_unique_pass_kernel<V, false><<<grid_i, 256, 0, ctx->stream>>>(ep_inner, present, slots)
                    if (valw == 0) { MBC_UNIQUE(0); }
                    else if (valw == 1) { MBC_UNIQUE(1); }
                    else if (valw == 2) { MBC_UNIQUE(2); }
                    else { MBC_UNIQUE(4); }
#undef MBC_UNIQUE
                    ctx->launches += 2;
                    unique_fast = true;
                }
            }
        }
        if (!unique_fast && inner->nrows > 0) {
            join_agg_pass_kernel<2><<<grid_i, 256, 0, ctx->stream>>>(ep_inner);
            ctx->launches++;
        }
        {
            int overflow = 0;
            JCUDA(cudaMemcpyAsync(&overflow, ep.overflow, 4, cudaMemcpyDeviceToHost, ctx->stream));
            JCUDA(cudaMemcpyAsync(part.data(), ep.partials, part.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
            JCUDA(cudaStreamSynchronize(ctx->stream));
            if (overflow) return fail((set_error("join: hash table overflow"), MBC_ERR_CUDA));
            const int na = ep_inner.nagg;
            const int cs = count_slot >= 0 ? count_slot : nagg;
            long long cnt = 0;
            if (inner->nrows > 0) for (int b = 0; b < grid_i; ++b) cnt += (long long)part[(size_t)cs * grid_i + b];
            npairs = cnt;
            (void)na;
            if (inner->nrows > 0) {
                for (int a = 0; a < nagg; ++a) {
                    const bool mine = ja[a].side == 0 || ja[a].side == 2 || unique_fast;
                    if (!mine) continue;
                    const bool integral = ja[a].kind == MBC_AGG_COUNT || ja[a].type == MBC_ATTR_INTEGER;
                    const bool additive = ja[a].kind == MBC_AGG_COUNT || ja[a].kind == MBC_AGG_SUM;
                    long long ri = additive ? 0 : ja[a].kind == MBC_AGG_MIN ? (long long)INT32_MAX : (long long)INT32_MIN;
                    double rf = additive ? 0.0 : ja[a].kind == MBC_AGG_MIN ? INFINITY : -INFINITY;
                    for (int b = 0; b < grid_i; ++b) {
                        unsigned long long raw = part[(size_t)a * grid_i + b];
                        long long xi = (long long)raw;
                        double xf;
                        memcpy(&xf, &raw, 8);
                        ri = additive ? ri + xi : ja[a].kind == MBC_AGG_MIN ? std::min(ri, xi) : std::max(ri, xi);
                        rf = additive ? rf + xf : ja[a].kind == MBC_AGG_MIN ? std::min(rf, xf) : std::max(rf, xf);
                    }
                    if (integral) agg_raw[a] = (unsigned long long)ri; else memcpy(&agg_raw[a], &rf, 8);
                }
            }
        }
        // outer pass: outer-side aggregates weighted by n_inner
        bool any_outer_agg = false;
        for (int a = 0; a < nagg; ++a) any_outer_agg |= ja[a].side == 1;
        if (any_outer_agg && outer->nrows > 0 && !unique_fast) {
            JCUDA(cudaMemsetAsync(ep.partials, 0, (size_t)std::max(nagg, 1) * pgrid * 8, ctx->stream));
            join_agg_pass_kernel<1><<<grid_o, 256, 0, ctx->stream>>>(ep);
            ctx->launches++;
            part.resize((size_t)std::max(nagg, 1) * pgrid);
            JTRY(fold(1, grid_o));
        }

        // ---- pair list ------------------------------------------------------------------------------
        if (want_pairs && npairs > 0) {
            if (npairs > (1ll << 31)) return fail((set_error("join: %lld result pairs; ask for aggregates only", (long long)npairs), MBC_ERR_UNSUPPORTED));
            mbc_result *ro = nullptr, *ri = nullptr;
            JTRY(compact_side(inner, ep.inner_match, &ri));
            // outer rows that are selected (a scan over the selection bitmap, or all rows)
            int32_t s2 = compact_side(outer, so.sel, &ro);
            if (s2 != MBC_OK) { mbc_result_free(ri); return fail(s2); }
            const int64_t nim = ri->count, nol = ro->count;
            uint32_t *keys = nullptr, *vals = nullptr, *ocnt = nullptr, *ogrp = nullptr;
            unsigned long long *gstart = nullptr, *ooff = nullptr;
            int32_t s3 = MBC_OK;
            if ((s3 = talloc((void**)&keys, (size_t)std::max<int64_t>(nim, 1) * 4, false)) != MBC_OK ||
                (s3 = talloc((void**)&vals, (size_t)std::max<int64_t>(nim, 1) * 4, false)) != MBC_OK ||
                (s3 = talloc((void**)&ocnt, (size_t)std::max<int64_t>(nol, 1) * 4, false)) != MBC_OK ||
                (s3 = talloc((void**)&ogrp, (size_t)std::max<int64_t>(nol, 1) * 4, false)) != MBC_OK ||
                (s3 = talloc((void**)&gstart, ((size_t)g.ngroups + 1) * 8, false)) != MBC_OK ||
                (s3 = talloc((void**)&ooff, ((size_t)nol + 1) * 8, false)) != MBC_OK ||
                (s3 = dev_alloc(ctx, (void**)&d_pair_o, (size_t)npairs * 8, false)) != MBC_OK ||
                (s3 = dev_alloc(ctx, (void**)&d_pair_i, (size_t)npairs * 8, false)) != MBC_OK) {
                mbc_result_free(ri); mbc_result_free(ro);
                return fail(s3);
            }
            join_group_keys_kernel<<<grid_for(ctx, nim), 256, 0, ctx->stream>>>(g, ri->d_pos, nim, inner->pos_base, keys, vals);
            ctx->launches++;
            int key_bits = 1;
            while ((1ull << key_bits) < (unsigned long long)g.ngroups) ++key_bits;
            s3 = radix_sort_pairs(ctx, keys, vals, nim, key_bits);
            if (s3 == MBC_OK) s3 = exclusive_scan_u32(ctx, ep.n_inner, g.ngroups, gstart);
            if (s3 == MBC_OK) {
                join_outer_counts_kernel<<<grid_for(ctx, nol), 256, 0, ctx->stream>>>(g, ro->d_pos, nol, outer->pos_base, ep.n_inner, ocnt, ogrp);
                ctx->launches++;
                s3 = exclusive_scan_u32(ctx, ocnt, nol, ooff);
            }
            if (s3 == MBC_OK) {
                join_fill_pairs_kernel<<<grid_for(ctx, npairs), 256, 0, ctx->stream>>>(ooff, nol, ro->d_pos, ogrp, gstart, vals,
                                                                                    inner->pos_base, npairs, d_pair_o, d_pair_i);
                ctx->launches++;
                if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) s3 = MBC_ERR_CUDA;
            }
            mbc_result_free(ri);
            mbc_result_free(ro);
            if (s3 != MBC_OK) { dev_free(ctx, d_pair_o); dev_free(ctx, d_pair_i); return fail(s3); }
        }
    } else {
        // ---- THETA path -----------------------------------------------------------------------------
        mbc_result *ro = nullptr, *ri = nullptr;
        JTRY(compact_side(outer, so.sel, &ro));
        int32_t s2 = compact_side(inner, si.sel, &ri);
        if (s2 != MBC_OK) { mbc_result_free(ro); return fail(s2); }
        ThetaParams tp;
        memset(&tp, 0, sizeof(tp));
        tp.outer_pos = ro->d_pos; tp.inner_pos = ri->d_pos;
        tp.n_outer = ro->count; tp.n_inner = ri->count;
        tp.outer_base = outer->pos_base; tp.inner_base = inner->pos_base;
        tp.nterms = njoin;
        memcpy(tp.terms, jt, sizeof(JoinTerm) * njoin);
        tp.chunks = (int)std::max<int64_t>(1, (tp.n_inner + kThetaChunk - 1) / kThetaChunk);
        int32_t s3 = MBC_OK;
        unsigned long long* offs = nullptr;
        if (tp.n_outer > 0 && tp.n_inner > 0) {
            if (tp.chunks > 65535 || tp.n_outer * (int64_t)tp.chunks > (1ll << 31))
                s3 = (set_error("theta join of %lld x %lld survivors is too large for the nested-loop path", (long long)tp.n_outer, (long long)tp.n_inner), MBC_ERR_UNSUPPORTED);
            const int64_t ncnt = tp.n_outer * tp.chunks;
            if (s3 == MBC_OK) s3 = talloc((void**)&tp.counts, (size_t)ncnt * 4, false);
            if (s3 == MBC_OK) s3 = talloc((void**)&offs, ((size_t)ncnt + 1) * 8, false);
            if (s3 == MBC_OK) {
                dim3 grid((unsigned)tp.n_outer, (unsigned)tp.chunks);
                join_theta_kernel<false><<<grid, kThetaThreads, 0, ctx->stream>>>(tp);
                ctx->launches++;
                s3 = exclusive_scan_u32(ctx, tp.counts, ncnt, offs);
                unsigned long long total = 0;
                if (s3 == MBC_OK && (cudaMemcpyAsync(&total, offs + ncnt, 8, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
                                     cudaStreamSynchronize(ctx->stream) != cudaSuccess)) s3 = MBC_ERR_CUDA;
                npairs = (int64_t)total;
                if (s3 == MBC_OK && npairs > 0) {
                    if (npairs > (1ll << 31)) s3 = (set_error("theta join: %lld result pairs", (long long)npairs), MBC_ERR_UNSUPPORTED);
                    if (s3 == MBC_OK) s3 = dev_alloc(ctx, (void**)&d_pair_o, (size_t)npairs * 8, false);
                    if (s3 == MBC_OK) s3 = dev_alloc(ctx, (void**)&d_pair_i, (size_t)npairs * 8, false);
                    if (s3 == MBC_OK) {
                        tp.offsets = offs; tp.out_o = d_pair_o; tp.out_i = d_pair_i;
                        join_theta_kernel<true><<<grid, kThetaThreads, 0, ctx->stream>>>(tp);
                        ctx->launches++;
                        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) s3 = MBC_ERR_CUDA;
                    }
                }
            }
        }
        mbc_result_free(ro);
        mbc_result_free(ri);
        if (s3 != MBC_OK) { dev_free(ctx, d_pair_o); dev_free(ctx, d_pair_i); return fail(s3); }
    }

    // ---- materialise: positions + projected columns ----------------------------------------------------------
    r->count = npairs;
    r->capacity = npairs;
    r->d_pos = d_pair_o;
    r->d_pos2 = d_pair_i;
    const bool need_cols = ((want & (MBC_WANT_COLUMNS | MBC_WANT_TUPLES)) != 0 || (!equi && nagg > 0)) && nproj > 0;
    if (need_cols) {
        const int64_t cap = round_up(std::max<int64_t>(npairs, 1), kPadRows);     // padded: the scan engine may read these
        for (int f = 0; f < nproj; ++f) {
            const mbc_table* t = proj[f].rel == MBC_OPERAND_OUTER ? outer : inner;
            const Column& c = t->cols[proj[f].col];
            mbc_result::Col rc{c.type, c.width, c.stride, nullptr, nullptr};
            JTRY(dev_alloc(ctx, &rc.d, (size_t)cap * c.stride, true));
            r->cols.push_back(rc);
            if (npairs > 0) {
                GatherParams gp;
                gp.pos = proj[f].rel == MBC_OPERAND_OUTER ? d_pair_o : d_pair_i;
                gp.base = t->pos_base;
                gp.npairs = npairs;
                gp.src = c.d;
                gp.dst = rc.d;
                gp.stride = c.stride;
                gp.pad = 0;
                join_gather_kernel<<<grid_for(ctx, npairs), 256, 0, ctx->stream>>>(gp);
                ctx->launches++;
            }
        }
    }
    if (!equi && nagg > 0) {
        // aggregates of the theta path: a scan with no predicate over the projected result columns
        mbc_table view;
        view.ctx = ctx;
        view.nrows = npairs;
        view.nrows_pad = round_up(std::max<int64_t>(npairs, 1), kPadRows);
        view.words_pad = view.nrows_pad / 32;
        std::vector<mbc_aggspec> specs(aggs, aggs + nagg);
        for (auto& rc : r->cols) {
            Column c;
            c.type = rc.type; c.width = rc.width; c.stride = rc.stride; c.d = rc.d;
            view.cols.push_back(c);
        }
        view.bm.resize(view.cols.size());
        ScanRequest rq;
        rq.table = &view;
        rq.want = MBC_WANT_AGG;
        rq.aggs = specs.data();
        rq.nagg = nagg;
        mbc_result* ar = nullptr;
        int32_t s4 = run_scan(rq, &ar);
        view.cols.clear();
        if (s4 != MBC_OK) return fail(s4);
        r->aggs = ar->aggs;
        mbc_result_free(ar);
    } else {
        r->aggs.resize(nagg);
        for (int a = 0; a < nagg; ++a) {
            mbc_result::Agg& g = r->aggs[a];
            g.kind = ja[a].kind;
            g.type = ja[a].type;
            const bool integral = g.kind == MBC_AGG_COUNT || g.type == MBC_ATTR_INTEGER;
            if (integral) { g.i = (int64_t)agg_raw[a]; g.f = (double)g.i; }
            else { double d; memcpy(&d, &agg_raw[a], 8); g.f = d; g.i = real_agg_as_i64(d); }
            g.valid = (g.kind == MBC_AGG_COUNT || g.kind == MBC_AGG_SUM) ? 1 : (npairs > 0);
            if (!g.valid) { g.i = 0; g.f = 0.0; }
        }
    }
    end_timing(ctx);
    JCUDA(cudaGetLastError());
    for (void* t : temps) dev_free(ctx, t);
    temps.clear();
    if (!(want & (MBC_WANT_COLUMNS | MBC_WANT_TUPLES))) {
        // columns were only needed for the aggregates
        for (auto& c : r->cols) dev_free(ctx, c.d);
        r->cols.clear();
    }
    if (!(want & MBC_WANT_POSITIONS)) {
        // keep the device lists (NCCL callers), but do not copy them to the host
    }
    int32_t s5 = finish_result_host(r);
    if (s5 != MBC_OK) { mbc_result_free(r); return s5; }
#undef JTRY
#undef JCUDA
    *out = r;
    return MBC_OK;
}
