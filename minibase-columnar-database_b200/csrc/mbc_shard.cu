// mbc_shard.cu -- TID-range shards on the GPUs of one node: the result gather over NVLink peer memory, under the C ABI.
//
// SURVEY.md 8(e): rows shard by contiguous position range, every GPU scans its slice with no data-path collective, and
// only counts, aggregates and the qualifying rows travel.  Rank order is position order, so the whole table's result is
// the concatenation of the ranks' results: rank r's rows start at the sum of the counts of ranks < r.
//
// The root rank owns a WINDOW in its HBM (cudaMalloc, exported with cudaIpcGetMemHandle; peers map it with
// cudaIpcOpenMemHandle, or -- inside one process, the shape a single JVM driving 8 GPUs has -- reach it through
// cudaDeviceEnablePeerAccess).  One kernel per rank and step (shard_push_kernel) then does the whole exchange:
//   1. (shard_publish_kernel, right behind the scan) the rank's count and its COUNT/SUM/MIN/MAX block are published in the
//      window's control area (release, system scope),
//   2. the push reads the counts of the lower ranks from the same area (they ran the same scan at the same time) -> its offset,
//   3. stores its positions and projected columns straight into the root's buffers at that offset (coalesced stores over
//      NVLink; nothing is staged, padded or sent to ranks that do not need it),
//   4. signals completion.
// The root waits for every rank's signal with a one-warp kernel and folds the aggregate blocks (the all-reduce of
// COUNT/SUM/MIN/MAX is a fold of `world` 72-byte blocks).  No NCCL kernel runs next to the scans, and the bytes that cross
// NVLink are exactly the gathered rows.  Two window slots alternate so that step i's push may overlap step i+1's scans.
//
// This is the reference-facing replacement of "run the same query on every partition and concatenate": the reference
// itself has no partitioning (SURVEY F2); the operator it accelerates is still iterator/ColumnarFileScan.java:156-188.
#include <cstring>
#include <algorithm>

#include "mbc_internal.cuh"

namespace mbc {

constexpr int kShardMaxWorld = 32;
constexpr int kShardSlots = 2;
constexpr unsigned long long kCountMask = (1ull << 40) - 1ull;     // published word = epoch << 40 | count

struct ShardCtl {                       // one per (slot, rank), 128 bytes
    unsigned long long pub;             // epoch << 40 | count: the rank's result size of this step
    unsigned long long done;            // epoch: the rank's rows have landed in the window
    unsigned long long aggs[kMaxAgg + 1];
    unsigned long long dropped;         // rows that did not fit the window (0 in a correct run)
    unsigned long long pad[16 - (kMaxAgg + 1) - 3];
};
static_assert(sizeof(ShardCtl) == 128, "control block layout");

struct ShardHeader {                    // start of the window
    unsigned long long consumed;        // the root has released every step <= consumed
    unsigned long long pad[15];
};

struct PushParams {
    ShardHeader* hdr;                   // root memory
    ShardCtl* ctl;                      // root memory: the slot's [world] control blocks
    int32_t rank, world;
    unsigned long long epoch;
    const unsigned long long* my_aggs;  // local: kMaxAgg aggregates, then the count
    int64_t cap_rows;
    const int64_t* src_pos;
    int64_t* dst_pos;
    int32_t ncols, pad;
    const void* src[kMaxProj];
    void* dst[kMaxProj];
    int32_t stride[kMaxProj];
    unsigned int* blocks_done;          // local
};

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Copy nbytes (a multiple of 4; src and dst 4-byte aligned) with 128-bit stores wherever dst allows: the destination is the
// root's HBM behind NVLink, where a 16-byte store per thread (512 bytes per warp instruction) fills the link's packets; the
// source is local HBM, read with whatever alignment the (arbitrary) output offset leaves it.
__device__ __forceinline__ void push_copy(const char* __restrict__ src, char* __restrict__ dst, long long nbytes) {
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    long long head = (16 - (long long)(reinterpret_cast<uintptr_t>(dst) & 15)) & 15;
    if (head > nbytes) head = nbytes;
    if (tid < head / 4) reinterpret_cast<uint32_t*>(dst)[tid] = reinterpret_cast<const uint32_t*>(src)[tid];
    const char* s = src + head;
    char* d = dst + head;
    const long long n16 = (nbytes - head) / 16;
    if ((reinterpret_cast<uintptr_t>(s) & 15) == 0) {              // grid-uniform: both sides 16-byte aligned
        const uint4* s4 = reinterpret_cast<const uint4*>(s);
        uint4* d4 = reinterpret_cast<uint4*>(d);
        long long i = tid;
        for (; i + 3 * nthreads < n16; i += 4 * nthreads) {        // four independent loads in flight per thread
            const uint4 a = s4[i], b = s4[i + nthreads], c = s4[i + 2 * nthreads], e = s4[i + 3 * nthreads];
            d4[i] = a; d4[i + nthreads] = b; d4[i + 2 * nthreads] = c; d4[i + 3 * nthreads] = e;
        }
        for (; i < n16; i += nthreads) d4[i] = s4[i];
    } else {
        const uint32_t* s1 = reinterpret_cast<const uint32_t*>(s);
        uint4* d4 = reinterpret_cast<uint4*>(d);
        long long i = tid;
        for (; i + nthreads < n16; i += 2 * nthreads) {
            const uint4 a = make_uint4(s1[4 * i], s1[4 * i + 1], s1[4 * i + 2], s1[4 * i + 3]);
            const long long k = i + nthreads;
            const uint4 b = make_uint4(s1[4 * k], s1[4 * k + 1], s1[4 * k + 2], s1[4 * k + 3]);
            d4[i] = a; d4[k] = b;
        }
        for (; i < n16; i += nthreads) d4[i] = make_uint4(s1[4 * i], s1[4 * i + 1], s1[4 * i + 2], s1[4 * i + 3]);
    }
    const long long done = head + n16 * 16;
    const long long tail = (nbytes - done) / 4;
    if (tid < tail) reinterpret_cast<uint32_t*>(dst + done)[tid] = reinterpret_cast<const uint32_t*>(src + done)[tid];
}

__global__ void __launch_bounds__(256) shard_push_kernel(const __grid_constant__ PushParams p) {
    __shared__ long long s_off, s_cnt;
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        const long long count = (long long)p.my_aggs[kMaxAgg];      // published by shard_publish_kernel when the scan finished
        // the slot was last used by step epoch - kShardSlots: the root must have released it
        if (lane == 0)
            while (ld_acquire_sys(&p.hdr->consumed) + kShardSlots < p.epoch) __nanosleep(200);
        long long off = 0;
        if (lane < p.rank) {                                        // counts of the lower ranks: they run the same step
            unsigned long long v = ld_acquire_sys(&p.ctl[lane].pub);
            while ((v >> 40) != p.epoch) {
                __nanosleep(200);
                v = ld_acquire_sys(&p.ctl[lane].pub);
            }
            off = (long long)(v & kCountMask);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) off += __shfl_xor_sync(0xFFFFFFFFu, off, o);
        if (lane == 0) { s_off = off; s_cnt = count; }
    }
    __syncthreads();
    const long long off = s_off;
    long long n = s_cnt;
    if (off + n > p.cap_rows) n = max(0ll, p.cap_rows - off);       // never write past the window; the loss is reported
    if (p.src_pos) push_copy(reinterpret_cast<const char*>(p.src_pos), reinterpret_cast<char*>(p.dst_pos + off), n * 8);
    for (int c = 0; c < p.ncols; ++c) {
        const long long st = p.stride[c];
        push_copy(reinterpret_cast<const char*>(p.src[c]), reinterpret_cast<char*>(p.dst[c]) + off * st, n * st);
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int prev = atomicAdd(p.blocks_done, 1u);
        if (prev == gridDim.x - 1) {                                // every block's stores are fenced: signal the root
            *p.blocks_done = 0u;
            ShardCtl* mine = p.ctl + p.rank;
            mine->dropped = (unsigned long long)(s_cnt - n);
            __threadfence_system();
            st_release_sys(&mine->done, p.epoch);
        }
    }
}

// The rank's count and aggregate block reach the root's control area before any row is pushed: a rank's push only waits
// for the (80-byte) publications of the lower ranks, never for their rows.
__global__ void shard_publish_kernel(ShardCtl* ctl, int rank, unsigned long long epoch, const unsigned long long* my_aggs) {
    if (threadIdx.x == 0) {
        ShardCtl* mine = ctl + rank;
        for (int a = 0; a <= kMaxAgg; ++a) mine->aggs[a] = my_aggs[a];
        __threadfence_system();
        st_release_sys(&mine->pub, (epoch << 40) | (my_aggs[kMaxAgg] & kCountMask));
    }
}

// Copy-engine form of the push: this one-warp kernel only resolves the rank's offset (and waits for the window slot); the
// rows then travel as cudaMemcpyAsync peer copies (DMA engines, no SM), and shard_done_kernel signals the root behind them.
__global__ void shard_offset_kernel(const ShardHeader* hdr, const ShardCtl* ctl, int rank, unsigned long long epoch, const unsigned long long* my_aggs,
                                    long long cap_rows, long long* out /* host-mapped: offset, rows that fit, rows dropped */) {
    const int lane = threadIdx.x;
    if (lane == 0)
        while (ld_acquire_sys(&hdr->consumed) + kShardSlots < epoch) __nanosleep(200);
    long long off = 0;
    if (lane < rank) {
        unsigned long long v = ld_acquire_sys(&ctl[lane].pub);
        while ((v >> 40) != epoch) {
            __nanosleep(200);
            v = ld_acquire_sys(&ctl[lane].pub);
        }
        off = (long long)(v & kCountMask);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) off += __shfl_xor_sync(0xFFFFFFFFu, off, o);
    if (lane == 0) {
        const long long count = (long long)my_aggs[kMaxAgg];
        long long n = count;
        if (off + n > cap_rows) n = max(0ll, cap_rows - off);
        out[0] = off;
        out[1] = n;
        out[2] = count - n;
        __threadfence_system();
    }
}

__global__ void shard_done_kernel(ShardCtl* ctl, int rank, unsigned long long epoch, unsigned long long dropped) {
    if (threadIdx.x == 0) {
        ctl[rank].dropped = dropped;
        __threadfence_system();
        st_release_sys(&ctl[rank].done, epoch);
    }
}

// root: wait until every rank's rows of step `epoch` have landed, then leave the per-rank counts and aggregate blocks in
// `summary` ([world] x {count, dropped, aggs[kMaxAgg]})
__global__ void shard_wait_kernel(const ShardCtl* ctl, int world, unsigned long long epoch, unsigned long long* summary) {
    const int lane = threadIdx.x;
    if (lane < world) {
        while (ld_acquire_sys(&ctl[lane].done) != epoch) __nanosleep(200);
        unsigned long long* o = summary + (size_t)lane * (kMaxAgg + 2);
        o[0] = ld_acquire_sys(&ctl[lane].pub) & kCountMask;
        o[1] = ctl[lane].dropped;
        for (int a = 0; a < kMaxAgg; ++a) o[2 + a] = ctl[lane].aggs[a];
    }
}

__global__ void shard_release_kernel(ShardHeader* hdr, unsigned long long epoch) {
    if (threadIdx.x == 0) st_release_sys(&hdr->consumed, epoch);
}

}  // namespace mbc

using namespace mbc;

struct mbc_shard {
    mbc_ctx* ctx = nullptr;
    int rank = 0, world = 1;
    char* win = nullptr;                // the root's window as seen from this rank
    bool owned = false, ipc = false;
    int64_t cap_rows = 0;
    int ncols = 0;
    int strides[kMaxProj] = {0};
    size_t off_ctl = 0, off_pos[kShardSlots] = {0}, off_col[kShardSlots][kMaxProj] = {{0}};
    size_t bytes = 0;
    cudaStream_t side = nullptr;        // pushes may run beside the next step's scans
    cudaEvent_t ev_scan = nullptr, ev_push = nullptr;
    cudaEvent_t ev_push0 = nullptr, ev_push1 = nullptr;   // device time of the last push (mbc_shard_push_ms)
    unsigned int* d_blocks_done = nullptr;
    unsigned long long epoch = 0;       // steps gathered so far (every rank calls mbc_shard_gather once per step)
    unsigned long long* d_summary = nullptr;
    unsigned long long* h_summary = nullptr;
    long long* h_off = nullptr;         // host-mapped: offset / rows / dropped of the copy-engine form
    long long* d_off = nullptr;
    cudaEvent_t ev_off = nullptr;
    int64_t total = 0, dropped = 0;
    unsigned long long collected = 0;   // the step mbc_shard_collect completed, until mbc_shard_release (0: none)
    unsigned long long* d_count_block = nullptr;   // zero aggregates + the count of a row or grouped result (shard_publish_kernel)
    std::vector<int64_t> counts;
    int push_ctas = 0;
};

static void layout_window(mbc_shard* s) {
    size_t o = sizeof(ShardHeader);
    s->off_ctl = o;
    o += sizeof(ShardCtl) * kShardSlots * kShardMaxWorld;
    for (int k = 0; k < kShardSlots; ++k) {
        o = (size_t)round_up((int64_t)o, 256);
        s->off_pos[k] = o;
        o += (size_t)s->cap_rows * 8;
        for (int c = 0; c < s->ncols; ++c) {
            o = (size_t)round_up((int64_t)o, 256);
            s->off_col[k][c] = o;
            o += (size_t)s->cap_rows * s->strides[c];
        }
    }
    s->bytes = (size_t)round_up((int64_t)o, 256);
}

static int32_t set_shape(mbc_shard* s, int64_t capacity_rows, int32_t ncols, const int32_t* col_strides) {
    if (capacity_rows <= 0 || ncols < 0 || ncols > kMaxProj || (ncols > 0 && !col_strides)) MBC_FAIL(MBC_ERR_ARG, "shard window: bad shape");
    for (int c = 0; c < ncols; ++c)
        if (col_strides[c] <= 0 || (col_strides[c] & 3)) MBC_FAIL(MBC_ERR_ARG, "shard window: column %d stride %d", c, col_strides[c]);
    s->cap_rows = capacity_rows;
    s->ncols = ncols;
    for (int c = 0; c < ncols; ++c) s->strides[c] = col_strides[c];
    layout_window(s);
    return MBC_OK;
}

// ---- root-side merges of the gathered rows ----------------------------------------------------------------------------
// The window's rows are the input, row id i = window row i; rank order is position order, so a stable sort of the row ids
// keeps equal keys in ascending global position.

static int32_t merge_check(const mbc_shard* s, const char* fn) {
    if (!s || !s->owned) MBC_FAIL(MBC_ERR_ARG, "%s: only the window's owner merges", fn);
    if (s->epoch == 0 || s->collected != s->epoch) MBC_FAIL(MBC_ERR_ARG, "%s: no collected step (mbc_shard_collect first, mbc_shard_release after)", fn);
    if (s->total > (int64_t)UINT32_MAX) MBC_FAIL(MBC_ERR_UNSUPPORTED, "%s: %lld gathered rows (max 2^32 - 1)", fn, (long long)s->total);
    return MBC_OK;
}

// window column c of the collected step as a table column of type/width d
static int32_t window_column(const mbc_shard* s, const char* fn, int c, const mbc_coldesc& d, Column* out) {
    int stride = 0;
    if ((d.type == MBC_ATTR_INTEGER || d.type == MBC_ATTR_REAL) && d.width == 4) stride = 4;
    else if (d.type == MBC_ATTR_STRING && d.width > 0 && d.width <= kMaxStrStride) stride = str_stride(d.width);
    if (stride == 0) MBC_FAIL(MBC_ERR_ARG, "%s: column %d: type %d width %d", fn, c, d.type, d.width);
    if (stride != s->strides[c]) MBC_FAIL(MBC_ERR_ARG, "%s: column %d has stride %d, the window %d", fn, c, stride, s->strides[c]);
    out->type = d.type;
    out->width = d.width;
    out->stride = stride;
    out->d = s->win + s->off_col[s->epoch % kShardSlots][c];
    return MBC_OK;
}

static int merge_grid(const mbc_ctx* ctx, int64_t n) {
    return (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8));
}

extern "C" {

int32_t mbc_shard_create(mbc_ctx* ctx, int32_t rank, int32_t world, mbc_shard** out) {
    if (!ctx || !out || world < 1 || world > kShardMaxWorld || rank < 0 || rank >= world)
        MBC_FAIL(MBC_ERR_ARG, "mbc_shard_create: rank %d of %d (max %d ranks)", rank, world, kShardMaxWorld);
    *out = nullptr;
    MBC_CUDA(cudaSetDevice(ctx->device));
    mbc_shard* s = new mbc_shard();
    s->ctx = ctx;
    ctx_retain(ctx);
    s->rank = rank;
    s->world = world;
    s->counts.assign(world, 0);
    s->push_ctas = std::max(8, ctx->sm_count / 2);                // enough stores in flight for NVLink; leaves SMs to the scans
    if (const char* e = getenv("MBC_SHARD_PUSH_CTAS")) s->push_ctas = std::max(1, atoi(e));
    if (cudaStreamCreateWithFlags(&s->side, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_scan, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_push, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreate(&s->ev_push0) != cudaSuccess || cudaEventCreate(&s->ev_push1) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_off, cudaEventDisableTiming) != cudaSuccess ||
        cudaHostAlloc((void**)&s->h_off, 64, cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer((void**)&s->d_off, s->h_off, 0) != cudaSuccess ||
        cudaMalloc((void**)&s->d_blocks_done, 64) != cudaSuccess || cudaMemset(s->d_blocks_done, 0, 64) != cudaSuccess ||
        cudaMalloc((void**)&s->d_count_block, (kMaxAgg + 1) * 8) != cudaSuccess ||
        cudaMemset(s->d_count_block, 0, (kMaxAgg + 1) * 8) != cudaSuccess) {
        set_error("mbc_shard_create: %s", cudaGetErrorString(cudaGetLastError()));
        mbc_shard_free(s);
        return MBC_ERR_CUDA;
    }
    *out = s;
    return MBC_OK;
}

void mbc_shard_free(mbc_shard* s) {
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    if (s->side) cudaStreamSynchronize(s->side);
    cudaStreamSynchronize(s->ctx->stream);
    if (s->win) {
        if (s->owned) cudaFree(s->win);
        else if (s->ipc) cudaIpcCloseMemHandle(s->win);
    }
    if (s->d_blocks_done) cudaFree(s->d_blocks_done);
    if (s->d_count_block) cudaFree(s->d_count_block);
    if (s->d_summary) cudaFree(s->d_summary);
    if (s->h_summary) cudaFreeHost(s->h_summary);
    if (s->h_off) cudaFreeHost(s->h_off);
    if (s->ev_off) cudaEventDestroy(s->ev_off);
    if (s->ev_scan) cudaEventDestroy(s->ev_scan);
    if (s->ev_push) cudaEventDestroy(s->ev_push);
    if (s->ev_push0) cudaEventDestroy(s->ev_push0);
    if (s->ev_push1) cudaEventDestroy(s->ev_push1);
    if (s->side) cudaStreamDestroy(s->side);
    mbc_ctx* ctx = s->ctx;
    delete s;
    ctx_release(ctx);
}

int32_t mbc_shard_window_create(mbc_shard* s, int64_t capacity_rows, int32_t ncols, const int32_t* col_strides, uint8_t* handle_out) {
    if (!s || s->win) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_window_create: bad shard (or window exists)");
    MBC_CUDA(cudaSetDevice(s->ctx->device));
    MBC_TRY(set_shape(s, capacity_rows, ncols, col_strides));
    MBC_CUDA(cudaMalloc((void**)&s->win, s->bytes));               // cudaMalloc, not the stream-ordered pool: IPC exports whole allocations
    MBC_CUDA(cudaMemset(s->win, 0, sizeof(ShardHeader) + sizeof(ShardCtl) * kShardSlots * kShardMaxWorld));
    s->owned = true;
    const size_t sum_bytes = (size_t)kShardMaxWorld * (kMaxAgg + 2) * 8;
    MBC_CUDA(cudaMalloc((void**)&s->d_summary, sum_bytes));
    MBC_CUDA(cudaHostAlloc((void**)&s->h_summary, sum_bytes, cudaHostAllocDefault));
    if (handle_out) {
        static_assert(sizeof(cudaIpcMemHandle_t) == MBC_IPC_HANDLE_BYTES, "IPC handle size");
        cudaIpcMemHandle_t h;
        MBC_CUDA(cudaIpcGetMemHandle(&h, s->win));
        memcpy(handle_out, &h, sizeof(h));
    }
    return MBC_OK;
}

int32_t mbc_shard_window_open(mbc_shard* s, const uint8_t* handle, int64_t capacity_rows, int32_t ncols, const int32_t* col_strides) {
    if (!s || s->win || !handle) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_window_open: bad argument");
    MBC_CUDA(cudaSetDevice(s->ctx->device));
    MBC_TRY(set_shape(s, capacity_rows, ncols, col_strides));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    MBC_CUDA(cudaIpcOpenMemHandle((void**)&s->win, h, cudaIpcMemLazyEnablePeerAccess));
    s->ipc = true;
    return MBC_OK;
}

int32_t mbc_shard_window_attach(mbc_shard* s, const mbc_shard* root) {
    if (!s || s->win || !root || !root->win || !root->owned) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_window_attach: bad argument");
    MBC_CUDA(cudaSetDevice(s->ctx->device));
    if (s->ctx->device != root->ctx->device) {
        int can = 0;
        MBC_CUDA(cudaDeviceCanAccessPeer(&can, s->ctx->device, root->ctx->device));
        if (!can) MBC_FAIL(MBC_ERR_UNSUPPORTED, "device %d cannot reach device %d's memory", s->ctx->device, root->ctx->device);
        cudaError_t e = cudaDeviceEnablePeerAccess(root->ctx->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) MBC_CUDA(e);
        cudaGetLastError();
    }
    MBC_TRY(set_shape(s, root->cap_rows, root->ncols, root->strides));
    s->win = root->win;
    return MBC_OK;
}

int32_t mbc_shard_gather(mbc_shard* s, const mbc_result* r, int32_t beside_next_scan) {
    if (!s || !s->win || !r) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_gather: no window / result");
    if (r->ctx != s->ctx) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_gather: the result belongs to another context");
    // the window columns this result fills, and where its count (after kMaxAgg aggregates) is read from
    const void* src[kMaxProj];
    int32_t src_stride[kMaxProj];
    int nsrc = (int)r->cols.size();
    for (int c = 0; c < nsrc && c < kMaxProj; ++c) {
        src[c] = r->cols[c].d;
        src_stride[c] = r->cols[c].stride;
    }
    bool own_count = false;             // rows / groups: the count comes from the host, through d_count_block
    switch (r->kind) {
        case mbc_result::kScan:
            break;
        case mbc_result::kRows:
            if (!(r->want & MBC_WANT_POSITIONS)) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_gather: a sorted result needs MBC_WANT_POSITIONS");
            own_count = true;
            break;
        case mbc_result::kGrouped: {
            // key columns, then one 8-byte column per aggregate: aggregate a's values are the block d_aggs + a * count
            if (nsrc + r->group_nagg > kMaxProj)
                MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_shard_gather: %d key columns + %d aggregates exceed the window's %d columns", nsrc,
                         r->group_nagg, kMaxProj);
            if ((r->want & (MBC_WANT_POSITIONS | MBC_WANT_COLUMNS)) != (MBC_WANT_POSITIONS | MBC_WANT_COLUMNS))
                MBC_FAIL(MBC_ERR_ARG, "mbc_shard_gather: a grouped result needs MBC_WANT_POSITIONS | MBC_WANT_COLUMNS");
            for (int a = 0; a < r->group_nagg; ++a) {
                src[nsrc] = r->d_aggs + (size_t)a * r->count;
                src_stride[nsrc++] = 8;
            }
            own_count = true;
            break;
        }
        default:
            MBC_FAIL(MBC_ERR_ARG, "mbc_shard_gather: only scan, sorted, top-k and grouped results can be gathered (not a join's pairs)");
    }
    if (nsrc != s->ncols) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_gather: result has %d columns, window %d", nsrc, s->ncols);
    for (int c = 0; c < s->ncols; ++c)
        if (src_stride[c] != s->strides[c]) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_gather: column %d stride %d, window %d", c, src_stride[c], s->strides[c]);
    mbc_ctx* ctx = s->ctx;
    MBC_CUDA(cudaSetDevice(ctx->device));
    const unsigned long long epoch = ++s->epoch;
    const int slot = (int)(epoch % kShardSlots);
    PushParams p;
    memset(&p, 0, sizeof(p));
    p.hdr = reinterpret_cast<ShardHeader*>(s->win);
    p.ctl = reinterpret_cast<ShardCtl*>(s->win + s->off_ctl) + (size_t)slot * kShardMaxWorld;
    p.rank = s->rank;
    p.world = s->world;
    p.epoch = epoch;
    p.my_aggs = own_count ? s->d_count_block : reinterpret_cast<const unsigned long long*>(r->d_aggs);
    p.cap_rows = s->cap_rows;
    p.src_pos = r->d_pos;
    p.dst_pos = reinterpret_cast<int64_t*>(s->win + s->off_pos[slot]);
    p.ncols = s->ncols;
    for (int c = 0; c < s->ncols; ++c) {
        p.src[c] = src[c];
        p.dst[c] = s->win + s->off_col[slot][c];
        p.stride[c] = s->strides[c];
    }
    p.blocks_done = s->d_blocks_done;
    // the exchange follows THIS result's kernels (its completion event), not whatever the context's stream holds by now:
    // the caller may already have queued the next step's scans
    cudaStream_t st = ctx->stream;
    if (beside_next_scan & 1) {
        if (r->ev_done) {
            MBC_CUDA(cudaStreamWaitEvent(s->side, r->ev_done, 0));
        } else {
            MBC_CUDA(cudaEventRecord(s->ev_scan, ctx->stream));
            MBC_CUDA(cudaStreamWaitEvent(s->side, s->ev_scan, 0));
        }
        st = s->side;
    }
    if (own_count) {
        unsigned long long blk[kMaxAgg + 1] = {0};
        blk[kMaxAgg] = (unsigned long long)r->count;
        MBC_CUDA(cudaStreamWaitEvent(st, s->ev_push, 0));           // the previous step's publish has read the block
        MBC_CUDA(cudaMemcpyAsync(s->d_count_block, blk, sizeof(blk), cudaMemcpyHostToDevice, st));
    }
    shard_publish_kernel<<<1, 32, 0, st>>>(p.ctl, s->rank, epoch, p.my_aggs);
    ctx->launches++;
    cudaEventRecord(s->ev_push0, st);
    if (beside_next_scan & 2) {
        // copy engines: offset on the host (one small wait), then one peer copy per buffer, then the done flag
        shard_offset_kernel<<<1, 32, 0, st>>>(p.hdr, p.ctl, s->rank, epoch, p.my_aggs, s->cap_rows, s->d_off);
        ctx->launches++;
        MBC_CUDA(cudaGetLastError());
        MBC_CUDA(cudaEventRecord(s->ev_off, st));
        MBC_CUDA(cudaEventSynchronize(s->ev_off));
        const long long off = s->h_off[0], n = s->h_off[1], dropped = s->h_off[2];
        if (n > 0) {
            if (p.src_pos) MBC_CUDA(cudaMemcpyAsync(p.dst_pos + off, p.src_pos, (size_t)n * 8, cudaMemcpyDeviceToDevice, st));
            for (int c = 0; c < s->ncols; ++c)
                MBC_CUDA(cudaMemcpyAsync((char*)p.dst[c] + (size_t)off * p.stride[c], p.src[c], (size_t)n * p.stride[c], cudaMemcpyDeviceToDevice, st));
        }
        shard_done_kernel<<<1, 32, 0, st>>>(p.ctl, s->rank, epoch, (unsigned long long)dropped);
        ctx->launches++;
        MBC_CUDA(cudaGetLastError());
    } else {
        shard_push_kernel<<<s->push_ctas, 256, 0, st>>>(p);
        ctx->launches++;
        MBC_CUDA(cudaGetLastError());
    }
    cudaEventRecord(s->ev_push1, st);
    MBC_CUDA(cudaEventRecord(s->ev_push, st));
    return MBC_OK;
}

float mbc_shard_push_ms(mbc_shard* s) {
    float ms = -1.f;
    if (!s || cudaEventSynchronize(s->ev_push1) != cudaSuccess || cudaEventElapsedTime(&ms, s->ev_push0, s->ev_push1) != cudaSuccess) return -1.f;
    return ms;
}

int32_t mbc_shard_fence(mbc_shard* s) {
    if (!s) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_fence: NULL");
    MBC_CUDA(cudaSetDevice(s->ctx->device));
    MBC_CUDA(cudaStreamWaitEvent(s->ctx->stream, s->ev_push, 0));  // later work of the stream (frees included) follows the push
    return MBC_OK;
}

int32_t mbc_shard_collect(mbc_shard* s, int64_t* total_rows, int64_t* rank_counts) {
    if (!s || !s->owned) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_collect: only the window's owner collects");
    if (s->epoch == 0) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_collect: nothing was gathered");
    s->collected = 0;
    mbc_ctx* ctx = s->ctx;
    MBC_CUDA(cudaSetDevice(ctx->device));
    const int slot = (int)(s->epoch % kShardSlots);
    const ShardCtl* ctl = reinterpret_cast<const ShardCtl*>(s->win + s->off_ctl) + (size_t)slot * kShardMaxWorld;
    // everything of the collect runs on the side stream: the context's stream may already hold the next step's scans, and
    // the host must not wait for those
    MBC_CUDA(cudaStreamWaitEvent(s->side, s->ev_push, 0));
    shard_wait_kernel<<<1, 32, 0, s->side>>>(ctl, s->world, s->epoch, s->d_summary);
    ctx->launches++;
    MBC_CUDA(cudaGetLastError());
    MBC_CUDA(cudaMemcpyAsync(s->h_summary, s->d_summary, (size_t)s->world * (kMaxAgg + 2) * 8, cudaMemcpyDeviceToHost, s->side));
    MBC_CUDA(cudaStreamSynchronize(s->side));
    s->total = s->dropped = 0;
    for (int k = 0; k < s->world; ++k) {
        s->counts[k] = (int64_t)s->h_summary[(size_t)k * (kMaxAgg + 2)];
        s->total += s->counts[k];
        s->dropped += (int64_t)s->h_summary[(size_t)k * (kMaxAgg + 2) + 1];
        if (rank_counts) rank_counts[k] = s->counts[k];
    }
    if (total_rows) *total_rows = s->total;
    if (s->dropped) MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_shard_collect: %lld rows did not fit the window of %lld rows", (long long)s->dropped, (long long)s->cap_rows);
    s->collected = s->epoch;
    return MBC_OK;
}

int32_t mbc_shard_agg(const mbc_shard* s, int32_t i, int32_t kind, int32_t type, int64_t* as_i64, double* as_f64, int32_t* valid) {
    if (!s || !s->owned || !s->h_summary || i < 0 || i >= kMaxAgg || kind < MBC_AGG_COUNT || kind > MBC_AGG_MAX)
        MBC_FAIL(MBC_ERR_ARG, "mbc_shard_agg: bad argument");
    const bool integral = kind == MBC_AGG_COUNT || type == MBC_ATTR_INTEGER;
    long long ai = 0;
    double af = 0.0;
    bool first = true;
    for (int k = 0; k < s->world; ++k) {                           // rank order = position order: a fixed association
        const unsigned long long raw = s->h_summary[(size_t)k * (kMaxAgg + 2) + 2 + i];
        const bool has = s->counts[k] > 0 || kind == MBC_AGG_COUNT || kind == MBC_AGG_SUM;
        if (!has) continue;                                        // MIN/MAX of an empty shard is the identity, not a value
        long long vi = (long long)raw;
        double vf;
        memcpy(&vf, &raw, 8);
        if (first) { ai = vi; af = vf; first = false; continue; }
        if (kind == MBC_AGG_COUNT || kind == MBC_AGG_SUM) { ai += vi; af += vf; }
        else if (kind == MBC_AGG_MIN) { ai = std::min(ai, vi); af = std::min(af, vf); }
        else { ai = std::max(ai, vi); af = std::max(af, vf); }
    }
    const bool ok = !first && (kind == MBC_AGG_COUNT || kind == MBC_AGG_SUM || s->total > 0);
    if (as_i64) *as_i64 = ok ? (integral ? ai : real_agg_as_i64(af)) : 0;
    if (as_f64) *as_f64 = ok ? (integral ? (double)ai : af) : 0.0;
    if (valid) *valid = ok ? 1 : 0;
    return MBC_OK;
}

int32_t mbc_shard_window_device(const mbc_shard* s, void** d_positions, int32_t col, void** d_column) {
    if (!s || !s->win || s->epoch == 0) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_window_device: no gathered step");
    const int slot = (int)(s->epoch % kShardSlots);
    if (d_positions) *d_positions = s->win + s->off_pos[slot];
    if (d_column) {
        if (col < 0 || col >= s->ncols) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_window_device: column %d of %d", col, s->ncols);
        *d_column = s->win + s->off_col[slot][col];
    }
    return MBC_OK;
}

int32_t mbc_shard_read(mbc_shard* s, int32_t col, int64_t first_row, int64_t nrows, void* host_out) {
    if (!s || !s->owned || s->epoch == 0 || !host_out || first_row < 0 || nrows < 0 || first_row + nrows > s->cap_rows || col < -1 || col >= s->ncols)
        MBC_FAIL(MBC_ERR_ARG, "mbc_shard_read: bad argument");
    MBC_CUDA(cudaSetDevice(s->ctx->device));
    const int slot = (int)(s->epoch % kShardSlots);
    const size_t stride = col < 0 ? 8 : (size_t)s->strides[col];
    const char* src = s->win + (col < 0 ? s->off_pos[slot] : s->off_col[slot][col]) + (size_t)first_row * stride;
    if (nrows) MBC_CUDA(cudaMemcpyAsync(host_out, src, (size_t)nrows * stride, cudaMemcpyDeviceToHost, s->side));
    MBC_CUDA(cudaStreamSynchronize(s->side));
    return MBC_OK;
}

int32_t mbc_shard_release(mbc_shard* s) {
    if (!s || !s->owned || s->epoch == 0) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_release: only the window's owner releases a gathered step");
    MBC_CUDA(cudaSetDevice(s->ctx->device));
    s->collected = 0;
    shard_release_kernel<<<1, 32, 0, s->side>>>(reinterpret_cast<ShardHeader*>(s->win), s->epoch);   // after the reads of the step
    s->ctx->launches++;
    MBC_CUDA(cudaGetLastError());
    return MBC_OK;
}

int32_t mbc_shard_topk(mbc_shard* s, const mbc_coldesc* descs, const int32_t* key_fields, int32_t nkeys, int32_t descending, int64_t k,
                       const int32_t* proj_fields, int32_t nproj, uint32_t want, mbc_result** out) {
    if (!out || !descs || !key_fields || nkeys <= 0 || nproj < 0 || (nproj > 0 && !proj_fields)) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_topk: bad argument");
    *out = nullptr;
    MBC_TRY(merge_check(s, "mbc_shard_topk"));
    if (k < 0) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_topk: k = %lld is negative", (long long)k);
    if (want & (MBC_WANT_AGG | MBC_WANT_BITMAP))
        MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_shard_topk: MBC_WANT_AGG / MBC_WANT_BITMAP are not available for a top-k");
    if (nkeys > kMaxTerms || nproj > kMaxProj) MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_shard_topk: %d key fields / %d projected fields", nkeys, nproj);
    Column cols[kMaxProj];
    for (int c = 0; c < s->ncols; ++c) MBC_TRY(window_column(s, "mbc_shard_topk", c, descs[c], &cols[c]));
    for (int q = 0; q < nkeys; ++q)
        if (key_fields[q] < 0 || key_fields[q] >= s->ncols) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_topk: key field %d of %d", key_fields[q], s->ncols);
    for (int c = 0; c < nproj; ++c)
        if (proj_fields[c] < 0 || proj_fields[c] >= s->ncols) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_topk: projected field %d of %d", proj_fields[c], s->ncols);
    mbc_ctx* ctx = s->ctx;
    MBC_CUDA(cudaSetDevice(ctx->device));
    const int64_t n = s->total, m = std::min<int64_t>(k, n);
    const int64_t* win_pos = reinterpret_cast<const int64_t*>(s->win + s->off_pos[s->epoch % kShardSlots]);
    begin_timing(ctx);
    mbc_result* r = new mbc_result();
    r->kind = mbc_result::kRows;
    r->ctx = ctx;
    ctx_retain(ctx);
    r->want = want;
    r->nrows = n;
    r->count = m;
    r->capacity = m;
    uint32_t *rows = nullptr, *keys = nullptr, *bits = nullptr;
    auto release = [&]() {
        for (void* p : {(void*)rows, (void*)keys, (void*)bits}) dev_free(ctx, p);
    };
    auto fail = [&](int32_t st) {
        release();
        cudaStreamSynchronize(ctx->stream);                           // nothing reads the window after the call returns
        mbc_result_free(r);
        return st;
    };
#define MTRY(x) do { int32_t _s = (x); if (_s != MBC_OK) return fail(_s); } while (0)
    // `rows` ends up holding the window rows in key order; the result is its first m
    if (m > 0) {
        MTRY(dev_alloc(ctx, (void**)&rows, (size_t)n * 4, false));
        MTRY(dev_alloc(ctx, (void**)&keys, (size_t)n * 4, false));
        MTRY(dev_alloc(ctx, (void**)&bits, 8, false));
        sort_iota_kernel<<<merge_grid(ctx, n), 256, 0, ctx->stream>>>(n, rows);
        ctx->launches++;
        for (int q = nkeys - 1; q >= 0; --q) MTRY(sort_rows_by_column(ctx, rows, n, cols[key_fields[q]], descending != 0, keys, bits));
    }
    if ((want & MBC_WANT_POSITIONS) && m > 0) {
        MTRY(dev_alloc(ctx, (void**)&r->d_pos, (size_t)m * 8, false));
        sort_gather_kernel<<<merge_grid(ctx, m), 256, 0, ctx->stream>>>(rows, m, win_pos, 8, r->d_pos);
        ctx->launches++;
    }
    if ((want & (MBC_WANT_COLUMNS | MBC_WANT_TUPLES)) && nproj > 0) {
        for (int c = 0; c < nproj; ++c) {
            const Column& col = cols[proj_fields[c]];
            mbc_result::Col rc{col.type, col.width, col.stride, nullptr, nullptr};
            MTRY(dev_alloc(ctx, &rc.d, (size_t)std::max<int64_t>(m, 1) * col.stride, false));
            r->cols.push_back(rc);
            if (m > 0) {
                sort_gather_kernel<<<merge_grid(ctx, m), 256, 0, ctx->stream>>>(rows, m, col.d, col.stride, rc.d);
                ctx->launches++;
            }
        }
    }
    end_timing(ctx);
    if (cudaGetLastError() != cudaSuccess) return fail((set_error("mbc_shard_topk: launch failed"), MBC_ERR_CUDA));
    MTRY(finish_result_host(r));
#undef MTRY
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return fail((set_error("mbc_shard_topk: merge failed"), MBC_ERR_CUDA));
    release();
    *out = r;
    return MBC_OK;
}

int32_t mbc_shard_group(mbc_shard* s, const mbc_coldesc* key_descs, int32_t nkeys, const int32_t* agg_kinds, const int32_t* agg_types,
                        int32_t nagg, uint32_t want, mbc_result** out) {
    if (!out || !key_descs || nkeys <= 0 || nagg < 0 || (nagg > 0 && (!agg_kinds || !agg_types)))
        MBC_FAIL(MBC_ERR_ARG, "mbc_shard_group: bad argument");
    *out = nullptr;
    MBC_TRY(merge_check(s, "mbc_shard_group"));
    if (want & (MBC_WANT_TUPLES | MBC_WANT_BITMAP))
        MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_shard_group: MBC_WANT_TUPLES / MBC_WANT_BITMAP are not available for groups");
    if (nkeys + nagg > kMaxProj || nagg > kMaxAgg)
        MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_shard_group: %d key columns + %d aggregates (max %d columns, %d aggregates)", nkeys, nagg, kMaxProj, kMaxAgg);
    if (s->ncols != nkeys + nagg)
        MBC_FAIL(MBC_ERR_ARG, "mbc_shard_group: %d key columns + %d aggregates for a window of %d columns", nkeys, nagg, s->ncols);
    Column keys[kMaxProj];
    for (int c = 0; c < nkeys; ++c) MBC_TRY(window_column(s, "mbc_shard_group", c, key_descs[c], &keys[c]));
    const int slot = (int)(s->epoch % kShardSlots);
    GroupAggSpec specs[kMaxAgg] = {};
    for (int a = 0; a < nagg; ++a) {
        const int kind = agg_kinds[a], type = agg_types[a];
        if (kind < MBC_AGG_COUNT || kind > MBC_AGG_MAX) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_group: aggregate %d: unknown kind %d", a, kind);
        if (kind != MBC_AGG_COUNT && type == MBC_ATTR_STRING) MBC_FAIL(MBC_ERR_UNSUPPORTED, "mbc_shard_group: aggregate %d over a string column", a);
        if (kind != MBC_AGG_COUNT && type != MBC_ATTR_INTEGER && type != MBC_ATTR_REAL)
            MBC_FAIL(MBC_ERR_ARG, "mbc_shard_group: aggregate %d: column type %d", a, type);
        if (s->strides[nkeys + a] != 8) MBC_FAIL(MBC_ERR_ARG, "mbc_shard_group: window column %d (aggregate %d) has stride %d, not 8", nkeys + a, a, s->strides[nkeys + a]);
        specs[a].kind = kind;
        specs[a].type = kind == MBC_AGG_COUNT ? MBC_ATTR_INTEGER : type;
        specs[a].src = s->win + s->off_col[slot][nkeys + a];
    }
    mbc_ctx* ctx = s->ctx;
    MBC_CUDA(cudaSetDevice(ctx->device));
    const int64_t n = s->total;
    begin_timing(ctx);
    mbc_result* r = new mbc_result();
    r->ctx = ctx;
    ctx_retain(ctx);
    r->want = want;
    r->nrows = n;
    uint32_t* rows = nullptr;
    int32_t st = dev_alloc(ctx, (void**)&rows, (size_t)std::max<int64_t>(n, 1) * 4, false);
    if (st == MBC_OK && n > 0) {
        sort_iota_kernel<<<merge_grid(ctx, n), 256, 0, ctx->stream>>>(n, rows);
        ctx->launches++;
    }
    // the partials of one group keep rank order through the stable sort, so the fold's association is fixed
    if (st == MBC_OK)
        st = group_rows(ctx, rows, n, keys, nkeys, specs, nagg, true, reinterpret_cast<const int64_t*>(s->win + s->off_pos[slot]), 0, r);
    dev_free(ctx, rows);
    if (st != MBC_OK) {
        cudaStreamSynchronize(ctx->stream);                           // nothing reads the window after the call returns
        mbc_result_free(r);
        return st;
    }
    *out = r;
    return MBC_OK;
}

int32_t mbc_init_devices(int32_t n_devices, const int32_t* device_ids, mbc_ctx** out) {
    if (n_devices <= 0 || !device_ids || !out) MBC_FAIL(MBC_ERR_ARG, "mbc_init_devices: bad argument");
    for (int i = 0; i < n_devices; ++i) out[i] = nullptr;
    for (int i = 0; i < n_devices; ++i) {
        const int32_t s = mbc_init(device_ids[i], &out[i]);
        if (s != MBC_OK) {
            for (int k = 0; k < i; ++k) { mbc_shutdown(out[k]); out[k] = nullptr; }
            return s;
        }
    }
    return MBC_OK;
}

}  // extern "C"
