/*
 * mbcol.h -- C ABI of libmbcol.so: the B200-native (sm_100a) columnar scan hot path
 * that sits under MiniBase-Columnar-Database's Java operator surface.
 *
 * The reference has no FFI seam of its own (it is 100% Java); the seam is the Java class
 * surface.  Every entry point below names the reference method(s) whose work it replaces
 * (paths relative to /root/reference/minijava/src).  The Java-side binding a maintainer
 * would add (Panama FFM / JNI) is shown in INTEGRATION.md.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  No torch / C++ types.
 *   - every function returns int32 status: 0 = MBC_OK, <0 = error; mbc_last_error() returns
 *     a thread-local message (the Java shim rethrows it as FileScanException/IndexException,
 *     iterator/ColumnarFileScan.java:80-98, index/ColumnIndexScan.java:107-112).
 *   - there is NO CPU fallback: mbc_init fails when no sm_100 device is present.
 *   - field numbers on the Java surface are 1-based; everything here is 0-based.
 *   - one caller thread per handle (the reference is single threaded).
 *   - host scalars are native little-endian; only mbc_result_tuples() emits the reference's
 *     big-endian Tuple wire format (heap/Tuple.java:369-440, global/Convert.java:163-275).
 */
#ifndef MBCOL_H
#define MBCOL_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MBC_ABI_VERSION 1

/* ---- status codes ---------------------------------------------------------------- */
#define MBC_OK              0
#define MBC_ERR_ARG        -1   /* bad argument (maps to the reference's checked exceptions)  */
#define MBC_ERR_CUDA       -2   /* CUDA runtime failure                                       */
#define MBC_ERR_NODEVICE   -3   /* no sm_100 device: the product path has no CPU fallback     */
#define MBC_ERR_UNSUPPORTED -4  /* outside the stated contract (e.g. string literal too wide) */
#define MBC_ERR_FORMAT     -5   /* malformed reference DB file                                */
#define MBC_ERR_NOINDEX    -6   /* bitmap index missing on a column a bitmap scan needs       */

/* ---- global/AttrType.java:10-14 --------------------------------------------------- */
#define MBC_ATTR_STRING   0
#define MBC_ATTR_INTEGER  1
#define MBC_ATTR_REAL     2
#define MBC_ATTR_SYMBOL   3

/* ---- global/AttrOperator.java:10-18 ------------------------------------------------ */
#define MBC_OP_EQ    0
#define MBC_OP_LT    1
#define MBC_OP_GT    2
#define MBC_OP_NE    3
#define MBC_OP_LE    4
#define MBC_OP_GE    5
#define MBC_OP_NOT   6   /* PredEval treats it as NE (iterator/PredEval.java:158-160)         */
#define MBC_OP_NOP   7   /* never true (PredEval.java:137-162 default branch)                  */
#define MBC_OP_RANGE 8   /* never true                                                         */

/* operand kinds of one CondExpr term (iterator/CondExpr.java:12-57, Operand.java:5-10) */
#define MBC_OPERAND_LITERAL 0
#define MBC_OPERAND_OUTER   1   /* RelSpec.outer    -> t1 (iterator/PredEval.java:79-91)      */
#define MBC_OPERAND_INNER   2   /* RelSpec.innerRel -> t2 (joins only)                         */

/* what a scan should materialise */
#define MBC_WANT_POSITIONS 0x01u  /* ascending positions (TID.position, global/TID.java:8-29)  */
#define MBC_WANT_COLUMNS   0x02u  /* projected values, one dense array per projected column    */
#define MBC_WANT_TUPLES    0x04u  /* projected tuples in the reference Tuple byte layout       */
#define MBC_WANT_AGG       0x08u  /* COUNT/SUM/MIN/MAX over the qualifying set                 */
#define MBC_WANT_BITMAP    0x10u  /* the qualifying set as a java.util.BitSet-compatible bitmap*/
#define MBC_WANT_HOST      0x20u  /* copy what was asked for to pinned host memory             */

/* aggregate kinds (absent from the reference; defined in SURVEY.md 8c and oracle/) */
#define MBC_AGG_COUNT 0
#define MBC_AGG_SUM   1
#define MBC_AGG_MIN   2
#define MBC_AGG_MAX   3

typedef struct mbc_ctx    mbc_ctx;
typedef struct mbc_table  mbc_table;
typedef struct mbc_result mbc_result;

/* One column of a Columnarfile (columnar/Columnarfile.java:257-323: types, sizes). */
typedef struct {
    int32_t type;    /* MBC_ATTR_*                                                       */
    int32_t width;   /* payload bytes: 4 for int/real, strSize for char(strSize)          */
} mbc_coldesc;

/* One side of a comparison (iterator/Operand.java:5-10). */
typedef struct {
    int32_t kind;           /* MBC_OPERAND_*                                              */
    int32_t type;           /* literal: MBC_ATTR_INTEGER/REAL/STRING; column: MBC_ATTR_SYMBOL */
    int32_t col;            /* 0-based column (symbol.offset-1) when kind != LITERAL      */
    int32_t lit_i;          /* integer literal                                            */
    float   lit_f;          /* real literal                                               */
    int32_t lit_slen;       /* string literal length in bytes                             */
    const uint8_t* lit_s;   /* string literal bytes (modified UTF-8, no terminator)       */
} mbc_operand;

/* One CondExpr of the CNF.  Terms with equal conj_id are ORed (the .next chain,
 * iterator/PredEval.java:54,164-167); conjunct groups are ANDed (the CondExpr[] array,
 * PredEval.java:51,171-176).  Terms must be sorted by conj_id.  nterms == 0 means
 * "p == null" -> every row qualifies (PredEval.java:46-49). */
typedef struct {
    int32_t     op;         /* MBC_OP_*                                                   */
    int32_t     conj_id;
    mbc_operand lhs;        /* comparison type = type of the lhs (PredEval.java:64-89)    */
    mbc_operand rhs;
} mbc_term;

typedef struct {
    int32_t kind;           /* MBC_AGG_*                                                  */
    int32_t col;            /* 0-based column; ignored for COUNT                          */
} mbc_aggspec;

/* A projected output field of a join (iterator/Projection.java:28-83). */
typedef struct {
    int32_t rel;            /* MBC_OPERAND_OUTER or MBC_OPERAND_INNER                     */
    int32_t col;            /* 0-based column of that relation                            */
} mbc_projspec;

/* ---- context ----------------------------------------------------------------------- */
/* One context = one GPU.  Multi-GPU runs shard rows by position range, one context per GPU (in one process or in
 * one process per GPU), and gather their results through the mbc_shard_* calls below.  Replaces the role of
 * global/SystemDefs.java:7-96 (buffer pool + DB singletons): device HBM is the pool. */
int32_t mbc_init(int32_t device_id, mbc_ctx** out);
/* SURVEY.md 8(b)'s mbc_init(n_devices, ids): one context per listed device, all or nothing. */
int32_t mbc_init_devices(int32_t n_devices, const int32_t* device_ids, mbc_ctx** out /* [n_devices] */);
void    mbc_shutdown(mbc_ctx* ctx);
/* Run every later launch of this context on `cuda_stream` (a cudaStream_t; NULL = the
 * context's own stream) so callers can time with events on their stream. */
int32_t mbc_set_stream(mbc_ctx* ctx, void* cuda_stream);
int32_t mbc_sync(mbc_ctx* ctx);
const char* mbc_last_error(void);
int32_t mbc_abi_version(void);
/* Pinned host memory for staging (what a Panama MemorySegment / direct ByteBuffer would wrap). */
int32_t mbc_host_alloc(void** p, int64_t bytes);
void    mbc_host_free(void* p);
/* Number of this library's kernels launched by the context since creation. */
int64_t mbc_kernel_launches(const mbc_ctx* ctx);
/* Bytes mbc_scan_host has moved host -> device since the context was created: explicit copies plus the
 * survivors' rows it read in place from pinned host columns (late materialisation). */
int64_t mbc_h2d_bytes(const mbc_ctx* ctx);
/* Device-time of the last scan/bitmap/join call's kernels, CUDA events on the ctx stream. */
float   mbc_last_kernel_ms(const mbc_ctx* ctx);

/* ---- tables (columnar/Columnarfile.java:239-359 open; the read side only) ---------- */
/* position_base: global position of local row 0 (TID-range sharding; positions are
 * int64 = position_base + local row, SURVEY.md 8c). */
int32_t mbc_table_create(mbc_ctx* ctx, int32_t ncols, const mbc_coldesc* cols,
                         int64_t nrows, int64_t position_base, mbc_table** out);
void    mbc_table_free(mbc_table* t);
int64_t mbc_table_nrows(const mbc_table* t);
int32_t mbc_table_ncols(const mbc_table* t);
int32_t mbc_table_coldesc(const mbc_table* t, int32_t col, mbc_coldesc* out);
/* Already-columnar path: host array of nrows packed values (int32 / float32 little-endian,
 * or nrows*width bytes of zero-padded strings without the 2-byte length prefix). */
int32_t mbc_table_load_column(mbc_table* t, int32_t col, const void* host_packed, int64_t nrows);
/* Read one column back (tests / K1 parity). out must hold nrows*width bytes. */
int32_t mbc_table_read_column(mbc_table* t, int32_t col, void* host_out, int64_t nrows);
/* Device pointer + row stride of a resident column (for NCCL / zero-copy callers). */
int32_t mbc_table_column_device(mbc_table* t, int32_t col, void** dev_ptr, int32_t* stride_bytes);
/* Fill a column with the stateless counter-RNG synthetic data of SURVEY.md 8d
 * (kind 0: int uniform [0,domain); 1: real uniform [0,1000); 2: printable char(width);
 *  3: int (position*2654435761+12345) mod domain, a permutation of [0,domain) when nrows == domain).
 * Rows are keyed by global position, so any shard reproduces the same table. */
int32_t mbc_table_generate(mbc_table* t, int32_t col, int32_t kind, uint64_t seed, int64_t domain);
/* K1: decode a reference-format DB file image (diskmgr/DB.java:866-871,998-1000 directory;
 * heap/HFPage.java:31-40 pages; heap/Heapfile.java:262-289 position arithmetic;
 * columnar/Columnarfile.java:257-323 .hdr schema) into a device-resident table.
 * Replaces heap/Scan.java:84-114 + global/Convert.java:18-126 + columnar/TupleScan.java:55-89. */
int32_t mbc_table_ingest_dbfile(mbc_ctx* ctx, const uint8_t* db_bytes, int64_t db_len,
                                const char* cf_name, mbc_table** out);
/* columnar/Columnarfile.java:1138 getMarkedDeleted(): bit p set = position p deleted.
 * Words are java.util.BitSet.toLongArray() order (bit p -> word p/64, bit p%64). */
int32_t mbc_table_set_deleted(mbc_table* t, const uint64_t* bitset_words, int64_t nwords);

/* ---- K2: fused CNF filter -> ordered compaction -> projection -> aggregates ---------- */
/* Replaces iterator/ColumnarFileScan.java:156-188 (get_next/get_next_tid loop) +
 * iterator/PredEval.java:25-183 + iterator/Projection.java:103-144 for the whole table at once. */
int32_t mbc_scan(mbc_table* t, const mbc_term* terms, int32_t nterms,
                 const int32_t* proj_cols, int32_t nproj, uint32_t want,
                 const mbc_aggspec* aggs, int32_t nagg, mbc_result** out);
/* Same scan over host-resident columns: rows are streamed to the GPU in chunks (H2D on a copy
 * stream overlapped with the scan of the previous chunk) and the result is copied back.
 * host_cols[c] follows the mbc_table_load_column layout.  This is the end-to-end path.
 * Late materialisation: a column that is only projected / aggregated (never compared) whose buffer is pinned
 * host memory (mbc_host_alloc, cudaHostAlloc, cudaHostRegister), 16-byte aligned and laid out like the device
 * column is not uploaded when a first 256 Ki-row sample shows that at most 1/5 of the rows qualify: the write
 * pass then reads the survivors' values in place over PCIe.  Results are identical either way; pageable buffers
 * always take the upload path.  mbc_h2d_bytes() counts what crossed. */
int32_t mbc_scan_host(mbc_ctx* ctx, int32_t ncols, const mbc_coldesc* cols, const void* const* host_cols,
                      int64_t nrows, int64_t position_base,
                      const mbc_term* terms, int32_t nterms, const int32_t* proj_cols, int32_t nproj,
                      uint32_t want, const mbc_aggspec* aggs, int32_t nagg, mbc_result** out);

/* ---- K3: bitmap index build (columnar/Columnarfile.java:698-753) -------------------- */
int32_t mbc_bitmap_build(mbc_table* t, int32_t col);
int32_t mbc_bitmap_exists(const mbc_table* t, int32_t col);                 /* Columnarfile.java:1027 */
/* Columnarfile.java:1096 getBitmapValues(): distinct indexed values, ascending.
 * ints: n int32; strings: n*width bytes. *values stays owned by the table. */
int32_t mbc_bitmap_values(mbc_table* t, int32_t col, const void** values, int64_t* n);
/* Columnarfile.java:1103-1127 getBitmapIndex(col,value).getBitSet(): copies the value's bitmap
 * into out_words (BitSet.toLongArray() order); all-zero when the value was never indexed. */
int32_t mbc_bitmap_get(mbc_table* t, int32_t col, const void* value, uint64_t* out_words, int64_t nwords);
/* Physical layout of a column's bitmap index, chosen by mbc_bitmap_build; every call above returns the same either way.
 *   DENSE : one uncompressed bitset per distinct value, D * N/8 bytes of HBM.
 *   SPARSE: the indexed row ids sorted by value (4 bytes per row) plus the N/8-byte bitmap of the rows the index
 *           covers; taken when the column has more than 2^19 distinct values or its bitsets do not fit the device.
 * Returns the MBC_BITMAP_* layout (NONE when the column has no index) and, when device_bytes is not NULL, the
 * index's HBM bytes; < 0 on a bad argument. */
#define MBC_BITMAP_NONE   0
#define MBC_BITMAP_DENSE  1
#define MBC_BITMAP_SPARSE 2
int32_t mbc_bitmap_layout(const mbc_table* t, int32_t col, int64_t* device_bytes);

/* ---- K4 (+K5): bitmap CNF scan ------------------------------------------------------- */
/* Replaces index/ColumnarIndexScan.java:79-182,185-268 (CNF over per-term bitsets),
 * index/ColumnIndexScan.java:656-740 (term -> OR of the bitmaps of satisfying values),
 * :600-624 (skip markedDeleted) and :287-308 (gather of projected columns).
 * Every term must be `column op literal`; every referenced column needs a bitmap index. */
int32_t mbc_bitmap_scan(mbc_table* t, const mbc_term* terms, int32_t nterms,
                        const int32_t* proj_cols, int32_t nproj, uint32_t want,
                        const mbc_aggspec* aggs, int32_t nagg, mbc_result** out);

/* ---- K6: bitmap equi-join (input/BitMapQuery.java:187-305) --------------------------- */
/* outer_sel/inner_sel: results holding MBC_WANT_BITMAP of the side filters
 * (BitMapQuery.getConstraintBitset :322-345), or NULL for "all rows".
 * join terms: lhs = outer column, rhs = inner column, op as written by the user (the
 * reference reverses it internally, :453).  Pairs are ordered outer position ascending,
 * then inner position ascending (:227,269).  Aggregate specs address the projected field
 * list (col = index into proj). */
int32_t mbc_bitmap_join(mbc_table* outer, mbc_table* inner,
                        const mbc_result* outer_sel, const mbc_result* inner_sel,
                        const mbc_term* join_terms, int32_t njoin,
                        const mbc_projspec* proj, int32_t nproj, uint32_t want,
                        const mbc_aggspec* aggs, int32_t nagg, mbc_result** out);

/* ---- sort (input/ColumnarSort.java:73-400: `sort DB CF [sort columns] [projection] ASC|DSC ...`) --------------
 * Rows ordered by the key columns, first key most significant: ints numerically, strings in byte order
 * (= String.compareTo for BMP text, the comparator of ColumnarSort.java:163-205), reals numerically; `descending`
 * reverses all keys at once.  Equal keys come out in ascending position (the reference's external merge leaves the
 * order of ties unspecified).  Deleted rows are skipped.  The result carries the positions in sorted order
 * (MBC_WANT_POSITIONS) and the projected columns / Tuple bytes of those rows (MBC_WANT_COLUMNS / MBC_WANT_TUPLES). */
int32_t mbc_sort(mbc_table* t, const int32_t* key_cols, int32_t nkeys, int32_t descending,
                 const int32_t* proj_cols, int32_t nproj, uint32_t want, mbc_result** out);

/* ---- sharding: TID-range shards on the GPUs of one node (SURVEY.md 8e) ----------------------------------------
 * The reference has no partitioning (it is one Java thread); this is what running its ColumnarFileScan
 * (iterator/ColumnarFileScan.java:156-188) over a table whose position ranges live on several GPUs needs: every rank
 * scans its slice (mbc_scan on a table created with position_base = first position of the slice), then the ranks'
 * results are concatenated in rank (= position) order in a WINDOW in the root rank's HBM, and COUNT/SUM/MIN/MAX are
 * folded.  The rows cross NVLink once, as peer-memory stores from a kernel of this library; there is no NCCL call.
 *
 *   every rank:  mbc_shard_create(ctx, rank, world, &sh)
 *   root:        mbc_shard_window_create(sh, capacity_rows, ncols, strides, handle)      allocates + exports the window
 *   peers:       mbc_shard_window_open(sh, handle, ...)      another process: the host ships the 64 handle bytes
 *            or  mbc_shard_window_attach(sh, root_sh)        same process (one JVM, several GPUs): peer access
 *   per step, every rank (root included), after its mbc_scan:
 *                mbc_shard_gather(sh, result, beside_next_scan)   asynchronous; then mbc_shard_fence(sh) before the
 *                                                                 result is freed when beside_next_scan != 0
 *   root:        mbc_shard_collect(sh, &total, counts)       waits for every rank's rows; mbc_shard_agg folds aggregates;
 *                mbc_shard_read / mbc_shard_window_device     the gathered rows;   mbc_shard_release(sh) ends the step.
 * Every rank must call mbc_shard_gather exactly once per step (the calls are matched by a step counter), with results
 * of the same projection; the root must release a step before the ranks can gather the step after the next one. */
typedef struct mbc_shard mbc_shard;
#define MBC_IPC_HANDLE_BYTES 64
int32_t mbc_shard_create(mbc_ctx* ctx, int32_t rank, int32_t world, mbc_shard** out);
void    mbc_shard_free(mbc_shard* sh);
/* col_strides: device row stride of every projected column (mbc_result_column_device). handle_out: 64 bytes or NULL. */
int32_t mbc_shard_window_create(mbc_shard* sh, int64_t capacity_rows, int32_t ncols, const int32_t* col_strides,
                                uint8_t* handle_out);
int32_t mbc_shard_window_open(mbc_shard* sh, const uint8_t* handle, int64_t capacity_rows, int32_t ncols,
                              const int32_t* col_strides);
int32_t mbc_shard_window_attach(mbc_shard* sh, const mbc_shard* root);
/* Push this rank's positions, projected columns, count and aggregates of `r` into the window.  `mode` bit 0: the push
 * runs on a side stream behind r's kernels, so scans queued afterwards overlap it.  Bit 1: the rows travel as peer copies on
 * the copy engines (no SM; the call then waits until r's kernels have finished, to learn the rank's offset) instead of
 * peer-memory stores from a kernel. */
#define MBC_GATHER_BESIDE_NEXT_SCAN 1
#define MBC_GATHER_COPY_ENGINES     2
int32_t mbc_shard_gather(mbc_shard* sh, const mbc_result* r, int32_t mode);
int32_t mbc_shard_fence(mbc_shard* sh);
/* device time of this rank's last push kernel (waits for it), ms; < 0 if none */
float   mbc_shard_push_ms(mbc_shard* sh);
int32_t mbc_shard_collect(mbc_shard* root, int64_t* total_rows, int64_t* rank_counts /* [world] or NULL */);
/* aggregate i of the gathered results folded over the ranks; kind / type as in the scan's mbc_aggspec / column type */
int32_t mbc_shard_agg(const mbc_shard* root, int32_t i, int32_t kind, int32_t type, int64_t* as_i64, double* as_f64,
                      int32_t* valid);
/* device pointers of the last gathered step (root: its own memory; peers: the mapped window) */
int32_t mbc_shard_window_device(const mbc_shard* sh, void** d_positions, int32_t col, void** d_column);
/* copy rows [first_row, first_row + nrows) of the gathered positions (col = -1, int64) or of column `col` to the host */
int32_t mbc_shard_read(mbc_shard* root, int32_t col, int64_t first_row, int64_t nrows, void* host_out);
int32_t mbc_shard_release(mbc_shard* root);

/* ---- results -------------------------------------------------------------------------- */
/* A device-resident result of mbc_scan (no MBC_WANT_HOST / MBC_WANT_TUPLES) completes asynchronously:
 * mbc_scan returns with its kernels queued on the context's stream, and the first call of
 * mbc_result_count / mbc_result_agg / mbc_result_kernel_ms waits for them.  The device buffers of
 * mbc_result_device are valid in stream order at once. */
int64_t        mbc_result_count(const mbc_result* r);
/* Device time of the kernels that produced this result (CUDA events around them), ms; < 0 if unknown. */
float          mbc_result_kernel_ms(const mbc_result* r);
/* The same per kernel for a scan over a resident table: ms4 = {pass 1 (filter_kernel / select_bitmap_kernel),
 * tile_offsets_kernel, write pass (write_kernel + write_staged_kernel), agg_finish_kernel}; -1 where unknown.  The three
 * extra events between the launches are recorded only when the environment has MBC_PHASE_EVENTS set (profiling). */
int32_t        mbc_result_phase_ms(const mbc_result* r, float* ms4);
/* ascending positions, int64 (host; needs MBC_WANT_POSITIONS|MBC_WANT_HOST). For joins:
 * outer positions; mbc_result_positions2 gives the matching inner positions. */
const int64_t* mbc_result_positions(const mbc_result* r);
const int64_t* mbc_result_positions2(const mbc_result* r);
/* projected field i as a dense host array (int32/float32 LE, or count*width string bytes) */
const void*    mbc_result_column(const mbc_result* r, int32_t i, int32_t* width);
/* reference Tuple byte layout, big-endian: [fldCnt:2][fldOffset[0..n]:2 each][fields],
 * strings as [len:2][modified UTF-8][zero pad] (heap/Tuple.java:369-440). */
const uint8_t* mbc_result_tuples(const mbc_result* r, int32_t* tuple_len);
/* aggregate i: valid=0 for MIN/MAX over an empty set. Integer aggregates are exact in as_i64;
 * real SUM is a double sum, MIN/MAX of reals are exact floats widened to double. */
int32_t        mbc_result_agg(const mbc_result* r, int32_t i, int64_t* as_i64, double* as_f64, int32_t* valid);
/* qualifying set as BitSet.toLongArray() words (needs MBC_WANT_BITMAP|MBC_WANT_HOST) */
const uint64_t* mbc_result_bitmap(const mbc_result* r, int64_t* nwords);
/* device-resident views (always available for what was asked): for NCCL gathers */
int32_t        mbc_result_device(const mbc_result* r, void** d_positions, void** d_positions2,
                                 void** d_bitmap, void** d_aggs);
int32_t        mbc_result_column_device(const mbc_result* r, int32_t i, void** d_ptr, int32_t* stride_bytes);
void           mbc_result_free(mbc_result* r);

#ifdef __cplusplus
}
#endif
#endif /* MBCOL_H */
