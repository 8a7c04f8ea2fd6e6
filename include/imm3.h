/*
 * imm3.h — C ABI of the B200-native scan / filter / project path of immutable3.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference has no FFI of its own: the seam
 * is the Scala operator family.  Every entry point below cites the reference interface it
 * replaces (paths relative to the reference checkout).  A JVM shim (JNI or Panama, see
 * INTEGRATION.md) binds exactly these symbols; the Python tests and bench.py bind the same
 * symbols through ctypes.  Plain pointers and sizes only — no C++ or torch types.
 *
 * Threading: one thread at a time per imm3_db (the reference is not safe for concurrent
 * queries either — SegmentManager.scala:101-106 shares ByteBuffer positions).  The library
 * sets the CUDA device explicitly on every call and never relies on caller thread state.
 *
 * Errors: every entry point returns 0 on success or a negative imm3_status; the message is
 * available from imm3_last_error() (thread-local).  Validation happens before any launch, so a
 * shim can map a non-zero status to Left(Throwable) (Engine.scala:193-196) and never hangs
 * (the reference hangs on worker failure — Engine.scala:182-188).
 *
 * There is no CPU fallback: if no CUDA device is usable, imm3_open fails with IMM3_ERR_CUDA
 * unless IMM3_OPEN_HOST_ONLY is requested (metadata/plan inspection only; queries refuse).
 */
#ifndef IMM3_H
#define IMM3_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IMM3_ABI_VERSION 1

typedef struct imm3_db imm3_db;         /* replaces `new SegmentManager(dataDir)`      */
typedef struct imm3_result imm3_result; /* replaces the Iterator[Row] of Engine.execute */
typedef struct imm3_writer imm3_writer; /* replaces SegmentWriter + LoaderCli roll logic */

typedef enum imm3_status {
    IMM3_OK = 0,
    IMM3_ERR_NOT_FOUND = -1,   /* unknown table / column (Table.scala:13, SegmentManager.scala:92) */
    IMM3_ERR_UNSUPPORTED = -2, /* predicate not defined for the column type (Select.scala:41,80,118,156),
                                  NotMatch/NoOp (Select.scala:22), or a documented library limit */
    IMM3_ERR_BAD_FORMAT = -3,  /* malformed _table.meta / .meta / segment bytes */
    IMM3_ERR_CUDA = -4,
    IMM3_ERR_OOM = -5,
    IMM3_ERR_INVALID_ARG = -6,
    IMM3_ERR_IO = -7,
    IMM3_ERR_STATE = -8,       /* call sequence error (e.g. fetch before begin, close with open results) */
    IMM3_ERR_COMM = -9         /* count exchange between the GPUs failed (peer mailbox unmappable, a peer's count late) */
} imm3_status;

/* ColumnType enumeration, Column.scala:13-16 */
typedef enum imm3_column_type {
    IMM3_COL_INT = 0, IMM3_COL_TINYINT = 1, IMM3_COL_STRING = 2,
    IMM3_COL_COUNT = 3,   /* aggregate results only: int64 (CountAggr, ProjectAggregate.scala:21-35)                 */
    IMM3_COL_DOUBLE = 4,  /* aggregate results only: IEEE double (Min/MaxDoubleAggr, ProjectAggregate.scala:37-59)    */
    IMM3_COL_INT64 = 5    /* aggregate results only: int64, an exact SUM (imm3_query_agg_ext)                          */
} imm3_column_type;

/* CodecType enumeration (same order), Codec.scala:20-23 */
typedef enum imm3_codec {
    IMM3_CODEC_PFOR_INT = 0,
    IMM3_CODEC_DENSE_INT = 1,
    IMM3_CODEC_DENSE_TINYINT = 2,
    IMM3_CODEC_DENSE_STRING = 3
} imm3_codec;

/* SelectCondition, Query.scala:3-9.  NotMatch / NoOp exist in the ADT but SelectOp.iterator
 * throws on them (Select.scala:22); they are accepted here only to return IMM3_ERR_UNSUPPORTED. */
typedef enum imm3_op {
    IMM3_OP_GT = 1,      /* GT(gt: Double)  Select.scala:53-89  */
    IMM3_OP_LT = 2,      /* LT(lt: Double)  Select.scala:91-127 */
    IMM3_OP_EQ = 3,      /* EQ(eq: Double)  Select.scala:129-165 */
    IMM3_OP_MATCH = 4,   /* Match(values)   Select.scala:25-51  */
    IMM3_OP_NOTMATCH = 5,
    IMM3_OP_NOOP = 6
} imm3_op;

/* One Select(col, cond) leaf (Query.scala:14).  The caller flattens the And/Or tree left to
 * right exactly as PipelineThread.runOps does (Engine.scala:237-245): the AND/OR tag is dropped
 * there, so the list is always evaluated as a conjunction (SURVEY.md §3.4-7). */
typedef struct imm3_pred {
    const char* col;
    int32_t op;               /* imm3_op */
    double num;               /* GT / LT / EQ constant, narrowed inside with JVM d2i / i2b rules */
    const char* const* strs;  /* MATCH literals (NUL-terminated) */
    int32_t nstrs;
} imm3_pred;

#define IMM3_OPEN_HOST_ONLY 0x1u  /* parse + validate + lay out, no device work (CPU tests)   */
#define IMM3_OPEN_KEEP_HOST 0x2u  /* keep a pinned host mirror so imm3_reupload can re-stage  */
#define IMM3_OPEN_NO_TMA    0x4u  /* force the direct-load variant of the dense kernel (A/B)  */
#define IMM3_OPEN_FORCE_BLOCKS 0x8u /* run every query through the block-mode kernel (cross-check) */
#define IMM3_OPEN_NO_STATS  0x10u /* do not compute per-block min/max of the encoded INT columns (no block pruning) */

typedef struct imm3_open_opts {
    int32_t device;  /* CUDA ordinal */
    int32_t rank;    /* this process's shard: canonical segment slice [rank*n/world, (rank+1)*n/world) */
    int32_t world;   /* 1 = whole table */
    uint32_t flags;
} imm3_open_opts;

typedef struct imm3_table_desc {
    int32_t ncols;
    int32_t block_size;        /* Table.blockSize (Table.scala:9)                            */
    int32_t nsegments;         /* SegmentManager.getTableSegmentCount (SegmentManager.scala:94-99), whole table */
    int32_t seg_begin;         /* canonical slice owned by this handle                        */
    int32_t seg_end;
    int64_t nrows;             /* rows in the owned slice                                     */
    int64_t nblocks;           /* reference blocks (= batches) in the owned slice             */
    int64_t resident_bytes;    /* encoded bytes held in HBM for the slice                     */
} imm3_table_desc;

typedef struct imm3_column_desc {
    char name[64];
    int32_t column_type;  /* imm3_column_type */
    int32_t codec;        /* imm3_codec */
    int32_t width;        /* decoded value width in bytes: 4, 1 or dtypeAttrs("size") (Column.scala:60) */
    int32_t reserved;
    int64_t encoded_bytes; /* file bytes of the owned slice */
} imm3_column_desc;

/* ---- SegmentManager path: SegmentManager.scala:20-112, Segment.scala:33-58,154-181 ---------- */
int imm3_open(const char* data_dir, const imm3_open_opts* opts, imm3_db** out);
int imm3_close(imm3_db* db);
int imm3_table_count(imm3_db* db);                                   /* SegmentManager.tables            */
const char* imm3_table_name(imm3_db* db, int idx);
int imm3_table_info(imm3_db* db, const char* table, imm3_table_desc* out);   /* getTable / getTableSegmentCount */
int imm3_column_info(imm3_db* db, const char* table, int col_idx, imm3_column_desc* out); /* Table.columns */
/* Canonical (file-name-sorted, SegmentManager.scala:41) position -> numeric id in `col_<id>.dat`. */
int imm3_segment_file_id(imm3_db* db, const char* table, int canonical_idx, int32_t* out_id);
/* Re-stage the named columns (NULL/0 = all) of a table from the pinned host mirror into HBM.
 * Needs IMM3_OPEN_KEEP_HOST.  Asynchronous on the db stream; the next query is ordered after it. */
int imm3_reupload(imm3_db* db, const char* table, const char* const* cols, int ncols, int64_t* out_bytes);
/* Use an externally owned cudaStream_t (e.g. torch's) for everything the db launches; NULL restores its own. */
int imm3_set_stream(imm3_db* db, void* cuda_stream);
int imm3_sync(imm3_db* db);

/* ---- Scan -> Select* -> Project(limit): Engine.execute Project branch, Engine.scala:158-198 ---
 * imm3_query = begin + (count exchange is a no-op) + fetch of all rows this handle may emit.
 * Rows come back column-major, in canonical order (segment list order, block, position;
 * SURVEY.md §3.4-8), limit <= 0 meaning unlimited (Project.scala:73-77). */
int imm3_query(imm3_db* db, const char* table, const imm3_pred* preds, int npreds,
               const char* const* proj_cols, int nproj, int64_t limit, imm3_result** out);

/* Two-phase form for segment-sharded execution (one handle per GPU): begin launches the fused
 * kernels and returns once the local match count (capped at `limit`) is known; the host
 * exchanges counts (NCCL all-gather), decides how many leading local rows survive the global
 * LIMIT cut, and fetch copies exactly those rows to host memory. */
int imm3_query_begin(imm3_db* db, const char* table, const imm3_pred* preds, int npreds,
                     const char* const* proj_cols, int nproj, int64_t limit, imm3_result** out);
int64_t imm3_result_local_count(const imm3_result* r);

/* ---- Real OR (SURVEY.md 8f-4; an EXTENSION: not the reference's behaviour) ----
 * The reference parses `a or b` into Or(a, b) (Query.scala:13) and then drops the tag: PipelineThread.runOps applies every
 * leaf as a conjunction (Engine.scala:236-245), so imm3_query / imm3_query_begin evaluate Or exactly like And - that is
 * what parity with the reference means, and what the Scala engine's callers get today.  This entry point is the
 * disjunction the query language promises, for the maintainer who fixes that: the select tree in disjunctive normal
 * form, `nterms` conjunctions laid out back to back in `preds`, term i holding term_sizes[i] predicates
 * (sum = length of preds; a term of size 0 is `true`).  A row survives if it satisfies EVERY predicate of AT LEAST ONE
 * term.  Rows, order, LIMIT and the sharded count exchange are those of imm3_query_begin.  Each term runs the filter
 * kernel once and ORs its rows into the selection bitmap, so every predicate has to sit on a dense column
 * (IMM3_ERR_UNSUPPORTED otherwise); a term that can never hold (wrong-length literal, empty range) drops out. */
#define IMM3_MAX_OR_TERMS 16
int imm3_query_begin_dnf(imm3_db* db, const char* table, const imm3_pred* preds, const int32_t* term_sizes, int nterms,
                         const char* const* proj_cols, int nproj, int64_t limit, imm3_result** out);
/* The same disjunction with options.  flags = 0: imm3_query_begin_dnf, word for word (rows, route, launches, status and
 * message); unknown flag bits give IMM3_ERR_INVALID_ARG.
 * IMM3_DNF_ENCODED_FILTER: a term may also hold ranges (GT / LT / EQ) on sorted-int-codec (PFOR_INT) columns, alone or beside
 * dense predicates.  When at least two terms remain and one of them tests an encoded column, every term runs the block
 * pipeline's filter front (blocks pruned from their min / max where the term's predicates allow it; a term of dense
 * predicates alone takes the mini-block kernel) and blocks_or_merge ORs its per-block selection into the first term's, which
 * the emit kernels then read: e.g. "blocks_prune;blocks_filter_lane/w=11/s=2;blocks_prune;blocks_filter_lane/w=11/s=2;
 * blocks_or_merge;blocks_scan_emit".  Rows, order, LIMIT and the sharded count exchange are those of imm3_query_begin.
 * The table's blocks must hold at most 1024 rows (else IMM3_ERR_UNSUPPORTED).  Terms that touch no encoded column take
 * imm3_query_begin_dnf's row-space path; a single remaining term is the plain conjunction of imm3_query_begin. */
#define IMM3_DNF_ENCODED_FILTER 0x4u /* the bit of IMM3_AGG_ENCODED_FILTER */
int imm3_query_begin_dnf_ext(imm3_db* db, const char* table, const imm3_pred* preds, const int32_t* term_sizes, int nterms,
                             const char* const* proj_cols, int nproj, int64_t limit, uint32_t flags, imm3_result** out);

/* ---- The fan-in across GPUs: ResultQueueOp (ResultQueue.scala:7-56) + the queue of Engine.scala:166,190-196 ----
 * The reference funnels every worker's batches through one queue; across segment-sharded GPUs the ordered
 * concatenation and the LIMIT cut need only the match count of every rank (global order = rank order).  The GPUs
 * exchange those counts THEMSELVES: each rank owns a small mailbox in its HBM, exported as an IPC handle; once every
 * rank has mapped every mailbox (imm3_comm_connect), imm3_query_begin appends a one-warp kernel to the query that
 * stores the local count into every peer's mailbox over NVLink and waits for the peers' counts - no host round trip,
 * no collective library.  Bootstrap: each rank calls imm3_comm_local_handle, the IMM3_COMM_HANDLE_BYTES-byte handles
 * are all-gathered by whatever channel the host processes share (the JVM shim: its own RPC; bench/tests:
 * torch.distributed), rank order = imm3_open_opts.rank, then each rank calls imm3_comm_connect with all of them.
 * One process per GPU on one NVLink-connected node; every rank must issue the same queries in the same order. */
#define IMM3_COMM_HANDLE_BYTES 64
int imm3_comm_local_handle(imm3_db* db, void* handle_out /* IMM3_COMM_HANDLE_BYTES */);
int imm3_comm_connect(imm3_db* db, const void* handles /* world x IMM3_COMM_HANDLE_BYTES, rank order */, int nhandles);
/* After imm3_query_begin on a connected handle (a single handle reports offset 0, take = count = local count): */
int64_t imm3_result_global_offset(const imm3_result* r); /* ordinal of this rank's first row in the global result  */
int64_t imm3_result_take(const imm3_result* r);          /* leading local rows that survive the global LIMIT cut    */
int64_t imm3_result_global_count(const imm3_result* r);  /* rows of the whole result: min(limit, sum of counts)     */
int imm3_result_rank_counts(const imm3_result* r, int64_t* counts, int cap); /* local count of every rank; returns world */
int imm3_result_fetch(imm3_result* r, int64_t nrows);
/* Asynchronous form of fetch: the device->host copies are queued on the handle's copy stream and
 * the call returns; imm3_result_wait blocks until the rows are in host memory.  The consumer of
 * the reference is lazy too - ProjectOp.ProjectIterator materialises rows as they are pulled
 * (Project.scala:22-81) - so a caller can overlap the read-back of one query with staging the
 * next one's inputs (imm3_reupload) over the full-duplex PCIe link.  The result (and its device
 * buffers) must stay open until the wait has returned. */
int imm3_result_fetch_async(imm3_result* r, int64_t nrows);
int imm3_result_wait(imm3_result* r);

/* ---- Scan -> Select* -> ProjectAgg: Engine.execute ProjectAgg branch (Engine.scala:200-232), ProjectAggOp
 *      (ProjectAggregate.scala:115-226), ProjectAggregateQueueOp (ProjectAggregateQueue.scala:9-54) -------------------
 * count / min / max over the selected rows, grouped by `group_cols` (none = one group, reported only if a row was
 * selected).  The aggregate kinds are the ones Engine.resolveProjectOp accepts (Engine.scala:130-156): Min / Max on INT
 * and TINYINT columns (the reference widens to Double: results are IMM3_COL_DOUBLE), Count on any column
 * (IMM3_COL_COUNT); Sum / Avg throw there ("Unknown Aggregate type") and return IMM3_ERR_UNSUPPORTED here, as do Min / Max
 * on STRING columns (the reference maps both to MaxStringAggr, Engine.scala:137,147).
 * Result: one row per group, in the order the groups first appear in canonical row order (what the reference's
 * LinkedHashMaps produce with one worker); columns = the group columns (their own types), then one column per aggregate in
 * select-list order, named <col>_count / <col>_min / <col>_max (Engine.scala:136-152).  imm3_result_format_row prints the
 * aggregates only, as the reference does (Row of the aggregators' repr, ProjectAggregateQueue.scala:48-50).
 * Library limits (IMM3_ERR_UNSUPPORTED): group cells must pack into 7 bytes (a sorted-int-codec INT cell takes 4); aggregate
 * and group columns may be dense or sorted-int-codec (PFOR_INT), but one query decodes at most 4 distinct sorted-int-codec
 * columns, from blocks of at most 1024 rows; predicates on a sorted-int-codec column cannot be combined with aggregation
 * here (imm3_query_agg_ext with IMM3_AGG_ENCODED_FILTER accepts them).  On a sharded handle the result holds
 * this rank's groups (partials); imm3_query_agg_global below merges them on the GPUs. */
typedef enum imm3_agg_op { IMM3_AGG_COUNT = 0, IMM3_AGG_MIN = 1, IMM3_AGG_MAX = 2, IMM3_AGG_SUM = 3, IMM3_AGG_AVG = 4 } imm3_agg_op;
typedef struct imm3_agg {
    const char* col;
    int32_t op;  /* imm3_agg_op */
} imm3_agg;
int imm3_query_agg(imm3_db* db, const char* table, const imm3_pred* preds, int npreds, const imm3_agg* aggs, int naggs,
                   const char* const* group_cols, int ngroup, imm3_result** out);
/* The aggregate fan-in across segment-sharded GPUs (ProjectAggregateQueueOp, ProjectAggregateQueue.scala:9-54): the same
 * arguments, validation and result layout as imm3_query_agg, but every rank of a connected handle (imm3_comm_connect) gets
 * the WHOLE table's groups - the same rows on every rank, in first-appearance order over the global canonical order (rank
 * order, then the rank's own order), COUNT summed and MIN / MAX taken over the ranks.  Each rank compacts its partial
 * groups into an exchange buffer beside its mailbox, announces their number through the mailbox ring, and merges every
 * rank's buffer over NVLink into its own table: one stream, one synchronisation, no host round trip.  On a world == 1
 * handle the result is exactly imm3_query_agg's; a world > 1 handle that is not connected returns IMM3_ERR_STATE.
 * imm3_result_rank_counts reports every rank's partial group count, imm3_result_global_count the merged groups.
 * A refusal of one rank's slice (more groups than its table holds, blocks of more than 1024 rows, shared memory) is
 * exchanged too: every rank returns the same IMM3_ERR_UNSUPPORTED.  IMM3_AGG_SLOTS above 65536 is refused.  Every rank
 * must issue the same queries (aggregates and Project queries alike) in the same order. */
int imm3_query_agg_global(imm3_db* db, const char* table, const imm3_pred* preds, int npreds, const imm3_agg* aggs, int naggs,
                          const char* const* group_cols, int ngroup, imm3_result** out);
/* Sum and Avg, which the query language has and the reference engine refuses, behind an entry point of their own (the
 * two above keep refusing them).  flags = 0: imm3_query_agg; IMM3_AGG_GLOBAL: imm3_query_agg_global.  Without a Sum /
 * Avg the result - rows, names, types, route, status and message - is the one that entry point returns; unknown flag
 * bits give IMM3_ERR_INVALID_ARG.
 *   Sum(c), c INT or TINYINT (dense or PFOR_INT): the exact sum of the group's selected values, column <c>_sum,
 *           IMM3_COL_INT64.
 *   Avg(c): (double)sum / (double)count, computed once on the host in IEEE double, column <c>_avg, IMM3_COL_DOUBLE;
 *           imm3_result_format_row prints it as Double.toString does (shortest round-trip digits).
 * Sum / Avg on a STRING column give IMM3_ERR_UNSUPPORTED.  A query with a Sum or Avg carries one Count of the group's
 * rows: its own first Count, else a hidden one that is not in the result; visible plus hidden aggregates must be at most
 * 8 (else IMM3_ERR_UNSUPPORTED).  Every add, on the GPU and in the merge, is a 64-bit two's-complement add, so a sum is
 * exact whenever its group has at most 2^32 rows; a group with more rows (on a global aggregate: after the merge)
 * returns IMM3_ERR_UNSUPPORTED, never a wrapped value.
 * IMM3_AGG_ENCODED_FILTER: predicates on sorted-int-codec (PFOR_INT) columns are accepted - ranges (GT / LT / EQ), alone or
 * mixed with predicates on dense columns - and decided by the block pipeline's filter kernels (blocks pruned from their
 * min / max statistics where every predicate is such a range), whose per-block selection the aggregation kernel reads;
 * the route then ends in agg_blocks<NG,NA>/bsel.  The table's blocks must hold at most 1024 rows (else
 * IMM3_ERR_UNSUPPORTED).  A query with no predicate on an encoded column is unaffected by the flag: the same rows, names,
 * types, route, status and message.  Combines with IMM3_AGG_GLOBAL and with Sum / Avg.  Without the flag (and in the two
 * entry points above) such predicates keep giving IMM3_ERR_UNSUPPORTED. */
#define IMM3_AGG_GLOBAL 0x1u
#define IMM3_AGG_ENCODED_FILTER 0x4u
int imm3_query_agg_ext(imm3_db* db, const char* table, const imm3_pred* preds, int npreds, const imm3_agg* aggs, int naggs,
                       const char* const* group_cols, int ngroup, uint32_t flags, imm3_result** out);

/* Same query text the reference CLI takes (SQLParser.scala:8-129; SqlCli.scala:60). */
int imm3_query_sql(imm3_db* db, const char* sql, imm3_result** out);

int64_t imm3_result_nrows(const imm3_result* r);            /* rows fetched to host                    */
int imm3_result_ncols(const imm3_result* r);
int imm3_result_col_type(const imm3_result* r, int col);    /* imm3_column_type                         */
int imm3_result_col_width(const imm3_result* r, int col);   /* bytes per cell: 4 (LE int32), 1 (int8), k */
const char* imm3_result_col_name(const imm3_result* r, int col);
const void* imm3_result_col_data(const imm3_result* r, int col); /* host, pinned, nrows*width bytes    */
const void* imm3_result_col_device(const imm3_result* r, int col); /* device copy (valid until free)    */
/* Row.toString (Record.scala:13): writes "Row(v1,v2,...)" for row i; returns length or <0. */
int imm3_result_format_row(const imm3_result* r, int64_t row, char* buf, size_t buflen);
double imm3_result_device_ms(const imm3_result* r);         /* CUDA-event time of the kernels of begin  */
/* Kernels launched by begin / imm3_query_agg, count exchanges included: the number of entries in imm3_result_route (0 when
 * it is ""). */
int imm3_result_kernel_launches(const imm3_result* r);
/* The kernels imm3_query_begin / imm3_query_agg queued, in launch order, separated by ';' ("" when none ran): kernel names
 * (select_all, filter(tma|direct), offset_scan, emit_stream, emit, emit_general, blocks_prune, blocks_filter_lane,
 * blocks_filter_quad, blocks_filter, blocks_or_merge, blocks_group_emit, blocks_scan_emit, blocks_emit(rowspace|blocks), scan_blocks,
 * count_exchange, agg_init, agg<NG,NA>, agg_blocks<NG,NA>, agg_compact, agg_exchange, agg_merge) with "/key=value" parameters: /s= ring stages,
 * /w= warps per CTA of the lane kernel, /ctas= the group emit kernel's grid; "/prefix" marks the prefix pass of a small
 * LIMIT; "/sum" the SUM instantiation of agg<NG,NA> / agg_blocks<NG,NA> (imm3_query_agg_ext with a Sum or Avg); "/bsel" (after
 * "/sum" when both) agg_blocks<NG,NA> over the block filter's selection (IMM3_AGG_ENCODED_FILTER with a predicate on an encoded
 * column, whose filter kernels - blocks_prune, blocks_filter*, offset_scan - are recorded as for a Project query), e.g.
 * "agg_init;blocks_prune;blocks_filter_lane/w=11/s=2;agg_blocks<1,3>/bsel;agg_compact".  E.g. "blocks_prune;blocks_filter_lane/w=11/s=2;blocks_group_emit/ctas=148"; a global aggregate on a connected
 * handle: "agg_init;filter(tma)/s=4;agg<1,2>;agg_compact;agg_exchange;agg_init;agg_merge;agg_compact" (a rank with an empty
 * slice starts at agg_exchange).  Owned by the result (valid until imm3_result_free). */
const char* imm3_result_route(const imm3_result* r);
/* CUDA-event time of one stage of begin: 0 = filter (+scan) kernel, 1 = emit kernel (multi-pass path);
 * the fused single-pass kernels report everything as stage 0. */
double imm3_result_stage_ms(const imm3_result* r, int stage);
/* Wall clock (microseconds) spent inside imm3_query_begin, by phase: 0 = validation + logical plan, 1 = result buffers + device
 * plan, 2 = queueing the launches, 3 = waiting for the GPU (kernels + count exchange + the 200-byte read-back), 4 = epilogue. */
double imm3_result_host_us(const imm3_result* r, int phase);
int64_t imm3_result_algorithmic_bytes(const imm3_result* r);/* SURVEY.md §8d formula for this query     */
int imm3_result_free(imm3_result* r);

/* Selection bitmap of the conjunctive filter alone (north_star stage 3; Select.scala keeps it in
 * FilledColumnVectorBatch.selected): bit i of word w = canonical row 32*w+i of the owned slice.
 * `words` receives a library-owned host array of ceil(nrows/32) uint32, valid until the next call
 * on this db. */
int imm3_filter_bitmap(imm3_db* db, const char* table, const imm3_pred* preds, int npreds,
                       const uint32_t** words, int64_t* nwords, int64_t* nselected);

/* Host-side plan of a query as JSON (narrowed constants, merged ranges, kernel choice); works on
 * IMM3_OPEN_HOST_ONLY handles.  Library-owned string, valid until the next call on this db. */
int imm3_explain(imm3_db* db, const char* table, const imm3_pred* preds, int npreds,
                 const char* const* proj_cols, int nproj, int64_t limit, const char** json);

/* ---- Writer side: SegmentWriter (Segment.scala:70-152) + LoaderCli roll logic
 *      (LoaderCli.scala:113-154) + TableIO.store (Table.scala:50-59) ---------------------------
 * col_specs uses the loader's syntax "name:CODEC[:k=v;k=v]" (LoaderCli.scala:66-80), plus PFOR_INT,
 * which the reference loader cannot create (SURVEY.md §3.4 B3) but Column.make accepts. */
int imm3_writer_open(const char* data_dir, const char* table, const char* const* col_specs, int ncols,
                     int32_t block_size, int32_t segment_size, int32_t first_segment_id,
                     int write_table_meta, imm3_writer** out);
/* Append nrows rows given one typed array per column: int32 for INT, int8 for TINYINT, nrows*k
 * bytes for STRING(k). */
int imm3_writer_append(imm3_writer* w, const void* const* col_data, int64_t nrows);
/* CSV body line(s) exactly as LoaderCli splits them (split on ',', trim). */
int imm3_writer_append_csv_line(imm3_writer* w, const char* line);
int imm3_writer_close(imm3_writer* w);
/* Whole-file CSV loader: first line is a header and is discarded (LoaderCli.scala:115-116). */
int imm3_load_csv(const char* data_dir, const char* table, const char* const* col_specs, int ncols,
                  int32_t block_size, int32_t segment_size, const char* csv_path);
/* PFORCodecInt.encode (PFORCodec.scala:17-28): n int32 -> big-endian words + 8 zero bytes.
 * Returns bytes written or <0; call with out==NULL to size. */
int64_t imm3_pfor_encode(const int32_t* values, int32_t n, uint8_t* out, int64_t out_cap);
/* The same encoder on the GPU for a whole column (SURVEY.md 8f-1): `n` values are cut into blocks of
 * `block_rows` values (the SegmentWriter's blocks, Segment.scala:99-151: every block restarts the
 * delta chain at 0), every block is encoded exactly as imm3_pfor_encode encodes it and the blocks are
 * written back to back; block_off (nblocks+1 entries, may be NULL) receives their byte offsets -
 * SegmentMeta.blockOffsets (Segment.scala:33).  block_rows: a multiple of 32, at most 1024.
 * Returns the bytes written, or the bytes needed when out == NULL, or <0. */
int64_t imm3_pfor_encode_blocks_gpu(int device, const int32_t* values, int64_t n, int32_t block_rows,
                                    uint8_t* out, int64_t out_cap, int64_t* block_off);

/* Deterministic synthetic tables of BASELINE.md (id=row index, age uniform [0,100), state uniform
 * over 51 two-letter codes; counter-based PRNG, seed 42).  Writes the canonical segments
 * [seg_begin, seg_end) of an nrows table laid out exactly as the loader would (S*B+1 rows per full
 * segment).  id_codec is IMM3_CODEC_DENSE_INT or IMM3_CODEC_PFOR_INT. */
int imm3_synth_write(const char* data_dir, const char* table, int64_t nrows, int32_t block_size,
                     int32_t segment_size, int32_t id_codec, int32_t seg_id_begin, int32_t seg_id_end,
                     int write_table_meta);
/* Value of the synthetic generator for one row (so tests can check it without files). */
void imm3_synth_row(int64_t row, int32_t* id, int8_t* age, char state[2]);

const char* imm3_last_error(void);
int imm3_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* IMM3_H */
