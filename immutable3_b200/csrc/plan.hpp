// plan.hpp — the query plan handed to the kernels (POD, passed as a __grid_constant__ parameter)
// and the host-side planner that produces it from the reference's Query shape
// (Query.scala:3-46 flattened by Engine.resolveSelectOps / PipelineThread.runOps,
// Engine.scala:108-128, 237-245).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "common.hpp"

namespace imm3 {

constexpr int kMaxFilterCols = 8;   // distinct columns carrying predicates
constexpr int kMaxProjCols = 16;    // select-list length (duplicates allowed, Project.scala:55-57)
constexpr int kMaxPforCols = 4;     // PFOR_INT columns touched by one query
constexpr int kLitPoolBytes = 512;  // MATCH literals of all filter columns, packed
constexpr int kDenseTileRowsPerWord = 8192;  // dense kernel: 8 compute warps x 32 lanes x 32 rows per bitmap word
constexpr int kDenseTileMinRows = 400;  // an 8192-row tile with at least this many selected rows (4.9 %) is streamed, not gathered:
                                        // measured crossover of the two emit kernels (age < t sweep, 100 M rows: equal at 5 %)
constexpr int kDenseMaxTileRows = 4 * kDenseTileRowsPerWord;  // tile = 8192 * W rows, W in {1, 2, 4}
constexpr int kBlockThreads = 256;  // block-mode kernel: threads per CTA
constexpr int kMaxBlockRows = 8192; // block-mode kernel: largest reference block it stages
// Tile-status arrays of the dense kernel (counts, then offsets) are padded to whole scanner rounds of 256 tiles.
constexpr long long status_round_up(long long ntiles) { return ((ntiles + 255) & ~255ll) + 256; }
constexpr int kMaxFilterStages = 8;  // TMA ring depth of the multi-pass filter kernel

enum FilterKind : int32_t {
    kFilterI8Range = 0,   // TINYINT: lo <= v <= hi   (merged GT/LT/EQ, Select.scala:53-165)
    kFilterI32Range = 1,  // INT
    kFilterStrMatch = 2,  // STRING(k): cell equals one of nlit literals (Select.scala:25-51)
};

struct FilterCol {
    const uint8_t* base;  // device arena of the column (dense) or nullptr (PFOR: decoded in shared memory)
    int32_t width;        // bytes per decoded value
    int32_t kind;         // FilterKind
    int32_t lo;           // ranges: inclusive lower bound
    uint32_t span;        // ranges: (uint32)(hi - lo)
    int32_t nlit;         // match: number of literals (each `width` bytes) ...
    int32_t lit_off;      // ... at lits[lit_off]
    int32_t smem_off;     // dense kernel: byte offset of this column's tile inside a stage, -1 = read from global
    int32_t pfor_slot;    // block kernel: index into ScanPlan::pfor, -1 = dense column
    int32_t keep_l2;      // multi-pass: the column is projected too and small enough to stay in L2 until the emit kernel
    int32_t pad;
};

struct ProjCol {
    const uint8_t* base;  // device arena (dense) or nullptr (PFOR)
    uint8_t* out;         // device result column
    int32_t width;
    int32_t filter_idx;   // >= 0: same column as filter[filter_idx] (its staged tile can be reused)
    int32_t pfor_slot;
    int32_t stage_off;    // fused dense kernel: byte offset of this column's 1024-row span in a warp's staging buffer
};

struct PforCol {
    const uint32_t* words;     // device arena viewed as big-endian 32-bit words
    const uint32_t* word_off;  // nblocks+1 word offsets of the blocks (file order = canonical order)
};

struct ScanPlan {
    int64_t nrows;        // rows in the owned slice
    int64_t limit;        // rows wanted (INT64_MAX = unlimited)
    int64_t ntiles;       // dense: ceil(nrows / 8192); block mode: number of reference blocks
    const uint64_t* row_start;  // block mode: nblocks+1 canonical row ordinals
    uint32_t* bitmap;     // filter-bitmap mode: selection bitmap out (else nullptr)
    unsigned long long* trace;  // debugging (IMM3_TRACE): 8 globaltimer stamps per tile, else nullptr
    uint32_t epoch;       // tags the tile-status words of this launch
    int32_t nfilter;
    int32_t nproj;
    int32_t npfor;
    int32_t stages;       // dense: TMA pipeline depth (0 = direct loads, no staging)
    int32_t stage_bytes;  // dense: bytes of one stage
    int32_t max_block_rows;  // block mode: rows of the largest block (shared-memory sizing)
    int32_t lit_bytes;       // bytes of `lits` in use
    int32_t blk_words_cap;   // block-mode multi-pass: 32-bit words of the largest encoded PFOR block (+ slack), per-warp scratch
    int32_t blk_tile_bytes;  // blocks_filter_kernel: bytes reserved per staged encoded column in a ring slot (largest 8-block tile)
    int32_t scan_inline;     // 1: the filter kernel's last CTA turns the tile counts into offsets; 0: offset_scan_kernel does (large tables)
    uint32_t pfor_filter_mask;  // blocks_filter_kernel: PFOR slots that carry a predicate (their tiles are staged)
    int32_t pad0;            // unused: keeps the offsets of the members behind it (kernel parameter layout)
    int32_t or_accumulate;   // filter kernel: OR this conjunction's bits into the bitmap already there (second and later terms of a disjunction)
    uint32_t debug;          // IMM3_DEBUG env bits (timing experiments only; bit 0: skip the look-back -> WRONG offsets)
    FilterCol filter[kMaxFilterCols];
    ProjCol proj[kMaxProjCols];
    PforCol pfor[kMaxPforCols];
    uint8_t lits[kLitPoolBytes];
};

// What blocks_scan_emit_kernel needs of a plan (k_blocks_scanemit.cuh): a parameter block of 72 bytes instead of ScanPlan's 4 KB.
struct LeanPlan {
    const uint64_t* row_start;   // nblocks + 1 canonical row ordinals
    const uint32_t* words;       // the projected encoded column: big-endian word stream ...
    const uint32_t* word_off;    // ... and one word offset per block (+ 1)
    uint8_t* out;                // result column (int32 values)
    int64_t limit;               // rows wanted (INT64_MAX = unlimited)
    int64_t ntiles;              // 8-block tiles
    unsigned long long* trace;   // debugging (IMM3_DEBUG=16 + IMM3_TRACE), else nullptr
    uint32_t debug;
    uint32_t pad;
};

// Block pruning (k_blocks_prune.cuh): exact signed min / max of every block of an encoded INT column, computed on the GPU
// when the table is opened, and the plan of the kernel that decides whole blocks from them.
struct alignas(8) BlockStat {
    int32_t mn, mx;
};
struct PrunePlan {
    const BlockStat* stats[kMaxFilterCols];  // per predicate: the block statistics of its column
    int32_t lo[kMaxFilterCols], hi[kMaxFilterCols];  // inclusive signed window
    int32_t nfilter;
    int32_t group_shift;  // work-list granularity: tiles of 1 << group_shift blocks (5: quad filter kernel, 3: blocks_filter_kernel)
};

// Aggregation (k_agg.cuh; ProjectAggOp, ProjectAggregate.scala:115-226): count / min / max over the rows the filter
// kernel selected, grouped by up to kMaxGroupCols columns whose cells pack into at most 7 key bytes.  A MIN / MAX input or
// a group column in the sorted-int codec is decoded per block inside agg_blocks_kernel (its slot in agg_pfor / group_pfor).
constexpr int kMaxAggs = 8;
constexpr int kMaxGroupCols = 4;
enum AggOp : int32_t { kAggCount = 0, kAggMin = 1, kAggMax = 2, kAggSum = 3 };  // (kAggSum: imm3_query_agg_ext only)
struct AggCol {
    const uint8_t* base;  // device arena of the aggregated column (dense INT / TINYINT; unused for COUNT)
    int32_t width;        // 4 or 1
    int32_t op;           // AggOp
};
struct GroupCol {
    const uint8_t* base;
    int32_t width;        // bytes per cell
    int32_t key_shift;    // bit position of this column's cell inside the packed 64-bit key
};
struct AggPlan {
    int64_t nrows;
    int64_t ntiles;        // 8192-row tiles of the row-space bitmap
    int32_t naggs, ngroup;
    uint32_t table_slots;  // global hash table size (power of two)
    int32_t pad;
    AggCol agg[kMaxAggs];
    GroupCol group[kMaxGroupCols];
    // agg_blocks_kernel only (after the fields agg_kernel reads, which keep their parameter offsets):
    int8_t agg_pfor[kMaxAggs];          // index into pfor[] of a MIN / MAX / SUM input in the sorted-int codec, -1 = dense
    int8_t group_pfor[kMaxGroupCols];   // ... of a group column, -1 = dense
    int32_t npfor;                      // distinct encoded columns decoded per block
    int32_t blk_words_cap;              // per-warp scratch for one encoded block, in 32-bit words (from the columns' max_block_words)
    int64_t nblocks;                    // reference blocks of the owned slice
    const uint64_t* row_start;          // nblocks + 1 row ordinals of the blocks (row space of the dense arenas)
    PforCol pfor[kMaxPforCols];
};
// One group in the global table / in the compacted result.  val[i]: COUNT -> the count, MIN / MAX -> the extreme as int64,
// SUM -> the sum modulo 2^64.
struct AggEntry {
    unsigned long long key;        // packed group cells, ~0 = empty slot
    unsigned long long first_row;  // canonical ordinal of the group's first selected row (groups are reported in that order)
    long long val[kMaxAggs];
};

// Device-resident control block of one db (reset by the last CTA of every launch).
struct ScanCtrl {
    unsigned int ticket;   // next tile to hand out
    unsigned int done;     // LIMIT reached: later tiles are dead
    unsigned int exited;   // CTAs that have left the kernel
    unsigned int error;    // watchdog: a bounded spin expired (never hang the GPU)
    unsigned long long total;  // rows emitted (min(limit, matches)) or matches in bitmap mode
    unsigned int scanner;  // dense kernel: the grid's scanner warp has been elected
    unsigned int ticket2;  // multi-pass: next tile of the streaming emit kernel (reset by the filter kernel's last CTA)
    unsigned long long dense_rows;  // multi-pass: selected rows living in tiles with >= 1 selected row in 32 (emit-kernel choice)
};

// ---------------------------------------------------------------------------------------------
// Multi-GPU count exchange over NVLink peer memory (k_comm.cuh).  Every rank owns a MAILBOX in its HBM:
// kCommRing rounds x kMaxWorld senders of one 64-bit word  [63:40] exchange epoch, [39:0] match count.
// Rank r stores its word into slot [epoch % ring][r] of EVERY rank's mailbox (peer stores through NVLink,
// the pointers come from cudaIpcOpenMemHandle) and then polls its own mailbox until all `world` words of the
// epoch have arrived.  Replaces the fan-in of ResultQueue.scala:7-56 / Engine.scala:166,190-196.
// ---------------------------------------------------------------------------------------------
constexpr int kMaxWorld = 16;
constexpr int kCommRing = 4;
constexpr size_t kMailboxBytes = (size_t)kCommRing * kMaxWorld * sizeof(unsigned long long);

struct CommPlan {
    unsigned long long* peer[kMaxWorld];  // mailbox of every rank as mapped in THIS process (peer[rank] = the local one)
    int32_t rank, world;
    uint32_t epoch;                       // exchange sequence number of this db (identical on all ranks)
    int32_t has_count;                    // 0: this rank ran no kernel (empty slice) - it contributes 0
    long long limit;                      // INT64_MAX = unlimited
    unsigned long long timeout_ns;
    struct CtrlBlock* pub;                // pinned host control block to publish into (nullptr: the host copies it itself)
    unsigned long long pub_seq;
};

// Global aggregation (imm3_query_agg_global, k_comm.cuh agg_exchange_kernel / k_agg.cuh agg_merge_kernel): the mailbox's
// allocation also holds this rank's EXCHANGE AREA, two buffers of kAggXchgSlots AggEntry at kAggXchgOff bytes from the
// mailbox base - peers reach them at the base they already mapped.  Aggregate s of a db compacts its partial groups into
// buffer s & 1 (s = agg_seq, identical on all ranks); the ring word of the exchange round carries the group count.
constexpr size_t kAggXchgOff = 4096;
constexpr uint32_t kAggXchgSlots = 1u << 16;
constexpr unsigned long long kAggXchgError = 1ull << 32;  // ring word payload: [32] this rank's partials are unusable, [31:0] its group count
constexpr size_t kCommAllocBytes = kAggXchgOff + 2 * (size_t)kAggXchgSlots * sizeof(AggEntry);  // mailbox + exchange area (~10 MiB)
static_assert(kMailboxBytes <= kAggXchgOff, "the exchange area starts behind the mailbox ring");

struct AggXPlan {
    unsigned long long* peer[kMaxWorld];  // mailbox of every rank as mapped in THIS process (peer[rank] = the local one)
    int32_t rank, world;
    uint32_t epoch;                       // exchange round (db->comm_epoch, shared with the count exchange)
    int32_t has_local;                    // 0: no local kernels ran (empty slice, or a refusal of this slice): 0 groups
    int32_t refused;                      // 1: this slice refuses the query (posted as the error bit)
    int32_t pad;
    unsigned long long timeout_ns;
};
// What agg_exchange_kernel leaves for agg_merge_kernel and the host.
struct AggXOut {
    unsigned long long counts[kMaxWorld];  // partial group count of every rank
    unsigned int err_mask;                 // bit r: rank r posted the error bit (local overflow or a refusal of its slice)
    unsigned int late;                     // 1: a peer's word did not arrive before the timeout
};
struct AggMergePlan {
    const AggEntry* buf[kMaxWorld];  // this aggregate's exchange buffer of every rank, as mapped here
    int32_t world;
    uint32_t slots;                  // merged table size (power of two)
    int32_t naggs;
    int32_t op[kMaxAggs];            // AggOp of every aggregate
};

// What the exchange kernel leaves behind for the host (copied back together with ScanCtrl).
struct CommOut {
    unsigned long long g_offset;  // global ordinal of this rank's first row = sum of the counts of the ranks before it
    unsigned long long g_take;    // rows of this rank that survive the global LIMIT cut
    unsigned long long g_total;   // rows of the whole result (min(limit, sum of counts))
    unsigned int error;           // 1 = a peer's count did not arrive before the timeout
    unsigned int world;
    unsigned long long counts[kMaxWorld];  // local count of every rank (each capped at LIMIT)
};

struct CtrlBlock {
    ScanCtrl c;
    CommOut x;
    unsigned long long pub_seq;  // host copy only: [63:41] the query whose control block the GPU itself has written there (see below)
};
// "Publish": the last kernel of a query (blocks_scan_emit_kernel, or count_exchange_kernel on a sharded table) stores the
// control block straight into the handle's pinned host copy and then the query's sequence number; the host polls that word
// instead of queueing a device-to-host copy and synchronising the stream (measured: 11 us from the last kernel's end to the
// return of cudaStreamSynchronize, ~2 us with the poll).

// ---------------------------------------------------------------------------------------------
// Host-side logical plan (independent of device pointers; testable on CPU through imm3_explain).
// ---------------------------------------------------------------------------------------------
struct LogicalFilter {
    int col_idx = -1;          // index in TableMeta::cols
    int kind = 0;              // FilterKind
    int64_t lo = 0, hi = 0;    // inclusive range after merging every GT/LT/EQ on the column
    std::vector<std::string> lits;  // k-byte literals surviving the intersection of all Match lists
};

struct LogicalPlan {
    const TableMeta* table = nullptr;
    std::vector<LogicalFilter> filters;   // one per distinct filter column, first-appearance order
    std::vector<int> proj;                // column indices in select-list order
    int64_t limit = 0;                    // <= 0: unlimited
    bool always_empty = false;            // a predicate can never hold (lo > hi, no literal of length k)
    bool uses_pfor = false;
    // Narrowed constants per input predicate, for imm3_explain and the tests of SURVEY.md §8c.
    struct Narrowed { std::string col; int op; int32_t ival; int8_t bval; };
    std::vector<Narrowed> narrowed;
};

int find_col(const TableMeta& t, const char* name);  // column index by name, -1: none (or NULL)
int build_logical_plan(const TableMeta& table, const imm3_pred* preds, int npreds, const char* const* proj_cols,
                       int nproj, int64_t limit, LogicalPlan* out);
std::string explain_json(const LogicalPlan& lp, const char* kernel);

// SQLParser.parseAll restatement (SQLParser.scala:8-129) for the Project form of the grammar.
struct ParsedQuery {
    std::string table;
    std::vector<std::string> pred_cols;
    std::vector<imm3_pred> preds;              // .col / .strs point into the vectors below
    std::vector<std::vector<std::string>> pred_strs;
    std::vector<std::vector<const char*>> pred_str_ptrs;
    std::vector<std::string> proj;
    int64_t limit = 0;
    void fix_pointers();
};
int parse_sql(const char* sql, ParsedQuery* out);

}  // namespace imm3
