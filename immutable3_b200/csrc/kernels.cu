// kernels.cu - sm_100a kernels of the scan -> filter -> project path (one translation unit; the device code lives in the
// k_*.cuh fragments included below, this file holds the launchers).  Each launcher owns its kernel's sizing: the sizing
// rule beside it turns a plan into the kernel's ring, shared memory, CTA width, occupancy and grid, from the layout
// constants of the kernel's fragment, so the planner (engine.cu) never sees them.
//
// Reference path: ScanOp / DenseCodec*.decode / sorted-int codec (Scan.scala:28-70, DenseCodec.scala:34-74,
// PFORCodec.scala:12-28) -> conjunctive RangeFilter / MatchFilter (Select.scala:14-165) -> Project with an exact LIMIT in
// canonical row order (Project.scala:37-80).
//
//   k_multipass.cuh      dense tables (default): filter_kernel -> offset scan by its last CTA -> emit_stream_kernel (dense
//                        results, TMA-streamed) or emit_kernel / emit_general_kernel (sparse results, gathers)
//   k_blocks_multi.cuh   any query touching a sorted-int-codec column: blocks_filter_kernel (or the dense filter kernel in
//                        row space when no predicate touches an encoded column) -> blocks_emit_kernel, one warp per block
//   k_blocks_or.cuh      blocks_or_merge_kernel: real OR over encoded columns, the union of two block filter selections
//   k_blocks_single.cuh  scan_blocks_kernel: single-pass block kernel with decoupled look-back (blocks > 1024 rows, bitmaps)
//   k_rowspace.cuh       predicates (SIMD within a register), selection vectors, gathers, plan tables in shared memory
//   k_ptx.cuh            mbarrier / TMA / L2-policy / relaxed-load helpers
//
// Tiles are handed out by atomic tickets, so a tile only ever waits on tiles that are already running (forward progress
// without relying on block scheduling order).  No spin is unbounded: a watchdog traps instead of hanging the GPU.
#include <cuda_runtime.h>
#include <algorithm>
#include <type_traits>

#include <climits>
#include <cstdint>
#include <cstdlib>
#include <cstring>

#include "kernels.hpp"
#include "plan.hpp"

namespace imm3 {

#include "k_ptx.cuh"
#include "k_rowspace.cuh"
#include "k_blocks_single.cuh"
#include "k_multipass.cuh"
#include "k_blocks_multi.cuh"
#include "k_blocks_scanemit.cuh"
#include "k_blocks_groupemit.cuh"
#include "k_blocks_filter.cuh"
#include "k_blocks_lane.cuh"
#include "k_blocks_prune.cuh"
#include "k_blocks_or.cuh"
#include "k_comm.cuh"
#include "k_agg.cuh"

// =============================================================================================
// Launchers
// =============================================================================================
constexpr int kSmemCap = 200 * 1024;      // opt-in dynamic shared memory of the kernels configure_device sets up ...
constexpr int kLaneSmemCap = 222 * 1024;  // ... and of blocks_filter_lane_kernel (one CTA per SM)

cudaError_t configure_device() {
    cudaError_t e = cudaSuccess;
#define IMM3_SET_SMEM(K) if ((e = cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemCap)) != cudaSuccess) return e
    IMM3_SET_SMEM(emit_stream_kernel);
    IMM3_SET_SMEM(blocks_filter_kernel);
    IMM3_SET_SMEM(blocks_filter_quad_kernel);
    if ((e = cudaFuncSetAttribute(blocks_filter_lane_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLaneSmemCap)) != cudaSuccess) return e;
    IMM3_SET_SMEM(block_stats_kernel);
    IMM3_SET_SMEM(blocks_emit_kernel<true>);
    IMM3_SET_SMEM(blocks_emit_kernel<false>);
    IMM3_SET_SMEM(emit_general_kernel);
    IMM3_SET_SMEM(filter_kernel<true>);
    IMM3_SET_SMEM(filter_kernel<false>);
#undef IMM3_SET_SMEM
    return cudaFuncSetAttribute(scan_blocks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemCap);
}

// Every cudaLaunchKernelEx launch.  pdl: a programmatic dependent of the stream's previous kernel - it may start while that
// kernel finishes, and waits for its results in griddepcontrol.wait.
template <typename... Params, typename... Args>
static cudaError_t launch_ex(void (*kernel)(Params...), int grid, int block, size_t smem, cudaStream_t stream, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, args...);
}

static std::string with_stages(const char* name, int stages) { return std::string(name) + "/s=" + std::to_string(stages); }

// Per-warp scratch of the block decoders: the byte-swapped words of the largest encoded block, plus slack.
static int block_words_cap(int64_t max_block_words) { return (int)std::min<int64_t>(1120, ((max_block_words + 4 + 31) / 32) * 32); }

// Row-space filter kernel: tiles of 8192 rows; a TMA ring of ~32 KiB, so that four CTAs share an SM.  A stage holds one
// 8192-row sub-tile of every filter column.
cudaError_t size_filter(ScanPlan* sp, bool no_tma, KernelShape* ks) {
    int stage_bytes = 0;
    for (int i = 0; i < sp->nfilter; i++) stage_bytes += kDenseTileRowsPerWord * sp->filter[i].width;
    const bool stage_ok = !no_tma && stage_bytes > 0 && stage_bytes <= 56 * 1024;
    for (int i = 0, off = 0; i < sp->nfilter; i++) {  // where each column sits inside a stage
        sp->filter[i].smem_off = stage_ok ? off : -1;
        off += kDenseTileRowsPerWord * sp->filter[i].width;
    }
    int stages = 0;
    if (stage_ok) stages = std::max(2, std::min(kMaxFilterStages, (32 * 1024) / stage_bytes));
    if (const char* e = getenv("IMM3_FILTER_STAGES")) {
        int v = atoi(e);
        if (stage_ok && v >= 2 && v <= kMaxFilterStages && (size_t)v * stage_bytes <= kSmemCap) stages = v;
    }
    sp->stages = stages;
    sp->stage_bytes = stage_bytes;
    ks->smem = (size_t)stages * (size_t)stage_bytes;
    if (ks->smem > 0) return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ks->occupancy, filter_kernel<true>, kComputeThreads + 32, ks->smem);
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ks->occupancy, filter_kernel<false>, kComputeThreads + 32, ks->smem);
}
cudaError_t launch_filter(const ScanPlan& plan, uint32_t* bitmap, uint32_t* span_cnt, uint32_t* tile_cnt, unsigned long long* tile_off,
                          ScanCtrl* ctrl, int grid, size_t dyn_smem, cudaStream_t stream, std::string* route) {
    if (plan.nfilter == 0) {  // no predicate: nothing to read - the selection metadata is written analytically
        select_all_kernel<<<grid, kComputeThreads, 0, stream>>>(plan, bitmap, span_cnt, tile_cnt, tile_off, ctrl);
        *route = "select_all";
    } else if (plan.stages > 0) {
        filter_kernel<true><<<grid, kComputeThreads + 32, dyn_smem, stream>>>(plan, bitmap, span_cnt, tile_cnt, tile_off, ctrl);
        *route = with_stages("filter(tma)", plan.stages);
    } else {
        filter_kernel<false><<<grid, kComputeThreads + 32, dyn_smem, stream>>>(plan, bitmap, span_cnt, tile_cnt, tile_off, ctrl);
        *route = "filter(direct)";
    }
    return cudaGetLastError();
}
// Who turns the tile counts into offsets: the filter kernel's last CTA (small tables), or offset_scan_kernel - one CTA per
// 4096 counts, launched behind the filter kernel (large tables: 122 K counts at 1 B rows take one SM ~50 us).
bool scan_inline_for(long long ntiles) {
    if (const char* e = getenv("IMM3_SCAN")) {
        if (!strcmp(e, "inline")) return true;
        if (!strcmp(e, "kernel")) return false;
    }
    return ntiles <= kScanInlineMaxTiles;
}

// The dense pipeline's emit kernels: the gather kernel (8 spans of 1024 rows per tile) and the streaming one (dense results).
cudaError_t size_emit(ScanPlan* sp, bool no_tma, int num_sms, EmitShape* es) {
    es->general = sp->nproj > 4 || getenv("IMM3_EMIT_GENERAL");
    for (int i = 0; i < sp->nproj; i++) es->general = es->general || !(sp->proj[i].width == 1 || sp->proj[i].width == 2 || sp->proj[i].width == 4);
    int occ = 0;
    cudaError_t e = es->general ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, emit_general_kernel, kComputeThreads, kComputeWarps * 1024 * 2)
                                : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, emit_kernel, kComputeThreads, kComputeWarps * kEmitWarpSmemBytes);
    if (e != cudaSuccess) return e;
    const int64_t nspans = sp->ntiles * (kDenseTileRowsPerWord / 1024);
    es->grid = (int)std::max<int64_t>(1, std::min<int64_t>((nspans + 7) / 8, (int64_t)num_sms * std::max(1, occ)));
    // Streaming emit kernel: a stage = bitmap words + span counts + one 8192-row tile of every projected column, if that fits.
    int pstage = 0;
    for (int i = 0; i < sp->nproj; i++) {
        sp->proj[i].stage_off = pstage;
        pstage += 1024 * sp->proj[i].width;
    }
    KernelShape& s = es->stream;
    s.stage_bytes = 0;
    if (sp->nproj > 0 && 8 * pstage <= 64 * 1024 && !no_tma && !getenv("IMM3_NO_EMIT_STREAM")) {
        s.stage_bytes = kEmitHdrBytes + 8 * pstage;
        s.stages = std::max(2, std::min(4, (80 * 1024) / s.stage_bytes));
        if (const char* v = getenv("IMM3_EMIT_STAGES")) {
            int n = atoi(v);
            if (n >= 2 && n <= 4) s.stages = n;
        }
        s.smem = (size_t)kComputeWarps * 1024 * 2 + (size_t)s.stages * (size_t)s.stage_bytes + 16;
        if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&s.occupancy, emit_stream_kernel, kComputeThreads + 32, s.smem)) != cudaSuccess) return e;
        if (s.occupancy < 1) s.stage_bytes = 0;
        s.grid = (int)std::max<int64_t>(1, std::min<int64_t>(sp->ntiles, (int64_t)num_sms * std::max(1, s.occupancy)));
    }
    return cudaSuccess;
}
cudaError_t launch_emit(const ScanPlan& plan, const uint32_t* bitmap, const uint32_t* span_cnt, const unsigned long long* tile_off,
                        int spans_per_tile, long long nspans, const EmitShape& es, int dense_off, const ScanCtrl* ctrl, bool pdl,
                        cudaStream_t stream) {
    if (es.general)
        return launch_ex(emit_general_kernel, es.grid, kComputeThreads, kComputeWarps * 1024 * 2, stream, pdl, plan, bitmap, span_cnt, tile_off,
                         spans_per_tile, nspans, dense_off, ctrl);
    return launch_ex(emit_kernel, es.grid, kComputeThreads, kComputeWarps * kEmitWarpSmemBytes, stream, pdl, plan, bitmap, span_cnt, tile_off,
                     spans_per_tile, nspans, dense_off, ctrl);
}
cudaError_t launch_emit_stream(const ScanPlan& plan, const uint32_t* bitmap, const uint32_t* span_cnt, const uint32_t* tile_cnt,
                               const unsigned long long* tile_off, long long nsub, const KernelShape& ks, int dense_mode, ScanCtrl* ctrl,
                               bool pdl, cudaStream_t stream) {
    return launch_ex(emit_stream_kernel, ks.grid, kComputeThreads + 32, ks.smem, stream, pdl, plan, bitmap, span_cnt, tile_cnt, tile_off, nsub,
                     ks.stages, ks.stage_bytes, dense_mode, ctrl);
}

// Exact signed min / max of every block of an encoded INT column (imm3_open).
cudaError_t launch_block_stats(const PforCol& pc, const uint64_t* row_start, long long nblocks, int64_t max_block_words, int num_sms, BlockStat* stats,
                               cudaStream_t stream) {
    const int words_cap = block_words_cap(max_block_words);
    const size_t smem = (size_t)kComputeWarps * (size_t)(words_cap + kBlkVals) * 4;
    int occ = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, block_stats_kernel, kComputeThreads, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) return cudaErrorInvalidConfiguration;
    const long long grid = std::max<long long>(1, std::min<long long>((nblocks + kComputeWarps - 1) / kComputeWarps, (long long)num_sms * occ));
    block_stats_kernel<<<(unsigned)grid, kComputeThreads, smem, stream>>>(pc, row_start, nblocks, words_cap, stats);
    return cudaGetLastError();
}
cudaError_t launch_blocks_prune(const PrunePlan& q, const uint64_t* row_start, long long nblocks, long long ntiles8, uint32_t* blk_cnt,
                                uint32_t* tile_cnt, unsigned int* work, int num_sms, cudaStream_t stream, uint32_t* grp_sum) {
    const long long groups = (nblocks + 31) / 32;
    const long long grid = std::max<long long>(1, std::min<long long>((groups + kComputeWarps - 1) / kComputeWarps, (long long)num_sms * 8));
    blocks_prune_kernel<<<(unsigned)grid, kComputeThreads, 0, stream>>>(q, row_start, nblocks, ntiles8, blk_cnt, tile_cnt, work, grp_sum);
    return cudaGetLastError();
}

cudaError_t launch_blocks_or_merge(const uint64_t* row_start, long long nblocks, long long ntiles8, uint32_t* acc_words, uint32_t* acc_cnt,
                                   const uint32_t* term_words, const uint32_t* term_cnt, uint32_t* tile_cnt, ScanCtrl* ctrl, int num_sms,
                                   cudaStream_t stream) {
    const long long groups = (nblocks + 31) / 32;
    const long long grid = std::max<long long>(1, std::min<long long>((groups + kComputeWarps - 1) / kComputeWarps, (long long)num_sms * 8));
    blocks_or_merge_kernel<<<(unsigned)grid, kComputeThreads, 0, stream>>>(row_start, nblocks, ntiles8, acc_words, acc_cnt, term_words, term_cnt,
                                                                           tile_cnt, ctrl);
    return cudaGetLastError();
}

// count / min / max / sum ... group by: empty table -> (filter front, launched by the caller) -> agg_kernel or
// agg_blocks_kernel -> compaction.  The instantiation: exact for <= 2 group-by columns and 1 .. 4 aggregates, the general
// forms beyond; a plan with a SUM takes the SUM instantiations (it carries a COUNT too: 2 .. 4 aggregates exact, else 8).
AggShape agg_shape(const AggPlan& a, bool blocks, bool bsel) {
    AggShape s;
    s.ng = a.ngroup <= 2 ? a.ngroup : 4;
    s.na = (a.naggs >= 1 && a.naggs <= 4) ? a.naggs : 8;
    s.nsum = 0;
    for (int i = 0; i < a.naggs && i < kMaxAggs; i++) s.nsum += a.agg[i].op == kAggSum;
    if (s.nsum > 0 && s.na < 2) s.na = 2;
    s.blocks = blocks;
    s.bsel = blocks && bsel;
    return s;
}
std::string agg_route(const AggShape& s) {
    return std::string(s.blocks ? "agg_blocks<" : "agg<") + std::to_string(s.ng) + "," + std::to_string(s.na) + ">" + (s.nsum > 0 ? "/sum" : "") +
           (s.bsel ? "/bsel" : "");
}
cudaError_t launch_agg_init(AggEntry* table, uint32_t slots, const AggPlan& a, unsigned int* counters, cudaStream_t stream) {
    AggOps ops;
    for (int i = 0; i < kMaxAggs; i++) ops.op[i] = i < a.naggs ? (a.agg[i].op == kAggSum ? kAggCount : a.agg[i].op) : 0;  // (a SUM starts at 0, as a COUNT)
    ops.naggs = a.naggs;
    agg_init_kernel<<<(slots + kComputeThreads - 1) / kComputeThreads, kComputeThreads, 0, stream>>>(table, slots, ops, counters);
    return cudaGetLastError();
}
static size_t agg_blocks_smem_bytes(const AggShape& s, int npfor, int words_cap) {
    return agg_blocks_state_bytes(s.na, s.nsum) + (size_t)kComputeWarps * (size_t)agg_blocks_warp_words(npfor, words_cap) * 4;
}
size_t size_agg_blocks(AggPlan* ap, const AggShape& s, int64_t max_block_words) {
    ap->blk_words_cap = block_words_cap(max_block_words);
    return agg_blocks_smem_bytes(s, ap->npfor, ap->blk_words_cap) + 1024;  // (1 KB: the kernel's static shared memory)
}
// The kernel of a shape.  These switches instantiate every aggregation kernel of the library: agg_kernel<NG, NA, S> and
// agg_blocks_kernel<NG, NA, S, BS> for NG in {0, 1, 2, 4}, NA in {1, 2, 3, 4, 8} (S = false) or {2, 3, 4, 8} (S = true).
using AggKernel = void (*)(AggPlan, const uint32_t*, const uint32_t*, AggEntry*, unsigned int*, const ScanCtrl*);
template <int NG, int NA, bool S>
static AggKernel agg_kernel_of(const AggShape& s) {
    if (!s.blocks) return agg_kernel<NG, NA, S>;
    return s.bsel ? agg_blocks_kernel<NG, NA, S, true> : agg_blocks_kernel<NG, NA, S, false>;
}
template <int NG>
static AggKernel agg_kernel_of(const AggShape& s) {
    if (s.nsum > 0) return s.na == 2 ? agg_kernel_of<NG, 2, true>(s) : s.na == 3 ? agg_kernel_of<NG, 3, true>(s) : s.na == 4 ? agg_kernel_of<NG, 4, true>(s) : agg_kernel_of<NG, 8, true>(s);
    return s.na == 1 ? agg_kernel_of<NG, 1, false>(s) : s.na == 2 ? agg_kernel_of<NG, 2, false>(s) : s.na == 3 ? agg_kernel_of<NG, 3, false>(s)
         : s.na == 4 ? agg_kernel_of<NG, 4, false>(s) : agg_kernel_of<NG, 8, false>(s);
}
cudaError_t launch_agg(const AggPlan& a, const AggShape& s, const uint32_t* bitmap, const uint32_t* span_cnt, AggEntry* table, unsigned int* counters,
                       const ScanCtrl* ctrl, int num_sms, cudaStream_t stream) {
    const AggKernel kern = s.ng == 0 ? agg_kernel_of<0>(s) : s.ng == 1 ? agg_kernel_of<1>(s) : s.ng == 2 ? agg_kernel_of<2>(s) : agg_kernel_of<4>(s);
    const size_t smem = s.blocks ? agg_blocks_smem_bytes(s, a.npfor, a.blk_words_cap) : agg_smem_bytes(s.na, s.nsum);
    cudaError_t e = cudaSuccess;
    // (a per-device attribute, set per launch: one driver call per aggregation query)
    if (smem > 48 * 1024 && (e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kComputeThreads, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) return cudaErrorInvalidConfiguration;
    const long long units = s.blocks ? a.nblocks : a.ntiles * 8;  // one warp per block, or per 1024-row span
    const long long grid = std::max<long long>(1, std::min<long long>((units + kComputeWarps - 1) / kComputeWarps, (long long)num_sms * occ));
    kern<<<(unsigned)grid, kComputeThreads, smem, stream>>>(a, bitmap, span_cnt, table, counters + 1, ctrl);
    return cudaGetLastError();
}
cudaError_t launch_agg_compact(const AggEntry* table, uint32_t slots, AggEntry* out, unsigned int* counters, cudaStream_t stream) {
    agg_compact_kernel<<<(slots + kComputeThreads - 1) / kComputeThreads, kComputeThreads, 0, stream>>>(table, slots, out, counters);
    return cudaGetLastError();
}

// Global aggregate: every rank's partial groups (exchange buffers) -> the freshly initialised table (compaction follows).
cudaError_t launch_agg_merge(const AggMergePlan& m, const AggXOut* x, AggEntry* table, unsigned int* counters, int num_sms, cudaStream_t stream) {
    agg_merge_kernel<<<(unsigned)std::max(1, num_sms), kComputeThreads, 0, stream>>>(m, x, table, counters + 1);
    return cudaGetLastError();
}

cudaError_t launch_offset_scan(const uint32_t* tile_cnt, unsigned long long* tile_off, long long ntiles, long long limit, uint32_t epoch,
                               unsigned long long* partials, ScanCtrl* ctrl, unsigned int* tile_list, cudaStream_t stream) {
    return launch_ex(offset_scan_kernel, (int)((ntiles + kComputeThreads * 16 - 1) / (kComputeThreads * 16)), kComputeThreads, 0, stream, true,
                     tile_cnt, tile_off, ntiles, limit, epoch, partials, ctrl, tile_list);
}

// The emit kernels of one projected encoded column read the LeanPlan: the parts of the ScanPlan they use.
static LeanPlan lean_plan(const ScanPlan& plan) {
    LeanPlan lp;
    const int slot = plan.proj[0].pfor_slot;
    lp.row_start = plan.row_start;
    lp.words = plan.pfor[slot].words;
    lp.word_off = plan.pfor[slot].word_off;
    lp.out = plan.proj[0].out;
    lp.limit = plan.limit;
    lp.ntiles = plan.ntiles;
    lp.trace = plan.trace;
    lp.debug = plan.debug;
    lp.pad = 0;
    return lp;
}

// Offset scan + emit in one kernel (one encoded column projected): a persistent grid of small CTAs, at least one per scan chunk.
cudaError_t blocks_scan_emit_grid(int num_sms, long long ntiles8, int* grid) {
    int occ = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, blocks_scan_emit_kernel, kComputeThreads, 0);
    if (e != cudaSuccess) return e;
    const long long nchunks = (ntiles8 + kComputeThreads * 16 - 1) / (kComputeThreads * 16);
    const long long g = (long long)num_sms * occ;
    *grid = (occ >= 1 && nchunks <= g) ? (int)g : 0;  // 0: does not apply (every chunk CTA has to be resident)
    return cudaSuccess;
}
cudaError_t launch_blocks_scan_emit(const ScanPlan& plan, const uint32_t* bitmapB, const uint32_t* blk_cnt, const uint32_t* tile_cnt,
                                    unsigned long long* tile_off, long long nblocks, uint32_t epoch, unsigned long long* partials, ScanCtrl* ctrl,
                                    unsigned int* tile_list, bool pdl, int grid, cudaStream_t stream, CtrlBlock* pub, unsigned long long pub_seq) {
    return launch_ex(blocks_scan_emit_kernel, grid, kComputeThreads, 0, stream, pdl, lean_plan(plan), bitmapB, blk_cnt, tile_cnt, tile_off, nblocks,
                     epoch, partials, ctrl, tile_list, pub, pub_seq);
}

// Emit without an offset scan (k_blocks_groupemit.cuh): a persistent grid of small CTAs next to the filter kernel.
cudaError_t blocks_group_emit_grid(int num_sms, long long nblocks, int* grid, size_t* sum_bytes) {
    int occ = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, blocks_group_emit_kernel, kComputeThreads, 0);
    if (e != cudaSuccess) return e;
    const long long ng = (nblocks + (1ll << kGrpShift) - 1) >> kGrpShift;
    if (const char* e = getenv("IMM3_GE_CTAS")) occ = std::max(1, std::min(occ, atoi(e)));  // experiment: CTAs per SM
    *grid = (occ >= 1 && ng <= kGrpMaxGroups) ? num_sms * occ : 0;  // 0: does not apply
    *sum_bytes = (size_t)kGrpSumWords * 4;
    return cudaSuccess;
}
cudaError_t launch_blocks_group_emit(const ScanPlan& plan, const uint32_t* bitmapB, const uint32_t* blk_cnt, uint32_t* grp_sum, long long nblocks,
                                     ScanCtrl* ctrl, bool pdl, int grid, cudaStream_t stream, CtrlBlock* pub, unsigned long long pub_seq) {
    const int ngroups = (int)std::min<long long>((nblocks + (1ll << kGrpShift) - 1) >> kGrpShift, kGrpMaxGroups);
    return launch_ex(blocks_group_emit_kernel, grid, kComputeThreads, 0, stream, pdl, lean_plan(plan), bitmapB, blk_cnt, grp_sum, nblocks, ngroups,
                     ctrl, pub, pub_seq);
}

// The quad and lane kernels stage CTA tiles of 32 blocks of their one column: a ring slot holds such a tile (padded) behind
// its header.
static int quad_slot_bytes(int64_t max_tile32_bytes, int* tile_cap) {
    *tile_cap = (int)((max_tile32_bytes + 16 + 15) & ~15ll);
    return kQuadHdrBytes + *tile_cap;
}
// Quad kernel (lane = (block, super-block), CTA tile of 32 blocks) if such a tile of this column fits a ring slot (i.e. the
// column actually compresses); its lane = block successor if a CTA of 8 warps holds a two-slot ring per warp (unless
// IMM3_NO_LANE).  Otherwise the mini-block kernel.
BlockFilter single_range_block_filter(int64_t max_tile32_bytes) {
    int cap = 0;
    const int qslot = quad_slot_bytes(max_tile32_bytes, &cap);
    if (qslot > 40 * 1024) return BlockFilter::kMini;
    return (2 * 8 * (size_t)qslot <= kLaneSmemCap && !getenv("IMM3_NO_LANE")) ? BlockFilter::kLane : BlockFilter::kQuad;
}
// Mini-block kernel: a TMA ring of raw tiles (8 blocks of every encoded column that carries a predicate + metadata).  Quad
// kernel: tiles of 32 blocks of its one column.  Lane kernel: every warp of the CTA runs its own ring of 2 .. 4 such slots;
// one CTA per SM with as many warps (8 .. 16) as its shared memory holds two-slot rings for.
cudaError_t size_block_filter(BlockFilter f, ScanPlan* sp, int64_t max_tile_bytes, int64_t max_tile32_bytes, KernelShape* ks) {
    const char* ring_env = getenv("IMM3_BLOCKS_STAGES");
    if (f == BlockFilter::kMini) {
        sp->blk_tile_bytes = (int)((max_tile_bytes + 16 + 15) & ~15ll);
        const int slot_bytes = blk_filter_slot_bytes(__builtin_popcount(sp->pfor_filter_mask), sp->blk_tile_bytes);
        int ring = std::max(2, std::min(kMaxFilterStages, (48 * 1024) / slot_bytes));
        if (ring_env) ring = std::max(2, std::min(kMaxFilterStages, atoi(ring_env)));
        while (ring > 2 && (size_t)ring * slot_bytes > kSmemCap) ring--;
        sp->stages = ring;
        sp->stage_bytes = slot_bytes;
        ks->smem = (size_t)ring * (size_t)slot_bytes;
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ks->occupancy, blocks_filter_kernel, kComputeThreads + 32, ks->smem);
    }
    const int qslot = quad_slot_bytes(max_tile32_bytes, &sp->blk_tile_bytes);
    sp->stage_bytes = qslot;
    if (f == BlockFilter::kQuad) {
        int qring = std::max(2, std::min(4, (40 * 1024) / qslot));
        if (ring_env) qring = std::max(2, std::min(kMaxFilterStages, atoi(ring_env)));
        sp->stages = qring;
        ks->smem = (size_t)qring * (size_t)qslot;
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ks->occupancy, blocks_filter_quad_kernel, kComputeThreads + 32, ks->smem);
    }
    int lring = 2;
    if (const char* e = getenv("IMM3_LANE_STAGES")) lring = std::max(2, std::min(4, atoi(e)));
    while (lring > 2 && (size_t)lring * 4 * (size_t)qslot > kLaneSmemCap) lring--;
    int lw = (int)std::min<size_t>(16, kLaneSmemCap / ((size_t)lring * (size_t)qslot));
    if (const char* e = getenv("IMM3_LANE_WARPS")) lw = std::max(4, std::min(lw, atoi(e)));
    ks->lane_warps = lw;
    sp->stages = lring;
    ks->smem = (size_t)lring * (size_t)lw * (size_t)qslot;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ks->occupancy, blocks_filter_lane_kernel, lw * 32, ks->smem);
}
cudaError_t launch_blocks_filter(const ScanPlan& plan, uint32_t* bitmapB, uint32_t* blk_cnt, uint32_t* tile_cnt, unsigned long long* tile_off,
                                 ScanCtrl* ctrl, long long nblocks, int grid, BlockFilter filter, const KernelShape& ks, const unsigned int* work,
                                 uint32_t* grp_sum, cudaStream_t stream, std::string* route) {
    if (filter != BlockFilter::kMini) {  // CTA tiles of 32 blocks (quad), 32 blocks per warp (lane)
        const long long per_cta = 32 * (filter == BlockFilter::kLane ? ks.lane_warps : 1);
        grid = (int)std::max<long long>(1, std::min<long long>(grid, (nblocks + per_cta - 1) / per_cta));
    }
    if (filter == BlockFilter::kLane) {
        blocks_filter_lane_kernel<<<grid, ks.lane_warps * 32, ks.smem, stream>>>(plan, bitmapB, blk_cnt, tile_cnt, tile_off, ctrl, nblocks, work, grp_sum);
        *route = "blocks_filter_lane/w=" + std::to_string(ks.lane_warps) + "/s=" + std::to_string(plan.stages);
    } else if (filter == BlockFilter::kQuad) {
        blocks_filter_quad_kernel<<<grid, kComputeThreads + 32, ks.smem, stream>>>(plan, bitmapB, blk_cnt, tile_cnt, tile_off, ctrl, nblocks, work);
        *route = with_stages("blocks_filter_quad", plan.stages);
    } else {
        blocks_filter_kernel<<<grid, kComputeThreads + 32, ks.smem, stream>>>(plan, bitmapB, blk_cnt, tile_cnt, tile_off, ctrl, nblocks, work);
        *route = with_stages("blocks_filter", plan.stages);
    }
    return cudaGetLastError();
}

// Block emit kernel: one warp per block, every warp with its own decode scratch.
cudaError_t size_blocks_emit(ScanPlan* sp, bool rowspace, int64_t max_block_words, long long nblocks, int num_sms, KernelShape* ks) {
    sp->blk_words_cap = block_words_cap(max_block_words);
    ks->smem = (size_t)kComputeWarps * blk_emit_warp_words(sp->npfor, sp->blk_words_cap) * 4;
    cudaError_t e = rowspace ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ks->occupancy, blocks_emit_kernel<true>, kComputeThreads, ks->smem)
                             : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ks->occupancy, blocks_emit_kernel<false>, kComputeThreads, ks->smem);
    ks->grid = (int)std::max<int64_t>(1, std::min<int64_t>((nblocks + 7) / 8, (int64_t)num_sms * std::max(1, ks->occupancy)));
    return e;
}
cudaError_t launch_blocks_emit(const ScanPlan& plan, const uint32_t* bitmap, const uint32_t* cnts, const unsigned int* tile_list, const unsigned long long* tile_off,
                               long long nblocks, const ScanCtrl* ctrl, bool rowspace, bool pdl, const KernelShape& ks, cudaStream_t stream) {
    const int grid = (int)std::min<long long>(ks.grid, (nblocks + 7) / 8);
    if (rowspace) return launch_ex(blocks_emit_kernel<true>, grid, kComputeThreads, ks.smem, stream, pdl, plan, bitmap, cnts, tile_list, tile_off, nblocks, ctrl);
    return launch_ex(blocks_emit_kernel<false>, grid, kComputeThreads, ks.smem, stream, pdl, plan, bitmap, cnts, tile_list, tile_off, nblocks, ctrl);
}

// The count exchange rides behind the query's last kernel as a programmatic dependent (its launch overlaps that kernel).
cudaError_t launch_count_exchange(const CommPlan& plan, const ScanCtrl* ctrl, CommOut* out, cudaStream_t stream) {
    return launch_ex(count_exchange_kernel, 1, 32, 0, stream, true, plan, ctrl, out);
}
// ... and so does the exchange of a global aggregate (behind the compaction of the local groups).
cudaError_t launch_agg_exchange(const AggXPlan& plan, const unsigned int* counters, const ScanCtrl* ctrl, AggXOut* out, cudaStream_t stream) {
    return launch_ex(agg_exchange_kernel, 1, 32, 0, stream, true, plan, counters, ctrl, out);
}

// scan_blocks stages whole blocks.
cudaError_t size_scan_blocks(const ScanPlan& sp, int max_block_rows, KernelShape* ks) {
    const size_t maxb = (size_t)((max_block_rows + 31) & ~31), nmb = maxb / 32;
    const size_t words = (size_t)sp.npfor * maxb + (sp.npfor > 0 ? maxb + nmb + 64 : 0) + nmb + (nmb + 1) + nmb + nmb;
    ks->smem = words * 4 + nmb * 2 + nmb + 64;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ks->occupancy, scan_blocks_kernel, kBlockThreads, ks->smem);
}
cudaError_t launch_scan_blocks(const ScanPlan& plan, ScanCtrl* ctrl, unsigned long long* status, int grid, size_t dyn_smem,
                               cudaStream_t stream) {
    scan_blocks_kernel<<<grid, kBlockThreads, dyn_smem, stream>>>(plan, ctrl, status);
    return cudaGetLastError();
}

}  // namespace imm3
