// kernels.cu - sm_100a kernels of the scan -> filter -> project path (one translation unit; the device code lives in the
// k_*.cuh fragments included below, this file holds the launchers).
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
#include <mutex>

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
size_t blocks_kernel_smem_bytes(int npfor, int max_block_rows) {
    const size_t maxb = (size_t)((max_block_rows + 31) & ~31), nmb = maxb / 32;
    size_t words = (size_t)npfor * maxb + (npfor > 0 ? maxb + nmb + 64 : 0) + nmb + (nmb + 1) + nmb + nmb;
    return words * 4 + nmb * 2 + nmb + 64;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute: one process may hold handles on several GPUs
// (one GpuEngine per GPU, INTEGRATION.md), so the kernels are configured once per device ordinal, for the device that is
// current on the calling thread (every entry point of engine.cu has called cudaSetDevice(db->device) by now).
static cudaError_t configure_device();
static cudaError_t configure_once() {
    static std::mutex mu;
    static bool done[64] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    if (dev >= 0 && dev < 64 && done[dev]) return cudaSuccess;
    e = configure_device();
    if (e == cudaSuccess && dev >= 0 && dev < 64) done[dev] = true;
    return e;
}
static cudaError_t configure_device() {
    {
        cudaError_t e = cudaSuccess;
#define IMM3_SET_SMEM(K) if ((e = cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)) != cudaSuccess) return e
        IMM3_SET_SMEM(emit_stream_kernel);
        IMM3_SET_SMEM(blocks_filter_kernel);
        IMM3_SET_SMEM(blocks_filter_quad_kernel);
        if ((e = cudaFuncSetAttribute(blocks_filter_lane_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 222 * 1024)) != cudaSuccess) return e;
        IMM3_SET_SMEM(block_stats_kernel);
        IMM3_SET_SMEM(blocks_emit_kernel<true>);
        IMM3_SET_SMEM(blocks_emit_kernel<false>);
        IMM3_SET_SMEM(emit_general_kernel);
        IMM3_SET_SMEM(filter_kernel<true>);
        IMM3_SET_SMEM(filter_kernel<false>);
#undef IMM3_SET_SMEM
        return cudaFuncSetAttribute(scan_blocks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    }
}

cudaError_t blocks_kernel_occupancy(size_t dyn_smem, int* blocks_per_sm) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, scan_blocks_kernel, kBlockThreads, dyn_smem);
}

cudaError_t filter_kernel_occupancy(size_t dyn_smem, int* blocks_per_sm) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    if (dyn_smem > 0) return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, filter_kernel<true>, kComputeThreads + 32, dyn_smem);
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, filter_kernel<false>, kComputeThreads + 32, dyn_smem);
}
cudaError_t emit_kernel_occupancy(bool general, int* blocks_per_sm) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    if (general) return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, emit_general_kernel, kComputeThreads, kComputeWarps * 1024 * 2);
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, emit_kernel, kComputeThreads, kComputeWarps * kEmitWarpSmemBytes);
}
cudaError_t launch_filter(const ScanPlan& plan, uint32_t* bitmap, uint32_t* span_cnt, uint32_t* tile_cnt, unsigned long long* tile_off,
                          ScanCtrl* ctrl, int grid, size_t dyn_smem, cudaStream_t stream) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    if (plan.nfilter == 0) {  // no predicate: nothing to read - the selection metadata is written analytically
        select_all_kernel<<<grid, kComputeThreads, 0, stream>>>(plan, bitmap, span_cnt, tile_cnt, tile_off, ctrl);
        return cudaGetLastError();
    }
    if (plan.stages > 0) filter_kernel<true><<<grid, kComputeThreads + 32, dyn_smem, stream>>>(plan, bitmap, span_cnt, tile_cnt, tile_off, ctrl);
    else filter_kernel<false><<<grid, kComputeThreads + 32, dyn_smem, stream>>>(plan, bitmap, span_cnt, tile_cnt, tile_off, ctrl);
    return cudaGetLastError();
}
cudaError_t launch_emit(const ScanPlan& plan, const uint32_t* bitmap, const uint32_t* span_cnt, const unsigned long long* tile_off,
                        int spans_per_tile, long long nspans, int grid, int dense_off, const ScanCtrl* ctrl, bool general, bool pdl,
                        cudaStream_t stream) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kComputeThreads);
    cfg.dynamicSmemBytes = kComputeWarps * kEmitWarpSmemBytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (general) {
        cfg.dynamicSmemBytes = kComputeWarps * 1024 * 2;
        return cudaLaunchKernelEx(&cfg, emit_general_kernel, plan, bitmap, span_cnt, tile_off, spans_per_tile, nspans, dense_off, ctrl);
    }
    return cudaLaunchKernelEx(&cfg, emit_kernel, plan, bitmap, span_cnt, tile_off, spans_per_tile, nspans, dense_off, ctrl);
}
size_t emit_stream_smem_bytes(int stage_bytes, int ring) { return (size_t)kComputeWarps * 1024 * 2 + (size_t)ring * (size_t)stage_bytes + 16; }
int emit_stream_header_bytes() { return kEmitHdrBytes; }
cudaError_t emit_stream_occupancy(size_t dyn_smem, int* blocks_per_sm) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, emit_stream_kernel, kComputeThreads + 32, dyn_smem);
}
cudaError_t launch_emit_stream(const ScanPlan& plan, const uint32_t* bitmap, const uint32_t* span_cnt, const uint32_t* tile_cnt,
                               const unsigned long long* tile_off, long long nsub, int ring, int stage_bytes, int dense_mode, int grid,
                               size_t dyn_smem, ScanCtrl* ctrl, bool pdl, cudaStream_t stream) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kComputeThreads + 32);
    cfg.dynamicSmemBytes = dyn_smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, emit_stream_kernel, plan, bitmap, span_cnt, tile_cnt, tile_off, nsub, ring, stage_bytes, dense_mode, ctrl);
}

// Exact signed min / max of every block of an encoded INT column (imm3_open).
cudaError_t launch_block_stats(const PforCol& pc, const uint64_t* row_start, long long nblocks, int words_cap, int num_sms, BlockStat* stats,
                               cudaStream_t stream) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    const size_t smem = (size_t)kComputeWarps * (size_t)(words_cap + kBlkVals) * 4;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, block_stats_kernel, kComputeThreads, smem);
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
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    AggOps ops;
    for (int i = 0; i < kMaxAggs; i++) ops.op[i] = i < a.naggs ? (a.agg[i].op == kAggSum ? kAggCount : a.agg[i].op) : 0;  // (a SUM starts at 0, as a COUNT)
    ops.naggs = a.naggs;
    agg_init_kernel<<<(slots + kComputeThreads - 1) / kComputeThreads, kComputeThreads, 0, stream>>>(table, slots, ops, counters);
    return cudaGetLastError();
}
size_t agg_blocks_smem_bytes(const AggShape& s, int npfor, int words_cap) {
    return agg_blocks_state_bytes(s.na, s.nsum) + (size_t)kComputeWarps * (size_t)agg_blocks_warp_words(npfor, words_cap) * 4;
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
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    const AggKernel kern = s.ng == 0 ? agg_kernel_of<0>(s) : s.ng == 1 ? agg_kernel_of<1>(s) : s.ng == 2 ? agg_kernel_of<2>(s) : agg_kernel_of<4>(s);
    const size_t smem = s.blocks ? agg_blocks_smem_bytes(s, a.npfor, a.blk_words_cap) : agg_smem_bytes(s.na, s.nsum);
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
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    agg_merge_kernel<<<(unsigned)std::max(1, num_sms), kComputeThreads, 0, stream>>>(m, x, table, counters + 1);
    return cudaGetLastError();
}

long long scan_inline_max_tiles() { return kScanInlineMaxTiles; }
cudaError_t launch_offset_scan(const uint32_t* tile_cnt, unsigned long long* tile_off, long long ntiles, long long limit, uint32_t epoch,
                               unsigned long long* partials, ScanCtrl* ctrl, unsigned int* tile_list, cudaStream_t stream) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((ntiles + kComputeThreads * 16 - 1) / (kComputeThreads * 16)));
    cfg.blockDim = dim3(kComputeThreads);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, offset_scan_kernel, tile_cnt, tile_off, ntiles, limit, epoch, partials, ctrl, tile_list);
}

// Offset scan + emit in one kernel (one encoded column projected): a persistent grid of small CTAs, at least one per scan chunk.
cudaError_t blocks_scan_emit_grid(int num_sms, long long ntiles8, int* grid) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, blocks_scan_emit_kernel, kComputeThreads, 0);
    if (e != cudaSuccess) return e;
    const long long nchunks = (ntiles8 + kComputeThreads * 16 - 1) / (kComputeThreads * 16);
    const long long g = (long long)num_sms * occ;
    *grid = (occ >= 1 && nchunks <= g) ? (int)g : 0;  // 0: does not apply (every chunk CTA has to be resident)
    return cudaSuccess;
}
cudaError_t launch_blocks_scan_emit(const ScanPlan& plan, const uint32_t* bitmapB, const uint32_t* blk_cnt, const uint32_t* tile_cnt,
                                    unsigned long long* tile_off, long long nblocks, uint32_t epoch, unsigned long long* partials, ScanCtrl* ctrl,
                                    unsigned int* tile_list, bool pdl, int grid, cudaStream_t stream, CtrlBlock* pub, unsigned long long pub_seq) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kComputeThreads);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
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
    return cudaLaunchKernelEx(&cfg, blocks_scan_emit_kernel, lp, bitmapB, blk_cnt, tile_cnt, tile_off, nblocks, epoch, partials, ctrl, tile_list, pub, pub_seq);
}

// Emit without an offset scan (k_blocks_groupemit.cuh): a persistent grid of small CTAs next to the filter kernel.
int blocks_group_emit_max_groups() { return kGrpMaxGroups; }
size_t blocks_group_sum_bytes() { return (size_t)kGrpSumWords * 4; }
cudaError_t blocks_group_emit_grid(int num_sms, long long nblocks, int* grid, int* ngroups) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, blocks_group_emit_kernel, kComputeThreads, 0);
    if (e != cudaSuccess) return e;
    const long long ng = (nblocks + (1ll << kGrpShift) - 1) >> kGrpShift;
    *ngroups = (int)std::min<long long>(ng, kGrpMaxGroups);
    if (const char* e = getenv("IMM3_GE_CTAS")) occ = std::max(1, std::min(occ, atoi(e)));  // experiment: CTAs per SM
    *grid = (occ >= 1 && ng <= kGrpMaxGroups) ? num_sms * occ : 0;  // 0: does not apply
    return cudaSuccess;
}
cudaError_t launch_blocks_group_emit(const ScanPlan& plan, const uint32_t* bitmapB, const uint32_t* blk_cnt, uint32_t* grp_sum, long long nblocks,
                                     int ngroups, ScanCtrl* ctrl, bool pdl, int grid, cudaStream_t stream, CtrlBlock* pub, unsigned long long pub_seq) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kComputeThreads);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
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
    return cudaLaunchKernelEx(&cfg, blocks_group_emit_kernel, lp, bitmapB, blk_cnt, grp_sum, nblocks, ngroups, ctrl, pub, pub_seq);
}

size_t blocks_filter_smem_bytes(int nstaged, int tile_cap_bytes, int ring) { return (size_t)ring * (size_t)blk_filter_slot_bytes(nstaged, tile_cap_bytes); }
int blocks_filter_slot_bytes(int nstaged, int tile_cap_bytes) { return blk_filter_slot_bytes(nstaged, tile_cap_bytes); }
size_t blocks_emit_smem_bytes(int npfor, int words_cap) { return (size_t)kComputeWarps * blk_emit_warp_words(npfor, words_cap) * 4; }
int blocks_filter_quad_slot_bytes(int tile_cap_bytes) { return kQuadHdrBytes + tile_cap_bytes; }
cudaError_t blocks_filter_occupancy(size_t filter_smem, BlockFilter filter, int lane_warps, int* blocks_per_sm) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    return filter == BlockFilter::kLane   ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, blocks_filter_lane_kernel, lane_warps * 32, filter_smem)
           : filter == BlockFilter::kQuad ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, blocks_filter_quad_kernel, kComputeThreads + 32, filter_smem)
                                          : cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, blocks_filter_kernel, kComputeThreads + 32, filter_smem);
}
cudaError_t blocks_emit_occupancy(size_t emit_smem, bool rowspace, int* blocks_per_sm) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    if (rowspace) return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, blocks_emit_kernel<true>, kComputeThreads, emit_smem);
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, blocks_emit_kernel<false>, kComputeThreads, emit_smem);
}
cudaError_t launch_blocks_filter(const ScanPlan& plan, uint32_t* bitmapB, uint32_t* blk_cnt, uint32_t* tile_cnt, unsigned long long* tile_off,
                                 ScanCtrl* ctrl, long long nblocks, int grid, size_t dyn_smem, BlockFilter filter, int lane_warps,
                                 const unsigned int* work, cudaStream_t stream, uint32_t* grp_sum) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    if (filter == BlockFilter::kLane) blocks_filter_lane_kernel<<<grid, lane_warps * 32, dyn_smem, stream>>>(plan, bitmapB, blk_cnt, tile_cnt, tile_off, ctrl, nblocks, work, grp_sum);
    else if (filter == BlockFilter::kQuad) blocks_filter_quad_kernel<<<grid, kComputeThreads + 32, dyn_smem, stream>>>(plan, bitmapB, blk_cnt, tile_cnt, tile_off, ctrl, nblocks, work);
    else blocks_filter_kernel<<<grid, kComputeThreads + 32, dyn_smem, stream>>>(plan, bitmapB, blk_cnt, tile_cnt, tile_off, ctrl, nblocks, work);
    return cudaGetLastError();
}
cudaError_t launch_blocks_emit(const ScanPlan& plan, const uint32_t* bitmap, const uint32_t* cnts, const unsigned int* tile_list, const unsigned long long* tile_off,
                               long long nblocks, const ScanCtrl* ctrl, bool rowspace, bool pdl, int grid, size_t dyn_smem, cudaStream_t stream) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kComputeThreads);
    cfg.dynamicSmemBytes = dyn_smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const long long nb = nblocks;
    if (rowspace) return cudaLaunchKernelEx(&cfg, blocks_emit_kernel<true>, plan, bitmap, cnts, tile_list, tile_off, nb, ctrl);
    return cudaLaunchKernelEx(&cfg, blocks_emit_kernel<false>, plan, bitmap, cnts, tile_list, tile_off, nb, ctrl);
}

// The count exchange rides behind the query's last kernel as a programmatic dependent (its launch overlaps that kernel).
cudaError_t launch_count_exchange(const CommPlan& plan, const ScanCtrl* ctrl, CommOut* out, cudaStream_t stream) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(1);
    cfg.blockDim = dim3(32);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, count_exchange_kernel, plan, ctrl, out);
}
// ... and so does the exchange of a global aggregate (behind the compaction of the local groups).
cudaError_t launch_agg_exchange(const AggXPlan& plan, const unsigned int* counters, const ScanCtrl* ctrl, AggXOut* out, cudaStream_t stream) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(1);
    cfg.blockDim = dim3(32);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, agg_exchange_kernel, plan, counters, ctrl, out);
}

cudaError_t launch_scan_blocks(const ScanPlan& plan, ScanCtrl* ctrl, unsigned long long* status, int grid, size_t dyn_smem,
                               cudaStream_t stream) {
    cudaError_t e = configure_once();
    if (e != cudaSuccess) return e;
    scan_blocks_kernel<<<grid, kBlockThreads, dyn_smem, stream>>>(plan, ctrl, status);
    return cudaGetLastError();
}

}  // namespace imm3
