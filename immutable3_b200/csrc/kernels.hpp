// kernels.hpp — host-callable launchers of kernels.cu, and the sizing rules that shape their launches.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <string>

#include "plan.hpp"

namespace imm3 {

// The opt-in dynamic shared memory of the kernels that take more than 48 KB, on the calling thread's current device (a
// per-device attribute: imm3_open runs it for its device before the first launch).
cudaError_t configure_device();

// One kernel's launch as its sizing rule decided it.  A rule that stages through a TMA ring writes that ring (stages,
// stage_bytes) into the device plan the kernel reads; the streaming emit kernel takes it as arguments, here.
struct KernelShape {
    size_t smem = 0;      // dynamic shared memory per CTA
    int occupancy = 0;    // CTAs per SM at that shared memory
    int grid = 0;         // CTAs
    int stages = 0, stage_bytes = 0;
    int lane_warps = 0;   // blocks_filter_lane_kernel: warps per CTA
};
// The dense pipeline's emit kernels: the gather kernel (emit_kernel, or emit_general_kernel when `general`) and the
// streaming one (stream.stage_bytes = 0: not usable).
struct EmitShape {
    bool general = false;
    int grid = 0;
    KernelShape stream;
};

// Row-space filter kernel: where each filter column sits in a TMA stage (sp->filter[].smem_off), its ring (sp->stages,
// sp->stage_bytes; no ring without TMA) and occupancy.
cudaError_t size_filter(ScanPlan* sp, bool no_tma, KernelShape* ks);
// The kernel that ran goes to *route, its name in Result.route ("select_all", "filter(tma)/s=4", "filter(direct)").
cudaError_t launch_filter(const ScanPlan& plan, uint32_t* bitmap, uint32_t* span_cnt, uint32_t* tile_cnt, unsigned long long* tile_off,
                          ScanCtrl* ctrl, int grid, size_t dyn_smem, cudaStream_t stream, std::string* route);
// Whether the filter kernel's last CTA turns `ntiles` tile counts into offsets (else offset_scan_kernel does).
bool scan_inline_for(long long ntiles);
// Gather and streaming emit kernels over sp->ntiles tiles: sp->proj[].stage_off and both kernels' shapes.
cudaError_t size_emit(ScanPlan* sp, bool no_tma, int num_sms, EmitShape* es);
cudaError_t launch_emit(const ScanPlan& plan, const uint32_t* bitmap, const uint32_t* span_cnt, const unsigned long long* tile_off,
                        int spans_per_tile, long long nspans, const EmitShape& es, int dense_off, const ScanCtrl* ctrl, bool pdl,
                        cudaStream_t stream);
cudaError_t launch_emit_stream(const ScanPlan& plan, const uint32_t* bitmap, const uint32_t* span_cnt, const uint32_t* tile_cnt,
                               const unsigned long long* tile_off, long long nsub, const KernelShape& ks, int dense_mode, ScanCtrl* ctrl,
                               bool pdl, cudaStream_t stream);
// The aggregation kernel's instantiation (agg_shape is the one place that chooses it): NG group-by columns, NA aggregates,
// nsum SUMs; blocks: agg_blocks_kernel, else agg_kernel; bsel: agg_blocks_kernel reads the block filter's selection (32
// words and one count per block), not the row-space filter's.
struct AggShape { int ng, na, nsum; bool blocks, bsel; };
AggShape agg_shape(const AggPlan& a, bool blocks, bool bsel);
std::string agg_route(const AggShape& s);  // its name in Result.route, e.g. "agg<1,2>", "agg_blocks<0,3>/sum/bsel"
// agg_blocks_kernel over encoded blocks of at most max_block_words words: sets ap->blk_words_cap and returns the shared
// memory (dynamic and static) one CTA needs.
size_t size_agg_blocks(AggPlan* ap, const AggShape& s, int64_t max_block_words);
cudaError_t launch_agg_init(AggEntry* table, uint32_t slots, const AggPlan& a, unsigned int* counters, cudaStream_t stream);
cudaError_t launch_agg(const AggPlan& a, const AggShape& s, const uint32_t* bitmap, const uint32_t* span_cnt, AggEntry* table, unsigned int* counters,
                       const ScanCtrl* ctrl, int num_sms, cudaStream_t stream);
cudaError_t launch_agg_compact(const AggEntry* table, uint32_t slots, AggEntry* out, unsigned int* counters, cudaStream_t stream);
cudaError_t launch_offset_scan(const uint32_t* tile_cnt, unsigned long long* tile_off, long long ntiles, long long limit, uint32_t epoch,
                               unsigned long long* partials, ScanCtrl* ctrl, unsigned int* tile_list, cudaStream_t stream);
cudaError_t blocks_scan_emit_grid(int num_sms, long long ntiles8, int* grid);
cudaError_t launch_blocks_scan_emit(const ScanPlan& plan, const uint32_t* bitmapB, const uint32_t* blk_cnt, const uint32_t* tile_cnt,
                                    unsigned long long* tile_off, long long nblocks, uint32_t epoch, unsigned long long* partials, ScanCtrl* ctrl,
                                    unsigned int* tile_list, bool pdl, int grid, cudaStream_t stream, CtrlBlock* pub = nullptr,
                                    unsigned long long pub_seq = 0);
// grid 0: does not apply; *sum_bytes: the size of the group-sum buffer it reads.
cudaError_t blocks_group_emit_grid(int num_sms, long long nblocks, int* grid, size_t* sum_bytes);
cudaError_t launch_blocks_group_emit(const ScanPlan& plan, const uint32_t* bitmapB, const uint32_t* blk_cnt, uint32_t* grp_sum, long long nblocks,
                                     ScanCtrl* ctrl, bool pdl, int grid, cudaStream_t stream, CtrlBlock* pub = nullptr,
                                     unsigned long long pub_seq = 0);
// The block filter kernels: lane = mini-block (blocks_filter_kernel), quad (blocks_filter_quad_kernel), lane = block
// (blocks_filter_lane_kernel, lane_warps warps per CTA).
enum class BlockFilter { kMini, kQuad, kLane };
// The kernel for a query whose only predicate is a range on one encoded column, from that column's largest tile of 32
// blocks: quad or lane if such a tile fits their ring slots, else mini-block.
BlockFilter single_range_block_filter(int64_t max_tile32_bytes);
// Ring (sp->blk_tile_bytes, sp->stages, sp->stage_bytes), lane warps and occupancy of block filter kernel `f`, from the
// largest tile of the encoded predicate columns: of 8 blocks (mini-block kernel), of 32 blocks (quad and lane kernels).
cudaError_t size_block_filter(BlockFilter f, ScanPlan* sp, int64_t max_tile_bytes, int64_t max_tile32_bytes, KernelShape* ks);
// grid: the persistent grid over the tiles, clamped to the quad and lane kernels' CTA tiles.  grp_sum: blocks_group_emit_kernel
// follows (lane kernel only).  The kernel that ran goes to *route ("blocks_filter/s=4", "blocks_filter_lane/w=16/s=2", ...).
cudaError_t launch_blocks_filter(const ScanPlan& plan, uint32_t* bitmapB, uint32_t* blk_cnt, uint32_t* tile_cnt, unsigned long long* tile_off,
                                 ScanCtrl* ctrl, long long nblocks, int grid, BlockFilter filter, const KernelShape& ks, const unsigned int* work,
                                 uint32_t* grp_sum, cudaStream_t stream, std::string* route);
cudaError_t launch_block_stats(const PforCol& pc, const uint64_t* row_start, long long nblocks, int64_t max_block_words, int num_sms, BlockStat* stats,
                               cudaStream_t stream);
cudaError_t launch_blocks_prune(const PrunePlan& q, const uint64_t* row_start, long long nblocks, long long ntiles8, uint32_t* blk_cnt,
                                uint32_t* tile_cnt, unsigned int* work, int num_sms, cudaStream_t stream, uint32_t* grp_sum = nullptr);
// Real OR over encoded columns: acc_* (the block filter's selection of the terms so far) |= term_* (the next term's), in the
// same contract - every block's count, the words of partial blocks only - and every 8-block tile count rewritten.
cudaError_t launch_blocks_or_merge(const uint64_t* row_start, long long nblocks, long long ntiles8, uint32_t* acc_words, uint32_t* acc_cnt,
                                   const uint32_t* term_words, const uint32_t* term_cnt, uint32_t* tile_cnt, ScanCtrl* ctrl, int num_sms,
                                   cudaStream_t stream);
// Block emit kernel over encoded blocks of at most max_block_words words (sp->blk_words_cap); occupancy < 1: it does not fit.
cudaError_t size_blocks_emit(ScanPlan* sp, bool rowspace, int64_t max_block_words, long long nblocks, int num_sms, KernelShape* ks);
// rowspace: the bitmap / counts come from the dense filter kernel (row space), not from blocks_filter_kernel (block-local)
cudaError_t launch_blocks_emit(const ScanPlan& plan, const uint32_t* bitmap, const uint32_t* cnts, const unsigned int* tile_list, const unsigned long long* tile_off,
                               long long nblocks, const ScanCtrl* ctrl, bool rowspace, bool pdl, const KernelShape& ks, cudaStream_t stream);
cudaError_t launch_count_exchange(const CommPlan& plan, const ScanCtrl* ctrl, CommOut* out, cudaStream_t stream);
cudaError_t launch_agg_exchange(const AggXPlan& plan, const unsigned int* counters, const ScanCtrl* ctrl, AggXOut* out, cudaStream_t stream);
cudaError_t launch_agg_merge(const AggMergePlan& m, const AggXOut* x, AggEntry* table, unsigned int* counters, int num_sms, cudaStream_t stream);
// scan_blocks_kernel over blocks of at most max_block_rows rows.
cudaError_t size_scan_blocks(const ScanPlan& sp, int max_block_rows, KernelShape* ks);
cudaError_t launch_scan_blocks(const ScanPlan& plan, ScanCtrl* ctrl, unsigned long long* status, int grid, size_t dyn_smem,
                               cudaStream_t stream);

}  // namespace imm3
