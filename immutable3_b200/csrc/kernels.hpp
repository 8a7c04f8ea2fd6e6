// kernels.hpp — host-callable launchers of kernels.cu.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <string>

#include "plan.hpp"

namespace imm3 {

size_t blocks_kernel_smem_bytes(int npfor, int max_block_rows);
cudaError_t blocks_kernel_occupancy(size_t dyn_smem, int* blocks_per_sm);
cudaError_t filter_kernel_occupancy(size_t dyn_smem, int* blocks_per_sm);
cudaError_t emit_kernel_occupancy(bool general, int* blocks_per_sm);
cudaError_t launch_filter(const ScanPlan& plan, uint32_t* bitmap, uint32_t* span_cnt, uint32_t* tile_cnt, unsigned long long* tile_off,
                          ScanCtrl* ctrl, int grid, size_t dyn_smem, cudaStream_t stream);
cudaError_t launch_emit(const ScanPlan& plan, const uint32_t* bitmap, const uint32_t* span_cnt, const unsigned long long* tile_off,
                        int spans_per_tile, long long nspans, int grid, int dense_off, const ScanCtrl* ctrl, bool general, bool pdl,
                        cudaStream_t stream);
size_t emit_stream_smem_bytes(int stage_bytes, int ring);
int emit_stream_header_bytes();
cudaError_t emit_stream_occupancy(size_t dyn_smem, int* blocks_per_sm);
cudaError_t launch_emit_stream(const ScanPlan& plan, const uint32_t* bitmap, const uint32_t* span_cnt, const uint32_t* tile_cnt,
                               const unsigned long long* tile_off, long long nsub, int ring, int stage_bytes, int dense_mode, int grid,
                               size_t dyn_smem, ScanCtrl* ctrl, bool pdl, cudaStream_t stream);
// The aggregation kernel's instantiation (agg_shape is the one place that chooses it): NG group-by columns, NA aggregates,
// nsum SUMs; blocks: agg_blocks_kernel, else agg_kernel; bsel: agg_blocks_kernel reads the block filter's selection (32
// words and one count per block), not the row-space filter's.
struct AggShape { int ng, na, nsum; bool blocks, bsel; };
AggShape agg_shape(const AggPlan& a, bool blocks, bool bsel);
std::string agg_route(const AggShape& s);  // its name in Result.route, e.g. "agg<1,2>", "agg_blocks<0,3>/sum/bsel"
size_t agg_blocks_smem_bytes(const AggShape& s, int npfor, int words_cap);  // dynamic shared memory of agg_blocks_kernel
cudaError_t launch_agg_init(AggEntry* table, uint32_t slots, const AggPlan& a, unsigned int* counters, cudaStream_t stream);
cudaError_t launch_agg(const AggPlan& a, const AggShape& s, const uint32_t* bitmap, const uint32_t* span_cnt, AggEntry* table, unsigned int* counters,
                       const ScanCtrl* ctrl, int num_sms, cudaStream_t stream);
cudaError_t launch_agg_compact(const AggEntry* table, uint32_t slots, AggEntry* out, unsigned int* counters, cudaStream_t stream);
long long scan_inline_max_tiles();
cudaError_t launch_offset_scan(const uint32_t* tile_cnt, unsigned long long* tile_off, long long ntiles, long long limit, uint32_t epoch,
                               unsigned long long* partials, ScanCtrl* ctrl, unsigned int* tile_list, cudaStream_t stream);
cudaError_t blocks_scan_emit_grid(int num_sms, long long ntiles8, int* grid);
cudaError_t launch_blocks_scan_emit(const ScanPlan& plan, const uint32_t* bitmapB, const uint32_t* blk_cnt, const uint32_t* tile_cnt,
                                    unsigned long long* tile_off, long long nblocks, uint32_t epoch, unsigned long long* partials, ScanCtrl* ctrl,
                                    unsigned int* tile_list, bool pdl, int grid, cudaStream_t stream, CtrlBlock* pub = nullptr,
                                    unsigned long long pub_seq = 0);
int blocks_group_emit_max_groups();
size_t blocks_group_sum_bytes();
cudaError_t blocks_group_emit_grid(int num_sms, long long nblocks, int* grid, int* ngroups);
cudaError_t launch_blocks_group_emit(const ScanPlan& plan, const uint32_t* bitmapB, const uint32_t* blk_cnt, uint32_t* grp_sum, long long nblocks,
                                     int ngroups, ScanCtrl* ctrl, bool pdl, int grid, cudaStream_t stream, CtrlBlock* pub = nullptr,
                                     unsigned long long pub_seq = 0);
size_t blocks_filter_smem_bytes(int nstaged, int tile_cap_bytes, int ring);
int blocks_filter_slot_bytes(int nstaged, int tile_cap_bytes);
size_t blocks_emit_smem_bytes(int npfor, int words_cap);
int blocks_filter_quad_slot_bytes(int tile_cap_bytes);
// The block filter kernels: lane = mini-block (blocks_filter_kernel), quad (blocks_filter_quad_kernel), lane = block
// (blocks_filter_lane_kernel, lane_warps warps per CTA).
enum class BlockFilter { kMini, kQuad, kLane };
cudaError_t blocks_filter_occupancy(size_t filter_smem, BlockFilter filter, int lane_warps, int* blocks_per_sm);
cudaError_t blocks_emit_occupancy(size_t emit_smem, bool rowspace, int* blocks_per_sm);
cudaError_t launch_blocks_filter(const ScanPlan& plan, uint32_t* bitmapB, uint32_t* blk_cnt, uint32_t* tile_cnt, unsigned long long* tile_off,
                                 ScanCtrl* ctrl, long long nblocks, int grid, size_t dyn_smem, BlockFilter filter, int lane_warps,
                                 const unsigned int* work, cudaStream_t stream, uint32_t* grp_sum = nullptr);  // grp_sum: blocks_group_emit_kernel follows (lane kernel only)
cudaError_t launch_block_stats(const PforCol& pc, const uint64_t* row_start, long long nblocks, int words_cap, int num_sms, BlockStat* stats,
                               cudaStream_t stream);
cudaError_t launch_blocks_prune(const PrunePlan& q, const uint64_t* row_start, long long nblocks, long long ntiles8, uint32_t* blk_cnt,
                                uint32_t* tile_cnt, unsigned int* work, int num_sms, cudaStream_t stream, uint32_t* grp_sum = nullptr);
// Real OR over encoded columns: acc_* (the block filter's selection of the terms so far) |= term_* (the next term's), in the
// same contract - every block's count, the words of partial blocks only - and every 8-block tile count rewritten.
cudaError_t launch_blocks_or_merge(const uint64_t* row_start, long long nblocks, long long ntiles8, uint32_t* acc_words, uint32_t* acc_cnt,
                                   const uint32_t* term_words, const uint32_t* term_cnt, uint32_t* tile_cnt, ScanCtrl* ctrl, int num_sms,
                                   cudaStream_t stream);
// rowspace: the bitmap / counts come from the dense filter kernel (row space), not from blocks_filter_kernel (block-local)
cudaError_t launch_blocks_emit(const ScanPlan& plan, const uint32_t* bitmap, const uint32_t* cnts, const unsigned int* tile_list, const unsigned long long* tile_off,
                               long long nblocks, const ScanCtrl* ctrl, bool rowspace, bool pdl, int grid, size_t dyn_smem,
                               cudaStream_t stream);
cudaError_t launch_count_exchange(const CommPlan& plan, const ScanCtrl* ctrl, CommOut* out, cudaStream_t stream);
cudaError_t launch_agg_exchange(const AggXPlan& plan, const unsigned int* counters, const ScanCtrl* ctrl, AggXOut* out, cudaStream_t stream);
cudaError_t launch_agg_merge(const AggMergePlan& m, const AggXOut* x, AggEntry* table, unsigned int* counters, int num_sms, cudaStream_t stream);
cudaError_t launch_scan_blocks(const ScanPlan& plan, ScanCtrl* ctrl, unsigned long long* status, int grid, size_t dyn_smem,
                               cudaStream_t stream);

}  // namespace imm3
