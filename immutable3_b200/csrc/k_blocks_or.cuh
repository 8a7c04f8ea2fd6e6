// k_blocks_or.cuh - real OR over block-space selections (imm3_query_begin_dnf_ext with IMM3_DNF_ENCODED_FILTER)
// Fragment of kernels.cu (one translation unit, included inside namespace imm3 in the order listed there).
#pragma once

// =============================================================================================
// blocks_or_merge_kernel: the union of two selections of the block filter front (blocks_prune + the lane / quad / mini-block
// filter kernels), left in that front's own output contract so that the emit kernels read it unchanged: a selected-row count
// for EVERY block; the block's 32 bitmap words only where 0 < count < rows (the words of an empty or a full block are stale
// and are never read); the count of every tile of 8 blocks.  acc_* holds the terms merged so far and receives the union,
// term_* the next term's front.  Per block, a = accumulated count, c = the term's, n = rows:
//   a == n or c == 0   unchanged, no words read;
//   a == 0 or c == n   the term's count, and its words if 0 < c < n;
//   both partial       the two blocks' words ORed (masked to the block's rows) and counted; written only if not full.
// One lane per block, 32 blocks per warp: counts move coalesced and tile counts come from shuffles over 8 lanes.  Then the
// whole warp serves, one word per lane, each block of its ballot that needs words.
// =============================================================================================
__global__ void __launch_bounds__(kComputeThreads) blocks_or_merge_kernel(const uint64_t* __restrict__ row_start, long long nblocks, long long ntiles8,
                                                                         uint32_t* __restrict__ acc_words, uint32_t* __restrict__ acc_cnt,
                                                                         const uint32_t* __restrict__ term_words, const uint32_t* __restrict__ term_cnt,
                                                                         uint32_t* __restrict__ tile_cnt, ScanCtrl* ctrl) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long ngroups32 = (nblocks + 31) >> 5;
    for (long long T = warp0; T < ngroups32; T += nwarps) {
        const long long b = T * 32 + lane;
        unsigned n = 0, a = 0, c = 0;  // (lanes past the last block: all 0, i.e. unchanged)
        if (b < nblocks) {
            n = (unsigned)(__ldg(row_start + b + 1) - __ldg(row_start + b));
            a = acc_cnt[b];
            c = __ldg(term_cnt + b);
        }
        IMM3_CHECK(ctrl, a <= n && c <= n, 11);  // a selection never holds more rows than its block
        const bool keep = a == n || c == 0;
        const bool both = !keep && a != 0 && c != n;
        unsigned m = keep ? a : c;
        const unsigned todo = __ballot_sync(0xFFFFFFFFu, !keep && c != n);
        for (unsigned w = todo; w; w &= w - 1u) {
            const int j = __ffs((int)w) - 1;
            const unsigned nj = __shfl_sync(0xFFFFFFFFu, n, j);
            const bool bj = __shfl_sync(0xFFFFFFFFu, (int)both, j) != 0;
            const long long at = (T * 32 + j) * 32 + lane;
            const int left = (int)nj - lane * 32;
            uint32_t word = __ldg(term_words + at);
            if (bj) word |= acc_words[at];
            word &= left >= 32 ? 0xFFFFFFFFu : (left <= 0 ? 0u : ((1u << left) - 1u));
            const unsigned u = __reduce_add_sync(0xFFFFFFFFu, (unsigned)__popc(word));
            if (u < nj) acc_words[at] = word;
            if (lane == j) m = u;
        }
        if (b < nblocks) acc_cnt[b] = m;
        unsigned c8 = m;
        c8 += __shfl_xor_sync(0xFFFFFFFFu, c8, 1);
        c8 += __shfl_xor_sync(0xFFFFFFFFu, c8, 2);
        c8 += __shfl_xor_sync(0xFFFFFFFFu, c8, 4);
        const long long t8 = T * 4 + (lane >> 3);
        if ((lane & 7) == 0 && t8 < ntiles8) tile_cnt[t8] = c8;
    }
}
