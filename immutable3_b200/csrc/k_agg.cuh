// k_agg.cuh - count / min / max ... group by over the selection bitmap (ProjectAggOp, ProjectAggregate.scala:115-226)
// Fragment of kernels.cu (one translation unit, included inside namespace imm3 in the order listed there).
#pragma once

// =============================================================================================
// The reference aggregates per segment worker into a LinkedHashMap keyed by the group values (ProjectAggregate.scala:
// 160-166) and merges the per-segment maps in ProjectAggregateQueueOp (ProjectAggregateQueue.scala:21-45).  Here:
//   filter_kernel            the same K1 as every query: selection bitmap + span / tile counts (nothing is projected)
//   agg_kernel               one warp per 1024-row span with selected rows: the span's selection vector (append_selection),
//                            then 64 selected rows per iteration (two steps of 32, the gathers of both issued before the
//                            first update) - a lane gathers its row's group cells (packed into a 64-bit key) and aggregate
//                            inputs, finds the group's slot in the CTA's key table through a hash -> slot cache (two loads,
//                            no probing) and updates the WARP's own partial aggregates of that slot: MIN / MAX read the
//                            value first and only issue an atomic when the row improves it (after the first rows of a
//                            group almost never), COUNT is one native 32-bit shared-memory atomic; at the end the CTA
//                            folds its warps' values per slot and adds the groups to the global table
//   agg_blocks_kernel        instead of agg_kernel when a MIN / MAX input or a group column is in the sorted-int codec: one
//                            warp per reference BLOCK with selected rows, the block's encoded columns decoded into the
//                            warp's shared memory, then agg_kernel's row loop (see below)
//   agg_compact_kernel       occupied slots of the global table -> a dense array (any order; the host sorts the groups by
//                            the canonical ordinal of their first row, the order the reference reports them in with one
//                            worker) and clears the table for the next query
//   agg_merge_kernel         imm3_query_agg_global only: every rank's compacted partial groups (behind k_comm.cuh's
//                            agg_exchange_kernel) into a fresh global table, then agg_compact_kernel again
// Exact integer arithmetic: counts are 64-bit, min / max are taken on the raw int32 / int8 values (the reference widens to
// Double, which is exact for both types; the host formats them as Doubles).
// SUM (imm3_query_agg_ext only, DESIGN §4.4c) runs its own instantiations, agg_kernel / agg_blocks_kernel<NG, NA, true>: the
// same row loop with a 64-bit per-warp partial per SUM and slot, every add modulo 2^64.  Past the fold a SUM travels as
// a COUNT (the global table, agg_init_kernel and agg_merge_kernel add it with the same 64-bit atomicAdd).
// =============================================================================================
constexpr unsigned long long kAggEmpty = ~0ull;

__device__ __forceinline__ uint32_t agg_hash(unsigned long long k) {
    k ^= k >> 33;
    k *= 0xFF51AFD7ED558CCDull;
    k ^= k >> 33;
    return (uint32_t)k;
}

// Shared-memory state of a CTA (dynamic shared memory, in this order):
//   dict   2^14 bytes   hash(key) -> slot: a CACHE in front of the key table (any byte value is a valid guess: the key table
//                       confirms it), so a row finds its group with two loads and no probing; written without atomics
//   keys   256 x u64    the CTA's groups: open addressing, a slot is claimed with one CAS and never moves
//   vals   per WARP (NA + 1) x 256 x int32: the warp's own partial aggregates of every slot - a low-cardinality group-by
//                       (51 states) on one table per CTA serialised every warp of the SM on the same few words (5.2 ms for the
//                       reference's example on 100 M rows).  Value NA is the group's first row as the warp saw it.
//   sel    per warp 1024 x u16: the selection vector of the span in hand
// MIN, MAX and the first row share one update - "read the slot, atomicMax only if the row beats it": a MIN column is kept
// as the MAX of the complemented inputs (~x reverses the order of int32 without overflow) and complemented back when the
// table leaves shared memory; after a group's first rows the atomics all but disappear.  COUNT is one native 32-bit
// shared-memory atomic per row (a warp counts far fewer than 2^32 rows).
// A SUM's partial is 64-bit: its low words sit in the aggregate's own plane, its high words in one more plane per SUM
// behind the first-row plane (plane NA + 1 + j for the j-th SUM of the plan).  A 64-bit atomicAdd on shared memory is a
// CAS loop on sm_100a (ATOMS.CAST.SPIN.64), so a row adds its value with one native 32-bit atomicAdd on the low word and
// carries into the high word from the old value it returns: the high word moves only on a carry or a negative input.
constexpr int kAggSlots = 256;
constexpr int kAggDictBits = 14;
constexpr size_t agg_smem_bytes(int na, int nsum = 0) {
    return ((size_t)1 << kAggDictBits) + (size_t)kAggSlots * 8 + (size_t)kComputeWarps * (na + 1 + nsum) * kAggSlots * 4 + (size_t)kComputeWarps * 1024 * 2;
}
// Bit a set = aggregate a is a SUM (S: a SUM instantiation; elsewhere no plan has one).
template <int NA, bool S>
__device__ __forceinline__ unsigned agg_sum_mask(const AggPlan& A) {
    unsigned m = 0;
    if constexpr (S) {
#pragma unroll
        for (int a = 0; a < NA; a++) m |= A.agg[a].op == kAggSum ? 1u << a : 0u;
    }
    return m;
}
// x into the 64-bit partial of aggregate a (a SUM) at slot: lo = the low word in the aggregate's plane, V = the warp's values.
template <int NA>
__device__ __forceinline__ void agg_sum_add(int* V, int* lo, unsigned sum_mask, int a, int slot, int x) {
    const unsigned old = atomicAdd(reinterpret_cast<unsigned int*>(lo), (unsigned)x);
    const int dhi = (x >> 31) + (old + (unsigned)x < old ? 1 : 0);  // sign extension + carry out of the low word
    if (dhi != 0) atomicAdd(V + (NA + 1 + __popc(sum_mask & ((1u << a) - 1u))) * kAggSlots + slot, dhi);
}
// Warp partial of SUM a at slot i as a 64-bit two's-complement value (W = the warp's values).
template <int NA>
__device__ __forceinline__ long long agg_sum_read(const int* W, unsigned sum_mask, int a, int i) {
    const unsigned lo = (unsigned)W[a * kAggSlots + i], hi = (unsigned)W[(NA + 1 + __popc(sum_mask & ((1u << a) - 1u))) * kAggSlots + i];
    return (long long)(((unsigned long long)hi << 32) | lo);
}
__device__ __forceinline__ uint32_t agg_hash32(unsigned long long k) {
    return ((uint32_t)k * 0x9E3779B1u) ^ ((uint32_t)(k >> 32) * 0x85EBCA6Bu);
}
// Slot of `key` in the CTA's key table (claimed if new), -1 if the table has no room near the key's home slot.
__device__ __forceinline__ int agg_cta_slot(uint8_t* dict, unsigned long long* keys, unsigned long long key) {
    const uint32_t hh = agg_hash32(key);
    volatile uint8_t* const guess = dict + (hh >> (32 - kAggDictBits));
    uint32_t h = *guess;
    if (*reinterpret_cast<volatile unsigned long long*>(&keys[h]) == key) return (int)h;  // (nearly every row after a group's first)
    h = hh >> 24;
    for (int p = 0; p < 16; p++, h = (h + 1) & (kAggSlots - 1)) {  // (16 taken slots in a row: the table is as good as full)
        unsigned long long cur = *reinterpret_cast<volatile unsigned long long*>(&keys[h]);
        if (cur == kAggEmpty) {
            const unsigned long long old = atomicCAS(&keys[h], kAggEmpty, key);
            cur = old == kAggEmpty ? key : old;
        }
        if (cur == key) {
            *guess = (uint8_t)h;
            return (int)h;
        }
    }
    return -1;
}

// Slot of `key` in the global table (claimed if new), -1 = table full.
__device__ __forceinline__ int agg_global_slot(AggEntry* table, uint32_t slots, unsigned long long key) {
    uint32_t h = agg_hash(key) & (slots - 1);
    for (uint32_t p = 0; p < slots; p++, h = (h + 1) & (slots - 1)) {
        unsigned long long* kp = &table[h].key;
        unsigned long long cur = *reinterpret_cast<volatile unsigned long long*>(kp);
        if (cur == kAggEmpty) {
            const unsigned long long old = atomicCAS(kp, kAggEmpty, key);
            cur = old == kAggEmpty ? key : old;
        }
        if (cur == key) return (int)h;
    }
    return -1;
}

__device__ __forceinline__ void agg_update(long long* v, int op, long long x) {
    if (op == kAggCount) atomicAdd(reinterpret_cast<unsigned long long*>(v), (unsigned long long)x);
    else if (op == kAggMin) atomicMin(v, x);
    else atomicMax(v, x);
}
__device__ __forceinline__ long long agg_identity(int op) { return op == kAggCount ? 0ll : (op == kAggMin ? LLONG_MAX : LLONG_MIN); }

// One group's partial (x[a]: a count, or an extreme as int64) into the global table.  (K: agg_blocks_kernel calls its own
// copy, K = 1, agg_merge_kernel K = 2 and the SUM instantiations K = 3 and 4, so that agg_kernel's call
// graph - and with it agg_kernel's register allocation - is the one it had alone.)
template <int K = 0>
__device__ __noinline__ void agg_to_global(AggEntry* table, uint32_t slots, unsigned int* overflow, unsigned long long key, unsigned long long fr,
                                           const long long* x, const AggCol* aggs, int naggs) {
    const int gs = agg_global_slot(table, slots, key);
    if (gs < 0) {
        atomicExch(overflow, 1u);
        return;
    }
    atomicMin(&table[gs].first_row, fr);
    for (int a = 0; a < naggs; a++) agg_update(&table[gs].val[a], aggs[a].op, x[a]);
}
// The fold of a SUM instantiation (agg_kernel: K = 3, agg_blocks_kernel: K = 4): thread t folds slot t over the
// CTA's warps in 64 bits - COUNT and SUM add modulo 2^64, MIN / MAX take the extreme - and hands the group to the global
// table, where a SUM is added as a COUNT.  nplanes = 32-bit planes per warp; first_row(w, ord) = the row of warp w's ordinal.
template <int NA, int K, class FirstRow>
__device__ __forceinline__ void agg_fold_sum(const AggPlan& A, int naggs, const unsigned long long* keys, const int* vals, int nplanes, unsigned sum_mask,
                                             AggEntry* table, unsigned int* overflow, const AggCol* s_agg, int tid, FirstRow first_row) {
    for (int i = tid; i < kAggSlots; i += kComputeThreads) {
        const unsigned long long key = keys[i];
        if (key == kAggEmpty) continue;
        unsigned long long first = ~0ull;
        unsigned long long acc[kMaxAggs];
#pragma unroll
        for (int a = 0; a < NA; a++) acc[a] = (A.agg[a].op == kAggMin || A.agg[a].op == kAggMax) ? (unsigned long long)(long long)INT_MIN : 0ull;
        for (int w = 0; w < kComputeWarps; w++) {
            const int* const W = vals + w * nplanes * kAggSlots;
            const int fo = W[NA * kAggSlots + i];
            if (fo == INT_MIN) continue;  // warp w never saw this group
            const unsigned long long r = first_row(w, (unsigned)~fo);
            first = r < first ? r : first;
#pragma unroll
            for (int a = 0; a < NA; a++) {
                if (NA == 8 && a >= naggs) break;
                const int op = A.agg[a].op, v = W[a * kAggSlots + i];
                if (op == kAggCount) acc[a] += (unsigned)v;
                else if (op == kAggSum) acc[a] += (unsigned long long)agg_sum_read<NA>(W, sum_mask, a, i);
                else if ((long long)v > (long long)acc[a]) acc[a] = (unsigned long long)(long long)v;
            }
        }
        if (first == ~0ull) continue;
        long long xl[kMaxAggs];
#pragma unroll
        for (int a = 0; a < NA; a++) xl[a] = A.agg[a].op == kAggMin ? (long long)~(int)acc[a] : (long long)acc[a];
        agg_to_global<K>(table, A.table_slots, overflow, key, first, xl, s_agg, naggs);
    }
}

// NG = group-by columns (0, 1, 2 exact; 4 = A.ngroup of them, up to 4), NA = aggregates (1 .. 4 exact; 8 = A.naggs of them, up to 8):
// the loops over the plan are unrolled with compile-time indices into the kernel's parameter block, so the per-column
// descriptors are constant-bank operands - nothing about the query is decoded per row and nothing of it lives in registers.
// S = true: the SUM instantiations (a plan with a SUM); with S = false the code is the one agg_kernel had before SUM existed.
template <int NG, int NA, bool S>
__global__ void __launch_bounds__(kComputeThreads, 3) agg_kernel(const __grid_constant__ AggPlan A, const uint32_t* __restrict__ bitmap,
                                                                  const uint32_t* __restrict__ span_cnt, AggEntry* __restrict__ table,
                                                                  unsigned int* __restrict__ overflow, const ScanCtrl* ctrl) {
    extern __shared__ __align__(128) uint8_t agg_smem[];
    const unsigned sum_mask = agg_sum_mask<NA, S>(A);
    const int nplanes = NA + 1 + (S ? __popc(sum_mask) : 0);  // 32-bit planes per warp
    uint8_t* const dict = agg_smem;
    unsigned long long* const keys = reinterpret_cast<unsigned long long*>(agg_smem + (1u << kAggDictBits));
    int* const vals = reinterpret_cast<int*>(agg_smem + (1u << kAggDictBits) + kAggSlots * 8);
    unsigned short* const sel_all = reinterpret_cast<unsigned short*>(vals + kComputeWarps * nplanes * kAggSlots);
    __shared__ AggCol s_agg[kMaxAggs];  // (for the cold paths only: a row or a group that goes to the global table)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#pragma unroll
    for (int i = 0; i < kMaxAggs; i++)
        if (tid == i) {
            s_agg[i] = A.agg[i];
            if (S && A.agg[i].op == kAggSum) s_agg[i].op = kAggCount;  // (the global table adds a SUM as a COUNT)
        }
    const int naggs = NA == 8 ? A.naggs : NA, ngroup = NG == 4 ? A.ngroup : NG;
    for (int i = tid; i < (1 << kAggDictBits) / 4; i += kComputeThreads) reinterpret_cast<uint32_t*>(dict)[i] = 0u;
    for (int i = tid; i < kAggSlots; i += kComputeThreads) keys[i] = kAggEmpty;
    int* const V = vals + warp * nplanes * kAggSlots;  // this warp's values: V[a * kAggSlots + slot]
    for (int i = lane; i < kAggSlots; i += 32) {
#pragma unroll
        for (int a = 0; a < NA; a++) V[a * kAggSlots + i] = (A.agg[a].op == kAggCount || (S && A.agg[a].op == kAggSum)) ? 0 : INT_MIN;
        V[NA * kAggSlots + i] = INT_MIN;
        if (S)
            for (int p = NA + 1; p < nplanes; p++) V[p * kAggSlots + i] = 0;
    }
    __syncthreads();

    // The group key and the aggregate inputs of row `r` of the span in hand, in two halves so that the loads of several rows
    // are in flight together: fetch_raw ISSUES the loads (cells of 1, 2 and 4 bytes: the aligned 32-bit word that holds them -
    // the arenas are padded to whole tiles - one load type, no branch on the width, 32-bit offsets) and consumes nothing;
    // decode turns the words into the key and the inputs (MIN inputs complemented).  gp / ap = the columns at the span's
    // first row.  Group cells of other widths are gathered byte-wise in decode.
    const uint8_t* gp[NG > 0 ? NG : 1];
    const uint8_t* ap[NA];
    auto fetch_raw = [&](unsigned r, uint32_t (&gw)[NG > 0 ? NG : 1], uint32_t (&aw)[NA]) {
#pragma unroll
        for (int g = 0; g < NG; g++) {
            gw[g] = 0;
            if (NG == 4 && g >= ngroup) break;
            const unsigned w = (unsigned)A.group[g].width;
            if (w <= 4u && (w & (w - 1u)) == 0u) gw[g] = __ldg(reinterpret_cast<const uint32_t*>(gp[g] + ((r * w) & ~3u)));
        }
#pragma unroll
        for (int a = 0; a < NA; a++) {
            aw[a] = 0;
            if (NA == 8 && a >= naggs) break;
            if (A.agg[a].op != kAggCount) aw[a] = __ldg(reinterpret_cast<const uint32_t*>(ap[a] + ((r * (unsigned)A.agg[a].width) & ~3u)));
        }
    };
    auto decode = [&](unsigned r, const uint32_t (&gw)[NG > 0 ? NG : 1], const uint32_t (&aw)[NA], unsigned long long& key, int (&x)[NA]) {
        key = 0;
#pragma unroll
        for (int g = 0; g < NG; g++) {
            if (NG == 4 && g >= ngroup) break;
            const unsigned w = (unsigned)A.group[g].width;
            const unsigned off = r * w;
            unsigned long long cell = 0;
            if (w <= 4u && (w & (w - 1u)) == 0u) {
                cell = (gw[g] >> ((off & 3u) * 8u)) & (0xFFFFFFFFu >> (32u - 8u * w));
            } else {
                for (unsigned b = 0; b < w; b++) cell |= (unsigned long long)__ldg(gp[g] + off + b) << (8u * b);
            }
            key |= cell << A.group[g].key_shift;
        }
#pragma unroll
        for (int a = 0; a < NA; a++) {
            x[a] = 0;
            if (NA == 8 && a >= naggs) break;
            const int op = A.agg[a].op;
            if (op != kAggCount) {
                const unsigned w = (unsigned)A.agg[a].width;  // 4 (INT) or 1 (TINYINT, sign-extended)
                const int v = (int)(aw[a] << ((4u - w - ((r * w) & 3u)) * 8u)) >> ((4u - w) * 8u);
                x[a] = v ^ (op == kAggMin ? -1 : 0);
            }
        }
    };
    // one row into its group: `ord` = the row's ordinal in this warp's own sequence of rows (ascending: a group's first row
    // is the one that creates its entry in the warp's values)
    auto apply = [&](long long row, unsigned ord, unsigned long long key, const int (&x)[NA]) {
        const int slot = agg_cta_slot(dict, keys, key);
        if (slot >= 0) {
#pragma unroll
            for (int a = 0; a < NA; a++) {
                if (NA == 8 && a >= naggs) break;
                int* const v = V + a * kAggSlots + slot;
                if (A.agg[a].op == kAggCount) atomicAdd(reinterpret_cast<unsigned int*>(v), 1u);
                else if (S && A.agg[a].op == kAggSum) agg_sum_add<NA>(V, v, sum_mask, a, slot, x[a]);
                else if (x[a] > *reinterpret_cast<volatile int*>(v)) atomicMax(v, x[a]);  // (a stale read is only ever too low: at worst one atomic too many)
            }
            int* const f = V + NA * kAggSlots + slot;
            const int fo = ~(int)ord;
            if (fo > *reinterpret_cast<volatile int*>(f)) atomicMax(f, fo);
        } else {  // the CTA's table is full
            long long xl[kMaxAggs];
#pragma unroll
            for (int a = 0; a < NA; a++) xl[a] = A.agg[a].op == kAggCount ? 1ll : (long long)(A.agg[a].op == kAggMin ? ~x[a] : x[a]);
            agg_to_global<S ? 3 : 0>(table, A.table_slots, overflow, key, (unsigned long long)row, xl, s_agg, naggs);
        }
    };

    asm volatile("griddepcontrol.wait;" ::: "memory");  // the filter kernel's bitmap and counts are final
    const long long span_stride = (long long)gridDim.x * kComputeWarps, span_first = (long long)blockIdx.x * kComputeWarps + warp;
    if (__ldcg(&ctrl->total) != 0ull) {
        unsigned short* const sel_w = sel_all + warp * 1024;
        const long long nspans = A.ntiles * 8;
        unsigned ord0 = 0;  // 1024 x the number of spans this warp has been through (< 2^31: a warp sees every (8 x grid)-th span)
        for (long long span = span_first; span < nspans; span += span_stride, ord0 += 1024u) {
            const unsigned n = __ldg(span_cnt + span);
            if (n == 0) continue;
            const uint32_t m = __ldg(bitmap + span * 32 + lane);
            __syncwarp();
            append_selection(m, lane, sel_w, 0u);
            __syncwarp();
            const long long row0 = span * 1024;
#pragma unroll
            for (int g = 0; g < NG; g++) gp[g] = A.group[g].base + row0 * A.group[g].width;
#pragma unroll
            for (int a = 0; a < NA; a++) ap[a] = A.agg[a].base + row0 * A.agg[a].width;
            // 64 selected rows per iteration (two steps of 32), software-pipelined: the loads of the NEXT iteration are issued
            // before this iteration's updates and consumed after them, so the global-memory latency hides behind the
            // shared-memory work
            constexpr int NGW = NG > 0 ? NG : 1;
            unsigned s0 = lane < n ? sel_w[lane] : 0u, s1 = 32u + lane < n ? sel_w[32 + lane] : 0u;
            uint32_t g0[NGW], g1[NGW], a0[NA], a1[NA];
            fetch_raw(s0, g0, a0);
            fetch_raw(s1, g1, a1);
            for (unsigned i0 = 0; i0 < n; i0 += 64) {
                const bool live0 = i0 + lane < n, live1 = i0 + 32 + lane < n;
                unsigned long long k0, k1;
                int x0[NA], x1[NA];
                decode(s0, g0, a0, k0, x0);
                decode(s1, g1, a1, k1, x1);
                const unsigned c0 = s0, c1 = s1;
                if (i0 + 64 < n) {  // (rows past the selection vector's end fetch row 0 of the span: harmless, never applied)
                    s0 = i0 + 64 + lane < n ? sel_w[i0 + 64 + lane] : 0u;
                    s1 = i0 + 96 + lane < n ? sel_w[i0 + 96 + lane] : 0u;
                    fetch_raw(s0, g0, a0);
                    fetch_raw(s1, g1, a1);
                }
                if (live0) apply(row0 + c0, ord0 + c0, k0, x0);
                if (live1) apply(row0 + c1, ord0 + c1, k1, x1);
            }
        }
    }
    // thread t folds slot t over the CTA's warps and hands the group to the global table
    __syncthreads();
    if constexpr (S) {
        agg_fold_sum<NA, 3>(A, naggs, keys, vals, nplanes, sum_mask, table, overflow, s_agg, tid, [&](int w, unsigned ord) -> unsigned long long {
            return ((unsigned long long)((long long)blockIdx.x * kComputeWarps + w + (long long)(ord >> 10) * span_stride) << 10) | (ord & 1023u);
        });
    } else {
        for (int i = tid; i < kAggSlots; i += kComputeThreads) {
            const unsigned long long key = keys[i];
            if (key == kAggEmpty) continue;
            unsigned long long first = ~0ull;
            int acc[NA];
#pragma unroll
            for (int a = 0; a < NA; a++) acc[a] = A.agg[a].op == kAggCount ? 0 : INT_MIN;
            for (int w = 0; w < kComputeWarps; w++) {
                const int* const W = vals + w * (NA + 1) * kAggSlots;
                const int fo = W[NA * kAggSlots + i];
                if (fo == INT_MIN) continue;  // warp w never saw this group
                const unsigned ord = (unsigned)~fo;
                const unsigned long long r = ((unsigned long long)((long long)blockIdx.x * kComputeWarps + w + (long long)(ord >> 10) * span_stride) << 10) | (ord & 1023u);
                first = r < first ? r : first;
#pragma unroll
                for (int a = 0; a < NA; a++) {
                    if (NA == 8 && a >= naggs) break;
                    const int v = W[a * kAggSlots + i];
                    acc[a] = A.agg[a].op == kAggCount ? (int)((unsigned)acc[a] + (unsigned)v) : (v > acc[a] ? v : acc[a]);  // (a CTA counts < 2^32 rows)
                }
            }
            if (first == ~0ull) continue;
            long long xl[kMaxAggs];
#pragma unroll
            for (int a = 0; a < NA; a++) xl[a] = A.agg[a].op == kAggCount ? (long long)(unsigned int)acc[a] : (long long)(A.agg[a].op == kAggMin ? ~acc[a] : acc[a]);
            agg_to_global(table, A.table_slots, overflow, key, first, xl, s_agg, naggs);
        }
    }
}

// agg_blocks_kernel's per-row work, as functions of the plan: the same steps as agg_kernel's lambdas (fetch_raw / decode /
// apply / the fold), which stay written out in agg_kernel - routed through these functions its generated code changes.
// A CTA's empty state: no dict guesses, no keys, this warp's values at their identities (first row: "never seen").
// (S: a SUM instantiation - SUM partials and the high-word planes behind the first-row plane start at 0.)
template <int NA, bool S = false>
__device__ __forceinline__ void agg_state_init(const AggPlan& A, uint8_t* dict, unsigned long long* keys, int* V, int tid, int lane, int nplanes = NA + 1) {
    for (int i = tid; i < (1 << kAggDictBits) / 4; i += kComputeThreads) reinterpret_cast<uint32_t*>(dict)[i] = 0u;
    for (int i = tid; i < kAggSlots; i += kComputeThreads) keys[i] = kAggEmpty;
    for (int i = lane; i < kAggSlots; i += 32) {
#pragma unroll
        for (int a = 0; a < NA; a++) V[a * kAggSlots + i] = (A.agg[a].op == kAggCount || (S && A.agg[a].op == kAggSum)) ? 0 : INT_MIN;
        V[NA * kAggSlots + i] = INT_MIN;
        if (S)
            for (int p = NA + 1; p < nplanes; p++) V[p * kAggSlots + i] = 0;
    }
}
// The words fetched for row `r` (gw / aw: the aligned 32-bit word holding each cell; gp = the group columns at the row
// the offsets count from) -> the packed group key and the aggregate inputs (MIN inputs complemented).  Group cells of
// other widths are gathered byte-wise.
template <int NG, int NA>
__device__ __forceinline__ void agg_decode(const AggPlan& A, int ngroup, int naggs, const uint8_t* const (&gp)[NG > 0 ? NG : 1], unsigned r,
                                           const uint32_t (&gw)[NG > 0 ? NG : 1], const uint32_t (&aw)[NA], unsigned long long& key, int (&x)[NA]) {
    key = 0;
#pragma unroll
    for (int g = 0; g < NG; g++) {
        if (NG == 4 && g >= ngroup) break;
        const unsigned w = (unsigned)A.group[g].width;
        const unsigned off = r * w;
        unsigned long long cell = 0;
        if (w <= 4u && (w & (w - 1u)) == 0u) {
            cell = (gw[g] >> ((off & 3u) * 8u)) & (0xFFFFFFFFu >> (32u - 8u * w));
        } else {
            for (unsigned b = 0; b < w; b++) cell |= (unsigned long long)__ldg(gp[g] + off + b) << (8u * b);
        }
        key |= cell << A.group[g].key_shift;
    }
#pragma unroll
    for (int a = 0; a < NA; a++) {
        x[a] = 0;
        if (NA == 8 && a >= naggs) break;
        const int op = A.agg[a].op;
        if (op != kAggCount) {
            const unsigned w = (unsigned)A.agg[a].width;  // 4 (INT) or 1 (TINYINT, sign-extended)
            const int v = (int)(aw[a] << ((4u - w - ((r * w) & 3u)) * 8u)) >> ((4u - w) * 8u);
            x[a] = v ^ (op == kAggMin ? -1 : 0);
        }
    }
}
// One row into its group: `ord` = the row's ordinal in this warp's own sequence of rows (ascending: a group's first row
// is the one that creates its entry in the warp's values); `row` = its row ordinal (the cold path's first row).
template <int NA, bool S = false>
__device__ __forceinline__ void agg_apply(const AggPlan& A, int naggs, uint8_t* dict, unsigned long long* keys, int* V, AggEntry* table,
                                          unsigned int* overflow, const AggCol* s_agg, long long row, unsigned ord, unsigned long long key,
                                          const int (&x)[NA], unsigned sum_mask = 0u) {
    const int slot = agg_cta_slot(dict, keys, key);
    if (slot >= 0) {
#pragma unroll
        for (int a = 0; a < NA; a++) {
            if (NA == 8 && a >= naggs) break;
            int* const v = V + a * kAggSlots + slot;
            if (A.agg[a].op == kAggCount) atomicAdd(reinterpret_cast<unsigned int*>(v), 1u);
            else if (S && A.agg[a].op == kAggSum) agg_sum_add<NA>(V, v, sum_mask, a, slot, x[a]);
            else if (x[a] > *reinterpret_cast<volatile int*>(v)) atomicMax(v, x[a]);  // (a stale read is only ever too low: at worst one atomic too many)
        }
        int* const f = V + NA * kAggSlots + slot;
        const int fo = ~(int)ord;
        if (fo > *reinterpret_cast<volatile int*>(f)) atomicMax(f, fo);
    } else {  // the CTA's table is full
        long long xl[kMaxAggs];
#pragma unroll
        for (int a = 0; a < NA; a++) xl[a] = A.agg[a].op == kAggCount ? 1ll : (long long)(A.agg[a].op == kAggMin ? ~x[a] : x[a]);
        agg_to_global<S ? 4 : 1>(table, A.table_slots, overflow, key, (unsigned long long)row, xl, s_agg, naggs);
    }
}
// Thread t folds slot t over the CTA's warps and hands the group to the global table; first_row(w, ord) = the row ordinal
// of warp w's ordinal `ord`.
template <int NA, class FirstRow>
__device__ __forceinline__ void agg_fold(const AggPlan& A, int naggs, const unsigned long long* keys, const int* vals, AggEntry* table,
                                         unsigned int* overflow, const AggCol* s_agg, int tid, FirstRow first_row) {
    for (int i = tid; i < kAggSlots; i += kComputeThreads) {
        const unsigned long long key = keys[i];
        if (key == kAggEmpty) continue;
        unsigned long long first = ~0ull;
        int acc[NA];
#pragma unroll
        for (int a = 0; a < NA; a++) acc[a] = A.agg[a].op == kAggCount ? 0 : INT_MIN;
        for (int w = 0; w < kComputeWarps; w++) {
            const int* const W = vals + w * (NA + 1) * kAggSlots;
            const int fo = W[NA * kAggSlots + i];
            if (fo == INT_MIN) continue;  // warp w never saw this group
            const unsigned long long r = first_row(w, (unsigned)~fo);
            first = r < first ? r : first;
#pragma unroll
            for (int a = 0; a < NA; a++) {
                if (NA == 8 && a >= naggs) break;
                const int v = W[a * kAggSlots + i];
                acc[a] = A.agg[a].op == kAggCount ? (int)((unsigned)acc[a] + (unsigned)v) : (v > acc[a] ? v : acc[a]);  // (a CTA counts < 2^32 rows)
            }
        }
        if (first == ~0ull) continue;
        long long xl[kMaxAggs];
#pragma unroll
        for (int a = 0; a < NA; a++) xl[a] = A.agg[a].op == kAggCount ? (long long)(unsigned int)acc[a] : (long long)(A.agg[a].op == kAggMin ? ~acc[a] : acc[a]);
        agg_to_global<1>(table, A.table_slots, overflow, key, first, xl, s_agg, naggs);
    }
}

// agg_blocks_kernel: the same aggregation when a MIN / MAX input or a group column is in the sorted-int codec.  The filter
// is the same row-space filter_kernel (no predicate touches an encoded column); the work unit is a reference block instead
// of a 1024-row span, because an encoded column can only be decoded block by block:
//   one warp per block with selected rows (blocks warp0, warp0 + nwarps, ...: round robin, like blocks_emit_kernel<true>);
//   the block's selection bits = the row-space bitmap funnel-shifted to its first row R0; every encoded column the query
//   reads is decoded into the warp's own shared memory - the dense sorted shape into dense_prepare's O(1)-per-row form,
//   anything else by pfor_decode_warp - and never written to HBM; then agg_kernel's row loop: dense cells gathered at
//   R0 + row, encoded cells read from shared memory, the same key packing, slot cache, per-warp partials and fold.
// A warp's ordinal of a row is k * 1024 + row-in-block, k = the warp's round-robin position, so the fold recovers the
// block (warp0 + k * nwarps) and the first row (row_start[block] + row-in-block).
// Per warp, after agg_kernel's state (without its selection vectors): max(words_cap, 512) words - the block's byte-swapped
// encoded words while a column is decoded, then the block's selection vector - and per encoded column kBlkVals decoded
// values + 32 mini-block bases.
__host__ __device__ constexpr int agg_blocks_warp_words(int npfor, int words_cap) { return (words_cap > 512 ? words_cap : 512) + npfor * (kBlkVals + 32); }
constexpr size_t agg_blocks_state_bytes(int na, int nsum = 0) { return agg_smem_bytes(na, nsum) - (size_t)kComputeWarps * 1024 * 2; }

// S = true: the SUM instantiations, as agg_kernel's.
// BS = true: the selection is the BLOCK filter's output (imm3_query_agg_ext with IMM3_AGG_ENCODED_FILTER, DESIGN §4.4d):
// `bitmap` = 32 words per block (bit r of block b = row R0 + r), `span_cnt` = the selected rows per block (blk_cnt).  A block
// is a candidate iff its count is not 0; its words are read only if 0 < count < rows (blocks_prune_kernel and the filter
// kernels write no words for an empty or a fully selected block: those words are stale from earlier queries).
template <int NG, int NA, bool S, bool BS>
__global__ void __launch_bounds__(kComputeThreads, 2) agg_blocks_kernel(const __grid_constant__ AggPlan A, const uint32_t* __restrict__ bitmap,
                                                                         const uint32_t* __restrict__ span_cnt, AggEntry* __restrict__ table,
                                                                         unsigned int* __restrict__ overflow, const ScanCtrl* ctrl) {
    extern __shared__ __align__(128) uint8_t agg_smem[];
    const unsigned sum_mask = agg_sum_mask<NA, S>(A);
    const int nsum = S ? __popc(sum_mask) : 0, nplanes = NA + 1 + nsum;
    uint8_t* const dict = agg_smem;
    unsigned long long* const keys = reinterpret_cast<unsigned long long*>(agg_smem + (1u << kAggDictBits));
    int* const vals = reinterpret_cast<int*>(agg_smem + (1u << kAggDictBits) + kAggSlots * 8);
    __shared__ AggCol s_agg[kMaxAggs];
    __shared__ PforCol s_pfor[kMaxPforCols];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#pragma unroll
    for (int i = 0; i < kMaxAggs; i++)
        if (tid == i) {
            s_agg[i] = A.agg[i];
            if (S && A.agg[i].op == kAggSum) s_agg[i].op = kAggCount;  // (the global table adds a SUM as a COUNT)
        }
#pragma unroll
    for (int i = 0; i < kMaxPforCols; i++)
        if (tid == 32 + i) s_pfor[i] = A.pfor[i];
    const int naggs = NA == 8 ? A.naggs : NA, ngroup = NG == 4 ? A.ngroup : NG, npfor = A.npfor;
    int* const V = vals + warp * nplanes * kAggSlots;
    agg_state_init<NA, S>(A, dict, keys, V, tid, lane, nplanes);
    uint32_t* const Wb = reinterpret_cast<uint32_t*>(agg_smem + agg_blocks_state_bytes(NA, nsum)) + warp * agg_blocks_warp_words(npfor, A.blk_words_cap);
    uint32_t* const dec = Wb + (A.blk_words_cap > 512 ? A.blk_words_cap : 512);  // [slot][kBlkVals]
    uint32_t* const bases = dec + npfor * kBlkVals;                                 // [slot][mini-block]
    unsigned short* const sel_w = reinterpret_cast<unsigned short*>(Wb);
    __syncthreads();

    const long long nblocks = A.nblocks, warp0 = (long long)blockIdx.x * kComputeWarps + warp, nwarps = (long long)gridDim.x * kComputeWarps;
    // block metadata in ONE round trip: lanes 0,1 = row ordinals, lanes 2+2s, 3+2s = word offsets of encoded column s
    auto load_meta = [&](long long b) -> unsigned long long {
        unsigned long long m = 0;
        if (b < nblocks) {
            if (lane < 2) m = A.row_start[b + lane];
            else if (lane < 2 + 2 * npfor) m = s_pfor[(lane - 2) >> 1].word_off[b + (lane & 1)];
            else if (BS && lane == 31) m = __ldcg(span_cnt + b);  // (BS: the block's count; 2 + 2 * kMaxPforCols < 31)
        }
        return m;
    };
    const uint8_t* gp[NG > 0 ? NG : 1];
    const uint8_t* ap[NA];
    // One block (its index and metadata): selection bits, decode, then 64 selected rows per iteration as in agg_kernel.
    auto handle = [&](long long blk, unsigned long long meta) {
        const long long R0 = (long long)__shfl_sync(0xFFFFFFFFu, meta, 0);
        const int n = (int)((long long)__shfl_sync(0xFFFFFFFFu, meta, 1) - R0);
        uint32_t myword;
        if constexpr (BS) {
            // the block's count (lane 31 of the metadata): all rows, or its own 32 words
            const unsigned bc = (unsigned)__shfl_sync(0xFFFFFFFFu, meta, 31);
            IMM3_CHECK(ctrl, bc <= (unsigned)n, 10);
            myword = bc == (unsigned)n ? 0xFFFFFFFFu : __ldg(bitmap + blk * 32 + lane);
        } else {
            const long long bit0 = R0 + 32 * lane;
            const uint32_t lo = __ldg(bitmap + (bit0 >> 5)), hi = __ldg(bitmap + (bit0 >> 5) + 1);
            myword = __funnelshift_r(lo, hi, (uint32_t)(bit0 & 31));
        }
        const int left = n - lane * 32;
        myword &= left >= 32 ? 0xFFFFFFFFu : (left <= 0 ? 0u : ((1u << left) - 1u));
        if (__ballot_sync(0xFFFFFFFFu, myword != 0u) == 0u) return;
        IMM3_CHECK(ctrl, n > 0 && n <= kBlkRows, 9);  // (the host refuses tables with larger blocks)
        __syncwarp();  // (the previous block's readers are done with the scratch)
        unsigned dense_slots = 0;  // encoded columns held in dense_prepare's form
#pragma unroll 1
        for (int s = 0; s < npfor; s++) {
            const uint32_t wo0 = (uint32_t)__shfl_sync(0xFFFFFFFFu, meta, 2 + 2 * s), wo1 = (uint32_t)__shfl_sync(0xFFFFFFFFu, meta, 3 + 2 * s);
            const DenseRegs dr = dense_issue(s_pfor[s].words, wo0, wo1, n, lane);
            if (dense_prepare(dr, dec + s * kBlkVals, lane)) {
                dense_slots |= 1u << s;
                continue;
            }
            IMM3_CHECK(ctrl, wo1 >= wo0 + 3u && (int)(wo1 - wo0) <= A.blk_words_cap, 8);  // the block's words fit the decode scratch
            bases[s * 32 + lane] = pfor_decode_warp(s_pfor[s].words, wo0, wo1, n, Wb, A.blk_words_cap, dec + s * kBlkVals, lane);
            __syncwarp();
        }
        append_selection(myword, lane, sel_w, 0u);  // (over the encoded words: every column is decoded by now)
        const unsigned cnt = __reduce_add_sync(0xFFFFFFFFu, (unsigned)__popc(myword));
        __syncwarp();
        // value of row r of the block in encoded column s
        auto enc = [&](int s, unsigned r) -> uint32_t {
            const uint32_t* const vs = dec + s * kBlkVals;
            return ((dense_slots >> s) & 1u) ? dense_value(vs, (int)r) : vs[(r >> 5) * kBlkLane + (r & 31u)] + bases[s * 32 + (r >> 5)];
        };
        // Dense cells: the words are addressed from the row R0 & ~3 (4-byte aligned whatever the width), row r of the block
        // is row r + d from there.  An encoded cell is 4 bytes at offset 0 of its word, the form agg_decode expects of it.
        const long long R0a = R0 & ~3ll;
        const unsigned d = (unsigned)(R0 - R0a);
#pragma unroll
        for (int g = 0; g < NG; g++) gp[g] = A.group[g].base + R0a * A.group[g].width;
#pragma unroll
        for (int a = 0; a < NA; a++) ap[a] = A.agg[a].base + R0a * A.agg[a].width;
        auto fetch_raw = [&](unsigned r, uint32_t (&gw)[NG > 0 ? NG : 1], uint32_t (&aw)[NA]) {
            const unsigned rd = r + d;
#pragma unroll
            for (int g = 0; g < NG; g++) {
                gw[g] = 0;
                if (NG == 4 && g >= ngroup) break;
                const unsigned w = (unsigned)A.group[g].width;
                if (A.group_pfor[g] >= 0) gw[g] = enc(A.group_pfor[g], r);
                else if (w <= 4u && (w & (w - 1u)) == 0u) gw[g] = __ldg(reinterpret_cast<const uint32_t*>(gp[g] + ((rd * w) & ~3u)));
            }
#pragma unroll
            for (int a = 0; a < NA; a++) {
                aw[a] = 0;
                if (NA == 8 && a >= naggs) break;
                if (A.agg[a].op == kAggCount) continue;
                if (A.agg_pfor[a] >= 0) aw[a] = enc(A.agg_pfor[a], r);
                else aw[a] = __ldg(reinterpret_cast<const uint32_t*>(ap[a] + ((rd * (unsigned)A.agg[a].width) & ~3u)));
            }
        };
        const unsigned ord0 = (unsigned)((blk - warp0) / nwarps) << 10;
        constexpr int NGW = NG > 0 ? NG : 1;
        unsigned s0 = lane < cnt ? sel_w[lane] : 0u, s1 = 32u + lane < cnt ? sel_w[32 + lane] : 0u;
        uint32_t g0[NGW], g1[NGW], a0[NA], a1[NA];
        fetch_raw(s0, g0, a0);
        fetch_raw(s1, g1, a1);
        for (unsigned i0 = 0; i0 < cnt; i0 += 64) {
            const bool live0 = i0 + lane < cnt, live1 = i0 + 32 + lane < cnt;
            unsigned long long k0, k1;
            int x0[NA], x1[NA];
            agg_decode<NG, NA>(A, ngroup, naggs, gp, s0 + d, g0, a0, k0, x0);
            agg_decode<NG, NA>(A, ngroup, naggs, gp, s1 + d, g1, a1, k1, x1);
            const unsigned c0 = s0, c1 = s1;
            if (i0 + 64 < cnt) {  // (the next rows' loads are in flight during this iteration's updates)
                s0 = i0 + 64 + lane < cnt ? sel_w[i0 + 64 + lane] : 0u;
                s1 = i0 + 96 + lane < cnt ? sel_w[i0 + 96 + lane] : 0u;
                fetch_raw(s0, g0, a0);
                fetch_raw(s1, g1, a1);
            }
            if (live0) agg_apply<NA, S>(A, naggs, dict, keys, V, table, overflow, s_agg, R0 + c0, ord0 + c0, k0, x0, sum_mask);
            if (live1) agg_apply<NA, S>(A, naggs, dict, keys, V, table, overflow, s_agg, R0 + c1, ord0 + c1, k1, x1, sum_mask);
        }
    };

    asm volatile("griddepcontrol.wait;" ::: "memory");  // (a no-op unless launched as a programmatic dependent)
    // 32 of the warp's blocks at a time, a lane each.  Fewer selected rows than blocks (most blocks empty): a lane tests its
    // block through the counts of the (at most two) 1024-row spans it overlaps; otherwise every block is a candidate.  (BS:
    // a block is a candidate iff its own count is not 0 - one coalesced load per lane.)  The warp then handles the
    // candidates in order, the next one's metadata in flight.  (One call site of `handle`: with two, the compiler keeps it
    // as a called function and the row loop's arrays in local memory.)
    const unsigned long long total = __ldcg(&ctrl->total);
    const bool sparse = total < (unsigned long long)nblocks;
#pragma unroll 1
    for (long long b0 = warp0; total != 0ull && b0 < nblocks; b0 += 32 * nwarps) {
        const long long b = b0 + lane * nwarps;
        bool cand = b < nblocks;
        if (BS) {
            if (cand) cand = __ldcg(span_cnt + b) != 0u;
        } else if (cand && sparse) {
            const unsigned long long r0 = A.row_start[b], r1 = A.row_start[b + 1];
            const long long q0 = (long long)(r0 >> 10), q1 = (long long)((r1 - 1) >> 10);
            const unsigned c = __ldg(span_cnt + q0) + (q1 != q0 ? __ldg(span_cnt + q1) : 0u);
            cand = c != 0u;
        }
        unsigned todo = __ballot_sync(0xFFFFFFFFu, cand);
        if (!todo) continue;
        int nsrc = __ffs((int)todo) - 1;
        long long nblk = __shfl_sync(0xFFFFFFFFu, b, nsrc);
        unsigned long long meta_n = load_meta(nblk);
#pragma unroll 1
        while (todo) {
            todo &= todo - 1u;
            const unsigned long long meta = meta_n;
            const long long blk = nblk;
            if (todo) {
                nsrc = __ffs((int)todo) - 1;
                nblk = __shfl_sync(0xFFFFFFFFu, b, nsrc);
                meta_n = load_meta(nblk);
            }
            handle(blk, meta);
        }
    }
    __syncthreads();
    auto first_row = [&](int w, unsigned ord) -> unsigned long long {
        return A.row_start[(long long)blockIdx.x * kComputeWarps + w + (long long)(ord >> 10) * nwarps] + (ord & 1023u);
    };
    if constexpr (S) agg_fold_sum<NA, 4>(A, naggs, keys, vals, nplanes, sum_mask, table, overflow, s_agg, tid, first_row);
    else agg_fold<NA>(A, naggs, keys, vals, table, overflow, s_agg, tid, first_row);
}

// Occupied slots -> out[0 .. *nout), in any order (the host sorts the groups by first_row).
__global__ void __launch_bounds__(kComputeThreads) agg_compact_kernel(const AggEntry* __restrict__ table, uint32_t slots, AggEntry* __restrict__ out,
                                                                     unsigned int* __restrict__ nout) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < slots; i += gridDim.x * blockDim.x) {
        const AggEntry e = table[i];
        if (e.key != kAggEmpty) out[atomicAdd(nout, 1u)] = e;
    }
}

// agg_merge_kernel: the global aggregate's fan-in (ProjectAggregateQueueOp, ProjectAggregateQueue.scala:21-45), behind
// agg_exchange_kernel (k_comm.cuh).  Grid-stride over the partial groups of every rank - this rank's exchange buffer in
// HBM, the peers' over NVLink - into the freshly initialised global table.  An entry's order key is (rank << 48) | its
// first row in the rank's slice: sorted by it, the groups come out in first-appearance order over the global canonical
// order (rank order, then the rank's own order) without any rank knowing another's row count.  Nothing is merged when a
// rank posted the error bit or was late: every rank then reports the same error.
__global__ void __launch_bounds__(kComputeThreads) agg_merge_kernel(const __grid_constant__ AggMergePlan M, const AggXOut* x, AggEntry* __restrict__ table,
                                                                    unsigned int* __restrict__ overflow) {
    __shared__ AggCol s_agg[kMaxAggs];
    if (threadIdx.x < kMaxAggs) {
        s_agg[threadIdx.x].base = nullptr;
        s_agg[threadIdx.x].width = 0;
        s_agg[threadIdx.x].op = M.op[threadIdx.x];
    }
    __syncthreads();
    if (x->err_mask != 0u || x->late != 0u) return;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (int r = 0; r < M.world; r++) {
        const unsigned long long n = x->counts[r];
        const AggEntry* const src = M.buf[r];
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
            const AggEntry e = src[i];
            agg_to_global<2>(table, M.slots, overflow, e.key, ((unsigned long long)r << 48) | e.first_row, e.val, s_agg, M.naggs);
        }
    }
}

// An empty table for this query's aggregates (identities: 0 for COUNT, +inf / -inf for MIN / MAX).
struct AggOps {
    int32_t op[kMaxAggs];
    int32_t naggs;
};
__global__ void __launch_bounds__(kComputeThreads) agg_init_kernel(AggEntry* __restrict__ table, uint32_t slots, AggOps ops, unsigned int* __restrict__ counters) {
    if (blockIdx.x == 0 && threadIdx.x < 2) counters[threadIdx.x] = 0;  // [0] = groups compacted, [1] = overflow flag
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < slots; i += gridDim.x * blockDim.x) {
        AggEntry e;
        e.key = kAggEmpty;
        e.first_row = ~0ull;
#pragma unroll
        for (int a = 0; a < kMaxAggs; a++) e.val[a] = a < ops.naggs ? agg_identity(ops.op[a]) : 0;
        table[i] = e;
    }
}
