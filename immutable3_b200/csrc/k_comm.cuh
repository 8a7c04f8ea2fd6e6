// k_comm.cuh - the only cross-GPU step of the path: the per-rank match counts, exchanged by the GPUs themselves over NVLink
// Fragment of kernels.cu (one translation unit, included inside namespace imm3 in the order listed there).
#pragma once

// =============================================================================================
// count_exchange_kernel (one warp): the fan-in of the reference (every worker pushes its batches into ONE queue that the
// consumer drains in order - ResultQueue.scala:7-56, Engine.scala:166,190-196) needs, across segment-sharded GPUs, only
// the match count of every rank: global order = rank order, so rank r's rows start at the sum of the counts before it
// and the LIMIT cut is a clamp on that offset (Project.scala:73-77).
//
// Lane j stores this rank's count into rank j's mailbox (a peer store through NVLink/NVSwitch: the mailbox of every rank
// is mapped into this process by cudaIpcOpenMemHandle), then polls lane j's slot of the LOCAL mailbox until rank j's
// word of this epoch has landed.  No host round trip, no library collective: the kernel is launched behind the query's
// last kernel as a programmatic dependent, so its launch latency is hidden and the host synchronises once per query.
// A word is self-describing ([63:40] epoch, [39:0] count), 8-byte aligned -> a single atomic store/load, no fences.
// =============================================================================================
__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(32) count_exchange_kernel(const __grid_constant__ CommPlan C, const ScanCtrl* ctrl, CommOut* out) {
    __shared__ unsigned long long* s_peer[kMaxWorld];
    const int lane = threadIdx.x;
#pragma unroll
    for (int i = 0; i < kMaxWorld; i++)
        if (lane == i) s_peer[i] = C.peer[i];  // (compile-time indices into the parameter bank)
    __syncwarp();
    asm volatile("griddepcontrol.wait;" ::: "memory");  // the query's kernels are complete: ctrl->total is final
    constexpr unsigned long long kCountMask = (1ull << 40) - 1ull;
    const unsigned long long ep = (unsigned long long)(C.epoch & 0xFFFFFFu);
    const unsigned long long mine = C.has_count ? (__ldcg(&ctrl->total) & kCountMask) : 0ull;
    const int slot = (int)(C.epoch % (unsigned)kCommRing) * kMaxWorld;
    if (lane < C.world) st_relaxed_sys_u64(s_peer[lane] + slot + C.rank, (ep << 40) | mine);
    unsigned long long c = 0;
    bool late = false;
    if (lane < C.world) {
        const unsigned long long* src = s_peer[C.rank] + slot + lane;
        unsigned long long v = ld_relaxed_sys_u64(src);
        if ((v >> 40) != ep) {
            const uint64_t t0 = globaltimer_ns();
            unsigned spins = 0;
            while (((v = ld_relaxed_sys_u64(src)) >> 40) != ep) {
                __nanosleep(40);
                if ((++spins & 255u) == 0 && globaltimer_ns() - t0 > C.timeout_ns) {  // never hang the GPU: report and go on
                    late = true;
                    break;
                }
            }
        }
        c = late ? 0ull : (v & kCountMask);
    }
    const unsigned any_late = __ballot_sync(0xFFFFFFFFu, late);
    unsigned long long incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long nb = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += nb;
    }
    const unsigned long long sum = __shfl_sync(0xFFFFFFFFu, incl, 31);
    if (lane < kMaxWorld) out->counts[lane] = c;
    if (lane == C.rank) {
        const unsigned long long off = incl - c, lim = (unsigned long long)C.limit;
        out->g_offset = off;
        out->g_take = off >= lim ? 0ull : (lim - off < c ? lim - off : c);
        out->g_total = sum < lim ? sum : lim;
        out->error = any_late ? 1u : 0u;
        out->world = (unsigned)C.world;
    }
    if (C.pub) {  // publish: the whole control block goes to the host's pinned copy, then the sequence number the host polls
        volatile CtrlBlock* hp = C.pub;
        if (lane < kMaxWorld) hp->x.counts[lane] = c;
        if (lane == C.rank) {
            const unsigned long long off = incl - c, lim = (unsigned long long)C.limit;
            hp->x.g_offset = off;
            hp->x.g_take = off >= lim ? 0ull : (lim - off < c ? lim - off : c);
            hp->x.g_total = sum < lim ? sum : lim;
            hp->x.error = any_late ? 1u : 0u;
            hp->x.world = (unsigned)C.world;
        }
        if (lane == 0) {
            hp->c.total = __ldcg(&ctrl->total);
            hp->c.error = __ldcg(&ctrl->error);
            hp->c.dense_rows = __ldcg(&ctrl->dense_rows);
        }
        __threadfence_system();
        __syncwarp();
        if (lane == 0) asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(&C.pub->pub_seq), "l"((C.pub_seq & 0x7FFFFFull) << 41) : "memory");
    }
}

// =============================================================================================
// agg_exchange_kernel (one warp): the fan-in of a global aggregate (ProjectAggregateQueueOp, ProjectAggregateQueue.scala:
// 9-54).  Every rank has compacted its partial groups into its own exchange buffer (plan.hpp kAggXchgOff) before this
// kernel; what travels through the mailbox ring is one word per rank, [63:40] epoch, [32] error bit, [31:0] group count,
// in the ring slot and epoch scheme of count_exchange_kernel (the two kernels share db->comm_epoch).
// Unlike the count, the word announces DATA the peers then read over NVLink, so it is not self-describing: the poster
// fences at system scope and stores with release semantics (its compacted groups are visible to any reader that sees
// the word), the poller loads with acquire semantics at system scope before agg_merge_kernel - queued behind this kernel
// on the same stream - reads a peer's buffer.  Error bit: this rank's local table overflowed, its filter / aggregation
// watchdog fired, or its slice refuses the query (plan.refused); every rank sees every bit, so every rank returns the
// same status without waiting for anything.
// =============================================================================================
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(32) agg_exchange_kernel(const __grid_constant__ AggXPlan P, const unsigned int* counters, const ScanCtrl* ctrl,
                                                          AggXOut* out) {
    __shared__ unsigned long long* s_peer[kMaxWorld];
    const int lane = threadIdx.x;
#pragma unroll
    for (int i = 0; i < kMaxWorld; i++)
        if (lane == i) s_peer[i] = P.peer[i];
    __syncwarp();
    asm volatile("griddepcontrol.wait;" ::: "memory");  // the local aggregation and its compaction are complete
    const unsigned long long ep = (unsigned long long)(P.epoch & 0xFFFFFFu);
    unsigned long long mine = P.refused ? kAggXchgError : 0ull;
    if (P.has_local) {
        mine = (unsigned long long)__ldcg(&counters[0]);
        if (__ldcg(&counters[1]) != 0u || __ldcg(&ctrl->error) != 0u) mine = kAggXchgError;
    }
    const int slot = (int)(P.epoch % (unsigned)kCommRing) * kMaxWorld;
    if (lane < P.world) {
        __threadfence_system();  // (the compaction kernel's stores to this rank's exchange buffer, before the word)
        st_release_sys_u64(s_peer[lane] + slot + P.rank, (ep << 40) | mine);
    }
    unsigned long long w = 0;
    bool late = false;
    if (lane < P.world) {
        const unsigned long long* src = s_peer[P.rank] + slot + lane;
        unsigned long long v = ld_acquire_sys_u64(src);
        if ((v >> 40) != ep) {
            const uint64_t t0 = globaltimer_ns();
            unsigned spins = 0;
            while (((v = ld_acquire_sys_u64(src)) >> 40) != ep) {
                __nanosleep(40);
                if ((++spins & 255u) == 0 && globaltimer_ns() - t0 > P.timeout_ns) {  // never hang the GPU: report and go on
                    late = true;
                    break;
                }
            }
        }
        w = late ? kAggXchgError : (v & ((1ull << 40) - 1ull));
    }
    const unsigned any_late = __ballot_sync(0xFFFFFFFFu, late);
    const unsigned errs = __ballot_sync(0xFFFFFFFFu, lane < P.world && (w & kAggXchgError) != 0ull);
    if (lane < kMaxWorld) out->counts[lane] = (w & kAggXchgError) ? 0ull : (w & 0xFFFFFFFFull);
    if (lane == 0) {
        out->err_mask = errs;
        out->late = any_late ? 1u : 0u;
    }
    __threadfence_system();  // (every peer word this warp acquired is ordered before the merge kernel's reads of its buffer)
}
