// engine.cu — the C ABI of include/imm3.h: SegmentManager upload path + query execution.
//
//  imm3_open        = new SegmentManager(dataDir)            SegmentManager.scala:20-112
//                     + staging of every owned segment into HBM through pinned async copies
//  imm3_query*      = Engine.execute, Project branch         Engine.scala:158-198
//                     = ScanOp -> SelectOp* -> ProjectOp      Scan.scala, Select.scala, Project.scala
//  result accessors = Iterator[Row] / Row                    Project.scala:17-81, Record.scala:3-14
//
// HBM layout: one arena per (table, column) holding the owned segments' block bytes back to back in
// canonical order.  For DENSE_* columns that is a flat array of values indexed by the canonical row
// ordinal (blocks and segments need no per-block metadata on the device); the arena is padded to a
// whole tile so the last TMA bulk copy stays in bounds.  For PFOR_INT columns it is the stream of
// big-endian words plus a word offset per block.
//
// There is no CPU execution path in this file: every query runs the CUDA kernels of kernels.cu.
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fcntl.h>
#include <time.h>
#include <unistd.h>

#include <atomic>
#include <cerrno>
#include <charconv>
#include <cmath>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "kernels.hpp"
#include "plan.hpp"
#include "store.hpp"

using namespace imm3;

#define CUDA_TRY(expr)                                                                                     \
    do {                                                                                                   \
        cudaError_t e_ = (expr);                                                                           \
        if (e_ != cudaSuccess)                                                                             \
            return fail(e_ == cudaErrorMemoryAllocation ? IMM3_ERR_OOM : IMM3_ERR_CUDA, "%s: %s (%s:%d)", #expr, \
                        cudaGetErrorString(e_), __FILE__, __LINE__);                                       \
    } while (0)

namespace {

struct Buf {
    void* p = nullptr;
    size_t cap = 0;
};

inline double now_us() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec * 1e6 + (double)ts.tv_nsec * 1e-3;
}

// Grow-only cache of device / pinned-host buffers: result columns are handed back on
// imm3_result_free and reused by the next query (cudaMalloc / cudaMallocHost cost milliseconds).
struct BufPool {
    bool pinned_host = false;
    std::vector<Buf> free_list;
    int acquire(size_t bytes, Buf* out) {
        if (bytes < 256) bytes = 256;
        int best = -1;
        for (size_t i = 0; i < free_list.size(); i++)
            if (free_list[i].cap >= bytes && (best < 0 || free_list[i].cap < free_list[(size_t)best].cap)) best = (int)i;
        if (best >= 0) {
            *out = free_list[(size_t)best];
            free_list.erase(free_list.begin() + best);
            return 0;
        }
        // drop the largest cached buffer that is too small, so the pool does not accumulate
        if (!free_list.empty()) {
            size_t big = 0;
            for (size_t i = 1; i < free_list.size(); i++)
                if (free_list[i].cap > free_list[big].cap) big = i;
            if (pinned_host) cudaFreeHost(free_list[big].p); else cudaFree(free_list[big].p);
            free_list.erase(free_list.begin() + (long)big);
        }
        size_t cap = bytes + bytes / 8;
        cap = (cap + 255) & ~(size_t)255;
        void* p = nullptr;
        cudaError_t e = pinned_host ? cudaMallocHost(&p, cap) : cudaMalloc(&p, cap);
        if (e != cudaSuccess) {
            cudaGetLastError();
            release_all();
            e = pinned_host ? cudaMallocHost(&p, cap) : cudaMalloc(&p, cap);
        }
        if (e != cudaSuccess)
            return fail(IMM3_ERR_OOM, "%s of %zu bytes failed: %s", pinned_host ? "cudaMallocHost" : "cudaMalloc", cap,
                        cudaGetErrorString(e));
        out->p = p;
        out->cap = cap;
        return 0;
    }
    void release(Buf b) {
        if (b.p) free_list.push_back(b);
    }
    void release_all() {
        for (auto& b : free_list) {
            if (pinned_host) cudaFreeHost(b.p); else cudaFree(b.p);
        }
        free_list.clear();
    }
};

}  // namespace

struct imm3_db {
    std::string dir;
    int device = 0, rank = 0, world = 1;
    uint32_t flags = 0;
    bool host_only = false;
    std::vector<TableStore> tables;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t copy_stream = nullptr;      // imm3_result_fetch_async: device->host copies overlap the next query's staging
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_mid = nullptr;
    ScanCtrl* d_ctrl = nullptr;   // first member of a device CtrlBlock (ScanCtrl + CommOut)
    CtrlBlock* h_ctrl = nullptr;  // pinned copy, refreshed once per launch sequence
    unsigned long long pub_seq = 0;  // publish (plan.hpp): sequence number of the last query whose last kernel writes h_ctrl itself
    unsigned long long ev_seq = 0, query_seq = 0;  // the query ev0 / ev1 were recorded for (device times are read lazily)
    int live_results = 0;         // imm3_result objects that still point at this db (imm3_close refuses while > 0)
    // Count exchange over NVLink peer memory (imm3_comm_*): the local mailbox, every rank's mailbox as mapped here.
    unsigned long long* d_mailbox = nullptr;
    unsigned long long* comm_peer[kMaxWorld] = {};
    bool comm_on = false;
    uint32_t comm_epoch = 0;
    uint32_t agg_seq = 0;  // global aggregates exchanged since imm3_comm_connect (identical on all ranks): exchange buffer agg_seq & 1
    unsigned long long comm_timeout_ns = 30000000000ull;
    unsigned long long* d_status = nullptr;
    size_t status_cap = 0;
    uint32_t epoch = 0;
    int num_sms = 0;
    BufPool dev_pool, host_pool;
    Buf d_bitmap, h_bitmap;
    Buf d_span_cnt, d_tile_cnt, d_tile_off;  // multi-pass pipeline scratch (grow-only)
    Buf d_agg_table, d_agg_out, d_agg_cnt;   // aggregation: global hash table, compacted groups, [groups, overflow] counters
    Buf h_agg_out;                           // pinned read-back of the compacted groups
    Buf d_work;                              // blocks_prune_kernel: work list of tiles for the filter kernel ([0] = count)
    Buf d_scan_part;                         // offset_scan_kernel: epoch-tagged chunk sums (zeroed when (re)allocated)
    Buf d_tile_list;                         // offset_scan_kernel (block pipeline): the non-empty tiles, for the emit kernel
    Buf d_grp_sum;                           // blocks_group_emit_kernel: match counts per group of 1024 blocks (zero between queries)
    Buf d_or_bitmap, d_or_cnt;               // real OR over encoded columns: a later term's block selection (words, counts)
    uint32_t scan_epoch = 0;
    Buf d_trace;                             // IMM3_TRACE debugging buffer
    // Emit-kernel feedback: result density class (1 dense, 0 sparse) last seen for a query shape (table, filter
    // columns and kinds, select list).  A known class launches only the matching emit kernel; both kernels are correct
    // for any result, so a stale hint costs time, never rows.
    std::unordered_map<std::string, int> emit_hint;
    std::string explain_buf;
};

struct imm3_result {
    imm3_db* db = nullptr;
    int ncols = 0;
    std::vector<std::string> names;
    std::vector<int> types, widths;
    std::vector<Buf> d_cols, h_cols;
    int64_t local_count = 0;
    int64_t g_offset = 0, g_take = 0, g_total = 0;  // after the count exchange (single handle: 0, local_count, local_count)
    int world = 1;
    int64_t rank_counts[kMaxWorld] = {};
    int agg_first_col = -1;  // aggregate result: index of the first aggregate column (rows live in host buffers only)
    uint32_t avg_cols = 0;   // bit a: aggregate column a is an AVG (printed with every digit, not as an integral MIN / MAX)
    int64_t fetched = 0;
    int64_t pending = -1;        // rows of an imm3_result_fetch_async still in flight (-1 = none)
    cudaEvent_t copied = nullptr;  // recorded on the copy stream after the last device->host copy
    double device_ms = 0;            // < 0: not read yet (timing_seq says which query's events hold it)
    unsigned long long timing_seq = 0;
    double stage_ms[2] = {0, 0};
    double host_us[5] = {0, 0, 0, 0, 0};  // wall clock inside imm3_query_begin: plan, buffers + device plan, launches, wait for the GPU, epilogue
    std::string route;  // imm3_result_route: "kernel[/key=value...];kernel..." in launch order, an entry per kernel launch
    int64_t alg_bytes = 0;
};

namespace {

TableStore* find_table(imm3_db* db, const char* name) {
    if (!name) { set_error("table name is NULL"); return nullptr; }
    for (auto& t : db->tables)
        if (t.meta.name == name) return &t;
    // SegmentManager.getTable, SegmentManager.scala:89-92
    fail(IMM3_ERR_NOT_FOUND, "Table %s does not exist in SegmentManager", name);
    return nullptr;
}

int use_device(imm3_db* db) {
    if (db->host_only) return fail(IMM3_ERR_STATE, "handle was opened with IMM3_OPEN_HOST_ONLY: no device work (there is no CPU fallback)");
    CUDA_TRY(cudaSetDevice(db->device));
    return 0;
}

// What one query reports about its launches, created by the entry point and passed down.
struct Run {
    std::string route;     // imm3_result_route: one entry per queued kernel, in launch order, recorded on the host only
    const char* tag = "";  // appended to every entry: "/prefix" while phase A of a small LIMIT is queued
    double t_launched = 0, t_synced = 0;  // host stamps of the last phase: last launch queued, GPU done
    bool eager_times = false;             // a two-phase LIMIT query adds its phases' device times up: no lazy reading
    double device_ms = 0, stage_ms[2] = {0, 0};
    void note(const std::string& name) {
        if (!route.empty()) route += ';';
        route += name;
        route += tag;
    }
};

// ---- SegmentManager upload path: files -> pinned staging -> HBM --------------------------------
// The owned slice of every column is one contiguous byte range in canonical order (its segments' block bytes back to
// back).  It is cut into pieces of at most kStageBytes; a pool of I/O threads takes pieces off a shared counter, pread()s
// each piece from the segment files (page cache / tmpfs) STRAIGHT into one of its two pinned staging buffers - no mmap,
// no intermediate copy - and queues the host->device copy on its own stream, so file reads, PCIe copies of different
// threads and the refill of the other buffer all overlap.  (Round 1: one thread memcpy-ing mmap pages into a 2 x 32 MiB
// ring - 1.4 GB/s.)  The same piece reader fills the pinned host mirror that imm3_reupload re-stages from.
constexpr size_t kStageBytes = 4u << 20;
constexpr int kMaxStageThreads = 12;

struct Piece {
    ColumnStore* col;
    size_t off;    // byte offset inside the column's payload
    size_t bytes;
    size_t seg;    // first segment file touched, and the offset inside it
    size_t seg_off;
};

void cut_pieces(ColumnStore& col, std::vector<Piece>* out) {
    size_t seg = 0, seg_off = 0, off = 0;
    const size_t total = (size_t)col.encoded_bytes;
    while (off < total) {
        while (seg < col.segs.size() && seg_off >= (size_t)col.segs[seg].nbytes) { seg++; seg_off = 0; }
        const size_t take = std::min(kStageBytes, total - off);
        out->push_back(Piece{&col, off, take, seg, seg_off});
        size_t left = take;  // advance (seg, seg_off) by `take` bytes
        while (left) {
            const size_t in_seg = (size_t)col.segs[seg].nbytes - seg_off;
            if (left < in_seg) { seg_off += left; left = 0; }
            else { left -= in_seg; seg++; seg_off = 0; }
        }
        off += take;
    }
}

// pread the bytes of one piece into dst (host memory).
int read_piece(const Piece& pc, uint8_t* dst) {
    size_t seg = pc.seg, seg_off = pc.seg_off, done = 0;
    while (done < pc.bytes) {
        const SegmentFile& sf = pc.col->segs[seg];
        const size_t take = std::min(pc.bytes - done, (size_t)sf.nbytes - seg_off);
        if (take) {
            int fd = ::open(sf.path.c_str(), O_RDONLY);
            if (fd < 0) return fail(IMM3_ERR_IO, "open %s: %s", sf.path.c_str(), strerror(errno));
            size_t got = 0;
            while (got < take) {
                const ssize_t r = ::pread(fd, dst + done + got, take - got, (off_t)(seg_off + got));
                if (r <= 0) {
                    ::close(fd);
                    return fail(IMM3_ERR_IO, "read %s: %s", sf.path.c_str(), r < 0 ? strerror(errno) : "file is shorter than its block offsets");
                }
                got += (size_t)r;
            }
            ::close(fd);
        }
        done += take;
        seg++;
        seg_off = 0;
    }
    return 0;
}

// Run `pieces` on the I/O pool.  to_device: through pinned staging buffers into the columns' arenas; otherwise straight into
// the columns' pinned host mirrors.
int run_pieces(imm3_db* db, const std::vector<Piece>& pieces, bool to_device) {
    if (pieces.empty()) return 0;
    const int nthreads = std::max(1, std::min<int>(std::min(io_threads(), kMaxStageThreads), (int)pieces.size()));
    // Pinning memory is the slow part of a staged upload (tens of ms per 16 MiB, serialised inside the driver): ONE pinned
    // block for all staging threads, allocated on first use and kept for the life of the process.
    uint8_t* pool_base = nullptr;
    if (to_device) {
        static std::mutex pin_mu;
        static uint8_t* pin_block = nullptr;
        std::lock_guard<std::mutex> lock(pin_mu);
        if (!pin_block) CUDA_TRY(cudaHostAlloc(&pin_block, (size_t)kMaxStageThreads * 2 * kStageBytes, cudaHostAllocPortable));
        pool_base = pin_block;
    }
    static std::mutex run_mu;  // (one staged upload at a time per process: the pinned block is shared)
    std::unique_lock<std::mutex> run_lock(run_mu, std::defer_lock);
    if (to_device) run_lock.lock();
    std::atomic<size_t> next(0);
    std::atomic<int> first_rc(0);
    std::atomic<long long> us_alloc(0), us_read(0), us_wait(0);  // summed over the threads (IMM3_OPEN_TRACE)
    std::mutex mu;
    std::string why;
    auto report = [&](int rc) {
        std::lock_guard<std::mutex> lock(mu);
        if (!first_rc.load()) {
            why = last_error();
            first_rc.store(rc);
        }
    };
    auto work = [&](int tid) {
        uint8_t* stage[2] = {nullptr, nullptr};
        cudaEvent_t ev[2] = {nullptr, nullptr};
        cudaStream_t st = nullptr;
        auto body = [&]() -> int {
            if (to_device) {
                const double ta = now_us();
                CUDA_TRY(cudaSetDevice(db->device));
                CUDA_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
                for (int i = 0; i < 2; i++) {
                    stage[i] = pool_base + ((size_t)tid * 2 + (size_t)i) * kStageBytes;  // (carved out of the process-wide pinned block)
                    CUDA_TRY(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
                }
                us_alloc += (long long)(now_us() - ta);
            }
            int cur = 0;
            bool used[2] = {false, false};
            for (;;) {
                const size_t i = next.fetch_add(1);
                if (i >= pieces.size() || first_rc.load()) break;
                const Piece& pc = pieces[i];
                if (!to_device) {
                    int rc = read_piece(pc, pc.col->h_mirror + pc.off);
                    if (rc) return rc;
                    continue;
                }
                const double tw = now_us();
                if (used[cur]) CUDA_TRY(cudaEventSynchronize(ev[cur]));  // the buffer's previous copy has retired
                const double tr = now_us();
                int rc = read_piece(pc, stage[cur]);
                if (rc) return rc;
                us_wait += (long long)(tr - tw);
                us_read += (long long)(now_us() - tr);
                CUDA_TRY(cudaMemcpyAsync(pc.col->d_arena + pc.off, stage[cur], pc.bytes, cudaMemcpyHostToDevice, st));
                CUDA_TRY(cudaEventRecord(ev[cur], st));
                used[cur] = true;
                cur ^= 1;
            }
            if (st) CUDA_TRY(cudaStreamSynchronize(st));
            return 0;
        };
        const int rc = body();
        if (rc) report(rc);
        if (st) cudaStreamSynchronize(st);
        for (int i = 0; i < 2; i++)
            if (ev[i]) cudaEventDestroy(ev[i]);
        if (st) cudaStreamDestroy(st);
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < nthreads; t++) pool.emplace_back(work, t);
    work(0);
    for (auto& th : pool) th.join();
    if (int rc = first_rc.load()) return fail(rc, "%s", why.c_str());
    if (getenv("IMM3_OPEN_TRACE") && to_device)
        fprintf(stderr, "[imm3_open] %d staging threads; per thread: pinned buffers %.1f ms, file reads %.1f ms, waiting for copies %.1f ms\n", nthreads,
                us_alloc.load() * 1e-3 / nthreads, us_read.load() * 1e-3 / nthreads, us_wait.load() * 1e-3 / nthreads);
    return 0;
}

int upload_all(imm3_db* db) {
    const bool otrace = getenv("IMM3_OPEN_TRACE") != nullptr;
    const double t0 = now_us();
    std::vector<Piece> pieces;
    for (auto& t : db->tables) {
        for (auto& col : t.cols) {
            const bool dense = col.meta.codec != IMM3_CODEC_PFOR_INT;
            const size_t payload = (size_t)col.encoded_bytes;
            size_t arena = dense ? (size_t)((t.nrows + kDenseMaxTileRows - 1) / kDenseMaxTileRows) * kDenseMaxTileRows * (size_t)col.meta.width : payload;
            arena += 256;
            CUDA_TRY(cudaMalloc(&col.d_arena, arena));
            col.arena_bytes = arena;
            CUDA_TRY(cudaMemsetAsync(col.d_arena + payload, 0, arena - payload, db->stream));  // zero padding up to a whole tile
            if (!dense) {
                CUDA_TRY(cudaMalloc(&col.d_word_off, col.word_off.size() * sizeof(uint32_t) + 256));  // (+256: the filter kernels' TMA reads up to 36 entries per tile)
                CUDA_TRY(cudaMemcpyAsync(col.d_word_off, col.word_off.data(), col.word_off.size() * sizeof(uint32_t),
                                         cudaMemcpyHostToDevice, db->stream));
            }
            cut_pieces(col, &pieces);
        }
        CUDA_TRY(cudaMalloc(&t.d_row_start, t.row_start.size() * sizeof(uint64_t) + 512));  // (+512: ... and up to 34 row ordinals)
        CUDA_TRY(cudaMemcpyAsync(t.d_row_start, t.row_start.data(), t.row_start.size() * sizeof(uint64_t),
                                 cudaMemcpyHostToDevice, db->stream));
    }
    const double t1 = now_us();
    int rc = run_pieces(db, pieces, true);
    cudaError_t e = cudaStreamSynchronize(db->stream);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(IMM3_ERR_CUDA, "upload: %s", cudaGetErrorString(e));
    if (otrace) {
        size_t bytes = 0;
        for (auto& pc : pieces) bytes += pc.bytes;
        fprintf(stderr, "[imm3_open] arenas allocated in %.1f ms; %zu pieces, %.1f MB staged in %.1f ms = %.1f GB/s\n", (t1 - t0) * 1e-3, pieces.size(),
                bytes * 1e-6, (now_us() - t1) * 1e-3, bytes * 1e-3 / (now_us() - t1));
    }
    const double t2 = now_us();
    // Block statistics of the encoded INT columns (exact min / max per block, one decode pass on the GPU): what the stubs
    // SegmentStats / check() of the reference (Segment.scala:18-30) were meant to hold.  Range queries prune with them.
    if (!(db->flags & IMM3_OPEN_NO_STATS)) {
        for (auto& t : db->tables) {
            if (t.max_block_rows > 1024 || t.nblocks == 0) continue;  // (the warp-per-block decoder takes blocks of <= 1024 rows)
            for (auto& col : t.cols) {
                if (col.meta.codec != IMM3_CODEC_PFOR_INT) continue;
                CUDA_TRY(cudaMalloc(&col.d_stats, (size_t)t.nblocks * sizeof(BlockStat)));
                PforCol pc;
                pc.words = reinterpret_cast<const uint32_t*>(col.d_arena);
                pc.word_off = col.d_word_off;
                CUDA_TRY(launch_block_stats(pc, t.d_row_start, t.nblocks, col.max_block_words, db->num_sms, (BlockStat*)col.d_stats, db->stream));
            }
        }
        CUDA_TRY(cudaStreamSynchronize(db->stream));
        if (otrace) fprintf(stderr, "[imm3_open] block statistics in %.1f ms\n", (now_us() - t2) * 1e-3);
    }
    return 0;
}

// Pinned host mirror of a column's payload, built on first use (imm3_reupload): the open path never pins a whole column.
int ensure_mirror(imm3_db* db, ColumnStore& col) {
    if (col.h_mirror || !col.encoded_bytes) return 0;
    CUDA_TRY(cudaMallocHost(&col.h_mirror, (size_t)col.encoded_bytes));
    std::vector<Piece> pieces;
    cut_pieces(col, &pieces);
    return run_pieces(db, pieces, false);
}

void free_device_side(imm3_db* db) {
    if (db->host_only) return;
    cudaSetDevice(db->device);
    if (db->stream) cudaStreamSynchronize(db->stream);
    for (auto& t : db->tables) {
        for (auto& c : t.cols) {
            if (c.d_arena) cudaFree(c.d_arena);
            if (c.d_word_off) cudaFree(c.d_word_off);
            if (c.d_stats) cudaFree(c.d_stats);
            if (c.h_mirror) cudaFreeHost(c.h_mirror);
        }
        if (t.d_row_start) cudaFree(t.d_row_start);
    }
    db->dev_pool.release_all();
    db->host_pool.release_all();
    if (db->d_bitmap.p) cudaFree(db->d_bitmap.p);
    if (db->d_span_cnt.p) cudaFree(db->d_span_cnt.p);
    if (db->d_tile_cnt.p) cudaFree(db->d_tile_cnt.p);
    if (db->d_tile_off.p) cudaFree(db->d_tile_off.p);
    if (db->d_trace.p) cudaFree(db->d_trace.p);
    if (db->d_scan_part.p) cudaFree(db->d_scan_part.p);
    if (db->d_tile_list.p) cudaFree(db->d_tile_list.p);
    if (db->d_grp_sum.p) cudaFree(db->d_grp_sum.p);
    if (db->d_or_bitmap.p) cudaFree(db->d_or_bitmap.p);
    if (db->d_or_cnt.p) cudaFree(db->d_or_cnt.p);
    if (db->d_work.p) cudaFree(db->d_work.p);
    if (db->d_agg_table.p) cudaFree(db->d_agg_table.p);
    if (db->d_agg_out.p) cudaFree(db->d_agg_out.p);
    if (db->d_agg_cnt.p) cudaFree(db->d_agg_cnt.p);
    if (db->h_agg_out.p) cudaFreeHost(db->h_agg_out.p);
    if (db->h_bitmap.p) cudaFreeHost(db->h_bitmap.p);
    if (db->d_status) cudaFree(db->d_status);
    if (db->d_ctrl) cudaFree(db->d_ctrl);
    if (db->h_ctrl) cudaFreeHost(db->h_ctrl);
    for (int i = 0; i < kMaxWorld; i++)
        if (db->comm_peer[i] && db->comm_peer[i] != db->d_mailbox) cudaIpcCloseMemHandle(db->comm_peer[i]);
    if (db->d_mailbox) cudaFree(db->d_mailbox);
    if (db->ev0) cudaEventDestroy(db->ev0);
    if (db->ev1) cudaEventDestroy(db->ev1);
    if (db->ev_mid) cudaEventDestroy(db->ev_mid);
    if (db->copy_stream) cudaStreamDestroy(db->copy_stream);
    if (db->own_stream) cudaStreamDestroy(db->own_stream);
    cudaGetLastError();
}

// ---- query planning on top of the logical plan --------------------------------------------------
// The kernels of a query, chosen once per plan (choose_route); sizing (fill_scan_plan) and launching (run_scan_once) follow it.
enum class Pipeline {
    kDense,       // dense table: filter kernel over the row space -> offset scan -> emit kernels
    kRowSpace,    // block table, no predicate on an encoded column: the same filter kernel over the row space (dense columns are
                  // contiguous in HBM whatever the block framing) -> block emit kernel (decodes only blocks with surviving rows)
    kBlocks,      // block table: [blocks_prune ->] block filter kernel -> offset scan + block emit, scan-emit or group emit
    kSinglePass,  // block table: scan_blocks, one kernel with a look-back chain (selection bitmaps, blocks of more than 1024 rows)
};

struct Prepared {
    TableStore* table = nullptr;
    LogicalPlan lp;
    bool for_bitmap = false;    // imm3_filter_bitmap: the selection bitmap is the result
    Pipeline pipeline = Pipeline::kDense;
    BlockFilter block_filter = BlockFilter::kMini;  // kBlocks: the filter kernel
    bool prune = false;         // kBlocks: every predicate is a range on an encoded column with block statistics: blocks_prune_kernel first
    PrunePlan pp;
    std::vector<int> pfor_cols;  // table columns of sp.pfor, in slot order
    int64_t prefix_blocks = 0;  // small LIMIT on a block table: the pipeline first runs over this many leading blocks (0 = no prefix)
    int64_t prefix_rows = 0;    // small LIMIT on a dense table: ... over this many leading rows (a multiple of the tile size)
    std::string shape_key;    // key of imm3_db::emit_hint
    ScanPlan sp;
    KernelShape front;        // the filter kernel (row space or block), or scan_blocks; grid: its persistent grid (plan_grid)
    EmitShape emit;           // kDense: the gather and streaming emit kernels
    KernelShape blocks_emit;  // kRowSpace, kBlocks: the block emit kernel
    // real OR (imm3_query_begin_dnf): the second and later conjunctions of the disjunction - their filter kernels run behind this
    // plan's and OR their rows into its bitmap; counts, offsets and the emit kernels then see the union.  On kBlocks (a term
    // with a predicate on an encoded column, IMM3_DNF_ENCODED_FILTER) each term's block filter front runs into the term
    // buffers and blocks_or_merge_kernel ORs that selection into this plan's.
    std::vector<std::unique_ptr<Prepared>> or_terms;
};

bool is_pfor(const TableStore& t, int ci) { return t.cols[(size_t)ci].meta.codec == IMM3_CODEC_PFOR_INT; }

// Slot of column ci among the distinct sorted-int-codec columns a kernel decodes (`cols`, in slot order); -1: not encoded.
int pfor_slot(const TableStore& t, std::vector<int>* cols, int ci) {
    if (!is_pfor(t, ci)) return -1;
    for (size_t i = 0; i < cols->size(); i++)
        if ((*cols)[i] == ci) return (int)i;
    cols->push_back(ci);
    return (int)cols->size() - 1;
}

// The block filter kernel of a query with a predicate on an encoded column (kBlocks, and aggregates over such predicates):
// the only predicate is a range on one encoded column (C4): the quad or lane kernel if that column's tiles fit them
// (single_range_block_filter).  Otherwise (and with IMM3_NO_QUAD) the mini-block kernel.
void choose_block_filter(Prepared* pr) {
    const TableStore& t = *pr->table;
    const LogicalPlan& lp = pr->lp;
    pr->block_filter = BlockFilter::kMini;
    if (lp.filters.size() == 1 && is_pfor(t, lp.filters[0].col_idx) && lp.filters[0].kind == kFilterI32Range && !getenv("IMM3_NO_QUAD"))
        pr->block_filter = single_range_block_filter(t.cols[(size_t)lp.filters[0].col_idx].max_tile32_bytes);
}

// Pipeline and block filter kernel of a query, from the table's codecs and block sizes, the logical plan, whether a selection
// bitmap is wanted and the switches IMM3_PATH=fused, IMM3_NO_HYBRID, IMM3_NO_QUAD, IMM3_NO_LANE and IMM3_OPEN_FORCE_BLOCKS
// (tests: cross-check the dense and block kernels).
void choose_route(const imm3_db* db, Prepared* pr) {
    const TableStore& t = *pr->table;
    const LogicalPlan& lp = pr->lp;
    pr->block_filter = BlockFilter::kMini;
    if (!lp.uses_pfor && !(db->flags & IMM3_OPEN_FORCE_BLOCKS)) {
        pr->pipeline = Pipeline::kDense;
        return;
    }
    const char* path = getenv("IMM3_PATH");
    if (pr->for_bitmap || t.max_block_rows > 1024 || (path && !strcmp(path, "fused"))) {
        pr->pipeline = Pipeline::kSinglePass;
        return;
    }
    bool filters_dense = true;
    for (auto& f : lp.filters) filters_dense = filters_dense && !is_pfor(t, f.col_idx);
    pr->pipeline = filters_dense && !getenv("IMM3_NO_HYBRID") ? Pipeline::kRowSpace : Pipeline::kBlocks;
    if (pr->pipeline == Pipeline::kBlocks && !filters_dense) choose_block_filter(pr);
}

// imm3_explain's name of the kernels
const char* explain_kernel(const imm3_db* db, const Prepared& pr) {
    if (pr.lp.always_empty) return "none(always_empty)";
    if (pr.pipeline != Pipeline::kDense) return "blocks_filter -> blocks_emit";
    return (db->flags & IMM3_OPEN_NO_TMA) ? "filter(direct) -> emit" : "filter(tma) -> emit";
}

int prepare(imm3_db* db, const char* table, const imm3_pred* preds, int npreds, const char* const* proj, int nproj,
            int64_t limit, bool for_bitmap, Prepared* pr) {
    pr->table = find_table(db, table);
    if (!pr->table) return IMM3_ERR_NOT_FOUND;
    int rc = build_logical_plan(pr->table->meta, preds, npreds, proj, nproj, limit, &pr->lp);
    if (rc) return rc;
    pr->for_bitmap = for_bitmap;
    choose_route(db, pr);
    pr->shape_key = pr->table->meta.name + "|";
    for (auto& f : pr->lp.filters) pr->shape_key += std::to_string(f.col_idx) + ":" + std::to_string(f.kind) + ",";
    pr->shape_key += "|";
    for (int c : pr->lp.proj) pr->shape_key += std::to_string(c) + ",";
    return 0;
}

// A small LIMIT is served "prefix first": the multi-pass pipelines have no early exit, so phase A scans a leading part of the
// slice (64 rows per requested row, at least 4 M rows) and phase B the whole slice only if that did not fill the LIMIT.  (The
// single-pass kernel does stop early, but its look-back chain costs 13 ns per block when the rows come late.)  With a
// communicator every rank must run the same rounds, so the policy depends only on the query: phase A everywhere (a rank whose
// slice is too small for a prefix scans all of it), then - unless RANK 0's phase A alone fills the LIMIT, in which case the
// global result is its first `limit` rows - phase B everywhere.
bool small_limit(const LogicalPlan& lp) { return lp.limit > 0 && lp.limit <= (1 << 20) && !getenv("IMM3_NO_PREFIX"); }
// rows phase A wants (0: no prefix phase)
int64_t prefix_rows_wanted(const LogicalPlan& lp) {
    if (!small_limit(lp)) return 0;
    const int64_t min_rows = getenv("IMM3_PREFIX_ROWS") ? std::max(1024, atoi(getenv("IMM3_PREFIX_ROWS"))) : (4 << 20);  // (tests shrink it)
    return std::max<int64_t>(min_rows, lp.limit * 64);
}
// ... as leading blocks of a block table (0: no prefix phase - the prefix would be half the table or more)
int64_t prefix_blocks_wanted(const Prepared& pr) {
    const int64_t nb = (prefix_rows_wanted(pr.lp) + 1023) / 1024;
    return nb * 2 <= pr.table->nblocks ? nb : 0;
}

// The part of every device plan that does not depend on the pipeline: columns, literals, encoded-column slots, the L2 hint,
// the epoch and IMM3_DEBUG.
int plan_columns(imm3_db* db, Prepared* pr) {
    TableStore& t = *pr->table;
    const LogicalPlan& lp = pr->lp;
    ScanPlan& sp = pr->sp;
    std::memset(&sp, 0, sizeof sp);
    sp.nrows = t.nrows;
    sp.limit = lp.limit > 0 ? lp.limit : INT64_MAX;
    sp.row_start = t.d_row_start;
    sp.max_block_rows = t.max_block_rows;
    sp.nfilter = (int)lp.filters.size();
    sp.nproj = (int)lp.proj.size();
    pr->pfor_cols.clear();
    int lit_at = 0;
    for (int i = 0; i < sp.nfilter; i++) {
        const LogicalFilter& lf = lp.filters[(size_t)i];
        const ColumnStore& c = t.cols[(size_t)lf.col_idx];
        FilterCol& f = sp.filter[i];
        f.width = c.meta.width;
        f.kind = lf.kind;
        f.pfor_slot = pfor_slot(t, &pr->pfor_cols, lf.col_idx);
        f.base = f.pfor_slot >= 0 ? nullptr : c.d_arena;
        f.smem_off = -1;
        if (lf.kind == kFilterStrMatch) {
            f.nlit = (int)lf.lits.size();
            f.lit_off = lit_at;
            for (auto& s : lf.lits) {
                std::memcpy(sp.lits + lit_at, s.data(), (size_t)f.width);
                lit_at += f.width;
            }
        } else {
            f.lo = (int32_t)lf.lo;
            f.span = (uint32_t)(lf.hi - lf.lo);
        }
    }
    sp.lit_bytes = lit_at;
    for (int i = 0; i < sp.nproj; i++) {
        const int ci = lp.proj[(size_t)i];
        const ColumnStore& c = t.cols[(size_t)ci];
        ProjCol& p = sp.proj[i];
        p.width = c.meta.width;
        p.pfor_slot = pfor_slot(t, &pr->pfor_cols, ci);
        p.base = p.pfor_slot >= 0 ? nullptr : c.d_arena;
        p.filter_idx = -1;
        for (int k = 0; k < sp.nfilter; k++)
            if (lp.filters[(size_t)k].col_idx == ci) p.filter_idx = k;
    }
    // A filter column that is also projected is read again by the emit kernel: ask L2 to keep it if all such
    // columns together fit in ~2/3 of the 126 MB L2.
    {
        int64_t again = 0;
        for (int i = 0; i < sp.nproj; i++)
            if (sp.proj[i].filter_idx >= 0) again += t.nrows * sp.filter[sp.proj[i].filter_idx].width;
        for (int i = 0; i < sp.nproj; i++)
            if (sp.proj[i].filter_idx >= 0) sp.filter[sp.proj[i].filter_idx].keep_l2 = (again > 0 && again <= (int64_t)(getenv("IMM3_KEEP_L2_MB") ? atoi(getenv("IMM3_KEEP_L2_MB")) : 84) << 20) ? 1 : 0;
    }
    sp.npfor = (int)pr->pfor_cols.size();
    for (int i = 0; i < sp.npfor; i++) {
        const ColumnStore& c = t.cols[(size_t)pr->pfor_cols[(size_t)i]];
        sp.pfor[i].words = reinterpret_cast<const uint32_t*>(c.d_arena);
        sp.pfor[i].word_off = c.d_word_off;
    }
    if (++db->epoch >= 0x3FFFFFu) {  // 22-bit tag wrapped: clear the status words once
        if (db->d_status) CUDA_TRY(cudaMemsetAsync(db->d_status, 0, db->status_cap * sizeof(unsigned long long), db->stream));
        db->epoch = 1;
    }
    sp.epoch = db->epoch;
    if (const char* e = getenv("IMM3_DEBUG")) sp.debug = (uint32_t)atoi(e);
    return 0;
}

// Filter kernel over the row space (kDense, kRowSpace, aggregation): tiles of 8192 rows, its ring from size_filter.
int size_dense_filter(imm3_db* db, Prepared* pr) {
    pr->sp.ntiles = (pr->table->nrows + kDenseTileRowsPerWord - 1) / kDenseTileRowsPerWord;
    CUDA_TRY(size_filter(&pr->sp, db->flags & IMM3_OPEN_NO_TMA, &pr->front));
    return 0;
}

// kBlocks: pruning, if every predicate is a range on an encoded column that has block statistics.
void size_prune(Prepared* pr) {
    const TableStore& t = *pr->table;
    const ScanPlan& sp = pr->sp;
    pr->prune = false;
    if (sp.nfilter == 0 || getenv("IMM3_NO_PRUNE")) return;
    bool ok = true;
    std::memset(&pr->pp, 0, sizeof pr->pp);
    for (int i = 0; i < sp.nfilter && ok; i++) {
        const FilterCol& f = sp.filter[i];
        ok = f.pfor_slot >= 0 && f.kind == kFilterI32Range && t.cols[(size_t)pr->pfor_cols[(size_t)f.pfor_slot]].d_stats != nullptr;
        if (ok) {
            pr->pp.stats[i] = (const BlockStat*)t.cols[(size_t)pr->pfor_cols[(size_t)f.pfor_slot]].d_stats;
            pr->pp.lo[i] = f.lo;
            pr->pp.hi[i] = (int32_t)((int64_t)f.lo + (int64_t)f.span);
        }
    }
    pr->pp.nfilter = sp.nfilter;
    pr->pp.group_shift = pr->block_filter == BlockFilter::kMini ? 3 : 5;
    pr->prune = ok;
    // a pruned scan decides whole blocks from 8 bytes each: the whole slice costs what a prefix would - no prefix phase (with a
    // communicator phase A then is this rank's whole slice and phase B the count exchange alone: the protocol is unchanged)
    if (ok) pr->prefix_blocks = 0;
}

// kBlocks, and aggregates over encoded predicates: the block filter front on tiles of 8 blocks (the offset scan's), its
// filter kernel's ring over the encoded predicate columns' tiles (size_block_filter), and pruning.
int size_block_front(Prepared* pr) {
    const TableStore& t = *pr->table;
    ScanPlan& sp = pr->sp;
    sp.ntiles = (t.nblocks + 7) / 8;
    sp.pfor_filter_mask = 0;
    int64_t tile8 = 0, tile32 = 0;
    for (int i = 0; i < sp.nfilter; i++)
        if (sp.filter[i].pfor_slot >= 0) {
            const ColumnStore& c = t.cols[(size_t)pr->pfor_cols[(size_t)sp.filter[i].pfor_slot]];
            sp.pfor_filter_mask |= 1u << sp.filter[i].pfor_slot;
            tile8 = std::max<int64_t>(tile8, c.max_tile_bytes);
            tile32 = std::max<int64_t>(tile32, c.max_tile32_bytes);
        }
    CUDA_TRY(size_block_filter(pr->block_filter, &sp, tile8, tile32, &pr->front));
    size_prune(pr);
    return 0;
}

// kRowSpace, kBlocks: the block emit kernel.
int size_block_emit(imm3_db* db, Prepared* pr) {
    const TableStore& t = *pr->table;
    int64_t words = 0;
    for (int ci : pr->pfor_cols) words = std::max<int64_t>(words, t.cols[(size_t)ci].max_block_words);
    CUDA_TRY(size_blocks_emit(&pr->sp, pr->pipeline == Pipeline::kRowSpace, words, t.nblocks, db->num_sms, &pr->blocks_emit));
    if (pr->blocks_emit.occupancy < 1)
        return fail(IMM3_ERR_CUDA, "block emit kernel does not fit on an SM (dynamic shared memory %zu bytes)", pr->blocks_emit.smem);
    return 0;
}

// The filter kernel's persistent grid from its occupancy, and the status words of the tiles.
int plan_grid(imm3_db* db, Prepared* pr) {
    const ScanPlan& sp = pr->sp;
    KernelShape& ks = pr->front;
    if (sp.ntiles >= (int64_t)0x7FFFFFFF) return fail(IMM3_ERR_UNSUPPORTED, "too many tiles (%lld)", (long long)sp.ntiles);
    if (ks.occupancy < 1) return fail(IMM3_ERR_CUDA, "kernel does not fit on an SM (dynamic shared memory %zu bytes)", ks.smem);
    const int64_t persistent = (int64_t)db->num_sms * ks.occupancy;
    ks.grid = (int)std::max<int64_t>(1, std::min<int64_t>(sp.ntiles, persistent));
    const size_t status_need = 2 * (size_t)status_round_up(sp.ntiles);  // tile counts + (dense kernel) tile offsets
    if (status_need > db->status_cap) {
        if (db->d_status) CUDA_TRY(cudaFree(db->d_status));
        db->d_status = nullptr;
        size_t cap = status_need + status_need / 4 + 1024;
        CUDA_TRY(cudaMalloc(&db->d_status, cap * sizeof(unsigned long long)));
        CUDA_TRY(cudaMemsetAsync(db->d_status, 0, cap * sizeof(unsigned long long), db->stream));
        db->status_cap = cap;
    }
    return 0;
}

// Fill the device plan of the query's pipeline (everything but result pointers and the bitmap).
int fill_scan_plan(imm3_db* db, Prepared* pr) {
    const TableStore& t = *pr->table;
    int rc = plan_columns(db, pr);
    if (rc) return rc;
    const int64_t prefix = prefix_rows_wanted(pr->lp);
    switch (pr->pipeline) {
    case Pipeline::kDense: {
        const int64_t want = (prefix + kDenseTileRowsPerWord - 1) / kDenseTileRowsPerWord * kDenseTileRowsPerWord;
        if (want * 2 <= t.nrows) pr->prefix_rows = want;
        if ((rc = size_dense_filter(db, pr))) return rc;
        CUDA_TRY(size_emit(&pr->sp, db->flags & IMM3_OPEN_NO_TMA, db->num_sms, &pr->emit));
        break;
    }
    case Pipeline::kRowSpace:
    case Pipeline::kBlocks: {
        pr->prefix_blocks = prefix_blocks_wanted(*pr);
        rc = pr->pipeline == Pipeline::kRowSpace ? size_dense_filter(db, pr) : size_block_front(pr);
        if (rc || (rc = size_block_emit(db, pr))) return rc;
        break;
    }
    case Pipeline::kSinglePass:
        if (t.max_block_rows > kMaxBlockRows)
            return fail(IMM3_ERR_UNSUPPORTED, "block-mode kernel stages blocks of at most %d rows, table %s has a block of %d",
                        kMaxBlockRows, t.meta.name.c_str(), t.max_block_rows);
        pr->sp.ntiles = t.nblocks;
        CUDA_TRY(size_scan_blocks(pr->sp, t.max_block_rows, &pr->front));
        break;
    }
    return plan_grid(db, pr);
}

bool has_encoded_filter(const Prepared& pr) {
    for (auto& f : pr.lp.filters)
        if (is_pfor(*pr.table, f.col_idx)) return true;
    return false;
}

// Real OR over encoded columns (IMM3_DNF_ENCODED_FILTER): every term on kBlocks - a term of dense predicates alone takes the
// mini-block kernel, which decides them per block (what IMM3_NO_HYBRID runs for a conjunction).
void force_blocks(Prepared* pr) {
    pr->pipeline = Pipeline::kBlocks;
    choose_block_filter(pr);
}

// ... the plan of every term but the first (which carries the projection and the emit plan, fill_scan_plan): its own filter
// kernel, ring and pruning over the table's tiles of 8 blocks.  A prefix phase runs unless every term is pruned.
int fill_or_terms_plan(imm3_db* db, Prepared* pr) {
    bool pruned = pr->prune;
    for (auto& tm : pr->or_terms) {
        int rc = plan_columns(db, tm.get());
        if (rc || (rc = size_block_front(tm.get())) || (rc = plan_grid(db, tm.get()))) return rc;
        pruned = pruned && tm->prune;
    }
    pr->prefix_blocks = pruned ? 0 : prefix_blocks_wanted(*pr);
    return 0;
}

int ensure_buf(Buf* b, size_t bytes) {
    if (b->cap >= bytes) return 0;
    if (b->p) cudaFree(b->p);
    *b = Buf();
    size_t cap = bytes + bytes / 8 + 4096;
    CUDA_TRY(cudaMalloc(&b->p, cap));
    b->cap = cap;
    return 0;
}

// Tile counts and offsets, in whole rounds (4096 tiles) of the offset scan.
int ensure_tile_scratch(imm3_db* db, int64_t ntiles) {
    const size_t ntiles_pad = ((size_t)ntiles + 4095) / 4096 * 4096 + 16;
    int rc = ensure_buf(&db->d_tile_cnt, ntiles_pad * 4);
    return rc ? rc : ensure_buf(&db->d_tile_off, ntiles_pad * 8);
}

// Scratch of the filter kernel over the row space: the selection bitmap (unless the plan brings its own), span counts, tile
// counts and offsets.  (+64 bitmap words: the row-space emit kernel reads, for every lane of a block's warp, the word holding
// bit R0 + 32*lane and the one after it - up to 33 words past the last row's word for a 1-row tail block at the end of the slice)
int ensure_row_space(imm3_db* db, ScanPlan& sp) {
    int rc;
    if (!sp.bitmap) {
        if ((rc = ensure_buf(&db->d_bitmap, (size_t)(sp.ntiles * kDenseTileRowsPerWord / 32 + 64) * 4))) return rc;
        sp.bitmap = (uint32_t*)db->d_bitmap.p;
    }
    if ((rc = ensure_buf(&db->d_span_cnt, (size_t)(sp.ntiles * (kDenseTileRowsPerWord / 1024) + 8) * 4))) return rc;
    return ensure_tile_scratch(db, sp.ntiles);
}

// Launch the count-exchange kernel of one round (every rank of the communicator must launch the same rounds in the same
// order).  has_count = 0: this rank ran no kernel in this query (empty slice) and contributes 0.
int launch_exchange(imm3_db* db, Run* run, int64_t limit, int has_count, unsigned long long pub_seq = 0) {
    CommPlan cp;
    std::memset(&cp, 0, sizeof cp);
    cp.pub = pub_seq ? db->h_ctrl : nullptr;
    cp.pub_seq = pub_seq;
    for (int i = 0; i < db->world; i++) cp.peer[i] = db->comm_peer[i];
    cp.rank = db->rank;
    cp.world = db->world;
    if (((++db->comm_epoch) & 0xFFFFFFu) == 0) ++db->comm_epoch;  // tag 0 is what an untouched mailbox holds
    cp.epoch = db->comm_epoch;
    cp.has_count = has_count;
    cp.limit = limit;
    cp.timeout_ns = db->comm_timeout_ns;
    CUDA_TRY(launch_count_exchange(cp, db->d_ctrl, &reinterpret_cast<CtrlBlock*>(db->d_ctrl)->x, db->stream));
    run->note("count_exchange");
    return 0;
}

// A round of the exchange without a scan of this rank's own: its slice is empty (has_count = 0) or its previous phase
// already covered the whole slice (has_count = 1: ctrl->total still holds that count).
int exchange_only(imm3_db* db, Run* run, int64_t limit, int has_count) {
    int rc = launch_exchange(db, run, limit, has_count);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(db->h_ctrl, db->d_ctrl, sizeof(CtrlBlock), cudaMemcpyDeviceToHost, db->stream));
    CUDA_TRY(cudaStreamSynchronize(db->stream));
    if (db->h_ctrl->x.error)
        return fail(IMM3_ERR_COMM, "count exchange: a peer's count did not arrive within %llu ms (ranks must issue the same queries in the same order)",
                    db->comm_timeout_ns / 1000000ull);
    return 0;
}

// Whether the block filter front's last CTA runs the offset scan over `ntiles` tiles (scan_inline_for; the lane kernel's
// inline scan is written for 8 warps)
int block_scan_inline(const Prepared& pr, int64_t ntiles) { return scan_inline_for(ntiles) && !(pr.block_filter == BlockFilter::kLane && pr.front.lane_warps < 8); }
int prepare_scan_buffers(imm3_db* db, int64_t ntiles, bool want_list) {
    if (want_list) {
        int rc = ensure_buf(&db->d_tile_list, (size_t)(ntiles + 16) * 4);
        if (rc) return rc;
    }
    const size_t nchunks = (size_t)((ntiles + 4095) / 4096);
    if (db->d_scan_part.cap < nchunks * 16 + 512) {  // (+ the scan-emit kernel's chunks-done counter, 128 bytes behind the sums)
        if (db->d_scan_part.p) cudaFree(db->d_scan_part.p);
        db->d_scan_part = Buf();
        const size_t cap = nchunks * 16 + 4096;
        CUDA_TRY(cudaMalloc(&db->d_scan_part.p, cap));
        CUDA_TRY(cudaMemsetAsync(db->d_scan_part.p, 0, cap, db->stream));
        db->d_scan_part.cap = cap;
    }
    if (((++db->scan_epoch) & 0xFFFFFFu) == 0) ++db->scan_epoch;  // (tag 0 = never written)
    return 0;
}
int launch_scan_kernel(imm3_db* db, const ScanPlan& sp, int64_t ntiles, Run* run, bool want_list = false) {
    int rc = prepare_scan_buffers(db, ntiles, want_list);
    if (rc) return rc;
    CUDA_TRY(launch_offset_scan((const uint32_t*)db->d_tile_cnt.p, (unsigned long long*)db->d_tile_off.p, ntiles, sp.limit, db->scan_epoch,
                                (unsigned long long*)db->d_scan_part.p, db->d_ctrl, want_list ? (unsigned int*)db->d_tile_list.p : nullptr, db->stream));
    run->note("offset_scan");
    return 0;
}

// The part of the slice one phase scans (see small_limit): all of it, or phase A's leading prefix_rows rows or prefix_blocks
// blocks.
struct Extent {
    int64_t nrows, ntiles, nblocks;
};
Extent phase_extent(const Prepared& pr, bool prefix) {
    const TableStore& t = *pr.table;
    const int64_t nb = pr.prefix_blocks;
    if (!prefix) return {pr.sp.nrows, pr.sp.ntiles, t.nblocks};
    if (pr.prefix_rows > 0) return {pr.prefix_rows, pr.prefix_rows / kDenseTileRowsPerWord, nb};
    if (pr.pipeline != Pipeline::kRowSpace) return {pr.sp.nrows, (nb + 7) / 8, nb};
    const int64_t rows = (int64_t)t.row_start[(size_t)nb];
    return {rows, (rows + kDenseTileRowsPerWord - 1) / kDenseTileRowsPerWord, nb};
}
// A filter kernel's grid over a phase's tiles: its plan's persistent grid, fewer CTAs for a shorter phase.
int phase_grid(const Prepared& p, int64_t ntiles) { return (int)std::max<int64_t>(1, std::min<int64_t>(p.front.grid, ntiles)); }
// A later term's device plan of a real OR in one phase: its own, over the first term's rows, tiles and bitmap.
ScanPlan term_plan(const Prepared& tm, const ScanPlan& first) {
    ScanPlan sp = tm.sp;
    sp.nrows = first.nrows;
    sp.ntiles = first.ntiles;
    sp.bitmap = first.bitmap;
    return sp;
}

// What a pipeline's launch function tells the epilogue of run_scan_once.
struct Queued {
    unsigned long long pub_seq;  // publish (plan.hpp): sequence number of this launch sequence
    bool publish;                // the pipeline's last kernel may write the pinned control block itself
    bool published = false;      // ... and does
    bool have_mid = false;       // ev_mid splits the device time into two stages
};

// No event may sit between a kernel and its programmatic dependent: without PDL (IMM3_NO_PDL, or nothing to emit) ev_mid
// marks the end of the filter stage.
int mark_mid(imm3_db* db, bool pdl, Queued* q) {
    if (pdl) return 0;
    CUDA_TRY(cudaEventRecord(db->ev_mid, db->stream));
    q->have_mid = true;
    return 0;
}

// IMM3_DEBUG bit 16 + IMM3_TRACE (debugging): phase stamps, min / max over CTAs or warps, then `extra` words
int setup_phase_trace(imm3_db* db, ScanPlan& sp, size_t extra) {
    if (!(sp.debug & 16u) || !getenv("IMM3_TRACE")) return 0;
    int rc = ensure_buf(&db->d_trace, (64 + extra) * 8);
    if (rc) return rc;
    std::vector<unsigned long long> init(64 + extra);
    for (int i = 0; i < 64; i++) init[(size_t)i] = (i & 1) ? 0ull : ~0ull;
    CUDA_TRY(cudaMemcpyAsync(db->d_trace.p, init.data(), init.size() * 8, cudaMemcpyHostToDevice, db->stream));
    CUDA_TRY(cudaStreamSynchronize(db->stream));
    sp.trace = (unsigned long long*)db->d_trace.p;
    return 0;
}

// The filter kernel over the row space (from ev0 on) - for a real OR the first term's, then each later term's, ORing its rows
// into the same bitmap (same span / tile counts: every pass rewrites the counts of the union so far) - and the offset scan
// unless the last pass's last CTA runs it.
int launch_row_space_filter(imm3_db* db, const Prepared& pr, ScanPlan& sp, Run* run) {
    const bool scan_inline = sp.nfilter == 0 || scan_inline_for(sp.ntiles);
    auto filter = [&](const Prepared& p, ScanPlan& f, bool last) {
        f.scan_inline = last && scan_inline;
        std::string route;
        CUDA_TRY(launch_filter(f, sp.bitmap, (uint32_t*)db->d_span_cnt.p, (uint32_t*)db->d_tile_cnt.p, (unsigned long long*)db->d_tile_off.p,
                               db->d_ctrl, phase_grid(p, f.ntiles), p.front.smem, db->stream, &route));
        run->note(route);
        return 0;
    };
    CUDA_TRY(cudaEventRecord(db->ev0, db->stream));
    int rc = filter(pr, sp, pr.or_terms.empty());
    for (size_t i = 0; !rc && i < pr.or_terms.size(); i++) {
        ScanPlan term = term_plan(*pr.or_terms[i], sp);
        rc = filter(*pr.or_terms[i], term, i + 1 == pr.or_terms.size());
    }
    if (rc) return rc;
    return scan_inline ? 0 : launch_scan_kernel(db, sp, sp.ntiles, run);
}

// kDense: filter kernel -> emit kernels.  Two emit kernels, one of which does the work: which one is decided on the device
// from the match count, unless an earlier query of this shape said which (see emit_hint).
int launch_dense(imm3_db* db, const Prepared& pr, ScanPlan& sp, Run* run, Queued* q) {
    int rc;
    if ((rc = setup_phase_trace(db, sp, 0)) || (rc = ensure_row_space(db, sp))) return rc;
    const int stream_ok = pr.emit.stream.stage_bytes > 0 && sp.nproj > 0;
    const char* force = getenv("IMM3_EMIT");  // experiment: "stream" / "gather" = that kernel takes every result, "both" = no feedback
    int hint = -1;
    if (stream_ok && !(force && !strcmp(force, "both"))) {
        auto it = db->emit_hint.find(pr.shape_key);
        if (it != db->emit_hint.end()) hint = it->second;
        if (force && !strcmp(force, "stream")) hint = 1;
        if (force && !strcmp(force, "gather")) hint = 0;
    }
    const bool only_stream = stream_ok && hint == 1, only_gather = stream_ok && hint == 0;
    // The first emit kernel is launched as a programmatic dependent of the filter kernel (its prologue overlaps the filter
    // kernel's tail); IMM3_NO_PDL=1 restores per-stage timing.
    const bool pdl = sp.nproj > 0 && !getenv("IMM3_NO_PDL");
    if ((rc = launch_row_space_filter(db, pr, sp, run)) || (rc = mark_mid(db, pdl, q))) return rc;
    if (sp.nproj == 0) return 0;
    const int64_t nspans = sp.ntiles * (kDenseTileRowsPerWord / 1024);
    if (stream_ok && !only_gather) {
        CUDA_TRY(launch_emit_stream(sp, sp.bitmap, (const uint32_t*)db->d_span_cnt.p, (const uint32_t*)db->d_tile_cnt.p,
                                    (const unsigned long long*)db->d_tile_off.p, sp.ntiles, pr.emit.stream, only_stream ? -1 : 1, db->d_ctrl,
                                    pdl, db->stream));
        run->note("emit_stream/s=" + std::to_string(pr.emit.stream.stages));
    }
    if (!only_stream) {
        CUDA_TRY(launch_emit(sp, sp.bitmap, (const uint32_t*)db->d_span_cnt.p, (const unsigned long long*)db->d_tile_off.p, 8,
                             nspans, pr.emit, stream_ok && !only_gather, db->d_ctrl, pdl && (only_gather || !stream_ok), db->stream));
        run->note(pr.emit.general ? "emit_general" : "emit");
    }
    return 0;
}

// kRowSpace: filter kernel over the row space -> block emit kernel.
int launch_row_space(imm3_db* db, const Prepared& pr, ScanPlan& sp, int64_t nblocks, Run* run, Queued* q) {
    const bool pdl = sp.nproj > 0 && !getenv("IMM3_NO_PDL");
    int rc;
    if ((rc = ensure_row_space(db, sp)) || (rc = launch_row_space_filter(db, pr, sp, run)) || (rc = mark_mid(db, pdl, q))) return rc;
    if (sp.nproj == 0) return 0;
    CUDA_TRY(launch_blocks_emit(sp, sp.bitmap, (const uint32_t*)db->d_span_cnt.p, nullptr, (const unsigned long long*)db->d_tile_off.p,
                                nblocks, db->d_ctrl, true, pdl, pr.blocks_emit, db->stream));
    run->note("blocks_emit(rowspace)");
    return 0;
}

// Scratch of the block filter front over `ntiles` tiles: 32 bitmap words and one count per block, tile counts and offsets,
// and (pruned) the work list of the tiles blocks_prune_kernel leaves to the filter kernel.
int ensure_block_filter(imm3_db* db, const Prepared& pr, int64_t ntiles, int64_t nblocks) {
    int rc;
    if ((rc = ensure_buf(&db->d_bitmap, (size_t)(nblocks * 32 + 2) * 4))) return rc;
    if ((rc = ensure_buf(&db->d_span_cnt, (size_t)(nblocks + 8 + 1024) * 4))) return rc;  // (+ whole 16-byte loads of a group's counts)
    if ((rc = ensure_tile_scratch(db, ntiles))) return rc;
    return pr.prune ? ensure_buf(&db->d_work, (size_t)((nblocks + 7) / 8 + 2) * 4) : 0;
}

// The block filter front, shared by Project queries (kBlocks) and aggregates over encoded predicates: [blocks_prune ->]
// block filter kernel [-> offset scan, when `scan` and the filter kernel's last CTA does not run it].  Per block it leaves
// the selected row count in d_span_cnt and - only for a partially selected block - the block's 32 words in d_bitmap.
// Buffers: ensure_block_filter first.  grp_sum: blocks_group_emit_kernel follows (lane kernel only).  The selection goes to
// (words, cnts): db->d_bitmap / d_span_cnt, or a later term's buffers of a real OR.
int launch_block_filter_front(imm3_db* db, const Prepared& pr, const ScanPlan& sp, int64_t nblocks, Run* run, uint32_t* grp_sum, bool scan,
                              uint32_t* words, uint32_t* cnts) {
    const TableStore& t = *pr.table;
    const int64_t ntiles = sp.ntiles;
    const unsigned int* work = pr.prune ? (const unsigned int*)db->d_work.p : nullptr;
    if (pr.prune) {
        // whole blocks decided from their min / max; only the tiles a window edge cuts through reach the filter kernel
        CUDA_TRY(cudaMemsetAsync(db->d_work.p, 0, 4, db->stream));
        CUDA_TRY(launch_blocks_prune(pr.pp, t.d_row_start, nblocks, ntiles, cnts, (uint32_t*)db->d_tile_cnt.p,
                                     (unsigned int*)db->d_work.p, db->num_sms, db->stream, grp_sum));
        run->note("blocks_prune");
    }
    std::string route;
    CUDA_TRY(launch_blocks_filter(sp, words, cnts, (uint32_t*)db->d_tile_cnt.p, (unsigned long long*)db->d_tile_off.p, db->d_ctrl, nblocks,
                                  phase_grid(pr, ntiles), pr.block_filter, pr.front, work, grp_sum, db->stream, &route));
    run->note(route);
    return (scan && !sp.scan_inline) ? launch_scan_kernel(db, sp, ntiles, run, true) : 0;
}

// Real OR over encoded columns: the scratch of every term's front, and the term buffers (grow-only).
int ensure_or_terms(imm3_db* db, const Prepared& pr, int64_t nblocks) {
    int rc;
    for (auto& tm : pr.or_terms)
        if ((rc = ensure_block_filter(db, *tm, tm->sp.ntiles, nblocks))) return rc;
    if ((rc = ensure_buf(&db->d_or_bitmap, (size_t)(nblocks * 32 + 2) * 4))) return rc;
    return ensure_buf(&db->d_or_cnt, (size_t)(nblocks + 8 + 1024) * 4);
}

// ... behind the first term's front: each later term's front into the term buffers, then blocks_or_merge_kernel into
// d_bitmap / d_span_cnt.  Every term runs over the first term's blocks and tiles - in a prefix phase too - and runs no scan:
// the tile counts it leaves are rewritten by the merge (a term's plan keeps the scan_inline = 0 of plan_columns).
int launch_or_merges(imm3_db* db, const Prepared& pr, const ScanPlan& sp, int64_t nblocks, Run* run) {
    for (auto& tm : pr.or_terms) {
        const int rc = launch_block_filter_front(db, *tm, term_plan(*tm, sp), nblocks, run, nullptr, false, (uint32_t*)db->d_or_bitmap.p,
                                                 (uint32_t*)db->d_or_cnt.p);
        if (rc) return rc;
        CUDA_TRY(launch_blocks_or_merge(pr.table->d_row_start, nblocks, sp.ntiles, (uint32_t*)db->d_bitmap.p, (uint32_t*)db->d_span_cnt.p,
                                        (const uint32_t*)db->d_or_bitmap.p, (const uint32_t*)db->d_or_cnt.p, (uint32_t*)db->d_tile_cnt.p,
                                        db->d_ctrl, db->num_sms, db->stream));
        run->note("blocks_or_merge");
    }
    return 0;
}

// kBlocks: [blocks_prune ->] block filter kernel -> group emit (lane kernel, one encoded column projected: every emit warp finds
// its rows from the group sums, no scan), scan-emit (one encoded column projected: offset scan + emit in one small-footprint
// kernel, resident while the filter kernel runs) or offset scan + block emit kernel.  A real OR over encoded columns merges
// its later terms' fronts (launch_or_merges) before the emit; group emit needs a single term's group sums and is not used.
int launch_blocks(imm3_db* db, const Prepared& pr, ScanPlan& sp, int64_t nblocks, Run* run, Queued* q) {
    const int64_t ntiles = sp.ntiles;
    const bool lane = pr.block_filter == BlockFilter::kLane;
    const bool merge = !pr.or_terms.empty();
    int rc;
    if ((rc = ensure_block_filter(db, pr, ntiles, nblocks)) || (merge && (rc = ensure_or_terms(db, pr, nblocks)))) return rc;
    int fused_grid = 0;  // > 0: blocks_scan_emit_kernel
    int group_grid = 0;  // > 0: blocks_group_emit_kernel
    if (sp.nproj == 1 && sp.proj[0].pfor_slot >= 0 && !getenv("IMM3_NO_SCANEMIT")) {
        size_t sum_bytes = 0;
        if (lane && !merge && !getenv("IMM3_NO_GROUPEMIT")) CUDA_TRY(blocks_group_emit_grid(db->num_sms, nblocks, &group_grid, &sum_bytes));
        if (group_grid > 0) {
            if (!db->d_grp_sum.p) {
                CUDA_TRY(cudaMalloc(&db->d_grp_sum.p, sum_bytes));
                db->d_grp_sum.cap = sum_bytes;
                CUDA_TRY(cudaMemsetAsync(db->d_grp_sum.p, 0, db->d_grp_sum.cap, db->stream));
            }
        } else {
            CUDA_TRY(blocks_scan_emit_grid(db->num_sms, ntiles, &fused_grid));
            if (fused_grid > 0 && (rc = prepare_scan_buffers(db, ntiles, true))) return rc;
        }
    }
    const bool emit_scans = group_grid > 0 || fused_grid > 0;  // (these emit kernels find the offsets themselves)
    sp.scan_inline = !merge && !emit_scans && block_scan_inline(pr, ntiles);
    uint32_t* const grp_sum = group_grid > 0 ? (uint32_t*)db->d_grp_sum.p : nullptr;
    if ((rc = setup_phase_trace(db, sp, 1024))) return rc;
    CUDA_TRY(cudaEventRecord(db->ev0, db->stream));
    if ((rc = launch_block_filter_front(db, pr, sp, nblocks, run, grp_sum, !emit_scans && !merge, (uint32_t*)db->d_bitmap.p,
                                        (uint32_t*)db->d_span_cnt.p)))
        return rc;
    if (merge && ((rc = launch_or_merges(db, pr, sp, nblocks, run)) || (!emit_scans && (rc = launch_scan_kernel(db, sp, ntiles, run, true)))))
        return rc;
    CtrlBlock* const pub = q->publish ? db->h_ctrl : nullptr;
    const unsigned long long pub_seq = q->publish ? q->pub_seq : 0;
    if (emit_scans) {
        const bool pdl = !getenv("IMM3_NO_PDL");
        if ((rc = mark_mid(db, pdl, q))) return rc;
        if (group_grid > 0) {
            CUDA_TRY(launch_blocks_group_emit(sp, (const uint32_t*)db->d_bitmap.p, (const uint32_t*)db->d_span_cnt.p, grp_sum, nblocks, db->d_ctrl,
                                              pdl, group_grid, db->stream, pub, pub_seq));
            run->note("blocks_group_emit/ctas=" + std::to_string(group_grid));
        } else {
            CUDA_TRY(launch_blocks_scan_emit(sp, (const uint32_t*)db->d_bitmap.p, (const uint32_t*)db->d_span_cnt.p, (const uint32_t*)db->d_tile_cnt.p,
                                             (unsigned long long*)db->d_tile_off.p, nblocks, db->scan_epoch, (unsigned long long*)db->d_scan_part.p,
                                             db->d_ctrl, (unsigned int*)db->d_tile_list.p, pdl, fused_grid, db->stream, pub, pub_seq));
            run->note("blocks_scan_emit");
        }
        q->published = q->publish;
    } else {
        const bool pdl = sp.nproj > 0 && !getenv("IMM3_NO_PDL");
        if ((rc = mark_mid(db, pdl, q))) return rc;
        if (sp.nproj > 0) {
            CUDA_TRY(launch_blocks_emit(sp, (const uint32_t*)db->d_bitmap.p, (const uint32_t*)db->d_span_cnt.p,
                                        sp.scan_inline ? nullptr : (const unsigned int*)db->d_tile_list.p,
                                        (const unsigned long long*)db->d_tile_off.p, nblocks, db->d_ctrl, false, pdl, pr.blocks_emit, db->stream));
            run->note("blocks_emit(blocks)");
        }
    }
    return 0;
}

// Launch the kernels of one phase over `ex` and wait for the match count.
int run_scan_once(imm3_db* db, const Prepared& pr, const Extent& ex, Run* run, int64_t* total, bool exchange) {
    ScanPlan sp = pr.sp;  // this phase's device plan: the pipeline binds its bitmap and decides scan_inline
    sp.nrows = ex.nrows;
    sp.ntiles = ex.ntiles;
    // publish (plan.hpp): the query's last kernel writes the pinned control block itself and the host polls it
    const bool publish_ok = !getenv("IMM3_NO_PUBLISH");
    const bool sharded = exchange && db->comm_on;  // (a sharded table: the exchange kernel publishes)
    Queued q{++db->pub_seq, publish_ok && !sharded};
    int rc = 0;
    switch (pr.pipeline) {
    case Pipeline::kDense: rc = launch_dense(db, pr, sp, run, &q); break;
    case Pipeline::kRowSpace: rc = launch_row_space(db, pr, sp, ex.nblocks, run, &q); break;
    case Pipeline::kBlocks: rc = launch_blocks(db, pr, sp, ex.nblocks, run, &q); break;
    case Pipeline::kSinglePass:
        CUDA_TRY(cudaEventRecord(db->ev0, db->stream));
        CUDA_TRY(launch_scan_blocks(sp, db->d_ctrl, db->d_status, pr.front.grid, pr.front.smem, db->stream));
        run->note("scan_blocks");
        break;
    }
    if (rc) return rc;
    if (sharded) {
        // The per-rank counts are exchanged by the GPUs themselves (k_comm.cuh), behind the query's last kernel: no host
        // round trip between the kernels and the exchange, one synchronisation per query.
        if ((rc = launch_exchange(db, run, sp.limit, 1, publish_ok ? q.pub_seq : 0))) return rc;
        q.published = publish_ok;
    }
    CUDA_TRY(cudaEventRecord(db->ev1, db->stream));
    db->ev_seq = ++db->query_seq;
    if (q.published) {
        run->t_launched = now_us();
        const volatile unsigned long long* ps = &db->h_ctrl->pub_seq;
        bool seen = false;
        for (unsigned spins = 0;; spins++) {
            const unsigned long long word = __atomic_load_n(ps, __ATOMIC_ACQUIRE);
            if ((word >> 41) == (q.pub_seq & 0x7FFFFFull)) {
                if (!sharded) {  // (blocks_scan_emit_kernel packs what the host needs into the word itself)
                    db->h_ctrl->c.total = word & ((1ull << 40) - 1ull);
                    db->h_ctrl->c.error = (word >> 40) & 1u ? 1u : 0u;
                    db->h_ctrl->c.dense_rows = 0;
                }
                seen = true;
                break;
            }
            if ((spins & 0xFFFu) == 0xFFFu && now_us() - run->t_launched > 2e5) break;  // 0.2 s: something is wrong - ask the runtime
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
        }
        if (!seen) {  // (a kernel fault, or a peer that never came: the ordinary path reports it)
            CUDA_TRY(cudaMemcpyAsync(db->h_ctrl, db->d_ctrl, sizeof(CtrlBlock) - sizeof(unsigned long long), cudaMemcpyDeviceToHost, db->stream));
            CUDA_TRY(cudaStreamSynchronize(db->stream));
        }
        run->t_synced = now_us();
    } else {
        CUDA_TRY(cudaMemcpyAsync(db->h_ctrl, db->d_ctrl, sizeof(CtrlBlock) - sizeof(unsigned long long), cudaMemcpyDeviceToHost, db->stream));
        run->t_launched = now_us();
        CUDA_TRY(cudaStreamSynchronize(db->stream));
        run->t_synced = now_us();
    }
    if (db->h_ctrl->c.error) return fail(IMM3_ERR_CUDA, "kernel watchdog fired (code %u)", db->h_ctrl->c.error);
    if (sharded && db->h_ctrl->x.error)
        return fail(IMM3_ERR_COMM, "count exchange: a peer's count did not arrive within %llu ms (ranks must issue the same queries in the same order)",
                    db->comm_timeout_ns / 1000000ull);
    if (q.published && !q.have_mid && !run->eager_times && !getenv("IMM3_EAGER_TIMES")) {
        run->device_ms = -1.0;  // read lazily (imm3_result_device_ms): the events complete a moment after the publish, waiting for them here costs 2-3 us
        run->stage_ms[0] = -1.0, run->stage_ms[1] = 0;
    } else {
        float f = 0, a = 0, b = 0;
        if (q.published) CUDA_TRY(cudaEventSynchronize(db->ev1));
        CUDA_TRY(cudaEventElapsedTime(&f, db->ev0, db->ev1));
        a = f;
        if (q.have_mid) {
            CUDA_TRY(cudaEventElapsedTime(&a, db->ev0, db->ev_mid));
            CUDA_TRY(cudaEventElapsedTime(&b, db->ev_mid, db->ev1));
        }
        run->device_ms += f;  // (two-phase LIMIT queries: the phases' times add up)
        run->stage_ms[0] += a;
        run->stage_ms[1] += b;
    }
    *total = (int64_t)db->h_ctrl->c.total;
    if (pr.pipeline == Pipeline::kDense && sp.nproj > 0 && pr.emit.stream.stage_bytes > 0)  // feedback for the next query of this shape
        db->emit_hint[pr.shape_key] = (db->h_ctrl->c.total > 0 && db->h_ctrl->c.dense_rows * 2 >= db->h_ctrl->c.total) ? 1 : 0;
    if (sp.trace) {
        unsigned long long h[64];
        CUDA_TRY(cudaMemcpy(h, sp.trace, sizeof h, cudaMemcpyDeviceToHost));
        if (FILE* f = fopen(getenv("IMM3_TRACE"), "w")) {
            const char* names[] = {"K1 entry", "K1 cta done", "K1 scan start", "K1 scan end", "K3s entry", "K3s first tile", "K3s cta done", "-",
                                   "K3b entry", "K3b dep ready", "K3b tiles seen", "K3b tile meta", "K3b block start", "K3b block done", "K3b warp done", "K3b words here", "K3b store start", "K3b store done"};
            for (int i = 0; i < 18; i++)
                if (h[2 * i] != ~0ull)
                    fprintf(f, "%-16s min %9.2f us  max %9.2f us\n", names[i], (double)(h[2 * i] - h[0]) / 1e3, (double)(h[2 * i + 1] - h[0]) / 1e3);
            for (int i = 0; i < 8; i++)
                if (h[32 + i] != ~0ull && h[32 + i] != 0) fprintf(f, "scan round %d after block scan: %9.2f us\n", i, (double)(h[32 + i] - h[0]) / 1e3);
            if (pr.block_filter == BlockFilter::kLane) {  // per CTA of the lane kernel: done time, SM, tiles decided
                std::vector<unsigned long long> pc(1024);
                if (cudaMemcpy(pc.data(), sp.trace + 64, 1024 * 8, cudaMemcpyDeviceToHost) == cudaSuccess)
                    for (int i = 0; i < 512 && pc[2 * i]; i++)
                        fprintf(f, "cta %3d done %9.2f us  sm %3llu  tiles %llu\n", i, (double)(pc[2 * i] - h[0]) / 1e3, pc[2 * i + 1] >> 32, pc[2 * i + 1] & 0xFFFFFFFFull);
            }
            fclose(f);
        }
    }
    return 0;
}

// Launch the kernels of one query and wait for the match count (see small_limit for the two-phase LIMIT).
int run_scan(imm3_db* db, const Prepared& pr, Run* run, int64_t* total) {
    const bool comm = db->comm_on && !pr.for_bitmap;
    const bool local_prefix = pr.prefix_blocks > 0 || pr.prefix_rows > 0;
    if (!(comm ? small_limit(pr.lp) : local_prefix)) return run_scan_once(db, pr, phase_extent(pr, false), run, total, comm);
    // phase A: the leading blocks / rows only
    run->eager_times = true;
    if (local_prefix) run->tag = "/prefix";
    int rc = run_scan_once(db, pr, phase_extent(pr, local_prefix), run, total, comm);
    run->tag = "";
    if (rc || (comm ? (int64_t)db->h_ctrl->x.counts[0] >= pr.lp.limit : *total >= pr.lp.limit)) return rc;
    // phase B: the prefix did not fill the LIMIT - the whole table
    if (!local_prefix) return exchange_only(db, run, pr.sp.limit, 1);  // (comm only: phase A was this rank's whole slice already)
    return run_scan_once(db, pr, phase_extent(pr, false), run, total, comm);
}

// java.lang.Double.toString for an integral value of int32 magnitude (all Min/MaxDoubleAggr ever hold here): "18.0",
// "-128.0", and computerized scientific notation from 10^7 on ("1.0E7", "2.147483647E9").
std::string java_double_to_string_integral(double v) {
    if (v == 0) return "0.0";
    const bool neg = v < 0;
    long long a = (long long)(neg ? -v : v);
    std::string digits = std::to_string(a);
    std::string out = neg ? "-" : "";
    if (a < 10000000ll) return out + digits + ".0";
    const int exp10 = (int)digits.size() - 1;
    std::string frac = digits.substr(1);
    while (frac.size() > 1 && frac.back() == '0') frac.pop_back();
    return out + digits.substr(0, 1) + "." + frac + "E" + std::to_string(exp10);
}

// java.lang.Double.toString for any finite or infinite double (AVG results): the shortest digits that round-trip
// (std::to_chars), plain notation with at least one fractional digit for 10^-3 <= |v| < 10^7 ("21.5", "0.001"), else
// computerized scientific notation ("1.0E7", "-2.5E-4").
std::string java_double_to_string(double v) {
    if (std::isnan(v)) return "NaN";
    if (std::isinf(v)) return v > 0 ? "Infinity" : "-Infinity";
    if (v == 0) return std::signbit(v) ? "-0.0" : "0.0";
    char buf[64];
    const std::to_chars_result tc = std::to_chars(buf, buf + sizeof buf, std::fabs(v), std::chars_format::scientific);  // d[.ddd]e[+-]xx
    const std::string sci(buf, tc.ptr);
    const size_t e = sci.find('e');
    const int exp10 = std::atoi(sci.c_str() + e + 1);
    const std::string digits = sci.substr(0, 1) + (e > 1 ? sci.substr(2, e - 2) : std::string());  // v = 0.digits x 10^(exp10 + 1)
    const std::string sign = v < 0 ? "-" : "";
    const double a = std::fabs(v);
    if (a >= 1e-3 && a < 1e7) {
        if (exp10 < 0) return sign + "0." + std::string((size_t)(-exp10 - 1), '0') + digits;
        const size_t ni = (size_t)exp10 + 1;
        std::string ip = digits.substr(0, std::min(ni, digits.size()));
        ip.append(ni - ip.size(), '0');
        return sign + ip + "." + (digits.size() > ni ? digits.substr(ni) : std::string("0"));
    }
    return sign + digits.substr(0, 1) + "." + (digits.size() > 1 ? digits.substr(1) : std::string("0")) + "E" + std::to_string(exp10);
}

// Queue the device->host copies of the first nrows rows of every column of a result on `stream`.
int copy_columns(imm3_result* r, int64_t nrows, cudaStream_t stream) {
    imm3_db* db = r->db;
    for (int i = 0; i < r->ncols; i++) {
        const size_t bytes = (size_t)nrows * (size_t)r->widths[(size_t)i];
        if (r->h_cols[(size_t)i].cap < bytes || !r->h_cols[(size_t)i].p) {
            db->host_pool.release(r->h_cols[(size_t)i]);
            r->h_cols[(size_t)i] = Buf();
            int rc = db->host_pool.acquire(bytes, &r->h_cols[(size_t)i]);
            if (rc) return rc;
        }
        if (bytes) CUDA_TRY(cudaMemcpyAsync(r->h_cols[(size_t)i].p, r->d_cols[(size_t)i].p, bytes, cudaMemcpyDeviceToHost, stream));
    }
    return 0;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

const char* imm3_last_error(void) { return last_error(); }
int imm3_abi_version(void) { return IMM3_ABI_VERSION; }

int imm3_open(const char* data_dir, const imm3_open_opts* opts, imm3_db** out) {
    if (!data_dir || !out) return fail(IMM3_ERR_INVALID_ARG, "imm3_open: NULL argument");
    imm3_open_opts o = {0, 0, 1, 0};
    if (opts) o = *opts;
    if (o.world < 1 || o.rank < 0 || o.rank >= o.world) return fail(IMM3_ERR_INVALID_ARG, "imm3_open: rank %d of world %d", o.rank, o.world);
    std::unique_ptr<imm3_db> db(new imm3_db());
    db->dir = data_dir;
    db->device = o.device;
    db->rank = o.rank;
    db->world = o.world;
    db->flags = o.flags;
    db->host_only = (o.flags & IMM3_OPEN_HOST_ONLY) != 0;
    db->host_pool.pinned_host = true;
    const bool otrace = getenv("IMM3_OPEN_TRACE") != nullptr;  // phase times of the open path on stderr
    const double t_open0 = now_us();
    int rc = load_tables(db->dir, o.rank, o.world, &db->tables);
    if (rc) return rc;
    if (otrace) fprintf(stderr, "[imm3_open] metadata + validation %.1f ms (%d I/O threads)\n", (now_us() - t_open0) * 1e-3, io_threads());
    if (!db->host_only) {
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0) {
            cudaGetLastError();
            return fail(IMM3_ERR_CUDA, "no usable CUDA device (%s); this library has no CPU fallback",
                        e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        }
        if (o.device < 0 || o.device >= ndev) return fail(IMM3_ERR_INVALID_ARG, "imm3_open: device %d of %d", o.device, ndev);
        auto body = [&]() -> int {
            CUDA_TRY(cudaSetDevice(db->device));
            cudaDeviceProp prop;
            CUDA_TRY(cudaGetDeviceProperties(&prop, db->device));
            if (prop.major < 10) return fail(IMM3_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", db->device, prop.major, prop.minor);
            CUDA_TRY(configure_device());
            db->num_sms = prop.multiProcessorCount;
            if (const char* g = getenv("IMM3_L2_FETCH")) {  // experiment: DRAM->L2 fetch granularity hint (32 / 64 / 128 bytes)
                CUDA_TRY(cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)atoi(g)));
            }
            CUDA_TRY(cudaStreamCreateWithFlags(&db->own_stream, cudaStreamNonBlocking));
            db->stream = db->own_stream;
            CUDA_TRY(cudaEventCreate(&db->ev0));
            CUDA_TRY(cudaEventCreate(&db->ev1));
            CUDA_TRY(cudaEventCreate(&db->ev_mid));
            CUDA_TRY(cudaMalloc(&db->d_ctrl, sizeof(CtrlBlock)));
            CUDA_TRY(cudaMemsetAsync(db->d_ctrl, 0, sizeof(CtrlBlock), db->stream));
            CUDA_TRY(cudaMallocHost(&db->h_ctrl, sizeof(CtrlBlock)));
            std::memset(db->h_ctrl, 0, sizeof(CtrlBlock));
            if (const char* e = getenv("IMM3_COMM_TIMEOUT_MS")) db->comm_timeout_ns = (unsigned long long)std::max(1, atoi(e)) * 1000000ull;
            if (otrace) fprintf(stderr, "[imm3_open] device + stream setup at %.1f ms\n", (now_us() - t_open0) * 1e-3);
            return upload_all(db.get());
        };
        rc = body();
        if (rc) {
            std::string why = last_error();
            free_device_side(db.get());
            return fail(rc, "%s", why.c_str());
        }
    }
    *out = db.release();
    return 0;
}

int imm3_close(imm3_db* db) {
    if (!db) return 0;
    // Results borrow buffers from the db's pools and dereference it in fetch / wait / free: closing under them would be a
    // use-after-free.  The caller frees its results first (the Python mirror does so in SegmentManager.close).
    if (db->live_results > 0)
        return fail(IMM3_ERR_STATE, "imm3_close: %d result(s) of this handle are still open (imm3_result_free them first)", db->live_results);
    free_device_side(db);
    delete db;
    return 0;
}

// ---- count exchange over NVLink peer memory -----------------------------------------------------
int imm3_comm_local_handle(imm3_db* db, void* handle_out) {
    if (!db || !handle_out) return fail(IMM3_ERR_INVALID_ARG, "imm3_comm_local_handle: NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == IMM3_COMM_HANDLE_BYTES, "IMM3_COMM_HANDLE_BYTES must be sizeof(cudaIpcMemHandle_t)");
    int rc = use_device(db);
    if (rc) return rc;
    if (db->world > kMaxWorld) return fail(IMM3_ERR_UNSUPPORTED, "count exchange supports at most %d ranks (world = %d)", kMaxWorld, db->world);
    if (!db->d_mailbox) {
        CUDA_TRY(cudaMalloc(&db->d_mailbox, kCommAllocBytes));  // the mailbox ring, then the exchange area of global aggregates
        CUDA_TRY(cudaMemset(db->d_mailbox, 0, kMailboxBytes));
    }
    cudaIpcMemHandle_t h;
    CUDA_TRY(cudaIpcGetMemHandle(&h, db->d_mailbox));
    std::memcpy(handle_out, &h, sizeof h);
    return 0;
}

int imm3_comm_connect(imm3_db* db, const void* handles, int nhandles) {
    if (!db || !handles) return fail(IMM3_ERR_INVALID_ARG, "imm3_comm_connect: NULL argument");
    int rc = use_device(db);
    if (rc) return rc;
    if (nhandles != db->world) return fail(IMM3_ERR_INVALID_ARG, "imm3_comm_connect: %d handles for a world of %d", nhandles, db->world);
    if (!db->d_mailbox) return fail(IMM3_ERR_STATE, "imm3_comm_connect: call imm3_comm_local_handle first");
    if (db->comm_on) return fail(IMM3_ERR_STATE, "imm3_comm_connect: already connected");
    for (int i = 0; i < db->world; i++) {
        if (i == db->rank) {
            db->comm_peer[i] = db->d_mailbox;
            continue;
        }
        cudaIpcMemHandle_t h;
        std::memcpy(&h, (const uint8_t*)handles + (size_t)i * sizeof h, sizeof h);
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            for (int k = 0; k < i; k++) {
                if (db->comm_peer[k] && db->comm_peer[k] != db->d_mailbox) cudaIpcCloseMemHandle(db->comm_peer[k]);
                db->comm_peer[k] = nullptr;
            }
            return fail(IMM3_ERR_COMM, "imm3_comm_connect: cannot map the mailbox of rank %d (%s); the ranks must be processes on one NVLink-connected node", i,
                        cudaGetErrorString(e));
        }
        db->comm_peer[i] = (unsigned long long*)p;
    }
    db->comm_on = db->world > 1;
    db->comm_epoch = 0;
    db->agg_seq = 0;
    return 0;
}

int imm3_table_count(imm3_db* db) { return db ? (int)db->tables.size() : IMM3_ERR_INVALID_ARG; }

const char* imm3_table_name(imm3_db* db, int idx) {
    if (!db || idx < 0 || idx >= (int)db->tables.size()) return nullptr;
    return db->tables[(size_t)idx].meta.name.c_str();
}

int imm3_table_info(imm3_db* db, const char* table, imm3_table_desc* out) {
    if (!db || !out) return fail(IMM3_ERR_INVALID_ARG, "imm3_table_info: NULL argument");
    TableStore* t = find_table(db, table);
    if (!t) return IMM3_ERR_NOT_FOUND;
    out->ncols = (int)t->cols.size();
    out->block_size = t->meta.block_size;
    out->nsegments = t->nsegments;
    out->seg_begin = t->seg_begin;
    out->seg_end = t->seg_end;
    out->nrows = t->nrows;
    out->nblocks = t->nblocks;
    out->resident_bytes = 0;
    for (auto& c : t->cols) out->resident_bytes += c.encoded_bytes;
    return 0;
}

int imm3_column_info(imm3_db* db, const char* table, int col_idx, imm3_column_desc* out) {
    if (!db || !out) return fail(IMM3_ERR_INVALID_ARG, "imm3_column_info: NULL argument");
    TableStore* t = find_table(db, table);
    if (!t) return IMM3_ERR_NOT_FOUND;
    if (col_idx < 0 || col_idx >= (int)t->cols.size()) return fail(IMM3_ERR_NOT_FOUND, "column index %d out of range", col_idx);
    const ColumnStore& c = t->cols[(size_t)col_idx];
    std::memset(out, 0, sizeof *out);
    snprintf(out->name, sizeof out->name, "%s", c.meta.name.c_str());
    out->column_type = c.meta.ctype;
    out->codec = c.meta.codec;
    out->width = c.meta.width;
    out->encoded_bytes = c.encoded_bytes;
    return 0;
}

int imm3_segment_file_id(imm3_db* db, const char* table, int canonical_idx, int32_t* out_id) {
    if (!db || !out_id) return fail(IMM3_ERR_INVALID_ARG, "imm3_segment_file_id: NULL argument");
    TableStore* t = find_table(db, table);
    if (!t) return IMM3_ERR_NOT_FOUND;
    if (canonical_idx < 0 || canonical_idx >= t->nsegments) return fail(IMM3_ERR_NOT_FOUND, "segment index %d out of range", canonical_idx);
    *out_id = t->file_ids[(size_t)canonical_idx];
    return 0;
}

int imm3_set_stream(imm3_db* db, void* cuda_stream) {
    if (!db) return fail(IMM3_ERR_INVALID_ARG, "imm3_set_stream: db is NULL");
    int rc = use_device(db);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(db->stream));
    db->stream = cuda_stream ? (cudaStream_t)cuda_stream : db->own_stream;
    return 0;
}

int imm3_sync(imm3_db* db) {
    if (!db) return fail(IMM3_ERR_INVALID_ARG, "imm3_sync: db is NULL");
    int rc = use_device(db);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(db->stream));
    return 0;
}

int imm3_reupload(imm3_db* db, const char* table, const char* const* cols, int ncols, int64_t* out_bytes) {
    if (!db) return fail(IMM3_ERR_INVALID_ARG, "imm3_reupload: db is NULL");
    int rc = use_device(db);
    if (rc) return rc;
    if (!(db->flags & IMM3_OPEN_KEEP_HOST)) return fail(IMM3_ERR_STATE, "imm3_reupload needs IMM3_OPEN_KEEP_HOST");
    TableStore* t = find_table(db, table);
    if (!t) return IMM3_ERR_NOT_FOUND;
    int64_t bytes = 0;
    for (auto& c : t->cols) {
        bool want = ncols <= 0 || !cols;
        for (int i = 0; !want && i < ncols; i++) want = cols[i] && c.meta.name == cols[i];
        if (!want || !c.encoded_bytes) continue;
        if ((rc = ensure_mirror(db, c))) return rc;  // first use: pin + read the column's files once
        CUDA_TRY(cudaMemcpyAsync(c.d_arena, c.h_mirror, (size_t)c.encoded_bytes, cudaMemcpyHostToDevice, db->stream));
        bytes += c.encoded_bytes;
    }
    if (ncols > 0 && cols)
        for (int i = 0; i < ncols; i++) {
            bool found = false;
            for (auto& c : t->cols) found = found || (cols[i] && c.meta.name == cols[i]);
            if (!found) return fail(IMM3_ERR_NOT_FOUND, "Column %s does not exist in table %s", cols[i] ? cols[i] : "(null)", t->meta.name.c_str());
        }
    if (out_bytes) *out_bytes = bytes;
    return 0;
}

int imm3_explain(imm3_db* db, const char* table, const imm3_pred* preds, int npreds, const char* const* proj_cols,
                 int nproj, int64_t limit, const char** json) {
    if (!db || !json) return fail(IMM3_ERR_INVALID_ARG, "imm3_explain: NULL argument");
    Prepared pr;
    int rc = prepare(db, table, preds, npreds, proj_cols, nproj, limit, false, &pr);
    if (rc) return rc;
    db->explain_buf = explain_json(pr.lp, explain_kernel(db, pr));
    *json = db->explain_buf.c_str();
    return 0;
}

namespace {

// Validation and logical plan of every term, before any device work.  A term that can never hold (a wrong-length literal, an
// empty range) drops out of a disjunction; the first term that can hold carries the query, the others only add their filter
// kernels.
int plan_terms(imm3_db* db, const char* table, const std::vector<std::pair<const imm3_pred*, int>>& terms, const char* const* proj_cols,
               int nproj, int64_t limit, std::unique_ptr<Prepared>* main, std::vector<std::unique_ptr<Prepared>>* extra) {
    std::vector<std::unique_ptr<Prepared>> prepared;
    for (auto& tm : terms) {
        prepared.emplace_back(new Prepared());
        if (int rc = prepare(db, table, tm.first, tm.second, proj_cols, nproj, limit, false, prepared.back().get())) return rc;
    }
    size_t main_i = 0;
    while (main_i + 1 < prepared.size() && prepared[main_i]->lp.always_empty) main_i++;
    *main = std::move(prepared[main_i]);
    for (size_t i = main_i + 1; i < prepared.size(); i++)
        if (!prepared[i]->lp.always_empty) extra->push_back(std::move(prepared[i]));
    return 0;
}

// How a disjunction runs: every term's filter kernel over the row space, ORing into one bitmap (launch_row_space_filter), or -
// block_or: encoded_or and a term tests an encoded column - every term's block filter front, merged in block space
// (launch_or_merges).
int choose_or(const Prepared& pr, const std::vector<std::unique_ptr<Prepared>>& extra, bool encoded_or, bool* block_or) {
    if (!encoded_or || extra.empty()) return 0;
    *block_or = has_encoded_filter(pr);
    for (auto& tm : extra) *block_or = *block_or || has_encoded_filter(*tm);
    const TableStore& t = *pr.table;
    if (*block_or && std::max(t.max_block_rows, t.meta.block_size) > 1024)
        return fail(IMM3_ERR_UNSUPPORTED, "imm3_query_begin_dnf_ext: a disjunction over a sorted-int-codec column filters blocks of at most 1024 rows, table %s has blocks of %d",
                    t.meta.name.c_str(), std::max(t.max_block_rows, t.meta.block_size));
    return 0;
}

// The result's schema, and a device column of up to `limit` rows per projected column.
int result_columns(imm3_db* db, const Prepared& pr, int64_t limit, imm3_result* r) {
    const TableStore& t = *pr.table;
    const int64_t capacity = limit > 0 ? std::min<int64_t>(limit, t.nrows) : t.nrows;
    r->ncols = (int)pr.lp.proj.size();
    for (int i = 0; i < r->ncols; i++) {
        const ColumnMeta& c = t.meta.cols[(size_t)pr.lp.proj[(size_t)i]];
        r->names.push_back(c.name);
        r->types.push_back(c.ctype);
        r->widths.push_back(c.width);
        Buf b;
        if (int rc = db->dev_pool.acquire((size_t)capacity * (size_t)c.width, &b)) return rc;
        r->d_cols.push_back(b);
        r->h_cols.emplace_back();
    }
    return 0;
}

// The device plans of the main term, which writes the result's columns, and of the OR terms.
int plan_device(imm3_db* db, Prepared* pr, std::vector<std::unique_ptr<Prepared>> extra, bool block_or, const imm3_result& r) {
    if (block_or) {
        force_blocks(pr);
        for (auto& tm : extra) force_blocks(tm.get());
    }
    int rc = fill_scan_plan(db, pr);
    if (rc) return rc;
    for (int i = 0; i < r.ncols; i++) pr->sp.proj[i].out = (uint8_t*)r.d_cols[(size_t)i].p;
    if (block_or) {
        pr->or_terms = std::move(extra);
        return fill_or_terms_plan(db, pr);
    }
    if (extra.empty()) return 0;
    // real OR: every term's predicates are decided by the row-space filter kernel (dense columns); a disjunction over
    // an encoded column would need the block filter kernels to accumulate as well - not built
    auto row_space = [](const Prepared& p) { return p.pipeline == Pipeline::kDense || p.pipeline == Pipeline::kRowSpace; };
    bool ok = row_space(*pr);
    for (auto& tm : extra) {
        if ((rc = fill_scan_plan(db, tm.get()))) return rc;
        ok = ok && row_space(*tm);
        tm->sp.or_accumulate = 1;
    }
    if (!ok) return fail(IMM3_ERR_UNSUPPORTED, "imm3_query_begin_dnf: a disjunction needs every predicate on a dense (DENSE_INT / DENSE_TINYINT / DENSE_STRING) column");
    pr->or_terms = std::move(extra);
    return 0;
}

// This rank's scan, or - its slice is empty (more ranks than segments) - its part in every round of the exchange.  (A
// predicate that can never hold is a property of the query, known to every rank: nobody exchanges anything.)
int run_query(imm3_db* db, const Prepared& pr, bool local, Run* run, imm3_result* r) {
    if (local) {
        const int rc = run_scan(db, pr, run, &r->local_count);
        r->timing_seq = db->ev_seq;
        return rc;
    }
    if (!db->comm_on || pr.lp.always_empty) return 0;
    const int64_t lim = pr.lp.limit > 0 ? pr.lp.limit : INT64_MAX;
    int rc = exchange_only(db, run, lim, 0);
    if (!rc && small_limit(pr.lp) && (int64_t)db->h_ctrl->x.counts[0] < pr.lp.limit) rc = exchange_only(db, run, lim, 0);
    return rc;
}

// Global placement of this rank's rows (SURVEY.md 8e): from the on-device exchange, or trivially for a single handle.
void place_rows(const imm3_db* db, const LogicalPlan& lp, imm3_result* r) {
    r->world = db->comm_on ? db->world : 1;
    r->g_offset = 0;
    r->g_take = r->g_total = r->local_count;
    r->rank_counts[0] = r->local_count;
    if (!db->comm_on || lp.always_empty) return;
    const CommOut& x = db->h_ctrl->x;
    r->g_offset = (int64_t)x.g_offset;
    r->g_take = (int64_t)x.g_take;
    r->g_total = (int64_t)x.g_total;
    for (int i = 0; i < db->world; i++) r->rank_counts[i] = (int64_t)x.counts[i];
}

// Algorithmic bytes (SURVEY.md §8d): filter columns' encoded bytes once + per surviving row the
// project-only widths read and every projected width written (+ 4 B/block for PFOR offsets).
int64_t query_alg_bytes(const Prepared& pr, int64_t rows) {
    const TableStore& t = *pr.table;
    int64_t a = 0, per_row = 0;
    std::vector<int> seen;
    auto count_filters = [&](const LogicalPlan& lp) {
        for (auto& f : lp.filters) {
            if (std::find(seen.begin(), seen.end(), f.col_idx) != seen.end()) continue;  // (a column several terms of a disjunction test: once)
            const ColumnStore& c = t.cols[(size_t)f.col_idx];
            a += c.encoded_bytes + (c.meta.codec == IMM3_CODEC_PFOR_INT ? 4 * t.nblocks : 0);
            seen.push_back(f.col_idx);
        }
    };
    count_filters(pr.lp);
    for (auto& tm : pr.or_terms) count_filters(tm->lp);
    for (int ci : pr.lp.proj) {
        per_row += t.cols[(size_t)ci].meta.width;
        if (std::find(seen.begin(), seen.end(), ci) == seen.end()) {
            per_row += t.cols[(size_t)ci].meta.width;
            seen.push_back(ci);
        }
    }
    return a + per_row * rows;
}

// The launch record and the times: device and stage times, and the wall clock inside imm3_query_begin by phase - plan,
// buffers + device plan, launches, wait for the GPU, epilogue (two-phase LIMIT queries: the last phase's stamps).
void report_run(imm3_result* r, const Run& run, double t_in, double t_plan, double t_dev) {
    const double t_out = now_us();
    r->route = run.route;
    r->device_ms = run.device_ms;
    r->stage_ms[0] = run.stage_ms[0], r->stage_ms[1] = run.stage_ms[1];
    r->host_us[0] = t_plan - t_in;
    r->host_us[1] = t_dev - t_plan;
    if (run.t_launched > 0) {
        r->host_us[2] = run.t_launched - t_dev;
        r->host_us[3] = run.t_synced - run.t_launched;
        r->host_us[4] = t_out - run.t_synced;
    }
}

}  // namespace

// One conjunction (imm3_query_begin) or a disjunction of conjunctions (imm3_query_begin_dnf): terms[i] = (predicates, count).
// encoded_or (IMM3_DNF_ENCODED_FILTER): a disjunction whose terms test an encoded column runs on the block pipeline.
static int query_begin_terms(imm3_db* db, const char* table, const std::vector<std::pair<const imm3_pred*, int>>& terms,
                             const char* const* proj_cols, int nproj, int64_t limit, imm3_result** out, bool encoded_or = false) {
    if (!db || !out) return fail(IMM3_ERR_INVALID_ARG, "imm3_query_begin: NULL argument");
    const double t_in = now_us();
    std::unique_ptr<Prepared> pr;
    std::vector<std::unique_ptr<Prepared>> extra;
    bool block_or = false;
    int rc;
    if ((rc = plan_terms(db, table, terms, proj_cols, nproj, limit, &pr, &extra)) || (rc = choose_or(*pr, extra, encoded_or, &block_or)) ||
        (rc = use_device(db)))
        return rc;
    const double t_plan = now_us();
    std::unique_ptr<imm3_result, int (*)(imm3_result*)> r(new imm3_result(), imm3_result_free);  // (every error path: buffers back to the pools)
    r->db = db;
    db->live_results++;
    const bool local = !pr->lp.always_empty && pr->table->nrows > 0;
    if ((rc = result_columns(db, *pr, limit, r.get())) || (local && (rc = plan_device(db, pr.get(), std::move(extra), block_or, *r)))) return rc;
    const double t_dev = local ? now_us() : t_plan;
    Run run;
    if ((rc = run_query(db, *pr, local, &run, r.get()))) return rc;
    place_rows(db, pr->lp, r.get());
    r->alg_bytes = query_alg_bytes(*pr, r->local_count);
    report_run(r.get(), run, t_in, t_plan, t_dev);
    *out = r.release();
    return 0;
}

int imm3_query_begin(imm3_db* db, const char* table, const imm3_pred* preds, int npreds, const char* const* proj_cols,
                     int nproj, int64_t limit, imm3_result** out) {
    if (npreds < 0 || (npreds > 0 && !preds)) return fail(IMM3_ERR_INVALID_ARG, "imm3_query_begin: predicates");
    return query_begin_terms(db, table, {{preds, npreds}}, proj_cols, nproj, limit, out);
}

static int query_begin_dnf(imm3_db* db, const char* table, const imm3_pred* preds, const int32_t* term_sizes, int nterms,
                           const char* const* proj_cols, int nproj, int64_t limit, bool encoded_or, imm3_result** out) {
    if (!term_sizes || nterms < 1 || nterms > IMM3_MAX_OR_TERMS) return fail(IMM3_ERR_INVALID_ARG, "imm3_query_begin_dnf: 1 .. %d terms", IMM3_MAX_OR_TERMS);
    std::vector<std::pair<const imm3_pred*, int>> terms;
    int at = 0;
    for (int i = 0; i < nterms; i++) {
        if (term_sizes[i] < 0 || (term_sizes[i] > 0 && !preds)) return fail(IMM3_ERR_INVALID_ARG, "imm3_query_begin_dnf: term %d", i);
        if (term_sizes[i] == 0) return query_begin_terms(db, table, {{nullptr, 0}}, proj_cols, nproj, limit, out);  // `... or true`: every row
        terms.push_back({preds + at, term_sizes[i]});
        at += term_sizes[i];
    }
    return query_begin_terms(db, table, terms, proj_cols, nproj, limit, out, encoded_or);
}

int imm3_query_begin_dnf(imm3_db* db, const char* table, const imm3_pred* preds, const int32_t* term_sizes, int nterms,
                         const char* const* proj_cols, int nproj, int64_t limit, imm3_result** out) {
    return query_begin_dnf(db, table, preds, term_sizes, nterms, proj_cols, nproj, limit, false, out);
}

int imm3_query_begin_dnf_ext(imm3_db* db, const char* table, const imm3_pred* preds, const int32_t* term_sizes, int nterms,
                             const char* const* proj_cols, int nproj, int64_t limit, uint32_t flags, imm3_result** out) {
    const uint32_t known = IMM3_DNF_ENCODED_FILTER;
    if (flags & ~known) return fail(IMM3_ERR_INVALID_ARG, "imm3_query_begin_dnf_ext: unknown flag bits 0x%x", flags & ~known);
    return query_begin_dnf(db, table, preds, term_sizes, nterms, proj_cols, nproj, limit, (flags & IMM3_DNF_ENCODED_FILTER) != 0, out);
}

int64_t imm3_result_local_count(const imm3_result* r) { return r ? r->local_count : IMM3_ERR_INVALID_ARG; }
int64_t imm3_result_global_offset(const imm3_result* r) { return r ? r->g_offset : IMM3_ERR_INVALID_ARG; }
int64_t imm3_result_take(const imm3_result* r) { return r ? r->g_take : IMM3_ERR_INVALID_ARG; }
int64_t imm3_result_global_count(const imm3_result* r) { return r ? r->g_total : IMM3_ERR_INVALID_ARG; }
int imm3_result_rank_counts(const imm3_result* r, int64_t* counts, int cap) {
    if (!r || !counts || cap < r->world) return fail(IMM3_ERR_INVALID_ARG, "imm3_result_rank_counts: need room for %d counts", r ? r->world : 0);
    for (int i = 0; i < r->world; i++) counts[i] = r->rank_counts[i];
    return r->world;
}

int imm3_result_fetch(imm3_result* r, int64_t nrows) {
    if (!r) return fail(IMM3_ERR_INVALID_ARG, "imm3_result_fetch: result is NULL");
    if (nrows < 0 || nrows > r->local_count) return fail(IMM3_ERR_INVALID_ARG, "imm3_result_fetch: %lld rows of %lld", (long long)nrows, (long long)r->local_count);
    if (r->agg_first_col >= 0) return 0;  // (aggregate results are materialised on the host by imm3_query_agg)
    imm3_db* db = r->db;
    int rc = use_device(db);
    if (rc) return rc;
    if ((rc = copy_columns(r, nrows, db->stream))) return rc;
    CUDA_TRY(cudaStreamSynchronize(db->stream));
    r->fetched = nrows;
    return 0;
}

int imm3_result_fetch_async(imm3_result* r, int64_t nrows) {
    if (!r) return fail(IMM3_ERR_INVALID_ARG, "imm3_result_fetch_async: result is NULL");
    if (nrows < 0 || nrows > r->local_count) return fail(IMM3_ERR_INVALID_ARG, "imm3_result_fetch_async: %lld rows of %lld", (long long)nrows, (long long)r->local_count);
    if (r->agg_first_col >= 0) return 0;
    imm3_db* db = r->db;
    int rc = use_device(db);
    if (rc) return rc;
    if (!db->copy_stream) CUDA_TRY(cudaStreamCreateWithFlags(&db->copy_stream, cudaStreamNonBlocking));
    // (imm3_query_begin returned after the kernels had finished: the rows are final, the copy stream needs no event)
    if ((rc = copy_columns(r, nrows, db->copy_stream))) return rc;
    if (!r->copied) CUDA_TRY(cudaEventCreateWithFlags(&r->copied, cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(r->copied, db->copy_stream));
    r->pending = nrows;
    return 0;
}

int imm3_result_wait(imm3_result* r) {
    if (!r) return fail(IMM3_ERR_INVALID_ARG, "imm3_result_wait: result is NULL");
    if (r->pending < 0) return 0;  // nothing in flight
    int rc = use_device(r->db);
    if (rc) return rc;
    CUDA_TRY(cudaEventSynchronize(r->copied));
    r->fetched = r->pending;
    r->pending = -1;
    return 0;
}

int imm3_query(imm3_db* db, const char* table, const imm3_pred* preds, int npreds, const char* const* proj_cols,
               int nproj, int64_t limit, imm3_result** out) {
    imm3_result* r = nullptr;
    int rc = imm3_query_begin(db, table, preds, npreds, proj_cols, nproj, limit, &r);
    if (rc) return rc;
    if ((rc = imm3_result_fetch(r, r->g_take))) {  // (a single handle: all local rows; with a communicator: this rank's share)
        std::string why = last_error();
        imm3_result_free(r);
        return fail(rc, "%s", why.c_str());
    }
    *out = r;
    return 0;
}

namespace {

// An aggregate between the steps of query_agg.
struct AggQuery {
    const char* fn = nullptr;        // the entry point, in messages
    bool xchg = false;               // a global aggregate of a sharded handle: the ranks' groups are merged over the communicator
    Prepared pr;                     // the validated logical plan; the filter front's device plan after plan_agg_slice
    AggPlan ap;                      // naggs: the visible aggregates and a hidden COUNT
    AggShape shape{};                // the aggregation kernel's instantiation
    std::unique_ptr<imm3_result> r;  // schema from plan_agg, rows from agg_rows
    std::vector<int> pfor_cols;      // distinct sorted-int-codec columns decoded per block (MIN / MAX / SUM inputs, group columns)
    int count_slot = -1;             // the plan's first COUNT (a SUM / AVG query's group sizes)
    bool has_sum = false;
    bool enc_filter = false;         // a predicate on a sorted-int-codec column: the block filter front decides it
    int smem_optin = 0;              // agg_blocks_kernel: the device's shared memory per CTA (cudaDevAttrMaxSharedMemoryPerBlockOptin)
    size_t blocks_smem = 0;          // ... and what one of its CTAs needs (size_agg_blocks)
};

// Validation and plan of an aggregate, before any device work: group and aggregate columns, the result schema, the COUNT a
// SUM / AVG query carries, the encoded predicates and the hash table's size.
int plan_agg(imm3_db* db, const char* table, const imm3_pred* preds, int npreds, const imm3_agg* aggs, int naggs, const char* const* group_cols,
             int ngroup, bool global, bool allow_sum_avg, bool encoded_filter, bool have_out, AggQuery* q) {
    const char* const fn = q->fn = global ? "imm3_query_agg_global" : "imm3_query_agg";
    if (!db || !have_out || (naggs > 0 && !aggs) || (ngroup > 0 && !group_cols)) return fail(IMM3_ERR_INVALID_ARG, "%s: NULL argument", fn);
    // A sharded handle merges over the communicator; a single handle's partials are the global result already.
    q->xchg = global && db->world > 1;
    if (q->xchg && !db->comm_on)
        return fail(IMM3_ERR_STATE, "%s: a sharded handle (rank %d of %d) merges over the communicator: call imm3_comm_connect first", fn, db->rank, db->world);
    if (naggs < 1) return fail(IMM3_ERR_INVALID_ARG, "%s: no aggregates", fn);
    if (naggs > kMaxAggs) return fail(IMM3_ERR_UNSUPPORTED, "%s: at most %d aggregates", fn, kMaxAggs);
    if (ngroup > kMaxGroupCols) return fail(IMM3_ERR_UNSUPPORTED, "%s: at most %d group-by columns", fn, kMaxGroupCols);
    Prepared& pr = q->pr;
    int rc = prepare(db, table, preds, npreds, nullptr, 0, 0, false, &pr);
    if (rc) return rc;
    const TableStore& t = *pr.table;
    AggPlan& ap = q->ap;
    std::memset(&ap, 0, sizeof ap);
    q->r.reset(new imm3_result());
    imm3_result* const r = q->r.get();
    r->db = db;
    for (int i = 0; i < kMaxAggs; i++) ap.agg_pfor[i] = -1;
    for (int i = 0; i < kMaxGroupCols; i++) ap.group_pfor[i] = -1;
    int key_bits = 0;
    for (int g = 0; g < ngroup; g++) {
        const int ci = find_col(t.meta, group_cols[g]);
        if (ci < 0) return fail(IMM3_ERR_NOT_FOUND, "Column %s does not exist in table %s", group_cols[g] ? group_cols[g] : "(null)", t.meta.name.c_str());
        const ColumnStore& c = t.cols[(size_t)ci];
        if (key_bits + 8 * c.meta.width > 56) return fail(IMM3_ERR_UNSUPPORTED, "group-by cells must pack into 7 bytes");
        ap.group[g].base = c.d_arena;
        ap.group[g].width = c.meta.width;
        ap.group[g].key_shift = key_bits;
        ap.group_pfor[g] = (int8_t)pfor_slot(t, &q->pfor_cols, ci);
        key_bits += 8 * c.meta.width;
        r->names.push_back(c.meta.name);
        r->types.push_back(c.meta.ctype);
        r->widths.push_back(c.meta.width);
    }
    for (int a = 0; a < naggs; a++) {
        const int ci = find_col(t.meta, aggs[a].col);
        if (ci < 0) return fail(IMM3_ERR_NOT_FOUND, "Column %s does not exist in table %s", aggs[a].col ? aggs[a].col : "(null)", t.meta.name.c_str());
        const ColumnStore& c = t.cols[(size_t)ci];
        const char* suffix = "_count";
        int rtype = IMM3_COL_DOUBLE;
        if (aggs[a].op == IMM3_AGG_COUNT) {
            ap.agg[a].op = kAggCount;
            rtype = IMM3_COL_COUNT;
            if (q->count_slot < 0) q->count_slot = a;
        } else if (aggs[a].op == IMM3_AGG_MIN || aggs[a].op == IMM3_AGG_MAX) {
            if (c.meta.ctype == IMM3_COL_STRING)
                return fail(IMM3_ERR_UNSUPPORTED, "min / max on a STRING column (the reference maps both to MaxStringAggr, Engine.scala:137,147)");
            ap.agg[a].op = aggs[a].op == IMM3_AGG_MIN ? kAggMin : kAggMax;
            ap.agg_pfor[a] = (int8_t)pfor_slot(t, &q->pfor_cols, ci);  // (COUNT never reads its column)
            suffix = aggs[a].op == IMM3_AGG_MIN ? "_min" : "_max";
        } else if (allow_sum_avg && (aggs[a].op == IMM3_AGG_SUM || aggs[a].op == IMM3_AGG_AVG)) {
            if (c.meta.ctype == IMM3_COL_STRING) return fail(IMM3_ERR_UNSUPPORTED, "sum / avg on a STRING column (%s)", c.meta.name.c_str());
            ap.agg[a].op = kAggSum;  // (AVG = the SUM over the group's COUNT, divided on the host)
            ap.agg_pfor[a] = (int8_t)pfor_slot(t, &q->pfor_cols, ci);
            q->has_sum = true;
            suffix = aggs[a].op == IMM3_AGG_SUM ? "_sum" : "_avg";
            if (aggs[a].op == IMM3_AGG_SUM) rtype = IMM3_COL_INT64;
            else r->avg_cols |= 1u << a;
        } else {
            return fail(IMM3_ERR_UNSUPPORTED, "Unknown Aggregate type (Engine.scala:153: only Min, Max and Count are resolved)");
        }
        ap.agg[a].base = c.d_arena;
        ap.agg[a].width = c.meta.width;
        r->names.push_back(c.meta.name + suffix);  // alias.getOrElse(col + "_max"), Engine.scala:136-152
        r->types.push_back(rtype);
        r->widths.push_back(8);
    }
    // A SUM / AVG query carries one COUNT of the group's rows: the query's own, else a hidden one behind the visible
    // aggregates (in the plan, never in the result).
    ap.naggs = naggs;
    if (q->has_sum && q->count_slot < 0) {
        if (naggs + 1 > kMaxAggs)
            return fail(IMM3_ERR_UNSUPPORTED, "imm3_query_agg_ext: at most %d aggregates, including the COUNT a sum / avg query carries (the query has %d and no COUNT)",
                        kMaxAggs, naggs);
        q->count_slot = ap.naggs++;
        ap.agg[q->count_slot].op = kAggCount;
        ap.agg[q->count_slot].width = 4;
    }
    r->ncols = ngroup + naggs;
    r->agg_first_col = ngroup;
    r->h_cols.resize((size_t)r->ncols);
    ap.ngroup = ngroup;
    // A predicate on a sorted-int-codec column: the block filter front decides it (IMM3_AGG_ENCODED_FILTER only).
    for (auto& f : pr.lp.filters)
        if (is_pfor(t, f.col_idx)) {
            if (!encoded_filter)
                return fail(IMM3_ERR_UNSUPPORTED, "aggregation with a predicate on a sorted-int-codec column (%s) is not supported yet", t.cols[(size_t)f.col_idx].meta.name.c_str());
            q->enc_filter = true;
        }
    // A MIN / MAX input or a group column in the sorted-int codec: agg_blocks_kernel decodes them block by block.  It also
    // aggregates every block-space selection (blocks are not aligned to agg_kernel's 1024-row spans).
    q->shape = agg_shape(ap, !q->pfor_cols.empty() || q->enc_filter, q->enc_filter);
    if (q->pfor_cols.size() > (size_t)kMaxPforCols)
        return fail(IMM3_ERR_UNSUPPORTED, "aggregation decodes at most %d distinct sorted-int-codec columns, the query reads %zu", kMaxPforCols, q->pfor_cols.size());
    ap.table_slots = 1u << 16;
    if (const char* e = getenv("IMM3_AGG_SLOTS")) {  // (tests shrink it to exercise the overflow report)
        uint32_t v = (uint32_t)atoi(e);
        if (v >= 64 && (v & (v - 1)) == 0) ap.table_slots = v;
    }
    if (q->xchg && ap.table_slots > kAggXchgSlots)
        return fail(IMM3_ERR_UNSUPPORTED, "%s: IMM3_AGG_SLOTS = %u exceeds the exchange buffer of %u groups", fn, ap.table_slots, kAggXchgSlots);
    return 0;
}

// Limits of this rank's slice (query_agg's refuse_slice applies them).  Blocks of more than 1024 rows, before any device
// work: agg_blocks_kernel decodes, and the block filter front filters, no larger ones (the single-pass kernel, which takes
// larger blocks, leaves no block-space selection behind).
int check_agg_block_rows(const AggQuery& q) {
    const TableStore& t = *q.pr.table;
    if (t.max_block_rows <= 1024) return 0;
    if (!q.pfor_cols.empty())
        return fail(IMM3_ERR_UNSUPPORTED, "aggregation over sorted-int-codec columns decodes blocks of at most 1024 rows, table %s has a block of %d",
                    t.meta.name.c_str(), t.max_block_rows);
    if (q.enc_filter)
        return fail(IMM3_ERR_UNSUPPORTED, "aggregation with a predicate on a sorted-int-codec column filters blocks of at most 1024 rows, table %s has a block of %d",
                    t.meta.name.c_str(), t.max_block_rows);
    return 0;
}
// ... and, once the slice is planned, agg_blocks_kernel's shared memory against the device's opt-in limit.
int check_agg_smem(const AggQuery& q) {
    if (!q.shape.blocks || q.blocks_smem <= (size_t)q.smem_optin) return 0;
    return fail(IMM3_ERR_UNSUPPORTED, "aggregation over %d sorted-int-codec columns with %d aggregates needs %zu bytes of shared memory per CTA, the device has %d",
                q.ap.npfor, q.ap.naggs, q.blocks_smem, q.smem_optin);
}

// The device plans of this rank's slice: the filter front, then the AggPlan's columns.  An encoded predicate: the block
// pipeline's front (DESIGN §4.4d) leaves per block a count and - partially selected blocks only - 32 bitmap words, which
// agg_blocks_kernel<.., BS> reads.  Otherwise the dense filter kernel in row space, as for a Project query without a select list.
int plan_agg_slice(imm3_db* db, AggQuery* q) {
    Prepared& pr = q->pr;
    ScanPlan& sp = pr.sp;
    const TableStore& t = *pr.table;
    int rc = plan_columns(db, &pr);
    if (rc) return rc;
    if (q->enc_filter) {
        pr.pipeline = Pipeline::kBlocks;  // (IMM3_PATH=fused and IMM3_NO_HYBRID choose Project pipelines only)
        choose_block_filter(&pr);
    }
    rc = q->enc_filter ? size_block_front(&pr) : size_dense_filter(db, &pr);
    if (rc || (rc = plan_grid(db, &pr)) || (rc = q->enc_filter ? ensure_block_filter(db, pr, sp.ntiles, t.nblocks) : ensure_row_space(db, sp))) return rc;
    sp.scan_inline = q->enc_filter ? block_scan_inline(pr, sp.ntiles) : 1;  // (row space: only the total matters here, the last CTA's scan provides it)
    AggPlan& ap = q->ap;
    ap.nrows = t.nrows;
    ap.ntiles = sp.ntiles;
    if (q->shape.blocks) {
        int64_t words = 0;
        ap.npfor = (int)q->pfor_cols.size();
        for (int i = 0; i < ap.npfor; i++) {
            const ColumnStore& c = t.cols[(size_t)q->pfor_cols[(size_t)i]];
            ap.pfor[i].words = reinterpret_cast<const uint32_t*>(c.d_arena);
            ap.pfor[i].word_off = c.d_word_off;
            words = std::max<int64_t>(words, c.max_block_words);
        }
        q->blocks_smem = size_agg_blocks(&ap, q->shape, words);
        ap.nblocks = t.nblocks;
        ap.row_start = t.d_row_start;
        CUDA_TRY(cudaDeviceGetAttribute(&q->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, db->device));
    }
    return 0;
}

// Local step: empty table -> filter front -> aggregation kernel -> compaction of this rank's groups into `out`.
int launch_agg_local(imm3_db* db, const AggQuery* q, AggEntry* out, Run* run) {
    const Prepared& pr = q->pr;
    const ScanPlan& sp = pr.sp;
    AggEntry* const table = (AggEntry*)db->d_agg_table.p;
    unsigned int* const counters = (unsigned int*)db->d_agg_cnt.p;
    CUDA_TRY(launch_agg_init(table, q->ap.table_slots, q->ap, counters, db->stream));
    run->note("agg_init");
    if (q->enc_filter) {
        const int rc = launch_block_filter_front(db, pr, sp, pr.table->nblocks, run, nullptr, true, (uint32_t*)db->d_bitmap.p,
                                                 (uint32_t*)db->d_span_cnt.p);
        if (rc) return rc;
    } else {
        std::string route;
        CUDA_TRY(launch_filter(sp, (uint32_t*)db->d_bitmap.p, (uint32_t*)db->d_span_cnt.p, (uint32_t*)db->d_tile_cnt.p,
                               (unsigned long long*)db->d_tile_off.p, db->d_ctrl, pr.front.grid, pr.front.smem, db->stream, &route));
        run->note(route);
    }
    CUDA_TRY(launch_agg(q->ap, q->shape, (const uint32_t*)db->d_bitmap.p, (const uint32_t*)db->d_span_cnt.p, table, counters, db->d_ctrl,
                        db->num_sms, db->stream));
    run->note(agg_route(q->shape));
    CUDA_TRY(launch_agg_compact(table, q->ap.table_slots, out, counters, db->stream));
    run->note("agg_compact");
    return 0;
}

// This aggregate's exchange buffer of `rank`, as mapped here (DESIGN §4.3a: two per rank, used in turn).
AggEntry* agg_xbuf(const imm3_db* db, int rank) {
    return reinterpret_cast<AggEntry*>((uint8_t*)db->comm_peer[rank] + kAggXchgOff + (size_t)(db->agg_seq & 1u) * kAggXchgSlots * sizeof(AggEntry));
}

// Merge step of a global aggregate (DESIGN §4.3): this rank's group count - or that its slice ran nothing, or refused the
// query - posted to the peers -> a fresh table -> every rank's groups merged into it -> compaction into the result buffer.
int launch_agg_merge_step(imm3_db* db, const AggQuery& q, bool has_local, bool refused, Run* run) {
    const AggPlan& ap = q.ap;
    AggEntry* const table = (AggEntry*)db->d_agg_table.p;
    unsigned int* const counters = (unsigned int*)db->d_agg_cnt.p;
    AggXOut* const d_x = reinterpret_cast<AggXOut*>((uint8_t*)db->d_agg_cnt.p + 64);
    AggXPlan xp;
    std::memset(&xp, 0, sizeof xp);
    for (int i = 0; i < db->world; i++) xp.peer[i] = db->comm_peer[i];
    xp.rank = db->rank;
    xp.world = db->world;
    if (((++db->comm_epoch) & 0xFFFFFFu) == 0) ++db->comm_epoch;  // (the count exchange's rounds: tag 0 is an untouched mailbox)
    xp.epoch = db->comm_epoch;
    xp.has_local = has_local ? 1 : 0;
    xp.refused = refused ? 1 : 0;
    xp.timeout_ns = db->comm_timeout_ns;
    CUDA_TRY(launch_agg_exchange(xp, counters, db->d_ctrl, d_x, db->stream));
    run->note("agg_exchange");
    AggMergePlan mp;
    std::memset(&mp, 0, sizeof mp);
    for (int i = 0; i < db->world; i++) mp.buf[i] = agg_xbuf(db, i);
    db->agg_seq++;  // (posted: the next aggregate compacts into the other buffer)
    mp.world = db->world;
    mp.slots = ap.table_slots;
    mp.naggs = ap.naggs;
    for (int a = 0; a < ap.naggs; a++) mp.op[a] = ap.agg[a].op == kAggSum ? kAggCount : ap.agg[a].op;  // (a SUM merges as a COUNT: a 64-bit add)
    CUDA_TRY(launch_agg_init(table, ap.table_slots, ap, counters, db->stream));
    run->note("agg_init");
    CUDA_TRY(launch_agg_merge(mp, d_x, table, counters, db->num_sms, db->stream));
    run->note("agg_merge");
    CUDA_TRY(launch_agg_compact(table, ap.table_slots, (AggEntry*)db->d_agg_out.p, counters, db->stream));
    run->note("agg_compact");
    return 0;
}

// Read-back: the counters, the exchange's output and (local step) the control block, one synchronisation, the errors, the
// device time, the groups in first-row order and every rank's partial group count.
int read_agg_groups(imm3_db* db, const AggQuery& q, bool local, bool merge, const std::string& refusal, std::vector<AggEntry>* groups) {
    imm3_result* const r = q.r.get();
    const uint32_t slots = q.ap.table_slots;
    struct { unsigned int counters[16]; AggXOut x; } hc;
    static_assert(sizeof hc.counters == 64, "the exchange output sits 64 bytes into d_agg_cnt");
    if (local) CUDA_TRY(cudaMemcpyAsync(db->h_ctrl, db->d_ctrl, sizeof(CtrlBlock), cudaMemcpyDeviceToHost, db->stream));
    CUDA_TRY(cudaMemcpyAsync(&hc, db->d_agg_cnt.p, merge ? sizeof hc : sizeof hc.counters, cudaMemcpyDeviceToHost, db->stream));
    CUDA_TRY(cudaStreamSynchronize(db->stream));
    if (local && db->h_ctrl->c.error) return fail(IMM3_ERR_CUDA, "kernel watchdog fired (code %u)", db->h_ctrl->c.error);
    if (merge) {
        if (hc.x.late)
            return fail(IMM3_ERR_COMM, "aggregate exchange: a peer's groups were not announced within %llu ms (ranks must issue the same queries in the same order)",
                        db->comm_timeout_ns / 1000000ull);
        if (!refusal.empty()) return fail(IMM3_ERR_UNSUPPORTED, "%s", refusal.c_str());
        if ((hc.x.err_mask >> db->rank) & 1u) return fail(IMM3_ERR_UNSUPPORTED, "aggregation: more than %u groups in the slice of rank %d", slots, db->rank);
        if (hc.x.err_mask)
            return fail(IMM3_ERR_UNSUPPORTED, "%s: rank %d refused the query (more than %u groups in its slice, or a limit of its slice)", q.fn,
                        __builtin_ctz(hc.x.err_mask), slots);
    }
    if (hc.counters[1]) return fail(IMM3_ERR_UNSUPPORTED, "aggregation: more than %u groups", slots);
    float f = 0;
    CUDA_TRY(cudaEventElapsedTime(&f, db->ev0, db->ev1));
    r->device_ms = f;
    r->stage_ms[0] = f;
    groups->resize((size_t)hc.counters[0]);
    if (!groups->empty()) CUDA_TRY(cudaMemcpy(groups->data(), db->d_agg_out.p, groups->size() * sizeof(AggEntry), cudaMemcpyDeviceToHost));
    std::sort(groups->begin(), groups->end(), [](const AggEntry& x, const AggEntry& y) { return x.first_row < y.first_row; });
    if (merge)
        for (int i = 0; i < db->world; i++) r->rank_counts[i] = (int64_t)hc.x.counts[i];
    return 0;
}

// Algorithmic bytes of the local step: filter columns once + every decoded encoded column once (its words and 4 B of word
// offsets per block) + per selected row the cells of the dense group and aggregate columns (MIN / MAX / SUM / AVG inputs).
// (With a predicate on an encoded column: every filter column once, and an encoded column that is filtered and decoded once
// - its words once, plus the word offsets the decode reads.)
int64_t agg_alg_bytes(const AggQuery& q, int64_t selected_rows) {
    const TableStore& t = *q.pr.table;
    const AggPlan& ap = q.ap;
    int64_t bytes = 0, per_row = 0;
    std::vector<int> counted;
    auto seen = [&](int ci) { return std::find(counted.begin(), counted.end(), ci) != counted.end(); };
    for (auto& f : q.pr.lp.filters) {
        if (q.enc_filter && seen(f.col_idx)) continue;
        counted.push_back(f.col_idx);
        bytes += t.cols[(size_t)f.col_idx].encoded_bytes;
    }
    for (int ci : q.pfor_cols) bytes += (seen(ci) ? 0 : t.cols[(size_t)ci].encoded_bytes) + 4 * (int64_t)t.nblocks;
    for (int g = 0; g < ap.ngroup; g++)
        if (ap.group_pfor[g] < 0) per_row += ap.group[g].width;
    for (int a = 0; a < ap.naggs; a++)
        if (ap.agg[a].op != kAggCount && ap.agg_pfor[a] < 0) per_row += ap.agg[a].width;
    return bytes + per_row * selected_rows;
}

// The result's rows - group cells, then the aggregates (COUNT / SUM: int64, MIN / MAX / AVG: double) - and counts.
// SUM / AVG: every add on the way here was modulo 2^64, so a sum is exact when it fits int64 - certain for at most 2^32
// int32 inputs (2^32 x 2^31 <= 2^63); a larger group (on a global aggregate: the merged count) is refused, not wrapped.
int agg_rows(imm3_db* db, const AggQuery& q, const std::vector<AggEntry>& groups) {
    imm3_result* const r = q.r.get();
    const AggPlan& ap = q.ap;
    const int64_t n = (int64_t)groups.size();
    if (q.has_sum)
        for (const AggEntry& e : groups)
            if ((unsigned long long)e.val[q.count_slot] > (1ull << 32))
                return fail(IMM3_ERR_UNSUPPORTED, "imm3_query_agg_ext: a group of %lld rows: sum / avg are exact for groups of at most 2^32 rows", e.val[q.count_slot]);
    for (int c = 0; c < r->ncols; c++) {
        const size_t w = (size_t)r->widths[(size_t)c];
        if (const int rc = db->host_pool.acquire(std::max<size_t>(1, (size_t)n * w), &r->h_cols[(size_t)c])) {
            for (auto& b : r->h_cols) db->host_pool.release(b);
            return rc;
        }
        uint8_t* dst = (uint8_t*)r->h_cols[(size_t)c].p;
        for (int64_t i = 0; i < n; i++) {
            const AggEntry& e = groups[(size_t)i];
            if (c < ap.ngroup) {
                const unsigned long long cell = e.key >> ap.group[c].key_shift;
                for (size_t b = 0; b < w; b++) dst[(size_t)i * w + b] = (uint8_t)(cell >> (8 * b));
            } else {
                const int a = c - ap.ngroup;
                const bool avg = (r->avg_cols >> a) & 1u;
                double v = (double)e.val[a];  // MIN / MAX: value.toDouble, ProjectAggregate.scala:176-178
                if (avg) v /= (double)e.val[q.count_slot];  // AVG, once, in IEEE double
                if (ap.agg[a].op == kAggCount || (ap.agg[a].op == kAggSum && !avg)) std::memcpy(dst + (size_t)i * 8, &e.val[a], 8);
                else std::memcpy(dst + (size_t)i * 8, &v, 8);
            }
        }
    }
    r->local_count = r->fetched = r->g_take = r->g_total = n;  // (g_offset 0)
    r->world = q.xchg ? db->world : 1;  // (a global aggregate: rank_counts = every rank's partial group count)
    return 0;
}

// imm3_query_agg (global = false), imm3_query_agg_global and imm3_query_agg_ext, step by step.  The global form on a
// connected handle compacts this rank's partial groups into its exchange buffer instead of the result buffer and queues the
// exchange and the merge behind them (k_comm.cuh agg_exchange_kernel, k_agg.cuh agg_merge_kernel; DESIGN §4.3).
// allow_sum_avg (imm3_query_agg_ext only) resolves Sum / Avg (DESIGN §4.4c).
int query_agg(imm3_db* db, const char* table, const imm3_pred* preds, int npreds, const imm3_agg* aggs, int naggs, const char* const* group_cols,
              int ngroup, bool global, bool allow_sum_avg, bool encoded_filter, imm3_result** out) {
    AggQuery q;
    int rc = plan_agg(db, table, preds, npreds, aggs, naggs, group_cols, ngroup, global, allow_sum_avg, encoded_filter, out != nullptr, &q);
    if (rc) return rc;
    // Refusals that depend on this rank's slice: a global aggregate posts them to the peers (every rank then returns the
    // same status) instead of returning before the exchange.
    std::string refusal;
    auto refuse_slice = [&](int code) -> int {
        if (!code || !q.xchg) return code;
        refusal = last_error();
        return 0;
    };
    if ((rc = refuse_slice(check_agg_block_rows(q))) || (rc = use_device(db))) return rc;
    const bool merge = q.xchg && !q.pr.lp.always_empty;  // every rank of a connected handle takes part, an empty slice too
    bool local = !q.pr.lp.always_empty && q.pr.table->nrows > 0 && refusal.empty();
    if (local && ((rc = plan_agg_slice(db, &q)) || (rc = refuse_slice(check_agg_smem(q))))) return rc;
    local = local && refusal.empty();
    std::vector<AggEntry> groups;
    if (local || merge) {
        const size_t table_bytes = (size_t)q.ap.table_slots * sizeof(AggEntry);
        if ((rc = ensure_buf(&db->d_agg_table, table_bytes)) || (rc = ensure_buf(&db->d_agg_out, table_bytes)) ||
            (rc = ensure_buf(&db->d_agg_cnt, 64 + sizeof(AggXOut))))  // [groups, overflow] counters, then the exchange's AggXOut
            return rc;
        // every kernel noted (Run::note) between ev0 and ev1: the result's route and launch count; the local groups go to this
        // aggregate's exchange buffer when they are merged, else straight to the result buffer
        Run run;
        CUDA_TRY(cudaEventRecord(db->ev0, db->stream));
        if (local && (rc = launch_agg_local(db, &q, merge ? agg_xbuf(db, db->rank) : (AggEntry*)db->d_agg_out.p, &run))) return rc;
        if (merge && (rc = launch_agg_merge_step(db, q, local, !refusal.empty(), &run))) return rc;
        CUDA_TRY(cudaEventRecord(db->ev1, db->stream));
        q.r->route = run.route;
        if ((rc = read_agg_groups(db, q, local, merge, refusal, &groups))) return rc;
    }
    if (local) q.r->alg_bytes = agg_alg_bytes(q, (int64_t)db->h_ctrl->c.total);
    if ((rc = agg_rows(db, q, groups))) return rc;
    db->live_results++;
    *out = q.r.release();
    return 0;
}

}  // namespace

int imm3_query_agg(imm3_db* db, const char* table, const imm3_pred* preds, int npreds, const imm3_agg* aggs, int naggs,
                   const char* const* group_cols, int ngroup, imm3_result** out) {
    return query_agg(db, table, preds, npreds, aggs, naggs, group_cols, ngroup, false, false, false, out);
}

int imm3_query_agg_global(imm3_db* db, const char* table, const imm3_pred* preds, int npreds, const imm3_agg* aggs, int naggs,
                          const char* const* group_cols, int ngroup, imm3_result** out) {
    return query_agg(db, table, preds, npreds, aggs, naggs, group_cols, ngroup, true, false, false, out);
}

int imm3_query_agg_ext(imm3_db* db, const char* table, const imm3_pred* preds, int npreds, const imm3_agg* aggs, int naggs,
                       const char* const* group_cols, int ngroup, uint32_t flags, imm3_result** out) {
    const uint32_t known = IMM3_AGG_GLOBAL | IMM3_AGG_ENCODED_FILTER;
    if (flags & ~known) return fail(IMM3_ERR_INVALID_ARG, "imm3_query_agg_ext: unknown flag bits 0x%x", flags & ~known);
    return query_agg(db, table, preds, npreds, aggs, naggs, group_cols, ngroup, (flags & IMM3_AGG_GLOBAL) != 0, true, (flags & IMM3_AGG_ENCODED_FILTER) != 0, out);
}

int imm3_query_sql(imm3_db* db, const char* sql, imm3_result** out) {
    if (!db || !out) return fail(IMM3_ERR_INVALID_ARG, "imm3_query_sql: NULL argument");
    ParsedQuery q;
    int rc = parse_sql(sql, &q);
    if (rc) return rc;
    std::vector<const char*> proj;
    for (auto& s : q.proj) proj.push_back(s.c_str());
    return imm3_query(db, q.table.c_str(), q.preds.data(), (int)q.preds.size(), proj.data(), (int)proj.size(), q.limit, out);
}

int64_t imm3_result_nrows(const imm3_result* r) { return r ? r->fetched : IMM3_ERR_INVALID_ARG; }
int imm3_result_ncols(const imm3_result* r) { return r ? r->ncols : IMM3_ERR_INVALID_ARG; }
int imm3_result_col_type(const imm3_result* r, int c) { return (r && c >= 0 && c < r->ncols) ? r->types[(size_t)c] : IMM3_ERR_INVALID_ARG; }
int imm3_result_col_width(const imm3_result* r, int c) { return (r && c >= 0 && c < r->ncols) ? r->widths[(size_t)c] : IMM3_ERR_INVALID_ARG; }
const char* imm3_result_col_name(const imm3_result* r, int c) { return (r && c >= 0 && c < r->ncols) ? r->names[(size_t)c].c_str() : nullptr; }
const void* imm3_result_col_data(const imm3_result* r, int c) { return (r && c >= 0 && c < r->ncols) ? r->h_cols[(size_t)c].p : nullptr; }
const void* imm3_result_col_device(const imm3_result* r, int c) { return (r && c >= 0 && c < r->ncols && (size_t)c < r->d_cols.size()) ? r->d_cols[(size_t)c].p : nullptr; }
// Device times of a published query (plan.hpp) are read from the events on first use - as long as no later query has
// recorded them again (then the figure is gone: -1).
static void resolve_times(imm3_result* r) {
    if (r->device_ms >= 0 || !r->db || r->timing_seq == 0 || r->db->ev_seq != r->timing_seq) return;
    imm3_db* db = r->db;
    if (use_device(db)) return;
    float f = 0;
    if (cudaEventSynchronize(db->ev1) != cudaSuccess || cudaEventElapsedTime(&f, db->ev0, db->ev1) != cudaSuccess) return;
    r->device_ms = f;
    r->stage_ms[0] = f;
}
double imm3_result_device_ms(const imm3_result* r) {
    if (!r) return -1.0;
    resolve_times(const_cast<imm3_result*>(r));
    return r->device_ms;
}
int imm3_result_kernel_launches(const imm3_result* r) { return r ? (r->route.empty() ? 0 : 1 + (int)std::count(r->route.begin(), r->route.end(), ';')) : IMM3_ERR_INVALID_ARG; }
const char* imm3_result_route(const imm3_result* r) { return r ? r->route.c_str() : nullptr; }
double imm3_result_host_us(const imm3_result* r, int phase) { return (r && phase >= 0 && phase < 5) ? r->host_us[phase] : -1.0; }
double imm3_result_stage_ms(const imm3_result* r, int stage) {
    if (!r || stage < 0 || stage >= 2) return -1.0;
    resolve_times(const_cast<imm3_result*>(r));
    return r->stage_ms[stage];
}
int64_t imm3_result_algorithmic_bytes(const imm3_result* r) { return r ? r->alg_bytes : IMM3_ERR_INVALID_ARG; }

// Row.toString = xs.mkString("Row(", ",", ")")  (Record.scala:13)
int imm3_result_format_row(const imm3_result* r, int64_t row, char* buf, size_t buflen) {
    if (!r || !buf || row < 0 || row >= r->fetched) return fail(IMM3_ERR_INVALID_ARG, "imm3_result_format_row: bad arguments");
    std::string s = "Row(";
    const int c0 = r->agg_first_col >= 0 ? r->agg_first_col : 0;  // aggregate rows print the aggregators' repr only (ProjectAggregateQueue.scala:48-50)
    for (int c = c0; c < r->ncols; c++) {
        if (c > c0) s += ",";
        const uint8_t* p = (const uint8_t*)r->h_cols[(size_t)c].p + (size_t)row * (size_t)r->widths[(size_t)c];
        if (r->types[(size_t)c] == IMM3_COL_COUNT || r->types[(size_t)c] == IMM3_COL_INT64) {
            int64_t v;
            std::memcpy(&v, p, 8);
            s += std::to_string(v);  // Long.toString
        } else if (r->types[(size_t)c] == IMM3_COL_DOUBLE) {
            double v;
            std::memcpy(&v, p, 8);
            s += (r->avg_cols >> (c - c0)) & 1u ? java_double_to_string(v) : java_double_to_string_integral(v);
        } else if (r->types[(size_t)c] == IMM3_COL_INT) {
            int32_t v;
            std::memcpy(&v, p, 4);
            s += std::to_string(v);
        } else if (r->types[(size_t)c] == IMM3_COL_TINYINT) {
            s += std::to_string((int)(int8_t)p[0]);
        } else {
            s.append((const char*)p, (size_t)r->widths[(size_t)c]);
        }
    }
    s += ")";
    if (s.size() + 1 > buflen) return fail(IMM3_ERR_INVALID_ARG, "imm3_result_format_row: buffer too small (%zu needed)", s.size() + 1);
    std::memcpy(buf, s.c_str(), s.size() + 1);
    return (int)s.size();
}

int imm3_result_free(imm3_result* r) {
    if (!r) return 0;
    if (r->pending >= 0) cudaEventSynchronize(r->copied);  // never hand buffers back while a copy is reading them
    if (r->copied) cudaEventDestroy(r->copied);
    for (auto& b : r->d_cols) r->db->dev_pool.release(b);
    for (auto& b : r->h_cols) r->db->host_pool.release(b);
    r->db->live_results--;
    delete r;
    return 0;
}

int imm3_filter_bitmap(imm3_db* db, const char* table, const imm3_pred* preds, int npreds, const uint32_t** words,
                       int64_t* nwords, int64_t* nselected) {
    if (!db || !words || !nwords || !nselected) return fail(IMM3_ERR_INVALID_ARG, "imm3_filter_bitmap: NULL argument");
    Prepared pr;
    int rc = prepare(db, table, preds, npreds, nullptr, 0, 0, true, &pr);
    if (rc) return rc;
    if ((rc = use_device(db))) return rc;
    TableStore& t = *pr.table;
    const size_t need_words = (size_t)((t.nrows + kDenseMaxTileRows - 1) / kDenseMaxTileRows) * (kDenseMaxTileRows / 32) + 2;
    if ((rc = ensure_buf(&db->d_bitmap, need_words * 4))) return rc;
    if (db->h_bitmap.cap < need_words * 4) {
        if (db->h_bitmap.p) cudaFreeHost(db->h_bitmap.p);
        db->h_bitmap = Buf();
        CUDA_TRY(cudaMallocHost(&db->h_bitmap.p, need_words * 4));
        db->h_bitmap.cap = need_words * 4;
    }
    CUDA_TRY(cudaMemsetAsync(db->d_bitmap.p, 0, need_words * 4, db->stream));
    int64_t total = 0;
    if (!pr.lp.always_empty && t.nrows > 0) {
        if ((rc = fill_scan_plan(db, &pr))) return rc;
        pr.sp.bitmap = (uint32_t*)db->d_bitmap.p;
        pr.sp.limit = INT64_MAX;
        Run run;
        if ((rc = run_scan(db, pr, &run, &total))) return rc;
    }
    const size_t out_words = (size_t)((t.nrows + 31) / 32);
    if (out_words) CUDA_TRY(cudaMemcpyAsync(db->h_bitmap.p, db->d_bitmap.p, out_words * 4, cudaMemcpyDeviceToHost, db->stream));
    CUDA_TRY(cudaStreamSynchronize(db->stream));
    *words = (const uint32_t*)db->h_bitmap.p;
    *nwords = (int64_t)out_words;
    *nselected = total;
    return 0;
}

}  // extern "C"
