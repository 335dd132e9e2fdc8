// capi.cu -- the C ABI of libbydbgpu.so (include/bydb_gpu.h): context, HBM part cache, query
// orchestration on CUDA streams.  Host logic only; every byte of page decoding happens in
// scan_kernels.cu.  There is no CPU fallback here: unsupported encodings surface as BYDB_ENOTSUP.
#include <cuda_runtime.h>
#include <unistd.h>

#include <algorithm>
#include <cstdio>
#include <chrono>
#include <condition_variable>
#include <cstdlib>
#include <deque>
#include <functional>
#include <thread>
#include <future>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/bydb_gpu.h"
#include "part_dir.hpp"
#include "scan_kernels.cuh"
#include "index_kernels.cuh"

using namespace bydb;

namespace {

thread_local std::string g_last_error;
thread_local uint32_t g_last_dev_err = 0;  // DevErr of the last failed scan on this thread (drives the lazy unpack retry)
int fail(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}
// No exception may cross the C ABI ("never abort"): allocation failures and anything a hostile part provokes in the
// standard library become error codes.
template <class F>
int guarded(F &&f) {
    try {
        return f();
    } catch (const std::bad_alloc &) {
        return fail(BYDB_ENOMEM, "out of host memory");
    } catch (const std::exception &e) {
        return fail(BYDB_EINVAL, std::string("internal error: ") + e.what());
    } catch (...) {
        return fail(BYDB_EIO, "internal error: unknown exception");
    }
}
#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess)                                                                  \
            return fail(BYDB_EIO, std::string(#expr) + ": " + cudaGetErrorString(_e));          \
    } while (0)

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Part {
    uint64_t id = 0;
    PartDir dir;
    uint8_t *d_arena = nullptr;       // all file images, each 256 B aligned and padded
    uint8_t *d_dir = nullptr;         // DevBlock[] | DevCol[] | file pointer table
    uint8_t *d_unpack = nullptr;      // fallback pages rewritten at admission (unpack_kernels.cu); file slot `n_files`
    uint64_t unpacked_pages = 0, unpack_skipped = 0;
    const DevBlock *d_blocks = nullptr;
    const DevCol *d_cols = nullptr;
    const uint8_t *const *d_files = nullptr;
    uint64_t hbm_bytes = 0;
    int device = 0;
    cudaStream_t pool_stream = nullptr;  // transient parts (host path) live in the stream-ordered pool
    ~Part() {
        if (pool_stream) {
            if (d_arena) cudaFreeAsync(d_arena, pool_stream);
            if (d_dir) cudaFreeAsync(d_dir, pool_stream);
            if (d_unpack) cudaFreeAsync(d_unpack, pool_stream);
        } else {
            if (d_arena) cudaFree(d_arena);
            if (d_dir) cudaFree(d_dir);
            if (d_unpack) cudaFree(d_unpack);
        }
    }
};

// One in-flight call: stream, events and a pinned staging buffer.
struct ExecSlot {
    cudaStream_t stream = nullptr;
    static constexpr int kMaxBatches = 8;  // pipelined cold path: one set of events / zero page per batch
    cudaEvent_t ev[4 * kMaxBatches] = {};
    uint8_t *pinned = nullptr;
    size_t pinned_bytes = 0;
    uint8_t *zpage = nullptr;  // 256 B pinned: read-back of the per-query zero page (errors + counters)
    cudaEvent_t busy = nullptr;  // recorded by a call that returned before its work finished (asynchronous scan_partials)
    bool busy_pending = false;
    void wait_idle() {
        if (busy_pending) cudaEventSynchronize(busy);
        busy_pending = false;
    }
    // Page-locked allocations (and frees) are implicit synchronisation points of the device: no kernel issued after one starts
    // before every kernel issued before it has finished.  When several ranks share a device, a rank whose wait kernel is spinning
    // for a peer would then never see that peer's kernels start (the peer's call just allocated staging memory) -- a 60 s
    // stall ending in BYDB_EIO.  So: every slot is created with kInitialPinned bytes at bydb_init, grows geometrically and
    // rarely, and nothing is freed before bydb_shutdown.
    static constexpr size_t kInitialPinned = 1u << 20;
    std::vector<uint8_t *> retired;
    int ensure_pinned(size_t n) {
        if (n <= pinned_bytes) return 0;
        size_t want = align_up(std::max(n, 2 * pinned_bytes), 1 << 16);
        uint8_t *fresh = nullptr;
        if (cudaMallocHost(reinterpret_cast<void **>(&fresh), want) != cudaSuccess) {
            cudaGetLastError();
            want = align_up(n, 1 << 16);
            if (cudaMallocHost(reinterpret_cast<void **>(&fresh), want) != cudaSuccess) return -1;
        }
        if (pinned) retired.push_back(pinned);  // copies from it may still be in flight; freed at shutdown
        pinned = fresh;
        pinned_bytes = want;
        return 0;
    }
    int create() {
        if (cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking) != cudaSuccess) return -1;
        for (auto &e : ev)
            if (cudaEventCreate(&e) != cudaSuccess) return -1;
        if (cudaMallocHost(reinterpret_cast<void **>(&zpage), 256 * kMaxBatches) != cudaSuccess) return -1;
        if (cudaEventCreateWithFlags(&busy, cudaEventDisableTiming) != cudaSuccess) return -1;
        return ensure_pinned(kInitialPinned);
    }
};

}  // namespace

// A few persistent host threads for the cold path's block-index parsing: creating a dozen threads per query costs
// more (~0.5 ms, serialised on the calling thread) than parsing the first primary block.
class WorkPool {
  public:
    ~WorkPool() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto &t : th_) t.join();
    }
    void submit(std::function<void()> fn) {
        {
            std::lock_guard<std::mutex> lk(mu_);
            if (th_.empty()) {
                unsigned hw = std::thread::hardware_concurrency();
                const unsigned n = std::max(2u, std::min(32u, hw ? hw / 2 : 4u));  // index parsing + page gathering: memory-bound helpers
                for (unsigned i = 0; i < n; ++i) th_.emplace_back([this] { run(); });
            }
            q_.push_back(std::move(fn));
        }
        cv_.notify_one();
    }

  private:
    void run() {
        for (;;) {
            std::function<void()> fn;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [this] { return stop_ || !q_.empty(); });
                if (q_.empty()) return;  // stop_ and drained
                fn = std::move(q_.front());
                q_.pop_front();
            }
            fn();
        }
    }
    std::mutex mu_;
    std::condition_variable cv_;
    std::deque<std::function<void()>> q_;
    std::vector<std::thread> th_;
    bool stop_ = false;
};

// Peer mailboxes of the multi-GPU reduce (bydb_comm_*).  Layout of one rank's mailbox (device memory of that rank):
//   [0, 4096)        control: arrival flags (u64 epoch per writer rank) at 0, status words (epoch << 32 | host-side error of
//                    that rank's call) at 1024, `done` epoch at 2048, error word of this rank's wait kernels at 2056
//   [4096, ...)      2 parities x nranks slots of slot_bytes each (partial tables written by the peers)
constexpr int kCommMaxRanks = 64;
constexpr size_t kCommCtl = 4096, kCommStatusOff = 1024, kCommDoneOff = 2048, kCommErrOff = 2056, kCommArgsOff = 2112;
struct Comm {
    int rank = -1, nranks = 0;
    uint8_t *mine = nullptr;            // this rank's mailbox (cudaMalloc)
    size_t slot_bytes = 0, mailbox_bytes = 0;
    std::vector<uint8_t *> peer;        // device-visible base of every rank's mailbox
    std::vector<bool> ipc_opened;
    std::vector<size_t> peer_slot_bytes;
    uint64_t epoch = 0;
    std::vector<uint64_t> last_use;     // [root * 2 + parity] epoch of the previous collective that used that root's slots of that parity
    std::mutex mu;                      // collective calls are issued one at a time per context
    // A peer lives on THIS GPU (tests on a one-GPU box, more ranks than GPUs): no wait kernel may spin there.  CUDA gives no
    // forward-progress guarantee between streams of one device -- they share a handful of hardware queues, and work queued
    // behind the dependants of a spinning kernel in the same queue never launches, so a rank could wait forever for a peer
    // whose kernels sit behind its own wait kernel (seen as collectives that stalled until the 60 s bound, depending on how
    // many streams the process had created before).  In this mode the HOST polls the flags and the prepared form keeps the
    // plain path.  Ranks on different GPUs keep the device-side waits.
    bool shared_device = false;
    cudaStream_t poll_stream = nullptr;
    unsigned long long *poll_buf = nullptr;  // pinned, kCommMaxRanks words
};

// Pinned staging ring of the gather path (host images in PAGEABLE memory): the pages a query touches are collected into
// these buffers by the worker pool and go up with asynchronous copies, chunk k+1 being gathered while chunk k is on the bus.
struct StageRing {
    static constexpr int kBufs = 3;
    static constexpr size_t kBytes = 64u << 20;
    uint8_t *buf[kBufs] = {};
    cudaEvent_t done[kBufs] = {};
    bool pending[kBufs] = {};
    int next = 0;
    std::mutex mu;  // one gathering call at a time per context
};

struct bydb_ctx {
    int device = 0;
    int sm_count = 0;
    int ctas_per_sm = 2;       // slow lane (general decoder)
    int ctas_per_sm_fast = 2;  // fast lane
    uint64_t hbm_budget = 0;
    uint64_t hbm_used = 0;
    bool host_index = false;   // BYDB_CFG_HOST_INDEX: parse the block index of resident parts on the host (part_dir.cc)
    std::mutex mu;
    NameTable names;
    std::unordered_map<bydb_part_h, std::shared_ptr<Part>> parts;
    std::unordered_map<uint64_t, bydb_part_h> by_id;
    bydb_part_h next_handle = 1;
    std::vector<std::unique_ptr<ExecSlot>> free_slots;
    WorkPool pool;
    Comm comm;
    StageRing stage;
};

namespace {

struct SlotLease {
    bydb_ctx *ctx;
    std::unique_ptr<ExecSlot> slot;
    SlotLease(bydb_ctx *c) : ctx(c) {
        std::lock_guard<std::mutex> lk(c->mu);
        if (!c->free_slots.empty()) {
            slot = std::move(c->free_slots.back());
            c->free_slots.pop_back();
        }
    }
    int init() {
        if (slot) {
            slot->wait_idle();  // its pinned staging may still feed an asynchronous call's copies
            return 0;
        }
        slot.reset(new ExecSlot());   // more concurrent callers than slots made at bydb_init
        return slot->create();
    }
    ~SlotLease() {
        if (!slot) return;
        std::lock_guard<std::mutex> lk(ctx->mu);
        ctx->free_slots.push_back(std::move(slot));
    }
};

struct ResultOwner {
    std::vector<int32_t> group_id;
    std::vector<int64_t> rows;
    std::vector<uint8_t> is_float;
    std::vector<int64_t> val_i64;
    std::vector<double> val_f64;
};

// query after name resolution
struct Plan {
    std::vector<std::shared_ptr<Part>> parts;
    std::vector<std::string> fcols;       // distinct aggregated fields
    std::vector<int> agg_fcol;
    int32_t n_groups = 1;
    uint32_t total_blocks = 0;
    uint64_t n_series = 0;
};

const char *dev_err_text(uint32_t code) {
    switch (code) {
        case kErrPlainPage: return "numeric fallback page (EncodeTypePlain: null cells or non-decimal floats) is not decoded on the device yet";
        case kErrZstdDict: return "dictionary page with a zstd-compressed value block is not decoded on the device yet";
        case kErrBigBlock: return "row predicate on a block larger than the shared-memory row mask (8448 rows)";
        case kErrCorrupt: return "corrupt page: varint stream / header does not match the block's row count";
        case kErrTypeMix: return "a field is stored with different value types across blocks";
        case kErrBadEnc: return "unknown encode type byte";
        case kErrTagPlain: return "high-cardinality string tag page (plain bytes block) is not decoded on the device yet";
        case kErrOverlap: return "a series lives in several parts with overlapping time spans and the dedup pass did not run (internal error)";
        case kErrPredType: return "predicate literal type does not match the stored tag column type";
        case kErrTmaTimeout: return "internal error: a TMA bulk copy did not complete";
        case kErrPeerTimeout: return "multi-GPU reduce: a peer rank did not deliver its partial table in time";
        case kErrKeyCap: return "per-row group key: more distinct key values than bydb_group_key.max_values";
        case kErrKeyLong: return "per-row group key: a key value longer than 64 bytes";
    }
    return "unknown device error";
}
int dev_err_code(uint32_t code) { return code == kErrKeyCap ? BYDB_ENOMEM : (code == kErrCorrupt || code == kErrBadEnc || code == kErrTypeMix || code == kErrPredType) ? BYDB_EINVAL : (code == kErrTmaTimeout || code == kErrPeerTimeout) ? BYDB_EIO : BYDB_ENOTSUP; }

int validate_query(const bydb_query *q, bool need_parts) {
    if (!q) return fail(BYDB_EINVAL, "query is NULL");
    if (need_parts && (q->n_parts == 0 || !q->parts)) return fail(BYDB_EINVAL, "query has no parts");
    if (q->n_parts > kMaxParts) return fail(BYDB_EINVAL, "too many parts in one query (max 64)");
    if (q->n_series > 0 && !q->series_ids) return fail(BYDB_EINVAL, "series_ids is NULL");
    if (q->n_series > 0x7fffffffull) return fail(BYDB_EINVAL, "too many series");
    if (q->n_aggs == 0 || q->n_aggs > 32 || !q->aggs) return fail(BYDB_EINVAL, "need 1..32 aggregations");
    if (q->n_preds > kMaxPreds) return fail(BYDB_EINVAL, "too many predicates (max 8)");
    if (q->n_preds > 0 && !q->preds) return fail(BYDB_EINVAL, "preds is NULL");
    if (q->series_group && q->n_groups < 1) return fail(BYDB_EINVAL, "n_groups must be >= 1 when series_group is given");
    for (uint64_t i = 1; i < q->n_series; ++i)
        if (q->series_ids[i] <= q->series_ids[i - 1]) return fail(BYDB_EINVAL, "series_ids must be ascending and unique (query.go:601)");
    if (q->series_group)
        for (uint64_t i = 0; i < q->n_series; ++i)
            if (q->series_group[i] < 0 || q->series_group[i] >= q->n_groups) return fail(BYDB_EINVAL, "series_group out of range");
    for (uint32_t a = 0; a < q->n_aggs; ++a) {
        if (!q->aggs[a].field) return fail(BYDB_EINVAL, "aggregation without a field");
        if (q->aggs[a].func < BYDB_AGG_MEAN || q->aggs[a].func > BYDB_AGG_SUM) return fail(BYDB_EINVAL, "unknown aggregation function");
    }
    for (uint32_t i = 0; i < q->n_preds; ++i) {
        const bydb_pred &p = q->preds[i];
        if (!p.family || !p.tag) return fail(BYDB_EINVAL, "predicate without family/tag");
        if (p.op < BYDB_OP_EQ || p.op > BYDB_OP_GE) return fail(BYDB_EINVAL, "unknown predicate operator");
        if (p.value_type != BYDB_VT_INT64 && p.value_type != BYDB_VT_STR && p.value_type != BYDB_VT_BINARY)
            return fail(BYDB_EINVAL, "predicate literal must be int64, string or binary");
        if (p.value_type != BYDB_VT_INT64 && p.lit_len > kMaxLit) return fail(BYDB_ENOTSUP, "string predicate literal longer than 64 bytes");
        if (p.value_type != BYDB_VT_INT64 && p.lit_len > 0 && !p.lit) return fail(BYDB_EINVAL, "predicate literal is NULL");
    }
    if (q->top_n < 0 || (q->top_n > 0 && (q->top_agg < 0 || static_cast<uint32_t>(q->top_agg) >= q->n_aggs)))
        return fail(BYDB_EINVAL, "bad top_n / top_agg");
    // checked before anything is enqueued: a refusal after run_scan would leave work in flight on a pooled stream
    if (q->top_n > kMaxDeviceTopN) return fail(BYDB_ENOTSUP, "top_n larger than 2048 is not supported on the device path");
    return 0;
}

void distinct_fields(const bydb_query *q, std::vector<std::string> &fcols, std::vector<int> &agg_fcol) {
    for (uint32_t a = 0; a < q->n_aggs; ++a) {
        std::string f = q->aggs[a].field;
        int idx = -1;
        for (size_t i = 0; i < fcols.size(); ++i)
            if (fcols[i] == f) idx = static_cast<int>(i);
        if (idx < 0) {
            fcols.push_back(f);
            idx = static_cast<int>(fcols.size() - 1);
        }
        agg_fcol.push_back(idx);
    }
}

// partial-table layout for (G groups, F fields); see bydb_gpu.h
struct TableLayout {
    size_t G, F, GF;
    size_t off_sum_f64, off_max_f64, off_negmin_f64, off_sum_i64, off_cnt, off_rows, off_max_i64, off_notmin_i64, off_coltype, total;
    TableLayout(size_t g, size_t f) : G(g), F(f), GF(g * f) {
        size_t o = 0;
        off_sum_f64 = o; o += GF * 8;
        off_max_f64 = o; o += GF * 8;
        off_negmin_f64 = o; o += GF * 8;
        off_sum_i64 = o; o += GF * 8;
        off_cnt = o; o += GF * 8;
        off_rows = o; o += G * 8;
        off_max_i64 = o; o += GF * 8;
        off_notmin_i64 = o; o += GF * 8;
        off_coltype = o; o += F * 8;
        total = o;
    }
};

// zero_copy: the data files stay in (pinned, device-mapped) host memory and the kernels read the
// pages they need straight over PCIe; only the block directory is uploaded.
int unpack_fallback_pages(bydb_ctx *ctx, Part &part, size_t n_files, cudaStream_t s);
int build_part_dir_device(bydb_ctx *ctx, const std::vector<FileImage> &imgs, Part &part, const std::vector<std::string> &families, cudaStream_t s, size_t n_files,
                          size_t *dir_bytes_out);

int register_part_locked_free(bydb_ctx *ctx, uint64_t part_id, const bydb_part_files *files, std::shared_ptr<Part> &out, uint64_t *h2d,
                              bool zero_copy = false, bool transient = false, size_t batch = 0, size_t n_batches = 1, bool unpack = false,
                              PartDir *parsed = nullptr, bool device_index = false) {
    if (!files || files->n_files == 0 || !files->files) return fail(BYDB_EINVAL, "no files");
    std::vector<FileImage> imgs;
    for (uint32_t i = 0; i < files->n_files; ++i) {
        const bydb_file &f = files->files[i];
        if (!f.name || (!f.data && f.len)) return fail(BYDB_EINVAL, "file without name/data");
        imgs.push_back(FileImage{f.name, f.data, f.len});
    }
    auto part = std::make_shared<Part>();
    part->id = part_id;
    part->device = ctx->device;
    std::string err;
    // resident parts: the block index is inflated and parsed by kernels (index_kernels.cu); the host only decides the file table
    const bool dev_index = device_index && !parsed && n_batches == 1 && !zero_copy;
    std::vector<std::string> families;
    if (dev_index) {
        for (const auto &f : imgs)
            if (f.name.size() > 4 && f.name.compare(f.name.size() - 4, 4, ".tfm") == 0) families.push_back(f.name.substr(0, f.name.size() - 4));
        std::sort(families.begin(), families.end());
        if (families.size() > 250) return fail(BYDB_EINVAL, "too many tag family files");
        part->dir.files = {"timestamps.bin", "fv.bin"};
        for (const auto &fam : families) part->dir.files.push_back(fam + ".tf");
    } else if (parsed) {
        part->dir = std::move(*parsed);  // the caller parsed this slice of the block index already (cold path, in the background)
    } else {
        int rc = build_part_dir(imgs, ctx->names, part->dir, err, batch, n_batches);
        if (rc) return fail(rc, "part " + std::to_string(part_id) + ": " + err);
    }
    // arena: each data file 256 B aligned with >= 256 B of slack after it (TMA over-read, bit windows)
    std::vector<size_t> offs;
    size_t arena = 0;
    std::vector<const FileImage *> order;
    for (const auto &name : part->dir.files) {
        const FileImage *img = nullptr;
        for (const auto &f : imgs)
            if (f.name == name) img = &f;
        if (!img) return fail(BYDB_ENOENT, "missing file " + name);
        order.push_back(img);
        offs.push_back(arena);
        arena = align_up(arena + img->len + 256, 256);
    }
    std::vector<const uint8_t *> mapped(order.size(), nullptr);
    if (zero_copy) {
        for (size_t i = 0; i < order.size(); ++i) {
            if (order[i]->len == 0) continue;
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, order[i]->data) != cudaSuccess || at.type != cudaMemoryTypeHost || !at.devicePointer) {
                cudaGetLastError();
                return fail(BYDB_EINVAL, "BYDB_Q_HOST_ZERO_COPY needs file images in pinned, device-mapped host memory (" + order[i]->name + ")");
            }
            if (reinterpret_cast<uintptr_t>(at.devicePointer) & 15) return fail(BYDB_EINVAL, "zero-copy file images must be 16-byte aligned");
            mapped[i] = static_cast<const uint8_t *>(at.devicePointer);
        }
        arena = 0;
    }
    const size_t nb = part->dir.blocks.size(), nc = part->dir.cols.size(), nf = order.size();
    const size_t dir_bytes = dev_index ? 0 : align_up(nb * sizeof(DevBlock), 256) + align_up(nc * sizeof(DevCol), 256) + align_up((nf + 1) * sizeof(void *), 256);
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (ctx->hbm_budget && ctx->hbm_used + arena + dir_bytes > ctx->hbm_budget) return fail(BYDB_ENOMEM, "HBM budget exceeded");
        ctx->hbm_used += arena + dir_bytes;
    }
    part->hbm_bytes = arena + dir_bytes;
    auto undo_budget = [&]() {
        std::lock_guard<std::mutex> lk(ctx->mu);
        ctx->hbm_used -= part->hbm_bytes;
    };
    SlotLease lease(ctx);
    if (lease.init()) {
        undo_budget();
        return fail(BYDB_EIO, "cannot create stream");
    }
    cudaStream_t s = lease.slot->stream;
    bool alloc_ok;
    if (transient) {
        part->pool_stream = s;
        alloc_ok = cudaMallocAsync(reinterpret_cast<void **>(&part->d_arena), arena ? arena : 256, s) == cudaSuccess &&
                   (dev_index || cudaMallocAsync(reinterpret_cast<void **>(&part->d_dir), dir_bytes ? dir_bytes : 256, s) == cudaSuccess);
    } else {
        alloc_ok = cudaMalloc(reinterpret_cast<void **>(&part->d_arena), arena ? arena : 256) == cudaSuccess &&
                   (dev_index || cudaMalloc(reinterpret_cast<void **>(&part->d_dir), dir_bytes ? dir_bytes : 256) == cudaSuccess);
    }
    if (!alloc_ok) {
        undo_budget();
        return fail(BYDB_ENOMEM, "device allocation failed for part " + std::to_string(part_id));
    }
    cudaError_t e = cudaSuccess;
    if (!zero_copy) {
        e = cudaMemsetAsync(part->d_arena, 0, arena ? arena : 256, s);
        for (size_t i = 0; i < nf && e == cudaSuccess; ++i)
            if (order[i]->len) e = cudaMemcpyAsync(part->d_arena + offs[i], order[i]->data, order[i]->len, cudaMemcpyHostToDevice, s);
    }
    if (dev_index) {
        if (e != cudaSuccess) {
            undo_budget();
            return fail(BYDB_EIO, std::string("part upload: ") + cudaGetErrorString(e));
        }
        size_t dbytes = 0;
        int rc = build_part_dir_device(ctx, imgs, *part, families, s, nf, &dbytes);
        std::vector<const uint8_t *> table(nf + 1, nullptr);
        for (size_t i = 0; i < nf; ++i) table[i] = part->d_arena + offs[i];
        if (!rc && cudaMemcpyAsync(const_cast<uint8_t **>(reinterpret_cast<const uint8_t *const *>(part->d_files)), table.data(), nf * sizeof(void *),
                                   cudaMemcpyHostToDevice, s) != cudaSuccess)
            rc = fail(BYDB_EIO, "part upload: file table");
        if (!rc && cudaStreamSynchronize(s) != cudaSuccess) rc = fail(BYDB_EIO, "part upload: synchronize");
        if (rc) {
            cudaStreamSynchronize(s);
            undo_budget();
            return rc;
        }
        if (h2d) {
            for (size_t i = 0; i < nf; ++i) *h2d += order[i]->len;
            *h2d += dbytes;
        }
        if (unpack) {
            rc = unpack_fallback_pages(ctx, *part, nf, s);
            if (rc) {
                undo_budget();
                return rc;
            }
        }
        out = part;
        return 0;
    }
    // directory
    if (lease.slot->ensure_pinned(dir_bytes ? dir_bytes : 256)) {
        undo_budget();
        return fail(BYDB_ENOMEM, "cudaMallocHost failed");
    }
    uint8_t *hdir = lease.slot->pinned;  // the directory goes up from pinned staging in one copy
    if (nb) memcpy(hdir, part->dir.blocks.data(), nb * sizeof(DevBlock));
    const size_t off_cols = align_up(nb * sizeof(DevBlock), 256);
    if (nc) memcpy(hdir + off_cols, part->dir.cols.data(), nc * sizeof(DevCol));
    const size_t off_files = off_cols + align_up(nc * sizeof(DevCol), 256);
    for (size_t i = 0; i < nf; ++i) {
        const uint8_t *pfile = zero_copy ? mapped[i] : part->d_arena + offs[i];
        memcpy(hdir + off_files + i * sizeof(void *), &pfile, sizeof(void *));
    }
    if (e == cudaSuccess && dir_bytes) e = cudaMemcpyAsync(part->d_dir, hdir, dir_bytes, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) {
        undo_budget();
        return fail(BYDB_EIO, std::string("part upload: ") + cudaGetErrorString(e));
    }
    part->d_blocks = reinterpret_cast<const DevBlock *>(part->d_dir);
    part->d_cols = reinterpret_cast<const DevCol *>(part->d_dir + off_cols);
    part->d_files = reinterpret_cast<const uint8_t *const *>(part->d_dir + off_files);
    if (h2d) {
        if (!zero_copy)
            for (size_t i = 0; i < nf; ++i) *h2d += order[i]->len;
        *h2d += dir_bytes;
    }
    if (unpack) {
        const int rc = unpack_fallback_pages(ctx, *part, nf, s);
        if (rc) {
            undo_budget();
            return rc;
        }
    }
    out = part;
    return 0;
}


// ------------------------------------------------------------------------------------------------
// Block index on the device (index_kernels.cu): meta.bin / primary.bin / *.tfm go up as they are, the zstd frames are
// inflated and the blockMetadata records walked by kernels; the host only sizes the buffers between the phases and maps
// the handful of interned column names to the context's ids.  Fills part.dir (host copy of the directory) and writes
// DevBlock[] / DevCol[] straight into the part's device directory.
// ------------------------------------------------------------------------------------------------
struct DevTmp {
    uint8_t *p = nullptr;
    cudaStream_t s = nullptr;
    ~DevTmp() {
        if (p) cudaFreeAsync(p, s);
    }
    int alloc(size_t n, cudaStream_t st) {
        s = st;
        return cudaMallocAsync(reinterpret_cast<void **>(&p), n ? n : 256, st) == cudaSuccess ? 0 : -1;
    }
};

const char *index_err_text(uint32_t e) {
    switch (e) {
        case kIdxBadMeta: return "meta.bin: not a zstd frame of 40-byte primaryBlockMetadata records in order inside primary.bin";
        case kIdxBadFrame: return "primary block does not inflate to its declared size";
        case kIdxBadBlock: return "corrupt blockMetadata";
        case kIdxBadEnc: return "unexpected timestamps encode type";
        case kIdxBadColumn: return "corrupt columnMetadata";
        case kIdxFamily: return "tag family: missing or truncated .tf/.tfm";
        case kIdxOrder: return "blockMetadata out of order";
        case kIdxNames: return "too many / too long column names for the device index";
        case kIdxTooManyFamilies: return "more than 16 tag families in a block";
    }
    return "block index error";
}

// files: the part's file table (timestamps.bin, fv.bin, <family>.tf ...) is already decided by the caller; d_dir_* are
// allocated here once the counts are known.
int build_part_dir_device(bydb_ctx *ctx, const std::vector<FileImage> &imgs, Part &part, const std::vector<std::string> &families, cudaStream_t s,
                          size_t n_files, size_t *dir_bytes_out) {
    auto find = [&](const std::string &name) -> const FileImage * {
        for (const auto &f : imgs)
            if (f.name == name) return &f;
        return nullptr;
    };
    const FileImage *meta = find("meta.bin"), *primary = find("primary.bin"), *tsf = find("timestamps.bin"), *fvf = find("fv.bin");
    if (!meta || !primary || !tsf || !fvf) return fail(BYDB_ENOENT, "part needs meta.bin, primary.bin, timestamps.bin and fv.bin");
    // ---- the index files go up verbatim: [meta | primary | tfm ... | family names]
    std::vector<const FileImage *> tfm(families.size()), tf(families.size());
    size_t up = align_up(meta->len, 256) + align_up(primary->len, 256);
    const size_t off_primary = align_up(meta->len, 256);
    std::vector<size_t> off_tfm(families.size()), off_name(families.size());
    for (size_t i = 0; i < families.size(); ++i) {
        tfm[i] = find(families[i] + ".tfm");
        tf[i] = find(families[i] + ".tf");
        if (!tfm[i] || !tf[i]) return fail(BYDB_EINVAL, "tag family '" + families[i] + "': missing .tf/.tfm");
        off_tfm[i] = up;
        up += align_up(tfm[i]->len, 256);
    }
    for (size_t i = 0; i < families.size(); ++i) {
        off_name[i] = up;
        up += align_up(families[i].size(), 16);
    }
    const size_t off_fams = align_up(up, 256);
    up = off_fams + align_up(families.size() * sizeof(IndexFamily), 256);
    const size_t off_ctl = up;
    up += 256;
    const size_t off_names = up;
    up += kIndexMaxNames * sizeof(IndexName);
    const size_t off_map = up;
    up += align_up(kIndexMaxNames * sizeof(uint16_t), 256);
    DevTmp in;
    if (in.alloc(up, s)) return fail(BYDB_ENOMEM, "device allocation failed (index files)");
    CUDA_TRY(cudaMemsetAsync(in.p + off_ctl, 0, 256 + kIndexMaxNames * sizeof(IndexName), s));
    if (meta->len) CUDA_TRY(cudaMemcpyAsync(in.p, meta->data, meta->len, cudaMemcpyHostToDevice, s));
    if (primary->len) CUDA_TRY(cudaMemcpyAsync(in.p + off_primary, primary->data, primary->len, cudaMemcpyHostToDevice, s));
    std::vector<IndexFamily> fams(families.size());
    for (size_t i = 0; i < families.size(); ++i) {
        if (tfm[i]->len) CUDA_TRY(cudaMemcpyAsync(in.p + off_tfm[i], tfm[i]->data, tfm[i]->len, cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemcpyAsync(in.p + off_name[i], families[i].data(), families[i].size(), cudaMemcpyHostToDevice, s));
        memset(&fams[i], 0, sizeof fams[i]);
        fams[i].name = in.p + off_name[i];
        fams[i].name_len = static_cast<uint32_t>(families[i].size());
        fams[i].tfm = in.p + off_tfm[i];
        fams[i].tfm_len = tfm[i]->len;
        fams[i].tf_len = tf[i]->len;
        fams[i].file_id = static_cast<uint8_t>(2 + i);
    }
    if (!fams.empty()) CUDA_TRY(cudaMemcpyAsync(in.p + off_fams, fams.data(), fams.size() * sizeof(IndexFamily), cudaMemcpyHostToDevice, s));
    IndexCtl ctl0;
    memset(&ctl0, 0, sizeof ctl0);
    ctl0.min_ts = INT64_MAX;
    ctl0.max_ts = INT64_MIN;
    CUDA_TRY(cudaMemcpyAsync(in.p + off_ctl, &ctl0, sizeof ctl0, cudaMemcpyHostToDevice, s));
    IndexParams ip;
    memset(&ip, 0, sizeof ip);
    ip.meta = in.p;
    ip.primary = in.p + off_primary;
    ip.meta_len = meta->len;
    ip.primary_len = primary->len;
    ip.ts_len = tsf->len;
    ip.fv_len = fvf->len;
    ip.n_families = static_cast<uint32_t>(families.size());
    ip.families = reinterpret_cast<const IndexFamily *>(in.p + off_fams);
    ip.ctl = reinterpret_cast<IndexCtl *>(in.p + off_ctl);
    ip.names = reinterpret_cast<IndexName *>(in.p + off_names);
    ip.name_map = reinterpret_cast<const uint16_t *>(in.p + off_map);
    IndexCtl ctl;
    auto read_ctl = [&]() -> int {
        CUDA_TRY(cudaMemcpyAsync(&ctl, in.p + off_ctl, sizeof ctl, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        if (ctl.err) return fail(BYDB_EINVAL, "part " + std::to_string(part.id) + ": " + index_err_text(ctl.err) + " (#" + std::to_string(ctl.err_where) + ")");
        return 0;
    };
    // ---- meta.bin: size, then inflate + the primary frames' sizes
    DevTmp scratch0;
    if (scratch0.alloc(index_scratch_stride(), s)) return fail(BYDB_ENOMEM, "device allocation failed (index scratch)");
    ip.scratch = scratch0.p;
    launch_index_meta(ip, 0, s);
    int rc = read_ctl();
    if (rc) return rc;
    const size_t n_primary = static_cast<size_t>(ctl.meta_raw / 40);
    DevTmp meta_raw, pbs;
    if (meta_raw.alloc(ctl.meta_raw, s) || pbs.alloc(n_primary * sizeof(IndexPrimary), s)) return fail(BYDB_ENOMEM, "device allocation failed (index)");
    CUDA_TRY(cudaMemsetAsync(pbs.p, 0, n_primary ? n_primary * sizeof(IndexPrimary) : 256, s));
    ip.meta_raw = meta_raw.p;
    ip.meta_raw_cap = ctl.meta_raw;
    ip.pb = reinterpret_cast<IndexPrimary *>(pbs.p);
    launch_index_meta(ip, 1, s);
    rc = read_ctl();
    if (rc) return rc;
    // ---- primary blocks: inflate, count
    ip.n_primary = static_cast<uint32_t>(n_primary);
    DevTmp raw, scratch;
    if (raw.alloc(ctl.raw_total + 256, s) || scratch.alloc(std::max<size_t>(1, n_primary) * index_scratch_stride(), s))
        return fail(BYDB_ENOMEM, "device allocation failed (inflated index)");
    ip.raw = raw.p;
    ip.scratch = scratch.p;
    launch_index_inflate(ip, s);
    launch_index_walk(ip, false, s);
    std::vector<IndexPrimary> hpb(n_primary);
    std::vector<IndexName> hnames(kIndexMaxNames);
    if (n_primary) CUDA_TRY(cudaMemcpyAsync(hpb.data(), pbs.p, n_primary * sizeof(IndexPrimary), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(hnames.data(), in.p + off_names, kIndexMaxNames * sizeof(IndexName), cudaMemcpyDeviceToHost, s));
    rc = read_ctl();
    if (rc) return rc;
    uint64_t nb = 0, nc = 0;
    for (auto &e : hpb) {
        e.block_base = nb;
        e.col_base = nc;
        nb += e.n_blocks;
        nc += e.n_cols;
    }
    if (nb > 0x7fffffffull || nc > 0xffffffffull) return fail(BYDB_EINVAL, "too many blocks / columns");
    // ---- the interned names -> the context's ids (a few dozen short strings: the only index bytes the host looks at)
    std::vector<uint16_t> map(kIndexMaxNames, 0);
    for (uint32_t i = 0; i < ctl.n_names && i < kIndexMaxNames; ++i) {
        const IndexName &e = hnames[i];
        std::string key = e.kind == 'f' ? "f:" : "t:" + families[e.fam] + "/";
        key.append(reinterpret_cast<const char *>(e.bytes), e.len);
        map[i] = ctx->names.intern(key);
    }
    if (n_primary) CUDA_TRY(cudaMemcpyAsync(pbs.p, hpb.data(), n_primary * sizeof(IndexPrimary), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(in.p + off_map, map.data(), kIndexMaxNames * sizeof(uint16_t), cudaMemcpyHostToDevice, s));
    // ---- the part's device directory, filled by the second walk
    const size_t off_cols = align_up(nb * sizeof(DevBlock), 256);
    const size_t off_files = off_cols + align_up(nc * sizeof(DevCol), 256);
    const size_t dir_bytes = off_files + align_up((n_files + 1) * sizeof(void *), 256);
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (ctx->hbm_budget && ctx->hbm_used + dir_bytes > ctx->hbm_budget) return fail(BYDB_ENOMEM, "HBM budget exceeded");
        ctx->hbm_used += dir_bytes;
    }
    part.hbm_bytes += dir_bytes;
    *dir_bytes_out = dir_bytes;
    const cudaError_t ae = part.pool_stream ? cudaMallocAsync(reinterpret_cast<void **>(&part.d_dir), dir_bytes, s) : cudaMalloc(reinterpret_cast<void **>(&part.d_dir), dir_bytes);
    if (ae != cudaSuccess) {
        part.d_dir = nullptr;
        return fail(BYDB_ENOMEM, "device allocation failed for the directory of part " + std::to_string(part.id));
    }
    ip.blocks = reinterpret_cast<DevBlock *>(part.d_dir);
    ip.cols = reinterpret_cast<DevCol *>(part.d_dir + off_cols);
    ip.n_blocks = nb;
    launch_index_walk(ip, true, s);
    launch_index_order(ip, s);
    part.dir.blocks.resize(nb);
    part.dir.cols.resize(nc);
    if (nb) CUDA_TRY(cudaMemcpyAsync(part.dir.blocks.data(), ip.blocks, nb * sizeof(DevBlock), cudaMemcpyDeviceToHost, s));
    if (nc) CUDA_TRY(cudaMemcpyAsync(part.dir.cols.data(), ip.cols, nc * sizeof(DevCol), cudaMemcpyDeviceToHost, s));
    rc = read_ctl();
    if (rc) return rc;
    part.dir.total_rows = ctl.total_rows;
    part.dir.max_block_rows = ctl.max_block_rows;
    part.dir.min_ts = nb ? ctl.min_ts : 0;
    part.dir.max_ts = nb ? ctl.max_ts : 0;
    part.d_blocks = ip.blocks;
    part.d_cols = ip.cols;
    part.d_files = reinterpret_cast<const uint8_t *const *>(part.d_dir + off_files);
    return 0;
}

// Rewrites the part's fallback pages (EncodeTypePlain numeric pages, zstd-compressed string blocks) into a side
// arena in HBM so the scan kernels never meet zstd or per-cell byte strings; see unpack_kernels.cu.
int unpack_fallback_pages(bydb_ctx *ctx, Part &part, size_t n_files, cudaStream_t s) {
    const size_t nb = part.dir.blocks.size(), nc = part.dir.cols.size();
    if (nb == 0 || nc == 0) return 0;
    if (n_files >= 255) return 0;
    struct Tmp {
        uint8_t *p = nullptr;
        cudaStream_t s = nullptr;
        ~Tmp() {
            if (p) cudaFreeAsync(p, s);
        }
    } jobs, scratch;
    jobs.s = scratch.s = s;
    const size_t jobs_off = 256;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&jobs.p), jobs_off + nc * sizeof(UnpackJob), s));
    CUDA_TRY(cudaMemsetAsync(jobs.p, 0, jobs_off, s));
    UnpackParams up{};
    up.blocks = part.d_blocks;
    up.cols = const_cast<DevCol *>(part.d_cols);
    up.files = part.d_files;
    up.n_blocks = static_cast<uint32_t>(nb);
    up.arena_file_id = static_cast<uint32_t>(n_files);
    up.counters = reinterpret_cast<unsigned long long *>(jobs.p);
    up.jobs = reinterpret_cast<UnpackJob *>(jobs.p + jobs_off);
    up.max_jobs = nc;
    launch_classify_pages(up, s);
    unsigned long long cnt[5] = {0, 0, 0, 0, 0};
    CUDA_TRY(cudaMemcpyAsync(cnt, jobs.p, sizeof cnt, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    part.unpack_skipped = cnt[3];
    if (cnt[0] == 0) return 0;
    const size_t arena = align_up(cnt[1] + 256, 256);
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (ctx->hbm_budget && ctx->hbm_used + arena > ctx->hbm_budget) return fail(BYDB_ENOMEM, "HBM budget exceeded while unpacking fallback pages");
        ctx->hbm_used += arena;
    }
    part.hbm_bytes += arena;
    cudaError_t e = part.pool_stream ? cudaMallocAsync(reinterpret_cast<void **>(&part.d_unpack), arena, s)
                                     : cudaMalloc(reinterpret_cast<void **>(&part.d_unpack), arena);
    if (e != cudaSuccess) return fail(BYDB_ENOMEM, "device allocation failed for the unpack arena");
    const int n_warps = static_cast<int>(std::min<unsigned long long>(cnt[0], 8ull * static_cast<unsigned long long>(ctx->sm_count)));
    const int n_warps4 = (n_warps + 3) / 4 * 4;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&scratch.p), static_cast<size_t>(n_warps4) * unpack_scratch_stride(), s));
    // publish the arena as one more file of the part
    const uint8_t *ap = part.d_unpack;
    CUDA_TRY(cudaMemcpyAsync(const_cast<uint8_t **>(reinterpret_cast<const uint8_t *const *>(part.d_files)) + n_files, &ap, sizeof ap,
                             cudaMemcpyHostToDevice, s));
    up.n_jobs = cnt[0];
    up.arena = part.d_unpack;
    up.scratch = scratch.p;
    launch_unpack_pages(up, n_warps4, s);
    CUDA_TRY(cudaMemcpyAsync(cnt, jobs.p, sizeof cnt, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    part.unpacked_pages = cnt[4];
    part.unpack_skipped = cnt[3];
    return 0;
}

struct Scratch {
    uint8_t *base = nullptr;
    size_t bytes = 0;
    cudaStream_t stream = nullptr;
    ~Scratch() {
        if (base) cudaFreeAsync(base, stream);
    }
};

// Runs plan -> scan -> series_reduce -> group_reduce on `stream`, leaving the partial table at
// `d_table` (device).  Synchronises the stream.  Fills stats.
// one pass of a group-key query (bydb_scan_agg_keyed): where in the composite table the pass writes, and its side outputs
struct KeyedPass {
    size_t group_off;   // first group row of this pass's slice
    int64_t *coltype;   // [F] the pass's own column types + status (merged by permute_table)
    int64_t *kts;       // [n_series] see ReduceParams::Kts
    uint32_t *krow;     // [n_series]
};

int run_scan(bydb_ctx *ctx, const bydb_query *q, Plan &plan, ExecSlot &slot, cudaStream_t stream, uint8_t *d_table, const TableLayout &tl,
             bydb_stats *stats, int batch = 0, bool presized = false, const KeyedPass *kp = nullptr) {
    cudaEvent_t *ev = slot.ev + 4 * batch;
    uint8_t *zpage = slot.zpage + 256 * batch;
    memset(zpage, 0, 256);  // a failure before the read-back is enqueued must not leave a previous call's status behind
    const size_t F = plan.fcols.size();
    const size_t NS = q->n_series;
    const size_t NB = plan.total_blocks;
    const int32_t G = plan.n_groups;
    // ---- host staging: sids | order | group_start
    std::vector<int32_t> order(NS), gstart(static_cast<size_t>(G) + 1, 0);
    if (q->series_group) {
        for (size_t i = 0; i < NS; ++i) gstart[static_cast<size_t>(q->series_group[i]) + 1]++;
        for (int32_t g = 0; g < G; ++g) gstart[g + 1] += gstart[g];
        std::vector<int32_t> cur(gstart.begin(), gstart.end() - 1);
        for (size_t i = 0; i < NS; ++i) order[cur[q->series_group[i]]++] = static_cast<int32_t>(i);
    } else {
        for (size_t i = 0; i < NS; ++i) order[i] = static_cast<int32_t>(i);
        gstart[1] = static_cast<int32_t>(NS);
    }
    // ---- device scratch layout
    size_t o = 0;
    auto carve = [&](size_t bytes) {
        size_t at = o;
        o = align_up(o + bytes, 256);
        return at;
    };
    const size_t off_zero = carve(256);  // work_count, work_next, err[2], stats[4], col_type[F]
    // sids | order | group_start sit back to back, exactly like in the pinned staging: one copy brings all three
    const size_t off_sids = carve(NS * 12 + (static_cast<size_t>(G) + 1) * 4);
    const size_t off_order = off_sids + NS * 8;
    const size_t off_gstart = off_sids + NS * 12;
    const size_t off_worklist = carve(NB * 4);
    const size_t off_slowlist = carve(NB * 4);
    const size_t off_restlist = carve(NB * 4);
    const size_t off_qsid = carve(NB * 4);
    const size_t off_P = carve(NB * F * sizeof(BlockPartial));
    const size_t off_Prows = carve(NB * 4);
    const size_t off_Pfirst = carve(kp ? NB * 4 : 0);
    const size_t off_S = carve(NS * F * sizeof(BlockPartial));
    const size_t off_Srows = carve(NS * 8);
    const size_t n_first = NS * plan.parts.size();
    const bool use_first = n_first > 0 && n_first <= (16u << 20);
    const size_t off_first = carve(use_first ? n_first * 4 : 0);
    const size_t off_dd_index = carve(NB * 4), off_dd_rowoff = carve(NB * 8), off_dd_list = carve(NB * 4);
    Scratch sc;
    sc.stream = stream;
    sc.bytes = o;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&sc.base), o, stream));
    uint8_t *d = sc.base;
    const size_t stage_bytes = NS * 8 + NS * 4 + (static_cast<size_t>(G) + 1) * 4;
    const size_t stage_stride = align_up(stage_bytes + 256, 256);
    if (!presized && slot.ensure_pinned(stage_stride * static_cast<size_t>(batch + 1))) return fail(BYDB_ENOMEM, "cudaMallocHost failed");
    uint8_t *h = slot.pinned + stage_stride * static_cast<size_t>(batch);
    if (NS) memcpy(h, q->series_ids, NS * 8);
    if (NS) memcpy(h + NS * 8, order.data(), NS * 4);
    memcpy(h + NS * 12, gstart.data(), (static_cast<size_t>(G) + 1) * 4);
    CUDA_TRY(cudaMemsetAsync(d + off_zero, 0, 256, stream));
    if (use_first) CUDA_TRY(cudaMemsetAsync(d + off_first, 0xff, n_first * 4, stream));
    CUDA_TRY(cudaMemcpyAsync(d + off_sids, h, stage_bytes, cudaMemcpyHostToDevice, stream));
    if (stats) stats->h2d_bytes += stage_bytes;

    // zero page: [0] work_count [1] work_next [2..3] err [4..11] stats (u64 x4) [16..] col_type
    uint32_t *z32 = reinterpret_cast<uint32_t *>(d + off_zero);
    ScanParams sp;
    memset(&sp, 0, sizeof sp);
    ReduceParams rp;
    memset(&rp, 0, sizeof rp);
    uint32_t base = 0;
    for (size_t i = 0; i < plan.parts.size(); ++i) {
        DevPartRef r;
        r.blocks = plan.parts[i]->d_blocks;
        r.cols = plan.parts[i]->d_cols;
        r.files = plan.parts[i]->d_files;
        r.n_blocks = static_cast<uint32_t>(plan.parts[i]->dir.blocks.size());
        r.block_base = base;
        base += r.n_blocks;
        sp.parts[i] = r;
        rp.parts[i] = r;
    }
    sp.n_parts = rp.n_parts = static_cast<uint32_t>(plan.parts.size());
    sp.total_blocks = static_cast<uint32_t>(NB);
    sp.q_sids = reinterpret_cast<const uint64_t *>(d + off_sids);
    sp.n_series = static_cast<uint32_t>(NS);
    sp.n_fcols = static_cast<uint32_t>(F);
    sp.n_preds = q->n_preds;
    sp.tmin = q->tmin;
    sp.tmax = q->tmax;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        for (size_t c = 0; c < F; ++c) sp.fcol_name[c] = ctx->names.find("f:" + plan.fcols[c]);
        for (uint32_t a = 0; a < q->n_aggs; ++a) {
            const int fn = q->aggs[a].func;
            uint8_t need = (fn == BYDB_AGG_SUM || fn == BYDB_AGG_MEAN) ? 1 : (fn == BYDB_AGG_MIN || fn == BYDB_AGG_MAX) ? 2 : 0;
            sp.fcol_need[plan.agg_fcol[a]] |= need;
        }
        for (uint32_t i = 0; i < q->n_preds; ++i) {
            const bydb_pred &p = q->preds[i];
            DevPred &dp = sp.preds[i];
            dp.name_id = ctx->names.find(std::string("t:") + p.family + "/" + p.tag);
            dp.op = static_cast<uint8_t>(p.op);
            dp.value_type = static_cast<uint8_t>(p.value_type == BYDB_VT_BINARY ? BYDB_VT_STR : p.value_type);
            dp.lit_i64 = p.lit_i64;
            dp.lit_len = p.value_type == BYDB_VT_INT64 ? 0 : static_cast<uint32_t>(p.lit_len);
            if (dp.lit_len) memcpy(dp.lit, p.lit, dp.lit_len);
        }
    }
    sp.worklist = reinterpret_cast<uint32_t *>(d + off_worklist);
    sp.work_count = z32 + 0;
    sp.work_next = z32 + 1;
    sp.slow_list = reinterpret_cast<uint32_t *>(d + off_slowlist);
    sp.slow_count = z32 + 28;  // bytes 112..119 of the zero page
    sp.slow_next = z32 + 29;
    sp.err = z32 + 2;
    sp.stats = reinterpret_cast<unsigned long long *>(d + off_zero + 16);
    sp.col_type = reinterpret_cast<int32_t *>(d + off_zero + 64);
    sp.block_qsid = reinterpret_cast<int32_t *>(d + off_qsid);
    sp.first_block = use_first ? reinterpret_cast<uint32_t *>(d + off_first) : nullptr;
    sp.P = reinterpret_cast<BlockPartial *>(d + off_P);
    sp.Prows = reinterpret_cast<uint32_t *>(d + off_Prows);
    sp.Pfirst = kp ? reinterpret_cast<uint32_t *>(d + off_Pfirst) : nullptr;

    rp.n_series = static_cast<uint32_t>(NS);
    rp.n_fcols = static_cast<uint32_t>(F);
    rp.n_groups = G;
    rp.q_sids = sp.q_sids;
    rp.order = reinterpret_cast<const int32_t *>(d + off_order);
    rp.group_start = reinterpret_cast<const int32_t *>(d + off_gstart);
    rp.block_qsid = sp.block_qsid;
    rp.first_block = sp.first_block;
    rp.P = sp.P;
    rp.Prows = sp.Prows;
    rp.col_type = sp.col_type;
    rp.S = reinterpret_cast<BlockPartial *>(d + off_S);
    rp.Srows = reinterpret_cast<int64_t *>(d + off_Srows);
    rp.err = sp.err;
    rp.sum_f64 = reinterpret_cast<double *>(d_table + tl.off_sum_f64);
    rp.max_f64 = reinterpret_cast<double *>(d_table + tl.off_max_f64);
    rp.negmin_f64 = reinterpret_cast<double *>(d_table + tl.off_negmin_f64);
    rp.sum_i64 = reinterpret_cast<int64_t *>(d_table + tl.off_sum_i64);
    rp.cnt = reinterpret_cast<int64_t *>(d_table + tl.off_cnt);
    rp.rows = reinterpret_cast<int64_t *>(d_table + tl.off_rows);
    rp.max_i64 = reinterpret_cast<int64_t *>(d_table + tl.off_max_i64);
    rp.notmin_i64 = reinterpret_cast<int64_t *>(d_table + tl.off_notmin_i64);
    rp.coltype = reinterpret_cast<int64_t *>(d_table + tl.off_coltype);
    if (kp) {
        const size_t go = kp->group_off, gf = kp->group_off * F;
        rp.sum_f64 += gf, rp.max_f64 += gf, rp.negmin_f64 += gf;
        rp.sum_i64 += gf, rp.cnt += gf, rp.max_i64 += gf, rp.notmin_i64 += gf;
        rp.rows += go;
        rp.coltype = kp->coltype;
        rp.Pfirst = sp.Pfirst;
        rp.Kts = kp->kts;
        rp.Krow = kp->krow;
    }

    CUDA_TRY(cudaEventRecord(ev[0], stream));
    launch_plan_blocks(sp, stream);
    // ---- version dedup: only when two parts of the query overlap in time at all (host-side precheck on
    //      the part directories); then the device finds the series that really overlap
    Scratch dd_scratch;
    dd_scratch.stream = stream;
    uint32_t extra_launches = 0;
    bool parts_overlap = false;
    for (size_t a = 0; a < plan.parts.size() && !parts_overlap; ++a)
        for (size_t b = a + 1; b < plan.parts.size() && !parts_overlap; ++b) {
            const PartDir &x = plan.parts[a]->dir, &y = plan.parts[b]->dir;
            if (x.blocks.empty() || y.blocks.empty()) continue;
            const int64_t lo = std::max(std::max(x.min_ts, y.min_ts), q->tmin), hi = std::min(std::min(x.max_ts, y.max_ts), q->tmax);
            parts_overlap = lo <= hi;
        }
    if (parts_overlap && NB > 0 && NS > 0) {
        sp.dd_index = reinterpret_cast<int32_t *>(d + off_dd_index);
        sp.dd_row_off = reinterpret_cast<unsigned long long *>(d + off_dd_rowoff);
        sp.dd_list = reinterpret_cast<uint32_t *>(d + off_dd_list);
        sp.dd_counts = reinterpret_cast<unsigned long long *>(d + off_zero + 96);
        CUDA_TRY(cudaMemsetAsync(sp.dd_index, 0xff, NB * 4, stream));
        launch_detect_overlap(sp, stream);
        CUDA_TRY(cudaMemcpyAsync(zpage + 128, d + off_zero + 96, 16, cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
        const unsigned long long n_ddb = reinterpret_cast<unsigned long long *>(zpage + 128)[0];
        const unsigned long long n_ddr = reinterpret_cast<unsigned long long *>(zpage + 128)[1];
        extra_launches += 1;
        if (stats) stats->d2h_bytes += 16;
        if (n_ddb > 0) {
            const size_t b_ts = align_up(n_ddr * 8, 256), b_sh = align_up(n_ddb * kMaskWords * 4, 256);
            CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&dd_scratch.base), 2 * b_ts + b_sh, stream));
            sp.dd_ts = reinterpret_cast<int64_t *>(dd_scratch.base);
            sp.dd_ver = reinterpret_cast<int64_t *>(dd_scratch.base + b_ts);
            sp.dd_shadow = reinterpret_cast<uint32_t *>(dd_scratch.base + 2 * b_ts);
            sp.n_dd_blocks = static_cast<uint32_t>(n_ddb);
            launch_dedup(sp, ctx->sm_count * ctx->ctas_per_sm, stream);
            extra_launches += 2;
        }
        rp.dedup_done = 1;
    }
    {
        // express lane (scan_sum_express_kernel): all-rows SUM / MEAN / COUNT without row predicates or version dedup -- the
        // group-by-sum shape; every block it cannot take (time-range cut, non-delta page, ...) goes on to the regular lane
        bool sums_only = q->n_preds == 0 && !parts_overlap && NB > 0;
        for (size_t c = 0; c < F; ++c) sums_only = sums_only && (sp.fcol_need[c] & 2) == 0;
        static const bool no_express = getenv("BYDB_NO_EXPRESS") != nullptr;  // A/B timing of the two lanes
        if (sums_only && !no_express) {
            sp.rest_list = reinterpret_cast<uint32_t *>(d + off_restlist);
            sp.rest_count = z32 + 30;  // bytes 120..127 of the zero page
            sp.rest_next = z32 + 31;
            if (stats) stats->kernel_launches += 1;
        }
    }
    CUDA_TRY(cudaEventRecord(ev[1], stream));
    launch_scan_blocks(sp, ctx->sm_count * ctx->ctas_per_sm_fast, ctx->sm_count * ctx->ctas_per_sm, stream);
    CUDA_TRY(cudaEventRecord(ev[2], stream));
    launch_series_reduce(rp, stream);
    bool small_groups = true;  // every group has at most 32 series: the warp-per-group reduce (bit-identical sums)
    for (int32_t g = 0; g < G && small_groups; ++g) small_groups = gstart[g + 1] - gstart[g] <= 32;
    launch_group_reduce(rp, stream, small_groups);
    CUDA_TRY(cudaEventRecord(ev[3], stream));
    // read back the zero page (errors + counters); the caller synchronises and then calls collect_scan
    CUDA_TRY(cudaMemcpyAsync(zpage, d + off_zero, 256, cudaMemcpyDeviceToHost, stream));
    if (stats) {
        stats->kernel_launches += (NB ? 1u : 0u) + 2u + (NS ? 1u : 0u) + 1u + extra_launches;
        stats->d2h_bytes += 256;
    }
    // the scratch must outlive the kernels: it is freed stream-ordered (after them) when `sc` goes out of scope
    return 0;
}

// after the stream is synchronised: device errors + counters of the scan
int collect_scan(ExecSlot &slot, bydb_stats *stats, int batch = 0) {
    cudaEvent_t *ev = slot.ev + 4 * batch;
    const uint32_t *hz = reinterpret_cast<const uint32_t *>(slot.zpage + 256 * batch);
    if (stats) {
        const unsigned long long *hs = reinterpret_cast<const unsigned long long *>(slot.zpage + 256 * batch + 16);
        stats->rows_scanned += hs[0];
        stats->rows_matched += hs[1];
        stats->page_bytes += hs[2];
        stats->blocks_scanned += hs[3];
        stats->blocks_slow_lane += static_cast<uint32_t>(hs[4]);
        stats->slow_lane_reasons |= static_cast<uint32_t>(hs[5]);
        float ms = 0;
        cudaEventElapsedTime(&ms, ev[1], ev[2]);
        stats->scan_kernel_ms += ms;
        cudaEventElapsedTime(&ms, ev[0], ev[3]);
        stats->device_ms += ms;
    }
    if (hz[2] != 0) g_last_dev_err = hz[2];  // reset by the API entry points; a later clean slice must not hide it
    if (hz[2] != 0) {
        char buf[96];
        snprintf(buf, sizeof buf, " (block/series #%u)", hz[3]);
        return fail(dev_err_code(hz[2]), std::string(dev_err_text(hz[2])) + buf);
    }
    return 0;
}

struct FinalLayout {
    size_t o_out = 0, o_cnt = 0, o_isf = 0, o_sg = 0, o_sr = 0, o_si = 0, o_sf = 0, out_bytes = 0, cap = 0, A = 0;
    uint32_t launches = 0;
};

// finalize_to_host up to (and including) the read-back copy, without the synchronisation and the parsing; the result
// lands at slot.pinned + host_off so that the staging area of run_scan (at the start of slot.pinned) stays intact
int finalize_enqueue(const bydb_query *q, const Plan &plan, ExecSlot &slot, cudaStream_t stream, const uint8_t *d_table, const TableLayout &tl,
                     size_t host_off, FinalLayout &fl, Scratch &sc) {
    const size_t F = plan.fcols.size();
    const int32_t G = plan.n_groups;
    const size_t A = q->n_aggs;
    const size_t cap = q->top_n > 0 ? std::min<size_t>(static_cast<size_t>(q->top_n), static_cast<size_t>(G)) : static_cast<size_t>(G);
    size_t o = 0;
    auto carve = [&](size_t bytes) {
        size_t at = o;
        o = align_up(o + bytes, 256);
        return at;
    };
    const size_t o_vi = carve(static_cast<size_t>(G) * A * 8), o_vf = carve(static_cast<size_t>(G) * A * 8), o_keys = carve(static_cast<size_t>(G) * 8),
                 o_kst = carve(static_cast<size_t>(G));
    fl.o_out = o;
    fl.o_cnt = carve(16);
    fl.o_isf = carve(A);
    fl.o_sg = carve(cap * 4);
    fl.o_sr = carve(cap * 8);
    fl.o_si = carve(cap * A * 8);
    fl.o_sf = carve(cap * A * 8);
    fl.out_bytes = o - fl.o_out;
    fl.cap = cap;
    fl.A = A;
    sc.stream = stream;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&sc.base), o, stream));
    uint8_t *d = sc.base;
    FinalizeParams fp;
    memset(&fp, 0, sizeof fp);
    fp.n_groups = G;
    fp.n_fcols = static_cast<uint32_t>(F);
    fp.n_aggs = static_cast<uint32_t>(A);
    fp.row_path_types = (q->flags & BYDB_Q_ROW_PATH_TYPES) ? 1u : 0u;
    for (size_t a = 0; a < A; ++a) {
        fp.agg_fcol[a] = plan.agg_fcol[a];
        fp.agg_func[a] = q->aggs[a].func;
    }
    fp.sum_f64 = reinterpret_cast<const double *>(d_table + tl.off_sum_f64);
    fp.max_f64 = reinterpret_cast<const double *>(d_table + tl.off_max_f64);
    fp.negmin_f64 = reinterpret_cast<const double *>(d_table + tl.off_negmin_f64);
    fp.sum_i64 = reinterpret_cast<const int64_t *>(d_table + tl.off_sum_i64);
    fp.cnt = reinterpret_cast<const int64_t *>(d_table + tl.off_cnt);
    fp.rows = reinterpret_cast<const int64_t *>(d_table + tl.off_rows);
    fp.max_i64 = reinterpret_cast<const int64_t *>(d_table + tl.off_max_i64);
    fp.notmin_i64 = reinterpret_cast<const int64_t *>(d_table + tl.off_notmin_i64);
    fp.coltype = reinterpret_cast<const int64_t *>(d_table + tl.off_coltype);
    fp.out_i64 = reinterpret_cast<int64_t *>(d + o_vi);
    fp.out_f64 = reinterpret_cast<double *>(d + o_vf);
    fp.out_is_float = d + fl.o_isf;
    fp.err_out = reinterpret_cast<uint32_t *>(d + fl.o_cnt + 8);
    SelectParams sp;
    memset(&sp, 0, sizeof sp);
    sp.n_groups = G;
    sp.n_fcols = static_cast<uint32_t>(F);
    sp.n_aggs = static_cast<uint32_t>(A);
    sp.top_n = q->top_n;
    sp.top_agg = q->top_n > 0 ? q->top_agg : 0;
    sp.top_desc = q->top_desc;
    sp.top_fcol = plan.agg_fcol[sp.top_agg];
    sp.top_is_count = q->aggs[sp.top_agg].func == BYDB_AGG_COUNT;
    sp.rows = fp.rows;
    sp.cnt = fp.cnt;
    sp.val_i64 = fp.out_i64;
    sp.val_f64 = fp.out_f64;
    sp.is_float = fp.out_is_float;
    sp.keys = reinterpret_cast<uint64_t *>(d + o_keys);
    sp.kstate = d + o_kst;
    sp.sel_count = reinterpret_cast<uint32_t *>(d + fl.o_cnt);
    sp.sel_group = reinterpret_cast<int32_t *>(d + fl.o_sg);
    sp.sel_rows = reinterpret_cast<int64_t *>(d + fl.o_sr);
    sp.sel_i64 = reinterpret_cast<int64_t *>(d + fl.o_si);
    sp.sel_f64 = reinterpret_cast<double *>(d + fl.o_sf);
    fl.launches = launch_finalize_select(fp, sp, stream);
    if (slot.ensure_pinned(host_off + fl.out_bytes)) return fail(BYDB_ENOMEM, "cudaMallocHost failed");
    CUDA_TRY(cudaMemcpyAsync(slot.pinned + host_off, d + fl.o_out, fl.out_bytes, cudaMemcpyDeviceToHost, stream));
    return 0;
}

void finalize_parse(const uint8_t *h, const FinalLayout &fl, bydb_result *out) {
    const size_t A = fl.A;
    const size_t R = std::min<size_t>(*reinterpret_cast<const uint32_t *>(h + (fl.o_cnt - fl.o_out)), fl.cap);
    auto owner = new ResultOwner();
    const int32_t *sg = reinterpret_cast<const int32_t *>(h + (fl.o_sg - fl.o_out));
    const int64_t *sr = reinterpret_cast<const int64_t *>(h + (fl.o_sr - fl.o_out));
    const int64_t *si = reinterpret_cast<const int64_t *>(h + (fl.o_si - fl.o_out));
    const double *sf = reinterpret_cast<const double *>(h + (fl.o_sf - fl.o_out));
    owner->group_id.assign(sg, sg + R);
    owner->rows.assign(sr, sr + R);
    owner->is_float.assign(h + (fl.o_isf - fl.o_out), h + (fl.o_isf - fl.o_out) + A);
    owner->val_i64.assign(si, si + R * A);
    owner->val_f64.assign(sf, sf + R * A);
    out->n_rows = static_cast<int32_t>(R);
    out->n_aggs = static_cast<int32_t>(A);
    out->group_id = owner->group_id.data();
    out->rows = owner->rows.data();
    out->is_float = owner->is_float.data();
    out->val_i64 = owner->val_i64.data();
    out->val_f64 = owner->val_f64.data();
    out->owner = owner;
}


// finalisation + row selection + read-back of the result rows, synchronised and parsed
int finalize_to_host(bydb_ctx *ctx, const bydb_query *q, const Plan &plan, ExecSlot &slot, cudaStream_t stream, const uint8_t *d_table,
                     const TableLayout &tl, bydb_result *out, bool check_inband_status = false) {
    (void)ctx;
    FinalLayout fl;
    Scratch sc;
    int rc = finalize_enqueue(q, plan, slot, stream, d_table, tl, 0, fl, sc);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(stream));
    CUDA_TRY(cudaGetLastError());
    out->stats.d2h_bytes += fl.out_bytes;
    out->stats.kernel_launches += fl.launches;
    if (check_inband_status) {
        // the table came from bydb_scan_partials / a peer's mailbox slot (possibly another rank's): its status is in the table
        const uint32_t e = *reinterpret_cast<const uint32_t *>(slot.pinned + (fl.o_cnt - fl.o_out) + 8);
        g_last_dev_err = e;
        if (e != 0) return fail(dev_err_code(e), std::string(dev_err_text(e)) + " (status carried in a partial table)");
    }
    finalize_parse(slot.pinned, fl, out);
    return 0;
}

int make_plan(bydb_ctx *ctx, const bydb_query *q, const std::vector<std::shared_ptr<Part>> *given, Plan &plan) {
    if (given) {
        plan.parts = *given;
    } else {
        std::lock_guard<std::mutex> lk(ctx->mu);
        for (uint32_t i = 0; i < q->n_parts; ++i) {
            auto it = ctx->parts.find(q->parts[i]);
            if (it == ctx->parts.end()) return fail(BYDB_ENOENT, "unknown part handle");
            plan.parts.push_back(it->second);
        }
    }
    distinct_fields(q, plan.fcols, plan.agg_fcol);
    if (plan.fcols.size() > kMaxFcols) return fail(BYDB_EINVAL, "too many distinct aggregated fields (max 8)");
    plan.n_groups = q->series_group ? q->n_groups : 1;
    uint64_t nb = 0;
    for (auto &p : plan.parts) nb += p->dir.blocks.size();
    if (nb > 0x7fffffffull) return fail(BYDB_EINVAL, "too many blocks");
    plan.total_blocks = static_cast<uint32_t>(nb);
    plan.n_series = q->n_series;
    return 0;
}

int scan_agg_impl(bydb_ctx *ctx, const bydb_query *q, const std::vector<std::shared_ptr<Part>> *given, bydb_result *out, uint64_t h2d_pre) {
    Plan plan;
    int rc = make_plan(ctx, q, given, plan);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    SlotLease lease(ctx);
    if (lease.init()) return fail(BYDB_EIO, "cannot create stream");
    ExecSlot &slot = *lease.slot;
    TableLayout tl(static_cast<size_t>(plan.n_groups), plan.fcols.size());
    Scratch table;
    table.stream = slot.stream;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&table.base), tl.total, slot.stream));
    memset(&out->stats, 0, sizeof out->stats);
    out->stats.h2d_bytes = h2d_pre;
    {
        // size the pinned staging once: it must not be reallocated while copies from/to it are in flight
        const size_t G = static_cast<size_t>(plan.n_groups), A = q->n_aggs, NS = q->n_series;
        if (slot.ensure_pinned(NS * 12 + (G + 1) * 4 + G * (12 + 16 * A) + 16 * A + 8192)) return fail(BYDB_ENOMEM, "cudaMallocHost failed");
    }
    rc = run_scan(ctx, q, plan, slot, slot.stream, table.base, tl, &out->stats);
    // finalisation is enqueued behind the scan; one synchronisation covers both
    if (!rc) rc = finalize_to_host(ctx, q, plan, slot, slot.stream, table.base, tl, out);
    if (rc) {
        // a failure after something was enqueued: the slot (and, on the host path, the transient parts the kernels read)
        // go back to their pools when this returns, so nothing may still be in flight
        cudaStreamSynchronize(slot.stream);
        const std::string keep = g_last_error;
        (void)collect_scan(slot, nullptr);  // a device-side error of the scan, if any, still drives the lazy-unpack retry
        g_last_error = keep;
        bydb_result_free(ctx, out);
        return rc;
    }
    int rc2 = collect_scan(slot, &out->stats);
    if (rc2) {
        bydb_result_free(ctx, out);
        return rc2;
    }
    return rc;
}


// ------------------------------------------------------------------------------------------------
// Prepared queries: the whole step (staging copy, plan, scan, reduce, finalize, row selection, read-back) captured once
// into a CUDA graph and replayed.  A query executed many times (dashboards, alert rules) then costs one graph launch and
// one synchronisation instead of ~20 runtime calls.  Everything here is additive: bydb_scan_agg is untouched.
// ------------------------------------------------------------------------------------------------
}  // namespace

struct bydb_prepared {
    // deep copy of the query: the caller's arrays only live for the duration of bydb_query_prepare
    std::vector<bydb_part_h> parts;
    std::vector<uint64_t> sids;
    std::vector<int32_t> groups;
    std::vector<std::string> agg_names, pred_family, pred_tag;
    std::vector<std::vector<uint8_t>> pred_lit;
    std::vector<bydb_agg> aggs;
    std::vector<bydb_pred> preds;
    bydb_query q{};
    std::mutex mu;                     // one execution at a time per prepared query
    std::unique_ptr<ExecSlot> slot;    // dedicated stream + pinned staging: their addresses are baked into the graph
    cudaGraphExec_t exec = nullptr;
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    FinalLayout fl;
    size_t host_off = 0;
    std::vector<std::shared_ptr<Part>> held;  // the parts whose device pointers are baked into the graph stay alive with it
    bydb_stats captured{};             // host-side counters of one step (launch counts, byte counts)
    uint64_t runs = 0;
    bool capturable = true;
    // the collective form (bydb_scan_reduce_prepared): one captured graph per (root, slot parity)
    struct ReduceGraph {
        cudaGraphExec_t exec = nullptr;
        FinalLayout fl;
        bydb_stats captured{};
        std::vector<std::shared_ptr<Part>> held;
    };
    std::unordered_map<int, ReduceGraph> reduce_graphs;  // key = root * 2 + parity
    uint64_t reduce_runs = 0;
    bool reduce_capturable = true;
};

namespace {

void prepared_destroy(bydb_prepared *p) {
    if (!p) return;
    if (p->exec) cudaGraphExecDestroy(p->exec);
    for (auto &kv : p->reduce_graphs)
        if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    if (p->t0) cudaEventDestroy(p->t0);
    if (p->t1) cudaEventDestroy(p->t1);
    if (p->slot) {
        if (p->slot->stream) cudaStreamDestroy(p->slot->stream);
        for (auto &e : p->slot->ev)
            if (e) cudaEventDestroy(e);
        if (p->slot->busy) cudaEventDestroy(p->slot->busy);
        if (p->slot->pinned) cudaFreeHost(p->slot->pinned);
        for (uint8_t *r : p->slot->retired) cudaFreeHost(r);
        if (p->slot->zpage) cudaFreeHost(p->slot->zpage);
    }
    delete p;
}

// captures one step into p->exec; returns 0, or a code after leaving the stream out of capture mode
int prepared_capture(bydb_ctx *ctx, bydb_prepared *p) {
    Plan plan;
    int rc = make_plan(ctx, &p->q, nullptr, plan);
    if (rc) return rc;
    // the version-dedup precheck of run_scan synchronises: parts that overlap in time keep the uncaptured path
    for (size_t a = 0; a < plan.parts.size(); ++a)
        for (size_t b = a + 1; b < plan.parts.size(); ++b) {
            const PartDir &x = plan.parts[a]->dir, &y = plan.parts[b]->dir;
            if (x.blocks.empty() || y.blocks.empty()) continue;
            if (std::max(std::max(x.min_ts, y.min_ts), p->q.tmin) <= std::min(std::min(x.max_ts, y.max_ts), p->q.tmax)) {
                p->capturable = false;
                return 0;
            }
        }
    ExecSlot &slot = *p->slot;
    TableLayout tl(static_cast<size_t>(plan.n_groups), plan.fcols.size());
    const size_t G = static_cast<size_t>(plan.n_groups), A = p->q.n_aggs, NS = p->q.n_series;
    const size_t stage = align_up(NS * 12 + (G + 1) * 4 + 512, 256);
    p->host_off = stage;  // results land behind the staging area, which must survive from replay to replay
    if (slot.ensure_pinned(stage + G * (12 + 16 * A) + 16 * A + 16384)) return fail(BYDB_ENOMEM, "cudaMallocHost failed");
    memset(&p->captured, 0, sizeof p->captured);
    cudaError_t e = cudaStreamBeginCapture(slot.stream, cudaStreamCaptureModeThreadLocal);
    if (e != cudaSuccess) return fail(BYDB_EIO, std::string("cudaStreamBeginCapture: ") + cudaGetErrorString(e));
    {
        Scratch table, fin;
        table.stream = slot.stream;
        rc = cudaMallocAsync(reinterpret_cast<void **>(&table.base), tl.total, slot.stream) == cudaSuccess ? 0 : fail(BYDB_ENOMEM, "cudaMallocAsync (capture)");
        if (!rc) rc = run_scan(ctx, &p->q, plan, slot, slot.stream, table.base, tl, &p->captured, 0, true);
        if (!rc) rc = finalize_enqueue(&p->q, plan, slot, slot.stream, table.base, tl, p->host_off, p->fl, fin);
        // table / fin are released here: inside the capture, i.e. as free nodes of the graph
    }
    cudaGraph_t graph = nullptr;
    e = cudaStreamEndCapture(slot.stream, &graph);
    if (rc || e != cudaSuccess || !graph) {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        p->capturable = false;  // fall back to the uncaptured path for good
        return rc ? rc : 0;
    }
    e = cudaGraphInstantiate(&p->exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) {
        cudaGetLastError();
        p->exec = nullptr;
        p->capturable = false;
    }
    p->captured.kernel_launches += p->fl.launches;  // finalize + select_rows (one fused launch for few groups)
    p->captured.d2h_bytes += p->fl.out_bytes;
    p->held = plan.parts;
    return 0;
}

}  // namespace

// ================================================================================================
extern "C" {

const char *bydb_last_error(void) { return g_last_error.c_str(); }
const char *bydb_version(void) { return "bydb-b200 0.1 (sm_100a)"; }

int bydb_init(const bydb_cfg *cfg, bydb_ctx **out) {
    return guarded([&]() -> int {
    if (!out) return fail(BYDB_EINVAL, "out is NULL");
    *out = nullptr;
    int dev = cfg ? cfg->device : 0;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return fail(BYDB_EIO, "no CUDA device: libbydbgpu has no CPU fallback");
    if (dev < 0 || dev >= n) return fail(BYDB_EINVAL, "bad device ordinal");
    CUDA_TRY(cudaSetDevice(dev));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    if (prop.major < 10) return fail(BYDB_ENOTSUP, std::string("device '") + prop.name + "' is not sm_100 (Blackwell); this library is built for sm_100a only");
    auto ctx = new bydb_ctx();
    ctx->device = dev;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->hbm_budget = cfg ? cfg->hbm_budget_bytes : 0;
    ctx->host_index = cfg && (cfg->flags & BYDB_CFG_HOST_INDEX) != 0;
    if (upload_pow10_table()) {
        delete ctx;
        return fail(BYDB_EIO, "cannot upload constant tables (is the library built for this GPU?)");
    }
    {
        // keep freed stream-ordered allocations in the pool: every query allocates its scratch with
        // cudaMallocAsync, and the default threshold (0) would hand the memory back at each sync
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            uint64_t thr = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
            // never let the allocator satisfy a request by making the requesting stream wait for ANOTHER stream's pending free:
            // with several ranks on one device that other stream may sit behind a wait kernel spinning for this very rank
            // (the collective then stalls until the 60 s bound; seen as a test that failed only after the pool had history)
            int no = 0;
            cudaMemPoolSetAttribute(pool, cudaMemPoolReuseAllowInternalDependencies, &no);
        }
    }
    // execution slots (stream, events, pinned staging) for the first concurrent callers: made now, not inside a query
    for (int i = 0; i < 2; ++i) {
        std::unique_ptr<ExecSlot> sl(new ExecSlot());
        if (sl->create() != 0) {
            cudaGetLastError();
            break;
        }
        ctx->free_slots.push_back(std::move(sl));
    }
    preload_kernels();
    preload_unpack_kernels();
    preload_index_kernels();
    preload_encode_kernels();
    int occ_fast = 1, occ_slow = 1;
    scan_max_ctas_per_sm(&occ_fast, &occ_slow);
    int want = (cfg && cfg->warps_per_sm > 0) ? (cfg->warps_per_sm + kWarpsPerCta - 1) / kWarpsPerCta : 64;
    ctx->ctas_per_sm = std::max(1, std::min(want, occ_slow));
    ctx->ctas_per_sm_fast = std::max(1, std::min(want, occ_fast));
    *out = ctx;
    return 0;
    });
}

void bydb_shutdown(bydb_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (auto &s : ctx->free_slots) {
        if (s->stream) cudaStreamDestroy(s->stream);
        for (auto &e : s->ev)
            if (e) cudaEventDestroy(e);
        if (s->busy) cudaEventDestroy(s->busy);
        if (s->pinned) cudaFreeHost(s->pinned);
        for (uint8_t *r : s->retired) cudaFreeHost(r);
        if (s->zpage) cudaFreeHost(s->zpage);
    }
    ctx->free_slots.clear();
    ctx->parts.clear();
    for (int i = 0; i < StageRing::kBufs; ++i) {
        if (ctx->stage.buf[i]) cudaFreeHost(ctx->stage.buf[i]);
        if (ctx->stage.done[i]) cudaEventDestroy(ctx->stage.done[i]);
    }
    for (size_t r = 0; r < ctx->comm.peer.size(); ++r)
        if (ctx->comm.ipc_opened[r] && ctx->comm.peer[r]) cudaIpcCloseMemHandle(ctx->comm.peer[r]);
    if (ctx->comm.mine) cudaFree(ctx->comm.mine);
    if (ctx->comm.poll_stream) cudaStreamDestroy(ctx->comm.poll_stream);
    if (ctx->comm.poll_buf) cudaFreeHost(ctx->comm.poll_buf);
    delete ctx;
}

int bydb_part_register(bydb_ctx *ctx, uint64_t part_id, const bydb_part_files *files, bydb_part_h *out) {
    return guarded([&]() -> int {
    if (!ctx || !out) return fail(BYDB_EINVAL, "ctx/out is NULL");
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        auto it = ctx->by_id.find(part_id);
        if (it != ctx->by_id.end()) {  // idempotent per part_id
            *out = it->second;
            return 0;
        }
    }
    CUDA_TRY(cudaSetDevice(ctx->device));
    std::shared_ptr<Part> part;
    int rc = register_part_locked_free(ctx, part_id, files, part, nullptr, false, false, 0, 1, true, nullptr, !ctx->host_index);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    auto again = ctx->by_id.find(part_id);
    if (again != ctx->by_id.end()) {
        // another thread registered the same part meanwhile: keep its copy, drop ours (idempotent per part_id)
        ctx->hbm_used -= part->hbm_bytes;
        *out = again->second;
        return 0;
    }
    bydb_part_h h = ctx->next_handle++;
    ctx->parts[h] = part;
    ctx->by_id[part_id] = h;
    *out = h;
    return 0;
    });
}

int bydb_part_release(bydb_ctx *ctx, bydb_part_h h) {
    return guarded([&]() -> int {
    if (!ctx) return fail(BYDB_EINVAL, "ctx is NULL");
    std::shared_ptr<Part> victim;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        auto it = ctx->parts.find(h);
        if (it == ctx->parts.end()) return fail(BYDB_ENOENT, "unknown part handle");
        victim = it->second;
        ctx->by_id.erase(victim->id);
        ctx->parts.erase(it);
        ctx->hbm_used -= victim->hbm_bytes;
    }
    cudaSetDevice(ctx->device);
    victim.reset();  // frees HBM once no in-flight query holds the part
    return 0;
    });
}

int bydb_part_info(bydb_ctx *ctx, bydb_part_h h, uint64_t *hbm_bytes, uint64_t *n_blocks, uint64_t *n_rows) {
    return guarded([&]() -> int {
    if (!ctx) return fail(BYDB_EINVAL, "ctx is NULL");
    std::lock_guard<std::mutex> lk(ctx->mu);
    auto it = ctx->parts.find(h);
    if (it == ctx->parts.end()) return fail(BYDB_ENOENT, "unknown part handle");
    if (hbm_bytes) *hbm_bytes = it->second->hbm_bytes;
    if (n_blocks) *n_blocks = it->second->dir.blocks.size();
    if (n_rows) *n_rows = it->second->dir.total_rows;
    return 0;
    });
}

int bydb_part_fallback_pages(bydb_ctx *ctx, bydb_part_h h, uint64_t *unpacked, uint64_t *left) {
    return guarded([&]() -> int {
    if (!ctx) return fail(BYDB_EINVAL, "ctx is NULL");
    std::lock_guard<std::mutex> lk(ctx->mu);
    auto it = ctx->parts.find(h);
    if (it == ctx->parts.end()) return fail(BYDB_ENOENT, "unknown part handle");
    if (unpacked) *unpacked = it->second->unpacked_pages;
    if (left) *left = it->second->unpack_skipped;
    return 0;
    });
}

int bydb_part_directory(bydb_ctx *ctx, bydb_part_h h, void *blocks_out, uint64_t blocks_cap_bytes, void *cols_out, uint64_t cols_cap_bytes, uint64_t *n_blocks,
                        uint64_t *n_cols) {
    return guarded([&]() -> int {
    if (!ctx) return fail(BYDB_EINVAL, "ctx is NULL");
    std::shared_ptr<Part> part;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        auto it = ctx->parts.find(h);
        if (it == ctx->parts.end()) return fail(BYDB_ENOENT, "unknown part handle");
        part = it->second;
    }
    const uint64_t nb = part->dir.blocks.size(), nc = part->dir.cols.size();
    if (n_blocks) *n_blocks = nb;
    if (n_cols) *n_cols = nc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (blocks_out) {
        if (blocks_cap_bytes < nb * sizeof(DevBlock)) return fail(BYDB_EINVAL, "blocks buffer too small");
        if (nb) CUDA_TRY(cudaMemcpy(blocks_out, part->d_blocks, nb * sizeof(DevBlock), cudaMemcpyDeviceToHost));
    }
    if (cols_out) {
        if (cols_cap_bytes < nc * sizeof(DevCol)) return fail(BYDB_EINVAL, "cols buffer too small");
        if (nc) CUDA_TRY(cudaMemcpy(cols_out, part->d_cols, nc * sizeof(DevCol), cudaMemcpyDeviceToHost));
    }
    return 0;
    });
}

int bydb_scan_agg(bydb_ctx *ctx, const bydb_query *q, bydb_result *out) {
    return guarded([&]() -> int {
    if (!ctx || !out) return fail(BYDB_EINVAL, "ctx/out is NULL");
    memset(out, 0, sizeof *out);
    int rc = validate_query(q, true);
    if (rc) return rc;
    return scan_agg_impl(ctx, q, nullptr, out, 0);
    });
}


// ------------------------------------------------------------------------------------------------
// Gather path of the cold query (host images in pageable memory, e.g. BanyanDB's mmap'd part files): instead of copying
// every file of the part to HBM (12.8 GB for the 1e9 bench part, 1.1 s from pageable memory), the host selects the blocks
// like plan_blocks does and collects ONLY the pages the query reads -- the timestamps page, the aggregated fields, the
// predicate tags -- into one arena image per slice: [DevBlock[] | DevCol[] | file table | pages], every page offset
// rewritten into the arena.  The image goes up through the pinned staging ring in 64 MB chunks.
// ------------------------------------------------------------------------------------------------

namespace {
struct KeyedOwner {
    std::vector<int32_t> key_id;
    std::vector<uint32_t> key_off;
    std::vector<uint8_t> key_bytes;
};

// The checks every group-key entry point makes before it touches the device: the key, its value cap, the predicate budget,
// the plan, and no two parts that overlap in time.
int keyed_prepare(bydb_ctx *ctx, const bydb_query *q, const bydb_group_key *key, Plan &plan, uint32_t &cap) {
    int rc = validate_query(q, true);
    if (rc) return rc;
    if (!key || !key->family || !key->tag) return fail(BYDB_EINVAL, "group key without family/tag");
    cap = key->max_values ? key->max_values : 64u;
    if (cap > kMaxKeyValues) return fail(BYDB_EINVAL, "bydb_group_key.max_values above 256");
    if (q->n_preds + 1 > kMaxPreds) return fail(BYDB_ENOTSUP, "a group-key query takes at most 7 predicates");
    rc = make_plan(ctx, q, nullptr, plan);
    if (rc) return rc;
    for (size_t a = 0; a < plan.parts.size(); ++a)
        for (size_t b = a + 1; b < plan.parts.size(); ++b) {
            const PartDir &x = plan.parts[a]->dir, &y = plan.parts[b]->dir;
            if (x.blocks.empty() || y.blocks.empty()) continue;
            if (std::max(std::max(x.min_ts, y.min_ts), q->tmin) <= std::min(std::min(x.max_ts, y.max_ts), q->tmax))
                return fail(BYDB_ENOTSUP, "group-key query over parts that overlap in time (version dedup) is not supported on the device path");
        }
    return 0;
}

// Step 1 of a group-key query: the distinct key values of the selected blocks.  The device copies stay in `sc`: the query's
// series ids at d_sids, the packed values (cap x kMaxLit bytes) at d_vals, their lengths at d_lens.
struct KeyValues {
    Scratch sc;
    const uint64_t *d_sids = nullptr;
    const uint8_t *d_vals = nullptr;
    const uint32_t *d_lens = nullptr;
    std::vector<std::vector<uint8_t>> values;
};

int keyed_values(bydb_ctx *ctx, const bydb_query *q, const bydb_group_key *key, uint32_t cap, const Plan &plan, ExecSlot &slot, bydb_stats *stats,
                 KeyValues &kv) {
    cudaStream_t stream = slot.stream;
    const size_t NS = q->n_series, NB = plan.total_blocks;
    size_t o = 0;
    auto carve = [&](size_t bytes) {
        size_t at = o;
        o = align_up(o + bytes, 256);
        return at;
    };
    const size_t a_sids = carve(NS * 8), a_slots = carve(kKeySlots * 8), a_ctl = carve(16), a_vals = carve(static_cast<size_t>(cap) * kMaxLit),
                 a_lens = carve(static_cast<size_t>(cap) * 4);
    const size_t a_total = o;
    Scratch &ka = kv.sc;
    ka.stream = stream;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&ka.base), a_total, stream));
    kv.d_sids = reinterpret_cast<const uint64_t *>(ka.base + a_sids);
    kv.d_vals = ka.base + a_vals;
    kv.d_lens = reinterpret_cast<const uint32_t *>(ka.base + a_lens);
    const size_t back_bytes = a_total - a_ctl;  // ctl | vals | lens come back in one copy
    if (slot.ensure_pinned(std::max(back_bytes, NS * 8) + 256)) return fail(BYDB_ENOMEM, "cudaMallocHost failed");
    if (NS) memcpy(slot.pinned, q->series_ids, NS * 8);
    if (NS) CUDA_TRY(cudaMemcpyAsync(ka.base + a_sids, slot.pinned, NS * 8, cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaMemsetAsync(ka.base + a_slots, 0, a_total - a_slots, stream));
    KeyParams kpar;
    memset(&kpar, 0, sizeof kpar);
    {
        uint32_t base = 0;
        for (size_t i = 0; i < plan.parts.size(); ++i) {
            DevPartRef r;
            r.blocks = plan.parts[i]->d_blocks;
            r.cols = plan.parts[i]->d_cols;
            r.files = plan.parts[i]->d_files;
            r.n_blocks = static_cast<uint32_t>(plan.parts[i]->dir.blocks.size());
            r.block_base = base;
            base += r.n_blocks;
            kpar.parts[i] = r;
        }
    }
    kpar.n_parts = static_cast<uint32_t>(plan.parts.size());
    kpar.total_blocks = static_cast<uint32_t>(NB);
    kpar.q_sids = reinterpret_cast<const uint64_t *>(ka.base + a_sids);
    kpar.n_series = static_cast<uint32_t>(NS);
    kpar.cap = cap;
    kpar.tmin = q->tmin;
    kpar.tmax = q->tmax;
    kpar.key_name = ctx->names.find(std::string("t:") + key->family + "/" + key->tag);
    kpar.slots = reinterpret_cast<unsigned long long *>(ka.base + a_slots);
    kpar.count = reinterpret_cast<uint32_t *>(ka.base + a_ctl);
    kpar.err = reinterpret_cast<uint32_t *>(ka.base + a_ctl) + 1;
    kpar.vals = ka.base + a_vals;
    kpar.lens = reinterpret_cast<uint32_t *>(ka.base + a_lens);
    launch_key_values(kpar, ctx->sm_count * 4, stream);
    CUDA_TRY(cudaStreamSynchronize(stream));  // the staging of the series ids must be consumed before the read-back reuses it
    CUDA_TRY(cudaMemcpyAsync(slot.pinned, ka.base + a_ctl, back_bytes, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    CUDA_TRY(cudaGetLastError());
    stats->kernel_launches += 2;
    stats->h2d_bytes += NS * 8;
    stats->d2h_bytes += back_bytes;
    const uint32_t *ctl = reinterpret_cast<const uint32_t *>(slot.pinned);
    if (ctl[1] != 0) {
        g_last_dev_err = ctl[1];
        char buf[64];
        snprintf(buf, sizeof buf, " (block #%u)", ctl[2]);
        return fail(dev_err_code(ctl[1]), std::string(dev_err_text(ctl[1])) + buf);
    }
    const size_t V = std::min<size_t>(ctl[0], cap);
    kv.values.assign(V, {});
    const uint8_t *hv = slot.pinned + (a_vals - a_ctl);
    const uint32_t *hl = reinterpret_cast<const uint32_t *>(slot.pinned + (a_lens - a_ctl));
    for (size_t v = 0; v < V; ++v) kv.values[v].assign(hv + v * kMaxLit, hv + v * kMaxLit + hl[v]);
    return 0;
}

// Step 2: one scan pass per value v (the key as an extra predicate) into slice v of a composite table of V x G groups
// (value-major) at `table` with layout `tl`; pass v leaves its column types at coltype[v * F] and, per series, where it first
// shows v at kts / krow[v * NS].  Every pass is synchronised and its device errors collected.
int keyed_passes(bydb_ctx *ctx, const bydb_query *q, const bydb_group_key *key, Plan &plan, ExecSlot &slot, const KeyValues &kv, uint8_t *table,
                 const TableLayout &tl, int64_t *coltype, int64_t *kts, uint32_t *krow, bydb_stats *stats) {
    cudaStream_t stream = slot.stream;
    const size_t F = plan.fcols.size(), NS = q->n_series, G = static_cast<size_t>(plan.n_groups);
    std::vector<bydb_pred> preds(q->preds, q->preds + q->n_preds);
    preds.emplace_back();
    bydb_query qv = *q;
    qv.n_preds = q->n_preds + 1;
    for (size_t v = 0; v < kv.values.size(); ++v) {
        bydb_pred &kpred = preds.back();
        memset(&kpred, 0, sizeof kpred);
        kpred.family = key->family;
        kpred.tag = key->tag;
        kpred.op = kv.values[v].empty() ? kOpEqOrNil : BYDB_OP_EQ;  // a nil cell and "" are the same key (groupby.go:226-254)
        kpred.value_type = BYDB_VT_STR;
        kpred.lit = kv.values[v].data();
        kpred.lit_len = kv.values[v].size();
        qv.preds = preds.data();
        KeyedPass pass;
        pass.group_off = v * G;
        pass.coltype = coltype + v * F;
        pass.kts = kts + v * NS;
        pass.krow = krow + v * NS;
        int rc = run_scan(ctx, &qv, plan, slot, stream, table, tl, stats, 0, true, &pass);
        cudaError_t ce = cudaStreamSynchronize(stream);  // also on failure: nothing may be in flight when the slot goes back
        if (!rc && ce != cudaSuccess) rc = fail(BYDB_EIO, cudaGetErrorString(ce));
        if (!rc) rc = collect_scan(slot, stats);
        if (rc) return rc;
    }
    return 0;
}

// order | group_start of the series groups (run_scan's copies live in its own scratch), uploaded into `sc` through the staging
int upload_group_order(const bydb_query *q, size_t G, ExecSlot &slot, Scratch &sc, const int32_t **order_out, const int32_t **gstart_out) {
    const size_t NS = q->n_series;
    std::vector<int32_t> order(NS), gstart(G + 1, 0);
    if (q->series_group) {
        for (size_t i = 0; i < NS; ++i) gstart[static_cast<size_t>(q->series_group[i]) + 1]++;
        for (size_t g = 0; g < G; ++g) gstart[g + 1] += gstart[g];
        std::vector<int32_t> cur(gstart.begin(), gstart.end() - 1);
        for (size_t i = 0; i < NS; ++i) order[cur[q->series_group[i]]++] = static_cast<int32_t>(i);
    } else {
        for (size_t i = 0; i < NS; ++i) order[i] = static_cast<int32_t>(i);
        gstart[1] = static_cast<int32_t>(NS);
    }
    sc.stream = slot.stream;
    const size_t c_gstart = align_up(NS * 4, 256);
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&sc.base), c_gstart + (G + 1) * 4, slot.stream));
    if (NS) memcpy(slot.pinned, order.data(), NS * 4);
    memcpy(slot.pinned + c_gstart, gstart.data(), (G + 1) * 4);
    CUDA_TRY(cudaMemcpyAsync(sc.base, slot.pinned, c_gstart + (G + 1) * 4, cudaMemcpyHostToDevice, slot.stream));
    *order_out = reinterpret_cast<const int32_t *>(sc.base);
    *gstart_out = reinterpret_cast<const int32_t *>(sc.base + c_gstart);
    return 0;
}

TablePtrs table_ptrs(uint8_t *t, const TableLayout &tl) {
    TablePtrs tp;
    tp.sum_f64 = reinterpret_cast<double *>(t + tl.off_sum_f64);
    tp.max_f64 = reinterpret_cast<double *>(t + tl.off_max_f64);
    tp.negmin_f64 = reinterpret_cast<double *>(t + tl.off_negmin_f64);
    tp.sum_i64 = reinterpret_cast<int64_t *>(t + tl.off_sum_i64);
    tp.cnt = reinterpret_cast<int64_t *>(t + tl.off_cnt);
    tp.rows = reinterpret_cast<int64_t *>(t + tl.off_rows);
    tp.max_i64 = reinterpret_cast<int64_t *>(t + tl.off_max_i64);
    tp.notmin_i64 = reinterpret_cast<int64_t *>(t + tl.off_notmin_i64);
    tp.coltype = reinterpret_cast<int64_t *>(t + tl.off_coltype);
    return tp;
}

// The finalised rows carry the position of their composite group in insertion order: back to (group of the series, key value)
void keyed_split_rows(bydb_keyed_result *out, const std::vector<int32_t> &perm, size_t G) {
    auto *owner = static_cast<KeyedOwner *>(out->owner);
    auto *ro = static_cast<ResultOwner *>(out->base.owner);
    owner->key_id.resize(ro->group_id.size());
    for (size_t r = 0; r < ro->group_id.size(); ++r) {
        const int32_t comp = perm[static_cast<size_t>(ro->group_id[r])];
        owner->key_id[r] = comp / static_cast<int32_t>(G);
        ro->group_id[r] = comp % static_cast<int32_t>(G);
    }
    out->key_id = owner->key_id.data();
}
}  // namespace

void bydb_keyed_result_free(bydb_ctx *ctx, bydb_keyed_result *r);
void bydb_encoded_pages_free(bydb_ctx *ctx, bydb_encoded_pages *r);

// Group-by on a stored tag (per-row key): see "Group key" in scan_kernels.cu for the device side.
int bydb_scan_agg_keyed(bydb_ctx *ctx, const bydb_query *q, const bydb_group_key *key, bydb_keyed_result *out) {
    return guarded([&]() -> int {
    if (!ctx || !out) return fail(BYDB_EINVAL, "ctx/out is NULL");
    memset(out, 0, sizeof *out);
    Plan plan;
    uint32_t cap = 0;
    int rc = keyed_prepare(ctx, q, key, plan, cap);
    if (rc) return rc;
    g_last_dev_err = 0;
    CUDA_TRY(cudaSetDevice(ctx->device));
    SlotLease lease(ctx);
    if (lease.init()) return fail(BYDB_EIO, "cannot create stream");
    ExecSlot &slot = *lease.slot;
    cudaStream_t stream = slot.stream;
    const size_t F = plan.fcols.size(), NS = q->n_series, G = static_cast<size_t>(plan.n_groups);
    memset(&out->base.stats, 0, sizeof out->base.stats);

    // ---- 1. the distinct key values of the selected blocks
    KeyValues kv;
    rc = keyed_values(ctx, q, key, cap, plan, slot, &out->base.stats, kv);
    if (rc) return rc;
    const std::vector<std::vector<uint8_t>> &values = kv.values;
    const size_t V = values.size();
    auto owner = new KeyedOwner();
    out->owner = owner;
    bool done = false;
    struct Undo {  // a failure past this point must not leave a half-filled result with the caller
        bydb_ctx *ctx;
        bydb_keyed_result *out;
        bool *done;
        ~Undo() {
            if (!*done) bydb_keyed_result_free(ctx, out);
        }
    } undo{ctx, out, &done};
    owner->key_off.push_back(0);
    for (size_t v = 0; v < V; ++v) {
        owner->key_bytes.insert(owner->key_bytes.end(), values[v].begin(), values[v].end());
        owner->key_off.push_back(static_cast<uint32_t>(owner->key_bytes.size()));
    }
    if (owner->key_bytes.empty()) owner->key_bytes.push_back(0);
    out->n_keys = static_cast<int32_t>(V);
    out->key_off = owner->key_off.data();
    out->key_bytes = owner->key_bytes.data();
    if (V == 0) {  // no block selected: no rows (n_rows = 0)
        done = true;
        return 0;
    }

    // ---- 2. one scan pass per value into slice v of the composite table (V x G groups, value-major)
    const size_t GP = G * V;
    if (GP > 0x7fffffffull / std::max<size_t>(F, 1)) return fail(BYDB_ENOMEM, "group-key query: too many composite groups");
    TableLayout tlc(GP, F);
    size_t o = 0;
    auto carve = [&](size_t bytes) {
        size_t at = o;
        o = align_up(o + bytes, 256);
        return at;
    };
    const size_t b_src = carve(tlc.total), b_dst = carve(tlc.total), b_ct = carve(V * F * 8), b_kts = carve(V * NS * 8), b_krow = carve(V * NS * 4),
                 b_slot = carve(NS * V * 4), b_first = carve(GP * 4), b_perm = carve(GP * 4), b_np = carve(16);
    Scratch kb;
    kb.stream = stream;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&kb.base), o, stream));
    CUDA_TRY(cudaMemsetAsync(kb.base + b_ct, 0, V * F * 8, stream));
    CUDA_TRY(cudaMemsetAsync(kb.base + b_slot, 0xff, NS * V * 4, stream));
    {
        const size_t A = q->n_aggs;
        if (slot.ensure_pinned(NS * 12 + (G + 1) * 4 + GP * (12 + 16 * A) + 16 * A + 8192)) return fail(BYDB_ENOMEM, "cudaMallocHost failed");
    }
    rc = keyed_passes(ctx, q, key, plan, slot, kv, kb.base + b_src, tlc, reinterpret_cast<int64_t *>(kb.base + b_ct),
                      reinterpret_cast<int64_t *>(kb.base + b_kts), reinterpret_cast<uint32_t *>(kb.base + b_krow), &out->base.stats);
    if (rc) return rc;

    // ---- 3. insertion order of the composite groups, table reordered, ordinary finalisation / Top-N on it
    KeyOrderParams ko;
    memset(&ko, 0, sizeof ko);
    ko.n_groups = static_cast<int32_t>(G);
    ko.n_values = static_cast<uint32_t>(V);
    ko.n_series = static_cast<uint32_t>(NS);
    Scratch kc;
    rc = upload_group_order(q, G, slot, kc, &ko.order, &ko.group_start);
    if (rc) return rc;
    ko.Kts = reinterpret_cast<const int64_t *>(kb.base + b_kts);
    ko.Krow = reinterpret_cast<const uint32_t *>(kb.base + b_krow);
    ko.slot = reinterpret_cast<int32_t *>(kb.base + b_slot);
    ko.first_series = reinterpret_cast<int32_t *>(kb.base + b_first);
    ko.perm = reinterpret_cast<int32_t *>(kb.base + b_perm);
    ko.n_present = reinterpret_cast<uint32_t *>(kb.base + b_np);
    launch_key_order(ko, stream);
    launch_permute_table(table_ptrs(kb.base + b_dst, tlc), table_ptrs(kb.base + b_src, tlc), ko.perm, static_cast<uint32_t>(GP), static_cast<uint32_t>(F),
                         reinterpret_cast<const int64_t *>(kb.base + b_ct), static_cast<uint32_t>(V), stream);
    CUDA_TRY(cudaStreamSynchronize(stream));  // the staging above is reused by the finalisation's read-back
    out->base.stats.kernel_launches += 3;
    Plan planc = plan;
    planc.n_groups = static_cast<int32_t>(GP);
    rc = finalize_to_host(ctx, q, planc, slot, stream, kb.base + b_dst, tlc, &out->base, true);
    if (rc) {
        cudaStreamSynchronize(stream);
        return rc;
    }
    std::vector<int32_t> perm(GP);
    CUDA_TRY(cudaMemcpyAsync(perm.data(), kb.base + b_perm, GP * 4, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    out->base.stats.d2h_bytes += GP * 4;
    keyed_split_rows(out, perm, G);
    done = true;
    return 0;
    });
}

void bydb_keyed_result_free(bydb_ctx *ctx, bydb_keyed_result *r) {
    if (!r) return;
    bydb_result_free(ctx, &r->base);
    delete static_cast<KeyedOwner *>(r->owner);
    memset(r, 0, sizeof *r);
}


namespace {
struct EncodedOwner {
    std::vector<uint64_t> page_off;
    std::vector<uint8_t> bytes, needs_cpu;
};
}  // namespace

// Write side (f4): numeric field pages encoded on the device, see encode_kernels.cu.
int bydb_encode_pages(bydb_ctx *ctx, const bydb_encode_input *in, bydb_encoded_pages *out) {
    return guarded([&]() -> int {
    if (!ctx || !in || !out) return fail(BYDB_EINVAL, "ctx/in/out is NULL");
    memset(out, 0, sizeof *out);
    if (in->value_type != BYDB_VT_INT64 && in->value_type != BYDB_VT_FLOAT64) return fail(BYDB_EINVAL, "bydb_encode_pages takes int64 or float64 columns");
    if (in->n_blocks > 0 && (!in->block_rows || !in->values)) return fail(BYDB_EINVAL, "block_rows / values is NULL");
    const size_t NB = in->n_blocks;
    const bool is_float = in->value_type == BYDB_VT_FLOAT64;
    std::vector<uint64_t> block_off(NB + 1, 0), slot_off(NB + 1, 0);
    for (size_t b = 0; b < NB; ++b) {
        if (in->block_rows[b] == 0) return fail(BYDB_EINVAL, "a block without rows");
        block_off[b + 1] = block_off[b] + in->block_rows[b];
        slot_off[b + 1] = slot_off[b] + align_up(11 + 10 * static_cast<size_t>(in->block_rows[b]), 16);  // a varint takes at most 10 bytes
    }
    const size_t NV = block_off[NB];
    auto owner = new EncodedOwner();
    out->owner = owner;
    out->n_blocks = in->n_blocks;
    owner->page_off.assign(NB + 1, 0);
    owner->needs_cpu.assign(std::max<size_t>(NB, 1), 0);
    owner->bytes.assign(1, 0);
    out->page_off = owner->page_off.data();
    out->needs_cpu = owner->needs_cpu.data();
    out->bytes = owner->bytes.data();
    if (NB == 0) return 0;
    bool done = false;
    struct Undo {
        bydb_ctx *ctx;
        bydb_encoded_pages *out;
        bool *done;
        ~Undo() {
            if (!*done) bydb_encoded_pages_free(ctx, out);
        }
    } undo{ctx, out, &done};
    CUDA_TRY(cudaSetDevice(ctx->device));
    SlotLease lease(ctx);
    if (lease.init()) return fail(BYDB_EIO, "cannot create stream");
    cudaStream_t stream = lease.slot->stream;
    size_t o = 0;
    auto carve = [&](size_t bytes) {
        size_t at = o;
        o = align_up(o + bytes, 256);
        return at;
    };
    const size_t d_vals = carve(NV * 8), d_boff = carve((NB + 1) * 8), d_soff = carve((NB + 1) * 8), d_scr = carve(is_float ? NV * 8 : 0),
                 d_exp = carve(is_float ? NV * 2 : 0), d_len = carve(NB * 4), d_st = carve(NB), d_ooff = carve((NB + 1) * 8), d_slots = carve(slot_off[NB]);
    Scratch sc;
    sc.stream = stream;
    if (cudaMallocAsync(reinterpret_cast<void **>(&sc.base), o, stream) != cudaSuccess) {
        cudaGetLastError();
        return fail(BYDB_ENOMEM, "bydb_encode_pages: device allocation failed");
    }
    uint8_t *d = sc.base;
    cudaEvent_t ev0 = lease.slot->ev[0], ev1 = lease.slot->ev[1], ev2 = lease.slot->ev[2], ev3 = lease.slot->ev[3];
    CUDA_TRY(cudaMemcpyAsync(d + d_vals, in->values, NV * 8, cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaMemcpyAsync(d + d_boff, block_off.data(), (NB + 1) * 8, cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaMemcpyAsync(d + d_soff, slot_off.data(), (NB + 1) * 8, cudaMemcpyHostToDevice, stream));
    EncodeParams ep;
    memset(&ep, 0, sizeof ep);
    ep.values = d + d_vals;
    ep.block_off = reinterpret_cast<const uint64_t *>(d + d_boff);
    ep.n_blocks = static_cast<uint32_t>(NB);
    ep.is_float = is_float ? 1u : 0u;
    ep.scratch = reinterpret_cast<int64_t *>(d + d_scr);
    ep.exps = reinterpret_cast<int16_t *>(d + d_exp);
    ep.slots = d + d_slots;
    ep.slot_off = reinterpret_cast<const uint64_t *>(d + d_soff);
    ep.page_len = reinterpret_cast<uint32_t *>(d + d_len);
    ep.status = d + d_st;
    const int grid = ctx->sm_count * 4;
    CUDA_TRY(cudaEventRecord(ev0, stream));
    launch_encode_pages(ep, grid, stream);
    CUDA_TRY(cudaEventRecord(ev1, stream));
    std::vector<uint32_t> page_len(NB);
    CUDA_TRY(cudaMemcpyAsync(page_len.data(), d + d_len, NB * 4, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaMemcpyAsync(owner->needs_cpu.data(), d + d_st, NB, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    CUDA_TRY(cudaGetLastError());
    for (size_t b = 0; b < NB; ++b) {
        owner->page_off[b + 1] = owner->page_off[b] + page_len[b];
        out->n_cpu_blocks += owner->needs_cpu[b] ? 1u : 0u;
    }
    const size_t total = owner->page_off[NB];
    owner->bytes.assign(std::max<size_t>(total, 1), 0);
    out->bytes = owner->bytes.data();
    Scratch compact;
    compact.stream = stream;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&compact.base), std::max<size_t>(total, 256), stream));
    CUDA_TRY(cudaMemcpyAsync(d + d_ooff, owner->page_off.data(), (NB + 1) * 8, cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaEventRecord(ev2, stream));
    launch_gather_pages(ep, reinterpret_cast<const uint64_t *>(d + d_ooff), compact.base, grid, stream);
    CUDA_TRY(cudaEventRecord(ev3, stream));
    if (total) CUDA_TRY(cudaMemcpyAsync(owner->bytes.data(), compact.base, total, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    CUDA_TRY(cudaGetLastError());
    float ms = 0, ms2 = 0;  // the two kernels only: the host's prefix sum of the page lengths lies between them
    cudaEventElapsedTime(&ms, ev0, ev1);
    cudaEventElapsedTime(&ms2, ev2, ev3);
    out->device_ms = ms + ms2;
    done = true;
    return 0;
    });
}

void bydb_encoded_pages_free(bydb_ctx *, bydb_encoded_pages *r) {
    if (!r) return;
    delete static_cast<EncodedOwner *>(r->owner);
    memset(r, 0, sizeof *r);
}

struct GatherSeg {
    const uint8_t *src;
    size_t dst;
    size_t len;
};
struct GatherImage {
    std::vector<DevBlock> blocks;
    std::vector<DevCol> cols;
    std::vector<GatherSeg> segs;  // ascending dst
    size_t off_cols = 0, off_files = 0, off_pages = 0, bytes = 0;
    uint64_t page_bytes = 0;
};

static int plan_gather(bydb_ctx *ctx, const std::vector<FileImage> &imgs, const bydb_query *q, const Plan &base, const PartDir &dir, GatherImage &g) {
    std::vector<uint16_t> need;
    for (const auto &f : base.fcols) need.push_back(ctx->names.find("f:" + f));
    for (uint32_t i = 0; i < q->n_preds; ++i) need.push_back(ctx->names.find(std::string("t:") + q->preds[i].family + "/" + q->preds[i].tag));
    std::vector<const FileImage *> file_of(dir.files.size(), nullptr);
    for (size_t i = 0; i < dir.files.size(); ++i)
        for (const auto &f : imgs)
            if (f.name == dir.files[i]) file_of[i] = &f;
    if (file_of.empty() || !file_of[0]) return fail(BYDB_ENOENT, "missing timestamps.bin");
    const uint64_t *sb = q->series_ids, *se = q->series_ids + q->n_series;
    struct Page {
        const uint8_t *src;
        uint32_t len;
    };
    std::vector<Page> pages;
    for (const DevBlock &b : dir.blocks) {
        const uint64_t *it = std::lower_bound(sb, se, b.sid);
        if (it == se || *it != b.sid || b.ts_max < q->tmin || b.ts_min > q->tmax) continue;  // plan_blocks' selection (part_iter.go:232-241)
        DevBlock nb = b;
        nb.col_begin = static_cast<uint32_t>(g.cols.size());
        pages.push_back({file_of[0]->data + b.ts_off, b.ts_size});
        uint16_t kept = 0;
        for (uint32_t c = 0; c < b.n_cols; ++c) {
            const DevCol &col = dir.cols[b.col_begin + c];
            if (col.name_id == 0 || std::find(need.begin(), need.end(), col.name_id) == need.end()) continue;
            if (col.file_id >= file_of.size() || !file_of[col.file_id]) return fail(BYDB_ENOENT, "missing file of a column page");
            DevCol nc = col;
            nc.file_id = 0;
            pages.push_back({file_of[col.file_id]->data + col.off, col.size});
            g.cols.push_back(nc);
            ++kept;
        }
        nb.n_cols = kept;
        g.blocks.push_back(nb);
    }
    // layout: directory first, then the pages (16 B aligned, >= 8 B apart: bit windows read a few bytes past a page)
    g.off_cols = align_up(g.blocks.size() * sizeof(DevBlock), 256);
    g.off_files = g.off_cols + align_up(g.cols.size() * sizeof(DevCol), 256);
    g.off_pages = g.off_files + 256;
    size_t cur = g.off_pages, pi = 0;
    g.segs.reserve(pages.size() + 3);
    if (!g.blocks.empty()) g.segs.push_back({reinterpret_cast<const uint8_t *>(g.blocks.data()), 0, g.blocks.size() * sizeof(DevBlock)});
    if (!g.cols.empty()) g.segs.push_back({reinterpret_cast<const uint8_t *>(g.cols.data()), g.off_cols, g.cols.size() * sizeof(DevCol)});
    g.segs.push_back({nullptr, g.off_files, 2 * sizeof(void *)});  // the file table: filled in once the arena address is known
    size_t ci = 0;
    for (DevBlock &nb : g.blocks) {
        nb.ts_off = cur;
        g.segs.push_back({pages[pi].src, cur, pages[pi].len});
        g.page_bytes += pages[pi].len;
        cur = align_up(cur + pages[pi].len + 8, 16);
        ++pi;
        for (uint16_t c = 0; c < nb.n_cols; ++c, ++ci, ++pi) {
            g.cols[ci].off = cur;
            g.segs.push_back({pages[pi].src, cur, pages[pi].len});
            g.page_bytes += pages[pi].len;
            cur = align_up(cur + pages[pi].len + 8, 16);
        }
    }
    g.bytes = align_up(cur + 256, 256);
    return 0;
}

// uploads the image through the staging ring onto `stream`; the copies of one chunk are spread over the worker pool
// the pinned staging ring of the gather path: made at the first pageable cold query -- or at bydb_comm_connect, because a
// page-locked allocation INSIDE a collective can stall peers that share the device (see ExecSlot::ensure_pinned)
static int ensure_stage_ring(bydb_ctx *ctx) {
    StageRing &ring = ctx->stage;
    for (int i = 0; i < StageRing::kBufs; ++i) {
        if (ring.buf[i]) continue;
        if (cudaMallocHost(reinterpret_cast<void **>(&ring.buf[i]), StageRing::kBytes) != cudaSuccess ||
            cudaEventCreateWithFlags(&ring.done[i], cudaEventDisableTiming) != cudaSuccess)
            return fail(BYDB_ENOMEM, "cannot allocate the pinned staging ring");
    }
    return 0;
}

static int upload_gather(bydb_ctx *ctx, GatherImage &g, uint8_t *d_arena, cudaStream_t stream) {
    StageRing &ring = ctx->stage;
    if (int rrc = ensure_stage_ring(ctx)) return rrc;
    const uint8_t *table[2] = {d_arena, d_arena};  // every page lives in the arena: "file" 0 (and a spare slot)
    size_t si = 0;
    for (size_t c0 = 0; c0 < g.bytes; c0 += StageRing::kBytes) {
        const size_t c1 = std::min(g.bytes, c0 + StageRing::kBytes);
        const int bi = ring.next;
        ring.next = (ring.next + 1) % StageRing::kBufs;
        if (ring.pending[bi]) {
            CUDA_TRY(cudaEventSynchronize(ring.done[bi]));
            ring.pending[bi] = false;
        }
        uint8_t *stage = ring.buf[bi];
        // segments that intersect [c0, c1); a segment cut by the chunk edge is copied in two parts
        while (si < g.segs.size() && g.segs[si].dst + g.segs[si].len <= c0) ++si;
        size_t sj = si;
        while (sj < g.segs.size() && g.segs[sj].dst < c1) ++sj;
        const size_t n = sj - si;
        const size_t tasks = std::max<size_t>(1, std::min<size_t>(32, n / 64));
        std::vector<std::future<void>> futs;
        for (size_t t = 0; t < tasks; ++t) {
            const size_t a = si + n * t / tasks, b = si + n * (t + 1) / tasks;
            auto task = std::make_shared<std::packaged_task<void()>>([&g, &table, stage, c0, c1, a, b] {
                for (size_t k = a; k < b; ++k) {
                    const GatherSeg &sg = g.segs[k];
                    const size_t lo = std::max(sg.dst, c0), hi = std::min(sg.dst + sg.len, c1);
                    if (lo >= hi) continue;
                    const uint8_t *src = sg.src ? sg.src : reinterpret_cast<const uint8_t *>(table);
                    memcpy(stage + (lo - c0), src + (lo - sg.dst), hi - lo);
                }
            });
            futs.push_back(task->get_future());
            if (t + 1 < tasks) ctx->pool.submit([task] { (*task)(); });
            else (*task)();  // the calling thread takes the last share itself
        }
        for (auto &f : futs) f.get();
        // the gaps between pages travel too (they are padding): one contiguous copy per chunk
        CUDA_TRY(cudaMemcpyAsync(d_arena + c0, stage, c1 - c0, cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaEventRecord(ring.done[bi], stream));
        ring.pending[bi] = true;
    }
    return 0;
}

// Cold path, one zero-copy part: the block index is parsed in slices and the scan of slice k runs on the
// GPU (pulling its pages over PCIe) while the host parses slice k+1; the per-slice partial tables are
// combined on the device.  A series may straddle slices: partial tables merge exactly.
// gather = the images are in pageable memory: the touched pages of every slice are collected and staged (see above).
static int scan_agg_host_pipelined(bydb_ctx *ctx, const bydb_part_files *files, const bydb_query *q, bydb_result *out, bool gather = false) {
    constexpr int K = ExecSlot::kMaxBatches;  // most slices (scan launches) per call
    std::unique_lock<std::mutex> ring_lock(ctx->stage.mu, std::defer_lock);
    if (gather) ring_lock.lock();
    SlotLease lease(ctx);
    if (lease.init()) return fail(BYDB_EIO, "cannot create stream");
    ExecSlot &slot = *lease.slot;
    Plan base;
    distinct_fields(q, base.fcols, base.agg_fcol);
    if (base.fcols.size() > kMaxFcols) return fail(BYDB_EINVAL, "too many distinct aggregated fields (max 8)");
    base.n_groups = q->series_group ? q->n_groups : 1;
    base.n_series = q->n_series;
    TableLayout tl(static_cast<size_t>(base.n_groups), base.fcols.size());
    std::vector<FileImage> imgs;
    for (uint32_t i = 0; i < files->n_files; ++i) {
        const bydb_file &f = files->files[i];
        if (!f.name || (!f.data && f.len)) return fail(BYDB_EINVAL, "file without name/data");
        imgs.push_back(FileImage{f.name, f.data, f.len});
    }
    size_t n_primary = 0;
    {
        std::string err;
        const int rc0 = count_primary_blocks(imgs, &n_primary, err);
        if (rc0) return fail(rc0, err);
    }
    Scratch tables;
    tables.stream = slot.stream;
    CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&tables.base), tl.total * K, slot.stream));
    {
        const size_t G = static_cast<size_t>(base.n_groups), A = q->n_aggs, NS = q->n_series;
        const size_t stage_stride = align_up(NS * 12 + (G + 1) * 4 + 256, 256);
        if (slot.ensure_pinned(std::max(stage_stride * K, G * (12 + 16 * A) + 16 * A + 8192))) return fail(BYDB_ENOMEM, "cudaMallocHost failed");
    }
    memset(&out->stats, 0, sizeof out->stats);
    // The block index is parsed in the background from the start, one task per group of primary blocks (they are
    // independent zstd frames).  The main thread takes the pieces in order: whatever is parsed by the time the GPU can
    // take more work becomes the next slice -- first slice = the first piece (shortest wait before the first launch),
    // later slices grow with what the parsers delivered meanwhile, the last allowed slice takes the rest.
    struct Parsed {
        PartDir dir;
        std::string err;
        int rc = 0;
    };
    // pieces of one or two primary blocks: the first piece (= the first slice the GPU can start on) is parsed in well under a
    // millisecond; with 32 pieces it took 4.8 ms of a 45 ms step before anything was launched (traced step, r02n)
    const size_t T = std::max<size_t>(1, std::min<size_t>(n_primary, 128));
    const bool trace = getenv("BYDB_TRACE") != nullptr;  // host-side timeline of the cold path on stderr (read per call: a caller can trace one step)
    const auto t_begin = std::chrono::steady_clock::now();
    auto since = [&] { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_begin).count(); };
    std::vector<std::future<Parsed>> parses;
    for (size_t t = 0; t < T; ++t) {
        auto task = std::make_shared<std::packaged_task<Parsed()>>([ctx, &imgs, t, T] {
            Parsed r;
            r.rc = build_part_dir(imgs, ctx->names, r.dir, r.err, t, T);
            return r;
        });
        parses.push_back(task->get_future());
        ctx->pool.submit([task] { (*task)(); });
    }
    std::vector<std::shared_ptr<Part>> keep;
    std::vector<std::shared_ptr<GatherImage>> gathered;
    int rc = 0, n_slices = 0;
    size_t next = 0;
    while (next < T) {
        std::vector<PartDir> pieces;
        auto take = [&] {
            Parsed pr = parses[next++].get();
            if (pr.rc && !rc) rc = fail(pr.rc, "block index: " + pr.err);
            pieces.push_back(std::move(pr.dir));
        };
        take();
        if (rc || n_slices == K - 1) {
            while (next < T) take();  // the last slice takes the rest; after a failure every task is still joined
        } else {
            while (next < T && parses[next].wait_for(std::chrono::seconds(0)) == std::future_status::ready) take();
        }
        if (rc) break;
        PartDir merged;
        {
            std::string err;
            const int mrc = merge_part_dirs(pieces, merged, err);
            if (mrc) {
                rc = fail(mrc, err);
                continue;
            }
        }
        const int k = n_slices++;
        if (trace) fprintf(stderr, "[bydb cold] slice %d = pieces ..%zu of %zu, parsed at %.0f us (%zu blocks)\n", k, next, T, since(), merged.blocks.size());
        std::shared_ptr<Part> p;
        uint64_t h2d = 0;
        if (gather) {
            auto gi = std::make_shared<GatherImage>();
            rc = plan_gather(ctx, imgs, q, base, merged, *gi);
            if (rc) continue;
            if (gi->blocks.empty() && (next < T || n_slices > 1)) {
                --n_slices;  // nothing of this slice is selected (a query that selects nothing at all still runs one empty slice)
                continue;
            }
            p = std::make_shared<Part>();
            p->id = ~0ull - static_cast<uint64_t>(k);
            p->device = ctx->device;
            p->pool_stream = slot.stream;
            p->hbm_bytes = gi->bytes;
            {
                std::lock_guard<std::mutex> lk(ctx->mu);
                if (ctx->hbm_budget && ctx->hbm_used + gi->bytes > ctx->hbm_budget) {
                    rc = fail(BYDB_ENOMEM, "HBM budget exceeded");
                    continue;
                }
                ctx->hbm_used += gi->bytes;
            }
            if (cudaMallocAsync(reinterpret_cast<void **>(&p->d_arena), gi->bytes, slot.stream) != cudaSuccess) {
                p->d_arena = nullptr;
                std::lock_guard<std::mutex> lk(ctx->mu);
                ctx->hbm_used -= gi->bytes;
                rc = fail(BYDB_ENOMEM, "device allocation failed for the gathered pages");
                continue;
            }
            keep.push_back(p);
            rc = upload_gather(ctx, *gi, p->d_arena, slot.stream);
            if (rc) continue;
            p->d_blocks = reinterpret_cast<const DevBlock *>(p->d_arena);
            p->d_cols = reinterpret_cast<const DevCol *>(p->d_arena + gi->off_cols);
            p->d_files = reinterpret_cast<const uint8_t *const *>(p->d_arena + gi->off_files);
            p->dir.blocks = std::move(gi->blocks);   // only the sizes are read from here on
            p->dir.files = {"arena"};
            p->dir.min_ts = merged.min_ts;
            p->dir.max_ts = merged.max_ts;
            h2d = gi->bytes;
            gathered.push_back(gi);                  // the directory vectors feed the staged copies: keep them until the end
        } else {
            rc = register_part_locked_free(ctx, ~0ull - static_cast<uint64_t>(k), files, p, &h2d, true, true, 0, 1, false, &merged);
            if (rc) continue;
            keep.push_back(p);
        }
        out->stats.h2d_bytes += h2d;
        Plan plan = base;
        plan.parts = {p};
        plan.total_blocks = static_cast<uint32_t>(p->dir.blocks.size());
        rc = run_scan(ctx, q, plan, slot, slot.stream, tables.base + tl.total * static_cast<size_t>(k), tl, &out->stats, k, true);
        if (trace) fprintf(stderr, "[bydb cold] slice %d enqueued at %.0f us\n", k, since());
    }
    while (next < T) (void)parses[next++].get();
    if (!rc && n_slices > 0) {
        launch_combine_tables(reinterpret_cast<uint64_t *>(tables.base), static_cast<uint32_t>(n_slices), tl.total / 8, tl.off_sum_f64 / 8,
                              tl.off_max_f64 / 8, tl.off_max_f64 / 8, tl.off_sum_i64 / 8, tl.off_sum_i64 / 8, tl.off_max_i64 / 8, tl.off_max_i64 / 8,
                              tl.total / 8, slot.stream);
        out->stats.kernel_launches += 1;
        // the pinned staging of the last slices may still be in flight: finalize copies into it only after the kernels
        rc = finalize_to_host(ctx, q, base, slot, slot.stream, tables.base, tl, out);
        if (rc) cudaStreamSynchronize(slot.stream);  // nothing of this call may be in flight when the slot and the parts go back
        if (trace) fprintf(stderr, "[bydb cold] finalized at %.0f us\n", since());
    } else {
        cudaStreamSynchronize(slot.stream);
    }
    for (int k = 0; k < static_cast<int>(keep.size()); ++k) {
        int rc2 = collect_scan(slot, &out->stats, k);
        if (!rc && rc2) {
            bydb_result_free(ctx, out);
            rc = rc2;
        }
    }
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        for (auto &p : keep) ctx->hbm_used -= p->hbm_bytes;
    }
    if (!rc && !gather) out->stats.h2d_bytes += out->stats.page_bytes;  // pages were read in place over PCIe
    return rc;
}

int bydb_scan_agg_host(bydb_ctx *ctx, uint32_t n_parts, const bydb_part_files *parts, const bydb_query *q, bydb_result *out) {
    return guarded([&]() -> int {
    if (!ctx || !out) return fail(BYDB_EINVAL, "ctx/out is NULL");
    memset(out, 0, sizeof *out);
    int rc = validate_query(q, false);
    if (rc) return rc;
    if (n_parts == 0 || !parts || n_parts > kMaxParts) return fail(BYDB_EINVAL, "need 1..64 host parts");
    CUDA_TRY(cudaSetDevice(ctx->device));
    // The cold path first scans the pages as they are; only when a block turns out to hold fallback pages
    // (EncodeTypePlain numeric pages, zstd string blocks) are the parts unpacked on the device and scanned again.
    auto wants_unpack = [](int code) {
        return code == BYDB_ENOTSUP && (g_last_dev_err == kErrPlainPage || g_last_dev_err == kErrZstdDict || g_last_dev_err == kErrTagPlain);
    };
    g_last_dev_err = 0;
    if (n_parts == 1) {
        // pinned by the caller: pages pulled in place over PCIe; pageable: the touched pages gathered and staged
        rc = scan_agg_host_pipelined(ctx, &parts[0], q, out, (q->flags & BYDB_Q_HOST_ZERO_COPY) == 0);
        if (!wants_unpack(rc)) return rc;
    }
    for (int attempt = rc ? 1 : 0; attempt < 2; ++attempt) {
        std::vector<std::shared_ptr<Part>> tmp;
        uint64_t h2d = 0;
        rc = 0;
        g_last_dev_err = 0;
        memset(out, 0, sizeof *out);
        for (uint32_t i = 0; i < n_parts; ++i) {
            std::shared_ptr<Part> p;
            rc = register_part_locked_free(ctx, ~0ull - i, &parts[i], p, &h2d, (q->flags & BYDB_Q_HOST_ZERO_COPY) != 0, true, 0, 1, attempt == 1);
            if (rc) break;
            tmp.push_back(p);
        }
        if (!rc) rc = scan_agg_impl(ctx, q, &tmp, out, h2d);
        if (!rc && (q->flags & BYDB_Q_HOST_ZERO_COPY)) out->stats.h2d_bytes += out->stats.page_bytes;  // pages were read in place over PCIe
        {
            std::lock_guard<std::mutex> lk(ctx->mu);
            for (auto &p : tmp) ctx->hbm_used -= p->hbm_bytes;
        }
        if (!wants_unpack(rc)) break;
    }
    return rc;
    });
}

void bydb_result_free(bydb_ctx *, bydb_result *r) {
    if (!r) return;
    delete static_cast<ResultOwner *>(r->owner);
    memset(r, 0, sizeof *r);
}

int bydb_partials_layout(const bydb_query *q, bydb_partials_layout_t *out) {
    return guarded([&]() -> int {
    if (!q || !out) return fail(BYDB_EINVAL, "NULL argument");
    int rc = validate_query(q, false);
    if (rc) return rc;
    std::vector<std::string> fcols;
    std::vector<int> agg_fcol;
    distinct_fields(q, fcols, agg_fcol);
    TableLayout tl(static_cast<size_t>(q->series_group ? q->n_groups : 1), fcols.size());
    out->total_bytes = tl.total;
    out->off_sum_f64 = tl.off_sum_f64;
    out->n_sum_f64 = tl.GF;
    out->off_max_f64 = tl.off_max_f64;
    out->n_max_f64 = 2 * tl.GF;
    out->off_sum_i64 = tl.off_sum_i64;
    out->n_sum_i64 = 2 * tl.GF + tl.G;
    out->off_max_i64 = tl.off_max_i64;
    out->n_max_i64 = 2 * tl.GF + tl.F;
    return 0;
    });
}

int bydb_scan_partials(bydb_ctx *ctx, const bydb_query *q, void *d_partials, uint64_t bytes, void *stream, bydb_stats *stats) {
    return guarded([&]() -> int {
    if (!ctx || !d_partials) return fail(BYDB_EINVAL, "ctx/d_partials is NULL");
    int rc = validate_query(q, true);
    if (rc) return rc;
    Plan plan;
    rc = make_plan(ctx, q, nullptr, plan);
    if (rc) return rc;
    TableLayout tl(static_cast<size_t>(plan.n_groups), plan.fcols.size());
    if (bytes < tl.total) return fail(BYDB_EINVAL, "partial table buffer too small");
    CUDA_TRY(cudaSetDevice(ctx->device));
    SlotLease lease(ctx);
    if (lease.init()) return fail(BYDB_EIO, "cannot create stream");
    cudaStream_t s = static_cast<cudaStream_t>(stream);  // NULL = the legacy default stream, like every partial-table call
    bydb_stats local;
    memset(&local, 0, sizeof local);
    rc = run_scan(ctx, q, plan, *lease.slot, s, static_cast<uint8_t *>(d_partials), tl, &local);
    if (!rc && !stats) {
        // asynchronous form: nothing is read back here.  A device-side failure travels in the table (coltype words)
        // and surfaces in bydb_reduce_finalize on whichever rank finalises.
        CUDA_TRY(cudaEventRecord(lease.slot->busy, s));
        lease.slot->busy_pending = true;
        return 0;
    }
    if (!rc) {
        CUDA_TRY(cudaStreamSynchronize(s));
        CUDA_TRY(cudaGetLastError());
        rc = collect_scan(*lease.slot, &local);
    }
    if (stats) *stats = local;
    return rc;
    });
}

int bydb_partials_combine(bydb_ctx *ctx, const bydb_query *q, void *d_tables, uint32_t n_tables, uint64_t bytes_each, void *stream) {
    return guarded([&]() -> int {
    if (!ctx || !d_tables || n_tables == 0) return fail(BYDB_EINVAL, "NULL argument");
    int rc = validate_query(q, false);
    if (rc) return rc;
    std::vector<std::string> fcols;
    std::vector<int> agg_fcol;
    distinct_fields(q, fcols, agg_fcol);
    TableLayout tl(static_cast<size_t>(q->series_group ? q->n_groups : 1), fcols.size());
    if (bytes_each != tl.total) return fail(BYDB_EINVAL, "partial tables must be exactly bydb_partials_layout().total_bytes each");
    CUDA_TRY(cudaSetDevice(ctx->device));
    launch_combine_tables(static_cast<uint64_t *>(d_tables), n_tables, tl.total / 8, tl.off_sum_f64 / 8, tl.off_max_f64 / 8, tl.off_max_f64 / 8,
                          tl.off_sum_i64 / 8, tl.off_sum_i64 / 8, tl.off_max_i64 / 8, tl.off_max_i64 / 8, tl.total / 8,
                          static_cast<cudaStream_t>(stream));
    CUDA_TRY(cudaGetLastError());
    return 0;
    });
}

int bydb_reduce_finalize(bydb_ctx *ctx, const bydb_query *q, const void *d_partials, uint64_t bytes, void *stream, bydb_result *out) {
    return guarded([&]() -> int {
    if (!ctx || !d_partials || !out) return fail(BYDB_EINVAL, "NULL argument");
    memset(out, 0, sizeof *out);
    int rc = validate_query(q, false);
    if (rc) return rc;
    Plan plan;
    distinct_fields(q, plan.fcols, plan.agg_fcol);
    plan.n_groups = q->series_group ? q->n_groups : 1;
    TableLayout tl(static_cast<size_t>(plan.n_groups), plan.fcols.size());
    if (bytes < tl.total) return fail(BYDB_EINVAL, "partial table buffer too small");
    CUDA_TRY(cudaSetDevice(ctx->device));
    SlotLease lease(ctx);
    if (lease.init()) return fail(BYDB_EIO, "cannot create stream");
    cudaStream_t s = static_cast<cudaStream_t>(stream);  // NULL = the legacy default stream, like every partial-table call
    return finalize_to_host(ctx, q, plan, *lease.slot, s, static_cast<const uint8_t *>(d_partials), tl, out, true);
    });
}


int bydb_query_prepare(bydb_ctx *ctx, const bydb_query *q, bydb_prepared **out) {
    return guarded([&]() -> int {
    if (!ctx || !out) return fail(BYDB_EINVAL, "ctx/out is NULL");
    *out = nullptr;
    int rc = validate_query(q, true);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    auto p = new bydb_prepared();
    p->parts.assign(q->parts, q->parts + q->n_parts);
    p->sids.assign(q->series_ids, q->series_ids + q->n_series);
    if (q->series_group) p->groups.assign(q->series_group, q->series_group + q->n_series);
    p->aggs.assign(q->aggs, q->aggs + q->n_aggs);
    p->agg_names.resize(q->n_aggs);
    for (uint32_t a = 0; a < q->n_aggs; ++a) p->agg_names[a] = q->aggs[a].field;
    for (uint32_t a = 0; a < q->n_aggs; ++a) p->aggs[a].field = p->agg_names[a].c_str();
    p->preds.assign(q->preds, q->preds + q->n_preds);
    p->pred_family.resize(q->n_preds);
    p->pred_tag.resize(q->n_preds);
    p->pred_lit.resize(q->n_preds);
    for (uint32_t i = 0; i < q->n_preds; ++i) {
        p->pred_family[i] = q->preds[i].family;
        p->pred_tag[i] = q->preds[i].tag;
        if (q->preds[i].lit && q->preds[i].lit_len) p->pred_lit[i].assign(q->preds[i].lit, q->preds[i].lit + q->preds[i].lit_len);
    }
    for (uint32_t i = 0; i < q->n_preds; ++i) {
        p->preds[i].family = p->pred_family[i].c_str();
        p->preds[i].tag = p->pred_tag[i].c_str();
        p->preds[i].lit = p->pred_lit[i].empty() ? nullptr : p->pred_lit[i].data();
    }
    p->q = *q;
    p->q.parts = p->parts.data();
    p->q.series_ids = p->sids.data();
    p->q.series_group = q->series_group ? p->groups.data() : nullptr;
    p->q.aggs = p->aggs.data();
    p->q.preds = p->preds.data();
    // a dedicated slot: stream, events, pinned staging
    p->slot.reset(new ExecSlot());
    bool ok = p->slot->create() == 0;  // with its pinned staging: nothing page-locked is allocated inside an execution
    if (ok) {
        // sized for this query now (see ExecSlot::ensure_pinned: a page-locked allocation inside a collective can stall the peers)
        const size_t G = q->series_group ? static_cast<size_t>(q->n_groups) : 1, A = q->n_aggs, NS = q->n_series;
        ok = p->slot->ensure_pinned(NS * 12 + (G + 1) * 4 + G * (12 + 16 * A) + 16 * A + 16384) == 0;
    }
    ok = ok && cudaEventCreate(&p->t0) == cudaSuccess && cudaEventCreate(&p->t1) == cudaSuccess;
    if (!ok) {
        prepared_destroy(p);
        return fail(BYDB_EIO, "cannot create the stream / events of a prepared query");
    }
    *out = p;
    return 0;
    });
}

void bydb_query_release(bydb_ctx *ctx, bydb_prepared *p) {
    if (ctx) cudaSetDevice(ctx->device);
    prepared_destroy(p);
}

int bydb_scan_agg_prepared(bydb_ctx *ctx, bydb_prepared *p, bydb_result *out) {
    return guarded([&]() -> int {
    if (!ctx || !p || !out) return fail(BYDB_EINVAL, "NULL argument");
    memset(out, 0, sizeof *out);
    std::lock_guard<std::mutex> lk(p->mu);
    g_last_dev_err = 0;
    CUDA_TRY(cudaSetDevice(ctx->device));
    // the first execution runs the ordinary path (it also performs the one-time kernel attribute setup); the second one
    // captures; from then on the graph is replayed
    const uint64_t run = p->runs++;
    if (run == 0 || !p->capturable) return scan_agg_impl(ctx, &p->q, nullptr, out, 0);
    if (!p->exec) {
        const int rc = prepared_capture(ctx, p);
        if (rc) return rc;
        if (!p->exec) return scan_agg_impl(ctx, &p->q, nullptr, out, 0);
    }
    {
        // the graph reads the parts through the device pointers captured with it: every handle must still name the very
        // part object that was captured (a released part makes the call fail like bydb_scan_agg would, a re-registered one
        // drops the graph and captures again)
        std::lock_guard<std::mutex> lk2(ctx->mu);
        bool same = p->held.size() == p->parts.size();
        bool missing = false;
        for (size_t i = 0; i < p->parts.size(); ++i) {
            auto it = ctx->parts.find(p->parts[i]);
            if (it == ctx->parts.end()) missing = true;
            else if (same && it->second != p->held[i]) same = false;
        }
        if (missing || !same) {
            cudaGraphExecDestroy(p->exec);
            p->exec = nullptr;
            p->held.clear();
            if (missing) return fail(BYDB_ENOENT, "unknown part handle");
        }
    }
    if (!p->exec) {
        const int rc = prepared_capture(ctx, p);
        if (rc) return rc;
        if (!p->exec) return scan_agg_impl(ctx, &p->q, nullptr, out, 0);
    }
    ExecSlot &slot = *p->slot;
    CUDA_TRY(cudaEventRecord(p->t0, slot.stream));
    CUDA_TRY(cudaGraphLaunch(p->exec, slot.stream));
    CUDA_TRY(cudaEventRecord(p->t1, slot.stream));
    CUDA_TRY(cudaStreamSynchronize(slot.stream));
    CUDA_TRY(cudaGetLastError());
    out->stats = p->captured;
    const uint32_t *hz = reinterpret_cast<const uint32_t *>(slot.zpage);
    const unsigned long long *hs = reinterpret_cast<const unsigned long long *>(slot.zpage + 16);
    out->stats.rows_scanned = hs[0];
    out->stats.rows_matched = hs[1];
    out->stats.page_bytes = hs[2];
    out->stats.blocks_scanned = hs[3];
    out->stats.blocks_slow_lane = static_cast<uint32_t>(hs[4]);
    out->stats.slow_lane_reasons = static_cast<uint32_t>(hs[5]);
    float ms = 0;
    cudaEventElapsedTime(&ms, p->t0, p->t1);
    out->stats.device_ms = ms;
    out->stats.scan_kernel_ms = 0;  // per-kernel events are not available inside a graph replay
    if (hz[2] != 0) {
        g_last_dev_err = hz[2];
        char buf[96];
        snprintf(buf, sizeof buf, " (block/series #%u)", hz[3]);
        return fail(dev_err_code(hz[2]), std::string(dev_err_text(hz[2])) + buf);
    }
    finalize_parse(slot.pinned + p->host_off, p->fl, out);
    return 0;
    });
}


struct PartialRowsOwner {
    std::vector<int32_t> group_id;
    std::vector<uint8_t> is_float;
    std::vector<int64_t> val_i64, cnt_i64;
    std::vector<double> val_f64, cnt_f64;
};

int bydb_partials_rows(bydb_ctx *ctx, const bydb_query *q, const void *d_partials, uint64_t bytes, void *stream, bydb_partial_rows *out) {
    return guarded([&]() -> int {
    if (!ctx || !d_partials || !out) return fail(BYDB_EINVAL, "NULL argument");
    memset(out, 0, sizeof *out);
    int rc = validate_query(q, false);
    if (rc) return rc;
    std::vector<std::string> fcols;
    std::vector<int> agg_fcol;
    distinct_fields(q, fcols, agg_fcol);
    const size_t G = static_cast<size_t>(q->series_group ? q->n_groups : 1), F = fcols.size(), A = q->n_aggs;
    TableLayout tl(G, F);
    if (bytes < tl.total) return fail(BYDB_EINVAL, "partial table buffer too small");
    CUDA_TRY(cudaSetDevice(ctx->device));
    std::vector<uint8_t> h(tl.total);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CUDA_TRY(cudaMemcpyAsync(h.data(), d_partials, tl.total, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    const double *sum_f = reinterpret_cast<const double *>(h.data() + tl.off_sum_f64), *max_f = reinterpret_cast<const double *>(h.data() + tl.off_max_f64),
                 *negmin_f = reinterpret_cast<const double *>(h.data() + tl.off_negmin_f64);
    const int64_t *sum_i = reinterpret_cast<const int64_t *>(h.data() + tl.off_sum_i64), *cnt = reinterpret_cast<const int64_t *>(h.data() + tl.off_cnt),
                  *rows = reinterpret_cast<const int64_t *>(h.data() + tl.off_rows), *max_i = reinterpret_cast<const int64_t *>(h.data() + tl.off_max_i64),
                  *notmin_i = reinterpret_cast<const int64_t *>(h.data() + tl.off_notmin_i64), *coltype = reinterpret_cast<const int64_t *>(h.data() + tl.off_coltype);
    uint32_t dev_err = 0;
    for (size_t c = 0; c < F; ++c) dev_err = std::max(dev_err, static_cast<uint32_t>(coltype[c] >> 8));
    if (dev_err) return fail(dev_err_code(dev_err), std::string(dev_err_text(dev_err)) + " (status carried in a partial table)");
    auto owner = std::make_unique<PartialRowsOwner>();
    owner->is_float.resize(A);
    for (size_t a = 0; a < A; ++a) owner->is_float[a] = (coltype[agg_fcol[a]] & 0xff) == BYDB_VT_FLOAT64 ? 1 : 0;
    for (size_t g = 0; g < G; ++g) {
        if (rows[g] <= 0) continue;  // the group never appeared on this node
        owner->group_id.push_back(static_cast<int32_t>(g));
        for (size_t a = 0; a < A; ++a) {
            const size_t o = g * F + static_cast<size_t>(agg_fcol[a]);
            const bool isf = owner->is_float[a] != 0;
            const int64_t n = cnt[o];
            int64_t vi = 0, ci = 0;
            double vf = 0.0, cf = 0.0;
            switch (q->aggs[a].func) {
                case BYDB_AGG_SUM: vi = sum_i[o]; vf = sum_f[o]; break;
                case BYDB_AGG_COUNT: vi = n; vf = static_cast<double>(n); break;
                case BYDB_AGG_MAX: vi = n > 0 ? max_i[o] : INT64_MIN; vf = n > 0 ? max_f[o] : -1.7976931348623157e308; break;
                case BYDB_AGG_MIN: vi = n > 0 ? ~notmin_i[o] : INT64_MAX; vf = n > 0 ? -negmin_f[o] : 1.7976931348623157e308; break;
                case BYDB_AGG_MEAN: vi = sum_i[o]; vf = sum_f[o]; ci = n; cf = static_cast<double>(n); break;
            }
            owner->val_i64.push_back(isf ? 0 : vi);
            owner->val_f64.push_back(isf ? vf : 0.0);
            owner->cnt_i64.push_back(isf ? 0 : ci);
            owner->cnt_f64.push_back(isf ? cf : 0.0);
        }
    }
    out->n_rows = static_cast<int32_t>(owner->group_id.size());
    out->n_aggs = static_cast<int32_t>(A);
    out->group_id = owner->group_id.data();
    out->is_float = owner->is_float.data();
    out->val_i64 = owner->val_i64.data();
    out->val_f64 = owner->val_f64.data();
    out->cnt_i64 = owner->cnt_i64.data();
    out->cnt_f64 = owner->cnt_f64.data();
    out->owner = owner.release();
    return 0;
    });
}

void bydb_partial_rows_free(bydb_ctx *, bydb_partial_rows *r) {
    if (!r) return;
    delete static_cast<PartialRowsOwner *>(r->owner);
    memset(r, 0, sizeof *r);
}

// ------------------------------------------------------------------------------------------------
// Multi-GPU reduce behind the C ABI: peer mailboxes over NVLink (see scan_kernels.cu, comm_*_kernel)
// ------------------------------------------------------------------------------------------------
struct CommBlob {  // what travels inside a bydb_comm_handle
    uint32_t magic, device;
    uint64_t pid, raw_ptr, slot_bytes, mailbox_bytes;
    cudaIpcMemHandle_t ipc;
    unsigned char uuid[16];  // the physical GPU (device ordinals differ between processes under CUDA_VISIBLE_DEVICES)
};
static_assert(sizeof(CommBlob) <= sizeof(bydb_comm_handle), "bydb_comm_handle too small");

int bydb_comm_export(bydb_ctx *ctx, uint64_t max_table_bytes, int32_t max_ranks, bydb_comm_handle *out) {
    return guarded([&]() -> int {
    if (!ctx || !out) return fail(BYDB_EINVAL, "ctx/out is NULL");
    if (max_ranks < 1 || max_ranks > kCommMaxRanks) return fail(BYDB_EINVAL, "max_ranks must be 1..64");
    if (max_table_bytes == 0 || max_table_bytes > (1ull << 32)) return fail(BYDB_EINVAL, "bad max_table_bytes");
    CUDA_TRY(cudaSetDevice(ctx->device));
    Comm &cm = ctx->comm;
    std::lock_guard<std::mutex> lk(cm.mu);
    if (cm.mine) return fail(BYDB_EINVAL, "bydb_comm_export was already called on this context");
    cm.slot_bytes = align_up(max_table_bytes, 256);
    cm.mailbox_bytes = kCommCtl + 2 * static_cast<size_t>(max_ranks) * cm.slot_bytes;
    {
        std::lock_guard<std::mutex> lk2(ctx->mu);
        if (ctx->hbm_budget && ctx->hbm_used + cm.mailbox_bytes > ctx->hbm_budget) return fail(BYDB_ENOMEM, "HBM budget exceeded (mailbox)");
        ctx->hbm_used += cm.mailbox_bytes;
    }
    if (cudaMalloc(reinterpret_cast<void **>(&cm.mine), cm.mailbox_bytes) != cudaSuccess) {
        cm.mine = nullptr;
        return fail(BYDB_ENOMEM, "device allocation failed for the mailbox");
    }
    CUDA_TRY(cudaMemset(cm.mine, 0, cm.mailbox_bytes));
    CommBlob b;
    memset(&b, 0, sizeof b);
    b.magic = 0xB1DBC011u;
    b.device = static_cast<uint32_t>(ctx->device);
    b.pid = static_cast<uint64_t>(getpid());
    b.raw_ptr = reinterpret_cast<uint64_t>(cm.mine);
    b.slot_bytes = cm.slot_bytes;
    b.mailbox_bytes = cm.mailbox_bytes;
    CUDA_TRY(cudaIpcGetMemHandle(&b.ipc, cm.mine));
    {
        cudaDeviceProp prop;
        CUDA_TRY(cudaGetDeviceProperties(&prop, ctx->device));
        static_assert(sizeof prop.uuid.bytes == sizeof b.uuid, "uuid size");
        memcpy(b.uuid, prop.uuid.bytes, sizeof b.uuid);
    }
    memset(out, 0, sizeof *out);
    memcpy(out, &b, sizeof b);
    return 0;
    });
}

int bydb_comm_connect(bydb_ctx *ctx, int32_t rank, int32_t nranks, const bydb_comm_handle *all) {
    return guarded([&]() -> int {
    if (!ctx || !all) return fail(BYDB_EINVAL, "ctx/handles is NULL");
    if (nranks < 1 || nranks > kCommMaxRanks || rank < 0 || rank >= nranks) return fail(BYDB_EINVAL, "bad rank / nranks");
    CUDA_TRY(cudaSetDevice(ctx->device));
    Comm &cm = ctx->comm;
    std::lock_guard<std::mutex> lk(cm.mu);
    if (!cm.mine) return fail(BYDB_EINVAL, "call bydb_comm_export first");
    if (cm.nranks) return fail(BYDB_EINVAL, "bydb_comm_connect was already called on this context");
    std::vector<uint8_t *> peer(static_cast<size_t>(nranks), nullptr);
    std::vector<bool> opened(static_cast<size_t>(nranks), false);
    std::vector<size_t> slots(static_cast<size_t>(nranks), 0);
    bool shares_device = false;  // another rank lives on this GPU (tests, a box with fewer GPUs than ranks)
    unsigned char my_uuid[16];
    {
        cudaDeviceProp prop;
        CUDA_TRY(cudaGetDeviceProperties(&prop, ctx->device));
        memcpy(my_uuid, prop.uuid.bytes, sizeof my_uuid);
    }
    for (int r = 0; r < nranks; ++r) {
        CommBlob b;
        memcpy(&b, &all[r], sizeof b);
        if (b.magic != 0xB1DBC011u) return fail(BYDB_EINVAL, "handle of rank " + std::to_string(r) + " is not a bydb_comm_handle");
        if (kCommCtl + 2 * static_cast<uint64_t>(nranks) * b.slot_bytes > b.mailbox_bytes)
            return fail(BYDB_EINVAL, "mailbox of rank " + std::to_string(r) + " was exported for fewer ranks");
        slots[r] = b.slot_bytes;
        if (r != rank && memcmp(b.uuid, my_uuid, sizeof my_uuid) == 0) shares_device = true;
        if (r == rank) {
            if (b.raw_ptr != reinterpret_cast<uint64_t>(cm.mine)) return fail(BYDB_EINVAL, "handles[rank] is not this context's own handle");
            peer[r] = cm.mine;
        } else if (b.pid == static_cast<uint64_t>(getpid())) {
            // same process (several contexts, one per GPU, or tests): the pointer is valid as it is once peer access is on
            if (static_cast<int>(b.device) != ctx->device) {
                int can = 0;
                cudaDeviceCanAccessPeer(&can, ctx->device, static_cast<int>(b.device));
                if (!can) return fail(BYDB_ENOTSUP, "no peer access between device " + std::to_string(ctx->device) + " and " + std::to_string(b.device));
                const cudaError_t e = cudaDeviceEnablePeerAccess(static_cast<int>(b.device), 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(BYDB_EIO, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
                cudaGetLastError();
            }
            peer[r] = reinterpret_cast<uint8_t *>(b.raw_ptr);
        } else {
            void *p = nullptr;
            const cudaError_t e = cudaIpcOpenMemHandle(&p, b.ipc, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) {
                for (int k = 0; k < r; ++k)
                    if (opened[k]) cudaIpcCloseMemHandle(peer[k]);
                return fail(BYDB_EIO, std::string("cudaIpcOpenMemHandle (rank ") + std::to_string(r) + "): " + cudaGetErrorString(e));
            }
            peer[r] = static_cast<uint8_t *>(p);
            opened[r] = true;
        }
    }
    cm.peer = std::move(peer);
    cm.ipc_opened = std::move(opened);
    cm.peer_slot_bytes = std::move(slots);
    cm.rank = rank;
    cm.nranks = nranks;
    cm.epoch = 0;
    cm.last_use.assign(2 * static_cast<size_t>(nranks), 0);
    // ranks that share a device must not make page-locked allocations inside a collective (ExecSlot::ensure_pinned): the
    // staging ring of the pageable cold path is made now
    if (shares_device && ensure_stage_ring(ctx) != 0) g_last_error.clear();
    if (shares_device) {
        // host-polled waits (see Comm::shared_device): the polling stream and its pinned words are made now
        if (cudaStreamCreateWithFlags(&cm.poll_stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaMallocHost(reinterpret_cast<void **>(&cm.poll_buf), sizeof(unsigned long long) * kCommMaxRanks) != cudaSuccess)
            return fail(BYDB_EIO, "cannot create the polling stream of a shared-device collective");
        cm.shared_device = true;
    }
    return 0;
    });
}

// given: the parts to scan instead of q->parts (the host-buffer form); pre_rc: a failure that already happened on this
// rank (its transient parts could not be admitted) -- the rank still takes part in the collective and reports it
// Host-side form of comm_wait_kernel for ranks that share a device (Comm::shared_device): polls n words until all have reached
// `epoch`; bounded like the kernel (60 s).  Returns 0 or kErrPeerTimeout.
static uint32_t comm_wait_host(Comm &cm, const unsigned long long *dev_words, uint32_t n, unsigned long long epoch) {
    const auto t0 = std::chrono::steady_clock::now();
    for (uint32_t spins = 0;; ++spins) {
        if (cudaMemcpyAsync(cm.poll_buf, dev_words, sizeof(unsigned long long) * n, cudaMemcpyDeviceToHost, cm.poll_stream) != cudaSuccess ||
            cudaStreamSynchronize(cm.poll_stream) != cudaSuccess) {
            cudaGetLastError();
            return kErrPeerTimeout;
        }
        bool all = true;
        for (uint32_t i = 0; i < n; ++i) all = all && cm.poll_buf[i] >= epoch;
        if (all) return 0;
        if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(60)) return kErrPeerTimeout;
        if (spins > 64) std::this_thread::sleep_for(std::chrono::microseconds(20));
        else std::this_thread::yield();
    }
}

static int scan_reduce_impl(bydb_ctx *ctx, const bydb_query *q, const std::vector<std::shared_ptr<Part>> *given, int pre_rc, uint64_t h2d_pre, int32_t root,
                            bydb_result *out) {
    {
    const std::string pre_msg = pre_rc ? g_last_error : std::string();
    Comm &cm = ctx->comm;
    std::lock_guard<std::mutex> lk(cm.mu);
    if (cm.nranks == 0) return fail(BYDB_EINVAL, "bydb_comm_connect was not called on this context");
    if (root < 0 || root >= cm.nranks) return fail(BYDB_EINVAL, "bad root");
    CUDA_TRY(cudaSetDevice(ctx->device));
    SlotLease lease(ctx);
    if (lease.init()) return fail(BYDB_EIO, "cannot create stream");
    ExecSlot &es = *lease.slot;
    cudaStream_t s = es.stream;
    // From here on this rank ALWAYS raises its arrival flag (with a status word in front of it), whatever fails on the
    // host side: the other ranks' calls must neither hang nor fall out of step (every rank counts the same epochs).
    const uint64_t epoch = ++cm.epoch;
    const size_t parity = static_cast<size_t>(epoch & 1u);
    const size_t slot = cm.peer_slot_bytes[static_cast<size_t>(root)];
    uint8_t *root_mb = cm.peer[static_cast<size_t>(root)];
    uint8_t *slots0 = root_mb + kCommCtl + parity * static_cast<size_t>(cm.nranks) * slot;
    uint8_t *my_slot = slots0 + static_cast<size_t>(cm.rank) * slot;
    unsigned long long *flags = reinterpret_cast<unsigned long long *>(root_mb);
    unsigned long long *status = reinterpret_cast<unsigned long long *>(root_mb + kCommStatusOff);
    unsigned long long *done = reinterpret_cast<unsigned long long *>(root_mb + kCommDoneOff);
    uint32_t *my_err = reinterpret_cast<uint32_t *>(cm.mine + kCommErrOff);
    Plan plan;
    int rc = pre_rc ? fail(pre_rc, pre_msg) : validate_query(q, given == nullptr);
    if (!rc) rc = make_plan(ctx, q, given, plan);
    TableLayout tl(static_cast<size_t>(rc ? 1 : plan.n_groups), rc ? 1 : plan.fcols.size());
    if (!rc && tl.total > slot) rc = fail(BYDB_EINVAL, "partial table larger than the mailbox slots (bydb_comm_export max_table_bytes)");
    if (!rc) {
        const size_t G = static_cast<size_t>(plan.n_groups), A = q->n_aggs, NS = q->n_series;
        if (es.ensure_pinned(NS * 12 + (G + 1) * 4 + G * (12 + 16 * A) + 16 * A + 8192)) rc = fail(BYDB_ENOMEM, "cudaMallocHost failed");
    }
    memset(&out->stats, 0, sizeof out->stats);
    out->stats.h2d_bytes = h2d_pre;
    // the slots' previous use -- the last collective with THIS root and parity, the same epoch on every rank -- must have been
    // consumed by the root (its `done` word only ever grows) before they are overwritten
    const uint64_t prev_use = cm.last_use[2 * static_cast<size_t>(root) + parity];
    cm.last_use[2 * static_cast<size_t>(root) + parity] = epoch;
    uint32_t host_perr = 0;  // outcome of the host-polled waits (shared-device mode)
    if (prev_use) {
        if (cm.shared_device) host_perr = comm_wait_host(cm, done, 1, prev_use);
        else launch_comm_wait(done, 1, prev_use, my_err, kErrPeerTimeout, s);
    }
    // map: this rank's group_reduce writes the table straight into the root's memory (P2P stores over NVLink)
    if (!rc) rc = run_scan(ctx, q, plan, es, s, my_slot, tl, &out->stats);
    const std::string my_msg = rc ? g_last_error : std::string();
    const unsigned long long st_word = (epoch << 32) | static_cast<unsigned long long>(static_cast<uint32_t>(-rc));
    cudaMemcpyAsync(status + cm.rank, &st_word, sizeof st_word, cudaMemcpyHostToDevice, s);  // pageable source: staged before the call returns
    launch_comm_signal(flags + cm.rank, epoch, s);
    unsigned long long peer_status[kCommMaxRanks] = {0};
    bool finalized = false;
    int frc = 0;
    if (cm.rank == root) {
        // reduce: wait for every rank's table, combine in rank order (deterministic float sums), finalise
        if (cm.shared_device) {
            const uint32_t e2 = comm_wait_host(cm, flags, static_cast<uint32_t>(cm.nranks), epoch);  // own flag included: own table is complete
            host_perr = host_perr ? host_perr : e2;
        } else {
            launch_comm_wait(flags, static_cast<uint32_t>(cm.nranks), epoch, my_err, kErrPeerTimeout, s);
        }
        if (!rc) {
            launch_combine_tables(reinterpret_cast<uint64_t *>(slots0), static_cast<uint32_t>(cm.nranks), tl.total / 8, tl.off_sum_f64 / 8, tl.off_max_f64 / 8,
                                  tl.off_max_f64 / 8, tl.off_sum_i64 / 8, tl.off_sum_i64 / 8, tl.off_max_i64 / 8, tl.off_max_i64 / 8, tl.total / 8, s,
                                  slot / 8);
            out->stats.kernel_launches += 3;
            frc = finalize_to_host(ctx, q, plan, es, s, slots0, tl, out, true);  // synchronises
            finalized = frc == 0;
        }
        cudaStreamSynchronize(s);
        cudaMemcpy(peer_status, status, sizeof(unsigned long long) * static_cast<size_t>(cm.nranks), cudaMemcpyDeviceToHost);
        // the slots of this parity are free again: nothing reads them any more
        cudaMemcpyAsync(done, &epoch, sizeof epoch, cudaMemcpyHostToDevice, s);
    }
    cudaStreamSynchronize(s);
    uint32_t perr = 0;
    if (cudaMemcpy(&perr, my_err, sizeof perr, cudaMemcpyDeviceToHost) == cudaSuccess && perr != 0) cudaMemset(my_err, 0, sizeof perr);
    if (!perr) perr = host_perr;
    // ---- outcome, most specific first: this rank's own host-side failure, its device-side scan error, a peer's failure
    if (rc) {
        if (finalized) bydb_result_free(ctx, out);
        return fail(rc, my_msg);
    }
    int crc = collect_scan(es, &out->stats);
    if (!crc && perr) crc = fail(dev_err_code(perr), dev_err_text(perr));
    if (!crc && cm.rank == root) {
        for (int r = 0; r < cm.nranks && !crc; ++r) {
            const unsigned long long w = peer_status[r];
            if ((w >> 32) == (epoch & 0xffffffffull) && static_cast<uint32_t>(w) != 0)
                crc = fail(-static_cast<int>(static_cast<uint32_t>(w)), "multi-GPU reduce: rank " + std::to_string(r) + " failed before its scan");
        }
        if (!crc) crc = frc;
    }
    if (crc && finalized) bydb_result_free(ctx, out);
    return crc;
    }
}

int bydb_scan_reduce(bydb_ctx *ctx, const bydb_query *q, int32_t root, bydb_result *out) {
    return guarded([&]() -> int {
    if (!ctx || !out) return fail(BYDB_EINVAL, "ctx/out is NULL");
    memset(out, 0, sizeof *out);
    return scan_reduce_impl(ctx, q, nullptr, 0, 0, root, out);
    });
}

// ------------------------------------------------------------------------------------------------
// Keyed collective (bydb_scan_reduce_keyed): group-by on a stored tag over the peer mailboxes.  Each rank finds its own
// distinct key values and runs one pass per value with its composite table landing straight in its slot of the root's
// mailbox; the root unites the dictionaries, folds the slices through the remap and restores the single-context insertion
// order (see "Keyed collective" in scan_kernels.cu).
// ------------------------------------------------------------------------------------------------
namespace {
// One rank's slot, every piece 256-byte aligned:
//   u32 V_r | u32 lens[cap] | bytes[cap x kMaxLit] (the rank's dictionary) | first appearance of composite group (v, g):
//   u64 sid[cap x G], i64 Kts[cap x G], u32 Krow[cap x G] | i64 pass column types[cap x F] | composite table TableLayout(cap x G, F),
//   value-major (slice v = groups v*G .. v*G + G - 1; only the first V_r slices are written)
struct KeyedSlotLayout {
    TableLayout tl;
    size_t off_nv = 0, off_lens = 0, off_vals = 0, off_fsid = 0, off_fts = 0, off_frow = 0, off_ct = 0, off_table = 0, total = 0;
    KeyedSlotLayout(size_t cap, size_t G, size_t F) : tl(cap * G, F) {
        auto carve = [&](size_t bytes) {
            const size_t at = total;
            total = align_up(total + bytes, 256);
            return at;
        };
        off_nv = carve(16);
        off_lens = carve(cap * 4);
        off_vals = carve(cap * kMaxLit);
        off_fsid = carve(cap * G * 8);
        off_fts = carve(cap * G * 8);
        off_frow = carve(cap * G * 4);
        off_ct = carve(cap * F * 8);
        off_table = carve(tl.total);
    }
};
}  // namespace

int bydb_keyed_reduce_layout(const bydb_query *q, const bydb_group_key *key, uint64_t *slot_bytes) {
    return guarded([&]() -> int {
    if (!slot_bytes) return fail(BYDB_EINVAL, "slot_bytes is NULL");
    int rc = validate_query(q, false);
    if (rc) return rc;
    if (!key || !key->family || !key->tag) return fail(BYDB_EINVAL, "group key without family/tag");
    const uint32_t cap = key->max_values ? key->max_values : 64u;
    if (cap > kMaxKeyValues) return fail(BYDB_EINVAL, "bydb_group_key.max_values above 256");
    std::vector<std::string> fcols;
    std::vector<int> agg_fcol;
    distinct_fields(q, fcols, agg_fcol);
    if (fcols.size() > kMaxFcols) return fail(BYDB_EINVAL, "too many distinct aggregated fields (max 8)");
    const size_t G = q->series_group ? static_cast<size_t>(q->n_groups) : 1;
    *slot_bytes = KeyedSlotLayout(cap, G, fcols.size()).total;
    return 0;
    });
}

int bydb_scan_reduce_keyed(bydb_ctx *ctx, const bydb_query *q, const bydb_group_key *key, int32_t root, bydb_keyed_result *out) {
    return guarded([&]() -> int {
    if (!ctx || !out) return fail(BYDB_EINVAL, "ctx/out is NULL");
    memset(out, 0, sizeof *out);
    Comm &cm = ctx->comm;
    std::lock_guard<std::mutex> lk(cm.mu);
    if (cm.nranks == 0) return fail(BYDB_EINVAL, "bydb_comm_connect was not called on this context");
    if (root < 0 || root >= cm.nranks) return fail(BYDB_EINVAL, "bad root");
    CUDA_TRY(cudaSetDevice(ctx->device));
    g_last_dev_err = 0;
    SlotLease lease(ctx);
    if (lease.init()) return fail(BYDB_EIO, "cannot create stream");
    ExecSlot &es = *lease.slot;
    cudaStream_t s = es.stream;
    // From here on this rank ALWAYS raises its arrival flag with a status word in front of it (scan_reduce_impl's protocol): a
    // failure on any rank reaches the root through the status words, and every rank counts the same epochs.
    const uint64_t epoch = ++cm.epoch;
    const size_t parity = static_cast<size_t>(epoch & 1u);
    const size_t slot = cm.peer_slot_bytes[static_cast<size_t>(root)];
    uint8_t *root_mb = cm.peer[static_cast<size_t>(root)];
    uint8_t *slots0 = root_mb + kCommCtl + parity * static_cast<size_t>(cm.nranks) * slot;
    uint8_t *my_slot = slots0 + static_cast<size_t>(cm.rank) * slot;
    unsigned long long *flags = reinterpret_cast<unsigned long long *>(root_mb);
    unsigned long long *status = reinterpret_cast<unsigned long long *>(root_mb + kCommStatusOff);
    unsigned long long *done = reinterpret_cast<unsigned long long *>(root_mb + kCommDoneOff);
    uint32_t *my_err = reinterpret_cast<uint32_t *>(cm.mine + kCommErrOff);
    Plan plan;
    uint32_t cap = 64;
    int rc = keyed_prepare(ctx, q, key, plan, cap);
    const size_t G = rc ? 1 : static_cast<size_t>(plan.n_groups), F = rc ? 1 : plan.fcols.size(), NS = rc ? 0 : q->n_series, A = rc ? 1 : q->n_aggs;
    const KeyedSlotLayout kl(cap, G, F);
    if (!rc && kl.total > slot) rc = fail(BYDB_EINVAL, "group-key table larger than the mailbox slots (size them with bydb_keyed_reduce_layout)");
    if (!rc && cap * G > 0x7fffffffull / F) rc = fail(BYDB_ENOMEM, "group-key query: too many composite groups");
    // the staging at its largest (the root's finalisation of up to cap x G groups) before any wait can spin (ExecSlot::ensure_pinned)
    if (!rc && es.ensure_pinned(std::max(NS * 12 + (G + 1) * 4 + cap * G * (12 + 16 * A) + 16 * A + 8192, cap * (kMaxLit + 4) + NS * 8 + 4096)))
        rc = fail(BYDB_ENOMEM, "cudaMallocHost failed");
    memset(&out->base.stats, 0, sizeof out->base.stats);
    bydb_stats &st = out->base.stats;
    // the slots' previous use must have been consumed by the root before this rank writes into them
    const uint64_t prev_use = cm.last_use[2 * static_cast<size_t>(root) + parity];
    cm.last_use[2 * static_cast<size_t>(root) + parity] = epoch;
    uint32_t host_perr = 0;
    if (prev_use) {
        if (cm.shared_device) host_perr = comm_wait_host(cm, done, 1, prev_use);
        else launch_comm_wait(done, 1, prev_use, my_err, kErrPeerTimeout, s);
    }
    // map: distinct values, one pass per value into this rank's slot, the dictionary and the first appearances next to it
    KeyValues kv;
    Scratch kb, kc;
    if (!rc) rc = [&]() -> int {
        int r2 = keyed_values(ctx, q, key, cap, plan, es, &st, kv);
        if (r2) return r2;
        const size_t V = kv.values.size();
        KeyFirstParams kf;
        memset(&kf, 0, sizeof kf);
        if (V) {
            const size_t kts_bytes = align_up(V * NS * 8, 256);
            kb.stream = s;
            CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&kb.base), kts_bytes + V * NS * 4 + 256, s));
            int64_t *kts = reinterpret_cast<int64_t *>(kb.base);
            uint32_t *krow = reinterpret_cast<uint32_t *>(kb.base + kts_bytes);
            CUDA_TRY(cudaMemsetAsync(my_slot + kl.off_ct, 0, V * F * 8, s));
            r2 = keyed_passes(ctx, q, key, plan, es, kv, my_slot + kl.off_table, kl.tl, reinterpret_cast<int64_t *>(my_slot + kl.off_ct), kts, krow, &st);
            if (r2) return r2;
            r2 = upload_group_order(q, G, es, kc, &kf.order, &kf.group_start);
            if (r2) return r2;
            kf.Kts = kts;
            kf.Krow = krow;
        }
        CUDA_TRY(cudaMemcpyAsync(my_slot + kl.off_lens, kv.d_lens, static_cast<size_t>(cap) * 4, cudaMemcpyDeviceToDevice, s));
        CUDA_TRY(cudaMemcpyAsync(my_slot + kl.off_vals, kv.d_vals, static_cast<size_t>(cap) * kMaxLit, cudaMemcpyDeviceToDevice, s));
        kf.n_groups = static_cast<int32_t>(G);
        kf.n_values = static_cast<uint32_t>(V);
        kf.q_sids = kv.d_sids;
        kf.n_series = static_cast<uint32_t>(NS);
        kf.n_values_out = reinterpret_cast<uint32_t *>(my_slot + kl.off_nv);
        kf.first_sid = reinterpret_cast<uint64_t *>(my_slot + kl.off_fsid);
        kf.first_ts = reinterpret_cast<int64_t *>(my_slot + kl.off_fts);
        kf.first_row = reinterpret_cast<uint32_t *>(my_slot + kl.off_frow);
        launch_key_first(kf, s);
        st.kernel_launches += 1;
        return 0;
    }();
    const std::string my_msg = rc ? g_last_error : std::string();
    const unsigned long long st_word = (epoch << 32) | static_cast<unsigned long long>(static_cast<uint32_t>(-rc));
    cudaMemcpyAsync(status + cm.rank, &st_word, sizeof st_word, cudaMemcpyHostToDevice, s);  // pageable source: staged before the call returns
    launch_comm_signal(flags + cm.rank, epoch, s);
    unsigned long long peer_status[kCommMaxRanks] = {0};
    int frc = 0;
    if (cm.rank == root) {
        if (cm.shared_device) {
            const uint32_t e2 = comm_wait_host(cm, flags, static_cast<uint32_t>(cm.nranks), epoch);
            host_perr = host_perr ? host_perr : e2;
        } else {
            launch_comm_wait(flags, static_cast<uint32_t>(cm.nranks), epoch, my_err, kErrPeerTimeout, s);
        }
        cudaStreamSynchronize(s);
        cudaMemcpy(peer_status, status, sizeof(unsigned long long) * static_cast<size_t>(cm.nranks), cudaMemcpyDeviceToHost);
        uint32_t werr = 0;
        cudaMemcpy(&werr, my_err, sizeof werr, cudaMemcpyDeviceToHost);
        // reduce only over slots that every rank filled: a failed rank's slot holds nothing of this epoch
        bool all_ok = !rc && !host_perr && !werr;
        for (int r = 0; r < cm.nranks && all_ok; ++r)
            all_ok = !((peer_status[r] >> 32) == (epoch & 0xffffffffull) && static_cast<uint32_t>(peer_status[r]) != 0);
        if (all_ok) frc = [&]() -> int {
            // 1. key union over the ranks' dictionaries
            const size_t R = static_cast<size_t>(cm.nranks), n = R * cap;
            size_t hash_slots = 64;
            while (hash_slots < 2 * n) hash_slots <<= 1;
            size_t o = 0;
            auto carve = [&](size_t bytes) {
                const size_t at = o;
                o = align_up(o + bytes, 256);
                return at;
            };
            const size_t u_hash = carve(hash_slots * 4), u_rep = carve(n * 4), u_remap = carve(n * 4), u_inv = carve(n * 4), u_ctl = carve(16),
                         u_lens = carve(static_cast<size_t>(cap) * 4), u_vals = carve(static_cast<size_t>(cap) * kMaxLit);
            Scratch ua;
            ua.stream = s;
            CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&ua.base), o, s));
            CUDA_TRY(cudaMemsetAsync(ua.base + u_hash, 0, hash_slots * 4, s));
            CUDA_TRY(cudaMemsetAsync(ua.base + u_remap, 0xff, u_ctl - u_remap, s));
            CUDA_TRY(cudaMemsetAsync(ua.base + u_ctl, 0, o - u_ctl, s));
            KeyUnionParams up;
            memset(&up, 0, sizeof up);
            up.n_ranks = static_cast<uint32_t>(R);
            up.cap = cap;
            up.slots = slots0;
            up.slot_bytes = slot;
            up.off_nv = kl.off_nv;
            up.off_lens = kl.off_lens;
            up.off_vals = kl.off_vals;
            up.hash = reinterpret_cast<uint32_t *>(ua.base + u_hash);
            up.hash_slots = static_cast<uint32_t>(hash_slots);
            up.rep = reinterpret_cast<int32_t *>(ua.base + u_rep);
            up.remap = reinterpret_cast<int32_t *>(ua.base + u_remap);
            up.inv = reinterpret_cast<int32_t *>(ua.base + u_inv);
            up.ctl = reinterpret_cast<uint32_t *>(ua.base + u_ctl);
            up.g_lens = reinterpret_cast<uint32_t *>(ua.base + u_lens);
            up.g_vals = ua.base + u_vals;
            launch_key_union(up, s);
            const size_t back = o - u_ctl;  // ctl | lens | vals
            CUDA_TRY(cudaMemcpyAsync(es.pinned, ua.base + u_ctl, back, cudaMemcpyDeviceToHost, s));
            CUDA_TRY(cudaStreamSynchronize(s));
            CUDA_TRY(cudaGetLastError());
            st.kernel_launches += 1;
            st.d2h_bytes += back;
            const uint32_t *ctl = reinterpret_cast<const uint32_t *>(es.pinned);
            if (ctl[1] != 0) {
                g_last_dev_err = ctl[1];
                return fail(dev_err_code(ctl[1]), std::string(dev_err_text(ctl[1])) + " (the union of the ranks' values)");
            }
            const size_t Vg = ctl[0];
            auto owner = new KeyedOwner();
            out->owner = owner;
            owner->key_off.push_back(0);
            const uint32_t *hl = reinterpret_cast<const uint32_t *>(es.pinned + (u_lens - u_ctl));
            const uint8_t *hv = es.pinned + (u_vals - u_ctl);
            for (size_t v = 0; v < Vg; ++v) {
                owner->key_bytes.insert(owner->key_bytes.end(), hv + v * kMaxLit, hv + v * kMaxLit + hl[v]);
                owner->key_off.push_back(static_cast<uint32_t>(owner->key_bytes.size()));
            }
            if (owner->key_bytes.empty()) owner->key_bytes.push_back(0);
            out->n_keys = static_cast<int32_t>(Vg);
            out->key_off = owner->key_off.data();
            out->key_bytes = owner->key_bytes.data();
            if (Vg == 0) return 0;  // no rank selected a block: no rows
            // 2. keyed combine, 3. order, then the single-context tail: permute, finalise, rows back to (series group, key)
            const size_t GP = Vg * G;
            const TableLayout tlc(GP, F);
            o = 0;
            const size_t c_comb = carve(tlc.total), c_dst = carve(tlc.total), c_ct = carve(Vg * F * 8), c_fsid = carve(GP * 8), c_fts = carve(GP * 8),
                         c_frow = carve(GP * 4), c_perm = carve(GP * 4);
            size_t sort_bytes = 0;
            if (launch_key_rank(nullptr, nullptr, nullptr, nullptr, static_cast<uint32_t>(GP), nullptr, &sort_bytes, s))
                return fail(BYDB_EIO, "cannot size the device sort of the composite groups");
            const size_t c_sort = carve(sort_bytes);
            Scratch ub;
            ub.stream = s;
            CUDA_TRY(cudaMallocAsync(reinterpret_cast<void **>(&ub.base), o, s));
            KeyCombineParams cp;
            memset(&cp, 0, sizeof cp);
            cp.n_ranks = static_cast<uint32_t>(R);
            cp.cap = cap;
            cp.n_values = static_cast<uint32_t>(Vg);
            cp.n_fcols = static_cast<uint32_t>(F);
            cp.n_groups = static_cast<int32_t>(G);
            cp.slot_bytes = slot;
            cp.src = table_ptrs(slots0 + kl.off_table, kl.tl);
            cp.src_ct = reinterpret_cast<const int64_t *>(slots0 + kl.off_ct);
            cp.src_fsid = reinterpret_cast<const uint64_t *>(slots0 + kl.off_fsid);
            cp.src_fts = reinterpret_cast<const int64_t *>(slots0 + kl.off_fts);
            cp.src_frow = reinterpret_cast<const uint32_t *>(slots0 + kl.off_frow);
            cp.inv = up.inv;
            cp.dst = table_ptrs(ub.base + c_comb, tlc);
            cp.dst_ct = reinterpret_cast<int64_t *>(ub.base + c_ct);
            cp.fsid = reinterpret_cast<uint64_t *>(ub.base + c_fsid);
            cp.fts = reinterpret_cast<int64_t *>(ub.base + c_fts);
            cp.frow = reinterpret_cast<uint32_t *>(ub.base + c_frow);
            launch_key_combine(cp, s);
            int32_t *d_perm = reinterpret_cast<int32_t *>(ub.base + c_perm);
            if (launch_key_rank(cp.fsid, cp.fts, cp.frow, d_perm, static_cast<uint32_t>(GP), ub.base + c_sort, &sort_bytes, s))
                return fail(BYDB_EIO, "device sort of the composite groups failed");
            launch_permute_table(table_ptrs(ub.base + c_dst, tlc), cp.dst, d_perm, static_cast<uint32_t>(GP), static_cast<uint32_t>(F), cp.dst_ct,
                                 static_cast<uint32_t>(Vg), s);
            st.kernel_launches += 4;  // combine, iota, the merge sort (counted once), permute
            Plan planc = plan;
            planc.n_groups = static_cast<int32_t>(GP);
            int r2 = finalize_to_host(ctx, q, planc, es, s, ub.base + c_dst, tlc, &out->base, true);
            if (r2) return r2;
            std::vector<int32_t> perm(GP);
            CUDA_TRY(cudaMemcpyAsync(perm.data(), d_perm, GP * 4, cudaMemcpyDeviceToHost, s));
            CUDA_TRY(cudaStreamSynchronize(s));
            st.d2h_bytes += GP * 4;
            keyed_split_rows(out, perm, G);
            return 0;
        }();
        cudaStreamSynchronize(s);
        // the slots of this parity are free again: nothing reads them any more
        cudaMemcpyAsync(done, &epoch, sizeof epoch, cudaMemcpyHostToDevice, s);
    }
    cudaStreamSynchronize(s);
    uint32_t perr = 0;
    if (cudaMemcpy(&perr, my_err, sizeof perr, cudaMemcpyDeviceToHost) == cudaSuccess && perr != 0) cudaMemset(my_err, 0, sizeof perr);
    if (!perr) perr = host_perr;
    // ---- outcome, most specific first: this rank's own failure, a failed wait, a peer's failure, the root's reduce
    int crc = rc ? fail(rc, my_msg) : perr ? fail(dev_err_code(perr), dev_err_text(perr)) : 0;
    if (!crc && cm.rank == root) {
        for (int r = 0; r < cm.nranks && !crc; ++r) {
            const unsigned long long w = peer_status[r];
            if ((w >> 32) == (epoch & 0xffffffffull) && static_cast<uint32_t>(w) != 0)
                crc = fail(-static_cast<int>(static_cast<uint32_t>(w)), "multi-GPU keyed reduce: rank " + std::to_string(r) + " failed");
        }
        if (!crc) crc = frc;
    }
    if (crc) bydb_keyed_result_free(ctx, out);
    return crc;
    });
}

// The collective as a prepared query: from its second execution on (per root and slot parity) the rank's whole step -- argument
// refresh, wait for the slots, staging copy, block selection, scan, reduce into the root's mailbox, status + arrival flag, and on
// the root the wait for all ranks, combine, finalisation, row selection, `done` word and read-back -- is ONE captured CUDA graph:
// one launch and one synchronisation per call.  Semantics are bydb_scan_reduce's; ranks may mix the two freely.
int bydb_scan_reduce_prepared(bydb_ctx *ctx, bydb_prepared *p, int32_t root, bydb_result *out) {
    return guarded([&]() -> int {
    if (!ctx || !p || !out) return fail(BYDB_EINVAL, "NULL argument");
    memset(out, 0, sizeof *out);
    std::lock_guard<std::mutex> lkp(p->mu);
    Comm &cm = ctx->comm;
    if (cm.nranks == 0) return fail(BYDB_EINVAL, "bydb_comm_connect was not called on this context");
    if (root < 0 || root >= cm.nranks) return fail(BYDB_EINVAL, "bad root");
    CUDA_TRY(cudaSetDevice(ctx->device));
    g_last_dev_err = 0;
    const uint64_t run = p->reduce_runs++;
    if (run == 0 || !p->reduce_capturable || cm.shared_device) return scan_reduce_impl(ctx, &p->q, nullptr, 0, 0, root, out);
    std::unique_lock<std::mutex> lk(cm.mu);
    const uint64_t epoch = cm.epoch + 1;
    const size_t parity = static_cast<size_t>(epoch & 1u);
    const size_t slot_bytes = cm.peer_slot_bytes[static_cast<size_t>(root)];
    uint8_t *root_mb = cm.peer[static_cast<size_t>(root)];
    uint8_t *slots0 = root_mb + kCommCtl + parity * static_cast<size_t>(cm.nranks) * slot_bytes;
    uint8_t *my_slot = slots0 + static_cast<size_t>(cm.rank) * slot_bytes;
    unsigned long long *flags = reinterpret_cast<unsigned long long *>(root_mb);
    unsigned long long *status = reinterpret_cast<unsigned long long *>(root_mb + kCommStatusOff);
    unsigned long long *done = reinterpret_cast<unsigned long long *>(root_mb + kCommDoneOff);
    uint32_t *my_err = reinterpret_cast<uint32_t *>(cm.mine + kCommErrOff);
    CommArgs *d_args = reinterpret_cast<CommArgs *>(cm.mine + kCommArgsOff);
    ExecSlot &es = *p->slot;
    // pinned words of this prepared query that the graph's memcpy nodes read / write: the last two zero pages of its slot
    CommArgs *h_args = reinterpret_cast<CommArgs *>(es.zpage + 256 * 7);
    uint8_t *h_back = es.zpage + 256 * 6;  // [0,4) this rank's wait-kernel error word, [8, 8 + 8 * nranks) the status words (root)
    if (static_cast<size_t>(cm.nranks) * 8 + 8 > 256) {  // more ranks than the pinned read-back page holds status words for
        lk.unlock();
        return scan_reduce_impl(ctx, &p->q, nullptr, 0, 0, root, out);
    }
    auto &rg = p->reduce_graphs[root * 2 + static_cast<int>(parity)];
    // a graph reads its parts through the pointers captured with it (same rule as bydb_scan_agg_prepared)
    if (rg.exec) {
        std::lock_guard<std::mutex> lk2(ctx->mu);
        bool same = rg.held.size() == p->parts.size(), missing = false;
        for (size_t i = 0; i < p->parts.size(); ++i) {
            auto it = ctx->parts.find(p->parts[i]);
            if (it == ctx->parts.end()) missing = true;
            else if (same && it->second != rg.held[i]) same = false;
        }
        if (missing || !same) {
            cudaGraphExecDestroy(rg.exec);
            rg.exec = nullptr;
            rg.held.clear();
        }
    }
    if (!rg.exec) {
        Plan plan;
        int rc = make_plan(ctx, &p->q, nullptr, plan);
        if (rc) {
            lk.unlock();
            return scan_reduce_impl(ctx, &p->q, nullptr, 0, 0, root, out);  // takes part in the collective and reports the failure
        }
        bool overlap = false;  // the version-dedup precheck synchronises: such queries keep the plain path
        for (size_t a = 0; a < plan.parts.size(); ++a)
            for (size_t b = a + 1; b < plan.parts.size(); ++b) {
                const PartDir &x = plan.parts[a]->dir, &y = plan.parts[b]->dir;
                if (x.blocks.empty() || y.blocks.empty()) continue;
                if (std::max(std::max(x.min_ts, y.min_ts), p->q.tmin) <= std::min(std::min(x.max_ts, y.max_ts), p->q.tmax)) overlap = true;
            }
        TableLayout tl(static_cast<size_t>(plan.n_groups), plan.fcols.size());
        const size_t G = static_cast<size_t>(plan.n_groups), A = p->q.n_aggs, NS = p->q.n_series;
        const size_t stage = align_up(NS * 12 + (G + 1) * 4 + 512, 256);
        p->host_off = stage;
        if (overlap || tl.total > slot_bytes || es.ensure_pinned(stage + G * (12 + 16 * A) + 16 * A + 16384)) {
            p->reduce_capturable = false;
            lk.unlock();
            return scan_reduce_impl(ctx, &p->q, nullptr, 0, 0, root, out);
        }
        memset(&rg.captured, 0, sizeof rg.captured);
        cudaStream_t s = es.stream;
        cudaGetLastError();  // a stale error of an earlier call must not be blamed on the capture
        cudaError_t e = cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal);
        const char *bad_step = nullptr;  // first step of the capture the runtime objected to (BYDB_TRACE prints it)
        if (e == cudaSuccess) {
            Scratch fin;
            auto step = [&](const char *name, bool good) {
                const cudaError_t le = cudaGetLastError();
                if ((!good || le != cudaSuccess) && !bad_step) {
                    bad_step = name;
                    if (le != cudaSuccess) e = le;
                }
            };
            step("args copy", cudaMemcpyAsync(d_args, h_args, sizeof(CommArgs), cudaMemcpyHostToDevice, s) == cudaSuccess);
            launch_comm_wait_args(done, 1, d_args, 1, my_err, kErrPeerTimeout, s);
            step("wait for the slots", true);
            step("scan", run_scan(ctx, &p->q, plan, es, s, my_slot, tl, &rg.captured, 0, true) == 0);
            launch_comm_signal_args(flags + cm.rank, status + cm.rank, d_args, s);
            step("signal", true);
            if (cm.rank == root) {
                launch_comm_wait_args(flags, static_cast<uint32_t>(cm.nranks), d_args, 0, my_err, kErrPeerTimeout, s);
                step("wait for the ranks", true);
                launch_combine_tables(reinterpret_cast<uint64_t *>(slots0), static_cast<uint32_t>(cm.nranks), tl.total / 8, tl.off_sum_f64 / 8,
                                      tl.off_max_f64 / 8, tl.off_max_f64 / 8, tl.off_sum_i64 / 8, tl.off_sum_i64 / 8, tl.off_max_i64 / 8, tl.off_max_i64 / 8,
                                      tl.total / 8, s, slot_bytes / 8);
                step("combine", true);
                step("finalize", finalize_enqueue(&p->q, plan, es, s, slots0, tl, p->host_off, rg.fl, fin) == 0);
                launch_comm_done_args(done, d_args, s);
                step("done word", true);
                step("status read-back",
                     cudaMemcpyAsync(h_back + 8, status, sizeof(unsigned long long) * static_cast<size_t>(cm.nranks), cudaMemcpyDeviceToHost, s) == cudaSuccess);
                rg.captured.kernel_launches += 3 + rg.fl.launches;
            }
            step("error read-back", cudaMemcpyAsync(h_back, my_err, sizeof(uint32_t), cudaMemcpyDeviceToHost, s) == cudaSuccess);
            rg.captured.kernel_launches += 2;
        }
        cudaGraph_t graph = nullptr;
        if (e == cudaSuccess || bad_step) {
            const cudaError_t ee = cudaStreamEndCapture(s, &graph);  // always leave capture mode
            if (!bad_step && ee != cudaSuccess) {
                bad_step = "end capture";
                e = ee;
            }
        }
        if (!bad_step && graph) {
            e = cudaGraphInstantiate(&rg.exec, graph, 0);
            if (e != cudaSuccess) bad_step = "instantiate";
        }
        if (graph) cudaGraphDestroy(graph);
        if (bad_step || !rg.exec) {
            static const bool trace = getenv("BYDB_TRACE") != nullptr;
            if (trace) fprintf(stderr, "[bydb] prepared collective: capture failed at '%s' (%s); keeping the plain path\n", bad_step ? bad_step : "?", cudaGetErrorString(e));
            cudaGetLastError();
            if (rg.exec) cudaGraphExecDestroy(rg.exec);
            rg.exec = nullptr;
            p->reduce_capturable = false;  // the plain path from here on
            lk.unlock();
            return scan_reduce_impl(ctx, &p->q, nullptr, 0, 0, root, out);
        }
        rg.held = plan.parts;
    }
    // ---- replay
    cm.epoch = epoch;
    const uint64_t prev_use = cm.last_use[2 * static_cast<size_t>(root) + parity];
    cm.last_use[2 * static_cast<size_t>(root) + parity] = epoch;
    h_args->epoch = epoch;
    h_args->prev_use = prev_use;
    memset(h_back, 0, 256);
    memset(es.zpage, 0, 256);
    cudaStream_t s = es.stream;
    CUDA_TRY(cudaEventRecord(p->t0, s));
    CUDA_TRY(cudaGraphLaunch(rg.exec, s));
    CUDA_TRY(cudaEventRecord(p->t1, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaGetLastError());
    out->stats = rg.captured;
    const uint32_t *hz = reinterpret_cast<const uint32_t *>(es.zpage);
    const unsigned long long *hs = reinterpret_cast<const unsigned long long *>(es.zpage + 16);
    out->stats.rows_scanned = hs[0];
    out->stats.rows_matched = hs[1];
    out->stats.page_bytes = hs[2];
    out->stats.blocks_scanned = hs[3];
    out->stats.blocks_slow_lane = static_cast<uint32_t>(hs[4]);
    out->stats.slow_lane_reasons = static_cast<uint32_t>(hs[5]);
    float ms = 0;
    cudaEventElapsedTime(&ms, p->t0, p->t1);
    out->stats.device_ms = ms;
    out->stats.scan_kernel_ms = 0;  // per-kernel events are not available inside a graph replay
    const uint32_t perr = *reinterpret_cast<const uint32_t *>(h_back);
    if (perr != 0) cudaMemset(my_err, 0, sizeof perr);
    if (hz[2] != 0) {
        g_last_dev_err = hz[2];
        char buf[96];
        snprintf(buf, sizeof buf, " (block/series #%u)", hz[3]);
        return fail(dev_err_code(hz[2]), std::string(dev_err_text(hz[2])) + buf);
    }
    if (perr != 0) return fail(dev_err_code(perr), dev_err_text(perr));
    if (cm.rank != root) return 0;
    const unsigned long long *peer_status = reinterpret_cast<const unsigned long long *>(h_back + 8);
    for (int r = 0; r < cm.nranks; ++r) {
        const unsigned long long w = peer_status[r];
        if ((w >> 32) == (epoch & 0xffffffffull) && static_cast<uint32_t>(w) != 0)
            return fail(-static_cast<int>(static_cast<uint32_t>(w)), "multi-GPU reduce: rank " + std::to_string(r) + " failed before its scan");
    }
    const uint8_t *h = es.pinned + p->host_off;
    const uint32_t e_in = *reinterpret_cast<const uint32_t *>(h + (rg.fl.o_cnt - rg.fl.o_out) + 8);
    if (e_in != 0) {
        g_last_dev_err = e_in;
        return fail(dev_err_code(e_in), std::string(dev_err_text(e_in)) + " (status carried in a partial table)");
    }
    finalize_parse(h, rg.fl, out);
    return 0;
    });
}

// The collective with HOST file images on every rank (the end-to-end form of a cold distributed query): each rank's parts
// are admitted for the duration of the call (BYDB_Q_HOST_ZERO_COPY: directory upload only, pages pulled over PCIe by the
// scan), scanned into the root's mailbox and dropped.  q->parts / q->n_parts are ignored.
int bydb_scan_reduce_host(bydb_ctx *ctx, uint32_t n_parts, const bydb_part_files *parts, const bydb_query *q, int32_t root, bydb_result *out) {
    return guarded([&]() -> int {
    if (!ctx || !out) return fail(BYDB_EINVAL, "ctx/out is NULL");
    memset(out, 0, sizeof *out);
    CUDA_TRY(cudaSetDevice(ctx->device));
    g_last_dev_err = 0;
    std::vector<std::shared_ptr<Part>> tmp;
    uint64_t h2d = 0;
    int rc = validate_query(q, false);
    if (!rc && (n_parts == 0 || !parts || n_parts > kMaxParts)) rc = fail(BYDB_EINVAL, "need 1..64 host parts");
    const bool zc = !rc && (q->flags & BYDB_Q_HOST_ZERO_COPY) != 0;
    for (uint32_t i = 0; i < n_parts && !rc; ++i) {
        std::shared_ptr<Part> p;
        // fallback pages are unpacked up front here: a collective cannot be re-run by one rank alone
        rc = register_part_locked_free(ctx, ~0ull - i, &parts[i], p, &h2d, zc, true, 0, 1, !zc);
        if (!rc) tmp.push_back(p);
    }
    rc = scan_reduce_impl(ctx, q, &tmp, rc, h2d, root, out);
    if (!rc && zc) out->stats.h2d_bytes += out->stats.page_bytes;  // pages were read in place over PCIe
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        for (auto &p : tmp) ctx->hbm_used -= p->hbm_bytes;
    }
    return rc;
    });
}

}  // extern "C"
