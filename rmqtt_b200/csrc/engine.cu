// libgpumqtt: C ABI (include/gpumqtt.h) over the host mirror (host_trie.cpp) and the sm_100a kernels
// (kernels.cuh).  There is no CPU fallback: without a CUDA device every entry point that would match
// returns GM_ERR_NO_DEVICE.
#include <cuda_runtime.h>
#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <cctype>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/gpumqtt.h"
#include "host_trie.h"
#include "comm.cuh"
#include "kernels.cuh"
#include "relations.cuh"
#include "retain_kernels.cuh"
#include "retain_tree.h"
#include "pipeline.h"
#include "router_host.h"

using namespace gm;

namespace {

thread_local std::string g_err;

#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            g_err = std::string(#expr) + ": " + cudaGetErrorString(_e);                             \
            return (_e == cudaErrorNoDevice || _e == cudaErrorInsufficientDriver) ? GM_ERR_NO_DEVICE : GM_ERR_CUDA; \
        }                                                                                           \
    } while (0)

struct DevBuf {   // owning device allocation (freed on destruction, also on the early-return error paths)
    void* p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept { if (this != &o) { release(); p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; } return *this; }
    void* detach() { void* q = p; p = nullptr; cap = 0; return q; }
    ~DevBuf() { release(); }
    cudaError_t ensure(size_t bytes, bool keep = false, cudaStream_t s = nullptr) {
        if (bytes <= cap) return cudaSuccess;
        size_t ncap = std::max(bytes, cap + cap / 2);
        ncap = (ncap + 255) & ~size_t(255);
        void* np = nullptr;
        cudaError_t e = cudaMalloc(&np, ncap);
        if (e != cudaSuccess) return e;
        if (keep && p && cap) { e = cudaMemcpyAsync(np, p, cap, cudaMemcpyDeviceToDevice, s); if (e != cudaSuccess) return e; cudaStreamSynchronize(s); }
        if (p) cudaFree(p);
        p = np; cap = ncap;
        return cudaSuccess;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return static_cast<T*>(p); }
};

static_assert(GM_ERR_INVALID_TOPIC == -2, "k_tokenize writes the per-topic status code directly");

// pipeline.h's launcher on a CUDA stream: counts the launches in *launches; the timing points go to one slot of the event ring
struct CudaLauncher {
    cudaStream_t s;
    cudaEvent_t* ev;                // the ring slot, or nullptr: no timing
    u64* ring_n;
    u64* launches;
    template <class... P, class... A>
    int launch(void (*k)(P...), u32 grid, u32 block, size_t smem, A... a) {
        k<<<grid, block, smem, s>>>(a...);
        ++*launches;
        CUDA_TRY(cudaGetLastError());
        return GM_OK;
    }
    int memset(void* p, int v, size_t bytes) { CUDA_TRY(cudaMemsetAsync(p, v, bytes, s)); return GM_OK; }
    int copy(void* dst, const void* src, size_t bytes) { CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s)); return GM_OK; }
    int mark(int i) {
        if (!ev) return GM_OK;
        CUDA_TRY(cudaEventRecord(ev[i], s));
        if (i == 3) ++*ring_n;
        return GM_OK;
    }
};

}  // namespace

struct SmallGraph;
static void small_graph_destroy(SmallGraph* g);
constexpr int GM_SMALL_NOT_APPLICABLE = 1000;     // internal: the small-batch fast path declined, take the pipelined path

// One match CONTEXT = everything a match call needs besides the (read-only) tables: its own streams, events, kernel
// scratch and staging buffers.  Host-buffer calls take a free context from the engine's pool, enqueue, RELEASE THE
// ENGINE LOCK, and wait on their own events — so several batches are in flight at once (the reference serves many
// concurrent readers under its RwLock, rmqtt/src/router.rs:166) and a mutation never waits behind a D2H copy.
struct MatchCtx {
    static constexpr int MAXC = 32;  // chunks per pipelined host call
    cudaStream_t sc = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_h2d[MAXC] = {}, ev_comp[MAXC] = {};
    cudaEvent_t ev_done = nullptr;   // after the last kernel of the last match enqueued with this context's scratch
    bool recorded = false, busy = false;
    unsigned long long* h_cur = nullptr;             // pinned: cursor snapshot after every chunk
    DevBuf d_tok, d_tok8, d_meta, d_slow, d_ctrl, d_gstack, d_gpool, d_sort, d_hist;   // kernel scratch
    DevBuf d_blob, d_offs, d_spans, d_ids, d_status, d_trees;                          // staging of host-buffer calls
    // small-batch fast path: the whole call (H2D, memsets, 5 kernels, D2H) as ONE CUDA-graph launch (see SmallGraph)
    struct SmallGraph* small[2] = {nullptr, nullptr};
    // the scratch pointers a captured graph has baked in: a later, larger call may re-allocate any of them
    u64 scratch_sig() const {
        u64 h = 0x9E3779B97F4A7C15ull;
        for (const DevBuf* b : {&d_tok, &d_tok8, &d_meta, &d_slow, &d_ctrl, &d_gstack, &d_gpool, &d_sort, &d_hist}) h = (h ^ reinterpret_cast<uintptr_t>(b->p)) * 0x100000001B3ull;
        return h;
    }
    int init() {
        CUDA_TRY(cudaStreamCreateWithFlags(&sc, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&s_h2d, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&s_d2h, cudaStreamNonBlocking));
        for (int i = 0; i < MAXC; ++i) {
            CUDA_TRY(cudaEventCreateWithFlags(&ev_h2d[i], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&ev_comp[i], cudaEventDisableTiming));
        }
        CUDA_TRY(cudaEventCreateWithFlags(&ev_done, cudaEventDisableTiming));
        CUDA_TRY(cudaMallocHost(&h_cur, MAXC * sizeof(unsigned long long)));
        return GM_OK;
    }
    void destroy();
};

struct gm_engine {
    // LOCK ORDER: mu (host mirror: mutations, flush, statistics) -> mu_dev (device enqueue state: contexts, view, events).
    // A match takes mu only to flush pending mutations (auto-flush engines) and mu_dev only while it ENQUEUES.
    std::mutex mu, mu_dev, mu_ret;   // mu_ret serialises retained lookups (their scratch is engine-wide)
    std::condition_variable cv_ctx;
    int device = 0;
    u32 flags = 0;
    int num_sms = 0;
    HostTrie trie;
    RetainTreeHost rtree{&trie};     // retained-message tree (shares the level dictionary)
    static constexpr int NCTX = 3;   // host-buffer matches in flight
    MatchCtx ctxs[NCTX];
    MatchCtx devctx;                 // scratch of the device-buffer entry points (they run on the CALLER's stream)
    cudaStream_t side = nullptr;     // flush
    static constexpr int MAXC = MatchCtx::MAXC;
    static constexpr int RING = 64;   // per-kernel timing events of the last RING match calls
    cudaEvent_t ev_flush = nullptr;
    cudaEvent_t ev_ring[RING][4] = {};
    u64 ring_n = 0;
    u64 view_epoch = 0;               // bumped by every flush that changed what the kernels see
    // device tables
    DevBuf d_edges, d_ranges, d_values, d_dict, d_pool, d_cfilter, d_tree_slots;
    ShipMarks up;                    // what the device tables hold
    // flush staging: patches are gathered into PINNED host memory and scattered by kernels on the side stream —
    // the flush never synchronises the host with the device
    DevBuf d_patch;
    char* h_patch = nullptr; size_t h_patch_cap = 0;
    cudaEvent_t ev_patch = nullptr;  // the previous flush has consumed h_patch
    bool patch_pending = false;
    struct Retired { void* p; u64 gen; };
    std::vector<Retired> retired;    // table buffers replaced by an epoch swap: freed once every match that could see them is done
    u64 flush_gen = 0;
    // retained tree (device copy of the flattened arrays) + scratch of the retained lookup
    DevBuf d_rnodes, d_rkids, d_redges, d_rvals;
    DevBuf d_rfront[2], d_rdescs, d_rctl, d_rq, d_rstage[5];
    u32 r_cap_items = 1u << 22, r_cap_desc = 1u << 22;   // totals over the RQ slices of each queue
    u64 launches = 0;
    bool k2_attr_set = false;
    // fused gather over peer memory (comm.cuh): one block per rank holding every rank's slab; the peers' blocks are opened by CUDA IPC
    struct Gather : GatherLayout {
        char* block = nullptr;
        u32 rank = 0, epoch = 0;
        char* peer[8] = {};
        DevBuf d_ptrs;      // device arrays for k_gather_finish: counts pointers [8], flags pointers [8]
        bool connected = false;
    } gather;
    // multi-GPU (comm.cuh): NCCL communicator of the root-hash shards, scratch of the size exchange
    ncclComm_t comm = nullptr;
    u32 comm_rank = 0, comm_world = 1;
    DevBuf d_comm, d_part;
    unsigned long long* h_comm = nullptr;   // pinned [2 * world + 64]
    // tuning / diagnostics knobs, read from the environment once at creation
    struct Knobs { u32 site_bits = 14, sub_bits = 0; bool sorted_rows = true; int k2_ctas = 0; u32 diag_flags = 0; u32 tile_chunk = 1; bool tok_bulk = true; u32 e2e_chunk = 262144; bool small_graphs = true; bool retain_stats = false; bool gather_bcast = false; bool gather_direct = false; } knobs;
    void read_knobs() {
        if (const char* ev = getenv("GM_BUCKET_BITS")) { int a = 14, b = 0; if (sscanf(ev, "%d,%d", &a, &b) >= 1 && a >= 10 && b >= 0 && a + b <= int(MAX_BUCKET_BITS)) { knobs.site_bits = a; knobs.sub_bits = b; } }
        if (const char* ev = getenv("GM_SORTED_ROWS")) knobs.sorted_rows = atoi(ev) != 0;
        if (const char* ev = getenv("GM_K2_CTAS")) knobs.k2_ctas = atoi(ev);
        if (const char* ev = getenv("GM_TILE_CHUNK")) { int v = atoi(ev); if (v >= 1 && v <= 1024) knobs.tile_chunk = static_cast<u32>(v); }
        if (getenv("GM_DIAG_NO_PUBLISH")) knobs.diag_flags |= MP_DIAG_NO_PUBLISH;
        if (const char* ev = getenv("GM_TOK_BULK")) knobs.tok_bulk = atoi(ev) != 0;
        if (const char* ev = getenv("GM_ALLGATHERV")) knobs.gather_bcast = std::string(ev) == "bcast";
        if (const char* ev = getenv("GM_GATHER_DIRECT")) knobs.gather_direct = atoi(ev) != 0;
        if (const char* ev = getenv("GM_SMALL_GRAPHS")) knobs.small_graphs = atoi(ev) != 0;
        if (const char* ev = getenv("GM_E2E_CHUNK")) { int v = atoi(ev); if (v >= 1024) knobs.e2e_chunk = static_cast<u32>(v); }
    }

    explicit gm_engine(u32 max_levels) : trie(max_levels) {}

    // The view the kernels get is a SNAPSHOT taken when the tables were last shipped (flush): with
    // GM_FLAG_MANUAL_FLUSH the host mirror may already have grown / re-hashed a table that the device has not seen yet.
    TrieView dev_view{};
    RetainView dev_rview{};

    // ---- flush: ship the staged mutations to HBM on the side stream WITHOUT stopping the matches ------------------------
    // Phase A (no fence; only the host-mirror lock `mu` is held, matches keep running):
    //   * a table that was re-hashed / outgrew its buffer / was compacted goes into a NEW device buffer (epoch swap);
    //   * appended tails (values, ranges, string pool, retained child blocks / values) are copied behind the part the
    //     running kernels can reach — no published record refers to them yet;
    //   * changed 32-byte slots are gathered into PINNED memory and copied to a device staging area.
    // Phase B (under mu_dev, microseconds of host time, no host<->device synchronisation):
    //   * the side stream waits for every match enqueued so far (their ev_done), the new buffers are swapped in, the
    //     staged slots are scattered by k_apply_patches, ev_flush is recorded; matches enqueued from now on wait for
    //     ev_flush on the device and use the new view;
    //   * replaced buffers are retired and freed by a later flush once that ev_flush has passed.
    struct alignas(32) Blk32 { u32 w[8]; };
    struct PatchJob { DevBuf* table; u32 elem, n; size_t off_idx, off_data; };
    struct Swap { DevBuf* dst; DevBuf fresh; };
    std::vector<PatchJob> jobs_;
    std::vector<Swap> swaps_;
    size_t stage_used_ = 0;
    int arena_ = 0;
    char* h_arena_[2] = {nullptr, nullptr}; size_t h_arena_cap_[2] = {0, 0};
    cudaEvent_t ev_arena_[2] = {nullptr, nullptr}; bool arena_pending_[2] = {false, false};

    MatchGeometry geometry() const {
        MatchGeometry g;
        g.num_sms = static_cast<u32>(num_sms); g.k2_ctas = knobs.k2_ctas; g.site_bits = knobs.site_bits; g.sub_bits = knobs.sub_bits;
        g.sorted_rows = knobs.sorted_rows; g.tok_bulk = knobs.tok_bulk; g.gather_direct = knobs.gather_direct;
        g.diag_flags = knobs.diag_flags; g.tile_chunk = knobs.tile_chunk;
        return g;
    }

    int stage_reserve(size_t bytes) {
        if (bytes <= h_arena_cap_[arena_]) return GM_OK;
        size_t ncap = std::max(bytes, h_arena_cap_[arena_] * 2 + (size_t(1) << 20));
        char* np = nullptr;
        CUDA_TRY(cudaMallocHost(&np, ncap));
        if (h_arena_[arena_]) { std::memcpy(np, h_arena_[arena_], stage_used_); cudaFreeHost(h_arena_[arena_]); }
        h_arena_[arena_] = np; h_arena_cap_[arena_] = ncap;
        return GM_OK;
    }

    // ---- the shipper of pipeline.h's ship() ----
    // gather the listed (already final) host slots into the pinned arena; they are scattered in phase B
    template <class V>
    int patch(DevBuf& buf, const V& host, std::vector<u32>& dirty) {
        using T = std::remove_cv_t<std::remove_reference_t<decltype(host[0])>>;
        static_assert(sizeof(T) == 32 || sizeof(T) == 8 || sizeof(T) == 4 || sizeof(T) == 1, "patchable element sizes");
        std::sort(dirty.begin(), dirty.end());
        dirty.erase(std::unique(dirty.begin(), dirty.end()), dirty.end());
        const u32 nd = static_cast<u32>(dirty.size());
        if (nd == 0) return GM_OK;
        const size_t off_idx = (stage_used_ + 31) & ~size_t(31);
        const size_t off_data = (off_idx + nd * sizeof(u32) + 31) & ~size_t(31);
        int st = stage_reserve(off_data + nd * sizeof(T));
        if (st != GM_OK) return st;
        char* base = h_arena_[arena_];
        std::memcpy(base + off_idx, dirty.data(), nd * sizeof(u32));
        T* data = reinterpret_cast<T*>(base + off_data);
        for (u32 i = 0; i < nd; ++i) data[i] = host[dirty[i]];
        stage_used_ = off_data + nd * sizeof(T);
        jobs_.push_back(PatchJob{&buf, static_cast<u32>(sizeof(T)), nd, off_idx, off_data});
        dirty.clear();
        return GM_OK;
    }

    // whole array into a fresh device buffer (swapped in at the fence)
    int fresh(DevBuf& buf, const void* src, size_t bytes, size_t cap_bytes) {
        DevBuf nb;
        CUDA_TRY(nb.ensure(cap_bytes));
        if (bytes) CUDA_TRY(cudaMemcpyAsync(nb.p, src, bytes, cudaMemcpyHostToDevice, side));
        swaps_.push_back(Swap{&buf, std::move(nb)});
        return GM_OK;
    }
    // a tail behind the part the running kernels can reach
    int append(DevBuf& buf, size_t off, const void* src, size_t bytes) {
        CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(buf.p) + off, src, bytes, cudaMemcpyHostToDevice, side));
        return GM_OK;
    }
    size_t capacity(const DevBuf& buf) const { return buf.cap; }
    TableBufs<DevBuf> tables() { return {&d_edges, &d_dict, &d_ranges, &d_values, &d_pool, &d_cfilter, &d_tree_slots, &d_rnodes, &d_rkids, &d_redges, &d_rvals}; }

    void free_retired(bool all) {
        if (retired.empty()) return;
        if (!all && cudaEventQuery(ev_flush) != cudaSuccess) return;     // the last fence has not passed yet: some match may still read them
        for (const Retired& r : retired) cudaFree(r.p);
        retired.clear();
    }

    // A flush that fails half-way (a cudaMalloc of a fresh table buffer, a copy) has already advanced the "shipped up to here"
    // marks and cleared dirty lists for the parts it handled: nothing may be assumed about what reached the device any more.
    // The next flush therefore ships every table whole into new buffers; until then the kernels keep the last complete view.
    int flush_locked() {      // caller holds `mu`
        const int st = flush_impl();
        if (st != GM_OK && !(flags & GM_FLAG_HOST_ONLY) && st != GM_ERR_TOO_LARGE) {
            jobs_.clear(); swaps_.clear(); stage_used_ = 0;               // (fresh buffers not yet swapped in are freed here)
            up.forget_all();
            trie.full_edges = trie.full_dict = true; trie.cfilter_dirty = true; trie.trees_dirty = true; trie.root_dirty = true;
            rtree.dirty = true; rtree.full = true;
        }
        return st;
    }

    int flush_impl() {        // caller holds `mu`
        if (flags & GM_FLAG_HOST_ONLY) {
            if (!trie.sync()) { g_err = "more than 2^32 live value words"; return GM_ERR_TOO_LARGE; }
            if (rtree.dirty) { rtree.prepare_flush(); rtree.shipped(); }
            return GM_OK;
        }
        if (!trie.any_dirty() && !rtree.dirty) return GM_OK;
        CUDA_TRY(cudaSetDevice(device));
        if (!trie.sync()) { g_err = "more than 2^32 live value words"; return GM_ERR_TOO_LARGE; }
        free_retired(false);
        // ---------------- phase A ----------------
        arena_ ^= 1;
        if (arena_pending_[arena_]) { CUDA_TRY(cudaEventSynchronize(ev_arena_[arena_])); arena_pending_[arena_] = false; }   // two flushes ago: long done
        jobs_.clear(); swaps_.clear(); stage_used_ = 0;
        bool r_shipped = false;
        const int rs = ship(*this, tables(), trie, rtree, up, &r_shipped);
        if (rs != GM_OK) return rs;
        if (stage_used_) {
            CUDA_TRY(d_patch.ensure(stage_used_));
            CUDA_TRY(cudaMemcpyAsync(d_patch.p, h_arena_[arena_], stage_used_, cudaMemcpyHostToDevice, side));
        }
        // ---------------- phase B: the fence ----------------
        {
            std::lock_guard<std::mutex> gd(mu_dev);
            for (MatchCtx* c : all_ctxs()) if (c->recorded) CUDA_TRY(cudaStreamWaitEvent(side, c->ev_done, 0));   // never patch under a running match
            for (Swap& sw : swaps_) {
                if (sw.dst->p) retired.push_back(Retired{sw.dst->detach(), flush_gen});
                *sw.dst = std::move(sw.fresh);
            }
            swaps_.clear();
            for (const PatchJob& j : jobs_) {
                const u32* idx = reinterpret_cast<const u32*>(static_cast<char*>(d_patch.p) + j.off_idx);
                const void* data = static_cast<char*>(d_patch.p) + j.off_data;
                const unsigned grid = (j.n + 255) / 256;
                if (j.elem == 32) k_apply_patches<Blk32><<<grid, 256, 0, side>>>(j.table->as<Blk32>(), idx, static_cast<const Blk32*>(data), j.n);
                else if (j.elem == 8) k_apply_patches<Range><<<grid, 256, 0, side>>>(j.table->as<Range>(), idx, static_cast<const Range*>(data), j.n);
                else if (j.elem == 4) k_apply_patches<u32><<<grid, 256, 0, side>>>(j.table->as<u32>(), idx, static_cast<const u32*>(data), j.n);
                else k_apply_patches<u8><<<grid, 256, 0, side>>>(j.table->as<u8>(), idx, static_cast<const u8*>(data), j.n);
                launches++;
            }
            CUDA_TRY(cudaGetLastError());
            if (stage_used_) { CUDA_TRY(cudaEventRecord(ev_arena_[arena_], side)); arena_pending_[arena_] = true; }
            dev_view = make_trie_view(trie, {d_edges.as<EdgeSlot>(), d_ranges.as<Range>(), d_values.as<u32>(), d_dict.as<DictSlot>(), d_pool.as<u8>(),
                                             d_cfilter.as<u32>(), d_tree_slots.as<u32>()});
            dev_rview = make_retain_view(rtree, {d_rkids.as<RKid>(), d_redges.as<REdge>(), d_rvals.as<u32>()});
            view_epoch++;
            CUDA_TRY(cudaEventRecord(ev_flush, side));
            flush_gen++;
        }
        if (r_shipped) rtree.shipped();
        return GM_OK;
    }

    std::vector<MatchCtx*> all_ctxs() { std::vector<MatchCtx*> v; for (auto& c : ctxs) v.push_back(&c); v.push_back(&devctx); return v; }

    // ---- the match pipeline (pipeline.h), all on `s`, all buffers on the device; scratch from context `c` (caller holds mu_dev) ----
    int enqueue_match(MatchCtx& c, const MatchJob& j, cudaStream_t s) {
        if (j.n == 0) { if (j.d_needed) CUDA_TRY(cudaMemsetAsync(j.d_needed, 0, sizeof(u64), s)); return GM_OK; }
        if (j.n > 0xFFFFFFF0ull) { g_err = "batch too large"; return GM_ERR_TOO_LARGE; }
        const MatchGeometry g = geometry();
        const MatchPlan p = plan_match(g, j, dev_view.max_depth);
        CUDA_TRY(c.d_tok.ensure(p.tok));
        CUDA_TRY(c.d_tok8.ensure(p.tok8));
        CUDA_TRY(c.d_meta.ensure(p.meta));
        CUDA_TRY(c.d_slow.ensure(p.slow));
        CUDA_TRY(c.d_ctrl.ensure(p.ctrl));
        CUDA_TRY(c.d_sort.ensure(p.sort));
        CUDA_TRY(c.d_hist.ensure(p.hist));
        CUDA_TRY(c.d_gstack.ensure(p.gstack));
        CUDA_TRY(c.d_gpool.ensure(p.gpool));
        const bool small = j.hdr != nullptr;
        if (!small) {      // (a captured graph carries these dependencies as its launch order; events of other streams cannot be waited on while capturing)
            CUDA_TRY(cudaStreamWaitEvent(s, ev_flush, 0));
            if (c.recorded) CUDA_TRY(cudaStreamWaitEvent(s, c.ev_done, 0));   // this context's scratch: one match at a time
        }
        if (!k2_attr_set) {
            for (MatchFastKernel k : match_fast_kernels())
                CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, int(k2_smem_bytes<K2_FAST_L, K2_THREADS>())));
            k2_attr_set = true;
        }
        CudaLauncher l{s, j.timing ? ev_ring[ring_n % RING] : nullptr, &ring_n, &launches};
        const int st = match_pipeline(l, g, j, p, dev_view, {c.d_tok.as<u32>(), c.d_tok8.as<u32>(), c.d_meta.as<u32>(), c.d_slow.as<u32>(), c.d_ctrl.as<Ctrl>(),
                                                          c.d_sort.as<u32>(), c.d_hist.as<u32>(), c.d_gstack.as<u64>(), c.d_gpool.as<Desc>()});
        if (st != GM_OK) return st;
        if (!small) { CUDA_TRY(cudaEventRecord(c.ev_done, s)); c.recorded = true; }
        return GM_OK;
    }

    // ---- retained lookup (pipeline.h) on the engine-wide scratch ----
    int enqueue_retain(const RetainJob& j, cudaStream_t s) {
        std::lock_guard<std::mutex> gd(mu_dev);     // enqueue only; the caller (holding mu_ret) synchronises afterwards without it
        MatchCtx& c = devctx;
        const RetainPlan p = plan_retain(j.n, dev_rview.max_depth, r_cap_items, r_cap_desc);
        CUDA_TRY(c.d_tok.ensure(p.tok));
        CUDA_TRY(c.d_tok8.ensure(p.tok8));
        CUDA_TRY(c.d_meta.ensure(p.meta));
        CUDA_TRY(d_rq.ensure(p.rq));
        CUDA_TRY(d_rctl.ensure(p.ctl));
        CUDA_TRY(d_rfront[0].ensure(p.front));
        CUDA_TRY(d_rfront[1].ensure(p.front));
        CUDA_TRY(d_rdescs.ensure(p.descs));
        CUDA_TRY(cudaStreamWaitEvent(s, ev_flush, 0));
        if (c.recorded) CUDA_TRY(cudaStreamWaitEvent(s, c.ev_done, 0));
        CudaLauncher l{s, ev_ring[ring_n % RING], &ring_n, &launches};
        const int st = retain_pipeline(l, j, p, dev_view, dev_rview, {c.d_tok.as<u32>(), c.d_tok8.as<u32>(), c.d_meta.as<u32>(), d_rq.as<u32>(), d_rctl.as<RCtl>(),
                                                                   {d_rfront[0].as<RTask>(), d_rfront[1].as<RTask>()}, d_rdescs.as<RDesc>()}, static_cast<u32>(num_sms));
        if (st != GM_OK) return st;
        CUDA_TRY(cudaEventRecord(c.ev_done, s));
        c.recorded = true;
        return GM_OK;
    }

    // runs the pipeline, growing the frontier / descriptor scratch until nothing overflowed; leaves *total
    int run_retain(RetainJob j, cudaStream_t s, u64* total) {
        j.stats = knobs.retain_stats;
        for (int attempt = 0; attempt < RETAIN_ATTEMPTS; ++attempt) {
            int st = enqueue_retain(j, s);
            if (st != GM_OK) return st;
            RCtl h{};
            CUDA_TRY(cudaMemcpyAsync(&h, d_rctl.p, sizeof(RCtl), cudaMemcpyDeviceToHost, s));
            CUDA_TRY(cudaStreamSynchronize(s));
            if (h.err == 0 && knobs.retain_stats) {      // diagnostics: work counters of the instrumented kernels + tasks per round
                const u32 depth = dev_rview.max_depth;
                std::vector<u32> cnt(static_cast<size_t>(depth + 3) * RQ);
                CUDA_TRY(cudaMemcpy(cnt.data(), static_cast<char*>(d_rctl.p) + offsetof(RCtl, counts), cnt.size() * sizeof(u32), cudaMemcpyDeviceToHost));
                fprintf(stderr, "retain stats: visited %llu probes %llu hits %llu; tasks per round:", h.stats[0], h.stats[1], h.grand);
                for (u32 l = 0; l <= depth + 1; ++l) { unsigned long long t = 0; for (u32 k = 0; k < RQ; ++k) t += cnt[static_cast<size_t>(l) * RQ + k]; fprintf(stderr, " %llu", t); }
                unsigned long long nd = 0; for (u32 k = 0; k < RQ; ++k) nd += h.n_desc[k];
                fprintf(stderr, "; descriptors %llu\n", nd);
            }
            if (h.err == 0) { *total = h.grand; return GM_OK; }
            if (!retain_grow(h.err, r_cap_items, r_cap_desc)) break;
        }
        g_err = "retained lookup: frontier does not fit the scratch limits, split the batch";
        return GM_ERR_TOO_LARGE;
    }
};

// =====================================================================================================
extern "C" {

const char* gm_version(void) { return "libgpumqtt 0.1 (sm_100a)"; }
const char* gm_last_error(gm_engine*) { return g_err.c_str(); }

int32_t gm_create(const gm_config* cfg, gm_engine** out) {
    if (!out) return GM_ERR_INVALID_ARG;
    *out = nullptr;
    gm_config c{};
    c.struct_size = sizeof(gm_config); c.device = -1;
    if (cfg) std::memcpy(&c, cfg, std::min<size_t>(cfg->struct_size ? cfg->struct_size : sizeof(gm_config), sizeof(gm_config)));
    if (c.flags & GM_FLAG_HOST_ONLY) {   // staging mirror only (tests, off-device shard preparation): nothing can match
        gm_engine* eng = new gm_engine(c.max_levels ? c.max_levels : 128u);
        eng->flags = c.flags;
        eng->device = -1;
        if (c.filters_hint) eng->trie.reserve(c.filters_hint);
        *out = eng;
        return GM_OK;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) { g_err = "no CUDA device: libgpumqtt has no CPU fallback"; return GM_ERR_NO_DEVICE; }
    int dev = c.device;
    if (dev < 0) CUDA_TRY(cudaGetDevice(&dev));
    if (dev >= ndev) { g_err = "device ordinal out of range"; return GM_ERR_INVALID_ARG; }
    CUDA_TRY(cudaSetDevice(dev));
    gm_engine* eng = new gm_engine(c.max_levels ? c.max_levels : 128u);
    struct Guard { gm_engine* e; ~Guard() { if (e) gm_destroy(e); } } guard{eng};   // a failing CUDA call below must not leak the half-built engine
    eng->device = dev;
    eng->flags = c.flags;
    eng->read_knobs();
    cudaDeviceProp prop{};
    CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    eng->num_sms = prop.multiProcessorCount;
    CUDA_TRY(cudaStreamCreateWithFlags(&eng->side, cudaStreamNonBlocking));
    for (MatchCtx* cx : eng->all_ctxs()) { int st = cx->init(); if (st != GM_OK) return st; }
    CUDA_TRY(cudaEventCreateWithFlags(&eng->ev_flush, cudaEventDisableTiming));
    for (auto& ev : eng->ev_arena_) CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    for (auto& q : eng->ev_ring) for (auto& ev : q) CUDA_TRY(cudaEventCreate(&ev));
    CUDA_TRY(cudaEventRecord(eng->ev_flush, eng->side));
    // L2 fetch granularity: a miss on one 32-byte sector makes the L2 fetch 64 bytes from HBM by default.  Every hot access
    // of this engine is a RANDOM 32-byte slot, so the second half of each fetch is wasted DRAM bandwidth; GM_L2_FETCH=32
    // (or gm_config.flags & GM_FLAG_L2_FETCH_32) asks for 32-byte fetches.  It is a per-context limit, hence opt-in.
    if (const char* ev = getenv("GM_L2_FETCH")) { const int v = atoi(ev); if (v == 32 || v == 64 || v == 128) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, static_cast<size_t>(v)); }
    else if (c.flags & GM_FLAG_L2_FETCH_32) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, 32);
    if (c.filters_hint) eng->trie.reserve(c.filters_hint);
    guard.e = nullptr;
    *out = eng;
    return GM_OK;
}

void MatchCtx::destroy() {
    for (DevBuf* b : {&d_tok, &d_tok8, &d_meta, &d_slow, &d_ctrl, &d_gstack, &d_gpool, &d_sort, &d_hist, &d_blob, &d_offs, &d_spans, &d_ids, &d_status, &d_trees}) b->release();
    for (auto& g : small) if (g) { small_graph_destroy(g); g = nullptr; }
    if (sc) cudaStreamDestroy(sc);
    if (s_h2d) cudaStreamDestroy(s_h2d);
    if (s_d2h) cudaStreamDestroy(s_d2h);
    for (int i = 0; i < MAXC; ++i) { if (ev_h2d[i]) cudaEventDestroy(ev_h2d[i]); if (ev_comp[i]) cudaEventDestroy(ev_comp[i]); }
    if (ev_done) cudaEventDestroy(ev_done);
    if (h_cur) cudaFreeHost(h_cur);
}

void gm_destroy(gm_engine* e) {
    if (!e) return;
    if (e->flags & GM_FLAG_HOST_ONLY) { delete e; return; }
    cudaSetDevice(e->device);
    cudaDeviceSynchronize();
    e->free_retired(true);
    for (MatchCtx* cx : e->all_ctxs()) cx->destroy();
    for (DevBuf* b : {&e->d_cfilter, &e->d_tree_slots, &e->d_edges, &e->d_ranges, &e->d_values, &e->d_dict, &e->d_pool, &e->d_patch, &e->d_rnodes, &e->d_rkids, &e->d_redges,
                      &e->d_rvals, &e->d_rfront[0], &e->d_rfront[1], &e->d_rdescs, &e->d_rctl, &e->d_rq, &e->d_rstage[0], &e->d_rstage[1], &e->d_rstage[2],
                      &e->d_rstage[3], &e->d_rstage[4]})
        b->release();
    if (e->side) cudaStreamDestroy(e->side);
    if (e->comm) { NcclApi::get().CommDestroy(e->comm); e->comm = nullptr; }
    if (e->h_comm) cudaFreeHost(e->h_comm);
    e->d_comm.release(); e->d_part.release();
    if (e->gather.block) { for (u32 w = 0; w < e->gather.world; ++w) if (w != e->gather.rank && e->gather.peer[w]) cudaIpcCloseMemHandle(e->gather.peer[w]); cudaFree(e->gather.block); e->gather.block = nullptr; }
    e->gather.d_ptrs.release();
    for (auto& hp : e->h_arena_) if (hp) cudaFreeHost(hp);
    for (auto& ev : e->ev_arena_) if (ev) cudaEventDestroy(ev);
    if (e->ev_flush) cudaEventDestroy(e->ev_flush);
    for (auto& q : e->ev_ring) for (auto& ev : q) if (ev) cudaEventDestroy(ev);
    delete e;
}

static int32_t map_parse(int st, const char* what) {
    if (st == PARSE_OK) return GM_OK;
    if (st == PARSE_TOO_DEEP) { g_err = std::string(what) + ": filter deeper than max_levels"; return GM_ERR_TOO_DEEP; }
    g_err = std::string(what) + ": invalid topic filter";
    return GM_ERR_INVALID_TOPIC;
}

int32_t gm_sub_add(gm_engine* e, const char* filter, uint32_t len, uint32_t value, int32_t* changed) {
    if (!e || (!filter && len)) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    bool ch = false;
    int st = e->trie.insert(filter, len, value, &ch);
    if (changed) *changed = ch ? 1 : 0;
    return map_parse(st, "gm_sub_add");
}

int32_t gm_sub_remove(gm_engine* e, const char* filter, uint32_t len, uint32_t value, int32_t* changed) {
    if (!e || (!filter && len)) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    bool ch = false;
    int st = e->trie.remove(filter, len, value, &ch);
    if (changed) *changed = ch ? 1 : 0;
    return map_parse(st, "gm_sub_remove");
}

int32_t gm_sub_add_tree(gm_engine* e, uint32_t tree, const char* filter, uint32_t len, uint32_t value, int32_t* changed) {
    if (!e || (!filter && len) || tree >= HostTrie::MAX_TREES) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    bool ch = false;
    int st = e->trie.insert(filter, len, value, &ch, tree);
    if (changed) *changed = ch ? 1 : 0;
    return map_parse(st, "gm_sub_add_tree");
}

int32_t gm_sub_remove_tree(gm_engine* e, uint32_t tree, const char* filter, uint32_t len, uint32_t value, int32_t* changed) {
    if (!e || (!filter && len) || tree >= HostTrie::MAX_TREES) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    bool ch = false;
    int st = e->trie.remove(filter, len, value, &ch, tree);
    if (changed) *changed = ch ? 1 : 0;
    return map_parse(st, "gm_sub_remove_tree");
}

int32_t gm_bulk_load(gm_engine* e, const char* blob, const uint32_t* offsets, const uint32_t* values, uint64_t n, uint64_t* n_changed) {
    if (!e || (n && (!blob || !offsets || !values))) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    e->trie.reserve(n);
    uint64_t ok = 0;
    if (getenv("GM_BULK_ONE_BY_ONE")) {       // A/B switch for the host-side bulk-load measurement
        for (uint64_t i = 0; i < n; ++i) { bool ch = false; e->trie.insert(blob + offsets[i], offsets[i + 1] - offsets[i], values[i], &ch); ok += ch; }
    } else ok = e->trie.insert_batch(blob, offsets, values, n);
    if (n_changed) *n_changed = ok;
    return GM_OK;
}

int32_t gm_compact(gm_engine* e) {
    if (!e) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    // the retained tree interns its levels in the same dictionary: carry its tokens over and re-label its nodes
    const std::vector<u32> keep = e->rtree.used_tokens();
    std::vector<u32> remap;
    e->trie.compact(&keep, &remap);
    e->rtree.remap_tokens(remap);
    e->up.forget_trie(e->trie.values_epoch);
    return (e->flags & GM_FLAG_HOST_ONLY) ? GM_OK : e->flush_locked();
}

int32_t gm_flush(gm_engine* e) {
    if (!e) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    return e->flush_locked();
}

// pending mutations become visible before a match unless the caller fences explicitly (GM_FLAG_MANUAL_FLUSH)
static int32_t auto_flush(gm_engine* e, bool need_retained = false) {
    if ((e->flags & GM_FLAG_MANUAL_FLUSH) && e->d_edges.p && (!need_retained || e->d_rnodes.p)) return GM_OK;
    std::lock_guard<std::mutex> g(e->mu);
    return e->flush_locked();
}

// shared implementation of the device-buffer entry points
static int32_t match_device_impl(gm_engine* e, const void* d_blob, uint64_t blob_bytes, const uint32_t* d_offs, uint64_t n_entries, const uint32_t* d_sel,
                                 uint64_t n, gm_span* d_spans, void* d_out, uint64_t cap, uint64_t* d_needed, int32_t* d_status, void* stream,
                                 bool desc, gm_work* work, const uint32_t* d_trees = nullptr) {
    if (!e || (n && (!d_offs || !d_spans || !d_status))) return GM_ERR_INVALID_ARG;
    if (blob_bytes > 0xFFFFFFFFull) { g_err = "topic blob >= 4 GiB"; return GM_ERR_TOO_LARGE; }
    if (e->flags & GM_FLAG_HOST_ONLY) { g_err = "host-only engine cannot match: there is no CPU fallback"; return GM_ERR_NO_DEVICE; }
    CUDA_TRY(cudaSetDevice(e->device));
    { int st = auto_flush(e); if (st != GM_OK) return st; }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    std::unique_lock<std::mutex> gd(e->mu_dev);
    MatchJob job;
    job.blob = d_blob; job.blob_bytes = blob_bytes; job.offs = d_offs; job.sel = d_sel; job.n = n;
    job.spans = d_spans; job.out = d_out; job.cap = cap; job.d_needed = d_needed; job.status = d_status; job.trees = d_trees;
    job.mode = desc ? MatchJob::DESCRIPTORS : MatchJob::IDS;
    job.stats = work != nullptr;
    int st = e->enqueue_match(e->devctx, job, s);
    if (st != GM_OK || !work) return st;
    std::memset(work, 0, sizeof(*work));
    if (n == 0) return GM_OK;
    Ctrl h{};
    std::vector<u32> meta(n), offs(n_entries + 1), sel(d_sel ? n : 0);
    CUDA_TRY(cudaMemcpyAsync(&h, e->devctx.d_ctrl.p, sizeof(Ctrl), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(meta.data(), e->devctx.d_meta.p, n * sizeof(u32), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(offs.data(), d_offs, (n_entries + 1) * sizeof(u32), cudaMemcpyDeviceToHost, s));
    if (d_sel) CUDA_TRY(cudaMemcpyAsync(sel.data(), d_sel, n * sizeof(u32), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    work->visited = h.stats[0]; work->probed = h.stats[1]; work->filters = h.stats[2]; work->ids = h.stats[3];
    work->deferred = h.slow_count;
    for (int k = 0; k < 8; ++k) { work->probes_by_depth[k] = h.stats[4 + k]; work->misses_by_depth[k] = h.stats[12 + k]; }
    work->slot_loads = h.stats[20];
    for (uint64_t i = 0; i < n; ++i)
        if (!(meta[i] & META_INVALID)) { const u64 j = d_sel ? sel[i] : i; work->levels += meta[i] & META_NLEV_MASK; work->bytes += offs[j + 1] - offs[j]; }
    return GM_OK;
}

int32_t gm_match_batch_device(gm_engine* e, const void* d_blob, uint64_t blob_bytes, const uint32_t* d_offs, uint64_t n,
                              gm_span* d_spans, uint32_t* d_ids, uint64_t cap_ids, uint64_t* d_needed, int32_t* d_status, void* stream) {
    return match_device_impl(e, d_blob, blob_bytes, d_offs, n, nullptr, n, d_spans, d_ids, cap_ids, d_needed, d_status, stream, false, nullptr);
}

int32_t gm_match_batch_device_stats(gm_engine* e, const void* d_blob, uint64_t blob_bytes, const uint32_t* d_offs, uint64_t n,
                                    gm_span* d_spans, uint32_t* d_ids, uint64_t cap_ids, uint64_t* d_needed, int32_t* d_status,
                                    void* stream, gm_work* work) {
    if (!work) return GM_ERR_INVALID_ARG;
    return match_device_impl(e, d_blob, blob_bytes, d_offs, n, nullptr, n, d_spans, d_ids, cap_ids, d_needed, d_status, stream, false, work);
}

int32_t gm_match_batch_device_ex(gm_engine* e, const gm_match_args* a) {
    if (!a || a->struct_size < offsetof(gm_match_args, d_trees)) return GM_ERR_INVALID_ARG;
    if (a->d_sel && a->n > a->n_entries) return GM_ERR_INVALID_ARG;
    return match_device_impl(e, a->d_blob, a->blob_bytes, a->d_offsets, a->d_sel ? a->n_entries : a->n, a->d_sel, a->n, a->d_spans, a->d_out, a->cap,
                             a->d_needed, a->d_status, a->stream, (a->flags & GM_MATCH_DESCRIPTORS) != 0, a->work,
                             a->struct_size >= offsetof(gm_match_args, d_trees) + sizeof(a->d_trees) ? a->d_trees : nullptr);
}

}  // extern "C"

// ---- small batches: one CUDA-graph launch per call ---------------------------------------------------------------------
// A PUBLISH-sized batch (1 .. 2048 topics) costs the same five kernels, two memsets and four copies as a million-topic
// batch: at that size the call is pure launch latency.  Per context and capacity tier the whole sequence
//     H2D(pinned in-block) -> memsets -> k_tokenize -> k_bucket_scan -> k_bucket_scatter -> k_match_fast -> k_match_slow
//     -> D2H(pinned out-block)
// is captured ONCE into a CUDA graph sized for the tier's capacity; the real batch size and text length travel in the
// first words of the in-block (`hdr`), which the kernels read at run time.  A call then is: fill the pinned in-block,
// cudaGraphLaunch, wait for one event, copy the results out of the pinned out-block.  The kernels carry the table view
// by value, so the graph is re-captured (cudaGraphExecUpdate) when a flush has changed the view.
struct SmallGraph {
    u32 cap_n = 0, cap_blob = 0, cap_out = 0;
    size_t elem = 0;
    u64 view_epoch = ~0ull, scratch_sig = 0;
    cudaGraphExec_t exec = nullptr;
    char *h_in = nullptr, *h_out = nullptr;
    size_t in_bytes = 0, out_bytes = 0, off_offs = 0, off_trees = 0, off_blob = 0, off_spans = 0, off_status = 0, off_out = 0;
    DevBuf d_in, d_out;
    bool warmed = false;
};
static void small_graph_destroy(SmallGraph* g) {
    if (!g) return;
    if (g->exec) cudaGraphExecDestroy(g->exec);
    if (g->h_in) cudaFreeHost(g->h_in);
    if (g->h_out) cudaFreeHost(g->h_out);
    delete g;
}

static int small_graph_match(gm_engine* e, MatchCtx& c, std::unique_lock<std::mutex>& gd, const char* blob, const uint32_t* offsets, uint64_t n,
                             gm_span* out_spans, void* out, size_t elem, uint64_t cap_user, uint64_t* needed, int32_t* status, const uint32_t* trees) {
    const u64 b0 = offsets[0], blob_bytes = offsets[n] - b0;
    int tier;
    if (n <= 64 && blob_bytes <= 8 * 1024) tier = 0;
    else if (n <= 2048 && blob_bytes <= 192 * 1024) tier = 1;
    else return GM_SMALL_NOT_APPLICABLE;
    SmallGraph*& g = c.small[tier];
    if (!g) {
        g = new SmallGraph();
        g->cap_n = tier == 0 ? 64u : 2048u; g->cap_blob = tier == 0 ? 8u * 1024u : 192u * 1024u; g->cap_out = tier == 0 ? 4096u : 128u * 1024u;
        g->off_offs = 16; g->off_trees = g->off_offs + (g->cap_n + 1) * sizeof(u32); g->off_blob = (g->off_trees + g->cap_n * sizeof(u32) + 255) & ~size_t(255);
        g->in_bytes = g->off_blob + g->cap_blob + 32;
        g->off_spans = 16; g->off_status = g->off_spans + g->cap_n * sizeof(gm_span); g->off_out = (g->off_status + g->cap_n * sizeof(int32_t) + 255) & ~size_t(255);
        g->out_bytes = g->off_out + static_cast<size_t>(g->cap_out) * 8;
        CUDA_TRY(cudaMallocHost(&g->h_in, g->in_bytes));
        CUDA_TRY(cudaMallocHost(&g->h_out, g->out_bytes));
        CUDA_TRY(g->d_in.ensure(g->in_bytes));
        CUDA_TRY(g->d_out.ensure(g->out_bytes));
        std::memset(g->h_in, 0, g->in_bytes);
    }
    const bool desc = elem == 8;
    auto enqueue = [&](cudaStream_t s) -> int {
        char* di = static_cast<char*>(g->d_in.p);
        char* dout = static_cast<char*>(g->d_out.p);
        MatchJob j;
        j.blob = di + g->off_blob; j.blob_bytes = j.readable_bytes = g->cap_blob; j.offs = reinterpret_cast<const u32*>(di + g->off_offs);
        j.n = g->cap_n; j.hdr = reinterpret_cast<const u32*>(di);
        j.spans = reinterpret_cast<gm_span*>(dout + g->off_spans); j.out = dout + g->off_out; j.cap = g->cap_out;
        j.d_needed = reinterpret_cast<u64*>(dout); j.status = reinterpret_cast<int32_t*>(dout + g->off_status); j.trees = reinterpret_cast<const u32*>(di + g->off_trees);
        j.mode = desc ? MatchJob::DESCRIPTORS : MatchJob::IDS;
        j.timing = false;
        j.bucket_bits = 10;
        return e->enqueue_match(c, j, s);
    };
    if (!g->warmed) {      // allocate the scratch and set kernel attributes outside any capture: one empty (n = 0) pass
        CUDA_TRY(cudaMemsetAsync(g->d_in.p, 0, g->in_bytes, c.sc));
        int st = enqueue(c.sc);
        if (st != GM_OK) return st;
        CUDA_TRY(cudaStreamSynchronize(c.sc));
        g->warmed = true;
    }
    if (g->exec && g->scratch_sig != c.scratch_sig()) {      // a larger call re-allocated this context's scratch since the capture:
        CUDA_TRY(cudaMemsetAsync(g->d_in.p, 0, g->in_bytes, c.sc));   // size it again (empty pass), then re-capture with the new pointers
        int st = enqueue(c.sc);
        if (st != GM_OK) return st;
        CUDA_TRY(cudaStreamSynchronize(c.sc));
    }
    if (!g->exec || g->view_epoch != e->view_epoch || g->elem != elem || g->scratch_sig != c.scratch_sig()) {
        cudaGraph_t graph = nullptr;
        CUDA_TRY(cudaStreamBeginCapture(c.sc, cudaStreamCaptureModeRelaxed));
        cudaError_t ce = cudaMemcpyAsync(g->d_in.p, g->h_in, g->in_bytes, cudaMemcpyHostToDevice, c.sc);
        int st = ce == cudaSuccess ? enqueue(c.sc) : GM_ERR_CUDA;
        if (st == GM_OK) ce = cudaMemcpyAsync(g->h_out, g->d_out.p, g->out_bytes, cudaMemcpyDeviceToHost, c.sc);
        cudaError_t ee = cudaStreamEndCapture(c.sc, &graph);
        if (st != GM_OK || ce != cudaSuccess || ee != cudaSuccess) { if (graph) cudaGraphDestroy(graph); g_err = "small-batch graph capture failed"; return st != GM_OK ? st : GM_ERR_CUDA; }
        bool ok = false;
        if (g->exec) {
            cudaGraphExecUpdateResultInfo info{};
            ok = cudaGraphExecUpdate(g->exec, graph, &info) == cudaSuccess;
            if (!ok) { cudaGetLastError(); cudaGraphExecDestroy(g->exec); g->exec = nullptr; }
        }
        if (!ok) CUDA_TRY(cudaGraphInstantiate(&g->exec, graph, 0));
        cudaGraphDestroy(graph);
        g->view_epoch = e->view_epoch; g->elem = elem; g->scratch_sig = c.scratch_sig();
    }
    // fill the pinned in-block: {n, text bytes} | offsets re-based to 0 | text
    u32* hdr = reinterpret_cast<u32*>(g->h_in);
    hdr[0] = static_cast<u32>(n); hdr[1] = static_cast<u32>(blob_bytes);
    u32* ho = reinterpret_cast<u32*>(g->h_in + g->off_offs);
    for (u64 i = 0; i <= n; ++i) ho[i] = static_cast<u32>(offsets[i] - b0);
    if (blob_bytes) std::memcpy(g->h_in + g->off_blob, blob + b0, blob_bytes);
    if (trees) std::memcpy(g->h_in + g->off_trees, trees, n * sizeof(u32)); else std::memset(g->h_in + g->off_trees, 0, n * sizeof(u32));
    CUDA_TRY(cudaStreamWaitEvent(c.sc, e->ev_flush, 0));
    CUDA_TRY(cudaGraphLaunch(g->exec, c.sc));
    CUDA_TRY(cudaEventRecord(c.ev_done, c.sc));
    c.recorded = true;
    e->launches += 5;
    gd.unlock();
    CUDA_TRY(cudaEventSynchronize(c.ev_done));
    const u64 total = *reinterpret_cast<const u64*>(g->h_out);
    if (total > g->cap_out) return GM_SMALL_NOT_APPLICABLE;      // more output than the tier holds: the pipelined path handles it
    if (needed) *needed = total;
    std::memcpy(status, g->h_out + g->off_status, n * sizeof(int32_t));
    if (total > cap_user) { g_err = "output buffer too small"; return GM_ERR_CAPACITY; }
    std::memcpy(out_spans, g->h_out + g->off_spans, n * sizeof(gm_span));
    if (total) std::memcpy(out, g->h_out + g->off_out, total * elem);
    return GM_OK;
}

extern "C" {

// a free context of the pool (blocks while all NCTX are in flight); release() hands it back
struct CtxLease {
    gm_engine* e; MatchCtx* c = nullptr;
    explicit CtxLease(gm_engine* e_) : e(e_) {}
    void acquire(std::unique_lock<std::mutex>& lk) {     // lk holds e->mu_dev
        for (;;) {
            for (auto& cx : e->ctxs) if (!cx.busy) { cx.busy = true; c = &cx; return; }
            e->cv_ctx.wait(lk);
        }
    }
    ~CtxLease() {
        if (!c) return;
        { std::lock_guard<std::mutex> g(e->mu_dev); c->busy = false; }
        e->cv_ctx.notify_one();
    }
};

// shared implementation of the host-buffer entry points; `elem` = bytes per output element (4: ids, 8: descriptors)
static int32_t match_host_impl(gm_engine* e, const char* blob, const uint32_t* offsets, uint64_t n, gm_span* out_spans, void* out, size_t elem,
                               uint64_t cap_ids, uint64_t* needed, int32_t* status, const uint32_t* trees = nullptr) {
    if (!e || (n && (!offsets || !out_spans || !status)) || (cap_ids && !out)) return GM_ERR_INVALID_ARG;
    if (needed) *needed = 0;
    if (n == 0) return GM_OK;
    if (n > 0xFFFFFFF0ull) { g_err = "batch too large"; return GM_ERR_TOO_LARGE; }
    const bool desc = elem == 8;
    if (e->flags & GM_FLAG_HOST_ONLY) { g_err = "host-only engine cannot match: there is no CPU fallback"; return GM_ERR_NO_DEVICE; }
    CUDA_TRY(cudaSetDevice(e->device));
    { int st = auto_flush(e); if (st != GM_OK) return st; }
    const u64 blob_bytes = offsets[n];
    if (cap_ids > 0xFFFFFFFFull) cap_ids = 0xFFFFFFFFull;
    CtxLease lease(e);
    std::unique_lock<std::mutex> gd(e->mu_dev);
    lease.acquire(gd);
    MatchCtx& c = *lease.c;
    // ---- small batches: the whole call as ONE CUDA-graph launch (no per-kernel launch latency) ----
    if (e->knobs.small_graphs) {
        int st = small_graph_match(e, c, gd, blob, offsets, n, out_spans, out, elem, cap_ids, needed, status, trees);
        if (st != GM_SMALL_NOT_APPLICABLE) return st;       // (gd was released inside while waiting)
        if (!gd.owns_lock()) gd.lock();
    }
    CUDA_TRY(c.d_blob.ensure(blob_bytes + 16));
    CUDA_TRY(c.d_offs.ensure((n + 1) * sizeof(u32)));
    CUDA_TRY(c.d_spans.ensure(n * sizeof(gm_span)));
    CUDA_TRY(c.d_status.ensure(n * sizeof(int32_t)));
    CUDA_TRY(c.d_ids.ensure(std::max<u64>(cap_ids, 1) * elem));
    if (trees) { CUDA_TRY(c.d_trees.ensure(n * sizeof(u32))); CUDA_TRY(cudaMemcpyAsync(c.d_trees.p, trees, n * sizeof(u32), cudaMemcpyHostToDevice, c.s_h2d)); }
    // Pipelined in chunks over three streams: H2D of chunk c+1 and D2H of chunk c-1 overlap the kernels of
    // chunk c.  All chunks share one bump cursor, so the output of chunk c is the contiguous range
    // [cursor after c-1, cursor after c) and can be copied out as soon as that chunk's kernels finished.
    const u64 chunk = std::max<u64>(e->knobs.e2e_chunk, (n + gm_engine::MAXC - 1) / gm_engine::MAXC);
    const int nchunks = static_cast<int>((n + chunk - 1) / chunk);
    if (c.recorded) CUDA_TRY(cudaStreamWaitEvent(c.s_h2d, c.ev_done, 0));   // (cannot happen for a leased context; cheap insurance)
    for (int k = 0; k < nchunks; ++k) {
        const u64 c0 = k * chunk, c1 = std::min<u64>(n, c0 + chunk);
        const u64 b0 = offsets[c0], b1 = offsets[c1];
        if (b1 > b0) CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(c.d_blob.p) + b0, blob + b0, b1 - b0, cudaMemcpyHostToDevice, c.s_h2d));
        CUDA_TRY(cudaMemcpyAsync(c.d_offs.as<u32>() + c0, offsets + c0, (c1 - c0 + 1) * sizeof(u32), cudaMemcpyHostToDevice, c.s_h2d));
        CUDA_TRY(cudaEventRecord(c.ev_h2d[k], c.s_h2d));
    }
    for (int k = 0; k < nchunks; ++k) {
        const u64 c0 = k * chunk, c1 = std::min<u64>(n, c0 + chunk);
        CUDA_TRY(cudaStreamWaitEvent(c.sc, c.ev_h2d[k], 0));
        MatchJob j;
        j.blob = c.d_blob.p; j.blob_bytes = offsets[c1]; j.readable_bytes = (offsets[c1] + 15) & ~u64(15);
        j.offs = c.d_offs.as<u32>() + c0; j.n = c1 - c0;
        j.spans = c.d_spans.as<gm_span>() + c0; j.out = c.d_ids.p; j.cap = cap_ids; j.status = c.d_status.as<int32_t>() + c0;
        j.trees = trees ? c.d_trees.as<u32>() + c0 : nullptr;
        j.mode = desc ? MatchJob::DESCRIPTORS : MatchJob::IDS;
        j.keep_cursor = k != 0;
        int st = e->enqueue_match(c, j, c.sc);
        if (st != GM_OK) return st;
        CUDA_TRY(cudaMemcpyAsync(&c.h_cur[k], &c.d_ctrl.as<Ctrl>()->cursor, sizeof(u64), cudaMemcpyDeviceToHost, c.sc));
        CUDA_TRY(cudaEventRecord(c.ev_comp[k], c.sc));
    }
    gd.unlock();        // everything is enqueued: other calls (and flushes) proceed while this one waits for its copies
    u64 done = 0;
    for (int k = 0; k < nchunks; ++k) {
        const u64 c0 = k * chunk, c1 = std::min<u64>(n, c0 + chunk);
        CUDA_TRY(cudaEventSynchronize(c.ev_comp[k]));
        const u64 cur = c.h_cur[k];
        CUDA_TRY(cudaMemcpyAsync(out_spans + c0, c.d_spans.as<gm_span>() + c0, (c1 - c0) * sizeof(gm_span), cudaMemcpyDeviceToHost, c.s_d2h));
        CUDA_TRY(cudaMemcpyAsync(status + c0, c.d_status.as<int32_t>() + c0, (c1 - c0) * sizeof(int32_t), cudaMemcpyDeviceToHost, c.s_d2h));
        const u64 hi = std::min<u64>(cur, cap_ids);
        if (hi > done) {
            CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(out) + done * elem, static_cast<char*>(c.d_ids.p) + done * elem, (hi - done) * elem, cudaMemcpyDeviceToHost, c.s_d2h));
            done = hi;
        }
    }
    CUDA_TRY(cudaStreamSynchronize(c.s_d2h));
    const u64 total = c.h_cur[nchunks - 1];
    if (needed) *needed = total;
    if (total > 0xFFFFFFFFull) { g_err = "batch produces >= 2^32 output elements: split it"; return GM_ERR_TOO_LARGE; }
    if (total > cap_ids) { g_err = "output buffer too small"; return GM_ERR_CAPACITY; }
    return GM_OK;
}

int32_t gm_match_batch(gm_engine* e, const char* blob, const uint32_t* offsets, uint64_t n, gm_span* out_spans, uint32_t* out_ids,
                       uint64_t cap_ids, uint64_t* needed, int32_t* status) {
    return match_host_impl(e, blob, offsets, n, out_spans, out_ids, sizeof(uint32_t), cap_ids, needed, status);
}

int32_t gm_match_batch_trees(gm_engine* e, const char* blob, const uint32_t* offsets, const uint32_t* trees, uint64_t n, gm_span* out_spans, uint32_t* out_ids,
                             uint64_t cap_ids, uint64_t* needed, int32_t* status) {
    return match_host_impl(e, blob, offsets, n, out_spans, out_ids, sizeof(uint32_t), cap_ids, needed, status, trees);
}

int32_t gm_match_batch_desc(gm_engine* e, const char* blob, const uint32_t* offsets, uint64_t n, gm_span* out_spans, gm_desc* out_descs,
                            uint64_t cap_descs, uint64_t* needed, int32_t* status) {
    static_assert(sizeof(gm_desc) == 8, "descriptor = one 64-bit value-set reference");
    return match_host_impl(e, blob, offsets, n, out_spans, out_descs, sizeof(gm_desc), cap_descs, needed, status);
}

int32_t gm_values_view(gm_engine* e, gm_values* out) {
    if (!e || !out) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    out->values = e->trie.values.data(); out->n_values = e->trie.values.size();
    out->ranges = reinterpret_cast<const gm_span*>(e->trie.ranges.data()); out->n_ranges = e->trie.ranges.size();
    out->epoch = e->trie.values_epoch;
    return GM_OK;
}

int32_t gm_desc_expand(gm_engine* e, const gm_desc* descs, uint64_t n, uint32_t* out_ids, uint64_t cap_ids, uint64_t* needed) {
    if (!e || (n && !descs) || (cap_ids && !out_ids)) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    const u32* vals = e->trie.values.data();
    const u64 nvals = e->trie.values.size();
    u64 w = 0;
    for (uint64_t i = 0; i < n; ++i) {
        u32 ref = descs[i].ref, cnt = descs[i].cnt;
        if (cnt == 1) { if (w < cap_ids) out_ids[w] = ref; ++w; continue; }
        u64 off = ref;
        if (cnt == CNT_BIG) { if (ref >= e->trie.ranges.size()) { g_err = "gm_desc_expand: stale descriptor"; return GM_ERR_INVALID_ARG; } off = e->trie.ranges[ref].off; cnt = e->trie.ranges[ref].cnt; }
        if (off + cnt > nvals) { g_err = "gm_desc_expand: stale descriptor (values were compacted since the match)"; return GM_ERR_INVALID_ARG; }
        if (w + cnt <= cap_ids) std::memcpy(out_ids + w, vals + off, cnt * sizeof(u32));
        w += cnt;
    }
    if (needed) *needed = w;
    if (w > cap_ids) { g_err = "out_ids too small"; return GM_ERR_CAPACITY; }
    return GM_OK;
}

// ---- retained-message tree ----------------------------------------------------------------------------
int32_t gm_retain_set(gm_engine* e, const char* topic, uint32_t len, uint32_t value, int32_t* had_old, uint32_t* old_value) {
    if (!e || (!topic && len)) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    bool had = false; u32 old = 0;
    int st = e->rtree.set(topic, len, value, &had, &old);
    if (had_old) *had_old = had ? 1 : 0;
    if (old_value && had) *old_value = old;
    return map_parse(st, "gm_retain_set");
}

int32_t gm_retain_remove(gm_engine* e, const char* topic, uint32_t len, int32_t* had_old, uint32_t* old_value) {
    if (!e || (!topic && len)) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    bool had = false; u32 old = 0;
    int st = e->rtree.remove(topic, len, &had, &old);
    if (had_old) *had_old = had ? 1 : 0;
    if (old_value && had) *old_value = old;
    return map_parse(st, "gm_retain_remove");
}

int32_t gm_retain_remove_batch(gm_engine* e, const char* blob, const uint32_t* offsets, uint64_t n, uint32_t* old_values, uint64_t* n_removed) {
    if (!e || (n && (!blob || !offsets))) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    uint64_t removed = 0;
    for (uint64_t i = 0; i < n; ++i) {
        bool had = false; u32 old = 0;
        const int st = e->rtree.remove(blob + offsets[i], offsets[i + 1] - offsets[i], &had, &old);
        if (old_values) old_values[i] = (st == PARSE_OK && had) ? old : 0xFFFFFFFFu;
        removed += (st == PARSE_OK && had) ? 1 : 0;
    }
    if (n_removed) *n_removed = removed;
    return GM_OK;
}

int32_t gm_retain_bulk_load(gm_engine* e, const char* blob, const uint32_t* offsets, const uint32_t* values, uint64_t n, uint64_t* n_set) {
    if (!e || (n && (!blob || !offsets || !values))) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    const uint64_t ok = e->rtree.set_batch(blob, offsets, values, n);
    if (n_set) *n_set = ok;
    return GM_OK;
}

int32_t gm_retain_match_batch_device(gm_engine* e, const void* d_blob, uint64_t blob_bytes, const uint32_t* d_offs, uint64_t n,
                                     gm_span* d_spans, uint32_t* d_ids, uint64_t cap_ids, uint64_t* needed, int32_t* d_status, void* stream) {
    if (!e || (n && (!d_offs || !d_spans || !d_status))) return GM_ERR_INVALID_ARG;
    if (needed) *needed = 0;
    if (n == 0) return GM_OK;
    if (blob_bytes > 0xFFFFFFFFull || n > 0xFFFFFFF0ull) { g_err = "filter batch too large"; return GM_ERR_TOO_LARGE; }
    if (e->flags & GM_FLAG_HOST_ONLY) { g_err = "host-only engine cannot match: there is no CPU fallback"; return GM_ERR_NO_DEVICE; }
    CUDA_TRY(cudaSetDevice(e->device));
    std::lock_guard<std::mutex> gr(e->mu_ret);      // the retained lookup's scratch is engine-wide: one lookup at a time
    { int st = auto_flush(e, true); if (st != GM_OK) return st; }
    RetainJob j;
    j.blob = d_blob; j.blob_bytes = blob_bytes; j.offs = d_offs; j.n = n; j.spans = d_spans; j.ids = d_ids; j.cap_ids = std::min<u64>(cap_ids, 0xFFFFFFFFull); j.status = d_status;
    u64 total = 0;
    int st = e->run_retain(j, static_cast<cudaStream_t>(stream), &total);
    if (st != GM_OK) return st;
    if (needed) *needed = total;
    if (total > 0xFFFFFFFFull) { g_err = "batch produces >= 2^32 ids: split it"; return GM_ERR_TOO_LARGE; }
    if (total > cap_ids) { g_err = "out_ids too small"; return GM_ERR_CAPACITY; }
    return GM_OK;
}

int32_t gm_retain_match_batch(gm_engine* e, const char* blob, const uint32_t* offsets, uint64_t n, gm_span* out_spans, uint32_t* out_ids,
                              uint64_t cap_ids, uint64_t* needed, int32_t* status) {
    if (!e || (n && (!offsets || !out_spans || !status)) || (cap_ids && !out_ids)) return GM_ERR_INVALID_ARG;
    if (needed) *needed = 0;
    if (n == 0) return GM_OK;
    if (n > 0xFFFFFFF0ull) { g_err = "filter batch too large"; return GM_ERR_TOO_LARGE; }
    if (e->flags & GM_FLAG_HOST_ONLY) { g_err = "host-only engine cannot match: there is no CPU fallback"; return GM_ERR_NO_DEVICE; }
    CUDA_TRY(cudaSetDevice(e->device));
    std::lock_guard<std::mutex> gr(e->mu_ret);
    { int st = auto_flush(e, true); if (st != GM_OK) return st; }
    const u64 blob_bytes = offsets[n];
    MatchCtx& c = e->devctx;                          // staging of the retained host call (guarded by mu_ret)
    cudaStream_t s = c.sc;
    DevBuf &rb = e->d_rstage[0], &ro = e->d_rstage[1], &rs = e->d_rstage[2], &rt = e->d_rstage[3], &ri = e->d_rstage[4];
    CUDA_TRY(rb.ensure(blob_bytes + 16));
    CUDA_TRY(ro.ensure((n + 1) * sizeof(u32)));
    CUDA_TRY(rs.ensure(n * sizeof(gm_span)));
    CUDA_TRY(rt.ensure(n * sizeof(int32_t)));
    CUDA_TRY(ri.ensure(std::max<u64>(cap_ids, 1) * sizeof(u32)));
    if (blob_bytes) CUDA_TRY(cudaMemcpyAsync(rb.p, blob, blob_bytes, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(ro.p, offsets, (n + 1) * sizeof(u32), cudaMemcpyHostToDevice, s));
    RetainJob j;
    j.blob = rb.p; j.blob_bytes = blob_bytes; j.offs = ro.as<u32>(); j.n = n; j.spans = rs.as<gm_span>(); j.ids = ri.as<u32>();
    j.cap_ids = std::min<u64>(cap_ids, 0xFFFFFFFFull); j.status = rt.as<int32_t>();
    u64 total = 0;
    int st = e->run_retain(j, s, &total);
    if (st != GM_OK) return st;
    CUDA_TRY(cudaMemcpyAsync(status, rt.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(out_spans, rs.p, n * sizeof(gm_span), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    if (needed) *needed = total;
    if (total > 0xFFFFFFFFull) { g_err = "batch produces >= 2^32 ids: split it"; return GM_ERR_TOO_LARGE; }
    if (total > cap_ids) { g_err = "out_ids too small"; return GM_ERR_CAPACITY; }
    if (total) {
        CUDA_TRY(cudaMemcpyAsync(out_ids, ri.p, total * sizeof(u32), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
    }
    return GM_OK;
}

// ---- GpuRouter (router_host.cpp) ------------------------------------------------------------------------
struct gm_router { GpuRouter impl; explicit gm_router(gm_engine* e) : impl(e) {} };

static GpuRouter::Id to_id(const gm_id* id) {
    GpuRouter::Id r;
    r.node_id = id->node_id; r.tag = id->tag;
    if (id->client_id) r.client_id.assign(id->client_id, id->client_len);
    return r;
}

int32_t gmr_create(gm_engine* e, gm_router** out) {
    if (!e || !out) return GM_ERR_INVALID_ARG;
    *out = new gm_router(e);
    return GM_OK;
}
void gmr_destroy(gm_router* r) { delete r; }

int32_t gmr_add(gm_router* r, const char* filter, uint32_t len, const gm_id* id, const gm_sub_opts* opts) {
    if (!r || !id || (!filter && len)) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(r->impl.mu);
    GpuRouter::Opts o;
    if (opts) { o.qos = opts->qos; o.is_v5 = opts->is_v5; o.no_local = opts->no_local; o.sub_id = opts->sub_id; if (opts->shared_group) o.group.assign(opts->shared_group, opts->shared_group_len); }
    return r->impl.add(filter, len, to_id(id), o);
}
int32_t gmr_remove(gm_router* r, const char* filter, uint32_t len, const gm_id* id, int32_t* removed) {
    if (!r || !id || (!filter && len)) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(r->impl.mu);
    bool rm = false;
    int32_t rc = r->impl.remove(filter, len, to_id(id), &rm);
    if (removed) *removed = rm ? 1 : 0;
    return rc;
}
int32_t gmr_add_batch_numbered(gm_router* r, const char* blob, const uint32_t* offsets, uint64_t n, const uint64_t* node_ids, const uint32_t* client_nums,
                               const uint8_t* flags, const uint32_t* sub_ids, uint64_t* n_added) {
    if (!r || (n && (!blob || !offsets || !client_nums))) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(r->impl.mu);
    uint64_t ok = 0;
    char cid[24];
    for (uint64_t i = 0; i < n; ++i) {
        GpuRouter::Id id;
        id.node_id = node_ids ? node_ids[i] : 1; id.tag = client_nums[i];
        id.client_id.assign(cid, static_cast<size_t>(snprintf(cid, sizeof cid, "c%u", client_nums[i])));
        GpuRouter::Opts o;
        if (flags) { o.is_v5 = flags[i] & 1; o.no_local = (flags[i] >> 1) & 1; }
        if (sub_ids) o.sub_id = sub_ids[i];
        if (r->impl.add(blob + offsets[i], offsets[i + 1] - offsets[i], id, o) == GM_OK) ++ok;
    }
    if (n_added) *n_added = ok;
    return GM_OK;
}
int32_t gmr_last_timing(gm_router* r, double* device_ms, double* host_ms) {
    if (!r) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(r->impl.mu);
    if (device_ms) *device_ms = r->impl.last_device_ms;
    if (host_ms) *host_ms = r->impl.last_host_ms;
    return GM_OK;
}
int64_t gmr_topics(gm_router* r) { return r ? r->impl.topics() : 0; }
int64_t gmr_routes(gm_router* r) { return r ? r->impl.routes() : 0; }

int32_t gmr_matches_batch(gm_router* r, const gm_id* publishers, const char* blob, const uint32_t* offs, uint64_t n, gm_span* out_spans,
                          gm_sub_relation* out_rels, uint64_t cap_rels, uint32_t* out_sub_ids, uint64_t cap_sub_ids, uint64_t* needed_rels,
                          uint64_t* needed_sub_ids, int32_t* status) {
    if (!r || (n && (!offs || !out_spans || !status))) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(r->impl.mu);
    const int32_t rc = r->impl.matches_batch(publishers, blob, offs, n, out_spans, out_rels, cap_rels, out_sub_ids, cap_sub_ids, needed_rels, needed_sub_ids, status);
    if (rc == GM_ERR_CAPACITY) g_err = "gmr_matches_batch: output too small";
    return rc;
}

int32_t gmr_matched_filters_batch(gm_router* r, const char* blob, const uint32_t* offs, uint64_t n, gm_span* out_spans, uint32_t* out_filters, uint64_t cap_filters,
                                  uint64_t* needed, int32_t* status) {
    if (!r || (n && (!offs || !out_spans || !status))) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(r->impl.mu);
    std::vector<gm_span> spans; std::vector<uint32_t> fl; std::vector<int32_t> st;
    const int32_t rc = r->impl.matched_filters_batch(blob, offs, n, spans, fl, st);
    if (rc != GM_OK) return rc;
    if (needed) *needed = fl.size();
    std::copy(st.begin(), st.end(), status);
    if (fl.size() > cap_filters) { g_err = "gmr_matched_filters_batch: output too small"; return GM_ERR_CAPACITY; }
    std::copy(spans.begin(), spans.end(), out_spans);
    std::copy(fl.begin(), fl.end(), out_filters);
    return GM_OK;
}

int32_t gmr_filter(gm_router* r, uint32_t filter_idx, const char** filter, uint32_t* filter_len, uint64_t* out_node_ids, uint32_t cap_nodes, uint32_t* n_nodes) {
    if (!r || !filter || !filter_len) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(r->impl.mu);
    const std::string* f;
    std::vector<uint64_t> nodes;
    if (!r->impl.filter(filter_idx, &f, nodes)) return GM_ERR_INVALID_ARG;
    *filter = f->data(); *filter_len = static_cast<uint32_t>(f->size());
    if (n_nodes) *n_nodes = static_cast<uint32_t>(nodes.size());
    if (out_node_ids) for (uint32_t k = 0; k < nodes.size() && k < cap_nodes; ++k) out_node_ids[k] = nodes[k];
    return GM_OK;
}

int32_t gmr_relation(gm_router* r, uint32_t handle, const char** filter, uint32_t* filter_len, const char** client, uint32_t* client_len) {
    if (!r || !filter || !filter_len || !client || !client_len) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(r->impl.mu);
    const std::string *f, *c;
    if (!r->impl.relation(handle, &f, &c)) return GM_ERR_INVALID_ARG;
    *filter = f->data(); *filter_len = static_cast<uint32_t>(f->size()); *client = c->data(); *client_len = static_cast<uint32_t>(c->size());
    return GM_OK;
}

// ---- multi-GPU: NCCL communicator, device partition of a mixed batch, all-gatherv of match lists (comm.cuh) ----------
#define NCCL_TRY(expr)                                                                          \
    do {                                                                                        \
        ncclResult_t _r = (expr);                                                               \
        if (_r != ncclSuccess) { g_err = std::string(#expr) + ": " + nc.GetErrorString(_r); return GM_ERR_COMM; } \
    } while (0)

int32_t gm_comm_unique_id(uint8_t* out_id) {
    if (!out_id) return GM_ERR_INVALID_ARG;
    NcclApi& nc = NcclApi::get();
    if (!nc.ok()) { g_err = nc.error; return GM_ERR_COMM; }
    static_assert(GM_COMM_ID_BYTES == NCCL_UNIQUE_ID_BYTES, "gm_comm_unique_id hands out an ncclUniqueId");
    ncclUniqueId id;
    NCCL_TRY(nc.GetUniqueId(&id));
    std::memcpy(out_id, id.internal, GM_COMM_ID_BYTES);
    return GM_OK;
}

int32_t gm_comm_init(gm_engine* e, const uint8_t* id128, uint32_t rank, uint32_t world) {
    if (!e || !id128 || world == 0 || rank >= world) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu_dev);
    if (e->flags & GM_FLAG_HOST_ONLY) { g_err = "host-only engine has no device to communicate from"; return GM_ERR_NO_DEVICE; }
    NcclApi& nc = NcclApi::get();
    if (!nc.ok()) { g_err = nc.error; return GM_ERR_COMM; }
    CUDA_TRY(cudaSetDevice(e->device));
    if (e->comm) { nc.CommDestroy(e->comm); e->comm = nullptr; }
    ncclUniqueId id;
    std::memcpy(id.internal, id128, GM_COMM_ID_BYTES);
    NCCL_TRY(nc.CommInitRank(&e->comm, static_cast<int>(world), id, static_cast<int>(rank)));
    e->comm_rank = rank; e->comm_world = world;
    CUDA_TRY(e->d_comm.ensure((2 + 2 * static_cast<size_t>(world)) * sizeof(unsigned long long) + (static_cast<size_t>(world) + 2) * sizeof(u32)));
    if (e->h_comm) { cudaFreeHost(e->h_comm); e->h_comm = nullptr; }
    CUDA_TRY(cudaMallocHost(&e->h_comm, (2 * static_cast<size_t>(world) + 64) * sizeof(unsigned long long)));
    return GM_OK;
}

int32_t gm_comm_destroy(gm_engine* e) {
    if (!e) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu_dev);
    if (e->comm) { cudaSetDevice(e->device); NcclApi::get().CommDestroy(e->comm); e->comm = nullptr; }
    e->comm_world = 1; e->comm_rank = 0;
    return GM_OK;
}

int32_t gm_partition_batch_device(gm_engine* e, const void* d_blob, uint64_t blob_bytes, const uint32_t* d_offsets, uint64_t n, uint32_t n_shards,
                                  uint32_t rank, uint32_t* d_sel, uint32_t* d_shard, uint64_t* n_local, uint64_t* shard_counts, void* stream) {
    if (!e || !n_local || n_shards == 0 || n_shards > 4096 || rank >= n_shards || (n && (!d_blob || !d_offsets || !d_sel))) return GM_ERR_INVALID_ARG;
    if (blob_bytes > 0xFFFFFFFFull || n > 0xFFFFFFF0ull) { g_err = "batch too large"; return GM_ERR_TOO_LARGE; }
    *n_local = 0;
    std::lock_guard<std::mutex> g(e->mu_dev);
    if (e->flags & GM_FLAG_HOST_ONLY) { g_err = "host-only engine has no device"; return GM_ERR_NO_DEVICE; }
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    DevBuf& cb = e->d_part;
    CUDA_TRY(cb.ensure((static_cast<size_t>(n_shards) + 1) * sizeof(u32)));
    CUDA_TRY(cudaMemsetAsync(cb.p, 0, (static_cast<size_t>(n_shards) + 1) * sizeof(u32), s));
    if (n) {
        k_partition<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(static_cast<const u8*>(d_blob), static_cast<u32>(blob_bytes), d_offsets, static_cast<u32>(n),
                                                                            n_shards, rank, d_sel, d_shard, cb.as<u32>());
        e->launches++;
        CUDA_TRY(cudaGetLastError());
    }
    std::vector<u32> h(n_shards + 1);
    CUDA_TRY(cudaMemcpyAsync(h.data(), cb.p, h.size() * sizeof(u32), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    *n_local = h[n_shards];
    if (shard_counts) for (u32 r = 0; r < n_shards; ++r) shard_counts[r] = h[r];
    return GM_OK;
}

int32_t gm_allgatherv_device(gm_engine* e, const uint32_t* d_index, const gm_span* d_spans, uint64_t k, const uint32_t* d_ids, const uint64_t* d_m,
                             uint32_t* d_all_index, gm_span* d_all_spans, uint64_t cap_topics, uint32_t* d_all_ids, uint64_t cap_ids, uint64_t* sizes,
                             void* stream) {
    if (!e || !d_m || !sizes || (k && (!d_index || !d_spans)) || !d_all_index || !d_all_spans || !d_all_ids) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu_dev);
    if (!e->comm) { g_err = "gm_allgatherv_device: call gm_comm_init first"; return GM_ERR_INVALID_ARG; }
    NcclApi& nc = NcclApi::get();
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const u32 W = e->comm_world, R = e->comm_rank;
    unsigned long long* d_send = e->d_comm.as<unsigned long long>();
    unsigned long long* d_all = d_send + 2;
    // 1. sizes: (k, m) of every rank.  m lives on the device (the match kernels' cursor): no host hop before the exchange.
    k_comm_sizes<<<1, 1, 0, s>>>(d_send, k, reinterpret_cast<const unsigned long long*>(d_m));
    NCCL_TRY(nc.AllGather(d_send, d_all, 2, ncclUint64, e->comm, s));
    CUDA_TRY(cudaMemcpyAsync(e->h_comm, d_all, 2 * static_cast<size_t>(W) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));      // NCCL needs the counts on the host: the one host synchronisation of the collective
    u64 K = 0, M = 0;
    for (u32 r = 0; r < W; ++r) { sizes[2 * r] = e->h_comm[2 * r]; sizes[2 * r + 1] = e->h_comm[2 * r + 1]; K += sizes[2 * r]; M += sizes[2 * r + 1]; }
    if (M > 0xFFFFFFFFull) { g_err = "gathered match lists exceed 2^32 ids: split the batch"; return GM_ERR_TOO_LARGE; }
    if (K > cap_topics || M > cap_ids) { g_err = "gm_allgatherv_device: output too small (sizes[] holds what every rank contributes)"; return GM_ERR_CAPACITY; }
    // 2. one grouped launch, straight out of the buffers the match kernels wrote.  Default: point-to-point (every rank sends
    //    its three arrays to every peer and receives theirs — each pair has its own NVSwitch path); GM_ALLGATHERV=bcast
    //    selects one ncclBroadcast per (rank, array) instead (A/B, profiles/).
    std::vector<u64> kof(W + 1, 0), mof(W + 1, 0);
    for (u32 r = 0; r < W; ++r) { kof[r + 1] = kof[r] + sizes[2 * r]; mof[r + 1] = mof[r] + sizes[2 * r + 1]; }
    if (e->knobs.gather_bcast) {
        NCCL_TRY(nc.GroupStart());
        for (u32 r = 0; r < W; ++r) {
            const u64 kr = sizes[2 * r], mr = sizes[2 * r + 1];
            if (kr) {
                NCCL_TRY(nc.Broadcast(r == R ? static_cast<const void*>(d_index) : d_all_index + kof[r], d_all_index + kof[r], kr, ncclUint32, static_cast<int>(r), e->comm, s));
                NCCL_TRY(nc.Broadcast(r == R ? static_cast<const void*>(d_spans) : d_all_spans + kof[r], d_all_spans + kof[r], kr, ncclUint64, static_cast<int>(r), e->comm, s));
            }
            if (mr) NCCL_TRY(nc.Broadcast(r == R ? static_cast<const void*>(d_ids) : d_all_ids + mof[r], d_all_ids + mof[r], mr, ncclUint32, static_cast<int>(r), e->comm, s));
        }
        NCCL_TRY(nc.GroupEnd());
    } else {
        const u64 kR = sizes[2 * R], mR = sizes[2 * R + 1];
        // own part: device-to-device copies on the same stream
        if (kR) {
            CUDA_TRY(cudaMemcpyAsync(d_all_index + kof[R], d_index, kR * sizeof(u32), cudaMemcpyDeviceToDevice, s));
            CUDA_TRY(cudaMemcpyAsync(d_all_spans + kof[R], d_spans, kR * sizeof(gm_span), cudaMemcpyDeviceToDevice, s));
        }
        if (mR) CUDA_TRY(cudaMemcpyAsync(d_all_ids + mof[R], d_ids, mR * sizeof(u32), cudaMemcpyDeviceToDevice, s));
        if (W > 1) {
            NCCL_TRY(nc.GroupStart());
            for (u32 d = 1; d < W; ++d) {
                const u32 to = (R + d) % W, from = (R + W - d) % W;          // staggered pairs: no two ranks target the same peer first
                if (kR) { NCCL_TRY(nc.Send(d_index, kR, ncclUint32, static_cast<int>(to), e->comm, s)); NCCL_TRY(nc.Send(d_spans, kR, ncclUint64, static_cast<int>(to), e->comm, s)); }
                if (mR) NCCL_TRY(nc.Send(d_ids, mR, ncclUint32, static_cast<int>(to), e->comm, s));
                const u64 kf = sizes[2 * from], mf = sizes[2 * from + 1];
                if (kf) { NCCL_TRY(nc.Recv(d_all_index + kof[from], kf, ncclUint32, static_cast<int>(from), e->comm, s)); NCCL_TRY(nc.Recv(d_all_spans + kof[from], kf, ncclUint64, static_cast<int>(from), e->comm, s)); }
                if (mf) NCCL_TRY(nc.Recv(d_all_ids + mof[from], mf, ncclUint32, static_cast<int>(from), e->comm, s));
            }
            NCCL_TRY(nc.GroupEnd());
        }
    }
    // 3. spans of rank r index rank r's ids: re-base them onto the gathered id array
    if (K) { k_rebase_spans<<<static_cast<unsigned>((K + 255) / 256), 256, 0, s>>>(reinterpret_cast<uint2*>(d_all_spans), d_all, W, static_cast<u32>(K)); e->launches++; }
    e->launches++;
    CUDA_TRY(cudaGetLastError());
    return GM_OK;
}

// ---- fused gather over peer memory ------------------------------------------------------------------------------------
int32_t gm_gather_create(gm_engine* e, uint32_t world, uint32_t rank, uint64_t slab_topics, uint64_t slab_ids, uint8_t* out_handle) {
    if (!e || !out_handle || world == 0 || world > 8 || rank >= world || slab_topics == 0 || slab_ids == 0) return GM_ERR_INVALID_ARG;
    const GatherLayout layout = gather_layout(world, slab_topics, slab_ids);
    if (layout.slab_ids * world > 0xFFFFFFFFull || layout.slab_topics * world > 0xFFFFFFF0ull) { g_err = "gathered arrays exceed 32-bit offsets"; return GM_ERR_TOO_LARGE; }
    if (e->flags & GM_FLAG_HOST_ONLY) { g_err = "host-only engine has no device"; return GM_ERR_NO_DEVICE; }
    std::lock_guard<std::mutex> g(e->mu_dev);
    CUDA_TRY(cudaSetDevice(e->device));
    gm_engine::Gather& G = e->gather;
    if (G.block) { g_err = "gm_gather_create: already created (gm_gather_destroy first)"; return GM_ERR_INVALID_ARG; }
    static_cast<GatherLayout&>(G) = layout;
    G.rank = rank; G.epoch = 0; G.connected = false;
    void* p = nullptr;
    CUDA_TRY(cudaMalloc(&p, G.bytes));
    G.block = static_cast<char*>(p);
    CUDA_TRY(cudaMemset(G.block + G.off_counts, 0, G.bytes - G.off_counts));
    const unsigned long long geo[3] = {world, G.slab_topics, G.slab_ids};       // the layout must be the same on every rank: checked at connect
    CUDA_TRY(cudaMemcpy(G.block, geo, sizeof(geo), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaDeviceSynchronize());
    cudaIpcMemHandle_t h;
    static_assert(sizeof(h) == GM_IPC_HANDLE_BYTES, "gm_gather_create hands out a cudaIpcMemHandle_t");
    CUDA_TRY(cudaIpcGetMemHandle(&h, G.block));
    std::memcpy(out_handle, &h, sizeof(h));
    return GM_OK;
}

int32_t gm_gather_connect(gm_engine* e, const uint8_t* handles) {
    if (!e || !handles) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu_dev);
    gm_engine::Gather& G = e->gather;
    if (!G.block) { g_err = "gm_gather_connect: gm_gather_create first"; return GM_ERR_INVALID_ARG; }
    CUDA_TRY(cudaSetDevice(e->device));
    for (u32 w = 0; w < G.world; ++w) {
        if (w == G.rank) { G.peer[w] = G.block; continue; }
        cudaIpcMemHandle_t h;
        std::memcpy(&h, handles + static_cast<size_t>(w) * GM_IPC_HANDLE_BYTES, sizeof(h));
        void* p = nullptr;
        cudaError_t ce = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (ce != cudaSuccess) { g_err = std::string("cudaIpcOpenMemHandle (peer-to-peer access between the ranks' GPUs is required): ") + cudaGetErrorString(ce); cudaGetLastError(); return GM_ERR_COMM; }
        G.peer[w] = static_cast<char*>(p);
        unsigned long long geo[3] = {0, 0, 0};
        CUDA_TRY(cudaMemcpy(geo, G.peer[w], sizeof(geo), cudaMemcpyDeviceToHost));
        if (geo[0] != G.world || geo[1] != G.slab_topics || geo[2] != G.slab_ids) {
            g_err = "gm_gather_connect: rank " + std::to_string(w) + " created its block with a different (world, slab_topics, slab_ids): the layout must be identical on every rank";
            return GM_ERR_INVALID_ARG;
        }
    }
    void* ptrs[24] = {};
    for (u32 w = 0; w < G.world; ++w) { ptrs[w] = G.peer[w] + G.off_counts; ptrs[8 + w] = G.peer[w] + G.off_flags; ptrs[16 + w] = G.peer[w]; }
    CUDA_TRY(G.d_ptrs.ensure(sizeof(ptrs)));
    CUDA_TRY(cudaMemcpy(G.d_ptrs.p, ptrs, sizeof(ptrs), cudaMemcpyHostToDevice));
    G.connected = true;
    return GM_OK;
}

int32_t gm_match_gather_device(gm_engine* e, const void* d_blob, uint64_t blob_bytes, const uint32_t* d_offsets, uint64_t n_entries, const uint32_t* d_sel,
                               uint64_t n, int32_t* d_status, void* stream) {
    if (!e || (n && (!d_offsets || !d_status))) return GM_ERR_INVALID_ARG;
    if (blob_bytes > 0xFFFFFFFFull) { g_err = "topic blob >= 4 GiB"; return GM_ERR_TOO_LARGE; }
    if (d_sel && n > n_entries) return GM_ERR_INVALID_ARG;
    gm_engine::Gather& G = e->gather;
    if (!G.connected) { g_err = "gm_match_gather_device: gm_gather_create + gm_gather_connect first"; return GM_ERR_INVALID_ARG; }
    if (n > G.slab_topics) { g_err = "gm_match_gather_device: more rows than this rank's slab holds"; return GM_ERR_CAPACITY; }
    CUDA_TRY(cudaSetDevice(e->device));
    { int st = auto_flush(e); if (st != GM_OK) return st; }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    std::lock_guard<std::mutex> gd(e->mu_dev);
    MatchJob j;
    j.blob = d_blob; j.blob_bytes = blob_bytes; j.offs = d_offsets; j.sel = d_sel; j.n = n; j.cap = G.slab_ids; j.status = d_status;
    j.mode = MatchJob::GATHER; j.gather = &G; j.blocks = G.peer; j.rank = G.rank;
    int st = e->enqueue_match(e->devctx, j, s);
    if (st != GM_OK) return st;
    // contribution (rows, ids) into every rank's counts + the epoch barrier: when it has passed on a rank, all ranks' data is there
    G.epoch++;
    const unsigned long long* d_m = n ? &e->devctx.d_ctrl.as<Ctrl>()->cursor : nullptr;
    if (!d_m) { CUDA_TRY(e->devctx.d_ctrl.ensure(sizeof(Ctrl))); CUDA_TRY(cudaMemsetAsync(e->devctx.d_ctrl.p, 0, sizeof(Ctrl), s)); d_m = &e->devctx.d_ctrl.as<Ctrl>()->cursor; }
    void** dp = G.d_ptrs.as<void*>();
    CudaLauncher l{s, nullptr, &e->ring_n, &e->launches};
    if ((st = gather_push(l, G, e->knobs.gather_direct, static_cast<u32>(e->num_sms), reinterpret_cast<char* const*>(dp + 16), G.rank, n, d_m)) != GM_OK) return st;
    if ((st = gather_finish(l, G, G.block, reinterpret_cast<unsigned long long* const*>(dp), reinterpret_cast<u32* const*>(dp + 8), G.rank, n, d_m, G.epoch)) != GM_OK) return st;
    CUDA_TRY(cudaEventRecord(e->devctx.ev_done, s));
    e->devctx.recorded = true;
    return GM_OK;
}

int32_t gm_gather_get(gm_engine* e, gm_gather_view* out, void* stream) {
    if (!e || !out) return GM_ERR_INVALID_ARG;
    gm_engine::Gather& G = e->gather;
    if (!G.block) return GM_ERR_INVALID_ARG;
    CUDA_TRY(cudaSetDevice(e->device));
    CUDA_TRY(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    u32 err = 0;
    CUDA_TRY(cudaMemcpy(&err, G.block + G.off_flags + 32 * 4, 4, cudaMemcpyDeviceToHost));
    out->d_ids = reinterpret_cast<const uint32_t*>(G.block + GatherLayout::off_ids); out->d_spans = reinterpret_cast<const gm_span*>(G.block + G.off_spans);
    out->d_index = reinterpret_cast<const uint32_t*>(G.block + G.off_index); out->d_counts = reinterpret_cast<const uint64_t*>(G.block + G.off_counts);
    out->slab_topics = G.slab_topics; out->slab_ids = G.slab_ids; out->world = G.world; out->rank = G.rank;
    if (err) { g_err = "fused gather: a rank did not reach the end-of-step barrier"; return GM_ERR_COMM; }
    return GM_OK;
}

int32_t gm_gather_destroy(gm_engine* e) {
    if (!e) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu_dev);
    gm_engine::Gather& G = e->gather;
    if (!G.block) return GM_OK;
    cudaSetDevice(e->device);
    cudaDeviceSynchronize();
    for (u32 w = 0; w < G.world; ++w) if (w != G.rank && G.peer[w]) cudaIpcCloseMemHandle(G.peer[w]);
    cudaFree(G.block);
    G = gm_engine::Gather{};
    return GM_OK;
}

int32_t gm_device_read(gm_engine* e, const void* d_src, void* h_dst, uint64_t bytes) {
    if (!e || !d_src || !h_dst) return GM_ERR_INVALID_ARG;
    CUDA_TRY(cudaSetDevice(e->device));
    CUDA_TRY(cudaMemcpy(h_dst, d_src, bytes, cudaMemcpyDeviceToHost));
    return GM_OK;
}

int32_t gm_relations_expand_device(gm_engine* e, const gm_span* d_spans, const uint32_t* d_ids, uint64_t n, const uint32_t* d_publishers,
                                   const gm_rel* d_rels, uint64_t n_rels, const gm_rel_out* o, void* stream) {
    if (!e || !o || !o->d_needed || (n && (!d_spans || !o->d_spans || !o->d_status))) return GM_ERR_INVALID_ARG;
    if (n > 0xFFFFFFF0ull || n_rels > 0xFFFFFFFFull) { g_err = "batch too large"; return GM_ERR_TOO_LARGE; }
    if (e->flags & GM_FLAG_HOST_ONLY) { g_err = "host-only engine has no device"; return GM_ERR_NO_DEVICE; }
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CUDA_TRY(cudaMemsetAsync(o->d_needed, 0, 3 * sizeof(uint64_t), s));
    if (n == 0) return GM_OK;
    RelParams rp{};
    rp.spans = reinterpret_cast<const uint2*>(d_spans); rp.ids = d_ids; rp.n = static_cast<u32>(n); rp.pubs = d_publishers;
    rp.rels = d_rels; rp.n_rels = static_cast<u32>(n_rels);
    rp.out_spans = reinterpret_cast<uint2*>(o->d_spans); rp.out_rels = o->d_rels; rp.cap_rels = o->cap_rels;
    rp.out_sub_ids = o->d_sub_ids; rp.cap_sub_ids = o->cap_sub_ids;
    rp.needed = reinterpret_cast<unsigned long long*>(o->d_needed); rp.status = o->d_status;
    const unsigned grid = static_cast<unsigned>(std::min<u64>((n + 7) / 8, static_cast<u64>(e->num_sms) * 8));
    k_relations<<<grid, 256, 0, s>>>(rp);
    { std::lock_guard<std::mutex> g(e->mu_dev); e->launches++; }
    CUDA_TRY(cudaGetLastError());
    return GM_OK;
}

int32_t gm_tokenize_batch(gm_engine* e, const char* blob, const uint32_t* offsets, uint64_t n, uint32_t max_tok, uint32_t* out_tokens, uint32_t* out_meta) {
    if (!e || !max_tok || (n && (!offsets || !out_tokens || !out_meta))) return GM_ERR_INVALID_ARG;
    if (n == 0) return GM_OK;
    if (e->flags & GM_FLAG_HOST_ONLY) { g_err = "host-only engine cannot match: there is no CPU fallback"; return GM_ERR_NO_DEVICE; }
    CUDA_TRY(cudaSetDevice(e->device));
    { std::lock_guard<std::mutex> g(e->mu); int st = e->flush_locked(); if (st != GM_OK) return st; }
    std::lock_guard<std::mutex> g(e->mu_dev);
    cudaStream_t s = e->devctx.sc;
    DevBuf t_blob, t_offs;
    const u64 blob_bytes = offsets[n];
    DevBuf tok, tok8, meta, stat;
    CUDA_TRY(t_blob.ensure(blob_bytes + 16));
    CUDA_TRY(t_offs.ensure((n + 1) * sizeof(u32)));
    CUDA_TRY(tok.ensure(static_cast<size_t>(max_tok) * n * sizeof(u32)));
    CUDA_TRY(tok8.ensure(static_cast<size_t>(n) * TOK8 * sizeof(u32)));
    CUDA_TRY(meta.ensure(n * sizeof(u32)));
    CUDA_TRY(stat.ensure(n * sizeof(int)));
    if (blob_bytes) CUDA_TRY(cudaMemcpyAsync(t_blob.p, blob, blob_bytes, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(t_offs.p, offsets, (n + 1) * sizeof(u32), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemsetAsync(tok.p, 0, static_cast<size_t>(max_tok) * n * sizeof(u32), s));
    CUDA_TRY(cudaStreamWaitEvent(s, e->ev_flush, 0));
    auto k1 = e->knobs.tok_bulk ? k_tokenize<true> : k_tokenize<false>;
    k1<<<(static_cast<u32>(n) + TOK_THREADS - 1) / TOK_THREADS, TOK_THREADS, 0, s>>>(
        t_blob.as<u8>(), static_cast<u32>(blob_bytes), static_cast<u32>((blob_bytes + 15) & ~u64(15)), t_offs.as<u32>(), nullptr, static_cast<u32>(n), nullptr, e->dev_view, max_tok, tok8.as<u32>(), tok.as<u32>(), meta.as<u32>(), stat.as<int>(), nullptr, nullptr, 0u, 0u);
    e->launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out_tokens, tok.p, static_cast<size_t>(max_tok) * n * sizeof(u32), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(out_meta, meta.p, n * sizeof(u32), cudaMemcpyDeviceToHost, s));
    std::vector<u32> rows(static_cast<size_t>(n) * TOK8);
    CUDA_TRY(cudaMemcpyAsync(rows.data(), tok8.p, rows.size() * sizeof(u32), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    for (uint64_t i = 0; i < n; ++i)          // levels 0..7 live in the per-topic row; present them level-major too
        for (u32 l = 0; l < TOK8 && l < max_tok; ++l) out_tokens[static_cast<size_t>(l) * n + i] = rows[i * TOK8 + l];
    return GM_OK;
}

int32_t gm_get_stats(gm_engine* e, gm_stats* out) {
    if (!e || !out) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    std::memset(out, 0, sizeof(*out));
    const HostTrie& t = e->trie;
    out->values = t.values_size(); out->nodes = t.nodes_size(); out->device_nodes = t.node_count() - 1;
    out->edges = t.edge_count(); out->edge_slots = t.edges.size();
    out->dict_entries = t.dict_count(); out->dict_slots = t.dict.size();
    out->plus_nodes = t.plus_count();
    out->value_words = t.values.size(); out->garbage_value_words = t.garbage_values;
    out->device_bytes = e->d_edges.cap + e->d_ranges.cap + e->d_values.cap + e->d_dict.cap + e->d_pool.cap;
    out->max_depth = t.max_depth;
    out->pending = (t.any_dirty() || e->rtree.dirty) ? 1 : 0;
    out->retained_values = e->rtree.values_size(); out->retained_nodes = e->rtree.nodes_size();
    out->device_bytes += e->d_rnodes.cap + e->d_rkids.cap + e->d_redges.cap + e->d_rvals.cap;
    return GM_OK;
}

int32_t gm_kernel_ms_ring(gm_engine* e, float* out_ms, uint32_t max_calls, uint32_t* n_calls) {
    if (!e || !out_ms || !n_calls) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu_dev);
    *n_calls = 0;
    if (e->flags & GM_FLAG_HOST_ONLY) return GM_OK;
    CUDA_TRY(cudaSetDevice(e->device));
    const u64 have = std::min<u64>(e->ring_n, gm_engine::RING);
    const u64 take = std::min<u64>(have, max_calls);
    for (u64 k = 0; k < take; ++k) {                       // oldest first
        cudaEvent_t* ev = e->ev_ring[(e->ring_n - take + k) % gm_engine::RING];
        CUDA_TRY(cudaEventSynchronize(ev[3]));
        for (int j = 0; j < 3; ++j) CUDA_TRY(cudaEventElapsedTime(&out_ms[3 * k + j], ev[j], ev[j + 1]));
    }
    *n_calls = static_cast<uint32_t>(take);
    return GM_OK;
}

uint64_t gm_kernel_launches(gm_engine* e) { return e ? e->launches : 0; }

int32_t gm_debug_table(gm_engine* e, uint32_t which, const void** ptr, uint64_t* count) {
    if (!e || !ptr || !count) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    e->trie.sync();
    const HostTrie& t = e->trie;
    static thread_local uint32_t root[8];
    static thread_local uint64_t rstat[6];
    switch (which) {
        case 0: *ptr = t.edges.data(); *count = t.edges.size(); break;
        case 2: *ptr = t.ranges.data(); *count = t.ranges.size(); break;
        case 3: *ptr = t.values.data(); *count = t.values.size(); break;
        case 4: *ptr = t.dict.data(); *count = t.dict.size(); break;
        case 5: *ptr = t.pool.data(); *count = t.pool.size(); break;
        case 6: root[0] = t.root_plus; root[1] = t.root_hash_ref; root[2] = t.root_mask; root[3] = t.max_depth; root[4] = t.root_hash_cnt;
                root[5] = t.win_mask(); root[6] = t.win_shift(); root[7] = t.nwin_mask(); *ptr = root; *count = 8; break;
        case 12: *ptr = t.cfilter.data(); *count = t.cfilter.size(); break;
        case 10: e->rtree.prepare_flush(); *ptr = e->rtree.redges.data(); *count = e->rtree.redges.size(); break;
        case 11: e->rtree.debug_stats(rstat); *ptr = rstat; *count = 6; break;
        case 7: e->rtree.prepare_flush(); *ptr = e->rtree.rnodes.data(); *count = e->rtree.rnodes.size(); break;
        case 8: e->rtree.prepare_flush(); *ptr = e->rtree.rkids.data(); *count = e->rtree.rkids.size(); break;
        case 9: e->rtree.prepare_flush(); *ptr = e->rtree.rvals.data(); *count = e->rtree.rvals.size(); break;
        default: return GM_ERR_INVALID_ARG;
    }
    return GM_OK;
}

int32_t gm_debug_knob(gm_engine* e, const char* name, int64_t value) {
    if (!e || !name) return GM_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu_dev);
    const std::string k(name);
    if (k == "tile_chunk" && value >= 1 && value <= 1024) e->knobs.tile_chunk = static_cast<u32>(value);
    else if (k == "k2_ctas" && value >= 0 && value <= 8) e->knobs.k2_ctas = static_cast<int>(value);
    else if (k == "sorted_rows") e->knobs.sorted_rows = value != 0;
    else if (k == "bucket_bits" && value / 100 >= 10 && value % 100 + value / 100 <= int64_t(MAX_BUCKET_BITS)) { e->knobs.site_bits = static_cast<u32>(value / 100); e->knobs.sub_bits = static_cast<u32>(value % 100); }
    else if (k == "diag_flags") e->knobs.diag_flags = static_cast<u32>(value);
    else if (k == "tok_bulk") e->knobs.tok_bulk = value != 0;
    else if (k == "small_graphs") e->knobs.small_graphs = value != 0;
    else if (k == "gather_bcast") e->knobs.gather_bcast = value != 0;
    else if (k == "gather_direct") e->knobs.gather_direct = value != 0;
    else if (k == "retain_stats") e->knobs.retain_stats = value != 0;
    else if (k == "e2e_chunk" && value >= 1024) e->knobs.e2e_chunk = static_cast<u32>(value);
    else return GM_ERR_INVALID_ARG;
    return GM_OK;
}

uint32_t gm_shard_of(const char* s, uint32_t len, uint32_t n_shards) {
    if (!s || n_shards == 0) return 0xFFFFFFFFu;
    uint32_t l0 = 0;
    while (l0 < len && s[l0] != '/') ++l0;
    if (l0 == 1 && (s[0] == '+' || s[0] == '#')) return 0xFFFFFFFFu;
    return shard_of_hash(HostTrie::level0_hash(s, len), n_shards);
}

int32_t gm_shard_of_batch(const char* blob, const uint32_t* offsets, uint64_t n, uint32_t n_shards, uint32_t* out_shard) {
    if ((n && (!blob || !offsets || !out_shard)) || n_shards == 0) return GM_ERR_INVALID_ARG;
    for (uint64_t i = 0; i < n; ++i) out_shard[i] = gm_shard_of(blob + offsets[i], offsets[i + 1] - offsets[i], n_shards);
    return GM_OK;
}

// ---- NUMA placement of the host side (2-socket GPU servers: a pinned buffer on the far socket halves the PCIe rate and
//      makes 8 ranks contend for the inter-socket link) ------------------------------------------------------------------
static int device_numa_node(int device) {
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) return -1;
    for (char* c = bus; *c; ++c) *c = static_cast<char>(tolower(*c));
    const std::string path = std::string("/sys/bus/pci/devices/") + bus + "/numa_node";
    FILE* f = fopen(path.c_str(), "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    return node;
}

int32_t gm_device_numa_node(int32_t device) {
    if (device < 0 && cudaGetDevice(&device) != cudaSuccess) return -1;
    return device_numa_node(device);
}

int32_t gm_bind_thread_near_device(int32_t device) {
    const int node = gm_device_numa_node(device);
    if (node < 0) return GM_OK;                       // no NUMA information: nothing to do
    const std::string path = "/sys/devices/system/node/node" + std::to_string(node) + "/cpulist";
    FILE* f = fopen(path.c_str(), "r");
    if (!f) return GM_OK;
    char buf[4096] = {0};
    const bool ok = fgets(buf, sizeof(buf), f) != nullptr;
    fclose(f);
    if (!ok) return GM_OK;
    cpu_set_t allowed, want;
    CPU_ZERO(&allowed); CPU_ZERO(&want);
    sched_getaffinity(0, sizeof(allowed), &allowed);
    int n_want = 0;
    for (char* p = buf; *p;) {
        char* e;
        long a = strtol(p, &e, 10), b = a;
        if (e == p) break;
        if (*e == '-') { p = e + 1; b = strtol(p, &e, 10); }
        for (long k = a; k <= b && k < CPU_SETSIZE; ++k) if (CPU_ISSET(k, &allowed)) { CPU_SET(k, &want); ++n_want; }
        if (*e != ',') break;
        p = e + 1;
    }
    if (n_want) sched_setaffinity(0, sizeof(want), &want);
    unsigned long mask[16] = {0};
    mask[node / (8 * sizeof(long))] |= 1ul << (node % (8 * sizeof(long)));
    syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, static_cast<unsigned long>(node + 2));
    return GM_OK;
}

void* gm_host_alloc_near(gm_engine* e, uint64_t bytes) {
    const int node = (e && !(e->flags & GM_FLAG_HOST_ONLY)) ? device_numa_node(e->device) : -1;
    unsigned long mask[16] = {0};
    if (node >= 0) {
        mask[node / (8 * sizeof(long))] |= 1ul << (node % (8 * sizeof(long)));
        syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, static_cast<unsigned long>(node + 2));
    }
    void* p = nullptr;
    if (e && !(e->flags & GM_FLAG_HOST_ONLY)) cudaSetDevice(e->device);
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) p = nullptr;
    if (node >= 0) syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0ul);
    return p;
}

void* gm_host_alloc(uint64_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    return p;
}
void gm_host_free(void* p) { if (p) cudaFreeHost(p); }

}  // extern "C"
