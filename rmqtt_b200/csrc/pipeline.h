// What the engine enqueues on the device, decided once for libgpumqtt (engine.cu) and for the CPU emulation of the
// kernels (tests/native/emu/emu_driver.cpp): the match pipeline, the fused-gather steps, the retained lookup, and the
// shipping policy of a flush.  Plain C++: a caller supplies HOW an operation is carried out, this header decides WHAT runs.
//
// A launcher `L` (CUDA stream / CPU emulation) has four operations, each returning a GM_* code:
//   l.launch(kernel, grid, block, smem_bytes, args...)   launch (and count) one kernel
//   l.memset(ptr, value, bytes)                          device memory
//   l.copy(dst, src, bytes)                              device to device
//   l.mark(i)                                            timing point i = 0..3 of the call (no-op without timing)
// A shipper `S` (flush staging / byte image) and its buffer type `B` have four more:
//   sh.fresh(buf, src, bytes, cap_bytes)    buf becomes a new buffer of cap_bytes holding src[0, bytes)
//   sh.append(buf, off, src, bytes)         bytes at offset `off` of the current buffer (beyond what kernels can reach)
//   sh.patch(buf, host, dirty)              the listed elements of `host` into the current buffer; clears `dirty`
//   sh.capacity(buf)                        bytes of the current buffer (0: none yet)
#pragma once
#include <algorithm>
#include <array>
#include <cstddef>
#include <type_traits>
#include <vector>

#include "../../include/gpumqtt.h"
#include "comm.cuh"
#include "host_trie.h"
#include "kernels.cuh"
#include "retain_kernels.cuh"
#include "retain_tree.h"

namespace gm {

struct Ctrl {                       // device control block of a match, zeroed before every match
    unsigned long long cursor;
    unsigned long long stats[24];
    u32 slow_count;
    u32 tile_counter;
};

// fast-path geometry (see DESIGN.md): one topic per thread, 512 threads per CTA, 3 CTAs per SM (64 KB of shared memory each)
constexpr int K2_FAST_L = 8;       // levels staged in shared memory; deeper topics take the deferred kernel
constexpr int K2_THREADS = 512;
constexpr int K2_CTAS_PER_SM = 3;
constexpr u32 K2_POOL_ROWS = 24;   // matched value sets per topic beyond the 8 held in shared memory, before the topic is deferred

using MatchFastKernel = void (*)(MatchParams, Desc*, u32);

// The k_match_fast instantiations the pipeline launches: [stats][descriptors], then the gather form.  They use more
// dynamic shared memory than a CUDA launch allows by default.
template <int FAST_L = K2_FAST_L, int THREADS = K2_THREADS, int CTAS = K2_CTAS_PER_SM>
std::array<MatchFastKernel, 5> match_fast_kernels() {
    return {k_match_fast<FAST_L, THREADS, CTAS, true, false>, k_match_fast<FAST_L, THREADS, CTAS, true, true>,
            k_match_fast<FAST_L, THREADS, CTAS, false, false>, k_match_fast<FAST_L, THREADS, CTAS, false, true>,
            k_match_fast<FAST_L, THREADS, CTAS, false, false, true>};
}

// ---- fused gather: one block per rank holding every rank's slab ------------------------------------------------------------
struct GatherLayout {
    static constexpr size_t off_ids = 256;      // the block starts with a 256-byte header {world, slab_topics, slab_ids}
    u32 world = 0;
    u64 slab_topics = 0, slab_ids = 0;
    size_t off_spans = 0, off_index = 0, off_counts = 0, off_flags = 0, bytes = 0;
};

inline GatherLayout gather_layout(u32 world, u64 slab_topics, u64 slab_ids) {
    GatherLayout g;
    g.world = world;
    g.slab_topics = (slab_topics + 3) & ~u64(3); g.slab_ids = (slab_ids + 3) & ~u64(3);       // every slab starts on a 16-byte boundary
    const size_t a = 256;
    g.off_spans = (GatherLayout::off_ids + static_cast<size_t>(world) * g.slab_ids * 4 + a - 1) / a * a;
    g.off_index = g.off_spans + static_cast<size_t>(world) * g.slab_topics * 8;
    g.off_counts = (g.off_index + static_cast<size_t>(world) * g.slab_topics * 4 + a - 1) / a * a;
    g.off_flags = g.off_counts + static_cast<size_t>(world) * 16;
    g.bytes = g.off_flags + 256;
    return g;
}

// ---- the match pipeline: k_tokenize -> k_bucket_scan -> k_bucket_scatter -> k_match_fast -> k_match_slow ---------------------
struct MatchGeometry {              // the device and the engine's tuning
    u32 num_sms = 0;
    int k2_ctas = 0;                // k_match_fast CTAs per SM (outside 1..K2_CTAS_PER_SM: K2_CTAS_PER_SM)
    u32 pool_rows = K2_POOL_ROWS;
    u32 site_bits = 14, sub_bits = 0;   // locality buckets: 2^(site_bits + sub_bits)
    bool sorted_rows = true, tok_bulk = true, gather_direct = false;
    u32 diag_flags = 0, tile_chunk = 1;
};

struct MatchJob {                   // one match call; every pointer is device memory
    const void* blob = nullptr;
    u64 blob_bytes = 0, readable_bytes = 0;   // the tokeniser may read up to max(blob_bytes, readable_bytes)
    const u32* offs = nullptr;
    const u32* sel = nullptr;       // optional selection: row t matches entry sel[t] of the packed batch
    u64 n = 0;                      // rows (with `hdr`: the capacity the kernels are launched for)
    const u32* hdr = nullptr;       // small-batch graphs: {n, blob_bytes} read by the kernels at run time
    gm_span* spans = nullptr;
    void* out = nullptr;            // ids, or descriptors (uint2) in DESCRIPTORS mode
    u64 cap = 0;
    u64* d_needed = nullptr;        // optional: receives the output cursor
    int32_t* status = nullptr;
    const u32* trees = nullptr;     // optional: the tree every row is matched against
    enum Mode { IDS, DESCRIPTORS, GATHER } mode = IDS;
    bool stats = false;             // instrumented instantiations (work counters in Ctrl::stats)
    bool keep_cursor = false;       // the output cursor carries on from the previous call (chunks of one host call)
    bool timing = true;
    u32 bucket_bits = 0;            // non-zero: 2^bucket_bits locality buckets instead of the geometry's
    // GATHER mode: results go to the slab of `rank` in the blocks of every rank (blocks[w]: rank w's block)
    const GatherLayout* gather = nullptr;
    char* const* blocks = nullptr;
    u32 rank = 0;
};

struct MatchPlan {                  // launch shape and the scratch (bytes) the caller provides
    u32 n, S, site_bits, sub_bits, nbuckets, stack_cap;
    int k2_grid, k3_blocks;
    size_t tok, tok8, meta, slow, ctrl, sort, hist, gstack, gpool;
};

struct MatchScratch {
    u32 *tok, *tok8, *meta, *slow;
    Ctrl* ctrl;
    u32 *sort, *hist;
    u64* gstack;
    Desc* gpool;
};

inline MatchPlan plan_match(const MatchGeometry& g, const MatchJob& j, u32 max_depth) {
    MatchPlan p{};
    const u32 n = static_cast<u32>(j.n);
    p.n = n;
    p.S = std::max<u32>(1u, max_depth);
    p.site_bits = j.bucket_bits ? j.bucket_bits : g.site_bits;
    p.sub_bits = j.bucket_bits ? 0u : g.sub_bits;
    p.nbuckets = 1u << (p.site_bits + p.sub_bits);
    p.stack_cap = 32u * (max_depth + 2u) + 64u;
    const int k2_ctas = (g.k2_ctas >= 1 && g.k2_ctas <= K2_CTAS_PER_SM) ? g.k2_ctas : K2_CTAS_PER_SM;
    const int sms = static_cast<int>(g.num_sms);
    const bool small = j.hdr != nullptr;     // capacity-sized launches: the grids shrink with the capacity
    p.k2_grid = small ? std::max(1, std::min<int>(sms * k2_ctas, (n + K2_THREADS - 1) / K2_THREADS)) : sms * k2_ctas;
    p.k3_blocks = small ? std::max(1, std::min<int>(sms, (n + 7) / 8)) : sms * 4;
    p.tok = p.S > TOK8 ? static_cast<size_t>(p.S) * n * sizeof(u32) : 256;
    p.tok8 = static_cast<size_t>(n) * TOK8 * sizeof(u32);
    p.meta = n * sizeof(u32);
    p.slow = n * sizeof(u32);
    p.ctrl = sizeof(Ctrl);
    p.sort = static_cast<size_t>(n) * 11 * sizeof(u32) + 64;      // bkey, perm, meta_sorted [n] + tok8_sorted [n][8]
    p.hist = 2 * static_cast<size_t>(p.nbuckets) * sizeof(u32);   // histogram + cursor
    p.gstack = static_cast<size_t>(g.num_sms) * 4 * 8 * p.stack_cap * sizeof(u64);
    p.gpool = static_cast<size_t>(g.num_sms) * k2_ctas * K2_THREADS * g.pool_rows * sizeof(Desc);
    return p;
}

// Enqueues the pipeline for j.n > 0 rows (the caller has provided the scratch of `p` and ordered the call after the
// last flush and the scratch's previous user).
template <class L>
int match_pipeline(L& l, const MatchGeometry& g, const MatchJob& j, const MatchPlan& p, const TrieView& tv, const MatchScratch& m) {
    const u32 n = p.n;
    const bool desc = j.mode == MatchJob::DESCRIPTORS, gather = j.mode == MatchJob::GATHER;
    u32* bkey = m.sort;
    u32* perm = bkey + n;
    u32* meta_sorted = perm + n;
    u32* tok8_sorted = meta_sorted + n + ((8 - (3 * static_cast<size_t>(n)) % 8) % 8);   // 32-byte aligned rows
    u32* hist = m.hist;
    u32* bcursor = hist + p.nbuckets;
    int st;
    // the bump cursor over the output survives between the chunks of one pipelined host call
    if (j.keep_cursor) st = l.memset(reinterpret_cast<char*>(m.ctrl) + sizeof(unsigned long long), 0, sizeof(Ctrl) - sizeof(unsigned long long));
    else st = l.memset(m.ctrl, 0, sizeof(Ctrl));
    if (st != GM_OK || (st = l.memset(hist, 0, p.nbuckets * sizeof(u32))) != GM_OK || (st = l.mark(0)) != GM_OK) return st;
    auto k1 = g.tok_bulk ? k_tokenize<true> : k_tokenize<false>;
    if ((st = l.launch(k1, (n + TOK_THREADS - 1) / TOK_THREADS, TOK_THREADS, 0, static_cast<const u8*>(j.blob), static_cast<u32>(j.blob_bytes),
                       static_cast<u32>(std::max<u64>(j.blob_bytes, j.readable_bytes)), j.offs, j.sel, n, j.hdr, tv, p.S, m.tok8, m.tok, m.meta, j.status,
                       bkey, hist, p.site_bits, p.sub_bits)) != GM_OK) return st;
    if ((st = l.launch(k_bucket_scan, 1, 1024, 0, hist, bcursor, p.nbuckets)) != GM_OK) return st;
    if ((st = l.launch(k_bucket_scatter, (n + 255) / 256, 256, 0, bkey, bcursor, n, j.hdr, perm, m.tok8, m.meta,
                       g.sorted_rows ? tok8_sorted : nullptr, meta_sorted)) != GM_OK) return st;
    if ((st = l.mark(1)) != GM_OK) return st;

    MatchParams mp{};
    mp.tv = tv; mp.tok8 = m.tok8; mp.tok = m.tok; mp.meta = m.meta; mp.n = n; mp.n_ptr = j.hdr; mp.tok_levels = p.S;
    mp.spans = reinterpret_cast<uint2*>(j.spans); mp.out_ids = static_cast<u32*>(j.out); mp.out_desc = static_cast<uint2*>(j.out);
    mp.cap_ids = std::min<u64>(j.cap, 0xFFFFFFFFull);       // spans carry 32-bit offsets
    mp.status = j.status;
    mp.trees = j.trees;
    mp.cursor = &m.ctrl->cursor; mp.slow_list = m.slow; mp.slow_count = &m.ctrl->slow_count;
    mp.tile_counter = &m.ctrl->tile_counter; mp.stats = m.ctrl->stats;
    mp.perm = perm; mp.tok8_sorted = tok8_sorted; mp.meta_sorted = meta_sorted;
    mp.flags = (g.sorted_rows ? MP_SORTED_ROWS : 0u) | g.diag_flags;
    mp.tile_chunk = g.tile_chunk;
    if (gather) {
        const GatherLayout& G = *j.gather;
        mp.g_base_topics = static_cast<u32>(j.rank * G.slab_topics); mp.g_base_ids = j.rank * G.slab_ids; mp.g_sel = j.sel;
        const u32 w0 = g.gather_direct ? 0 : j.rank, w1 = g.gather_direct ? G.world : j.rank + 1;
        mp.g_world = w1 - w0;   // direct: the publish phase stores into every rank's block; else into its own, k_gather_push copies
        for (u32 w = w0; w < w1; ++w) {
            mp.g_ids[w - w0] = reinterpret_cast<u32*>(j.blocks[w] + GatherLayout::off_ids); mp.g_spans[w - w0] = reinterpret_cast<uint2*>(j.blocks[w] + G.off_spans);
            mp.g_index[w - w0] = reinterpret_cast<u32*>(j.blocks[w] + G.off_index);
        }
    }
    const std::array<MatchFastKernel, 5> k2s = match_fast_kernels();
    const MatchFastKernel k2 = gather ? k2s[4] : k2s[(j.stats ? 0 : 2) + (desc ? 1 : 0)];
    if ((st = l.launch(k2, p.k2_grid, K2_THREADS, k2_smem_bytes<K2_FAST_L, K2_THREADS>(), mp, m.gpool, g.pool_rows)) != GM_OK || (st = l.mark(2)) != GM_OK) return st;
    auto k3 = gather ? k_match_slow<false, false, true>
                     : j.stats ? (desc ? k_match_slow<true, true> : k_match_slow<true, false>) : (desc ? k_match_slow<false, true> : k_match_slow<false, false>);
    if ((st = l.launch(k3, p.k3_blocks, 256, 0, mp, m.gstack, p.stack_cap)) != GM_OK || (st = l.mark(3)) != GM_OK) return st;
    return j.d_needed ? l.copy(j.d_needed, &m.ctrl->cursor, sizeof(u64)) : GM_OK;
}

// End of a fused-gather step, part 1 (push form only): k_gather_push copies this rank's slab into every peer's block.
// `blocks` is an array the kernel can read.
template <class L>
int gather_push(L& l, const GatherLayout& G, bool direct, u32 num_sms, char* const* blocks, u32 rank, u64 n, const unsigned long long* d_m) {
    if (direct || G.world <= 1) return GM_OK;
    return l.launch(k_gather_push, num_sms * 4, 256, 0, blocks, rank, G.world, GatherLayout::off_ids, G.off_spans, G.off_index,
                    static_cast<unsigned long long>(rank * G.slab_topics), static_cast<unsigned long long>(rank * G.slab_ids), static_cast<unsigned long long>(n), d_m);
}

// ... part 2: this rank's contribution into every rank's counts, then the epoch barrier.  The error word reports on THIS
// step only: a straggler of an earlier step (a rank that arrived after the bounded wait) must not make every later step
// fail (only this rank's own k_gather_finish ever writes the word).  `counts` / `flags` are arrays the kernel can read.
template <class L>
int gather_finish(L& l, const GatherLayout& G, char* own_block, unsigned long long* const* counts, u32* const* flags, u32 rank, u64 n,
                  const unsigned long long* d_m, u32 epoch) {
    u32* my_flags = reinterpret_cast<u32*>(own_block + G.off_flags);
    const int st = l.memset(my_flags + 32, 0, sizeof(u32));
    if (st != GM_OK) return st;
    return l.launch(k_gather_finish, 1, 32, 0, counts, flags, my_flags, rank, G.world, static_cast<unsigned long long>(n), d_m, epoch, my_flags + 32);
}

// ---- retained lookup: tokenise filters -> frontier BFS (one step kernel per tree level) -> publish ---------------------------
// counts[(max_depth + 3) * RQ] (tasks per round and queue slice; the first RQ are the member) and then claim[max_depth + 3]
// follow the struct in the same allocation
struct RCtl { unsigned long long grand; unsigned long long stats[2]; u32 err; u32 pad; u32 n_desc[RQ]; u32 counts[RQ]; };

constexpr int RETAIN_ATTEMPTS = 12;   // scratch growths before a lookup gives up

// After an overflow (RCtl::err bit 0: tasks, bit 1: descriptors) the scratch grows x4; false: past 2^30, give up.
inline bool retain_grow(u32 err, u32& cap_items, u32& cap_desc) {
    if (err & 1u) { if (cap_items > (1u << 30)) return false; cap_items *= 4; }
    if (err & 2u) { if (cap_desc > (1u << 30)) return false; cap_desc *= 4; }
    return true;
}

struct RetainJob {                  // one lookup; every pointer is device memory
    const void* blob = nullptr;
    u64 blob_bytes = 0;
    const u32* offs = nullptr;
    u64 n = 0;
    gm_span* spans = nullptr;
    u32* ids = nullptr;
    u64 cap_ids = 0;
    int32_t* status = nullptr;
    bool stats = false;             // instrumented instantiations
};

struct RetainPlan {
    u32 nq, depth, S, slice_items, slice_desc;
    size_t tok, tok8, meta, rq, ctl, front, descs;   // scratch bytes (front: each of the two frontier queues)
};

struct RetainScratch {
    u32 *tok, *tok8, *meta, *rq;
    RCtl* ctl;
    RTask* front[2];
    RDesc* descs;
};

// cap_items / cap_desc: totals over the RQ slices of each queue
inline RetainPlan plan_retain(u64 n, u32 depth, u32 cap_items, u32 cap_desc) {
    RetainPlan p{};
    const u32 nq = static_cast<u32>(n);
    p.nq = nq; p.depth = depth;
    p.S = depth + 2;                // the walk reads filter levels pos and pos+1 with pos <= tree depth
    p.slice_items = cap_items / RQ; p.slice_desc = cap_desc / RQ;
    p.tok = p.S > TOK8 ? static_cast<size_t>(p.S) * nq * sizeof(u32) : 256;
    p.tok8 = static_cast<size_t>(nq) * TOK8 * sizeof(u32);
    p.meta = nq * sizeof(u32);
    p.rq = static_cast<size_t>(nq) * 3 * sizeof(u32);
    p.ctl = sizeof(RCtl) + static_cast<size_t>(depth + 3) * RQ * sizeof(u32) + static_cast<size_t>(depth + 3) * sizeof(u32);
    p.front = static_cast<size_t>(p.slice_items) * RQ * sizeof(RTask);
    p.descs = static_cast<size_t>(p.slice_desc) * RQ * sizeof(RDesc);
    return p;
}

template <class L>
int retain_pipeline(L& l, const RetainJob& j, const RetainPlan& p, const TrieView& tv, const RetainView& rv, const RetainScratch& m, u32 num_sms) {
    const u32 nq = p.nq, depth = p.depth;
    RCtl* ctl = m.ctl;
    u32* qtotal = m.rq;
    u32* qbase = qtotal + nq;
    u32* qcur = qbase + nq;
    int st;
    if ((st = l.memset(ctl, 0, p.ctl)) != GM_OK || (st = l.memset(m.rq, 0, p.rq)) != GM_OK || (st = l.mark(0)) != GM_OK) return st;
    if ((st = l.launch(k_tokenize<false>, (nq + TOK_THREADS - 1) / TOK_THREADS, TOK_THREADS, 0, static_cast<const u8*>(j.blob), static_cast<u32>(j.blob_bytes),
                       static_cast<u32>(j.blob_bytes), j.offs, static_cast<const u32*>(nullptr), nq, static_cast<const u32*>(nullptr), tv, p.S, m.tok8, m.tok, m.meta,
                       j.status, static_cast<u32*>(nullptr), static_cast<u32*>(nullptr), 0u, 0u)) != GM_OK || (st = l.mark(1)) != GM_OK) return st;
    RetainParams rp{};
    rp.v = rv; rp.qtok8 = m.tok8; rp.qtok = m.tok; rp.qmeta = m.meta; rp.nq = nq; rp.tok_levels = p.S;
    rp.descs = m.descs; rp.n_desc = ctl->n_desc; rp.cap_items = p.slice_items; rp.cap_desc = p.slice_desc;
    rp.qtotal = qtotal; rp.err = &ctl->err;
    // round 0 follows every filter's literal prefix; every later round expands the wildcard tasks the round before
    // queued.  A task descends at least one tree level, so depth + 1 rounds drain every queue (late rounds find
    // theirs empty and return at once).
    rp.stats = ctl->stats;
    auto kri = j.stats ? k_retain_init<true> : k_retain_init<false>;
    auto krr = j.stats ? k_retain_round<true> : k_retain_round<false>;
    if ((st = l.launch(kri, (nq + 255) / 256, 256, 0, rp, m.front[0], &ctl->counts[0])) != GM_OK) return st;
    const u32 rgrid = num_sms * GM_RETAIN_CTAS;   // exactly the resident CTAs (launch bound of k_retain_round): tasks are claimed dynamically
    for (u32 lvl = 0; lvl <= depth; ++lvl)
        if ((st = l.launch(krr, rgrid, 256, 0, rp, m.front[lvl & 1], &ctl->counts[static_cast<size_t>(lvl) * RQ], m.front[(lvl + 1) & 1],
                           &ctl->counts[static_cast<size_t>(lvl + 1) * RQ], &ctl->counts[static_cast<size_t>(depth + 3) * RQ + lvl])) != GM_OK) return st;
    if ((st = l.mark(2)) != GM_OK) return st;
    if ((st = l.launch(k_retain_scan, 1, 1024, 0, qtotal, nq, qbase, reinterpret_cast<uint2*>(j.spans), &ctl->grand)) != GM_OK) return st;
    if ((st = l.launch(k_retain_expand, num_sms * 8, 256, 0, m.descs, ctl->n_desc, p.slice_desc, rv.vals, qbase, qcur, j.ids,
                       static_cast<unsigned long long>(j.cap_ids))) != GM_OK) return st;
    return l.mark(3);
}

// ---- tables: the views the kernels get, and what a flush ships -----------------------------------------------------------------
struct TrieTables { const EdgeSlot* edges; const Range* ranges; const u32* values; const DictSlot* dict; const u8* pool; const u32* cfilter; const u32* tree_slots; };
struct RetainTables { const RKid* kids; const REdge* edges; const u32* vals; };

inline TrieView make_trie_view(const HostTrie& trie, const TrieTables& d) {
    TrieView v{};
    v.edges = d.edges; v.ranges = d.ranges; v.values = d.values; v.dict = d.dict; v.pool = d.pool;
    v.cfilter = d.cfilter; v.cfilter_mask = static_cast<u32>(trie.cfilter.size() - 1);
    v.edge_mask = static_cast<u32>(trie.edges.size() - 1);
    v.win_mask = trie.win_mask(); v.win_shift = trie.win_shift(); v.nwin_mask = trie.nwin_mask();
    v.dict_mask = static_cast<u32>(trie.dict.size() - 1);
    v.root_plus = trie.root_plus; v.root_hash_ref = trie.root_hash_ref; v.root_hash_cnt = trie.root_hash_cnt; v.root_mask = trie.root_mask;
    v.max_depth = trie.max_depth;
    v.tree_slots = d.tree_slots; v.n_trees = d.tree_slots ? static_cast<u32>(trie.tree_slots.size()) : 0u;
    return v;
}

inline RetainView make_retain_view(const RetainTreeHost& rtree, const RetainTables& d) {
    RetainView v{};
    v.kids = d.kids; v.edges = d.edges; v.vals = d.vals;
    v.edge_mask = static_cast<u32>(rtree.redges.size() - 1);
    if (!rtree.rnodes.empty()) { v.root_first_kid = rtree.rnodes[0].first_kid; v.root_nk_flags = rtree.rnodes[0].nkids | (rtree.rnodes[0].flags << 28); }
    v.root_plain_kids = rtree.root_plain_kids; v.root_plain_val_hi = rtree.root_plain_val_hi; v.max_depth = rtree.max_depth;
    v.n_kids = static_cast<u32>(rtree.rkids.size());
    return v;
}

// The device copies, one buffer per table (rnodes only marks "the retained tree was shipped": its records travel in rkids / redges).
template <class B> struct TableBufs { B *edges, *dict, *ranges, *values, *pool, *cfilter, *tree_slots, *rnodes, *rkids, *redges, *rvals; };

// What the device copies hold: how far each appendable array was shipped, the slot count each hash table was shipped with
// (0: nothing that may be assumed, ship whole), the value-store generation.
struct ShipMarks {
    size_t ranges = 0, values = 0, pool = 0, edges_slots = 0, dict_slots = 0;
    size_t rkids = 0, rvals = 0, redges_slots = 0;
    u64 values_epoch = 0;
    // the subscription tables were rebuilt (a compaction) or the device copy is unknown: re-ship them whole
    void forget_trie(u64 epoch) { ranges = values = pool = edges_slots = dict_slots = 0; values_epoch = epoch; }
    void forget_all() { forget_trie(values_epoch); rkids = rvals = redges_slots = 0; }
};

template <class V> using elem_t = std::remove_cv_t<std::remove_reference_t<decltype(std::declval<const V&>()[0])>>;

// capacity of a fresh buffer: room for `bytes + slack_bytes`, at least min_bytes, whole 256-byte units
inline size_t fresh_capacity(size_t bytes, size_t min_bytes, size_t slack_bytes = 0) {
    const size_t c = std::max({bytes + slack_bytes, min_bytes, size_t(256)});
    return (c + 255) & ~size_t(255);
}

template <class S, class B, class V>
int ship_fresh(S& sh, B& buf, const V& host, size_t min_bytes, size_t slack_bytes = 0) {
    const size_t bytes = host.size() * sizeof(elem_t<V>);
    return sh.fresh(buf, host.data(), bytes, fresh_capacity(bytes, min_bytes, slack_bytes));
}

// Hash tables (edges, dict): whole table into a new buffer after a re-hash or when most of it changed, else patches.
template <class S, class B, class V>
int ship_table(S& sh, B& buf, const V& host, bool& full, std::vector<u32>& dirty, size_t& up_slots) {
    int st;
    if (full || up_slots != host.size() || dirty.size() * 8 > host.size()) {
        if ((st = ship_fresh(sh, buf, host, 0)) != GM_OK) return st;
        up_slots = host.size();
        dirty.clear();
    } else if ((st = sh.patch(buf, host, dirty)) != GM_OK) return st;
    full = false;
    return GM_OK;
}

// Append-only arrays (ranges, values, pool, retained child blocks / values): copy the new tail in place (no running
// kernel can reach it yet); a grown or rebuilt array goes into a new buffer; older entries that changed are patched.
template <class S, class B, class V>
int ship_appendable(S& sh, B& buf, const V& host, size_t& up, std::vector<u32>* dirty) {
    using T = elem_t<V>;
    const size_t bytes = host.size() * sizeof(T);
    if ((up == 0 && (host.size() > 0 || !sh.capacity(buf))) || bytes > sh.capacity(buf)) {    // first shipment, rebuilt content, or out of room: new buffer with room to append
        int st = ship_fresh(sh, buf, host, std::max(bytes * 2, size_t(4096)));
        if (st != GM_OK) return st;
        up = host.size();
        if (dirty) dirty->clear();
        return GM_OK;
    }
    const size_t before = up;
    if (host.size() > up) {
        int st = sh.append(buf, up * sizeof(T), host.data() + up, (host.size() - up) * sizeof(T));
        if (st != GM_OK) return st;
        up = host.size();
    }
    if (dirty) {
        dirty->erase(std::remove_if(dirty->begin(), dirty->end(), [&](u32 i) { return i >= before; }), dirty->end());
        int st = sh.patch(buf, host, *dirty);
        if (st != GM_OK) return st;
        dirty->clear();
    }
    return GM_OK;
}

// Everything a flush ships after trie.sync(); *r_shipped: the retained tree went too (the caller calls rtree.shipped()
// once the shipment is complete).
template <class S, class B>
int ship(S& sh, const TableBufs<B>& d, HostTrie& trie, RetainTreeHost& rtree, ShipMarks& up, bool* r_shipped) {
    if (trie.values_epoch != up.values_epoch) { up.values = up.ranges = 0; up.values_epoch = trie.values_epoch; }   // value sets were compacted: re-ship whole
    int rs;
    *r_shipped = false;
    if (rtree.dirty) {   // retained tree: whole arrays after a (re)flatten, else only the entries set / remove edited in place
        rtree.prepare_flush();
        if (rtree.full) {
            const std::vector<u32> marker{0u};
            if ((rs = ship_fresh(sh, *d.rnodes, marker, 0)) != GM_OK) return rs;
            if ((rs = ship_fresh(sh, *d.rkids, rtree.rkids, 0, (rtree.rkids.size() / 4 + 1024) * sizeof(RKid))) != GM_OK) return rs;   // room for in-place appends
            if ((rs = ship_fresh(sh, *d.redges, rtree.redges, 0)) != GM_OK) return rs;
            if ((rs = ship_fresh(sh, *d.rvals, rtree.rvals, 0, 4096)) != GM_OK) return rs;
            up.rkids = rtree.rkids.size(); up.rvals = rtree.rvals.size(); up.redges_slots = rtree.redges.size();
        } else {
            bool full_edges = false;
            if ((rs = ship_appendable(sh, *d.rkids, rtree.rkids, up.rkids, &rtree.dirty_kids)) != GM_OK) return rs;
            if ((rs = ship_table(sh, *d.redges, rtree.redges, full_edges, rtree.dirty_edges, up.redges_slots)) != GM_OK) return rs;
            if ((rs = ship_appendable(sh, *d.rvals, rtree.rvals, up.rvals, &rtree.dirty_vals)) != GM_OK) return rs;
        }
        *r_shipped = true;
    }
    if ((rs = ship_table(sh, *d.edges, trie.edges, trie.full_edges, trie.dirty_edges, up.edges_slots)) != GM_OK) return rs;
    if ((rs = ship_table(sh, *d.dict, trie.dict, trie.full_dict, trie.dirty_dict, up.dict_slots)) != GM_OK) return rs;
    if ((rs = ship_appendable(sh, *d.ranges, trie.ranges, up.ranges, nullptr)) != GM_OK) return rs;
    if ((rs = ship_appendable(sh, *d.values, trie.values, up.values, nullptr)) != GM_OK) return rs;
    if ((rs = ship_appendable(sh, *d.pool, trie.pool, up.pool, nullptr)) != GM_OK) return rs;
    if (trie.cfilter_dirty) {   // child filter of wide nodes: a few MB, shipped whole into a new buffer (a rebuild changes its geometry)
        if ((rs = ship_fresh(sh, *d.cfilter, trie.cfilter, 0)) != GM_OK) return rs;
        trie.cfilter_dirty = false;
    }
    if (trie.trees_dirty) {      // root records of the extra trees (ACL rules, rewrite rules, ...): a tiny array, shipped whole
        if ((rs = ship_fresh(sh, *d.tree_slots, trie.tree_slots, 0)) != GM_OK) return rs;
        trie.trees_dirty = false;
    }
    trie.root_dirty = false;
    return GM_OK;
}

}  // namespace gm
