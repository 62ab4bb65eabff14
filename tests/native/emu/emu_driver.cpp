// TEST INFRASTRUCTURE: the engine's own match, fused-gather and retained-lookup pipelines and its flush shipping policy
// (rmqtt_b200/csrc/pipeline.h, which engine.cu runs on the device) over HOST memory, with the REAL kernel sources
// (kernels.cuh, retain_kernels.cuh, comm.cuh, relations.cuh compiled with -DGM_CPU_EMU) run by the CPU emulation in
// cuda_runtime.h.  This file supplies only how an operation is carried out there: a launcher (emu::launch, std::memset),
// a shipper into a byte image of every table, and host buffers for the scratch the pipelines size.  Exposed as a small C
// interface for tests/test_emu_kernels.py, which compares the results with the oracle.  Build (tests/test_emu_kernels.py does it):
//   g++ -O1 -g -std=c++17 -DGM_CPU_EMU -Itests/native/emu -Irmqtt_b200/csrc -shared -fPIC tests/native/emu/emu_driver.cpp \
//       rmqtt_b200/csrc/host_trie.cpp rmqtt_b200/csrc/retain_tree.cpp -o <out>.so     (+ -fsanitize=address,undefined for the ASan run)
#include <cuda_runtime.h>      // the emulation (this directory is first on the include path)

#include <cstring>
#include <vector>

#include "../../../include/gpumqtt.h"
#include "pipeline.h"
#include "relations.cuh"

using namespace gm;

namespace {

constexpr u32 EMU_SMS = 2;               // the emulated part has two SMs: several CTAs per kernel, dynamic tile hand-out exercised

// host stand-in for a cudaMalloc'd buffer: 256-byte aligned, whole 256-byte units
struct Bytes {
    struct alignas(256) Unit { unsigned char b[256]; };
    std::vector<Unit> v;
    Bytes() = default;
    Bytes(size_t bytes, int fill) { alloc(bytes, fill); }
    void alloc(size_t bytes, int fill) {
        v.assign((bytes + 255) / 256, Unit{});
        if (!v.empty()) std::memset(static_cast<void*>(v.data()), fill, v.size() * sizeof(Unit));
    }
    template <class T> T* as() { return v.empty() ? nullptr : reinterpret_cast<T*>(v.data()); }
    size_t cap() const { return v.size() * sizeof(Unit); }
};

// pipeline.h's launcher: kernels run to completion one after the other, on the calling thread
struct EmuLauncher {
    template <class... P, class... A>
    int launch(void (*k)(P...), u32 grid, u32 block, size_t, A... a) {
        emu::launch(dim3(grid), dim3(block), [&] { k(a...); });
        return GM_OK;
    }
    int memset(void* p, int v, size_t bytes) { std::memset(p, v, bytes); return GM_OK; }
    int copy(void* dst, const void* src, size_t bytes) { std::memcpy(dst, src, bytes); return GM_OK; }
    int mark(int) { return GM_OK; }
};

// pipeline.h's shipper into a byte image per table: a slot the host mirror changed without listing it as dirty stays
// stale there — and shows up as a wrong match.  Bytes never shipped read 0xCD (garbage, as on a device).
struct ImageShipper {
    int fresh(Bytes& b, const void* src, size_t bytes, size_t cap_bytes) {
        b.alloc(cap_bytes, 0xCD);
        if (bytes) std::memcpy(b.as<char>(), src, bytes);
        return GM_OK;
    }
    int append(Bytes& b, size_t off, const void* src, size_t bytes) { std::memcpy(b.as<char>() + off, src, bytes); return GM_OK; }
    template <class V>
    int patch(Bytes& b, const V& host, std::vector<u32>& dirty) {
        using T = elem_t<V>;
        for (u32 i : dirty) std::memcpy(b.as<char>() + static_cast<size_t>(i) * sizeof(T), &host[i], sizeof(T));
        dirty.clear();
        return GM_OK;
    }
    size_t capacity(const Bytes& b) const { return b.cap(); }
};

struct MatchBufs {                       // the scratch of one match, as plan_match sized it
    Bytes tok, tok8, meta, slow, ctrl, sort, hist, gstack, gpool;
    explicit MatchBufs(const MatchPlan& p)
        : tok(p.tok, 0), tok8(p.tok8, 0), meta(p.meta, 0), slow(p.slow, 0), ctrl(p.ctrl, 0), sort(p.sort, 0), hist(p.hist, 0), gstack(p.gstack, 0), gpool(p.gpool, 0) {}
    MatchScratch scratch() {
        return {tok.as<u32>(), tok8.as<u32>(), meta.as<u32>(), slow.as<u32>(), ctrl.as<Ctrl>(), sort.as<u32>(), hist.as<u32>(), gstack.as<u64>(), gpool.as<Desc>()};
    }
};

struct EmuEngine {
    HostTrie trie{128};
    RetainTreeHost rtree{&trie};
    u32 pool_rows = K2_POOL_ROWS;        // (tests lower it to push topics onto the deferred kernel)
    // optional device image (emu_use_image): the kernels then read copies that only flush() updates
    bool image = false, manual_flush = false;
    Bytes d_edges, d_dict, d_ranges, d_values, d_pool, d_cfilter, d_tree_slots, d_rnodes, d_rkids, d_redges, d_rvals;
    ShipMarks up;
    TrieView dev_view{}; RetainView dev_rview{};

    bool flush() {                       // gm_engine::flush_impl, into the image
        if (!trie.any_dirty() && !rtree.dirty) return true;
        if (!trie.sync()) return false;
        ImageShipper sh;
        bool r_shipped = false;
        ship(sh, TableBufs<Bytes>{&d_edges, &d_dict, &d_ranges, &d_values, &d_pool, &d_cfilter, &d_tree_slots, &d_rnodes, &d_rkids, &d_redges, &d_rvals},
             trie, rtree, up, &r_shipped);
        dev_view = make_trie_view(trie, {d_edges.as<EdgeSlot>(), d_ranges.as<Range>(), d_values.as<u32>(), d_dict.as<DictSlot>(), d_pool.as<u8>(),
                                         d_cfilter.as<u32>(), d_tree_slots.as<u32>()});
        dev_rview = make_retain_view(rtree, {d_rkids.as<RKid>(), d_redges.as<REdge>(), d_rvals.as<u32>()});
        if (r_shipped) rtree.shipped();
        return true;
    }
    // what a match sees: the live host arrays, or — with the device image — the copies as of the last flush (engine.cu
    // auto_flush: GM_FLAG_MANUAL_FLUSH engines flush only when told to, once the tables they need were shipped)
    bool prepare(bool retained) {
        if (!image) { if (!trie.sync()) return false; if (retained) { rtree.prepare_flush(); rtree.shipped(); } return true; }
        if (manual_flush && d_edges.cap() && (!retained || d_rnodes.cap())) return true;
        return flush();
    }
    TrieView view() {
        if (image) return dev_view;
        return make_trie_view(trie, {trie.edges.data(), trie.ranges.data(), trie.values.data(), trie.dict.data(), trie.pool.data(), trie.cfilter.data(), trie.tree_slots.data()});
    }
    RetainView rview() { return image ? dev_rview : make_retain_view(rtree, {rtree.rkids.data(), rtree.redges.data(), rtree.rvals.data()}); }
    MatchGeometry geometry(bool tok_bulk) const {
        MatchGeometry g;
        g.num_sms = EMU_SMS; g.pool_rows = pool_rows; g.site_bits = 10; g.tok_bulk = tok_bulk;
        return g;
    }
};

}  // namespace

extern "C" {

void* emu_new() { return new EmuEngine(); }
void emu_free(void* h) { delete static_cast<EmuEngine*>(h); }
void emu_set_pool_rows(void* h, uint32_t rows) { static_cast<EmuEngine*>(h)->pool_rows = rows; }
// the kernels read a device IMAGE that only flushes update (manual != 0: only emu_flush, like GM_FLAG_MANUAL_FLUSH)
void emu_use_image(void* h, uint32_t manual) { EmuEngine* e = static_cast<EmuEngine*>(h); e->image = true; e->manual_flush = manual != 0; }
void emu_retain_counters(void* h, uint64_t* out6) { uint64_t o[6]; static_cast<EmuEngine*>(h)->rtree.debug_stats(o); std::memcpy(out6, o, sizeof(o)); }   // {full rebuilds, in-place patches, ...}
int32_t emu_flush(void* h) { return static_cast<EmuEngine*>(h)->flush() ? 0 : -7; }
int32_t emu_compact(void* h) {           // gm_compact: dictionary + value compaction, the retained tree re-labelled
    EmuEngine* e = static_cast<EmuEngine*>(h);
    const std::vector<u32> keep = e->rtree.used_tokens();
    std::vector<u32> remap;
    e->trie.compact(&keep, &remap);
    e->rtree.remap_tokens(remap);
    e->up.forget_trie(e->trie.values_epoch);
    return 0;
}

int32_t emu_sub_add(void* h, const char* f, uint32_t len, uint32_t value, uint32_t tree) {
    bool ch = false;
    return static_cast<EmuEngine*>(h)->trie.insert(f, len, value, &ch, tree);
}
int32_t emu_sub_remove(void* h, const char* f, uint32_t len, uint32_t value, uint32_t tree) {
    bool ch = false;
    return static_cast<EmuEngine*>(h)->trie.remove(f, len, value, &ch, tree);
}
int32_t emu_retain_set(void* h, const char* t, uint32_t len, uint32_t value) {
    bool had; u32 old;
    return static_cast<EmuEngine*>(h)->rtree.set(t, len, value, &had, &old);
}
int32_t emu_retain_remove(void* h, const char* t, uint32_t len) {
    bool had; u32 old;
    return static_cast<EmuEngine*>(h)->rtree.remove(t, len, &had, &old);
}

// gm_bulk_load / gm_retain_bulk_load: the all-host-threads builds (host_trie.cpp insert_batch_parallel, retain_tree.cpp set_batch_build)
uint64_t emu_bulk_load(void* h, const char* blob, const uint32_t* offs, const uint32_t* vals, uint64_t n) {
    EmuEngine& e = *static_cast<EmuEngine*>(h);
    e.trie.reserve(n);
    return e.trie.insert_batch(blob, offs, vals, n);
}
uint64_t emu_retain_bulk_load(void* h, const char* blob, const uint32_t* offs, const uint32_t* vals, uint64_t n) {
    return static_cast<EmuEngine*>(h)->rtree.set_batch(blob, offs, vals, n);
}

// Router::matches for a batch through the match pipeline.
// flags: bit 0 descriptor mode (the descriptors are expanded here from the host mirror, so `out_ids` holds ids either way),
//        bit 1 the bulk-staged tokeniser, bit 2 the instrumented (STATS) instantiations; work[4] = V, E, F, M then.
// Returns 0, or -3 with *needed when cap_ids is too small (the engine's capacity protocol).
//        bit 3 the batch is a SELECTION: row t matches entry sel[t] of the packed batch (n rows, n_entries entries; gm_match_args.d_sel),
//        bit 4 the small-batch-graph form: the kernels are launched for a CAPACITY larger than the batch and read the real
//              batch size / text length from a header in memory (engine.cu small_graph_match).
int32_t emu_match_ex(void* h, const char* blob_in, const uint32_t* offs, uint64_t n_entries, const uint32_t* sel, uint64_t n64, const uint32_t* trees, uint32_t flags,
                     gm_span* out_spans, uint32_t* out_ids, uint64_t cap_ids, uint64_t* needed, int32_t* status, uint64_t* work, uint32_t* deferred) {
    EmuEngine& e = *static_cast<EmuEngine*>(h);
    const bool desc = flags & 1u, bulk = flags & 2u, stats = flags & 4u, graph_form = flags & 16u;
    if (!(flags & 8u)) sel = nullptr;
    const u32 n_real = static_cast<u32>(n64);
    *needed = 0;
    if (n_real == 0) return 0;
    if (!e.prepare(false)) return -7;
    const TrieView tv = e.view();
    const u32 blob_bytes = offs[n_entries];
    const u32 n = graph_form ? n_real + 37u : n_real;            // launch size (rows beyond the real batch must stay untouched)
    u32 hdr_store[4] = {n_real, blob_bytes, 0u, 0u};
    std::vector<u32> offs_cap;
    if (graph_form) {                                             // the in-block holds capacity + 1 offsets; the tail is never read
        offs_cap.assign(offs, offs + n_entries + 1);
        offs_cap.resize(static_cast<size_t>(n) + 1, 0xDEADBEEFu);
        offs = offs_cap.data();
    }
    // the bulk stage wants a 16-byte aligned blob that may be read up to a 16-byte boundary
    const size_t readable = (static_cast<size_t>(blob_bytes) + 15) & ~size_t(15);
    Bytes blob(readable + 64, 0);
    std::memcpy(blob.as<char>(), blob_in, blob_bytes);
    std::vector<uint2> descs;
    std::vector<u32> ids_tmp;
    void* d_out = out_ids;
    if (desc) { descs.resize(cap_ids + 1); d_out = descs.data(); }
    std::vector<int32_t> status_cap;
    int32_t* status_k = status;
    if (graph_form) { status_cap.assign(n, 0x7F7F7F7F); status_k = status_cap.data(); }
    for (u32 i = 0; i < n_real; ++i) status[i] = 0x7F7F7F7F;   // every row must be written by the tokeniser
    std::vector<gm_span> spans_cap;
    gm_span* spans_k = out_spans;
    if (graph_form) { spans_cap.assign(n, gm_span{0xABABABABu, 0xABABABABu}); spans_k = spans_cap.data(); }

    MatchJob j;
    j.blob = blob.as<u8>(); j.blob_bytes = blob_bytes; j.readable_bytes = readable; j.offs = offs; j.sel = sel; j.n = n; j.hdr = graph_form ? hdr_store : nullptr;
    j.spans = spans_k; j.out = d_out; j.cap = cap_ids; j.status = status_k; j.trees = trees;
    j.mode = desc ? MatchJob::DESCRIPTORS : MatchJob::IDS;
    j.stats = stats;
    const MatchGeometry g = e.geometry(bulk);
    const MatchPlan p = plan_match(g, j, tv.max_depth);
    MatchBufs m(p);
    EmuLauncher l;
    match_pipeline(l, g, j, p, tv, m.scratch());
    const Ctrl& ctrl = *m.ctrl.as<Ctrl>();
    if (graph_form) {
        for (u32 i = n_real; i < n; ++i) if (status_cap[i] != 0x7F7F7F7F) return -50;      // a row beyond the real batch was touched
        std::memcpy(status, status_cap.data(), n_real * sizeof(int32_t));
        for (u32 i = n_real; i < n; ++i) if (spans_cap[i].off != 0xABABABABu) return -51;
        std::memcpy(out_spans, spans_cap.data(), n_real * sizeof(gm_span));
    }
    if (deferred) *deferred = ctrl.slow_count;
    if (work) for (int k = 0; k < 4; ++k) work[k] = ctrl.stats[k];
    *needed = ctrl.cursor;
    if (ctrl.cursor > cap_ids) return -3;
    if (!desc) return 0;
    // descriptor mode: expand (ref, cnt) into ids out of the host mirror, per topic, so that the caller compares id lists
    u64 w = 0;
    for (u32 t = 0; t < n_real; ++t) {
        const u32 off = out_spans[t].off, cnt = out_spans[t].cnt;
        const u64 begin = w;
        for (u32 k = 0; k < cnt; ++k) {
            const uint2 d = descs[off + k];
            if (d.y == 1) ids_tmp.push_back(d.x);
            else {
                u64 o = d.x, c = d.y;
                if (d.y == CNT_BIG) { o = e.trie.ranges[d.x].off; c = e.trie.ranges[d.x].cnt; }
                for (u64 q = 0; q < c; ++q) ids_tmp.push_back(e.trie.values[o + q]);
            }
        }
        w = ids_tmp.size();
        out_spans[t] = gm_span{static_cast<u32>(begin), static_cast<u32>(w - begin)};
    }
    *needed = w;                      // (in descriptor mode the capacity the caller must offer is the expanded size)
    if (w > cap_ids) return -3;
    std::memcpy(out_ids, ids_tmp.data(), w * sizeof(u32));
    return 0;
}

int32_t emu_match(void* h, const char* blob_in, const uint32_t* offs, uint64_t n64, const uint32_t* trees, uint32_t flags, gm_span* out_spans, uint32_t* out_ids,
                  uint64_t cap_ids, uint64_t* needed, int32_t* status, uint64_t* work, uint32_t* deferred) {
    return emu_match_ex(h, blob_in, offs, n64, nullptr, n64, trees, flags & ~8u, out_spans, out_ids, cap_ids, needed, status, work, deferred);
}

// gm_partition_batch_device: k_partition.  counts[n_shards + 1] (the last entry = rows appended to sel)
int32_t emu_partition(const char* blob, const uint32_t* offs, uint64_t n, uint32_t n_shards, uint32_t rank, uint32_t* sel, uint32_t* shard_out, uint32_t* counts) {
    std::memset(counts, 0, (static_cast<size_t>(n_shards) + 1) * sizeof(u32));
    if (n == 0) return 0;
    const u32 blob_bytes = offs[n];
    emu::launch(dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), [&] {
        k_partition(reinterpret_cast<const u8*>(blob), blob_bytes, offs, static_cast<u32>(n), n_shards, rank, sel, shard_out, counts);
    });
    return 0;
}

// ---- the fused gather over "peer memory": every rank's block lives in host memory of this one process ---------------------------
struct GatherWorld : GatherLayout {
    std::vector<Bytes> store;
    std::vector<char*> block;
    std::vector<u32> epoch;
    std::vector<unsigned long long> cursor;      // the match cursor of every rank's last step (k_gather_push / k_gather_finish read it)
};
void* emu_gather_new(uint32_t world, uint64_t slab_topics, uint64_t slab_ids) {       // gm_gather_create
    GatherWorld* g = new GatherWorld();
    static_cast<GatherLayout&>(*g) = gather_layout(world, slab_topics, slab_ids);
    g->store.resize(world); g->block.resize(world); g->epoch.assign(world, 0); g->cursor.assign(world, 0);
    for (u32 w = 0; w < world; ++w) {
        g->store[w].alloc(g->bytes, 0xEE);                                  // (stale bytes must never be read as results)
        g->block[w] = g->store[w].as<char>();
        std::memset(g->block[w] + g->off_counts, 0, g->bytes - g->off_counts);
    }
    return g;
}
void emu_gather_free(void* p) { delete static_cast<GatherWorld*>(p); }
uint64_t emu_gather_slab_ids(void* p) { return static_cast<GatherWorld*>(p)->slab_ids; }
uint64_t emu_gather_slab_topics(void* p) { return static_cast<GatherWorld*>(p)->slab_topics; }

// gm_match_gather_device of ONE rank: its rows (sel / n) through the GATHER instantiations of the match kernels, then — push form —
// k_gather_push copies the rank's slab into every peer's block.  direct != 0: the publish phase stores into every block itself.
int32_t emu_match_gather(void* gw, uint32_t rank, void* h, const char* blob_in, const uint32_t* offs, uint64_t n_entries, const uint32_t* sel, uint64_t n64,
                         uint32_t direct, int32_t* status) {
    GatherWorld& G = *static_cast<GatherWorld*>(gw);
    EmuEngine& e = *static_cast<EmuEngine*>(h);
    const u32 n = static_cast<u32>(n64);
    if (n > G.slab_topics) return -3;
    G.cursor[rank] = 0;
    if (n) {
        if (!e.prepare(false)) return -7;
        const TrieView tv = e.view();
        const u32 blob_bytes = offs[n_entries];
        const size_t readable = (static_cast<size_t>(blob_bytes) + 15) & ~size_t(15);
        Bytes blob(readable + 64, 0);
        std::memcpy(blob.as<char>(), blob_in, blob_bytes);
        MatchJob j;
        j.blob = blob.as<u8>(); j.blob_bytes = blob_bytes; j.readable_bytes = readable; j.offs = offs; j.sel = sel; j.n = n; j.cap = G.slab_ids; j.status = status;
        j.mode = MatchJob::GATHER; j.gather = &G; j.blocks = G.block.data(); j.rank = rank;
        MatchGeometry g = e.geometry(false);
        g.gather_direct = direct != 0;
        const MatchPlan p = plan_match(g, j, tv.max_depth);
        MatchBufs m(p);
        EmuLauncher l;
        match_pipeline(l, g, j, p, tv, m.scratch());
        G.cursor[rank] = m.ctrl.as<Ctrl>()->cursor;
        if (G.cursor[rank] > G.slab_ids) return -3;
    }
    EmuLauncher l;
    gather_push(l, G, direct != 0, EMU_SMS, G.block.data(), rank, n, &G.cursor[rank]);
    return 0;
}

// the end-of-step kernel of one rank (counts + flag to every block, bounded wait for the others' flags); returns the rank's error word
int32_t emu_gather_finish(void* gw, uint32_t rank, uint64_t n, uint32_t new_epoch) {
    GatherWorld& G = *static_cast<GatherWorld*>(gw);
    if (new_epoch) G.epoch[rank]++;
    std::vector<unsigned long long*> counts(G.world);
    std::vector<u32*> flags(G.world);
    for (u32 w = 0; w < G.world; ++w) { counts[w] = reinterpret_cast<unsigned long long*>(G.block[w] + G.off_counts); flags[w] = reinterpret_cast<u32*>(G.block[w] + G.off_flags); }
    EmuLauncher l;
    gather_finish(l, G, G.block[rank], counts.data(), flags.data(), rank, n, &G.cursor[rank], G.epoch[rank]);
    return static_cast<int32_t>(reinterpret_cast<u32*>(G.block[rank] + G.off_flags)[32]);
}

// one rank's view of the gathered arrays (gm_gather_get + the copies Engine.gather_result makes)
void emu_gather_read(void* gw, uint32_t rank, uint64_t* counts, uint32_t* index, gm_span* spans, uint32_t* ids) {
    GatherWorld& G = *static_cast<GatherWorld*>(gw);
    const char* b = G.block[rank];
    std::memcpy(counts, b + G.off_counts, static_cast<size_t>(G.world) * 16);
    std::memcpy(index, b + G.off_index, static_cast<size_t>(G.world) * G.slab_topics * 4);
    std::memcpy(spans, b + G.off_spans, static_cast<size_t>(G.world) * G.slab_topics * 8);
    std::memcpy(ids, b + GatherLayout::off_ids, static_cast<size_t>(G.world) * G.slab_ids * 4);
}

// RetainStorage::get for a batch of filters through the retained-lookup pipeline, growing the scratch from cap_items / cap_desc
// like gm_engine::run_retain; *grew = how many times it grew.  Returns 0, -3 with *needed when cap_ids is too small, or
// GM_ERR_TOO_LARGE when the scratch could not grow any further.
int32_t emu_retain_match(void* h, const char* blob_in, const uint32_t* offs, uint64_t n64, uint32_t stats_on, uint32_t cap_items, uint32_t cap_desc, gm_span* out_spans,
                         uint32_t* out_ids, uint64_t cap_ids, uint64_t* needed, int32_t* status, uint64_t* work, uint32_t* grew) {
    EmuEngine& e = *static_cast<EmuEngine*>(h);
    const u32 nq = static_cast<u32>(n64);
    *needed = 0;
    *grew = 0;
    if (nq == 0) return 0;
    if (!e.prepare(true)) return -7;
    const TrieView tv = e.view();
    const RetainView rv = e.rview();
    const u32 blob_bytes = offs[nq];
    Bytes blob(static_cast<size_t>(blob_bytes) + 64, 0);
    std::memcpy(blob.as<char>(), blob_in, blob_bytes);
    RetainJob j;
    j.blob = blob.as<u8>(); j.blob_bytes = blob_bytes; j.offs = offs; j.n = nq; j.spans = out_spans; j.ids = out_ids; j.cap_ids = cap_ids; j.status = status;
    j.stats = stats_on != 0;
    for (int attempt = 0; attempt < RETAIN_ATTEMPTS; ++attempt) {
        for (u32 i = 0; i < nq; ++i) status[i] = 0x7F7F7F7F;
        const RetainPlan p = plan_retain(nq, rv.max_depth, cap_items, cap_desc);
        Bytes tok(p.tok, 0), tok8(p.tok8, 0), meta(p.meta, 0), rq(p.rq, 0), ctl(p.ctl, 0), front0(p.front, 0), front1(p.front, 0), descs(p.descs, 0);
        EmuLauncher l;
        retain_pipeline(l, j, p, tv, rv, {tok.as<u32>(), tok8.as<u32>(), meta.as<u32>(), rq.as<u32>(), ctl.as<RCtl>(), {front0.as<RTask>(), front1.as<RTask>()}, descs.as<RDesc>()},
                        EMU_SMS);
        const RCtl& c = *ctl.as<RCtl>();
        if (c.err == 0) {
            if (work) { work[0] = c.stats[0]; work[1] = c.stats[1]; }
            *needed = c.grand;
            return c.grand > cap_ids ? -3 : 0;
        }
        if (!retain_grow(c.err, cap_items, cap_desc)) break;
        ++*grew;
    }
    return GM_ERR_TOO_LARGE;
}

// gm_relations_expand_device over host arrays (k_relations)
int32_t emu_relations(const gm_span* spans, const uint32_t* ids, uint64_t n, const uint32_t* pubs, const gm_rel* rels, uint64_t n_rels, gm_span* out_spans,
                      gm_sub_relation* out_rels, uint64_t cap_rels, uint32_t* out_sub_ids, uint64_t cap_sub_ids, uint64_t* needed3, int32_t* status) {
    needed3[0] = needed3[1] = needed3[2] = 0;
    if (n == 0) return 0;
    RelParams rp{};
    rp.spans = reinterpret_cast<const uint2*>(spans); rp.ids = ids; rp.n = static_cast<u32>(n); rp.pubs = pubs; rp.rels = rels; rp.n_rels = static_cast<u32>(n_rels);
    rp.out_spans = reinterpret_cast<uint2*>(out_spans); rp.out_rels = out_rels; rp.cap_rels = cap_rels; rp.out_sub_ids = out_sub_ids; rp.cap_sub_ids = cap_sub_ids;
    rp.needed = reinterpret_cast<unsigned long long*>(needed3); rp.status = status;
    const unsigned grid = static_cast<unsigned>(std::min<u64>((n + 7) / 8, static_cast<u64>(EMU_SMS) * 8));
    emu::launch(dim3(grid), dim3(256), [&] { k_relations(rp); });
    return 0;
}

}  // extern "C"
