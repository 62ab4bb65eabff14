"""CPU tier: the REAL kernel sources (rmqtt_b200/csrc/kernels.cuh, retain_kernels.cuh, relations.cuh) executed on the CPU by
the small CUDA-model emulation under tests/native/emu (threads of a CTA as fibers, warp collectives and barriers as
rendezvous points), driven like engine.cu drives them, and compared with the oracle — bit-exact sorted multisets, plus the
exact work counters V / E / F / M of the instrumented instantiations.

What this tier adds to the GPU tier: it runs HERE (no device), so a logic or indexing regression in a kernel shows up in the
`-m "not gpu"` suite; and the second build puts the kernels under AddressSanitizer + UBSan (out-of-bounds shared / global
accesses, misaligned vector accesses, shifts).  What it cannot see: memory ordering, scheduling, performance — the GPU tier
and compute-sanitizer cover those.  The product (`libgpumqtt.so`) is built from the same sources without GM_CPU_EMU and never
contains any of this."""
import ctypes as C
import random
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import oracle as orc
from rmqtt_b200.engine import MatchResult, pack

from _gen import rand_filter, rand_topic

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "rmqtt_b200" / "csrc"
EMU = ROOT / "tests" / "native" / "emu"

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")


class Span(C.Structure):
    _fields_ = [("off", C.c_uint32), ("cnt", C.c_uint32)]


def _build(tmp, san: bool):
    out = tmp / ("libemu_asan.so" if san else "libemu.so")
    cmd = ["g++", "-O1", "-g", "-std=c++17", "-DGM_CPU_EMU", f"-I{EMU}", f"-I{CSRC}", "-shared", "-fPIC", "-pthread", "-fno-omit-frame-pointer",
           *(["-fsanitize=address,undefined", "-fno-sanitize-recover=undefined"] if san else []),
           "-o", str(out), str(EMU / "emu_driver.cpp"), str(CSRC / "host_trie.cpp"), str(CSRC / "retain_tree.cpp")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0 and "sanitize" in r.stderr and "cannot find" in r.stderr:
        pytest.skip("sanitizer runtime not installed")
    assert r.returncode == 0, r.stderr[-3000:]
    return out


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    lib = C.CDLL(str(_build(tmp_path_factory.mktemp("emu"), san=False)))
    lib.emu_new.restype = C.c_void_p
    for f in ("emu_sub_add", "emu_sub_remove", "emu_retain_set", "emu_retain_remove", "emu_match", "emu_retain_match", "emu_relations", "emu_partition"):
        getattr(lib, f).restype = C.c_int32
    return lib


class Emu:
    def __init__(self, lib):
        self.lib, self.h = lib, C.c_void_p(lib.emu_new())

    def close(self):
        if self.h:
            self.lib.emu_free(self.h)
            self.h = None

    def add(self, f, v, tree=0):
        b = f.encode() if isinstance(f, str) else f
        return self.lib.emu_sub_add(self.h, b, len(b), v, tree)

    def remove(self, f, v, tree=0):
        b = f.encode() if isinstance(f, str) else f
        return self.lib.emu_sub_remove(self.h, b, len(b), v, tree)

    def retain_set(self, t, v):
        b = t.encode()
        return self.lib.emu_retain_set(self.h, b, len(b), v)

    def retain_remove(self, t):
        b = t.encode()
        return self.lib.emu_retain_remove(self.h, b, len(b))

    def match(self, blob, offs, flags=0, trees=None):
        n = len(offs) - 1
        spans = np.zeros((n, 2), dtype=np.uint32)
        status = np.zeros(n, dtype=np.int32)
        work = np.zeros(4, dtype=np.uint64)
        deferred, needed = C.c_uint32(0), C.c_uint64(0)
        cap = 1024
        blob = np.ascontiguousarray(blob if len(blob) else np.zeros(1, np.uint8))
        while True:
            ids = np.zeros(cap, dtype=np.uint32)
            rc = self.lib.emu_match(self.h, C.c_void_p(blob.ctypes.data), C.c_void_p(offs.ctypes.data), C.c_uint64(n), C.c_void_p(trees.ctypes.data) if trees is not None else None, flags,
                                    C.c_void_p(spans.ctypes.data), C.c_void_p(ids.ctypes.data), C.c_uint64(cap), C.byref(needed), C.c_void_p(status.ctypes.data), C.c_void_p(work.ctypes.data), C.byref(deferred))
            if rc == -3:
                cap = int(needed.value) + 16
                continue
            assert rc == 0, rc
            return MatchResult(spans, ids[:int(needed.value)], status, int(needed.value)), work, int(deferred.value)

    def retain_match(self, blob, offs, stats=0, cap_items=1 << 14, cap_desc=1 << 14):
        n = len(offs) - 1
        spans = np.zeros((n, 2), dtype=np.uint32)
        status = np.zeros(n, dtype=np.int32)
        work = np.zeros(2, dtype=np.uint64)
        needed, grew = C.c_uint64(0), C.c_uint32(0)
        cap = 1024
        blob = np.ascontiguousarray(blob if len(blob) else np.zeros(1, np.uint8))
        while True:
            ids = np.zeros(cap, dtype=np.uint32)
            rc = self.lib.emu_retain_match(self.h, C.c_void_p(blob.ctypes.data), C.c_void_p(offs.ctypes.data), C.c_uint64(n), stats, cap_items, cap_desc, C.c_void_p(spans.ctypes.data), C.c_void_p(ids.ctypes.data),
                                           C.c_uint64(cap), C.byref(needed), C.c_void_p(status.ctypes.data), C.c_void_p(work.ctypes.data), C.byref(grew))
            if rc == -3:
                cap = int(needed.value) + 16
                continue
            assert rc == 0, rc
            return MatchResult(spans, ids[:int(needed.value)], status, int(needed.value)), work, int(grew.value)


def _canon(want):
    ids = want["ids"].copy()
    o = want["offsets"]
    for i in range(len(o) - 1):
        ids[o[i]:o[i + 1]].sort()
    return want["counts"], ids


def _same(res, want):
    counts, ids = res.canonical()
    wc, wi = _canon(want)
    assert (counts == wc).all(), f"counts differ at {np.nonzero(counts != wc)[0][:5]}: {counts[counts != wc][:5]} vs {wc[counts != wc][:5]}"
    assert len(ids) == len(wi) and (ids == wi).all()


def _random_trie(e, tree, rng, n_filters, removals=0):
    fs = []
    for _ in range(n_filters):
        f, v = rand_filter(rng), rng.randint(0, 40)
        ok = e.add(f, v) == 0
        try:
            tree.insert(f, v)
            assert ok, f
            fs.append((f, v))
        except ValueError:
            assert not ok, f
    for f, v in rng.sample(fs, min(removals, len(fs))):
        assert e.remove(f, v) == 0
        tree.remove(f, v)


@pytest.mark.parametrize("seed,flags", [(1, 0), (2, 1), (3, 2), (4, 3), (5, 4), (6, 5)])
def test_publish_pipeline_on_the_emulator_equals_the_oracle(emu, seed, flags):
    """k_tokenize (plain and bulk-staged) -> k_bucket_scan -> k_bucket_scatter -> k_match_fast (ids / descriptors, plain /
    instrumented) -> k_match_slow over a random trie with every special case of SURVEY §8a in the alphabet."""
    rng = random.Random(seed)
    e, tree = Emu(emu), orc.TopicTree()
    # (removals leave pruned nodes behind as dead device records until gm_compact: results are unaffected, but the kernels then
    #  VISIT more nodes than the reference algorithm — the exact-counter runs therefore use a trie without removals)
    _random_trie(e, tree, rng, 1500, removals=0 if flags & 4 else 200)
    topics = [rand_topic(rng) for _ in range(1500)] + ["", "/", "//", "$SYS", "$SYS/a", "+", "#", "a/+", "a/#", "a/#/b", "a+/b", "x" * 200, "/".join(["a"] * 9)]
    tb, to = pack(topics)
    res, work, _ = e.match(tb, to, flags)
    want = tree.match_batch(tb, to)
    _same(res, want)
    assert (res.status[want["counts"] < 0] == -2).all() and (res.status[want["counts"] >= 0] == 0).all()
    if flags & 4:                                # the instrumented instantiations count exactly what the reference algorithm does
        c = want["counters"]
        assert [int(x) for x in work] == [c["V"], c["E"], c["F"], c["M"]]
    e.close()


def test_deferred_kernel_deep_topics_heavy_hitters_and_huge_sets(emu):
    """Everything k_match_fast hands to k_match_slow: more than 8 levels, more matched value sets than the staging pool holds
    (pool_rows lowered to 1: 9 sets), a value set of >= 65535 members (the `ranges` indirection) — in ids and descriptor mode."""
    e, tree = Emu(emu), orc.TopicTree()
    emu.emu_set_pool_rows(e.h, 1)
    deep = "/".join(f"l{i}" for i in range(20))
    fl = [deep, "/".join(["+"] * 20), "l0/l1/#", deep + "/#", "/".join(["l0"] + ["+"] * 10) + "/#", "#", "+/#", "l0/#", "l0/+/#", "l0/l1/+/#", "l0/l1/l2/#",
          "l0/l1/l2/+/#", "+/l1/#", "+/+/l2/#", "+/+/+/#", "l0/+/l2/#"]
    for i, f in enumerate(fl):
        assert e.add(f, i) == 0
        tree.insert(f, i)
    for v in range(66000):
        e.add("hot/+", v)
    tree.bulk_insert(*pack(["hot/+"] * 66000), np.arange(66000, dtype=np.uint32))
    for v in range(300):
        e.add("warm/#", v); tree.insert("warm/#", v)
    topics = [deep, deep + "/x", "l0/l1", "hot/a", "hot", "warm/x/y", "l0/" + "/".join(["q"] * 19), "l0/l1/l2/l3/l4"] * 9
    tb, to = pack(topics)
    for flags in (0, 1, 4, 5):
        res, work, deferred = e.match(tb, to, flags)
        want = tree.match_batch(tb, to)
        _same(res, want)
        assert deferred >= 9 * 5                  # the deep ones, the 9+-set ones and the huge set really took the deferred kernel
        if flags & 4:
            c = want["counters"]
            assert [int(x) for x in work] == [c["V"], c["E"], c["F"], c["M"]]
    e.close()


def test_extra_trees_rows_of_the_same_batch(emu):
    """gm_match_batch_trees: a row names the tree it is matched against; the `$`-rule applies at each tree's own root."""
    rng = random.Random(77)
    e = Emu(emu)
    trees = {0: orc.TopicTree(), 1: orc.TopicTree(), 5: orc.TopicTree()}
    for k, t in trees.items():
        for _ in range(300):
            f, v = rand_filter(rng), rng.randint(0, 20)
            try:
                t.insert(f, v)
            except ValueError:
                continue
            assert e.add(f, v, tree=k) == 0
    topics = [rand_topic(rng) for _ in range(600)]
    rows = np.asarray([rng.choice([0, 1, 5, 9]) for _ in topics], dtype=np.uint32)       # 9: no such tree -> nothing matches
    tb, to = pack(topics)
    res, _, _ = e.match(tb, to, 0, trees=rows)
    for i, (t, k) in enumerate(zip(topics, rows)):
        if orc.topic_parse(t) is None:
            want = None                               # Topic::from_str Err: whatever the tree
        else:
            want = sorted(trees[int(k)].matches(t)) if int(k) in trees else []
        assert res.sorted_list(i) == want, (t, k)
    e.close()


@pytest.mark.parametrize("seed", [11, 12])
def test_retained_pipeline_on_the_emulator_equals_the_oracle(emu, seed):
    """k_tokenize -> k_retain_init -> k_retain_round x (depth + 1) -> k_retain_scan -> k_retain_expand over a random retained
    tree (bulk-built image, then in-place edits), incl. literal '+' / '#' levels that shadow wildcard expansion and a scratch
    that starts too small (the overflow bits make the driver grow it, as gm_engine::run_retain does)."""
    rng = random.Random(seed)
    e, tree = Emu(emu), orc.RetainTree()
    names = []
    for i in range(2500):
        t = rand_topic(rng, max_depth=6) if rng.random() < 0.93 else rand_filter(rng, 5)
        if e.retain_set(t, i) != 0:
            with pytest.raises(ValueError):
                tree.insert(t, i)
            continue
        tree.remove(t)
        tree.insert(t, i)
        names.append(t)
    filters = [rand_filter(rng, 7) for _ in range(700)] + ["#", "+/#", "+", "$SYS/#", "+/+/+/+/+/+", "a/+/#", "+/+/#", "a/#"]
    fb, fo = pack(filters)
    res, work, grew = e.retain_match(fb, fo, stats=1, cap_items=64, cap_desc=64)
    assert grew >= 1
    _same(res, tree.match_batch(fb, fo))
    for t in rng.sample(names, 400):              # in-place edits of the image, then again
        e.retain_remove(t)
        tree.remove(t)
    for i in range(300):
        t = rand_topic(rng, max_depth=6)
        if e.retain_set(t, 100000 + i) == 0:
            tree.remove(t)
            tree.insert(t, 100000 + i)
    res, _, _ = e.retain_match(fb, fo)
    _same(res, tree.match_batch(fb, fo))
    e.close()


def test_kernels_under_asan_ubsan(tmp_path):
    """The same pipelines, kernels and host builders compiled with AddressSanitizer + UBSan, in a subprocess (the sanitizer
    runtime must be loaded first): a mixed publish batch incl. the deferred path, and a retained batch."""
    so = _build(tmp_path, san=True)
    script = tmp_path / "run.py"
    script.write_text(f"""
import sys, random, ctypes as C
sys.path.insert(0, {str(ROOT)!r}); sys.path.insert(0, {str(ROOT / 'tests')!r})
import numpy as np
import test_emu_kernels as T
from oracle import oracle as orc
from rmqtt_b200.engine import pack
lib = C.CDLL({str(so)!r})
lib.emu_new.restype = C.c_void_p
for f in ("emu_sub_add", "emu_sub_remove", "emu_retain_set", "emu_retain_remove", "emu_match", "emu_retain_match", "emu_relations", "emu_partition"):
    getattr(lib, f).restype = C.c_int32
rng = random.Random(5)
e, tree = T.Emu(lib), orc.TopicTree()
lib.emu_set_pool_rows(e.h, 2)
T._random_trie(e, tree, rng, 800, removals=100)
for v in range(40):
    e.add("+/#", 1000 + v); tree.insert("+/#", 1000 + v)
topics = [T.rand_topic(rng) for _ in range(700)] + ["", "x" * 300, "/".join(["a"] * 12)]
tb, to = pack(topics)
for flags in (0, 1, 2, 3, 4):
    res, _, _ = e.match(tb, to, flags)
    T._same(res, tree.match_batch(tb, to))
rt = orc.RetainTree()
for i in range(1200):
    t = T.rand_topic(rng, max_depth=6)
    if e.retain_set(t, i) == 0:
        rt.remove(t); rt.insert(t, i)
fb, fo = pack([T.rand_filter(rng, 7) for _ in range(300)] + ["#", "+/#", "+/+/+"])
res, _, _ = e.retain_match(fb, fo, cap_items=128, cap_desc=128)
T._same(res, rt.match_batch(fb, fo))
e.close()
# the other entry points of the driver, through the test functions themselves
T.test_selection_and_capacity_sized_launches(lib, 25)
T.test_partition_kernel_equals_the_host_shard_function(lib)
T.test_fused_gather_over_emulated_peer_memory(lib, 3, 0)
T.test_fused_gather_over_emulated_peer_memory(lib, 3, 1)
T.test_relation_expansion_kernel_against_a_python_model(lib)
print("asan run ok")
""")
    libasan = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    env = {"PATH": "/usr/bin:/bin", "LD_PRELOAD": libasan, "ASAN_OPTIONS": "detect_leaks=0:detect_stack_use_after_return=0", "PYTHONPATH": str(ROOT)}
    import os
    import sys
    for k in ("HOME", "LD_LIBRARY_PATH", "VIRTUAL_ENV"):
        if k in os.environ:
            env[k] = os.environ[k]
    run = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=1500, env=env)
    assert run.returncode == 0 and "asan run ok" in run.stdout, (run.stdout[-1500:], run.stderr[-4000:])


def test_relation_expansion_kernel_against_a_python_model(emu):
    """k_relations (router.rs:182-239 + types.rs:478-508 on the device): no_local, pass-through of v3 / shared-group members,
    per-client de-dup of v5 relations with accumulation of subscription identifiers, the > 256-relation hand-over — on synthetic
    match lists (duplicates, dead and out-of-range handles included) against a direct Python restatement."""
    from rmqtt_b200 import _native as N

    class GmRel(C.Structure):                               # include/gpumqtt.h gm_rel (24 bytes)
        _fields_ = [("node_id", C.c_uint64), ("client_key", C.c_uint32), ("id_idx", C.c_uint32), ("sub_id", C.c_uint32), ("flags", C.c_uint32)]

    rng = random.Random(99)
    n_rels = 900
    rels = (GmRel * n_rels)()
    table = []
    for h in range(n_rels):
        live = rng.random() < 0.9
        v5 = rng.random() < 0.6
        group = rng.choice([0, 0, 0, 1, 2])
        flags = (1 if live else 0) | (2 if v5 else 0) | (4 if rng.random() < 0.3 else 0) | (group << 8)
        r = dict(node_id=rng.randint(1, 3), client_key=rng.randint(0, 120), id_idx=rng.randint(0, 200), sub_id=rng.choice([0, 0, 3, 7, 9]), flags=flags)
        table.append(r)
        rels[h].node_id, rels[h].client_key, rels[h].id_idx, rels[h].sub_id, rels[h].flags = r["node_id"], r["client_key"], r["id_idx"], r["sub_id"], r["flags"]
    lists = []
    for t in range(120):
        k = rng.choice([0, 1, 5, 40, 300, 700]) if t % 10 else 700
        lst = [rng.randint(0, n_rels + 20) for _ in range(k)]
        if lst and rng.random() < 0.5:
            lst += lst[:3]                                  # the same handle twice (literal '+' / '#' topic levels)
        lists.append(lst)
    n = len(lists)
    spans = np.zeros((n, 2), dtype=np.uint32)
    ids = np.asarray([h for l in lists for h in l] + [0], dtype=np.uint32)
    o = 0
    for i, l in enumerate(lists):
        spans[i] = (o, len(l)); o += len(l)
    pubs = np.asarray([rng.choice([0xFFFFFFFF, rng.randint(0, 200)]) for _ in range(n)], dtype=np.uint32)
    cap_r, cap_s = len(ids) + 8, len(ids) + 8
    out_spans = np.zeros((n, 2), dtype=np.uint32)
    out_rels = (N.GmSubRelation * cap_r)()
    out_subs = np.zeros(cap_s, dtype=np.uint32)
    needed = np.zeros(3, dtype=np.uint64)
    status = np.zeros(n, dtype=np.int32)
    rc = emu.emu_relations(C.c_void_p(spans.ctypes.data), C.c_void_p(ids.ctypes.data), C.c_uint64(n), C.c_void_p(pubs.ctypes.data), rels, C.c_uint64(n_rels),
                           C.c_void_p(out_spans.ctypes.data), out_rels, C.c_uint64(cap_r), C.c_void_p(out_subs.ctypes.data), C.c_uint64(cap_s),
                           C.c_void_p(needed.ctypes.data), C.c_void_p(status.ctypes.data))
    assert rc == 0
    tot_r = tot_s = 0
    flagged = 0
    for t, lst in enumerate(lists):
        direct, v5 = [], []
        for h in lst:
            if h >= n_rels:
                continue
            r = table[h]
            if not r["flags"] & 1:
                continue
            if (r["flags"] & 2) and (r["flags"] & 4) and pubs[t] != 0xFFFFFFFF and r["id_idx"] == pubs[t]:
                continue                                    # no_local: the publisher's own subscription
            (v5 if (r["flags"] & 2) and (r["flags"] >> 8) == 0 else direct).append(h)
        want = [(table[h]["node_id"], h, table[h]["flags"] >> 8, ()) for h in direct]
        if len(v5) > 256:                                   # handed over un-deduplicated, the topic is flagged
            want += [(table[h]["node_id"], h, 0, ()) for h in v5]
            assert status[t] == 1
            flagged += 1
        else:
            assert status[t] == 0
            by_client = {}
            for h in v5:
                by_client.setdefault(table[h]["client_key"], []).append(h)
            for key, hs in by_client.items():
                rep = min(hs)
                subs = tuple(table[h]["sub_id"] for h in hs if table[h]["sub_id"])
                want.append((table[rep]["node_id"], rep, 0, subs))
                tot_s += len(subs)
        off, cnt = int(out_spans[t, 0]), int(out_spans[t, 1])
        got = []
        for k in range(cnt):
            sr = out_rels[off + k]
            got.append((sr.node_id, sr.handle, sr.group, tuple(int(x) for x in out_subs[sr.sub_ids_off:sr.sub_ids_off + sr.sub_ids_cnt])))
        assert sorted(got) == sorted(want), t
        tot_r += cnt
    assert flagged >= 1 and int(needed[0]) == tot_r and int(needed[1]) == tot_s


def _match_ex(e, blob, offs, sel, flags):
    n_entries, n = len(offs) - 1, len(sel)
    spans = np.zeros((n, 2), dtype=np.uint32)
    status = np.zeros(n, dtype=np.int32)
    needed = C.c_uint64(0)
    cap = 1024
    e.lib.emu_match_ex.restype = C.c_int32
    while True:
        ids = np.zeros(cap, dtype=np.uint32)
        rc = e.lib.emu_match_ex(e.h, C.c_void_p(blob.ctypes.data), C.c_void_p(offs.ctypes.data), C.c_uint64(n_entries), C.c_void_p(sel.ctypes.data), C.c_uint64(n), None, flags,
                                C.c_void_p(spans.ctypes.data), C.c_void_p(ids.ctypes.data), C.c_uint64(cap), C.byref(needed), C.c_void_p(status.ctypes.data), None, None)
        if rc == -3:
            cap = int(needed.value) + 16
            continue
        assert rc == 0, rc
        return MatchResult(spans, ids[:int(needed.value)], status, int(needed.value))


@pytest.mark.parametrize("flags", [8, 9, 16, 17, 24])
def test_selection_and_capacity_sized_launches(emu, flags):
    """gm_match_args.d_sel (row t = entry sel[t]: a rank's share of a mixed batch) and the small-batch-graph form (kernels launched
    for a capacity, the real batch size read from a header; rows beyond the batch must stay untouched)."""
    rng = random.Random(200 + flags)
    e, tree = Emu(emu), orc.TopicTree()
    _random_trie(e, tree, rng, 900)
    topics = [rand_topic(rng) for _ in range(500)]
    tb, to = pack(topics)
    rows = np.asarray(rng.sample(range(len(topics)), 180) if flags & 8 else list(range(len(topics))), dtype=np.uint32)
    res = _match_ex(e, tb, to, rows, flags)
    for t, ent in enumerate(rows):
        w = tree.matches(topics[int(ent)])
        assert res.sorted_list(t) == (None if w is None else sorted(w)), topics[int(ent)]
    e.close()


def _shard_of(s, world):
    from rmqtt_b200 import _native as N
    b = s.encode()
    return int(N.lib().gm_shard_of(b, len(b), world))


def test_partition_kernel_equals_the_host_shard_function(emu):
    rng = random.Random(31)
    topics = [rand_topic(rng) for _ in range(1000)] + ["+", "#", "+/a", "#/x", "", "/a"]
    tb, to = pack(topics)
    n = len(topics)
    for world in (1, 2, 8, 1500):                     # 1500 shards: the histogram leaves shared memory
        for rank in (0, world - 1):
            sel = np.full(n, 0xFFFFFFFF, dtype=np.uint32)
            shard = np.zeros(n, dtype=np.uint32)
            counts = np.zeros(world + 1, dtype=np.uint32)
            assert emu.emu_partition(C.c_void_p(tb.ctypes.data), C.c_void_p(to.ctypes.data), C.c_uint64(n), world, rank, C.c_void_p(sel.ctypes.data), C.c_void_p(shard.ctypes.data),
                                     C.c_void_p(counts.ctypes.data)) == 0
            want = np.asarray([0 if t.split("/")[0] in ("+", "#") else _shard_of(t, world) for t in topics], dtype=np.uint32)
            assert (shard == want).all()
            assert (counts[:world] == np.bincount(want, minlength=world)).all()
            k = int(counts[world])
            assert sorted(sel[:k].tolist()) == np.nonzero(want == rank)[0].tolist() and (sel[k:] == 0xFFFFFFFF).all()


@pytest.mark.parametrize("world,direct", [(2, 0), (2, 1), (8, 0), (8, 1), (5, 0)])
def test_fused_gather_over_emulated_peer_memory(emu, world, direct):
    """The multi-GPU step with the exchange fused into the match kernels, ALL ranks emulated in this process (a peer's block is
    just another host buffer): k_partition -> k_match_fast<GATHER> / k_match_slow<GATHER> -> k_gather_push (push form) or stores
    into every block from the publish phase (direct form) -> k_gather_finish.  Every rank's block must then hold every topic's
    list exactly once, equal to the unsharded oracle — at 2, 5 and 8 ranks (the 8-rank push form had no GPU run of its own)."""
    for f in ("emu_match_gather", "emu_gather_finish"):
        getattr(emu, f).restype = C.c_int32
    emu.emu_gather_new.restype = C.c_void_p
    emu.emu_gather_slab_ids.restype = C.c_uint64
    emu.emu_gather_slab_topics.restype = C.c_uint64
    rng = random.Random(1000 + 10 * world + direct)
    tree = orc.TopicTree()
    engines = [Emu(emu) for _ in range(world)]
    for en in engines:
        emu.emu_set_pool_rows(en.h, 2)                # some topics take the deferred kernel on every rank
    roots = ["a", "b", "c", "d", "e", "f", "g", "h", "r1", "r2", "r3", "r4", "r5", "r6", "r7", "r8", "", "$SYS"]
    for _ in range(2500):
        f, v = rand_filter(rng), rng.randint(0, 30)
        if rng.random() < 0.7:
            f = rng.choice(roots) + "/" + f
        try:
            tree.insert(f, v)
        except ValueError:
            continue
        s = _shard_of(f, world)
        for r, en in enumerate(engines):
            if s == 0xFFFFFFFF or s == r:             # root wildcards are replicated on every shard
                assert en.add(f, v) == 0
    for v in range(40):                               # a replicated filter with many values: > 2 + 8 matched sets for deep topics
        tree.insert("+/#", 5000 + v)
        for en in engines:
            en.add("+/#", 5000 + v)
    topics = [(rng.choice(roots) + "/" if rng.random() < 0.7 else "") + rand_topic(rng) for _ in range(1200)] + ["+/a", "#", "/".join(["a"] * 11)]
    tb, to = pack(topics)
    n = len(topics)
    want = tree.match_batch(tb, to)
    gw = C.c_void_p(emu.emu_gather_new(world, n, int(want["counts"].clip(0).sum()) + 64))
    slab_t, slab_i = int(emu.emu_gather_slab_topics(gw)), int(emu.emu_gather_slab_ids(gw))
    n_local = []
    for r, en in enumerate(engines):
        sel = np.zeros(n, dtype=np.uint32)
        counts = np.zeros(world + 1, dtype=np.uint32)
        emu.emu_partition(C.c_void_p(tb.ctypes.data), C.c_void_p(to.ctypes.data), C.c_uint64(n), world, r, C.c_void_p(sel.ctypes.data), None, C.c_void_p(counts.ctypes.data))
        k = int(counts[world])
        n_local.append(k)
        status = np.zeros(max(k, 1), dtype=np.int32)
        rc = emu.emu_match_gather(gw, r, en.h, C.c_void_p(tb.ctypes.data), C.c_void_p(to.ctypes.data), C.c_uint64(n), C.c_void_p(sel.ctypes.data), C.c_uint64(k), direct,
                                  C.c_void_p(status.ctypes.data))
        assert rc == 0, rc
    assert sum(n_local) == n
    # end of step: on a real node the ranks run this concurrently; here one after the other — the early ones give up waiting
    # (bounded spin, error word set), the last one sees every flag; a second look at the same epoch then passes everywhere
    first = [emu.emu_gather_finish(gw, r, C.c_uint64(n_local[r]), 1) for r in range(world)]
    assert first[-1] == 0 and (world == 1 or first[0] == 1)
    assert [emu.emu_gather_finish(gw, r, C.c_uint64(n_local[r]), 0) for r in range(world)] == [0] * world
    wc, wi = _canon(want)
    blocks = []
    for r in range(world):
        counts = np.zeros((world, 2), dtype=np.uint64)
        index = np.zeros(world * slab_t, dtype=np.uint32)
        spans = np.zeros((world * slab_t, 2), dtype=np.uint32)
        ids = np.zeros(world * slab_i, dtype=np.uint32)
        emu.emu_gather_read(gw, r, C.c_void_p(counts.ctypes.data), C.c_void_p(index.ctypes.data), C.c_void_p(spans.ctypes.data), C.c_void_p(ids.ctypes.data))
        assert [int(c) for c in counts[:, 0]] == n_local
        rows = np.concatenate([np.arange(q * slab_t, q * slab_t + n_local[q]) for q in range(world)])
        idx = index[rows]
        assert sorted(idx.tolist()) == list(range(n))                       # every topic exactly once
        order = np.argsort(idx)
        got = MatchResult(spans[rows][order], ids, np.where(wc < 0, -2, 0).astype(np.int32), 0)
        cg, ig = got.canonical()
        assert (cg == wc).all() and len(ig) == len(wi) and (ig == wi).all(), f"rank {r}"
        blocks.append((idx, spans[rows], [int(c) for c in counts[:, 1]]))
    for r in range(1, world):                                               # and every rank holds the same thing
        assert (blocks[r][0] == blocks[0][0]).all() and (blocks[r][1] == blocks[0][1]).all() and blocks[r][2] == blocks[0][2]
    emu.emu_gather_free(gw)
    for en in engines:
        en.close()


# ---- hypothesis-driven (the strategies of tests/test_hypothesis_cpu.py): arbitrary add / remove interleavings, matched by the
#      emulated kernels — the CPU twin of tests/test_gpu_hypothesis.py ------------------------------------------------------------------
from hypothesis import HealthCheck, given, settings, strategies as st          # noqa: E402

from test_hypothesis_cpu import ops as hyp_ops, path as hyp_path, retain_ops as hyp_retain_ops   # noqa: E402

import os as _os                                                                  # noqa: E402

_HYP = dict(deadline=None, max_examples=int(_os.environ.get("GM_HYP_EMU_EXAMPLES", "40")), suppress_health_check=[HealthCheck.too_slow, HealthCheck.function_scoped_fixture])


@settings(**_HYP)
@given(ops=hyp_ops, topics=st.lists(hyp_path, min_size=1, max_size=30), flags=st.sampled_from([0, 1, 2]))
def test_hypothesis_subscription_trie_emulated_kernels_vs_oracle(emu, ops, topics, flags):
    e, tree = Emu(emu), orc.TopicTree()
    for op, f, v in ops:
        rc = e.add(f, v) if op == "add" else e.remove(f, v)
        if rc != 0:
            continue
        tree.insert(f, v) if op == "add" else tree.remove(f, v)
    tb, to = pack(topics)
    res, _, _ = e.match(tb, to, flags)
    for i, t in enumerate(topics):
        assert res.sorted_list(i) == tree.matches(t), t
    e.close()


@settings(**_HYP)
@given(ops=hyp_retain_ops, filters=st.lists(hyp_path, min_size=1, max_size=30))
def test_hypothesis_retained_tree_emulated_kernels_vs_oracle(emu, ops, filters):
    e, tree = Emu(emu), orc.RetainTree()
    fb0, fo0 = pack(["#"])
    for op, t, v in ops:
        if op == "flush":                            # make the image current (later operations edit it in place)
            e.retain_match(fb0, fo0)
            continue
        rc = e.retain_set(t, v) if op == "set" else e.retain_remove(t)
        if rc != 0:
            continue
        tree.insert(t, v) if op == "set" else tree.remove(t)
    fb, fo = pack(filters)
    res, _, _ = e.retain_match(fb, fo)
    for i, f in enumerate(filters):
        assert res.sorted_list(i) == tree.matches(f), f
    e.close()


def test_workload_generator_shapes_on_parallel_built_tables(emu):
    """C3- and C4-shaped data from the workload generator (64-way fan-out at the top: wide nodes with the child filter, several
    windows of the edge table, the locality sort with populated buckets), the tables built by the all-host-threads bulk paths —
    the emulated kernels against the oracle, exact work counters included."""
    from rmqtt_b200 import workload as wl
    emu.emu_bulk_load.restype = C.c_uint64
    emu.emu_retain_bulk_load.restype = C.c_uint64
    cfg = wl.C3.scaled(n_subs=300_000, n_topics=8_000)
    sb, so, sv = wl.gen_subs(cfg)
    tb, to = wl.gen_topics(cfg)
    e, tree = Emu(emu), orc.TopicTree()
    assert emu.emu_bulk_load(e.h, C.c_void_p(sb.ctypes.data), C.c_void_p(so.ctypes.data), C.c_void_p(sv.ctypes.data), C.c_uint64(len(sv))) == len(sv)
    tree.bulk_insert(sb, so, sv, nthreads=4)
    want = tree.match_batch(tb, to, nthreads=4)
    for flags in (4, 1):
        res, work, _ = e.match(tb, to, flags)
        _same(res, want)
        if flags & 4:
            c = want["counters"]
            assert [int(x) for x in work] == [c["V"], c["E"], c["F"], c["M"]]
    rcfg = wl.C4.scaled(n_subs=200_000, n_topics=1_000)
    rb, ro, rv = wl.gen_retained(rcfg)
    fb, fo = wl.gen_retain_filters(rcfg)
    rt = orc.RetainTree()
    assert emu.emu_retain_bulk_load(e.h, C.c_void_p(rb.ctypes.data), C.c_void_p(ro.ctypes.data), C.c_void_p(rv.ctypes.data), C.c_uint64(len(rv))) == rt.bulk_insert(rb, ro, rv)
    res, _, _ = e.retain_match(fb, fo)
    _same(res, rt.match_batch(fb, fo, nthreads=4))
    e.close()


@pytest.mark.parametrize("seed,tiny", [(41, False), (42, True), (43, False)])
def test_device_image_is_kept_current_by_the_dirty_lists_alone(emu, seed, tiny, monkeypatch):
    """The kernels read a COPY of every table that only the engine's shipping policy updates (whole table after a re-hash,
    appended tails, the 32-byte slots the host mirror listed as dirty — rmqtt_b200/csrc/pipeline.h ship(), which gm_engine::flush_impl runs).  A slot
    the mirror changed without listing it would stay stale in the copy and show up as a wrong match.  Rounds of single
    add / remove, a bulk load in between (tables re-hashed), a compaction; subscription trie and retained tree."""
    if tiny:
        monkeypatch.setenv("GM_WIN_MIN_SLOTS_LOG2", "3")
    rng = random.Random(seed)
    for f in ("emu_flush", "emu_compact"):
        getattr(emu, f).restype = C.c_int32
    emu.emu_bulk_load.restype = C.c_uint64
    e, tree, rt = Emu(emu), orc.TopicTree(), orc.RetainTree()
    emu.emu_use_image(e.h, 0)
    live, names, hist = [], [], []
    for rnd in range(7):
        for _ in range(400):
            r = rng.random()
            if r < 0.45 or not live:
                f, v = rand_filter(rng), rng.randint(0, 30)
                if e.add(f, v) == 0:
                    tree.insert(f, v); live.append((f, v))
            elif r < 0.7:
                f, v = live.pop(rng.randrange(len(live)))
                assert e.remove(f, v) == 0
                tree.remove(f, v)
            elif r < 0.9 or not names:
                # (plain levels except in round 5: a stored literal '+' / '#' level makes the host give the in-place image up
                #  and re-flatten — shipped whole — which would hide the patch path this test is about)
                t = rand_topic(rng, max_depth=6) if rnd == 5 else "/".join(rng.choice(["a", "b", "c", "d", "", "x" * 30, "$SYS"]) for _ in range(rng.randint(1, 5)))
                v = rng.randint(0, 10**6)
                if e.retain_set(t, v) == 0:
                    rt.insert(t, v); names.append(t)
            else:
                t = names.pop(rng.randrange(len(names)))
                e.retain_remove(t); rt.remove(t)
        if rnd == 2:                                   # a bulk load through the all-threads path: edge table re-hashed, shipped whole
            monkeypatch.setenv("GM_HOST_PAR_MIN", "1"); monkeypatch.setenv("GM_HOST_THREADS", "4")
            fs = [rand_filter(rng) for _ in range(3000)]
            ok = []
            for f in fs:
                try:
                    tree.insert(f, 77); ok.append(f)
                except ValueError:
                    pass
            fb, fo = pack(fs)
            assert emu.emu_bulk_load(e.h, C.c_void_p(fb.ctypes.data), C.c_void_p(fo.ctypes.data), C.c_void_p(np.full(len(fs), 77, np.uint32).ctypes.data), C.c_uint64(len(fs))) >= 1
            live += [(f, 77) for f in set(ok)]
            monkeypatch.delenv("GM_HOST_PAR_MIN"); monkeypatch.delenv("GM_HOST_THREADS")
        if rnd == 4:
            assert emu.emu_compact(e.h) == 0
        topics = [rand_topic(rng) for _ in range(300)]
        tb, to = pack(topics)
        res, _, _ = e.match(tb, to, rnd % 2)           # ids and descriptor mode alternate
        _same(res, tree.match_batch(tb, to))
        filters = [rand_filter(rng, 6) for _ in range(150)] + ["#", "+/#"]
        qb, qo = pack(filters)
        rres, _, _ = e.retain_match(qb, qo)
        _same(rres, rt.match_batch(qb, qo))
        ctr = np.zeros(6, dtype=np.uint64)
        emu.emu_retain_counters(e.h, C.c_void_p(ctr.ctypes.data))
        hist.append((int(ctr[0]), int(ctr[1])))
    # some round of plain topics edited the shipped image in place without a re-flatten (re-packs happen too: garbage, the compaction)
    assert any(b[0] == a[0] and b[1] > a[1] for a, b in zip(hist, hist[1:])), hist
    e.close()


def test_manual_flush_engines_match_the_last_shipped_snapshot(emu):
    """GM_FLAG_MANUAL_FLUSH: between fences the kernels keep matching the tables as of the last flush, whatever the host mirror has
    become meanwhile (new filters, a table that grew and re-hashed)."""
    emu.emu_flush.restype = C.c_int32
    rng = random.Random(7)
    e, tree = Emu(emu), orc.TopicTree()
    emu.emu_use_image(e.h, 1)
    _random_trie(e, tree, rng, 600)
    topics = [rand_topic(rng) for _ in range(300)]
    tb, to = pack(topics)
    res, _, _ = e.match(tb, to, 0)                     # (first match ships the tables)
    before = tree.match_batch(tb, to)
    _same(res, before)
    for f, v in [(rand_filter(rng), rng.randint(0, 9)) for _ in range(5000)]:      # enough to grow and re-hash the edge table
        if e.add(f, v) == 0:
            tree.insert(f, v)
    res, _, _ = e.match(tb, to, 0)
    _same(res, before)                                 # not flushed: the old snapshot answers
    assert emu.emu_flush(e.h) == 0
    res, _, _ = e.match(tb, to, 0)
    after = tree.match_batch(tb, to)
    assert int(after["counts"].clip(0).sum()) > int(before["counts"].clip(0).sum())
    _same(res, after)
    e.close()


# ---- the reference's own unit-test vectors (tests/golden/reference_asserts.json: trie.rs:417-498, retain.rs:451-475 and the derived
#      `$` / literal-wildcard cases) replayed through the emulated kernels --------------------------------------------------------------
def _emu_matches(e, topic, flags=0):
    tb, to = pack([topic])
    res, _, _ = e.match(tb, to, flags)
    return res.sorted_list(0)


def _emu_retain_matches(e, filt):
    fb, fo = pack([filt])
    res, _, _ = e.retain_match(fb, fo)
    return res.sorted_list(0)


def test_golden_trie_vectors_through_the_emulated_kernels(emu, golden):
    g = golden["trie_A1"]
    e = Emu(emu)
    for f, v in g["inserts"]:
        assert e.add(f, v) == 0
    for topic, want in g["matches"]:
        assert _emu_matches(e, topic) == sorted(want), topic
    for topic, bad in g["not_matches"]:
        assert _emu_matches(e, topic) != sorted(bad)
    for f, v, _want in g["removes"]:
        e.remove(f, v)
    for topic, want in g["after_remove_matches"]:
        assert _emu_matches(e, topic, 1) == sorted(want), topic
    e.close()
    g = golden["trie_A2"]
    e = Emu(emu)
    for f, v in g["inserts"]:
        e.add(f, v)
    r = g["range_inserts"]
    for v in range(r["lo"], r["hi"]):
        e.add(r["pattern_each"].format(v=v), v)
    for v in range(r["lo"], r["hi"]):
        e.add(r["pattern_same"], v)
    for topic, want in g["matches"]:
        assert _emu_matches(e, topic) == sorted(want), topic
    assert _emu_matches(e, "/iot/x") == sorted(list(range(1, 10000)) + [3])      # 10 000 ids in one set
    for f, v in g["stage2_inserts"]:
        e.add(f, v)
    for topic, want in g["stage2_matches"]:
        assert _emu_matches(e, topic) == sorted(want), topic
    for f, v in g["stage3_inserts"]:
        e.add(f, v)
    for topic, want in g["stage3_matches"]:
        assert _emu_matches(e, topic) == sorted(want), topic                     # the same id under two filters is reported twice
    e.close()
    g = golden["derived_A5"]["trie"]
    e = Emu(emu)
    for f, v in g["inserts"]:
        e.add(f, v)
    for topic, want in g["matches"]:
        assert _emu_matches(e, topic) == sorted(want), topic
    e.close()


def test_golden_retain_vectors_through_the_emulated_kernels(emu, golden):
    g = golden["retain_A3"]
    e = Emu(emu)
    for topic, v in g["inserts"]:
        assert e.retain_set(topic, v & 0xFFFFFFFF) == 0
    for f, want in g["matches"]:
        assert _emu_retain_matches(e, f) == sorted(w & 0xFFFFFFFF for w in want), f
    for f, bad in g["not_matches"]:
        assert _emu_retain_matches(e, f) != sorted(bad)
    for topic, v in g["more_inserts"]:
        e.retain_set(topic, v & 0xFFFFFFFF)
    for f, want in g["more_matches"] + golden["derived_A5"]["retain_on_A3"]:
        assert _emu_retain_matches(e, f) == sorted(w & 0xFFFFFFFF for w in want), f
    e.close()


def test_value_set_size_boundary_wide_nodes_tiny_windows_and_an_empty_spill_pool(emu, monkeypatch):
    """Edges of the layout: a value set of 65534 members is the largest that stays in-line for the fast kernel, 65535 goes through
    the `ranges` indirection on the deferred kernel; nodes with more than 48 children (child filter) in 8-slot windows (linear
    probing wraps, windows overflow and the table re-hashes); no spill rows for matched sets (the 9th set defers the topic)."""
    emu.emu_bulk_load.restype = C.c_uint64
    for nset, want_deferred in ((65534, 0), (65535, 3)):
        e, tree = Emu(emu), orc.TopicTree()
        fb, fo = pack(["big/+", "big/#"] * nset)
        vals = np.repeat(np.arange(nset, dtype=np.uint32), 2)
        assert emu.emu_bulk_load(e.h, C.c_void_p(fb.ctypes.data), C.c_void_p(fo.ctypes.data), C.c_void_p(vals.ctypes.data), C.c_uint64(len(vals))) == len(vals)
        tree.bulk_insert(fb, fo, vals)
        e.add("big/x", 7); tree.insert("big/x", 7)
        tb, to = pack(["big/x", "big", "big/x/y", "small"])
        for flags in (0, 1, 5):
            res, work, deferred = e.match(tb, to, flags)
            want = tree.match_batch(tb, to)
            _same(res, want)
            assert deferred == want_deferred
            if flags & 4:
                c = want["counters"]
                assert [int(x) for x in work] == [c["V"], c["E"], c["F"], c["M"]]
        e.close()
    monkeypatch.setenv("GM_WIN_MIN_SLOTS_LOG2", "3")
    rng = random.Random(3)
    e, tree = Emu(emu), orc.TopicTree()
    emu.emu_set_pool_rows(e.h, 0)
    for _ in range(3000):
        f = f"w/{rng.randrange(200)}/{rng.choice(['+', 'a', 'b', '#'])}" if rng.random() < 0.7 else f"{rng.randrange(120)}/x/{rng.randrange(5)}"
        v = rng.randrange(50)
        tree.insert(f, v)
        assert e.add(f, v) == 0
    for v in range(12):
        for f in ("#", "+/#", "w/#", "w/+/#", "w/+/+", "+/+/+", "+/+/#", "w/+/a", "+/5/+", "w/5/#"):
            tree.insert(f, 1000 + v); e.add(f, 1000 + v)
    topics = [f"w/{rng.randrange(220)}/{rng.choice(['a', 'b', 'c'])}" for _ in range(1200)] + [f"{rng.randrange(130)}/x/{rng.randrange(6)}" for _ in range(400)]
    tb, to = pack(topics)
    for flags in (0, 1, 2):
        res, _, deferred = e.match(tb, to, flags)
        _same(res, tree.match_batch(tb, to))
        assert deferred > 500                     # more than 8 matched sets and nowhere to spill them
    e.close()


def test_retained_lookup_beyond_the_eight_level_token_row(emu):
    """Retained topics and filters of up to 14 levels (levels >= 8 live in the level-major token array), literal '+' / '#' levels
    that shadow wildcard expansion, `$` roots, removals — scratch starting small."""
    rng = random.Random(8)
    e, rt = Emu(emu), orc.RetainTree()

    def deep_topic():
        lv = [rng.choice(["a", "b", "c", "", "dd"]) if rng.random() < 0.93 else rng.choice(["+", "#"]) for _ in range(rng.randint(1, 14))]
        if rng.random() < 0.1:
            lv[0] = "$x"
        return "/".join(lv)

    def deep_filter():
        lv = [rng.choice(["a", "b", "c", "", "dd", "+", "+"]) for _ in range(rng.randint(1, 14))]
        if rng.random() < 0.3:
            lv[-1] = "#"
        if rng.random() < 0.05:
            lv[0] = "$x"
        return "/".join(lv)

    for i in range(5000):
        t = deep_topic()
        if e.retain_set(t, i) == 0:
            rt.insert(t, i)
        if i % 7 == 3:
            t2 = deep_topic()
            if e.retain_remove(t2) == 0:
                rt.remove(t2)
    fl = [deep_filter() for _ in range(1200)] + ["#", "+/#", "+/+/+/+/+/+/+/+/+/#", "a/a/a/a/a/a/a/a/a/a/+", "/".join(["+"] * 12)]
    fb, fo = pack(fl)
    res, _, grew = e.retain_match(fb, fo, cap_items=256, cap_desc=256)
    assert grew >= 1
    _same(res, rt.match_batch(fb, fo))
    e.close()
