"""CPU tier: the CONTROL FLOW of bench.py's own arm, which no GPU-less box can otherwise execute.

`run_own` is driven end to end against a fake engine whose answers come from the oracle (so the parity self-check inside the
bench really compares lists), with torch on "cpu".  What this pins: every name the function uses exists on every path, the
line carries the contract keys, a failing secondary leg lands under `errors` without taking the headline down (the C4 and
relations legs need entry points the fake does not have), and the abnormal-end paths (`_bail`, the watchdog) print
the headline measured so far exactly once.  Numbers are meaningless here; the GPU tier and the driver's run measure."""
import argparse
import ctypes as C
import io
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


class _FakeEngine:
    """The slice of rmqtt_b200.engine.Engine that bench.run_own touches; matching is done by the oracle's TopicTree."""
    _h = None

    def __init__(self, device=-1, filters_hint=0, **_):
        from oracle import oracle as orc
        self.tree = orc.TopicTree()
        self.n_values = 0
        self.cache = {}
        self.launches = 0
        self._world = 1

    def bulk_load(self, blob, offs, values):
        self.n_values += self.tree.bulk_insert(blob, offs, values)
        return len(values)

    def flush(self):
        pass

    def close(self):
        pass

    def stats(self):
        return {"values": self.n_values, "nodes": self.tree.nodes_size(), "edges": self.tree.nodes_size(), "edge_slots": 1 << 20, "dict_entries": 1,
                "plus_nodes": 1, "device_bytes": 1 << 30, "max_depth": 6}

    @staticmethod
    def comm_unique_id():
        return b"\0" * 128

    def comm_init(self, uid, rank, world):
        self._world = world

    def _match(self, d_blob, d_offs):
        key = (d_blob.data_ptr(), d_offs.data_ptr())
        if key not in self.cache:
            blob = d_blob.numpy()
            offs = d_offs.numpy().view(np.uint32)
            self.cache[key] = self.tree.match_batch(blob, offs, nthreads=2, want_ids=True)
        return self.cache[key]

    def match_batch_device(self, d_blob, d_offs, d_spans, d_ids, d_needed, d_status, stream, work=False):
        return self.match_batch_device_ex(d_blob, d_offs, d_spans, d_ids, d_needed, d_status, stream, work=work)

    def match_batch_device_ex(self, d_blob, d_offs, d_spans, d_out, d_needed, d_status, stream, *, desc=False, d_sel=None, n_sel=None, work=False):
        r = self._match(d_blob, d_offs)
        n = len(r["counts"])
        self.launches += 5
        m = int(r["offsets"][-1])
        d_needed[0] = m
        if not desc and m <= d_out.numel():
            d_spans.numpy()[:n, 0] = r["offsets"][:-1].astype(np.int64)
            d_spans.numpy()[:n, 1] = np.maximum(r["counts"], 0)
            d_out.numpy()[:m] = r["ids"].view(np.int32)
            d_status.numpy()[:n] = 0
        if work:
            c = r["counters"]
            return {"visited": c["V"], "probed": c["E"], "filters": c["F"], "ids": m, "levels": 6 * n, "bytes": int(d_blob.numel()), "deferred": 0, "slot_loads": c["E"],
                    "probes_by_depth": [0] * 8, "misses_by_depth": [0] * 8}
        return None

    def partition_batch_device(self, d_blob, d_offs, n_shards, rank, d_sel, stream, d_shard=None):
        n = d_offs.numel() - 1
        d_sel.numpy()[:n] = np.arange(n)
        return n, np.array([n], dtype=np.int64)

    def allgatherv_device(self, d_index, d_spans, k, d_ids, d_m, a_idx, a_spans, a_ids, stream):
        m = int(d_m[0])
        a_idx.numpy()[:k] = d_index.numpy()[:k]
        a_spans.numpy()[:k] = d_spans.numpy()[:k]
        a_ids.numpy()[:m] = d_ids.numpy()[:m]
        return np.array([[k, m]], dtype=np.int64)

    peer_memory = True                   # class switch: False = gm_gather_connect fails (no peer-to-peer access)

    def gather_create(self, world, rank, slab_topics, slab_ids):
        if not self.peer_memory:
            raise RuntimeError("no peer memory on a CPU box")
        self._slab_ids = slab_ids
        return b"\0" * 64

    def gather_connect(self, handles):
        pass

    def match_gather_device(self, d_blob, d_offs, d_status, stream, d_sel=None, n_sel=None):
        self._gathered = self._match(d_blob, d_offs)
        self.launches += 7

    def gather_result(self, stream):
        r = self._gathered
        n, m = len(r["counts"]), int(r["offsets"][-1])
        spans = np.stack([r["offsets"][:-1].astype(np.uint32), np.maximum(r["counts"], 0).astype(np.uint32)], axis=1)
        ids = np.zeros(max(self._slab_ids, m), dtype=np.uint32)
        ids[:m] = r["ids"]
        return np.array([[n, m]], dtype=np.int64), np.arange(n, dtype=np.uint32), spans, ids

    def debug_knob(self, name, value):
        pass

    def kernel_ms(self, max_calls=64):
        return np.full((max_calls, 3), 0.1, dtype=np.float32)

    def kernel_launches(self):
        return self.launches


class _FakeLib:
    """libgpumqtt entry points bench.run_own calls directly (host-buffer calls are not executed: rc 0, sizes filled in)."""

    def __init__(self, real=None):
        self.bufs = {}
        self._real = real

    def __getattr__(self, name):                 # pure host functions (gm_shard_of ...) are the real library's; the router's gmr_* are
        if name.startswith("gm_") and self._real is not None:      # not served, also where a device would let them run
            return getattr(self._real, name)
        raise AttributeError(name)

    def gm_bind_thread_near_device(self, dev):
        return 0

    def gm_host_alloc_near(self, h, nbytes):
        b = C.create_string_buffer(int(nbytes))
        self.bufs[C.addressof(b)] = b
        return C.addressof(b)

    def gm_host_free(self, p):
        self.bufs.pop(p, None)

    def gm_device_numa_node(self, dev):
        return 0

    def gm_last_error(self, h):
        return b"fake"

    def gm_match_batch(self, h, pb, po, n, spans, ids, cap, need, status):
        need._obj.value = 7
        return 0

    gm_match_batch_desc = gm_match_batch

    def gm_churn_probe(self, *a):
        return 0

    def gm_batcher_probe(self, *a):
        return 0


class _Event:
    def __init__(self, enable_timing=False):
        pass

    def record(self):
        pass

    def elapsed_time(self, other):
        return 1.0


class _Stream:
    cuda_stream = 0


@pytest.fixture
def fake_gpu(monkeypatch):
    import torch
    import bench
    from rmqtt_b200 import _native as N
    from rmqtt_b200 import engine as E
    monkeypatch.setattr(bench, "_DEVICE_KIND", "cpu")
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a: None)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a: _Stream())
    monkeypatch.setattr(torch.cuda, "Event", _Event)
    monkeypatch.setattr(E, "Engine", _FakeEngine)
    fake = _FakeLib(real=N.lib())
    monkeypatch.setattr(N, "lib", lambda: fake)
    out = io.StringIO()
    monkeypatch.setattr(bench, "_RESULT_OUT", out)
    monkeypatch.setattr(bench, "_EMITTED", False)
    bench._PARTIAL.clear()
    monkeypatch.setenv("RANK", "0")
    monkeypatch.setenv("WORLD_SIZE", "1")
    monkeypatch.setenv("LOCAL_RANK", "0")
    monkeypatch.setattr(bench.ClockSampler, "start", lambda self: None)
    yield bench, out
    bench._PARTIAL.clear()


def _ns(**kw):
    d = dict(gpus=1, steps=3, warmup=3, impl="own", subs=20_000, topics=2_000, batches=2, no_cpu_baseline=False, e2e_steps=None, no_c4=False,
             dump_outputs=None)
    d.update(kw)
    return argparse.Namespace(**d)


CONTRACT = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
            "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks", "multi_gpu", "parity_check", "c4", "latency", "churn", "relations")


def test_run_own_walks_every_leg_and_isolates_the_failing_ones(fake_gpu):
    bench, out = fake_gpu
    bench.run_own(_ns())
    lines = [l for l in out.getvalue().splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in CONTRACT:
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["higher_is_better"] is True and d["scaling"] == "weak" and "workload" in d["config"]
    assert d["value"] > 0 and d["gpu_launches"] == 15
    for k in ("value", "h2d_bytes_per_step", "d2h_bytes_per_step", "ids_mode", "single_caller"):
        assert k in d["e2e"], k
    assert set(d["e2e"]["by_caller_threads"]) == {"2", "3"} and d["e2e"]["value"] == max(d["e2e"]["by_caller_threads"].values())
    assert d["e2e"]["caller_threads"] in (2, 3)
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["kernel"] == "k_match_fast" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert abs(r["descriptor_mode"]["frac"] - r["descriptor_mode"]["achieved"] / r["peak"]) < 1e-12
    assert d["parity_check"]["ok"] is True and d["parity_check"]["topics"] == 2000          # the oracle-backed fake really was compared
    assert d["multi_gpu"]["strong_fused"]["value"] > 0 and d["parity_check"]["fused_ok"] is True      # the peer-memory leg and its self-check
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0 and d["cpu_baseline"]["cores"] >= 1
    assert len(d["churn"]["legs"]) == 4 and d["churn"]["port_single_thread_ops_per_s"] > 0
    assert len(d["latency"]["table"]) == 5
    # the two legs the fake cannot serve (retained tree, GpuRouter): reported, not fatal
    assert d["c4"] is None and d["relations"] is None
    assert set(d["errors"]) == {"c4", "relations"}, d["errors"]
    # C1 / C2 through tools/bench_configs.py and the Zipf batch ride on the fake too (count parity is real: oracle vs oracle-backed fake)
    assert set(d["configs"]) == {"C1", "C2", "C3-zipf"} and d["configs"]["C1"]["count_parity"] is True and d["configs"]["C2"]["count_parity"] is True
    assert d["configs"]["C3-zipf"]["topics_per_s"] > 0


def test_run_own_without_the_cpu_legs(fake_gpu, monkeypatch):
    bench, out = fake_gpu
    monkeypatch.setattr(_FakeEngine, "peer_memory", False)          # GPUs without peer access: the NCCL path only
    bench.run_own(_ns(no_cpu_baseline=True))
    d = json.loads(out.getvalue())
    assert d["cpu_baseline"] is None and d["churn"] is None and "errors" not in d and d["parity_check"]["ok"] is True
    assert "unavailable" in d["multi_gpu"]["strong_fused"] and "fused_ok" not in d["parity_check"]


def test_an_exception_after_the_headline_still_leaves_the_headline(fake_gpu, monkeypatch):
    bench, out = fake_gpu

    def boom(*a, **k):
        raise RuntimeError("collective leg died")

    monkeypatch.setattr(_FakeEngine, "partition_batch_device", boom)
    with pytest.raises(RuntimeError):
        bench.run_own(_ns(no_cpu_baseline=True))
    assert out.getvalue() == ""                               # nothing printed yet: __main__'s handler prints _PARTIAL through _bail
    p = bench._PARTIAL
    assert p["value"] > 0 and p["e2e"]["value"] > 0 and p["roofline"]["frac"] > 0 and p["multi_gpu"] is None


_BAIL = r"""
import sys, time
sys.path.insert(0, {root!r})
import bench
bench._PARTIAL.update({{"metric": "m", "value": 1.5, "e2e": {{"value": 1.0}}}})
mode = sys.argv[1]
if mode == "bail":
    bench._bail("RuntimeError: leg 3 died", 1)
elif mode == "empty":
    bench._PARTIAL.clear()
    bench._bail("early failure", 1)
elif mode == "rank1":
    bench._bail("x", 1)
elif mode == "watchdog":
    bench._watchdog(0.3)
    time.sleep(30)
"""


@pytest.mark.parametrize("mode, env, rc, printed", [("bail", {}, 0, True), ("empty", {}, 1, False), ("rank1", {"RANK": "1", "WORLD_SIZE": "2"}, 0, False),
                                                    ("watchdog", {}, 0, True)])
def test_abnormal_ends_print_the_partial_line_once(mode, env, rc, printed, tmp_path):
    import os
    script = tmp_path / "bail.py"
    script.write_text(_BAIL.format(root=str(ROOT)))
    e = dict(os.environ)
    e.pop("RANK", None)
    e.update(env)
    r = subprocess.run([sys.executable, str(script), mode], capture_output=True, text=True, timeout=120, env=e)
    assert r.returncode == rc, (r.returncode, r.stderr[-500:])
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == (1 if printed else 0), r.stdout
    if printed:
        d = json.loads(lines[0])
        assert d["value"] == 1.5 and "bench" in d["errors"]


@pytest.mark.parametrize("steps, batch", [(2, 1), (3, 0)])
def test_dump_outputs_holds_the_lists_of_the_last_timed_step(fake_gpu, tmp_path, steps, batch):
    """--dump-outputs: the sorted per-topic lists of the batch the last timed step matched (step k matches batch k % batches),
    as float64, equal to the oracle's lists of that batch."""
    from oracle import oracle as orc
    from rmqtt_b200 import workload as wl
    bench, out = fake_gpu
    args = _ns(steps=steps, batches=2, no_cpu_baseline=True, dump_outputs=str(tmp_path / "dump"))
    bench.run_own(args)
    d = {k: np.load(tmp_path / "dump" / f"{k}.npy") for k in ("topics", "status", "counts", "ids")}
    assert all(a.dtype == np.float64 for a in d.values())
    cfg = bench._cfg(args)
    tree = orc.TopicTree()
    tree.bulk_insert(*wl.gen_subs(cfg))
    want = tree.match_batch(*wl.gen_topics(cfg, cfg.n_topics, stream=batch))
    seg = np.repeat(np.arange(cfg.n_topics), np.maximum(want["counts"], 0))
    assert (d["topics"] == np.arange(cfg.n_topics)).all() and (d["status"] == 0).all()
    assert (d["counts"] == want["counts"]).all() and (d["ids"] == want["ids"][np.lexsort((want["ids"], seg))]).all()


def test_dump_outputs_samples_a_large_batch_the_same_way_within_the_byte_budget(tmp_path, monkeypatch):
    import bench
    from rmqtt_b200.engine import MatchResult
    n, per = 5000, 7
    spans = np.stack([np.arange(n, dtype=np.uint32) * per, np.full(n, per, np.uint32)], axis=1)
    ids = np.random.default_rng(1).integers(0, 1 << 32, n * per, dtype=np.uint64).astype(np.uint32)
    status = np.zeros(n, np.int32)
    status[::97] = -2
    monkeypatch.setattr(bench, "_DUMP_TOPICS", 1000)
    monkeypatch.setattr(bench, "_DUMP_BYTES", 8 * 6000)      # about 600 of the 1000 sampled topics fit (topic, status, count, 7 ids)
    for run in ("a", "b"):
        bench._dump_outputs(str(tmp_path / run), spans, ids, status)
    d = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in ("topics", "status", "counts", "ids")}
    for k, a in d.items():
        assert (a == np.load(tmp_path / "b" / f"{k}.npy")).all(), k
    t = d["topics"].astype(np.int64)
    assert 600 <= len(t) < 1000 and (np.diff(t) > 0).all() and t[-1] > len(t)
    counts, sorted_ids = MatchResult(spans[t], ids, status[t], len(ids)).canonical()
    assert (d["status"] == status[t]).all() and (d["counts"] == counts).all() and (d["ids"] == sorted_ids).all()
    words = sum(a.size for a in d.values())
    assert 6000 - (3 + per) < words <= 6000                 # the next sampled topic would not have fit


def test_a_missed_gather_barrier_keeps_the_fused_timings(fake_gpu, monkeypatch):
    bench, out = fake_gpu

    def boom(self, stream):
        raise RuntimeError("fused gather: a rank did not reach the end-of-step barrier")

    monkeypatch.setattr(_FakeEngine, "gather_result", boom)
    bench.run_own(_ns(no_cpu_baseline=True))
    d = json.loads(out.getvalue())
    f = d["multi_gpu"]["strong_fused"]
    assert f["value"] > 0 and f["gather_get_errors"] and "fused_ok" not in d["parity_check"] and d["parity_check"]["ok"] is True


def test_rank_zero_of_a_two_rank_launch_walks_the_multi_rank_branches(fake_gpu, monkeypatch):
    """WORLD_SIZE=2 with torch.distributed replaced by single-process stand-ins: rank 0 takes every `world > 1` branch of run_own
    (sharded generators, the library communicator, value_with_gather, the broadcast A/B of the collective, the direct-store A/B of
    the fused gather, max-over-ranks reductions).  The fake holds only rank 0's shard, so the gathered lists do not equal the
    unsharded oracle here — the line must say so (`parity_check.ok` false) rather than crash."""
    import torch.distributed as dist
    bench, out = fake_gpu
    monkeypatch.setenv("WORLD_SIZE", "2")
    monkeypatch.setattr(dist, "init_process_group", lambda *a, **k: None)
    monkeypatch.setattr(dist, "destroy_process_group", lambda *a, **k: None)
    monkeypatch.setattr(dist, "barrier", lambda *a, **k: None)
    monkeypatch.setattr(dist, "all_reduce", lambda t, op=None: None)
    monkeypatch.setattr(dist, "broadcast_object_list", lambda objs, src=0: None)

    def all_gather_object(outs, obj):
        for i in range(len(outs)):
            outs[i] = obj
    monkeypatch.setattr(dist, "all_gather_object", all_gather_object)

    def partition(self, d_blob, d_offs, n_shards, rank, d_sel, stream, d_shard=None):      # everything lands on rank 0
        n = d_offs.numel() - 1
        d_sel.numpy()[:n] = np.arange(n)
        counts = np.zeros(n_shards, dtype=np.int64)
        counts[0] = n
        return n, counts

    def allgatherv(self, d_index, d_spans, k, d_ids, d_m, a_idx, a_spans, a_ids, stream):
        m = int(d_m[0])
        a_idx.numpy()[:k] = d_index.numpy()[:k]
        a_spans.numpy()[:k] = d_spans.numpy()[:k]
        a_ids.numpy()[:m] = d_ids.numpy()[:m]
        sizes = np.zeros((self._world, 2), dtype=np.int64)
        sizes[0] = (k, m)
        return sizes

    def gather_result(self, stream):
        r = self._gathered
        n, m = len(r["counts"]), int(r["offsets"][-1])
        spans = np.stack([r["offsets"][:-1].astype(np.uint32), np.maximum(r["counts"], 0).astype(np.uint32)], axis=1)
        ids = np.zeros(2 * max(self._slab_ids, m), dtype=np.uint32)
        ids[:m] = r["ids"]
        return np.array([[n, m], [0, 0]], dtype=np.int64), np.arange(n, dtype=np.uint32), spans, ids

    monkeypatch.setattr(_FakeEngine, "partition_batch_device", partition)
    monkeypatch.setattr(_FakeEngine, "allgatherv_device", allgatherv)
    monkeypatch.setattr(_FakeEngine, "gather_result", gather_result)
    bench.run_own(_ns(gpus=2))
    d = json.loads(out.getvalue())
    assert d["n_gpus"] == 2 and d["value_with_gather"] > 0 and d["multi_gpu"]["collective"].startswith("gm_allgatherv_device")
    assert d["multi_gpu"]["strong"]["all_gatherv_ms_with_broadcasts"] > 0 and d["multi_gpu"]["strong"]["shard_load"]["per_shard"][1] == 0
    assert d["multi_gpu"]["strong_fused"]["ms_per_step_direct_stores"] > 0
    assert d["cpu_baseline"] is None and d["c4"] is None and "sharded by topic-root hash over 2 GPUs" in d["config"]["workload"]
    assert d["parity_check"]["topics"] == 2000 and isinstance(d["parity_check"]["ok"], bool)
