#!/usr/bin/env python
"""Benchmark of the north-star path: Router::matches for a batch of PUBLISH topics at 10 M subscriptions.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl own|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path (tokenise -> trie walk -> per-topic match lists) over one batch of
synthetic topics (workload C3 of BASELINE.json: 10 M subscriptions, 30 % '+', 5 % '#', 6-level IoT topics,
1 M-topic batch).  N > 1 is launched by torchrun, one process per GPU: the subscription set is sharded by
topic-root hash (root-wildcard filters replicated).  `value` is the weak-scaling leg (every rank matches its own
batch of topics of its shard, no collective -> "scaling": "weak"); `multi_gpu` adds the collective on the data path:
`value_with_gather` (the same plus ONE all-gatherv of all match lists, libgpumqtt's gm_allgatherv_device) and the
strong-scaling leg (one mixed batch partitioned by a device kernel, matched, gathered), and `parity_check` verifies
the gathered lists of a 60 K-topic sample against the oracle on rank 0.

Prints ONE JSON line (rank 0).  See DESIGN.md §"Measurement" for every key.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import traceback
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
_DEVICE_KIND = "cuda"          # tests/test_bench_flow.py runs the control flow of run_own against a fake engine on "cpu"


def _args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--subs", type=int, default=None, help="override subscription count (non-default => not the headline config)")
    ap.add_argument("--topics", type=int, default=None, help="override topics per batch")
    ap.add_argument("--batches", type=int, default=4, help="distinct topic batches rotated through the timed loop")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--no-c4", action="store_true", help="skip the retained-tree (config C4) leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the match lists of the last timed step (a fixed sample of its topics, rank 0) "
                         "as DIR/<name>.npy, so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "own":
        ap.error("--dump-outputs writes what the own arm's timed path computed; use it with --impl own")
    return a


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _regions_of_rank(cfg, rank: int, world: int):
    from rmqtt_b200 import workload as wl
    from rmqtt_b200.engine import shard_of
    if world == 1:
        return list(range(cfg.R))
    return [r for r in range(cfg.R) if shard_of(wl.region_name(r), world) == rank]


def _cfg(args):
    from rmqtt_b200 import workload as wl
    cfg = wl.C3
    if args.subs or args.topics:
        cfg = cfg.scaled(n_subs=args.subs, n_topics=args.topics, name="C3-scaled")
    return cfg


def _workload_desc(cfg, world):
    return (f"{cfg.name}: {cfg.n_subs} subscriptions (30% '+', 5% '#', 0.6% root '+'), 6-level IoT topics "
            f"reg/site/dev/sen/met/ch over R{cfg.R}xS{cfg.S}xD{cfg.D}xK{cfg.K}xM{cfg.M}xF{cfg.F}, "
            f"{cfg.n_topics}-topic uniform batch per GPU, seed {cfg.seed:#x}"
            + (f", subscriptions sharded by topic-root hash over {world} GPUs (root-wildcards replicated)" if world > 1 else "")
            + "; L2: the device tables (GBs) and the rotated distinct batches are far larger than the 126 MB L2, no flush between steps")


_DUMP_TOPICS = 1 << 16             # topics of the batch that --dump-outputs samples
_DUMP_BYTES = 60 << 20             # array bytes of one dump: with the .npy headers it stays under 64 MB


def _dump_outputs(out_dir, spans, ids, status):
    """--dump-outputs: one step's match lists (spans uint32[n, 2], ids uint32[], status int32[n]) in a form in which two builds
    compare equal when they match alike.  The topics are a fixed seeded sample of the batch (all of it when it is small), each
    topic's ids are sorted (the kernels leave them in any order), and everything is float64, which holds every u32 id exactly.
    Files: topics (index in the batch), status, counts (-1 for an invalid topic) and ids (concatenated in topic order)."""
    from rmqtt_b200.engine import MatchResult
    n = len(spans)
    topics = np.arange(n) if n <= _DUMP_TOPICS else np.sort(np.random.default_rng(0).choice(n, _DUMP_TOPICS, replace=False))
    counts, sorted_ids = MatchResult(spans[topics], ids, status[topics], len(ids)).canonical()
    # the longest prefix of the sample whose topic, status, count and ids fit the byte budget
    keep = int(np.searchsorted(np.cumsum(3 + np.maximum(counts, 0)), _DUMP_BYTES // 8, side="right"))
    arrays = {"topics": topics[:keep], "status": status[topics[:keep]], "counts": counts[:keep],
              "ids": sorted_ids[:int(np.maximum(counts[:keep], 0).sum())]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float64))


# ======================================================================================================
def run_reference(args):
    """The reference's own CPU implementation of the path.  rmqtt is Rust and cannot be built here (no
    cargo/rustc), so this arm times the C++ restatement of DefaultRouter::_matches (oracle/oracle.cpp) on
    all host cores against the SAME subscription set; each step matches a bounded sample of the batch."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    from rmqtt_b200 import workload as wl
    cfg = _cfg(args)
    threads = orc.hardware_threads()
    orc.numa_interleave(True)          # tree pages spread over the sockets: the 128-reader baseline must not depend on page luck
    sb, so, sv = wl.gen_subs(cfg)
    router = orc.Router()
    t0 = time.time()
    router.bulk_add(sb, so, sv, nthreads=min(threads, 64))
    build_s = time.time() - t0
    # bounded sample per step: sized so that warmup + steps stay within a few minutes on the host cores
    sample = min(cfg.n_topics, max(2_000, 25_000_000 // max(1, args.steps + args.warmup)))
    tb, to = wl.gen_topics(cfg, sample)
    tried = {}
    for k in range(max(2, args.warmup)):                 # warm-up doubles as the choice of the reader-thread count: all allowed
        t = threads if k % 2 == 0 else max(1, threads // 2)   # CPUs, or one per two (SMT siblings idle) — whichever serves the port better
        tried[t] = min(tried.get(t, float("inf")), router.match_batch(tb, to, nthreads=t)["seconds"])
    all_threads, threads = threads, min(tried, key=tried.get)
    secs, ids = 0.0, 0
    for _ in range(args.steps):
        r = router.match_batch(tb, to, nthreads=threads)
        secs += r["seconds"]
        ids = r["total_ids"]
    value = sample * args.steps / secs
    line = {
        "impl": "reference", "metric": "topic-matches/sec @10M subs", "value": value, "unit": "topics/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": _workload_desc(cfg, max(1, args.gpus))},      # the same workload definition as the own arm's line
        "details": {"sample": f"{sample} topics of the batch per step, matched against the whole (unsharded) subscription set on the host cores",
                    "oracle_build_s": round(build_s, 1), "matched_ids_per_topic": ids / sample},
        "cpu_baseline": {"value": value, "unit": "topics/s", "cores": threads, "kind": "port",
                         "sample": f"{sample}-topic sample x {args.steps} steps, C++ restatement of DefaultRouter::_matches (Rust reference not buildable here: no cargo)",
                         "allowed_cpus": all_threads, "threads_tried_topics_per_s": {str(t): sample / v for t, v in tried.items()}},
        "e2e": {"value": value, "unit": "topics/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)


# ======================================================================================================
class _Pinned:
    """Pinned host buffers from the library's NUMA-aware allocator (placed next to the engine's GPU)."""

    def __init__(self, lib, eng):
        self.lib, self.eng, self.ptrs = lib, eng, []

    def alloc(self, nbytes, dtype, shape):
        p = self.lib.gm_host_alloc_near(self.eng._h, max(1, int(nbytes)))
        assert p, "gm_host_alloc_near failed"
        self.ptrs.append(p)
        return p, np.frombuffer((C.c_uint8 * max(1, int(nbytes))).from_address(p), dtype=dtype)[:int(np.prod(shape))].reshape(shape)

    def free(self):
        for p in self.ptrs:
            self.lib.gm_host_free(p)
        self.ptrs = []


def _c4_leg(torch, dev, stream, peak, small: bool):
    """BASELINE.json config C4 (retained tree: 5 M retained topics, 100 K wildcard SUBSCRIBE filters) on this GPU:
    device-resident filters, CUDA-event kernel times from the engine's ring, algorithmic bytes from the oracle's counters
    of the same batch (SURVEY §8(d), retained form), count parity against the oracle."""
    from oracle import oracle as orc
    from rmqtt_b200 import workload as wl
    from rmqtt_b200.engine import Engine
    cfg = wl.C4.scaled(n_subs=500_000, n_topics=20_000, name="C4-scaled") if small else wl.C4
    rb, ro, rv = wl.gen_retained(cfg)
    fb, fo = wl.gen_retain_filters(cfg)
    n = len(fo) - 1
    eng = Engine()
    t0 = time.time()
    eng.retain_bulk_load(rb, ro, rv)
    eng.flush()
    build_s = time.time() - t0
    d_blob, d_offs = torch.from_numpy(fb).to(dev), torch.from_numpy(fo.view(np.int32)).to(dev)
    d_spans = torch.zeros((n, 2), dtype=torch.int32, device=dev)
    d_status = torch.zeros(n, dtype=torch.int32, device=dev)
    d_ids = torch.empty(1 << 22, dtype=torch.int32, device=dev)
    need = C.c_uint64(0)
    from rmqtt_b200 import _native as N
    rc = N.lib().gm_retain_match_batch_device(eng._h, d_blob.data_ptr(), d_blob.numel(), d_offs.data_ptr(), n, d_spans.data_ptr(), d_ids.data_ptr(), d_ids.numel(),
                                              C.byref(need), d_status.data_ptr(), stream)
    if rc == N.GM_ERR_CAPACITY:
        d_ids = torch.empty(int(need.value) + 1024, dtype=torch.int32, device=dev)
    reps = 10
    for _ in range(reps + 3):
        hits = eng.retain_match_batch_device(d_blob, d_offs, d_spans, d_ids, d_status, stream)
    torch.cuda.synchronize()
    k = eng.kernel_ms(reps).mean(axis=0)
    tree = orc.RetainTree()
    tree.bulk_insert(rb, ro, rv)
    o = tree.match_batch(fb, fo, nthreads=orc.hardware_threads(), want_ids=False)
    counts = d_spans.cpu().numpy()[:, 1].astype(np.int64)
    c = o["counters"]
    walk_bytes = 32 * c["V"] + 16 * c["E"] + 4 * c["M"] + 8 * n
    ms = float(k.sum())
    eng.close()
    return {"workload": f"{cfg.name}: {cfg.n_subs} retained topics, {n} wildcard SUBSCRIBE filters (85% '+', 15% '#'), seed {cfg.seed:#x}",
            "filters_per_s": n / (ms * 1e-3), "ms": ms, "kernel_ms": {"tokenize": float(k[0]), "walk": float(k[1]), "publish": float(k[2])},
            "hits_per_filter": hits / n, "visited_nodes_per_filter": c["V"] / n,
            "algorithmic_bytes": walk_bytes, "achieved_GBps": walk_bytes / (float(k[1] + k[2]) * 1e-3) / 1e9,
            "frac": walk_bytes / (float(k[1] + k[2]) * 1e-3) / 1e9 / peak,
            "cpu_filters_per_s": n / o["seconds"], "cpu_threads": orc.hardware_threads(),
            "count_parity": bool((counts == o["counts"]).all()), "build_s": round(build_s, 1)}


def _relations_leg(small: bool):
    """Router::matches END TO END at the router level (config C2: 1 M subscriptions, 100 K-topic batch): engine match +
    device-side relation expansion (k_relations: no_local, v5 per-client de-dup) + host assembly of gm_sub_relation records."""
    from rmqtt_b200 import workload as wl
    from rmqtt_b200 import _native as N
    from rmqtt_b200.router import GpuRouter
    cfg = wl.C2.scaled(n_subs=100_000, n_topics=20_000, name="C2-scaled") if small else wl.C2
    sb, so, sv = wl.gen_subs(cfg)
    tb, to = wl.gen_topics(cfg)
    n = cfg.n_topics
    r = GpuRouter()
    lib = N.lib()
    rng = np.random.default_rng(7)
    nodes = rng.integers(1, 4, size=len(sv)).astype(np.uint64)
    clients = (sv // 2).astype(np.uint32)                      # every client holds two subscriptions: de-dup has work to do
    flags = (rng.random(len(sv)) < 0.5).astype(np.uint8)       # half of the clients speak v5
    flags = flags[clients % len(flags)] | ((rng.random(len(sv)) < 0.1).astype(np.uint8) << 1)
    sub_ids = np.where(flags & 1, 1 + (sv % 7), 0).astype(np.uint32)
    added = C.c_uint64(0)
    t0 = time.time()
    rc = lib.gmr_add_batch_numbered(r._h, sb.ctypes.data, so.ctypes.data, len(sv), nodes.ctypes.data, clients.ctypes.data, flags.ctypes.data, sub_ids.ctypes.data, C.byref(added))
    assert rc == 0
    build_s = time.time() - t0
    spans = np.zeros((n, 2), dtype=np.uint32)
    status = np.zeros(n, dtype=np.int32)
    cap_r, cap_s = 64 * n, 16 * n
    rels = (N.GmSubRelation * cap_r)()
    sids = np.zeros(cap_s, dtype=np.uint32)
    nr, ns = C.c_uint64(0), C.c_uint64(0)
    dev_ms, host_ms, wall = [], [], []
    for k in range(6):
        t0 = time.perf_counter()
        rc = lib.gmr_matches_batch(r._h, None, tb.ctypes.data, to.ctypes.data, n, spans.ctypes.data, rels, cap_r, sids.ctypes.data, cap_s, C.byref(nr), C.byref(ns), status.ctypes.data)
        assert rc == 0, rc
        wall.append((time.perf_counter() - t0) * 1e3)
        d, h = C.c_double(0), C.c_double(0)
        lib.gmr_last_timing(r._h, C.byref(d), C.byref(h))
        dev_ms.append(d.value); host_ms.append(h.value)
    return {"workload": f"{cfg.name}: {int(added.value)} subscriptions (every client subscribes twice, half of them v5, 10% no_local), {n}-topic batch, host buffers",
            "relations_per_batch": int(nr.value), "sub_ids_per_batch": int(ns.value),
            "device_ms": float(np.median(dev_ms[1:])), "host_assembly_ms": float(np.median(host_ms[1:])), "call_ms": float(np.median(wall[1:])),
            "topics_per_s": n / (float(np.median(wall[1:])) * 1e-3), "relations_per_s": int(nr.value) / (float(np.median(wall[1:])) * 1e-3),
            "device_part": "H2D topics, k_tokenize..k_match_fast, k_relations (no_local, v5 per-client de-dup, sub-id accumulation), D2H handles",
            "host_part": "handle -> gm_sub_relation{node_id, handle, group, sub ids}: table look-ups only", "router_build_s": round(build_s, 1)}


def _configs_leg(torch, eng, cfg, dev, stream, timed_device_loop, d_spans, d_ids, d_needed, d_status, small: bool):
    """The other single-GPU rows of BASELINE.json in the same run: C1 and C2 through tools/bench_configs.py (own engines; kernel
    times from the engine's ring, the CPU port on 1 and all threads beside them, count parity of every topic), and the secondary
    publish distribution of SURVEY §8(d) — Zipf(1.0) over devices — as one more batch on the C3 engine."""
    from rmqtt_b200 import workload as wl
    sys.path.insert(0, str(ROOT / "tools"))
    import bench_configs as bc
    bc.dev, bc.stream = dev, stream          # the tool's module-level device / stream: this process's
    out = {}
    for name in ("C1", "C2"):
        c = wl.CONFIGS[name]
        if small and name == "C2":
            c = c.scaled(n_subs=100_000, n_topics=20_000, name="C2-scaled")
        out[name] = bc.publish_config(c, reps=20)
    zb, zo = wl.gen_topics_zipf(cfg)
    n = len(zo) - 1
    d_zb, d_zo = torch.from_numpy(zb).to(dev), torch.from_numpy(zo.view(np.int32)).to(dev)
    ids = d_ids
    eng.match_batch_device(d_zb, d_zo, d_spans, ids, d_needed, d_status, stream)
    need = int(d_needed.item())
    if need > ids.numel():
        ids = torch.empty(need + 1024, dtype=torch.int32, device=dev)
    steps = 20
    ms_z = timed_device_loop(lambda k: eng.match_batch_device(d_zb, d_zo, d_spans, ids, d_needed, d_status, stream), steps, 3)
    kz = eng.kernel_ms(steps).mean(axis=0)
    out["C3-zipf"] = {"workload": f"{cfg.name} subscriptions, {n}-topic batch drawn Zipf(1.0) over devices (SURVEY 8d, secondary distribution)",
                      "topics_per_s": n * steps / (ms_z / 1e3), "ms_per_step": ms_z / steps, "ids_per_topic": need / n,
                      "kernel_ms": {"k_tokenize+k_bucket_scan+k_bucket_scatter": float(kz[0]), "k_match_fast": float(kz[1]), "k_match_slow": float(kz[2])}}
    return out


def run_own(args):
    import torch
    import torch.distributed as dist
    from rmqtt_b200 import workload as wl
    from rmqtt_b200 import _native as N
    from rmqtt_b200.engine import Engine, MatchResult

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    lib = N.lib()
    if world > 1:
        lib.gm_bind_thread_near_device(local)      # one process per GPU: its host threads and buffers live next to its GPU (2-socket hosts)
        os.environ.setdefault("GM_HOST_THREADS", str(max(1, min(64, (os.cpu_count() or 1) // world))))   # the bulk build of every rank runs at the same time
    torch.cuda.set_device(local)
    dev = torch.device(_DEVICE_KIND, local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = _cfg(args)
    regions = _regions_of_rank(cfg, rank, world)
    small = cfg.n_subs < 5_000_000                 # developer runs with --subs/--topics: shrink the secondary legs too

    # ---- build the device-resident trie for this rank's shard -------------------------------------
    t0 = time.time()
    if world == 1:
        sb, so, sv = wl.gen_subs(cfg)
    else:
        sb, so, sv = wl.gen_subs_sharded(cfg, regions)
    t1 = time.time()
    eng = Engine(device=local, filters_hint=len(sv))
    t2 = time.time()
    eng.bulk_load(sb, so, sv)
    t3 = time.time()
    eng.flush()
    build_s = time.time() - t0
    # gm_bulk_load + the first gm_flush are the library's build (all host threads, host_trie.cpp insert_batch_parallel); the
    # generator of the synthetic filters is single-threaded and not part of it
    build_parts = {"generate_filters_s": round(t1 - t0, 2), "create_and_reserve_s": round(t2 - t1, 2), "bulk_load_s": round(t3 - t2, 2),
                   "flush_s": round(time.time() - t3, 2), "host_threads": int(os.environ.get("GM_HOST_THREADS", min(64, os.cpu_count() or 1)))}
    st = eng.stats()
    del sb, so
    uid = [Engine.comm_unique_id() if rank == 0 else None]
    if world > 1:
        dist.broadcast_object_list(uid, src=0)
    eng.comm_init(uid[0], rank, world)             # the library's own NCCL communicator (gm_allgatherv_device)

    # ---- topic batches, resident in HBM before the timed region ---------------------------------
    n = cfg.n_topics
    B = max(1, args.batches)
    host_batches = [wl.gen_topics(cfg, n, regions=regions if world > 1 else None, stream=rank * 1000 + b) for b in range(B)]
    d_batches = [(torch.from_numpy(tb).to(dev), torch.from_numpy(to.view(np.int32)).to(dev)) for tb, to in host_batches]
    d_spans = torch.zeros((n, 2), dtype=torch.int32, device=dev)
    d_status = torch.zeros(n, dtype=torch.int32, device=dev)
    d_needed = torch.zeros(1, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    cap = 64 * n
    d_ids = torch.empty(cap, dtype=torch.int32, device=dev)
    needed_max, works = 0, []
    for tb, to in d_batches:   # untimed instrumented pass: exact work counters + output sizing
        while True:
            w = eng.match_batch_device(tb, to, d_spans, d_ids, d_needed, d_status, stream, work=True)
            need = int(d_needed.item())
            if need <= d_ids.numel():
                break
            d_ids = torch.empty(int(need * 1.1) + 1024, dtype=torch.int32, device=dev)
        works.append(w)
        needed_max = max(needed_max, need)
    if d_ids.numel() > 2 * needed_max + 1024:
        d_ids = torch.empty(int(needed_max * 1.25) + 1024, dtype=torch.int32, device=dev)
    desc_max = int(max(w["filters"] for w in works))

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_device_loop(step, steps, warm):
        for k in range(warm):
            step(k)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(steps):
            step(k)
        e1.record()
        sync_all()
        return max_over_ranks(e0.elapsed_time(e1))

    # ---- leg 1 (headline `value`): ids mode, inputs resident in HBM ------------------------------------------------
    def step(k):
        tb, to = d_batches[k % B]
        eng.match_batch_device(tb, to, d_spans, d_ids, d_needed, d_status, stream)

    for k in range(max(3, args.warmup)):
        step(k)
    sync_all()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.2)
    launches0 = eng.kernel_launches()
    ms = timed_device_loop(step, args.steps, 0)
    launches = eng.kernel_launches() - launches0
    kms = eng.kernel_ms(min(64, args.steps))
    clocks = sampler.stop() if sampler else None
    value = world * n * args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:            # the buffers still hold the last timed step's lists (batch (steps - 1) % B)
        m = int(d_needed.item())
        assert m <= d_ids.numel(), "the last timed step's ids did not fit the output buffer"
        _dump_outputs(args.dump_outputs, d_spans.cpu().numpy().view(np.uint32), d_ids[:m].cpu().numpy().view(np.uint32), d_status.cpu().numpy())

    # the same loop in descriptor mode (8 B per matched filter instead of 4 B per matched id): explains the e2e number
    d_desc = torch.empty((int(desc_max * 1.25) + 1024, 2), dtype=torch.int32, device=dev)

    def step_desc(k):
        tb, to = d_batches[k % B]
        eng.match_batch_device_ex(tb, to, d_spans, d_desc, d_needed, d_status, stream, desc=True)

    side_steps = max(5, min(args.steps, 50))
    ms_desc = timed_device_loop(step_desc, side_steps, 3)
    kms_desc = eng.kernel_ms(min(64, side_steps))
    value_desc = world * n * side_steps / (ms_desc / 1e3)

    # ---- leg 2 (e2e): through the C ABI with pinned HOST buffers: H2D + kernels + D2H inside the timed region, batches rotated
    pin = _Pinned(lib, eng)
    p_in = []
    for hb, ho in host_batches:
        pb, ab = pin.alloc(len(hb), np.uint8, (len(hb),))
        po, ao = pin.alloc(4 * (n + 1), np.uint32, (n + 1,))
        ab[:] = hb
        ao[:] = ho
        p_in.append((pb, po, len(hb)))
    ids_cap = int(needed_max * 1.25) + 1024
    desc_cap = int(desc_max * 1.25) + 1024
    p_spans, _ = pin.alloc(8 * n, np.uint32, (n, 2))
    p_status, _ = pin.alloc(4 * n, np.int32, (n,))
    p_ids, _ = pin.alloc(4 * ids_cap, np.uint32, (ids_cap,))
    p_desc, _ = pin.alloc(8 * desc_cap, np.uint32, (desc_cap, 2))
    e2e_steps = args.e2e_steps or max(3, min(args.steps, 10))
    need = C.c_uint64(0)

    def e2e_ids(k):
        pb, po, _ = p_in[k % B]
        rc = lib.gm_match_batch(eng._h, pb, po, n, p_spans, p_ids, ids_cap, C.byref(need), p_status)
        assert rc == 0, lib.gm_last_error(eng._h)

    def e2e_desc(k):
        pb, po, _ = p_in[k % B]
        rc = lib.gm_match_batch_desc(eng._h, pb, po, n, p_spans, p_desc, desc_cap, C.byref(need), p_status)
        assert rc == 0, lib.gm_last_error(eng._h)

    def timed_host_loop(fn, steps):
        for k in range(2):
            fn(k)
        sync_all()
        t0 = time.perf_counter()
        for k in range(steps):
            fn(k)
        torch.cuda.synchronize()
        return max_over_ranks(time.perf_counter() - t0)

    s_ids = timed_host_loop(e2e_ids, e2e_steps)
    need_ids = int(need.value)
    s_desc = timed_host_loop(e2e_desc, e2e_steps)
    need_desc = int(need.value)

    # the same descriptor-mode call issued by SEVERAL caller threads (the reference's Router::matches is called from many
    # tokio workers at once; the engine keeps three batches in flight): the D2H tail of one call overlaps the H2D head of
    # the next.  Every thread has its own output buffers; every call still moves its whole batch in and its result out.
    # Measured with 2 and with 3 callers (= the engine's three match contexts); the better one is `e2e.value`, both are reported.
    def run_with_callers(T):
        outs = []
        for _ in range(T):
            ps, _a = pin.alloc(8 * n, np.uint32, (n, 2))
            pt, _b = pin.alloc(4 * n, np.int32, (n,))
            pd, _c = pin.alloc(8 * desc_cap, np.uint32, (desc_cap, 2))
            outs.append((ps, pt, pd))
        steps_t = max(2, e2e_steps // T) * T
        errs = []

        def caller(tid, count):
            nd = C.c_uint64(0)
            ps, pt, pd = outs[tid]
            for k in range(count):
                pb, po, _ = p_in[(tid + T * k) % B]
                rc = lib.gm_match_batch_desc(eng._h, pb, po, n, ps, pd, desc_cap, C.byref(nd), pt)
                if rc != 0:
                    errs.append(rc)

        def run_callers(count):
            ths = [threading.Thread(target=caller, args=(t, count)) for t in range(T)]
            for t in ths:
                t.start()
            for t in ths:
                t.join()

        run_callers(1)
        sync_all()
        t0 = time.perf_counter()
        run_callers(steps_t // T)
        torch.cuda.synchronize()
        secs = max_over_ranks(time.perf_counter() - t0)
        assert not errs, errs
        return steps_t, secs

    by_callers = {T: run_with_callers(T) for T in (2, 3)}
    rate = {T: world * n * st_ / sec_ for T, (st_, sec_) in by_callers.items()}      # identical on every rank (max over ranks inside)
    T2 = max(rate, key=rate.get)
    steps2, s_desc2 = by_callers[T2]
    h2d = int(np.mean([x[2] for x in p_in]) + 4 * (n + 1))
    e2e = {"value": world * n * steps2 / s_desc2, "unit": "topics/s", "mode": "descriptors (gm_match_batch_desc: per topic the matched value sets by reference, "
           "8 B per matched filter; the host reads members from its mirror through gm_values_view); several caller threads per GPU "
           "(the better of 2 and 3, see caller_threads / by_caller_threads), each call moves its whole batch in and its result out",
           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(8 + 4 * n + 8 * n + 8 * need_desc), "steps": steps2, "caller_threads": T2,
           "by_caller_threads": {str(T): v for T, v in rate.items()},
           "single_caller": {"value": world * n * e2e_steps / s_desc, "unit": "topics/s", "steps": e2e_steps},
           "ids_mode": {"value": world * n * e2e_steps / s_ids, "unit": "topics/s", "entry": "gm_match_batch (every matched id materialised in host memory)",
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(8 + 4 * n + 8 * n + 4 * need_ids)},
           "buffers": f"pinned, NUMA node {lib.gm_device_numa_node(local)} (gm_host_alloc_near), {B} batches rotated"}

    # ---- roofline of the dominant kernel (k_match_fast) -------------------------------------------
    peak, peak_src = _peaks()
    W = {k: sum(w[k] for w in works) / len(works) for k in works[0] if not isinstance(works[0][k], list)}   # mean per launch over the rotated batches
    diag = {"probes_by_depth": works[0]["probes_by_depth"], "misses_by_depth": works[0]["misses_by_depth"], "slot_loads": works[0]["slot_loads"]}
    k2_bytes = 16 * W["visited"] + 16 * W["probed"] + 8 * W["filters"] + 4 * W["ids"] + 8 * n     # SURVEY §8(d), walk terms
    k1_bytes = W["bytes"] + 8 * n + 16 * W["levels"]                                              # SURVEY §8(d), tokeniser terms
    k_mean = kms.mean(axis=0) if len(kms) else np.zeros(3)
    k2_ms = float(k_mean[1])
    achieved = k2_bytes / (k2_ms * 1e-3) / 1e9 if k2_ms > 0 else None
    traffic, traffic_src = None, "not measured in this run (ncu cannot run inside the timed bench)"
    prof = ROOT / "profiles" / "k_match_fast_traffic.json"      # written next to the committed ncu report it was read from
    traffic_same_build = None
    if prof.exists():
        try:
            pj = json.loads(prof.read_text())
            traffic, traffic_src = pj.get("dram_bytes_per_launch"), pj.get("source")
            if rank == 0 and pj.get("library_sass_md5"):        # is the library that just ran the one that was profiled?  (machine code, not timestamps)
                import hashlib
                sass = subprocess.run(["cuobjdump", "-sass", str(ROOT / "rmqtt_b200" / "libgpumqtt.so")], capture_output=True, timeout=120).stdout
                traffic_same_build = bool(sass) and hashlib.md5(sass).hexdigest() == pj["library_sass_md5"]
        except Exception:
            pass
    kd = kms_desc.mean(axis=0) if len(kms_desc) else np.zeros(3)
    roofline = {"bound": "hbm", "kernel": "k_match_fast", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_src, "traffic_same_machine_code": traffic_same_build, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": k2_bytes, "kernel_ms": {"k_tokenize+k_bucket_scan+k_bucket_scatter": float(k_mean[0]), "k_match_fast": k2_ms, "k_match_slow": float(k_mean[2])},
                "pipeline": {"algorithmic_bytes_per_step": k1_bytes + k2_bytes,
                             "achieved": (k1_bytes + k2_bytes) / (float(k_mean.sum()) * 1e-3) / 1e9 if k_mean.sum() > 0 else None,
                             "frac_of_step": (k1_bytes + k2_bytes) / (ms / args.steps * 1e-3) / 1e9 / peak},
                "descriptor_mode_kernel_ms": {"k_tokenize+k_bucket_scan+k_bucket_scatter": float(kd[0]), "k_match_fast": float(kd[1]), "k_match_slow": float(kd[2])}}
    # the same kernel in descriptor mode (the mode the e2e path runs): the publish phase writes one 8-byte value-set reference per
    # matched filter instead of 4 bytes per matched id, everything else is the same walk
    k2_bytes_desc = 16 * W["visited"] + 16 * W["probed"] + 8 * W["filters"] + 8 * W["filters"] + 8 * n
    if kd[1] > 0:
        ach_d = k2_bytes_desc / (float(kd[1]) * 1e-3) / 1e9
        roofline["descriptor_mode"] = {"kernel": "k_match_fast<DESC>", "algorithmic_bytes_per_launch": k2_bytes_desc, "achieved": ach_d, "unit": "GB/s",
                                       "frac": ach_d / peak}

    # ---- the headline is complete here: keep it where the watchdog / exception path finds it (rank 0) -------------------
    if rank == 0:
        _PARTIAL.update({
            "metric": "topic-matches/sec @10M subs", "value": value, "unit": "topics/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": _workload_desc(cfg, world)},
            "details": {"l2": f"device tables {st['device_bytes'] / 1e9:.2f} GB >> 126 MB L2; {B} distinct topic batches rotated",
                        "matched_ids_per_topic": W["ids"] / n, "matched_filters_per_topic": W["filters"] / n, "visited_nodes_per_topic": W["visited"] / n,
                        "deferred_topics_per_batch": W["deferred"], "probe_diag": diag,
                        "trie": {k: st[k] for k in ("values", "nodes", "edges", "edge_slots", "dict_entries", "plus_nodes", "device_bytes", "max_depth")},
                        "build_s": round(build_s, 1), "build": build_parts, "e2e_timing": "perf_counter around synchronous C-ABI calls (pinned host buffers), max over ranks"},
            "value_descriptor_mode": value_desc,
            "e2e": e2e,
            "gpu_launches": int(launches),
            "roofline": roofline,
            "cpu_baseline": None, "multi_gpu": None, "parity_check": None, "c4": None, "latency": None, "churn": None, "relations": None, "configs": None,
            "clocks": clocks,
        })

    # ---- leg 3 (C5): the collective on the data path ---------------------------------------------------------------
    # (a) weak + gather: every rank matches its own batch, then ONE all-gatherv makes every rank hold all world*n lists
    # (b) strong: ONE mixed batch (identical on every rank, uniform over all roots) is partitioned by a device kernel,
    #     every rank matches its share, the all-gatherv completes the batch on every rank
    multi = None
    parity = None
    coll_steps = max(3, min(args.steps, 20))
    mb, mo = wl.gen_topics(cfg, n, stream=424242)                         # the mixed batch: same bytes on every rank
    d_mb, d_mo = torch.from_numpy(mb).to(dev), torch.from_numpy(mo.view(np.int32)).to(dev)
    d_sel = torch.zeros(n, dtype=torch.int32, device=dev)
    a_cap_t = world * n if world > 1 else n
    a_idx = torch.empty(a_cap_t, dtype=torch.int32, device=dev)
    a_spans = torch.empty((a_cap_t, 2), dtype=torch.int32, device=dev)
    a_ids = torch.empty(int(needed_max * 1.3) * world + 4096, dtype=torch.int32, device=dev)
    d_own_index = torch.arange(rank * n, (rank + 1) * n, dtype=torch.int32, device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    phase = np.zeros(3)
    shard_counts = None

    def strong_step(k, record=False):
        nonlocal shard_counts
        if record:
            ev[0].record()
        kk, shard_counts = eng.partition_batch_device(d_mb, d_mo, world, rank, d_sel, stream)
        if record:
            ev[1].record()
        eng.match_batch_device_ex(d_mb, d_mo, d_spans, d_ids, d_needed, d_status, stream, d_sel=d_sel, n_sel=kk)
        if record:
            ev[2].record()
        sizes = eng.allgatherv_device(d_sel, d_spans, kk, d_ids, d_needed, a_idx, a_spans, a_ids, stream)
        if record:
            ev[3].record()
            torch.cuda.synchronize()
            for j in range(3):
                phase[j] += ev[j].elapsed_time(ev[j + 1])
        return sizes

    def weak_gather_step(k):
        tb, to = d_batches[k % B]
        eng.match_batch_device(tb, to, d_spans, d_ids, d_needed, d_status, stream)
        eng.allgatherv_device(d_own_index, d_spans, n, d_ids, d_needed, a_idx, a_spans, a_ids, stream)

    ms_strong = timed_device_loop(strong_step, coll_steps, 3)
    for k in range(coll_steps):
        strong_step(k, record=True)
    ph = [max_over_ranks(float(x)) / coll_steps for x in phase]
    sizes = strong_step(0)
    torch.cuda.synchronize()
    multi = {"strong": {"workload": f"one mixed {n}-topic batch (uniform over all roots, identical on every rank) partitioned on the device by root hash",
                        "value": n * coll_steps / (ms_strong / 1e3), "unit": "topics/s", "ms_per_step": ms_strong / coll_steps, "steps": coll_steps,
                        "phase_ms_max_over_ranks": {"partition": ph[0], "match": ph[1], "all_gatherv": ph[2]},
                        "limiter": ["partition", "match", "all_gatherv"][int(np.argmax(ph))],
                        "shard_load": {"max": int(shard_counts.max()), "mean": float(shard_counts.mean()), "per_shard": [int(x) for x in shard_counts]},
                        "gathered_ids_per_step": int(sizes[:, 1].sum())}}
    if world > 1:
        ms_wg = timed_device_loop(weak_gather_step, coll_steps, 3)
        multi["value_with_gather"] = world * n * coll_steps / (ms_wg / 1e3)
        multi["weak_gather_ms_per_step"] = ms_wg / coll_steps
        multi["collective"] = "gm_allgatherv_device: ncclAllGather of (topics, ids) per rank + one grouped launch of ncclSend/ncclRecv pairs out of the match kernels' buffers"
        # A/B of the data movement inside the collective: per-rank ncclBroadcasts instead of point-to-point pairs
        eng.debug_knob("gather_bcast", 1)
        phase[:] = 0
        for k in range(coll_steps):
            strong_step(k, record=True)
        multi["strong"]["all_gatherv_ms_with_broadcasts"] = max_over_ranks(float(phase[2])) / coll_steps
        eng.debug_knob("gather_bcast", 0)

    # ---- (c) the same strong-scaling step with the exchange FUSED into the match kernels over peer memory (CUDA IPC) ----
    fused_res = None
    try:
        slab_ids = int(needed_max * 1.3) + 4096
        if world > 1:                                         # the block layout must be identical on every rank
            t_sl = torch.tensor([slab_ids], dtype=torch.int64, device=dev)
            dist.all_reduce(t_sl, op=dist.ReduceOp.MAX)
            slab_ids = int(t_sl.item())
        hnd = eng.gather_create(world, rank, n, slab_ids)
        hs = [hnd]
        if world > 1:
            hs = [None] * world
            dist.all_gather_object(hs, hnd)
        eng.gather_connect(hs)
        fused_ok = True
    except Exception as ex:                                   # no peer-to-peer access between the GPUs: NCCL path only
        fused_ok = False
        multi["strong_fused"] = {"unavailable": str(ex)[:200]}
    if world > 1:                                             # every rank must take the same branch
        t_ok = torch.tensor([1 if fused_ok else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(t_ok, op=dist.ReduceOp.MIN)
        fused_ok = bool(int(t_ok.item()))
    if fused_ok:
        try:
            def fused_step(k):
                kk, _ = eng.partition_batch_device(d_mb, d_mo, world, rank, d_sel, stream)
                eng.match_gather_device(d_mb, d_mo, d_status, stream, d_sel=d_sel, n_sel=kk)

            def read_back():                                      # rank 0's gathered block; a barrier a rank missed is reported, the timings stand
                try:
                    return eng.gather_result(stream) if rank == 0 else None
                except Exception as ex:                           # noqa: BLE001
                    gather_get_errors.append(f"{type(ex).__name__}: {ex}"[:200])
                    return None

            gather_get_errors = []
            ms_fused = timed_device_loop(fused_step, coll_steps, 3)
            fused_step(0)
            sync_all()
            fused_res = read_back()
            ms_direct = None
            if world > 1:                                         # A/B: the publish phase storing into every rank's block itself
                eng.debug_knob("gather_direct", 1)
                ms_direct = timed_device_loop(fused_step, coll_steps, 2)
                eng.debug_knob("gather_direct", 0)
                fused_step(0)
                sync_all()
                fused_res = read_back()
            multi["strong_fused"] = {"how": "gm_match_gather_device over peer memory (CUDA IPC): the match kernels publish this rank's rows into its own block, "
                                            "k_gather_push copies the slab into every peer's block with 16-byte stores over NVLink, a one-warp kernel writes the counts "
                                            "and runs a flag barrier; no NCCL call, no host synchronisation",
                                     "ms_per_step_direct_stores": (ms_direct / coll_steps) if ms_direct else None,
                                     "value": n * coll_steps / (ms_fused / 1e3), "unit": "topics/s", "ms_per_step": ms_fused / coll_steps, "steps": coll_steps,
                                     "vs_nccl_step": (ms_strong / coll_steps) / (ms_fused / coll_steps)}
            if gather_get_errors:
                multi["strong_fused"]["gather_get_errors"] = gather_get_errors
            sync_all()
        except Exception as ex:                               # noqa: BLE001 - e.g. GM_ERR_COMM from the flag barrier: reported, the NCCL numbers stand
            traceback.print_exc(file=sys.stderr)
            fused_res = None
            multi["strong_fused"] = {"error": f"{type(ex).__name__}: {ex}"[:300]}

    # ---- parity self-check of the sharded path: gathered lists of a >= 50 K-topic sample against the oracle (rank 0) ----
    sizes = strong_step(0)
    torch.cuda.synchronize()
    if rank == 0:
        from oracle import oracle as orc
        orc.numa_interleave(True)
        m_tot = int(sizes[:, 1].sum())
        k_tot = int(sizes[:, 0].sum())
        idx = a_idx[:k_tot].cpu().numpy()
        sp = a_spans[:k_tot].cpu().numpy().view(np.uint32)
        gi = a_ids[:m_tot].cpu().numpy().view(np.uint32)
        ok = k_tot == n and (np.sort(idx) == np.arange(n)).all()
        sample = min(n, 60_000)
        fsb, fso, fsv = wl.gen_subs(cfg)
        tree = orc.TopicTree()
        tree.bulk_insert(fsb, fso, fsv, nthreads=min(orc.hardware_threads(), 64))
        del fsb, fso
        want = tree.match_batch(mb[:int(mo[sample])], mo[:sample + 1], nthreads=orc.hardware_threads(), want_ids=True)
        del tree
        if ok:
            order = np.argsort(idx)[:sample]                      # rows of topics 0 .. sample-1
            res = MatchResult(sp[order], gi, np.zeros(sample, np.int32), m_tot)
            cg, ig = res.canonical()
            seg = np.repeat(np.arange(sample, dtype=np.int64), np.maximum(want["counts"], 0))
            iw = want["ids"][np.lexsort((want["ids"], seg))]
            ok = bool((cg == want["counts"]).all() and len(ig) == len(iw) and (ig == iw).all())
        parity = {"topics": sample, "ok": bool(ok), "path": f"gm_partition_batch_device -> gm_match_batch_device_ex -> gm_allgatherv_device over {world} rank(s), "
                  "sorted id multiset of every sampled topic vs the oracle's TopicTree::matches"}
        if fused_res is not None:                             # the fused (peer-memory) gather must deliver the same lists
            fcounts, fidx, fspans, fids = fused_res
            fok = int(fcounts[:, 0].sum()) == n and (np.sort(fidx) == np.arange(n)).all()
            if fok:
                fo = np.argsort(fidx)[:sample]
                cg2, ig2 = MatchResult(fspans[fo], fids, np.zeros(sample, np.int32), int(fcounts[:, 1].sum())).canonical()
                fok = bool((cg2 == want["counts"]).all() and len(ig2) == len(iw) and (ig2 == iw).all())
            parity["fused_ok"] = bool(fok)
    sync_all()
    pin.free()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- single-rank legs: each one isolated (an exception lands under `errors`, the other legs and the headline stand) ----
    _PARTIAL["multi_gpu"], _PARTIAL["parity_check"] = multi, parity
    errors: dict = {}
    if world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as orc
        threads = orc.hardware_threads()
        orc.numa_interleave(True)
        sb, so, sv2 = wl.gen_subs(cfg)
        nch = min(200_000, len(sv2))
        port: dict = {}

        def cpu_leg():
            """CPU baseline: the oracle's DefaultRouter::_matches restatement on the host cores"""
            router = orc.Router()
            router.bulk_add(sb, so, sv2, nthreads=min(threads, 64))
            port["router"] = router
            sample = min(n, 250_000)
            stb, sto = wl.gen_topics(cfg, sample)
            tried = {}
            for k in range(4):                               # warm-up + choice of the reader-thread count (all allowed CPUs, or one per two)
                t = threads if k % 2 == 0 else max(1, threads // 2)
                tried[t] = min(tried.get(t, float("inf")), router.match_batch(stb, sto, nthreads=t)["seconds"])
            use = min(tried, key=tried.get)
            runs = []
            secs = 0.0
            while secs < 4.0 and len(runs) < 50:
                r = router.match_batch(stb, sto, nthreads=use)["seconds"]
                runs.append(sample / r)
                secs += r
            one_n = min(20000, sample)
            one = router.match_batch(stb[:int(sto[one_n])], sto[:one_n + 1], nthreads=1)
            return {"value": sample * len(runs) / secs, "unit": "topics/s", "cores": use, "kind": "port", "allowed_cpus": threads,
                    "threads_tried_topics_per_s": {str(t): sample / v for t, v in tried.items()},
                    "sample": f"{sample}-topic sample x {len(runs)} reps of the same workload; C++ restatement of DefaultRouter::_matches "
                              f"(oracle/oracle.cpp; the Rust reference cannot be built here: no cargo); reader threads pinned one per allowed CPU, "
                              f"tree pages interleaved over NUMA nodes, work handed out in chunks",
                    "best_rep": max(runs), "worst_rep": min(runs), "single_thread_value": one_n / one["seconds"]}

        def churn_leg():
            """subscribe / unsubscribe load from a second thread while this thread keeps matching (device buffers)"""
            router = port.pop("router", None)
            # the port's write-lock path: Router::remove + Router::add of existing subscriptions, one thread
            port_churn_ops = (2 * nch / router.churn(sb, so, sv2[:nch])) if router is not None else None
            del router
            churn = {"filters_cycled": nch, "port_single_thread_ops_per_s": port_churn_ops, "legs": [],
                     "how": "gm_churn_probe in its own thread: remove + re-add of existing subscriptions at the target rate, gm_flush every 1 ms "
                            "(asynchronous: patches are scattered on a side stream between match kernels; a re-hash goes to a second table + pointer swap); "
                            "the bench thread runs the device-resident match loop meanwhile (auto-flush engine)"}
            ch_steps = 1200
            for label, rate in (("no churn", None), ("1%/s", 0.01 * cfg.n_subs), ("10%/s", 0.10 * cfg.n_subs), ("unthrottled", 0.0)):
                out = N.GmChurn()
                rcbox = []
                th = None
                if rate is not None:
                    th = threading.Thread(target=lambda: rcbox.append(lib.gm_churn_probe(eng._h, sb.ctypes.data, so.ctypes.data, sv2.ctypes.data, nch, float(rate), 1500, 1000, C.byref(out))))
                    th.start()
                    time.sleep(0.15)
                try:
                    ms_c = timed_device_loop(step, ch_steps, 3)
                finally:
                    if th:
                        th.join()
                if th:
                    assert rcbox == [0], lib.gm_last_error(eng._h)
                d = out.as_dict()
                churn["legs"].append({"churn": label, "target_ops_per_s": rate, "match_topics_per_s": n * ch_steps / (ms_c / 1e3),
                                      "mutation_ops_per_s": d["ops_per_s"], "flushes_per_s": d["flushes_per_s"], "mean_flush_us": d["mean_flush_us"], "max_flush_us": d["max_flush_us"]})
            base = churn["legs"][0]["match_topics_per_s"]
            for leg in churn["legs"]:
                leg["match_throughput_vs_no_churn"] = leg["match_topics_per_s"] / base
            return churn

        def latency_leg():
            """per-PUBLISH latency through the single-call front end (gm_submit -> batcher -> small-batch graph / pipelined path)"""
            lat = N.GmLatency()
            hb0, ho0 = host_batches[0]
            table = []
            for burst, rounds in ((1, 2000), (32, 400), (1024, 60), (32768, 12), (n, 4)):
                burst = min(burst, n)
                rc = lib.gm_batcher_probe(eng._h, hb0.ctypes.data, ho0.ctypes.data, n, burst, rounds, 0, C.byref(lat))
                assert rc == 0, lib.gm_last_error(eng._h)
                d = lat.as_dict()
                table.append({"offered_burst": burst, "p50_us": d["p50_us"], "p99_us": d["p99_us"], "mean_us": d["mean_us"], "topics_per_s": d["topics_per_s"], "samples": d["samples"]})
            out = {"front_end": "gm_submit (MPSC queue) -> 2 dispatcher threads -> gm_match_batch; bursts <= 2048 topics run as ONE CUDA-graph launch; "
                                "closed loop: the next burst is offered when every callback of the previous one has run; max_wait_us = 0",
                   "table": table}
            one_thread = (_PARTIAL.get("cpu_baseline") or {}).get("single_thread_value")
            if one_thread:
                cpu_lat_us = 1e6 / one_thread
                cross = next((r["offered_burst"] for r in table if r["topics_per_s"] > one_thread), None)
                out["cpu_port_single_thread_us_per_publish"] = cpu_lat_us
                out["crossover"] = (f"one CPU thread answers a PUBLISH in {cpu_lat_us:.1f} us; the GPU front end's throughput passes one CPU thread "
                                    f"at an offered burst of {cross} topics")
            return out

        _PARTIAL["cpu_baseline"] = _leg("cpu_baseline", cpu_leg, errors)
        _PARTIAL["churn"] = _leg("churn", churn_leg, errors)
        port.clear()
        _PARTIAL["latency"] = _leg("latency", latency_leg, errors)
        if not args.no_c4:
            _PARTIAL["c4"] = _leg("c4", lambda: _c4_leg(torch, dev, stream, peak, small), errors)
        _PARTIAL["relations"] = _leg("relations", lambda: _relations_leg(small), errors)
        _PARTIAL["configs"] = _leg("configs", lambda: _configs_leg(torch, eng, cfg, dev, stream, timed_device_loop, d_spans, d_ids, d_needed, d_status, small), errors)

    line = dict(_PARTIAL)
    if errors:
        line["errors"] = errors
    if multi and "value_with_gather" in multi:
        line["value_with_gather"] = multi["value_with_gather"]
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


_RESULT_OUT = sys.stdout
_PARTIAL: dict = {}            # rank 0: the result line as far as it has been measured (see _bail)
_EMIT_LOCK = threading.Lock()
_EMITTED = False


def _jsonable(o):
    if isinstance(o, np.generic):
        return o.item()
    if isinstance(o, np.ndarray):
        return o.tolist()
    return str(o)


def _emit(line: dict) -> None:
    """Exactly ONE line on the real stdout, whoever gets here first (normal end, exception handler or watchdog)."""
    global _EMITTED
    with _EMIT_LOCK:
        if _EMITTED:
            return
        print(json.dumps(line, default=_jsonable), file=_RESULT_OUT, flush=True)
        _EMITTED = True


def _leg(name: str, fn, errors: dict):
    """A secondary leg (single-rank, no collective inside) must not take the headline down with it: its exception is
    recorded under `errors` in the line, the key of the leg stays null."""
    try:
        return fn()
    except Exception as ex:                                   # noqa: BLE001 - anything a leg throws is reported, not raised
        errors[name] = f"{type(ex).__name__}: {ex}"[:300]
        traceback.print_exc(file=sys.stderr)
        return None


def _bail(why: str, code: int) -> None:
    """Abnormal end (exception in a collective leg, or the watchdog's deadline): rank 0 prints the headline measured so far —
    the timed loops, e2e and roofline come first in run_own — with the reason under `errors`; then the process ends at once
    (other ranks may be blocked in a collective that will never complete).  Exit code 0 when the line carries the headline."""
    rank0 = int(os.environ.get("RANK", "0")) == 0
    if rank0 and "value" in _PARTIAL and not _EMITTED:
        line = dict(_PARTIAL)
        line.setdefault("errors", {})["bench"] = why[:400]
        _emit(line)
        code = 0
    elif _EMITTED or not rank0:
        code = 0                                              # the verdict is rank 0's line (or its absence), not this exit code
    sys.stderr.flush()
    os._exit(code)


def _watchdog(seconds: float) -> None:
    t = threading.Timer(seconds, _bail, args=(f"deadline of {seconds:.0f} s reached (BENCH_DEADLINE_S); secondary legs still running were cut off", 3))
    t.daemon = True
    t.start()


if __name__ == "__main__":
    a = _args()
    # stdout carries exactly ONE line (the JSON result): keep a private handle to it and point fd 1 at stderr so that
    # library chatter written by native code (e.g. NCCL's "NCCL version ..." banner) cannot land on it.
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    # a normal run takes 2 - 4 minutes; the driver's limits are 1800 s (N=1) and 870 s per N of the scaling run
    _watchdog(float(os.environ.get("BENCH_DEADLINE_S", "780")))
    try:
        if a.impl == "reference":
            run_reference(a)
        else:
            run_own(a)
    except BaseException as ex:                               # noqa: BLE001
        if isinstance(ex, SystemExit) and not ex.code:
            raise
        traceback.print_exc(file=sys.stderr)
        if int(os.environ.get("RANK", "0")) != 0 and int(os.environ.get("WORLD_SIZE", "1")) > 1:
            # a failing non-zero rank must not make torchrun tear rank 0 down before it has printed what it measured:
            # stay until the watchdog (here or on rank 0) ends the job
            threading.Event().wait()
        _bail(f"{type(ex).__name__}: {ex}", 1)
