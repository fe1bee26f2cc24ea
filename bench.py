#!/usr/bin/env python
"""bench.py — BASELINE.json's headline metric on B200.

Headline workload (config.workload): BASELINE config 4 — 5-term SHOULD BooleanQuery (DisjunctionSumScorer)
BM25 top-100, batch 4096, 100M-doc synthetic Zipfian index (1M terms), evaluated by IndexSearcher::search
through the C ABI.  One "step" = one pass of the whole query batch.

  value  : queries/sec, whole job, kernels only (plan + index resident in HBM), max over ranks
  e2e    : queries/sec through rg_search_batch with HOST query arrays in and HOST TopDocs out
           (planning, H2D of the plan, kernels, D2H of results inside the timed region)
  roofline: the evaluation kernels (k_eval_or_ms + k_eval_or, or k_eval_and): algorithmic bytes per launch
           (SURVEY 8d) / CUDA-event time, against MEASURED_PEAKS.json
  cpu_baseline: the oracle (C++ restatement of the reference's CPU path, kind "port") timed on the box's
           usable host cores on a bounded sample of the same batch; the GPU result is checked against it
  workloads: with the default command line at N=1 also BASELINE configs 3 (2-term MUST, 10M docs) and 5
           (8 segments, mixed AND/OR, batch 8192), each with its own parity verdict
  forutil_decode: BASELINE config 2 — uniform-width blocks, the realistic blocks of the 100M index, a
           per-width sweep and the raw-stream kernel, GB/s vs the measured HBM peak

N>1 (torchrun): the index is split into docid-range segments (c4/c3: N of them; c5: always 8), contiguous
leaves per rank; every rank evaluates the whole batch on its leaves (search_parallel semantics), ONE NCCL
all-gather moves the per-leaf top-k records and every rank replays finish_parallel in leaf order.  Rank 0
then rebuilds ALL leaves for the oracle and checks a sample, so every N carries a parity verdict.
`--impl reference` times the oracle alone (rank 0 only).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED_INDEX = 0x5EED0001
SEED_BLOCKS = 0x5EED0002

WORKLOADS = {
    # name: docs, terms, batch, k, segments (0 = one per rank), index seed, query seed
    "c4": dict(docs=100_000_000, terms=1_000_000, batch=4096, k=100, segments=0, seed_index=SEED_INDEX,
               seed_queries=0x5EED0004,
               what="C4: 5-term SHOULD BooleanQuery (DisjunctionSumScorer)"),
    "c3": dict(docs=10_000_000, terms=100_000, batch=1024, k=10, segments=0, seed_index=SEED_INDEX,
               seed_queries=0x5EED0003,
               what="C3: 2-term MUST BooleanQuery (ConjunctionScorer)"),
    "c5": dict(docs=100_000_000, terms=1_000_000, batch=8192, k=100, segments=8, seed_index=0x5EED0005,
               seed_queries=0x5EED0005,
               what="C5: alternating 2-3-term MUST / 3-5-term SHOULD BooleanQuerys, search_parallel over 8 segments"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--docs", type=int, default=int(os.environ.get("RUCENE_BENCH_DOCS", 0)))
    ap.add_argument("--terms", type=int, default=int(os.environ.get("RUCENE_BENCH_TERMS", 0)))
    ap.add_argument("--batch", type=int, default=int(os.environ.get("RUCENE_BENCH_BATCH", 0)))
    ap.add_argument("--k", type=int, default=0)
    ap.add_argument("--cpu-sample", type=int, default=int(os.environ.get("RUCENE_BENCH_CPU_SAMPLE", 1024)),
                    help="upper bound on the queries of the batch the CPU baseline evaluates")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="time bound of the CPU baseline sample")
    ap.add_argument("--range-postings", type=int, default=0)
    ap.add_argument("--no-decode", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the C3 / C5 legs and the A/B legs of the default run")
    ap.add_argument("--no-columns", action="store_true",
                    help="RG_CFG_NO_COLUMNS: evaluate every clause from its block stream (A/B runs)")
    ap.add_argument("--no-lists", action="store_true", help="RG_CFG_NO_LISTS: no scored posting lists (A/B runs)")
    ap.add_argument("--tf-planes", action="store_true", help="RG_CFG_TFPLANES: three-level per-document bound (A/B runs)")
    ap.add_argument("--stats", action="store_true", help="RG_CFG_STATS: event counters of k_eval_or_ms in the line")
    ap.add_argument("--maxscore", action="store_true",
                    help="RG_CFG_MAXSCORE: disjunctions through k_eval_or_ms (bitmaps + per-document bound) (A/B runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the TopDocs of the last timed step of the headline workload to DIR/*.npy")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    w = dict(WORKLOADS[a.workload])
    for key in ("docs", "terms", "batch", "k"):
        if getattr(a, key):
            w[key] = getattr(a, key)
    a.w = w
    a.scaled = any(getattr(a, key) for key in ("docs", "terms", "batch", "k"))
    return a


def usable_cores():
    """Cores this process may actually use: CPU affinity, capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, p = f.read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(p))))
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = int(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                p = int(f.read())
            if q > 0:
                n = min(n, max(1, q // p))
        except Exception:
            pass
    return max(1, n)


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.p, self.t, self.index = [], None, None, index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None
            return
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].startswith("Active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------ queries
def _rank_sample(rng, n_terms):
    """SURVEY §8d: rank r = floor(V^U) (log-uniform) -> 0-based term id."""
    r = int(np.floor(float(n_terms) ** rng.random()))
    return min(max(r, 1), n_terms) - 1


def gen_queries(name, n_terms, batch, seed):
    """-> list of (occur, [term ids]); occur 'must' | 'should'.  Terms distinct within a query."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(batch):
        if name == "c4":
            occ, t = "should", 5
        elif name == "c3":
            occ, t = "must", 2
        else:  # c5: alternate by index
            occ = "must" if i % 2 == 0 else "should"
            t = int(rng.integers(2, 4)) if occ == "must" else int(rng.integers(3, 6))
        chosen = []
        while len(chosen) < t:
            c = _rank_sample(rng, n_terms)
            if c not in chosen:
                chosen.append(c)
        out.append((occ, chosen))
    return out


def build_query_arrays(qs, weight_of, E):
    """-> rg_query[], rg_clause[] for BooleanQuery::build(musts | shoulds of TermQuery)."""
    n_cl = sum(len(t) for _, t in qs)
    q = np.zeros(len(qs), E.QUERY_DTYPE)
    c = np.zeros(n_cl, E.CLAUSE_DTYPE)
    pos = 0
    for i, (occ, terms) in enumerate(qs):
        q["clause_begin"][i] = pos
        q["n_clauses"][i] = len(terms)
        for t in terms:
            c["occur"][pos] = E.MUST if occ == "must" else E.SHOULD
            c["term_id"][pos] = t
            c["weight"][pos] = weight_of(t)
            pos += 1
    q["flags"] = E.Q_BOOLEAN
    return q, c


def oracle_queries(ob, qs):
    specs = [("bool", [((ob.MUST if occ == "must" else ob.SHOULD), int(t)) for t in terms], 0) for occ, terms in qs]
    return ob.make_queries(specs)


def oracle_mod():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding as ob
    return ob


def query_costs(qs, df_by_seg):
    """postings the reference's scorers iterate per query (sum of df over clauses, over all leaves)."""
    df = np.sum(np.stack(df_by_seg), axis=0)
    return np.array([int(df[np.asarray(ts)].sum()) for _, ts in qs], np.int64)


def same_topdocs(got, want, idx):
    """got: full-batch (hits, counts, total); want: the sample's; idx: sample -> batch index."""
    gh, gc, gt = got
    wh, wc, wt = want
    if not (np.array_equal(gt[idx], wt) and np.array_equal(gc[idx], wc)):
        return False
    for j, i in enumerate(idx):
        n = int(wc[j])
        if not (np.array_equal(gh[i][:n]["doc"], wh[j][:n]["doc"]) and
                np.array_equal(gh[i][:n]["score"].view(np.uint32), wh[j][:n]["score"].view(np.uint32))):
            return False
    return True


class _CudaArray:
    """__cuda_array_interface__ view of engine-owned device memory (for torch.as_tensor)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False),
                                         "version": 2, "strides": None}


def seg_layout(w, world):
    """-> (n_segments, docs per segment)."""
    n = w["segments"] or world
    return n, w["docs"] // n


def workload_config(name, w, world):
    n_seg, seg_docs = seg_layout(w, world)
    return {"workload": "%s BM25 top-%d, batch %d, %d-doc Zipfian synthetic index, %d terms"
                        % (w["what"], w["k"], w["batch"], w["docs"], w["terms"]),
            "name": name, "batch": w["batch"], "k": w["k"], "docs": w["docs"], "terms": w["terms"],
            "segments": n_seg, "segment_docs": seg_docs,
            "parallelism": ("%d docid-range segments, %d per GPU" % (n_seg, n_seg // world)) if n_seg > 1 else "single GPU, one segment",
            "cache": "index image + score columns (GBs) exceed the 126 MB L2; no explicit flush"}


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_sample_run(ob, ix, qs, costs, k, mode, cores, max_queries, seconds):
    """The oracle on `cores` threads over a sample of the batch: longest-first order (dynamic scheduling, so
    the wall time is not the tail of one heavy query), 256 queries first, more while the time bound allows."""
    n = len(qs)
    first = min(256, n, max_queries)
    order = np.arange(first)
    order = order[np.argsort(-costs[order], kind="stable")]
    oq, oc = oracle_queries(ob, [qs[i] for i in order])
    t0 = time.perf_counter()
    res = ix.search_batch(oq, oc, k, parallel_mode=mode, n_threads=cores)
    dt = time.perf_counter() - t0
    idx, want, wall = order, res, dt
    more = min(max_queries, n) - first
    if more > 0 and dt * (more / first) < max(0.0, seconds - dt):
        order2 = np.arange(first, first + more)
        order2 = order2[np.argsort(-costs[order2], kind="stable")]
        oq, oc = oracle_queries(ob, [qs[i] for i in order2])
        t0 = time.perf_counter()
        res2 = ix.search_batch(oq, oc, k, parallel_mode=mode, n_threads=cores)
        dt2 = time.perf_counter() - t0
        idx = np.concatenate([order, order2])
        want = tuple(np.concatenate([a, b]) for a, b in zip(res, res2))
        wall = dt + dt2
    return idx, want, wall


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port) on the usable host cores."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from rucene_b200 import codec
    name, w = args.workload, args.w
    world = args.gpus
    n_seg, seg_docs = seg_layout(w, world)
    ob = oracle_mod()
    ix = ob.Index(1.2, 0.75)
    dfs = []
    for s in range(n_seg):
        seg = codec.synth_segment(w["seed_index"] + s, seg_docs, w["terms"], doc_version=1)
        ix.add_segment(seg)
        dfs.append(seg.terms["doc_freq"].astype(np.int64))
    qs = gen_queries(name, w["terms"], w["batch"], w["seed_queries"])
    costs = query_costs(qs, dfs)
    cores = usable_cores()
    mode = 1 if n_seg > 1 else 0
    # size the per-step sample from a probe so that steps+warmup stay within a few minutes (~6 s per step)
    probe = min(128, len(qs))
    pq, pc = oracle_queries(ob, qs[:probe])
    t0 = time.perf_counter()
    ix.search_batch(pq, pc, w["k"], parallel_mode=mode, n_threads=cores)
    rate = probe / max(1e-6, time.perf_counter() - t0)
    sample = int(min(len(qs), max(min(256, len(qs)), rate * 6.0)))
    times = []
    for step in range(args.warmup + args.steps):
        lo = (step * sample) % max(1, len(qs) - sample + 1)
        sel = np.arange(lo, lo + sample)
        sel = sel[np.argsort(-costs[sel], kind="stable")]
        q, c = oracle_queries(ob, [qs[i] for i in sel])
        t0 = time.perf_counter()
        ix.search_batch(q, c, w["k"], parallel_mode=mode, n_threads=cores)
        dt = time.perf_counter() - t0
        if step >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = sample / (ms / 1e3)
    line = {"impl": "reference", "metric": "queries/sec", "value": value, "unit": "queries/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32/f32",
            "data": "synthetic", "config": workload_config(name, w, world),
            "cpu_baseline": {"value": value, "unit": "queries/s", "cores": cores, "kind": "port",
                             "os_cpu_count": os.cpu_count(),
                             "sample": "%d queries of the batch per step (a sliding window, longest first), one query per "
                                       "thread, dynamic scheduling" % sample},
            "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ GPU arm
class Ctx:
    pass


def run_workload(ctx, name, w, args, steps, warmup, cpu_queries, cpu_seconds, flags=0, light=False):
    """One workload on the current process group.  light: value only (A/B legs)."""
    import torch
    import torch.distributed as dist
    from rucene_b200 import codec, engine

    world, rank, dev, stream = ctx.world, ctx.rank, ctx.dev, ctx.stream
    n_seg, seg_docs = seg_layout(w, world)
    assert n_seg % world == 0, "segments must divide evenly over the ranks"
    per_rank = n_seg // world
    my_segs = list(range(rank * per_rank, (rank + 1) * per_rank))
    t0 = time.perf_counter()
    segs = [codec.synth_segment(w["seed_index"] + s, seg_docs, w["terms"], doc_version=1) for s in my_segs]
    t_gen = time.perf_counter() - t0
    eng = engine.Engine(device=ctx.local_rank, range_postings=args.range_postings, flags=flags)
    eng.set_stream(stream.cuda_stream)
    t0 = time.perf_counter()
    for s, seg in zip(my_segs, segs):
        eng.upload_segment(seg, doc_base=s * seg_docs)
    t_up = time.perf_counter() - t0

    # ---- weights: statistics of the largest leaf = leaf 0 (searcher.rs:311-351,732-767), same on every rank
    df0 = torch.from_numpy(segs[0].terms["doc_freq"].astype(np.int32)).to(dev)
    st0 = torch.tensor([segs[0].doc_count, segs[0].sum_total_term_freq], dtype=torch.int64, device=dev)
    if world > 1:
        dist.broadcast(df0, 0)
        dist.broadcast(st0, 0)
    df0 = df0.cpu().numpy()
    doc_count, sum_ttf = int(st0[0]), int(st0[1])
    avgdl = codec.bm25_avg_field_length(sum_ttf, doc_count, w["docs"])
    eng.set_norm_cache(0, codec.bm25_norm_cache(1.2, 0.75, avgdl))
    idf_cache = {}

    def weight_of(t):
        if t not in idf_cache:
            idf_cache[t] = np.float32(codec.bm25_idf(int(df0[t]), doc_count))  # boost 1.0
        return idf_cache[t]

    qs = gen_queries(name, w["terms"], w["batch"], w["seed_queries"])
    q, c = build_query_arrays(qs, weight_of, engine)
    nq, k = len(qs), w["k"]
    mode = engine.MODE_SEARCH_PARALLEL if n_seg > 1 else engine.MODE_SEARCH

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- first batch on a cold engine (score columns are built here), then the resident plan
    barrier()
    t0 = time.perf_counter()
    batch = eng.prepare(q, c, k, k1=1.2, mode=mode)
    batch.run()
    torch.cuda.synchronize()
    first_batch_ms = (time.perf_counter() - t0) * 1e3
    col_stats_cold = eng.column_stats()
    rec_bytes = 16 + 8 * k
    gathered = local_rec = None
    if world > 1:
        rec_ptr, _ = batch.leaf_records()
        local_rec = torch.as_tensor(_CudaArray(rec_ptr, per_rank * rec_bytes * nq), device=dev)
        gathered = torch.empty(world * per_rank * rec_bytes * nq, dtype=torch.uint8, device=dev)

    def one_step():
        batch.run()
        if world > 1:  # kernels -> one all-gather -> leaf-order merge, all on one stream; the result stays on the device
            dist.all_gather_into_tensor(gathered, local_rec)
            eng.merge_leaf_records_device(gathered.data_ptr(), n_seg, nq, k)

    for _ in range(warmup):
        one_step()
    barrier()
    sampler = ClockSampler(ctx.local_rank)
    if rank == 0 and not light:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = eng.launch_count()
    ev0.record(stream)
    for _ in range(steps):
        one_step()
    ev1.record(stream)
    barrier()
    clocks = sampler.stop() if (rank == 0 and not light) else None
    ms_total = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
    ms_step = float(ms_total[0]) / steps
    launches = eng.launch_count() - launches0
    # the TopDocs of the last timed step, copied back without running the batch again
    result = batch.fetch() if world == 1 else eng.merge_fetch()
    if world > 1:
        batch.fetch()  # populates the per-kernel CUDA-event timings of the last run
    eval_ms = eng.last_kernel_ms("eval")
    replay_ms = eng.last_kernel_ms("replay")
    bstats = batch.stats()
    n_cols, col_bytes = batch.columns()
    dbg_all = batch.debug()
    dbg = dbg_all if (flags & engine.CFG_STATS) else None
    out = {"value": nq / (ms_step / 1e3), "ms_per_step": ms_step, "config": workload_config(name, w, world)}
    per_rank_eval = [eval_ms]
    if world > 1:
        t = torch.tensor([eval_ms], dtype=torch.float64, device=dev)
        allv = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allv, t)
        per_rank_eval = [float(x[0]) for x in allv]
    if light:
        batch.close()
        eng.close()
        return out

    # ---- e2e: host arrays in, host TopDocs out.  Timed on batches the engine has NOT seen (fresh query seeds, same
    # distribution): the persistent score columns / scored lists only help where a term recurs across or within
    # batches, and whatever a new batch still has to build is inside its rg_batch_prepare, i.e. inside the timed region.
    # The repeated-batch figure (every cache hot) is reported next to it.
    def e2e_step(qa, ca):
        if world == 1:
            return eng.search_batch(qa, ca, k, k1=1.2, mode=mode)
        b2 = eng.prepare(qa, ca, k, k1=1.2, mode=mode)
        b2.run()
        p2, _ = b2.leaf_records()
        loc = torch.as_tensor(_CudaArray(p2, per_rank * rec_bytes * nq), device=dev)
        dist.all_gather_into_tensor(gathered, loc)
        res = eng.merge_leaf_records(gathered.data_ptr(), n_seg, nq, k)
        b2.close()
        return res

    e2e_steps = steps
    fresh = [build_query_arrays(gen_queries(name, w["terms"], w["batch"], w["seed_queries"] + 7919 * (i + 1)), weight_of, engine)
             for i in range(e2e_steps)]
    e2e_res = e2e_step(q, c)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step(q, c)
    barrier()
    rep_ms = torch.tensor([(time.perf_counter() - t0) * 1e3 / e2e_steps], dtype=torch.float64, device=dev)
    cache0 = (eng.column_stats(), eng.list_stats())
    barrier()
    t0 = time.perf_counter()
    for qa, ca in fresh:
        e2e_step(qa, ca)
    barrier()
    e2e_ms = torch.tensor([(time.perf_counter() - t0) * 1e3 / e2e_steps], dtype=torch.float64, device=dev)
    cache1 = (eng.column_stats(), eng.list_stats())
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(rep_ms, op=dist.ReduceOp.MAX)
    e2e_ms, rep_ms = float(e2e_ms[0]), float(rep_ms[0])
    # the same unseen batches through the split calls, two in flight: batch i+1 is planned and uploaded (copy stream)
    # while batch i runs; the fetch waits for batch i only
    pipe_ms = None
    if world == 1:
        more = [build_query_arrays(gen_queries(name, w["terms"], w["batch"], w["seed_queries"] + 7919 * (i + 101)), weight_of, engine)
                for i in range(e2e_steps + 1)]
        torch.cuda.synchronize()
        nxt = eng.prepare(more[0][0], more[0][1], k, k1=1.2, mode=mode)
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            cur = nxt
            cur.run()
            nxt = eng.prepare(more[i + 1][0], more[i + 1][1], k, k1=1.2, mode=mode)
            cur.fetch()
            cur.close()
        pipe_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
        nxt.close()
    e2e_split = fresh_split = None
    if world == 1:  # where the e2e time goes (one extra step through the split calls): the repeated batch, a new one
        def split_of(qa, ca):
            torch.cuda.synchronize()
            ta = time.perf_counter()
            b3 = eng.prepare(qa, ca, k, k1=1.2, mode=mode)
            tb = time.perf_counter()
            b3.run()
            torch.cuda.synchronize()
            tc = time.perf_counter()
            b3.fetch()
            td = time.perf_counter()
            b3.close()
            return {"prepare_ms": (tb - ta) * 1e3, "run_ms": (tc - tb) * 1e3, "fetch_ms": (td - tc) * 1e3}
        e2e_split = split_of(q, c)
        fresh_split = split_of(*build_query_arrays(gen_queries(name, w["terms"], w["batch"], w["seed_queries"] + 7919 * 17), weight_of, engine))
    d2h = nq * k * 8 + nq * 4 + nq * 8
    h2d = bstats["h2d_bytes"] + q.nbytes + c.nbytes
    consistent = bool(np.array_equal(result[0]["doc"], e2e_res[0]["doc"]) and np.array_equal(result[2], e2e_res[2]))

    out.update({"e2e": {"value": nq / (e2e_ms / 1e3), "unit": "queries/s", "ms_per_step": e2e_ms,
                        "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "batches": "%d batches the engine had not seen (query seeds +7919*i), one per step" % e2e_steps,
                        "split": fresh_split,
                        "pipelined": None if pipe_ms is None else {
                            "value": nq / (pipe_ms / 1e3), "ms_per_step": pipe_ms,
                            "note": "rg_batch_prepare of batch i+1 overlaps rg_batch_run of batch i (plan uploads and result "
                                    "fetches ride the engine's copy stream); unseen batches, host arrays in, host TopDocs out"},
                        "built_during_these_steps": {"score_columns": cache1[0]["built"] - cache0[0]["built"],
                                                     "scored_lists": cache1[1]["built"] - cache0[1]["built"]},
                        "repeated_batch": {"value": nq / (rep_ms / 1e3), "ms_per_step": rep_ms, "split": e2e_split,
                                           "same_result_as_resident_path": consistent}},
                "gpu_launches": int(launches), "clocks": clocks,
                "first_batch_ms": first_batch_ms, "kernel_events": dbg,
                "per_rank_eval_ms": per_rank_eval,
                "setup": {"index_gen_s": t_gen, "upload_s": t_up, "index_image_bytes": eng.index_bytes(),
                          "doc_file_bytes": int(sum(s.doc_file.size for s in segs)),
                          "upload_GBs_of_doc_file": sum(s.doc_file.size for s in segs) / t_up / 1e9,
                          "postings": int(sum(s.sum_doc_freq for s in segs)), "host_cores": usable_cores()}})
    ctx.eng_for_decode = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        algo_bytes = bstats["algorithmic_bytes"]
        upper_bytes = None
        if name == "c3" and dbg_all["and_touched_bytes"] > 0:
            # conjunctions: SURVEY 8d asks for TOUCHED blocks — counted by the kernel itself (lead list in full +
            # the blocks / table entries / column cells it probed); the planner's figure is the upper bound
            upper_bytes, algo_bytes = algo_bytes, dbg_all["and_touched_bytes"] + nq * k * 8
        achieved = algo_bytes / (eval_ms / 1e3) / 1e9 if eval_ms > 0 else 0.0
        out["roofline"] = {
            "bound": "hbm", "kernel": "k_eval_and" if name == "c3" else ("k_eval_or_ms (+ k_eval_or)" if flags & engine.CFG_MAXSCORE else "k_eval_or"),
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": ctx.traffic.get(name),
            "peak_source": peak_src, "algorithmic_bytes_per_launch": algo_bytes, "upper_bound_bytes_all_lists": upper_bytes,
            "kernel_ms": eval_ms,
            "replay_ms": replay_ms, "postings_per_launch": bstats["postings"], "work_items": bstats["items"],
            "candidate_slots": bstats["candidate_slots"],
            "note": "algorithmic bytes = SURVEY 8d: every clause's encoded blocks + tails + 12 B/block of tables + one "
                    "norm byte per posting (conjunctions: the bytes the kernel itself counted — lead list + touched "
                    "blocks / table entries / column cells).  Dense clauses that have a score column are read from it "
                    "(4 B per docid) instead of being decoded; traffic = DRAM bytes actually moved (ncu, profiles/)",
            "scored_lists": dict(eng.list_stats(), note="(docid, f32 score) pairs of disjunction clauses two queries of a batch share, "
                                 "1 KB per 128-posting block; kept across batches in the engine's list arena (a ring of slabs, <= 1/6 of the free HBM)"),
            "score_columns": {"n": n_cols, "bytes": col_bytes, "built_by_first_batch": col_stats_cold["built"],
                              "engine_cache": eng.column_stats(),
                              "note": "persistent across batches (LRU, <= 1/3 of the free HBM); the timed steps hit the "
                                      "cache, first_batch_ms includes building them"}}
    # ---- parity: the reference's algorithm on the host, sample of the batch (rank 0; all leaves)
    if rank == 0:
        ob = oracle_mod()
        ix = ob.Index(1.2, 0.75)
        dfs = []
        for s in range(n_seg):
            seg = segs[s - my_segs[0]] if s in my_segs else codec.synth_segment(w["seed_index"] + s, seg_docs, w["terms"], doc_version=1)
            ix.add_segment(seg)
            dfs.append(seg.terms["doc_freq"].astype(np.int64))
        costs = query_costs(qs, dfs)
        cores = usable_cores()
        idx, want, wall = cpu_sample_run(ob, ix, qs, costs, k, 1 if n_seg > 1 else 0, cores, cpu_queries, cpu_seconds)
        ok = same_topdocs(result, want, idx)
        cpu = {"value": len(idx) / wall, "unit": "queries/s", "cores": cores, "kind": "port",
               "os_cpu_count": os.cpu_count(),
               "sample": "%d queries of the batch (the first %d, longest first), one query per thread, dynamic scheduling, "
                         "%.2f s wall" % (len(idx), len(idx), wall),
               "sample_postings": int(costs[idx].sum()),
               "postings_per_s_all_cores": float(costs[idx].sum() / wall),
               "parity_on_sample": "identical TopDocs" if ok else "MISMATCH"}
        if name == "c4" and world == 1:  # single-thread figure on a few queries (bounded by postings)
            pick, acc = [], 0
            for i in range(len(qs)):
                if acc >= 120_000_000 or len(pick) >= 16:
                    break
                pick.append(i)
                acc += int(costs[i])
            oq, oc = oracle_queries(ob, [qs[i] for i in pick])
            t0 = time.perf_counter()
            ix.search_batch(oq, oc, k, parallel_mode=0, n_threads=1)
            dt = time.perf_counter() - t0
            cpu["single_thread"] = {"queries": len(pick), "queries_per_s": len(pick) / dt,
                                    "postings_per_s": float(costs[pick].sum() / dt)}
        out["cpu_baseline"] = cpu
        del ix
    ctx.last_engine, ctx.last_batch, ctx.last_result = eng, batch, result
    return out


def decode_bench(eng, stream, have_full_index):
    """BASELINE config 2 on an engine that still holds the C4 segment."""
    import torch
    from rucene_b200 import codec
    peak, _ = measured_peaks()
    res = {}
    nb = 1_000_000

    def time_staged(bs_handle, reps=20):
        for _ in range(3):
            bs_handle.decode()
        torch.cuda.synchronize()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record(stream)
        for _ in range(reps):
            bs_handle.decode()
        d1.record(stream)
        torch.cuda.synchronize()
        return d0.elapsed_time(d1) / reps

    # (i) uniform widths 1..32, staged 16-byte aligned parts
    bs = codec.synth_blocks(SEED_BLOCKS, nb, mode=0, doc_version=1)
    st = eng.stage_blocks(bs.stream, bs.offsets, 1, codec.forutil_table())
    dms = time_staged(st)
    s = st.stats()
    rw = (s["encoded_bytes"] + s["decoded_bytes"]) / (dms / 1e3) / 1e9
    res.update({"blocks": nb, "ms": dms, "read_write_GBs": rw, "read_only_GBs": s["encoded_bytes"] / (dms / 1e3) / 1e9,
                "frac_of_hbm_peak": rw / peak, "bytes_read": s["encoded_bytes"], "bytes_written": s["decoded_bytes"],
                "note": "(i) staged 16B-aligned blocks, uniform widths 1..32; 777 MB/pass > L2"})
    st.close()
    # the raw codec stream (unaligned bytes), same blocks: k_decode_raw, kernel time only
    eng.forutil_decode(bs.stream, bs.offsets[:200_000], 1, codec.forutil_table())
    eng.forutil_decode(bs.stream, bs.offsets[:200_000], 1, codec.forutil_table())
    raw_ms = eng.last_kernel_ms("decode")
    enc = int(bs.offsets[200_000] - bs.offsets[0])
    res["raw_stream"] = {"kernel": "k_decode_raw", "blocks": 200_000, "ms": raw_ms,
                         "read_write_GBs": (enc + 200_000 * 512) / (raw_ms / 1e3) / 1e9,
                         "frac_of_hbm_peak": (enc + 200_000 * 512) / (raw_ms / 1e3) / 1e9 / peak}
    del bs
    # (iii) per-width sweep (staged)
    sweep = {}
    for b in (0, 1, 2, 4, 7, 8, 12, 16, 20, 24, 28, 31, 32):
        bsw = codec.synth_blocks(SEED_BLOCKS + 100 + b, 500_000, mode=1, param=b, doc_version=1)
        stw = eng.stage_blocks(bsw.stream, bsw.offsets, 1, codec.forutil_table())
        ms = time_staged(stw, reps=10)
        sw = stw.stats()
        sweep[str(b)] = round((sw["encoded_bytes"] + sw["decoded_bytes"]) / (ms / 1e3) / 1e9, 1)
        stw.close()
        del bsw
    res["width_sweep_read_write_GBs"] = sweep
    # (ii) realistic: every doc-delta + freq block pair of the index, in file order
    if have_full_index:
        eng.segment_decode(0)
        stats, _ = eng.segment_decode(0)
        ms = eng.last_kernel_ms("decode")
        rwb = stats["encoded_bytes"] + stats["decoded_bytes"]
        res["realistic"] = {"kernel": "k_decode_segment", "block_pairs": stats["blocks"], "ms": ms,
                            "read_write_GBs": rwb / (ms / 1e3) / 1e9, "frac_of_hbm_peak": rwb / (ms / 1e3) / 1e9 / peak,
                            "read_only_GBs": stats["encoded_bytes"] / (ms / 1e3) / 1e9,
                            "bytes_read": stats["encoded_bytes"], "bytes_written": stats["decoded_bytes"],
                            "note": "(ii) all doc-delta and freq blocks of the bench index in file order"}
    return res


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, result):
    """TopDocs as a caller of the timed path receives them, one row per query: doc ids (float64: exact for every
    int32), scores (float32), hit counts and total hits.  Slots past a row's hit count are not part of its TopDocs
    and are written as doc -1, score 0.  Above DUMP_LIMIT_BYTES a fixed seeded sample of rows is written;
    query_rows.npy holds the batch index of each row."""
    hits, counts, total = result
    nq, k = hits.shape
    rows = np.arange(nq)
    row_bytes = k * (8 + 4) + 8 + 8 + 8
    if nq * row_bytes > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0x5EED00D0).choice(nq, DUMP_LIMIT_BYTES // row_bytes, replace=False))
    hits, counts, total = hits[rows], counts[rows], total[rows]
    valid = np.arange(k)[None, :] < counts[:, None]
    arrays = {"docs": np.where(valid, hits["doc"], -1).astype(np.float64),
              "scores": np.where(valid, hits["score"], np.float32(0)).astype(np.float32),
              "counts": counts.astype(np.float64), "total_hits": total.astype(np.float64),
              "query_rows": rows.astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_traffic():
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist
    from rucene_b200 import engine

    ctx = Ctx()
    ctx.world = int(os.environ.get("WORLD_SIZE", "1"))
    ctx.rank = int(os.environ.get("RANK", "0"))
    ctx.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(ctx.local_rank)
    ctx.dev = torch.device("cuda", ctx.local_rank)
    if ctx.world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=ctx.dev)
    # a dedicated (non-default) torch stream: the engine launches on it and torch.cuda.Event timing sees
    # exactly those launches
    ctx.stream = torch.cuda.Stream(device=ctx.dev)
    torch.cuda.set_stream(ctx.stream)
    tr = load_traffic()
    ctx.traffic = {} if args.scaled else {n: tr.get(n) for n in WORKLOADS}

    flags = ((engine.CFG_NO_COLUMNS if args.no_columns else 0) | (engine.CFG_NO_LISTS if args.no_lists else 0) |
             (engine.CFG_MAXSCORE if (args.maxscore or args.tf_planes) else 0) |
             (engine.CFG_STATS if args.stats else 0) | (engine.CFG_TFPLANES if args.tf_planes else 0))
    name, w = args.workload, args.w
    main_res = run_workload(ctx, name, w, args, args.steps, args.warmup, args.cpu_sample, args.cpu_seconds, flags=flags)
    eng, batch = ctx.last_engine, ctx.last_batch
    if args.dump_outputs and ctx.rank == 0:
        dump_outputs(args.dump_outputs, ctx.last_result)
    decode = None
    if ctx.rank == 0 and not args.no_decode:
        decode = decode_bench(eng, ctx.stream, have_full_index=True)
    batch.close()
    eng.close()
    extra = {}
    ab = {}
    if not args.no_extra and not args.scaled and name == "c4" and (flags & ~engine.CFG_STATS) == 0:
        # A/B legs on the same workload: what the other evaluation routes deliver (2 steps each)
        for label, fl in (("block_streams_only", engine.CFG_NO_COLUMNS | engine.CFG_NO_LISTS),
                          ("score_columns_no_scored_lists", engine.CFG_NO_LISTS),
                          ("bitmaps_per_document_bound", engine.CFG_MAXSCORE),
                          ("bitmaps_bound_with_tf_planes", engine.CFG_MAXSCORE | engine.CFG_TFPLANES)):
            r = run_workload(ctx, name, w, args, args.steps, args.warmup, 0, 0, flags=fl, light=True)
            ab[label] = {"queries_per_s": r["value"], "ms_per_step": r["ms_per_step"]}
        if ctx.world == 1:
            for other in ("c3", "c5"):
                r = run_workload(ctx, other, dict(WORKLOADS[other]), args, args.steps, args.warmup, 256, 8.0)
                ctx.last_batch.close()
                ctx.last_engine.close()
                extra[other] = {kk: r[kk] for kk in ("value", "ms_per_step", "config", "e2e", "first_batch_ms", "roofline",
                                                     "cpu_baseline", "gpu_launches") if kk in r}
    if ctx.rank == 0:
        line = {"metric": "queries/sec", "value": main_res["value"], "unit": "queries/s", "n_gpus": ctx.world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"],
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32/f32",
                "data": "synthetic", "config": main_res["config"], "e2e": main_res["e2e"],
                "gpu_launches": main_res["gpu_launches"], "clocks": main_res["clocks"],
                "roofline": main_res.get("roofline"), "cpu_baseline": main_res.get("cpu_baseline"),
                "first_batch_ms": main_res["first_batch_ms"], "per_rank_eval_ms": main_res["per_rank_eval_ms"],
                "step_breakdown": {"slowest_rank_eval_kernels_ms": max(main_res["per_rank_eval_ms"]),
                                   "rank_skew_ms": max(main_res["per_rank_eval_ms"]) - min(main_res["per_rank_eval_ms"]),
                                   "outside_eval_kernels_ms": main_res["ms_per_step"] - max(main_res["per_rank_eval_ms"]),
                                   "note": "ms_per_step = slowest rank's evaluation kernels + heap replay (+ all-gather and "
                                           "leaf-order merge at N > 1); against N = 1 the remainder is the per-leaf "
                                           "collectors' weaker theta (search_parallel semantics), not the exchange"},
                "kernel_events": main_res.get("kernel_events"),
                "forutil_decode": decode, "ab": ab or None, "workloads": extra or None, "setup": main_res["setup"]}
        print(json.dumps(line))
    if ctx.world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
