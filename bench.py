#!/usr/bin/env python
"""bench.py — BM25 top-k queries/sec on the 10M-doc synthetic corpus (BASELINE.json metric).

One "step" = one pass of the hot path over one batch of synthetic queries.
  value     : whole-job queries/s with the prepared batch already resident in HBM (kernels only, CUDA events)
  e2e       : the same through the C-ABI call with HOST buffers (canonicalise + H2D + kernels + D2H) per step
  roofline  : algorithmic bytes of the search kernel ÷ its device time vs the measured HBM copy peak
  cpu_baseline / --impl reference : the restated reference algorithm (Block-max WAND, oracle/) on the host cores

Launch: `python bench.py --gpus N --steps K --warmup W` (N>1: under torchrun, one rank per GPU; queries are
sharded across ranks with the index replicated — weak scaling: every rank runs its own full batch).  Every timed loop
runs K steps.  `--dump-outputs DIR` writes the result rows of the last timed step as DIR/<name>.npy (dump_outputs()).
"""
import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs (SURVEY.md §8d); the metric is quoted on the 10M-doc corpus, top-10
    "c3": dict(docs=10_000_000, vocab=100_000, doclen=128, queries=100_000, tmin=3, tmax=3, zipf=0.0, k=10,
               seed=0xB25C0DE0 + 3, desc="C3: 10M docs, vocab 100k uniform, 128 terms/doc, 100k 3-term OR queries"),
    "c2": dict(docs=1_000_000, vocab=30_000, doclen=64, queries=10_000, tmin=1, tmax=1, zipf=0.0, k=10,
               seed=0xB25C0DE0 + 2, desc="C2: 1M docs, vocab 30k, 64 terms/doc, 10k 1-term queries"),
    "c1": dict(docs=1_000, vocab=1_000, doclen=32, queries=100, tmin=3, tmax=3, zipf=0.0, k=10,
               seed=0xB25C0DE0 + 1, desc="C1: 1k docs, 100 3-term queries"),
    "c4": dict(docs=10_000_000, vocab=100_000, doclen=128, queries=4_000, tmin=8, tmax=8, zipf=1.0, k=10,
               seed=0xB25C0DE0 + 4, desc="C4: 10M docs Zipf(1), 8-term queries (4000-query subset; --no-prune = exhaustive)"),
    "c5": dict(docs=50_000_000, vocab=100_000, doclen=128, queries=1_000_000, tmin=1, tmax=8, zipf=0.0, k=10,
               seed=0xB25C0DE0 + 5, scaling="strong",
               desc="C5: 50M docs replicated, ONE batch of 1M mixed 1-8 term queries sharded over the GPUs, top-10"),
}


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {v}")
    return v


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=10, help="timed steps of every timed loop")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--docs", type=int)
    ap.add_argument("--queries", type=int)
    ap.add_argument("--k", type=int)
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling side leg of the default run")
    ap.add_argument("--no-prune", action="store_true", help="disable MaxScore-style pruning (exhaustive streaming)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's results of the last timed step as DIR/<name>.npy (see dump_outputs)")
    return ap.parse_args()


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            atexit.register(self._end)   # a run that fails between start() and stop() must not leave nvidia-smi behind
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def _end(self):
        if self.proc and self.proc.poll() is None:
            self.proc.terminate()
            self.proc.wait()

    def stop(self):
        self._end()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


METRIC = "queries/sec + achieved HBM GB/s, 10M-doc synthetic corpus, top-10"   # BASELINE.json's metric, both arms
REF_SAMPLE = 20_000   # queries per step of the CPU arms: the FIRST 20k queries of the batch, on every box


def effective_cores():
    """Host threads this process may really use: the affinity mask, capped by the cgroup CPU quota
    (os.cpu_count() ignores both: round 1 reported 128 "cores" on a box that granted ~12)."""
    n = len(os.sched_getaffinity(0))
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    eff = n if quota is None else max(1, min(n, int(quota + 0.5)))
    return eff, {"affinity": n, "cgroup_quota": quota, "os_cpu_count": os.cpu_count()}


def measured_traffic(workload, nq, k):
    """dram__bytes_read.sum + dram__bytes_write.sum of the search kernel from the COMMITTED ncu capture of this exact
    launch (profiles/*_traffic.json — newest kernel first; not measured in this run), else None."""
    for name in ("r3_traffic.json", "r2_traffic.json"):
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", name)))
            if t["workload"] == workload and t["queries"] == nq and t["k"] == k:
                return t["dram_bytes_read"] + t["dram_bytes_write"]
        except Exception:
            pass
    return None


def kernel_name(tmax, k, zipf=0.0):
    """The kernel instance the library launches for the widest query class of the workload (bm25x_search.cu)."""
    cls = next(c for c in (1, 2, 3, 4, 8, 16, 32) if c >= tmax)
    kp = 64 if k <= 32 else 256 if k <= 224 else 2048 if k <= 1024 else 131072
    # 2..8 terms, k within the champion lists (128), no prefilter: the seeded launch (doc-id-only rings); the launch that
    # follows it (RCfg<..,4>: queries handed back for pruning) finds an empty list on this corpus
    if 2 <= cls <= 8 and k <= 128:
        # (Zipf workloads: head terms next to rare ones — the seeded launch hands those queries back, the plain kernel of
        # the launch behind it does the work)
        return f"k_search_ring<RCfg<{cls},{kp},4>> (plain kernel over the queries the seeded launch RCfg<{cls},{kp},3> handed back)" \
            if zipf > 0 else f"k_search_ring<RCfg<{cls},{kp},3>>"
    return f"k_search_ring<RCfg<{cls},{kp},0>>"


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def cpu_reference(oix, q_off, q_terms, k, n, threads):
    """Times the restated reference algorithm (Block-max WAND, search.rs:28-282) on the first n queries."""
    n = min(n, len(q_off) - 1)
    sub_off = (q_off[:n + 1] - q_off[0]).astype(np.uint32)
    t0 = time.perf_counter()
    _, _, _, st = oix.search_batch(sub_off, q_terms[q_off[0]:q_off[n]], k, nthreads=threads, wand=True)
    dt = time.perf_counter() - t0
    return n / dt, n, dt, st


DUMP_BYTES = 60_000_000  # --dump-outputs: array bytes in all (under 64 MB with the .npy headers)
DUMP_SEED = 0xB25D0       # --dump-outputs: the row sample when all rows would not fit


def dump_outputs(d, res):
    """--dump-outputs: the result rows a caller of the timed path receives, as DIR/<name>.npy — doc ids and row counts
    as float64 (exact), scores in their own precision (score f32, score64 f64).  Slots past a row's count n are not
    defined by the C ABI and are written as 0.  When every row would take more than DUMP_BYTES, a fixed seeded sample of
    rows is written instead; DIR/query.npy holds the query number of each written row."""
    doc = res["doc"]
    nq, k = doc.shape
    n = res["n"].astype(np.int64)
    arrays = {"doc": (doc, np.float64), "score": (res.get("score"), np.float32),
              "score64": (res.get("score64"), np.float64)}
    arrays = {name: (a, dt) for name, (a, dt) in arrays.items() if a is not None}
    row_bytes = 2 * 8 + k * sum(np.dtype(dt).itemsize for _, dt in arrays.values())   # n + query + the k-wide arrays
    rows = np.arange(nq)
    if nq * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(DUMP_SEED).choice(nq, DUMP_BYTES // row_bytes, replace=False))
    os.makedirs(d, exist_ok=True)
    valid = np.arange(k)[None, :] < n[rows, None]
    for name, (a, dt) in arrays.items():
        np.save(os.path.join(d, f"{name}.npy"), np.where(valid, a[rows], 0).astype(dt))
    np.save(os.path.join(d, "n.npy"), n[rows].astype(np.float64))
    np.save(os.path.join(d, "query.npy"), rows.astype(np.float64))


STRONG_MIX_QUERIES = 400_000   # side leg of the default run: C5's query mix, strong scaling, on the corpus already in HBM


def strong_leg(m, torch, dist, index, stream, q_off_all, q_terms_all, k, rank, world, local_rank, reps):
    """Strong scaling with the gather INSIDE the clock (north_star: "per-GPU results are gathered on the host"):
    one batch, contiguous query shards (shard.shard_queries), every rank answers its shard through the C ABI from
    page-locked host buffers (canonicalise + H2D + kernels), the result rows travel GPU → GPU to rank 0 (one
    dist.gather per array over NCCL/NVLink) and rank 0 copies the whole batch's rows to its page-locked host buffers.
    Host clock, synchronize + barrier on both sides, max over ranks."""
    from vectorchord_bm25_b200 import shard
    nq_total = len(q_off_all) - 1
    sub_off, sub_terms, lo, hi = shard.shard_queries(q_off_all, q_terms_all, rank, world)
    n_local = hi - lo
    dev = torch.device("cuda", local_rank)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    sub_off, sub_terms = pin(sub_off), pin(sub_terms)
    widths = {"doc": 4 * k, "score": 4 * k, "n": 4}
    host = {name: torch.empty((nq_total, w), dtype=torch.uint8, pin_memory=True) for name, w in widths.items()} \
        if rank == 0 else None

    def once():
        t0 = time.perf_counter()
        b = index.prepare(sub_off, sub_terms, k)
        b.run(stream=stream.cuda_stream, timed=False)
        dr = b.device_results()
        parts = {name: torch.as_tensor(shard._DevArray(*dr[name]), device=dev).view(n_local, widths[name])
                 for name in widths}
        stream.synchronize()
        t1 = time.perf_counter()
        g = shard.gather_rows(parts, nq_total, rank, world)
        if rank == 0:
            for name in widths:
                host[name].copy_(g[name], non_blocking=True)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        b.close()
        return t1 - t0, t2 - t1

    once()
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        ts, tg = once()
        if world > 1:
            dist.barrier()
        times.append((time.perf_counter() - t0, ts, tg))
    t = torch.tensor(min(times), dtype=torch.float64, device=dev)   # best repetition of this rank ...
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)                     # ... slowest rank
    total, ts, tg = (float(x) for x in t)
    res = None
    if rank == 0:
        res = {"queries": nq_total, "value": nq_total / total, "unit": "queries/s", "ms": 1e3 * total,
               "search_ms": 1e3 * ts, "gather_and_d2h_ms": 1e3 * tg, "n_gpus": world, "scaling": "strong",
               "h2d_bytes": int(4 * (len(q_off_all) + len(q_terms_all))), "d2h_bytes": nq_total * (8 * k + 4),
               "note": "one batch sharded over the ranks; rows gathered GPU->GPU to rank 0 (dist.gather, NCCL), then "
                       "one D2H of the whole batch on rank 0; host clock, max over ranks",
               "doc_sha": __import__("hashlib").sha256(host["doc"].numpy().tobytes()).hexdigest()[:16]}
    return res


def reference_arm(a, wl, k, cores, cores_how):
    """`--impl reference`: the reference's own CPU algorithm for this path (oracle/: Block-max WAND restatement, the
    reference itself is Rust + pgrx and cannot be built here) on the host cores.  Corpus and queries come from the
    oracle's own generator (bit-identical to the product's, tests/test_abi.py): the product library is never loaded."""
    from oracle import oracle
    oracle.build()
    t0 = time.time()
    oc = oracle.Corpus.synth_bulk(wl["seed"], wl["docs"], wl["vocab"], wl["doclen"], wl["doclen"], wl["zipf"],
                                  nthreads=cores)
    t_gen = time.time() - t0
    q_off, q_terms = oracle.gen_queries_bulk(wl["seed"] + 1000, wl["queries"], wl["vocab"], wl["tmin"], wl["tmax"],
                                             oc.post_off, wl["zipf"])
    nq = wl["queries"]
    oix = oracle.OracleIndex(oc)
    n = min(REF_SAMPLE, nq)
    sub_off, sub_terms = q_off[:n + 1].astype(np.uint32), q_terms[:q_off[n]]
    for _ in range(max(1, a.warmup)):
        oix.search_batch(sub_off, sub_terms, k, nthreads=cores, wand=True)
    t0 = time.perf_counter()
    for _ in range(a.steps):
        od, os_, on, _ = oix.search_batch(sub_off, sub_terms, k, nthreads=cores, wand=True)
    el = time.perf_counter() - t0
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"doc": od, "score64": os_, "n": on})
    qps = n * a.steps / el
    config = {"workload": wl["desc"], "n_docs": wl["docs"], "vocab": wl["vocab"], "doc_len": wl["doclen"],
              "queries_per_gpu_per_step": nq, "terms_per_query": [wl["tmin"], wl["tmax"]], "k": k,
              "zipf_s": wl["zipf"], "postings": int(oc.post_off[-1]), "gen_s": round(t_gen, 1)}
    line = {"impl": "reference", "metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * el / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "cores_how": cores_how, "kind": "port",
                             "sample": f"first {n} of the {nq} queries per step, Block-max WAND restatement of "
                                       f"crates/bm25/src/search.rs (oracle/bm25_oracle.c), one query per OpenMP thread"},
            "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wl = dict(WORKLOADS[a.workload])
    if a.docs:
        wl["docs"] = a.docs
    if a.queries:
        wl["queries"] = a.queries
    if a.k:
        wl["k"] = a.k
    k = wl["k"]
    cores, cores_how = effective_cores()

    if a.impl == "reference":
        if rank == 0:
            reference_arm(a, wl, k, cores, cores_how)
        return  # the reference arm runs on rank 0 only; it never loads the product library
    if world > 1:  # the ranks of one box share its cores: each takes its share for the host side of the C ABI
        os.environ.setdefault("BM25X_HOST_THREADS", str(max(1, cores // world)))
    import _pkg
    m = _pkg.load()
    m.load_library()
    use_gpu = True
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # rank 0 generates the corpus and builds the index; the other ranks receive a replica over NCCL (load time only)
    t0 = time.time()
    corpus = None
    if rank == 0:
        corpus = m.synth_corpus(wl["seed"], wl["docs"], wl["vocab"], wl["doclen"], wl["doclen"], wl["zipf"], cores)
    t_gen = time.time() - t0
    index, t_index, t_repl = None, 0.0, 0.0
    if use_gpu:
        t0 = time.time()
        if rank == 0:
            index = m.Index.from_corpus(corpus, device=local_rank)
        t_index = time.time() - t0
        if world > 1:
            from vectorchord_bm25_b200 import shard
            dist.barrier()
            t0 = time.time()
            index = shard.replicate_index(index, rank, local_rank)
            dist.barrier()
            t_repl = time.time() - t0
        df = index.df()
        post_off_like = np.concatenate([[0], np.cumsum(df, dtype=np.uint64)]).astype(np.uint64)
        n_postings = int(post_off_like[-1])
    else:
        post_off_like, n_postings = corpus.post_off, int(corpus.n_postings)
    strong = wl.get("scaling") == "strong"
    q_all = None
    if strong:
        # strong scaling: ONE batch (same seed on every rank), rank r answers its contiguous shard
        from vectorchord_bm25_b200 import shard
        q_all = m.synth_queries(wl["seed"] + 1000, wl["queries"], wl["vocab"], wl["tmin"], wl["tmax"], post_off_like,
                                wl["zipf"])
        q_off, q_terms, _lo, _hi = shard.shard_queries(q_all[0], q_all[1], rank, world)
        nq, nq_job = _hi - _lo, wl["queries"]
    else:
        # weak scaling: rank r runs its own batch (different query seed per rank) against its replica
        q_off, q_terms = m.synth_queries(wl["seed"] + 1000 + 7919 * rank, wl["queries"], wl["vocab"], wl["tmin"],
                                         wl["tmax"], post_off_like, wl["zipf"])
        nq, nq_job = wl["queries"], world * wl["queries"]
    config = {"workload": wl["desc"], "n_docs": wl["docs"], "vocab": wl["vocab"], "doc_len": wl["doclen"],
              "queries_per_gpu_per_step": nq, "terms_per_query": [wl["tmin"], wl["tmax"]], "k": k,
              "zipf_s": wl["zipf"], "postings": n_postings,
              "parallelism": f"queries sharded over {world} GPU(s), index replicated (NCCL broadcast at load)",
              "l2": "index (8 B/posting) is far larger than the 126 MB L2; no flush needed",
              "k_note": "BASELINE.json's metric says top-10, its configs[2] words the same 10M-doc case as top-100: "
                        "`value` is top-10, the `top100` object is the same batch at k=100",
              "gen_s": round(t_gen, 1), "index_build_s": round(t_index, 1), "replicate_s": round(t_repl, 2)}

    info = index.info()
    if a.no_prune:
        index.set_option("prune", 0)

    cpu_baseline = None
    if rank == 0 and a.gpus == 1 and not a.no_cpu_baseline:
        from oracle import oracle
        oracle.build()
        oc = oracle.Corpus(corpus.n_docs, corpus.doc_len, corpus.n_terms, corpus.post_off, corpus.post_doc,
                           corpus.post_tf)
        oix = oracle.OracleIndex(oc)
        qps, n, dt, st = cpu_reference(oix, q_off, q_terms, k, REF_SAMPLE, cores)
        qps1, n1, dt1, _ = cpu_reference(oix, q_off, q_terms, k, max(200, REF_SAMPLE // 20), 1)
        cpu_baseline = {"value": qps, "unit": "queries/s", "cores": cores, "cores_how": cores_how, "kind": "port",
                        "sample": f"first {n} of the {nq} queries ({dt:.1f} s), Block-max WAND restatement of "
                                  f"crates/bm25/src/search.rs (oracle/bm25_oracle.c), one query per OpenMP thread",
                        "single_thread_qps": qps1, "single_thread_sample": n1,
                        "wand_postings_touched_frac": st.postings_touched / max(1, sum(
                            int(corpus.post_off[t + 1] - corpus.post_off[t]) for t in q_terms[:q_off[n]]))}
        del oix, oc

    stream = torch.cuda.Stream()  # a real (non-default) stream: the handle is passed through the C ABI
    torch.cuda.set_stream(stream)
    batch = index.prepare(q_off, q_terms, k)
    # ---- value: prepared batch resident in HBM, kernels only ----
    sampler = ClockSampler(local_rank)   # started before the warm-up: nvidia-smi needs a moment to come up
    sampler.start()
    for _ in range(a.warmup):
        batch.run(stream=stream.cuda_stream, timed=False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(a.steps):
        batch.run(stream=stream.cuda_stream, timed=False)
    ev1.record(stream)
    torch.cuda.synchronize()
    ms_total = ev0.elapsed_time(ev1)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, batch.fetch(want_f64=True))
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    st = batch.run(stream=stream.cuda_stream, timed=True)  # per-launch kernel time + algorithmic bytes
    kernel_ms_samples = [batch.run(stream=stream.cuda_stream, timed=True).kernel_ms for _ in range(3)]
    res_dev = batch.fetch(want_f64=False)

    # ---- e2e: host buffers in, host buffers out, every step ----
    def pinned(shape, dtype, src=None):  # page-locked host memory, as the bench contract asks for the e2e leg
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        buf = torch.empty(max(n, 1), dtype=torch.uint8, pin_memory=True).numpy()[:n].view(dtype).reshape(shape)
        if src is not None:
            buf[...] = src
        return buf

    out = {"doc": pinned((nq, k), np.uint32), "score": pinned((nq, k), np.float32), "score64": None,
           "payload": None, "n": pinned((nq,), np.uint32)}
    q_off, q_terms = pinned(q_off.shape, np.uint32, q_off), pinned(q_terms.shape, np.uint32, q_terms)
    index.search_batch(q_off, q_terms, k, want_f64=False, out=out)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_steps = a.steps
    for _ in range(e2e_steps):
        index.search_batch(q_off, q_terms, k, want_f64=False, out=out)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop()
    assert np.array_equal(out["doc"], res_dev["doc"]) and np.array_equal(out["n"], res_dev["n"])

    # ---- the same corpus and queries at top-100 (BASELINE.json configs[2] words the 10M-doc case as top-100) ----
    top100 = None
    if world == 1 and k != 100 and a.workload == "c3":
        b100 = index.prepare(q_off, q_terms, 100)
        for _ in range(a.warmup):
            b100.run(stream=stream.cuda_stream, timed=False)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(a.steps):
            b100.run(stream=stream.cuda_stream, timed=False)
        e1.record(stream)
        torch.cuda.synchronize()
        ms100 = e0.elapsed_time(e1) / a.steps
        top100 = {"value": nq / (ms100 / 1e3), "unit": "queries/s", "ms_per_step": ms100, "k": 100}
        b100.close()

    # ---- strong scaling, gather to rank 0's host inside the clock (collective: every rank takes part) ----
    strong_obj = None
    if strong:
        strong_obj = strong_leg(m, torch, dist, index, stream, q_all[0], q_all[1], k, rank, world, local_rank, a.steps)
    elif a.workload == "c3" and not a.no_strong:
        qs = m.synth_queries(0xB25C0DE0 + 5 + 1000, STRONG_MIX_QUERIES, wl["vocab"], 1, 8, post_off_like, 0.0)
        strong_obj = strong_leg(m, torch, dist, index, stream, qs[0], qs[1], k, rank, world, local_rank, a.steps)
        if strong_obj:
            strong_obj["workload"] = (f"C5's query mix (1-8 terms, seed of configs[4]) on THIS corpus ({wl['docs']} docs): "
                                      f"one batch of {STRONG_MIX_QUERIES} queries; the 50M-doc corpus itself: --workload c5")

    t = torch.tensor([ms_total, 1e3 * e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms = float(t[0]), float(t[1])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    ms_step = ms_total / a.steps
    value = nq_job / (ms_step / 1e3)
    e2e_value = nq_job * e2e_steps / (e2e_ms / 1e3)
    peak, peak_src = hbm_peak()
    kms = statistics.mean(kernel_ms_samples)
    # algorithmic bytes (SURVEY §8d): 8 B per posting touched + 8 B per result slot + 16 B per query term.  With pruning
    # only the postings actually streamed count (never more than the exhaustive figure: chunk tails are loaded twice).
    fetched = int(st.postings_fetched)
    touched = min(int(st.postings), fetched) if fetched else int(st.postings)
    bytes_algo = 8 * touched + (int(st.bytes_algo) - 8 * int(st.postings))
    achieved = bytes_algo / (kms / 1e3) / 1e9
    h2d = 4 * (len(q_off) + len(q_terms) + nq)       # class-grouped ids + offsets + terms
    d2h = nq * k * 8 + nq * 4
    line = {"metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "f32 filter + f64 exact re-score (u32 doc ids)", "data": "synthetic", "config": config,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None if a.no_prune else measured_traffic(a.workload, nq, k), "peak_source": peak_src, "kernel": kernel_name(wl["tmax"], k, wl["zipf"]),
                         "kernel_ms": kms, "algorithmic_bytes_per_launch": bytes_algo,
                         "postings_exhaustive": int(st.postings), "postings_streamed": fetched,
                         "pruning": "off" if a.no_prune else "on",
                         "note": "achieved = ALGORITHMIC bytes (8 B per posting, SURVEY 8d) / kernel time; the seeded kernel streams "
                                 "doc ids only (4 B per posting), so `traffic` (DRAM bytes of the same launch, committed ncu "
                                 "capture) is about half of that",
                         "skipped_frac": max(0.0, 1.0 - touched / max(1, int(st.postings)))},
            "cpu_baseline": cpu_baseline,
            "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / e2e_steps, "note": "bm25x_search_batch: host q_off/q_terms in, "
                    "host doc ids + f32 scores + counts out (page-locked host buffers)"},
            "top100": top100, "strong_scaling": strong_obj, "gpu_launches": int(st.launches) * a.steps, "clocks": clocks,
            "index": {"device_bytes": int(info.device_bytes), "blocks": int(info.n_blocks), "avgdl": info.avgdl}}
    if strong:   # the job's end-to-end number is the sharded batch WITH the gather to rank 0's host
        line["e2e"] = {"value": strong_obj["value"], "unit": "queries/s", "h2d_bytes_per_step": strong_obj["h2d_bytes"],
                       "d2h_bytes_per_step": strong_obj["d2h_bytes"], "ms_per_step": strong_obj["ms"],
                       "note": strong_obj["note"], "per_rank_search_batch_qps": e2e_value}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
