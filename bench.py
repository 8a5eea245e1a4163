#!/usr/bin/env python
"""ehb200 benchmark — batched k-NN over the HNSW graph at the north-star configurations.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ehb200|reference] [--workload auto|c2|c3|...]
                  [--dump-outputs DIR]

Default workload ("auto"): ONE GPU -> BASELINE.json configs[2] (C3: N=10M d=768 Q=10k k=10 ef=128 InnerProduct,
the north-star target, 30.7 GB of vectors on one B200); N > 1 GPUs -> configs[4] (C5: d=128 Q=10k k=100 ef=256
cosine, range-sharded, 12.5M points per GPU = 100M at 8 GPUs).  A step = one pass of the hot path over one
batch of Q synthetic queries.
  value        queries/s over the WHOLE index (Q / step time), index and queries resident in HBM, device-timed
               with CUDA events on the launch stream, L2 flushed between steps, max over ranks
  e2e          the same through the host entry point (ehb_index_search): pinned host queries -> H2D -> walk ->
               D2H of labels / distances / counts, all inside the timed region
  roofline     algorithmic bytes of the walk kernel (hnswlib hop / distance-evaluation counters of that very
               launch, SURVEY.md §8d) / its CUDA-event duration, against the measured HBM copy bandwidth
  cpu_baseline the CPU oracle (hnswlib restatement) walking the SAME graph with the SAME queries on the host
               cores of this box: threads pinned one per CPU, best and median of 5 passes (rank 0, N=1 only)
  parity       at a stated sub-sample N' of the same data: recall@k of the oracle on its OWN CPU-built graph
               (= the reference's behaviour), of the GPU-built graph walked by the GPU, and of the GPU-built
               graph walked by the oracle, all at the same ef, against exact ground truth
--impl reference times the oracle end to end on the host cores (its own CPU-built graph over a time-bounded
prefix of the same base set).

Multi-GPU (torchrun, one rank per GPU): the index is range-sharded, every rank searches all Q queries over its
own shard, the per-shard top-k lists meet in ONE exchange step (default: the library's peer-memory exchange —
one push + flag + merge kernel per rank over NVLink, no collective; --exchange nccl: one ncclAllGather + merge
kernel).  Weak scaling: the shard size per GPU is fixed, so the index grows with N; `value` stays Q / step
time (queries answered over N_total points) and `shard_searches_per_s` = N x that is the aggregate of
shard-level searches.
"""
import argparse
import ctypes as C
import json
import os
import platform
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: N per GPU, d, Q, k, ef, metric
    "c2": dict(N=1_000_000, d=128, Q=1000, k=10, ef=64, metric="l2",
               desc="HNSW N=1M d=128 Q=1k k=10 ef=64 L2 (BASELINE.json configs[1])"),
    "c2s": dict(N=100_000, d=128, Q=1000, k=10, ef=64, metric="l2", desc="C2 at N=100k (smoke)"),
    "c3s": dict(N=1_000_000, d=768, Q=10000, k=10, ef=128, metric="ip",
                desc="C3 shape at N=1M: d=768 Q=10k k=10 ef=128 InnerProduct"),
    "c3": dict(N=10_000_000, d=768, Q=10000, k=10, ef=128, metric="ip",
               desc="HNSW N=10M d=768 Q=10k k=10 ef=128 InnerProduct (BASELINE.json configs[2])"),
    "c5s": dict(N=1_000_000, d=128, Q=10000, k=100, ef=256, metric="cosine",
                desc="C5 shape at N=1M per GPU: d=128 Q=10k k=100 ef=256 cosine"),
    "c5": dict(N=12_500_000, d=128, Q=10000, k=100, ef=256, metric="cosine",
               desc="HNSW N=100M d=128 Q=10k k=100 ef=256 cosine range-sharded over 8 GPUs = 12.5M per GPU "
                    "(BASELINE.json configs[4]; with fewer ranks the total shrinks accordingly)"),
    # brute force on the bf16 tensor-core path (tcgen05 GEMM + fp32 re-rank); recall is measured against the
    # exact fp32 path
    "c4s": dict(N=1_000_000, d=768, Q=4096, k=100, ef=0, metric="ip", brute="bf16",
                desc="brute force N=1M d=768 Q=4096 k=100 bf16 tensor-core path (C4 shape at N=1M)"),
    "c4": dict(N=10_000_000, d=768, Q=4096, k=100, ef=0, metric="ip", brute="bf16",
               desc="brute-force N=10M d=768 Q=4096 k=100 bf16 tensor-core GEMM path (BASELINE.json configs[3])"),
}
BASE_SEED, QUERY_SEED = 1234, 4321  # SURVEY.md §8d
CHUNK = 1 << 20                     # rows per generated chunk (SURVEY.md §8d: chunks of 1M rows)

DIST = "gaussian"   # --dist gmm: report-only secondary distribution (SURVEY.md §8d): 1024-centre GMM, sigma 0.3


def gen_chunks(n, d, seed):
    """Yields (first_row, rows[<=1M][d]) of the prescribed stream: numpy default_rng(seed) (PCG64)
    standard_normal float32, generated in chunks of 1M rows; a prefix of the stream is the same data."""
    rng = np.random.default_rng(seed)
    centres = np.random.default_rng(99).standard_normal((1024, d), dtype=np.float32) if DIST == "gmm" else None
    for i in range(0, n, CHUNK):
        m = min(CHUNK, n - i)
        x = rng.standard_normal((m, d), dtype=np.float32)
        if centres is not None:
            x *= np.float32(0.3)
            x += centres[rng.integers(0, 1024, m)]
        yield i, x


def gen(n, d, seed):
    out = np.empty((n, d), np.float32)
    for i, x in gen_chunks(n, d, seed):
        out[i:i + x.shape[0]] = x
    return out


def prefetched(it, depth=2):
    """Runs a generator in a background thread (numpy releases the GIL while filling)."""
    import queue

    qu, end = queue.Queue(maxsize=depth), object()

    def run():
        try:
            for item in it:
                qu.put(item)
        finally:
            qu.put(end)

    threading.Thread(target=run, daemon=True).start()
    while True:
        item = qu.get()
        if item is end:
            return
        yield item


def shared_config(wl, world):
    """`config` of a bench line: identical for the GPU arm and the reference arm of one workload / rank count."""
    return {"workload": wl["desc"], "N_per_gpu": wl["N"], "N_total": wl["N"] * world, "d": wl["d"], "Q": wl["Q"],
            "k": wl["k"], "ef": wl["ef"], "metric_space": wl["metric"], "M": 16, "ef_construction": 200}


def recall_at_k(found, truth):
    k = truth.shape[1]
    return float(np.mean([len(set(a.tolist()) & set(b.tolist())) / k for a, b in zip(found, truth)]))


def dump_outputs(out_dir, labels, dists, counts):
    """Writes the last timed step's result as <out_dir>/{labels,distances,counts}.npy so that two builds can be
    compared output for output.  Labels go through int64 (NO_LABEL -> -1) to float64, exact below 2^53; the
    largest workload (C5: Q=10k, k=100) writes about 12 MB, so every array is stored whole."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "labels.npy"), np.asarray(labels).view(np.int64).astype(np.float64))
    np.save(os.path.join(out_dir, "distances.npy"), np.asarray(dists, dtype=np.float32))
    np.save(os.path.join(out_dir, "counts.npy"), np.asarray(counts).astype(np.float32))


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.p = gpu_index, [], None

    def start(self):
        for q in (self.Q, self.Q.replace("clocks_event_reasons", "clocks_throttle_reasons")):
            try:
                probe = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}",
                                        "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=20)
                if probe.returncode != 0 or "not a valid" in (probe.stdout + probe.stderr).lower():
                    continue
                self.p = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}",
                                           "--format=csv,noheader,nounits", "-lms", "20"],
                                          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                threading.Thread(target=self._read, daemon=True).start()
                time.sleep(0.3)
                return
            except Exception:
                self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.p:
            self.p.terminate()
            try:
                self.p.wait(timeout=2)
            except Exception:
                self.p.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                   r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_cpus():
    try:
        return sorted(os.sched_getaffinity(0))
    except Exception:
        return list(range(os.cpu_count() or 1))


def host_info():
    model = platform.processor() or ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    load = None
    try:
        load = os.getloadavg()[0]
    except Exception:
        pass
    return {"cpu_model": model, "nproc": len(host_cpus()), "loadavg_1m_before": load,
            "cgroup_cpu_limit": cgroup_cpu_limit()}


def cgroup_cpu_limit():
    """CPUs' worth of quota the container may use (None = unlimited / unknown)."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        return None if q == "max" else float(q) / float(per)
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / per
    except Exception:
        return None


def calibrate_threads(run, cores, sample_desc):
    """The CPU arm gets the thread count that serves it best on THIS box: a short sample is timed at
    nproc, nproc/2, ... (oversubscribed hyper-threads, NUMA and container CPU quotas make "all logical CPUs"
    the slowest choice on some hosts — round 1 saw 4.4x between two boxes).  run(threads) -> seconds."""
    lim = cgroup_cpu_limit()
    cand = {cores, cores // 2, cores // 4, cores // 8, 32, 16, 8}
    if lim:
        cand |= {int(round(lim)), int(round(lim * 1.5)), int(round(lim * 2))}   # a CPU quota: stay near it
    cand = sorted({c for c in cand if 1 <= c <= cores}, reverse=True)
    sweep = {}
    for c in cand:
        run(c)                      # warm
        sweep[c] = min(run(c), run(c))
    best = min(sweep, key=sweep.get)
    return best, {"sample": sample_desc, "seconds_by_threads": {str(k): round(v, 4) for k, v in sweep.items()}}


def timed_passes(fn, passes=5, min_passes=3, budget_s=30.0):
    """Best and median wall time of repeated passes (perf_counter), bounded by a time budget."""
    fn()  # warm
    ts, t_all = [], time.perf_counter()
    while len(ts) < passes and (len(ts) < min_passes or time.perf_counter() - t_all < budget_s):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return min(ts), float(np.median(ts)), len(ts)


def oracle_build_prefix(orc, wl, budget_s, cores, cap, tune=None):
    """CPU construction (the reference's path: one addPoint per row, here multi-threaded) over as long a prefix
    of the prescribed base stream as the time budget allows.  Returns (oracle, rows kept, seconds).  With
    `tune` (a dict), the thread count is calibrated on the first 20k points and recorded there."""
    d = wl["d"]
    o = orc.OracleHNSW(d, wl["metric"], cap)
    kept, built, t0 = [], 0, time.perf_counter()
    step = 20000
    threads = cores
    for first, x in gen_chunks(cap, d, BASE_SEED):
        off = 0
        while off < x.shape[0] and time.perf_counter() - t0 < budget_s:
            m = min(step, x.shape[0] - off)
            o.add(x[off:off + m], np.arange(built, built + m, dtype=np.uint64), threads=threads)
            built += m
            off += m
            if tune is not None and "threads" not in tune:
                qs = gen(2048, d, QUERY_SEED)
                t_cal = time.perf_counter()

                def run(c):
                    t1 = time.perf_counter()
                    o.search(qs, wl["k"], ef=wl["ef"], threads=c)
                    return time.perf_counter() - t1

                threads, tune["sweep"] = calibrate_threads(run, cores, f"2048 queries on the first {built} points")
                tune["threads"] = threads
                t0 += time.perf_counter() - t_cal      # calibration is not construction time
        kept.append(x[:off])
        if off < x.shape[0] or time.perf_counter() - t0 >= budget_s:
            break
    return o, np.concatenate(kept) if kept else np.empty((0, d), np.float32), time.perf_counter() - t0


# ---------------------------------------------------------------------------------------------
def run_reference(args, wl):
    """The reference arm: the CPU oracle (hnswlib restatement; oracle/_ref cannot exist because the hnswlib
    headers are not in /root/reference) with every host thread pinned, its own CPU-built graph."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc

    orc.set_thread_pinning(True)
    cpus = host_cpus()
    cores = len(cpus)
    info = host_info()
    N, d, Q, k, ef = wl["N"], wl["d"], wl["Q"], wl["k"], wl["ef"]
    brute = bool(wl.get("brute"))
    q = gen(Q, d, QUERY_SEED)
    if brute:
        ns, qs = min(N, 200_000), min(Q, 256)
        base = gen(ns, d, BASE_SEED)
        for _ in range(max(args.warmup, 1)):
            orc.bruteforce(base, q[:qs], k, wl["metric"], threads=cores)
        steps_ms = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            labels, dists = orc.bruteforce(base, q[:qs], k, wl["metric"], threads=cores)
            steps_ms.append((time.perf_counter() - t0) * 1e3)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, labels, dists, np.full(qs, min(k, ns)))
        med = float(np.median(steps_ms)) * 1e-3
        best = min(steps_ms) * 1e-3
        qps = qs / med * (ns / N)
        sample = (f"oracle exact scan of {qs} queries over the first {ns} base vectors on {cores} pinned threads, "
                  f"scaled by {ns}/{N}; median of {args.steps} steps")
        built, rec, t_build = ns, 1.0, 0.0
    else:
        tune = {}
        o, base, t_build = oracle_build_prefix(orc, wl, args.ref_build_budget, cores, min(N, args.ref_max_points), tune)
        built = base.shape[0]
        cores = tune.get("threads", cores)
        info["thread_sweep"] = tune.get("sweep")
        o.set_ef(ef)
        t0 = time.perf_counter()
        o.search(q, k, ef=ef, threads=cores)
        t_one = time.perf_counter() - t0
        # a step is a bounded sample of the workload: all Q queries unless K steps of that would run past ~150 s
        Qs = Q if t_one * (args.steps + args.warmup) <= 150.0 else max(256, int(Q * 150.0 / (t_one * (args.steps + args.warmup))))
        qstep = q[:Qs]
        for _ in range(max(args.warmup, 1)):
            o.search(qstep, k, ef=ef, threads=cores)
        steps_ms = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            labels, dists, counts = o.search(qstep, k, ef=ef, threads=cores)
            steps_ms.append((time.perf_counter() - t0) * 1e3)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, labels, dists, counts)
        med = float(np.median(steps_ms)) * 1e-3
        best = min(steps_ms) * 1e-3
        gt, _ = orc.bruteforce(base, q[:200], k, wl["metric"], threads=cores)
        rec = recall_at_k(labels[:200], gt)
        qps = Qs / med
        sample = (f"graph built on the CPU over the first {built} of {N} base vectors in {t_build:.0f}s ({cores} pinned "
                  f"threads); each step = {Qs} of the {Q} queries at ef={ef}; value = queries of a step / median step "
                  f"time of {args.steps} steps")
    line = {
        "impl": "reference", "metric": "k-NN queries/s", "value": qps, "unit": "queries/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": med * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the same `config` dict as the GPU arm prints for this workload and rank count; arm-specific facts
        # (the sub-sample the CPU graph was built over) go to `details`
        "config": shared_config(wl, max(args.gpus, 1)),
        "details": {"N_sample": built, "graph": "CPU-built by the oracle over a time-bounded prefix of the same base stream"},
        "recall_at_k": rec,
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample,
                         "best_queries_per_s": (Qs if not brute else qs * ns / N) / best, "build_s": round(t_build, 1),
                         "step_ms_min_median_max": [min(steps_ms), float(np.median(steps_ms)), max(steps_ms)],
                         "pinned": True, **info},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
def parity_block(ehb, orc, wl, budget_s, cores, device):
    """Recall parity at a matched sub-sample N' (SURVEY.md §8d parity gate), same data, same queries, same ef."""
    d, k, ef, metric = wl["d"], wl["k"], wl["ef"], wl["metric"]
    nq = 1000
    q = gen(nq, d, QUERY_SEED)
    tune = {}
    o, base, t_cpu = oracle_build_prefix(orc, wl, budget_s, cores, min(wl["N"], 1_000_000), tune)
    cores = tune.get("threads", cores)
    n1 = base.shape[0]
    ix = ehb.NativeIndex(d, metric=metric, capacity=n1, device=device)
    ix.add(base)
    t0 = time.perf_counter()
    ix.build()
    t_gpu = time.perf_counter() - t0
    gt, _, _ = ix.search_bruteforce(q, k)
    ol, od, _ = o.search(q, k, ef=ef, threads=cores)
    al, _, _ = ix.search(q, k, ef=ef)       # automatic warps per query (what a batch of this size gets)
    ix.set_search_width(1)                  # one warp per query = hnswlib's expansion order: the identity check
    gl, gd, _ = ix.search(q, k, ef=ef)
    o2 = orc.OracleHNSW(d, metric, n1)
    o2.import_graph(ix.export_graph())
    xl, xd, _ = o2.search(q, k, ef=ef, threads=cores)
    same = gl == xl
    rel = float(np.max(np.abs(gd[same] - xd[same]) / np.maximum(np.abs(xd[same]), 1e-6))) if same.any() else None
    out = {"N_prime": n1, "queries": nq, "ef": ef, "k": k,
           "recall_oracle_built_oracle_walk": recall_at_k(ol, gt),
           "recall_gpu_built_gpu_walk": recall_at_k(gl, gt),
           "recall_gpu_built_gpu_walk_auto_width": recall_at_k(al, gt),
           "recall_gpu_built_oracle_walk": recall_at_k(xl, gt),
           "ids_equal_gpu_vs_oracle_walk_same_graph": float(same.mean()),
           "max_rel_dist_err_same_graph": rel,
           "cpu_build_s": round(t_cpu, 1), "gpu_build_s": round(t_gpu, 2),
           "gate": "recall(GPU) >= recall(oracle) - 0.005 at the same ef (two builds of the oracle itself differ by "
                   "about that much); ids of the two walks on the same graph equal; |dist - oracle dist| <= 1e-4 relative"}
    out["gate_passed"] = bool(out["recall_gpu_built_gpu_walk"] >= out["recall_oracle_built_oracle_walk"] - 0.005 and
                              out["ids_equal_gpu_vs_oracle_walk_same_graph"] >= 0.995 and (rel is None or rel <= 1e-4))
    del ix, o, o2
    return out


def run_ehb(args, wl):
    import torch
    import torch.distributed as dist

    import embeddinghub_b200 as ehb
    from embeddinghub_b200._native import check, lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; ehb200 has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    N, d, Q, k, ef, metric = wl["N"], wl["d"], wl["Q"], wl["k"], wl["ef"], wl["metric"]
    brute = bool(wl.get("brute"))
    steps, warmup = args.steps, max(args.warmup, 3)
    t_setup0 = time.time()

    # ---- build the shard (setup, untimed): generated chunk by chunk, added as it comes -----------------
    ix = ehb.NativeIndex(d, metric=metric, capacity=N, device=local)
    if args.walk_prefetch >= 0:
        ix.set_option("walk_prefetch", args.walk_prefetch)
    t0 = time.time()
    for first, x in prefetched(gen_chunks(N, d, BASE_SEED + 1000 * rank)):
        ix.add(x, np.arange(rank * N + first, rank * N + first + x.shape[0], dtype=np.uint64))  # global labels
    t_ingest = time.time() - t0
    t1 = time.time()
    if not brute:
        ix.build()
    t_build = time.time() - t1
    nbatch = warmup + steps
    qsets = [gen(Q, d, QUERY_SEED + i) for i in range(min(nbatch, 8))]  # rotated query batches
    stream = torch.cuda.Stream()  # a real (non-default) stream: handle 0 would mean "the index's own stream"
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream
    dq = [torch.from_numpy(x).cuda() for x in qsets]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    from embeddinghub_b200.sharded import ShardedSearcher

    searcher = ShardedSearcher(ix, world, local, exchange=args.exchange)
    last = {}

    def step_dev(i):
        # per-shard walk -> (world > 1: ONE exchange step: push + flag + merge kernel over peer memory)
        last["l"], last["d"], last["c"] = searcher.search_dev(dq[i % len(dq)], k, ef, sptr, bruteforce=brute,
                                                              precision=1 if brute else 0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident-input timing: K steps, L2 flushed between steps, device events --------------------------
    for i in range(warmup):
        step_dev(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    kernel_ms, alg_bytes, counters = [], [], []
    barrier()
    for i in range(steps):
        flush.zero_()            # untimed: evicts L2 between timed iterations
        ev[i][0].record(stream)
        step_dev(warmup + i)
        ev[i][1].record(stream)
        if i < 4 or i == steps - 1:   # kernel duration + counters of THIS launch (syncs on its events)
            ev[i][1].synchronize()
            kernel_ms.append(ix.last_kernel_ms())
            s_i = ix.stats()
            alg_bytes.append(0 if brute else s_i["algorithmic_bytes"])
            counters.append(s_i)
    barrier()
    dev_ms = sum(a.elapsed_time(b) for a, b in ev) / steps
    clocks = sampler.stop() if rank == 0 else None
    st = counters[-1]
    kernel_name = ix.last_kernel_name()
    labels_dev = last["l"].cpu().numpy().view(np.uint64).copy()
    if args.dump_outputs and rank == 0:     # every rank holds the same merged top-k
        dump_outputs(args.dump_outputs, labels_dev, last["d"].cpu().numpy(), last["c"].cpu().numpy())

    # the local shard alone (no exchange), same steps: lets a reader separate the walk from the exchange
    shard_ms = None
    if world > 1:
        solo = ShardedSearcher(ix, 1, local)
        for i in range(2):
            solo.search_dev(dq[i % len(dq)], k, ef, sptr, bruteforce=brute, precision=1 if brute else 0)
        barrier()
        ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(min(steps, 10))]
        for i, (a, b) in enumerate(ev2):
            flush.zero_()
            a.record(stream)
            solo.search_dev(dq[(warmup + i) % len(dq)], k, ef, sptr, bruteforce=brute, precision=1 if brute else 0)
            b.record(stream)
        barrier()
        shard_ms = sum(a.elapsed_time(b) for a, b in ev2) / len(ev2)

    # ---- end to end through the host entry point (pinned host buffers) ------------------------------------
    hq = [torch.from_numpy(x).pin_memory() for x in qsets]
    hl = torch.empty((Q, k), dtype=torch.int64).pin_memory()
    hd = torch.empty((Q, k), dtype=torch.float32).pin_memory()
    hc = torch.empty(Q, dtype=torch.int32).pin_memory()
    L, h = lib(), ix._h

    dq_e2e = torch.empty((Q, d), dtype=torch.float32, device="cuda")

    def step_e2e(i):
        if world == 1 and brute:
            check(L.ehb_index_search_bruteforce(h, Q, C.c_void_p(hq[i % len(hq)].data_ptr()), k, 1,
                                                C.c_void_p(hl.data_ptr()), C.c_void_p(hd.data_ptr()),
                                                C.c_void_p(hc.data_ptr())))
        elif world == 1:
            # the public host entry point: host queries in, host labels/distances/counts out
            check(L.ehb_index_search(h, Q, C.c_void_p(hq[i % len(hq)].data_ptr()), k, ef,
                                     C.c_void_p(hl.data_ptr()), C.c_void_p(hd.data_ptr()), C.c_void_p(hc.data_ptr())))
        else:
            # sharded: H2D of the queries, per-shard walk, exchange + merge, D2H of the merged result
            dq_e2e.copy_(hq[i % len(hq)], non_blocking=True)
            ml_, md_, mc_ = searcher.search_dev(dq_e2e, k, ef, sptr, bruteforce=brute, precision=1 if brute else 0)
            hl.copy_(ml_, non_blocking=True)
            hd.copy_(md_, non_blocking=True)
            hc.copy_(mc_, non_blocking=True)
            stream.synchronize()

    for i in range(warmup):
        step_e2e(i)
    barrier()
    t_e2e = 0.0
    for i in range(steps):
        flush.zero_()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0e = time.perf_counter()
        step_e2e(warmup + i)     # returns after the D2H of the results completed
        t_e2e += time.perf_counter() - t0e
    e2e_ms = t_e2e / steps * 1e3

    # max over ranks
    if world > 1:
        t = torch.tensor([dev_ms, e2e_ms, shard_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms, shard_ms = t[0].item(), t[1].item(), t[2].item()

    # ---- recall vs exact ground truth (own kernels: exact fp32 brute force, same exchange + merge) -----------
    qi = (warmup + steps - 1) % len(dq)
    nrec = min(Q, args.recall_queries)
    gl_t, _, _ = searcher.search_dev(dq[qi][:nrec].contiguous(), k, ef, sptr, bruteforce=True)
    torch.cuda.synchronize()
    gt_l = gl_t.cpu().numpy().view(np.uint64).copy()
    rec = recall_at_k(labels_dev[:nrec], gt_l)
    timed_out = 0
    if world > 1 and searcher.exchange == "peer":
        tmo = C.c_uint32()
        check(L.ehb_exchange_timed_out(searcher._ex, C.byref(tmo)))
        timed_out = tmo.value

    if rank != 0:
        if world > 1:
            dist.barrier()          # rank 0 may still run its CPU legs
            dist.destroy_process_group()
        return

    # ---- roofline of the walk kernel ------------------------------------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peaks = json.load(open(peaks_path)) if os.path.exists(peaks_path) else {}
    if peaks:
        peak, peak_src = peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    k_ms = float(np.mean(kernel_ms))
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "walk_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        ent = tj.get(args.workload)
        if isinstance(ent, dict):
            traffic, traffic_src = ent.get("dram_bytes_per_launch"), ent.get("source")
        elif ent is not None:
            traffic = ent
    if brute:
        tpeak = peaks.get("bf16_tflops_sustained", 1400.0)
        flops = 2.0 * Q * N * d
        ach = flops / (k_ms * 1e-3) / 1e12
        roofline = {"bound": "tensor", "achieved": ach, "peak": tpeak, "unit": "TFLOP/s", "frac": ach / tpeak,
                    "traffic": traffic, "peak_source": "measured sustained cuBLAS bf16 (MEASURED_PEAKS.json)"
                    if peaks else "fallback (B200_PROFILING.md)", "kernel": "bf16_topk_gemm_kernel (persistent tcgen05 "
                    "GEMM, selection fused into the epilogue) + compaction + fp32 re-rank: the whole brute-force "
                    "pipeline is timed", "kernel_ms": k_ms, "flops_per_launch": flops}
    else:
        achieved = float(np.mean(alg_bytes)) / (k_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "kernel": kernel_name,
                    "kernel_ms": k_ms, "algorithmic_bytes_per_launch": float(np.mean(alg_bytes)),
                    "evals_per_query": st["dist_evals"] / Q, "hops_per_query": st["hops_base"] / Q,
                    "visited_overflow_queries": st["visited_overflow"]}

    # ---- CPU legs (rank 0): baseline on the SAME graph (N=1) and the recall parity block --------------------
    cpu, parity = None, None
    if not args.no_cpu_baseline:
        from oracle import oracle as orc

        orc.set_thread_pinning(True)
        cores = len(host_cpus())
        info = host_info()
    if world == 1 and not args.no_cpu_baseline and brute:
        ns, qs = min(N, 200_000), min(Q, 256)
        base_s = gen(ns, d, BASE_SEED)
        best, med, passes = timed_passes(lambda: orc.bruteforce(base_s, qsets[qi][:qs], k, metric, threads=cores), 3, 2, 60)
        cpu = {"value": qs / med * (ns / N), "unit": "queries/s", "cores": cores, "kind": "port", "pinned": True, **info,
               "sample": f"oracle exact scan (hnswlib BruteforceSearch semantics) of {qs} queries over the first {ns} base "
                         f"vectors on {cores} pinned threads, scaled by {ns}/{N} to the full base set; median of {passes}"}
    elif world == 1 and not args.no_cpu_baseline:
        g = ix.export_graph()
        o = orc.OracleHNSW(d, metric, N)
        o.import_graph(g)
        del g
        qq = qsets[qi]  # the oracle normalises cosine queries itself
        res = {}

        def cal(c):
            t1 = time.perf_counter()
            o.search(qq[:1024], k, ef=ef, threads=c)
            return time.perf_counter() - t1

        cores, info["thread_sweep"] = calibrate_threads(cal, cores, f"1024 of the {Q} queries on the full graph")

        def one_pass():
            res["l"] = o.search(qq, k, ef=ef, threads=cores)[0]

        best, med, passes = timed_passes(one_pass, 5, 3, 40)
        cl = res["l"]
        # hnswlib's own counters for the same graph and queries (metric_hops / metric_distance_computations):
        # the roofline numerator WITHOUT anything the GPU walk adds (re-evaluations after a visited-table
        # overflow, speculative expansions of the team walk)
        o.metrics(reset=True)
        one_pass()
        om = o.metrics(reset=True)
        clean_bytes = om["hops_upper"] * 4.0 * 16 + om["hops0"] * 8.0 * 16 + om["evals"] * 4.0 * d + Q * 4.0 * d
        roofline["hnswlib_counters"] = {
            "evals_per_query": om["evals"] / Q, "hops_per_query": om["hops0"] / Q,
            "algorithmic_bytes_per_launch": clean_bytes,
            "achieved": clean_bytes / (k_ms * 1e-3) / 1e9, "frac": clean_bytes / (k_ms * 1e-3) / 1e9 / peak,
            "note": "same kernel duration, bytes from the oracle's counters on the same graph and queries"}
        t0c = time.perf_counter()
        o.search(qq[:max(Q // 20, 50)], k, ef=ef, threads=1)
        cpu_1t = max(Q // 20, 50) / (time.perf_counter() - t0c)
        # "reference as shipped": the reference never calls setEf, so it runs ef = max(10, k) (index.cc:14-15,41)
        ef_ship = max(10, k)

        def ship_pass():
            res["s"] = o.search(qq, k, ef=ef_ship, threads=cores)[0]

        sbest, smed, _ = timed_passes(ship_pass, 3, 2, 15)
        for _ in range(3):
            gl_s, _, _ = ix.search(qsets[qi], k, ef=ef_ship)
        ship_ms = ix.last_kernel_ms()
        shipped = {"ef": ef_ship, "gpu_kernel_queries_per_s": Q / (ship_ms * 1e-3),
                   "gpu_recall_at_k": recall_at_k(gl_s[:nrec], gt_l), "cpu_queries_per_s": Q / smed,
                   "cpu_recall_at_k": recall_at_k(res["s"][:nrec], gt_l), "cpu_threads": cores}
        cpu = {"value": Q / med, "unit": "queries/s", "cores": cores, "kind": "port", "pinned": True, **info,
               "best_queries_per_s": Q / best, "median_queries_per_s": Q / med, "passes": passes,
               "reference_as_shipped": shipped,
               "sample": f"oracle (hnswlib restatement) searching the same {N}-point graph exported from the GPU "
                         f"build, same {Q} queries, ef={ef}; median of {passes} passes on {cores} pinned threads",
               "single_thread_queries_per_s": cpu_1t, "recall_at_k": recall_at_k(cl[:nrec], gt_l),
               "ids_equal_to_gpu_frac": float(np.mean(cl == labels_dev))}
        del o
    if not args.no_cpu_baseline and not args.no_parity and not brute:
        parity = parity_block(ehb, orc, wl, args.parity_budget, cores, local)

    h2d = Q * d * 4
    d2h = Q * k * 12 + Q * 4
    launches_per_step = 1 + (1 if metric == "cosine" else 0) + (1 if world > 1 else 0)
    if brute:  # pad + 2x to_bf16 (first step) + per (q-chunk, n-chunk): GEMM, select, merge + fill + re-rank
        nchunks = -(-Q // 2048) * -(-N // 131072)
        launches_per_step = 3 + 3 * nchunks + 2 + (1 if world > 1 else 0)
    global_qps = Q / (dev_ms * 1e-3)
    line = {
        "metric": "k-NN queries/s", "value": global_qps, "unit": "queries/s", "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic" if DIST == "gaussian" else "synthetic (gmm)",
        "config": shared_config(wl, world),
        "details": {"path": "bruteforce bf16 tcgen05 + fp32 re-rank" if brute else "graph walk",
                    "l2": "flushed between timed steps (256 MB write) and the index (vectors+links) is larger than L2",
                    "parallelism": f"range-sharded x{world}, one {searcher.exchange} exchange of per-shard top-k + merge"
                    if world > 1 else "single GPU", "exchange": searcher.exchange, "build_s": round(t_build, 2),
                    "ingest_s": round(t_ingest, 1), "setup_s": round(time.time() - t_setup0, 1)},
        "shard_searches_per_s": world * global_qps,
        "shard_only_ms_per_step": shard_ms,
        "recall_at_k": rec, "recall_queries": nrec,
        "e2e": {"value": Q / (e2e_ms * 1e-3), "unit": "queries/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms},
        "gpu_launches": launches_per_step * steps,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "parity": parity,
        "clocks": clocks,
    }
    if timed_out:
        line["exchange_timed_out"] = True
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ehb200", choices=["ehb200", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto"] + sorted(WORKLOADS))
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--walk-prefetch", type=int, default=-1, help="A/B: 0/1 sets the library option, -1 keeps its default")
    ap.add_argument("--parity-budget", type=float, default=45.0, help="seconds of CPU construction for the parity block")
    ap.add_argument("--ref-build-budget", type=float, default=100.0)
    ap.add_argument("--ref-max-points", type=int, default=1_000_000)
    ap.add_argument("--recall-queries", type=int, default=2000)
    ap.add_argument("--dist", default="gaussian", choices=["gaussian", "gmm"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the labels, distances and counts of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global DIST
    DIST = args.dist
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    if args.workload == "auto":
        args.workload = "c3" if max(world, args.gpus) == 1 else "c5"
    wl = dict(WORKLOADS[args.workload])
    if DIST != "gaussian":
        wl["desc"] += " [secondary distribution: 1024-centre GMM, sigma 0.3]"
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ehb(args, wl)


if __name__ == "__main__":
    main()
