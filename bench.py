#!/usr/bin/env python
"""bench.py -- QPS of the Vamana batched search (BASELINE.json metric) on B200, one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1], the configuration the metric is quoted on): synthetic 1M x 96-d
float32, L2, Vamana search_window=128, batch = 10k queries, k = 10; graph built once per box by the
reference's own CPU builder (oracle/_ref, R=64, window 128, alpha 1.2) and cached in the system's temporary
directory.  oracle/_ref can only be compiled where the reference's sources are; without it (and without a cached
graph) the graph comes from the project's GPU builder (svsb200_build_vamana, same parameters), and the line's
config.graph_builder says which.  A "step" = one full pass of the hot path over the 10k-query batch.
--dump-outputs DIR writes the results of the last timed step (ids as float64, distances as float32) to
DIR/ids.npy and DIR/distances.npy.  Data and queries come from fixed seeds and the graph is cached per box, so runs
with the same arguments search the same inputs and two builds can be compared output for output (a graph built
afresh can differ in a few edges: both builders' results depend on thread timing).

Lines printed (rank 0 only):
  value     whole-job QPS with queries/results resident in HBM (CUDA events, max over ranks)
  e2e       same metric through the C ABI with HOST buffers (pinned), H2D + D2H inside the timed region
  roofline  algorithmic HBM bytes of the search kernel / its CUDA-event duration vs MEASURED_PEAKS.json
  cpu_baseline  the reference's own AVX-512 CPU path (oracle/_ref) on this box's host cores
`--impl reference` times that CPU path alone under the same metric/config.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: n, dim, dtype, metric, nq, k, window, max_degree, build window
    "c2-1Mx96-f32-L2-w128": dict(n=1_000_000, dim=96, dtype="float32", metric="l2", nq=10_000, k=10, window=128,
                                 max_degree=64, build_window=128, alpha=1.2),
    # reduced-size stand-ins for BASELINE configs[2..4] (the full sizes need a GPU graph builder: the reference's
    # CPU builder takes ~36 s per million 96-d vectors on the box's 16-core quota)
    "c3s-200kx768-f16-IP-w128": dict(n=200_000, dim=768, dtype="float16", metric="ip", nq=10_000, k=10, window=128,
                                     max_degree=64, build_window=128, alpha=0.95),
    "c4s-1Mx96-lvq8-L2-w128": dict(n=1_000_000, dim=96, dtype="float32", metric="l2", nq=10_000, k=10, window=128,
                                   max_degree=64, build_window=128, alpha=1.2, storage="lvq8",
                                   graph_from="c2-1Mx96-f32-L2-w128"),
    "c5s-2Mx96-f16-L2-sharded": dict(n=2_000_000, dim=96, dtype="float16", metric="l2", nq=10_000, k=10, window=128,
                                     max_degree=64, build_window=128, alpha=1.2, sharded=True),
    # BASELINE configs[2..4] at their stated sizes; graphs from the GPU builder (svsb200_build_vamana: the reference's
    # CPU builder needs minutes to hours at these sizes) -- both arms then search that same graph
    "c3-1Mx768-f16-IP-w128": dict(n=1_000_000, dim=768, dtype="float16", metric="ip", nq=10_000, k=10, window=128,
                                  max_degree=64, build_window=128, alpha=0.95, builder="gpu"),
    "c4-10Mx96-lvq8-L2-w128": dict(n=10_000_000, dim=96, dtype="float32", metric="l2", nq=10_000, k=10, window=128,
                                   max_degree=64, build_window=128, alpha=1.2, storage="lvq8", builder="gpu"),
    "c5-100Mx96-f16-L2-sharded": dict(n=100_000_000, dim=96, dtype="float16", metric="l2", nq=100_000, k=10, window=128,
                                      max_degree=64, build_window=128, alpha=1.2, sharded=True, builder="gpu",
                                      per_shard_data=True),
    "tiny-100kx96-f32-L2-w128": dict(n=100_000, dim=96, dtype="float32", metric="l2", nq=10_000, k=10, window=128,
                                     max_degree=64, build_window=128, alpha=1.2),
}
FALLBACK_HBM_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md, used only without MEASURED_PEAKS.json
FALLBACK_BF16_TFLOPS = 2250.0   # nominal dense bf16 (same guide), used only without MEASURED_PEAKS.json


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def effective_cpus():
    """Host cores this process may actually use: min(os.cpu_count, affinity mask, cgroup CPU quota).  On the
    GPU boxes the container sees 128 logical CPUs but `cpu.max` grants 16; the reference's spin-waiting
    thread pool collapses when oversubscribed, so its arm is run at the granted count."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ------------------------------------------------------------------------------------------------
# workload: data + graph (cached per box in the temporary directory, rank 0 builds)
# ------------------------------------------------------------------------------------------------
def graph_cache_path(tag, w):
    key = hashlib.sha1(json.dumps({k: w.get(k) for k in ("n", "dim", "dtype", "metric", "max_degree", "build_window",
                                                           "alpha", "builder")}, sort_keys=True).encode()).hexdigest()[:12]
    return os.path.join(os.environ.get("SVSB200_CACHE") or os.path.join(tempfile.gettempdir(), "svsb200_cache"),
                        f"graph_{tag}_{key}.npy")


def graph_source(tag, w):
    """`w` with the builder its graph comes from: the reference's CPU builder where oracle/_ref is built or its graph
    is cached, otherwise the GPU builder (oracle/_ref needs the reference's sources to compile)."""
    from oracle.bindings import RefLib
    if w.get("builder") or os.path.exists(graph_cache_path(tag, w)) or RefLib.available():
        return w
    log(f"oracle/_ref/libsvsref.so is not built: graph {tag} from the GPU builder (svsb200_build_vamana)")
    return dict(w, builder="gpu")


def build_graph_cached(tag, w, base, rank_builds, barrier):
    """Vamana graph from the GPU builder or the reference's own CPU builder (oracle/_ref), cached per box in the
    temporary directory."""
    cache = graph_cache_path(tag, w)
    if w.get("per_shard_data") and w.get("builder") == "gpu":
        # multi-GB shard graphs: built in place on this rank's GPU, never written to disk
        from scalablevectorsearch_b200 import DistanceType, VamanaBuildParameters, build_graph
        t1 = time.time()
        graph, ep = build_graph(base, {"l2": DistanceType.L2, "ip": DistanceType.MIP}[w["metric"]],
                                VamanaBuildParameters(alpha=w["alpha"], graph_max_degree=w["max_degree"],
                                                      window_size=w["build_window"]),
                                device=int(os.environ.get("LOCAL_RANK", 0)))
        log(f"GPU graph build {tag} n={base.shape[0]} dim={base.shape[1]} R={w['max_degree']}: {time.time() - t1:.1f} s, "
            f"avg degree {graph[:, 0].mean():.1f}")
        barrier()
        return ep, graph
    if rank_builds and not os.path.exists(cache) and w.get("builder") == "gpu":
        from scalablevectorsearch_b200 import DistanceType, VamanaBuildParameters, build_graph
        os.makedirs(os.path.dirname(cache), exist_ok=True)
        t1 = time.time()
        graph, ep = build_graph(base, {"l2": DistanceType.L2, "ip": DistanceType.MIP}[w["metric"]],
                                VamanaBuildParameters(alpha=w["alpha"], graph_max_degree=w["max_degree"],
                                                      window_size=w["build_window"]),
                                device=int(os.environ.get("LOCAL_RANK", 0)))
        log(f"GPU graph build {tag} n={base.shape[0]} dim={base.shape[1]} R={w['max_degree']}: {time.time() - t1:.1f} s, "
            f"avg degree {graph[:, 0].mean():.1f}")
        tmp = cache + f".tmp{os.getpid()}"
        with open(tmp, "wb") as f:
            np.save(f, np.concatenate([np.array([[ep] + [0] * w["max_degree"]], dtype=np.uint32), graph]))
        os.replace(tmp, cache)
    if rank_builds and not os.path.exists(cache):
        from oracle.bindings import RefLib   # checker/baseline infrastructure: builds the graph only
        if not RefLib.available():
            raise SystemExit("oracle/_ref/libsvsref.so is missing: run `python -c 'import __graft_entry__ as g; "
                             "g.build()'` where /root/reference exists (the graph comes from the reference builder)")
        os.makedirs(os.path.dirname(cache), exist_ok=True)
        t1 = time.time()
        threads = max(1, effective_cpus() // w.get("build_share", 1))
        graph, ep = RefLib().build(base, w["metric"], w["max_degree"], w["build_window"], alpha=w["alpha"],
                                   threads=threads)
        log(f"reference auto_build {tag} n={base.shape[0]} dim={base.shape[1]} R={w['max_degree']} on {threads} threads: "
            f"{time.time() - t1:.1f} s, avg degree {graph[:, 0].mean():.1f}")
        tmp = cache + f".tmp{os.getpid()}"
        with open(tmp, "wb") as f:
            np.save(f, np.concatenate([np.array([[ep] + [0] * w["max_degree"]], dtype=np.uint32), graph]))
        os.replace(tmp, cache)
    barrier()
    blob = np.load(cache, mmap_mode="r")
    return int(blob[0, 0]), np.ascontiguousarray(blob[1:])


def load_workload(name, rank, world, barrier):
    from scalablevectorsearch_b200.synthetic import clustered_unit_vectors
    w = WORKLOADS[name]
    t0 = time.time()
    base, queries = clustered_unit_vectors(w["n"], w["nq"], w["dim"])
    if w["dtype"] == "float16":
        base = base.astype(np.float16)
    gname = w.get("graph_from", name)
    gw = graph_source(gname, WORKLOADS[gname])
    w = dict(w, builder=gw.get("builder"))
    ep, graph = build_graph_cached(gname, gw, base, rank == 0, barrier)
    log(f"rank {rank}: workload {name} ready in {time.time() - t0:.1f} s (entry point {ep})")
    return w, base, queries, graph, ep


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].startswith("Active") for r in self.rows if len(r) >= 7)]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(sm)}


def algorithmic_bytes(hops, evals, rows_read, w, row_bytes, qbytes):
    """SURVEY.md §8(d) per query: sum_hops 4*(1+deg) + rows * row_bytes + D*sizeof(Tq) + k*8.
    `evals` = entry points + sum of out-degrees and `hops` = expanded nodes (the counts a reference
    GreedySearchTracker reports).  `rows_read` is the number of base-vector rows charged: `evals` for the
    reference-equivalent figure (the CPU path re-reads every neighbour: visited set off by default), or the
    kernel's own `fetched` counter (rows that pass its exact visited filter) for the bytes the kernel must move."""
    hops, evals, rows_read = hops.astype(np.float64), evals.astype(np.float64), rows_read.astype(np.float64)
    per_query = 4.0 * (hops + (evals - 1.0)) + rows_read * row_bytes + qbytes + w["k"] * 8.0
    return float(per_query.sum()), float(per_query.mean())


# ------------------------------------------------------------------------------------------------
# reference arm (CPU): the reference's own AVX-512 path via oracle/_ref
# ------------------------------------------------------------------------------------------------
def time_reference(w, base, queries, graph, ep, steps, warmup, threads):
    from oracle.bindings import RefLib
    ref = RefLib()
    idx = ref.index(base, graph, ep, w["metric"], threads=threads)
    for _ in range(warmup):
        idx.search(queries, w["k"], w["window"], w["window"])
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        ids, dists = idx.search(queries, w["k"], w["window"], w["window"])
        times.append(time.perf_counter() - t0)
    return times, ids, dists, ref


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    w, base, queries, graph, ep = load_workload(args.workload, 0, 1, lambda: None)
    if args.window:
        w = dict(w, window=args.window)
    threads = effective_cpus()
    # the CPU path's QPS does not depend on how many GPUs our arm uses: each step is one 10k-query batch of the
    # same workload (a bounded sample of the N x 10k global batch of the weak-scaling run)
    times, ids, dists, ref = time_reference(w, base, queries, graph, ep, args.steps, args.warmup, threads)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ids=ids, distances=dists)
    total = sum(times)
    qps = w["nq"] * len(times) / total
    line = {
        "impl": "reference", "metric": "QPS", "value": qps, "unit": "queries/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True,
        "scaling": "weak" if args.weak else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": run_config(args.workload, w, graph, args.gpus, args.weak),
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "kind": "reference",
                         "sample": f"full {w['nq']}-query batch x {len(times)} steps, {threads} threads = container CPU quota "
                                   f"(os.cpu_count()={os.cpu_count()}), avx512={ref.avx512()}, "
                                   f"{REF_PAGES}"},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


REF_PAGES = ("reference data+graph in lib::Allocator memory = 4 KiB pages (transparent hugepages per the host's THP "
             "setting); its HugepageAllocator (core/allocator.h:94-150) is not used by this arm")


def dump_outputs(directory, **arrays):
    """Save each result array of the last timed step as DIR/<name>.npy: integer ids as float64 (exact below 2^53),
    distances as float32."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
        np.save(os.path.join(directory, f"{name}.npy"), a.astype(np.float64 if a.dtype.kind in "iu" else np.float32))


def run_config(name, w, graph, gpus, weak):
    """The `config` object, identical in both arms (the driver compares them)."""
    return dict(workload_config(name, w, graph), global_batch=w["nq"] * (gpus if weak else 1),
                batch_per_gpu=w["nq"] if weak else -(-w["nq"] // gpus))


def workload_config(name, w, graph):
    return {"workload": name, "n": w["n"], "dim": w["dim"], "base_dtype": w["dtype"], "distance": w["metric"],
            "batch": w["nq"], "k": w["k"], "search_window": w["window"], "graph_max_degree": w["max_degree"],
            "graph_avg_degree": round(float(graph[:, 0].mean()), 2), "graph_builder": w.get("builder") or "reference cpu",
            "l2_policy": "index (vectors+graph) is several times larger than the 126 MB L2; no explicit flush"}


# ------------------------------------------------------------------------------------------------
# our arm (GPU)
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from scalablevectorsearch_b200 import DistanceType, SearchBufferConfig, Vamana, _lib
    from scalablevectorsearch_b200.multi_gpu import ReplicatedSearch, balance, cuda_local_search

    rank, local_rank, world = dist_env()
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL prints its version banner there at NCCL_DEBUG=VERSION *and*
        # WARN (the boxes export one of them); INFO/TRACE are left alone for whoever asks for them explicitly
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            del os.environ["NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=dev)
    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)

    w, base, queries, graph, ep = load_workload(args.workload, rank, world, barrier)
    if args.window:
        w = dict(w, window=args.window)
    if args.batch:
        w = dict(w, nq=args.batch)
        queries = queries[:args.batch]
    metric = {"l2": DistanceType.L2, "ip": DistanceType.MIP, "cosine": DistanceType.Cosine}[w["metric"]]
    row_bytes = w["dim"] * base.dtype.itemsize
    lvq = None
    if w.get("storage") == "lvq8":
        from scalablevectorsearch_b200 import lvq8_compress
        rows, mean = lvq8_compress(base, device=local_rank)
        lvq = (rows, mean)
        row_bytes = rows.shape[1]
        index = Vamana.from_arrays(rows, graph, ep, metric, device=local_rank, lvq8=(w["dim"], mean))
    else:
        index = Vamana.from_arrays(base, graph, ep, metric, device=local_rank)
    index.search_parameters.buffer_config = SearchBufferConfig(w["window"])
    for opt in ("warps_per_cta", "ctas_per_sm", "rows_in_flight"):
        if getattr(args, opt):
            index.set_option(opt, getattr(args, opt))
    index.set_option("visited_filter_slots", args.filter_slots)
    for kv in args.opt:
        name, val = kv.split("=")
        index.set_option(name, int(val))
    lib = _lib.lib()
    k = w["k"]
    searcher = ReplicatedSearch(cuda_local_search(index, id_dtype=torch.int32), id_dtype=torch.int32)

    # Two batch shapes (SURVEY.md 8e mode A).  STRONG -- the metric's own configuration: ONE batch of w["nq"] queries
    # split over the GPUs with threads::balance; this is `value`.  WEAK: every GPU keeps a whole w["nq"]-query batch
    # (global batch N x that; block 0 is the single-GPU batch), reported beside it under "weak".
    from scalablevectorsearch_b200.synthetic import clustered_queries
    q_strong = queries
    q_weak = queries if world == 1 else np.concatenate(
        [queries] + [clustered_queries(w["nq"], w["dim"], r) for r in range(1, world)])

    kernel_kind = {}

    def time_mode(q_np):
        """W warm-ups, K timed steps of the device-resident multi-GPU search (local search -> one NCCL all-gather of
        the result rows), CUDA events on this rank's stream, max over ranks."""
        q_dev = torch.from_numpy(q_np).to(dev)
        for _ in range(max(args.warmup, 3)):
            out = searcher.search(q_dev, k)
        torch.cuda.synchronize()
        barrier()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = lib.svsb200_launch_count()
        start.record()
        for _ in range(args.steps):
            out = searcher.search(q_dev, k)
        stop.record()
        torch.cuda.synchronize()
        launched = lib.svsb200_launch_count() - l0
        out = tuple(t.clone() for t in out)   # the multi-GPU gather reuses its buffers on the next call
        barrier()
        ms = start.elapsed_time(stop)
        kern = []
        for _ in range(3):
            searcher.search(q_dev, k)
            torch.cuda.synchronize()
            kern.append(index.last_kernel_ms())
        kernel_kind["timed"] = index.get_option("last_kernel")
        t = torch.tensor([ms, float(np.mean(kern))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), out, q_dev, launched

    # ---- per-query work counters (reference tracker equivalents) for the roofline, on the strong batch ----
    nq = q_strong.shape[0]
    lo, hi = balance(nq, world, rank)
    q_dev = torch.from_numpy(q_strong).to(dev)
    index.set_counting(True)
    searcher.search(q_dev, k)
    torch.cuda.synchronize()
    hops, evals = index.counters(hi - lo)
    fetched = index.fetched(hi - lo)
    index.set_counting(False)
    qb = w["dim"] * queries.dtype.itemsize
    shard_bytes, bytes_per_query = algorithmic_bytes(hops, evals, fetched, w, row_bytes, qb)
    shard_ref_bytes, ref_bytes_per_query = algorithmic_bytes(hops, evals, evals, w, row_bytes, qb)

    with ClockSampler(local_rank) as clocks:
        elapsed_ms, kern_ms, (ids_all, d_all), q_dev, launches = time_mode(q_strong)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ids=ids_all, distances=d_all)
    qps = nq * args.steps / (elapsed_ms * 1e-3)
    weak = None
    if world > 1:
        w_ms, w_kern, _, _, _ = time_mode(q_weak)
        weak = {"value": q_weak.shape[0] * args.steps / (w_ms * 1e-3), "unit": "queries/s", "ms_per_step": w_ms / args.steps,
                "kernel_ms": w_kern, "global_batch": int(q_weak.shape[0]), "batch_per_gpu": int(w["nq"])}

    # the same kernel with its visited filter off reads every neighbour row, like the CPU path does:
    # that run is the apples-to-apples HBM-bandwidth measurement against the reference-equivalent bytes
    nofilter_ms = []
    index.set_option("visited_filter_slots", 0)
    for i in range(4):
        searcher.search(q_dev, k)
        torch.cuda.synchronize()
        if i:
            nofilter_ms.append(index.last_kernel_ms())
    index.set_option("visited_filter_slots", args.filter_slots)
    t = torch.tensor([shard_bytes, shard_ref_bytes, float(np.mean(nofilter_ms))], dtype=torch.float64, device=dev)
    if world > 1:
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_bytes, total_ref_bytes, nofilter = float(tsum[0]), float(tsum[1]), float(t[2])
    else:
        total_bytes, total_ref_bytes, nofilter = float(t[0]), float(t[1]), float(t[2])

    # ---- end to end with HOST buffers, through the call a user makes ----
    cfg = index.search_parameters.buffer_config
    if world == 1:
        # svsb200_search (C ABI): pinned host queries in, host ids + distances out, H2D + kernels + D2H per step
        q_host = torch.from_numpy(q_strong).pin_memory()
        out_ids = torch.empty((nq, k), dtype=torch.int64).pin_memory()
        out_d = torch.empty((nq, k), dtype=torch.float32).pin_memory()

        def step_e2e():
            _lib.check(lib.svsb200_search(index._h, q_host.data_ptr(), 0, nq, k, cfg.search_window_size,
                                          cfg.search_buffer_capacity, 0, out_ids.data_ptr(), 8, out_d.data_ptr(), None))
        e2e_path = "svsb200_search (C ABI): pinned host queries in, host ids + distances out"
        h2d, d2h = int(nq * w["dim"] * 4), int(nq * k * 12)
    else:
        # every rank: H2D of its query slice, local search, NCCL all-gather of the rows; rank 0: D2H of the whole result
        q_host = torch.from_numpy(np.ascontiguousarray(q_strong[lo:hi])).pin_memory()
        q_stage = torch.empty((nq, w["dim"]), dtype=torch.float32, device=dev)
        out_ids = torch.empty((nq, k), dtype=torch.int32).pin_memory()
        out_d = torch.empty((nq, k), dtype=torch.float32).pin_memory()

        def step_e2e():
            q_stage[lo:hi].copy_(q_host, non_blocking=True)
            ids, dd = searcher.search(q_stage, k)
            if rank == 0:
                out_ids.copy_(ids, non_blocking=True)
                out_d.copy_(dd, non_blocking=True)
            torch.cuda.synchronize()
        e2e_path = ("per rank: pinned host query slice -> HBM, local search, NCCL all-gather of the result rows; rank 0: "
                    "whole result -> pinned host; wall clock between barriers, max over ranks")
        h2d, d2h = int(nq * w["dim"] * 4), int(nq * k * 8)
    for _ in range(3):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_qps = nq * args.steps / float(te[0])
    same = bool(rank != 0 or np.array_equal(out_ids.numpy().astype(np.int64), ids_all.cpu().numpy().astype(np.int64)))

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"
        achieved = total_bytes / (kern_ms * 1e-3) / 1e9 / world   # per-GPU GB/s of the search kernel
        ref_achieved = total_ref_bytes / (kern_ms * 1e-3) / 1e9 / world
        nofilter_achieved = total_ref_bytes / (nofilter * 1e-3) / 1e9 / world
        ncu_traffic = None
        ncu_path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(ncu_path) and world == 1:
            ncu_traffic = json.load(open(ncu_path)).get(args.workload, {}).get("dram_bytes_per_launch")
        # recall@10 on a sample against the exact top-k (svsb200_exhaustive_device: the search path's own distance code,
        # ties by id; checked against the oracle in tests/test_gpu_parity.py::test_exhaustive_scan_is_exact_topk)
        # (uncompressed data: the tensor-core flat search over the whole batch -- exact by construction, equal to that
        # scan bit for bit, tests/test_gpu_flat.py; LVQ-8: the scan on a 1000-query sample)
        sample = nq if lvq is None else min(1000, nq)
        gt_ids = torch.empty((sample, k), dtype=torch.int64, device=dev)
        gt_d = torch.empty((sample, k), dtype=torch.float32, device=dev)
        gt_stream = torch.cuda.current_stream(dev).cuda_stream or 1
        if lvq is None:
            index.flat_search_device(q_dev.data_ptr(), queries.dtype, sample, k, gt_ids.data_ptr(), gt_d.data_ptr(),
                                     stream=gt_stream)
        else:
            index.exhaustive_device(q_dev.data_ptr(), queries.dtype, sample, k, gt_ids.data_ptr(), gt_d.data_ptr(),
                                    stream=gt_stream)
        torch.cuda.synchronize()
        ground_truth = None
        if lvq is None:   # the call above built the tiles; time one more (the whole batch's exact top-k)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fb = index.flat_search_device(q_dev.data_ptr(), queries.dtype, sample, k, gt_ids.data_ptr(),
                                          gt_d.data_ptr(), stream=gt_stream)
            e1.record()
            torch.cuda.synchronize()
            gt_ms = e0.elapsed_time(e1)
            tf_peak = (float(json.load(open(peaks_path)).get("bf16_tflops", FALLBACK_BF16_TFLOPS))
                       if os.path.exists(peaks_path) else FALLBACK_BF16_TFLOPS)
            tflops = 2.0 * sample * w["n"] * w["dim"] / (gt_ms * 1e-3) / 1e12
            ground_truth = {"kernel": "flat_gemm_topk_kernel (tcgen05 fp16 x fp16 -> fp32, fused top-k) + exact rescore",
                            "queries": sample, "ms": gt_ms, "tflops_whole_call": tflops, "peak_tflops": tf_peak,
                            "frac_of_bf16_peak": tflops / tf_peak, "queries_sent_to_exact_scan": int(fb),
                            "note": "whole svsb200_flat_search_device call (GEMM + per-tile top-k + bit-exact rescoring + "
                                    "verification), not the GEMM alone; a 96-wide K is epilogue-bound (DESIGN.md 9)"}
        gt = gt_ids.cpu().numpy()
        got = ids_all[:sample].cpu().numpy()
        recall = float(np.mean([len(set(got[i].tolist()) & set(gt[i].tolist())) for i in range(sample)])) / k

        cpu = None
        if not args.no_cpu_baseline and world == 1:   # reported at N=1 only; `--impl reference` covers every N
            try:
                if lvq is not None:
                    raise NotImplementedError("LVQ is closed source in the reference: no reference arm for this workload")
                threads = effective_cpus()
                nb = min(w["nq"], args.cpu_sample or w["nq"])   # the metric's batch (or a bounded sample of it)
                reps = 5 if nb == w["nq"] and w["n"] * w["dim"] <= 2e8 else 1
                times, ref_ids, ref_d, ref = time_reference(w, base, queries[:nb], graph, ep, reps, 1 if reps > 1 else 0,
                                                            threads)
                cpu_qps = nb / min(times)
                ids_equal = bool(np.array_equal(ref_ids, ids_all[:nb].cpu().numpy().astype(np.uint64)))
                d_equal = bool(np.array_equal(ref_d.view(np.uint32), d_all[:nb].cpu().numpy().view(np.uint32)))
                cpu = {"value": nb * len(times) / sum(times), "best": cpu_qps, "unit": "queries/s", "cores": threads,
                       "kind": "reference",
                       "sample": f"reference AVX-512 path (oracle/_ref, avx512={ref.avx512()}), first {nb} queries of the "
                                 f"batch, {len(times)} timed searches on {threads} threads = the container's CPU quota "
                                 f"(os.cpu_count()={os.cpu_count()}); {REF_PAGES}",
                       "ids_identical_to_gpu": ids_equal, "distances_bit_identical_to_gpu": d_equal}
            except NotImplementedError:
                from oracle.bindings import OracleLib   # own-spec LVQ-8: the CPU checker is the baseline ("port")
                oidx = OracleLib().lvq8_index(lvq[0], w["dim"], lvq[1], graph, ep, w["metric"])
                ns = 256
                t0 = time.perf_counter()
                o_ids, o_d = oidx.search(queries[:ns], k, w["window"], w["window"])
                dt = time.perf_counter() - t0
                cpu = {"value": ns / dt, "unit": "queries/s", "cores": 1, "kind": "port",
                       "sample": f"oracle/vamana_oracle.c LVQ-8 restatement, first {ns} queries, 1 thread (scalar)",
                       "ids_identical_to_gpu": bool(np.array_equal(o_ids, ids_all[:ns].cpu().numpy().astype(np.uint64))),
                       "distances_bit_identical_to_gpu": bool(np.array_equal(
                           o_d.view(np.uint32), d_all[:ns].cpu().numpy().view(np.uint32)))}
            except Exception as e:   # noqa: BLE001
                cpu = {"value": None, "unit": "queries/s", "cores": 0, "kind": "reference", "sample": f"unavailable: {e}"}
        dram_frac = (ncu_traffic / (kern_ms * 1e-3) / 1e9 / peak) if ncu_traffic else None
        line = {
            "metric": "QPS", "value": qps, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None,
            "dtype": "f32" if lvq is None else "f32 (fused LVQ-8 decode)", "data": "synthetic",
            "config": run_config(args.workload, w, graph, world, False),
            "weak": weak,
            "recall_at_10": round(recall, 4),
            "ground_truth": ground_truth,
            "parallelism": f"replicas x{world}: queries split with threads::balance, one NCCL all-gather of the top-k rows",
            "kernel": {1: "vamana_search_fast_kernel", 0: "vamana_search_kernel"}[kernel_kind["timed"]],
            "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "matches_device_path": same, "path": e2e_path},
            "gpu_launches": int(launches),
            "roofline": {
                "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic, "peak_source": peak_src, "kernel_ms": kern_ms,
                "frac_must_move": achieved / peak, "frac_survey_8d": ref_achieved / peak, "frac_dram_ncu": dram_frac,
                "judged_on": "frac_must_move (the 0.60 target of BASELINE.json north_star)",
                "algorithmic_bytes_per_query": bytes_per_query, "hops_per_query": float(hops.mean()),
                "evals_per_query": float(evals.mean()), "rows_fetched_per_query": float(fetched.mean()),
                "definition": "frac = frac_must_move = (adjacency rows + the base-vector rows that pass the kernel's exact "
                              "visited filter + query + results) / kernel time / peak, per GPU: the bytes this kernel must "
                              "move.  frac_survey_8d charges every neighbour evaluation of the CPU path (visited set off) "
                              "one row (SURVEY.md 8d; above 1 because the filter skips the re-reads the CPU performs).  "
                              "frac_dram_ncu = ncu dram__bytes per launch (profiles/ncu_traffic.json) / kernel time / peak.",
                "reference_equivalent": {"bytes_per_query": ref_bytes_per_query, "achieved": ref_achieved,
                                         "frac": ref_achieved / peak},
                "filter_off": {
                    "kernel_ms": nofilter, "achieved": nofilter_achieved, "frac": nofilter_achieved / peak,
                    "definition": "generic kernel, visited filter disabled: reads every row the reference reads; "
                                  "reference-equivalent bytes / its own kernel time"}},
            "cpu_baseline": cpu,
            "clocks": clocks.summary(),
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_sharded(args):
    """Mode B (SURVEY.md 8e, BASELINE configs[4] shape): base vectors split into one contiguous id range per GPU,
    each shard with its own reference-built graph and entry point; every rank searches all queries, NCCL all-gather
    of the per-shard top-k, TotalOrder merge on the GPU.  Checker: the reference on each shard + the same merge."""
    import torch
    import torch.distributed as dist
    from scalablevectorsearch_b200 import DistanceType, SearchBufferConfig, Vamana
    from scalablevectorsearch_b200.multi_gpu import (ShardedSearch, balance, cuda_local_search,
                                                     merge_topk_reference_order)
    from scalablevectorsearch_b200.synthetic import clustered_unit_vectors
    rank, local_rank, world = dist_env()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            del os.environ["NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=dev)
    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)
    w = WORKLOADS[args.workload]
    # --shards-total S > world: this run holds only the first `world` of S shards (rank r = shard r) -- one GPU's
    # share of the S-GPU job, for sizing it; the line says so
    total_shards = max(world, args.shards_total)
    lo, hi = balance(w["n"], total_shards, rank)
    if w.get("per_shard_data"):
        from scalablevectorsearch_b200.synthetic import clustered_base_block, clustered_queries
        queries = clustered_queries(w["nq"], w["dim"], 0)
        shard = clustered_base_block(hi - lo, w["dim"], rank)
    else:
        base, queries = clustered_unit_vectors(w["n"], w["nq"], w["dim"])
        shard = base[lo:hi]
        del base
    shard = np.ascontiguousarray(shard.astype(np.float16 if w["dtype"] == "float16" else np.float32))
    ws = dict(w, n=hi - lo, build_share=world)
    t_build = time.time()
    ep, graph = build_graph_cached(f"{args.workload}_shard{rank}of{total_shards}", ws, shard, True, lambda: None)
    t_build = time.time() - t_build
    barrier()
    metric = {"l2": DistanceType.L2, "ip": DistanceType.MIP}[w["metric"]]
    index = Vamana.from_arrays(shard, graph, ep, metric, device=local_rank)
    index.search_parameters.buffer_config = SearchBufferConfig(w["window"])
    nq, k = w["nq"], w["k"]
    q_dev = torch.from_numpy(queries).to(dev)
    searcher = ShardedSearch(cuda_local_search(index), id_offset=lo, greater=w["metric"] != "l2")
    for _ in range(max(args.warmup, 3)):
        ids, d = searcher.search(q_dev, k)
    torch.cuda.synchronize()
    barrier()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(args.steps):
        ids, d = searcher.search(q_dev, k)
    stop.record()
    torch.cuda.synchronize()
    barrier()
    t = torch.tensor([start.elapsed_time(stop)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    # checker: reference CPU search on this shard for a sample, gathered and merged on the host
    from oracle.bindings import RefLib
    ns = 200
    r_ids, r_d = RefLib().index(shard, graph, ep, w["metric"], threads=max(1, effective_cpus() // world)).search(
        queries[:ns], k, w["window"], w["window"])
    r_ids = r_ids.astype(np.int64) + lo
    # exact top-k of the same sample on this shard (tensor-core flat search), for the recall of the merged result
    gt_i = torch.empty((ns, k), dtype=torch.int64, device=dev)
    gt_d = torch.empty((ns, k), dtype=torch.float32, device=dev)
    index.flat_search_device(q_dev.data_ptr(), queries.dtype, ns, k, gt_i.data_ptr(), gt_d.data_ptr(),
                             stream=torch.cuda.current_stream(dev).cuda_stream or 1)
    torch.cuda.synchronize()
    parts, gts = [None] * world, [None] * world
    if world > 1:
        dist.all_gather_object(parts, (r_ids, r_d))
        dist.all_gather_object(gts, (gt_i.cpu().numpy() + lo, gt_d.cpu().numpy()))
    else:
        parts, gts = [(r_ids, r_d)], [(gt_i.cpu().numpy() + lo, gt_d.cpu().numpy())]
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, ids=ids, distances=d)
        gt_ids, _ = merge_topk_reference_order(np.stack([g_[0] for g_ in gts]), np.stack([g_[1] for g_ in gts]), k,
                                               w["metric"] != "l2")
        got = ids[:ns].cpu().numpy()
        recall = float(np.mean([len(set(got[i].tolist()) & set(gt_ids[i].tolist())) for i in range(ns)])) / k
        want_ids, want_d = merge_topk_reference_order(np.stack([p_[0] for p_ in parts]), np.stack([p_[1] for p_ in parts]), k,
                                                      w["metric"] != "l2")
        ok = bool(np.array_equal(want_ids, ids[:ns].cpu().numpy()) and np.array_equal(want_d, d[:ns].cpu().numpy()))
        qps = nq * args.steps / (float(t[0]) * 1e-3)
        print(json.dumps({
            "metric": "QPS", "value": qps, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": float(t[0]) / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "n": w["n"], "shards": total_shards, "shards_in_this_run": world,
                       "rows_per_shard": hi - lo, "graph_seconds_rank0": round(t_build, 1),
                       "graph_builder": w.get("builder", "reference cpu"), "dim": w["dim"], "base_dtype": w["dtype"],
                       "distance": w["metric"], "batch": nq, "k": k, "search_window": w["window"],
                       "parallelism": f"index sharded x{world} (own graph per shard), NCCL all-gather + TotalOrder merge"},
            "matches_reference_per_shard_plus_merge": ok, "checked_queries": ns, "recall_at_10": round(recall, 4)}),
            flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", default=os.environ.get("SVSB200_WORKLOAD", "c2-1Mx96-f32-L2-w128"),
                    choices=sorted(WORKLOADS))
    ap.add_argument("--window", type=int, default=0)
    ap.add_argument("--batch", type=int, default=0, help="use only the first BATCH queries (experiments)")
    ap.add_argument("--warps-per-cta", dest="warps_per_cta", type=int, default=0)
    ap.add_argument("--ctas-per-sm", dest="ctas_per_sm", type=int, default=0)
    ap.add_argument("--rows-in-flight", dest="rows_in_flight", type=int, default=0)
    ap.add_argument("--filter-slots", dest="filter_slots", type=int, default=-1)
    ap.add_argument("--opt", action="append", default=[], help="library option name=value (svsb200_set_option)")
    ap.add_argument("--shards-total", dest="shards_total", type=int, default=0,
                    help="sharded workloads: split the base into this many shards and hold only the first --gpus of them")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--weak", action="store_true",
                    help="reference arm only: label the line as the weak-scaling batch (our arm reports the strong "
                         "result as `value` and the weak one under `weak` in the same line)")
    ap.add_argument("--cpu-sample", dest="cpu_sample", type=int, default=0,
                    help="cpu_baseline: time only the first N queries of the batch (bounded sample for big workloads)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", default=None, metavar="DIR",
                    help="write the results of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if WORKLOADS[args.workload].get("sharded"):
        run_sharded(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
