#!/usr/bin/env python
"""bench.py — QPS of the HNSW-Slim search hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our CUDA engine (C ABI)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU search

A "step" = one pass of the hot path over one batch of synthetic queries:
HierarchicalNSWSlim::searchKnn for every query of the batch (hnsw_slim_strategy.h:112-114)
== ONE hs_search_batch_device launch.  Workload at every N: BASELINE.json configs[0], the
configuration the north-star target is quoted on — SIFT-shaped synthetic 1M x 128 L2,
hnsw_slim M=16 ef_construction=200, k=10 ef_search=100, 10k queries per batch.  With N GPUs
the 1M index is replicated and every rank searches its own 10k-query batch (north_star:
"1M-scale indices are replicated and queries are split with no collective") => weak scaling,
value = N * 10k * K / max-over-ranks device time.  `--workload deep-sharded` runs the
sharded path instead (one sub-graph per shard, NCCL all-gather + top-k merge).

Prints ONE JSON line (rank 0).  Inputs (corpus, queries, .graph) are generated once and cached
in $HS_DATA_CACHE (default /tmp/hs_data_cache); the .graph is built by the engine's own host
builder (hs_build_slim_graph), not by anything under oracle/.

`--dump-outputs DIR` writes what the last timed step returned (rank 0) as DIR/<name>.npy: the
labels (as float64, exact) and distances (float32) of the whole batch, and DIR/inputs.json with
SHA-256 digests of the index and of the query batch.  Corpus and queries are seeded, and the
.graph is then built deterministically (the multi-threaded host build differs from run to run) and
cached as its own file: by the GPU builder (about 2 s at 1M x 128), for hnsw_slimq by the host
builder on one thread (more than 8 minutes at 1M rows).  So two builds of the project run with the
same arguments search the same inputs and can be compared output for output.  Indices that live
in HBM only (the sharded and ef-sweep workloads) are digested through hs_save_index.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CACHE = os.environ.get("HS_DATA_CACHE", "/tmp/hs_data_cache")

WORKLOADS = {
    # BASELINE.json configs[0]
    "sift1m": dict(n=1_000_000, dim=128, metric=0, M=16, efc=200, rank=14, nq=10_000, k=10, ef=100,
                   desc="SIFT-shaped synthetic 1Mx128 L2, hnsw_slim M=16 efc=200 (rank-14 latent Gaussian, seed 1)"),
    # BASELINE.json configs[3] shape (DEEP 96-dim, 8 sub-graphs, NVLink top-k merge), scaled from
    # 100M to what the host can index inside a benchmark run: 8 shards x 500k rows.
    "deep-sharded": dict(n=8_000_000, shards=8, dim=96, metric=0, M=16, efc=200, rank=12, nq=10_000, k=10, ef=100,
                         desc="DEEP-shaped synthetic {n}x96 L2 in 8 sub-graphs of {rows} rows (the 100M config scaled to "
                              "what can be indexed inside a benchmark run), hnsw_slim M=16 efc=200, rows exchanged over "
                              "NVLink + top-k merge"),
    # BASELINE.json configs[1]: GIST-shaped, ef_search sweep 50-400 (tools/perf_probe.py --efs ...)
    "gist1m": dict(n=1_000_000, dim=960, metric=0, M=32, efc=200, rank=24, nq=10_000, k=10, ef=100, curve=True,
                   desc="GIST-shaped synthetic 1Mx960 L2, hnsw_slim M=32 efc=200 (rank-24 latent Gaussian, seed 1)"),
    # BASELINE.json configs[2]: COHERE-shaped, inner product on unit vectors
    # (rank 16: with rank 24 the pruned graph stays below recall 0.95 up to ef=400, profiles/r01_probe_gist_cohere_final.txt)
    "cohere1m": dict(n=1_000_000, dim=768, metric=1, M=32, efc=200, rank=16, nq=10_000, k=10, ef=100, curve=True,
                     desc="COHERE-shaped synthetic 1Mx768 inner product (unit rows), hnsw_slim M=32 efc=200 "
                          "(rank-16 latent Gaussian, seed 1)"),
    # BASELINE.json configs[4] shape (MSTuring 96-dim, hnsw-slimq = RaBitQ codes + exact rerank) on one GPU
    "msturing1m-slimq": dict(n=1_000_000, dim=96, metric=0, M=16, efc=200, rank=12, nq=10_000, k=10, ef=100,
                             kind="slimq",
                             desc="MSTuring-shaped synthetic 1Mx96 L2, hnsw_slimq (16 clusters, 1-bit RaBitQ codes + exact "
                                  "rerank) M=16 efc=200 (rank-12 latent Gaussian, seed 1)"),
    # ... and sharded like configs[4]: 8 sub-graphs over 1/2/4/8 GPUs, scaled from 100M to 8 x 500k rows
    "msturing-sharded-slimq": dict(n=8_000_000, shards=8, dim=96, metric=0, M=16, efc=200, rank=12, nq=10_000, k=10,
                                   ef=100, kind="slimq",
                                   desc="MSTuring-shaped synthetic {n}x96 L2 in 8 hnsw_slimq sub-graphs of {rows} rows (100M "
                                        "config scaled down), M=16 efc=200, rows exchanged over NVLink + top-k merge"),
    # reduced-size variants for quick local runs (not contract lines)
    # the reference's ground-truth producer (BruteForce::solve writes k=100 rows, brute_force_strategy.h:15-45):
    # the one dense contraction of the system, on the tcgen05 tensor cores (bruteforce_tc.cu)
    "bruteforce1m": dict(n=1_000_000, dim=128, metric=0, rank=14, nq=10_000, k=100, exact=True,
                         desc="exact kNN (ground truth, k=100) over SIFT-shaped synthetic 1M x 128 L2, 10k queries per step"),
    "sift200k": dict(n=200_000, dim=128, metric=0, M=16, efc=200, rank=14, nq=10_000, k=10, ef=100,
                     desc="SIFT-shaped synthetic 200kx128 L2 (dev size)"),
    "gist200k": dict(n=200_000, dim=960, metric=0, M=32, efc=200, rank=24, nq=10_000, k=10, ef=100, curve=True,
                     desc="GIST-shaped synthetic 200kx960 L2 (dev size; 768 MB of vectors, still >> L2)"),
    "msturing200k-slimq": dict(n=200_000, dim=96, metric=0, M=16, efc=200, rank=12, nq=10_000, k=10, ef=100,
                               kind="slimq", desc="MSTuring-shaped synthetic 200kx96 hnsw_slimq (dev size)"),
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def env_rank():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def prepare_inputs(w: dict, n_query_batches: int, build_rank: bool, reference_builder: bool = False,
                   deterministic: bool = False, device: int = 0):
    """Synthetic corpus + query batches + the .graph over the corpus (cached on disk).  The reference arm
    (reference_builder=True, `--impl reference`, which the driver runs first on a box) builds the hnsw_slim
    graph with the REFERENCE's own builder (addPoint loop + convertFromHNSW through oracle/_ref), so that both
    arms search the graph BASELINE.md specifies; the engine's arm never executes oracle/: it takes the cached
    file, or builds one with its own host builder (profiles/r02_refgraph_probe.txt: same recall and QPS on
    reference-built, host-built and GPU-built graphs).  deterministic=True (--dump-outputs): the .graph is the
    same file on every machine, cached under its own name: built by the GPU builder (levels drawn from a seed,
    atomics only for statistics) and saved with hs_save_index, or for hnsw_slimq by the host builder on one
    thread (its GPU path clusters on all host threads)."""
    from hnsw_slim_b200 import capi
    from hnsw_slim_b200.synth import latent_gaussian
    os.makedirs(CACHE, exist_ok=True)
    slimq = w.get("kind") == "slimq"
    tag = (f"n{w['n']}_d{w['dim']}_m{w['metric']}_r{w['rank']}_M{w['M']}_e{w['efc']}_b4_s1"
           + (("_t1" if slimq else "_gpu") if deterministic else ""))
    threads = 1 if deterministic else 0
    graph = os.path.join(CACHE, f"hnsw_{'slimq' if slimq else 'slim'}_{tag}.graph")
    base = None
    if slimq:      # the raw rows are part of a hnsw_slimq index (exact rerank, setDataset)
        base = latent_gaussian(w["n"], w["dim"], rank=w["rank"], seed=1)
    if not os.path.exists(graph) and build_rank:
        t0 = time.time()
        if base is None:
            base = latent_gaussian(w["n"], w["dim"], rank=w["rank"], seed=1, normalize=(w["metric"] == 1))
        t1 = time.time()
        tmp = graph + f".tmp{os.getpid()}"
        who = "engine host builder"
        if slimq:
            capi.build_slimq_graph(base, tmp, M=w["M"], ef_construction=w["efc"], branching="4", threads=threads)
        else:
            built = False
            if deterministic:
                gix = capi.Index.build_gpu(base, metric=w["metric"], M=w["M"], ef_construction=w["efc"], branching="4",
                                           device=device)
                gix.save(tmp)
                gix.close()
                built, who = True, "engine GPU builder (hs_build_slim_index_gpu, saved by hs_save_index)"
            if reference_builder and not deterministic:
                from oracle import refharness as rh
                if rh.ref_slim_path() is not None:
                    rh.ref_slim_build(base, tmp, metric=w["metric"], M=w["M"], ef_construction=w["efc"], branching="4")
                    built, who = True, "reference builder (oracle/_ref)"
            if not built:
                capi.build_slim_graph(base, tmp, metric=w["metric"], M=w["M"], ef_construction=w["efc"], branching="4",
                                      threads=threads)
        os.replace(tmp, graph)
        with open(graph + ".builder", "w") as f:
            f.write(who)
        log(f"[bench] generated corpus in {t1-t0:.1f}s, built {graph} with the {who} in {time.time()-t1:.1f}s "
            f"({os.cpu_count()} host threads)")
    queries = [latent_gaussian(w["nq"], w["dim"], rank=w["rank"], seed=1, normalize=(w["metric"] == 1),
                               stream=1 + b) for b in range(n_query_batches)]
    return graph, base, queries


def file_sha256(path: str) -> str:
    import hashlib
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 24), b""):
            h.update(blk)
    return h.hexdigest()


def index_sha256(ix) -> str:
    """Digest of an index that lives in HBM only (GPU-built): of the file hs_save_index writes for it."""
    import tempfile
    with tempfile.TemporaryDirectory(prefix="hs_bench_") as td:
        path = os.path.join(td, "index.graph")
        ix.save(path)
        return file_sha256(path)


def dump_outputs(out_dir: str, labels: np.ndarray, dists: np.ndarray, inputs: dict) -> None:
    """--dump-outputs: labels[nq,k] (ids, stored as float64: exact below 2**53), dists[nq,k] float32, and
    inputs.json with digests of the index and the query batch the step searched: a comparison of two runs
    refuses to compare outputs of different inputs."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "labels.npy"), labels.astype(np.float64))
    np.save(os.path.join(out_dir, "distances.npy"), dists.astype(np.float32))
    with open(os.path.join(out_dir, "inputs.json"), "w") as f:
        json.dump(inputs, f, indent=1, sort_keys=True)
    log(f"[bench] outputs of the last timed step ({labels.shape[0]} x {labels.shape[1]}) written to {out_dir}")


def query_sha256(q: np.ndarray) -> str:
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(q, dtype=np.float32).tobytes()).hexdigest()


def graph_builder_of(graph: str) -> str:
    try:
        with open(graph + ".builder") as f:
            return f.read().strip()
    except OSError:
        return "unknown (cached file)"


class ClockSampler:
    """Samples SM clock / throttle reasons through NVML during the timed region."""

    def __init__(self, device_index: int, interval_s: float = 0.004):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.interval_s = interval_s
        self.power_w = []
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.nv = None
            log(f"[bench] NVML unavailable: {e}")

    def _run(self):
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                self.power_w.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            self._stop.wait(self.interval_s)

    def __enter__(self):
        if self.nv and not os.environ.get("HS_BENCH_NO_SAMPLER"):
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "power_w_max": max(self.power_w) if self.power_w else None}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def cpu_reference_qps_slimq(graph: str, base: np.ndarray, w: dict, queries: np.ndarray, threads: int, passes: int):
    """hnsw_slimq: the reference's search is not re-entrant (member search_pool_, slimq.h:220,1814) and its
    strategy loops serially (hnsw_slimq_strategy.h:157-159): `threads` only applies to the plain-C port."""
    from oracle import refharness as rh
    if rh.ref_slimq_path() is not None:
        ix = rh.RefSlimQ(graph, base)
        ix.search(queries[:200], w["k"], w["ef"])
        t = 0.0
        for _ in range(passes):
            _, sec = ix.search(queries, w["k"], w["ef"])
            t += sec
        return len(queries) * passes / t, "reference", t, 1
    return None, "port", 0.0, 1


def cpu_port_qps_slimq(graph: str, base: np.ndarray, w: dict, queries: np.ndarray, t_const: float, threads: int):
    """The plain-C restatement (oracle/hs_oracle_slimq.c), one index shared by `threads` OpenMP threads."""
    from oracle import refharness as rh
    orc = rh.OracleQ(graph, base, t_const=t_const)
    orc.search(queries[:200], w["k"], w["ef"], order=rh.ORDER_REF, threads=threads)
    t0 = time.time()
    orc.search(queries, w["k"], w["ef"], order=rh.ORDER_REF, threads=threads)
    t = time.time() - t0
    return len(queries) / t, t


def cpu_reference_qps(graph: str, w: dict, queries: np.ndarray, threads: int, passes: int, budget_s: float = 0.0):
    """The reference's own search (oracle/_ref, compiled unmodified) on this host's cores.  Runs `passes`
    passes over `queries`, then keeps going until `budget_s` seconds of search time are spent; the rate is
    taken from the MEDIAN pass (host cores are shared with whatever else the box runs)."""
    from oracle import refharness as rh
    if rh.ref_slim_path() is not None:
        ix = rh.RefSlim(graph, w["dim"], w["n"], w["metric"])
        ix.search(queries[: min(2000, len(queries))], w["k"], w["ef"], threads)      # warm-up: per-thread visited lists
        times = []
        while len(times) < passes or (sum(times) < budget_s and len(times) < 400):
            _, sec, _ = ix.search(queries, w["k"], w["ef"], threads)
            times.append(sec)
        return len(queries) / float(np.median(times)), "reference", float(sum(times)), len(times)
    orc = rh.Oracle(graph, w["dim"], w["metric"])                              # plain-C port
    times = []
    while len(times) < passes or (sum(times) < budget_s and len(times) < 400):
        t0 = time.time()
        orc.search(queries, w["k"], w["ef"], order=rh.ORDER_REF, threads=threads if threads != 1 else 1)
        times.append(time.time() - t0)
    return len(queries) / float(np.median(times)), "port", float(sum(times)), len(times)


def run_reference(args, w):
    rank, _, world = env_rank()
    if rank != 0:
        return
    from oracle import refharness as rh
    graph, base, qb = prepare_inputs(w, 1, True, reference_builder=True)
    q = qb[0]
    cores = os.cpu_count() or 1
    slimq = w.get("kind") == "slimq"
    how = ("omp parallel for schedule(dynamic) over queries (hnsw_slim_client_update_patch.cc:223-226), "
           f"{cores} threads")
    if slimq:
        from hnsw_slim_b200 import capi
        if rh.ref_slimq_path():
            ix, orc, kind = "copies", None, "reference"
            how = (f"{cores} OpenMP threads, each searching its own copy of the index over one shared raw dataset "
                   "(one index copy per thread, BASELINE.md §2: the reference's hnsw_slimq search is not re-entrant, "
                   "member search_pool_, slimq.h:220,1814); copies are loaded once per step, outside the timed loop")
        else:
            pd = (w["dim"] + 63) // 64 * 64
            ix, orc, kind = None, rh.OracleQ(graph, base, t_const=capi.slimq_default_tconst(pd)), "port"
    else:
        ix = rh.RefSlim(graph, w["dim"], w["n"], w["metric"]) if rh.ref_slim_path() else None
        kind = "reference" if ix is not None else "port"
        orc = None if ix is not None else rh.Oracle(graph, w["dim"], w["metric"])

    def step():
        if ix is not None and slimq:
            return rh.ref_slimq_search_copies(graph, base, q, w["k"], w["ef"], threads=cores, passes=1)[1]
        if ix is not None:
            _, sec, _ = ix.search(q, w["k"], w["ef"], 0)         # omp dynamic, all cores
            return sec
        t0 = time.time()
        orc.search(q, w["k"], w["ef"], order=rh.ORDER_REF, threads=0)
        return time.time() - t0

    for _ in range(max(1, args.warmup)):
        step()
    total = sum(step() for _ in range(args.steps))
    qps = len(q) * args.steps / total
    sample = f"{args.steps} x {len(q)} queries, ef={w['ef']}, k={w['k']}, {how}"
    out = {
        "impl": "reference", "metric": "QPS at recall@10>=0.95", "value": qps, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["desc"], "k": w["k"], "ef_search": w["ef"], "queries_per_step": len(q),
                   "graph_built_by": graph_builder_of(graph)},
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


def run_gpu(args, w):
    import torch
    rank, local_rank, world = env_rank()
    from hnsw_slim_b200 import capi
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    distributed = world > 1
    if distributed:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    n_batches = min(8, args.warmup + args.steps)
    # rank 0 builds the graph (all host threads); the others wait, then read the cache
    if rank == 0:
        graph, base, qbatches = prepare_inputs(w, n_batches, True, deterministic=bool(args.dump_outputs),
                                               device=local_rank)
    barrier()
    if rank != 0:
        graph, base, qbatches = prepare_inputs(w, n_batches, False, deterministic=bool(args.dump_outputs))
    # each rank takes its own batches (different streams) in the replicated/weak-scaling mode
    if distributed:
        from hnsw_slim_b200.synth import latent_gaussian
        qbatches = [latent_gaussian(w["nq"], w["dim"], rank=w["rank"], seed=1, normalize=(w["metric"] == 1),
                                    stream=1 + b + 100 * rank) for b in range(n_batches)]

    t0 = time.time()
    slimq = w.get("kind") == "slimq"
    if slimq:
        ix = capi.Index(graph, w["dim"], kind=capi.HS_KIND_SLIMQ, raw_base=base, device=local_rank)
    else:
        ix = capi.Index(graph, w["dim"], metric=w["metric"], device=local_rank)
    ix.set_ef(w["ef"])
    ix.set_overlap(not args.no_overlap)
    info = ix.info()
    log(f"[bench] rank {rank}: index resident in {time.time()-t0:.1f}s, {info['device_bytes']/2**20:.0f} MiB HBM, "
        f"maxlevel {info['maxlevel']}, avg deg0 {info['sum_deg0']/info['n']:.2f}")

    nq, k, dim = w["nq"], w["k"], w["dim"]
    stream = torch.cuda.Stream()
    d_q = [torch.from_numpy(q).cuda() for q in qbatches]
    d_lab = torch.empty((nq, k), dtype=torch.int32, device="cuda")
    d_dist = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()

    def step(i):
        ix.search_device(d_q[i % n_batches].data_ptr(), nq, k, d_lab.data_ptr(), d_dist.data_ptr(), stream.cuda_stream)

    # ---- device-resident number ----
    for i in range(args.warmup):
        step(i)
    stream.synchronize()
    ix.reset_stats()
    barrier()
    # only the two bracketing events sit on the stream: an event between two launches would split
    # the programmatic-serialization edge that lets consecutive batches overlap (hs_set_overlap)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    clocks = ClockSampler(local_rank)
    barrier()
    with clocks:
        ev[0].record(stream)
        for i in range(args.steps):
            step(args.warmup + i)
        ev[1].record(stream)
        stream.synchronize()
    barrier()
    ms_total = ev[0].elapsed_time(ev[-1])
    if args.dump_outputs and rank == 0:      # before the sustained stream below reuses the buffers
        dump_outputs(args.dump_outputs, d_lab.cpu().numpy().view(np.uint32), d_dist.cpu().numpy(),
                     {"workload": args.workload, "k": k, "ef_search": w["ef"], "index_sha256": file_sha256(graph),
                      "queries_sha256": query_sha256(qbatches[(args.warmup + args.steps - 1) % n_batches])})
    st = ix.stats()
    if distributed:
        t = torch.tensor([ms_total], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    value = world * nq * args.steps / (ms_total * 1e-3)

    # ---- sustained: the same step back to back for about args.sustained seconds, with its own clock record
    #      (the K timed steps above are a ~20 ms burst; a long stream may clock and cache differently) ----
    sustained = None
    if args.sustained > 0:
        n_sus = max(args.steps, int(args.sustained * 1e3 / max(ms_total / args.steps, 1e-3)))
        sev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        clocks_s = ClockSampler(local_rank, 0.05)
        barrier()
        with clocks_s:
            sev[0].record(stream)
            for i in range(n_sus):
                step(args.warmup + args.steps + i)
            sev[1].record(stream)
            stream.synchronize()
        barrier()
        t = torch.tensor([sev[0].elapsed_time(sev[1])], device="cuda", dtype=torch.float64)
        if distributed:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sus_ms = float(t.item())
        sustained = {"value": world * nq * n_sus / (sus_ms * 1e-3), "unit": "queries/s", "steps": n_sus,
                     "ms_per_step": sus_ms / n_sus, "seconds": sus_ms * 1e-3, "clocks": clocks_s.summary()}

    # ---- roofline of the traversal kernel (the only kernel in the step) ----
    launch_ms = ev[0].elapsed_time(ev[-1]) / args.steps
    n_dist = st["n_dist"] / args.steps
    n_hops = st["n_hops"] / args.steps
    avg_deg0 = info["sum_deg0"] / info["n"]
    if slimq:
        # SURVEY.md §8(d): per estimate the code record (padded_dim/8 B code + 2 factors + cluster id = one
        # 32-byte record at padded_dim 128), per expansion the adjacency list and one raw row for the rerank
        n_rerank = st["n_rerank"] / args.steps
        alg_bytes = (n_dist * (info["padded_dim_q"] // 8 + 16) + n_rerank * 4 * info["dim_padded"]
                     + n_hops * (8 + 4 * avg_deg0))
    else:
        alg_bytes = n_dist * 4 * info["dim_padded"] + n_hops * (8 + 4 * avg_deg0)      # SURVEY.md §8(d)
    peaks, peak_src = measured_peaks()
    achieved = alg_bytes / (launch_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")     # dram bytes/launch from the committed ncu capture
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(args.workload, {}).get("dram_bytes_per_launch")
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": traffic, "peak_source": peak_src,
                "kernel": "hs::traverse_slimq_kernel" if slimq else "hs::traverse_kernel",
                "algorithmic_bytes_per_launch": alg_bytes,
                "dist_evals_per_query": n_dist / nq, "hops_per_query": n_hops / nq, "launch_ms": launch_ms}

    # ---- end to end through the host-buffer C-ABI calls (pinned host memory in, pinned host memory out) ----
    # Every step's queries start in pinned host memory and its results end there; the transfers happen inside
    # the timed region (the kernel reads/writes the mapped buffers over PCIe/C2C, or staged copies when
    # HS_ZERO_COPY=0).  Headline = a stream of batches with three in flight (hs_search_batch_submit/_wait_oldest, what a
    # server front end does); the strictly synchronous hs_search_batch call per step is reported beside it.
    h_q = [torch.from_numpy(q).pin_memory() for q in qbatches]
    depth = 3
    h_lab = [torch.empty((nq, k), dtype=torch.int32).pin_memory() for _ in range(depth)]
    h_dist = [torch.empty((nq, k), dtype=torch.float32).pin_memory() for _ in range(depth)]
    for i in range(args.warmup):
        ix.search_ptr(h_q[i % n_batches].data_ptr(), nq, k, h_lab[0].data_ptr(), h_dist[0].data_ptr())
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        ix.search_ptr(h_q[(args.warmup + i) % n_batches].data_ptr(), nq, k, h_lab[0].data_ptr(), h_dist[0].data_ptr())
    e2e_sync_s = time.perf_counter() - t0
    checksum = 0
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        if i >= depth:                                  # ring slot i % depth is being reused: its batch must be done
            ix.wait_oldest()
            checksum += int(h_lab[i % depth][0, 0])     # ... and is consumed on the host
        ix.submit_ptr(h_q[(args.warmup + i) % n_batches].data_ptr(), nq, k, h_lab[i % depth].data_ptr(),
                      h_dist[i % depth].data_ptr())
    ix.wait()
    e2e_s = time.perf_counter() - t0
    if distributed:
        t = torch.tensor([e2e_s, e2e_sync_s], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s, e2e_sync_s = float(t[0].item()), float(t[1].item())
    e2e = {"value": world * nq * args.steps / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": nq * dim * 4,
           "d2h_bytes_per_step": nq * k * 8,
           "timing": "host wall clock; hs_search_batch_submit / hs_search_batch_wait_oldest with three batches in flight, "
                     "pinned host buffers read/written in place by the kernel",
           "sync_value": world * nq * args.steps / e2e_sync_s,
           "sync_timing": "host wall clock around one synchronous hs_search_batch call per step"}

    # ---- recall of what was just measured (exact kNN on the GPU, outside the timed regions) ----
    recall = None
    if rank == 0 and not args.no_recall:
        if base is None:
            from hnsw_slim_b200.synth import latent_gaussian
            base = latent_gaussian(w["n"], dim, rank=w["rank"], seed=1, normalize=(w["metric"] == 1))
        ns = min(1000, nq)
        gt, _ = capi.bruteforce_knn(base, qbatches[0][:ns], k, metric=w["metric"], device=local_rank)
        lab, _ = ix.search(qbatches[0][:ns], k)
        recall = float(np.mean([len(set(a) & set(b)) / k for a, b in zip(lab, gt)]))

    # ---- the reference's CPU search on this host, bounded sample (rank 0, N=1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        if slimq:
            from oracle import refharness as rh
            if rh.ref_slimq_path() is not None and hasattr(rh.slimq_lib(), "refq_search_copies"):
                # all cores: one index copy per thread (BASELINE.md §2; the reference's slimq search is not re-entrant)
                _, sec, thr = rh.ref_slimq_search_copies(graph, base, qbatches[0], w["k"], w["ef"], threads=cores, passes=3)
                qps_1, _, secs1, _ = cpu_reference_qps_slimq(graph, base, w, qbatches[0][:2000], 1, 1)
                cpu = {"value": nq / sec, "unit": "queries/s", "cores": thr, "kind": "reference",
                       "sample": f"3 passes x {nq} queries of the same workload (median), {thr} OpenMP threads each searching "
                                 f"its OWN copy of the index over one shared raw dataset (the reference's hnsw_slimq "
                                 f"searchKnn is not re-entrant: member search_pool_, slimq.h:220,1814); its serial loop "
                                 f"(hnsw_slimq_strategy.h:157-159) on 2000 queries: {qps_1:.0f} queries/s"}
            else:
                qps_port, secs_p = cpu_port_qps_slimq(graph, base, w, qbatches[0], ix.query_tconst, cores)
                cpu = {"value": qps_port, "unit": "queries/s", "cores": cores, "kind": "port",
                       "sample": f"{nq} queries of the same workload, plain-C restatement, omp over queries ({secs_p:.1f}s)"}
        else:
            qps_all, kind, secs, np_all = cpu_reference_qps(graph, w, qbatches[0], 0, 4, budget_s=10.0)
            qps_1, _, secs1, _ = cpu_reference_qps(graph, w, qbatches[0][:2000], 1, 1)
            cpu = {"value": qps_all, "unit": "queries/s", "cores": cores, "kind": kind,
                   "sample": f"{np_all} passes x {nq} queries of the same workload, omp dynamic over queries, {cores} "
                             f"threads ({secs:.1f}s of search, rate of the median pass); serial 1-thread loop "
                             f"(hnsw_slim_strategy.h:112-114) on 2000 queries: {qps_1:.0f} queries/s"}

    # ---- the sharded path of the same run (north_star (4), BASELINE.json configs[3] shape): the driver's
    #      --gpus 1/2/4/8 runs thereby record its strong-scaling curve next to the replicated headline ----
    sharded = None
    if not args.no_sharded and args.workload == "sift1m":
        del ix, d_q, h_q
        torch.cuda.empty_cache()
        ws = dict(WORKLOADS["deep-sharded"])
        if args.shard_rows or args.shards:
            rows = args.shard_rows or ws["n"] // ws["shards"]
            ws["shards"] = args.shards or ws["shards"]
            ws["n"] = rows * ws["shards"]
            ws["desc"] = ws["desc"].replace("in 8 ", f"in {ws['shards']} ")
        sargs = argparse.Namespace(**vars(args))
        sargs.ef = None
        sargs.dump_outputs = None
        # the object times --steps steps like the headline (before, at least 200): at 8 GPUs a window of a few
        # ~0.3 ms steps is dominated by the ranks' start-up skew, so multi-GPU runs want a larger --steps
        try:
            sharded = measure_sharded(sargs, ws, rank, local_rank, world, dist if distributed else None)
        except Exception as e:          # the headline stands on its own; say why the object is missing
            log(f"[bench] rank {rank}: sharded measurement failed: {e!r}")
            sharded = {"error": repr(e)} if rank == 0 else None

    if rank == 0:
        out = {
            "metric": "QPS at recall@10>=0.95", "value": value, "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": w["desc"], "k": k, "ef_search": w["ef"], "queries_per_step_per_gpu": nq,
                       "parallelism": f"replicated index x{world}, queries split, no collective",
                       "recall_at_10": recall, "graph_built_by": graph_builder_of(graph),
                       "batch_overlap": (not args.no_overlap) and "hs_set_overlap: the next step's grid is launched with "
                                        "programmatic stream serialization and fills SMs while this step's last queries "
                                        "drain; ms_per_step = timed region / steps",
                       "l2": "index (vectors+adjacency) %.0f MiB > 126 MB L2; a different query batch every step"
                             % (info["device_bytes"] / 2**20)},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "sustained": sustained, "gpu_launches": args.steps,
            "clocks": clocks.summary(), "sharded": sharded,
        }
        print(json.dumps(out), flush=True)
    if distributed:
        dist.barrier()
        dist.destroy_process_group()


def run_gpu_bruteforce(args, w):
    """--workload bruteforce1m: a step = hs_bruteforce_knn_device over one 10k-query batch (BruteForce::solve's loop of
    BruteforceSearch::searchKnn, bruteforce.h:106-135, for a whole batch).  N GPUs: base replicated, queries split."""
    import torch
    rank, local_rank, world = env_rank()
    from hnsw_slim_b200 import capi
    from hnsw_slim_b200.synth import latent_gaussian
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    distributed = world > 1
    if distributed:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    n, dim, nq, k = w["n"], w["dim"], w["nq"], w["k"]
    n_batches = min(4, args.warmup + args.steps)
    base = latent_gaussian(n, dim, rank=w["rank"], seed=1)
    qb = [latent_gaussian(nq, dim, rank=w["rank"], seed=1, stream=1 + b + 100 * rank) for b in range(n_batches)]
    d_base = torch.from_numpy(base).cuda()
    d_q = [torch.from_numpy(q).cuda() for q in qb]
    d_lab = torch.empty((nq, k), dtype=torch.int32, device="cuda")
    d_dist = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    stream = torch.cuda.Stream()

    def step(i):
        capi.bruteforce_knn_device(d_base.data_ptr(), n, dim, d_q[i % n_batches].data_ptr(), nq, k, d_lab.data_ptr(),
                                   d_dist.data_ptr(), metric=w["metric"], stream=stream.cuda_stream)

    for i in range(args.warmup):
        step(i)
    stream.synchronize()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    clocks = ClockSampler(local_rank, 0.02)
    with clocks:
        ev[0].record(stream)
        for i in range(args.steps):
            step(args.warmup + i)
        ev[1].record(stream)
        stream.synchronize()
    barrier()
    ms_total = ev[0].elapsed_time(ev[1])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_lab.cpu().numpy().view(np.uint32), d_dist.cpu().numpy(),
                     {"workload": args.workload, "k": k, "base_sha256": query_sha256(base),
                      "queries_sha256": query_sha256(qb[(args.warmup + args.steps - 1) % n_batches])})
    if distributed:
        t = torch.tensor([ms_total], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    value = world * nq * args.steps / (ms_total * 1e-3)
    step_ms = ev[0].elapsed_time(ev[1]) / args.steps

    # end to end: host buffers in, host buffers out through hs_bruteforce_knn (base uploaded inside the call)
    h_lab = np.empty((nq, k), np.uint32)
    t0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 3))
    for i in range(e2e_steps):
        h_lab, _ = capi.bruteforce_knn(base, qb[i % n_batches], k, metric=w["metric"], device=local_rank)
    e2e_s = time.perf_counter() - t0
    e2e = {"value": world * nq * e2e_steps / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": (n + nq) * dim * 4,
           "d2h_bytes_per_step": nq * k * 8, "steps": e2e_steps,
           "timing": "host wall clock around hs_bruteforce_knn: pageable host base + queries in (the 512 MB base is "
                     "uploaded inside every call, as the reference's strategy re-reads its .fvecs), labels + distances out"}
    peaks, peak_src = measured_peaks()
    flop = 2.0 * n * nq * dim
    achieved = flop / (step_ms * 1e-3) / 1e12
    pipe = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            pipe = json.load(f).get("bruteforce1m")
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peaks.get("bf16_tflops", 1640.9), "unit": "TFLOP/s",
                "frac": achieved / peaks.get("bf16_tflops", 1640.9), "traffic": None, "peak_source": peak_src,
                "kernel": "hs::bf_tc_kernel (+ split / threshold / finish kernels inside the step)",
                "algorithmic_flop_per_step": flop, "step_ms": step_ms,
                "note": "algorithmic 2*n*nq*dim against the bf16 burst peak; the kernel issues 3x that in "
                        "tcgen05.mma.kind::tf32 work (hi.hi + hi.lo + lo.hi: bit-exact fp32 results need the split), "
                        "and the tf32 rate is half the bf16 rate",
                "tensor_pipe": pipe}
    recall = None
    cpu = None
    if rank == 0:
        # parity of what was measured: identical to the fp32 scan path on a sample (and, below, to the reference)
        ns = 64
        lab_tc, _ = capi.bruteforce_knn(base, qb[0][:ns], k, metric=w["metric"], device=local_rank)
        if world == 1 and not args.no_cpu_baseline:
            from oracle import refharness as rh
            cores = os.cpu_count() or 1
            if rh.ref_slim_path() is not None:
                ref_l, sec = rh.ref_bruteforce(base, qb[0][:256], k, metric=w["metric"], threads=0)
                same = float(np.mean([set(a) == set(b) for a, b in zip(ref_l[:ns], lab_tc)]))
                cpu = {"value": 256 / sec, "unit": "queries/s", "cores": cores, "kind": "reference",
                       "sample": f"256 queries of the same workload through the reference's BruteforceSearch::searchKnn under "
                                 f"omp ({sec:.1f}s; brute_force_strategy.h:24-36); k-sets identical to the engine's on "
                                 f"{same*100:.0f}% of the first {ns}"}
                recall = same
    if rank == 0:
        out = {
            "metric": "exact kNN QPS (k=100 ground-truth path)", "value": value, "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 (tf32x3 tensor-core prefilter + exact fp32 re-scoring)",
            "data": "synthetic",
            "config": {"workload": w["desc"], "k": k, "queries_per_step_per_gpu": nq,
                       "parallelism": f"replicated base x{world}, queries split, no collective",
                       "identical_to_reference": recall,
                       "l2": "base 512 MB > 126 MB L2; a different query batch every step"},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": args.steps,
            "clocks": clocks.summary(),
        }
        print(json.dumps(out), flush=True)
    if distributed:
        dist.barrier()
        dist.destroy_process_group()


def device_rows(n: int, dim: int, rank: int, normalize: bool, device: int):
    """n x dim rows of the latent model generated on the GPU (see shard_rows_device)."""
    w = {"n": n, "shards": 1, "dim": dim, "rank": rank}
    rows = shard_rows_device(w, 0, device)
    if normalize:
        rows /= rows.norm(dim=1, keepdim=True)
    return rows


def run_gpu_curve(args, w):
    """BASELINE.json configs[1] / [2] (GIST-shaped ef sweep, COHERE-shaped recall-QPS curve) on ONE GPU: rows
    generated on the GPU, index built on the GPU (hs_build_slim_index_gpu), an ef_search sweep with recall@10
    against exact kNN, and the headline fields for the smallest ef of the sweep that reaches recall >= 0.95;
    the reference's OpenMP search on the same graph (saved in saveIndex's format) beside it."""
    import torch
    from hnsw_slim_b200 import capi
    from hnsw_slim_b200.synth import latent_gaussian
    rank, local_rank, world = env_rank()
    if world != 1:
        raise SystemExit("bench.py: the curve workloads are single-GPU measurements (--gpus 1)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    n, dim, k, nq, metric = w["n"], w["dim"], w["k"], w["nq"], w["metric"]
    t0 = time.time()
    rows = device_rows(n, dim, w["rank"], metric == 1, local_rank)
    torch.cuda.synchronize()
    t1 = time.time()
    ix = capi.Index.build_gpu(None, base_ptr=rows.data_ptr(), n=n, dim=dim, metric=metric, M=w["M"],
                              ef_construction=w["efc"], branching="4", device=local_rank)
    t_build = time.time() - t1
    info = ix.info()
    log(f"[bench] {n}x{dim} rows generated on the GPU in {t1-t0:.1f}s, index built on the GPU in {t_build:.1f}s "
        f"({info['device_bytes']/2**20:.0f} MiB HBM, avg deg0 {info['sum_deg0']/n:.2f}, maxlevel {info['maxlevel']})")
    n_batches = min(8, args.warmup + args.steps)
    qb = [latent_gaussian(nq, dim, rank=w["rank"], seed=1, normalize=(metric == 1), stream=1 + b) for b in range(n_batches)]
    d_q = [torch.from_numpy(q).cuda() for q in qb]
    ns = min(1000, nq)
    gl = torch.empty((ns, k), dtype=torch.int32, device="cuda")
    capi.bruteforce_knn_device(rows.data_ptr(), n, dim, d_q[0].data_ptr(), ns, k, gl.data_ptr(), None, metric=metric,
                               stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    gt = gl.cpu().numpy().view(np.uint32)
    del rows
    torch.cuda.empty_cache()
    ix.set_overlap(not args.no_overlap)
    stream = torch.cuda.Stream()
    d_lab = torch.empty((nq, k), dtype=torch.int32, device="cuda")
    d_dist = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    peaks, peak_src = measured_peaks()
    avg_deg0 = info["sum_deg0"] / n

    def measure(ef, steps):
        ix.set_ef(ef)
        lab, _ = ix.search(qb[0][:ns], k)
        rec = float(np.mean([len(set(a) & set(b)) / k for a, b in zip(lab, gt)]))
        for i in range(args.warmup):
            ix.search_device(d_q[i % n_batches].data_ptr(), nq, k, d_lab.data_ptr(), d_dist.data_ptr(), stream.cuda_stream)
        stream.synchronize()
        ix.reset_stats()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clocks = ClockSampler(local_rank)
        torch.cuda.synchronize()
        with clocks:
            e0.record(stream)
            for i in range(steps):
                ix.search_device(d_q[(args.warmup + i) % n_batches].data_ptr(), nq, k, d_lab.data_ptr(), d_dist.data_ptr(),
                                 stream.cuda_stream)
            e1.record(stream)
            stream.synchronize()
        ms = e0.elapsed_time(e1)
        if args.dump_outputs:
            last_out[ef] = (d_lab.cpu().numpy().view(np.uint32), d_dist.cpu().numpy())
        st = ix.stats()
        alg = (st["n_dist"] * 4 * info["dim_padded"] + st["n_hops"] * (8 + 4 * avg_deg0)) / steps
        gbs = alg / (ms / steps * 1e-3) / 1e9
        return {"ef_search": ef, "recall_at_10": rec, "qps": nq * steps / (ms * 1e-3), "ms_per_step": ms / steps,
                "hbm_gbs_algorithmic": gbs, "frac": gbs / peaks["hbm_gbs"], "dist_evals_per_query": st["n_dist"] / steps / nq,
                "alg_bytes": alg, "clocks": clocks.summary()}

    efs = [args.ef] if args.ef else [50, 100, 200, 400]
    last_out = {}
    curve = [measure(ef, args.steps) for ef in efs]
    for c in curve:
        log(f"[bench] ef={c['ef_search']}: recall {c['recall_at_10']:.4f}, {c['qps']/1e6:.3f} M QPS, "
            f"{c['hbm_gbs_algorithmic']:.0f} GB/s algorithmic ({c['frac']:.2f} of peak)")
    ok = [c for c in curve if c["recall_at_10"] >= 0.95]
    head = min(ok, key=lambda c: c["ef_search"]) if ok else max(curve, key=lambda c: c["recall_at_10"])
    ef = head["ef_search"]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *last_out[ef],
                     {"workload": args.workload, "k": k, "ef_search": ef, "index_sha256": index_sha256(ix),
                      "queries_sha256": query_sha256(qb[(args.warmup + args.steps - 1) % n_batches])})

    # end to end: pinned host batches in, pinned host rows out, three batches in flight (as the headline workload)
    ix.set_ef(ef)
    h_q = [torch.from_numpy(q).pin_memory() for q in qb]
    depth = 3
    h_lab = [torch.empty((nq, k), dtype=torch.int32).pin_memory() for _ in range(depth)]
    h_dist = [torch.empty((nq, k), dtype=torch.float32).pin_memory() for _ in range(depth)]
    for i in range(args.warmup):
        ix.search_ptr(h_q[i % n_batches].data_ptr(), nq, k, h_lab[0].data_ptr(), h_dist[0].data_ptr())
    t0 = time.perf_counter()
    for i in range(args.steps):
        if i >= depth:
            ix.wait_oldest()
        ix.submit_ptr(h_q[(args.warmup + i) % n_batches].data_ptr(), nq, k, h_lab[i % depth].data_ptr(),
                      h_dist[i % depth].data_ptr())
    ix.wait()
    e2e_s = time.perf_counter() - t0
    e2e = {"value": nq * args.steps / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": nq * dim * 4,
           "d2h_bytes_per_step": nq * k * 8,
           "timing": "host wall clock; hs_search_batch_submit / _wait_oldest, three batches in flight, pinned host buffers"}

    cpu = None
    if not args.no_cpu_baseline:
        try:
            from oracle import refharness as rh
            if rh.ref_slim_path() is not None:
                os.makedirs(CACHE, exist_ok=True)
                path = os.path.join(CACHE, f"gpu_built_{args.workload}_{os.getpid()}.graph")
                ix.save(path)
                ref = rh.RefSlim(path, dim, n, metric)
                qs = qb[0][:2000]
                ref.search(qs[:500], k, ef, 0)
                times = []
                while sum(times) < 10.0 and len(times) < 100:
                    _, sec, _ = ref.search(qs, k, ef, 0)
                    times.append(sec)
                ref.close()
                os.remove(path)
                cores = os.cpu_count() or 1
                cpu = {"value": len(qs) / float(np.median(times)), "unit": "queries/s", "cores": cores, "kind": "reference",
                       "sample": f"{len(times)} passes x {len(qs)} queries at ef={ef} on the same graph (saved by "
                                 f"hs_save_index, loaded by the reference's loadIndex), omp dynamic over queries, {cores} threads"}
        except Exception as e:
            log(f"[bench] CPU baseline failed: {e!r}")
    out = {
        "metric": "QPS at recall@10>=0.95", "value": head["qps"], "unit": "queries/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["desc"], "k": k, "ef_search": ef, "queries_per_step": nq,
                   "recall_at_10": head["recall_at_10"], "reached_0.95": bool(ok),
                   "curve": [{kk: c[kk] for kk in ("ef_search", "recall_at_10", "qps", "hbm_gbs_algorithmic", "frac",
                                                    "dist_evals_per_query")} for c in curve],
                   "graph_built_by": f"hs_build_slim_index_gpu in {t_build:.1f}s (rows generated on the GPU)",
                   "l2": "index %.0f MiB >> 126 MB L2; a different query batch every step" % (info["device_bytes"] / 2**20)},
        "roofline": {"bound": "hbm", "achieved": head["hbm_gbs_algorithmic"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": head["frac"], "traffic": None, "peak_source": peak_src, "kernel": "hs::traverse_kernel",
                     "algorithmic_bytes_per_launch": head["alg_bytes"]},
        "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": args.steps, "clocks": head["clocks"],
    }
    print(json.dumps(out), flush=True)


def shard_paths(w: dict):
    fam = "hnsw_slimq" if w.get("kind") == "slimq" else "hnsw_slim"
    return [os.path.join(CACHE, f"{fam}_shard{s}of{w['shards']}_n{w['n']}_d{w['dim']}_r{w['rank']}_M{w['M']}"
                                f"_e{w['efc']}_b4_s1_v2.graph") for s in range(w["shards"])]


def shard_rows(w: dict, s: int) -> np.ndarray:
    """Rows of shard s of the sharded corpus (chunk-addressable generator: only this shard is drawn)."""
    from hnsw_slim_b200 import sharding
    from hnsw_slim_b200.synth import latent_gaussian_rows
    lo, hi = sharding.shard_ranges(w["n"], w["shards"])[s]
    return latent_gaussian_rows(lo, hi, w["dim"], rank=w["rank"], seed=1)


def prepare_shards(w: dict, my_shards, threads: int):
    """Shard graphs with GLOBAL labels (label = row index in the full corpus), cached on disk."""
    from hnsw_slim_b200 import capi, sharding
    os.makedirs(CACHE, exist_ok=True)
    ranges = sharding.shard_ranges(w["n"], w["shards"])
    slimq = w.get("kind") == "slimq"
    paths = shard_paths(w)
    raws = []
    for s in my_shards:
        rows = None
        if not os.path.exists(paths[s]):
            lo, hi = ranges[s]
            t0 = time.time()
            rows = shard_rows(w, s)
            tmp = paths[s] + f".tmp{os.getpid()}"
            if slimq:
                capi.build_slimq_graph(rows, tmp, M=w["M"], ef_construction=w["efc"], branching="4",
                                       threads=threads, labels=np.arange(lo, hi, dtype=np.uint64))
            else:
                capi.build_slim_graph(rows, tmp, metric=w["metric"], M=w["M"], ef_construction=w["efc"],
                                      branching="4", threads=threads, labels=np.arange(lo, hi, dtype=np.uint64))
            os.replace(tmp, paths[s])
            log(f"[bench] built shard {s} [{lo},{hi}) in {time.time()-t0:.1f}s with {threads} threads")
        if slimq:
            raws.append(rows if rows is not None else shard_rows(w, s))
    return paths, (raws if slimq else None)


def sharded_queries(w: dict, n_batches: int):
    from hnsw_slim_b200.synth import latent_gaussian_rows
    return [latent_gaussian_rows(0, w["nq"], w["dim"], rank=w["rank"], seed=1, stream=1 + b) for b in range(n_batches)]


def sharded_ground_truth(w: dict, q: np.ndarray, k: int, device: int):
    """Exact top-k over the whole sharded corpus, shard by shard on the GPU (hs_bruteforce_knn), merged on the
    host: the corpus never has to exist in one piece."""
    from hnsw_slim_b200 import capi, sharding
    ranges = sharding.shard_ranges(w["n"], w["shards"])
    labs, dsts = [], []
    for s, (lo, hi) in enumerate(ranges):
        l, d = capi.bruteforce_knn(shard_rows(w, s), q, k, metric=w["metric"], device=device)
        labs.append(l.astype(np.int64) + lo)
        dsts.append(d)
    lab, dst = np.concatenate(labs, 1), np.concatenate(dsts, 1)
    order = np.argsort(dst, axis=1, kind="stable")[:, :k]       # shards are in label order: ties -> smaller label
    return np.take_along_axis(lab, order, 1).astype(np.uint32)


def shard_rows_device(w: dict, s: int, device: int):
    """Rows of shard s generated ON the GPU (torch's Philox stream, one generator per 65536-row chunk, the
    latent model of synth.py with the same mixing matrix): the 100M-shaped corpora never touch the host.
    Deterministic in (row, dim, rank, seed) for this torch build, whatever the number of ranks."""
    import torch
    from hnsw_slim_b200 import sharding
    lo, hi = sharding.shard_ranges(w["n"], w["shards"])[s]
    chunk = 1 << 16
    dev = torch.device("cuda", device)
    A = torch.from_numpy(np.random.default_rng(1).standard_normal((w["rank"], w["dim"])).astype(np.float32)).to(dev)
    out = torch.empty((hi - lo, w["dim"]), dtype=torch.float32, device=dev)
    g = torch.Generator(device=dev)
    for c in range(lo // chunk, (hi + chunk - 1) // chunk):
        g.manual_seed(0x5EED0000 + c)
        z = torch.randn((chunk, w["rank"]), generator=g, device=dev)
        eps = torch.randn((chunk, w["dim"]), generator=g, device=dev)
        rows = torch.addmm(eps * 0.1, z, A)
        a, b = max(lo, c * chunk), min(hi, (c + 1) * chunk)
        out[a - lo: b - lo] = rows[a - c * chunk: b - c * chunk]
    return out


def build_shards_gpu(w: dict, my_shards, device: int, gt_queries, k: int, slimq: bool = False):
    """This rank's shards built on its GPU (hs_build_slim_index_gpu) from device-generated rows, plus — while
    the rows are at hand — the shard-local exact top-k of `gt_queries` for the recall of the merged result."""
    import torch
    from hnsw_slim_b200 import capi, sharding
    ranges = sharding.shard_ranges(w["n"], w["shards"])
    shards, gt_parts = [], []
    d_gq = torch.from_numpy(gt_queries).cuda() if gt_queries is not None else None
    for s in my_shards:
        lo, hi = ranges[s]
        t0 = time.time()
        rows = shard_rows_device(w, s, device)
        torch.cuda.synchronize()
        t1 = time.time()
        if d_gq is not None:
            ns = d_gq.shape[0]
            gl = torch.empty((ns, k), dtype=torch.int32, device="cuda")
            gd = torch.empty((ns, k), dtype=torch.float32, device="cuda")
            capi.bruteforce_knn_device(rows.data_ptr(), hi - lo, w["dim"], d_gq.data_ptr(), ns, k, gl.data_ptr(),
                                       gd.data_ptr(), metric=w["metric"], stream=torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            gt_parts.append((gl.cpu().numpy().view(np.uint32).astype(np.int64) + lo, gd.cpu().numpy()))
        t2 = time.time()
        ix = capi.Index.build_gpu(None, base_ptr=rows.data_ptr(), n=hi - lo, dim=w["dim"], metric=w["metric"], M=w["M"],
                                  ef_construction=w["efc"], branching="4", labels=np.arange(lo, hi, dtype=np.uint64),
                                  device=device, kind=capi.HS_KIND_SLIMQ if slimq else capi.HS_KIND_SLIM)
        del rows
        torch.cuda.empty_cache()
        log(f"[bench] shard {s} [{lo},{hi}): rows generated on the GPU in {t1-t0:.1f}s, exact top-k {t2-t1:.1f}s, "
            f"index built on the GPU in {time.time()-t2:.1f}s")
        shards.append(ix)
    return shards, gt_parts


def merge_ground_truth(parts, k: int):
    """[(labels[ns,k] int64 global, dists[ns,k])] over all shards -> exact global top-k labels."""
    lab = np.concatenate([p[0] for p in parts], 1)
    dst = np.concatenate([p[1] for p in parts], 1)
    order = np.argsort(dst, axis=1, kind="stable")[:, :k]        # parts arrive in label order: ties -> smaller label
    return np.take_along_axis(lab, order, 1).astype(np.uint32)


EF_LADDER = [10, 12, 16, 20, 24, 28, 32, 40, 48, 64, 80, 100, 128, 200]


def measure_sharded(args, w, rank, local_rank, world, dist):
    """The sharded path (north_star (4)): S sub-graphs over N ranks, every rank searches the whole batch on
    its shards, rows are exchanged by the traversal kernels (hs_shardgroup) or one NCCL all-gather, top-k
    merge.  Total work is fixed => strong scaling.  Returns the result dict (rank 0) or None."""
    import torch
    from hnsw_slim_b200 import capi, sharding

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    slimq = w.get("kind") == "slimq"
    w = dict(w, desc=w["desc"].format(n=w["n"], rows=w["n"] // w["shards"]))
    mine = sharding.shards_of_rank(w["shards"], rank, world)
    nq, k = w["nq"], w["k"]
    n_batches = min(8, args.warmup + args.steps)
    qb = sharded_queries(w, n_batches)
    ns = min(1000, nq)
    builder = args.builder
    t_build = time.time()
    paths, gt = None, None
    if builder == "gpu":
        shards, gt_parts = build_shards_gpu(w, mine, local_rank, None if args.no_recall else qb[0][:ns], k, slimq)
        if not args.no_recall:
            if world > 1:
                allp = [None] * world
                dist.all_gather_object(allp, gt_parts)
                gt_parts = [p for rp in allp for p in rp]
            gt = merge_ground_truth(gt_parts, k) if rank == 0 else None
        barrier()
        t_build = time.time() - t_build
        ix = sharding.ShardedIndex.from_indices(shards, w["dim"], device=local_rank)
    else:
        paths, raws = prepare_shards(w, mine, max(1, (os.cpu_count() or 1) // world))
        barrier()
        t_build = time.time() - t_build
        ix = sharding.ShardedIndex([paths[s] for s in mine], w["dim"], metric=w["metric"], device=local_rank,
                                   kind=capi.HS_KIND_SLIMQ if slimq else capi.HS_KIND_SLIM, raw_bases=raws)
        if rank == 0 and not args.no_recall:
            gt = sharded_ground_truth(w, qb[0][:ns], k, local_rank)
    # a rank that stops submitting leaves the others waiting for its flags: bound every GPU phase
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("HS_BENCH_WATCHDOG_S", "240")), exit=True)
    d_q = [torch.from_numpy(q).cuda() for q in qb]
    depth = 4
    fused = args.exchange == "fused"
    if fused:       # rows go straight into every rank's gather table (peer memory); flags instead of a collective
        try:
            ix.connect(rank, world, nq, k, depth=depth)
        except Exception as e:      # raised on every rank (connect is collective): fall back to the NCCL exchange
            log(f"[bench] rank {rank}: fused exchange unavailable ({e}); using NCCL all-gather")
            fused = False
        barrier()
    ring = 2 * depth
    outs = [(torch.empty((nq, k), dtype=torch.int32, device="cuda"), torch.empty((nq, k), device="cuda"))
            for _ in range(ring)]

    def step(i):
        if fused:
            ix.submit(d_q[i % n_batches].data_ptr(), nq, outs[i % ring][0].data_ptr(), outs[i % ring][1].data_ptr())
            return outs[i % ring]
        return ix.search(d_q[i % n_batches], nq, k, exchange="nccl")

    # ---- per-shard ef: the smallest rung of the ladder whose recall@10 of the MERGED result is >= 0.95 ----
    ef, recall, ladder = w["ef"], None, []
    if args.ef is None and not args.no_recall:
        for ef in EF_LADDER:
            ix.set_ef(ef)
            out = step(0)
            ix.join()
            torch.cuda.synchronize()
            ok = torch.zeros(1, device="cuda")
            if rank == 0:
                lab = out[0][:ns].cpu().numpy().view(np.uint32)
                recall = float(np.mean([len(set(a) & set(b)) / k for a, b in zip(lab, gt)]))
                ladder.append((ef, round(recall, 4)))
                ok += float(recall >= 0.95)
            if world > 1:
                dist.broadcast(ok, 0)
            if ok.item() > 0:
                break
    ix.set_ef(ef)
    if rank == 0:
        log(f"[bench] sharded: {w['shards']} shards over {world} GPUs, per-shard ef {ef}, recall ladder {ladder}")

    for i in range(args.warmup):
        out = step(i)
    ix.join()
    for s_ in ix.shards:
        s_.reset_stats()
    barrier()
    if fused:
        ss, ms_ = ix.group.streams()
        s0, s1 = torch.cuda.ExternalStream(ss), torch.cuda.ExternalStream(ms_)
    else:
        s0 = s1 = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clocks = ClockSampler(local_rank)       # NVML start-up happens before the barrier, not inside the timed region
    barrier()
    with clocks:
        e0.record(s0)
        for i in range(args.steps):
            out = step(args.warmup + i)
        if not fused:
            ix.join()
        e1.record(s1)               # the merge stream: behind the last batch's merge
        ix.join()
        torch.cuda.synchronize()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        digests = [file_sha256(paths[s]) if paths is not None else index_sha256(s_) for s, s_ in zip(mine, ix.shards)]
        dump_outputs(args.dump_outputs, out[0].cpu().numpy().view(np.uint32), out[1].cpu().numpy(),
                     {"workload": args.workload, "k": k, "ef_search_per_shard": ef, "shards": w["shards"],
                      "rows_per_shard": w["n"] // w["shards"], "builder": builder, "shard_index_sha256": digests,
                      "queries_sha256": query_sha256(qb[(args.warmup + args.steps - 1) % n_batches])})
    if rank == 0:
        log(f"[bench] sharded: {args.steps} steps in {ms:.2f} ms on rank 0")
    stats = [s_.stats() for s_ in ix.shards]          # counters of the K timed steps (before the sustained stream)
    infos = [s_.info() for s_ in ix.shards]
    # ---- sustained: the same step, back to back for about args.sustained seconds (its own clock record) ----
    sustained = None
    if args.sustained > 0:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        if world > 1:               # every rank must submit the SAME number of batches
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        n_sus = max(args.steps, int(args.sustained * 1e3 / max(float(t.item()) / args.steps, 1e-3)))
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clocks_s = ClockSampler(local_rank, 0.05)
        barrier()
        with clocks_s:
            f0.record(s0)
            for i in range(n_sus):
                step(args.warmup + args.steps + i)
            if not fused:
                ix.join()
            f1.record(s1)
            ix.join()
            torch.cuda.synchronize()
        barrier()
        t = torch.tensor([f0.elapsed_time(f1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sustained = {"value": nq * n_sus / (float(t.item()) * 1e-3), "unit": "queries/s", "steps": n_sus,
                     "ms_per_step": float(t.item()) / n_sus, "seconds": float(t.item()) * 1e-3,
                     "clocks": clocks_s.summary()}
    if rank == 0 and gt is not None:
        b_last = (args.warmup + args.steps - 1) % n_batches
        if b_last == 0:
            lab = out[0][:ns].cpu().numpy().view(np.uint32)
            recall = float(np.mean([len(set(a) & set(b)) / k for a, b in zip(lab, gt)]))
    if slimq:
        alg = sum(st["n_dist"] * (inf["padded_dim_q"] // 8 + 16) + st["n_rerank"] * 4 * inf["dim_padded"]
                  + st["n_hops"] * (8 + 4 * inf["sum_deg0"] / inf["n"]) for st, inf in zip(stats, infos)) / args.steps
    else:
        alg = sum(st["n_dist"] * 4 * inf["dim_padded"] + st["n_hops"] * (8 + 4 * inf["sum_deg0"] / inf["n"])
                  for st, inf in zip(stats, infos)) / args.steps
    evals = sum(st["n_dist"] for st in stats) / args.steps / nq

    # ---- end to end: the batch starts in pinned host memory on every rank (the "broadcast" of north_star:
    #      each rank's kernels read it in place) and the merged rows end in pinned host memory ----
    e2e = None
    if fused:
        h_q = [torch.from_numpy(q).pin_memory() for q in qb]
        h_out = [(torch.empty((nq, k), dtype=torch.int32).pin_memory(), torch.empty((nq, k)).pin_memory())
                 for _ in range(ring)]
        for i in range(args.warmup):
            ix.submit(h_q[i % n_batches].data_ptr(), nq, h_out[i % ring][0].data_ptr(), h_out[i % ring][1].data_ptr())
        ix.join()
        barrier()
        t0 = time.perf_counter()
        checksum = 0
        for i in range(args.steps):
            if i >= depth:                       # keep `depth` batches in flight; consume the oldest on the host
                ix.group.wait_oldest()
                checksum += int(h_out[(i - depth) % ring][0][0, 0])
            ix.submit(h_q[(args.warmup + i) % n_batches].data_ptr(), nq, h_out[i % ring][0].data_ptr(),
                      h_out[i % ring][1].data_ptr())
        ix.join()
        e2e_s = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t.item())
        e2e = {"value": nq * args.steps / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": nq * w["dim"] * 4 * len(mine),
               "d2h_bytes_per_step": nq * k * 8,
               "timing": f"host wall clock, max over ranks; hs_shardgroup_submit / _wait_oldest with {depth} batches in "
                         "flight; every rank's kernels read the pinned host batch in place (once per local shard) and "
                         "its merge kernel writes the rows to pinned host memory"}
    if world > 1:
        t = torch.tensor([ms, alg], device="cuda", dtype=torch.float64)
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        ms, alg_total = float(tmax[0]), float(t[1])
        evals_t = torch.tensor([evals], device="cuda", dtype=torch.float64)
        dist.all_reduce(evals_t, op=dist.ReduceOp.SUM)
        evals = float(evals_t.item())
    else:
        alg_total = alg

    # ---- the reference's CPU search on ONE shard (rank 0, N=1 only; bounded sample) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not slimq:
        try:
            if paths is None:           # GPU-built shards live in HBM only: write shard 0 in saveIndex's format
                os.makedirs(CACHE, exist_ok=True)
                paths = [os.path.join(CACHE, f"gpu_built_shard0_{os.getpid()}.graph")]
                ix.shards[0].save(paths[0])
            cpu = cpu_sharded_baseline(w, paths, qb[0], ef, budget_s=8.0)
        except Exception as e:
            log(f"[bench] CPU baseline of the sharded workload failed: {e!r}")
        finally:
            if builder == "gpu" and paths and os.path.exists(paths[0]):
                os.remove(paths[0])
    ix.close()
    faulthandler.cancel_dump_traceback_later()
    if rank != 0:
        return None
    peaks, peak_src = measured_peaks()
    per_gpu = alg_total / world / (ms / args.steps * 1e-3) / 1e9
    rows = w["n"] // w["shards"]
    return {
        "metric": "QPS at recall@10>=0.95", "value": nq * args.steps / (ms * 1e-3), "unit": "queries/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["desc"], "k": k, "ef_search_per_shard": ef, "queries_per_step": nq,
                   "shards": w["shards"], "rows_per_shard": rows, "shards_per_gpu": len(mine),
                   "exchange": ("fused: rows stored into every rank's gather table by the traversal kernels (peer memory "
                                "over NVLink), flags raised by the last warp of a batch, merge kernel on a second stream; "
                                f"up to {depth} batches in flight, no collective" if fused else
                                "nccl: one all_gather(nq*k*8 B per rank) + hs_topk_merge_device per batch"),
                   "recall_at_10": recall, "ef_ladder": ladder, "dist_evals_per_query_all_shards": evals,
                   "graph_build_s": round(t_build, 1),
                   "graph_builder": (("hs_build_slimq_index_gpu" if slimq else "hs_build_slim_index_gpu") +
                                     ": rows generated and indexed on each rank's GPU (HNSW build + convertFromHNSW"
                                     + (" + RaBitQ codes" if slimq else "") + " on the device)" if builder == "gpu" else
                                     "host builder (hs_build_slim_graph / hs_build_slimq_graph), cached .graph files"),
                   "l2": "each shard (%.0f MB of rows) vs 126 MB L2; a different query batch every step"
                         % (rows * w["dim"] * 4 / 1e6)},
        "roofline": {"bound": "hbm", "achieved": per_gpu, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": per_gpu / peaks["hbm_gbs"], "traffic": None, "peak_source": peak_src,
                     "kernel": ("hs::traverse_slimq_kernel" if slimq else "hs::traverse_kernel")
                               + " (per GPU, algorithmic bytes of all local shard launches / whole step incl. merge)"},
        "cpu_baseline": cpu, "e2e": e2e, "sustained": sustained, "gpu_launches": args.steps * (len(mine) + 1),
        "clocks": clocks.summary(),
    }


def cpu_sharded_baseline(w, paths, queries, ef, budget_s):
    """The reference's OpenMP search on shard 0 alone; a query of the sharded corpus visits all S shards, so the
    whole-corpus rate of the same algorithm on this host is that rate / S."""
    from oracle import refharness as rh
    cores = os.cpu_count() or 1
    rows = w["n"] // w["shards"]
    if rh.ref_slim_path() is None:
        return None
    ix = rh.RefSlim(paths[0], w["dim"], rows, w["metric"])
    qs = queries[:2000]
    ix.search(qs, w["k"], ef, 0)
    times = []
    while sum(times) < budget_s and len(times) < 200:
        _, sec, _ = ix.search(qs, w["k"], ef, 0)
        times.append(sec)
    shard_qps = len(qs) / float(np.median(times))
    return {"value": shard_qps / w["shards"], "unit": "queries/s", "cores": cores, "kind": "reference",
            "sample": f"{len(times)} passes x {len(qs)} queries on shard 0 of {w['shards']} ({rows} rows) at ef={ef}, omp dynamic "
                      f"over queries, {cores} threads: {shard_qps:.0f} queries/s on one shard; every query visits all "
                      f"{w['shards']} shards, so the corpus rate is 1/{w['shards']} of it"}


def run_gpu_sharded(args, w):
    import torch
    import torch.distributed as dist
    rank, local_rank, world = env_rank()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    line = measure_sharded(args, w, rank, local_rank, world, dist)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="sift1m", choices=sorted(WORKLOADS))
    ap.add_argument("--ef", type=int, default=None)
    ap.add_argument("--no-recall", action="store_true")
    ap.add_argument("--no-overlap", action="store_true",
                    help="do not let consecutive batches overlap on the stream (hs_set_overlap off)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--builder", default="gpu", choices=["gpu", "host"],
                    help="sharded workloads: build the shard graphs on the GPU (default) or with the host builder")
    ap.add_argument("--shards", type=int, default=None, help="sharded workloads: number of sub-graphs (default 8)")
    ap.add_argument("--sustained", type=float, default=2.0,
                    help="seconds of the back-to-back stream reported as \"sustained\" (0: skip)")
    ap.add_argument("--shard-rows", type=int, default=None,
                    help="sharded workloads: rows per shard (default: the workload's n / shards)")
    ap.add_argument("--exchange", default="fused", choices=["nccl", "fused"],
                    help="sharded workloads: NCCL all-gather, or the exchange fused into the traversal kernels")
    ap.add_argument("--no-sharded", action="store_true",
                    help="default workload: skip the embedded deep-sharded measurement (\"sharded\" object)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the labels and distances of the last timed step to DIR/labels.npy, DIR/distances.npy, "
                         "digests of its inputs to DIR/inputs.json; host-built graphs are then built single-threaded")
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("bench.py: --steps must be at least 1")
    args.warmup = max(3, args.warmup) if args.impl == "ours" else max(1, args.warmup)
    w = dict(WORKLOADS[args.workload])
    if args.ef:
        w["ef"] = args.ef
    if "shards" in w and (args.shard_rows or args.shards):
        rows = args.shard_rows or w["n"] // w["shards"]
        w["shards"] = args.shards or w["shards"]
        w["n"] = rows * w["shards"]
        w["desc"] = w["desc"].replace("in 8 ", f"in {w['shards']} ")
    if args.impl == "reference" and w.get("exact"):
        raise SystemExit("bench.py: --impl reference is defined for the graph-search workloads; the exact-kNN workload "
                         "times the reference's brute force inside its own line (cpu_baseline)")
    if args.dump_outputs and args.impl == "reference":
        raise SystemExit("bench.py: --dump-outputs is defined for the engine (--impl ours)")
    if args.impl == "reference":
        run_reference(args, w)
    elif w.get("exact"):
        run_gpu_bruteforce(args, w)
    elif "shards" in w:
        run_gpu_sharded(args, w)
    elif w.get("curve") and args.builder == "gpu":
        run_gpu_curve(args, w)
    else:
        run_gpu(args, w)


if __name__ == "__main__":
    main()
