"""Saves GPU-built hnsw_slimq indices with hs_save_index and measures the round trip.

Per size: hs_build_slimq_index_gpu, hs_save_index, hs_load of the saved file with the same rows; the reloaded
index must return the in-memory index's labels, distance bits and per-query counters on every query.  Reports
build, save and load seconds, the file size, and the card's name and power limit.  With --cpu-baseline it also
builds the host builder's file for the same rows and times the C oracle port (oracle/hs_oracle_slimq.c, all
cores) on both files, and the reference's own search (single-threaded, as its strategy runs) where oracle/_ref
is built: the CPU baseline on GPU-built files.

    python tools/slimq_save_probe.py --n 1000000 --cpu-baseline
    python tools/slimq_save_probe.py --n 12500000
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hnsw_slim_b200 import capi  # noqa: E402
from hnsw_slim_b200.synth import latent_gaussian_rows  # noqa: E402
from oracle import refharness as rh  # noqa: E402


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power = (s.strip() for s in out.split(","))
    return {"gpu": name, "power_limit": power}


def cpu_qps(graph, base, q, k, ef, t_const):
    """(C oracle port queries/s on all cores, reference queries/s on one thread or None)"""
    orc = rh.OracleQ(graph, base, t_const=t_const)
    orc.search(q[:500], k, ef, order=rh.ORDER_REF, threads=0)
    t0 = time.time()
    orc.search(q, k, ef, order=rh.ORDER_REF, threads=0)
    port = len(q) / (time.time() - t0)
    ref = None
    if rh.ref_slimq_path() is not None:
        r = rh.RefSlimQ(graph, base)
        r.t_const = t_const
        r.search(q[:200], k, ef)
        _, sec = r.search(q, k, ef)
        ref = len(q) / sec
    return port, ref


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=96)
    ap.add_argument("--rank", type=int, default=12)
    ap.add_argument("--M", type=int, default=16)
    ap.add_argument("--efc", type=int, default=200)
    ap.add_argument("--clusters", type=int, default=16)
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--efs", default="10,100,300")
    ap.add_argument("--cpu-baseline", action="store_true")
    ap.add_argument("--tmp", default=None, help="directory for the .graph files (default: the system temp dir)")
    ap.add_argument("--out", default=None, help="also append the JSON result line to this file")
    a = ap.parse_args()
    res = {"n": a.n, "dim": a.dim, "M": a.M, "efc": a.efc, "clusters": a.clusters, **card()}
    base = latent_gaussian_rows(0, a.n, a.dim, rank=a.rank, seed=1)
    q = latent_gaussian_rows(0, a.nq, a.dim, rank=a.rank, seed=1, stream=1)
    with tempfile.TemporaryDirectory(dir=a.tmp) as td:
        path = os.path.join(td, "gpu.graph")
        t0 = time.time()
        gpu = capi.Index.build_gpu(base, kind=capi.HS_KIND_SLIMQ, M=a.M, ef_construction=a.efc,
                                   num_cluster=a.clusters)
        res["build_s"] = time.time() - t0
        t0 = time.time()
        gpu.save(path)
        res["save_s"] = time.time() - t0
        res["file_bytes"] = os.path.getsize(path)
        t0 = time.time()
        again = capi.Index(path, a.dim, kind=capi.HS_KIND_SLIMQ, raw_base=base)
        res["load_s"] = time.time() - t0
        assert again.info()["device_bytes"] == gpu.info()["device_bytes"]
        for ef in (int(e) for e in a.efs.split(",")):
            for k in sorted({a.k, ef}):
                gpu.set_ef(ef)
                again.set_ef(ef)
                la, da, ca = gpu.search(q, k, counts=True)
                lb, db, cb = again.search(q, k, counts=True)
                same = (np.array_equal(la, lb) and np.array_equal(da.view(np.uint32), db.view(np.uint32))
                        and np.array_equal(ca, cb))
                res[f"identical_ef{ef}_k{k}"] = bool(same)
                if not same:
                    raise SystemExit(f"saved index differs from the in-memory one at ef={ef} k={k}: {res}")
        t_const = gpu.query_tconst
        del gpu, again
        if a.cpu_baseline:
            host = os.path.join(td, "host.graph")
            t0 = time.time()
            capi.build_slimq_graph(base, host, M=a.M, ef_construction=a.efc, num_cluster=a.clusters)
            res["host_build_s"] = time.time() - t0
            res["cpu_threads"] = os.cpu_count()
            for name, g in (("gpu_built", path), ("host_built", host)):
                port, ref = cpu_qps(g, base, q, a.k, 100, t_const)
                res[f"port_qps_{name}"] = port
                res[f"ref_qps_{name}"] = ref if ref is not None else "not measured (oracle/_ref not built)"
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
