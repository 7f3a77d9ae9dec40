"""A/B probe for traversal-kernel changes: bench.py lines of two (or more) builds of the project, measured in one
session, alternating arm by arm (A B A B ...), with the GPU's name, power limit and SM clocks recorded next to them.

    python tools/hop_rows_probe.py --arm old=/path/to/baseline/checkout --arm new=. [--runs 5] [--out FILE]

Every arm is a checkout of the project whose library is built; its own bench.py runs from its own directory, with
its own input cache (HS_DATA_CACHE under a temporary directory), so the deterministic GPU-built graphs of the two
builds are compared by digest as well.  An arm may add environment variables: --arm new-wpc1=.,HS_WPC=1.

Cases (--cases): sift1m at ef 100 (the bench default), 50 and 200, msturing1m-slimq.  Every sift1m run passes
--dump-outputs, so it searches the GPU-built graph, and the first run of every arm also measures recall; the labels
and distances of the arms' first runs are compared byte for byte, together with the digests of index and queries.
--no-cpu-baseline and --no-sharded leave out the parts of a bench line that do not time this kernel."""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

CASES = {
    "ef100": ("sift1m", []),
    "ef50": ("sift1m", ["--ef", "50"]),
    "ef200": ("sift1m", ["--ef", "200"]),
    "slimq": ("msturing1m-slimq", []),
}


def gpu_state() -> str:
    q = "name,power.limit,power.max_limit,clocks.sm,clocks.max.sm,clocks.mem,temperature.gpu,driver_version"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv"], capture_output=True, text=True,
                           timeout=60)
        return r.stdout.strip() or r.stderr.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        return f"nvidia-smi unavailable: {e!r}"


def file_digest(path: str) -> str:
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def run_bench(arm_dir: str, env_extra: dict, cache: str, workload: str, extra: list, steps: int, warmup: int,
              first: bool, dump: str | None, timeout: float) -> dict:
    cmd = [sys.executable, os.path.join(arm_dir, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup",
           str(warmup), "--workload", workload, "--no-cpu-baseline", "--no-sharded"] + extra
    if not first:
        cmd.append("--no-recall")
    if dump:
        cmd += ["--dump-outputs", dump]
    env = dict(os.environ, HS_DATA_CACHE=cache, **env_extra)
    t0 = time.time()
    r = subprocess.run(cmd, cwd=arm_dir, env=env, capture_output=True, text=True, timeout=timeout)
    line = None
    for ln in r.stdout.splitlines():
        if ln.startswith("{"):
            line = ln
    if r.returncode != 0 or line is None:
        sys.stderr.write(r.stderr[-4000:])
        raise SystemExit(f"bench.py failed in {arm_dir} ({' '.join(extra)}): exit {r.returncode}")
    out = json.loads(line)
    out["_wall_s"] = time.time() - t0
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--arm", action="append", required=True, help="NAME=DIR[,VAR=VAL...]; the first arm is the baseline")
    ap.add_argument("--cases", default="ef100,ef50,ef200")
    ap.add_argument("--runs", default="5", help="runs per arm: one number, or CASE=N,... (others take 5)")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the report here")
    a = ap.parse_args()

    arms = []
    for spec in a.arm:
        name, rest = spec.split("=", 1)
        parts = rest.split(",")
        env = dict(p.split("=", 1) for p in parts[1:])
        arms.append((name, os.path.abspath(parts[0]), env))
    runs = {}
    if "=" in a.runs:
        runs = {k: int(v) for k, v in (p.split("=") for p in a.runs.split(","))}
    nruns = lambda c: runs.get(c, 5) if runs else int(a.runs)  # noqa: E731

    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").close()

    def say(s=""):          # the report is written as it grows: a failed run leaves what came before it
        print(s, flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(s + "\n")

    say(f"# hop_rows_probe: bench.py --steps {a.steps} --warmup {a.warmup} --no-cpu-baseline --no-sharded, arms "
        f"alternated run by run; {time.strftime('%Y-%m-%d %H:%M:%S')}")
    say("# GPU before:\n" + gpu_state())
    for name, d, env in arms:
        say(f"# arm {name}: {d} {env or ''}")
    tmp = tempfile.mkdtemp(prefix="hs_hop_probe_")
    results = {}
    for case in a.cases.split(","):
        workload, extra = CASES[case]
        for r in range(nruns(case)):
            for name, d, env in arms:
                # one cache per checkout: arms that share a directory share the graph
                cache = os.path.join(tmp, "cache_" + hashlib.sha1(d.encode()).hexdigest()[:8])
                dump = os.path.join(tmp, f"dump_{name}_{case}") if workload == "sift1m" and r == 0 else None
                if workload == "sift1m" and dump is None:
                    dump = os.path.join(tmp, f"dump_scratch_{name}")       # same (GPU-built) graph on every run
                res = run_bench(d, env, cache, workload, extra, a.steps, a.warmup, r == 0, dump,
                                timeout=1800 if r == 0 else 600)
                results.setdefault(case, {}).setdefault(name, []).append(res)
                sus = (res.get("sustained") or {}).get("value")
                rf = res.get("roofline") or {}
                say(f"{case:6s} run {r} {name:10s} value {res['value'] / 1e6:7.3f} M QPS  ms/step {res['ms_per_step']:.4f}  "
                    f"sustained {sus / 1e6 if sus else float('nan'):7.3f} M  dist/q {rf.get('dist_evals_per_query', 0):.2f}  "
                    f"hops/q {rf.get('hops_per_query', 0):.2f}  recall {res['config'].get('recall_at_10')}  "
                    f"clocks {json.dumps(res.get('clocks'))}  ({res['_wall_s']:.0f} s)")
    say("\n# summary: median [min, max] of value and sustained (M QPS), change of the median against the first arm")
    base = arms[0][0]
    for case, by_arm in results.items():
        med0 = statistics.median(x["value"] for x in by_arm[base])
        sus0 = [(x.get("sustained") or {}).get("value") for x in by_arm[base]]
        for name, rs in by_arm.items():
            v = [x["value"] / 1e6 for x in rs]
            s = [(x.get("sustained") or {}).get("value", 0) / 1e6 for x in rs]
            sm0 = statistics.median(x for x in sus0 if x) / 1e6 if all(sus0) else float("nan")
            say(f"{case:6s} {name:10s} n={len(v)} value {statistics.median(v):7.3f} [{min(v):.3f}, {max(v):.3f}] "
                f"({(statistics.median(v) * 1e6 / med0 - 1) * 100:+.1f} %)   sustained {statistics.median(s):7.3f} "
                f"[{min(s):.3f}, {max(s):.3f}] ({(statistics.median(s) / sm0 - 1) * 100:+.1f} %)")
    say("\n# outputs of the first run of every arm (sift1m cases): inputs.json, labels.npy, distances.npy")
    for case in results:
        if CASES[case][0] != "sift1m":
            continue
        ref = None
        for name, _, _ in arms:
            dd = os.path.join(tmp, f"dump_{name}_{case}")
            with open(os.path.join(dd, "inputs.json")) as f:
                inputs = json.load(f)
            dig = {fn: file_digest(os.path.join(dd, fn)) for fn in ("labels.npy", "distances.npy")}
            cur = (inputs, dig)
            same = "reference" if ref is None else ("IDENTICAL" if cur == ref else "DIFFERENT")
            ref = ref or cur
            say(f"{case:6s} {name:10s} index {inputs['index_sha256'][:16]} queries {inputs['queries_sha256'][:16]} "
                f"labels {dig['labels.npy'][:16]} distances {dig['distances.npy'][:16]}  {same}")
    say("# GPU after:\n" + gpu_state())
    shutil.rmtree(tmp, ignore_errors=True)
    if a.out:
        with open(os.path.splitext(a.out)[0] + ".jsonl", "w") as f:
            for case, by_arm in results.items():
                for name, rs in by_arm.items():
                    for i, x in enumerate(rs):
                        f.write(json.dumps({"case": case, "arm": name, "run": i, "line": x}) + "\n")


if __name__ == "__main__":
    main()
