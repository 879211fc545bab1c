"""Time Problem.covariance (ba_cuda_covariance) next to one LM iteration of the same workload.

usage: python profiles/tools/covariance_time.py [OUT.json] [--workloads hongo,cfg2,cfg3] [--calls 25]

Per workload: the problem is solved first (default options), then
  - covariance: host clock around the call (it ends in a stream synchronise), 3 warm-up calls, then --calls timed calls;
  - the per-kernel split of one call with options.profile_kernels = 1 (CUDA events around every launch, a run of its own);
  - one LM iteration: bench.py's options (5 rows per solve, no early stop), solve time / rows, median of 10 solves; for the
    rig-size workloads (one-CTA whole-loop kernel) also the multi-kernel pipeline (BA_RIG=0), which the covariance uses.
The card's name and power limit (nvidia-smi, read only) are recorded in the same run.
"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from realsensecalibration_b200 import abi, cuda  # noqa: E402


def stats_ms(samples_s):
    a = np.asarray(samples_s) * 1e3
    return {"median_ms": float(np.median(a)), "min_ms": float(a.min()), "max_ms": float(a.max()),
            "p10_ms": float(np.percentile(a, 10)), "p90_ms": float(np.percentile(a, 90)), "n": int(a.size)}


def lm_iteration(P, rig_off):
    old = os.environ.get("BA_RIG")
    if rig_off:
        os.environ["BA_RIG"] = "0"
    try:
        opts = bench.bench_options(cuda, profile=False)
        per_it, path = [], None
        for rep in range(13):
            P.restore_parameters()
            t0 = time.perf_counter()
            s, rows = P.solve(opts)
            dt = time.perf_counter() - t0
            path = s.path_used
            if rep >= 3:
                per_it.append(dt / max(len(rows) - 1, 1))   # row 0 is the initial evaluation
        out = stats_ms(per_it)
        out["path_used"] = {abi.PATH_GENERIC: "generic", abi.PATH_RIG: "rig"}.get(path, str(path))
        return out
    finally:
        if rig_off:
            if old is None:
                os.environ.pop("BA_RIG", None)
            else:
                os.environ["BA_RIG"] = old


def run(name, calls):
    pr = bench.make_workload(name)
    P = cuda.Problem(0)
    P.set_model_b(pr.n_cam, pr.n_time, pr.n_marker, pr.time_idx, pr.cam_idx, pr.marker_idx, pr.obs8, pr.intr, pr.marker_side, 1)
    P.set_parameters(pr.params)
    P.save_parameters()
    rec = {"workload": name, "desc": bench.WORKLOADS[name]["desc"], "n_marker_obs": int(pr.n_mobs),
           "reduced_system_n": 6 * (pr.n_cam + pr.n_marker), "n_frames": int(pr.n_time)}
    rec["lm_iteration"] = lm_iteration(P, rig_off=False)
    if rec["lm_iteration"]["path_used"] == "rig":
        rec["lm_iteration_multi_kernel"] = lm_iteration(P, rig_off=True)
    P.restore_parameters()
    s, rows = P.solve()
    rec["solve"] = {"iterations": len(rows), "final_cost": s.final_cost}
    for _ in range(3):
        kept, frames, ratio = P.covariance()
    t = []
    for _ in range(calls):
        t0 = time.perf_counter()
        P.covariance()
        t.append(time.perf_counter() - t0)
    rec["covariance"] = stats_ms(t)
    rec["smallest_pivot_ratio"] = ratio
    o = cuda.default_options()
    o.profile_kernels = 1
    P.covariance(o)            # warm the event pool
    P.reset_stats()
    P.covariance(o)
    rec["covariance_kernels"] = {k["name"]: {"launches": k["launches"], "ms": k["total_ms"],
                                             "algorithmic_bytes_per_launch": k["algorithmic_bytes_per_launch"]}
                                 for k in P.kernel_stats()}
    P.close()
    return rec


def main():
    args = sys.argv[1:]
    out = args[0] if args and not args[0].startswith("--") else None
    workloads = ["hongo", "cfg2", "cfg3"]
    calls = 25
    for i, a in enumerate(args):
        if a == "--workloads":
            workloads = args[i + 1].split(",")
        if a == "--calls":
            calls = int(args[i + 1])
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True).stdout
    res = {"gpu": smi.strip().splitlines()[1:] if smi else None, "runs": []}
    for w in workloads:
        r = run(w, calls)
        res["runs"].append(r)
        cov, it = r["covariance"], r["lm_iteration"]
        line = "%-6s n = %4d: covariance %.3f ms (p10 %.3f, p90 %.3f)  LM iteration %.3f ms (%s)" % (
            w, r["reduced_system_n"], cov["median_ms"], cov["p10_ms"], cov["p90_ms"], it["median_ms"], it["path_used"])
        if "lm_iteration_multi_kernel" in r:
            line += ", multi-kernel %.3f ms" % r["lm_iteration_multi_kernel"]["median_ms"]
        print(line, flush=True)
        for k, v in sorted(r["covariance_kernels"].items(), key=lambda kv: -kv[1]["ms"]):
            print("    %-22s %3d launches %9.4f ms" % (k, v["launches"], v["ms"]))
    print("gpu:", res["gpu"])
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
