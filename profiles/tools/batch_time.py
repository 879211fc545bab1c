"""Time Problem.solve_batch (ba_cuda_solve_batch: k solves of one structure in one launch, one CTA each) against k
sequential Problem.solve calls on the same inputs.

usage: python profiles/tools/batch_time.py OUT_PREFIX [--ks 1,148,1184,9472] [--calls 10] [--workloads hongo,test2,two_cam,rig156]

Per workload and k: k starts (the workload's start + N(0, 1e-3)) and k observation sets (+ N(0, 0.3 px)), fixed seeds.
  - batch: host clock around solve_batch (it ends in a stream synchronise), rows_cap = 0 (no progress rows copied back),
    2 warm-up calls, then the median of --calls calls;
  - sequential: set_parameters + solve + get_parameters per instance (the model is set up with the instance's observations
    outside the clock), host clock per solve over min(k, 148) instances after 3 warm-up solves; the time of k sequential
    solves is k x the mean of those.
Solves/s and LM iterations/s (summed num_linear_solves) per call.  The card's name and power limit (nvidia-smi, read only)
are recorded in the same run.  Writes OUT_PREFIX.json and OUT_PREFIX.txt.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from realsensecalibration_b200 import cuda, synthetic as S  # noqa: E402
from tests import helpers as H  # noqa: E402


def workload(name):
    """(set_model(P, obs), observations, start)"""
    if name in ("hongo", "test2"):
        pb, intr, side, fix0 = H.hongo() if name == "hongo" else H.test2()
        def load(P, obs):
            P.set_model_b(pb.n_cam, pb.n_time, pb.n_marker, pb.time_idx, pb.cam_idx, pb.marker_idx, obs, intr, side, fix0)
        return load, pb.obs8, np.asarray(pb.params, np.float64)
    if name == "two_cam":
        pa, intr = H.two_cam()
        def load(P, obs):
            P.set_model_a(pa.n_cam, pa.n_pt, pa.cam_idx, pa.pt_idx, obs, intr)
        return load, pa.obs_xy, np.asarray(pa.params, np.float64)
    if name == "rig156":   # n = 6 (4 + 22) = 156, 7744 residual rows: the largest the one-CTA path takes
        pr = S.marker_rig_b(4, 22, 11, 7)
        def load(P, obs):
            P.set_model_b(pr.n_cam, pr.n_time, pr.n_marker, pr.time_idx, pr.cam_idx, pr.marker_idx, obs, pr.intr, pr.marker_side, 1)
        return load, pr.obs8, pr.params
    raise KeyError(name)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True,
                              timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "nvidia-smi failed: %s" % e


def run(name, ks, calls):
    load, obs0, x_start = workload(name)
    out = []
    P, Q = cuda.Problem(0), cuda.Problem(0)
    for k in ks:
        rng = np.random.default_rng(k)
        x0 = x_start[None] + rng.normal(0.0, 1e-3, (k, x_start.shape[0]))
        obs = obs0[None] + rng.normal(0.0, 0.3, (k,) + obs0.shape)
        load(P, obs0)
        times = []
        for rep in range(calls + 2):
            t0 = time.perf_counter()
            xs, sums, _ = P.solve_batch(x0, obs, rows_cap=0)
            if rep >= 2:
                times.append(time.perf_counter() - t0)
        t_batch = float(np.median(times))
        its = int(sum(s.num_linear_solves for s in sums))
        m = min(k, 148)
        per = []
        for i in list(range(min(3, m))) + list(range(m)):   # the first solves warm up
            load(Q, obs[i])
            Q.set_parameters(x0[i])
            t0 = time.perf_counter()
            s, _ = Q.solve()
            Q.get_parameters()
            per.append(time.perf_counter() - t0)
        per = np.asarray(per[min(3, m):])
        t_seq = k * float(per.mean())
        r = {"workload": name, "k": k, "batch_call_s": t_batch, "batch_call_s_min": float(min(times)),
             "batch_call_s_max": float(max(times)), "calls": calls, "batch_solves_per_s": k / t_batch,
             "batch_lm_iterations_per_s": its / t_batch, "lm_iterations": its,
             "sequential_solve_s_mean": float(per.mean()), "sequential_solve_s_median": float(np.median(per)),
             "sequential_instances_timed": m, "sequential_s": t_seq, "sequential_solves_per_s": k / t_seq,
             "sequential_lm_iterations_per_s": its / t_seq, "speedup": t_seq / t_batch,
             "converged": int(sum(s.termination_type == 0 for s in sums))}
        print(json.dumps(r), flush=True)
        out.append(r)
    P.close(); Q.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--ks", default="1,148,1184,9472")
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--workloads", default="hongo,test2,two_cam,rig156")
    a = ap.parse_args()
    info = card()
    res = {"card": info, "method": __doc__.strip().splitlines()[3:12], "results": []}
    for w in a.workloads.split(","):
        res["results"] += run(w, [int(k) for k in a.ks.split(",")], a.calls)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out + ".json", "w") as f:
        json.dump(res, f, indent=1)
    with open(a.out + ".txt", "w") as f:
        f.write("%s\n\n" % info)
        f.write("%-8s %6s %12s %14s %14s %14s %14s %8s\n" % ("workload", "k", "batch ms", "batch solve/s", "batch LM it/s",
                                                            "seq solve/s", "seq LM it/s", "speedup"))
        for r in res["results"]:
            f.write("%-8s %6d %12.3f %14.0f %14.0f %14.0f %14.0f %8.1f\n" % (
                r["workload"], r["k"], 1e3 * r["batch_call_s"], r["batch_solves_per_s"], r["batch_lm_iterations_per_s"],
                r["sequential_solves_per_s"], r["sequential_lm_iterations_per_s"], r["speedup"]))


if __name__ == "__main__":
    main()
