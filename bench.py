#!/usr/bin/env python
"""bench.py -- LM iterations/s of the bundle-adjustment hot path on B200 (and the CPU reference arm beside it).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg5] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W     (one rank per GPU)

A "step" is ONE Levenberg-Marquardt iteration (one row of Ceres' progress table: Schur elimination of the
current Jacobian, reduced-camera-system solve, back-substitution, candidate cost, accept/reject, and on
acceptance the residual + Jacobian evaluation at the new point) on the synthetic problem named by
--workload.  A bundle-adjustment solve only runs 5-10 such iterations before it converges, so the K timed
steps are run as ceil(K / ITERS_PER_SOLVE) solves that each restart from the same initial guess (a
device-to-device restore); the initial evaluation every solve starts with (TrustRegionMinimizer's iteration
zero) IS inside the timed region but is not counted as a step, so `value` under-reports rather than
over-reports.

  value   K / device time of those solves, problem resident in HBM (CUDA events on the solve stream, max over ranks)
  e2e     the same K steps through the public C ABI from HOST buffers: ba_cuda_set_model_a (observations,
          indices -> HBM, structure build) + ba_cuda_set_parameters + ba_cuda_solve + ba_cuda_get_parameters,
          all inside the timed region
  roofline      the kernel with the largest share of device time: algorithmic bytes (DESIGN.md) / its
                CUDA-event duration, against MEASURED_PEAKS.json
  cpu_baseline  the CPU oracle (oracle/, a restatement of the Ceres 1.14 path the reference runs) on the host cores

--impl reference times that CPU oracle alone, with all host threads, on the same workload/metric.

--dump-outputs DIR writes, after the timed steps, what the timed path returned to its caller in its last step (see
dump_outputs) as DIR/<name>.npy.  The workloads are generated from fixed seeds, so two builds run with the same
arguments can be compared output for output.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ITERS_PER_SOLVE = 5

# --dump-outputs: a parameter vector of up to DUMP_MAX_FULL entries (32 MB in float64) is written whole; a larger one
# (cfg5 has 12M) as a sample of DUMP_SAMPLE entries drawn with DUMP_SEED, beside their positions, 32 MB in all
DUMP_MAX_FULL = 1 << 22
DUMP_SAMPLE = 1 << 21
DUMP_SEED = 0xBAD0
DUMP_ROW_FIELDS = ("cost", "cost_change", "gradient_max_norm", "step_norm", "trust_region_radius", "linear_solver_iterations",
                   "step_is_successful")

# name -> (description, model, generator kwargs, rcs solver)
WORKLOADS = {
    "hongo": dict(desc="the reference's own fixture Common/Correspondence/hongo/correspondence.txt (Model B, Main_Calibration dispatch): "
                       "4 cameras x 6 frames x 11 markers, 68 marker observations (272 corner observations)",
                  kind="hongo", args=()),
    "cfg1": dict(desc="Test1_BundleAdjustment-shaped synthetic (Model A): 2 cameras (one relative pose), 1 ArUco marker (4 corners) x 50 frames "
                      "= 200 points, 200 observations",
                 kind="two_cam", args=(50, 0xBA01)),
    "cfg3a": dict(desc="large rig, Model A reading: 8 cameras x 100 markers x 1000 frames = 400k corner points, 3.2M observations",
                  kind="rig_a", args=(8, 100, 1000, 0xBA03)),
    "cfg4": dict(desc="BAL-shaped synthetic: 1000 cameras x 1M points x 5M observations (window 20)",
                 kind="bal", args=(1000, 1000000, 5, 20, 0xBA04)),
    "cfg5": dict(desc="BAL-shaped synthetic: 10000 cameras x 4M points x ~30M observations (Poisson 2..16 per point, window 30)",
                 kind="bal", args=(10000, 4000000, 7.5, 30, 0xBA05), kwargs=dict(variable_degree=True)),
    "small": dict(desc="smoke-sized BAL-shaped synthetic: 50 cameras x 20k points x 100k observations",
                  kind="bal", args=(50, 20000, 5, 12, 0xBA00)),
    "cfg2": dict(desc="Main_Calibration shape (Model B): 4 cameras x 20 markers x 200 frames = 16k marker observations (64k corner "
                      "observations), camera 0 and marker 0 fixed",
                 kind="rig_b", args=(4, 20, 200, 0xBA02)),
    "cfg3": dict(desc="large rig (Model B): 8 cameras x 100 markers x 1000 frames = 800k marker observations (3.2M corner observations)",
                 kind="rig_b", args=(8, 100, 1000, 0xBA03)),
}
# The default is the problem BASELINE.json's north_star sets its targets on (30M observations, PCG on the reduced camera
# system; it fits one B200), so that the 1 -> 8 GPU runs of the driver measure strong scaling on that problem.
DEFAULT_WORKLOAD = "cfg5"


def host_threads():
    """Host threads the CPU arm may use: the process' CPU affinity, NOT omp_get_max_threads() -- torch.distributed.run
    exports OMP_NUM_THREADS=1 to its workers, which would turn "all host cores" into one."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def kernel_source_hash():
    """Identifies the kernels a profile was taken on (profiles/traffic.json): sha256 over csrc/*.cu*."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "realsensecalibration_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            with open(os.path.join(d, f), "rb") as fh:
                h.update(fh.read())
    return h.hexdigest()[:16]


def make_workload(name):
    from realsensecalibration_b200 import synthetic as S
    w = WORKLOADS[name]
    if w["kind"] == "hongo":
        from realsensecalibration_b200 import formats as F
        from tests import helpers as H
        pb, intr, side, fix0 = H.hongo()
        counts = np.zeros((pb.n_time, pb.n_cam), np.int32)
        np.add.at(counts, (pb.time_idx, pb.cam_idx), 1)
        return S.ModelB(pb.n_cam, pb.n_time, pb.n_marker, pb.time_idx, pb.cam_idx, pb.marker_idx, pb.obs8, np.asarray(intr, np.float64),
                        pb.params, pb.params, side, counts)
    if w["kind"] == "two_cam":
        return S.two_cam_like(*w["args"])
    if w["kind"] == "rig_a":
        return S.marker_rig_a(*w["args"])
    if w["kind"] == "rig_b":
        return S.marker_rig_b(*w["args"])
    return S.bal_like(*w["args"], **w.get("kwargs", {}))


class Job:
    """One workload as the bench sees it: the rank-local shard, how to hand it to the C ABI, the CPU oracle call."""

    def __init__(self, name, rank, world):
        from realsensecalibration_b200 import sharding
        self.pr = pr = make_workload(name)
        self.model = "B" if WORKLOADS[name]["kind"] in ("rig_b", "hongo") else "A"
        if self.model == "A":
            sh = sharding.shard_model_a(pr.n_cam, pr.n_pt, pr.cam_idx, pr.pt_idx, pr.obs_xy, pr.params, rank, world)
            self.local = (sh.n_pt, sh.cam_idx, sh.pt_idx, np.asarray(sh.obs_xy), sh.params)
            self.n_obs = pr.n_obs                    # corner observations (2 residuals each)
            self.jac_bytes_per_obs = 184
            self.blocks = {"n_cameras": pr.n_cam, "n_points": pr.n_pt, "n_obs": pr.n_obs}
            self.sharded = "points"
        else:
            sh = sharding.shard_model_b(pr.n_cam, pr.n_time, pr.n_marker, pr.time_idx, pr.cam_idx, pr.marker_idx, pr.obs8, pr.params, rank, world)
            self.local = (sh.n_time, sh.time_idx, sh.cam_idx, sh.marker_idx, np.asarray(sh.obs8), sh.params)
            self.n_obs = pr.n_mobs                   # marker observations (8 residuals each)
            self.jac_bytes_per_obs = 1292
            self.blocks = {"n_cameras": pr.n_cam, "n_frames": pr.n_time, "n_markers": pr.n_marker, "n_marker_obs": pr.n_mobs,
                           "n_corner_obs": 4 * pr.n_mobs}
            self.sharded = "frames"
        self.lo, self.hi = sh.lo, sh.hi
        self.params = self.local[-1]
        self.h2d = sum(np.asarray(a).nbytes for a in self.local[1:]) + pr.intr.nbytes

    def pin(self):
        """The rank-local input arrays (and nothing else) move to pinned host memory, as the e2e contract says: the
        library's cudaMemcpyAsync calls then run as direct DMA instead of being staged by the driver."""
        import torch

        def pinned(a):
            t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
            self._keep.append(t)
            return t.numpy()
        self._keep = []
        self.local = (self.local[0],) + tuple(pinned(a) for a in self.local[1:])
        self.params = self.local[-1]
        self.result = pinned(np.zeros_like(self.params))   # where ba_cuda_get_parameters writes the solution

    def set_model(self, P):
        pr = self.pr
        if self.model == "A":
            n_pt, cam, pt, obs, _ = self.local
            P.set_model_a(pr.n_cam, n_pt, cam, pt, obs, pr.intr)
        else:
            n_time, ti, ci, mi, obs8, _ = self.local
            P.set_model_b(pr.n_cam, n_time, pr.n_marker, ti, ci, mi, obs8, pr.intr, pr.marker_side, True)

    def merge(self, shard_results):
        """(lo, hi, rank-local parameter vector) of every rank -> the parameter vector of the whole problem."""
        from realsensecalibration_b200 import sharding
        pr = self.pr
        if self.model == "A":
            return sharding.merge_model_a(pr.n_cam, pr.n_pt, shard_results)
        return sharding.merge_model_b(pr.n_cam, pr.n_time, pr.n_marker, shard_results)

    def oracle_solver(self, O):
        # the rule BA_RCS_AUTO applies (ba_cuda.cu, kDenseAutoMaxN): dense Cholesky up to dimension 1536, PCG above
        n_kept = self.pr.n_cam if self.model == "A" else self.pr.n_cam + self.pr.n_marker
        return O.SCHUR_DENSE if 6 * n_kept <= 1536 else O.SCHUR_PCG

    def oracle_solve(self, O, opts, threads):
        pr = self.pr
        if self.model == "A":
            return O.solve_model_a(pr.n_cam, pr.n_pt, pr.cam_idx, pr.pt_idx, pr.obs_xy, pr.intr, pr.params, options=opts,
                                   linear_solver=self.oracle_solver(O), n_threads=threads)
        return O.solve_model_b(pr, pr.intr, pr.marker_side, True, options=opts, linear_solver=self.oracle_solver(O), n_threads=threads)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [l for t, l in self.lines if t0 - 0.05 <= t <= t1 + 0.15] or [l for _, l in self.lines]
        for l in rows:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); smax = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def bench_options(cuda, profile):
    o = cuda.default_options()
    o.max_num_iterations = ITERS_PER_SOLVE
    o.function_tolerance = 0.0      # never stop early: exactly ITERS_PER_SOLVE rows per solve
    o.parameter_tolerance = 0.0
    o.gradient_tolerance = 0.0
    o.profile_kernels = 1 if profile else 0
    return o


def run_steps(P, opts, k):
    """k LM iterations as solves of ITERS_PER_SOLVE, each restarting from the saved initial guess."""
    done = 0
    while done < k:
        n = min(ITERS_PER_SOLVE, k - done)
        P.restore_parameters()
        if n == opts.max_num_iterations:   # the one-call API (what BAManager::Solve uses): ba_cuda_solve
            out = P.solve(opts)
        else:
            P.solve_begin(opts)
            P.solve_iterate(n)
            out = P.solve_end()
        check_steps(out[1], n)
        done += n
    return out


def check_steps(rows, n):
    """A solve that stopped before its n LM iterations would make K / time over-report: refuse to count it."""
    if len(rows) != n + 1:   # row 0 is the initial evaluation
        raise RuntimeError("a solve asked for %d LM iterations ran %d: the timed steps would not be --steps" % (n, len(rows) - 1))


def oracle_steps(job, k, threads):
    """The reference arm: the CPU oracle on the same workload, same restart rule; returns (seconds, rows, summary, x) of
    the last solve."""
    from oracle import oracle_py as O
    o = O.default_options()
    o.function_tolerance = 0.0; o.parameter_tolerance = 0.0; o.gradient_tolerance = 0.0
    done, t, rows = 0, 0.0, []
    while done < k:
        n = min(ITERS_PER_SOLVE, k - done)
        o.max_num_iterations = n
        t0 = time.perf_counter()
        x, s, rows = job.oracle_solve(O, o, threads)
        t += time.perf_counter() - t0
        check_steps(rows, n)
        done += n
    return t, rows, s, x


def dump_outputs(out_dir, x, summary, rows):
    """--dump-outputs: what the timed path handed its caller after its last step, one float64 .npy file per array --
    the parameter vector (what ba_cuda_get_parameters returns, or the oracle's solution on --impl reference; a fixed,
    seeded sample of it above DUMP_MAX_FULL entries, with the positions of the sample in parameters_index), the progress rows of the last solve (row 0 is the cost it started
    from) and its final cost."""
    os.makedirs(out_dir, exist_ok=True)
    x = np.asarray(x, np.float64)
    arrays = {}
    if x.size <= DUMP_MAX_FULL:
        arrays["parameters"] = x
    else:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(x.size, DUMP_SAMPLE, replace=False))
        arrays["parameters"] = x[idx]
        arrays["parameters_index"] = idx.astype(np.float64)
    for k in DUMP_ROW_FIELDS:
        arrays[k] = np.array([r[k] for r in rows], np.float64)
    arrays["final_cost"] = np.array([summary.final_cost], np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def config_of(job, name, n_gpus, rcs_solver, rcs_dim):
    """The `config` object both arms print (the driver compares them key by key)."""
    ws_mb = job.n_obs * (job.jac_bytes_per_obs if job.model == "B" else 72) / 1e6 / n_gpus
    l2_note = ("per-step working set of %.0f MB per rank exceeds the 126 MB L2; no explicit flush" % ws_mb if ws_mb > 126 else
               "per-step working set of %.0f MB per rank fits the 126 MB L2 (this is the reference's own problem size); no flush: the "
               "real workload is L2 resident too" % ws_mb)
    return {"workload": name, "description": WORKLOADS[name]["desc"], **job.blocks, "iters_per_solve": ITERS_PER_SOLVE,
            "parallelism": "%s sharded over %d rank(s), kept blocks (cameras%s) replicated" %
                           (job.sharded, n_gpus, "" if job.model == "A" else ", markers"),
            "l2": l2_note, "rcs_solver": {1: "dense_cholesky", 2: "pcg"}.get(int(rcs_solver), "?"), "rcs_dim": int(rcs_dim)}


def committed_trace(name):
    """Oracle rows of the bench solve (ITERS_PER_SOLVE iterations from the bench start), tests/golden/synth_traces.json."""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "synth_traces.json")) as f:
            return json.load(f).get(name)
    except (OSError, ValueError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-jacobian", action="store_true", help="skip the standalone residual+Jacobian kernel timing")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path computed in its last step to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K, W = a.steps, max(a.warmup, 0)
    metric, unit = "LM iterations/sec", "it/s"
    wl = WORKLOADS[a.workload]

    if a.impl == "reference":
        if rank != 0:
            return 0
        from oracle import oracle_py as O
        job = Job(a.workload, 0, 1)
        threads = host_threads()
        if W > 0:
            oracle_steps(job, min(W, 1), threads)
        secs, rows, osum, x = oracle_steps(job, K, threads)
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, x, osum, rows)
        v = K / secs
        print(json.dumps({
            "impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": a.gpus, "steps": K, "warmup": W,
            "ms_per_step": 1e3 * secs / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic" if wl["kind"] != "hongo" else "reference fixture (tests/golden)",
            "config": config_of(job, a.workload, a.gpus, 1 if job.oracle_solver(O) == O.SCHUR_DENSE else 2, osum.rcs_dim),
            "cpu_baseline": {"value": v, "unit": unit, "cores": threads, "kind": "port",
                             "threads_from": "CPU affinity of the process, passed to the oracle's num_threads clauses (OMP_NUM_THREADS is ignored)",
                             "final_cost": float(osum.final_cost),
                             "sample": "full workload, %d LM iterations in solves of %d (problem construction + initial evaluation "
                                       "of each solve included)" % (K, ITERS_PER_SOLVE)},
            "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "jacobian_mobs_per_sec": None, "gpu_launches": 0}))
        return 0

    # libraries (NCCL's version banner, for one) write to stdout: keep fd 1 for the one JSON line
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import torch
    from realsensecalibration_b200 import cuda
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    job = Job(a.workload, rank, world)
    job.pin()
    pr, par_l = job.pr, job.params
    stream = torch.cuda.Stream()
    P = cuda.Problem(local_rank)
    P.set_stream(stream.cuda_stream)
    if world > 1:
        ids = [cuda.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        P.comm_init(rank, world, ids[0])

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident measurement ("value") ----------------------------------------------------
    job.set_model(P)
    P.set_parameters(par_l)
    P.save_parameters()
    opts = bench_options(cuda, profile=False)
    if W > 0:
        run_steps(P, opts, W)
    barrier()
    P.reset_stats()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    with torch.cuda.stream(stream):
        e0.record(stream)
        summary, rows = run_steps(P, opts, K)
        e1.record(stream)
    barrier()
    t_wall1 = time.time()
    ms = e0.elapsed_time(e1)
    launches = P.num_launches()
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if dist is not None:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = K / (ms * 1e-3)
    if a.dump_outputs:
        # now, before the passes below overwrite the problem's parameters
        x = P.get_parameters()
        if dist is not None:
            got = [None] * world
            dist.all_gather_object(got, (job.lo, job.hi, x))
            x = job.merge(got)
        if rank == 0:
            dump_outputs(a.dump_outputs, x, summary, rows)

    # the same K steps once more with an event pair around every kernel (costs a few us per launch, which is why it is
    # not the timed pass): per-kernel device times for the roofline and the kernel shares
    P.reset_stats()
    with torch.cuda.stream(stream):
        e0.record(stream)
        summary, rows = run_steps(P, bench_options(cuda, profile=True), K)
        e1.record(stream)
    barrier()
    ms_prof = e0.elapsed_time(e1)
    stats = P.kernel_stats()

    # residual+Jacobian throughput (the other half of BASELINE.json's metric): the standalone K1 kernel (residual and
    # analytic Jacobian written to HBM, what ba_cuda_eval runs; the LM loop of Model A uses the fused passes instead,
    # where r and J never leave the SM), timed by the library's own CUDA events on the solve stream
    peak, peak_src = peaks()
    jacobian = None
    jac_mobs = None
    if not a.no_jacobian:
        P.restore_parameters()
        with torch.cuda.stream(stream):
            for _ in range(2):
                P.eval(False, False)
            ts = []
            for _ in range(5):
                P.eval(False, False)
                ts.append(P.last_kernel_ms())
        jms = float(np.median(ts))
        if dist is not None:
            t = torch.tensor([jms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            jms = float(t.item())
        jac_mobs = job.n_obs / 1e6 / (jms * 1e-3)   # whole job: shards run concurrently
        gbs = job.jac_bytes_per_obs * job.n_obs / world / (jms * 1e-3) / 1e9
        jacobian = {"kernel": "k_fa_jac" if job.model == "A" else "k_jac_b", "ms": jms, "mobs_per_sec": jac_mobs,
                    "unit_of_obs": "corner observation (2 residuals)" if job.model == "A" else "marker observation (8 residuals)",
                    "algorithmic_bytes_per_obs": job.jac_bytes_per_obs, "achieved_gbs_per_gpu": gbs, "frac_of_hbm_peak": gbs / peak}

    # roofline of the dominant kernel
    timed = [s for s in stats if s["total_ms"] > 0 and s["algorithmic_bytes_per_launch"] > 0]
    roofline = None
    if timed:
        top = max(timed, key=lambda s: s["total_ms"])
        avg_s = top["total_ms"] / top["launches"] * 1e-3
        ach = top["algorithmic_bytes_per_launch"] / avg_s / 1e9
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                ent = json.load(f).get(a.workload, {}).get(top["name"])
            # only a capture of THESE kernels counts: the profile records the hash of the kernel sources it was taken on
            if ent and world == 1 and ent.get("kernel_source_hash") == kernel_source_hash():
                traffic, traffic_src = ent["bytes"], ent["source"]
        except (OSError, ValueError):
            pass
        roofline = {"bound": "hbm", "kernel": top["name"], "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": traffic, "traffic_source": traffic_src,
                    "algorithmic_bytes_per_launch": top["algorithmic_bytes_per_launch"], "peak_source": peak_src, "avg_launch_ms": avg_s * 1e3, "launches": top["launches"],
                    "share_of_step": top["total_ms"] / ms_prof,
                    "all_kernels": [{"name": s["name"], "launches": s["launches"], "ms_per_launch": s["total_ms"] / s["launches"],
                                     "share": s["total_ms"] / ms_prof,
                                     "gbs": (s["algorithmic_bytes_per_launch"] / (s["total_ms"] / s["launches"] * 1e-3) / 1e9)
                                     if s["total_ms"] > 0 and s["algorithmic_bytes_per_launch"] > 0 else None} for s in stats]}

    # ---- end to end through the public C ABI from host buffers ("e2e") ------------------------------
    e2e = None
    if not a.no_e2e:
        opts_e = bench_options(cuda, profile=False)
        h2d = job.h2d
        d2h = par_l.nbytes
        def e2e_solves(k):
            done = 0
            x = None
            while done < k:
                n = min(ITERS_PER_SOLVE, k - done)
                opts_e.max_num_iterations = n
                job.set_model(P)
                P.set_parameters(par_l)
                P.solve(opts_e)
                x = P.get_parameters(out=job.result)
                done += n
            return x
        e2e_solves(min(W, ITERS_PER_SOLVE) or 1)
        barrier()
        t0 = time.perf_counter()
        e2e_solves(K)
        barrier()
        secs = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([secs], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            secs = float(t.item())
        n_solves = (K + ITERS_PER_SOLVE - 1) // ITERS_PER_SOLVE
        e2e = {"value": K / secs, "unit": unit, "h2d_bytes_per_step": int(h2d * n_solves / K), "d2h_bytes_per_step": int(d2h * n_solves / K),
               "ms_per_step": 1e3 * secs / K, "timed": "host wall clock around set_model_a + set_parameters + solve + get_parameters, max over ranks"}

    # ---- CPU baseline (rank 0, N=1 only) -------------------------------------------------------------
    cpu = None
    parity = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        from oracle import oracle_py as O
        threads = host_threads()
        kc = min(K, ITERS_PER_SOLVE)
        secs, _, osum, _ = oracle_steps(job, kc, threads)
        cpu = {"value": kc / secs, "unit": unit, "cores": threads, "kind": "port",
               "threads_from": "CPU affinity of the process, passed to the oracle's num_threads clauses",
               "final_cost": float(osum.final_cost),
               "sample": "full workload, one solve of %d LM iterations (problem construction + initial evaluation included), "
                         "oracle/ba_oracle.cpp with OpenMP" % kc}
        if WORKLOADS[a.workload]["kind"] in ("hongo", "two_cam") and threads > 1:
            # at the reference's own problem sizes OpenMP's fork / join can cost more than it buys: best of three solves on ONE thread too
            best = min(oracle_steps(job, kc, 1)[0] for _ in range(3))
            cpu["single_thread_value"] = kc / best
        if kc == ITERS_PER_SOLVE and K >= ITERS_PER_SOLVE:
            # relative to the final cost, but never below 1e-12 of the initial cost: a zero-residual problem (cfg1) ends at round-off
            scale = max(abs(float(osum.final_cost)), 1e-12 * abs(float(osum.initial_cost)), 1e-300)
            parity = {"oracle_final_cost": float(osum.final_cost), "gpu_final_cost": float(summary.final_cost),
                      "rel": abs(float(summary.final_cost) - float(osum.final_cost)) / scale,
                      "source": "cpu_baseline leg of this run (same options, same start, %d LM iterations)" % kc}
    if parity is None and rank == 0 and K >= ITERS_PER_SOLVE and K % ITERS_PER_SOLVE == 0:
        tr = committed_trace(a.workload)
        if tr:
            oc = float(tr["rows"][-1]["cost"])
            parity = {"oracle_final_cost": oc, "gpu_final_cost": float(summary.final_cost),
                      "rel": abs(float(summary.final_cost) - oc) / abs(oc), "source": "tests/golden/synth_traces.json (oracle, %s)" % tr["how"]}

    if rank == 0:
        out = {
            "metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic" if wl["kind"] != "hongo" else "reference fixture (tests/golden)",
            "config": config_of(job, a.workload, world, summary.rcs_solver_used, summary.rcs_dim),
            "path_used": {0: "generic", 1: "fused_tiles", 2: "fused_strips", 3: "rig_one_cta"}.get(int(summary.path_used), "?"),
            "parity": parity, "us_per_solve": 1e3 * ms / K * ITERS_PER_SOLVE,
            "jacobian_mobs_per_sec": jac_mobs, "jacobian": jacobian, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches,
            "clocks": clocks, "final_cost_last_solve": float(summary.final_cost), "ms_per_step_profiled_pass": ms_prof / K,
            "device_ms": {"jacobian": summary.ms_jacobian, "schur": summary.ms_schur, "rcs_solve": summary.ms_rcs_solve,
                          "update": summary.ms_update, "cost": summary.ms_cost, "collective": summary.ms_collective, "of_last_solve": True},
        }
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(out) + "\n").encode())
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
