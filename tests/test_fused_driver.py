"""The host sequence of the fused Model A path (fused_linearize / fused_step in ba_cuda.cu) through each of its
branches, on both pass-1 geometries: strips (BA_SA=2) and single tiles (BA_SA=0).  One problem that fits strips,
held to the oracle's rows at the tolerances of test_gpu_parity.py."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from realsensecalibration_b200 import abi, cuda, synthetic as S
from tests import helpers as H
from tests.test_gpu_parity import POSE_ATOL, _check_rows, _Env, _solve_a

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PCG_K = 10

# options on top of max_num_iterations = 5 and the dense solver
CASES = {
    "one_pass": {},                                # iteration 0 linearises, scales and eliminates in one pass
    "no_jacobi_scaling": dict(jacobi_scaling=0),
    "max_iterations_0": dict(max_num_iterations=0),   # cost and gradient only; on tiles the scaling has a pass of its own
    "max_iterations_1": dict(max_num_iterations=1),
    "pcg_fixed_count": dict(rcs_solver=abi.RCS_PCG, pcg_min_iterations=PCG_K, pcg_max_iterations=PCG_K),
}
GEOMETRIES = {"strips": (2, abi.PATH_FUSED_STRIPS), "tiles": (0, abi.PATH_FUSED_TILES)}


@pytest.fixture(scope="module")
def gpu():
    if cuda.device_count() == 0:
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box")
    P = cuda.Problem(0)
    yield P
    P.close()


def _problem():
    return S.bal_like(60, 5000, 6, 16, 13, variable_degree=True)


def _options(mod, case):
    o = mod.default_options()
    o.max_num_iterations = 5
    o.rcs_solver = abi.RCS_DENSE_CHOLESKY
    for k, v in CASES[case].items():
        setattr(o, k, v)
    return o


_oracle_runs = {}


def _oracle_solve(oracle, pr, case):
    if case not in _oracle_runs:
        pcg = CASES[case].get("rcs_solver") == abi.RCS_PCG
        kw = dict(linear_solver=oracle.SCHUR_PCG) if pcg else {}
        xo, so, rows_o = oracle.solve_model_a(pr.n_cam, pr.n_pt, pr.cam_idx, pr.pt_idx, pr.obs_xy, pr.intr, pr.params,
                                              options=_options(oracle, case), n_threads=4, **kw)
        _oracle_runs[case] = (xo, rows_o)
    return _oracle_runs[case]


def _check(case, rows, x, rows_o, xo):
    if CASES[case].get("rcs_solver") == abi.RCS_PCG:   # as test_pcg_with_a_fixed_iteration_count_is_the_same_method
        assert len(rows) == len(rows_o)
        for a, b in zip(rows, rows_o):
            assert a["linear_solver_iterations"] == b["linear_solver_iterations"] == (PCG_K if a["iteration"] > 0 else 0)
            assert a["step_is_successful"] == b["step_is_successful"]
            assert H.rel(a["cost"], b["cost"]) <= 1e-9, (a, b)
    else:
        _check_rows(rows, rows_o)
    assert np.abs(np.asarray(x) - xo).max() < POSE_ATOL


@pytest.mark.parametrize("geometry", sorted(GEOMETRIES))
@pytest.mark.parametrize("case", sorted(CASES))
def test_fused_driver_branch_matches_oracle(gpu, oracle, case, geometry):
    pr = _problem()
    xo, rows_o = _oracle_solve(oracle, pr, case)
    sa, path = GEOMETRIES[geometry]
    with _Env(BA_SA=sa, BA_RIG=0):
        s, rows, x = _solve_a(gpu, pr, _options(cuda, case))
    assert s.path_used == path
    _check(case, rows, x, rows_o, xo)


_CHILD = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
from realsensecalibration_b200 import abi, cuda
from tests.test_fused_driver import _options, _problem
pr = _problem()
P = cuda.Problem(0)
P.set_model_a(pr.n_cam, pr.n_pt, pr.cam_idx, pr.pt_idx, pr.obs_xy, pr.intr)
P.set_parameters(pr.params)
s, rows = P.solve(_options(cuda, sys.argv[2]))
print(json.dumps({"rows": rows, "x": P.get_parameters().tolist(), "path": s.path_used}))
P.close()
"""


@pytest.mark.parametrize("case", ["one_pass", "max_iterations_1"])
def test_tiles_scaling_in_a_pass_of_its_own_matches_oracle(oracle, case):
    # BA_FA_FIRST=0: iteration 0 on tiles takes the Jacobi scaling from a pass of its own (FA_NORMS) before the full
    # pass.  The variable is read once per process, hence the child.
    env = dict(os.environ, BA_SA="0", BA_RIG="0", BA_FA_FIRST="0")
    r = subprocess.run([sys.executable, "-c", _CHILD, ROOT, case], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["path"] == abi.PATH_FUSED_TILES
    xo, rows_o = _oracle_solve(oracle, _problem(), case)
    _check(case, out["rows"], out["x"], rows_o, xo)
