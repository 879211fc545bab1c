"""The three dense solvers of the reduced camera system, launched directly and compared with a reference solution of the same
fp64 input that is accurate far below fp64 rounding.

    k_ldlt_small   (ba_rig.cuh)            panel L D L^T, the factorisation of the rig kernel; every n <= 160 on the default path
    k_chol_solve   (ba_dense.cuh)          single-CTA Cholesky, n <= 160 under BA_DENSE_LDLT=0
    k_chol_blocked (ba_dense_blocked.cuh)  blocked DMMA Cholesky over the grid, n > 160 and the covariance's factorisation

tests/probe/dense_probe.cu launches them the way the library does, on device buffers given by torch; it is compiled here with the
nvcc flags of csrc/Makefile.

Bounds, with eps = 2^-53 and C = 4 for every solver and matrix:
    backward error   |b - A y|_inf / (|A|_inf |y|_inf + |b|_inf)      <= C n eps
    forward error    |y - x|_2 / |x|_2                                <= C n eps kappa_2(A)
    factor residual  |(A - L L^T) z|_inf / (|A|_inf |z|_inf)           <= C n eps    (k_chol_blocked, 4 random z)
A Cholesky-type solve is backward stable: (A + dA) y = b with |dA| <= gamma_{3n+1} |L||L^T| (Higham, Accuracy and Stability of
Numerical Algorithms, 2nd ed., Thm 10.4), gamma_{3n+1} = (3n + 1) eps / (1 - (3n + 1) eps) < 4 n eps for the n here.  For an SPD
matrix factored without pivoting |L||L^T| stays of the size of |A| (its worst case, a factor n more, needs a matrix far from
these); the kernels' reciprocal-and-multiply in place of a division adds one rounding per entry, inside the margin of 3n + 1 to
4n.  The forward bound is the first-order perturbation bound kappa * (backward error) with the same C, the factor residual the
same gamma bound on A - L L^T itself.

The reference: scipy's cho_solve, then two steps of iterative refinement with the residual b - A x in np.longdouble (64-bit
mantissa), x kept in np.longdouble.  test_reference_against_mpmath checks it against a 40-digit mpmath solve."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.linalg as sla

from realsensecalibration_b200 import abi, formats as F, synthetic as S
from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "realsensecalibration_b200", "csrc")
PROBE_SRC = os.path.join(ROOT, "tests", "probe", "dense_probe.cu")
PROBE_LIB = os.path.join(ROOT, "tests", "probe", "build", "libdense_probe.so")   # build/ is ignored by git

EPS = 2.0 ** -53
C = 4.0
LD = np.longdouble
SMALL = ("ldlt_small", "chol_solve")
SOLVERS = SMALL + ("chol_blocked",)
BLOCKED_N = (1, 2, 31, 32, 33, 63, 64, 65, 97, 127, 128, 129, 159, 160, 161, 191, 192, 193, 255, 256, 257, 385, 636, 1023, 1535,
             1536, 1537, 2049, 6000)


# ---- the probe library ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="session")
def probe_lib():
    """Compiles tests/probe/dense_probe.cu against the csrc headers with the library's own nvcc command line."""
    cmd = subprocess.run(["make", "-s", "--no-print-directory", "-C", CSRC, "--eval", "probe-cmd: ; @echo $(NVCC) $(NVCCFLAGS)",
                          "probe-cmd"], check=True, capture_output=True, text=True).stdout.split()
    assert cmd and "arch=compute_100a,code=sm_100a" in cmd, cmd
    os.makedirs(os.path.dirname(PROBE_LIB), exist_ok=True)
    tmp = "%s.%d" % (PROBE_LIB, os.getpid())
    r = subprocess.run(cmd + ["-I.", "-shared", "-o", tmp, PROBE_SRC], cwd=CSRC, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    os.replace(tmp, PROBE_LIB)
    lib = ctypes.CDLL(PROBE_LIB)
    for name in ("probe_ldlt_small", "probe_chol_solve", "probe_chol_blocked"):
        getattr(lib, name).argtypes = [ctypes.c_int] + [ctypes.c_void_p] * 5
        getattr(lib, name).restype = ctypes.c_int
    lib.probe_blocked_reset.restype = None
    lib.probe_blocked_bad_flag.restype = ctypes.c_int
    lib.probe_blocked_work_capacity.restype = ctypes.c_size_t
    lib.probe_last_error.restype = ctypes.c_char_p
    return lib


def test_probe_compiles_and_the_single_cta_cholesky_refuses_n_above_160(probe_lib):
    # no device needed: launch_chol_solve refuses before it touches CUDA
    rc = probe_lib.probe_chol_solve(161, None, None, None, None, None)
    assert rc == abi.ERR_UNSUPPORTED and b"161" in probe_lib.probe_last_error()


@pytest.fixture(scope="module")
def probe(probe_lib):
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box")
    probe_lib.probe_blocked_reset()
    yield probe_lib
    torch.cuda.synchronize()
    probe_lib.probe_blocked_reset()


GUARD = 64               # elements of a known value on each side of every buffer a solver gets
SENTINEL = -3.0e300      # a value no solver writes
SENTINEL_I = 0x5A5A5A5A


class Run:
    """One solver call on device copies of (A, b); .get() synchronises and returns (y, status, A after the call).  Each buffer
    sits between two guard zones, and .get() checks that no solver wrote into them.  For k_chol_blocked it also checks that the
    workspace's solve buffer was sized for n before the launch."""

    def __init__(self, probe, solver, A, b):
        import torch
        n = A.shape[0]
        self.n = n
        self.bufs = [self._guarded(torch, np.ascontiguousarray(v, np.float64).ravel(), SENTINEL, torch.float64)
                     for v in (A, b, np.full(n, 7.0))]   # y = 7.0 is not a solution: every entry must be written
        self.bufs.append(self._guarded(torch, np.zeros(1, np.int32), SENTINEL_I, torch.int32))
        (_, self.A, _), (_, self.b, _), (_, self.y, _), (_, self.status, _) = self.bufs
        rc = getattr(probe, "probe_" + solver)(n, self.A.data_ptr(), self.b.data_ptr(), self.y.data_ptr(), self.status.data_ptr(), None)
        assert rc == abi.BA_OK, (solver, n, rc, probe.probe_last_error())
        if solver == "chol_blocked":
            assert probe.probe_blocked_work_capacity() >= n, (n, probe.probe_blocked_work_capacity())

    @staticmethod
    def _guarded(torch, values, sentinel, dtype):
        whole = torch.full((values.size + 2 * GUARD,), sentinel, dtype=dtype, device="cuda")   # GUARD keeps 16-byte alignment
        whole[GUARD:GUARD + values.size] = torch.from_numpy(values).cuda()
        return whole, whole[GUARD:GUARD + values.size], sentinel

    def get(self):
        import torch
        torch.cuda.synchronize()
        for whole, _, sentinel in self.bufs:
            g = torch.cat([whole[:GUARD], whole[-GUARD:]]).cpu().numpy()
            assert np.all(g == sentinel), (self.n, "a solver wrote outside its buffer")
        return self.y.cpu().numpy(), int(self.status.item()), self.A.cpu().numpy().reshape(self.n, self.n)


def nan_upper(A):
    A = A.copy()
    A[np.triu_indices(A.shape[0], 1)] = np.nan
    return A


# ---- matrices and the reference ------------------------------------------------------------------------------------------------
def spd(n, kappa, rng):
    """Q diag(l) Q^T, Q Haar-random, the eigenvalues log-spaced from 1 to 1 / kappa in random order."""
    Q, R = np.linalg.qr(rng.standard_normal((n, n)))
    Q *= np.sign(np.diag(R))
    lam = rng.permutation(np.logspace(0.0, -np.log10(kappa), n)) if n > 1 else np.ones(1)
    A = (Q * lam) @ Q.T
    return 0.5 * (A + A.T)


def rcs_shaped(n, rng):
    """A reduced camera system of a synthetic rig: 6x6 blocks over [4 cameras | markers], observations (frame, camera, marker)
    with random 8x6 Jacobians, the frames eliminated, a small LM diagonal, Jacobi-scaled to a unit diagonal; the leading n x n."""
    nf = -(-n // 6)
    ncam, nm = min(nf, 4), max(nf - 4, 0)
    T = max(1, nf // 2)
    nd = 6 * (T + nf)
    Hm = np.zeros((nd, nd))
    for t in range(T):
        seen = rng.choice(nm, min(nm, 3), replace=False) + ncam if nm else [None]
        for m in seen:
            for c in rng.choice(ncam, min(ncam, 2), replace=False):
                idx = np.r_[6 * t:6 * t + 6, 6 * (T + c):6 * (T + c) + 6]
                if m is not None:
                    idx = np.r_[idx, 6 * (T + m):6 * (T + m) + 6]
                J = rng.standard_normal((8, idx.size))
                Hm[np.ix_(idx, idx)] += J.T @ J
    e, f = slice(0, 6 * T), slice(6 * T, nd)
    Sr = Hm[f, f] - Hm[f, e] @ np.linalg.solve(Hm[e, e], Hm[e, f])
    Sr += 1e-4 * np.diag(np.maximum(np.diag(Hm[f, f]), 1.0))
    s = 1.0 / np.sqrt(np.diag(Sr))
    Sr = (Sr * s[:, None] * s[None, :])[:n, :n]
    Sr = 0.5 * (Sr + Sr.T)
    np.fill_diagonal(Sr, 1.0)
    return Sr


def real_rcs(oracle, which):
    """The reduced camera system of a reference fixture or a synthetic rig at its start, from the oracle's Jacobian."""
    if which == "hongo":
        pb, intr, side, fix0 = H.hongo()
    else:
        pr = S.marker_rig_b(*which, visibility=0.5)
        pb = F.ModelBFile(pr.n_time, pr.n_cam, pr.n_marker, pr.counts, pr.time_idx, pr.cam_idx, pr.marker_idx, pr.obs8, pr.params)
        intr, side, fix0 = pr.intr, pr.marker_side, 1
    Sr = H.reduced_system(oracle, pb, intr, side, fix0, pb.params)
    return 0.5 * (Sr + Sr.T)


def matvec_ld(A, v):
    out = np.empty(A.shape[0], LD)
    for i in range(0, A.shape[0], 512):
        out[i:i + 512] = A[i:i + 512].astype(LD) @ v
    return out


def reference(A, b):
    cf = sla.cho_factor(A, lower=True)
    x = sla.cho_solve(cf, b).astype(LD)
    for _ in range(2):
        r = b.astype(LD) - matvec_ld(A, x)
        x = x + sla.cho_solve(cf, r.astype(np.float64)).astype(LD)
    return x


def backward_error(A, b, y):
    r = b.astype(LD) - matvec_ld(A, y.astype(LD))
    return float(np.abs(r).max() / (np.abs(A).sum(axis=1).max() * np.abs(y).max() + np.abs(b).max()))


def forward_error(y, x):
    return float(np.sqrt(((y.astype(LD) - x) ** 2).sum() / (x ** 2).sum()))


def factor_residual(A, L, rng):
    Z = rng.standard_normal((A.shape[0], 4))
    worst = 0.0
    for z in Z.T:
        r = matvec_ld(A, z.astype(LD)) - matvec_ld(L, matvec_ld(np.ascontiguousarray(L.T), z.astype(LD)).astype(np.float64))
        worst = max(worst, float(np.abs(r).max() / (np.abs(A).sum(axis=1).max() * np.abs(z).max())))
    return worst


def negative_pivot(A, k):
    """A with its k-th pivot of L D L^T (no pivoting) moved to -1/2 of its value."""
    A = A.copy()
    d = A[k, k] - A[k, :k] @ np.linalg.solve(A[:k, :k], A[:k, k]) if k else A[0, 0]
    A[k, k] -= 1.5 * d
    return A


def pivots(A):
    """The pivots of L D L^T without pivoting, the order every solver here eliminates in."""
    A = A.copy()
    d = np.empty(A.shape[0])
    for k in range(A.shape[0]):
        d[k] = A[k, k]
        A[k + 1:, k + 1:] -= np.outer(A[k + 1:, k], A[k, k + 1:]) / d[k]
    return d


class Case:
    def __init__(self, name, A, kappa, rng):
        self.name, self.A, self.n = name, A, A.shape[0]
        self.b = rng.standard_normal(self.n)
        self.kappa = kappa if kappa is not None else float(np.linalg.cond(A))
        self.x = reference(A, self.b)
        self.fwd_bound = C * self.n * EPS * self.kappa
        self.bwd_bound = C * self.n * EPS


def cases_at(n, rng, kinds=("k1", "k1e6", "k1e12", "rcs")):
    for k in kinds:
        if k == "rcs":
            yield Case("rcs-shaped n=%d" % n, rcs_shaped(n, rng), None, rng)
        else:
            kappa = float(k[1:]) if n > 1 else 1.0   # a 1 x 1 matrix has kappa = 1 whatever was asked for
            yield Case("spd kappa=%g n=%d" % (kappa, n), spd(n, kappa, rng), kappa, rng)


WORST = {}   # solver -> largest backward and forward error seen, and each over its bound (printed with -s)


def record(solver, case, bwd, fwd):
    w = WORST.setdefault(solver, {"bwd": 0.0, "fwd": 0.0, "bwd_rel": 0.0, "fwd_rel": 0.0})
    w["bwd"], w["fwd"] = max(w["bwd"], bwd), max(w["fwd"], fwd)
    w["bwd_rel"], w["fwd_rel"] = max(w["bwd_rel"], bwd / case.bwd_bound), max(w["fwd_rel"], fwd / case.fwd_bound)


def check_solution(solver, case, y, status):
    assert status == 0, (solver, case.name, status)
    bwd, fwd = backward_error(case.A, case.b, y), forward_error(y, case.x)
    record(solver, case, bwd, fwd)
    assert bwd <= case.bwd_bound, (solver, case.name, bwd, case.bwd_bound)
    assert fwd <= case.fwd_bound, (solver, case.name, fwd, case.fwd_bound, case.kappa)


def check_small_solvers(probe, case):
    """k_ldlt_small and k_chol_solve on the lower triangle (strict upper = NaN), twice, and on the full symmetric matrix;
    k_chol_blocked on the same input: the three agree."""
    A_nan = nan_upper(case.A)
    runs = {s: [Run(probe, s, A_nan, case.b), Run(probe, s, A_nan, case.b), Run(probe, s, case.A, case.b)] for s in SMALL}
    runs["chol_blocked"] = [Run(probe, "chol_blocked", A_nan, case.b)]
    ys = {}
    for s in SMALL:
        (y, st, A_after), (y2, st2, _), (y3, st3, _) = (r.get() for r in runs[s])
        check_solution(s, case, y, st)
        assert st2 == st3 == 0
        assert np.array_equal(y, y2), (s, case.name, "repeat is not bit-identical")
        assert np.array_equal(y, y3), (s, case.name, "the upper triangle changed the result")
        assert np.array_equal(A_after, A_nan, equal_nan=True), (s, case.name, "S was modified")
        ys[s] = y
    y, st, _ = runs["chol_blocked"][0].get()
    check_solution("chol_blocked", case, y, st)
    ys["chol_blocked"] = y
    for a in SOLVERS:
        for b in SOLVERS:
            if a < b:
                d = forward_error(ys[a], ys[b].astype(LD))
                assert d <= case.fwd_bound, (a, b, case.name, d, case.fwd_bound)


def check_blocked(probe, case, rng):
    A_nan = nan_upper(case.A)
    r1, r2, r3 = Run(probe, "chol_blocked", A_nan, case.b), Run(probe, "chol_blocked", A_nan, case.b), \
        Run(probe, "chol_blocked", case.A, case.b)
    (y, st, F1), (y2, st2, F2), (y3, st3, F3) = r1.get(), r2.get(), r3.get()
    check_solution("chol_blocked", case, y, st)
    assert st2 == st3 == 0
    lo = np.tril_indices(case.n)
    assert np.array_equal(y, y2) and np.array_equal(F1, F2, equal_nan=True), (case.name, "repeat is not bit-identical")
    assert np.array_equal(y, y3) and np.array_equal(F1[lo], F3[lo]), (case.name, "the upper triangle changed the result")
    assert np.isnan(F1[np.triu_indices(case.n, 1)]).all(), (case.name, "the strict upper triangle was written")
    fr = factor_residual(case.A, np.tril(F1), rng)
    WORST.setdefault("chol_blocked_factor", {"res": 0.0})
    WORST["chol_blocked_factor"]["res"] = max(WORST["chol_blocked_factor"]["res"], fr)
    assert fr <= C * case.n * EPS, (case.name, fr)


# ---- CPU: the reference ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [3, 8, 17])
def test_reference_against_mpmath(n):
    # the reference must be far more accurate than anything the solvers are held to: 1 / 100 of the forward bound
    import mpmath
    mpmath.mp.dps = 40
    rng = np.random.default_rng(100 + n)
    for case in list(cases_at(n, rng)):
        xm = mpmath.lu_solve(mpmath.matrix(case.A.tolist()), mpmath.matrix(case.b.tolist()))
        x = mpmath.matrix([mpmath.mpf(float(v)) + mpmath.mpf(float(v - LD(float(v)))) for v in case.x])   # exact: two doubles
        err = mpmath.norm(x - xm) / mpmath.norm(xm)
        assert float(err) <= 0.01 * case.fwd_bound, (case.name, float(err), case.fwd_bound)


def test_failure_matrices_have_the_pivot_where_intended():
    for k in (0, 8, 32, 64, 140, 154, 156):
        d = pivots(negative_pivot(spd(157, 10.0, np.random.default_rng(k)), k))
        assert np.all(d[:k] > 0) and d[k] < 0, (k, d[k])


# ---- GPU ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["k1", "k1e6", "k1e12", "rcs"])
def test_small_solvers_every_n_up_to_160(probe, kind):
    rng = np.random.default_rng({"k1": 1, "k1e6": 2, "k1e12": 3, "rcs": 4}[kind])
    for n in range(1, 161):
        for case in cases_at(n, rng, (kind,)):
            check_small_solvers(probe, case)
    print("worst so far:", json.dumps(WORST))


@pytest.mark.gpu
def test_blocked_cholesky_at_every_size_class(probe):
    rng = np.random.default_rng(5)
    for n in BLOCKED_N:
        kinds = ("k1", "k1e6", "k1e12", "rcs") if n <= 1023 else ("k1e6",)   # the reference costs seconds above
        for case in cases_at(n, rng, kinds):
            check_blocked(probe, case, rng)
    print("worst so far:", json.dumps(WORST))


@pytest.mark.gpu
def test_real_reduced_camera_systems(probe, oracle):
    rng = np.random.default_rng(6)
    for which in ("hongo", (4, 20, 50, 5), (4, 40, 60, 6)):
        Sr = real_rcs(oracle, which)
        case = Case("rcs of %s n=%d" % (which, Sr.shape[0]), Sr, None, rng)
        if case.n <= 160:
            check_small_solvers(probe, case)
        check_blocked(probe, case, rng)
    print("worst so far:", json.dumps(WORST))


@pytest.mark.gpu
@pytest.mark.parametrize("bad", ["nan", "negative"])
def test_a_bad_pivot_raises_bit_2_and_returns_zero(probe, bad):
    # column 0, the panel boundaries 8 (k_ldlt_small), 32 and 64 (k_chol_blocked's panel and tile), inside the last partial panel
    # (152..156 of 8 columns, 128..156 of 32) and the last column
    for n, ks, solvers in ((157, (0, 8, 32, 64, 140, 154, 156), SOLVERS), (205, (0, 8, 32, 64, 197, 204), ("chol_blocked",))):
        rng = np.random.default_rng(n)
        A0 = spd(n, 10.0, rng)
        b = rng.standard_normal(n)
        good = Case("good n=%d" % n, A0, 10.0, rng)
        for k in ks:
            A = A0.copy()
            if bad == "nan":
                A[k, k] = np.nan
            else:
                A = negative_pivot(A, k)
            for s in solvers:
                y, st, _ = Run(probe, s, nan_upper(A), b).get()
                assert st == 2 and np.all(y == 0.0), (s, n, k, st, y[:4])
                if s == "chol_blocked":
                    assert probe.probe_blocked_bad_flag() == 1
                    # the next call on the same workspace starts clean
                    y, st, _ = Run(probe, s, nan_upper(good.A), good.b).get()
                    assert probe.probe_blocked_bad_flag() == 0
                    check_solution(s, good, y, st)


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["nan", "inf"])
def test_a_non_finite_right_hand_side_raises_bit_4(probe, what):
    for n, solvers in ((157, SOLVERS), (205, ("chol_blocked",))):
        rng = np.random.default_rng(n)
        A = spd(n, 10.0, rng)
        for j in (0, n // 2, n - 1):
            b = rng.standard_normal(n)
            b[j] = np.nan if what == "nan" else np.inf
            for s in solvers:
                y, st, _ = Run(probe, s, nan_upper(A), b).get()
                assert st == 4 and not np.all(np.isfinite(y)), (s, n, j, st)


@pytest.mark.gpu
def test_blocked_workspace_reuse_is_bit_identical_to_a_fresh_workspace(probe):
    rng = np.random.default_rng(7)
    mats = {n: (spd(n, 1e6, rng), rng.standard_normal(n)) for n in (161, 1537)}
    fresh = {}
    for n, (A, b) in mats.items():
        probe.probe_blocked_reset()
        fresh[n] = Run(probe, "chol_blocked", nan_upper(A), b).get()
        assert fresh[n][1] == 0
    probe.probe_blocked_reset()
    for n in (161, 1537, 161, 1537):   # a larger system after a smaller one, and the reverse
        y, st, Fn = Run(probe, "chol_blocked", nan_upper(mats[n][0]), mats[n][1]).get()
        assert st == 0 and np.array_equal(y, fresh[n][0]) and np.array_equal(Fn, fresh[n][2], equal_nan=True), n


# ---- the solver paths behind BA_DENSE_LDLT=0, at solve level ------------------------------------------------------------------
_CHILD = r"""
import json, sys
import torch
sys.path.insert(0, sys.argv[1])
from realsensecalibration_b200 import cuda, formats as F, synthetic as S
from tests import helpers as H
if sys.argv[2] == "hongo":
    pb, intr, side, fix0 = H.hongo()
else:
    pr = S.marker_rig_b(4, 20, 50, 5, visibility=0.5)
    pb = F.ModelBFile(pr.n_time, pr.n_cam, pr.n_marker, pr.counts, pr.time_idx, pr.cam_idx, pr.marker_idx, pr.obs8, pr.params)
    intr, side, fix0 = pr.intr, pr.marker_side, 1
P = cuda.Problem(0)
P.set_model_b(pb.n_cam, pb.n_time, pb.n_marker, pb.time_idx, pb.cam_idx, pb.marker_idx, pb.obs8, intr, side, fix0)
P.set_parameters(pb.params)
o = cuda.default_options()
o.force_generic_path = 1
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:   # which kernels ran
    s, rows = P.solve(o)
    torch.cuda.synchronize()
kernels = sorted({e.key for e in prof.key_averages()})
print(json.dumps({"rows": rows, "x": P.get_parameters().tolist(), "path": s.path_used, "rcs_dim": s.rcs_dim,
                  "solver": s.rcs_solver_used, "kernels": kernels}))
P.close()
"""


@pytest.mark.gpu
@pytest.mark.parametrize("which,n", [("hongo", 78), ("rig", 132)])
def test_cholesky_fallback_solves_match_the_oracle(oracle, which, n):
    # BA_DENSE_LDLT=0 with the default BA_DENSE_SMEM_MAX_N=96: hongo (n = 78) runs on k_chol_solve, the rig (n = 132) on
    # k_chol_blocked.  Both variables are read once per process, hence the child; its kernel trace shows which solver ran.
    from tests.test_gpu_parity import _check_rows
    env = dict(os.environ, BA_DENSE_LDLT="0")
    env.pop("BA_DENSE_SMEM_MAX_N", None)
    r = subprocess.run([sys.executable, "-c", _CHILD, ROOT, which], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["path"] == abi.PATH_GENERIC and out["rcs_dim"] == n and out["solver"] == abi.RCS_DENSE_CHOLESKY
    ran = {k for k in ("k_ldlt_small", "k_chol_solve", "k_chol_blocked") if any(k in name for name in out["kernels"])}
    assert ran == {"k_chol_solve" if which == "hongo" else "k_chol_blocked"}, (ran, out["kernels"])
    if which == "hongo":
        pb, intr, side, fix0 = H.hongo()
    else:
        pr = S.marker_rig_b(4, 20, 50, 5, visibility=0.5)
        pb = F.ModelBFile(pr.n_time, pr.n_cam, pr.n_marker, pr.counts, pr.time_idx, pr.cam_idx, pr.marker_idx, pr.obs8, pr.params)
        intr, side, fix0 = pr.intr, pr.marker_side, 1
    xo, _, rows_o = oracle.solve_model_b(pb, intr, side, fix0)
    _check_rows(out["rows"], rows_o)
    x = np.array(out["x"])
    assert np.abs(x - xo).max() < 1e-9
    if which == "hongo":
        H.check_hongo_golden(x, 1e-10, 1e-10)
