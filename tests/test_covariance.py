"""ba_cuda_covariance (ceres::Covariance of Model B) against a numpy twin: (J^T J)^-1 over the free parameter blocks, J from the
CPU oracle (rows of a marker observation scaled by sqrt(rho'(|r|^2)) under a robust loss: Ceres 1.14's Corrector, whose alpha is
0 for Huber and Cauchy because rho'' <= 0).  The twin itself is pinned by a Monte Carlo experiment on the CPU."""
import os
import re
import subprocess

import numpy as np
import pytest

from realsensecalibration_b200 import abi, cuda, formats as F, synthetic as S
from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "realsensecalibration_b200", "host", "ba_main_calibration")


# ---- the numpy twin ----------------------------------------------------------------------------------------------------------
def _rho1(loss, a, s):
    if loss == abi.LOSS_HUBER:
        return np.where(s > a * a, a / np.sqrt(np.maximum(s, 1e-300)), 1.0)
    if loss == abi.LOSS_CAUCHY:
        return 1.0 / (1.0 + s / (a * a))
    return np.ones_like(s)


def normal_equations(oracle, pb, intr, side, fix0, x, loss=abi.LOSS_NONE, scale=1.0):
    """J^T J as a dense [6 nblk]^2 matrix over the blocks [cameras | frames | markers] and the mask of the free blocks.
    Accumulated block-wise (np.add.at over the 3 x 3 block pairs of every marker observation)."""
    C, T, M = pb.n_cam, pb.n_time, pb.n_marker
    _, res, jac = oracle.eval_model_b(pb, intr, side, fix0, params=x)
    w = np.sqrt(_rho1(loss, scale, (res ** 2).sum(axis=1)))
    J = jac.reshape(-1, 3, 8, 6).transpose(0, 2, 1, 3) * w[:, None, None, None]   # [obs, row, block, col]
    blk = np.stack([pb.cam_idx, C + pb.time_idx, C + T + pb.marker_idx], 1)
    nb = C + T + M
    Hb = np.zeros((nb, nb, 6, 6))
    for a in range(3):
        for b in range(3):
            np.add.at(Hb, (blk[:, a], blk[:, b]), np.einsum("nri,nrj->nij", J[:, :, a], J[:, :, b]))
    free = np.zeros(nb, bool)
    free[blk.ravel()] = True
    free[0] = False                       # camera 0 is never a parameter block
    if fix0:
        free[C + T] = False               # marker 0 under the Main dispatch
    return Hb.transpose(0, 2, 1, 3).reshape(6 * nb, 6 * nb), free


def twin(oracle, pb, intr, side, fix0, x, loss=abi.LOSS_NONE, scale=1.0):
    """(cov_kept [6(C+M)]^2 in the order [cameras | markers], cov_frames [T, 6, 6]) as ba_cuda_covariance lays them out."""
    C, T, M = pb.n_cam, pb.n_time, pb.n_marker
    Hd, free = normal_equations(oracle, pb, intr, side, fix0, x, loss, scale)
    fs = np.repeat(free, 6)
    cov = np.zeros_like(Hd)
    cov[np.ix_(fs, fs)] = np.linalg.inv(Hd[np.ix_(fs, fs)])
    kept = np.r_[np.arange(6 * C), np.arange(6 * (C + T), 6 * (C + T + M))]
    frames = np.stack([cov[6 * (C + t):6 * (C + t + 1), 6 * (C + t):6 * (C + t + 1)] for t in range(T)]) if T else np.zeros((0, 6, 6))
    return cov[np.ix_(kept, kept)], frames


def reduced_pivots(oracle, pb, intr, side, fix0, x):
    """Pivots of L D L^T (no pivoting) of the Jacobi-scaled reduced system over the free kept blocks, and its diagonal."""
    C, T = pb.n_cam, pb.n_time
    Hd, free = normal_equations(oracle, pb, intr, side, fix0, x)
    s = 1.0 / (1.0 + np.sqrt(np.diag(Hd)))
    Hs = Hd * s[:, None] * s[None, :]
    fs = np.repeat(free, 6)
    is_frame = np.zeros(Hd.shape[0], bool)
    is_frame[6 * C:6 * (C + T)] = True
    e, f = np.flatnonzero(fs & is_frame), np.flatnonzero(fs & ~is_frame)
    Ssys = Hs[np.ix_(f, f)] - Hs[np.ix_(f, e)] @ np.linalg.solve(Hs[np.ix_(e, e)], Hs[np.ix_(e, f)])
    A = Ssys.copy()
    d = np.zeros(A.shape[0])
    for k in range(A.shape[0]):
        d[k] = A[k, k]
        if k + 1 < A.shape[0]:
            A[k + 1:, k + 1:] -= np.outer(A[k + 1:, k], A[k, k + 1:]) / d[k]
    return d, np.diag(Ssys)


# ---- CPU: the twin is the right quantity -------------------------------------------------------------------------------------
def test_monte_carlo_pins_the_twin(oracle):
    # 300 solves from the truth with fresh noise of sigma px per coordinate: the spread of camera 1 and 2 must be
    # sigma^2 (J^T J)^-1 at the truth
    sigma, trials = 0.5, 300
    pr = S.marker_rig_b(3, 6, 20, 11, noise_px=0.0)
    assert pr.n_mobs == 360
    clean = pr.obs8.copy()
    base = F.ModelBFile(pr.n_time, pr.n_cam, pr.n_marker, pr.counts, pr.time_idx, pr.cam_idx, pr.marker_idx, clean, pr.truth)
    kept, _ = twin(oracle, base, pr.intr, pr.marker_side, 1, pr.truth)
    rng = np.random.default_rng(2024)
    dev = np.zeros((trials, 12))
    for k in range(trials):
        pb = F.ModelBFile(pr.n_time, pr.n_cam, pr.n_marker, pr.counts, pr.time_idx, pr.cam_idx, pr.marker_idx,
                          clean + rng.normal(0.0, sigma, clean.shape), pr.truth)
        x, s, _ = oracle.solve_model_b(pb, pr.intr, pr.marker_side, 1)
        assert s.termination_type == abi.CONVERGENCE
        dev[k] = (x - pr.truth)[6:18]              # cameras 1 and 2
    sd_twin = sigma * np.sqrt(np.diag(kept)[6:18])
    ratio = dev.std(axis=0) / sd_twin
    assert np.all((ratio > 0.75) & (ratio < 1.25)), ratio
    C1 = sigma ** 2 * kept[6:12, 6:12]
    maha = np.einsum("ni,ij,nj->n", dev[:, :6], np.linalg.inv(C1), dev[:, :6])
    assert 0.75 * 6 <= maha.mean() <= 1.25 * 6, maha.mean()


def test_twin_pivot_test_on_the_reference_fixtures(oracle):
    # test2 (marker 0 free): the gauge freedom of frame poses against marker poses is a 6-dimensional null space
    pb, intr, side, fix0 = H.test2()
    x, _, _ = oracle.solve_model_b(pb, intr, side, fix0)
    d, diag = reduced_pivots(oracle, pb, intr, side, fix0, x)
    assert d.shape[0] == 30
    assert (d <= 1e-12 * diag.max()).sum() == 6
    # hongo (marker 0 fixed): well posed
    pb, intr, side, fix0 = H.hongo()
    x, _, _ = oracle.solve_model_b(pb, intr, side, fix0)
    d, diag = reduced_pivots(oracle, pb, intr, side, fix0, x)
    assert d.shape[0] == 78
    assert d.min() / diag.max() > 1e-4


# ---- GPU ---------------------------------------------------------------------------------------------------------------------
def _problem(pb, intr, side, fix0):
    P = cuda.Problem(0)
    P.set_model_b(pb.n_cam, pb.n_time, pb.n_marker, pb.time_idx, pb.cam_idx, pb.marker_idx, pb.obs8, intr, side, fix0)
    P.set_parameters(pb.params)
    return P


def _rig(*args, **kw):
    pr = S.marker_rig_b(*args, **kw)
    pb = F.ModelBFile(pr.n_time, pr.n_cam, pr.n_marker, pr.counts, pr.time_idx, pr.cam_idx, pr.marker_idx, pr.obs8, pr.params)
    return pb, pr.intr, pr.marker_side, 1


def _check_against_twin(oracle, name, pb, intr, side, fix0, options=None, loss=abi.LOSS_NONE, scale=1.0):
    P = _problem(pb, intr, side, fix0)
    P.solve(options)
    x = P.get_parameters()
    kept, frames, ratio = P.covariance(options)
    P.close()
    tk, tf = twin(oracle, pb, intr, side, fix0, x, loss, scale)
    big = max(np.abs(tk).max(), np.abs(tf).max())
    err_k, err_f = np.abs(kept - tk).max() / big, np.abs(frames - tf).max() / big
    print("covariance %s: n = %d, max |gpu - twin| / max |twin| = %.2e (kept) %.2e (frames), smallest pivot ratio %.3e" %
          (name, kept.shape[0], err_k, err_f, ratio))
    assert err_k <= 1e-9 and err_f <= 1e-9, (err_k, err_f)
    assert np.array_equal(kept, kept.T)
    assert np.array_equal(frames, frames.transpose(0, 2, 1))
    assert np.all(kept[:6] == 0) and np.all(kept[:, :6] == 0)          # camera 0 is not a parameter
    if fix0:
        m0 = 6 * pb.n_cam
        assert np.all(kept[m0:m0 + 6] == 0) and np.all(kept[:, m0:m0 + 6] == 0)
    return kept, frames, ratio


@pytest.mark.gpu
def test_gpu_hongo_matches_the_twin(oracle):
    _, _, ratio = _check_against_twin(oracle, "hongo", *H.hongo())
    assert 1e-4 < ratio <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(4, 20, 50, 5), (4, 40, 60, 6)])   # n = 144 and 264: both sides of the single-CTA limit 160
def test_gpu_synthetic_rigs_match_the_twin(oracle, shape):
    pb, intr, side, fix0 = _rig(*shape, visibility=0.5)
    _check_against_twin(oracle, "rig %s" % (shape,), pb, intr, side, fix0)


@pytest.mark.gpu
def test_gpu_cfg3_shaped_rig_matches_the_twin(oracle):
    pb, intr, side, fix0 = _rig(8, 100, 50, 3)
    kept, _, _ = _check_against_twin(oracle, "8 x 100 x 50", pb, intr, side, fix0)
    assert kept.shape == (648, 648)


@pytest.mark.gpu
@pytest.mark.parametrize("loss", [abi.LOSS_HUBER, abi.LOSS_CAUCHY])
def test_gpu_robust_loss_matches_the_twin_with_the_corrector(oracle, loss):
    pr = S.marker_rig_b(4, 12, 30, 7)
    rng = np.random.default_rng(4)
    obs8 = pr.obs8.copy()
    idx = rng.choice(obs8.shape[0], 40, replace=False)
    obs8[idx] += rng.normal(0.0, 25.0, (40, 8))
    pb = F.ModelBFile(pr.n_time, pr.n_cam, pr.n_marker, pr.counts, pr.time_idx, pr.cam_idx, pr.marker_idx, obs8, pr.params)
    o = cuda.default_options()
    o.loss_function = loss; o.loss_scale = 3.0
    _, res, _ = oracle.eval_model_b(pb, pr.intr, pr.marker_side, 1)
    assert ((res ** 2).sum(axis=1) > 9.0).sum() >= 30           # the outliers are in the robust regime
    _check_against_twin(oracle, "loss %d" % loss, pb, pr.intr, pr.marker_side, 1, o, loss, 3.0)


@pytest.mark.gpu
def test_gpu_test2_is_rank_deficient():
    P = _problem(*H.test2())
    P.solve()
    with pytest.raises(cuda.BAError) as e:
        P.covariance()
    P.close()
    assert e.value.code == abi.ERR_RANK_DEFICIENT and str(abi.ERR_RANK_DEFICIENT) in str(e.value)
    assert e.value.smallest_pivot_ratio < 1e-12


@pytest.mark.gpu
def test_gpu_refusals():
    pa, intr = H.two_cam()
    P = cuda.Problem(0)
    P.set_model_a(pa.n_cam, pa.n_pt, pa.cam_idx, pa.pt_idx, pa.obs_xy, intr)
    P.set_parameters(pa.params)
    with pytest.raises(cuda.BAError) as e:
        P.covariance()
    assert e.value.code == abi.ERR_UNSUPPORTED and "gauge" in str(e.value)
    P.close()
    P = _problem(*H.hongo())
    P.solve_begin()
    with pytest.raises(cuda.BAError) as e:
        P.covariance()
    assert e.value.code == abi.ERR_STATE
    while not P.solve_iterate(100):
        pass
    P.solve_end()
    P.covariance()   # after the solve it runs
    P.close()


@pytest.mark.gpu
def test_gpu_covariance_is_deterministic():
    pb, intr, side, fix0 = _rig(4, 40, 60, 6, visibility=0.5)
    P = _problem(pb, intr, side, fix0)
    P.solve()
    a = P.covariance()
    b = P.covariance()
    P.close()
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2] == b[2]


def _rows_without_times(rows):
    return [{k: v for k, v in r.items() if k != "iteration_time_s"} for r in rows]


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["hongo", "generic"])
def test_gpu_covariance_does_not_disturb_a_later_solve(which):
    pb, intr, side, fix0 = H.hongo() if which == "hongo" else _rig(4, 20, 50, 5, visibility=0.5)
    out = []
    for with_cov in (False, True):
        P = _problem(pb, intr, side, fix0)
        P.save_parameters()
        s, _ = P.solve()
        assert s.path_used == (abi.PATH_RIG if which == "hongo" else abi.PATH_GENERIC)
        if with_cov:
            P.covariance()
        P.restore_parameters()
        s, rows = P.solve()
        out.append((_rows_without_times(rows), P.get_parameters()))
        P.close()
    assert out[0][0] == out[1][0]
    assert np.array_equal(out[0][1], out[1][1])


@pytest.mark.gpu
def test_gpu_host_program_prints_the_camera_standard_deviations(tmp_path, oracle):
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "realsensecalibration_b200", "host")])
    r = subprocess.run([EXE, H.GOLDEN, str(tmp_path), "covariance"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    got = {int(m.group(1)): np.array(m.group(2).split(), float)
           for m in re.finditer(r"^covariance: camera (\d+) sd (.*)$", r.stdout, re.M)}
    pb, intr, side, fix0 = H.hongo()
    assert sorted(got) == list(range(pb.n_cam))
    xo, _, _ = oracle.solve_model_b(pb, intr, side, fix0)
    kept, _ = twin(oracle, pb, intr, side, fix0, xo)
    for c in range(pb.n_cam):
        sd = np.sqrt(np.diag(kept)[6 * c:6 * c + 6])
        assert np.all(np.abs(got[c] - sd) <= 6e-7 * sd + 1e-300), (c, got[c], sd)
    # the default mode prints no covariance
    r = subprocess.run([EXE, H.GOLDEN, str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "covariance:" not in r.stdout
