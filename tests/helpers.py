"""Shared fixtures-as-functions for the parity tests (host-side numpy only)."""
import os

import numpy as np

from realsensecalibration_b200 import abi, formats as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_common")

# Known-answer traces of the reference's fixtures (SURVEY.md 8c / BASELINE.md 2): the
# end states match the reference's committed Ceres outputs to 1e-15.
HONGO_COSTS = [1.387966960542683e+05, 1.044261171521932e+05, 1.619009257909599e+04, 1.140581757675756e+04,
               5.783243408891863e+02, 1.441617307924972e+02, 1.436293888518609e+02]
HONGO_RADII = [1e4, 9.589347493e3, 2.876804248e4, 2.770715625e4, 8.312146876e4, 2.493644063e5, 7.480932188e5]
TEST2_COSTS = [1.357816158655430e+02, 1.343560334876707e+01, 1.330172662558997e+01, 1.330170910708654e+01]
TEST2_RADII = [1e4, 3e4, 9e4, 2.7e5]
TWO_CAM_COSTS = [5.617747098021e+00, 2.512595816529e-04, 2.734342332794e-12]
# G2's configuration is no longer in the reference source tree (SURVEY.md 8c, appendix A-7)
TEST2_MARKER_SIDE = 0.048
TEST2_SERIALS = ("819612072493", "825312072048")
TEST1_SERIAL = "825312072048"  # serial_numbers[1], Test1_BundleAdjustment/main.cpp:21,73


def intrinsics(serials):
    return np.stack([F.load_intrinsics(os.path.join(GOLDEN, "Calibration", "Intrinsics", "%s.xml" % s))[0] for s in serials])


def hongo():
    pb = F.load_correspondence(os.path.join(GOLDEN, "Correspondence", "hongo", "correspondence.txt"))
    return pb, intrinsics(F.SERIAL_NUMBERS), F.MARKER_SIDE, 1


def test2():
    pb = F.load_correspondence(os.path.join(GOLDEN, "Correspondence", "test2", "correspondence_test.txt"))
    return pb, intrinsics(TEST2_SERIALS), TEST2_MARKER_SIDE, 0


def two_cam():
    pa = F.load_two_cam_data(os.path.join(GOLDEN, "Correspondence", "two_cam_data.txt"))
    return pa, intrinsics((TEST1_SERIAL,))[0]


def rodrigues_np(rvec):
    """cv::Rodrigues rvec -> R, numpy twin used to compare against XML goldens."""
    r = np.asarray(rvec, np.float64)
    t = np.linalg.norm(r)
    if t < np.finfo(np.float64).eps:
        return np.eye(3)
    k = r / t
    K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.cos(t) * np.eye(3) + (1 - np.cos(t)) * np.outer(k, k) + np.sin(t) * K


def check_hongo_golden(x, tol_R=5e-14, tol_t=5e-14):
    gold = F.load_opencv_xml(os.path.join(GOLDEN, "Correspondence", "hongo", "Camera_Transform.xml"))
    for c in range(4):
        assert np.abs(rodrigues_np(x[6 * c:6 * c + 3]) - gold["R%d" % c]).max() <= tol_R, c
        assert np.abs(x[6 * c + 3:6 * c + 6] - gold["t%d" % c].ravel()).max() <= tol_t, c


def check_test2_golden(x, tol=5e-14):
    gold = F.load_opencv_xml(os.path.join(GOLDEN, "Correspondence", "test2", "Camera_Transform.xml"))
    for c in range(2):
        assert np.abs(x[6 * c:6 * c + 3] - gold["R%d" % c].ravel()).max() <= tol, c
        assert np.abs(x[6 * c + 3:6 * c + 6] - gold["t%d" % c].ravel()).max() <= tol, c


def rel(a, b):
    return abs(a - b) / max(abs(b), 1e-300)


# ---- the numpy twin of the normal equations (test_covariance.py, test_dense_solvers.py) ----
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


def reduced_system(oracle, pb, intr, side, fix0, x):
    """The Jacobi-scaled reduced camera system over the free kept blocks (the frames eliminated), without an LM diagonal."""
    C, T = pb.n_cam, pb.n_time
    Hd, free = normal_equations(oracle, pb, intr, side, fix0, x)
    s = 1.0 / (1.0 + np.sqrt(np.diag(Hd)))
    Hs = Hd * s[:, None] * s[None, :]
    fs = np.repeat(free, 6)
    is_frame = np.zeros(Hd.shape[0], bool)
    is_frame[6 * C:6 * (C + T)] = True
    e, f = np.flatnonzero(fs & is_frame), np.flatnonzero(fs & ~is_frame)
    return Hs[np.ix_(f, f)] - Hs[np.ix_(f, e)] @ np.linalg.solve(Hs[np.ix_(e, e)], Hs[np.ix_(e, f)])
