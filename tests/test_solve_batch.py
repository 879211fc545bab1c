"""ba_cuda_solve_batch: k independent solves of one structure in one launch, one CTA each.

Every instance must give, bit for bit, what a fresh problem gives when it is set up with the instance's observations and
start and solved alone: the parameters, every row field except iteration_time_s, every summary field except total_time_s
and the ms_* timings."""
import ctypes as C

import numpy as np
import pytest

from realsensecalibration_b200 import abi, cuda, synthetic as S
from tests import helpers as H

SUMMARY_SKIP = {"total_time_s", "ms_jacobian", "ms_schur", "ms_rcs_solve", "ms_update", "ms_cost", "ms_collective"}


@pytest.fixture(scope="module")
def gpu():
    if cuda.device_count() == 0:
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box")
    P = cuda.Problem(0)
    yield P
    P.close()


@pytest.fixture(scope="module")
def solo():
    P = cuda.Problem(0)
    yield P
    P.close()


# ---- cases: (kind, data, width of an observation, start, setter) ----------------------------------------------------
class Case:
    def __init__(self, kind, d, intr, side=None, fix0=None):
        self.kind, self.d, self.intr, self.side, self.fix0 = kind, d, intr, side, fix0
        self.obs = d.obs8 if kind == "B" else d.obs_xy
        self.start = np.asarray(d.params, np.float64)

    def load(self, P, obs=None):
        d = self.d
        o = self.obs if obs is None else obs
        if self.kind == "B":
            P.set_model_b(d.n_cam, d.n_time, d.n_marker, d.time_idx, d.cam_idx, d.marker_idx, o, self.intr, self.side, self.fix0)
        else:
            P.set_model_a(d.n_cam, d.n_pt, d.cam_idx, d.pt_idx, o, self.intr)


def case(name):
    if name == "hongo":
        pb, intr, side, fix0 = H.hongo()
        return Case("B", pb, intr, side, fix0)
    if name == "test2":
        pb, intr, side, fix0 = H.test2()
        return Case("B", pb, intr, side, fix0)
    if name == "two_cam":
        pa, intr = H.two_cam()
        return Case("A", pa, intr)
    if name == "two_cam_like":
        pa = S.two_cam_like(50, 11)
        return Case("A", pa, pa.intr)
    if name == "rig156":
        pr = S.marker_rig_b(4, 22, 11, 7)   # at the limits: n = 6 (4 + 22) = 156, 8 x 968 = 7744 residual rows
        return Case("B", pr, pr.intr, pr.marker_side, 1)
    raise KeyError(name)


def starts_and_obs(c, k, seed, dx=1e-3, px=0.3):
    rng = np.random.default_rng(seed)
    x = c.start[None, :] + rng.normal(0.0, dx, (k, c.start.shape[0]))
    obs = c.obs[None] + rng.normal(0.0, px, (k,) + c.obs.shape)
    return x, obs


def bits(v):
    return np.float64(v).tobytes()


def assert_same(got, want, tag):
    (x, s, rows), (xo, so, rows_o) = got, want
    assert x.tobytes() == xo.tobytes(), (tag, np.abs(x - xo).max())
    for name, _ in abi.Summary._fields_:
        if name not in SUMMARY_SKIP:
            assert bits(getattr(s, name)) == bits(getattr(so, name)), (tag, name, getattr(s, name), getattr(so, name))
    assert len(rows) == len(rows_o), (tag, len(rows), len(rows_o))
    for r, ro in zip(rows, rows_o):
        for name in r:
            if name != "iteration_time_s":
                assert bits(r[name]) == bits(ro[name]), (tag, r["iteration"], name, r[name], ro[name])


def solve_alone(P, c, x0, obs, opts):
    c.load(P, obs)
    P.set_parameters(x0)
    s, rows = P.solve(opts)
    return P.get_parameters(), s, rows


def check_batch(gpu, solo, c, x0, obs, opts=None, sample=None):
    c.load(gpu)
    xs, sums, rows = gpu.solve_batch(x0, obs, opts)
    idx = range(x0.shape[0]) if sample is None else sample
    for i in idx:
        want = solve_alone(solo, c, x0[i], None if obs is None else obs[i], opts or cuda.default_options())
        assert_same((xs[i], sums[i], rows[i]), want, i)
        assert sums[i].path_used == abi.PATH_RIG
    return xs, sums, rows


# ---- 1. bitwise equal to solo solves ----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hongo", "test2", "two_cam", "two_cam_like", "rig156"])
def test_matches_solo_solves(gpu, solo, name):
    c = case(name)
    x0, obs = starts_and_obs(c, 6, 100 + len(name))
    _, sums, _ = check_batch(gpu, solo, c, x0, obs)
    if name == "rig156":
        assert 6 * (c.d.n_cam + c.d.n_marker) == 156 and sums[0].num_residuals == 7744


@pytest.mark.gpu
@pytest.mark.parametrize("loss", [abi.LOSS_HUBER, abi.LOSS_CAUCHY])
def test_matches_solo_robust_loss(gpu, solo, loss):
    c = case("hongo")
    x0, obs = starts_and_obs(c, 5, 7 + loss, px=2.0)
    o = cuda.default_options()
    o.loss_function, o.loss_scale = loss, 1.5
    check_batch(gpu, solo, c, x0, obs, o)


@pytest.mark.gpu
def test_matches_solo_without_jacobi_scaling(gpu, solo):
    c = case("hongo")
    x0, obs = starts_and_obs(c, 5, 31)
    o = cuda.default_options()
    o.jacobi_scaling = 0
    check_batch(gpu, solo, c, x0, obs, o)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hongo", "two_cam_like"])
def test_matches_solo_with_the_models_observations(gpu, solo, name):
    c = case(name)
    x0, _ = starts_and_obs(c, 4, 9)
    check_batch(gpu, solo, c, x0, None)


# ---- 2. every wave shape ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 147, 148, 149])
def test_wave_shapes(gpu, solo, k):
    c = case("hongo")
    x0, obs = starts_and_obs(c, k, 1000 + k)
    check_batch(gpu, solo, c, x0, obs)


@pytest.mark.gpu
def test_thousand_instances_repeat_and_sample(gpu, solo):
    c = case("hongo")
    x0, obs = starts_and_obs(c, 1000, 4242)
    sample = np.random.default_rng(1).choice(1000, 60, replace=False)
    xs, sums, rows = check_batch(gpu, solo, c, x0, obs, sample=sample)
    xs2, sums2, rows2 = gpu.solve_batch(x0, obs)
    assert xs.tobytes() == xs2.tobytes()
    for i in range(1000):
        assert_same((xs2[i], sums2[i], rows2[i]), (xs[i], sums[i], rows[i]), i)


# ---- 3. instances that end differently in one launch ------------------------------------------------------------------
@pytest.mark.gpu
def test_instances_that_end_differently(gpu, solo):
    c = case("hongo")
    c.load(solo)
    solo.set_parameters(c.start)
    solo.solve()
    x_sol = solo.get_parameters()
    d = np.random.default_rng(5).normal(0.0, 1.0, x_sol.shape)
    x0 = np.stack([x_sol + sc * d for sc in (0.0, 1e-3, 1e-2, 3e-2, 0.1, 0.3)] + [np.full_like(x_sol, np.nan)])
    obs = np.repeat(c.obs[None], x0.shape[0], axis=0)
    o = cuda.default_options()
    o.max_num_iterations = 5
    _, sums, _ = check_batch(gpu, solo, c, x0, obs, o)
    reasons = [s.termination_reason for s in sums]
    assert abi.REASON_FUNCTION_TOLERANCE in reasons and abi.REASON_MAX_ITERATIONS in reasons, reasons
    assert reasons[-1] == abi.REASON_INITIAL_EVALUATION_FAILED and sums[-1].termination_type == abi.FAILURE
    assert any(s.num_unsuccessful_steps > 0 for s in sums)


# ---- 4. past the row cap ----------------------------------------------------------------------------------------------
def long_options():
    o = cuda.default_options()
    o.max_num_iterations = 300
    o.function_tolerance = o.gradient_tolerance = o.parameter_tolerance = 0.0
    o.max_trust_region_radius = 1e-2
    return o


@pytest.mark.gpu
def test_past_the_row_cap(gpu, solo):
    c = case("hongo")
    x0, obs = starts_and_obs(c, 3, 77)
    o = long_options()
    xs, sums, rows = check_batch(gpu, solo, c, x0, obs, o)
    assert all(s.num_iterations == 301 and len(r) == 301 for s, r in zip(sums, rows))
    # fewer rows kept than recorded, and none
    xs_c, sums_c, rows_c = gpu.solve_batch(x0, obs, o, rows_cap=100)
    xs_n, sums_n, rows_n = gpu.solve_batch(x0, obs, o, rows_cap=0)
    assert xs_c.tobytes() == xs.tobytes() and xs_n.tobytes() == xs.tobytes()
    for i in range(3):
        assert sums_c[i].num_iterations == 301 and sums_n[i].num_iterations == 301
        assert bits(sums_n[i].initial_cost) == bits(sums[i].initial_cost) and bits(sums_n[i].final_cost) == bits(sums[i].final_cost)
        assert len(rows_c[i]) == 100 and rows_n[i] == []
        for r, ro in zip(rows_c[i], rows[i][:100]):
            assert all(bits(r[n]) == bits(ro[n]) for n in r if n != "iteration_time_s")


# ---- 5. the problem is left alone -------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_problem_is_left_alone(gpu, solo):
    c = case("hongo")
    x0, obs = starts_and_obs(c, 8, 3)

    def sequence(P, batch):
        c.load(P)
        P.set_parameters(c.start)
        P.save_parameters()
        s1, r1 = P.solve()
        if batch:
            P.solve_batch(x0, obs, long_options())
        x1, rows1 = P.get_parameters(), P._rows()
        P.restore_parameters()
        x_restored = P.get_parameters()
        s2, r2 = P.solve()
        return x1, rows1, x_restored, P.get_parameters(), s2, r2

    a, b = sequence(gpu, True), sequence(solo, False)
    assert a[0].tobytes() == b[0].tobytes()
    assert_same((a[0], abi.Summary(), a[1]), (b[0], abi.Summary(), b[1]), "rows")
    assert a[2].tobytes() == c.start.tobytes() == b[2].tobytes()
    assert_same((a[3], a[4], a[5]), (b[3], b[4], b[5]), "later solve")


# ---- 6. Monte Carlo agrees with the covariance ------------------------------------------------------------------------
@pytest.mark.gpu
def test_monte_carlo_agrees_with_the_covariance(gpu):
    sigma, trials = 0.5, 2000
    pr = S.marker_rig_b(3, 6, 20, 11, noise_px=0.0)
    c = Case("B", pr, pr.intr, pr.marker_side, 1)
    c.load(gpu)
    gpu.set_parameters(pr.truth)
    kept, _, _ = gpu.covariance()
    rng = np.random.default_rng(2025)
    obs = pr.obs8[None] + rng.normal(0.0, sigma, (trials,) + pr.obs8.shape)
    xs, sums, _ = gpu.solve_batch(np.repeat(pr.truth[None], trials, axis=0), obs, rows_cap=0)
    assert all(s.termination_type == abi.CONVERGENCE for s in sums)
    dev = (xs - pr.truth[None])[:, 6:18]   # cameras 1 and 2
    ratio = dev.std(axis=0) / (sigma * np.sqrt(np.diag(kept)[6:18]))
    assert np.all((ratio >= 0.9) & (ratio <= 1.1)), ratio
    maha = np.einsum("ni,ij,nj->n", dev[:, :6], np.linalg.inv(sigma ** 2 * kept[6:12, 6:12]), dev[:, :6])
    assert 0.92 * 6 <= maha.mean() <= 1.08 * 6, maha.mean()


# ---- 7. refusals ------------------------------------------------------------------------------------------------------
def refused(code, fn):
    with pytest.raises(cuda.BAError) as e:
        fn()
    assert e.value.code == code, e.value


@pytest.mark.gpu
def test_refusals_leave_the_problem_usable(gpu, solo):
    c = case("hongo")
    x0, obs = starts_and_obs(c, 2, 8)
    pr = S.marker_rig_b(4, 20, 200, 0xBA02)
    cfg2 = Case("B", pr, pr.intr, pr.marker_side, 1)
    cfg2.load(gpu)
    assert pr.n_mobs == 16000
    refused(abi.ERR_UNSUPPORTED, lambda: gpu.solve_batch(np.repeat(pr.params[None], 2, axis=0)))
    c.load(gpu)
    o = cuda.default_options(); o.rcs_solver = abi.RCS_PCG
    refused(abi.ERR_UNSUPPORTED, lambda: gpu.solve_batch(x0, obs, o))
    o = cuda.default_options(); o.force_generic_path = 1
    refused(abi.ERR_UNSUPPORTED, lambda: gpu.solve_batch(x0, obs, o))
    refused(abi.ERR_INVALID_ARGUMENT, lambda: gpu.solve_batch(x0[:0], obs[:0]))
    o = cuda.default_options(); o.loss_function = abi.LOSS_HUBER; o.loss_scale = 0.0
    refused(abi.ERR_INVALID_ARGUMENT, lambda: gpu.solve_batch(x0, obs, o))
    gpu.set_parameters(c.start)
    gpu.solve_begin()
    refused(abi.ERR_STATE, lambda: gpu.solve_batch(x0, obs))
    gpu.solve_iterate(1 << 30)
    gpu.solve_end()
    empty = cuda.Problem(0)
    try:
        refused(abi.ERR_STATE, lambda: empty.solve_batch(np.zeros((2, 6))))
    finally:
        empty.close()
    check_batch(gpu, solo, c, x0, obs)   # still solves, and as a fresh problem does


@pytest.mark.gpu
def test_invalid_arguments_of_the_c_abi(gpu):
    c = case("hongo")
    c.load(gpu)
    n = gpu.num_parameters()
    x = np.repeat(c.start[None], 2, axis=0)
    L = cuda.lib()
    rows = (abi.Iteration * 4)()
    assert L.ba_cuda_solve_batch(gpu._h, None, C.c_int32(2), None, None, None, None, C.c_int32(0)) == abi.ERR_INVALID_ARGUMENT
    assert L.ba_cuda_solve_batch(gpu._h, None, C.c_int32(-1), x.ctypes.data_as(C.c_void_p), None, None, None, C.c_int32(0)) == abi.ERR_INVALID_ARGUMENT
    assert L.ba_cuda_solve_batch(gpu._h, None, C.c_int32(2), x.ctypes.data_as(C.c_void_p), None, None, rows, C.c_int32(0)) == abi.ERR_INVALID_ARGUMENT
    # NULL options are the defaults, NULL summaries and rows are allowed
    assert L.ba_cuda_solve_batch(gpu._h, None, C.c_int32(2), x.ctypes.data_as(C.c_void_p), None, None, None, C.c_int32(0)) == 0
    assert x.shape == (2, n) and np.isfinite(x).all() and x[0].tobytes() == x[1].tobytes()


def cpu_problem(model, n_obs):
    """A Problem object with no device behind it: enough for the shape checks, which run before the library is called."""
    P = cuda.Problem.__new__(cuda.Problem)
    P._h = C.c_void_p()
    P.model, P.n_obs = model, n_obs
    return P


def test_shape_errors_are_raised_before_the_library_is_called():
    for model, width in (("A", 2), ("B", 8)):
        P = cpu_problem(model, 5)   # num_parameters() of no problem is 0
        with pytest.raises(ValueError):
            P.solve_batch(np.zeros((3, 4)))
        with pytest.raises(ValueError):
            P.solve_batch(np.zeros(3))
        with pytest.raises(ValueError):
            P.solve_batch(np.zeros((3, 0)), np.zeros((3, 5, 10 - width)))
        with pytest.raises(ValueError):
            P.solve_batch(np.zeros((3, 0)), np.zeros((2, 5, width)))
        with pytest.raises(ValueError):
            P.solve_batch(np.zeros((3, 0)), np.zeros((3, 4, width)))


# ---- 8. kernel stats --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_kernel_stats_name_the_batch_kernel(gpu):
    c = case("hongo")
    c.load(gpu)
    x0, obs = starts_and_obs(c, 3, 12)
    gpu.reset_stats()
    gpu.solve_batch(x0, obs, long_options())
    stats = {s["name"]: s["launches"] for s in gpu.kernel_stats()}
    assert stats.get("rig_lm_batch") == 2, stats   # 301 rows: one relaunch past the 256-row cap
    assert "rig_lm_whole_loop" not in stats
