"""ctypes binding of csrc/libba_cuda.so (the ba_cuda_* C ABI of include/ba_cuda.h).

Host-side plumbing for tests and bench.py: numpy arrays in, numpy arrays out, all
arithmetic happens in the CUDA library.  There is no fallback: a missing library or a
missing GPU raises.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from .abi import UNIQUE_ID_BYTES, Iteration, KernelStat, Options, Summary

_CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc")
LIB_PATH = os.path.join(_CSRC, "libba_cuda.so")
_LIB = None

EXPORTS = [
    "ba_cuda_options_init", "ba_cuda_create", "ba_cuda_destroy", "ba_cuda_last_error", "ba_cuda_device_count",
    "ba_cuda_comm_unique_id", "ba_cuda_comm_init", "ba_cuda_shard_blocks", "ba_cuda_set_model_a", "ba_cuda_set_model_b",
    "ba_cuda_set_parameters", "ba_cuda_get_parameters", "ba_cuda_num_parameters", "ba_cuda_solve",
    "ba_cuda_get_iterations", "ba_cuda_eval", "ba_cuda_last_kernel_ms", "ba_cuda_reprojection_error",
    "ba_cuda_project_points_error", "ba_cuda_model_b_outputs", "ba_cuda_solve_begin", "ba_cuda_solve_iterate",
    "ba_cuda_solve_end", "ba_cuda_set_stream", "ba_cuda_get_kernel_stats", "ba_cuda_num_launches", "ba_cuda_reset_stats",
    "ba_cuda_save_parameters", "ba_cuda_restore_parameters", "ba_cuda_project_points_error_rt",
    "ba_cuda_release_cached_memory", "ba_cuda_marker_corners", "ba_cuda_compose_poses", "ba_cuda_covariance",
    "ba_cuda_solve_batch",
]


class BAError(RuntimeError):
    """A ba_cuda_* call failed; `code` is its ba_status (abi.ERR_*)."""

    def __init__(self, message, code=None):
        super().__init__(message)
        self.code = code


def build():
    """Compiles libba_cuda.so for sm_100a in tree (nvcc cross-compiles without a GPU)."""
    subprocess.check_call(["make", "-s", "-C", _CSRC])


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise BAError("CUDA library %s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.ba_cuda_last_error.restype = C.c_char_p
        L.ba_cuda_num_parameters.restype = C.c_int64
        L.ba_cuda_last_kernel_ms.restype = C.c_double
        L.ba_cuda_num_launches.restype = C.c_int64
        L.ba_cuda_reset_stats.restype = None
        L.ba_cuda_release_cached_memory.restype = None
        L.ba_cuda_options_init.argtypes = [C.POINTER(Options)]
        _LIB = L
    return _LIB


def _error(rc):
    return BAError("ba_cuda error %d: %s" % (rc, lib().ba_cuda_last_error().decode()), rc)


def _check(rc):
    if rc != 0:
        raise _error(rc)


def default_options():
    o = Options()
    lib().ba_cuda_options_init(C.byref(o))
    return o


def device_count():
    return int(lib().ba_cuda_device_count())


def release_cached_memory():
    lib().ba_cuda_release_cached_memory()


def shard_blocks(weights, world_size):
    w = np.ascontiguousarray(weights, np.int64)
    out = np.zeros(world_size + 1, np.int64)
    _check(lib().ba_cuda_shard_blocks(C.c_int64(w.shape[0]), w.ctypes, C.c_int(world_size), out.ctypes))
    return out


def comm_unique_id():
    buf = (C.c_uint8 * UNIQUE_ID_BYTES)()
    _check(lib().ba_cuda_comm_unique_id(buf))
    return bytes(buf)


class Problem:
    """One ba_cuda_problem bound to one GPU."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        _check(lib().ba_cuda_create(C.byref(self._h), C.c_int(device)))
        self.model = None
        self.n_obs = 0

    def close(self):
        if self._h:
            lib().ba_cuda_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def comm_init(self, rank, world_size, unique_id):
        buf = (C.c_uint8 * UNIQUE_ID_BYTES).from_buffer_copy(unique_id)
        _check(lib().ba_cuda_comm_init(self._h, C.c_int(rank), C.c_int(world_size), buf))

    def set_model_a(self, n_cam, n_pt, cam_idx, pt_idx, obs_xy, intr):
        cam_idx = np.ascontiguousarray(cam_idx, np.int32); pt_idx = np.ascontiguousarray(pt_idx, np.int32)
        obs_xy = np.ascontiguousarray(obs_xy, np.float64); intr = np.ascontiguousarray(intr, np.float64)
        if intr.size == 4 * n_cam:
            stride = 4
        elif intr.size == 4:
            stride = 0
        else:
            raise ValueError("intr must hold 4 or 4*n_cam doubles")
        _check(lib().ba_cuda_set_model_a(self._h, C.c_int32(n_cam), C.c_int64(n_pt), C.c_int64(cam_idx.shape[0]),
                                         cam_idx.ctypes, pt_idx.ctypes, obs_xy.ctypes, intr.ctypes, C.c_int32(stride)))
        self.model, self.n_obs = "A", int(cam_idx.shape[0])

    def set_model_b(self, n_cam, n_time, n_marker, time_idx, cam_idx, marker_idx, obs8, intr4, marker_side, fix_marker0):
        ti = np.ascontiguousarray(time_idx, np.int32); ci = np.ascontiguousarray(cam_idx, np.int32)
        mi = np.ascontiguousarray(marker_idx, np.int32); ob = np.ascontiguousarray(obs8, np.float64)
        K = np.ascontiguousarray(intr4, np.float64)
        _check(lib().ba_cuda_set_model_b(self._h, C.c_int32(n_cam), C.c_int32(n_time), C.c_int32(n_marker), C.c_int64(ti.shape[0]),
                                         ti.ctypes, ci.ctypes, mi.ctypes, ob.ctypes, K.ctypes, C.c_double(marker_side),
                                         C.c_int32(1), C.c_int32(int(fix_marker0))))
        self.model, self.n_obs = "B", int(ti.shape[0])
        self.n_cam, self.n_time, self.n_marker = n_cam, n_time, n_marker

    def num_parameters(self):
        return int(lib().ba_cuda_num_parameters(self._h))

    def set_parameters(self, params):
        x = np.ascontiguousarray(params, np.float64)
        _check(lib().ba_cuda_set_parameters(self._h, x.ctypes, C.c_int64(x.shape[0])))

    def get_parameters(self, out=None):
        """`out`: an optional float64 array of num_parameters() to receive the result (e.g. pinned memory)."""
        x = np.empty(self.num_parameters(), np.float64) if out is None else out
        assert x.dtype == np.float64 and x.flags.c_contiguous and x.size == self.num_parameters()
        _check(lib().ba_cuda_get_parameters(self._h, x.ctypes, C.c_int64(x.size)))
        return x

    def save_parameters(self):
        _check(lib().ba_cuda_save_parameters(self._h))

    def restore_parameters(self):
        _check(lib().ba_cuda_restore_parameters(self._h))

    def solve(self, options=None):
        opts = options or default_options()
        s = Summary()
        _check(lib().ba_cuda_solve(self._h, C.byref(opts), C.byref(s)))
        n = lib().ba_cuda_get_iterations(self._h, None, C.c_int(0))
        rows = (Iteration * max(n, 1))()
        lib().ba_cuda_get_iterations(self._h, rows, C.c_int(n))
        return s, [rows[i].as_dict() for i in range(n)]

    def solve_batch(self, params, observations=None, options=None, rows_cap=None):
        """k independent solves of this problem's structure in one launch (ba_cuda_solve_batch, include/ba_cuda.h).

        params: [k, n_params] starts.  observations: None (the model's own) or [k, n_obs, 2] (Model A) / [k, n_mobs, 8]
        (Model B) in the order given to set_model_*.  rows_cap: progress rows kept per instance (None: all of them,
        options.max_num_iterations + 1; 0: none).  Returns (solutions [k, n_params], k summaries, k row lists), the summaries
        and rows as `solve` returns them."""
        opts = options or default_options()
        x = np.array(params, dtype=np.float64, order="C", copy=True)   # the library writes the solutions into it
        obs = None
        if self.model is not None:   # without a model the library refuses the call (BA_ERR_STATE)
            if x.ndim != 2 or x.shape[1] != self.num_parameters():
                raise ValueError("params must have shape [k, %d], got %s" % (self.num_parameters(), x.shape))
            if observations is not None:
                obs = np.ascontiguousarray(observations, np.float64)
                width = 2 if self.model == "A" else 8
                if obs.shape != (x.shape[0], self.n_obs, width):
                    raise ValueError("observations must have shape [%d, %d, %d], got %s" % (x.shape[0], self.n_obs, width, obs.shape))
        k = x.shape[0] if x.ndim == 2 else 1
        if rows_cap is None:
            rows_cap = max(1, int(opts.max_num_iterations) + 1)
        summaries = (Summary * max(k, 1))()
        rows = (Iteration * (k * rows_cap))() if rows_cap > 0 and k > 0 else None
        _check(lib().ba_cuda_solve_batch(self._h, C.byref(opts), C.c_int32(k), x.ctypes.data_as(C.c_void_p),
                                         None if obs is None else obs.ctypes.data_as(C.c_void_p), summaries,
                                         rows, C.c_int32(rows_cap)))
        out_rows = []
        for i in range(k):
            n = min(summaries[i].num_iterations, rows_cap) if rows is not None else 0
            out_rows.append([rows[i * rows_cap + r].as_dict() for r in range(n)])
        return x, [summaries[i] for i in range(k)], out_rows

    def _rows(self):
        n = lib().ba_cuda_get_iterations(self._h, None, C.c_int(0))
        rows = (Iteration * max(n, 1))()
        lib().ba_cuda_get_iterations(self._h, rows, C.c_int(n))
        return [rows[i].as_dict() for i in range(n)]

    def solve_begin(self, options=None):
        opts = options or default_options()
        _check(lib().ba_cuda_solve_begin(self._h, C.byref(opts)))

    def solve_iterate(self, max_new_iterations):
        fin = C.c_int32(0)
        _check(lib().ba_cuda_solve_iterate(self._h, C.c_int32(max_new_iterations), C.byref(fin)))
        return bool(fin.value)

    def solve_end(self):
        s = Summary()
        _check(lib().ba_cuda_solve_end(self._h, C.byref(s)))
        return s, self._rows()

    def set_stream(self, cuda_stream_handle):
        _check(lib().ba_cuda_set_stream(self._h, C.c_void_p(cuda_stream_handle)))

    def kernel_stats(self):
        n = lib().ba_cuda_get_kernel_stats(self._h, None, C.c_int(0))
        buf = (KernelStat * max(n, 1))()
        lib().ba_cuda_get_kernel_stats(self._h, buf, C.c_int(n))
        return [buf[i].as_dict() for i in range(n)]

    def num_launches(self):
        return int(lib().ba_cuda_num_launches(self._h))

    def reset_stats(self):
        lib().ba_cuda_reset_stats(self._h)

    def eval(self, want_residuals=True, want_jac=True):
        rd, jw = (2, 18) if self.model == "A" else (8, 144)
        cost = C.c_double(0)
        res = np.zeros((self.n_obs, rd)) if want_residuals else None
        jac = np.zeros((self.n_obs, jw)) if want_jac else None
        _check(lib().ba_cuda_eval(self._h, C.byref(cost), None if res is None else res.ctypes.data_as(C.c_void_p),
                                  None if jac is None else jac.ctypes.data_as(C.c_void_p)))
        return cost.value, res, jac

    def covariance(self, options=None, min_pivot_ratio=0.0):
        """ceres::Covariance of the free parameters at the current parameters (Model B; include/ba_cuda.h):
        (cov_kept [6(C+M), 6(C+M)] in parameter order [cameras | markers], cov_frames [T, 6, 6], smallest_pivot_ratio).
        A rank-deficient problem raises BAError with code abi.ERR_RANK_DEFICIENT and the ratio as `smallest_pivot_ratio`."""
        kept = frames = None   # no Model B: the library refuses the call (BA_ERR_STATE / BA_ERR_UNSUPPORTED) and writes nothing
        if self.model == "B":
            nk = 6 * (self.n_cam + self.n_marker)
            kept = np.zeros((nk, nk)); frames = np.zeros((self.n_time, 6, 6))
        ratio = C.c_double(0.0)
        rc = lib().ba_cuda_covariance(self._h, None if options is None else C.byref(options), C.c_double(min_pivot_ratio),
                                      None if kept is None else kept.ctypes.data_as(C.c_void_p),
                                      None if frames is None else frames.ctypes.data_as(C.c_void_p), C.byref(ratio))
        if rc != 0:
            err = _error(rc)
            err.smallest_pivot_ratio = ratio.value
            raise err
        return kept, frames, ratio.value

    def last_kernel_ms(self):
        return float(lib().ba_cuda_last_kernel_ms(self._h))

    def reprojection_error(self):
        err = C.c_double(0); rms = C.c_double(0)
        _check(lib().ba_cuda_reprojection_error(self._h, C.byref(err), C.byref(rms)))
        return err.value, rms.value

    def project_points_error(self, xyz, cam_of_point, rvec_tvec6, intr4, image_xy, want_reprojected=True):
        xyz = np.ascontiguousarray(xyz, np.float64); cam = np.ascontiguousarray(cam_of_point, np.int32)
        rt = np.ascontiguousarray(rvec_tvec6, np.float64).reshape(-1, 6); K = np.ascontiguousarray(intr4, np.float64)
        img = np.ascontiguousarray(image_xy, np.float32)
        n = xyz.shape[0]
        err = C.c_double(0); rms = C.c_double(0)
        rep = np.zeros((n, 2)) if want_reprojected else None
        _check(lib().ba_cuda_project_points_error(self._h, C.c_int64(n), xyz.ctypes, cam.ctypes, C.c_int32(rt.shape[0]), rt.ctypes,
                                                  K.ctypes, img.ctypes, C.byref(err), C.byref(rms),
                                                  None if rep is None else rep.ctypes.data_as(C.c_void_p)))
        return err.value, rms.value, rep

    def marker_corners(self, rvec_tvec6, marker_side):
        """Correspondencer::GetCornersInCameraWorld for n poses -> [n, 4, 3] (top left, top right, bottom right, bottom left)."""
        rt = np.ascontiguousarray(rvec_tvec6, np.float64).reshape(-1, 6)
        out = np.zeros((rt.shape[0], 4, 3))
        _check(lib().ba_cuda_marker_corners(self._h, C.c_int64(rt.shape[0]), rt.ctypes, C.c_double(marker_side), out.ctypes))
        return out

    def compose_poses(self, a6, b6, invert_b=False):
        """out = a o b, or a o b^-1 (rvec | tvec rows, cv::Rodrigues conventions)."""
        a = np.ascontiguousarray(a6, np.float64).reshape(-1, 6); b = np.ascontiguousarray(b6, np.float64).reshape(-1, 6)
        out = np.zeros_like(a)
        _check(lib().ba_cuda_compose_poses(self._h, C.c_int64(a.shape[0]), a.ctypes, b.ctypes, C.c_int32(1 if invert_b else 0), out.ctypes))
        return out

    def model_b_outputs(self):
        rot = np.zeros((self.n_cam, 9)); inv = np.zeros((self.n_cam, 12)); corners = np.zeros((self.n_obs * 4, 3))
        _check(lib().ba_cuda_model_b_outputs(self._h, rot.ctypes, inv.ctypes, corners.ctypes))
        return rot.reshape(-1, 3, 3), inv.reshape(-1, 3, 4), corners
