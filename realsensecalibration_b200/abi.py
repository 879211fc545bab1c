"""ctypes mirror of include/ba_cuda.h (PODs and enums only)."""
import ctypes as C

BA_OK = 0
RCS_AUTO, RCS_DENSE_CHOLESKY, RCS_PCG = 0, 1, 2
CONVERGENCE, NO_CONVERGENCE, FAILURE = 0, 1, 2
(REASON_NONE, REASON_GRADIENT_TOLERANCE, REASON_PARAMETER_TOLERANCE, REASON_FUNCTION_TOLERANCE,
 REASON_MIN_TRUST_REGION_RADIUS, REASON_MAX_ITERATIONS, REASON_TOO_MANY_INVALID_STEPS,
 REASON_INITIAL_EVALUATION_FAILED) = range(8)
UNIQUE_ID_BYTES = 128
PATH_GENERIC, PATH_FUSED_TILES, PATH_FUSED_STRIPS, PATH_RIG = 0, 1, 2, 3
LOSS_NONE, LOSS_HUBER, LOSS_CAUCHY = 0, 1, 2
(ERR_INVALID_ARGUMENT, ERR_CUDA, ERR_STATE, ERR_NCCL, ERR_OUT_OF_MEMORY, ERR_NO_DEVICE, ERR_UNSUPPORTED,
 ERR_RANK_DEFICIENT) = range(-1, -9, -1)


class Options(C.Structure):
    _fields_ = [
        ("max_num_iterations", C.c_int32),
        ("max_num_consecutive_invalid_steps", C.c_int32),
        ("jacobi_scaling", C.c_int32),
        ("rcs_solver", C.c_int32),
        ("pcg_max_iterations", C.c_int32),
        ("pcg_min_iterations", C.c_int32),
        ("pcg_residual_reset_period", C.c_int32),
        ("minimizer_progress_to_stdout", C.c_int32),
        ("profile_kernels", C.c_int32),
        ("force_generic_path", C.c_int32),
        ("initial_trust_region_radius", C.c_double),
        ("max_trust_region_radius", C.c_double),
        ("min_trust_region_radius", C.c_double),
        ("min_relative_decrease", C.c_double),
        ("min_lm_diagonal", C.c_double),
        ("max_lm_diagonal", C.c_double),
        ("function_tolerance", C.c_double),
        ("gradient_tolerance", C.c_double),
        ("parameter_tolerance", C.c_double),
        ("pcg_eta", C.c_double),
        ("pcg_r_tolerance", C.c_double),
        ("loss_function", C.c_int32),
        ("reserved_", C.c_int32),
        ("loss_scale", C.c_double),
    ]


class Iteration(C.Structure):
    _fields_ = [
        ("iteration", C.c_int32),
        ("step_is_valid", C.c_int32),
        ("step_is_successful", C.c_int32),
        ("linear_solver_iterations", C.c_int32),
        ("cost", C.c_double),
        ("cost_change", C.c_double),
        ("gradient_max_norm", C.c_double),
        ("gradient_norm", C.c_double),
        ("step_norm", C.c_double),
        ("relative_decrease", C.c_double),
        ("trust_region_radius", C.c_double),
        ("iteration_time_s", C.c_double),
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class KernelStat(C.Structure):
    _fields_ = [
        ("name", C.c_char * 32),
        ("launches", C.c_int64),
        ("total_ms", C.c_double),
        ("algorithmic_bytes_per_launch", C.c_double),
    ]

    def as_dict(self):
        return {"name": self.name.decode(), "launches": int(self.launches), "total_ms": float(self.total_ms),
                "algorithmic_bytes_per_launch": float(self.algorithmic_bytes_per_launch)}


class Summary(C.Structure):
    _fields_ = [
        ("termination_type", C.c_int32),
        ("termination_reason", C.c_int32),
        ("num_iterations", C.c_int32),
        ("num_successful_steps", C.c_int32),
        ("num_unsuccessful_steps", C.c_int32),
        ("rcs_solver_used", C.c_int32),
        ("rcs_dim", C.c_int32),
        ("num_jacobian_evaluations", C.c_int32),
        ("num_cost_evaluations", C.c_int32),
        ("num_linear_solves", C.c_int32),
        ("num_residuals", C.c_int64),
        ("num_free_parameters", C.c_int64),
        ("initial_cost", C.c_double),
        ("final_cost", C.c_double),
        ("total_time_s", C.c_double),
        ("ms_jacobian", C.c_double),
        ("ms_schur", C.c_double),
        ("ms_rcs_solve", C.c_double),
        ("ms_update", C.c_double),
        ("ms_cost", C.c_double),
        ("ms_collective", C.c_double),
        ("path_used", C.c_int32),
        ("reserved_", C.c_int32),
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}
