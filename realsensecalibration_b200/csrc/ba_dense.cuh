// ba_dense.cuh -- K3a: dense Cholesky solve of a rig-sized reduced camera system in ONE CTA.
// Replaces Ceres' DenseSchurComplementSolver -> Eigen LLT (options.linear_solver_type = DENSE_SCHUR,
// bundle_adjustment_manager.cpp:91).  The whole matrix lives in shared memory, so n <= 160
// (n^2 * 8 B <= 205 KB of the 227 KB a CTA may use on sm_100a); larger systems go to ba_dense_blocked.cuh.
// Only the lower triangle and the diagonal of S are read.
#pragma once
#include "ba_util.cuh"

namespace ba {

constexpr int CHOL_SMEM_MAX_N = 160;

// status |= 2 (and y = 0) if a pivot is not positive, |= 4 if the solution is not finite.
__global__ void __launch_bounds__(1024)
k_chol_solve(int n, const double* __restrict__ S, const double* __restrict__ rhs, double* __restrict__ y, int* status) {
  extern __shared__ double sh[];
  double* A = sh;
  double* col = sh + (size_t)n * n;
  double* bv = col + n;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  for (int i = tid; i < n * n; i += nt) A[i] = S[i];
  for (int i = tid; i < n; i += nt) bv[i] = rhs[i];
  bool bad = false;
  for (int j = 0; j < n; ++j) {
    __syncthreads();
    const double d = A[(size_t)j * n + j];
    if (!(d > 0.0) || !isfinite(d)) { bad = true; break; }  // uniform across the CTA
    const double l = sqrt(d), inv = 1.0 / l;
    for (int i = j + tid; i < n; i += nt) {
      const double v = (i == j) ? l : A[(size_t)i * n + j] * inv;
      col[i] = v;
      if (i != j) A[(size_t)i * n + j] = v;   // the diagonal is still being read as d by slower warps (racecheck, round 2)
    }
    __syncthreads();
    if (tid == 0) A[(size_t)j * n + j] = l;
    for (int i = j + 1 + warp; i < n; i += nw) {
      const double ci = col[i];
      double* row = A + (size_t)i * n;
      for (int k = j + 1 + lane; k <= i; k += 32) row[k] -= ci * col[k];
    }
  }
  __syncthreads();
  if (bad) {
    if (tid == 0) atomicOr(status, 2);
    for (int i = tid; i < n; i += nt) y[i] = 0.0;
    return;
  }
  // forward substitution L t = b
  for (int j = 0; j < n; ++j) {
    __syncthreads();
    const double yj = bv[j] / A[(size_t)j * n + j];
    __syncthreads();
    if (tid == 0) bv[j] = yj;
    for (int i = j + 1 + tid; i < n; i += nt) bv[i] -= A[(size_t)i * n + j] * yj;
  }
  // backward substitution L^T y = t
  for (int j = n - 1; j >= 0; --j) {
    __syncthreads();
    const double yj = bv[j] / A[(size_t)j * n + j];
    __syncthreads();
    if (tid == 0) bv[j] = yj;
    for (int i = tid; i < j; i += nt) bv[i] -= A[(size_t)j * n + i] * yj;
  }
  __syncthreads();
  for (int i = tid; i < n; i += nt) {
    const double v = bv[i];
    y[i] = v;
    if (!isfinite(v)) atomicOr(status, 4);
  }
}

inline int launch_chol_solve(int n, const double* S, const double* rhs, double* y, int* status, cudaStream_t st) {
  if (n > CHOL_SMEM_MAX_N) return fail(BA_ERR_UNSUPPORTED, "dense RCS of dimension %d is too large for the single-CTA solver", n);
  const size_t smem = ((size_t)n * n + 2 * (size_t)n) * sizeof(double);
  // the opt-in limit belongs to the device the stream runs on; setting it costs microseconds, a process-wide
  // "done" flag would leave a second GPU without it
  if (smem > 48 * 1024) BA_CUDA_TRY(cudaFuncSetAttribute(k_chol_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  k_chol_solve<<<1, 1024, smem, st>>>(n, S, rhs, y, status);
  BA_CUDA_TRY(cudaGetLastError());
  return BA_OK;
}

}  // namespace ba
