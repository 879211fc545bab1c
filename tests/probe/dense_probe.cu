// dense_probe.cu -- test-only entry points that launch the dense reduced-camera-system solvers of csrc/ exactly as the
// library does, on caller-provided device buffers (tests/test_dense_solvers.py).  Not part of libba_cuda.so.
//
//   S      n x n row-major, only its lower triangle and diagonal are read; k_chol_blocked overwrites that part with L
//   rhs    n;  y  n (output);  status  one int the solvers OR their bits into (2: pivot not positive, 4: y not finite)
// Every entry point returns a BA_* code; the launches are asynchronous on `stream`.
#include "ba_dense.cuh"
#include "ba_dense_blocked.cuh"
#include "ba_rig.cuh"

using namespace ba;

namespace {
CholBlockedWork* g_blocked = nullptr;   // one workspace across calls, as a ba_cuda_problem keeps it
}

extern "C" {

// k_ldlt_small, with the shared-memory opt-in dense_solve (ba_cuda.cu) sets
int probe_ldlt_small(int n, const double* S, const double* rhs, double* y, int* status, cudaStream_t stream) {
  if (n < 1 || n > RIG_MAX_N) return fail(BA_ERR_UNSUPPORTED, "k_ldlt_small takes 1 <= n <= %d, not %d", RIG_MAX_N, n);
  const size_t smem = rig_smem_bytes(n);
  if (smem > 48 * 1024) BA_CUDA_TRY(cudaFuncSetAttribute(k_ldlt_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rig_smem_bytes(RIG_MAX_N)));
  k_ldlt_small<<<1, RIG_THREADS, smem, stream>>>(n, S, rhs, y, status);
  BA_CUDA_TRY(cudaGetLastError());
  return BA_OK;
}

int probe_chol_solve(int n, const double* S, const double* rhs, double* y, int* status, cudaStream_t stream) {
  return launch_chol_solve(n, S, rhs, y, status, stream);
}

int probe_chol_blocked(int n, double* S, const double* rhs, double* y, int* status, cudaStream_t stream) {
  int device = 0;
  BA_CUDA_TRY(cudaGetDevice(&device));
  if (!g_blocked) g_blocked = new CholBlockedWork();
  return launch_chol_blocked(*g_blocked, n, S, rhs, y, status, device, stream);
}

// drops the workspace: the next probe_chol_blocked starts from a fresh one
void probe_blocked_reset() {
  delete g_blocked;
  g_blocked = nullptr;
}

// the workspace's `bad` flag as the last k_chol_blocked left it (-1 without a workspace); synchronises the device
int probe_blocked_bad_flag() {
  if (!g_blocked || !g_blocked->bad.p) return -1;
  int v = -1;
  if (cudaMemcpy(&v, g_blocked->bad.p, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return v;
}

// doubles the workspace's solve buffer holds (0 without a workspace): launch_chol_blocked must have made it >= n before the launch
size_t probe_blocked_work_capacity() { return g_blocked ? g_blocked->work.n : 0; }

const char* probe_last_error() { return err_buf(); }

}  // extern "C"
