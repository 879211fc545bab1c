// ba_cov.cuh -- covariance of the free parameters of Model B at the current x (ceres::Covariance, dense, apply_loss_function
// = true): C = (J^T J)^-1, recovered from the undamped Schur complement of the frame poses.
//
// With J Jacobi scaled (J_s = J diag(s)) and split into frame columns E and kept columns F (cameras | markers),
//   U_e = E_e^T E_e = L_e L_e^T         (k_e_chol, per frame)
//   Y_i = L_e^-1 E_e^T F_f(i)          (k_inc_Y, per incidence (frame e, kept block f(i)); stored as Yt)
//   S   = F^T F - sum_e W_e^T U_e^-1 W_e = L L^T   (k_assemble_dense + k_diag_rhs_dense, then k_chol_blocked)
// the kept blocks' covariance is S^-1 and the diagonal block of frame e is
//   C_ee = L_e^-T (I + sum_{k,l} Y_k S^-1[f_k, f_l] Y_l^T) L_e^-1,
// both unscaled by diag(s) on the way out.  The kernels here take it from the Cholesky factor L in the lower triangle of Sd:
//   k_cov_linv      X = L^-1, one CTA per 32 columns: forward substitution by 32-row blocks, the block products on DMMA
//   k_cov_inverse   S^-1 = X^T X on 64 x 64 output tiles (DMMA, as k_chol_blocked's trailing update), one triangle computed
//                   and mirrored (exactly symmetric); the epilogue also writes diag(sf) S^-1 diag(sf) in parameter order
//   k_cov_frames    C_ee, one CTA per frame: the frame's Yt records staged in shared memory, S^-1 read out of L2
// Every sum runs in a fixed order and nothing is accumulated with atomics: two calls give the same bits.
#pragma once
#include "ba_dense_blocked.cuh"
#include "ba_kernels.cuh"

namespace ba {

constexpr int CV_THREADS = 256;
constexpr int CV_NB = 32;   // column block of k_cov_linv
constexpr int CV_TB = 64;   // output tile of k_cov_inverse
constexpr int CV_LD = 36;   // shared-memory row stride of a 32-wide tile (doubles), conflict-free DMMA fragment loads

__device__ __forceinline__ bool f_active(const int64_t* __restrict__ f_act_ptr, int64_t f) { return f_act_ptr[f + 1] > f_act_ptr[f]; }

// Blocks no observation references would make the undamped system singular: unit diagonals in E^T E of unobserved frames and
// in F^T F of kept blocks that are not parameters (camera 0, marker 0 under fix_marker0).  Their output is zero.
template <int DE>
__global__ void k_cov_unit_unused(int64_t ne, const int64_t* __restrict__ e_ptr, double* __restrict__ ME, int64_t nf,
                                  const int64_t* __restrict__ f_act_ptr, double* __restrict__ HG) {
  constexpr int NVE = DE * (DE + 1) / 2 + DE;
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t < ne) {
    if (e_ptr[t + 1] == e_ptr[t])
      for (int a = 0; a < DE; ++a) ME[t * NVE + a * DE - a * (a - 1) / 2] = 1.0;
  } else if (t < ne + nf) {
    const int64_t f = t - ne;
    if (!f_active(f_act_ptr, f))
      for (int a = 0; a < 6; ++a) HG[f * NV_F + sym_idx6(a, a)] = 1.0;
  }
}

__global__ void k_cov_save_diag(int n, const double* __restrict__ S, double* __restrict__ diag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) diag[i] = S[(size_t)i * n + i];
}

// min_k L_kk^2 / max_k S_kk over the scalar rows of parameter blocks (L_kk^2 is the k-th pivot of L D L^T); 1 when there is none.
// Launched <<<1, 1024>>>.
__global__ void k_cov_pivot_ratio(int n, const double* __restrict__ L, const double* __restrict__ diag,
                                  const int64_t* __restrict__ f_act_ptr, double* __restrict__ out) {
  __shared__ double sm[32];
  double mn = -INFINITY, mx = 0.0;   // mn holds -min
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    if (f_active(f_act_ptr, i / 6)) {
      const double l = L[(size_t)i * n + i];
      mn = fmax(mn, -(l * l));
      mx = fmax(mx, diag[i]);
    }
  mn = block_max(mn, sm);
  __syncthreads();
  if (threadIdx.x == 0) sm[31] = mn;
  __syncthreads();
  mn = -sm[31];
  mx = block_max(mx, sm);
  if (threadIdx.x == 0) *out = mn == INFINITY ? 1.0 : mn / mx;
}

// X = L^-1 (lower triangle; rows above a column's diagonal block are left as the caller's zeros).  CTA j owns columns
// [32 j, 32 j + 32) and walks the row blocks I >= j:  X_Ij = L_II^-1 (delta_Ij - sum_{j <= K < I} L_IK X_Kj).
// The block products run on DMMA (warp w: row tile w & 3, column tiles 2 (w >> 2) and 2 (w >> 2) + 1, K and k in order);
// the 32 x 32 triangular solve by warps (4 columns each, lane = row).  X_Kj is read back from global memory (L2), where this
// CTA wrote it at step K.
__global__ void __launch_bounds__(CV_THREADS)
k_cov_linv(int n, const double* __restrict__ L, double* __restrict__ X) {
  __shared__ __align__(16) double La[CV_NB * CV_LD];       // L_IK, row i, column k
  __shared__ __align__(16) double Xb[CV_NB * CV_LD];       // X_Kj transposed: column c, row k
  __shared__ double Ld[CV_NB * (CV_NB + 1)];                // L_II
  __shared__ double T[CV_NB * (CV_NB + 1)];                 // right-hand side of the block row
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nblk = (n + CV_NB - 1) / CV_NB, j = blockIdx.x, c0 = CV_NB * j, cb = min(CV_NB, n - c0);
  const size_t ld = (size_t)n;
  const int wr = warp & 3, wc = 2 * (warp >> 2), fr = lane >> 2, fc = lane & 3;
  for (int I = j; I < nblk; ++I) {
    const int r0 = CV_NB * I, rb = min(CV_NB, n - r0);
    double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
    for (int K = j; K < I; ++K) {   // K < I <= nblk - 1: block K is a full 32 rows / columns
      const int k0 = CV_NB * K;
      __syncthreads();
      for (int i = tid; i < CV_NB * CV_NB; i += CV_THREADS) {
        const int r = i / CV_NB, c = i % CV_NB;
        La[r * CV_LD + c] = r < rb ? L[(r0 + r) * ld + k0 + c] : 0.0;
        Xb[c * CV_LD + r] = c < cb ? X[(k0 + r) * ld + c0 + c] : 0.0;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < CV_NB / 4; ++kk) {
        const double a = La[(8 * wr + fr) * CV_LD + 4 * kk + fc];
#pragma unroll
        for (int t = 0; t < 2; ++t) dmma_m8n8k4(acc[t][0], acc[t][1], a, Xb[(8 * (wc + t) + fr) * CV_LD + 4 * kk + fc]);
      }
    }
    __syncthreads();
#pragma unroll
    for (int t = 0; t < 2; ++t)
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int row = 8 * wr + fr, col = 8 * (wc + t) + 2 * fc + q;
        T[row * (CV_NB + 1) + col] = (r0 + row == c0 + col ? 1.0 : 0.0) - acc[t][q];
      }
    for (int i = tid; i < CV_NB * CV_NB; i += CV_THREADS) {
      const int r = i / CV_NB, c = i % CV_NB;
      Ld[r * (CV_NB + 1) + c] = (r < rb && c <= r) ? L[(r0 + r) * ld + r0 + c] : 0.0;
    }
    __syncthreads();
    double x[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) x[q] = T[lane * (CV_NB + 1) + 4 * warp + q];
    for (int jr = 0; jr < rb; ++jr) {   // uniform trip count: every lane takes part in the shuffles
      const double djj = Ld[jr * (CV_NB + 1) + jr], ljr = Ld[lane * (CV_NB + 1) + jr];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const double xj = __shfl_sync(0xffffffffu, x[q], jr) / djj;
        if (lane == jr) x[q] = xj;
        else if (lane > jr) x[q] -= ljr * xj;
      }
    }
    if (lane < rb)
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (4 * warp + q < cb) X[(r0 + lane) * ld + c0 + 4 * warp + q] = x[q];
  }
}

// S^-1 = X^T X on the 64 x 64 tiles (I, J), I >= J, of the lower triangle; the sum over rows r >= 64 I (X[r, a] = 0 for r < a)
// in chunks of 32, each chunk staged transposed and multiplied on DMMA as in k_chol_blocked.  Every element is computed once
// and written to both triangles of Sig; C = diag(sf) Sig diag(sf) with the rows and columns of blocks that are not
// parameters set to 0 (C is in parameter order [cameras | markers] because the kept blocks are numbered that way).
__global__ void __launch_bounds__(CV_THREADS)
k_cov_inverse(int n, const double* __restrict__ X, const double* __restrict__ sf, const int64_t* __restrict__ f_act_ptr,
              double* __restrict__ Sig, double* __restrict__ C) {
  __shared__ __align__(16) double Pa[CV_TB * CV_LD];
  __shared__ __align__(16) double Pb[CV_TB * CV_LD];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t ld = (size_t)n;
  const int t = blockIdx.x;
  int I = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
  while ((I + 1) * (I + 2) / 2 <= t) ++I;
  while (I * (I + 1) / 2 > t) --I;
  const int J = t - I * (I + 1) / 2;
  const int ri = CV_TB * I, rj = CV_TB * J;
  double acc[8][2];
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[c][0] = acc[c][1] = 0.0;
  const int fr = lane >> 2, fc = lane & 3;
  for (int r0 = ri; r0 < n; r0 += CV_NB) {
    __syncthreads();
    for (int i = tid; i < CV_TB * CV_NB; i += CV_THREADS) {
      const int a = i % CV_TB, kk = i / CV_TB;   // consecutive threads read consecutive columns of a row of X
      const bool rok = r0 + kk < n;
      Pa[a * CV_LD + kk] = (rok && ri + a < n) ? X[(r0 + kk) * ld + ri + a] : 0.0;
      Pb[a * CV_LD + kk] = (rok && rj + a < n) ? X[(r0 + kk) * ld + rj + a] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < CV_NB / 4; ++kk) {
      const double a = Pa[(8 * warp + fr) * CV_LD + 4 * kk + fc];
#pragma unroll
      for (int c = 0; c < 8; ++c) dmma_m8n8k4(acc[c][0], acc[c][1], a, Pb[(8 * c + fr) * CV_LD + 4 * kk + fc]);
    }
  }
  const int row = ri + 8 * warp + fr;
  if (row >= n) return;
  const bool row_act = f_active(f_act_ptr, row / 6);
  const double srow = sf[row];
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int col = rj + 8 * c + 2 * fc + q;
      if (col >= n || col > row) continue;
      const double v = acc[c][q];
      const double cv = (row_act && f_active(f_act_ptr, col / 6)) ? srow * v * sf[col] : 0.0;
      Sig[row * ld + col] = v; Sig[col * ld + row] = v;
      C[row * ld + col] = cv; C[col * ld + row] = cv;
    }
}

inline size_t cov_frames_smem(int DE, int64_t nf) { return ((size_t)2 * DE * 6 * nf + DE * DE) * sizeof(double) + (size_t)6 * nf * sizeof(int); }

// C_ee of every frame, one CTA per frame e with incidences i0 .. i0 + m (kept blocks f_0 .. f_{m-1}), w = 6 m:
//   Yc[d][6 l + b] = Y_l[d][b]                          (shared memory)
//   T[6 k + a][d]  = sum_{l,b} Sig[6 f_k + a][6 f_l + b] Yc[d][6 l + b]   (warp per row of T, lanes along the row of Sig)
//   M = Yc T (lower triangle, mirrored), C_ee = diag(se) L_e^-T (I + M) L_e^-1 diag(se) (lower triangle, mirrored).
// Frames without observations get 0.  Dynamic shared memory: cov_frames_smem(DE, nf).
template <int DE>
__global__ void __launch_bounds__(CV_THREADS)
k_cov_frames(int64_t ne, const int64_t* __restrict__ e_ptr, const int64_t* __restrict__ einc_ptr, const int32_t* __restrict__ inc_f,
             const double* __restrict__ Yt, const double* __restrict__ Lb, const double* __restrict__ se, const double* __restrict__ Sig,
             int n, double* __restrict__ out) {
  extern __shared__ __align__(16) double cov_sm[];
  const int64_t e = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double* o = out + e * DE * DE;
  if (e_ptr[e + 1] == e_ptr[e]) {
    if (tid < DE * DE) o[tid] = 0.0;
    return;
  }
  const int64_t i0 = einc_ptr[e];
  const int m = (int)(einc_ptr[e + 1] - i0), w = 6 * m;
  double* Yc = cov_sm;
  double* T = Yc + DE * w;
  double* M = T + DE * w;
  int* col = reinterpret_cast<int*>(M + DE * DE);
  for (int t = tid; t < DE * w; t += CV_THREADS) {
    const int d = t / w, c = t % w;
    Yc[t] = Yt[(i0 + c / 6) * DE * 6 + d * 6 + c % 6];
  }
  for (int c = tid; c < w; c += CV_THREADS) col[c] = 6 * inc_f[i0 + c / 6] + c % 6;
  __syncthreads();
  for (int r = warp; r < w; r += CV_THREADS / 32) {
    const double* srow = Sig + (size_t)col[r] * n;
    double acc[DE];
#pragma unroll
    for (int d = 0; d < DE; ++d) acc[d] = 0.0;
    for (int c = lane; c < w; c += 32) {
      const double g = srow[col[c]];
#pragma unroll
      for (int d = 0; d < DE; ++d) acc[d] = fma(g, Yc[d * w + c], acc[d]);
    }
    group_sum_store<DE, 32>(acc, lane, T + r * DE, true);
  }
  __syncthreads();
  for (int q = warp; q < DE * (DE + 1) / 2; q += CV_THREADS / 32) {
    int d1 = 0;
    while ((d1 + 1) * (d1 + 2) / 2 <= q) ++d1;
    const int d2 = q - d1 * (d1 + 1) / 2;
    double s = 0.0;
    for (int r = lane; r < w; r += 32) s = fma(Yc[d1 * w + r], T[r * DE + d2], s);
    s = warp_sum(s);
    if (lane == 0) { M[d1 * DE + d2] = s; M[d2 * DE + d1] = s; }
  }
  __syncthreads();
  if (tid != 0) return;
  double L[DE * DE], A[DE * DE], x[DE];
#pragma unroll
  for (int k = 0; k < DE * DE; ++k) { L[k] = Lb[e * DE * DE + k]; A[k] = (k % (DE + 1) == 0 ? 1.0 : 0.0) + M[k]; }
#pragma unroll
  for (int c = 0; c < DE; ++c) {   // A <- L^-T A, by columns
#pragma unroll
    for (int r = 0; r < DE; ++r) x[r] = A[r * DE + c];
    bwd_small<DE>(L, x);
#pragma unroll
    for (int r = 0; r < DE; ++r) A[r * DE + c] = x[r];
  }
#pragma unroll
  for (int r = 0; r < DE; ++r) {   // A <- A L^-1, by rows: (A L^-1)[r, :] = L^-T A[r, :]^T
#pragma unroll
    for (int c = 0; c < DE; ++c) x[c] = A[r * DE + c];
    bwd_small<DE>(L, x);
#pragma unroll
    for (int c = 0; c < DE; ++c) A[r * DE + c] = x[c];
  }
#pragma unroll
  for (int a = 0; a < DE; ++a)
#pragma unroll
    for (int b = 0; b <= a; ++b) {
      const double v = se[e * DE + a] * A[a * DE + b] * se[e * DE + b];
      o[a * DE + b] = v; o[b * DE + a] = v;
    }
}

}  // namespace ba
