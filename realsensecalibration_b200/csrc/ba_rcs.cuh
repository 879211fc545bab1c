// ba_rcs.cuh -- K3b: the reduced camera system as a block-sparse symmetric matrix and its
// block-Jacobi preconditioned conjugate-gradient solve in ONE persistent cooperative kernel.
//
// Replaces, for BAL-scale camera counts, what the reference gets from
// options.linear_solver_type (bundle_adjustment_manager.cpp:91) -> Ceres' Schur complement solvers.
// The CG recurrence, its x0 = 0 start, the Q-based stopping rule (q_tolerance = eta), the
// disabled r_tolerance and the residual reset every 10 iterations restate Ceres 1.14's
// ConjugateGradientsSolver as LevenbergMarquardtStrategy drives it (SURVEY.md 5.9, oracle
// solve_schur_pcg); the preconditioner is the inverse of the 6x6 diagonal blocks of S
// (SCHUR_JACOBI).
//
// Storage: only the destination blocks d = (fa <= fb) that some eliminated block couples
// are stored, 36 doubles each, row-major with rows = fa (HBM: ndest * 288 B; cfg4 ~ 6 MB and
// cfg5 ~ 90 MB, i.e. L2 resident).  A static row index lists, for every camera row f, the
// stored blocks of both triangles as (dest << 1 | transposed).  One warp owns one block row;
// every reduction is a fixed tree over a fixed ownership map, so the solve is bitwise
// reproducible.  Two grid-wide barriers per CG iteration.
#pragma once
#include <cooperative_groups.h>

#include "ba_structure.cuh"

namespace ba {
namespace cg = cooperative_groups;

struct RcsPattern {
  int nd = 0;         // stored blocks (upper triangle incl. every diagonal block)
  int64_t nf = 0;
  int64_t nnzb = 0;   // row-index entries (both triangles)
  DVec<uint64_t> keys;      // fa * nf + fb ascending
  DVec<int32_t> fa, fb, diag;
  DVec<int64_t> row_ptr;
  DVec<int32_t> row_ent, row_col;
  DVec<int32_t> l2g;        // this rank's destination block -> stored block (identity on one GPU)
};

__global__ void k_row_keys(const int32_t* __restrict__ fa, const int32_t* __restrict__ fb, int nd, int32_t* __restrict__ keys,
                           int32_t* __restrict__ ent, int32_t* __restrict__ col) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= nd) return;
  keys[2 * d] = fa[d]; ent[2 * d] = d << 1; col[2 * d] = fb[d];
  const bool off = fa[d] != fb[d];
  keys[2 * d + 1] = off ? fb[d] : INT32_MAX; ent[2 * d + 1] = (d << 1) | 1; col[2 * d + 1] = fa[d];
}
__global__ void k_map_keys(const uint64_t* __restrict__ local, int nl, const uint64_t* __restrict__ global, int ng, int32_t* __restrict__ l2g) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= nl) return;
  l2g[d] = (int32_t)lower_bound_u64(global, ng, local[d]);
}

// keys: device array of nd ascending unique (fa * nf + fb) with fa <= fb, containing every (f, f).
inline int build_rcs_pattern(RcsPattern& R, const uint64_t* keys, int nd, int64_t nf, cudaStream_t st) {
  R.nd = nd; R.nf = nf;
  BA_TRY(R.keys.alloc(nd));
  BA_CUDA_TRY(cudaMemcpyAsync(R.keys.p, keys, sizeof(uint64_t) * nd, cudaMemcpyDeviceToDevice, st));
  BA_TRY(R.fa.alloc(nd)); BA_TRY(R.fb.alloc(nd)); BA_TRY(R.diag.alloc(nf));
  k_dest_finish<<<grid_for(nd, 256), 256, 0, st>>>(R.keys.p, nd, nf, R.fa.p, R.fb.p, R.diag.p);
  DVec<int32_t> k, e, c, es;
  BA_TRY(k.alloc(2 * (size_t)nd)); BA_TRY(e.alloc(2 * (size_t)nd)); BA_TRY(c.alloc(2 * (size_t)nd));
  k_row_keys<<<grid_for(nd, 256), 256, 0, st>>>(R.fa.p, R.fb.p, nd, k.p, e.p, c.p);
  // two stable sorts by the same key keep (ent, col) aligned
  DVec<int64_t> ptr2;
  BA_TRY(sort_to_csr(k.p, e.p, 2 * (int64_t)nd, nf, R.row_ptr, R.row_ent, st));
  BA_TRY(sort_to_csr(k.p, c.p, 2 * (int64_t)nd, nf, ptr2, R.row_col, st));
  int64_t nnzb = 0;
  BA_CUDA_TRY(cudaMemcpyAsync(&nnzb, R.row_ptr.p + nf, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  R.nnzb = nnzb;
  BA_CUDA_TRY(cudaGetLastError());
  return BA_OK;
}

// Stored block value = Q - P of this rank's destination block (F^T F off-diagonal part minus the eliminated
// blocks' contribution); the diagonal F^T F blocks and the LM diagonal are added after the cross-GPU sum.
__global__ void k_assemble_bsr(int ndest, const int32_t* __restrict__ l2g, const double* __restrict__ P, const double* __restrict__ Q,
                               double* __restrict__ Sb) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= (int64_t)ndest * 36) return;
  const int d = (int)(t / 36), q = (int)(t % 36);
  Sb[(int64_t)l2g[d] * 36 + q] = (Q ? Q[t] : 0.0) - P[t];
}

// diagonal block += F^T F + D_f^2, rhs = F^T r - sum v.  DOFF >= 0: the LM diagonal is taken from diag F^T F at HG[DOFF..]
// (the strip record, whose packed block is F^T (I - U^T U) F); -1: from the packed block itself.
template <int DOFF = -1>
__global__ void k_diag_rhs_bsr(int64_t nf, const int32_t* __restrict__ diag, const double* __restrict__ HG, int hg_stride,
                               const double* __restrict__ vsum, int v_stride, const double* __restrict__ radius_p, double min_diag, double max_diag, double* __restrict__ Sb,
                               double* __restrict__ rhs) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= nf * 6) return;
  const int64_t f = t / 6;
  const int a = (int)(t % 6);
  const double* H = HG + f * hg_stride;
  double* B = Sb + (int64_t)diag[f] * 36;
#pragma unroll
  for (int b = 0; b < 6; ++b) {
    double h = H[a <= b ? sym_idx6(a, b) : sym_idx6(b, a)];
    if (a == b) { const double d = sqrt(fmin(fmax(DOFF < 0 ? h : H[DOFF + a], min_diag), max_diag) / *radius_p); h += d * d; }
    B[a * 6 + b] += h;
  }
  rhs[t] = H[21 + a] - vsum[f * v_stride + a];
}

struct PcgParams {
  int nf;
  const int64_t* row_ptr; const int32_t* row_ent; const int32_t* row_col; const int32_t* diag;
  const double* Sb; const double* b;
  double* x; double* r; double* z; double* p0; double* p1; double* q; double* Minv;
  double* partial;   // 4 * total warps
  int max_it, min_it, reset_period;
  double eta, r_tol;
  int* out_iters; int* status;
};

// sums of n per-warp partials (K arrays at once), identical (bitwise) in every thread of every CTA: strided per-thread
// sums, warp trees, then EVERY warp folds the per-warp values with the same tree -- two barriers per call
template <int K>
__device__ __forceinline__ void pcg_totals(const double* const* partial, int n, double* sm /* K * 32 */, double* out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  double v[K];
#pragma unroll
  for (int k = 0; k < K; ++k) v[k] = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] += __ldcg(partial[k] + i);
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    v[k] = warp_sum(v[k]);
    if (lane == 0) sm[32 * k + warp] = v[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const double x = warp_sum(lane < nw ? sm[32 * k + lane] : 0.0);
    out[k] = __shfl_sync(0xffffffffu, x, 0);
  }
  __syncthreads();
}
__device__ __forceinline__ double pcg_total(const double* partial, int n, double* sm) {
  const double* arr[1] = {partial};
  double out[1];
  pcg_totals<1>(arr, n, sm, out);
  return out[0];
}

// (S v)_f with v = a + beta * b2 (b2 may be null); result valid in every lane
__device__ __forceinline__ void pcg_spmv_row(const PcgParams& P, int f, const double* a, const double* b2, double beta, int lane,
                                             double* acc) {
#pragma unroll
  for (int i = 0; i < 6; ++i) acc[i] = 0.0;
  for (int64_t k = P.row_ptr[f] + lane; k < P.row_ptr[f + 1]; k += 32) {
    const int ent = P.row_ent[k];
    const int g = P.row_col[k];
    double v[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) v[j] = __ldcg(a + 6 * (int64_t)g + j) + (b2 ? beta * __ldcg(b2 + 6 * (int64_t)g + j) : 0.0);
    const double* B = P.Sb + 36 * (int64_t)(ent >> 1);
    double blk[36];
#pragma unroll
    for (int j = 0; j < 18; ++j) { const double2 w = reinterpret_cast<const double2*>(B)[j]; blk[2 * j] = w.x; blk[2 * j + 1] = w.y; }
    if (ent & 1) {
#pragma unroll
      for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = 0; j < 6; ++j) acc[i] += blk[j * 6 + i] * v[j];
    } else {
#pragma unroll
      for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = 0; j < 6; ++j) acc[i] += blk[i * 6 + j] * v[j];
    }
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
  }
}

// K tile sums of a CTA (fixed tree); result valid in thread 0
template <int K>
__device__ __forceinline__ void pcg_block_sums(double* v, double* sm /* K * 32 */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    v[k] = warp_sum(v[k]);
    if (lane == 0) sm[32 * k + warp] = v[k];
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] = warp_sum(lane < nw ? sm[32 * k + lane] : 0.0);
  }
  __syncthreads();
}

// r, z = M^-1 r and the partial sums of one block row, by the six lanes base .. base + 5 of a warp (lane base + c owns
// component c and holds x_c, r_c); every lane of the warp must call (shuffles), `on` says whether this lane has a row
__device__ __forceinline__ void pcg_finish_row(const PcgParams& P, int f, bool on, int base, int c, double xv, double rv,
                                               double& s_q, double& s_rz, double& s_rr) {
  const int64_t o = 6 * (int64_t)f + c;
  const double* Mi = P.Minv + 36 * (int64_t)f + 6 * c;
  double m[6];
#pragma unroll
  for (int j = 0; j < 6; ++j) m[j] = on ? Mi[j] : 0.0;
  double s = 0.0;
#pragma unroll
  for (int j = 0; j < 6; ++j) s += m[j] * __shfl_sync(0xffffffffu, rv, base + j);
  if (on) {
    P.r[o] = rv;
    P.z[o] = s;
    s_q += xv * (P.b[o] + rv);
    s_rr += rv * rv;
    s_rz += rv * s;
  }
}

// One cooperative launch per linear solve.  Block rows are dealt one per WARP for the products with S (lane = stored
// block of the row) and one per THREAD / per six lanes for everything that is local to a row (block-Jacobi factors,
// vector updates), so no phase runs on one lane of a warp; the dot products leave every CTA as one partial each.
__global__ void __launch_bounds__(256, 2) k_pcg(PcgParams P) {
  __shared__ double sm[128];
  cg::grid_group grid = cg::this_grid();
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  const int gw = blockIdx.x * wpb + (threadIdx.x >> 5);
  const int GW = gridDim.x * wpb;
  const int gt = blockIdx.x * blockDim.x + threadIdx.x, GT = gridDim.x * blockDim.x;
  const int NB = gridDim.x;
  double* pa = P.partial; double* pb = pa + NB; double* pc = pb + NB; double* pd = pc + NB;
  const int grp = lane / 6, comp = lane - 6 * grp;   // six lanes per row, five rows per warp (lanes 30, 31 idle)

  // ---- setup: block-Jacobi preconditioner, x = 0, r = b, z = M^-1 r (one thread per block row) ----
  {
    double v[2] = {0.0, 0.0};   // b.b, r.z
    for (int f = gt; f < P.nf; f += GT) {
      double L[36];
      const double* D = P.Sb + 36 * (int64_t)P.diag[f];
#pragma unroll
      for (int k = 0; k < 36; ++k) L[k] = D[k];
      double* Mi = P.Minv + 36 * (int64_t)f;
      double rv[6], zv[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) { rv[i] = P.b[6 * (int64_t)f + i]; v[0] += rv[i] * rv[i]; zv[i] = 0.0; }
      if (!chol_small<6>(L)) {
        atomicOr(P.status, 8);
#pragma unroll
        for (int k = 0; k < 36; ++k) Mi[k] = 0.0;
      } else {
#pragma unroll
        for (int c = 0; c < 6; ++c) {
          double col[6];
#pragma unroll
          for (int i = 0; i < 6; ++i) col[i] = (i == c) ? 1.0 : 0.0;
          fwd_small<6>(L, col);
          bwd_small<6>(L, col);
#pragma unroll
          for (int i = 0; i < 6; ++i) { Mi[i * 6 + c] = col[i]; zv[i] += col[i] * rv[c]; }
        }
      }
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        const int64_t o = 6 * (int64_t)f + i;
        P.x[o] = 0.0; P.r[o] = rv[i]; P.z[o] = zv[i]; P.p0[o] = 0.0;
        v[1] += rv[i] * zv[i];
      }
    }
    pcg_block_sums<2>(v, sm);
    if (threadIdx.x == 0) { pa[blockIdx.x] = v[0]; pc[blockIdx.x] = v[1]; }
  }
  grid.sync();
  double tot0[2];
  {
    const double* arr[2] = {pa, pc};
    pcg_totals<2>(arr, NB, sm, tot0);
  }
  const double norm_b = sqrt(tot0[0]);
  double rho = tot0[1], last_rho = 1.0, Q0 = 0.0;
  const double tol_r = P.r_tol * norm_b;
  int iters = 0;
  bool failed = false;
  int cur = 0;
  if (norm_b != 0.0) {
    for (int it = 1;; ++it) {
      iters = it;
      if (rho == 0.0 || !isfinite(rho)) { failed = true; break; }
      double beta = 0.0;
      if (it > 1) {
        beta = rho / last_rho;
        if (beta == 0.0 || !isfinite(beta)) { failed = true; break; }
      }
      double* pold = cur ? P.p1 : P.p0;
      double* pnew = cur ? P.p0 : P.p1;
      // ---- phase 1: p = z + beta p_old (formed on the fly for the neighbours), q = S p, partial p.q ----
      {
        double v[1] = {0.0};
        for (int f = gw; f < P.nf; f += GW) {
          double acc[6];
          pcg_spmv_row(P, f, P.z, it > 1 ? pold : nullptr, beta, lane, acc);
          double a = acc[0];
#pragma unroll
          for (int i = 1; i < 6; ++i) a = (lane == i) ? acc[i] : a;
          if (lane < 6) {
            const int64_t o = 6 * (int64_t)f + lane;
            const double pv = P.z[o] + (it > 1 ? beta * pold[o] : 0.0);
            pnew[o] = pv;
            P.q[o] = a;
            v[0] += pv * a;
          }
        }
        pcg_block_sums<1>(v, sm);
        if (threadIdx.x == 0) pb[blockIdx.x] = v[0];
      }
      grid.sync();
      const double pq = pcg_total(pb, NB, sm);
      if (pq <= 0.0 || !isfinite(pq)) break;  // keep the current x (Ceres: LINEAR_SOLVER_NO_CONVERGENCE)
      const double alpha = rho / pq;
      if (!isfinite(alpha)) { failed = true; break; }
      const bool reset = (it % P.reset_period) == 0;
      // ---- phase 2: x += alpha p ; r ; z = M^-1 r ; partial sums ----
      {
        double v[3] = {0.0, 0.0, 0.0};   // x.(b + r), r.z, r.r
        if (reset) {  // r = b - S x from scratch
          for (int i = gt; i < 6 * P.nf; i += GT) P.x[i] += alpha * pnew[i];
          grid.sync();
          for (int f = gw; f < P.nf; f += GW) {
            double acc[6];
            pcg_spmv_row(P, f, P.x, nullptr, 0.0, lane, acc);
            double a = acc[0];
#pragma unroll
            for (int i = 1; i < 6; ++i) a = (lane == i) ? acc[i] : a;
            const bool on = lane < 6;
            const int64_t o = 6 * (int64_t)f + (on ? lane : 0);
            const double xv = on ? P.x[o] : 0.0, rv = on ? P.b[o] - a : 0.0;
            pcg_finish_row(P, f, on, 0, on ? lane : 0, xv, rv, v[0], v[1], v[2]);
          }
        } else {      // r -= alpha q: five rows per warp, six lanes each
          for (int f0 = 5 * gw; f0 < P.nf; f0 += 5 * GW) {
            const int f = f0 + grp;
            const bool on = lane < 30 && f < P.nf;
            const int64_t o = 6 * (int64_t)(on ? f : 0) + comp;
            double xv = 0.0, rv = 0.0;
            if (on) { xv = P.x[o] + alpha * pnew[o]; P.x[o] = xv; rv = P.r[o] - alpha * P.q[o]; }
            pcg_finish_row(P, on ? f : 0, on, 6 * (grp < 5 ? grp : 0), comp, xv, rv, v[0], v[1], v[2]);
          }
        }
        pcg_block_sums<3>(v, sm);
        if (threadIdx.x == 0) { pa[blockIdx.x] = v[0]; pc[blockIdx.x] = v[1]; pd[blockIdx.x] = v[2]; }
      }
      grid.sync();
      double tot[3];
      {
        const double* arr[3] = {pa, pc, pd};
        pcg_totals<3>(arr, NB, sm, tot);
      }
      const double Q1 = -tot[0];
      const double zeta = it * (Q1 - Q0) / Q1;
      last_rho = rho;
      rho = tot[1];
      const double rr = tot[2];
      cur ^= 1;
      if (zeta < P.eta && it >= P.min_it) break;
      Q0 = Q1;
      if (sqrt(rr) <= tol_r && it >= P.min_it) break;
      if (it >= P.max_it) break;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    *P.out_iters = iters;
    if (failed) atomicOr(P.status, 16);
  }
  if (failed) {  // invalid step: make sure nothing non-finite leaks into the back-substitution
    for (int i = gt; i < 6 * P.nf; i += GT) P.x[i] = 0.0;
  }
}

struct PcgWork {
  DVec<double> r, z, p0, p1, q, Minv, partial;
  DVec<int> iters;
  int grid = 0;
};

inline int pcg_prepare(PcgWork& W, int64_t nf, int device) {
  BA_TRY(W.r.alloc(6 * nf)); BA_TRY(W.z.alloc(6 * nf)); BA_TRY(W.p0.alloc(6 * nf)); BA_TRY(W.p1.alloc(6 * nf)); BA_TRY(W.q.alloc(6 * nf));
  BA_TRY(W.Minv.alloc(36 * nf)); BA_TRY(W.iters.alloc(1));
  int sms = 0, per_sm = 0;
  BA_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  BA_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pcg, 256, 0));
  if (per_sm < 1) return fail(BA_ERR_CUDA, "k_pcg cannot be made resident");
  const int64_t want = (nf + 7) / 8;  // one warp per block row, 8 warps per CTA
  W.grid = (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)sms * std::min(per_sm, 2), want));
  BA_TRY(W.partial.alloc(4 * (size_t)W.grid * 8));
  return BA_OK;
}

inline int launch_pcg(PcgWork& W, const RcsPattern& R, const double* Sb, const double* rhs, double* x, int* status,
                      const ba_cuda_options& opt, cudaStream_t st) {
  PcgParams P;
  P.nf = (int)R.nf; P.row_ptr = R.row_ptr.p; P.row_ent = R.row_ent.p; P.row_col = R.row_col.p; P.diag = R.diag.p;
  P.Sb = Sb; P.b = rhs; P.x = x; P.r = W.r.p; P.z = W.z.p; P.p0 = W.p0.p; P.p1 = W.p1.p; P.q = W.q.p; P.Minv = W.Minv.p;
  P.partial = W.partial.p; P.max_it = opt.pcg_max_iterations; P.min_it = opt.pcg_min_iterations;
  P.reset_period = opt.pcg_residual_reset_period > 0 ? opt.pcg_residual_reset_period : 10;
  P.eta = opt.pcg_eta; P.r_tol = opt.pcg_r_tolerance; P.out_iters = W.iters.p; P.status = status;
  void* args[] = {&P};
  BA_CUDA_TRY(cudaLaunchCooperativeKernel((const void*)k_pcg, dim3(W.grid), dim3(256), args, 0, st));
  return BA_OK;
}

}  // namespace ba
