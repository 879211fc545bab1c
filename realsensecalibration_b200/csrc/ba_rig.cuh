// ba_rig.cuh -- the rig-size latency path: the whole trust-region loop of ceres::Solve in ONE launch of ONE CTA.
//
// The reference's own problems (Common/Correspondence/hongo: 68 marker observations; Test1/Test2_BundleAdjustment: 16..200
// observations; Main_Calibration/bundle_adjustment_manager.cpp:16-96) are three orders of magnitude below what fills a
// B200: on the multi-kernel pipeline one LM iteration is ~40 launches and two host round trips, all latency.  Here one
// CTA of 256 threads walks the same phases (the item functions d_* of ba_kernels.cuh, so the arithmetic per observation,
// per block and per incidence is the generic pipeline's) separated by __syncthreads instead of launches; the reduced camera
// system lives in shared memory and is factorised there (L D L^T by panels of 8 columns with look-ahead, the right-hand side
// riding along as one more row; rig_ldlt_solve below); TrustRegionMinimizer's loop variables and its decisions (lm_begin /
// lm_iterate of ba_cuda.cu, statement for statement) are taken by thread 0 between barriers, and the iteration rows are
// written to HBM for the host to read after the launch.  Every sum is a fixed tree: results are bitwise reproducible.
#pragma once
#include "ba_kernels.cuh"

namespace ba {

constexpr int RIG_THREADS = 256;        // 255 registers per thread: measured on B200 against 320 / 384 / 512 threads (168 / 168 / 128 registers):
                                        // hongo 8300 vs 6530 / 6840 / 6970 LM it/s.  At the register cap ptxas puts every shared-memory load right
                                        // in front of its use and the dependent chains of the dense solve run 3-5x longer
constexpr int RIG_ROWS_CAP = 256;       // iteration rows one launch can record
constexpr int RIG_MAX_N = 160;       // reduced camera system dimension that fits shared memory (n * (n | 1) doubles)
constexpr int64_t RIG_MAX_ROWS = 8192;    // residual rows (nb * RD); measured crossover with the multi-kernel pipeline ~9k rows (profiles/r02_rig_crossover.txt)

struct RigState {   // LmState of ba_cuda.cu, on the device
  double radius, decrease_factor, x_cost, gmax, gnorm;
  int32_t num_invalid, go, n_rows, term_type, term_reason;
  int32_t n_jac, n_solves, n_success, n_unsuccess, last_iteration, pad_;
  double last_gmax, last_gnorm;      // gradient norms of the previous row (an invalid step repeats them)
};

struct RigParams {
  int64_t nb, ne, nf, ninc;
  int ndest, n, ld;
  // structure (ba_structure.cuh)
  const int32_t *ob_e, *ob_f0, *ob_f1, *ob_cam;
  const int64_t* e_ptr;
  const int32_t *inc_e, *inc_f;
  const int64_t* einc_ptr;
  const int64_t* incobs_ptr; const int32_t* incobs;
  const int64_t *finc_ptr, *fobs_ptr; const int32_t *finc, *fobs;
  const int32_t *dest_fa, *dest_fb;
  const int64_t* dpair_ptr; const int2* pairs;
  const int64_t* dobs_ptr; const int32_t* dobs;
  const int64_t* f_act_ptr;
  // model data
  const double2* uv; const double* obs8; const double* intr_f; double half_side;
  // parameters, scaling, tables
  double *xe, *xf, *xe_c, *xf_c, *se, *sf, *tab_f, *tab_e, *tabc_f, *tabc_e;
  // workspace of the generic pipeline
  double *RES, *JE, *JF0, *JF1, *ME, *HG, *Wt, *Qacc, *Lb, *zb, *Yt, *vb, *Pacc, *vsum, *yf, *ye;
  RigState* state;
  ba_cuda_iteration* rows;
  int32_t rows_base;  // rows recorded by earlier launches of this solve
  int32_t begin;      // 1: start from `init` and run iteration zero first (TrustRegionMinimizer::IterationZero)
  int32_t max_new;    // at most this many loop iterations in this launch (begin + max_new <= RIG_ROWS_CAP)
  RigState init;
  long long* clk;     // BA_RIG_CLOCKS=1: SM cycles per phase (16 slots), thread 0's view
  ba_cuda_options opt;
  LossSpec loss;
};

// ---- CTA-wide helpers --------------------------------------------------------------------------------------
__device__ __forceinline__ double rig_sum(double v, double* red) {   // every thread gets the sum
  v = block_sum(v, red);
  __syncthreads();
  if (threadIdx.x == 0) red[32] = v;
  __syncthreads();
  return red[32];
}
__device__ __forceinline__ double rig_max(double v, double* red) {
  v = block_max(v, red);
  __syncthreads();
  if (threadIdx.x == 0) red[32] = v;
  __syncthreads();
  return red[32];
}
// N values at once (sum, or maximum where is_max): one pair of barriers for all of them; every thread gets the results in v
template <int N>
__device__ __forceinline__ void rig_reduce(double* v, const bool* is_max, double* red /* N * 8 + N */) {
  constexpr int NW = RIG_THREADS / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < N; ++k) {
    double x = v[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double y = __shfl_down_sync(0xffffffffu, x, o);
      x = is_max[k] ? fmax(x, y) : x + y;
    }
    if (lane == 0) red[k * NW + warp] = x;
  }
  __syncthreads();
  if (threadIdx.x < N) {
    const int k = threadIdx.x;
    double x = red[k * NW];
#pragma unroll
    for (int w = 1; w < NW; ++w) x = is_max[k] ? fmax(x, red[k * NW + w]) : x + red[k * NW + w];
    red[N * NW + k] = x;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < N; ++k) v[k] = red[N * NW + k];
  __syncthreads();   // red may be reused right away
}
__device__ __forceinline__ double rig_now_s() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return 1e-9 * (double)t;
}

// tables at x (candidate = false) or at the candidate point
template <int MODEL>
__device__ __forceinline__ void rig_tables(const RigParams& P, bool candidate) {
  const double* xf = candidate ? P.xf_c : P.xf;
  double* tf = candidate ? P.tabc_f : P.tab_f;
  if (MODEL == 1) {   // one pass over both kinds of block (sin / cos make this the longest per-thread chain of the evaluation)
    const double* xe = candidate ? P.xe_c : P.xe;
    double* te = candidate ? P.tabc_e : P.tab_e;
    for (int64_t i = threadIdx.x; i < P.nf + P.ne; i += RIG_THREADS) {
      const bool isf = i < P.nf;
      const int64_t j = isf ? i : i - P.nf;
      d_tables(j, isf ? xf : xe, isf ? P.intr_f : nullptr, isf ? P.sf : P.se, isf ? tf : te);
    }
  } else {
    for (int64_t i = threadIdx.x; i < P.nf; i += RIG_THREADS) d_tables(i, xf, P.intr_f, P.sf, tf);
  }
  __syncthreads();
}

// K1: residuals and scaled Jacobian at x; returns sum r^2 (or sum rho)
template <int MODEL>
__device__ __forceinline__ double rig_jacobian(const RigParams& P, double* red) {
  rig_tables<MODEL>(P, false);
  double sq = 0.0;
  if (MODEL == 0) {
    for (int64_t base = 0; base < P.nb; base += RIG_THREADS) {
      const int64_t o = base + threadIdx.x;
      if (o < P.nb) {
        double jf[12], je[6];
        sq += d_jac_a(o, P.ob_e, P.ob_f0, P.uv, P.tab_f, P.xe, P.se, P.RES, jf, je, P.loss);
        double2* pf = reinterpret_cast<double2*>(P.JF0 + 12 * o);
#pragma unroll
        for (int k = 0; k < 6; ++k) pf[k] = make_double2(jf[2 * k], jf[2 * k + 1]);
        double2* pe = reinterpret_cast<double2*>(P.JE + 6 * o);
#pragma unroll
        for (int k = 0; k < 3; ++k) pe[k] = make_double2(je[2 * k], je[2 * k + 1]);
      }
    }
  } else {
    for (int64_t base = 0; base < 4 * P.nb; base += RIG_THREADS) {   // whole warps: the robust loss sums over a marker's 4 lanes
      const int64_t t = base + threadIdx.x;
      double je12[12], jc12[12], jm12[12];
      sq += d_jac_b(t, P.nb, P.ob_e, P.ob_f0, P.ob_f1, P.ob_cam, P.obs8, P.tab_f, P.tab_e, P.half_side, P.RES, je12, jc12, jm12, P.loss);
      if ((t >> 2) < P.nb) {
        double2* a = reinterpret_cast<double2*>(P.JE + 12 * t);
        double2* b = reinterpret_cast<double2*>(P.JF0 + 12 * t);
        double2* c = reinterpret_cast<double2*>(P.JF1 + 12 * t);
#pragma unroll
        for (int k = 0; k < 6; ++k) {
          a[k] = make_double2(je12[2 * k], je12[2 * k + 1]);
          b[k] = make_double2(jc12[2 * k], jc12[2 * k + 1]);
          c[k] = make_double2(jm12[2 * k], jm12[2 * k + 1]);
        }
      }
    }
  }
  return rig_sum(sq, red);   // its barriers also publish RES / J
}

// K5: cost only, at the candidate
template <int MODEL>
__device__ __forceinline__ double rig_cost_candidate(const RigParams& P, double* red) {
  rig_tables<MODEL>(P, true);
  double sq = 0.0;
  if (MODEL == 0) {
    for (int64_t o = threadIdx.x; o < P.nb; o += RIG_THREADS) sq += d_cost_a(o, P.ob_e, P.ob_f0, P.uv, P.tabc_f, P.xe_c, P.loss);
  } else {
    for (int64_t base = 0; base < 4 * P.nb; base += RIG_THREADS)
      sq += d_cost_b(base + threadIdx.x, P.nb, P.ob_e, P.ob_f0, P.ob_f1, P.ob_cam, P.obs8, P.tabc_f, P.tabc_e, P.half_side, P.loss);
  }
  return rig_sum(sq, red);
}

// K2, the part that depends on J only (run_normal_parts)
template <int RD, int DE, int GE>
__device__ __forceinline__ void rig_normal_parts(const RigParams& P) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NW = RIG_THREADS / 32;
  for (int64_t f = warp; f < P.nf; f += NW) {
    double acc[NV_F];
    d_fobs_seg<RD>(lane, P.fobs_ptr[f], P.fobs_ptr[f + 1], P.fobs, P.RES, P.JF0, P.JF1, acc);
    group_sum_store<NV_F, 32>(acc, lane, P.HG + f * NV_F, true);
  }
  for (int64_t base = 0; base < P.ne * GE; base += RIG_THREADS) d_e_M<RD, DE, GE>(base + threadIdx.x, P.ne, P.e_ptr, P.RES, P.JE, P.ME);
  if (RD == 8) {   // Model B
    for (int64_t base = 0; base < P.ninc * RD; base += RIG_THREADS)
      d_inc_W<RD>(base + threadIdx.x, P.ninc, P.incobs_ptr, P.incobs, P.JE, P.JF0, P.JF1, P.Wt);
    // a destination of a rig holds a handful of observations (the frames that saw the pair): 8 lanes (= rows) per destination
    for (int base = 0; base < P.ndest; base += RIG_THREADS / 8) {
      const int d = base + (threadIdx.x >> 3), r = threadIdx.x & 7;
      const bool live = d < P.ndest;
      double acc[36];
#pragma unroll
      for (int k = 0; k < 36; ++k) acc[k] = 0.0;
      if (live) {
        const int64_t end = P.dobs_ptr[d + 1];
#pragma unroll 4
        for (int64_t idx = P.dobs_ptr[d]; idx < end; ++idx) {
          const int64_t row = (int64_t)RD * P.dobs[idx] + r;
          double ra[6], rb[6];
          load_row6(P.JF0 + row * 6, ra);
          load_row6(P.JF1 + row * 6, rb);
#pragma unroll
          for (int a = 0; a < 6; ++a)
#pragma unroll
            for (int b = 0; b < 6; ++b) acc[a * 6 + b] = fma(ra[a], rb[b], acc[a * 6 + b]);
        }
      }
      group_sum_store<36, 8>(acc, lane, P.Qacc + (int64_t)(live ? d : 0) * 36, live);
    }
  }
  __syncthreads();
}

// gradient norms at x (EvaluateGradientAndJacobian): max and 2-norm over the active blocks
template <int DE>
__device__ __forceinline__ void rig_gradient(const RigParams& P, double* red, double& gmax, double& gnorm) {
  constexpr int NU = DE * (DE + 1) / 2;
  double mx = 0.0, sqe = 0.0, sqf = 0.0;
  for (int64_t t = threadIdx.x; t < P.ne * DE; t += RIG_THREADS) {
    double m = 0.0, s = 0.0;
    d_gradient_norm<DE, NU + DE, NU>(t, P.e_ptr, P.xe, P.se, P.ME, m, s);
    mx = fmax(mx, m); sqe += s;
  }
  for (int64_t t = threadIdx.x; t < P.nf * 6; t += RIG_THREADS) {
    double m = 0.0, s = 0.0;
    d_gradient_norm<6, NV_F, 21>(t, P.f_act_ptr, P.xf, P.sf, P.HG, m, s);
    mx = fmax(mx, m); sqf += s;
  }
  double v[3] = {sqe, sqf, mx};
  const bool is_max[3] = {false, false, true};
  rig_reduce<3>(v, is_max, red);
  const double g2e = v[0], g2f = v[1];
  gmax = v[2];
  gnorm = sqrt(g2e + g2f);
}

// S = L' D^-1 L'^T in place in shared memory (lower triangle; L' keeps the pivots d_k on its diagonal, invd[k] = 1 / d_k),
// blocked by panels of 8 columns: (a) ONE thread factorises the 8 x 8 diagonal block in its registers; (b) one thread per row
// below solves its 8 panel entries against that block; (c) rank-8 update of the trailing triangle, a warp per row, a lane
// per column.  Three barriers per 8 columns.  The right-hand side is row n of S and rides through (b) and (c): that is the
// forward substitution.  The backward substitution runs by panels too (8 dependent steps in warp 0, then one thread per row
// above).  Returns false (uniformly) when a pivot is not positive.
__device__ __forceinline__ bool rig_ldlt_solve(double* S, int n, int ld, double* rhs, double* invd, double* tacc, double* blk /* 64 + 1 */,
                                               double* __restrict__ y_out, long long* sclk) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NW = RIG_THREADS / 32;
  constexpr int NB = 8;
  // (a) the 8 x 8 diagonal block at k0 in warp 0's registers: lane = (row r = lane >> 2, column pair g = lane & 3) holds
  // A[r][2g], A[r][2g+1]; a pivot step is four broadcasts (pivot, the lane's row factor, its two column factors), one
  // reciprocal, two fmas.  When `upd` the block first takes the rank-8 update of the previous panel (columns kp..kp+7), so
  // the factorisation of panel p + 1 starts while the other warps are still in the trailing update of panel p (look-ahead).
  auto diag_block = [&](int k0, bool upd, int kp) {
    const int w = min(NB, n - k0);
    const int r = lane >> 2, g = lane & 3, c0 = 2 * g, c1 = 2 * g + 1;
    const bool in0 = r < w && c0 <= r, in1 = r < w && c1 <= r;
    double* row = S + (k0 + (r < w ? r : 0)) * ld;
    double a0 = in0 ? row[k0 + c0] : (r == c0 ? 1.0 : 0.0);   // identity below a partial last panel
    double a1 = in1 ? row[k0 + c1] : (r == c1 ? 1.0 : 0.0);
    if (upd) {
      const double* rc0 = S + (k0 + (c0 < w ? c0 : 0)) * ld + kp;
      const double* rc1 = S + (k0 + (c1 < w ? c1 : 0)) * ld + kp;
      double li[NB], v0[NB], v1[NB];
#pragma unroll
      for (int kk = 0; kk < NB; ++kk) { li[kk] = row[kp + kk] * invd[kp + kk]; v0[kk] = rc0[kk]; v1[kk] = rc1[kk]; }
      double u0 = 0.0, u1 = 0.0;
#pragma unroll
      for (int kk = 0; kk < NB; ++kk) { u0 = fma(li[kk], v0[kk], u0); u1 = fma(li[kk], v1[kk], u1); }
      if (in0) a0 -= u0;
      if (in1) a1 -= u1;
    }
    bool ok = true;
#pragma unroll
    for (int kk = 0; kk < NB; ++kk) {
      const double mine = (kk & 1) ? a1 : a0;   // this lane's entry of column kk if g == kk / 2
      const double d = __shfl_sync(0xffffffffu, mine, 4 * kk + (kk >> 1));
      const double inv = (d > 0.0 && isfinite(d)) ? __drcp_rn(d) : 0.0;   // = 1.0 / d, correctly rounded
      ok = ok && inv != 0.0;
      const double lrk = __shfl_sync(0xffffffffu, mine, (lane & 28) | (kk >> 1)) * inv;   // A[r][kk] / d_kk
      const double l0 = __shfl_sync(0xffffffffu, mine, 4 * c0 + (kk >> 1));               // A[c0][kk]
      const double l1 = __shfl_sync(0xffffffffu, mine, 4 * c1 + (kk >> 1));               // A[c1][kk]
      if (r > kk) {
        if (c0 > kk && c0 <= r) a0 = fma(-lrk, l0, a0);
        if (c1 > kk && c1 <= r) a1 = fma(-lrk, l1, a1);
        if (g == 0) blk[r * NB + kk] = lrk;   // the block scaled by D^-1, for (b)
      }
      if (lane == 0 && kk < w) invd[k0 + kk] = inv;
    }
    if (in0) row[k0 + c0] = a0;
    if (in1) row[k0 + c1] = a1;
    if (lane == 0) blk[NB * NB] = ok ? 1.0 : 0.0;
  };
  if (warp == 0) diag_block(0, false, 0);
  __syncthreads();
  for (int k0 = 0; k0 < n; k0 += NB) {
    if (blk[NB * NB] == 0.0) return false;   // a pivot of this panel is not positive (uniform: read after a barrier)
    const int w = min(NB, n - k0);
    // rows below the panel, and the right-hand side as one more row (row n of S): its panel solve and trailing update ARE the
    // forward substitution, so after the last panel row n holds v_k = d_k u_k of L' u = rhs at no extra dependent step
    const int i0 = k0 + w;
    const int m = n + 1 - i0;
    long long tq = 0;
    if (sclk && threadIdx.x == 0) tq = clock64();
    for (int r = threadIdx.x; r < m; r += RIG_THREADS) {   // (b)
      double* row = S + (i0 + r) * ld + k0;
      double x[NB];
#pragma unroll
      for (int c = 0; c < NB; ++c) x[c] = c < w ? row[c] : 0.0;
      // column by column: once x[q] is final its NB - 1 - q updates are independent, and their block entries are loaded together
      // (row by row the compiler put every shared-memory load right in front of the fma that waits for it: 28 round trips)
#pragma unroll
      for (int q = 0; q < NB - 1; ++q) {
        double bq[NB];
#pragma unroll
        for (int kk = q + 1; kk < NB; ++kk) bq[kk] = blk[kk * NB + q];
#pragma unroll
        for (int kk = q + 1; kk < NB; ++kk) x[kk] = fma(-x[q], bq[kk], x[kk]);
      }
#pragma unroll
      for (int c = 1; c < NB; ++c)
        if (c < w) row[c] = x[c];
    }
    if (sclk && threadIdx.x == 0) { const long long q = clock64(); sclk[13] += q - tq; tq = q; }
    __syncthreads();
    if (sclk && threadIdx.x == 0) { const long long q = clock64(); sclk[14] += q - tq; tq = q; }
    if (i0 < n) {   // (c), w == NB here: warp 0 takes the next diagonal block (and factorises it), the others the rows below it
      const int nd = min(NB, n - i0);
      if (warp == 0) {
        diag_block(i0, true, k0);
        if (sclk && threadIdx.x == 0) { const long long q = clock64(); sclk[15] += q - tq; tq = q; }
      } else {
        double iv[NB];
#pragma unroll
        for (int kk = 0; kk < NB; ++kk) iv[kk] = invd[k0 + kk];
        const int cols = n - i0;   // trailing columns
#pragma unroll 1
        for (int r = nd + warp - 1; r < m; r += NW - 1) {
          double* row = S + (i0 + r) * ld + k0;
          double li[NB];
#pragma unroll
          for (int kk = 0; kk < NB; ++kk) li[kk] = row[kk] * iv[kk];
          const int cmax = min(r, cols - 1);
#pragma unroll 1
          for (int c = lane; c <= cmax; c += 32) {
            const double* rj = S + (i0 + c) * ld + k0;
            double rv[NB];
#pragma unroll
            for (int kk = 0; kk < NB; ++kk) rv[kk] = rj[kk];
            double acc0 = row[NB + c], acc1 = 0.0;   // two chains of four
#pragma unroll
            for (int kk = 0; kk < NB; kk += 2) { acc0 = fma(-li[kk], rv[kk], acc0); acc1 = fma(-li[kk + 1], rv[kk + 1], acc1); }
            row[NB + c] = acc0 + acc1;
          }
        }
      }
      __syncthreads();
    }
  }
  long long t_f = 0;
  if (sclk && threadIdx.x == 0) t_f = clock64();
  {
    // backward, L'^T x = v  (x_k = (v_k - sum_{i>k} L'[i][k] x_i) / d_k; v = row n of S), panels from the last: tacc[k] collects the sum over
    // the rows already solved; warp 0 finishes the panel, then one thread per row above adds the panel's contribution
    for (int i = threadIdx.x; i < n; i += RIG_THREADS) tacc[i] = 0.0;
    __syncthreads();
    for (int k0 = ((n - 1) / NB) * NB; k0 >= 0; k0 -= NB) {
      const int w = min(NB, n - k0);
      if (warp == 0) {
        double av = lane < w ? tacc[k0 + lane] : 0.0;
        const double uv = lane < w ? rhs[k0 + lane] : 0.0;
        const double iv = lane < w ? invd[k0 + lane] : 0.0;
        double lv[NB];   // column `lane` of the block: L'[k0 + kk][k0 + lane], kk > lane
#pragma unroll
        for (int kk = 0; kk < NB; ++kk) lv[kk] = (lane < kk && kk < w) ? S[(k0 + kk) * ld + k0 + lane] : 0.0;
        double xv = 0.0;
#pragma unroll
        for (int kk = NB - 1; kk >= 0; --kk) {
          const double mine = (uv - av) * iv;   // meaningful in lane kk once the rows below it are in av
          const double xk = __shfl_sync(0xffffffffu, mine, kk);
          if (lane == kk) xv = xk;
          av = fma(lv[kk], xk, av);
        }
        if (lane < w) { rhs[k0 + lane] = xv; y_out[k0 + lane] = xv; }
      }
      __syncthreads();
      for (int i = threadIdx.x; i < k0; i += RIG_THREADS) {
        double sv[NB], xv[NB];
#pragma unroll
        for (int kk = 0; kk < NB; ++kk) { sv[kk] = kk < w ? S[(k0 + kk) * ld + i] : 0.0; xv[kk] = kk < w ? rhs[k0 + kk] : 0.0; }
        double av = tacc[i];
#pragma unroll
        for (int kk = 0; kk < NB; ++kk) av = fma(sv[kk], xv[kk], av);
        tacc[i] = av;
      }
      __syncthreads();
    }
  }
  if (sclk && threadIdx.x == 0) sclk[12] += clock64() - t_f;
  __syncthreads();
  return true;
}

// ---- the kernel ----------------------------------------------------------------------------------------------
template <int RD, int DE, int GE, int NSLOT>
__global__ void __launch_bounds__(RIG_THREADS, 1) k_rig_lm(const RigParams P) {
  constexpr int MODEL = RD == 8 ? 1 : 0;
  constexpr int NU = DE * (DE + 1) / 2;
  extern __shared__ __align__(16) double dsm[];
  double* S = dsm;                          // n x ld
  double* rhs = S + (size_t)P.n * P.ld;     // row n of S: the right-hand side rides through the factorisation
  double* invd = rhs + P.ld;                // n
  double* tacc = invd + P.n;                // n: the backward solve's running sums
  double* blk = tacc + P.n;                 // 65: the scaled diagonal block of the current panel, and its verdict
  __shared__ double red[48];   // rig_reduce<5>: 5 * 8 warps + 5; rig_sum: 32 + 1
  __shared__ RigState st;
  __shared__ int status;
  __shared__ double sh_radius;
  __shared__ int sh_flow;                   // thread 0's decision: 0 continue the loop body, 1 next iteration, 2 leave
  __shared__ long long sclk[16];
  long long clk_last = 0;
  const ba_cuda_options& opt = P.opt;
  const int tid = threadIdx.x;
  if (P.clk && tid == 0) { for (int k = 0; k < 16; ++k) sclk[k] = 0; clk_last = clock64(); }
  auto lap = [&](int slot) { if (P.clk && tid == 0) { const long long now = clock64(); sclk[slot] += now - clk_last; clk_last = now; } };
  const int lane = tid & 31, warp = tid >> 5;
  constexpr int NW = RIG_THREADS / 32;
  if (tid == 0) st = P.begin ? P.init : *P.state;
  __syncthreads();

  // FinalizeIterationAndCheckIfMinimizerCanContinue (lm_finalize), by thread 0
  auto finalize = [&](ba_cuda_iteration& row, double t0) -> bool {
    if (row.step_is_successful) st.n_success++; else st.n_unsuccess++;
    row.trust_region_radius = st.radius;
    row.iteration_time_s = rig_now_s() - t0;
    if (st.n_rows - P.rows_base < RIG_ROWS_CAP) P.rows[st.n_rows - P.rows_base] = row;
    st.n_rows++;
    st.last_iteration = row.iteration;
    st.last_gmax = row.gradient_max_norm; st.last_gnorm = row.gradient_norm;
    if (row.iteration >= opt.max_num_iterations) { st.term_type = BA_NO_CONVERGENCE; st.term_reason = BA_REASON_MAX_ITERATIONS; return false; }
    if (row.step_is_successful && row.gradient_max_norm <= opt.gradient_tolerance) { st.term_type = BA_CONVERGENCE; st.term_reason = BA_REASON_GRADIENT_TOLERANCE; return false; }
    if (row.trust_region_radius <= opt.min_trust_region_radius) { st.term_type = BA_CONVERGENCE; st.term_reason = BA_REASON_MIN_TRUST_REGION_RADIUS; return false; }
    return true;
  };
  auto zero_row = [](ba_cuda_iteration& row) {
    row.iteration = 0; row.step_is_valid = 0; row.step_is_successful = 0; row.linear_solver_iterations = 0;
    row.cost = 0.0; row.cost_change = 0.0; row.gradient_max_norm = 0.0; row.gradient_norm = 0.0; row.step_norm = 0.0;
    row.relative_decrease = 0.0; row.trust_region_radius = 0.0; row.iteration_time_s = 0.0;
  };
  // One loop, one copy of every phase: at its top EvaluateGradientAndJacobian when a row is waiting for it (row 0 of
  // IterationZero / lm_begin, or the row of an accepted step), then the body of lm_iterate.
  bool need_eval = P.begin != 0, first = P.begin != 0;
  ba_cuda_iteration row;
  double t0 = rig_now_s();
  int32_t it = 0;
  for (;;) {
    if (need_eval) {
      if (first) {
        for (int64_t t = tid; t < P.ne * DE; t += RIG_THREADS) P.se[t] = 1.0;
        for (int64_t t = tid; t < P.nf * 6; t += RIG_THREADS) P.sf[t] = 1.0;
        __syncthreads();
      }
      const int passes = (first && opt.jacobi_scaling) ? 2 : 1;   // iteration 0: the second pass has the Jacobian column scaled
      double cost = 0.0;
      lap(11);
#pragma unroll 1
      for (int pass = 0; pass < passes; ++pass) {
        if (pass == 1) {
          for (int64_t t = tid; t < P.ne * DE; t += RIG_THREADS) d_jacobi_scale<DE, NU + DE>(t, P.ME, P.se);
          for (int64_t t = tid; t < P.nf * 6; t += RIG_THREADS) d_jacobi_scale<6, NV_F>(t, P.HG, P.sf);
          __syncthreads();
        }
        cost = rig_jacobian<MODEL>(P, red);
        lap(0);
        rig_normal_parts<RD, DE, GE>(P);
        lap(1);
      }
      double gmax, gnorm;
      rig_gradient<DE>(P, red, gmax, gnorm);
      lap(2);
      if (tid == 0) {
        st.x_cost = 0.5 * cost; st.gmax = gmax; st.gnorm = gnorm; st.n_jac++;
        if (first) {
          zero_row(row);
          if (!isfinite(st.x_cost)) {
            st.term_type = BA_FAILURE; st.term_reason = BA_REASON_INITIAL_EVALUATION_FAILED; st.go = 0;
          } else {
            row.iteration = 0; row.step_is_valid = 1; row.step_is_successful = 1; row.cost = st.x_cost;
            row.gradient_max_norm = st.gmax; row.gradient_norm = st.gnorm;
            st.go = finalize(row, t0) ? 1 : 0;
          }
        } else {
          row.step_is_successful = 1;
          row.cost = st.x_cost; row.gradient_max_norm = st.gmax; row.gradient_norm = st.gnorm;
          st.go = finalize(row, t0) ? 1 : 0;
        }
      }
      __syncthreads();
      need_eval = false; first = false;
    }
    if (!st.go || it >= P.max_new) break;   // st.go is read after a barrier: uniform
    ++it;
    t0 = rig_now_s();
    // ---- compute_step -------------------------------------------------------------------------
    if (tid == 0) { status = 0; sh_radius = st.radius; }
    __syncthreads();
    const double radius = sh_radius;
    for (int64_t e = tid; e < P.ne; e += RIG_THREADS) d_e_chol<DE>(e, P.ME, radius, opt.min_lm_diagonal, opt.max_lm_diagonal, P.Lb, P.zb, &status);
    __syncthreads();
    for (int64_t i = tid; i < P.ninc; i += RIG_THREADS) {
      if (MODEL == 0) d_inc_Y<RD, DE, true>(i, P.inc_e, P.JE, P.JF0, nullptr, P.Lb, P.zb, P.Yt, P.vb);
      else d_inc_Y<RD, DE, false>(i, P.inc_e, nullptr, nullptr, P.Wt, P.Lb, P.zb, P.Yt, P.vb);
    }
    for (int idx = tid; idx < P.n * P.ld; idx += RIG_THREADS) S[idx] = 0.0;
    __syncthreads();
    lap(3);
    for (int64_t f = warp; f < P.nf; f += NW) {
      double acc[6];
      d_finc_seg(lane, P.finc_ptr[f], P.finc_ptr[f + 1], P.finc, P.vb, acc);
      group_sum_store<6, 32>(acc, lane, P.vsum + f * 6, true);
    }
    if (P.ndest >= 2 * NW) {   // many destinations with short pair lists (a rig): 8 lanes (= rows of Yt) per destination
      for (int base = 0; base < P.ndest; base += RIG_THREADS / 8) {
        const int d = base + (tid >> 3), r = tid & 7;
        const bool live = d < P.ndest;
        double acc[36];
#pragma unroll
        for (int q = 0; q < 36; ++q) acc[q] = 0.0;
        if (live && r < DE) {
          const int64_t end = P.dpair_ptr[d + 1];
#pragma unroll 4
          for (int64_t idx = P.dpair_ptr[d]; idx < end; ++idx) {
            const int2 pr = P.pairs[idx];
            if (pr.x < 0) continue;
            double yi[6], yj[6];
            load_row6(P.Yt + ((int64_t)DE * pr.x + r) * 6, yi);
            load_row6(P.Yt + ((int64_t)DE * pr.y + r) * 6, yj);
#pragma unroll
            for (int a = 0; a < 6; ++a)
#pragma unroll
              for (int b = 0; b < 6; ++b) acc[a * 6 + b] = fma(yi[a], yj[b], acc[a * 6 + b]);
          }
        }
        group_sum_store<36, 8>(acc, lane, P.Pacc + (int64_t)(live ? d : 0) * 36, live);
      }
    } else {
      for (int d = warp; d < P.ndest; d += NW) {
        double acc[36];
        d_pairs_seg<DE>(lane, P.dpair_ptr[d], P.dpair_ptr[d + 1], P.pairs, P.Yt, acc);
        group_sum_store<36, 32>(acc, lane, P.Pacc + (int64_t)d * 36, true);
      }
    }
    __syncthreads();
    lap(4);
    for (int64_t t = tid; t < (int64_t)P.ndest * 36; t += RIG_THREADS)
      d_assemble_dense(t, P.dest_fa, P.dest_fb, P.Pacc, MODEL == 1 ? P.Qacc : nullptr, P.ld, S);
    __syncthreads();
    for (int64_t t = tid; t < P.nf * 6; t += RIG_THREADS)
      d_diag_rhs_dense(t, P.HG, NV_F, P.vsum, 6, &sh_radius, opt.min_lm_diagonal, opt.max_lm_diagonal, P.ld, S, rhs);
    __syncthreads();
    lap(5);
    const bool pd = rig_ldlt_solve(S, P.n, P.ld, rhs, invd, tacc, blk, P.yf, P.clk ? sclk : nullptr);
    lap(6);
    if (!pd) {
      for (int t = tid; t < P.n; t += RIG_THREADS) P.yf[t] = 0.0;
      if (tid == 0) status |= 2;
      __syncthreads();
    }
    for (int64_t base = 0; base < P.ne * GE; base += RIG_THREADS)
      d_e_backsub<DE, GE>(base + tid, P.ne, P.einc_ptr, P.inc_f, P.Yt, P.Lb, P.zb, P.yf, P.ye);
    __syncthreads();
    double acc = 0.0;
    for (int64_t rr = tid; rr < P.nb * RD; rr += RIG_THREADS)
      acc += d_model_cost_row<RD, DE, NSLOT>(rr, P.ob_e, P.ob_f0, P.ob_f1, P.RES, P.JE, P.JF0, P.JF1, P.ye, P.yf);
    lap(7);
    double x2e = 0.0, d2e = 0.0, x2f = 0.0, d2f = 0.0;
    for (int64_t t = tid; t < P.ne * DE; t += RIG_THREADS) { double a = 0.0, b = 0.0; d_candidate<DE>(t, P.e_ptr, P.xe, P.se, P.ye, P.xe_c, a, b); x2e += a; d2e += b; }
    for (int64_t t = tid; t < P.nf * 6; t += RIG_THREADS) { double a = 0.0, b = 0.0; d_candidate<6>(t, P.f_act_ptr, P.xf, P.sf, P.yf, P.xf_c, a, b); x2f += a; d2f += b; }
    double sv[5] = {acc, x2e, d2e, x2f, d2f};
    const bool no_max[5] = {false, false, false, false, false};
    rig_reduce<5>(sv, no_max, red);
    const double mcc = sv[0], xe2 = sv[1], de2 = sv[2], xf2 = sv[3], df2 = sv[4];
    lap(8);
    const double cand = rig_cost_candidate<MODEL>(P, red);
    lap(9);

    // ---- the decisions of lm_iterate, by thread 0 ---------------------------------------------
    if (tid == 0) {
      zero_row(row);
      sh_flow = 0;
      st.n_solves++;
      row.iteration = st.last_iteration + 1;
      const double model_cost_change = -mcc;
      const bool solve_ok = status == 0 && isfinite(model_cost_change);
      row.step_is_valid = solve_ok && model_cost_change > 0.0;
      if (!row.step_is_valid) {   // HandleInvalidStep
        if (++st.num_invalid >= opt.max_num_consecutive_invalid_steps) {
          st.term_type = BA_FAILURE; st.term_reason = BA_REASON_TOO_MANY_INVALID_STEPS; st.go = 0;
          sh_flow = 2;
        } else {
          st.radius = st.radius / st.decrease_factor; st.decrease_factor *= 2.0;
          row.cost = st.x_cost; row.cost_change = 0.0;
          row.gradient_max_norm = st.last_gmax; row.gradient_norm = st.last_gnorm;
          st.go = finalize(row, t0) ? 1 : 0;
          sh_flow = 1;
        }
      } else {
        st.num_invalid = 0;
        const double cand_cost = 0.5 * cand;
        const double x_norm = sqrt(xe2 + xf2);
        row.step_norm = sqrt(de2 + df2);
        row.cost_change = st.x_cost - cand_cost;
        if (row.step_norm <= opt.parameter_tolerance * (x_norm + opt.parameter_tolerance)) {   // ParameterToleranceReached
          st.term_type = BA_CONVERGENCE; st.term_reason = BA_REASON_PARAMETER_TOLERANCE; st.go = 0;
          sh_flow = 2;
        } else if (fabs(row.cost_change) <= opt.function_tolerance * st.x_cost) {              // FunctionToleranceReached
          st.term_type = BA_CONVERGENCE; st.term_reason = BA_REASON_FUNCTION_TOLERANCE; st.go = 0;
          sh_flow = 2;
        } else {
          row.relative_decrease = row.cost_change / model_cost_change;
          if (row.relative_decrease > opt.min_relative_decrease) {   // HandleSuccessfulStep
            const double q = 2.0 * row.relative_decrease - 1.0;
            st.radius = st.radius / fmax(1.0 / 3.0, 1.0 - q * q * q);
            st.radius = fmin(opt.max_trust_region_radius, st.radius);
            st.decrease_factor = 2.0;
            sh_flow = 3;   // accept: x <- candidate, evaluate there
          } else {       // HandleUnsuccessfulStep
            st.radius = st.radius / st.decrease_factor; st.decrease_factor *= 2.0;
            row.cost = cand_cost;
            st.go = finalize(row, t0) ? 1 : 0;
            sh_flow = 1;
          }
        }
      }
    }
    __syncthreads();
    lap(10);
    const int flow = sh_flow;
    if (flow == 2) break;
    if (flow == 3) {
      for (int64_t t = tid; t < P.ne * DE; t += RIG_THREADS) P.xe[t] = P.xe_c[t];
      for (int64_t t = tid; t < P.nf * 6; t += RIG_THREADS) P.xf[t] = P.xf_c[t];
      __syncthreads();
      need_eval = true;
    }
  }
  __syncthreads();
  if (tid == 0) *P.state = st;
  if (P.clk && tid == 0) for (int k = 0; k < 16; ++k) P.clk[k] = sclk[k];
}

// The same factorisation as a kernel of its own: the dense reduced-system solve of the multi-kernel pipeline for n <= RIG_MAX_N
// (S row-major n x n in HBM, not modified; only its lower triangle and diagonal are read).  As the other dense solvers:
// status |= 2 and y = 0 when a pivot is not positive, status |= 4 when the solution is not finite.
__global__ void __launch_bounds__(RIG_THREADS, 1)
k_ldlt_small(int n, const double* __restrict__ Sg, const double* __restrict__ rhs_g, double* __restrict__ y, int* status) {
  extern __shared__ __align__(16) double dsm[];
  const int ld = n | 1;
  double* S = dsm;
  double* rhs = S + (size_t)n * ld;
  double* invd = rhs + ld;
  double* tacc = invd + n;
  double* blk = tacc + n;
  for (int idx = threadIdx.x; idx < n * n; idx += RIG_THREADS) {
    const int i = idx / n, j = idx - i * n;
    S[i * ld + j] = Sg[idx];
  }
  for (int i = threadIdx.x; i < n; i += RIG_THREADS) rhs[i] = rhs_g[i];
  __syncthreads();
  if (!rig_ldlt_solve(S, n, ld, rhs, invd, tacc, blk, y, nullptr)) {
    for (int i = threadIdx.x; i < n; i += RIG_THREADS) y[i] = 0.0;
    if (threadIdx.x == 0) atomicOr(status, 2);
    return;
  }
  for (int i = threadIdx.x; i < n; i += RIG_THREADS)   // rhs holds the solution (rig_ldlt_solve ends on a barrier)
    if (!isfinite(rhs[i])) atomicOr(status, 4);
}

inline size_t rig_smem_bytes(int n) { return sizeof(double) * (((size_t)n + 1) * (n | 1) + 2 * (size_t)n + 66); }

}  // namespace ba

