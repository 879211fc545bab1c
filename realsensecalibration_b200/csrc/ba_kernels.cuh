// ba_kernels.cuh -- the hot-path kernels (fp64 throughout).
//
//   K1  residual + analytic Jacobian      k_tables, k_jac_a, k_jac_b       (replaces the AutoDiff functors,
//                                          Test1 bundle_adjustmenter.cpp:122-141, bundle_adjustment.h:74-125 ...)
//   K2  Schur elimination / RCS assembly  k_fobs_partial, k_e_M, k_inc_W, k_e_chol, k_inc_Y, k_finc_partial,
//                                          k_pairs_partial, k_dobs_partial, k_seg_final, k_assemble_*, k_diag_rhs
//   K4  back-substitution / model cost / candidate   k_e_backsub, k_model_cost, k_candidate
//   K5  cost-only evaluation              k_cost_a, k_cost_b  (same projection as reprojection_check.cpp:69,81)
//
// Data layout in HBM (all per sorted observation "o", sorted by eliminated block):
//   RES[o][RD]  JE[o][RD][DE]  JF0[o][RD][6]  JF1[o][RD][6]      AoS records, so both the sequential
//   passes and the per-camera / per-pair gathers touch whole 32-byte sectors.
//   Yt[i][DE][6]  (= L^-1 W_i^T, k-major)  v[i][6]               per incidence i = (e,f)
//   tab[block][32] = R(9) | A = left Jacobian of SO(3) (9) | t(3) | fx fy ppx ppy (4) | small-angle flag | scale s(6)
//
// The item functions (d_*) are shared with the single-CTA rig kernel (ba_rig.cuh), which rewrites tables and Jacobians
// inside one launch: no explicit __ldg here (the kernels' const __restrict__ parameters still get the read-only path).
//
// Every reduction is a fixed-shape tree over a list produced by a stable sort: no floating
// point atomics anywhere, results are bitwise reproducible run to run.
#pragma once
#include <cfloat>

#include "ba_util.cuh"

namespace ba {

constexpr int TAB = 32;      // doubles per block table
constexpr int NV_F = 27;     // 21 packed upper of F^T F diagonal block + 6 of F^T r
__host__ __device__ constexpr int packed_upper(int d) { return d * (d + 1) / 2; }
__device__ __forceinline__ int sym_idx6(int a, int b) { return a * 6 - a * (a - 1) / 2 + (b - a); }  // a <= b

// ---------------------------------------------------------------------------------------
// Block tables.  R is evaluated with the expression sequence of ceres::AngleAxisRotatePoint
// (Ceres 1.14 rotation.h) applied to the basis vectors, including its theta^2 <= epsilon
// first-order branch; A is the SO(3) left Jacobian, so that d(R(w)X)/dw = -[R X]x A, which
// is the exact derivative the reference's Jets evaluate.  In the small-angle branch Ceres
// differentiates X + w x X, i.e. the derivative is -[X]x: flag = 1, A = I, and the kernels
// use X in place of R X.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void d_tables(int64_t i, const double* __restrict__ x6, const double* __restrict__ intr4,
                                         const double* __restrict__ s6, double* __restrict__ tab) {
  const double w0 = x6[6 * i], w1 = x6[6 * i + 1], w2 = x6[6 * i + 2];
  double R[9], A[9], flag;
  const double theta2 = w0 * w0 + w1 * w1 + w2 * w2;
  if (theta2 > DBL_EPSILON) {
    const double theta = sqrt(theta2);
    const double c = cos(theta), sn = sin(theta);
    const double ti = 1.0 / theta;
    const double k0 = w0 * ti, k1 = w1 * ti, k2 = w2 * ti;
    const double omc = 1.0 - c;
    const double t0 = k0 * omc, t1 = k1 * omc, t2 = k2 * omc;  // (k . e_col) (1 - cos)
    // column 0: pt = e0, k x pt = (0, k2, -k1)
    R[0] = c + k0 * t0;        R[3] = k2 * sn + k1 * t0;  R[6] = -k1 * sn + k2 * t0;
    // column 1: pt = e1, k x pt = (-k2, 0, k0)
    R[1] = -k2 * sn + k0 * t1; R[4] = c + k1 * t1;        R[7] = k0 * sn + k2 * t1;
    // column 2: pt = e2, k x pt = (k1, -k0, 0)
    R[2] = k1 * sn + k0 * t2;  R[5] = -k0 * sn + k1 * t2; R[8] = c + k2 * t2;
    const double a1 = sn / theta;
    const double hs = sin(0.5 * theta);
    const double a3 = 2.0 * hs * hs / theta;
    const double a2 = 1.0 - a1;
    A[0] = a1 + a2 * k0 * k0;      A[1] = a2 * k0 * k1 - a3 * k2; A[2] = a2 * k0 * k2 + a3 * k1;
    A[3] = a2 * k1 * k0 + a3 * k2; A[4] = a1 + a2 * k1 * k1;      A[5] = a2 * k1 * k2 - a3 * k0;
    A[6] = a2 * k2 * k0 - a3 * k1; A[7] = a2 * k2 * k1 + a3 * k0; A[8] = a1 + a2 * k2 * k2;
    flag = 0.0;
  } else {
    R[0] = 1.0; R[1] = -w2; R[2] = w1;
    R[3] = w2;  R[4] = 1.0; R[5] = -w0;
    R[6] = -w1; R[7] = w0;  R[8] = 1.0;
#pragma unroll
    for (int q = 0; q < 9; ++q) A[q] = (q % 4 == 0) ? 1.0 : 0.0;
    flag = 1.0;
  }
  double* T = tab + TAB * i;
#pragma unroll
  for (int q = 0; q < 9; ++q) { T[q] = R[q]; T[9 + q] = A[q]; }
  T[18] = x6[6 * i + 3]; T[19] = x6[6 * i + 4]; T[20] = x6[6 * i + 5];
#pragma unroll
  for (int q = 0; q < 4; ++q) T[21 + q] = intr4 ? intr4[4 * i + q] : 0.0;
  T[25] = flag;
#pragma unroll
  for (int q = 0; q < 6; ++q) T[26 + q] = s6 ? s6[6 * i + q] : 1.0;
}
__global__ void k_tables(const double* __restrict__ x6, const double* __restrict__ intr4, const double* __restrict__ s6,
                         int64_t n, double* __restrict__ tab) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) d_tables(i, x6, intr4, s6, tab);
}

__device__ __forceinline__ void load_tab(const double* __restrict__ tab, int64_t blk, double* T) {
  const double2* p = reinterpret_cast<const double2*>(tab + TAB * blk);
#pragma unroll
  for (int q = 0; q < TAB / 2; ++q) { const double2 v = (*(p + q)); T[2 * q] = v.x; T[2 * q + 1] = v.y; }
}
__device__ __forceinline__ void mat3_vec(const double* R, const double* x, double* y) {
  y[0] = R[0] * x[0] + R[1] * x[1] + R[2] * x[2];
  y[1] = R[3] * x[0] + R[4] * x[1] + R[5] * x[2];
  y[2] = R[6] * x[0] + R[7] * x[1] + R[8] * x[2];
}
// Robust loss of one residual block (ceres::HuberLoss / ceres::CauchyLoss, loss_function.cc) and Ceres' Corrector
// (corrector.cc): for both losses rho'' <= 0, so the corrected residuals and Jacobian rows are the plain ones times
// sqrt(rho'(s)); the block's cost term is rho(s) / 2.  type 0 (the reference: NULL loss) leaves everything untouched.
struct LossSpec { int type; double a; };
__host__ __device__ __forceinline__ void loss_apply(const LossSpec L, double s, double* rho, double* w) {
  *rho = s; *w = 1.0;
  if (L.type == 1) {            // Huber: rho = s below a^2, 2 a sqrt(s) - a^2 above
    const double b = L.a * L.a;
    if (s > b) { const double r = sqrt(s); *rho = 2.0 * L.a * r - b; *w = sqrt(fmax(DBL_MIN, L.a / r)); }
  } else if (L.type == 2) {     // Cauchy: rho = a^2 log(1 + s / a^2)
    const double b = L.a * L.a, sum = 1.0 + s / b, inv = 1.0 / sum;
    *rho = b * log(sum); *w = sqrt(fmax(DBL_MIN, inv));
  }
}

// D[:,k] = A[:,k] x b  (= -[b]x A), the derivative of the rotated point w.r.t. the angle-axis
__device__ __forceinline__ void rot_deriv(const double* A, const double* b, double* D /*3x3 row-major*/) {
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double a0 = A[k], a1 = A[3 + k], a2 = A[6 + k];
    D[k] = a1 * b[2] - a2 * b[1];
    D[3 + k] = a2 * b[0] - a0 * b[2];
    D[6 + k] = a0 * b[1] - a1 * b[0];
  }
}

// Coalesced AoS store: every thread of the CTA owns W consecutive doubles of dst (record tid of the CTA's
// contiguous slice starting at dst); a direct store would scatter 16-byte pieces W * 8 bytes apart.  The records go
// through shared memory (row stride WS doubles, chosen so that the double2 stores are conflict free) and leave as
// full 128-byte lines.  All threads of the CTA must call; n_valid = records of this CTA that exist.
template <int W, int WS>
__device__ __forceinline__ void staged_store(double* stage, const double* vals, bool valid, double* __restrict__ dst, int n_valid) {
  static_assert(W % 2 == 0 && WS % 2 == 0 && WS >= W, "double2 granularity");
  if (valid) {
    double2* row = reinterpret_cast<double2*>(stage + (size_t)threadIdx.x * WS);
#pragma unroll
    for (int k = 0; k < W / 2; ++k) row[k] = make_double2(vals[2 * k], vals[2 * k + 1]);
  }
  __syncthreads();
  const double2* src = reinterpret_cast<const double2*>(stage);
  double2* out = reinterpret_cast<double2*>(dst);
  for (int g = threadIdx.x; g < n_valid * (W / 2); g += blockDim.x) out[g] = src[(g / (W / 2)) * (WS / 2) + g % (W / 2)];
  __syncthreads();
}

// ---------------------------------------------------------------------------------------
// Model A.  One thread per observation (sorted by point).
// ---------------------------------------------------------------------------------------
// one observation: residual (written), the two Jacobian rows of the camera (jf) and of the point (je), |r|^2 (or rho)
__device__ __forceinline__ double d_jac_a(int64_t o, const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f0,
                                          const double2* __restrict__ uv, const double* __restrict__ tab_f,
                                          const double* __restrict__ xe, const double* __restrict__ se, double* __restrict__ RES,
                                          double* jf, double* je, LossSpec L) {
  double sq;
  {
    const int32_t e = ob_e[o], c = ob_f0[o];
    double T[TAB];
    load_tab(tab_f, c, T);
    const double X[3] = {xe[3 * (int64_t)e], xe[3 * (int64_t)e + 1], xe[3 * (int64_t)e + 2]};
    const double s0 = se[3 * (int64_t)e], s1 = se[3 * (int64_t)e + 1], s2 = se[3 * (int64_t)e + 2];
    double q[3];
    mat3_vec(T, X, q);
    const double p0 = q[0] + T[18], p1 = q[1] + T[19], p2 = q[2] + T[20];
    const double2 ob = uv[o];
    double r0 = T[21] * p0 / p2 + T[23] - ob.x;
    double r1 = T[22] * p1 / p2 + T[24] - ob.y;
    sq = r0 * r0 + r1 * r1;
    const double iz = 1.0 / p2;
    const double a = T[21] * iz, bb = -T[21] * p0 * iz * iz, cc = T[22] * iz, dd = -T[22] * p1 * iz * iz;
    double D[9];
    rot_deriv(T + 9, T[25] != 0.0 ? X : q, D);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      jf[k] = (a * D[k] + bb * D[6 + k]) * T[26 + k];
      jf[6 + k] = (cc * D[3 + k] + dd * D[6 + k]) * T[26 + k];
    }
    jf[3] = a * T[29]; jf[4] = 0.0;        jf[5] = bb * T[31];
    jf[9] = 0.0;       jf[10] = cc * T[30]; jf[11] = dd * T[31];
    je[0] = (a * T[0] + bb * T[6]) * s0; je[1] = (a * T[1] + bb * T[7]) * s1; je[2] = (a * T[2] + bb * T[8]) * s2;
    je[3] = (cc * T[3] + dd * T[6]) * s0; je[4] = (cc * T[4] + dd * T[7]) * s1; je[5] = (cc * T[5] + dd * T[8]) * s2;
    if (L.type != 0) {
      double w;
      loss_apply(L, sq, &sq, &w);
      r0 *= w; r1 *= w;
#pragma unroll
      for (int k = 0; k < 12; ++k) jf[k] *= w;
#pragma unroll
      for (int k = 0; k < 6; ++k) je[k] *= w;
    }
    reinterpret_cast<double2*>(RES)[o] = make_double2(r0, r1);
  }
  return sq;
}
__global__ void __launch_bounds__(256)
k_jac_a(int64_t nb, const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f0, const double2* __restrict__ uv,
        const double* __restrict__ tab_f, const double* __restrict__ xe, const double* __restrict__ se,
        double* __restrict__ RES, double* __restrict__ JE, double* __restrict__ JF0, double* __restrict__ cost_partial, LossSpec L) {
  __shared__ double sm[32];
  __shared__ __align__(16) double stage[256 * 14];
  const int64_t o0 = blockIdx.x * (int64_t)blockDim.x;
  const int64_t o = o0 + threadIdx.x;
  const int n_valid = (int)min((int64_t)blockDim.x, nb - o0);
  double sq = 0.0;
  double jf[12], je[6];
  if (o < nb) sq = d_jac_a(o, ob_e, ob_f0, uv, tab_f, xe, se, RES, jf, je, L);
  staged_store<12, 14>(stage, jf, o < nb, JF0 + 12 * o0, n_valid);
  staged_store<6, 6>(stage, je, o < nb, JE + 6 * o0, n_valid);
  sq = block_sum(sq, sm);
  if (threadIdx.x == 0) cost_partial[blockIdx.x] = sq;
}

__device__ __forceinline__ double d_cost_a(int64_t o, const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f0,
                                           const double2* __restrict__ uv, const double* __restrict__ tab_f,
                                           const double* __restrict__ xe, LossSpec L) {
  double sq;
  {
    const int32_t e = ob_e[o], c = ob_f0[o];
    const double* T = tab_f + TAB * (int64_t)c;
    const double X[3] = {xe[3 * (int64_t)e], xe[3 * (int64_t)e + 1], xe[3 * (int64_t)e + 2]};
    double R[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = (*(T + k));
    double q[3];
    mat3_vec(R, X, q);
    const double p0 = q[0] + (*(T + 18)), p1 = q[1] + (*(T + 19)), p2 = q[2] + (*(T + 20));
    const double2 ob = uv[o];
    const double r0 = (*(T + 21)) * p0 / p2 + (*(T + 23)) - ob.x;
    const double r1 = (*(T + 22)) * p1 / p2 + (*(T + 24)) - ob.y;
    sq = r0 * r0 + r1 * r1;
    if (L.type != 0) { double w; loss_apply(L, sq, &sq, &w); }
  }
  return sq;
}
__global__ void __launch_bounds__(256)
k_cost_a(int64_t nb, const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f0, const double2* __restrict__ uv,
         const double* __restrict__ tab_f, const double* __restrict__ xe, double* __restrict__ cost_partial, LossSpec L) {
  __shared__ double sm[32];
  const int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  double sq = o < nb ? d_cost_a(o, ob_e, ob_f0, uv, tab_f, xe, L) : 0.0;
  sq = block_sum(sq, sm);
  if (threadIdx.x == 0) cost_partial[blockIdx.x] = sq;
}

// ---------------------------------------------------------------------------------------
// Model B.  One thread per (marker observation, corner); 4 consecutive threads share an obs.
// f-block index space: [0,C) cameras, [C,C+M) markers; e = frame.  ob_f0 / ob_f1 are -1
// where the functor of the reference does not take that block (camera 0; marker 0 under
// the Main dispatch), and then that transform is not applied at all.
// ---------------------------------------------------------------------------------------
struct BPoint {
  double p3[3];       // point in the target camera
  double G[9], H[9];  // d p3 / d p2, d p3 / d p1
  double bc[3], bt[3], bm[3];
};

__device__ __forceinline__ void model_b_chain(const double* Tc, const double* Tt, const double* Tm, double half, int corner,
                                              bool want_deriv, BPoint& P) {
  double q0[3] = {(corner == 0 || corner == 3) ? -half : half, (corner < 2) ? half : -half, 0.0};
  double p1[3], p2[3], r[3];
  if (Tm) {
    mat3_vec(Tm, q0, r);
    p1[0] = r[0] + Tm[18]; p1[1] = r[1] + Tm[19]; p1[2] = r[2] + Tm[20];
    if (want_deriv) { const double* b = Tm[25] != 0.0 ? q0 : r; P.bm[0] = b[0]; P.bm[1] = b[1]; P.bm[2] = b[2]; }
  } else {
    p1[0] = q0[0]; p1[1] = q0[1]; p1[2] = q0[2];
  }
  mat3_vec(Tt, p1, r);
  p2[0] = r[0] + Tt[18]; p2[1] = r[1] + Tt[19]; p2[2] = r[2] + Tt[20];
  if (want_deriv) { const double* b = Tt[25] != 0.0 ? p1 : r; P.bt[0] = b[0]; P.bt[1] = b[1]; P.bt[2] = b[2]; }
  if (Tc) {
    mat3_vec(Tc, p2, r);
    P.p3[0] = r[0] + Tc[18]; P.p3[1] = r[1] + Tc[19]; P.p3[2] = r[2] + Tc[20];
    if (want_deriv) {
      const double* b = Tc[25] != 0.0 ? p2 : r; P.bc[0] = b[0]; P.bc[1] = b[1]; P.bc[2] = b[2];
#pragma unroll
      for (int k = 0; k < 9; ++k) P.G[k] = Tc[k];
    }
  } else {
    P.p3[0] = p2[0]; P.p3[1] = p2[1]; P.p3[2] = p2[2];
    if (want_deriv) {
#pragma unroll
      for (int k = 0; k < 9; ++k) P.G[k] = (k % 4 == 0) ? 1.0 : 0.0;
    }
  }
  if (want_deriv) {
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) P.H[3 * i + j] = P.G[3 * i] * Tt[j] + P.G[3 * i + 1] * Tt[3 + j] + P.G[3 * i + 2] * Tt[6 + j];
  }
}

// rows (2 x 6) of one block's Jacobian: [a 0 bb; 0 cc dd] * Mleft * [Drot | I], scaled by s
__device__ __forceinline__ void b_rows(const double* Mleft /*3x3 or nullptr = I*/, const double* A, const double* b, const double* s,
                                       double a, double bb, double cc, double dd, double* row0, double* row1) {
  double D[9];
  rot_deriv(A, b, D);
  double u[3], v[3];  // u = row0 of proj * Mleft, v = row1 of proj * Mleft
  if (Mleft) {
#pragma unroll
    for (int j = 0; j < 3; ++j) { u[j] = a * Mleft[j] + bb * Mleft[6 + j]; v[j] = cc * Mleft[3 + j] + dd * Mleft[6 + j]; }
  } else {
    u[0] = a; u[1] = 0.0; u[2] = bb; v[0] = 0.0; v[1] = cc; v[2] = dd;
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    row0[k] = (u[0] * D[k] + u[1] * D[3 + k] + u[2] * D[6 + k]) * s[k];
    row1[k] = (v[0] * D[k] + v[1] * D[3 + k] + v[2] * D[6 + k]) * s[k];
    row0[3 + k] = u[k] * s[3 + k];
    row1[3 + k] = v[k] * s[3 + k];
  }
}

// one (marker observation, corner): the two residuals (written) and the two rows of the three Jacobian blocks; returns
// |r|^2 (robust loss: rho of the marker observation in its corner-0 lane).  Called by whole warps (the loss uses shuffles).
__device__ __forceinline__ double d_jac_b(int64_t t, int64_t nb, const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f0,
                                          const int32_t* __restrict__ ob_f1, const int32_t* __restrict__ ob_cam,
                                          const double* __restrict__ obs8, const double* __restrict__ tab_f,
                                          const double* __restrict__ tab_e, double half, double* __restrict__ RES, double* je12,
                                          double* jc12, double* jm12, LossSpec L) {
  const int64_t o = t >> 2;
  const int corner = (int)(t & 3);
  double sq = 0.0, rr0 = 0.0, rr1 = 0.0;
#pragma unroll
  for (int k = 0; k < 12; ++k) { je12[k] = 0.0; jc12[k] = 0.0; jm12[k] = 0.0; }
  if (o < nb) {
    const int32_t f0 = ob_f0[o], f1 = ob_f1[o];
    double Tc[TAB], Tt[TAB], Tm[TAB];
    load_tab(tab_e, ob_e[o], Tt);
    if (f0 >= 0) load_tab(tab_f, f0, Tc);
    if (f1 >= 0) load_tab(tab_f, f1, Tm);
    const double* K = tab_f + TAB * (int64_t)ob_cam[o] + 21;
    const double fx = (*(K)), fy = (*(K + 1)), ppx = (*(K + 2)), ppy = (*(K + 3));
    BPoint P;
    model_b_chain(f0 >= 0 ? Tc : nullptr, Tt, f1 >= 0 ? Tm : nullptr, half, corner, true, P);
    const double p0 = P.p3[0], p1 = P.p3[1], p2 = P.p3[2];
    const double r0 = fx * p0 / p2 + ppx - obs8[8 * o + 2 * corner];
    const double r1 = fy * p1 / p2 + ppy - obs8[8 * o + 2 * corner + 1];
    sq = r0 * r0 + r1 * r1;
    const double iz = 1.0 / p2;
    const double a = fx * iz, bb = -fx * p0 * iz * iz, cc = fy * iz, dd = -fy * p1 * iz * iz;
    double row0[6], row1[6];
    b_rows(P.G, Tt + 9, P.bt, Tt + 26, a, bb, cc, dd, row0, row1);
#pragma unroll
    for (int k = 0; k < 6; ++k) { je12[k] = row0[k]; je12[6 + k] = row1[k]; }
    if (f0 >= 0) b_rows(nullptr, Tc + 9, P.bc, Tc + 26, a, bb, cc, dd, row0, row1);
#pragma unroll
    for (int k = 0; k < 6; ++k) { jc12[k] = f0 >= 0 ? row0[k] : 0.0; jc12[6 + k] = f0 >= 0 ? row1[k] : 0.0; }
    if (f1 >= 0) b_rows(P.H, Tm + 9, P.bm, Tm + 26, a, bb, cc, dd, row0, row1);
#pragma unroll
    for (int k = 0; k < 6; ++k) { jm12[k] = f1 >= 0 ? row0[k] : 0.0; jm12[6 + k] = f1 >= 0 ? row1[k] : 0.0; }
    rr0 = r0; rr1 = r1;
  }
  if (L.type != 0) {   // the residual block is the marker observation: |r|^2 over its four corners (four consecutive lanes)
    double s = sq;
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    double rho, w;
    loss_apply(L, s, &rho, &w);
    sq = corner == 0 ? rho : 0.0;
    rr0 *= w; rr1 *= w;
#pragma unroll
    for (int k = 0; k < 12; ++k) { je12[k] *= w; jc12[k] *= w; jm12[k] *= w; }
  }
  if (o < nb) {
    RES[8 * o + 2 * corner] = rr0;
    RES[8 * o + 2 * corner + 1] = rr1;
  }
  return sq;
}
__global__ void __launch_bounds__(128)
k_jac_b(int64_t nb, const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f0, const int32_t* __restrict__ ob_f1,
        const int32_t* __restrict__ ob_cam, const double* __restrict__ obs8, const double* __restrict__ tab_f,
        const double* __restrict__ tab_e, double half, double* __restrict__ RES, double* __restrict__ JE,
        double* __restrict__ JF0, double* __restrict__ JF1, double* __restrict__ cost_partial, LossSpec L) {
  __shared__ double sm[32];
  __shared__ __align__(16) double stage[128 * 14];
  const int64_t t0 = blockIdx.x * (int64_t)blockDim.x;   // (marker observation, corner) records are contiguous: 12 doubles each
  const int64_t t = t0 + threadIdx.x;
  const int64_t o = t >> 2;
  const int n_valid = (int)min((int64_t)blockDim.x, 4 * nb - t0);
  double je12[12], jc12[12], jm12[12];
  double sq = d_jac_b(t, nb, ob_e, ob_f0, ob_f1, ob_cam, obs8, tab_f, tab_e, half, RES, je12, jc12, jm12, L);
  staged_store<12, 14>(stage, je12, o < nb, JE + 12 * t0, n_valid);
  staged_store<12, 14>(stage, jc12, o < nb, JF0 + 12 * t0, n_valid);
  staged_store<12, 14>(stage, jm12, o < nb, JF1 + 12 * t0, n_valid);
  sq = block_sum(sq, sm);
  if (threadIdx.x == 0) cost_partial[blockIdx.x] = sq;
}

__device__ __forceinline__ double d_cost_b(int64_t t, int64_t nb, const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f0,
                                           const int32_t* __restrict__ ob_f1, const int32_t* __restrict__ ob_cam,
                                           const double* __restrict__ obs8, const double* __restrict__ tab_f,
                                           const double* __restrict__ tab_e, double half, LossSpec L) {
  const int64_t o = t >> 2;
  const int corner = (int)(t & 3);
  double sq = 0.0;
  if (o < nb) {
    const int32_t f0 = ob_f0[o], f1 = ob_f1[o];
    double Tc[TAB], Tt[TAB], Tm[TAB];
    load_tab(tab_e, ob_e[o], Tt);
    if (f0 >= 0) load_tab(tab_f, f0, Tc);
    if (f1 >= 0) load_tab(tab_f, f1, Tm);
    const double* K = tab_f + TAB * (int64_t)ob_cam[o] + 21;
    BPoint P;
    model_b_chain(f0 >= 0 ? Tc : nullptr, Tt, f1 >= 0 ? Tm : nullptr, half, corner, false, P);
    const double r0 = (*(K)) * P.p3[0] / P.p3[2] + (*(K + 2)) - obs8[8 * o + 2 * corner];
    const double r1 = (*(K + 1)) * P.p3[1] / P.p3[2] + (*(K + 3)) - obs8[8 * o + 2 * corner + 1];
    sq = r0 * r0 + r1 * r1;
  }
  if (L.type != 0) {
    double s = sq;
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    double rho, w;
    loss_apply(L, s, &rho, &w);
    sq = corner == 0 ? rho : 0.0;
  }
  return sq;
}
__global__ void __launch_bounds__(128)
k_cost_b(int64_t nb, const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f0, const int32_t* __restrict__ ob_f1,
         const int32_t* __restrict__ ob_cam, const double* __restrict__ obs8, const double* __restrict__ tab_f,
         const double* __restrict__ tab_e, double half, double* __restrict__ cost_partial, LossSpec L) {
  __shared__ double sm[32];
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;   // one thread per (marker observation, corner)
  double sq = d_cost_b(t, nb, ob_e, ob_f0, ob_f1, ob_cam, obs8, tab_f, tab_e, half, L);
  sq = block_sum(sq, sm);
  if (threadIdx.x == 0) cost_partial[blockIdx.x] = sq;
}

// ---------------------------------------------------------------------------------------
// K2: generic over RD (residuals / obs), DE (size of the eliminated block).
// ---------------------------------------------------------------------------------------
// F^T F diagonal block (packed 21) and F^T r (6) of one f-block, chunk partials.  One warp per chunk; a lane owns one
// residual row of one observation (32 / RD observations per step), so a warp reads whole 48-byte rows side by side.
__device__ __forceinline__ void load_row6(const double* __restrict__ p, double* row) {
  const double2* q = reinterpret_cast<const double2*>(p);
#pragma unroll
  for (int k = 0; k < 3; ++k) { const double2 v = q[k]; row[2 * k] = v.x; row[2 * k + 1] = v.y; }
}
// this lane's share of list entries [begin, end) (sum the 27 values over the warp afterwards)
template <int RD>
__device__ __forceinline__ void d_fobs_seg(int lane, int64_t begin, int64_t end, const int32_t* __restrict__ fobs,
                                           const double* __restrict__ RES, const double* __restrict__ JF0,
                                           const double* __restrict__ JF1, double* acc) {
  static_assert(32 % RD == 0, "rows of an observation share a warp");
  constexpr int OPW = 32 / RD;
  const int sub = lane / RD, rr = lane % RD;
#pragma unroll
  for (int k = 0; k < NV_F; ++k) acc[k] = 0.0;
#pragma unroll 2
  for (int64_t idx = begin + sub; idx < end; idx += OPW) {
    const int32_t ent = fobs[idx];
    const int64_t o = ent >> 1;
    double row[6];
    load_row6(((ent & 1) ? JF1 : JF0) + ((int64_t)RD * o + rr) * 6, row);
    const double rv = RES[(int64_t)RD * o + rr];
    int q = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
      for (int b = a; b < 6; ++b) { acc[q] = fma(row[a], row[b], acc[q]); ++q; }
#pragma unroll
    for (int a = 0; a < 6; ++a) acc[21 + a] = fma(row[a], rv, acc[21 + a]);
  }
}
template <int RD>
__global__ void __launch_bounds__(128)
k_fobs_partial(int nchunks, int ch, const int32_t* __restrict__ chunk_seg, const int64_t* __restrict__ chunk_begin,
               const int64_t* __restrict__ fobs_ptr, const int32_t* __restrict__ fobs, const double* __restrict__ RES,
               const double* __restrict__ JF0, const double* __restrict__ JF1, double* __restrict__ partial) {
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= nchunks) return;
  const int64_t begin = chunk_begin[c];
  const int64_t end = min(begin + ch, fobs_ptr[chunk_seg[c] + 1]);
  double acc[NV_F];
  d_fobs_seg<RD>(lane, begin, end, fobs, RES, JF0, JF1, acc);
  group_sum_store<NV_F, 32>(acc, lane, partial + (int64_t)c * NV_F, true);
}

// out[seg][NV] = sum of the chunk partials of the segment, fixed order.  One warp per segment.
template <int NV>
__global__ void __launch_bounds__(128)
k_seg_final(int nseg, const int32_t* __restrict__ seg_first, const double* __restrict__ partial, double* __restrict__ out) {
  const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (s >= nseg) return;
  const int c0 = seg_first[s], c1 = seg_first[s + 1];
  for (int v = 0; v < NV; ++v) {
    double a = 0.0;
    for (int c = c0 + lane; c < c1; c += 32) a += partial[(int64_t)c * NV + v];
    a = warp_sum(a);
    if (lane == 0) out[(int64_t)s * NV + v] = a;
  }
}

// E^T E (packed upper) and E^T r per eliminated block; G lanes cooperate on one block.
template <int RD, int DE, int G>
__device__ __forceinline__ void d_e_M(int64_t t, int64_t ne, const int64_t* __restrict__ e_ptr, const double* __restrict__ RES,
                                      const double* __restrict__ JE, double* __restrict__ ME) {   // whole warps call this
  constexpr int NU = DE * (DE + 1) / 2, NV = NU + DE;
  const int64_t e = t / G;
  const int g = (int)(t % G);
  const bool live = e < ne;
  double acc[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) acc[k] = 0.0;
  if constexpr (G >= RD && G % RD == 0 && DE == 6) {
    // a lane owns one residual row; G / RD observations per step, rows read side by side
    const int sub = g / RD, rr = g % RD;
    if (live) {
#pragma unroll 2
      for (int64_t o = e_ptr[e] + sub; o < e_ptr[e + 1]; o += G / RD) {
        double row[6];
        load_row6(JE + ((int64_t)RD * o + rr) * 6, row);
        const double rv = RES[(int64_t)RD * o + rr];
        int q = 0;
#pragma unroll
        for (int a = 0; a < 6; ++a)
#pragma unroll
          for (int b = a; b < 6; ++b) { acc[q] = fma(row[a], row[b], acc[q]); ++q; }
#pragma unroll
        for (int a = 0; a < 6; ++a) acc[NU + a] = fma(row[a], rv, acc[NU + a]);
      }
    }
  } else
  if (live) {
    for (int64_t o = e_ptr[e] + g; o < e_ptr[e + 1]; o += G) {
      const double* J = JE + (int64_t)RD * DE * o;
      const double* r = RES + (int64_t)RD * o;
#pragma unroll
      for (int rr = 0; rr < RD; ++rr) {
        double row[DE];
#pragma unroll
        for (int k = 0; k < DE; ++k) row[k] = J[rr * DE + k];
        const double rv = r[rr];
        int q = 0;
#pragma unroll
        for (int a = 0; a < DE; ++a)
#pragma unroll
          for (int b = a; b < DE; ++b) acc[q++] += row[a] * row[b];
#pragma unroll
        for (int a = 0; a < DE; ++a) acc[NU + a] += row[a] * rv;
      }
    }
  }
  group_sum_store<NV, G>(acc, g, ME + (live ? e : 0) * NV, live);
}
template <int RD, int DE, int G>
__global__ void __launch_bounds__(128)
k_e_M(int64_t ne, const int64_t* __restrict__ e_ptr, const double* __restrict__ RES, const double* __restrict__ JE,
      double* __restrict__ ME) {
  d_e_M<RD, DE, G>(blockIdx.x * (int64_t)blockDim.x + threadIdx.x, ne, e_ptr, RES, JE, ME);
}

// Model B: W_i^T = sum over the observations of incidence i of JE^T JF  (6 x 6, k-major).  RD lanes per incidence, a lane
// owns one residual row: the group walks the incidence's observations one at a time and reads both 384-byte records whole.
template <int RD>
__device__ __forceinline__ void d_inc_W(int64_t t, int64_t ninc, const int64_t* __restrict__ incobs_ptr, const int32_t* __restrict__ incobs,
                                        const double* __restrict__ JE, const double* __restrict__ JF0,
                                        const double* __restrict__ JF1, double* __restrict__ Wt) {   // whole warps call this
  static_assert(32 % RD == 0, "one lane per residual row, a group inside a warp");   // used for Model B only (RD = 8)
  constexpr int G = RD;
  const int64_t i = t / G;
  const int g = (int)(t % G);
  const bool live = i < ninc;
  double acc[36];
#pragma unroll
  for (int k = 0; k < 36; ++k) acc[k] = 0.0;
  if (live) {
    const int64_t q1 = incobs_ptr[i + 1];
#pragma unroll 2
    for (int64_t q = incobs_ptr[i]; q < q1; ++q) {
      const int32_t ent = incobs[q];
      const int64_t row = (int64_t)RD * (ent >> 1) + g;
      double re[6], rf[6];
      load_row6(JE + row * 6, re);
      load_row6(((ent & 1) ? JF1 : JF0) + row * 6, rf);
#pragma unroll
      for (int k = 0; k < 6; ++k)
#pragma unroll
        for (int a = 0; a < 6; ++a) acc[k * 6 + a] = fma(re[k], rf[a], acc[k * 6 + a]);
    }
  }
  group_sum_store<36, G>(acc, g, Wt + (live ? i : 0) * 36, live);
}
template <int RD>
__global__ void __launch_bounds__(128)
k_inc_W(int64_t ninc, const int64_t* __restrict__ incobs_ptr, const int32_t* __restrict__ incobs, const double* __restrict__ JE,
        const double* __restrict__ JF0, const double* __restrict__ JF1, double* __restrict__ Wt) {
  d_inc_W<RD>(blockIdx.x * (int64_t)blockDim.x + threadIdx.x, ninc, incobs_ptr, incobs, JE, JF0, JF1, Wt);
}

// (E^T E + D_e^2) = L L^T and z = L^-1 E^T r per eliminated block.  D_e = sqrt(clamp(diag)/radius)
// (LevenbergMarquardtStrategy::ComputeStep).  status bit 0 is raised when a block is not PD.
template <int DE>
__device__ __forceinline__ void d_e_chol(int64_t e, const double* __restrict__ ME, double radius, double min_diag, double max_diag,
                                         double* __restrict__ Lb, double* __restrict__ zb, int* status) {
  constexpr int NU = DE * (DE + 1) / 2, NV = NU + DE;
  double M[DE * DE], g[DE];
  int q = 0;
#pragma unroll
  for (int a = 0; a < DE; ++a)
#pragma unroll
    for (int b = a; b < DE; ++b) { const double v = ME[e * NV + q++]; M[a * DE + b] = v; M[b * DE + a] = v; }
#pragma unroll
  for (int a = 0; a < DE; ++a) {
    g[a] = ME[e * NV + NU + a];
    const double d = sqrt(fmin(fmax(M[a * DE + a], min_diag), max_diag) / radius);
    M[a * DE + a] += d * d;
  }
  if (!chol_small<DE>(M)) {
    atomicOr(status, 1);
#pragma unroll
    for (int k = 0; k < DE * DE; ++k) M[k] = (k % (DE + 1) == 0) ? 1.0 : 0.0;
  }
  fwd_small<DE>(M, g);
#pragma unroll
  for (int k = 0; k < DE * DE; ++k) Lb[e * DE * DE + k] = M[k];
#pragma unroll
  for (int k = 0; k < DE; ++k) zb[e * DE + k] = g[k];
}
template <int DE>
__global__ void __launch_bounds__(256)
k_e_chol(int64_t ne, const double* __restrict__ ME, const double* __restrict__ radius_p, double min_diag, double max_diag,
         double* __restrict__ Lb, double* __restrict__ zb, int* status) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e < ne) d_e_chol<DE>(e, ME, *radius_p, min_diag, max_diag, Lb, zb, status);
}

// Yt_i = L^-1 W_i^T (DE x 6, k-major) and v_i = Yt_i^T z per incidence.  FROM_J: the incidence is a single
// observation (Model A) and W_i^T = JE^T JF0 is formed on the fly.
template <int RD, int DE, bool FROM_J>
__device__ __forceinline__ void d_inc_Y(int64_t i, const int32_t* __restrict__ inc_e, const double* __restrict__ JE,
                                        const double* __restrict__ JF0, const double* __restrict__ Wt, const double* __restrict__ Lb,
                                        const double* __restrict__ zb, double* __restrict__ Yt, double* __restrict__ vb) {
  const int64_t e = inc_e[i];
  double W[DE * 6];
  if (FROM_J) {
#pragma unroll
    for (int k = 0; k < DE * 6; ++k) W[k] = 0.0;
#pragma unroll
    for (int rr = 0; rr < RD; ++rr) {
      double re[DE], rf[6];
#pragma unroll
      for (int k = 0; k < DE; ++k) re[k] = JE[(int64_t)RD * DE * i + rr * DE + k];
#pragma unroll
      for (int a = 0; a < 6; ++a) rf[a] = JF0[(int64_t)RD * 6 * i + rr * 6 + a];
#pragma unroll
      for (int k = 0; k < DE; ++k)
#pragma unroll
        for (int a = 0; a < 6; ++a) W[k * 6 + a] += re[k] * rf[a];
    }
  } else {
#pragma unroll
    for (int k = 0; k < DE * 6; ++k) W[k] = Wt[i * DE * 6 + k];
  }
  double v[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
  for (int k = 0; k < DE; ++k) {
    const double inv = 1.0 / Lb[e * DE * DE + k * DE + k];
    const double zk = zb[e * DE + k];
#pragma unroll
    for (int a = 0; a < 6; ++a) {
      double s = W[k * 6 + a];
#pragma unroll
      for (int m = 0; m < DE; ++m)
        if (m < k) s -= Lb[e * DE * DE + k * DE + m] * W[m * 6 + a];
      s *= inv;
      W[k * 6 + a] = s;
      v[a] += s * zk;
    }
  }
  double2* py = reinterpret_cast<double2*>(Yt + i * DE * 6);
#pragma unroll
  for (int k = 0; k < DE * 3; ++k) py[k] = make_double2(W[2 * k], W[2 * k + 1]);
  double2* pv = reinterpret_cast<double2*>(vb + i * 6);
#pragma unroll
  for (int k = 0; k < 3; ++k) pv[k] = make_double2(v[2 * k], v[2 * k + 1]);
}
template <int RD, int DE, bool FROM_J>
__global__ void __launch_bounds__(128)
k_inc_Y(int64_t ninc, const int32_t* __restrict__ inc_e, const double* __restrict__ JE, const double* __restrict__ JF0,
        const double* __restrict__ Wt, const double* __restrict__ Lb, const double* __restrict__ zb, double* __restrict__ Yt,
        double* __restrict__ vb) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < ninc) d_inc_Y<RD, DE, FROM_J>(i, inc_e, JE, JF0, Wt, Lb, zb, Yt, vb);
}

// sum of v_i over the incidences of one f-block, chunk partials (6 values).
__device__ __forceinline__ void d_finc_seg(int lane, int64_t begin, int64_t end, const int32_t* __restrict__ finc,
                                           const double* __restrict__ vb, double* acc) {
#pragma unroll
  for (int k = 0; k < 6; ++k) acc[k] = 0.0;
  for (int64_t idx = begin + lane; idx < end; idx += 32) {
    const double2* p = reinterpret_cast<const double2*>(vb + 6 * (int64_t)finc[idx]);
#pragma unroll
    for (int k = 0; k < 3; ++k) { const double2 v = p[k]; acc[2 * k] += v.x; acc[2 * k + 1] += v.y; }
  }
}
__global__ void __launch_bounds__(128)
k_finc_partial(int nchunks, int ch, const int32_t* __restrict__ chunk_seg, const int64_t* __restrict__ chunk_begin,
               const int64_t* __restrict__ finc_ptr, const int32_t* __restrict__ finc, const double* __restrict__ vb,
               double* __restrict__ partial) {
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= nchunks) return;
  const int64_t begin = chunk_begin[c];
  const int64_t end = min(begin + ch, finc_ptr[chunk_seg[c] + 1]);
  double acc[6];
  d_finc_seg(lane, begin, end, finc, vb, acc);
  group_sum_store<6, 32>(acc, lane, partial + (int64_t)c * 6, true);
}

// sum over incidence pairs (i,j) of Y_i Y_j^T = Yt_i^T Yt_j for one destination block, chunk partials (36 values).
// One warp per chunk; a lane owns one row k of the two Yt records of a pair (groups of 8 lanes, or 4 when DE <= 4).
template <int DE>
__device__ __forceinline__ void d_pairs_seg(int lane, int64_t begin, int64_t end, const int2* __restrict__ pairs,
                                            const double* __restrict__ Yt, double* acc) {
  constexpr int G = DE <= 4 ? 4 : 8;
  static_assert(DE <= G, "one lane per row of Yt");
  const int sub = lane / G, k = lane % G;
#pragma unroll
  for (int q = 0; q < 36; ++q) acc[q] = 0.0;
  if (k < DE) {
#pragma unroll 2
    for (int64_t idx = begin + sub; idx < end; idx += 32 / G) {
      const int2 pr = pairs[idx];
      if (pr.x < 0) continue;
      double yi[6], yj[6];
      load_row6(Yt + ((int64_t)DE * pr.x + k) * 6, yi);
      load_row6(Yt + ((int64_t)DE * pr.y + k) * 6, yj);
#pragma unroll
      for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int b = 0; b < 6; ++b) acc[a * 6 + b] = fma(yi[a], yj[b], acc[a * 6 + b]);
    }
  }
}
template <int DE>
__global__ void __launch_bounds__(128)
k_pairs_partial(int nchunks, int ch, const int32_t* __restrict__ chunk_seg, const int64_t* __restrict__ chunk_begin,
                const int64_t* __restrict__ dpair_ptr, const int2* __restrict__ pairs, const double* __restrict__ Yt,
                double* __restrict__ partial) {
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= nchunks) return;
  const int64_t begin = chunk_begin[c];
  const int64_t end = min(begin + ch, dpair_ptr[chunk_seg[c] + 1]);
  double acc[36];
  d_pairs_seg<DE>(lane, begin, end, pairs, Yt, acc);
  group_sum_store<36, 32>(acc, lane, partial + (int64_t)c * 36, true);
}

// Model B: sum over observations with (f0,f1) == (fa,fb) of JF0^T JF1, chunk partials (36 values).  One warp per chunk,
// a lane owns one residual row of one observation.
template <int RD>
__device__ __forceinline__ void d_dobs_seg(int lane, int64_t begin, int64_t end, const int32_t* __restrict__ dobs,
                                           const double* __restrict__ JF0, const double* __restrict__ JF1, double* acc) {
  static_assert(32 % RD == 0, "rows of an observation share a warp");
  constexpr int OPW = 32 / RD;
  const int sub = lane / RD, rr = lane % RD;
#pragma unroll
  for (int k = 0; k < 36; ++k) acc[k] = 0.0;
#pragma unroll 2
  for (int64_t idx = begin + sub; idx < end; idx += OPW) {
    const int64_t row = (int64_t)RD * dobs[idx] + rr;
    double ra[6], rb[6];
    load_row6(JF0 + row * 6, ra);
    load_row6(JF1 + row * 6, rb);
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
      for (int b = 0; b < 6; ++b) acc[a * 6 + b] = fma(ra[a], rb[b], acc[a * 6 + b]);
  }
}
template <int RD>
__global__ void __launch_bounds__(128)
k_dobs_partial(int nchunks, int ch, const int32_t* __restrict__ chunk_seg, const int64_t* __restrict__ chunk_begin,
               const int64_t* __restrict__ dobs_ptr, const int32_t* __restrict__ dobs, const double* __restrict__ JF0,
               const double* __restrict__ JF1, double* __restrict__ partial) {
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= nchunks) return;
  const int64_t begin = chunk_begin[c];
  const int64_t end = min(begin + ch, dobs_ptr[chunk_seg[c] + 1]);
  double acc[36];
  d_dobs_seg<RD>(lane, begin, end, dobs, JF0, JF1, acc);
  group_sum_store<36, 32>(acc, lane, partial + (int64_t)c * 36, true);
}

// Dense RCS: S[fa,fb] = Q - P (and its transpose).  One thread per (dest, entry).
__device__ __forceinline__ void d_assemble_dense(int64_t t, const int32_t* __restrict__ dest_fa, const int32_t* __restrict__ dest_fb,
                                                 const double* __restrict__ P, const double* __restrict__ Q, int64_t n /* row stride */,
                                                 double* __restrict__ S) {
  const int d = (int)(t / 36), q = (int)(t % 36), a = q / 6, b = q % 6;
  const int64_t fa = dest_fa[d], fb = dest_fb[d];
  const double v = (Q ? Q[t] : 0.0) - P[t];
  S[(6 * fa + a) * n + 6 * fb + b] = v;
  if (fa != fb) S[(6 * fb + b) * n + 6 * fa + a] = v;
}
__global__ void k_assemble_dense(int ndest, const int32_t* __restrict__ dest_fa, const int32_t* __restrict__ dest_fb,
                                 const double* __restrict__ P, const double* __restrict__ Q, int64_t n, double* __restrict__ S) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t < (int64_t)ndest * 36) d_assemble_dense(t, dest_fa, dest_fb, P, Q, n, S);
}

// After the (optional) cross-GPU sum: add F^T F diagonal blocks and the LM diagonal D_f^2, form the rhs.  DOFF as in
// k_diag_rhs_bsr (ba_rcs.cuh).
template <int DOFF = -1>
__device__ __forceinline__ void d_diag_rhs_dense(int64_t t, const double* __restrict__ HG, int hg_stride, const double* __restrict__ vsum,
                                                 int v_stride, const double* __restrict__ radius_p, double min_diag, double max_diag,
                                                 int64_t n /* row stride */, double* __restrict__ S, double* __restrict__ rhs) {
  const int64_t f = t / 6;
  const int a = (int)(t % 6);
  const double* H = HG + f * hg_stride;
#pragma unroll
  for (int b = 0; b < 6; ++b) {
    double h = H[a <= b ? sym_idx6(a, b) : sym_idx6(b, a)];
    if (a == b) { const double d = sqrt(fmin(fmax(DOFF < 0 ? h : H[DOFF + a], min_diag), max_diag) / *radius_p); h += d * d; }
    S[(6 * f + a) * n + 6 * f + b] += h;
  }
  rhs[t] = H[21 + a] - vsum[f * v_stride + a];
}
template <int DOFF = -1>
__global__ void k_diag_rhs_dense(int64_t nf, const double* __restrict__ HG, int hg_stride, const double* __restrict__ vsum,
                                 int v_stride, const double* __restrict__ radius_p, double min_diag, double max_diag, int64_t n,
                                 double* __restrict__ S, double* __restrict__ rhs) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t < nf * 6) d_diag_rhs_dense<DOFF>(t, HG, hg_stride, vsum, v_stride, radius_p, min_diag, max_diag, n, S, rhs);
}

// ---------------------------------------------------------------------------------------
// K4
// ---------------------------------------------------------------------------------------
// y_e = L^-T (z - sum_i Yt_i y_f(i)); G lanes per eliminated block.
template <int DE, int G>
__device__ __forceinline__ void d_e_backsub(int64_t t, int64_t ne, const int64_t* __restrict__ einc_ptr, const int32_t* __restrict__ inc_f,
                                            const double* __restrict__ Yt, const double* __restrict__ Lb, const double* __restrict__ zb,
                                            const double* __restrict__ yf, double* __restrict__ ye) {   // whole warps call this
  const int64_t e = t / G;
  const int g = (int)(t % G);
  const bool live = e < ne;
  double acc[DE];
#pragma unroll
  for (int k = 0; k < DE; ++k) acc[k] = 0.0;
  if (live) {
    for (int64_t i = einc_ptr[e] + g; i < einc_ptr[e + 1]; i += G) {
      const double* y = yf + 6 * (int64_t)inc_f[i];
      const double* Y = Yt + i * DE * 6;
#pragma unroll
      for (int k = 0; k < DE; ++k) {
        double s = 0.0;
#pragma unroll
        for (int a = 0; a < 6; ++a) s += Y[k * 6 + a] * y[a];
        acc[k] += s;
      }
    }
  }
  if (G > 1) {
#pragma unroll
    for (int k = 0; k < DE; ++k)
#pragma unroll
      for (int off = G / 2; off > 0; off >>= 1) acc[k] += __shfl_down_sync(0xffffffffu, acc[k], off, G);
  }
  if (live && g == 0) {
    double L[DE * DE], x[DE];
#pragma unroll
    for (int k = 0; k < DE * DE; ++k) L[k] = Lb[e * DE * DE + k];
#pragma unroll
    for (int k = 0; k < DE; ++k) x[k] = zb[e * DE + k] - acc[k];
    bwd_small<DE>(L, x);
#pragma unroll
    for (int k = 0; k < DE; ++k) ye[e * DE + k] = x[k];
  }
}
template <int DE, int G>
__global__ void __launch_bounds__(128)
k_e_backsub(int64_t ne, const int64_t* __restrict__ einc_ptr, const int32_t* __restrict__ inc_f, const double* __restrict__ Yt,
            const double* __restrict__ Lb, const double* __restrict__ zb, const double* __restrict__ yf, double* __restrict__ ye) {
  d_e_backsub<DE, G>(blockIdx.x * (int64_t)blockDim.x + threadIdx.x, ne, einc_ptr, inc_f, Yt, Lb, zb, yf, ye);
}

// model_cost_change partials: with step = -y,  sum_o (J step) . (r + J step / 2)   (the caller negates).
// One thread per residual row: consecutive lanes read consecutive rows of JE / JF0 / JF1.
template <int RD, int DE, int NSLOT>
__device__ __forceinline__ double d_model_cost_row(int64_t row, const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f0,
                                                   const int32_t* __restrict__ ob_f1, const double* __restrict__ RES,
                                                   const double* __restrict__ JE, const double* __restrict__ JF0,
                                                   const double* __restrict__ JF1, const double* __restrict__ ye,
                                                   const double* __restrict__ yf) {
  const int64_t o = row / RD;
  {
    const int64_t e = ob_e[o];
    const int32_t f0 = ob_f0[o];
    const int32_t f1 = NSLOT == 2 ? ob_f1[o] : -1;
    double m = 0.0;
#pragma unroll
    for (int k = 0; k < DE; ++k) m = fma(JE[row * DE + k], -ye[e * DE + k], m);
    if (f0 >= 0) {
      double j[6];
      load_row6(JF0 + row * 6, j);
#pragma unroll
      for (int k = 0; k < 6; ++k) m = fma(j[k], -yf[6 * (int64_t)f0 + k], m);
    }
    if (NSLOT == 2 && f1 >= 0) {
      double j[6];
      load_row6(JF1 + row * 6, j);
#pragma unroll
      for (int k = 0; k < 6; ++k) m = fma(j[k], -yf[6 * (int64_t)f1 + k], m);
    }
    return m * (RES[row] + m / 2.0);
  }
}
template <int RD, int DE, int NSLOT>
__global__ void __launch_bounds__(256)
k_model_cost(int64_t nb, const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f0, const int32_t* __restrict__ ob_f1,
             const double* __restrict__ RES, const double* __restrict__ JE, const double* __restrict__ JF0,
             const double* __restrict__ JF1, const double* __restrict__ ye, const double* __restrict__ yf,
             double* __restrict__ partial) {
  __shared__ double sm[32];
  const int64_t row = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  double acc = row / RD < nb ? d_model_cost_row<RD, DE, NSLOT>(row, ob_e, ob_f0, ob_f1, RES, JE, JF0, JF1, ye, yf) : 0.0;
  acc = block_sum(acc, sm);
  if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}

// candidate = x - s .* y over blocks of width W; partial sums of x^2 and (x - candidate)^2 over active blocks.
template <int W>
__device__ __forceinline__ void d_candidate(int64_t t, const int64_t* __restrict__ ptr, const double* __restrict__ x,
                                            const double* __restrict__ s, const double* __restrict__ y, double* __restrict__ xc,
                                            double& x2, double& d2) {
  const int64_t b = t / W;
  const double xv = x[t];
  const double c = xv + (-(y[t]) * s[t]);
  xc[t] = c;
  if (ptr[b + 1] > ptr[b]) { x2 = xv * xv; const double d = xv - c; d2 = d * d; }
}
template <int W>
__global__ void __launch_bounds__(256)
k_candidate(int64_t nblk, const int64_t* __restrict__ ptr /*block is active iff ptr[b+1] > ptr[b]*/, const double* __restrict__ x,
            const double* __restrict__ s, const double* __restrict__ y, double* __restrict__ xc, double* __restrict__ p_x2,
            double* __restrict__ p_d2) {
  __shared__ double sm[32];
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  double x2 = 0.0, d2 = 0.0;
  if (t < nblk * W) d_candidate<W>(t, ptr, x, s, y, xc, x2, d2);
  x2 = block_sum(x2, sm);
  d2 = block_sum(d2, sm);
  if (threadIdx.x == 0) { p_x2[blockIdx.x] = x2; p_d2[blockIdx.x] = d2; }
}

// |x - Plus(x, -g)| max and squared-sum partials (TrustRegionMinimizer::EvaluateGradientAndJacobian);
// g (unscaled) = g_scaled / s.  src holds per block NVB values with the gradient at offset GOFF.
template <int W, int NVB, int GOFF>
__device__ __forceinline__ void d_gradient_norm(int64_t t, const int64_t* __restrict__ ptr, const double* __restrict__ x,
                                                const double* __restrict__ s, const double* __restrict__ src, double& mx, double& sq) {
  const int64_t b = t / W;
  const int k = (int)(t % W);
  if (ptr[b + 1] > ptr[b]) {
    const double g = src[b * NVB + GOFF + k] / s[t];
    const double xv = x[t];
    const double d = xv - (xv + (-g));
    mx = fabs(d); sq = d * d;
  }
}
template <int W, int NVB, int GOFF>
__global__ void __launch_bounds__(256)
k_gradient_norm(int64_t nblk, const int64_t* __restrict__ ptr, const double* __restrict__ x, const double* __restrict__ s,
                const double* __restrict__ src, double* __restrict__ p_max, double* __restrict__ p_sq) {
  __shared__ double sm[32];
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  double mx = 0.0, sq = 0.0;
  if (t < nblk * W) d_gradient_norm<W, NVB, GOFF>(t, ptr, x, s, src, mx, sq);
  mx = block_max(mx, sm);
  sq = block_sum(sq, sm);
  if (threadIdx.x == 0) { p_max[blockIdx.x] = mx; p_sq[blockIdx.x] = sq; }
}

// Jacobi scaling s = 1 / (1 + sqrt(|column|^2)) from the packed normal-equation diagonals (iteration 0 only), or, DOFF >= 0,
// from the W column norms stored at src[DOFF..] of each block.
template <int W, int NVB, int DOFF = -1>
__device__ __forceinline__ void d_jacobi_scale(int64_t t, const double* __restrict__ src, double* __restrict__ s) {
  const int64_t b = t / W;
  const int k = (int)(t % W);
  const int di = DOFF < 0 ? k * W - k * (k - 1) / 2 : DOFF + k;  // packed index of (k,k), or a separate diagonal
  s[t] = 1.0 / (1.0 + sqrt(src[b * NVB + di]));
}
template <int W, int NVB, int DOFF = -1>
__global__ void k_jacobi_scale(int64_t nblk, const double* __restrict__ src, double* __restrict__ s) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t < nblk * W) d_jacobi_scale<W, NVB, DOFF>(t, src, s);
}

__global__ void k_fill(double* a, int64_t n, double v) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) a[i] = v;
}

}  // namespace ba
