// ba_rig_loop.cuh -- the body of the one-CTA rig kernels (ba_rig.cuh: k_rig_lm, k_rig_lm_batch): the whole trust-region loop
// of ceres::Solve on `const RigParams& P`, template parameters RD, DE, GE, NSLOT.  Included inside a kernel body only.
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
