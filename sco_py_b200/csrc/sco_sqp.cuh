// sco_sqp.cuh -- per-problem penalty-SQP state machine, run by the team that owns the problem.
//
// Replaces Solver._penalty_sqp / _min_merit_fn and its predicates
// (sco_py/sco_osqp/solver.py:62-283), Prob.find_closest_feasible_point (prob.py:369-412),
// Prob.update_obj's penalty bookkeeping (prob.py:414-426, quirks C-1..C-3 of SURVEY.md
// Appendix C), Prob.get_value / get_approx_value / get_max_cnt_violation (prob.py:547-630),
// Prob.add_trust_region / save / restore (prob.py:514-519,639-652; variable.py:37-73).
// Every scalar decision is taken on team-uniform values, so control flow never diverges
// inside a team; different problems (teams) follow different paths freely.
#pragma once
#include "sco_device.cuh"
#include "sco_families.cuh"
#include "sco_qp.cuh"

struct SqpOut {
  int verdict;
  double merit, objective, max_vio;
  int sqp_iters, qp_solves, admm_iters, last_status;
  int nonconv;  // prob.nonconverged_groups of the last evaluation of solver.py:206-235 (bit g / bit 16+g)
#ifdef SCO_TIMING
  long long cyc_total, cyc_setup, cyc_loop, cyc_check, cyc_cvx;  // clock64() ticks per phase
#endif
};

template <int TEAM, int DK>
struct SqpSolver {
  const DevStruct &S;
  const DevSettings &st;
  QPW &w;
  const double *prm;
  Sh xc;        // current iterate (shared memory)
  double *Jg;   // unscaled Jacobian entries of the last convexification (global scratch)
  const int tid, n, m_nl, ng;
  // work queue of the launch (k_solve): once it is drained the remaining problems decide when the launch ends
  const unsigned long long *queue = nullptr;
  long long queue_len = 0;

  __device__ SqpSolver(const DevStruct &S_, const DevSettings &st_, QPW &w_, const double *prm_,
                       double *Jg_)
      : S(S_), st(st_), w(w_), prm(prm_), xc(w_.xc), Jg(Jg_), tid(threadIdx.x), n(S_.n),
        m_nl(S_.m_nl), ng(S_.m_nl ? S_.n_groups : 0) {}

  __device__ __forceinline__ void sync() { Team<TEAM>::sync(); }

  // quadratic part of the objective at xc: 0.5 x'Qx + q'x + c (QuadExpr.eval, expr.py:205-206)
  __device__ double objective_quad() {
    const double *Qg = field_ptr(S, S.Q, prm), *qg = field_ptr(S, S.q, prm), *cg = field_ptr(S, S.c, prm);
    const double *qag = field_ptr(S, S.qa, prm);  // AffExpr objective terms: exact value a'x (expr.py:173-174)
    double v[1] = {0.0};
    for (int k = tid; k < n; k += TEAM) {
      double acc = 0.0;
      if (Qg)
        for (int j = 0; j < n; j++) acc += Qg[j * n + k] * xc[j];
      v[0] += xc[k] * (0.5 * acc + (qg ? qg[k] : 0.0) + (qag ? qag[k] : 0.0));
    }
    Team<TEAM>::reduce_sum(v, w.red);
    return v[0] + (cg ? cg[0] : 0.0);
  }

  // term t of the objective blocks: its block and row
  __device__ __forceinline__ const DevObjBlock &obj_term(int t, int &r) const {
    int b = 0;
    while (b + 1 < S.n_ob && t >= S.ob[b + 1].t0) b++;
    r = t - S.ob[b].t0;
    return S.ob[b];
  }
  // term t's model in the term-model area (DevObjBlock)
  __device__ __forceinline__ Sh obj_model(const DevObjBlock &B, int r) const {
    return w.ot + (B.toff + r * (B.n_in * (B.n_in + 1) / 2 + B.n_in + 1));
  }
  // entry (i, j) of a term's packed upper triangle, i <= j
  static __device__ __forceinline__ int tri(int i, int j, int nn) { return i * nn - i * (i - 1) / 2 + (j - i); }

  // exact objective: quadratic terms + the non-quadratic terms, sum_t f_t (prob.py:573-574)
  __device__ double objective() {
    double v = objective_quad();
    if (S.n_ob) {
      double t[1] = {0.0};
      for (int k = tid; k < S.n_terms; k += TEAM) {
        int r;
        const DevObjBlock &B = obj_term(k, r);
        t[0] += vm_eval(field_ptr(S, B.prog, prm), B.m, r, xc, S.ob_cols + B.coff + r * B.n_in, -1, 0.0, -1, 0.0);
      }
      Team<TEAM>::reduce_sum(t, w.red);
      v += t[0];
    }
    return v;
  }

  // objective of the convex model: quadratic terms + the sum of the terms' degree-2 models at the last
  // convexification (prob.py:624-626), from the assembled model (w.Hv on the pattern of P, w.gq, w.oc)
  __device__ double objective_model() {
    double v = objective_quad();
    if (S.n_ob) {
      double t[1] = {0.0};
      for (int k = tid; k < n; k += TEAM) {
        double acc = 0.0;
        for (int p = __ldg(S.P_cptr + k); p < __ldg(S.P_cptr + k + 1); p++) acc += w.Hv[p] * xc[__ldg(S.P_row + p)];
        t[0] += xc[k] * (0.5 * acc + w.gq[k]);
      }
      Team<TEAM>::reduce_sum(t, w.red);
      v += t[0] + w.oc[0];
    }
    return v;
  }

  // Expr.convexify degree 2 of every non-quadratic objective term at xc, each on its own (expr.py:143-153):
  // H_t = numeric Hessian over the term's inputs shifted by -min(lambda_min, 0) I, A_t = grad - x'H_t,
  // b_t = 0.5 x'H_t x - grad.x + f_t.  Leaves the per-term models in w.ot, their sum on the pattern of P in w.Hv, its
  // linear term in w.gq and its constant (sum_t b_t) in w.oc.  Every sum runs in a fixed order (no atomics).
  __device__ void convexify_objective() {
    const int NT = S.n_terms;
    int nh = 0, ng_ = 0;  // Hessian entries (upper triangles) and gradient entries of all terms
    for (int b = 0; b < S.n_ob; b++) {
      nh += S.ob[b].m * (S.ob[b].n_in * (S.ob[b].n_in + 1) / 2);
      ng_ += S.ob[b].m * S.ob[b].n_in;
    }
    for (int k = tid; k < NT; k += TEAM) {
      int r;
      const DevObjBlock &B = obj_term(k, r);
      obj_model(B, r)[B.n_in * (B.n_in + 1) / 2 + B.n_in] =
          vm_eval(field_ptr(S, B.prog, prm), B.m, r, xc, S.ob_cols + B.coff + r * B.n_in, -1, 0.0, -1, 0.0);
    }
    sync();
    for (int e = tid; e < nh + ng_; e += TEAM) {
      int b = 0, q = e < nh ? e : e - nh;
      const bool hess = e < nh;
      for (;;) {  // the block of entry q
        const int cnt = S.ob[b].m * (hess ? S.ob[b].n_in * (S.ob[b].n_in + 1) / 2 : S.ob[b].n_in);
        if (q < cnt || b + 1 == S.n_ob) break;
        q -= cnt;
        b++;
      }
      const DevObjBlock &B = S.ob[b];
      const int nn = B.n_in, ntri = nn * (nn + 1) / 2;
      const int r = q / (hess ? ntri : nn);
      q -= r * (hess ? ntri : nn);
      const double *prog = field_ptr(S, B.prog, prm);
      const int *cols = S.ob_cols + B.coff + r * nn;
      const Sh h = obj_model(B, r);
      if (hess) {
        int i = 0;
        while (q >= nn - i) { q -= nn - i; i++; }
        h[tri(i, i + q, nn)] = vm_fd2(prog, B.m, r, xc, cols, i, i + q, h[ntri + nn]);
      } else if (B.flags & 1) {  // gradient: the program's own derivative, or finite differences
        double d;
        vm_eval_dual(prog, B.m, r, xc, cols, q, &d);
        h[ntri + q] = d;
      } else {
        h[ntri + q] = vm_fd1(prog, B.m, r, xc, cols, q);
      }
    }
    sync();
    {
      // smallest eigenvalue of every H_t: cyclic Jacobi on a scratch copy, one warp per term.  The rotations come in the
      // serial (p, q) order and every element is computed by the formula of a one-thread sweep; the lanes only share the
      // elements of the two columns, then of the two rows, a rotation touches.
      const int wid = tid >> 5, lane = tid & 31;
      if (wid < S.nwj) {
        const Sh A = w.jac + wid * S.n_in_max * S.n_in_max;
        for (int k = wid; k < NT; k += S.nwj) {
          int r;
          const DevObjBlock &B = obj_term(k, r);
          const int nn = B.n_in;
          const Sh h = obj_model(B, r);
          for (int e = lane; e < nn * nn; e += 32) {
            const int i = e / nn, j = e % nn;
            A[e] = h[i <= j ? tri(i, j, nn) : tri(j, i, nn)];
          }
          __syncwarp();
          for (int sweep = 0; sweep < 50; sweep++) {
            double off = 0.0, dg = 0.0;
            for (int p = lane; p < nn; p += 32)
              for (int q = 0; q < nn; q++) (p == q ? dg : off) += A[p * nn + q] * A[p * nn + q];
            off = warp_sum(off); dg = warp_sum(dg);
            if (off <= 1e-30 * dg || off == 0.0) break;
            for (int p = 0; p < nn - 1; p++)
              for (int q = p + 1; q < nn; q++) {
                const double apq = A[p * nn + q], app = A[p * nn + p], aqq = A[q * nn + q];
                __syncwarp();
                if (apq == 0.0) continue;
                const double theta = (aqq - app) / (2.0 * apq);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
                for (int k2 = lane; k2 < nn; k2 += 32) {  // columns p, q
                  const double akp = A[k2 * nn + p], akq = A[k2 * nn + q];
                  A[k2 * nn + p] = c * akp - sn * akq;
                  A[k2 * nn + q] = sn * akp + c * akq;
                }
                __syncwarp();
                for (int k2 = lane; k2 < nn; k2 += 32) {  // rows p, q
                  const double apk = A[p * nn + k2], aqk = A[q * nn + k2];
                  A[p * nn + k2] = c * apk - sn * aqk;
                  A[q * nn + k2] = sn * apk + c * aqk;
                }
                __syncwarp();
              }
          }
          double lam = A[0];
          for (int p = 1; p < nn; p++) lam = fmin(lam, A[p * nn + p]);
          if (lam < 0.0)
            for (int j = lane; j < nn; j += 32) h[tri(j, j, nn)] -= lam;
          __syncwarp();
        }
      }
    }
    sync();
    double t[1] = {0.0};
    for (int e = tid; e < ng_; e += TEAM) {
      int b = 0, q = e;
      while (b + 1 < S.n_ob && q >= S.ob[b].m * S.ob[b].n_in) { q -= S.ob[b].m * S.ob[b].n_in; b++; }
      const DevObjBlock &B = S.ob[b];
      const int nn = B.n_in, ntri = nn * (nn + 1) / 2, r = q / nn, k = q - r * nn;
      const int *cols = S.ob_cols + B.coff + r * nn;
      const Sh h = obj_model(B, r);
      double acc = 0.0;
      for (int j = 0; j < nn; j++) acc += h[j <= k ? tri(j, k, nn) : tri(k, j, nn)] * xc[__ldg(cols + j)];  // (x'H)_k
      const double g = h[ntri + k], xk = xc[__ldg(cols + k)];
      h[ntri + k] = g - acc;
      t[0] += xk * (0.5 * acc - g);
    }
    Team<TEAM>::reduce_sum(t, w.red);
    if (tid == 0) {
      double f = 0.0;
      for (int k = 0; k < NT; k++) {
        int r;
        const DevObjBlock &B = obj_term(k, r);
        const double fk = obj_model(B, r)[B.n_in * (B.n_in + 1) / 2 + B.n_in];
        f = k ? f + fk : fk;
      }
      w.oc[0] = t[0] + f;
    }
    // the model's sum on the pattern of P and on q: every entry from its list of term entries, in term order
    for (int p = tid; p < S.nnz_p; p += TEAM) {
      const int a0 = __ldg(S.hv_ptr + p), a1 = __ldg(S.hv_ptr + p + 1);
      double v = a0 < a1 ? w.ot[__ldg(S.hv_src + a0)] : 0.0;
      for (int a = a0 + 1; a < a1; a++) v += w.ot[__ldg(S.hv_src + a)];
      w.Hv[p] = v;
    }
    for (int j = tid; j < n; j += TEAM) {
      const int a0 = __ldg(S.gq_ptr + j), a1 = __ldg(S.gq_ptr + j + 1);
      double v = a0 < a1 ? w.ot[__ldg(S.gq_src + a0)] : 0.0;
      for (int a = a0 + 1; a < a1; a++) v += w.ot[__ldg(S.gq_src + a)];
      w.gq[j] = v;
    }
    sync();
  }

  // violations from w.fv (raw f at xc): out[0] = sum, out[1] = max, out[2+g] = group sums
  __device__ void violation_sums(double *out) {
    double v[1 + SCO_DEV_MAX_GROUPS], mx[1] = {0.0};
    for (int k = 0; k < 1 + SCO_DEV_MAX_GROUPS; k++) v[k] = 0.0;
    for (int bi = 0; bi < S.n_blocks; bi++) {
      const DevBlock &B = S.blocks[bi];
      const double *val = field_ptr(S, B.val, prm);
      for (int r = tid; r < B.m; r += TEAM) {
        const double d = w.fv[B.row0 + r] - (val ? val[r] : 0.0);
        const double vio = B.cnt_type ? fabs(d) : fmax(d, 0.0);  // prob.py:582-590
        v[0] += vio;
        mx[0] = fmax(mx[0], vio);
        for (int g = 0; g < ng; g++)
          if ((B.group_mask >> g) & 1) v[1 + g] += vio;
      }
    }
    Team<TEAM>::reduce_sum(v, w.red);
    Team<TEAM>::reduce_max(mx, w.red);
    out[0] = v[0];
    out[1] = mx[0];
    for (int g = 0; g < SCO_DEV_MAX_GROUPS; g++) out[2 + g] = v[1 + g];
  }

  // penalties of the affine models at xc (unmasked J, prob.py:624-630): out[0] = sum, out[2+g]
  __device__ void model_sums(double *out) {
    double v[1 + SCO_DEV_MAX_GROUPS];
    for (int k = 0; k < 1 + SCO_DEV_MAX_GROUPS; k++) v[k] = 0.0;
    for (int i = tid; i < m_nl; i += TEAM) {
      const int go = __ldg(S.row_goff + (i)), wd = __ldg(S.row_w + (i));
      double acc = w.bb[i];
      for (int k = 0; k < wd; k++) acc += Jg[go + k] * xc[__ldg(S.jcol_g + (go + k))];
      const double pen = __ldg(S.row_eq + (i)) ? fabs(acc) : fmax(acc, 0.0);
      v[0] += pen;
      const int gm = __ldg(S.row_gmask + (i));
      for (int g = 0; g < ng; g++)
        if ((gm >> g) & 1) v[1 + g] += pen;
    }
    Team<TEAM>::reduce_sum(v, w.red);
    out[0] = v[0];
    out[1] = 0.0;
    for (int g = 0; g < SCO_DEV_MAX_GROUPS; g++) out[2 + g] = v[1 + g];
  }

  // Prob.convexify at xc: fv, Jg, bb = f - J x - val ; first call freezes the sparsity masks
  __device__ void convexify(bool &mask_set) {
    if (S.n_ob) convexify_objective();
    eval_blocks<TEAM>(S, prm, xc, w.fv, Jg, w.stage);
    for (int bi = 0; bi < S.n_blocks; bi++) {
      const DevBlock &B = S.blocks[bi];
      const double *val = field_ptr(S, B.val, prm);
      for (int r = tid; r < B.m; r += TEAM) {
        const int i = B.row0 + r, go = __ldg(S.row_goff + (i)), wd = __ldg(S.row_w + (i));
        double acc = 0.0;
        uint32_t mk = 0;
        for (int k = 0; k < wd; k++) {
          const double jv = Jg[go + k];
          acc += jv * xc[__ldg(S.jcol_g + (go + k))];
          if (jv != 0.0) mk |= (1u << (k & 31));
          if ((k & 31) == 31 || k == wd - 1) {  // one 32-bit word of the row's mask is complete
            if (!mask_set) w.msk[i * S.mw + (k >> 5)] = st.freeze_sparsity ? mk : 0xffffffffu;
            mk = 0;
          }
        }
        w.bb[i] = -acc + w.fv[i] - (val ? val[r] : 0.0);
      }
    }
    mask_set = true;
    sync();
  }

  __device__ SqpOut run(const double *x0) {
    SqpOut o;
    o.verdict = 0; o.merit = 0; o.objective = 0; o.max_vio = 0;
    o.sqp_iters = 0; o.qp_solves = 0; o.admm_iters = 0; o.last_status = 0; o.nonconv = 0;
#ifdef SCO_TIMING
    o.cyc_setup = o.cyc_loop = o.cyc_check = o.cyc_cvx = 0;
    const long long t_run = clock64();
#endif
    for (int j = tid; j < n; j += TEAM) xc[j] = x0[j];
    sync();
    double mu = st.initial_penalty_coeff;
    double vs[2 + SCO_DEV_MAX_GROUPS], ms_[2 + SCO_DEV_MAX_GROUPS];
    bool finished = false;
    // ---- find_closest_feasible_point (prob.py:369-412): default OSQP settings (solver.py:81)
    {
      // bounds of the projection = whatever is on the scalar variables (osqp_utils.py:165-189): the user's
      const double *lb0 = field_ptr(S, S.lb0, prm), *ub0 = field_ptr(S, S.ub0, prm);
      for (int j = tid; j < n; j += TEAM) {
        w.xs[j] = xc[j];
        w.lb[j] = lb0 ? lb0[j] : -INFINITY;
        w.ub[j] = ub0 ? ub0[j] : INFINITY;
      }
      sync();
      QPArgs a;
      a.prm = prm; a.Jg = nullptr; a.pi = 0.0; a.kd = 0.0; a.wa = 0.0; a.use_pen = 0; a.closest = 1; a.has_hq = 0; a.tail = 0;
      a.warm = 0;
      DevSettings d = st;
      d.eps_abs = 1e-6; d.eps_rel = 1e-9; d.max_iter = 100000; d.rho = 0.1; d.sigma = 5e-10;
      d.adaptive_rho = 0;
      QPSolver<TEAM, DK> qp(S, d, w, a);
      QPResult r = qp.solve();
      o.qp_solves++; o.admm_iters += r.iters; o.last_status = r.status;
      if (r.status == 1 || r.status == 2) {
        for (int j = tid; j < n; j += TEAM) xc[j] = w.x[j];
        sync();
      } else {
        finished = true;  // solver.py:81-82 -> False
      }
    }
    double pi = 1.0, kd = 0.0;
    double wa = 0.0;  // weight of the AffExpr objective terms in the QP (quirk C-4)
    bool mask_set = false;
    if (!finished) {
      bool success = false;
      int verdict = 0;
      for (int inc = 0; inc < st.max_merit_coeff_increases && !finished; inc++) {
        // ---------------- _min_merit_fn(prob, mu, delta0) ----------------
        double delta = st.initial_trust_region_size;
        bool done_mm = false;
        success = false;
        while (!done_mm) {
          if (o.sqp_iters >= st.max_sqp_iters) { verdict = -1; finished = true; break; }
          o.sqp_iters++;
#ifdef SCO_TIMING
          const long long t_cvx = clock64();
#endif
          convexify(mask_set);
#ifdef SCO_TIMING
          o.cyc_cvx += clock64() - t_cvx;
#endif
          kd = st.duplicate_rows ? kd + 1.0 : 1.0;      // prob.py:508-509
          pi = st.compound_penalty ? pi * mu : mu;      // prob.py:424-426
          wa = st.aff_obj_quirk ? (wa + 1.0) * mu : 1.0;  // prob.py:220-221,240-249 then :424-426
          bool first_qp = true;  // of this convexification (warm start, sco_settings.warm_start)
          violation_sums(vs);
          const double merit = objective() + mu * vs[0];
          double mvec[SCO_DEV_MAX_GROUPS];
          for (int g = 0; g < SCO_DEV_MAX_GROUPS; g++) mvec[g] = vs[2 + g];
          for (int j = tid; j < n; j += TEAM) w.xs[j] = xc[j];  // prob.save()
          sync();
          while (true) {  // trust-region loop, solver.py:136-251
            for (int j = tid; j < n; j += TEAM) { w.lb[j] = w.xs[j] - delta; w.ub[j] = w.xs[j] + delta; }
            sync();
            QPArgs a;
            a.prm = prm; a.Jg = Jg; a.pi = pi; a.kd = kd; a.wa = wa; a.use_pen = 1; a.closest = 0; a.has_hq = S.n_ob != 0;
            // warm_start 1: QPs of one trust-region loop (same J, b, weights; only the box moves); 2: every penalty QP
            // after the problem's first one
            a.warm = (st.warm_start == 1 && !first_qp) || (st.warm_start >= 2 && o.qp_solves > 1) ? 1 : 0;
            first_qp = false;
            // one thread looks at the queue and the team agrees on the answer (a per-thread read could
            // split the team at the moment the queue runs dry)
            if (tid == 0)
              w.red[0] = (queue && *(const volatile unsigned long long *)queue >= (unsigned long long)queue_len) ? 1.0 : 0.0;
            sync();
            a.tail = w.red[0] != 0.0;
            sync();
            QPSolver<TEAM, DK> qp(S, st, w, a);
            QPResult r = qp.solve();
            o.qp_solves++; o.admm_iters += r.iters; o.last_status = r.status;
#ifdef SCO_TIMING
            o.cyc_setup += r.cyc_setup; o.cyc_loop += r.cyc_loop; o.cyc_check += r.cyc_check;
#endif
            if (r.status == 1 || r.status == 2) {  // prob.py:197-205
              for (int j = tid; j < n; j += TEAM) xc[j] = w.x[j];
              sync();
            }
            model_sums(ms_);
            const double obj_new = objective();
            const double model_merit = (S.n_ob ? objective_model() : obj_new) + mu * ms_[0];
            eval_blocks<TEAM>(S, prm, xc, w.fv, nullptr, w.stage);
            violation_sums(vs);
            const double new_merit = obj_new + mu * vs[0];
            double approx = merit - model_merit;
            if (approx == 0.0) approx += 1e-12;  // solver.py:151-153
            const double exact = merit - new_merit;
            const double ratio = exact / approx;
            bool restore = false, ret = false, retval = false;
            if (approx < -1e-5) { restore = true; ret = true; retval = false; }          // _bad_model
            else if (approx < st.min_approx_improve) { restore = true; ret = true; retval = true; }  // _y_converged
            else {
              int ma = 0, mb = 0;  // solver.py:209-235: first loop (with the overlap rule), second loop (without)
              for (int g = 0; g < ng; g++) {
                const double av = mvec[g] - ms_[2 + g];
                if (mvec[g] > st.cnt_tolerance && av < st.min_approx_improve) {
                  mb |= 1 << g;
                  bool ov = false;
                  for (int g2 = 0; g2 < ng; g2++)
                    if (g2 != g && ((S.overlap[g] >> g2) & 1) && (mvec[g2] - ms_[2 + g2]) > st.min_approx_improve)
                      ov = true;
                  if (!ov) ma |= 1 << g;
                }
              }
              o.nonconv = ma ? (ma | (mb << 16)) : 0;  // the reference clears the list at every evaluation
              if (ma) { restore = true; ret = true; retval = true; }
            }
            if (ret) {
              for (int j = tid; j < n; j += TEAM) xc[j] = w.xs[j];
              sync();
              success = retval;
              done_mm = true;
              break;
            }
            if (exact < 0.0 || ratio < st.improve_ratio_threshold) {  // _shrink_trust_region
              for (int j = tid; j < n; j += TEAM) xc[j] = w.xs[j];
              sync();
              delta *= st.trust_shrink_ratio;
            } else {
              delta *= st.trust_expand_ratio;
              break;  // next SQP iteration
            }
            if (delta < st.min_trust_region_size) {  // _x_converged
              success = true;
              done_mm = true;
              break;
            }
            (void)restore;
          }
        }
        if (finished) break;
        // ---------------- solver.py:94-101 ----------------
        eval_blocks<TEAM>(S, prm, xc, w.fv, nullptr, w.stage);
        violation_sums(vs);
        if (vs[1] > st.cnt_tolerance) {
          if (inc + 1 < st.max_merit_coeff_increases) mu *= st.merit_coeff_increase_ratio;
        } else {
          verdict = success ? 1 : 0;
          finished = true;
        }
      }
      o.verdict = verdict;  // falling out of the loop: solver.py:105 -> False
    }
    // final report at xc with the last penalty coefficient used
    eval_blocks<TEAM>(S, prm, xc, w.fv, nullptr, w.stage);
    violation_sums(vs);
    o.objective = objective();
    o.merit = o.objective + mu * vs[0];
    o.max_vio = vs[1];
#ifdef SCO_TIMING
    o.cyc_total = clock64() - t_run;
#endif
    return o;
  }
};
