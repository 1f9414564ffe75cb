// sco_qp.cuh -- the in-house batched OSQP-style ADMM QP solve, one QP per thread team,
// working set resident in shared memory.
//
// Replaces osqp.OSQP().setup()/solve() as driven by sco_py/sco_osqp/osqp_utils.py:195-216 for
// the penalty QP of SURVEY.md Appendix A:
//
//   min  0.5 x' Psym x + q'x + pi * 1's
//   s.t. A_lin x in [l_lin, u_lin]
//        (J.*M) x - s1 (+ s2) {<=, =} -b          (each row present `kd` times, quirk C-3)
//        lbx <= x <= ubx ,  s >= 0
//
// The iteration is the one of OSQP 0.6.2 (Ruiz equilibration + cost scaling, per-row rho,
// alpha-relaxed ADMM from x=z=y=0, termination tests every check_termination iterations on the
// unscaled residuals, SURVEY.md Appendix B) so that iterates agree with the CPU oracle to
// rounding.  What differs is the linear algebra: instead of an LDL' of the (n_q+m_q) KKT matrix
// the team eliminates the constraint block (nu = R(A xt - z) + y), then the slack variables
// (their diagonal blocks are 1x1 / 2x2), and keeps the explicit inverse of the remaining
// n x n SPD matrix  S = Psym^ + sigma I + A_x' R A_x - (slack Schur terms)  in shared memory, so
// one ADMM iteration is three small mat-vecs with no sequential triangular solve.
// Duplicate penalty rows are never materialised: they share z, y, E and rho by symmetry, so they
// enter as the weight `kd` wherever A' multiplies a row-space vector.
#pragma once
#include "sco_device.cuh"

struct QPArgs {
  const double *prm;  // problem parameter block
  const double *Jg;   // unscaled Jacobian entries, global layout (may be null when !use_pen)
  double pi;          // slack cost (compounded penalty weight)
  double kd;          // copies of every penalty row
  double wa;          // weight of the AffExpr objective terms (S.qa) in q
  int use_pen;        // 0: no penalty rows / slacks (closest feasible point)
  int closest;        // objective |x - xs|^2
  int has_hq;         // add the degree-2 model of a non-quadratic objective term (w.Hq, w.gq)
  int tail;           // the launch's work queue is drained: favour the latency of this problem (sco_dense.cuh)
  int warm;           // same J, b, pi, kd as the previous solve of this team (only the box changed): reuse
};

struct QPResult {
  int status, iters;
  double pri_res, dua_res;
#ifdef SCO_TIMING
  long long cyc_loop, cyc_check, cyc_setup;  // clock64() ticks: ADMM loop (incl. checks), checks, setup
  long long cyc_c[5];                        // stages of the termination test / phases of the generic loops
  long long cyc_scale;                       // generic setup: load + Ruiz (the rest of cyc_setup is S and its inverse)
#endif
};

// rho for a row with scaled bounds [l, u] (OSQP set_rho_vec)
__device__ __forceinline__ double rho_of(double l, double u, double rho) {
  if (l < -OSQP_INFTY * OSQP_MIN_SCALING && u > OSQP_INFTY * OSQP_MIN_SCALING) return OSQP_RHO_MIN;
  if (u - l < OSQP_RHO_TOL) return OSQP_RHO_EQ_OVER_RHO_INEQ * rho;
  return rho;
}

__device__ __forceinline__ double clampd(double v, double lo, double hi) {
  v = v < lo ? lo : v;
  v = v > hi ? hi : v;
  return v;
}

// project dy on the polar of the recession cone of [l,u] (OSQP is_primal_infeasible)
__device__ __forceinline__ double proj_dy(double dy, double l, double u) {
  if (u > OSQP_INFTY * OSQP_MIN_SCALING) {
    if (l < -OSQP_INFTY * OSQP_MIN_SCALING) return 0.0;
    return fmin(dy, 0.0);
  } else if (l < -OSQP_INFTY * OSQP_MIN_SCALING) {
    return fmax(dy, 0.0);
  }
  return dy;
}

// OSQP check_termination on the team-reduced, unscaled norms, for every ADMM loop: pri_res, max(|z|, |Ax|), the dual
// residual times c, max(|q|, |A'y|, |Px|), and the first stage of the primal (|E dy|_inf, u'dy+ + l'dy-) and of the dual
// (|D dx|_inf, q'dx) infeasibility certificates.  Returns 1 / 2 (solved / solved inaccurate), -7 or 0; `cert` gets
// bit 0 / bit 1 when the test failed on the primal / dual side and that certificate's first stage holds, so that
// its second stage has to run.  `approximate`: all tolerances x10 (the last test at max_iter).
__device__ __forceinline__ int qp_termination(double pri_res, double pri_scale, double dua_c, double dua_scale, double nvp,
                                              double lhs, double nvd, double qd, double c, double cinv, double eps_abs,
                                              double eps_rel, double eps_pinf, double eps_dinf, bool approximate,
                                              double &pri_out, double &dua_out, int &cert) {
  const double f = approximate ? 10.0 : 1.0;
  const double ea = f * eps_abs, er = f * eps_rel, epi = f * eps_pinf, edi = f * eps_dinf;
  const double dua_res = cinv * dua_c;
  pri_out = pri_res;
  dua_out = dua_res;
  cert = 0;
  if (pri_res > OSQP_INFTY || dua_res > OSQP_INFTY) return -7;
  const double eps_p = ea + er * pri_scale;
  const double eps_d = ea + er * cinv * dua_scale;
  const bool prim_ok = pri_res < eps_p, dual_ok = dua_res < eps_d;
  if (prim_ok && dual_ok) return approximate ? 2 : 1;
  if (!prim_ok && nvp > epi && lhs < -epi * nvp) cert |= 1;
  if (!dual_ok && nvd > edi && qd < -(c * edi * nvd)) cert |= 2;
  return 0;
}

#include "sco_dense.cuh"

// Per-entity terms of the termination test in the QPSolver mapping, accumulated into the caller's v[6] / sums[2]
// as maxima of absolute values (exact in any order): v[0] pri_res, v[1] max(|z|, |Ax|), v[2] the dual residual,
// v[3] max(|q|, |A'y|, |Px|) (each scaled back by E or D), v[4] / sums[0] the primal and v[5] / sums[1] the dual
// certificate's first stage -- the arguments of qp_termination once the team has reduced them.
// Unscaled primal residual terms of one row of A with scale E
__device__ __forceinline__ void qp_term_pri(double *v, double ax, double z, double E) {
  const double ei = 1.0 / E;
  v[0] = fmax(v[0], fabs((ax - z) * ei)); v[1] = fmax(v[1], fmax(fabs(z * ei), fabs(ax * ei)));
}
// First stage of the dual certificate for one variable (scale D, linear cost q^) with step dx
__device__ __forceinline__ void qp_term_dx(double *v, double *sums, double D, double dx, double q) {
  v[5] = fmax(v[5], fabs(D * dx));
  sums[1] += q * dx;
}
// A linear row (wt = 1) or a penalty row (wt = kd copies) [l, u] with its dual step dy
__device__ __forceinline__ void qp_term_row(double *v, double *sums, double ax, double z, double E, double dy, double l,
                                            double u, double wt) {
  qp_term_pri(v, ax, z, E);
  dy = proj_dy(dy, l, u);
  v[4] = fmax(v[4], fabs(E * dy));
  sums[0] += wt * (u * fmax(dy, 0.0) + l * fmin(dy, 0.0));
}
// A slack with its bound row [0, +inf): residuals and the primal certificate (qp_term_dx adds its dual one).
// qs = c pi Ds, aty = kd sl yp + bs ys
__device__ __forceinline__ void qp_term_slack(double *v, double *sums, double axs, double zs, double Es, double Ds,
                                              double qs, double aty, double dys) {
  qp_term_pri(v, axs, zs, Es);
  const double di = 1.0 / Ds;
  v[2] = fmax(v[2], fabs((qs + aty) * di)); v[3] = fmax(v[3], fmax(fabs(qs * di), fabs(aty * di)));
  const double us = OSQP_INFTY * Es;
  dys = proj_dy(dys, 0.0, us);
  v[4] = fmax(v[4], fabs(Es * dys));
  sums[0] += us * fmax(dys, 0.0);
}
// A variable with its box row [lb, ub]: ax = bx x, px = (P^ x)_j, aty = (A'y)_j including the box row
__device__ __forceinline__ void qp_term_var(double *v, double *sums, double ax, double zb, double Eb, double D, double q,
                                            double px, double aty, double dyb, double lb, double ub, double dx) {
  qp_term_row(v, sums, ax, zb, Eb, dyb, lb, ub, 1.0);
  const double di = 1.0 / D;
  v[2] = fmax(v[2], fabs((q + px + aty) * di));
  v[3] = fmax(v[3], fmax(fabs(q * di), fmax(fabs(aty * di), fabs(px * di))));
  qp_term_dx(v, sums, D, dx, q);
}

template <int TEAM, int DK>
struct QPSolver {
  const DevStruct &S;
  const DevSettings &st;
  QPW &w;
  const QPArgs &a;
  const int tid;
  const int n, m_lin, m_nl, ms;
  const double *Qg;  // global Q (may be null = zeros)
  double c;          // cost scaling
  double rho;        // current scalar rho

  __device__ QPSolver(const DevStruct &S_, const DevSettings &st_, QPW &w_, const QPArgs &a_)
      : S(S_), st(st_), w(w_), a(a_), tid(threadIdx.x), n(S_.n), m_lin(S_.m_lin),
        m_nl(a_.use_pen ? S_.m_nl : 0), ms(S_.m_nl), Qg(field_ptr(S_, S_.Q, a_.prm)), c(1.0),
        rho(st_.rho) {}

  __device__ __forceinline__ void sync() { Team<TEAM>::sync(); }

  // Every method starts with SCO_QP_LOCALS: by-value copies that shadow the members of the same name
  // (see DevIdx), followed by the small helpers as lambdas over those locals.
  //   psym(i, j)          entry of the symmetrised objective matrix (osqp_utils.py:153-163)
  //   gatherAT(j, vl, vp) A' * (row-space vector) for user variable j: linear rows (vl) and penalty
  //                       rows (vp; the caller folds the multiplicity kd into vp); bound row by the caller
  //   lin_row_dot / pen_row_dot   one row of A times a variable-space vector
  //   pcol_norm(j)        column j of c D |Psym| D
// S = P + sigma I + A'RA and its inverse: in shared memory (W_Sm), or -- for structures whose n x n matrix does not fit
// next to the rest of the working set (DevStruct::sws != 0) -- in the team's global workspace w.Sg (L2 / HBM)
// SM_GLOBAL: which of the two, as the expanding function knows it (a template parameter in the setup functions)
#define SM_GLOBAL (w.Sg != nullptr)
#define SM_LD(i) (SM_GLOBAL ? w.Sg[i] : W_Sm[i])
#define SM_ST(i, v)              \
  do {                           \
    if (SM_GLOBAL) w.Sg[i] = (v); \
    else W_Sm[i] = (v);          \
  } while (0)
#define SCO_QP_LOCALS                                                                                       \
  const DevStruct &SS = this->S;                                                                            \
  const QPW w = this->w; /* offsets as individual scalars: registers, not a struct in local memory */        \
  const Sh W_Js = w.Js, W_Sm = w.Sm, W_Als = w.Als, W_x = w.x, W_xt = w.xt, W_xt2 = w.xt2,                  \
      W_qh = w.qh, W_D = w.D, W_bx = w.bx, W_rb = w.rb, W_lb = w.lb, W_ub = w.ub, W_zb = w.zb,              \
      W_yb = w.yb, W_Eb = w.Eb, W_dxv = w.dxv, W_dyb = w.dyb, W_xs = w.xs, W_El = w.El,                     \
      W_rl = w.rl, W_ll = w.ll, W_ul = w.ul, W_zl = w.zl, W_yl = w.yl, W_wl = w.wl, W_dyl = w.dyl,          \
      W_Ep = w.Ep, W_rp = w.rp, W_lp = w.lp, W_up = w.up, W_zp = w.zp, W_yp = w.yp, W_wp = w.wp,            \
      W_bb = w.bb, W_fv = w.fv, W_dyp = w.dyp, W_s = w.s, W_Ds = w.Ds, W_sl = w.sl, W_bs = w.bs,            \
      W_zs = w.zs, W_ys = w.ys, W_Es = w.Es, W_gs = w.gs, W_hs = w.hs, W_rs = w.rs, W_dss = w.dss,          \
      W_dys = w.dys, W_Minv = w.Minv, W_red = w.red, W_stage = w.stage, W_Hq = w.Hq, W_gq = w.gq,           \
      W_xc = w.xc, W_ps = w.ps;                                                                             \
  const ShU32 W_msk = w.msk;                                                                                \
  (void)W_msk; (void)W_Js; (void)W_Sm; (void)W_Als; (void)W_x; (void)W_xt; (void)W_xt2; (void)W_qh; (void)W_D; (void)W_bx; (void)W_rb; (void)W_lb; (void)W_ub; (void)W_zb; (void)W_yb; (void)W_Eb; (void)W_dxv; (void)W_dyb; (void)W_xs; (void)W_El; (void)W_rl;\
  (void)W_ll; (void)W_ul; (void)W_zl; (void)W_yl; (void)W_wl; (void)W_dyl; (void)W_Ep; (void)W_rp; (void)W_lp; (void)W_up; (void)W_zp; (void)W_yp; (void)W_wp; (void)W_bb; (void)W_fv; (void)W_dyp; (void)W_s; (void)W_Ds; (void)W_sl; (void)W_bs;\
  (void)W_zs; (void)W_ys; (void)W_Es; (void)W_gs; (void)W_hs; (void)W_rs; (void)W_dss; (void)W_dys; (void)W_Minv; (void)W_red; (void)W_stage; (void)W_Hq; (void)W_gq; (void)W_xc; (void)W_ps;\
  const DevIdx S(this->S);                                                                                  \
  const DevSettings st = this->st;                                                                          \
  const QPArgs a = this->a;                                                                                 \
  const int tid = this->tid, n = this->n, m_lin = this->m_lin, m_nl = this->m_nl, ms = this->ms;            \
  const double *const Qg = this->Qg;                                                                        \
  double c = this->c, rho = this->rho;                                                                      \
  (void)SS; (void)ms; (void)rho;                                                                            \
  auto psym = [&](int i, int j) -> double {                                                                 \
    if (a.closest) return i == j ? 2.0 : 0.0;                                                               \
    double v = Qg ? 0.5 * (Qg[i * n + j] + Qg[j * n + i]) : 0.0;                                            \
    if (a.has_hq) v += 0.5 * (W_Hq[i * n + j] + W_Hq[j * n + i]); /* prob.py:348-367 */                     \
    return v;                                                                                               \
  };                                                                                                        \
  auto gatherAT = [&](int j, Sh vl, Sh vp) -> double {                                                      \
    double acc = 0.0;                                                                                       \
    if (m_lin)                                                                                              \
      for (int p = __ldg(S.lin_cptr + (j)); p < __ldg(S.lin_cptr + (j + 1)); p++) acc += W_Als[__ldg(S.lin_centry + (p))] * vl[__ldg(S.lin_crow + (p))]; \
    if (m_nl) {                                                                                             \
      double accp = 0.0;                                                                                    \
      for (int p = __ldg(S.pc_ptr + (j)); p < __ldg(S.pc_ptr + (j + 1)); p++) accp += W_Js[__ldg(S.pc_e + (p))] * vp[__ldg(S.pc_r + (p))];          \
      acc += accp;                                                                                          \
    }                                                                                                       \
    return acc;                                                                                             \
  };                                                                                                        \
  auto lin_row_dot = [&](int r, Sh v) -> double {                                                           \
    double acc = 0.0;                                                                                       \
    for (int p = __ldg(S.lin_rowptr + (r)); p < __ldg(S.lin_rowptr + (r + 1)); p++) acc += W_Als[p] * v[__ldg(S.lin_col + (p))];          \
    return acc;                                                                                             \
  };                                                                                                        \
  auto pen_row_dot = [&](int i, Sh v) -> double {                                                           \
    const int so = __ldg(S.row_soff + (i)), go = __ldg(S.row_goff + (i)), wd = __ldg(S.row_w + (i));                                      \
    double acc = 0.0;                                                                                       \
    for (int k = 0; k < wd; k++) acc += W_Js[so + k] * v[__ldg(S.jcol_g + (go + k))];                                 \
    return acc;                                                                                             \
  };                                                                                                        \
  /* column j of c D |Psym| D over the pattern of Psym (closest point: 2 I; objective model: dense) */        \
  auto pcol_norm = [&](int j) -> double {                                                                   \
    double cp = 0.0;                                                                                        \
    if (a.closest) cp = W_D[j] * fabs(SM_LD(j * n + j));                                                     \
    else if (a.has_hq) { for (int i = 0; i < n; i++) cp = fmax(cp, W_D[i] * fabs(SM_LD(i * n + j))); }       \
    else for (int p = __ldg(S.P_cptr + (j)); p < __ldg(S.P_cptr + (j + 1)); p++) {                              \
      const int i = __ldg(S.P_row + (p));                                                                     \
      cp = fmax(cp, W_D[i] * fabs(SM_LD(i * n + j)));                                                      \
    }                                                                                                       \
    return cp * c * W_D[j];                                                                                 \
  };                                                                                                        \
  /* (Psym v)_j for a variable-space vector v in shared memory */                                          \
  auto psym_dot = [&](int j, Sh v) -> double {                                                              \
    double px = 0.0;                                                                                        \
    if (a.closest) px = 2.0 * v[j];                                                                         \
    else if (a.has_hq) { for (int k = 0; k < n; k++) px += psym(k, j) * v[k]; }                             \
    else if (Qg) for (int p = __ldg(S.P_cptr + (j)); p < __ldg(S.P_cptr + (j + 1)); p++) {                      \
      const int k = __ldg(S.P_row + (p));                                                                     \
      px += 0.5 * (Qg[k * n + j] + Qg[j * n + k]) * v[k];                                                   \
    }                                                                                                       \
    return px;                                                                                              \
  };                                                                                                        \
  (void)psym; (void)gatherAT; (void)lin_row_dot; (void)pen_row_dot; (void)pcol_norm; (void)psym_dot;

  // ================================================================== setup
  // expects (unscaled): W_lb/W_ub bounds on x, W_bb = b, W_msk, W_xs (closest point target)
#undef SM_GLOBAL
#define SM_GLOBAL SG  // compile-time in the two setup functions: no test per matrix element
  template <bool SG>
  __device__ __noinline__ void load_and_scale() {
    SCO_QP_LOCALS
    const double *qg = field_ptr(SS, SS.q, a.prm), *qag = field_ptr(SS, SS.qa, a.prm);
    const double *llg = field_ptr(SS, SS.lin_l, a.prm), *ulg = field_ptr(SS, SS.lin_u, a.prm);
    for (int e = tid; e < n * n; e += TEAM) SM_ST(e, psym(e / n, e % n));
    for (int j = tid; j < n; j += TEAM) {
      W_qh[j] = a.closest ? -2.0 * W_xs[j]
                          : (qg ? qg[j] : 0.0) + (qag ? a.wa * qag[j] : 0.0) + (a.has_hq ? W_gq[j] : 0.0);
      W_D[j] = 1.0;
      W_bx[j] = 1.0;
      W_Eb[j] = 1.0;
    }
    for (int e = tid; e < S.nnz_lin; e += TEAM) W_Als[e] = __ldg(S.lin_val + (e));
    for (int r = tid; r < m_lin; r += TEAM) W_El[r] = 1.0;
    for (int i = tid; i < m_nl; i += TEAM) {
      const int so = __ldg(S.row_soff + (i)), go = __ldg(S.row_goff + (i)), wd = __ldg(S.row_w + (i));
      const int mo = i * SS.mw;
      for (int k = 0; k < wd; k++) W_Js[so + k] = ((W_msk[mo + (k >> 5)] >> (k & 31)) & 1u) ? a.Jg[go + k] : 0.0;
      W_Ep[i] = 1.0;
      W_sl[i] = -1.0; W_bs[i] = 1.0; W_Ds[i] = 1.0; W_Es[i] = 1.0;
      if (__ldg(S.row_eq + (i))) {
        W_sl[ms + i] = 1.0; W_bs[ms + i] = 1.0; W_Ds[ms + i] = 1.0; W_Es[ms + i] = 1.0;
      }
    }
    c = 1.0;
    sync();
    const int nq = n + (a.use_pen ? S.n_slack : 0);
    // Ruiz passes.  temporaries: Dt -> xt, Etb -> xt2, Etl -> wl, Etp -> wp, Dts -> gs, Ets -> dys
    for (int it = 0; it < st.scaling; it++) {
      for (int j = tid; j < n; j += TEAM) {
        const double cp = pcol_norm(j);
        double ca = fabs(W_bx[j]);
        if (m_lin)
          for (int p = __ldg(S.lin_cptr + (j)); p < __ldg(S.lin_cptr + (j + 1)); p++)
            ca = fmax(ca, fabs(W_Als[__ldg(S.lin_centry + (p))]));
        if (m_nl)
          for (int p = __ldg(S.pc_ptr + (j)); p < __ldg(S.pc_ptr + (j + 1)); p++) ca = fmax(ca, fabs(W_Js[__ldg(S.pc_e + (p))]));
        W_xt[j] = 1.0 / sqrt(limit_scaling(fmax(cp, ca)));
        W_xt2[j] = 1.0 / sqrt(limit_scaling(fabs(W_bx[j])));
      }
      for (int r = tid; r < m_lin; r += TEAM) {
        double rn = 0.0;
        for (int p = __ldg(S.lin_rowptr + (r)); p < __ldg(S.lin_rowptr + (r + 1)); p++) rn = fmax(rn, fabs(W_Als[p]));
        W_wl[r] = 1.0 / sqrt(limit_scaling(rn));
      }
      for (int i = tid; i < m_nl; i += TEAM) {
        const int so = __ldg(S.row_soff + (i)), wd = __ldg(S.row_w + (i)), eq = __ldg(S.row_eq + (i));
        double rn = fabs(W_sl[i]);
        if (eq) rn = fmax(rn, fabs(W_sl[ms + i]));
        for (int k = 0; k < wd; k++) rn = fmax(rn, fabs(W_Js[so + k]));
        W_wp[i] = 1.0 / sqrt(limit_scaling(rn));
        for (int k2 = 0; k2 <= eq; k2++) {
          const int si = k2 * ms + i;
          W_gs[si] = 1.0 / sqrt(limit_scaling(fmax(fabs(W_sl[si]), fabs(W_bs[si]))));
          W_dys[si] = 1.0 / sqrt(limit_scaling(fabs(W_bs[si])));
        }
      }
      sync();
      for (int r = tid; r < m_lin; r += TEAM) {
        const double er = W_wl[r];
        for (int p = __ldg(S.lin_rowptr + (r)); p < __ldg(S.lin_rowptr + (r + 1)); p++)
          W_Als[p] *= er * W_xt[__ldg(S.lin_col + (p))];
        W_El[r] *= er;
      }
      for (int i = tid; i < m_nl; i += TEAM) {
        const int so = __ldg(S.row_soff + (i)), go = __ldg(S.row_goff + (i)), wd = __ldg(S.row_w + (i)), eq = __ldg(S.row_eq + (i));
        const double er = W_wp[i];
        for (int k = 0; k < wd; k++) W_Js[so + k] *= er * W_xt[__ldg(S.jcol_g + (go + k))];
        W_Ep[i] *= er;
        for (int k2 = 0; k2 <= eq; k2++) {
          const int si = k2 * ms + i;
          W_sl[si] *= er * W_gs[si];
          W_bs[si] *= W_dys[si] * W_gs[si];
          W_Ds[si] *= W_gs[si];
          W_Es[si] *= W_dys[si];
        }
      }
      sync();  // column data of Js / Als final before D changes (pcol_norm below reads D only)
      for (int j = tid; j < n; j += TEAM) {
        W_bx[j] *= W_xt2[j] * W_xt[j];
        W_Eb[j] *= W_xt2[j];
        W_qh[j] *= W_xt[j];
        W_D[j] *= W_xt[j];
      }
      sync();
      // cost normalisation
      double vs[1] = {0.0}, vm[1] = {0.0};
      for (int j = tid; j < n; j += TEAM) {
        vs[0] += pcol_norm(j);
        vm[0] = fmax(vm[0], fabs(W_qh[j]));
      }
      if (m_nl) {
        const double cq = fabs(c * a.pi);
        for (int i = tid; i < m_nl; i += TEAM)
          for (int k2 = 0; k2 <= __ldg(S.row_eq + (i)); k2++) vm[0] = fmax(vm[0], cq * W_Ds[k2 * ms + i]);
      }
      Team<TEAM>::reduce_sum(vs, W_red);
      Team<TEAM>::reduce_max(vm, W_red);
      const double mean = vs[0] / (double)nq;
      const double ct = 1.0 / limit_scaling(fmax(mean, limit_scaling(vm[0])));
      for (int j = tid; j < n; j += TEAM) W_qh[j] *= ct;
      c *= ct;
      sync();
    }
    // scaled bounds
    for (int j = tid; j < n; j += TEAM) {
      const double eb = W_Eb[j];
      W_lb[j] = eb * fmax(W_lb[j], -OSQP_INFTY);
      W_ub[j] = eb * fmin(W_ub[j], OSQP_INFTY);
    }
    for (int r = tid; r < m_lin; r += TEAM) {
      W_ll[r] = W_El[r] * fmax(llg ? llg[r] : 0.0, -OSQP_INFTY);
      W_ul[r] = W_El[r] * fmin(ulg ? ulg[r] : 0.0, OSQP_INFTY);
    }
    for (int i = tid; i < m_nl; i += TEAM) {
      const double hi = clampd(-W_bb[i], -OSQP_INFTY, OSQP_INFTY);
      W_up[i] = W_Ep[i] * hi;
      W_lp[i] = __ldg(S.row_eq + (i)) ? W_Ep[i] * hi : -OSQP_INFTY * W_Ep[i];
    }
    this->c = c;
    sync();
  }
#undef SM_GLOBAL
#define SM_GLOBAL (w.Sg != nullptr)

  __device__ void set_rho() {
    SCO_QP_LOCALS
    rho = fmin(fmax(rho, OSQP_RHO_MIN), OSQP_RHO_MAX);
    this->rho = rho;
    for (int j = tid; j < n; j += TEAM) W_rb[j] = rho_of(W_lb[j], W_ub[j], rho);
    for (int r = tid; r < m_lin; r += TEAM) W_rl[r] = rho_of(W_ll[r], W_ul[r], rho);
    for (int i = tid; i < m_nl; i += TEAM) {
      W_rp[i] = rho_of(W_lp[i], W_up[i], rho);
      for (int k2 = 0; k2 <= __ldg(S.row_eq + (i)); k2++)
        W_rs[k2 * ms + i] = rho_of(0.0, OSQP_INFTY * W_Es[k2 * ms + i], rho);
    }
    sync();
  }

  // S = Psym^ + sigma I + A_x' R A_x - slack Schur terms, then S <- S^-1 (in place).
  // `reload`: Sm does not hold the unscaled Psym any more (rho update) -> fetch it again.
#undef SM_GLOBAL
#define SM_GLOBAL SG
  template <bool SG>
  __device__ __noinline__ void assemble_and_invert(bool reload) {
    SCO_QP_LOCALS
    const double sigma = st.sigma;
    for (int i = tid; i < m_nl; i += TEAM) {
      const double kr = a.kd * W_rp[i];
      const double s1 = W_sl[i], b1 = W_bs[i];
      const double m11 = sigma + kr * s1 * s1 + W_rs[i] * b1 * b1;
      double coef;
      if (__ldg(S.row_eq + (i))) {
        const double s2 = W_sl[ms + i], b2 = W_bs[ms + i];
        const double m22 = sigma + kr * s2 * s2 + W_rs[ms + i] * b2 * b2;
        const double m12 = kr * s1 * s2;
        const double det = m11 * m22 - m12 * m12;
        const double i11 = m22 / det, i22 = m11 / det, i12 = -m12 / det;
        W_Minv[3 * i] = i11; W_Minv[3 * i + 1] = i12; W_Minv[3 * i + 2] = i22;
        const double h1 = kr * (i11 * s1 + i12 * s2), h2 = kr * (i12 * s1 + i22 * s2);
        W_hs[i] = h1; W_hs[ms + i] = h2;
        coef = kr - kr * (s1 * h1 + s2 * h2);
      } else {
        const double i11 = 1.0 / m11;
        W_Minv[3 * i] = i11; W_Minv[3 * i + 1] = 0.0; W_Minv[3 * i + 2] = 0.0;
        const double h1 = kr * i11 * s1;
        W_hs[i] = h1;
        coef = kr - kr * s1 * h1;
      }
      W_wp[i] = coef;
    }
    for (int e = tid; e < n * n; e += TEAM) {
      const int i = e / n, j = e % n;
      const double pv = reload ? psym(i, j) : SM_LD(e);
      double v = c * W_D[i] * pv * W_D[j];
      if (i == j) v += sigma + W_rb[j] * W_bx[j] * W_bx[j];
      SM_ST(e, v);
    }
    sync();
    for (int j = tid; j < n; j += TEAM) {
      if (m_lin) {
        for (int p = __ldg(S.lin_cptr + (j)); p < __ldg(S.lin_cptr + (j + 1)); p++) {
          const int r = __ldg(S.lin_crow + (p));
          const double f = W_rl[r] * W_Als[__ldg(S.lin_centry + (p))];
          for (int q2 = __ldg(S.lin_rowptr + (r)); q2 < __ldg(S.lin_rowptr + (r + 1)); q2++) {
            const int e2 = __ldg(S.lin_col + (q2)) * n + j;
            SM_ST(e2, SM_LD(e2) + f * W_Als[q2]);
          }
        }
      }
      if (m_nl) {
        for (int p = __ldg(S.pc_ptr + (j)); p < __ldg(S.pc_ptr + (j + 1)); p++) {
          const int r = __ldg(S.pc_r + (p));
          const double f = W_wp[r] * W_Js[__ldg(S.pc_e + (p))];
          const int so = __ldg(S.row_soff + (r)), go = __ldg(S.row_goff + (r)), wd = __ldg(S.row_w + (r));
          for (int k = 0; k < wd; k++) {
            const int e2 = __ldg(S.jcol_g + (go + k)) * n + j;
            SM_ST(e2, SM_LD(e2) + f * W_Js[so + k]);
          }
        }
      }
    }
    sync();
    // in-place Gauss-Jordan inverse (S is SPD: no pivoting).  xt = pivot row, xt2 = pivot column.
    // S is banded for trajectory structures (half-bandwidth s_bw): beyond row / column k + s_bw the pivot row and
    // column of step k are still exact zeros, so the sweep only touches the leading mk x mk block (the same
    // arithmetic on every element it changes, a third of the work for a narrow band).
    const int bw = SS.s_bw;
    for (int k = 0; k < n; k++) {
      const int mk = (k + bw + 1) < n ? (k + bw + 1) : n;
      const double d = 1.0 / SM_LD(k * n + k);
      for (int j = tid; j < mk; j += TEAM) {
        W_xt[j] = SM_LD(k * n + j) * d;
        W_xt2[j] = SM_LD(j * n + k);
      }
      sync();
      int i = tid / mk, j = tid - i * mk;
      const int di = TEAM / mk, dj = TEAM - di * mk;
      while (i < mk) {
        const int e = i * n + j;
        double v;
        if (i == k) v = (j == k) ? d : W_xt[j];
        else if (j == k) v = -W_xt2[i] * d;
        else v = SM_LD(e) - W_xt2[i] * W_xt[j];
        SM_ST(e, v);
        j += dj;
        i += di;
        if (j >= mk) { j -= mk; i++; }
      }
      sync();
    }
  }

#undef SM_GLOBAL
#define SM_GLOBAL (w.Sg != nullptr)

  // ================================================================== termination
  // Returns a terminal status or 0.  Scratch: xt (D.*x), wp (kd*yp).  sc[], when given, receives the scaled
  // norms needed by the rho estimate: {|Ax-z|, max(|z|, |Ax|), |Px+q+A'y|, max(|q|, |A'y|, |Px|)}.
  __device__ __noinline__ int check(int approximate, double &pri_res_out, double &dua_res_out, double *sc) {
    SCO_QP_LOCALS
    // v[6], sums[2]: see qp_term_pri.  The per-thread order of the sums is the one the certificates' first stage is
    // defined with: linear rows, penalty rows with their slacks, variables, then the slacks' dual-certificate terms.
    double v[6] = {0, 0, 0, 0, 0, 0};
    double u[4] = {0, 0, 0, 0};  // v[0..3] in the scaled problem, for the rho estimate
    const bool rho_est = sc != nullptr;  // u only then: the loops get a version with fewer live values for the tests
    double sums[2] = {0.0, 0.0};
    for (int r = tid; r < m_lin; r += TEAM) {
      const double ax = lin_row_dot(r, W_x), z = W_zl[r];
      qp_term_row(v, sums, ax, z, W_El[r], W_dyl[r], W_ll[r], W_ul[r], 1.0);
      if (rho_est) { u[0] = fmax(u[0], fabs(ax - z)); u[1] = fmax(u[1], fmax(fabs(z), fabs(ax))); }
    }
    for (int i = tid; i < m_nl; i += TEAM) {
      const int eq = __ldg(S.row_eq + (i));
      double ax = pen_row_dot(i, W_x) + W_sl[i] * W_s[i];
      if (eq) ax += W_sl[ms + i] * W_s[ms + i];
      const double z = W_zp[i];
      qp_term_row(v, sums, ax, z, W_Ep[i], W_dyp[i], W_lp[i], W_up[i], a.kd);
      if (rho_est) { u[0] = fmax(u[0], fabs(ax - z)); u[1] = fmax(u[1], fmax(fabs(z), fabs(ax))); }
      for (int k2 = 0; k2 <= eq; k2++) {
        const int si = k2 * ms + i;
        const double axs = W_bs[si] * W_s[si], zs = W_zs[si];
        // slack variable: q^ + A'y (its P block is zero)
        const double qs = c * a.pi * W_Ds[si];
        const double aty = a.kd * W_sl[si] * W_yp[i] + W_bs[si] * W_ys[si];
        qp_term_slack(v, sums, axs, zs, W_Es[si], W_Ds[si], qs, aty, W_dys[si]);
        if (rho_est) {
          u[0] = fmax(u[0], fabs(axs - zs)); u[1] = fmax(u[1], fmax(fabs(zs), fabs(axs)));
          u[2] = fmax(u[2], fabs(qs + aty)); u[3] = fmax(u[3], fmax(fabs(qs), fabs(aty)));
        }
      }
    }
    for (int i = tid; i < m_nl; i += TEAM) W_wp[i] = a.kd * W_yp[i];
    for (int j = tid; j < n; j += TEAM) W_xt[j] = W_D[j] * W_x[j];
    sync();
    for (int j = tid; j < n; j += TEAM) {
      const double ax = W_bx[j] * W_x[j], z = W_zb[j];
      double px = psym_dot(j, W_xt);
      px *= c * W_D[j];
      const double aty = gatherAT(j, W_yl, W_wp) + W_bx[j] * W_yb[j];
      const double q = W_qh[j];
      qp_term_var(v, sums, ax, z, W_Eb[j], W_D[j], q, px, aty, W_dyb[j], W_lb[j], W_ub[j], W_dxv[j]);
      if (rho_est) {
        u[0] = fmax(u[0], fabs(ax - z)); u[1] = fmax(u[1], fmax(fabs(z), fabs(ax)));
        u[2] = fmax(u[2], fabs(q + px + aty)); u[3] = fmax(u[3], fmax(fabs(q), fmax(fabs(aty), fabs(px))));
      }
    }
    for (int i = tid; i < m_nl; i += TEAM)
      for (int k2 = 0; k2 <= __ldg(S.row_eq + (i)); k2++) {
        const int si = k2 * ms + i;
        qp_term_dx(v, sums, W_Ds[si], W_dss[si], c * a.pi * W_Ds[si]);
      }
    Team<TEAM>::template reduce_mixed<6, 2>(v, sums, W_red);
    if (rho_est) {
      Team<TEAM>::reduce_max(u, W_red);
      for (int k = 0; k < 4; k++) sc[k] = u[k];
    }
    int cert;
    const int status = qp_termination(v[0], v[1], v[2], v[3], v[4], sums[0], v[5], sums[1], c, 1.0 / c, st.eps_abs,
                                      st.eps_rel, st.eps_prim_inf, st.eps_dual_inf, approximate != 0, pri_res_out,
                                      dua_res_out, cert);
    if (status != 0) return status;
    const double f = approximate ? 10.0 : 1.0;
    const bool pinf = (cert & 1) && primal_infeasible(f * st.eps_prim_inf, v[4]);
    const bool dinf = (cert & 2) && dual_infeasible(f * st.eps_dual_inf, v[5]);
    if (pinf) return approximate ? 3 : -3;
    if (dinf) return approximate ? 4 : -4;
    return 0;
  }

  // Second stage of OSQP is_primal_infeasible on delta_y of the last iteration: dyl (lin), dyp (pen), dyb (x bounds),
  // dys (slack bounds).  Entered when the first stage holds: nv = |E dy|_inf, reduced by check().
  __device__ __noinline__ bool primal_infeasible(double eps, double nv) {
    SCO_QP_LOCALS
    for (int r = tid; r < m_lin; r += TEAM) W_dyl[r] = proj_dy(W_dyl[r], W_ll[r], W_ul[r]);
    for (int i = tid; i < m_nl; i += TEAM) {
      const double dy = proj_dy(W_dyp[i], W_lp[i], W_up[i]);
      W_dyp[i] = dy;
      W_wp[i] = a.kd * dy;
      for (int k2 = 0; k2 <= __ldg(S.row_eq + (i)); k2++) {
        const int si = k2 * ms + i;
        W_dys[si] = proj_dy(W_dys[si], 0.0, OSQP_INFTY * W_Es[si]);
      }
    }
    for (int j = tid; j < n; j += TEAM) W_dyb[j] = proj_dy(W_dyb[j], W_lb[j], W_ub[j]);
    sync();
    double mv[1] = {0.0};
    for (int j = tid; j < n; j += TEAM) {
      const double aty = gatherAT(j, W_dyl, W_wp) + W_bx[j] * W_dyb[j];
      mv[0] = fmax(mv[0], fabs(aty / W_D[j]));
    }
    for (int i = tid; i < m_nl; i += TEAM)
      for (int k2 = 0; k2 <= __ldg(S.row_eq + (i)); k2++) {
        const int si = k2 * ms + i;
        const double aty = W_sl[si] * W_wp[i] + W_bs[si] * W_dys[si];
        mv[0] = fmax(mv[0], fabs(aty / W_Ds[si]));
      }
    Team<TEAM>::reduce_max(mv, W_red);
    sync();
    return mv[0] < eps * nv;
  }

  // Second stage of OSQP is_dual_infeasible on delta_x of the last iteration: dxv (user variables), dss (slacks).
  // Entered when the first stage holds: nv = |D dx|_inf, reduced by check().
  __device__ __noinline__ bool dual_infeasible(double eps, double nv) {
    SCO_QP_LOCALS
    for (int j = tid; j < n; j += TEAM) W_xt[j] = W_D[j] * W_dxv[j];
    sync();
    bool res = false;
    const double thr = c * eps * nv;
    double pv[1] = {0.0};
    for (int j = tid; j < n; j += TEAM) {
      const double px = psym_dot(j, W_xt);
      pv[0] = fmax(pv[0], fabs(c * px));  // Dinv .* (c D Psym D dx) = c * Psym (D dx)
    }
    Team<TEAM>::reduce_max(pv, W_red);
    if (pv[0] < thr) {
      const double lim = eps * nv;
      double bad[1] = {0.0};
      for (int r = tid; r < m_lin; r += TEAM) {
        const double adx = lin_row_dot(r, W_dxv) / W_El[r];
        if ((W_ul[r] < OSQP_INFTY * OSQP_MIN_SCALING && adx > lim) ||
            (W_ll[r] > -OSQP_INFTY * OSQP_MIN_SCALING && adx < -lim)) bad[0] = 1.0;
      }
      for (int i = tid; i < m_nl; i += TEAM) {
        double adx = pen_row_dot(i, W_dxv) + W_sl[i] * W_dss[i];
        if (__ldg(S.row_eq + (i))) adx += W_sl[ms + i] * W_dss[ms + i];
        adx /= W_Ep[i];
        if ((W_up[i] < OSQP_INFTY * OSQP_MIN_SCALING && adx > lim) ||
            (W_lp[i] > -OSQP_INFTY * OSQP_MIN_SCALING && adx < -lim)) bad[0] = 1.0;
        for (int k2 = 0; k2 <= __ldg(S.row_eq + (i)); k2++) {
          const int si = k2 * ms + i;
          const double ads = W_bs[si] * W_dss[si] / W_Es[si];
          if ((OSQP_INFTY * W_Es[si] < OSQP_INFTY * OSQP_MIN_SCALING && ads > lim) || ads < -lim)
            bad[0] = 1.0;
        }
      }
      for (int j = tid; j < n; j += TEAM) {
        const double adx = W_bx[j] * W_dxv[j] / W_Eb[j];
        if ((W_ub[j] < OSQP_INFTY * OSQP_MIN_SCALING && adx > lim) ||
            (W_lb[j] > -OSQP_INFTY * OSQP_MIN_SCALING && adx < -lim)) bad[0] = 1.0;
      }
      Team<TEAM>::reduce_max(bad, W_red);
      res = bad[0] == 0.0;
    }
    sync();
    return res;
  }


#ifdef SCO_TIMING
#define SCO_PH(k) { sync(); const long long tq_ = clock64(); res.cyc_c[k] += tq_ - tph; tph = tq_; }
#else
#define SCO_PH(k)
#endif

  // ================================================================== the ADMM loop, ONE THREAD PER ENTITY
  // Same iteration as generic_loop below (same formulas in the same order; y / rho is y * (1 / rho) as in the
  // reference's rho_inv_vec), different machine mapping: a thread owns ONE entity for the whole QP --
  //   warps [0, nV)        variable j with its box row          (x, zb, yb)
  //   warps [nV, nV + nL)  linear row r                         (z, y)
  //   then nP warps        penalty row i with its one / two slacks
  // (every role starts on a warp boundary) -- and keeps that entity's iterates AND constants in registers,
  // including the first entries of its row of A (rows: SCO_EN) or of its column of A (variables: SCO_EH from
  // linear rows + SCO_EH from penalty rows): coefficient + shared-memory index of the operand, padded with zero
  // coefficients so that the products run without a branch -- an iteration touches no index array at all.
  // generic_loop re-reads every constant from shared memory and every index from global memory in every iteration
  // and strides TEAM threads over the entities (12,110 / 8,525 cycles per iteration for the arm / point robot;
  // profiles/r1_cycles.txt).  S^-1 rhs is split over all threads (column segments, partial sums through shared
  // memory).  Iterates go back to the shared-memory arrays only when the termination test runs (every
  // check_termination iterations) or the loop ends, so check() / the certificates / the epilogue of solve() are
  // shared with generic_loop.
  // The three roles run three instantiations of fast_role<ROLE>, each with its own register allocation (one
  // function holding the state of all three roles needs ~150 registers; a 512-thread team has 128).  All of them
  // execute the same sequence of team barriers; the barrier only counts arrivals.
  // Requires ceil32(n) + ceil32(m_lin) + ceil32(m_nl) <= TEAM and no adaptive rho.
#define SCO_EN 8
#define SCO_EH 4
  // Everything the hot loop needs, by value: a handful of shared-memory offsets and scalars.  The loop must not touch
  // the solver object (QPW offsets, settings, index arrays live in local memory: with 512 threads per team and
  // ~150 KB of shared memory the L1 that backs local memory is a few dozen KB, and every such access is an L2 round
  // trip -- measured: 1,500 cycles for a phase that does one multiply-add).
  struct FastCtx {
    int id;        // index of the entity inside its role
    int act;       // 0: padding lane of a role's last warp
    int n, ms;
    int K3, j3, s3, c0, c1, p3_active;  // S^-1 rhs: column segment [c0, c1) of row j3
    int o_Sm, o_xt, o_xt2, o_ps, o_wl, o_wp;  // shared-memory offsets (doubles)
    int max_iter, chk, has_pen, m_nl;
    int o_red, inline_test;  // the termination test inside the register loop (fast_role): reduction scratch, applicable?
    double sigma, alpha, kd, cpi;
    double c, eps_abs, eps_rel, eps_pinf, eps_dinf;
  };

  // Hand-over of the iterates (and, at a test iteration, of the last step's deltas) to the shared-memory arrays that
  // check() / the certificates / the epilogue of solve() work on, followed by the termination test.  Out of line: the
  // ~20 array offsets it needs are loaded here, once per check_termination iterations, not carried through the loop.
  //   ROLE 0: v = x zb yb, d = dx dyb          ROLE 1: v = z y, d = dy
  //   ROLE 2: v = zp yp s1 zs1 ys1 s2 zs2 ys2, d = dyp dss1 dys1 dss2 dys2
  template <int ROLE>
  // `store_d`: the deltas go to shared memory too -- at a tested iteration and at the last one, whose final tests
  // (QPSolver::solve) evaluate the certificates on the deltas of that iteration, as OSQP does
  __device__ __noinline__ int fast_flush(int id, int act, int eq, int can_check, int store_d, QPResult &res, double v0,
                                         double v1, double v2, double v3, double v4, double v5, double v6, double v7,
                                         double d0, double d1, double d2, double d3, double d4) {
    const QPW &wq = this->w;
    const int ms = this->ms;
    if (act) {
      if (ROLE == 0) {
        wq.x[id] = v0; wq.zb[id] = v1; wq.yb[id] = v2;
        if (store_d) { wq.dxv[id] = d0; wq.dyb[id] = d1; }
      } else if (ROLE == 1) {
        wq.zl[id] = v0; wq.yl[id] = v1;
        if (store_d) wq.dyl[id] = d0;
      } else if (ROLE == 2) {
        wq.zp[id] = v0; wq.yp[id] = v1;
        wq.s[id] = v2; wq.zs[id] = v3; wq.ys[id] = v4;
        if (eq) { wq.s[ms + id] = v5; wq.zs[ms + id] = v6; wq.ys[ms + id] = v7; }
        if (store_d) {
          wq.dyp[id] = d0; wq.dss[id] = d1; wq.dys[id] = d2;
          if (eq) { wq.dss[ms + id] = d3; wq.dys[ms + id] = d4; }
        }
      }
    }
    sync();
    int status = 0;
    if (can_check) {
#ifdef SCO_TIMING
      const long long tc0 = clock64();
#endif
      status = check(0, res.pri_res, res.dua_res, nullptr);
#ifdef SCO_TIMING
      res.cyc_check += clock64() - tc0;
#endif
      if (status == 0) sync();
    }
    return status;
  }

  // DENSE = 1: structures whose penalty rows are dense (QUADFORM / VM rows over all n <= 32 variables, m_nl <= 48,
  // no linear rows -- the QCQP shapes with more than 32 rows, which the two-warp dense kernel does not take): a
  // penalty-row thread keeps its whole row of J (SCO_DN coefficients), a variable thread its whole column (SCO_DM),
  // operands are read with broadcast 128-bit loads; no addresses are stored.
#define SCO_DN 32
#define SCO_DM 48
  template <int ROLE, int DENSE>  // ROLE: 0 variable, 1 linear row, 2 penalty row of a structure without equality rows,
  // 4 penalty row (one or two slacks), 3 none (idle warps still do their share of S^-1 rhs)
  __device__ __noinline__ int fast_role(const FastCtx f, int &iter_out, bool &checked_out, QPResult &res) {
    constexpr bool PEN = ROLE == 2 || ROLE == 4, EQS = ROLE == 4;
    constexpr int NEC = DENSE ? (ROLE == 0 ? SCO_DM : SCO_DN) : SCO_EN;  // coefficient slots of this role
    // the in-loop termination test costs ~20 registers: not at the 128-register budget of the 512-thread team
    constexpr bool INL = !DENSE && TEAM <= 256;
    const int id = f.id, n = f.n;
    const bool act = f.act != 0;
    const double sigma = f.sigma, alpha = f.alpha, oma = 1.0 - f.alpha, kd = f.kd;
    const int max_iter = f.max_iter, chk = f.chk;
    int iter = 0, status = 0, next_check = chk ? chk : max_iter + 1;
    bool checked = false;
    while (iter < max_iter) {
      // ---- (re)load the entity: constants, entries of A and iterates, all from shared memory.  This happens at the
      // start and after every termination test: the test is a call, and whatever lives across a call is given a home
      // in LOCAL memory by the compiler and re-read from there in every iteration (L1 does not keep it: 98 % misses
      // measured) -- so nothing is kept across it.  Unused entry slots multiply the coefficient 0 with ps[0], which
      // always holds a finite number.
      double ec[NEC];
      int ea[SCO_EN];
#pragma unroll
      for (int k = 0; k < NEC; k++) ec[k] = 0.0;
#pragma unroll
      for (int k = 0; k < SCO_EN; k++) ea[k] = f.o_ps;
      double x = 0.0, zb = 0.0, yb = 0.0, qh = 0.0, bx = 0.0, rb = 1.0, rbi = 1.0, lb = 0.0, ub = 0.0;   // variable
      double z = 0.0, y = 0.0, rr = 1.0, rri = 1.0, lo = 0.0, hi = 0.0;                                   // row (lin / pen)
      double mi11 = 0.0, mi12 = 0.0, mi22 = 0.0;                                                          // pen
      double s1 = 0.0, zs1 = 0.0, ys1 = 0.0, sl1 = 0.0, bs1 = 0.0, rs1 = 1.0, rsi1 = 1.0, cd1 = 0.0, us1 = 0.0, hs1 = 0.0, g1 = 0.0;
      double s2 = 0.0, zs2 = 0.0, ys2 = 0.0, sl2 = 0.0, bs2 = 0.0, rs2 = 1.0, rsi2 = 1.0, cd2 = 0.0, us2 = 0.0, hs2 = 0.0, g2 = 0.0;
      double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0, d4 = 0.0;  // deltas of the last iteration (certificates)
      // scaling factors the in-loop termination test needs: variable Eb, D | linear row El | penalty row Ep, Es1, Ds1, Es2, Ds2
      double k0 = 1.0, k1 = 1.0, k2s = 1.0, k3 = 1.0, k4 = 1.0;
      double pq[4] = {0.0, 0.0, 0.0, 0.0};  // variable: its column of Psym (<= 4 entries) ...
      int pa[4] = {f.o_ps, f.o_ps, f.o_ps, f.o_ps};  // ... and where the operands (D x)_k are published
      int eq = 0;
      {
        const QPW &wq = this->w;
        const DevStruct &SS = this->S;
        const int m_lin = this->m_lin, m_nl = this->m_nl, ms = f.ms;
        if (ROLE == 0 && act) {
          const int j = id;
          x = wq.x[j]; zb = wq.zb[j]; yb = wq.yb[j];
          k0 = wq.Eb[j]; k1 = wq.D[j];
          if (INL && f.inline_test) {
            if (this->a.closest) { pq[0] = 2.0; pa[0] = f.o_xt + j; }
            else if (this->Qg) {
              const double *Qg_ = this->Qg;
              const int p0 = __ldg(SS.P_cptr + (j)), p1 = __ldg(SS.P_cptr + (j + 1));
#pragma unroll
              for (int k = 0; k < 4; k++)
                if (p0 + k < p1) {
                  const int r = __ldg(SS.P_row + (p0 + k));
                  pq[k] = 0.5 * (Qg_[r * n + j] + Qg_[j * n + r]);
                  pa[k] = f.o_xt + r;
                }
            }
          }
          qh = wq.qh[j]; bx = wq.bx[j]; rb = wq.rb[j]; rbi = 1.0 / rb; lb = wq.lb[j]; ub = wq.ub[j];
          int pl0 = 0, pl1 = 0, pp0 = 0, pp1 = 0;
          if (m_lin) { pl0 = __ldg(SS.lin_cptr + (j)); pl1 = __ldg(SS.lin_cptr + (j + 1)); }
          if (m_nl) { pp0 = __ldg(SS.pc_ptr + (j)); pp1 = __ldg(SS.pc_ptr + (j + 1)); }
          if (DENSE) {  // column j of the dense J: entry (row k, column j)
#pragma unroll
            for (int k = 0; k < NEC; k++)
              if (k < m_nl) ec[k] = wq.Js[__ldg(SS.row_soff + (k)) + j];
          } else
#pragma unroll
          for (int k = 0; k < SCO_EH; k++) {
            if (pl0 + k < pl1) {
              ec[k] = wq.Als[__ldg(SS.lin_centry + (pl0 + k))];
              ea[k] = f.o_wl + __ldg(SS.lin_crow + (pl0 + k));
            }
            if (pp0 + k < pp1) {
              ec[SCO_EH + k] = wq.Js[__ldg(SS.pc_e + (pp0 + k))];
              ea[SCO_EH + k] = f.o_wp + __ldg(SS.pc_r + (pp0 + k));
            }
          }
        } else if (ROLE == 1 && act) {
          const int r = id;
          z = wq.zl[r]; y = wq.yl[r];
          k0 = wq.El[r];
          rr = wq.rl[r]; rri = 1.0 / rr; lo = wq.ll[r]; hi = wq.ul[r];
          const int p0 = __ldg(SS.lin_rowptr + (r)), p1 = __ldg(SS.lin_rowptr + (r + 1));
#pragma unroll
          for (int k = 0; k < SCO_EN; k++)
            if (p0 + k < p1) { ec[k] = wq.Als[p0 + k]; ea[k] = f.o_xt2 + __ldg(SS.lin_col + (p0 + k)); }
        } else if (PEN && act) {
          const int i = id;
          eq = EQS ? __ldg(SS.row_eq + (i)) : 0;
          z = wq.zp[i]; y = wq.yp[i];
          k0 = wq.Ep[i]; k1 = wq.Es[i]; k2s = wq.Ds[i];
          if (EQS && eq) { k3 = wq.Es[ms + i]; k4 = wq.Ds[ms + i]; }
          rr = wq.rp[i]; rri = 1.0 / rr; lo = wq.lp[i]; hi = wq.up[i];
          mi11 = wq.Minv[3 * i]; mi12 = wq.Minv[3 * i + 1]; mi22 = wq.Minv[3 * i + 2];
          s1 = wq.s[i]; zs1 = wq.zs[i]; ys1 = wq.ys[i];
          sl1 = wq.sl[i]; bs1 = wq.bs[i]; rs1 = wq.rs[i]; rsi1 = 1.0 / rs1; cd1 = f.cpi * wq.Ds[i]; us1 = OSQP_INFTY * wq.Es[i]; hs1 = wq.hs[i];
          if (EQS && eq) {
            const int i2 = ms + i;
            s2 = wq.s[i2]; zs2 = wq.zs[i2]; ys2 = wq.ys[i2];
            sl2 = wq.sl[i2]; bs2 = wq.bs[i2]; rs2 = wq.rs[i2]; rsi2 = 1.0 / rs2; cd2 = f.cpi * wq.Ds[i2]; us2 = OSQP_INFTY * wq.Es[i2]; hs2 = wq.hs[i2];
          }
          const int so = __ldg(SS.row_soff + (i)), go = __ldg(SS.row_goff + (i)), wd = __ldg(SS.row_w + (i));
          if (DENSE) {
#pragma unroll
            for (int k = 0; k < NEC; k++)
              if (k < n) ec[k] = wq.Js[so + k];
          } else
#pragma unroll
          for (int k = 0; k < SCO_EN; k++)
            if (k < wd) { ec[k] = wq.Js[so + k]; ea[k] = f.o_xt2 + __ldg(SS.jcol_g + (go + k)); }
        }
      }
      const int K3 = f.K3, j3 = f.j3, s3 = f.s3, c0 = f.c0, c1 = f.c1;
      const bool p3_active = f.p3_active != 0;
      const int o_Sm = f.o_Sm, o_xt = f.o_xt, o_xt2 = f.o_xt2, o_ps = f.o_ps, o_wl = f.o_wl, o_wp = f.o_wp;
      const bool has_pen = f.has_pen != 0;
      // ---- iterations up to (and including) the next tested / last one that needs the out-of-line test: no call inside
      bool leave = false, tested = false;
      while (!leave) {
        iter++;
#ifdef SCO_TIMING
        long long tph = clock64();
#endif
        // ---- P1: row weights w = rho z - y ; slack elimination (registers -> wl / wp)
        if (ROLE == 1 && act) {
          sco_smem[o_wl + id] = rr * z - y;
        } else if (PEN && act) {
          const double wpen = rr * z - y;
          const double kr = kd * rr;
          const double r1 = sigma * s1 - cd1 + kd * sl1 * wpen + bs1 * (rs1 * zs1 - ys1);
          if (EQS && eq) {
            const double r2 = sigma * s2 - cd2 + kd * sl2 * wpen + bs2 * (rs2 * zs2 - ys2);
            g1 = mi11 * r1 + mi12 * r2;
            g2 = mi12 * r1 + mi22 * r2;
            sco_smem[o_wp + id] = kd * wpen - kr * (sl1 * g1 + sl2 * g2);
          } else {
            g1 = mi11 * r1;
            sco_smem[o_wp + id] = kd * wpen - kr * sl1 * g1;
          }
        }
        sync();
        SCO_PH(0)
        // ---- P2: reduced right-hand side (variables)
        if (ROLE == 0 && act) {
          double acc = 0.0, accp = 0.0;
          if (DENSE) {  // J' w over all penalty rows: four chains, operands by broadcast 128-bit loads
            double b0 = 0.0, b1 = 0.0, b2 = 0.0, b3 = 0.0;
            const double2 *wv = sco_smem2 + (o_wp >> 1);
#pragma unroll
            for (int k = 0; k < NEC; k += 4) {
              if (k < f.m_nl) {  // team-uniform; wp is zero-padded to a multiple of four
                const double2 w01 = wv[k >> 1], w23 = wv[(k >> 1) + 1];
                b0 = fma(ec[k], w01.x, b0);
                b1 = fma(ec[k + 1], w01.y, b1);
                b2 = fma(ec[k + 2], w23.x, b2);
                b3 = fma(ec[k + 3], w23.y, b3);
              }
            }
            accp = (b0 + b2) + (b1 + b3);
          } else
#pragma unroll
          for (int k = 0; k < SCO_EH; k++) {
            acc = fma(ec[k], sco_smem[ea[k]], acc);
            accp = fma(ec[SCO_EH + k], sco_smem[ea[SCO_EH + k]], accp);
          }
          if (has_pen) acc += accp;
          sco_smem[o_xt + id] = sigma * x - qh + bx * (rb * zb - yb) + acc;
        }
        sync();
        SCO_PH(1)
        // ---- P3: partial sums of x~ = S^-1 rhs (every thread of the team, whatever its role)
        if (p3_active) {
          double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
          int cc = c0;
          const double *Sc = sco_smem + o_Sm + j3;
          const double2 *xv = sco_smem2 + (o_xt >> 1);
#pragma unroll 2
          for (; cc + 3 < c1; cc += 4) {
            const double q0 = Sc[cc * n], q1 = Sc[(cc + 1) * n], q2 = Sc[(cc + 2) * n], q3 = Sc[(cc + 3) * n];
            const double2 x01 = xv[cc >> 1], x23 = xv[(cc >> 1) + 1];  // c0 is a multiple of 4
            a0 = fma(q0, x01.x, a0);
            a1 = fma(q1, x01.y, a1);
            a2 = fma(q2, x23.x, a2);
            a3 = fma(q3, x23.y, a3);
          }
          for (; cc < c1; cc++) a0 = fma(Sc[cc * n], sco_smem[o_xt + cc], a0);
          sco_smem[o_ps + s3 * n + j3] = (a0 + a2) + (a1 + a3);
        }
        sync();
        SCO_PH(2)
        // ---- P4a: x~, x and the box rows (variables)
        if (ROLE == 0 && act) {
          double xtil = sco_smem[o_ps + id];
          for (int k = 1; k < K3; k++) xtil += sco_smem[o_ps + k * n + id];
          sco_smem[o_xt2 + id] = xtil;
          const double xo = x;
          const double xn = alpha * xtil + oma * xo;
          x = xn;
          const double zt = bx * xtil;
          const double vv = alpha * zt + oma * zb;
          const double zn = clampd(vv + yb * rbi, lb, ub);
          const double dy = rb * (vv - zn);
          yb += dy;
          zb = zn;
          d0 = xn - xo; d1 = dy;
        }
        sync();
        // ---- P4b: rows
        if ((ROLE == 1 || PEN) && act) {
          double t = 0.0;
          if (DENSE && PEN) {  // J x~ over all variables
            double b0 = 0.0, b1 = 0.0, b2 = 0.0, b3 = 0.0;
            const double2 *xv2 = sco_smem2 + (o_xt2 >> 1);
#pragma unroll
            for (int k = 0; k < NEC; k += 4) {
              if (k < n) {  // xt2 is zero-padded to a multiple of four
                const double2 x01 = xv2[k >> 1], x23 = xv2[(k >> 1) + 1];
                b0 = fma(ec[k], x01.x, b0);
                b1 = fma(ec[k + 1], x01.y, b1);
                b2 = fma(ec[k + 2], x23.x, b2);
                b3 = fma(ec[k + 3], x23.y, b3);
              }
            }
            t = (b0 + b2) + (b1 + b3);
          } else
#pragma unroll
          for (int k = 0; k < SCO_EN; k++) t = fma(ec[k], sco_smem[ea[k]], t);
          double zt = t;
          if (PEN) {
            {
              const double stil = g1 - hs1 * t;
              zt += sl1 * stil;
              const double so_ = s1;
              const double sn = alpha * stil + oma * so_;
              s1 = sn;
              const double zts = bs1 * stil;
              const double vs = alpha * zts + oma * zs1;
              const double zns = clampd(vs + ys1 * rsi1, 0.0, us1);
              const double dys = rs1 * (vs - zns);
              ys1 += dys;
              zs1 = zns;
              d1 = sn - so_; d2 = dys;
            }
            if (EQS && eq) {
              const double stil = g2 - hs2 * t;
              zt += sl2 * stil;
              const double so_ = s2;
              const double sn = alpha * stil + oma * so_;
              s2 = sn;
              const double zts = bs2 * stil;
              const double vs = alpha * zts + oma * zs2;
              const double zns = clampd(vs + ys2 * rsi2, 0.0, us2);
              const double dys = rs2 * (vs - zns);
              ys2 += dys;
              zs2 = zns;
              d3 = sn - so_; d4 = dys;
            }
          }
          const double vv = alpha * zt + oma * z;
          const double zn = clampd(vv + y * rri, lo, hi);
          const double dy = rr * (vv - zn);
          y += dy;
          z = zn;
          d0 = dy;
        }
        SCO_PH(3)
        if (iter == next_check) {
          next_check += chk;
          tested = true;
          leave = true;
          if (INL && f.inline_test && iter < max_iter) {
            // ---- the termination test of check(), from the registers: same quantities, same arithmetic, one mixed
            // reduction.  Only when it ends the solve -- or a certificate's first stage holds -- the iterates go to
            // shared memory and check() itself decides (out of line: its code is cold, 17-36 k cycles a visit).
            sync();  // P4b of the row roles still reads x~ from xt2
            if (act) {
              if (ROLE == 0) { sco_smem[o_xt2 + id] = x; sco_smem[o_xt + id] = k1 * x; }
              else if (ROLE == 1) sco_smem[o_wl + id] = y;
              else if (PEN) sco_smem[o_wp + id] = kd * y;
            }
            sync();
            double v[6] = {0, 0, 0, 0, 0, 0};
            double sums[2] = {0.0, 0.0};
            if (act) {
              if (ROLE == 1 || PEN) {
                double ax = 0.0;
#pragma unroll
                for (int k = 0; k < SCO_EN; k++) ax = fma(ec[k], sco_smem[ea[k]], ax);
                if (ROLE == 1) {
                  qp_term_row(v, sums, ax, z, k0, d0, lo, hi, 1.0);
                } else {
                  ax = ax + sl1 * s1;
                  if (EQS && eq) ax += sl2 * s2;
                  qp_term_row(v, sums, ax, z, k0, d0, lo, hi, kd);
                  qp_term_slack(v, sums, bs1 * s1, zs1, k1, k2s, cd1, kd * sl1 * y + bs1 * ys1, d2);
                  qp_term_dx(v, sums, k2s, d1, cd1);
                  if (EQS && eq) {
                    qp_term_slack(v, sums, bs2 * s2, zs2, k3, k4, cd2, kd * sl2 * y + bs2 * ys2, d4);
                    qp_term_dx(v, sums, k4, d3, cd2);
                  }
                }
              } else if (ROLE == 0) {
                double px = 0.0;
#pragma unroll
                for (int k = 0; k < 4; k++) px = fma(pq[k], sco_smem[pa[k]], px);
                px *= f.c * k1;
                double acc = 0.0, accp = 0.0;
#pragma unroll
                for (int k = 0; k < SCO_EH; k++) {
                  acc = fma(ec[k], sco_smem[ea[k]], acc);
                  accp = fma(ec[SCO_EH + k], sco_smem[ea[SCO_EH + k]], accp);
                }
                if (has_pen) acc += accp;
                qp_term_var(v, sums, bx * x, zb, k0, k1, qh, px, acc + bx * yb, d1, lb, ub, d0);
              }
            }
            Team<TEAM>::template reduce_mixed<6, 2>(v, sums, Sh{f.o_red});
            double pri_res, dua_res;
            int cert;
            if (qp_termination(v[0], v[1], v[2], v[3], v[4], sums[0], v[5], sums[1], f.c, 1.0 / f.c, f.eps_abs, f.eps_rel,
                               f.eps_pinf, f.eps_dinf, false, pri_res, dua_res, cert) == 0 && cert == 0) {
              leave = false;
              tested = false;
            }
            SCO_PH(4)
          }
        } else if (iter >= max_iter) {
          leave = true;
        }
      }
      // ---- the tested (and not waved through) or the last iteration.  Iterates (+ deltas) -> shared memory, then check().
      const int can_check = tested ? 1 : 0, store_d = tested || iter >= max_iter ? 1 : 0;
#ifdef SCO_TIMING
      long long tph = clock64();
#endif
      if (ROLE == 0) status = fast_flush<0>(id, act, 0, can_check, store_d, res, x, zb, yb, 0, 0, 0, 0, 0, d0, d1, 0, 0, 0);
      else if (ROLE == 1) status = fast_flush<1>(id, act, 0, can_check, store_d, res, z, y, 0, 0, 0, 0, 0, 0, d0, 0, 0, 0, 0);
      else if (PEN) status = fast_flush<2>(id, act, eq, can_check, store_d, res, z, y, s1, zs1, ys1, s2, zs2, ys2, d0, d1, d2, d3, d4);
      else status = fast_flush<3>(id, 0, 0, can_check, store_d, res, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0);
      checked = can_check != 0;
      SCO_PH(4)
      if (status != 0) break;
    }
    iter_out = status != 0 ? iter : max_iter + 1;  // generic_loop's convention: the loop variable after the loop
    checked_out = checked;
    return status;
  }

  // Warm start of the thread-per-entity loop (sco_settings.warm_start; OSQP's osqp_warm_start): the iterate arrays
  // hold the UNSCALED x, s and duals the previous QP of this team ended with (solve() unscales them when the setting
  // is on); x^ = D^-1 x, y^ = c E^-1 y, z^ = A^ x^ with the scaling of this QP.
  __device__ __noinline__ void warm_init() {
    SCO_QP_LOCALS
    for (int j = tid; j < n; j += TEAM) {
      const double xh = W_x[j] / W_D[j];
      W_x[j] = xh;
      W_zb[j] = W_bx[j] * xh;
      W_yb[j] = c * W_yb[j] / W_Eb[j];
    }
    for (int i = tid; i < m_nl; i += TEAM)
      for (int k2 = 0; k2 <= __ldg(S.row_eq + (i)); k2++) {
        const int si = k2 * ms + i;
        const double sh = W_s[si] / W_Ds[si];
        W_s[si] = sh;
        W_zs[si] = W_bs[si] * sh;
        W_ys[si] = c * W_ys[si] / W_Es[si];
      }
    sync();
    for (int r = tid; r < m_lin; r += TEAM) {
      W_zl[r] = lin_row_dot(r, W_x);
      W_yl[r] = c * W_yl[r] / W_El[r];
    }
    for (int i = tid; i < m_nl; i += TEAM) {
      double ax = pen_row_dot(i, W_x) + W_sl[i] * W_s[i];
      if (__ldg(S.row_eq + (i))) ax += W_sl[ms + i] * W_s[ms + i];
      W_zp[i] = ax;
      W_yp[i] = c * (W_yp[i] / a.kd) / W_Ep[i];  // the stored dual is the sum over the kd copies of the row
    }
    sync();
  }

  // roles start on warp boundaries: ceil32(n) variable lanes, ceil32(m_lin) linear-row lanes, ceil32(m_nl) penalty-row lanes
  // ... and every row of A has at most SCO_EN entries, every column at most SCO_EH from linear and SCO_EH from
  // penalty rows (S.fast_ok, checked once by sco_create)
  __device__ __forceinline__ bool fast_fits() const {
    return !S.sws && (S.fast_ok || (S.fast_dense && m_lin == 0)) && ((n + 31) & ~31) + ((m_lin + 31) & ~31) + ((m_nl + 31) & ~31) <= TEAM;
  }

  __device__ __noinline__ int fast_loop(int &iter_out, bool &checked_out, QPResult &res) {
    const int n = this->n, m_lin = this->m_lin, m_nl = this->m_nl, tid = this->tid;
    const QPW &wq = this->w;
    const int nV = (n + 31) & ~31, nL = (m_lin + 31) & ~31, nP = (m_nl + 31) & ~31;
    FastCtx f;
    const int role = tid < nV ? 0 : tid < nV + nL ? 1 : tid < nV + nL + nP ? 2 : 3;
    f.id = role == 0 ? tid : role == 1 ? tid - nV : tid - nV - nL;
    f.act = role == 0 ? f.id < n : role == 1 ? f.id < m_lin : role == 2 ? f.id < m_nl : 0;
    f.n = n; f.ms = this->ms;
    // S^-1 rhs: thread (j3, s3) sums the columns [c0, c1) of row j3 (S^-1 is symmetric: column access)
    f.K3 = (TEAM / n) < 4 ? (TEAM / n) : 4;
    f.j3 = tid % n;
    f.s3 = tid / n;
    const int CS = ((n + f.K3 - 1) / f.K3 + 3) & ~3;
    f.c0 = f.s3 * CS;
    f.c1 = (f.s3 + 1) * CS < n ? (f.s3 + 1) * CS : n;
    f.p3_active = f.s3 < f.K3 && f.c0 < n;
    f.o_Sm = wq.Sm.off; f.o_xt = wq.xt.off; f.o_xt2 = wq.xt2.off; f.o_ps = wq.ps.off; f.o_wl = wq.wl.off; f.o_wp = wq.wp.off;
    f.max_iter = this->st.max_iter; f.chk = this->st.check_termination; f.has_pen = m_nl != 0; f.m_nl = m_nl;
    f.sigma = this->st.sigma; f.alpha = this->st.alpha; f.kd = this->a.kd; f.cpi = this->c * this->a.pi;
    f.o_red = wq.red.off; f.c = this->c;
    f.eps_abs = this->st.eps_abs; f.eps_rel = this->st.eps_rel; f.eps_pinf = this->st.eps_prim_inf; f.eps_dinf = this->st.eps_dual_inf;
    // in-loop test: the objective matrix has at most four entries per column (or is the closest-point 2 I)
    f.inline_test = (this->a.closest || this->S.p_narrow) && !this->a.has_hq;
    for (int e = tid; e < f.K3 * n; e += TEAM) wq.ps[e] = 0.0;  // segments beyond n contribute exact zeros
    // ADMM starts from x = z = y = 0 (osqp_utils.py:195 builds a new OSQP object per call) unless the opt-in warm
    // start applies; fast_role reads its iterates from these arrays
    if (this->a.warm) warm_init();
    else {
    for (int j = tid; j < n; j += TEAM) { wq.x[j] = 0.0; wq.zb[j] = 0.0; wq.yb[j] = 0.0; }
    for (int r = tid; r < m_lin; r += TEAM) { wq.zl[r] = 0.0; wq.yl[r] = 0.0; }
    for (int i = tid; i < m_nl; i += TEAM) {
      wq.zp[i] = 0.0; wq.yp[i] = 0.0;
      wq.s[i] = 0.0; wq.zs[i] = 0.0; wq.ys[i] = 0.0;
      if (__ldg(this->S.row_eq + (i))) { wq.s[f.ms + i] = 0.0; wq.zs[f.ms + i] = 0.0; wq.ys[f.ms + i] = 0.0; }
    }
    }
    // the dense variants read their operands in groups of four: pad wp / xt2 with zeros (the arrays behind them are
    // rewritten before they are read)
    if (tid < 4) { wq.wp[m_nl + tid] = 0.0; wq.xt2[n + tid] = 0.0; }
    sync();
    if constexpr (TEAM <= 256) {  // the dense variants need ~200 registers: teams that have them
      if (!this->S.fast_ok) {
        f.inline_test = 0;  // team-uniform: the idle role below is the <3, 0> instantiation and must not test alone
        if (role == 0) return fast_role<0, 1>(f, iter_out, checked_out, res);
        if (role == 2) return this->S.nsl == 2 ? fast_role<4, 1>(f, iter_out, checked_out, res) : fast_role<2, 1>(f, iter_out, checked_out, res);
        return fast_role<3, 0>(f, iter_out, checked_out, res);
      }
    }
    if (role == 0) return fast_role<0, 0>(f, iter_out, checked_out, res);
    if (role == 1) return fast_role<1, 0>(f, iter_out, checked_out, res);
    if (role == 2) return this->S.nsl == 2 ? fast_role<4, 0>(f, iter_out, checked_out, res) : fast_role<2, 0>(f, iter_out, checked_out, res);
    return fast_role<3, 0>(f, iter_out, checked_out, res);
  }

  // ================================================================== the ADMM loop
  // On return W_x (user variables) and W_s (slacks) hold the UNSCALED solution.
  // generic shared-memory ADMM loop; returns the status (0 = max_iter reached without a verdict)
  __device__ __noinline__ int generic_loop(int &iter_out, bool &checked_out, QPResult &res) {
    SCO_QP_LOCALS
    const double sigma = st.sigma, alpha = st.alpha, oma = 1.0 - st.alpha;
    for (int j = tid; j < n; j += TEAM) { W_x[j] = 0.0; W_zb[j] = 0.0; W_yb[j] = 0.0; }
    for (int r = tid; r < m_lin; r += TEAM) { W_zl[r] = 0.0; W_yl[r] = 0.0; }
    for (int i = tid; i < m_nl; i += TEAM) {
      W_zp[i] = 0.0; W_yp[i] = 0.0;
      for (int k2 = 0; k2 <= __ldg(S.row_eq + (i)); k2++) {
        const int si = k2 * ms + i;
        W_s[si] = 0.0; W_zs[si] = 0.0; W_ys[si] = 0.0;
      }
    }
    sync();
    const double cpi = c * a.pi;
    int interval = st.adaptive_rho_interval;
    if (st.adaptive_rho && interval == 0) interval = st.check_termination ? 4 * st.check_termination : 100;
    int iter, status = 0;
    bool checked = false;
    for (iter = 1; iter <= st.max_iter; iter++) {
      const bool can_check = st.check_termination && (iter % st.check_termination == 0);
      const bool do_rho = st.adaptive_rho && interval && (iter % interval == 0);
      const bool want_delta = can_check || do_rho;
      // the deltas of the last iteration also feed the final tests after the loop (QPSolver::solve)
      const bool keep_delta = want_delta || iter == st.max_iter;
#ifdef SCO_TIMING
      long long tph = clock64();
#endif
      // ---- P1: row weights  w = rho z - y, slack elimination
      for (int r = tid; r < m_lin; r += TEAM) W_wl[r] = W_rl[r] * W_zl[r] - W_yl[r];
      for (int i = tid; i < m_nl; i += TEAM) {
        const double wpen = W_rp[i] * W_zp[i] - W_yp[i];
        const double kr = a.kd * W_rp[i];
        const double r1 = sigma * W_s[i] - cpi * W_Ds[i] + a.kd * W_sl[i] * wpen +
                          W_bs[i] * (W_rs[i] * W_zs[i] - W_ys[i]);
        if (__ldg(S.row_eq + (i))) {
          const int i2 = ms + i;
          const double r2 = sigma * W_s[i2] - cpi * W_Ds[i2] + a.kd * W_sl[i2] * wpen +
                            W_bs[i2] * (W_rs[i2] * W_zs[i2] - W_ys[i2]);
          const double g1 = W_Minv[3 * i] * r1 + W_Minv[3 * i + 1] * r2;
          const double g2 = W_Minv[3 * i + 1] * r1 + W_Minv[3 * i + 2] * r2;
          W_gs[i] = g1; W_gs[i2] = g2;
          W_wp[i] = a.kd * wpen - kr * (W_sl[i] * g1 + W_sl[i2] * g2);
        } else {
          const double g1 = W_Minv[3 * i] * r1;
          W_gs[i] = g1;
          W_wp[i] = a.kd * wpen - kr * W_sl[i] * g1;
        }
      }
      sync();
      SCO_PH(0)
      // ---- P2: reduced right-hand side
      for (int j = tid; j < n; j += TEAM)
        W_xt[j] = sigma * W_x[j] - W_qh[j] + W_bx[j] * (W_rb[j] * W_zb[j] - W_yb[j]) +
                  gatherAT(j, W_wl, W_wp);
      sync();
      SCO_PH(1)
      // ---- P3: x~ = S^-1 rhs ; x, bound rows
      for (int j = tid; j < n; j += TEAM) {
        // four independent chains, loads issued ahead of the FMAs (a two-chain loop waited for every
        // shared-memory round trip: 28 cycles per term)
        double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
        int k = 0;
        if (w.Sg) {  // S^-1 streamed from this team's global workspace (coalesced over j; same chains, same order)
          const double *Sg = w.Sg + j;
#pragma unroll 4
          for (; k + 3 < n; k += 4) {
            const double s0 = __ldcg(Sg + (size_t)k * n), s1 = __ldcg(Sg + (size_t)(k + 1) * n),
                         s2 = __ldcg(Sg + (size_t)(k + 2) * n), s3 = __ldcg(Sg + (size_t)(k + 3) * n);
            acc0 = fma(s0, W_xt[k], acc0);
            acc1 = fma(s1, W_xt[k + 1], acc1);
            acc2 = fma(s2, W_xt[k + 2], acc2);
            acc3 = fma(s3, W_xt[k + 3], acc3);
          }
          for (; k < n; k++) acc0 = fma(__ldcg(Sg + (size_t)k * n), W_xt[k], acc0);
        } else {
#pragma unroll 2
        for (; k + 3 < n; k += 4) {
          const double s0 = W_Sm[k * n + j], s1 = W_Sm[(k + 1) * n + j], s2 = W_Sm[(k + 2) * n + j], s3 = W_Sm[(k + 3) * n + j];
          acc0 = fma(s0, W_xt[k], acc0);
          acc1 = fma(s1, W_xt[k + 1], acc1);
          acc2 = fma(s2, W_xt[k + 2], acc2);
          acc3 = fma(s3, W_xt[k + 3], acc3);
        }
        for (; k < n; k++) acc0 = fma(W_Sm[k * n + j], W_xt[k], acc0);
        }
        acc0 += acc2;
        acc1 += acc3;
        const double xtil = acc0 + acc1;
        W_xt2[j] = xtil;
        const double xo = W_x[j];
        const double xn = alpha * xtil + oma * xo;
        W_x[j] = xn;
        const double zt = W_bx[j] * xtil;
        const double vv = alpha * zt + oma * W_zb[j];
        const double zn = clampd(vv + W_yb[j] / W_rb[j], W_lb[j], W_ub[j]);
        const double dy = W_rb[j] * (vv - zn);
        W_yb[j] += dy;
        W_zb[j] = zn;
        if (keep_delta) { W_dxv[j] = xn - xo; W_dyb[j] = dy; }
      }
      sync();
      SCO_PH(2)
      // ---- P4: rows
      for (int r = tid; r < m_lin; r += TEAM) {
        const double zt = lin_row_dot(r, W_xt2);
        const double vv = alpha * zt + oma * W_zl[r];
        const double zn = clampd(vv + W_yl[r] / W_rl[r], W_ll[r], W_ul[r]);
        const double dy = W_rl[r] * (vv - zn);
        W_yl[r] += dy;
        W_zl[r] = zn;
        if (keep_delta) W_dyl[r] = dy;
      }
      for (int i = tid; i < m_nl; i += TEAM) {
        const double t = pen_row_dot(i, W_xt2);
        const int eq = __ldg(S.row_eq + (i));
        double zt = t;
        for (int k2 = 0; k2 <= eq; k2++) {
          const int si = k2 * ms + i;
          const double stil = W_gs[si] - W_hs[si] * t;
          zt += W_sl[si] * stil;
          const double so = W_s[si];
          const double sn = alpha * stil + oma * so;
          W_s[si] = sn;
          const double zts = W_bs[si] * stil;
          const double vs = alpha * zts + oma * W_zs[si];
          const double zns = clampd(vs + W_ys[si] / W_rs[si], 0.0, OSQP_INFTY * W_Es[si]);
          const double dys = W_rs[si] * (vs - zns);
          W_ys[si] += dys;
          W_zs[si] = zns;
          if (keep_delta) { W_dss[si] = sn - so; W_dys[si] = dys; }
        }
        const double vv = alpha * zt + oma * W_zp[i];
        const double zn = clampd(vv + W_yp[i] / W_rp[i], W_lp[i], W_up[i]);
        const double dy = W_rp[i] * (vv - zn);
        W_yp[i] += dy;
        W_zp[i] = zn;
        if (keep_delta) W_dyp[i] = dy;
      }
      SCO_PH(3)
      checked = false;
      if (want_delta) {
        sync();
        double sc[4];
        status = check(0, res.pri_res, res.dua_res, do_rho ? sc : nullptr);
        checked = can_check;
        if (can_check && status != 0) break;
        status = 0;
        if (do_rho) {
          double pri = sc[0] / (sc[1] + 1e-10);
          double dua = sc[2] / (sc[3] + 1e-10);
          double rn = rho * sqrt(pri / (dua + 1e-10));
          rn = fmin(fmax(rn, OSQP_RHO_MIN), OSQP_RHO_MAX);
          if (rn > rho * 5.0 || rn < rho / 5.0) {
            this->rho = rn;
            set_rho();
            rho = this->rho;
            if (w.Sg) assemble_and_invert<true>(true); else assemble_and_invert<false>(true);
          }
        }
        sync();
      }
      SCO_PH(4)
    }
    iter_out = iter;
    checked_out = checked;
    return status;
  }

  __device__ __noinline__ QPResult solve() {
    // dense hinge-only structures: the specialised two-warp solve (same iteration, sco_dense.cuh).
    // The size table is kept in sync with sco_create (sco_abi.cu).
    if constexpr (TEAM == 64 && DK != 0) {
      if (!st.force_generic && !st.adaptive_rho && a.use_pen) {
        if constexpr (DK == 1) return dense_qp_solve<8, 6>(S, st, w, a);
        else if constexpr (DK == 2) return dense_qp_solve<12, 16>(S, st, w, a);
        else if constexpr (DK == 3) return dense_qp_solve<20, 30>(S, st, w, a);
        else return dense_qp_solve<32, 32>(S, st, w, a);
      }
    }
#ifdef SCO_TIMING
    const long long t_begin = clock64();
#endif
    if (w.Sg) load_and_scale<true>(); else load_and_scale<false>();
#ifdef SCO_TIMING
    const long long t_scaled = clock64();
#endif
    rho = st.rho;
    set_rho();
    if (w.Sg) assemble_and_invert<true>(false); else assemble_and_invert<false>(false);
    QPResult res;
    res.status = 0; res.iters = 0; res.pri_res = 0.0; res.dua_res = 0.0;
#ifdef SCO_TIMING
    res.cyc_check = 0;
    for (int k = 0; k < 5; k++) res.cyc_c[k] = 0;
    res.cyc_setup = clock64() - t_begin;
    res.cyc_scale = t_scaled - t_begin;
    const long long t_loop = clock64();
#endif
    int iter = 0, status = 0;
    bool checked = false;
    // one thread per entity when the team is large enough (sco_create sizes it so); adaptive rho re-factorises
    // inside the loop and stays on the shared-memory loop
    if (fast_fits() && !st.adaptive_rho && !st.force_generic) status = fast_loop(iter, checked, res);
    else status = generic_loop(iter, checked, res);
#ifdef SCO_TIMING
    res.cyc_loop = clock64() - t_loop;
#endif
    if (status == 0) {
      iter = st.max_iter;
      if (!checked) {
        sync();
        status = check(0, res.pri_res, res.dua_res, nullptr);
      }
      if (status == 0) {
        sync();
        status = check(1, res.pri_res, res.dua_res, nullptr);
        if (status == 0) status = -2;
      }
    }
    sync();
    // unscale
    for (int j = tid; j < n; j += TEAM) w.x[j] *= w.D[j];
    for (int i = tid; i < m_nl; i += TEAM)
      for (int k2 = 0; k2 <= __ldg(S.row_eq + (i)); k2++) w.s[k2 * ms + i] *= w.Ds[k2 * ms + i];
    if (st.warm_start) {  // duals too (y = E y^ / c), for the warm start of this team's next QP (warm_init)
      const double ci = 1.0 / c;
      for (int j = tid; j < n; j += TEAM) w.yb[j] *= w.Eb[j] * ci;
      for (int r = tid; r < m_lin; r += TEAM) w.yl[r] *= w.El[r] * ci;
      for (int i = tid; i < m_nl; i += TEAM) {
        w.yp[i] *= a.kd * w.Ep[i] * ci;
        for (int k2 = 0; k2 <= __ldg(S.row_eq + (i)); k2++) w.ys[k2 * ms + i] *= w.Es[k2 * ms + i] * ci;
      }
    }
    sync();
    res.status = status;
    res.iters = iter;
    return res;
  }
};
