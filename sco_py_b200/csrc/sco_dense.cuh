// sco_dense.cuh -- the penalty QP of a dense hinge-only structure (one QUADFORM block of LEq rows,
// no linear rows: BASELINE.json configs[3], the headline workload), solved by a team of TWO warps
// with every size a compile-time bound.
//
// Same algorithm, same scaling, same termination tests as the generic QPSolver of sco_qp.cuh (the
// OSQP 0.6.2 iteration of SURVEY.md Appendix B as driven by sco_py/sco_osqp/osqp_utils.py:195-216);
// what is specialised is the machine mapping:
//   * warp 0, lane i = penalty row i with its slack;  warp 1, lane j = variable j with its box row.
//     Everything that is "per row" or "per variable" (scaling factors, bounds, rho, iterates) lives
//     in that lane's registers from the first Ruiz pass to the unscaling of the solution.
//   * the working set has a compile-time layout at the start of dynamic shared memory (DenseL) and is
//     addressed with 32-bit shared-window addresses: no offset table behind a generic pointer, no
//     index arrays in global memory -- in the generic code every shared store was followed by
//     re-loads of both, and the kernel was 640 KB of SASS that missed the instruction cache in
//     every rarely-executed block.
//   * one ADMM iteration = one (n+m)-term dot product of the lane's register-resident row of
//         [ S^-1  K ; K'  G ],   K = S^-1 J',  G = J S^-1 J'
//     with the exchange vector (c, wp) read by broadcast 128-bit shared loads, the lane-local
//     update, one 8-byte store, one barrier.
//   * the termination test is one combined reduction (redux.sync on the bit patterns of the
//     non-negative norms) and one exchange between the two warps.
#pragma once
#include "sco_device.cuh"


__device__ __forceinline__ double lds_f64(uint32_t addr) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
// max(v, 0) through the sign bit (integer pipe; a double compare-and-select is four times the latency)
__device__ __forceinline__ double relu_bits(double v) {
  const int hi = __double2hiint(v), msk = ~(hi >> 31);
  return __hiloint2double(hi & msk, __double2loint(v) & msk);
}
// maximum of two non-negative doubles (3 instructions; fmax() costs 7 with its NaN fix-up)
__device__ __forceinline__ double max_nn(double a, double b) { return a > b ? a : b; }

// lane-constant view of the scaled QP (kept in shared memory, DL::LA; the ADMM loop holds only the
// first five in registers)
struct DenseLane {
  double u0, u1, u2, lo, hi, r0, r1, r2, e0, e1, e2, rbj;
  // variable lane: u0=q^ u1=bx u2=rho_j lo/hi=box   r0=1/Eb r1=1/D        e0=Eb e1=D
  // row lane     : u0=c pi Ds u1=sl u2=bs lo=kd sl hi=up r0=1/Ep r1=1/Es r2=1/Ds e0=Ep e1=Es e2=Ds
};
// proj_dy (sco_qp.cuh) with selects instead of branches, the same value in every case: l and u differ
// from lane to lane, and a branch would split the basic block the dense loop overlaps with an ADMM
// iteration (the generic loops keep the branches, which cost them fewer registers)
__device__ __forceinline__ double proj_dy_sel(double dy, double l, double u) {
  const bool u_inf = u > OSQP_INFTY * OSQP_MIN_SCALING, l_inf = l < -OSQP_INFTY * OSQP_MIN_SCALING;
  const double upper_only = l_inf ? 0.0 : fmin(dy, 0.0), lower_only = l_inf ? fmax(dy, 0.0) : dy;
  return u_inf ? upper_only : lower_only;
}
template <bool B> struct BoolC { static constexpr bool value = B; };  // a compile-time flag passed to a generic lambda
struct DenseState {
  double p0, z0, y0, s, zs, ys;   // (x, zb, yb) or (-, zp, yp, s, zs, ys)
  double pp0, py0, ps, pys;       // the same before the last iteration
};

template <int NP, int MP>
__device__ __forceinline__ uint32_t dense_la(const uint32_t sb, const bool rowwarp, const int lane, const int k) {
  using DL = DenseL<NP, MP>;
  return sb + 8u * (DL::LA + ((rowwarp ? 0 : DL::NLA) + k) * 32 + lane);
}
template <int NP, int MP>
__device__ __forceinline__ double dense_sc(const uint32_t sb, const int k) {
  return lds_f64(sb + 8u * (DenseL<NP, MP>::Sc + k));
}

// ---- termination test (OSQP check_termination on the unscaled residuals), both warps: the dense
// layout's norms and certificate first stages, decided by qp_termination (sco_qp.cuh).
//
// First half, one warp (ROW: the penalty-row warp): this lane's terms of state X (dense_test_terms),
// then their reduction over the warp, which lane 0 stores into the warp's slots of DL::Red
// (dense_test_publish).  Expects Xs / Ys of state X published and a barrier passed.  The lane passes
// the five constants its ADMM loop keeps in registers; the rest comes from DL::LA / DL::Sc.  Nothing in
// it depends on the ADMM iterates in registers, so the dense loop runs it beside the next iteration
// (dense_qp_solve) and one barrier publishes both.
struct DenseTestTerms {
  double v0, v12, v3, v456, nvp, nvd, s0, s1, mvs, rej;
};
template <int NP, int MP, bool ROW>
__device__ __forceinline__ DenseTestTerms dense_test_terms(const uint32_t sb, const int lane, const double u0,
                                                           const double u1, const double u2, const double lo,
                                                           const double hi, const DenseState &X, const bool tail) {
  using DL = DenseL<NP, MP>;
  constexpr int LDJ = DL::LDJ;
  const double r0 = lds_f64(dense_la<NP, MP>(sb, ROW, lane, 5)), r1 = lds_f64(dense_la<NP, MP>(sb, ROW, lane, 6));
  const double e0 = lds_f64(dense_la<NP, MP>(sb, ROW, lane, 8)), e1 = lds_f64(dense_la<NP, MP>(sb, ROW, lane, 9));
  const double kd = dense_sc<NP, MP>(sb, 8);
  double v0, v12, v3, v456, nvp, nvd, s0, s1;
  // Tail mode (the launch's queue is drained, this problem is on the critical path): lane-local parts of
  // the SECOND stage of the certificates that can only refute them -- mvs = slack columns of |A' dy| / D
  // (primal), rej = how far A dx leaves the recession cone on slack-bound and box rows (dual).  The first
  // stage holds in 15-22 % of the tests although these QPs are feasible and bounded; with the two values
  // almost none of them needs dense_certificates (a lone problem runs 7 % faster; on a full machine the
  // extra instructions cost 4 %, hence only in tail mode -- profiles/README.md).
  double mvs = 0.0, rej = 0.0;
  if (ROW) {
    const double r2 = lds_f64(dense_la<NP, MP>(sb, true, lane, 7)), e2 = lds_f64(dense_la<NP, MP>(sb, true, lane, 10));
    // lanes beyond the padded row / column count read row / column 0: what lies behind the matrices may
    // be stale shared memory (a NaN pattern times their zero scale factor would still be NaN)
    const uint32_t jr = sb + 8u * (DL::Js + (lane < MP ? lane : 0) * LDJ), xs = sb + 8u * DL::Xs;
    double a0 = 0.0, a1 = 0.0;
#pragma unroll
    for (int k = 0; k < NP; k += 2) {
      const double2 xk = lds_v2(xs + 8u * k);
      a0 = fma(lds_f64(jr + 8u * k), xk.x, a0);
      if (k + 1 < NP) a1 = fma(lds_f64(jr + 8u * k + 8u), xk.y, a1);
    }
    const double ax = (a0 + a1) + u1 * X.s;
    v0 = fabs((ax - X.z0) * r0);
    v12 = max_nn(fabs(X.z0 * r0), fabs(ax * r0));
    const double axs = u2 * X.s;
    v0 = max_nn(v0, fabs(__dsub_rn(axs, X.zs) * r1));
    v12 = max_nn(v12, max_nn(fabs(X.zs * r1), fabs(axs * r1)));
    const double aty = lo * X.y0 + u2 * X.ys;
    v3 = fabs((u0 + aty) * r2);
    v456 = max_nn(fabs(u0 * r2), fabs(aty * r2));
    // first stage of the certificates, lane-local part
    const double lpl = -OSQP_INFTY * e0, usmax = OSQP_INFTY * e1;
    const double d1 = proj_dy_sel(X.y0 - X.py0, lpl, hi), d2 = proj_dy_sel(X.ys - X.pys, 0.0, usmax);
    nvp = max_nn(fabs(e0 * d1), fabs(e1 * d2));
    s0 = kd * (hi * fmax(d1, 0.0) + lpl * fmin(d1, 0.0)) + usmax * fmax(d2, 0.0);
    const double dss = X.s - X.ps;
    nvd = fabs(e2 * dss);
    s1 = u0 * dss;
    if (tail) {
      mvs = fabs((u1 * (kd * d1) + u2 * d2) * r2);
      const double ads = u2 * dss * r1;  // slack-bound row [0, usmax]
      rej = max_nn(usmax < OSQP_INFTY * OSQP_MIN_SCALING ? ads : 0.0, max_nn(-ads, 0.0));
    }
  } else {
    const int col = lane < NP ? lane : 0;
    const uint32_t pc = sb + 8u * (DL::Ph + col), jc = sb + 8u * (DL::Js + col);
    const uint32_t xs = sb + 8u * DL::Xs, ys = sb + 8u * DL::Ys;
    const double ax = u1 * X.p0;
    v0 = fabs(__dsub_rn(ax, X.z0) * r0);
    v12 = max_nn(fabs(X.z0 * r0), fabs(ax * r0));
    double p0 = 0.0, p1 = 0.0, t0 = 0.0, t1 = 0.0;
#pragma unroll
    for (int k = 0; k < NP; k += 2) {
      const double2 xk = lds_v2(xs + 8u * k);
      p0 = fma(lds_f64(pc + 8u * (k * NP)), xk.x, p0);
      if (k + 1 < NP) p1 = fma(lds_f64(pc + 8u * ((k + 1) * NP)), xk.y, p1);
    }
#pragma unroll
    for (int i = 0; i < MP; i += 2) {
      const double2 yi = lds_v2(ys + 8u * i);
      t0 = fma(lds_f64(jc + 8u * (i * LDJ)), yi.x, t0);
      if (i + 1 < MP) t1 = fma(lds_f64(jc + 8u * ((i + 1) * LDJ)), yi.y, t1);
    }
    const double px = p0 + p1, aty = (t0 + t1) + u1 * X.y0;
    v3 = fabs((u0 + px + aty) * r1);
    v456 = max_nn(fabs(u0 * r1), max_nn(fabs(aty * r1), fabs(px * r1)));
    const double d3 = proj_dy_sel(X.y0 - X.py0, lo, hi);
    nvp = fabs(e0 * d3);
    s0 = hi * fmax(d3, 0.0) + lo * fmin(d3, 0.0);
    const double dx = X.p0 - X.pp0;
    nvd = fabs(e1 * dx);
    s1 = u0 * dx;
    if (tail) {
      const double adx = u1 * dx * r0;  // box row [lo, hi]
      rej = max_nn(hi < OSQP_INFTY * OSQP_MIN_SCALING ? adx : 0.0, max_nn(lo > -OSQP_INFTY * OSQP_MIN_SCALING ? -adx : 0.0, 0.0));
    }
  }
  return DenseTestTerms{v0, v12, v3, v456, nvp, nvd, s0, s1, mvs, rej};
}
template <int NP, int MP, bool ROW>
__device__ __forceinline__ void dense_test_publish(const uint32_t sb, const int lane, DenseTestTerms t, const bool tail) {
  using DL = DenseL<NP, MP>;
  // one combined warp reduction
  t.v0 = warp_max_nonneg(t.v0); t.v12 = warp_max_nonneg(t.v12); t.v3 = warp_max_nonneg(t.v3);
  t.v456 = warp_max_nonneg(t.v456); t.nvp = warp_max_nonneg(t.nvp); t.nvd = warp_max_nonneg(t.nvd);
  if (tail) { t.mvs = warp_max_nonneg(t.mvs); t.rej = warp_max_nonneg(t.rej); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    t.s0 += __shfl_xor_sync(0xffffffffu, t.s0, o);
    t.s1 += __shfl_xor_sync(0xffffffffu, t.s1, o);
  }
  const uint32_t mine = sb + 8u * (DL::Red + (ROW ? 0 : 16));
  if (lane == 0) {
    sts_f64(mine, t.v0); sts_f64(mine + 8u, t.v12); sts_f64(mine + 16u, t.v3); sts_f64(mine + 24u, t.v456);
    sts_f64(mine + 32u, t.nvp); sts_f64(mine + 40u, t.nvd); sts_f64(mine + 48u, t.s0); sts_f64(mine + 56u, t.s1);
    if (tail) { sts_f64(mine + 64u, t.mvs); sts_f64(mine + 72u, t.rej); }
  }
}

// Second half, both warps, after a barrier that published both warps' slots: the team's norms (this
// warp's value first, as max_nn is not symmetric in a NaN), decided by qp_termination.  Returns 1 / 2
// (solved / solved inaccurate), -7, or 0; `want_cert` tells the caller which infeasibility certificates
// passed their first stage (bit 0 primal, bit 1 dual) and have to be evaluated in full by
// dense_certificates, which reads the reduced first stage from the per-warp slots of DL::Red.
template <int NP, int MP>
__device__ __forceinline__ int dense_test_decide(const uint32_t sb, const bool rowwarp, const bool approximate,
                                                 const bool tail, double &pri_out, double &dua_out, int &want_cert) {
  using DL = DenseL<NP, MP>;
  const uint32_t mine = sb + 8u * (DL::Red + (rowwarp ? 0 : 16)), other = sb + 8u * (DL::Red + (rowwarp ? 16 : 0));
  double mvs = 0.0, rej = 0.0;
  if (tail) { mvs = max_nn(lds_f64(mine + 64u), lds_f64(other + 64u)); rej = max_nn(lds_f64(mine + 72u), lds_f64(other + 72u)); }
  const double v0 = max_nn(lds_f64(mine), lds_f64(other)), v12 = max_nn(lds_f64(mine + 8u), lds_f64(other + 8u));
  const double v3 = max_nn(lds_f64(mine + 16u), lds_f64(other + 16u)), v456 = max_nn(lds_f64(mine + 24u), lds_f64(other + 24u));
  const double nvp = max_nn(lds_f64(mine + 32u), lds_f64(other + 32u)), nvd = max_nn(lds_f64(mine + 40u), lds_f64(other + 40u));
  // fixed order (rows + variables) so that both warps take the same decision
  const uint32_t r0a = sb + 8u * DL::Red;
  const double s0 = lds_f64(r0a + 48u) + lds_f64(r0a + 128u + 48u);
  const double s1 = lds_f64(r0a + 56u) + lds_f64(r0a + 128u + 56u);
  const double eps_pinf = dense_sc<NP, MP>(sb, 2), eps_dinf = dense_sc<NP, MP>(sb, 3);
  const int status = qp_termination(v0, v12, v3, v456, nvp, s0, nvd, s1, dense_sc<NP, MP>(sb, 4), dense_sc<NP, MP>(sb, 5),
                                    dense_sc<NP, MP>(sb, 0), dense_sc<NP, MP>(sb, 1), eps_pinf, eps_dinf, approximate,
                                    pri_out, dua_out, want_cert);
  // in tail mode, drop a certificate whose second stage the lane-local part already refutes
  if (tail) {
    const double f = approximate ? 10.0 : 1.0;
    if (mvs >= f * eps_pinf * nvp) want_cert &= ~1;
    if (rej > f * eps_dinf * nvd) want_cert &= ~2;
  }
  return status;
}

// the whole test on state X, both warps (expects Xs / Ys of X published and a barrier passed)
template <int NP, int MP>
__device__ __forceinline__ int dense_test(const uint32_t sb, const bool rowwarp, const int lane,
                                          const double u0, const double u1, const double u2, const double lo,
                                          const double hi, const DenseState &X, const bool approximate,
                                          const bool tail, double &pri_out, double &dua_out, int &want_cert) {
  if (rowwarp) dense_test_publish<NP, MP, true>(sb, lane, dense_test_terms<NP, MP, true>(sb, lane, u0, u1, u2, lo, hi, X, tail), tail);
  else dense_test_publish<NP, MP, false>(sb, lane, dense_test_terms<NP, MP, false>(sb, lane, u0, u1, u2, lo, hi, X, tail), tail);
  __syncthreads();
  return dense_test_decide<NP, MP>(sb, rowwarp, approximate, tail, pri_out, dua_out, want_cert);
}

// ---- rare paths.  Both work on the iterates spilled to DL::Sp and rebuild the lane constants from
// shared memory; they are separate functions so that their code stays out of the ADMM loop.
template <int NP, int MP>
__device__ __forceinline__ void dense_spill(const uint32_t sb, const bool rowwarp, const int lane, const DenseState &X) {
  using DL = DenseL<NP, MP>;
  const uint32_t a = sb + 8u * (DL::Sp + lane);
  if (rowwarp) {
    sts_f64(a + 8u * 160, X.s); sts_f64(a + 8u * 192, X.zs); sts_f64(a + 8u * 224, X.ys); sts_f64(a + 8u * 256, X.z0);
    sts_f64(a + 8u * 288, X.y0); sts_f64(a + 8u * 320, X.ps); sts_f64(a + 8u * 352, X.pys); sts_f64(a + 8u * 384, X.py0);
  } else {
    sts_f64(a, X.p0); sts_f64(a + 8u * 32, X.z0); sts_f64(a + 8u * 64, X.y0); sts_f64(a + 8u * 96, X.pp0);
    sts_f64(a + 8u * 128, X.py0);
  }
}
template <int NP, int MP>
__device__ __forceinline__ void dense_unspill(const uint32_t sb, const bool rowwarp, const int lane, DenseState &X) {
  using DL = DenseL<NP, MP>;
  const uint32_t a = sb + 8u * (DL::Sp + lane);
  X.p0 = X.z0 = X.y0 = X.s = X.zs = X.ys = X.pp0 = X.py0 = X.ps = X.pys = 0.0;
  if (rowwarp) {
    X.s = lds_f64(a + 8u * 160); X.zs = lds_f64(a + 8u * 192); X.ys = lds_f64(a + 8u * 224); X.z0 = lds_f64(a + 8u * 256);
    X.y0 = lds_f64(a + 8u * 288); X.ps = lds_f64(a + 8u * 320); X.pys = lds_f64(a + 8u * 352); X.py0 = lds_f64(a + 8u * 384);
  } else {
    X.p0 = lds_f64(a); X.z0 = lds_f64(a + 8u * 32); X.y0 = lds_f64(a + 8u * 64); X.pp0 = lds_f64(a + 8u * 96);
    X.py0 = lds_f64(a + 8u * 128);
  }
}
template <int NP, int MP>
__device__ __forceinline__ void dense_reload(const uint32_t sb, const bool rowwarp, const int lane, DenseLane &L,
                                             DenseState &X) {
  dense_unspill<NP, MP>(sb, rowwarp, lane, X);
  L.u0 = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 0)); L.u1 = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 1));
  L.u2 = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 2)); L.lo = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 3));
  L.hi = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 4)); L.r0 = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 5));
  L.r1 = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 6)); L.r2 = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 7));
  L.e0 = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 8)); L.e1 = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 9));
  L.e2 = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 10)); L.rbj = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 11));
}

// team maximum / sum through DL::Red (both warps, two barriers)
template <int NP, int MP>
__device__ __forceinline__ void dense_team2(const uint32_t sb, const bool rowwarp, const int lane, double &mx, double &sm) {
  using DL = DenseL<NP, MP>;
  mx = warp_max_nonneg(mx);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, o);
  const uint32_t r = sb + 8u * DL::Red;
  __syncthreads();
  if (lane == 0) { sts_f64(r + (rowwarp ? 0u : 128u), mx); sts_f64(r + (rowwarp ? 8u : 136u), sm); }
  __syncthreads();
  mx = max_nn(lds_f64(r), lds_f64(r + 128u));
  sm = lds_f64(r + 8u) + lds_f64(r + 136u);
}

// Second stage of OSQP is_primal_infeasible / is_dual_infeasible on delta_y / delta_x of the last
// iteration, for the certificates whose first stage dense_test found to hold (the dense layout's
// QPSolver::primal_infeasible / dual_infeasible).  Returns bit 0 = primal infeasible, bit 1 = dual
// infeasible.
template <int NP, int MP>
__device__ __noinline__ int dense_certificates(const uint32_t sb, const int n, const int m, const bool approximate,
                                               const bool need_p, const bool need_d) {
  using DL = DenseL<NP, MP>;
  constexpr int LDJ = DL::LDJ;
  const int tid = threadIdx.x, lane = tid & 31;
  const bool rowwarp = tid < 32;
  const bool act = rowwarp ? lane < m : lane < n;
  // |E dy|_inf and |D dx|_inf as dense_test reduced them (rows, then variables: dense_team2's order),
  // read before dense_team2 reuses the slots
  const uint32_t red = sb + 8u * DL::Red;
  const double nvp = max_nn(lds_f64(red + 32u), lds_f64(red + 128u + 32u));
  const double nvd = max_nn(lds_f64(red + 40u), lds_f64(red + 128u + 40u));
  DenseLane L;
  DenseState X;
  dense_reload<NP, MP>(sb, rowwarp, lane, L, X);
  const double f = approximate ? 10.0 : 1.0;
  const double kd = dense_sc<NP, MP>(sb, 8), c = dense_sc<NP, MP>(sb, 4);
  int res = 0;
  if (need_p) {
    const double eps = f * dense_sc<NP, MP>(sb, 2);
    double d1 = 0.0, d2 = 0.0, d3 = 0.0;
    if (rowwarp) {
      d1 = proj_dy(X.y0 - X.py0, -OSQP_INFTY * L.e0, L.hi); d2 = proj_dy(X.ys - X.pys, 0.0, OSQP_INFTY * L.e1);
      sts_f64(sb + 8u * (DL::Ys + lane), kd * d1);
    } else {
      d3 = proj_dy(X.y0 - X.py0, L.lo, L.hi);
    }
    __syncthreads();  // publishes Ys
    double mv, dummy = 0.0;
    if (rowwarp) {
      mv = fabs((L.u1 * (kd * d1) + L.u2 * d2) * L.r2);
    } else {
      double t = 0.0;
      for (int i = 0; i < MP; i++) t = fma(lds_f64(sb + 8u * (DL::Js + i * LDJ + (lane < NP ? lane : 0))), lds_f64(sb + 8u * (DL::Ys + i)), t);
      mv = fabs((t + L.u1 * d3) * L.r1);
    }
    dense_team2<NP, MP>(sb, rowwarp, lane, mv, dummy);
    if (mv < eps * nvp) res |= 1;
  }
  if (need_d) {
    const double eps = f * dense_sc<NP, MP>(sb, 3);
    double dx = 0.0, dss = 0.0;
    if (rowwarp) {
      dss = X.s - X.ps;
    } else {
      dx = X.p0 - X.pp0;
      sts_f64(sb + 8u * (DL::Xs + lane), dx);
    }
    __syncthreads();  // publishes Xs = delta_x
    const double thr = c * eps * nvd;
    double pv = 0.0, dummy = 0.0;
    if (!rowwarp) {  // |c Psym (D dx)|_j = |(Ph dx)_j / D_j|
      double t = 0.0;
      for (int k = 0; k < NP; k++) t = fma(lds_f64(sb + 8u * (DL::Ph + k * NP + (lane < NP ? lane : 0))), lds_f64(sb + 8u * (DL::Xs + k)), t);
      pv = fabs(t * L.r1);
    }
    dense_team2<NP, MP>(sb, rowwarp, lane, pv, dummy);
    if (pv < thr) {
      const double lim = eps * nvd;
      double bad = 0.0;
      if (rowwarp) {
        double t = 0.0;
        for (int k = 0; k < NP; k++) t = fma(lds_f64(sb + 8u * (DL::Js + (lane < MP ? lane : 0) * LDJ + k)), lds_f64(sb + 8u * (DL::Xs + k)), t);
        const double adx = (t + L.u1 * dss) * L.r0;
        const double lpl = -OSQP_INFTY * L.e0, usmax = OSQP_INFTY * L.e1;
        if (act && ((L.hi < OSQP_INFTY * OSQP_MIN_SCALING && adx > lim) ||
                    (lpl > -OSQP_INFTY * OSQP_MIN_SCALING && adx < -lim))) bad = 1.0;
        const double ads = L.u2 * dss * L.r1;  // slack row [0, +inf)
        if (act && ((usmax < OSQP_INFTY * OSQP_MIN_SCALING && ads > lim) || ads < -lim)) bad = 1.0;
      } else {
        const double adx = L.u1 * dx * L.r0;
        if (act && ((L.hi < OSQP_INFTY * OSQP_MIN_SCALING && adx > lim) ||
                    (L.lo > -OSQP_INFTY * OSQP_MIN_SCALING && adx < -lim))) bad = 1.0;
      }
      dense_team2<NP, MP>(sb, rowwarp, lane, bad, dummy);
      if (bad == 0.0) res |= 2;
    }
  }
  __syncthreads();
  return res;
}

// the tests OSQP runs when max_iter is reached (exact if the last iteration was not tested, then
// with all tolerances x10), on the spilled iterates
template <int NP, int MP>
__device__ __noinline__ int dense_final_tests(const uint32_t sb, const int n, const int m, const bool checked,
                                              double &pri, double &dua) {
  using DL = DenseL<NP, MP>;
  const int tid = threadIdx.x, lane = tid & 31;
  const bool rowwarp = tid < 32;
  DenseLane L;
  DenseState X;
  dense_reload<NP, MP>(sb, rowwarp, lane, L, X);
  const double kd = dense_sc<NP, MP>(sb, 8);
  sts_f64(sb + 8u * ((rowwarp ? DL::Ys : DL::Xs) + lane), rowwarp ? kd * X.y0 : X.p0);
  __syncthreads();
  for (int approx = checked ? 1 : 0; approx < 2; approx++) {
    int cert;
    int status = dense_test<NP, MP>(sb, rowwarp, lane, L.u0, L.u1, L.u2, L.lo, L.hi, X, approx != 0, true, pri, dua, cert);
    if (status == 0 && cert) {
      const int r = dense_certificates<NP, MP>(sb, n, m, approx != 0, (cert & 1) != 0, (cert & 2) != 0);
      if (r & 1) status = approx ? 3 : -3;
      else if (r & 2) status = approx ? 4 : -4;
      // dense_certificates overwrote Xs / Ys: publish them again
      sts_f64(sb + 8u * ((rowwarp ? DL::Ys : DL::Xs) + lane), rowwarp ? kd * X.y0 : X.p0);
    }
    if (status != 0) return status;
    __syncthreads();
  }
  return -2;
}

// ======================================================================================
// The solve.  Inputs (generic working set of the SQP driver, run-time offsets): unscaled box
// w.lb / w.ub, affine offsets w.bb, frozen-sparsity masks w.msk; a.Jg, a.prm, a.pi, a.kd.
// Outputs: w.x (unscaled x) and w.s (unscaled slacks).
template <int NP, int MP>
__device__ __noinline__ QPResult dense_qp_solve(const DevStruct &S_, const DevSettings &st_, const QPW &w_,
                                                const QPArgs &a_) {
  using DL = DenseL<NP, MP>;
  constexpr int LDJ = DL::LDJ, NV = DL::NV, VLD = DL::VLD;
  static_assert(NP <= 32 && MP <= 32, "one lane per variable / row");
#ifdef SCO_TIMING
  const long long t_begin = clock64();
#endif
  // ---- by-value copies: nothing below reads through a generic pointer except J, Q, q in HBM
  const int tid = threadIdx.x, lane = tid & 31;
  const bool rowwarp = tid < 32;
  const int n = S_.n, m = S_.m_nl;
  const bool act = rowwarp ? lane < m : lane < n;
  const double sigma = st_.sigma, alpha = st_.alpha, oma = 1.0 - st_.alpha;
  const double rho = fmin(fmax(st_.rho, OSQP_RHO_MIN), OSQP_RHO_MAX), rhoi = 1.0 / rho;
  const int max_iter = st_.max_iter, chk = st_.check_termination, scaling = st_.scaling;
  const double pi = a_.pi, kd = a_.kd;
  const bool tail = a_.tail != 0;
  const double *__restrict__ Jg = a_.Jg;
  const double *__restrict__ Qg = field_ptr(S_, S_.Q, a_.prm);
  const double *__restrict__ qg = field_ptr(S_, S_.q, a_.prm);
  const double *__restrict__ qag = field_ptr(S_, S_.qa, a_.prm);
  const int o_lb = w_.lb.off, o_ub = w_.ub.off, o_bb = w_.bb.off, o_msk = w_.msk.off, o_x = w_.x.off, o_s = w_.s.off;
  // warm start (sco_settings.warm_start): the unscaled duals of this team's previous QP are parked in the generic
  // working set's y arrays, which the dense solve does not use otherwise
  const int o_yp = w_.yp.off, o_ys = w_.ys.off, o_yb = w_.yb.off;
  const bool warm = a_.warm != 0, keep_duals = st_.warm_start != 0;
  const uint32_t sb = (uint32_t)__cvta_generic_to_shared(sco_smem);
  const int half = tid >> 5;  // 0 / 1: the two warps split matrix rows

  // ================================================================== load
  // Psym (unscaled) -> Si, zero padding; J masked -> Js
  for (int i = half; i < NP; i += 2) {
    if (lane < NP) {
      double v = 0.0;
      if (Qg && i < n && lane < n) v = 0.5 * (Qg[i * n + lane] + Qg[lane * n + i]);
      sts_f64(sb + 8u * (DL::Si + i * NP + lane), v);
      sts_f64(sb + 8u * (DL::Ph + i * NP + lane), 0.0);
    }
  }
  for (int i = half; i < MP; i += 2) {
    if (lane < LDJ) {
      double v = 0.0;
      if (i < m && lane < n) {
        const uint32_t mk = lds_u32(sb + 8u * o_msk + 4u * i);
        if ((mk >> lane) & 1u) v = Jg[i * n + lane];
      }
      sts_f64(sb + 8u * (DL::Js + i * LDJ + lane), v);
    }
  }
  // lane-resident scaling state.  variable lane: (D, Eb, bx, qh);  row lane: (Ep, Es, Ds, sl, bs)
  double D = 1.0, Eb = 1.0, bx = act ? 1.0 : 0.0, qh = 0.0;
  double Ep = 1.0, Es = 1.0, Ds = 1.0, sl = act ? -1.0 : 0.0, bs = act ? 1.0 : 0.0;
  double c = 1.0;
  if (!rowwarp) {
    if (act && qg) qh = qg[lane];
    if (act && qag) qh += a_.wa * qag[lane];
    sts_f64(sb + 8u * (DL::D + lane), 1.0);
  }
  __syncthreads();
  // ================================================================== Ruiz equilibration
  const int nq = n + m;
  for (int it = 0; it < scaling; it++) {
    double e_row = 1.0, d_sl = 1.0, e_sl = 1.0, d_var = 1.0, e_box = 1.0;
    if (rowwarp) {
      // all norms are maxima of absolute values: max_nn (3 instructions) on two independent chains
      double rn = fabs(sl), rn2 = 0.0;
      const uint32_t jr = sb + 8u * (DL::Js + lane * LDJ);
#pragma unroll 4
      for (int k = 0; k < NP; k += 2) {
        rn = max_nn(rn, fabs(lds_f64(jr + 8u * k)));
        if (k + 1 < NP) rn2 = max_nn(rn2, fabs(lds_f64(jr + 8u * (k + 1))));
      }
      rn = max_nn(rn, rn2);
      if (!act) rn = 0.0;
      e_row = 1.0 / sqrt(limit_scaling(rn));
      d_sl = 1.0 / sqrt(limit_scaling(fmax(fabs(sl), fabs(bs))));
      e_sl = 1.0 / sqrt(limit_scaling(fabs(bs)));
    } else {
      double cp = 0.0, cp2 = 0.0, ca = fabs(bx), ca2 = 0.0;
      const uint32_t pc = sb + 8u * (DL::Si + lane), jc = sb + 8u * (DL::Js + lane), dd = sb + 8u * DL::D;
#pragma unroll 4
      for (int i = 0; i < NP; i += 2) {
        const double2 di = lds_v2(dd + 8u * i);
        cp = max_nn(cp, di.x * fabs(lds_f64(pc + 8u * (i * NP))));
        if (i + 1 < NP) cp2 = max_nn(cp2, di.y * fabs(lds_f64(pc + 8u * ((i + 1) * NP))));
      }
      cp = max_nn(cp, cp2) * c * D;
#pragma unroll 4
      for (int i = 0; i < MP; i += 2) {
        ca = max_nn(ca, fabs(lds_f64(jc + 8u * (i * LDJ))));
        if (i + 1 < MP) ca2 = max_nn(ca2, fabs(lds_f64(jc + 8u * ((i + 1) * LDJ))));
      }
      ca = max_nn(ca, ca2);
      if (!act) { cp = 0.0; ca = 0.0; }
      d_var = 1.0 / sqrt(limit_scaling(fmax(cp, ca)));
      e_box = 1.0 / sqrt(limit_scaling(fabs(bx)));
      sts_f64(sb + 8u * (DL::t1 + lane), d_var);
    }
    __syncthreads();
    if (rowwarp) {
      const uint32_t jr = sb + 8u * (DL::Js + lane * LDJ), tt = sb + 8u * DL::t1;
      if (act)
        for (int k = 0; k < NP; k++) sts_f64(jr + 8u * k, lds_f64(jr + 8u * k) * (e_row * lds_f64(tt + 8u * k)));
      Ep *= e_row;
      sl *= e_row * d_sl;
      bs *= e_sl * d_sl;
      Ds *= d_sl;
      Es *= e_sl;
    } else {
      bx *= e_box * d_var;
      Eb *= e_box;
      qh *= d_var;
      D *= d_var;
      sts_f64(sb + 8u * (DL::D + lane), D);
    }
    __syncthreads();
    // cost normalisation
    double vs = 0.0, vm = 0.0;
    if (rowwarp) {
      if (act) vm = fabs(c * pi) * Ds;
    } else {
      if (act) {
        double cp = 0.0, cp2 = 0.0;
        const uint32_t pc = sb + 8u * (DL::Si + lane), dd = sb + 8u * DL::D;
#pragma unroll 4
        for (int i = 0; i < NP; i += 2) {
          const double2 di = lds_v2(dd + 8u * i);
          cp = max_nn(cp, di.x * fabs(lds_f64(pc + 8u * (i * NP))));
          if (i + 1 < NP) cp2 = max_nn(cp2, di.y * fabs(lds_f64(pc + 8u * ((i + 1) * NP))));
        }
        vs = max_nn(cp, cp2) * c * D;
        vm = fabs(qh);
      }
    }
    dense_team2<NP, MP>(sb, rowwarp, lane, vm, vs);
    const double mean = vs / (double)nq;
    const double ct = 1.0 / limit_scaling(fmax(mean, limit_scaling(vm)));
    qh *= ct;
    c *= ct;
  }
  const double cpi = c * pi;
  if (tid == 0) {
    const uint32_t sc = sb + 8u * DL::Sc;
    sts_f64(sc, st_.eps_abs); sts_f64(sc + 8u, st_.eps_rel); sts_f64(sc + 16u, st_.eps_prim_inf);
    sts_f64(sc + 24u, st_.eps_dual_inf); sts_f64(sc + 32u, c); sts_f64(sc + 40u, 1.0 / c); sts_f64(sc + 48u, cpi);
    sts_f64(sc + 56u, rho); sts_f64(sc + 64u, kd);
  }
  // ================================================================== bounds, rho, slack elimination
  // lane constants of the ADMM loop (registers) and of the termination test (DL::LA)
  double u0, u1, u2, u3, lo, hi, Mi = 0.0;
  {
    double r0, r1, r2 = 0.0, e0, e1, e2 = 0.0, rbj = 1.0;
    if (rowwarp) {
      double bbi = 0.0;
      if (act) bbi = lds_f64(sb + 8u * (o_bb + lane));
      hi = act ? Ep * clampd(-bbi, -OSQP_INFTY, OSQP_INFTY) : 0.0;
      const double kr = kd * rho;
      const double m11 = sigma + kr * sl * sl + rho * bs * bs;
      Mi = act ? 1.0 / m11 : 0.0;
      const double hs = kr * Mi * sl;
      const double coef = act ? kr - kr * sl * hs : 0.0;
      u0 = act ? cpi * Ds : 0.0;
      u1 = sl;
      u2 = bs;
      u3 = hs;
      lo = kd * sl;
      e0 = act ? Ep : 0.0; e1 = act ? Es : 0.0; e2 = act ? Ds : 0.0;
      r0 = act ? 1.0 / Ep : 0.0; r1 = act ? 1.0 / Es : 0.0; r2 = act ? 1.0 / Ds : 0.0;
      sts_f64(sb + 8u * (DL::cf + lane), coef);
    } else {
      double lbx = 0.0, ubx = 0.0;
      if (act) { lbx = lds_f64(sb + 8u * (o_lb + lane)); ubx = lds_f64(sb + 8u * (o_ub + lane)); }
      lo = act ? Eb * fmax(lbx, -OSQP_INFTY) : 0.0;
      hi = act ? Eb * fmin(ubx, OSQP_INFTY) : 0.0;
      rbj = act ? rho_of(lo, hi, rho) : 1.0;
      u0 = qh;
      u1 = bx;
      u2 = rbj;
      u3 = 1.0 / rbj;
      e0 = act ? Eb : 0.0; e1 = act ? D : 0.0;
      r0 = act ? 1.0 / Eb : 0.0; r1 = act ? 1.0 / D : 0.0;
      sts_f64(sb + 8u * (DL::dg + lane), sigma + rbj * bx * bx);
    }
    sts_f64(dense_la<NP, MP>(sb, rowwarp, lane, 0), u0); sts_f64(dense_la<NP, MP>(sb, rowwarp, lane, 1), u1);
    sts_f64(dense_la<NP, MP>(sb, rowwarp, lane, 2), u2); sts_f64(dense_la<NP, MP>(sb, rowwarp, lane, 3), lo);
    sts_f64(dense_la<NP, MP>(sb, rowwarp, lane, 4), hi); sts_f64(dense_la<NP, MP>(sb, rowwarp, lane, 5), r0);
    sts_f64(dense_la<NP, MP>(sb, rowwarp, lane, 6), r1); sts_f64(dense_la<NP, MP>(sb, rowwarp, lane, 7), r2);
    sts_f64(dense_la<NP, MP>(sb, rowwarp, lane, 8), e0); sts_f64(dense_la<NP, MP>(sb, rowwarp, lane, 9), e1);
    sts_f64(dense_la<NP, MP>(sb, rowwarp, lane, 10), e2); sts_f64(dense_la<NP, MP>(sb, rowwarp, lane, 11), rbj);
  }
  __syncthreads();
  // ================================================================== S = P^ + diag + J' diag(coef) J, then S^-1
  for (int i = half; i < n; i += 2) {
    if (lane < n) {
      const double pv = c * lds_f64(sb + 8u * (DL::D + i)) * lds_f64(sb + 8u * (DL::Si + i * NP + lane)) * lds_f64(sb + 8u * (DL::D + lane));
      double v = pv;
      if (i == lane) v += lds_f64(sb + 8u * (DL::dg + lane));
      const uint32_t ji = sb + 8u * (DL::Js + i), jl = sb + 8u * (DL::Js + lane), cf = sb + 8u * DL::cf;
      double v2 = 0.0;
#pragma unroll 4
      for (int r = 0; r < MP; r += 2) {
        const double2 cr = lds_v2(cf + 8u * r);
        v = fma(cr.x * lds_f64(jl + 8u * (r * LDJ)), lds_f64(ji + 8u * (r * LDJ)), v);
        if (r + 1 < MP) v2 = fma(cr.y * lds_f64(jl + 8u * ((r + 1) * LDJ)), lds_f64(ji + 8u * ((r + 1) * LDJ)), v2);
      }
      v += v2;
      sts_f64(sb + 8u * (DL::Ph + i * NP + lane), pv);
      sts_f64(sb + 8u * (DL::Si + i * NP + lane), v);  // in place: every element reads only itself from Si
    }
  }
  __syncthreads();
  // in-place Gauss-Jordan inverse (S is SPD: no pivoting); pivot row / column staged in t1 / Xs
  for (int k = 0; k < n; k++) {
    const double d = 1.0 / lds_f64(sb + 8u * (DL::Si + k * NP + k));
    if (tid < n) {
      sts_f64(sb + 8u * (DL::t1 + tid), lds_f64(sb + 8u * (DL::Si + k * NP + tid)) * d);
      sts_f64(sb + 8u * (DL::Xs + tid), lds_f64(sb + 8u * (DL::Si + tid * NP + k)));
    }
    __syncthreads();
    for (int i = half; i < n; i += 2) {
      if (lane < n) {
        const uint32_t e = sb + 8u * (DL::Si + i * NP + lane);
        const double rowk = lds_f64(sb + 8u * (DL::t1 + lane)), colk = lds_f64(sb + 8u * (DL::Xs + i));
        double v;
        if (i == k) v = (lane == k) ? d : rowk;
        else if (lane == k) v = -colk * d;
        else v = lds_f64(e) - colk * rowk;
        sts_f64(e, v);
      }
    }
    __syncthreads();
  }
  // ================================================================== K = S^-1 J'  (Ks[j*MP + i])
  for (int j = half; j < n; j += 2) {
    if (lane < MP) {  // padded rows (lane >= m) hold zeros in Js, so their K entries are exact zeros
      double a0 = 0.0, a1 = 0.0;
      const uint32_t sj = sb + 8u * (DL::Si + j), jr = sb + 8u * (DL::Js + lane * LDJ);
#pragma unroll 2
      for (int k = 0; k < NP; k += 2) {
        a0 = fma(lds_f64(sj + 8u * (k * NP)), lds_f64(jr + 8u * k), a0);
        if (k + 1 < NP) a1 = fma(lds_f64(sj + 8u * ((k + 1) * NP)), lds_f64(jr + 8u * (k + 1)), a1);
      }
      sts_f64(sb + 8u * (DL::Ks + j * MP + lane), a0 + a1);
    }
  }
  // zero the exchange buffers meanwhile
  for (int e = tid; e < 2 * VLD + 64; e += 64) sts_f64(sb + 8u * (DL::Vb + e), 0.0);
  __syncthreads();
  // ---- this lane's row of [S^-1 K ; K' G] -> registers
  double Mr[NV];
  if (rowwarp) {
#pragma unroll
    for (int k = 0; k < NP; k++) Mr[k] = (act && k < n) ? lds_f64(sb + 8u * (DL::Ks + k * MP + lane)) : 0.0;
    // G row: all MP accumulators in flight, one pass over k (K rows are read as broadcast 128-bit words)
    const uint32_t jr = sb + 8u * (DL::Js + (act ? lane : 0) * LDJ);
#pragma unroll
    for (int l = 0; l < MP; l++) Mr[NP + l] = 0.0;
    for (int k = 0; k < n; k++) {
      const double jv = act ? lds_f64(jr + 8u * k) : 0.0;
      const uint32_t kr = sb + 8u * (DL::Ks + k * MP);
#pragma unroll
      for (int l = 0; l < MP; l += 2) {
        const double2 kk = lds_v2(kr + 8u * l);
        Mr[NP + l] = fma(jv, kk.x, Mr[NP + l]);
        Mr[NP + l + 1] = fma(jv, kk.y, Mr[NP + l + 1]);
      }
    }
  } else {
#pragma unroll
    for (int k = 0; k < NP; k++) Mr[k] = (act && k < n) ? lds_f64(sb + 8u * (DL::Si + k * NP + lane)) : 0.0;
#pragma unroll
    for (int i = 0; i < MP; i++) Mr[NP + i] = (act && i < m) ? lds_f64(sb + 8u * (DL::Ks + lane * MP + i)) : 0.0;
  }
  QPResult res;
  res.status = 0; res.iters = 0; res.pri_res = 0.0; res.dua_res = 0.0;
#ifdef SCO_TIMING
  res.cyc_check = 0;
  for (int k = 0; k < 5; k++) res.cyc_c[k] = 0;
  res.cyc_setup = clock64() - t_begin;
  res.cyc_scale = 0;
  const long long t_loop = clock64();
#endif
  // ================================================================== ADMM
  DenseState X;
  X.p0 = X.z0 = X.y0 = X.s = X.zs = X.ys = X.pp0 = X.py0 = X.ps = X.pys = 0.0;
  double g = Mi * (-u0);
  // this lane's entry of (c, wp); lanes that own none store into the dump slot at the end of the row
  const bool publishes = rowwarp ? lane < MP : lane < NP;
  const uint32_t vb0 = sb + 8u * DL::Vb, vb1 = vb0 + 8u * VLD;
  const uint32_t my_out = 8u * (uint32_t)(publishes ? (rowwarp ? NP + lane : lane) : VLD - 1);
  const uint32_t my_chk = sb + 8u * ((rowwarp ? DL::Ys : DL::Xs) + lane);
  double first_out = rowwarp ? -(rho * lo) * g : -u0;  // this lane's entry of (c, wp) for x = z = y = 0
  if (warm) {
    // OSQP's warm start (osqp_warm_start): x^ = D^-1 x, y^ = c E^-1 y, z^ = A^ x^ with the scaling of THIS QP; x, s and
    // the duals are those the previous QP of this problem ended with.  The reference never warm-starts (it builds a
    // new OSQP object per call, osqp_utils.py:195): opt-in, results agree to the QP tolerances, not bit for bit.
    const double e0 = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 8)), e1 = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 9));
    if (!rowwarp) {
      if (act) {
        X.p0 = lds_f64(sb + 8u * (o_x + lane)) / e1;        // / D
        X.y0 = c * lds_f64(sb + 8u * (o_yb + lane)) / e0;   // c y / Eb
        X.z0 = u1 * X.p0;
      }
      sts_f64(sb + 8u * (DL::Xs + lane), X.p0);
    } else if (act) {
      const double e2 = lds_f64(dense_la<NP, MP>(sb, true, lane, 10));
      X.s = lds_f64(sb + 8u * (o_s + lane)) / e2;             // / Ds
      X.ys = c * lds_f64(sb + 8u * (o_ys + lane)) / e1;       // c y / Es
      X.zs = u2 * X.s;
      X.y0 = c * (lds_f64(sb + 8u * (o_yp + lane)) / kd) / e0;  // the stored dual is the sum over the kd copies
    }
    __syncthreads();
    if (rowwarp) {
      const uint32_t jr = sb + 8u * (DL::Js + (lane < MP ? lane : 0) * LDJ), xs = sb + 8u * DL::Xs;
      double t = 0.0;
      for (int k = 0; k < NP; k++) t = fma(lds_f64(jr + 8u * k), lds_f64(xs + 8u * k), t);
      if (act) X.z0 = t + u1 * X.s;
      const double wpen = rho * X.z0 - X.y0;
      const double rr = (sigma * X.s - u0) + u2 * (rho * X.zs - X.ys) + lo * wpen;
      g = Mi * rr;
      first_out = kd * wpen - (rho * lo) * g;
    } else {
      first_out = (sigma * X.p0 - u0) + u1 * (u2 * X.z0 - X.y0);
    }
    __syncthreads();
  }
  if (publishes) sts_f64(vb0 + my_out, first_out);
  int iter = 0, status = 0;
  bool checked = false;
  int next_check = chk ? chk : max_iter + 1;
  __syncthreads();

  // one ADMM iteration: the dot product of this lane's row with (c, wp) at `vcur` ...
  auto lane_dot = [&](const uint32_t vcur) {
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
    for (int k = 0; k < NV / 4; k++) {
      const double2 va = lds_v2(vcur + 32u * k), vc = lds_v2(vcur + 32u * k + 16u);
      a0 = fma(Mr[4 * k], va.x, a0);
      a1 = fma(Mr[4 * k + 1], va.y, a1);
      a2 = fma(Mr[4 * k + 2], vc.x, a2);
      a3 = fma(Mr[4 * k + 3], vc.y, a3);
    }
    if (NV % 4) {
      const double2 va = lds_v2(vcur + 8u * (NV - 2));
      a0 = fma(Mr[NV - 2], va.x, a0);
      a1 = fma(Mr[NV - 1], va.y, a1);
    }
    return (a0 + a1) + (a2 + a3);
  };
  // ... then the lane-local update, which returns this lane's entry of (c, wp) for the next iteration.
  // The updates are those of the generic loop (sco_qp.cuh generic_loop P1..P4) with the exact
  // identities  y+ = y + rho (v - z+) = rho (t - z+),  rho z+ - y+ = rho (2 z+ - t),  t = v + y / rho,
  // which shorten the dependent chain behind the dot product from 16 to 10 FP64 operations.  A product
  // feeding a subtraction is written as an explicit fma: left to ptxas, which multiply it fuses depends
  // on the surrounding code, and the plain and the tested iterations would round differently.
  auto row_update = [&](const double acc) {
    // t = acc ; slack and penalty-row updates, then wp for the next iteration
    const double stil = fma(acc, -u3, g);
    const double sn = alpha * stil + oma * X.s;
    const double ts = (alpha * u2) * stil + (oma * X.zs + X.ys * rhoi);
    const double zns = relu_bits(ts);
    X.ys = rho * (ts - zns);
    const double zt = acc + u1 * stil;
    const double tz = alpha * zt + (oma * X.z0 + X.y0 * rhoi);
    const double zn = tz < hi ? tz : hi;
    X.y0 = rho * (tz - zn);
    X.s = sn;
    X.zs = zns;
    X.z0 = zn;
    const double wpen = rho * (2.0 * zn - tz);
    const double rr = fma(lo, wpen, fma(u2, rho * (2.0 * zns - ts), fma(sigma, sn, -u0)));
    g = Mi * rr;
    return fma(kd, wpen, -((rho * lo) * g));
  };
  auto var_update = [&](const double acc) {
    // x~ = acc ; x and box-row updates, then c for the next iteration
    const double xn = alpha * acc + oma * X.p0;
    const double tz = (alpha * u1) * acc + (oma * X.z0 + X.y0 * u3);
    const double zn = clampd(tz, lo, hi);
    X.y0 = u2 * (tz - zn);
    X.p0 = xn;
    X.z0 = zn;
    return fma(u1 * u2, 2.0 * zn - tz, fma(sigma, xn, -u0));
  };
  // reads (c, wp) at `vcur`, publishes this lane's new entry at `vnext`
  auto iterate = [&](const uint32_t vcur, const uint32_t vnext) {
    const double acc = lane_dot(vcur);
    const double out = rowwarp ? row_update(acc) : var_update(acc);
    sts_f64(vnext + my_out, out);
  };
  // iteration k+1 with the first half of the termination test of iteration k (Xs / Ys published, its
  // iterates spilled to DL::Sp) in its shadow: neither depends on the other, and with the warp's role and
  // the tail mode fixed at compile time each warp runs both in one basic block, so the test's loads, dot
  // products and lane-local terms fill the latency of the iteration's dependent chain.  The barrier after
  // it publishes the test's partials with (c, wp).
  auto iterate_and_test = [&](const uint32_t vcur, const uint32_t vnext, auto row, auto tl) {
    constexpr bool ROW = decltype(row)::value, TAIL = decltype(tl)::value;
    DenseState Xk;
    dense_unspill<NP, MP>(sb, ROW, lane, Xk);
    const double acc = lane_dot(vcur);
    const DenseTestTerms t = dense_test_terms<NP, MP, ROW>(sb, lane, u0, u1, u2, lo, hi, Xk, TAIL);
    const double out = ROW ? row_update(acc) : var_update(acc);
    dense_test_publish<NP, MP, ROW>(sb, lane, t, TAIL);  // after the update: a warp collective is a scheduling fence
    sts_f64(vnext + my_out, out);
  };
  int p = 0;
  while (iter < max_iter) {
    // ---- plain iterations up to (not including) the next tested / last one
    const int seg_end = next_check < max_iter ? next_check : max_iter;
    for (int i = iter + 1; i < seg_end; i++) {
      iterate(p ? vb1 : vb0, p ? vb0 : vb1);
      p ^= 1;
      __syncthreads();
    }
    // ---- the tested (or last) iteration: the certificates need delta_x / delta_y of it
    X.pp0 = X.p0; X.py0 = X.y0; X.ps = X.s; X.pys = X.ys;
    iterate(p ? vb1 : vb0, p ? vb0 : vb1);
    p ^= 1;
    iter = seg_end;
    checked = false;
    if (iter != next_check) { __syncthreads(); break; }
    next_check += chk;
    checked = true;
    sts_f64(my_chk, rowwarp ? kd * X.y0 : X.p0);
    if (chk >= 2 && iter + 1 < max_iter) {
      // ---- pipelined test of iteration k = iter, decided after iteration k+1.  Iteration k+1 is never
      // tested itself (chk >= 2) nor the last one, so the max_iter epilogue never sees this path.  State k
      // goes to DL::Sp: the test reads it from there, and a verdict on k restores it.
      dense_spill<NP, MP>(sb, rowwarp, lane, X);
      __syncthreads();
      const uint32_t vcur = p ? vb1 : vb0, vnext = p ? vb0 : vb1;
      if (rowwarp) {
        if (tail) iterate_and_test(vcur, vnext, BoolC<true>(), BoolC<true>());
        else iterate_and_test(vcur, vnext, BoolC<true>(), BoolC<false>());
      } else {
        if (tail) iterate_and_test(vcur, vnext, BoolC<false>(), BoolC<true>());
        else iterate_and_test(vcur, vnext, BoolC<false>(), BoolC<false>());
      }
      p ^= 1;
      __syncthreads();
#ifdef SCO_TIMING
      const long long tc0 = clock64();
#endif
      int cert;
      status = dense_test_decide<NP, MP>(sb, rowwarp, false, tail, res.pri_res, res.dua_res, cert);
      if (status == 0 && cert) {  // Xs / Ys / Red are free again: the decision has been read
        const int r = dense_certificates<NP, MP>(sb, n, m, false, (cert & 1) != 0, (cert & 2) != 0);
        if (r & 1) status = -3;
        else if (r & 2) status = -4;
      }
      if (status != 0) dense_unspill<NP, MP>(sb, rowwarp, lane, X);  // the result is iteration k's
      else iter++;
#ifdef SCO_TIMING
      res.cyc_check += clock64() - tc0;
#endif
      if (status != 0) break;
      continue;
    }
    // ---- unpipelined test (check_termination 1, or k+1 = max_iter)
#ifdef SCO_TIMING
    const long long tc0 = clock64();
#endif
    __syncthreads();
    int cert;
    status = dense_test<NP, MP>(sb, rowwarp, lane, u0, u1, u2, lo, hi, X, false, tail, res.pri_res, res.dua_res, cert);
    if (status != 0) break;
    if (cert) {
      dense_spill<NP, MP>(sb, rowwarp, lane, X);
      __syncthreads();
      const int r = dense_certificates<NP, MP>(sb, n, m, false, (cert & 1) != 0, (cert & 2) != 0);
      if (r & 1) { status = -3; break; }
      if (r & 2) { status = -4; break; }
    }
#ifdef SCO_TIMING
    res.cyc_check += clock64() - tc0;
#endif
  }
#ifdef SCO_TIMING
  res.cyc_loop = clock64() - t_loop;
#endif
  __syncthreads();
  if (status == 0) {  // max_iter reached without a verdict
    dense_spill<NP, MP>(sb, rowwarp, lane, X);
    __syncthreads();
    status = dense_final_tests<NP, MP>(sb, n, m, checked, res.pri_res, res.dua_res);
    iter = max_iter;
  }
  // ---- unscale into the SQP driver's arrays
  if (act) {  // D / Ds are e1 / e2 of the lane-constant block
    if (rowwarp) sts_f64(sb + 8u * (o_s + lane), X.s * lds_f64(dense_la<NP, MP>(sb, true, lane, 10)));
    else sts_f64(sb + 8u * (o_x + lane), X.p0 * lds_f64(dense_la<NP, MP>(sb, false, lane, 9)));
    if (keep_duals) {  // y = E y^ / c, for the next QP's warm start
      const double e0 = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 8)), e1 = lds_f64(dense_la<NP, MP>(sb, rowwarp, lane, 9));
      const double cinv = dense_sc<NP, MP>(sb, 5);
      if (rowwarp) {
        sts_f64(sb + 8u * (o_yp + lane), kd * e0 * X.y0 * cinv);
        sts_f64(sb + 8u * (o_ys + lane), e1 * X.ys * cinv);
      } else {
        sts_f64(sb + 8u * (o_yb + lane), e0 * X.y0 * cinv);
      }
    }
  }
  __syncthreads();
  res.status = status;
  res.iters = iter;
  return res;
}
