// sco_kernels.cuh -- the __global__ entry points, templated on the team size (threads per problem).
// Compiled once per team size by sco_team.cu (-DSCO_TEAM=32|64|128|256) so the four
// instantiations build in parallel; sco_abi.cu holds only host code.
#pragma once
#include "sco_device.cuh"
#include "sco_families.cuh"
#include "sco_qp.cuh"
#include "sco_sqp.cuh"

// Register budget per thread.  The register file is split over the four SM sub-partitions (16 K
// registers each), so the steps are 255 (2 warps per sub-partition), 168 (3), 128 (4).  Left alone,
// ptxas aims a 64-thread kernel at 168 and the dense loop's matrix rows (100 registers) spill to
// local memory inside the ADMM loop; the dense kinds therefore take the full 255.
#ifndef SCO_DK
#define SCO_DK 0
#endif
#if defined(SCO_TEAM) && SCO_TEAM >= 512
// A warp's registers come out of its SM sub-partition's 16,384: a 512-thread team has four warps on each, so 128
// registers per thread is its ceiling (a 448-thread team has the same problem: 4 + 4 + 3 + 3 warps).  A 256-thread
// team keeps the full budget (one team per SM): at 128 registers two teams fit, but the penalty-row role spills and
// the point robot's 1,024-problem batch -- whose step is set by one 794 k-iteration problem -- ran at 1,050
// instead of 1,535 problems/s (profiles/r2_generic_cycles.txt).
#define SCO_MAXNREG 128
#else
#define SCO_MAXNREG 255
#endif

template <int TEAM, int DK>
__global__ void __maxnreg__(SCO_MAXNREG)
k_solve(const __grid_constant__ DevStruct S, const __grid_constant__ DevSettings st, long long B,
        const double *__restrict__ params, const double *__restrict__ x0, double *__restrict__ x_out,
        int *__restrict__ verdict, double *__restrict__ merit, double *__restrict__ objective,
        double *__restrict__ max_vio, int *__restrict__ stats, double *__restrict__ Jscr,
        unsigned long long *counter, const int *__restrict__ order, int *__restrict__ nonconv,
        const int *__restrict__ order_err) {
  __shared__ long long next;
  if (order_err && *order_err != 0) {  // sco_solve_batch_ordered: the order is not a permutation (checked by k_check_order)
    for (long long b = (long long)blockIdx.x * TEAM + threadIdx.x; b < B; b += (long long)gridDim.x * TEAM) verdict[b] = -3;
    return;
  }
  QPW w;
  w.bind(S.L);
  const Sh xc = w.xc;  // n doubles appended after the layout
  double *Jg = Jscr + (size_t)blockIdx.x * (S.jnnz + S.sws);
  if (S.sws) w.Sg = Jg + S.jnnz;
  const int tid = threadIdx.x;
  while (true) {
    if (tid == 0) next = (long long)atomicAdd(counter, 1ull);
    Team<TEAM>::sync();
    const long long slot = next;
    Team<TEAM>::sync();
    if (slot >= B) break;
    const long long b = order ? (long long)order[slot] : slot;  // optional processing order (longest first)
    const double *prm = params + b * S.stride;
    SqpSolver<TEAM, DK> sq(S, st, w, prm, Jg);
    sq.queue = counter;
    sq.queue_len = B;
    SqpOut o = sq.run(x0 + b * S.n);
    for (int j = tid; j < S.n; j += TEAM) x_out[b * S.n + j] = xc[j];
    if (tid == 0) {
      verdict[b] = o.verdict;
      if (merit) merit[b] = o.merit;
      if (objective) objective[b] = o.objective;
      if (max_vio) max_vio[b] = o.max_vio;
      if (stats) {
        stats[4 * b] = o.sqp_iters; stats[4 * b + 1] = o.qp_solves;
        stats[4 * b + 2] = o.admm_iters; stats[4 * b + 3] = o.last_status;
      }
      if (nonconv) nonconv[b] = o.nonconv;
#ifdef SCO_TIMING
      // diagnostic build only: the report slots carry the per-phase clock64() totals instead
      if (merit) merit[b] = (double)o.cyc_total;
      if (objective) objective[b] = (double)o.cyc_setup;
      if (max_vio) max_vio[b] = (double)o.cyc_loop;
      x_out[b * S.n] = (double)o.cyc_check;
      x_out[b * S.n + 1] = (double)o.cyc_cvx;
#endif
    }
    Team<TEAM>::sync();
  }
}

template <int TEAM>
__global__ void __launch_bounds__(TEAM)
k_convexify(const __grid_constant__ DevStruct S, long long B, const double *__restrict__ params,
            const double *__restrict__ x, double *__restrict__ f, double *__restrict__ J,
            double *__restrict__ bvec, double *__restrict__ obj, double *__restrict__ Jscr, double *__restrict__ Hq,
            double *__restrict__ gq, double *__restrict__ cq) {
  QPW w;
  w.bind(S.L);
  const Sh xc = w.xc;
  const int tid = threadIdx.x;
  DevSettings st;
  memset(&st, 0, sizeof(st));
  st.freeze_sparsity = 1;
  for (long long b = blockIdx.x; b < B; b += gridDim.x) {
    const double *prm = params + b * S.stride;
    double *Jg = J ? J + b * S.jnnz : Jscr + (size_t)blockIdx.x * S.jnnz;
    SqpSolver<TEAM, 0> sq(S, st, w, prm, Jg);
    for (int j = tid; j < S.n; j += TEAM) xc[j] = x[b * S.n + j];
    Team<TEAM>::sync();
    bool mask_set = false;
    sq.convexify(mask_set);
    for (int i = tid; i < S.m_nl; i += TEAM) {
      if (f) f[b * S.m_nl + i] = w.fv[i];
      if (bvec) bvec[b * S.m_nl + i] = w.bb[i];
    }
    if (obj) {
      const double ov = sq.objective();
      if (tid == 0) obj[b] = ov;
    }
    if (S.n_ob) {  // Expr.convexify degree 2 of the non-quadratic objective terms, summed (expr.py:143-153)
      const int n = S.n;
      if (Hq)  // column j by one thread: zeros, then the model's entries on the pattern of P
        for (int j = tid; j < n; j += TEAM) {
          double *Hb = Hq + (size_t)b * n * n;
          for (int i = 0; i < n; i++) Hb[(size_t)i * n + j] = 0.0;
          for (int p = S.P_cptr[j]; p < S.P_cptr[j + 1]; p++) Hb[(size_t)S.P_row[p] * n + j] = w.Hv[p];
        }
      if (gq) for (int e = tid; e < n; e += TEAM) gq[b * n + e] = w.gq[e];
      if (cq && tid == 0) cq[b] = w.oc[0];
    }
    Team<TEAM>::sync();
  }
}

template <int TEAM, int DK>
__global__ void __maxnreg__(SCO_MAXNREG)
k_qp(const __grid_constant__ DevStruct S, const __grid_constant__ DevSettings st, long long B,
     const double *__restrict__ params, const double *__restrict__ J, const double *__restrict__ bvec,
     const uint32_t *__restrict__ mask, const double *__restrict__ lbx, const double *__restrict__ ubx,
     const double *__restrict__ pi, const int *__restrict__ kdup, const double *__restrict__ wa,
     const double *__restrict__ xref,
     int use_pen, int closest, double *__restrict__ xq, int *__restrict__ status,
     int *__restrict__ iters, double *__restrict__ scr) {
  QPW w;
  w.bind(S.L);
  if (S.sws) w.Sg = scr + (size_t)blockIdx.x * (S.jnnz + S.sws) + S.jnnz;
  const int tid = threadIdx.x;
  const int n = S.n, ms = S.m_nl;
  for (long long b = blockIdx.x; b < B; b += gridDim.x) {
    for (int j = tid; j < n; j += TEAM) {
      w.lb[j] = lbx ? lbx[b * n + j] : -INFINITY;
      w.ub[j] = ubx ? ubx[b * n + j] : INFINITY;
      w.xs[j] = xref ? xref[b * n + j] : 0.0;
    }
    if (use_pen) {
      for (int i = tid; i < ms; i += TEAM) w.bb[i] = bvec[b * ms + i];
      for (int i = tid; i < ms * S.mw; i += TEAM) w.msk[i] = mask ? mask[b * ms * S.mw + i] : 0xffffffffu;
    }
    Team<TEAM>::sync();
    QPArgs a;
    a.prm = params + b * S.stride;
    a.Jg = use_pen ? J + b * S.jnnz : nullptr;
    a.pi = pi ? pi[b] : 0.0;
    a.kd = kdup ? (double)kdup[b] : 1.0;
    a.wa = wa ? wa[b] : 1.0;
    a.warm = 0;
    a.use_pen = use_pen;
    a.closest = closest;
    a.has_hq = 0;
    a.tail = 0;
    QPSolver<TEAM, DK> qp(S, st, w, a);
    QPResult r = qp.solve();
    const int nq = use_pen ? S.n_q : n;
    for (int j = tid; j < n; j += TEAM) xq[b * nq + j] = w.x[j];
    if (use_pen) {
      int so = n;
      for (int bi = 0; bi < S.n_blocks; bi++) {
        const DevBlock &Bk = S.blocks[bi];
        for (int r2 = tid; r2 < Bk.m; r2 += TEAM) {
          xq[b * nq + so + r2] = w.s[Bk.row0 + r2];
          if (Bk.cnt_type) xq[b * nq + so + Bk.m + r2] = w.s[ms + Bk.row0 + r2];
        }
        so += Bk.m * (Bk.cnt_type ? 2 : 1);
      }
    }
    if (tid == 0) {
      status[b] = r.status;
      iters[b] = r.iters;
#ifdef SCO_TIMING
      xq[b * nq] = (double)r.cyc_loop; xq[b * nq + 1] = (double)r.cyc_check; xq[b * nq + 2] = (double)r.cyc_setup;
      for (int k = 0; k < 5; k++) xq[b * nq + 3 + k] = (double)r.cyc_c[k];
      xq[b * nq + 8] = (double)r.cyc_scale;
#endif
    }
    Team<TEAM>::sync();
  }
}

template <int TEAM>
__global__ void __launch_bounds__(TEAM)
k_merit(const __grid_constant__ DevStruct S, long long B, const double *__restrict__ params,
        const double *__restrict__ x, const double *__restrict__ J, const double *__restrict__ bvec,
        const double *__restrict__ mu, double *__restrict__ merit, double *__restrict__ model,
        double *__restrict__ max_vio, double *__restrict__ gv, double *__restrict__ gm) {
  QPW w;
  w.bind(S.L);
  const Sh xc = w.xc;
  const int tid = threadIdx.x;
  DevSettings st;
  memset(&st, 0, sizeof(st));
  for (long long b = blockIdx.x; b < B; b += gridDim.x) {
    const double *prm = params + b * S.stride;
    SqpSolver<TEAM, 0> sq(S, st, w, prm, const_cast<double *>(J ? J + b * S.jnnz : nullptr));
    for (int j = tid; j < S.n; j += TEAM) xc[j] = x[b * S.n + j];
    if (bvec)
      for (int i = tid; i < S.m_nl; i += TEAM) w.bb[i] = bvec[b * S.m_nl + i];
    Team<TEAM>::sync();
    eval_blocks<TEAM>(S, prm, xc, w.fv, nullptr, w.stage);
    double vs[2 + SCO_DEV_MAX_GROUPS], msum[2 + SCO_DEV_MAX_GROUPS];
    sq.violation_sums(vs);
    const double ov = sq.objective();
    const double m = mu ? mu[b] : 1.0;
    if (J && bvec) sq.model_sums(msum);
    if (tid == 0) {
      if (merit) merit[b] = ov + m * vs[0];
      if (max_vio) max_vio[b] = vs[1];
      if (model && J && bvec) model[b] = ov + m * msum[0];
      for (int g = 0; g < S.n_groups; g++) {
        if (gv) gv[b * S.n_groups + g] = vs[2 + g];
        if (gm && J && bvec) gm[b * S.n_groups + g] = msum[2 + g];
      }
    }
    Team<TEAM>::sync();
  }
}

