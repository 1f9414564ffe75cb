// sco_families.cuh -- batched expression evaluation and convexification on device.
//
// Replaces Expr.eval / Expr.grad / Expr._num_grad (sco_py/expr.py:34-41,61-69,78-100) for the
// closed constraint families the engine supports, and the affine-model offset of
// Expr.convexify degree 1 (expr.py:139-142) + Eq/LEqExpr.convexify (expr.py:327-328,366-367):
//   J = grad f(x),  b = f(x) - J x - val.
// A team evaluates one problem: x is in shared memory, the family parameters are streamed from
// the problem's parameter block in HBM with coalesced loads (a warp reads 32 consecutive doubles).
#pragma once
#include "sco_device.cuh"

#define FAM_QUADFORM 1
#define FAM_CIRCLE2D 2
#define FAM_FK7 3
#define FAM_VM 4

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- QUADFORM: f_j = 0.5 x'P_j x + a_j'x, P_j packed upper row-major, one warp per row ----
// With a column map x is the row's n_in inputs, gathered into the staging buffer behind P_j.
template <int TEAM>
__device__ void eval_quadform(const DevStruct &S, const DevBlock &B, const double *par,
                              Sh xg, Sh f, double *Jout, Sh stage) {
  const int *cm = B.n_in ? S.jcol_g + B.joff : nullptr;  // column map
  const int n = cm ? B.n_in : S.n, ntri = n * (n + 1) / 2, m = B.m;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const Sh buf = stage + warp * S.stage_per_warp;
  const Sh x = cm ? buf + ntri : xg;
  const double *A = par + (size_t)m * ntri;
  for (int j = warp; j < m; j += TEAM / 32) {
    const double *Pj = par + (size_t)j * ntri;
    for (int e = lane; e < ntri; e += 32) buf[e] = __ldg(Pj + e);
    if (cm)
      for (int i = lane; i < n; i += 32) x[i] = xg[__ldg(cm + j * n + i)];
    __syncwarp();
    double fj = 0.0;
    for (int r = lane; r < n; r += 32) {
      double acc = 0.0;
      for (int cc = 0; cc < r; cc++) acc += buf[cc * n - (cc * (cc - 1)) / 2 + (r - cc)] * x[cc];
      const int base = r * n - (r * (r - 1)) / 2 - r;
      for (int cc = r; cc < n; cc++) acc += buf[base + cc] * x[cc];
      const double aj = __ldg(A + j * n + r);
      if (Jout) Jout[j * n + r] = acc + aj;
      fj += x[r] * (0.5 * acc + aj);
    }
    fj = warp_sum(fj);
    if (lane == 0) f[j] = fj;
    __syncwarp();
  }
}

// ---- CIRCLE2D: row t*K+k: R_k - |p_t - c_k| ----
// With a column map row r reads the point (x[cols[2r]], x[cols[2r+1]]).
template <int TEAM>
__device__ void eval_circle2d(const DevStruct &S, const DevBlock &B, const double *par,
                              Sh x, Sh f, double *Jout) {
  const int K = B.ipar[1], m = B.m;
  const int *cm = B.n_in ? S.jcol_g + B.joff : nullptr;  // column map
  for (int r = threadIdx.x; r < m; r += TEAM) {
    const int t = r / K, k = r % K;
    const int i0 = cm ? __ldg(cm + 2 * r) : 2 * t, i1 = cm ? __ldg(cm + 2 * r + 1) : 2 * t + 1;
    const double dx = x[i0] - par[2 * k], dy = x[i1] - par[2 * k + 1];
    const double dist = sqrt(dx * dx + dy * dy);
    f[r] = par[2 * K + k] - dist;
    if (Jout) {
      Jout[2 * r] = -dx / dist;
      Jout[2 * r + 1] = -dy / dist;
    }
  }
}

// ---- FK7: flange position of a 7-link modified-DH chain.  tab = a[7] d[7] cos(alpha)[7]
// sin(alpha)[7] flange base_step ----
// Every operation is rounded on its own (__dmul_rn / __dadd_rn are never contracted into FMAs) and three-term
// sums run left to right: the very sequence of oracle/families.py:fk7_pos, so that the two sides differ only
// through sin / cos.  profiles/arm_sensitivity.py: ~10 ulp of difference in f make the SQP of an occasional
// arm problem stop one iteration earlier or later (|dx| ~ 1e-3); ~1 ulp does not.
__device__ __forceinline__ double dot3_rn(double a0, double b0, double a1, double b1, double a2, double b2) {
  return __dadd_rn(__dadd_rn(__dmul_rn(a0, b0), __dmul_rn(a1, b1)), __dmul_rn(a2, b2));
}
__device__ __forceinline__ void fk7_pos(const double *q, const double *tab, double out[3]) {
  double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  double p[3] = {0, 0, 0};
  for (int i = 0; i < 7; i++) {
    const double ai = tab[i], di = tab[7 + i], ca = tab[14 + i], sa = tab[21 + i];
    double st, ct;
    sincos(q[i], &st, &ct);
    const double Ri[9] = {ct, -st, 0.0, __dmul_rn(st, ca), __dmul_rn(ct, ca), -sa, __dmul_rn(st, sa), __dmul_rn(ct, sa), ca};
    const double pi3[3] = {ai, __dmul_rn(-sa, di), __dmul_rn(ca, di)};
    for (int r = 0; r < 3; r++)
      p[r] = __dadd_rn(p[r], dot3_rn(R[3 * r], pi3[0], R[3 * r + 1], pi3[1], R[3 * r + 2], pi3[2]));
    double Rn[9];
    for (int r = 0; r < 3; r++)
      for (int cc = 0; cc < 3; cc++)
        Rn[3 * r + cc] = dot3_rn(R[3 * r], Ri[cc], R[3 * r + 1], Ri[3 + cc], R[3 * r + 2], Ri[6 + cc]);
    for (int e = 0; e < 9; e++) R[e] = Rn[e];
  }
  const double fl = tab[28];
  for (int r = 0; r < 3; r++) out[r] = __dadd_rn(p[r], dot3_rn(R[3 * r], 0.0, R[3 * r + 1], 0.0, R[3 * r + 2], fl));
}

// Central differences at steps h and 2h, Richardson-combined -- the scheme of
// oracle/shims/numdifftools (restating numdifftools.Jacobian as called at expr.py:67).
// Without a column map one instance on x[n-7:n]; with one, instance i (rows 3i..3i+2) on x[cols[21i + k]], its joints
// gathered into stage[98..104] (sco_create gives a structure with a mapped FK7 block a stage of >= 106 doubles).
template <int TEAM>
__device__ void eval_fk7(const DevStruct &S, const DevBlock &B, const double *tab, Sh x, Sh f,
                         double *Jout, Sh stage) {
  const int n = S.n, t = threadIdx.x;
  const int ninst = B.n_in ? B.m / 3 : 1;
  for (int inst = 0; inst < ninst; inst++) {
    const int *cm = B.n_in ? S.jcol_g + B.joff + inst * 21 : nullptr;  // column map of the instance's first row
    const Sh q = cm ? stage + 98 : x + (n - 7);                           // its joints
    if (cm) {
      Team<TEAM>::sync();  // the stage may still be read (previous instance or block)
      for (int k = t; k < 7; k += TEAM) q[k] = x[__ldg(cm + k)];
      Team<TEAM>::sync();
    }
    if (t == 0) {
      double o[3], q0[7];
      for (int k = 0; k < 7; k++) q0[k] = q[k];
      fk7_pos(q0, tab, o);
      f[3 * inst] = o[0]; f[3 * inst + 1] = o[1]; f[3 * inst + 2] = o[2];
    }
    if (Jout) {
      // thread e = col*4 + (mult_idx*2 + sign): 28 evaluations -> stage[e*3 .. e*3+2]; stage[84+..] = hh
      for (int e = t; e < 28; e += TEAM) {
        const int col = e >> 2, mi = (e >> 1) & 1, sg = e & 1;
        double qq[7];
        for (int k = 0; k < 7; k++) qq[k] = q[k];
        const double h0 = tab[29] * fmax(log1p(fabs(q[col])), 1.0);
        const double h = h0 * (mi ? 2.0 : 1.0);
        const double xp = q[col] + h, xm = q[col] - h;
        qq[col] = sg ? xm : xp;
        double o[3];
        fk7_pos(qq, tab, o);
        stage[e * 3] = o[0]; stage[e * 3 + 1] = o[1]; stage[e * 3 + 2] = o[2];
        if (sg == 0) stage[84 + col * 2 + mi] = xp - xm;
      }
      Team<TEAM>::sync();
      double *J = Jout + inst * 21;
      for (int e = t; e < 21; e += TEAM) {
        const int r = e / 7, col = e % 7;
        const double d1 = (stage[(col * 4 + 0) * 3 + r] - stage[(col * 4 + 1) * 3 + r]) / stage[84 + col * 2];
        const double d2 = (stage[(col * 4 + 2) * 3 + r] - stage[(col * 4 + 3) * 3 + r]) / stage[84 + col * 2 + 1];
        J[r * 7 + col] = (4.0 * d1 - d2) / 3.0;
      }
    }
  }
}


// ---- VM: rows given as stack programs (sco_py_b200/sym.py).  Program = m row offsets, then
// (opcode, operand) pairs of doubles; opcodes END 0, PUSH_X 1, PUSH_C 2, ADD 3, SUB 4, MUL 5, DIV 6,
// NEG 7, POWI 8, SQRT 9, LOG 10, EXP 11, SIN 12, COS 13, ABS 14, MIN 15, MAX 16, TEE 17 (copy the top of the stack
// into temporary k), LOAD 18 (push temporary k).  Up to two variables may be replaced by
// given values (the perturbed points of the finite differences) without copying x.  `cols` is the row's column map
// (PUSH_X k reads x[cols[k]]) or null (PUSH_X k reads x[k]); pi / pj / wrt name local inputs.
#define SCO_VM_STACK 16
#define SCO_VM_SLOTS 128  // a seven-link kinematic chain keeps ~100 rotation entries alive
#define SCO_FD_JAC_STEP 5.477420592293901e-07    // eps^(1/2.5): numdifftools base step, first derivatives
#define SCO_FD_HESS_STEP 9.843133202303692e-03  // eps^(1/7.8): second derivatives (oracle/shims/numdifftools)

static __device__ __noinline__ double vm_eval(const double *prog, int m, int row, Sh x, const int *cols, int pi, double vi,
                                              int pj, double vj) {
  const double *ins = prog + m;
  int pc = (int)prog[row];
  double stk[SCO_VM_STACK], slot[SCO_VM_SLOTS];
  int sp = 0;
  for (;;) {
    const int op = (int)ins[2 * pc];
    const double arg = ins[2 * pc + 1];
    pc++;
    if (op == 0) break;
    if (op == 1) {
      const int i = (int)arg;
      stk[sp++] = i == pi ? vi : (i == pj ? vj : x[cols ? __ldg(cols + i) : i]);
    } else if (op == 2) {
      stk[sp++] = arg;
    } else if (op <= 6) {
      const double b = stk[--sp], a = stk[sp - 1];
      stk[sp - 1] = op == 3 ? a + b : op == 4 ? a - b : op == 5 ? a * b : a / b;
    } else if (op == 7) {
      stk[sp - 1] = -stk[sp - 1];
    } else if (op == 8) {
      const double a = stk[sp - 1];
      double v = 1.0;
      for (int k = (int)arg; k > 0; k--) v = v * a;
      stk[sp - 1] = v;
    } else if (op <= 13) {
      const double a = stk[sp - 1];
      stk[sp - 1] = op == 9 ? sqrt(a) : op == 10 ? log(a) : op == 11 ? exp(a) : op == 12 ? sin(a) : cos(a);
    } else if (op == 14) {
      stk[sp - 1] = fabs(stk[sp - 1]);
    } else if (op <= 16) {
      const double b = stk[--sp], a = stk[sp - 1];
      stk[sp - 1] = op == 15 ? (a <= b ? a : b) : (a >= b ? a : b);
    } else if (op == 17) {
      slot[(int)arg] = stk[sp - 1];
    } else {
      stk[sp++] = slot[(int)arg];
    }
  }
  return stk[sp - 1];
}

// The same program in forward mode: value and d/dx_wrt, the exact counterpart of a user-supplied gradient
// (Expr(f, grad), expr.py:86-88); SymExpr(..., analytic=True).  Rules as in sym.eval_program_dual.
static __device__ __noinline__ double vm_eval_dual(const double *prog, int m, int row, Sh x, const int *cols, int wrt,
                                                   double *dout) {
  const double *ins = prog + m;
  int pc = (int)prog[row];
  double stk[SCO_VM_STACK], dsk[SCO_VM_STACK], slot[SCO_VM_SLOTS], dslot[SCO_VM_SLOTS];
  int sp = 0;
  for (;;) {
    const int op = (int)ins[2 * pc];
    const double arg = ins[2 * pc + 1];
    pc++;
    if (op == 0) break;
    if (op == 1) {
      const int i = (int)arg;
      stk[sp] = x[cols ? __ldg(cols + i) : i];
      dsk[sp++] = i == wrt ? 1.0 : 0.0;
    } else if (op == 2) {
      stk[sp] = arg;
      dsk[sp++] = 0.0;
    } else if (op <= 6) {
      --sp;
      const double b = stk[sp], db = dsk[sp], a = stk[sp - 1], da = dsk[sp - 1];
      if (op == 3) { stk[sp - 1] = a + b; dsk[sp - 1] = da + db; }
      else if (op == 4) { stk[sp - 1] = a - b; dsk[sp - 1] = da - db; }
      else if (op == 5) { stk[sp - 1] = a * b; dsk[sp - 1] = da * b + a * db; }
      else { const double q = a / b; stk[sp - 1] = q; dsk[sp - 1] = (da - q * db) / b; }
    } else if (op == 7) {
      stk[sp - 1] = -stk[sp - 1];
      dsk[sp - 1] = -dsk[sp - 1];
    } else if (op == 8) {
      const double a = stk[sp - 1];
      const int k = (int)arg;
      double v = 1.0, vm1 = 1.0;
      for (int t = 0; t < k; t++) { vm1 = v; v = v * a; }
      stk[sp - 1] = v;
      dsk[sp - 1] = k > 0 ? k * vm1 * dsk[sp - 1] : 0.0;
    } else if (op <= 13) {
      const double a = stk[sp - 1], da = dsk[sp - 1];
      if (op == 9) { const double v = sqrt(a); stk[sp - 1] = v; dsk[sp - 1] = da != 0.0 ? da / (2.0 * v) : 0.0; }  // sqrt of a constant 0 is flat
      else if (op == 10) { stk[sp - 1] = log(a); dsk[sp - 1] = da / a; }
      else if (op == 11) { const double v = exp(a); stk[sp - 1] = v; dsk[sp - 1] = v * da; }
      else if (op == 12) { stk[sp - 1] = sin(a); dsk[sp - 1] = cos(a) * da; }
      else { stk[sp - 1] = cos(a); dsk[sp - 1] = -sin(a) * da; }
    } else if (op == 14) {
      const double a = stk[sp - 1];
      stk[sp - 1] = fabs(a);
      if (!(a >= 0.0)) dsk[sp - 1] = -dsk[sp - 1];
    } else if (op <= 16) {
      --sp;
      const double b = stk[sp], a = stk[sp - 1];
      const bool keep_a = op == 15 ? a <= b : a >= b;
      if (!keep_a) { stk[sp - 1] = b; dsk[sp - 1] = dsk[sp]; }
    } else if (op == 17) {
      slot[(int)arg] = stk[sp - 1];
      dslot[(int)arg] = dsk[sp - 1];
    } else {
      stk[sp] = slot[(int)arg];
      dsk[sp++] = dslot[(int)arg];
    }
  }
  *dout = dsk[sp - 1];
  return stk[sp - 1];
}

// d f_row / d x_j by two central differences, Richardson-combined (numdifftools.Jacobian as called at
// expr.py:67; the scheme of oracle/shims/numdifftools.jacobian_fd)
static __device__ double vm_fd1(const double *prog, int m, int row, Sh x, const int *cols, int j) {
  const double xj = x[cols ? __ldg(cols + j) : j];
  const double h0 = SCO_FD_JAC_STEP * fmax(log1p(fabs(xj)), 1.0);
  double est[2];
  for (int k = 0; k < 2; k++) {
    const double h = h0 * (k ? 2.0 : 1.0);
    const double xp = xj + h, xm = xj - h;
    est[k] = (vm_eval(prog, m, row, x, cols, j, xp, -1, 0.0) - vm_eval(prog, m, row, x, cols, j, xm, -1, 0.0)) / (xp - xm);
  }
  return (4.0 * est[0] - est[1]) / 3.0;
}

// d2 f_row / d x_i d x_j: central second differences at h and 2h, Richardson-combined (numdifftools.Hessian as called
// at expr.py:108; oracle/shims/numdifftools.hessian_fd).  i, j are local inputs of the row (x[cols[i]] with a map).
static __device__ double vm_fd2(const double *prog, int m, int row, Sh x, const int *cols, int i, int j, double f0) {
  const double xi = x[cols ? __ldg(cols + i) : i], xj = x[cols ? __ldg(cols + j) : j];
  const double hi0 = SCO_FD_HESS_STEP * fmax(log1p(fabs(xi)), 1.0), hj0 = SCO_FD_HESS_STEP * fmax(log1p(fabs(xj)), 1.0);
  double est[2];
  for (int k = 0; k < 2; k++) {
    const double hi = hi0 * (k ? 2.0 : 1.0), hj = hj0 * (k ? 2.0 : 1.0);
    if (i == j) {
      est[k] = (vm_eval(prog, m, row, x, cols, i, xi + 2.0 * hi, -1, 0.0) - 2.0 * f0 + vm_eval(prog, m, row, x, cols, i, xi - 2.0 * hi, -1, 0.0)) /
               (4.0 * hi * hi);
    } else {
      est[k] = (vm_eval(prog, m, row, x, cols, i, xi + hi, j, xj + hj) - vm_eval(prog, m, row, x, cols, i, xi + hi, j, xj - hj) -
                vm_eval(prog, m, row, x, cols, i, xi - hi, j, xj + hj) + vm_eval(prog, m, row, x, cols, i, xi - hi, j, xj - hj)) /
               (4.0 * hi * hj);
    }
  }
  return (4.0 * est[0] - est[1]) / 3.0;
}

// With a column map row r is a function of its n_in inputs: n_in Jacobian entries per row instead of n.
template <int TEAM>
__device__ void eval_vm(const DevStruct &S, const DevBlock &B, const double *prog, Sh x, Sh f, double *Jout) {
  const int *cm = B.n_in ? S.jcol_g + B.joff : nullptr;  // column map
  const int n = cm ? B.n_in : S.n, m = B.m;
  for (int r = threadIdx.x; r < m; r += TEAM) f[r] = vm_eval(prog, m, r, x, cm ? cm + r * n : nullptr, -1, 0.0, -1, 0.0);
  if (Jout) {
    if (B.ipar[3]) {  // analytic: the program differentiated in forward mode (one pass per entry)
      for (int e = threadIdx.x; e < m * n; e += TEAM) {
        double d;
        vm_eval_dual(prog, m, e / n, x, cm ? cm + (e / n) * n : nullptr, e % n, &d);
        Jout[e] = d;
      }
    } else {
      for (int e = threadIdx.x; e < m * n; e += TEAM) Jout[e] = vm_fd1(prog, m, e / n, x, cm ? cm + (e / n) * n : nullptr, e % n);
    }
  }
}

// Evaluate every block at x: fv[row] = f_row(x); if Jg != null also the stored Jacobian entries.
// Ends with a team sync.
template <int TEAM>
__device__ __noinline__ void eval_blocks(const DevStruct &S, const double *prm, Sh x, Sh fv, double *Jg, Sh stage) {
  for (int bi = 0; bi < S.n_blocks; bi++) {
    const DevBlock &B = S.blocks[bi];
    const double *par = field_ptr(S, B.par, prm);
    const Sh f = fv + B.row0;
    double *J = Jg ? Jg + B.joff : nullptr;
    if (B.family == FAM_QUADFORM) eval_quadform<TEAM>(S, B, par, x, f, J, stage);
    else if (B.family == FAM_CIRCLE2D) eval_circle2d<TEAM>(S, B, par, x, f, J);
    else if (B.family == FAM_FK7) eval_fk7<TEAM>(S, B, par, x, f, J, stage);
    else if (B.family == FAM_VM) eval_vm<TEAM>(S, B, par, x, f, J);
  }
  Team<TEAM>::sync();
}
