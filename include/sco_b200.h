/*
 * sco_b200.h -- C ABI of the B200-native batched penalty-SQP engine.
 *
 * Drop-in boundary for the hot path of Algorithmic-Alignment-Lab/sco_py's OSQP
 * backend (the "backend package triple" Prob / Solver / Variable, SURVEY.md
 * section 8b).  One handle = one problem STRUCTURE (shared by a batch of B
 * independent problems) bound to one CUDA device.  All pointers named d_* are
 * device pointers (e.g. torch.Tensor.data_ptr()), row-major, batch-major,
 * float64 / int32, 16-byte aligned, owned by the caller.  Functions return 0 on
 * success or a negative error code; sco_last_error() (thread-local) explains.
 * There is no CPU fallback: every entry point fails with SCO_ERR_CUDA if no
 * sm_100 device is usable.
 *
 * Reference interfaces replaced (paths relative to the reference repository):
 *   sco_create / sco_destroy   <- Prob.add_obj_expr / add_cnt_expr bookkeeping and the
 *                                 variable ordering + row layout of osqp_utils.optimize
 *                                 (sco_py/sco_osqp/prob.py:88-144, osqp_utils.py:136-189)
 *   sco_solve_batch            <- Solver.solve(prob, method="penalty_sqp", ...)
 *                                 (sco_py/sco_osqp/solver.py:30-253)
 *   sco_convexify              <- Prob.convexify (prob.py:522-544), Expr.eval/grad/convexify
 *                                 (sco_py/expr.py:34-41,78-100,130-142), Eq/LEqExpr.convexify
 *                                 (expr.py:314-332,353-371)
 *   sco_qp_solve               <- Prob.update_obj + Prob.add_trust_region + Prob.optimize ->
 *                                 osqp_utils.optimize -> osqp.OSQP().setup/solve
 *                                 (prob.py:146-205,414-512,514-519; osqp_utils.py:113-221)
 *   sco_merit                  <- Prob.get_value / get_approx_value / get_max_cnt_violation
 *                                 (prob.py:547-630)
 */
#ifndef SCO_B200_H
#define SCO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCO_MAX_BLOCKS 16
#define SCO_MAX_GROUPS 8
#define SCO_MAX_OBJ_BLOCKS 4

/* nonlinear constraint families evaluated on device (closed set; the reference takes
 * black-box Python callables, sco_py/expr.py:22-25) */
#define SCO_FAM_QUADFORM 1 /* f_j = 0.5 x'P_j x + a_j'x ; par = P packed-upper [m][n(n+1)/2], a [m][n] */
#define SCO_FAM_CIRCLE2D 2 /* f_{t,k} = R_k - |p_t - c_k| ; ipar = {T, K} ; par = c [K][2], R [K]      */
#define SCO_FAM_FK7 3      /* flange position of a 7-link DH chain on x[n-7:n], finite-difference Jacobian */
#define SCO_FAM_VM 4       /* rows given as stack programs (sco_py_b200/sym.py): par = m row offsets, then
                              (opcode, operand) pairs; ipar = {n, m, instructions, analytic}; analytic = 0:
                              finite-difference Jacobian, like a black-box Expr without grad (expr.py:61-69);
                              analytic = 1: the program differentiated in forward mode, like Expr(f, grad) (:86-88) */
/* Column maps (sco_block_desc.cols, the Variable a BoundExpr is bound to, expr.py:413-437).  cols = NULL: the
 * columns above, every row over all n variables (CIRCLE2D: x[2t], x[2t+1]; FK7: x[n-7:n]).  Otherwise row r
 * reads x[cols[r*n_in + i]] as its local input i, and the formulas above hold with n replaced by n_in:
 *   QUADFORM, VM: row r is a function of its n_in local inputs; P_r is packed over n_in, a_r has n_in entries,
 *                 PUSH_X operands are local indices, ipar[0] = n_in.  Rows of different maps may share a block.
 *   CIRCLE2D:     n_in = 2; row r reads the point (x[cols[2r]], x[cols[2r+1]]) against circle r % K; T = m / K.
 *   FK7:          n_in = 7; m is a multiple of 3, rows 3i..3i+2 are instance i (one flange position), have the
 *                 same map, and every instance uses the block's one DH table.
 * Indices lie in [0, n) and do not repeat within a row.  A block with a map never takes the dense QP kernels
 * (sco_dense.cuh), which assume rows over all n variables. */

#define SCO_CNT_LEQ 0 /* LEqExpr -> hinge penalty, one slack per row  (expr.py:353-371) */
#define SCO_CNT_EQ 1  /* EqExpr  -> abs penalty, two slacks per row   (expr.py:314-332) */

/* OSQP status codes as consumed at prob.py:197 */
#define SCO_QP_SOLVED 1
#define SCO_QP_SOLVED_INACCURATE 2
#define SCO_QP_PRIMAL_INFEASIBLE_INACCURATE 3
#define SCO_QP_DUAL_INFEASIBLE_INACCURATE 4
#define SCO_QP_MAX_ITER_REACHED (-2)
#define SCO_QP_PRIMAL_INFEASIBLE (-3)
#define SCO_QP_DUAL_INFEASIBLE (-4)
#define SCO_QP_NON_CVX (-7)

/* per-problem verdicts of sco_solve_batch (Solver.solve returns bool; the reason is extra) */
#define SCO_VERDICT_FAILED 0        /* solve() would return False                         */
#define SCO_VERDICT_CONVERGED 1     /* solve() would return True                          */
#define SCO_VERDICT_ITER_CAP (-1)   /* safety cap on SQP iterations hit (reference: none) */
#define SCO_VERDICT_BAD_ORDER (-3)  /* sco_solve_batch_ordered: d_order is not a permutation of 0..B-1 */

#define SCO_OK 0
#define SCO_ERR_ARG (-1)
#define SCO_ERR_CUDA (-2)
#define SCO_ERR_UNSUPPORTED (-3)

typedef struct sco_handle sco_handle;

typedef struct {
  int64_t off;    /* offset in doubles inside the per-problem (or shared) block; -1 = absent (zeros) */
  int32_t shared; /* 1: lives in the shared block, 0: once per problem */
  int32_t pad_;
} sco_field;

typedef struct {
  int32_t family;     /* SCO_FAM_*  */
  int32_t cnt_type;   /* SCO_CNT_*  */
  int32_t m;          /* rows */
  int32_t group_mask; /* bit g set <=> member of constraint group g (prob.py:135-142) */
  int32_t jw;         /* Jacobian entries stored per row */
  int32_t n_in;       /* inputs per row when cols != NULL (see the column maps above); ignored otherwise */
  int32_t ipar[8];
  sco_field par; /* family parameters */
  sco_field val; /* CompExpr.val, m doubles */
  const int32_t *cols; /* host, m * n_in column indices, row-major, or NULL (implied columns) */
} sco_block_desc;

typedef struct {
  int32_t m;           /* terms, one scalar program row each */
  int32_t n_in;        /* inputs per term, 1..64 */
  int32_t n_instr;     /* instructions of the packed program */
  int32_t flags;       /* bit 0: forward-mode gradient (SymExpr analytic=True) */
  sco_field prog;      /* m row offsets, then 2*n_instr */
  const int32_t *cols; /* host, m*n_in column indices (the Variable's order) */
} sco_obj_block_desc;

typedef struct {
  int32_t n;        /* user variables (sorted-name order, osqp_utils.py:136-143) */
  int32_t m_lin;    /* linear Eq/LEq rows added at add_cnt_expr time (prob.py:317-346) */
  int32_t n_blocks; /* nonlinear constraint blocks */
  int32_t n_groups;
  int64_t stride;     /* doubles per problem block */
  int64_t shared_len; /* doubles in the shared block */
  sco_field Q;        /* n*n row-major, QuadExpr.Q (symmetrised as osqp_utils.py:153-163) */
  sco_field q;        /* n, QuadExpr.A */
  sco_field c;        /* 1, QuadExpr.b */
  sco_field lin_l;    /* m_lin */
  sco_field lin_u;    /* m_lin */
  const int32_t *lin_rowptr; /* host, CSR of the linear rows; pattern and values shared by the batch */
  const int32_t *lin_col;
  const double *lin_val;
  const double *shared;         /* host, shared_len doubles */
  const int32_t *group_overlap; /* host, n_groups*n_groups or NULL */
  sco_block_desc blocks[SCO_MAX_BLOCKS];
  /* non-quadratic objective term (prob.py:97-103 _nonquad_obj_exprs): one scalar stack program, convexified to
   * degree 2 every SQP iteration -- finite-difference gradient and Hessian, eigenvalue shift (expr.py:102-156) */
  sco_field obj_prog;
  int32_t obj_prog_len;   /* instructions; 0 = none */
  int32_t obj_prog_flags; /* bit 0: gradient by forward-mode differentiation of the program (Expr(f, grad),
                             expr.py:86-88) instead of finite differences; the Hessian stays numerical (expr.py:102-109) */
  /* AffExpr objective terms (prob.py:97-103 files them under _quad_obj_exprs): the sum of their A rows, n doubles
   * (their constants go into c).  The exact merit uses a'x (AffExpr.eval, expr.py:173-174); the QP uses
   * w * a'x with the weight of quirk C-4 (prob.py:220-221,240-249,424-426: every update_obj appends another
   * copy and multiplies all copies by the penalty coefficient, w <- (w + 1) * mu) unless
   * sco_settings.aff_obj_quirk = 0 (w = 1, the Gurobi backend's semantics). */
  sco_field qa;
  /* user bounds of the scalar variables (OSQPVar lb / ub), n doubles each; honoured by the closest-point QP
   * (prob.py:369-412) -- the first trust region overwrites them (variable.py:37-45).  -1 = (-inf, +inf). */
  sco_field lb0;
  sco_field ub0;
  /* Non-quadratic objective terms, each bound to its own Variable (prob.py:97-103; BoundExpr, expr.py:413-437).
   * Terms with the same input count and derivative mode share a block: one scalar program row per term, and a
   * column map like that of a constraint block -- term r of a block reads x[cols[r*n_in + i]] as its local input i.
   * Every term is convexified on its own, as Expr.convexify(degree=2) does per term (expr.py:143-153): H_t = the
   * numerical Hessian over its n_in inputs, H_t+ = H_t - min(lambda_min(H_t), 0) I, A_t = g_t - x_t'H_t+,
   * b_t = 0.5 x_t'H_t+ x_t - g_t.x_t + f_t; the QP adds sum_t scatter(H_t+) to P and sum_t scatter(A_t) to q
   * (prob.py:348-367), the merits sum_t f_t (prob.py:573-574) and sum_t of the models (prob.py:624-626).
   * Indices lie in [0, n) and do not repeat within a term, 1 <= n_in <= 64.  obj_prog above is the same thing for
   * one term over all n variables in QP order (n <= 64); a structure has one or the other, not both.  Hosts that
   * memset this struct get n_obj_blocks = 0. */
  int32_t n_obj_blocks;
  sco_obj_block_desc obj_blocks[SCO_MAX_OBJ_BLOCKS];
} sco_structure_desc;

typedef struct {
  /* Solver attributes, sco_py/sco_osqp/solver.py:17-28 */
  double improve_ratio_threshold;
  double min_trust_region_size;
  double min_approx_improve;
  double trust_shrink_ratio;
  double trust_expand_ratio;
  double cnt_tolerance;
  double merit_coeff_increase_ratio;
  double initial_trust_region_size;
  double initial_penalty_coeff;
  int32_t max_merit_coeff_increases;
  int32_t max_sqp_iters; /* safety cap on convexifications per problem (reference has none, solver.py:126) */
  /* OSQP settings, osqp_utils.py:10-15,197-214 (+ upstream defaults, SURVEY.md Appendix B) */
  double osqp_eps_abs;
  double osqp_eps_rel;
  double osqp_rho;
  double osqp_sigma;
  double osqp_alpha;
  double osqp_eps_prim_inf;
  double osqp_eps_dual_inf;
  int32_t osqp_max_iter;
  int32_t osqp_scaling;
  int32_t osqp_check_termination;
  int32_t osqp_adaptive_rho;
  int32_t osqp_adaptive_rho_interval;
  /* OSQP-backend quirks (SURVEY.md Appendix C); 1 = behave like the reference */
  int32_t compound_penalty; /* C-1, prob.py:424-426 */
  int32_t freeze_sparsity;  /* C-2, prob.py:488-504 */
  int32_t duplicate_rows;   /* C-3, prob.py:508-509 */
  int32_t threads_per_problem; /* 0 = choose from the structure */
  int32_t force_generic;       /* 1 = never take the register-resident dense ADMM loop (A/B parity checks) */
  int32_t aff_obj_quirk;       /* C-4, prob.py:240-249: AffExpr objectives weighted like penalty terms */
  int32_t warm_start;          /* 0 = every QP starts from x = z = y = 0 like the reference (osqp_utils.py:195 builds a
                                  new OSQP object per call); 1 = QPs inside one trust-region loop (only l, u change,
                                  solver.py:136-146) reuse scaling and factorisation and start from the previous
                                  iterates; 2 = additionally warm-start x, y across SQP iterations */
  int32_t pad_;
} sco_settings;

const char *sco_last_error(void);
void sco_default_settings(sco_settings *s);

int sco_create(const sco_structure_desc *desc, int device, sco_handle **out);
int sco_destroy(sco_handle *h);

/* sizes derived from the structure: out[0]=n, [1]=m_nl, [2]=n_slack, [3]=jnnz (stored Jacobian
 * entries per problem), [4]=n_q, [5]=shared-memory bytes per problem, [6]=threads per problem,
 * [7]=resident problems per SM */
int sco_query(sco_handle *h, int64_t *out8);

/* Full penalty-SQP on B problems.  stats[b] = {sqp_iters, qp_solves, admm_iters, last_qp_status}. */
int sco_solve_batch(sco_handle *h, int64_t B, const double *d_params, const double *d_x0,
                    const sco_settings *s, double *d_x_out, int32_t *d_verdict, double *d_merit,
                    double *d_objective, double *d_max_vio, int32_t *d_stats, void *stream);

/* Same, with a processing order: the work queue hands out problem d_order[0], d_order[1], ... (a permutation
 * of 0..B-1 on the device; NULL = index order).  Results stay at their own index.  Iteration counts are
 * heavy-tailed and a problem is sequential, so a launch ends when its longest problem does; a caller that
 * re-solves similar batches (replanning, MPC) passes last time's stats[:, 2] sorted in descending order. */
int sco_solve_batch_ordered(sco_handle *h, int64_t B, const double *d_params, const double *d_x0,
                            const sco_settings *s, double *d_x_out, int32_t *d_verdict, double *d_merit,
                            double *d_objective, double *d_max_vio, int32_t *d_stats, const int32_t *d_order,
                            void *stream);

/* The general form: every buffer of a batch in one struct (device pointers; NULL = not wanted / not given).
 *   nonconverged[b]: bit g      <=> constraint group g (sorted group ids, prob.py:540-542) is in
 *                                   prob.nonconverged_groups after the first loop of solver.py:209-225,
 *                    bit 16 + g <=> group g is appended again by the second loop (solver.py:231-233);
 *                    the value of the last evaluation of that block, like the attribute of the reference.
 *   order: see sco_solve_batch_ordered.  An order that is not a permutation of 0..B-1 is detected on the
 *          device before the solve starts; every verdict of the batch is then SCO_VERDICT_BAD_ORDER and nothing
 *          else is written.
 *   y_warm / x_warm: reserved (must be NULL). */
typedef struct {
  const double *d_params, *d_x0;
  double *d_x_out;
  int32_t *d_verdict;
  double *d_merit, *d_objective, *d_max_vio;
  int32_t *d_stats;
  int32_t *d_nonconverged;
  const int32_t *d_order;
  const double *d_x_warm, *d_y_warm;
} sco_batch_io;
int sco_solve_batch_io(sco_handle *h, int64_t B, const sco_batch_io *io, const sco_settings *s, void *stream);

/* Launches of one handle may be in flight on several streams at once (each owns one of SCO_LAUNCH_SLOTS launch
 * slots: work-queue counter + Jacobian scratch); calls on one handle must come from one host thread. */
#define SCO_LAUNCH_SLOTS 16
#define SCO_STAGING_SETS 8

/* Same with HOST buffers: copies in, solves, copies out -- all enqueued on `stream`, no host
 * synchronisation (pinned buffers make the copies asynchronous; the caller synchronises the stream
 * before reading the outputs).  Up to SCO_STAGING_SETS calls may be in flight (one staging set each).
 * `nonconverged` may be NULL (see sco_batch_io). */
int sco_solve_batch_host_async(sco_handle *h, int64_t B, const double *params, const double *x0,
                               const sco_settings *s, double *x_out, int32_t *verdict, double *merit,
                               double *objective, double *max_vio, int32_t *stats, void *stream);
int sco_solve_batch_host_groups(sco_handle *h, int64_t B, const double *params, const double *x0,
                                const sco_settings *s, double *x_out, int32_t *verdict, double *merit,
                                double *objective, double *max_vio, int32_t *stats, int32_t *nonconverged,
                                void *stream);

/* Same on the default stream, then synchronises (pinned or pageable buffers). */
int sco_solve_batch_host(sco_handle *h, int64_t B, const double *params, const double *x0,
                         const sco_settings *s, double *x_out, int32_t *verdict, double *merit,
                         double *objective, double *max_vio, int32_t *stats);

/* ---- stage entry points (parity tests / integration of single steps) ---- */

/* f[B,m_nl] = block functions at x ; J[B,jnnz] stored Jacobian entries ; b[B,m_nl] = f - Jx - val ;
 * obj[B] = 0.5x'Qx + q'x + c.  Any output may be NULL. */
int sco_convexify(sco_handle *h, int64_t B, const double *d_params, const double *d_x, double *d_f,
                  double *d_J, double *d_b, double *d_obj, void *stream);
/* Same, plus the convex degree-2 model of the non-quadratic objective terms (Expr.hess / _num_hess and
 * Expr.convexify degree 2, expr.py:102-128,143-153), each term convexified on its own and the models summed:
 * H+ = sum_t scatter(H_t - min(lambda_min(H_t), 0) I) [B,n,n], A = sum_t scatter(grad_t - x_t'H_t+) [B,n],
 * b = sum_t (0.5 x_t'H_t+ x_t - grad_t.x_t + f_t) [B].  Any output may be NULL; an error if the structure has no such
 * term. */
int sco_convexify_model(sco_handle *h, int64_t B, const double *d_params, const double *d_x, double *d_f,
                        double *d_J, double *d_b, double *d_obj, double *d_H, double *d_g, double *d_c,
                        void *stream);

/* One penalty QP per problem:  min 0.5 x'sym(Q)x + q'x + pi*1's  s.t. lin rows, kdup copies of the
 * penalty rows (J.*mask) x -/+ s {<=,=} -b, lbx <= x <= ubx, s >= 0.   use_penalty=0 drops the
 * penalty rows and slacks; closest_point=1 replaces the objective by |x - xref|^2 (prob.py:369-412).
 * d_mask[B,m_nl,W] uint32, W = ceil(widest stored Jacobian row / 32) (1 for rows of up to 32 entries):
 * bit (s & 31) of word s >> 5 <=> slot s of the row participates (NULL = all).
 * Outputs: x[B,n_q] (user variables then slacks, unscaled), status[B], iters[B]. */
int sco_qp_solve(sco_handle *h, int64_t B, const double *d_params, const double *d_J,
                 const double *d_b, const uint32_t *d_mask, const double *d_lbx, const double *d_ubx,
                 const double *d_pi, const int32_t *d_kdup, const double *d_xref, int use_penalty,
                 int closest_point, const sco_settings *s, double *d_xq, int32_t *d_status,
                 int32_t *d_iters, void *stream);
/* Same with the weight of the AffExpr objective terms per problem (d_wa[B]; NULL = 1, see sco_structure_desc.qa). */
int sco_qp_solve_w(sco_handle *h, int64_t B, const double *d_params, const double *d_J,
                   const double *d_b, const uint32_t *d_mask, const double *d_lbx, const double *d_ubx,
                   const double *d_pi, const int32_t *d_kdup, const double *d_wa, const double *d_xref,
                   int use_penalty, int closest_point, const sco_settings *s, double *d_xq, int32_t *d_status,
                   int32_t *d_iters, void *stream);

/* merit[B] = obj + mu*sum(viol), model[B] = obj + mu*sum(pen(Jx+b)) (J, b from a previous
 * sco_convexify at another point), max_vio[B], group sums gv[B,n_groups] / gm[B,n_groups]. */
int sco_merit(sco_handle *h, int64_t B, const double *d_params, const double *d_x, const double *d_J,
              const double *d_b, const double *d_mu, double *d_merit, double *d_model,
              double *d_max_vio, double *d_gv, double *d_gm, void *stream);

/* ---- measurement helper (bench.py): sustained FP64 FMA rate of the device in TFLOP/s, the
 * compute roofline of the shared-memory-resident ADMM kernel.  Not on the solve path; the
 * reference has no counterpart. */
int sco_probe_fp64(int device, double *tflops_out);

#ifdef __cplusplus
}
#endif
#endif /* SCO_B200_H */
