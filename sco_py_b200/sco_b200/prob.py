"""Prob: the problem container of the backend, with the method surface of
sco_py/sco_osqp/prob.py (add_var :106, add_osqp_var :109, add_obj_expr :88, add_cnt_expr :112,
optimize :146, find_closest_feasible_point :369, update_obj :414, add_trust_region :514,
convexify :522, get_value :547, get_max_cnt_violation :592, get_approx_value :605, save :639,
restore :647, nonconverged_groups).

`Solver.solve(prob)` / `Solver.solve_batch(probs)` run the whole penalty SQP in one kernel
(sco_solve_batch).  The step methods of this class (convexify, update_obj, add_trust_region,
optimize, get_value, ...) drive the same device code one stage at a time through the stage entry
points of the C ABI (sco_convexify / sco_qp_solve / sco_merit) for a batch of one, with the
reference's bookkeeping quirks kept: the penalty weight compounds across update_obj calls (C-1), the
Jacobian sparsity is frozen at the first convexification (C-2), every update_obj adds another copy
of the penalty rows (C-3).  Nothing numerical runs on the host.
"""
from collections import OrderedDict

import numpy as np

from .. import batch
from .. import expr as E


class Prob(object):
    def __init__(self, callback=None):
        self._vars = []
        self._osqp_vars = []
        self._quad_obj_exprs = []
        self._nonquad_obj_exprs = []
        self._lin_cnt_exprs = []      # (BoundExpr, "eq" | "leq")
        self._nonlin_cnt_exprs = []
        self._cnt_groups = OrderedDict()
        self._cnt_groups_overlap = OrderedDict()
        self.nonconverged_groups = []
        self._callback = callback if callback is not None else (lambda: None)
        self._stage = None            # device state of the step-by-step path

    # ------------------------------------------------------------------ building
    def add_var(self, var):
        if not any(v is var for v in self._vars):
            self._vars.append(var)
        self._stage = None

    def add_osqp_var(self, osqp_var):
        if not any(v is osqp_var for v in self._osqp_vars):
            self._osqp_vars.append(osqp_var)
        self._stage = None

    def add_obj_expr(self, bound_expr):
        if isinstance(bound_expr.expr, (E.AffExpr, E.QuadExpr)):
            self._quad_obj_exprs.append(bound_expr)
        else:
            self._nonquad_obj_exprs.append(bound_expr)
        self.add_var(bound_expr.var)

    def add_cnt_expr(self, bound_expr, group_ids=None):
        comp = bound_expr.expr
        assert isinstance(comp, E.CompExpr)
        if isinstance(comp, E.LExpr):
            raise NotImplementedError("LExpr constraints: the reference's OSQP backend silently ignores the "
                                      "affine ones and crashes on the nonlinear ones (prob.py:126-130,582-590)")
        if isinstance(comp.expr, E.AffExpr):
            self._lin_cnt_exprs.append((bound_expr, "eq" if isinstance(comp, E.EqExpr) else "leq"))
        else:
            self._nonlin_cnt_exprs.append(bound_expr)
            for gid in (group_ids if group_ids is not None else ["all"]):
                self._cnt_groups.setdefault(gid, []).append(bound_expr)
                for other in (group_ids or []):
                    if other != gid:
                        self._cnt_groups_overlap.setdefault(gid, set()).add(other)
        self.add_var(bound_expr.var)

    # ------------------------------------------------------------------ state
    def save(self):
        for var in self._vars:
            var.save()

    def restore(self):
        for var in self._vars:
            var.restore()

    def add_trust_region(self, trust_region_size):
        for var in self._vars:
            var.add_trust_region(trust_region_size)

    def _update_vars(self):
        for var in self._vars:
            var.update()

    # ------------------------------------------------------------------ device stages (batch of one)
    def _dev(self):
        if self._stage is None:
            from ..engine import Engine
            st, params, x0, cps = batch.compile_batch([self])
            self._stage = dict(st=st, params=params, cp=cps[0], eng=Engine(st), J=None, b=None, mask=None,
                               pi=1.0, kdup=0, wa=0.0)
        return self._stage

    def _x(self):
        s = self._dev()
        x = np.empty(s["st"].n)
        for var, k, j in s["cp"].slots:
            x[j] = var.get_value().ravel()[k]
        return x[None, :]

    def _settings(self, **osqp):
        from ..engine import make_settings
        return make_settings(osqp=osqp)

    def convexify(self):
        """Affine models of the nonlinear constraints at the current value (prob.py:522-544)."""
        s = self._dev()
        if s["st"].obj_prog_len or s["st"].obj_blocks:
            raise NotImplementedError("the step-by-step methods do not carry the degree-2 model of a non-quadratic "
                                      "objective between calls; use Solver.solve (one kernel does the whole SQP)")
        if s["st"].m_nl == 0:
            return
        f, J, b, _ = s["eng"].convexify(s["params"], self._x())
        s["J"], s["b"] = J, b
        if s["mask"] is None:  # prob.py:264,301: the row pattern is frozen at the first convexification
            Jn = J.cpu().numpy()[0]
            bits, e = [], 0
            for blk in s["st"].blocks:
                for _ in range(blk.m):
                    w = 0
                    for k in range(blk.jw):
                        if Jn[e + k] != 0.0:
                            w |= 1 << k
                    bits.append(w)
                    e += blk.jw
            s["mask"] = np.asarray(bits, dtype=np.uint32).view(np.int32)[None, :]

    def update_obj(self, penalty_coeff=0.0):
        """Rebuilds the penalty objective for `penalty_coeff` (prob.py:414-426)."""
        s = self._dev()
        # AffExpr objective terms are re-appended and every copy is scaled by the coefficient (quirk C-4,
        # prob.py:220-221,240-249,424-426)
        s["wa"] = (s["wa"] + 1.0) * penalty_coeff
        if s["st"].m_nl and s["J"] is not None:
            s["pi"] = s["pi"] * penalty_coeff   # prob.py:424-426: the stored weight is multiplied in place
            s["kdup"] += 1                      # prob.py:508-509: the penalty rows are appended again

    def _bounds(self):
        s = self._dev()
        lb = np.array([[float(ov.get_lower_bound()) for ov in s["cp"].ovars]])
        ub = np.array([[float(ov.get_upper_bound()) for ov in s["cp"].ovars]])
        return lb, ub

    def _deliver(self, xq):
        s = self._dev()
        batch.scatter_solution(s["cp"], xq[: s["st"].n])
        self._callback()

    def optimize(self, osqp_eps_abs=1e-6, osqp_eps_rel=1e-9, osqp_max_iter=int(1e5), rho=0.1,
                 adaptive_rho=False, sigma=5e-10, verbose=False):
        """One QP solve of the current convex model; True iff OSQP-status solved / solved inaccurate
        (prob.py:146-205)."""
        s = self._dev()
        lb, ub = self._bounds()
        pen = s["st"].m_nl > 0 and s["J"] is not None and s["kdup"] > 0
        kw = dict(J=s["J"], b=s["b"], mask=s["mask"], pi=np.array([s["pi"]]),
                  kdup=np.array([s["kdup"]], np.int32)) if pen else {}
        xq, status, _ = s["eng"].qp_solve(s["params"], self._settings(
            eps_abs=osqp_eps_abs, eps_rel=osqp_eps_rel, max_iter=osqp_max_iter, rho=rho,
            adaptive_rho=adaptive_rho, sigma=sigma), lbx=lb, ubx=ub, use_penalty=pen, wa=np.array([s["wa"]]), **kw)
        if int(status.cpu()[0]) not in (1, 2):
            return False
        self._deliver(xq.cpu().numpy()[0])
        return True

    def find_closest_feasible_point(self, **_ignored):
        """Projection of the current value on the linear constraints (prob.py:369-412; default OSQP
        settings whatever the caller passed, quirk C-7)."""
        s = self._dev()
        lb, ub = self._bounds()
        xq, status, _ = s["eng"].qp_solve(s["params"], self._settings(), lbx=lb, ubx=ub, xref=self._x(),
                                          use_penalty=False, closest_point=True)
        if int(status.cpu()[0]) not in (1, 2):
            return False
        self._deliver(xq.cpu().numpy()[0])
        return True

    def _merit(self, penalty_coeff, with_model):
        s = self._dev()
        J, b = (s["J"], s["b"]) if with_model else (None, None)
        return [t.cpu().numpy()[0] for t in
                s["eng"].merit(s["params"], self._x(), np.array([float(penalty_coeff)]), J=J, b=b)]

    def get_value(self, penalty_coeff, vectorize=False):
        """Exact penalty merit, or per-group violation sums (prob.py:547-580)."""
        merit, _, _, gv, _ = self._merit(penalty_coeff, False)
        return np.array(gv[: len(self._cnt_groups)]) if vectorize else float(merit)

    def get_approx_value(self, penalty_coeff, vectorize=False):
        """Merit of the convex model of the last convexification (prob.py:605-630)."""
        _, model, _, _, gm = self._merit(penalty_coeff, True)
        return np.array(gm[: len(self._cnt_groups)]) if vectorize else float(model)

    def get_max_cnt_violation(self):
        if not self._nonlin_cnt_exprs:
            return 0.0
        return float(self._merit(0.0, False)[2])
