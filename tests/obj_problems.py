"""API problems with non-quadratic objective terms bound to Variables (BoundExpr(SymExpr, var), one term per call of
Prob.add_obj_expr, as a per-step cost is written in the reference), each also writable "lifted": every term a
function of all n variables in QP order (PUSH_X re-indexed), still its own term -- the same optimisation problem
with the same per-term convexification.  "summed": one term, the sum of all, over all variables (the structure of
earlier versions; a different QP by design, since the eigenvalue shift of a sum is not the sum of the shifts)."""
import numpy as np

import bound_problems as BP
from sco_py_b200 import expr as E
from sco_py_b200 import sym


def remap(e, idx):
    """The expression with input j replaced by input idx[j]."""
    if e.op == sym.PUSH_X:
        return sym.Sym(sym.PUSH_X, value=float(idx[int(e.value)]))
    return sym.Sym(e.op, tuple(remap(a, idx) for a in e.args), e.value)


def add_terms(prob, ov, x0, terms, form="bound", analytic=False):
    """terms: [(f over local inputs 0..k-1, QP columns of those inputs)]."""
    n = ov.shape[0]
    if form == "summed":
        tot = sym.Sym.wrap(0.0)
        for f, cols in terms:
            tot = tot + remap(f, list(cols))
        prob.add_obj_expr(E.BoundExpr(E.SymExpr([tot], n, analytic=analytic), BP._sub(ov, x0, np.arange(n))))
        return prob
    for f, cols in terms:
        if form == "bound":
            prob.add_obj_expr(E.BoundExpr(E.SymExpr([f], len(cols), analytic=analytic), BP._sub(ov, x0, cols)))
        else:
            prob.add_obj_expr(E.BoundExpr(E.SymExpr([remap(f, list(cols))], n, analytic=analytic),
                                          BP._sub(ov, x0, np.arange(n))))
    return prob


def soft_obstacle(c=(0.3, -0.2), w=0.5):
    """w exp(-|p - c|^2): indefinite Hessian near the centre."""
    x = sym.variables(2)
    return w * sym.exp(-((x[0] - c[0]) ** 2 + (x[1] - c[1]) ** 2))


def convex_cost(c=(0.3, -0.2), w=0.5):
    """w sqrt(1 + |p - c|^2): convex with bounded curvature, so a term lifted to all variables gets the same (zero)
    shift as the bound one."""
    x = sym.variables(2)
    return w * sym.sqrt(1.0 + (x[0] - c[0]) ** 2 + (x[1] - c[1]) ** 2)


def pair_cost(w=0.05):
    """w (|p_{t+1} - p_t|^2 - 0.1)^2 over the four coordinates of two consecutive steps."""
    x = sym.variables(4)
    return w * ((x[2] - x[0]) ** 2 + (x[3] - x[1]) ** 2 - 0.1) ** 2


def robot(i, T=12, K=2, form="bound", cost="step", analytic=False, groups=None):
    """bound_problems.robot (obstacle rows as bound SymExpr constraints) with per-step soft-obstacle costs
    (cost="step", n_in = 2), convex per-step costs (cost="convex") or pairwise costs over consecutive steps
    (cost="pair", n_in = 4)."""
    prob = BP.robot(i, T=T, K=K, form="bound", analytic=analytic, groups=groups)
    ov = np.array([[v] for v in sorted(prob._osqp_vars, key=lambda v: v.var_name)], dtype=object)
    x0 = prob._vars[0].get_value().ravel()  # the Variable of all scalar variables (bound_problems._start)
    rng = np.random.default_rng(100 + i)
    if cost == "step":
        terms = [(soft_obstacle(c=tuple(rng.uniform(-0.5, 0.5, 2))), np.array([2 * t, 2 * t + 1])) for t in range(T)]
    elif cost == "convex":
        terms = [(convex_cost(c=tuple(rng.uniform(-0.5, 0.5, 2))), np.array([2 * t, 2 * t + 1])) for t in range(T)]
    else:
        terms = [(pair_cost(), np.arange(2 * t, 2 * t + 4)) for t in range(T - 1)]
    return add_terms(prob, ov, x0, terms, form=form, analytic=analytic)
