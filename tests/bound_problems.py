"""API problems whose nonlinear constraints are bound to Variables of a few scalar variables (BoundExpr(expr, var)
with `var` a step of a trajectory or a subset of the unknowns), each also written "lifted": the same constraint as a
function of all n variables in QP order (zero-padded P / a, PUSH_X re-indexed, the FK7 joints placed last).  The
two forms are the same optimisation problem with the same penalty rows in the same order."""
import numpy as np

from sco_py_b200 import expr as E
from sco_py_b200 import sym
from sco_py_b200 import workloads as W
from sco_py_b200.sco_b200.osqp_utils import OSQPVar
from sco_py_b200.sco_b200.prob import Prob
from sco_py_b200.sco_b200.variable import Variable

FORMS = ("bound", "lifted")


def _scalars(names):
    ov = np.empty((len(names), 1), dtype=object)
    for j, nm in enumerate(names):
        ov[j, 0] = OSQPVar(nm)
    return ov


def _start(ov, x0):
    prob = Prob()
    for v in ov[:, 0]:
        prob.add_osqp_var(v)
    allv = Variable(ov, np.asarray(x0, dtype=float).reshape(-1, 1))
    prob.add_var(allv)
    return prob, allv


def _sub(ov, x0, idx):
    idx = np.asarray(idx)
    return Variable(ov[idx], np.asarray(x0, dtype=float).reshape(-1, 1)[idx])


def robot(i, T=8, K=2, form="bound", analytic=False, groups=None):
    """Point robot (workloads.gen_point_robot's numbers): obstacle rows R_k - |p_t - c_k| <= 0 as SymExprs, one per
    step bound to that step's Variable, or lifted: one SymExpr over all 2T variables.  groups(t): the group ids of
    step t's constraint (bound form)."""
    st, params, x0 = W.gen_point_robot(1, T=T, K=K, first=i)
    row, x0 = params[0], x0[0]
    n = 2 * T
    ov = _scalars(["p%03d%s" % (t, "xy"[d]) for t in range(T) for d in range(2)])
    prob, allv = _start(ov, x0)
    Q = np.asarray(st.shared[:n * n]).reshape(n, n)
    prob.add_obj_expr(E.BoundExpr(E.QuadExpr(Q, np.zeros((1, n)), np.zeros((1, 1))), allv))
    A = np.zeros((4, n))
    A[0, 0] = A[1, 1] = A[2, n - 2] = A[3, n - 1] = 1.0
    pin = np.asarray(st.get(st.lin_u, row, 4)).reshape(4, 1)
    prob.add_cnt_expr(E.BoundExpr(E.EqExpr(E.AffExpr(A, np.zeros((4, 1))), pin), allv))
    par = np.asarray(st.get(st.blocks[0].par, row, 3 * K))
    cen, rad = par[:2 * K].reshape(K, 2), par[2 * K:]

    def rows(x, a, b):
        return [rad[k] - sym.sqrt((x[a] - cen[k, 0]) ** 2 + (x[b] - cen[k, 1]) ** 2) for k in range(K)]

    if form == "bound":
        for t in range(T):
            x = sym.variables(2)
            e = E.SymExpr(rows(x, 0, 1), 2, analytic=analytic)
            prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(e, np.zeros((K, 1))), _sub(ov, x0, [2 * t, 2 * t + 1])),
                              group_ids=None if groups is None else groups(t))
    else:
        x = sym.variables(n)
        e = E.SymExpr([r for t in range(T) for r in rows(x, 2 * t, 2 * t + 1)], n, analytic=analytic)
        prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(e, np.zeros((T * K, 1))), allv))
    return prob


def qcqp(i, n=8, m=6, k=3, form="bound", sel_seed=None):
    """QCQP (workloads.gen_qcqp's numbers) whose row j reads only k of the n variables, in a permuted order: one
    QuadFormExpr per row bound to a Variable of those k, or lifted: one QuadFormExpr with zero-padded P / a.  The
    variables of each row are drawn from sel_seed (default: per problem); problems of one sel_seed share a structure."""
    st, params, x0 = W.gen_qcqp(1, n=n, m=m, first=i)
    row, x0 = params[0], x0[0]
    ntri = n * (n + 1) // 2
    par = np.asarray(st.get(st.blocks[0].par, row, m * ntri + m * n))
    iu = np.triu_indices(n)
    P = np.zeros((m, n, n))
    for j in range(m):
        P[j][iu] = par[j * ntri:(j + 1) * ntri]
        P[j] = P[j] + P[j].T - np.diag(np.diag(P[j]))
    a = par[m * ntri:].reshape(m, n)
    val = np.asarray(st.get(st.blocks[0].val, row, m)).reshape(m, 1)
    ov = _scalars(["x%05d" % j for j in range(n)])
    prob, allv = _start(ov, x0)
    Q = np.asarray(st.get(st.Q, row, n * n)).reshape(n, n)
    prob.add_obj_expr(E.BoundExpr(E.QuadExpr(Q, np.asarray(st.get(st.q, row, n)).reshape(1, n), np.zeros((1, 1))), allv))
    rng = np.random.default_rng(77 + i if sel_seed is None else sel_seed)
    sel = [rng.choice(n, k, replace=False) for _ in range(m)]
    if form == "bound":
        for j in range(m):
            c = sel[j]
            e = E.QuadFormExpr(P[j][np.ix_(c, c)][None], a[j, c][None])
            prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(e, val[j:j + 1]), _sub(ov, x0, c)))
    else:
        Pl, al = np.zeros((m, n, n)), np.zeros((m, n))
        for j in range(m):
            c = sel[j]
            Pl[j][np.ix_(c, c)] = P[j][np.ix_(c, c)]
            al[j, c] = a[j, c]
        prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(E.QuadFormExpr(Pl, al), val), allv))
    return prob


def circle(i, T=6, K=2, form="bound"):
    """Point robot with its CircleDistExpr obstacles: one CircleDistExpr(1) per step bound to that step's Variable
    (one block per step: CIRCLE2D constraints are never packed), or lifted: one CircleDistExpr(T) on all variables."""
    st, params, x0 = W.gen_point_robot(1, T=T, K=K, first=i)
    row, x0 = params[0], x0[0]
    n = 2 * T
    ov = _scalars(["p%03d%s" % (t, "xy"[d]) for t in range(T) for d in range(2)])
    prob, allv = _start(ov, x0)
    Q = np.asarray(st.shared[:n * n]).reshape(n, n)
    prob.add_obj_expr(E.BoundExpr(E.QuadExpr(Q, np.zeros((1, n)), np.zeros((1, 1))), allv))
    A = np.zeros((4, n))
    A[0, 0] = A[1, 1] = A[2, n - 2] = A[3, n - 1] = 1.0
    pin = np.asarray(st.get(st.lin_u, row, 4)).reshape(4, 1)
    prob.add_cnt_expr(E.BoundExpr(E.EqExpr(E.AffExpr(A, np.zeros((4, 1))), pin), allv))
    par = np.asarray(st.get(st.blocks[0].par, row, 3 * K))
    cen, rad = par[:2 * K].reshape(K, 2), par[2 * K:]
    if form == "bound":
        for t in range(T):
            e = E.CircleDistExpr(1, cen, rad)
            prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(e, np.zeros((K, 1))), _sub(ov, x0, [2 * t, 2 * t + 1])))
    else:
        prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(E.CircleDistExpr(T, cen, rad), np.zeros((T * K, 1))), allv))
    return prob


def arm(i, T=3, form="bound", per_step=False):
    """7-DOF arm (workloads.gen_arm's numbers): flange == target at the last step, FK7Expr(7) bound to that step's
    Variable, or lifted: FK7Expr(n) on all variables (the last step's joints are the last seven).  per_step=True
    (bound form only) adds an FK7 instance per intermediate step: flange <= target + 0.1 there."""
    st, params, x0 = W.gen_arm(1, T=T, first=i)
    row, x0 = params[0], x0[0]
    n = 7 * T
    ov = _scalars(["q%03d_%d" % (t, j) for t in range(T) for j in range(7)])
    prob, allv = _start(ov, x0)
    Q = np.asarray(st.shared[:n * n]).reshape(n, n)
    prob.add_obj_expr(E.BoundExpr(E.QuadExpr(Q, np.zeros((1, n)), np.zeros((1, 1))), allv))
    lo = np.asarray(st.get(st.lin_l, row, st.m_lin))
    hi = np.asarray(st.get(st.lin_u, row, st.m_lin))
    lim = np.full((2 * n, 1), W.JOINT_LIMIT)
    prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(E.AffExpr(np.vstack([np.eye(n), -np.eye(n)]), np.zeros((2 * n, 1))), lim), allv))
    prob.add_cnt_expr(E.BoundExpr(E.EqExpr(E.AffExpr(np.eye(7, n), np.zeros((7, 1))), hi[2 * n:].reshape(7, 1)), allv))
    assert np.array_equal(lo[2 * n:], hi[2 * n:])
    target = np.asarray(st.get(st.blocks[0].val, row, 3)).reshape(3, 1)
    if per_step:
        assert form == "bound"
        for t in range(1, T - 1):
            step = _sub(ov, x0, np.arange(7 * t, 7 * t + 7))
            prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(E.FK7Expr(7), target + 0.1), step))
    if form == "bound":
        prob.add_cnt_expr(E.BoundExpr(E.EqExpr(E.FK7Expr(7), target), _sub(ov, x0, np.arange(n - 7, n))))
    else:
        prob.add_cnt_expr(E.BoundExpr(E.EqExpr(E.FK7Expr(n), target), allv))
    return prob


BUILDERS = {"vm": robot, "quadform": qcqp, "circle2d": circle, "fk7": arm}
