"""BASELINE.json configs[0]: the toy non-convex problems of the reference's own solver test
(tests/sco_osqp/test_solver.py:91-169, hyper-parameters :15-25, pass mark atol 5e-4 on the optimum :87).

All nine are assembled exactly as helper_test_prob (:32-87) does: one quadratic objective, one
black-box objective term f, one linear LEq row block, one nonlinear LEq block g, one nonlinear Eq
block h, absent pieces being the reference's placeholders (f = 0, g = -1e5, h = 0).
  * "quadform" variants (prob0, 2, 3, 5, 6): f folded into the QuadExpr, g / h as QuadFormExpr
    (a linear g is a quadratic form with P = 0) -- the closed-family path.
  * "sym" variants (all nine): f, g, h written in the expression language of sco_py_b200.sym, i.e. black
    boxes without analytic derivatives like the reference's lambdas: finite-difference Jacobians, and
    for f the finite-difference Hessian + eigenvalue shift of Expr.convexify degree 2 (expr.py:143-153).
"""
import numpy as np
import pytest

import sqp_port
from sco_py_b200 import batch
from sco_py_b200 import workloads as W
import ref_builder
from sco_py_b200 import sym
from sco_py_b200.expr import AffExpr, BoundExpr, EqExpr, LEqExpr, QuadExpr, QuadFormExpr, SymExpr
from sco_py_b200.sco_b200.osqp_utils import OSQPVar
from sco_py_b200.sco_b200.prob import Prob
from sco_py_b200.sco_b200.solver import Solver
from sco_py_b200.sco_b200.variable import Variable

N = 2
ANG = (np.arange(1, 7) * 2 * np.pi / 6).reshape(6, 1)
HEX_A = np.hstack((np.cos(ANG), np.sin(ANG)))
HEX_q = -np.array([[np.cos(np.pi / 6), np.sin(np.pi / 6)]])


def quadform(rows):
    """rows: list of (P 2x2, a 2, const) -> (QuadFormExpr, val) with f_j = 0.5 x'P_j x + a_j'x <= / == -const."""
    P = np.array([r[0] for r in rows], dtype=float)
    a = np.array([r[1] for r in rows], dtype=float)
    val = -np.array([[r[2]] for r in rows], dtype=float)
    return QuadFormExpr(P, a), val


Z = np.zeros((2, 2))
PROBLEMS = {
    # name: (x0, x_true, Q, q, c, A_ineq, b_ineq, g rows, h rows)
    "prob0": ([1.0, 1.0], [1.5, 1.5], 2 * np.eye(2), np.zeros((1, 2)), 0.0, None, None,
              [(Z, [-1.0, -1.0], 3.0)], None),                                   # g = 3 - x1 - x2
    "prob2": ([10.0, 1.0], [0.0, 0.0], 2 * np.array([[1.0, -1.0], [-1.0, 1.0]]), np.array([[0.0, 1.0]]), 1e-5,
              None, None, [(Z, [0.0, -1.0], 0.0)], None),                        # f = x2 + 1e-5 + (x2-x1)^2 ; g = -x2
    "prob3": ([10.0, 1.0], [1.0, 1.0], 2 * np.diag([1.0, 0.0]), np.array([[-2.0, 0.0]]), 1.0, None, None, None,
              [(np.array([[-20.0, 0.0], [0.0, 0.0]]), [0.0, 10.0], 0.0)]),       # h = 10 (x2 - x1^2)
    "prob5": ([0.0, 0.0], [1.0, np.tan(np.pi / 6)], Z, HEX_q, 0.0, HEX_A, np.ones((6, 1)), None, None),
    "prob6": ([0.0, 0.0], [1.0, np.tan(np.pi / 6)], 0.1 * np.eye(2), HEX_q, 0.0, None, None,
              [(Z, 0.01 * HEX_A[k], -0.01) for k in range(6)], None),            # g = 0.01 (A x - 1)
}


def build(name, x0=None):
    x0_, x_true, Q, q, c, A_ineq, b_ineq, g, h = PROBLEMS[name]
    x0 = np.array(x0_ if x0 is None else x0, dtype=float).reshape(2, 1)
    prob = Prob()
    ov = np.array([[OSQPVar("x1")], [OSQPVar("x2")]], dtype=object)
    for v in ov[:, 0]:
        prob.add_osqp_var(v)
    var = Variable(ov, value=x0)
    prob.add_var(var)
    prob.add_obj_expr(BoundExpr(QuadExpr(Q, q, np.array([[c]])), var))
    if A_ineq is None:
        A_ineq, b_ineq = np.zeros((1, N)), np.zeros((1, 1))
    prob.add_cnt_expr(BoundExpr(LEqExpr(AffExpr(A_ineq, -b_ineq), np.zeros(b_ineq.shape)), var))
    ge, gval = quadform(g if g is not None else [(Z, [0.0, 0.0], -1e5)])       # neginffunc
    prob.add_cnt_expr(BoundExpr(LEqExpr(ge, gval), var))
    he, hval = quadform(h if h is not None else [(Z, [0.0, 0.0], 0.0)])        # zerofunc
    prob.add_cnt_expr(BoundExpr(EqExpr(he, hval), var))
    return prob, var, np.array(x_true)


def _solver():
    s = Solver()
    for k, v in W.SOLVER_SETTINGS.items():
        setattr(s, k, v)
    return s


@pytest.mark.parametrize("name", sorted(PROBLEMS))
def test_oracle_reaches_the_reference_answers(name):
    """The modelling above is the reference's problem: the oracle port lands on x_true at atol 5e-4."""
    prob, var, x_true = build(name)
    st, params, x0, _ = batch.compile_batch([prob])
    r = sqp_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    assert np.allclose(r["x"], x_true, atol=5e-4), (name, r["x"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(PROBLEMS))
def test_device_reaches_the_reference_answers(name):
    prob, var, x_true = build(name)
    _solver().solve(prob, method="penalty_sqp")
    assert np.allclose(var.get_value()[:, 0], x_true, atol=5e-4), (name, var.get_value()[:, 0])


@pytest.mark.gpu
def test_jittered_batch_of_toy_problems():
    """SURVEY.md C1: B copies with x0 jittered by N(0, 0.1^2), seed 1 -- one launch, same optimum."""
    rng = np.random.default_rng(1)
    for name in ("prob0", "prob3"):
        built = [build(name, x0=np.array(PROBLEMS[name][0]) + rng.normal(0.0, 0.1, 2)) for _ in range(16)]
        _solver().solve_batch([b[0] for b in built], method="penalty_sqp")
        for prob, var, x_true in built:
            assert np.allclose(var.get_value()[:, 0], x_true, atol=5e-4), (name, var.get_value()[:, 0])


# ------------------------------------------------------------------ all nine, as black boxes (sym)
X = sym.variables(2)
x1, x2 = X
HEXROWS = [0.01 * (float(HEX_A[k, 0]) * x1 + float(HEX_A[k, 1]) * x2 - 1.0) for k in range(6)]
SYM_PROBLEMS = {
    # name: (x0, x_true, Q, q, A_ineq, b_ineq, f, g rows, h rows)       tests/sco_osqp/test_solver.py:91-169
    "prob0": ([1.0, 1.0], [1.5, 1.5], Z, np.zeros((1, 2)), None, None, x1 ** 2 + x2 ** 2, [3 - x1 - x2], None),
    "prob1": ([-2.0, 1.0], [1.0, 1.0], Z, np.zeros((1, 2)), None, None, (x2 - x1 ** 2) ** 2 + (1 - x1) ** 2,
              [-1.5 - x2], None),
    "prob2": ([10.0, 1.0], [0.0, 0.0], Z, np.zeros((1, 2)), None, None, x2 + 1e-5 + (x2 - x1) ** 2, [-x2], None),
    "prob3": ([10.0, 1.0], [1.0, 1.0], Z, np.zeros((1, 2)), None, None, (1 - x1) ** 2, None, [10 * (x2 - x1 ** 2)]),
    "prob4": ([2.0, 2.0], [0.0, np.sqrt(3)], Z, np.zeros((1, 2)), None, None, sym.log(1 + x1 ** 2) - x2, None,
              [(1 + x1 ** 2) ** 2 + x2 ** 2 - 4]),
    "prob5": ([0.0, 0.0], [1.0, np.tan(np.pi / 6)], Z, HEX_q, HEX_A, np.ones((6, 1)), None, None, None),
    "prob6": ([0.0, 0.0], [1.0, np.tan(np.pi / 6)], 0.1 * np.eye(2), HEX_q, None, None, None, HEXROWS, None),
    "prob7": ([0.0, 0.0], [2.0, 1.0], Z, np.zeros((1, 2)), None, None, x1 ** 4 + x2 ** 4, [3 - x1 - x2], [x1 - 2 * x2]),
    "prob8": ([5.0, 5.0], [0.0, 0.0], np.eye(2), np.zeros((1, 2)), None, None, None,
              [x1 ** 2 + x2 ** 2 - 4, -((x1 - 1) ** 2 + (x2 - 1) ** 2 - 0.25), -((x1 + 1) ** 2 + (x2 - 1) ** 2 - 0.25),
               -(x1 ** 2 + 7 * (x2 + 1 - x1 ** 2 / 2) ** 2 - 0.8)], None),
}


def build_sym(name, x0=None, analytic=False):
    """analytic=True: the functions come with their exact derivatives (Expr(f, grad), expr.py:86-88) instead of being
    finite-differenced (the objective keeps its numerical Hessian, expr.py:102-109)."""
    x0_, x_true, Q, q, A_ineq, b_ineq, f, g, h = SYM_PROBLEMS[name]
    x0 = np.array(x0_ if x0 is None else x0, dtype=float).reshape(2, 1)
    prob = Prob()
    ov = np.array([[OSQPVar("x1")], [OSQPVar("x2")]], dtype=object)
    for v in ov[:, 0]:
        prob.add_osqp_var(v)
    var = Variable(ov, value=x0)
    prob.add_var(var)
    prob.add_obj_expr(BoundExpr(QuadExpr(Q, q, np.zeros((1, 1))), var))
    prob.add_obj_expr(BoundExpr(SymExpr([f if f is not None else sym.Sym.wrap(0.0)], 2, analytic=analytic), var))    # zerofunc
    if A_ineq is None:
        A_ineq, b_ineq = np.zeros((1, N)), np.zeros((1, 1))
    prob.add_cnt_expr(BoundExpr(LEqExpr(AffExpr(A_ineq, -b_ineq), np.zeros(b_ineq.shape)), var))
    g = g if g is not None else [sym.Sym.wrap(-1e5)]                                               # neginffunc
    prob.add_cnt_expr(BoundExpr(LEqExpr(SymExpr(g, 2, analytic=analytic), np.zeros((len(g), 1))), var))
    h = h if h is not None else [sym.Sym.wrap(0.0)]                                                # zerofunc
    prob.add_cnt_expr(BoundExpr(EqExpr(SymExpr(h, 2, analytic=analytic), np.zeros((len(h), 1))), var))
    return prob, var, np.array(x_true)


@pytest.mark.parametrize("name", sorted(SYM_PROBLEMS))
def test_oracle_reaches_the_reference_answers_sym(name):
    prob, var, x_true = build_sym(name)
    st, params, x0, _ = batch.compile_batch([prob])
    r = sqp_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    assert np.allclose(r["x"], x_true, atol=5e-4), (name, r["x"])


@pytest.mark.skipif(not ref_builder.reference_available(), reason="needs an upstream sco_py checkout at SCO_REFERENCE_ROOT")
@pytest.mark.parametrize("name", ["prob1", "prob4", "prob7", "prob8"])
def test_port_equals_the_unmodified_reference_on_black_box_objectives(name):
    """The unmodified reference (Solver.solve on the shims) on the same functions as Python callables."""
    prob, var, x_true = build_sym(name)
    st, params, x0, _ = batch.compile_batch([prob])
    a = sqp_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    b = ref_builder.solve_with_reference(ref_builder.import_reference(), st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    assert a["success"] == b["success"]
    assert np.abs(a["x"] - b["x"]).max() <= 1e-7, (a["x"], b["x"])
    assert np.allclose(b["x"], x_true, atol=5e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SYM_PROBLEMS))
def test_device_reaches_the_reference_answers_sym(name):
    prob, var, x_true = build_sym(name)
    st, params, x0, _ = batch.compile_batch([prob])
    ref = sqp_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    ok = _solver().solve(prob, method="penalty_sqp")
    assert ok == ref["success"], name
    assert np.allclose(var.get_value()[:, 0], x_true, atol=5e-4), (name, var.get_value()[:, 0])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["prob4", "prob8"])
def test_vm_family_values_and_fd_jacobians_match_the_oracle(name):
    """Stage level: the stack-program family on the device (values, finite-difference Jacobian, affine
    offsets) against the oracle's interpreter + numdifftools shim."""
    from sco_py_b200.engine import Engine
    prob, var, _ = build_sym(name)
    st, params, x0, _ = batch.compile_batch([prob])
    eng = Engine(st)
    f, J, b, obj = [t.cpu().numpy()[0] for t in eng.convexify(params, x0)]
    pp = sqp_port.PortProblem(st, params[0], x0[0])
    pp.convexify()
    r0 = e0 = 0
    for bi, blk in enumerate(st.blocks):
        np.testing.assert_allclose(f[r0:r0 + blk.m], pp.blocks[bi].f(pp.x)[:, 0], rtol=1e-13, atol=1e-13)
        np.testing.assert_allclose(J[e0:e0 + blk.m * blk.jw].reshape(blk.m, blk.jw), pp.J[bi], rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(b[r0:r0 + blk.m], pp.b[bi][:, 0], rtol=1e-9, atol=1e-8)
        r0 += blk.m
        e0 += blk.m * blk.jw
    assert abs(obj - pp.objective(pp.x)) <= 1e-12 * max(1.0, abs(obj))
    eng.close()


# ------------------------------------------------------------------ analytic derivatives (Expr(f, grad)) and the Hessian stage
@pytest.mark.skipif(not ref_builder.reference_available(), reason="needs an upstream sco_py checkout at SCO_REFERENCE_ROOT")
@pytest.mark.parametrize("name", ["prob1", "prob4", "prob7", "prob8"])
def test_port_equals_the_unmodified_reference_with_analytic_gradients(name):
    """The same functions handed to the unmodified reference as Expr(f, grad) with exact gradients."""
    prob, var, x_true = build_sym(name, analytic=True)
    st, params, x0, _ = batch.compile_batch([prob])
    assert st.obj_prog_flags == 1 and all(b.ipar[3] == 1 for b in st.blocks)
    a = sqp_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    b = ref_builder.solve_with_reference(ref_builder.import_reference(), st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    assert a["success"] == b["success"]
    assert np.abs(a["x"] - b["x"]).max() <= 1e-7, (a["x"], b["x"])
    assert np.allclose(b["x"], x_true, atol=5e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SYM_PROBLEMS))
def test_device_reaches_the_reference_answers_with_analytic_gradients(name):
    prob, var, x_true = build_sym(name, analytic=True)
    st, params, x0, _ = batch.compile_batch([prob])
    ref = sqp_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    ok = _solver().solve(prob, method="penalty_sqp")
    assert ok == ref["success"], name
    assert np.allclose(var.get_value()[:, 0], x_true, atol=5e-4), (name, var.get_value()[:, 0])
    assert np.abs(var.get_value()[:, 0] - ref["x"]).max() <= 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["prob1", "prob4", "prob7"])
@pytest.mark.parametrize("analytic", [False, True])
def test_objective_model_stage_matches_the_oracle(name, analytic):
    """Stage level (SURVEY.md row a3): numerical Hessian (central second differences, Richardson), smallest eigenvalue
    by Jacobi sweeps, shift H - min(lambda, 0) I, A = grad - x'H, b = 0.5 x'Hx - grad.x + f on the device against the
    oracle's Expr.hess / Expr.convexify(degree=2) restatement (expr.py:102-128,143-153), at points where the Hessian is
    indefinite (the shift is active) and where it is not."""
    from sco_py_b200.engine import Engine
    rng = np.random.default_rng(11)
    pts = np.vstack([np.array(SYM_PROBLEMS[name][0]), rng.uniform(-2.0, 2.0, (7, 2))])
    probs = [build_sym(name, x0=p, analytic=analytic)[0] for p in pts]
    st, params, x0, _ = batch.compile_batch(probs)
    eng = Engine(st)
    H, g, c = [t.cpu().numpy() for t in eng.convexify_model(params, x0)]
    shifted = 0
    for i in range(len(pts)):
        pp = sqp_port.PortProblem(st, params[i], x0[i])
        pp.convexify()
        scale = max(1.0, np.abs(pp.Hq).max())
        assert np.abs(H[i] - pp.Hq).max() <= 1e-6 * scale, (name, i, H[i], pp.Hq)
        assert np.abs(g[i] - pp.aq).max() <= 1e-6 * max(1.0, np.abs(pp.aq).max()), (name, i)
        assert abs(c[i] - pp.bq) <= 1e-6 * max(1.0, abs(pp.bq)), (name, i)
        assert np.linalg.eigvalsh(H[i]).min() >= -1e-7 * scale  # convex after the shift
        shifted += int(np.linalg.eigvalsh(pp.Hq).min() < 1e-9 * scale)
    eng.close()
