"""Sizes beyond the first round's hard limits, same parity bars as tests/test_gpu_parity.py:
  * penalty rows wider than 32 stored Jacobian entries (a QCQP over 40 variables): the frozen-sparsity
    mask of quirk C-2 (prob.py:488-504) is ceil(width / 32) words per row;
  * a non-quadratic objective over 40 (stage level) and 20 (full solve) variables (Expr.convexify degree 2,
    expr.py:143-153: numerical Hessian, eigenvalue shift -- a warp-parallel Jacobi sweep on the device);
    up to 64 variables are accepted;
  * up to 16 constraint blocks per structure;
  * structures whose n x n system matrix exceeds one SM's shared memory (n = 240): S and its inverse live in
    global memory and are streamed by the ADMM loop.
"""
import numpy as np
import pytest

import helpers
import sqp_port
from sco_py_b200 import batch
from sco_py_b200 import sym
from sco_py_b200 import workloads as W
from sco_py_b200.expr import AffExpr, BoundExpr, LEqExpr, QuadExpr, QuadFormExpr, SymExpr
from sco_py_b200.sco_b200.osqp_utils import OSQPVar
from sco_py_b200.sco_b200.prob import Prob
from sco_py_b200.sco_b200.variable import Variable

WIDE_N, WIDE_M, WIDE_B = 40, 6, 6
CHAIN_STAGE_N, CHAIN_SOLVE_N = 40, 20


def build_chain(x0, analytic=False):
    """A Rosenbrock chain over len(x0) variables (indefinite Hessian away from the valley) inside a ball."""
    n = len(x0)
    X = sym.variables(n)
    f = sym.Sym.wrap(0.0)
    for i in range(n - 1):
        f = f + (X[i + 1] - X[i] ** 2) ** 2 + 0.1 * (1 - X[i]) ** 2
    ball = sym.Sym.wrap(-9.0)
    for i in range(n):
        ball = ball + X[i] ** 2
    prob = Prob()
    ov = np.array([[OSQPVar("x%02d" % i)] for i in range(n)], dtype=object)
    for v in ov[:, 0]:
        prob.add_osqp_var(v)
    var = Variable(ov, value=np.asarray(x0, dtype=float).reshape(n, 1))
    prob.add_var(var)
    prob.add_obj_expr(BoundExpr(QuadExpr(np.zeros((n, n)), np.zeros((1, n)), np.zeros((1, 1))), var))
    prob.add_obj_expr(BoundExpr(SymExpr([f], n, analytic=analytic), var))
    prob.add_cnt_expr(BoundExpr(LEqExpr(SymExpr([ball], n, analytic=analytic), np.zeros((1, 1))), var))
    return prob, var


def chain_points(k, n):
    rng = np.random.default_rng(5)
    return rng.uniform(-1.0, 1.0, (k, n))


def test_host_side_accepts_the_larger_sizes():
    st = W.qcqp_structure(n=WIDE_N, m=WIDE_M)
    assert st.blocks[0].jw == WIDE_N
    stc, params, x0, _ = batch.compile_batch([build_chain(p)[0] for p in chain_points(2, CHAIN_STAGE_N)])
    assert stc.n == CHAIN_STAGE_N and stc.obj_prog_len > 0
    with pytest.raises(batch.UnsupportedProblem):
        batch.compile_batch([build_chain(np.zeros(65))[0]])
    # sixteen constraint blocks in one structure
    prob = Prob()
    ov = np.array([[OSQPVar("a")], [OSQPVar("b")]], dtype=object)
    for v in ov[:, 0]:
        prob.add_osqp_var(v)
    var = Variable(ov, value=np.zeros((2, 1)))
    prob.add_var(var)
    prob.add_obj_expr(BoundExpr(QuadExpr(np.eye(2), np.zeros((1, 2)), np.zeros((1, 1))), var))
    for k in range(16):
        P = np.eye(2) * (1.0 + k)
        prob.add_cnt_expr(BoundExpr(LEqExpr(QuadFormExpr([P], np.zeros((1, 2))), np.full((1, 1), 4.0 + k)), var))
    st16, _, _, _ = batch.compile_batch([prob])
    assert len(st16.blocks) == 16
    prob.add_cnt_expr(BoundExpr(LEqExpr(QuadFormExpr([np.eye(2)], np.zeros((1, 2))), np.ones((1, 1))), var))
    with pytest.raises(batch.UnsupportedProblem):
        batch.compile_batch([prob])


@pytest.fixture(scope="module")
def wide():
    from sco_py_b200.engine import Engine
    st, params, x0 = W.gen_qcqp(WIDE_B, n=WIDE_N, m=WIDE_M)
    eng = Engine(st)
    assert eng.mask_words == 2
    yield eng, st, params, x0
    eng.close()


def _settings(**kw):
    from sco_py_b200.engine import make_settings
    return make_settings(solver=W.SOLVER_SETTINGS, **kw)


@pytest.mark.gpu
def test_wide_rows_convexify_and_masked_qp_stage(wide):
    eng, st, params, x0 = wide
    B = x0.shape[0]
    f, J, b, _ = eng.convexify(params, x0)
    Jn, bn = J.cpu().numpy(), b.cpu().numpy()
    for i in range(B):
        pp = sqp_port.PortProblem(st, params[i], x0[i])
        pp.convexify()
        np.testing.assert_allclose(helpers.split_J(st, Jn[i])[0], pp.J[0], rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(bn[i], pp.b[0][:, 0], rtol=1e-9, atol=1e-8)
    rng = np.random.default_rng(78)
    keep = rng.random((B, st.m_nl, 64)) > 1.0 / 3.0
    words = (keep.reshape(B, st.m_nl, 2, 32) * (1 << np.arange(32, dtype=np.uint64))).sum(axis=3).astype(np.uint32)
    lbx, ubx = x0 - 0.5, x0 + 0.5
    for mask in (None, words):
        xq, status, iters = eng.qp_solve(params, _settings(), J=J, b=b, lbx=lbx, ubx=ubx, pi=np.full(B, 10.0),
                                         kdup=np.full(B, 2, np.int32),
                                         mask=None if mask is None else mask.view(np.int32))
        xq, status, iters = xq.cpu().numpy(), status.cpu().numpy(), iters.cpu().numpy()
        for i in range(B):
            P, q, A, l, u = helpers.stage_qp(st, params[i], Jn[i], bn[i], lbx[i], ubx[i], 10.0, 2,
                                             bits=None if mask is None else mask[i])
            res = helpers.oracle_qp(P, q, A, l, u)
            assert status[i] == res.info.status_val and iters[i] == res.info.iter, (i, status[i], iters[i], res.info.iter)
            assert np.abs(xq[i] - res.x).max() <= 1e-7 * max(1.0, np.abs(res.x).max())


@pytest.mark.gpu
def test_wide_rows_full_solve_matches_port(wide):
    eng, st, params, x0 = wide
    out = eng.solve_batch(params, x0, _settings())
    x, verdict, vio = out["x"].cpu().numpy(), out["verdict"].cpu().numpy(), out["max_vio"].cpu().numpy()
    for i in range(x0.shape[0]):
        ref = sqp_port.solve(st, params[i], x0[i], solver=W.SOLVER_SETTINGS)
        assert (verdict[i] == 1) == ref["success"], (i, out["stats"][i].tolist(), ref["stats"])
        assert np.abs(x[i] - ref["x"]).max() <= 1e-4 * max(1.0, np.abs(ref["x"]).max())
        assert abs(vio[i] - ref["max_vio"]) <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("analytic", [False, True])
def test_objective_model_over_40_variables(analytic):
    from sco_py_b200.engine import Engine
    pts = chain_points(2, CHAIN_STAGE_N)
    st, params, x0, _ = batch.compile_batch([build_chain(p, analytic=analytic)[0] for p in pts])
    eng = Engine(st)
    H, g, c = [t.cpu().numpy() for t in eng.convexify_model(params, x0)]
    shifted = 0
    for i in range(len(pts)):
        pp = sqp_port.PortProblem(st, params[i], x0[i])
        pp.convexify()
        scale = max(1.0, np.abs(pp.Hq).max())
        assert np.abs(H[i] - pp.Hq).max() <= 1e-6 * scale, (i, np.abs(H[i] - pp.Hq).max())
        assert np.abs(g[i] - pp.aq).max() <= 1e-6 * max(1.0, np.abs(pp.aq).max())
        assert abs(c[i] - pp.bq) <= 1e-6 * max(1.0, abs(pp.bq))
        assert np.linalg.eigvalsh(H[i]).min() >= -1e-7 * scale
        shifted += int(np.linalg.eigvalsh(pp.Hq).min() < 1e-9 * scale)
    assert shifted > 0  # the shift was active somewhere
    eng.close()


@pytest.mark.gpu
def test_full_solve_with_an_objective_over_20_variables():
    from sco_py_b200.engine import Engine
    pts = chain_points(1, CHAIN_SOLVE_N)
    st, params, x0, _ = batch.compile_batch([build_chain(p, analytic=True)[0] for p in pts])
    eng = Engine(st)
    out = eng.solve_batch(params, x0, _settings())
    ref = sqp_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    assert (int(out["verdict"][0]) == 1) == ref["success"], (out["stats"][0].tolist(), ref["stats"])
    xr = ref["x"]
    assert np.abs(out["x"][0].cpu().numpy() - xr).max() <= 1e-4 * max(1.0, np.abs(xr).max())
    eng.close()


# ------------------------------------------------------------------ n beyond what one SM's shared memory holds
BIG_T = 120  # point robot over 120 time steps: n = 240, 360 penalty rows; S = P + sigma I + A'RA is 240 x 240 = 460 KB


@pytest.fixture(scope="module")
def big():
    from sco_py_b200.engine import Engine
    st, params, x0 = W.gen_point_robot(3, T=BIG_T)
    eng = Engine(st)
    yield eng, st, params, x0
    eng.close()


@pytest.mark.gpu
def test_large_structure_keeps_S_in_global_memory_qp_stage(big):
    """The n x n matrix of the reduced KKT system does not fit next to the rest of the working set: it lives in a
    per-team global workspace and the (strided) ADMM loop streams its inverse every iteration.  Same bars as the
    shared-memory path: identical status and iteration count, |dx| <= 1e-7."""
    eng, st, params, x0 = big
    assert st.n == 2 * BIG_T and 8 * st.n * st.n > 227 * 1024 > eng.smem_bytes
    B = 2
    f, J, b, _ = eng.convexify(params[:B], x0[:B])
    Jn, bn = J.cpu().numpy(), b.cpu().numpy()
    lbx, ubx = x0[:B] - 1.0, x0[:B] + 1.0
    xq, status, iters = eng.qp_solve(params[:B], _settings(), J=J, b=b, lbx=lbx, ubx=ubx, pi=np.full(B, 10.0),
                                     kdup=np.full(B, 1, np.int32))
    xq, status, iters = xq.cpu().numpy(), status.cpu().numpy(), iters.cpu().numpy()
    for i in range(B):
        P, q, A, l, u = helpers.stage_qp(st, params[i], Jn[i], bn[i], lbx[i], ubx[i], 10.0, 1)
        res = helpers.oracle_qp(P, q, A, l, u)
        assert status[i] == res.info.status_val and iters[i] == res.info.iter, (i, status[i], iters[i], res.info.iter)
        assert np.abs(xq[i] - res.x).max() <= 1e-7 * max(1.0, np.abs(res.x).max())


@pytest.mark.gpu
def test_large_structure_full_solve_matches_port(big):
    eng, st, params, x0 = big
    out = eng.solve_batch(params, x0, _settings())
    x, verdict, vio = out["x"].cpu().numpy(), out["verdict"].cpu().numpy(), out["max_vio"].cpu().numpy()
    for i in range(x0.shape[0]):
        ref = sqp_port.solve(st, params[i], x0[i], solver=W.SOLVER_SETTINGS)
        assert (verdict[i] == 1) == ref["success"], (i, out["stats"][i].tolist(), ref["stats"])
        assert np.abs(x[i] - ref["x"]).max() <= 1e-4 * max(1.0, np.abs(ref["x"]).max())
        assert abs(vio[i] - ref["max_vio"]) <= 1e-5
