"""CPU tests of the oracle (test infrastructure): pinned on the reference's own test-suite, on the
unmodified reference run on the shims, and on the committed golden vectors."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import helpers
import ref_builder
import sqp_port
from sco_py_b200 import workloads as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
needs_reference = pytest.mark.skipif(not ref_builder.reference_available(),
                                     reason="needs an upstream sco_py checkout at SCO_REFERENCE_ROOT")


@needs_reference
def test_reference_suite_passes_on_the_oracle_shims():
    """tests/sco_osqp/*.py of the reference, unmodified, with oracle/shims standing in for the two
    absent third-party modules: every known-answer QP / merit / SQP test the reference holds
    (SURVEY.md section 8c) pins oracle/osqp_core.c and the numdifftools shim."""
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "oracle", "shims"), ref_builder.REFERENCE_ROOT])
    p = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider",
                        os.path.join(ref_builder.REFERENCE_ROOT, "tests", "sco_osqp")],
                       env=env, capture_output=True, text=True, cwd="/tmp")
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-2000:]
    assert "54 passed" in p.stdout, p.stdout[-500:]


@pytest.mark.parametrize("name,idx", [("qcqp", i) for i in range(6)] + [("point_robot", i) for i in range(4)]
                         + [("arm", i) for i in range(4)])
def test_port_matches_the_unmodified_reference(name, idx):
    """Against what the unmodified reference returned for the same problem, every problem stored in
    tests/golden/ref_<config>.npz (written by oracle/gen_golden.py)."""
    g = np.load(os.path.join(GOLDEN, "ref_%s.npz" % name))
    st, params, x0 = W.GENERATORS[name](1, first=idx)
    a = sqp_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    assert a["success"] == bool(g["success"][idx])
    assert np.abs(a["x"] - g["x"][idx]).max() <= 1e-8
    assert abs(a["max_vio"] - g["max_vio"][idx]) <= 1e-9


@pytest.mark.parametrize("name,indices", [("qcqp", [3, 5]), ("point_robot", [1, 2, 3]), ("arm", [2, 3])])
def test_port_matches_golden_reference_solutions(name, indices):
    g = np.load(os.path.join(GOLDEN, "ref_%s.npz" % name))
    for idx in indices:
        st, params, x0 = W.GENERATORS[name](1, first=idx)
        r = sqp_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
        assert r["success"] == bool(g["success"][idx])
        assert np.abs(r["x"] - g["x"][idx]).max() <= 1e-8, (name, idx)
        assert abs(r["max_vio"] - g["max_vio"][idx]) <= 1e-9


@pytest.mark.parametrize("name", ["qcqp", "point_robot", "arm"])
def test_osqp_core_reproduces_golden_qps(name):
    """(P, q, A, l, u) captured at the reference's osqp.OSQP().setup call site (osqp_utils.py:195-214)
    -> x, status, iterations."""
    g = np.load(os.path.join(GOLDEN, "ref_%s.npz" % name))
    for k in range(len(g["qp_index"])):
        mats = {}
        for key in ("A", "P"):
            mats[key] = sp.csr_matrix((g["qp%d_%s_data" % (k, key)], g["qp%d_%s_indices" % (k, key)],
                                       g["qp%d_%s_indptr" % (k, key)]), shape=tuple(g["qp%d_%s_shape" % (k, key)]))
        rho, sigma, ea, er, mi, ar = g["qp%d_settings" % k]
        res = helpers.oracle_qp(mats["P"].toarray() + np.triu(mats["P"].toarray(), 1).T, g["qp%d_q" % k],
                                sp.csc_matrix(mats["A"]), g["qp%d_l" % k], g["qp%d_u" % k], rho=rho, sigma=sigma,
                                eps_abs=ea, eps_rel=er, max_iter=int(mi), adaptive_rho=bool(ar))
        status, iters = g["qp%d_status" % k]
        assert res.info.status_val == status and res.info.iter == iters
        np.testing.assert_allclose(res.x, g["qp%d_x" % k], rtol=0, atol=1e-12)


def test_osqp_core_known_answers():
    """Known optima of tiny QPs as the reference's tests state them (tests/sco_osqp/test_prob.py:119-144
    -> [2, 0]; test_variable.py:69-96 -> trust region clamps to 3.0)."""
    # min x1^2 + x2^2 - 4 x1  s.t.  x1 + x2 <= 4 (free otherwise)  -> (2, 0)
    P = np.array([[2.0, 0.0], [0.0, 2.0]])
    q = np.array([-4.0, 0.0])
    A = sp.csc_matrix(np.array([[1.0, 1.0], [1.0, 0.0], [0.0, 1.0]]))
    res = helpers.oracle_qp(P, q, A, np.array([-np.inf, -np.inf, -np.inf]), np.array([4.0, np.inf, np.inf]))
    assert res.info.status_val == 1
    np.testing.assert_allclose(res.x, [2.0, 0.0], atol=1e-5)
    # min (x - 5)^2 with x in [1, 3] -> 3
    res = helpers.oracle_qp(np.array([[2.0]]), np.array([-10.0]), sp.csc_matrix(np.array([[1.0]])),
                            np.array([1.0]), np.array([3.0]))
    np.testing.assert_allclose(res.x, [3.0], atol=1e-5)
    # infeasible: x <= 0 and x >= 1
    res = helpers.oracle_qp(np.array([[2.0]]), np.array([0.0]), sp.csc_matrix(np.array([[1.0], [1.0]])),
                            np.array([-np.inf, 1.0]), np.array([0.0, np.inf]))
    assert res.info.status_val in (-3, 3)


def test_numdifftools_shim_on_the_reference_test_functions():
    """tests/sco_osqp/test_expr.py:13-17,71-78: numeric Jacobian of x, x^2, x^3 at 1, 2, -1, 0."""
    import numdifftools as nd
    for f, df in ((lambda x: x, lambda x: 1.0), (lambda x: x ** 2, lambda x: 2 * x), (lambda x: x ** 3, lambda x: 3 * x ** 2)):
        for x in (1.0, 2.0, -1.0, 0.0):
            J = nd.Jacobian(lambda v: f(v))(np.array([x]))
            assert np.allclose(J, df(x))
    H = nd.Hessian(lambda v: v[0] ** 3 + v[0] * v[1])(np.array([1.0, 2.0]))
    assert np.allclose(H, [[6.0, 1.0], [1.0, 0.0]], atol=1e-5)
