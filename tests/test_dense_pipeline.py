"""The pipelined termination test of the two-warp dense ADMM loop (sco_dense.cuh, dense_qp_solve) against the OSQP
oracle, at every dense kind.

The loop runs the test of a tested iteration k beside iteration k+1 and decides after the barrier of k+1; a verdict on
k restores iteration k's state, which the loop spilled to shared memory.  Where there is no iteration k+1 to hide the
test in (k + 1 >= max_iter, or a test interval below 2) it tests k unpipelined.  So the cases that matter are a cap
on k, k+1 and k+2 of the iteration the oracle solves at, test intervals 1, 2 and 3, and an infeasibility certificate
found on the restored state, with and without keeping the duals for a warm start.

Bars of test_qp_edges: identical status, identical ADMM iteration count, and |dx| <= 1e-7 max(1, |x|) where the
status carries a solution.
"""
import numpy as np
import pytest

import helpers
from sco_py_b200 import workloads as W

KINDS = {"dense1": (8, 6), "dense2": (12, 16), "dense3": (20, 30), "dense4": (32, 32)}  # full fill of each kind
B = 3
PI, KDUP = 10.0, 2


@pytest.fixture(scope="module")
def dense_qps():
    """kind -> (Engine, structure, params, x0, J, b), created once per module."""
    from sco_py_b200.engine import Engine
    cache = {}

    def get(kind):
        if kind not in cache:
            n, m = KINDS[kind]
            st, params, x0 = W.gen_qcqp(B, n=n, m=m)
            eng = Engine(st)
            assert eng.team == 64, "expected the two-warp dense loop"
            _, J, b, _ = eng.convexify(params, x0)
            cache[kind] = (eng, st, params, x0, J, b)
        return cache[kind]
    yield get
    for e in cache.values():
        e[0].close()


def _settings(**kw):
    from sco_py_b200.engine import make_settings
    return make_settings(solver=W.SOLVER_SETTINGS, **kw)


def _solve(eng, params, J, b, lbx, ubx, bits=None, **kw):
    n = params.shape[0]
    mask = None if bits is None else np.ascontiguousarray(bits).view(np.int32)
    xq, status, iters = eng.qp_solve(params, _settings(**kw), J=J, b=b, lbx=lbx, ubx=ubx, pi=np.full(n, PI),
                                     kdup=np.full(n, KDUP, np.int32), mask=mask)
    return xq.cpu().numpy(), status.cpu().numpy(), iters.cpu().numpy()


def _qps(st, params, J, b, lbx, ubx, bits=None):
    Jn, bn = J.cpu().numpy(), b.cpu().numpy()
    return [helpers.stage_qp(st, params[i], Jn[i], bn[i], lbx[i], ubx[i], PI, KDUP,
                             bits=None if bits is None else bits[i]) for i in range(params.shape[0])]


def _match(got, qps, where, **oracle_kw):
    """Device results against the oracle -> the oracle statuses."""
    x, status, iters = got
    seen = []
    for i, qp in enumerate(qps):
        res = helpers.oracle_qp(*qp, **oracle_kw)
        info = (where, i, "device", int(status[i]), int(iters[i]), "oracle", res.info.status_val, res.info.iter)
        assert status[i] == res.info.status_val, info
        assert iters[i] == res.info.iter, info
        if res.info.status_val in (1, 2, -2):
            err = np.abs(x[i] - res.x).max()
            assert err <= 1e-7 * max(1.0, np.abs(res.x).max()), info + (err,)
        seen.append(res.info.status_val)
    return seen


@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(KINDS))
def test_cap_on_the_tested_iteration_and_the_two_after_it(dense_qps, kind):
    """max_iter = k, k+1, k+2 for the iteration k the oracle solves at: k and k+1 test k unpipelined, k+2 decides on k
    after iteration k+1 and has to return k's iterates, status and count."""
    eng, st, params, x0, J, b = dense_qps(kind)
    lbx, ubx = x0 - 1.0, x0 + 1.0
    qps = _qps(st, params, J, b, lbx, ubx)
    for i in range(B):
        k = helpers.oracle_qp(*qps[i]).info.iter
        for cap in (k, k + 1, k + 2):
            got = _solve(eng, params[i:i + 1], J[i:i + 1], b[i:i + 1], lbx[i:i + 1], ubx[i:i + 1], osqp_max_iter=cap)
            assert _match(got, qps[i:i + 1], (kind, i, "cap", k, cap), max_iter=cap) == [1], (kind, i, cap)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(KINDS))
@pytest.mark.parametrize("ct", [1, 2, 3])
def test_short_test_intervals(dense_qps, kind, ct):
    """Interval 1 tests unpipelined; at 2 the next test follows the decision of the last one directly."""
    eng, st, params, x0, J, b = dense_qps(kind)
    lbx, ubx = x0 - 1.0, x0 + 1.0
    got = _solve(eng, params, J, b, lbx, ubx, osqp_check_termination=ct)
    assert set(_match(got, _qps(st, params, J, b, lbx, ubx), (kind, "ct", ct), check_termination=ct)) == {1}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(KINDS))
@pytest.mark.parametrize("warm_start", [0, 2])
def test_certificate_stop_returns_the_tested_iteration(dense_qps, kind, warm_start):
    """No quadratic term, every Jacobian slot masked off and no box: the dual certificate (-4) holds, found by
    dense_certificates on the spilled state of the tested iteration after iteration k+1 has run."""
    eng, st, params, x0, J, b = dense_qps(kind)
    n = st.n
    flat = params.copy()
    flat[:, st.Q.off:st.Q.off + n * n] = 0.0
    bits = np.zeros((B, st.m_nl, eng.mask_words), np.uint32)
    inf = np.full((B, n), np.inf)
    got = _solve(eng, flat, J, b, -inf, inf, bits, warm_start=warm_start)
    assert set(_match(got, _qps(st, flat, J, b, -inf, inf, bits), (kind, "dinf", warm_start))) == {-4}
