"""Constraint groups (Prob.add_cnt_expr(bexpr, group_ids), prob.py:112-144; the per-group
convergence test of Solver._min_merit_fn, solver.py:206-235): compiler output on CPU, oracle port
against the unmodified reference, device against the port."""
import numpy as np
import pytest

import api_builder
import ref_builder
import sqp_port
from sco_py_b200 import batch
from sco_py_b200 import expr as E
from sco_py_b200 import workloads as W
from sco_py_b200.sco_b200.osqp_utils import OSQPVar
from sco_py_b200.sco_b200.prob import Prob
from sco_py_b200.sco_b200.solver import Solver
from sco_py_b200.sco_b200.variable import Variable


def build(i, n=8, m=6):
    """QCQP i with its m rows split into two blocks: rows [0, m/2) in groups {a, b}, the rest in {b}."""
    st, params, x0 = W.gen_qcqp(1, n=n, m=m, first=i)
    fam = api_builder.family_expr(st, st.blocks[0], params[0])
    val = np.asarray(st.get(st.blocks[0].val, params[0], m)).reshape(-1, 1)
    prob = Prob()
    ov = np.empty((n, 1), dtype=object)
    for j in range(n):
        ov[j, 0] = OSQPVar("x%05d" % j)
        prob.add_osqp_var(ov[j, 0])
    var = Variable(ov, x0[0].reshape(n, 1))
    prob.add_var(var)
    Q = np.asarray(st.get(st.Q, params[0], n * n)).reshape(n, n)
    q = np.asarray(st.get(st.q, params[0], n)).reshape(1, n)
    prob.add_obj_expr(E.BoundExpr(E.QuadExpr(Q, q, np.zeros((1, 1))), var))
    h = m // 2
    prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(E.QuadFormExpr(fam.P[:h], fam.a[:h]), val[:h]), var), group_ids=["a", "b"])
    prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(E.QuadFormExpr(fam.P[h:], fam.a[h:]), val[h:]), var), group_ids=["b"])
    return prob, var


def _solver():
    s = Solver()
    for k, v in W.SOLVER_SETTINGS.items():
        setattr(s, k, v)
    return s


def test_groups_compile_to_masks_and_overlap():
    prob, _ = build(0)
    st, params, x0, _ = batch.compile_batch([prob])
    assert st.n_groups == 2 and [b.group_mask for b in st.blocks] == [0b11, 0b10]
    assert st.group_overlap.tolist() == [[0, 1], [1, 0]]  # "a" and "b" were named together (prob.py:139-142)
    pp = sqp_port.PortProblem(st, params[0], x0[0])
    v = pp.get_value(1.0, vectorize=True)
    sums = [float(np.sum(b.violation(pp.x))) for b in pp.blocks]
    assert np.allclose(v, [sums[0], sums[0] + sums[1]])


@pytest.mark.skipif(not ref_builder.reference_available(), reason="needs an upstream sco_py checkout at SCO_REFERENCE_ROOT")
@pytest.mark.parametrize("i", [0, 1, 2])
def test_port_equals_the_unmodified_reference_with_groups(i):
    prob, _ = build(i)
    st, params, x0, _ = batch.compile_batch([prob])
    a = sqp_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    b = ref_builder.solve_with_reference(ref_builder.import_reference(), st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    assert a["success"] == b["success"]
    assert np.abs(a["x"] - b["x"]).max() <= 1e-8


@pytest.mark.gpu
def test_device_matches_the_port_with_groups():
    built = [build(i) for i in range(6)]
    ok = _solver().solve_batch([p for p, _ in built], method="penalty_sqp")
    for i, (prob, var) in enumerate(built):
        st, params, x0, _ = batch.compile_batch([build(i)[0]])
        ref = sqp_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
        assert ok[i] == ref["success"], i
        assert np.abs(var.get_value()[:, 0] - ref["x"]).max() <= 1e-4 * max(1.0, np.abs(ref["x"]).max()), i
        assert np.allclose(prob.get_value(1.0, vectorize=True),
                           sqp_port.PortProblem(st, params[0], var.get_value()[:, 0]).get_value(1.0, vectorize=True), atol=1e-9)
