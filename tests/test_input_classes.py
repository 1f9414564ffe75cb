"""Input classes beyond the three benchmark configurations: AffExpr objective terms (quirk C-4,
prob.py:220-221,240-249; pinned by tests/sco_osqp/test_prob.py:95-117), user bounds on the scalar variables
(find_closest_feasible_point honours them, prob.py:369-412), constraint groups with the
nonconverged_groups report (solver.py:206-235) and the callback hook (prob.py:204).
CPU: structure compiler + oracle port against the unmodified reference.  GPU: device against the port."""
import numpy as np
import pytest

import api_builder
import ref_builder
import sqp_port
from sco_py_b200 import batch
from sco_py_b200 import workloads as W
from sco_py_b200.sco_b200.solver import Solver, nonconverged_list

needs_reference = pytest.mark.skipif(not ref_builder.reference_available(),
                                     reason="needs an upstream sco_py checkout at SCO_REFERENCE_ROOT")

GROUPS = [(slice(0, 2), ["a", "b"]), (slice(2, 4), ["b"]), (slice(4, 5), ["c"]), (slice(5, 6), [])]
VARIANTS = {
    "aff": dict(aff=True),
    "bounds": dict(bounds=True),
    "groups": dict(groups=GROUPS),
    "nogroup": dict(groups=[(slice(0, 6), [])]),
    "all": dict(aff=True, bounds=True, groups=GROUPS),
}
# tighter than the benchmark settings so that the per-group stall test of solver.py:209-235 fires on some problems
GROUP_SETTINGS = dict(W.SOLVER_SETTINGS, max_merit_coeff_increases=2, min_approx_improve=1e-3)


def _solver(settings):
    s = Solver()
    for k, v in settings.items():
        setattr(s, k, v)
    return s


def test_compiler_fields():
    prob, _ = api_builder.build_qcqp_variant(0, **VARIANTS["all"])
    st, params, x0, cps = batch.compile_batch([prob])
    assert st.qa.off >= 0 and st.lb0.off >= 0 and st.ub0.off >= 0
    assert st.n_groups == 3 and [b.group_mask for b in st.blocks] == [0b011, 0b010, 0b100, 0]
    pp = sqp_port.PortProblem(st, params[0], x0[0])
    assert np.isfinite(pp.lb0).all() and pp.qa is not None
    prob, _ = api_builder.build_qcqp_variant(0, **VARIANTS["nogroup"])
    st, _, _, _ = batch.compile_batch([prob])
    assert st.n_groups == 0 and st.blocks[0].group_mask == 0


def test_nonconverged_list_decoding():
    assert nonconverged_list(["a", "b", "c"], 0) == []
    assert nonconverged_list(["a", "b", "c"], 0b010 | (0b110 << 16)) == ["b", "b", "c"]


@needs_reference
@pytest.mark.parametrize("variant", sorted(VARIANTS))
@pytest.mark.parametrize("i", [0, 1, 2, 3])
def test_port_equals_the_unmodified_reference(variant, i):
    settings = GROUP_SETTINGS if "group" in variant or variant == "all" else W.SOLVER_SETTINGS
    prob, _ = api_builder.build_qcqp_variant(i, **VARIANTS[variant])
    st, params, x0, cps = batch.compile_batch([prob])
    a = sqp_port.solve(st, params[0], x0[0], solver=settings)
    b = ref_builder.solve_with_reference(ref_builder.import_reference(), st, params[0], x0[0], solver=settings)
    assert a["success"] == b["success"]
    assert np.abs(a["x"] - b["x"]).max() <= 1e-8
    # ref_builder names group g of the structure "g%02d": same sorted order as the structure's indices
    assert ["g%02d" % g for g in a["nonconverged"]] == b["nonconverged"]


def test_some_group_problem_reports_nonconverged_groups():
    """The parity above must not be vacuous: at least one of the group problems ends with a non-empty list."""
    hits = 0
    for i in range(12):
        prob, _ = api_builder.build_qcqp_variant(i, **VARIANTS["groups"])
        st, params, x0, _ = batch.compile_batch([prob])
        hits += bool(sqp_port.solve(st, params[0], x0[0], solver=GROUP_SETTINGS)["nonconverged"])
    assert hits > 0


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_device_matches_the_port(variant):
    settings = GROUP_SETTINGS if "group" in variant or variant == "all" else W.SOLVER_SETTINGS
    count = 12
    built = [api_builder.build_qcqp_variant(i, **VARIANTS[variant]) for i in range(count)]
    calls = []
    for i, (p, _) in enumerate(built):
        p._callback = (lambda i=i: calls.append(i))
    ok = _solver(settings).solve_batch([p for p, _ in built], method="penalty_sqp")
    assert sorted(calls) == list(range(count))  # the callback hook ran once per problem
    for i, (prob, var) in enumerate(built):
        fresh, _ = api_builder.build_qcqp_variant(i, **VARIANTS[variant])
        st, params, x0, cps = batch.compile_batch([fresh])
        ref = sqp_port.solve(st, params[0], x0[0], solver=settings)
        assert ok[i] == ref["success"], i
        assert np.abs(var.get_value()[:, 0] - ref["x"]).max() <= 1e-4 * max(1.0, np.abs(ref["x"]).max()), i
        assert prob.nonconverged_groups == [cps[0].gids[g] for g in ref["nonconverged"]], i


@pytest.mark.gpu
def test_affexpr_objective_known_answer_of_the_reference_suite():
    """tests/sco_osqp/test_prob.py:95-117: min x^2 - 2x (QuadExpr) + (-2x) (AffExpr), update_obj(0), optimize -> 1.0
    on the OSQP backend (the AffExpr term is scaled by the penalty coefficient 0); the Gurobi backend's twin
    (tests/sco_gurobi/test_prob.py:105-125) expects the true minimiser 2.0."""
    from sco_py_b200 import expr as E
    from sco_py_b200.sco_b200.osqp_utils import OSQPVar
    from sco_py_b200.sco_b200.prob import Prob
    from sco_py_b200.sco_b200.variable import Variable
    quad = E.QuadExpr(2 * np.eye(1), -2 * np.ones((1, 1)), np.zeros((1, 1)))
    aff = E.AffExpr(-2 * np.ones((1, 1)), np.zeros((1, 1)))
    for coeff, want in ((0.0, 1.0), (1.0, 2.0)):  # weight (0 + 1) * coeff on the AffExpr term
        prob = Prob()
        ov = OSQPVar("x")
        prob.add_osqp_var(ov)
        var = Variable(np.array([[ov]]), np.zeros((1, 1)))
        prob.add_var(var)
        prob.add_obj_expr(E.BoundExpr(quad, var))
        prob.add_obj_expr(E.BoundExpr(aff, var))
        prob.update_obj(penalty_coeff=coeff)
        assert prob.optimize()
        assert np.allclose(var.get_value(), np.array([[want]]))
