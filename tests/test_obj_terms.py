"""Non-quadratic objective terms as the reference takes them (prob.py:97-103, 522-544; expr.py:143-153, 431-437): any
number, each a scalar SymExpr bound to any Variable, each convexified on its own -- from the structure compiler
(Structure.obj_blocks) through the C ABI (sco_obj_block_desc) to the device's per-term convexification, the QP on the
union pattern of P and the merits."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest

import bound_port
import bound_problems as BP
import obj_legacy
import obj_port
import obj_problems as OP
import ref_builder
import test_c1_toy as C1
import test_caps as CAPS
from sco_py_b200 import _lib, batch, batchfile
from sco_py_b200 import expr as E
from sco_py_b200 import sym
from sco_py_b200 import workloads as W
from sco_py_b200.structure import Field, ObjBlock

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# sha256 of repr(batch.signature(st)) of the chains of test_caps.py (one term over all variables in QP order) as
# computed by the version before objective blocks existed: they keep the obj_prog structure
SIGNATURES = {
    (20, False): '0659bd1a741b91453f080f536192e7edf9fd162dbd50f825dccad91755697509',
    (20, True): 'd061cbc6e6c6fadb9ae260024901fe911819bf0bff5c96bdf6e0ca1d77988ebf',
    (40, False): 'b05523679bffcb67f4843c3df1ded51d41262dba1bcbcf4f0404ece2dc460695',
    (40, True): '28450bc754e79888908ca75b9de8469666f509f025d7318d0002f5962d3cf107',
}


def _compile(probs):
    return batch.compile_batch(probs)


def _names(n):
    return ["v%02d" % j for j in range(n)]


def _free_prob(n, x0=None):
    ov = BP._scalars(_names(n))
    x0 = np.linspace(0.1, 0.5, n) if x0 is None else np.asarray(x0, dtype=float)
    prob, allv = BP._start(ov, x0)
    prob.add_obj_expr(E.BoundExpr(E.QuadExpr(0.1 * np.eye(n), np.zeros((1, n)), np.zeros((1, 1))), allv))
    return prob, ov, x0


def _permuted_c1(name, analytic=False):
    """C1 problem `name` with its non-quadratic objective bound to the Variable (x2, x1)."""
    prob, var, x_true = C1.build_sym(name, analytic=analytic)
    f = prob._nonquad_obj_exprs[0].expr.rows[0]
    prob._nonquad_obj_exprs.clear()
    ov = var.get_osqp_vars()
    pv = BP.Variable(ov[[1, 0]], var.get_value()[[1, 0]])
    prob.add_obj_expr(E.BoundExpr(E.SymExpr([OP.remap(f, [1, 0])], 2, analytic=analytic), pv))
    return prob, var, x_true


# ---------------------------------------------------------------------------------------------------- CPU
def test_per_step_terms_compile_to_one_mapped_block():
    st, params, x0, _ = _compile([OP.robot(0, T=5)])
    assert st.obj_prog_len == 0 and st.obj_prog.off < 0 and len(st.obj_blocks) == 1
    ob = st.obj_blocks[0]
    assert (ob.m, ob.n_in, ob.flags) == (5, 2, 0)
    np.testing.assert_array_equal(ob.cols, np.arange(10).reshape(5, 2))
    prog = st.get(ob.prog, params[0], ob.m + 2 * ob.n_instr)
    assert prog[0] == 0 and np.all(np.diff(prog[:ob.m]) > 0)  # row offsets of the packed program


def test_subset_in_permuted_order_and_two_input_counts():
    prob, ov, x0 = _free_prob(6)
    x = sym.variables(3)
    OP.add_terms(prob, ov, x0, [(x[0] * x[1] - x[2] ** 2, np.array([4, 1, 2]))])
    y = sym.variables(2)
    OP.add_terms(prob, ov, x0, [(y[0] ** 3 - y[1], np.array([5, 0]))], analytic=True)
    OP.add_terms(prob, ov, x0, [(x[2] * x[0] + x[1], np.array([0, 3, 5]))])
    st, params, _, _ = _compile([prob])
    assert [(o.m, o.n_in, o.flags) for o in st.obj_blocks] == [(2, 3, 0), (1, 2, 1)]
    np.testing.assert_array_equal(st.obj_blocks[0].cols, [[4, 1, 2], [0, 3, 5]])
    np.testing.assert_array_equal(st.obj_blocks[1].cols, [[5, 0]])
    # the port evaluates term r of a block on x[cols[r]]
    terms = obj_port.terms_of(st, params[0])
    xv = np.linspace(-1.0, 1.0, 6)
    assert terms[0][0](xv[[4, 1, 2]]) == pytest.approx(xv[4] * xv[1] - xv[2] ** 2)
    assert terms[1][0](xv[[0, 3, 5]]) == pytest.approx(xv[5] * xv[0] + xv[3])
    assert terms[2][0](xv[[5, 0]]) == pytest.approx(xv[5] ** 3 - xv[0])


def test_legacy_objective_keeps_its_fields_and_signature():
    for n in (20, 40):
        for analytic in (False, True):
            st, params, _, cps = _compile([CAPS.build_chain(p, analytic=analytic)[0] for p in CAPS.chain_points(2, n)])
            assert st.obj_prog_len > 0 and st.obj_blocks == [] and st.obj_prog_flags == int(analytic)
            assert hashlib.sha256(repr(batch.signature(st)).encode()).hexdigest() == SIGNATURES[(n, analytic)]
            for c, row in zip(cps, params):  # the program of the one-term block is the term's own
                (pk, _), = c.obj_blocks
                (term,) = pk.parts
                assert np.array_equal(pk.params(), term.params())
                assert np.array_equal(st.get(st.obj_prog, row, 1 + 2 * st.obj_prog_len), term.params())


def test_refusals_name_their_limit():
    prob, ov, x0 = _free_prob(4)
    prob.add_obj_expr(E.BoundExpr(E.Expr(lambda v: float(np.sum(v ** 2))), BP._sub(ov, x0, [0, 1])))
    with pytest.raises(batch.UnsupportedProblem, match="black-box.*no CPU fallback"):
        _compile([prob])
    prob, ov, x0 = _free_prob(70)
    x = sym.variables(65)
    OP.add_terms(prob, ov, x0, [(sum(x[1:], x[0] ** 2), np.arange(65))])
    with pytest.raises(batch.UnsupportedProblem, match="65 variables.*limit is 64"):
        _compile([prob])
    prob, ov, x0 = _free_prob(4)
    x = sym.variables(2)
    prob.add_obj_expr(E.BoundExpr(E.SymExpr([x[0] * x[1]], 2), BP._sub(ov, x0, [1, 1])))
    with pytest.raises(batch.UnsupportedProblem, match="more than once"):
        _compile([prob])
    prob, ov, x0 = _free_prob(8)
    for k in range(1, 6):  # five input counts: five blocks
        x = sym.variables(k)
        OP.add_terms(prob, ov, x0, [(sum(x[1:], x[0] ** 4), np.arange(k))])
    with pytest.raises(batch.UnsupportedProblem, match="5 objective blocks.*limit is 4"):
        _compile([prob])


def test_blocks_enter_the_batch_identity_and_the_batch_file(tmp_path):
    p1, p2 = OP.robot(0, T=4), OP.robot(1, T=4)
    c1, c2 = batch.compile_problem(p1), batch.compile_problem(p2)
    assert batch.group_key(c1) == batch.group_key(c2)
    prob, ov, x0 = _free_prob(8)
    OP.add_terms(prob, ov, x0, [(OP.soft_obstacle(), np.array([0, 1])), (OP.soft_obstacle(), np.array([2, 3]))])
    other, ov2, x02 = _free_prob(8)
    OP.add_terms(other, ov2, x02, [(OP.soft_obstacle(), np.array([0, 1])), (OP.soft_obstacle(), np.array([3, 2]))])
    ca, cb = batch.compile_problem(prob), batch.compile_problem(other)
    assert batch.group_key(ca) != batch.group_key(cb)  # same sizes, different maps
    with pytest.raises(batch.UnsupportedProblem, match="does not share the structure"):
        batch.compile_batch([prob, other])
    sta = batch.compile_batch([prob])[0]
    stb = batch.compile_batch([other])[0]
    assert batch.signature(sta) != batch.signature(stb)
    st, params, x0s, _ = batch.compile_batch([p1, p2])
    path = str(tmp_path / "b.npz")
    batchfile.save_batch(path, st, params, x0s)
    st2, params2, _, meta = batchfile.load_batch(path)
    assert batch.signature(st2) == batch.signature(st) and len(st2.obj_blocks) == 1
    np.testing.assert_array_equal(st2.obj_blocks[0].cols, st.obj_blocks[0].cols)
    np.testing.assert_array_equal(params2, params)
    # a file written before objective blocks existed
    st3, _, _, _ = batchfile.load_batch(os.path.join(ROOT, "tests", "golden", "batch_parent_point_robot.npz"))
    assert st3.obj_blocks == []


def test_c_layout_of_the_objective_blocks_matches_ctypes(tmp_path):
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "sco_b200.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(sco_structure_desc),\n'
                   '         offsetof(sco_structure_desc, n_obj_blocks), offsetof(sco_structure_desc, obj_blocks),\n'
                   '         sizeof(sco_obj_block_desc), offsetof(sco_obj_block_desc, m), offsetof(sco_obj_block_desc, n_in),\n'
                   '         offsetof(sco_obj_block_desc, n_instr), offsetof(sco_obj_block_desc, flags),\n'
                   '         offsetof(sco_obj_block_desc, prog), offsetof(sco_obj_block_desc, cols));\n  return 0;\n}\n')
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    S, O = _lib.CStructure, _lib.CObjBlock
    assert got == [ctypes.sizeof(S), S.n_obj_blocks.offset, S.obj_blocks.offset, ctypes.sizeof(O), O.m.offset,
                   O.n_in.offset, O.n_instr.offset, O.flags.offset, O.prog.offset, O.cols.offset]
    assert _lib.MAX_OBJ_BLOCKS == 4


def test_port_convexifies_every_term_on_its_own():
    """f1 = x0 x1 and f2 = -x0 x1 on one Variable: each term's Hessian has eigenvalues +-1 and is shifted by 1, so the
    model is 2 I; the model of the sum would be 0."""
    prob, ov, x0 = _free_prob(2)
    x = sym.variables(2)
    OP.add_terms(prob, ov, x0, [(x[0] * x[1], np.array([0, 1])), (-(x[0] * x[1]), np.array([0, 1]))])
    st, params, x0s, _ = _compile([prob])
    H, A, c = obj_port.model_at(st, params[0], x0s[0])
    np.testing.assert_allclose(H, 2.0 * np.eye(2), atol=1e-8)


@pytest.mark.parametrize("i", [0, 1])
def test_port_mapped_terms_equal_the_lifted_ones(i):
    """Convex per-step costs (zero shift either way): bound to each step's Variable, or each lifted to all variables
    (zero-padded inputs, still one term per step) -- the same optimisation problem."""
    rs = []
    for form in ("bound", "lifted"):
        st, params, x0, _ = _compile([OP.robot(i, T=5, form=form, cost="convex")])
        rs.append(obj_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS))
    a, b = rs
    assert a["success"] == b["success"]
    assert (a["stats"]["sqp_iters"], a["stats"]["qp_solves"]) == (b["stats"]["sqp_iters"], b["stats"]["qp_solves"])
    assert np.abs(a["x"] - b["x"]).max() <= 1e-9 * max(1.0, np.abs(b["x"]).max())


@pytest.mark.skipif(not ref_builder.reference_available(), reason="needs an upstream sco_py checkout at SCO_REFERENCE_ROOT")
def test_port_equals_the_unmodified_reference_on_bound_terms():
    """The reference's own Prob with one BoundExpr(Expr(f_t), v_t) per term, v_t a Variable of the term's scalars."""
    ref = ref_builder.import_reference()
    st, params, x0, _ = _compile([OP.robot(0, T=4)])
    with bound_port.mapped_port():
        prob, var = ref_builder.build_prob(ref, st, params[0], x0[0])
    ovars = var.get_osqp_vars()
    for f, _, c in obj_port.terms_of(st, params[0]):
        v = ref["variable"].Variable(ovars[c], value=np.asarray(x0[0])[c].reshape(-1, 1))
        prob.add_var(v)
        prob.add_obj_expr(ref["expr"].BoundExpr(ref["expr"].Expr(lambda x, f=f: f(np.asarray(x).ravel())), v))
    solv = ref["solver"].Solver()
    for k, val in W.SOLVER_SETTINGS.items():
        setattr(solv, k, val)
    ok = solv.solve(prob, method="penalty_sqp")
    mine = obj_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    xr = var.get_value()[:, 0]
    assert mine["success"] == bool(ok)
    assert np.abs(mine["x"] - xr).max() <= 1e-6 * max(1.0, np.abs(xr).max())


# ---------------------------------------------------------------------------------------------------- GPU
def _engine(st):
    from sco_py_b200.engine import Engine
    return Engine(st)


def _settings(**kw):
    from sco_py_b200.engine import make_settings
    return make_settings(solver=W.SOLVER_SETTINGS, **kw)


def _overlapping_prob(i):
    prob, ov, x0 = _free_prob(7, x0=np.random.default_rng(i).uniform(-1, 1, 7))
    x = sym.variables(3)
    OP.add_terms(prob, ov, x0, [(sym.sin(x[0] * x[1]) + x[2] ** 4 - x[0] * x[2], np.array([0, 1, 2])),
                                (sym.cos(x[0] + x[1]) * x[2], np.array([2, 1, 4])),
                                (x[0] ** 2 * x[1] - x[2], np.array([6, 2, 5]))])
    OP.add_terms(prob, ov, x0, [(OP.pair_cost(), np.array([3, 5, 1, 0]))], analytic=True)
    return prob


MODEL_CASES = {
    "per_step": lambda i: OP.robot(i, T=12),
    "overlapping": _overlapping_prob,
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(MODEL_CASES))
def test_convexify_model_matches_the_port(case):
    probs = [MODEL_CASES[case](i) for i in range(3)]
    st, params, x0, _ = _compile(probs)
    eng = _engine(st)
    H, g, c = [t.cpu().numpy() for t in eng.convexify_model(params, x0)]
    eng.close()
    analytic = any(o.flags & 1 for o in st.obj_blocks)
    for i in range(len(probs)):
        Hr, gr, cr = obj_port.model_at(st, params[i], x0[i])
        tol = 1e-7
        np.testing.assert_allclose(H[i], Hr, rtol=tol, atol=tol)
        np.testing.assert_allclose(g[i], gr, rtol=tol, atol=tol * (1 + np.abs(gr).max()))
        assert abs(c[i] - cr) <= tol * max(1.0, abs(cr))
    assert analytic == (case == "overlapping")


@pytest.mark.gpu
def test_device_convexifies_every_term_on_its_own():
    prob, ov, x0 = _free_prob(2)
    x = sym.variables(2)
    OP.add_terms(prob, ov, x0, [(x[0] * x[1], np.array([0, 1])), (-(x[0] * x[1]), np.array([0, 1]))])
    st, params, x0s, _ = _compile([prob])
    eng = _engine(st)
    H, g, c = [t.cpu().numpy() for t in eng.convexify_model(params, x0s)]
    eng.close()
    np.testing.assert_allclose(H[0], 2.0 * np.eye(2), atol=1e-7)


SOLVE_CASES = {
    # (a) per-step soft-obstacle costs: union pattern <= 4 entries per column, thread-per-entity loop + inline test
    "robot12_step": lambda i: OP.robot(i, T=12),
    # (b) C2's point robot size, n = 80 > 64
    "robot40_step": lambda i: OP.robot(i, T=40, K=3),
    # (c) pairwise costs over consecutive steps with bound SymExpr constraints in groups
    "robot10_pair": lambda i: OP.robot(i, T=10, cost="pair", groups=lambda t: [t % 2]),
}
SOLVE_CASES.update({"c1_" + nm: (lambda i, nm=nm: _permuted_c1(nm, analytic=bool(i % 2))[0]) for nm in sorted(C1.SYM_PROBLEMS)})


def _pattern_columns(st):
    n = st.n
    P = np.asarray(st.get(st.Q, st.shared, n * n) if st.Q.shared else np.ones(n * n)).reshape(n, n) != 0
    P = P | P.T
    for o in st.obj_blocks:
        for c in o.cols:
            P[np.ix_(c, c)] = True
    return P.sum(axis=0)


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(SOLVE_CASES))
def test_full_solve_matches_the_port(case):
    B = 2 if case.startswith("c1_") else 3
    probs = [SOLVE_CASES[case](i) for i in range(B)]
    if case.startswith("c1_"):  # analytic and FD gradients are different structures: one launch each
        groups = [[p] for p in probs]
    else:
        groups = [probs]
    for grp in groups:
        st, params, x0, _ = _compile(grp)
        if case == "robot12_step":
            assert _pattern_columns(st).max() <= 4  # the in-loop termination test applies
        eng = _engine(st)
        outs = []
        for fg in (0, 1):
            r = eng.solve_batch(params, x0, _settings(force_generic=fg))
            outs.append({k: v.cpu().numpy() for k, v in r.items()})
        eng.close()
        a, b = outs
        # thread-per-entity loop == strided loop.  Not for C1 prob3 with finite differences: there the two loops take
        # different SQP paths in the version before objective blocks too (tests/golden/obj_legacy_parent.npz:
        # 7 / 8 against 8 / 9 SQP iterations / QPs, |dx| 5e-10), so only the port comparison below applies.
        split = case == "c1_prob3" and not any(o.flags & 1 for o in st.obj_blocks)
        for i in range(x0.shape[0] if not split else 0):
            assert a["verdict"][i] == b["verdict"][i] and (a["stats"][i] == b["stats"][i]).all(), (i, a["stats"][i], b["stats"][i])
            assert np.abs(a["x"][i] - b["x"][i]).max() <= 1e-9 * max(1.0, np.abs(b["x"][i]).max())
        for i in range(x0.shape[0]):
            ref = obj_port.solve(st, params[i], x0[i], solver=W.SOLVER_SETTINGS)
            for o in (a, b) if split else (a,):
                assert (o["verdict"][i] == 1) == ref["success"], (case, i, o["stats"][i].tolist(), ref["stats"])
                assert abs(o["max_vio"][i] - ref["max_vio"]) <= 1e-5
                assert abs(o["objective"][i] - ref["objective"]) <= 1e-5 * max(1.0, abs(ref["objective"]))
                assert np.abs(o["x"][i] - ref["x"]).max() <= 1e-4 * max(1.0, np.abs(ref["x"]).max())


def _desc_error(st):
    from sco_py_b200.engine import Engine
    with pytest.raises(RuntimeError) as ei:
        Engine(st)
    return str(ei.value)


@pytest.mark.gpu
def test_sco_create_refuses_bad_objective_blocks():
    import copy
    st0, _, _, _ = _compile([OP.robot(0, T=4)])

    def bad(fn):
        st = copy.deepcopy(st0)
        fn(st)
        return _desc_error(st)

    ob = lambda st: st.obj_blocks[0]  # noqa: E731
    assert "error -1" in bad(lambda st: ob(st).cols.__setitem__((0, 0), st.n)) and "outside" in bad(
        lambda st: ob(st).cols.__setitem__((0, 0), st.n))
    assert "repeats" in bad(lambda st: ob(st).cols.__setitem__((1, 1), ob(st).cols[1, 0]))

    def wide(st):
        o = ob(st)
        st.obj_blocks[0] = ObjBlock(o.prog, 1, 65, o.n_instr, o.flags, np.arange(65, dtype=np.int32)[None, :] % st.n)
    assert "n_in = 65" in bad(wide)
    assert "outside its parameter block" in bad(
        lambda st: setattr(ob(st), "prog", Field(st.stride - 1, False)) if not ob(st).prog.shared else setattr(
            ob(st), "prog", Field(len(st.shared) - 1, True)))

    def both(st):
        st.obj_prog, st.obj_prog_len = Field(0, False), 1
    assert "both set" in bad(both)


@pytest.mark.gpu
def test_legacy_objectives_give_the_parent_bits():
    ref = np.load(obj_legacy.GOLDEN)
    got = obj_legacy.compute()
    assert sorted(got) == sorted(ref.files)
    diff = [k for k in ref.files if not np.array_equal(got[k], ref[k], equal_nan=True)]
    assert not diff, diff
