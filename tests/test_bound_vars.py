"""Nonlinear constraints bound to any Variable (BoundExpr(expr, var), expr.py:413-437): per-row column maps of
constraint blocks (Block.cols, include/sco_b200.h), from the structure compiler through the device families, the QP
stage and the full solve."""
import os
import re
import subprocess

import numpy as np
import pytest

import bound_port
import bound_problems as BP
import helpers
import sqp_port
from sco_py_b200 import batch, batchfile
from sco_py_b200 import expr as E
from sco_py_b200 import sym
from sco_py_b200 import workloads as W
from sco_py_b200.sco_b200.osqp_utils import OSQPVar
from sco_py_b200.sco_b200.prob import Prob
from sco_py_b200.sco_b200.solver import Solver
from sco_py_b200.sco_b200.variable import Variable
from sco_py_b200.structure import FAM_CIRCLE2D, FAM_FK7, FAM_QUADFORM, FAM_VM, Block, Field, Structure

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# sha256 of repr(batch.signature(st)) for problems whose constraints are bound to all variables in QP order, as
# computed by the version before column maps existed: such problems must compile to the same structures
SIGNATURES = {
    "qcqp[('m', 6), ('n', 8)]": 'a6572eafed93323c223d245ae9db0871f31fffb76174fd655c136272d0985209',
    "qcqp[('m', 30), ('n', 20)]": '4c1cf5f3fc6db10a10f7c2ad0e333289b7678e2f7fb6d7d1c554bb8c590caca1',
    "point_robot[('K', 3), ('T', 12)]": '96502cfcaeea5b19720d1d1a3b49b33f60b68c816350dbea74ac810c6169d92d',
}


def _small_prob(names=("c", "a", "g", "e", "b", "f", "d")):
    """Scalar variables added in a scrambled order; QP order is the names' order a..g."""
    prob = Prob()
    ov = {nm: OSQPVar(nm) for nm in names}
    for nm in names:
        prob.add_osqp_var(ov[nm])
    allv = Variable(np.array([[ov[nm]] for nm in sorted(names)], dtype=object), np.arange(len(names), dtype=float)[:, None] * 0.1)
    prob.add_var(allv)
    n = len(names)
    prob.add_obj_expr(E.BoundExpr(E.QuadExpr(np.eye(n), np.zeros((1, n)), np.zeros((1, 1))), allv))
    return prob, ov


def _var(ov, names):
    return Variable(np.array([[ov[nm]] for nm in names], dtype=object), np.linspace(0.1, 0.9, len(names))[:, None])


# ---------------------------------------------------------------------------------------------------- CPU
def test_columns_follow_the_variable_order():
    prob, ov = _small_prob()
    P = np.array([[[2.0, 0.5], [0.5, 1.0]]])
    prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(E.QuadFormExpr(P, np.ones((1, 2))), np.ones((1, 1))), _var(ov, "db")))
    x = sym.variables(3)
    prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(E.SymExpr([x[0] * x[1] - x[2], x[2] ** 2], 3), np.ones((2, 1))),
                                  _var(ov, "gac")))
    prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(E.CircleDistExpr(2, [[0.0, 0.0]], [0.5]), np.zeros((2, 1))),
                                  _var(ov, "edba")))
    prob.add_cnt_expr(E.BoundExpr(E.EqExpr(E.FK7Expr(7), np.zeros((3, 1))), _var(ov, "gfedcba")))
    st, _, _, _ = batch.compile_batch([prob])
    fams = [(b.family, b.m, b.jw, b.n_in) for b in st.blocks]
    assert fams == [(FAM_QUADFORM, 1, 2, 2), (FAM_VM, 2, 3, 3), (FAM_CIRCLE2D, 2, 2, 2), (FAM_FK7, 3, 7, 7)]
    assert st.blocks[0].cols.tolist() == [[3, 1]]
    assert st.blocks[1].cols.tolist() == [[6, 0, 2]] * 2
    assert st.blocks[1].ipar[:4] == [3, 2, st.blocks[1].ipar[2], 0]
    assert st.blocks[2].cols.tolist() == [[4, 3], [1, 0]]
    assert st.blocks[3].cols.tolist() == [[6, 5, 4, 3, 2, 1, 0]] * 3
    for bi in range(4):
        assert np.array_equal(st.jac_cols(bi), st.blocks[bi].cols)
        assert st.blocks[bi].cols.dtype == np.int32


def test_bound_to_everything_in_qp_order_keeps_the_structure():
    import hashlib
    got = {}
    for key, kw in (("qcqp", dict(n=8, m=6)), ("qcqp", dict(n=20, m=30)), ("point_robot", dict(T=12, K=3))):
        import api_builder
        st, params, x0 = W.GENERATORS[key](1, **kw)
        prob = api_builder.build_prob(st, params[0], x0[0])[0]
        stc = batch.compile_batch([prob])[0]
        assert all(b.cols is None for b in stc.blocks)
        got["%s%s" % (key, sorted(kw.items()))] = hashlib.sha256(repr(batch.signature(stc)).encode()).hexdigest()
    assert got == SIGNATURES


def test_bound_constraints_of_one_kind_share_a_device_block():
    prob, ov = _small_prob()
    x = sym.variables(2)
    sq = lambda: E.SymExpr([x[0] * x[0] + x[1]], 2)
    P1 = np.array([[[1.0, 0.0], [0.0, 1.0]]])
    add = lambda e, names, **kw: prob.add_cnt_expr(E.BoundExpr(e, _var(ov, names)), **kw)
    add(E.LEqExpr(sq(), np.full((1, 1), 1.0)), "ab")                               # VM leq           -> block 0
    add(E.LEqExpr(E.QuadFormExpr(P1, np.ones((1, 2))), np.full((1, 1), 2.0)), "cd")  # QUADFORM leq   -> block 1
    add(E.LEqExpr(sq(), np.full((1, 1), 3.0)), "ge")                               # VM leq           -> block 0
    add(E.EqExpr(sq(), np.full((1, 1), 4.0)), "bc")                                # VM eq            -> block 2
    add(E.LEqExpr(sq(), np.full((1, 1), 5.0)), "fa", group_ids=["g1"])             # other group set  -> block 3
    add(E.LEqExpr(E.SymExpr([x[0] * x[1]], 2, analytic=True), np.full((1, 1), 6.0)), "cf")  # analytic -> block 4
    xs = sym.variables(3)
    add(E.LEqExpr(E.SymExpr([xs[0] + xs[1] * xs[2]], 3), np.full((1, 1), 7.0)), "abc")     # 3 inputs -> block 5
    add(E.LEqExpr(E.QuadFormExpr(P1 * 2, np.zeros((1, 2))), np.full((1, 1), 8.0)), "ag")  # QUADFORM leq   -> block 1
    add(E.LEqExpr(sq(), np.full((1, 1), 9.0)), "dg")                               # VM leq           -> block 0
    st, params, x0, cps = batch.compile_batch([prob])
    assert [(b.family, b.cnt_type, b.m, b.n_in) for b in st.blocks] == [
        (FAM_VM, 0, 3, 2), (FAM_QUADFORM, 0, 2, 2), (FAM_VM, 1, 1, 2), (FAM_VM, 0, 1, 2), (FAM_VM, 0, 1, 2),
        (FAM_VM, 0, 1, 3)]
    assert st.blocks[0].cols.tolist() == [[0, 1], [6, 4], [3, 6]]
    assert st.blocks[1].cols.tolist() == [[2, 3], [0, 6]]
    vals = [st.get(b.val, params[0], b.m).tolist() for b in st.blocks]
    assert vals == [[1.0, 3.0, 9.0], [2.0, 8.0], [4.0], [5.0], [6.0], [7.0]]
    assert st.blocks[4].ipar[3] == 1 and st.blocks[0].ipar[3] == 0
    # the packed program is the three programs with re-offset row tables: it evaluates row by row like them
    prog = st.get(st.blocks[0].par, params[0], 3 + 2 * st.blocks[0].ipar[2])
    for r, names in enumerate(("ab", "ge", "dg")):
        xv = x0[0][st.blocks[0].cols[r]]
        assert sym.eval_program(prog, 3, x0[0][st.blocks[0].cols[r]])[r] == xv[0] * xv[0] + xv[1]
    # QUADFORM: P of every row first, then a of every row
    ntri = 3
    par = st.get(st.blocks[1].par, params[0], 2 * ntri + 4)
    assert par.tolist() == [1.0, 0.0, 1.0, 2.0, 0.0, 2.0, 1.0, 1.0, 0.0, 0.0]


def test_forty_step_constraints_fit_in_one_block_and_the_limit_counts_device_blocks():
    st = batch.compile_batch([BP.robot(0, T=40, K=3)])[0]
    assert [(b.family, b.m, b.n_in) for b in st.blocks] == [(FAM_VM, 120, 2)]
    assert st.blocks[0].cols.tolist() == [[2 * t, 2 * t + 1] for t in range(40) for _ in range(3)]
    st = batch.compile_batch([BP.circle(0, T=16, K=1)])[0]  # CIRCLE2D constraints are never packed
    assert len(st.blocks) == 16
    with pytest.raises(batch.UnsupportedProblem, match="17 device constraint blocks"):
        batch.compile_batch([BP.circle(0, T=17, K=1)])


def test_a_variable_that_repeats_a_scalar_is_refused():
    prob, ov = _small_prob()
    x = sym.variables(2)
    prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(E.SymExpr([x[0] - x[1]], 2), np.zeros((1, 1))), _var(ov, "ee")))
    with pytest.raises(batch.UnsupportedProblem, match="'e' more than once"):
        batch.compile_batch([prob])
    prob, ov = _small_prob()
    prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(E.SymExpr([x[0] - x[1]], 2), np.zeros((1, 1))), _var(ov, "abc")))
    with pytest.raises(batch.UnsupportedProblem, match="over 2 variables is bound to a Variable of 3"):
        batch.compile_batch([prob])


def test_maps_enter_the_batch_key_and_the_signature():
    a = batch.compile_problem(BP.qcqp(0))
    b = batch.compile_problem(BP.qcqp(1))  # other subsets per row
    assert batch.group_key(a) != batch.group_key(b)
    with pytest.raises(batch.UnsupportedProblem):
        batch.compile_batch(None, compiled=[a, b])
    sa = batch.compile_batch(None, compiled=[a])[0]
    sb = batch.compile_batch(None, compiled=[b])[0]
    assert batch.signature(sa) != batch.signature(sb)
    assert batch.group_key(a) == batch.group_key(batch.compile_problem(BP.qcqp(0)))


def test_batch_files_keep_the_maps(tmp_path):
    st, params, x0, _ = batch.compile_batch([BP.arm(0, T=4, per_step=True)])
    path = str(tmp_path / "arm.npz")
    batchfile.save_batch(path, st, params, x0)
    st2, p2, x2, meta = batchfile.load_batch(path)
    assert batch.signature(st2) == batch.signature(st)
    assert [b.cols.tolist() for b in st2.blocks] == [b.cols.tolist() for b in st.blocks]
    assert np.array_equal(p2, params) and np.array_equal(x2, x0)
    # a file of the version before maps existed still loads, with its own signature
    st3, p3, x3, meta3 = batchfile.load_batch(os.path.join(GOLDEN, "batch_parent_point_robot.npz"))
    assert meta3["signature"] == "0e3c9e6e21c4ebe24e9695141a47840cd0fad907e0ee862ac9321cf930666988"
    assert all(b.cols is None for b in st3.blocks)
    ref = W.gen_point_robot(2, T=4, K=2)
    assert batch.signature(st3) == batch.signature(ref[0]) and np.array_equal(p3, ref[1])


def test_ctypes_mirror_matches_the_header(tmp_path):
    from sco_py_b200 import _lib
    fields = {"sco_block_desc": _lib.CBlock, "sco_structure_desc": _lib.CStructure}
    lines = ['#include <stddef.h>', '#include <stdio.h>', '#include "sco_b200.h"', 'int main(void) {']
    for cname, ct in fields.items():
        lines.append('  printf("%s size %%zu\\n", sizeof(%s));' % (cname, cname))
        for f in ct._fields_:
            lines.append('  printf("%s %s %%zu\\n", offsetof(%s, %s));' % (cname, f[0], cname, f[0]))
    lines.append('  return 0;\n}\n')
    src = tmp_path / "off.c"
    src.write_text("\n".join(lines))
    exe = str(tmp_path / "off")
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe])
    out = subprocess.check_output([exe], text=True).split("\n")
    got = {tuple(l.split()[:2]): int(l.split()[2]) for l in out if l}
    for cname, ct in fields.items():
        assert got[(cname, "size")] == __import__("ctypes").sizeof(ct), cname
        for f in ct._fields_:
            assert got[(cname, f[0])] == getattr(ct, f[0]).offset, (cname, f[0])


@pytest.mark.parametrize("family", sorted(BP.BUILDERS))
@pytest.mark.parametrize("i", [0, 1])
def test_port_solves_bound_and_lifted_forms_alike(family, i):
    res = {}
    for form in BP.FORMS:
        st, params, x0, _ = batch.compile_batch([BP.BUILDERS[family](i, form=form)])
        assert all((b.cols is None) == (form == "lifted") for b in st.blocks)
        res[form] = bound_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    a, b = res["bound"], res["lifted"]
    assert a["success"] == b["success"]
    assert [a["stats"][k] for k in ("sqp_iters", "qp_solves")] == [b["stats"][k] for k in ("sqp_iters", "qp_solves")]
    assert np.abs(a["x"] - b["x"]).max() <= 1e-9


# ---------------------------------------------------------------------------------------------------- GPU
def _multi_fk7(B=3, seed=0):
    """Hand-built: one FK7 block of three instances (rows 3i..3i+2) with permuted maps, on 21 variables."""
    from sco_py_b200.families_host import fk7_table
    n = 21
    rng = np.random.default_rng(seed)
    cols = np.vstack([np.tile(rng.permutation(np.arange(7 * i, 7 * i + 7)), (3, 1)) for i in (2, 0, 1)]).astype(np.int32)
    blk = Block(FAM_FK7, 1, 9, Field(0, True), Field(0, False), ipar=[3, 0, 0, 0, 0, 0, 0, 0], jw=7, cols=cols)
    st = Structure(n=n, stride=9, Q=Field(-1, False), q=Field(-1, False), c=Field(-1, False), blocks=[blk],
                   shared=fk7_table())
    return st, rng.normal(0.0, 0.2, (B, 9)), rng.uniform(-1.0, 1.0, (B, n))


def _permuted_circle(i):
    """CircleDistExpr(3, K=2) bound to a Variable that lists the way-points in reverse step order."""
    prob, ov = _small_prob(names=tuple("abcdef"))
    var = _var(ov, "efcdab")
    prob.add_cnt_expr(E.BoundExpr(E.LEqExpr(E.CircleDistExpr(3, [[0.2, 0.1], [0.5, 0.4]], [0.3, 0.6 + 0.1 * i]),
                                            np.zeros((6, 1))), var))
    return prob


def _convexify_cases():
    return {
        "vm_fd": lambda i: BP.robot(i, T=6, K=2),
        "vm_analytic": lambda i: BP.robot(i, T=6, K=2, analytic=True),
        "quadform": lambda i: BP.qcqp(i, n=10, m=8, k=4, sel_seed=5),
        "circle2d_steps": lambda i: BP.circle(i, T=5, K=2),
        "circle2d_permuted": _permuted_circle,
        "fk7_steps": lambda i: BP.arm(i, T=4, per_step=True),
    }


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(_convexify_cases()) + ["fk7_instances"])
def test_convexify_stage_through_maps_matches_the_port(case):
    from sco_py_b200.engine import Engine
    if case == "fk7_instances":
        st, params, x = _multi_fk7()
    else:
        st, params, x0, _ = batch.compile_batch([_convexify_cases()[case](i) for i in range(4)])
        x = x0 + np.random.default_rng(3).normal(0.0, 0.3, x0.shape)
    assert all(b.cols is not None for b in st.blocks)
    eng = Engine(st)
    f, J, b, _ = [t.cpu().numpy() for t in eng.convexify(params, x)]
    fd = any(blk.family == FAM_FK7 or (blk.family == FAM_VM and not blk.ipar[3]) for blk in st.blocks)
    with bound_port.mapped_port():
        for i in range(x.shape[0]):
            pp = sqp_port.PortProblem(st, params[i], x[i])
            Js = helpers.split_J(st, J[i])
            bs = helpers.split_b(st, b[i])
            r0 = 0
            for bi, (blk, fn) in enumerate(zip(st.blocks, pp.blocks)):
                fr = fn.f(pp.x)[:, 0]
                Jr = fn.grad(pp.x)
                np.testing.assert_allclose(f[i, r0:r0 + blk.m], fr, rtol=1e-9, atol=1e-9)
                tol = 1e-7 if fd else 1e-9
                np.testing.assert_allclose(Js[bi], Jr, rtol=tol, atol=tol)
                np.testing.assert_allclose(bs[bi], fr - Jr @ x[i] - fn.val[:, 0], rtol=tol, atol=tol * 10)
                r0 += blk.m
    eng.close()


def _fast_ok(st):
    """The thread-per-entity ADMM loop's condition (sco_create): rows of <= 8 entries, columns with <= 4 linear and
    <= 4 penalty entries."""
    rows_ok = all(b.jw <= 8 for b in st.blocks)
    pen = np.zeros(st.n, int)
    for bi in range(len(st.blocks)):
        np.add.at(pen, st.jac_cols(bi).ravel(), 1)
    lin = np.bincount(np.asarray(st.lin_col if st.m_lin else [], dtype=int), minlength=st.n)
    lin_rows = np.diff(st.lin_rowptr) if st.m_lin else np.zeros(0)
    return rows_ok and (lin_rows <= 8).all() and (pen <= 4).all() and (lin <= 4).all()


@pytest.mark.gpu
@pytest.mark.parametrize("case,fast", [("robot", True), ("qcqp_wide", False)])
def test_qp_stage_through_maps_matches_osqp(case, fast):
    from sco_py_b200.engine import Engine, make_settings
    probs = ([BP.robot(i, T=10, K=2) for i in range(4)] if case == "robot" else
             [BP.qcqp(i, n=12, m=10, k=9, sel_seed=5) for i in range(4)])
    st, params, x0, _ = batch.compile_batch(probs)
    assert _fast_ok(st) == fast
    eng = Engine(st)
    ent = sum(-(-k // 32) * 32 for k in (st.n, st.m_lin, st.m_nl))
    assert eng.team == next(t for t in (32, 64, 128, 256, 512) if t >= ent)  # one thread per variable / row
    B = x0.shape[0]
    _, J, b, _ = eng.convexify(params, x0)
    Jn, bn = J.cpu().numpy(), b.cpu().numpy()
    rng = np.random.default_rng(11)
    for masks in ("random", "on"):
        bits = None
        if masks == "random":
            keep = rng.random((B, st.m_nl, 32)) > 1.0 / 3.0
            keep[:, :, max(blk.jw for blk in st.blocks):] = False
            bits = (keep * (1 << np.arange(32, dtype=np.uint64))).sum(axis=2).astype(np.uint32)[:, :, None]
        for pi, kdup, delta in ((10.0, 1, 0.5), (1e3, 2, 0.1)):
            lbx, ubx = x0 - delta, x0 + delta
            xq, status, iters = eng.qp_solve(params, make_settings(solver=W.SOLVER_SETTINGS), J=J, b=b, lbx=lbx,
                                             ubx=ubx, pi=np.full(B, pi), kdup=np.full(B, kdup, np.int32),
                                             mask=None if bits is None else bits.view(np.int32))
            xq, status, iters = xq.cpu().numpy(), status.cpu().numpy(), iters.cpu().numpy()
            with bound_port.mapped_port():
                for i in range(B):
                    qp = helpers.stage_qp(st, params[i], Jn[i], bn[i], lbx[i], ubx[i], pi, kdup,
                                          bits=None if bits is None else bits[i])
                    res = helpers.oracle_qp(*qp)
                    info = (case, masks, pi, i, int(status[i]), int(iters[i]), res.info.status_val, res.info.iter)
                    assert status[i] == res.info.status_val and iters[i] == res.info.iter, info
                    if res.info.status_val in (1, 2, -2):
                        assert np.abs(xq[i] - res.x).max() <= 1e-7 * max(1.0, np.abs(res.x).max()), info
    eng.close()


def _full_case(name):
    if name == "robot_fd":
        return [BP.robot(i, T=10, K=2) for i in range(12)]
    if name == "robot_analytic":
        return [BP.robot(i, T=10, K=2, analytic=True) for i in range(12)]
    return [BP.arm(i, T=4, per_step=True) for i in range(6)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["robot_fd", "robot_analytic", "arm_steps"])
def test_full_solves_through_maps_match_the_port(name):
    from sco_py_b200.engine import Engine, make_settings
    st, params, x0, _ = batch.compile_batch(_full_case(name))
    eng = Engine(st)
    out = eng.solve_batch_host(params, x0, make_settings(solver=W.SOLVER_SETTINGS))
    for i in range(x0.shape[0]):
        ref = bound_port.solve(st, params[i], x0[i], solver=W.SOLVER_SETTINGS)
        info = (name, i, int(out["verdict"][i]), ref["success"], out["stats"][i].tolist(), ref["stats"])
        assert (out["verdict"][i] == 1) == ref["success"], info
        assert abs(out["max_vio"][i] - ref["max_vio"]) <= 1e-5, info
        assert abs(out["objective"][i] - ref["objective"]) <= 1e-5 * max(1.0, abs(ref["objective"])), info
        assert np.abs(out["x"][i] - ref["x"]).max() <= 1e-4 * max(1.0, np.abs(ref["x"]).max()), info
    eng.close()


@pytest.mark.gpu
def test_solver_and_prob_entry_points_with_maps():
    # Solver.solve_batch: two structures with maps in one call (bucketed), results written into the Variables
    probs = [BP.robot(i, T=6, K=2) for i in range(3)] + [BP.qcqp(i) for i in range(2)]
    inputs = [batch.compile_batch([p])[:3] for p in probs]  # before the solve writes the solutions into the Variables
    oks = Solver().solve_batch(probs, method="penalty_sqp")
    for p, ok, (st, params, x0) in zip(probs, oks, inputs):
        ref = bound_port.solve(st, params[0], x0[0])  # Solver() and the port both default to solver.py:17-28
        assert ok == ref["success"]
        assert np.abs(batch.compile_batch([p])[2][0] - ref["x"]).max() <= 1e-4 * max(1.0, np.abs(ref["x"]).max())
    # the Prob step methods against the port's first two SQP iterations
    prob = BP.robot(4, T=6, K=2)
    st, params, x0, cps = batch.compile_batch([BP.robot(4, T=6, K=2)])
    allv = prob._vars[0]
    mu, delta = 3.0, 0.5
    with bound_port.mapped_port():
        pp = sqp_port.PortProblem(st, params[0], x0[0])
        assert abs(prob.get_value(mu) - pp.get_value(mu)) <= 1e-9 * max(1.0, abs(pp.get_value(mu)))
        for it in range(2):
            prob.convexify()
            prob.update_obj(mu)
            prob.save()
            prob.add_trust_region(delta)
            pp.convexify()
            pp.update_obj(mu)
            xs = pp.x[:, 0].copy()
            ok_ref = pp.solve_qp(xs - delta, xs + delta, True, sqp_port.DEFAULT_OSQP)
            assert prob.optimize() == ok_ref
            assert np.abs(allv.get_value()[:, 0] - pp.x[:, 0]).max() <= 1e-6
            assert abs(prob.get_approx_value(mu) - pp.get_approx_value(mu)) <= 1e-6 * max(1.0, abs(pp.get_approx_value(mu)))
            assert abs(prob.get_value(mu) - pp.get_value(mu)) <= 1e-6 * max(1.0, abs(pp.get_value(mu)))


def _grouped_robot(i):
    """Per-step obstacle SymExprs in groups spread over the steps: even steps in "a", odd ones in "a" and "b", the
    first half of the trajectory also in "c" (four packed blocks)."""
    return BP.robot(i, T=8, K=2, groups=lambda t: (["a"] if t % 2 == 0 else ["a", "b"]) + (["c"] if t < 4 else []))


@pytest.mark.gpu
def test_nonconverged_groups_across_packed_rows():
    probs = [_grouped_robot(i) for i in range(8)]
    st, params, x0, cps = batch.compile_batch(probs)
    assert len(st.blocks) == 4 and st.n_groups == 3
    solver = Solver()
    solver.solve_batch(probs, method="penalty_sqp")
    for i, p in enumerate(probs):
        ref = bound_port.solve(st, params[i], x0[i])  # Solver() and the port both default to solver.py:17-28
        assert [cps[i].gids[g] for g in ref["nonconverged"]] == p.nonconverged_groups, i


@pytest.mark.gpu
@pytest.mark.parametrize("bad", ["out_of_range", "negative", "repeat", "n_in_circle", "n_in_fk7", "fk7_rows",
                                 "fk7_m"])
def test_bad_maps_are_refused(bad):
    from sco_py_b200.engine import Engine
    if "fk7" in bad:
        st = _multi_fk7()[0]
    else:
        st = batch.compile_batch([_permuted_circle(0) if bad == "n_in_circle" else BP.robot(0, T=4, K=2)])[0]
    blk = st.blocks[0]
    cols = blk.cols.copy()
    if bad == "out_of_range":
        cols[1, 0] = st.n
    elif bad == "negative":
        cols[0, 1] = -1
    elif bad == "repeat":
        cols[2, 1] = cols[2, 0]
    elif bad == "n_in_circle":
        cols = np.hstack([cols, cols[:, :1]])
    elif bad == "n_in_fk7":
        cols = cols[:, :6]
    elif bad == "fk7_rows":
        cols[4] = cols[4][::-1]
    else:
        cols, blk.m, blk.val = cols[:8], 8, Field(0, False)
    blk.cols = np.ascontiguousarray(cols, dtype=np.int32)
    with pytest.raises(RuntimeError) as e:
        Engine(st)
    msg = str(e.value)
    assert msg.startswith("sco_b200 error -1: ")
    want = {"out_of_range": "outside", "negative": "outside", "repeat": "repeats", "n_in_circle": "n_in",
            "n_in_fk7": "n_in = 6", "fk7_rows": "different maps", "fk7_m": "m % 3"}[bad]
    assert want in msg, msg
