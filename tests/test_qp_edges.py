"""The penalty QP at every machine mapping of its ADMM loop, at every fill of the dense loops' compile-time bounds and
through the loops' rare exits, against the OSQP oracle.

sco_create (sco_abi.cu) routes a QCQP of n variables and m hinge rows to
  * the two-warp dense loop of the first kind in KINDS whose bounds (NP, MP) hold it (sco_dense.cuh,
    dense_qp_solve<NP, MP>).  Below the bounds, variable lanes n <= j < NP and row lanes m <= i < MP are padding and
    must not reach a norm, a sum or the cost scaling;
  * the thread-per-entity loop with dense penalty rows (sco_qp.cuh: fast_role<ROLE, 1>) up to n = 32, m = 48;
  * the strided shared-memory loop (generic_loop) beyond that, and for every structure under force_generic = 1.
The point robot (sparse rows, linear equality rows) runs the thread-per-entity loop, the 7-DOF arm the same loop on a
512-thread team.

Bars of test_gpu_parity.test_qp_stage_matches_oracle: identical status, identical ADMM iteration count, and
|dx| <= 1e-7 max(1, |x|) where the status carries a solution.  The rare exits are the end of max_iter (an exact
re-test when the last iteration was not tested, then the x10-tolerance test: status 2 / -2), termination test
intervals other than 25, the infeasibility certificates (-3 / -4, and 3 / 4 under the x10 tolerances), box rows with
infinite bounds (rho = RHO_MIN) and with equal bounds (rho x 1e3).
"""
import os
import re

import numpy as np
import pytest

import helpers
import sqp_port
from sco_py_b200 import workloads as W

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "sco_py_b200", "csrc")

KINDS = ((8, 6), (12, 16), (20, 30), (32, 32))  # (NP, MP) of dense kinds 1..4
SHAPES = {  # loop -> QCQP shapes (n, m) it solves: per dense kind full fill, one below both bounds, lopsided
    "dense1": [(8, 6), (7, 5), (1, 1), (8, 1)],
    "dense2": [(12, 16), (9, 7), (3, 16)],
    "dense3": [(20, 30), (13, 17), (2, 29), (20, 17)],
    "dense4": [(32, 32), (31, 31), (2, 31), (31, 2)],
    "entity": [(32, 33), (32, 48), (5, 40)],
    "strided": [(32, 49), (33, 6)],
}
ALL_SHAPES = [(loop, s) for loop, shapes in SHAPES.items() for s in shapes]
DENSE_SHAPES = [(loop, s) for loop, s in ALL_SHAPES if loop.startswith("dense")]
STAGE_B = 3  # problems per shape in the stage tests
STAGE_SETTINGS = [(1, 1.0, 1.0), (3, 10.0, 0.1), (7, 1000.0, 2e-5)]  # (kdup, pi, delta) of test_gpu_parity


def route(n, m):
    """The loop sco_create gives a QCQP.  Its dense rows (n entries each; with m > 32 more than four entries in every
    column) never fit the sparse thread-per-entity loop."""
    for k, (NP, MP) in enumerate(KINDS):
        if n <= NP and m <= MP:
            return "dense%d" % (k + 1)
    return "entity" if n <= 32 and m <= 48 else "strided"


def _shape_id(v):
    return "%dx%d" % v if isinstance(v, tuple) else str(v)


def test_routing_table_matches_the_sources():
    """The kind table of sco_create, the instantiations of QPSolver::solve and the build's kind list are the ones this
    file covers, and every shape above lands in the loop it is listed under."""
    abi = open(os.path.join(CSRC, "sco_abi.cu")).read()
    table = re.search(r"static const int table\[\]\[2\]\s*=\s*\{(.*?)\};", abi, re.S)
    assert table, "dense kind table not found in sco_abi.cu"
    assert tuple((int(a), int(b)) for a, b in re.findall(r"\{\s*(\d+)\s*,\s*(\d+)\s*\}", table.group(1))) == KINDS
    assert re.search(r"desc->m_lin == 0 && n <= 32 && m_nl > 0 && m_nl <= 48;", abi), "thread-per-entity dense bounds"
    qp = open(os.path.join(CSRC, "sco_qp.cuh")).read()
    solve = qp[qp.index("QPResult solve()"):]
    solve = solve[:solve.index("load_and_scale")]
    inst = re.findall(r"(?:DK == (\d+)\)|else) return dense_qp_solve<\s*(\d+)\s*,\s*(\d+)\s*>", solve)
    assert [(int(k or len(KINDS)), int(a), int(b)) for k, a, b in inst] == [(k + 1,) + s for k, s in enumerate(KINDS)]
    from sco_py_b200 import build
    assert tuple(build.DENSE_KINDS) == tuple(range(1, len(KINDS) + 1))
    for loop, shapes in SHAPES.items():
        for n, m in shapes:
            assert route(n, m) == loop, (n, m, loop)
    for k, (NP, MP) in enumerate(KINDS):
        mine = SHAPES["dense%d" % (k + 1)]
        assert (NP, MP) in mine and any(n < NP and m < MP for n, m in mine)
        assert any(n <= NP // 4 or m <= MP // 4 for n, m in mine)  # lopsided


# ------------------------------------------------------------------ device side
def _settings(**kw):
    from sco_py_b200.engine import make_settings
    return make_settings(solver=W.SOLVER_SETTINGS, **kw)


def _oracle_kw(kw):
    """CSettings field names -> oracle_qp keywords."""
    return {k[len("osqp_"):]: v for k, v in kw.items() if k.startswith("osqp_")}


def _gen(key, B):
    if key[0] == "qcqp":
        return W.gen_qcqp(B, n=key[1], m=key[2])
    if key[0] == "point_robot":
        return W.gen_point_robot(B, T=20, K=1)
    return W.gen_arm(B, T=20)


@pytest.fixture(scope="module")
def engine():
    """key -> (Engine, structure, params, x0) of STAGE_B problems, created once per module."""
    from sco_py_b200.engine import Engine
    cache = {}

    def get(key):
        if key not in cache:
            st, params, x0 = _gen(key, STAGE_B)
            cache[key] = (Engine(st), st, params, x0)
        return cache[key]
    yield get
    for e in cache.values():
        e[0].close()


def _bits(eng, st, B, rng, off_rows=None):
    """Mask words (B, m_nl, words): a third of the stored slots off at random, or every slot on but the rows
    `off_rows[i]` of problem i entirely off."""
    m, jw, words = st.m_nl, st.blocks[0].jw, eng.mask_words
    if off_rows is None:
        keep = rng.random((B, m, 32 * words)) > 1.0 / 3.0
    else:
        keep = np.ones((B, m, 32 * words), dtype=bool)
        for i, r in enumerate(off_rows):
            keep[i, r] = False
    keep[:, :, jw:] = False
    w = (keep.reshape(B, m, words, 32) * (1 << np.arange(32, dtype=np.uint64))).sum(axis=3)
    return w.astype(np.uint32)


def _stage(eng, params, J, b, lbx, ubx, pi, kdup, bits=None, **kw):
    """Device penalty QPs, one per problem -> host (x, status, iters)."""
    B = params.shape[0]
    xq, status, iters = eng.qp_solve(params, _settings(**kw), J=J, b=b, lbx=lbx, ubx=ubx, pi=np.full(B, float(pi)),
                                     kdup=np.full(B, kdup, np.int32),
                                     mask=None if bits is None else np.ascontiguousarray(bits).view(np.int32))
    return xq.cpu().numpy(), status.cpu().numpy(), iters.cpu().numpy()


def _closest(eng, params, x0, lbx=None, ubx=None, **kw):
    xq, status, iters = eng.qp_solve(params, _settings(**kw), xref=x0, lbx=lbx, ubx=ubx, use_penalty=False,
                                     closest_point=True)
    return xq.cpu().numpy(), status.cpu().numpy(), iters.cpu().numpy()


def _match(got, qps, where, **oracle_kw):
    """Device results against the oracle on the expanded QPs -> the oracle statuses."""
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


def _same(a, b, where):
    """Two loops on the same QPs: same status, same iteration count, x to 1e-9 where there is a solution."""
    assert np.array_equal(a[1], b[1]), (where, a[1], b[1])
    assert np.array_equal(a[2], b[2]), (where, a[2], b[2])
    sol = np.isin(a[1], (1, 2, -2))
    assert np.abs(a[0][sol] - b[0][sol]).max(initial=0.0) <= 1e-9, where


def _penalty_qps(st, params, Jn, bn, lbx, ubx, pi, kdup, bits=None):
    return [helpers.stage_qp(st, params[i], Jn[i], bn[i], lbx[i], ubx[i], pi, kdup,
                             bits=None if bits is None else bits[i]) for i in range(params.shape[0])]


def _closest_qps(st, params, x0, lbx=None, ubx=None):
    inf = np.full(st.n, np.inf)
    return [helpers.expand_qp(st, params[i], [], [], [], -inf if lbx is None else lbx[i],
                              inf if ubx is None else ubx[i], 0.0, 0, closest_xref=x0[i], use_penalty=False)
            for i in range(params.shape[0])]


@pytest.mark.gpu
@pytest.mark.parametrize("loop,shape", ALL_SHAPES, ids=[l + "-" + _shape_id(s) for l, s in ALL_SHAPES])
def test_qp_stage_matches_oracle_at_every_fill(engine, loop, shape):
    """Random and all-on masks at the three (kdup, pi, delta) settings of test_gpu_parity, whole rows switched off
    (a zero row norm in the Ruiz passes), a non-symmetric Q (both sides solve with (Q + Q') / 2), pi at 1e-3 and 1e8,
    and the closest-point projection.  The dense kinds also against the strided loop on the same QPs."""
    eng, st, params, x0 = engine(("qcqp",) + shape)
    assert (eng.team == 64) == loop.startswith("dense")
    B, n, m = params.shape[0], shape[0], shape[1]
    f, J, b, _ = eng.convexify(params, x0)
    Jn, bn = J.cpu().numpy(), b.cpu().numpy()
    rng = np.random.default_rng(1000 * n + m)
    cases = []
    for kdup, pi, delta in STAGE_SETTINGS:
        cases.append(("kdup%d/all" % kdup, params, kdup, pi, delta, None))
        cases.append(("kdup%d/masked" % kdup, params, kdup, pi, delta, _bits(eng, st, B, rng)))
    cases.append(("row-off", params, 2, 10.0, 0.5, _bits(eng, st, B, rng, off_rows=[0, m - 1, m // 2][:B])))
    skew = params.copy()
    R = rng.standard_normal((B, n, n))
    skew[:, st.Q.off:st.Q.off + n * n] += (R - np.transpose(R, (0, 2, 1))).reshape(B, -1)
    cases.append(("nonsymmetric-Q", skew, 2, 10.0, 0.5, None))
    cases.append(("pi=1e-3", params, 2, 1e-3, 0.5, None))
    cases.append(("pi=1e8", params, 2, 1e8, 0.5, _bits(eng, st, B, rng)))
    for label, prm, kdup, pi, delta, bits in cases:
        lbx, ubx = x0 - delta, x0 + delta
        got = _stage(eng, prm, J, b, lbx, ubx, pi, kdup, bits)
        _match(got, _penalty_qps(st, prm, Jn, bn, lbx, ubx, pi, kdup, bits), (loop, shape, label))
        if loop.startswith("dense"):
            _same(got, _stage(eng, prm, J, b, lbx, ubx, pi, kdup, bits, force_generic=1), (loop, shape, label))
    _match(_closest(eng, params, x0), _closest_qps(st, params, x0), (loop, shape, "closest-point"))


# ------------------------------------------------------------------ rare exits
# (loop, structure, force_generic): each dense kind full and padded, the thread-per-entity loop with dense rows and
# with sparse and linear rows, the strided loop on its own shapes and under force_generic
EXIT_CASES = ([("dense%d" % (k + 1), ("qcqp",) + s, 0) for k in range(len(KINDS)) for s in SHAPES["dense%d" % (k + 1)][:2]]
              + [("entity", ("qcqp", 32, 48), 0), ("entity", ("qcqp", 5, 40), 0), ("entity", ("point_robot",), 0),
                 ("entity", ("arm",), 0),
                 ("strided", ("qcqp", 33, 6), 0), ("strided", ("qcqp", 32, 49), 0), ("strided", ("qcqp", 8, 6), 1),
                 ("strided", ("qcqp", 20, 30), 1), ("strided", ("qcqp", 32, 48), 1), ("strided", ("point_robot",), 1),
                 ("strided", ("arm",), 1)])
EXITS = ["max_iter", "check_termination", "scaling", "mixed_box", "dual_infeasible", "primal_infeasible"]


def _exit_params():
    out = []
    for loop, key, gen in EXIT_CASES:
        for ex in EXITS:
            if ex == "dual_infeasible" and key[0] != "qcqp":
                continue  # the shared objective of the point robot and the arm is bounded below on its pinned rows
            if ex == "primal_infeasible" and key[0] == "qcqp":
                continue  # a penalty QP over hinge rows and a box alone is always feasible
            out.append(pytest.param(loop, key, gen, ex, id="%s-%s%s-%s" % (
                loop, "x".join(str(v) for v in key), "-generic" if gen else "", ex)))
    return out


def _caps(qp, ct=25):
    """max_iter caps, chosen by asking the oracle, at which it ends in -2, 2 and 1: per (status, cap is a multiple of
    the test interval) the last cap found for -2 and the first for the others, from a scan below the iteration at
    which the QP converges."""
    k = helpers.oracle_qp(*qp).info.iter
    found = {}
    for c in sorted(set(c for j in range(1, k // ct + 2) for c in (ct * j - 13, ct * j - 1, ct * j) if c > 0)):
        s = helpers.oracle_qp(*qp, max_iter=c).info.status_val
        if s == -2:
            found[(s, c % ct == 0)] = c
        else:
            found.setdefault((s, c % ct == 0), c)
    return found


def _pin_row(st, row, x0):
    """(column, value) of a linear equality row that pins one variable."""
    pp = sqp_port.PortProblem(st, row, x0)
    A = pp.A_lin.toarray()
    for r in range(A.shape[0]):
        (cols,) = np.nonzero(A[r])
        if len(cols) == 1 and pp.l_lin[r] == pp.u_lin[r]:
            return int(cols[0]), pp.l_lin[r] / A[r, cols[0]]
    raise AssertionError("no pinned variable")


@pytest.mark.gpu
@pytest.mark.parametrize("loop,key,generic,exit_", _exit_params())
def test_rare_exits_match_oracle(engine, loop, key, generic, exit_):
    eng, st, params, x0 = engine(key)
    B, n = params.shape[0], st.n
    f, J, b, _ = eng.convexify(params, x0)
    Jn, bn = J.cpu().numpy(), b.cpu().numpy()
    where = (loop, key, generic, exit_)
    kw0 = dict(force_generic=generic)
    lbx, ubx = x0 - 1.0, x0 + 1.0
    runs = []  # (label, settings, penalty QP args or None for the closest-point QP, lbx, ubx, params, bits)
    if exit_ == "max_iter":
        found = _caps(_penalty_qps(st, params[:1], Jn[:1], bn[:1], lbx[:1], ubx[:1], 10.0, 2)[0])
        caps = sorted(set(found.values()))
        assert {s for s, _ in found} >= {-2, 2, 1}, found
        assert any(c % 25 == 0 for c in caps) and any(c % 25 for c in caps), found
        runs += [("cap%d" % c, dict(osqp_max_iter=c), params, lbx, ubx, None) for c in caps]
    elif exit_ == "check_termination":
        runs += [("ct0", dict(osqp_check_termination=0, osqp_max_iter=3000), params, lbx, ubx, None),
                 ("ct1", dict(osqp_check_termination=1), params, lbx, ubx, None),
                 ("ct7", dict(osqp_check_termination=7), params, lbx, ubx, None)]
    elif exit_ == "scaling":
        runs += [("scaling%d" % s, dict(osqp_scaling=s), params, lbx, ubx, None) for s in (0, 1)]
    elif exit_ == "mixed_box":  # equal bounds on every other variable, infinite ones on every fourth
        lo, hi = x0 - 0.5, x0 + 0.5
        lo[:, ::2] = hi[:, ::2] = x0[:, ::2]
        lo[:, 1::4], hi[:, 1::4] = -np.inf, np.inf
        runs += [("mixed-box", {}, params, lo, hi, None), ("mixed-box-ct1", dict(osqp_check_termination=1), params,
                                                            lo, hi, None)]
    elif exit_ == "dual_infeasible":  # no quadratic term, every Jacobian slot masked off, no box
        flat = params.copy()
        flat[:, st.Q.off:st.Q.off + n * n] = 0.0
        bits = np.zeros((B, st.m_nl, eng.mask_words), np.uint32)
        inf = np.full((B, n), np.inf)
        runs += [("dinf", {}, flat, -inf, inf, bits)]
        runs += [("dinf-cap%d" % c, dict(osqp_max_iter=c), flat, -inf, inf, bits) for c in (1, 10, 24)]
        runs += [("dinf-ct7", dict(osqp_check_termination=7), flat, -inf, inf, bits)]
    else:  # primal infeasible: the box of a pinned variable excludes its pinned value
        lo, hi = np.full((B, n), -np.inf), np.full((B, n), np.inf)
        for i in range(B):
            j, v = _pin_row(st, params[i], x0[i])
            lo[i, j], hi[i, j] = v + 1.0, v + 2.0
        runs += [("pinf-closest", {}, None, lo, hi, None), ("pinf-closest-cap30", dict(osqp_max_iter=30), None, lo, hi,
                                                            None)]
        lp, hp = lbx.copy(), ubx.copy()
        lp[lo > -np.inf], hp[hi < np.inf] = lo[lo > -np.inf], hi[hi < np.inf]
        runs += [("pinf-penalty", {}, params, lp, hp, None)]
    seen = set()
    for label, kw, prm, lo, hi, bits in runs:
        s = dict(kw0, **kw)
        if prm is None:
            seen |= set(_match(_closest(eng, params, x0, lo, hi, **s), _closest_qps(st, params, x0, lo, hi),
                               where + (label,), **_oracle_kw(s)))
        else:
            seen |= set(_match(_stage(eng, prm, J, b, lo, hi, 10.0, 2, bits, **s),
                               _penalty_qps(st, prm, Jn, bn, lo, hi, 10.0, 2, bits), where + (label,),
                               **_oracle_kw(s)))
    print("oracle statuses %s: %s" % ("/".join(map(str, where)), sorted(seen)))
    want = {"max_iter": {-2, 2, 1}, "dual_infeasible": {-4}, "primal_infeasible": {-3}}.get(exit_, set())
    assert seen >= want, (where, seen)


# ------------------------------------------------------------------ full solves and the non-tail regime
FULL_B = {"dense1": 8, "dense2": 8, "dense3": 6, "dense4": 2}  # the port needs up to minutes for one 20 x 17 or 32 x 32 problem
CAP_SHAPES = [(8, 6), (12, 16), (31, 2)]


def _full_solve_check(st, out, refs, where):
    x, verdict = out["x"].cpu().numpy(), out["verdict"].cpu().numpy()
    vio, obj, stats = out["max_vio"].cpu().numpy(), out["objective"].cpu().numpy(), out["stats"].cpu().numpy()
    for i, ref in refs.items():
        info = (where, i, stats[i].tolist(), ref["stats"])
        assert (verdict[i] == 1) == ref["success"], info
        assert abs(vio[i] - ref["max_vio"]) <= 1e-5, info
        assert np.abs(x[i] - ref["x"]).max() <= 1e-4 * max(1.0, np.abs(ref["x"]).max()), info
        assert abs(obj[i] - ref["objective"]) <= 1e-5 * max(1.0, abs(ref["objective"])), info
        # no finite differences, no sin / cos: the same SQP trajectory, QP by QP
        assert stats[i][:3].tolist() == [ref["stats"]["sqp_iters"], ref["stats"]["qp_solves"],
                                         ref["stats"]["admm_iters"]], info


@pytest.mark.gpu
@pytest.mark.parametrize("loop,shape", DENSE_SHAPES, ids=[l + "-" + _shape_id(s) for l, s in DENSE_SHAPES])
def test_full_solve_matches_port_at_every_fill(loop, shape):
    from sco_py_b200.engine import Engine
    n, m = shape
    st, params, x0 = W.gen_qcqp(FULL_B[loop], n=n, m=m)
    eng = Engine(st)
    out = eng.solve_batch(params, x0, _settings())
    eng.close()
    refs = helpers.port_solve_many("qcqp", range(x0.shape[0]), W.SOLVER_SETTINGS, gen_kw=dict(n=n, m=m))
    _full_solve_check(st, out, refs, (loop, shape))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", CAP_SHAPES, ids=[_shape_id(s) for s in CAP_SHAPES])
def test_full_solve_with_a_small_osqp_cap_matches_port(shape):
    """QPs that stop at max_iter inside the SQP: the status gate of the reference (only solved / solved-inaccurate QPs
    are accepted) and quirk C-5; the cap is one at which the sample has both verdicts."""
    from sco_py_b200.engine import Engine
    n, m = shape
    st, params, x0 = W.gen_qcqp(8, n=n, m=m)
    for cap in (30, 60, 100, 200):
        refs = helpers.port_solve_many("qcqp", range(8), W.SOLVER_SETTINGS, gen_kw=dict(n=n, m=m),
                                       osqp_kw={"max_iter": cap})
        if len(set(r["success"] for r in refs.values())) == 2:
            break
    else:
        raise AssertionError("no cap gives both verdicts")
    eng = Engine(st)
    out = eng.solve_batch(params, x0, _settings(osqp_max_iter=cap))
    eng.close()
    _full_solve_check(st, out, refs, (shape, cap))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", range(1, len(KINDS) + 1))
def test_dense_kinds_give_the_same_results_on_a_full_machine(kind):
    """With twice as many problems as resident teams the dense loop tests termination without the tail-mode
    refutation terms; the first 32 problems alone run in tail mode.  Both must return the same bits."""
    import torch
    from sco_py_b200.engine import Engine
    n, m = KINDS[kind - 1]
    st = W.qcqp_structure(n, m)
    eng = Engine(st)
    B = 2 * torch.cuda.get_device_properties(eng.device).multi_processor_count * eng.occupancy
    _, params, x0 = W.gen_batch("qcqp", B, n=n, m=m)
    full = eng.solve_batch(params, x0, _settings())
    alone = eng.solve_batch(params[:32], x0[:32], _settings())
    for k in ("x", "verdict", "stats", "max_vio", "objective"):
        assert np.array_equal(full[k][:32].cpu().numpy(), alone[k].cpu().numpy()), (kind, B, k)
    assert (full["verdict"].cpu().numpy() == 1).mean() > 0.5
    eng.close()
