"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same inputs.

Tolerances (float64 path, BASELINE.json north_star: 1e-4 relative on the solution, 1e-5 absolute
on violation, same verdict):
  * expression values / Jacobians / affine offsets: 1e-9 (analytic), 1e-7 (finite-difference FK)
  * one QP (same scaling, same ADMM iteration, different linear algebra): |dx| <= 1e-7 * max(1,|x|),
    identical status, identical iteration count
  * full penalty-SQP solve: identical verdict, |d max_vio| <= 1e-5, objective within 1e-5 relative
    (1e-4 for the arm) and |dx| <= 1e-4 * max(1,|x|) for all three configurations.  Round 1 needed 2e-3 for the
    arm and blamed sin / cos; the cause was the forward kinematics itself: the oracle summed its 3-vector products
    in BLAS order, the kernel with contracted FMAs, ~10 ulp apart -- and profiles/arm_sensitivity.py shows that
    10 ulp in f (not 1) make the SQP of an occasional arm problem stop one iteration earlier or later.  Both sides
    now evaluate the chain in one fixed order (oracle/families.py:fk7_pos, sco_families.cuh:fk7_pos) and differ
    only through sin / cos: 64 arm problems agree to 1e-8 (bench.py detail.other_configs.arm.audit)
"""
import os
import numpy as np
import pytest

import helpers
import sqp_port
from sco_py_b200 import workloads as W

pytestmark = pytest.mark.gpu

CONFIGS = [("qcqp", 64), ("point_robot", 16), ("arm", 16)]   # full solves (the oracle runs on every host core)
STAGE_N = {"qcqp": 8, "point_robot": 4, "arm": 4}            # problems of the batch used by the stage-level tests
X_TOL = {"qcqp": 1e-4, "point_robot": 1e-4, "arm": 1e-4}
OBJ_TOL = {"qcqp": 1e-5, "point_robot": 1e-5, "arm": 1e-4}
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def engines():
    import torch
    from sco_py_b200.engine import Engine
    assert torch.cuda.is_available()
    out = {}
    for name, B in CONFIGS:
        st, params, x0 = W.GENERATORS[name](B)
        out[name] = (Engine(st), st, params, x0)
    yield out
    for e in out.values():
        e[0].close()


def _settings(**kw):
    from sco_py_b200.engine import make_settings
    return make_settings(solver=W.SOLVER_SETTINGS, **kw)


@pytest.mark.parametrize("name", [c[0] for c in CONFIGS])
def test_convexify_matches_oracle(engines, name):
    eng, st, params, x0 = engines[name]
    f, J, b, obj = [t.cpu().numpy() for t in eng.convexify(params, x0)]
    tol = 1e-7 if name == "arm" else 1e-9
    for i in range(min(x0.shape[0], 2 * STAGE_N[name])):
        pp = sqp_port.PortProblem(st, params[i], x0[i])
        pp.convexify()
        Jd = helpers.split_J(st, J[i])
        r0 = 0
        for bi, blk in enumerate(st.blocks):
            fo = pp.blocks[bi].f(pp.x)[:, 0]
            np.testing.assert_allclose(f[i, r0:r0 + blk.m], fo, rtol=1e-12, atol=1e-12)
            np.testing.assert_allclose(Jd[bi], pp.J[bi], rtol=tol, atol=tol)
            np.testing.assert_allclose(b[i, r0:r0 + blk.m], pp.b[bi][:, 0], rtol=tol, atol=tol * 10)
            r0 += blk.m
        assert abs(obj[i] - pp.objective(pp.x)) <= 1e-10 * max(1.0, abs(obj[i]))


@pytest.mark.parametrize("name", [c[0] for c in CONFIGS])
@pytest.mark.parametrize("kdup,pi,delta,masked", [(1, 1.0, 1.0, False), (3, 10.0, 0.1, True), (7, 1000.0, 2e-5, True)])
def test_qp_stage_matches_oracle(engines, name, kdup, pi, delta, masked):
    """One penalty QP per problem.  `masked`: a non-trivial frozen-sparsity pattern (quirk C-2, prob.py:488-504):
    a third of the stored Jacobian slots is switched off, on the device through d_mask and in the oracle's A."""
    eng, st, params, x0 = engines[name]
    B = STAGE_N[name]
    params, x0 = params[:B], x0[:B]
    f, J, b, _ = eng.convexify(params, x0)
    Jn, bn = J.cpu().numpy(), b.cpu().numpy()
    lbx, ubx = x0 - delta, x0 + delta
    bits = None
    if masked:
        rng = np.random.default_rng(77)
        keep = rng.random((B, st.m_nl, 32)) > 1.0 / 3.0
        bits = (keep * (1 << np.arange(32, dtype=np.uint64))[None, None, :]).sum(axis=2).astype(np.uint32)
    xq, status, iters = eng.qp_solve(params, _settings(), J=J, b=b, lbx=lbx, ubx=ubx, pi=np.full(B, pi),
                                     kdup=np.full(B, kdup, np.int32),
                                     mask=None if bits is None else bits.view(np.int32))
    xq, status, iters = xq.cpu().numpy(), status.cpu().numpy(), iters.cpu().numpy()
    for i in range(B):
        # bit s of row r <=> stored slot s of that row participates
        P, q, A, l, u = helpers.stage_qp(st, params[i], Jn[i], bn[i], lbx[i], ubx[i], pi, kdup,
                                         bits=None if bits is None else bits[i])
        res = helpers.oracle_qp(P, q, A, l, u)
        assert status[i] == res.info.status_val, (i, status[i], res.info.status_val, iters[i], res.info.iter)
        assert iters[i] == res.info.iter, (i, iters[i], res.info.iter)
        if res.info.status_val in (1, 2, -2):
            err = np.abs(xq[i] - res.x).max()
            assert err <= 1e-7 * max(1.0, np.abs(res.x).max()), (i, err)


@pytest.mark.parametrize("name", [c[0] for c in CONFIGS])
def test_closest_point_qp_matches_oracle(engines, name):
    eng, st, params, x0 = engines[name]
    B = STAGE_N[name]
    params, x0 = params[:B], x0[:B]
    xq, status, iters = eng.qp_solve(params, _settings(), xref=x0, use_penalty=False, closest_point=True)
    xq, status, iters = xq.cpu().numpy(), status.cpu().numpy(), iters.cpu().numpy()
    inf = np.full(st.n, np.inf)
    for i in range(B):
        P, q, A, l, u = helpers.expand_qp(st, params[i], [], [], [], -inf, inf, 0.0, 0,
                                          closest_xref=x0[i], use_penalty=False)
        res = helpers.oracle_qp(P, q, A, l, u)
        assert status[i] == res.info.status_val
        assert iters[i] == res.info.iter
        assert np.abs(xq[i] - res.x).max() <= 1e-7 * max(1.0, np.abs(res.x).max())


@pytest.mark.parametrize("name", [c[0] for c in CONFIGS])
def test_full_solve_matches_port(engines, name):
    eng, st, params, x0 = engines[name]
    out = eng.solve_batch(params, x0, _settings())
    x = out["x"].cpu().numpy()
    verdict = out["verdict"].cpu().numpy()
    vio = out["max_vio"].cpu().numpy()
    obj = out["objective"].cpu().numpy()
    stats = out["stats"].cpu().numpy()
    refs = helpers.port_solve_many(name, range(x0.shape[0]), W.SOLVER_SETTINGS)
    for i in range(x0.shape[0]):
        ref = refs[i]
        info = (name, i, stats[i].tolist(), ref["stats"])
        assert (verdict[i] == 1) == ref["success"], info
        err = np.abs(x[i] - ref["x"]).max()
        assert err <= X_TOL[name] * max(1.0, np.abs(ref["x"]).max()), info + (err,)
        assert abs(vio[i] - ref["max_vio"]) <= 1e-5, info
        assert abs(obj[i] - ref["objective"]) <= OBJ_TOL[name] * max(1.0, abs(ref["objective"])), info


@pytest.mark.parametrize("name", [c[0] for c in CONFIGS])
def test_full_solve_matches_golden_reference(engines, name):
    """Against what the UNMODIFIED reference (Solver.solve on the oracle shims) produced in the build
    container: tests/golden/ref_<config>.npz written by oracle/gen_golden.py."""
    eng, st, params, x0 = engines[name]
    g = np.load(os.path.join(GOLDEN, "ref_%s.npz" % name))
    B = min(x0.shape[0], int(g["count"]))
    out = eng.solve_batch(params[:B], x0[:B], _settings())
    x = out["x"].cpu().numpy()
    verdict = out["verdict"].cpu().numpy()
    vio = out["max_vio"].cpu().numpy()
    for i in range(B):
        assert (verdict[i] == 1) == bool(g["success"][i]), (name, i)
        err = np.abs(x[i] - g["x"][i]).max()
        assert err <= X_TOL[name] * max(1.0, np.abs(g["x"][i]).max()), (name, i, err)
        assert abs(vio[i] - g["max_vio"][i]) <= 1e-5, (name, i)


def test_host_buffer_entry_matches_device_entry(engines):
    eng, st, params, x0 = engines["qcqp"]
    a = eng.solve_batch(params, x0, _settings())
    b = eng.solve_batch_host(params, x0, _settings())
    assert np.array_equal(a["x"].cpu().numpy(), b["x"])
    assert np.array_equal(a["verdict"].cpu().numpy(), b["verdict"])
    assert np.array_equal(a["stats"].cpu().numpy(), b["stats"])


def test_batch_properties_at_scale(engines):
    """Size-independent properties on a batch too large for the CPU oracle: every converged problem
    satisfies its constraints to cnt_tolerance, the reported violation / objective are those of
    the returned x, and results do not depend on batch composition or order."""
    eng, st, _, _ = engines["qcqp"]
    B = 4096
    _, params, x0 = W.gen_batch("qcqp", B)
    s = _settings()
    out = eng.solve_batch(params, x0, s)
    verdict = out["verdict"].cpu().numpy()
    vio = out["max_vio"].cpu().numpy()
    x = out["x"].cpu().numpy()
    assert (verdict == 1).mean() > 0.9
    assert (vio[verdict == 1] <= 1e-4).all()
    f, _, _, obj = eng.convexify(params, out["x"])
    val = params[:, st.blocks[0].val.off:st.blocks[0].val.off + st.blocks[0].m]
    assert np.allclose(np.maximum(f.cpu().numpy() - val, 0.0).max(axis=1), vio, atol=1e-12)
    assert np.allclose(obj.cpu().numpy(), out["objective"].cpu().numpy(), rtol=1e-12, atol=1e-12)
    # batch composition / order independence (dynamic work queue must not leak state)
    perm = np.random.default_rng(0).permutation(B)[:512]
    out2 = eng.solve_batch(params[perm], x0[perm], s)
    assert np.array_equal(out2["x"].cpu().numpy(), x[perm])
    assert np.array_equal(out2["verdict"].cpu().numpy(), verdict[perm])
    # a processing order (longest first) changes the schedule, not the results
    import torch
    order = torch.argsort(out["stats"][:, 2], descending=True).to(torch.int32)
    out3 = eng.solve_batch(params, x0, s, order=order)
    assert np.array_equal(out3["x"].cpu().numpy(), x) and np.array_equal(out3["verdict"].cpu().numpy(), verdict)


def test_dense_register_path_matches_generic_path(engines):
    """The two-warp register-resident ADMM loop (sco_dense.cuh) against the generic shared-memory
    loop on the same QPs: same status, same iteration count, x to 1e-9; and the same SQP outcome."""
    from sco_py_b200.engine import make_settings
    eng, st, params, x0 = engines["qcqp"]
    assert eng.team == 64
    B = x0.shape[0]
    f, J, b, _ = eng.convexify(params, x0)
    for kdup, pi, delta in [(1, 1.0, 1.0), (4, 100.0, 0.01), (9, 1e4, 3e-5)]:
        kw = dict(J=J, b=b, lbx=x0 - delta, ubx=x0 + delta, pi=np.full(B, pi), kdup=np.full(B, kdup, np.int32))
        xa, sa, ia = eng.qp_solve(params, _settings(), **kw)
        xb, sb, ib = eng.qp_solve(params, _settings(force_generic=1), **kw)
        assert np.array_equal(sa.cpu().numpy(), sb.cpu().numpy())
        assert np.array_equal(ia.cpu().numpy(), ib.cpu().numpy())
        assert np.abs(xa.cpu().numpy() - xb.cpu().numpy()).max() <= 1e-9
    _, p2, x2 = W.gen_batch("qcqp", 64)
    a = eng.solve_batch(p2, x2, _settings())
    g = eng.solve_batch(p2, x2, _settings(force_generic=1))
    va, vg = a["verdict"].cpu().numpy(), g["verdict"].cpu().numpy()
    assert (va == vg).mean() >= 0.98
    same = va == vg
    dx = np.abs(a["x"].cpu().numpy() - g["x"].cpu().numpy()).max(axis=1)
    assert np.quantile(dx[same], 0.9) <= 1e-4


def test_adaptive_rho_reaches_the_same_qp_optimum(engines):
    """`adaptive_rho=True` is selectable through Solver.solve (solver.py:39).  Upstream OSQP picks the
    adaptation interval from wall-clock setup time, so iteration counts are not comparable; the QP
    optimum is (SURVEY.md Appendix B-8): same status class and x to 1e-5 against the oracle run with
    the same flag, on the generic path and on a dense structure (which falls back to it)."""
    for name in ("qcqp", "point_robot"):
        eng, st, params, x0 = engines[name]
        B = x0.shape[0]
        f, J, b, _ = eng.convexify(params, x0)
        Jn, bn = J.cpu().numpy(), b.cpu().numpy()
        lbx, ubx = x0 - 0.3, x0 + 0.3
        s = _settings()
        s.osqp_adaptive_rho = 1
        xq, status, iters = eng.qp_solve(params, s, J=J, b=b, lbx=lbx, ubx=ubx, pi=np.full(B, 10.0),
                                         kdup=np.full(B, 2, np.int32))
        xq, status = xq.cpu().numpy(), status.cpu().numpy()
        for i in range(min(B, 3)):
            P, q, A, l, u = helpers.stage_qp(st, params[i], Jn[i], bn[i], lbx[i], ubx[i], 10.0, 2)
            res = helpers.oracle_qp(P, q, A, l, u, adaptive_rho=True)
            assert status[i] in (1, 2) and res.info.status_val in (1, 2), (name, i, status[i], res.info.status_val)
            assert np.abs(xq[i] - res.x).max() <= 1e-5 * max(1.0, np.abs(res.x).max()), (name, i)


def test_intended_semantics_mode_matches_the_port(engines):
    """The OSQP-backend quirks switched off (compound_penalty = freeze_sparsity = duplicate_rows = 0:
    fixed penalty weight, fresh sparsity, one copy of the penalty rows -- the maths of the reference's
    Gurobi backend, SURVEY.md section 8f-2): device against the port with the same switches, and the
    default penalty coefficient 1e3 of Solver() becomes usable (with the quirks it drives |q| to 1e18)."""
    eng, st, params, x0 = engines["qcqp"]
    off = dict(compound_penalty=0, freeze_sparsity=0, duplicate_rows=0)
    out = eng.solve_batch(params, x0, _settings(**off))
    x, verdict = out["x"].cpu().numpy(), out["verdict"].cpu().numpy()
    refs = helpers.port_solve_many("qcqp", range(16), W.SOLVER_SETTINGS, quirks={k: False for k in off})
    for i in range(16):
        ref = refs[i]
        assert (verdict[i] == 1) == ref["success"], i
        assert np.abs(x[i] - ref["x"]).max() <= 1e-4 * max(1.0, np.abs(ref["x"]).max()), i


def test_handles_of_one_team_size_do_not_disturb_each_other():
    """Kernel attributes (dynamic shared-memory limit, carve-out) belong to the kernel, not to a handle: creating a
    handle with a SMALLER working set of the same team size must not break launches of an earlier, larger one."""
    from sco_py_b200.engine import Engine
    st_big, p_big, x_big = W.gen_point_robot(4, T=40)
    st_small, p_small, x_small = W.gen_point_robot(4, T=33)
    big = Engine(st_big)
    a = big.solve_batch(p_big, x_big, _settings())
    small = Engine(st_small)
    assert small.team == big.team and small.smem_bytes < big.smem_bytes
    c = small.solve_batch(p_small, x_small, _settings())
    b = big.solve_batch(p_big, x_big, _settings())  # round 1: cudaErrorInvalidValue here
    d = small.solve_batch(p_small, x_small, _settings())
    assert np.array_equal(a["x"].cpu().numpy(), b["x"].cpu().numpy())
    assert np.array_equal(c["x"].cpu().numpy(), d["x"].cpu().numpy())
    big.close()
    small.close()


def test_bad_processing_order_is_refused(engines):
    """sco_solve_batch_ordered: an order that is not a permutation would solve some problems twice and skip
    others; the device check turns the whole batch into SCO_VERDICT_BAD_ORDER instead."""
    import torch
    eng, st, params, x0 = engines["qcqp"]
    B = 16
    order = torch.arange(B, dtype=torch.int32)
    order[3] = 5  # 5 twice, 3 never
    out = eng.solve_batch(params[:B], x0[:B], _settings(), order=order)
    assert (out["verdict"].cpu().numpy() == -3).all()
    order[3] = B  # out of range
    out = eng.solve_batch(params[:B], x0[:B], _settings(), order=order)
    assert (out["verdict"].cpu().numpy() == -3).all()
    good = eng.solve_batch(params[:B], x0[:B], _settings(), order=torch.arange(B - 1, -1, -1, dtype=torch.int32))
    ref = eng.solve_batch(params[:B], x0[:B], _settings())
    assert np.array_equal(good["x"].cpu().numpy(), ref["x"].cpu().numpy())


@pytest.mark.parametrize("name", ["point_robot", "arm", "qcqp"])
def test_thread_per_entity_loop_matches_the_strided_loop(engines, name):
    """sco_qp.cuh: fast_loop (one thread per variable / row, iterates and constants in registers) against
    generic_loop (the round-1 shared-memory loop, force_generic = 1) on the same QPs: same status, same iteration
    count, x to 1e-9 -- for penalty QPs and for the closest-point projection."""
    eng, st, params, x0 = engines[name]
    B = STAGE_N[name]
    params, x0 = params[:B], x0[:B]
    f, J, b, _ = eng.convexify(params, x0)
    for kdup, pi, delta in [(1, 1.0, 1.0), (3, 10.0, 0.1), (6, 1e3, 3e-5)]:
        kw = dict(J=J, b=b, lbx=x0 - delta, ubx=x0 + delta, pi=np.full(B, pi), kdup=np.full(B, kdup, np.int32))
        xa, sa, ia = eng.qp_solve(params, _settings(), **kw)
        xb, sb, ib = eng.qp_solve(params, _settings(force_generic=1), **kw)
        assert np.array_equal(sa.cpu().numpy(), sb.cpu().numpy()), (name, kdup)
        assert np.array_equal(ia.cpu().numpy(), ib.cpu().numpy()), (name, kdup, ia.cpu().numpy(), ib.cpu().numpy())
        assert np.abs(xa.cpu().numpy() - xb.cpu().numpy()).max() <= 1e-9, (name, kdup)
    xa, sa, ia = eng.qp_solve(params, _settings(), xref=x0, use_penalty=False, closest_point=True)
    xb, sb, ib = eng.qp_solve(params, _settings(force_generic=1), xref=x0, use_penalty=False, closest_point=True)
    assert np.array_equal(sa.cpu().numpy(), sb.cpu().numpy()) and np.array_equal(ia.cpu().numpy(), ib.cpu().numpy())
    assert np.abs(xa.cpu().numpy() - xb.cpu().numpy()).max() <= 1e-9


@pytest.mark.parametrize("name", [c[0] for c in CONFIGS])
@pytest.mark.parametrize("level", [1, 2])
def test_warm_start_mode_agrees_with_cold_start(engines, name, level):
    """sco_settings.warm_start (SURVEY.md section 8f-3): QPs start from the previous QP's (x, y) -- level 1 inside one
    trust-region loop (only l, u change between those QPs, solver.py:136-146), level 2 across the whole SQP.  The
    reference never warm-starts (osqp_utils.py:195 builds a new OSQP object per call), so this is an opt-in mode judged
    against the cold-start results of the same engine: every QP still ends on OSQP's termination criteria, the SQP
    trajectories differ at that level."""
    eng, st, params, x0 = engines[name]
    cold = eng.solve_batch(params, x0, _settings())
    warm = eng.solve_batch(params, x0, _settings(warm_start=level))
    vc, vw = cold["verdict"].cpu().numpy(), warm["verdict"].cpu().numpy()
    xc, xw = cold["x"].cpu().numpy(), warm["x"].cpu().numpy()
    ic, iw = cold["stats"][:, 2].cpu().numpy().astype(float), warm["stats"][:, 2].cpu().numpy().astype(float)
    same = vc == vw
    rel = np.abs(xc - xw).max(axis=1) / np.maximum(1.0, np.abs(xc).max(axis=1))
    print("warm_start=%d %s: verdicts equal %d/%d, rel |dx| median %.1e, ADMM iterations %.0f -> %.0f per problem" % (
        level, name, same.sum(), same.size, np.median(rel[same]), ic.mean(), iw.mean()))
    assert same.mean() >= 0.9
    # every QP ends on OSQP's tolerances (eps_abs 1e-6), the SQP on its own (min_approx_improve, trust region 1e-5):
    # two valid trajectories end within ~1e-4 of each other in the flat directions of the smoothness objectives
    assert np.median(rel[same]) <= 1e-3
    both = (vc == 1) & (vw == 1)
    assert (warm["max_vio"].cpu().numpy()[both] <= 1e-4).all()  # converged means feasible, warm or cold
    assert iw.sum() <= 1.05 * ic.sum()
