"""clock64() phase breakdown of the whole penalty-SQP solve (needs a library built with
SCO_NVCC_FLAGS=-DSCO_TIMING python -m sco_py_b200.build --force).  In that diagnostic build the
merit / objective / max_vio / x[:, 0:2] outputs carry cycle totals per problem:
total, QP setup (scaling + factorisation), ADMM loop (incl. termination tests), termination tests,
convexification.
    python profiles/time_solve.py [config] [batch]

"Termination tests" counts what a test still exposes.  The dense loop (sco_dense.cuh) runs the first half of the
test of iteration k beside iteration k+1; their shared barrier ends the ADMM-loop share.  The test's count runs
from there to the decision, plus the certificates and the restore of iteration k, the test that ends the solve
included.  Where the dense loop tests unpipelined (check_termination 1, or k+1 = max_iter), and in the other
loops, it runs from the end of the tested iteration to the decision, the ending test excluded.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from sco_py_b200 import workloads as W  # noqa: E402
from sco_py_b200.engine import Engine, make_settings  # noqa: E402

name = sys.argv[1] if len(sys.argv) > 1 else "qcqp"
B = int(sys.argv[2]) if len(sys.argv) > 2 else 2368
st, params, x0 = W.gen_batch(name, B)
eng = Engine(st)
s = make_settings(solver=W.SOLVER_SETTINGS)
out = eng.solve_batch(params, x0, s)
torch.cuda.synchronize()
tot = out["merit"].cpu().numpy()
setup = out["objective"].cpu().numpy()
loop = out["max_vio"].cpu().numpy()
x = out["x"].cpu().numpy()
chk, cvx = x[:, 0], x[:, 1]
stats = out["stats"].cpu().numpy()
it, qps = stats[:, 2].astype(float), stats[:, 1].astype(float)
T = tot.sum()
print("%s B=%d team %d ctas/sm %d | cycles/problem %.3g | per ADMM iteration (all-in) %.0f" % (
    name, B, eng.team, eng.occupancy, tot.mean(), T / it.sum()))
print("  share: qp setup %.1f%% | admm loop w/o tests %.1f%% | termination tests %.1f%% | convexify %.1f%% | rest %.1f%%" % (
    100 * setup.sum() / T, 100 * (loop.sum() - chk.sum()) / T, 100 * chk.sum() / T, 100 * cvx.sum() / T,
    100 * (T - setup.sum() - loop.sum() - cvx.sum()) / T))
print("  per QP: setup %.0f cycles | per iteration: loop %.0f, tests %.0f (= %.0f per test) | iters/QP %.0f" % (
    setup.sum() / qps.sum(), (loop.sum() - chk.sum()) / it.sum(), chk.sum() / it.sum(), 25 * chk.sum() / it.sum(),
    it.sum() / qps.sum()))
