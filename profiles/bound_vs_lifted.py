"""Point-robot obstacle workload written two ways, solved on the GPU (B problems each):
  lifted  one SymExpr over all 2T variables (rows of width 2T: 2T finite-difference columns per row)
  bound   one SymExpr per step bound to that step's Variable (column maps: rows of 2 inputs, packed into one block)
Prints, per form, the structure (rows, stored Jacobian entries per row, threads per problem, whether the
thread-per-entity ADMM loop applies), converged problems/s over `reps` timed solves of the whole batch after one
warm-up, and the verdict agreement of the two forms; with $OUT set, also writes them to $OUT/bound_vs_lifted.json.
    python profiles/bound_vs_lifted.py [B] [T] [K] [reps]
"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bound_problems as BP  # noqa: E402  (tests/bound_problems.py)
from sco_py_b200 import batch  # noqa: E402
from sco_py_b200 import workloads as W  # noqa: E402
from sco_py_b200.engine import Engine, make_settings  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
T = int(sys.argv[2]) if len(sys.argv) > 2 else 16
K = int(sys.argv[3]) if len(sys.argv) > 3 else 2
reps = int(sys.argv[4]) if len(sys.argv) > 4 else 3


def fast_ok(st):
    """sco_create's condition for the thread-per-entity loop: rows <= 8 entries, columns <= 4 + 4 entries."""
    pen = np.zeros(st.n, int)
    for bi in range(len(st.blocks)):
        np.add.at(pen, st.jac_cols(bi).ravel(), 1)
    lin = np.bincount(np.asarray(st.lin_col, dtype=int), minlength=st.n) if st.m_lin else np.zeros(st.n, int)
    rows = np.diff(st.lin_rowptr) if st.m_lin else np.zeros(0, int)
    return bool(all(b.jw <= 8 for b in st.blocks) and (rows <= 8).all() and (pen <= 4).all() and (lin <= 4).all())


props = torch.cuda.get_device_properties(0)
report = dict(device=props.name, B=B, T=T, K=K, reps=reps, forms={})
settings = make_settings(solver=W.SOLVER_SETTINGS)
verdicts = {}
for form in BP.FORMS:
    t0 = time.time()
    st, params, x0, _ = batch.compile_batch([BP.robot(i, T=T, K=K, form=form) for i in range(B)])
    t_compile = time.time() - t0
    eng = Engine(st)
    p_d = torch.as_tensor(params, device="cuda")
    x_d = torch.as_tensor(x0, device="cuda")
    out = eng.solve_batch(p_d, x_d, settings)  # warm-up
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = eng.solve_batch(p_d, x_d, settings)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    v = out["verdict"].cpu().numpy()
    verdicts[form] = v
    conv = int((v == 1).sum())
    med = float(np.median(times))
    r = dict(blocks=[(int(b.m), int(b.jw)) for b in st.blocks], team=eng.team, occupancy=eng.occupancy,
             fast_ok=fast_ok(st), compile_s=round(t_compile, 2), solve_s=times, converged=conv,
             converged_per_s=conv / med, mean_admm_iters=float(out["stats"][:, 2].double().mean()))
    report["forms"][form] = r
    print("%-6s blocks (m, entries/row) %s | team %d x %d/SM | thread-per-entity loop %s | %d / %d converged | "
          "median %.3f s -> %.0f converged problems/s" % (form, r["blocks"], eng.team, eng.occupancy, r["fast_ok"],
                                                          conv, B, med, r["converged_per_s"]), flush=True)
    eng.close()
report["same_verdicts"] = int((verdicts["bound"] == verdicts["lifted"]).sum())
print("verdicts equal in %d / %d problems; bound / lifted throughput %.2fx" % (
    report["same_verdicts"], B, report["forms"]["bound"]["converged_per_s"] / report["forms"]["lifted"]["converged_per_s"]))
if os.environ.get("OUT"):
    os.makedirs(os.environ["OUT"], exist_ok=True)
    with open(os.path.join(os.environ["OUT"], "bound_vs_lifted.json"), "w") as f:
        json.dump(report, f, indent=1)
