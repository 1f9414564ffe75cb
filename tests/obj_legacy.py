"""Outputs of the objective problems that keep the one-term obj_prog structure (a scalar SymExpr over every variable
in QP order), on seeded inputs: the 20-variable chain of test_caps.py (full solves, both ADMM loops), the
40-variable chain (sco_convexify_model, finite-difference and analytic gradients) and the nine C1 problems of
test_c1_toy.py (full solves, both gradient modes).  tests/golden/obj_legacy_parent.npz holds them as computed by the
version before objective blocks existed; the device must reproduce them bit for bit.

    python tests/obj_legacy.py OUT.npz     # record with the library sco_py_b200 loads (SCO_B200_LIB to choose)
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "oracle", "shims")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

GOLDEN = os.path.join(HERE, "golden", "obj_legacy_parent.npz")


def compute():
    import torch
    import test_c1_toy as C1
    import test_caps as CAPS
    from sco_py_b200 import batch
    from sco_py_b200 import workloads as W
    from sco_py_b200.engine import Engine, make_settings
    out = {}

    def solves(key, probs):
        st, params, x0, _ = batch.compile_batch(probs)
        eng = Engine(st)
        for fg in (0, 1):
            r = eng.solve_batch(params, x0, make_settings(solver=W.SOLVER_SETTINGS, force_generic=fg))
            torch.cuda.synchronize()
            for k in ("x", "verdict", "merit", "objective", "max_vio", "stats"):
                out["%s_fg%d_%s" % (key, fg, k)] = r[k].cpu().numpy()
        eng.close()

    solves("chain20", [CAPS.build_chain(p)[0] for p in CAPS.chain_points(8, CAPS.CHAIN_SOLVE_N)])
    for analytic in (False, True):
        st, params, x0, _ = batch.compile_batch([CAPS.build_chain(p, analytic=analytic)[0]
                                                 for p in CAPS.chain_points(4, CAPS.CHAIN_STAGE_N)])
        eng = Engine(st)
        res = tuple(eng.convexify(params, x0)) + tuple(eng.convexify_model(params, x0))
        torch.cuda.synchronize()
        for k, v in zip(("f", "J", "b", "obj", "H", "g", "c"), res):
            out["chain40_a%d_%s" % (analytic, k)] = v.cpu().numpy()
        eng.close()
        for name in sorted(C1.SYM_PROBLEMS):
            solves("c1_%s_a%d" % (name, analytic), [C1.build_sym(name, analytic=analytic)[0]])
    return out


if __name__ == "__main__":
    res = compute()
    np.savez_compressed(sys.argv[1], **res)
    print("recorded %d arrays to %s" % (len(res), sys.argv[1]))
