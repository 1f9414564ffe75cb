"""Objective terms bound to Variables (Structure.obj_blocks): converged problems per second and clock64() phase cycles
at B = 4,096 on one GPU.

    python profiles/obj_terms.py --lib NEW.so --timing-lib NEW_TIMING.so \
        [--parent-lib OLD.so --parent-timing-lib OLD_TIMING.so] [--repeats 3] [--out result.json]

Cases (16 distinct seeded problems tiled to B):
  robot40_step   C2's point robot at T = 40 (n = 80) with a soft-obstacle cost per step (bound to that step)
  chain20        the 20-variable chain of tests/test_caps.py (one term over all variables: obj_prog), on the new
                 library and -- with --parent-lib -- on the build before objective blocks, alternated
  robot30_step / robot30_summed   T = 30 (n = 60): the same costs as per-step terms, or summed into one term over all
                 60 variables (the only form earlier versions took).  The two are different QPs by design (each term's
                 eigenvalue shift vs one shift of the sum), so they are reported side by side per QP and per
                 convexification, not as a speed-up.
Every measurement runs in a subprocess of its own with SCO_B200_LIB set to the library it measures.  The timing
libraries are SCO_NVCC_FLAGS=-DSCO_TIMING builds (see profiles/time_solve.py): their merit / objective / max_vio /
x[:, 0:2] outputs carry cycle totals.  Card name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "oracle", "shims")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

B = 4096


def problems(case):
    import obj_problems as OP
    import test_caps as CAPS
    if case == "robot40_step":
        return [OP.robot(i, T=40, K=3) for i in range(16)]
    if case == "robot30_step":
        return [OP.robot(i, T=30, K=3) for i in range(16)]
    if case == "robot30_summed":
        return [_summed_robot(i, T=30, K=3) for i in range(16)]
    if case == "chain20":
        return [CAPS.build_chain(p)[0] for p in CAPS.chain_points(16, CAPS.CHAIN_SOLVE_N)]
    raise KeyError(case)


def _summed_robot(i, T, K):
    import bound_problems as BP
    import obj_problems as OP
    prob = BP.robot(i, T=T, K=K, form="bound")
    ov = np.array([[v] for v in sorted(prob._osqp_vars, key=lambda v: v.var_name)], dtype=object)
    x0 = prob._vars[0].get_value().ravel()
    rng = np.random.default_rng(100 + i)  # the centres of obj_problems.robot(cost="step")
    terms = [(OP.soft_obstacle(c=tuple(rng.uniform(-0.5, 0.5, 2))), np.array([2 * t, 2 * t + 1])) for t in range(T)]
    return OP.add_terms(prob, ov, x0, terms, form="summed")


def worker(case, timing, reps):
    import torch
    from sco_py_b200 import batch
    from sco_py_b200 import workloads as W
    from sco_py_b200.engine import Engine, make_settings
    st, params, x0, _ = batch.compile_batch(problems(case))
    reps_ = (B + params.shape[0] - 1) // params.shape[0]
    params, x0 = np.tile(params, (reps_, 1))[:B], np.tile(x0, (reps_, 1))[:B]
    eng = Engine(st)
    s = make_settings(solver=W.SOLVER_SETTINGS)
    res = dict(case=case, B=B, n=st.n, team=eng.team, occupancy=eng.occupancy, smem_bytes=eng.smem_bytes,
               obj_blocks=[(o.m, o.n_in) for o in st.obj_blocks], obj_prog_len=st.obj_prog_len)
    out = eng.solve_batch(params, x0, s)  # warm-up (module load)
    torch.cuda.synchronize()
    if timing:
        st_ = out["stats"].cpu().numpy().astype(float)
        x = out["x"].cpu().numpy()
        setup, loop = out["objective"].cpu().numpy(), out["max_vio"].cpu().numpy()
        cvx = x[:, 1]
        res.update(cyc_cvx_per_convexification=float(cvx.sum() / st_[:, 0].sum()),
                   cyc_qp_per_qp=float((setup.sum() + loop.sum()) / st_[:, 1].sum()),
                   cyc_total_per_problem=float(out["merit"].cpu().numpy().mean()),
                   sqp_iters=float(st_[:, 0].mean()), qp_solves=float(st_[:, 1].mean()),
                   admm_iters_per_qp=float(st_[:, 2].sum() / st_[:, 1].sum()))
    else:
        times = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = eng.solve_batch(params, x0, s)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        v = out["verdict"].cpu().numpy()
        stt = out["stats"].cpu().numpy().astype(float)
        res.update(seconds=times, converged=int((v == 1).sum()),
                   converged_per_s=[float((v == 1).sum() / t) for t in times],
                   sqp_iters=float(stt[:, 0].mean()), qp_solves=float(stt[:, 1].mean()),
                   us_per_qp=[1e6 * t / stt[:, 1].sum() for t in times],
                   us_per_problem=[1e6 * t / B for t in times])
    eng.close()
    print("RESULT " + json.dumps(res))


def run(case, lib, timing, reps):
    env = dict(os.environ, SCO_B200_LIB=os.path.abspath(lib))
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", case, "--timing", str(int(timing)),
                        "--repeats", str(reps)], env=env, capture_output=True, text=True)
    for line in p.stdout.splitlines():
        if line.startswith("RESULT "):
            r = json.loads(line[7:])
            r["lib"] = os.path.basename(lib)
            return r
    raise RuntimeError("%s on %s failed:\n%s\n%s" % (case, lib, p.stdout[-2000:], p.stderr[-4000:]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", default=None)
    ap.add_argument("--timing", type=int, default=0)
    ap.add_argument("--lib", default=os.path.join(ROOT, "sco_py_b200", "libsco_b200.so"))
    ap.add_argument("--timing-lib", default=None)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--parent-timing-lib", default=None)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.worker:
        return worker(a.worker, a.timing, a.repeats)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    results = dict(gpu=gpu, B=B, runs=[])
    for case in ("robot40_step", "robot30_step", "robot30_summed"):
        results["runs"].append(run(case, a.lib, False, a.repeats))
        if a.timing_lib:
            results["runs"].append(run(case, a.timing_lib, True, 1))
    for k in range(a.repeats):  # new and parent alternated
        results["runs"].append(run("chain20", a.lib, False, 1))
        if a.parent_lib:
            results["runs"].append(run("chain20", a.parent_lib, False, 1))
    if a.timing_lib:
        results["runs"].append(run("chain20", a.timing_lib, True, 1))
    if a.parent_timing_lib:
        results["runs"].append(run("chain20", a.parent_timing_lib, True, 1))
    print(json.dumps(results, indent=1))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
