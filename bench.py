#!/usr/bin/env python
"""bench.py -- converged penalty-SQP problems per second (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--batch B] [--dump-outputs DIR]

Own arm (default): one "step" = one pass of the hot path (sco_solve_batch: closest feasible
point, convexification, penalty-QP assembly, ADMM, merit / trust-region state machine) over a
batch of B synthetic problems per GPU.  Workload = BASELINE.json configs[3]: C4 non-convex QCQP,
n=20, m=30, problem i drawn from default_rng(4000+i) (sco_py_b200/workloads.py), B=65,536 per GPU
("weak" scaling: rank r solves problems [r*B, (r+1)*B), no data-path collective).
`value` is timed with inputs resident in HBM; `e2e` is the same batch through the host-buffer
C-ABI entry (sco_solve_batch_host_async) from pinned memory, copies inside the timed region, for the
same number of steps.  After the timed regions (never inside them) the run
  * audits a random subsample of the batch against the CPU oracle (`detail.audit`; the same CPU pass
    is the `cpu_baseline` sample), and
  * times the two trajectory configurations, C2 point robot B=1,024 and C3 arm B=4,096
    (`detail.other_configs`, each with its own roofline and audit).

Reference arm (--impl reference): the reference's algorithm on the host CPUs -- the oracle port
(oracle/sqp_port.py + oracle/osqp_core.c, equal to /root/reference's sco_py run on the oracle shims;
upstream OSQP is not installable in this image) -- one process per core, bounded by WALL CLOCK: problems
are dealt one at a time until the budget (SCO_REF_BUDGET_S, default 150 s) is spent; whatever is still
running then is abandoned and value = converged problems / elapsed.  A single problem can need tens of
minutes on a core (penalty SQP has no iteration cap), so a sample bounded by count never ends in time.

Under torchrun (WORLD_SIZE > 1) every rank runs its shard; rank 0 prints ONE JSON line.
"""
import argparse
import json
import os
import signal
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "converged SQP problems/sec"
UNIT = "problems/s"
CONFIG_NAMES = {"qcqp": "C4 non-convex QCQP n=20 m=30 (BASELINE.json configs[3]), rng seeds 4000+i",
                "point_robot": "C2 point robot T=40 K=3 (configs[1]), rng seeds 2000+i",
                "arm": "C3 7-DOF arm T=20 (configs[2]), rng seeds 3000+i"}
PORT_NOTE = ("oracle port = the reference's penalty-SQP restated on structured inputs + restated OSQP 0.6.2 "
             "(equal to /root/reference run on the oracle shims to 1e-8, tests/test_oracle.py; upstream OSQP is "
             "not installable in this image)")


# ------------------------------------------------------------------------------ CPU arm
def _cpu_init():
    for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "oracle", "shims")):
        if p not in sys.path:
            sys.path.insert(0, p)
    signal.signal(signal.SIGTERM, signal.SIG_DFL)
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass
    import sqp_port  # noqa: F401  (import cost outside the timed region)


def _cpu_solve_one(job):
    name, index = job
    import sqp_port
    from sco_py_b200 import workloads as W
    st, params, x0 = W.GENERATORS[name](1, first=index)
    t0 = time.time()
    r = sqp_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    return dict(index=index, success=bool(r["success"]), seconds=time.time() - t0, x=r["x"],
                max_vio=float(r["max_vio"]), objective=float(r["objective"]),
                qp_solves=int(r["stats"]["qp_solves"]), admm_iters=int(r["stats"]["admm_iters"]))


class CpuArm(object):
    """The oracle port on every host core, one process per core, bounded by wall clock."""

    def __init__(self, name, cores=None):
        import multiprocessing as mp
        self.name = name
        self.cores = cores or (os.cpu_count() or 1)
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import build as oracle_build
        oracle_build.build()
        self.pool = mp.get_context("fork").Pool(self.cores, initializer=_cpu_init)
        self.pool.map(abs, range(self.cores * 4))  # workers up, imports done

    def run(self, indices, budget_s, on_result=None):
        """Deals `indices` one at a time; stops at the deadline.  -> dict(results, wall, dealt, complete)."""
        jobs = [(self.name, int(i)) for i in indices]
        t0 = time.time()
        it = self.pool.imap_unordered(_cpu_solve_one, jobs, chunksize=1)
        results = []
        complete = False
        import multiprocessing as mp
        while True:
            left = budget_s - (time.time() - t0)
            if left <= 0:
                break
            try:
                r = it.next(timeout=left)
            except mp.TimeoutError:
                break
            except StopIteration:
                complete = True
                break
            results.append(r)
            if on_result is not None:
                on_result(r, time.time() - t0)
        wall = time.time() - t0
        return dict(results=results, wall=wall, dealt=len(jobs), complete=complete)

    def close(self):
        self.pool.terminate()  # abandons whatever is still running
        self.pool.join()


def reference_line(args, value, conv, done, wall, cores, sample):
    return {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(args, args.config, args.batch),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "detail": {"converged": conv, "problems_completed": done, "wall_s": wall},
    }


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    budget = float(os.environ.get("SCO_REF_BUDGET_S", "150"))
    arm = CpuArm(args.config, args.cpu_cores)
    state = dict(conv=0, done=0, wall=0.0, printed=False, t0=time.time())

    def emit():
        if state["printed"]:
            return
        state["printed"] = True
        wall = max(state["wall"], 1e-9)
        sample = ("problems 0.. of the %s workload dealt one at a time to %d processes for %.0f s of wall clock (no "
                  "warm-up: a process pool has none); %d completed, the ones still running at the deadline are "
                  "abandoned and not counted; %s" % (args.config, arm.cores, wall, state["done"], PORT_NOTE))
        print(json.dumps(reference_line(args, state["conv"] / wall, state["conv"], state["done"], wall, arm.cores, sample)))
        sys.stdout.flush()

    def on_result(r, elapsed):
        state["done"] += 1
        state["conv"] += 1 if r["success"] else 0
        state["wall"] = elapsed

    def on_term(signum, frame):  # the driver's timeout: report what has been measured so far
        state["wall"] = time.time() - state["t0"]
        emit()
        try:
            arm.pool.terminate()
        except Exception:
            pass
        os._exit(0)

    signal.signal(signal.SIGTERM, on_term)
    signal.signal(signal.SIGINT, on_term)
    state["t0"] = time.time()
    out = arm.run(range(0, arm.cores * 256), budget, on_result)
    state["wall"] = out["wall"]
    emit()
    arm.close()
    return 0


# ------------------------------------------------------------------------------ helpers
def workload_config(args, name, per_gpu_batch):
    n_streams = max(1, min(getattr(args, "streams", 1), 8))
    return {"workload": CONFIG_NAMES[name], "batch_per_gpu": per_gpu_batch,
            "global_batch": per_gpu_batch * args.gpus, "parallelism": "problems sharded, dp%d" % args.gpus,
            "pipelining": "steps (independent batches) round-robin over %d CUDA streams" % n_streams,
            "queue_order": getattr(args, "order", "index"),
            "solver": "penalty_sqp, test_solver.py:15-25 hyper-parameters (mu0=1), OSQP eps_abs 1e-6 eps_rel 1e-9 "
                      "rho 0.1 fixed, reference quirks C-1..C-4 on, cold-started QPs",
            "l2": "inputs (%.2f GB of parameters per GPU) exceed the 126 MB L2; no flush needed"
                  % (per_gpu_batch * 58800 / 1e9) if name == "qcqp" else
                  "parameters are small (L2-resident after the first step, as they are for the reference's CPU "
                  "caches); the kernel's working set lives in shared memory"}


class ClockSampler(object):
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except Exception:
                continue
            for k, nm in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def algorithmic_bytes(st, stats):
    """SURVEY.md section 8(d): per problem sum_qp B_qp + sum_sqp B_cvx + 8(2n+4), resident regime."""
    n = st.n
    m_nl, n_slack = st.m_nl, st.n_slack
    nnz_lin = int(st.lin_rowptr[-1]) if st.m_lin else 0
    jnnz = sum(b.m * b.jw for b in st.blocks)
    n_q = n + n_slack
    m_q = st.m_lin + m_nl + n_q
    p = n * (n + 1) // 2
    a = jnnz + nnz_lin
    b_qp = 8 * (p + a + n_q + 2 * m_q) + 8 * (n_q + m_q) + 16
    per_problem_params = st.stride - (n * n - p if st.Q.off >= 0 and not st.Q.shared else 0)
    b_cvx = 8 * (per_problem_params + n) + 8 * (jnnz + m_nl + 1)
    qp_solves = stats[:, 1].astype(np.float64).sum()
    sqp_iters = stats[:, 0].astype(np.float64).sum()
    B = stats.shape[0]
    return float(qp_solves * b_qp + sqp_iters * b_cvx + B * 8 * (2 * n + 4)), b_qp, b_cvx


def admm_flops(st, stats):
    """FP64 flops of the ADMM iterations alone (2 flops per FMA of the three mat-vecs
    S^-1 rhs, J x~, J' w plus ~12 per row / variable of vector updates)."""
    n = st.n
    jnnz = sum(b.m * b.jw for b in st.blocks)
    nnz_lin = int(st.lin_rowptr[-1]) if st.m_lin else 0
    per_iter = 2.0 * (n * n + 2 * jnnz + 2 * nnz_lin) + 12.0 * (st.m_nl + st.n_slack + n + st.m_lin)
    return float(stats[:, 2].astype(np.float64).sum() * per_iter), per_iter


DUMP_LIMIT_BYTES = 64 << 20
NPY_HEADER_BYTES = 128  # what np.save puts before the data of a float64 array of up to two axes


def dump_outputs(out_dir, batches):
    """`--dump-outputs`: batches = {prefix: (problem numbers, {field: result array, one row per problem})} -> one
    out_dir/<prefix><field>.npy per field, in float64 (the integer fields -- verdict, stats, nonconverged -- are exact in
    it), and out_dir/<prefix>problem.npy, the problem number of every row.  If the files would exceed DUMP_LIMIT_BYTES
    in all, every batch keeps the same share of its problems: a subset fixed by a seed, so that two runs with the same
    arguments write the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    files = sum(1 + len(fields) for _, fields in batches.values())
    total = sum(8 * len(idx) * (1 + sum(a[:1].size for a in fields.values())) for idx, fields in batches.values())
    share = min(1.0, (DUMP_LIMIT_BYTES - NPY_HEADER_BYTES * files) / total) if total else 1.0
    for prefix, (idx, fields) in batches.items():
        rows = np.arange(len(idx))
        if share < 1.0:
            rows = np.sort(np.random.default_rng(0).permutation(len(idx))[:int(len(idx) * share)])
        np.save(os.path.join(out_dir, prefix + "problem.npy"), np.asarray(idx, dtype=np.float64)[rows])
        for name, a in fields.items():
            np.save(os.path.join(out_dir, prefix + name + ".npy"), np.asarray(a, dtype=np.float64)[rows])


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def roofline_of(name, st, stats, ms_step, fp64_peak, B):
    """The dominant (only) kernel of a step is k_solve.  Its working set is resident in shared memory, so the
    binding resource is the FP64 pipe; the HBM view SURVEY.md 8(d) asks for is reported beside it."""
    peaks = load_peaks()
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    abytes, b_qp, b_cvx = algorithmic_bytes(st, stats)
    flops, per_iter = admm_flops(st, stats)
    achieved_tf = flops / (ms_step * 1e-3) / 1e12
    achieved_gbs = abytes / (ms_step * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(name, {}).get("dram_bytes_per_problem")
            if traffic is not None:
                traffic = traffic * B
        except Exception:
            traffic = None
    return {
        "kernel": "k_solve (fused convexify + penalty-QP assembly + ADMM + merit/trust-region, one launch per step)",
        "regime": "resident: the whole QP working set lives in shared memory / registers for the solve",
        "bound": "fp64", "achieved": achieved_tf, "peak": fp64_peak, "unit": "TFLOP/s",
        "frac": achieved_tf / fp64_peak if fp64_peak else None,
        "peak_source": "sco_probe_fp64: dependent-free DFMA loop measured in this run (MEASURED_PEAKS.json carries no FP64 "
                       "figure; nominal 64 FMA/clk/SM x 148 SMs x 1.965 GHz = 37.2 TFLOP/s)",
        "flops_per_admm_iter": per_iter, "traffic": traffic,
        "hbm": {"achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": abytes, "bytes_per_qp": b_qp,
                "bytes_per_convexification": b_cvx,
                "note": "SURVEY.md 8(d) formula; small by construction in the resident regime (DESIGN.md section 4)"},
    }


def audit_against_oracle(name, indices, dev, budget_s, cores, first=0):
    """Solves problems `indices` (batch-local) of config `name` with the CPU oracle, for at most `budget_s` of wall
    clock, and compares them with the device results `dev` (numpy dict of the whole batch).
    -> (audit dict, cpu_baseline dict)."""
    arm = CpuArm(name, cores)
    out = arm.run([first + int(i) for i in indices], budget_s)
    arm.close()
    res = out["results"]
    rel, dvio, dobj, match, conv = [], [], [], 0, 0
    for r in res:
        i = r["index"] - first
        ok_dev = bool(dev["verdict"][i] == 1)
        match += int(ok_dev == r["success"])
        conv += int(r["success"])
        rel.append(float(np.abs(dev["x"][i] - r["x"]).max() / max(1.0, np.abs(r["x"]).max())))
        dvio.append(abs(float(dev["max_vio"][i]) - r["max_vio"]))
        dobj.append(abs(float(dev["objective"][i]) - r["objective"]) / max(1.0, abs(r["objective"])))
    n = len(res)
    audit = {"problems": n, "requested": len(indices), "budget_s": budget_s, "complete": out["complete"],
             "selection": "random subsample of the batch (rng 12345), dealt in that order; problems still running at the "
                          "deadline are dropped",
             "verdict_match": match, "converged_on_cpu": conv,
             "rel_dx": {"p50": float(np.percentile(rel, 50)) if n else None, "p99": float(np.percentile(rel, 99)) if n else None,
                        "max": max(rel) if n else None},
             "dvio_max": max(dvio) if n else None, "dobj_rel_max": max(dobj) if n else None,
             "tolerance": "north_star: 1e-4 relative on x, 1e-5 absolute on violation, same verdict"}
    cpu = {"value": conv / out["wall"] if out["wall"] > 0 else None, "unit": UNIT, "cores": arm.cores, "kind": "port",
           "sample": "%d random problems of the same batch completed in %.1f s of wall clock on %d processes (the audit "
                     "pass; unfinished ones dropped); %s" % (n, out["wall"], arm.cores, PORT_NOTE),
           "admm_iters_per_problem": float(np.mean([r["admm_iters"] for r in res])) if n else None}
    return audit, cpu


# ------------------------------------------------------------------------------ GPU arm
def time_config(args, name, B, steps, warmup, dev, local, rank, world, dist, sampler_on, e2e=True):
    """Generates config `name` (problems [rank*B, (rank+1)*B)), times `steps` device-resident steps and the same number
    of end-to-end steps.  -> dict of measurements + host copies of the results."""
    import torch
    from sco_py_b200 import workloads as W
    from sco_py_b200.engine import Engine, make_settings
    t_gen = time.time()
    st0 = W.GENERATORS[name](1)[0]
    h_params = torch.empty((B, st0.stride), dtype=torch.float64, pin_memory=True)
    h_x0 = torch.empty((B, st0.n), dtype=torch.float64, pin_memory=True)
    # SCO_BENCH_SHARD=r (diagnostic, single GPU): solve the shard rank r of a multi-rank job would hold
    shard = rank + int(os.environ.get("SCO_BENCH_SHARD", "0"))
    st, _, _ = W.gen_batch(name, B, first=shard * B, out_params=h_params.numpy(), out_x0=h_x0.numpy())
    t_gen = time.time() - t_gen
    eng = Engine(st, device=local)
    settings = make_settings(solver=W.SOLVER_SETTINGS)
    d_params = h_params.to(dev, non_blocking=True)
    d_x0 = h_x0.to(dev, non_blocking=True)
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(v, op):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    # Steps are independent batches: they are pipelined over `--streams` CUDA streams (launch slots of the
    # handle), so the tail of one launch -- a few long problems on a handful of SMs -- overlaps the next
    # launches.  The timed region is still K whole steps.
    n_streams = max(1, min(args.streams, 8))
    streams = [torch.cuda.Stream(device=dev) for _ in range(n_streams)]
    cur = torch.cuda.current_stream(dev)
    order = [None]

    def run_steps(count):
        outs = []
        for s_ in streams:
            s_.wait_stream(cur)
        for i in range(count):
            outs.append(eng.solve_batch(d_params, d_x0, settings, stream=streams[i % n_streams], order=order[0]))
        for s_ in streams:
            cur.wait_stream(s_)
        return outs

    warm = run_steps(warmup)
    if args.order == "profile" and warm:
        torch.cuda.synchronize()
        order[0] = torch.argsort(warm[-1]["stats"][:, 2], descending=True).to(torch.int32)
        run_steps(1)
    del warm
    barrier()
    sampler = ClockSampler(local) if sampler_on else None
    if sampler is not None:
        sampler.start()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record(cur)
    outs = run_steps(steps)
    e1.record(cur)
    barrier()
    ms_local = e0.elapsed_time(e1)
    ms_total = reduce(ms_local, dist.ReduceOp.MAX if world > 1 else None)
    clocks = sampler.stop() if sampler is not None else None
    out = outs[-1]
    for o_ in outs[:-1]:
        if not torch.equal(o_["verdict"], out["verdict"]) or not torch.equal(o_["x"], out["x"]):
            raise SystemExit("bench.py: two steps over the same batch disagree")
    host = {k: v.cpu().numpy() for k, v in out.items()}
    del outs
    verdict, stats = host["verdict"], host["stats"]
    converged = reduce(float((verdict == 1).sum()), dist.ReduceOp.SUM if world > 1 else None)
    res = dict(st=st, eng=eng, host=host, ms_local=ms_local, ms_total=ms_total, clocks=clocks, converged=converged,
               value=converged * steps / (ms_total * 1e-3), t_gen=t_gen, n_streams=n_streams, B=B, first=shard * B)

    if e2e:
        # end-to-end: host buffers through the C ABI (sco_solve_batch_host_async), the H2D copy of every step's
        # inputs and the D2H copy of its results inside the timed region, same pipelining, same number of steps
        def host_out():
            return dict(x=torch.empty((B, st.n), dtype=torch.float64, pin_memory=True).numpy(),
                        verdict=torch.empty(B, dtype=torch.int32, pin_memory=True).numpy(),
                        merit=torch.empty(B, dtype=torch.float64, pin_memory=True).numpy(),
                        objective=torch.empty(B, dtype=torch.float64, pin_memory=True).numpy(),
                        max_vio=torch.empty(B, dtype=torch.float64, pin_memory=True).numpy(),
                        stats=torch.empty((B, 4), dtype=torch.int32, pin_memory=True).numpy())

        e2e_steps = max(1, min(steps, args.e2e_steps if args.e2e_steps > 0 else steps))
        h_outs = [host_out() for _ in range(min(e2e_steps, n_streams))]

        def run_e2e(count):
            for i in range(count):
                eng.solve_batch_host(h_params.numpy(), h_x0.numpy(), settings, out=h_outs[i % len(h_outs)],
                                     stream=streams[i % n_streams])
            for s_ in streams:
                s_.synchronize()

        run_e2e(min(len(h_outs), 2))  # warm-up (staging allocations)
        barrier()
        t0 = time.perf_counter()
        run_e2e(e2e_steps)
        barrier()
        e2e_s = reduce(time.perf_counter() - t0, dist.ReduceOp.MAX if world > 1 else None)
        e2e_conv = reduce(float((h_outs[0]["verdict"] == 1).sum()), dist.ReduceOp.SUM if world > 1 else None)
        for ho in h_outs:
            if not np.array_equal(ho["verdict"], verdict) or not np.array_equal(ho["x"], host["x"]):
                raise SystemExit("bench.py: host-buffer path and device path disagree")
        res["e2e"] = {"value": e2e_conv * e2e_steps / e2e_s, "unit": UNIT,
                      "h2d_bytes_per_step": h_params.numel() * 8 + h_x0.numel() * 8,
                      "d2h_bytes_per_step": sum(v.nbytes for v in h_outs[0].values()),
                      "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s / e2e_steps}
        del h_outs
    del d_params, d_x0, h_params, h_x0
    return res


def measure_warm_start(args, eng, main, host):
    """`--batch` problems again with sco_settings.warm_start = 2 (every penalty QP after a problem's first starts from
    the previous QP's x and duals): throughput, iteration counts and agreement with the cold-start results."""
    import torch
    from sco_py_b200 import workloads as W
    from sco_py_b200.engine import make_settings
    B = main["B"]
    dev = eng.device
    st0 = eng.st
    h_params = torch.empty((B, st0.stride), dtype=torch.float64, pin_memory=True)
    h_x0 = torch.empty((B, st0.n), dtype=torch.float64, pin_memory=True)
    W.gen_batch(args.config, B, first=0, out_params=h_params.numpy(), out_x0=h_x0.numpy())
    d_params, d_x0 = h_params.to(dev), h_x0.to(dev)
    settings = make_settings(solver=W.SOLVER_SETTINGS, warm_start=2)
    n_streams = max(1, min(args.streams, 8))
    streams = [torch.cuda.Stream(device=dev) for _ in range(n_streams)]
    cur = torch.cuda.current_stream(dev)
    steps = min(args.steps, 4)

    def run(count):
        outs = []
        for s_ in streams:
            s_.wait_stream(cur)
        for i in range(count):
            outs.append(eng.solve_batch(d_params, d_x0, settings, stream=streams[i % n_streams]))
        for s_ in streams:
            cur.wait_stream(s_)
        return outs

    run(1)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(cur)
    outs = run(steps)
    e1.record(cur)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    out = {k: v.cpu().numpy() for k, v in outs[-1].items()}
    vc, vw = host["verdict"], out["verdict"]
    same = vc == vw
    rel = np.abs(host["x"] - out["x"]).max(axis=1) / np.maximum(1.0, np.abs(host["x"]).max(axis=1))
    conv = int((vw == 1).sum())
    return {"mode": "sco_settings.warm_start = 2 (opt-in; cold start is the default and the parity mode)",
            "value": conv / (ms * 1e-3), "unit": UNIT, "steps": steps, "ms_per_step": ms, "converged": conv,
            "verdicts_equal_to_cold": int(same.sum()), "problems": int(same.size),
            "rel_dx_vs_cold": {"p50": float(np.percentile(rel[same], 50)), "p99": float(np.percentile(rel[same], 99))},
            "max_vio_of_converged_max": float(out["max_vio"][vw == 1].max()) if conv else None,
            "mean_admm_iters": float(out["stats"][:, 2].mean()), "mean_admm_iters_cold": float(host["stats"][:, 2].mean()),
            "mean_qp_solves": float(out["stats"][:, 1].mean()), "mean_qp_solves_cold": float(host["stats"][:, 1].mean())}


def run_b200_arm(args):
    import torch
    import torch.distributed as dist
    from sco_py_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line: anything libraries print meanwhile (NCCL's version banner)
    # goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback (use --impl reference "
                         "for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    main = time_config(args, args.config, B, args.steps, args.warmup, dev, local, rank, world, dist,
                       sampler_on=(rank == 0))
    st, eng, host = main["st"], main["eng"], main["host"]
    stats, verdict = host["stats"], host["verdict"]
    ms_step = main["ms_total"] / args.steps
    # per-rank view of the tail: every rank's own device time and its longest problem (the step ends
    # when the rank that holds the longest problems is done)
    per_rank = [[main["ms_local"] / args.steps, float(stats[:, 2].max()), float(stats[:, 2].astype(np.float64).sum())]]
    if world > 1:
        t = torch.tensor(per_rank[0], dtype=torch.float64, device=dev)
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank = [a.cpu().tolist() for a in allt]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"": (main["first"] + np.arange(B), host)})

    import ctypes
    tf = ctypes.c_double(0.0)
    _lib.check(eng.lib.sco_probe_fp64(local, ctypes.byref(tf)))
    roofline = roofline_of(args.config, st, stats, ms_step, tf.value, B)
    team, smem_bytes, occupancy = eng.team, eng.smem_bytes, eng.occupancy
    # ---- opt-in warm start (sco_settings.warm_start = 2; the reference never warm-starts): same batch, outside the
    # timed regions of the headline numbers, judged against the cold-start results above
    warm_report = None
    if world == 1 and not args.no_warm_start:
        try:
            warm_report = measure_warm_start(args, eng, main, host)
        except Exception as ex:
            warm_report = {"error": repr(ex)}
    eng.close()

    # ---- oracle audit + CPU baseline: one CPU pass over a random subsample of the batch (outside every timed region)
    cpu, audit = None, None
    if world == 1 and args.audit > 0 and not args.no_cpu_baseline:
        idx = np.random.default_rng(12345).permutation(B)[:args.audit]
        audit, cpu = audit_against_oracle(args.config, idx, host, args.audit_seconds, args.cpu_cores, first=rank * B)

    # ---- the trajectory configurations (BASELINE.json configs[1], configs[2]) at their own batch sizes
    others = {}
    if world == 1 and not args.no_other_configs and args.config == "qcqp":
        for name, Bo in (("point_robot", 1024), ("arm", 4096)):
            try:
                r = time_config(args, name, Bo, steps=2, warmup=1, dev=dev, local=local, rank=0, world=1, dist=dist,
                                sampler_on=False, e2e=True)
                h = r["host"]
                ms_o = r["ms_total"] / 2
                entry = {"config": workload_config(args, name, Bo), "value": r["value"], "unit": UNIT, "steps": 2, "warmup": 1,
                         "ms_per_step": ms_o, "e2e": r["e2e"], "gpu_launches": 2,
                         "roofline": roofline_of(name, r["st"], h["stats"], ms_o, tf.value, Bo),
                         "converged": int((h["verdict"] == 1).sum()), "problems": Bo,
                         "mean_admm_iters": float(h["stats"][:, 2].mean()), "max_admm_iters": int(h["stats"][:, 2].max()),
                         "team": r["eng"].team, "smem_bytes": r["eng"].smem_bytes, "ctas_per_sm": r["eng"].occupancy}
                r["eng"].close()
                if args.audit > 0 and not args.no_cpu_baseline:
                    idx = np.random.default_rng(12345).permutation(Bo)[:min(args.audit, 64)]
                    entry["audit"], entry["cpu_baseline"] = audit_against_oracle(name, idx, h, args.other_audit_seconds,
                                                                                 args.cpu_cores)
                others[name] = entry
            except Exception as ex:  # never lose the headline line to a side measurement
                others[name] = {"error": repr(ex)}

    busiest = max(range(len(per_rank)), key=lambda r: per_rank[r][0])
    line = {
        "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, args.config, B),
        "clocks": main["clocks"],
        "e2e": main["e2e"],
        "gpu_launches": args.steps,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "detail": {"converged": int(main["converged"]), "problems": B * world,
                   "verdict_counts": {str(k): int((verdict == k).sum()) for k in (-1, 0, 1)},
                   "mean_sqp_iters": float(stats[:, 0].mean()), "mean_qp_solves": float(stats[:, 1].mean()),
                   "mean_admm_iters": float(stats[:, 2].mean()), "max_admm_iters": int(stats[:, 2].max()),
                   "audit": audit, "warm_start": warm_report,
                   "per_rank": [{"rank": r, "ms_per_step": round(v[0], 1), "max_admm_iters": int(v[1]),
                                 "busy_fraction": round(v[0] / ms_step, 3), "total_admm_iters": int(v[2])}
                                for r, v in enumerate(per_rank)],
                   "limiter": "rank %d: a problem is sequential, its longest one needs %d ADMM iterations (k_solve tail); "
                              "every rank holds the same total work within 2 %%" % (busiest, int(per_rank[busiest][1])),
                   "team": team, "smem_bytes": smem_bytes, "ctas_per_sm": occupancy,
                   "gen_seconds": main["t_gen"], "other_configs": others},
    }
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line))
    sys.stdout.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0



# ------------------------------------------------------------------------------ C5: mixed shapes
def run_mixed(args):
    """BASELINE.json configs[4]: `--batch` mixed-shape problems per GPU (global problem numbers [rank*B, (rank+1)*B),
    i.i.d. mixture of nine structures, workloads.gen_mixed), bucketed by structure; every bucket is one launch of its
    own engine, all buckets of a step run concurrently on their own streams.  Reports verdict counts per bucket, an
    audit of a random subsample of every bucket against the CPU oracle (rank 0, time-bounded) and the usual line."""
    import torch
    import torch.distributed as dist
    from sco_py_b200 import workloads as W
    from sco_py_b200.engine import Engine, make_settings
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    t0 = time.time()
    cores = os.cpu_count() or 1
    buckets = W.gen_mixed(B, first=rank * B, workers=max(1, min(32, cores // max(world, 1))))
    t_gen = time.time() - t0
    settings = make_settings(solver=W.SOLVER_SETTINGS)
    for bk in buckets:
        bk["eng"] = Engine(bk["structure"], device=local)
        bk["d_params"] = torch.as_tensor(bk["params"]).to(dev)
        bk["d_x0"] = torch.as_tensor(bk["x0"]).to(dev)
        bk["stream"] = torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()
    cur = torch.cuda.current_stream(dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        outs = []
        for bk in buckets:  # the long buckets first: they decide when the step ends
            bk["stream"].wait_stream(cur)
            outs.append(bk["eng"].solve_batch(bk["d_params"], bk["d_x0"], settings, stream=bk["stream"]))
        for bk in buckets:
            cur.wait_stream(bk["stream"])
        return outs

    buckets.sort(key=lambda bk: -bk["structure"].n * len(bk["indices"]))
    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler is not None:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    bucket_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in buckets]
    e0.record(cur)
    outs = None
    for k in range(args.steps):
        if k == args.steps - 1:  # per-bucket device time of the last step
            outs = []
            for bk, (a, b) in zip(buckets, bucket_ev):
                bk["stream"].wait_stream(cur)
                a.record(bk["stream"])
                outs.append(bk["eng"].solve_batch(bk["d_params"], bk["d_x0"], settings, stream=bk["stream"]))
                b.record(bk["stream"])
            for bk in buckets:
                cur.wait_stream(bk["stream"])
        else:
            step()
    e1.record(cur)
    barrier()
    ms_local = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler is not None else None
    rows = []
    conv_local = 0
    for bk, out, (a, b) in zip(buckets, outs, bucket_ev):
        v = out["verdict"].cpu().numpy()
        stt = out["stats"].cpu().numpy()
        bk["host"] = {k: t.cpu().numpy() for k, t in out.items()}
        conv_local += int((v == 1).sum())
        rows.append([bk["bucket"], len(v), int((v == 1).sum()), int((v == 0).sum()), int((v == -1).sum()),
                     float(stt[:, 2].astype(np.float64).sum()), float(stt[:, 2].max()), a.elapsed_time(b),
                     bk["eng"].team, bk["eng"].occupancy])
    t = torch.tensor([ms_local, float(conv_local)], dtype=torch.float64, device=dev)
    table = torch.zeros((len(W.MIXED_BUCKETS), 10), dtype=torch.float64, device=dev)
    for r in rows:
        table[int(r[0])] = torch.tensor(r, dtype=torch.float64, device=dev)
    if world > 1:
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        allb = [torch.zeros_like(table) for _ in range(world)]
        dist.all_gather(allb, table)
    else:
        allt, allb = [t], [table]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"bucket%d_" % bk["bucket"]: (bk["indices"], bk["host"]) for bk in buckets})
    per_rank = [a.cpu().tolist() for a in allt]
    ms_total = max(v[0] for v in per_rank)
    converged = sum(v[1] for v in per_rank)
    tabs = np.stack([a.cpu().numpy() for a in allb])  # [world, buckets, 10]
    bucket_report = []
    for bi, (name, kw) in enumerate(W.MIXED_BUCKETS):
        tt = tabs[:, bi, :]
        n_prob = int(tt[:, 1].sum())
        if n_prob == 0:
            continue
        bucket_report.append({"bucket": bi, "shape": name, "kw": kw, "problems": n_prob, "converged": int(tt[:, 2].sum()),
                              "failed": int(tt[:, 3].sum()), "iter_cap": int(tt[:, 4].sum()),
                              "mean_admm_iters": float(tt[:, 5].sum() / n_prob), "max_admm_iters": int(tt[:, 6].max()),
                              "device_ms_last_step_max_over_ranks": float(tt[:, 7].max()), "team": int(tt[:, 8].max()),
                              "ctas_per_sm": int(tt[:, 9].max())})
    # ---- audit (rank 0's problems, every bucket, time-bounded) against the oracle port
    audits = {}
    if args.audit > 0 and not args.no_cpu_baseline:
        per_bucket_s = args.audit_seconds / max(1, len(buckets))
        for bk in buckets:
            name = bk["name"]
            take = np.random.default_rng(12345).permutation(len(bk["indices"]))[:args.audit]
            arm = MixedCpuArm(name, bk["kw"], args.cpu_cores)
            out = arm.run([int(bk["indices"][i]) for i in take], per_bucket_s)
            arm.close()
            pos = {int(bk["indices"][i]): int(i) for i in take}
            rel, dvio, match = [], [], 0
            for r in out["results"]:
                i = pos[r["index"]]
                match += int(bool(bk["host"]["verdict"][i] == 1) == r["success"])
                rel.append(float(np.abs(bk["host"]["x"][i] - r["x"]).max() / max(1.0, np.abs(r["x"]).max())))
                dvio.append(abs(float(bk["host"]["max_vio"][i]) - r["max_vio"]))
            audits[str(bk["bucket"])] = {"problems": len(out["results"]), "requested": int(len(take)), "verdict_match": match,
                                         "rel_dx_max": max(rel) if rel else None, "dvio_max": max(dvio) if dvio else None,
                                         "wall_s": out["wall"]}
    value = converged * args.steps / (ms_total * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "C5 mixed TAMP-shaped subproblems (BASELINE.json configs[4]): 50 % QCQP n/m in "
                               "(10,15),(20,30),(30,45), 30 % point robot T in 20,40 x K in 1,3, 20 % arm T in 10,20; "
                               "problem i from default_rng(5000+i)",
                   "batch_per_gpu": B, "global_batch": B * world, "parallelism": "problems sharded, dp%d" % world,
                   "pipelining": "the buckets of a step run concurrently on one stream each",
                   "solver": workload_config(args, "qcqp", B)["solver"]},
        "clocks": clocks, "gpu_launches": args.steps * len(buckets),
        "detail": {"converged": int(converged), "problems": B * world, "buckets": bucket_report,
                   "audit_rank0": audits, "gen_seconds_rank0": t_gen,
                   "per_rank": [{"rank": r, "ms_per_step": v[0] / args.steps, "converged": int(v[1])} for r, v in enumerate(per_rank)]},
    }
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line))
    sys.stdout.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0


def _cpu_solve_mixed(job):
    name, kw, index = job
    import sqp_port
    from sco_py_b200 import workloads as W
    st, params, x0 = W.GENERATORS[name](1, seed_base=W.MIXED_SEED, indices=[index], **kw)
    r = sqp_port.solve(st, params[0], x0[0], solver=W.SOLVER_SETTINGS)
    return dict(index=index, success=bool(r["success"]), x=r["x"], max_vio=float(r["max_vio"]),
                objective=float(r["objective"]), admm_iters=int(r["stats"]["admm_iters"]))


class MixedCpuArm(CpuArm):
    def __init__(self, name, kw, cores=None):
        CpuArm.__init__(self, name, cores)
        self.kw = kw

    def run(self, indices, budget_s, on_result=None):
        import multiprocessing as mp
        jobs = [(self.name, self.kw, int(i)) for i in indices]
        t0 = time.time()
        it = self.pool.imap_unordered(_cpu_solve_mixed, jobs, chunksize=1)
        results, complete = [], False
        while True:
            left = budget_s - (time.time() - t0)
            if left <= 0:
                break
            try:
                results.append(it.next(timeout=left))
            except mp.TimeoutError:
                break
            except StopIteration:
                complete = True
                break
        return dict(results=results, wall=time.time() - t0, dealt=len(jobs), complete=complete)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="qcqp", choices=["qcqp", "point_robot", "arm", "mixed"])
    ap.add_argument("--batch", type=int, default=65536, help="problems per GPU")
    ap.add_argument("--e2e-steps", type=int, default=0, help="end-to-end steps (0 = as many as --steps)")
    ap.add_argument("--order", default="index", choices=["index", "profile"],
                    help="work-queue order: index (default) or profile = longest first by the ADMM iteration counts "
                         "of the last warm-up step (sco_solve_batch_ordered; for callers that re-solve similar batches)")
    ap.add_argument("--streams", type=int, default=8, help="CUDA streams the steps are pipelined over (1..8)")
    ap.add_argument("--audit", type=int, default=256, help="problems of the batch audited against the CPU oracle after "
                                                            "the timed regions (0 = none); the same pass is the cpu_baseline")
    ap.add_argument("--audit-seconds", type=float, default=60.0, help="wall-clock budget of the audit pass")
    ap.add_argument("--other-audit-seconds", type=float, default=20.0)
    ap.add_argument("--cpu-cores", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU pass (audit and cpu_baseline)")
    ap.add_argument("--no-other-configs", action="store_true", help="skip detail.other_configs (C2 / C3)")
    ap.add_argument("--no-warm-start", action="store_true", help="skip detail.warm_start (the opt-in warm-start mode)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step (rank 0's problems) as DIR/<name>.npy, float64, at "
                         "most 64 MB in all, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's results; the reference arm has no timed steps")
    args.cpu_cores = args.cpu_cores or None
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        args.gpus = world
    if args.impl == "reference":
        if args.config == "mixed":
            args.config = "qcqp"
        return run_reference_arm(args)
    if args.config == "mixed":
        return run_mixed(args)
    return run_b200_arm(args)


if __name__ == "__main__":
    sys.exit(main())
