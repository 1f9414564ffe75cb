"""Host-side logic that needs no GPU: workloads, structure description, settings, sharding."""
import os
import sys

import numpy as np
import pytest

from sco_py_b200 import workloads as W
from sco_py_b200.shard import shard_range, shard_sizes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("name", ["qcqp", "point_robot", "arm"])
def test_generators_are_reproducible_per_problem(name):
    st, p, x = W.GENERATORS[name](4)
    st2, p2, x2 = W.GENERATORS[name](2, first=2)
    assert np.array_equal(p[2:], p2) and np.array_equal(x[2:], x2)
    assert p.shape == (4, st.stride) and x.shape == (4, st.n)


def test_parallel_generation_matches_serial():
    st, p, x = W.gen_qcqp(200)
    st2, p2, x2 = W.gen_batch("qcqp", 200, workers=2)
    assert np.array_equal(p, p2) and np.array_equal(x, x2)


def test_config_sizes_follow_the_survey():
    st, _, _ = W.gen_qcqp(1)
    assert (st.n, st.m_nl, st.n_slack, st.stride) == (20, 30, 30, 7350)
    st, _, _ = W.gen_point_robot(1)
    assert (st.n, st.m_nl, st.m_lin) == (80, 120, 4)
    st, _, _ = W.gen_arm(1)
    assert (st.n, st.m_nl, st.m_lin, st.n_slack) == (140, 3, 287, 6)


def test_settings_from_solver_attributes():
    from sco_py_b200.engine import make_settings
    s = make_settings(solver=W.SOLVER_SETTINGS, osqp=dict(eps_abs=1e-5, adaptive_rho=True))
    assert s.initial_penalty_coeff == 1.0 and s.max_merit_coeff_increases == 5
    assert s.min_trust_region_size == 1e-5 and s.osqp_eps_abs == 1e-5 and s.osqp_adaptive_rho == 1
    with pytest.raises(KeyError):
        make_settings(solver=dict(no_such_attribute=1))


def test_shard_ranges_partition_the_batch():
    for B in (0, 1, 7, 65536, 65537):
        for world in (1, 2, 3, 8):
            ranges = [shard_range(B, r, world) for r in range(world)]
            assert ranges[0][0] == 0 and ranges[-1][1] == B
            assert all(ranges[r][1] == ranges[r + 1][0] for r in range(world - 1))
            sizes = shard_sizes(B, world)
            assert max(sizes) - min(sizes) <= 1 and sum(sizes) == B


def _gather_worker(rank, world, port, B, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    from sco_py_b200.shard import gather_results, shard_range
    lo, hi = shard_range(B, rank, world)
    idx = torch.arange(lo, hi, dtype=torch.float64)
    local = dict(x=idx[:, None] * torch.ones(1, 3, dtype=torch.float64), verdict=(idx % 2).to(torch.int32))
    full = gather_results(local, B)
    ok = bool(torch.equal(full["x"][:, 0], torch.arange(B, dtype=torch.float64))
              and torch.equal(full["verdict"], (torch.arange(B) % 2).to(torch.int32)))
    q.put((rank, ok))
    dist.destroy_process_group()


def test_result_gather_world_size_2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, 7, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert res == [(0, True), (1, True)]


def test_dump_outputs_writes_float64_rows_within_the_limit(tmp_path, monkeypatch):
    """bench.py --dump-outputs: every field as float64 with the problem number of each row; past the size limit the
    same seeded subset of problems in every field and in every run."""
    import bench
    B = 1000
    host = dict(x=np.random.default_rng(1).normal(size=(B, 20)), verdict=np.arange(B, dtype=np.int32) % 3 - 1,
                stats=np.arange(4 * B, dtype=np.int32).reshape(B, 4))
    bench.dump_outputs(str(tmp_path / "all"), {"": (500 + np.arange(B), host)})
    for name, a in host.items():
        d = np.load(tmp_path / "all" / (name + ".npy"))
        assert d.dtype == np.float64 and np.array_equal(d, a)
    assert np.array_equal(np.load(tmp_path / "all" / "problem.npy"), 500 + np.arange(B))
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 8 * 25 * B // 4)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"": (np.arange(B), host), "second_": (np.arange(B), host)})
    files = sorted(os.listdir(tmp_path / "a"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_LIMIT_BYTES
    rows = np.load(tmp_path / "a" / "problem.npy").astype(int)
    assert 0 < len(rows) < B
    for f in files:
        d = np.load(tmp_path / "a" / f)
        assert np.array_equal(d, np.load(tmp_path / "b" / f))
        if not f.endswith("problem.npy"):
            assert np.array_equal(d, host[f[:-4].replace("second_", "")][rows])


def test_reference_arm_prints_one_line_within_its_budget_single_and_under_torchrun():
    """`bench.py --impl reference` (the CPU arm the driver times next to the GPU arm): one JSON line with the contract's
    keys inside a wall-clock budget, also when the time runs out mid-problem; under torchrun rank 0 alone works and
    prints, the other ranks exit 0."""
    import json
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, SCO_REF_BUDGET_S="4")
    for cmd in ([sys.executable, "bench.py", "--impl", "reference", "--steps", "20", "--warmup", "5", "--cpu-cores", "2"],
                [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                 "127.0.0.1", "--master-port", "29533", "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "20",
                 "--warmup", "5", "--cpu-cores", "2"]):
        p = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=240)
        assert p.returncode == 0, p.stderr[-2000:]
        lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
        assert len(lines) == 1, p.stdout
        d = json.loads(lines[0])
        assert d["impl"] == "reference" and d["metric"] == "converged SQP problems/sec" and d["unit"] == "problems/s"
        assert d["higher_is_better"] is True and d["gpu_launches"] == 0
        assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 2
        assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
        assert d["detail"]["wall_s"] <= 10.0 and d["value"] >= 0.0
