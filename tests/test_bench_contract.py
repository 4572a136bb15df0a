"""bench.py contract checks: byte formulas of SURVEY.md §8(d), the JSON line of the reference arm and --dump-outputs
(all but the last test need no GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_algorithmic_bytes_match_the_survey():
    assert bench.algorithmic_bytes_per_asset_step(50, 50, 5, 0.0, False) == pytest.approx(8.5)          # Mode S, A=50
    assert bench.algorithmic_bytes_per_asset_step(100, 50, 5, 0.0, False) == pytest.approx(8.25)
    assert bench.algorithmic_bytes_per_asset_step(500, 50, 5, 0.0025, False) == pytest.approx(12.05)    # commission: + w_last
    assert bench.algorithmic_bytes_per_asset_step(100, 50, 5, 0.0, True) == pytest.approx(1208.25)      # Mode O
    assert bench.algorithmic_bytes_per_asset_step(50, 50, 5, 0.0, True) == pytest.approx(1208.5)


def test_workloads_are_the_baseline_configs():
    w = bench.WORKLOADS
    assert w["c2"][:3] == (4096, 50, 50) and w["c3"][:3] == (65536, 100, 50) and w["c5"][:3] == (262144, 500, 50)
    assert w["c4_shard"][0] * 8 == 1048576 and w["c4_shard"][1:3] == (100, 50)
    assert w["c5"][4] == 0.0025 and not w["c5"][5]                     # commission, state-only
    assert w["c4"][:3] == (1048576, 100, 50)                           # config 4 whole (divided over the ranks: strong scaling)


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, PMRL_BENCH_REF_SECONDS="0.2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3",
                          "--workload", "c2"], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["value"] > 0 and line["config"]["workload"] == "c2"
    from oracle import live_reference as live
    want_kind = "reference" if live.locate() else "port"                # BASELINE.md §3 step 2: the live tree first, else the port
    assert line["cpu_baseline"]["kind"] == want_kind and line["cpu_baseline"]["cores"] >= 1
    cfg = bench.shared_config(type("A", (), dict(workload="c2", envs=0, tune=[], graph=0, burst=0))(), 1)
    assert line["config"] == cfg                                        # both arms print the same config object
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_falls_back_to_the_port_without_the_tree():
    env = dict(os.environ, PMRL_BENCH_REF_SECONDS="0.2", PMRL_REFERENCE_ROOT="/nonexistent")
    code = ("import sys; sys.path.insert(0, %r); from oracle import live_reference as live; live.locate = lambda: None; import bench; "
            "print(bench.cpu_baseline(11, 8, 0.0, seconds=0.2, context=False)['kind'])" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0 and out.stdout.strip().splitlines()[-1] == "port", out.stderr[-2000:]


def test_reference_arm_other_ranks_exit_without_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, env=env, timeout=60)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_whole_or_one_seeded_env_sample(tmp_path):
    E = 1000
    arrays = {"obs": (torch.arange(E * 6, dtype=torch.float32).reshape(E, 2, 3), 0),
              "reward": (torch.arange(E, dtype=torch.float32) / 7, 0),
              "done": ((torch.arange(E) % 3 == 0).to(torch.uint8), 0),
              "burst_reward": (torch.arange(3 * E, dtype=torch.float32).reshape(3, E), 1)}
    bench.dump_outputs(str(tmp_path / "whole"), arrays, E)
    assert sorted(os.listdir(tmp_path / "whole")) == ["burst_reward.npy", "done.npy", "obs.npy", "reward.npy"]
    for name, (t, _) in arrays.items():
        a = np.load(tmp_path / "whole" / f"{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, t.numpy().astype(np.float32)), name

    limit = 200 * (4 * (6 + 1 + 1 + 3) + 8)                   # room for 200 of the 1,000 envs
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, E, limit=limit)
    idx = np.load(tmp_path / "a" / "env_index.npy")
    assert idx.dtype == np.float64 and len(idx) == 200 and np.all(np.diff(idx) > 0) and 0 <= idx[0] and idx[-1] < E
    i = idx.astype(np.int64)
    assert i[-1] - i[0] > E // 2                              # spread over the batch, not its first rows
    for name, (t, ax) in arrays.items():
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert np.array_equal(a, b), name                     # the same sample every run
        assert np.array_equal(a, np.take(t.numpy(), i, axis=ax).astype(np.float32)), name
    assert sum(np.load(tmp_path / "a" / f).nbytes for f in os.listdir(tmp_path / "a")) <= limit


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_of_exactly_steps_timed_steps(tmp_path):
    """bench.py --dump-outputs writes what the last of its --steps timed steps returned (before the e2e leg reuses the
    env): the same seeded inputs stepped warmup + steps times after the pre-roll give the same bits."""
    steps, warmup = 4, 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c2", "--steps", str(steps), "--warmup",
                          str(warmup), "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["warmup"] == warmup and "e2e" in line
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= 64e6
    got = {n: np.load(tmp_path / f"{n}.npy") for n in ("obs", "reward", "done", "env_index")}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())

    ctx = bench.Ctx()
    E, A, W, F, c, obs, _ = bench.WORKLOADS["c2"]
    env = bench.make_env(ctx, E, A, W, F, c, 0)
    pool = bench.action_pool(ctx, E, A)
    env.reset(obs=True)
    for i in range(W):
        env.step(pool[i % 4], obs=False)
    for i in range(warmup + steps):
        o, r, d = env.step(pool[i % 4], obs=True)
    idx = torch.from_numpy(got["env_index"].astype(np.int64)).to(ctx.dev)
    assert got["obs"].shape == (len(idx), A, W, F)
    assert np.array_equal(got["obs"], o[idx].cpu().numpy())
    assert np.array_equal(got["reward"], r[idx].cpu().numpy())
    assert np.array_equal(got["done"], d[idx].float().cpu().numpy())
