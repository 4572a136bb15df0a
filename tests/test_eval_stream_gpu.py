"""Streaming evaluation metrics (BatchedTradingEnv.track_eval_metrics, pmrl_eval_stream_*) against the trace path
(`pmrl_eval_metrics` on the value / weight histories `loops.evaluate` builds) and an fp64 numpy restatement: return and
max drawdown bit-equal, Sharpe / Sortino / turnover within 1e-6 (fp64 sums taken in another order)."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RTOL = 1e-6
PERIODS = 252


def make_env(E, A, W, L=60, commission=0.0, reward="step_log", seed=1234, obs_dtype="float32", T=None, collect_stats=False):
    import pmrl_b200
    from pmrl_b200 import synth
    from pmrl_b200.env import BatchedTradingEnv
    T = T or (W + L + 64)
    tbl = synth.gbm_ohlc(T, A, seed)
    t0 = synth.episode_offsets(E, T, W, L)
    cfg = pmrl_b200.EnvConfig(num_envs=E, num_assets=A, window_size=W, num_features=5, commission=commission, reward=reward,
                              episode_len=L, obs_dtype=obs_dtype)
    return BatchedTradingEnv(cfg, prices=tbl, t0=t0, collect_stats=collect_stats)


def actions(steps, E, A, seed=7):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randn(E, A, generator=g, device="cuda") * 2.0 for _ in range(steps)]   # raw scores: softmax branch


def last_weights(env, rows=None):
    rows = torch.arange(env.E, device="cuda") if rows is None else rows
    return env.hist[rows, (env.idx[rows].long() - 1) % env.W]


class Trace:
    """What `loops.evaluate(traces=True)` keeps: value and last-weight rows of every call, and the rewards."""

    def __init__(self, env, rows=None):
        self.env, self.rows = env, rows
        self.v, self.w, self.r = [], [], []

    def record(self, r=None):
        rows = self.rows
        self.v.append((self.env.value if rows is None else self.env.value[rows]).clone())
        self.w.append(last_weights(self.env, rows).clone())
        self.r.append(None if r is None else (r if rows is None else r[rows]).clone())

    def metrics(self, calls, rf=0.0):
        """(total [n], trace metrics [n, 4], values [n, N] f64, weights [n, N, A] f64) over the given call indices."""
        from pmrl_b200.metrics import eval_metrics
        V = torch.stack([self.v[c] for c in calls], 1)
        Wt = torch.stack([self.w[c] for c in calls], 1)
        total = torch.zeros_like(self.v[0])
        for c in calls[1:]:
            total += self.r[c]
        return total, eval_metrics(V, Wt, rf=rf, periods=PERIODS), V.double().cpu().numpy(), Wt.double().cpu().numpy()


def same_bits(a, b):
    a, b = torch.as_tensor(a).float(), torch.as_tensor(b).float()
    return bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())


def numpy_metrics(v, w, rf=0.0):
    r = v[:, 1:] / v[:, :-1] - 1 - ((1.0 + rf) ** (1 / PERIODS) - 1 if rf else 0.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        sharpe = r.mean(1) / r.std(1, ddof=1) * np.sqrt(PERIODS)
        sortino = r.mean(1) / np.sqrt((np.minimum(r, 0) ** 2).sum(1) / r.shape[1]) * np.sqrt(PERIODS)
    mdd = (v / np.maximum.accumulate(v, axis=1)).min(1) - 1
    to = np.abs(np.diff(w, axis=1)).sum(-1).mean(1)
    return np.stack([sharpe, sortino, mdd, to], 1)


def assert_matches_trace(got, total, want, msg=""):
    """got [n, 5] streaming rows vs the trace path's total [n] and metrics [n, 4]."""
    got, want = got.cpu(), want.cpu()
    assert same_bits(got[:, 0], total.cpu()), f"{msg}: return differs"
    assert same_bits(got[:, 3], want[:, 2]), f"{msg}: max drawdown differs"
    for j, k, name in ((1, 0, "sharpe"), (2, 1, "sortino"), (4, 3, "turnover")):
        np.testing.assert_allclose(got[:, j].numpy(), want[:, k].numpy(), rtol=RTOL, atol=0, equal_nan=True, err_msg=f"{msg}: {name}")


def assert_matches_numpy(got, v, w, rf=0.0, msg=""):
    ref = numpy_metrics(v, w, rf)
    got = got.cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(got[:, 1], ref[:, 0], rtol=1e-4, equal_nan=True, err_msg=f"{msg}: sharpe vs numpy")
    np.testing.assert_allclose(got[:, 2], ref[:, 1], rtol=1e-4, equal_nan=True, err_msg=f"{msg}: sortino vs numpy")
    np.testing.assert_allclose(got[:, 3], ref[:, 2], rtol=1e-5, atol=1e-6, err_msg=f"{msg}: mdd vs numpy")
    np.testing.assert_allclose(got[:, 4], ref[:, 3], rtol=1e-5, err_msg=f"{msg}: turnover vs numpy")


def acc_bytes(m):
    return m.acc.cpu().numpy().tobytes()


# (A, W, commission, reward, obs, rf): every A / W / commission / reward mode and obs on and off
SHAPES = [
    (11, 2, 0.0, "step_log", True, 0.0),
    (11, 50, 0.0025, "returns", False, 0.04),
    (50, 5, 0.0, "log_returns", True, 0.0),
    (50, 50, 0.0025, "sharpe_ratio", True, 0.04),
    (100, 50, 0.0, "step_log", True, 0.04),
    (100, 2, 0.0025, "sharpe_ratio", False, 0.0),
    (100, 5, 0.0025, "returns", True, 0.0),
    (500, 50, 0.0025, "step_log", False, 0.0),
    (500, 5, 0.0, "log_returns", True, 0.04),
    (500, 2, 0.0, "returns", True, 0.0),
]


@pytest.mark.parametrize("A,W,c,reward,obs,rf", SHAPES)
def test_running_matches_the_trace_path(A, W, c, reward, obs, rf):
    E, steps = 37, 30
    env = make_env(E, A, W, L=40, commission=c, reward=reward)
    m = env.track_eval_metrics(rf=rf, periods=PERIODS)
    tr = Trace(env)
    env.reset(obs=obs)
    tr.record()
    for a in actions(steps, E, A):
        _, r, _ = env.step(a, obs=obs)
        tr.record(r)
    got, count = m.running()
    total, want, v, w = tr.metrics(list(range(steps + 1)), rf=rf)
    assert_matches_trace(got, total, want, f"A={A} W={W}")
    assert_matches_numpy(got, v, w, rf, f"A={A} W={W}")
    assert int(count.sum()) == 0


def test_episode_records_match_each_episodes_segment():
    E, A, W, L, calls = 29, 50, 5, 7, 40
    env = make_env(E, A, W, L=L, commission=0.0025)
    m = env.track_eval_metrics()
    tr = Trace(env)
    env.reset(obs=False)
    tr.record()
    records, dones = [], torch.zeros(E, dtype=torch.int32, device="cuda")
    for k, a in enumerate(actions(calls, E, A), start=1):
        _, r, d = env.step(a, obs=False)
        tr.record(r)
        dones += d.int()
        if bool(d.any()):
            assert bool(d.all())                              # lockstep episodes: every env ends on the same call
            records.append((k, *m.last_episode()))
    assert [k for k, _, _ in records] == [7, 15, 23, 31, 39]  # calls 8, 16, ... are the auto-resets
    for j, (k, rec, count) in enumerate(records):
        total, want, v, w = tr.metrics(list(range(k - L, k + 1)))
        assert_matches_trace(rec, total, want, f"episode {j}")
        assert_matches_numpy(rec, v, w, msg=f"episode {j}")
        assert bool((count == j + 1).all())
    mean, count = m.episode_mean()
    assert torch.equal(count, dones)
    recs = np.stack([rec.cpu().numpy().astype(np.float64) for _, rec, _ in records])
    np.testing.assert_allclose(mean.cpu().numpy(), recs.mean(0), rtol=RTOL)
    running, _ = m.running()                                  # call 40 auto-reset every env: an empty running episode
    assert bool((running[:, 0] == 0).all()) and bool((running[:, 3] == 0).all())
    assert bool(torch.isnan(running[:, [1, 2, 4]]).all())


def test_masked_reset_restarts_only_the_masked_envs():
    E, A, W = 24, 11, 8
    env = make_env(E, A, W, L=50)
    m = env.track_eval_metrics()
    tr = Trace(env)
    acts = actions(9, E, A)
    env.reset()
    tr.record()
    for k in range(5):
        _, r, _ = env.step(acts[k])
        tr.record(r)
    mask = (torch.arange(E) % 3 == 0).to(torch.uint8)
    env.reset(mask=mask)                                          # call 6
    tr.record(torch.zeros(E, device="cuda"))
    for k in range(5, 9):
        _, r, _ = env.step(acts[k])
        tr.record(r)
    got, _ = m.running()
    sel = mask.bool().cuda()
    total, want, v, w = tr.metrics([6, 7, 8, 9, 10])
    assert_matches_trace(got[sel], total[sel], want[sel], "masked envs")
    total, want, v, w = tr.metrics([0, 1, 2, 3, 4, 5, 7, 8, 9, 10])
    assert_matches_trace(got[~sel], total[~sel], want[~sel], "unmasked envs")


def test_a_missed_update_invalidates_only_that_env_until_its_reset():
    from pmrl_b200 import _lib
    E, A, W, k = 16, 50, 5, 5
    env, twin = make_env(E, A, W), make_env(E, A, W)
    m, mt = env.track_eval_metrics(), twin.track_eval_metrics()
    acts = actions(8, E, A)
    for e in (env, twin):
        e.reset(obs=False)
        for a in acts[:3]:
            e.step(a, obs=False)
    # envs [0, k) take one step through the C-ABI with no update after it
    c = env._c_cfg
    sub = _lib.PmrlEnvCfg(k, c.A, c.W, c.F, c.T, c.episode_len, c.reward_mode, c.mu_max_iter, c.flags, c.initial_cash,
                          c.commission, c.reward_scale, c.risk_free)
    rc = env.lib.pmrl_env_step(ctypes.byref(sub), env._p_tbl, env._p_st, acts[3].data_ptr(), None, env.reward.data_ptr(),
                               env.done.data_ptr(), None, 0, None, _lib.current_stream())
    assert rc == 0
    got, _ = m.running()
    assert bool(torch.isnan(got[:k]).all())                       # stepped since the last update: not trusted
    assert bool(torch.isfinite(got[k:, 3]).all())
    env.step(acts[4], obs=False)
    twin.step(acts[4], obs=False)
    got, _ = m.running()
    assert bool(torch.isnan(got[:k]).all())
    assert acc_bytes(m)[k * 128:] == acc_bytes(mt)[k * 128:]      # the other envs are untouched
    mask = torch.zeros(E, dtype=torch.uint8)
    mask[:k] = 1
    env.reset(mask=mask, obs=False)
    got, _ = m.running()
    assert bool((got[:k, 0] == 0).all()) and bool((got[:k, 3] == 0).all()) and bool(torch.isnan(got[:k, 1]).all())
    env.step(acts[5], obs=False)
    env.step(acts[6], obs=False)
    got, _ = m.running()
    assert bool(torch.isfinite(got[:k, [0, 3, 4]]).all())


def test_a_zeroed_accumulator_that_first_sees_a_step_reads_nan():
    E, A, W = 8, 11, 4
    env = make_env(E, A, W)
    acts = actions(4, E, A)
    env.step(acts[0], obs=False)
    m = env.track_eval_metrics()                                  # enabled mid-episode
    env.step(acts[1], obs=False)
    assert bool(torch.isnan(m.running()[0]).all())
    env.reset(obs=False)
    env.step(acts[2], obs=False)
    assert bool(torch.isfinite(m.running()[0][:, [0, 3, 4]]).all())
    m.clear()
    env.step(acts[3], obs=False)
    out, count = m.running()
    assert bool(torch.isnan(out).all()) and int(count.sum()) == 0
    assert bool(torch.isnan(m.last_episode()[0]).all()) and bool(torch.isnan(m.episode_mean()[0]).all())


# ------------------------------------------------------------------------------------------------ dispatch paths
def run_eager(env, acts, obs=True):
    m = env.track_eval_metrics()
    env.reset(obs=obs)
    for a in acts:
        env.step(a, obs=obs)
    return m


@pytest.mark.parametrize("A,W,L", [(100, 50, 12), (11, 5, 9), (500, 8, 12)])
def test_every_step_path_leaves_the_same_accumulator(A, W, L):
    E, steps = 33, 30
    acts = actions(steps, E, A)
    ref = acc_bytes(run_eager(make_env(E, A, W, L=L, commission=0.0025), acts))

    env = make_env(E, A, W, L=L, commission=0.0025)
    m = env.track_eval_metrics()
    env.reset()
    rew = torch.empty(E, device="cuda"); dn = torch.empty(E, dtype=torch.uint8, device="cuda")
    vs = torch.empty(E, device="cuda"); ws = torch.empty(E, A, device="cuda")
    for a in acts:
        env.step_io(a, reward=rew, done=dn, value_sink=vs, weight_sink=ws, action_sink=torch.empty(E, A, device="cuda"))
    assert acc_bytes(m) == ref, "step_io"

    env = make_env(E, A, W, L=L, commission=0.0025)
    m = env.track_eval_metrics()
    env.reset()
    for a in acts:
        env.step_host(a.cpu().pin_memory())
    assert acc_bytes(m) == ref, "step_host"

    for K in (1, 15):
        env = make_env(E, A, W, L=L, commission=0.0025)
        m = env.track_eval_metrics()
        env.reset()
        static, replay = env.graphed_step(steps=K)
        for i in range(0, steps, K):
            if K == 1:
                static.copy_(acts[i])
            else:
                static.copy_(torch.stack(acts[i:i + K]))
            replay()
        assert acc_bytes(m) == ref, f"graphed_step(steps={K})"

    env = make_env(E, A, W, L=L, commission=0.0025, obs_dtype="bfloat16")
    assert acc_bytes(run_eager(env, acts)) == ref, "bf16 obs"


def test_step_burst_refuses_while_tracking():
    from pmrl_b200._lib import PmrlError
    E, A, W = 8, 11, 4
    env = make_env(E, A, W)
    env.step_burst(torch.randn(3, E, A, device="cuda"))           # allowed before tracking
    env.track_eval_metrics()
    with pytest.raises(PmrlError, match="track_eval_metrics"):
        env.step_burst(torch.randn(3, E, A, device="cuda"))


def test_two_tracked_envs_on_two_streams_stay_independent():
    E, A, W, steps = 64, 100, 50, 20
    a1, a2 = actions(steps, E, A, seed=1), actions(steps, E, A, seed=2)
    ref1 = acc_bytes(run_eager(make_env(E, A, W, L=9), a1))
    ref2 = acc_bytes(run_eager(make_env(E, A, W, L=9, seed=99), a2))
    e1, e2 = make_env(E, A, W, L=9), make_env(E, A, W, L=9, seed=99)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    s1.wait_stream(torch.cuda.current_stream()); s2.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s1):
        m1 = e1.track_eval_metrics(); e1.reset()
    with torch.cuda.stream(s2):
        m2 = e2.track_eval_metrics(); e2.reset()
    for k in range(steps):
        with torch.cuda.stream(s1):
            e1.step(a1[k])
        with torch.cuda.stream(s2):
            e2.step(a2[k])
    torch.cuda.synchronize()
    assert acc_bytes(m1) == ref1 and acc_bytes(m2) == ref2


# ------------------------------------------------------------------------------------------------ full size
def test_full_size_c4_shard_with_obs():
    import bench
    E, A, W, steps, S = 131072, 100, 50, 60, 512
    env = make_env(E, A, W, L=bench.EPISODE_LEN, T=bench.TABLE_ROWS)
    acts = actions(4, E, A)
    env.reset()
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    m = env.track_eval_metrics()
    rows = torch.randperm(E, generator=torch.Generator().manual_seed(5))[:S].cuda()
    env.reset()
    v, w, rs = [env.value[rows].clone()], [last_weights(env, rows).clone()], []
    for k in range(steps):
        _, r, _ = env.step(acts[k % 4])
        v.append(env.value[rows].clone()); w.append(last_weights(env, rows).clone()); rs.append(r[rows].clone())
    torch.cuda.synchronize()
    extra = torch.cuda.memory_allocated() - before - sum(t.numel() * t.element_size() for t in v + w + rs) - rows.numel() * 8
    assert extra <= 128 * E, f"tracker holds {extra} bytes for {E} envs"
    got, _ = m.running()
    from pmrl_b200.metrics import eval_metrics
    want = eval_metrics(torch.stack(v, 1), torch.stack(w, 1), periods=PERIODS)
    total = torch.zeros(S, device="cuda")
    for r in rs:
        total += r
    assert_matches_trace(got[rows], total, want, "c4_shard sample")
    assert bool(torch.isfinite(got[:, [0, 1, 3, 4]]).all())


# ------------------------------------------------------------------------------------------------ loops.evaluate
@pytest.mark.parametrize("num_items,L,rf", [(50, 60, 0.0), (31, 30, 0.04)])
def test_evaluate_without_traces_equals_with_traces(num_items, L, rf):
    from pmrl_b200 import loops
    E, A, W = 40, 11, 8
    proj = torch.randn(W * 5, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3)) * 2e-3

    def act_fn(s):
        return s.reshape(E, A, W * 5) @ proj
    tot_t, met_t = loops.evaluate(make_env(E, A, W, L=L), act_fn, num_items, rf=rf, traces=True)
    tot_s, met_s = loops.evaluate(make_env(E, A, W, L=L), act_fn, num_items, rf=rf, traces=False)
    assert tot_s.shape == (E,) and met_s.shape == (E, 4)
    assert_matches_trace(torch.cat([tot_s[:, None], met_s], 1), tot_t, met_t, "evaluate")
