"""Randomised episode starts (BatchedTradingEnv.sample_episode_starts, pmrl_env_draw_starts) against the CPU statement of
the draw (oracle/starts_oracle.py) and the CPU env oracle with its t0 overwritten from those draws."""
import numpy as np
import pytest
import torch

from oracle import starts_oracle as so
from tests.util import assert_rewards_close, assert_values_close

pytestmark = pytest.mark.gpu


def tables(T, A, F, seed=1234):
    from pmrl_b200 import synth
    tbl = synth.gbm_ohlc(T, A, seed)
    feats = tbl
    if F != 5:                                                  # OHLC + seeded extra channels
        g = torch.Generator().manual_seed(seed + 1)
        feats = torch.cat([tbl, torch.rand(T, A, F - 5, generator=g)], dim=-1)
    return tbl, feats


def make_env(E, A, W, L, F=5, c=0.0, T=None, seed=1234, first_env=0, obs_dtype="float32", t0=None):
    import pmrl_b200
    from pmrl_b200 import synth
    from pmrl_b200.env import BatchedTradingEnv
    T = T or (W + 4 * L + 64)
    tbl, feats = tables(T, A, F, seed)
    if t0 is None:
        t0 = synth.episode_offsets(E, T, W, L, first_env=first_env)
    cfg = pmrl_b200.EnvConfig(num_envs=E, num_assets=A, window_size=W, num_features=F, commission=c, episode_len=L,
                              obs_dtype=obs_dtype)
    return BatchedTradingEnv(cfg, prices=tbl, features=feats if F != 5 else None, t0=t0)


def actions(steps, E, A, seed=7):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randn(E, A, generator=g, device="cuda") * 2.0 for _ in range(steps)]


def host(t):
    return t.detach().cpu().numpy()


def u32(t):
    return host(t).astype(np.int64) & so.MASK32


class Ref:
    """The CPU side of a sampler: t0 / draw counters advanced by the oracle's draw."""

    def __init__(self, env, s, kind, beta=None):
        self.kind, self.lo, self.hi, self.beta = kind, s.low, s.high, beta
        self.seed, self.base = s.dist.seed, s.dist.env_base
        self.t0, self.ep = host(env.t0).astype(np.int32), np.zeros(env.E, np.int64)
        self.q = np.full(env.E, np.nan)

    def draw(self, select):
        self.t0, self.ep, q = so.draw(self.kind, self.lo, self.hi, self.seed, self.base, self.t0, self.ep, select, self.beta)
        self.q = np.where(np.asarray(select, bool), q, self.q)


def assert_draws_equal(env, s, ref, msg=""):
    got = host(env.t0).astype(np.int64)
    assert np.array_equal(u32(s.episodes), ref.ep), f"{msg}: draw counters"
    bad = got != ref.t0
    if ref.kind == so.GEOMETRIC and bad.any():
        # the device's fp64 log1p may differ from the host's in the last bit: only a quotient within 1e-9 of an integer
        # may then floor one apart
        q = ref.q[bad]
        near = np.abs(q - np.round(q)) < 1e-9
        assert near.all() and (np.abs(got[bad] - ref.t0[bad]) == 1).all(), f"{msg}: geometric draws differ"
    else:
        assert not bad.any(), f"{msg}: t0 differs at {np.flatnonzero(bad)[:5]}: {got[bad][:5]} vs {ref.t0[bad][:5]}"


# ------------------------------------------------------------------------------------------------ draws
@pytest.mark.parametrize("E", [1, 37, 4096])
@pytest.mark.parametrize("distribution", ["uniform", "geometric"])
def test_mask_and_due_draws_equal_the_reference(E, distribution):
    W, L = 5, 7
    kind, beta = (so.UNIFORM, None) if distribution == "uniform" else (so.GEOMETRIC, 0.01)
    for seed, first_env in ((0, 0), (12345, 1000), ((1 << 64) - 1, (1 << 33) + 5)):
        env = make_env(E, 11, W, L, T=600)
        s = env.sample_episode_starts(seed=seed, distribution=distribution, beta=beta, first_env=first_env)
        ref = Ref(env, s, kind, beta)
        assert ref.hi == 600 - L - W
        g = torch.Generator().manual_seed(seed % 1000 + E)
        for _ in range(3):                                      # masked draws: only the masked envs move
            mask = (torch.rand(E, generator=g) < 0.5).to(torch.uint8)
            before = host(env.t0).copy()
            s.draw_mask(mask.cuda())
            ref.draw(mask.numpy())
            assert_draws_equal(env, s, ref, f"mask seed={seed}")
            assert np.array_equal(host(env.t0)[mask.numpy() == 0], before[mask.numpy() == 0])
        s.draw_mask(None)
        ref.draw(np.ones(E, bool))
        assert_draws_equal(env, s, ref, f"all seed={seed}")
        for _ in range(3):                                      # due draws on arbitrary local steps
            t = torch.randint(0, L + 3, (E,), generator=g, dtype=torch.int32)
            env.t.copy_(t)
            t0_before, ep_before = env.t0.clone(), s.episodes.clone()
            s.draw_due()
            ref.draw(so.due(t.numpy(), L))
            assert_draws_equal(env, s, ref, f"due seed={seed}")
            keep = torch.from_numpy(~so.due(t.numpy(), L)).cuda()
            assert torch.equal(env.t0[keep], t0_before[keep]) and torch.equal(s.episodes[keep], ep_before[keep])
            assert bool((env.t0 >= s.low).all()) and bool((env.t0 <= s.high).all())


# ------------------------------------------------------------------------------------------------ trajectories
@pytest.mark.parametrize("A", [11, 100, 500])
@pytest.mark.parametrize("W", [2, 50])
@pytest.mark.parametrize("F", [5, 7])
@pytest.mark.parametrize("c", [0.0, 0.0025])
def test_trajectories_match_the_oracle_with_drawn_starts(A, W, F, c):
    from oracle.env_oracle import OracleEnv
    E, L, T = 19, 4, 160
    episodes = 3
    steps = episodes * (L + 1)
    env = make_env(E, A, W, L, F=F, c=c, T=T)
    tbl, feats = tables(T, A, F)
    ora = OracleEnv(E, A, W, F, close=tbl[:, :, 3].numpy(), feat=feats.numpy(), t0=host(env.t0), episode_len=L,
                    commission=c)
    s = env.sample_episode_starts(seed=31 + A, low=3, first_env=7)
    ref = Ref(env, s, so.UNIFORM)
    obs = env.reset()
    ref.draw(np.ones(E, bool))
    ora.t0 = ref.t0.copy(); ora.reset()
    np.testing.assert_array_equal(host(env.t0), ref.t0)
    np.testing.assert_array_equal(host(obs)[..., :F - 1], ora.obs()[..., :F - 1])
    idx = torch.empty(E, dtype=torch.int32, device="cuda")
    resets = 0
    for k, a in enumerate(actions(steps, E, A)):
        due = so.due(ora.t, L)
        resets += int(due.any())
        ref.draw(due)
        ora.t0 = ref.t0.copy()
        obs, r, d = env.step_io(a, index_sink=idx)
        r_o, d_o = ora.step(host(a))
        msg = f"A={A} W={W} F={F} c={c} step {k}"
        np.testing.assert_array_equal(host(env.t0), ref.t0, err_msg=msg)
        np.testing.assert_array_equal(u32(s.episodes), ref.ep, err_msg=msg)
        np.testing.assert_array_equal(host(idx), ora.t0 + ora.t, err_msg=msg)
        got = host(obs)
        want = ora.obs()
        np.testing.assert_array_equal(got[..., :F - 1], want[..., :F - 1], err_msg=msg)
        np.testing.assert_allclose(got[..., F - 1], want[..., F - 1], rtol=1e-5, atol=1e-6, err_msg=msg)
        assert_rewards_close(host(r), r_o, msg)
        assert_values_close(host(env.value), ora.value, msg)
        np.testing.assert_array_equal(host(d), d_o, err_msg=msg)
    assert resets == episodes                                  # the last call is the third auto-reset
    assert (ref.ep == episodes + 1).all()


# ------------------------------------------------------------------------------------------------ dispatch paths
E_D, STEPS, L_D = 33, 30, 6


def _run(env, mode, acts, obs=True):
    """Drive one env through `mode`; returns the bytes that must not depend on the dispatch path."""
    s = env.sample_episode_starts(seed=99, first_env=11)
    env.reset(obs=obs)
    rewards, last = [], None
    if mode.startswith("graphed"):
        K = int(mode[len("graphed"):])
        static, replay = env.graphed_step(obs=obs, steps=K)
        for i in range(0, len(acts), K):
            static.copy_(acts[i] if K == 1 else torch.stack(acts[i:i + K]))
            last, r, _ = replay()
            rewards += [r.clone()] if K == 1 else [r[k].clone() for k in range(K)]
    else:
        for a in acts:
            if mode == "step":
                last, r, _ = env.step(a, obs=obs)
            elif mode == "step_io":
                last, r, _ = env.step_io(a, obs=obs, reward=torch.empty(env.E, device="cuda"),
                                         done=torch.empty(env.E, dtype=torch.uint8, device="cuda"),
                                         index_sink=torch.empty(env.E, dtype=torch.int32, device="cuda"))
            elif mode in ("host_zero_copy", "host_sliced"):
                last, r, _ = env.step_host(a.cpu().pin_memory(), obs=obs, chunks=0 if mode == "host_zero_copy" else 3)
            rewards.append(r.clone().cuda())
    torch.cuda.synchronize()
    out = {"value": env.value, "hist": env.hist, "idx": env.idx, "is_full": env.is_full, "t": env.t, "t0": env.t0,
           "ep_return": env.ep_return, "episodes": s.episodes, "rewards": torch.stack(rewards)}
    out = {k: host(v).tobytes() for k, v in out.items()}
    if obs:
        out["obs"] = last.clone()
    return out


def _same(got, ref, what):
    for k, v in ref.items():
        if k == "obs":                                          # a bf16 env's obs is the bf16 rounding of the fp32 obs
            assert torch.equal(got[k], v.to(got[k].dtype)), f"{what}: obs"
        else:
            assert got[k] == v, f"{what}: {k}"


@pytest.mark.parametrize("A,W", [(100, 50), (11, 5), (500, 8)])
def test_every_dispatch_path_gives_the_same_run(A, W):
    from pmrl_b200 import _lib
    acts = actions(STEPS, E_D, A)
    mk = lambda **kw: make_env(E_D, A, W, L_D, c=0.0025, **kw)   # noqa: E731
    ref = _run(mk(), "step", acts)
    for mode in ("step_io", "host_zero_copy", "host_sliced", "graphed1", "graphed15"):
        _same(_run(mk(), mode, acts), ref, mode)
    _same(_run(mk(obs_dtype="bfloat16"), "step", acts), ref, "bf16 obs")
    # the fallbacks the tuning keys select (their default is 1: fused kernel, TMA ring loads, staged wide step when large)
    for key, value, what in ((_lib.TUNE_FUSED, 0, "two-kernel step + obs"), (_lib.TUNE_RING_TMA, 0, "register-ring fused")):
        _lib.set_tuning(key, value)
        try:
            _same(_run(mk(), "step", acts), ref, what)
        finally:
            _lib.set_tuning(key, 1)
    if A > 128 and A % 4 == 0:                                  # the staged wide-env state-only step, at this small batch too
        ref_s = _run(mk(), "step", acts, obs=False)
        _lib.set_tuning(_lib.TUNE_STAGED, 2)
        try:
            _same(_run(mk(), "step", acts, obs=False), ref_s, "staged wide-A step")
        finally:
            _lib.set_tuning(_lib.TUNE_STAGED, 1)


def test_two_half_batches_reproduce_the_whole_batch():
    E, A, W, L = 64, 50, 8, 5
    acts = actions(20, E, A)
    whole = make_env(E, A, W, L)
    sw = whole.sample_episode_starts(seed=5, first_env=0)
    halves = [make_env(E // 2, A, W, L, first_env=b) for b in (0, E // 2)]
    sh = [h.sample_episode_starts(seed=5, first_env=b) for h, b in zip(halves, (0, E // 2))]
    assert torch.equal(torch.cat([h.t0 for h in halves]), whole.t0)
    whole.reset()
    for h in halves:
        h.reset()
    for a in acts:
        _, r, _ = whole.step(a)
        rh = [h.step(a[i * (E // 2):(i + 1) * (E // 2)].contiguous())[1].clone() for i, h in enumerate(halves)]
        assert torch.equal(torch.cat(rh), r)
    for name in ("t0", "value", "t", "idx", "hist"):
        assert torch.equal(torch.cat([getattr(h, name) for h in halves]), getattr(whole, name)), name
    assert torch.equal(torch.cat([s.episodes for s in sh]), sw.episodes)
    assert int(sw.episodes.min()) == 1 + 20 // (L + 1)


def test_masked_reset_draws_exactly_the_masked_envs():
    E, A, W, L = 40, 11, 4, 9
    env = make_env(E, A, W, L)
    s = env.sample_episode_starts(seed=3)
    ref = Ref(env, s, so.UNIFORM)
    mask = (torch.arange(E) % 3 == 1).to(torch.uint8)
    for a in actions(3, E, A):
        env.step(a)
    t_before = env.t.clone()
    obs = env.reset(mask=mask)
    ref.draw(mask.numpy() == 1)
    np.testing.assert_array_equal(host(env.t0), ref.t0)
    np.testing.assert_array_equal(u32(s.episodes), ref.ep)
    sel = mask.bool().cuda()
    assert bool((env.t[sel] == 0).all()) and torch.equal(env.t[~sel], t_before[~sel])
    tbl, _ = tables(W + 4 * L + 64, A, 5)
    for e in torch.nonzero(sel).flatten().tolist():             # the reset obs of a masked env starts at its new t0
        r0 = int(ref.t0[e])
        np.testing.assert_array_equal(host(obs[e])[..., :4], tbl[r0:r0 + W].permute(1, 0, 2).numpy())


def test_the_last_offset_reads_the_last_table_row():
    E, A, W, L, T = 8, 11, 6, 5, 80
    env = make_env(E, A, W, L, T=T)
    s = env.sample_episode_starts(low=T - L - W, seed=1)            # high defaults to T - L - W: one admissible offset
    assert s.low == s.high == T - L - W
    env.reset()
    tbl, _ = tables(T, A, 5)
    idx = torch.empty(E, dtype=torch.int32, device="cuda")
    for k, a in enumerate(actions(L, E, A), start=1):
        obs, _, d = env.step_io(a, index_sink=idx)
    assert bool(d.all()) and bool((idx == T - W).all())             # item index t0 + L
    np.testing.assert_array_equal(host(obs)[..., :4], np.broadcast_to(tbl[T - W:T].permute(1, 0, 2).numpy(), (E, A, W, 4)))


@pytest.mark.parametrize("distribution,beta", [("uniform", None), ("geometric", 0.05)])
def test_distributions_over_a_million_draws(distribution, beta):
    from scipy import stats
    E, draws, lo, hi = 1 << 16, 16, 20, 119                         # 2^20 draws over 100 offsets
    env = make_env(E, 2, 2, 1, T=200)
    s = env.sample_episode_starts(low=lo, high=hi, seed=2024, distribution=distribution, beta=beta)
    counts = torch.zeros(hi - lo + 1, dtype=torch.int64, device="cuda")
    for _ in range(draws):
        s.draw_mask(None)
        counts += torch.bincount((env.t0 - lo).long(), minlength=hi - lo + 1)
    counts = host(counts).astype(np.float64)
    assert counts.sum() == E * draws
    j = np.arange(hi - lo + 1)
    if distribution == "uniform":
        p = np.full(len(j), 1.0 / len(j))
    else:
        p = beta * (1 - beta) ** (hi - lo - j)                       # offset lo + j is j' = hi - lo - j rows before hi
        p /= p.sum()
    _, pval = stats.chisquare(counts, counts.sum() * p)
    assert pval > 1e-4, f"{distribution}: chi-square p = {pval}"
    assert bool((s.episodes == draws).all())


def test_step_burst_refuses_while_sampling_and_works_after_detach():
    from pmrl_b200._lib import PmrlError
    E, A, W, L = 8, 11, 4, 3
    env = make_env(E, A, W, L)
    s = env.sample_episode_starts(seed=1)
    env.reset()
    with pytest.raises(PmrlError, match="sample_episode_starts"):
        env.step_burst(torch.randn(5, E, A, device="cuda"))
    t0 = env.t0.clone()
    s.detach()
    env.step_burst(torch.randn(5, E, A, device="cuda"))             # crosses an episode end: offsets are kept
    env.reset()
    assert torch.equal(env.t0, t0) and bool((s.episodes == 1).all())


def test_one_extra_launch_per_call_with_a_sampler_and_none_without():
    E, A, W, L = 16, 11, 4, 3
    plain, sampled, detached = make_env(E, A, W, L), make_env(E, A, W, L), make_env(E, A, W, L)
    sampled.sample_episode_starts(seed=1)
    detached.sample_episode_starts(seed=1).detach()
    lib = plain.lib
    a = torch.randn(E, A, device="cuda")
    idx = torch.empty(E, dtype=torch.int32, device="cuda")
    calls = {"reset": lambda env: env.reset(), "reset_mask": lambda env: env.reset(mask=torch.ones(E, dtype=torch.uint8)),
             "step": lambda env: env.step(a), "step_state": lambda env: env.step(a, obs=False),
             "step_io": lambda env: env.step_io(a, index_sink=idx), "step_host": lambda env: env.step_host(a.cpu().pin_memory())}
    for name, call in calls.items():
        n = {}
        for key, env in (("plain", plain), ("sampled", sampled), ("detached", detached)):
            c0 = lib.pmrl_launch_count()
            call(env)
            n[key] = lib.pmrl_launch_count() - c0
        assert n["sampled"] == n["plain"] + 1 and n["detached"] == n["plain"], f"{name}: {n}"


def test_episode_returns_with_eval_metrics_equal_the_step_reward_sums():
    E, A, W, L = 24, 50, 8, 5
    env = make_env(E, A, W, L, c=0.0025)
    env.sample_episode_starts(seed=8, distribution="geometric", beta=0.02)
    m = env.track_eval_metrics()
    env.reset()
    total = torch.zeros(E, device="cuda")
    ends = 0
    for a in actions(3 * (L + 1), E, A):
        _, r, d = env.step(a)
        total += r
        if bool(d.any()):
            assert bool(d.all())
            rec, count = m.last_episode()
            assert torch.equal(rec[:, 0], total), "episode return"
            assert bool(torch.isfinite(rec[:, 1:]).all())
            ends += 1
            assert bool((count == ends).all())
            total.zero_()
    assert ends == 3


def test_full_size_c4_shard_crosses_an_episode_boundary():
    import bench
    E, A, W, L, S = 131072, 100, 50, 3, 256
    T = bench.TABLE_ROWS
    env = make_env(E, A, W, L, T=T)
    s = env.sample_episode_starts(seed=11)
    env.reset()
    t0_first = host(env.t0)
    acts = actions(2, E, A)
    for k in range(L + 1):                                         # L steps, then the auto-reset call
        obs, _, d = env.step(acts[k % 2])
    torch.cuda.synchronize()
    assert bool((env.t == 0).all()) and bool((s.episodes == 2).all())
    t0 = host(env.t0)
    rows = np.random.default_rng(5).choice(E, S, replace=False)
    for e in rows:
        assert t0_first[e] == so.draw_one(so.UNIFORM, 0, T - L - W, 11, int(e), 0)[0]
        assert t0[e] == so.draw_one(so.UNIFORM, 0, T - L - W, 11, int(e), 1)[0]
    tbl, _ = tables(T, A, 5)
    got = host(obs[torch.from_numpy(rows).cuda()])[..., :4]
    want = np.stack([tbl[r:r + W].permute(1, 0, 2).numpy() for r in t0[rows]])
    np.testing.assert_array_equal(got, want)
    assert len(np.unique(t0)) > 2000                               # the batch now covers many windows, not 131,072 fixed ones


def test_observe_after_a_done_step_shows_the_finished_episode():
    """t0 is redrawn at the call after a done step, so observe() in between still shows the finished episode's window."""
    E, A, W, L = 12, 11, 5, 4
    env = make_env(E, A, W, L)
    s = env.sample_episode_starts(seed=21)
    env.reset()
    t0_episode = env.t0.clone()
    for a in actions(L, E, A):
        obs, _, d = env.step(a)
    assert bool(d.all())
    done_obs = obs.clone()
    assert torch.equal(env.observe(out=torch.empty_like(done_obs)), done_obs)
    assert torch.equal(env.t0, t0_episode) and bool((s.episodes == 1).all())
    env.step(actions(1, E, A, seed=8)[0])                          # the auto-reset call draws the next start
    assert bool((s.episodes == 2).all()) and bool((env.t == 0).all())
    ref = Ref(env, s, so.UNIFORM)
    ref.ep[:] = 1
    ref.draw(np.ones(E, bool))
    np.testing.assert_array_equal(host(env.t0), ref.t0)


def test_a_batch_larger_than_the_grid_walks_every_env():
    """More envs than the launch's threads (SMs x 8 blocks x 256): the grid-stride loop takes several passes."""
    from pmrl_b200._lib import load
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    E, W, L, T = 1 << 20, 2, 1, 64
    assert E > sms * 8 * 256
    env = make_env(E, 2, W, L, T=T)
    s = env.sample_episode_starts(seed=77, first_env=3)
    n = load().pmrl_launch_count()
    s.draw_mask(None)
    assert load().pmrl_launch_count() == n + 1
    assert bool((s.episodes == 1).all())
    t = torch.randint(0, L + 2, (E,), generator=torch.Generator().manual_seed(4), dtype=torch.int32)
    env.t.copy_(t)
    s.draw_due()
    due = host(t) >= L
    assert np.array_equal(u32(s.episodes), 1 + due.astype(np.int64))
    rows = np.unique(np.concatenate([np.arange(64), np.arange(E - 64, E),
                                     np.random.default_rng(1).choice(E, 1024, replace=False),
                                     np.arange(sms * 8 * 256 - 32, sms * 8 * 256 + 32)]))
    t0 = host(env.t0)
    for e in rows:
        want = so.draw_one(so.UNIFORM, 0, T - L - W, 77, 3 + int(e), 1 if due[e] else 0)[0]
        assert t0[e] == want, f"env {e}"


@pytest.mark.parametrize("bad", ["short", "long", "dtype", "host"])
def test_draw_mask_refuses_a_mask_that_does_not_fit_the_batch(bad):
    E = 16
    env = make_env(E, 11, 4, 3)
    s = env.sample_episode_starts(seed=1)
    mask = {"short": torch.ones(E - 1, dtype=torch.uint8, device="cuda"),
            "long": torch.ones(E + 1, dtype=torch.uint8, device="cuda"),
            "dtype": torch.ones(E, dtype=torch.int32, device="cuda"),
            "host": torch.ones(E, dtype=torch.uint8)}[bad]
    before = (env.t0.clone(), s.episodes.clone())
    with pytest.raises(ValueError, match="mask"):
        s.draw_mask(mask)
    if bad in ("short", "long"):
        with pytest.raises(ValueError, match="mask"):
            env.reset(mask=mask)
    assert torch.equal(env.t0, before[0]) and torch.equal(s.episodes, before[1])


def test_a_captured_graph_keeps_the_sampler_counters_it_writes_alive():
    import gc
    import weakref
    E, A, W, L = 8, 11, 4, 3
    env = make_env(E, A, W, L)
    old = env.sample_episode_starts(seed=1)
    env.reset()
    _, replay = env.graphed_step(steps=1)
    ref = weakref.ref(old.episodes)
    env.sample_episode_starts(seed=2)                              # replaces the sampler the graph was captured with
    del old
    gc.collect()
    assert ref() is not None, "the graph's draw counters were freed while the graph can still replay"
    for _ in range(L + 1):                                         # replays cross an episode end: the captured draw runs
        replay()
    torch.cuda.synchronize()
    assert bool((ref() == 2).all())
