"""Window-relative observations (EnvConfig.obs_relative_to, PMRL_OBS_REL) against a plain twin env fed the same actions:
the relative obs must equal, bit for bit, the plain obs with its masked channels divided by torch (`a / b` on CUDA is the
correctly rounded IEEE quotient) and the CPU restatement of oracle/obs_relative_oracle.py on the table windows; state,
reward and done must be identical to the plain twin's."""
import numpy as np
import pytest
import torch

from oracle.obs_relative_oracle import relative_obs

pytestmark = pytest.mark.gpu


def _mods():
    import pmrl_b200
    from pmrl_b200 import synth
    from pmrl_b200.env import BatchedTradingEnv
    return pmrl_b200, synth, BatchedTradingEnv


def features_for(tbl4, F):
    """[T, A, F-1] table: OHLC for F = 5, else a deterministic mix of the OHLC channels (as tests/test_obs_bf16_gpu.py)."""
    if F - 1 == 4:
        return tbl4
    return torch.stack([tbl4[..., i % 4] * (1.0 + 0.25 * (i // 4)) for i in range(F - 1)], dim=-1).contiguous()


def make_pair(E, A, W, F=5, ref=3, channels=None, episode_len=60, commission=0.0, seed=1234, features=None, T=None,
              obs_dtype="float32", starts=False):
    """(plain fp32 env, window-relative env) on the same tables and offsets."""
    pmrl, synth, Env = _mods()
    T = T or (W + episode_len + 64)
    tbl4 = synth.gbm_ohlc(T, A, seed)
    feat = features_for(tbl4, F) if features is None else features
    t0 = synth.episode_offsets(E, T, W, episode_len)
    envs = []
    for kw in (dict(), dict(obs_relative_to=ref, obs_relative_channels=channels, obs_dtype=obs_dtype)):
        cfg = pmrl.EnvConfig(num_envs=E, num_assets=A, window_size=W, num_features=F, commission=commission,
                             episode_len=episode_len, **kw)
        env = Env(cfg, prices=tbl4, features=feat, t0=t0)
        if starts:
            env.sample_episode_starts(seed=77)
        envs.append(env)
    return envs


def torch_rel(obs, cfg):
    """The caller-side normalisation pass: masked feature channels divided by channel ref of the window's last row."""
    out = obs.clone()
    div = obs[:, :, -1:, cfg.obs_relative_to]
    for c in cfg.obs_relative_channels:
        out[..., c] = obs[..., c] / div
    return out


def assert_bits(got, want, msg=""):
    assert got.dtype == want.dtype and got.shape == want.shape, msg
    nan = torch.isnan(want.float())
    assert torch.equal(torch.isnan(got.float()), nan), msg + ": NaN positions"
    it = torch.int32 if got.dtype is torch.float32 else torch.int16
    bad = (got.view(it) != want.view(it)) & ~nan
    assert not bool(bad.any()), f"{msg}: {int(bad.sum())} elements differ, first at {bad.nonzero()[:3].tolist()}"


def assert_same_state(ep, er, msg=""):
    names = ["value", "hist", "idx", "is_full", "t", "t0", "ep_return", "reward", "done"]
    for n in names:
        a, b = getattr(ep, n), getattr(er, n)
        assert a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes(), f"{msg}: {n} differs"


def oracle_check(er, o_rel, o_plain):
    """Feature channels against the CPU restatement applied to the table windows at the env's rows; weight channel = plain."""
    F, W = er.F, er.W
    feat = er.feat_am.permute(1, 0, 2).cpu().numpy()                     # [T, A, F-1]
    rows = (er.t0.long() + er.t.long()).cpu().numpy()
    win = np.stack([feat[r:r + W].transpose(1, 0, 2) for r in rows])     # [E, A, W, F-1]
    full = np.concatenate([win, o_plain[..., F - 1:].cpu().numpy()], axis=-1)
    want = torch.from_numpy(relative_obs(full, er.cfg.obs_relative_to, er.cfg.obs_relative_channels))
    got = o_rel.float().cpu() if o_rel.dtype is torch.float32 else o_rel.cpu()
    if o_rel.dtype is torch.bfloat16:
        want = want.to(torch.bfloat16)
    assert_bits(got, want, "oracle")


def check(ep, er, o_plain, o_rel, msg):
    want = torch_rel(o_plain.float(), er.cfg)
    if o_rel.dtype is torch.bfloat16:
        want = want.to(torch.bfloat16)
    assert_bits(o_rel, want, msg)
    assert_same_state(ep, er, msg)


def run_pair(ep, er, steps, seed=7, oracle_every=0):
    E, A = ep.E, ep.A
    g = torch.Generator(device="cuda").manual_seed(seed)
    op, orl = ep.reset(), er.reset()
    check(ep, er, op, orl, "reset")
    for k in range(steps):
        a = torch.randn(E, A, generator=g, device="cuda")
        op, _, _ = ep.step(a)
        orl, _, _ = er.step(a)
        check(ep, er, op, orl, f"step {k + 1}")
        if oracle_every and (k + 1) % oracle_every == 0:
            oracle_check(er, orl, op)
    oracle_check(er, orl, op)
    return op, orl


# (E, A, W, F, commission, ref, channels) — every obs path: fused kernel (F = 5 / 9, W compiled in or not, divisor lane and
# chunk moving across 32), the register-staged tile kernel (A < 32, A > 128), the generic tile kernel (F = 7, 13, W > 64)
SHAPES = [
    (45, 100, 50, 5, 0.0, 3, None),
    (45, 100, 50, 5, 0.0025, 3, (0, 1, 3)),
    (48, 50, 31, 5, 0.0, 0, None),
    (48, 50, 33, 5, 0.0025, 2, None),
    (37, 64, 64, 5, 0.0, 3, (1, 2, 3)),
    (30, 100, 2, 5, 0.0, 3, None),
    (45, 100, 50, 9, 0.0, 3, None),
    (37, 64, 33, 9, 0.0025, 5, (0, 2, 4, 5, 7)),
    (30, 36, 31, 13, 0.0, 11, None),
    (20, 100, 50, 7, 0.0025, 1, (0, 1, 4)),
    (48, 11, 50, 5, 0.0, 3, None),
    (21, 500, 50, 5, 0.0025, 3, (3,)),
    (9, 500, 64, 9, 0.0, 0, (0, 3)),
    (9, 40, 70, 5, 0.0, 3, None),
]


@pytest.mark.parametrize("E,A,W,F,commission,ref,channels", SHAPES)
def test_relative_obs_through_ring_fill_and_auto_reset(E, A, W, F, commission, ref, channels):
    """Steps cross the ring fill and an episode end with its auto-reset, with random episode starts drawn at every reset."""
    ep, er = make_pair(E, A, W, F, ref, channels, episode_len=W + 2, commission=commission, starts=True)
    run_pair(ep, er, W + 5, oracle_every=max(1, (W + 5) // 3))


@pytest.mark.parametrize("E,A,W,F,commission,ref,channels",
                         [s for s in SHAPES if s[:4] in {(45, 100, 50, 5), (48, 50, 31, 5), (48, 50, 33, 5), (45, 100, 50, 9),
                                                         (30, 36, 31, 13), (48, 11, 50, 5), (9, 500, 64, 9)}])
def test_bf16_relative_is_the_rounding_of_fp32_relative(E, A, W, F, commission, ref, channels):
    """bf16 x REL (paired-row fill at F = 5 with even W, lanes-over-rows otherwise, tile kernels) = RNE of fp32 REL."""
    pmrl, synth, Env = _mods()
    ep, er16 = make_pair(E, A, W, F, ref, channels, episode_len=W + 2, commission=commission, obs_dtype="bfloat16")
    _, er32 = make_pair(E, A, W, F, ref, channels, episode_len=W + 2, commission=commission)
    g = torch.Generator(device="cuda").manual_seed(3)
    o32, o16 = er32.reset(), er16.reset()
    assert_bits(o16, o32.to(torch.bfloat16), "reset")
    for k in range(W + 5):
        a = torch.randn(E, A, generator=g, device="cuda")
        o32, _, _ = er32.step(a)
        o16, _, _ = er16.step(a)
        assert_bits(o16, o32.to(torch.bfloat16), f"step {k + 1}")
        assert_same_state(er32, er16, f"step {k + 1}")


def _tuned(key, value, fn):
    from pmrl_b200 import _lib
    _lib.set_tuning(key, value)
    try:
        return fn()
    finally:
        _lib.set_tuning(key, 1)


@pytest.mark.parametrize("F,obs_dtype", [(5, "float32"), (9, "float32"), (5, "bfloat16")])
def test_every_dispatch_path_writes_the_same_bytes(F, obs_dtype):
    """step, step_io into a rollout slot, step_host (zero-copy, growing / equal / pageable slices), graphed_step(1) and
    graphed_step(15), and the tuning fallbacks (two kernels, generic tile kernel, register-ring fused kernel) all write the
    obs `step` writes; masked reset and observe agree with the torch-normalised plain twin."""
    from pmrl_b200 import _lib
    E, A, W, L, N = 40, 100, 50, 30, 60
    acts = torch.randn(N, E, A, generator=torch.Generator().manual_seed(5))

    def fresh():
        return make_pair(E, A, W, F, 3, (0, 1, 3) if F == 5 else None, episode_len=L, obs_dtype=obs_dtype)

    def run(stepper):
        ep, er = fresh()
        ep.reset(); er.reset()
        outs = []
        for k in range(N):
            op, _, _ = ep.step(acts[k].cuda())
            outs.append((stepper(er, k), op.clone()))
        return ep, er, outs

    ref_ep, ref_er, ref = run(lambda er, k: er.step(acts[k].cuda())[0].clone())
    for k in (0, W - 2, W, L, N - 1):
        want = torch_rel(ref[k][1], ref_er.cfg)
        assert_bits(ref[k][0], want if obs_dtype == "float32" else want.to(torch.bfloat16), f"step {k}")
    slot = torch.empty(3, E, A, W, F, dtype=ref_er.obs_dtype, device="cuda")
    variants = {
        "step_io": lambda er, k: er.step_io(acts[k].cuda(), out=slot[k % 3])[0].clone(),
        "host0": lambda er, k: er.step_host(acts[k].pin_memory(), chunks=0)[0].clone(),
        "host3": lambda er, k: er.step_host(acts[k].pin_memory(), chunks=3)[0].clone(),
        "host-4": lambda er, k: er.step_host(acts[k].pin_memory(), chunks=-4)[0].clone(),
        "host_pageable": lambda er, k: er.step_host(acts[k].clone(), chunks=0)[0].clone(),
    }
    for name, fn in variants.items():
        _, er, got = run(fn)
        for k in range(N):
            assert_bits(got[k][0], ref[k][0], f"{name} step {k}")
        assert_same_state(ref_er, er, name)
    for key, value, name in ((_lib.TUNE_FUSED, 0, "two kernels"), (_lib.TUNE_FAST_FILL, 0, "generic tiles"),
                             (_lib.TUNE_RING_TMA, 0, "register rings")):
        _, er, got = _tuned(key, value, lambda: run(lambda er, k: er.step(acts[k].cuda())[0].clone()))
        for k in range(N):
            assert_bits(got[k][0], ref[k][0], f"{name} step {k}")
    for K in (1, 15):
        ep, er = fresh()
        er.reset()
        static, replay = er.graphed_step(steps=K)
        for b in range(N // K):
            static.copy_(acts[b * K:(b + 1) * K].reshape(static.shape).cuda())
            o, _, _ = replay()
            assert_bits(o, ref[(b + 1) * K - 1][0], f"graphed_step({K}) burst {b}")
    # masked reset and observe on the state the reference run ended in
    mask = torch.zeros(E, dtype=torch.uint8); mask[::3] = 1
    sentinel = torch.full((E, A, W, F), -2.5, dtype=ref_er.obs_dtype, device="cuda")
    out = sentinel.clone()
    ref_er.reset(mask=mask, out=out)
    op = ref_ep.reset(mask=mask).clone()
    m = mask.bool().cuda()
    want = torch_rel(op, ref_er.cfg)
    want = want if obs_dtype == "float32" else want.to(torch.bfloat16)
    assert_bits(out[m], want[m], "masked reset")
    assert torch.equal(out[~m], sentinel[~m])
    for _ in range(3):
        a = torch.randn(E, A, device="cuda")
        ref_ep.step(a); ref_er.step(a)
    check(ref_ep, ref_er, ref_ep.observe().clone(), ref_er.observe(), "observe")


SPECIALS = np.array([0x00000000, 0x80000000, 0x00000001, 0x807FFFFF, 0x00400000, 0x0B000000, 0x73800000,   # ±0, subnormals,
                     0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00001,                                      # 2^-105, 2^40 ... ±inf,
                     0x1D800000, 0x1E800000, 0x60800000, 0x61800000, 0x7F7FFFFF, 0xFF7FFFFF,              # NaNs, 2^-68 .. 2^68,
                     0x3F800000, 0xBF800000, 0xC2C80000], dtype=np.uint32).view(np.float32)              # max, ±1, -100


@pytest.mark.parametrize("A,W,F,obs_dtype", [(64, 50, 5, "float32"), (64, 33, 9, "float32"), (64, 24, 5, "bfloat16"),
                                             (11, 50, 5, "float32"), (40, 20, 13, "float32"), (100, 50, 9, "bfloat16")])
def test_edge_divisors_and_numerators_follow_ieee_division(A, W, F, obs_dtype):
    """Tables with zero, negative, subnormal, out-of-range (beyond 2^±60), infinite and NaN values among normal ones, as
    divisors and as numerators: the obs equals torch's division wherever the shared-reciprocal path or __fdiv_rn runs."""
    E, L = 12, 20
    T = W + L + 64
    rs = np.random.RandomState(A + W + F)
    feat = rs.lognormal(4.0, 0.3, size=(T, A, F - 1)).astype(np.float32)
    hit = rs.rand(T, A, F - 1) < 0.3
    feat[hit] = rs.choice(SPECIALS, size=int(hit.sum()))
    ep, er = make_pair(E, A, W, F, 0, None, episode_len=L, features=torch.from_numpy(feat), T=T, obs_dtype=obs_dtype)
    run_pair(ep, er, W + 3, oracle_every=4)


def _collect_twins(mode, obs_dtype="float32", E=8, A=100, W=10, items=30, F=5, ref=3, channels=(0, 1, 3)):
    """Two window-relative envs of one config driven by the same actions, one into a full-mode rollout buffer (stores the
    obs the env wrote) and one into an index-mode buffer (regenerates them)."""
    pmrl, synth, Env = _mods()
    from pmrl_b200 import loops
    from pmrl_b200.buffers import DeviceRolloutBuffer
    T = items + W + 80
    tbl = synth.gbm_ohlc(T, A)
    t0 = synth.episode_offsets(E, T, W, items)
    bufs = []
    for m in ("full", mode):
        cfg = pmrl.EnvConfig(num_envs=E, num_assets=A, window_size=W, num_features=F, episode_len=items, obs_dtype=obs_dtype,
                             obs_relative_to=ref, obs_relative_channels=channels)
        env = Env(cfg, prices=tbl, features=features_for(tbl, F), t0=t0)
        gen = torch.Generator(device="cuda").manual_seed(8)
        rel = dict(obs_relative_to=ref, obs_relative_channels=channels) if m == "index" else {}
        buf = DeviceRolloutBuffer(F, items, E, A, W, batch_size=4, mode=m, feat_am=env.feat_am, y_tm=env.y_tm,
                                  obs_dtype=obs_dtype, **rel)
        loops.collect_on_policy(env, lambda s, gen=gen: torch.randn(E, A, generator=gen, device="cuda"), buf, items)
        if m == "full":
            buf.fill_prices(env)
        bufs.append(buf)
    return bufs


@pytest.mark.parametrize("obs_dtype,F", [("float32", 5), ("bfloat16", 5), ("float32", 9)])
def test_index_rollout_gather_returns_the_obs_the_env_wrote(obs_dtype, F):
    full, index = _collect_twins("index", obs_dtype, F=F, channels=None if F == 9 else (0, 1, 3))
    rs = np.random.RandomState(0)
    slots = rs.randint(1, full.S - 1, 32); envs = rs.randint(0, full.E, 32)
    gf, gi = full.gather(slots, envs), index.gather(slots, envs)
    assert_bits(gi[0], gf[0], "s")
    for x, y, name in zip(gi[1:], gf[1:], ("a", "r", "pv", "pa")):
        assert torch.equal(x, y), name


@pytest.mark.parametrize("obs_dtype", ["float32", "bfloat16"])
def test_replay_gather_divides_each_window_by_its_own_last_row(obs_dtype):
    """s and s' of the relative replay gather = the plain gather's windows normalised by torch, s by row i + W - 1 and s' by
    row i + W — and the plain gather regenerates exactly the env's obs (tests/test_features_buffers_gpu.py)."""
    pmrl, synth, Env = _mods()
    from pmrl_b200 import loops
    from pmrl_b200.buffers import DeviceReplayBuffer
    E, A, W, F, items, ref, chans = 6, 40, 8, 9, 40, 3, (0, 1, 3, 6)
    tbl = synth.gbm_ohlc(128, A)
    cfg = pmrl.EnvConfig(num_envs=E, num_assets=A, window_size=W, num_features=F, episode_len=items)
    env = Env(cfg, prices=tbl, features=features_for(tbl, F))
    proj = torch.randn(W * F, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0)) * 2e-3
    size = 3 * (items - 2 * (W - 1))
    plain = DeviceReplayBuffer(env.feat_am, F, items, E, A, W, buffer_size=size, batch_size=4)
    for ep in range(3):
        loops.collect_off_policy(env, lambda s: s.reshape(E, A, W * F) @ proj, plain, ep, items)
    rel = DeviceReplayBuffer(env.feat_am, F, items, E, A, W, buffer_size=size, batch_size=4, obs_dtype=obs_dtype,
                             obs_relative_to=ref, obs_relative_channels=chans)
    rel.bi.copy_(plain.bi); rel.ba.copy_(plain.ba); rel.br.copy_(plain.br)
    rel.curr_epoch, rel.newest_epoch, rel.full = plain.curr_epoch, plain.newest_epoch, plain.full
    rcfg = pmrl.EnvConfig(num_features=F, obs_relative_to=ref, obs_relative_channels=chans)
    for sampler in ("traj", "buffer"):
        s, a, r, s2 = plain.sample(torch.Generator().manual_seed(11), sampler=sampler)
        sr, ar, rr, s2r = rel.sample(torch.Generator().manual_seed(11), sampler=sampler)
        for got, base, name in ((sr, s, "s"), (s2r, s2, "s_")):
            want = torch_rel(base, rcfg)
            assert_bits(got, want if obs_dtype == "float32" else want.to(torch.bfloat16), f"{sampler} {name}")
        assert torch.equal(a, ar) and torch.equal(r, rr)


def test_collect_loops_refuse_a_buffer_with_another_transform():
    pmrl, synth, Env = _mods()
    from pmrl_b200 import loops
    from pmrl_b200.buffers import DeviceReplayBuffer, DeviceRolloutBuffer
    E, A, W, items = 4, 12, 6, 12
    ep, er = make_pair(E, A, W, 5, 3, None, episode_len=items)
    act = lambda s: torch.zeros(E, A, device="cuda")
    plain_idx = DeviceRolloutBuffer(5, items, E, A, W, mode="index", feat_am=er.feat_am, y_tm=er.y_tm)
    other_idx = DeviceRolloutBuffer(5, items, E, A, W, mode="index", feat_am=er.feat_am, y_tm=er.y_tm, obs_relative_to=0)
    rel_idx = DeviceRolloutBuffer(5, items, E, A, W, mode="index", feat_am=er.feat_am, y_tm=er.y_tm, obs_relative_to=3)
    for env, buf in ((er, plain_idx), (er, other_idx), (ep, rel_idx)):
        with pytest.raises(ValueError, match="obs_relative_to"):
            loops.collect_on_policy(env, act, buf, items)
    loops.collect_on_policy(er, act, rel_idx, items)                          # matching settings
    loops.collect_on_policy(er, act, DeviceRolloutBuffer(5, items, E, A, W), items)   # a full-mode buffer stores what it gets
    rb = DeviceReplayBuffer(er.feat_am, 5, 40, E, A, W)
    with pytest.raises(ValueError, match="obs_relative_to"):
        loops.collect_off_policy(er, act, rb, 0, items)
    with pytest.raises(ValueError):
        DeviceReplayBuffer(er.feat_am, 5, 40, E, A, W, obs_relative_to=4)


def test_full_size_c4_shard_step():
    """One step at 131,072 envs x 100 assets x window 50 (ring full), checked on a seeded sample of 4,096 envs."""
    E, A, W = 131072, 100, 50
    ep, er = make_pair(E, A, W, 5, 3, None, episode_len=100)
    ep.reset(obs=False); er.reset(obs=False)
    g = torch.Generator(device="cuda").manual_seed(2)
    for _ in range(W):
        a = torch.randn(E, A, generator=g, device="cuda")
        ep.step(a, obs=False); er.step(a, obs=False)
    a = torch.randn(E, A, generator=g, device="cuda")
    op, _, _ = ep.step(a)
    orl, _, _ = er.step(a)
    torch.cuda.synchronize()
    idx = torch.randperm(E, generator=torch.Generator().manual_seed(0))[:4096].cuda()
    assert_bits(orl[idx], torch_rel(op[idx], er.cfg), "c4 shard sample")
    assert_same_state(ep, er, "c4 shard")
