"""bf16 observations (EnvConfig.obs_dtype = "bfloat16", PMRL_OBS_BF16) against the fp32 path, which the oracle and the live
reference pin: twin envs fed the same actions must agree bit for bit — the bf16 obs is the round-to-nearest-even of the fp32
obs element by element, and state, reward and done are identical."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _mods():
    import pmrl_b200
    from pmrl_b200 import synth
    from pmrl_b200.env import BatchedTradingEnv
    return pmrl_b200, synth, BatchedTradingEnv


def features_for(tbl4, F):
    """[T, A, F-1] table: OHLC for F = 5, else a deterministic mix of the OHLC channels (as tests/test_env_gpu.py)."""
    if F - 1 == 4:
        return tbl4
    return torch.stack([tbl4[..., i % 4] * (1.0 + 0.25 * (i // 4)) for i in range(F - 1)], dim=-1).contiguous()


def make_twins(E, A, W, F=5, episode_len=60, commission=0.0, reward="step_log", seed=1234, features=None, T=None):
    pmrl, synth, Env = _mods()
    T = T or (W + episode_len + 64)
    tbl4 = synth.gbm_ohlc(T, A, seed)
    feat = features_for(tbl4, F) if features is None else features
    t0 = synth.episode_offsets(E, T, W, episode_len)
    envs = []
    for dt in ("float32", "bfloat16"):
        cfg = pmrl.EnvConfig(num_envs=E, num_assets=A, window_size=W, num_features=F, commission=commission, reward=reward,
                             episode_len=episode_len, obs_dtype=dt)
        envs.append(Env(cfg, prices=tbl4, features=feat, t0=t0))
    return envs


def rne_bits(x32: np.ndarray) -> np.ndarray:
    """Round-to-nearest-even fp32 → bf16 bit patterns computed on the host (NaN positions are not meaningful)."""
    u = x32.view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)


def assert_bf16_of(o16, o32, msg=""):
    assert o16.dtype is torch.bfloat16 and o32.dtype is torch.float32 and o16.shape == o32.shape, msg
    nan = torch.isnan(o32)
    assert torch.equal(torch.isnan(o16.float()), nan), msg + ": NaN positions"
    want = o32.to(torch.bfloat16).view(torch.int16)
    got = o16.view(torch.int16)
    bad = (got != want) & ~nan
    assert not bool(bad.any()), f"{msg}: {int(bad.sum())} bf16 elements differ, first at {bad.nonzero()[:3].tolist()}"


def assert_same_state(e32, e16, msg=""):
    names = ["value", "hist", "idx", "is_full", "t", "ep_return", "reward", "done"] + (["sharpe"] if e32.sharpe is not None else [])
    for n in names:                                           # bitwise (the Sharpe reward is NaN on an episode's first step)
        a, b = getattr(e32, n), getattr(e16, n)
        assert a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes(), f"{msg}: {n} differs"


def run_twins(e32, e16, steps, seed=7, compare_every=1):
    E, A = e32.E, e32.A
    g = torch.Generator(device="cuda").manual_seed(seed)
    o32, o16 = e32.reset(), e16.reset()
    assert_bf16_of(o16, o32, "reset")
    for k in range(steps):
        a = torch.randn(E, A, generator=g, device="cuda")
        o32, r32, d32 = e32.step(a)
        o16, r16, d16 = e16.step(a)
        if (k + 1) % compare_every == 0 or k + 1 == steps:
            assert_bf16_of(o16, o32, f"step {k + 1}")
            assert_same_state(e32, e16, f"step {k + 1}")


# (E, A, W, F, commission, reward) — one per dispatch path of the obs
SHAPES = [
    (45, 100, 50, 5, 0.0, "step_log"),        # headline fused kernel, paired-row bf16 tile fill, partial last group
    (45, 100, 50, 5, 0.0025, "sharpe_ratio"),  # the same with commission and the running Sharpe reward
    (48, 50, 50, 5, 0.0, "step_log"),         # two envs per warp
    (37, 64, 24, 5, 0.0025, "step_log"),      # run-time W, paired rows
    (37, 64, 25, 5, 0.0, "step_log"),         # odd W: the lanes-over-rows fill with split 16/32-bit stores
    (45, 100, 50, 9, 0.0, "step_log"),        # F = 9, 13, 17
    (37, 64, 24, 13, 0.0, "step_log"),
    (30, 36, 20, 17, 0.0025, "step_log"),
    (30, 36, 20, 6, 0.0, "step_log"),         # channel-padded table, F = 6, 7
    (20, 100, 50, 7, 0.0, "step_log"),
    (20, 100, 24, 8, 0.0, "step_log"),        # dense F = 8 / 16
    (19, 32, 8, 16, 0.0, "step_log"),
    (48, 11, 50, 5, 0.0, "step_log"),         # A < 32: step kernel + obs tile kernel
    (48, 33, 6, 5, 0.0, "step_log"),          # W·A % 4 != 0: two kernels
    (21, 500, 50, 5, 0.0025, "step_log"),     # A > 128: staged step + tiles
    (40, 130, 16, 7, 0.0, "step_log"),        # A > 128 at F = 7: generic tile kernel
    (9, 40, 70, 5, 0.0, "step_log"),          # W > 64: two kernels
]


@pytest.mark.parametrize("E,A,W,F,commission,reward", SHAPES)
def test_twin_envs_agree_through_ring_fill_and_auto_reset(E, A, W, F, commission, reward):
    """Steps cross the ring fill (W - 1, W, W + 1) and an episode end with its auto-reset."""
    e32, e16 = make_twins(E, A, W, F, episode_len=W + 2, commission=commission, reward=reward)
    run_twins(e32, e16, W + 5)


def test_masked_reset_leaves_unmasked_bf16_rows_untouched():
    e32, e16 = make_twins(24, 100, 50, 5)
    run_twins(e32, e16, 53)
    mask = torch.zeros(24, dtype=torch.uint8); mask[::3] = 1
    sentinel = torch.full((24, 100, 50, 5), -3.5, dtype=torch.bfloat16, device="cuda")
    out16 = sentinel.clone()
    e16.reset(mask=mask, out=out16)
    o32 = e32.reset(mask=mask).clone()
    m = mask.bool().cuda()
    assert_bf16_of(out16[m], o32[m], "masked rows")
    assert torch.equal(out16[~m].view(torch.int16), sentinel[~m].view(torch.int16))
    assert_same_state(e32, e16, "after masked reset")


@pytest.mark.parametrize("A,W,F", [(100, 50, 5), (11, 50, 5), (64, 24, 13), (100, 24, 8)])
def test_observe(A, W, F):
    e32, e16 = make_twins(13, A, W, F)
    run_twins(e32, e16, W + 1)
    assert_bf16_of(e16.observe(), e32.observe(), "observe")


@pytest.mark.parametrize("chunks,pinned", [(0, True), (3, True), (-4, True), (0, False)])
def test_step_host(chunks, pinned):
    e32, e16 = make_twins(200, 100, 50, 5)
    e32.reset(); e16.reset()
    g = torch.Generator().manual_seed(3)
    for k in range(52):
        a = torch.randn(200, 100, generator=g)
        if pinned:
            a = a.pin_memory()
        o32, r32, d32 = e32.step_host(a, chunks=chunks)
        o16, r16, d16 = e16.step_host(a, chunks=chunks)
        assert torch.equal(r32, r16) and torch.equal(d32, d16)
    assert_bf16_of(o16, o32, "step_host")
    assert_same_state(e32, e16, "step_host")


def test_graphed_step_burst():
    e32, e16 = make_twins(40, 100, 50, 5, episode_len=30)
    e32.reset(); e16.reset()
    (a32, rep32), (a16, rep16) = e32.graphed_step(steps=15), e16.graphed_step(steps=15)
    g = torch.Generator(device="cuda").manual_seed(5)
    for _ in range(5):                                       # 75 steps: ring fill, episode end and auto-reset inside bursts
        a = torch.randn(15, 40, 100, generator=g, device="cuda")
        a32.copy_(a); a16.copy_(a)
        o32, r32, d32 = rep32()
        o16, r16, d16 = rep16()
        assert torch.equal(r32, r16) and torch.equal(d32, d16)
        assert_bf16_of(o16, o32, "graphed")
    assert_same_state(e32, e16, "graphed")


@pytest.mark.parametrize("A,W,F", [(100, 50, 5), (64, 24, 9), (11, 50, 5)])
def test_unaligned_out_view_takes_the_scalar_store(A, W, F):
    """An out= view 2 bytes past a 16-byte boundary: no tile can use the bulk store."""
    E = 10
    e32, e16 = make_twins(E, A, W, F)
    flat = torch.zeros(E * A * W * F + 8, dtype=torch.bfloat16, device="cuda")
    view = flat[1:1 + E * A * W * F].view(E, A, W, F)
    assert view.data_ptr() % 16 == 2
    e32.reset(); e16.reset(out=view)
    g = torch.Generator(device="cuda").manual_seed(9)
    for _ in range(W + 1):
        a = torch.randn(E, A, generator=g, device="cuda")
        o32, _, _ = e32.step(a)
        e16.step(a, out=view)
    assert_bf16_of(view, o32, "unaligned view")
    assert float(flat[0]) == 0.0 and bool((flat[1 + E * A * W * F:] == 0).all())


def test_rounding_edges_of_the_conversion():
    """Feature values at the edges of fp32 → bf16 rounding: exact ties (to even, up and down), subnormals and subnormal ties,
    -0.0, ±inf, NaN, the largest finite values, and values that round up to inf.  Pins the conversion itself against a host
    round-to-nearest-even, not only against torch."""
    specials = np.array([
        0x3F808000, 0x3F818000, 0x3F80C000, 0x3F807FFF, 0x3F808001,    # 1 + half ulp (tie → even, down / up), ± a bit
        0xBF808000, 0xBF818000,                                         # negative ties
        0x00000001, 0x00008000, 0x00018000, 0x00007FFF, 0x80008000,    # subnormals incl. ties
        0x80000000, 0x00000000, 0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00001, 0x7F800001,   # -0, +0, ±inf, NaNs
        0x7F7F7FFF, 0x7F7F8000, 0x7F7FFFFF, 0xFF7F8000,                # largest finite: stays / rounds up to ±inf
        0x00800000, 0x007FFFFF, 0x3F7FFFFF, 0x47800000,
    ], dtype=np.uint32).view(np.float32)
    E, A, W, F, L = 6, 64, 24, 5, 20
    pmrl, synth, Env = _mods()
    T = W + L + 64
    rs = np.random.RandomState(0)
    feat = rs.choice(specials, size=(T, A, F - 1)).astype(np.float32)
    e32, e16 = make_twins(E, A, W, F, episode_len=L, features=torch.from_numpy(feat), T=T)
    run_twins(e32, e16, W + 3, compare_every=4)
    o16 = e16.observe().cpu().view(torch.int16).numpy().view(np.uint16)
    o32 = e32.observe().cpu().numpy()
    nan = np.isnan(o32)
    assert np.array_equal(o16[~nan], rne_bits(o32[~nan]))
    assert np.all((o16[nan] & 0x7F80) == 0x7F80) and np.all((o16[nan] & 0x007F) != 0)     # NaN stays NaN
    assert nan.any() and np.isinf(o32).any() and (o16 == 0x7F80).sum() > (o32 == np.inf).sum()   # some finite values became inf


def _twin_collect(mode, E=8, A=100, W=10, items=30, obs_dtypes=("float32", "bfloat16")):
    pmrl, synth, Env = _mods()
    from pmrl_b200 import loops
    from pmrl_b200.buffers import DeviceRolloutBuffer
    T = items + W + 80
    tbl = synth.gbm_ohlc(T, A)
    t0 = synth.episode_offsets(E, T, W, items)
    out = []
    for dt in obs_dtypes:
        cfg = pmrl.EnvConfig(num_envs=E, num_assets=A, window_size=W, episode_len=items, obs_dtype=dt)
        env = Env(cfg, prices=tbl, t0=t0)
        gen = torch.Generator(device="cuda").manual_seed(8)
        buf = DeviceRolloutBuffer(5, items, E, A, W, batch_size=4, mode=mode, feat_am=env.feat_am, y_tm=env.y_tm, obs_dtype=dt)
        loops.collect_on_policy(env, lambda s, gen=gen: torch.randn(E, A, generator=gen, device="cuda"), buf, items)
        if mode == "full":
            buf.fill_prices(env)
        out.append(buf)
    return out


def _assert_batches(b32, b16, what):
    assert_bf16_of(b16[0], b32[0], what + " s")
    for got, want, name in zip(b16[1:], b32[1:], ("a", "r", "pv", "pa", "p")):
        assert torch.equal(got, want), f"{what} {name}"


@pytest.mark.parametrize("mode", ["full", "index"])
def test_rollout_buffer(mode):
    b32, b16 = _twin_collect(mode)
    if mode == "full":
        assert b16.s.dtype is torch.bfloat16
        assert_bf16_of(b16.s, b32.s, "stored s")
        assert 2 * (b32.nbytes() - b16.nbytes()) > b32.s.numel() * 4 * 0.99
    for t in ("a", "v", "r"):
        assert torch.equal(getattr(b32, t), getattr(b16, t))
    rs = np.random.RandomState(0)
    slots = rs.randint(1, b32.S - 1, 24); envs = rs.randint(0, b32.E, 24)
    _assert_batches(b32.gather(slots, envs), b16.gather(slots, envs), "gather")
    for k, (x32, x16) in enumerate(zip(b32.sample_random(np.random.RandomState(4)), b16.sample_random(np.random.RandomState(4)))):
        _assert_batches(x32, x16, f"sample_random {k}")
    for k, (x32, x16) in enumerate(zip(b32.sample(), b16.sample())):
        _assert_batches(x32, x16, f"sample {k}")


def test_rollout_buffer_add_converts():
    from pmrl_b200.buffers import DeviceRolloutBuffer
    E, A, W, F, items = 3, 12, 5, 5, 12
    b32 = DeviceRolloutBuffer(F, items, E, A, W)
    b16 = DeviceRolloutBuffer(F, items, E, A, W, obs_dtype="bfloat16")
    g = torch.Generator(device="cuda").manual_seed(1)
    for _ in range(items - 1):
        s = torch.randn(E, A, W, F, generator=g, device="cuda") * 100
        a, v, r = torch.rand(E, A, device="cuda"), torch.rand(E, device="cuda"), torch.rand(E, device="cuda")
        b32.add(s, a, v, r); b16.add(s, a, v, r)
    assert_bf16_of(b16.s, b32.s, "add")


def test_replay_buffer_sample():
    pmrl, synth, Env = _mods()
    from pmrl_b200 import loops
    from pmrl_b200.buffers import DeviceReplayBuffer
    E, A, W, F, items = 6, 40, 8, 9, 40
    T = 128
    tbl = synth.gbm_ohlc(T, A)
    feat = features_for(tbl, F)
    cfg = pmrl.EnvConfig(num_envs=E, num_assets=A, window_size=W, num_features=F, episode_len=items)
    env = Env(cfg, prices=tbl, features=feat)
    proj = torch.randn(W * F, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0)) * 2e-3
    act_fn = lambda s: s.reshape(E, A, W * F) @ proj
    bufs = [DeviceReplayBuffer(env.feat_am, F, items, E, A, W, buffer_size=3 * (items - 2 * (W - 1)), batch_size=4, obs_dtype=dt)
            for dt in ("float32", "bfloat16")]
    for ep in range(3):
        for b in bufs:
            loops.collect_off_policy(env, act_fn, b, ep, items)
    for sampler in ("traj", "buffer"):
        s32, a32, r32, n32 = bufs[0].sample(torch.Generator().manual_seed(11), sampler=sampler)
        s16, a16, r16, n16 = bufs[1].sample(torch.Generator().manual_seed(11), sampler=sampler)
        assert_bf16_of(s16, s32, sampler + " s"); assert_bf16_of(n16, n32, sampler + " s_")
        assert torch.equal(a32, a16) and torch.equal(r32, r16)


def test_dtype_errors():
    from pmrl_b200 import _lib, loops
    from pmrl_b200.buffers import DeviceRolloutBuffer
    e32, e16 = make_twins(4, 12, 6, 5)
    with pytest.raises(ValueError, match="bfloat16"):
        e16.step(torch.zeros(4, 12, device="cuda"), out=torch.empty(4, 12, 6, 5, device="cuda"))
    with pytest.raises(ValueError, match="float32"):
        e32.reset(out=torch.empty(4, 12, 6, 5, dtype=torch.bfloat16, device="cuda"))
    with pytest.raises(ValueError, match="bfloat16"):
        e16.observe(out=torch.empty(4, 12, 6, 5, device="cuda"))
    buf32 = DeviceRolloutBuffer(5, 12, 4, 12, 6)
    with pytest.raises(ValueError, match="obs_dtype"):
        loops.collect_on_policy(e16, lambda s: torch.zeros(4, 12, device="cuda"), buf32, 12)
    with pytest.raises(_lib.PmrlError, match="bfloat16"):
        e16.write_weight_channel(torch.zeros(4, 12, 6, 5, device="cuda"))
    with pytest.raises(ValueError):
        DeviceRolloutBuffer(5, 12, 4, 12, 6, obs_dtype="float16")


def test_full_size_c4_shard_step():
    """One step at 131,072 envs x 100 assets x window 50 (ring full), compared in chunks of 8,192 envs."""
    E, A, W = 131072, 100, 50
    e32, e16 = make_twins(E, A, W, 5, episode_len=100)
    e32.reset(obs=False); e16.reset(obs=False)
    g = torch.Generator(device="cuda").manual_seed(2)
    for _ in range(W):
        a = torch.randn(E, A, generator=g, device="cuda")
        e32.step(a, obs=False); e16.step(a, obs=False)
    a = torch.randn(E, A, generator=g, device="cuda")
    o32, _, _ = e32.step(a)
    o16, _, _ = e16.step(a)
    torch.cuda.synchronize()
    for c in range(0, E, 8192):
        assert_bf16_of(o16[c:c + 8192], o32[c:c + 8192], f"envs {c}..")
    assert_same_state(e32, e16, "c4 shard")
