"""Batched collect loops — the callers of the hot path (SURVEY.md §8(f) N1).

`collect_on_policy` is `Train._rollout` (train/on_policy.py:56-67) over E lockstep envs: the first loader item
is a reset (no action), every later item is act → step → buffer.add, with the observation written straight
into the rollout-buffer slot by the step kernel's consumer and no per-step host sync (the reference appends
host copies to `env.info` every step, trading_env.py:80-100).

`collect_off_policy` is `Train._collect` (train/off_policy.py:76-89) writing the (i, a, r) index-replay rows.
"""
from __future__ import annotations

import torch


def _check_relative(env, buffer):
    """A buffer that regenerates windows (index-mode rollout, replay) must divide them like the env does."""
    if buffer is None or getattr(buffer, "mode", "index") == "full":
        return
    want = (env.cfg.obs_relative_to, env.cfg.obs_relative_channels)
    got = (buffer.obs_relative_to, buffer.obs_relative_channels)
    if want != got:
        raise ValueError(f"the buffer regenerates windows with obs_relative_to / obs_relative_channels = {got}, the env makes "
                         f"them with {want}: a sample would not equal the obs the env returned; build the buffer with the "
                         "env config's settings")


@torch.no_grad()
def collect_on_policy(env, act_fn, buffer, num_items: int):
    """env: BatchedTradingEnv; act_fn(obs [E,A,W,F]) -> actions [E,A(,1)]; buffer: DeviceRolloutBuffer or None.
    Runs one episode of `num_items` loader items (1 reset + num_items-1 steps).  Returns the final obs.

    The step kernel writes the buffer rows itself (`buffer.sinks`): reward, raw action and post-step value of item k go
    to slot k - (W-1), and the obs the step returns — the obs stored WITH the next item (on_policy.py:65 stores the obs
    before the step) — is materialised directly in s[slot + 1].  No copy kernel, no second obs pass, no host sync."""
    _check_relative(env, buffer)
    if buffer is not None:
        buffer.reset()
    s = env.reset()
    for step in range(1, num_items):
        a = act_fn(s)
        if buffer is None:
            s, _, _ = env.step(a)
        else:
            s, _, _ = env.step_io(a, **buffer.sinks(step))
            buffer.advance()
    return s


@torch.no_grad()
def collect_off_policy(env, act_fn, buffer, epoch: int, num_items: int):
    """env: BatchedTradingEnv; buffer: DeviceReplayBuffer.  `buffer.add(epoch, step, a, r)` per item (off_policy.py:87),
    with the (i, a, r) row written by the step kernel: `i` is each env's OWN loader index t0[e] + k — the row the replay
    gather regenerates s and s' from (buffer.py:65-68) — not the lockstep counter."""
    _check_relative(env, buffer)
    s = env.reset()
    for step in range(1, num_items):
        a = act_fn(s)
        s, _, _ = env.step_io(a, **buffer.sinks(epoch, step))
    return s


@torch.no_grad()
def evaluate(env, act_fn, num_items: int, rf: float = 0.0, periods: int = 252, traces: bool = True):
    """`Train._evaluate` (train/on_policy.py:76-90) batched: rolls one episode and returns (total_reward [E],
    metrics [E, 4] = sharpe, sortino, max drawdown, average turnover).

    traces=True keeps the value / weight traces on the device ([E, N] + [E, N, A] floats) and computes the metrics from
    them at the end.  traces=False feeds a `metrics.StreamingEvalMetrics` after every step instead (128 bytes per env):
    the same total and drawdown bit for bit, Sharpe / Sortino / turnover up to the order of their fp64 sums.  It
    evaluates exactly one episode, so it refuses num_items - 1 > env.cfg.episode_len."""
    if not traces:
        L = env.cfg.episode_len
        if num_items < 2:
            raise ValueError(f"evaluate: num_items must be >= 2 (one reset and at least one step), got {num_items}")
        if L > 0 and num_items - 1 > L:
            raise ValueError(f"evaluate(traces=False): {num_items - 1} steps cross the episode end "
                             f"(episode_len = {L}); it evaluates exactly one episode")
        from .metrics import StreamingEvalMetrics
        tracker = StreamingEvalMetrics(env, rf=rf, periods=periods)
        s = env.reset()
        tracker.update()
        for _ in range(1, num_items):
            s, _, _ = env.step(act_fn(s))
            tracker.update()
        out, _ = tracker.running()
        return out[:, 0].contiguous(), out[:, 1:].contiguous()
    from .metrics import eval_metrics
    s = env.reset()
    E, A = env.E, env.A
    vals = torch.empty(E, num_items, device=env.device)
    wts = torch.empty(E, num_items, A, device=env.device)
    vals[:, 0] = env.value
    wts[:, 0] = env.weights_last
    total = torch.zeros(E, device=env.device)
    for step in range(1, num_items):
        s, r, _ = env.step(act_fn(s))
        total += r
        vals[:, step] = env.value
        wts[:, step] = env.weights_last
    return total, eval_metrics(vals, wts, rf=rf, periods=periods)
