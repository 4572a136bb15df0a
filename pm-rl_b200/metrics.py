"""Per-env evaluation metrics on device (util/eval.py:14-37): Sharpe, Sortino, max drawdown, average turnover."""
from __future__ import annotations

import math

import torch

from . import _lib

RUNNING, LAST_EPISODE, EPISODE_MEAN = 0, 1, 2          # include/pmrl_b200.h PMRL_EVAL_*


def eval_metrics(values, weights=None, rf: float = 0.0, periods: int = 252):
    """values [E, N] portfolio-value history (values[:, 0] = initial cash), weights [E, N, A] or None.
    Returns [E, 4] = (sharpe, sortino, max_drawdown, average_turnover)."""
    lib = _lib.load()
    v = values.to(torch.float32).contiguous()
    E, N = v.shape
    w = weights.to(torch.float32).contiguous() if weights is not None else None
    A = w.shape[2] if w is not None else 1
    out = torch.empty(E, 4, dtype=torch.float32, device=v.device)
    rc = lib.pmrl_eval_metrics(_lib.ptr(v), _lib.ptr(w), E, N, A, float(rf), int(periods), _lib.ptr(out), _lib.current_stream())
    _lib.check(rc, "pmrl_eval_metrics")
    return out


class StreamingEvalMetrics:
    """`eval_metrics` of every env's episodes, accumulated on the device one step at a time (C-ABI pmrl_eval_stream_*):
    `PMRL_EVAL_ACC_BYTES` (128) per env instead of the [E, N] value and [E, N, A] weight traces.

    `update()` must follow every reset and step of `env` on the same stream; `BatchedTradingEnv.track_eval_metrics`
    arranges that.  An env whose update was missed, or whose running episode began before the tracker existed, reads
    NaN until its next reset.  The readers return `(metrics [E, 5], count [E] int32)` with rows (return, sharpe, sortino,
    max drawdown, average turnover) — the return and drawdown bit-equal to the trace path, the others fp64 sums taken in
    another order — and the number of completed episodes; nothing here syncs with the host."""

    def __init__(self, env, rf: float = 0.0, periods: int = 252):
        rf = float(rf)
        if not math.isfinite(rf):
            raise ValueError(f"rf must be finite, got {rf}")
        if isinstance(periods, bool) or int(periods) != periods or periods < 1:
            raise ValueError(f"periods must be an integer >= 1, got {periods!r}")
        self.env, self.rf, self.periods = env, rf, int(periods)
        self.lib = _lib.load()
        self.acc = torch.zeros(env.E, _lib.EVAL_ACC_BYTES, dtype=torch.uint8, device=env.device)
        self._p_acc = self.acc.data_ptr()

    def update(self):
        """Fold the env's current state into the accumulators (enqueued on the current stream)."""
        env = self.env
        rc = self.lib.pmrl_eval_stream_update(env._p_cfg, env._p_st, self._p_acc, self.rf, self.periods,
                                              _lib.current_stream())
        if rc:
            _lib.check(rc, "pmrl_eval_stream_update")

    def _read(self, which):
        E, dev = self.env.E, self.env.device
        out = torch.empty(E, 5, dtype=torch.float32, device=dev)
        count = torch.empty(E, dtype=torch.int32, device=dev)
        rc = self.lib.pmrl_eval_stream_read(self.env._p_cfg, self.env._p_st, self._p_acc, which, self.rf, self.periods,
                                            _lib.ptr(out), _lib.ptr(count), _lib.current_stream())
        _lib.check(rc, "pmrl_eval_stream_read")
        return out, count

    def running(self):
        """Metrics of each env's running episode (after the step that ended an episode: that episode)."""
        return self._read(RUNNING)

    def last_episode(self):
        """Metrics of each env's last completed episode (NaN rows where none has completed)."""
        return self._read(LAST_EPISODE)

    def episode_mean(self):
        """Mean of the metric rows of each env's completed episodes (NaN rows where none has completed)."""
        return self._read(EPISODE_MEAN)

    def clear(self):
        """Forget everything: every env reads NaN until its next reset."""
        self.acc.zero_()
