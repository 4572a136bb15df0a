"""Randomised episode starts (C-ABI pmrl_env_draw_starts): every reset of an env gives it a fresh table offset t0[e],
drawn on the device, instead of replaying the one offset it was built with.

    starts = env.sample_episode_starts(seed=7)                                   # uniform over [0, T - episode_len - W]
    starts = env.sample_episode_starts(seed=7, distribution="geometric", beta=1e-3)   # favours the latest rows

A draw is a pure function of (seed, global env id, the env's draw count), so a rank whose shard starts at global env
`first_env` reproduces its part of the single-GPU run.  The formulas are in include/pmrl_b200.h.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib

UNIFORM, GEOMETRIC = 0, 1          # include/pmrl_b200.h PMRL_START_*
DRAW_DUE, DRAW_MASK = 0, 1         # include/pmrl_b200.h PMRL_DRAW_*
DISTRIBUTIONS = {"uniform": UNIFORM, "geometric": GEOMETRIC}


def _integer(name, x):
    if isinstance(x, bool) or int(x) != x:
        raise ValueError(f"{name} must be an integer, got {x!r}")
    return int(x)


def start_dist(T: int, episode_len: int, W: int, low=0, high=None, seed=0, distribution="uniform", beta=None,
               first_env=0) -> _lib.PmrlStartDist:
    """The PmrlStartDist of a sampler over table offsets [low, high] (high=None: T - episode_len - W, the last offset
    whose episode stays inside the tables).  Raises ValueError on what pmrl_env_draw_starts would refuse."""
    if T <= 0:
        raise ValueError("episode starts index the price / feature tables: this env has none")
    if distribution not in DISTRIBUTIONS:
        raise ValueError(f"distribution must be one of {sorted(DISTRIBUTIONS)}, got {distribution!r}")
    low = _integer("low", low)
    high = T - episode_len - W if high is None else _integer("high", high)
    if low < 0 or high < low:
        raise ValueError(f"need 0 <= low <= high, got low={low}, high={high}")
    if high + episode_len + W > T:
        raise ValueError(f"high + episode_len + W = {high + episode_len + W} > T = {T}: the episode would leave the tables")
    seed = _integer("seed", seed)
    if not 0 <= seed < 1 << 64:
        raise ValueError(f"seed must be in [0, 2**64), got {seed}")
    first_env = _integer("first_env", first_env)
    if not 0 <= first_env < 1 << 62:
        raise ValueError(f"first_env must be >= 0, got {first_env}")
    log1m_beta = geo_norm = 0.0
    if distribution == "geometric":
        if beta is None or not 0.0 < float(beta) < 1.0:          # NaN fails the comparison
            raise ValueError(f"the geometric distribution needs beta in (0, 1), got {beta!r}")
        log1m_beta = math.log1p(-float(beta))
        geo_norm = -math.expm1((high - low + 1) * log1m_beta)
    elif beta is not None:
        raise ValueError("beta only applies to distribution='geometric'")
    return _lib.PmrlStartDist(DISTRIBUTIONS[distribution], low, high, 0, seed, first_env, log1m_beta, geo_norm)


class EpisodeStarts:
    """The sampler `BatchedTradingEnv.sample_episode_starts` attaches.  `episodes` [E] int32 counts each env's draws (the
    Philox counter of its next draw); the env's own `t0` tensor receives the offsets.  `detach()` stops drawing and keeps
    the last offsets."""

    def __init__(self, env, dist: _lib.PmrlStartDist):
        self.env, self.dist = env, dist
        self.lib = _lib.load()
        self.episodes = torch.zeros(env.E, dtype=torch.int32, device=env.device)
        self._p_dist = C.byref(self.dist)
        self._p_t, self._p_t0, self._p_ep = env.t.data_ptr(), env.t0.data_ptr(), self.episodes.data_ptr()

    @property
    def low(self) -> int:
        return self.dist.lo

    @property
    def high(self) -> int:
        return self.dist.hi

    def draw_due(self):
        """New offsets for the envs the next step call auto-resets (enqueued on the current stream)."""
        env = self.env
        rc = self.lib.pmrl_env_draw_starts(env._p_cfg, self._p_dist, self._p_t, None, DRAW_DUE, self._p_t0, self._p_ep,
                                           _lib.current_stream())
        if rc:
            _lib.check(rc, "pmrl_env_draw_starts")

    def draw_mask(self, mask=None):
        """New offsets for the envs with mask[e] != 0 (all when None): what `reset(mask)` enqueues before it resets.
        mask: a contiguous CUDA uint8 tensor of E elements, or None."""
        if mask is not None and (mask.dtype is not torch.uint8 or mask.numel() != self.env.E or not mask.is_cuda
                                 or not mask.is_contiguous()):
            raise ValueError(f"mask must be a contiguous CUDA uint8 tensor of {self.env.E} elements, got {mask.dtype} "
                             f"{tuple(mask.shape)} on {mask.device}")
        rc = self.lib.pmrl_env_draw_starts(self.env._p_cfg, self._p_dist, None, _lib.ptr(mask), DRAW_MASK, self._p_t0,
                                           self._p_ep, _lib.current_stream())
        _lib.check(rc, "pmrl_env_draw_starts")

    def detach(self):
        """Stop drawing: later resets reuse each env's current offset, as without a sampler."""
        if self.env._starts is self:
            self.env._starts = None
