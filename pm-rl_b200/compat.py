"""Drop-in `TradingEnv` (E = 1) with the reference's exact call surface, executing on the CUDA kernels.

Mirrors env/sim/trading_env.py:7-105 so that `train/on_policy.py:_rollout`, `train/off_policy.py:_collect`
and `agent/pg` drive it unchanged:

    env = TradingEnv()                       # shapes from config.base like the reference (or an EnvConfig)
    s = env.reset(features)                  # features [A, W, F], last channel overwritten in place
    r, s_ = env.step(action, features, prices)
    env.value, env.weights.get_last(), env.weights.get_all(), env.info["values"|"actions"|"rewards"|"returns"]

`features` / `prices` are supplied by the caller exactly as in the reference (the loader owns the
windows), so the kernels run with external price relatives and only write the weight channel
(PMRL_OBS_WEIGHTS).  There is no CPU compute path.  A caller that keeps everything on the CPU (the reference's own loop)
goes through page-locked staging buffers: action and price relatives are copied into pinned memory the kernels read in
place, reward / done / weight channel are written by the kernels straight into pinned memory, and one stream
synchronisation per step makes them host tensors — no per-step torch H2D/D2H ops.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from .config import EnvConfig
from .env import BatchedTradingEnv, OBS_NONE, OBS_WEIGHTS


class _WeightsView:
    """ActionBuffer read surface (env/sim/weight_buffer.py:28-44) over the device ring."""

    def __init__(self, owner):
        self._o = owner

    @property
    def buffer(self):
        return self._o._env.hist[0]                       # [W, A]

    @property
    def idx(self):
        return int(self._o._env.idx[0].item())

    @property
    def is_full(self):
        return bool(self._o._env.is_full[0].item())

    def get_last(self):
        return self._o._env.weights_last[0]               # [A]

    def get_all(self):
        e = self._o._env
        # the WEIGHTS-mode kernel on a scratch [1, A, W, F] tensor; its last channel is get_all()
        scratch = torch.zeros(1, e.A, e.W, e.F, dtype=torch.float32, device=e.device)
        e.write_weight_channel(scratch)
        return scratch[0, :, :, -1]                       # [A, W]


class _RewardView:
    """Reward.* (env/reward.py:15-31) evaluated from the device-side value trace."""

    def __init__(self, owner):
        self._o = owner

    def _values(self):
        return self._o.info["values"]

    def returns(self):
        v = self._values()
        return np.float32(v[-1]) / np.float32(v[-2])

    def log_returns(self):
        return np.log(self.returns())

    def sharpe_ratio(self):
        v = np.array(self._values(), dtype=np.float64)
        g = v[1:] / v[:-1]
        with np.errstate(all="ignore"):
            return (np.mean(g) - self._o.cfg.risk_free_rate) / np.std(g, ddof=1)

    def get_reward(self):
        name = self._o.reward_name
        fn = {"returns": self.returns, "log_returns": self.log_returns, "sharpe_ratio": self.sharpe_ratio}[name]
        return self._o.cfg.reward_scale * fn()


class TradingEnv:
    def __init__(self, cfg: EnvConfig | None = None, device=None, three_tuple: bool = False):
        if cfg is None:
            try:
                cfg = EnvConfig.from_reference_config()
                import config.base as cb
                self.reward_name = getattr(cb, "REWARD", "log_returns")
            except ImportError:
                cfg = EnvConfig()
                self.reward_name = "log_returns"
        else:
            self.reward_name = cfg.reward if cfg.reward != "step_log" else "log_returns"
        # a single env, never "done" (the reference ends an episode at loader exhaustion), step reward = :99
        # (plain fp32 obs whatever cfg.obs_dtype / obs_relative_to say: this shim mirrors the reference's fp32 `features` tensor)
        self.cfg = EnvConfig(**{**cfg.__dict__, "num_envs": 1, "episode_len": 0, "reward": "step_log", "obs_dtype": "float32",
                                          "obs_relative_to": None, "obs_relative_channels": None})
        self._env = BatchedTradingEnv(self.cfg, prices=None, features=None, device=device)
        self.init_cash = self.cfg.initial_cash            # agent/dreamer/dreamer.py:197
        self.three_tuple = three_tuple
        self.weights = _WeightsView(self)
        self.reward = _RewardView(self)
        self._trace = None
        self._pin = None                                  # page-locked staging of the CPU-caller path, made on first use
        self._host_idx = 1                                # ring slot the next step writes (E = 1: known on the host)
        self._clear_trace()

    def _pinned(self):
        if self._pin is None:
            e = self._env
            A, W, F = e.A, e.W, e.F
            p = {"in": torch.zeros(2, A).pin_memory(), "obs": torch.zeros(1, A, W, F).pin_memory(),
                 "r": torch.zeros(1).pin_memory(), "d": torch.zeros(1, dtype=torch.uint8).pin_memory(),
                 "v": torch.zeros(1).pin_memory(), "w": torch.zeros(A).pin_memory()}
            p["ptr_a"], p["ptr_y"] = p["in"][0].data_ptr(), p["in"][1].data_ptr()   # device-addressable under unified addressing
            p["ptr_obs"], p["ptr_r"], p["ptr_d"] = p["obs"].data_ptr(), p["r"].data_ptr(), p["d"].data_ptr()
            self._pin = p
        return self._pin

    def _weights_to_host(self, features):
        """features[:, :, -1] = get_all() for a CPU `features`: the WEIGHTS-mode kernel writes the channel into a pinned
        scratch obs (posted writes over PCIe), the host copies the strided channel after the caller's synchronisation."""
        e, p = self._env, self._pinned()
        rc = e.lib.pmrl_obs_build(e._p_cfg, e._p_tbl, e._p_st, p["ptr_obs"], OBS_WEIGHTS, _lib.current_stream())
        if rc:
            _lib.check(rc, "pmrl_obs_build")

    def _step_host(self, action, features, prices):
        e, p = self._env, self._pinned()
        A, W, F = e.A, e.W, e.F
        if tuple(features.shape[-3:]) != (A, W, F):
            raise ValueError(f"features must be [{A}, {W}, {F}], got {tuple(features.shape)}")
        p["in"][0].copy_(action.reshape(A))
        p["in"][1].copy_(prices.reshape(A))
        stream = _lib.current_stream()
        rc = e.lib.pmrl_env_step(e._p_cfg, e._p_tbl, e._p_st, p["ptr_a"], p["ptr_y"], p["ptr_r"], p["ptr_d"], None,
                                 OBS_NONE, e._ptr_stats, stream)
        if rc:
            _lib.check(rc, "pmrl_env_step")
        self._weights_to_host(features)
        slot = self._host_idx
        p["v"].copy_(e.value, non_blocking=True)
        p["w"].copy_(e.hist[0, slot], non_blocking=True)
        torch.cuda.current_stream(e.device).synchronize()
        self._host_idx = (slot + 1) % W
        v, r = p["v"][0].clone(), p["r"][0].clone()
        t = self._trace
        t["values"].append(v)
        t["actions"].append(p["w"].clone())
        t["rewards"].append(r)
        v_before = t["values"][-2] if len(t["values"]) > 1 else self.cfg.initial_cash
        if not isinstance(v_before, float) and v_before.is_cuda:
            v_before = v_before.cpu()
        t["returns"].append(v / v_before if self.cfg.commission == 0 else torch.exp(r / self.cfg.reward_scale))
        features[..., -1] = p["obs"][0, :, :, -1]
        if self.three_tuple:
            return features, r, p["d"][0].clone()
        return r, features

    # -- info: the reference appends host copies every step (:80,85,90,100); here the trace stays on the
    #    device and is materialised only when `info` is read --
    def _clear_trace(self):
        self._trace = {"values": [], "actions": [], "rewards": [], "returns": []}
        self._first_action = self._env.weights_last[0].clone()

    @staticmethod
    def _stack(items):
        """One host tensor from a trace list (entries are CUDA tensors for CUDA callers, CPU tensors for CPU callers)."""
        if len({x.device for x in items}) == 1:
            return torch.stack(items).cpu()
        return torch.stack([x.cpu() for x in items])

    @property
    def info(self):
        t = self._trace
        vals = [float(self.cfg.initial_cash)] + ([] if not t["values"] else self._stack(t["values"]).tolist())
        acts = [self._first_action.cpu().numpy()] + [a for a in (self._stack(t["actions"]).numpy() if t["actions"] else [])]
        rews = [0] + ([] if not t["rewards"] else self._stack(t["rewards"]).tolist())
        rets = [0] + ([] if not t["returns"] else self._stack(t["returns"]).tolist())
        return {"values": vals, "actions": acts, "rewards": rews, "returns": rets}

    @property
    def value(self):
        """`self.value` of the reference: INITIAL_CASH (a float) after reset (:27), then the 0-dim value tensor of the last
        step ON THE CALLER'S DEVICE (:89) — a CPU caller gets a host tensor, so `RolloutBuffer.add(..., env.value, r)` →
        `np.array(v)` (rollout_buffer.py:55) works as it does on the reference."""
        t = self._trace["values"]
        return t[-1] if t else float(self.cfg.initial_cash)

    def _write_weights(self, features):
        A, W, F = self._env.A, self._env.W, self._env.F
        if tuple(features.shape[-3:]) != (A, W, F):
            raise ValueError(f"features must be [{A}, {W}, {F}], got {tuple(features.shape)}")
        if features.is_cuda and features.dtype == torch.float32 and features.is_contiguous():
            self._env.write_weight_channel(features.view(1, A, W, F))
        elif not features.is_cuda:
            self._weights_to_host(features)
            torch.cuda.current_stream(self._env.device).synchronize()
            features[..., -1] = self._pinned()["obs"][0, :, :, -1]
        else:
            dev = features.to(device=self._env.device, dtype=torch.float32).contiguous().view(1, A, W, F)
            self._env.write_weight_channel(dev)
            features[..., -1] = dev[0, :, :, -1].to(device=features.device, dtype=features.dtype)
        return features

    def reset(self, features):
        """trading_env.py:21-41."""
        self._env.reset(obs=False)
        self._clear_trace()
        self._host_idx = 1
        return self._write_weights(features)

    def step(self, action, features, prices):
        """trading_env.py:44-105 → (r, features) (or (features, r, done) with three_tuple=True)."""
        A = self._env.A
        if action.numel() != A:
            raise ValueError(f"Action must have shape ({A},), got {tuple(action.shape)}")    # weight_buffer.py:18-19
        if not (action.is_cuda or features.is_cuda or prices.is_cuda):
            return self._step_host(action, features, prices)
        e = self._env
        fast = (action.is_cuda and prices.is_cuda and action.dtype is torch.float32 and prices.dtype is torch.float32
                and action.is_contiguous() and prices.is_contiguous() and prices.numel() == A)
        if fast:                                           # device tensors as they are: no torch ops before the launch
            rc = e.lib.pmrl_env_step(e._p_cfg, e._p_tbl, e._p_st, action.data_ptr(), prices.data_ptr(), e._ptr_reward, e._ptr_done,
                                     None, OBS_NONE, e._ptr_stats, _lib.current_stream())
            if rc:
                _lib.check(rc, "pmrl_env_step")
            r, done = e.reward, e.done
        else:
            _, r, done = e.step(action.reshape(1, A), y=prices.reshape(1, A), obs=False)
        slot = self._host_idx                              # E = 1, no auto-reset: the ring pointer is known on the host
        self._host_idx = (slot + 1) % e.W
        t = self._trace
        v = e.value[0].clone()
        rr = r[0].clone()
        v_before = t["values"][-1] if t["values"] else self.cfg.initial_cash
        if not isinstance(v_before, float) and v_before.device != v.device:
            v_before = v_before.to(v.device)
        t["values"].append(v)
        t["actions"].append(e.hist[0, slot].clone())
        t["rewards"].append(rr)
        t["returns"].append(v / v_before if self.cfg.commission == 0 else torch.exp(rr / self.cfg.reward_scale))
        features = self._write_weights(features)
        if self.three_tuple:
            return features, rr, done[0].clone()
        return rr, features
