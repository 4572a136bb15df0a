"""BatchedTradingEnv — E lockstep portfolio environments on one B200, driven through the C-ABI.

Keeps the reference env's reset/step contract (env/sim/trading_env.py:21-105) batched over E:

    obs = env.reset()                       # [E, A, W, F]   (TradingEnv.reset, :21-41)
    obs, reward, done = env.step(actions)   # actions [E, A] (TradingEnv.step,  :44-105)

All state lives in device tensors owned by torch; the kernels only borrow the pointers for the
enqueued work.  Nothing here syncs with the host; `stats()` is the only call that reads back.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from .config import EnvConfig

OBS_NONE, OBS_FULL, OBS_WEIGHTS = 0, 1, 2
OBS_BF16 = 0x100                  # OR-ed into OBS_FULL: the obs is written as bf16 (include/pmrl_b200.h PMRL_OBS_BF16)
OBS_TORCH_DTYPES = {"float32": torch.float32, "bfloat16": torch.bfloat16}
STATS_LEN = 10
STAT_NAMES = ("n_envs", "sum_r", "sum_r2", "sum_v", "sum_lnv", "n_done", "sum_ep_return", "sum_ep_len",
              "max_v", "max_neg_v")


def _as_f32_cuda(x, device):
    t = torch.as_tensor(x)
    return t.to(device=device, dtype=torch.float32).contiguous()


class BatchedTradingEnv:
    """E independent `TradingEnv`s advanced by one fused CUDA launch per step.

    Args:
        cfg:       EnvConfig (reference config surface).
        prices:    [T, A, C] price table (OHLC; `close_channel` selects the close used for
                   y_t = close_t / close_{t-1}, data/instrument.py:79), or None if every step gets `y=`.
        features:  [T, A, F-1] feature table gathered into the obs window (defaults to `prices` when its
                   channel count is F-1); FFD'ed / scaled tables come from `pmrl_b200.features`.
        t0:        [E] int episode offsets into the table (default 0); redrawn at every reset once
                   `sample_episode_starts` attaches a sampler.
        collect_stats: accumulate the PMRL_STAT_* vector on device every step.

    With `cfg.obs_dtype == "bfloat16"` every obs this env returns or writes (`reset`, `step`, `step_io`, `step_host`,
    `graphed_step`, `observe`, and `out=` buffers, which must then be bfloat16) is the bf16 rounding of the fp32 obs;
    state, rewards and the buffer rows written through `step_io` stay fp32.

    With `cfg.obs_relative_to = ref` the same obs are window-relative: channel c in `cfg.obs_relative_channels` of every
    asset's window is divided (IEEE fp32 division) by channel `ref` of that window's last row, inside the obs kernels;
    the weight channel, state and rewards are unchanged.
    """

    @classmethod
    def from_tables(cls, cfg: EnvConfig, close_tm, feat_am, t0=None, device=None, collect_stats: bool = False):
        """Construct from tables already in the kernel layouts (close_tm [T, A], feat_am [A, T, F-1]), e.g. the
        output of `pmrl_b200.features.build_env_tables`."""
        return cls(cfg, t0=t0, device=device, collect_stats=collect_stats, _packed=(close_tm, feat_am))

    def __init__(self, cfg: EnvConfig, prices=None, features=None, t0=None, close_channel: int = 3,
                 device=None, collect_stats: bool = False, _packed=None):
        if not torch.cuda.is_available():
            raise _lib.PmrlError("BatchedTradingEnv needs a CUDA device (pmrl_b200 has no CPU fallback)")
        self.lib = _lib.load()
        self.cfg = cfg
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        E, A, W, F = cfg.num_envs, cfg.num_assets, cfg.window_size, cfg.num_features
        self.E, self.A, self.W, self.F = E, A, W, F
        self.obs_dtype = OBS_TORCH_DTYPES[cfg.obs_dtype]
        # obs_mode of every obs this env makes
        self._obs_full = OBS_FULL | (OBS_BF16 if self.obs_dtype is torch.bfloat16 else 0) | cfg.obs_relative_bits
        dev = self.device
        self.close_tm = None
        self.feat_am = None
        self.T = 0
        if _packed is not None:
            ctm, fam = _packed
            if ctm is not None:
                self.close_tm = _as_f32_cuda(ctm, dev)
                if self.close_tm.dim() != 2 or self.close_tm.shape[1] != A:
                    raise ValueError(f"close_tm must be [T, {A}]")
                self.T = self.close_tm.shape[0]
            if fam is not None:
                self.feat_am = _as_f32_cuda(fam, dev)
                if self.feat_am.dim() != 3 or self.feat_am.shape[0] != A or self.feat_am.shape[2] != F - 1:
                    raise ValueError(f"feat_am must be [{A}, T, {F - 1}]")
                if self.T and self.feat_am.shape[1] != self.T:
                    raise ValueError("close_tm and feat_am must have the same number of rows")
                self.T = self.feat_am.shape[1]
        if prices is not None:
            p = _as_f32_cuda(prices, dev)
            if p.dim() != 3 or p.shape[1] != A:
                raise ValueError(f"prices must be [T, {A}, C], got {tuple(p.shape)}")
            self.T = p.shape[0]
            self.close_tm = p[:, :, close_channel].contiguous()                  # [T, A]
            if features is None and p.shape[2] == F - 1:
                features = p
        if features is not None:
            f = _as_f32_cuda(features, dev)
            if f.dim() != 3 or f.shape[1] != A or f.shape[2] != F - 1:
                raise ValueError(f"features must be [T, {A}, {F - 1}], got {tuple(f.shape)}")
            if self.T and f.shape[0] != self.T:
                raise ValueError("prices and features must have the same number of rows")
            self.T = f.shape[0]
            self.feat_am = f.permute(1, 0, 2).contiguous()                       # [A, T, F-1]
        if t0 is None:
            self.t0 = torch.zeros(E, dtype=torch.int32, device=dev)
        else:
            self.t0 = torch.as_tensor(t0).to(device=dev, dtype=torch.int32).contiguous()
            if self.t0.shape != (E,):
                raise ValueError(f"t0 must be [{E}]")
        if W < 2:
            raise ValueError("window_size must be >= 2 (the reference ring indexes row 1 on reset, weight_buffer.py:9-10)")
        if self.T:
            if cfg.episode_len <= 0:
                # rows [t0 + k, t0 + k + W) are gathered from the tables: without an episode length k would leave them
                raise ValueError("episode_len must be > 0 when the env reads price / feature tables")
            need = int(self.t0.max().item()) + cfg.episode_len + W if E else 0
            if need > self.T:
                raise ValueError(f"table too short: max(t0) + episode_len + W = {need} > T = {self.T}")
            if E and int(self.t0.min().item()) < 0:
                raise ValueError("t0 must be >= 0")
        # ---- state (SURVEY.md Appendix A) ----
        self.value = torch.empty(E, dtype=torch.float32, device=dev)
        self.hist = torch.empty(E, W, A, dtype=torch.float32, device=dev)
        self.idx = torch.empty(E, dtype=torch.int32, device=dev)
        self.is_full = torch.empty(E, dtype=torch.uint8, device=dev)
        self.t = torch.empty(E, dtype=torch.int32, device=dev)
        self.sharpe = torch.zeros(E, 3, dtype=torch.float64, device=dev) if cfg.reward_mode == 3 else None
        self.ep_return = torch.zeros(E, dtype=torch.float32, device=dev)
        self.reward = torch.zeros(E, dtype=torch.float32, device=dev)
        self.done = torch.zeros(E, dtype=torch.uint8, device=dev)
        # work counters of the fused kernel's dynamic group hand-out: owned by THIS batch (two envs on two streams never share)
        self._ticket = torch.zeros(2, dtype=torch.int32, device=dev)
        self._stats = None
        if collect_stats:
            self._stats = torch.zeros(STATS_LEN, dtype=torch.float64, device=dev)
            self.clear_stats()
        self._obs = None
        # ---- C structs (built once; the hot call only passes pointers) ----
        self._c_cfg = _lib.PmrlEnvCfg(E, A, W, F, self.T, cfg.episode_len, cfg.reward_mode, cfg.mu_max_iter,
                                      1 if cfg.strict_reference else 0, cfg.initial_cash, cfg.commission,
                                      cfg.reward_scale, cfg.risk_free_rate)
        # price relatives y[t] = close[t] / close[t-1], once per table (instrument.py:79): the table the step kernels read
        self.y_tm = None
        if self.close_tm is not None:
            self.y_tm = torch.empty_like(self.close_tm)
            _lib.check(self.lib.pmrl_price_relatives(self.close_tm.data_ptr(), self.T, A, self.y_tm.data_ptr(),
                                                     _lib.current_stream()), "pmrl_price_relatives")
        # channel-padded copy of the feature table ([A, T, 4*ceil((F-1)/4)]) for the fused step+obs kernel when F - 1 is not a
        # multiple of four (e.g. OHLC + ema: F = 6, OHLC + bbands: F = 8); the pad channels are never copied to obs
        self.feat_am4 = None
        if self.feat_am is not None and (F - 1) % 4 != 0 and F <= 17:
            c4 = (F + 2) // 4
            self.feat_am4 = torch.zeros(A, self.T, 4 * c4, dtype=torch.float32, device=dev)
            self.feat_am4[:, :, :F - 1] = self.feat_am
        self._c_tbl = _lib.PmrlTables(_lib.ptr(self.y_tm), _lib.ptr(self.feat_am), _lib.ptr(self.feat_am4))
        self._c_st = _lib.PmrlEnvState(_lib.ptr(self.value), _lib.ptr(self.hist), _lib.ptr(self.idx),
                                       _lib.ptr(self.is_full), _lib.ptr(self.t), _lib.ptr(self.t0),
                                       _lib.ptr(self.sharpe), _lib.ptr(self.ep_return), _lib.ptr(self._ticket))
        self._io = _lib.PmrlStepIO()
        self._p_io = C.byref(self._io)
        self._p_cfg, self._p_tbl, self._p_st = C.byref(self._c_cfg), C.byref(self._c_tbl), C.byref(self._c_st)
        self._ptr_reward, self._ptr_done, self._ptr_stats = _lib.ptr(self.reward), _lib.ptr(self.done), _lib.ptr(self._stats)
        self._eval = None                 # StreamingEvalMetrics fed after every reset / step (track_eval_metrics)
        self._starts = None               # EpisodeStarts drawing t0 before every reset (sample_episode_starts)
        self.reset(obs=False)

    # ------------------------------------------------------------------------------------------
    def _obs_buffer(self, out):
        if out is not None:
            if out.shape != (self.E, self.A, self.W, self.F) or out.dtype != self.obs_dtype:
                raise ValueError(f"obs out must be {str(self.obs_dtype).replace('torch.', '')} [{self.E}, {self.A}, {self.W}, "
                                 f"{self.F}] (the env's obs_dtype), got {out.dtype} {tuple(out.shape)}")
            return out
        if self._obs is None:
            self._obs = torch.empty(self.E, self.A, self.W, self.F, dtype=self.obs_dtype, device=self.device)
        return self._obs

    def reset(self, mask=None, obs: bool = True, out=None):
        """TradingEnv.reset batched (trading_env.py:21-41): re-initialise the masked envs (all if None).
        Returns the obs buffer [E, A, W, F] (rows of unmasked envs are left untouched) or None."""
        m = None
        if mask is not None:
            m = torch.as_tensor(mask).to(device=self.device, dtype=torch.uint8).contiguous()
        want_obs = obs and self.feat_am is not None
        buf = self._obs_buffer(out) if want_obs else None
        if self._starts is not None:
            self._starts.draw_mask(m)
        rc = self.lib.pmrl_env_reset(self._p_cfg, self._p_tbl, self._p_st, _lib.ptr(m), _lib.ptr(buf),
                                     self._obs_full if want_obs else OBS_NONE, _lib.current_stream())
        _lib.check(rc, "pmrl_env_reset")
        if self._eval is not None:
            self._eval.update()
        return buf

    def step(self, actions, y=None, obs: bool = True, out=None):
        """TradingEnv.step batched (trading_env.py:44-105).

        actions [E, A] (raw scores or weights; also accepts [E, A, 1]); y: optional external price
        relatives [E, A] (else computed from the close table).  Returns (obs | None, reward [E], done [E] u8);
        the returned tensors are the env's own buffers and are overwritten by the next step."""
        a = actions
        if not (a.is_cuda and a.dtype is torch.float32 and a.is_contiguous() and a.numel() == self.E * self.A):   # else: hot path, no torch ops
            if a.dtype != torch.float32 or not a.is_cuda:
                a = a.to(device=self.device, dtype=torch.float32)
            a = a.reshape(self.E, self.A).contiguous()
        if y is not None:
            y = y.to(device=self.device, dtype=torch.float32).reshape(self.E, self.A).contiguous()
        want_obs = obs and self.feat_am is not None
        buf = self._obs_buffer(out) if want_obs else None
        if self._starts is not None:
            self._starts.draw_due()
        rc = self.lib.pmrl_env_step(self._p_cfg, self._p_tbl, self._p_st, a.data_ptr(), _lib.ptr(y),
                                    self._ptr_reward, self._ptr_done, buf.data_ptr() if buf is not None else None,
                                    self._obs_full if want_obs else OBS_NONE, self._ptr_stats,
                                    _lib.current_stream())
        if rc:
            _lib.check(rc, "pmrl_env_step")
        if self._eval is not None:
            self._eval.update()
        return buf, self.reward, self.done

    def step_io(self, actions, y=None, obs: bool = True, out=None, reward=None, done=None, action_sink=None,
                value_sink=None, weight_sink=None, index_sink=None):
        """`step` with the kernel writing straight into caller-owned rows (C-ABI pmrl_env_step_io): `reward` [E] f32 /
        `done` [E] u8 replace the env's own buffers (e.g. the r row of a rollout slot), `action_sink` [E, A] receives the raw
        action, `value_sink` [E] the post-step value, `weight_sink` [E, A] the post-drift weights, `index_sink` [E] i32 the
        loader item index t0 + k — the rows RolloutBuffer.add / ReplayBuffer.add would copy (rollout_buffer.py:51-57,
        buffer.py:31-37).  All tensors must be contiguous CUDA tensors of the exact dtype; nothing is copied or cast."""
        a = actions
        if not (a.is_cuda and a.dtype is torch.float32 and a.is_contiguous() and a.numel() == self.E * self.A):
            a = a.to(device=self.device, dtype=torch.float32).reshape(self.E, self.A).contiguous()
        if y is not None:
            y = y.to(device=self.device, dtype=torch.float32).reshape(self.E, self.A).contiguous()
        want_obs = obs and self.feat_am is not None
        buf = self._obs_buffer(out) if want_obs else None
        E, A = self.E, self.A
        for name, t, dt, n in (("reward", reward, torch.float32, E), ("done", done, torch.uint8, E),
                               ("action_sink", action_sink, torch.float32, E * A), ("value_sink", value_sink, torch.float32, E),
                               ("weight_sink", weight_sink, torch.float32, E * A), ("index_sink", index_sink, torch.int32, E)):
            if t is not None and (t.dtype is not dt or t.numel() != n or not t.is_cuda or not t.is_contiguous()):
                raise _lib.PmrlError(f"step_io: {name} must be a contiguous CUDA {dt} tensor of {n} elements")
        io = self._io
        io.actions, io.y_ext = a.data_ptr(), _lib.ptr(y)
        io.reward = reward.data_ptr() if reward is not None else self._ptr_reward
        io.done = done.data_ptr() if done is not None else self._ptr_done
        io.obs, io.obs_mode, io.stats = _lib.ptr(buf), (self._obs_full if want_obs else OBS_NONE), self._ptr_stats
        io.action_sink, io.value_sink = _lib.ptr(action_sink), _lib.ptr(value_sink)
        io.weight_sink, io.index_sink = _lib.ptr(weight_sink), _lib.ptr(index_sink)
        io.reward_host = io.done_host = None
        if self._starts is not None:
            self._starts.draw_due()
        rc = self.lib.pmrl_env_step_io(self._p_cfg, self._p_tbl, self._p_st, self._p_io, _lib.current_stream())
        if rc:
            _lib.check(rc, "pmrl_env_step_io")
        if self._eval is not None:
            self._eval.update()
        return buf, (reward if reward is not None else self.reward), (done if done is not None else self.done)

    def step_burst(self, actions, reward=None, done=None):
        """K state-only steps in ONE launch on pre-supplied actions [K, E, A] (imagination bursts, HORIZON = 15 in
        config/dreamer.py:54): returns (reward [K, E], done [K, E]); bit-identical to K calls of `step(obs=False)`."""
        if self._eval is not None:
            raise _lib.PmrlError("step_burst: this env tracks evaluation metrics (track_eval_metrics), which need every "
                                 "step's state; a burst keeps its intermediate states in registers — use step / graphed_step")
        if self._starts is not None:
            raise _lib.PmrlError("step_burst: this env draws episode starts (sample_episode_starts); an episode ending inside "
                                 "a burst would auto-reset with a stale t0 — use step / graphed_step, or detach() the sampler")
        a = actions
        if not (a.is_cuda and a.dtype is torch.float32 and a.is_contiguous() and a.dim() >= 2 and a[0].numel() == self.E * self.A):
            a = a.to(device=self.device, dtype=torch.float32).reshape(-1, self.E, self.A).contiguous()
        K = a.shape[0]
        if reward is None:
            reward = torch.empty(K, self.E, dtype=torch.float32, device=self.device)
        if done is None:
            done = torch.empty(K, self.E, dtype=torch.uint8, device=self.device)
        if reward.numel() != K * self.E or done.numel() != K * self.E or reward.dtype is not torch.float32 or done.dtype is not torch.uint8:
            raise _lib.PmrlError("step_burst: reward [K, E] float32 / done [K, E] uint8 expected")
        rc = self.lib.pmrl_env_step_burst(self._p_cfg, self._p_tbl, self._p_st, a.data_ptr(), K, _lib.ptr(reward), _lib.ptr(done),
                                          self._ptr_stats, _lib.current_stream())
        if rc:
            _lib.check(rc, "pmrl_env_step_burst")
        return reward, done

    # ------------------------------------------------------------------------------------------
    def step_host(self, actions_host, reward_host=None, done_host=None, obs: bool = True, out=None, chunks: int = 0):
        """One step driven from HOST buffers (the reference loop's call with CPU tensors, train/on_policy.py:64-65):
        `actions_host` [E, A] float32 (pinned, so the copies overlap) in, `reward_host` [E] f32 / `done_host` [E] u8 out.
        With `chunks` = 0 and pinned actions the kernel reads them in place over PCIe (zero-copy, one launch); otherwise
        pmrl_env_step_host issues the batch as env slices so that the host→device copy of slice c+1 and the
        device→host copy of slice c-1 run under the kernel of slice c (`chunks` > 0: that many geometrically growing
        slices, < 0: equal slices; pageable actions with 0: five slices).  Blocks until the results are on the host.
        Returns (obs | None, reward_host, done_host)."""
        E, A = self.E, self.A
        if actions_host.dtype != torch.float32 or actions_host.is_cuda or actions_host.numel() != E * A or not actions_host.is_contiguous():
            raise _lib.PmrlError("step_host: actions_host must be a contiguous CPU float32 tensor of E*A elements")
        if reward_host is None:
            reward_host = torch.empty(E, dtype=torch.float32).pin_memory()
        if done_host is None:
            done_host = torch.empty(E, dtype=torch.uint8).pin_memory()
        if (reward_host.dtype != torch.float32 or done_host.dtype != torch.uint8 or reward_host.numel() != E or done_host.numel() != E
                or reward_host.is_cuda or done_host.is_cuda or not reward_host.is_contiguous() or not done_host.is_contiguous()):
            raise _lib.PmrlError("step_host: reward_host [E] float32 / done_host [E] uint8 CPU tensors expected")
        stage = self.__dict__.get("_host_stage")
        if stage is None:
            stage = self._host_stage = torch.empty(E, A, dtype=torch.float32, device=self.device)
        want_obs = obs and self.feat_am is not None
        buf = self._obs_buffer(out) if want_obs else None
        if self._starts is not None:
            self._starts.draw_due()                       # every kernel of pmrl_env_step_host runs on this stream after it
        rc = self.lib.pmrl_env_step_host(self._p_cfg, self._p_tbl, self._p_st, actions_host.data_ptr(), stage.data_ptr(),
                                         self.reward.data_ptr(), self.done.data_ptr(), reward_host.data_ptr(),
                                         done_host.data_ptr(), _lib.ptr(buf), self._obs_full if want_obs else OBS_NONE,
                                         _lib.ptr(self._stats), int(chunks), _lib.current_stream())
        _lib.check(rc, "pmrl_env_step_host")
        if self._eval is not None:
            self._eval.update()
        return buf, reward_host, done_host

    def graphed_step(self, obs: bool = True, out=None, steps: int = 1):
        """Capture `steps` consecutive steps in ONE CUDA graph (launch-bound small batches: 4,096 x 50 moves 1.7 MB per
        state-only step; imagination rollouts advance in fixed bursts, cf. HORIZON = 15 in config/dreamer.py:54).
        Returns (static_actions, replay): fill `static_actions` ([E, A] for steps == 1, else [steps, E, A]) in place, then
        call `replay()`, which returns (obs, reward, done) like `step` — for steps > 1 reward and done are [steps, E]
        (one row per captured step; the obs buffer is rewritten by every step and holds the last one).  The kernels take no host-side decisions after
        validation, so the captured launches are valid for every later burst (auto-resets included).  Replays of one
        captured graph must not overlap each other (they share these static buffers)."""
        K = int(steps)
        if K < 1:
            raise ValueError("steps must be >= 1")
        shape = (self.E, self.A) if K == 1 else (K, self.E, self.A)
        static_actions = torch.zeros(*shape, dtype=torch.float32, device=self.device)
        acts = [static_actions] if K == 1 else [static_actions[k] for k in range(K)]
        rew = torch.zeros(K, self.E, dtype=torch.float32, device=self.device) if K > 1 else None
        dn = torch.zeros(K, self.E, dtype=torch.uint8, device=self.device) if K > 1 else None
        state = (self.value, self.hist, self.idx, self.is_full, self.t, self.ep_return) + ((self.sharpe,) if self.sharpe is not None else ())
        if self._eval is not None:
            state += (self._eval.acc,)                    # the captured steps include the metrics update
        if self._starts is not None:
            state += (self.t0, self._starts.episodes)     # ... and the episode-start draws

        def burst():
            res = None
            for k in range(K):
                res = self.step(acts[k], obs=obs, out=out)
                if K > 1:
                    rew[k].copy_(res[1]); dn[k].copy_(res[2])
            return res if K == 1 else (res[0], rew, dn)

        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):                        # warm-up launch outside capture (lazy module loading, smem attributes)
            snap = [t.clone() for t in state]
            stats_snap = self._stats.clone() if self._stats is not None else None
            self.step(acts[0], obs=obs, out=out)
            for dst, src in zip(state, snap):
                dst.copy_(src)                            # undo the warm-up transition
            if stats_snap is not None:
                self._stats.copy_(stats_snap)
        torch.cuda.current_stream(self.device).wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            result = burst()
        for dst, src in zip(state, snap):
            dst.copy_(src)                                # capture does not execute, but keep the state explicit
        if stats_snap is not None:
            self._stats.copy_(stats_snap)

        # the graph holds raw pointers into `state` (the metrics accumulator and the sampler's draw counters among them):
        # the closure keeps those tensors alive even if the tracker or sampler is replaced and dropped later
        def replay(_keep=state):
            g.replay()
            return result

        return static_actions, replay

    def track_eval_metrics(self, rf: float = 0.0, periods: int = 252):
        """Accumulate `loops.evaluate`'s metrics of every episode on the device as the env runs (util/eval.py:14-37),
        in 128 bytes per env instead of value / weight traces.  From now on `reset`, `step`, `step_io`, `step_host` and
        `graphed_step` (captured after this call) enqueue one `pmrl_eval_stream_update` right after their own launch;
        `step_burst` raises.  Metrics start at each env's next reset: an env that is mid-episode now reads NaN until
        then, an env at local step 0 starts at once.  A later call replaces the tracker.  Returns the
        `metrics.StreamingEvalMetrics` (`running()`, `last_episode()`, `episode_mean()`, `clear()`)."""
        from .metrics import StreamingEvalMetrics
        tracker = StreamingEvalMetrics(self, rf=rf, periods=periods)
        tracker.update()
        self._eval = tracker
        return tracker

    def sample_episode_starts(self, low: int = 0, high=None, seed: int = 0, distribution: str = "uniform", beta=None,
                              first_env: int = 0):
        """Give every env a freshly drawn table offset t0[e] at each of its resets, on the device, instead of replaying the
        offset it was built with.  From now on `reset(mask)` draws for the masked envs, and `step`, `step_io`, `step_host`
        and `graphed_step` (captured after this call) draw for the envs the step auto-resets, each before its own launch;
        `step_burst` raises.  The obs of a reset, `index_sink` and the rest of that episode use the new offset; between a
        done step and the next call `t0` still holds the finished episode's start.  The first draw happens at each env's
        next reset.

        distribution "uniform" draws t0 uniformly from [low, high]; "geometric" draws t0 = high - j with
        P(j) ∝ beta (1 - beta)^j, j < high - low + 1 (recent rows favoured).  high=None means T - episode_len - W.
        first_env is the global id of env 0 (a rank passes `dist.shard_range(...)[0]`): a draw depends only on (seed,
        global env id, that env's draw count).  A later call replaces the sampler.  Returns the `starts.EpisodeStarts`
        (`episodes`: draws per env; `detach()`)."""
        from .starts import EpisodeStarts, start_dist
        dist = start_dist(self.T, self.cfg.episode_len, self.W, low=low, high=high, seed=seed, distribution=distribution,
                          beta=beta, first_env=first_env)
        sampler = EpisodeStarts(self, dist)
        self._starts = sampler
        return sampler

    def write_weight_channel(self, obs):
        """features[:, :, -1] = weights.get_all() on a caller-filled obs [E, A, W, F] (trading_env.py:103).  fp32 envs only."""
        if self.obs_dtype is not torch.float32:
            raise _lib.PmrlError("write_weight_channel overwrites channel F-1 of a float32 obs; this env's obs_dtype is bfloat16")
        rc = self.lib.pmrl_obs_build(self._p_cfg, self._p_tbl, self._p_st, _lib.ptr(obs), OBS_WEIGHTS,
                                     _lib.current_stream())
        _lib.check(rc, "pmrl_obs_build")
        return obs

    def observe(self, out=None):
        """Materialise the obs of the current state without stepping."""
        buf = self._obs_buffer(out)
        rc = self.lib.pmrl_obs_build(self._p_cfg, self._p_tbl, self._p_st, _lib.ptr(buf), self._obs_full,
                                     _lib.current_stream())
        _lib.check(rc, "pmrl_obs_build")
        return buf

    # ------------------------------------------------------------------------------------------
    @property
    def weights_last(self):
        """ActionBuffer.get_last batched (weight_buffer.py:28-30) → [E, A]."""
        last = ((self.idx.long() - 1) % self.W)
        return self.hist[torch.arange(self.E, device=self.device), last]

    def clear_stats(self):
        if self._stats is not None:
            self._stats.zero_()
            self._stats[8:] = float("-inf")

    def stats(self, all_reduce: bool = False, clear: bool = True):
        """Read the device statistics vector (one host sync).  With all_reduce=True the vector is first
        summed (max for the extrema) across the ranks of the default process group."""
        if self._stats is None:
            raise _lib.PmrlError("construct the env with collect_stats=True")
        v = self._stats.clone()
        if all_reduce:
            from .dist import all_reduce_stats
            v = all_reduce_stats(v)
        h = v.cpu().tolist()
        if clear:
            self.clear_stats()
        d = dict(zip(STAT_NAMES, h))
        n = max(d["n_envs"], 1.0)
        d["mean_reward"] = d["sum_r"] / n
        d["mean_value"] = d["sum_v"] / n
        d["min_v"] = -d.pop("max_neg_v")
        d["mean_ep_return"] = d["sum_ep_return"] / max(d["n_done"], 1.0)
        return d
