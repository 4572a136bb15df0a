"""Device-resident rollout / replay buffers in the reference layouts, batched over E envs.

  DeviceRolloutBuffer  ↔ replay/rollout_buffer.py:7-142 (on-policy epoch buffer)
      s [S, E, A, W, F], a [S, E, A], v [S, E], r [S, E], prices y [S, E, A];  S = epoch_len + 1
  DeviceReplayBuffer   ↔ replay/buffer.py:6-79 / replay/traj_buffer.py:6-89 (off-policy *index* replay)
      i [P, L, E] int32, a [P, L, E, A], r [P, L, E]; windows are re-gathered from the feature table on sample

The step kernel can write its observation straight into `rollout.obs_slot(...)` ("obs directly into the
buffer layout"); `add` then only appends the small a / v / r rows.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from .config import obs_relative_bits, obs_relative_check

_OBS_FULL, _OBS_BF16 = 1, 0x100                               # include/pmrl_b200.h PMRL_OBS_FULL, PMRL_OBS_BF16
_OBS_DTYPES = {"float32": torch.float32, "bfloat16": torch.bfloat16}


def _obs_dtype(name):
    if name not in _OBS_DTYPES:
        raise ValueError(f"unknown obs_dtype {name!r}; expected one of {tuple(_OBS_DTYPES)}")
    return _OBS_DTYPES[name]


class DeviceRolloutBuffer:
    """On-policy epoch buffer (replay/rollout_buffer.py:7-142) batched over E envs, in one of two storage modes:

    mode="full"   s [S, E, A, W, F] is stored like the reference does (`np.zeros((E+1, A, W, F))`, :17) — 4·A·W·F bytes
                  per env-step (13 GB per slot at 131,072 envs x 100 assets): a handful of slots fit.
    mode="index"  per slot only the loader index bi [S, E], the raw action a [S, E, A], v, r and the un-wrapped history
                  of post-drift weights wp [S + W - 1, E, A]; `gather` regenerates s (window by index from the device
                  table, ring-ordered weight channel from wp) exactly like the off-policy buffer regenerates its windows
                  (replay/buffer.py:58-77).  8·A + 12 bytes per env-step: an epoch of 1,000 steps at 65,536 envs x 100
                  assets is 53 GB instead of 6.5 TB.  Needs the env's tables (`feat_am`, `y_tm`).

    Either way the rows of a slot are written by the step kernel itself: `sinks(step)` returns the keyword arguments for
    `BatchedTradingEnv.step_io` (reward → r[slot], action_sink → a[slot], value_sink → v[slot], obs out → s[slot + 1], …),
    so no copy kernel runs per step.  `add` keeps the reference's call (rollout_buffer.py:43-57) for callers that have
    the rows elsewhere.

    obs_dtype="bfloat16": s is stored (full mode) and returned by `gather` / `sample` / `sample_random` (both modes) as
    bf16, half the bytes; the env feeding it must have the same obs_dtype.  a, v, r, prices stay fp32.

    obs_relative_to / obs_relative_channels (index mode): the regenerated windows are window-relative like those of an env
    with the same `EnvConfig` settings, so a sample equals the obs the env returned.  A full-mode buffer stores what the env
    wrote and ignores them."""

    def __init__(self, num_features: int, train_len: int, num_envs: int, num_assets: int, window_size: int,
                 initial_cash: float = 25000.0, batch_size: int = 64, device=None, store_obs: bool = True,
                 mode: str = "full", feat_am=None, y_tm=None, obs_dtype: str = "float32",
                 obs_relative_to: int | None = None, obs_relative_channels=None):
        if not torch.cuda.is_available():
            raise _lib.PmrlError("DeviceRolloutBuffer needs a CUDA device (pmrl_b200 has no CPU fallback)")
        if mode not in ("full", "index"):
            raise ValueError("mode must be 'full' or 'index'")
        self.lib = _lib.load()
        self.mode = mode
        self.obs_dtype = _obs_dtype(obs_dtype)
        self._bf16 = self.obs_dtype is torch.bfloat16
        self.obs_relative_to = obs_relative_to
        self.obs_relative_channels = obs_relative_check(obs_relative_to, obs_relative_channels, num_features)
        self._obs_mode = _OBS_FULL | (_OBS_BF16 if self._bf16 else 0) | obs_relative_bits(obs_relative_to, self.obs_relative_channels)
        self.F, self.E, self.A, self.W = num_features, num_envs, num_assets, window_size
        self.step_offset = window_size - 1                      # rollout_buffer.py:10
        self.epoch_len = train_len - self.step_offset           # rollout_buffer.py:11
        self.S = self.epoch_len + 1
        self.batch_size = batch_size
        self.initial_cash = float(initial_cash)
        dev = torch.device(device or "cuda")
        self.device = dev
        S, E, A, W, F = self.S, self.E, self.A, self.W, self.F
        self.s = self.y = self.bi = self.wp = None
        self.feat_am, self.y_tm = feat_am, y_tm
        if mode == "full":
            self.s = torch.zeros(S, E, A, W, F, dtype=self.obs_dtype, device=dev) if store_obs else None
            self.y = torch.zeros(S, E, A, device=dev)           # `prices` (rollout_buffer.py:12), filled by set_prices/add
        else:
            if feat_am is None or y_tm is None:
                raise ValueError("mode='index' regenerates the windows on sample and needs feat_am [A, T, F-1] and y_tm [T, A]")
            self.T = feat_am.shape[1]
            self.bi = torch.zeros(S, E, dtype=torch.int32, device=dev)
            self.wp = torch.zeros(S + W - 1, E, A, device=dev)  # wp[m] = w' after step m; wp[0] = all cash
        self.a = torch.zeros(S, E, A, device=dev)
        self.v = torch.zeros(S, E, device=dev)
        self.r = torch.zeros(S, E, device=dev)
        self.reset()

    def nbytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in (self.s, self.y, self.bi, self.wp, self.a, self.v, self.r) if t is not None)

    def reset(self):
        """rollout_buffer.py:29-41 — slot 0 holds the all-cash action and the initial value."""
        if self.s is not None:
            self.s.zero_()
        self.a.zero_(); self.v.zero_(); self.r.zero_()
        self.a[0, :, 0] = 1.0
        self.v[0] = self.initial_cash
        if self.wp is not None:
            self.wp.zero_(); self.bi.zero_()
            self.wp[0, :, 0] = 1.0
        self.step = 1

    def set_prices(self, y):
        """y: price relatives per slot [S, E, A] (the reference passes train_prices[W-1:] at construction)."""
        if self.y is None:
            raise _lib.PmrlError("an index-mode rollout buffer reads the price relatives from y_tm")
        self.y.copy_(torch.as_tensor(y).to(self.device, torch.float32).reshape(self.S, self.E, self.A))

    def fill_prices(self, env):
        """`prices[W-1:]` of the reference constructor (rollout_buffer.py:12) for envs driven from a table: slot k holds the
        price relatives the step of that slot saw, y_tm[t0 + k + 2(W-1)].  One-time setup gather."""
        if self.y is None:
            return
        rows = env.t0.long()[None, :] + torch.arange(self.S, device=self.device)[:, None] + 2 * (self.W - 1)
        self.y.copy_(env.y_tm[rows.clamp_(max=env.T - 1)])

    def slot_of(self, step=None):
        """Slot that add() will write for loader step `step` (None → the current one), or -1 while step <= W-1."""
        st = self.step if step is None else step
        return st - self.step_offset if st > self.step_offset else -1

    def obs_slot(self, step=None):
        """View s[slot] ([E, A, W, F]) for the step kernel to write the observation into directly, or None."""
        k = self.slot_of(step)
        return self.s[k] if (0 <= k < self.S and self.s is not None) else None

    def sinks(self, step=None):
        """Keyword arguments for `BatchedTradingEnv.step_io` so that the kernel stepping loader item `step` writes this
        buffer's rows itself (then call `advance()` instead of `add()`): the obs the step RETURNS is the obs stored
        with the next step (on_policy.py:65 stores the obs before the step), so it goes to s[slot + 1]."""
        st = self.step if step is None else step
        k = self.slot_of(st)
        kw = {}
        if 0 <= k < self.S:
            kw.update(reward=self.r[k], action_sink=self.a[k], value_sink=self.v[k])
            if self.bi is not None:
                kw["index_sink"] = self.bi[k]
        if self.wp is not None and st < self.wp.shape[0]:
            kw["weight_sink"] = self.wp[st]
        nxt = self.obs_slot(st + 1)
        if nxt is not None:
            kw["out"] = nxt
        return kw

    def advance(self):
        self.step += 1

    def add(self, s, a, v, r, y=None):
        """rollout_buffer.py:43-57 batched: s [E,A,W,F] (None if already written through obs_slot), a [E,A(,1)], v [E], r [E]."""
        if self.mode == "index":
            raise _lib.PmrlError("an index-mode rollout buffer is filled through sinks() / step_io (it stores no observations)")
        if self.step > self.step_offset:
            slot = self.step - self.step_offset
            if slot >= self.S:
                raise IndexError("rollout buffer overflow: more steps than train_len")
            a2 = a.reshape(self.E, self.A).to(torch.float32).contiguous()
            v2 = v.reshape(self.E).to(torch.float32).contiguous()
            r2 = r.reshape(self.E).to(torch.float32).contiguous()
            s2 = None
            if s is not None and self.s is not None and s.data_ptr() != self.s[slot].data_ptr():
                if self._bf16:                                  # converting copy into the bf16 slot (round to nearest even)
                    self.s[slot].copy_(s.reshape(self.E, self.A, self.W, self.F))
                else:
                    s2 = s.reshape(self.E, self.A, self.W, self.F).to(torch.float32).contiguous()
            rc = self.lib.pmrl_rollout_add(self.E, self.A, self.W, self.F, slot, _lib.ptr(s2), _lib.ptr(a2), _lib.ptr(v2),
                                           _lib.ptr(r2), _lib.ptr(self.s), _lib.ptr(self.a), _lib.ptr(self.v),
                                           _lib.ptr(self.r), _lib.current_stream())
            _lib.check(rc, "pmrl_rollout_add")
            if y is not None:
                self.y[slot].copy_(y.reshape(self.E, self.A))
        self.step += 1

    def _check_slots(self, slots):
        """slot - 1 is read (rollout_buffer.py:130-131): slots must lie in [1, S).  Checked on the host when the indices
        are host data; device tensors are trusted (no sync on the sampling path)."""
        if not (torch.is_tensor(slots) and slots.is_cuda):
            arr = np.asarray(slots)
            if arr.size and (arr.min() < 1 or arr.max() >= self.S):
                raise IndexError(f"rollout gather: slots must be in [1, {self.S}), got [{arr.min()}, {arr.max()}]")

    def gather(self, slots, envs):
        """One minibatch (rollout_buffer.py:125-140): tensors shaped like the reference's
        (s [B,A,W,F], a [B,A,1], r [B,1,1], _v [B,1,1], _a [B,A,1], p [B,A,1])."""
        self._check_slots(slots)
        slots = torch.as_tensor(slots).to(self.device, torch.int32).contiguous()
        envs = torch.as_tensor(envs).to(self.device, torch.int32).contiguous()
        B = slots.numel()
        A, W, F, dev = self.A, self.W, self.F, self.device
        s = torch.empty(B, A, W, F, dtype=self.obs_dtype, device=dev)
        a = torch.empty(B, A, 1, device=dev); r = torch.empty(B, 1, 1, device=dev)
        pv = torch.empty(B, 1, 1, device=dev); pa = torch.empty(B, A, 1, device=dev); p = torch.empty(B, A, 1, device=dev)
        if self.mode == "index":
            rc = self.lib.pmrl_rollout_gather_index_obs(self.S, self.E, A, W, F, self.T, B, _lib.ptr(slots), _lib.ptr(envs),
                                                        _lib.ptr(self.bi), _lib.ptr(self.a), _lib.ptr(self.v), _lib.ptr(self.r),
                                                        _lib.ptr(self.wp), _lib.ptr(self.feat_am), _lib.ptr(self.y_tm),
                                                        _lib.ptr(s), _lib.ptr(a), _lib.ptr(r), _lib.ptr(pv), _lib.ptr(pa),
                                                        _lib.ptr(p), self._obs_mode, _lib.current_stream())
            _lib.check(rc, "pmrl_rollout_gather_index")
            return s, a, r, pv, pa, p
        if self.s is None:
            raise _lib.PmrlError("this rollout buffer was built with store_obs=False")
        gather = self.lib.pmrl_rollout_gather_bf16 if self._bf16 else self.lib.pmrl_rollout_gather
        rc = gather(self.S, self.E, A, W, F, B, _lib.ptr(slots), _lib.ptr(envs), _lib.ptr(self.s),
                                          _lib.ptr(self.a), _lib.ptr(self.v), _lib.ptr(self.r), _lib.ptr(self.y),
                                          _lib.ptr(s), _lib.ptr(a), _lib.ptr(r), _lib.ptr(pv), _lib.ptr(pa), _lib.ptr(p),
                                          _lib.current_stream())
        _lib.check(rc, "pmrl_rollout_gather")
        return s, a, r, pv, pa, p

    def sample(self):
        """rollout_buffer.py:59-101 — sequential minibatches over the slots of every env (env-major order)."""
        bs = self.epoch_len if self.batch_size == -1 else self.batch_size
        for env in range(self.E):
            cur = 1
            while cur < self.epoch_len and self.epoch_len - cur >= bs:
                sl = np.arange(cur, cur + bs)
                yield self.gather(sl, np.full(bs, env))
                cur += bs

    def sample_random(self, rng=np.random):
        """rollout_buffer.py:103-142 — a random permutation without replacement of the (slot ≥ 1, env) pairs.
        With E == 1 and the same numpy RNG state it yields exactly the reference's batches."""
        bs = self.epoch_len if self.batch_size == -1 else self.batch_size
        n_per_env = self.epoch_len - 1
        nb = (n_per_env * self.E) // bs if self.E > 1 else n_per_env // bs
        if self.E == 1:
            idxs = rng.choice(np.arange(1, self.epoch_len), (nb, bs), replace=False)       # :123
            envs = np.zeros_like(idxs)
        else:
            flat = rng.choice(n_per_env * self.E, (nb, bs), replace=False)
            idxs, envs = 1 + flat // self.E, flat % self.E
        for b in range(nb):
            yield self.gather(idxs[b], envs[b])


class DeviceReplayBuffer:
    """Off-policy index replay (replay/buffer.py:6-79, replay/traj_buffer.py:6-89).  obs_dtype="bfloat16": the windows
    `gather` / `sample` regenerate (s, s_) are returned as bf16, rounded from the fp32 table and actions.
    obs_relative_to / obs_relative_channels: s and s_ are window-relative like the obs of an env with the same `EnvConfig`
    settings (each window divided by its own last row)."""

    def __init__(self, feat_am, num_features: int, train_len: int, num_envs: int, num_assets: int, window_size: int,
                 buffer_size: int = 425000, batch_size: int = 32, include_last: bool = True, device=None,
                 obs_dtype: str = "float32", obs_relative_to: int | None = None, obs_relative_channels=None):
        if not torch.cuda.is_available():
            raise _lib.PmrlError("DeviceReplayBuffer needs a CUDA device (pmrl_b200 has no CPU fallback)")
        self.lib = _lib.load()
        self.obs_dtype = _obs_dtype(obs_dtype)
        self.obs_relative_to = obs_relative_to
        self.obs_relative_channels = obs_relative_check(obs_relative_to, obs_relative_channels, num_features)
        self._obs_mode = (_OBS_FULL | (_OBS_BF16 if self.obs_dtype is torch.bfloat16 else 0)
                          | obs_relative_bits(obs_relative_to, self.obs_relative_channels))
        self.feat_am = feat_am                                   # [A, T, F-1] device table (the `dataset`, buffer.py:8)
        self.T = feat_am.shape[1]
        self.F, self.E, self.A, self.W = num_features, num_envs, num_assets, window_size
        self.step_offset = 2 * (window_size - 1)                 # buffer.py:11
        self.epoch_len = train_len - self.step_offset            # buffer.py:12
        self.max_epoch = max(1, buffer_size // self.epoch_len)   # buffer.py:13
        self.batch_size, self.include_last = batch_size, include_last
        dev = torch.device(device or feat_am.device)
        self.device = dev
        P, L, E, A = self.max_epoch, self.epoch_len, self.E, self.A
        self.bi = torch.zeros(P, L, E, dtype=torch.int32, device=dev)      # "i" as int32 (the reference stores f32: quirk Q14)
        self.ba = torch.zeros(P, L, E, A, device=dev)
        self.br = torch.zeros(P, L, E, device=dev)
        self.curr_epoch = 0
        self.newest_epoch = 0                                    # buffer.py:38 `self.epoch = max(self.epoch, epoch)`
        self.full = False

    def __len__(self):
        return self.max_epoch if self.full else self.curr_epoch

    def add(self, e: int, i, a, r):
        """buffer.py:23-37 / traj_buffer.py:26-43 batched: `i` is the loader step (int, same for all envs, or an
        int32 tensor [E] of per-env loader indices), a [E, A], r [E]."""
        step_i = int(i) if not torch.is_tensor(i) else None
        lockstep = step_i if step_i is not None else int(i.flatten()[0].item())
        if lockstep < self.W - 1:
            return
        self.curr_epoch = int(e % self.max_epoch)
        self.newest_epoch = max(self.newest_epoch, self.curr_epoch)
        step = lockstep - self.step_offset
        if step < 0 or step >= self.epoch_len:
            # the reference would wrap a negative index into the tail of the epoch row (torch indexing); rows
            # W-1 <= i < 2(W-1) are never sampled as `end-1`, so they are dropped here instead of aliasing.
            return
        idx = i.to(self.device, torch.int32).reshape(self.E).contiguous() if torch.is_tensor(i) else \
            torch.full((self.E,), step_i, dtype=torch.int32, device=self.device)
        a2 = a.reshape(self.E, self.A).to(torch.float32).contiguous()
        r2 = r.reshape(self.E).to(torch.float32).contiguous()
        rc = self.lib.pmrl_replay_add(self.max_epoch, self.epoch_len, self.E, self.A, self.curr_epoch, step,
                                      _lib.ptr(idx), _lib.ptr(a2), _lib.ptr(r2), _lib.ptr(self.bi), _lib.ptr(self.ba),
                                      _lib.ptr(self.br), _lib.current_stream())
        _lib.check(rc, "pmrl_replay_add")
        if not self.full and self.curr_epoch == self.max_epoch - 1:
            self.full = True

    def sinks(self, e: int, step: int):
        """Keyword arguments for `BatchedTradingEnv.step_io` so that the kernel stepping loader item `step` of epoch `e`
        writes the (i, a, r) row itself — `i` is the env's own loader index t0 + k (buffer.py:31-37); {} for the items the
        reference skips.  Marks the epoch like `add` does."""
        if step < self.W - 1:
            return {}
        self.curr_epoch = int(e % self.max_epoch)
        self.newest_epoch = max(self.newest_epoch, self.curr_epoch)
        slot = step - self.step_offset
        if slot < 0 or slot >= self.epoch_len:
            return {}
        if not self.full and self.curr_epoch == self.max_epoch - 1:
            self.full = True
        ep = self.curr_epoch
        return dict(index_sink=self.bi[ep, slot], action_sink=self.ba[ep, slot], reward=self.br[ep, slot])

    def gather(self, epochs, envs, starts):
        """buffer.py:58-77 for explicit (epoch, env, start) triples → (s [B,A,W,F], a [B,A,1], r [B,1,1], s_ [B,A,W,F])."""
        dev = self.device
        ep = torch.as_tensor(epochs).to(dev, torch.int32).contiguous()
        en = torch.as_tensor(envs).to(dev, torch.int32).contiguous()
        st = torch.as_tensor(starts).to(dev, torch.int32).contiguous()
        B = ep.numel()
        A, W, F = self.A, self.W, self.F
        s = torch.empty(B, A, W, F, dtype=self.obs_dtype, device=dev); s2 = torch.empty(B, A, W, F, dtype=self.obs_dtype, device=dev)
        a = torch.empty(B, A, 1, device=dev); r = torch.empty(B, 1, 1, device=dev)
        rc = self.lib.pmrl_replay_gather_obs(self.max_epoch, self.epoch_len, self.E, A, W, F, self.T, B, _lib.ptr(ep),
                                             _lib.ptr(en), _lib.ptr(st), _lib.ptr(self.bi), _lib.ptr(self.ba), _lib.ptr(self.br),
                                             _lib.ptr(self.feat_am), _lib.ptr(s), _lib.ptr(a), _lib.ptr(r), _lib.ptr(s2),
                                             self._obs_mode, _lib.current_stream())
        _lib.check(rc, "pmrl_replay_gather")
        return s, a, r, s2

    def sample(self, generator=None, sampler: str = "traj", percent_latest: float = 0.5):
        """`ReplayBuffer.sample` with the reference's own draw sequence, so that with E == 1 and the same torch RNG state
        it returns exactly the reference's batch:

        sampler="traj"    replay/traj_buffer.py:52-60 (the class train/off_policy.py:10 imports): epochs = [current] +
                          randperm(stored epochs)[:B-1], ONE random start shared by the batch;
        sampler="buffer"  replay/buffer.py:45-49: int(percent_latest·B) copies of the newest epoch + randint epochs, one
                          random start per sample.
        Envs (the batch axis the reference does not have) are drawn last, uniformly, and only when E > 1."""
        B, L, W, g = self.batch_size, self.epoch_len, self.W, generator
        if sampler == "traj":
            n = self.max_epoch if self.full else self.curr_epoch                                  # traj_buffer.py:52
            if not self.include_last:
                raise _lib.PmrlError("INCLUDE_LAST = False removes curr_epoch from the choices (traj_buffer.py:53-54) "
                                     "and then indexes it anyway; only include_last=True is supported")
            rand = torch.randperm(n, generator=g)[:B - 1]                                          # :56
            epochs = torch.cat([torch.tensor([self.curr_epoch]), rand])                            # :57
            if epochs.numel() < B:
                raise IndexError(f"traj sampler: {n} stored epochs cannot fill a batch of {B} (traj_buffer.py:67 would index "
                                 "past `epochs`)")
            starts = torch.randint(0, L - W - 1, (1,), generator=g).repeat(B)                      # :59
        elif sampler == "buffer":
            n_last = int(percent_latest * B)                                                       # buffer.py:14
            last = torch.tensor([self.newest_epoch] * n_last, dtype=torch.long)                    # :45
            rand = torch.randint(0, self.newest_epoch + 1, (B - n_last,), generator=g)             # :46
            epochs = torch.cat((last, rand))
            starts = torch.randint(0, L - W - 1, (B,), generator=g)                                # :48
        else:
            raise ValueError("sampler must be 'traj' or 'buffer'")
        envs = torch.randint(0, self.E, (B,), generator=g) if self.E > 1 else torch.zeros(B, dtype=torch.long)
        return self.gather(epochs, envs, starts)
