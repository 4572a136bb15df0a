"""Environment configuration — the reference's config surface (config/base.py:28-29,47-53) as a dataclass.

The reference binds module-level constants at import (`from config.base import WINDOW_SIZE, NUM_ASSETS`);
`EnvConfig.from_reference_config()` reads the same names from an importable `config.base` so existing
config files keep working.
"""
from __future__ import annotations

from dataclasses import dataclass

REWARD_MODES = {"step_log": 0, "returns": 1, "log_returns": 2, "sharpe_ratio": 3}
OBS_DTYPES = ("float32", "bfloat16")


@dataclass
class EnvConfig:
    num_envs: int = 1                 # E (envs on this rank)
    num_assets: int = 32              # NUM_ASSETS   (config/base.py:29), asset 0 = cash
    window_size: int = 32             # WINDOW_SIZE  (config/base.py:28)
    num_features: int = 5             # F: o,h,l,c + the weight slot that replaces volume (trading_env.py:32)
    initial_cash: float = 25000.0     # INITIAL_CASH (config/base.py:47)
    commission: float = 0.0           # COMISSION [sic] (config/base.py:48)
    reward: str = "step_log"          # what TradingEnv.step returns (:99); or REWARD names (config/base.py:51)
    reward_scale: float = 1.0         # REWARD_SCALE (config/base.py:52)
    risk_free_rate: float = 0.04      # RISK_FREE_RATE (config/base.py:53)
    episode_len: int = 1000           # steps per episode (the reference ends at loader exhaustion)
    mu_max_iter: int = 16             # cap for the commission fixed-point loop (trading_env.py:70)
    strict_reference: bool = True     # reproduce the AND-condition normalisation quirk (trading_env.py:58)
    obs_dtype: str = "float32"        # "bfloat16": the kernels write the obs as bf16 (rounded from the fp32 values; state,
                                      # rewards and everything else stay fp32) — half the obs bytes for a bf16 network

    def __post_init__(self):
        if self.obs_dtype not in OBS_DTYPES:
            raise ValueError(f"unknown obs_dtype {self.obs_dtype!r}; expected one of {OBS_DTYPES}")

    @property
    def reward_mode(self) -> int:
        try:
            return REWARD_MODES[self.reward]
        except KeyError:
            raise ValueError(f"unknown reward {self.reward!r}; expected one of {sorted(REWARD_MODES)}") from None

    @classmethod
    def from_reference_config(cls, **overrides) -> "EnvConfig":
        """Read NUM_ASSETS, WINDOW_SIZE, INITIAL_CASH, COMISSION, REWARD_SCALE, RISK_FREE_RATE from `config.base`."""
        import config.base as cb  # the reference's (or the user's) config package
        kw = dict(num_assets=cb.NUM_ASSETS, window_size=cb.WINDOW_SIZE, initial_cash=float(cb.INITIAL_CASH),
                  commission=float(cb.COMISSION), reward_scale=float(cb.REWARD_SCALE),
                  risk_free_rate=float(cb.RISK_FREE_RATE))
        kw.update(overrides)
        return cls(**kw)
