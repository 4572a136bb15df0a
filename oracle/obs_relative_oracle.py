"""CPU restatement of the window-relative observation (include/pmrl_b200.h PMRL_OBS_REL): the masked feature channels of each
asset's window divided by channel `ref` of the window's last row, in IEEE fp32 (numpy's float32 division is correctly rounded,
keeps subnormals and follows IEEE for zero, infinite and NaN operands); the other feature channels and the weight channel F-1
are left as they are."""
from __future__ import annotations

import numpy as np


def relative_obs(obs, ref: int, channels) -> np.ndarray:
    """obs [..., W, F] float32 (feature channels 0..F-2, weight channel F-1) → the window-relative obs, float32."""
    x = np.asarray(obs, dtype=np.float32)
    F = x.shape[-1]
    chans = sorted(set(int(c) for c in channels))
    if not 0 <= ref < F - 1 or not chans or chans[0] < 0 or chans[-1] >= F - 1:
        raise ValueError("ref and channels must be feature channels 0 .. F-2")
    out = x.copy()
    div = x[..., -1:, ref]                                   # [..., 1]: row W-1 of every window
    with np.errstate(divide="ignore", invalid="ignore", over="ignore", under="ignore"):
        for c in chans:
            out[..., c] = x[..., c] / div
    return out
