"""CPU oracle for the episode-start draw (pmrl_env_draw_starts) — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A Python-int / numpy restatement of the formulas in include/pmrl_b200.h: Philox4x32-10 (Random123), the uniform map
lo + umul64hi(r64, n) in exact integers, and the truncated-geometric map in fp64 (the host's log1p, which may differ from
the device's in the last bit: a quotient within ~1e-9 of an integer may then floor one apart).
"""
from __future__ import annotations

import math

import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK32 = 0xFFFFFFFF
UNIFORM, GEOMETRIC = 0, 1
DRAW_DUE, DRAW_MASK = 0, 1


def philox4x32_10(ctr, key):
    """Random123 Philox4x32 with 10 rounds: ctr (4 x u32), key (2 x u32) → 4 x u32."""
    c0, c1, c2, c3 = (int(x) & MASK32 for x in ctr)
    k0, k1 = (int(x) & MASK32 for x in key)
    for r in range(10):
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & MASK32, p1 & MASK32, ((p0 >> 32) ^ c3 ^ k1) & MASK32, p0 & MASK32
        k0, k1 = (k0 + W0) & MASK32, (k1 + W1) & MASK32
    return c0, c1, c2, c3


def r64(seed: int, gid: int, episode: int) -> int:
    x = philox4x32_10((episode, gid & MASK32, gid >> 32, 0), (seed & MASK32, seed >> 32))
    return (x[0] << 32) | x[1]


def geometric_params(lo: int, hi: int, beta: float):
    """(log1m_beta, geo_norm) as the binding computes them."""
    L = math.log1p(-beta)
    return L, -math.expm1((hi - lo + 1) * L)


def draw_one(kind, lo, hi, seed, gid, episode, beta=None):
    """(t0, geometric quotient or None) of one draw."""
    r = r64(seed, gid, episode)
    n = hi - lo + 1
    if kind == UNIFORM:
        return lo + ((r * n) >> 64), None
    L, g = geometric_params(lo, hi, beta)
    u = (r >> 11) * 2.0 ** -53
    q = math.log1p(-u * g) / L
    return hi - min(n - 1, math.floor(q)), q


def draw(kind, lo, hi, seed, env_base, t0, episodes, select, beta=None):
    """Apply one draw to the selected envs: returns (t0', episodes', quotients) — quotients[e] is the geometric quotient of
    a drawn env (NaN otherwise), for the near-integer tolerance."""
    t0 = np.array(t0, np.int64).copy()
    ep = np.array(episodes, np.int64).copy()
    q = np.full(len(t0), np.nan)
    for e in np.flatnonzero(np.asarray(select, bool)):
        t0[e], qe = draw_one(kind, lo, hi, seed, env_base + int(e), int(ep[e]) & MASK32, beta)
        if qe is not None:
            q[e] = qe
        ep[e] = (ep[e] + 1) & MASK32
    return t0.astype(np.int32), ep, q


def due(t, episode_len):
    """The envs the next step auto-resets (the step kernels' test)."""
    t = np.asarray(t)
    return (t >= episode_len) if episode_len > 0 else np.zeros(t.shape, bool)
