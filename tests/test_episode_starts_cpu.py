"""Randomised episode starts (pmrl_env_draw_starts): header, ctypes mirror, argument checks that need no GPU, and the CPU
statement of the draw (oracle/starts_oracle.py) against the Random123 known-answer vectors and exact integer arithmetic."""
import ctypes
import math
import os
import re

import numpy as np
import pytest

from oracle import starts_oracle as so
from tests.test_capi_symbols import ROOT, declared_symbols

E_ARG, E_SHAPE = -1, -2


def _load():
    import __graft_entry__ as g
    g.build()
    from pmrl_b200 import _lib
    return _lib, _lib.load()


def _cfg(_lib, E=4, T=64, W=6, L=10):
    return _lib.PmrlEnvCfg(E, 8, W, 5, T, L, 0, 16, 1, 25000.0, 0.0, 1.0, 0.04)


def _dist(_lib, kind=0, lo=0, hi=48, seed=7, env_base=0, beta=0.1):
    L, g = so.geometric_params(lo, max(hi, lo), beta) if kind == so.GEOMETRIC else (0.0, 0.0)
    return _lib.PmrlStartDist(kind, lo, hi, 0, seed, env_base, L, g)


def _draw(lib, cfg, dist, t=16, mask=None, mode=0, t0=16, episode=16):
    return lib.pmrl_env_draw_starts(ctypes.byref(cfg) if cfg is not None else None,
                                    ctypes.byref(dist) if dist is not None else None, t, mask, mode, t0, episode, None)


def test_header_macros_struct_and_ctypes_table():
    syms = declared_symbols()
    assert "pmrl_env_draw_starts" in syms
    hdr = open(os.path.join(ROOT, "include", "pmrl_b200.h")).read()
    from pmrl_b200 import _lib, starts
    for name, value in (("START_UNIFORM", starts.UNIFORM), ("START_GEOMETRIC", starts.GEOMETRIC),
                        ("DRAW_DUE", starts.DRAW_DUE), ("DRAW_MASK", starts.DRAW_MASK)):
        assert int(re.search(rf"#define PMRL_{name}\s+(\d+)", hdr).group(1)) == value
    assert starts.DISTRIBUTIONS == {"uniform": starts.UNIFORM, "geometric": starts.GEOMETRIC}
    assert [f[0] for f in _lib.PmrlStartDist._fields_] == ["kind", "lo", "hi", "pad", "seed", "env_base", "log1m_beta",
                                                           "geo_norm"]
    args = _lib.SIGNATURES["pmrl_env_draw_starts"][1]
    assert len(args) == 8 and args[1] == ctypes.POINTER(_lib.PmrlStartDist) and args[4] == ctypes.c_int32
    _, lib = _load()
    assert lib.pmrl_abi_sizeof(4) == ctypes.sizeof(_lib.PmrlStartDist) == 48
    assert lib.pmrl_abi_sizeof(5) == -1
    assert lib.pmrl_abi_version() == 5


@pytest.mark.parametrize("null", ["cfg", "dist", "t0", "episode", "t_due"])
def test_null_pointers_are_refused(null):
    _lib, lib = _load()
    cfg, dist = _cfg(_lib), _dist(_lib)
    kw = dict(cfg=None if null == "cfg" else cfg, dist=None if null == "dist" else dist)
    if null in ("t0", "episode"):
        kw[null] = None
    if null == "t_due":
        kw["t"] = None
    n = lib.pmrl_launch_count()
    assert _draw(lib, **kw) == E_ARG
    assert lib.pmrl_launch_count() == n


def test_mask_mode_does_not_need_t():
    _lib, lib = _load()
    cfg, dist = _cfg(_lib, E=0), _dist(_lib)
    assert _draw(lib, cfg, dist, t=None, mode=so.DRAW_MASK) == 0


@pytest.mark.parametrize("kind,mode", [(2, 0), (-1, 0), (0, 2), (0, -1), (1, 7)])
def test_unknown_kind_or_mode_is_refused(kind, mode):
    _lib, lib = _load()
    dist = _dist(_lib)
    dist.kind = kind
    assert _draw(lib, _cfg(_lib), dist, mode=mode) == E_ARG


@pytest.mark.parametrize("log1m_beta,geo_norm", [(0.0, 0.5), (0.5, 0.5), (float("nan"), 0.5), (float("-inf"), 1.0),
                                                 (float("inf"), 0.5), (-0.1, 0.0), (-0.1, 1.5), (-0.1, float("nan"))])
def test_geometric_parameters_outside_their_range_are_refused(log1m_beta, geo_norm):
    _lib, lib = _load()
    dist = _dist(_lib, kind=so.GEOMETRIC)
    dist.log1m_beta, dist.geo_norm = log1m_beta, geo_norm
    assert _draw(lib, _cfg(_lib), dist) == E_ARG


@pytest.mark.parametrize("E,lo,hi,env_base,T", [(-1, 0, 48, 0, 64), (4, -1, 48, 0, 64), (4, 10, 9, 0, 64),
                                                (4, 0, 49, 0, 64), (4, 49, 49, 0, 64), (4, 0, 48, -1, 64)])
def test_bad_shapes_are_refused(E, lo, hi, env_base, T):
    _lib, lib = _load()
    n = lib.pmrl_launch_count()
    assert _draw(lib, _cfg(_lib, E=E, T=T), _dist(_lib, lo=lo, hi=hi, env_base=env_base)) == E_SHAPE
    assert lib.pmrl_launch_count() == n


def test_global_env_ids_that_would_overflow_are_refused():
    """gid = env_base + e must stay within int64 for every env of the batch."""
    _lib, lib = _load()
    int64_max = (1 << 63) - 1
    for E, base in ((4, int64_max - 3), (4, int64_max), (1, int64_max)):
        assert _draw(lib, _cfg(_lib, E=E), _dist(_lib, env_base=base)) == E_SHAPE
    assert _draw(lib, _cfg(_lib, E=0), _dist(_lib, env_base=int64_max)) == 0     # validated, then nothing to launch


def test_table_bound_is_the_constructor_bound():
    """hi + episode_len + W == T is the last admissible offset (window rows up to T - 1); without tables nothing bounds hi."""
    _lib, lib = _load()
    assert _draw(lib, _cfg(_lib, E=0, T=64), _dist(_lib, hi=48)) == 0
    assert _draw(lib, _cfg(_lib, E=0, T=0), _dist(_lib, hi=10 ** 6)) == 0


def test_empty_batch_launches_nothing():
    _lib, lib = _load()
    n = lib.pmrl_launch_count()
    assert _draw(lib, _cfg(_lib, E=0), _dist(_lib)) == 0
    assert _draw(lib, _cfg(_lib, E=0), _dist(_lib), mode=so.DRAW_MASK) == 0
    assert lib.pmrl_launch_count() == n


# ------------------------------------------------------------------------------------------------ CPU reference
@pytest.mark.parametrize("ctr,key,out", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_reference_philox_reproduces_the_random123_vectors(ctr, key, out):
    assert so.philox4x32_10(ctr, key) == out


def test_reference_counter_and_key_layout():
    seed, gid, ep = 0x0123456789ABCDEF, (5 << 32) | 17, 3
    x = so.philox4x32_10((ep, 17, 5, 0), (0x89ABCDEF, 0x01234567))
    assert so.r64(seed, gid, ep) == (x[0] << 32) | x[1]


@pytest.mark.parametrize("lo,hi", [(0, 0), (0, 1), (3, 2048 + 2), (0, 3045), (100, 100 + (1 << 20) - 1), (0, (1 << 31) - 2)])
def test_reference_uniform_mapping_is_exact(lo, hi):
    n = hi - lo + 1
    for seed, gid, ep in ((0, 0, 0), (7, 12345, 2), ((1 << 64) - 1, (1 << 40) + 3, 0xffffffff)):
        r = so.r64(seed, gid, ep)
        t0, q = so.draw_one(so.UNIFORM, lo, hi, seed, gid, ep)
        assert q is None and lo <= t0 <= hi
        # floor(r * n / 2^64): the multiply-high, checked through the defining inequality
        k = t0 - lo
        assert k * (1 << 64) <= r * n < (k + 1) * (1 << 64)
        if n & (n - 1) == 0:
            assert k == r >> (64 - (n.bit_length() - 1)) if n > 1 else k == 0


def test_reference_geometric_mapping():
    lo, hi, beta = 10, 109, 0.05
    n = hi - lo + 1
    L, g = so.geometric_params(lo, hi, beta)
    assert L == math.log1p(-beta) and g == -math.expm1(n * L)
    seen = []
    for gid in range(2000):
        t0, q = so.draw_one(so.GEOMETRIC, lo, hi, 99, gid, 0, beta)
        assert lo <= t0 <= hi and q >= 0
        seen.append(hi - t0)
    # recent rows favoured: P(j = 0) = beta / g ≈ 0.05, P(j < 14) ≈ 1 - 0.95^14 ≈ 0.51
    j = np.array(seen)
    assert 0.03 < (j == 0).mean() < 0.07 and 0.45 < (j < 14).mean() < 0.57


def test_reference_draw_touches_only_the_selected_envs():
    t0 = np.arange(8, dtype=np.int32)
    ep = np.array([0, 1, 2, 3, 0xffffffff, 5, 6, 7])
    sel = np.array([1, 0, 1, 0, 1, 0, 0, 0], bool)
    t1, ep1, _ = so.draw(so.UNIFORM, 0, 1000, 1, 100, t0, ep, sel)
    assert np.array_equal(t1[~sel], t0[~sel]) and np.array_equal(ep1[~sel], ep[~sel])
    assert list(ep1[sel]) == [1, 3, 0]                            # u32 wrap
    assert t1[0] == so.draw_one(so.UNIFORM, 0, 1000, 1, 100, 0)[0]
    assert list(so.due([0, 4, 5, 9], 5)) == [False, False, True, True] and not so.due([9], 0).any()


# ------------------------------------------------------------------------------------------------ Python arguments
class _NoDeviceEnv:
    """Stands in for a BatchedTradingEnv: argument checks must fail before any device is touched."""
    T, W, E = 200, 10, 4

    class cfg:
        episode_len = 50


@pytest.mark.parametrize("kw", [dict(low=-1), dict(low=50, high=49), dict(high=141), dict(low=141), dict(low=1.5),
                                dict(distribution="normal"), dict(distribution="geometric"),
                                dict(distribution="geometric", beta=0.0), dict(distribution="geometric", beta=1.0),
                                dict(distribution="geometric", beta=float("nan")), dict(beta=0.5), dict(seed=-1),
                                dict(seed=1 << 64), dict(seed=True), dict(first_env=-3)])
def test_sample_episode_starts_argument_errors(kw):
    from pmrl_b200.env import BatchedTradingEnv
    with pytest.raises(ValueError):
        BatchedTradingEnv.sample_episode_starts(_NoDeviceEnv(), **kw)


def test_sample_episode_starts_needs_tables():
    from pmrl_b200.env import BatchedTradingEnv
    env = _NoDeviceEnv()
    env.T = 0
    with pytest.raises(ValueError, match="tables"):
        BatchedTradingEnv.sample_episode_starts(env)


def test_default_high_is_the_last_offset_whose_episode_fits():
    from pmrl_b200 import starts
    d = starts.start_dist(200, 50, 10)
    assert (d.kind, d.lo, d.hi, d.seed, d.env_base) == (starts.UNIFORM, 0, 140, 0, 0)
    d = starts.start_dist(200, 50, 10, low=5, seed=(1 << 64) - 1, distribution="geometric", beta=0.01, first_env=1 << 33)
    assert (d.kind, d.lo, d.hi, d.seed, d.env_base) == (starts.GEOMETRIC, 5, 140, (1 << 64) - 1, 1 << 33)
    assert (d.log1m_beta, d.geo_norm) == so.geometric_params(5, 140, 0.01)
