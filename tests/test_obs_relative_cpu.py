"""Window-relative observations (PMRL_OBS_REL, EnvConfig.obs_relative_to): the parts that need no GPU — the header bits and
their Python mirror, obs modes and gather arguments refused before any launch, EnvConfig validation, and the CPU
restatement in oracle/obs_relative_oracle.py against the formula."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FULL, WEIGHTS, NONE, BF16, REL = 1, 2, 0, 0x100, 0x200


def rel_of(ref, mask):
    return REL | (ref << 10) | (mask << 14)


def _load():
    import __graft_entry__ as g
    g.build()
    from pmrl_b200 import _lib
    return _lib, _lib.load()


def _header_defines():
    src = open(os.path.join(ROOT, "include", "pmrl_b200.h")).read()
    return dict(re.findall(r"#define\s+(PMRL_OBS_\w+)\s+(0x[0-9a-fA-F]+|\d+)", src)), src


def test_header_bits_and_python_mirror_agree():
    from pmrl_b200 import config
    d, src = _header_defines()
    assert int(d["PMRL_OBS_REL"], 0) == REL == config.OBS_REL
    assert int(d["PMRL_OBS_REL_REF_SHIFT"]) == 10 == config.OBS_REL_REF_SHIFT
    assert int(d["PMRL_OBS_REL_MASK_SHIFT"]) == 14 == config.OBS_REL_MASK_SHIFT
    assert int(d["PMRL_OBS_BF16"], 0) == BF16 and REL & (BF16 | 0xFF) == 0
    assert "#define PMRL_OBS_REL_OF(ref, mask)" in src
    assert config.obs_relative_bits(3, (0, 1, 2, 3)) == rel_of(3, 0xF)
    assert config.obs_relative_bits(None, None) == 0
    widest = config.obs_relative_bits(15, tuple(range(16)))            # every bit the encoding has
    assert widest == rel_of(15, 0xFFFF) and 0 < widest | FULL | BF16 < 2 ** 31


def _cfg_state(_lib, F=5, W=6):
    # a shape every obs path accepts; the state pointers are never dereferenced because validation fails first
    cfg = _lib.PmrlEnvCfg(4, 8, W, F, 64, 10, 0, 16, 1, 25000.0, 0.0, 1.0, 0.04)
    st = _lib.PmrlEnvState(16, 16, 16, 16, 16, 16, None, None, None)
    tbl = _lib.PmrlTables(16, 16, None)
    return cfg, tbl, st


def _env_entry_points(lib, _lib, cfg, tbl, st, mode):
    B = ctypes.byref
    io = _lib.PmrlStepIO()
    io.actions, io.reward, io.done, io.obs, io.obs_mode = 16, 16, 16, 16, mode
    return {
        "step": lib.pmrl_env_step(B(cfg), B(tbl), B(st), 16, None, 16, 16, 16, mode, None, None),
        "step_io": lib.pmrl_env_step_io(B(cfg), B(tbl), B(st), B(io), None),
        "reset": lib.pmrl_env_reset(B(cfg), B(tbl), B(st), None, 16, mode, None),
        "step_host": lib.pmrl_env_step_host(B(cfg), B(tbl), B(st), 16, 16, 16, 16, 16, 16, 16, mode, None, 0, None),
        "obs_build": lib.pmrl_obs_build(B(cfg), B(tbl), B(st), 16, mode, None),
    }


# (obs_mode, expected code, text in pmrl_last_error) at F = 5: feature channels 0..3
BAD_F5 = [
    (NONE | rel_of(0, 1), -1, b"bad obs_mode"),
    (WEIGHTS | rel_of(0, 1), -1, b"bad obs_mode"),
    (FULL | REL, -1, b"empty channel mask"),
    (FULL | BF16 | REL | (2 << 10), -1, b"empty channel mask"),
    (FULL | rel_of(0, 0x10), -1, b"outside the feature channels"),        # mask bit 4 = F-1 (the weight channel)
    (FULL | rel_of(0, 0x8000), -1, b"outside the feature channels"),
    (FULL | rel_of(4, 1), -1, b"outside the feature channels"),           # ref = F-1
    (FULL | rel_of(15, 1), -1, b"outside the feature channels"),
    (FULL | rel_of(0, 1) | (1 << 30), -1, b"bad obs_mode"),               # unknown bit
    (FULL | rel_of(0, 1) | (1 << 31) - (1 << 32), -1, b"bad obs_mode"),   # negative
    (FULL | (3 << 10), -1, b"bad obs_mode"),                              # ref bits without PMRL_OBS_REL
    (FULL | (1 << 14), -1, b"bad obs_mode"),                              # mask bits without PMRL_OBS_REL
]


@pytest.mark.parametrize("mode,code,msg", BAD_F5)
def test_bad_relative_modes_are_refused_before_any_launch(mode, code, msg):
    _lib, lib = _load()
    cfg, tbl, st = _cfg_state(_lib)
    before = lib.pmrl_launch_count()
    for name, rc in _env_entry_points(lib, _lib, cfg, tbl, st, mode).items():
        if name == "obs_build" and mode & 0xFF == NONE:
            assert rc == -1                                              # (obs_build refuses NONE on its own)
            continue
        assert rc == code, name
        assert msg in lib.pmrl_last_error(), (name, lib.pmrl_last_error())
    assert lib.pmrl_launch_count() == before


def test_more_than_16_feature_channels_is_a_shape_error():
    _lib, lib = _load()
    cfg, tbl, st = _cfg_state(_lib, F=18, W=4)
    before = lib.pmrl_launch_count()
    for name, rc in _env_entry_points(lib, _lib, cfg, tbl, st, FULL | rel_of(3, 0xF)).items():
        assert rc == -2, name
        assert b"at most 16 feature channels" in lib.pmrl_last_error()
    assert lib.pmrl_launch_count() == before


def _rollout_index_obs(lib, mode, F=5, S=2, W=2, T=8):
    return lib.pmrl_rollout_gather_index_obs(S, 1, 1, W, F, T, 1, *([16] * 15), mode, None)


def _replay_obs(lib, mode, F=5, W=2, T=8):
    return lib.pmrl_replay_gather_obs(1, 1, 1, 1, W, F, T, 1, *([16] * 11), mode, None)


@pytest.mark.parametrize("gather", [_rollout_index_obs, _replay_obs])
def test_gather_obs_modes(gather):
    _lib, lib = _load()
    before = lib.pmrl_launch_count()
    for mode, code in [(NONE, -1), (WEIGHTS, -1), (NONE | BF16, -1), (WEIGHTS | rel_of(0, 1), -1), (FULL | REL, -1),
                       (FULL | rel_of(4, 1), -1), (FULL | rel_of(0, 0x10), -1), (FULL | rel_of(0, 1) | (1 << 30), -1), (-1, -1)]:
        assert gather(lib, mode) == code, hex(mode)
        assert b"bad obs_mode" in lib.pmrl_last_error()
    assert gather(lib, FULL | rel_of(0, 1), F=18) == -2
    # valid modes get as far as the size checks of the existing gathers
    for mode in (FULL, FULL | BF16, FULL | rel_of(3, 0xF), FULL | BF16 | rel_of(0, 0x5)):
        assert gather(lib, mode, T=1) == -2 and b"bad sizes" in lib.pmrl_last_error()
    assert lib.pmrl_launch_count() == before


def test_env_config_validation():
    from pmrl_b200 import EnvConfig
    assert EnvConfig().obs_relative_to is None and EnvConfig().obs_relative_channels is None
    assert EnvConfig().obs_relative_bits == 0
    c = EnvConfig(num_features=5, obs_relative_to=3)
    assert c.obs_relative_channels == (0, 1, 2, 3) and c.obs_relative_bits == rel_of(3, 0xF)
    c = EnvConfig(num_features=9, obs_relative_to=3, obs_relative_channels=[6, 0, 3, 3])
    assert c.obs_relative_channels == (0, 3, 6) and c.obs_relative_bits == rel_of(3, 0b1001001)
    assert EnvConfig(num_features=17, obs_relative_to=15).obs_relative_channels == tuple(range(16))
    bad = [dict(num_features=5, obs_relative_to=4), dict(num_features=5, obs_relative_to=-1),
           dict(num_features=5, obs_relative_to=1.0), dict(num_features=5, obs_relative_to=True),
           dict(num_features=5, obs_relative_to=0, obs_relative_channels=()),
           dict(num_features=5, obs_relative_to=0, obs_relative_channels=(4,)),
           dict(num_features=5, obs_relative_to=0, obs_relative_channels=(-1,)),
           dict(num_features=5, obs_relative_channels=(0,)),                  # channels without a divisor
           dict(num_features=18, obs_relative_to=0),                          # F - 1 > 16
           dict(num_features=1, obs_relative_to=0)]
    for kw in bad:
        with pytest.raises(ValueError):
            EnvConfig(**kw)


def _specials():
    return np.array([0x00000000, 0x80000000, 0x00000001, 0x807FFFFF, 0x00800000, 0x1F800000, 0x5F800000,   # ±0, subnormals,
                     0x7F800000, 0xFF800000, 0x7FC00000, 0x3F800000, 0xBF800000, 0x42C80000, 0xC2C80000,   # 2^-64, 2^64, ±inf,
                     0x7F7FFFFF, 0x1E800000, 0x60800000], dtype=np.uint32).view(np.float32)          # NaN, ±1, ±100, max


def test_oracle_restates_the_formula():
    """Against the formula with an independent rounding (fp64 quotient rounded once to fp32 — exact for a quotient of two
    fp32 values), on normal values and on every IEEE edge as numerator and as divisor."""
    from oracle.obs_relative_oracle import relative_obs
    rs = np.random.RandomState(0)
    E, A, W, F = 3, 7, 6, 6
    obs = (rs.lognormal(4.0, 0.5, size=(E, A, W, F))).astype(np.float32)
    sp = _specials()
    obs.reshape(-1)[rs.choice(obs.size, 120, replace=False)] = rs.choice(sp, 120)
    obs[0, 0, -1, 2] = 0.0; obs[0, 1, -1, 2] = -3.0; obs[0, 2, -1, 2] = sp[2]; obs[0, 3, -1, 2] = np.inf
    obs[0, 4, -1, 2] = np.nan; obs[0, 5, -1, 2] = sp[5]; obs[0, 6, -1, 2] = sp[6]; obs[1, 0, :, :] = 1.0
    ref, chans = 2, (0, 2, 3)
    got = relative_obs(obs, ref, chans)
    with np.errstate(all="ignore"):
        want = obs.copy()
        div = obs[..., -1:, ref].astype(np.float64)
        for c in chans:
            want[..., c] = (obs[..., c].astype(np.float64) / div).astype(np.float32)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    assert np.array_equal(got.view(np.uint32)[~nan], want.view(np.uint32)[~nan])
    assert np.array_equal(got[..., [1, 4, 5]], obs[..., [1, 4, 5]], equal_nan=True)                # unmasked and weight channel kept
    assert np.all(got[1, 0] == 1.0)                                                   # a cash row of ones stays ones
    assert np.all(np.isnan(got[0, 4, :, [0, 2, 3]]))                                  # NaN divisor → NaN row
    with pytest.raises(ValueError):
        relative_obs(obs, 5, (0,))
    with pytest.raises(ValueError):
        relative_obs(obs, 0, (5,))
