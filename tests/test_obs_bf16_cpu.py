"""bf16 observations (PMRL_OBS_BF16): argument checks that need no GPU — bad obs modes are refused before any launch."""
import ctypes

import pytest

FULL, WEIGHTS, NONE, BF16 = 1, 2, 0, 0x100
BAD_MODES = (WEIGHTS | BF16, NONE | BF16, FULL | 0x200, FULL | BF16 | 0x1000, 3, -1)


def _load():
    import __graft_entry__ as g
    g.build()
    from pmrl_b200 import _lib
    return _lib, _lib.load()


def _cfg_state(_lib):
    # a shape every obs path accepts; the state pointers are never dereferenced because validation fails first
    cfg = _lib.PmrlEnvCfg(4, 8, 6, 5, 64, 10, 0, 16, 1, 25000.0, 0.0, 1.0, 0.04)
    st = _lib.PmrlEnvState(16, 16, 16, 16, 16, 16, None, None, None)
    tbl = _lib.PmrlTables(16, 16, None)
    return cfg, tbl, st


@pytest.mark.parametrize("mode", BAD_MODES)
def test_bad_obs_modes_are_rejected_before_launch(mode):
    _lib, lib = _load()
    cfg, tbl, st = _cfg_state(_lib)
    B = ctypes.byref
    rc = lib.pmrl_env_step(B(cfg), B(tbl), B(st), 16, None, 16, 16, 16, mode, None, None)
    assert rc == -1 and b"bad obs_mode" in lib.pmrl_last_error()
    io = _lib.PmrlStepIO()
    io.actions, io.reward, io.done, io.obs, io.obs_mode = 16, 16, 16, 16, mode
    assert lib.pmrl_env_step_io(B(cfg), B(tbl), B(st), B(io), None) == -1
    assert lib.pmrl_env_reset(B(cfg), B(tbl), B(st), None, 16, mode, None) == -1
    assert lib.pmrl_env_step_host(B(cfg), B(tbl), B(st), 16, 16, 16, 16, 16, 16, 16, mode, None, 0, None) == -1
    if (mode & 0xff) != NONE:                   # (obs_build refuses NONE on its own)
        assert lib.pmrl_obs_build(B(cfg), B(tbl), B(st), 16, mode, None) == -1
    assert b"bad obs_mode" in lib.pmrl_last_error()


def test_bf16_flag_names_its_partner_mode():
    _lib, lib = _load()
    cfg, tbl, st = _cfg_state(_lib)
    B = ctypes.byref
    assert lib.pmrl_env_reset(B(cfg), B(tbl), B(st), None, 16, WEIGHTS | BF16, None) == -1
    assert b"PMRL_OBS_BF16 needs PMRL_OBS_FULL" in lib.pmrl_last_error()


def test_bf16_gathers_validate_like_the_fp32_ones():
    _lib, lib = _load()
    assert lib.pmrl_rollout_gather_bf16(0, 1, 1, 1, 1, 1, *([None] * 14)) == -2
    assert lib.pmrl_rollout_gather_bf16(1, 1, 1, 1, 1, 1, *([None] * 14)) == -1
    assert lib.pmrl_rollout_gather_index_bf16(2, 1, 1, 2, 2, 8, 1, *([None] * 16)) == -1
    assert lib.pmrl_replay_gather_bf16(1, 1, 1, 1, 2, 2, 8, 1, *([None] * 12)) == -1
    assert lib.pmrl_replay_gather_bf16(1, 1, 1, 1, 2, 2, 2, 1, *([None] * 12)) == -2


def test_env_config_obs_dtype():
    from pmrl_b200 import EnvConfig
    assert EnvConfig().obs_dtype == "float32"
    assert EnvConfig(obs_dtype="bfloat16").obs_dtype == "bfloat16"
    for bad in ("float16", "bf16", "fp8"):
        with pytest.raises(ValueError, match="obs_dtype"):
            EnvConfig(obs_dtype=bad)
