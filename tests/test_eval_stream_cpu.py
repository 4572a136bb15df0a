"""Streaming evaluation metrics (pmrl_eval_stream_*): header, ctypes table and argument checks that need no GPU — every
invalid argument is refused before any launch."""
import ctypes
import os
import re

import pytest

from tests.test_capi_symbols import ROOT, declared_symbols

E_ARG, E_SHAPE, E_ALIGN = -1, -2, -3


def _load():
    import __graft_entry__ as g
    g.build()
    from pmrl_b200 import _lib
    return _lib, _lib.load()


def _cfg_state(_lib, E=4, A=8, W=6, **null):
    cfg = _lib.PmrlEnvCfg(E, A, W, 5, 64, 10, 0, 16, 1, 25000.0, 0.0, 1.0, 0.04)
    f = {k: 16 for k in ("value", "hist", "idx", "is_full", "t", "t0", "ep_return")}
    f.update({k: None for k in null})
    st = _lib.PmrlEnvState(f["value"], f["hist"], f["idx"], f["is_full"], f["t"], f["t0"], None, f["ep_return"], None)
    return cfg, st


def _update(lib, cfg, st, acc=16, periods=252):
    return lib.pmrl_eval_stream_update(ctypes.byref(cfg), ctypes.byref(st), acc, 0.0, periods, None)


def _read(lib, cfg, st, acc=16, which=0, periods=252, out=16):
    return lib.pmrl_eval_stream_read(ctypes.byref(cfg), ctypes.byref(st), acc, which, 0.0, periods, out, None, None)


def test_header_declares_the_streaming_entry_points_and_the_ctypes_table_matches():
    syms = declared_symbols()
    assert "pmrl_eval_stream_update" in syms and "pmrl_eval_stream_read" in syms
    from pmrl_b200 import _lib
    assert _lib.SIGNATURES["pmrl_eval_stream_update"][1][2:] == [ctypes.c_void_p, ctypes.c_float, ctypes.c_int32, ctypes.c_void_p]
    assert len(_lib.SIGNATURES["pmrl_eval_stream_read"][1]) == 9
    hdr = open(os.path.join(ROOT, "include", "pmrl_b200.h")).read()
    acc_bytes = int(re.search(r"#define PMRL_EVAL_ACC_BYTES\s+(\d+)", hdr).group(1))
    assert acc_bytes == _lib.EVAL_ACC_BYTES <= 128
    from pmrl_b200 import metrics
    for name, mode in (("RUNNING", metrics.RUNNING), ("LAST_EPISODE", metrics.LAST_EPISODE), ("EPISODE_MEAN", metrics.EPISODE_MEAN)):
        assert int(re.search(rf"#define PMRL_EVAL_{name}\s+(\d+)", hdr).group(1)) == mode
    _, lib = _load()
    assert hasattr(lib, "pmrl_eval_stream_update") and hasattr(lib, "pmrl_eval_stream_read")


@pytest.mark.parametrize("null", ["value", "hist", "idx", "t", "ep_return"])
def test_null_state_pointers_are_refused(null):
    _lib, lib = _load()
    cfg, st = _cfg_state(_lib, **{null: True})
    assert _update(lib, cfg, st) == E_ARG
    assert _read(lib, cfg, st) == E_ARG


def test_null_acc_out_and_structs_are_refused():
    _lib, lib = _load()
    cfg, st = _cfg_state(_lib)
    assert _update(lib, cfg, st, acc=None) == E_ARG
    assert _read(lib, cfg, st, acc=None) == E_ARG
    assert _read(lib, cfg, st, out=None) == E_ARG
    assert lib.pmrl_eval_stream_update(None, ctypes.byref(st), 16, 0.0, 252, None) == E_ARG
    assert lib.pmrl_eval_stream_read(ctypes.byref(cfg), None, 16, 0, 0.0, 252, 16, None, None) == E_ARG


@pytest.mark.parametrize("which", [-1, 3, 100])
def test_unknown_read_mode_is_refused(which):
    _lib, lib = _load()
    cfg, st = _cfg_state(_lib)
    assert _read(lib, cfg, st, which=which) == E_ARG
    assert b"bad which" in lib.pmrl_last_error()


@pytest.mark.parametrize("shape,periods", [((-1, 8, 6), 252), ((4, 0, 6), 252), ((4, 1025, 6), 252), ((4, 8, 1), 252),
                                           ((4, 8, 6), 0), ((4, 8, 6), -5)])
def test_bad_shapes_are_refused(shape, periods):
    _lib, lib = _load()
    E, A, W = shape
    cfg, st = _cfg_state(_lib, E=E, A=A, W=W)
    assert _update(lib, cfg, st, periods=periods) == E_SHAPE
    assert _read(lib, cfg, st, periods=periods) == E_SHAPE


def test_misaligned_accumulator_is_refused():
    _lib, lib = _load()
    cfg, st = _cfg_state(_lib)
    assert _update(lib, cfg, st, acc=24) == E_ALIGN
    assert _read(lib, cfg, st, acc=24) == E_ALIGN


def test_empty_batch_launches_nothing():
    _lib, lib = _load()
    cfg, st = _cfg_state(_lib, E=0)
    n = lib.pmrl_launch_count()
    assert _update(lib, cfg, st) == 0 and _read(lib, cfg, st) == 0
    assert lib.pmrl_launch_count() == n


class _NoDeviceEnv:
    """Stands in for a BatchedTradingEnv: argument checks must fail before any attribute or device is touched."""
    class cfg:
        episode_len = 10


@pytest.mark.parametrize("kw", [dict(periods=0), dict(periods=-3), dict(periods=2.5), dict(periods=True),
                                dict(rf=float("nan")), dict(rf=float("inf"))])
def test_track_eval_metrics_argument_errors(kw):
    from pmrl_b200.env import BatchedTradingEnv
    with pytest.raises(ValueError):
        BatchedTradingEnv.track_eval_metrics(_NoDeviceEnv(), **kw)


@pytest.mark.parametrize("num_items", [0, 1, 12, 1000])
def test_evaluate_without_traces_refuses_what_is_not_one_episode(num_items):
    from pmrl_b200 import loops
    with pytest.raises(ValueError):
        loops.evaluate(_NoDeviceEnv(), lambda s: s, num_items, traces=False)


def test_evaluate_without_traces_checks_its_tracker_arguments():
    from pmrl_b200 import loops
    with pytest.raises(ValueError):
        loops.evaluate(_NoDeviceEnv(), lambda s: s, 5, periods=0, traces=False)
