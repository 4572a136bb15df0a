"""ctypes binding of libpmrl_b200.so — the only way the Python host reaches the CUDA kernels.

There is no CPU fallback: if the library cannot be loaded, or a call is made without a CUDA device,
the error is raised to the caller.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpmrl_b200.so")

c_float_p = C.c_void_p     # device pointers travel as integers
c_void_p = C.c_void_p
i32 = C.c_int32
f32 = C.c_float


class PmrlEnvCfg(C.Structure):
    _fields_ = [("E", i32), ("A", i32), ("W", i32), ("F", i32), ("T", i32),
                ("episode_len", i32), ("reward_mode", i32), ("mu_max_iter", i32), ("flags", C.c_uint32),
                ("initial_cash", f32), ("commission", f32), ("reward_scale", f32), ("risk_free", f32)]


class PmrlTables(C.Structure):
    _fields_ = [("y_tm", c_void_p), ("feat_am", c_void_p), ("feat_am4", c_void_p)]


class PmrlEnvState(C.Structure):
    _fields_ = [("value", c_void_p), ("hist", c_void_p), ("idx", c_void_p), ("is_full", c_void_p),
                ("t", c_void_p), ("t0", c_void_p), ("sharpe", c_void_p), ("ep_return", c_void_p), ("ticket", c_void_p)]


class PmrlStepIO(C.Structure):
    _fields_ = [("actions", c_void_p), ("y_ext", c_void_p), ("reward", c_void_p), ("done", c_void_p), ("obs", c_void_p),
                ("obs_mode", i32), ("stats", c_void_p), ("action_sink", c_void_p), ("value_sink", c_void_p),
                ("weight_sink", c_void_p), ("index_sink", c_void_p), ("reward_host", c_void_p), ("done_host", c_void_p),
                ("actions_ready", c_void_p), ("actions_ready_seq", C.c_uint32), ("actions_ready_shift", i32)]


class PmrlStartDist(C.Structure):
    _fields_ = [("kind", i32), ("lo", i32), ("hi", i32), ("pad", i32), ("seed", C.c_uint64), ("env_base", C.c_int64),
                ("log1m_beta", C.c_double), ("geo_norm", C.c_double)]


P = C.POINTER
# symbol → (restype, argtypes); must list every function declared in include/pmrl_b200.h
SIGNATURES = {
    "pmrl_abi_version": (C.c_int, []),
    "pmrl_abi_sizeof": (C.c_int, [i32]),
    "pmrl_launch_count": (C.c_uint64, []),
    "pmrl_last_error": (C.c_char_p, []),
    "pmrl_set_tuning": (C.c_int, [i32, i32]),
    "pmrl_env_reset": (C.c_int, [P(PmrlEnvCfg), P(PmrlTables), P(PmrlEnvState), c_void_p, c_void_p, i32, c_void_p]),
    "pmrl_env_step": (C.c_int, [P(PmrlEnvCfg), P(PmrlTables), P(PmrlEnvState), c_void_p, c_void_p,
                                c_void_p, c_void_p, c_void_p, i32, c_void_p, c_void_p]),
    "pmrl_env_step_io": (C.c_int, [P(PmrlEnvCfg), P(PmrlTables), P(PmrlEnvState), P(PmrlStepIO), c_void_p]),
    "pmrl_env_step_burst": (C.c_int, [P(PmrlEnvCfg), P(PmrlTables), P(PmrlEnvState), c_void_p, i32, c_void_p, c_void_p,
                                      c_void_p, c_void_p]),
    "pmrl_env_step_host": (C.c_int, [P(PmrlEnvCfg), P(PmrlTables), P(PmrlEnvState), c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, i32, c_void_p, i32, c_void_p]),
    "pmrl_price_relatives": (C.c_int, [c_void_p, i32, i32, c_void_p, c_void_p]),
    "pmrl_selftest_division": (C.c_int, [c_void_p, c_void_p, C.c_int64, c_void_p, c_void_p]),
    "pmrl_obs_build": (C.c_int, [P(PmrlEnvCfg), P(PmrlTables), P(PmrlEnvState), c_void_p, i32, c_void_p]),
    "pmrl_ffd_weights": (C.c_int, [c_void_p, i32, i32, f32, c_void_p, c_void_p, c_void_p]),
    "pmrl_ffd_transform": (C.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, i32, i32, i32, c_void_p, c_void_p]),
    "pmrl_scale_series": (C.c_int, [c_void_p, i32, i32, i32, c_void_p, c_void_p]),
    "pmrl_pack_features": (C.c_int, [c_void_p, c_void_p, i32, i32, i32, c_void_p, c_void_p, c_void_p]),
    "pmrl_indicator_layout": (C.c_int, [c_void_p, i32, c_void_p, c_void_p]),
    "pmrl_indicators": (C.c_int, [c_void_p, i32, i32, i32, c_void_p, i32, c_void_p, c_void_p]),
    "pmrl_rollout_add": (C.c_int, [i32, i32, i32, i32, i32, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pmrl_rollout_gather": (C.c_int, [i32, i32, i32, i32, i32, i32, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pmrl_rollout_gather_index": (C.c_int, [i32, i32, i32, i32, i32, i32, i32, c_void_p, c_void_p,
                                            c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                            c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pmrl_replay_add": (C.c_int, [i32, i32, i32, i32, i32, i32, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_void_p, c_void_p]),
    "pmrl_replay_gather": (C.c_int, [i32, i32, i32, i32, i32, i32, i32, i32, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pmrl_rollout_gather_bf16": (C.c_int, [i32, i32, i32, i32, i32, i32, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pmrl_rollout_gather_index_bf16": (C.c_int, [i32, i32, i32, i32, i32, i32, i32, c_void_p, c_void_p,
                                                 c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                 c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pmrl_replay_gather_bf16": (C.c_int, [i32, i32, i32, i32, i32, i32, i32, i32, c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pmrl_rollout_gather_index_obs": (C.c_int, [i32, i32, i32, i32, i32, i32, i32, c_void_p, c_void_p,
                                                c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, i32, c_void_p]),
    "pmrl_replay_gather_obs": (C.c_int, [i32, i32, i32, i32, i32, i32, i32, i32, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_void_p, c_void_p, i32, c_void_p]),
    "pmrl_pg_reward_fwd_bwd": (C.c_int, [i32, i32, i32, i32, f32, f32, i32, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p, f32, c_void_p]),
    "pmrl_eval_metrics": (C.c_int, [c_void_p, c_void_p, i32, i32, i32, f32, i32, c_void_p, c_void_p]),
    "pmrl_eval_stream_update": (C.c_int, [P(PmrlEnvCfg), P(PmrlEnvState), c_void_p, f32, i32, c_void_p]),
    "pmrl_eval_stream_read": (C.c_int, [P(PmrlEnvCfg), P(PmrlEnvState), c_void_p, i32, f32, i32, c_void_p, c_void_p,
                                        c_void_p]),
    "pmrl_env_draw_starts": (C.c_int, [P(PmrlEnvCfg), P(PmrlStartDist), c_void_p, c_void_p, i32, c_void_p, c_void_p,
                                       c_void_p]),
}

EVAL_ACC_BYTES = 128       # include/pmrl_b200.h PMRL_EVAL_ACC_BYTES: one streaming-metrics accumulator per env

_lib = None


class PmrlError(RuntimeError):
    pass


def load(build_if_missing: bool = False) -> C.CDLL:
    """dlopen libpmrl_b200.so (in-tree).  Raises if it is missing — there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if build_if_missing:
            from . import build as _b
            _b.build()
        else:
            raise PmrlError(f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(nvcc, sm_100a). pmrl_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here means header and library diverged
        fn.restype = res
        fn.argtypes = args
    if lib.pmrl_abi_version() != 5:
        raise PmrlError("libpmrl_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().pmrl_last_error().decode(errors="replace")
        raise PmrlError(f"{what} failed (rc={rc}): {msg}")


def ptr(t) -> int | None:
    """Device pointer of a CUDA tensor (or None)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise PmrlError("pmrl_b200 kernels need CUDA tensors (no CPU fallback)")
    if not t.is_contiguous():
        raise PmrlError("pmrl_b200 kernels need contiguous tensors")
    return t.data_ptr()


def current_stream() -> int:
    """Raw handle of torch's current CUDA stream (the stream every entry point enqueues on)."""
    import torch
    raw = getattr(torch._C, "_cuda_getCurrentRawStream", None)
    if raw is not None:                       # ~0.2 us instead of ~2 us for the Stream object round trip
        return raw(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


TUNE_GROUP_ENVS, TUNE_CTAS_PER_SM, TUNE_FUSED, TUNE_FAST_FILL, TUNE_RING_TMA, TUNE_STAGED, TUNE_HOST_STREAM, TUNE_HOST_MIRROR = 2, 3, 4, 5, 11, 12, 13, 14


def set_tuning(key: int, value: int) -> None:
    """Launch-shape tuning hook of the fused step kernel (include/pmrl_b200.h PMRL_TUNE_*); value <= 0 → heuristic."""
    check(load().pmrl_set_tuning(key, value), "pmrl_set_tuning")
