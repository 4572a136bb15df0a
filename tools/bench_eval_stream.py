#!/usr/bin/env python
"""Streaming evaluation metrics (BatchedTradingEnv.track_eval_metrics → k_eval_stream_update) on one GPU.

1. step alone vs step + update: two envs built alike (one tracked) run in alternating blocks of 5 warm-up + 20 timed steps
   (CUDA events, median block, ring full), at c4_shard, c3, c2, c5_obs (obs materialised) and c2_state (no obs).
2. the update kernel alone: CUDA events around each update that follows a step (20 steps), against its algorithmic bytes
   per env — two ring rows (8·A), the accumulator read + write (2 × 128), t, idx and V (12).
3. loops.evaluate(traces=True) vs traces=False at c3 with 200 items, alternating, two runs each: wall time (host clock
   around a synchronised call) and torch.cuda.max_memory_allocated above what the env already held; outputs compared.
4. a streaming 1,000-item evaluation at c4_shard and at config 4 whole (1,048,576 envs) on one GPU.

    python tools/bench_eval_stream.py [--out profiles/r03_eval_stream_1gpu.json] [--workloads c4_shard,c2] [--no-whole]
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402  (workload shapes, HBM rate, clock sampler)
import bench_obs_dtype as bod  # noqa: E402  (env construction, action pool, ring fill, block timer, GPU name)

WORKLOADS = ("c4_shard", "c3", "c2", "c5_obs", "c2_state")
ACC_BYTES = 128


def update_bytes_per_env(A):
    return 8.0 * A + 2.0 * ACC_BYTES + 12.0


def free():
    gc.collect(); torch.cuda.empty_cache(); torch.cuda.reset_peak_memory_stats()


def run_step_vs_update(name, peak, clocks):
    E, A, W, F, c, obs, desc = bench.WORKLOADS[name]
    pool = bod.action_pool(E, A)
    plain, tracked = bod.make_env(E, A, W, F, c, "float32"), bod.make_env(E, A, W, F, c, "float32")
    m = tracked.track_eval_metrics()                       # both envs are at local step 0: the tracker starts at once
    for env in (plain, tracked):
        bod.fill_ring(env, pool, W)

    def stepper(env):
        def step(i):
            env.step(pool[i % len(pool)], obs=obs)
        return step

    ms = {"step": [], "step_update": []}
    mark = clocks.mark()
    for b in range(bod.BLOCKS):
        first = b * (bod.WARMUP + bod.STEPS)
        ms["step"].append(bod.time_block(stepper(plain), first))
        ms["step_update"].append(bod.time_block(stepper(tracked), first))
    res = {"workload": name, "desc": desc, "E": E, "A": A, "W": W, "F": F, "commission": c, "obs": obs,
           "clocks": clocks.summary(mark)}
    for v, blocks in ms.items():
        res[v] = {"ms_per_step": statistics.median(blocks), "ms_blocks": blocks}
    res["update_overhead_frac"] = res["step_update"]["ms_per_step"] / res["step"]["ms_per_step"] - 1.0
    # the update kernel alone: events around each update that follows a step of the untracked env
    alone = type(m)(plain)
    plain.reset(obs=obs); alone.update()
    times = []
    for i in range(bod.WARMUP + bod.STEPS):
        plain.step(pool[i % len(pool)], obs=obs)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(); alone.update(); ev1.record()
        times.append((ev0, ev1))
    torch.cuda.synchronize()
    us = sorted(a.elapsed_time(b) * 1e3 for a, b in times[bod.WARMUP:])
    med = statistics.median(us)
    nbytes = E * update_bytes_per_env(A)
    res["update_alone"] = {"us_median": med, "us_min": us[0], "us_max": us[-1], "bytes_per_env": update_bytes_per_env(A),
                           "bytes": nbytes, "achieved_gbs": nbytes / (med * 1e-6) / 1e9,
                           "frac_of_roofline": nbytes / (med * 1e-6) / 1e9 / peak}
    out, _ = alone.running()
    res["update_alone"]["all_envs_valid"] = bool(torch.isfinite(out[:, 3]).all())
    del plain, tracked, m, alone, pool
    free()
    return res


def policy(E, A, W, F):
    # a cheap deterministic policy: the newest close-to-close change of the window as raw scores (signed: softmax branch)
    return lambda s: s[:, :, W - 1, 3] - s[:, :, W - 2, 3]


def same_or_close(t_tot, t_met, s_tot, s_met):
    nan_eq = lambda a, b: bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())
    close = bool(torch.isclose(s_met[:, [0, 1, 3]], t_met[:, [0, 1, 3]], rtol=1e-6, atol=0, equal_nan=True).all())
    return {"return_bit_equal": nan_eq(t_tot, s_tot), "mdd_bit_equal": nan_eq(t_met[:, 2], s_met[:, 2]),
            "sharpe_sortino_turnover_within_1e-6": close}


def run_evaluate_ab(name="c3", items=200, reps=2):
    from pmrl_b200 import loops
    E, A, W, F, c, _, desc = bench.WORKLOADS[name]
    env = bod.make_env(E, A, W, F, c, "float32")
    act = policy(E, A, W, F)
    loops.evaluate(env, act, 3, traces=True); loops.evaluate(env, act, 3, traces=False)     # warm-up
    res = {"workload": name, "desc": desc, "items": items, "traces_True": [], "traces_False": []}
    outs = {}
    for _ in range(reps):
        for traces in (True, False):
            torch.cuda.synchronize(); free()
            held = torch.cuda.memory_allocated()
            t = time.perf_counter()
            tot, met = loops.evaluate(env, act, items, traces=traces)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t
            res[f"traces_{traces}"].append({"wall_s": wall, "peak_extra_gb": (torch.cuda.max_memory_allocated() - held) / 1e9})
            outs[traces] = (tot, met)
    res["env_held_gb"] = held / 1e9
    res["trace_bytes_gb"] = E * items * (A + 1) * 4 / 1e9
    res["check"] = same_or_close(*outs[True], *outs[False])
    del env, outs
    free()
    return res


def run_streaming_eval(E, A, W, F, items, label):
    from pmrl_b200 import loops
    free()
    env = bod.make_env(E, A, W, F, 0.0, "float32")
    act = policy(E, A, W, F)
    torch.cuda.synchronize()
    held = torch.cuda.memory_allocated()
    t = time.perf_counter()
    tot, met = loops.evaluate(env, act, items, traces=False)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t
    res = {"workload": label, "E": E, "A": A, "W": W, "F": F, "items": items, "wall_s": wall,
           "ms_per_item": wall / (items - 1) * 1e3, "env_held_gb": held / 1e9,
           "peak_extra_gb": (torch.cuda.max_memory_allocated() - held) / 1e9,
           "trace_bytes_avoided_gb": E * items * (A + 1) * 4 / 1e9,
           "finite_envs": int(torch.isfinite(met[:, 2]).sum()), "mean_return": float(tot.double().mean())}
    del env, tot, met
    free()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_eval_stream_1gpu.json"))
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--no-whole", action="store_true", help="skip the 1,000-item evaluation of config 4 whole")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval_stream.py measures on a CUDA device; none found")
    torch.cuda.set_device(0)
    peak, peak_src = bench.measured_peak_gbs()
    clocks = bench.ClockSampler(0)
    clocks.start()
    out = {"gpu": bod.gpu_info(), "peak_gbs": peak, "peak_source": peak_src, "warmup": bod.WARMUP, "steps": bod.STEPS,
           "blocks": bod.BLOCKS, "timing": "CUDA events; step / step+update blocks alternate; update alone: events around "
           "each update after a step", "step_vs_update": []}
    for name in [w for w in args.workloads.split(",") if w]:
        r = run_step_vs_update(name, peak, clocks)
        out["step_vs_update"].append(r)
        print(json.dumps({"workload": name, "step_ms": round(r["step"]["ms_per_step"], 4),
                          "step_update_ms": round(r["step_update"]["ms_per_step"], 4),
                          "overhead": round(r["update_overhead_frac"], 4), "update_us": round(r["update_alone"]["us_median"], 2),
                          "update_frac_of_roofline": round(r["update_alone"]["frac_of_roofline"], 3)}), flush=True)
    out["evaluate_ab"] = run_evaluate_ab()
    print(json.dumps({"evaluate_ab": out["evaluate_ab"]}), flush=True)
    out["streaming_1000"] = [run_streaming_eval(131072, 100, 50, 5, 1000, "c4_shard")]
    if not args.no_whole:
        out["streaming_1000"].append(run_streaming_eval(1048576, 100, 50, 5, 1000, "c4_whole"))
    for r in out["streaming_1000"]:
        print(json.dumps(r), flush=True)
    out["clocks_all"] = clocks.stop()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    ok = all(out["evaluate_ab"]["check"].values()) and all(r["update_alone"]["all_envs_valid"] for r in out["step_vs_update"])
    print("wrote", args.out, "checks ok" if ok else "CHECK FAILED")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
