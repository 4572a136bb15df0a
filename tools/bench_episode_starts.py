#!/usr/bin/env python
"""Randomised episode starts (BatchedTradingEnv.sample_episode_starts → k_env_draw_starts) on one GPU.

1. step alone vs draw + step: two envs built alike (one with a uniform sampler) run in alternating blocks of 5 warm-up +
   20 timed steps (CUDA events, median block, ring full), at c4_shard, c3, c5_obs, c2 (obs materialised) and c2_state
   (no obs).  Episodes are bench.py's 1,000 steps, so in the timed steps the due draw reads every env's t and draws for
   none: the cost every step pays.
2. c2 through graphed_step(steps=15): the draws are captured in the same graph; ms per step = replay time / 15.
3. the draw kernel alone, CUDA events around each launch (20 launches, median): the due draw after a step (reads 4 B of t
   per env), and a draw for every env (mask = NULL: reads the counter, writes t0 and the counter, 12 B per env).

    python tools/bench_episode_starts.py [--out profiles/r03_episode_starts_1gpu.json] [--workloads c4_shard,c2]
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402  (workload shapes, HBM rate, clock sampler)
import bench_obs_dtype as bod  # noqa: E402  (env construction, action pool, ring fill, block timer, GPU name)

WORKLOADS = ("c4_shard", "c3", "c5_obs", "c2", "c2_state")
GRAPH_STEPS = 15


def free():
    gc.collect(); torch.cuda.empty_cache()


def time_launches(fn, n=bod.WARMUP + bod.STEPS, before=None):
    """Median / min / max microseconds of fn() between CUDA events (the first WARMUP launches dropped)."""
    times = []
    for i in range(n):
        if before is not None:
            before(i)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(); fn(); ev1.record()
        times.append((ev0, ev1))
    torch.cuda.synchronize()
    us = sorted(a.elapsed_time(b) * 1e3 for a, b in times[bod.WARMUP:])
    return {"us_median": statistics.median(us), "us_min": us[0], "us_max": us[-1]}


def run_step_vs_draw(name, peak, clocks):
    E, A, W, F, c, obs, desc = bench.WORKLOADS[name]
    pool = bod.action_pool(E, A)
    plain, sampled = bod.make_env(E, A, W, F, c, "float32"), bod.make_env(E, A, W, F, c, "float32")
    s = sampled.sample_episode_starts(seed=1)
    sampled.reset()                                            # first draw: every env gets a random start
    for env in (plain, sampled):
        bod.fill_ring(env, pool, W)

    def stepper(env):
        def step(i):
            env.step(pool[i % len(pool)], obs=obs)
        return step

    ms = {"step": [], "draw_step": []}
    mark = clocks.mark()
    for b in range(bod.BLOCKS):
        first = b * (bod.WARMUP + bod.STEPS)
        ms["step"].append(bod.time_block(stepper(plain), first))
        ms["draw_step"].append(bod.time_block(stepper(sampled), first))
    res = {"workload": name, "desc": desc, "E": E, "A": A, "W": W, "F": F, "commission": c, "obs": obs,
           "episode_len": bench.EPISODE_LEN, "clocks": clocks.summary(mark)}
    for v, blocks in ms.items():
        res[v] = {"ms_per_step": statistics.median(blocks), "ms_blocks": blocks}
    res["draw_overhead_frac"] = res["draw_step"]["ms_per_step"] / res["step"]["ms_per_step"] - 1.0
    # the draw alone: the due draw that precedes a step (no env is due), and a draw for every env
    res["due_draw_alone"] = time_launches(s.draw_due, before=lambda i: plain.step(pool[i % len(pool)], obs=obs))
    res["due_draw_alone"]["bytes"] = 4 * E
    res["all_draw_alone"] = time_launches(lambda: s.draw_mask(None))
    res["all_draw_alone"]["bytes"] = 12 * E
    for k in ("due_draw_alone", "all_draw_alone"):
        r = res[k]
        r["achieved_gbs"] = r["bytes"] / (r["us_median"] * 1e-6) / 1e9
        r["frac_of_roofline"] = r["achieved_gbs"] / peak
    t0 = sampled.t0
    res["t0_check"] = {"in_range": bool(((t0 >= s.low) & (t0 <= s.high)).all()), "distinct": int(torch.unique(t0).numel()),
                       "range": [s.low, s.high]}
    del plain, sampled, s, pool
    free()
    return res


def run_graphed(name, clocks, K=GRAPH_STEPS):
    E, A, W, F, c, obs, desc = bench.WORKLOADS[name]
    pool = bod.action_pool(E, A)
    plain, sampled = bod.make_env(E, A, W, F, c, "float32"), bod.make_env(E, A, W, F, c, "float32")
    sampled.sample_episode_starts(seed=1)
    sampled.reset()
    burst = torch.stack([pool[i % len(pool)] for i in range(K)])
    replays = {}
    for key, env in (("graph", plain), ("draw_graph", sampled)):
        bod.fill_ring(env, pool, W)
        static, replay = env.graphed_step(obs=obs, steps=K)
        static.copy_(burst)
        replays[key] = replay
    ms = {k: [] for k in replays}
    mark = clocks.mark()
    for _ in range(bod.BLOCKS):
        for key, replay in replays.items():
            ms[key].append(bod.time_block(lambda i: replay(), 0) / K)
    res = {"workload": name, "desc": desc, "steps_per_graph": K, "clocks": clocks.summary(mark)}
    for k, blocks in ms.items():
        res[k] = {"ms_per_step": statistics.median(blocks), "ms_blocks": blocks}
    res["draw_overhead_frac"] = res["draw_graph"]["ms_per_step"] / res["graph"]["ms_per_step"] - 1.0
    del plain, sampled, replays, pool
    free()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_episode_starts_1gpu.json"))
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_episode_starts.py measures on a CUDA device; none found")
    torch.cuda.set_device(0)
    peak, peak_src = bench.measured_peak_gbs()
    clocks = bench.ClockSampler(0)
    clocks.start()
    out = {"gpu": bod.gpu_info(), "peak_gbs": peak, "peak_source": peak_src, "warmup": bod.WARMUP, "steps": bod.STEPS,
           "blocks": bod.BLOCKS, "timing": "CUDA events; step / draw+step blocks alternate; draw alone: events around each "
           "launch", "step_vs_draw": []}
    for name in [w for w in args.workloads.split(",") if w]:
        r = run_step_vs_draw(name, peak, clocks)
        out["step_vs_draw"].append(r)
        print(json.dumps({"workload": name, "step_ms": round(r["step"]["ms_per_step"], 4),
                          "draw_step_ms": round(r["draw_step"]["ms_per_step"], 4),
                          "overhead": round(r["draw_overhead_frac"], 4),
                          "due_draw_us": round(r["due_draw_alone"]["us_median"], 2),
                          "all_draw_us": round(r["all_draw_alone"]["us_median"], 2)}), flush=True)
    out["graphed"] = run_graphed("c2", clocks)
    g = out["graphed"]
    print(json.dumps({"graphed_c2_ms": round(g["graph"]["ms_per_step"], 5),
                      "graphed_c2_draw_ms": round(g["draw_graph"]["ms_per_step"], 5),
                      "overhead": round(g["draw_overhead_frac"], 4)}), flush=True)
    out["clocks_all"] = clocks.stop()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    ok = all(r["t0_check"]["in_range"] for r in out["step_vs_draw"])
    print("wrote", args.out, "checks ok" if ok else "CHECK FAILED")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
