#!/usr/bin/env python
"""fp32 vs bf16 observations (EnvConfig.obs_dtype) on one GPU, device-timed with CUDA events.

For each workload three variants run in ONE process on the same tables, offsets and action sequence, in alternating
blocks (fp32, bf16, fp32 + `.to(torch.bfloat16)` — what a caller feeding a bf16 network does without the flag), each block
5 warm-up + 20 timed steps with the ring full.  Config 4 whole (1,048,576 envs) does not fit three times: there the two
dtypes run one after the other, one block each, freeing the first before the second is built.

Reported per variant: ms/step (median over blocks, every block listed), asset-steps/s, algorithmic bytes per asset-step
(fp32 obs 8 + 25/A + 4·W·F + 4·W, bf16 obs 8 + 25/A + 2·W·F + 4·W, the cast adds a 4·W·F read and a 2·W·F write), the
share of the HBM rate bench.py uses, with the GPU name, power limit and SM clock samples taken in the same run.  After
the last block the bf16 obs is compared bit for bit with the fp32 obs `.to(torch.bfloat16)` on a seeded sample of envs.

    python tools/bench_obs_dtype.py [--out profiles/r03_obs_bf16_1gpu.json] [--workloads c4_shard,c2] [--no-whole]
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402  (workload shapes, table size, HBM rate, clock sampler)

WORKLOADS = ("c4_shard", "c4_f9", "c2", "c5_obs")
WARMUP, STEPS, BLOCKS, CHECK_ENVS = 5, 20, 3, 512


def bytes_per_asset_step(A, W, F, variant):
    base = 8.0 + 25.0 / A + 4.0 * W
    if variant == "bf16":
        return base + 2.0 * W * F
    if variant == "fp32_cast":
        return base + 4.0 * W * F + 6.0 * W * F
    return base + 4.0 * W * F


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def make_env(E, A, W, F, commission, obs_dtype):
    import pmrl_b200
    from pmrl_b200 import synth
    from pmrl_b200.env import BatchedTradingEnv
    cfg = pmrl_b200.EnvConfig(num_envs=E, num_assets=A, window_size=W, num_features=F, commission=commission,
                              episode_len=bench.EPISODE_LEN, obs_dtype=obs_dtype)
    tbl = synth.gbm_ohlc(bench.TABLE_ROWS, A)
    feats = None
    if F != 5:                                                # as bench.make_env: OHLC + synthetic indicator channels
        g = torch.Generator().manual_seed(99)
        feats = torch.cat([tbl, torch.rand(bench.TABLE_ROWS, A, F - 5, generator=g)], dim=-1)
    t0 = synth.episode_offsets(E, bench.TABLE_ROWS, W, bench.EPISODE_LEN)
    env = BatchedTradingEnv(cfg, prices=tbl, features=feats, t0=t0)
    env.reset()
    return env


def action_pool(E, A, n=4):
    gen = torch.Generator(device="cuda").manual_seed(4321)
    return [torch.randn(E, A, generator=gen, device="cuda") for _ in range(n)]


def fill_ring(env, pool, W):
    for i in range(W):                                        # state-only steps: every ring is full before timing
        env.step(pool[i % len(pool)], obs=False)


def time_block(step, first):
    """WARMUP untimed + STEPS timed calls of step(i); ms per step from CUDA events around the timed calls."""
    for i in range(WARMUP):
        step(first + i)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(STEPS):
        step(first + WARMUP + i)
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / STEPS


def entry(ms_blocks, E, A, W, F, variant, peak):
    ms = statistics.median(ms_blocks)
    rate = E * A / (ms * 1e-3)
    bpa = bytes_per_asset_step(A, W, F, variant)
    gbs = rate * bpa / 1e9
    return {"ms_per_step": ms, "ms_blocks": ms_blocks, "asset_steps_per_s": rate, "bytes_per_asset_step": bpa,
            "achieved_gbs": gbs, "frac_of_peak": gbs / peak}


def check_sample(e32, e16, o32, o16, seed=0):
    g = torch.Generator().manual_seed(seed)
    idx = torch.randperm(e32.E, generator=g)[:CHECK_ENVS].cuda()
    want = o32[idx].to(torch.bfloat16).view(torch.int16)
    got = o16[idx].view(torch.int16)
    ok = bool(torch.equal(got, want)) and bool(torch.equal(e32.value[idx], e16.value[idx])) \
        and bool(torch.equal(e32.hist[idx], e16.hist[idx]))
    return {"envs_checked": int(idx.numel()), "bf16_bits_equal_and_state_equal": ok}


def run_workload(name, peak, clocks):
    E, A, W, F, c, _, desc = bench.WORKLOADS[name]
    pool = action_pool(E, A)
    e32, e16, e32c = make_env(E, A, W, F, c, "float32"), make_env(E, A, W, F, c, "bfloat16"), make_env(E, A, W, F, c, "float32")
    for env in (e32, e16, e32c):
        fill_ring(env, pool, W)
    last = {}

    def stepper(env, key, cast=False):
        def step(i):
            o, _, _ = env.step(pool[i % len(pool)])
            last[key] = o.to(torch.bfloat16) if cast else o
        return step

    ms = {"fp32": [], "bf16": [], "fp32_cast": []}
    mark = clocks.mark()
    for b in range(BLOCKS):
        first = b * (WARMUP + STEPS)
        ms["fp32"].append(time_block(stepper(e32, "fp32"), first))
        ms["bf16"].append(time_block(stepper(e16, "bf16"), first))
        ms["fp32_cast"].append(time_block(stepper(e32c, "fp32_cast", cast=True), first))
    res = {"workload": name, "desc": desc, "E": E, "A": A, "W": W, "F": F, "commission": c,
           "clocks": clocks.summary(mark), "check": check_sample(e32, e16, last["fp32"], last["bf16"])}
    res["check"]["cast_equals_bf16"] = bool(torch.equal(last["fp32_cast"].view(torch.int16), last["bf16"].view(torch.int16)))
    for v, blocks in ms.items():
        res[v] = entry(blocks, E, A, W, F, v, peak)
    res["speedup_bf16_over_fp32"] = res["fp32"]["ms_per_step"] / res["bf16"]["ms_per_step"]
    res["speedup_bf16_over_fp32_cast"] = res["fp32_cast"]["ms_per_step"] / res["bf16"]["ms_per_step"]
    res["bf16_roofline_ms"] = E * A * bytes_per_asset_step(A, W, F, "bf16") / (peak * 1e9) * 1e3
    res["bf16_frac_of_roofline"] = res["bf16_roofline_ms"] / res["bf16"]["ms_per_step"]
    del e32, e16, e32c, pool, last
    gc.collect(); torch.cuda.empty_cache()
    return res


def run_whole(peak, clocks):
    """Config 4 whole on one GPU: 1,048,576 envs x 100 x 50 (105 GB of fp32 obs), the dtypes one after the other."""
    E, A, W, F, c = 1048576, 100, 50, 5, 0.0
    res = {"workload": "c4_whole", "E": E, "A": A, "W": W, "F": F, "commission": c}
    obs_sample = {}
    for v, dt in (("fp32", "float32"), ("bf16", "bfloat16")):
        pool = action_pool(E, A, n=2)
        env = make_env(E, A, W, F, c, dt)
        fill_ring(env, pool, W)
        box = {}

        def step(i):
            box["o"] = env.step(pool[i % 2])[0]
        mark = clocks.mark()
        ms = time_block(step, 0)
        res[v] = entry([ms], E, A, W, F, v, peak)
        res[v]["clocks"] = clocks.summary(mark)
        res[v]["obs_gb"] = box["o"].numel() * box["o"].element_size() / 1e9
        res[v]["max_memory_allocated_gb"] = torch.cuda.max_memory_allocated() / 1e9
        g = torch.Generator().manual_seed(0)
        idx = torch.randperm(E, generator=g)[:CHECK_ENVS].cuda()
        obs_sample[v] = box["o"][idx].clone()
        del env, pool, box
        gc.collect(); torch.cuda.empty_cache(); torch.cuda.reset_peak_memory_stats()
    res["check"] = {"envs_checked": CHECK_ENVS, "bf16_bits_equal": bool(torch.equal(
        obs_sample["bf16"].view(torch.int16), obs_sample["fp32"].to(torch.bfloat16).view(torch.int16)))}
    res["speedup_bf16_over_fp32"] = res["fp32"]["ms_per_step"] / res["bf16"]["ms_per_step"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_obs_bf16_1gpu.json"))
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--no-whole", action="store_true", help="skip config 4 whole (1,048,576 envs)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_obs_dtype.py measures on a CUDA device; none found")
    torch.cuda.set_device(0)
    peak, peak_src = bench.measured_peak_gbs()
    clocks = bench.ClockSampler(0)
    clocks.start()
    out = {"gpu": gpu_info(), "peak_gbs": peak, "peak_source": peak_src, "warmup": WARMUP, "steps": STEPS, "blocks": BLOCKS,
           "timing": "CUDA events around the timed steps of each block; fp32 / bf16 / fp32+cast blocks alternate",
           "results": []}
    for name in [w for w in args.workloads.split(",") if w]:
        r = run_workload(name, peak, clocks)
        out["results"].append(r)
        print(json.dumps({k: r[k] for k in ("workload", "speedup_bf16_over_fp32", "bf16_frac_of_roofline")}
                         | {v: round(r[v]["ms_per_step"], 4) for v in ("fp32", "bf16", "fp32_cast")}), flush=True)
    if not args.no_whole:
        r = run_whole(peak, clocks)
        out["results"].append(r)
        print(json.dumps({"workload": "c4_whole", "fp32": r["fp32"]["ms_per_step"], "bf16": r["bf16"]["ms_per_step"]}), flush=True)
    out["clocks_all"] = clocks.stop()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    ok = all(r["check"].get("bf16_bits_equal_and_state_equal", r["check"].get("bf16_bits_equal")) for r in out["results"])
    print("wrote", args.out, "checks ok" if ok else "CHECK FAILED")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
