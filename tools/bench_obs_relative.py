#!/usr/bin/env python
"""Window-relative observations (EnvConfig.obs_relative_to, PMRL_OBS_REL) on one GPU, device-timed with CUDA events.

For each workload four variants run in ONE process on the same tables, offsets and action sequence, in alternating blocks
(plain fp32; REL in the kernels; plain fp32 followed by the caller-side torch pass `o[..., :F-1] /= o[:, :, -1:, ref:ref+1]`
with the divisor column cloned first — what a caller does without the flag; bf16 REL), each block 5 warm-up + 20 timed
steps with the ring full.  The divisor is the close (channel 3) and every feature channel is divided.

Reported per variant: ms/step (median over blocks, every block listed), asset-steps/s, algorithmic bytes per asset-step
(plain and REL 8 + 25/A + 4·W·F + 4·W, bf16 REL 8 + 25/A + 2·W·F + 4·W, the torch pass adds a read and a write of the
4·W·(F-1) feature bytes), and the share of the HBM rate bench.py uses, with the GPU name, power limit and SM clock samples
taken in the same run.  After the last block the REL obs is compared bit for bit with the torch pass on a seeded sample of
envs, and the bf16 REL obs with its rounding.

    python tools/bench_obs_relative.py [--out profiles/r03_obs_relative_1gpu.json] [--workloads c4_shard,c2]
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
VARIANTS = ("plain", "rel", "plain_torch", "rel_bf16")
WARMUP, STEPS, BLOCKS, CHECK_ENVS = 5, 20, 3, 512
REF = 3


def bytes_per_asset_step(A, W, F, variant):
    base = 8.0 + 25.0 / A + 4.0 * W
    if variant == "rel_bf16":
        return base + 2.0 * W * F
    if variant == "plain_torch":
        return base + 4.0 * W * F + 8.0 * W * (F - 1)
    return base + 4.0 * W * F


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def make_env(E, A, W, F, commission, variant):
    import pmrl_b200
    from pmrl_b200 import synth
    from pmrl_b200.env import BatchedTradingEnv
    kw = {}
    if variant in ("rel", "rel_bf16"):
        kw["obs_relative_to"] = REF
    if variant == "rel_bf16":
        kw["obs_dtype"] = "bfloat16"
    cfg = pmrl_b200.EnvConfig(num_envs=E, num_assets=A, window_size=W, num_features=F, commission=commission,
                              episode_len=bench.EPISODE_LEN, **kw)
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


def bits_equal(a, b):
    it = torch.int32 if a.dtype is torch.float32 else torch.int16
    return bool(torch.equal(a.view(it), b.view(it)))


def run_workload(name, peak, clocks):
    E, A, W, F, c, _, desc = bench.WORKLOADS[name]
    pool = action_pool(E, A)
    envs = {v: make_env(E, A, W, F, c, v) for v in VARIANTS}
    for env in envs.values():
        for i in range(W):                                    # state-only steps: every ring is full before timing
            env.step(pool[i % len(pool)], obs=False)
    last = {}

    def stepper(v):
        env = envs[v]

        def step(i):
            o, _, _ = env.step(pool[i % len(pool)])
            if v == "plain_torch":
                o[..., :F - 1] /= o[:, :, -1:, REF:REF + 1].clone()
            last[v] = o
        return step

    ms = {v: [] for v in VARIANTS}
    mark = clocks.mark()
    for b in range(BLOCKS):
        first = b * (WARMUP + STEPS)
        for v in VARIANTS:
            ms[v].append(time_block(stepper(v), first))
    idx = torch.randperm(E, generator=torch.Generator().manual_seed(0))[:CHECK_ENVS].cuda()
    check = {"envs_checked": int(idx.numel()),
             "rel_bits_equal_torch_pass": bits_equal(last["rel"][idx], last["plain_torch"][idx]),
             "rel_bf16_bits_equal_rounding": bits_equal(last["rel_bf16"][idx], last["rel"][idx].to(torch.bfloat16)),
             "state_equal": all(bool(torch.equal(envs["plain"].hist[idx], envs[v].hist[idx])) and
                                bool(torch.equal(envs["plain"].value[idx], envs[v].value[idx])) for v in VARIANTS)}
    res = {"workload": name, "desc": desc, "E": E, "A": A, "W": W, "F": F, "commission": c, "ref_channel": REF,
           "clocks": clocks.summary(mark), "check": check}
    for v, blocks in ms.items():
        res[v] = entry(blocks, E, A, W, F, v, peak)
    res["rel_over_plain"] = res["rel"]["ms_per_step"] / res["plain"]["ms_per_step"]
    res["speedup_rel_over_plain_torch"] = res["plain_torch"]["ms_per_step"] / res["rel"]["ms_per_step"]
    del envs, pool, last
    gc.collect(); torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_obs_relative_1gpu.json"))
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_obs_relative.py measures on a CUDA device; none found")
    torch.cuda.set_device(0)
    peak, peak_src = bench.measured_peak_gbs()
    clocks = bench.ClockSampler(0)
    clocks.start()
    out = {"gpu": gpu_info(), "peak_gbs": peak, "peak_source": peak_src, "warmup": WARMUP, "steps": STEPS, "blocks": BLOCKS,
           "timing": "CUDA events around the timed steps of each block; plain / rel / plain + torch pass / bf16 rel blocks "
                     "alternate", "results": []}
    for name in [w for w in args.workloads.split(",") if w]:
        r = run_workload(name, peak, clocks)
        out["results"].append(r)
        print(json.dumps({k: r[k] for k in ("workload", "rel_over_plain", "speedup_rel_over_plain_torch")}
                         | {v: round(r[v]["ms_per_step"], 4) for v in VARIANTS}), flush=True)
    out["clocks_all"] = clocks.stop()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    ok = all(all(v for k, v in r["check"].items() if k != "envs_checked") for r in out["results"])
    print("wrote", args.out, "checks ok" if ok else "CHECK FAILED")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
