#!/usr/bin/env python
"""bench.py — throughput of the portfolio-env hot path on B200 (driver contract in DESIGN.md §Measurement).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's CPU step on the host cores (live tree if present, else its port)

A "step" is one lockstep transition of every env on the rank: fused step kernel + observation
materialisation (Mode O).  Default workload = the per-GPU shard of BASELINE config 4
(1,048,576 envs x 100 assets x window 50 over 8 GPUs → 131,072 envs per GPU, weak scaling).
Prints ONE JSON line on rank 0.  With the default workload the line also carries `configs`: every other
BASELINE.json config (1: PG-in-the-loop on the CPU; 2, 3, 5 and config 4 whole; the burst / graph / collect-loop
variants), each timed on its own — after and outside the headline's timed region — with its own roofline entry.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (envs, assets, window, features, commission, obs materialised, description)
    # `envs` is per GPU for a headline run (`--workload X`: weak scaling, except c4) and the BASELINE total that is
    # divided over the ranks when the workload is timed as an entry of `configs`
    "c4_shard": (131072, 100, 50, 5, 0.0, True, "BASELINE config 4 shard: 131,072 envs/GPU x 100 assets x window 50, obs materialised"),
    "c4": (1048576, 100, 50, 5, 0.0, True, "BASELINE config 4 whole: 1,048,576 envs x 100 assets x window 50 divided over the ranks (strong scaling), obs materialised"),
    "c2": (4096, 50, 50, 5, 0.0, True, "BASELINE config 2: 4,096 envs x 50 assets, window 50, obs materialised"),
    "c2_state": (4096, 50, 50, 5, 0.0, False, "BASELINE config 2, state-only step (no obs)"),
    "c3": (65536, 100, 50, 5, 0.0, True, "BASELINE config 3: 65,536 envs x 100 assets, obs materialised"),
    "c5": (262144, 500, 50, 5, 0.0025, False, "BASELINE config 5: 262,144 envs x 500 assets, commission 0.0025, state-only"),
    "c5_obs": (32768, 500, 50, 5, 0.0025, True, "wide universe with obs: 32,768 envs x 500 assets x window 50, commission 0.0025, obs materialised"),
    "c4_state": (131072, 100, 50, 5, 0.0, False, "config 4 shard, state-only step (no obs)"),
    "c4_f9": (131072, 100, 50, 9, 0.0, True, "config 4 shard with the indicator set appended: F = 9 (OHLC + ema + bbands + weight channel)"),
    "c4_f13": (65536, 100, 50, 13, 0.0, True, "wider indicator set: F = 13 (OHLC + 8 indicator outputs + weight channel), 65,536 envs/GPU"),
    "c4_f17": (65536, 100, 50, 17, 0.0, True, "wider indicator set: F = 17 (OHLC + 12 indicator outputs + weight channel), 65,536 envs/GPU"),
    "c4_f6": (65536, 100, 50, 6, 0.0, True, "F = 6 (OHLC + ema + weight channel), 65,536 envs/GPU"),
    "c4_f8": (65536, 100, 50, 8, 0.0, True, "F = 8 (OHLC + bbands + weight channel), 65,536 envs/GPU"),
    "c4_f7": (65536, 100, 50, 7, 0.0, True, "F = 7 ((F - 1) % 4 != 0, e.g. OHLC + two indicator outputs): fused kernel on the channel-padded table, 65,536 envs/GPU"),
}
EPISODE_LEN = 1000
TABLE_ROWS = 4096
L2_BYTES = 126e6
DUMP_BYTES = 60 << 20                                         # --dump-outputs: under 64 MB with the .npy headers


def algorithmic_bytes_per_asset_step(A, W, F, commission, obs, sinks=0.0):
    """SURVEY.md §8(d): Mode S = 4 (action) + 4 (w' ring write) + 4·[c>0] (w_last) + 25/A;
    Mode O adds 4·W·F (obs write) + 4·W (ring read for the weight channel, subsumes w_last).
    `sinks`: extra bytes per asset-step the kernel writes into buffer rows (collect loops)."""
    b = 4.0 + 4.0 + 25.0 / A + sinks
    if obs:
        return b + 4.0 * W * F + 4.0 * W
    return b + (4.0 if commission > 0 else 0.0)


def ncu_traffic_bytes(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu --set full
    capture of this workload (profiles/traffic.json), or None if no capture exists for it."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            return json.load(fh).get(workload, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


def dump_outputs(out_dir, arrays, E, limit=DUMP_BYTES):
    """Writes `arrays` (name -> (tensor, env axis)) as out_dir/<name>.npy, float32 (int64 as float64, exact).  While
    they fit in `limit` bytes they go out whole; otherwise every array is cut to the same fixed, seeded sample of envs,
    in ascending order, and env_index.npy lists them."""
    import numpy as np
    import torch
    per_env = sum(4 * t.numel() // E for t, _ in arrays.values())
    if per_env * E > limit:
        idx = torch.randperm(E, generator=torch.Generator().manual_seed(0))[:limit // (per_env + 8)].sort().values
        arrays = {k: (t.index_select(ax, idx.to(t.device)), ax) for k, (t, ax) in arrays.items()}
        arrays["env_index"] = (idx, 0)
    os.makedirs(out_dir, exist_ok=True)
    for name, (t, _) in arrays.items():
        a = t.cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64 if a.dtype == np.int64 else np.float32))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self):
        return len(self.rows)

    def summary(self, since=0):
        rows = self.rows[since:]
        sm = [float(r[0]) for r in rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        return self.summary()


# ------------------------------------------------------------------------------------------------------------------
# CPU side: the reference's own step on the host cores
# ------------------------------------------------------------------------------------------------------------------
def reference_kind():
    """BASELINE.md §3 step 2: the live reference if its tree is on this box, else the op-for-op port."""
    from oracle import live_reference as live
    root = live.locate()
    return ("reference", root) if root else ("port", None)


def cpu_baseline(A, W, commission=0.0, seconds=12.0, context=True):
    """The reference's CPU step on every host core: `seconds` of single-env stepping per process, one single-thread
    process per core (BASELINE.md §3), raw N(0,1) actions (softmax branch) like the GPU arm."""
    from oracle.ref_port import time_all_cores, time_env
    kind, root = reference_kind()
    impl = "live" if kind == "reference" else "port"
    procs = len(os.sched_getaffinity(0))
    rate1 = time_env(impl, A, W, 500, 50, 5, 0, commission)         # calibrate (≈0.1 s)
    steps = max(500, int(rate1 * seconds))
    total, rates = time_all_cores(impl, A, W, steps, procs, commission)
    out = {"value": total * A, "unit": "asset-steps/s", "cores": procs, "kind": kind,
           "env_steps_per_s": total,
           "sample": f"{procs} single-thread processes x {steps} steps of one env ({A} assets, window {W}, commission {commission}), "
                     + (f"the live reference env/sim/trading_env.py at {root}" if kind == "reference" else
                        "oracle/ref_port.py (op-for-op torch-CPU port of env/sim/trading_env.py:44-105; no reference tree on this box)")}
    if context:
        # context only: the batched numpy restatement (oracle/env_oracle.py, one thread, state-only, no obs) — what a
        # vectorised CPU rewrite of the reference would reach per core — and the plain-C restatement with OpenMP
        import numpy as np
        from oracle.env_oracle import OracleEnv
        Eb = 4096
        env = OracleEnv(Eb, A, W, 5)
        rs = np.random.RandomState(0)
        acts = rs.standard_normal((4, Eb, A)).astype(np.float32)
        ys = (1 + 0.01 * rs.standard_normal((4, Eb, A))).astype(np.float32)
        env.step(acts[0], ys[0])
        t0 = time.perf_counter()
        nb = 12
        for i in range(nb):
            env.step(acts[i % 4], ys[i % 4])
        out["batched_numpy_1core_asset_steps_per_s"] = nb * Eb * A / (time.perf_counter() - t0)
        try:
            from oracle.c_oracle import time_all_cores as c_all
            out["c_port_openmp_all_cores_asset_steps_per_s"] = c_all(A, W)
        except Exception:
            out["c_port_openmp_all_cores_asset_steps_per_s"] = None
    return out


def config1_cpu(seconds=6.0):
    """BASELINE config 1: PG agent on the reference env/sim, 1 env, 11 assets, window 50, on the CPU — the loop of
    train/on_policy.py:59-67 (agent.act → env.step), one single-thread process per core.  Needs the live tree for the
    policy (agent/pg/pg.py:29-38, net/lsre_cann.py:94-123); without it only the env half can be timed (the port)."""
    from oracle.ref_port import time_all_cores, time_env
    kind, root = reference_kind()
    impl = "live" if kind == "reference" else "port"
    procs = len(os.sched_getaffinity(0))
    A, W = 11, 50
    out = {"description": "BASELINE config 1: PG agent on the reference env, 1 env x 11 assets x window 50, CPU",
           "cores": procs, "kind": kind, "assets": A, "window": W}
    r1 = time_env(impl, A, W, 500, 50, 5, 0)
    tot, _ = time_all_cores(impl, A, W, max(500, int(r1 * seconds / 2)), procs)
    out["env_only"] = {"env_steps_per_s_all_cores": tot, "env_steps_per_s_per_core": tot / procs, "asset_steps_per_s": tot * A}
    if kind == "reference":
        rp = time_env("live", A, W, 60, 10, 5, 0, 0.0, True)
        totp, _ = time_all_cores("live", A, W, max(60, int(rp * seconds / 2)), procs, 0.0, True)
        out["pg_in_loop"] = {"env_steps_per_s_all_cores": totp, "env_steps_per_s_per_core": totp / procs, "asset_steps_per_s": totp * A,
                             "policy": "agent.pg.pg.PG(5).act — LSRE-CANN, eval mode, torch CPU, 1 thread per process"}
    else:
        out["pg_in_loop"] = {"unavailable": "the PG policy is reference code (agent/pg/pg.py, net/lsre_cann.py); no reference tree "
                                            "at $PMRL_REFERENCE_ROOT, /root/reference or baseline/_ref on this box"}
    return out


def shared_config(args, world):
    """The `config` object both arms print (same keys, same values) for one workload."""
    E, A, W, F, commission, obs, desc = WORKLOADS[args.workload]
    if args.envs:
        E = args.envs
    strong = args.workload == "c4" and not args.envs
    if strong:
        E = E // world
    return {"workload": args.workload, "description": desc, "envs_per_gpu": E, "envs_total": world * E,
            "assets": A, "window": W, "features": F, "commission": commission, "obs_materialised": obs,
            "episode_len": EPISODE_LEN, "table_rows": TABLE_ROWS, "preroll_steps": W, "tune": args.tune,
            "cuda_graph": bool(args.graph), "graph_burst_steps": max(1, args.graph) if args.graph else None,
            "burst_kernel_steps": args.burst or None, "actions": "raw N(0,1) scores (softmax branch)",
            "parallelism": f"env-shard x{world}, no data-path collective" + (", NCCL stats all-reduce every step (async)" if world > 1 else ""),
            "l2_policy": "working set per step (obs write + ring) exceeds L2 (126 MB)" if E * A * W * 4 > L2_BYTES
                         else "working set smaller than L2: L2-resident by construction (a flushed-L2 timing is reported beside it in `configs`)"}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the host cores (rank 0 only)."""
    if rank != 0:
        return
    E, A, W, F, c, obs, desc = WORKLOADS[args.workload]
    t0 = time.perf_counter()
    # each "step" of this arm is a bounded sample: all cores stepping single envs for a fixed wall time
    per = max(2.0, min(20.0, 60.0 / max(1, args.steps + args.warmup)))
    per = float(os.environ.get("PMRL_BENCH_REF_SECONDS", per))          # tests shrink the sample
    vals = []
    for i in range(args.warmup + args.steps):
        b = cpu_baseline(A, W, c, seconds=per, context=False)
        if i >= args.warmup:
            vals.append(b)
    v = statistics.mean(x["value"] for x in vals)
    cores = vals[-1]["cores"]
    line = {"impl": "reference", "metric": "asset_steps_per_s", "value": v, "unit": "asset-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * (time.perf_counter() - t0) / max(1, args.steps + args.warmup),
            "higher_is_better": True, "scaling": "strong" if (args.workload == "c4" and not args.envs) else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": shared_config(args, world),
            "cpu_baseline": {"value": v, "unit": "asset-steps/s", "cores": cores, "kind": vals[-1]["kind"],
                             "sample": vals[-1]["sample"] + f"; {per:.0f} s per step"},
            "e2e": {"value": v, "unit": "asset-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------------------------
class Ctx:
    """Per-process state of a GPU run."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        from pmrl_b200 import _lib, dist as pdist
        self.torch, self.dist, self.lib = torch, dist, _lib.load()
        self.rank, self.world, self.local_rank = pdist.init_from_env()
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.peak, self.peak_src = measured_peak_gbs()
        self._flush = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        t = self.torch.tensor([ms], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps, warmup):
        """W untimed + exactly K timed calls of fn(i), CUDA events on the launching stream between barrier + synchronize
        on both sides, max over ranks.  Returns (ms total, kernels launched by libpmrl_b200 in the timed region)."""
        torch = self.torch
        for i in range(warmup):
            fn(i)
        self.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        l0 = self.lib.pmrl_launch_count()
        ev0.record()
        for i in range(steps):
            fn(warmup + i)
        ev1.record()
        launches = int(self.lib.pmrl_launch_count() - l0)
        self.barrier()
        return self.max_over_ranks(ev0.elapsed_time(ev1)), launches

    def timed_flushed(self, fn, steps, first):
        """Cold-L2 timing for workloads whose working set fits the 126 MB L2: a 512 MB fill between the steps evicts it,
        each step is bracketed by its own event pair, the sum is reported (max over ranks)."""
        torch = self.torch
        if self._flush is None:
            self._flush = torch.empty(512 << 20, dtype=torch.uint8, device=self.dev)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        self.barrier()
        for i, (a, b) in enumerate(evs):
            self._flush.fill_(i & 0xff)
            a.record()
            fn(first + i)
            b.record()
        self.barrier()
        return self.max_over_ranks(sum(a.elapsed_time(b) for a, b in evs))

    def free(self):
        import gc
        gc.collect()
        self.torch.cuda.empty_cache()


def make_env(ctx, E, A, W, F, commission, first_env, tables=None):
    import pmrl_b200
    from pmrl_b200 import synth
    from pmrl_b200.env import BatchedTradingEnv
    cfg = pmrl_b200.EnvConfig(num_envs=E, num_assets=A, window_size=W, num_features=F, commission=commission,
                              episode_len=EPISODE_LEN)
    if tables is not None:
        rows = tables["rows"]
        t0 = synth.episode_offsets(E, rows, W, EPISODE_LEN, first_env=first_env)
        return BatchedTradingEnv.from_tables(cfg, tables["close_tm"], tables["feat_am"], t0=t0, device=ctx.dev, collect_stats=True)
    tbl = synth.gbm_ohlc(TABLE_ROWS, A)
    feats = None
    if F != 5:                                                # wider feature sets: OHLC + synthetic indicator channels
        import torch
        g = torch.Generator().manual_seed(99)
        feats = torch.cat([tbl, torch.rand(TABLE_ROWS, A, F - 5, generator=g)], dim=-1)
    t0 = synth.episode_offsets(E, TABLE_ROWS, W, EPISODE_LEN, first_env=first_env)
    return BatchedTradingEnv(cfg, prices=tbl, features=feats, t0=t0, device=ctx.dev, collect_stats=True)


def action_pool(ctx, E, A, n=4):
    torch = ctx.torch
    gen = torch.Generator(device=ctx.dev).manual_seed(4321 + ctx.rank)
    return [torch.randn(E, A, generator=gen, device=ctx.dev) for _ in range(n)]     # "random actions": raw scores


def roofline_entry(ctx, value, world, bpa, E, A, workload, kernel):
    per_gpu_gbs = (value / world) * bpa / 1e9
    return {"bound": "hbm", "achieved": per_gpu_gbs, "peak": ctx.peak, "unit": "GB/s", "frac": per_gpu_gbs / ctx.peak,
            "traffic": ncu_traffic_bytes(workload), "algorithmic_bytes_per_launch": bpa * E * A,
            "bytes_per_asset_step": bpa, "peak_source": ctx.peak_src, "kernel": kernel}


def measure_e2e(ctx, env, pool, E, A, obs, steps, chunks=0):
    """The same metric end to end through the public host-buffer API (C-ABI pmrl_env_step_host): pinned actions in,
    reward/done on the host when the call returns, every step."""
    torch = ctx.torch
    h_act = [p.cpu().pin_memory() for p in pool[:2]]
    h_rew = torch.empty(E, dtype=torch.float32).pin_memory()
    h_done = torch.empty(E, dtype=torch.uint8).pin_memory()

    def e2e_step(i):
        env.step_host(h_act[i % 2], h_rew, h_done, obs=obs, chunks=chunks)

    for i in range(3):
        e2e_step(i)
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        e2e_step(i)
    e1.record()
    ctx.barrier()
    ems = ctx.max_over_ranks(e0.elapsed_time(e1))
    return {"value": ctx.world * E * A * steps / (ems * 1e-3), "unit": "asset-steps/s",
            "h2d_bytes_per_step": E * A * 4, "d2h_bytes_per_step": E * 5, "chunks": chunks,
            "transfer": ("zero-copy: ONE kernel reads the pinned host actions over PCIe and writes reward/done into mapped pinned memory"
                         if chunks == 0 else "sliced H2D/D2H copies overlapped with per-slice kernels"),
            "api": "BatchedTradingEnv.step_host -> C-ABI pmrl_env_step_host",
            "ms_per_step": ems / steps}


def kernel_name(obs, launches_per_step, A, F, burst=0, E=1 << 30):
    """Name of the dominant kernel of a workload (what `roofline` is about), from the launcher's own dispatch rules."""
    staged = A > 128 and A % 4 == 0 and E > 148 * 2 * 8            # env_kernels.cu:launch_step_s
    state = "k_env_step_staged" if staged else "k_env_step"
    if burst:
        return f"{state} x{burst} launches" if staged else "k_env_step_burst"
    if not obs:
        return state
    return "k_env_step_obs_rt" if launches_per_step <= 1.001 else f"{state} + k_obs_build_rows"


def config_entry(ctx, name, steps, warmup, mode="step", K=0, e2e=True, flushed=False):
    """One entry of `configs`: the named BASELINE workload (its total env count divided over the ranks), timed on its own."""
    torch = ctx.torch
    E_total, A, W, F, commission, obs, desc = WORKLOADS[name]
    per_gpu = name in ("c4_shard", "c4_state", "c5_obs", "c4_f9", "c4_f13", "c4_f17", "c4_f7", "c4_f6", "c4_f8")
    E = E_total if per_gpu else E_total // ctx.world
    env = make_env(ctx, E, A, W, F, commission, ctx.rank * E)
    pool = action_pool(ctx, E, A)
    env.reset(obs=obs)
    for i in range(W):                                        # steady state: ring full
        env.step(pool[i % 4], obs=False)
    n_pool = len(pool)
    if mode in ("burst", "graph"):
        steps = max(K, steps // K * K)
        warmup = max(K, -(-warmup // K) * K)
        bpool = [torch.stack([pool[(j + k) % n_pool] for k in range(K)]) for j in range(n_pool)]
    graph_launches = 0
    if mode == "burst":
        b_rew = torch.empty(K, E, dtype=torch.float32, device=ctx.dev)
        b_done = torch.empty(K, E, dtype=torch.uint8, device=ctx.dev)

        def fn(i):
            if i % K == 0:
                env.step_burst(bpool[(i // K) % n_pool], b_rew, b_done)
    elif mode == "graph":
        c0 = ctx.lib.pmrl_launch_count()
        static_actions, replay = env.graphed_step(obs=obs, steps=K)
        graph_launches = int(ctx.lib.pmrl_launch_count() - c0) // (K + 1)

        def fn(i):
            if i % K == 0:
                static_actions.copy_(bpool[(i // K) % n_pool] if K > 1 else pool[i % n_pool])
                replay()
    else:
        def fn(i):
            env.step(pool[i % n_pool], obs=obs)
    ms, launches = ctx.timed(fn, steps, warmup)
    if mode == "graph":
        launches = graph_launches * steps
    value = ctx.world * E * A * steps / (ms * 1e-3)
    bpa = algorithmic_bytes_per_asset_step(A, W, F, commission, obs)
    out = {"description": desc, "mode": mode + (f" x{K}" if K else ""), "envs_per_gpu": E, "envs_total": ctx.world * E,
           "assets": A, "window": W, "features": F, "commission": commission, "obs_materialised": obs,
           "scaling": "weak" if per_gpu else "strong", "steps": steps, "warmup": warmup,
           "ms_per_step": ms / steps, "value": value, "unit": "asset-steps/s", "env_steps_per_s": value / A,
           "gpu_launches": launches,
           "roofline": roofline_entry(ctx, value, ctx.world, bpa, E, A, name if mode == "step" else f"{name}_{mode}",
                                      kernel_name(obs, launches / steps, A, F, burst=(K if mode == "burst" else 0), E=E)),
           "l2": "working set > L2" if E * A * 4 * (W if obs else 2) > L2_BYTES else "L2-resident back to back"}
    if flushed:
        fms = ctx.timed_flushed(fn, steps, warmup + steps)
        out["l2_flushed"] = {"ms_per_step": fms / steps, "value": ctx.world * E * A * steps / (fms * 1e-3),
                             "how": "512 MB fill between steps, per-step CUDA events"}
    if e2e and mode == "step":
        out["e2e"] = measure_e2e(ctx, env, pool, E, A, obs, min(steps, 10))
    del env, pool
    ctx.free()
    return out


def config3_entry(ctx, steps, warmup):
    """BASELINE config 3: the SAC off-policy collect loop at 65,536 envs x 100 assets on FFD features — feature path
    (FFD → min-max → packed tables, `build_env_tables`) once, then per step the fused kernel writes the obs AND the
    (i, a, r) index-replay row itself (`step_io` with `DeviceReplayBuffer.sinks`), then `sample()` of B = 64."""
    torch = ctx.torch
    from pmrl_b200 import synth
    from pmrl_b200.buffers import DeviceReplayBuffer
    from pmrl_b200.features import build_env_tables
    E_total, A, W, F, commission, obs, desc = WORKLOADS["c3"]
    E = E_total // ctx.world
    raw = synth.gbm_ohlc(TABLE_ROWS + 2048, A).to(ctx.dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    build_env_tables(raw, d=0.4, thres=1e-4)                  # warm-up (module load)
    ev0.record()
    tabs = build_env_tables(raw, d=0.4, thres=1e-4)
    ev1.record()
    torch.cuda.synchronize()
    feat_ms = ev0.elapsed_time(ev1)
    env = make_env(ctx, E, A, W, F, commission, ctx.rank * E, tables=tabs)
    pool = action_pool(ctx, E, A)
    train_len = 64 + 2 * (W - 1)
    rb = DeviceReplayBuffer(tabs["feat_am"], F, train_len, E, A, W, buffer_size=2 * 64, batch_size=64)
    env.reset(obs=True)
    for i in range(W):
        env.step(pool[i % 4], obs=False)
    L = rb.epoch_len

    def fn(i):
        epoch, slot = divmod(i, L)
        env.step_io(pool[i % 4], **rb.sinks(epoch, 2 * (W - 1) + slot))
    ms, launches = ctx.timed(fn, steps, warmup)
    value = ctx.world * E * A * steps / (ms * 1e-3)
    bpa = algorithmic_bytes_per_asset_step(A, W, F, commission, True, sinks=4.0 + 4.0 / A)
    g = torch.Generator().manual_seed(0)
    rb.sample(g, sampler="buffer")
    torch.cuda.synchronize()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(10):
        rb.sample(g, sampler="buffer")
    s1.record()
    torch.cuda.synchronize()
    out = {"description": "BASELINE config 3: off-policy collect, 65,536 envs x 100 assets on FFD(d=0.4) + min-max features; the step "
                          "kernel writes obs and the (i, a, r) replay row", "mode": "collect_off_policy",
           "envs_per_gpu": E, "envs_total": ctx.world * E, "assets": A, "window": W, "features": F, "scaling": "strong",
           "steps": steps, "warmup": warmup, "ms_per_step": ms / steps, "value": value, "unit": "asset-steps/s",
           "env_steps_per_s": value / A, "gpu_launches": launches,
           "feature_path_ms": feat_ms, "feature_path": f"FFD + scale + pack of {A * 4} series x {raw.shape[0]} rows (max width {tabs['max_width']})",
           "replay_sample_ms": s0.elapsed_time(s1) / 10, "replay_sample": "B = 64 (s, a, r, s'), buffer.py sampler, incl. host draws",
           "roofline": roofline_entry(ctx, value, ctx.world, bpa, E, A, "c3_collect", kernel_name(True, launches / steps, A, F))}
    del env, pool, rb, tabs
    ctx.free()
    return out


def collect_on_policy_entry(ctx, steps, warmup, bare_ms):
    """On-policy collect at the headline shape with an index-mode rollout buffer: the step kernel writes obs plus the
    buffer rows (raw action, value, reward, loader index, post-drift weights) itself — no add() kernel, no obs copy."""
    torch = ctx.torch
    from pmrl_b200.buffers import DeviceRolloutBuffer
    E, A, W, F, commission, obs, desc = WORKLOADS["c4_shard"]
    env = make_env(ctx, E, A, W, F, commission, ctx.rank * E)
    pool = action_pool(ctx, E, A)
    slots = 24
    train_len = slots + W - 1
    buf = DeviceRolloutBuffer(F, train_len, E, A, W, mode="index", feat_am=env.feat_am, y_tm=env.y_tm, device=ctx.dev)
    env.reset(obs=True)
    for i in range(W):
        env.step(pool[i % 4], obs=False)

    def fn(i):
        env.step_io(pool[i % 4], **buf.sinks(W + (i % (slots - 1))))
    ms, launches = ctx.timed(fn, steps, warmup)
    value = ctx.world * E * A * steps / (ms * 1e-3)
    bpa = algorithmic_bytes_per_asset_step(A, W, F, commission, True, sinks=8.0 + 12.0 / A)
    out = {"description": "on-policy collect at the config-4 shard shape, index-mode rollout buffer rows written by the step kernel",
           "mode": "collect_on_policy(index)", "envs_per_gpu": E, "envs_total": ctx.world * E, "assets": A, "window": W,
           "scaling": "weak", "steps": steps, "warmup": warmup, "ms_per_step": ms / steps, "value": value, "unit": "asset-steps/s",
           "gpu_launches": launches, "bare_step_ms": bare_ms, "overhead_vs_bare_step": (ms / steps) / bare_ms - 1.0 if bare_ms else None,
           "buffer_bytes_per_env_step": 8 * A + 12, "epoch_of_1000_steps_at_65536_envs_gb": 65536 * 1000 * (8 * A + 12) / 1e9,
           "roofline": roofline_entry(ctx, value, ctx.world, bpa, E, A, "c4_collect", kernel_name(True, launches / steps, A, F))}
    del env, pool, buf
    ctx.free()
    return out


def config1_gpu_shim(ctx, steps=1500):
    """Config-1 shape through the drop-in E = 1 `compat.TradingEnv` with CPU caller tensors (one step at a time)."""
    import torch
    import pmrl_b200
    from pmrl_b200.compat import TradingEnv
    A, W, F = 11, 50, 5
    env = TradingEnv(pmrl_b200.EnvConfig(num_assets=A, window_size=W, num_features=F))
    g = torch.Generator().manual_seed(0)
    feat = torch.rand(A, W, F, generator=g)
    acts = torch.randn(64, 1, A, 1, generator=g)
    ys = 1 + 0.01 * torch.randn(64, A, generator=g)
    env.reset(feat)
    for s in range(50):
        env.step(acts[s % 64], feat, ys[s % 64])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for s in range(steps):
        if s % 500 == 499:
            env.reset(feat)
        r, _ = env.step(acts[s % 64], feat, ys[s % 64])
    float(r)
    torch.cuda.synchronize()
    return steps / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4_shard", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="override envs per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` block (the other BASELINE configs)")
    ap.add_argument("--configs", action="store_true", help="force the `configs` block for a non-default workload")
    ap.add_argument("--e2e-chunks", type=int, default=0,
                    help="env slices of the host-buffer step: >0 geometric x2.5, <0 equal, 0 library default (zero-copy)")
    ap.add_argument("--stats-every", type=int, default=1,
                    help="multi-GPU: all-reduce the stats vector over NCCL every K steps (SURVEY 8e: K = 1); 0 = only at the end")
    ap.add_argument("--graph", type=int, nargs="?", const=1, default=0, metavar="K",
                    help="replay the step from a CUDA graph (launch-bound small batches); K > 1 captures K-step bursts in one graph")
    ap.add_argument("--burst", type=int, default=0, metavar="K",
                    help="state-only workloads: advance K steps per launch through pmrl_env_step_burst (imagination bursts)")
    ap.add_argument("--tune", action="append", default=[], metavar="KEY=VAL",
                    help="kernel launch-shape override: group|ctas|fast|rt|staged = int (pmrl_set_tuning)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write what the last one returned (obs, reward, done; rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from pmrl_b200 import dist as pdist
    from pmrl_b200 import _lib

    ctx = Ctx()
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    try:                                                      # one rank per GPU: keep each Python loop on its own cores
        cores = sorted(os.sched_getaffinity(0))
        if world > 1 and len(cores) >= 2 * world:
            per = len(cores) // world
            os.sched_setaffinity(0, cores[ctx.local_rank * per:(ctx.local_rank + 1) * per])
    except Exception:
        pass
    tune_keys = {"group": _lib.TUNE_GROUP_ENVS, "ctas": _lib.TUNE_CTAS_PER_SM, "fast": _lib.TUNE_FAST_FILL, "rt": _lib.TUNE_RING_TMA, "staged": _lib.TUNE_STAGED, "hoststream": _lib.TUNE_HOST_STREAM}
    for kv in args.tune:
        k, v = kv.split("=")
        _lib.set_tuning(tune_keys[k], int(v))

    cfg_line = shared_config(args, world)
    E, A, W, F, commission, obs = (cfg_line[k] for k in ("envs_per_gpu", "assets", "window", "features", "commission", "obs_materialised"))
    strong = args.workload == "c4" and not args.envs
    env = make_env(ctx, E, A, W, F, commission, rank * E)     # weak scaling: rank r owns global envs [r*E, (r+1)*E)
    n_pool = 4
    pool = action_pool(ctx, E, A, n_pool)
    env.reset(obs=obs)
    # steady state of a 1,000-step episode: the weight ring is full after W-1 steps (95 % of all steps), and only
    # then does the obs weight channel read the whole ring.  Pre-roll W state-only steps (untimed) to get there.
    for i in range(W):
        env.step(pool[i % n_pool], obs=False)

    # multi-GPU: the 10-double stats vector is all-reduced over NCCL EVERY step (SURVEY.md §8(e), K = 1), issued
    # asynchronously behind a snapshot so the next step's kernel is not ordered after the collective
    reducer = pdist.AsyncStatsReducer(dev) if (world > 1 and args.stats_every > 0) else None
    stats_in_sync = None

    graph_launches_per_step = 0
    burst = max(1, args.graph or args.burst)
    if args.steps % burst:
        raise SystemExit(f"--steps must be a multiple of the {burst}-step burst")
    returned = [None]                                         # what the last timed step returned (--dump-outputs)
    if args.graph:
        if args.warmup % burst:
            args.warmup = max(burst, -(-args.warmup // burst) * burst)
        c0 = ctx.lib.pmrl_launch_count()
        static_actions, replay = env.graphed_step(obs=obs, steps=burst)
        graph_launches_per_step = int(ctx.lib.pmrl_launch_count() - c0) // (burst + 1)   # one warm-up step + the captured burst
        burst_pool = [torch.stack([pool[(j + k) % n_pool] for k in range(burst)]) if burst > 1 else pool[j] for j in range(n_pool)]

        def one_step(i):                                      # called once per env step; a burst is replayed on its first step
            if i % burst == 0:
                static_actions.copy_(burst_pool[(i // burst) % n_pool])   # the policy would write its actions here
                returned[0] = replay()
    elif args.burst:
        if obs:
            raise SystemExit("--burst is a state-only mode")
        args.warmup = max(burst, -(-args.warmup // burst) * burst)
        burst_pool = [torch.stack([pool[(j + k) % n_pool] for k in range(burst)]) for j in range(n_pool)]
        b_rew = torch.empty(burst, E, dtype=torch.float32, device=dev)
        b_done = torch.empty(burst, E, dtype=torch.uint8, device=dev)

        def one_step(i):
            if i % burst == 0:
                returned[0] = env.step_burst(burst_pool[(i // burst) % n_pool], b_rew, b_done)
    else:
        def one_step(i):
            returned[0] = env.step(pool[i % n_pool], obs=obs)
            if reducer is not None and i % args.stats_every == 0:
                reducer.launch(env._stats)

    sampler = ClockSampler(ctx.local_rank)
    if rank == 0:
        sampler.start()                                       # samples clocks / throttle reasons over warm-up + timed region
        time.sleep(0.25)                                      # nvidia-smi needs a moment before its first sample
    ms, gpu_launches = ctx.timed(one_step, args.steps, args.warmup)
    if args.graph:
        gpu_launches = graph_launches_per_step * args.steps      # replayed from the graph: counted at capture time
    clocks = sampler.summary() if rank == 0 else None
    if args.dump_outputs and rank == 0:                       # before anything else reuses the env's output buffers
        *o, rew, done = returned[0]                           # (obs | None, reward, done) or, from a burst, (reward, done)
        outs = {"reward": (rew, rew.dim() - 1), "done": (done, done.dim() - 1)}
        if o and o[0] is not None:
            outs["obs"] = (o[0], 0)
        dump_outputs(args.dump_outputs, outs, E)
    if reducer is not None:                                   # the last step's reduced vector must equal a fresh reduce
        last = reducer.result()
        fresh = pdist.all_reduce_stats(env._stats.clone())
        stats_in_sync = bool(torch.allclose(last, fresh, rtol=1e-12, atol=0.0)) if args.stats_every == 1 else None
    stats = env.stats(all_reduce=world > 1)                   # NCCL all-reduce of the 10-double stats vector

    # ---- end to end through the public API with host buffers (H2D actions, D2H reward/done every step) ----
    e2e = None if args.no_e2e else measure_e2e(ctx, env, pool, E, A, obs, args.steps, args.e2e_chunks)
    del env, pool
    ctx.free()

    # ---- the other BASELINE configs, each timed on its own (after and outside the headline's timed region) ----
    configs = None
    if (args.workload == "c4_shard" and not args.envs and not args.no_configs and not args.graph and not args.burst) or args.configs:
        configs = {}
        ks, kw = max(10, args.steps), max(3, args.warmup)

        def add(key, fn, *a, **k):
            mark = sampler.mark() if rank == 0 else 0
            try:
                ent = fn(*a, **k)
            except Exception as ex:                            # a config that cannot run (e.g. memory) is reported, not hidden
                ctx.free()
                ent = {"error": f"{type(ex).__name__}: {ex}"[:300]}
            if rank == 0 and isinstance(ent, dict):
                ent["clocks"] = sampler.summary(mark)
            configs[key] = ent

        add("c2", config_entry, ctx, "c2", 10 * ks, 2 * kw, flushed=True)
        add("c2_state", config_entry, ctx, "c2_state", 10 * ks, 2 * kw, flushed=True)
        add("c2_state_burst15", config_entry, ctx, "c2_state", 15 * ks, 15 * 2, mode="burst", K=15, flushed=False)
        add("c2_state_graph15", config_entry, ctx, "c2_state", 15 * ks, 15 * 2, mode="graph", K=15)
        add("c3", config_entry, ctx, "c3", ks, kw)
        add("c3_collect", config3_entry, ctx, ks, kw)
        add("c4_state", config_entry, ctx, "c4_state", ks, kw)
        add("c4_f9", config_entry, ctx, "c4_f9", ks, kw, e2e=False)
        add("c4_f7", config_entry, ctx, "c4_f7", ks, kw, e2e=False)
        add("c4_collect", collect_on_policy_entry, ctx, ks, kw, ms / args.steps)
        add("c5", config_entry, ctx, "c5", ks, kw)
        add("c5_burst15", config_entry, ctx, "c5", 15, 15, mode="burst", K=15)
        add("c5_obs", config_entry, ctx, "c5_obs", ks, kw, e2e=False)
        if world > 1 or torch.cuda.get_device_properties(dev).total_memory > 150e9:
            add("c4", config_entry, ctx, "c4", ks, kw)         # config 4 whole (1,048,576 envs): 126 GB on one GPU
        if rank == 0:
            c1 = {"gpu_shim": None}
            try:
                c1 = config1_cpu(float(os.environ.get("PMRL_BENCH_C1_SECONDS", 6.0)))
                c1["gpu_shim"] = {"env_steps_per_s": config1_gpu_shim(ctx), "what": "compat.TradingEnv (E = 1, CPU caller tensors, one step "
                                  "at a time like train/on_policy.py:59-67) on the CUDA kernels; latency-bound by construction"}
            except Exception as ex:
                c1["error"] = f"{type(ex).__name__}: {ex}"[:300]
            configs["c1"] = c1
    if rank == 0:
        sampler.stop()

    if rank == 0:
        sec = ms * 1e-3
        value = world * E * A * args.steps / sec
        bpa = algorithmic_bytes_per_asset_step(A, W, F, commission, obs)
        line = {
            "metric": "asset_steps_per_s", "value": value, "unit": "asset-steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "env_steps_per_s": value / A,
            "config": cfg_line,
            "roofline": roofline_entry(ctx, value, world, bpa, E, A, args.workload,
                                       kernel_name(obs, gpu_launches / args.steps, A, F, burst=args.burst, E=E)),
            "clocks": clocks,
            "gpu_launches": gpu_launches,
            "stats": {k: stats[k] for k in ("n_envs", "mean_reward", "mean_value", "n_done")},
        }
        if reducer is not None:
            line["stats_allreduce"] = {"every_steps": args.stats_every, "launches": reducer.launches, "last_equals_fresh_reduce": stats_in_sync}
        if e2e:
            line["e2e"] = e2e
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(A, W, commission)
        if configs is not None:
            line["configs"] = configs
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
