// env_kernels.cu — environment reset / step / observation kernels + their C-ABI entry points.
//
// Kernels (sm_100a):
//   k_env_step<NPL>      state-only transition ("Mode S"): persistent grid of warps, one env per warp.
//   k_env_reset          masked re-initialisation, one env per warp.
//   k_obs_build          one CTA per (env, asset-tile): gather window + weight channel into a shared
//                        tile that is the byte image of obs[e, a0:a0+na, :, :], then one TMA bulk store.
//   (the fused step+obs "Mode O" kernels live in env_step_rt.cu / env_step_fast.cu)
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>
#include "pmrl_b200.h"
#include "pmrl_device.cuh"
#include "env_step.cuh"
#include "obs_tile.cuh"
#include "host_util.h"
#include "env_launch.h"
#include <type_traits>

namespace pmrl {

constexpr int kStepThreads = 256;
constexpr int kStepWarps = kStepThreads / 32;
constexpr int kObsThreads = 256;

// ------------------------------------------------------------------------------------------------
// Mode S: state-only step.
// ------------------------------------------------------------------------------------------------
// Wide envs with commission keep w and the previous weights in registers through the mu iteration (2·NPL) and fetch the
// price relatives after it (LOADY = false): 80 registers → three resident CTAs per SM instead of two.
template <int NPL, bool HASC>
constexpr bool kDeferY = HASC && (NPL == 8 || NPL == 16);
// Resident CTAs per SM the register allocation aims for.  Narrow envs without the cross-env software pipeline (small
// batches: one env per warp, latency-bound) want every warp of the batch resident at once — 4,096 envs are 28 warps per SM.
template <int NPL, bool HASC, bool PIPE>
constexpr int kStepMinBlocks = PIPE ? 2 : NPL <= 2 ? 4 : NPL == 4 ? 3 : kDeferY<NPL, HASC> ? 3 : NPL == 32 ? 1 : 2;

template <int NPL, bool HASC, int VEC, bool PIPE, bool TAIL, bool NOSINKS = false>
__global__ void __launch_bounds__(kStepThreads, kStepMinBlocks<NPL, HASC, PIPE>) k_env_step(const StepParams p) {
    __shared__ double s_stats[kStepWarps * PMRL_STATS_LEN];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gw = blockIdx.x * kStepWarps + warp;
    const int nw = gridDim.x * kStepWarps;
    WarpStats ws;
    wstats_init(ws);
    StepOut so;
    if constexpr (PIPE) {
        // three envs of this warp in flight: scalars of e+2nw, vectors of e+nw, arithmetic of e
        EnvScalars s0, s1, s2;
        EnvVectors<NPL, HASC, VEC> v0, v1;
        int e = gw;
        if (e < p.E) { env_load_scalars(p, e, s0); env_load_vectors<NPL, HASC, VEC, TAIL>(p, e, lane, s0, v0); }
        if (e + nw < p.E) env_load_scalars(p, e + nw, s1);
        for (; e < p.E; e += nw) {
            if (e + 2 * nw < p.E) env_load_scalars(p, e + 2 * nw, s2);
            if (e + nw < p.E) env_load_vectors<NPL, HASC, VEC, TAIL>(p, e + nw, lane, s1, v1);
            env_compute_rows<NPL, HASC, VEC, TAIL, true, true, false, NoHook, false, NOSINKS>(p, e, lane, s0, v0.a, v0.y, v0.wl, so, ws);
            s0 = s1; s1 = s2; v0 = v1;
        }
    } else {
        // wide envs (NPL >= 8): no registers for a second env's vectors.  Keep the scalars of the next two envs in
        // registers and pull the next env's DRAM rows into L2 while this one computes: the dependent chain
        // scalars → row addresses → vectors then costs one L2 hit per env instead of two DRAM round trips.
        constexpr bool LOADY = !kDeferY<NPL, HASC>;
        EnvScalars s0, s1, s2;
        int e = gw;
        if (e < p.E) env_load_scalars(p, e, s0);
        if (e + nw < p.E) env_load_scalars(p, e + nw, s1);
        for (; e < p.E; e += nw) {
            EnvVectors<NPL, HASC, VEC> v;
            if (e + 2 * nw < p.E) env_load_scalars(p, e + 2 * nw, s2);
            env_load_rows<NPL, HASC, VEC, TAIL, true, LOADY>(p, e, lane, s0, v.a, v.y, v.wl);
            if (e + nw < p.E) env_prefetch_vectors<HASC>(p, e + nw, lane, s1);
            env_compute_rows<NPL, HASC, VEC, TAIL, LOADY>(p, e, lane, s0, v.a, v.y, v.wl, so, ws);
            s0 = s1; s1 = s2;
        }
    }
    if (p.stats) { wstats_store(ws, s_stats + warp * PMRL_STATS_LEN, lane); stats_flush_block(p.stats, s_stats, kStepWarps); }
}

// ------------------------------------------------------------------------------------------------
// Mode S, K-step burst: ONE launch advances every env by `p.burst` steps on pre-supplied actions [K, E, A]
// (imagination rollouts: HORIZON = 15, config/dreamer.py:54).  A warp keeps its env's V / ring pointer / local step /
// episode return in registers across the burst and writes them back once; the weights it has just written ARE the next
// step's previous weights (weight_buffer.py:30): the two register rows swap roles from step to step (w' of step k is
// read as w_last by step k+1 while the dead row receives the next action), so per step only the action row comes from
// DRAM — requested one step ahead (into registers for narrow envs, into L2 for wide ones).  Reward / done / the ring row
// are written every step; a burst is bit-identical to K eager steps.
// ------------------------------------------------------------------------------------------------
template <int NPL, bool HASC, int VEC, bool TAIL>
__global__ void __launch_bounds__(kStepThreads, kStepMinBlocks<NPL, HASC, false>) k_env_step_burst(const StepParams p) {
    __shared__ double s_stats[kStepWarps * PMRL_STATS_LEN];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gw = blockIdx.x * kStepWarps + warp;
    const int nw = gridDim.x * kStepWarps;
    WarpStats ws;
    wstats_init(ws);
    const int K = p.burst;
    const size_t EA = (size_t)p.E * p.A;
    constexpr bool REGPF = (NPL <= 4);                   // next step's action / y rows prefetched into registers
    constexpr bool LOADY = !kDeferY<NPL, HASC>;
    constexpr int WLN = HASC ? NPL : 1;
    for (int e = gw; e < p.E; e += nw) {
        StepParams q = p;                                 // per-step views: actions[k], reward[k], done[k]
        EnvScalars sc;
        env_load_scalars(p, e, sc);
        float X[NPL], Y[WLN], yv[NPL];                    // X / Y: (action → w', previous weights), roles swap every step (HASC)
        float an[REGPF ? NPL : 1], yn[REGPF ? NPL : 1];
        StepOut so;
        env_load_rows<NPL, HASC, VEC, TAIL, true, LOADY>(q, e, lane, sc, X, yv, Y);
        // one step: `a` holds the action (step 0 / narrow envs) or receives it here (wide envs, k > 0); `wl` = previous weights
        auto step = [&](float (&a)[NPL], float (&wl)[WLN], float (&nxt)[HASC ? NPL : NPL], int k) {
            EnvScalars sn = sc;                           // the local step after this one is known before the arithmetic,
            sn.k = env_needs_reset(p, sc) ? 0 : sc.k + 1; // so the next step's rows are requested now
            if (k + 1 < K) {
                StepParams qn = q;
                qn.actions = q.actions + EA;
                float none[1];
                if constexpr (REGPF) env_load_rows<NPL, false, VEC, TAIL, false, true>(qn, e, lane, sn, an, yn, none);
                else env_prefetch_vectors<false>(qn, e, lane, sn);
            }
            if constexpr (!REGPF) {
                if (k > 0) { float none[1]; env_load_rows<NPL, false, VEC, TAIL, false, LOADY>(q, e, lane, sc, a, yv, none); }
            }
            // (pmrl_env_step_burst takes no sinks / host mirrors: their per-step null tests are compiled out)
            env_compute_rows<NPL, HASC, VEC, TAIL, LOADY, false, false, NoHook, false, /*NOSINKS=*/true>(q, e, lane, sc, a, yv, wl, so, ws);
            sc.V = so.V; sc.i = so.idx_new; sc.full = so.is_full; sc.k = so.k; sc.epr = so.epr;
            q.actions += EA; q.reward += p.E; q.done += p.E;
            if constexpr (REGPF) {                        // narrow envs: the prefetched rows move into the row that is now dead
                if (k + 1 < K) {
#pragma unroll
                    for (int j = 0; j < NPL; ++j) { nxt[j] = an[j]; yv[j] = yn[j]; }
                }
            }
        };
        if constexpr (HASC) {
            for (int k = 0; k < K; k += 2) {
                step(X, Y, Y, k);                         // w' → X; next action → Y
                if (k + 1 < K) step(Y, X, X, k + 1);      // w' → Y; next action → X
            }
        } else {
            for (int k = 0; k < K; ++k) step(X, Y, X, k);
        }
        if (lane == 0) {                                  // the scalar state goes back once per burst
            p.value[e] = sc.V; p.idx[e] = sc.i; p.is_full[e] = (uint8_t)sc.full; p.t[e] = sc.k;
            if (p.ep_return) p.ep_return[e] = sc.epr;
        }
    }
    if (p.stats) { wstats_store(ws, s_stats + warp * PMRL_STATS_LEN, lane); stats_flush_block(p.stats, s_stats, kStepWarps); }
}

// ------------------------------------------------------------------------------------------------
// Masked reset (trading_env.py:28-29, weight_buffer.py:46-50).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kStepThreads) k_env_reset(const StepParams p) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gw = blockIdx.x * kStepWarps + warp;
    const int nw = gridDim.x * kStepWarps;
    for (int e = gw; e < p.E; e += nw) {
        if (p.mask && !p.mask[e]) continue;
        ring_reset_warp(p.hist + (size_t)e * p.W * p.A, p.W, p.A, lane);
        if (lane == 0) {
            p.value[e] = p.initial_cash;
            p.idx[e] = 1; p.is_full[e] = 0; p.t[e] = 0;
            if (p.sharpe) { p.sharpe[3 * (size_t)e] = 0.0; p.sharpe[3 * (size_t)e + 1] = 0.0; p.sharpe[3 * (size_t)e + 2] = 0.0; }
            if (p.ep_return) p.ep_return[e] = 0.0f;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Observation tiles from the current state.
// ------------------------------------------------------------------------------------------------
// OT: obs element type (float, or uint16_t bf16 bits — PMRL_OBS_BF16); the fp32 and bf16 kernels below share this body.
template <typename OT>
__device__ __forceinline__ void obs_build(const StepParams& p) {
    extern __shared__ __align__(128) unsigned char smem_obs[];
    OT* const tile = reinterpret_cast<OT*>(smem_obs);
    const int e = blockIdx.x / p.tiles_per_env;
    const int ti = blockIdx.x - e * p.tiles_per_env;
    if (p.mask && !p.mask[e]) return;
    const int a0 = ti * p.tile_assets;
    const int na = min(p.tile_assets, p.A - a0);
    const int tid = threadIdx.x;
    const int idx = p.idx[e], full = p.is_full[e];
    if (p.obs_mode == PMRL_OBS_FULL) {
        const int row0 = (p.t0 ? p.t0[e] : 0) + p.t[e];
        obs_tile_fill_features(p, tile, a0, na, row0, tid, kObsThreads);
    }
    obs_tile_fill_weights(p, tile, p.hist + (size_t)e * p.W * p.A, a0, na, idx, full, nullptr, -1, tid, kObsThreads);
    fence_proxy_async_smem();
    __syncthreads();
    obs_tile_store(p, tile, e, a0, na, tid, kObsThreads);
    if (p.obs_mode == PMRL_OBS_FULL && p.obs_bulk_ok && tid == 0) bulk_wait_read<0>();
}
__global__ void __launch_bounds__(kObsThreads) k_obs_build(const StepParams p) { obs_build<float>(p); }
__global__ void __launch_bounds__(kObsThreads) k_obs_build_bf16(const StepParams p) { obs_build<uint16_t>(p); }


// The same tile for the common shape (4 feature channels + weight slot, W <= 64, 32-asset tiles), without the
// per-element index divisions of the generic fill: a warp owns an asset row of the feature window (lanes over window
// rows, one float4 per row), and lanes run over assets for the weight channel (coalesced 128-byte ring rows).  All
// loads of a thread are issued before the first shared store; the L2-resident table loads go first so that no
// DRAM-latency ring load sits ahead of them in the L1 return queue.
__global__ void __launch_bounds__(kObsThreads) k_obs_build_rows(const StepParams p) {
    extern __shared__ __align__(128) float tile[];                  // [32][W][5]
    const int A = p.A, W = p.W, T = p.T;
    const int e = blockIdx.x / p.tiles_per_env;
    const int ti = blockIdx.x - e * p.tiles_per_env;
    if (p.mask && !p.mask[e]) return;
    const int a0 = ti * 32;
    const int na = min(32, A - a0);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int idx = p.idx[e], full = p.is_full[e];
    const int row0 = p.t0[e] + p.t[e];
    const int shift = full ? 0 : (W - idx);                         // weight_buffer.py:38-42
    const bool w0 = lane < W, w1 = lane + 32 < W;
    const float4* __restrict__ tbl = reinterpret_cast<const float4*>(p.feat_am) + ((size_t)a0 * T + row0 + lane);
    float4 fv[4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int al = warp + 8 * i;
        if (al < na) {
            const float4* __restrict__ src = tbl + (size_t)al * T;
            if (w0) fv[i][0] = ld_keep4(src, kPolicyEvictLast);
            if (w1) fv[i][1] = ld_keep4(src + 32, kPolicyEvictLast);
        }
    }
    const float* __restrict__ ring = p.hist + (size_t)e * W * A + a0 + lane;
    float rv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int w = warp + 8 * j, slot = w - shift;
        rv[j] = (w < W && slot >= 0 && lane < na) ? ld_once(ring + (size_t)slot * A, kPolicyEvictFirst) : 0.0f;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int al = warp + 8 * i;
        if (al < na) {
            float* d = tile + (al * W + lane) * 5;
            if (w0) { const float4 v = fv[i][0]; d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w; }
            if (w1) { const float4 v = fv[i][1]; d[160] = v.x; d[161] = v.y; d[162] = v.z; d[163] = v.w; }
        }
    }
    if (lane < na) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int w = warp + 8 * j;
            if (w < W) tile[(lane * W + w) * 5 + 4] = rv[j];
        }
    }
    fence_proxy_async_smem();
    __syncthreads();
    float* __restrict__ dst = p.obs + ((size_t)e * A + a0) * W * 5;
    const int n = na * W * 5;
    if (((((uintptr_t)dst) | ((size_t)n * 4)) & 15) == 0) {
        if (tid == 0) { bulk_store_s2g(dst, tile, (uint32_t)n * 4u, kPolicyEvictFirst); bulk_commit(); bulk_wait_read<0>(); }
    } else {
        for (int q = tid; q < n; q += kObsThreads) dst[q] = tile[q];
    }
}

// k_obs_build_rows with the tile in obs element type OT (instantiated for bf16 bits: k_obs_build_rows_bf16).  The fp32
// kernel above keeps its own code: compiled through this template its SASS comes out reordered.
template <typename OT>
__device__ __forceinline__ void obs_build_rows(const StepParams& p) {
    extern __shared__ __align__(128) unsigned char smem_obs[];
    OT* const tile = reinterpret_cast<OT*>(smem_obs);               // [32][W][5]
    const int A = p.A, W = p.W, T = p.T;
    const int e = blockIdx.x / p.tiles_per_env;
    const int ti = blockIdx.x - e * p.tiles_per_env;
    if (p.mask && !p.mask[e]) return;
    const int a0 = ti * 32;
    const int na = min(32, A - a0);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int idx = p.idx[e], full = p.is_full[e];
    const int row0 = p.t0[e] + p.t[e];
    const int shift = full ? 0 : (W - idx);                         // weight_buffer.py:38-42
    const bool w0 = lane < W, w1 = lane + 32 < W;
    const float4* __restrict__ tbl = reinterpret_cast<const float4*>(p.feat_am) + ((size_t)a0 * T + row0 + lane);
    float4 fv[4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int al = warp + 8 * i;
        if (al < na) {
            const float4* __restrict__ src = tbl + (size_t)al * T;
            if (w0) fv[i][0] = ld_keep4(src, kPolicyEvictLast);
            if (w1) fv[i][1] = ld_keep4(src + 32, kPolicyEvictLast);
        }
    }
    const float* __restrict__ ring = p.hist + (size_t)e * W * A + a0 + lane;
    float rv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int w = warp + 8 * j, slot = w - shift;
        rv[j] = (w < W && slot >= 0 && lane < na) ? ld_once(ring + (size_t)slot * A, kPolicyEvictFirst) : 0.0f;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int al = warp + 8 * i;
        if (al < na) {
            OT* d = tile + (al * W + lane) * 5;
            if (w0) { const float4 v = fv[i][0]; d[0] = obs_cvt<OT>(v.x); d[1] = obs_cvt<OT>(v.y); d[2] = obs_cvt<OT>(v.z); d[3] = obs_cvt<OT>(v.w); }
            if (w1) { const float4 v = fv[i][1]; d[160] = obs_cvt<OT>(v.x); d[161] = obs_cvt<OT>(v.y); d[162] = obs_cvt<OT>(v.z); d[163] = obs_cvt<OT>(v.w); }
        }
    }
    if (lane < na) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int w = warp + 8 * j;
            if (w < W) tile[(lane * W + w) * 5 + 4] = obs_cvt<OT>(rv[j]);
        }
    }
    fence_proxy_async_smem();
    __syncthreads();
    OT* __restrict__ dst = reinterpret_cast<OT*>(p.obs) + ((size_t)e * A + a0) * W * 5;
    const int n = na * W * 5;
    if (((((uintptr_t)dst) | ((size_t)n * sizeof(OT))) & 15) == 0) {
        if (tid == 0) { bulk_store_s2g(dst, tile, (uint32_t)n * (uint32_t)sizeof(OT), kPolicyEvictFirst); bulk_commit(); bulk_wait_read<0>(); }
    } else {
        for (int q = tid; q < n; q += kObsThreads) dst[q] = tile[q];
    }
}

__global__ void __launch_bounds__(kObsThreads) k_obs_build_rows_bf16(const StepParams p) { obs_build_rows<uint16_t>(p); }

}  // namespace pmrl

// ================================================================================================
// Host side: validation, tiling choice, launches.
// ================================================================================================
using namespace pmrl;

// Pick the asset-tile of the obs kernels: the biggest tile ≤ cap bytes whose start offsets stay
// 16-byte aligned (so the TMA bulk store applies) with the least ragged last tile.  esz: bytes per obs element.
static void choose_obs_tile(int A, int W, int F, size_t esz, size_t cap_bytes, const void* obs, StepParams& p) {
    const size_t per = (size_t)W * F * esz;
    int max_ta = (int)(cap_bytes / per);
    if (max_ta > A) max_ta = A;
    if (max_ta < 1) max_ta = 1;
    const bool env_aligned = (((size_t)A * W * F * esz) % 16 == 0) && (((uintptr_t)obs) % 16 == 0);
    int best = -1; long best_waste = 0;
    if (env_aligned) {
        for (int pass = 0; pass < 2 && best < 0; ++pass) {
            const int lo = pass == 0 ? (max_ta + 1) / 2 : 1;
            for (int ta = max_ta; ta >= lo; --ta) {
                if (((size_t)ta * W * F * esz) % 16 != 0 && ta < A) continue;
                const long tiles = (A + ta - 1) / ta;
                const long waste = tiles * ta - A;
                if (best < 0 || waste < best_waste) { best = ta; best_waste = waste; }
            }
        }
    }
    if (best > 0) { p.tile_assets = best; p.obs_bulk_ok = 1; }
    else { p.tile_assets = max_ta; p.obs_bulk_ok = 0; }
    p.tiles_per_env = (A + p.tile_assets - 1) / p.tile_assets;
}

static int fill_params(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st, StepParams& p) {
    if (!cfg || !st) return pmrl_fail(PMRL_E_ARG, "cfg/state is NULL");
    if (cfg->E < 0 || cfg->A < 1 || cfg->W < 1 || cfg->F < 1) return pmrl_fail(PMRL_E_SHAPE, "E>=0, A>=1, W>=1, F>=1 required");
    if (!st->value || !st->hist || !st->idx || !st->is_full || !st->t) return pmrl_fail(PMRL_E_ARG, "state pointer is NULL");
    memset(&p, 0, sizeof(p));
    p.E = cfg->E; p.A = cfg->A; p.W = cfg->W; p.F = cfg->F; p.T = cfg->T;
    p.episode_len = cfg->episode_len; p.reward_mode = cfg->reward_mode;
    p.mu_max_iter = cfg->mu_max_iter > 0 ? cfg->mu_max_iter : 16;
    p.flags = cfg->flags;
    p.initial_cash = cfg->initial_cash; p.commission = cfg->commission;
    p.reward_scale = cfg->reward_scale; p.risk_free = cfg->risk_free;
    const double c = (double)cfg->commission;
    p.mu0 = (float)(1.0 - 2.0 * c + c * c);
    p.c2 = (float)(2.0 * c - c * c);
    if (tbl) { p.y_tm = tbl->y_tm; p.feat_am = tbl->feat_am; p.feat_am4 = tbl->feat_am4; }
    p.value = st->value; p.hist = st->hist; p.idx = st->idx; p.is_full = st->is_full; p.t = st->t;
    p.t0 = st->t0; p.sharpe = st->sharpe; p.ep_return = st->ep_return;
    p.ticket = st->ticket;
    return 0;
}

// obs_mode as passed by the caller (PMRL_OBS_BF16 included); the rest of the library works with the base mode and a bf16 flag
static int check_obs_args(const StepParams& p, const float* obs, int obs_mode_arg) {
    if (int rc = pmrl_check_obs_mode(obs_mode_arg)) return rc;
    const int obs_mode = obs_mode_arg & ~PMRL_OBS_BF16;
    if (obs_mode == PMRL_OBS_NONE) return 0;
    if (!obs) return pmrl_fail(PMRL_E_ARG, "obs is NULL but obs_mode != NONE");
    if (p.F < 2 && obs_mode == PMRL_OBS_FULL) return pmrl_fail(PMRL_E_SHAPE, "F >= 2 required for a full obs");
    if (obs_mode == PMRL_OBS_FULL) {
        if (!p.feat_am) return pmrl_fail(PMRL_E_ARG, "feat_am is NULL but obs_mode == FULL");
        if (!p.t0) return pmrl_fail(PMRL_E_ARG, "t0 is NULL but obs_mode == FULL");
        if (p.F - 1 == 4 && ((uintptr_t)p.feat_am) % 16 != 0) return pmrl_fail(PMRL_E_ALIGN, "feat_am must be 16-byte aligned");
        if (p.T < p.W) return pmrl_fail(PMRL_E_SHAPE, "T < W");
        // the window rows are [t0 + k, t0 + k + W): without an episode length k grows without bound and would leave the table
        if (p.episode_len <= 0) return pmrl_fail(PMRL_E_SHAPE, "obs_mode FULL gathers from the feature table and needs episode_len > 0");
    }
    if ((size_t)p.W * p.F * 4 > kObsTileCapBytes) return pmrl_fail(PMRL_E_SHAPE, "W*F*4 exceeds the obs tile capacity");
    return 0;
}

// Launch-shape knobs (pmrl_set_tuning).
static int g_tune_group = 0, g_tune_ctas_per_sm = 0, g_tune_fused = 1, g_tune_fast = 1, g_tune_rt = 1;

// obs_mode: base mode (FULL / WEIGHTS); bf16: PMRL_OBS_BF16 was set (FULL only, checked by check_obs_args)
static int launch_obs(StepParams& p, float* obs, int obs_mode, bool bf16, cudaStream_t s) {
    p.obs = obs; p.obs_mode = obs_mode;
    const size_t esz = bf16 ? 2 : 4;
    if (obs_mode == PMRL_OBS_FULL && p.F == 5 && p.W <= 64 && p.t0 && g_tune_fast) {      // division-free tile kernel
        if (p.E == 0) return 0;
        p.tile_assets = 32;
        p.tiles_per_env = (p.A + 31) / 32;
        const long grid = (long)p.E * p.tiles_per_env;
        if (grid > 2147483647L) return pmrl_fail(PMRL_E_SHAPE, "E * tiles_per_env exceeds the grid limit");
        if (bf16) {
            k_obs_build_rows_bf16<<<(unsigned)grid, kObsThreads, (size_t)32 * p.W * 5 * esz, s>>>(p);
            return pmrl_check_launch("k_obs_build_rows_bf16");
        }
        k_obs_build_rows<<<(unsigned)grid, kObsThreads, (size_t)32 * p.W * 5 * 4, s>>>(p);
        return pmrl_check_launch("k_obs_build_rows");
    }
    choose_obs_tile(p.A, p.W, p.F, esz, kObsTileCapBytes, obs, p);
    if (p.E == 0) return 0;
    const size_t smem = (size_t)p.tile_assets * p.W * p.F * esz;
    const long grid = (long)p.E * p.tiles_per_env;
    if (grid > 2147483647L) return pmrl_fail(PMRL_E_SHAPE, "E * tiles_per_env exceeds the grid limit");
    if (bf16) {
        k_obs_build_bf16<<<(unsigned)grid, kObsThreads, smem, s>>>(p);
        return pmrl_check_launch("k_obs_build_bf16");
    }
    k_obs_build<<<(unsigned)grid, kObsThreads, smem, s>>>(p);
    return pmrl_check_launch("k_obs_build");
}

// (NPL, VEC) dispatch shared by the eager and the burst launchers: F is a generic lambda called with
// std::integral_constant<int, NPL>, <int, VEC>.
template <typename Fn>
static int dispatch_npl_vec(int npl, int vec, Fn&& f) {
#define PMRL_NV(N, V) if (npl == N && vec == V) return f(std::integral_constant<int, N>{}, std::integral_constant<int, V>{})
    PMRL_NV(1, 1); PMRL_NV(2, 1); PMRL_NV(2, 2); PMRL_NV(4, 1); PMRL_NV(4, 2); PMRL_NV(4, 4);
    PMRL_NV(8, 1); PMRL_NV(8, 4); PMRL_NV(16, 1); PMRL_NV(16, 4); PMRL_NV(32, 1); PMRL_NV(32, 4);
#undef PMRL_NV
    return pmrl_fail(PMRL_E_SHAPE, "unsupported (slots per lane, vector width)");
}

static int g_tune_staged = 1;

static int launch_step_s(const StepParams& p, int npl, int vec, cudaStream_t s) {
    if (g_tune_staged && npl >= 8 && (g_tune_staged == 2 || (p.E + kStepWarps - 1) / kStepWarps > pmrl_sm_count() * 2)) {
        // wide envs, more than one env per warp: rows staged one env ahead through shared memory (env_step_staged.cu)
        const int rc = pmrl_launch_step_staged(p, npl, vec, g_tune_ctas_per_sm, s);
        if (rc != -100) return rc;
    }
    const int want = (p.E + kStepWarps - 1) / kStepWarps;
    const int cap = pmrl_sm_count() * 8;
    const int grid = want < cap ? want : cap;
    const bool hasc = p.commission > 0.0f;
    return dispatch_npl_vec(npl, vec, [&](auto N, auto V) {
        constexpr int NPL = decltype(N)::value, VEC = decltype(V)::value;
        // TAIL: every group of 32·VEC asset slots but the last is full → only the last group carries validity guards
        const bool tail = env_tail_ok<NPL, VEC>(p.A);
        // (the pipelined form — large batches of narrow envs — has a variant without the per-env null tests of the PmrlStepIO sinks)
        const bool nosinks = !p.action_sink && !p.weight_sink && !p.value_sink && !p.index_sink && !p.reward_host;
        auto go = [&](auto H, auto P, auto T) {
            if constexpr (decltype(P)::value) {
                if (nosinks) {
                    k_env_step<NPL, decltype(H)::value, VEC, true, decltype(T)::value, true><<<grid, kStepThreads, 0, s>>>(p);
                    return pmrl_check_launch("k_env_step");
                }
            }
            k_env_step<NPL, decltype(H)::value, VEC, decltype(P)::value, decltype(T)::value><<<grid, kStepThreads, 0, s>>>(p);
            return pmrl_check_launch("k_env_step");
        };
        using Tr = std::true_type; using Fa = std::false_type;
        // 3-stage software pipeline over the envs of a warp while the registers allow it (narrow envs) and a warp has more
        // than one env; a batch that fits one wave runs the plain form at full occupancy
        if constexpr (NPL <= 4) {
            if (want > cap) {
                if (hasc) return tail ? go(Tr{}, Tr{}, Tr{}) : go(Tr{}, Tr{}, Fa{});
                return tail ? go(Fa{}, Tr{}, Tr{}) : go(Fa{}, Tr{}, Fa{});
            }
        }
        if (hasc) return tail ? go(Tr{}, Fa{}, Tr{}) : go(Tr{}, Fa{}, Fa{});
        return tail ? go(Fa{}, Fa{}, Tr{}) : go(Fa{}, Fa{}, Fa{});
    });
}

static int launch_step_burst(const StepParams& p, int npl, int vec, cudaStream_t s) {
    const int want = (p.E + kStepWarps - 1) / kStepWarps;
    const int cap = pmrl_sm_count() * 8;
    const int grid = want < cap ? want : cap;
    const bool hasc = p.commission > 0.0f;
    return dispatch_npl_vec(npl, vec, [&](auto N, auto V) {
        constexpr int NPL = decltype(N)::value, VEC = decltype(V)::value;
        const bool tail = env_tail_ok<NPL, VEC>(p.A);
        if (hasc) { if (tail) k_env_step_burst<NPL, true, VEC, true><<<grid, kStepThreads, 0, s>>>(p); else k_env_step_burst<NPL, true, VEC, false><<<grid, kStepThreads, 0, s>>>(p); }
        else      { if (tail) k_env_step_burst<NPL, false, VEC, true><<<grid, kStepThreads, 0, s>>>(p); else k_env_step_burst<NPL, false, VEC, false><<<grid, kStepThreads, 0, s>>>(p); }
        return pmrl_check_launch("k_env_step_burst");
    });
}

extern "C" int pmrl_set_tuning(int32_t key, int32_t value) {
    switch (key) {
        case PMRL_TUNE_GROUP_ENVS: g_tune_group = value; return 0;
        case PMRL_TUNE_CTAS_PER_SM: g_tune_ctas_per_sm = value; return 0;
        case PMRL_TUNE_FUSED: g_tune_fused = value; return 0;
        case PMRL_TUNE_FAST_FILL: g_tune_fast = value; return 0;
        case PMRL_TUNE_RING_TMA: g_tune_rt = value; return 0;
        case PMRL_TUNE_STAGED: g_tune_staged = value; return 0;
        case PMRL_TUNE_HOST_STREAM: pmrl_set_host_stream(value); return 0;
        case PMRL_TUNE_HOST_MIRROR: pmrl_set_host_mirror(value); return 0;
        default: return pmrl_fail(PMRL_E_ARG, "unknown tuning key");
    }
}

static int launch_fused(StepParams& p, float* obs, int npl, int vec, bool bf16, cudaStream_t s) {
    p.obs = obs; p.obs_mode = PMRL_OBS_FULL;
    if (!g_tune_fast) return -100;
    if (g_tune_rt) {                                  // ring rows through one TMA bulk load per env (env_step_rt.cu)
        p.prefetch_next = (g_tune_rt == 2) ? 0 : 1;
        const int rc = pmrl_launch_step_obs_rt(p, npl, vec, g_tune_group, g_tune_ctas_per_sm, bf16, s);
        if (rc != -100) return rc;
    }
    if (bf16) return -100;                            // no bf16 form of the register-staged kernel: its shapes take the two kernels
    // register-staged fill (env_step_fast.cu): F == 5, W <= 64, A <= 128 — the shapes RT's ring alignment excludes
    return pmrl_launch_step_obs_fast(p, npl, vec, g_tune_group, g_tune_ctas_per_sm, s);
    // -100: no fused kernel covers this shape (A > 128, F != 5, W > 64) → state-only step, then the obs tile kernel
}

extern "C" int pmrl_env_reset(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st,
                              const uint8_t* mask, float* obs, int32_t obs_mode, void* stream) {
    if (cfg && cfg->E == 0) return 0;                  // empty batch: nothing to do (state pointers may be NULL)
    StepParams p;
    if (int rc = fill_params(cfg, tbl, st, p)) return rc;
    if (int rc = check_obs_args(p, obs, obs_mode)) return rc;
    p.mask = mask;
    cudaStream_t s = (cudaStream_t)stream;
    const int want = (p.E + kStepWarps - 1) / kStepWarps;
    const int cap = pmrl_sm_count() * 8;
    k_env_reset<<<want < cap ? want : cap, kStepThreads, 0, s>>>(p);
    if (int rc = pmrl_check_launch("k_env_reset")) return rc;
    if (obs_mode != PMRL_OBS_NONE) return launch_obs(p, obs, obs_mode & ~PMRL_OBS_BF16, (obs_mode & PMRL_OBS_BF16) != 0, s);
    return 0;
}

// y_tm[t, a] = close_tm[t, a] / close_tm[t-1, a] (data/instrument.py:79), row 0 = 1: the IEEE division of the reference,
// done once per table instead of once per env-step.
__global__ void k_price_relatives(const float* __restrict__ close_tm, int T, int A, float* __restrict__ y_tm) {
    const size_t n = (size_t)T * A;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        y_tm[i] = (i < (size_t)A) ? 1.0f : __fdiv_rn(close_tm[i], close_tm[i - A]);
}

extern "C" int pmrl_price_relatives(const float* close_tm, int32_t T, int32_t A, float* y_tm, void* stream) {
    if (!close_tm || !y_tm) return pmrl_fail(PMRL_E_ARG, "price_relatives: null pointer");
    if (T < 1 || A < 1) return pmrl_fail(PMRL_E_SHAPE, "price_relatives: T >= 1, A >= 1 required");
    const size_t n = (size_t)T * A;
    const size_t want = (n + 255) / 256, cap = (size_t)pmrl_sm_count() * 16;
    k_price_relatives<<<(unsigned)(want < cap ? want : cap), 256, 0, (cudaStream_t)stream>>>(close_tm, T, A, y_tm);
    return pmrl_check_launch("k_price_relatives");
}

// Bit-for-bit comparison of the shared-reciprocal quotient (pmrl_device.cuh: unidiv) with IEEE division on caller-supplied
// operands: den[i / 32] divides num[i]; pairs outside the range the kernels accept are skipped and counted separately.
// Even i take the scalar form, odd i the packed (FMUL2 / FFMA2) form the step kernels use.
__global__ void k_selftest_division(const float* __restrict__ num, const float* __restrict__ den, long long n,
                                    unsigned long long* __restrict__ out /* [2]: mismatches, pairs tested */) {
    unsigned long long bad = 0, tested = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float a = num[i], b = den[i >> 5];
        if (!unidiv_in_range(b) || !(a == 0.0f || unidiv_in_range(a))) continue;
        const UniDiv d = unidiv_make(b);
        float q;
        if (i & 1) { float x[2] = {a, a}; lane_unidiv(x, d); q = x[1]; }
        else q = unidiv(a, d);
        const float ref = __fdiv_rn(a, b);
        ++tested;
        if (__float_as_uint(q) != __float_as_uint(ref)) ++bad;
    }
    if (bad) atomicAdd(out, bad);
    if (tested) atomicAdd(out + 1, tested);
}

extern "C" int pmrl_selftest_division(const float* num, const float* den, int64_t n, uint64_t* out, void* stream) {
    if (!num || !den || !out) return pmrl_fail(PMRL_E_ARG, "selftest_division: null pointer");
    if (n < 0) return pmrl_fail(PMRL_E_SHAPE, "selftest_division: n < 0");
    if (n == 0) return 0;
    k_selftest_division<<<pmrl_sm_count() * 8, 256, 0, (cudaStream_t)stream>>>(num, den, (long long)n, (unsigned long long*)out);
    return pmrl_check_launch("k_selftest_division");
}

extern "C" int pmrl_obs_build(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st,
                              float* obs, int32_t obs_mode, void* stream) {
    if (cfg && cfg->E == 0) return 0;                  // empty batch: nothing to do (state pointers may be NULL)
    StepParams p;
    if (int rc = fill_params(cfg, tbl, st, p)) return rc;
    if (obs_mode == PMRL_OBS_NONE) return pmrl_fail(PMRL_E_ARG, "obs_mode NONE makes no obs");
    if (int rc = check_obs_args(p, obs, obs_mode)) return rc;
    return launch_obs(p, obs, obs_mode & ~PMRL_OBS_BF16, (obs_mode & PMRL_OBS_BF16) != 0, (cudaStream_t)stream);
}

// validation shared by the step entry points; fills the per-step fields of p
static int prepare_step(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st, const PmrlStepIO* io, StepParams& p) {
    if (int rc = fill_params(cfg, tbl, st, p)) return rc;
    if (!io) return pmrl_fail(PMRL_E_ARG, "io is NULL");
    if (!io->actions || !io->reward || !io->done) return pmrl_fail(PMRL_E_ARG, "actions/reward/done is NULL");
    if (!io->y_ext) {
        if (!p.y_tm) return pmrl_fail(PMRL_E_ARG, "need y_tm (pmrl_price_relatives) or y_ext");
        if (!p.t0) return pmrl_fail(PMRL_E_ARG, "t0 is NULL but y comes from the price table");
        if (p.episode_len <= 0) return pmrl_fail(PMRL_E_SHAPE, "episode_len must be > 0 when y comes from the price table");
    }
    if (cfg->reward_mode < 0 || cfg->reward_mode > PMRL_REWARD_SHARPE) return pmrl_fail(PMRL_E_ARG, "bad reward_mode");
    if (cfg->reward_mode == PMRL_REWARD_SHARPE && !p.sharpe) return pmrl_fail(PMRL_E_ARG, "sharpe state is NULL");
    if (io->stats && !p.ep_return) return pmrl_fail(PMRL_E_ARG, "ep_return is NULL but stats requested");
    if ((io->reward_host == nullptr) != (io->done_host == nullptr)) return pmrl_fail(PMRL_E_ARG, "reward_host and done_host go together");
    if (io->index_sink && !p.t0) return pmrl_fail(PMRL_E_ARG, "index_sink needs t0");
    if (!env_npl_for(p.A)) return pmrl_fail(PMRL_E_SHAPE, "A > 1024 is not supported");
    p.actions = io->actions; p.y_ext = io->y_ext; p.reward = io->reward; p.done = io->done; p.stats = io->stats;
    p.action_sink = io->action_sink; p.value_sink = io->value_sink; p.index_sink = io->index_sink; p.weight_sink = io->weight_sink;
    p.reward_host = io->reward_host; p.done_host = io->done_host;
    if (io->actions_ready) {
        if (io->actions_ready_shift < 0 || io->actions_ready_shift > 30) return pmrl_fail(PMRL_E_ARG, "bad actions_ready_shift");
        p.act_ready = io->actions_ready; p.act_seq = io->actions_ready_seq; p.act_shift = io->actions_ready_shift;
    }
    return 0;
}

// 16-byte (VEC = 4) / 8-byte (VEC = 2) row accesses need every row base aligned: rows start at multiples of A floats
// from these bases, and A % VEC == 0 whenever VEC > 1.
static int vec_for_pointers(const StepParams& p, int npl) {
    int vec = env_vec_for(p.A, npl);
    uintptr_t m = (uintptr_t)p.actions | (uintptr_t)p.hist | (uintptr_t)p.action_sink | (uintptr_t)p.weight_sink;
    m |= p.y_ext ? (uintptr_t)p.y_ext : (uintptr_t)p.y_tm;
    while (vec > 1 && (m % (4u * vec)) != 0) vec = (vec == 4 && npl < 8 && p.A % 2 == 0) ? 2 : 1;
    return vec;
}

extern "C" int pmrl_env_step_io(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st,
                                const PmrlStepIO* io, void* stream) {
    if (cfg && cfg->E == 0) return 0;                  // empty batch: nothing to do (state pointers may be NULL)
    StepParams p;
    if (int rc = prepare_step(cfg, tbl, st, io, p)) return rc;
    float* obs = io->obs;
    if (int rc = check_obs_args(p, obs, io->obs_mode)) return rc;
    const int obs_mode = io->obs_mode & ~PMRL_OBS_BF16;
    const bool bf16 = (io->obs_mode & PMRL_OBS_BF16) != 0;
    const int npl = env_npl_for(p.A), vec = vec_for_pointers(p, npl);
    cudaStream_t s = (cudaStream_t)stream;
    if (obs_mode == PMRL_OBS_FULL && g_tune_fused && (size_t)p.W * p.F * 4 <= 36 * 1024) {
        const int rc = launch_fused(p, obs, npl, vec, bf16, s);
        if (rc != -100) return rc;                    // -100: no fused kernel for this shape → step kernel + obs kernel
    }
    if (int rc = launch_step_s(p, npl, vec, s)) return rc;
    if (obs_mode != PMRL_OBS_NONE) return launch_obs(p, obs, obs_mode, bf16, s);
    return 0;
}

extern "C" int pmrl_env_step(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st,
                             const float* actions, const float* y_ext,
                             float* reward, uint8_t* done, float* obs, int32_t obs_mode,
                             double* stats, void* stream) {
    PmrlStepIO io;
    memset(&io, 0, sizeof(io));
    io.actions = actions; io.y_ext = y_ext; io.reward = reward; io.done = done; io.obs = obs; io.obs_mode = obs_mode; io.stats = stats;
    return pmrl_env_step_io(cfg, tbl, st, &io, stream);
}

extern "C" int pmrl_env_step_burst(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st,
                                   const float* actions, int32_t K, float* reward, uint8_t* done,
                                   double* stats, void* stream) {
    if (cfg && cfg->E == 0) return 0;
    if (K < 1) return pmrl_fail(PMRL_E_SHAPE, "env_step_burst: K >= 1 required");
    PmrlStepIO io;
    memset(&io, 0, sizeof(io));
    io.actions = actions; io.reward = reward; io.done = done; io.stats = stats;
    StepParams p;
    if (int rc = prepare_step(cfg, tbl, st, &io, p)) return rc;
    p.burst = K;
    const int npl = env_npl_for(p.A), vec = vec_for_pointers(p, npl);
    if (g_tune_staged && npl >= 8 && (g_tune_staged == 2 || (p.E + kStepWarps - 1) / kStepWarps > pmrl_sm_count() * 2)) {
        // wide envs, large batches: the single-step kernel with its rows staged by TMA bulk copies is faster per step than
        // the register-resident burst (config 5: 0.335 vs 0.365 ms) and launch latency is negligible at this size, so the
        // burst is K of those launches enqueued here — the same arithmetic, bit-identical results
        p.burst = 0;
        const size_t EA = (size_t)p.E * p.A;
        for (int k = 0; k < K; ++k) {
            const int rc = pmrl_launch_step_staged(p, npl, vec, g_tune_ctas_per_sm, (cudaStream_t)stream);
            if (rc == -100) { if (k == 0) { p.burst = K; return launch_step_burst(p, npl, vec, (cudaStream_t)stream); } return pmrl_fail(PMRL_E_ARG, "env_step_burst: staged launch refused mid-burst"); }
            if (rc != 0) return rc;
            p.actions += EA; p.reward += p.E; p.done += p.E;
        }
        return 0;
    }
    return launch_step_burst(p, npl, vec, (cudaStream_t)stream);
}
