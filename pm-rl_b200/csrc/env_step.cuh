// env_step.cuh — one warp advances one environment by one step.
//
// Restates, batched and in registers, the reference transition
//   TradingEnv.step            env/sim/trading_env.py:54-100
//   ActionBuffer.update/get_last  env/sim/weight_buffer.py:13-30
//   Reward.*                   env/reward.py:15-31
//   y_t = close_t / close_{t-1}   data/instrument.py:79  (precomputed once per table: pmrl_price_relatives)
// keeping the reference association of every fp32 operation (no FMA contraction, IEEE div,
// expf/logf without fast-math) so values stay within 1e-5 relative over 1,000 compounding steps.
//
// Asset → register map.  A lane owns NPL asset slots in groups of VEC consecutive assets:
//     asset(lane, j) = ((j / VEC) * 32 + lane) * VEC + j % VEC
// so that with VEC = 4 (A % 4 == 0) every row access — raw action, price relatives, previous weights, the ring
// write — is ONE 16-byte instruction per group (VEC = 2: 8 bytes when A is even, VEC = 1: the lane-strided scalar
// map).  Every kernel that advances envs uses this one map (and env_vec_for / env_npl_for to choose it), so a
// given env shape runs the same operations in the same order whichever kernel steps it.
//
// The elementwise arithmetic runs on sm_100's packed fp32 pipe (FADD2 / FMUL2 / FFMA2: two IEEE-rn results per
// instruction, bit-identical to the scalar forms) and the 3-input FMNMX3; only expf stays scalar.
//
// The transition is split into three stages so that the state-only kernel can software-pipeline them
// across consecutive envs of a warp (scalars of env n+2, vectors of env n+1 and the arithmetic of env n
// are in flight together):
//   env_load_scalars   V, ring pointer, is_full, local step, episode offset
//   env_load_vectors   raw action, the price-relative row (or external y), previous weights (commission only)
//   env_compute_store  everything else
#pragma once
#include "pmrl_device.cuh"

namespace pmrl {

// Per-warp partial of the PMRL_STAT_* vector, held in registers TRANSPOSED over the lanes: lane q < 8 accumulates statistic q
// (one double), the two extrema are warp-uniform floats (a max of floats is exact).  Every value an env contributes is
// warp-uniform after the step, so adding it is a handful of non-divergent selects + one DADD per env — the former layout
// (10 doubles in shared memory, updated by lane 0 inside a divergent branch) cost ~100 issue slots per env.
struct WarpStats { double acc; float mx, mneg; };
__device__ __forceinline__ void wstats_init(WarpStats& s) { s.acc = 0.0; s.mx = -INFINITY; s.mneg = -INFINITY; }
__device__ __forceinline__ void wstats_add(WarpStats& s, int lane, float r, float Vn, int dn, float epr, int k_new) {
    const float fd = dn ? 1.0f : 0.0f;
    // Σ ln V is a monitoring statistic: the fast logarithm (lg2.approx, |err| < 4e-7 for V of order 1e4) — the reward's own
    // logf stays the accurate one
    float x = 1.0f;                                                    // PMRL_STAT_N_ENVS
    x = lane == PMRL_STAT_SUM_R ? r : x;
    x = lane == PMRL_STAT_SUM_R2 ? __fmul_rn(r, r) : x;
    x = lane == PMRL_STAT_SUM_V ? Vn : x;
    x = lane == PMRL_STAT_SUM_LNV ? __logf(Vn) : x;
    x = lane == PMRL_STAT_N_DONE ? fd : x;
    x = lane == PMRL_STAT_SUM_EPRET ? (dn ? epr : 0.0f) : x;
    x = lane == PMRL_STAT_SUM_EPLEN ? (dn ? (float)k_new : 0.0f) : x;
    s.acc += (double)x;
    s.mx = fmaxf(s.mx, Vn);
    s.mneg = fmaxf(s.mneg, -Vn);
}
// warp partial → its row of the block's shared staging array [warps][10]; then stats_flush_block
__device__ __forceinline__ void wstats_store(const WarpStats& s, double* __restrict__ sm_warp, int lane) {
    if (lane < PMRL_STAT_MAX_V) sm_warp[lane] = s.acc;
    else if (lane == PMRL_STAT_MAX_V) sm_warp[lane] = (double)s.mx;
    else if (lane == PMRL_STAT_MAX_NEGV) sm_warp[lane] = (double)s.mneg;
}

struct StepOut {       // warp-uniform result of one env transition
    int idx_new;       // ring pointer after the step
    int slot_written;  // ring row that received w' (or -1 on auto-reset)
    int is_full;
    int k;             // local step after the call
    int did_reset;
    float V, reward, epr;
    int done;
};

struct EnvScalars { float V, epr; int i, full, k, t0e; };   // epr: running episode return (only when p.ep_return)

template <int NPL, bool HASC, int VEC = 1>
struct EnvVectors {
    static_assert(NPL % VEC == 0, "NPL must be a multiple of VEC");
    float a[NPL];                   // raw action → weights → holdings → w'  (updated in place)
    float y[NPL];                   // price relative close_t / close_{t-1} (table row or external)
    float wl[HASC ? NPL : 1];       // previous post-drift weights (only read when commission > 0)
};

// Slots per lane / vector width for an env of A assets (host and device agree through these two functions).
__host__ __device__ constexpr int env_npl_for(int A) {
    return A <= 32 ? 1 : A <= 64 ? 2 : A <= 128 ? 4 : A <= 256 ? 8 : A <= 512 ? 16 : A <= 1024 ? 32 : 0;
}
__host__ __device__ constexpr int env_vec_for(int A, int npl) {
    if (npl >= 8) return (A % 4 == 0) ? 4 : 1;          // wide envs: 16-byte groups or the scalar map
    if (A % 4 == 0 && npl >= 4) return 4;
    if (A % 2 == 0 && npl >= 2) return 2;
    return 1;
}

template <int VEC>
__device__ __forceinline__ int asset_of(int lane, int j) { return ((j / VEC) * 32 + lane) * VEC + (j % VEC); }

// Is asset slot j of this lane a real asset?  With TAIL the caller guarantees that every group of 32·VEC assets but
// the last is full, so the test folds to `true` at compile time for all but the last group (all BASELINE shapes:
// A = 11, 50, 100, 500).  A % VEC == 0, so the slots of a group are valid together.
template <int NPL, int VEC, bool TAIL>
__device__ __forceinline__ bool slot_ok(int j, int lane, int A) {
    if (TAIL && j / VEC < NPL / VEC - 1) return true;
    return ((j / VEC) * 32 + lane) * VEC < A;
}
template <int NPL, int VEC>
__host__ __device__ constexpr bool env_tail_ok(int A) { return A > 32 * (NPL - VEC); }

// ---- VEC-wide row accesses ----
template <int VEC>
__device__ __forceinline__ void ld_once_v(const float* p, float* d) {        // read-once stream: no L1, evict-first in L2
    if constexpr (VEC == 4) {
        asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                     : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3]) : "l"(p), "l"(kPolicyEvictFirst));
    } else if constexpr (VEC == 2) {
        asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.f32 {%0,%1}, [%2], %3;"
                     : "=f"(d[0]), "=f"(d[1]) : "l"(p), "l"(kPolicyEvictFirst));
    } else {
        d[0] = ld_once(p, kPolicyEvictFirst);
    }
}
template <int VEC>
__device__ __forceinline__ void ld_keep_v(const float* p, float* d) {        // L2-resident table rows
    if constexpr (VEC == 4) {
        asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                     : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3]) : "l"(p), "l"(kPolicyEvictLast));
    } else if constexpr (VEC == 2) {
        asm volatile("ld.global.nc.L2::cache_hint.v2.f32 {%0,%1}, [%2], %3;"
                     : "=f"(d[0]), "=f"(d[1]) : "l"(p), "l"(kPolicyEvictLast));
    } else {
        d[0] = ld_keep(p, kPolicyEvictLast);
    }
}
template <int VEC>
__device__ __forceinline__ void ld_plain_v(const float* p, float* d) {       // ring rows (written by earlier launches)
    if constexpr (VEC == 4) { const float4 v = *reinterpret_cast<const float4*>(p); d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w; }
    else if constexpr (VEC == 2) { const float2 v = *reinterpret_cast<const float2*>(p); d[0] = v.x; d[1] = v.y; }
    else d[0] = *p;
}
template <int VEC>
__device__ __forceinline__ void lds_v(uint32_t saddr, float* d) {            // staged rows (env_step_staged.cu): ld.shared
    if constexpr (VEC == 4) asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3]) : "r"(saddr));
    else if constexpr (VEC == 2) asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(d[0]), "=f"(d[1]) : "r"(saddr));
    else asm volatile("ld.shared.f32 %0, [%1];" : "=f"(d[0]) : "r"(saddr));
}
template <int VEC>
__device__ __forceinline__ void st_v(float* p, const float* s) {
    if constexpr (VEC == 4) *reinterpret_cast<float4*>(p) = make_float4(s[0], s[1], s[2], s[3]);
    else if constexpr (VEC == 2) *reinterpret_cast<float2*>(p) = make_float2(s[0], s[1]);
    else *p = s[0];
}

// ---- packed fp32 helpers over a lane's NPL slots (pairs (j, j+1); NPL == 1 falls back to the scalar op) ----
__device__ __forceinline__ float min3_nan(float a, float b, float c) {       // NaN-propagating 3-input minimum (FMNMX3.NAN)
    float r;
    asm("min.NaN.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}
__device__ __forceinline__ float min3f(float a, float b, float c) {
    float r;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}
__device__ __forceinline__ float max3f(float a, float b, float c) {
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}
template <int N>
__device__ __forceinline__ float lane_sum(const float (&x)[N]) {             // Σ_j x[j] of this lane: pairwise tree on packed adds
    if constexpr (N == 1) return x[0];
    else if constexpr (N == 2) return __fadd_rn(x[0], x[1]);
    else {
        float t[N / 2];
#pragma unroll
        for (int j = 0; j < N / 2; j += 2) {                                 // (x[2j], x[2j+1]) + (x[2j+2], x[2j+3]), two sums per FADD2
            const float2 r = __fadd2_rn(make_float2(x[2 * j], x[2 * j + 1]), make_float2(x[2 * j + 2], x[2 * j + 3]));
            t[j] = r.x; t[j + 1] = r.y;
        }
        return lane_sum(t);
    }
}
// The two sums every value of the env is divided by — Σ exp(a) and V' = Σ port — carry their rounding error straight into
// the compounding portfolio value (V' = V·Σ w_i y_i·(1 − δ_Σe + δ_ΣV)), so they are accumulated in fp64 across the lanes
// (and within the lane while that is ≤ 4 conversions) and rounded to fp32 once: what is left against the reference is
// the reference's own summation error (SURVEY.md hard part 1: fp64-accumulate measured within 1e-5 over 1,000 steps).
template <int N>
__device__ __forceinline__ float env_sum_f64(const float (&x)[N]) {
    double d;
    if constexpr (N <= 4) {
        d = (double)x[0];
#pragma unroll
        for (int j = 1; j < N; ++j) d += (double)x[j];
    } else {
        d = (double)lane_sum(x);
    }
    return __double2float_rn(warp_sum(d));
}
template <int N>
__device__ __forceinline__ void lane_unidiv(float (&x)[N], const UniDiv& d) {  // x[j] /= b, shared reciprocal (see unidiv)
    if constexpr (N == 1) x[0] = unidiv(x[0], d);
    else {
        const float2 r2 = make_float2(d.r, d.r), nb2 = make_float2(d.nb, d.nb);
#pragma unroll
        for (int j = 0; j < N; j += 2) {
            const float2 a = make_float2(x[j], x[j + 1]);
            const float2 q0 = __fmul2_rn(a, r2);
            const float2 e = __ffma2_rn(nb2, q0, a);
            const float2 q = __ffma2_rn(r2, e, q0);
            x[j] = q.x; x[j + 1] = q.y;
        }
    }
}

// Zero the ring of env e and set the all-cash row (weight_buffer.py:46-50).
__device__ __forceinline__ void ring_reset_warp(float* __restrict__ hist_e, int W, int A, int lane) {
    const int n = W * A;
    for (int i = lane; i < n; i += 32) hist_e[i] = (i == 0) ? 1.0f : 0.0f;
}

__device__ __forceinline__ void env_load_scalars(const StepParams& p, int e, EnvScalars& s) {
    s.V = p.value[e];
    s.i = p.idx[e];
    s.full = p.is_full[e];
    s.k = p.t[e];
    s.t0e = p.t0 ? p.t0[e] : 0;
    s.epr = p.ep_return ? p.ep_return[e] : 0.0f;
}

__device__ __forceinline__ bool env_needs_reset(const StepParams& p, const EnvScalars& s) {
    return episode_due_reset(p.episode_len, s.k);                // train/on_policy.py:60-61
}

// Where the price relatives of the step after local step s.k live: the caller's [E, A] array or row t0 + k_new + W − 1 of the
// table (the last row of the new window).
__device__ __forceinline__ const float* env_y_row(const StepParams& p, int e, const EnvScalars& s) {
    return p.y_ext ? p.y_ext + (size_t)e * p.A : p.y_tm + (size_t)(s.t0e + s.k + p.W) * p.A;
}

// Streamed-in actions (PmrlStepIO.actions_ready): block until the chunk holding env e's row has landed in device memory.
// One lane polls the flag with a system-scope acquire load (the writer is the copy engine: flag after data in stream order).
__device__ __forceinline__ void env_wait_actions_lane(const StepParams& p, int e) {
    const uint32_t* f = p.act_ready + (e >> p.act_shift);
    for (uint32_t spin = 0;; ++spin) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
        if (v == p.act_seq) break;
        if (spin > (1u << 22)) __trap();                             // ≈ seconds: a protocol bug traps instead of hanging the GPU
        __nanosleep(128);
    }
}
__device__ __forceinline__ void env_wait_actions(const StepParams& p, int e, int lane) {
    if (p.act_ready) {
        if (lane == 0) env_wait_actions_lane(p, e);
        __syncwarp();
    }
}

// Raw action, price relatives and (commission only) previous weights of env e into a lane's slots.
// LOADWL = false: the caller supplies the previous weights itself (burst kernel: the w' it wrote one step earlier).
// LOADY = false: the price relatives are fetched inside env_compute_store, after the mu iteration (wide envs with
// commission: 16 fewer live registers through the iteration buy a third resident CTA per SM).
template <int NPL, bool HASC, int VEC, bool TAIL = false, bool LOADWL = true, bool LOADY = true>
__device__ __forceinline__ void env_load_rows(const StepParams& p, int e, int lane, const EnvScalars& s,
                                              float (&va)[NPL], float (&vy)[NPL], float (&vwl)[HASC ? NPL : 1]) {
    if (env_needs_reset(p, s)) return;                           // nothing is read on the auto-reset call
    env_wait_actions(p, e, lane);
    constexpr bool WL = HASC && LOADWL;
    const int A = p.A, W = p.W;
    const float* __restrict__ act = p.actions + (size_t)e * A;
    const float* __restrict__ wrow = p.hist;
    if (WL) wrow += ((size_t)e * W + (s.i == 0 ? W : s.i) - 1) * A;   // buffer[(idx - 1) % W], weight_buffer.py:30
    const bool ext = p.y_ext != nullptr;
    const float* __restrict__ yrow = env_y_row(p, e, s);
    // one validity test per group shared by the three loads (slots beyond A read as 0 everywhere)
#pragma unroll
    for (int g = 0; g < NPL / VEC; ++g) {
        const int a = (g * 32 + lane) * VEC;
        if (slot_ok<NPL, VEC, TAIL>(g * VEC, lane, A)) {
            ld_once_v<VEC>(act + a, &va[g * VEC]);
            if (LOADY) { if (ext) ld_once_v<VEC>(yrow + a, &vy[g * VEC]); else ld_keep_v<VEC>(yrow + a, &vy[g * VEC]); }
            if (WL) ld_plain_v<VEC>(wrow + a, &vwl[g * VEC]);
        } else {
#pragma unroll
            for (int c = 0; c < VEC; ++c) { va[g * VEC + c] = 0.0f; if (LOADY) vy[g * VEC + c] = 0.0f; if (WL) vwl[g * VEC + c] = 0.0f; }
        }
    }
}
template <int NPL, bool HASC, int VEC, bool TAIL = false>
__device__ __forceinline__ void env_load_vectors(const StepParams& p, int e, int lane, const EnvScalars& s,
                                                 EnvVectors<NPL, HASC, VEC>& v) {
    env_load_rows<NPL, HASC, VEC, TAIL>(p, e, lane, s, v.a, v.y, v.wl);
}

// Pull the DRAM-resident rows env e will read (its raw action, and its previous weights when commission > 0) into L2
// one env ahead of the warp, without holding registers for them: one 128-byte line per lane (A <= 1024: one pass).  The
// price-relative row lives in the L2-resident table already.
template <bool WL>
__device__ __forceinline__ void env_prefetch_vectors(const StepParams& p, int e, int lane, const EnvScalars& s) {
    if (env_needs_reset(p, s)) return;
    const int A = p.A, a = lane * 32;
    if (a < A) {
        prefetch_l2(p.actions + (size_t)e * A + a);
        if (WL) prefetch_l2(p.hist + ((size_t)e * p.W + (s.i == 0 ? p.W : s.i) - 1) * A + a);
    }
}

// One transition of env e on the rows in va / vy / vwl.  On return va[] holds w' (the post-drift weights, in the asset
// map above).  STORE_STATE = false leaves the scalar state (V, ring pointer, local step, episode return) in `out` only —
// the burst kernel writes it back once per burst; reward / done / the ring row / the sinks are always written.
struct NoHook { __device__ __forceinline__ void before_y() const {} __device__ __forceinline__ void after_y() const {} };

// WLS: the previous weights are not held in registers through the mu iteration but re-read from their staged shared-memory
// row (`wl_stage`) in every iteration (env_step_staged.cu, single-stage shape: 16 fewer live registers → more resident warps).
// `hook.before_y()` / `hook.after_y()` bracket the late read of the price relatives (LOADY = false) so the staging kernel
// can wait for / refill that row.
// YSTAGE: the late price-relative read always comes from `y_stage` (no runtime source test per group).  NOSINKS: the launcher
// has checked that no PmrlStepIO sink / host mirror is set, so their per-env null tests are compiled out.
template <int NPL, bool HASC, int VEC, bool TAIL = false, bool LOADY = true, bool STORE_STATE = true, bool WLS = false, typename Hook = NoHook,
          bool YSTAGE = false, bool NOSINKS = false>
__device__ __forceinline__ void env_compute_rows(const StepParams& p, int e, int lane, const EnvScalars& sc,
                                                 float (&va)[NPL], float (&vy)[NPL], float (&vwl)[(HASC && !WLS) ? NPL : 1],
                                                 StepOut& out, WarpStats& ws, uint32_t y_stage = 0u, uint32_t wl_stage = 0u,
                                                 const Hook& hook = Hook()) {
    const int A = p.A, W = p.W;
    float* __restrict__ hist_e = p.hist + (size_t)e * W * A;

    // ---- auto-reset instead of a step (train/on_policy.py:60-61) ----
    if (env_needs_reset(p, sc)) {
        ring_reset_warp(hist_e, W, A, lane);
        if (lane == 0) {
            p.value[e] = p.initial_cash;
            p.idx[e] = 1; p.is_full[e] = 0; p.t[e] = 0;
            p.reward[e] = 0.0f; p.done[e] = 0;
            if (p.reward_host) { p.reward_host[e] = 0.0f; p.done_host[e] = 0; }
            if (p.value_sink) p.value_sink[e] = p.initial_cash;
            if (p.index_sink) p.index_sink[e] = sc.t0e;
            if (p.sharpe) { p.sharpe[3 * (size_t)e] = 0.0; p.sharpe[3 * (size_t)e + 1] = 0.0; p.sharpe[3 * (size_t)e + 2] = 0.0; }
            if (p.ep_return) p.ep_return[e] = 0.0f;
        }
#pragma unroll
        for (int j = 0; j < NPL; ++j) va[j] = (asset_of<VEC>(lane, j) == 0) ? 1.0f : 0.0f;
        if (p.action_sink || p.weight_sink) {                    // the slot of a reset item holds the all-cash row (rollout_buffer.py:36)
#pragma unroll
            for (int g = 0; g < NPL / VEC; ++g)
                if (slot_ok<NPL, VEC, TAIL>(g * VEC, lane, A)) {
                    if (p.action_sink) st_v<VEC>(p.action_sink + (size_t)e * A + (g * 32 + lane) * VEC, &va[g * VEC]);
                    if (p.weight_sink) st_v<VEC>(p.weight_sink + (size_t)e * A + (g * 32 + lane) * VEC, &va[g * VEC]);
                }
        }
        out.idx_new = 1; out.slot_written = -1; out.is_full = 0; out.k = 0; out.did_reset = 1;
        out.V = p.initial_cash; out.reward = 0.0f; out.done = 0; out.epr = 0.0f;
        return;
    }

    float V = sc.V;
    const int i = sc.i;
    int full = sc.full;
    const int k_new = sc.k + 1;

    // the raw action row of a rollout / replay slot (replay/rollout_buffer.py:53, replay/buffer.py:35), written by the
    // kernel that read it instead of a separate copy
    if (!NOSINKS && p.action_sink) {
#pragma unroll
        for (int g = 0; g < NPL / VEC; ++g)
            if (slot_ok<NPL, VEC, TAIL>(g * VEC, lane, A)) st_v<VEC>(p.action_sink + (size_t)e * A + (g * 32 + lane) * VEC, &va[g * VEC]);
    }

    // ---- normalise (trading_env.py:58-60; quirks Q1-Q3) ----
    // slots beyond A hold 0: neutral for the sum, and for the minimum too, which is only ever compared with 0 (has_neg)
    // and with the −41 bound of the shared-reciprocal softmax below (a smaller minimum only makes that test stricter)
    float s = lane_sum(va), mn = INFINITY;
    if constexpr (NPL == 1) mn = nanmin(mn, va[0]);
    else {
#pragma unroll
        for (int j = 0; j < NPL; j += 2) mn = min3_nan(mn, va[j], va[j + 1]);
    }
    s = warp_sum(s);
    mn = warp_min_nan(mn);
    const bool strict = (p.flags & PMRL_FLAG_STRICT_REFERENCE) != 0;
    const bool not_close = !isclose_one(s);
    const bool has_neg = mn < 0.0f;
    const bool normalise = strict ? (not_close && has_neg) : (not_close || has_neg);
    if (normalise) {
        float mx = 0.0f;
        if (!strict) {                                           // stabilised softmax (agent/pg/pg.py:53)
            mx = -INFINITY;
#pragma unroll
            for (int j = 0; j < NPL; ++j) if (slot_ok<NPL, VEC, TAIL>(j, lane, A)) mx = fmaxf(mx, va[j]);
            mx = warp_max(mx);
#pragma unroll
            for (int j = 0; j < NPL; ++j) va[j] = __fsub_rn(va[j], mx);
        }
#pragma unroll
        for (int j = 0; j < NPL; ++j) {
            const float ex = expf(va[j]);
            va[j] = slot_ok<NPL, VEC, TAIL>(j, lane, A) ? ex : 0.0f;
        }
        const float se = env_sum_f64(va);
        // e_j / Σe over one divisor.  min_j e_j = exp(min_j a_j − mx) and max_j e_j ≤ Σe, so the shared-reciprocal form is
        // exact when the smallest raw score is above −41 (e^-41 > 2^-60) and Σe is in range; NaNs fail both tests.
        if (__fsub_rn(mn, mx) >= -41.0f && se >= kUniDivLo && se <= kUniDivHi) {
            lane_unidiv(va, unidiv_make(se));
        } else {
#pragma unroll
            for (int j = 0; j < NPL; ++j) va[j] = __fdiv_rn(va[j], se);
        }
    }

    // ---- transaction remainder factor mu (trading_env.py:67-75; upstream PGPortfolio relu form) ----
    const float V_prev = V;
    if (HASC) {
        const float c = p.commission;
        const float w0 = __shfl_sync(PMRL_FULL_MASK, va[0], 0);
        float wl0;
        if constexpr (WLS) { float t0[1]; lds_v<1>(wl_stage, t0); wl0 = t0[0]; }
        else wl0 = __shfl_sync(PMRL_FULL_MASK, vwl[0], 0);
        const float denom = __fsub_rn(1.0f, __fmul_rn(c, w0));
        const float cw = __fmul_rn(c, wl0);
        float mu_last = 1.0f, mu = p.mu0;
        int it = 0;
        // the sum runs over assets i >= 1: asset 0 (cash) is taken out by a hugely negative previous weight (its term is
        // relu(−1e30 − mu·w) = 0), the slots beyond A hold wl = w = 0 and contribute relu(0) = 0 — no per-slot guard
        // inside the iteration.  relu is evaluated as (d + |d|) / 2: d + |d| is 2d or 0 exactly and a sum of doubled
        // terms is the doubled sum bit for bit, so halving the total restores Σ relu(d) in the same rounding sequence
        // with two packed instructions per pair instead of two FMNMX and one packed add.
        if (!WLS && lane == 0) vwl[0] = -1e30f;
        while (fabsf(__fsub_rn(mu, mu_last)) > 1e-10f && it < p.mu_max_iter) {
            mu_last = mu;
            float part;
            if constexpr (WLS) {
                static_assert(!WLS || VEC == 4, "staged previous weights need the 16-byte asset map");
                const float2 mu2 = make_float2(mu, mu), neg1 = make_float2(-1.0f, -1.0f);
                float t[NPL];
#pragma unroll
                for (int g = 0; g < NPL / VEC; ++g) {
                    float w4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                    if (slot_ok<NPL, VEC, TAIL>(g * VEC, lane, A)) lds_v<4>(wl_stage + 16u * (uint32_t)(g * 32 + lane), w4);
                    if (g == 0 && lane == 0) w4[0] = -1e30f;
#pragma unroll
                    for (int h = 0; h < 4; h += 2) {
                        const int j = g * 4 + h;
                        const float2 m = __fmul2_rn(mu2, make_float2(va[j], va[j + 1]));
                        const float2 d = __ffma2_rn(m, neg1, make_float2(w4[h], w4[h + 1]));
                        const float2 r2 = __fadd2_rn(d, make_float2(fabsf(d.x), fabsf(d.y)));
                        t[j] = r2.x; t[j + 1] = r2.y;
                    }
                }
                part = __fmul_rn(lane_sum(t), 0.5f);
            } else if constexpr (NPL == 1) {
                part = fmaxf(__fsub_rn(vwl[0], __fmul_rn(mu, va[0])), 0.0f);
            } else {
                const float2 mu2 = make_float2(mu, mu), neg1 = make_float2(-1.0f, -1.0f);
                float t[NPL];
#pragma unroll
                for (int j = 0; j < NPL; j += 2) {
                    const float2 m = __fmul2_rn(mu2, make_float2(va[j], va[j + 1]));
                    const float2 d = __ffma2_rn(m, neg1, make_float2(vwl[j], vwl[j + 1]));    // wl − mu·w, both roundings kept
                    const float2 r2 = __fadd2_rn(d, make_float2(fabsf(d.x), fabsf(d.y)));
                    t[j] = r2.x; t[j + 1] = r2.y;
                }
                part = __fmul_rn(lane_sum(t), 0.5f);
            }
            part = warp_sum(part);
            const float numer = __fsub_rn(__fsub_rn(1.0f, cw), __fmul_rn(p.c2, part));
            mu = __fdiv_rn(numer, denom);
            ++it;
        }
        V = __fmul_rn(mu, V);                                    // trading_env.py:75
    }

    if constexpr (!LOADY) {                                      // price relatives fetched late (see env_load_rows)
        hook.before_y();
        const bool ext = !YSTAGE && p.y_ext != nullptr;
        const float* __restrict__ yrow = YSTAGE ? nullptr : env_y_row(p, e, sc);
#pragma unroll
        for (int g = 0; g < NPL / VEC; ++g) {
            const int a = (g * 32 + lane) * VEC;
            if (slot_ok<NPL, VEC, TAIL>(g * VEC, lane, A)) {
                if (YSTAGE) lds_v<VEC>(y_stage + 4u * (uint32_t)a, &vy[g * VEC]);         // row staged in shared memory by a bulk copy
                else if (ext) ld_once_v<VEC>(yrow + a, &vy[g * VEC]); else ld_keep_v<VEC>(yrow + a, &vy[g * VEC]);
            } else {
#pragma unroll
                for (int c = 0; c < VEC; ++c) vy[g * VEC + c] = 0.0f;
            }
        }
        hook.after_y();
    }

    // ---- value, drift, return (trading_env.py:78-90) ----
    float lo = INFINITY, hi = 0.0f;                          // range of |port_j| for the shared-reciprocal division
    if constexpr (NPL == 1) {
        va[0] = slot_ok<NPL, VEC, TAIL>(0, lane, A) ? __fmul_rn(V, __fmul_rn(va[0], vy[0])) : 0.0f;
        const float ap = slot_ok<NPL, VEC, TAIL>(0, lane, A) ? fabsf(va[0]) : 1.0f;
        lo = ap; hi = ap;
    } else {
        const float2 V2 = make_float2(V, V);
#pragma unroll
        for (int j = 0; j < NPL; j += 2) {
            const float2 pr = __fmul2_rn(V2, __fmul2_rn(make_float2(va[j], va[j + 1]), make_float2(vy[j], vy[j + 1])));
            const bool ok = slot_ok<NPL, VEC, TAIL>(j, lane, A);
            va[j] = ok ? pr.x : 0.0f; va[j + 1] = ok ? pr.y : 0.0f;
            const float a0 = ok ? fabsf(pr.x) : 1.0f, a1 = ok ? fabsf(pr.y) : 1.0f;
            lo = min3f(lo, a0, a1);
            hi = max3f(hi, a0, a1);
        }
    }
    const float Vn = env_sum_f64(va);
    // w' = port / V' (trading_env.py:83): one divisor for the whole env.  A zero, denormal, huge or NaN holding anywhere in
    // the env (fminf/fmaxf drop NaNs, so those are caught through V') sends the warp down the plain IEEE division.
    const bool uni = __all_sync(PMRL_FULL_MASK, lo >= kUniDivLo && hi <= kUniDivHi) && unidiv_in_range(Vn);
    if (uni) {
        lane_unidiv(va, unidiv_make(Vn));
    } else {
#pragma unroll
        for (int j = 0; j < NPL; ++j) va[j] = __fdiv_rn(va[j], Vn);
    }
    const float ret = __fdiv_rn(Vn, V);

    // ---- ring write (weight_buffer.py:21-26) ----
#pragma unroll
    for (int g = 0; g < NPL / VEC; ++g)
        if (slot_ok<NPL, VEC, TAIL>(g * VEC, lane, A)) {
            st_v<VEC>(hist_e + (size_t)i * A + (g * 32 + lane) * VEC, &va[g * VEC]);
            if (!NOSINKS && p.weight_sink) st_v<VEC>(p.weight_sink + (size_t)e * A + (g * 32 + lane) * VEC, &va[g * VEC]);   // un-wrapped history row
        }
    const int i_new = (i + 1 == W) ? 0 : i + 1;
    if (i_new == 0) full = 1;

    // ---- reward (trading_env.py:99; env/reward.py:15-31) ----
    float r;
    if (p.reward_mode == PMRL_REWARD_STEP_LOG) {
        r = __fmul_rn(logf(ret), p.reward_scale);
    } else if (p.reward_mode == PMRL_REWARD_RETURNS) {
        r = __fmul_rn(__fdiv_rn(Vn, V_prev), p.reward_scale);
    } else if (p.reward_mode == PMRL_REWARD_LOG_RETURNS) {
        r = __fmul_rn(logf(__fdiv_rn(Vn, V_prev)), p.reward_scale);
    } else {  // running Sharpe over the episode's value history, fp64 like numpy (reward.py:26-31)
        r = 0.0f;
        if (lane == 0) {
            double* sh = p.sharpe + 3 * (size_t)e;
            double n = sh[0], mean = sh[1], m2 = sh[2];
            const double g = (double)Vn / (double)V_prev;
            n += 1.0;
            const double d1 = g - mean;
            mean += d1 / n;
            m2 += d1 * (g - mean);
            sh[0] = n; sh[1] = mean; sh[2] = m2;
            const double sd = sqrt(m2 / (n - 1.0));              // ddof=1 → NaN at n == 1 (quirk Q11)
            r = (float)(((mean - (double)p.risk_free) / sd) * (double)p.reward_scale);
        }
        r = __shfl_sync(PMRL_FULL_MASK, r, 0);
    }

    const int dn = (p.episode_len > 0 && k_new == p.episode_len) ? 1 : 0;
    const float epr = __fadd_rn(sc.epr, r);
    if (lane == 0) {
        p.reward[e] = r; p.done[e] = (uint8_t)dn;
        if (!NOSINKS) {
            if (p.reward_host) { p.reward_host[e] = r; p.done_host[e] = (uint8_t)dn; }   // mapped pinned host memory: posted PCIe writes
            if (p.value_sink) p.value_sink[e] = Vn;              // RolloutBuffer.v[slot] (on_policy.py:65)
            if (p.index_sink) p.index_sink[e] = sc.t0e + k_new;  // loader item of this step (off_policy.py:87 → buffer.py:34)
        }
        if (STORE_STATE) {
            p.value[e] = Vn;
            p.idx[e] = i_new; p.is_full[e] = (uint8_t)full; p.t[e] = k_new;
            if (p.ep_return) p.ep_return[e] = epr;
        }
    }
    if (p.stats) wstats_add(ws, lane, r, Vn, dn, epr, k_new);
    out.idx_new = i_new; out.slot_written = i; out.is_full = full; out.k = k_new; out.did_reset = 0;
    out.V = Vn; out.reward = r; out.done = dn; out.epr = epr;
}
template <int NPL, bool HASC, int VEC, bool TAIL = false>
__device__ __forceinline__ void env_compute_store(const StepParams& p, int e, int lane, const EnvScalars& sc,
                                                  EnvVectors<NPL, HASC, VEC>& v, StepOut& out, WarpStats& ws) {
    env_compute_rows<NPL, HASC, VEC, TAIL>(p, e, lane, sc, v.a, v.y, v.wl, out, ws);
}

// The three stages back to back (fused kernel phase 1).
template <int NPL, bool HASC, int VEC>
__device__ __forceinline__ void env_step_warp(const StepParams& p, int e, int lane, EnvVectors<NPL, HASC, VEC>& v,
                                              StepOut& out, WarpStats& ws) {
    EnvScalars sc;
    env_load_scalars(p, e, sc);
    env_load_vectors<NPL, HASC, VEC>(p, e, lane, sc, v);
    env_compute_store<NPL, HASC, VEC>(p, e, lane, sc, v, out, ws);
}

// Block-level flush of the per-warp partials: thread q < 10 folds column q over the warps → 10 atomics per CTA.
__device__ __forceinline__ void stats_flush_block(double* __restrict__ stats, const double* sm /* [warps*10] */, int nwarps) {
    __syncthreads();
    if (threadIdx.x < PMRL_STATS_LEN) {
        const int q = threadIdx.x;
        double v = sm[q];
        for (int wi = 1; wi < nwarps; ++wi) {
            const double o = sm[wi * PMRL_STATS_LEN + q];
            v = (q >= PMRL_STAT_MAX_V) ? fmax(v, o) : v + o;
        }
        if (q >= PMRL_STAT_MAX_V) { if (v > -INFINITY) atomic_max_double(stats + q, v); }
        else if (v != 0.0) atomicAdd(stats + q, v);
    }
}

}  // namespace pmrl
