// eval_stream.cu — streaming per-env evaluation metrics (util/eval.py:14-37): the quantities k_eval_metrics computes from
// [E, N] value / [E, N, A] weight traces, accumulated in a fixed PMRL_EVAL_ACC_BYTES per env by one small kernel after
// every env call.  The two weight rows a step's turnover needs are still in the env's ring: after the step w'_t is row
// (idx-1) mod W and w'_{t-1} row (idx-2) mod W (W >= 2).
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "pmrl_b200.h"
#include "pmrl_device.cuh"
#include "host_util.h"

namespace pmrl {

// One env's accumulator.  All-zero = never started.  state: 0 never started, 1 running episode valid, 2 invalid (an
// update was missed) until the next reset.
struct __align__(16) EvalAcc {
    int32_t state;
    int32_t k_seen;          // the env's local step t at the last update
    double n, mean, m2;      // Welford over the excess simple returns of the running episode
    double dn;               // Σ min(r, 0)²
    double to;               // Σ_steps Σ_a |w'_t[a] − w'_{t-1}[a]|
    float v_prev, peak, mdd; // previous V, running max of V, running min of V / peak (starts at 1)
    int32_t ep_count;        // completed episodes
    float last[5];           // last completed episode: return, sharpe, sortino, mdd − 1, turnover
    int32_t pad;
    double sum[5];           // Σ over completed episodes of the five entries of `last`
};
static_assert(sizeof(EvalAcc) == PMRL_EVAL_ACC_BYTES, "PMRL_EVAL_ACC_BYTES must match the accumulator layout");
static_assert(PMRL_EVAL_ACC_BYTES == 8 * sizeof(uint4), "lanes 0-7 move one accumulator as eight 16-byte words");

constexpr int kEsThreads = 256;
constexpr int kEsWarps = kEsThreads / 32;

// sharpe, sortino, mdd − 1, turnover of the running episode: the expressions of k_eval_metrics (eval_metrics.cu:57-71)
__device__ __forceinline__ void acc_metrics(const EvalAcc& a, double ann, float* m) {
    const double n = a.n;
    const double sd = sqrt(a.m2 / (n - 1.0));                  // ddof = 1 → NaN at n == 1
    m[0] = n > 0.0 ? (float)(a.mean / sd * ann) : NAN;
    m[1] = n > 0.0 ? (float)(a.mean / sqrt(a.dn / n) * ann) : NAN;
    m[2] = a.mdd - 1.0f;
    m[3] = n > 0.0 ? (float)(a.to / n) : NAN;
}

// Σ_a |(double)w1[a] − (double)w0[a]| over the warp (every lane gets the sum).
template <bool V4>
__device__ __forceinline__ double turnover_rows(const float* __restrict__ w1, const float* __restrict__ w0, int A, int lane) {
    double s = 0.0;
    if constexpr (V4) {
        const float4* __restrict__ x4 = reinterpret_cast<const float4*>(w1);
        const float4* __restrict__ y4 = reinterpret_cast<const float4*>(w0);
#pragma unroll 2
        for (int j = lane; j < (A >> 2); j += 32) {
            const float4 x = ld_stream4(x4 + j), y = ld_stream4(y4 + j);
            s += fabs((double)x.x - (double)y.x);
            s += fabs((double)x.y - (double)y.y);
            s += fabs((double)x.z - (double)y.z);
            s += fabs((double)x.w - (double)y.w);
        }
    } else {
        for (int j = lane; j < A; j += 32) s += fabs((double)ld_stream(w1 + j) - (double)ld_stream(w0 + j));
    }
    return warp_sum(s);
}

// One warp per env (persistent grid): lanes 0-7 move the accumulator as eight 16-byte words through a per-warp shared
// copy, lane 0 applies the update rule, all lanes read the two ring rows when a step is to be added.
template <bool V4>
__global__ void __launch_bounds__(kEsThreads) k_eval_stream_update(int E, int A, int W, int episode_len,
                                                                   const float* __restrict__ value,
                                                                   const float* __restrict__ hist,
                                                                   const int32_t* __restrict__ idx,
                                                                   const int32_t* __restrict__ tstep,
                                                                   const float* __restrict__ ep_return,
                                                                   EvalAcc* __restrict__ acc, double rf_period, double ann) {
    __shared__ EvalAcc s_acc[kEsWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gw = blockIdx.x * kEsWarps + warp;
    const int nw = gridDim.x * kEsWarps;
    EvalAcc& a = s_acc[warp];
    uint4* const a_words = reinterpret_cast<uint4*>(&a);
    for (int e = gw; e < E; e += nw) {
        uint4* const g_words = reinterpret_cast<uint4*>(acc + e);
        if (lane < 8) a_words[lane] = g_words[lane];
        const int t = tstep[e], i = idx[e];
        const float V = value[e];
        __syncwarp();
        // 0: nothing to do, 1: restart at a reset, 2: add one step, 3: invalidate
        int act;
        if (t == 0) act = 1;
        else if (a.state != 1) act = 3;
        else if (t == a.k_seen) act = 0;
        else if (t == a.k_seen + 1 && i >= 0 && i < W) act = 2;
        else act = 3;
        double to = 0.0;
        if (act == 2) {
            const int r1 = i >= 1 ? i - 1 : i - 1 + W;             // w'_t
            const int r0 = r1 >= 1 ? r1 - 1 : r1 - 1 + W;          // w'_{t-1}
            const float* __restrict__ h = hist + (size_t)e * W * A;
            to = turnover_rows<V4>(h + (size_t)r1 * A, h + (size_t)r0 * A, A, lane);
        }
        if (lane == 0 && act != 0) {
            if (act == 1) {
                a.state = 1; a.k_seen = 0;
                a.n = 0.0; a.mean = 0.0; a.m2 = 0.0; a.dn = 0.0; a.to = 0.0;
                a.v_prev = V; a.peak = V; a.mdd = 1.0f;
            } else if (act == 3) {
                a.state = 2;
            } else {
                const double r = (double)V / (double)a.v_prev - 1.0 - rf_period;   // eval_metrics.cu:40
                a.n += 1.0;
                const double d = r - a.mean;
                a.mean += d / a.n;
                a.m2 += d * (r - a.mean);
                const double neg = r < 0.0 ? r : 0.0;
                a.dn += neg * neg;
                a.to += to;
                a.peak = fmaxf(a.peak, V);                         // the trace kernel's prefix max, then V / max
                a.mdd = fminf(a.mdd, V / a.peak);
                a.v_prev = V;
                a.k_seen = t;
                if (episode_len > 0 && t == episode_len) {         // the step that returned done = 1 (env_step.cuh:552)
                    float m[5];
                    m[0] = ep_return[e];
                    acc_metrics(a, ann, m + 1);
#pragma unroll
                    for (int j = 0; j < 5; ++j) { a.last[j] = m[j]; a.sum[j] += (double)m[j]; }
                    a.ep_count += 1;
                }
            }
        }
        __syncwarp();
        if (lane < 8 && act != 0) g_words[lane] = a_words[lane];
        __syncwarp();                                              // s_acc is refilled by the next env
    }
}

// One thread per env: accumulator → out [E, 5] (+ count).
__global__ void __launch_bounds__(kEsThreads) k_eval_stream_read(int E, const int32_t* __restrict__ tstep,
                                                                 const float* __restrict__ ep_return,
                                                                 const EvalAcc* __restrict__ acc, int which, double ann,
                                                                 float* __restrict__ out, int32_t* __restrict__ count) {
    for (int e = blockIdx.x * kEsThreads + threadIdx.x; e < E; e += gridDim.x * kEsThreads) {
        const EvalAcc a = acc[e];
        float m[5];
        if (which == PMRL_EVAL_RUNNING) {
            if (a.state == 1 && tstep[e] == a.k_seen) {
                m[0] = ep_return[e];
                acc_metrics(a, ann, m + 1);
            } else {
#pragma unroll
                for (int j = 0; j < 5; ++j) m[j] = NAN;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 5; ++j)
                m[j] = a.ep_count <= 0 ? NAN
                     : which == PMRL_EVAL_LAST_EPISODE ? a.last[j] : (float)(a.sum[j] / (double)a.ep_count);
        }
#pragma unroll
        for (int j = 0; j < 5; ++j) out[5 * (size_t)e + j] = m[j];
        if (count) count[e] = a.ep_count;
    }
}

}  // namespace pmrl

using namespace pmrl;

static int eval_stream_check(const PmrlEnvCfg* cfg, const PmrlEnvState* st, const void* acc, int32_t periods, const char* who) {
    if (!cfg || !st || !acc) return pmrl_fail(PMRL_E_ARG, who);
    if (!st->value || !st->hist || !st->idx || !st->t || !st->ep_return)
        return pmrl_fail(PMRL_E_ARG, "eval_stream: value, hist, idx, t and ep_return are required");
    if (cfg->E < 0 || cfg->A < 1 || cfg->A > 1024 || cfg->W < 2 || periods < 1)
        return pmrl_fail(PMRL_E_SHAPE, "eval_stream: need E >= 0, 1 <= A <= 1024, W >= 2, periods >= 1");
    if ((uintptr_t)acc % 16) return pmrl_fail(PMRL_E_ALIGN, "eval_stream: acc must be 16-byte aligned");
    return 0;
}

// resident blocks of a kernel per SM (queried once per kernel: callers keep it in a function-local static)
static int eval_stream_occupancy(const void* kernel) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kEsThreads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
    return per_sm;
}

// persistent grid: no more blocks than are resident at once (a second, partial wave would lengthen the per-warp env chain)
static int eval_stream_blocks(int E, int per_block, int per_sm) {
    const int blocks = (E + per_block - 1) / per_block;
    const int cap = pmrl_sm_count() * per_sm;
    return blocks < cap ? blocks : cap;
}

extern "C" int pmrl_eval_stream_update(const PmrlEnvCfg* cfg, const PmrlEnvState* st, void* acc, float rf, int32_t periods,
                                       void* stream) {
    if (int rc = eval_stream_check(cfg, st, acc, periods, "eval_stream_update: NULL cfg, state or acc")) return rc;
    const int E = cfg->E, A = cfg->A;
    if (E == 0) return 0;
    const double rf_period = pmrl_rf_period(rf, periods), ann = sqrt((double)periods);
    static const int occ_v4 = eval_stream_occupancy((const void*)k_eval_stream_update<true>);
    static const int occ_v1 = eval_stream_occupancy((const void*)k_eval_stream_update<false>);
    EvalAcc* const a = static_cast<EvalAcc*>(acc);
    const cudaStream_t s = (cudaStream_t)stream;
    if (A % 4 == 0 && (uintptr_t)st->hist % 16 == 0)
        k_eval_stream_update<true><<<eval_stream_blocks(E, kEsWarps, occ_v4), kEsThreads, 0, s>>>(
            E, A, cfg->W, cfg->episode_len, st->value, st->hist, st->idx, st->t, st->ep_return, a, rf_period, ann);
    else
        k_eval_stream_update<false><<<eval_stream_blocks(E, kEsWarps, occ_v1), kEsThreads, 0, s>>>(
            E, A, cfg->W, cfg->episode_len, st->value, st->hist, st->idx, st->t, st->ep_return, a, rf_period, ann);
    return pmrl_check_launch("k_eval_stream_update");
}

extern "C" int pmrl_eval_stream_read(const PmrlEnvCfg* cfg, const PmrlEnvState* st, const void* acc, int32_t which, float rf,
                                     int32_t periods, float* out, int32_t* count, void* stream) {
    (void)rf;
    if (int rc = eval_stream_check(cfg, st, acc, periods, "eval_stream_read: NULL cfg, state or acc")) return rc;
    if (!out) return pmrl_fail(PMRL_E_ARG, "eval_stream_read: NULL out");
    if (which != PMRL_EVAL_RUNNING && which != PMRL_EVAL_LAST_EPISODE && which != PMRL_EVAL_EPISODE_MEAN)
        return pmrl_fail(PMRL_E_ARG, "eval_stream_read: bad which");
    const int E = cfg->E;
    if (E == 0) return 0;
    static const int occ_read = eval_stream_occupancy((const void*)k_eval_stream_read);
    k_eval_stream_read<<<eval_stream_blocks(E, kEsThreads, occ_read), kEsThreads, 0, (cudaStream_t)stream>>>(
        E, st->t, st->ep_return, static_cast<const EvalAcc*>(acc), which, sqrt((double)periods), out, count);
    return pmrl_check_launch("k_eval_stream_read");
}
