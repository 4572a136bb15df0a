// eval_metrics.cu — per-env evaluation metrics on device (util/eval.py:14-37): Sharpe, Sortino, maximum
// drawdown and average turnover from the value / weight histories.  One warp per env.
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "pmrl_b200.h"
#include "pmrl_device.cuh"
#include "host_util.h"

namespace pmrl {

constexpr int kEvalThreads = 256;

__global__ void __launch_bounds__(kEvalThreads) k_eval_metrics(const float* __restrict__ values,
                                                               const float* __restrict__ weights,
                                                               int E, int N, int A, double rf_period, int periods,
                                                               float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int gw = (blockIdx.x * kEvalThreads + threadIdx.x) >> 5;
    const int nw = (gridDim.x * kEvalThreads) >> 5;
    for (int e = gw; e < E; e += nw) {
        const float* __restrict__ v = values + (size_t)e * N;
        const int n = N - 1;                                   // number of returns
        // pass 1: mean of excess returns, downside sum, drawdown (running max via warp scan + carry)
        double s = 0.0, dn = 0.0;
        float carry = -INFINITY, mdd = INFINITY;
        for (int base = 0; base < N; base += 32) {
            const int i = base + lane;
            const float vi = (i < N) ? v[i] : -INFINITY;
            float m = vi;                                      // inclusive prefix max over the 32 lanes
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const float up = __shfl_up_sync(PMRL_FULL_MASK, m, o);
                if (lane >= o) m = fmaxf(m, up);
            }
            m = fmaxf(m, carry);
            if (i < N) mdd = fminf(mdd, vi / m);
            carry = __shfl_sync(PMRL_FULL_MASK, m, 31);
            if (i >= 1 && i < N) {
                const double r = (double)vi / (double)v[i - 1] - 1.0 - rf_period;
                s += r;
                const double neg = r < 0.0 ? r : 0.0;
                dn += neg * neg;
            }
        }
        s = warp_sum(s); dn = warp_sum(dn);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mdd = fminf(mdd, __shfl_xor_sync(PMRL_FULL_MASK, mdd, o));
        const double mean = n > 0 ? s / n : NAN;
        // pass 2: sample variance (ddof = 1)
        double q = 0.0;
        for (int i = 1 + lane; i < N; i += 32) {
            const double r = (double)v[i] / (double)v[i - 1] - 1.0 - rf_period;
            q += (r - mean) * (r - mean);
        }
        q = warp_sum(q);
        const double sd = sqrt(q / (double)(n - 1));
        const double ann = sqrt((double)periods);
        // turnover
        double to = 0.0;
        if (weights) {
            const float* __restrict__ w = weights + (size_t)e * N * A;
            const size_t tot = (size_t)N * A;
            for (size_t k = (size_t)A + lane; k < tot; k += 32) to += fabs((double)w[k] - (double)w[k - A]);
            to = warp_sum(to);
        }
        if (lane == 0) {
            out[4 * (size_t)e + 0] = (float)(mean / sd * ann);
            out[4 * (size_t)e + 1] = (float)(mean / sqrt(dn / (double)n) * ann);
            out[4 * (size_t)e + 2] = mdd - 1.0f;
            out[4 * (size_t)e + 3] = weights ? (float)(to / (double)n) : NAN;
        }
    }
}

}  // namespace pmrl

using namespace pmrl;

extern "C" int pmrl_eval_metrics(const float* values, const float* weights, int32_t E, int32_t N, int32_t A,
                                 float rf, int32_t periods, float* out, void* stream) {
    if (!values || !out) return pmrl_fail(PMRL_E_ARG, "eval_metrics: NULL pointer");
    if (E < 0 || N < 2 || A < 1 || periods < 1) return pmrl_fail(PMRL_E_SHAPE, "eval_metrics: need N >= 2, A >= 1, periods >= 1");
    if (E == 0) return 0;
    const double rf_period = pmrl_rf_period(rf, periods);
    const int warps = kEvalThreads / 32;
    int blocks = (E + warps - 1) / warps;
    const int cap = pmrl_sm_count() * 8;
    if (blocks > cap) blocks = cap;
    k_eval_metrics<<<blocks, kEvalThreads, 0, (cudaStream_t)stream>>>(values, weights, E, N, A, rf_period, periods, out);
    return pmrl_check_launch("k_eval_metrics");
}
