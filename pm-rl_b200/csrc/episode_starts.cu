// episode_starts.cu — randomised episode starts: a fresh table offset t0[e] for every env about to be reset, drawn on the
// device so that it can run before each step (eagerly or inside a captured graph) without a host round trip.  The draw is
// a pure function of (seed, global env id, the env's draw count): Philox4x32-10 (Random123, Salmon et al. 2011) with the
// env's draw count as the first counter word.  The mapping to an offset is written down in include/pmrl_b200.h.
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "pmrl_b200.h"
#include "pmrl_device.cuh"
#include "host_util.h"

namespace pmrl {

constexpr int kDrawThreads = 256;

// Philox4x32-10: ten rounds of two 32x32→64 multiplies, the key bumped by the Weyl constants between rounds.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
    constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
        const uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += W0; k.y += W1;                                   // the bump after the last round is never used
    }
    return c;
}

struct StartDraw {
    int kind, lo, hi;
    uint64_t n;                                                 // hi - lo + 1
    uint2 key;
    uint64_t env_base;
    double log1m_beta, geo_norm;
};

// One thread per env (grid-stride): only the drawn envs touch episode[] and t0[].
__global__ void __launch_bounds__(kDrawThreads) k_env_draw_starts(int E, int episode_len, int mode, StartDraw d,
                                                                  const int32_t* __restrict__ t,
                                                                  const uint8_t* __restrict__ mask,
                                                                  int32_t* __restrict__ t0, uint32_t* __restrict__ episode) {
    for (int e = blockIdx.x * kDrawThreads + threadIdx.x; e < E; e += gridDim.x * kDrawThreads) {
        const bool draw = mode == PMRL_DRAW_DUE ? episode_due_reset(episode_len, t[e]) : (mask == nullptr || mask[e] != 0);
        if (!draw) continue;
        const uint32_t n_ep = episode[e];
        const uint64_t gid = d.env_base + (uint64_t)e;           // env_base + E <= INT64_MAX (checked on the host)
        const uint4 x = philox4x32_10(make_uint4(n_ep, (uint32_t)gid, (uint32_t)(gid >> 32), 0u), d.key);
        const uint64_t r64 = ((uint64_t)x.x << 32) | x.y;
        int32_t start;
        if (d.kind == PMRL_START_UNIFORM) {
            start = d.lo + (int32_t)__umul64hi(r64, d.n);
        } else {
            const double u = (double)(r64 >> 11) * 0x1p-53;
            const double q = floor(log1p(-u * d.geo_norm) / d.log1m_beta);
            const int64_t j = q < (double)(d.n - 1) ? (int64_t)q : (int64_t)(d.n - 1);
            start = d.hi - (int32_t)j;
        }
        t0[e] = start;
        episode[e] = n_ep + 1u;
    }
}

}  // namespace pmrl

using namespace pmrl;

extern "C" int pmrl_env_draw_starts(const PmrlEnvCfg* cfg, const PmrlStartDist* dist, const int32_t* t, const uint8_t* mask,
                                    int32_t mode, int32_t* t0, uint32_t* episode, void* stream) {
    if (!cfg || !dist || !t0 || !episode) return pmrl_fail(PMRL_E_ARG, "env_draw_starts: NULL cfg, dist, t0 or episode");
    if (mode != PMRL_DRAW_DUE && mode != PMRL_DRAW_MASK) return pmrl_fail(PMRL_E_ARG, "env_draw_starts: bad mode");
    if (mode == PMRL_DRAW_DUE && !t) return pmrl_fail(PMRL_E_ARG, "env_draw_starts: PMRL_DRAW_DUE reads t, which is NULL");
    if (dist->kind != PMRL_START_UNIFORM && dist->kind != PMRL_START_GEOMETRIC)
        return pmrl_fail(PMRL_E_ARG, "env_draw_starts: bad kind");
    if (dist->kind == PMRL_START_GEOMETRIC) {
        // beta in (0, 1) <=> log1p(-beta) finite and < 0; NaN fails both tests
        if (!(dist->log1m_beta < 0.0 && isfinite(dist->log1m_beta)))
            return pmrl_fail(PMRL_E_ARG, "env_draw_starts: geometric needs beta in (0, 1) (log1m_beta finite and < 0)");
        if (!(dist->geo_norm > 0.0 && dist->geo_norm <= 1.0))
            return pmrl_fail(PMRL_E_ARG, "env_draw_starts: geometric needs geo_norm in (0, 1]");
    }
    if (cfg->E < 0 || dist->lo < 0 || dist->hi < dist->lo || dist->env_base < 0 || dist->env_base > INT64_MAX - cfg->E)
        return pmrl_fail(PMRL_E_SHAPE, "env_draw_starts: need E >= 0, 0 <= lo <= hi, 0 <= env_base <= INT64_MAX - E");
    if (cfg->T > 0 && (int64_t)dist->hi + cfg->episode_len + cfg->W > cfg->T)
        return pmrl_fail(PMRL_E_SHAPE, "env_draw_starts: hi + episode_len + W > T (the episode would leave the tables)");
    const int E = cfg->E;
    if (E == 0) return 0;
    StartDraw d;
    d.kind = dist->kind; d.lo = dist->lo; d.hi = dist->hi;
    d.n = (uint64_t)((int64_t)dist->hi - dist->lo + 1);
    d.key = make_uint2((uint32_t)dist->seed, (uint32_t)(dist->seed >> 32));
    d.env_base = (uint64_t)dist->env_base;
    d.log1m_beta = dist->log1m_beta; d.geo_norm = dist->geo_norm;
    int blocks = (E + kDrawThreads - 1) / kDrawThreads;
    const int cap = pmrl_sm_count() * 8;
    if (blocks > cap) blocks = cap;
    k_env_draw_starts<<<blocks, kDrawThreads, 0, (cudaStream_t)stream>>>(E, cfg->episode_len, mode, d, t, mask, t0, episode);
    return pmrl_check_launch("k_env_draw_starts");
}
