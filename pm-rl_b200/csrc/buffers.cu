// buffers.cu — device-resident rollout / replay storage in the reference layouts.
//
//   pmrl_rollout_add / _gather   RolloutBuffer.add / sample / sample_random   replay/rollout_buffer.py:43-142
//   pmrl_replay_add / _gather    ReplayBuffer.add / sample                    replay/buffer.py:23-79,
//                                                                             replay/traj_buffer.py:26-89
// The off-policy buffer is an *index* replay (it stores (i, a, r) and regenerates the windows on
// sample, buffer.py:65-70); the gather re-uses the obs-tile builder of the step kernel.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include "pmrl_b200.h"
#include "pmrl_device.cuh"
#include "obs_tile.cuh"
#include "host_util.h"

namespace pmrl {

constexpr int kCopyThreads = 256;

// contiguous fp32 copy by the whole CTA (float4 when both ends are 16-byte aligned)
__device__ __forceinline__ void cta_copy_f32(float* __restrict__ dst, const float* __restrict__ src, size_t n,
                                             int tid, int nthreads) {
    if ((((uintptr_t)dst | (uintptr_t)src) & 15) == 0) {
        const size_t n4 = n >> 2;
        const float4* __restrict__ s4 = reinterpret_cast<const float4*>(src);
        float4* __restrict__ d4 = reinterpret_cast<float4*>(dst);
        for (size_t q = tid; q < n4; q += nthreads) d4[q] = s4[q];
        for (size_t q = (n4 << 2) + tid; q < n; q += nthreads) dst[q] = src[q];
    } else {
        for (size_t q = tid; q < n; q += nthreads) dst[q] = src[q];
    }
}

// the same for bf16 bit patterns (uint4 = 8 elements when both ends are 16-byte aligned)
__device__ __forceinline__ void cta_copy_u16(uint16_t* __restrict__ dst, const uint16_t* __restrict__ src, size_t n,
                                             int tid, int nthreads) {
    if ((((uintptr_t)dst | (uintptr_t)src) & 15) == 0) {
        const size_t n8 = n >> 3;
        const uint4* __restrict__ s8 = reinterpret_cast<const uint4*>(src);
        uint4* __restrict__ d8 = reinterpret_cast<uint4*>(dst);
        for (size_t q = tid; q < n8; q += nthreads) d8[q] = s8[q];
        for (size_t q = (n8 << 3) + tid; q < n; q += nthreads) dst[q] = src[q];
    } else {
        for (size_t q = tid; q < n; q += nthreads) dst[q] = src[q];
    }
}

// grid-stride contiguous copy (whole grid)
__global__ void __launch_bounds__(kCopyThreads) k_copy_f32(float* __restrict__ dst, const float* __restrict__ src, size_t n) {
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (size_t)gridDim.x * blockDim.x;
    if ((((uintptr_t)dst | (uintptr_t)src) & 15) == 0) {
        const size_t n4 = n >> 2;
        const float4* __restrict__ s4 = reinterpret_cast<const float4*>(src);
        float4* __restrict__ d4 = reinterpret_cast<float4*>(dst);
        for (size_t q = tid; q < n4; q += nt) d4[q] = ld_stream4(s4 + q);
        for (size_t q = (n4 << 2) + tid; q < n; q += nt) dst[q] = src[q];
    } else {
        for (size_t q = tid; q < n; q += nt) dst[q] = src[q];
    }
}
__global__ void k_copy_i32(int32_t* __restrict__ dst, const int32_t* __restrict__ src, size_t n) {
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (size_t)gridDim.x * blockDim.x;
    for (size_t q = tid; q < n; q += nt) dst[q] = src[q];
}

// One CTA per (sample b, chunk): gathers the six tensors of a RolloutBuffer minibatch (rollout_buffer.py:125-140).
// OT: element type of s / s_out (float, or uint16_t bf16 bits: the pointers below then hold uint16_t).
struct RolloutGatherParams {
    int S, E, A, W, F, B;
    const int32_t* slots; const int32_t* envs;
    const float *s, *a, *v, *r, *y;
    float *s_out, *a_out, *r_out, *pv_out, *pa_out, *p_out;
};
__global__ void __launch_bounds__(kCopyThreads) k_rollout_gather(const RolloutGatherParams g) {
    const int b = blockIdx.x, chunk = blockIdx.y, nchunks = gridDim.y;
    const int slot = g.slots[b], env = g.envs[b];
    const size_t row = (size_t)g.A * g.W * g.F;
    const size_t se = (size_t)slot * g.E + env;
    // obs row split across the chunks of this sample
    const size_t per = ((row + nchunks - 1) / nchunks + 3) & ~(size_t)3;
    const size_t lo = (size_t)chunk * per;
    if (lo < row) {
        const size_t n = (row - lo < per) ? row - lo : per;
        cta_copy_f32(g.s_out + (size_t)b * row + lo, g.s + se * row + lo, n, threadIdx.x, kCopyThreads);
    }
    if (chunk == 0) {
        const size_t sp = (size_t)(slot - 1) * g.E + env;             // idx-1 (rollout_buffer.py:130-131)
        for (int q = threadIdx.x; q < g.A; q += kCopyThreads) {
            g.a_out[(size_t)b * g.A + q] = g.a[se * g.A + q];
            g.pa_out[(size_t)b * g.A + q] = g.a[sp * g.A + q];
            g.p_out[(size_t)b * g.A + q] = g.y[se * g.A + q];
        }
        if (threadIdx.x == 0) { g.r_out[b] = g.r[se]; g.pv_out[b] = g.v[sp]; }
    }
}
// k_rollout_gather with the obs in element type OT (instantiated for bf16 bits: k_rollout_gather_bf16; the fp32 kernel above keeps
// its own code, whose SASS the template would reorder).
template <typename OT>
__device__ __forceinline__ void rollout_gather(const RolloutGatherParams& g) {
    const int b = blockIdx.x, chunk = blockIdx.y, nchunks = gridDim.y;
    const int slot = g.slots[b], env = g.envs[b];
    const size_t row = (size_t)g.A * g.W * g.F;
    const size_t se = (size_t)slot * g.E + env;
    // obs row split across the chunks of this sample (chunk starts stay 16-byte aligned)
    constexpr size_t kVec = 16 / sizeof(OT);
    const size_t per = ((row + nchunks - 1) / nchunks + (kVec - 1)) & ~(kVec - 1);
    const size_t lo = (size_t)chunk * per;
    if (lo < row) {
        const size_t n = (row - lo < per) ? row - lo : per;
        if constexpr (sizeof(OT) == 4) cta_copy_f32(g.s_out + (size_t)b * row + lo, g.s + se * row + lo, n, threadIdx.x, kCopyThreads);
        else cta_copy_u16(reinterpret_cast<uint16_t*>(g.s_out) + (size_t)b * row + lo,
                          reinterpret_cast<const uint16_t*>(g.s) + se * row + lo, n, threadIdx.x, kCopyThreads);
    }
    if (chunk == 0) {
        const size_t sp = (size_t)(slot - 1) * g.E + env;             // idx-1 (rollout_buffer.py:130-131)
        for (int q = threadIdx.x; q < g.A; q += kCopyThreads) {
            g.a_out[(size_t)b * g.A + q] = g.a[se * g.A + q];
            g.pa_out[(size_t)b * g.A + q] = g.a[sp * g.A + q];
            g.p_out[(size_t)b * g.A + q] = g.y[se * g.A + q];
        }
        if (threadIdx.x == 0) { g.r_out[b] = g.r[se]; g.pv_out[b] = g.v[sp]; }
    }
}
__global__ void __launch_bounds__(kCopyThreads) k_rollout_gather_bf16(const RolloutGatherParams g) { rollout_gather<uint16_t>(g); }

// One CTA per (sample b, asset-tile, which ∈ {s, s'}): window from the feature table by stored index,
// action history spliced into the last channel (buffer.py:58-77).
struct ReplayGatherParams {
    StepParams p;                 // A, W, F, T, feat_am, tile_assets, tiles_per_env, obs_bulk_ok are used
    int P, L, E, B;
    const int32_t *epochs, *envs, *starts;
    const int32_t* bi; const float *ba, *br;
    float *s_out, *a_out, *r_out, *s2_out;
};
__global__ void __launch_bounds__(kCopyThreads) k_replay_gather(const ReplayGatherParams g) {
    extern __shared__ __align__(128) float tile[];
    StepParams p = g.p;
    const int b = blockIdx.x, ti = blockIdx.y, which = blockIdx.z;   // which: 0 → s, 1 → s'
    const int A = p.A, W = p.W, F = p.F;
    const int ep = g.epochs[b], env = g.envs[b], start = g.starts[b];
    const int end = start + W;
    const int tid = threadIdx.x;
    const size_t le = (size_t)ep * g.L;
    const int i = g.bi[(le + end - 1) * g.E + env];                   // stored loader index (buffer.py:65)
    const int a0 = ti * p.tile_assets;
    const int na = min(p.tile_assets, A - a0);
    obs_tile_fill_features(p, tile, a0, na, i + which, tid, kCopyThreads);
    // channel F-1 ← a_hist[:, which : which+W]ᵀ  (buffer.py:69-70); asset fastest → coalesced action rows
    const int n = W * na;
    for (int q = tid; q < n; q += kCopyThreads) {
        const int w = q / na, al = q - w * na;
        tile[(al * W + w) * F + (F - 1)] = g.ba[((le + start + which + w) * g.E + env) * A + a0 + al];
    }
    fence_proxy_async_smem();
    __syncthreads();
    p.obs = which ? g.s2_out : g.s_out;
    p.obs_mode = PMRL_OBS_FULL;
    obs_tile_store(p, tile, b, a0, na, tid, kCopyThreads);
    if (which == 0 && ti == 0) {
        for (int q = tid; q < A; q += kCopyThreads)
            g.a_out[(size_t)b * A + q] = g.ba[((le + end) * g.E + env) * A + q];      // a[:, -1] (buffer.py:72)
        if (tid == 0) g.r_out[b] = g.br[(le + end - 1) * g.E + env];                 // buffer.py:60
    }
    if (p.obs_bulk_ok && tid == 0) bulk_wait_read<0>();
}
// k_replay_gather with the obs in element type OT (instantiated for bf16 bits: k_replay_gather_bf16; the fp32 kernel above keeps
// its own code, whose SASS the template would reorder).
template <typename OT>
__device__ __forceinline__ void replay_gather(const ReplayGatherParams& g) {
    extern __shared__ __align__(128) unsigned char smem_tile[];
    OT* const tile = reinterpret_cast<OT*>(smem_tile);
    StepParams p = g.p;
    const int b = blockIdx.x, ti = blockIdx.y, which = blockIdx.z;   // which: 0 → s, 1 → s'
    const int A = p.A, W = p.W, F = p.F;
    const int ep = g.epochs[b], env = g.envs[b], start = g.starts[b];
    const int end = start + W;
    const int tid = threadIdx.x;
    const size_t le = (size_t)ep * g.L;
    const int i = g.bi[(le + end - 1) * g.E + env];                   // stored loader index (buffer.py:65)
    const int a0 = ti * p.tile_assets;
    const int na = min(p.tile_assets, A - a0);
    obs_tile_fill_features(p, tile, a0, na, i + which, tid, kCopyThreads);
    // channel F-1 ← a_hist[:, which : which+W]ᵀ  (buffer.py:69-70); asset fastest → coalesced action rows
    const int n = W * na;
    for (int q = tid; q < n; q += kCopyThreads) {
        const int w = q / na, al = q - w * na;
        tile[(al * W + w) * F + (F - 1)] = obs_cvt<OT>(g.ba[((le + start + which + w) * g.E + env) * A + a0 + al]);
    }
    fence_proxy_async_smem();
    __syncthreads();
    p.obs = which ? g.s2_out : g.s_out;
    p.obs_mode = PMRL_OBS_FULL;
    obs_tile_store(p, tile, b, a0, na, tid, kCopyThreads);
    if (which == 0 && ti == 0) {
        for (int q = tid; q < A; q += kCopyThreads)
            g.a_out[(size_t)b * A + q] = g.ba[((le + end) * g.E + env) * A + q];      // a[:, -1] (buffer.py:72)
        if (tid == 0) g.r_out[b] = g.br[(le + end - 1) * g.E + env];                 // buffer.py:60
    }
    if (p.obs_bulk_ok && tid == 0) bulk_wait_read<0>();
}
__global__ void __launch_bounds__(kCopyThreads) k_replay_gather_bf16(const ReplayGatherParams g) { replay_gather<uint16_t>(g); }

// Index-mode rollout gather: the buffer keeps (loader index, raw action, value, reward) per slot plus the un-wrapped history of
// post-drift weights, and the observation s[slot] is REGENERATED here — feature window by index from the device table, weight
// channel from the history with ActionBuffer.get_all's ring order (weight_buffer.py:38-39; stored slots always have a full
// ring: slot >= 1 ↔ step n >= W) — exactly like the off-policy buffer regenerates its windows (replay/buffer.py:58-77).
// 8·A + 12 bytes per env-step instead of 4·A·W·F.
struct RolloutIndexGatherParams {
    StepParams p;                 // A, W, F, T, feat_am, tile_assets, tiles_per_env, obs_bulk_ok are used
    int S, E, B, off;             // off = W - 1: step number of a slot = slot + off (rollout_buffer.py:51-57)
    const int32_t *slots, *envs;
    const int32_t* bi;            // [S, E] loader item index t0 + n of the step stored in the slot
    const float *a, *v, *r;       // [S, E, A], [S, E], [S, E]
    const float* wp;              // [S + off, E, A] w' after step m (row 0 = all-cash)
    const float* y_tm;            // [T, A]
    float *s_out, *a_out, *r_out, *pv_out, *pa_out, *p_out;
};
__global__ void __launch_bounds__(kCopyThreads) k_rollout_gather_index(const RolloutIndexGatherParams g) {
    extern __shared__ __align__(128) float tile[];
    StepParams p = g.p;
    const int b = blockIdx.x, ti = blockIdx.y;
    const int A = p.A, W = p.W, F = p.F;
    const int slot = g.slots[b], env = g.envs[b];
    const int tid = threadIdx.x;
    const size_t se = (size_t)slot * g.E + env;
    const int i = g.bi[se];                                           // loader item of the step; the obs BEFORE it is item i - 1
    const int t = slot + g.off - 1;                                   // steps taken when that obs was made (>= W - 1: ring full)
    const int a0 = ti * p.tile_assets;
    const int na = min(p.tile_assets, A - a0);
    obs_tile_fill_features(p, tile, a0, na, i - 1, tid, kCopyThreads);
    const int n = W * na;
    for (int q = tid; q < n; q += kCopyThreads) {
        const int w = q / na, al = q - w * na;                        // asset fastest → coalesced history rows
        int d = (t - w) % W;                                          // column w shows ring slot w = newest step m <= t with m ≡ w (mod W)
        const int m = t - d;
        tile[(al * W + w) * F + (F - 1)] = g.wp[((size_t)m * g.E + env) * A + a0 + al];
    }
    fence_proxy_async_smem();
    __syncthreads();
    p.obs = g.s_out;
    p.obs_mode = PMRL_OBS_FULL;
    obs_tile_store(p, tile, b, a0, na, tid, kCopyThreads);
    if (ti == 0) {
        const size_t sp = (size_t)(slot - 1) * g.E + env;             // idx-1 (rollout_buffer.py:130-131)
        const float* __restrict__ yrow = g.y_tm + (size_t)(i + W - 1) * A;   // prices[idx]: the price relatives the step saw
        for (int q = tid; q < A; q += kCopyThreads) {
            g.a_out[(size_t)b * A + q] = g.a[se * A + q];
            g.pa_out[(size_t)b * A + q] = g.a[sp * A + q];
            g.p_out[(size_t)b * A + q] = yrow[q];
        }
        if (tid == 0) { g.r_out[b] = g.r[se]; g.pv_out[b] = g.v[sp]; }
    }
    if (p.obs_bulk_ok && tid == 0) bulk_wait_read<0>();
}
// k_rollout_gather_index with the obs in element type OT (instantiated for bf16 bits: k_rollout_gather_index_bf16; the fp32 kernel above keeps
// its own code, whose SASS the template would reorder).
template <typename OT>
__device__ __forceinline__ void rollout_gather_index(const RolloutIndexGatherParams& g) {
    extern __shared__ __align__(128) unsigned char smem_tile[];
    OT* const tile = reinterpret_cast<OT*>(smem_tile);
    StepParams p = g.p;
    const int b = blockIdx.x, ti = blockIdx.y;
    const int A = p.A, W = p.W, F = p.F;
    const int slot = g.slots[b], env = g.envs[b];
    const int tid = threadIdx.x;
    const size_t se = (size_t)slot * g.E + env;
    const int i = g.bi[se];                                           // loader item of the step; the obs BEFORE it is item i - 1
    const int t = slot + g.off - 1;                                   // steps taken when that obs was made (>= W - 1: ring full)
    const int a0 = ti * p.tile_assets;
    const int na = min(p.tile_assets, A - a0);
    obs_tile_fill_features(p, tile, a0, na, i - 1, tid, kCopyThreads);
    const int n = W * na;
    for (int q = tid; q < n; q += kCopyThreads) {
        const int w = q / na, al = q - w * na;                        // asset fastest → coalesced history rows
        int d = (t - w) % W;                                          // column w shows ring slot w = newest step m <= t with m ≡ w (mod W)
        const int m = t - d;
        tile[(al * W + w) * F + (F - 1)] = obs_cvt<OT>(g.wp[((size_t)m * g.E + env) * A + a0 + al]);
    }
    fence_proxy_async_smem();
    __syncthreads();
    p.obs = g.s_out;
    p.obs_mode = PMRL_OBS_FULL;
    obs_tile_store(p, tile, b, a0, na, tid, kCopyThreads);
    if (ti == 0) {
        const size_t sp = (size_t)(slot - 1) * g.E + env;             // idx-1 (rollout_buffer.py:130-131)
        const float* __restrict__ yrow = g.y_tm + (size_t)(i + W - 1) * A;   // prices[idx]: the price relatives the step saw
        for (int q = tid; q < A; q += kCopyThreads) {
            g.a_out[(size_t)b * A + q] = g.a[se * A + q];
            g.pa_out[(size_t)b * A + q] = g.a[sp * A + q];
            g.p_out[(size_t)b * A + q] = yrow[q];
        }
        if (tid == 0) { g.r_out[b] = g.r[se]; g.pv_out[b] = g.v[sp]; }
    }
    if (p.obs_bulk_ok && tid == 0) bulk_wait_read<0>();
}
__global__ void __launch_bounds__(kCopyThreads) k_rollout_gather_index_bf16(const RolloutIndexGatherParams g) {
    rollout_gather_index<uint16_t>(g);
}

}  // namespace pmrl

using namespace pmrl;

static int copy_f32(float* dst, const float* src, size_t n, cudaStream_t s) {
    if (n == 0) return 0;
    size_t blocks = (n / 4 + kCopyThreads - 1) / kCopyThreads;
    const size_t cap = (size_t)pmrl_sm_count() * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    k_copy_f32<<<(unsigned)blocks, kCopyThreads, 0, s>>>(dst, src, n);
    return pmrl_check_launch("k_copy_f32");
}

extern "C" int pmrl_rollout_add(int32_t E, int32_t A, int32_t W, int32_t F, int32_t slot,
                                const float* obs, const float* action, const float* value, const float* reward,
                                float* s, float* a, float* v, float* r, void* stream) {
    if (E < 0 || A < 1 || W < 1 || F < 1 || slot < 0) return pmrl_fail(PMRL_E_SHAPE, "rollout_add: bad sizes");
    if (!action || !value || !reward || !a || !v || !r) return pmrl_fail(PMRL_E_ARG, "rollout_add: NULL pointer");
    if (obs && !s) return pmrl_fail(PMRL_E_ARG, "rollout_add: obs given but s is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t row = (size_t)A * W * F;
    int rc = 0;
    if (obs) rc = copy_f32(s + (size_t)slot * E * row, obs, (size_t)E * row, st);
    if (!rc) rc = copy_f32(a + (size_t)slot * E * A, action, (size_t)E * A, st);
    if (!rc) rc = copy_f32(v + (size_t)slot * E, value, (size_t)E, st);
    if (!rc) rc = copy_f32(r + (size_t)slot * E, reward, (size_t)E, st);
    return rc;
}

// s / s_out: float, or uint16_t bf16 bits (bf16 = true)
static int rollout_gather(int32_t S, int32_t E, int32_t A, int32_t W, int32_t F, int32_t B,
                          const int32_t* slots, const int32_t* envs,
                          const void* s, const float* a, const float* v, const float* r, const float* y,
                          void* s_out, float* a_out, float* r_out, float* pv_out, float* pa_out, float* p_out,
                          bool bf16, void* stream) {
    if (S < 1 || E < 1 || A < 1 || W < 1 || F < 1 || B < 0) return pmrl_fail(PMRL_E_SHAPE, "rollout_gather: bad sizes");
    if (!slots || !envs || !s || !a || !v || !r || !y || !s_out || !a_out || !r_out || !pv_out || !pa_out || !p_out)
        return pmrl_fail(PMRL_E_ARG, "rollout_gather: NULL pointer");
    if (B == 0) return 0;
    RolloutGatherParams g{S, E, A, W, F, B, slots, envs, (const float*)s, a, v, r, y, (float*)s_out, a_out, r_out, pv_out, pa_out, p_out};
    const size_t row = (size_t)A * W * F;
    int chunks = (int)((row * (bf16 ? 2 : 4) + 32767) / 32768);
    if (chunks < 1) chunks = 1;
    if (chunks > 65535) chunks = 65535;
    if (bf16) {
        k_rollout_gather_bf16<<<dim3(B, chunks), kCopyThreads, 0, (cudaStream_t)stream>>>(g);
        return pmrl_check_launch("k_rollout_gather_bf16");
    }
    k_rollout_gather<<<dim3(B, chunks), kCopyThreads, 0, (cudaStream_t)stream>>>(g);
    return pmrl_check_launch("k_rollout_gather");
}

extern "C" int pmrl_rollout_gather(int32_t S, int32_t E, int32_t A, int32_t W, int32_t F, int32_t B,
                                   const int32_t* slots, const int32_t* envs,
                                   const float* s, const float* a, const float* v, const float* r, const float* y,
                                   float* s_out, float* a_out, float* r_out, float* pv_out, float* pa_out, float* p_out,
                                   void* stream) {
    return rollout_gather(S, E, A, W, F, B, slots, envs, s, a, v, r, y, s_out, a_out, r_out, pv_out, pa_out, p_out, false, stream);
}

extern "C" int pmrl_rollout_gather_bf16(int32_t S, int32_t E, int32_t A, int32_t W, int32_t F, int32_t B,
                                        const int32_t* slots, const int32_t* envs,
                                        const uint16_t* s, const float* a, const float* v, const float* r, const float* y,
                                        uint16_t* s_out, float* a_out, float* r_out, float* pv_out, float* pa_out, float* p_out,
                                        void* stream) {
    return rollout_gather(S, E, A, W, F, B, slots, envs, s, a, v, r, y, s_out, a_out, r_out, pv_out, pa_out, p_out, true, stream);
}

extern "C" int pmrl_replay_add(int32_t P, int32_t L, int32_t E, int32_t A, int32_t epoch_slot, int32_t step_slot,
                               const int32_t* item_index, const float* action, const float* reward,
                               int32_t* bi, float* ba, float* br, void* stream) {
    if (P < 1 || L < 1 || E < 0 || A < 1) return pmrl_fail(PMRL_E_SHAPE, "replay_add: bad sizes");
    if (epoch_slot < 0 || epoch_slot >= P || step_slot < 0 || step_slot >= L) return pmrl_fail(PMRL_E_SHAPE, "replay_add: slot out of range");
    if (!item_index || !action || !reward || !bi || !ba || !br) return pmrl_fail(PMRL_E_ARG, "replay_add: NULL pointer");
    if (E == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t at = (size_t)epoch_slot * L + step_slot;
    k_copy_i32<<<(E + 255) / 256, 256, 0, st>>>(bi + at * E, item_index, (size_t)E);
    if (int rc = pmrl_check_launch("k_copy_i32")) return rc;
    if (int rc = copy_f32(ba + at * E * A, action, (size_t)E * A, st)) return rc;
    return copy_f32(br + at * E, reward, (size_t)E, st);
}

// same tile chooser as the env obs kernels (env_kernels.cu) restricted to what the gather needs; esz: bytes per obs element
static void choose_tile(int A, int W, int F, size_t esz, const void* o1, const void* o2, StepParams& p) {
    const size_t per = (size_t)W * F * esz;
    int max_ta = (int)(kObsTileCapBytes / per);
    if (max_ta > A) max_ta = A;
    if (max_ta < 1) max_ta = 1;
    const bool aligned = (((size_t)A * W * F * esz) % 16 == 0) && (((uintptr_t)o1 | (uintptr_t)o2) % 16 == 0);
    int best = -1; long best_waste = 0;
    if (aligned) {
        for (int ta = max_ta; ta >= 1; --ta) {
            if (((size_t)ta * W * F * esz) % 16 != 0 && ta < A) continue;
            const long waste = (long)((A + ta - 1) / ta) * ta - A;
            if (best < 0 || waste < best_waste) { best = ta; best_waste = waste; }
            if (ta <= (max_ta + 1) / 2 && best > 0) break;
        }
    }
    p.tile_assets = best > 0 ? best : max_ta;
    p.obs_bulk_ok = best > 0;
    p.tiles_per_env = (A + p.tile_assets - 1) / p.tile_assets;
}

// s_out / s2_out: float, or uint16_t bf16 bits (bf16 = true)
static int replay_gather(int32_t P, int32_t L, int32_t E, int32_t A, int32_t W, int32_t F, int32_t T, int32_t B,
                         const int32_t* epochs, const int32_t* envs, const int32_t* starts,
                         const int32_t* bi, const float* ba, const float* br, const float* feat_am,
                         void* s_out, float* a_out, float* r_out, void* s2_out, bool bf16, void* stream) {
    if (P < 1 || L < 1 || E < 1 || A < 1 || W < 1 || F < 2 || T < W + 1 || B < 0) return pmrl_fail(PMRL_E_SHAPE, "replay_gather: bad sizes");
    if (!epochs || !envs || !starts || !bi || !ba || !br || !feat_am || !s_out || !a_out || !r_out || !s2_out)
        return pmrl_fail(PMRL_E_ARG, "replay_gather: NULL pointer");
    if ((size_t)W * F * 4 > kObsTileCapBytes) return pmrl_fail(PMRL_E_SHAPE, "replay_gather: W*F*4 exceeds the tile capacity");
    if (F - 1 == 4 && ((uintptr_t)feat_am) % 16 != 0) return pmrl_fail(PMRL_E_ALIGN, "feat_am must be 16-byte aligned");
    if (B == 0) return 0;
    ReplayGatherParams g;
    memset(&g, 0, sizeof(g));
    g.p.A = A; g.p.W = W; g.p.F = F; g.p.T = T; g.p.feat_am = feat_am;
    const size_t esz = bf16 ? 2 : 4;
    choose_tile(A, W, F, esz, s_out, s2_out, g.p);
    g.P = P; g.L = L; g.E = E; g.B = B;
    g.epochs = epochs; g.envs = envs; g.starts = starts; g.bi = bi; g.ba = ba; g.br = br;
    g.s_out = (float*)s_out; g.a_out = a_out; g.r_out = r_out; g.s2_out = (float*)s2_out;
    const size_t smem = (size_t)g.p.tile_assets * W * F * esz;
    if (bf16) {
        k_replay_gather_bf16<<<dim3(B, g.p.tiles_per_env, 2), kCopyThreads, smem, (cudaStream_t)stream>>>(g);
        return pmrl_check_launch("k_replay_gather_bf16");
    }
    k_replay_gather<<<dim3(B, g.p.tiles_per_env, 2), kCopyThreads, smem, (cudaStream_t)stream>>>(g);
    return pmrl_check_launch("k_replay_gather");
}

extern "C" int pmrl_replay_gather(int32_t P, int32_t L, int32_t E, int32_t A, int32_t W, int32_t F, int32_t T, int32_t B,
                                  const int32_t* epochs, const int32_t* envs, const int32_t* starts,
                                  const int32_t* bi, const float* ba, const float* br, const float* feat_am,
                                  float* s_out, float* a_out, float* r_out, float* s2_out, void* stream) {
    return replay_gather(P, L, E, A, W, F, T, B, epochs, envs, starts, bi, ba, br, feat_am, s_out, a_out, r_out, s2_out, false, stream);
}

extern "C" int pmrl_replay_gather_bf16(int32_t P, int32_t L, int32_t E, int32_t A, int32_t W, int32_t F, int32_t T, int32_t B,
                                       const int32_t* epochs, const int32_t* envs, const int32_t* starts,
                                       const int32_t* bi, const float* ba, const float* br, const float* feat_am,
                                       uint16_t* s_out, float* a_out, float* r_out, uint16_t* s2_out, void* stream) {
    return replay_gather(P, L, E, A, W, F, T, B, epochs, envs, starts, bi, ba, br, feat_am, s_out, a_out, r_out, s2_out, true, stream);
}

// s_out: float, or uint16_t bf16 bits (bf16 = true)
static int rollout_gather_index(int32_t S, int32_t E, int32_t A, int32_t W, int32_t F, int32_t T, int32_t B,
                                const int32_t* slots, const int32_t* envs,
                                const int32_t* bi, const float* a, const float* v, const float* r,
                                const float* wp, const float* feat_am, const float* y_tm,
                                void* s_out, float* a_out, float* r_out, float* pv_out, float* pa_out, float* p_out,
                                bool bf16, void* stream) {
    if (S < 2 || E < 1 || A < 1 || W < 2 || F < 2 || T < W + 1 || B < 0) return pmrl_fail(PMRL_E_SHAPE, "rollout_gather_index: bad sizes");
    if (!slots || !envs || !bi || !a || !v || !r || !wp || !feat_am || !y_tm || !s_out || !a_out || !r_out || !pv_out || !pa_out || !p_out)
        return pmrl_fail(PMRL_E_ARG, "rollout_gather_index: NULL pointer");
    if ((size_t)W * F * 4 > kObsTileCapBytes) return pmrl_fail(PMRL_E_SHAPE, "rollout_gather_index: W*F*4 exceeds the tile capacity");
    if (F - 1 == 4 && ((uintptr_t)feat_am) % 16 != 0) return pmrl_fail(PMRL_E_ALIGN, "feat_am must be 16-byte aligned");
    if (B == 0) return 0;
    RolloutIndexGatherParams g;
    memset(&g, 0, sizeof(g));
    g.p.A = A; g.p.W = W; g.p.F = F; g.p.T = T; g.p.feat_am = feat_am;
    const size_t esz = bf16 ? 2 : 4;
    choose_tile(A, W, F, esz, s_out, s_out, g.p);
    g.S = S; g.E = E; g.B = B; g.off = W - 1;
    g.slots = slots; g.envs = envs; g.bi = bi; g.a = a; g.v = v; g.r = r; g.wp = wp; g.y_tm = y_tm;
    g.s_out = (float*)s_out; g.a_out = a_out; g.r_out = r_out; g.pv_out = pv_out; g.pa_out = pa_out; g.p_out = p_out;
    const size_t smem = (size_t)g.p.tile_assets * W * F * esz;
    if (bf16) {
        k_rollout_gather_index_bf16<<<dim3(B, g.p.tiles_per_env), kCopyThreads, smem, (cudaStream_t)stream>>>(g);
        return pmrl_check_launch("k_rollout_gather_index_bf16");
    }
    k_rollout_gather_index<<<dim3(B, g.p.tiles_per_env), kCopyThreads, smem, (cudaStream_t)stream>>>(g);
    return pmrl_check_launch("k_rollout_gather_index");
}

extern "C" int pmrl_rollout_gather_index(int32_t S, int32_t E, int32_t A, int32_t W, int32_t F, int32_t T, int32_t B,
                                         const int32_t* slots, const int32_t* envs,
                                         const int32_t* bi, const float* a, const float* v, const float* r,
                                         const float* wp, const float* feat_am, const float* y_tm,
                                         float* s_out, float* a_out, float* r_out, float* pv_out, float* pa_out, float* p_out,
                                         void* stream) {
    return rollout_gather_index(S, E, A, W, F, T, B, slots, envs, bi, a, v, r, wp, feat_am, y_tm, s_out, a_out, r_out, pv_out,
                                pa_out, p_out, false, stream);
}

extern "C" int pmrl_rollout_gather_index_bf16(int32_t S, int32_t E, int32_t A, int32_t W, int32_t F, int32_t T, int32_t B,
                                              const int32_t* slots, const int32_t* envs,
                                              const int32_t* bi, const float* a, const float* v, const float* r,
                                              const float* wp, const float* feat_am, const float* y_tm,
                                              uint16_t* s_out, float* a_out, float* r_out, float* pv_out, float* pa_out,
                                              float* p_out, void* stream) {
    return rollout_gather_index(S, E, A, W, F, T, B, slots, envs, bi, a, v, r, wp, feat_am, y_tm, s_out, a_out, r_out, pv_out,
                                pa_out, p_out, true, stream);
}
