// env_step_rt.cu — fused step + observation kernel, variant "RT": the weight ring of an env enters the SM as ONE
// contiguous TMA bulk load (W·A·4 bytes, e.g. 20 KB) instead of 8 register loads per thread and tile.
//
// Same structure as env_step_fast.cu (persistent CTAs, groups of G <= 8 envs — 16 for A <= 64, two per warp —,
// 32-asset-row tiles, register-staged table loads, one TMA bulk store per tile) with these differences:
//   * ring rows never travel through registers or the L1 load queue: thread 0 issues cp.async.bulk global→shared for
//     the whole ring of env el (2-4 rings resident: envs el .. el+NB-1), completion on an mbarrier; the weight
//     channel of a tile is then filled from shared memory (lanes over assets: conflict-free).  The L1 queue only
//     carries the L2-hit table loads, so no DRAM-latency load can sit in front of them, and DRAM sees one
//     page-friendly 20 KB read per env instead of 200 scattered 128-byte reads;
//   * 2 CTAs per SM (110 KB of shared memory each), up to 128 registers, no spills;
//   * groups are handed out through a self-resetting global ticket counter (no static stride: no 55-or-56-round tail,
//     and a CTA delayed by a concurrent kernel just takes fewer groups); while a group streams, the next group's
//     actions and scalar state are prefetched into L2.
// Requires (W·A) % 4 == 0 (16-byte alignment of every env's ring) and 2·W·A·4 + tiles to fit in shared memory.
// Weight channel semantics: ActionBuffer.get_all (weight_buffer.py:32-44), fresh row from shared memory.
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include "pmrl_b200.h"
#include "pmrl_device.cuh"
#include "env_step.cuh"
#include "env_launch.h"
#include "host_util.h"

namespace pmrl {

constexpr int kRtThreads = 256;
constexpr int kRtWarps = kRtThreads / 32;
constexpr int kRtGroup = kRtWarps;                 // envs per group, one per warp (A > 64)
constexpr int kRtGroupNarrow = 2 * kRtWarps;       // A <= 64: two envs per warp

struct RtEnv { int row0, shift, fresh_slot, pad; };

// Tile geometry for C4 = ceil((F - 1) / 4) float4 chunks per (asset, table row): F <= 5, 9, 13, 17 (OHLC, OHLC + indicator
// outputs).  When (F - 1) % 4 != 0 the chunks come from the channel-padded table PmrlTables.feat_am4 and the last chunk of a
// row stores only its (F - 1) - 4 (C4 - 1) real channels.
// A warp owns RPW asset rows of a tile and stages ≤ 8 float4 per thread one tile ahead, so wider rows mean lower tiles:
// 32 rows at F = 5 (32 KB at W = 50), 16 at F = 9 (28.8 KB), 8 at F = 13 / 17.
template <int C4> struct RtGeom {
    static constexpr int RPW = C4 == 1 ? 4 : C4 == 2 ? 2 : 1;      // asset rows per warp and tile
    static constexpr int TR = 8 * RPW;                             // asset rows per tile
    static constexpr int NSUB = 32 / TR;                           // lane groups sharing the weight channel of a tile row
    static constexpr int JMAX = 8 / NSUB;                          // window slots (stride 8) per lane, W <= 64
};
template <int C4, int WT> struct RtFeat {
    static constexpr int MW = ((WT ? WT : 64) + 31) / 32 * C4;     // float4 chunks of one window run per lane (W <= 64)
    float4 fv[RtGeom<C4>::RPW][MW];
};

// bf16 tile stores (OT = uint16_t).  Four channels of one (window row, chunk) at halfword offset d: two 32-bit words when d is
// even, else 16 + 32 + 16 bits.  A 32-bit store only ever covers two feature channels of the same chunk, never the weight
// slot, which other threads fill in the same phase.
__device__ __forceinline__ void st_bf16x4(uint16_t* d, const float4 v) {
    if ((reinterpret_cast<uintptr_t>(d) & 2) == 0) {
        reinterpret_cast<uint32_t*>(d)[0] = bf16x2_bits(v.x, v.y);
        reinterpret_cast<uint32_t*>(d)[1] = bf16x2_bits(v.z, v.w);
    } else {
        d[0] = bf16_bits(v.x);
        *reinterpret_cast<uint32_t*>(d + 1) = bf16x2_bits(v.y, v.z);
        d[3] = bf16_bits(v.w);
    }
}

// PAD = false: F = 4 C4 + 1 is a compile-time constant (every tile offset folds); PAD = true: F = p.F at run time, chunks from
// the channel-padded table (measured: a run-time F in the headline instantiation costs 8 %, hence the split).
template <int NPL, bool HASC, int VEC, int WT, int C4, bool PAD = false>
__global__ void __launch_bounds__(kRtThreads, 2) k_env_step_obs_rt(const StepParams p) {
    using Geo = RtGeom<C4>;
    using Feat = RtFeat<C4, WT>;
    constexpr int RPW = Geo::RPW, TR = Geo::TR, NSUB = Geo::NSUB, JMAX = Geo::JMAX, MW = Feat::MW;
    const int F = PAD ? p.F : 4 * C4 + 1;                            // PAD: 4 (C4 - 1) + 1 < F < 4 C4 + 1
    const int cv = PAD ? F - 1 - 4 * (C4 - 1) : 4;                   // real channels in the last chunk of a row
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ double s_stats[kRtWarps * PMRL_STATS_LEN];
    __shared__ RtEnv s_env[kRtGroupNarrow];
    __shared__ __align__(8) uint64_t s_rbar[4];
    __shared__ int s_next;
    const int W = WT ? WT : p.W;
    const int A = p.A, T = p.T, G = p.group_envs;
    const int WA = W * A;
    const int tile_floats = TR * W * F;
    float* const tile0 = reinterpret_cast<float*>(smem_raw);
    float* const tile1 = tile0 + tile_floats;
    float* const s_ring = tile1 + tile_floats;                       // [NB][W*A] rings of consecutive envs
    const int NB = p.ring_bufs;                                      // rings resident at once (2 at A = 100, up to 4 for narrow envs)
    float* const s_wnew = s_ring + NB * WA;                          // [G*A]    w' per asset-row of the group
    int* const s_ea = reinterpret_cast<int*>(s_wnew + G * A);        // [G*A]    (env-in-group << 16) | asset
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_groups = (p.E + G - 1) / G;
    const size_t row_floats = (size_t)W * F;
    if (tid == 0) { for (int b = 0; b < 4; ++b) mbar_init(&s_rbar[b], 1); mbar_fence_init(); }
    WarpStats ws;
    wstats_init(ws);
    __syncthreads();

    // feature window of one asset = W·C4 contiguous float4 chunks of the table; lane l stages the C4 chunks of window rows
    // l and l + 32 and scatters chunk (w, q) to tile offset w·F + 4q of its asset row: with lanes over w the shared stores
    // of one instruction hit banks (F·l + const) mod 32 — F is odd, so all 32 differ (lanes over consecutive chunks, the
    // first version, gave two-way conflicts at F = 9: 312 conflicts per tile, mio_throttle 1.6 per issue)
    const int rl = lane % TR, sub = lane / TR;                       // weight channel: tile row of this lane, its window-slot phase
    const int wbase = (rl * W + warp + 8 * sub) * F + (F - 1);
    const int n8 = max(0, (W - warp + 7) >> 3);                      // window slots warp, warp + 8, … below W
    const int nj = n8 > sub ? (n8 - sub + NSUB - 1) / NSUB : 0;
    const float4* __restrict__ tbl = reinterpret_cast<const float4*>(PAD ? p.feat_am4 : p.feat_am) + lane * C4;
    // Even F (PAD instantiations only): a row pitch of F floats puts the lanes-over-window-rows stores on 32 / gcd(F, 32) banks.
    // With 2-way conflicts the chunk form still wins (F = 6 at 65,536 x 100: 2.13 ms = 0.66 against 3.12 ms dense), with 8-way
    // it does not (F = 8: 3.78 ms = 0.48 against 3.16 ms = 0.57 dense), so F = 8 and 16 take the DENSE form: lane l owns floats l, l + 32, … of the asset row's W·F-float image, loads feature (w, c) = (n / F, n % F)
    // as a scalar from the UNPADDED table (index n - w: consecutive lanes read consecutive floats but for one gap per
    // window row) and stores it to offset n — consecutive banks, conflict-free for every F.  The weight slot c = F - 1 is
    // skipped (the weight pass below fills it).
    const bool dense = PAD && (F & 7) == 0;
    const unsigned inv_f = PAD ? (65536u + (unsigned)F - 1u) / (unsigned)F : 0u;   // n / F = (n * inv_f) >> 16 for n < 64 * 17
    constexpr int MD = 8 * C4;                                       // floats of a row image per lane (W <= 64, F <= 4 C4 + 1)

    int buf = 0;
    int ebase = 0;                                                   // envs streamed by this CTA so far (ring buffer / phase index)
    // Groups are handed out dynamically: the first one is the CTA's own index, every further one a ticket from a global
    // counter.  A static stride leaves 16,384 groups on 296 CTAs as 55 or 56 rounds (a 1.8 % tail), and a CTA that starts
    // late — e.g. behind a concurrent NCCL kernel holding its SM's shared memory — would finish a whole round late.
    int grp = blockIdx.x;
    while (grp < n_groups) {
        const int e0 = grp * G;
        const int ne = min(G, p.E - e0);
        unsigned int ticket = 0;
        if (tid == 0) ticket = p.ticket ? atomicAdd(p.ticket, 1u)    // consumed after phase 1: its latency hides under the step
                                        : (unsigned int)(grp - (int)blockIdx.x);   // no counters: static stride over the groups
        // ---------------- phase 1: one warp per env (two per warp for narrow envs: groups of up to 16) ----------------
        auto publish = [&](int el, const EnvVectors<NPL, HASC, VEC>& ev, const StepOut& so) {
#pragma unroll
            for (int j = 0; j < NPL; ++j) {
                const int a = asset_of<VEC>(lane, j);
                if (a < A) { s_wnew[el * A + a] = ev.a[j]; s_ea[el * A + a] = (el << 16) | a; }
            }
            if (lane == 0) {
                RtEnv ge;
                ge.row0 = p.t0[e0 + el] + so.k;
                ge.shift = so.is_full ? 0 : (W - so.idx_new);          // weight_buffer.py:38-42
                ge.fresh_slot = so.did_reset ? 0 : so.slot_written;     // the row written by this launch comes from smem
                ge.pad = 0;
                s_env[el] = ge;
            }
        };
        if constexpr (NPL <= 2) {
            // A <= 64: an env is only 50-odd rows of streaming, so the step latency weighs twice as much per byte as at
            // A = 100.  Each warp advances two envs with their loads issued together (scalars, then vectors, then the math).
            const int el0 = warp, el1 = warp + kRtWarps;
            EnvScalars sc0, sc1;
            EnvVectors<NPL, HASC, VEC> ev0, ev1;
            StepOut so;
            if (el0 < ne) env_load_scalars(p, e0 + el0, sc0);
            if (el1 < ne) env_load_scalars(p, e0 + el1, sc1);
            if (el0 < ne) env_load_vectors<NPL, HASC, VEC>(p, e0 + el0, lane, sc0, ev0);
            if (el1 < ne) env_load_vectors<NPL, HASC, VEC>(p, e0 + el1, lane, sc1, ev1);
            if (el0 < ne) { env_compute_store<NPL, HASC, VEC>(p, e0 + el0, lane, sc0, ev0, so, ws); publish(el0, ev0, so); }
            if (el1 < ne) { env_compute_store<NPL, HASC, VEC>(p, e0 + el1, lane, sc1, ev1, so, ws); publish(el1, ev1, so); }
        } else if (warp < ne) {
            EnvVectors<NPL, HASC, VEC> ev;
            StepOut so;
            env_step_warp<NPL, HASC, VEC>(p, e0 + warp, lane, ev, so, ws);
            publish(warp, ev, so);
        }
        if (tid == 0) s_next = p.ticket ? (int)(gridDim.x + ticket) : grp + (int)gridDim.x;
        __syncthreads();
        const int next_grp = s_next;                                  // (rewritten only after the tile loop's barriers)
        // pull what phase 1 of the next group will read from DRAM (raw actions, scalar state) into L2 while this group
        // streams: its dependent chain scalars → addresses → vectors then runs on L2 hits
        if (p.prefetch_next && next_grp < n_groups) {
            const int ne_next = min(G, p.E - next_grp * G);
            const size_t a_first = (size_t)next_grp * G * A;
            const int a_lines = (ne_next * A + 31) >> 5;              // 128-byte lines of the group's action rows
            for (int q = tid; q < a_lines; q += kRtThreads) prefetch_l2(p.actions + a_first + (size_t)q * 32);
            if (tid == 32) { prefetch_l2(p.value + next_grp * G); prefetch_l2(p.idx + next_grp * G); prefetch_l2(p.t + next_grp * G); }
            if (tid == 64) { prefetch_l2(p.t0 + next_grp * G); prefetch_l2(p.is_full + next_grp * G); if (p.ep_return) prefetch_l2(p.ep_return + next_grp * G); }
        }
        // ---------------- phase 2 ----------------
        const int R = ne * A;
        const int ntiles = (R + TR - 1) / TR, nfull = R / TR;
        const float* __restrict__ hist_g = p.hist + (size_t)e0 * WA;
        float* const obs_grp = p.obs + (size_t)e0 * A * row_floats;
        int issued = 0;                                               // envs of this group whose ring load has been issued
        auto issue_rings = [&](int upto) {                            // thread 0 only
            for (; issued < upto; ++issued) {
                const int n = ebase + issued;
                const int b = n % NB;
                mbar_arrive_expect_tx(&s_rbar[b], (uint32_t)WA * 4u);
                bulk_load_g2s(s_ring + b * WA, hist_g + (size_t)issued * WA, (uint32_t)WA * 4u, &s_rbar[b], kPolicyEvictFirst);
            }
        };
        if (tid == 0) issue_rings(min(ne, NB));
        int wel = rl / A, wa = rl - wel * A;                          // (env-in-group, asset) of this lane's weight row

        auto load_feat = [&](Feat& fr, int r0, auto partial) {
            constexpr bool PARTIAL = decltype(partial)::value;
            const int nr = PARTIAL ? R - r0 : TR;
#pragma unroll
            for (int i = 0; i < RPW; ++i) {
                if (!PARTIAL || warp + 8 * i < nr) {
                    const int ea = s_ea[r0 + warp + 8 * i];
                    if constexpr (PAD) {
                        if (dense) {
                            const float* __restrict__ srcd = p.feat_am + (size_t)((ea & 0xffff) * T + s_env[ea >> 16].row0) * (F - 1);
                            float* const dv = reinterpret_cast<float*>(&fr.fv[i][0]);
                            const int nrow = W * F;
#pragma unroll
                            for (int m = 0; m < MD; ++m) {
                                const int n = lane + 32 * m;
                                const int w = (int)(((unsigned)n * inv_f) >> 16);
                                if (n < nrow && n - w * F != F - 1) dv[m] = ld_keep(srcd + (n - w), kPolicyEvictLast);
                            }
                            continue;
                        }
                    }
                    const float4* __restrict__ src = tbl + (size_t)((ea & 0xffff) * T + s_env[ea >> 16].row0) * C4;
#pragma unroll
                    for (int m = 0; m < MW; ++m)                      // m = (m / C4)-th window row of this lane, chunk m % C4
                        if (lane + 32 * (m / C4) < W) fr.fv[i][m] = ld_keep4(src + 32 * C4 * (m / C4) + (m % C4), kPolicyEvictLast);
                }
            }
        };
        auto spill_tile = [&](const Feat& fr, float* __restrict__ tile, int r0, auto partial) {
            constexpr bool PARTIAL = decltype(partial)::value;
            const int nr = PARTIAL ? R - r0 : TR;
#pragma unroll
            for (int i = 0; i < RPW; ++i) {
                if (!PARTIAL || warp + 8 * i < nr) {
                    float* drow = tile + (warp + 8 * i) * W * F;
                    if constexpr (PAD) {
                        if (dense) {
                            const float* const dv = reinterpret_cast<const float*>(&fr.fv[i][0]);
                            const int nrow = W * F;
#pragma unroll
                            for (int m = 0; m < MD; ++m) {
                                const int n = lane + 32 * m;
                                const int w = (int)(((unsigned)n * inv_f) >> 16);
                                if (n < nrow && n - w * F != F - 1) drow[n] = dv[m];
                            }
                            continue;
                        }
                    }
#pragma unroll
                    for (int m = 0; m < MW; ++m) {
                        const int w = lane + 32 * (m / C4);
                        if (w < W) {
                            float* d = drow + w * F + 4 * (m % C4);
                            const float4 v = fr.fv[i][m];
                            if (!PAD || m % C4 < C4 - 1) { d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w; }
                            else {                                    // last chunk of the row: cv real channels, the rest is padding
                                d[0] = v.x;
                                if (cv > 1) d[1] = v.y;
                                if (cv > 2) d[2] = v.z;
                                if (cv > 3) d[3] = v.w;
                            }
                        }
                    }
                }
            }
            if (!PARTIAL || rl < nr) {                                // weight channel straight from the staged ring
                const int n = ebase + wel;
                const int b = n % NB;
                mbar_wait(&s_rbar[b], (uint32_t)((n / NB) & 1));
                const RtEnv ge = s_env[wel];
                const float* __restrict__ rs = s_ring + b * WA + wa;
                const float fresh = s_wnew[r0 + rl];
#pragma unroll
                for (int j = 0; j < JMAX; ++j) {
                    if (j < nj) {
                        const int slot = warp + 8 * (j * NSUB + sub) - ge.shift;
                        float v = 0.0f;                               // zero front padding while the ring is not full
                        if (slot >= 0) v = (slot == ge.fresh_slot) ? fresh : rs[slot * A];
                        tile[wbase + 8 * NSUB * F * j] = v;
                    }
                }
            }
            wa += TR;
            while (wa >= A) { wa -= A; ++wel; }
        };

        Feat fr;
        if (nfull > 0) load_feat(fr, 0, std::false_type{}); else load_feat(fr, 0, std::true_type{});
        for (int ti = 0; ti < ntiles; ++ti) {
            // ONE CTA barrier per tile.  The buffer filled now was last read by the bulk store issued two tiles ago; thread 0
            // waited for that store to finish reading shared memory BEFORE it arrived at the previous tile's barrier, so
            // every thread that is past that barrier may overwrite it.  (Round 1 had a second barrier at the top of the tile
            // for exactly this hand-over; barrier stalls were the largest stall reason, 2.0 per issue at F = 5, 2.8 at F = 9.)
            float* const tile = buf ? tile1 : tile0;
            const int r0 = ti * TR;
            if (ti < nfull) spill_tile(fr, tile, r0, std::false_type{}); else spill_tile(fr, tile, r0, std::true_type{});
            if (ti + 1 < ntiles) {
                if (ti + 1 < nfull) load_feat(fr, r0 + TR, std::false_type{}); else load_feat(fr, r0 + TR, std::true_type{});
            }
            fence_proxy_async_smem();
            if (tid == 0) bulk_wait_read<0>();                        // the previous tile's store (other buffer) has drained: see above
            __syncthreads();
            const int nr = min(TR, R - r0);
            float* const gdst = obs_grp + (size_t)r0 * row_floats;
            const int n = nr * W * F;
            if (((((uintptr_t)gdst) | ((size_t)n * 4)) & 15) == 0) {
                if (tid == 0) { bulk_store_s2g(gdst, tile, (uint32_t)n * 4u, kPolicyEvictFirst); bulk_commit(); }
            } else {
                for (int q = tid; q < n; q += kRtThreads) gdst[q] = tile[q];   // (done before this thread reaches the next barrier,
            }                                                                  //  and the tile is refilled only after that one)
            // envs below (r0+TR)/A are complete (every thread passed the barrier after its last read of their ring):
            // their buffers can take the rings of the envs NB positions further on
            if (tid == 0) issue_rings(min(ne, (r0 + TR) / A + NB));
            buf ^= 1;
        }
        ebase += ne;
        grp = next_grp;
    }
    if (tid == 0) {
        bulk_wait_read<0>();
        // the last CTA out re-arms the batch's counters for its next launch
        if (p.ticket) {
            __threadfence();
            if (atomicAdd(p.ticket + 1, 1u) == gridDim.x - 1) { p.ticket[0] = 0u; p.ticket[1] = 0u; __threadfence(); }
        }
    }
    if (p.stats) { wstats_store(ws, s_stats + warp * PMRL_STATS_LEN, lane); stats_flush_block(p.stats, s_stats, kRtWarps); }
}

// The same kernel with the obs written as bf16 (PMRL_OBS_BF16): k_env_step_obs_rt_bf16.  OT is the obs element type; the
// shared tile is the byte image of the obs slab in that type, so a bf16 tile and its bulk store are half the bytes.  The
// body is the fp32 kernel's above with the tile stores rounding (obs_cvt, bf16x2 words) and byte-counted alignment; it is
// instantiated for bf16 only.  The fp32 kernel keeps its own copy: routing it through this template compiles to different
// (reordered, re-allocated) SASS for all 108 fp32 instantiations, and the fp32 path is the measured, pinned reference.
// (#128 "loop is not reachable": with W = 50 compiled in, the bf16 paired-row fill `continue`s past the generic one)
#pragma nv_diag_suppress 128
template <typename OT, int NPL, bool HASC, int VEC, int WT, int C4, bool PAD>
__device__ __forceinline__ void env_step_obs_rt(const StepParams& p) {
    constexpr bool BF = sizeof(OT) == 2;
    using Geo = RtGeom<C4>;
    using Feat = RtFeat<C4, WT>;
    constexpr int RPW = Geo::RPW, TR = Geo::TR, NSUB = Geo::NSUB, JMAX = Geo::JMAX, MW = Feat::MW;
    const int F = PAD ? p.F : 4 * C4 + 1;                            // PAD: 4 (C4 - 1) + 1 < F < 4 C4 + 1
    const int cv = PAD ? F - 1 - 4 * (C4 - 1) : 4;                   // real channels in the last chunk of a row
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ double s_stats[kRtWarps * PMRL_STATS_LEN];
    __shared__ RtEnv s_env[kRtGroupNarrow];
    __shared__ __align__(8) uint64_t s_rbar[4];
    __shared__ int s_next;
    const int W = WT ? WT : p.W;
    const int A = p.A, T = p.T, G = p.group_envs;
    const int WA = W * A;
    const int tile_floats = TR * W * F;                              // (elements of type OT)
    OT* const tile0 = reinterpret_cast<OT*>(smem_raw);
    OT* const tile1 = tile0 + tile_floats;
    float* const s_ring = reinterpret_cast<float*>(tile1 + tile_floats);   // [NB][W*A] rings of consecutive envs
    const int NB = p.ring_bufs;                                      // rings resident at once (2 at A = 100, up to 4 for narrow envs)
    float* const s_wnew = s_ring + NB * WA;                          // [G*A]    w' per asset-row of the group
    int* const s_ea = reinterpret_cast<int*>(s_wnew + G * A);        // [G*A]    (env-in-group << 16) | asset
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_groups = (p.E + G - 1) / G;
    const size_t row_floats = (size_t)W * F;
    if (tid == 0) { for (int b = 0; b < 4; ++b) mbar_init(&s_rbar[b], 1); mbar_fence_init(); }
    WarpStats ws;
    wstats_init(ws);
    __syncthreads();

    // feature window of one asset = W·C4 contiguous float4 chunks of the table; lane l stages the C4 chunks of window rows
    // l and l + 32 and scatters chunk (w, q) to tile offset w·F + 4q of its asset row: with lanes over w the shared stores
    // of one instruction hit banks (F·l + const) mod 32 — F is odd, so all 32 differ (lanes over consecutive chunks, the
    // first version, gave two-way conflicts at F = 9: 312 conflicts per tile, mio_throttle 1.6 per issue)
    const int rl = lane % TR, sub = lane / TR;                       // weight channel: tile row of this lane, its window-slot phase
    const int wbase = (rl * W + warp + 8 * sub) * F + (F - 1);
    const int n8 = max(0, (W - warp + 7) >> 3);                      // window slots warp, warp + 8, … below W
    const int nj = n8 > sub ? (n8 - sub + NSUB - 1) / NSUB : 0;
    const float4* __restrict__ tbl = reinterpret_cast<const float4*>(PAD ? p.feat_am4 : p.feat_am) + lane * C4;
    // Even F (PAD instantiations only): a row pitch of F floats puts the lanes-over-window-rows stores on 32 / gcd(F, 32) banks.
    // With 2-way conflicts the chunk form still wins (F = 6 at 65,536 x 100: 2.13 ms = 0.66 against 3.12 ms dense), with 8-way
    // it does not (F = 8: 3.78 ms = 0.48 against 3.16 ms = 0.57 dense), so F = 8 and 16 take the DENSE form: lane l owns floats l, l + 32, … of the asset row's W·F-float image, loads feature (w, c) = (n / F, n % F)
    // as a scalar from the UNPADDED table (index n - w: consecutive lanes read consecutive floats but for one gap per
    // window row) and stores it to offset n — consecutive banks, conflict-free for every F.  The weight slot c = F - 1 is
    // skipped (the weight pass below fills it).
    const bool dense = PAD && (F & 7) == 0;
    const unsigned inv_f = PAD ? (65536u + (unsigned)F - 1u) / (unsigned)F : 0u;   // n / F = (n * inv_f) >> 16 for n < 64 * 17
    constexpr int MD = 8 * C4;                                       // floats of a row image per lane (W <= 64, F <= 4 C4 + 1)
    // bf16 at F = 5 with an even W (even row pitch W·F): lane l owns window rows 2l and 2l + 1, i.e. the 10 halfwords at word
    // offset 5l of the asset row — three 32-bit stores (bank 5l + const: conflict-free) and two 16-bit ones next to the
    // weight slots, 2.5 stores per window row instead of 5 for the lanes-over-rows mapping
    [[maybe_unused]] const bool pair = BF && C4 == 1 && !PAD && (W & 1) == 0;

    int buf = 0;
    int ebase = 0;                                                   // envs streamed by this CTA so far (ring buffer / phase index)
    // Groups are handed out dynamically: the first one is the CTA's own index, every further one a ticket from a global
    // counter.  A static stride leaves 16,384 groups on 296 CTAs as 55 or 56 rounds (a 1.8 % tail), and a CTA that starts
    // late — e.g. behind a concurrent NCCL kernel holding its SM's shared memory — would finish a whole round late.
    int grp = blockIdx.x;
    while (grp < n_groups) {
        const int e0 = grp * G;
        const int ne = min(G, p.E - e0);
        unsigned int ticket = 0;
        if (tid == 0) ticket = p.ticket ? atomicAdd(p.ticket, 1u)    // consumed after phase 1: its latency hides under the step
                                        : (unsigned int)(grp - (int)blockIdx.x);   // no counters: static stride over the groups
        // ---------------- phase 1: one warp per env (two per warp for narrow envs: groups of up to 16) ----------------
        auto publish = [&](int el, const EnvVectors<NPL, HASC, VEC>& ev, const StepOut& so) {
#pragma unroll
            for (int j = 0; j < NPL; ++j) {
                const int a = asset_of<VEC>(lane, j);
                if (a < A) { s_wnew[el * A + a] = ev.a[j]; s_ea[el * A + a] = (el << 16) | a; }
            }
            if (lane == 0) {
                RtEnv ge;
                ge.row0 = p.t0[e0 + el] + so.k;
                ge.shift = so.is_full ? 0 : (W - so.idx_new);          // weight_buffer.py:38-42
                ge.fresh_slot = so.did_reset ? 0 : so.slot_written;     // the row written by this launch comes from smem
                ge.pad = 0;
                s_env[el] = ge;
            }
        };
        if constexpr (NPL <= 2) {
            // A <= 64: an env is only 50-odd rows of streaming, so the step latency weighs twice as much per byte as at
            // A = 100.  Each warp advances two envs with their loads issued together (scalars, then vectors, then the math).
            const int el0 = warp, el1 = warp + kRtWarps;
            EnvScalars sc0, sc1;
            EnvVectors<NPL, HASC, VEC> ev0, ev1;
            StepOut so;
            if (el0 < ne) env_load_scalars(p, e0 + el0, sc0);
            if (el1 < ne) env_load_scalars(p, e0 + el1, sc1);
            if (el0 < ne) env_load_vectors<NPL, HASC, VEC>(p, e0 + el0, lane, sc0, ev0);
            if (el1 < ne) env_load_vectors<NPL, HASC, VEC>(p, e0 + el1, lane, sc1, ev1);
            if (el0 < ne) { env_compute_store<NPL, HASC, VEC>(p, e0 + el0, lane, sc0, ev0, so, ws); publish(el0, ev0, so); }
            if (el1 < ne) { env_compute_store<NPL, HASC, VEC>(p, e0 + el1, lane, sc1, ev1, so, ws); publish(el1, ev1, so); }
        } else if (warp < ne) {
            EnvVectors<NPL, HASC, VEC> ev;
            StepOut so;
            env_step_warp<NPL, HASC, VEC>(p, e0 + warp, lane, ev, so, ws);
            publish(warp, ev, so);
        }
        if (tid == 0) s_next = p.ticket ? (int)(gridDim.x + ticket) : grp + (int)gridDim.x;
        __syncthreads();
        const int next_grp = s_next;                                  // (rewritten only after the tile loop's barriers)
        // pull what phase 1 of the next group will read from DRAM (raw actions, scalar state) into L2 while this group
        // streams: its dependent chain scalars → addresses → vectors then runs on L2 hits
        if (p.prefetch_next && next_grp < n_groups) {
            const int ne_next = min(G, p.E - next_grp * G);
            const size_t a_first = (size_t)next_grp * G * A;
            const int a_lines = (ne_next * A + 31) >> 5;              // 128-byte lines of the group's action rows
            for (int q = tid; q < a_lines; q += kRtThreads) prefetch_l2(p.actions + a_first + (size_t)q * 32);
            if (tid == 32) { prefetch_l2(p.value + next_grp * G); prefetch_l2(p.idx + next_grp * G); prefetch_l2(p.t + next_grp * G); }
            if (tid == 64) { prefetch_l2(p.t0 + next_grp * G); prefetch_l2(p.is_full + next_grp * G); if (p.ep_return) prefetch_l2(p.ep_return + next_grp * G); }
        }
        // ---------------- phase 2 ----------------
        const int R = ne * A;
        const int ntiles = (R + TR - 1) / TR, nfull = R / TR;
        const float* __restrict__ hist_g = p.hist + (size_t)e0 * WA;
        OT* const obs_grp = reinterpret_cast<OT*>(p.obs) + (size_t)e0 * A * row_floats;
        int issued = 0;                                               // envs of this group whose ring load has been issued
        auto issue_rings = [&](int upto) {                            // thread 0 only
            for (; issued < upto; ++issued) {
                const int n = ebase + issued;
                const int b = n % NB;
                mbar_arrive_expect_tx(&s_rbar[b], (uint32_t)WA * 4u);
                bulk_load_g2s(s_ring + b * WA, hist_g + (size_t)issued * WA, (uint32_t)WA * 4u, &s_rbar[b], kPolicyEvictFirst);
            }
        };
        if (tid == 0) issue_rings(min(ne, NB));
        int wel = rl / A, wa = rl - wel * A;                          // (env-in-group, asset) of this lane's weight row

        auto load_feat = [&](Feat& fr, int r0, auto partial) {
            constexpr bool PARTIAL = decltype(partial)::value;
            const int nr = PARTIAL ? R - r0 : TR;
#pragma unroll
            for (int i = 0; i < RPW; ++i) {
                if (!PARTIAL || warp + 8 * i < nr) {
                    const int ea = s_ea[r0 + warp + 8 * i];
                    if constexpr (PAD) {
                        if (dense) {
                            const float* __restrict__ srcd = p.feat_am + (size_t)((ea & 0xffff) * T + s_env[ea >> 16].row0) * (F - 1);
                            float* const dv = reinterpret_cast<float*>(&fr.fv[i][0]);
                            const int nrow = W * F;
#pragma unroll
                            for (int m = 0; m < MD; ++m) {
                                const int n = lane + 32 * m;
                                const int w = (int)(((unsigned)n * inv_f) >> 16);
                                if (n < nrow && n - w * F != F - 1) dv[m] = ld_keep(srcd + (n - w), kPolicyEvictLast);
                            }
                            continue;
                        }
                    }
                    const float4* __restrict__ src = tbl + (size_t)((ea & 0xffff) * T + s_env[ea >> 16].row0) * C4;
                    if constexpr (BF && C4 == 1 && !PAD) {
                        if (pair) {                                   // rows 2l, 2l + 1 (tbl already points at row l)
                            if (2 * lane < W) { fr.fv[i][0] = ld_keep4(src + lane, kPolicyEvictLast); fr.fv[i][1] = ld_keep4(src + lane + 1, kPolicyEvictLast); }
                            continue;
                        }
                    }
#pragma unroll
                    for (int m = 0; m < MW; ++m)                      // m = (m / C4)-th window row of this lane, chunk m % C4
                        if (lane + 32 * (m / C4) < W) fr.fv[i][m] = ld_keep4(src + 32 * C4 * (m / C4) + (m % C4), kPolicyEvictLast);
                }
            }
        };
        auto spill_tile = [&](const Feat& fr, OT* __restrict__ tile, int r0, auto partial) {
            constexpr bool PARTIAL = decltype(partial)::value;
            const int nr = PARTIAL ? R - r0 : TR;
#pragma unroll
            for (int i = 0; i < RPW; ++i) {
                if (!PARTIAL || warp + 8 * i < nr) {
                    OT* drow = tile + (warp + 8 * i) * W * F;
                    if constexpr (PAD) {
                        if (dense) {
                            const float* const dv = reinterpret_cast<const float*>(&fr.fv[i][0]);
                            const int nrow = W * F;
#pragma unroll
                            for (int m = 0; m < MD; ++m) {
                                const int n = lane + 32 * m;
                                const int w = (int)(((unsigned)n * inv_f) >> 16);
                                if (n < nrow && n - w * F != F - 1) drow[n] = obs_cvt<OT>(dv[m]);
                            }
                            continue;
                        }
                    }
                    if constexpr (BF && C4 == 1 && !PAD) {
                        if (pair) {
                            if (2 * lane < W) {
                                const float4 a = fr.fv[i][0], b = fr.fv[i][1];
                                uint32_t* const dw = reinterpret_cast<uint32_t*>(drow) + 5 * lane;
                                dw[0] = bf16x2_bits(a.x, a.y);
                                dw[1] = bf16x2_bits(a.z, a.w);
                                drow[10 * lane + 5] = bf16_bits(b.x);   // (halfword 10l + 4: weight slot of row 2l)
                                dw[3] = bf16x2_bits(b.y, b.z);
                                drow[10 * lane + 8] = bf16_bits(b.w);   // (halfword 10l + 9: weight slot of row 2l + 1)
                            }
                            continue;
                        }
                    }
#pragma unroll
                    for (int m = 0; m < MW; ++m) {
                        const int w = lane + 32 * (m / C4);
                        if (w < W) {
                            OT* d = drow + w * F + 4 * (m % C4);
                            const float4 v = fr.fv[i][m];
                            if (!PAD || m % C4 < C4 - 1) {
                                if constexpr (BF) st_bf16x4(d, v);
                                else { d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w; }
                            } else {                                  // last chunk of the row: cv real channels, the rest is padding
                                d[0] = obs_cvt<OT>(v.x);
                                if (cv > 1) d[1] = obs_cvt<OT>(v.y);
                                if (cv > 2) d[2] = obs_cvt<OT>(v.z);
                                if (cv > 3) d[3] = obs_cvt<OT>(v.w);
                            }
                        }
                    }
                }
            }
            if (!PARTIAL || rl < nr) {                                // weight channel straight from the staged ring
                const int n = ebase + wel;
                const int b = n % NB;
                mbar_wait(&s_rbar[b], (uint32_t)((n / NB) & 1));
                const RtEnv ge = s_env[wel];
                const float* __restrict__ rs = s_ring + b * WA + wa;
                const float fresh = s_wnew[r0 + rl];
#pragma unroll
                for (int j = 0; j < JMAX; ++j) {
                    if (j < nj) {
                        const int slot = warp + 8 * (j * NSUB + sub) - ge.shift;
                        float v = 0.0f;                               // zero front padding while the ring is not full
                        if (slot >= 0) v = (slot == ge.fresh_slot) ? fresh : rs[slot * A];
                        tile[wbase + 8 * NSUB * F * j] = obs_cvt<OT>(v);
                    }
                }
            }
            wa += TR;
            while (wa >= A) { wa -= A; ++wel; }
        };

        Feat fr;
        if (nfull > 0) load_feat(fr, 0, std::false_type{}); else load_feat(fr, 0, std::true_type{});
        for (int ti = 0; ti < ntiles; ++ti) {
            // ONE CTA barrier per tile.  The buffer filled now was last read by the bulk store issued two tiles ago; thread 0
            // waited for that store to finish reading shared memory BEFORE it arrived at the previous tile's barrier, so
            // every thread that is past that barrier may overwrite it.  (Round 1 had a second barrier at the top of the tile
            // for exactly this hand-over; barrier stalls were the largest stall reason, 2.0 per issue at F = 5, 2.8 at F = 9.)
            OT* const tile = buf ? tile1 : tile0;
            const int r0 = ti * TR;
            if (ti < nfull) spill_tile(fr, tile, r0, std::false_type{}); else spill_tile(fr, tile, r0, std::true_type{});
            if (ti + 1 < ntiles) {
                if (ti + 1 < nfull) load_feat(fr, r0 + TR, std::false_type{}); else load_feat(fr, r0 + TR, std::true_type{});
            }
            fence_proxy_async_smem();
            if (tid == 0) bulk_wait_read<0>();                        // the previous tile's store (other buffer) has drained: see above
            __syncthreads();
            const int nr = min(TR, R - r0);
            OT* const gdst = obs_grp + (size_t)r0 * row_floats;
            const int n = nr * W * F;
            if (((((uintptr_t)gdst) | ((size_t)n * sizeof(OT))) & 15) == 0) {   // (alignment in bytes)
                if (tid == 0) { bulk_store_s2g(gdst, tile, (uint32_t)n * (uint32_t)sizeof(OT), kPolicyEvictFirst); bulk_commit(); }
            } else {
                for (int q = tid; q < n; q += kRtThreads) gdst[q] = tile[q];   // (done before this thread reaches the next barrier,
            }                                                                  //  and the tile is refilled only after that one)
            // envs below (r0+TR)/A are complete (every thread passed the barrier after its last read of their ring):
            // their buffers can take the rings of the envs NB positions further on
            if (tid == 0) issue_rings(min(ne, (r0 + TR) / A + NB));
            buf ^= 1;
        }
        ebase += ne;
        grp = next_grp;
    }
    if (tid == 0) {
        bulk_wait_read<0>();
        // the last CTA out re-arms the batch's counters for its next launch
        if (p.ticket) {
            __threadfence();
            if (atomicAdd(p.ticket + 1, 1u) == gridDim.x - 1) { p.ticket[0] = 0u; p.ticket[1] = 0u; __threadfence(); }
        }
    }
    if (p.stats) { wstats_store(ws, s_stats + warp * PMRL_STATS_LEN, lane); stats_flush_block(p.stats, s_stats, kRtWarps); }
}
#pragma nv_diag_default 128

template <int NPL, bool HASC, int VEC, int WT, int C4, bool PAD = false>
__global__ void __launch_bounds__(kRtThreads, 2) k_env_step_obs_rt_bf16(const StepParams p) {
    env_step_obs_rt<uint16_t, NPL, HASC, VEC, WT, C4, PAD>(p);
}

}  // namespace pmrl

using namespace pmrl;

template <bool BF, int NPL, bool HASC, int VEC, int WT, int C4, bool PAD>
static int launch_rt_t(StepParams& p, size_t smem, int grid, cudaStream_t s) {
    constexpr auto kernel = BF ? k_env_step_obs_rt_bf16<NPL, HASC, VEC, WT, C4, PAD> : k_env_step_obs_rt<NPL, HASC, VEC, WT, C4, PAD>;
    const char* const name = BF ? "k_env_step_obs_rt_bf16" : "k_env_step_obs_rt";
    static bool attr_done[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !attr_done[dev]) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024);
        if (e != cudaSuccess) return pmrl_fail((int)e, BF ? "cudaFuncSetAttribute(k_env_step_obs_rt_bf16) failed" : "cudaFuncSetAttribute(k_env_step_obs_rt) failed");
        attr_done[dev] = true;
    }
    kernel<<<grid, kRtThreads, smem, s>>>(p);
    return pmrl_check_launch(name);
}

template <bool BF, int NPL, int VEC, int C4, bool PAD>
static int launch_rt_w(StepParams& p, size_t smem, int grid, cudaStream_t s) {
    const bool hasc = p.commission > 0.0f;
    if (p.W == 50) return hasc ? launch_rt_t<BF, NPL, true, VEC, 50, C4, PAD>(p, smem, grid, s) : launch_rt_t<BF, NPL, false, VEC, 50, C4, PAD>(p, smem, grid, s);
    return hasc ? launch_rt_t<BF, NPL, true, VEC, 0, C4, PAD>(p, smem, grid, s) : launch_rt_t<BF, NPL, false, VEC, 0, C4, PAD>(p, smem, grid, s);
}

// Envs per group for a batch of E envs on `slots` persistent CTAs.  A CTA's time is (rounds it runs) x (envs per group +
// about one env-time of per-group overhead: barriers and the un-overlapped step phase), and every CTA waits for the
// slowest, so minimise ceil(ceil(E/g)/slots) * (g + 1).  Measured on 4,096 x 50 (config 2): g = 7 → 2 full rounds,
// 58.6 us; the former power-of-two choice g = 4 → 3.46 → 4 rounds, 67.2 us (with 16-env groups and four resident
// rings: g = 14 → one round, 53.4 us).  Large batches end up at the maximum.  Only multiples of `step` are considered.
static int pick_group(int E, int slots, int gmax, int step) {
    int best = step;
    long best_cost = -1;
    for (int g = gmax; g >= step; --g) {
        if (g % step) continue;
        const long n = (E + g - 1) / g;
        const long rounds = (n + slots - 1) / slots;
        const long cost = rounds * (g + 1);
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = g; }
    }
    return best;
}

int pmrl_launch_step_obs_rt(StepParams& p, int npl, int vec, int group, int ctas_per_sm, bool bf16, cudaStream_t s) {
    // four feature channels per float4 chunk of the asset-major table: F = 5, 9, 13, 17 read feat_am directly, every other
    // F in [2, 17] needs the channel-padded copy feat_am4
    if (p.F < 2 || p.F > 17) return -100;
    const float* tbl = (p.F - 1) % 4 == 0 || p.F % 8 == 0 ? p.feat_am : p.feat_am4;   // F = 8, 16: dense scalar loads from feat_am
    if (!tbl || (p.F % 8 != 0 && ((uintptr_t)tbl) % 16 != 0)) return -100;
    const int c4 = (p.F + 2) / 4;                                     // ceil((F - 1) / 4)
    if (p.W > 64 || npl > 4 || p.A < 32) return -100;                 // A >= 32: a tile spans at most two envs
    if (((size_t)p.W * p.A) % 4 != 0 || ((uintptr_t)p.hist) % 16 != 0) return -100;   // every env's ring 16-byte aligned
    if ((size_t)p.A * p.T * c4 >= (1u << 31) || p.A >= 65536) return -100;
    const int per_sm = ctas_per_sm > 0 ? ctas_per_sm : 2;
    const int slots = pmrl_sm_count() * per_sm;
    const int gmax = npl <= 2 ? kRtGroupNarrow : kRtGroup;
    // a group's obs starts at env e0 = group · G; the bulk stores need it 16-byte aligned, which a bf16 env of A·W·F·2 bytes
    // (a multiple of 8 here) only guarantees for even G.  fp32 envs are multiples of 16 bytes: step 1, the heuristic as ever.
    const int gstep = ((size_t)p.A * p.W * p.F * (bf16 ? 2 : 4)) % 16 == 0 ? 1 : 2;
    int G = group > 0 ? group : pick_group(p.E, slots, gmax, gstep);
    if (G > gmax) G = gmax;
    p.group_envs = G;
    const int tr = c4 == 1 ? 32 : c4 == 2 ? 16 : 8;
    p.tile_assets = tr;
    // ring buffers: a tile may touch two envs, and the ring of env n+NB can only be requested once env n is
    // done — with two buffers a 50-asset env gets its ring one tile (≈2 us) before it is needed, less than a DRAM round
    // trip under load.  Narrow envs have small rings: keep up to four resident.
    const size_t budget = (size_t)(226 * 1024) / per_sm - 1024;
    const size_t esz = bf16 ? 2 : 4;                                  // obs element: the two tiles are bf16 or fp32 slab images
    const size_t fixed = (size_t)2 * tr * p.W * p.F * esz + (size_t)G * p.A * 8, ring_bytes = (size_t)p.W * p.A * 4;
    if (fixed + 2 * ring_bytes > budget) return -100;
    int nb = (int)((budget - fixed) / ring_bytes);
    p.ring_bufs = nb > 4 ? 4 : nb;
    const size_t smem = fixed + (size_t)p.ring_bufs * ring_bytes;
    const int n_groups = (p.E + G - 1) / G;
    const int grid = n_groups < slots ? n_groups : slots;
    const bool pad = (p.F - 1) % 4 != 0;
#define RT_CASE(N, V, C) if (npl == N && vec == V && c4 == C && !pad) \
        return bf16 ? launch_rt_w<true, N, V, C, false>(p, smem, grid, s) : launch_rt_w<false, N, V, C, false>(p, smem, grid, s)
#define RT_PAD(N, V, C) if (npl == N && vec == V && c4 == C && pad) \
        return bf16 ? launch_rt_w<true, N, V, C, true>(p, smem, grid, s) : launch_rt_w<false, N, V, C, true>(p, smem, grid, s)
    RT_CASE(1, 1, 1); RT_CASE(2, 1, 1); RT_CASE(2, 2, 1); RT_CASE(4, 1, 1); RT_CASE(4, 2, 1); RT_CASE(4, 4, 1);
    // wider feature sets and padded tables: the even / 16-byte asset maps only (odd asset counts take the two-kernel path)
    RT_CASE(2, 2, 2); RT_CASE(4, 2, 2); RT_CASE(4, 4, 2);
    RT_CASE(2, 2, 3); RT_CASE(4, 2, 3); RT_CASE(4, 4, 3);
    RT_CASE(2, 2, 4); RT_CASE(4, 2, 4); RT_CASE(4, 4, 4);
    RT_PAD(2, 2, 1); RT_PAD(4, 2, 1); RT_PAD(4, 4, 1);
    RT_PAD(2, 2, 2); RT_PAD(4, 2, 2); RT_PAD(4, 4, 2);
    RT_PAD(2, 2, 3); RT_PAD(4, 2, 3); RT_PAD(4, 4, 3);
    RT_PAD(2, 2, 4); RT_PAD(4, 2, 4); RT_PAD(4, 4, 4);
#undef RT_CASE
#undef RT_PAD
    return -100;
}
