// obs_tile.cuh — build one observation tile obs[e, a0:a0+na, :, :] in shared memory and stream it out.
//
// Restates the sliding-window gather + weight-channel overwrite of the reference:
//   window rows [i, i+W) per asset          data/instrument.py:351-356
//   features[:, :, -1] = weights.get_all()  env/sim/trading_env.py:32,103
//   get_all(): not full → zero front padding + chronological rows; full → raw ring order (quirk Q8)
//                                           env/sim/weight_buffer.py:32-44
// The tile is the exact byte image of the [na, W, F] slab of the reference obs layout, so it leaves
// the SM as one contiguous TMA bulk store (cp.async.bulk shared::cta → global).  OT is the obs element type: float, or
// uint16_t holding bf16 bits (PMRL_OBS_BF16: each element rounded from the fp32 value as the tile is filled).
#pragma once
#include "pmrl_device.cuh"

namespace pmrl {

// Feature channels 0..F-2 of the tile from the asset-major table (rows row0 .. row0+W-1).  REL (PMRL_OBS_REL): the channels
// in rel.mask are divided by channel rel.ref of row row0+W-1 of their asset (rel_quot: the bits of IEEE division).
template <typename OT, bool REL = false>
__device__ __forceinline__ void obs_tile_fill_features(const StepParams& p, OT* __restrict__ tile,
                                                       int a0, int na, int row0, int tid, int nthreads,
                                                       const ObsRel& rel = ObsRel{0, 0u}) {
    const int W = p.W, F = p.F, Fm1 = p.F - 1, T = p.T;
    const uint64_t pol_keep = l2_policy_evict_last();
    if (Fm1 == 4) {
        // one float4 (o,h,l,c) per (asset,row); consecutive threads walk consecutive rows of one asset:
        // 16-byte coalesced loads of an 800-byte run, stride-5 conflict-free shared stores.
        const float4* __restrict__ tbl = reinterpret_cast<const float4*>(p.feat_am);
        const int n = na * W;
        for (int r = tid; r < n; r += nthreads) {
            const int al = r / W, w = r - al * W;
            float4 v = ld_keep4(tbl + (size_t)(a0 + al) * T + row0 + w, pol_keep);
            if constexpr (REL) {        // the divisor row: the same 16 bytes for the W threads of one asset (L1 hits)
                const float b = f4_get(ld_keep4(tbl + (size_t)(a0 + al) * T + row0 + W - 1, pol_keep), rel.ref);
                const bool b_ok = unidiv_in_range(b);
                const UniDiv dv = unidiv_make(b);
                if (rel.mask & 1u) v.x = rel_quot(v.x, b, dv, b_ok);
                if (rel.mask & 2u) v.y = rel_quot(v.y, b, dv, b_ok);
                if (rel.mask & 4u) v.z = rel_quot(v.z, b, dv, b_ok);
                if (rel.mask & 8u) v.w = rel_quot(v.w, b, dv, b_ok);
            }
            OT* d = tile + r * 5;
            d[0] = obs_cvt<OT>(v.x); d[1] = obs_cvt<OT>(v.y); d[2] = obs_cvt<OT>(v.z); d[3] = obs_cvt<OT>(v.w);
        }
    } else {
        // any channel count: a warp owns an asset row of the tile (its window is ONE contiguous run of W·(F-1) floats in
        // the asset-major table), lanes walk the run 32 floats at a time — coalesced 128-byte loads — and carry their
        // (window row, channel) position incrementally: no integer division per element.
        const int per_asset = W * Fm1;
        const int lane = tid & 31, warp = tid >> 5, nwarps = nthreads >> 5;
        const int dq = 32 / Fm1, dr = 32 - dq * Fm1;               // a stride of 32 floats = dq rows + dr channels
        const int w_first = lane / Fm1, c_first = lane - w_first * Fm1;
        for (int al = warp; al < na; al += nwarps) {
            const float* __restrict__ src = p.feat_am + ((size_t)(a0 + al) * T + row0) * Fm1;
            OT* __restrict__ drow = tile + al * W * F;
            float b = 0.0f;
            bool b_ok = false;
            UniDiv dv = {0.0f, 0.0f};
            if constexpr (REL) {        // one broadcast load of the divisor per asset row
                b = ld_keep(src + (W - 1) * Fm1 + rel.ref, pol_keep);
                b_ok = unidiv_in_range(b);
                dv = unidiv_make(b);
            }
            int w = w_first, c = c_first;
            for (int rem = lane; rem < per_asset; rem += 32) {
                float x = ld_keep(src + rem, pol_keep);
                if constexpr (REL) { if ((rel.mask >> c) & 1u) x = rel_quot(x, b, dv, b_ok); }
                drow[w * F + c] = obs_cvt<OT>(x);
                w += dq; c += dr;
                if (c >= Fm1) { c -= Fm1; ++w; }
            }
        }
    }
}

// Weight channel F-1 of the tile from the ring (get_all semantics).  `fresh`/`fresh_slot`: optional
// shared-memory copy of the row written by this very step (fused kernel), else fresh_slot = -1.
template <typename OT>
__device__ __forceinline__ void obs_tile_fill_weights(const StepParams& p, OT* __restrict__ tile,
                                                      const float* __restrict__ hist_e, int a0, int na,
                                                      int idx, int is_full,
                                                      const float* __restrict__ fresh, int fresh_slot,
                                                      int tid, int nthreads) {
    const int W = p.W, F = p.F, A = p.A;
    const int shift = is_full ? 0 : (W - idx);      // column w shows ring slot w - shift (weight_buffer.py:38-42)
    const int lane = tid & 31, warp = tid >> 5, nwarps = nthreads >> 5;
    for (int w = warp; w < W; w += nwarps) {          // lanes over assets → coalesced ring-row reads, no division per element
        const int slot = w - shift;
        for (int al = lane; al < na; al += 32) {
            float v = 0.0f;
            if (slot >= 0) v = (slot == fresh_slot) ? fresh[a0 + al] : ld_stream(hist_e + (size_t)slot * A + a0 + al);
            tile[(al * W + w) * F + (F - 1)] = obs_cvt<OT>(v);
        }
    }
}

// Tile → obs.  mode FULL: whole slab (bulk store when aligned); mode WEIGHTS: channel F-1 only.
// All threads of the CTA call this after `fence_proxy_async_smem(); __syncthreads();` following the
// fills (every writer fences its own generic-proxy stores before the barrier, then one thread issues
// the async-proxy bulk store).  WEIGHTS mode is fp32 only.
template <typename OT>
__device__ __forceinline__ void obs_tile_store(const StepParams& p, const OT* __restrict__ tile,
                                               int e, int a0, int na, int tid, int nthreads) {
    const int W = p.W, F = p.F;
    OT* __restrict__ dst = reinterpret_cast<OT*>(p.obs) + ((size_t)e * p.A + a0) * W * F;
    const int n = na * W * F;
    if (p.obs_mode == PMRL_OBS_FULL) {
        if (p.obs_bulk_ok) {
            if (tid == 0) {
                bulk_store_s2g(dst, tile, (uint32_t)n * (uint32_t)sizeof(OT), l2_policy_evict_first());
                bulk_commit();
            }
        } else {
            for (int q = tid; q < n; q += nthreads) dst[q] = tile[q];
        }
    } else {  // PMRL_OBS_WEIGHTS
        const int rows = na * W;
        for (int r = tid; r < rows; r += nthreads) dst[(size_t)r * F + (F - 1)] = tile[r * F + (F - 1)];
    }
}

}  // namespace pmrl
