// host_util.h — host-side helpers shared by the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <math.h>
#include "pmrl_b200.h"

// largest obs tile staged in shared memory by k_obs_build (fits the default 48 KB dynamic limit)
static const size_t kObsTileCapBytes = 40 * 1024;

int pmrl_fail(int code, const char* msg);          // records msg for pmrl_last_error(), returns code
int pmrl_check_launch(const char* what);           // cudaGetLastError() → 0 or positive cudaError_t
int pmrl_sm_count(void);                           // SMs of the current device (cached per device)

// obs_mode of the env entry points: PMRL_OBS_NONE / FULL / WEIGHTS, optionally | PMRL_OBS_BF16 and | PMRL_OBS_REL_OF(ref, mask)
// with FULL; F: obs channels of the env.  0, PMRL_E_ARG or PMRL_E_SHAPE.
static inline int pmrl_check_obs_mode(int obs_mode, int F) {
    const bool rel = obs_mode >= 0 && (obs_mode & PMRL_OBS_REL);
    const int rel_bits = PMRL_OBS_REL | (0xF << PMRL_OBS_REL_REF_SHIFT) | (0xFFFF << PMRL_OBS_REL_MASK_SHIFT);
    const int base = obs_mode & ~(PMRL_OBS_BF16 | (rel ? rel_bits : 0));
    if (base != PMRL_OBS_NONE && base != PMRL_OBS_FULL && base != PMRL_OBS_WEIGHTS) return pmrl_fail(PMRL_E_ARG, "bad obs_mode");
    if ((obs_mode & PMRL_OBS_BF16) && base != PMRL_OBS_FULL) return pmrl_fail(PMRL_E_ARG, "bad obs_mode: PMRL_OBS_BF16 needs PMRL_OBS_FULL");
    if (!rel) return 0;
    if (base != PMRL_OBS_FULL) return pmrl_fail(PMRL_E_ARG, "bad obs_mode: PMRL_OBS_REL needs PMRL_OBS_FULL");
    const int ref = (obs_mode >> PMRL_OBS_REL_REF_SHIFT) & 0xF;
    const unsigned mask = ((unsigned)obs_mode >> PMRL_OBS_REL_MASK_SHIFT) & 0xFFFFu;
    if (mask == 0u) return pmrl_fail(PMRL_E_ARG, "bad obs_mode: PMRL_OBS_REL with an empty channel mask");
    if (F - 1 > 16) return pmrl_fail(PMRL_E_SHAPE, "PMRL_OBS_REL covers at most 16 feature channels (F - 1 <= 16)");
    if (ref >= F - 1 || (mask >> (F > 1 ? F - 1 : 0)) != 0u)
        return pmrl_fail(PMRL_E_ARG, "bad obs_mode: PMRL_OBS_REL reference channel or mask bit outside the feature channels 0..F-2");
    return 0;
}

// per-period risk-free rate (1 + rf)^(1/periods) - 1 that the evaluation metrics subtract from every simple return
// (util/eval.py:14-24), evaluated in double like Python does; shared by the trace and the streaming metrics
static inline double pmrl_rf_period(float rf, int periods) {
    return rf != 0.0f ? pow(1.0 + (double)rf, 1.0 / (double)periods) - 1.0 : 0.0;
}
