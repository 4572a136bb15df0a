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

// obs_mode of the env entry points: PMRL_OBS_NONE / FULL / WEIGHTS, optionally | PMRL_OBS_BF16 with FULL.  0 or PMRL_E_ARG.
static inline int pmrl_check_obs_mode(int obs_mode) {
    const int base = obs_mode & ~PMRL_OBS_BF16;
    if (base != PMRL_OBS_NONE && base != PMRL_OBS_FULL && base != PMRL_OBS_WEIGHTS) return pmrl_fail(PMRL_E_ARG, "bad obs_mode");
    if ((obs_mode & PMRL_OBS_BF16) && base != PMRL_OBS_FULL) return pmrl_fail(PMRL_E_ARG, "bad obs_mode: PMRL_OBS_BF16 needs PMRL_OBS_FULL");
    return 0;
}

// per-period risk-free rate (1 + rf)^(1/periods) - 1 that the evaluation metrics subtract from every simple return
// (util/eval.py:14-24), evaluated in double like Python does; shared by the trace and the streaming metrics
static inline double pmrl_rf_period(float rf, int periods) {
    return rf != 0.0f ? pow(1.0 + (double)rf, 1.0 / (double)periods) - 1.0 : 0.0;
}
