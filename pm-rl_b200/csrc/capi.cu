// capi.cu — ABI version, error reporting and device-query helpers of libpmrl_b200.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>
#include <stddef.h>
#include "pmrl_b200.h"
#include "host_util.h"

#include <atomic>

static thread_local char g_err[256] = "";
static std::atomic<unsigned long long> g_launches{0};

int pmrl_fail(int code, const char* msg) {
    snprintf(g_err, sizeof(g_err), "pmrl_b200: %s", msg);
    return code;
}

int pmrl_check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (e == cudaSuccess) return 0;
    snprintf(g_err, sizeof(g_err), "pmrl_b200: launch of %s failed: %s", what, cudaGetErrorString(e));
    return (int)e;
}

int pmrl_sm_count(void) {
    static int cached[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

extern "C" uint64_t pmrl_launch_count(void) { return (uint64_t)g_launches.load(std::memory_order_relaxed); }
extern "C" int pmrl_abi_version(void) { return PMRL_ABI_VERSION; }
extern "C" const char* pmrl_last_error(void) { return g_err; }

// sizeof / selected field offsets of the boundary structs as compiled here (the ctypes mirror is checked against them)
extern "C" int pmrl_abi_sizeof(int32_t which) {
    switch (which) {
        case 0: return (int)sizeof(PmrlEnvCfg);
        case 1: return (int)sizeof(PmrlTables);
        case 2: return (int)sizeof(PmrlEnvState);
        case 3: return (int)sizeof(PmrlStepIO);
        case 4: return (int)sizeof(PmrlStartDist);
        case 100: return (int)offsetof(PmrlStepIO, stats);
        case 101: return (int)offsetof(PmrlStepIO, done_host);
        case 102: return (int)offsetof(PmrlEnvState, ticket);
        case 103: return (int)offsetof(PmrlEnvCfg, initial_cash);
        default: return -1;
    }
}
