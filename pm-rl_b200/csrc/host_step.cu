// host_step.cu — pmrl_env_step_host: one lockstep transition driven from HOST buffers.
//
// The reference's caller hands CPU tensors to TradingEnv.step and reads the reward back on the host
// (train/on_policy.py:64-65).  This entry point is that call for a batch: pinned actions in, reward/done out,
// it returns when the results are on the host.  Envs are independent, so the batch is issued as env slices:
// the host→device copy of slice c+1 runs on a copy stream under the kernel of slice c, and the device→host
// copy of slice c runs on a third stream under the kernel of slice c+1.  Slices grow geometrically (the H2D copy
// of N envs costs about a third of their kernel time over PCIe 5), which keeps the two exposed ends — the
// first copy in and the last copy out — a few tens of microseconds.
//
// When the action buffer is page-locked and mapped (cudaHostAlloc / cudaHostRegister / torch pin_memory: under
// unified addressing the kernel can dereference it), the default is better still: ONE kernel over the whole
// batch whose stepper warps read the actions straight from host memory over PCIe.  Each action is read exactly
// once (4 of the 1,208 algorithmic bytes per asset-step), so the PCIe reads hide under the HBM-bound obs fill
// and there are no slice boundaries at all (measured on config 4: 2.82 ms vs 2.94–3.0 ms sliced vs 3.72 serial).
#include <cuda_runtime.h>
#include <mutex>
#include <string.h>
#include "pmrl_b200.h"
#include "host_util.h"
#include "env_launch.h"

namespace {

constexpr int kMaxSlices = 32;
constexpr int kMaxDevices = 64;

constexpr int kMaxChunks = 64;

struct HostPipe {
    bool ready = false;
    std::mutex busy;                   // held for a whole sliced / streamed call: the streams, events and flags below are per device
    cudaStream_t copy_in = nullptr, copy_out = nullptr;
    cudaEvent_t start = nullptr, in_ev[kMaxSlices], k_ev[kMaxSlices];
    uint32_t* flags_dev = nullptr;     // [kMaxChunks] chunk-arrival flags of the streamed path (device memory)
    uint32_t* seq_src = nullptr;       // [kMaxChunks] page-locked source of the flag writes (all = the call's sequence number)
    uint32_t seq = 0;
};

int g_host_stream = 0, g_host_mirror = 1;

std::mutex g_mu;
HostPipe g_pipes[kMaxDevices];

// streams/events of the calling device, created on first use (the only state this library keeps; per device, lives
// for the process)
HostPipe* pipe_for_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return nullptr;
    std::lock_guard<std::mutex> lk(g_mu);
    HostPipe& p = g_pipes[dev];
    if (!p.ready) {
        if (cudaStreamCreateWithFlags(&p.copy_in, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
        if (cudaStreamCreateWithFlags(&p.copy_out, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
        if (cudaEventCreateWithFlags(&p.start, cudaEventDisableTiming) != cudaSuccess) return nullptr;
        for (int i = 0; i < kMaxSlices; ++i) {
            if (cudaEventCreateWithFlags(&p.in_ev[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
            if (cudaEventCreateWithFlags(&p.k_ev[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
        }
        if (cudaMalloc((void**)&p.flags_dev, kMaxChunks * sizeof(uint32_t)) != cudaSuccess) return nullptr;
        if (cudaMemset(p.flags_dev, 0, kMaxChunks * sizeof(uint32_t)) != cudaSuccess) return nullptr;
        if (cudaHostAlloc((void**)&p.seq_src, kMaxChunks * sizeof(uint32_t), cudaHostAllocDefault) != cudaSuccess) return nullptr;
        p.ready = true;
    }
    return &p;
}

// device-visible alias of a page-locked, mapped host pointer (cudaHostAlloc / cudaHostRegister / torch pin_memory), or null
template <typename T>
T* mapped_alias(const T* host) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, host) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer)
        return (T*)at.devicePointer;
    (void)cudaGetLastError();
    return nullptr;
}

// slice boundaries: slices > 0 → geometric growth ×2.5 from the first; slices < 0 → |slices| equal parts.
// Interior boundaries are multiples of 64 envs (keeps every slice's ring/obs base 16-byte aligned for any A).
int slice_bounds(int E, int slices, int* bounds) {
    int n = slices < 0 ? -slices : slices;
    if (n < 1) n = 1;
    if (n > kMaxSlices) n = kMaxSlices;
    double total = 0.0, w = 1.0;
    for (int i = 0; i < n; ++i) { total += w; if (slices > 0) w *= 2.5; }
    bounds[0] = 0;
    double acc = 0.0;
    w = 1.0;
    int m = 0;
    for (int i = 0; i < n; ++i) {
        acc += w;
        if (slices > 0) w *= 2.5;
        long long b = (i == n - 1) ? E : (long long)((double)E * acc / total);
        if (i != n - 1) b = (b / 64) * 64;
        if (b > E) b = E;
        if (b > bounds[m]) bounds[++m] = (int)b;
    }
    if (bounds[m] != E) bounds[++m] = E;
    return m;                                     // number of non-empty slices
}

#define PMRL_CUDA(call, what)                                                             \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) { pmrl_fail((int)e_, what); return (int)e_; }              \
    } while (0)

}  // namespace

void pmrl_set_host_stream(int value) { g_host_stream = value; }
void pmrl_set_host_mirror(int value) { g_host_mirror = value; }

extern "C" int pmrl_env_step_host(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st,
                                  const float* actions_host, float* actions_stage,
                                  float* reward, uint8_t* done, float* reward_host, uint8_t* done_host,
                                  float* obs, int32_t obs_mode, double* stats, int32_t slices, void* stream) {
    if (cfg && cfg->E == 0) return 0;
    if (!cfg || !tbl || !st || !actions_host || !actions_stage || !reward || !done || !reward_host || !done_host)
        return pmrl_fail(PMRL_E_ARG, "env_step_host: null argument");
    if (cfg->E <= 0 || cfg->A <= 0 || cfg->W <= 0 || cfg->F <= 0) return pmrl_fail(PMRL_E_SHAPE, "env_step_host: bad sizes");
    if (int rc = pmrl_check_obs_mode(obs_mode)) return rc;
    if (obs_mode != PMRL_OBS_NONE && !obs) return pmrl_fail(PMRL_E_ARG, "env_step_host: obs_mode set but obs is null");
    cudaStream_t s = (cudaStream_t)stream;
    const size_t A = (size_t)cfg->A, WA = (size_t)cfg->W * A;
    const size_t obs_env_bytes = WA * (size_t)cfg->F * ((obs_mode & PMRL_OBS_BF16) ? 2 : 4);   // bf16 obs: 2-byte elements

    if (slices == 0) {
        const float* act_dev = mapped_alias(actions_host);
        float* r_dev = mapped_alias(reward_host);
        uint8_t* d_dev = mapped_alias(done_host);
        const bool mirrored = g_host_mirror && r_dev && d_dev;   // the kernel writes reward / done straight into mapped host memory (posted PCIe writes)
        // Streaming vs zero-copy reads, measured on three boxes (tools/e2e_ab.py, alternating repetitions on one box): with the
        // obs materialised one box gave config 4 shard 2.773 → 2.738 ms and config 3 1.438 → 1.410 ms, two others gave equal
        // times at config 4 (2.81–2.89 ms in both modes) and streaming 2.5 % SLOWER at config 3; state-only steps are PCIe-bound
        // either way (131,072 x 100: 1.21 ms zero-copy vs 1.38 ms streamed; 262,144 x 500: 10.66 vs 9.94 ms); small batches lose
        // (4,096 x 50: 94 us vs 105 us).  No robust gain → zero-copy is the default and streaming stays an option.
        const size_t act_bytes = (size_t)cfg->E * A * sizeof(float);
        const size_t stream_from = (obs_mode & ~PMRL_OBS_BF16) == PMRL_OBS_FULL ? ((size_t)2 << 20) : ((size_t)128 << 20);
        if (act_dev && (g_host_stream == 2 || (g_host_stream == 1 && act_bytes >= stream_from))) {
            // streamed path (opt-in, PMRL_TUNE_HOST_STREAM): ONE kernel over the whole batch while the copy engine brings the action rows into
            // device memory chunk by chunk; every group of chunks is followed on the copy stream by its flag words, and
            // a warp waits for the flag of its env's chunk before it reads the row (PmrlStepIO.actions_ready).
            // The groups are taken in ascending env order, the copy runs at PCIe speed (52 MB in ≈1 ms at config 4) against
            // a 2.7 ms kernel, so only the first chunk is ever waited for.  Unlike zero-copy reads the step phase never pays a
            // PCIe round trip (L2 prefetch does not apply to host memory), and unlike the sliced pipeline there are no kernel
            // boundaries.  The flags carry a per-call sequence number, so they are never reset.
            HostPipe* hp = pipe_for_device();
            if (!hp) return pmrl_fail(PMRL_E_ARG, "env_step_host: could not create the copy streams");
            std::lock_guard<std::mutex> busy(hp->busy);
            int shift = 0;
            while (((cfg->E + (1 << shift) - 1) >> shift) > 32 || ((size_t)(1 << shift) * A * sizeof(float) < (256u << 10) && (1 << shift) < cfg->E)) ++shift;
            const int n = (cfg->E + (1 << shift) - 1) >> shift;
            if (n <= kMaxChunks) {
                if (++hp->seq == 0) hp->seq = 1;
                for (int c = 0; c < n; ++c) hp->seq_src[c] = hp->seq;
                PMRL_CUDA(cudaEventRecord(hp->start, s), "env_step_host: event record");
                PMRL_CUDA(cudaStreamWaitEvent(hp->copy_in, hp->start, 0), "env_step_host: stream wait");   // earlier work on s may still read the stage
                // The copies are enqueued BEFORE the kernel: a launch that blocks the host (a profiler or debugger serialising
                // kernels, CUDA_LAUNCH_BLOCKING=1) must find every chunk it will wait for already on its way.  They cover
                // 2, 4, 8, 18 chunks (a small first copy so the kernel finds its first rows on arrival, few large ones after it:
                // every copy and every flag write costs the copy engine and the host a fixed few microseconds).
                for (int c = 0, c1 = 0; c < n; c = c1) {
                    c1 = c == 0 ? 2 : c == 2 ? 6 : c == 6 ? 14 : n;
                    if (c1 > n) c1 = n;
                    const size_t lo = (size_t)c << shift;
                    const size_t hi = ((size_t)c1 << shift) < (size_t)cfg->E ? ((size_t)c1 << shift) : (size_t)cfg->E;
                    cudaError_t e1 = cudaMemcpyAsync(actions_stage + lo * A, actions_host + lo * A, (hi - lo) * A * sizeof(float), cudaMemcpyHostToDevice, hp->copy_in);
                    cudaError_t e2 = cudaMemcpyAsync(hp->flags_dev + c, hp->seq_src + c, (size_t)(c1 - c) * sizeof(uint32_t), cudaMemcpyHostToDevice, hp->copy_in);
                    if (e1 != cudaSuccess || e2 != cudaSuccess) {
                        cudaStreamSynchronize(hp->copy_in);
                        pmrl_fail((int)(e1 != cudaSuccess ? e1 : e2), "env_step_host: H2D action chunk");
                        return (int)(e1 != cudaSuccess ? e1 : e2);
                    }
                }
                PmrlStepIO io;
                memset(&io, 0, sizeof(io));
                io.actions = actions_stage; io.reward = reward; io.done = done; io.obs = obs; io.obs_mode = obs_mode; io.stats = stats;
                io.actions_ready = hp->flags_dev; io.actions_ready_seq = hp->seq; io.actions_ready_shift = shift;
                if (mirrored) { io.reward_host = r_dev; io.done_host = d_dev; }
                int rc = pmrl_env_step_io(cfg, tbl, st, &io, stream);
                if (rc != 0) { cudaStreamSynchronize(hp->copy_in); return rc; }
                if (!mirrored) {
                    PMRL_CUDA(cudaMemcpyAsync(reward_host, reward, (size_t)cfg->E * sizeof(float), cudaMemcpyDeviceToHost, s), "env_step_host: D2H reward");
                    PMRL_CUDA(cudaMemcpyAsync(done_host, done, (size_t)cfg->E, cudaMemcpyDeviceToHost, s), "env_step_host: D2H done");
                }
                PMRL_CUDA(cudaStreamSynchronize(s), "env_step_host: synchronize");
                PMRL_CUDA(cudaStreamSynchronize(hp->copy_in), "env_step_host: synchronize");   // (chunks of envs that only auto-reset are not waited for by the kernel)
                return 0;
            }
        }
        // zero-copy path: the kernel reads the mapped host actions itself over PCIe — ONE launch and ONE synchronisation
        if (act_dev) {
            PmrlStepIO io;
            memset(&io, 0, sizeof(io));
            io.actions = act_dev; io.reward = reward; io.done = done; io.obs = obs; io.obs_mode = obs_mode; io.stats = stats;
            if (mirrored) { io.reward_host = r_dev; io.done_host = d_dev; }
            int rc = pmrl_env_step_io(cfg, tbl, st, &io, stream);
            if (rc != 0) return rc;
            if (!mirrored) {
                PMRL_CUDA(cudaMemcpyAsync(reward_host, reward, (size_t)cfg->E * sizeof(float), cudaMemcpyDeviceToHost, s), "env_step_host: D2H reward");
                PMRL_CUDA(cudaMemcpyAsync(done_host, done, (size_t)cfg->E, cudaMemcpyDeviceToHost, s), "env_step_host: D2H done");
            }
            PMRL_CUDA(cudaStreamSynchronize(s), "env_step_host: synchronize");
            return 0;
        }
        // pageable actions: fall through to the copy pipeline
    }
    HostPipe* p = pipe_for_device();
    if (!p) return pmrl_fail(PMRL_E_ARG, "env_step_host: could not create the copy streams");
    std::lock_guard<std::mutex> busy(p->busy);        // one sliced call per device at a time (shared streams / events)
    int bounds[kMaxSlices + 2];
    const int n = slice_bounds(cfg->E, slices == 0 ? 5 : slices, bounds);
    // on any failure: drain what is already in flight on the caller's buffers before reporting it
    auto drain = [&](int rc) { cudaStreamSynchronize(p->copy_in); cudaStreamSynchronize(s); cudaStreamSynchronize(p->copy_out); return rc; };
#define PMRL_CUDA_DRAIN(call, what)                                                       \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) { pmrl_fail((int)e_, what); return drain((int)e_); }       \
    } while (0)

    PMRL_CUDA_DRAIN(cudaEventRecord(p->start, s), "env_step_host: event record");
    PMRL_CUDA_DRAIN(cudaStreamWaitEvent(p->copy_in, p->start, 0), "env_step_host: stream wait");   // earlier work on s may still read the stage
    for (int c = 0; c < n; ++c) {
        const int lo = bounds[c], cnt = bounds[c + 1] - lo;
        PMRL_CUDA_DRAIN(cudaMemcpyAsync(actions_stage + lo * A, actions_host + lo * A, (size_t)cnt * A * sizeof(float),
                                        cudaMemcpyHostToDevice, p->copy_in), "env_step_host: H2D actions");
        PMRL_CUDA_DRAIN(cudaEventRecord(p->in_ev[c], p->copy_in), "env_step_host: event record");
        PMRL_CUDA_DRAIN(cudaStreamWaitEvent(s, p->in_ev[c], 0), "env_step_host: stream wait");

        PmrlEnvCfg ccfg = *cfg;
        ccfg.E = cnt;
        PmrlEnvState cst = *st;
        cst.value = st->value + lo;
        cst.hist = st->hist + lo * WA;
        cst.idx = st->idx + lo;
        cst.is_full = st->is_full + lo;
        cst.t = st->t + lo;
        cst.t0 = st->t0 ? st->t0 + lo : nullptr;
        cst.sharpe = st->sharpe ? st->sharpe + 3 * (size_t)lo : nullptr;
        cst.ep_return = st->ep_return ? st->ep_return + lo : nullptr;
        int rc = pmrl_env_step(&ccfg, tbl, &cst, actions_stage + lo * A, nullptr, reward + lo, done + lo,
                               obs ? (float*)((char*)obs + lo * obs_env_bytes) : nullptr, obs_mode, stats, stream);
        if (rc != 0) return drain(rc);

        PMRL_CUDA_DRAIN(cudaEventRecord(p->k_ev[c], s), "env_step_host: event record");
        PMRL_CUDA_DRAIN(cudaStreamWaitEvent(p->copy_out, p->k_ev[c], 0), "env_step_host: stream wait");
        PMRL_CUDA_DRAIN(cudaMemcpyAsync(reward_host + lo, reward + lo, (size_t)cnt * sizeof(float), cudaMemcpyDeviceToHost, p->copy_out),
                        "env_step_host: D2H reward");
        PMRL_CUDA_DRAIN(cudaMemcpyAsync(done_host + lo, done + lo, (size_t)cnt, cudaMemcpyDeviceToHost, p->copy_out),
                        "env_step_host: D2H done");
    }
    PMRL_CUDA_DRAIN(cudaStreamSynchronize(p->copy_out), "env_step_host: synchronize");   // last D2H is behind the last kernel
#undef PMRL_CUDA_DRAIN
    return 0;
}
