/*
 * pmrl_b200.h — C-ABI of libpmrl_b200.so: the B200 (sm_100a) implementation of the
 * pm-rl portfolio-environment hot path, batched over E lockstep environments.
 *
 * Every entry point is `extern "C"`, takes plain device pointers + sizes + a CUDA
 * stream handle (as void*), enqueues work on that stream and returns immediately
 * (no host sync, no allocation, no global state; graph-capturable).  Return value:
 * 0 = ok, negative = PMRL_E_* (argument/shape problem, nothing was launched),
 * positive = a cudaError_t from the launch.  `pmrl_last_error()` gives the text.
 *
 * Reference interfaces replaced (all paths relative to the pm-rl tree):
 *   pmrl_env_reset      <- TradingEnv.reset              env/sim/trading_env.py:21-41
 *                          ActionBuffer.reset            env/sim/weight_buffer.py:46-50
 *   pmrl_env_step       <- TradingEnv.step               env/sim/trading_env.py:44-105
 *   pmrl_env_step_host  <- the same call with CPU tensors train/on_policy.py:64-65
 *   pmrl_price_relatives<- y = close / close.shift(1)        data/instrument.py:79
 *                          ActionBuffer.update/get_last  env/sim/weight_buffer.py:13-30
 *                          ActionBuffer.get_all          env/sim/weight_buffer.py:32-44
 *                          Reward.get_reward & variants  env/reward.py:15-31
 *                          y_t = close_t/close_{t-1}     data/instrument.py:79
 *                          window rows [i, i+W)          data/instrument.py:351-356
 *   pmrl_obs_build      <- features[:, :, -1] = weights.get_all()   trading_env.py:32,103
 *   pmrl_ffd_weights    <- FixedFracDiff._objective (weights/width) data/ffd.py:38-47
 *   pmrl_ffd_transform  <- FixedFracDiff.transform       data/ffd.py:80-89
 *   pmrl_scale_series   <- Instrument.scale              data/instrument.py:318-336
 *   pmrl_pack_features  <- Instrument.window / get_feature_tensor layout (instrument.py:339-356)
 *   pmrl_indicators     <- Instrument.add_indicators (TA-Lib windows)     data/instrument.py:207-232, config/base.py:30-44
 *   pmrl_rollout_add    <- RolloutBuffer.add             replay/rollout_buffer.py:43-57
 *   pmrl_rollout_gather <- RolloutBuffer.sample[_random] replay/rollout_buffer.py:59-142
 *   pmrl_replay_add     <- ReplayBuffer.add              replay/buffer.py:23-37, replay/traj_buffer.py:26-43
 *   pmrl_replay_gather  <- ReplayBuffer.sample           replay/buffer.py:39-79, replay/traj_buffer.py:45-89
 *   pmrl_pg_reward_*    <- PG._reward (fwd + grad wrt a) agent/pg/pg.py:40-82
 *   pmrl_eval_metrics   <- Metrics.sharpe/sortino/mdd/average_turnover  util/eval.py:14-37
 *   pmrl_eval_stream_*  <- the same metrics, accumulated per step   util/eval.py:14-37
 *   pmrl_env_draw_starts<- the loader's episode start (every reset replays one fixed offset t0[e] otherwise);
 *                          random starts as in online stochastic batch learning (Jiang, Xu & Liang 2017) and the
 *                          recency-weighted sampling of replay/buffer.py (PERCENT_LATEST)
 *
 * Device data layout (all fp32 unless noted; E = envs on this GPU, A = assets incl.
 * cash at index 0, W = window, F = obs channels incl. the weight slot which is LAST):
 *   y_tm     [T, A]        time-major price relatives y_t[a] = close[t,a] / close[t-1,a] (pmrl_price_relatives)
 *   feat_am  [A, T, F-1]   asset-major feature table (OHLC, or FFD'ed + scaled series)
 *   value    [E]           portfolio value V
 *   hist     [E, W, A]     ring of post-drift weights (reference ActionBuffer.buffer per env)
 *   idx      [E] i32       ring write pointer;  is_full [E] u8;  t [E] i32 local step k
 *   t0       [E] i32       episode offset: at local step k the env sees table rows
 *                          [t0+k, t0+k+W) and the price relative of row t0+k+W-1
 *   obs      [E, A, W, F]  reference observation layout (net/lsre_cann.py:105); fp32, or bf16 bit patterns with
 *                          PMRL_OBS_BF16 (everything else stays fp32)
 */
#ifndef PMRL_B200_H
#define PMRL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PMRL_ABI_VERSION 5   /* 5: PmrlTables.feat_am4 (channel-padded feature table: fused kernel for any F <= 17);
                                3: PmrlEnvState.ticket, PmrlStepIO + pmrl_env_step_io, pmrl_env_step_burst, pmrl_rollout_gather_index;
                                4: PmrlStepIO.actions_ready (action rows streamed in under the kernel) */

/* error codes (negative) */
#define PMRL_E_ARG        (-1)   /* null pointer / bad enum */
#define PMRL_E_SHAPE      (-2)   /* unsupported or inconsistent sizes */
#define PMRL_E_ALIGN      (-3)   /* pointer alignment requirement not met */

/* reward_mode (env/reward.py:15-18, trading_env.py:93-99) */
#define PMRL_REWARD_STEP_LOG    0   /* ln(V'/V_post_mu) * scale  — what TradingEnv.step returns (:99) */
#define PMRL_REWARD_RETURNS     1   /* Reward.returns      (env/reward.py:20-21) */
#define PMRL_REWARD_LOG_RETURNS 2   /* Reward.log_returns  (env/reward.py:23-24) */
#define PMRL_REWARD_SHARPE      3   /* Reward.sharpe_ratio (env/reward.py:26-31), running over the episode */

/* cfg.flags */
#define PMRL_FLAG_STRICT_REFERENCE 1u  /* reproduce quirk Q1: normalise only if (!isclose(sum,1) AND min<0).
                                          cleared: OR-condition + max-subtracted softmax (agent/pg/pg.py:52-53) */

/* obs_mode of pmrl_env_step / pmrl_env_reset */
#define PMRL_OBS_NONE    0   /* state-only step ("Mode S") */
#define PMRL_OBS_FULL    1   /* gather feature window + weight channel into obs ("Mode O") */
#define PMRL_OBS_WEIGHTS 2   /* overwrite only channel F-1 of a caller-filled obs (compat shim; trading_env.py:103) */
#define PMRL_OBS_BF16    0x100  /* OR-ed into PMRL_OBS_FULL only (pmrl_env_reset, pmrl_env_step, PmrlStepIO.obs_mode,
                                   pmrl_env_step_host, pmrl_obs_build): the `float* obs` argument then points to [E, A, W, F]
                                   uint16_t bf16 bit patterns, each the round-to-nearest-even (cvt.rn.bf16.f32) of the fp32 value
                                   the plain FULL mode writes; half the obs bytes.  State, tables, reward, done, stats and sinks
                                   stay fp32 and bit-identical to an fp32 run.  Accepted for exactly the shapes FULL accepts;
                                   WEIGHTS | BF16, NONE | BF16 and unknown bits fail with PMRL_E_ARG before any launch.  A library
                                   built before this flag rejects it with "bad obs_mode" (PMRL_E_ARG): that is how a binding
                                   detects support (PMRL_ABI_VERSION is unchanged). */

typedef struct PmrlEnvCfg {
    int32_t E, A, W, F;        /* envs on this device, assets, window, obs channels (weight slot = F-1) */
    int32_t T;                 /* rows of y_tm / feat_am */
    int32_t episode_len;       /* L_ep: done when local step == L_ep; <= 0 → episodes never end */
    int32_t reward_mode;       /* PMRL_REWARD_* */
    int32_t mu_max_iter;       /* cap on the commission fixed-point iterations (trading_env.py:70) */
    uint32_t flags;            /* PMRL_FLAG_* */
    float initial_cash;        /* config/base.py:47 INITIAL_CASH */
    float commission;          /* config/base.py:48 COMISSION [sic] */
    float reward_scale;        /* config/base.py:52 REWARD_SCALE */
    float risk_free;           /* config/base.py:53 RISK_FREE_RATE */
} PmrlEnvCfg;

typedef struct PmrlTables {
    const float* y_tm;         /* [T, A] price relatives y[t] = close[t] / close[t-1] (row 0 = 1) built by
                                  pmrl_price_relatives from the time-major close plane, or NULL when y is supplied externally */
    const float* feat_am;      /* [A, T, F-1] or NULL when obs_mode != PMRL_OBS_FULL */
    const float* feat_am4;     /* optional: the same table with every (asset, row) padded to a multiple of four channels,
                                  [A, T, 4*ceil((F-1)/4)], 16-byte aligned (pad values are never copied to obs).  With it the
                                  fused step+obs kernel covers every F in [2, 17]; without it only (F-1) % 4 == 0, other widths
                                  take the state-only step followed by the obs tile kernel.  NULL → not provided. */
} PmrlTables;

typedef struct PmrlEnvState {
    float*    value;           /* [E] */
    float*    hist;            /* [E, W, A] */
    int32_t*  idx;             /* [E] */
    uint8_t*  is_full;         /* [E] */
    int32_t*  t;               /* [E] */
    const int32_t* t0;         /* [E] (may be NULL when y_ext is used and obs_mode != FULL) */
    double*   sharpe;          /* [E, 3] running (n, mean, M2) of gross returns; required for PMRL_REWARD_SHARPE */
    float*    ep_return;       /* [E] running sum of rewards in the episode; required when stats != NULL */
    uint32_t* ticket;          /* [2] zero-initialised work counters of THIS env batch ({next env group, CTAs finished}; the fused
                                  step+obs kernel hands its env groups out through them and re-zeroes them before it exits), or
                                  NULL → static group stride.  Owned by the batch, not by the library, so launches of different
                                  env batches on different streams (eager or inside captured graphs) never share a counter;
                                  launches of ONE batch must be stream-ordered anyway (they update the same state). */
} PmrlEnvState;

/* Per-step inputs / outputs of pmrl_env_step_io.  Zero-initialise, then set what is used. */
typedef struct PmrlStepIO {
    const float* actions;      /* [E, A] raw scores or weights */
    const float* y_ext;        /* [E, A] external price relatives or NULL → table row t0+k+W-1 */
    float*    reward;          /* [E] out */
    uint8_t*  done;            /* [E] out */
    float*    obs;             /* [E, A, W, F] out (FULL), in/out (WEIGHTS), NULL (NONE) */
    int32_t   obs_mode;        /* PMRL_OBS_* */
    double*   stats;           /* [PMRL_STATS_LEN] or NULL */
    /* optional sinks: rows of a rollout / replay buffer slot written by the step kernel itself instead of by a separate
     * copy (replay/rollout_buffer.py:51-57 stores a, v, r; replay/buffer.py:31-37 stores i, a, r) — `reward` may point
     * straight at the r row of the slot, `obs` at s[slot + 1] */
    float*    action_sink;     /* [E, A] raw action as received */
    float*    value_sink;      /* [E] portfolio value after the step (train/on_policy.py:65 stores env.value) */
    float*    weight_sink;     /* [E, A] post-drift weights w' of this step: the un-wrapped weight history an index-mode rollout
                                  buffer regenerates the obs weight channel from (pmrl_rollout_gather_index) */
    int32_t*  index_sink;      /* [E] loader item index t0 + k of this step (train/off_policy.py:87) */
    /* optional host mirrors: device-visible addresses of page-locked mapped host memory (cudaHostGetDevicePointer);
     * the kernel writes reward / done there as well (posted PCIe writes), so a host caller needs no D2H copy */
    float*    reward_host;     /* [E] or NULL */
    uint8_t*  done_host;       /* [E] or NULL (set together with reward_host) */
    /* optional: the action rows arrive WHILE the kernel runs (pmrl_env_step_host streams them in with the copy engine under the
     * kernel): actions_ready[c] becomes == actions_ready_seq (a release by the writer: copy-engine stream order) once the rows
     * of envs [c << actions_ready_shift, (c + 1) << actions_ready_shift) are in `actions`; a warp waits for its env's flag
     * before it reads the row (bounded: a flag that never arrives traps instead of hanging the GPU).  NULL → all rows are in
     * `actions` when the kernel starts. */
    const uint32_t* actions_ready;
    uint32_t  actions_ready_seq;
    int32_t   actions_ready_shift;
} PmrlStepIO;

/* stats vector written by pmrl_env_step (accumulated with atomics; caller zeroes it) */
#define PMRL_STATS_LEN 10
#define PMRL_STAT_N_ENVS     0   /* envs that took a real step */
#define PMRL_STAT_SUM_R      1
#define PMRL_STAT_SUM_R2     2
#define PMRL_STAT_SUM_V      3
#define PMRL_STAT_SUM_LNV    4
#define PMRL_STAT_N_DONE     5
#define PMRL_STAT_SUM_EPRET  6   /* Σ episode return over envs that finished this step */
#define PMRL_STAT_SUM_EPLEN  7
#define PMRL_STAT_MAX_V      8   /* max V   (caller initialises to -inf) */
#define PMRL_STAT_MAX_NEGV   9   /* max −V  (caller initialises to -inf) → min V = −this */

int         pmrl_abi_version(void);
/* sizeof of a boundary struct as compiled into the library (0 PmrlEnvCfg, 1 PmrlTables, 2 PmrlEnvState, 3 PmrlStepIO,
 * 4 PmrlStartDist; 100+:
 * selected field offsets) — lets a foreign-language binding verify its mirror of the structs; -1 for an unknown code. */
int         pmrl_abi_sizeof(int32_t which);
const char* pmrl_last_error(void);

/* Launch-shape tuning hook (process-wide; for benchmarking the kernel variants, not part of the reference surface).
 * value <= 0 restores the built-in heuristic. */
#define PMRL_TUNE_GROUP_ENVS  2   /* envs a CTA advances together (1..16) */
#define PMRL_TUNE_CTAS_PER_SM 3   /* persistent CTAs per SM of the fused step+obs kernel; for the staged wide-env step: 3 = three 8-warp CTAs
                                     with single-stage rows (default: two CTAs, double-buffered rows) */
#define PMRL_TUNE_FUSED       4   /* 1 (default): fused step+obs kernel where one covers the shape, else k_env_step followed by the
                                     obs tile kernel; 0: always the two kernels */
#define PMRL_TUNE_FAST_FILL   5   /* 1 (default): specialised obs kernels (fused RT / register-staged, division-free tile fill);
                                     0: generic k_obs_build after the state-only step */
#define PMRL_TUNE_RING_TMA    11  /* 1 (default): fused kernel that loads each env's weight ring with one TMA bulk copy
                                     (env_step_rt.cu); 2: the same without the next-group L2 prefetch; 0: register ring loads
                                     (env_step_fast.cu) */
#define PMRL_TUNE_STAGED      12  /* 1 (default): state-only step of wide envs (A > 128, A % 4 == 0) with the action / previous-weight /
                                     price-relative rows staged one env ahead through shared memory by TMA bulk copies
                                     (env_step_staged.cu) when a warp has more than one env; 2: also for small batches; 0: register loads +
                                     L2 prefetch (k_env_step) */
#define PMRL_TUNE_HOST_STREAM 13  /* pmrl_env_step_host with page-locked actions: 0 (default) zero-copy, the kernel reads the host buffer
                                     over PCIe itself; 1: the copy engine streams the action rows into device memory in chunks under
                                     the kernel, which waits per chunk (PmrlStepIO.actions_ready), for batches of >= 2 MB of actions
                                     with the obs materialised (>= 128 MB state-only); 2: streamed at any size.  Measured equal
                                     within the run-to-run spread (DESIGN.md §3.1), hence not the default */
#define PMRL_TUNE_HOST_MIRROR 14  /* pmrl_env_step_host with page-locked result buffers: 1 the kernel writes reward / done straight into
                                     the mapped host buffers; 0 two device→host copies after the kernel */
int pmrl_set_tuning(int32_t key, int32_t value);

/* Kernels this library has launched in this process so far (every entry point counts its own launches; bench.py reports
 * the difference over its timed region as `gpu_launches`). */
uint64_t pmrl_launch_count(void);

/* Re-initialise the envs with mask[e] != 0 (mask == NULL → all): V ← initial_cash, ring ← 0 with
 * hist[e,0,0] = 1, idx ← 1, is_full ← 0, t ← 0, sharpe/ep_return cleared.  If obs_mode != NONE the
 * obs of the (re)initialised envs is written (window rows [t0, t0+W) + reset weight channel). */
int pmrl_env_reset(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st,
                   const uint8_t* mask, float* obs, int32_t obs_mode, void* stream);

/* One lockstep transition of all E envs.
 *   actions [E, A]  raw scores or weights (normalised in-kernel like trading_env.py:58-60)
 *   y_ext   [E, A]  externally supplied price relatives, or NULL → row t0+k+W-1 of tbl->y_tm
 *   reward  [E]     out;  done [E] u8 out (local step reached episode_len)
 *   obs             out [E,A,W,F] (FULL), in/out (WEIGHTS), or NULL (NONE)
 *   stats           double[PMRL_STATS_LEN] device vector or NULL
 * An env whose local step already equals episode_len on entry is auto-reset instead of stepped
 * (reward 0, done 0, action ignored) — the reference loop's `if step == 0: env.reset(data)`
 * (train/on_policy.py:60-61). */
int pmrl_env_step(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st,
                  const float* actions, const float* y_ext,
                  float* reward, uint8_t* done, float* obs, int32_t obs_mode,
                  double* stats, void* stream);

/* The same transition with the optional sinks / host mirrors of PmrlStepIO (pmrl_env_step is this call with none set). */
int pmrl_env_step_io(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st,
                     const PmrlStepIO* io, void* stream);

/* K consecutive state-only transitions in ONE launch on pre-supplied actions — imagination rollouts advance in fixed
 * bursts (HORIZON = 15, config/dreamer.py:54; agent/dreamer/dreamer.py:104-158).  actions [K, E, A], reward [K, E],
 * done [K, E]; price relatives come from tbl->y_tm.  Bit-identical to K calls of pmrl_env_step with obs_mode NONE
 * (auto-resets included); each env's scalar state and newest weight row stay in registers across the burst. */
int pmrl_env_step_burst(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st,
                        const float* actions, int32_t K, float* reward, uint8_t* done,
                        double* stats, void* stream);

/* The same transition driven from HOST buffers — the call the reference's loop makes with CPU tensors
 * (`r, obs = env.step(action, …)` then `env.value` read on the host, train/on_policy.py:64-65).
 *   actions_host [E, A]  host (pinned for overlap) in;  actions_stage [E, A] device staging buffer (caller-owned)
 *   reward/done          device buffers as in pmrl_env_step;  reward_host [E] f32 / done_host [E] u8  host out
 *   slices  0 (default): page-locked mapped actions_host → one kernel reads them in place over PCIe (zero-copy);
 *                pageable → as slices = 5.   > 0: that many env slices growing ×2.5 (the H2D copy of slice c+1 and
 *                the D2H copy of slice c-1 run under the kernel of slice c);  < 0: |slices| equal slices
 * Unlike every other entry point this one BLOCKS until reward_host/done_host are written (it is not
 * graph-capturable) and keeps two copy streams per device, created on first use. */
int pmrl_env_step_host(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st,
                       const float* actions_host, float* actions_stage,
                       float* reward, uint8_t* done, float* reward_host, uint8_t* done_host,
                       float* obs, int32_t obs_mode, double* stats, int32_t slices, void* stream);

/* y_tm[t, a] = close_tm[t, a] / close_tm[t-1, a] (data/instrument.py:79: `close / close.shift(1)`), row 0 = 1.
 * Builds PmrlTables.y_tm: the reference divides once per loader item on the host, the step kernels read the quotient.
 * close_tm, y_tm [T, A]; the two must not alias (row t reads close row t-1). */
int pmrl_price_relatives(const float* close_tm, int32_t T, int32_t A, float* y_tm, void* stream);

/* Self-test of the kernels' shared-divisor quotient against IEEE division: den[i / 32] divides num[i] (n numerators,
 * ceil(n/32) divisors, device pointers); out[0] += pairs whose bits differ, out[1] += pairs tested (operands outside
 * the range in which the kernels use the shared-divisor form are skipped).  out: uint64[2] device, caller-zeroed. */
int pmrl_selftest_division(const float* num, const float* den, int64_t n, uint64_t* out, void* stream);

/* Materialise obs for the current state without stepping (obs_mode FULL or WEIGHTS). */
int pmrl_obs_build(const PmrlEnvCfg* cfg, const PmrlTables* tbl, const PmrlEnvState* st,
                   float* obs, int32_t obs_mode, void* stream);

/* ---- feature path (data/ffd.py, data/instrument.py) ---- */

/* Binomial FFD weights per series: w[n,0]=1, w[n,k]=w[n,k-1]*(1-(d[n]+1)/k) (sequential product in a double accumulator rounded to fp32 per prefix, like torch.cumprod on the CPU;
 * ffd.py:38-40; d is a host-precision double like the reference's Python float, rounded to fp32 after
 * the +1); widths[n] = max{k : |w[n,k]| > thres} (ffd.py:43).  d [N] f64 (device), weights [N, T], widths [N] i32. */
int pmrl_ffd_weights(const double* d, int32_t N, int32_t T, float thres,
                     float* weights, int32_t* widths, void* stream);

/* Valid convolution with the first widths[n] taps (the tap at index width is dropped, ffd.py:47),
 * tail-aligned to T - max_width outputs (ffd.py:81-88):
 *   out[n, j] = Σ_{k<width_n} w[n,k] · x[n, max_width + j − k],  j ∈ [0, T−max_width)
 * Series with d[n] <= 0 are copied (x[n, max_width + j]).  x [N, T], out [N, T − max_width]. */
int pmrl_ffd_transform(const float* x, const double* d, const float* weights, const int32_t* widths,
                       int32_t N, int32_t T, int32_t max_width, float* out, void* stream);

/* Per-series scaling over [0, L): method 0 = min-max (x−min)/(max−min), 1 = standard (x−mean)/std (population
 * std), constant series follow sklearn (scale treated as 1).  In place allowed (out == x).  x [N, L]. */
int pmrl_scale_series(const float* x, int32_t N, int32_t L, int32_t method, float* out, void* stream);

/* Pack series-major planes into the two table layouts the env kernels read:
 *   series [A*C, L] (series index = a*C + c)  →  feat_am [A, L, C];  close [A, L] → close_tm [L, A]. */
int pmrl_pack_features(const float* series, const float* close, int32_t A, int32_t C, int32_t L,
                       float* feat_am, float* close_tm, void* stream);

/* Technical-indicator windows (data/instrument.py:207-232; TA-Lib's published algorithms in double precision, outputs
 * fp32 with NaN over each indicator's lookback — TA-Lib is not vendored: parity UNPINNED).
 * specs: HOST array [n_specs, 2] of (PMRL_IND_*, period); series [A*C, L] with channels o,h,l,c[,v] (index a*C + c);
 * out [A, n_out, L] where n_out / the maximum lookback come from pmrl_indicator_layout (BBANDS: upper, middle, lower;
 * MACD 12/26/9: macd, signal, hist; STOCH 5/3/3: slowk, slowd; the others one output). */
#define PMRL_IND_SMA    0
#define PMRL_IND_EMA    1
#define PMRL_IND_RSI    2
#define PMRL_IND_ATR    3
#define PMRL_IND_BBANDS 4
#define PMRL_IND_MACD   5
#define PMRL_IND_OBV    6   /* needs the volume channel (C >= 5) */
#define PMRL_IND_ADOSC  7   /* 3 / 10; needs the volume channel */
#define PMRL_IND_CCI    8
#define PMRL_IND_STOCH  9   /* 5 / 3 / 3: slowk, slowd */
#define PMRL_IND_DX     10  /* Wilder directional movement index */
#define PMRL_IND_ADX    11  /* Wilder-smoothed DX */
int pmrl_indicator_layout(const int32_t* specs, int32_t n_specs, int32_t* n_out, int32_t* lookback);
int pmrl_indicators(const float* series, int32_t A, int32_t C, int32_t L, const int32_t* specs, int32_t n_specs,
                    float* out, void* stream);

/* ---- buffers (replay/rollout_buffer.py, replay/buffer.py, replay/traj_buffer.py) ---- */

/* On-policy store, batched over envs: slot = step − (W−1) when step > W−1 (rollout_buffer.py:51-57).
 * Buffers: s [S, E, A, W, F], a [S, E, A], v [S, E], r [S, E].  Copies obs/action/value/reward of all E
 * envs into `slot` (the step kernel can also write obs straight into s[slot] — then pass obs == NULL). */
int pmrl_rollout_add(int32_t E, int32_t A, int32_t W, int32_t F, int32_t slot,
                     const float* obs, const float* action, const float* value, const float* reward,
                     float* s, float* a, float* v, float* r, void* stream);

/* Minibatch gather (rollout_buffer.py:125-140): for b < B with (slot_b, env_b):
 *   s_out[b] = s[slot,env], a_out[b] = a[slot,env], r_out[b] = r[slot,env],
 *   pv_out[b] = v[slot−1,env], pa_out[b] = a[slot−1,env], p_out[b] = y[slot,env] (price relatives [S,E,A]). */
int pmrl_rollout_gather(int32_t S, int32_t E, int32_t A, int32_t W, int32_t F, int32_t B,
                        const int32_t* slots, const int32_t* envs,
                        const float* s, const float* a, const float* v, const float* r, const float* y,
                        float* s_out, float* a_out, float* r_out, float* pv_out, float* pa_out, float* p_out,
                        void* stream);

/* The same minibatch from an INDEX-mode rollout buffer, which stores per slot only bi [S, E] i32 (loader item index t0 + n of
 * the step, PmrlStepIO.index_sink), a [S, E, A], v [S, E], r [S, E] plus the un-wrapped weight history wp [S + W - 1, E, A]
 * (wp[m] = w' after step m, PmrlStepIO.weight_sink; wp[0] = all-cash): s_out[b] is regenerated — rows [i-1, i-1+W) of feat_am
 * and the ring-ordered weight channel of ActionBuffer.get_all (weight_buffer.py:38-39) from wp — like ReplayBuffer.sample
 * regenerates its windows (replay/buffer.py:58-77); p_out[b] = y_tm[i + W - 1].  8·A + 12 bytes per env-step of storage
 * instead of 4·A·W·F.  Slots are >= 1 (slot - 1 is read, rollout_buffer.py:130-131). */
int pmrl_rollout_gather_index(int32_t S, int32_t E, int32_t A, int32_t W, int32_t F, int32_t T, int32_t B,
                              const int32_t* slots, const int32_t* envs,
                              const int32_t* bi, const float* a, const float* v, const float* r,
                              const float* wp, const float* feat_am, const float* y_tm,
                              float* s_out, float* a_out, float* r_out, float* pv_out, float* pa_out, float* p_out,
                              void* stream);

/* The two rollout gathers for a buffer whose observations are bf16 (PMRL_OBS_BF16): the same parameters, but s (full mode)
 * and s_out are uint16_t bf16 bit patterns; the regenerated obs of the index-mode gather is rounded from the fp32 values like
 * the step kernels round theirs.  The other outputs stay fp32. */
int pmrl_rollout_gather_bf16(int32_t S, int32_t E, int32_t A, int32_t W, int32_t F, int32_t B,
                             const int32_t* slots, const int32_t* envs,
                             const uint16_t* s, const float* a, const float* v, const float* r, const float* y,
                             uint16_t* s_out, float* a_out, float* r_out, float* pv_out, float* pa_out, float* p_out,
                             void* stream);
int pmrl_rollout_gather_index_bf16(int32_t S, int32_t E, int32_t A, int32_t W, int32_t F, int32_t T, int32_t B,
                                   const int32_t* slots, const int32_t* envs,
                                   const int32_t* bi, const float* a, const float* v, const float* r,
                                   const float* wp, const float* feat_am, const float* y_tm,
                                   uint16_t* s_out, float* a_out, float* r_out, float* pv_out, float* pa_out, float* p_out,
                                   void* stream);

/* Off-policy index replay: store (i, a, r) of all E envs at [epoch_slot, step_slot] (buffer.py:31-37).
 * Buffers: bi [P, L, E] i32, ba [P, L, E, A], br [P, L, E]. */
int pmrl_replay_add(int32_t P, int32_t L, int32_t E, int32_t A, int32_t epoch_slot, int32_t step_slot,
                    const int32_t* item_index, const float* action, const float* reward,
                    int32_t* bi, float* ba, float* br, void* stream);

/* Off-policy sample (buffer.py:58-77): for b < B with (epoch_b, env_b, start_b), end = start+W:
 *   i = bi[epoch, end−1, env];  s[b] = window rows [i, i+W) of feat_am, s_[b] = rows [i+1, i+1+W);
 *   channel F−1 of s ← ba[epoch, start:end, env, :]ᵀ, of s_ ← ba[epoch, start+1:end+1, env, :]ᵀ;
 *   a[b] = ba[epoch, end, env, :];  r[b] = br[epoch, end−1, env]. */
int pmrl_replay_gather(int32_t P, int32_t L, int32_t E, int32_t A, int32_t W, int32_t F, int32_t T, int32_t B,
                       const int32_t* epochs, const int32_t* envs, const int32_t* starts,
                       const int32_t* bi, const float* ba, const float* br, const float* feat_am,
                       float* s_out, float* a_out, float* r_out, float* s2_out, void* stream);
/* The same sample with s_out / s2_out as uint16_t bf16 bit patterns (PMRL_OBS_BF16 rounding); a_out, r_out stay fp32. */
int pmrl_replay_gather_bf16(int32_t P, int32_t L, int32_t E, int32_t A, int32_t W, int32_t F, int32_t T, int32_t B,
                            const int32_t* epochs, const int32_t* envs, const int32_t* starts,
                            const int32_t* bi, const float* ba, const float* br, const float* feat_am,
                            uint16_t* s_out, float* a_out, float* r_out, uint16_t* s2_out, void* stream);

/* ---- differentiable batched reward (agent/pg/pg.py:40-82) ---- */

/* Forward: per row b: a' = softmax(a) if normalise else a; mu (commission) ; v = Σ pv·(a'·p); ret = v/(mu·pv);
 * rew[b] = {ret, ln ret}·scale;  Backward: grad_a[b,:] = d(mean_b rew)/d a[b,:]·gscale.
 * a [B, A], pv [B], pa [B, A] (previous weights), p [B, A].  mode: PMRL_REWARD_RETURNS | _LOG_RETURNS. */
int pmrl_pg_reward_fwd_bwd(int32_t B, int32_t A, int32_t mode, int32_t normalise, float commission, float scale,
                           int32_t mu_max_iter,
                           const float* a, const float* pv, const float* pa, const float* p,
                           float* rew, float* grad_a, float gscale, void* stream);

/* ---- evaluation metrics on device (util/eval.py:14-37) ---- */

/* values [E, N] per-env portfolio-value history (values[:,0] = initial cash), weights [E, N, A] or NULL.
 * out [E, 4] = {sharpe, sortino, max drawdown, average turnover} with simple returns r_i = V_i/V_{i-1} - 1,
 * excess e_i = r_i - ((1+rf)^(1/periods) - 1):
 *   sharpe  = mean(e)/std(e, ddof=1)*sqrt(periods);  sortino = mean(e)/sqrt(sum(min(e,0)^2)/n)*sqrt(periods)
 *   (the published quantstats formulas util/eval.py:14-24 calls — quantstats itself is not vendored: UNPINNED);
 *   mdd     = min_i(V_i / max_{j<=i} V_j) - 1                         (util/eval.py:26-30)
 *   turnover = mean_{i>=1} sum_a |w[i,a] - w[i-1,a]|                   (util/eval.py:32-37, pinned) */
int pmrl_eval_metrics(const float* values, const float* weights, int32_t E, int32_t N, int32_t A,
                      float rf, int32_t periods, float* out, void* stream);

/* Streaming form of the same metrics (util/eval.py:14-37): O(E) memory instead of [E, N] / [E, N, A] traces.
 * acc is a caller-owned device buffer of E accumulators, PMRL_EVAL_ACC_BYTES each, 16-byte aligned; all-zero means
 * "no episode seen".  Each holds the running episode (Welford mean / M2 of the excess returns, downside sum of squares,
 * turnover sum in fp64; previous V, peak and min V/peak in fp32) and the record of completed episodes: the last one's
 * (return, sharpe, sortino, mdd - 1, turnover), fp64 sums of those five and an episode count.
 *
 * pmrl_eval_stream_update: enqueue once after EVERY reset / step of the env batch (same stream).  Per env, with t the
 * local step after the call: t == 0 restarts the running episode (V_prev = peak = V, the record is kept); t == last
 * t + 1 adds the step (r = V/V_prev - 1 - ((1+rf)^(1/periods) - 1), turnover sum_a |w'_t - w'_{t-1}| from ring rows
 * (idx-1) mod W and (idx-2) mod W) and, when t == episode_len (the step that returned done = 1), appends the episode to
 * the record with its return ep_return[e]; t == last t does nothing; anything else (a missed update, or an accumulator
 * that never saw a reset) marks the env invalid until its next reset.  rf / periods must be the same on every call.
 * pmrl_eval_stream_read: out [E, 5] = (return, sharpe, sortino, mdd - 1, turnover) with the formulas of
 * pmrl_eval_metrics (sd with ddof = 1, sortino over sqrt(downside / n), turnover = sum / n), for
 *   which = PMRL_EVAL_RUNNING       the running episode (return = ep_return[e]); n = 0: sharpe, sortino, turnover NaN,
 *                                    mdd 0; n = 1: sharpe NaN; an invalid env, or one stepped since its last update: NaN
 *           PMRL_EVAL_LAST_EPISODE  the last completed episode (NaN without one)
 *           PMRL_EVAL_EPISODE_MEAN  the mean of every completed episode's row (NaN without one)
 * count [E] i32 (or NULL) receives the number of completed episodes.  rf is not used by the read (the update formed
 * the excess returns); periods annualises sharpe and sortino.
 * Both: NULL acc / value / hist / idx / t / ep_return (or out) → PMRL_E_ARG; E < 0, A outside [1, 1024], W < 2,
 * periods < 1 → PMRL_E_SHAPE; acc not 16-byte aligned → PMRL_E_ALIGN; an unknown `which` → PMRL_E_ARG. */
#define PMRL_EVAL_ACC_BYTES     128
#define PMRL_EVAL_RUNNING       0
#define PMRL_EVAL_LAST_EPISODE  1
#define PMRL_EVAL_EPISODE_MEAN  2
int pmrl_eval_stream_update(const PmrlEnvCfg* cfg, const PmrlEnvState* st, void* acc, float rf, int32_t periods,
                            void* stream);
int pmrl_eval_stream_read(const PmrlEnvCfg* cfg, const PmrlEnvState* st, const void* acc, int32_t which, float rf,
                          int32_t periods, float* out, int32_t* count, void* stream);

/* ---- randomised episode starts ---- */

/* Draw a fresh table offset t0[e] for envs about to be reset, on the device (enqueue it BEFORE the reset / step call that
 * reads the offset; the call after it then writes its obs, index_sink and every later row of the episode from the new t0).
 *
 * The draw of env e depends only on (seed, gid = env_base + e, episode[e]) — not on the stream, launch shape or how many
 * GPUs share the batch:
 *   (x0, x1, x2, x3) = Philox4x32-10(counter = (episode[e], gid & 0xffffffff, gid >> 32, 0),
 *                                    key     = (seed & 0xffffffff, seed >> 32))          (Random123, Salmon et al. 2011)
 *   r64 = (uint64)x0 << 32 | x1;   n = hi - lo + 1;   then episode[e] += 1 (u32)
 *   PMRL_START_UNIFORM    t0 = lo + umul64hi(r64, n)                                      (integer only)
 *   PMRL_START_GEOMETRIC  P(t0 = hi - j) ∝ beta (1 - beta)^j for j < n (recent rows favoured):
 *                         u = (r64 >> 11) * 2^-53,  j = min(n - 1, floor(log1p(-u * geo_norm) / log1m_beta)),  t0 = hi - j
 *                         with log1m_beta = log1p(-beta) and geo_norm = -expm1(n * log1m_beta), both double, from the caller
 *                         (the device evaluates one fp64 log1p and one fp64 division per draw)
 * mode PMRL_DRAW_DUE   draws for the envs the NEXT pmrl_env_step / _io / _host call auto-resets: episode_len > 0 and
 *                      t[e] >= episode_len (the step kernels' own test); enqueue it right before that call.
 *      PMRL_DRAW_MASK  draws for mask[e] != 0 (mask == NULL → every env); enqueue it right before pmrl_env_reset with the
 *                      same mask.
 * Envs that are not drawn are not written (t0 and episode keep their bytes).  t is read in DUE mode only (may be NULL
 * otherwise).  t0 [E] i32 is the array PmrlEnvState.t0 points to, passed here writable; episode [E] u32 is caller-owned,
 * zero-initialised for a fresh sequence.
 * NULL cfg / dist / t0 / episode (or t in DUE mode), an unknown kind or mode, a geometric log1m_beta that is not finite
 * and < 0 (beta outside (0, 1) or NaN) or a geo_norm outside (0, 1] → PMRL_E_ARG; E < 0, lo < 0, hi < lo, env_base outside
 * [0, INT64_MAX - E] (global ids must not overflow),
 * or T > 0 and hi + episode_len + W > T (the window of the last step would leave the tables) → PMRL_E_SHAPE. */
#define PMRL_START_UNIFORM    0
#define PMRL_START_GEOMETRIC  1
#define PMRL_DRAW_DUE         0
#define PMRL_DRAW_MASK        1
typedef struct PmrlStartDist {
    int32_t kind;              /* PMRL_START_* */
    int32_t lo, hi;            /* offsets drawn from [lo, hi] */
    int32_t pad;
    uint64_t seed;             /* Philox key */
    int64_t env_base;          /* global id of env 0 of this batch (a rank's first env) */
    double log1m_beta;         /* GEOMETRIC: log1p(-beta) */
    double geo_norm;           /* GEOMETRIC: -expm1((hi - lo + 1) * log1m_beta) */
} PmrlStartDist;
int pmrl_env_draw_starts(const PmrlEnvCfg* cfg, const PmrlStartDist* dist, const int32_t* t, const uint8_t* mask,
                         int32_t mode, int32_t* t0, uint32_t* episode, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PMRL_B200_H */
