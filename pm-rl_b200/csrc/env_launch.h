// env_launch.h — internal: launchers shared between the env translation units.
#pragma once
#include <cuda_runtime.h>
#include "pmrl_device.cuh"

// Fused step+obs kernel whose weight rings enter shared memory as one TMA bulk load per env (env_step_rt.cu).
// bf16: obs as bf16 bit patterns (PMRL_OBS_BF16).  Returns -100 if the shape is not covered by this kernel (caller falls back).
int pmrl_launch_step_obs_rt(pmrl::StepParams& p, int npl, int vec, int group, int ctas_per_sm, bool bf16, cudaStream_t s);

// Register-staged fused step+obs kernel (env_step_fast.cu).  Returns -100 if the shape is not covered.
int pmrl_launch_step_obs_fast(pmrl::StepParams& p, int npl, int vec, int group, int ctas_per_sm, cudaStream_t s);

// State-only step for wide envs with the rows staged through shared memory by TMA bulk copies (env_step_staged.cu).
// Returns -100 if the shape is not covered.
int pmrl_launch_step_staged(const pmrl::StepParams& p, int npl, int vec, int shape, cudaStream_t s);

// host_step.cu: 1 = stream page-locked actions in with the copy engine under the kernel (default), 0 = zero-copy reads.
void pmrl_set_host_stream(int value);
void pmrl_set_host_mirror(int value);
