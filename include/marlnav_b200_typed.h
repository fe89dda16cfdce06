/*
 * include/marlnav_b200_typed.h -- observation element types of libmarlnav_b200.so
 *
 * Included by marlnav_b200.h; additive to ABI 4 (no struct or existing entry point changes).
 *
 * The `_typed` entry points are the `_f32` ones with the observations' element type as an
 * argument.  MARLNAV_OBS_F32 is exactly the `_f32` call.  With MARLNAV_OBS_F16 / MARLNAV_OBS_BF16
 * every observation is written as IEEE half / bfloat16: the float32 value the `_f32` call would
 * have written (after the io normaliser, if any), rounded to nearest-even, subnormals kept -- the
 * same bits as torch's `obs32.to(torch.float16 / torch.bfloat16)` (NaN payloads unspecified).
 * Everything else -- states, obstacles, target, step_num, terminates, rewards, terminated,
 * truncated, stats -- is bit-identical to the float32 call: rewards and flags are computed from the
 * float32 values, only the stored copy is rounded.
 *
 * A 16-bit `obs` may start at any 2-byte aligned address; 16-byte aligned buffers take the bulk
 * (TMA) stores, others plain stores with the same results.  An unknown `obs_dtype` returns
 * MARLNAV_ERR_BAD_ARG before anything is launched.  marlnav_step_launch_info reports the float32
 * kernels.  The 16-bit actor, critic and fused actor+step entries are declared in
 * marlnav_b200_rollout_typed.h.
 */
#ifndef MARLNAV_B200_TYPED_H
#define MARLNAV_B200_TYPED_H

#include "marlnav_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define MARLNAV_OBS_F32  0   /* float32 (the `_f32` entry points) */
#define MARLNAV_OBS_F16  1   /* IEEE binary16, round to nearest-even */
#define MARLNAV_OBS_BF16 2   /* bfloat16, round to nearest-even */

/* marlnav_observe_f32 with `obs` (B,A,S) of element type `obs_dtype`. */
int marlnav_observe_typed(const marlnav_env_params* params,
                          const float* states, const float* obstacles, const float* target,
                          void* obs, int obs_dtype, void* stream);

/* marlnav_step_f32 with `obs` (B,A,S) of element type `obs_dtype`. */
int marlnav_step_typed(const marlnav_env_params* params, const marlnav_reset_spec* reset,
                       float* states, float* obstacles, float* target,
                       float* step_num, uint8_t* terminates,
                       const float* actions,
                       void* obs, int obs_dtype, float* rewards, uint8_t* terminated, uint8_t* truncated,
                       unsigned long long* stats,
                       const marlnav_io_transform* io, void* stream);

/* marlnav_step_call_f32 with call->obs holding `obs_dtype` elements (read as void*). */
int marlnav_step_call_typed(const marlnav_step_call* call, int obs_dtype);

/* marlnav_step_host_f32 with `obs_dev` / `obs_host` of element type `obs_dtype`: the download
 * moves 2 bytes per observation instead of 4. */
int marlnav_step_host_typed(marlnav_host_pipe* pipe,
                            const marlnav_env_params* params, const marlnav_reset_spec* reset,
                            float* states, float* obstacles, float* target,
                            float* step_num, uint8_t* terminates,
                            const float* actions_host, float* actions_dev,
                            void* obs_dev, float* rewards_dev,
                            uint8_t* terminated_dev, uint8_t* truncated_dev,
                            void* obs_host, float* rewards_host,
                            uint8_t* terminated_host, uint8_t* truncated_host,
                            unsigned long long* stats,
                            const marlnav_io_transform* io, void* stream, int obs_dtype);

#ifdef __cplusplus
}
#endif
#endif /* MARLNAV_B200_TYPED_H */
