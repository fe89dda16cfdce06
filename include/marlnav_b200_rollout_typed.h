/*
 * include/marlnav_b200_rollout_typed.h -- 16-bit observations for the rollout entry points
 *
 * Included by marlnav_b200.h after marlnav_b200_typed.h, whose MARLNAV_OBS_* codes it uses;
 * additive to ABI 4 (no struct or existing entry point changes).
 *
 * These are the float32 actor, critic and fused actor+step entries with the observations'
 * element type as an argument; MARLNAV_OBS_F32 is exactly the float32 call.  With MARLNAV_OBS_F16 /
 * MARLNAV_OBS_BF16 the policy and the critic read each stored 16-bit observation widened exactly to
 * float32, so a 16-bit input gives bit for bit what its float32 copy (torch's `.float()`) gives.
 * Everything that is not an observation -- weights, eps, actions, log-probs, mu / var, values,
 * rewards, flags, the env state -- keeps its float32 type.  An unknown `obs_dtype` returns
 * MARLNAV_ERR_BAD_ARG, with "obs_dtype" in the message, before anything is checked or launched.
 * The actor and critic report their errors through marlnav_rollout_last_error, the fused
 * actor+step through marlnav_last_error, as the float32 entries do.
 */
#ifndef MARLNAV_B200_ROLLOUT_TYPED_H
#define MARLNAV_B200_ROLLOUT_TYPED_H

#include "marlnav_b200.h"
#include "marlnav_b200_typed.h"

#ifdef __cplusplus
extern "C" {
#endif

/* The float32 actor sample with `obs` (N,S) of element type `obs_dtype`. */
int marlnav_actor_sample_typed(const void* obs, int obs_dtype, long long N, int S, int H,
                               const float* w1, const float* b1, const float* w_mu, const float* b_mu,
                               const float* w_std, const float* b_std,
                               const float* eps, uint64_t seed, uint64_t counter, const uint64_t* counter_dev,
                               uint64_t row_offset,
                               float* actions, float* log_probs, float* mu_out, float* var_out, void* stream);

/* The float32 critic with `obs` (B,K) of element type `obs_dtype`; same batch-size dispatch and
 * summation order, hence the bits of the float32 call on the widened values. */
int marlnav_critic_value_typed(const void* obs, int obs_dtype, long long B, int K, int H,
                               const float* w1, const float* b1, const float* w2, const float* b2,
                               float* values, void* stream);

/* The float32 fused actor+step with `obs_in` (the actor's input, the previous step's output) and
 * `obs` (this step's output), both (B,A,S) of element type `obs_dtype`: the same bits as the typed
 * actor sample followed by the typed step. */
int marlnav_act_step_typed(const marlnav_env_params* params, const marlnav_reset_spec* reset,
                           float* states, float* obstacles, float* target, float* step_num, uint8_t* terminates,
                           const marlnav_actor_spec* actor, const void* obs_in,
                           float* actions_out, float* log_probs_out,
                           void* obs, int obs_dtype, float* rewards, uint8_t* terminated, uint8_t* truncated,
                           unsigned long long* stats, const marlnav_io_transform* io, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MARLNAV_B200_ROLLOUT_TYPED_H */
