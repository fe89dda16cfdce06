/*
 * include/marlnav_b200_final.h -- final observations of auto-reset envs, truncation-aware GAE
 *
 * Included by marlnav_b200.h after marlnav_b200_typed.h, whose MARLNAV_OBS_* codes it uses;
 * additive to ABI 4 (no struct or existing entry point changes).
 *
 * Every step auto-resets the envs it finishes and returns their post-reset observations.  The
 * `_final` steps also write `final_obs` (B,A,S), of element type `obs_dtype`: for every env whose
 * terminated | truncated this step sets, final_obs[b] holds the observations its rewards and flags
 * were computed from (post-move, pre-reset; normalised when `io` has the normaliser), the same bits
 * a non-resetting env gets in `obs`.  Rows of envs that did not finish are not written.
 * `final_obs` may start at any address its element type allows.  A NULL `final_obs`, one equal to
 * `obs` or an unknown `obs_dtype` returns MARLNAV_ERR_BAD_ARG before anything is launched; callers
 * that do not want the final observations use marlnav_step_typed / marlnav_step_call_typed.
 * There is no fused actor+step or host-pipeline form.  Errors: marlnav_last_error.
 */
#ifndef MARLNAV_B200_FINAL_H
#define MARLNAV_B200_FINAL_H

#include "marlnav_b200.h"
#include "marlnav_b200_typed.h"

#ifdef __cplusplus
extern "C" {
#endif

/* marlnav_step_typed that also writes the finished envs' pre-reset observations to `final_obs`. */
int marlnav_step_final_typed(const marlnav_env_params* params, const marlnav_reset_spec* reset,
                             float* states, float* obstacles, float* target,
                             float* step_num, uint8_t* terminates,
                             const float* actions,
                             void* obs, int obs_dtype, void* final_obs,
                             float* rewards, uint8_t* terminated, uint8_t* truncated,
                             unsigned long long* stats,
                             const marlnav_io_transform* io, void* stream);

/* marlnav_step_call_typed with `final_obs`, as marlnav_step_final_typed. */
int marlnav_step_call_final_typed(const marlnav_step_call* call, int obs_dtype, void* final_obs);

/* Generalised advantage estimation that tells truncation from termination, per env b over
 * (T,B) row-major float32 inputs, for t = T-1 .. 0 (gl = gamma * lam, computed once):
 *     nv = t == T-1 ? last_values[b] (0 if NULL) : values[t+1,b]
 *     terminated[t,b]:  nv = 0,                                cont = 0
 *     else truncated:   nv = final_values[t,b] (0 if NULL),    cont = 0
 *     else:                                                    cont = 1
 *     delta = (r + gamma * nv) - v;  adv = cont ? delta + gl * adv_next : delta;  ret = adv + v
 * Outputs advantages / returns (T,B) float64.  Every operation is a float64 operation rounded to
 * nearest, without fused multiply-adds.  Errors: marlnav_rollout_last_error. */
int marlnav_gae_f64(const float* rewards, const float* values, const uint8_t* terminated,
                    const uint8_t* truncated, const float* final_values, const float* last_values,
                    double gamma, double lam, int T, long long B,
                    double* advantages, double* returns, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MARLNAV_B200_FINAL_H */
