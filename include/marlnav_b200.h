/*
 * include/marlnav_b200.h -- C ABI of libmarlnav_b200.so
 *
 * Drop-in boundary for ONE path of JussiM01/MARL-nav: the batched environment
 * step, marlnav/environment.py (Env.__init__ :11-68, Env.step :92-107,
 * Env.observations :139-180).  The reference has no FFI of its own -- the seam
 * is the duck-typed Python class `Env` (SURVEY.md section 8b) -- so these entry
 * points are what a ctypes binding of that class needs and nothing more; the
 * binding itself is marlnav_b200/env.py and is shown in INTEGRATION.md.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch types.
 *   - Every `float*` / `uint8_t*` / `unsigned long long*` below is a DEVICE
 *     pointer into caller-owned memory unless the name ends in `_host`.
 *   - Tensors use the reference's layouts, contiguous, float32:
 *       states (B,A,5) = [x, y, dir_x, dir_y, speed]     environment.py:28, utils.py:386
 *       obstacles (B,O,2), target (B,1,2)                 environment.py:29-30
 *       actions (B,A,2) = [turn angle rad, acceleration]  environment.py:115-119
 *       obs (B,A,S), S = 2 + 2*O + 2*(A-1), field order of the reference's
 *         `Observations` namedtuple (utils.py:13-15):
 *         [target_angle | target_distance | obstacles_angles(O) |
 *          obstacles_distances(O) | others_angles(A-1) | others_distances(A-1)]
 *       step_num (B) float32 (environment.py:38), terminates (B) 1-byte bool
 *       (environment.py:39), rewards (B), terminated/truncated (B) 1-byte bool.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).
 *     All calls are asynchronous on that stream; none allocates or synchronises
 *     (marlnav_step_host_f32 enqueues copies on the streams of a caller-owned
 *     marlnav_host_pipe; the caller synchronises).
 *   - Every struct passed by pointer starts with `struct_size` = its sizeof in the
 *     caller's build (ABI 4); an entry that receives another size fails with
 *     MARLNAV_ERR_BAD_ARG instead of reading past the caller's struct.
 *   - Threading: the library keeps no mutable state between calls except caches of
 *     idempotent facts (proven constant divisors, per-device kernel attributes; both
 *     safe to race) and the calling thread's last-error string.  Calls on different
 *     streams / devices may come from different threads; a marlnav_host_pipe must not
 *     be used by two calls at a time.
 *   - Return value: 0 on success, a cudaError_t (>0) for a CUDA failure,
 *     <0 for an argument error; marlnav_last_error() describes the last failure
 *     of the calling thread.
 *   - There is no CPU fallback: without a CUDA device every compute entry fails.
 */
#ifndef MARLNAV_B200_H
#define MARLNAV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MARLNAV_ABI_VERSION 4
#define MARLNAV_MAX_AGENTS 26     /* torch.cdist's direct formula holds up to 25 columns */
#define MARLNAV_MAX_OBSTACLES 64

#define MARLNAV_ERR_BAD_ARG   (-1)
#define MARLNAV_ERR_BAD_SHAPE (-2)
#define MARLNAV_ERR_ALIGN     (-3)

/* Everything Env.__init__ reads from params (environment.py:13-19,32-35,48-53) plus
 * the geometry constants it hard-codes (environment.py:56-68) and the obstacle box
 * of TriangleIntitializer (utils.py:344-347).  Passed by pointer, read on the host. */
typedef struct marlnav_env_params {
    uint32_t struct_size;    /* sizeof(marlnav_env_params) */
    int32_t num_envs;        /* B = num_parallel (this process's slice) */
    int32_t num_agents;      /* A, 2..MARLNAV_MAX_AGENTS */
    int32_t num_obstacles;   /* O, 1..MARLNAV_MAX_OBSTACLES */
    int32_t episode_len;     /* truncated = step_num > episode_len - 1 */
    float min_speed, max_speed, min_accel, max_accel;
    float risk_factor, distance_factor, heading_factor, target_factor, soft_factor, bond_factor;
    float ob_risk_dist, ag_risk_dist, ob_coll_dist, ag_coll_dist;
    float agents_min_d, agents_max_d, max_at_prop_d, max_angle_diff;
    float target_radius, cap_distance, bond_sharpness, ideal_dist, init_dist;
    float obst_x_range, obst_x_mean, obst_y_range, obst_y_mean;
} marlnav_env_params;

/* Where re-initialised envs get their state (Env._reinit, environment.py:76-90).
 *   env stride 0  -> one template shared by all envs (TriangleIntitializer's
 *                    constant agents/target, utils.py:349-368)
 *   env stride >0 -> per-env templates (MockInitializer, utils.py:310-319)
 *   tmpl_obstacles == NULL -> obstacles re-sampled uniformly in the box with
 *                    Philox4x32-10 addressed by (seed; global env id,
 *                    step_counter, obstacle pair) -- replaces the global
 *                    mt19937 draw of utils.py:390-398.
 *   alias_first_step != 0 -> reproduce MockInitializer's aliasing on the first
 *                    step: the template IS the current state (SURVEY.md B-6). */
/* flags: no element of a SHARED tmpl_states (states_env_stride == 0) has its sign bit set,
 * so 0*template == +0 and the blend of a not-reset env reduces to old + 0 (no template reads).
 * A binding should set it whenever it holds (marlnav_b200.Env checks the template): together with
 * states_env_stride == 0, alias_first_step == 0, no MARLNAV_RESET_NOISY_AGENTS and the reference's
 * geometry constants it selects the step kernels specialised for the default reset source (1-2 %
 * faster); every other combination runs the general kernels, with identical results. */
#define MARLNAV_RESET_TMPL_NONNEG 1
/* TriangleIntitializer with noisy_ags = True (utils.py:25, 381-388; shared template only): every
 * (re-)initialised agent gets Gaussian position noise  pos += noise_mult * (noise_chol * z)  with
 * z ~ N(0, I) (MultivariateNormal(0, diag(ags_std)).sample(): noise_chol = sqrt(ags_std),
 * noise_mult = ags_dist) and its template heading rotated by angle_range * (u - 1/2).  The draws are
 * Philox4x32-10 addressed by (seed; global env id, step_counter, 0x40000000 + agent): words 0-1
 * -> Box-Muller normals, word 2 -> u.  Like the reference, which samples the whole batch every
 * step and blends by mask, envs that do not reset evaluate the literal blend old + 0 * new. */
#define MARLNAV_RESET_NOISY_AGENTS 2

typedef struct marlnav_reset_spec {
    uint32_t struct_size;      /* sizeof(marlnav_reset_spec) */
    int32_t flags;             /* MARLNAV_RESET_* bits */
    const float* tmpl_states;
    const float* tmpl_obstacles;
    const float* tmpl_target;
    int64_t states_env_stride, obstacles_env_stride, target_env_stride;   /* in floats */
    int32_t alias_first_step;
    float noise_chol, noise_mult, angle_range;   /* MARLNAV_RESET_NOISY_AGENTS only */
    uint64_t seed;
    uint64_t step_counter;     /* 0 at construction, k for the k-th step() call */
    uint64_t env_id_offset;    /* global id of local env 0 (multi-GPU sharding) */
    const uint64_t* step_counter_dev;  /* if non-NULL the kernels use `step_counter` + this DEVICE word
                                        * (ABI 3), so a captured CUDA graph draws fresh reset positions
                                        * on every replay: either bump the word with marlnav_counter_add
                                        * before each step and pass step_counter = 0, or pass the step's
                                        * 1-based index inside a batch of T steps and add T once after
                                        * the batch */
} marlnav_reset_spec;

/* Optional fused caller-side transforms (SURVEY.md section 8(f)-1):
 *   ObsNormalizer  utils.py:519-532   obs_norm[k] = (obs[k] - mean[k]) / scale[k]
 *   ActionScaler   utils.py:535-547   action[k]   = scale[k] * raw[k] + mean[k]
 * All pointers device; NULL disables the corresponding transform. */
typedef struct marlnav_io_transform {
    uint64_t struct_size;      /* sizeof(marlnav_io_transform) */
    const float* obs_mean;     /* (S) */
    const float* obs_scale;    /* (S) */
    const float* act_mean;     /* (2) */
    const float* act_scale;    /* (2) */
} marlnav_io_transform;

int         marlnav_abi_version(void);
const char* marlnav_last_error(void);
/* sizeof of the structs in the library's build: a binding asserts they equal its own layouts. */
size_t      marlnav_sizeof_env_params(void);
size_t      marlnav_sizeof_reset_spec(void);
size_t      marlnav_sizeof_io_transform(void);
size_t      marlnav_sizeof_actor_spec(void);
size_t      marlnav_sizeof_step_call(void);
/* S = 2 + 2*O + 2*(A-1); 0 for invalid (A,O). */
int         marlnav_obs_size(int num_agents, int num_obstacles);
/* Number of CUDA devices visible (0 when there is none / no driver). */
int         marlnav_device_count(void);

/* *counter += inc on the stream (one-thread kernel; graph-capturable).  Used to advance the
 * device-resident step counters of marlnav_reset_spec / marlnav_actor_sample_f32. */
int marlnav_counter_add(uint64_t* counter, uint64_t inc, void* stream);

/* Env.__init__'s first `self._init_sampler()` + counters (environment.py:26-40):
 * fills states/obstacles/target from `reset` (step_counter is used as given,
 * normally 0) and zeroes step_num / terminates. */
int marlnav_init_f32(const marlnav_env_params* params, const marlnav_reset_spec* reset,
                     float* states, float* obstacles, float* target,
                     float* step_num, uint8_t* terminates, void* stream);

/* Env.observations() (environment.py:139-180): obs <- f(states, obstacles, target). */
int marlnav_observe_f32(const marlnav_env_params* params,
                        const float* states, const float* obstacles, const float* target,
                        float* obs, void* stream);

/* Env.step(actions) (environment.py:92-107) as ONE kernel launch:
 * move -> count -> observe -> rewards/terminal flags -> episode stats ->
 * masked re-initialisation -> observe again (returned obs are post-reset).
 *   in-out: states, obstacles, target, step_num, terminates
 *   out   : obs (B,A,S), rewards (B), terminated (B), truncated (B)
 *   stats : device uint64[3], += (num_trunc, num_col, num_tar)  environment.py:98,210,211
 *   io    : may be NULL.  With io->act_* set, `actions` are the policy's raw
 *           [-1,1] outputs; with io->obs_* set, `obs` receives normalised values. */
int marlnav_step_f32(const marlnav_env_params* params, const marlnav_reset_spec* reset,
                     float* states, float* obstacles, float* target,
                     float* step_num, uint8_t* terminates,
                     const float* actions,
                     float* obs, float* rewards, uint8_t* terminated, uint8_t* truncated,
                     unsigned long long* stats,
                     const marlnav_io_transform* io, void* stream);

/* marlnav_step_f32 with its arguments in one caller-owned struct: a binding fills it once and
 * changes only what differs between steps (actions, outputs, stream; the step counter lives in
 * *reset).  Through Python's ctypes a 1-argument call costs ~2 us less than the 15-argument one,
 * which is most of what a step of ~1000 envs costs on the host. */
typedef struct marlnav_step_call {
    uint64_t struct_size;      /* sizeof(marlnav_step_call) */
    const marlnav_env_params* params;
    const marlnav_reset_spec* reset;
    float *states, *obstacles, *target, *step_num;
    uint8_t* terminates;
    const float* actions;
    float *obs, *rewards;
    uint8_t *terminated, *truncated;
    unsigned long long* stats;
    const marlnav_io_transform* io;
    void* stream;
} marlnav_step_call;
int marlnav_step_call_f32(const marlnav_step_call* call);

/* Streams and events of the host-stepping pipeline below, owned by the caller: created on the
 * current device, used by one marlnav_step_host_f32 call at a time, destroyed by the caller.
 * (The only entry points that allocate.) */
typedef struct marlnav_host_pipe marlnav_host_pipe;
int  marlnav_host_pipe_create(marlnav_host_pipe** pipe);
void marlnav_host_pipe_destroy(marlnav_host_pipe* pipe);

/* Same step for a HOST-resident policy: `actions_host` is copied H2D, the step
 * runs, and obs/rewards/flags are copied D2H; the batch is cut into chunks whose
 * upload, step and download overlap on `stream` and the two streams of `pipe`;
 * `stream` ends up waiting for the last download.  Host
 * buffers should be pinned for the copies to be asynchronous.  `actions_dev`,
 * `obs_dev`, `rewards_dev`, `terminated_dev`, `truncated_dev` are device staging
 * buffers of the usual shapes owned by the caller.  Environment state stays on
 * the device (it never leaves HBM between steps). */
int marlnav_step_host_f32(marlnav_host_pipe* pipe,
                          const marlnav_env_params* params, const marlnav_reset_spec* reset,
                          float* states, float* obstacles, float* target,
                          float* step_num, uint8_t* terminates,
                          const float* actions_host, float* actions_dev,
                          float* obs_dev, float* rewards_dev,
                          uint8_t* terminated_dev, uint8_t* truncated_dev,
                          float* obs_host, float* rewards_host,
                          uint8_t* terminated_host, uint8_t* truncated_host,
                          unsigned long long* stats,
                          const marlnav_io_transform* io, void* stream);

/* Launch geometry the library would use for (A,O,B): for bench/roofline reporting.
 * Writes grid, block, dynamic smem bytes, envs per CTA; returns 0 or an error. */
int marlnav_step_launch_info(const marlnav_env_params* params,
                             int* grid, int* block, int* smem_bytes, int* envs_per_cta);

/* ---- caller-side rows that come next after the step (SURVEY.md section 8(f)-2, 8(f)-3) ---- */

/* Actor.forward + dist.sample() + dist.log_prob(actions), marlnav/models.py:27-36,113-115, for
 * N = B*A rows of normalised observations (obs_size S, hidden H; the reference has S=12, H=50):
 *   h = fc1(x)  (no activation, models.py:29);  mu = tanh(fc_mu(h));  var = softplus(fc_std(h))
 *   dist = MultivariateNormal(mu, covariance_matrix=diag(var))        (models.py:32-34)
 *   actions = mu + sqrt(var)*eps;  log_probs = dist.log_prob(actions)
 * Weights are torch.nn.Linear layouts: w1 (H,S), b1 (H), w_mu/w_std (2,H), b_mu/b_std (2).
 * eps (N,2): standard-normal draws to use (parity tests) or NULL -> Philox4x32-10 + Box-Muller
 * addressed by (seed; row_offset + row, counter); counter_dev, if non-NULL, is a DEVICE word added to
 * `counter` (CUDA-graph replays, same convention as marlnav_reset_spec.step_counter_dev).
 * row_offset = the global index of local row 0 (env_id_offset * A for a sharded batch), so N ranks
 * draw what one process would (ABI 4).  mu_out/var_out (N,2) may be NULL. */
int marlnav_actor_sample_f32(const float* obs, long long N, int S, int H,
                             const float* w1, const float* b1, const float* w_mu, const float* b_mu,
                             const float* w_std, const float* b_std,
                             const float* eps, uint64_t seed, uint64_t counter, const uint64_t* counter_dev,
                             uint64_t row_offset,
                             float* actions, float* log_probs, float* mu_out, float* var_out, void* stream);

/* The same actor as one struct, for the fused {actor -> step} launch. */
typedef struct marlnav_actor_spec {
    uint64_t struct_size;         /* sizeof(marlnav_actor_spec) */
    const float *w1, *b1, *w_mu, *b_mu, *w_std, *b_std;   /* device, torch.nn.Linear layouts as above */
    int32_t S, H;                 /* obs_size (must equal the env's), hidden (<= 256) */
    uint64_t seed, counter;       /* Philox addressing, as in marlnav_actor_sample_f32 */
    const uint64_t* counter_dev;  /* optional DEVICE word added to `counter` */
    uint64_t row_offset;          /* global index of local row 0 (env_id_offset * A) */
} marlnav_actor_spec;

/* SURVEY.md section 8(f)-2, end state: MAPPO.get_data's inner iteration (models.py:113-122) as ONE
 * launch -- actor forward + sample + log_prob on the normalised observations `obs_in` (B,A,S) of the
 * current state, ActionScaler, the environment step, ObsNormalizer on the new observations.
 * Writes actions_out (B*A,2) raw sampled actions, log_probs_out (B*A), and the step's outputs as
 * marlnav_step_f32.  Requires `io` with both transforms and a team shape with a thread-per-env
 * kernel (3 agents, 1..6 obstacles); returns MARLNAV_ERR_BAD_SHAPE otherwise (callers then use
 * marlnav_actor_sample_f32 + marlnav_step_f32, which give the same bits). */
int marlnav_act_step_f32(const marlnav_env_params* params, const marlnav_reset_spec* reset,
                         float* states, float* obstacles, float* target, float* step_num, uint8_t* terminates,
                         const marlnav_actor_spec* actor, const float* obs_in,
                         float* actions_out, float* log_probs_out,
                         float* obs, float* rewards, uint8_t* terminated, uint8_t* truncated,
                         unsigned long long* stats, const marlnav_io_transform* io, void* stream);

/* Critic.forward, marlnav/models.py:39-56: values (B) = fc2(relu(fc1(x))) for x = the env's
 * flattened normalised observations (K = A*S inputs, hidden H <= 64; reference: 36 -> 50 -> 1).
 * w1 (H,K), b1 (H), w2 (1,H), b2 (1) in torch.nn.Linear layout. */
int marlnav_critic_value_f32(const float* obs, long long B, int K, int H,
                             const float* w1, const float* b1, const float* w2, const float* b2,
                             float* values, void* stream);

/* The backward scan of MAPPO._process_rewards, marlnav/models.py:131-139, in float64 like the
 * reference: out[t] = done[t] ? 0 : rewards[t] + gamma * out[t+1], t = T-1..0, (T,B) row-major. */
int marlnav_discounted_returns_f64(const float* rewards, const uint8_t* done, double gamma,
                                   int T, long long B, double* out, void* stream);

const char* marlnav_rollout_last_error(void);

#ifdef __cplusplus
}
#endif

/* float16 / bfloat16 observations: the `_typed` entry points of the step, then of the rollout;
 * final observations of auto-reset envs and truncation-aware GAE */
#include "marlnav_b200_typed.h"
#include "marlnav_b200_rollout_typed.h"
#include "marlnav_b200_final.h"

#endif /* MARLNAV_B200_H */
