// marlnav_b200/csrc/marlnav_abi.cu
//
// The step library's C ABI (include/marlnav_b200.h): argument checks, the step dispatcher and the
// host pipeline.  The kernels are in marlnav_step_env.cu, marlnav_step_team.cu and
// marlnav_step_generic.cu; their declarations and entry points are in marlnav_step_launch.cuh.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <mutex>

#include "../../include/marlnav_b200.h"
#include "marlnav_step_launch.cuh"

// ============================================================================= C ABI

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, const char* detail = "") {
    snprintf(g_err, sizeof g_err, fmt, detail);
    return code;
}

}  // namespace

int mnl::cuda_fail(cudaError_t e, const char* where) {
    snprintf(g_err, sizeof g_err, "%s: %s", where, cudaGetErrorString(e));
    return (int)e;
}

namespace {

using mnl::cuda_fail;
using mnl::dispatch_observe;
using mnl::kMaxActorHidden;

const char* const kSizeMsg = "%s.struct_size does not match this library's layout (binding built against another ABI?)";

int check_params(const marlnav_env_params* p) {
    if (!p) return fail(MARLNAV_ERR_BAD_ARG, "params is NULL");
    if (p->struct_size != sizeof(marlnav_env_params)) return fail(MARLNAV_ERR_BAD_ARG, kSizeMsg, "marlnav_env_params");
    if (p->num_envs < 1) return fail(MARLNAV_ERR_BAD_SHAPE, "num_envs must be >= 1");
    if (p->num_agents < 2 || p->num_agents > MARLNAV_MAX_AGENTS)
        return fail(MARLNAV_ERR_BAD_SHAPE, "num_agents must be in [2, 26] (the reference needs >= 2 agents; "
                                           "torch.cdist changes formula above 25 columns)");
    if (p->num_obstacles < 1 || p->num_obstacles > MARLNAV_MAX_OBSTACLES)
        return fail(MARLNAV_ERR_BAD_SHAPE, "num_obstacles must be in [1, 64]");
    return 0;
}

using mnl::current_device;

bool aligned16(const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; }

// Is  q = x*rc; q += fma(-q, c, x)*rc  (rc = RN(1/c)) the correctly rounded x/c for EVERY x?
// All three steps scale exactly with powers of two while nothing leaves the normal range, so
// it is enough to try every significand once: the 2^23 floats of [1, 2).  The device code
// (mn::div_const) additionally restricts |x| to [1e-20, 1e20] and we restrict c to
// (1e-6, 1e6), which keeps every intermediate normal.  ~10 ms per constant, cached.
bool const_div_ok(float c) {
    static std::mutex mu;
    static std::map<uint32_t, bool> cache;
    uint32_t key; memcpy(&key, &c, 4);
    std::lock_guard<std::mutex> lock(mu);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    bool ok = c > 1e-6f && c < 1e6f;
    if (ok) {
        const volatile float rc_v = 1.0f / c;
        const float rc = rc_v;
        for (uint32_t m = 0; m < (1u << 23); ++m) {
            const uint32_t xb = 0x3f800000u | m;
            float x; memcpy(&x, &xb, 4);
            const volatile float q = x * rc;          // volatile: no host-side contraction
            const float got = fmaf(fmaf(-q, c, x), rc, q);
            if (got != x / c) { ok = false; break; }
        }
    }
    cache[key] = ok;
    return ok;
}
float safe_rcp(float c) {
    int e;
    if (c > 1e-6f && c < 1e6f && frexpf(c, &e) == 0.5f) return -(1.0f / c);   // power of two: exact scaling
    return const_div_ok(c) ? 1.0f / c : 0.0f;
}

// batch size up to which a team of 3 runs thread-per-agent (MARLNAV_TEAM3_MAX_ENVS overrides; 0 = never)
int team3_max_envs() {
    static const int v = [] {
        const char* e = getenv("MARLNAV_TEAM3_MAX_ENVS");
        return e ? atoi(e) : 32768;     // measured on B200: 16384 envs 5.97 vs 9.0 us, 32768: 7.24 vs 10.1, 65536: a tie
    }();
    return v;
}

// OT: the observations' element type (float, __half, __nv_bfloat16)
template <class OT = float>
int dispatch_step(const mn::StepArgs& a, cudaStream_t st, int* info) {
    const int A = a.p.num_agents, O = a.p.num_obstacles;
    if (A == 3 && O <= 6 && a.p.num_envs <= team3_max_envs()) {
        // small batches of the reference's team: less than a wave of warps either way, so the
        // thread-per-agent mapping (a third of the dependent chain) wins on latency; same bits
        const int rc = mnl::launch_team3<OT>(a, st, info);
        if (rc != -1) return rc;
    }
    if (A == 3) {       // the reference's team (TriangleIntitializer, utils.py:349-368) with `-no` 1..6
        const int rc = mnl::launch_env3<OT>(a, st, info);
        if (rc != -1) return rc;
    }
    if (A == 8 && O == 16) return mnl::launch_team8x16<OT>(a, st, info);
    return mnl::launch_generic<OT>(a, st, info);
}

// the observation element type of a marlnav_*_typed call; 0 for an unknown MARLNAV_OBS_* code
size_t obs_elem_size(int obs_dtype) {
    return obs_dtype == MARLNAV_OBS_F32 ? 4 : (obs_dtype == MARLNAV_OBS_F16 || obs_dtype == MARLNAV_OBS_BF16) ? 2 : 0;
}
int check_obs_dtype(int obs_dtype) {
    if (obs_elem_size(obs_dtype) == 0)
        return fail(MARLNAV_ERR_BAD_ARG, "obs_dtype must be MARLNAV_OBS_F32 (0), MARLNAV_OBS_F16 (1) or MARLNAV_OBS_BF16 (2)");
    return 0;
}
int dispatch_step_typed(const mn::StepArgs& a, int obs_dtype, cudaStream_t st) {
    // the fused-actor kernels have no final-observation build
    if (a.obs_in && a.final_obs) return fail(MARLNAV_ERR_BAD_ARG, "final_obs cannot be combined with the fused actor");
    switch (obs_dtype) {
        case MARLNAV_OBS_F16: return dispatch_step<__half>(a, st, nullptr);
        case MARLNAV_OBS_BF16: return dispatch_step<__nv_bfloat16>(a, st, nullptr);
        default: return dispatch_step<float>(a, st, nullptr);
    }
}

// The StepArgs fields every step launch fills the same way; `actions` is NULL for the fused
// actor, whose launch then sets the actor's fields.
mn::StepArgs step_args(const marlnav_env_params* params, const marlnav_reset_spec* reset, float* states,
                       float* obstacles, float* target, float* step_num, uint8_t* terminates, const float* actions,
                       void* obs, float* rewards, uint8_t* terminated, uint8_t* truncated,
                       unsigned long long* stats, const marlnav_io_transform* io) {
    mn::StepArgs a;
    a.p = *params; a.rs = *reset;
    a.states = states; a.obstacles = obstacles; a.target = target; a.step_num = step_num;
    a.terminates = terminates; a.actions = actions; a.obs = static_cast<float*>(obs); a.rewards = rewards;
    a.terminated = terminated; a.truncated = truncated; a.stats = stats;
    if (io) a.io = *io; else memset(&a.io, 0, sizeof a.io);
    memset(&a.actor, 0, sizeof a.actor); a.obs_in = nullptr; a.act_out = nullptr; a.logp_out = nullptr;
    a.final_obs = nullptr;
    a.vec_ok = aligned16(states) && aligned16(obstacles) && aligned16(target) && aligned16(actions) &&
               aligned16(obs);
    a.act8 = actions && (reinterpret_cast<uintptr_t>(actions) & 7u) == 0;
    a.rc_init_dist = safe_rcp(params->init_dist);
    a.rc_prop_d = safe_rcp(params->max_at_prop_d);
    a.rc_sharp = safe_rcp(params->bond_sharpness);
    a.rc_R = safe_rcp((float)(params->num_agents - 1));
    a.rc_A = safe_rcp((float)params->num_agents);
    return a;
}

int check_reset(const marlnav_reset_spec* rs) {
    if (!rs) return fail(MARLNAV_ERR_BAD_ARG, "reset spec is NULL");
    if (rs->struct_size != sizeof(marlnav_reset_spec)) return fail(MARLNAV_ERR_BAD_ARG, kSizeMsg, "marlnav_reset_spec");
    if ((rs->flags & MARLNAV_RESET_NOISY_AGENTS) && (rs->states_env_stride != 0 || rs->alias_first_step))
        return fail(MARLNAV_ERR_BAD_ARG, "MARLNAV_RESET_NOISY_AGENTS needs a shared agent template (utils.py:381-388)");
    if (!rs->alias_first_step && (!rs->tmpl_states || !rs->tmpl_target))
        return fail(MARLNAV_ERR_BAD_ARG, "reset spec needs tmpl_states and tmpl_target");
    return 0;
}

}  // namespace

extern "C" {

int marlnav_abi_version(void) { return MARLNAV_ABI_VERSION; }
const char* marlnav_last_error(void) { return g_err; }
size_t marlnav_sizeof_env_params(void) { return sizeof(marlnav_env_params); }
size_t marlnav_sizeof_reset_spec(void) { return sizeof(marlnav_reset_spec); }
size_t marlnav_sizeof_io_transform(void) { return sizeof(marlnav_io_transform); }
size_t marlnav_sizeof_actor_spec(void) { return sizeof(marlnav_actor_spec); }
size_t marlnav_sizeof_step_call(void) { return sizeof(marlnav_step_call); }

int marlnav_obs_size(int A, int O) {
    if (A < 2 || A > MARLNAV_MAX_AGENTS || O < 1 || O > MARLNAV_MAX_OBSTACLES) return 0;
    return 2 + 2 * O + 2 * (A - 1);
}

int marlnav_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int marlnav_counter_add(uint64_t* counter, uint64_t inc, void* stream) {
    if (!counter) return fail(MARLNAV_ERR_BAD_ARG, "counter is NULL");
    mn::counter_add_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(reinterpret_cast<unsigned long long*>(counter), inc);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail(e, "counter_add launch");
}

int marlnav_init_f32(const marlnav_env_params* params, const marlnav_reset_spec* reset, float* states,
                     float* obstacles, float* target, float* step_num, uint8_t* terminates, void* stream) {
    if (int rc = check_params(params)) return rc;
    if (int rc = check_reset(reset)) return rc;
    if (reset->alias_first_step) return fail(MARLNAV_ERR_BAD_ARG, "alias_first_step is meaningless for init");
    if (!states || !obstacles || !target || !step_num || !terminates)
        return fail(MARLNAV_ERR_BAD_ARG, "NULL tensor pointer");
    const int threads = 128, grid = (params->num_envs + threads - 1) / threads;
    mn::init_kernel<<<grid, threads, 0, (cudaStream_t)stream>>>(*params, *reset, states, obstacles, target,
                                                                step_num, terminates);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail(e, "init kernel launch");
}

int marlnav_observe_typed(const marlnav_env_params* params, const float* states, const float* obstacles,
                          const float* target, void* obs, int obs_dtype, void* stream) {
    if (int rc = check_obs_dtype(obs_dtype)) return rc;
    if (int rc = check_params(params)) return rc;
    if (!states || !obstacles || !target || !obs) return fail(MARLNAV_ERR_BAD_ARG, "NULL tensor pointer");
    mn::ObserveArgs a;
    a.p = *params; a.states = states; a.obstacles = obstacles; a.target = target; a.obs = static_cast<float*>(obs);
    memset(&a.io, 0, sizeof a.io);
    a.vec_ok = aligned16(states) && aligned16(obstacles) && aligned16(target) && aligned16(obs);
    switch (obs_dtype) {
        case MARLNAV_OBS_F16: return dispatch_observe<__half>(a, (cudaStream_t)stream);
        case MARLNAV_OBS_BF16: return dispatch_observe<__nv_bfloat16>(a, (cudaStream_t)stream);
        default: return dispatch_observe<float>(a, (cudaStream_t)stream);
    }
}

int marlnav_observe_f32(const marlnav_env_params* params, const float* states, const float* obstacles,
                        const float* target, float* obs, void* stream) {
    return marlnav_observe_typed(params, states, obstacles, target, obs, MARLNAV_OBS_F32, stream);
}

}  // extern "C"

namespace {
// marlnav_step_typed, and marlnav_step_final_typed with a non-NULL final_obs
int step_typed(const marlnav_env_params* params, const marlnav_reset_spec* reset, float* states, float* obstacles,
               float* target, float* step_num, uint8_t* terminates, const float* actions, void* obs, int obs_dtype,
               void* final_obs, float* rewards, uint8_t* terminated, uint8_t* truncated, unsigned long long* stats,
               const marlnav_io_transform* io, void* stream) {
    if (int rc = check_obs_dtype(obs_dtype)) return rc;
    if (int rc = check_params(params)) return rc;
    if (int rc = check_reset(reset)) return rc;
    if (!states || !obstacles || !target || !step_num || !terminates || !actions || !obs || !rewards ||
        !terminated || !truncated || !stats)
        return fail(MARLNAV_ERR_BAD_ARG, "NULL tensor pointer");
    if (io && io->struct_size != sizeof(marlnav_io_transform)) return fail(MARLNAV_ERR_BAD_ARG, kSizeMsg, "marlnav_io_transform");
    if (io && ((io->obs_mean == nullptr) != (io->obs_scale == nullptr) ||
               (io->act_mean == nullptr) != (io->act_scale == nullptr)))
        return fail(MARLNAV_ERR_BAD_ARG, "io transform needs mean and scale together");
    mn::StepArgs a = step_args(params, reset, states, obstacles, target, step_num, terminates, actions, obs,
                               rewards, terminated, truncated, stats, io);
    a.final_obs = final_obs;
    return dispatch_step_typed(a, obs_dtype, (cudaStream_t)stream);
}
}  // namespace

extern "C" {

int marlnav_step_typed(const marlnav_env_params* params, const marlnav_reset_spec* reset, float* states,
                       float* obstacles, float* target, float* step_num, uint8_t* terminates,
                       const float* actions, void* obs, int obs_dtype, float* rewards, uint8_t* terminated,
                       uint8_t* truncated, unsigned long long* stats, const marlnav_io_transform* io,
                       void* stream) {
    return step_typed(params, reset, states, obstacles, target, step_num, terminates, actions, obs, obs_dtype,
                      nullptr, rewards, terminated, truncated, stats, io, stream);
}

int marlnav_step_final_typed(const marlnav_env_params* params, const marlnav_reset_spec* reset, float* states,
                             float* obstacles, float* target, float* step_num, uint8_t* terminates,
                             const float* actions, void* obs, int obs_dtype, void* final_obs, float* rewards,
                             uint8_t* terminated, uint8_t* truncated, unsigned long long* stats,
                             const marlnav_io_transform* io, void* stream) {
    if (!final_obs) return fail(MARLNAV_ERR_BAD_ARG, "final_obs is NULL (marlnav_step_typed is the step without it)");
    if (final_obs == obs) return fail(MARLNAV_ERR_BAD_ARG, "final_obs and obs must be different buffers");
    return step_typed(params, reset, states, obstacles, target, step_num, terminates, actions, obs, obs_dtype,
                      final_obs, rewards, terminated, truncated, stats, io, stream);
}

int marlnav_step_f32(const marlnav_env_params* params, const marlnav_reset_spec* reset, float* states,
                     float* obstacles, float* target, float* step_num, uint8_t* terminates,
                     const float* actions, float* obs, float* rewards, uint8_t* terminated,
                     uint8_t* truncated, unsigned long long* stats, const marlnav_io_transform* io,
                     void* stream) {
    return marlnav_step_typed(params, reset, states, obstacles, target, step_num, terminates, actions, obs,
                              MARLNAV_OBS_F32, rewards, terminated, truncated, stats, io, stream);
}

int marlnav_step_call_typed(const marlnav_step_call* c, int obs_dtype) {
    if (int rc = check_obs_dtype(obs_dtype)) return rc;
    if (!c) return fail(MARLNAV_ERR_BAD_ARG, "call is NULL");
    if (c->struct_size != sizeof(marlnav_step_call)) return fail(MARLNAV_ERR_BAD_ARG, kSizeMsg, "marlnav_step_call");
    return marlnav_step_typed(c->params, c->reset, c->states, c->obstacles, c->target, c->step_num, c->terminates,
                              c->actions, c->obs, obs_dtype, c->rewards, c->terminated, c->truncated, c->stats, c->io,
                              c->stream);
}

int marlnav_step_call_f32(const marlnav_step_call* c) { return marlnav_step_call_typed(c, MARLNAV_OBS_F32); }

int marlnav_step_call_final_typed(const marlnav_step_call* c, int obs_dtype, void* final_obs) {
    if (int rc = check_obs_dtype(obs_dtype)) return rc;
    if (!c) return fail(MARLNAV_ERR_BAD_ARG, "call is NULL");
    if (c->struct_size != sizeof(marlnav_step_call)) return fail(MARLNAV_ERR_BAD_ARG, kSizeMsg, "marlnav_step_call");
    return marlnav_step_final_typed(c->params, c->reset, c->states, c->obstacles, c->target, c->step_num,
                                    c->terminates, c->actions, c->obs, obs_dtype, final_obs, c->rewards,
                                    c->terminated, c->truncated, c->stats, c->io, c->stream);
}

int marlnav_act_step_typed(const marlnav_env_params* params, const marlnav_reset_spec* reset, float* states,
                           float* obstacles, float* target, float* step_num, uint8_t* terminates,
                           const marlnav_actor_spec* actor, const void* obs_in, float* actions_out,
                           float* log_probs_out, void* obs, int obs_dtype, float* rewards, uint8_t* terminated,
                           uint8_t* truncated, unsigned long long* stats, const marlnav_io_transform* io,
                           void* stream) {
    if (int rc = check_obs_dtype(obs_dtype)) return rc;
    if (int rc = check_params(params)) return rc;
    if (int rc = check_reset(reset)) return rc;
    if (!states || !obstacles || !target || !step_num || !terminates || !actor || !obs_in || !actions_out ||
        !log_probs_out || !obs || !rewards || !terminated || !truncated || !stats)
        return fail(MARLNAV_ERR_BAD_ARG, "NULL tensor pointer");
    if (actor->struct_size != sizeof(marlnav_actor_spec)) return fail(MARLNAV_ERR_BAD_ARG, kSizeMsg, "marlnav_actor_spec");
    if (!actor->w1 || !actor->b1 || !actor->w_mu || !actor->b_mu || !actor->w_std || !actor->b_std)
        return fail(MARLNAV_ERR_BAD_ARG, "NULL actor weight pointer");
    if (io && io->struct_size != sizeof(marlnav_io_transform)) return fail(MARLNAV_ERR_BAD_ARG, kSizeMsg, "marlnav_io_transform");
    if (!io || !io->obs_mean || !io->obs_scale || !io->act_mean || !io->act_scale)
        return fail(MARLNAV_ERR_BAD_ARG, "the fused actor needs both io transforms (normalised observations, scaled actions)");
    if (params->num_agents != 3 || params->num_obstacles > 6)
        return fail(MARLNAV_ERR_BAD_SHAPE, "the fused actor exists for the thread-per-env kernels (3 agents, 1..6 obstacles)");
    if (actor->S != marlnav_obs_size(params->num_agents, params->num_obstacles) || actor->H < 1 ||
        actor->H > kMaxActorHidden)
        return fail(MARLNAV_ERR_BAD_SHAPE, "actor obs_size must equal the env's and 1 <= hidden <= 256");
    if (obs_in == obs) return fail(MARLNAV_ERR_BAD_ARG, "obs_in and obs must be different buffers");
    mn::StepArgs a = step_args(params, reset, states, obstacles, target, step_num, terminates, nullptr, obs, rewards,
                               terminated, truncated, stats, io);
    a.actor = *actor; a.obs_in = obs_in; a.act_out = actions_out; a.logp_out = log_probs_out;
    return dispatch_step_typed(a, obs_dtype, (cudaStream_t)stream);
}

int marlnav_act_step_f32(const marlnav_env_params* params, const marlnav_reset_spec* reset, float* states,
                         float* obstacles, float* target, float* step_num, uint8_t* terminates,
                         const marlnav_actor_spec* actor, const float* obs_in, float* actions_out,
                         float* log_probs_out, float* obs, float* rewards, uint8_t* terminated,
                         uint8_t* truncated, unsigned long long* stats, const marlnav_io_transform* io,
                         void* stream) {
    return marlnav_act_step_typed(params, reset, states, obstacles, target, step_num, terminates, actor, obs_in,
                                  actions_out, log_probs_out, obs, MARLNAV_OBS_F32, rewards, terminated, truncated,
                                  stats, io, stream);
}

// Host-resident policy: the batch is cut into chunks and the three legs of each chunk -- H2D of
// its actions, the fused step on it, D2H of its observations / rewards / flags -- run on three
// streams chained by events, so chunk c's download overlaps chunk c+1's upload and compute
// (PCIe is full duplex and the download is 6x the upload).  Chunk boundaries are multiples of
// 128 envs, which keeps every slice 16-byte aligned for the TMA path.  The caller's stream
// waits for the last download, so synchronising it is enough.
struct marlnav_host_pipe {
    int device = -1;
    cudaStream_t s_in = nullptr, s_out = nullptr;
    cudaEvent_t entry = nullptr, exit_ev = nullptr;
    cudaEvent_t up[16] = {}, done[16] = {};
};

void marlnav_host_pipe_destroy(marlnav_host_pipe* hp) {
    if (!hp) return;
    for (int i = 0; i < 16; ++i) { if (hp->up[i]) cudaEventDestroy(hp->up[i]); if (hp->done[i]) cudaEventDestroy(hp->done[i]); }
    if (hp->entry) cudaEventDestroy(hp->entry);
    if (hp->exit_ev) cudaEventDestroy(hp->exit_ev);
    if (hp->s_in) cudaStreamDestroy(hp->s_in);
    if (hp->s_out) cudaStreamDestroy(hp->s_out);
    delete hp;
}

int marlnav_host_pipe_create(marlnav_host_pipe** out) {
    if (!out) return fail(MARLNAV_ERR_BAD_ARG, "pipe is NULL");
    *out = nullptr;
    marlnav_host_pipe* hp = new marlnav_host_pipe;
    hp->device = current_device();
    cudaError_t e = cudaStreamCreateWithFlags(&hp->s_in, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&hp->s_out, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&hp->entry, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&hp->exit_ev, cudaEventDisableTiming);
    for (int i = 0; i < 16 && e == cudaSuccess; ++i) {
        e = cudaEventCreateWithFlags(&hp->up[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&hp->done[i], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) { marlnav_host_pipe_destroy(hp); return cuda_fail(e, "host pipeline streams/events"); }
    *out = hp;
    return 0;
}

int marlnav_step_host_typed(marlnav_host_pipe* hp, const marlnav_env_params* params, const marlnav_reset_spec* reset,
                            float* states, float* obstacles, float* target, float* step_num, uint8_t* terminates,
                            const float* actions_host, float* actions_dev, void* obs_dev, float* rewards_dev,
                            uint8_t* terminated_dev, uint8_t* truncated_dev, void* obs_host,
                            float* rewards_host, uint8_t* terminated_host, uint8_t* truncated_host,
                            unsigned long long* stats, const marlnav_io_transform* io, void* stream, int obs_dtype) {
    if (int rc = check_obs_dtype(obs_dtype)) return rc;
    if (int rc = check_params(params)) return rc;
    if (int rc = check_reset(reset)) return rc;
    if (!actions_host || !actions_dev || !obs_dev || !rewards_dev || !terminated_dev || !truncated_dev ||
        !obs_host || !rewards_host || !terminated_host || !truncated_host)
        return fail(MARLNAV_ERR_BAD_ARG, "NULL host/staging pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const long long B = params->num_envs;
    const size_t A = params->num_agents, O = params->num_obstacles;
    const size_t S = (size_t)marlnav_obs_size(params->num_agents, params->num_obstacles);
    const size_t esz = obs_elem_size(obs_dtype);     // bytes per observation element
    char* const obs_dev_b = static_cast<char*>(obs_dev);
    char* const obs_host_b = static_cast<char*>(obs_host);
    if (!hp) return fail(MARLNAV_ERR_BAD_ARG, "pipe is NULL (marlnav_host_pipe_create)");
    if (hp->device != current_device()) return fail(MARLNAV_ERR_BAD_ARG, "the host pipe belongs to another device");

    // up to 8 chunks of at least 32768 envs, boundaries on multiples of 128 envs
    int nchunk = (int)(B / 32768);
    nchunk = nchunk < 1 ? 1 : (nchunk > 8 ? 8 : nchunk);
    long long per = ((B + nchunk - 1) / nchunk + 127) / 128 * 128;

    cudaError_t e;
    if ((e = cudaEventRecord(hp->entry, st)) != cudaSuccess) return cuda_fail(e, "event record");
    if ((e = cudaStreamWaitEvent(hp->s_in, hp->entry, 0)) != cudaSuccess) return cuda_fail(e, "stream wait");
    if ((e = cudaStreamWaitEvent(hp->s_out, hp->entry, 0)) != cudaSuccess) return cuda_fail(e, "stream wait");
    // the first two chunks are 1/4 and 1/2 of a chunk: the first download starts after a quarter of the
    // fill (one chunk's upload and step) -- median 3.004 vs 3.041 ms per 1M-env step over 6 + 6
    // interleaved runs (by an A/B script removed once the ramp became unconditional)
    int c = 0;
    long long n = 0;
    for (long long lo = 0; lo < B; lo += n, ++c) {
        long long want = per;
        if (nchunk >= 4 && c < 2) want = (per >> (2 - c)) / 128 * 128;
        if (c == 15) want = B - lo;              // 16 events per pipe
        n = (B - lo) < want ? (B - lo) : want;
        if ((e = cudaMemcpyAsync(actions_dev + lo * A * 2, actions_host + lo * A * 2, (size_t)n * A * 2 * sizeof(float),
                                 cudaMemcpyHostToDevice, hp->s_in)) != cudaSuccess) return cuda_fail(e, "H2D actions");
        cudaEventRecord(hp->up[c], hp->s_in);
        cudaStreamWaitEvent(st, hp->up[c], 0);
        marlnav_env_params pc = *params;
        pc.num_envs = (int32_t)n;
        marlnav_reset_spec rc2 = *reset;
        rc2.env_id_offset += (uint64_t)lo;
        if (rc2.tmpl_states) rc2.tmpl_states += lo * rc2.states_env_stride;
        if (rc2.tmpl_obstacles) rc2.tmpl_obstacles += lo * rc2.obstacles_env_stride;
        if (rc2.tmpl_target) rc2.tmpl_target += lo * rc2.target_env_stride;
        if (int rc = marlnav_step_typed(&pc, &rc2, states + lo * A * 5, obstacles + lo * O * 2, target + lo * 2,
                                        step_num + lo, terminates + lo, actions_dev + lo * A * 2,
                                        obs_dev_b + lo * A * S * esz, obs_dtype, rewards_dev + lo, terminated_dev + lo,
                                        truncated_dev + lo, stats, io, stream))
            return rc;
        cudaEventRecord(hp->done[c], st);
        cudaStreamWaitEvent(hp->s_out, hp->done[c], 0);
        if ((e = cudaMemcpyAsync(obs_host_b + lo * A * S * esz, obs_dev_b + lo * A * S * esz, (size_t)n * A * S * esz,
                                 cudaMemcpyDeviceToHost, hp->s_out)) != cudaSuccess) return cuda_fail(e, "D2H obs");
    }
    // rewards and flags once for the whole batch, behind the last chunk's observations: as 3 x nchunk
    // small copies they cost ~4 us each on the link (scripts/pcie_probe.py: 2.93 vs 2.85 ms per step)
    if ((e = cudaMemcpyAsync(rewards_host, rewards_dev, (size_t)B * sizeof(float), cudaMemcpyDeviceToHost,
                             hp->s_out)) != cudaSuccess) return cuda_fail(e, "D2H rewards");
    if ((e = cudaMemcpyAsync(terminated_host, terminated_dev, (size_t)B, cudaMemcpyDeviceToHost,
                             hp->s_out)) != cudaSuccess) return cuda_fail(e, "D2H terminated");
    if ((e = cudaMemcpyAsync(truncated_host, truncated_dev, (size_t)B, cudaMemcpyDeviceToHost,
                             hp->s_out)) != cudaSuccess) return cuda_fail(e, "D2H truncated");
    if ((e = cudaEventRecord(hp->exit_ev, hp->s_out)) != cudaSuccess) return cuda_fail(e, "event record");
    if ((e = cudaStreamWaitEvent(st, hp->exit_ev, 0)) != cudaSuccess) return cuda_fail(e, "stream wait");
    return 0;
}

int marlnav_step_host_f32(marlnav_host_pipe* hp, const marlnav_env_params* params, const marlnav_reset_spec* reset, float* states,
                          float* obstacles, float* target, float* step_num, uint8_t* terminates,
                          const float* actions_host, float* actions_dev, float* obs_dev, float* rewards_dev,
                          uint8_t* terminated_dev, uint8_t* truncated_dev, float* obs_host,
                          float* rewards_host, uint8_t* terminated_host, uint8_t* truncated_host,
                          unsigned long long* stats, const marlnav_io_transform* io, void* stream) {
    return marlnav_step_host_typed(hp, params, reset, states, obstacles, target, step_num, terminates, actions_host,
                                   actions_dev, obs_dev, rewards_dev, terminated_dev, truncated_dev, obs_host,
                                   rewards_host, terminated_host, truncated_host, stats, io, stream, MARLNAV_OBS_F32);
}

int marlnav_step_launch_info(const marlnav_env_params* params, int* grid, int* block, int* smem_bytes,
                             int* envs_per_cta) {
    if (int rc = check_params(params)) return rc;
    mn::StepArgs a; memset(&a, 0, sizeof a); a.p = *params;
    int info[4] = {0, 0, 0, 0};
    if (int rc = dispatch_step<float>(a, nullptr, info)) return rc;
    if (grid) *grid = info[0];
    if (block) *block = info[1];
    if (smem_bytes) *smem_bytes = info[2];
    if (envs_per_cta) *envs_per_cta = info[3];
    return 0;
}

}  // extern "C"
