// marlnav_b200/csrc/marlnav_step_launch.cuh
//
// Host-side launch code shared by the step library's units: the launch path of the two
// one-warp-CTA kernel families (step_env_kernel, step_team_kernel), and the entry point each
// kernel-family unit exports to the dispatcher in marlnav_abi.cu.  Every kernel template is
// defined, instantiated and launched in one unit; the others see only these entry points.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stddef.h>

#include <type_traits>

#include "marlnav_launch.cuh"
#include "marlnav_step.cuh"

namespace mn {
// defined in marlnav_step_env.cu and marlnav_step_team.cu; launch_step_tile_n names both
template <int TA, int TO, class OT> struct EnvTile;
template <int TA, int TO, class OT> struct TeamTile;
template <int TA, int TO, bool NORM, class DM, bool ACTOR, class OT> __global__ void step_env_kernel(const StepArgs args);
template <int TA, int TO, bool NORM, class DM, bool ACTOR, class OT> __global__ void step_team_kernel(const StepArgs args);
// defined in marlnav_step_generic.cu, launched by marlnav_init_f32 and marlnav_counter_add
__global__ void init_kernel(const marlnav_env_params p, const marlnav_reset_spec rs, float* states,
                            float* obstacles, float* target, float* step_num, uint8_t* terminates);
__global__ void counter_add_kernel(unsigned long long* ctr, unsigned long long inc);
}  // namespace mn

namespace mnl {

// Records a failed CUDA call for marlnav_last_error() (defined in marlnav_abi.cu) and returns its code.
int cuda_fail(cudaError_t e, const char* where);

constexpr int kMaxActorHidden = 256;

// Launch a one-warp-CTA step kernel with programmatic stream serialization: consecutive step
// kernels of a stream overlap the next one's prologue with this one's tail (1M x 3 x 3: 70.9 ->
// 68.9 us per step; (8,16): 170.1 -> 167.9).  The fused-actor launches of a rollout do not use
// it: inside a captured graph with the critic on a parallel branch it measured slower (11.9 ->
// 13.7 us per iteration at 1 024 envs).
template <typename Kernel>
cudaError_t launch_pdl(Kernel kernel, int grid, size_t smem, cudaStream_t st, const mn::StepArgs& a, bool allow) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(32); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = allow ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, a);
}

inline int div_mode_of(float c, float rc) {
    return c == 1.0f ? mn::DIV_UNIT : rc < 0.0f ? mn::DIV_POW2 : rc > 0.0f ? mn::DIV_PROVEN : mn::DIV_RT;
}
template <class DM>
bool div_modes_match(const mn::StepArgs& a) {
    const bool wash_only = (a.rs.flags & MARLNAV_RESET_TMPL_NONNEG) != 0 && a.rs.alias_first_step == 0 &&
                           (a.rs.flags & MARLNAV_RESET_NOISY_AGENTS) == 0 && a.rs.states_env_stride == 0;
    return (DM::kWash == 0 || wash_only) &&
           div_mode_of(a.p.init_dist, a.rc_init_dist) == DM::kInit && div_mode_of(a.p.max_at_prop_d, a.rc_prop_d) == DM::kProp &&
           div_mode_of(a.p.bond_sharpness, a.rc_sharp) == DM::kSharp &&
           div_mode_of((float)(a.p.num_agents - 1), a.rc_R) == DM::kR && div_mode_of((float)a.p.num_agents, a.rc_A) == DM::kA;
}
// The one-warp-CTA step kernels: step_env_kernel (one env per lane) for Tile = EnvTile,
// step_team_kernel (one agent per lane) for Tile = TeamTile.
template <template <int, int, class> class Tile, int TA, int TO, bool NORM, class DM, bool ACTOR, class OT>
int launch_step_tile_n(const mn::StepArgs& a, cudaStream_t st, int* info) {
    using W = Tile<TA, TO, OT>;
    constexpr bool kTeam = std::is_same_v<W, mn::TeamTile<TA, TO, OT>>;
    constexpr auto kernel = [] {
        if constexpr (kTeam) return mn::step_team_kernel<TA, TO, NORM, DM, ACTOR, OT>;
        else return mn::step_env_kernel<TA, TO, NORM, DM, ACTOR, OT>;
    }();
    // fused actor: its weights sit behind the tile and the mbarrier
    const auto actor_bytes = [](int H) { return ACTOR ? 8 + ((size_t)H * W::S + 5 * (size_t)H) * 4 : (size_t)0; };
    const size_t smem = W::smem_bytes() + actor_bytes(a.actor.H);
    const int grid = (a.p.num_envs + W::ENVS - 1) / W::ENVS;
    if (info) { info[0] = grid; info[1] = 32; info[2] = (int)smem; info[3] = W::ENVS; return 0; }
    if (cudaError_t e = mnl::set_attributes_once<kernel>(W::smem_bytes() + actor_bytes(kMaxActorHidden), true))
        return cuda_fail(e, kTeam ? "cudaFuncSetAttribute(step_team)" : "cudaFuncSetAttribute(step_env)");
    cudaError_t e = launch_pdl(kernel, grid, smem, st, a, !ACTOR);
    if (e == cudaSuccess) e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail(e, kTeam ? "step_team kernel launch" : "step_env kernel launch");
}
template <template <int, int, class> class Tile, int TA, int TO, class DM, class OT>
int launch_step_tile_d(const mn::StepArgs& a, cudaStream_t st, int* info) {
    // the fused actor exists for the reference's team only (it needs io), and not with final_obs
    if constexpr (TA < 4 && DM::kFinal == 0) {
        if (a.obs_in) return launch_step_tile_n<Tile, TA, TO, true, DM, true, OT>(a, st, info);
    }
    return a.io.obs_mean ? launch_step_tile_n<Tile, TA, TO, true, DM, false, OT>(a, st, info)
                         : launch_step_tile_n<Tile, TA, TO, false, DM, false, OT>(a, st, info);
}
// The kernel specialised on the shape's constant divisors DMD when the launch has them (the
// host's verdict on each divisor matches DMD), the run-time-mode build otherwise.
template <template <int, int, class> class Tile, int TA, int TO, class DMD, class OT>
int launch_step_tile(const mn::StepArgs& a, cudaStream_t st, int* info) {
    // `info` queries carry no constants; the launch geometry does not depend on the profile
    if (!info && a.final_obs) return launch_step_tile_d<Tile, TA, TO, mn::DivModesFinal, OT>(a, st, info);
    if (info || div_modes_match<DMD>(a)) return launch_step_tile_d<Tile, TA, TO, DMD, OT>(a, st, info);
    return launch_step_tile_d<Tile, TA, TO, mn::DivModesRT, OT>(a, st, info);
}

// The kernel-family entry points, for OT = float, __half and __nv_bfloat16.  Each returns 0 or a
// CUDA error code (positive); with `info` set it fills the launch geometry instead of launching.
// launch_env3 / launch_team3 return -1 when num_obstacles is outside 1..6 (no build for it).
template <class OT> int launch_env3(const mn::StepArgs& a, cudaStream_t st, int* info);       // marlnav_step_env.cu
template <class OT> int launch_team3(const mn::StepArgs& a, cudaStream_t st, int* info);      // marlnav_step_team.cu
template <class OT> int launch_team8x16(const mn::StepArgs& a, cudaStream_t st, int* info);   // marlnav_step_team.cu
template <class OT> int launch_generic(const mn::StepArgs& a, cudaStream_t st, int* info);    // marlnav_step_generic.cu
template <class OT> int dispatch_observe(const mn::ObserveArgs& a, cudaStream_t st);          // marlnav_step_generic.cu

}  // namespace mnl
