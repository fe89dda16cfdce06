// marlnav_b200/csrc/marlnav_step_generic.cu
//
// The CTA-tiled kernels and their launchers: the generic step_kernel (shape read at run time, for
// every team the one-warp kernels do not cover) and observe_kernel; and init_kernel and
// counter_add_kernel, which marlnav_abi.cu launches.  Device code shared with the other step
// kernels is in marlnav_step.cuh.
#include "marlnav_step_launch.cuh"

namespace mn {

// ----------------------------------------------------------------------------- the step kernel

// OTF: the observations' element type OT, or FinalObs<OT> for the build that also copies the
// pre-reset observations of the finished envs to args.final_obs (a tag type, not a template
// parameter, so that no existing kernel is renamed)
template <class OT> struct FinalObs {};
template <class T> struct ObsType { using type = T; static constexpr bool kFinal = false; };
template <class T> struct ObsType<FinalObs<T>> { using type = T; static constexpr bool kFinal = true; };

template <int TA, int TO, int LPE, int THREADS, bool NORM, class OTF = float>
__global__ void __launch_bounds__(THREADS, (THREADS == 128 ? 7 : 3))
step_kernel(const StepArgs args) {
    using OT = typename ObsType<OTF>::type;
    constexpr bool FINAL = ObsType<OTF>::kFinal;
    using G = Geo<TA, TO, LPE, THREADS>;
    constexpr int TILE = G::TILE;
    const marlnav_env_params& p = args.p;
    const marlnav_reset_spec& rs = args.rs;
    const G g(p.num_agents, p.num_obstacles);
    const int A = g.A, O = g.O, S = g.S;
    const DivConsts rc{args.rc_init_dist, args.rc_prop_d, args.rc_sharp, args.rc_R, args.rc_A};

    extern __shared__ float4 smem_raw[];
    const Smem<G, OT> sm(g, reinterpret_cast<float*>(smem_raw));
    OT* const obs = reinterpret_cast<OT*>(args.obs);
    const int obs_stride = g.template obs_stride_of<OT>();

    const int tid = threadIdx.x;
    const long long env0 = (long long)blockIdx.x * TILE;
    const int nenv = (int)min((long long)TILE, (long long)p.num_envs - env0);
    const bool vec = args.vec_ok != 0;

    const int le = tid / LPE;            // local env
    const int la = tid % LPE;            // lane within the env's group
    const bool active = le < nenv;
    const long long env = env0 + le;
    const bool leader = active && la == 0;

    // ---- P0: stage in.  Actions are read once by their own thread: straight to registers.
    float2 acts[LPE == 1 ? (G::kStatic ? TA : 1) : 1];
    if constexpr (G::kStatic) {
        if (active) {
#pragma unroll
            for (int i = 0; i < (LPE == 1 ? A : 1); ++i) acts[i] = load_action(args.actions, env * A + (LPE == 1 ? i : la), args.act8 != 0);
        }
    }
    copy_in<THREADS, false>(sm.st, args.states + env0 * g.st_row, nenv * g.st_row, vec);
    if (g.ob_stride == g.ob_row) copy_in<THREADS, false>(sm.ob, args.obstacles + env0 * g.ob_row, nenv * g.ob_row, vec);
    else copy_in_rows<THREADS>(sm.ob, g.ob_stride, args.obstacles + env0 * g.ob_row, g.ob_row, nenv);
    copy_in<THREADS, false>(sm.tg, args.target + env0 * 2, nenv * 2, vec);
    if (tid < 4) sm.cnt[tid] = 0u;
    __syncthreads();

    if (active) {
        // ---- P1: move (ActionScaler, utils.py:546-547, folded into the action load)
        float* st_env = sm.st + le * g.st_row;
        const bool scale_act = args.io.act_scale != nullptr;
        const float am0 = scale_act ? __ldg(args.io.act_mean + 0) : 0.f;
        const float am1 = scale_act ? __ldg(args.io.act_mean + 1) : 0.f;
        const float as0 = scale_act ? __ldg(args.io.act_scale + 0) : 1.f;
        const float as1 = scale_act ? __ldg(args.io.act_scale + 1) : 1.f;
#pragma unroll
        for (int i = 0; i < (LPE == 1 ? A : 1); ++i) {
            const int a = LPE == 1 ? i : la;
            float2 act;
            if constexpr (G::kStatic) act = acts[i];
            else act = load_action(args.actions, env * A + a, args.act8 != 0);
            if (scale_act) { act.x = (as0 * act.x) + am0; act.y = (as1 * act.y) + am1; }
            float s[5];
#pragma unroll
            for (int k = 0; k < 5; ++k) s[k] = st_env[5 * a + k];
            move_agent(p, s, act.x, act.y);
#pragma unroll
            for (int k = 0; k < 5; ++k) st_env[5 * a + k] = s[k];
        }
    }
    if (LPE > 1) __syncwarp();

    // ---- work loop: iteration 0 observes this thread's own env (P2) and does the per-env
    // bookkeeping (P3, P4a); later iterations re-observe single agents of the envs that were
    // reset (P4b).  One loop so that the (large) observation code exists once in the binary.
    int e_cur = le, a_lo = (LPE == 1 ? 0 : la), a_hi = (LPE == 1 ? A : la + 1);
    bool have = active, first = true;
    int w = tid, n_items = 0, ndone = 0;
#pragma unroll 1
    while (true) {
        bool all_in = true, coll_any = false;
        float sum_out = 0.f, sum_in = 0.f, r_out = 0.f, r_in = 0.f;
        if (have) {
            const float* st_env = sm.st + e_cur * g.st_row;
            const float* ob_env = sm.ob + e_cur * g.ob_stride;
            const float2 tg = *reinterpret_cast<const float2*>(sm.tg + e_cur * 2);
#pragma unroll 1
            for (int a = a_lo; a < a_hi; ++a) {
                ObsRow<NORM, OT> sink;
                if constexpr (G::kObsSmem) sink.row = sm.obs + ((size_t)e_cur * A + a) * obs_stride;
                else sink.row = obs + ((size_t)(env0 + e_cur) * A + a) * S;
                sink.mean = args.io.obs_mean; sink.scale = args.io.obs_scale;
                AgentTerms tm;
                observe_agent<G, NORM>(g, p, rc, st_env, ob_env, tg.x, tg.y, a, sink, tm);
                all_in = all_in && tm.in_t;
                coll_any = coll_any || tm.coll;
                agent_reward2(p, tm, r_out, r_in);
                if constexpr (!G::kRewardSmem) { sum_out = sum_out + r_out; sum_in = sum_in + r_in; }
                else if constexpr (LPE == 1) { sm.rw[(e_cur * A + a) * 2] = r_out; sm.rw[(e_cur * A + a) * 2 + 1] = r_in; }
            }
        }
        if (first) {
            first = false;
            float reward = 0.f;
            if constexpr (LPE > 1) {
                // combine over the env's lanes (groups are aligned sub-warps)
                const unsigned lane = tid & 31u;
                const unsigned gmask = (LPE == 32 ? 0xffffffffu : ((1u << LPE) - 1u)) << (lane & ~(unsigned)(LPE - 1));
                const unsigned b_in = __ballot_sync(0xffffffffu, all_in);
                const unsigned b_co = __ballot_sync(0xffffffffu, coll_any);
                all_in = (b_in & gmask) == gmask;
                coll_any = (b_co & gmask) != 0u;
                if (active) sm.rw[le * A + la] = all_in ? r_in : r_out;
                __syncwarp();
                if (leader) reward = div_const(torch_row_sum(sm.rw + le * A, A), (float)A, rc.A);
            } else if (active) {
                if constexpr (!G::kRewardSmem) {
                    // torch.mean over A < 4 agents: sequential sum from 0, then three idle accumulators
                    reward = div_const((all_in ? sum_in : sum_out) + 0.0f, (float)A, rc.A);
                } else {
                    float r[G::kStatic ? TA : MARLNAV_MAX_AGENTS];
                    for (int a = 0; a < A; ++a) r[a] = sm.rw[(le * A + a) * 2 + (all_in ? 1 : 0)];
                    reward = div_const(torch_row_sum(r, A), (float)A, rc.A);
                }
            }

            // ---- P3: per-env flags, counters, outputs (environment.py:96-103, 209-221)
            bool done = false, trunc = false;
            if (leader) {
                const float sn = args.step_num[env] + 1.0f;
                trunc = sn > (float)(p.episode_len - 1);
                const bool term_old = args.terminates[env] != 0;
                const bool term = coll_any || term_old;
                done = term || trunc;
                args.terminates[env] = (uint8_t)((!term_old) && all_in);
                args.rewards[env] = reward;
                args.terminated[env] = (uint8_t)term;
                args.truncated[env] = (uint8_t)trunc;
                args.step_num[env] = done ? ((0.0f * sn) + 0.0f) : (sn + 0.0f);   // (1-m)*sn + m*0
                if (done) sm.done[atomicAdd(&sm.cnt[0], 1u)] = le;
            }
            {
                const unsigned b_tr = __ballot_sync(0xffffffffu, leader && trunc);
                const unsigned b_co = __ballot_sync(0xffffffffu, leader && coll_any);
                const unsigned b_ta = __ballot_sync(0xffffffffu, leader && all_in);
                if ((tid & 31) == 0) {
                    if (b_tr) atomicAdd(&sm.cnt[1], (unsigned)__popc(b_tr));
                    if (b_co) atomicAdd(&sm.cnt[2], (unsigned)__popc(b_co));
                    if (b_ta) atomicAdd(&sm.cnt[3], (unsigned)__popc(b_ta));
                }
            }
            if constexpr (LPE > 1) done = __shfl_sync(0xffffffffu, (int)done, (tid & 31) & ~(LPE - 1)) != 0;

            // ---- P4a: masked re-initialisation (environment.py:76-90): x = (1-m)*x + m*new
            if (active) {
                float* st_env = sm.st + le * g.st_row;
                float* ob_env = sm.ob + le * g.ob_stride;
                const bool alias = rs.alias_first_step != 0;
                const bool noisy = (rs.flags & MARLNAV_RESET_NOISY_AGENTS) != 0;
                const float* ts = rs.tmpl_states + env * rs.states_env_stride;
#pragma unroll 1
                for (int i = 0; i < (LPE == 1 ? A : 1); ++i) {
                    const int a = LPE == 1 ? i : la;
                    float nv[5];
                    if (noisy) sample_agent_noisy(rs, reset_counter(rs), rs.env_id_offset + (uint64_t)env, a, ts + 5 * a, nv);
#pragma unroll
                    for (int k = 0; k < 5; ++k) {
                        const float old_v = st_env[5 * a + k];
                        const float new_v = noisy ? nv[k] : (alias ? old_v : __ldg(ts + 5 * a + k));
                        // m = 1: 0*old + 1*new ; m = 0: 1*old + 0*new
                        st_env[5 * a + k] = done ? ((0.0f * old_v) + new_v) : (old_v + (0.0f * new_v));
                    }
                }
                if (done) {
                    // obstacles / target are rewritten only for envs that reset; for the others
                    // (1-0)*x + 0*new == x for every value the initialisers can produce
                    if (rs.tmpl_obstacles || alias) {
                        const float* to = alias ? nullptr : rs.tmpl_obstacles + env * rs.obstacles_env_stride;
                        for (int c = la; c < g.ob_row; c += LPE) {
                            const float old_v = ob_env[c];
                            ob_env[c] = (0.0f * old_v) + (alias ? old_v : __ldg(to + c));
                        }
                    } else {
                        for (int pr = la; 2 * pr < O; pr += LPE) {
                            float nw[4];
                            sample_obstacle_pair(p, rs.seed, reset_counter(rs), rs.env_id_offset + (uint64_t)env, pr, nw);
#pragma unroll
                            for (int c = 0; c < 4; ++c)
                                if (4 * pr + c < g.ob_row) ob_env[4 * pr + c] = (0.0f * ob_env[4 * pr + c]) + nw[c];
                        }
                    }
                    if (la == 0) {
                        const float* tt = rs.tmpl_target + env * rs.target_env_stride;
#pragma unroll
                        for (int c = 0; c < 2; ++c) {
                            const float old_v = sm.tg[le * 2 + c];
                            sm.tg[le * 2 + c] = (0.0f * old_v) + (alias ? old_v : __ldg(tt + c));
                        }
                    }
                }
            }
            __syncthreads();
            ndone = (int)sm.cnt[0];
            n_items = ndone * A;        // P4b work items: (reset env, agent)
            w = tid;
            if constexpr (FINAL) {
                // the finished envs' rows, complete in global memory, before P4b rewrites them
                static_assert(!G::kObsSmem, "the final-observation copy reads rows from global memory");
                OT* const fin = static_cast<OT*>(args.final_obs);
                const int per = A * S;
                for (int i = tid; i < ndone * per; i += THREADS) {
                    const size_t at = (size_t)(env0 + sm.done[i / per]) * per + i % per;
                    fin[at] = obs[at];
                }
                __syncthreads();
            }
        } else {
            w += THREADS;
        }
        if (w >= n_items) break;
        e_cur = sm.done[w / A];
        a_lo = w % A; a_hi = a_lo + 1;
        have = true;
    }
    __syncthreads();

    // ---- P5: stage out
    copy_out<THREADS>(args.states + env0 * g.st_row, sm.st, nenv * g.st_row, vec);
    if constexpr (G::kObsSmem)
        copy_out_obs<THREADS>(obs + (size_t)env0 * A * S, sm.obs, S, obs_stride, nenv * A, vec);
    {
        const int per = g.ob_row + 2;
        for (int i = tid; i < ndone * per; i += THREADS) {
            const int e2 = sm.done[i / per], c = i % per;
            if (c < g.ob_row) args.obstacles[(env0 + e2) * g.ob_row + c] = sm.ob[e2 * g.ob_stride + c];
            else args.target[(env0 + e2) * 2 + (c - g.ob_row)] = sm.tg[e2 * 2 + (c - g.ob_row)];
        }
    }
    if (tid >= 1 && tid < 4 && sm.cnt[tid]) atomicAdd(args.stats + (tid - 1), (unsigned long long)sm.cnt[tid]);
}


// ----------------------------------------------------------------------------- observe-only kernel

template <int TA, int TO, int LPE, int THREADS, class OT = float>
__global__ void __launch_bounds__(THREADS)
observe_kernel(const ObserveArgs args) {
    using G = Geo<TA, TO, LPE, THREADS>;
    constexpr int TILE = G::TILE;
    const marlnav_env_params& p = args.p;
    const G g(p.num_agents, p.num_obstacles);
    const int A = g.A, S = g.S;
    const DivConsts rc{0.f, 0.f, 0.f, 0.f, 0.f};
    extern __shared__ float4 smem_raw[];
    const Smem<G, OT> sm(g, reinterpret_cast<float*>(smem_raw));
    OT* const obs = reinterpret_cast<OT*>(args.obs);
    const int obs_stride = g.template obs_stride_of<OT>();
    const int tid = threadIdx.x;
    const long long env0 = (long long)blockIdx.x * TILE;
    const int nenv = (int)min((long long)TILE, (long long)p.num_envs - env0);
    const bool vec = args.vec_ok != 0;

    copy_in<THREADS, true>(sm.st, args.states + env0 * g.st_row, nenv * g.st_row, vec);
    if (g.ob_stride == g.ob_row) copy_in<THREADS, true>(sm.ob, args.obstacles + env0 * g.ob_row, nenv * g.ob_row, vec);
    else copy_in_rows<THREADS>(sm.ob, g.ob_stride, args.obstacles + env0 * g.ob_row, g.ob_row, nenv);
    copy_in<THREADS, true>(sm.tg, args.target + env0 * 2, nenv * 2, vec);
    __syncthreads();

    const int le = tid / LPE, la = tid % LPE;
    if (le < nenv) {
        const float2 tg = *reinterpret_cast<const float2*>(sm.tg + le * 2);
        const int a_lo = LPE == 1 ? 0 : la, a_hi = LPE == 1 ? A : la + 1;
#pragma unroll 1
        for (int a = a_lo; a < a_hi; ++a) {
            ObsRow<false, OT> sink;
            if constexpr (G::kObsSmem) sink.row = sm.obs + ((size_t)le * A + a) * obs_stride;
            else sink.row = obs + ((size_t)(env0 + le) * A + a) * S;
            sink.mean = nullptr; sink.scale = nullptr;
            AgentTerms unused;
            observe_agent<G, false>(g, p, rc, sm.st + le * g.st_row, sm.ob + le * g.ob_stride, tg.x, tg.y, a, sink, unused);
        }
    }
    if constexpr (G::kObsSmem) {
        __syncthreads();
        copy_out_obs<THREADS>(obs + (size_t)env0 * A * S, sm.obs, S, obs_stride, nenv * A, vec);
    }
}


// ----------------------------------------------------------------------------- init kernel

// Env.__init__'s first sampler call + counters (environment.py:26-40).
__global__ void init_kernel(const marlnav_env_params p, const marlnav_reset_spec rs, float* states,
                            float* obstacles, float* target, float* step_num, uint8_t* terminates) {
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.num_envs) return;
    const int A = p.num_agents, O = p.num_obstacles;
    const float* ts = rs.tmpl_states + env * rs.states_env_stride;
    if (rs.flags & MARLNAV_RESET_NOISY_AGENTS) {
        for (int a = 0; a < A; ++a) {
            float nv[5];
            sample_agent_noisy(rs, reset_counter(rs), rs.env_id_offset + (uint64_t)env, a, ts + 5 * a, nv);
            for (int k = 0; k < 5; ++k) states[env * 5 * A + 5 * a + k] = nv[k];
        }
    } else {
        for (int k = 0; k < 5 * A; ++k) states[env * 5 * A + k] = __ldg(ts + k);
    }
    if (rs.tmpl_obstacles) {
        const float* to = rs.tmpl_obstacles + env * rs.obstacles_env_stride;
        for (int k = 0; k < 2 * O; ++k) obstacles[env * 2 * O + k] = __ldg(to + k);
    } else {
        for (int pr = 0; 2 * pr < O; ++pr) {
            float nw[4];
            sample_obstacle_pair(p, rs.seed, reset_counter(rs), rs.env_id_offset + (uint64_t)env, pr, nw);
            for (int c = 0; c < 4; ++c)
                if (4 * pr + c < 2 * O) obstacles[env * 2 * O + 4 * pr + c] = nw[c];
        }
    }
    const float* tt = rs.tmpl_target + env * rs.target_env_stride;
    target[env * 2 + 0] = __ldg(tt + 0); target[env * 2 + 1] = __ldg(tt + 1);
    step_num[env] = 0.f; terminates[env] = 0;
}

__global__ void counter_add_kernel(unsigned long long* ctr, unsigned long long inc) { *ctr += inc; }

}  // namespace mn

namespace mnl {

template <int TA, int TO, int LPE, int THREADS, bool NORM, bool FINAL, class OT>
int launch_step_n(const mn::StepArgs& a, cudaStream_t st, int* info) {
    using G = mn::Geo<TA, TO, LPE, THREADS>;
    const G g(a.p.num_agents, a.p.num_obstacles);
    const size_t smem = g.template smem_bytes<OT>();
    const int grid = (a.p.num_envs + G::TILE - 1) / G::TILE;
    if (info) { info[0] = grid; info[1] = THREADS; info[2] = (int)smem; info[3] = G::TILE; return 0; }
    // launches with final_obs take the build that copies the finished envs' rows out
    constexpr auto kernel = mn::step_kernel<TA, TO, LPE, THREADS, NORM, std::conditional_t<FINAL, mn::FinalObs<OT>, OT>>;
    if (cudaError_t e = mnl::set_attributes_once<kernel>(smem, true))
        return cuda_fail(e, "cudaFuncSetAttribute(step)");
    kernel<<<grid, THREADS, smem, st>>>(a);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail(e, "step kernel launch");
}
template <int TA, int TO, int LPE, int THREADS, class OT>
int launch_step(const mn::StepArgs& a, cudaStream_t st, int* info) {
    if (a.final_obs)
        return a.io.obs_mean ? launch_step_n<TA, TO, LPE, THREADS, true, true, OT>(a, st, info)
                             : launch_step_n<TA, TO, LPE, THREADS, false, true, OT>(a, st, info);
    return a.io.obs_mean ? launch_step_n<TA, TO, LPE, THREADS, true, false, OT>(a, st, info)
                         : launch_step_n<TA, TO, LPE, THREADS, false, false, OT>(a, st, info);
}

template <int TA, int TO, int LPE, int THREADS, class OT>
int launch_observe(const mn::ObserveArgs& a, cudaStream_t st) {
    using G = mn::Geo<TA, TO, LPE, THREADS>;
    const G g(a.p.num_agents, a.p.num_obstacles);
    const size_t smem = g.template smem_bytes<OT>();
    const int grid = (a.p.num_envs + G::TILE - 1) / G::TILE;
    if (cudaError_t e = mnl::set_attributes_once<mn::observe_kernel<TA, TO, LPE, THREADS, OT>>(smem, false))
        return cuda_fail(e, "cudaFuncSetAttribute(observe)");
    mn::observe_kernel<TA, TO, LPE, THREADS, OT><<<grid, THREADS, smem, st>>>(a);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail(e, "observe kernel launch");
}

template <class OT>
int launch_generic(const mn::StepArgs& a, cudaStream_t st, int* info) {
    return launch_step<0, 0, 1, 128, OT>(a, st, info);
}
template <class OT = float>
int dispatch_observe(const mn::ObserveArgs& a, cudaStream_t st) {
    const int A = a.p.num_agents, O = a.p.num_obstacles;
    if (A == 3 && O == 3) return launch_observe<3, 3, 1, 128, OT>(a, st);
    if (A == 3 && O == 1) return launch_observe<3, 1, 1, 128, OT>(a, st);
    if (A == 8 && O == 16) return launch_observe<8, 16, 8, 256, OT>(a, st);
    return launch_observe<0, 0, 1, 128, OT>(a, st);
}

template int launch_generic<float>(const mn::StepArgs&, cudaStream_t, int*);
template int launch_generic<__half>(const mn::StepArgs&, cudaStream_t, int*);
template int launch_generic<__nv_bfloat16>(const mn::StepArgs&, cudaStream_t, int*);
template int dispatch_observe<float>(const mn::ObserveArgs&, cudaStream_t);
template int dispatch_observe<__half>(const mn::ObserveArgs&, cudaStream_t);
template int dispatch_observe<__nv_bfloat16>(const mn::ObserveArgs&, cudaStream_t);

}  // namespace mnl
