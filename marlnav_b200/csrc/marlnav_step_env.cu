// marlnav_b200/csrc/marlnav_step_env.cu
//
// The thread-per-env step kernel (step_env_kernel) and its launch entry: the reference's team of
// 3 with 1..6 obstacles.  Device code shared with the other step kernels is in marlnav_step.cuh.
#include "marlnav_actor.cuh"
#include "marlnav_step_launch.cuh"

namespace mn {

// ---- thread-per-env kernel for small static teams (A < 4: the headline (3,3) path and (3,1)).
// One warp = one CTA = 32 consecutive envs, end to end: its own shared-memory tile, its own
// mbarrier, its own TMA bulk copies, no barrier wider than __syncwarp.
//
//   lane 0     mbarrier.init; expect_tx; cp.async.bulk global->shared x3 (states, obstacles,
//              target: one contiguous range each, 16-byte multiples)
//   all lanes  LDG own actions / step_num / terminates (issued first; overlaps the bulk copies);
//              wait on the mbarrier; P1..P4 with warp-level sync only
//   lane 0     fence.proxy.async; cp.async.bulk shared->global x2 (states, observations);
//              commit_group; wait_group.read
// Ragged warps (fewer than 32 envs left, or unaligned base pointers) stage with plain coalesced
// loads/stores into the same layout.
//
// What the B200 measurements (1M x 3 x 3) decided -- all variants bit-identical, see DESIGN.md 5:
//   * one-warp CTAs: a CTA's registers and shared memory are only released when its slowest warp
//     is done, and the tail of the last wave shrinks: 4-warp 82.0 us, 2-warp 80.2, 1-warp 78.8;
//   * P2 is split in two blocks, each smaller than the one rolled agent-loop body it replaces
//     (368 instructions at (3,3)): P2a, straight-line, evaluates each unordered agent pair ONCE for
//     both agents (geometry, bond quotient, compares; only the angle is taken per direction); P2b,
//     rolled over the team, takes the target and the obstacles.  P2a hands each agent's bond term to
//     P2b through the lane's dead obstacle / target tile slots and its flags and pair count through
//     one register of bit fields: no local memory, no larger tile.  (Unrolling the whole team
//     instead removes 15 % of the instructions but the hot path then exceeds the 32 KB L1.5
//     instruction cache, stall_no_inst 10 % -> 18 %: 83.2 us, no gain.);
//   * persistent warps with double-buffered TMA prefetch (91-121 us) and observation rows stored
//     straight from registers with 256-bit STG (86 us) both lost to this layout;
//   * one range test per env (min |component|, max d^2 over all its pairs, NaN-propagating)
//     selects between the guard-free arithmetic and a guarded re-evaluation of that env;
//   * constant divisions specialised at compile time (DivModes), guard-free bond quotients.
template <int TA, int TO, class OT = float>
struct EnvTile {
    static constexpr int A = TA, O = TO, R = TA - 1, S = 2 + 2 * TO + 2 * (TA - 1);
    // Obstacles and target go through the shared-memory tile.  Loading them straight from global
    // memory into the registers of their env's lane instead (the reset re-observation fetching them
    // by shuffle) shrinks the tile at (3,3) from 7 560 to 6 536 bytes:
    // 30 resident one-warp CTAs per SM instead of 27, and a slice of 131 072 envs (configs[3] split
    // over 8 GPUs: 4 096 CTAs) fits in ONE wave.  Bit-identical (full GPU suite); measured on B200:
    // 66.0 vs 66.5 us at 1M envs, 10.6 vs 11.9 us at 65 536, but 13.55 vs 12.96 us at 131 072 -- one
    // wave of phase-aligned warps loads, computes and stores in lock step, the 1.03 waves of the
    // tiled build overlap -- and the 8-GPU split of configs[3] runs at exactly that size, so the
    // tile stays.  (With __launch_bounds__(32, 30) the same 59 registers schedule worse: 68.3 us.)
    static constexpr int ENVS = 32;                 // envs per CTA: one per lane
    static constexpr int ST = 32 * 5 * TA, OB = 32 * 2 * TO, TG = 32 * 2;   // floats
    static constexpr int OBS = 32 * TA * S;         // observation elements (OT)
    // the mbarrier sits behind the observations (OBS * sizeof(OT) is a multiple of 16 for every shape)
    static constexpr int BYTES = (ST + OB + TG) * 4 + OBS * (int)sizeof(OT);
    static_assert(ST % 4 == 0 && OB % 4 == 0 && TG % 4 == 0 && (OBS * sizeof(OT)) % 16 == 0, "bulk copies need 16-byte multiples");
    static constexpr bool kRowVec = S % 4 == 0;     // float4 row stores into the tile (odd obstacle counts)
    static constexpr size_t smem_bytes() { return (size_t)BYTES + 8; }
    // resident CTAs per SM the compiler schedules for.  Shared memory, not registers, bounds the
    // occupancy (26 CTAs/SM at (3,3), 55-64 registers either way); a looser bound lets ptxas schedule
    // better: measured at 1M x 3 x 3 on B200, 28: 66.5 us, 24: 66.45, 20: 66.3, 16 / 12 / 8: 65.85
    // with one rolled agent loop; with the split P2, 26: 65.7, 16: 64.26, 8: 63.81 (medians of 6;
    // 4 and 1 give the same code as 8).
    static constexpr int CTAS = 8;
};

// Where P2a leaves each agent's bond term for P2b: this lane's obstacle / target slots of the tile,
// dead once P2 holds them in registers (P4a rewrites them from registers for the envs it resets
// before P4b reads them, P5 never stores them, the guarded fallback takes them from registers).
// 2 * O + 2 >= A slots for every O >= 1.
template <int A, int O>
__device__ __forceinline__ float* bond_slot(float* ob_env, float* tg_env, int a) {
    static_assert(2 * O + 2 >= A, "slots");
    if constexpr (2 * O >= A) return ob_env + a;
    else return a < 2 * O ? ob_env + a : tg_env + (a - 2 * O);
}

// P2a: every agent pair of the env once, on the branch-free fast path (see pair_obs), straight-line.
// For i < j the geometry of (i -> j) serves (j -> i) as well: on the fast path every component is
// non-zero, so cdist(j, i) == cdist(i, j) and normalize(i - j) is exactly -normalize(j - i); only
// the angle, taken against each agent's own heading, is evaluated per direction.  The bond quotient
// and the compares depend on the distance alone.  Writes the others' columns of every agent's row
// and leaves, per agent a, its bond term in bond_slot(a) and in `flags` bits 4a..4a+3: ag_risk,
// ag_coll and the count of agents between agents_min_d and agents_max_d (0..R).
template <int A, int O, class DM, bool NORM, class OT>
__device__ __forceinline__ void observe_agent_pairs(const marlnav_env_params& p, const DivConsts& rc,
                                                    const float* __restrict__ st_env, OT* obs_env,
                                                    ObsRow<NORM, OT> sink, float* ob_env, float* tg_env,
                                                    float& lo, float& dmin, unsigned& flags) {
    constexpr int R = A - 1, S = EnvTile<A, O>::S;
    static_assert(4 * A <= 32 && R <= 3, "flag bits");
    const float cap = p.cap_distance;
    float an[A][R > 0 ? R : 1], di[A][R > 0 ? R : 1], q[A][R > 0 ? R : 1];   // [agent][k-th other]
    unsigned fl = 0u;
#pragma unroll
    for (int i = 0; i < A; ++i) {
#pragma unroll
        for (int j = i + 1; j < A; ++j) {
            const int ki = j - 1, kj = i;                   // j among i's others, i among j's (:22-24)
            float d, nx, ny;
            geom_fast(st_env[5 * j + 0] - st_env[5 * i + 0], st_env[5 * j + 1] - st_env[5 * i + 1], d, nx, ny, lo);
            pair_finish<false>(d, nx, ny, st_env[5 * i + 2], st_env[5 * i + 3], cap, an[i][ki], di[i][ki]);
            pair_finish<false>(d, -nx, -ny, st_env[5 * j + 2], st_env[5 * j + 3], cap, an[j][kj], di[j][kj]);
            dmin = fminf(dmin, d);
            const unsigned both = (1u << (4 * i)) | (1u << (4 * j));
            if (d < p.ag_risk_dist) fl |= both;
            if (d < p.ag_coll_dist) fl |= both << 1;
            if (p.agents_min_d < d && d < p.agents_max_d) fl += both << 2;
            const float sd = div_mode<DM::kSharp, false>(d - p.ideal_dist, p.bond_sharpness, rc.sharp);
            q[i][ki] = q[j][kj] = rcp_rn_normal(1.0f + sd * sd);
        }
    }
#pragma unroll
    for (int a = 0; a < A; ++a) {
        float cols[2 * R];
#pragma unroll
        for (int k = 0; k < R; ++k) { cols[k] = an[a][k]; cols[R + k] = di[a][k]; }
        sink.row = obs_env + a * S;
        sink.template put_cols<2 + 2 * O, 2 * R, EnvTile<A, O>::kRowVec>(cols);
        *bond_slot<A, O>(ob_env, tg_env, a) = div_mode<DM::kR, false>(torch_row_sum(q[a], R), (float)R, rc.R);
    }
    flags = fl;
}

// P2b: agent `a` against the target and the O obstacles on the fast path, the rest of its row, and
// its reward ingredients with the agent-pair terms P2a left for it (environment.py:186-202).
template <int A, int O, class DM, bool NORM, class OT>
__device__ __forceinline__ void observe_agent_objects(const marlnav_env_params& p, const DivConsts& rc,
                                                      const float* __restrict__ st_env, const float (&OBX)[O],
                                                      const float (&OBY)[O], float tx, float ty, int a,
                                                      const ObsRow<NORM, OT>& sink, float bond, unsigned flags,
                                                      float& lo, float& dmin, AgentTerms& tm) {
    constexpr int N = 1 + O;
    const float ox = st_env[5 * a + 0], oy = st_env[5 * a + 1];
    const float hx = st_env[5 * a + 2], hy = st_env[5 * a + 3];
    const float cap = p.cap_distance;
    float px[N], py[N], an[N], di[N];
    px[0] = tx; py[0] = ty;
#pragma unroll
    for (int j = 0; j < O; ++j) { px[1 + j] = OBX[j]; py[1 + j] = OBY[j]; }
#pragma unroll
    for (int i = 0; i < N; ++i) {
        float d, nx, ny;
        geom_fast(px[i] - ox, py[i] - oy, d, nx, ny, lo);
        pair_finish<false>(d, nx, ny, hx, hy, cap, an[i], di[i]);
    }
#pragma unroll
    for (int i = 0; i + 1 < N; i += 2) dmin = min3f(dmin, di[i], di[i + 1]);
    if constexpr (N % 2 == 1) dmin = fminf(dmin, di[N - 1]);
    float row[2 + 2 * O];
    row[0] = an[0]; row[1] = di[0];
    bool ob_risk = false, ob_coll = false;
#pragma unroll
    for (int j = 0; j < O; ++j) {
        row[2 + j] = an[1 + j]; row[2 + O + j] = di[1 + j];
        ob_risk |= di[1 + j] < p.ob_risk_dist; ob_coll |= di[1 + j] < p.ob_coll_dist;
    }
    sink.template put_cols<0, 2 + 2 * O, EnvTile<A, O>::kRowVec>(row);
    const unsigned f = flags >> (4 * a);
    tm.risk = (ob_risk || (f & 1u) != 0u) ? 1.f : 0.f;
    tm.coll = ob_coll || (f & 2u) != 0u;
    tm.in_t = di[0] < p.target_radius;
    const float cnt = (float)((f >> 2) & 3u);            // the reference's sum of 0/1 terms, exact
    const float capped = cnt > p.max_at_prop_d ? p.max_at_prop_d : cnt;
    tm.dsc = div_mode<DM::kProp, false>(capped, p.max_at_prop_d, rc.prop_d);
    tm.head = fabsf(an[0]) < p.max_angle_diff ? 1.f : 0.f;
    // 2^-39 < di[0] < 2^50 (the caller's range test), inside the proven sequence's range
    tm.soft = -1.0f * div_mode<DM::kInit, true>(di[0], p.init_dist, rc.init_dist);
    tm.bond = bond;
}

// ACTOR: the actions are not read but sampled here, from the reference's Actor applied to the
// (normalised) observations of the current state -- SURVEY 8(f)-2's end state, "feeding actions
// straight to the step": one launch per rollout step instead of two.  mna::actor_row is the code
// of the stand-alone actor kernel, so both routes give the same bits.
//
// OT: the observations' element type (float, or float32 values rounded into __half / __nv_bfloat16;
// 16-bit observations are never read back from the tile).  The fused actor reads the previous
// step's observations, args.obs_in, from global memory as OT and widens them exactly to float32.
template <int TA, int TO, bool NORM, class DM, bool ACTOR = false, class OT = float>
__global__ void __launch_bounds__(32, EnvTile<TA, TO, OT>::CTAS)
step_env_kernel(const StepArgs args) {
    using W = EnvTile<TA, TO, OT>;
    using G = Geo<TA, TO, 1, 128>;
    constexpr int A = TA, O = TO, R = TA - 1, S = W::S, N = 1 + O + R;
    static_assert(TA < 4, "sequential torch.mean order only holds below 4 agents");
    const marlnav_env_params& p = args.p;
    const marlnav_reset_spec& rs = args.rs;
    const DivConsts rc{args.rc_init_dist, args.rc_prop_d, args.rc_sharp, args.rc_R, args.rc_A};

    extern __shared__ float4 smem_raw[];
    const int lane = threadIdx.x;
    float* const w_st = reinterpret_cast<float*>(smem_raw);
    float* const w_ob = w_st + W::ST;
    float* const w_tg = w_ob + W::OB;
    OT* const w_obs = reinterpret_cast<OT*>(w_tg + W::TG);
    uint64_t* const bar = reinterpret_cast<uint64_t*>(reinterpret_cast<char*>(smem_raw) + W::BYTES);

    // Odd steps visit the tiles in reverse (CTA i takes tile gridDim.x - 1 - i): each step starts on
    // the tiles the previous one finished last, whose state is the likeliest to be still in L2
    // (the parity is the host's step counter: no load before the bulk copies are issued).  The
    // fused-actor build keeps the launch order: it steps rollouts of small, L2-resident batches, and
    // there the reversal measured 0.8 % slower per rollout iteration at 1 024 envs.
    const unsigned tile = (!ACTOR && (rs.step_counter & 1u)) ? gridDim.x - 1u - blockIdx.x : blockIdx.x;
    const long long wenv0 = (long long)tile << 5;
    const long long left = (long long)p.num_envs - wenv0;
    const int nenv = left < 32 ? (int)left : 32;
    const bool bulk = args.vec_ok != 0 && nenv == 32;
    const bool active = lane < nenv;
    const long long env = wenv0 + lane;

    float* const g_st = args.states + wenv0 * (5 * A);
    float* const g_ob = args.obstacles + wenv0 * (2 * O);
    float* const g_tg = args.target + wenv0 * 2;
    OT* const g_obs = reinterpret_cast<OT*>(args.obs) + (size_t)wenv0 * A * S;

    // ---- P0: the tile by TMA bulk copies, per-env scalars and actions straight to registers.
    // Everything is requested before anything is consumed: the loaded step counter / terminates
    // flag stay raw until P3 (a consumer placed here would expose one DRAM latency before the
    // bulk copies are even issued -- measured: 7 % of all stall samples).
    pdl_launch_dependents();
    pdl_wait();
    if constexpr (ACTOR) {
        // after the dependency wait: FusedActor.refresh() rewrites the weights on the stream
        mna::stage_actor_weights(reinterpret_cast<float*>(bar + 2), S, args.actor.H, args.actor.w1, args.actor.b1,
                                 args.actor.w_mu, args.actor.w_std, lane, 32);
    }
    if (bulk) {
        if (lane == 0) {
            mbar_init(bar, 1);
            mbar_expect_tx(bar, (W::ST + W::OB + W::TG) * 4);
            bulk_g2s(w_st, g_st, W::ST * 4, bar);
            bulk_g2s(w_ob, g_ob, W::OB * 4, bar);
            bulk_g2s(w_tg, g_tg, W::TG * 4, bar);
        }
        __syncwarp();
    }
    float2 acts[A];
    float sn_in = 0.f;
    unsigned char term_raw = 0;
    float OBX[O], OBY[O];                   // this env's obstacles and target (from the tile in P2)
    float2 tg = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < O; ++j) { OBX[j] = 0.f; OBY[j] = 0.f; }
    if (active) {
        if constexpr (!ACTOR) {
#pragma unroll
            for (int i = 0; i < A; ++i) acts[i] = load_action(args.actions, env * A + i, args.act8 != 0);
        }
        sn_in = args.step_num[env];
        term_raw = args.terminates[env];
    }
    if constexpr (ACTOR) {
        // the policy, while the bulk copies are in flight (models.py:27-36, 113-115)
        float* const s_actor = reinterpret_cast<float*>(bar + 2);
        const int H = args.actor.H;
        __syncwarp();
        if (active) {
            const mna::ActorWeights aw(s_actor, S, H);
            const OT* const obs_in = static_cast<const OT*>(args.obs_in);
            const uint64_t counter = args.actor.counter +
                (args.actor.counter_dev ? __ldg(reinterpret_cast<const unsigned long long*>(args.actor.counter_dev)) : 0ull);
#pragma unroll 1
            for (int a = 0; a < A; ++a) {
                const long long row = env * A + a;
                float x[S];
#pragma unroll
                for (int k = 0; k < S; ++k) x[k] = mna::widen(obs_in[row * S + k]);
                const mna::ActorOut o = mna::actor_row<S>(x, S, H, aw, args.actor.b_mu, args.actor.b_std, nullptr,
                                                          args.actor.seed, counter, row, args.actor.row_offset + (uint64_t)row);
                args.act_out[row * 2] = o.a0; args.act_out[row * 2 + 1] = o.a1;
                args.logp_out[row] = o.logp;
                // (rolled loop: the action goes through a register array indexed by a constant below)
                if (a == 0) acts[0] = make_float2(o.a0, o.a1);
                if (A > 1 && a == 1) acts[A > 1 ? 1 : 0] = make_float2(o.a0, o.a1);
                if (A > 2 && a == 2) acts[A > 2 ? 2 : 0] = make_float2(o.a0, o.a1);
            }
        }
    }
    if (bulk) {
        mbar_wait(bar, 0);
    } else {
#pragma unroll 1
        for (int i = lane; i < nenv * 5 * A; i += 32) w_st[i] = g_st[i];
#pragma unroll 1
        for (int i = lane; i < nenv * 2 * O; i += 32) w_ob[i] = g_ob[i];
#pragma unroll 1
        for (int i = lane; i < nenv * 2; i += 32) w_tg[i] = g_tg[i];
        __syncwarp();
    }

    bool all_in = true, coll_any = false, done = false, trunc = false;
    float* const st_env = w_st + lane * (5 * A);
    float* const ob_env = w_ob + lane * (2 * O);
    // The blend of an env that does NOT reset, 1*old + 0*new (environment.py:86-90), is old + (+0)
    // when every template element is +0 or positive: its only effect is -0 -> +0.  That wash is
    // folded into the move's store (x + (-0) == x for every x when it does not apply).  The sign
    // of a zero coordinate or heading component cannot reach any observation, reward or flag
    // (squares, |.|, comparisons against non-zero thresholds, acos(+-0) and `orth > 0` agree), and
    // a reset computes 0*old + new, which is new for either zero; so washing before observing is
    // bit-identical to the reference's order.
    const bool wash_early = DM::kWash != 0 || ((rs.flags & MARLNAV_RESET_TMPL_NONNEG) != 0 && rs.alias_first_step == 0);
    const float wash = wash_early ? 0.0f : -0.0f;
    if (active) {
        // ---- P1: move (ActionScaler, utils.py:546-547, folded into the action load)
        const bool scale_act = args.io.act_scale != nullptr;
        float am0 = 0.f, am1 = 0.f, as0 = 1.f, as1 = 1.f;
        if (scale_act) {
            am0 = __ldg(args.io.act_mean + 0); am1 = __ldg(args.io.act_mean + 1);
            as0 = __ldg(args.io.act_scale + 0); as1 = __ldg(args.io.act_scale + 1);
        }
        float cmax = 0.f;                                   // max |coordinate| of the env (agents, obstacles, target)
#pragma unroll
        for (int a = 0; a < A; ++a) {
            float2 act = acts[a];
            if (scale_act) { act.x = (as0 * act.x) + am0; act.y = (as1 * act.y) + am1; }
            float s[5];
#pragma unroll
            for (int k = 0; k < 5; ++k) s[k] = st_env[5 * a + k];
            move_agent(p, s, act.x, act.y);
            cmax = max3_nan_abs(cmax, s[0], s[1]);
#pragma unroll
            for (int k = 0; k < 5; ++k) st_env[5 * a + k] = s[k] + wash;
        }

        // ---- P2: observe + per-agent reward terms
#pragma unroll
        for (int j = 0; j < O; ++j) {
            const float2 ob = *reinterpret_cast<const float2*>(ob_env + 2 * j);
            OBX[j] = ob.x; OBY[j] = ob.y;
        }
        tg = *reinterpret_cast<const float2*>(w_tg + lane * 2);
#pragma unroll
        for (int j = 0; j < O; ++j) cmax = max3_nan_abs(cmax, OBX[j], OBY[j]);
        cmax = max3_nan_abs(cmax, tg.x, tg.y);
        float lo = 3.0e38f, dmin = 3.0e38f;                 // min |component|, min distance over the env's pairs
        float sum_out = 0.f, sum_in = 0.f;
        ObsRow<NORM, OT> sink;
        sink.mean = args.io.obs_mean; sink.scale = args.io.obs_scale;
        OT* const obs_env = w_obs + lane * A * S;
        float* const tg_env = w_tg + lane * 2;
        unsigned pair_flags;
        // ---- P2a: agent pairs, each once (straight-line)
        observe_agent_pairs<A, O, DM>(p, rc, st_env, obs_env, sink, ob_env, tg_env, lo, dmin, pair_flags);
        // ---- P2b: target and obstacles, rolled over the team (code size, see above); the reward
        // terms summed from agent 0 up as torch does
#pragma unroll 1
        for (int a = 0; a < A; ++a) {
            sink.row = obs_env + a * S;
            AgentTerms tm;
            observe_agent_objects<A, O, DM>(p, rc, st_env, OBX, OBY, tg.x, tg.y, a, sink,
                                            *bond_slot<A, O>(ob_env, tg_env, a), pair_flags, lo, dmin, tm);
            all_in = all_in && tm.in_t;
            coll_any = coll_any || tm.coll;
            float r_out, r_in;
            agent_reward2(p, tm, r_out, r_in);
            sum_out = sum_out + r_out; sum_in = sum_in + r_in;
        }
        // ---- P2c: guarded fallback
        // Fast-path validity (see pair_obs, geom_fast): every |ex|, |ey| > 2^-39, every coordinate
        // below 2^48 (=> every d^2 < 2^100) and every distance >= cap (the fast path leaves the cap
        // rule out).  Anything else (exactly aligned agents, absurd magnitudes, coincident points)
        // re-evaluates the whole env with the guarded IEEE sequences.
        if (__builtin_expect(!fast_path_ok(lo, cmax, dmin, p.cap_distance), 0)) {
            const G g(TA, TO);
            all_in = true; coll_any = false; sum_out = 0.f; sum_in = 0.f;
            float ob_loc[2 * O];                            // the guarded routine takes the obstacles by pointer
#pragma unroll
            for (int j = 0; j < O; ++j) { ob_loc[2 * j] = OBX[j]; ob_loc[2 * j + 1] = OBY[j]; }
#pragma unroll 1
            for (int a = 0; a < A; ++a) {
                sink.row = obs_env + a * S;
                AgentTerms tm;
                observe_agent<G, NORM, false>(g, p, rc, st_env, ob_loc, tg.x, tg.y, a, sink, tm);
                all_in = all_in && tm.in_t;
                coll_any = coll_any || tm.coll;
                float r_out, r_in;
                agent_reward2(p, tm, r_out, r_in);
                sum_out = sum_out + r_out; sum_in = sum_in + r_in;
            }
        }

        // ---- P3 (environment.py:96-103, 209-221)
        // torch.mean over A < 4 agents: sequential sum from 0, then three idle accumulators
        const float reward = div_mode<DM::kA, false>((all_in ? sum_in : sum_out) + 0.0f, (float)A, rc.A);
        const float sn = sn_in + 1.0f;
        trunc = sn > (float)(p.episode_len - 1);
        const bool term_old = term_raw != 0;
        const bool term = coll_any || term_old;
        done = term || trunc;
        args.terminates[env] = (uint8_t)((!term_old) && all_in);
        args.rewards[env] = reward;
        args.terminated[env] = (uint8_t)term;
        args.truncated[env] = (uint8_t)trunc;
        args.step_num[env] = done ? ((0.0f * sn) + 0.0f) : (sn + 0.0f);   // (1-m)*sn + m*0
    }
    const unsigned b_tr = __ballot_sync(0xffffffffu, active && trunc);
    const unsigned b_co = __ballot_sync(0xffffffffu, active && coll_any);
    const unsigned b_ta = __ballot_sync(0xffffffffu, active && all_in);
    const unsigned dmask = __ballot_sync(0xffffffffu, done);
    if (lane == 0) {
        if (b_tr) atomicAdd(args.stats + 0, (unsigned long long)__popc(b_tr));
        if (b_co) atomicAdd(args.stats + 1, (unsigned long long)__popc(b_co));
        if (b_ta) atomicAdd(args.stats + 2, (unsigned long long)__popc(b_ta));
    }
    if constexpr (DM::kFinal) {
        // the finished envs' rows, which the rewards and flags were computed from, before P4b
        // re-observes them (finished envs one after the other, the warp copying each row block)
        __syncwarp();
        OT* const g_fin = static_cast<OT*>(args.final_obs) + (size_t)wenv0 * A * S;
        for (unsigned m = dmask; m != 0u; m &= m - 1u) {
            const int e2 = __ffs((int)m) - 1;
            copy_final_rows(g_fin + (size_t)e2 * A * S, w_obs + e2 * A * S, A, S, S, lane);
        }
    }
    // ---- P4a: masked re-initialisation (environment.py:76-90): x = (1-m)*x + m*new
    // (A cooperative form -- the warp taking its reset envs one after the other, one state element /
    // Philox obstacle pair per lane instead of ~320 instructions on the reset env's own lane -- was
    // built, is bit-identical and measured SLOWER, 66.0 vs 64.9 us: 72 registers, and the divergent
    // lane groups cost more than the idle lanes they replace.)
    if (active) {
        const bool alias = DM::kWash == 0 && rs.alias_first_step != 0;
        const float* ts = rs.tmpl_states + env * rs.states_env_stride;
        if (done || !wash_early) {          // (an env that keeps going was already blended by the move's store)
            const bool noisy = DM::kWash == 0 && (rs.flags & MARLNAV_RESET_NOISY_AGENTS) != 0;
#pragma unroll 1
            for (int a = 0; a < A; ++a) {
                float nv[5];
                if (noisy) sample_agent_noisy(rs, reset_counter(rs), rs.env_id_offset + (uint64_t)env, a, ts + 5 * a, nv);
#pragma unroll
                for (int k = 0; k < 5; ++k) {
                    const float old_v = st_env[5 * a + k];
                    const float new_v = noisy ? nv[k] : (alias ? old_v : __ldg(ts + 5 * a + k));
                    st_env[5 * a + k] = done ? ((0.0f * old_v) + new_v) : (old_v + (0.0f * new_v));
                }
            }
        }
        if (done) {
            // obstacles / target of a reset env: x = 0*old + new (environment.py:86-90 with m = 1)
            if (rs.tmpl_obstacles || alias) {
                const float* to = alias ? nullptr : rs.tmpl_obstacles + env * rs.obstacles_env_stride;
#pragma unroll
                for (int j = 0; j < O; ++j) {
                    OBX[j] = (0.0f * OBX[j]) + (alias ? OBX[j] : __ldg(to + 2 * j));
                    OBY[j] = (0.0f * OBY[j]) + (alias ? OBY[j] : __ldg(to + 2 * j + 1));
                }
            } else {
#pragma unroll
                for (int pr = 0; 2 * pr < O; ++pr) {
                    float nw[4];
                    sample_obstacle_pair(p, rs.seed, reset_counter(rs), rs.env_id_offset + (uint64_t)env, pr, nw);
                    OBX[2 * pr] = (0.0f * OBX[2 * pr]) + nw[0]; OBY[2 * pr] = (0.0f * OBY[2 * pr]) + nw[1];
                    if (2 * pr + 1 < O) {
                        OBX[2 * pr + 1 < O ? 2 * pr + 1 : 0] = (0.0f * OBX[2 * pr + 1 < O ? 2 * pr + 1 : 0]) + nw[2];
                        OBY[2 * pr + 1 < O ? 2 * pr + 1 : 0] = (0.0f * OBY[2 * pr + 1 < O ? 2 * pr + 1 : 0]) + nw[3];
                    }
                }
            }
            const float* tt = rs.tmpl_target + env * rs.target_env_stride;
            tg.x = (0.0f * tg.x) + (alias ? tg.x : __ldg(tt + 0));
            tg.y = (0.0f * tg.y) + (alias ? tg.y : __ldg(tt + 1));
            // only reset envs rewrite obstacles / target in HBM
#pragma unroll
            for (int j = 0; j < O; ++j) { g_ob[lane * (2 * O) + 2 * j] = OBX[j]; g_ob[lane * (2 * O) + 2 * j + 1] = OBY[j]; }
            g_tg[lane * 2 + 0] = tg.x; g_tg[lane * 2 + 1] = tg.y;
            // the re-observation below reads them from the tile
#pragma unroll
            for (int j = 0; j < O; ++j) { ob_env[2 * j] = OBX[j]; ob_env[2 * j + 1] = OBY[j]; }
            w_tg[lane * 2 + 0] = tg.x; w_tg[lane * 2 + 1] = tg.y;
        }
    }
    __syncwarp();

    // ---- P4b: re-observe this warp's reset envs (environment.py:105), ONE (env, agent, object)
    // pair per lane.  Rewards were taken from the pre-reset observations, so only angles and
    // distances are needed here; spreading the 18 pairs of a reset env over 18 lanes instead of
    // its three agents over three lanes cuts the warp's tail six-fold.
    {
        const int n_pairs = __popc(dmask) * (A * N);
        const float cap = p.cap_distance;
#pragma unroll 1
        for (int base = 0; base < n_pairs; base += 32) {
            const int w2 = base + lane;
            const bool on = w2 < n_pairs;
            const int e2 = on ? (int)__fns(dmask, 0, w2 / (A * N) + 1) : 0;
            const int rem = w2 % (A * N), a = on ? rem / N : 0, obj = on ? rem - (rem / N) * N : 0;
            const float* st2 = w_st + e2 * (5 * A);
            float px, py;
            int col_a, col_d;
            if (obj == 0) {
                px = w_tg[e2 * 2]; py = w_tg[e2 * 2 + 1];
                col_a = 0; col_d = 1;
            } else if (obj <= O) {
                px = w_ob[e2 * (2 * O) + 2 * (obj - 1)]; py = w_ob[e2 * (2 * O) + 2 * (obj - 1) + 1];
                col_a = 1 + obj; col_d = 1 + O + obj;
            } else {
                const int k = obj - 1 - O, jj = k + (k >= a ? 1 : 0);
                px = st2[5 * jj]; py = st2[5 * jj + 1];
                col_a = 2 + 2 * O + k; col_d = 2 + 2 * O + (A - 1) + k;
            }
            if (on) {
                float ang, dist;
                // (guarded arithmetic for every pair: a freshly reset team has exactly aligned agents, so with
                // pair_obs both of its branches would run in every iteration)
                pair_guarded(st2[5 * a], st2[5 * a + 1], st2[5 * a + 2], st2[5 * a + 3], px, py, cap, ang, dist);
                ObsRow<NORM, OT> sink;
                sink.row = w_obs + (e2 * A + a) * S; sink.mean = args.io.obs_mean; sink.scale = args.io.obs_scale;
                sink.put(col_a, ang); sink.put(col_d, dist);
            }
        }
    }

    // ---- P5: stage out
    // (the warp storing the tile itself with coalesced float4 stores -- no wait before exit --
    // measured 73.4 vs 70.8 us: the bulk stores stay)
    if (bulk) {
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
            bulk_s2g(g_st, w_st, W::ST * 4);
            bulk_s2g(g_obs, w_obs, W::OBS * sizeof(OT));
            bulk_commit_wait_read();
        }
    } else {
        __syncwarp();
#pragma unroll 1
        for (int i = lane; i < nenv * 5 * A; i += 32) g_st[i] = w_st[i];
#pragma unroll 1
        for (int i = lane; i < nenv * A * S; i += 32) g_obs[i] = w_obs[i];
    }
}

}  // namespace mn

namespace mnl {

template <class OT>
int launch_env3(const mn::StepArgs& a, cudaStream_t st, int* info) {
    switch (a.p.num_obstacles) {
        case 1: return launch_step_tile<mn::EnvTile, 3, 1, mn::DivModesDefault, OT>(a, st, info);
        case 2: return launch_step_tile<mn::EnvTile, 3, 2, mn::DivModesDefault, OT>(a, st, info);
        case 3: return launch_step_tile<mn::EnvTile, 3, 3, mn::DivModesDefault, OT>(a, st, info);
        case 4: return launch_step_tile<mn::EnvTile, 3, 4, mn::DivModesDefault, OT>(a, st, info);
        case 5: return launch_step_tile<mn::EnvTile, 3, 5, mn::DivModesDefault, OT>(a, st, info);
        case 6: return launch_step_tile<mn::EnvTile, 3, 6, mn::DivModesDefault, OT>(a, st, info);
        default: return -1;
    }
}
template int launch_env3<float>(const mn::StepArgs&, cudaStream_t, int*);
template int launch_env3<__half>(const mn::StepArgs&, cudaStream_t, int*);
template int launch_env3<__nv_bfloat16>(const mn::StepArgs&, cudaStream_t, int*);

}  // namespace mnl
