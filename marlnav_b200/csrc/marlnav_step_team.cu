// marlnav_b200/csrc/marlnav_step_team.cu
//
// The thread-per-agent step kernel (step_team_kernel) and its launch entries: the (8,16) team,
// and the reference's team of 3 with 1..6 obstacles on small batches.  Device code shared with
// the other step kernels is in marlnav_step.cuh.
#include "marlnav_actor.cuh"
#include "marlnav_step_launch.cuh"

namespace mn {

// ---- thread-per-agent kernel: big static teams ((8,16)), and the reference's team of 3 when the
// batch is small (one wave of warps: a third of the dependent chain of the thread-per-env kernel).
// One warp = one CTA = 32 / LPE consecutive envs, LPE = A rounded up to a power of two lanes per
// env (lanes beyond the team idle); lane = (env, agent).  Same staging as step_env_kernel; env-wide
// flags by __ballot_sync on aligned sub-warps, the A per-agent rewards gathered with __shfl_sync
// and summed in torch's order.  The pair loops stay rolled (instruction cache: fully unrolled,
// 23 % of the stall samples were stall_no_inst) but evaluate every pair on the guard-free fast
// path and test the whole agent once (observe_agent_team).
constexpr int ceil_pow2(int x) { int p = 1; while (p < x) p *= 2; return p; }
template <int TA, int TO, class OT = float>
struct TeamTile {
    static constexpr int A = TA, O = TO, R = TA - 1, S = 2 + 2 * TO + 2 * (TA - 1);
    static constexpr int LPE = ceil_pow2(TA);     // lanes per env
    static constexpr int ENVS = 32 / LPE;         // envs per warp
    static_assert(TA >= 2 && TA <= 32, "team size");
    // consecutive lanes write consecutive rows; a row stride that is an odd multiple of 16 bytes
    // spreads the banks (and then the tile is copied out by the warp instead of by TMA).  In elements
    // of OT: 16 bytes are 4 float32 or 8 16-bit observations.
    static constexpr int E16 = 16 / (int)sizeof(OT);
    static constexpr int OBS_STRIDE = (S % E16 == 0 && ((S / E16) % 2) == 0) ? S + E16 : S;
    static constexpr bool kObsBulk = OBS_STRIDE == S;
    // An obstacle row that is a multiple of 32 words (O = 16) puts "obstacle j" of every env of the
    // warp into the same banks (the lanes of one env broadcast-read it).  So the envs start their
    // obstacle loop at different obstacles (ob_rot) and the rows stay packed.  Staging such rows 4
    // words further apart instead (one bulk copy per env), which lets the loop be unrolled with
    // immediate offsets, measured on B200 at 262144 x 8 x 16: rolled 155.6 us (the three extra bulk
    // copies cost what the rotation saved), unrolled x2 154.9, x4 166-172, x8 185.7 us against 155.1
    // for the rotation: the unrolled body no longer fits the 6 KB L0 instruction cache
    // (stall_no_instruction 0.23 -> 1.74 warps per issue), so the rotation stays.
    static constexpr int ST = ENVS * 5 * TA, OB = ENVS * 2 * TO, TG = ENVS * 2;   // floats
    static constexpr int OBS = ENVS * TA * OBS_STRIDE;                            // observation elements (OT)
    static_assert((ST % 4) == 0 && (OB % 4) == 0 && (TG % 4) == 0 && (OBS * sizeof(OT)) % 16 == 0, "bulk copies need 16-byte multiples");
    static constexpr int BYTES = (ST + OB + TG) * 4 + OBS * (int)sizeof(OT);     // the mbarrier sits behind
    static constexpr int FLOATS = BYTES / 4;
    static constexpr size_t smem_bytes() { return (size_t)BYTES + 8; }
    // register budget the compiler schedules for (shared memory, not registers, bounds the occupancy:
    // 56-59 registers in use at (8,16); measured 20: 140.3 us, 16: 140.7, 24: 141.7, 26: 141.9).  Taking
    // the smallest agent distance and the in-band count from the distances read back by compile-time
    // column, after the pair loops, measured the same (140.7 vs 140.2 us) and was dropped.
    static constexpr int CTAS = (FLOATS * 4 + 8 + 1024) * 28 <= 233472 + 8 * 1024 ? 28 : 20;
    // copy-out of a padded observation tile: iterations after which (row, column) of a lane's 16-byte piece repeat
    static constexpr int gcd_(int a, int b) { return b == 0 ? a : gcd_(b, a % b); }
    static constexpr int kCopyPeriod = (S % E16 == 0) ? (S / E16) / gcd_(32, S / E16) : 1;
};

// One agent of a big team against its 1 + O + R objects: every pair on the guard-free fast path
// in rolled loops (one or two pair instances per loop in the binary), angles and distances written
// straight to the agent's shared-memory row, ONE range test for the whole agent afterwards; the
// rare agent that fails it (an exactly aligned pair, absurd magnitudes, a distance below the cap)
// is redone by the guarded observe_agent.  Under the test every distance is in (2^-39, 2^50), so
// the bond quotients and the soft term take their guard-free divisions.
//   * Obstacles go two at a time: one LDS.128 for both, one 8-byte store for the two angles and
//     one for the two distances (columns 2+j, 2+O+j with j even are 8-byte aligned).  With the
//     padded row stride (an odd multiple of 16 bytes) an 8-byte store of 32 rows takes 4
//     shared-memory wavefronts where two 4-byte stores took 8.
//   * `ob_rot`: the envs of one warp start their obstacle loop at different obstacles.  With 16
//     obstacles an env's obstacle row is exactly 32 banks wide, so the 4 envs' broadcast reads of
//     "obstacle j" all hit the same banks (4-way conflict on every read, ncu round 1); rotated by
//     4 obstacles per env they hit 4 different bank groups.  Nothing here depends on the order.
//   * `env_ok`: the coordinate bound of geom_fast, established for the whole env by the caller.
//   * Agent-agent pairs share their geometry: cdist(i, j) == cdist(j, i) bit for bit and
//     normalize(pos_j - pos_i) is the exact negation of normalize(pos_i - pos_j) (every step of the
//     sqrt / division sequences is odd-symmetric; a zero component, where +0 would break that,
//     fails the range test).  In round o = 1 .. (A-1)/2 lane a evaluates its FORWARD partner
//     (a + o) mod A and takes the pair with its BACKWARD partner (a - o) mod A from that lane's
//     registers (three shuffles; it was that lane's forward pair of the same round); even teams
//     finish with the opposite agent (a + A/2).  4 geometries per agent instead of 7 at A = 8.
//     Partner positions come by shuffle too.  Because a lane now consumes geometry another lane
//     range-tested, the fast-path verdict is taken per ENV (ballot), and ALL lanes of the warp
//     call this function (idle lanes compute on whatever their slot holds and store nothing).
//     The fused-normaliser build keeps the ascending-k loop (it needs the raw distances in
//     registers by k for the bond sum).
template <typename G, class DM, bool NORM, class OT = float>
__device__ __forceinline__ void observe_agent_team(const G& g, const marlnav_env_params& p, const DivConsts& rc,
                                                   const float* __restrict__ st_env,
                                                   const float* __restrict__ ob_env, float tx, float ty,
                                                   int a, bool active, unsigned lead, unsigned gmask, int ob_rot,
                                                   bool env_ok, const ObsRow<NORM, OT>& sink, AgentTerms& tm) {
    using SINK = ObsRow<NORM, OT>;
    static_assert(G::kStatic, "compile-time team shape");
    constexpr int A = G::kMaxR + 1, O = G::kStaticO, R = G::kMaxR;
    constexpr unsigned FULL = 0xffffffffu;
    const float ox = st_env[5 * a + 0], oy = st_env[5 * a + 1];
    const float hx = st_env[5 * a + 2], hy = st_env[5 * a + 3];
    const float cap = p.cap_distance;
    float lo = 3.0e38f;
    float ta, td;
    {
        float d, nx, ny;
        geom_fast(tx - ox, ty - oy, d, nx, ny, lo);
        pair_finish<false>(d, nx, ny, hx, hy, cap, ta, td);
        if (active) sink.put2(0, ta, td);
    }
    float ob_min = 3.0e38f;                                  // any(dist < x) == (min dist) < x; a NaN distance is never "<"
    constexpr int O2 = O & ~1;
    // kLean: power-of-two obstacle count, raw (not normalised) rows, every lane owning a row.  The loop
    // then carries ONE induction variable, the byte offset of the obstacle pair inside the env's
    // obstacle row (wrapping: the envs of a warp start at different obstacles, see ob_rot): the
    // LDS.128 address is base + off, the two 8-byte stores go to row + 8 + off/2 (+ 4 O), unpredicated.
    // 8 bookkeeping instructions per iteration instead of 12 (ptxas, sm_100a).
    constexpr bool kLean = !NORM && (O & (O - 1)) == 0 && O >= 2 && G::LPE == A;
    if constexpr (kLean) {
        const char* const ob_bytes = reinterpret_cast<const char*>(ob_env);
        // (an obstacle is 8 bytes of its row, its column 4 bytes of a float32 row, 2 of a 16-bit row)
        constexpr int kColShift = sizeof(OT) == 4 ? 1 : 2;
        char* const row_bytes = reinterpret_cast<char*>(sink.row + 2);
        int off = (ob_rot * 8) & (8 * O - 16);
#pragma unroll 1
        for (int it = 0; it < O / 2; ++it) {
            const float4 ob = *reinterpret_cast<const float4*>(ob_bytes + off);
            float d0, nx0, ny0, d1, nx1, ny1, a0, a1, t0, t1;
            geom_fast(ob.x - ox, ob.y - oy, d0, nx0, ny0, lo);
            geom_fast(ob.z - ox, ob.w - oy, d1, nx1, ny1, lo);
            pair_finish<false>(d0, nx0, ny0, hx, hy, cap, a0, t0);
            pair_finish<false>(d1, nx1, ny1, hx, hy, cap, a1, t1);
            OT* const dst = reinterpret_cast<OT*>(row_bytes + (off >> kColShift));   // column 2 + j, j = off / 8
            obs_store2(dst, a0, a1);
            obs_store2(dst + O, t0, t1);
            ob_min = min3f(ob_min, t0, t1);
            off = (off + 16) & (8 * O - 16);
        }
    } else {
#pragma unroll 1
    for (int jj = 0; jj < O2; jj += 2) {
        // rotation only for power-of-two counts
        const int j = ((O & (O - 1)) == 0) ? ((jj + ob_rot) & (O - 1)) : jj;
        float4 ob;
        if constexpr ((O % 2) == 0) ob = *reinterpret_cast<const float4*>(ob_env + 2 * j);      // env rows are 16-byte multiples
        else { const float2 o0 = *reinterpret_cast<const float2*>(ob_env + 2 * j), o1 = *reinterpret_cast<const float2*>(ob_env + 2 * j + 2);
               ob = make_float4(o0.x, o0.y, o1.x, o1.y); }
        float d0, nx0, ny0, d1, nx1, ny1, a0, a1, t0, t1;
        geom_fast(ob.x - ox, ob.y - oy, d0, nx0, ny0, lo);
        geom_fast(ob.z - ox, ob.w - oy, d1, nx1, ny1, lo);
        pair_finish<false>(d0, nx0, ny0, hx, hy, cap, a0, t0);
        pair_finish<false>(d1, nx1, ny1, hx, hy, cap, a1, t1);
        if (active) {
            sink.put2(2 + j, a0, a1);
            if constexpr ((O % 2) == 0) sink.put2(2 + O + j, t0, t1);
            else { sink.put(2 + O + j, t0); sink.put(2 + O + j + 1, t1); }
        }
        ob_min = min3f(ob_min, t0, t1);
    }
    }
    if constexpr (O % 2 == 1) {
        const float2 ob = *reinterpret_cast<const float2*>(ob_env + 2 * (O - 1));
        float d, nx, ny, ang, dist;
        geom_fast(ob.x - ox, ob.y - oy, d, nx, ny, lo);
        pair_finish<false>(d, nx, ny, hx, hy, cap, ang, dist);
        if (active) { sink.put(2 + (O - 1), ang); sink.put(2 + O + (O - 1), dist); }
        ob_min = fminf(ob_min, dist);
    }
    float ag_min = 3.0e38f;
    int cnt_i = 0;                 // sum_k [min_d < d_k] * [d_k < max_d] (:243-250): a small exact integer either way
    float dk[R];
    constexpr bool kShare = SINK::kReadBack;
    if constexpr (!kShare) {
        auto other = [&](int k, float& dist) {
            const int j = k + (k >= a ? 1 : 0);             // others in ascending index, skipping self (:22-24)
            float d, nx, ny, ang;
            geom_fast(st_env[5 * j + 0] - ox, st_env[5 * j + 1] - oy, d, nx, ny, lo);
            pair_finish<false>(d, nx, ny, hx, hy, cap, ang, dist);
            if (active) { sink.put(2 + 2 * O + k, ang); sink.put(2 + 2 * O + R + k, dist); }
            ag_min = fminf(ag_min, dist);
            cnt_i += (p.agents_min_d < dist && dist < p.agents_max_d) ? 1 : 0;
        };
        if constexpr (!SINK::kReadBack) {
            // the row holds normalised or 16-bit values: keep the raw distances in registers by k (unrolled)
#pragma unroll
            for (int k = 0; k < R; ++k) other(k, dk[k]);
        } else {
#pragma unroll 1
            for (int k = 0; k < R; ++k) { float dist; other(k, dist); }
        }
    } else {
        auto finish = [&](int j, float d, float nx, float ny) {
            float ang, dist;
            pair_finish<false>(d, nx, ny, hx, hy, cap, ang, dist);
            const int k = j - (j > a ? 1 : 0);              // column of agent j among the others of agent a (:22-24)
            if (active) {
                if constexpr (NORM) { sink.put(2 + 2 * O + k, ang); sink.put(2 + 2 * O + R + k, dist); }
                else { float* const dst = sink.row + (2 + 2 * O) + k; dst[0] = ang; dst[R] = dist; }
            }
            ag_min = fminf(ag_min, dist);
            cnt_i += (p.agents_min_d < dist && dist < p.agents_max_d) ? 1 : 0;
        };
        constexpr bool kPow2 = (A & (A - 1)) == 0;
        // The round loop stays ROLLED: unrolled, its 4 geometries + 7 finishes are ~5 KB of straight-line
        // code with many values live across the shuffles (75 registers, 24-25 CTAs/SM); rolled the
        // kernel needs 56 registers, shared memory becomes the occupancy limit (26 CTAs/SM) and the
        // body is fetched once per SM sub-partition instead of once per warp: 146.5 -> 140.5 us at
        // 262144 x 8 x 16 on B200 although it executes 1 % MORE instructions.
#pragma unroll 1
        for (int o = 1; o <= (A - 1) / 2; ++o) {
            const int jf = kPow2 ? ((a + o) & (A - 1)) : (a + o < A ? a + o : a + o - A);
            const int jb = kPow2 ? ((a - o) & (A - 1)) : (a - o >= 0 ? a - o : a - o + A);
            const float pxf = __shfl_sync(FULL, ox, lead + jf), pyf = __shfl_sync(FULL, oy, lead + jf);
            float d, nx, ny;
            geom_fast(pxf - ox, pyf - oy, d, nx, ny, lo);
            const float db = __shfl_sync(FULL, d, lead + jb);
            const float nxb = -__shfl_sync(FULL, nx, lead + jb), nyb = -__shfl_sync(FULL, ny, lead + jb);
            finish(jf, d, nx, ny);
            finish(jb, db, nxb, nyb);
        }
        if constexpr (A % 2 == 0) {
            const int jf = kPow2 ? (a ^ (A / 2)) : (a + A / 2 < A ? a + A / 2 : a - A / 2);
            const float pxf = __shfl_sync(FULL, ox, lead + jf), pyf = __shfl_sync(FULL, oy, lead + jf);
            float d, nx, ny;
            geom_fast(pxf - ox, pyf - oy, d, nx, ny, lo);
            finish(jf, d, nx, ny);
        }
    }
    // fast-path verdict of the whole env (a lane may hold geometry another lane tested)
    const bool mine_ok = !active || (lo > MN_FAST_LO && min3f(td, ob_min, ag_min) >= cap);
    const unsigned b_ok = __ballot_sync(FULL, mine_ok);
    if (__builtin_expect(!(env_ok && (b_ok & gmask) == gmask), 0)) {
        if (active) observe_agent<G, NORM, false>(g, p, rc, st_env, ob_env, tx, ty, a, sink, tm);
        return;
    }
    // bond terms; raw-row build: from the distances this lane just wrote to its own shared-memory row
    float q[R];
#pragma unroll
    for (int k = 0; k < R; ++k) {
        if constexpr (SINK::kReadBack) dk[k] = sink.row[2 + 2 * O + R + k];
        const float sd = div_mode<DM::kSharp, false>(dk[k] - p.ideal_dist, p.bond_sharpness, rc.sharp);
        q[k] = rcp_rn_normal(1.0f + sd * sd);
    }
    tm.risk = (ob_min < p.ob_risk_dist || ag_min < p.ag_risk_dist) ? 1.f : 0.f;    // clamp(ob + ag, max=1)
    tm.coll = ob_min < p.ob_coll_dist || ag_min < p.ag_coll_dist;
    tm.in_t = td < p.target_radius;
    const float cnt = (float)cnt_i;
    const float capped = cnt > p.max_at_prop_d ? p.max_at_prop_d : cnt;
    tm.dsc = div_mode<DM::kProp, false>(capped, p.max_at_prop_d, rc.prop_d);
    tm.head = fabsf(ta) < p.max_angle_diff ? 1.f : 0.f;
    tm.soft = -1.0f * div_mode<DM::kInit, true>(td, p.init_dist, rc.init_dist);
    tm.bond = div_mode<DM::kR, false>(torch_row_sum(q, R), (float)R, rc.R);
}


// Register budget of the fused-actor builds with 16-bit observations: that of 16 resident CTAs (128
// registers), as in step_env_kernel.  At the tile's 28 (72 registers) the actor's row spills 8-28 bytes
// for 1, 2, 4, 5 and 6 obstacles, and at 20 (96) still 4 bytes for 6 -- as the float32 fused-actor
// builds spill at 72, which keep the tile's budget unchanged.
template <bool ACTOR, class OT, int TILE_CTAS>
constexpr int team_ctas() { return ACTOR && sizeof(OT) == 2 && TILE_CTAS > 16 ? 16 : TILE_CTAS; }

template <int TA, int TO, bool NORM, class DM, bool ACTOR = false, class OT = float>
__global__ void __launch_bounds__(32, team_ctas<ACTOR, OT, TeamTile<TA, TO, OT>::CTAS>())
step_team_kernel(const StepArgs args) {
    using W = TeamTile<TA, TO, OT>;
    using G = Geo<TA, TO, W::LPE, 128>;
    constexpr int A = TA, O = TO, S = W::S, ENVS = W::ENVS, LPE = W::LPE, N = 1 + O + (A - 1);
    const marlnav_env_params& p = args.p;
    const marlnav_reset_spec& rs = args.rs;
    const G g(TA, TO);
    const DivConsts rc{args.rc_init_dist, args.rc_prop_d, args.rc_sharp, args.rc_R, args.rc_A};

    extern __shared__ float4 smem_raw[];
    const int lane = threadIdx.x;
    float* const w_st = reinterpret_cast<float*>(smem_raw);
    float* const w_ob = w_st + W::ST;
    float* const w_tg = w_ob + W::OB;
    OT* const w_obs = reinterpret_cast<OT*>(w_tg + W::TG);
    uint64_t* const bar = reinterpret_cast<uint64_t*>(reinterpret_cast<char*>(smem_raw) + W::BYTES);

    // odd steps visit the tiles in reverse, except in the fused-actor build (see step_env_kernel)
    const unsigned tile = (!ACTOR && (rs.step_counter & 1u)) ? gridDim.x - 1u - blockIdx.x : blockIdx.x;
    const long long wenv0 = (long long)tile * ENVS;
    const long long left = (long long)p.num_envs - wenv0;
    const int nenv = left < ENVS ? (int)left : ENVS;
    const bool bulk = args.vec_ok != 0 && nenv == ENVS;
    const int le = lane / LPE, la = lane % LPE;             // local env, agent
    const unsigned lead = (unsigned)(lane & ~(LPE - 1));    // lane of this env's agent 0
    const bool env_live = le < nenv;                        // (lanes beyond the team idle through P1-P3)
    const bool active = env_live && la < A;
    const bool leader = active && la == 0;
    const long long env = wenv0 + le;

    float* const g_st = args.states + wenv0 * (5 * A);
    float* const g_ob = args.obstacles + wenv0 * (2 * O);
    float* const g_tg = args.target + wenv0 * 2;
    OT* const g_obs = reinterpret_cast<OT*>(args.obs) + (size_t)wenv0 * A * S;

    // ---- P0: the tile by TMA bulk copies, per-env scalars and this agent's action straight to
    // registers; nothing is consumed before everything is requested (see step_env_kernel)
    pdl_launch_dependents();
    pdl_wait();
    if constexpr (ACTOR) {
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
    float2 act = make_float2(0.f, 0.f);
    float sn_in = 0.f;
    unsigned char term_raw = 0;
    if (active) {
        if constexpr (!ACTOR) act = load_action(args.actions, env * A + la, args.act8 != 0);
        if (la == 0) {
            sn_in = args.step_num[env];
            term_raw = args.terminates[env];
        }
    }
    if constexpr (ACTOR) {
        // the policy, one (env, agent) row per lane, while the bulk copies are in flight
        // (models.py:27-36, 113-115; see step_env_kernel)
        float* const s_actor = reinterpret_cast<float*>(bar + 2);
        const int H = args.actor.H;
        __syncwarp();
        if (active) {
            const uint64_t counter = args.actor.counter +
                (args.actor.counter_dev ? __ldg(reinterpret_cast<const unsigned long long*>(args.actor.counter_dev)) : 0ull);
            const long long row = env * A + la;
            const OT* const obs_in = static_cast<const OT*>(args.obs_in);
            float x[S];
#pragma unroll
            for (int k = 0; k < S; ++k) x[k] = mna::widen(obs_in[row * S + k]);
            const mna::ActorOut o = mna::actor_row<S>(x, S, H, mna::ActorWeights(s_actor, S, H), args.actor.b_mu,
                                                      args.actor.b_std, nullptr, args.actor.seed, counter, row,
                                                      args.actor.row_offset + (uint64_t)row);
            args.act_out[row * 2] = o.a0; args.act_out[row * 2 + 1] = o.a1;
            args.logp_out[row] = o.logp;
            act = make_float2(o.a0, o.a1);
        }
    }
    if (bulk) {
        mbar_wait(bar, 0);
    } else {
#pragma unroll 1
        for (int i = lane; i < nenv * 5 * A; i += 32) w_st[i] = g_st[i];
        // (env row, column) indexing, the same element as w_ob[i]: plain `i` changes the code
        // generated for 2 obstacles
#pragma unroll 1
        for (int i = lane; i < nenv * 2 * O; i += 32) w_ob[(i / (2 * O)) * (2 * O) + i % (2 * O)] = g_ob[i];
#pragma unroll 1
        for (int i = lane; i < nenv * 2; i += 32) w_tg[i] = g_tg[i];
        __syncwarp();
    }

    float* const st_env = w_st + le * (5 * A);
    float* const ob_env = w_ob + le * (2 * O);
    // the non-reset blend's -0 -> +0 wash, folded into the move's store (see step_env_kernel)
    const bool wash_early = DM::kWash != 0 || ((rs.flags & MARLNAV_RESET_TMPL_NONNEG) != 0 && rs.alias_first_step == 0);
    const float wash = wash_early ? 0.0f : -0.0f;
    // ---- P1: move (ActionScaler, utils.py:546-547, folded into the action load)
    float cmax = 0.f;                                       // this lane's share of max |coordinate| of its env
    if (active) {
        if (args.io.act_scale != nullptr) {
            act.x = (__ldg(args.io.act_scale + 0) * act.x) + __ldg(args.io.act_mean + 0);
            act.y = (__ldg(args.io.act_scale + 1) * act.y) + __ldg(args.io.act_mean + 1);
        }
        float s[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) s[k] = st_env[5 * la + k];
        move_agent(p, s, act.x, act.y);
        cmax = max3_nan_abs(cmax, s[0], s[1]);
#pragma unroll
        for (int k = 0; k < 5; ++k) st_env[5 * la + k] = s[k] + wash;
    }
    // The coordinate bound of the fast path (geom_fast), once per env: each lane takes its own
    // agent (above), its share of the env's obstacle row and the target; one ballot combines them.
    const unsigned gmask = (LPE == 32 ? 0xffffffffu : ((1u << LPE) - 1u)) << lead;
    bool env_ok;
    {
        if (env_live) {
            if constexpr (2 * O == 4 * LPE) {
                const float4 o4 = *reinterpret_cast<const float4*>(ob_env + 4 * la);
                cmax = max3_nan_abs(cmax, o4.x, o4.y);
                cmax = max3_nan_abs(cmax, o4.z, o4.w);
            } else {
                for (int c = la; c < 2 * O; c += LPE) cmax = max_nan(cmax, fabsf(ob_env[c]));
            }
            cmax = max3_nan_abs(cmax, w_tg[le * 2], w_tg[le * 2 + 1]);
        }
        const unsigned b_ok = __ballot_sync(0xffffffffu, cmax < MN_FAST_CMAX);
        env_ok = (b_ok & gmask) == gmask;
    }
    __syncwarp();                                           // P1's stores before P2's reads

    // ---- P2: observe own agent + its reward terms
    // (every lane of the warp takes part: agent pairs exchange their geometry by shuffle; lanes
    // without an agent store nothing and vote neutrally)
    bool all_in = true, coll_any = false;
    AgentTerms tm;
    tm.head = tm.dsc = tm.soft = tm.bond = tm.risk = 0.f; tm.coll = false; tm.in_t = true;
    {
        const float2 tg = *reinterpret_cast<const float2*>(w_tg + le * 2);
        ObsRow<NORM, OT> sink;
        // (lanes without an agent only ever read through it; with LPE == A every lane has a row of its
        // own in the tile, live env or not, and may store to it unpredicated)
        sink.row = w_obs + ((active || LPE == A) ? (le * A + la) * W::OBS_STRIDE : 0);
        sink.mean = args.io.obs_mean; sink.scale = args.io.obs_scale;
        observe_agent_team<G, DM, NORM>(g, p, rc, st_env, ob_env, tg.x, tg.y, la, active, lead, gmask, 4 * le, env_ok, sink, tm);
        if (active) { all_in = tm.in_t; coll_any = tm.coll; }
    }
    // combine over the env's lanes (aligned sub-warps): flags by ballot, the per-agent rewards
    // (environment.py:223-231, evaluated once the env-wide all_in_target flag is known) gathered
    // to every lane and summed in torch's order
    {
        const unsigned b_in = __ballot_sync(0xffffffffu, all_in);
        const unsigned b_co = __ballot_sync(0xffffffffu, coll_any);
        all_in = (b_in & gmask) == gmask;
        coll_any = (b_co & gmask) != 0u;
    }
    const float mine = (((((p.target_factor * (all_in ? 1.0f : 0.0f)) + (p.heading_factor * tm.head)) + (p.distance_factor * tm.dsc)) +
                         (p.soft_factor * tm.soft)) + (p.bond_factor * tm.bond)) - (p.risk_factor * tm.risk);
    float r[A];
#pragma unroll
    for (int i = 0; i < A; ++i) r[i] = __shfl_sync(0xffffffffu, mine, lead + i);
    const float reward = div_mode<DM::kA, false>(torch_row_sum(r, A), (float)A, rc.A);

    // ---- P3 (environment.py:96-103, 209-221)
    bool done = false, trunc = false;
    if (leader) {
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
    const unsigned b_tr = __ballot_sync(0xffffffffu, leader && trunc);
    const unsigned b_co2 = __ballot_sync(0xffffffffu, leader && coll_any);
    const unsigned b_ta = __ballot_sync(0xffffffffu, leader && all_in);
    const unsigned dmask = __ballot_sync(0xffffffffu, leader && done);     // one bit per reset env, at its leader lane
    if (lane == 0) {
        if (b_tr) atomicAdd(args.stats + 0, (unsigned long long)__popc(b_tr));
        if (b_co2) atomicAdd(args.stats + 1, (unsigned long long)__popc(b_co2));
        if (b_ta) atomicAdd(args.stats + 2, (unsigned long long)__popc(b_ta));
    }
    done = (dmask >> lead) & 1u;
    if constexpr (DM::kFinal) {
        // the finished envs' rows before P4b re-observes them (see step_env_kernel), unpadded
        __syncwarp();
        OT* const g_fin = static_cast<OT*>(args.final_obs) + (size_t)wenv0 * A * S;
        for (unsigned m = dmask; m != 0u; m &= m - 1u) {
            const int e2 = (__ffs((int)m) - 1) / LPE;
            copy_final_rows(g_fin + (size_t)e2 * A * S, w_obs + e2 * A * W::OBS_STRIDE, A, S, W::OBS_STRIDE, lane);
        }
    }
    // ---- P4a: masked re-initialisation (environment.py:76-90): x = (1-m)*x + m*new
    if (active) {
        const bool alias = DM::kWash == 0 && rs.alias_first_step != 0;
        const float* ts = rs.tmpl_states + env * rs.states_env_stride;
        const int k0 = 5 * la;                              // this lane's slice of the env's state row
        if (done || !wash_early) {          // (an env that keeps going was already blended by the move's store)
            const bool noisy = DM::kWash == 0 && (rs.flags & MARLNAV_RESET_NOISY_AGENTS) != 0;
            float nv[5];
            if (noisy) sample_agent_noisy(rs, reset_counter(rs), rs.env_id_offset + (uint64_t)env, la, ts + k0, nv);
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const float old_v = st_env[k0 + k];
                const float new_v = noisy ? nv[k] : (alias ? old_v : __ldg(ts + k0 + k));
                st_env[k0 + k] = done ? ((0.0f * old_v) + new_v) : (old_v + (0.0f * new_v));
            }
        }
    }
    if (env_live && done) {
        // obstacles / target are rewritten (smem and HBM) only for envs that reset; all LPE lanes
        // of the env share the work
        const bool alias = DM::kWash == 0 && rs.alias_first_step != 0;
        if (rs.tmpl_obstacles || alias) {
            const float* to = alias ? nullptr : rs.tmpl_obstacles + env * rs.obstacles_env_stride;
            for (int c = la; c < 2 * O; c += LPE) {
                const float old_v = ob_env[c];
                ob_env[c] = (0.0f * old_v) + (alias ? old_v : __ldg(to + c));
                g_ob[le * (2 * O) + c] = ob_env[c];
            }
        } else {
            for (int pr = la; 2 * pr < O; pr += LPE) {
                float nw[4];
                sample_obstacle_pair(p, rs.seed, reset_counter(rs), rs.env_id_offset + (uint64_t)env, pr, nw);
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (4 * pr + c < 2 * O) {
                        ob_env[4 * pr + c] = (0.0f * ob_env[4 * pr + c]) + nw[c];
                        g_ob[le * (2 * O) + 4 * pr + c] = ob_env[4 * pr + c];
                    }
            }
        }
        if (la == 0) {
            const float* tt = rs.tmpl_target + env * rs.target_env_stride;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const float old_v = w_tg[le * 2 + c];
                w_tg[le * 2 + c] = (0.0f * old_v) + (alias ? old_v : __ldg(tt + c));
                g_tg[le * 2 + c] = w_tg[le * 2 + c];
            }
        }
    }
    __syncwarp();

    // ---- P4b: re-observe this warp's reset envs, one (env, agent, object) pair per lane
    // (see step_env_kernel); reset envs one after the other (rarely more than one per warp), their
    // A * N pairs spread over the 32 lanes
    {
        const float cap = p.cap_distance;
#pragma unroll 1
        for (unsigned m = dmask; m != 0u; m &= m - 1u) {
            const int e2 = (__ffs((int)m) - 1) / LPE;
            const float* st2 = w_st + e2 * (5 * A);
#pragma unroll 1
            for (int w2 = lane; w2 < A * N; w2 += 32) {
                const int a = w2 / N, obj = w2 - a * N;
                float px, py;
                int col_a, col_d;
                if (obj == 0) {
                    px = w_tg[e2 * 2]; py = w_tg[e2 * 2 + 1]; col_a = 0; col_d = 1;
                } else if (obj <= O) {
                    px = w_ob[e2 * (2 * O) + 2 * (obj - 1)]; py = w_ob[e2 * (2 * O) + 2 * (obj - 1) + 1];
                    col_a = 1 + obj; col_d = 1 + O + obj;
                } else {
                    const int k = obj - 1 - O, jj = k + (k >= a ? 1 : 0);
                    px = st2[5 * jj]; py = st2[5 * jj + 1];
                    col_a = 2 + 2 * O + k; col_d = 2 + 2 * O + (A - 1) + k;
                }
                float ang, dist;
                // (guarded arithmetic for every pair: a freshly reset team has exactly aligned agents, so with
                // pair_obs both of its branches would run in every iteration)
                pair_guarded(st2[5 * a], st2[5 * a + 1], st2[5 * a + 2], st2[5 * a + 3], px, py, cap, ang, dist);
                ObsRow<NORM, OT> sink;
                sink.row = w_obs + (e2 * A + a) * W::OBS_STRIDE; sink.mean = args.io.obs_mean; sink.scale = args.io.obs_scale;
                sink.put(col_a, ang); sink.put(col_d, dist);
            }
        }
    }

    // ---- P5: stage out
    if (bulk) {
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
            bulk_s2g(g_st, w_st, W::ST * 4);
            if constexpr (W::kObsBulk) bulk_s2g(g_obs, w_obs, W::OBS * sizeof(OT));
            bulk_commit_wait_read();
        }
        if constexpr (!W::kObsBulk) {
            // padded rows: the warp copies its tile out itself (16-byte pieces, fully coalesced).  (One
            // bulk copy per lane of its own 192-byte row instead: 181.8 vs 169.9 us at (8,16) -- 32 small
            // TMA operations per warp cost more than the 12-step loop.)
            constexpr int s4 = S / W::E16, st4 = W::OBS_STRIDE / W::E16, TOT = ENVS * A * s4;
            const float4* src = reinterpret_cast<const float4*>(w_obs);
            // float4 i = lane + 32 * it of the tile sits in row i / s4, column i % s4.  Both repeat with
            // period PER = lcm(32, s4) / 32 iterations (32 * PER float4s = a whole number of rows), so
            // the PER (row, column) splits are taken once and every other address is an immediate.
            constexpr int PER = W::kCopyPeriod;
            if constexpr (PER <= 4 && TOT % (32 * PER) == 0) {
                int off[PER];
#pragma unroll
                for (int u = 0; u < PER; ++u) {
                    const int i = lane + 32 * u, r2 = i / s4;
                    off[u] = r2 * st4 + (i - r2 * s4);
                }
                constexpr int ROWS_PER = 32 * PER / s4;
#pragma unroll
                for (int mrep = 0; mrep < TOT / (32 * PER); ++mrep)
#pragma unroll
                    for (int u = 0; u < PER; ++u)
                        stg_stream4(reinterpret_cast<float4*>(g_obs) + (lane + 32 * (u + PER * mrep)),
                                    src[off[u] + mrep * ROWS_PER * st4]);
            } else {
#pragma unroll 4
                for (int i = lane; i < TOT; i += 32) {
                    const int r2 = i / s4, c = i - r2 * s4;
                    stg_stream4(reinterpret_cast<float4*>(g_obs) + i, src[r2 * st4 + c]);
                }
            }
        }
    } else {
        __syncwarp();
#pragma unroll 1
        for (int i = lane; i < nenv * 5 * A; i += 32) g_st[i] = w_st[i];
#pragma unroll 1
        for (int i = lane; i < nenv * A * S; i += 32) {
            const int r2 = i / S, c = i - r2 * S;
            g_obs[i] = w_obs[r2 * W::OBS_STRIDE + c];
        }
    }
}

}  // namespace mn

namespace mnl {

template <class OT>
int launch_team3(const mn::StepArgs& a, cudaStream_t st, int* info) {
    switch (a.p.num_obstacles) {
        case 1: return launch_step_tile<mn::TeamTile, 3, 1, mn::DivModesDefault, OT>(a, st, info);
        case 2: return launch_step_tile<mn::TeamTile, 3, 2, mn::DivModesDefault, OT>(a, st, info);
        case 3: return launch_step_tile<mn::TeamTile, 3, 3, mn::DivModesDefault, OT>(a, st, info);
        case 4: return launch_step_tile<mn::TeamTile, 3, 4, mn::DivModesDefault, OT>(a, st, info);
        case 5: return launch_step_tile<mn::TeamTile, 3, 5, mn::DivModesDefault, OT>(a, st, info);
        case 6: return launch_step_tile<mn::TeamTile, 3, 6, mn::DivModesDefault, OT>(a, st, info);
        default: return -1;
    }
}
template <class OT>
int launch_team8x16(const mn::StepArgs& a, cudaStream_t st, int* info) {
    return launch_step_tile<mn::TeamTile, 8, 16, mn::DivModesTeam8, OT>(a, st, info);
}
template int launch_team3<float>(const mn::StepArgs&, cudaStream_t, int*);
template int launch_team3<__half>(const mn::StepArgs&, cudaStream_t, int*);
template int launch_team3<__nv_bfloat16>(const mn::StepArgs&, cudaStream_t, int*);
template int launch_team8x16<float>(const mn::StepArgs&, cudaStream_t, int*);
template int launch_team8x16<__half>(const mn::StepArgs&, cudaStream_t, int*);
template int launch_team8x16<__nv_bfloat16>(const mn::StepArgs&, cudaStream_t, int*);

}  // namespace mnl
