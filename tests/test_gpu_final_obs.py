"""GPU: final observations of auto-reset envs (Env.step_fused(final_obs=...), collect_rollout /
RolloutGraph(final_obs=True)) and the truncation-aware GAE scan (marlnav_b200.gae).

For every env a step finishes, final_obs holds the observations its rewards and flags were computed
from -- the C oracle's `want_pre` rows, bit for bit (rounded for 16-bit envs, normalised with the
fused normaliser) -- and rows of the other envs keep whatever they held.  Asking for them changes
nothing else the step computes."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import action_pool, cpu_params

pytestmark = pytest.mark.gpu

INT_OF = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}
SENTINEL = {4: 0x7FBADBAD, 2: 0x7E5B}          # bit patterns no observation takes


def bits(t):
    return t.contiguous().view(INT_OF[t.element_size()])


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle as o
    o.lib()
    return o


def _params(B, A, O, seed=11, dtype=None, noisy=False, **kw):
    import marlnav_b200 as mb
    p = mb.default_env_params(B, A, O, sampling_style='policy', **kw) if A == 3 else \
        mb.template_env_params(B, A, O, **kw)
    p['seed'] = seed
    if dtype is not None:
        p['obs_dtype'] = dtype
    if noisy:
        p['init']['noisy_ags'] = True
    return p


def _io_params(A, O):
    max_d = math.sqrt(1500.0 ** 2 + 750.0 ** 2)
    lo = [-math.pi, 0.] + O * [-math.pi] + O * [0.] + (A - 1) * [-math.pi] + (A - 1) * [0.]
    hi = [math.pi, max_d] + O * [math.pi] + O * [max_d] + (A - 1) * [math.pi] + (A - 1) * [max_d]
    return dict(min_obs=lo, max_obs=hi), dict(min_action=[-math.pi, -0.5], max_action=[math.pi, 0.5])


def _final_buffer(env, offset=0):
    """(B,A,S) view `offset` elements into a sentinel-filled buffer (offset 1: a base misaligned by
    one element), and the whole buffer."""
    B, A, S = env.num_parallel, env.num_agents, env.obs_size
    raw = torch.empty(B * A * S + 8, dtype=env.obs_dtype, device=env.device)
    bits(raw).fill_(SENTINEL[raw.element_size()])
    return raw[offset:offset + B * A * S].view(B, A, S), raw


def _want(pre, dtype, io):
    """The oracle's pre-reset rows as the env stores them: normalised like the fused normaliser,
    rounded to the env's type."""
    if io is not None:
        pre = ((pre - io[0]).astype(np.float32) / io[1]).astype(np.float32)
    return torch.from_numpy(pre).to(dtype)


def _run_against_oracle(orc, params, steps=300, io=False, geometry=None, offset=0, angle=0.2, seed=11):
    """Steps an env with final_obs and the C oracle with want_pre side by side; returns the number of
    finished envs whose final rows were compared."""
    import marlnav_b200 as mb
    B, A, O = params['num_parallel'], params['num_agents'], params['num_obstacles']
    env = mb.Env(dict(params, seed=seed))
    oe = orc.OracleEnv(cpu_params(params), seed=seed)
    for k, v in (geometry or {}).items():
        setattr(env._c_params, k, v)
        setattr(oe.p, k, v)
    io_np = None
    if io:
        norm, scal = _io_params(A, O)
        env.fuse_io(norm, scal)
        lo, hi = torch.tensor(norm['min_obs']), torch.tensor(norm['max_obs'])
        io_np = ((0.5 * (lo + hi)).numpy(), (0.5 * (hi - lo)).numpy())
        a_lo, a_hi = torch.tensor(scal['min_action']), torch.tensor(scal['max_action'])
        a_scale, a_mean = (0.5 * (a_hi - a_lo)).numpy(), (0.5 * (a_lo + a_hi)).numpy()
    fin, raw = _final_buffer(env, offset)
    sentinel = bits(raw).clone()
    pool = action_pool(B, A, angle=angle)
    checked = 0
    for t in range(steps):
        act = pool[t % len(pool)]
        bits(raw).copy_(sentinel)
        obs, rew, term, trunc = env.step_fused(act.cuda(), final_obs=fin)
        o_act = ((a_scale * act.numpy()).astype(np.float32) + a_mean) if io else act.numpy()
        o_obs, o_rew, o_term, o_trunc, o_pre = oe.step_fused(o_act, want_pre=True)
        tag = f"step {t}"
        assert np.array_equal(term.cpu().numpy(), o_term) and np.array_equal(trunc.cpu().numpy(), o_trunc), tag
        assert np.array_equal(rew.cpu().numpy().view(np.uint32), o_rew.view(np.uint32)), tag
        assert torch.equal(bits(obs.cpu()), bits(_want(o_obs, env.obs_dtype, io_np))), tag
        done = torch.from_numpy(o_term | o_trunc)
        got = fin.cpu()
        assert torch.equal(bits(got[done]), bits(_want(o_pre, env.obs_dtype, io_np)[done])), tag
        assert bool((bits(got[~done]) == SENTINEL[got.element_size()]).all()), f"{tag}: rows of unfinished envs written"
        assert torch.equal(bits(raw)[:offset], sentinel[:offset]), tag
        assert torch.equal(bits(raw)[offset + fin.numel():], sentinel[offset + fin.numel():]), tag
        checked += int(done.sum())
    assert checked > 0
    return env, checked


def _expected_tile(B, A, O):
    """Envs per CTA of the kernel the dispatcher picks (MARLNAV_TEAM3_MAX_ENVS is read once per process)."""
    if A == 3 and O <= 6:
        limit = int(os.environ.get("MARLNAV_TEAM3_MAX_ENVS", "32768"))
        return 8 if B <= limit else 32
    if (A, O) == (8, 16):
        return 4
    return 128


# team of 3 below 32 768 envs (thread per agent), above it (thread per env), (8,16), generic shapes,
# ragged batch sizes
ORACLE_SHAPES = [(1000, 3, 1), (1000, 3, 2), (1000, 3, 3), (1000, 3, 4), (1000, 3, 5), (1000, 3, 6),
                 (40000, 3, 3), (40001, 3, 5), (1000, 8, 16), (301, 8, 16), (200, 4, 2), (203, 5, 7),
                 (1, 3, 3), (33, 3, 3), (130, 3, 6)]
DTYPES = [torch.float32, torch.float16, torch.bfloat16]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B,A,O", ORACLE_SHAPES)
def test_final_obs_equal_the_oracle_pre_reset_rows(orc, B, A, O, dtype):
    env, checked = _run_against_oracle(orc, _params(B, A, O, dtype=dtype), steps=300)
    assert env.launch_info()[3] == _expected_tile(B, A, O)
    if B >= 200:
        assert env._num_trunc > 0 and checked > env._num_trunc     # truncations and terminations both seen


@pytest.mark.parametrize("O", [1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("dtype", DTYPES)
def test_team3_small_batches(orc, O, dtype):
    """Small team-of-3 batches with episode_len 40: in this process thread per agent; run again below
    with MARLNAV_TEAM3_MAX_ENVS=0 through the thread-per-env kernel."""
    env, _ = _run_against_oracle(orc, _params(257, 3, O, dtype=dtype, episode_len=40), steps=300)
    assert env.launch_info()[3] == _expected_tile(257, 3, O)


def test_team3_small_batches_through_the_thread_per_env_kernel():
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, MARLNAV_TEAM3_MAX_ENVS="0")
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.join(here, "test_gpu_final_obs.py"), "-q", "-x",
                          "-m", "gpu", "-k", "test_team3_small_batches and not thread_per_env or mock_initializer",
                          "-p", "no:cacheprovider"], env=env, capture_output=True, text=True, cwd=os.path.dirname(here))
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-2000:]
    assert " passed" in res.stdout and "failed" not in res.stdout


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("B,A,O", [(777, 3, 3), (40000, 3, 3), (300, 8, 16), (200, 4, 2)])
def test_normalised_final_obs(orc, B, A, O, dtype):
    _run_against_oracle(orc, _params(B, A, O, dtype=dtype, episode_len=60), steps=200, io=True, angle=0.08)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B", [1000, 40000])
def test_noisy_resets(orc, B, dtype):
    _run_against_oracle(orc, _params(B, 3, 3, dtype=dtype, noisy=True, episode_len=50), steps=150)


@pytest.mark.parametrize("geometry", [
    dict(init_dist=1234.5, max_at_prop_d=3.0, bond_sharpness=2.0),
    dict(init_dist=1024.0, max_at_prop_d=1.0, bond_sharpness=0.7, ideal_dist=35.0, target_radius=45.0),
])
@pytest.mark.parametrize("B,A,O", [(1500, 3, 3), (40000, 3, 3), (300, 8, 16), (200, 5, 3)])
def test_custom_geometry_constants(orc, B, A, O, geometry):
    _run_against_oracle(orc, _params(B, A, O, episode_len=50), steps=120, geometry=geometry, seed=5)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("sn", [0, 1])
def test_mock_initializer_first_step_alias(orc, sn, dtype):
    """The reference's mock scenarios: the reset template is the state after the first move."""
    import marlnav_b200 as mb
    p = mb.default_env_params(sampler_num=sn, sampling_style='policy', episode_len=7)
    p['obs_dtype'] = dtype
    _run_against_oracle(orc, p, steps=40, angle=0.05)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B,A,O", [(40000, 3, 3), (1000, 3, 3), (33, 3, 3), (1000, 8, 16), (203, 5, 7)])
def test_misaligned_final_obs_gives_the_same_bits(orc, B, A, O, dtype):
    """A base one element off (4-byte aligned for float32, 2-byte for 16-bit)."""
    _run_against_oracle(orc, _params(B, A, O, dtype=dtype, episode_len=40), steps=100, offset=1)


@pytest.mark.parametrize("io", [False, True])
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B,A,O", [(40000, 3, 3), (1000, 3, 3), (1000, 8, 16), (203, 5, 7)])
def test_final_obs_has_no_side_effects(B, A, O, dtype, io):
    """Twins stepped with and without final_obs: identical states, obstacles, target, counters,
    observations, rewards, flags and episode stats."""
    import marlnav_b200 as mb
    twins = [mb.Env(_params(B, A, O, dtype=dtype, episode_len=30)) for _ in range(2)]
    if io:
        for e in twins:
            e.fuse_io(*_io_params(A, O))
    fin, _ = _final_buffer(twins[1])
    pool = [a.cuda() for a in action_pool(B, A, angle=0.3)]
    for t in range(90):
        a = twins[0].step_fused(pool[t % len(pool)])
        b = twins[1].step_fused(pool[t % len(pool)], final_obs=fin)
        for x, y, name in zip(a, b, ('obs', 'rewards', 'terminated', 'truncated')):
            assert torch.equal(bits(x), bits(y)), (t, name)
    for name in ('states', 'obstacles', 'target', '_step_num', '_terminates_u8', 'episode_stats'):
        assert torch.equal(bits(getattr(twins[0], name)), bits(getattr(twins[1], name))), name


def test_sharded_final_obs_equal_single_process():
    import marlnav_b200 as mb
    full = _params(600, 3, 3, seed=5, episode_len=30)
    e_full = mb.Env(full)
    shards = [mb.Env(mb.shard_env_params(full, r, 2)) for r in range(2)]
    f_full, _ = _final_buffer(e_full)
    f_parts = [_final_buffer(s)[0] for s in shards]
    pool = action_pool(600, 3)
    for t in range(150):
        act = pool[t % len(pool)].cuda()
        _, _, te, tr = e_full.step_fused(act, final_obs=f_full)
        for i, s in enumerate(shards):
            s.step_fused(act[i * 300:(i + 1) * 300].contiguous(), final_obs=f_parts[i])
        assert torch.equal(bits(f_full), bits(torch.cat(f_parts))), t
    assert torch.equal(e_full.states, torch.cat([s.states for s in shards]))


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("B", [300, 40000])
def test_cuda_graph_of_steps_with_final_obs_matches_eager(B, dtype):
    import marlnav_b200 as mb
    T = 64
    p = _params(B, 3, 3, seed=31, dtype=dtype, episode_len=25)
    pool = [a.cuda() for a in action_pool(B, 3, angle=0.3)]
    eager = mb.Env(dict(p))
    ref = []
    for i in range(2 * T):
        f, _ = _final_buffer(eager)
        out = eager.step_fused(pool[i % len(pool)], final_obs=f)
        ref.append([t.clone() for t in out] + [f.clone()])
    env = mb.Env(dict(p))
    env.use_device_counter(True)
    outs = [env._alloc_outputs() for _ in range(T)]
    fins = [_final_buffer(env)[0] for _ in range(T)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            env.batch_device_counter(True)
            for i in range(T):
                env.step_fused(pool[i % len(pool)], out=outs[i], final_obs=fins[i])
            env.batch_device_counter(False)
    torch.cuda.current_stream().wait_stream(side)
    ndone = 0
    for k in range(2):
        g.replay()
        torch.cuda.synchronize()
        for i in range(T):
            o, r, te, tr = outs[i]
            ro, rr, rte, rtr, rf = ref[k * T + i]
            assert torch.equal(bits(o), bits(ro)) and torch.equal(r, rr), (k, i)
            assert torch.equal(te.view(torch.bool), rte) and torch.equal(tr.view(torch.bool), rtr), (k, i)
            done = rte | rtr
            assert torch.equal(bits(fins[i][done]), bits(rf[done])), (k, i)
            ndone += int(done.sum())
    assert ndone > 0
    assert torch.equal(env.states, eager.states) and torch.equal(env.obstacles, eager.obstacles)


def test_bad_final_obs_buffers_are_refused():
    import marlnav_b200 as mb
    env = mb.Env(_params(64, 3, 3))
    B, A, S = 64, 3, env.obs_size
    act = torch.zeros(B, A, 2, device='cuda')
    out = env._alloc_outputs()
    bad = [torch.empty(B, A, S, dtype=torch.float16, device='cuda'),          # wrong dtype
           torch.empty(B * A * S - 1, device='cuda'),                         # short
           torch.empty(B, A, S),                                              # host memory
           torch.empty(B, A, 2 * S, device='cuda')[:, :, :S]]                 # not contiguous
    for f in bad:
        with pytest.raises(mb.MarlnavError, match="final_obs"):
            env.step_fused(act, final_obs=f)
    with pytest.raises(mb.MarlnavError, match="different buffers"):
        env.step_fused(act, out=out, final_obs=out[0])
    assert env._reset_counter == 0                                            # nothing was launched


# ---------------------------------------------------------------------------- rollouts

def _actor_weights(S=12, H=50, seed=0):
    g = torch.Generator().manual_seed(seed)
    w = {'fc1.weight': torch.empty(H, S), 'fc_mu.weight': torch.empty(2, H), 'fc_std.weight': torch.empty(2, H)}
    for v in w.values():
        torch.nn.init.orthogonal_(v, generator=g)
    w.update({'fc1.bias': torch.rand(H, generator=g) * 0.2 - 0.1, 'fc_mu.bias': torch.rand(2, generator=g) - 0.5,
              'fc_std.bias': torch.rand(2, generator=g) - 0.5})
    return w


def _critic_weights(K, H=50, seed=2):
    g = torch.Generator().manual_seed(seed)
    fc1, fc2 = torch.nn.Linear(K, H), torch.nn.Linear(H, 1)
    torch.nn.init.orthogonal_(fc1.weight, generator=g); torch.nn.init.orthogonal_(fc2.weight, generator=g)
    return {'fc1.weight': fc1.weight.detach(), 'fc1.bias': fc1.bias.detach(),
            'fc2.weight': fc2.weight.detach(), 'fc2.bias': fc2.bias.detach()}


def _rollout_env(B, O, dtype, seed=21):
    import marlnav_b200 as mb
    env = mb.Env(_params(B, 3, O, seed=seed, dtype=dtype, episode_len=25))
    env.fuse_io(*_io_params(3, O))
    return env


ROLLOUT_KEYS = ('obs', 'last_obs', 'actions', 'log_probs', 'rewards', 'done', 'values')


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("B,O", [(256, 3), (40000, 3), (1000, 5)])
def test_collect_rollout_final_obs(B, O, dtype):
    import marlnav_b200 as mb
    T, S = 60, 2 + 2 * O + 4
    w, cw = _actor_weights(S), _critic_weights(3 * S)
    runs = []
    for fin in (False, True):
        env = _rollout_env(B, O, dtype)
        runs.append(mb.collect_rollout(env, mb.FusedActor(w, seed=3), T, critic=mb.FusedCritic(cw), obs_dtype=dtype,
                                       final_obs=fin))
    plain, withf = runs
    for key in ROLLOUT_KEYS:
        assert torch.equal(bits(plain[key]), bits(withf[key])), key
    assert 'final_obs' not in plain
    assert torch.equal(withf['done'], withf['terminated'] | withf['truncated'])
    done = withf['done']
    assert int(done.sum()) > 0 and bool(withf['truncated'].any())
    # a twin env replaying the recorded actions through step_fused(final_obs=...)
    twin = _rollout_env(B, O, dtype)
    for t in range(T):
        f, _ = _final_buffer(twin)
        _, _, te, tr = twin.step_fused(withf['actions'][t].view(B, 3, 2), final_obs=f)
        assert torch.equal(te, withf['terminated'][t]) and torch.equal(tr, withf['truncated'][t]), t
        assert torch.equal(bits(f[done[t]]), bits(withf['final_obs'][t][done[t]])), t
    # final_values: the critic on those rows
    critic = mb.FusedCritic(cw)
    for t in range(T):
        v = critic(withf['final_obs'][t].view(B, 3 * S))
        assert torch.equal(bits(v[done[t]]), bits(withf['final_values'][t][done[t]])), t


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_rollout_graph_final_obs_replays_equal_the_eager_rollouts(dtype):
    import marlnav_b200 as mb
    B, O, T = 256, 3, 60
    w, cw = _actor_weights(), _critic_weights(36)

    def make():
        return _rollout_env(B, O, dtype, seed=12), mb.FusedActor(w, seed=3), mb.FusedCritic(cw)
    env_e, act_e, cri_e = make()
    mb.collect_rollout(env_e, act_e, 2, critic=cri_e, obs_dtype=dtype, final_obs=True)   # RolloutGraph's warm-up
    eager = [mb.collect_rollout(env_e, act_e, T, critic=cri_e, obs_dtype=dtype, final_obs=True) for _ in range(2)]
    env_g, act_g, cri_g = make()
    rg = mb.RolloutGraph(env_g, act_g, T, critic=cri_g, warmup_steps=2, obs_dtype=dtype, final_obs=True)
    for k in range(2):
        buf = rg.replay()
        torch.cuda.synchronize()
        for key in ROLLOUT_KEYS + ('terminated', 'truncated'):
            assert torch.equal(bits(buf[key]), bits(eager[k][key])), (k, key)
        done = eager[k]['done']
        assert int(done.sum()) > 0
        assert torch.equal(bits(buf['final_obs'][done]), bits(eager[k]['final_obs'][done])), k
        assert torch.equal(bits(buf['final_values'][done]), bits(eager[k]['final_values'][done])), k
    assert torch.equal(env_g.states, env_e.states) and torch.equal(env_g.obstacles, env_e.obstacles)


# ---------------------------------------------------------------------------- gae

def gae_reference(rewards, values, terminated, truncated, gamma, lam, final_values=None, last_values=None):
    """numpy float64 restatement, vectorised over envs: each operation one IEEE round-to-nearest
    float64 operation (numpy does not contract a*b+c)."""
    T, B = rewards.shape
    gamma, lam = np.float64(gamma), np.float64(lam)
    gl = gamma * lam
    r, v = rewards.astype(np.float64), values.astype(np.float64)
    fv = final_values.astype(np.float64) if final_values is not None else np.zeros((T, B))
    adv, ret = np.empty((T, B)), np.empty((T, B))
    a_next = np.zeros(B)
    for t in range(T - 1, -1, -1):
        if t == T - 1:
            nv = last_values.astype(np.float64) if last_values is not None else np.zeros(B)
        else:
            nv = v[t + 1]
        nv = np.where(terminated[t], 0.0, np.where(truncated[t], fv[t], nv))
        cont = ~(terminated[t] | truncated[t])
        delta = (r[t] + gamma * nv) - v[t]
        a_next = np.where(cont, delta + gl * a_next, delta)
        adv[t] = a_next
        ret[t] = a_next + v[t]
    return adv, ret


def _gae_inputs(T, B, p_term, p_trunc, seed):
    g = torch.Generator().manual_seed(seed)
    r = torch.randn(T, B, generator=g)
    v = torch.randn(T, B, 1, generator=g) * 3
    fv = torch.randn(T, B, 1, generator=g) * 3
    lv = torch.randn(B, generator=g)
    te = torch.rand(T, B, generator=g) < p_term
    tr = torch.rand(T, B, generator=g) < p_trunc
    return r, v, te, tr, fv, lv


@pytest.mark.parametrize("T,B,p_term,p_trunc", [
    (1, 5, 0.3, 0.3), (1000, 1024, 0.02, 0.02), (37, 129, 0.1, 0.2), (9, 33, 1.0, 0.0), (9, 33, 0.0, 1.0),
    (16, 7, 1.0, 1.0), (250, 1, 0.05, 0.05)])
@pytest.mark.parametrize("with_final,with_last", [(True, True), (False, True), (True, False), (False, False)])
def test_gae_bit_exact(T, B, p_term, p_trunc, with_final, with_last):
    import marlnav_b200 as mb
    r, v, te, tr, fv, lv = _gae_inputs(T, B, p_term, p_trunc, seed=T * 7 + B)
    if T > 1:
        tr[T - 1, : B // 2 + 1] = True            # truncation on the last step
        te[T - 1, 0] = True                       # ... and with terminated on the same step
    gamma, fv_arg, lv_arg = 0.99, fv if with_final else None, lv if with_last else None
    for lam in (0.0, 0.95, 1.0):
        adv, ret = mb.gae(r.cuda(), v.cuda(), te.cuda(), tr.cuda(), gamma, lam,
                          final_values=None if fv_arg is None else fv_arg.cuda(),
                          last_values=None if lv_arg is None else lv_arg.cuda())
        assert adv.dtype == torch.float64 and adv.shape == (T, B)
        want_a, want_r = gae_reference(r.numpy(), v.numpy()[..., 0], te.numpy(), tr.numpy(), gamma, lam,
                                       None if fv_arg is None else fv_arg.numpy()[..., 0],
                                       None if lv_arg is None else lv_arg.numpy())
        assert np.array_equal(adv.cpu().numpy().view(np.uint64), want_a.view(np.uint64)), lam
        assert np.array_equal(ret.cpu().numpy().view(np.uint64), want_r.view(np.uint64)), lam


def test_gae_at_lambda_one_with_zero_values_is_discounted_returns():
    """discounted_returns (the reference's scan) sets the return of a done step to 0, dropping that
    step's reward, where gae keeps it (adv = r).  With those rewards zeroed, values 0, no truncations
    and lambda 1, gae's returns are discounted_returns bit for bit; with them kept, the two differ."""
    import marlnav_b200 as mb
    r, _, te, _, _, _ = _gae_inputs(200, 300, 0.05, 0.0, seed=4)
    r, te = r.cuda(), te.cuda()
    zero, no_trunc = torch.zeros(200, 300, device='cuda'), torch.zeros_like(te)
    r0 = torch.where(te, torch.zeros_like(r), r)
    _, ret = mb.gae(r0, zero, te, no_trunc, 0.97, 1.0)
    assert torch.equal(bits(ret), bits(mb.discounted_returns(r0, te, 0.97)))
    _, ret_r = mb.gae(r, zero, te, no_trunc, 0.97, 1.0)
    assert torch.equal(ret_r[te], r[te].double())


def test_gae_refuses_bad_shapes():
    import marlnav_b200 as mb
    r = torch.zeros(4, 3, device='cuda')
    f = torch.zeros(4, 3, dtype=torch.bool, device='cuda')
    with pytest.raises(mb.MarlnavError, match="values"):
        mb.gae(r, torch.zeros(4, 2, device='cuda'), f, f, 0.9, 0.9)
    with pytest.raises(mb.MarlnavError, match="last_values"):
        mb.gae(r, r, f, f, 0.9, 0.9, last_values=torch.zeros(4, device='cuda'))
    with pytest.raises(mb.MarlnavError, match="truncated"):
        mb.gae(r, r, f, f[:3], 0.9, 0.9)
