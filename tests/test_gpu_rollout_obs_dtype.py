"""GPU: rollouts into float16 / bfloat16 observation buffers (collect_rollout / RolloutGraph with
obs_dtype).  The actor and the critic read a stored 16-bit observation widened exactly to float32, so
they give the bits of their float32 call on ``obs16.float()``; the fused act+step launch gives the
bits of the two-launch route; and a float32 twin env driven with a 16-bit rollout's recorded actions
reaches the same states, rewards and flags, its normalised observations rounded being the buffer."""
import math
import types

import pytest
import torch

pytestmark = pytest.mark.gpu

DTYPES = [torch.float16, torch.bfloat16]
INT_OF = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}


def bits(t):
    return t.contiguous().view(INT_OF[t.element_size()])


def assert_bits(tag, a, b):
    assert a.dtype == b.dtype and a.shape == b.shape, (tag, a.dtype, b.dtype, a.shape, b.shape)
    assert torch.equal(bits(a), bits(b)), (tag, int((bits(a) != bits(b)).sum()))


def assert_rounded(tag, o16, o32):
    """o16 == o32.to(dtype) bit for bit; NaN positions equal, payloads unspecified."""
    want = o32.to(o16.dtype)
    same = (bits(o16) == bits(want)) | (torch.isnan(o16) & torch.isnan(want))
    assert bool(same.all()), (tag, int((~same).sum()))


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


def _io_params(A, O):
    max_d = math.sqrt(1500.0 ** 2 + 750.0 ** 2)
    lo = [-math.pi, 0.] + O * [-math.pi] + O * [0.] + (A - 1) * [-math.pi] + (A - 1) * [0.]
    hi = [math.pi, max_d] + O * [math.pi] + O * [max_d] + (A - 1) * [math.pi] + (A - 1) * [max_d]
    return dict(min_obs=lo, max_obs=hi), dict(min_action=[-math.pi, -0.5], max_action=[math.pi, 0.5])


def _params(B, A, O, dtype=None, seed=21, **kw):
    import marlnav_b200 as mb
    p = mb.default_env_params(B, A, O, sampling_style='policy', **kw) if A == 3 else \
        mb.template_env_params(B, A, O, **kw)
    p['seed'] = seed
    if dtype is not None:
        p['obs_dtype'] = dtype
    return p


def _env(B, A, O, dtype=None, **kw):
    import marlnav_b200 as mb
    env = mb.Env(_params(B, A, O, dtype, **kw))
    env.fuse_io(*_io_params(A, O))
    return env


def _obs_size(A, O):
    return 2 + 2 * O + 2 * (A - 1)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("S,H", [(12, 50), (48, 256)])
@pytest.mark.parametrize("N", [33, 3072, 20001])
def test_actor_reads_16bit_as_its_float32_copy(S, H, N, dtype):
    """Both kernel builds (S <= 16 and S <= 64), injected eps and Philox noise, with the moments."""
    import marlnav_b200 as mb
    w = _actor_weights(S, H)
    g = torch.Generator().manual_seed(N)
    obs16 = (torch.rand(N, S, generator=g) * 2 - 1).to(dtype).cuda()
    eps = torch.randn(N, 2, generator=g).cuda()
    for e in (eps, None):
        got = mb.FusedActor(w, seed=5).act(obs16, eps=e, want_moments=True)
        want = mb.FusedActor(w, seed=5).act(obs16.float(), eps=e, want_moments=True)
        for name, a, b in zip(("actions", "log_probs", "mu", "var"), got, want):
            assert a.dtype == torch.float32
            assert_bits((e is None, name), a, b)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("K,H,B", [(36, 50, 1000),       # <= 2 048: 64 lanes per env
                                   (36, 50, 5000),       # 2 049 .. 32 768: 16 lanes per env
                                   (36, 64, 40001),      # 32 769 .. 262 144: 4 lanes per env
                                   (36, 50, 262145),     # > 262 144: thread per env
                                   (384, 50, 300)])      # weights over 48 KiB: thread per env
def test_critic_reads_16bit_as_its_float32_copy(K, H, B, dtype):
    import marlnav_b200 as mb
    g = torch.Generator().manual_seed(B)
    x16 = (torch.rand(B, K, generator=g) * 2 - 1).to(dtype).cuda()
    critic = mb.FusedCritic(_critic_weights(K, H))
    got, want = critic(x16), critic(x16.float())
    assert got.dtype == torch.float32 and got.shape == (B, 1)
    assert_bits("values", got, want)


ROLLOUT_KEYS = ('obs', 'last_obs', 'actions', 'log_probs', 'rewards', 'done')


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B,O,H", [(515, 3, 50), (40001, 3, 64), (64, 1, 7), (40001, 1, 50),
                                   (300, 4, 64), (40001, 4, 7), (33, 6, 50), (40000, 6, 64)])
def test_fused_actor_step_matches_two_launches_16bit(B, O, H, dtype):
    """Thread-per-agent (B <= 32 768) and thread-per-env kernels, ragged batches, resets.  At B = 515
    every odd obs_all[t] starts 8 bytes off a 16-byte boundary: the plain-store path."""
    import marlnav_b200 as mb
    A, T = 3, 40
    w = _actor_weights(_obs_size(A, O), H)
    bufs, envs = [], []
    for fuse in (True, False):
        env = _env(B, A, O, dtype, episode_len=15)
        fa = mb.FusedActor(w, seed=9)
        assert env.supports_fused_actor(fa)
        bufs.append(mb.collect_rollout(env, fa, T, fuse_actor=fuse, obs_dtype=dtype))
        envs.append(env)
    assert bufs[0]['obs'].dtype == dtype and bufs[0]['last_obs'].dtype == dtype
    for key in ROLLOUT_KEYS:
        assert_bits(key, bufs[0][key], bufs[1][key])
    assert bool(bufs[0]['done'].any())
    for name in ('states', 'obstacles', 'target', '_step_num', '_terminates_u8'):
        assert_bits(name, getattr(envs[0], name), getattr(envs[1], name))
    assert torch.equal(envs[0].episode_stats, envs[1].episode_stats)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B,A,O,fuse", [(515, 3, 3, True), (40001, 3, 3, True), (515, 3, 3, False),
                                        (300, 8, 16, True), (257, 5, 7, True)])
def test_16bit_rollout_is_the_rounded_float32_twin(B, A, O, fuse, dtype):
    """(8,16) and (5,7) have no fused actor kernel: the typed actor + step_fused route."""
    import marlnav_b200 as mb
    S, T = _obs_size(A, O), 30
    w = _actor_weights(S, 50)
    cw = _critic_weights(A * S)
    env = _env(B, A, O, dtype, episode_len=12)
    buf = mb.collect_rollout(env, mb.FusedActor(w, seed=3), T, critic=mb.FusedCritic(cw), fuse_actor=fuse,
                             obs_dtype=dtype)
    for key in ('actions', 'log_probs', 'rewards', 'values'):
        assert buf[key].dtype == torch.float32, key
    assert buf['obs'].dtype == dtype and buf['done'].dtype == torch.bool
    twin = _env(B, A, O, None, episode_len=12)
    mean, scale = twin._io_tensors[0], twin._io_tensors[1]
    fa, critic = mb.FusedActor(w, seed=3), mb.FusedCritic(cw)
    o32 = (twin.observations_fused() - mean) / scale
    for t in range(T):
        assert_rounded(("obs", t), buf['obs'][t], o32)
        act, lp = fa.act(buf['obs'][t].float())
        assert_bits(("actions", t), buf['actions'][t], act)
        assert_bits(("log_probs", t), buf['log_probs'][t], lp)
        assert_bits(("values", t), buf['values'][t], critic(buf['obs'][t].reshape(B, A * S).float()))
        o32, rew, term, trunc = twin.step_fused(buf['actions'][t].view(B, A, 2))
        assert_bits(("rewards", t), buf['rewards'][t], rew)
        assert torch.equal(buf['done'][t], term | trunc), t
    assert_rounded("last_obs", buf['last_obs'], o32)
    assert bool(buf['done'].any())
    torch.cuda.synchronize()
    for name in ('states', 'obstacles', 'target', '_step_num', '_terminates_u8'):
        assert_bits(name, getattr(env, name), getattr(twin, name))
    assert torch.equal(env.episode_stats, twin.episode_stats)


@pytest.mark.parametrize("dtype", DTYPES)
def test_rollout_graph_replays_equal_the_eager_16bit_rollouts(dtype):
    import marlnav_b200 as mb
    B, A, O, T = 256, 3, 3, 60
    w, cw = _actor_weights(), _critic_weights(A * 12)

    def make():
        return _env(B, A, O, dtype, seed=12, episode_len=25), mb.FusedActor(w, seed=3), mb.FusedCritic(cw)
    env_e, act_e, cri_e = make()
    mb.collect_rollout(env_e, act_e, 2, critic=cri_e, obs_dtype=dtype)          # RolloutGraph's warm-up
    eager = [mb.collect_rollout(env_e, act_e, T, critic=cri_e, obs_dtype=dtype) for _ in range(2)]
    env_g, act_g, cri_g = make()
    rg = mb.RolloutGraph(env_g, act_g, T, critic=cri_g, warmup_steps=2, obs_dtype=dtype)
    for k in range(2):
        buf = rg.replay()
        torch.cuda.synchronize()
        for key in ('obs', 'last_obs', 'actions', 'log_probs', 'rewards', 'done', 'values'):
            assert_bits((k, key), buf[key], eager[k][key])
    assert not torch.equal(eager[0]['actions'], eager[1]['actions'])
    assert torch.equal(env_g.states, env_e.states) and torch.equal(env_g.obstacles, env_e.obstacles)


@pytest.mark.parametrize("dtype", DTYPES)
def test_sharded_16bit_rollout_equals_single_process(dtype):
    import marlnav_b200 as mb
    B, A, O, T = 600, 3, 3, 60
    norm, scal = _io_params(A, O)
    w = _actor_weights(_obs_size(A, O), 50)
    full = _params(B, A, O, dtype, seed=8, episode_len=25)
    for fuse in (True, False):
        env = mb.Env(dict(full)); env.fuse_io(norm, scal)
        whole = mb.collect_rollout(env, mb.FusedActor(w, seed=13), T, fuse_actor=fuse, obs_dtype=dtype)
        parts = []
        for r in range(2):
            e = mb.Env(mb.shard_env_params(full, r, 2)); e.fuse_io(norm, scal)
            assert e.obs_dtype == dtype
            parts.append(mb.collect_rollout(e, mb.FusedActor(w, seed=13), T, fuse_actor=fuse, obs_dtype=dtype))
        for key in ('obs', 'actions', 'log_probs', 'rewards', 'done'):
            assert_bits((fuse, key), whole[key], torch.cat([p[key] for p in parts], dim=1))
        assert bool(whole['done'].any())


@pytest.mark.parametrize("dtype", DTYPES)
def test_mismatched_or_wrong_observation_buffers_are_refused(dtype):
    import marlnav_b200 as mb
    from marlnav_b200 import rollout
    B, A, O = 64, 3, 3
    S = _obs_size(A, O)
    other = torch.bfloat16 if dtype == torch.float16 else torch.float16
    w = _actor_weights(S, 50)
    e16, e32 = _env(B, A, O, dtype), _env(B, A, O)
    fa = mb.FusedActor(w, seed=1)
    assert e16.supports_fused_actor(fa) and e32.supports_fused_actor(fa)
    dev = 'cuda'

    def out(obs):
        return (torch.empty(B * A, 2, device=dev), torch.empty(B * A, device=dev), obs, torch.empty(B, device=dev),
                torch.empty(B, dtype=torch.uint8, device=dev), torch.empty(B, dtype=torch.uint8, device=dev))
    good_in, good_out = torch.zeros(B, A, S, dtype=dtype, device=dev), torch.empty(B, A, S, dtype=dtype, device=dev)
    # the requested dtype must be the env's, either way, and that is checked first
    for env, asked in ((e16, torch.float32), (e16, other), (e32, dtype)):
        pat = f"{asked}.*{env.obs_dtype}"
        with pytest.raises(mb.MarlnavError, match=pat):
            env.act_step_fused(fa, good_in, out(good_out), obs_dtype=asked)
        with pytest.raises(mb.MarlnavError, match=pat):
            rollout.collect_rollout(env, fa, 4, obs_dtype=asked)
        with pytest.raises(mb.MarlnavError, match=pat):
            rollout.RolloutGraph(env, fa, 4, obs_dtype=asked)
    # wrong-dtype or short buffers are refused, not overrun
    for name, obs_in, obs in (("obs_in", good_in.float(), good_out), ("obs_in", good_in.reshape(-1)[:-1], good_out),
                              ("obs_in", good_in.to(other), good_out),
                              ("out\\[2\\]", good_in, good_out.float()), ("out\\[2\\]", good_in, good_out.reshape(-1)[:-1])):
        with pytest.raises(mb.MarlnavError, match=name):
            e16.act_step_fused(fa, obs_in, out(obs), obs_dtype=dtype)
    a, lp, o, *_ = e16.act_step_fused(fa, good_in, out(good_out), obs_dtype=dtype)
    torch.cuda.synchronize()
    assert o.dtype == dtype and a.dtype == torch.float32 and bool(torch.isfinite(lp).all())
    # MappoRollout keeps handing the reference's learner float32 buffers
    with pytest.raises(mb.MarlnavError, match="float32"):
        rollout.MappoRollout(types.SimpleNamespace(env=e16))
