"""GPU: float16 / bfloat16 observations (params['obs_dtype']).  A 16-bit env and a float32 twin built
from the same params and seed, stepped with the same actions: the 16-bit observations are the float32
ones rounded to nearest-even (obs32.to(dtype), bit for bit, NaN positions equal), and everything else
-- states, obstacles, target, step counters, terminates, rewards, flags, episode stats -- is identical.
Shapes cover every kernel family and dispatch branch: thread-per-env and thread-per-agent team of 3,
(8,16), the generic kernel, ragged last warps, the normaliser / scaler, noisy resets, run-time
geometry constants, unaligned outputs, the host-stepping pipeline and CUDA-graph replays."""
import math
import types

import pytest
import torch

from helpers import action_pool

pytestmark = pytest.mark.gpu

DTYPES = [torch.float16, torch.bfloat16]
I16 = torch.int16


def _params(B, A, O, dtype=None, **kw):
    import marlnav_b200 as mb
    p = mb.default_env_params(B, A, O, sampling_style='policy', **kw) if A == 3 else \
        mb.template_env_params(B, A, O, **kw)
    p['seed'] = 11
    if dtype is not None:
        p['obs_dtype'] = dtype
    return p


def _twins(B, A, O, dtype, geometry=None, io=False, noisy=False, **kw):
    import marlnav_b200 as mb
    envs = []
    for d in (None, dtype):
        p = _params(B, A, O, d, **kw)
        if noisy:
            p['init']['noisy_ags'] = True
        e = mb.Env(p)
        for k, v in (geometry or {}).items():
            setattr(e._c_params, k, v)
        if io:
            e.fuse_io(*_io_params(A, O))
        envs.append(e)
    return envs


def _io_params(A, O):
    max_d = math.sqrt(1500.0 ** 2 + 750.0 ** 2)
    lo = [-math.pi, 0.] + O * [-math.pi] + O * [0.] + (A - 1) * [-math.pi] + (A - 1) * [0.]
    hi = [math.pi, max_d] + O * [math.pi] + O * [max_d] + (A - 1) * [math.pi] + (A - 1) * [max_d]
    return dict(min_obs=lo, max_obs=hi), dict(min_action=[-math.pi, -0.5], max_action=[math.pi, 0.5])


def assert_rounded(tag, o16, o32):
    """o16 == o32.to(dtype) bit for bit; NaN positions equal, payloads unspecified."""
    assert o16.dtype != torch.float32 and o16.shape == o32.shape, (tag, o16.dtype, o16.shape, o32.shape)
    want = o32.to(o16.dtype)
    same = (o16.view(I16) == want.view(I16)) | (torch.isnan(o16) & torch.isnan(want))
    if not bool(same.all()):
        idx = (~same).nonzero()[:5].tolist()
        raise AssertionError(f"{tag}: {int((~same).sum())} of {same.numel()} observations differ, e.g. "
                             f"{[(i, float(o16[tuple(i)]), float(o32[tuple(i)])) for i in idx]}")


def assert_same_state(tag, e16, e32):
    for name in ('states', 'obstacles', 'target', '_step_num'):
        a, b = getattr(e16, name), getattr(e32, name)
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (tag, name)
    assert torch.equal(e16._terminates_u8, e32._terminates_u8), (tag, 'terminates')
    assert torch.equal(e16.episode_stats, e32.episode_stats), (tag, 'stats')


def _run_twins(e32, e16, steps=30, scale=None):
    B, A = e32.num_parallel, e32.num_agents
    pool = [a.cuda() for a in action_pool(B, A, angle=0.3)]
    resets = 0
    for t in range(steps):
        act = pool[t % len(pool)]
        if scale is not None:
            act = act * scale
        o32, r32, te32, tr32 = e32.step_fused(act)
        o16, r16, te16, tr16 = e16.step_fused(act)
        assert_rounded(f"step {t}", o16, o32)
        assert torch.equal(r16.view(torch.int32), r32.view(torch.int32)), t
        assert torch.equal(te16, te32) and torch.equal(tr16, tr32), t
        resets += int((te32 | tr32).sum())
    torch.cuda.synchronize()
    assert_same_state("final", e16, e32)
    return resets


SHAPES = [
    (40000, 3, 3),    # thread-per-env
    (1000, 3, 3),     # team of 3, thread per agent
    (40000, 3, 1), (1000, 3, 1),
    (40000, 3, 6), (1000, 3, 6),
    (4096, 8, 16),    # team of 8
    (500, 5, 7), (300, 2, 1),                       # generic kernel
    (1, 3, 3), (31, 3, 3), (33, 3, 3), (20001, 3, 3), (40001, 3, 3), (33, 8, 16), (33, 5, 7),   # ragged
]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B,A,O", SHAPES)
def test_twin_envs_16bit_observations_are_rounded_float32(B, A, O, dtype):
    e32, e16 = _twins(B, A, O, dtype, episode_len=12)
    assert e16.obs_dtype == dtype and e32.obs_dtype == torch.float32
    resets = _run_twins(e32, e16)
    assert resets > 0


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B,A,O", [(40000, 3, 3), (1000, 3, 3), (4096, 8, 16), (500, 5, 7), (1000, 3, 6)])
def test_twin_envs_with_normalizer_and_scaler(B, A, O, dtype):
    """The value rounded is the normalised float32 value; actions go through the scaler."""
    e32, e16 = _twins(B, A, O, dtype, io=True, episode_len=12)
    assert _run_twins(e32, e16, scale=torch.tensor([0.1, 1.0], device='cuda')) > 0


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B", [40000, 1000])
def test_twin_envs_with_noisy_resets(B, dtype):
    e32, e16 = _twins(B, 3, 3, dtype, noisy=True, episode_len=12)
    assert _run_twins(e32, e16) > 0


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B,A,O", [(40000, 3, 3), (1000, 3, 3), (4096, 8, 16), (500, 5, 7)])
def test_twin_envs_with_custom_geometry(B, A, O, dtype):
    """Geometry constants that do not match the compiled-in division profile select the run-time-mode kernels."""
    geo = dict(init_dist=1234.5, max_at_prop_d=3.0, bond_sharpness=2.0)
    e32, e16 = _twins(B, A, O, dtype, geometry=geo, episode_len=12)
    assert _run_twins(e32, e16) > 0


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B,A,O", [(1000, 3, 3), (40000, 3, 3), (1000, 3, 1), (4096, 8, 16), (500, 5, 7), (33, 8, 16)])
def test_observations_are_rounded_float32(B, A, O, dtype):
    e32, e16 = _twins(B, A, O, dtype, episode_len=12)
    _run_twins(e32, e16, steps=5)
    f32, f16 = e32.observations_fused(), e16.observations_fused()
    S = e16.obs_size
    assert f16.dtype == dtype and f16.shape == (B, A, S)
    assert_rounded("observations_fused", f16, f32)
    fields16, fields32 = e16.observations(), e32.observations()
    assert type(fields16).__name__ == 'Observations'
    for a, b in zip(fields16, fields32):
        assert a.dtype == dtype and a.shape == b.shape
        assert_rounded("field", a, b)
    obs, rew, term, trunc = e16.step(action_pool(B, A, n=1)[0].cuda())
    assert all(f.dtype == dtype for f in obs) and obs.others_distances.shape == (B, A, A - 1)
    assert rew.dtype == torch.float32 and term.dtype == torch.bool and trunc.dtype == torch.bool


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B,A,O", [(40000, 3, 3), (1000, 3, 3), (4096, 8, 16), (500, 5, 7), (33, 3, 3)])
def test_unaligned_output_gives_the_same_bits(B, A, O, dtype):
    """step_fused(out=...) into buf[1:] (obs one element off a 16-byte boundary: plain 2-byte stores)
    equals the aligned output of a twin."""
    import marlnav_b200 as mb
    ea, eb = mb.Env(_params(B, A, O, dtype, episode_len=12)), mb.Env(_params(B, A, O, dtype, episode_len=12))
    S = ea.obs_size
    buf = torch.empty(B * A * S + 1, dtype=dtype, device='cuda')
    out = (buf[1:].view(B, A, S), torch.empty(B, device='cuda'), torch.empty(B, dtype=torch.uint8, device='cuda'),
           torch.empty(B, dtype=torch.uint8, device='cuda'))
    assert out[0].data_ptr() % 16 != 0
    pool = [a.cuda() for a in action_pool(B, A, angle=0.3)]
    for t in range(20):
        oa, ra, ta, tra = ea.step_fused(pool[t % len(pool)])
        ob, rb, tb, trb = eb.step_fused(pool[t % len(pool)], out=out)
        assert torch.equal(oa.view(I16), ob.view(I16)), t
        assert torch.equal(ra, rb) and torch.equal(ta, tb) and torch.equal(tra, trb), t
    assert_same_state("final", ea, eb)


@pytest.mark.parametrize("dtype", DTYPES)
def test_wrong_or_short_output_is_refused(dtype):
    import marlnav_b200 as mb
    B, A, O = 64, 3, 3
    e16 = mb.Env(_params(B, A, O, dtype))
    e32 = mb.Env(_params(B, A, O))
    S = e16.obs_size
    act = torch.zeros(B, A, 2, device='cuda')
    rest = (torch.empty(B, device='cuda'), torch.empty(B, dtype=torch.uint8, device='cuda'),
            torch.empty(B, dtype=torch.uint8, device='cuda'))
    with pytest.raises(mb.MarlnavError, match="out\\[0\\]"):
        e16.step_fused(act, out=(torch.empty(B, A, S, device='cuda'),) + rest)          # float32 buffer
    with pytest.raises(mb.MarlnavError, match="out\\[0\\]"):
        e16.step_fused(act, out=(torch.empty(B * A * S - 1, dtype=dtype, device='cuda'),) + rest)
    with pytest.raises(mb.MarlnavError, match="out\\[0\\]"):
        e32.step_fused(act, out=(torch.empty(B, A, S, dtype=dtype, device='cuda'),) + rest)
    with pytest.raises(mb.MarlnavError, match="obs_dtype"):
        mb.Env(_params(B, A, O, torch.float64))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B", [70001, 140001])
def test_host_stepper_equals_device_step(B, dtype):
    """Both chunking pipelines (2 chunks; 4 with the ramp-up chunks)."""
    import marlnav_b200 as mb
    A, O = 3, 3
    e_dev, e_host = mb.Env(_params(B, A, O, dtype, episode_len=12)), mb.Env(_params(B, A, O, dtype, episode_len=12))
    hs = mb.HostStepper(e_host)
    try:
        assert hs.obs_host.dtype == dtype and hs.obs_dev.dtype == dtype
        assert hs.d2h_bytes == B * A * e_host.obs_size * 2 + B * 4 + 2 * B
        pool = action_pool(B, A, angle=0.3)
        for t in range(14):
            act = pool[t % len(pool)]
            o, r, te, tr = e_dev.step_fused(act.cuda())
            hs.actions_host.copy_(act)
            hs.step()
            assert torch.equal(hs.obs_host.view(I16), o.cpu().view(I16)), t
            assert torch.equal(hs.rewards_host, r.cpu()), t
            assert torch.equal(hs.terminated_host.view(torch.bool), te.cpu()), t
            assert torch.equal(hs.truncated_host.view(torch.bool), tr.cpu()), t
        assert_same_state("final", e_host, e_dev)
    finally:
        hs.close()


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B", [1000, 40000])
def test_step_graph_replays_equal_the_eager_loop(B, dtype):
    import marlnav_b200 as mb
    p = _params(B, 3, 3, dtype, episode_len=25)
    pool = [a.cuda() for a in action_pool(B, 3, angle=0.3)]
    K = 2 * len(pool)
    acts = [pool[i % len(pool)] for i in range(K)]
    eager = mb.Env(dict(p))
    seq = [acts[0]] + acts + acts                         # StepGraph's warm-up step runs acts[0] once
    ref = [[t.clone() for t in eager.step_fused(a)] for a in seq]
    env = mb.Env(dict(p))
    sg = mb.StepGraph(env, acts, keep_outputs=True)
    for k in range(2):
        outs = sg.replay()
        torch.cuda.synchronize()
        for i in range(K):
            o, r, te, tr = outs[i]
            ro, rr, rte, rtr = ref[1 + k * K + i]
            assert o.dtype == dtype and torch.equal(o.view(I16), ro.view(I16)), (k, i)
            assert torch.equal(r, rr) and torch.equal(te.view(torch.bool), rte) and torch.equal(tr.view(torch.bool), rtr)
    assert torch.equal(env.states, eager.states) and torch.equal(env.obstacles, eager.obstacles)


@pytest.mark.parametrize("dtype", DTYPES)
def test_rollout_and_fused_actor_refuse_16bit_envs(dtype):
    import marlnav_b200 as mb
    from marlnav_b200 import rollout
    B, A, O = 64, 3, 3
    env = mb.Env(_params(B, A, O, dtype))
    env.fuse_io(*_io_params(A, O))
    assert env.supports_fused_actor(None) is False
    with pytest.raises(mb.MarlnavError, match="float32"):
        env.act_step_fused(None, None, None)
    with pytest.raises(mb.MarlnavError, match="float32"):
        rollout.collect_rollout(env, None, 4)
    with pytest.raises(mb.MarlnavError, match="float32"):
        rollout.RolloutGraph(env, None, 4)
    with pytest.raises(mb.MarlnavError, match="float32"):
        rollout.MappoRollout(types.SimpleNamespace(env=env))
