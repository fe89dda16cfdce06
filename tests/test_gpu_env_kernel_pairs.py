"""GPU: the thread-per-env kernel (team of 3, more than 32 768 envs) evaluates every agent pair once
and gives both agents its distance and the opposite unit vector.  Scenes built so that agent-agent
distances straddle ag_coll_dist, ag_risk_dist, agents_min_d, agents_max_d and cap_distance, and so
that some envs have agents with an exactly zero x or y component between them (the guarded
re-evaluation of the env), stepped against the C oracle bit for bit: observations (float32 /
float16 / bfloat16, with and without the fused normaliser), rewards, flags and final observations."""
import math

import numpy as np
import pytest
import torch

from helpers import cpu_params

pytestmark = pytest.mark.gpu

B = 33000                      # > 32 768: thread per env; 33 000 = 1031 * 32 + 8, a ragged last warp
THRESHOLDS = ('ag_coll_dist', 'ag_risk_dist', 'agents_min_d', 'agents_max_d', 'cap_distance')
INT_OF = {2: torch.int16, 4: torch.int32}


def bits(t):
    return t.contiguous().view(INT_OF[t.element_size()])


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle as o
    o.lib()
    return o


def _io_params(A, O):
    max_d = math.sqrt(1500.0 ** 2 + 750.0 ** 2)
    lo = [-math.pi, 0.] + O * [-math.pi] + O * [0.] + (A - 1) * [-math.pi] + (A - 1) * [0.]
    hi = [math.pi, max_d] + O * [math.pi] + O * [max_d] + (A - 1) * [math.pi] + (A - 1) * [max_d]
    return dict(min_obs=lo, max_obs=hi), dict(min_action=[-math.pi, -0.5], max_action=[math.pi, 0.5])


def _scene(states, p, rng):
    """Agents 1 and 2 placed around agent 0 at distances just below / above the pair thresholds.
    Each env's agents share heading, speed and action, so that the move keeps their offsets (up to
    rounding).  Envs 0, 9, 18, ...: agent 1 straight above or below agent 0 (zero x component),
    headings (0, +-1); envs 1, 10, ...: agent 2 level with agent 0 (zero y component), headings
    (+-1, 0); those envs turn by exactly 0 so the component stays zero."""
    st = states.copy()
    n = st.shape[0]
    th = np.array([getattr(p, k) for k in THRESHOLDS], np.float64)
    pick = rng.integers(0, len(th), size=(n, 2))
    width = np.maximum(0.5 * th[pick], 0.02) * 0.2
    dist = th[pick] + rng.uniform(-1.0, 1.0, size=(n, 2)) * width
    ang = rng.uniform(-math.pi, math.pi, size=(n, 2))
    hd = rng.uniform(-math.pi, math.pi, size=n)
    head = np.stack([np.cos(hd), np.sin(hd)], 1)
    x_al, y_al = np.arange(n) % 9 == 0, np.arange(n) % 9 == 1
    ang[x_al, 0] = np.where(rng.random(x_al.sum()) < 0.5, 0.5, -0.5) * math.pi
    ang[y_al, 1] = np.where(rng.random(y_al.sum()) < 0.5, 0.0, 1.0) * math.pi
    sgn = np.where(rng.random(n) < 0.5, 1.0, -1.0)
    head[x_al] = np.stack([np.zeros(x_al.sum()), sgn[x_al]], 1)
    head[y_al] = np.stack([sgn[y_al], np.zeros(y_al.sum())], 1)
    base = st[:, 0, :2].astype(np.float64)
    for k in (1, 2):
        st[:, k, 0] = (base[:, 0] + dist[:, k - 1] * np.cos(ang[:, k - 1])).astype(np.float32)
        st[:, k, 1] = (base[:, 1] + dist[:, k - 1] * np.sin(ang[:, k - 1])).astype(np.float32)
    st[x_al, 1, 0] = st[x_al, 0, 0]
    st[y_al, 2, 1] = st[y_al, 0, 1]
    st[:, :, 2:4] = head.astype(np.float32)[:, None, :]
    st[:, :, 4] = rng.uniform(3.0, 10.0, size=n).astype(np.float32)[:, None]
    return st, x_al | y_al


@pytest.mark.parametrize("final", [False, True])
@pytest.mark.parametrize("io", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("O", [1, 2, 3, 4, 5, 6])
def test_shared_agent_pairs_equal_the_oracle(orc, O, dtype, io, final):
    import marlnav_b200 as mb
    A, steps = 3, 4
    params = mb.default_env_params(B, A, O, sampling_style='policy', episode_len=3)
    params['seed'], params['obs_dtype'] = 7 + O, dtype
    env = mb.Env(dict(params))
    oe = orc.OracleEnv(cpu_params(params), seed=7 + O)
    S = env.obs_size
    rng = np.random.default_rng(100 * O + 3)
    st, aligned = _scene(env.states.cpu().numpy(), env._c_params, rng)
    env.states.copy_(torch.from_numpy(st))
    oe.states[...] = st
    io_np = None
    if io:
        norm, scal = _io_params(A, O)
        env.fuse_io(norm, scal)
        lo, hi = torch.tensor(norm['min_obs']), torch.tensor(norm['max_obs'])
        io_np = ((0.5 * (lo + hi)).numpy(), (0.5 * (hi - lo)).numpy())
        a_lo, a_hi = torch.tensor(scal['min_action']), torch.tensor(scal['max_action'])
        a_scale, a_mean = (0.5 * (a_hi - a_lo)).numpy(), (0.5 * (a_lo + a_hi)).numpy()

    def want(o):
        if io_np is not None:
            o = ((o - io_np[0]).astype(np.float32) / io_np[1]).astype(np.float32)
        return torch.from_numpy(o).to(dtype)

    fin = torch.empty(B, A, S, dtype=dtype, device='cuda') if final else None
    checked = 0
    for t in range(steps):
        act = np.empty((B, A, 2), np.float32)
        act[:, :, 0] = rng.uniform(-0.2, 0.2, size=B).astype(np.float32)[:, None]
        act[:, :, 1] = rng.uniform(-0.5, 0.5, size=B).astype(np.float32)[:, None]
        act[aligned, :, 0] = 0.0
        if io:
            act[:, :, 0] /= np.float32(math.pi)         # the scaler maps it back (its mean is 0)
            act[aligned, :, 0] = 0.0
        o_act = ((a_scale * act).astype(np.float32) + a_mean) if io else act
        obs, rew, term, trunc = env.step_fused(torch.from_numpy(act).cuda(), final_obs=fin)
        o_obs, o_rew, o_term, o_trunc, o_pre = oe.step_fused(o_act, want_pre=True)
        if t == 0:
            assert env.launch_info()[3] == 32                    # the thread-per-env kernel
            d = o_pre[:, :, 2 + 2 * O + (A - 1):].reshape(-1)
            for k in THRESHOLDS:
                v = getattr(env._c_params, k)
                near = d[np.abs(d - v) < max(0.2 * v, 0.02)]
                assert (near < v).any() and (near > v).any(), k
            # (envs this step finished were reset to the template and are left out)
            s = oe.states[aligned & ~(o_term | o_trunc)]
            assert len(s) > 1000 and ((s[:, 0, 0] == s[:, 1, 0]) | (s[:, 0, 1] == s[:, 2, 1])).all()
        tag = f"O={O} step {t}"
        assert np.array_equal(term.cpu().numpy(), o_term) and np.array_equal(trunc.cpu().numpy(), o_trunc), tag
        assert np.array_equal(rew.cpu().numpy().view(np.uint32), o_rew.view(np.uint32)), tag
        assert torch.equal(bits(obs.cpu()), bits(want(o_obs))), tag
        if final:
            done = torch.from_numpy(o_term | o_trunc)
            assert torch.equal(bits(fin.cpu()[done]), bits(want(o_pre)[done])), tag
            checked += int(done.sum())
    assert not final or checked > 0
