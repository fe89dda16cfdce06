"""The one-warp tile kernels visit their tiles in reverse order on every other step (the parity of
the step counter; it keeps the env state in L2 from one step to the next).  Results do not depend
on the order: every env's rows must be written on both parities, bit-identical to the C oracle,
for a ragged last tile, for misaligned base pointers and in a CUDA-graph replay of back-to-back
steps.  Outputs are filled with a sentinel before every step, so a tile skipped on one parity
cannot pass on the previous step's values."""
import numpy as np
import pytest
import torch

from helpers import action_pool, assert_bits_equal, cpu_params

pytestmark = pytest.mark.gpu

STEPS = 6          # three steps of each parity

# (B, A, O, envs per CTA): 32 k + 5 envs, so the last tile is ragged.  B above 32 768 runs the team
# of 3 through the thread-per-env kernel; smaller teams of 3 and the team of 8 thread per agent.
SHAPES = {"env_3x3": (32 * 1100 + 5, 3, 3, 32), "team_3x3": (32 * 40 + 5, 3, 3, 8),
          "team_8x16": (32 * 10 + 5, 8, 16, 4)}


def _params(B, A, O):
    import marlnav_b200 as mb
    kw = dict(episode_len=3)           # resets on both parities
    if A == 3:
        return mb.default_env_params(B, A, O, sampling_style='policy', **kw)
    return mb.template_env_params(B, A, O, **kw)


def _shifted(t):
    """Same values, storage one element past a 16-byte boundary (the kernels' non-TMA staging)."""
    flat = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)[1:]
    flat.copy_(t.reshape(-1))
    return flat.view(t.shape)


def _outputs(B, A, S, misaligned):
    obs = torch.empty(B * A * S + int(misaligned), device='cuda')[int(misaligned):].view(B, A, S)
    return obs, torch.empty(B, device='cuda'), torch.empty(B, dtype=torch.uint8, device='cuda'), \
        torch.empty(B, dtype=torch.uint8, device='cuda')


def _poison(out):
    out[0].fill_(float('nan')); out[1].fill_(float('nan')); out[2].fill_(0xAB); out[3].fill_(0xAB)


def _check(tag, out, want):
    o_obs, o_rew, o_term, o_trunc = want
    assert_bits_equal(f"{tag} obs", out[0].cpu().numpy(), o_obs)
    assert_bits_equal(f"{tag} rewards", out[1].cpu().numpy(), o_rew)
    assert_bits_equal(f"{tag} terminated", out[2].cpu().numpy(), o_term.astype(np.uint8))
    assert_bits_equal(f"{tag} truncated", out[3].cpu().numpy(), o_trunc.astype(np.uint8))


def _check_state(env, oe, tag):
    assert_bits_equal(f"{tag} states", env.states.cpu().numpy(), oe.states)
    assert_bits_equal(f"{tag} obstacles", env.obstacles.cpu().numpy(), oe.obstacles)
    assert_bits_equal(f"{tag} target", env.target.cpu().numpy().reshape(-1, 2), oe.target)
    assert_bits_equal(f"{tag} step_num", env._step_num.cpu().numpy(), oe.step_num)


@pytest.mark.parametrize("misaligned", [False, True], ids=["aligned", "misaligned"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_both_tile_orders_write_every_env(oracle, shape, misaligned):
    import marlnav_b200 as mb
    B, A, O, per_cta = SHAPES[shape]
    p = _params(B, A, O)
    env = mb.Env(dict(p, seed=21))
    assert env.launch_info()[3] == per_cta
    oe = oracle.OracleEnv(cpu_params(p), seed=21)
    if misaligned:
        env.states, env.obstacles, env.target = _shifted(env.states), _shifted(env.obstacles), _shifted(env.target)
        assert env.states.data_ptr() % 16 != 0
    out = _outputs(B, A, env.obs_size, misaligned)
    pool = action_pool(B, A, angle=0.3)
    done = 0
    for t in range(STEPS):
        act = pool[t % len(pool)]
        _poison(out)
        env.step_fused(act.cuda(), out=out)
        want = oe.step_fused(act.numpy())
        _check(f"{shape} step {t}", out, want)
        done += int((want[2] | want[3]).sum())
    _check_state(env, oe, f"{shape} final")
    assert done > 0


@pytest.mark.parametrize("shape", ["env_3x3", "team_8x16"])
def test_both_tile_orders_in_a_step_graph_replay(oracle, shape):
    """StepGraph passes the step's offset inside the captured batch as the host counter: consecutive
    captured steps alternate their tile order, and two replays continue the oracle's loop."""
    import marlnav_b200 as mb
    B, A, O, _ = SHAPES[shape]
    p = _params(B, A, O)
    env = mb.Env(dict(p, seed=33))
    oe = oracle.OracleEnv(cpu_params(p), seed=33)
    pool = action_pool(B, A, n=4, angle=0.3)
    acts = [a.cuda() for a in pool]
    sg = mb.StepGraph(env, acts, keep_outputs=True)
    torch.cuda.synchronize()
    oe.step_fused(pool[0].numpy())                         # StepGraph's warm-up step runs acts[0] once
    for rep in range(2):
        for out in sg.outputs:
            _poison(out)
        outs = sg.replay()
        torch.cuda.synchronize()
        for k, a in enumerate(pool):
            _check(f"{shape} replay {rep} step {k}", outs[k], oe.step_fused(a.numpy()))
    _check_state(env, oe, f"{shape} final")
