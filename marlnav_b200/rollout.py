"""Caller-side pieces around the fused step (SURVEY.md section 8(f)-2 and 8(f)-3).

* ``FusedActor``          -- the reference's ``Actor.forward`` + ``dist.sample()`` +
                             ``dist.log_prob()`` (/root/reference/marlnav/models.py:27-36,113-115)
                             as one kernel launch (``marlnav_actor_sample_typed``).
* ``discounted_returns``  -- the backward scan of ``MAPPO._process_rewards``
                             (models.py:131-139) as one kernel (``marlnav_discounted_returns_f64``),
                             optionally followed by its std/mean normalisation (models.py:141-145).
* ``gae``                 -- generalised advantage estimation that bootstraps time-limit truncations
                             from the final observations' values (``marlnav_gae_f64``).
* ``collect_rollout``     -- ``MAPPO.get_data`` (models.py:106-129) with device-resident (T, ...)
                             buffers instead of a Python list of lists: per step one actor launch and
                             one fused environment step (normaliser and action scaler folded in); the
                             observation buffer in the env's ``obs_dtype`` when the caller opts in.

The reference's learner itself (PPO losses, Adam) is out of scope and stays stock PyTorch; these
functions hand it tensors in the layouts it already uses.
"""
import ctypes

import torch

from . import _lib
from .env import OBS_DTYPES


def _rollout_check(rc, what):
    if rc != 0:
        msg = _lib.load().marlnav_rollout_last_error().decode(errors="replace")
        raise _lib.MarlnavError(f"{what} failed (code {rc}): {msg}")


class FusedActor:
    """Inference-side twin of the reference ``Actor`` (models.py:14-36): takes its weights
    (``fc1``, ``fc_mu``, ``fc_std``) and samples actions + log-probs in one launch."""

    def __init__(self, actor, device='cuda', seed=None, row_offset=None):
        """``row_offset``: global index of this process's first (env, agent) row -- the sampling noise
        is addressed by GLOBAL row, so N ranks stepping N slices draw what one process would.  Left
        at None, ``collect_rollout`` / ``Env.act_step_fused`` use the env's ``env_id_offset * A``."""
        self._lib = _lib.load()
        self.row_offset = row_offset
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise _lib.MarlnavError("FusedActor needs a CUDA device (no CPU fallback)")
        self.seed = int(torch.initial_seed() if seed is None else seed) & 0xFFFFFFFFFFFFFFFF
        self.counter = 0
        self._counter_dev = None
        self._counter_batch = False        # see Env.batch_device_counter
        self._counter_pending = 0
        self.w1 = None
        self.refresh(actor)

    def refresh(self, actor):
        """(Re-)read the weights, e.g. after optimiser steps.  ``actor`` is the reference's
        ``Actor`` module or its ``state_dict()``."""
        sd = actor if isinstance(actor, dict) else actor.state_dict()
        g = lambda k: sd[k].detach().to(device=self.device, dtype=torch.float32).contiguous()
        new = [g(k) for k in ('fc1.weight', 'fc1.bias', 'fc_mu.weight', 'fc_mu.bias', 'fc_std.weight', 'fc_std.bias')]
        if self.w1 is not None and all(o.shape == n.shape for o, n in zip(self._weights(), new)):
            for o, n in zip(self._weights(), new):       # in place: captured CUDA graphs keep pointing here
                o.copy_(n)
        else:
            self.w1, self.b1, self.w_mu, self.b_mu, self.w_std, self.b_std = new
        self.hidden, self.obs_size = self.w1.shape
        if self.w_mu.shape != (2, self.hidden) or self.w_std.shape != (2, self.hidden):
            raise _lib.MarlnavError("unexpected Actor head shapes (need 2 outputs)")

    def _weights(self):
        return [self.w1, self.b1, self.w_mu, self.b_mu, self.w_std, self.b_std]

    def use_device_counter(self, enable=True):
        """Keep the sampling counter in device memory so that CUDA-graph replays draw fresh noise."""
        if enable and self._counter_dev is None:
            self._counter_dev = torch.full((1,), self.counter, dtype=torch.int64, device=self.device)
        elif not enable and self._counter_dev is not None:
            self.batch_device_counter(False)
            self.counter = int(self._counter_dev.item())
            self._counter_dev = None

    def _advance_counter(self, stream):
        """The ``counter`` argument for the launch being made (ABI 3: the kernels add the device word)."""
        self.counter += 1
        if self._counter_dev is None:
            return self.counter
        if self._counter_batch:
            self._counter_pending += 1
            return self._counter_pending
        self._lib.marlnav_counter_add(self._counter_dev.data_ptr(), 1, stream)
        return 0

    def spec(self, counter):
        """``marlnav_actor_spec`` of this actor for one fused {actor -> step} launch."""
        sp = _lib.ActorSpec()
        sp.w1, sp.b1 = self.w1.data_ptr(), self.b1.data_ptr()
        sp.w_mu, sp.b_mu = self.w_mu.data_ptr(), self.b_mu.data_ptr()
        sp.w_std, sp.b_std = self.w_std.data_ptr(), self.b_std.data_ptr()
        sp.S, sp.H, sp.seed, sp.counter = self.obs_size, self.hidden, self.seed, counter
        sp.counter_dev = self._counter_dev.data_ptr() if self._counter_dev is not None else None
        sp.row_offset = int(self.row_offset or 0)
        return sp

    def batch_device_counter(self, enable=True):
        """Batch mode of the device-resident sampling counter (see ``Env.batch_device_counter``)."""
        if not enable:
            self.flush_device_counter()
        self._counter_batch = bool(enable) and self._counter_dev is not None

    def flush_device_counter(self):
        if self._counter_dev is not None and self._counter_pending:
            self._lib.marlnav_counter_add(self._counter_dev.data_ptr(), self._counter_pending,
                                          torch.cuda.current_stream(self.device).cuda_stream)
        self._counter_pending = 0

    def act(self, obs, eps=None, want_moments=False, out=None, row_offset=None):
        """``obs``: normalised observations (..., obs_size) on the device (e.g. the fused (B,A,S)
        buffer).  Returns ``(actions (N,2), log_probs (N,))`` with N = prod(leading dims), exactly
        what models.py:113-115 produces; ``eps`` (N,2) injects the normal draws (tests); ``out`` =
        preallocated contiguous ``(actions, log_probs)`` tensors to write into; ``row_offset``
        overrides ``self.row_offset`` for this call.  float16 / bfloat16 ``obs`` are read as they
        are and widened exactly in the kernel: the same bits as ``act(obs.float())``.  Other dtypes
        are converted to float32 first.  The outputs are float32."""
        if row_offset is None:
            row_offset = self.row_offset or 0
        x = obs.reshape(-1, self.obs_size)
        code = OBS_DTYPES.get(x.dtype, 0)
        dtype = x.dtype if code else torch.float32
        if x.dtype != dtype or not x.is_contiguous() or x.device != self.device:
            x = x.to(device=self.device, dtype=dtype).contiguous()
        n = x.shape[0]
        with torch.cuda.device(self.device):
            if out is not None:
                actions, log_probs = out
            else:
                actions = torch.empty(n, 2, device=self.device)
                log_probs = torch.empty(n, device=self.device)
            mu = torch.empty(n, 2, device=self.device) if want_moments else None
            var = torch.empty(n, 2, device=self.device) if want_moments else None
            if eps is not None:
                eps = eps.to(device=self.device, dtype=torch.float32).contiguous()
            p = lambda t: t.data_ptr() if t is not None else None
            stream = torch.cuda.current_stream(self.device).cuda_stream
            counter = self._advance_counter(stream)
            args = (n, self.obs_size, self.hidden, p(self.w1), p(self.b1), p(self.w_mu), p(self.b_mu),
                    p(self.w_std), p(self.b_std), p(eps), self.seed, counter, p(self._counter_dev), int(row_offset),
                    p(actions), p(log_probs), p(mu), p(var), stream)
            _rollout_check(self._lib.marlnav_actor_sample_typed(p(x), code, *args), "marlnav_actor_sample_typed")
        return (actions, log_probs, mu, var) if want_moments else (actions, log_probs)


class FusedCritic:
    """Inference-side twin of the reference ``Critic`` (models.py:39-56): one launch per batch."""

    def __init__(self, critic, device='cuda'):
        self._lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise _lib.MarlnavError("FusedCritic needs a CUDA device (no CPU fallback)")
        self.refresh(critic)

    def refresh(self, critic):
        sd = critic if isinstance(critic, dict) else critic.state_dict()
        g = lambda k: sd[k].detach().to(device=self.device, dtype=torch.float32).contiguous()
        new = [g('fc1.weight'), g('fc1.bias'), g('fc2.weight'), g('fc2.bias')]
        old = getattr(self, 'w1', None)
        if old is not None and all(o.shape == n.shape for o, n in zip([self.w1, self.b1, self.w2, self.b2], new)):
            for o, n in zip([self.w1, self.b1, self.w2, self.b2], new):     # in place (CUDA graphs)
                o.copy_(n)
        else:
            self.w1, self.b1, self.w2, self.b2 = new
        self.hidden, self.inputs = self.w1.shape

    def __call__(self, obs, out=None):
        """``obs``: (B, ...) normalised observations with prod(...) == inputs.  Returns (B,1) float32.
        float16 / bfloat16 ``obs`` are read as they are and widened exactly in the kernel: the same
        bits as ``self(obs.float())``.  Other dtypes are converted to float32 first."""
        x = obs.reshape(obs.shape[0], -1)
        if x.shape[1] != self.inputs:
            raise _lib.MarlnavError(f"critic expects {self.inputs} inputs per env, got {x.shape[1]}")
        code = OBS_DTYPES.get(x.dtype, 0)
        dtype = x.dtype if code else torch.float32
        if x.dtype != dtype or not x.is_contiguous() or x.device != self.device:
            x = x.to(device=self.device, dtype=dtype).contiguous()
        with torch.cuda.device(self.device):
            v = out if out is not None else torch.empty(x.shape[0], 1, device=self.device)
            args = (x.shape[0], self.inputs, self.hidden, self.w1.data_ptr(), self.b1.data_ptr(),
                    self.w2.data_ptr(), self.b2.data_ptr(), v.data_ptr(),
                    torch.cuda.current_stream(self.device).cuda_stream)
            _rollout_check(self._lib.marlnav_critic_value_typed(x.data_ptr(), code, *args), "marlnav_critic_value_typed")
        return v


_CRITIC_STREAMS = {}


def _critic_stream(dev):
    key = (dev.type, dev.index)
    if key not in _CRITIC_STREAMS:
        _CRITIC_STREAMS[key] = torch.cuda.Stream(device=dev)
    return _CRITIC_STREAMS[key]


def discounted_returns(rewards, done, gamma, normalize=False):
    """models.py:131-139: ``curr = where(done, 0, rew + gamma*curr)`` backwards over the buffer, in
    float64 like the reference.  ``rewards`` (T,B) float32, ``done`` (T,B) bool/uint8, on the device.
    ``normalize=True`` also applies models.py:141-145: ``(x - mean) / (std + 1e-12)`` over the buffer."""
    lib = _lib.load()
    if rewards.device.type != 'cuda':
        raise _lib.MarlnavError("discounted_returns needs CUDA tensors (no CPU fallback)")
    T, B = rewards.shape
    rewards = rewards.to(torch.float32).contiguous()
    done_u8 = (done.view(torch.uint8) if done.dtype == torch.bool else done.to(torch.uint8)).contiguous()
    with torch.cuda.device(rewards.device):
        out = torch.empty(T, B, dtype=torch.float64, device=rewards.device)
        _rollout_check(lib.marlnav_discounted_returns_f64(
            rewards.data_ptr(), done_u8.data_ptr(), float(gamma), int(T), int(B), out.data_ptr(),
            torch.cuda.current_stream(rewards.device).cuda_stream), "marlnav_discounted_returns_f64")
        if normalize:
            std, mean = torch.std_mean(out.reshape(-1))
            out = (out - mean) / (std + 1e-12)
    return out


def gae(rewards, values, terminated, truncated, gamma, lam, final_values=None, last_values=None):
    """Generalised advantage estimation that tells a time-limit truncation from a termination, as one
    kernel (``marlnav_gae_f64``).  Returns ``(advantages, returns)``, both (T,B) float64.

    ``rewards``, ``values`` (T,B) float32 (``values`` may be (T,B,1), e.g. ``collect_rollout``'s);
    ``terminated``, ``truncated`` (T,B) bool/uint8; ``final_values`` (T,B) or (T,B,1): the value of the
    observation an episode was cut off on (``collect_rollout(final_obs=True)``'s), read where
    ``truncated & ~terminated`` (None: 0); ``last_values`` (B,) or (B,1): the value of the state after
    the last step (None: 0).  Backwards over t, per env, with ``gl = gamma * lam``::

        nv = last_values if t == T-1 else values[t+1]
        terminated: nv = 0, cont = 0;  truncated: nv = final_values[t], cont = 0;  else cont = 1
        delta = (r + gamma*nv) - v;  adv = delta + gl*adv_next if cont else delta;  ret = adv + v

    Every operation is a float64 operation rounded to nearest, without fused multiply-adds."""
    lib = _lib.load()
    if rewards.device.type != 'cuda':
        raise _lib.MarlnavError("gae needs CUDA tensors (no CPU fallback)")
    if rewards.dim() != 2:
        raise _lib.MarlnavError(f"gae: rewards must be (T,B), got {tuple(rewards.shape)}")
    T, B = rewards.shape
    dev = rewards.device

    def f32(t, n, name):
        if t.numel() != n:
            raise _lib.MarlnavError(f"gae: {name} must hold {n} values (T = {T}, B = {B}), got {tuple(t.shape)}")
        return t.to(device=dev, dtype=torch.float32).reshape(-1).contiguous()

    def u8(t, name):
        if tuple(t.shape) != (T, B):
            raise _lib.MarlnavError(f"gae: {name} must be (T,B) = ({T}, {B}), got {tuple(t.shape)}")
        t = t.to(dev)
        return (t.view(torch.uint8) if t.dtype == torch.bool else (t != 0).to(torch.uint8)).contiguous()

    r, v = f32(rewards, T * B, 'rewards'), f32(values, T * B, 'values')
    te, tr = u8(terminated, 'terminated'), u8(truncated, 'truncated')
    fv = f32(final_values, T * B, 'final_values') if final_values is not None else None
    lv = f32(last_values, B, 'last_values') if last_values is not None else None
    p = lambda t: t.data_ptr() if t is not None else None
    with torch.cuda.device(dev):
        adv = torch.empty(T, B, dtype=torch.float64, device=dev)
        ret = torch.empty(T, B, dtype=torch.float64, device=dev)
        _rollout_check(lib.marlnav_gae_f64(p(r), p(v), p(te), p(tr), p(fv), p(lv), float(gamma), float(lam),
                                           int(T), int(B), p(adv), p(ret), torch.cuda.current_stream(dev).cuda_stream),
                       "marlnav_gae_f64")
    return adv, ret


def _require_obs_dtype(env, obs_dtype, what):
    """A rollout's observation buffer has the type the caller asked for, and it must be the env's: a
    16-bit buffer goes to a learner, whose float32 layers refuse it unless it casts, so a 16-bit env
    never hands one out unasked."""
    if obs_dtype != env.obs_dtype:
        raise _lib.MarlnavError(f"{what}: obs_dtype {obs_dtype} does not match the env's obs_dtype {env.obs_dtype} "
                                f"(pass obs_dtype={env.obs_dtype} for a buffer of that type)")


def _require_f32_obs(env, what):
    """MappoRollout hands its buffer to the reference's float32 learner."""
    if env.obs_dtype != torch.float32:
        raise _lib.MarlnavError(f"{what} needs an env with float32 observations; this env's obs_dtype is "
                                f"{env.obs_dtype}")


@torch.no_grad()
def collect_rollout(env, actor, buffer_len, critic=None, normalizer_params=None, scaler_params=None,
                    fuse_actor=True, obs_dtype=torch.float32, final_obs=False):
    """``MAPPO.get_data`` (models.py:106-129) on device-resident buffers.

    ``env``: a ``marlnav_b200.Env``; ``actor``: a ``FusedActor``; ``critic``: optional ``FusedCritic``
    or torch module taking (B, A*S) normalised observations (the reference's ``Critic``).  The env must have its
    normaliser / action scaler fused in (``env.fuse_io``); pass the reference's ``normalizer`` /
    ``scaler`` param dicts here to do that.  Returns a dict of tensors with a leading time axis:
    ``obs (T,B,A,S)``, ``actions (T,B*A,2)``, ``log_probs (T,B*A)``, ``rewards (T,B)``, ``done (T,B)``
    and ``values (T,B,1)`` when a critic is given.

    ``fuse_actor``: sample the actions inside the step launch (``marlnav_act_step_typed``: one launch
    per iteration instead of two) where that kernel exists -- 3 agents, 1..6 obstacles; same bits
    either way (``test_fused_actor_step_matches_two_launches``).

    ``obs_dtype``: the element type of ``obs`` and ``last_obs``; it must equal ``env.obs_dtype``.
    With ``torch.float16`` / ``torch.bfloat16`` every stored observation is the normalised float32
    value rounded to nearest-even (``obs32.to(obs_dtype)``), and the actor and a ``FusedCritic`` read
    those values widened exactly to float32; a torch-module critic gets ``obs.float()``.  Every other
    buffer stays float32 (``done``: bool).  Cast learner minibatches with ``.float()``.

    ``final_obs=True`` also returns, for a learner that bootstraps time-limit truncations (``gae``):
    ``final_obs (T,B,A,S)`` in ``obs_dtype``, where row ``[t,b]`` holds the observations env b's episode
    ended on at step t (valid where ``done[t,b]``, unspecified elsewhere), ``terminated`` and
    ``truncated`` (T,B) bool, and with a ``FusedCritic`` ``final_values (T,B,1)``, the critic on every
    ``final_obs`` row in one launch after the loop.  The fused actor+step kernels have no final
    observations, so this mode runs the actor and ``step_fused`` as two launches per step, with the
    same actions and outputs."""
    _require_obs_dtype(env, obs_dtype, "collect_rollout")
    if normalizer_params is not None or scaler_params is not None:
        env.fuse_io(normalizer_params, scaler_params)
    if env._io is None or not env._io.obs_mean or not env._io.act_scale:
        raise _lib.MarlnavError("collect_rollout needs env.fuse_io(normalizer, scaler) first")
    B, A, S, T = env.num_parallel, env.num_agents, env.obs_size, int(buffer_len)
    dev = env.device
    mean, scale = env._io_tensors[0], env._io_tensors[1]
    # every kernel writes straight into its slice of the buffers: one launch per step on the main
    # stream (two where there is no fused actor kernel), the critic beside it
    obs_all = torch.empty(T + 1, B, A, S, dtype=obs_dtype, device=dev)
    term = torch.empty(T, B, dtype=torch.uint8, device=dev)
    trunc = torch.empty(T, B, dtype=torch.uint8, device=dev)
    buf = dict(actions=torch.empty(T, B * A, 2, device=dev), log_probs=torch.empty(T, B * A, device=dev),
               rewards=torch.empty(T, B, device=dev))
    if critic is not None:
        buf['values'] = torch.empty(T, B, 1, device=dev)
    fin = torch.empty(T, B, A, S, dtype=obs_dtype, device=dev) if final_obs else None
    # models.py:110; a 16-bit buffer receives the float32 quotient rounded to nearest-even
    torch.div(env._observations_f32() - mean, scale, out=obs_all[0])
    # device-resident counters: each step passes its offset, ONE add per counter after the loop
    env.batch_device_counter(True)
    actor.batch_device_counter(True)
    # The critic only reads obs_all[t] and writes values[t]: it runs on a forked stream, off the
    # actor -> step critical path (in a captured graph: a parallel branch joined at the end).
    main = torch.cuda.current_stream(dev)
    side = _critic_stream(dev) if isinstance(critic, FusedCritic) else None
    fused = bool(fuse_actor) and not final_obs and env.supports_fused_actor(actor)
    try:
        for t in range(T):
            obs = obs_all[t]
            if side is not None:
                ready = torch.cuda.Event()
                ready.record(main)                                              # obs_all[t] is complete
                side.wait_event(ready)
                with torch.cuda.stream(side):
                    critic(obs.view(B, A * S), out=buf['values'][t])            # models.py:120
            if critic is not None and side is None:
                buf['values'][t].copy_(critic(obs.view(B, A * S).float()))
            if fused:
                # models.py:113-118,122 in one launch: sample from obs, scale, step, normalise
                env.act_step_fused(actor, obs, out=(buf['actions'][t], buf['log_probs'][t], obs_all[t + 1],
                                                    buf['rewards'][t], term[t], trunc[t]), obs_dtype=obs_dtype)
                continue
            actions, _ = actor.act(obs, out=(buf['actions'][t], buf['log_probs'][t]),     # models.py:113-115
                                   row_offset=actor.row_offset if actor.row_offset is not None else env._env_id_offset * A)
            # raw [-1,1] actions in, normalised next observations out (models.py:116-118,122)
            env.step_fused(actions.view(B, A, 2), out=(obs_all[t + 1], buf['rewards'][t], term[t], trunc[t]),
                           final_obs=None if fin is None else fin[t])
    finally:
        if side is not None:
            main.wait_stream(side)
        env.batch_device_counter(False)             # (adds the pending totals to the device words)
        actor.batch_device_counter(False)
    buf['obs'] = obs_all[:T]
    buf['last_obs'] = obs_all[T]
    buf['done'] = torch.logical_or(term.view(torch.bool), trunc.view(torch.bool))   # models.py:119
    if fin is not None:
        buf['final_obs'] = fin
        buf['terminated'], buf['truncated'] = term.view(torch.bool), trunc.view(torch.bool)
        if isinstance(critic, FusedCritic):
            buf['final_values'] = torch.empty(T, B, 1, device=dev)
            critic(fin.view(T * B, A * S), out=buf['final_values'].view(T * B, 1))
    return buf


class RolloutGraph:
    """``collect_rollout`` captured once in a CUDA graph (SURVEY.md section 8(f)-4): a rollout of
    ``buffer_len`` steps becomes one graph launch.  The environment's reset counter and the actor's
    sampling counter live in device memory, so every replay continues the same random streams an
    eager loop would use; ``FusedActor.refresh`` / ``FusedCritic.refresh`` update weights in place.
    ``replay()`` returns the SAME buffer tensors every time (clone what must outlive the next replay).
    ``obs_dtype`` and ``final_obs``: as in ``collect_rollout``."""

    def __init__(self, env, actor, buffer_len, critic=None, warmup_steps=2, obs_dtype=torch.float32,
                 final_obs=False):
        _require_obs_dtype(env, obs_dtype, "RolloutGraph")
        if critic is not None and not isinstance(critic, FusedCritic):
            raise _lib.MarlnavError("RolloutGraph needs a FusedCritic (or no critic)")
        self.env, self.actor, self.critic, self.buffer_len = env, actor, critic, int(buffer_len)
        env.use_device_counter(True)
        actor.use_device_counter(True)
        dev = env.device
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            if warmup_steps:                                  # lazy kernel attributes, allocator warm-up
                collect_rollout(env, actor, warmup_steps, critic=critic, obs_dtype=obs_dtype, final_obs=final_obs)
            side.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=side):
                self.buffers = collect_rollout(env, actor, self.buffer_len, critic=critic, obs_dtype=obs_dtype,
                                               final_obs=final_obs)
        torch.cuda.current_stream(dev).wait_stream(side)

    def replay(self):
        self.graph.replay()
        return self.buffers


class StepGraph:
    """``len(actions)`` back-to-back fused steps captured in ONE CUDA graph (SURVEY.md section 8(e):
    a rank that owns 1/8 of the batch steps it in ~12 us, less than a ctypes call + launch from
    Python, so an eager loop is bound by the host).  The reset counter lives in device memory in
    batch mode -- the captured steps pass their offset 1..K and the word is bumped once per replay --
    so every replay draws the reset positions an eager loop would draw
    (``test_cuda_graph_of_back_to_back_steps_matches_eager``).

    ``actions``: a list of (B,A,2) device tensors (or one (K,B,A,2) tensor); they are read at
    replay time, so a policy can refill them between replays.  ``keep_outputs=True`` gives every
    step its own (obs, rewards, terminated, truncated) buffers (``.outputs[k]``); otherwise the K
    steps write into one set (``.outputs[0]`` holds the last step's results)."""

    def __init__(self, env, actions, keep_outputs=False):
        self.env = env
        self.actions = list(actions)
        K = len(self.actions)
        if K < 1:
            raise _lib.MarlnavError("StepGraph needs at least one action tensor")
        dev = env.device
        env.use_device_counter(True)
        n_out = K if keep_outputs else 1
        self.outputs = [env._alloc_outputs() for _ in range(n_out)]
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            env.step_fused(self.actions[0], out=self.outputs[0])      # lazy kernel attributes, aliasing quirk B-6
            side.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=side):
                env.batch_device_counter(True)
                try:
                    for k in range(K):
                        env.step_fused(self.actions[k], out=self.outputs[k % n_out])
                finally:
                    env.batch_device_counter(False)
        torch.cuda.current_stream(dev).wait_stream(side)
        self.steps = K
        env._reset_counter -= K            # the capture advanced the host mirror; nothing ran yet

    def replay(self):
        """Run the K captured steps on the current stream; returns ``.outputs``."""
        self.graph.replay()
        self.env._reset_counter += self.steps          # host mirror of the device word
        return self.outputs


class MappoRollout:
    """``MAPPO.get_data`` (models.py:106-129) for the reference's own learner object, on the device:
    ``MappoRollout(mappo).attach()`` replaces ``mappo.get_data`` so that the training loop of
    marlnav/__main__.py:21-27 (``get_data`` -> ``train_actor`` -> ``train_critic``) runs unchanged, but the
    rollout is {fused actor sample -> fused step} x buffer_len with the critic beside it -- one CUDA-graph
    launch -- and the backward return scan (models.py:131-148) one kernel.

    ``mappo`` needs what the reference's ``MAPPO`` has: ``env`` (a ``marlnav_b200.Env``), ``actor``,
    ``critic``, ``_normalize`` / ``_scale_up`` (the reference's ``ObsNormalizer`` / ``ActionScaler``),
    ``buffer_len``, ``gamma``, ``num_parallel``, ``num_agents``, ``action_size``, ``_logs``,
    ``_update_epi_stats``.  After ``get_data()`` ``mappo.buffer`` holds, per step, the reference's
    ``[obs (B,A,S), actions (B,A,2), log_probs (B*A), values (B,1), returns (B) float64, done (B)]`` --
    views of the rollout's (T, ...) device buffers, valid until the next ``get_data()``.

    Differences from the reference's loop: the exploration noise is an addressed Philox stream
    instead of torch's global generator (same distribution), and nothing is printed per step.

    The env must have float32 observations: the buffer goes straight to the reference's own
    ``train_actor`` / ``train_critic``, whose float32 layers do not take 16-bit input."""

    def __init__(self, mappo, use_graph=True, seed=None):
        env = mappo.env
        _require_f32_obs(env, "MappoRollout")
        self.mappo, self.env, self.use_graph = mappo, env, bool(use_graph)
        norm, scal = mappo._normalize, mappo._scale_up
        env.fuse_io_tensors(norm.mean, norm.scale_tensor.reshape(-1, env.obs_size)[0],
                            scal.mean, scal.scale_tensor.reshape(-1, 2)[0])
        self.actor = FusedActor(mappo.actor, device=env.device, seed=seed)
        self.critic = FusedCritic(mappo.critic, device=env.device)
        self.graph = None

    def attach(self):
        self.mappo.get_data = self.get_data
        return self

    @torch.no_grad()
    def get_data(self):
        m, env = self.mappo, self.env
        T, B, A = int(m.buffer_len), env.num_parallel, env.num_agents
        self.actor.refresh(m.actor)                       # the optimisers stepped since the last rollout
        self.critic.refresh(m.critic)
        if self.use_graph:
            if self.graph is None:
                self.graph = RolloutGraph(env, self.actor, T, critic=self.critic)
            buf = self.graph.replay()
        else:
            buf = collect_rollout(env, self.actor, T, critic=self.critic)
        # models.py:131-148: discounted returns, normalised over the whole buffer
        ret = discounted_returns(buf['rewards'], buf['done'], float(m.gamma))
        std, mean_rew = torch.std_mean(ret.reshape(-1))
        ret = (ret - mean_rew) / (std + 1e-12)
        acts = buf['actions'].view(T, B, A, int(m.action_size))
        m.obs = buf['last_obs']
        # (unbind: the T views of each buffer in one call instead of T Python indexing operations)
        m.buffer = [list(row) for row in zip(buf['obs'].unbind(0), acts.unbind(0), buf['log_probs'].unbind(0),
                                             buf['values'].unbind(0), ret.unbind(0), buf['done'].unbind(0))]
        m._mean_rew = mean_rew
        m._logs['mean_rews'] += [mean_rew.item()]
        m._update_epi_stats()                             # models.py:151-158
        if m._mean_rew > m._max_rew:                      # models.py:127-129, literally
            torch.save(m.actor.state_dict(), m._actor_path)
            torch.save(m.critic.state_dict(), m._critic_path)
