"""Drop-in replacement for ``marlnav.environment.Env`` on one B200.

Same constructor argument (the reference's ``params['env']`` dict,
/root/reference/marlnav/utils.py:257-282), same methods and attributes the
reference's callers touch (SURVEY.md section 8b):

    Env(params)                       environment.py:11-68
    .step(actions) -> (Observations, rewards, terminated, truncated)   :92-107
    .observations() -> Observations   :139-180
    .sample_actions()                 :109-111
    .reset()                          :70-74   (a no-op in the reference too)
    .states (B,A,5) .obstacles (B,O,2) .target (B,1,2)                 :28-30
    ._num_trunc ._num_col ._num_tar   (read AND assigned by MAPPO, models.py:153-158)
    ._risk_factor ... ._bond_factor   (read by check_rews, utils.py:648-653)

but ``step`` is ONE launch of the fused sm_100a kernel in
``csrc/marlnav_step_*.cu`` through the C ABI of ``include/marlnav_b200.h``.
State tensors stay resident in HBM and are updated in place; outputs are fresh
tensors every step (the rollout buffer keeps references to them, models.py:121).

There is no CPU fallback: ``params['device']`` must be a CUDA device.

Differences from the reference, all documented in DESIGN.md:
  * re-initialised obstacles come from an addressed Philox4x32-10 stream keyed by
    (seed, global env id, step counter) instead of the global CPU mt19937 stream
    (utils.py:390-398); ``params['seed']`` or ``torch.initial_seed()`` seeds it.
  * ``params['env_id_offset']`` (default 0) is the global id of local env 0, so N
    processes stepping N slices reproduce the single-process run bit for bit.
  * ``init_method='template'`` accepts an explicit (A,5) agent template for team
    sizes the reference's 3-agent triangle cannot express.
  * ``params['obs_dtype']`` (default ``torch.float32``) may be ``torch.float16`` or
    ``torch.bfloat16``: every observation the env returns is then the float32 value
    rounded to nearest-even (``obs32.to(dtype)``, bit for bit); rewards, flags and the
    state are unchanged.
"""
import ctypes
import math
from collections import namedtuple

import torch

from . import _lib
from .params import GEOMETRY
from .samplers import action_sampler
from .slots import OutputSlots

# Same type the reference returns (utils.py:13-15).
Observations = namedtuple('Observations', ['target_angle', 'target_distance',
    'obstacles_angles', 'obstacles_distances', 'others_angles', 'others_distances'])


def _triangle_agents(init):
    """(3,5) float32 agent template, computed with the same float32 torch ops as
    TriangleIntitializer.__init__ (utils.py:349-368)."""
    pos_const = 0.5 * init['ags_dist']
    pos = pos_const * torch.tensor([[-1 / math.sqrt(3), 1.], [2 / math.sqrt(3), 0.],
                                    [-1 / math.sqrt(3), -1.]])
    pos = pos + torch.tensor([init['ags_cent_x'], init['ags_cent_y']]).unsqueeze(0).repeat(3, 1)
    heading = torch.tensor([[1., 0.]] * 3)
    speed = init['init_speed'] * torch.ones(3, 1)
    return torch.cat([pos, heading, speed], dim=1)


# observation element types: torch dtype -> MARLNAV_OBS_* code of the `_typed` entry points
OBS_DTYPES = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}


def split_observations(obs, num_agents, num_obstacles):
    """Six views of the fused (B,A,S) buffer, in the reference's field order."""
    O, R = num_obstacles, num_agents - 1
    o = 2
    return Observations(obs[:, :, 0:1], obs[:, :, 1:2], obs[:, :, o:o + O], obs[:, :, o + O:o + 2 * O],
                        obs[:, :, o + 2 * O:o + 2 * O + R], obs[:, :, o + 2 * O + R:o + 2 * O + 2 * R])


class Env(object):
    """Parallelised environment state + fused CUDA step (see module docstring)."""

    def __init__(self, params):
        self._lib = _lib.load()
        self.params = params
        dev = torch.device(params['device'])
        if dev.type != 'cuda':
            raise _lib.MarlnavError(
                f"marlnav_b200.Env needs a CUDA device, got {params['device']!r} "
                "(there is no CPU fallback; use the reference Env on CPU)")
        if not torch.cuda.is_available() or self._lib.marlnav_device_count() < 1:
            raise _lib.MarlnavError("no CUDA device visible")
        if dev.index is None:
            dev = torch.device('cuda', torch.cuda.current_device())
        self.device = dev
        self._dev_index = dev.index
        self.num_parallel = int(params['num_parallel'])
        self.num_agents = int(params['num_agents'])
        self._n_action_floats = self.num_parallel * self.num_agents * 2
        self.num_obstacles = int(params['num_obstacles'])
        self.max_step = params['max_step']
        self.episode_len = int(params['episode_len'])
        self.obs_size = self._lib.marlnav_obs_size(self.num_agents, self.num_obstacles)
        if self.obs_size == 0:
            raise _lib.MarlnavError(
                f"unsupported team shape A={self.num_agents}, O={self.num_obstacles} "
                "(need 2 <= A <= 26, 1 <= O <= 64)")
        # fixed for the env's life: output slots, captured graphs and host buffers are sized from it
        self.obs_dtype = params.get('obs_dtype', torch.float32)
        if self.obs_dtype not in OBS_DTYPES:
            raise _lib.MarlnavError(f"obs_dtype must be torch.float32, torch.float16 or torch.bfloat16, "
                                    f"got {self.obs_dtype!r}")
        self._obs_code = OBS_DTYPES[self.obs_dtype]
        self._sampler = action_sampler(params.get('sampler'))
        self._others_inds = torch.tensor(
            [[i for i in range(self.num_agents) if i != j] for j in range(self.num_agents)],
            device=dev)

        self.min_speed, self.max_speed = params['min_speed'], params['max_speed']
        self.min_accel, self.max_accel = params['min_accel'], params['max_accel']
        self._risk_factor = params['risk_factor']
        self._distance_factor = params['distance_factor']
        self._heading_factor = params['heading_factor']
        self._target_factor = params['target_factor']
        self._soft_factor = params['soft_factor']
        self._bond_factor = params['bond_factor']
        self._ob_risk_dist, self._ag_risk_dist = GEOMETRY['ob_risk_dist'], GEOMETRY['ag_risk_dist']
        self._ob_coll_dist, self._ag_coll_dist = GEOMETRY['ob_coll_dist'], GEOMETRY['ag_coll_dist']
        self._agents_min_d, self._agents_max_d = GEOMETRY['agents_min_d'], GEOMETRY['agents_max_d']
        self._max_at_prop_d = 2
        self._max_angle_diff = GEOMETRY['max_angle_diff']
        self._target_radius = GEOMETRY['target_radius']
        self._cap_distance = GEOMETRY['cap_distance']
        self._bond_sharpness = GEOMETRY['bond_sharpness']
        self._ideal_dist = GEOMETRY['ideal_dist']
        self._init_dist = GEOMETRY['init_dist']

        seed = params.get('seed')
        self._seed = int(torch.initial_seed() if seed is None else seed) & 0xFFFFFFFFFFFFFFFF
        self._env_id_offset = int(params.get('env_id_offset', 0))
        self._reset_counter = 0
        self._counter_dev = None          # device-resident copy of the counter (use_device_counter)
        self._counter_batch = False       # batch mode: steps pass their offset, one add per batch
        self._counter_pending = 0

        self._c_params = self._make_c_params()
        self._setup_reset_source(params['init'])

        B, A, O = self.num_parallel, self.num_agents, self.num_obstacles
        self._ring = OutputSlots(self._new_slot)      # reusable output slots of step()
        with torch.cuda.device(dev):
            self._states = torch.empty(B, A, 5, device=dev)
            self._obstacles = torch.empty(B, O, 2, device=dev)
            self._target = torch.empty(B, 1, 2, device=dev)
            self._step_num = torch.empty(B, device=dev)
            self._terminates_u8 = torch.empty(B, dtype=torch.uint8, device=dev)
            self._stats = torch.zeros(3, dtype=torch.int64, device=dev)   # trunc, col, tar
            rs = self._reset_spec(alias=False)
            _lib.check(self._lib.marlnav_init_f32(
                ctypes.byref(self._c_params), ctypes.byref(rs), self._ptr(self.states),
                self._ptr(self.obstacles), self._ptr(self.target), self._ptr(self._step_num),
                self._ptr(self._terminates_u8), self._stream()), "marlnav_init_f32")
        # MockInitializer aliasing (SURVEY.md Appendix B-6): until the first step, the
        # reset template IS the state tensor.
        self._alias_pending = self._per_env_template
        self._io = None
        self._io_tensors = None

    # ------------------------------------------------------------------ plumbing

    @staticmethod
    def _ptr(t):
        return ctypes.c_void_p(t.data_ptr())

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _raw_stream(self):
        """cudaStream_t of torch's current stream on this device, as an int."""
        try:
            return torch._C._cuda_getCurrentRawStream(self._dev_index)
        except AttributeError:            # (private fast path; the public route costs ~1.5 us more)
            return torch.cuda.current_stream(self.device).cuda_stream

    # The reference rebinds env.states / env.obstacles / env.target on every step
    # (environment.py:80-84) and callers may assign them; here they are updated in place, and an
    # assignment re-binds the tensor the kernels work on (the cached launch arguments are rebuilt).
    def _bind_state(self, name, value, shape):
        t = torch.as_tensor(value, dtype=torch.float32, device=self.device).reshape(shape).contiguous()
        setattr(self, name, t)
        self.__dict__.pop('_call_cache', None)

    states = property(lambda self: self._states,
                      lambda self, v: self._bind_state('_states', v, (self.num_parallel, self.num_agents, 5)))
    obstacles = property(lambda self: self._obstacles,
                         lambda self, v: self._bind_state('_obstacles', v, (self.num_parallel, self.num_obstacles, 2)))
    target = property(lambda self: self._target,
                      lambda self, v: self._bind_state('_target', v, (self.num_parallel, 1, 2)))

    def _make_c_params(self):
        p = _lib.EnvParams()
        p.num_envs, p.num_agents = self.num_parallel, self.num_agents
        p.num_obstacles, p.episode_len = self.num_obstacles, self.episode_len
        p.min_speed, p.max_speed = self.min_speed, self.max_speed
        p.min_accel, p.max_accel = self.min_accel, self.max_accel
        p.risk_factor, p.distance_factor = self._risk_factor, self._distance_factor
        p.heading_factor, p.target_factor = self._heading_factor, self._target_factor
        p.soft_factor, p.bond_factor = self._soft_factor, self._bond_factor
        for k, v in GEOMETRY.items():
            setattr(p, k, v)
        return p

    def _setup_reset_source(self, init):
        dev, B, A, O = self.device, self.num_parallel, self.num_agents, self.num_obstacles
        method = init['init_method']
        if method in ('triangle', 'template'):
            if method == 'triangle':
                if A != 3:
                    raise _lib.MarlnavError(
                        "init_method='triangle' is a 3-agent formation (utils.py:350-368); "
                        "use init_method='template' with an (A,5) agent_template")
                agents = _triangle_agents(init)
            else:
                agents = torch.as_tensor(init['agent_template'], dtype=torch.float32).reshape(A, 5)
            # utils.py:25,381-388: Gaussian position noise + heading rotation on every (re-)initialised
            # agent.  Constants with the reference's own float32 ops (utils.py:370-373: MultivariateNormal
            # keeps scale_tril = cholesky(diag(ags_std, ags_std))).
            self._noisy = bool(init.get('noisy_ags'))
            if self._noisy:
                chol = torch.linalg.cholesky(torch.diag(torch.tensor([init['ags_std'], init['ags_std']])))
                self._noise = (float(chol[0, 0]), float(init['ags_dist']), float(init['angle_range']))
            # (with noise the would-be sample of an env that does not reset can be negative, so the
            # literal blend old + 0*new is evaluated instead of the "+0" shortcut)
            self._tmpl_nonneg = not bool(torch.signbit(agents).any()) and not self._noisy
            self._tmpl_states = agents.to(dev).contiguous()
            self._tmpl_obstacles = None
            self._tmpl_target = torch.tensor([init['tar_pos_x'], init['tar_pos_y']], device=dev)
            self._per_env_template = False
            p = self._c_params      # utils.py:344-347
            p.obst_x_range = init['obst_max_x'] - init['obst_min_x']
            p.obst_y_range = init['obst_max_y'] - init['obst_min_y']
            p.obst_x_mean = 0.5 * (init['obst_min_x'] + init['obst_max_x'])
            p.obst_y_mean = 0.5 * (init['obst_min_y'] + init['obst_max_y'])
        elif method == 'mock_init':
            self._tmpl_states = torch.tensor(init['mock_states'], dtype=torch.float32,
                                             device=dev).reshape(B, A, 5).contiguous()
            self._tmpl_obstacles = torch.tensor(init['mock_obstacles'], dtype=torch.float32,
                                                device=dev).reshape(B, O, 2).contiguous()
            self._tmpl_target = torch.tensor(init['mock_target'], dtype=torch.float32,
                                             device=dev).reshape(B, 2).contiguous()
            self._per_env_template = True
            self._tmpl_nonneg = False
            self._noisy = False
        else:
            raise ValueError(f"unknown init_method {method!r}")

    def _reset_spec(self, alias):
        rs = _lib.ResetSpec()
        rs.tmpl_states = self._tmpl_states.data_ptr()
        rs.tmpl_obstacles = self._tmpl_obstacles.data_ptr() if self._tmpl_obstacles is not None else None
        rs.tmpl_target = self._tmpl_target.data_ptr()
        per_env = self._per_env_template
        rs.states_env_stride = self.num_agents * 5 if per_env else 0
        rs.obstacles_env_stride = self.num_obstacles * 2 if per_env else 0
        rs.target_env_stride = 2 if per_env else 0
        rs.alias_first_step = 1 if alias else 0
        rs.flags = _lib.RESET_TMPL_NONNEG if (not per_env and self._tmpl_nonneg) else 0
        if self._noisy:
            rs.flags |= _lib.RESET_NOISY_AGENTS
            rs.noise_chol, rs.noise_mult, rs.angle_range = self._noise
        rs.seed, rs.env_id_offset = self._seed, self._env_id_offset
        # ABI 3: the kernels use step_counter + *step_counter_dev
        rs.step_counter = self._reset_counter if self._counter_dev is None else self._counter_pending
        rs.step_counter_dev = self._counter_dev.data_ptr() if self._counter_dev is not None else None
        return rs

    # ------------------------------------------------------------------ episode statistics

    def _stat_get(self, i):
        return int(self._stats[i].item())

    def _stat_set(self, i, value):
        self._stats[i] = int(value)

    _num_trunc = property(lambda self: self._stat_get(0), lambda self, v: self._stat_set(0, v))
    _num_col = property(lambda self: self._stat_get(1), lambda self, v: self._stat_set(1, v))
    _num_tar = property(lambda self: self._stat_get(2), lambda self, v: self._stat_set(2, v))

    @property
    def episode_stats(self):
        """Device int64[3] = (num_trunc, num_col, num_tar) of this process's slice; no sync."""
        return self._stats

    @property
    def _terminates(self):
        return self._terminates_u8.view(torch.bool)

    # ------------------------------------------------------------------ reference API

    def reset(self):
        """environment.py:70-74.  The reference's reset() only sets a mask that step()
        overwrites before using it, i.e. it changes nothing (SURVEY.md Appendix B-5)."""
        return self.observations(), self.params

    def sample_actions(self):
        return self._sampler()

    def supports_fused_actor(self, actor):
        """Is there a fused {actor -> step} kernel (marlnav_act_step_typed) for this env and actor?"""
        return (self.num_agents == 3 and 1 <= self.num_obstacles <= 6 and self._io is not None
                and bool(self._io.obs_mean) and bool(self._io.act_scale)
                and getattr(actor, 'obs_size', None) == self.obs_size and getattr(actor, 'hidden', 10 ** 9) <= 256
                and getattr(getattr(actor, 'w1', None), 'device', None) == self.states.device)

    def act_step_fused(self, actor, obs_in, out, obs_dtype=torch.float32):
        """``actor.act(obs_in)`` + ``step_fused`` as ONE launch (SURVEY 8(f)-2; models.py:113-122).
        ``obs_in`` (B,A,S): the normalised observations of the current state; ``out`` = preallocated
        (actions (B*A,2), log_probs (B*A), next_obs (B,A,S), rewards (B), terminated_u8 (B),
        truncated_u8 (B)).  Needs ``fuse_io`` with both transforms.  ``obs_dtype`` is the element type
        of ``obs_in`` and ``next_obs`` and must be the env's ``obs_dtype``: the actor reads 16-bit
        observations widened exactly to float32, the same bits as ``actor.act(obs_in.float())``."""
        if obs_dtype != self.obs_dtype:
            raise _lib.MarlnavError(f"act_step_fused: obs_dtype {obs_dtype} does not match this env's obs_dtype "
                                    f"{self.obs_dtype}")
        if not self.supports_fused_actor(actor):
            raise _lib.MarlnavError("no fused actor+step kernel for this env/actor (see supports_fused_actor)")
        actions, log_probs, obs, rew, term, trunc = out
        n = self.num_parallel * self.num_agents * self.obs_size
        for name, t in (("obs_in", obs_in), ("out[2]", obs)):
            if t.dtype != obs_dtype or t.numel() < n:
                raise _lib.MarlnavError(f"act_step_fused: {name} must be {obs_dtype} with at least {n} elements, "
                                        f"got {t.dtype} with {t.numel()}")
        if obs_in.data_ptr() == obs.data_ptr():
            raise _lib.MarlnavError("act_step_fused: obs_in and the output observations must be different buffers")
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            sp = actor.spec(actor._advance_counter(stream))
            sp.row_offset = self._env_id_offset * self.num_agents if actor.row_offset is None else actor.row_offset
            rs = self._reset_spec(alias=self._alias_pending)
            rs.step_counter = self._next_step_counter(stream)
            _lib.check(self._lib.marlnav_act_step_typed(
                ctypes.byref(self._c_params), ctypes.byref(rs), self._ptr(self.states), self._ptr(self.obstacles),
                self._ptr(self.target), self._ptr(self._step_num), self._ptr(self._terminates_u8),
                ctypes.byref(sp), obs_in.data_ptr(), actions.data_ptr(), log_probs.data_ptr(), obs.data_ptr(),
                self._obs_code, rew.data_ptr(), term.data_ptr(), trunc.data_ptr(), self._ptr(self._stats),
                ctypes.byref(self._io), stream), "marlnav_act_step_typed")
            self._step_launched()
        return actions, log_probs, obs, rew, term, trunc

    def _next_step_counter(self, stream):
        """``step_counter`` argument of the step about to be launched; nothing on the host moves until
        ``_step_launched`` is called after the launch was accepted.  Host counter: its next value.
        Device counter: 0 after bumping the device word on ``stream``, or, in batch mode, the step's
        offset inside the batch (``flush_device_counter`` adds the total)."""
        if self._counter_dev is None:
            return self._reset_counter + 1
        if self._counter_batch:
            return self._counter_pending + 1
        self._lib.marlnav_counter_add(self._counter_dev.data_ptr(), 1, stream)
        return 0

    def _step_launched(self):
        """Host bookkeeping after a step launch was accepted: the reset step counter moves on, and
        the first step of an aliased template hands over its template."""
        self._reset_counter += 1
        if self._counter_dev is not None and self._counter_batch:
            self._counter_pending += 1
        if self._alias_pending:
            # the reference's template froze at "state after the first move" (B-6)
            self._tmpl_states = self._states.clone()
            self._alias_pending = False
            self.__dict__.pop('_call_cache', None)      # template pointer changed

    def batch_device_counter(self, enable=True):
        """Batch mode of the device-resident counter: steps address their Philox draws as
        ``device word + offset`` and ONE ``marlnav_counter_add`` per batch replaces one per step
        (``collect_rollout``: a third of the launches of a captured rollout)."""
        if not enable:
            self.flush_device_counter()
        self._counter_batch = bool(enable) and self._counter_dev is not None

    def flush_device_counter(self):
        if self._counter_dev is not None and self._counter_pending:
            self._lib.marlnav_counter_add(self._counter_dev.data_ptr(), self._counter_pending,
                                          torch.cuda.current_stream(self.device).cuda_stream)
        self._counter_pending = 0

    def use_device_counter(self, enable=True):
        """Keep the reset step counter in device memory (advanced by a one-thread kernel before
        every step) instead of passing it from the host.  Results are identical; the point is that
        a CUDA graph capturing ``step`` then draws fresh reset positions on every replay."""
        if enable and self._counter_dev is None:
            self._counter_dev = torch.full((1,), self._reset_counter, dtype=torch.int64, device=self.device)
        elif not enable and self._counter_dev is not None:
            self.batch_device_counter(False)
            self._reset_counter = int(self._counter_dev.item())
            self._counter_dev = None
        self.__dict__.pop('_call_cache', None)

    def fuse_io(self, normalizer_params=None, scaler_params=None):
        """Fold the caller-side ObsNormalizer (utils.py:519-532) and/or ActionScaler
        (utils.py:535-547) into the step kernel.  After this, ``step`` takes the
        policy's raw [-1,1] actions and/or returns normalised observations (use
        ``.normalized`` views via torch.cat as before or the fused buffer directly)."""
        dev = self.device
        io = _lib.IoTransform()
        keep = []
        if normalizer_params is not None:
            lo = torch.tensor(normalizer_params['min_obs'], dtype=torch.float32)
            hi = torch.tensor(normalizer_params['max_obs'], dtype=torch.float32)
            if lo.numel() != self.obs_size:
                raise _lib.MarlnavError(f"normalizer has {lo.numel()} entries, obs_size is {self.obs_size}")
            scale, mean = (0.5 * (hi - lo)).to(dev), (0.5 * (lo + hi)).to(dev)
            io.obs_mean, io.obs_scale = mean.data_ptr(), scale.data_ptr()
            keep += [mean, scale]
        if scaler_params is not None:
            lo = torch.tensor(scaler_params['min_action'], dtype=torch.float32)
            hi = torch.tensor(scaler_params['max_action'], dtype=torch.float32)
            scale, mean = (0.5 * (hi - lo)).to(dev), (0.5 * (lo + hi)).to(dev)
            io.act_mean, io.act_scale = mean.data_ptr(), scale.data_ptr()
            keep += [mean, scale]
        self._io, self._io_tensors = (io, keep) if keep else (None, None)
        self.__dict__.pop('_call_cache', None)

    def fuse_io_tensors(self, obs_mean=None, obs_scale=None, act_mean=None, act_scale=None):
        """``fuse_io`` from the tensors an existing ``ObsNormalizer`` / ``ActionScaler`` already holds
        (``.mean`` and one row of ``.scale_tensor``, utils.py:523-528,539-544): the kernel then divides /
        multiplies by exactly the values the reference's callables would."""
        dev = self.device
        io = _lib.IoTransform()
        keep = []
        cvt = lambda t, n: torch.as_tensor(t, dtype=torch.float32).detach().reshape(-1)[:n].to(dev).contiguous()
        if obs_mean is not None:
            mean, scale = cvt(obs_mean, self.obs_size), cvt(obs_scale, self.obs_size)
            if mean.numel() != self.obs_size or scale.numel() != self.obs_size:
                raise _lib.MarlnavError(f"normalizer needs {self.obs_size} entries")
            io.obs_mean, io.obs_scale = mean.data_ptr(), scale.data_ptr()
            keep += [mean, scale]
        if act_mean is not None:
            mean, scale = cvt(act_mean, 2), cvt(act_scale, 2)
            io.act_mean, io.act_scale = mean.data_ptr(), scale.data_ptr()
            keep += [mean, scale]
        self._io, self._io_tensors = (io, keep) if keep else (None, None)
        self.__dict__.pop('_call_cache', None)

    def _observe(self, dtype):
        """(B,A,S) observations of the current states in `dtype` (one kernel launch)."""
        with torch.cuda.device(self.device):
            obs = torch.empty(self.num_parallel, self.num_agents, self.obs_size, dtype=dtype, device=self.device)
            _lib.check(self._lib.marlnav_observe_typed(
                ctypes.byref(self._c_params), self._ptr(self.states), self._ptr(self.obstacles),
                self._ptr(self.target), self._ptr(obs), OBS_DTYPES[dtype], self._stream()), "marlnav_observe_typed")
        return obs

    def _observations_f32(self):
        """(B,A,S) float32 observations of the current states, whatever ``obs_dtype`` is: a 16-bit
        rollout normalises these before it rounds them (``collect_rollout``)."""
        return self._observe(torch.float32)

    def observations_fused(self):
        """(B,A,S) observation buffer of the current states, in ``obs_dtype`` (one kernel launch)."""
        return self._observe(self.obs_dtype)

    def observations(self):
        """environment.py:139-180"""
        return split_observations(self.observations_fused(), self.num_agents, self.num_obstacles)

    def _alloc_outputs(self):
        B, A, S = self.num_parallel, self.num_agents, self.obs_size
        n_obs_used = B * A * S * self.obs_dtype.itemsize
        n_obs = (n_obs_used + 15) & ~15               # rewards and flags stay 16-byte aligned
        n_rew = (B * 4 + 15) & ~15
        n_flag = (B + 15) & ~15
        buf = torch.empty(n_obs + n_rew + 2 * n_flag, dtype=torch.uint8, device=self.device)
        obs = buf[:n_obs_used].view(self.obs_dtype).view(B, A, S)
        rew = buf[n_obs:n_obs + B * 4].view(torch.float32)
        term = buf[n_obs + n_rew:n_obs + n_rew + B]
        trunc = buf[n_obs + n_rew + n_flag:n_obs + n_rew + n_flag + B]
        return obs, rew, term, trunc

    # ---- output slots (marlnav_b200/slots.py): buffers with prebuilt views and launch arguments,
    # recycled only when the caller holds none of their tensors

    def _new_slot(self):
        obs, rew, term, trunc = self._alloc_outputs()
        fields = split_observations(obs, self.num_agents, self.num_obstacles)
        tb, cb = term.view(torch.bool), trunc.view(torch.bool)
        return dict(obs=obs, rew=rew, term=tb, trunc=cb, fields=fields, storage=obs.untyped_storage(),
                    objs=(obs, rew, tb, cb, fields) + tuple(fields),
                    ptrs=(obs.data_ptr(), rew.data_ptr(), term.data_ptr(), trunc.data_ptr()),
                    u8=(term, trunc), call=_lib.StepCall(), epoch=0)

    def _take_slot(self):
        """-> (slot, stream): the raw current stream when this env's device is current, else None
        (the launch then switches devices itself and the slot is not shared with other streams)."""
        if torch.cuda.current_device() == self._dev_index:
            stream = self._raw_stream()
            return self._ring.take(stream), stream
        return self._ring.take(-1), None

    def _step_call_cache(self):
        """Launch arguments that do not change between steps (state tensors are updated in place;
        assigning env.states / .obstacles / .target, fuse_io, use_device_counter and the aliasing
        hand-over drop this cache): built once, because the per-step host cost is what bounds small
        batches.  `epoch` tells a slot's prebuilt marlnav_step_call that it is stale."""
        c = self.__dict__.get('_call_cache')
        if c is None:
            rs = self._reset_spec(alias=False)
            self._call_epoch = self.__dict__.get('_call_epoch', 0) + 1
            c = dict(rs=rs, epoch=self._call_epoch)
            self._call_cache = c
        return c

    def _fill_call(self, call, c, ptrs):
        """A marlnav_step_call for this env writing to the output pointers `ptrs`."""
        call.params = ctypes.addressof(self._c_params)
        call.reset = ctypes.addressof(c['rs'])
        call.states, call.obstacles, call.target = self._states.data_ptr(), self._obstacles.data_ptr(), self._target.data_ptr()
        call.step_num, call.terminates = self._step_num.data_ptr(), self._terminates_u8.data_ptr()
        call.obs, call.rewards, call.terminated, call.truncated = ptrs
        call.stats = self._stats.data_ptr()
        call.io = ctypes.addressof(self._io) if self._io is not None else None
        return call

    def _launch_step(self, actions, ptrs, slot=None, stream=None, final_ptr=None):
        """One fused step launch writing to the four output pointers `ptrs` (or to `slot`'s), on
        `stream` (raw handle of the current stream of this env's device; None = look it up);
        with `final_ptr` the finished envs' pre-reset observations go there too."""
        if actions.device != self.device or actions.dtype != torch.float32 or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.float32).contiguous()
        if actions.numel() != self._n_action_floats:
            raise _lib.MarlnavError(f"actions must be ({self.num_parallel},{self.num_agents},2), got {tuple(actions.shape)}")
        if stream is None:
            if torch.cuda.current_device() != self._dev_index:
                with torch.cuda.device(self.device):
                    return self._launch_step(actions, ptrs, slot, final_ptr=final_ptr)
            stream = self._raw_stream()
        c = self._step_call_cache()
        if slot is not None:
            call = slot['call']
            if slot['epoch'] != c['epoch']:
                self._fill_call(call, c, slot['ptrs'])
                slot['epoch'] = c['epoch']
        else:
            # caller-supplied outputs: their calls are remembered too (rollout buffers, CUDA-graph capture)
            calls = c.setdefault('out_calls', {})
            call = calls.get(ptrs)
            if call is None:
                if len(calls) >= 256:
                    calls.clear()
                call = calls[ptrs] = self._fill_call(_lib.StepCall(), c, ptrs)
        rs = c['rs']
        rs.step_counter = self._next_step_counter(stream)      # the host counters move after the launch
        if self._alias_pending:
            rs.alias_first_step = 1
        call.actions = actions.data_ptr()
        call.stream = stream
        if final_ptr is None:
            rc = self._lib.marlnav_step_call_typed(ctypes.addressof(call), self._obs_code)
            if rc:
                _lib.check(rc, "marlnav_step_call_typed")
        else:
            rc = self._lib.marlnav_step_call_final_typed(ctypes.addressof(call), self._obs_code, final_ptr)
            if rc:
                _lib.check(rc, "marlnav_step_call_final_typed")
        self._step_launched()

    def _final_obs_ptr(self, final_obs, out):
        n = self.num_parallel * self.num_agents * self.obs_size
        if not isinstance(final_obs, torch.Tensor) or final_obs.device != self.device \
                or final_obs.dtype != self.obs_dtype or final_obs.numel() < n or not final_obs.is_contiguous():
            got = (f"{final_obs.dtype} with {final_obs.numel()} elements on {final_obs.device}"
                   if isinstance(final_obs, torch.Tensor) else type(final_obs).__name__)
            raise _lib.MarlnavError(f"step_fused: final_obs must be a contiguous {self.obs_dtype} tensor on "
                                    f"{self.device} with at least {n} elements, got {got}")
        if out is not None and final_obs.data_ptr() == out[0].data_ptr():
            raise _lib.MarlnavError("step_fused: final_obs and out[0] must be different buffers")
        return final_obs.data_ptr()

    def step_fused(self, actions, out=None, final_obs=None):
        """One fused step.  Returns ``(obs (B,A,S), rewards (B), terminated (B) bool,
        truncated (B) bool)``; ``out`` may supply preallocated (obs, rewards,
        terminated_u8, truncated_u8) tensors to write into; ``obs`` must have the env's
        ``obs_dtype`` and at least B*A*S elements.

        ``final_obs`` (a (B,A,S) tensor of the env's ``obs_dtype`` on its device, not ``out[0]``)
        also receives, for every env this step finishes (terminated or truncated), the
        observations its rewards and flags were computed from, before the auto-reset replaced them
        (gymnasium's ``final_obs``): the bits a non-resetting env gets in ``obs``.  Rows of the
        other envs are left as they were."""
        final_ptr = None if final_obs is None else self._final_obs_ptr(final_obs, out)
        if out is not None:
            obs, rew, term, trunc = out
            if obs.dtype != self.obs_dtype or obs.numel() < self.num_parallel * self.num_agents * self.obs_size:
                raise _lib.MarlnavError(
                    f"step_fused: out[0] must be {self.obs_dtype} with at least "
                    f"{self.num_parallel * self.num_agents * self.obs_size} elements, got {obs.dtype} "
                    f"with {obs.numel()}")
            self._launch_step(actions, (obs.data_ptr(), rew.data_ptr(), term.data_ptr(), trunc.data_ptr()),
                              final_ptr=final_ptr)
            return obs, rew, term.view(torch.bool), trunc.view(torch.bool)
        slot, stream = self._take_slot()
        self._launch_step(actions, None, slot, stream, final_ptr)
        return slot['obs'], slot['rew'], slot['term'], slot['trunc']

    def step(self, actions):
        """environment.py:92-107"""
        slot, stream = self._take_slot()
        self._launch_step(actions, None, slot, stream)
        return slot['fields'], slot['rew'], slot['term'], slot['trunc']

    def launch_info(self):
        """(grid, block, dynamic smem bytes, envs per CTA) of the step kernel for this shape."""
        g, b, s, e = (ctypes.c_int() for _ in range(4))
        _lib.check(self._lib.marlnav_step_launch_info(ctypes.byref(self._c_params), ctypes.byref(g),
                                                      ctypes.byref(b), ctypes.byref(s), ctypes.byref(e)),
                   "marlnav_step_launch_info")
        return g.value, b.value, s.value, e.value


class HostStepper:
    """Steps an ``Env`` for a HOST-resident policy through ``marlnav_step_host_typed``:
    pinned host actions in, pinned host observations/rewards/flags out, env state
    resident in HBM.  This is the end-to-end path ``bench.py`` reports as ``e2e``."""

    def __init__(self, env):
        self.env = env
        B, A, S = env.num_parallel, env.num_agents, env.obs_size
        dev = env.device
        self.actions_host = torch.empty(B, A, 2, pin_memory=True)
        self.obs_host = torch.empty(B, A, S, dtype=env.obs_dtype, pin_memory=True)
        self.rewards_host = torch.empty(B, pin_memory=True)
        self.terminated_host = torch.empty(B, dtype=torch.uint8, pin_memory=True)
        self.truncated_host = torch.empty(B, dtype=torch.uint8, pin_memory=True)
        self.actions_dev = torch.empty(B, A, 2, device=dev)
        self.obs_dev = torch.empty(B, A, S, dtype=env.obs_dtype, device=dev)
        self.rewards_dev = torch.empty(B, device=dev)
        self.terminated_dev = torch.empty(B, dtype=torch.uint8, device=dev)
        self.truncated_dev = torch.empty(B, dtype=torch.uint8, device=dev)
        self.h2d_bytes = self.actions_host.numel() * 4
        self.d2h_bytes = self.obs_host.numel() * self.obs_host.element_size() + B * 4 + 2 * B
        # the pipeline's two side streams and events belong to this stepper (marlnav_host_pipe)
        self._pipe = ctypes.c_void_p()
        with torch.cuda.device(dev):
            _lib.check(env._lib.marlnav_host_pipe_create(ctypes.byref(self._pipe)), "marlnav_host_pipe_create")

    def close(self):
        pipe, self._pipe = getattr(self, '_pipe', None), None
        if pipe:
            torch.cuda.synchronize(self.env.device)
            self.env._lib.marlnav_host_pipe_destroy(pipe)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def step(self, actions=None, sync=True):
        """Consumes ``actions`` (a pinned CPU float32 tensor of shape (B,A,2); default
        ``self.actions_host``) and fills the ``*_host`` outputs."""
        env = self.env
        p = Env._ptr
        src = self.actions_host if actions is None else actions
        if src.device.type != 'cpu' or src.dtype != torch.float32 or not src.is_contiguous() \
                or src.numel() != self.actions_host.numel():
            raise _lib.MarlnavError("HostStepper.step needs a contiguous float32 CPU tensor of shape (B,A,2)")
        with torch.cuda.device(env.device):
            stream = torch.cuda.current_stream(env.device).cuda_stream
            rs = env._reset_spec(alias=env._alias_pending)
            rs.step_counter = env._next_step_counter(stream)
            args = (self._pipe, ctypes.byref(env._c_params), ctypes.byref(rs),
                    p(env.states), p(env.obstacles), p(env.target), p(env._step_num), p(env._terminates_u8),
                    p(src), p(self.actions_dev), p(self.obs_dev), p(self.rewards_dev),
                    p(self.terminated_dev), p(self.truncated_dev),
                    p(self.obs_host), p(self.rewards_host), p(self.terminated_host), p(self.truncated_host),
                    p(env._stats), ctypes.byref(env._io) if env._io is not None else None,
                    ctypes.c_void_p(stream), env._obs_code)
            _lib.check(env._lib.marlnav_step_host_typed(*args), "marlnav_step_host_typed")
            env._step_launched()
            if sync:
                torch.cuda.current_stream(env.device).synchronize()
