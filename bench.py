#!/usr/bin/env python
"""bench.py -- env-steps/s of the fused MARL-nav environment step on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[3]): 1,048,576 parallel envs x 3 agents x 3
obstacles per GPU, policy-like random actions (SURVEY.md section 8d: turn angle
~U(-0.2,0.2) rad, accel ~U(-0.5,0.5), a pool of 16 pre-generated action tensors cycled),
auto-reset on every termination/truncation, episode_len 200.  A "step" is ONE call of the
reference-facing ``Env.step(actions)`` (environment.py:92-107: fresh output tensors, the
Observations namedtuple) over the whole batch.  N>1 (torchrun, one rank per GPU): every
rank steps its own slice (weak scaling, no data-path collective); the three episode
counters are all-reduced over NCCL once after the timed region.

One JSON line on stdout (rank 0):
  value        env-steps/s, inputs resident in HBM, CUDA events, max over ranks
  e2e          the same metric through marlnav_step_host_f32: pinned HOST actions in,
               HOST observations/rewards/flags out, copies inside the timed region
  roofline     algorithmic bytes per launch / mean launch duration vs the measured HBM peak
  cpu_baseline the reference's own Env.step (baseline/_ref, unmodified; the torch-op port
               oracle.TorchPortEnv when the reference did not travel) on this box's cores
  configs      the other BASELINE.json configurations timed in the same process:
               262144x8x16 (configs[4], with its own roofline), 65536x3x3 (configs[2]),
               1024x3x3 (configs[1]: eager Env.step / step_fused(out=) / the whole rollout with
               the fused actor + critic as one CUDA graph), 2x3x3 (configs[0] scale)
  strong       configs[3] as BASELINE.json words it: 1,048,576 envs in TOTAL split over the N
               ranks, each rank's steps captured in a CUDA graph (StepGraph)
--impl reference times the reference's own CPU implementation alone: the real
marlnav.environment.Env from baseline/_ref (vendored, git-ignored, by __graft_entry__.build())
at the full batch size, all host threads; its line also carries ``reference_cuda`` -- the same
unmodified Env on device='cuda' (BASELINE.md 4.4's second bar).
--dump-outputs DIR writes what the last timed Env.step returned (see dump_outputs) so that two
builds can be compared output for output: the inputs depend only on the arguments.
"""
import argparse
import json
import math
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC, UNIT = "env_steps_per_sec", "env-steps/s"
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def algorithmic_bytes(A, O):
    """SURVEY.md section 8(d): every tensor read once + written once per env-step."""
    S = 2 + 2 * O + 2 * (A - 1)
    rd = 20 * A + 8 * A + 8 * O + 8 + 4 + 1
    wr = 20 * A + 4 + 1 + 4 * A * S + 4 + 1 + 1
    return rd + wr


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(A, O, B):
    """Per-launch DRAM bytes from the committed ncu capture, if one matches this shape."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            t = json.load(f)
        return t.get(f"{B}x{A}x{O}")
    except Exception:
        return None


def kernel_name(A, O, B):
    if A == 3 and O <= 6:
        return "mn::step_team_kernel" if B <= 32768 else "mn::step_env_kernel"
    return "mn::step_team_kernel" if (A, O) == (8, 16) else "mn::step_kernel"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML during the timed region.

    The thread is created and parked BEFORE the region and released by arm() only once every step
    of the region has been enqueued: the samples are taken while the GPU executes those steps, and
    neither a thread start-up nor an NVML call (driver locks, the GIL) competes with the launch loop
    -- at the driver's --steps 20 the region is 1.3 ms long and a first sample taken inside the
    loop cost 3-5 % of it."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self._go = threading.Event()
        self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._h = None

    def run(self):
        if self._h is None:
            return
        nv = self._nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        self._go.wait()
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004 if self.samples else 0.0002)    # (a failed first call is retried at once)

    def arm(self):
        self._go.set()

    def stop(self):
        self._halt.set()
        self._go.set()
        self.join(timeout=1.0)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "samples": len(s), "reasons": sorted(self.reasons)}


def make_action_pool(B, A, n, device, seed=1234, angle=0.2):
    """SURVEY.md section 8(d): turn angle ~ U(-angle, angle) -- 0.2 rad = "policy-like" (agents make
    progress, collide, reset), pi = trig stress -- and acceleration ~ U(-0.5, 0.5)."""
    g = torch.Generator().manual_seed(seed)
    pool = []
    for _ in range(n):
        ang = (torch.rand(B, A, generator=g) * 2 - 1) * angle
        acc = (torch.rand(B, A, generator=g) * 2 - 1) * 0.5
        pool.append(torch.stack([ang, acc], dim=2).contiguous().to(device))
    return pool


def env_params(B, A, O, device, offset=0):
    import marlnav_b200 as mb
    if A == 3:
        p = mb.default_env_params(B, A, O, sampling_style='policy', device=device)
    else:
        p = mb.template_env_params(B, A, O, device=device)
    p['seed'] = 0
    p['env_id_offset'] = offset
    return p


def workload_config(args, B_local):
    return {"workload": f"{B_local} envs x {args.agents} agents x {args.obstacles} obstacles per GPU, "
                        "random policy-like actions, auto-reset, episode_len 200 "
                        "(BASELINE.json configs[3]; configs[4] with --agents 8 --obstacles 16)",
            "envs_per_gpu": B_local, "num_agents": args.agents, "num_obstacles": args.obstacles,
            "action_pool": 16, "action_angle_range": args.angle,
            "l2_policy": "working set per step (states+actions+obs) exceeds the 126 MB L2"
            if B_local * algorithmic_bytes(args.agents, args.obstacles) > 2 * 126e6 else
            "working set may fit in L2 -- not an HBM number"}


# ----------------------------------------------------------------------------- CPU arm

def use_all_host_threads():
    try:        # torchrun exports OMP_NUM_THREADS=1; the CPU arm uses every core it may run on
        torch.set_num_threads(len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return torch.get_num_threads()


def load_reference():
    """The unmodified reference package from baseline/_ref (vendored by __graft_entry__.build();
    /root/reference itself does not exist on the GPU box).  matplotlib / PyQt5 are not installed and
    marlnav/utils.py imports matplotlib at module top: stub modules, nothing of the step uses them."""
    if not os.path.isdir(os.path.join(REF_DIR, "marlnav")):
        return None
    from unittest import mock
    for name in ('matplotlib', 'matplotlib.pyplot', 'matplotlib.animation'):
        sys.modules.setdefault(name, mock.MagicMock())
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    try:
        import marlnav.environment as env_mod
        return env_mod
    except Exception:
        return None


def reference_env(env_mod, B, A, O, device):
    """marlnav.environment.Env on the reference's own param dict (utils.py:257-282 restated in
    marlnav_b200.params: data only, no code of ours on the path)."""
    import marlnav_b200 as mb
    p = mb.default_env_params(B, A, O, sampling_style='policy', device=device)
    p['init'] = dict(p['init'], device=device)
    torch.manual_seed(0)
    return env_mod.Env(p)


def time_env_steps(env, pool, steps, warmup, sync=None):
    for i in range(warmup):
        env.step(pool[i % len(pool)])
    if sync:
        sync()
    t0 = time.perf_counter()
    for i in range(steps):
        env.step(pool[i % len(pool)])
    if sync:
        sync()
    return time.perf_counter() - t0


def time_cpu_reference(A, O, B, steps=None, warmup=1, budget_s=12.0):
    """Times the reference step on the host cores.  -> dict(value, cores, kind, sample, steps, ms, envs).
    kind "reference": the real marlnav Env; "port": oracle.TorchPortEnv (same op sequence and bits)
    when the reference is absent or cannot express the shape (its initialiser is 3-agent only)."""
    cores = use_all_host_threads()
    env_mod = load_reference() if A == 3 else None
    pool = make_action_pool(B, A, 4, 'cpu')
    if env_mod is not None:
        env, kind, what = reference_env(env_mod, B, A, O, 'cpu'), "reference", \
            "marlnav.environment.Env.step (unmodified reference, baseline/_ref)"
    else:
        from oracle import oracle as orc
        p = orc.default_env_params(B, A, O)
        if A != 3:
            p['init'] = dict(p['init'], init_method='template', agent_template=orc.ring_template(A))
        env, kind, what = orc.TorchPortEnv(p, seed=0), "port", \
            ("oracle.TorchPortEnv.step (torch-op port of the reference step: " +
             ("reference absent from baseline/_ref" if A == 3 else "the reference's initialiser is 3-agent only") + ")")
    t0 = time.perf_counter()
    for i in range(max(warmup, 1)):
        env.step(pool[i % 4])
    per = (time.perf_counter() - t0) / max(warmup, 1)
    if steps is None:
        steps = max(3, min(200, int(budget_s / max(per, 1e-6))))
    dt = time_env_steps(env, pool, steps, 0)
    desc = (f"{B} envs x {A} agents x {O} obstacles per step, {steps} timed steps ({dt:.1f} s) of {what}, "
            f"torch {torch.__version__} CPU, {cores} threads of {os.cpu_count()} cpus")
    return dict(value=B * steps / dt, cores=cores, kind=kind, sample=desc, steps=steps, ms=1e3 * dt / steps, envs=B)


def time_cuda_reference(A, O, B, steps=5, warmup=2):
    """BASELINE.md 4.4: the unmodified reference Env on device='cuda' (launch/sync bound)."""
    env_mod = load_reference() if A == 3 else None
    if env_mod is None or not torch.cuda.is_available():
        return {"unavailable": "reference absent from baseline/_ref" if env_mod is None else "no CUDA device"}
    try:
        env = reference_env(env_mod, B, A, O, 'cuda')
        pool = make_action_pool(B, A, 4, 'cuda')
        dt = time_env_steps(env, pool, steps, warmup, sync=torch.cuda.synchronize)
        return {"value": B * steps / dt, "unit": UNIT, "envs": B, "steps": steps, "ms_per_step": 1e3 * dt / steps,
                "what": "marlnav.environment.Env.step (unmodified reference) with params['device']='cuda', wall clock"}
    except Exception as e:                                   # e.g. out of memory at the full batch
        return {"unavailable": f"{type(e).__name__}: {str(e)[:200]}"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    A, O, B = args.agents, args.obstacles, args.envs
    # the full batch per step unless K + W steps of it would not end within a few minutes
    cores = use_all_host_threads()
    probe = time_cpu_reference(A, O, min(B, 65536), steps=1, warmup=1)
    est = (args.steps + max(args.warmup, 1)) * (probe['ms'] * 1e-3) * (B / probe['envs'])
    while est > 240 and B > 65536:
        B //= 2; est /= 2
    r = time_cpu_reference(A, O, B, steps=args.steps, warmup=max(args.warmup, 1))
    cfg = workload_config(args, B)
    if B != args.envs:
        cfg["workload"] = f"SAMPLE of {B} envs per step (the full {args.envs} would exceed the time bound): " + cfg["workload"]
    line = {
        "impl": "reference", "metric": METRIC, "value": r['value'], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r['steps'], "warmup": args.warmup, "ms_per_step": r['ms'], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": r['value'], "unit": UNIT, "cores": cores, "kind": r['kind'], "sample": r['sample']},
        "e2e": {"value": r['value'], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "reference_cuda": time_cuda_reference(A, O, min(B, args.ref_cuda_envs)) if not args.no_ref_cuda else None,
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------- GPU arm

def cuda_time(fn, reps):
    """ms per call of fn(i) over `reps` calls, CUDA events on the current stream."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def shape_record(B, A, O, dev, steps, warmup=20, modes=("step", "step_fused_out", "graph")):
    """One BASELINE configuration, device-resident: ms per step through Env.step (fresh outputs +
    namedtuple, what the reference's callers get), step_fused(out=) (reused buffers) and a StepGraph."""
    import marlnav_b200 as mb
    peak, _ = measured_peak()
    rec = {"envs": B, "num_agents": A, "num_obstacles": O, "kernel": kernel_name(A, O, B)}
    pool = make_action_pool(B, A, 16, dev)
    ws = B * algorithmic_bytes(A, O)
    for mode in modes:
        env = mb.Env(env_params(B, A, O, str(dev)))
        if mode == "graph":
            sg = mb.StepGraph(env, pool * 4)                 # 64 steps per replay
            for _ in range(2):
                sg.replay()
            torch.cuda.synchronize()
            reps = max(2, steps // sg.steps)
            ms = cuda_time(lambda i: sg.replay(), reps) / sg.steps
        else:
            out = env._alloc_outputs()
            f = (lambda i: env.step(pool[i % 16])) if mode == "step" else (lambda i: env.step_fused(pool[i % 16], out=out))
            for i in range(warmup):
                f(i)
            torch.cuda.synchronize()
            ms = cuda_time(f, steps)
        rec[mode] = {"ms_per_step": ms, "value": B / (ms * 1e-3)}
        del env
    best = min(rec[m]["ms_per_step"] for m in modes)
    gbs = ws / (best * 1e-3) / 1e9
    if ws > 2 * 126e6:
        rec["roofline"] = {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                           "traffic": ncu_traffic(A, O, B), "algorithmic_bytes_per_env_step": algorithmic_bytes(A, O)}
    else:
        rec["note"] = "working set fits in the 126 MB L2: not an HBM number"
    return rec


def rollout_record(B, dev, T=250):
    """BASELINE configs[1]: 1024 envs x 3 x 3 with the MAPPO actor (models.py:14-36, random init) and
    critic (models.py:39-56) in the loop, the whole T-step rollout as ONE CUDA graph (RolloutGraph)."""
    import marlnav_b200 as mb
    A, O = 3, 3
    env = mb.Env(env_params(B, A, O, str(dev)))
    max_d = math.sqrt(1500.0 ** 2 + 750.0 ** 2)
    lo = [-math.pi, 0.] + O * [-math.pi] + O * [0.] + (A - 1) * [-math.pi] + (A - 1) * [0.]
    hi = [math.pi, max_d] + O * [math.pi] + O * [max_d] + (A - 1) * [math.pi] + (A - 1) * [max_d]
    env.fuse_io(dict(min_obs=lo, max_obs=hi), dict(min_action=[-math.pi, -0.5], max_action=[math.pi, 0.5]))
    torch.manual_seed(5)
    S, H = env.obs_size, 50
    fc1, mu, std = torch.nn.Linear(S, H), torch.nn.Linear(H, 2), torch.nn.Linear(H, 2)
    c1, c2 = torch.nn.Linear(A * S, H), torch.nn.Linear(H, 1)
    actor = mb.FusedActor({'fc1.weight': fc1.weight, 'fc1.bias': fc1.bias, 'fc_mu.weight': mu.weight,
                           'fc_mu.bias': mu.bias, 'fc_std.weight': std.weight, 'fc_std.bias': std.bias},
                          device=dev, seed=1)
    critic = mb.FusedCritic({'fc1.weight': c1.weight, 'fc1.bias': c1.bias, 'fc2.weight': c2.weight, 'fc2.bias': c2.bias},
                            device=dev)
    rg = mb.RolloutGraph(env, actor, T, critic=critic)
    rg.replay()
    torch.cuda.synchronize()
    ms = cuda_time(lambda i: rg.replay(), 4) / T
    return {"envs": B, "buffer_len": T, "ms_per_iteration": ms, "value": B / (ms * 1e-3),
            "what": "RolloutGraph: {fused actor sample -> fused step} x T with the critic on a parallel branch, one graph launch per rollout"}


def dump_outputs(path, result, seed=0, budget=48 << 20):
    """Writes one Env.step result -- the six Observations fields, rewards, terminated, truncated --
    as float32 DIR/<name>.npy, env rows first.  A batch larger than `budget` bytes is cut to a fixed,
    seeded sample of env rows, the same rows in every array; env_index.npy (float64) lists them."""
    import numpy as np
    fields, rew, term, trunc = result
    arrays = dict(fields._asdict(), rewards=rew, terminated=term, truncated=trunc)
    B = rew.shape[0]
    per_env = 4 * sum(t[0].numel() for t in arrays.values()) + 8
    n = min(B, budget // per_env)
    idx = np.arange(B) if n == B else np.sort(np.random.default_rng(seed).choice(B, n, replace=False))
    rows = torch.from_numpy(idx).to(rew.device)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "env_index.npy"), idx.astype(np.float64))
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.index_select(0, rows).to(torch.float32).cpu().numpy())


def run_ours(args):
    import torch.distributed as dist
    import marlnav_b200 as mb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for --impl ours)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # rank 0 prints ONE JSON line on stdout: NCCL_DEBUG=VERSION (set on the GPU boxes) makes NCCL
        # printf its version banner there, and so does WARN; an explicit INFO/TRACE is left alone
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            del os.environ["NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=dev)

    A, O = args.agents, args.obstacles
    B = args.envs if args.scaling == "weak" else mb.shard_bounds(args.envs, rank, world)[1]
    offset = rank * B if args.scaling == "weak" else mb.shard_bounds(args.envs, rank, world)[0]
    env = mb.Env(env_params(B, A, O, f"cuda:{local_rank}", offset))
    pool = make_action_pool(B, A, 16, dev, angle=args.angle)
    K, W = args.steps, max(args.warmup, 3)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # Bring the device out of any idle P-state before the W warm-up steps (a fresh process starts
    # after seconds of interpreter start-up with the GPU idle, and W short steps are only ~1.5 ms).
    # Plain device copies on scratch tensors, nothing of the workload; --prewarm-s 0 disables it.
    scratch = torch.empty(2, 64 << 20, dtype=torch.float32, device=dev)
    t_ramp = time.perf_counter()
    while time.perf_counter() - t_ramp < args.prewarm_s:
        for _ in range(8):
            scratch[1].copy_(scratch[0])
        torch.cuda.synchronize()
    del scratch
    # ---- headline: the reference-facing Env.step (fresh output tensors every step, models.py:121)
    for i in range(W):
        env.step(pool[i % 16])
    sampler = ClockSampler(local_rank)
    sampler.start()                                  # parked until arm()
    legacy_sampler = os.environ.get("MARLNAV_BENCH_SAMPLER", "") == "legacy"     # A/B of the note above
    barrier()
    stats0 = env.episode_stats.clone()
    torch.cuda.synchronize()
    if legacy_sampler:
        sampler.arm()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K - 1):
        env.step(pool[i % 16])
    last = env.step(pool[(K - 1) % 16])              # kept for --dump-outputs
    e1.record()
    sampler.arm()                                    # the GPU is still executing the K steps
    barrier()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    stats_delta = env.episode_stats.clone() - stats0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    del last
    # the same loop writing into one reused output buffer (what the round-1 line timed)
    out = env._alloc_outputs()
    ms_fused = cuda_time(lambda i: env.step_fused(pool[i % 16], out=out), K) * K
    barrier()

    # ---- end-to-end leg: host actions -> device step -> host outputs, copies timed
    hs = mb.HostStepper(env)
    K2 = max(3, min(K, args.e2e_steps))
    host_pool = [p.cpu().pin_memory() for p in pool[:4]]     # the policy's outputs, in pinned host memory
    for i in range(2):
        hs.step(host_pool[i % 4])
    barrier()
    t0 = time.perf_counter()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    checksum = 0.0
    for i in range(K2):
        hs.step(host_pool[i % 4], sync=True)         # H2D actions -> fused step -> D2H obs/rewards/flags
        checksum += float(hs.rewards_host[0])        # the caller reads the step's result
    f1.record()
    barrier()
    ms_e2e = max(f0.elapsed_time(f1), 1e3 * (time.perf_counter() - t0))
    launch_info = env.launch_info()
    h2d, d2h = hs.h2d_bytes, hs.d2h_bytes
    del hs, env, out

    # ---- strong split of configs[3]: args.strong_envs in total over the ranks, steps in a CUDA graph
    strong = None
    if not args.no_strong and (A, O) == (3, 3):
        off_s, B_s = mb.shard_bounds(args.strong_envs, rank, world)
        env_s = mb.Env(env_params(B_s, A, O, f"cuda:{local_rank}", off_s))
        pool_s = make_action_pool(B_s, A, 16, dev, angle=args.angle)
        out_s = env_s._alloc_outputs()
        for i in range(W):
            env_s.step_fused(pool_s[i % 16], out=out_s)
        barrier()
        ms_eager = cuda_time(lambda i: env_s.step_fused(pool_s[i % 16], out=out_s), 256)
        sg = mb.StepGraph(env_s, pool_s * 4)                  # 64 steps per replay
        for _ in range(2):
            sg.replay()
        barrier()
        reps = 8
        ms_graph = cuda_time(lambda i: sg.replay(), reps) / sg.steps
        barrier()
        strong = [ms_graph, ms_eager, B_s, sg.steps * reps]
        del sg, env_s

    t = torch.tensor([ms, ms_e2e, ms_fused] + (strong[:2] if strong else [0.0, 0.0]), dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        mb.reduce_episode_stats(stats_delta)
    ms, ms_e2e, ms_fused, ms_sg, ms_se = (float(x) for x in t)

    if rank == 0:
        total_envs = B * world
        value = total_envs * K / (ms * 1e-3)
        e2e_value = total_envs * K2 / (ms_e2e * 1e-3)
        peak, peak_src = measured_peak()
        bytes_launch = B * algorithmic_bytes(A, O)
        achieved = bytes_launch / (ms / K * 1e-3) / 1e9
        g, blk, smem, tile = launch_info
        cpu = None
        configs = None
        if world == 1 and not args.no_cpu_baseline:
            r = time_cpu_reference(A, O, args.cpu_envs if A == 3 else 8192, budget_s=args.cpu_budget)
            cpu = {"value": r['value'], "unit": UNIT, "cores": r['cores'], "kind": r['kind'], "sample": r['sample']}
        if not args.no_configs and (A, O) == (3, 3):
            configs = {
                "262144x8x16": shape_record(262144, 8, 16, dev, 200),
                "65536x3x3": shape_record(65536, 3, 3, dev, 500),
                "1024x3x3": dict(shape_record(1024, 3, 3, dev, 2000), rollout=rollout_record(1024, dev)),
                "2x3x3": shape_record(2, 3, 3, dev, 2000),
            }
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(args, B), api="Env.step (fresh outputs + Observations namedtuple per step)",
                           prewarm=f"{args.prewarm_s} s of device copies before the warm-up steps",
                           grid=g, block=blk, smem_bytes=smem, envs_per_cta=tile,
                           agent_steps_per_sec=value * A,
                           step_fused_out_ms_per_step=ms_fused / K,
                           episode_events_in_timed_region=dict(zip(("trunc", "col", "tar"),
                                                                   [int(x) for x in stats_delta.tolist()]))),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic(A, O, B), "peak_source": peak_src,
                         "algorithmic_bytes_per_env_step": algorithmic_bytes(A, O),
                         "kernel": kernel_name(A, O, B),
                         "per": "one launch = one step of one GPU's slice"},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d * world,
                    "d2h_bytes_per_step": d2h * world, "steps": K2, "ms_per_step": ms_e2e / K2,
                    "path": "HostStepper -> marlnav_step_host_f32 (pinned host buffers)"},
            "strong": None if strong is None else {
                "envs_total": args.strong_envs, "envs_per_gpu": strong[2], "steps": strong[3],
                "ms_per_step": ms_sg, "value": args.strong_envs / (ms_sg * 1e-3),
                "launch": "StepGraph: 64 steps per CUDA-graph replay, device-resident reset counter",
                "eager_ms_per_step": ms_se, "eager_value": args.strong_envs / (ms_se * 1e-3),
                "note": "BASELINE.json configs[3]: 1,048,576 envs in total split over the ranks; "
                        "at 8 ranks each slice (131072 envs, 44 MB) is L2-resident"},
            "configs": configs,
            "gpu_launches": K,
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=("ours", "reference"), default="ours")
    ap.add_argument("--envs", type=int, default=1048576, help="envs per GPU (weak) or total (strong)")
    ap.add_argument("--agents", type=int, default=3)
    ap.add_argument("--obstacles", type=int, default=3)
    ap.add_argument("--scaling", choices=("weak", "strong"), default="weak")
    ap.add_argument("--strong-envs", type=int, default=1048576, help="total envs of the strong-split record")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configurations")
    ap.add_argument("--e2e-steps", type=int, default=50)
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU baseline work")
    ap.add_argument("--cpu-envs", type=int, default=262144, help="envs per step of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-cuda-envs", type=int, default=65536, help="batch of the reference-on-CUDA bar")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--angle", type=float, default=0.2,
                    help="turn-angle range of the random actions in rad (SURVEY 8d: 0.2 policy-like, 3.14159 trig stress)")
    ap.add_argument("--prewarm-s", type=float, default=0.5,
                    help="seconds of device copies before the warm-up steps (P-state ramp)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs (rank 0's slice) to DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
