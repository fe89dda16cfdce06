#!/usr/bin/env python
"""scripts/rollout_dtype_probe.py -- what 16-bit rollout observation buffers cost or buy on one GPU.

    python scripts/rollout_dtype_probe.py [--rounds 3] [--replays 5] [--launches 200]
                                          [--dtypes float32,float16,bfloat16] [--out FILE]

One JSON line (also written to --out, default profiles/r3_rollout_dtype_probe.json): the card's name,
power limit and max SM clock (read in this run), and per observation dtype, measured interleaved in
this one process (round r times every dtype before round r+1 starts; medians over rounds):
  * ``RolloutGraph`` replay time with ``FusedActor`` + ``FusedCritic`` (the reference's 12 -> 50 -> 2
    actor and 36 -> 50 -> 1 critic), buffer_len 250, at 1 024, 16 384 and 262 144 envs x 3 x 3:
    ms per replay and us per env-step iteration, CUDA events around ``--replays`` replays;
  * eager ``Env.act_step_fused`` us per launch at 1 048 576 x 3 x 3, ping-ponging two observation
    buffers as a rollout does, CUDA events around ``--launches`` launches;
  * the rollout buffer's bytes: ``torch.cuda.max_memory_allocated`` growth around one
    ``collect_rollout`` (1 024 envs x 3 x 3, buffer_len 1 000, the reference's ``-bl``), next to the
    bytes computed from the buffer shapes.
The float32 leg passes no argument the float32-only API lacks, so ``--dtypes float32`` runs on
builds without 16-bit rollouts too (A/B of the float32 path).
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NAMES = {"float32": torch.float32, "float16": torch.float16, "bfloat16": torch.bfloat16}
A, O, H = 3, 3, 50


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # (reported, not fatal: the timings stand on their own)
        q = f"unavailable: {e}"
    return name, q


def io_params():
    max_d = math.sqrt(1500.0 ** 2 + 750.0 ** 2)
    lo = [-math.pi, 0.] + O * [-math.pi] + O * [0.] + (A - 1) * [-math.pi] + (A - 1) * [0.]
    hi = [math.pi, max_d] + O * [math.pi] + O * [max_d] + (A - 1) * [math.pi] + (A - 1) * [max_d]
    return dict(min_obs=lo, max_obs=hi), dict(min_action=[-math.pi, -0.5], max_action=[math.pi, 0.5])


def weights(S):
    g = torch.Generator().manual_seed(0)
    actor = {'fc1.weight': torch.empty(H, S), 'fc_mu.weight': torch.empty(2, H), 'fc_std.weight': torch.empty(2, H)}
    for v in actor.values():
        torch.nn.init.orthogonal_(v, generator=g)
    actor.update({'fc1.bias': torch.rand(H, generator=g) * 0.2 - 0.1, 'fc_mu.bias': torch.rand(2, generator=g) - 0.5,
                  'fc_std.bias': torch.rand(2, generator=g) - 0.5})
    fc1, fc2 = torch.nn.Linear(A * S, H), torch.nn.Linear(H, 1)
    critic = {'fc1.weight': fc1.weight.detach(), 'fc1.bias': fc1.bias.detach(),
              'fc2.weight': fc2.weight.detach(), 'fc2.bias': fc2.bias.detach()}
    return actor, critic


def make_env(B, dtype):
    import marlnav_b200 as mb
    p = mb.default_env_params(B, A, O, sampling_style='policy')
    p['seed'] = 1
    if dtype != torch.float32:
        p['obs_dtype'] = dtype
    env = mb.Env(p)
    env.fuse_io(*io_params())
    return env


def dtype_kw(dtype):
    return {} if dtype == torch.float32 else {"obs_dtype": dtype}


def rollout_graph(B, dtype, T, aw, cw):
    import marlnav_b200 as mb
    env = make_env(B, dtype)
    return mb.RolloutGraph(env, mb.FusedActor(aw, seed=3), T, critic=mb.FusedCritic(cw), **dtype_kw(dtype))


def time_replays(rg, n):
    rg.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        rg.replay()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


class ActStep:
    """Eager fused act+step launches on two ping-ponged observation buffers."""

    def __init__(self, B, dtype, aw):
        import marlnav_b200 as mb
        self.env, self.actor, self.dtype = make_env(B, dtype), mb.FusedActor(aw, seed=3), dtype
        env, dev, S = self.env, self.env.device, self.env.obs_size
        mean, scale = env._io_tensors[0], env._io_tensors[1]
        obs0 = ((env.observations_fused().float() - mean) / scale).to(dtype)
        self.obs = [obs0, torch.empty(B, A, S, dtype=dtype, device=dev)]
        self.out = (torch.empty(B * A, 2, device=dev), torch.empty(B * A, device=dev), None,
                    torch.empty(B, device=dev), torch.empty(B, dtype=torch.uint8, device=dev),
                    torch.empty(B, dtype=torch.uint8, device=dev))
        self.i = 0

    def launch(self):
        src, dst = self.obs[self.i & 1], self.obs[(self.i + 1) & 1]
        out = self.out[:2] + (dst,) + self.out[3:]
        self.env.act_step_fused(self.actor, src, out, **dtype_kw(self.dtype))
        self.i += 1

    def time(self, n, warmup=10):
        for _ in range(warmup):
            self.launch()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            self.launch()
        e1.record()
        e1.synchronize()
        return 1e3 * e0.elapsed_time(e1) / n


def buffer_bytes(B, T, dtype, aw, cw):
    """(measured peak growth, bytes from the shapes) of one collect_rollout with a critic."""
    import marlnav_b200 as mb
    env = make_env(B, dtype)
    actor, critic = mb.FusedActor(aw, seed=3), mb.FusedCritic(cw)
    mb.collect_rollout(env, actor, 2, critic=critic, **dtype_kw(dtype))       # lazy kernel attributes
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    buf = mb.collect_rollout(env, actor, T, critic=critic, **dtype_kw(dtype))
    torch.cuda.synchronize()
    measured = torch.cuda.max_memory_allocated() - base
    S = env.obs_size
    shapes = {"obs_all": (T + 1) * B * A * S * dtype.itemsize, "actions": T * B * A * 2 * 4,
              "log_probs": T * B * A * 4, "rewards": T * B * 4, "values": T * B * 4,
              "terminated_truncated": 2 * T * B, "done": T * B}
    del buf
    return measured, shapes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--replays", type=int, default=5)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--buffer-len", type=int, default=250)
    ap.add_argument("--dtypes", default="float32,float16,bfloat16")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_rollout_dtype_probe.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rollout_dtype_probe needs a CUDA device")
    dtypes = [NAMES[d] for d in args.dtypes.split(",")]
    dn = lambda d: str(d).replace("torch.", "")
    name, power = card()
    S = 2 + 2 * O + 2 * (A - 1)
    aw, cw = weights(S)
    T = args.buffer_len
    out = {"card": name, "power_limit_and_max_sm_clock": power, "rounds": args.rounds, "buffer_len": T,
           "replays_per_round": args.replays, "launches_per_round": args.launches,
           "rollout_graph_ms_per_replay": {}, "rollout_graph_us_per_step": {}, "act_step_fused_us": {},
           "rollout_buffer_bytes": {}}
    for B in (1024, 16384, 262144):
        key = f"{B}x{A}x{O}"
        graphs = {d: rollout_graph(B, d, T, aw, cw) for d in dtypes}
        times = {d: [] for d in dtypes}
        for _ in range(args.rounds):
            for d in dtypes:
                times[d].append(time_replays(graphs[d], args.replays))
        for d in dtypes:
            ms = statistics.median(times[d])
            out["rollout_graph_ms_per_replay"].setdefault(key, {})[dn(d)] = {
                "median": round(ms, 4), "all": [round(t, 4) for t in times[d]]}
            out["rollout_graph_us_per_step"].setdefault(key, {})[dn(d)] = round(1e3 * ms / T, 3)
        del graphs
        torch.cuda.empty_cache()
    B = 1048576
    key = f"{B}x{A}x{O}"
    steppers = {d: ActStep(B, d, aw) for d in dtypes}
    times = {d: [] for d in dtypes}
    for _ in range(args.rounds):
        for d in dtypes:
            times[d].append(steppers[d].time(args.launches))
    for d in dtypes:
        out["act_step_fused_us"].setdefault(key, {})[dn(d)] = {
            "median": round(statistics.median(times[d]), 2), "all": [round(t, 2) for t in times[d]]}
    del steppers
    torch.cuda.empty_cache()
    B, TB = 1024, 1000
    key = f"{B}x{A}x{O}_T{TB}"
    for d in dtypes:
        measured, shapes = buffer_bytes(B, TB, d, aw, cw)
        out["rollout_buffer_bytes"].setdefault(key, {})[dn(d)] = {
            "max_memory_allocated_growth": measured, "from_shapes_total": sum(shapes.values()),
            "from_shapes": shapes}
        torch.cuda.empty_cache()
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
