#!/usr/bin/env python
"""scripts/final_obs_probe.py -- what asking for final observations costs on one GPU.

    python scripts/final_obs_probe.py [--rounds 3] [--steps 200] [--warmup 400] [--replays 5]
                                      [--out FILE]

One JSON line (also written to --out, default profiles/r3_final_obs_probe.json): the card's name,
power limit and max SM clock (read in this run), and, measured interleaved in this one process
(round r times every leg before round r+1 starts; medians over rounds):
  * eager ``Env.step_fused`` us per step without and with ``final_obs``, float32 and float16, at
    1 048 576 x 3 x 3 (thread-per-env kernel), 16 384 x 3 x 3 (thread-per-agent team of 3) and
    262 144 x 8 x 16.  Two twin envs per shape and dtype, each stepped ``--warmup`` times first so
    that resets run at their steady rate (episode_len 200), outputs into preallocated buffers,
    CUDA events around ``--steps`` steps;
  * ``RolloutGraph`` replay time at 1 024 x 3 x 3, buffer_len 250, ``FusedActor`` + ``FusedCritic``,
    without and with ``final_obs`` (which steps through the actor and ``step_fused`` as two launches
    and adds the critic over the final observations);
  * ``gae`` against ``discounted_returns`` at T = 1 000, B = 1 024: us per call of the Python
    functions (their input conversions and output allocations included).
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

H = 50


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # (reported, not fatal: the timings stand on their own)
        q = f"unavailable: {e}"
    return name, q


def io_params(A, O):
    max_d = math.sqrt(1500.0 ** 2 + 750.0 ** 2)
    lo = [-math.pi, 0.] + O * [-math.pi] + O * [0.] + (A - 1) * [-math.pi] + (A - 1) * [0.]
    hi = [math.pi, max_d] + O * [math.pi] + O * [max_d] + (A - 1) * [math.pi] + (A - 1) * [max_d]
    return dict(min_obs=lo, max_obs=hi), dict(min_action=[-math.pi, -0.5], max_action=[math.pi, 0.5])


def make_env(B, A, O, dtype, io=False):
    import marlnav_b200 as mb
    p = mb.default_env_params(B, A, O, sampling_style='policy') if A == 3 else mb.template_env_params(B, A, O)
    p['seed'] = 1
    p['obs_dtype'] = dtype
    env = mb.Env(p)
    if io:
        env.fuse_io(*io_params(A, O))
    return env


class Stepper:
    """One env stepped eagerly into preallocated outputs, with or without a final_obs buffer."""

    def __init__(self, B, A, O, dtype, final, pool):
        self.env, self.pool, self.i = make_env(B, A, O, dtype), pool, 0
        self.out = self.env._alloc_outputs()
        self.fin = torch.empty_like(self.out[0]) if final else None

    def step(self):
        self.env.step_fused(self.pool[self.i % len(self.pool)], out=self.out, final_obs=self.fin)
        self.i += 1

    def time(self, n):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            self.step()
        e1.record()
        e1.synchronize()
        return 1e3 * e0.elapsed_time(e1) / n


def action_pool(B, A, n=8, angle=0.2, accel=0.5):
    g = torch.Generator().manual_seed(1234)
    return [torch.stack([(torch.rand(B, A, generator=g) * 2 - 1) * angle,
                         (torch.rand(B, A, generator=g) * 2 - 1) * accel], dim=2).contiguous() for _ in range(n)]


def timed(fn, n):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def weights(S, A):
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


def summary(xs, nd):
    return {"median": round(statistics.median(xs), nd), "all": [round(x, nd) for x in xs]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=400)
    ap.add_argument("--replays", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_final_obs_probe.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("final_obs_probe needs a CUDA device")
    import marlnav_b200 as mb
    name, power = card()
    out = {"card": name, "power_limit_and_max_sm_clock": power, "rounds": args.rounds, "steps_per_round": args.steps,
           "warmup_steps": args.warmup, "step_fused_us": {}, "rollout_graph_ms_per_replay": {}, "gae_vs_returns_us": {}}

    for B, A, O in ((1048576, 3, 3), (16384, 3, 3), (262144, 8, 16)):
        key = f"{B}x{A}x{O}"
        pool = [a.cuda() for a in action_pool(B, A)]
        for dtype in (torch.float32, torch.float16):
            legs = {"plain": Stepper(B, A, O, dtype, False, pool), "final_obs": Stepper(B, A, O, dtype, True, pool)}
            for s in legs.values():
                for _ in range(args.warmup):
                    s.step()
            times = {k: [] for k in legs}
            for _ in range(args.rounds):
                for k, s in legs.items():
                    times[k].append(s.time(args.steps))
            res = {k: summary(v, 2) for k, v in times.items()}
            res["resets_per_step"] = round(
                float(legs["final_obs"].env.episode_stats[:2].sum()) / legs["final_obs"].i, 1)
            out["step_fused_us"].setdefault(key, {})[str(dtype).replace("torch.", "")] = res
            del legs
            torch.cuda.empty_cache()
        del pool

    B, A, O, T = 1024, 3, 3, 250
    aw, cw = weights(2 + 2 * O + 2 * (A - 1), A)
    graphs = {}
    for k, fin in (("plain", False), ("final_obs", True)):
        env = make_env(B, A, O, torch.float32, io=True)
        graphs[k] = mb.RolloutGraph(env, mb.FusedActor(aw, seed=3), T, critic=mb.FusedCritic(cw), final_obs=fin)
    times = {k: [] for k in graphs}
    for _ in range(args.rounds):
        for k, g in graphs.items():
            times[k].append(timed(g.replay, args.replays))
    out["rollout_graph_ms_per_replay"][f"{B}x{A}x{O}_T{T}"] = {k: summary(v, 4) for k, v in times.items()}
    del graphs
    torch.cuda.empty_cache()

    T, B = 1000, 1024
    g = torch.Generator().manual_seed(0)
    r = torch.randn(T, B, generator=g).cuda()
    v, fv = torch.randn(T, B, 1, generator=g).cuda(), torch.randn(T, B, 1, generator=g).cuda()
    te, tr = (torch.rand(T, B, generator=g) < 0.02).cuda(), (torch.rand(T, B, generator=g) < 0.02).cuda()
    legs = {"discounted_returns": lambda: mb.discounted_returns(r, te | tr, 0.99),
            "gae": lambda: mb.gae(r, v, te, tr, 0.99, 0.95, final_values=fv, last_values=v[-1])}
    times = {k: [] for k in legs}
    for _ in range(args.rounds):
        for k, fn in legs.items():
            times[k].append(1e3 * timed(fn, 50))
    out["gae_vs_returns_us"][f"T{T}_B{B}"] = {k: summary(t, 2) for k, t in times.items()}

    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
