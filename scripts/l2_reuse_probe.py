#!/usr/bin/env python
"""scripts/l2_reuse_probe.py -- does the env state stay in L2 from one step to the next?

    python scripts/l2_reuse_probe.py [--label NAME] [--steps 1000] [--warmup 400] [--rounds 3] [--out FILE]

Times eager ``Env.step_fused(out=)`` per step with CUDA events at B in {131 072, 262 144, 524 288,
786 432, 1 048 576, 1 310 720} x 3 x 3 and at 262 144 x 8 x 16: ``--warmup`` steps first (episode_len
200, so resets run at their steady rate), then ``--rounds`` windows of ``--steps`` steps.  Prints one
JSON line per size (appended to --out when given): the card's name, power limit, current and
maximum SM clock read right after the timing, us per step (median and all rounds) and ns per env.

What it shows without a profiler: the state that carries over between steps is 97 B/env at (3,3)
(states 60, obstacles 24, target 8, step counter 4, terminates 1), the streams -- actions in,
observations, rewards and flags out -- another 174 B/env.  While the whole working set fits the
126 MB L2 the time per env is flat; when a step's traffic no longer fits, a build that revisits the
tiles in the same order every step loses all its reuse at once (ns per env rises), a build that
keeps the state in L2 stays flat until the state alone (~1.3 M envs at (3,3)) outgrows it.
``MARLNAV_B200_LIB`` selects the library build, ``--label`` names it in the output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIZES = [(131072, 3, 3), (262144, 3, 3), (524288, 3, 3), (786432, 3, 3), (1048576, 3, 3), (1310720, 3, 3),
         (262144, 8, 16)]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                               "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # (reported, not fatal: the timings stand on their own)
        return f"unavailable: {e}"


def action_pool(B, A, n=8, angle=0.2, accel=0.5):
    g = torch.Generator().manual_seed(1234)
    return [torch.stack([(torch.rand(B, A, generator=g) * 2 - 1) * angle,
                         (torch.rand(B, A, generator=g) * 2 - 1) * accel], dim=2).contiguous().cuda() for _ in range(n)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--label", default=os.path.basename(os.environ.get("MARLNAV_B200_LIB", "") or "in-tree"))
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=400)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("l2_reuse_probe needs a CUDA device")
    import marlnav_b200 as mb
    for B, A, O in SIZES:
        p = mb.default_env_params(B, A, O, sampling_style='policy') if A == 3 else mb.template_env_params(B, A, O)
        p['seed'] = 1
        env = mb.Env(p)
        out = env._alloc_outputs()
        pool = action_pool(B, A)
        i = 0
        for _ in range(args.warmup):
            env.step_fused(pool[i % len(pool)], out=out)
            i += 1
        times = []
        for _ in range(args.rounds):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                env.step_fused(pool[i % len(pool)], out=out)
                i += 1
            e1.record()
            e1.synchronize()
            times.append(1e3 * e0.elapsed_time(e1) / args.steps)
        us = statistics.median(times)
        line = json.dumps({"label": args.label, "shape": f"{B}x{A}x{O}", "envs": B,
                           "card_power_limit_sm_clock_max_sm_clock": card(),
                           "warmup_steps": args.warmup, "steps_per_round": args.steps,
                           "us_per_step": round(us, 2), "us_per_step_all": [round(t, 2) for t in times],
                           "ns_per_env": round(1e3 * us / B, 4)})
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
        del env, out, pool
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
