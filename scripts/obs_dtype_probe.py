#!/usr/bin/env python
"""scripts/obs_dtype_probe.py -- what 16-bit observations (params['obs_dtype']) buy on one GPU.

    python scripts/obs_dtype_probe.py [--steps 1000] [--rounds 3] [--host-steps 30]

One JSON line: the card's name and power limit (read in this run), and per observation dtype
(float32, float16, bfloat16), measured interleaved in this one process (round r times every dtype
before round r+1 starts; the median over rounds is reported):
  * eager ``Env.step`` us/step at 1,048,576 x 3 x 3 and at 262,144 x 8 x 16, CUDA events around
    ``--steps`` steps after a warm-up;
  * ``HostStepper`` ms/step at 1,048,576 x 3 x 3 (pinned host actions in, pinned host
    observations / rewards / flags out, every step synchronised);
  * the algorithmic bytes per env-step (every tensor read once and written once; observations
    at 2 bytes for the 16-bit types) and the resulting share of the 6 555.8 GB/s HBM peak measured
    on this project's B200.
The working sets (336 MB at 1M x 3 x 3, 543 MB at 262144 x 8 x 16) are larger than the 126 MB L2.
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

PEAK_GBS = 6555.8          # HBM bandwidth measured on the B200 (DESIGN.md section 2)
DTYPES = (torch.float32, torch.float16, torch.bfloat16)


def algorithmic_bytes(A, O, esz):
    """bench.py's per-env-step bytes with the observations at `esz` bytes per element."""
    S = 2 + 2 * O + 2 * (A - 1)
    rd = 20 * A + 8 * A + 8 * O + 8 + 4 + 1
    wr = 20 * A + 4 + 1 + esz * A * S + 4 + 1 + 1
    return rd + wr


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # (reported, not fatal: the timings stand on their own)
        q = f"unavailable: {e}"
    return name, q


def make_env(B, A, O, dtype):
    import marlnav_b200 as mb
    p = mb.default_env_params(B, A, O, sampling_style='policy') if A == 3 else mb.template_env_params(B, A, O)
    p['seed'] = 1
    p['obs_dtype'] = dtype
    return mb.Env(p)


def action_pool(B, A, n=16, seed=0):
    g = torch.Generator().manual_seed(seed)
    return [torch.stack([(torch.rand(B, A, generator=g) * 2 - 1) * 0.2,
                         (torch.rand(B, A, generator=g) * 2 - 1) * 0.5], dim=2).contiguous() for _ in range(n)]


def time_steps(env, pool, steps, warmup=20):
    for i in range(warmup):
        env.step(pool[i % len(pool)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        env.step(pool[i % len(pool)])
    e1.record()
    e1.synchronize()
    return 1e3 * e0.elapsed_time(e1) / steps


def time_host(hs, host_pool, steps):
    import time
    for i in range(3):
        hs.step(host_pool[i % len(host_pool)])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        hs.step(host_pool[i % len(host_pool)], sync=True)
    return 1e3 * (time.perf_counter() - t0) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--host-steps", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("obs_dtype_probe needs a CUDA device")
    import marlnav_b200 as mb
    name, power = card()
    shapes = [(1048576, 3, 3), (262144, 8, 16)]
    out = {"card": name, "power_limit_and_max_sm_clock": power, "peak_gbs": PEAK_GBS, "steps": args.steps,
           "rounds": args.rounds, "step_us": {}, "host_ms": {}, "bytes_per_env_step": {}, "share_of_peak": {}}
    for B, A, O in shapes:
        key = f"{B}x{A}x{O}"
        pool = [a.cuda() for a in action_pool(B, A)]
        envs = {d: make_env(B, A, O, d) for d in DTYPES}
        times = {d: [] for d in DTYPES}
        for _ in range(args.rounds):
            for d in DTYPES:
                times[d].append(time_steps(envs[d], pool, args.steps))
        for d in DTYPES:
            dn = str(d).replace("torch.", "")
            us = statistics.median(times[d])
            nbytes = algorithmic_bytes(A, O, d.itemsize)
            out["step_us"].setdefault(key, {})[dn] = {"median": round(us, 2), "all": [round(t, 2) for t in times[d]]}
            out["bytes_per_env_step"].setdefault(key, {})[dn] = nbytes
            out["share_of_peak"].setdefault(key, {})[dn] = round(nbytes * B / (us * 1e-6) / 1e9 / PEAK_GBS, 4)
        del envs, pool
        torch.cuda.empty_cache()
    B, A, O = shapes[0]
    key = f"{B}x{A}x{O}"
    host_pool = [a.pin_memory() for a in action_pool(B, A, n=4)]
    steppers = {d: mb.HostStepper(make_env(B, A, O, d)) for d in DTYPES}
    htimes = {d: [] for d in DTYPES}
    for _ in range(args.rounds):
        for d in DTYPES:
            htimes[d].append(time_host(steppers[d], host_pool, args.host_steps))
    for d in DTYPES:
        dn = str(d).replace("torch.", "")
        out["host_ms"].setdefault(key, {})[dn] = {"median": round(statistics.median(htimes[d]), 3),
                                                  "all": [round(t, 3) for t in htimes[d]],
                                                  "d2h_bytes_per_step": steppers[d].d2h_bytes}
        steppers[d].close()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
