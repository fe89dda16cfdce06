"""bench.py's command-line contract on a box without a GPU: the reference arm's JSON line (alone and
under torchrun, where rank 0 alone prints), the product arm refusing to run without CUDA (no CPU
fallback), bad arguments refused; and on the GPU, --dump-outputs against the oracle.  The reference
arm steps the unmodified reference from baseline/_ref when __graft_entry__.build() has vendored it
there, else the oracle's torch-op port -- both CPU paths."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")
SMALL = ["--envs", "2048", "--steps", "2", "--warmup", "1", "--no-ref-cuda"]


def _json_lines(out):
    return [json.loads(l) for l in out.splitlines() if l.startswith("{")]


def _check_reference_line(d, n):
    assert d["impl"] == "reference" and "unavailable" not in d
    assert d["metric"] == "env_steps_per_sec" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == n and d["steps"] == 2 and d["warmup"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None
    assert abs(d["value"] - 2048 / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]
    assert d["config"]["envs_per_gpu"] == 2048 and d["config"]["num_agents"] == 3 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_line():
    r = subprocess.run([sys.executable, BENCH, "--impl", "reference", *SMALL], capture_output=True, text=True,
                       timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = _json_lines(r.stdout)
    assert len(lines) == 1
    _check_reference_line(lines[0], 1)


def test_reference_arm_under_torchrun_prints_once():
    """launched with torchrun for N > 1: every rank exits 0, rank 0 alone runs and prints"""
    import socket
    with socket.socket() as s:                  # a free port: the host may run other jobs
        s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), BENCH, "--impl", "reference",
                        "--gpus", "2", *SMALL], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = _json_lines(r.stdout)
    assert len(lines) == 1
    _check_reference_line(lines[0], 2)


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a box without CUDA")
def test_product_arm_refuses_without_cuda():
    r = subprocess.run([sys.executable, BENCH, "--steps", "2", "--warmup", "1"], capture_output=True, text=True,
                       timeout=300, cwd=ROOT)
    assert r.returncode != 0
    assert not _json_lines(r.stdout)
    assert "CUDA" in (r.stderr + r.stdout)


def test_bad_arguments_are_refused():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, BENCH, *extra], capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert r.returncode == 2 and not _json_lines(r.stdout), r.stderr[-2000:]


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path, oracle):
    """--dump-outputs writes what the K-th timed Env.step returned: the C oracle stepped through bench's
    W warm-up and K timed actions gives the same bits."""
    import numpy as np
    import bench
    from helpers import assert_bits_equal
    B, W, K = 4096, 3, 5
    r = subprocess.run([sys.executable, BENCH, "--envs", str(B), "--steps", str(K), "--warmup", str(W),
                        "--prewarm-s", "0", "--no-configs", "--no-strong", "--no-cpu-baseline", "--e2e-steps", "3",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert len(_json_lines(r.stdout)) == 1 and _json_lines(r.stdout)[0]["steps"] == K
    pool = bench.make_action_pool(B, 3, 16, "cpu")
    oe = oracle.OracleEnv(bench.env_params(B, 3, 3, "cpu"), seed=0)
    for act in pool[:W] + pool[:K]:
        fields, rew, term, trunc = oe.step(act.numpy())
    want = dict(fields._asdict(), rewards=rew, terminated=term, truncated=trunc)
    assert np.array_equal(np.load(tmp_path / "env_index.npy"), np.arange(B, dtype=np.float64))
    for name, a in want.items():
        got = np.load(tmp_path / f"{name}.npy")
        assert got.dtype == np.float32
        assert_bits_equal(name, got, np.ascontiguousarray(a, np.float32))
