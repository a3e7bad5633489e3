"""The bench's reference arm runs without a GPU (it times the oracle port on the host cores), so its side of the JSON
contract is checked here: ONE line on stdout with the agreed keys, rank 0 only under a multi-process launch.  The GPU
arm's line has the same keys plus ``roofline`` / ``parity_check`` / ``clocks`` (profiles/r02/75_bench.json)."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

from util import rel_err

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, extra_env=None):
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), *args], capture_output=True, text=True, env=env,
                          cwd=REPO, timeout=300)


def run_reference_arm(extra_env=None):
    return run_bench("--impl", "reference", "--config", "C2", "--steps", "2", "--warmup", "1", extra_env=extra_env)


def test_reference_arm_prints_one_contract_line():
    out = run_reference_arm()
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "chebyshev_spmm_steps_per_s" and line["unit"] == "steps/s"
    assert line["n_gpus"] == 1 and line["steps"] == 2 and line["warmup"] == 1
    assert line["higher_is_better"] is True and line["scaling"] == "weak" and line["vs_baseline"] is None
    assert line["dtype"] == "f64" and line["data"] == "synthetic" and "workload" in line["config"]
    assert line["value"] > 0 and abs(line["value"] * line["ms_per_step"] - 1e3) <= 1e-6 * 1e3
    cpu = line["cpu_baseline"]
    assert cpu["kind"] == "port" and cpu["cores"] >= 1 and cpu["value"] == line["value"] and cpu["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0


def test_reference_arm_is_silent_on_other_ranks():
    out = run_reference_arm({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert out.returncode == 0 and out.stdout.strip() == "", out.stdout + out.stderr[-2000:]


@pytest.mark.gpu
def test_steps_sets_the_timed_steps_and_dump_holds_the_moments(gpu_api, tmp_path):
    """``--steps K`` times K steps (K + 1 when an odd K meets a kernel that advances two steps per launch), and
    ``--dump-outputs`` writes the moments of that recursion: those chebyshev_moments returns for the same matrix, seed and
    scale."""
    from bodge_b200 import workloads

    K, W = 7, 3
    out = run_bench("--config", "C2", "--steps", str(K), "--warmup", str(W), "--no-cpu-baseline", "--no-e2e", "--no-plain",
                    "--dump-outputs", str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout)
    assert line["steps"] == K
    assert line["timed_steps"] == (K + 1 if line["run"]["kernel"] == "t2" else K)
    mu = np.load(tmp_path / "moments.npy")
    summed = np.load(tmp_path / "moments_summed.npy")
    assert mu.dtype == summed.dtype == np.float64 and mu.shape[1] == 8
    assert np.array_equal(np.load(tmp_path / "moment_index.npy"), np.arange(len(mu), dtype=np.float64))
    cfg = workloads.CONFIGS["C2"]
    system = gpu_api.Hamiltonian(gpu_api.CubicLattice(cfg["shape"]), device=0)
    system.fill(*cfg["build"](cfg["shape"]))
    want = system.chebyshev_moments(len(mu), vectors=8, seed=1234, scale=system.spectral_bound(), kernel="auto_moments")
    assert rel_err(mu, want) <= 1e-12
    assert rel_err(summed, want.sum(axis=1)) <= 1e-12
