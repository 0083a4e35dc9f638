"""bench.py's command line. Without a GPU: the reference arm (`--impl reference`: the CPU restatement of mcmc.js on the host cores)
prints ONE JSON line with the keys every bench line carries, for the same metric / config / unit as the GPU arm; the GPU arm refuses
to run without a GPU instead of falling back to anything. On a GPU: --dump-outputs writes the draws of the last timed step."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, timeout=240):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, capture_output=True, text=True, timeout=timeout)


def test_reference_arm_prints_the_contract_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["metric"].startswith("posterior draws/sec") and d["unit"] == "draws/s" and d["higher_is_better"] is True
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert "config 2" in d["config"]["workload"] and "model" not in d["config"]
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "draws per step" in cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_gpu_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return                                       # on a GPU box the arm itself is what the driver runs
    r = _run(["--steps", "1", "--warmup", "3", "--no-cpu"], timeout=120)
    assert r.returncode != 0
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]      # no number without the CUDA path


def test_bad_steps_and_dump_outputs_for_the_reference_arm_are_refused(tmp_path):
    r = _run(["--steps", "0"], timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr
    r = _run(["--impl", "reference", "--dump-outputs", str(tmp_path / "out")], timeout=120)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_dump_outputs_are_the_draws_of_the_last_timed_step(tmp_path, gpu_pkg):
    """--dump-outputs writes what the last timed step drew: the arrays sample() returns for the same sweeps of the same chains, and
    the same values again when bench.py runs a second time with the same arguments."""
    import numpy as np
    import models
    from conftest import config2_data
    args = ["--chains", "4096", "--iters", "10", "--burn", "20", "--steps", "2", "--warmup", "1", "--no-cpu"]
    for run in ("a", "b"):
        r = _run(args + ["--dump-outputs", str(tmp_path / run)], timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
        assert d["steps"] == 2 and d["warmup"] == 1
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("mu", "sigma")}
    assert sorted(os.listdir(tmp_path / "a")) == ["mu.npy", "sigma.npy"]
    for n, a in got.items():
        assert a.dtype == np.float64 and a.shape == (10, 4096), (n, a.dtype, a.shape)
        assert np.array_equal(a, np.load(tmp_path / "b" / f"{n}.npy")), n
    s = gpu_pkg.mcmc.AmwgSampler(models.PARAMS_NORM, models.norm_post_readme(gpu_pkg.ld), config2_data().tolist(), {"chains": 4096, "seed": 0})
    s.burn(20)
    for _ in range(1 + 2):                              # warm-up + timed steps
        want = s.sample(10)
    for n, a in got.items():
        assert np.array_equal(a, want[n]), n
