"""bench.py's contract: the reference arm prints ONE JSON line with the agreed keys, the product arm
refuses to run without CUDA (no CPU fallback), ``--steps`` is the number of timed steps, and
``--dump-outputs`` writes what the last timed step computed, the same from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, gpu=False):
    env = dict(os.environ) if gpu else dict(os.environ, OMP_NUM_THREADS="4", CUDA_VISIBLE_DEVICES="")
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, env=env,
                          capture_output=True, text=True, timeout=600)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "uq_sample_passes_per_sec"
    assert d["unit"] == "sample*members/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["config"]["workload"] == "ensemble16x512_1M"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] and "sample" in d["cpu_baseline"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None


def _dumped(d):
    return {name: np.load(os.path.join(d, name + ".npy")) for name in ("mean", "std")}


def test_reference_arm_dumps_the_same_outputs_from_run_to_run(tmp_path):
    runs = []
    for i in range(2):
        out = str(tmp_path / f"run{i}")
        r = _run("--impl", "reference", "--steps", "2", "--warmup", "1", "--dump-outputs", out)
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads(r.stdout.strip())
        assert d["steps"] == 2
        runs.append(_dumped(out))
    n = int(d["config"]["cpu_sample"].split()[0])
    for name, a in runs[0].items():
        assert a.dtype == np.float32 and a.shape == (n, 1), (name, a.dtype, a.shape)
        assert np.isfinite(a).all()
        np.testing.assert_array_equal(a, runs[1][name])


def test_steps_below_one_are_refused():
    r = _run("--impl", "reference", "--steps", "0")
    assert r.returncode != 0 and "--steps" in r.stderr


@pytest.mark.gpu
def test_product_arm_dumps_what_the_last_timed_step_computed(tmp_path):
    """Two runs with the same arguments time the same seeded inputs; the dumped (mean, std) agree
    up to the order of floating-point sums and stay within the bench's own bf16 parity bound."""
    runs = []
    for i in range(2):
        out = str(tmp_path / f"run{i}")
        r = _run("--workload", "ensemble32x128_4M", "--steps", "3", "--warmup", "1",
                 "--no-cpu-baseline", "--no-fp32-leg", "--no-metric-kernels", "--dump-outputs", out,
                 gpu=True)
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads(r.stdout.strip())
        assert d["steps"] == 3 and d["parity_max_err"]["bf16"]["max_err_of_scale"] <= 1e-2
        runs.append(_dumped(out))
    for name, a in runs[0].items():
        assert a.dtype == np.float32 and a.shape == (1 << 22, 1), (name, a.dtype, a.shape)
        assert np.isfinite(a).all()
        scale = float(np.abs(runs[0]["mean"]).max() + np.abs(runs[0]["std"]).max())
        np.testing.assert_allclose(a, runs[1][name], rtol=0, atol=1e-6 * scale)


def test_product_arm_fails_loudly_without_a_gpu():
    r = _run("--steps", "1", "--warmup", "1")
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stderr + r.stdout)
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]
