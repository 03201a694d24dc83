"""bench.py's reference arm runs without a GPU: check the JSON line the driver parses (keys, units, the
`impl`, `cpu_baseline` and `e2e` objects of the tier's contract) on a small mesh.  Also --dump-outputs: its size
cap and sample on the host, and in the GPU tier that its files are what the timed step returns."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra, env=None):
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1", "--factor", "1", "--scenarios", "3", "--solve-scenarios", "0"] + extra, cwd=ROOT, env=e, capture_output=True,
                         text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    return out.stdout.strip().splitlines()


def test_reference_arm_prints_the_contract_line():
    lines = _run([])
    assert len(lines) == 1
    b = json.loads(lines[0])
    assert b["impl"] == "reference" and b["metric"] == "fd_jacobian_plus_residual_evals_per_s"
    assert b["unit"] == "evals/s" and b["higher_is_better"] is True and b["scaling"] == "weak"
    # the arm honours the driver's --steps / --warmup / --scenarios
    assert b["n_gpus"] == 1 and b["steps"] == 2 and b["warmup"] == 1 and b["dtype"] == "f64" and b["data"] == "synthetic"
    assert b["config"]["scenarios_per_gpu"] == 3
    assert b["value"] > 0 and b["ms_per_step"] > 0 and b["vs_baseline"] is None and b["gpu_launches"] == 0
    assert "workload" in b["config"] and "model" not in b["config"]
    assert b["solves"] is None and b["solves_per_hour"] is None  # the solve leg (minutes of CPU work) is switched off here
    cb = b["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == b["value"] and cb["sample"]
    assert b["e2e"] == {"value": b["value"], "unit": b["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # value = evaluations of the step / time of the step
    evals = b["config"]["scenarios_per_gpu"] * b["config"]["evals_per_scenario_step"]
    assert abs(b["pairs_per_s"] - b["config"]["scenarios_per_gpu"] / (b["ms_per_step"] * 1e-3)) <= 1e-6 * b["pairs_per_s"]
    assert abs(b["value"] - evals / (b["ms_per_step"] * 1e-3)) <= 1e-6 * b["value"]


def test_dump_outputs_fits_the_budget_and_repeats(tmp_path, monkeypatch):
    """--dump-outputs: float64 files within the budget; an output too large for it keeps the same seeded columns in
    every run, one that fits is written whole."""
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench

    monkeypatch.setattr(bench, "DUMP_BYTES", 100_000)
    g = torch.arange(4 * 300, dtype=torch.float64).reshape(4, 300)
    pk = torch.arange(4 * 10_000, dtype=torch.float64).reshape(4, 10_000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"residuals": g, "jacobian_packed": pk})
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 100_000
    assert np.array_equal(np.load(tmp_path / "a" / "residuals.npy"), g.numpy())
    a, b = np.load(tmp_path / "a" / "jacobian_packed.npy"), np.load(tmp_path / "b" / "jacobian_packed.npy")
    assert a.dtype == np.float64 and 0 < a.shape[1] < 10_000 and np.array_equal(a, b)
    cols = a[0].astype(np.int64)
    assert np.all(np.diff(cols) > 0) and np.array_equal(a, pk.numpy()[:, cols])


@pytest.mark.gpu
def test_dump_outputs_are_what_the_timed_step_returns(tmp_path):
    """A short GPU run of bench.py --dump-outputs (outputs small enough to be written whole): the files equal the pair
    evaluation of the same scenarios at the same decision vectors through the host-buffer C ABI."""
    import numpy as np

    import bench
    from gelato_b200 import engine

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--factor", "1",
                          "--scenarios", "3", "--no-cpu-baseline", "--solve-scenarios", "0", "--sustained-seconds", "0",
                          "--preheat-seconds", "0", "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    plans, X, _ = bench.load_workload("example", 1, 3, 0, 3)
    E = engine.Engine(plans[0], device=0, scenario_plans=plans)
    g, pk = E.eval_pair_packed(X, 3)
    E.close()
    assert np.array_equal(np.load(tmp_path / "residuals.npy"), g)
    assert np.array_equal(np.load(tmp_path / "jacobian_packed.npy"), pk)


def test_reference_arm_other_ranks_stay_silent():
    """Under torchrun only rank 0 runs and prints the reference arm; the others exit 0 without work."""
    assert _run(["--gpus", "2"], env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}) == []
