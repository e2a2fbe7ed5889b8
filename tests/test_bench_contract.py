"""bench.py's reference arm (`--impl reference`: the oracle port timed on host cores) produces
the JSON line the driver parses.  Runs on CPU with a tiny bounded sample."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1", "--dim", "40", "--ref-seconds", "0.2"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1                                  # exactly one JSON line on stdout
    r = json.loads(lines[0])
    assert r["impl"] == "reference" and r["metric"] == "leapfrog_steps_per_sec" and r["unit"] == "leapfrog-steps/s"
    assert r["higher_is_better"] is True and r["n_gpus"] == 1 and r["steps"] == 2 and r["warmup"] == 1
    assert r["dtype"] == "f64" and r["data"] == "synthetic" and r["vs_baseline"] is None
    assert r["value"] > 0 and r["ms_per_step"] > 0 and "workload" in r["config"]
    cb = r["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == r["value"] and cb["sample"]
    assert r["e2e"] == {"value": r["value"], "unit": r["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert r["gpu_launches"] == 0                           # nothing of the CUDA path runs in this arm


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "0", "--dim", "40", "--ref-seconds", "0.1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_b200_arm_orchestration_emits_one_contract_line_with_stub_engine(tmp_path):
    """The b200 arm cannot run without a GPU; its ORCHESTRATION can: tests/bench_stub_driver.py replaces torch's CUDA entry
    points and the engine by stand-ins and runs bench.main() with the default configuration.  Checked: exactly one JSON line on
    stdout with every key of the contract, the roofline / cpu_baseline / e2e objects, the three auxiliary legs
    (user_model, c4_probe, c3_probe) present without an error, and the --dump-outputs files (names, shapes, dtype, size).
    (The numbers are the stand-in's and mean nothing.)"""
    dump = tmp_path / "dump"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "bench_stub_driver.py"), "--steps", "2", "--warmup", "3",
                          "--cpu-baseline-seconds", "0.2", "--dump-outputs", str(dump)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    r = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "gpu_launches", "clocks", "roofline", "cpu_baseline", "e2e"):
        assert k in r, k
    assert r["metric"] == "leapfrog_steps_per_sec" and r["n_gpus"] == 1 and r["steps"] == 2 and r["warmup"] == 3
    assert r["higher_is_better"] is True and r["scaling"] == "weak" and r["dtype"] == "f64" and r["vs_baseline"] is None
    assert "workload" in r["config"] and r["config"]["chains_per_gpu"] == 65536 and r["config"]["dim"] == 1000
    assert set(("bound", "achieved", "peak", "unit", "frac", "traffic")) <= set(r["roofline"]) and r["roofline"]["bound"] == "hbm"
    assert set(("value", "unit", "cores", "kind", "sample")) <= set(r["cpu_baseline"]) and r["cpu_baseline"]["kind"] == "port"
    assert set(("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step")) <= set(r["e2e"])
    assert r["e2e"]["h2d_bytes_per_step"] == 65536 * 1000 * 8 and r["e2e"]["d2h_bytes_per_step"] == 65536 * 2 * (1000 * 8 + 56 + 8)
    for leg in ("user_model", "c4_probe", "c3_probe"):
        assert leg in r and "error" not in r[leg] and r[leg]["value"] > 0 and r[leg]["unit"] == r["unit"], (leg, r.get(leg))
    assert r["user_model"]["model"] == "std_normal_user" and r["user_model"]["same_trees"] is True
    fields = ("pi", "depth", "left", "right", "acceptance_rate", "steps", "directions")
    names = {"chains", "posterior_matrix", "logdensities"} | {"tree_statistics_" + f for f in fields}
    assert {p.name for p in dump.iterdir()} == {n + ".npy" for n in names}
    a = {n: np.load(dump / (n + ".npy")) for n in names}
    assert all(v.dtype == np.float64 for v in a.values())
    assert sum(p.stat().st_size for p in dump.iterdir()) <= 64 << 20
    m = a["chains"].size                                    # a seeded sample: 65 536 chains x 2 draws x 1000 dims is 1 GB
    assert 1000 < m < 65536 and np.all(np.diff(a["chains"]) > 0) and a["chains"][-1] < 65536
    assert a["posterior_matrix"].shape == (m, 2, 1000) and all(a[n].shape == (m, 2) for n in names - {"chains", "posterior_matrix"})
