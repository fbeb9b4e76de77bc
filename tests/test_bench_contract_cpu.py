"""bench.py's reference arm (the UNMODIFIED reference module staged in baseline/_ref — or the oracle port when no copy of
the reference exists — on the host CPU) runs without a GPU and prints the contract line: one JSON object with the metric
BASELINE.json names, the cpu_baseline description and an e2e block."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, OMP_NUM_THREADS="1")                 # what torchrun exports: the arm must still take all cores
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--batch", "8"], capture_output=True, text=True, env=env, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["impl"] == "reference" and d["metric"].split(",")[0] in base["metric"]
    for k in ("value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["unit"] == "img/s" and d["higher_is_better"] is True and d["vs_baseline"] is None and d["value"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    sys.path.insert(0, ROOT)
    from oracle import reference_module as RM
    assert cb["kind"] == ("reference" if RM.find() else "port") and cb["value"] == d["value"] and cb["sample"]
    assert set(d["directions"]) == {"forward", "inverse"} and d["checks"]["recon_max_abs_err"] < 1e-3
    assert cb["cores"] == (os.cpu_count() or 1), "rank 0 must use every host core even under OMP_NUM_THREADS=1"
    assert d["e2e"] == {"value": d["value"], "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_writes_float_arrays_within_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    g = torch.Generator().manual_seed(0)
    arrays = {"log_likelihood": torch.randn(16, dtype=torch.float64, generator=g),
              "x_reconstructed": torch.randn(16, 3, 4, 4, generator=g)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    for k, v in arrays.items():
        a = np.load(tmp_path / "all" / f"{k}.npy")
        assert a.dtype == v.numpy().dtype and np.array_equal(a, v.numpy()), k
    monkeypatch.setattr(bench, "DUMP_LIMIT", 5 * (8 + 3 * 4 * 4 * 4) + 7)          # room for five images
    bench.dump_outputs(str(tmp_path / "cut"), arrays)
    for k, v in arrays.items():
        assert np.array_equal(np.load(tmp_path / "cut" / f"{k}.npy"), v.numpy()[:5]), k


def test_bench_rejects_bad_step_and_dump_arguments(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)],
                  ["--only-train", "--dump-outputs", str(tmp_path)]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                           timeout=60, cwd=ROOT)
        assert r.returncode == 2 and r.stdout == "", (extra, r.stderr)
    assert os.listdir(tmp_path) == []


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, env=env, timeout=300, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""
