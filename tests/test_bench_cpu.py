"""CPU-only: the bench.py contract the driver depends on, exercised through the reference arm (the only arm that runs
without a GPU) on a tiny configuration, plus the loud failure of the product arm when there is no B200."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


def run_bench(*args, env=None, timeout=600):
    proc = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=timeout,
                          cwd=str(ROOT), env=env)
    return proc


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    proc = run_bench("--impl", "reference", "--model", "tiny", "--batch", "4", "--seq", "32", "--new", "8", "--steps", "2",
                     "--warmup", "1", "--cpu-sample", "4")
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [ln for ln in proc.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    for k in ("metric", "value", "unit", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config"):
        assert k in d, k
    assert d["unit"] == "tokens/s" and d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_product_arm_fails_loudly_without_a_gpu():
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    proc = run_bench("--model", "tiny", "--batch", "4", "--seq", "32", "--new", "8", "--steps", "1", "--warmup", "3",
                     "--no-cpu-baseline")
    assert proc.returncode != 0
    assert "no CPU fallback" in (proc.stderr + proc.stdout) or "CUDA" in (proc.stderr + proc.stdout)
    assert not any(ln.lstrip().startswith("{") for ln in proc.stdout.splitlines())  # no number is reported


def test_dump_outputs_writes_the_tokens_and_stays_under_its_limit(tmp_path, monkeypatch):
    import numpy as np

    import bench

    tokens = np.arange(6 * 9).reshape(6, 9)
    bench.dump_tokens(tmp_path / "all", tokens)
    assert sorted(p.name for p in (tmp_path / "all").iterdir()) == ["generated_tokens.npy"]
    got = np.load(tmp_path / "all" / "generated_tokens.npy")
    assert got.dtype == np.float32 and np.array_equal(got, tokens)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 3 * (4 * 9 + 8))
    for d in ("s1", "s2"):
        bench.dump_tokens(tmp_path / d, tokens)
    rows = np.load(tmp_path / "s1" / "generated_tokens_rows.npy").astype(int)
    assert len(rows) == 3 and (np.diff(rows) > 0).all()
    assert np.array_equal(np.load(tmp_path / "s1" / "generated_tokens.npy"), tokens[rows])
    assert np.array_equal(rows, np.load(tmp_path / "s2" / "generated_tokens_rows.npy"))  # the same sample every run


def test_bench_rejects_zero_steps_and_dumps_on_the_reference_arm(tmp_path):
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        proc = run_bench(*args, timeout=120)
        assert proc.returncode == 2 and "error:" in proc.stderr and not proc.stdout.strip()
