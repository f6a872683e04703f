"""bench.py's reference arm (the one leg of the bench that runs without a GPU): it must print ONE JSON line with the
contract's keys, on the product arm's metric / unit / config, and never touch the CUDA library. Plus --dump-outputs:
refused on the reference arm, reproducible on the product arm."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"):
        assert k in d, k
    assert d["unit"] == "denoise-steps/s" and d["higher_is_better"] is True and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["config"]["id"] == "c2" and "768x768" in d["config"]["workload"]
    assert d["value"] > 0 and abs(d["value"] - 1e3 / d["ms_per_step"]) < 1e-6 * d["value"] + 1e-9
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert d["vs_baseline"] is None


def test_dump_outputs_is_refused_on_the_reference_arm(tmp_path):
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "o")],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr and not (tmp_path / "o").exists()


@pytest.mark.gpu
def test_dump_outputs_are_the_same_bits_from_run_to_run(tmp_path):
    """--dump-outputs writes the denoised latent after the last timed step and the end-to-end depth map, as float32;
    two runs with the same arguments write identical arrays, and `steps` in the line is the --steps asked for."""
    runs = []
    for i in range(2):
        d = tmp_path / f"run{i}"
        out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "2", "--warmup", "3", "--no-cpu-baseline",
                              "--no-library-baseline", "--no-kernel-roofline", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=1200, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
        assert len(lines) == 1, lines
        assert json.loads(lines[0])["steps"] == 2
        runs.append({p.stem: np.load(p) for p in d.glob("*.npy")})
    a, b = runs
    assert sorted(a) == ["depth", "latent"]
    assert a["latent"].shape == (1, 4, 96, 96) and a["depth"].shape == (768, 768)
    for k, v in a.items():
        assert v.dtype == np.float32 and np.isfinite(v).all(), k
        np.testing.assert_array_equal(v, b[k], err_msg=k)
