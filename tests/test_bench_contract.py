"""CPU-only checks of bench.py's driver contract: the reference arm prints exactly one JSON line with the agreed
keys, and the cuda_b200 arm refuses to run (non-zero exit, no JSON) on a box without a GPU — no CPU fallback."""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_contract_keys():
  out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "1", "--networks", "1"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600, check=True)
  lines = [l for l in out.stdout.splitlines() if l.strip()]
  assert len(lines) == 1, out.stdout
  d = json.loads(lines[0])
  assert d["impl"] == "reference" and d["metric"] == "pairwise contractions/s" and d["unit"] == "contractions/s"
  for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
            "config", "cpu_baseline", "e2e"):
    assert k in d, k
  assert d["vs_baseline"] is None and d["higher_is_better"] is True and d["value"] > 0
  # oracle/_ref installed (by build()) -> the unmodified reference times itself; only without it the oracle port
  from baseline import refenv
  assert d["cpu_baseline"]["kind"] == ("reference" if refenv.available() else "port") and d["cpu_baseline"]["cores"] >= 1
  assert set(d["by_dtype"]) == {"f32", "f64"} and all(v["value"] > 0 for v in d["by_dtype"].values())
  assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
  assert "workload" in d["config"]


def test_product_arm_fails_loudly_without_gpu():
  import pytest
  import torch
  if torch.cuda.is_available():
    pytest.skip("GPU present")
  out = subprocess.run([sys.executable, "bench.py", "--steps", "1", "--networks", "1", "--no-cpu-baseline"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
  assert out.returncode != 0
  assert not [l for l in out.stdout.splitlines() if l.strip().startswith("{")]
