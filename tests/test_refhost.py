"""Needs the reference installed in oracle/_ref by build(): the reference's own callers — tn.Node, tn.ncon,
contractors.greedy, split_node*, FiniteDMRG.run_two_site — run UNCHANGED on backend="cuda_b200".
The device layer is replaced by tests/fake_lib.py (host memory + numpy oracle), so this exercises
the adapter's host logic and the registration path; the kernels are checked by the -m gpu tests."""
import os
import subprocess
import sys
import pytest
from oracle import ref_shim

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = [pytest.mark.refhost,
              pytest.mark.skipif(not ref_shim.available(), reason="reference not installed in oracle/_ref")]


def _run(*extra):
  r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "refhost_runner.py")] + list(extra),
                     capture_output=True, text=True, cwd=ROOT, timeout=600)
  assert r.returncode == 0 and "REFHOST OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
  return r.stdout


def test_reference_callers_on_cuda_b200_adapter():
  _run()


def test_reference_two_site_dmrg_on_cuda_b200_adapter():
  out = _run("--dmrg")
  assert "case dmrg ok" in out


def test_reference_blocksparse_callers_on_symmetric_b200_adapter():
  """tests/symhost_runner.py: block-sparse tn.Node @ / split_node / ncon / svd on backend="symmetric_b200" against the
  reference's backend="symmetric" (host double of the library)."""
  r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "symhost_runner.py")],
                     capture_output=True, text=True, cwd=ROOT, timeout=600)
  assert r.returncode == 0 and "SYMHOST OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
