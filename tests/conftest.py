import json
import os
import sys
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

# The unmodified reference (oracle/_ref, installed by build()) must be imported BEFORE tensornetwork_b200 so that the
# backend subclasses the reference's real AbstractBackend and registers in its factory.
from baseline import refenv  # noqa: E402
REFERENCE = refenv.try_load()

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
  config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu)")
  config.addinivalue_line("markers", "refhost: needs the reference installed in oracle/_ref")


def _have_gpu():
  try:
    import torch
    return torch.cuda.is_available()
  except Exception:  # pylint: disable=broad-except
    return False


def pytest_collection_modifyitems(config, items):
  """`gpu` tests are skipped (not failed) on a machine without CUDA or without the built library."""
  lib = os.path.join(ROOT, "tensornetwork_b200", "lib", "libtnb200.so")
  if _have_gpu() and os.path.exists(lib):
    return
  skip = pytest.mark.skip(reason="needs a CUDA device and tensornetwork_b200/lib/libtnb200.so")
  for item in items:
    if "gpu" in item.keywords:
      item.add_marker(skip)


def load_golden(name):
  z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
  meta = json.loads(str(z["__meta__"]))
  return meta, z


@pytest.fixture(scope="session")
def golden():
  return load_golden


@pytest.fixture(scope="session")
def tn():
  """The unmodified reference package (oracle/_ref).  Its absence is an error, not a skip:
  the drop-in claim is only as good as these tests."""
  if REFERENCE is None:
    pytest.fail("oracle/_ref missing: build() installs the reference there (oracle/build_ref.py)")
  return REFERENCE
