"""Import the real reference (google/TensorNetwork 0.4.6) for fixture generation and for the
checks that run the reference's own callers.  Test infrastructure.

The import environment (three third-party stand-ins: h5py, graphviz, opt_einsum — SURVEY.md 8c /
Appendix A.1) lives in baseline/refenv.py; the package itself is the unmodified copy that oracle/build_ref.py installs into oracle/_ref.
"""
from baseline import refenv


def available() -> bool:
  return refenv.available()


def load():
  """Returns the imported reference `tensornetwork` module."""
  return refenv.load()
