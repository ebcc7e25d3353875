"""Import environment for the unmodified reference (google/TensorNetwork 0.4.6).

`oracle/build_ref.py` (run by `__graft_entry__.build()`) installs the reference, unmodified, into
`oracle/_ref` (git-ignored: a build product, never part of the repository).  The reference's
top-level import needs three third-party modules this image does not have (SURVEY.md 8c):
`h5py` (network_components.py:21,29 — only save/load use it), `graphviz`
(visualization/graphviz.py:16,23) and `opt_einsum` (path_contractors.py:18 — supplies only the
pairwise contraction ORDER).  `load()` pre-seeds `sys.modules` with minimal stand-ins for those
three and imports the package.  `opt_einsum.paths.{greedy,optimal}` are served by numpy's own
`_greedy_path` / `_optimal_path`, which reproduce the reference's path known-answer tests
(path_calculation_test.py:83-93; checked in tests/test_oracle_golden.py).

Nothing here is arithmetic: every flop of the reference arm is the reference's own code on its
own numpy backend.  Only the installed copy is imported.
"""
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
INSTALLED = os.path.join(os.path.dirname(HERE), "oracle", "_ref")


def location():
  if os.path.isdir(os.path.join(INSTALLED, "tensornetwork", "backends")):
    return INSTALLED
  return None


def available() -> bool:
  return location() is not None


def _seed_third_party():
  if "h5py" not in sys.modules:
    h5 = types.ModuleType("h5py")
    h5.Group = object
    h5.File = object
    h5.string_dtype = lambda encoding=None: object
    sys.modules["h5py"] = h5
  if "graphviz" not in sys.modules:
    gv = types.ModuleType("graphviz")
    gv.Graph = object
    sys.modules["graphviz"] = gv
  if "opt_einsum" not in sys.modules:
    from numpy._core.einsumfunc import _greedy_path, _optimal_path  # pylint: disable=import-outside-toplevel
    oe = types.ModuleType("opt_einsum")
    big = 2**62

    def greedy(i, o, s, memory_limit=None, **_unused):   # branch() passes nbranch=
      return _greedy_path(i, o, s, big if memory_limit is None else memory_limit)

    def optimal(i, o, s, memory_limit=None, **_unused):
      return _optimal_path(i, o, s, big if memory_limit is None else memory_limit)
    oe.paths = types.SimpleNamespace(greedy=greedy, optimal=optimal,
                                     dynamic_programming=optimal, branch=greedy)
    sys.modules["opt_einsum"] = oe


def load():
  """Returns the imported, unmodified reference `tensornetwork` module."""
  if "tensornetwork" in sys.modules:
    return sys.modules["tensornetwork"]
  loc = location()
  if loc is None:
    raise ImportError("reference not installed: oracle/_ref is missing (built by oracle/build_ref.py)")
  _seed_third_party()
  if loc not in sys.path:
    sys.path.insert(0, loc)
  import tensornetwork  # pylint: disable=import-outside-toplevel
  return tensornetwork


def try_load():
  try:
    return load()
  except ImportError:
    return None
