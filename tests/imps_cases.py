"""The reference's own InfiniteMPS (matrixproductstates/infinite_mps.py), unmodified, on a given backend.

`make_tensors` draws the unit cell with the reference's InfiniteMPS.random on backend numpy with np.random seeded (how
tools/gen_imps_golden.py made tests/golden/imps.npz); `canonicalize` runs InfiniteMPS.canonicalize and
check_canonical on backend `name` from those tensors and records what the tests compare: the dtype the state ends in,
the canonical-form deviation, the Schmidt values (1 / diag of the connector matrix, i.e. through backend.inv), the
returned lam_norm, and the operator applications of every backend.eigs call."""
import numpy as np

N_SITES, PHYS = 4, 2
SEED = 20261017
# (D, dtype) of tests/golden/imps.npz
GOLDEN_CASES = [(10, "float64"), (10, "complex128"), (64, "float64"), (64, "complex128"), (256, "float64"),
                (256, "complex128")]


def make_tensors(tn, D, dtype, seed=SEED):
  np.random.seed(seed)
  mps = tn.InfiniteMPS.random(d=[PHYS] * N_SITES, D=[D] * (N_SITES + 1), dtype=np.dtype(dtype), backend="numpy")
  return [np.array(t) for t in mps.tensors]


def checksum(tensors):
  return [float(np.sum(np.abs(t))) for t in tensors]


def golden_tensors(tn, meta):
  """the unit cell of a tests/golden/imps.npz case, redrawn from its seed and checked against the stored checksum"""
  tensors = make_tensors(tn, meta["D"], meta["dtype"], meta["seed"])
  np.testing.assert_allclose(checksum(tensors), meta["checksum"], rtol=1e-12)
  return tensors


def counting_eigs(be, calls):
  """Wraps be.eigs (on the instance) so that every call appends its number of operator applications to `calls`."""
  orig = be.eigs

  def eigs(*args, **kwargs):
    if "A" in kwargs:
      A = kwargs.pop("A")
    else:
      A, args = args[0], args[1:]
    n = [0]

    def counted(*x):
      n[0] += 1
      return A(*x)
    try:
      return orig(counted, *args, **kwargs)
    finally:
      calls.append(n[0])
  be.eigs = eigs
  return lambda: be.__dict__.pop("eigs", None)


def canonicalize(tn, name, tensors):
  be = tn.backends.backend_factory.get_backend(name)
  calls = []
  restore = counting_eigs(be, calls)
  try:
    mps = tn.InfiniteMPS([t.copy() for t in tensors], center_position=0, backend=name)
    lam_norm = mps.canonicalize()
    dev = float(np.abs(np.asarray(mps.check_canonical())))
  finally:
    restore()
  schmidt = 1.0 / np.diag(np.asarray(mps.connector_matrix))
  return dict(dtype=np.dtype(mps.dtype), tensor_dtypes=[np.asarray(t).dtype for t in mps.tensors], check=dev,
              schmidt=np.asarray(schmidt), lam_norm=complex(np.asarray(lam_norm)), matvecs=calls, mps=mps)
