"""Runs in a subprocess (tests/test_infinite_mps_host.py): the cuda_b200 adapter over the host double
test_infinite_mps_host.HostLib.  `imps`: the reference's InfiniteMPS.canonicalize / check_canonical on backend
"cuda_b200" against its numpy backend and tests/golden/imps.npz.  `api`: eigs argument errors, dense eigs against
np.linalg.eig, index_update, 0-d vs n-d comparisons, inv / eigh errors."""
import json
import os
import sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from baseline import refenv  # noqa: E402
tn = refenv.try_load()                   # reference first, so the adapter subclasses the real AbstractBackend
from tensornetwork_b200 import _lib, backend as tb_backend  # noqa: E402
import test_infinite_mps_host  # noqa: E402
_lib.set_lib(test_infinite_mps_host.HostLib())
tb_backend._CONFIG["device"] = "cpu"  # pylint: disable=protected-access
be = tb_backend.get_instance()


def expect(exc, fn, *args, **kwargs):
  try:
    fn(*args, **kwargs)
  except exc as e:
    return str(e)
  raise SystemExit("expected {} from {}".format(exc.__name__, getattr(fn, "__name__", fn)))


def api():
  import scipy.sparse.linalg  # pylint: disable=import-outside-toplevel
  rng = np.random.default_rng(5)
  x0 = be.convert_to_tensor(rng.standard_normal(40))
  mv = lambda v: v  # noqa: E731
  assert "LI" in expect(ValueError, be.eigs, mv, initial_state=x0, which="LI")
  expect(ValueError, be.eigs, mv, initial_state=x0, which="SI")
  expect(ValueError, be.eigs, mv, initial_state=x0, numeig=9, num_krylov_vecs=10)
  expect(ValueError, be.eigs, mv, shape=(40,))
  expect(TypeError, be.eigs, mv, initial_state=np.ones(40))
  # dense operators, real and complex, against np.linalg.eig
  for dt in (np.float64, np.complex128):
    M = rng.standard_normal((120, 120))
    if dt is np.complex128:
      M = M + 1j * rng.standard_normal((120, 120))
    Md = be.convert_to_tensor(M.astype(dt))
    ev = np.linalg.eigvals(M)
    for which, key in (("LM", lambda t: -np.abs(t)), ("LR", lambda t: -t.real), ("SR", lambda t: t.real)):
      for k in (1, 3):
        eta, vecs = be.eigs(lambda v: be.tensordot(Md, v, 1), initial_state=be.convert_to_tensor(rng.standard_normal(120).astype(dt)),
                            numeig=k, num_krylov_vecs=40, tol=1e-10, which=which, maxiter=200)
        want = ev[np.argsort(key(ev), kind="stable")[:k]]
        got = np.asarray(eta)
        assert got.dtype == np.complex128 and all(np.asarray(v).dtype == np.complex128 for v in vecs)
        for g in got:
          assert np.min(np.abs(want - g)) <= 1e-8 * np.abs(g), (dt, which, k, got, want)
        for g, v in zip(got, vecs):
          v = np.asarray(v)
          assert abs(np.linalg.norm(v) - 1) < 1e-12 and np.linalg.norm(M @ v - g * v) <= 1e-8 * abs(g)
  # non-convergence carries the converged pairs
  M = rng.standard_normal((200, 200))
  Md = be.convert_to_tensor(M)
  e = None
  try:
    be.eigs(lambda v: be.tensordot(Md, v, 1), initial_state=be.convert_to_tensor(rng.standard_normal(200)), numeig=4,
            num_krylov_vecs=8, tol=1e-14, which="SM", maxiter=2)
  except scipy.sparse.linalg.ArpackNoConvergence as err:
    e = err
  assert e is not None and hasattr(e, "eigenvalues") and hasattr(e, "eigenvectors")
  # comparisons: 0-d gives a python bool, n-d a device bool tensor
  s = be.convert_to_tensor(np.array(0.5))
  assert (s < 1.0) is True and (s >= 1.0) is False
  a = np.array([0.3, -1.0, 2.0, 1e-17, 0.0])
  t = be.convert_to_tensor(a)
  for op, ref in ((t <= 1e-16, a <= 1e-16), (t < 0.3, a < 0.3), (t > 0.0, a > 0.0), (t >= 2.0, a >= 2.0),
                  (0.3 >= t, 0.3 >= a), (t <= t, a <= a)):
    assert op.dtype == np.bool_ and np.array_equal(np.asarray(op), ref)
  # index_update: python scalar, size-1 device tensor, host mask
  mask = t <= 1e-16
  np.testing.assert_array_equal(np.asarray(be.index_update(t, mask, 0.0)), np.where(a <= 1e-16, 0.0, a))
  np.testing.assert_array_equal(np.asarray(be.index_update(t, mask, be.convert_to_tensor(np.array([7.0])))),
                                np.where(a <= 1e-16, 7.0, a))
  np.testing.assert_array_equal(np.asarray(be.index_update(t, a > 1.0, -3.0)), np.where(a > 1.0, -3.0, a))
  c = be.convert_to_tensor((a + 1j * a).astype(np.complex128))
  np.testing.assert_array_equal(np.asarray(be.index_update(c, mask, 0.0)), np.where(a <= 1e-16, 0.0, a + 1j * a))
  assert np.asarray(t).tolist() == a.tolist()       # the input is not modified
  # inv / eigh errors (numpy_backend.py:554-558; np.linalg)
  assert "Only matrices are supported" in expect(ValueError, be.inv, be.convert_to_tensor(np.ones((2, 2, 2))))
  expect(np.linalg.LinAlgError, be.inv, be.convert_to_tensor(np.ones((2, 3))))
  assert expect(np.linalg.LinAlgError, be.inv, be.convert_to_tensor(np.ones((3, 3)))) == "Singular matrix"
  B = rng.standard_normal((6, 6))
  np.testing.assert_allclose(np.asarray(be.inv(be.convert_to_tensor(B))), np.linalg.inv(B), rtol=1e-12, atol=1e-12)
  expect(np.linalg.LinAlgError, be.eigh, be.convert_to_tensor(np.ones((2, 3))))
  expect(TypeError, be.eigh, be.convert_to_tensor(np.ones((3, 3), dtype=np.int64)))
  w, v = be.eigh(be.convert_to_tensor(B))
  rw, rv = np.linalg.eigh(B)
  np.testing.assert_allclose(np.asarray(w), rw, atol=1e-12)
  print("api ok")


def imps():
  import imps_cases  # pylint: disable=import-outside-toplevel
  assert tn is not None, "reference missing"
  z = np.load(os.path.join(HERE, "golden", "imps.npz"), allow_pickle=False)
  meta = json.loads(str(z["__meta__"]))
  for i, m in enumerate(meta):
    if m["D"] > 64 or (m["D"] == 64 and m["dtype"] != "float64"):
      continue
    tensors = imps_cases.golden_tensors(tn, m)
    ref = imps_cases.canonicalize(tn, "numpy", tensors)
    got = imps_cases.canonicalize(tn, "cuda_b200", tensors)
    assert got["dtype"] == ref["dtype"] == np.dtype(m["final_dtype"]), (got["dtype"], ref["dtype"], m)
    assert got["tensor_dtypes"] == ref["tensor_dtypes"]
    assert got["check"] < 1e-12, got["check"]
    for want in (ref["schmidt"], z["c%d_schmidt" % i]):
      assert got["schmidt"].shape == want.shape and np.max(np.abs(got["schmidt"] - want)) <= 1e-10
    for want in (ref["lam_norm"], complex(*m["lam_norm"])):
      assert abs(got["lam_norm"] - want) <= 1e-10 * abs(want)
    assert len(got["matvecs"]) == len(m["matvecs"]) == 2
    for g, r in zip(got["matvecs"], m["matvecs"]):
      assert g <= 1.5 * r, (got["matvecs"], m["matvecs"])
    print("imps D=%d %s ok (matvecs %s vs ARPACK %s, check %.1e)" % (m["D"], m["dtype"], got["matvecs"], m["matvecs"], got["check"]))


if "api" in sys.argv:
  api()
if "imps" in sys.argv:
  imps()
print("IMPS HOST OK")
