"""The InfiniteMPS surface on the B200: tnb200_eigh (small one-CTA-per-matrix path and blocked path), tnb200_inv,
tnb200_compare / tnb200_masked_fill, and the Arnoldi eigensolver over tnb200_krylov_orth — each against numpy / scipy,
then the reference's own InfiniteMPS.canonicalize, unmodified, on backend="cuda_b200" against its numpy backend and
tests/golden/imps.npz, and tn.linalg.eigh / inv on tn.Tensor."""
import numpy as np
import pytest
import imps_cases

pytestmark = pytest.mark.gpu
EPS = {np.float32: np.finfo(np.float32).eps, np.float64: np.finfo(np.float64).eps,
       np.complex64: np.finfo(np.float32).eps, np.complex128: np.finfo(np.float64).eps}
DTYPES = [np.float32, np.float64, np.complex64, np.complex128]
SMALL_LIMIT = 64          # csrc/eigh.cu EIGH_SMALL_N


def _be():
  from tensornetwork_b200 import backend
  return backend.get_instance()


def _rand(rng, shape, dt):
  x = rng.standard_normal(shape)
  if np.issubdtype(dt, np.complexfloating):
    x = x + 1j * rng.standard_normal(shape)
  return x.astype(dt)


def _herm(rng, n, dt, batch=()):
  x = _rand(rng, batch + (n, n), dt)
  return ((x + np.conj(np.swapaxes(x, -1, -2))) / 2).astype(dt)


def _eigh_checked(be, a, dt):
  """device eigh with the info word; checks it against np.linalg.eigh on the same (lower-triangle) input."""
  info = be.torch.zeros(4, dtype=be.torch.int32, device=be.device)
  w, v = be._eigh(be.convert_to_tensor(a), info)  # pylint: disable=protected-access
  w, v, info = np.asarray(w), np.asarray(v), info.cpu().numpy()
  assert info[1] == 1, info
  assert w.dtype == np.empty(0, dt).real.dtype and v.dtype == dt
  n = a.shape[-1]
  h = np.tril(a) + np.conj(np.swapaxes(np.tril(a, -1), -1, -2))        # the Hermitian matrix numpy reads (UPLO='L')
  h = h.astype(np.complex128 if np.iscomplexobj(a) else np.float64)
  idx = np.arange(n)
  h[..., idx, idx] = h[..., idx, idx].real
  rw = np.linalg.eigvalsh(h)
  norm = max(np.linalg.norm(h.reshape(-1, n, n), ord=2, axis=(1, 2)).max(), 1e-300)
  tol = 10 * EPS[dt] * norm * max(n, 1)
  assert np.max(np.abs(w - rw)) <= tol, (np.max(np.abs(w - rw)), tol)
  assert np.all(np.diff(w, axis=-1) >= -tol)
  vv = v.astype(h.dtype)
  res = np.linalg.norm(h @ vv - vv * w[..., None, :].astype(h.dtype))
  orth = np.linalg.norm(np.conj(np.swapaxes(vv, -1, -2)) @ vv - np.eye(n))
  assert res <= tol * np.sqrt(n) * np.sqrt(max(1, np.prod(a.shape[:-2]))), res
  assert orth <= 10 * EPS[dt] * n * np.sqrt(max(1, np.prod(a.shape[:-2]))), orth
  return w, v


@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("n", [1, 2, 17, SMALL_LIMIT, SMALL_LIMIT + 1, 256, 1000])
def test_eigh_sizes(dt, n):
  be = _be()
  _eigh_checked(be, _herm(np.random.default_rng(n), n, dt), dt)


@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("shape", [(3, 17), (2, 2, 40), (2, 100)])
def test_eigh_stacks(dt, shape):
  be = _be()
  _eigh_checked(be, _herm(np.random.default_rng(7), shape[-1], dt, batch=shape[:-1]), dt)


@pytest.mark.parametrize("dt", [np.float64, np.complex128], ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("n", [40, 300])
def test_eigh_degenerate_spectra(dt, n):
  be = _be()
  rng = np.random.default_rng(11)
  _eigh_checked(be, np.eye(n, dtype=dt), dt)
  q, _ = np.linalg.qr(_rand(rng, (n, n), dt))
  lam = np.repeat(np.arange(1.0, n / 4 + 1), 4)[:n]
  _eigh_checked(be, ((q * lam) @ np.conj(q.T)).astype(dt), dt)
  x = _rand(rng, (n, n // 8), dt)          # rank-deficient PSD, many eigenvalues at ~0 (an iMPS fixed point's shape)
  _eigh_checked(be, (x @ np.conj(x.T) / n).astype(dt), dt)


@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("n", [30, 200])
def test_eigh_reads_only_the_lower_triangle(dt, n):
  be = _be()
  a = _rand(np.random.default_rng(3), (n, n), dt)          # not Hermitian; complex diagonal
  _eigh_checked(be, a, dt)


def test_eigh_errors():
  be = _be()
  with pytest.raises(np.linalg.LinAlgError):
    be.eigh(be.convert_to_tensor(np.ones((3, 4))))
  for dt in (np.int64, np.float16):
    with pytest.raises(TypeError):
      be.eigh(be.convert_to_tensor(np.ones((3, 3), dtype=dt)))


@pytest.mark.parametrize("dt", DTYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("n", [1, 5, 100, 513])
def test_inv(dt, n):
  be = _be()
  a = _rand(np.random.default_rng(n), (n, n), dt)
  got = np.asarray(be.inv(be.convert_to_tensor(a)))
  ref = np.linalg.inv(a.astype(np.complex128 if np.iscomplexobj(a) else np.float64))
  assert got.dtype == dt
  cond = np.linalg.cond(a.astype(ref.dtype))
  assert np.linalg.norm(got - ref) <= 50 * EPS[dt] * cond * np.linalg.norm(ref)
  # a strided (transposed) view
  got_t = np.asarray(be.inv(be.transpose(be.convert_to_tensor(a))))
  assert np.linalg.norm(got_t - ref.T) <= 50 * EPS[dt] * cond * np.linalg.norm(ref)


def test_inv_errors():
  be = _be()
  with pytest.raises(ValueError, match="Only matrices are supported"):
    be.inv(be.convert_to_tensor(np.ones((2, 2, 2))))
  with pytest.raises(np.linalg.LinAlgError):
    be.inv(be.convert_to_tensor(np.ones((2, 3))))
  for a in (np.ones((4, 4)), np.diag([1.0, 2.0, 0.0, 3.0]), np.zeros((1, 1), dtype=np.complex128)):
    with pytest.raises(np.linalg.LinAlgError, match="Singular matrix"):
      be.inv(be.convert_to_tensor(a))


@pytest.mark.parametrize("dt", [np.float32, np.float64, np.int64, np.complex128], ids=lambda d: np.dtype(d).name)
def test_masks_and_index_update(dt):
  be = _be()
  rng = np.random.default_rng(2)
  a = (rng.standard_normal((5, 7)) * 3).astype(np.float64)
  a[1, 2] = 1e-17
  t = be.convert_to_tensor(a)
  for got, ref in ((t <= 1e-16, a <= 1e-16), (t < 0.5, a < 0.5), (t > -1.0, a > -1.0), (t >= 0.0, a >= 0.0),
                   (t[0] <= t, a[0] <= a), (1.0 >= t, 1.0 >= a)):
    assert got.dtype == np.bool_ and np.array_equal(np.asarray(got), ref)
  assert (t[0, 0] < 1e30) is True                     # 0-d: a python bool (lanczos.py relies on it)
  x = (a + 1j * a).astype(dt) if np.issubdtype(dt, np.complexfloating) else a.astype(dt)
  xt = be.convert_to_tensor(x)
  mask = a <= 0.0
  for assignee, val in ((0.0, 0.0), (be.convert_to_tensor(np.array([5], dtype=np.int64)), 5),
                        (be.convert_to_tensor(np.array(-2.5)), -2.5)):
    ref = x.copy()
    ref[mask] = val
    got = be.index_update(xt, be.convert_to_tensor(mask), assignee)
    assert np.asarray(got).dtype == ref.dtype and np.array_equal(np.asarray(got), ref)
  ref = x.copy()
  ref[mask] = 0
  assert np.array_equal(np.asarray(be.index_update(xt, mask, 0)), ref)         # host mask
  assert np.array_equal(np.asarray(xt), x)


def _operator(rng, lam, dt):
  n = lam.size
  s = np.eye(n) + 0.05 * _rand(rng, (n, n), dt) / np.sqrt(n)
  return (s * lam) @ np.linalg.inv(s)


@pytest.mark.parametrize("dt", [np.float64, np.complex128], ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("which", ["LM", "LR", "SR", "SM"])
@pytest.mark.parametrize("numeig", [1, 2, 4])
def test_eigs_dense(dt, which, numeig):
  be = _be()
  rng = np.random.default_rng(numeig)
  n = 400
  if which == "SM":
    lam = np.concatenate([[0.01, 0.02, 0.03, 0.04, 0.05], np.linspace(1.0, 2.0, n - 5)])
  else:
    lam = np.concatenate([[-5.0, -4.5, -4.0, -3.5, -3.0], np.linspace(-1.0, 1.0, n - 10), [6.0, 6.5, 7.0, 7.5, 8.0]])
  m = _operator(rng, lam, dt).astype(dt)
  md = be.convert_to_tensor(m)
  x0 = be.convert_to_tensor(_rand(rng, (n,), dt))
  tol = 1e-10
  eta, vecs = be.eigs(lambda v: be.tensordot(md, v, 1), initial_state=x0, numeig=numeig, num_krylov_vecs=30, tol=tol,
                      which=which, maxiter=500)
  eta = np.asarray(eta)
  assert eta.dtype == np.complex128 and len(vecs) == numeig
  ev = np.linalg.eigvals(m)
  key = {"LM": lambda t: -np.abs(t), "SM": np.abs, "LR": lambda t: -t.real, "SR": lambda t: t.real}[which]
  want = ev[np.argsort(key(ev), kind="stable")[:numeig]]
  for e in eta:
    assert np.min(np.abs(want - e)) <= 100 * tol * max(1.0, abs(e)), (eta, want)
  for e, v in zip(eta, vecs):
    v = np.asarray(v)
    assert v.dtype == np.complex128 and v.shape == (n,)
    assert abs(np.linalg.norm(v) - 1.0) < 1e-12
    assert np.linalg.norm(m @ v - e * v) <= 100 * tol * abs(e)


def test_eigs_float32_output_is_complex64():
  be = _be()
  rng = np.random.default_rng(4)
  lam = np.concatenate([np.linspace(-1.0, 1.0, 195), [3.0, 3.5, 4.0, 4.5, 5.0]])
  m = _operator(rng, lam, np.float64).astype(np.float32)
  md = be.convert_to_tensor(m)
  eta, vecs = be.eigs(lambda v: be.tensordot(md, v, 1), shape=(200,), dtype=np.float32, numeig=1, num_krylov_vecs=20,
                      tol=1e-5, which="LR")
  assert np.asarray(eta).dtype == np.complex64 and np.asarray(vecs[0]).dtype == np.complex64
  assert abs(np.asarray(eta)[0] - 5.0) <= 5e-3        # f32 operator: its tensordot runs on TF32 tensor cores (DESIGN §5)


def _arms(tn, D, dt, tensors):
  be = _be()
  n0 = be.lib.tnb200_launch_count()
  got = imps_cases.canonicalize(tn, "cuda_b200", tensors)
  launches = be.lib.tnb200_launch_count() - n0
  ref = imps_cases.canonicalize(tn, "numpy", tensors)
  assert launches > 0
  assert got["dtype"] == ref["dtype"] and got["tensor_dtypes"] == ref["tensor_dtypes"]
  assert got["check"] < 1e-12, got["check"]
  assert got["schmidt"].shape == ref["schmidt"].shape and np.max(np.abs(got["schmidt"] - ref["schmidt"])) <= 1e-10
  assert abs(got["lam_norm"] - ref["lam_norm"]) <= 1e-10 * abs(ref["lam_norm"])
  for g, r in zip(got["matvecs"], ref["matvecs"]):
    assert g <= 1.5 * r, (got["matvecs"], ref["matvecs"])
  return got, ref


@pytest.mark.parametrize("D,dt", imps_cases.GOLDEN_CASES)
def test_reference_infinite_mps_canonicalize(tn, golden, D, dt):
  meta, z = golden("imps")
  i = next(k for k, m in enumerate(meta) if m["D"] == D and m["dtype"] == dt)
  tensors = imps_cases.golden_tensors(tn, meta[i])
  got, ref = _arms(tn, D, dt, tensors)
  assert str(got["dtype"]) == meta[i]["final_dtype"]
  stored = z["c%d_schmidt" % i]
  assert np.max(np.abs(ref["schmidt"] - stored)) <= 1e-10 and np.max(np.abs(got["schmidt"] - stored)) <= 1e-10
  assert abs(got["lam_norm"] - complex(*meta[i]["lam_norm"])) <= 1e-10 * abs(got["lam_norm"])


def test_reference_infinite_mps_d1024(tn):
  be = _be()
  tensors = imps_cases.make_tensors(tn, 1024, "float64")
  got = imps_cases.canonicalize(tn, "cuda_b200", tensors)
  assert got["check"] < 1e-12, got["check"]
  assert abs(np.linalg.norm(got["schmidt"]) - 1.0) < 1e-10
  mps = got["mps"]
  eta, l = mps.transfer_matrix_eigs("left", precision=1e-12)
  tl = mps.unit_cell_transfer_operator("left", l)
  lh, tlh, e = np.asarray(l), np.asarray(tl), complex(np.asarray(eta))
  assert np.linalg.norm(tlh - e * lh) <= 1e-10 * np.linalg.norm(lh)


def test_tn_linalg_eigh_and_inv(tn):
  rng = np.random.default_rng(8)
  for dt in (np.float64, np.complex128):
    a = _herm(rng, 90, dt)
    w1, v1 = tn.linalg.linalg.eigh(tn.Tensor(a, backend="cuda_b200"))
    w2, v2 = tn.linalg.linalg.eigh(tn.Tensor(a, backend="numpy"))
    assert np.max(np.abs(np.asarray(w1.array) - w2.array)) <= 1e-12 * np.abs(w2.array).max()
    p1, p2 = np.asarray(v1.array), v2.array                       # eigenvectors up to a phase each
    ph = np.sum(np.conj(p1) * p2, axis=0)
    assert np.allclose(np.abs(ph), 1.0, atol=1e-8)
    b = _rand(rng, (70, 70), dt)
    i1 = np.asarray(tn.linalg.linalg.inv(tn.Tensor(b, backend="cuda_b200")).array)
    i2 = tn.linalg.linalg.inv(tn.Tensor(b, backend="numpy")).array
    assert np.linalg.norm(i1 - i2) <= 1e-10 * np.linalg.norm(i2)
