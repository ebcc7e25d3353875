"""Row N1: the reference's own callers, UNMODIFIED, on backend="cuda_b200" with the real kernels.

The reference package is the copy build() installs under oracle/_ref (oracle/build_ref.py), imported
through baseline/refenv.py.  Every case of tests/ref_cases.py is run with backend="numpy" (the
reference's own numpy backend) and backend="cuda_b200" in the same process, on the same seeded
inputs, and compared (fp64: <= 1e-10 of the result scale; integers exact).  Both arms are also compared with the
numpy arm's results stored in tests/golden/ref_callers.npz (oracle/gen_golden.py:gen_ref_callers)."""
import numpy as np
import pytest
import ref_cases

pytestmark = pytest.mark.gpu


def _backend(tn):
  import tensornetwork_b200 as tb
  from tensornetwork_b200 import backend as tbb
  from tensornetwork.backends import abstract_backend, backend_factory
  assert tb.registered and tbb.HAVE_TENSORNETWORK
  be = backend_factory.get_backend("cuda_b200")
  assert isinstance(be, abstract_backend.AbstractBackend) and be.name == "cuda_b200"
  assert backend_factory.get_backend("cuda_b200") is be
  return be


@pytest.mark.parametrize("name,fn,tol", ref_cases.CASES, ids=[c[0] for c in ref_cases.CASES])
def test_reference_caller(tn, golden, name, fn, tol):
  be = _backend(tn)
  n0 = be.lib.tnb200_launch_count()
  got = fn(tn, "cuda_b200")
  launches = be.lib.tnb200_launch_count() - n0
  ref = fn(tn, "numpy")
  ref_cases.compare(name, got, ref, tol)
  meta, z = golden("ref_callers")
  stored = [z["%s__%d" % (name, i)] for i in range(next(m["outputs"] for m in meta if m["name"] == name))]
  ref_cases.compare(name, ref, stored, tol)
  ref_cases.compare(name, got, stored, tol)
  assert launches > 0, "no libtnb200 kernel ran for " + name


def test_results_live_on_the_device(tn):
  from tensornetwork_b200 import B200Tensor
  be = _backend(tn)
  a = tn.Node(np.ones((3, 4)), backend="cuda_b200")
  b = tn.Node(np.ones((4, 5)), backend="cuda_b200")
  a[1] ^ b[0]
  c = a @ b
  assert isinstance(c.tensor, B200Tensor) and c.tensor.t.is_cuda
  assert c.backend is be
  tn.set_default_backend("cuda_b200")
  try:
    assert tn.Node(np.ones(3)).backend.name == "cuda_b200"
  finally:
    tn.set_default_backend("numpy")


def test_reference_error_conventions(tn):
  be = _backend(tn)
  with pytest.raises(TypeError):
    be.convert_to_tensor([1, 2])
  with pytest.raises(ValueError):
    be.tensordot(be.convert_to_tensor(np.ones((2, 3))), be.convert_to_tensor(np.ones((4, 5))), [[1], [0]])
  a = tn.Node(np.ones((2, 2)), backend="cuda_b200")
  b = tn.Node(np.ones((2, 2)), backend="numpy")
  with pytest.raises(ValueError):
    a[0] ^ b[0]
    tn.contract_between(a, b)


def test_reference_greedy_mps_norm_D64_float32_and_complex(tn):
  """A larger <psi|psi> through contractors.greedy (path_contractors.py:87-90): the per-pair loop
  reaches the tcgen05 / DMMA / thin kernels rather than only the SIMT fallback.  float32 is checked
  twice: strict (fp32 FMA, 1e-4 after 23 chained contractions) and the tensor-core TF32 mode, whose
  2^-11 operand rounding accumulates over the chain (stated tolerance 2e-2)."""
  from tensornetwork_b200 import _lib as L
  be = _backend(tn)
  rng = np.random.default_rng(21)
  for dtype, mode, tol in ((np.float64, L.MATH_DEFAULT, 1e-10), (np.float32, L.MATH_STRICT, 1e-4),
                           (np.float32, L.MATH_DEFAULT, 2e-2), (np.complex128, L.MATH_DEFAULT, 1e-10)):
    kets = ref_cases.mps_kets(rng, 12, 64, np.float64)
    if np.issubdtype(dtype, np.complexfloating):
      kets = [k + 1j * rng.standard_normal(k.shape) / np.sqrt(k.shape[0]) for k in kets]
    kets = [k.astype(dtype) for k in kets]
    old = be.math_mode
    be.math_mode = mode
    try:
      got = np.asarray(tn.contractors.greedy(ref_cases._mps_norm_nodes(tn, "cuda_b200", kets)).tensor)
    finally:
      be.math_mode = old
    ref = np.asarray(tn.contractors.greedy(ref_cases._mps_norm_nodes(tn, "numpy", kets)).tensor)
    assert abs(got - ref) <= tol * abs(ref), (dtype, mode, got, ref)


def _canonical_mps_tensors(rng, N, D, centre):
  """left-orthonormal sites < centre, right-orthonormal sites > centre, normalised random centre tensor"""
  dims = [min(D, 2**min(i, N - i)) for i in range(N + 1)]
  ts = []
  for i in range(N):
    dl, dr = dims[i], dims[i + 1]
    if i < centre:
      q, _ = np.linalg.qr(rng.standard_normal((dl * 2, dr)))
      ts.append(np.ascontiguousarray(q.reshape(dl, 2, dr)))
    elif i > centre:
      q, _ = np.linalg.qr(rng.standard_normal((2 * dr, dl)))
      ts.append(np.ascontiguousarray(q.T.reshape(dl, 2, dr)))
    else:
      c = rng.standard_normal((dl, 2, dr))
      ts.append(c / np.linalg.norm(c))
  return ts


@pytest.mark.parametrize("D", [64, 1024])
def test_cfg5_two_site_update_full_bond_dimension(tn, D):
  """BASELINE cfg 5 (D=1024; D=64 is the quick sibling): ONE saturated two-site update of the reference's own
  FiniteDMRG._optimize_2s_local (matrixproductstates/dmrg.py:251-343: ncon -> eigsh_lanczos(two_site_matvec) -> svd
  truncation to D -> add_left_layer), identical inputs and identical update count on backend="numpy" and
  backend="cuda_b200".  Energy, the new bond's singular values and the updated left environment agree to 1e-8."""
  be = _backend(tn)
  lo = int(np.log2(D))
  N = 2 * lo + 2
  rng = np.random.default_rng(6)
  tensors = _canonical_mps_tensors(rng, N, D, lo)

  def arm(backend):
    mps = tn.FiniteMPS([t.copy() for t in tensors], canonicalize=False, backend=backend)
    mps.center_position = lo
    mpo = tn.FiniteXXZ(np.ones(N - 1), np.ones(N - 1), np.zeros(N), dtype=np.float64, backend=backend)
    dm = tn.FiniteDMRG(mps, mpo)
    dm.compute_left_envs()
    dm.compute_right_envs()
    e = dm._optimize_2s_local(max_bond_dim=D, sweep_dir="right", num_krylov_vecs=10, tol=1e-5, delta=1e-6, ndiag=10)
    nxt = np.asarray(mps.tensors[lo + 1])           # = diag(s) vh
    u = np.asarray(mps.tensors[lo])
    lenv = np.asarray(dm.left_envs[lo + 1])
    return float(np.real(np.asarray(e))), nxt, u, lenv, mps.center_position

  n0 = be.lib.tnb200_launch_count()
  e_g, nxt_g, u_g, l_g, c_g = arm("cuda_b200")
  assert be.lib.tnb200_launch_count() > n0
  e_n, nxt_n, u_n, l_n, c_n = arm("numpy")
  assert c_g == c_n == lo + 1 and nxt_g.shape == nxt_n.shape == (D, 2, D) and u_g.shape == u_n.shape
  assert abs(e_g - e_n) <= 1e-8 * abs(e_n), (e_g, e_n)
  s_g = np.linalg.norm(nxt_g.reshape(D, -1), axis=1)
  s_n = np.linalg.norm(nxt_n.reshape(D, -1), axis=1)
  np.testing.assert_allclose(s_g, s_n, rtol=0, atol=1e-8 * s_n[0])
  # gauge-invariant comparison of the factors: projector onto the kept left space, and the two-site state u s vh
  th_g = np.tensordot(u_g, nxt_g, [[2], [0]])
  th_n = np.tensordot(u_n, nxt_n, [[2], [0]])
  assert np.linalg.norm(th_g - th_n) <= 1e-7 * np.linalg.norm(th_n) or np.linalg.norm(th_g + th_n) <= 1e-7 * np.linalg.norm(th_n)
  ug = u_g.reshape(-1, D)
  np.testing.assert_allclose(ug.T @ ug, np.eye(D), atol=1e-9)


def test_reference_ncon_reaches_graph_replay_through_jit(tn):
  """`tn.ncon` -> `backend.jit(_jittable_ncon, static_argnums=(1..5))` (ncon_interface.py:654-660): call 1 eager, call 2
  captures the reference's own python loop in a CUDA graph, call 3 is ONE graph launch (no kernel launched from the host)
  on NEW input data, result equal to the numpy backend's."""
  be = _backend(tn)
  rng = np.random.default_rng(8)
  net = [[-1, 1, 2], [1, 3, -2], [2, 3, 4], [4, -3]]

  def data():
    return [rng.standard_normal(s) for s in ((6, 7, 8), (7, 9, 5), (8, 9, 4), (4, 3))]
  stats0 = dict(be.jit_stats)
  for call in range(4):
    xs = data()
    n0 = be.lib.tnb200_launch_count()
    r0 = be.jit_stats["replays"]
    got = tn.ncon([be.convert_to_tensor(x) for x in xs], net, backend="cuda_b200")
    launched = be.lib.tnb200_launch_count() - n0
    ref = tn.ncon(xs, net, backend="numpy")
    np.testing.assert_allclose(np.asarray(got), ref, rtol=0, atol=1e-12 * np.abs(ref).max())
    if call >= 2:
      assert launched == 0, (call, launched)                     # nothing but the graph replay
      assert be.jit_stats["replays"] - r0 == 1
  assert be.jit_stats["captures"] - stats0["captures"] == 1
  # results are values, not views of the captured buffers: an earlier result survives later calls
  keep = tn.ncon([be.convert_to_tensor(x) for x in xs], net, backend="cuda_b200")
  keep_host = np.asarray(keep).copy()
  tn.ncon([be.convert_to_tensor(x) for x in data()], net, backend="cuda_b200")
  np.testing.assert_array_equal(np.asarray(keep), keep_host)
  # a function that synchronises with the host (truncating svd) falls back to eager, permanently, without error
  f = be.jit(lambda t: be.svd(t, 1, max_truncation_error=1e-3, relative=True)[1], static_argnums=())
  x = be.convert_to_tensor(rng.standard_normal((20, 12)))
  a = [np.asarray(f(x)) for _ in range(3)]
  np.testing.assert_allclose(a[0], a[2])
  np.testing.assert_allclose(a[0], tn.backends.backend_factory.get_backend("numpy").svd(np.asarray(x), 1, max_truncation_error=1e-3, relative=True)[1], atol=1e-12)
