"""The reference's OWN callers, parametrised by backend name.

Each case builds its inputs from a fixed seed, drives the unmodified reference
(`oracle/_ref`, loaded through baseline/refenv.py) with `backend=<name>` and returns a list of
host arrays.  tests/test_gpu_reference_callers.py runs every case with backend="numpy" and
backend="cuda_b200" (the real libtnb200.so kernels) in the same process and compares;
tests/refhost_runner.py runs the same cases against the host test double.

Reference sites exercised (all unmodified, on our backend):
  network_components.py:1984-2095 contract_between (flip heuristic :2058-2080, axis sort :2082-2084)
  network_components.py:1367-1456 flatten_edges, :1802-1831 _contract_trace, :1834-1885 contract
  network_components.py:737-908   CopyNode / compute_contracted_tensor (einsum)
  ncon_interface.py:364-663       _jittable_ncon / ncon (through backend.jit)
  contractors/opt_einsum_paths/path_contractors.py:36-193 base / greedy / optimal
  contractors/bucket_contractor.py:21 bucket
  network_operations.py:130-588   split_node, split_node_qr, split_node_rq, split_node_full_svd
  matrixproductstates/dmrg.py:445-559 FiniteDMRG.run_two_site (+ eigsh_lanczos, svd, ncon)
"""
import numpy as np


def H(x):
  """backend tensor -> host ndarray."""
  return np.asarray(x)


def case_node_matmul(tn, be, seed=0):
  rng = np.random.default_rng(seed)
  a, b = rng.standard_normal((4, 5, 6)), rng.standard_normal((6, 5, 3))
  na, nb = tn.Node(a, backend=be), tn.Node(b, backend=be)
  na[2] ^ nb[0]
  na[1] ^ nb[1]
  c = na @ nb
  # matrix @ vector, vector @ vector (0-d result through the einsum fast path, numpy_backend.py:38-52)
  m, v = rng.standard_normal((7, 9)), rng.standard_normal(9)
  nm, nv = tn.Node(m, backend=be), tn.Node(v, backend=be)
  nm[1] ^ nv[0]
  d = nm @ nv
  v1, v2 = tn.Node(v, backend=be), tn.Node(2 * v, backend=be)
  v1[0] ^ v2[0]
  e = v1 @ v2
  return [H(c.tensor), H(d.tensor), H(e.tensor)]


def case_contract_between_flip(tn, be, seed=1):
  """node2 precedes node1 in the shared-edge axis order and the operands have unequal rank:
  exercises the flip heuristic and sorted axes of contract_between, plus output_edge_order and
  allow_outer_product."""
  rng = np.random.default_rng(seed)
  a = rng.standard_normal((3, 4, 5, 6))
  b = rng.standard_normal((6, 3))
  out = []
  for first in (0, 1):
    na, nb = tn.Node(a, backend=be), tn.Node(b, backend=be)
    na[3] ^ nb[0]
    na[0] ^ nb[1]
    c = tn.contract_between(nb, na) if first else tn.contract_between(na, nb)
    out.append(H(c.tensor))
  na, nb = tn.Node(a, backend=be), tn.Node(b, backend=be)
  e1 = na[3] ^ nb[0]
  c = tn.contract_between(na, nb, output_edge_order=[nb[1], na[2], na[0], na[1]])
  out.append(H(c.tensor))
  x, y = rng.standard_normal((2, 3)), rng.standard_normal((4,))
  o = tn.contract_between(tn.Node(x, backend=be), tn.Node(y, backend=be), allow_outer_product=True)
  out.append(H(o.tensor))
  out.append(H(tn.outer_product(tn.Node(x, backend=be), tn.Node(y, backend=be)).tensor))
  return out


def case_trace_and_flatten(tn, be, seed=2):
  rng = np.random.default_rng(seed)
  t = rng.standard_normal((3, 4, 3, 5, 4))
  nt = tn.Node(t, backend=be)
  nt[0] ^ nt[2]
  nt[1] ^ nt[4]
  r1 = tn.contract_trace_edges(nt)
  # flatten two parallel edges between two nodes, then contract the flattened edge
  a, b = rng.standard_normal((2, 3, 4, 5)), rng.standard_normal((5, 4, 3, 6))
  na, nb = tn.Node(a, backend=be), tn.Node(b, backend=be)
  e1 = na[1] ^ nb[2]
  e2 = na[2] ^ nb[1]
  e3 = na[3] ^ nb[0]
  da, db = na[0], nb[3]
  fe = tn.flatten_edges([e1, e2, e3])
  shapes = np.array(list(na.tensor.shape) + list(nb.tensor.shape))
  r2 = tn.contract(fe).reorder_edges([da, db])    # contract() picks node1/node2 by edge bookkeeping
  # flatten dangling edges of one node
  c = rng.standard_normal((2, 3, 4))
  nc = tn.Node(c, backend=be)
  tn.flatten_edges([nc[2], nc[0]])
  # flatten_all_edges / flatten_edges_between and contract_parallel
  na, nb = tn.Node(a, backend=be), tn.Node(b, backend=be)
  na[1] ^ nb[2]
  na[2] ^ nb[1]
  e = na[3] ^ nb[0]
  da, db = na[0], nb[3]
  r3 = tn.contract_parallel(e).reorder_edges([da, db])
  # trace edge flatten (both ends on one node)
  q = rng.standard_normal((3, 4, 3, 4, 2))
  nq = tn.Node(q, backend=be)
  t1 = nq[0] ^ nq[2]
  t2 = nq[1] ^ nq[3]
  tn.flatten_edges([t1, t2])
  r4 = tn.contract_trace_edges(nq)
  return [H(r1.tensor), shapes, H(r2.tensor), H(nc.tensor), H(r3.tensor), H(r4.tensor)]


def case_integer_nodes(tn, be, seed=3):
  """path_contractors_node_test.py:88-123 drives int64 tensors through contract_between."""
  a = tn.Node(np.arange(4).reshape((2, 2)), backend=be)
  b = tn.Node(np.arange(4).reshape((2, 2)) + 1, backend=be)
  c = tn.Node(np.arange(4).reshape((2, 2)) * 3, backend=be)
  a[1] ^ b[0]
  b[1] ^ c[0]
  r = tn.contractors.greedy([a, b, c], output_edge_order=[c[1], a[0]])
  return [H(r.tensor)]


NCON_CASES = [
    (((10, 10), (10, 10)), [(-1, 1), (1, -2)], None, None),
    (((3, 4, 4), (3, 5)), [(1, 2, 2), (1, -1)], None, None),                 # partial trace
    (((7, 3, 4), (7, 4, 5)), [(-1, -2, 1), (-1, 1, -3)], None, None),          # negative batch label
    (((2, 3), (4, 5)), [(-1, -2), (-3, -4)], None, [-3, -1, -4, -2]),          # outer product + out_order
    (((3, 4, 5), (5, 4, 6), (6, 3)), [(1, 2, 3), (3, 2, 4), (4, 1)], [3, 2, 4, 1], None),
    (((6, 3, 4), (6, 4, 5), (6, 5, 2)), [(1, -1, 2), (1, 2, 3), (1, 3, -2)], None, None),  # positive batch x3
    (((4, 5), (5,), (4,)), [(1, 2), (2,), (1,)], None, None),                   # scalar result
    (((3, 4, 3),), [(1, -1, 1)], None, None),                                  # single tensor, trace
    (((8, 2, 8), (8, 2, 8), (5, 5, 2, 2), (8, 8, 5)), [(1, 2, -1), (3, 4, -2), (5, -3, 4, 2), (3, 1, 5)],
     None, None),                                                              # DMRG add_left_layer shape
    (((3, 4), (4, 5)), [(-1, 1), (1, -2)], None, [-2, -1]),
]


def case_ncon(tn, be, seed=4):
  rng = np.random.default_rng(seed)
  out = []
  for shapes, net, con, order in NCON_CASES:
    ts = [rng.standard_normal(s) for s in shapes]
    out.append(H(tn.ncon(ts, net, con_order=con, out_order=order, backend=be)))
  # string labels (ncon_interface.py canonicalisation) and tn.Tensor inputs
  a, b = rng.standard_normal((3, 4)), rng.standard_normal((4, 5))
  out.append(H(tn.ncon([a, b], [["-a", "x"], ["x", "-b"]], backend=be)))
  # twice the same structure: second call goes through the cached jitted ncon
  for _ in range(2):
    ts = [rng.standard_normal(s) for s in NCON_CASES[4][0]]
    out.append(H(tn.ncon(ts, NCON_CASES[4][1], con_order=NCON_CASES[4][2], backend=be)))
  return out


def _mps_norm_nodes(tn, be, kets):
  L = len(kets)
  k = [tn.Node(x, backend=be) for x in kets]
  b = [tn.Node(np.conj(x), backend=be) for x in kets]
  for i in range(L):
    k[i][1] ^ b[i][1]
    if i + 1 < L:
      k[i][2] ^ k[i + 1][0]
      b[i][2] ^ b[i + 1][0]
  k[0][0] ^ b[0][0]
  k[-1][2] ^ b[-1][2]
  return k + b


def mps_kets(rng, L, D, dtype=np.float64):
  dims = [1] + [min(D, 2**min(i, L - i)) for i in range(1, L)] + [1]
  return [(rng.standard_normal((dims[i], 2, dims[i + 1])) / np.sqrt(dims[i])).astype(dtype)
          for i in range(L)]


def case_contractors(tn, be, seed=5):
  rng = np.random.default_rng(seed)
  kets = mps_kets(rng, 10, 16)
  out = [H(tn.contractors.greedy(_mps_norm_nodes(tn, be, kets)).tensor)]
  kets = mps_kets(rng, 3, 4)     # 6 nodes: the stand-in optimal search (numpy's brute force, baseline/refenv.py) is exponential
  out.append(H(tn.contractors.optimal(_mps_norm_nodes(tn, be, kets)).tensor))
  out.append(H(tn.contractors.auto(_mps_norm_nodes(tn, be, kets)).tensor))
  # open network with an output edge order (path_contractors.py:79-97)
  a, b, c = rng.standard_normal((4, 5)), rng.standard_normal((5, 6, 3)), rng.standard_normal((6, 7))
  na, nb, nc = tn.Node(a, backend=be), tn.Node(b, backend=be), tn.Node(c, backend=be)
  na[1] ^ nb[0]
  nb[1] ^ nc[0]
  r = tn.contractors.greedy([na, nb, nc], output_edge_order=[nc[1], nb[2], na[0]])
  out.append(H(r.tensor))
  # complex MPS
  kets = [k + 1j * rng.standard_normal(k.shape) for k in mps_kets(rng, 6, 8)]
  out.append(H(tn.contractors.greedy(_mps_norm_nodes(tn, be, kets)).tensor))
  return out


def case_split_node(tn, be, seed=6):
  """Returns reconstructions and singular values (the factors themselves are only defined up to
  per-vector phases)."""
  rng = np.random.default_rng(seed)
  t4 = rng.standard_normal((4, 5, 6, 3))
  out = []
  for kw in ({}, {"max_singular_values": 7}, {"max_truncation_err": 0.5, "relative": True},
             {"max_truncation_err": 2.0}):
    n = tn.Node(t4, backend=be)
    l, r, e = tn.split_node(n, [n[0], n[1]], [n[2], n[3]], **kw)
    out += [np.tensordot(H(l.tensor), H(r.tensor), 1), np.sort(np.abs(H(e)))[::-1]]
  n = tn.Node(t4, backend=be)
  u, s, vh, e = tn.split_node_full_svd(n, [n[1], n[0]], [n[3], n[2]], max_singular_values=5)  # mixed order
  out += [np.tensordot(np.tensordot(H(u.tensor), H(s.tensor), 1), H(vh.tensor), 1),
          np.diag(H(s.tensor)), np.sort(np.abs(H(e)))[::-1]]
  n = tn.Node(t4, backend=be)
  q, r = tn.split_node_qr(n, [n[0], n[1]], [n[2], n[3]])
  out += [H(q.tensor), H(r.tensor)]                   # LAPACK sign convention => factors comparable
  n = tn.Node(t4, backend=be)
  r, q = tn.split_node_rq(n, [n[0], n[1]], [n[2], n[3]])
  out += [H(r.tensor), H(q.tensor)]
  c4 = (t4 + 1j * rng.standard_normal(t4.shape)).astype(np.complex128)
  n = tn.Node(c4, backend=be)
  l, r, e = tn.split_node(n, [n[0], n[1]], [n[2], n[3]], max_singular_values=9)
  out += [np.tensordot(H(l.tensor), H(r.tensor), 1), np.sort(np.abs(H(e)))[::-1]]
  return out


def case_copy_node_and_bucket(tn, be, seed=7):
  """bucket_contractor_test.py: CNOT built from a CopyNode + XOR tensor; plus a rank-4 CopyNode
  contracted with three random partners (network_components.py:903-908)."""
  rng = np.random.default_rng(seed)
  out = []
  for bits_in, bits_out in (((0, 1), (0, 1)), ((1, 1), (1, 0)), ((1, 0), (1, 1))):
    def basis(b):
      v = np.zeros(2)
      v[b] = 1.0
      return v
    q0i, q1i = tn.Node(basis(bits_in[0]), backend=be), tn.Node(basis(bits_in[1]), backend=be)
    q0o, q1o = tn.Node(basis(bits_out[0]), backend=be), tn.Node(basis(bits_out[1]), backend=be)
    control = tn.CopyNode(rank=3, dimension=2, backend=be)
    xor = np.array([[[1, 0], [0, 1]], [[0, 1], [1, 0]]], dtype=np.float64)
    target = tn.Node(xor, backend=be)
    q0i[0] ^ control[0]
    q1i[0] ^ target[0]
    control[1] ^ target[1]
    control[2] ^ q0o[0]
    target[2] ^ q1o[0]
    net = tn.contractors.bucket([q0i, q1i, q0o, q1o, control, target], (control,))
    out.append(H(tn.contractors.greedy(net).tensor))
  cn = tn.CopyNode(rank=4, dimension=5, backend=be)
  a, b, c = rng.standard_normal((5, 3)), rng.standard_normal((4, 5, 2)), rng.standard_normal((5,))
  na, nb, nc = tn.Node(a, backend=be), tn.Node(b, backend=be), tn.Node(c, backend=be)
  cn[0] ^ na[0]
  cn[1] ^ nb[1]
  cn[2] ^ nc[0]
  d = rng.standard_normal((5, 6))
  nd = tn.Node(d, backend=be)
  cn[3] ^ nd[0]
  r = tn.contract_copy_node(cn)
  out.append(H(r.tensor))
  # a CopyNode's own tensor, contracted pairwise (Node @ CopyNode)
  cn = tn.CopyNode(rank=3, dimension=4, backend=be)
  x = tn.Node(rng.standard_normal((4, 6)), backend=be)
  cn[0] ^ x[0]
  out.append(H((cn @ x).tensor))
  return out


def case_dmrg(tn, be, seed=10, N=6, D=8, sweeps=4):
  """matrixproductstates/dmrg_test.py style: XXZ chain, energy after two-site sweeps."""
  np.random.seed(seed)
  mps = tn.FiniteMPS.random([2] * N, [D] * (N - 1), dtype=np.float64, backend=be)
  mpo = tn.FiniteXXZ(np.ones(N - 1), np.ones(N - 1), np.zeros(N), dtype=np.float64, backend=be)
  dmrg = tn.FiniteDMRG(mps, mpo)
  e = dmrg.run_two_site(max_bond_dim=D, num_sweeps=sweeps, num_krylov_vecs=10, verbose=0)
  bond_dims = np.array(mps.bond_dimensions)
  return [np.asarray(float(np.real(np.asarray(e)))), bond_dims]


def case_mps_ops(tn, be, seed=11):
  """base_mps.py canonicalisation (qr/rq/svd on the backend), norms and one-site expectation."""
  np.random.seed(seed)
  N, D = 8, 6
  mps = tn.FiniteMPS.random([2] * N, [D] * (N - 1), dtype=np.float64, backend=be, canonicalize=True)
  out = [np.asarray(float(np.real(np.asarray(mps.check_canonical()))))]
  mps.position(3)
  out.append(np.asarray(float(np.real(np.asarray(mps.check_canonical())))))
  sz = np.diag([0.5, -0.5])
  vals = mps.measure_local_operator([sz] * N, range(N))
  out.append(np.array([float(np.real(np.asarray(v))) for v in vals]))
  return out


CASES = [
    ("node_matmul", case_node_matmul, 1e-12),
    ("contract_between_flip", case_contract_between_flip, 1e-12),
    ("trace_and_flatten", case_trace_and_flatten, 1e-12),
    ("integer_nodes", case_integer_nodes, 0.0),
    ("ncon", case_ncon, 1e-12),
    ("contractors", case_contractors, 1e-11),
    ("split_node", case_split_node, 1e-10),
    ("copy_node_and_bucket", case_copy_node_and_bucket, 1e-12),
    ("mps_ops", case_mps_ops, 1e-9),
    ("dmrg", case_dmrg, 1e-8),
]


def compare(name, got, ref, tol):
  assert len(got) == len(ref), (name, len(got), len(ref))
  for i, (g, r) in enumerate(zip(got, ref)):
    g, r = np.asarray(g), np.asarray(r)
    assert g.shape == r.shape, "{}[{}]: shape {} vs {}".format(name, i, g.shape, r.shape)
    if r.dtype.kind in "iu" and g.dtype.kind in "iu":
      np.testing.assert_array_equal(g, r, err_msg="{}[{}]".format(name, i))
      continue
    scale = max(1.0, float(np.max(np.abs(r))) if r.size else 1.0)
    err = float(np.max(np.abs(g - r))) if r.size else 0.0
    assert err <= tol * scale, "{}[{}]: max abs err {:.3e} > {:.1e}*{:.2g}".format(name, i, err, tol, scale)
