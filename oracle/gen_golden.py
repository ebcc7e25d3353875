"""Generate tests/golden/*.npz by running the REAL reference (numpy backend).

Needs the reference installed in oracle/_ref (oracle/build_ref.py):  python -m oracle.gen_golden
Inputs are seeded; every array the reference returned is stored next to its inputs and
a JSON description of the call, so the fixtures can be replayed against (a) the oracle
restatement (tests/test_oracle_golden.py, CPU) and (b) the CUDA path (tests -m gpu).
"""
import json
import os
import numpy as np
from . import ref_shim

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                   "tests", "golden")


def _save(name, meta, arrays):
  os.makedirs(OUT, exist_ok=True)
  np.savez_compressed(os.path.join(OUT, name + ".npz"),
                      __meta__=np.array(json.dumps(meta)), **arrays)
  print("wrote", name, len(meta), "cases")


def gen_tensordot(tn):
  be = tn.backends.backend_factory.get_backend("numpy")
  rng = np.random.default_rng(101)
  cases = [
      # (shape_a, shape_b, axes, dtype, perm_a, perm_b)
      ((10, 10), (10, 10), [[1], [0]], "float64", None, None),
      ((2, 3, 4), (2, 3, 4), [[1, 2], [1, 2]], "float64", None, None),
      ((2, 3, 4), (4, 3, 2), [[0, 1, 2], [2, 1, 0]], "float64", None, None),
      ((5, 6, 7), (7, 6, 3), 1, "float64", None, None),
      ((4, 5), (6,), 0, "float32", None, None),
      ((16, 2, 16), (16, 2, 16), [[2], [0]], "float64", None, None),
      ((16, 2, 16), (16, 2, 16), [[0], [2]], "float64", None, None),
      ((16, 2, 16), (16, 2, 16), [[2], [2]], "float32", None, None),
      ((16, 2, 16), (16, 2, 16), [[0], [0]], "float32", None, None),
      ((16, 2, 16), (16, 2, 16), [[0, 1], [0, 1]], "float64", None, None),
      ((16, 2, 16), (16, 2, 16), [[1], [1]], "float64", None, None),
      ((6, 5, 4, 3), (3, 5, 7), [[2, 3], [0, 1]], "float64", (2, 0, 3, 1), None),
      ((6, 5, 4, 3), (3, 5, 7), [[3, 1], [2, 1]], "complex128", None, (2, 1, 0)),
      ((8, 9), (9, 8), [[0, 1], [1, 0]], "complex64", None, None),
      ((4, 4, 4), (4, 4), [[0], [1]], "int64", None, None),
      ((3, 1, 5), (5, 1, 2), [[2], [0]], "float16", None, None),
      ((33, 17), (17, 65), [[1], [0]], "float32", None, None),
      ((130, 70), (70, 129), [[1], [0]], "float64", None, None),
      ((0, 4), (4, 3), [[1], [0]], "float64", None, None),
      ((64, 2, 64), (64, 2, 64), [[2], [0]], "float32", None, None),
  ]
  meta, arrays = [], {}
  for i, (sa, sb, axes, dt, pa, pb) in enumerate(cases):
    def mk(shape):
      if dt.startswith("int"):
        return rng.integers(-5, 6, size=shape).astype(dt)
      x = rng.standard_normal(shape)
      if dt.startswith("complex"):
        x = x + 1j * rng.standard_normal(shape)
      return x.astype(dt)
    a, b = mk(sa), mk(sb)
    av = a if pa is None else be.transpose(a, pa)
    bv = b if pb is None else be.transpose(b, pb)
    # axes refer to the (possibly transposed) views that are passed in
    out = be.tensordot(av, bv, axes)
    meta.append(dict(axes=axes, dtype=dt, perm_a=pa, perm_b=pb))
    arrays["a%d" % i], arrays["b%d" % i], arrays["out%d" % i] = a, b, np.asarray(out)
  _save("tensordot", meta, arrays)


def gen_ncon(tn):
  rng = np.random.default_rng(102)
  r = lambda *s: rng.standard_normal(s)
  cases = [
      ([r(10, 10), r(10, 10)], [(-1, 1), (1, -2)], None, None),
      ([r(4, 5, 6), r(6, 5, 3)], [(-1, 1, 2), (2, 1, -2)], None, None),
      ([r(3, 4, 4), r(3, 5)], [(1, 2, 2), (1, -1)], None, None),         # partial trace
      ([r(3, 3, 4), r(4, 5), r(5,)], [(1, 1, 2), (2, 3), (3,)], None, None),
      ([r(2, 3), r(4, 5)], [(-1, -2), (-3, -4)], None, None),            # outer product
      ([r(2, 3), r(4, 5)], [(-1, -2), (-3, -4)], None, [-3, -1, -4, -2]),
      ([r(3, 4, 5), r(5, 4, 6), r(6, 3)], [(1, 2, 3), (3, 2, 4), (4, 1)], [3, 2, 4, 1], None),
      ([r(7, 3, 4), r(7, 4, 5)], [(-1, -2, 1), (-1, 1, -3)], None, None),  # batch (matmul)
      ([r(6, 3, 4), r(6, 4, 5), r(6, 5, 2)], [(1, -2, 2), (1, 2, 3), (1, 3, -3)], None, None),
      ([r(4, 5), r(5, 6), r(6, 7), r(7, 4)], [(1, 2), (2, 3), (3, 4), (4, 1)], None, None),
      ([r(3, 4, 5)], [(-3, -1, -2)], None, None),
      ([r(3, 4, 3)], [(1, -1, 1)], None, None),
      ([r(4, 2, 5), r(5, 2, 6), r(4, 2, 7), r(7, 2, 6)],
       [("a", "p1", "b"), ("b", "p2", "c"), ("a", "p1", "d"), ("d", "p2", "c")], None, None),
      ([r(3, 4), r(4, 5)], [("-x", "k"), ("k", "-y")], None, ["-y", "-x"]),
  ]
  meta, arrays = [], {}
  for i, (ts, net, con, out) in enumerate(cases):
    res = tn.ncon([t.copy() for t in ts], net, con_order=con, out_order=out,
                  backend="numpy")
    meta.append(dict(net=[list(n) for n in net], con=con, out=out, n=len(ts)))
    for j, t in enumerate(ts):
      arrays["c%d_t%d" % (i, j)] = t
    arrays["c%d_out" % i] = np.asarray(res)
  _save("ncon", meta, arrays)


def gen_decomp(tn):
  be = tn.backends.backend_factory.get_backend("numpy")
  rng = np.random.default_rng(103)
  meta, arrays = [], {}

  def add(kind, t, kwargs):
    i = len(meta)
    arrays["in%d" % i] = t
    res = getattr(be, kind)(t.copy(), **kwargs)
    for j, x in enumerate(res):
      arrays["out%d_%d" % (i, j)] = np.asarray(x)
    meta.append(dict(kind=kind, kwargs=kwargs, nout=len(res)))

  # decompositions_test.py:55-66 style: constructed spectrum 0..9
  def spectrum_matrix(n, svals, dtype="float64"):
    u = np.linalg.qr(rng.standard_normal((n, n)))[0]
    v = np.linalg.qr(rng.standard_normal((n, n)))[0]
    return (u @ np.diag(svals) @ v).astype(dtype)
  m = spectrum_matrix(10, np.arange(10.0))
  add("svd", m, dict(pivot_axis=1))
  add("svd", m, dict(pivot_axis=1, max_singular_values=7))
  add("svd", m, dict(pivot_axis=1, max_singular_values=20))
  add("svd", m, dict(pivot_axis=1, max_truncation_error=np.sqrt(5.1)))
  add("svd", spectrum_matrix(10, np.arange(2.0, 12.0)),
      dict(pivot_axis=1, max_truncation_error=0.5, relative=True))
  add("svd", spectrum_matrix(10, np.arange(2.0, 12.0)),
      dict(pivot_axis=1, max_truncation_error=0.5, relative=False))
  add("svd", rng.standard_normal((2, 3, 4, 5)), dict(pivot_axis=2))
  add("svd", rng.standard_normal((6, 4, 5)), dict(pivot_axis=1, max_singular_values=3))
  add("svd", rng.standard_normal((30, 12)).astype("float32"), dict(pivot_axis=1))
  add("svd", rng.standard_normal((12, 30)), dict(pivot_axis=1, max_singular_values=5,
                                                 max_truncation_error=1e-3, relative=True))
  add("svd", (rng.standard_normal((8, 8)) + 1j * rng.standard_normal((8, 8))),
      dict(pivot_axis=1, max_singular_values=4))
  add("svd", rng.standard_normal((64, 64)), dict(pivot_axis=1, max_singular_values=16))
  for nn in (False, True):
    add("qr", rng.standard_normal((2, 3, 4, 5)), dict(pivot_axis=2, non_negative_diagonal=nn))
    add("rq", rng.standard_normal((2, 3, 4, 5)), dict(pivot_axis=2, non_negative_diagonal=nn))
    add("qr", rng.standard_normal((20, 6)), dict(pivot_axis=1, non_negative_diagonal=nn))
    add("rq", rng.standard_normal((6, 20)), dict(pivot_axis=1, non_negative_diagonal=nn))
    add("qr", rng.standard_normal((6, 20)).astype("float32"),
        dict(pivot_axis=1, non_negative_diagonal=nn))
  _save("decomp", meta, arrays)


def _mps_norm_network(rng, L, D, d=2, dtype="float64"):
  """<psi|psi> closed network, SURVEY 8(d) cfg 2 (tensors scaled by 1/sqrt(contracted dims))."""
  dims = [1] + [min(D, d**min(i, L - i)) for i in range(1, L)] + [1]
  kets = []
  for i in range(L):
    t = rng.standard_normal((dims[i], d, dims[i + 1])) / np.sqrt(dims[i] * d)
    kets.append(t.astype(dtype))
  return kets


def mps_norm_labels(L):
  """ncon-style labels of <psi|psi>: ket i (k_i, p_i, k_{i+1}), bra i (b_i, p_i, b_{i+1});
  boundary legs (dimension 1) of ket and bra are tied together."""
  labels = []
  for i in range(L):
    labels.append(["k%d" % i if 0 < i else "e0", "p%d" % i,
                   "k%d" % (i + 1) if i + 1 < L else "eL"])
  for i in range(L):
    labels.append(["b%d" % i if 0 < i else "e0", "p%d" % i,
                   "b%d" % (i + 1) if i + 1 < L else "eL"])
  return labels


def gen_greedy(tn):
  rng = np.random.default_rng(104)
  meta, arrays = [], {}
  for ci, (L, D, dt) in enumerate([(6, 8, "float64"), (10, 16, "float64"),
                                   (8, 4, "float32")]):
    kets = _mps_norm_network(rng, L, D, dtype=dt)
    tensors = kets + [np.conj(k) for k in kets]
    labels = mps_norm_labels(L)
    nodes = [tn.Node(t, backend="numpy") for t in tensors]
    where = {}
    for n, labs in enumerate(labels):
      for ax, l in enumerate(labs):
        where.setdefault(l, []).append((n, ax))
    for l, ends in where.items():
      (n1, a1), (n2, a2) = ends
      tn.connect(nodes[n1][a1], nodes[n2][a2])
    res = tn.contractors.greedy(nodes)
    meta.append(dict(L=L, D=D, dtype=dt, labels=labels))
    for j, t in enumerate(kets):
      arrays["c%d_k%d" % (ci, j)] = t
    arrays["c%d_out" % ci] = np.asarray(res.tensor)
  # an open network: 3 tensors with dangling legs and an explicit output order
  a = rng.standard_normal((4, 5, 6))
  b = rng.standard_normal((6, 7, 3))
  c = rng.standard_normal((3, 5, 2))
  na, nb_, nc = [tn.Node(x, backend="numpy") for x in (a, b, c)]
  tn.connect(na[2], nb_[0]); tn.connect(nb_[2], nc[0]); tn.connect(na[1], nc[1])
  res = tn.contractors.greedy([na, nb_, nc], output_edge_order=[nc[2], na[0], nb_[1]])
  arrays["open_a"], arrays["open_b"], arrays["open_c"] = a, b, c
  arrays["open_out"] = np.asarray(res.tensor)
  meta.append(dict(open=True, labels=[["i", "x", "y"], ["y", "j", "z"], ["z", "x", "k"]],
                   out=["k", "i", "j"]))
  _save("greedy", meta, arrays)


def gen_split(tn):
  rng = np.random.default_rng(105)
  meta, arrays = [], {}
  t = rng.standard_normal((4, 5, 6, 3))
  arrays["t"] = t

  def rec(name, nodes_or_arrays):
    for j, x in enumerate(nodes_or_arrays):
      arrays["%s_%d" % (name, j)] = np.asarray(x.tensor if hasattr(x, "tensor") else x)
    meta.append(dict(name=name, n=len(nodes_or_arrays)))

  n = tn.Node(t, backend="numpy")
  l, r, terr = tn.split_node(n, [n[0], n[1]], [n[2], n[3]])
  rec("split_full", [l, r, terr])
  n = tn.Node(t, backend="numpy")
  l, r, terr = tn.split_node(n, [n[0], n[1]], [n[2], n[3]], max_singular_values=7)
  rec("split_k7", [l, r, terr])
  n = tn.Node(t, backend="numpy")
  l, r, terr = tn.split_node(n, [n[2], n[0]], [n[3], n[1]], max_singular_values=5)
  rec("split_mixed_k5", [l, r, terr])
  n = tn.Node(t, backend="numpy")
  u, s, vh, terr = tn.split_node_full_svd(n, [n[0], n[1]], [n[2], n[3]], max_singular_values=6)
  rec("fullsvd_k6", [u, s, vh, terr])
  n = tn.Node(t, backend="numpy")
  u, s, vh, terr = tn.split_node_full_svd(n, [n[0], n[1]], [n[2], n[3]],
                                          max_truncation_err=0.8, relative=True)
  rec("fullsvd_err", [u, s, vh, terr])
  n = tn.Node(t, backend="numpy")
  q, rr = tn.split_node_qr(n, [n[0], n[1]], [n[2], n[3]])
  rec("qr", [q, rr])
  n = tn.Node(t, backend="numpy")
  rr, q = tn.split_node_rq(n, [n[0], n[1]], [n[2], n[3]])
  rec("rq", [rr, q])
  _save("split", meta, arrays)


def gen_lanczos(tn):
  be = tn.backends.backend_factory.get_backend("numpy")
  rng = np.random.default_rng(106)
  meta, arrays = [], {}
  for i, (n, nk, reorth, numeig) in enumerate([(40, 20, False, 1), (64, 30, True, 2),
                                               (100, 10, False, 1)]):
    h = rng.standard_normal((n, n))
    h = (h + h.T) / 2
    x0 = rng.standard_normal((n,))

    def mv(x, mat):
      return mat @ x
    ev, vecs = be.eigsh_lanczos(mv, [h], x0.copy(), num_krylov_vecs=nk, numeig=numeig,
                                reorthogonalize=reorth, ndiag=5)
    arrays["h%d" % i], arrays["x%d" % i] = h, x0
    arrays["ev%d" % i] = np.asarray(ev)
    arrays["vec%d" % i] = np.stack(vecs)
    meta.append(dict(n=n, num_krylov_vecs=nk, reorthogonalize=reorth, numeig=numeig, ndiag=5))
  _save("lanczos", meta, arrays)


def gen_blocksparse(tn):
  """block_sparse.tensordot (cfg 4 family): inputs, result data vector AND the reference's own
  int64 block maps (`_find_transposed_diagonal_sparse_blocks`), so our map builder can be checked
  bit-exactly (SURVEY 8a row a11: 'int maps bit-exact')."""
  from tensornetwork.block_sparse import BlockSparseTensor, Index, U1Charge, tensordot
  from tensornetwork.block_sparse.blocksparse_utils import _find_transposed_diagonal_sparse_blocks
  meta, arrays = [], {}
  cases = [
      # (seed, leg dim, charge range, flows, axes, transpose of A before the product)
      (5, 8, 2, [False, False, True, True], ([2, 3], [2, 3]), None),
      (6, 10, 3, [False, True, False, True], ([1, 3], [1, 3]), None),
      (7, 6, 2, [True, False, False, True], ([0, 2], [0, 2]), (2, 0, 3, 1)),
      (8, 12, 2, [False, False, True], ([2], [2]), None),
      (5, 32, 8, [False, False, True, True], ([2, 3], [2, 3]), None),   # cfg 4 itself
  ]
  for ci, (seed, dim, q, flows, axes, perm) in enumerate(cases):
    np.random.seed(seed)
    legs = [Index(U1Charge.random(dim, -q, q), f) for f in flows]
    A = BlockSparseTensor.random(legs, dtype=np.float64)
    At = A if perm is None else A.transpose(perm)
    Bc = At.conj()
    C = tensordot(At, Bc, axes)
    for li, leg in enumerate(legs):
      arrays["c%d_q%d" % (ci, li)] = np.asarray(leg.flat_charges[0].charges).ravel().astype(np.int64)
    arrays["c%d_A" % ci] = np.asarray(A.data)
    arrays["c%d_C" % ci] = np.asarray(C.contiguous().data)
    arrays["c%d_Cdense" % ci] = np.asarray(C.todense()) if dim <= 12 else np.zeros(0)
    # the reference's gather maps of the first operand for this contraction
    free1 = sorted(set(range(At.ndim)) - set(axes[0]))
    new_order1 = [At._order[n] for n in free1] + [At._order[n] for n in axes[0]]
    flat_order_1 = [x for sub in new_order1 for x in sub]
    nleft = sum(len(At._order[n]) for n in free1)
    blocks, qn, shapes = _find_transposed_diagonal_sparse_blocks(At._charges, At._flows, nleft, flat_order_1)
    arrays["c%d_mapcat" % ci] = np.concatenate([np.asarray(b).ravel() for b in blocks]).astype(np.int64)
    arrays["c%d_mapoff" % ci] = np.insert(np.cumsum([np.asarray(b).size for b in blocks]), 0, 0).astype(np.int64)
    arrays["c%d_shapes" % ci] = np.asarray(shapes).astype(np.int64)
    arrays["c%d_qnums" % ci] = np.asarray(qn.unique_charges).ravel().astype(np.int64)
    meta.append(dict(flows=flows, axes=[list(axes[0]), list(axes[1])], perm=perm, nlegs=len(legs), dim=dim))
  _save("blocksparse", meta, arrays)


def gen_symsvd(tn):
  """SymmetricBackend.svd (backends/symmetric/decompositions.py:27-216): singular values (kept, sector-major),
  discarded values and the dense reconstruction, for several truncation settings."""
  from tensornetwork.block_sparse import BlockSparseTensor, Index, U1Charge
  be = tn.backends.backend_factory.get_backend("symmetric")
  meta, arrays = [], {}
  cases = [(11, 10, 2, [False, False, True, True], 2, {}),
           (12, 10, 2, [False, False, True, True], 2, {"max_singular_values": 12}),
           (13, 12, 3, [False, True, False, True], 2, {"max_truncation_error": 0.5}),
           (14, 12, 2, [False, False, True], 1, {"max_truncation_error": 0.05, "relative": True, "max_singular_values": 9}),
           (15, 8, 2, [True, False, True, False], 3, {"max_singular_values": 5})]
  for ci, (seed, dim, q, flows, pivot, kw) in enumerate(cases):
    np.random.seed(seed)
    legs = [Index(U1Charge.random(dim, -q, q), f) for f in flows]
    A = BlockSparseTensor.random(legs, dtype=np.float64)
    U, S, V, Sd = be.svd(A, pivot, **kw)
    for li, leg in enumerate(legs):
      arrays["c%d_q%d" % (ci, li)] = np.asarray(leg.flat_charges[0].charges).ravel().astype(np.int64)
    arrays["c%d_A" % ci] = np.asarray(A.data)
    arrays["c%d_S" % ci] = np.asarray(S.data)
    arrays["c%d_Sdisc" % ci] = np.asarray(Sd.data)
    ud, vd = U.todense(), V.todense()
    k = ud.shape[-1]
    rec = np.tensordot(ud * np.asarray(S.todense()), vd, 1) if k else np.zeros(A.shape)
    arrays["c%d_rec" % ci] = rec
    arrays["c%d_dense" % ci] = A.todense()
    meta.append(dict(flows=flows, pivot=pivot, kwargs=kw, nlegs=len(legs), k=int(k)))
  _save("symsvd", meta, arrays)


def gen_dmrg(tn):
  """FiniteDMRG.run_two_site (matrixproductstates/dmrg.py:445) on XXZ chains: initial MPS tensors, the
  reference's final energy, and the exact-diagonalisation energy (dmrg_test.py:161-191 style)."""
  meta, arrays = [], {}
  for ci, (N, D, sweeps) in enumerate([(6, 8, 4), (8, 16, 4), (10, 12, 3)]):
    np.random.seed(10 + ci)
    mps = tn.FiniteMPS.random([2] * N, [D] * (N - 1), dtype=np.float64, backend="numpy")
    for j, t in enumerate(mps.tensors):
      arrays["c%d_mps%d" % (ci, j)] = np.array(t)
    mpo = tn.FiniteXXZ(np.ones(N - 1), np.ones(N - 1), np.zeros(N), dtype=np.float64, backend="numpy")
    for j, t in enumerate(mpo.tensors):
      arrays["c%d_mpo%d" % (ci, j)] = np.array(t)
    center = mps.center_position
    dm = tn.FiniteDMRG(mps, mpo)
    e = float(dm.run_two_site(max_bond_dim=D, num_sweeps=sweeps, num_krylov_vecs=10, verbose=2))
    # exact diagonalisation of the same Hamiltonian
    sz = np.diag([-0.5, 0.5]); sp = np.array([[0, 0], [1.0, 0]]); sm = sp.T
    H = np.zeros((2**N, 2**N))
    def op(o, i):
      m = np.eye(1)
      for k in range(N):
        m = np.kron(m, o if k == i else np.eye(2))
      return m
    for i in range(N - 1):
      H += op(sz, i) @ op(sz, i + 1) + 0.5 * (op(sp, i) @ op(sm, i + 1) + op(sm, i) @ op(sp, i + 1))
    ed = float(np.linalg.eigvalsh(H)[0])
    meta.append(dict(N=N, D=D, sweeps=sweeps, center=int(center), energy=e, ed=ed))
  _save("dmrg", meta, arrays)


def gen_tree(tn):
  """tn.contractors.greedy (path_contractors.py:165-193) on backend numpy over a scaled-down copy of bench.py's 32-tensor
  tree network (the strong-scaling workload), seeded inputs as in tests/test_host_logic_r2.py: the closed network's value."""
  import bench  # pylint: disable=import-outside-toplevel
  labels, _, shapes, _ = bench.ttn_network({"b3": 24, "b2": 8, "b1": 4, "p": 3})
  rng = np.random.default_rng(2)
  kets = [rng.standard_normal(shapes[i]) / np.sqrt(np.prod(shapes[i][1:])) for i in range(len(labels) // 2)]
  nodes = [tn.Node(t, backend="numpy") for t in kets + [np.conj(k) for k in kets]]
  seen = {}
  for node, labs in zip(nodes, labels):
    for ax, l in enumerate(labs):
      if l in seen:
        seen[l] ^ node[ax]
      else:
        seen[l] = node[ax]
  value = float(tn.contractors.greedy(nodes).tensor)
  _save("tree", [dict(dims={"b3": 24, "b2": 8, "b1": 4, "p": 3}, seed=2, greedy=value)], {})


def gen_ref_callers(tn):
  """Every case of tests/ref_cases.py (the reference's own callers: Node @, contract_between, ncon, contractors, split_node*,
  CopyNode / bucket, FiniteMPS, FiniteDMRG) on backend numpy: the arrays tests/test_gpu_reference_callers.py compares the
  cuda_b200 arm against."""
  import sys  # pylint: disable=import-outside-toplevel
  sys.path.insert(0, os.path.dirname(OUT))
  import ref_cases  # pylint: disable=import-outside-toplevel
  meta, arrays = [], {}
  for name, fn, _ in ref_cases.CASES:
    out = fn(tn, "numpy")
    for i, a in enumerate(out):
      arrays["%s__%d" % (name, i)] = np.asarray(a)
    meta.append(dict(name=name, outputs=len(out)))
  _save("ref_callers", meta, arrays)


def main():
  tn = ref_shim.load()
  assert tn.__version__ == "0.4.6"
  gen_tensordot(tn)
  gen_ncon(tn)
  gen_decomp(tn)
  gen_greedy(tn)
  gen_split(tn)
  gen_lanczos(tn)
  gen_blocksparse(tn)
  gen_dmrg(tn)
  gen_symsvd(tn)
  gen_tree(tn)
  gen_ref_callers(tn)


if __name__ == "__main__":
  main()
