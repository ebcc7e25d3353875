"""CPU-only checks of host logic added in round 2: the jit key / skeleton machinery, the strong-scaling benchmark network and
its partition, the charge-degeneracy arithmetic of the block-sparse planner."""
import os
import sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)


def test_jit_skeleton_roundtrip_and_keys():
  from tensornetwork_b200 import jit

  class T:            # stand-in leaf: anything that is not a list / tuple / B200Tensor is a constant
    pass
  flat = []
  nest = ([1, (2, "a")], 3.5, [("x",), []])
  skel = jit._flatten(nest, flat)
  assert flat == [] and jit._unflatten(skel, []) == nest
  k1 = jit._skeleton_key(skel)
  k2 = jit._skeleton_key(jit._flatten(([1, (2, "a")], 3.5, [("x",), []]), []))
  k3 = jit._skeleton_key(jit._flatten(([1, (2, "b")], 3.5, [("x",), []]), []))
  assert k1 == k2 and k1 != k3 and hash(k1) == hash(k2)
  try:
    jit._skeleton_key(jit._flatten(({"unhashable": 1},), []))
    raise AssertionError("expected TypeError for an unhashable constant")
  except TypeError:
    pass


def test_strong_scaling_network_and_partition():
  """bench.ttn_network: 32 tensors, closed; the greedy path's tree fans out 8 ways (bound ~7.9); the partition used at 2 and 4
  ranks is balanced to 1 %, keeps ket and bra halves together (only small tensors cross ranks) and lets a rank send only
  after it has received everything it needs (no cyclic wait between two ranks)."""
  import bench
  from tensornetwork_b200 import drivers, parallel
  from oracle import np_network as nn
  labels, sizes, shapes, dims = bench.ttn_network(None)
  assert len(labels) == 32 and all(sum(l in labs for labs in labels) == 2 for labs in labels for l in labs)
  path = drivers.greedy_path(labels, [], sizes)
  flops = [2.0 * m * k * n for m, k, n in nn.network_flops(labels, path, sizes)]
  n = len(labels)
  ssa = parallel.path_to_ssa(n, path)
  lab = {i: list(l) for i, l in enumerate(labels)}
  for a, b, o in ssa:
    sh = [l for l in lab[a] if l in lab[b]]
    lab[o] = [l for l in lab[a] if l not in sh] + [l for l in lab[b] if l not in sh]
  for world in (2, 4, 8):
    owner, transfers, info = parallel.partition_tree(n, path, flops, world)
    assert info["total"] / info["critical"] > 7.5
    assert max(info["per_rank"]) <= 1.02 * info["total"] / world
    if world <= 4:
      assert max(int(np.prod([sizes[l] for l in lab[t]])) for t, _, _, _ in transfers) <= 16 * 64 * 64
    # per rank, in program order: every receive precedes every send (=> no two ranks can wait on each other)
    producer = {o: i for i, (_, _, o) in enumerate(ssa)}
    for r in range(world):
      recv_keys = [before for t, src, dst, before in transfers if dst == r]      # needed before this step
      send_keys = [producer.get(t, -1) for t, src, dst, before in transfers if src == r]
      if recv_keys and send_keys:
        # everything this rank sends is produced by a step that comes after the last step it needs a receive for
        assert min(send_keys) >= max(recv_keys), (world, r, recv_keys, send_keys)


def test_sharded_schedule_has_no_cyclic_wait_with_serialised_p2p():
  """parallel.schedule_completes: NCCL point-to-point operations that complete strictly in issue order on every rank (torch's
  eagerly initialised process group, large messages).  The tree plan of the benchmark network completes on 2, 4 and 8 ranks;
  on 3 ranks it would not (ShardedNetwork raises instead of hanging), and neither does the plan that gathers all small joins
  on one rank — removed after it hung an 8-GPU run."""
  import bench
  from tensornetwork_b200 import drivers, parallel
  from oracle import np_network as nn
  labels, sizes, shapes, dims = bench.ttn_network(None)
  path = drivers.greedy_path(labels, [], sizes)
  flops = [2.0 * m * k * n for m, k, n in nn.network_flops(labels, path, sizes)]
  n = len(labels)
  ssa = parallel.path_to_ssa(n, path)
  lab = {i: list(l) for i, l in enumerate(labels)}
  for a, b, o in ssa:
    sh = [l for l in lab[a] if l in lab[b]]
    lab[o] = [l for l in lab[a] if l not in sh] + [l for l in lab[b] if l not in sh]
  tb = {t: int(np.prod([sizes[l] for l in lab[t]] or [1])) * 8 for t in lab}

  def completes(world, tensor_bytes):
    owner, transfers, _ = parallel.partition_tree(n, path, flops, world, tensor_bytes=tensor_bytes)
    return parallel.schedule_completes(n, ssa, owner, transfers, world)
  ok = {world: completes(world, None) for world in range(2, 9)}
  assert ok[2] and ok[4] and ok[8], ok           # the world sizes the driver's scaling run uses
  assert not ok[3]                               # three ranks each open with a large send to the next: ShardedNetwork refuses
  assert not completes(8, tb)                    # the gathered-joins plan: rank 0 and rank 1 wait on each other


def test_blocksparse_degeneracy_arithmetic():
  from tensornetwork_b200 import blocksparse as bs
  rng = np.random.default_rng(3)
  for _ in range(100):
    n = int(rng.integers(1, 6))
    mod = [None, None, 2, 3, 5][rng.integers(0, 5)]
    idx = [bs.Index(rng.integers(-3, 4, rng.integers(1, 7)) if mod is None else rng.integers(0, mod, rng.integers(1, 7)),
                    bool(rng.integers(0, 2)), mod) for _ in range(n)]
    assert bs._count_allowed(idx) == bs._fused_allowed(idx).shape[0]
    shift = 0 if mod else int(sum(int(np.abs(bs._signed(ix)).max()) for ix in idx))
    nbins = int(mod) if mod else 2 * shift + 1
    h = bs._group_hist(idx, list(range(n)), shift, mod, nbins)
    fused = bs._fused_dense(idx, mod)
    ref = np.bincount(fused if mod else fused + shift, minlength=nbins)
    np.testing.assert_array_equal(h, ref)


def test_strong_scaling_network_oracle_equals_the_reference(golden):
  """The strong-scaling record checks the sharded result against the numpy oracle (`oracle.np_network.contract_path`); here the
  oracle itself is pinned, on a scaled-down copy of the same 32-tensor tree network, to the unmodified reference
  (`tn.contractors.greedy` on backend numpy, value stored by oracle/gen_golden.py:gen_tree in tests/golden/tree.npz)."""
  import bench
  from oracle import np_network as nn
  meta, _ = golden("tree")
  dims, seed, ref = meta[0]["dims"], meta[0]["seed"], meta[0]["greedy"]
  labels, sizes, shapes, _ = bench.ttn_network(dims)
  rng = np.random.default_rng(seed)
  n_ket = len(labels) // 2
  kets = [rng.standard_normal(shapes[i]) / np.sqrt(np.prod(shapes[i][1:])) for i in range(n_ket)]
  host = kets + [np.conj(k) for k in kets]
  path = nn.greedy_path(labels, [], sizes)
  want = float(nn.contract_path(host, labels, path, []))
  assert abs(ref - want) <= 1e-12 * abs(want)
