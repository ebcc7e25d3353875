#!/usr/bin/env python
"""bench.py — headline benchmark of the cuda_b200 hot path (contract: see DESIGN.md §Measurement).

A *step* is one full greedy contraction of the closed <psi|psi> network of an L=64,
bond-dim-512, phys-dim-2 MPS (BASELINE.json configs[1]; 128 tensors -> 127 pairwise
contractions, SURVEY.md 8(d) cfg 2, seed 3, tensors scaled by 1/sqrt(contracted dims)).
`value` = pairwise contractions per second with inputs resident in HBM; `e2e` = the same
metric through the public API with HOST (pinned) input buffers, H2D + D2H inside the timed
region.  `--impl reference` times the reference's own CPU algorithm (numpy backend restated
in oracle/, all host threads) on the same workload.  N > 1 (torchrun): every rank contracts
its own independent MPS sample (weak scaling, no data-path collective).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

L_SITES, BOND, PHYS = 64, 512, 2


# ----------------------------------------------------------------------------- workload
def mps_dims(L, D, d):
  return [1] + [min(D, d**min(i, L - i)) for i in range(1, L)] + [1]


def make_kets(L, D, d, seed):
  rng = np.random.default_rng(seed)
  dims = mps_dims(L, D, d)
  return [rng.standard_normal((dims[i], d, dims[i + 1])) / np.sqrt(dims[i] * d) for i in range(L)]


def norm_labels(L):
  labels = []
  for side in "kb":
    for i in range(L):
      labels.append(["e0" if i == 0 else "%s%d" % (side, i), "p%d" % i,
                     "eL" if i == L - 1 else "%s%d" % (side, i + 1)])
  return labels


def path_and_work(shapes, labels):
  from tensornetwork_b200 import drivers
  sizes = {l: s[ax] for s, labs in zip(shapes, labels) for ax, l in enumerate(labs)}
  path = drivers.greedy_path(labels, [], sizes)
  # algorithmic work per pairwise step: flops = 2MNK, bytes = (MK + KN + MN) * sizeof
  labs = [list(l) for l in labels]
  steps = []
  for a, b in path:
    l1, l2 = labs[a], labs[b]
    sh = [l for l in l1 if l in l2]
    K = int(np.prod([sizes[l] for l in sh])) if sh else 1
    M = int(np.prod([sizes[l] for l in l1 if l not in sh] or [1]))
    N = int(np.prod([sizes[l] for l in l2 if l not in sh] or [1]))
    steps.append((M, K, N))
    new = [l for l in l1 if l not in sh] + [l for l in l2 if l not in sh]
    for i in sorted([a, b], reverse=True):
      del labs[i]
    labs.append(new)
  return path, steps


# ------------------------------------------------------------------------------- output
_REAL_STDOUT = None


def quiet_stdout():
  """The driver reads ONE JSON line from stdout.  Libraries may write to file descriptor 1 directly (NCCL prints its
  version banner there): point fd 1 at stderr for the life of the process and keep the real stdout for emit()."""
  global _REAL_STDOUT
  if _REAL_STDOUT is None:
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line):
  data = (json.dumps(line) + "\n").encode()
  if _REAL_STDOUT is None:
    sys.stdout.write(data.decode())
    sys.stdout.flush()
  else:
    os.write(_REAL_STDOUT, data)


# ------------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
  QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
           "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
           "clocks_event_reasons.sw_power_cap,timestamp")

  def __init__(self, gpu_index=0):
    super().__init__(daemon=True)
    self.gpu = gpu_index
    self.samples = []
    self.times = []
    self.read_times = []
    self.window = None               # (t0, t1) host time of the timed region: summary() prefers samples inside it
    self.stop_flag = False

  def run(self):
    # one long-running nvidia-smi in loop mode (a fresh process per sample costs ~50 ms and would see
    # one or two samples of a 100 ms timed region)
    try:
      import shutil  # pylint: disable=import-outside-toplevel
      cmd = ["nvidia-smi", "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits", "-i", str(self.gpu), "-lms", "20"]
      if shutil.which("stdbuf"):
        cmd = ["stdbuf", "-oL"] + cmd              # line-buffered pipe: samples arrive as they are taken
      proc = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:  # pylint: disable=broad-except
      return
    try:
      for line in proc.stdout:
        f = [x.strip() for x in line.strip().split(",")]
        if len(f) >= 8:
          self.samples.append(f)
          t = time.time()                          # fallback: when the line was read
          self.read_times.append(t)
          if len(f) >= 9:
            try:                                   # nvidia-smi's own sampling time (the reader thread may lag behind)
              import datetime  # pylint: disable=import-outside-toplevel
              t = datetime.datetime.strptime(f[8], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except Exception:  # pylint: disable=broad-except
              pass
          self.times.append(t)
        if self.stop_flag:
          break
    finally:
      proc.terminate()
      try:
        proc.wait(timeout=2)
      except Exception:  # pylint: disable=broad-except
        proc.kill()

  def summary(self):
    if not self.samples:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    allsamples = self.samples
    if self.window is not None:
      for stamps in (self.times, self.read_times):      # nvidia-smi's own sampling time first, then arrival time
        inside = [s for s, t in zip(allsamples, stamps) if self.window[0] <= t <= self.window[1] + 0.05]
        if inside:
          self.samples = inside
          break
    sm = sorted(float(s[1]) for s in self.samples)
    reasons = []
    for name, col in (("hw_slowdown", 4), ("hw_thermal_slowdown", 5), ("sw_thermal_slowdown", 6),
                      ("sw_power_cap", 7)):
      if any(s[col].lower().startswith("active") for s in self.samples):
        reasons.append(name)
    return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][2]), "reasons": reasons,
            "samples": len(self.samples), "samples_total": len(allsamples)}


# ------------------------------------------------------------------------- reference arm
def tune_blas_threads(fn):
  """The reference's numpy backend is only as fast as its BLAS threading: on a many-core host OpenBLAS with ALL
  threads is slower on these mid-size GEMMs than with a few dozen.  Time `fn` (one network) under several thread
  limits and return (best_limit, context-manager factory) so the baseline is the reference at its best."""
  cores = os.cpu_count() or 1
  try:
    from threadpoolctl import threadpool_limits  # pylint: disable=import-outside-toplevel
  except ImportError:
    return cores, None
  best, best_t = cores, None
  for n in sorted({c for c in (8, 16, 32, 64, cores) if c <= cores}):
    with threadpool_limits(limits=n):
      fn()
      t0 = time.perf_counter()
      fn()
      dt = time.perf_counter() - t0
    if best_t is None or dt < best_t:
      best, best_t = n, dt
  return best, threadpool_limits


def reference_step_fn(np_dtype, nsamp):
  """One reference step = `nsamp` full <psi|psi> contractions through the reference's OWN code: tn.Node construction,
  edge wiring and `tn.contractors.greedy` (path_contractors.py:36-97,165-193 -> contract_between, network_components.py:1984-2095
  -> NumPyBackend.tensordot, numpy_backend.py:35-54) on backend="numpy", from the unmodified package installed under
  oracle/_ref by build().  Falls back to the oracle restatement (kind "port") only when that install is absent.
  Returns (step, kind, one_network)."""
  nets = [[k.astype(np_dtype) for k in make_kets(L_SITES, BOND, PHYS, 3 + b)] for b in range(nsamp)]
  from baseline import refenv  # pylint: disable=import-outside-toplevel
  tn = refenv.try_load()
  if tn is not None:
    def one(kets):
      n = len(kets)
      k = [tn.Node(x, backend="numpy") for x in kets]
      b = [tn.Node(np.conj(x), backend="numpy") for x in kets]
      for i in range(n):
        k[i][1] ^ b[i][1]
        if i + 1 < n:
          k[i][2] ^ k[i + 1][0]
          b[i][2] ^ b[i + 1][0]
      k[0][0] ^ b[0][0]
      k[-1][2] ^ b[-1][2]
      return tn.contractors.greedy(k + b).tensor
    kind = "reference"
  else:
    from oracle import np_network as nn  # pylint: disable=import-outside-toplevel
    labels = norm_labels(L_SITES)
    sizes = {l: t.shape[ax] for t, labs in zip(nets[0] + nets[0], labels) for ax, l in enumerate(labs)}

    def one(kets):
      path = nn.greedy_path(labels, [], sizes)   # the reference searches the path on every call
      return nn.contract_path(kets + [np.conj(k).copy() for k in kets], labels, path, [])
    kind = "port"

  def step():
    out = None
    for kets in nets:
      out = one(kets)
    return out
  return step, kind, (lambda: one(nets[0]))


def reference_measure(np_dtype, nsamp, steps, warmup):
  """-> dict(value, ms_per_step, cores, kind, sample, result): the reference at the BLAS thread count under which it is fastest"""
  step, kind, one = reference_step_fn(np_dtype, nsamp)
  threads, limiter = tune_blas_threads(one)
  import contextlib  # pylint: disable=import-outside-toplevel
  with (limiter(limits=threads) if limiter else contextlib.nullcontext()):
    for _ in range(warmup):
      step()
    t0 = time.perf_counter()
    for _ in range(steps):
      res = step()
    dt = time.perf_counter() - t0
  npair = 2 * L_SITES - 1
  return {"value": nsamp * npair * steps / dt, "ms_per_step": 1e3 * dt / steps, "cores": threads, "kind": kind,
          "result": float(np.real(res)),
          "sample": "%d network(s) per step x %d steps (127 pairwise each) through %s on numpy %s, BLAS threads = %d (fastest of "
                    "8/16/32/64/all on this host; %d logical cores)"
                    % (nsamp, steps, "the reference's tn.contractors.greedy (oracle/_ref)" if kind == "reference" else
                       "the oracle restatement", np.dtype(np_dtype).name, threads, os.cpu_count())}


NP_DTYPE = {"bf16": np.float32, "f32": np.float32, "f64": np.float64}


def run_reference(args, rank, world):
  """The reference arm: the UNMODIFIED reference (oracle/_ref) contracting the same workload on its own numpy backend,
  all the host threads it can use.  numpy has no bfloat16: for --dtype bf16 the reference computes in float32 (the narrowest
  type its BLAS supports) and the line says so; `by_dtype` carries the float32 AND float64 figures so that every GPU dtype
  has a like-for-like (or wider) reference number."""
  if rank != 0:
    return
  nsamp = min(max(1, args.networks), 2)
  main = reference_measure(NP_DTYPE[args.dtype], nsamp, args.steps, args.warmup)
  by = {}
  for name in ("f32", "f64"):
    if NP_DTYPE[args.dtype] == NP_DTYPE[name]:
      m = main
    else:
      m = reference_measure(NP_DTYPE[name], 1, max(1, min(args.steps, 3)), 1)
    by[name] = {"value": m["value"], "unit": "contractions/s", "cores": m["cores"], "kind": m["kind"], "sample": m["sample"]}
  val = main["value"]
  line = {
      "impl": "reference", "metric": "pairwise contractions/s", "value": val, "unit": "contractions/s",
      "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"],
      "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
      "dtype": "f32" if NP_DTYPE[args.dtype] == np.float32 else "f64", "data": "synthetic",
      "dtype_note": ("requested %s; numpy has no bfloat16, the reference computes in float32" % args.dtype) if args.dtype == "bf16" else None,
      "config": workload_config(args, 1),
      "cpu_baseline": {"value": val, "unit": "contractions/s", "cores": main["cores"], "kind": main["kind"], "sample": main["sample"]},
      "by_dtype": by,
      "e2e": {"value": val, "unit": "contractions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
      "result_check": main["result"],
  }
  emit(line)


def workload_config(args, world):
  return {"workload": "cfg2: <psi|psi> of MPS L=%d bond-dim %d phys-dim %d, greedy path, 127 pairwise contractions per network"
                      % (L_SITES, BOND, PHYS),
          "networks_per_step_per_gpu": max(1, args.networks), "launch_mode": "eager" if args.no_graph else "cuda-graph replay", "compute_dtype": args.dtype, "path_provider": "numpy greedy (opt_einsum stand-in)",
          "parallelism": "replicas x%d (independent MPS samples, no collective)" % world,
          "l2_policy": "no flush needed: one step reads %d x 128 input tensors = %.1f GB (bf16: 134 MB per network), far beyond the 126 MB L2"
                       % (max(1, args.networks), max(1, args.networks) * 0.134 * {"bf16": 1, "f32": 2, "f64": 4}[args.dtype])}


# ------------------------------------------------------------------------------ our arm
def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", default="cuda_b200", choices=["cuda_b200", "reference"])
  ap.add_argument("--dtype", default="bf16", choices=["bf16", "f32", "f64"])
  ap.add_argument("--networks", type=int, default=74,
                  help="independent MPS samples contracted in lock-step per step per GPU (batched kernels)")
  ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
  ap.add_argument("--cpu-baseline-steps", type=int, default=2)
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--no-e2e-overlap", action="store_true", help="e2e: copy and contract strictly in sequence (one compiled instance)")
  ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg1", "flagship", "flagship64", "cfg3", "cfg4", "cfg5", "tree32"],
                  help="cfg2 (default) is the headline line of the driver contract; the others are the remaining "
                       "SURVEY 8(d) configurations, single GPU, same JSON keys")
  ap.add_argument("--sub", action="store_true", help="internal: this process measures a sub-record of another bench line "
                  "(no nested sub-records, single BLAS thread setting for the CPU leg)")
  ap.add_argument("--no-strong-scaling", action="store_true", help="N > 1: skip the one-network strong-scaling sub-record")
  ap.add_argument("--no-subrecords", action="store_true", help="skip the by_dtype / configs sub-records of the default line")
  ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                  help="after the timed steps, write what the last timed step computed (the value of every network, "
                       "float64) to DIR/result.npy (DIR/result_rank<r>.npy with several ranks); the inputs are seeded, so "
                       "two builds run with the same arguments can be compared output for output")
  args = ap.parse_args()
  if args.dump_outputs is not None and (args.config != "cfg2" or args.impl != "cuda_b200"):
    ap.error("--dump-outputs writes the outputs of the default workload (--config cfg2 --impl cuda_b200)")
  quiet_stdout()
  args.warmup = max(args.warmup, 3) if args.impl == "cuda_b200" else max(args.warmup, 1)
  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  local = int(os.environ.get("LOCAL_RANK", "0"))

  if args.config != "cfg2":
    if rank == 0:
      run_config(args)
    return
  if args.impl == "reference":
    run_reference(args, rank, world)
    return

  import torch
  import torch.distributed as dist
  if world > 1:
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # rank 0's stdout carries exactly one JSON line
    import datetime  # pylint: disable=import-outside-toplevel
    dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=240))
  torch.cuda.set_device(local)
  import tensornetwork_b200 as tb
  from tensornetwork_b200 import drivers, _lib
  be = tb.get_backend()
  lib = be.lib
  sampler = ClockSampler(local)      # started early (nvidia-smi needs ~1 s to produce its first sample); only samples
  sampler.start()                    # inside the window [first warm-up step, end of the per-kernel pass] are reported

  code = {"bf16": _lib.BF16, "f32": _lib.F32, "f64": _lib.F64}[args.dtype]
  tdtype = {"bf16": torch.bfloat16, "f32": torch.float32, "f64": torch.float64}[args.dtype]
  esize = {"bf16": 2, "f32": 4, "f64": 8}[args.dtype]
  NB = max(1, args.networks)
  nbatch = 1 if NB > 1 else 0
  # NB independent MPS samples per rank, generated ON THE DEVICE by the library's Philox kernel (seeds differ
  # per rank / site; numpy would need ~30 s to draw 2.4e9 normals for NB = 74), scaled by 1/sqrt(contracted dims)
  dims = mps_dims(L_SITES, BOND, PHYS)
  labels = norm_labels(L_SITES)
  core_shapes = [(dims[i], PHYS, dims[i + 1]) for i in range(L_SITES)] * 2
  shapes = [((NB,) + cs) if nbatch else cs for cs in core_shapes]
  path, work = path_and_work(core_shapes, labels)
  npair = len(path)
  flops_step = NB * sum(2.0 * m * k * n for m, k, n in work)
  bytes_step = NB * sum((m * k + k * n + m * n) * esize for m, k, n in work)
  kets = []
  for i in range(L_SITES):
    t = be.randn(shapes[i], np.float32, seed=1 + 7919 * rank + i)
    t *= 1.0 / np.sqrt(dims[i] * PHYS)
    kets.append(be.astype(t, {"bf16": "bfloat16", "f32": np.float32, "f64": np.float64}[args.dtype]))
  # bra = conj(ket): the reference's caller builds it on the backend (`tn.conj(node)`); for real data conj is the
  # identity, so the 64 bra inputs are views of the ket buffers (conj_aliases) and only the kets cross PCIe
  dev = kets + list(kets)
  aliases = {L_SITES + i: i for i in range(L_SITES)}
  h2d_bytes = sum(int(np.prod(s)) * esize for s in shapes[:L_SITES])

  net = drivers.CompiledNetwork(be, shapes, {"bf16": "bfloat16", "f32": np.float32, "f64": np.float64}[args.dtype],
                                labels, [], path=path, nbatch=nbatch, conj_aliases=aliases) if not args.no_graph else None
  host = None
  if net is not None:
    net.load(dev)
    # the public API's pinned staging arena holds the step's 128 host tensors (filled once, outside the timed
    # region, with the same synthetic data; a user would generate / load their data straight into these views)
    host = net.host_staging()
    for dst, src in zip(host, dev):
      if dst is not None:
        dst.copy_(src.t)
  else:
    host = [d.t.cpu().pin_memory() for d in kets]
  torch.cuda.synchronize()

  def step_resident():
    if net is not None:
      return net()
    return drivers.contract_network(dev, labels, [], path=path, backend=be, nbatch=nbatch)

  def step_e2e():
    if net is not None:
      out = net.run_staged()    # ONE H2D of the pinned staging arena (all inputs), then graph replay
    else:
      ts = [tb.B200Tensor(h.to(be.device, non_blocking=True), code) for h in host]
      out = drivers.contract_network(ts + ts, labels, [], path=path, backend=be, nbatch=nbatch)
    return out.t.to("cpu")      # D2H of the result (one scalar per network; syncs)

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  # ---- device-resident timing ------------------------------------------------------
  win0 = time.time()
  for _ in range(args.warmup):
    res = step_resident()
  barrier()
  l0 = lib.tnb200_launch_count()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(args.steps):
    res = step_resident()
  e1.record()
  barrier()
  sampler.window = (win0, time.time())
  launches = (net.launches_per_replay * args.steps) if net is not None else (lib.tnb200_launch_count() - l0)
  ms = e0.elapsed_time(e1)
  result_host = np.atleast_1d(res.to_host().astype(np.float64))
  result_value = [float(x) for x in result_host]
  if args.dump_outputs is not None:
    os.makedirs(args.dump_outputs, exist_ok=True)
    np.save(os.path.join(args.dump_outputs, "result.npy" if world == 1 else "result_rank%d.npy" % rank), result_host)

  # ---- latency of ONE network (no sample batching): the same plan compiled for a single MPS sample
  single = None
  if nbatch and net is not None:
    one = [tb.B200Tensor(d.t[0], code) for d in dev]
    net1 = drivers.CompiledNetwork(be, core_shapes, {"bf16": "bfloat16", "f32": np.float32, "f64": np.float64}[args.dtype],
                                   labels, [], path=path, nbatch=0, conj_aliases=aliases)
    net1.load(one)
    for _ in range(3):
      net1()
    torch.cuda.synchronize()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(args.steps):
      net1()
    s1.record()
    torch.cuda.synchronize()
    ms1 = s0.elapsed_time(s1) / args.steps
    single = {"ms_per_network": ms1, "contractions_per_s": npair / (ms1 * 1e-3), "launches": net1.launches_per_replay,
              "note": "one network per graph replay (127 dependent launches, latency-bound)"}
    del net1, one

  # ---- per-kernel device times of one step (live, CUDA events) -> dominant kernel and its roofline
  if net is not None and getattr(net, "_nodes", None) is not None:
    kstats = net.profile(work, NB, esize)          # the nodes the graph replays (a chained launch is one node)
  else:
    kstats = kernel_profile(be, dev, labels, path, work, nbatch, NB, esize)

  torch.cuda.synchronize()
  sampler.window = (win0, time.time())   # warm-up + timed region + single-network + per-kernel pass: all compute load;
  sampler.stop_flag = True               # the PCIe-bound e2e section below is not part of the clock sample
  sampler.join(timeout=2)
  # ---- end-to-end timing (host buffers) ----------------------------------------------
  # Every step copies ITS inputs host->device (one transfer of the pinned staging arena) and reads ITS result back.
  # Two compiled instances ping-pong: the copy of step i+1 (copy stream) overlaps the contraction of step i (compute
  # stream); all contractions stay on one stream, in order.
  net_b = None
  if net is not None:
    nets = [net]
    if not args.no_e2e_overlap:
      try:
        net_b = drivers.CompiledNetwork(be, shapes, {"bf16": "bfloat16", "f32": np.float32, "f64": np.float64}[args.dtype],
                                        labels, [], path=path, nbatch=nbatch, conj_aliases=aliases)
        for dst, src in zip(net_b.host_staging(), dev):
          if dst is not None:
            dst.copy_(src.t)
        nets.append(net_b)
      except (RuntimeError, MemoryError) as exc:       # not enough device / pinned memory for a second instance
        sys.stderr.write("e2e overlap disabled (%s)\n" % str(exc).splitlines()[0])
        torch.cuda.empty_cache()
    copy_s, comp_s = torch.cuda.Stream(), torch.cuda.Stream()
    ev_in = [torch.cuda.Event() for _ in nets]
    ev_done = [torch.cuda.Event() for _ in nets]
    res_host = [torch.empty(max(NB, 1), dtype=tdtype).pin_memory() for _ in nets]

    def run_e2e(n):
      cur = torch.cuda.current_stream()
      copy_s.wait_stream(cur)
      comp_s.wait_stream(cur)
      for i in range(n):
        k = i % len(nets)
        with torch.cuda.stream(copy_s):
          if i >= len(nets):
            copy_s.wait_event(ev_done[k])          # instance k's previous step has consumed its inputs
          nets[k].stage()
          ev_in[k].record(copy_s)
        with torch.cuda.stream(comp_s):
          comp_s.wait_event(ev_in[k])
          out = nets[k]()
          res_host[k].copy_(out.t.reshape(-1), non_blocking=True)     # D2H of the step's result
          ev_done[k].record(comp_s)
      cur.wait_stream(copy_s)
      cur.wait_stream(comp_s)
  else:
    def run_e2e(n):
      for _ in range(n):
        step_e2e()
  run_e2e(args.warmup)
  barrier()
  t0 = torch.cuda.Event(enable_timing=True)
  t1 = torch.cuda.Event(enable_timing=True)
  t0.record()
  run_e2e(args.steps)
  t1.record()
  barrier()
  ms_e2e = t0.elapsed_time(t1)
  e2e_check = [float(x) for x in res_host[0][:4].float()] if net is not None else None

  e2e_mode = ("H2D of step i+1 overlapped with the contraction of step i (two compiled instances)"
              if (net is not None and len(nets) > 1) else "copy, contract, read back in sequence")
  strong = None
  if world > 1:
    tt = torch.tensor([ms, ms_e2e], device=be.device, dtype=torch.float64)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(tt[0]), float(tt[1])
    if not args.no_strong_scaling:
      # free the weak-scaling instances first (the tree network needs ~10 GB per rank)
      net = kets = dev = nets = net_b = host = res = None
      import gc  # pylint: disable=import-outside-toplevel
      gc.collect()
      torch.cuda.empty_cache()
      try:
        strong = strong_scaling_record(be, rank, world, dist, max(3, min(args.steps, 10)))
      except Exception as exc:  # pylint: disable=broad-except
        strong = {"error": "%s: %s" % (type(exc).__name__, str(exc).splitlines()[0] if str(exc) else "")}

  if rank == 0:
    peaks = {}
    try:
      peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # pylint: disable=broad-except
      pass
    if args.dtype == "bf16":
      peak, peak_src = peaks.get("bf16_tflops", 1590.0), ("measured" if peaks else "fallback")
      peak_note = "bf16 dense (cuBLAS burst), MEASURED_PEAKS.json" if peaks else "fallback 1.59 PF"
    elif args.dtype == "f32":
      peak = measured_peak("tf32")
      peak_src, peak_note = "measured", "tf32 dense: torch.matmul (cuBLAS, allow_tf32) 8192^3, best of 5, measured in this run"
    else:
      peak = measured_peak("f64")
      peak_src, peak_note = "measured", "fp64 dense: torch.matmul (cuBLAS DGEMM) 4096^3, best of 5, measured in this run"
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    if args.dtype == "bf16" and "bf16_tflops_sustained" in peaks:
      # the dominant kernel is timed inside a long step: the sustained figure is its tensor roof
      peak, peak_note = peaks["bf16_tflops_sustained"], "bf16 dense sustained (cuBLAS back to back), MEASURED_PEAKS.json"
    # dominant kernel = the family with the largest share of the step's device time
    ktot = sum(d["us"] for d in kstats.values())
    kern_name = max(kstats, key=lambda k: kstats[k]["us"])
    kd = kstats[kern_name]
    k_tf = kd["flops"] / (kd["us"] * 1e-6) / 1e12
    k_gbs = kd["bytes"] / (kd["us"] * 1e-6) / 1e9
    t_tensor, t_hbm = kd["flops"] / (peak * 1e12), kd["bytes"] / (hbm_peak * 1e9)
    if t_hbm >= t_tensor:
      roof = {"bound": "hbm", "achieved": k_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": k_gbs / hbm_peak}
    else:
      roof = {"bound": "tensor", "achieved": k_tf, "peak": peak, "unit": "TFLOP/s", "frac": k_tf / peak}
    traffic = None
    try:
      tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
      if tr.get("kernel") == kern_name and tr.get("dtype") == args.dtype and tr.get("networks") == NB:
        traffic = tr.get("dram_bytes_per_launch")
    except Exception:  # pylint: disable=broad-except
      pass
    roof.update({
        "traffic": traffic, "kernel": kern_name, "kernel_launches_per_step": kd["launches"],
        "kernel_us_per_launch": kd["us"] / kd["launches"], "kernel_share_of_step_time": kd["us"] / ktot,
        "algorithmic_mb_per_launch": kd["bytes"] / kd["launches"] / 1e6,
        "algorithmic_gflop_per_launch": kd["flops"] / kd["launches"] / 1e9,
        "kernel_tflops": k_tf, "kernel_gbs": k_gbs, "tensor_peak_tflops": peak, "hbm_peak_gbs": hbm_peak,
        "peak_source": peak_src, "peak_note": peak_note,
        "arithmetic_intensity_flop_per_byte": kd["flops"] / kd["bytes"], "ridge_flop_per_byte": peak * 1e3 / hbm_peak,
        "note": "dominant kernel timed live with CUDA events around each of its launches (eager replay of the "
                "step); algorithmic bytes = operands + result once, algorithmic flops = 2MNK; the binding roof "
                "is the one with the larger minimum time",
        "families": {k: {"launches": round(v["launches"], 2), "pairwise_steps": round(v.get("pairwise_steps", v["launches"]), 2),
                         "us": round(v["us"], 1),
                         "tflops": round(v["flops"] / (v["us"] * 1e-6) / 1e12, 1),
                         "gbs": round(v["bytes"] / (v["us"] * 1e-6) / 1e9, 1)} for k, v in kstats.items()},
    })
    achieved = flops_step * args.steps / (ms * 1e-3) / 1e12
    value = world * NB * npair * args.steps / (ms * 1e-3)
    line = {
        "metric": "pairwise contractions/s", "value": value, "unit": "contractions/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype,
        "data": "synthetic", "config": workload_config(args, world),
        "step_tflops": world * achieved,
        "step_hbm_gbs": world * bytes_step * args.steps / (ms * 1e-3) / 1e9,
        "launches_per_step": launches / args.steps,
        "algorithmic_gflop_per_step": flops_step / 1e9, "algorithmic_mb_per_step": bytes_step / 1e6,
        "roofline": roof,
        "e2e": {"value": world * NB * npair * args.steps / (ms_e2e * 1e-3), "unit": "contractions/s",
                "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": esize * NB,
                "ms_per_step": ms_e2e / args.steps, "result_check": e2e_check,
                "mode": e2e_mode},
        "gpu_launches": int(launches),
        "clocks": sampler.summary(),
        "result_check": result_value[:4],
        "single_network": single,
    }
    if strong is not None:
      line["strong_scaling"] = strong
    if not args.no_cpu_baseline and world == 1:
      line["cpu_baseline"] = cpu_baseline(args)
    if world == 1 and not args.sub and not args.no_subrecords and args.config == "cfg2":
      # release this process's device memory first: the sub-records run in fresh processes on the same GPU
      net = kets = dev = nets = net_b = host = res = None
      import gc  # pylint: disable=import-outside-toplevel
      gc.collect()
      torch.cuda.empty_cache()
      line.update(collect_subrecords(args))
    emit(line)
  if world > 1:
    dist.destroy_process_group()


def ttn_network(dims=None):
  """<T|T> of a binary tree tensor network: root -> 2 -> 4 -> 8 leaves (15 nodes) + a cap on the root's top leg = 16 ket
  nodes, 16 conj bra nodes, closed (scalar).  The heavy work sits at the 8 leaf groups (bond b3 between a leaf and its
  parent), the joins above are small: the contraction tree fans out 8 ways.  -> (labels, sizes, shapes)"""
  d = {"top": 4, "cap": 4, "b1": 16, "b2": 64, "b3": 1024, "p": 16}
  d.update(dims or {})
  lk, lb, sizes = [], [], {}
  bond = lambda tag, i: "%s%d" % (tag, i)
  for i in range(15):
    for tag, L in (("k", lk), ("b", lb)):
      if i == 0:
        L.append([tag + "top", bond(tag, 1), bond(tag, 2)])
      elif i < 7:
        L.append([bond(tag, i), bond(tag, 2 * i + 1), bond(tag, 2 * i + 2)])
      else:
        L.append([bond(tag, i), "p%da" % i, "p%db" % i])
  for tag, L in (("k", lk), ("b", lb)):
    L.append([tag + "top", "cap"])
    sizes[tag + "top"] = d["top"]
    for i in range(1, 15):
      sizes[bond(tag, i)] = d["b1" if i < 3 else ("b2" if i < 7 else "b3")]
  for i in range(7, 15):
    sizes["p%da" % i] = sizes["p%db" % i] = d["p"]
  sizes["cap"] = d["cap"]
  labels = lk + lb
  return labels, sizes, [tuple(sizes[l] for l in labs) for labs in labels], d


def strong_scaling_record(be, rank, world, dist, steps, b3=None):
  """ONE 32-node closed network (ttn_network, fp64) contracted on `world` GPUs by parallel.ShardedNetwork against the same
  network on one GPU (CompiledNetwork graph replay, measured on every rank at the same time; rank 0's time is reported).
  Device-timed, max over ranks.  Parity: against the numpy oracle on rank 0's host (fp64, 1e-10)."""
  import torch
  from tensornetwork_b200 import drivers, parallel
  labels, sizes, shapes, dims = ttn_network({"b3": b3} if b3 else None)
  path = drivers.greedy_path(labels, [], sizes)
  n_ket = len(labels) // 2
  kets = []
  for i in range(n_ket):
    t = be.randn(shapes[i], np.float64, seed=700 + i)
    t *= 1.0 / np.sqrt(float(np.prod(shapes[i][1:])))
    kets.append(t)
  dev = kets + list(kets)                      # bra = conj(ket); real data
  single = drivers.CompiledNetwork(be, shapes, np.float64, labels, [], path=path, conj_aliases={n_ket + i: i for i in range(n_ket)})
  single.load(dev)

  def timed(fn):
    for _ in range(3):
      fn()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
      out = fn()
    e1.record()
    torch.cuda.synchronize()
    dist.barrier()
    return e0.elapsed_time(e1) / steps, out
  ms1, out1 = timed(single)
  # Schedule: tree of joins, receives posted right before they are needed, join steps eager.  Measured at 4 GPUs against the
  # other ShardedNetwork knobs (graph-replayed join steps 3.840 ms, receives posted up front 3.905 ms, all small joins
  # gathered on one rank 3.892 ms — all within 2 %): 3.839 ms (profiles/r2_BENCH_default_n4_v1.json).  One schedule only in
  # the driver's run: the gathered plan DEADLOCKS at 8 GPUs (rank 0 sends a small tensor to rank 1 before it receives the
  # large one from it, and with an eagerly initialised NCCL group a rank's point-to-point operations are serialised on one
  # stream) and has been removed from ShardedNetwork.
  variants = {"tree joins, late receives, eager joins": dict(join_graphs=False)}
  var_ms, best = {}, None
  for name, kw in variants.items():
    shv = parallel.ShardedNetwork(be, shapes, np.float64, labels, path, rank, world, **kw)
    shv.load(dev)
    msv, outv = timed(shv.run)
    tv = torch.tensor([msv], device=be.device, dtype=torch.float64)
    dist.all_reduce(tv, op=dist.ReduceOp.MAX)
    var_ms[name] = float(tv[0])
    if best is None or var_ms[name] < best[0]:
      best = (var_ms[name], name, shv, outv)
  msn, best_name, sh, (outn, root_rank) = best
  tt = torch.tensor([ms1, msn], device=be.device, dtype=torch.float64)
  dist.all_reduce(tt, op=dist.ReduceOp.MAX)
  ms1_max, msn_max = float(tt[0]), float(tt[1])
  res = torch.zeros(2, device=be.device, dtype=torch.float64)
  if rank == root_rank:
    res[0] = outn.t.reshape(-1)[0]
  if rank == 0:
    res[1] = out1.t.reshape(-1)[0]
  dist.all_reduce(res, op=dist.ReduceOp.SUM)
  moved = torch.tensor([float(sh.p2p_bytes)], device=be.device, dtype=torch.float64)
  dist.all_reduce(moved, op=dist.ReduceOp.SUM)
  if rank != 0:
    return None
  from oracle import np_network as nn          # checker only (untimed)
  host = [k.to_host() for k in kets]
  ref = float(nn.contract_path(host + [np.conj(h) for h in host], labels, path, []))
  flops = sh.step_flops
  heavy = [f for f in flops if f >= 1e9]
  return {
      "network": "<T|T> of a 16-node binary tree tensor network (32 tensors, closed): bonds top=%d b1=%d b2=%d b3=%d, leaf legs %dx%d; "
                 "greedy path, %d pairwise steps, %d of them >= 1 GFLOP (%.1f-%.1f GFLOP each)"
                 % (dims["top"], dims["b1"], dims["b2"], dims["b3"], dims["p"], dims["p"], len(path), len(heavy), min(heavy) / 1e9, max(heavy) / 1e9),
      "dtype": "f64", "total_gflop": sum(flops) / 1e9,
      "ms_1gpu": ms1_max, "ms_sharded": msn_max, "n_gpus": world, "speedup": ms1_max / msn_max,
      "bound_total_over_critical": sh.info["total"] / sh.info["critical"],
      "bound_lpt_balance": sh.info["total"] / max(sh.info["per_rank"]),
      "per_rank_gflop": [x / 1e9 for x in sh.info["per_rank"]],
      "p2p_transfers": len(sh.transfers), "p2p_bytes_total": float(moved[0]) / 2.0,
      "executor": "per rank: local subtrees as CUDA-graph replays (CompiledNetwork); subtree results sent once, point to point (NCCL isend "
                  "/ irecv); no collective on the data path",
      "schedule": best_name, "ms_sharded_by_schedule": var_ms,
      "result_sharded": float(res[0]), "result_1gpu": float(res[1]), "result_oracle_fp64": ref,
      "parity_rel_err": abs(float(res[0]) - ref) / abs(ref), "parity_ok": bool(abs(float(res[0]) - ref) <= 1e-10 * abs(ref)),
      "tflops_1gpu": sum(flops) / ms1_max / 1e9, "tflops_sharded": sum(flops) / msn_max / 1e9,
  }


def _run_sub(extra, timeout=240):
  """Runs `bench.py <extra> --sub` in a fresh process and returns its JSON line (dict) or {"error": ...}."""
  cmd = [sys.executable, os.path.abspath(__file__)] + extra + ["--sub"]
  try:
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, check=False)
  except subprocess.TimeoutExpired:
    return {"error": "timeout after %d s" % timeout}
  for ln in reversed(r.stdout.strip().splitlines()):
    if ln.startswith("{"):
      try:
        return json.loads(ln)
      except ValueError:
        continue
  return {"error": "rc=%d %s" % (r.returncode, (r.stderr or "").strip().splitlines()[-1:] or "")}


def _compact(d, keys):
  return {k: d[k] for k in keys if k in d}


TOLERANCE = {"bf16": "bf16 operands and bf16 intermediates, fp32 accumulate: 3e-2 on the scalar of a 127-step network (tests/test_gpu_drivers.py)",
             "f32": "float32 storage, TF32 tensor-core products (10-bit mantissa operands, fp32 accumulate): 2e-2 on the scalar; "
                    "TNB200_MATH_STRICT=1 keeps fp32 FMA (1e-4)",
             "f64": "float64 DMMA: 1e-10"}


def collect_subrecords(args):
  """`by_dtype`: the same cfg2 step in float32 (TF32 tensor cores) and float64 (DMMA), each with its own roofline and a
  SAME-dtype cpu_baseline from the unmodified reference; `configs`: the other BASELINE.json configurations (flagship,
  cfg3 split, cfg4 block-sparse, cfg5 DMRG site update), each with time, roofline fraction, parity flag and a same-dtype
  reference baseline.  Every sub-record is measured by a fresh `bench.py ... --sub` process after this one has freed its
  device memory; none of it is inside this line's timed region."""
  out = {"by_dtype": {}, "configs": {}}
  for dt in ("f32", "f64"):
    if dt == args.dtype:
      continue
    d = _run_sub(["--dtype", dt, "--networks", str(args.networks), "--steps", "5", "--warmup", "3", "--cpu-baseline-steps", "1"])
    if "error" in d:
      out["by_dtype"][dt] = d
      continue
    rec = _compact(d, ["value", "unit", "ms_per_step", "step_tflops", "launches_per_step", "result_check", "cpu_baseline"])
    rec["e2e"] = _compact(d.get("e2e", {}), ["value", "unit", "ms_per_step", "h2d_bytes_per_step"])
    rec["roofline"] = _compact(d.get("roofline", {}), ["bound", "achieved", "peak", "unit", "frac", "kernel", "kernel_share_of_step_time",
                                                         "peak_source", "peak_note"])
    rec["tolerance"] = TOLERANCE[dt]
    if rec.get("cpu_baseline", {}).get("value"):
      rec["speedup_vs_reference_same_dtype"] = {"resident": rec["value"] / rec["cpu_baseline"]["value"],
                                                "e2e": rec["e2e"].get("value", 0.0) / rec["cpu_baseline"]["value"]}
    out["by_dtype"][dt] = rec
  for name, extra in (("flagship_bf16", ["--config", "flagship", "--dtype", "bf16", "--steps", "20"]),
                      ("flagship_f64", ["--config", "flagship", "--dtype", "f64", "--steps", "20"]),
                      ("flagship_batched64_bf16", ["--config", "flagship64", "--dtype", "bf16", "--steps", "10"]),
                      ("cfg3_split_svd_4096_f64", ["--config", "cfg3", "--dtype", "f64", "--steps", "2"]),
                      ("cfg4_blocksparse_f64", ["--config", "cfg4", "--dtype", "f64", "--steps", "20"]),
                      ("cfg5_dmrg_site_D1024_f64", ["--config", "cfg5", "--dtype", "f64", "--steps", "4"])):
    d = _run_sub(extra)
    if "error" in d:
      out["configs"][name] = d
      continue
    rec = _compact(d, ["metric", "value", "unit", "ms_per_step", "dtype", "parity", "parity_ok", "rel_err_vs_fp64", "gpu_launches",
                       "cpu_baseline", "sizes", "site_update_seconds", "energies"])
    rec["workload"] = d.get("config", {}).get("workload")
    rec["roofline"] = _compact(d.get("roofline") or {}, ["bound", "achieved", "peak", "unit", "frac", "kernel", "peak_source"])
    out["configs"][name] = rec
  return out


def kernel_profile(be, dev, labels, path, work, nbatch, nb, esize, reps=3):
  """Per-kernel device time of one step, measured LIVE with CUDA events on the launching stream: the plan is
  replayed eagerly `reps` times with an event pair around every pairwise contraction; the library reports which
  kernel family served it.  Returns {family: {"launches", "us", "flops", "bytes"}} averaged per step
  (bytes = algorithmic operand + result bytes of the contraction, each counted once)."""
  import torch
  from tensornetwork_b200 import drivers
  steps, _ = drivers.plan_path([t.shape for t in dev], labels, path, [], nbatch)
  stats = {}
  for rep in range(reps + 1):
    vals = list(dev)
    evs = []
    wi = 0
    for st in steps:
      if st[0] in ("tensordot", "batched"):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if st[0] == "tensordot":
          vals.append(be.tensordot(vals[st[1]], vals[st[2]], (st[3], st[4])))
        else:
          vals.append(be._contract(vals[st[1]], vals[st[2]], list(st[3]), list(st[4]), list(st[5]), list(st[6])))
        e1.record()
        evs.append((be.lib.tnb200_last_kernel().decode(), work[wi], e0, e1))
        wi += 1
      else:
        vals.append(be.transpose(vals[st[1]], st[2]))
    torch.cuda.synchronize()
    del vals
    if rep == 0:
      continue                                  # warm-up pass (allocator, descriptors)
    for name, (m, k, n), e0, e1 in evs:
      d = stats.setdefault(name, {"launches": 0, "us": 0.0, "flops": 0.0, "bytes": 0.0})
      d["launches"] += 1.0 / reps
      d["us"] += e0.elapsed_time(e1) * 1e3 / reps
      d["flops"] += nb * 2.0 * m * k * n / reps
      d["bytes"] += nb * float(m * k + k * n + m * n) * esize / reps
  return stats


def cpu_baseline(args):
  """The reference itself (oracle/_ref, numpy backend; oracle port only if that install is absent) on the host cores,
  bounded sample, at the dtype of this run (float32 for bf16: numpy has no bfloat16)."""
  m = reference_measure(NP_DTYPE[args.dtype], 1, args.cpu_baseline_steps, 1)
  return {"value": m["value"], "unit": "contractions/s", "cores": m["cores"], "kind": m["kind"],
          "dtype": np.dtype(NP_DTYPE[args.dtype]).name, "sample": m["sample"]}


# ------------------------------------------------------------------ the other SURVEY 8(d) configurations
def _peaks():
  try:
    return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
  except Exception:  # pylint: disable=broad-except
    return {}


_PEAK_CACHE = {}


def measured_peak(kind):
  """Dense GEMM peak of this board for `kind` in {"f64", "tf32"}, measured live the way MEASURED_PEAKS.json measures bf16:
  torch.matmul (cuBLAS) on 8192^3 (f64: 4096^3), best of 5, CUDA events.  TFLOP/s."""
  import torch
  if kind in _PEAK_CACHE:
    return _PEAK_CACHE[kind]
  n = 4096 if kind == "f64" else 8192
  dt = torch.float64 if kind == "f64" else torch.float32
  old = torch.backends.cuda.matmul.allow_tf32
  torch.backends.cuda.matmul.allow_tf32 = (kind == "tf32")
  try:
    a = torch.randn(n, n, device="cuda", dtype=dt)
    b = torch.randn(n, n, device="cuda", dtype=dt)
    c = torch.empty(n, n, device="cuda", dtype=dt)
    best = None
    for it in range(7):
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      torch.matmul(a, b, out=c)
      e1.record()
      torch.cuda.synchronize()
      if it >= 2:
        t = e0.elapsed_time(e1)
        best = t if best is None else min(best, t)
    del a, b, c
  finally:
    torch.backends.cuda.matmul.allow_tf32 = old
  _PEAK_CACHE[kind] = 2.0 * n**3 / (best * 1e-3) / 1e12
  return _PEAK_CACHE[kind]


def _ref_tn():
  from baseline import refenv  # pylint: disable=import-outside-toplevel
  return refenv.try_load()


def _time_gpu(fn, steps, warmup, flush=None):
  """CUDA-event time of `steps` calls of fn() (ms per call); `flush()` (untimed part excluded by its own
  events) is called between iterations when the inputs fit in L2."""
  import torch
  for _ in range(max(warmup, 3)):
    fn()
  torch.cuda.synchronize()
  tot = 0.0
  for _ in range(steps):
    if flush is not None:
      flush()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    tot += e0.elapsed_time(e1)
  return tot / steps


def _best_threads_time(fn, reps, warm=1, candidates=(8, 16, 32, 64, None)):
  """median time of fn under the BLAS thread limit that makes it fastest -> (seconds, threads)"""
  cores = os.cpu_count() or 1
  try:
    from threadpoolctl import threadpool_limits  # pylint: disable=import-outside-toplevel
  except ImportError:
    return _time_cpu(fn, reps, warm), cores
  best = None
  for c in candidates:
    n = cores if c is None else min(c, cores)
    with threadpool_limits(limits=n):
      t = _time_cpu(fn, reps, warm)
    if best is None or t < best[0]:
      best = (t, n)
  return best


def _time_cpu(fn, reps, warm=1):
  for _ in range(warm):
    fn()
  ts = []
  for _ in range(reps):
    t0 = time.perf_counter()
    fn()
    ts.append(time.perf_counter() - t0)
  return float(np.median(ts))


def run_config(args):
  """One JSON line per configuration, same keys as the headline line where they apply (N = 1)."""
  import torch
  torch.cuda.set_device(0)
  _ref_tn()                       # the reference first: tensornetwork_b200 then subclasses its AbstractBackend and registers in its factory
  import tensornetwork_b200 as tb
  from tensornetwork_b200 import drivers
  from oracle import np_backend as nb, np_network as nn          # cpu_baseline leg only
  be = tb.get_backend()
  lib = be.lib
  peaks = _peaks()
  hbm_peak = peaks.get("hbm_gbs", 6650.0)
  np_dt = {"bf16": np.float32, "f32": np.float32, "f64": np.float64}[args.dtype]
  be_dt = {"bf16": "bfloat16", "f32": np.float32, "f64": np.float64}[args.dtype]
  esize = {"bf16": 2, "f32": 4, "f64": 8}[args.dtype]
  tensor_peak = peaks.get("bf16_tflops", 1590.0) if args.dtype == "bf16" else measured_peak("tf32" if args.dtype == "f32" else "f64")
  fp64_peak = measured_peak("f64")
  peak_source = "MEASURED_PEAKS.json (bf16 burst)" if args.dtype == "bf16" else "cuBLAS %s GEMM measured in this run" % ("tf32" if args.dtype == "f32" else "fp64")
  cand = (16,) if args.sub else (8, 16, 32, 64, None)     # sub-records: one BLAS thread setting (16 was the fastest on this pool's hosts)
  tn_ref = _ref_tn()
  ref_kind = "reference" if tn_ref is not None else "port"
  ref_be = tn_ref.backends.backend_factory.get_backend("numpy") if tn_ref is not None else None
  flushbuf = torch.empty(256 << 20, dtype=torch.uint8, device=be.device)
  flush = lambda: flushbuf.zero_()                       # 256 MB write > 126 MB L2
  sampler = ClockSampler(0)
  sampler.start()
  cfg = args.config
  steps = args.steps
  line = {"n_gpus": 1, "steps": steps, "warmup": max(args.warmup, 3), "higher_is_better": True, "scaling": "weak",
          "vs_baseline": None, "dtype": args.dtype, "data": "synthetic"}
  l0 = lib.tnb200_launch_count()

  if cfg == "cfg1":
    # SURVEY 8(d) cfg 1: ncon of two 10x10 fp64 matrices — pure call-overhead number
    rng = np.random.default_rng(1)
    a, b = rng.standard_normal((10, 10)), rng.standard_normal((10, 10))
    A, B = be.convert_to_tensor(a), be.convert_to_tensor(b)
    net = [(-1, 1), (1, -2)]
    ms = _time_gpu(lambda: drivers.ncon([A, B], net, backend=be), steps, args.warmup)
    cpu = _time_cpu(lambda: nn.ncon([a, b], net), 200, 20)
    ok = np.allclose(drivers.ncon([A, B], net, backend=be).to_host(), nn.ncon([a, b], net), rtol=1e-12)
    line.update({"metric": "pairwise contractions/s", "value": 1e3 / ms, "unit": "contractions/s", "ms_per_step": ms, "dtype": "f64",
                 "config": {"workload": "cfg1: ncon([a,b],[(-1,1),(1,-2)]) on 10x10 fp64 (latency-bound, host plan + one launch)"},
                 "roofline": None, "parity_ok": bool(ok),
                 "cpu_baseline": {"value": 1.0 / cpu, "unit": "contractions/s", "cores": 1, "kind": "port",
                                  "sample": "200 calls of the numpy ncon restatement, median"}})
  elif cfg == "flagship":
    # SURVEY 8(d) flagship: A,B (512,2,512), tensordot over the shared bond -> (512,2,2,512); M=1024,K=512,N=1024
    rng = np.random.default_rng(2)
    a = (rng.standard_normal((512, 2, 512)) / np.sqrt(512)).astype(np_dt)
    b = (rng.standard_normal((512, 2, 512)) / np.sqrt(512)).astype(np_dt)
    A, B = be.astype(be.convert_to_tensor(a), be_dt), be.astype(be.convert_to_tensor(b), be_dt)
    ms = _time_gpu(lambda: be.tensordot(A, B, [[2], [0]]), steps, args.warmup, flush)
    kern = lib.tnb200_last_kernel().decode()
    flops, byts = 2.0 * 1024 * 512 * 1024, (1024 * 512 * 2 + 1024 * 1024) * esize
    out = be.tensordot(A, B, [[2], [0]]).to_host().astype(np.float64)
    ref = np.tensordot(A.to_host().astype(np.float64), B.to_host().astype(np.float64), [[2], [0]])
    err = float(np.linalg.norm(out - ref) / np.linalg.norm(ref))
    ref_td = (lambda: ref_be.tensordot(a, b, [[2], [0]])) if ref_be is not None else (lambda: nb.tensordot(a, b, [[2], [0]]))
    cpu, cpu_thr = _best_threads_time(ref_td, 10, 3, candidates=cand)
    tf, gbs = flops / ms / 1e9, byts / ms / 1e6
    t_t, t_h = flops / (tensor_peak * 1e12), byts / (hbm_peak * 1e9)
    tol = {"bf16": 4e-3, "f32": 2e-3, "f64": 1e-10}[args.dtype]
    line.update({"metric": "pairwise contractions/s", "value": 1e3 / ms, "unit": "contractions/s", "ms_per_step": ms,
                 "config": {"workload": "flagship: tensordot(A(512,2,512), B(512,2,512), [[2],[0]]), one unbatched call, L2 flushed "
                                        "(256 MB write) between timed calls"},
                 "roofline": {"bound": "tensor" if t_t >= t_h else "hbm", "achieved": tf if t_t >= t_h else gbs,
                              "peak": tensor_peak if t_t >= t_h else hbm_peak, "unit": "TFLOP/s" if t_t >= t_h else "GB/s",
                              "frac": (tf / tensor_peak) if t_t >= t_h else (gbs / hbm_peak), "traffic": None, "kernel": kern,
                              "kernel_tflops": tf, "kernel_gbs": gbs, "peak_source": peak_source,
                              "note": "single 1.07 GFLOP call on 148 SMs: 32 output tiles of 128x256 -> at most 32 SMs busy; "
                                      "the batched form of the same shape is the flagship64 record"},
                 "rel_err_vs_fp64": err, "parity_ok": bool(err <= tol),
                 "cpu_baseline": {"value": 1.0 / cpu, "unit": "contractions/s", "cores": cpu_thr, "kind": ref_kind,
                                  "dtype": np.dtype(np_dt).name,
                                  "sample": "NumPyBackend.tensordot of the %s in %s, median of 10, BLAS threads = %d of %d"
                                            % ("unmodified reference" if ref_be is not None else "oracle restatement",
                                               np.dtype(np_dt).name, cpu_thr, os.cpu_count()),
                                  "gflops": flops / cpu / 1e9}})
  elif cfg == "flagship64":
    # the flagship shape batched over 64 independent two-site pairs: matmul (64,1024,512) x (64,512,1024)
    nbt = 64
    A = be.astype(be.randn((nbt, 1024, 512), np.float32, seed=2) * (1.0 / np.sqrt(512)), be_dt)
    B = be.astype(be.randn((nbt, 512, 1024), np.float32, seed=3) * (1.0 / np.sqrt(512)), be_dt)
    def ten():                      # 10 launches per timed region: the ~10 us of host launch path per call is not kernel time
      for _ in range(10):
        be.matmul(A, B)
    ms = _time_gpu(ten, steps, args.warmup) / 10.0
    kern = lib.tnb200_last_kernel().decode()
    flops, byts = nbt * 2.0 * 1024 * 512 * 1024, nbt * (1024 * 512 * 2 + 1024 * 1024) * esize
    out = be.matmul(A, B)
    o0 = out.to_host()[:2].astype(np.float64)
    ref = np.matmul(A.to_host()[:2].astype(np.float64), B.to_host()[:2].astype(np.float64))
    err = float(np.linalg.norm(o0 - ref) / np.linalg.norm(ref))
    tol = {"bf16": 4e-3, "f32": 2e-3, "f64": 1e-10}[args.dtype]
    a2, b2 = A.to_host()[:2].astype(np_dt), B.to_host()[:2].astype(np_dt)
    ref_mm = (lambda: ref_be.matmul(a2, b2)) if ref_be is not None else (lambda: np.matmul(a2, b2))
    cpu, cpu_thr = _best_threads_time(ref_mm, 5, 2, candidates=cand)
    tf, gbs = flops / ms / 1e9, byts / ms / 1e6
    t_t, t_h = flops / (tensor_peak * 1e12), byts / (hbm_peak * 1e9)
    line.update({"metric": "pairwise contractions/s", "value": nbt * 1e3 / ms, "unit": "contractions/s", "ms_per_step": ms,
                 "config": {"workload": "flagship x64: matmul of 64 independent (1024 x 512)(512 x 1024) two-site products in one launch; "
                                        "operands 201 MB (bf16) > L2"},
                 "roofline": {"bound": "tensor" if t_t >= t_h else "hbm", "achieved": tf if t_t >= t_h else gbs,
                              "peak": tensor_peak if t_t >= t_h else hbm_peak, "unit": "TFLOP/s" if t_t >= t_h else "GB/s",
                              "frac": (tf / tensor_peak) if t_t >= t_h else (gbs / hbm_peak), "traffic": None, "kernel": kern,
                              "kernel_tflops": tf, "kernel_gbs": gbs, "peak_source": peak_source},
                 "rel_err_vs_fp64": err, "parity_ok": bool(err <= tol),
                 "cpu_baseline": {"value": 2.0 / cpu, "unit": "contractions/s", "cores": cpu_thr, "kind": ref_kind,
                                  "dtype": np.dtype(np_dt).name,
                                  "sample": "NumPyBackend.matmul on 2 of the 64 pairs in %s, median of 5, BLAS threads = %d" % (np.dtype(np_dt).name, cpu_thr)}})
  elif cfg == "cfg3":
    # SURVEY 8(d) cfg 3: split_node_full_svd of (64,64,64,64) with max_singular_values=256
    rng = np.random.default_rng(4)
    m = (rng.standard_normal((64, 64, 64, 64)) / 64.0).astype(np.float64 if args.dtype == "f64" else np.float32)
    M = be.convert_to_tensor(m)
    steps = min(steps, 3)
    res = {}
    def f():
      res["o"] = drivers.split_full_svd(M, [0, 1], [2, 3], max_singular_values=256, backend=be)
    ms = _time_gpu(f, steps, 1)
    u, s, vh, trun = res["o"]
    launches_per_split = (lib.tnb200_launch_count() - l0) / (steps + 3)
    ref_out = {}
    if tn_ref is not None:
      def fcpu():
        node = tn_ref.Node(m, backend="numpy")
        un, sn_, vn, tr = tn_ref.split_node_full_svd(node, [node[0], node[1]], [node[2], node[3]], max_singular_values=256)
        ref_out["o"] = (un.tensor, np.diag(sn_.tensor), vn.tensor, tr)
    else:
      def fcpu():
        ref_out["o"] = nb.svd(m, 2, 256, None, False)
    cpu, cpu_thr = _best_threads_time(fcpu, 1, 0, candidates=(16,) if args.sub else (16, 64, None))
    ru, rs, rvh, rtr = ref_out["o"]
    sv = np.diag(s.to_host())
    err_s = float(np.abs(sv - rs).max() / rs[0])
    err_rest = float(np.abs(trun.to_host() - np.asarray(rtr)).max() / rs[0])
    shapes_ok = u.shape == ru.shape and vh.shape == rvh.shape and tuple(trun.shape) == tuple(np.asarray(rtr).shape)
    rec = (u.to_host().reshape(4096, -1) * sv[None, :]) @ vh.to_host().reshape(sv.shape[0], 4096)
    rref = (ru.reshape(4096, -1) * rs[None, :]) @ rvh.reshape(rs.shape[0], 4096)
    err_rec = float(np.linalg.norm(rec - rref) / np.linalg.norm(rref))
    flops = 21.0 * 4096.0**3
    tol = 1e-10 if args.dtype == "f64" else 2e-5
    line.update({"metric": "split_node_full_svd/s", "value": 1e3 / ms, "unit": "splits/s", "ms_per_step": ms, "steps": steps,
                 "dtype": "f64" if args.dtype == "f64" else "f32 storage, f64 Jacobi iteration",
                 "config": {"workload": "cfg3: split_node_full_svd of a (64,64,64,64) tensor (4096x4096), max_singular_values=256"},
                 "roofline": {"bound": "fp64 pipe", "achieved": flops / ms / 1e9, "peak": fp64_peak, "unit": "TFLOP/s",
                              "frac": flops / ms / 1e9 / fp64_peak, "traffic": None, "kernel": lib.tnb200_last_kernel().decode(),
                              "peak_source": "cuBLAS fp64 GEMM measured in this run", "launches_per_split": launches_per_split,
                              "note": "flops by the 21 n^3 Golub-Reinsch convention (SURVEY 8d) irrespective of the Jacobi sweeps spent"},
                 "parity": {"singular_values_max_err_rel_s0": err_s, "s_rest_max_err_rel_s0": err_rest, "truncated_reconstruction_rel_err": err_rec,
                            "shapes_equal": bool(shapes_ok), "kept": int(sv.shape[0])},
                 "parity_ok": bool(shapes_ok and err_s <= tol and err_rest <= tol and err_rec <= 100 * tol),
                 "cpu_baseline": {"value": 1.0 / cpu, "unit": "splits/s", "cores": cpu_thr, "kind": ref_kind,
                                  "dtype": m.dtype.name,
                                  "sample": "1 call of %s (LAPACK gesdd) at BLAS threads = %d" %
                                            ("the reference's tn.split_node_full_svd on backend numpy" if tn_ref is not None else "the numpy restatement", cpu_thr),
                                  "seconds": cpu}})
  elif cfg == "cfg4":
    # SURVEY 8(d) cfg 4: U(1) block-sparse tensordot(A, conj(A), ([2,3],[2,3])), 4 legs of dim 32 (and the x2 scale-up)
    from tensornetwork_b200 import blocksparse as bs
    from oracle import np_blocksparse as nbs
    # library warm-up on an unrelated small structure: module load, memory pools (a cold process pays ~8 ms once)
    wl = [bs.Index(np.array([0, 1, -1, 0, 1]), f) for f in (False, False, True, True)]
    wA = bs.BlockSparseTensor.randn(wl, dtype=np.float64, seed=1, backend=be)
    bs.tensordot(wA, wA.conj(), ([2, 3], [2, 3]))
    torch.cuda.synchronize()
    outs = []
    for dim in (32, 64):
      rng = np.random.RandomState(5)
      charges = [rng.randint(-8, 9, dim).astype(np.int64) for _ in range(4)]
      flows = [False, False, True, True]
      legs = [bs.Index(c, f) for c, f in zip(charges, flows)]
      A = bs.BlockSparseTensor.randn(legs, dtype=np.float64, seed=5, backend=be)
      Ac = A.conj()
      torch.cuda.synchronize()
      t0 = time.perf_counter()
      C = bs.tensordot(A, Ac, ([2, 3], [2, 3]))       # first call of this charge structure: tables on the host, maps on the device
      torch.cuda.synchronize()
      first = time.perf_counter() - t0
      ms = _time_gpu(lambda: bs.tensordot(A, Ac, ([2, 3], [2, 3])), steps, args.warmup, flush)
      kern = lib.tnb200_last_kernel().decode()
      a_host = A.data.to_host()
      cref, _, _ = nbs.tensordot_trailing(a_host, charges, flows, np.conj(a_host), charges, [not f for f in flows], 2)   # checker
      if tn_ref is not None:
        rA = tn_ref.BlockSparseTensor.random([tn_ref.Index(tn_ref.U1Charge(c.astype(np.int16)), f) for c, f in zip(charges, flows)],
                                             dtype=np.float64)
        rAc = rA.conj()
        cpu = _time_cpu(lambda: tn_ref.block_sparse.tensordot(rA, rAc, ([2, 3], [2, 3])), 3, 1)
      else:
        cpu = _time_cpu(lambda: nbs.tensordot_trailing(a_host, charges, flows, np.conj(a_host), charges, [not f for f in flows], 2), 3, 0)
      err = float(np.linalg.norm(C.data.to_host() - cref) / np.linalg.norm(cref))
      nnz = a_host.shape[0]
      byts = (2 * nnz + cref.shape[0]) * 8 * 2.0          # payload + the int64 gather/scatter maps
      outs.append({"leg_dim": dim, "nnz_a": int(nnz), "nnz_c": int(cref.shape[0]), "mflop": C.last_flops / 1e6, "kernel": kern,
                   "gpu_ms_steady": ms, "gpu_ms_first_call_of_structure": first * 1e3, "gbs": byts / ms / 1e6,
                   "gflops": C.last_flops / ms / 1e6, "cpu_ms": cpu * 1e3, "rel_err": err})
    o = outs[0]
    line.update({"metric": "pairwise contractions/s", "value": 1e3 / o["gpu_ms_steady"], "unit": "contractions/s",
                 "ms_per_step": o["gpu_ms_steady"], "dtype": "f64",
                 "config": {"workload": "cfg4: U(1) block-sparse tensordot(A, conj(A), ([2,3],[2,3])), 4 legs x dim 32, charges in [-8,8] "
                                        "(one grouped gather-GEMM-scatter launch over all sectors; element maps built on the device, plan cached)"},
                 "roofline": {"bound": "hbm", "achieved": o["gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": o["gbs"] / hbm_peak,
                              "traffic": None, "kernel": o["kernel"],
                              "note": "3.8 MFLOP / 1 MB problem: launch-latency bound; the dim-64 scale-up (DMMA sector tiles) is in `sizes`"},
                 "sizes": outs, "parity_ok": bool(all(x["rel_err"] <= 1e-12 for x in outs)),
                 "cpu_baseline": {"value": 1e3 / o["cpu_ms"], "unit": "contractions/s", "cores": os.cpu_count(), "kind": ref_kind,
                                  "dtype": "float64",
                                  "sample": "median of 3 calls of %s (block maps rebuilt per call, as the reference does without its opt-in cache)"
                                            % ("the reference's block_sparse.tensordot" if tn_ref is not None else "the numpy restatement")}})
  elif cfg == "cfg5":
    # SURVEY 8(d) cfg 5: two-site DMRG of the XXZ chain at saturated bond dimension D: time per site update.
    # Both arms run the REFERENCE's own driver (FiniteDMRG._optimize_2s_local, matrixproductstates/dmrg.py:251-343) on identical
    # inputs for the same number of updates; only the backend differs ("cuda_b200" vs "numpy").
    D = int(os.environ.get("TNB200_CFG5_D", "1024"))
    lo = int(np.ceil(np.log2(D)))
    nup = max(2, min(steps, 4))                           # timed updates on the GPU arm (it does one more, untimed, first; the
                                                          # second one also records the CUDA graphs of the jitted ncon calls)
    N = 2 * lo + 2 + nup + 1
    rng = np.random.default_rng(6)
    dims = [min(D, 2**min(i, N - i)) for i in range(N + 1)]
    tensors = []
    for i in range(N):
      dl, dr = dims[i], dims[i + 1]
      if i < lo:
        q, _ = np.linalg.qr(rng.standard_normal((dl * 2, dr)))
        tensors.append(np.ascontiguousarray(q.reshape(dl, 2, dr)))
      elif i > lo:
        q, _ = np.linalg.qr(rng.standard_normal((2 * dr, dl)))
        tensors.append(np.ascontiguousarray(q.T.reshape(dl, 2, dr)))
      else:
        c = rng.standard_normal((dl, 2, dr))
        tensors.append(c / np.linalg.norm(c))
    if tn_ref is None:
      raise RuntimeError("cfg5 needs the reference driver (oracle/_ref, installed by build())")

    def arm(backend, count, sync):
      mps = tn_ref.FiniteMPS([t.copy() for t in tensors], canonicalize=False, backend=backend)
      mps.center_position = lo
      mpo = tn_ref.FiniteXXZ(np.ones(N - 1), np.ones(N - 1), np.zeros(N), dtype=np.float64, backend=backend)
      dm = tn_ref.FiniteDMRG(mps, mpo)
      dm.compute_left_envs()
      dm.compute_right_envs()
      times, energies = [], []
      for _ in range(count):
        sync()
        t0 = time.perf_counter()
        e = dm._optimize_2s_local(max_bond_dim=D, sweep_dir="right", num_krylov_vecs=10, tol=1e-5, delta=1e-6, ndiag=10)
        sync()
        times.append(time.perf_counter() - t0)
        energies.append(float(np.real(np.asarray(e))))
      return times, energies
    tg, eg = arm("cuda_b200", nup + 1, torch.cuda.synchronize)
    tc, ec, cpu_thr = [float("nan")], [], os.cpu_count()
    if not args.no_cpu_baseline:
      try:
        from threadpoolctl import threadpool_limits  # pylint: disable=import-outside-toplevel
        cpu_thr = min(16, os.cpu_count())
        with threadpool_limits(limits=cpu_thr):
          tc, ec = arm("numpy", 2, lambda: None)
      except ImportError:
        tc, ec = arm("numpy", 2, lambda: None)
    ms = float(np.median(tg[1:])) * 1e3
    e_err = max(abs(a_ - b_) / abs(b_) for a_, b_ in zip(eg, ec)) if ec else None
    flops_mv = 2.0 * (D * 5) * D * (2 * 2 * D) * 2 + 2.0 * (D * 2 * D * 2) * (5 * 2) * (5 * 2) * 2   # 4 tensordots per matvec
    line.update({"metric": "two-site DMRG site updates/s", "value": 1e3 / ms, "unit": "site-updates/s", "ms_per_step": ms,
                 "steps": len(tg) - 1, "dtype": "f64",
                 "config": {"workload": "cfg5: XXZ (Jz=Jxy=1, Bz=0) two-site DMRG, fp64, D=%d saturated, N=%d sites (interior site cost is "
                                        "independent of N), <=10 Krylov vectors, SVD truncation to D; the reference's FiniteDMRG driver on "
                                        "backend cuda_b200, wall clock incl. its Python" % (D, N)},
                 "roofline": {"bound": "fp64 pipe", "achieved": None, "peak": fp64_peak, "unit": "TFLOP/s", "frac": None, "traffic": None,
                              "kernel": "gemm_dmma_f64 + svd_pair_persistent", "approx_gflop_per_matvec": flops_mv / 1e9,
                              "peak_source": "cuBLAS fp64 GEMM measured in this run"},
                 "site_update_seconds": tg, "energies": {"cuda_b200": eg, "numpy": ec},
                 "parity": {"updates_compared": len(ec), "energy_max_rel_err": e_err},
                 "parity_ok": bool(e_err is not None and e_err <= 1e-8),
                 "cpu_baseline": {"value": 1.0 / float(np.median(tc)), "unit": "site-updates/s", "cores": cpu_thr, "kind": "reference",
                                  "dtype": "float64",
                                  "sample": "%d saturated site update(s) of the same reference driver on backend numpy, BLAS threads = %d" % (len(tc), cpu_thr),
                                  "site_update_seconds": tc}})
  elif cfg == "tree32":
    # SURVEY 8(d) 32-node network: <T|T> of a random 16-node tree tensor network, chi=128, d=2
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from multigpu_check import tree_network
    tensors, labels, sizes = tree_network(chi=128)
    host = [t.astype(np_dt) for t in tensors]
    dev = [be.astype(be.convert_to_tensor(t), be_dt) for t in host]
    path = drivers.greedy_path(labels, [], sizes)
    flops = float(sum(2.0 * m * k * n for m, k, n in nn.network_flops(labels, path, sizes)))
    net = drivers.CompiledNetwork(be, [t.shape for t in dev], be_dt, labels, [], path=path)
    net.load(dev)
    ms = _time_gpu(lambda: net(), steps, args.warmup, flush)
    out = float(net().to_host().astype(np.float64))
    ref = float(nn.contract_path([h.astype(np.float64) for h in host], labels, path, []))
    cpu, cpu_thr = _best_threads_time(lambda: nn.contract_path(host, labels, path, []), 3, 1)
    npair = len(path)
    line.update({"metric": "pairwise contractions/s", "value": npair * 1e3 / ms, "unit": "contractions/s", "ms_per_step": ms,
                 "config": {"workload": "tree32: <T|T> of a random 16-node tree tensor network (32 tensors, chi=128, d=2), greedy path, "
                                        "CUDA-graph replay, L2 flushed between replays"},
                 "roofline": {"bound": "tensor", "achieved": flops / ms / 1e9, "peak": tensor_peak, "unit": "TFLOP/s",
                              "frac": flops / ms / 1e9 / tensor_peak, "traffic": None, "kernel": "mixed (whole network)",
                              "algorithmic_gflop_per_step": flops / 1e9},
                 "result": out, "reference_result_fp64": ref, "rel_err": abs(out - ref) / abs(ref),
                 "cpu_baseline": {"value": npair / cpu, "unit": "contractions/s", "cores": cpu_thr, "kind": "port",
                                  "sample": "3 full networks in numpy %s, median, best BLAS thread count" % np.dtype(np_dt).name}})
  line["gpu_launches"] = int(lib.tnb200_launch_count() - l0)
  sampler.stop_flag = True
  sampler.join(timeout=2)
  line["clocks"] = sampler.summary()
  emit(line)


if __name__ == "__main__":
  main()
