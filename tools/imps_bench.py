"""InfiniteMPS benchmark: the reference's own InfiniteMPS.canonicalize (N = 4 sites, d = 2) on backend cuda_b200 against
its numpy backend, plus eigh and inv against numpy.  Prints ONE JSON line (and writes it to --out when given).

  python tools/imps_bench.py [--out FILE] [--quick]

* canonicalize: D in {64, 256, 512, 1024}, float64 and complex128, unit cell drawn as tests/imps_cases.py does; cuda_b200
  timed after one warm-up run of the same D and dtype (graph capture, workspace pools), host clock around work that
  ends in a device synchronise; the numpy arm for D <= 256.  Each entry also records the operator applications of every
  eigs call (ARPACK's for the numpy arm) and the Schmidt-value difference of the two arms.
* eigh / inv: n in {256, 1024, 2048}, float64 and complex128, random Hermitian / general input; device time after a
  warm-up, numpy (LAPACK) time on the host of the same machine.
The GPU name and power limit are read with nvidia-smi in the same run.  Needs build() (oracle/_ref holds the reference).
"""
import argparse
import json
import os
import subprocess
import sys
import time
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from baseline import refenv  # noqa: E402
tn = refenv.load()
import tensornetwork_b200  # noqa: E402,F401  pylint: disable=unused-import
from tensornetwork_b200 import backend as tbb  # noqa: E402
import imps_cases  # noqa: E402


def gpu_info():
  r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True, check=True)
  name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
  return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, sync):
  sync()
  t0 = time.perf_counter()
  out = fn()
  sync()
  return time.perf_counter() - t0, out


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--out")
  ap.add_argument("--quick", action="store_true", help="D in {64, 256} and n = 256 only")
  a = ap.parse_args()
  be = tbb.get_instance()
  sync = be.synchronize
  res = {"bench": "imps", **gpu_info(), "N": imps_cases.N_SITES, "d": imps_cases.PHYS, "canonicalize": [], "eigh": [], "inv": []}
  Ds = [64, 256] if a.quick else [64, 256, 512, 1024]
  for dt in ("float64", "complex128"):
    for D in Ds:
      tensors = imps_cases.make_tensors(tn, D, dt)
      imps_cases.canonicalize(tn, "cuda_b200", tensors)                                  # warm-up
      t, got = timed(lambda: imps_cases.canonicalize(tn, "cuda_b200", tensors), sync)    # pylint: disable=cell-var-from-loop
      e = {"D": D, "dtype": dt, "cuda_b200_s": round(t, 4), "eigs_matvecs": got["matvecs"], "check_canonical": got["check"]}
      if D <= 256:
        t0 = time.perf_counter()
        ref = imps_cases.canonicalize(tn, "numpy", tensors)
        e["numpy_s"] = round(time.perf_counter() - t0, 4)
        e["numpy_eigs_matvecs"] = ref["matvecs"]
        e["speedup"] = round(e["numpy_s"] / t, 2)
        e["schmidt_max_abs_diff"] = float(np.max(np.abs(got["schmidt"] - ref["schmidt"])))
      res["canonicalize"].append(e)
      print(json.dumps(e), file=sys.stderr)
  rng = np.random.default_rng(0)
  for dt in (np.float64, np.complex128):
    for n in ([256] if a.quick else [256, 1024, 2048]):
      x = rng.standard_normal((n, n))
      if dt is np.complex128:
        x = x + 1j * rng.standard_normal((n, n))
      h = (x + np.conj(x.T)) / 2
      hd, xd = be.convert_to_tensor(h), be.convert_to_tensor(x)
      info = be.torch.zeros(4, dtype=be.torch.int32, device=be.device)
      be._eigh(hd, info)   # pylint: disable=protected-access
      t, (w, _) = timed(lambda: be._eigh(hd, info), sync)   # pylint: disable=protected-access,cell-var-from-loop
      t0 = time.perf_counter()
      wn = np.linalg.eigvalsh(h)
      tn_ = time.perf_counter() - t0
      inf = info.cpu().numpy()
      res["eigh"].append({"n": n, "dtype": np.dtype(dt).name, "cuda_b200_s": round(t, 5), "numpy_s": round(tn_, 5),
                          "sweeps": int(inf[0]), "converged": int(inf[1]),
                          "max_abs_err_rel": float(np.max(np.abs(np.asarray(w) - wn)) / np.max(np.abs(wn)))})
      be.inv(xd)
      t, xi = timed(lambda: be.inv(xd), sync)   # pylint: disable=cell-var-from-loop
      t0 = time.perf_counter()
      xn = np.linalg.inv(x)
      tn_ = time.perf_counter() - t0
      res["inv"].append({"n": n, "dtype": np.dtype(dt).name, "cuda_b200_s": round(t, 5), "numpy_s": round(tn_, 5),
                         "rel_diff": float(np.linalg.norm(np.asarray(xi) - xn) / np.linalg.norm(xn))})
      print(json.dumps(res["eigh"][-1]), json.dumps(res["inv"][-1]), file=sys.stderr)
  line = json.dumps(res)
  print(line)
  if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
      f.write(line + "\n")


if __name__ == "__main__":
  main()
