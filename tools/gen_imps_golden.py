"""Generate tests/golden/imps.npz by running the REAL reference's InfiniteMPS on its numpy backend.

Needs the reference installed in oracle/_ref (oracle/build_ref.py):  python tools/gen_imps_golden.py
Per (D, dtype) of tests/imps_cases.GOLDEN_CASES: the Schmidt values, lam_norm, the final dtype and the operator
applications of each eigs call (ARPACK) of InfiniteMPS.canonicalize.  The unit cell is redrawn from the seed
(np.random's legacy stream is stable); a checksum of it is stored to catch a drift.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import ref_shim  # noqa: E402
from oracle.gen_golden import _save  # noqa: E402  pylint: disable=protected-access
import imps_cases  # noqa: E402


def main():
  tn = ref_shim.load()
  assert tn.__version__ == "0.4.6"
  meta, arrays = [], {}
  for i, (D, dt) in enumerate(imps_cases.GOLDEN_CASES):
    tensors = imps_cases.make_tensors(tn, D, dt)
    r = imps_cases.canonicalize(tn, "numpy", tensors)
    arrays["c%d_schmidt" % i] = r["schmidt"]
    meta.append(dict(D=D, dtype=dt, seed=imps_cases.SEED, checksum=imps_cases.checksum(tensors), final_dtype=str(r["dtype"]),
                     lam_norm=[r["lam_norm"].real, r["lam_norm"].imag], check=r["check"], matvecs=r["matvecs"]))
    print("imps", D, dt, r["matvecs"], r["check"])
  _save("imps", meta, arrays)


if __name__ == "__main__":
  main()
