"""CPU-only: the InfiniteMPS surface of the cuda_b200 adapter — eigh, eigs (arnoldi.py), inv, index_update and the n-d
comparisons — over a host double of the new C-ABI entry points (HostLib below, a tests/fake_lib.FakeLib subclass).
The reference's own InfiniteMPS.canonicalize / transfer_matrix_eigs / check_canonical run unmodified on
backend="cuda_b200" in a subprocess (imps_host_runner.py) and are compared with its numpy backend and with
tests/golden/imps.npz.  The kernels themselves are checked by tests/test_gpu_infinite_mps.py."""
import ctypes
import os
import subprocess
import sys
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, HERE):
  if p not in sys.path:
    sys.path.insert(0, p)
import fake_lib  # noqa: E402

_NP = dict(fake_lib._NP)  # pylint: disable=protected-access
_NP[8] = np.bool_


def _view(arg):
  """fake_lib._view with the TNB200_BOOL code (8)."""
  d = fake_lib._desc(arg)  # pylint: disable=protected-access
  dt = np.dtype(_NP[d.dtype])
  nd = d.ndim
  shape = tuple(d.shape[i] for i in range(nd))
  strides = tuple(d.stride[i] * dt.itemsize for i in range(nd))
  if any(s == 0 for s in shape):
    return np.zeros(shape, dtype=dt)
  span = sum((s - 1) * abs(st) for s, st in zip(shape, strides)) + dt.itemsize
  buf = (ctypes.c_char * span).from_address(d.data)
  return np.ndarray(shape, dtype=dt, buffer=buf, strides=strides)


def _at(ptr, n, dt):
  return fake_lib.FakeLib._vec(ptr, n, dt)  # pylint: disable=protected-access


class HostLib(fake_lib.FakeLib):
  """tnb200_eigh / inv / compare / masked_fill / krylov_orth on host memory (numpy), plus bool-aware copy."""

  def tnb200_copy(self, src, dst, conj, stream):
    if 8 in (fake_lib._desc(src).dtype, fake_lib._desc(dst).dtype):  # pylint: disable=protected-access
      _view(dst)[...] = _view(src)
      self._launches += 1
      return 0
    return super().tnb200_copy(src, dst, conj, stream)

  def tnb200_eigh(self, a, w, v, info, stream):
    A = _view(a)
    ww, vv = np.linalg.eigh(A)
    _view(w)[...] = ww
    _view(v)[...] = vv
    if info:
      _at(info, 4, np.int32)[...] = (1, 1, 0, 0)
    self._launches += 1
    return 0

  def tnb200_inv(self, a, out, info, stream):
    try:
      _view(out)[...] = np.linalg.inv(_view(a))
      _at(info, 1, np.int32)[0] = 0
    except np.linalg.LinAlgError:
      _at(info, 1, np.int32)[0] = 1
    self._launches += 1
    return 0

  def tnb200_compare(self, op, a, b, c, stream):
    _view(c)[...] = [np.less, np.less_equal, np.greater, np.greater_equal][op](_view(a), _view(b))
    self._launches += 1
    return 0

  def tnb200_masked_fill(self, src, mask, out, re, im, vptr, vdt, stream):
    S = _view(src)
    if vptr:
      val = fake_lib._scalar_at(vptr, vdt)[()] if vdt != 8 else _at(vptr, 1, np.bool_)[0]  # pylint: disable=protected-access
    else:
      val = complex(re, im) if np.iscomplexobj(S) else re
    _view(out)[...] = np.where(_view(mask), np.asarray(val).astype(S.dtype) if np.iscomplexobj(S) else np.real(val), S)
    self._launches += 1
    return 0

  def tnb200_krylov_orth(self, basis, w, k, h, stream):
    """CGS2 of w against basis rows 0..k-1, as csrc/krylov.cu (arithmetic in double)."""
    V = _view(basis)
    x = np.array(_view(w), dtype=np.complex128 if np.iscomplexobj(V) else np.float64)
    Vk = V[:k].astype(x.dtype)
    h1 = Vk.conj() @ x
    x = x - Vk.T @ h1
    h2 = Vk.conj() @ x
    x = x - Vk.T @ h2
    nrm = np.linalg.norm(x)
    V[k] = x / nrm if nrm > 0 else 0.0
    hh = _at(h, k + 1, V.dtype)
    hh[:k] = h1 + h2
    hh[k] = nrm
    self._launches += 4
    return 0


def _run(*extra):
  r = subprocess.run([sys.executable, os.path.join(HERE, "imps_host_runner.py")] + list(extra),
                     capture_output=True, text=True, cwd=ROOT, timeout=900)
  assert r.returncode == 0 and "IMPS HOST OK" in r.stdout, r.stdout[-3000:] + r.stderr[-4000:]
  return r.stdout


@pytest.mark.refhost
def test_reference_infinite_mps_canonicalize_on_cuda_b200_adapter(tn):  # pylint: disable=redefined-outer-name,unused-argument
  out = _run("imps")
  assert "imps D=10 float64 ok" in out and "imps D=10 complex128 ok" in out and "imps D=64 float64 ok" in out


def test_eigs_arguments_masks_index_update_and_inv_errors():
  _run("api")
