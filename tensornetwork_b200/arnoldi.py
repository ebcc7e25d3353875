"""Restarted Arnoldi eigensolver on device tensors — NumPyBackend.eigs (backends/numpy/numpy_backend.py:216-291, which
calls scipy.sparse.linalg.eigs, i.e. ARPACK) with the same arguments, checks and output types.

Split like lanczos.py: the host runs the control flow and the small dense problem (an m x m matrix, m =
num_krylov_vecs, with numpy / scipy); the Krylov vectors never leave the device.

* Basis: one contiguous (m + 1, n) device tensor V.  An Arnoldi step is the matvec A(v_j, *args) and one
  tnb200_krylov_orth call (CGS2 against V[:j+1], four launches), which writes v_{j+1} into V and column j of the
  Hessenberg matrix H into a device buffer: there is no host scalar inside a cycle.
* Restart: thick restart (Krylov-Schur, Stewart 2001).  At the end of a cycle H is copied to the host (the one D2H
  of a restart), its Schur form is ordered so that the `keep` best Ritz values lead — `numeig` plus a buffer of half
  the remaining basis, the role ARPACK's extra shifts play — and V[:keep] <- Z[:, :keep]^T V[:m] goes through
  tnb200_tensordot.  A real operator keeps a real Schur form, so it runs in real arithmetic throughout.
* Convergence: ARPACK's test |r^T y| <= tol * max(eps^(2/3), |theta|) for each of the `numeig` wanted Ritz pairs
  (theta, V y), r the residual row of the Krylov-Schur relation A V_m = V_m H_m + v_m r^T.  `maxiter` counts restarts
  (default n * 10, as scipy).  Breakdown (an invariant subspace) is read off H at the restart.
* Output, as scipy's: eigenvalues as a 1-d device tensor and unit-norm eigenvectors shaped like `initial_state`,
  always complex (c128 for f64 / c128 operators, c64 for f32 / c64).
"""
import numpy as np
import scipy.linalg
import scipy.sparse.linalg
from .tensor import B200Tensor
from . import _lib as L
from . import tensor as T

# sort keys: ascending key = most wanted first
_KEYS = {"LM": lambda t: -np.abs(t), "SM": np.abs, "LR": lambda t: -np.real(t), "SR": np.real}
_COMPLEX_OF = {L.F64: L.C128, L.C128: L.C128, L.F32: L.C64, L.C64: L.C64}


def eigs(be, A, args=None, initial_state=None, shape=None, dtype=None, num_krylov_vecs=50, numeig=6, tol=1e-8,
         which='LR', maxiter=None):
  if args is None:
    args = []
  if which in ('SI', 'LI'):
    raise ValueError(f'which = {which} is currently not supported.')
  if which not in _KEYS:
    raise ValueError("which must be one of 'LM', 'SM', 'LR', 'SR'; got {!r}".format(which))
  if numeig + 1 >= num_krylov_vecs:
    raise ValueError('`num_krylov_vecs` > `numeig + 1` required!')
  if initial_state is None:
    if (shape is None) or (dtype is None):
      raise ValueError("if no `initial_state` is passed, then `shape` and"
                       "`dtype` have to be provided")
    initial_state = be.randn(shape, dtype)
  if not isinstance(initial_state, B200Tensor):
    raise TypeError("Expected a `B200Tensor`. Got {}".format(type(initial_state)))
  be._no_capture("eigs")   # pylint: disable=protected-access
  shape = initial_state.shape
  code = initial_state.code
  if code in (L.I32, L.I64):
    code = L.F64
  if code not in _COMPLEX_OF:
    raise TypeError("eigs needs a float32/float64/complex operator, got dtype {}".format(initial_state.dtype))
  n = initial_state.size
  m = int(num_krylov_vecs)
  if m > n or numeig >= n - 1:
    raise ValueError("eigs: need numeig < n - 1 and num_krylov_vecs <= n for an operator of size n = {}".format(n))
  if maxiter is None:
    maxiter = n * 10
  cplx = T.is_complex_code(code)
  eps = float(np.finfo(np.float64 if code in (L.F64, L.C128) else np.float32).eps)
  key = _KEYS[which]

  V = be._new((m + 1, n), code)   # pylint: disable=protected-access
  Ht = be.zeros((m, m + 1), dtype=T.code_to_np(code))     # row j = column j of H (written by the device)
  h0 = be._new((m + 1,), code)    # pylint: disable=protected-access

  def orth(w, k, h_ptr):
    w = be.reshape(w, (n,))
    if w.code != code:
      w = be.astype(w, code)
    L.check(be.lib.tnb200_krylov_orth(V.ref(), w.ref(), k, h_ptr, be._stream()))   # pylint: disable=protected-access

  def row(j):
    return B200Tensor(V.t[j], code)

  def ritz_vectors(Y, mm):
    """V[:mm]^T Y (columns of Y = Ritz coefficients) -> list of unit-norm complex vectors shaped like the input."""
    Vm = B200Tensor(V.t[:mm], code)
    if cplx:
      X = be.tensordot(be.convert_to_tensor(np.ascontiguousarray(Y.T.astype(T.code_to_np(code)))), Vm, 1)
    else:
      rdt = T.code_to_np(code)
      X = be.astype(be.tensordot(be.convert_to_tensor(np.ascontiguousarray(Y.T.real.astype(rdt))), Vm, 1), _COMPLEX_OF[code])
      Xi = be.astype(be.tensordot(be.convert_to_tensor(np.ascontiguousarray(Y.T.imag.astype(rdt))), Vm, 1), _COMPLEX_OF[code])
      be.iadd(X, Xi, 1j)
    out = []
    for i in range(Y.shape[1]):
      x = B200Tensor(X.t[i], X.code)
      x /= be.norm(x)
      out.append(be.reshape(x, shape))
    return out

  def result(theta, Y, mm):
    eta = be.convert_to_tensor(np.asarray(theta, dtype=T.code_to_np(_COMPLEX_OF[code])))
    return eta, ritz_vectors(Y, mm)

  orth(be.reshape(initial_state, (n,)), 0, h0.t.data_ptr())
  H = np.zeros((m + 1, m), dtype=np.complex128 if cplx else np.float64)
  p = 0
  restarts = 0
  while True:
    for j in range(p, m):
      w = A(be.reshape(row(j), shape), *args)
      orth(w, j + 1, Ht.t[j].data_ptr())
    H[:, p:] = Ht.to_host()[p:, :].T          # the one device -> host copy of a restart
    restarts += 1
    # breakdown: a zero subdiagonal entry in the new columns means V[:mm] spans an invariant subspace
    sub = np.abs(H[np.arange(p + 1, m + 1), np.arange(p, m)])
    tiny = np.nonzero(sub <= eps * max(np.linalg.norm(H), np.finfo(np.float64).tiny))[0]
    mm = m if tiny.size == 0 else p + int(tiny[0]) + 1
    Hm = H[:mm, :mm]
    r = H[m, :mm] if mm == m else np.zeros(mm, dtype=H.dtype)
    theta, Y = scipy.linalg.eig(Hm)
    order = np.argsort(key(theta), kind="stable")
    want = order[:min(numeig, mm)]
    res = np.abs(r @ Y[:, want])
    conv = res <= tol * np.maximum(eps ** (2.0 / 3.0), np.abs(theta[want]))
    if conv.all() and want.size == numeig:
      return result(theta[want], Y[:, want], mm)
    if restarts >= maxiter or mm < m:
      good = want[conv]
      eta, vecs = result(theta[good], Y[:, good], mm) if good.size else (None, [])
      raise scipy.sparse.linalg.ArpackNoConvergence(
          "ARPACK error -1: No convergence ({} iterations, {}/{} eigenvectors converged)".format(
              restarts, int(good.size), numeig), eta, vecs)
    # thick restart: order the Schur form so the `keep` most wanted Ritz values lead
    keep = (m + numeig) // 2
    kv = np.sort(key(theta))
    thresh = kv[keep - 1] + 1e-12 * max(1.0, abs(kv[keep - 1]))
    if cplx:
      Tm, Z, sdim = scipy.linalg.schur(Hm, output="complex", sort=lambda z: key(np.array([z]))[0] <= thresh)
    else:
      Tm, Z, sdim = scipy.linalg.schur(Hm, output="real", sort=lambda x, y: key(np.array([complex(x, y)]))[0] <= thresh)
    p = int(min(max(sdim, numeig), m - 1))
    Zp = Z[:, :p]
    newv = be.tensordot(be.convert_to_tensor(np.ascontiguousarray(Zp.T.astype(T.code_to_np(code)))),
                        B200Tensor(V.t[:m], code), 1)
    L.check(be.lib.tnb200_copy(row(m).ref(), row(p).ref(), 0, be._stream()))   # pylint: disable=protected-access
    L.check(be.lib.tnb200_copy(newv.ref(), B200Tensor(V.t[:p], code).ref(), 0, be._stream()))   # pylint: disable=protected-access
    Hn = np.zeros_like(H)
    Hn[:p, :p] = Tm[:p, :p]
    Hn[p, :p] = r @ Zp
    H = Hn
