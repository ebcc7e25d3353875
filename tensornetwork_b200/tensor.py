"""B200Tensor — the backend's opaque tensor type.

A thin handle around a `torch.Tensor` that lives in B200 HBM.  torch is used ONLY as the
device-memory container (allocation, views, streams); every arithmetic operator below is
routed to a kernel of libtnb200.so.  The handle exposes the attributes the reference's
callers read from backend tensors: `.shape` (tuple), `.dtype` (a numpy dtype, because the
callers pass dtypes back to `backend.zeros/randn` as numpy dtypes — SURVEY 8b), `.ndim`,
`.item()`, in-place `/=` (dmrg.py:225,298,329; base_mps.py:172,197,222) and `__array__`
(device -> host copy) so `np.testing.assert_allclose(node.tensor, ...)` works unchanged.
"""
import ctypes
import operator
import numpy as np
from . import _lib as L


class BFloat16:
  """Stand-in dtype object for bfloat16 (numpy has no bf16)."""
  name = "bfloat16"
  itemsize = 2
  kind = "f"

  def __repr__(self):
    return "bfloat16"

  def __eq__(self, other):
    return isinstance(other, BFloat16) or other == "bfloat16"

  def __hash__(self):
    return hash("bfloat16")


bfloat16 = BFloat16()

_NP2CODE = {np.dtype(np.float64): L.F64, np.dtype(np.float32): L.F32, np.dtype(np.float16): L.F16,
            np.dtype(np.complex64): L.C64, np.dtype(np.complex128): L.C128,
            np.dtype(np.int32): L.I32, np.dtype(np.int64): L.I64, np.dtype(np.bool_): L.BOOL}
_CODE2NP = {v: k for k, v in _NP2CODE.items()}
_CODE2NP[L.BF16] = bfloat16
_REAL_OF = {L.C64: L.F32, L.C128: L.F64}
_torch = None
_CODE2TORCH = None
_TORCH2CODE = None


def _init_torch():
  global _torch, _CODE2TORCH, _TORCH2CODE
  if _torch is None:
    import torch  # pylint: disable=import-outside-toplevel
    _torch = torch
    _CODE2TORCH = {L.F64: torch.float64, L.F32: torch.float32, L.F16: torch.float16,
                   L.BF16: torch.bfloat16, L.C64: torch.complex64, L.C128: torch.complex128,
                   L.I32: torch.int32, L.I64: torch.int64, L.BOOL: torch.bool}
    _TORCH2CODE = {v: k for k, v in _CODE2TORCH.items()}
  return _torch


def dtype_code(dtype):
  """numpy dtype / python type / torch dtype / 'bfloat16' -> tnb200_dtype_t code."""
  if dtype is None:
    return L.F64
  if isinstance(dtype, BFloat16) or (isinstance(dtype, str) and dtype in ("bfloat16", "bf16")):
    return L.BF16
  if _TORCH2CODE is not None and dtype in _TORCH2CODE:
    return _TORCH2CODE[dtype]
  try:
    return _NP2CODE[np.dtype(dtype)]
  except (KeyError, TypeError):
    _init_torch()
    if dtype in _TORCH2CODE:
      return _TORCH2CODE[dtype]
    raise TypeError("cuda_b200 backend does not support dtype {!r}".format(dtype))


def code_to_np(code):
  return _CODE2NP[code]


def code_to_torch(code):
  _init_torch()
  return _CODE2TORCH[code]


def real_code(code):
  return _REAL_OF.get(code, code)


def is_complex_code(code):
  return code in (L.C64, L.C128)


_SYNC_GUARD = [None]      # set by the backend: raises jit.CaptureUnsupported while a CUDA graph is being recorded


def _host_sync_guard(what):
  g = _SYNC_GUARD[0]
  if g is not None:
    g(what)


class B200Tensor:
  """Handle of a (possibly strided) tensor in device memory."""
  __slots__ = ("t", "code", "_desc", "__weakref__")
  __array_priority__ = 1000  # numpy scalars defer to our reflected operators

  def __init__(self, t, code=None):
    self.t = t
    self.code = _TORCH2CODE[t.dtype] if code is None else code
    self._desc = None

  # ------------------------------------------------------------------ metadata
  @property
  def shape(self):
    return tuple(self.t.shape)

  @property
  def ndim(self):
    return self.t.dim()

  @property
  def dtype(self):
    return _CODE2NP[self.code]

  @property
  def size(self):
    return self.t.numel()

  def __len__(self):
    if self.t.dim() == 0:
      raise TypeError("len() of unsized object")
    return self.t.shape[0]

  def desc(self):
    """ctypes tnb200_tensor_t for this view (cached: handles are immutable)."""
    d = self._desc
    if d is None:
      t = self.t
      nd = t.dim()
      if nd > L.MAX_NDIM:
        raise ValueError("cuda_b200 supports at most {} axes".format(L.MAX_NDIM))
      d = L.TensorDesc()
      d.data = t.data_ptr()
      d.dtype = self.code
      d.ndim = nd
      if nd:
        d.shape[:nd] = t.shape
        d.stride[:nd] = t.stride()
      self._desc = d
    return d

  def ref(self):
    return ctypes.byref(self.desc())

  # ------------------------------------------------------------------ host access
  def to_host(self):
    """Device -> host copy as a numpy array (bf16 is widened to float32)."""
    _host_sync_guard("to_host")
    t = self.t
    if self.code == L.BF16:
      t = t.to(_torch.float32)
    return t.cpu().numpy()

  def __array__(self, dtype=None, copy=None):
    a = self.to_host()
    return a if dtype is None else a.astype(dtype)

  def item(self):
    _host_sync_guard("item")
    return self.t.item()

  def __float__(self):
    return float(self.item())

  def __complex__(self):
    return complex(self.item())

  def __int__(self):
    return int(self.item())

  def __bool__(self):
    if self.t.numel() != 1:
      raise ValueError("The truth value of a tensor with more than one element is ambiguous")
    return bool(self.item())

  def __repr__(self):
    return "B200Tensor(shape={}, dtype={}, device={})".format(self.shape, self.dtype, self.t.device)

  # comparisons: a 0-d tensor against a python number gives a python bool (Lanczos `abs(norm) < delta`); anything with
  # an axis gives a device bool tensor (InfiniteMPS.canonicalize's `eigvals <= cutoff` mask, infinite_mps.py:239)
  def _compare(self, o, op, pyop):
    if self.ndim == 0 and not (getattr(o, "ndim", 0) > 0):
      return pyop(self.item(), _scalar(o))
    return _be().compare(op, self, o)

  def __lt__(self, o):
    return self._compare(o, L.LT, operator.lt)

  def __le__(self, o):
    return self._compare(o, L.LE, operator.le)

  def __gt__(self, o):
    return self._compare(o, L.GT, operator.gt)

  def __ge__(self, o):
    return self._compare(o, L.GE, operator.ge)

  def __abs__(self):
    return _be().abs(self)

  # ------------------------------------------------------------------ views
  def __getitem__(self, idx):
    return B200Tensor(self.t[idx], self.code)

  @property
  def T(self):
    return _be().transpose(self)

  def conj(self):
    return _be().conj(self)

  def reshape(self, *shape):
    if len(shape) == 1 and not isinstance(shape[0], (int, np.integer)):
      shape = shape[0]
    return _be().reshape(self, shape)

  def transpose(self, *perm):
    if len(perm) == 1 and not isinstance(perm[0], (int, np.integer)):
      perm = perm[0]
    return _be().transpose(self, perm if perm else None)

  def astype(self, dtype):
    return _be().astype(self, dtype)

  def copy(self):
    return _be().copy(self)

  # ------------------------------------------------------------------ arithmetic
  def __add__(self, o):
    return _be().addition(self, o)

  def __radd__(self, o):
    return _be().addition(o, self)

  def __sub__(self, o):
    return _be().subtraction(self, o)

  def __rsub__(self, o):
    return _be().subtraction(o, self)

  def __mul__(self, o):
    return _be().multiply(self, o)

  def __rmul__(self, o):
    return _be().multiply(o, self)

  def __truediv__(self, o):
    return _be().divide(self, o)

  def __rtruediv__(self, o):
    return _be().divide(o, self)

  def __neg__(self):
    return _be().negative(self)

  def __pow__(self, o):
    return _be().power(self, o)

  def __matmul__(self, o):
    return _be().matmul(self, o) if self.ndim > 1 and o.ndim > 1 else _be().tensordot(self, o, 1)

  def __itruediv__(self, o):
    _be().idivide(self, o)
    return self

  def __imul__(self, o):
    _be().imultiply(self, o)
    return self

  def __iadd__(self, o):
    _be().iadd(self, o, 1.0)
    return self

  def __isub__(self, o):
    _be().iadd(self, o, -1.0)
    return self


def _scalar(o):
  return o.item() if isinstance(o, B200Tensor) else o


def _be():
  from . import backend  # pylint: disable=import-outside-toplevel
  return backend.get_instance()
