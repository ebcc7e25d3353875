"""`cuda_b200` — a TensorNetwork backend whose every compute method is a hand-written sm_100a
kernel behind the C ABI of libtnb200.so (include/tnb200.h).

Drop-in boundary (SURVEY.md 8b): this class implements the operator surface of
`tensornetwork.backends.abstract_backend.AbstractBackend` (abstract_backend.py:22) with the
same method names, argument meaning and error behaviour as the reference numpy backend
(backends/numpy/numpy_backend.py).  When the `tensornetwork` package is importable it
subclasses the real `AbstractBackend` and registers itself in
`backend_factory._BACKENDS["cuda_b200"]` (backend_factory.py:22-28), so `tn.Node`, `tn.ncon`,
`contractors.greedy`, `split_node*` and `FiniteDMRG` run unchanged with
`backend="cuda_b200"`.  Without it, the mirror base class in `_abstract.py` is used and the
drivers in `tensornetwork_b200.drivers` provide ncon / greedy / split on the same backend.

There is no CPU path: constructing the backend without a CUDA device raises.
"""
import ctypes
import os
import numpy as np

from . import _lib as L
from . import tensor as T
from .tensor import B200Tensor

try:  # the real plug-in base class, when the host library is installed
  from tensornetwork.backends import abstract_backend as _ab  # type: ignore
  _Base = _ab.AbstractBackend
  HAVE_TENSORNETWORK = True
except Exception:  # pylint: disable=broad-except
  from ._abstract import AbstractBackend as _Base
  HAVE_TENSORNETWORK = False

_INSTANCE = None
_CONFIG = {"device": None}  # tests may point this at "cpu" together with _lib.set_lib(...)

_I32P = ctypes.POINTER(ctypes.c_int32)
_EMPTY_I32 = (ctypes.c_int32 * 1)()


def _i32arr(seq):
  n = len(seq)
  if n == 0:
    return _EMPTY_I32
  return (ctypes.c_int32 * n)(*seq)


def get_instance():
  global _INSTANCE
  if _INSTANCE is None:
    _INSTANCE = CudaB200Backend()
  return _INSTANCE


def _prod(xs):
  p = 1
  for x in xs:
    p *= int(x)
  return p


class CudaB200Backend(_Base):
  """See the module docstring.  Tensors are `B200Tensor` handles."""

  def __init__(self, dtype=None):
    global _INSTANCE
    super().__init__()
    self.name = "cuda_b200"
    self.torch = T._init_torch()
    self.lib = L.load()
    dev = _CONFIG["device"]
    if dev is None:
      if not self.torch.cuda.is_available():
        raise RuntimeError("backend 'cuda_b200' needs a CUDA device (B200, sm_100a); "
                           "there is no CPU fallback")
      dev = self.torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
      self.torch.cuda.set_device(dev)
    self.device = self.torch.device(dev)
    self._on_cuda = self.device.type == "cuda"
    self.math_mode = L.MATH_DEFAULT
    self._seed = 0x5EED
    self._jit_cache = {}
    self._capturing = 0             # > 0 while jit.JitFunction records a CUDA graph
    self._cap_stream = None
    T._SYNC_GUARD[0] = self._no_capture
    self.jit_graphs = os.environ.get("TNB200_JIT", "1") != "0"      # jit(): CUDA-graph capture (0 = identity, like numpy's)
    self.jit_stats = {"eager": 0, "captures": 0, "replays": 0, "capture_failures": 0}
    if _INSTANCE is None:
      _INSTANCE = self

  # ------------------------------------------------------------------ plumbing
  def _stream(self):
    if self._on_cuda:
      return self.torch.cuda.current_stream().cuda_stream
    return 0

  def _capture_stream(self):
    if self._cap_stream is None:
      self._cap_stream = self.torch.cuda.Stream()
    return self._cap_stream

  def _no_capture(self, what):
    """Host-synchronising operations cannot be part of a CUDA graph: refuse cleanly (before any CUDA call) so that
    jit.JitFunction falls back to eager execution for this function."""
    if self._capturing:
      from .jit import CaptureUnsupported  # pylint: disable=import-outside-toplevel
      raise CaptureUnsupported(what + " synchronises with the host and cannot be captured in a CUDA graph")

  def _new(self, shape, code):
    return B200Tensor(self.torch.empty(tuple(int(s) for s in shape), dtype=T.code_to_torch(code),
                                       device=self.device), code)

  def _check_type(self, x, what="tensor"):
    if not isinstance(x, B200Tensor):
      raise TypeError("Expected a `B200Tensor` for {}. Got {}".format(what, type(x)))

  def _scalar_tensor(self, value, code):
    out = self._new((), code)
    v = complex(value)
    L.check(self.lib.tnb200_fill(out.ref(), v.real, v.imag, self._stream()))
    return out

  def _as_tensor(self, x, like_code=None):
    """operand of an arithmetic op -> B200Tensor (python / numpy scalars become 0-d tensors)."""
    if isinstance(x, B200Tensor):
      return x
    if isinstance(x, np.ndarray) and x.ndim > 0:
      return self.convert_to_tensor(x)
    if isinstance(x, np.ndarray):
      x = x.item()
    if like_code is None:
      code = T.dtype_code(np.result_type(x))
    elif like_code == L.BF16 or like_code == L.F16:
      code = like_code if not isinstance(x, complex) else L.C64
    else:
      code = T.dtype_code(np.result_type(T.code_to_np(like_code), x))
    return self._scalar_tensor(x, code)

  @staticmethod
  def _promote(c1, c2):
    if c1 == c2:
      return c1
    if L.BF16 in (c1, c2):
      other = c2 if c1 == L.BF16 else c1
      if other in (L.F16, L.I32, L.I64):
        return L.F32
      return other
    return T.dtype_code(np.result_type(T.code_to_np(c1), T.code_to_np(c2)))

  def astype(self, tensor, dtype):
    code = dtype if type(dtype) is int else T.dtype_code(dtype)  # pylint: disable=unidiomatic-typecheck
    if code == tensor.code:
      return tensor
    out = self._new(tensor.shape, code)
    L.check(self.lib.tnb200_copy(tensor.ref(), out.ref(), 0, self._stream()))
    return out

  def copy(self, tensor, conj=False):
    out = self._new(tensor.shape, tensor.code)
    L.check(self.lib.tnb200_copy(tensor.ref(), out.ref(), 1 if conj else 0, self._stream()))
    return out

  def contiguous(self, tensor):
    return tensor if tensor.t.is_contiguous() else self.copy(tensor)

  def to_host(self, tensor):
    return tensor.to_host()

  def synchronize(self):
    if self._on_cuda:
      self.torch.cuda.current_stream().synchronize()

  # ------------------------------------------------------------------ a1: tensordot
  def tensordot(self, a, b, axes, conj_a=False, conj_b=False):
    """numpy_backend.py:35-54.  Output = free axes of a, then free axes of b."""
    self._check_type(a, "a")
    self._check_type(b, "b")
    if isinstance(axes, (int, np.integer)):
      n = int(axes)
      if n < 0 or n > a.ndim or n > b.ndim:
        raise ValueError("shape-mismatch for sum")
      ax_a = list(range(a.ndim - n, a.ndim))
      ax_b = list(range(n))
    else:
      ax_a, ax_b = axes
      ax_a = [int(ax_a)] if isinstance(ax_a, (int, np.integer)) else [int(x) for x in ax_a]
      ax_b = [int(ax_b)] if isinstance(ax_b, (int, np.integer)) else [int(x) for x in ax_b]
      if len(ax_a) != len(ax_b):
        raise ValueError("shape-mismatch for sum")
    return self._contract(a, b, ax_a, ax_b, [], [], conj_a, conj_b)

  def _contract(self, a, b, ax_a, ax_b, bat_a, bat_b, conj_a=False, conj_b=False, out=None):
    if a.code != b.code:
      code = self._promote(a.code, b.code)
      a, b = self.astype(a, code), self.astype(b, code)
    nda, ndb = a.ndim, b.ndim
    na = [x + nda if x < 0 else x for x in ax_a]
    nb = [x + ndb if x < 0 else x for x in ax_b]
    ba = [x + nda if x < 0 else x for x in bat_a]
    bb = [x + ndb if x < 0 else x for x in bat_b]
    sa, sb = a.shape, b.shape
    used_a, used_b = set(na) | set(ba), set(nb) | set(bb)
    out_shape = [sa[i] for i in ba] + [sa[i] for i in range(nda) if i not in used_a] + \
        [sb[i] for i in range(ndb) if i not in used_b]
    if out is None:
      c = self._new(out_shape, a.code)
    else:                                   # preallocated result (static buffers of a compiled network)
      if tuple(out.shape) != tuple(out_shape) or out.code != a.code:
        raise ValueError("out has shape {} / dtype code {}, expected {} / {}".format(out.shape, out.code, out_shape, a.code))
      c = out
    flags = (L.CONJ_A if conj_a else 0) | (L.CONJ_B if conj_b else 0) | self.math_mode
    rc = self.lib.tnb200_tensordot(a.ref(), b.ref(), c.ref(), len(na), _i32arr(na), _i32arr(nb),
                                   len(ba), _i32arr(ba), _i32arr(bb), flags, self._stream())
    L.check(rc)
    return c

  def matmul(self, tensor1, tensor2):
    """numpy_backend.py:609-612: `...ab,...bc->...ac` with equal leading batch axes."""
    self._check_type(tensor1)
    self._check_type(tensor2)
    if tensor1.ndim <= 1 or tensor2.ndim <= 1:
      raise ValueError("inputs to `matmul` have to be a tensors of order > 1,")
    n1, n2 = tensor1.ndim, tensor2.ndim
    if n1 != n2:  # numpy broadcasting of batch dims: prepend 1-axes
      nd = max(n1, n2)
      tensor1 = self.reshape(tensor1, (1,) * (nd - n1) + tensor1.shape)
      tensor2 = self.reshape(tensor2, (1,) * (nd - n2) + tensor2.shape)
    nd = tensor1.ndim
    s1, s2 = tensor1.shape, tensor2.shape
    if s1[:-2] != s2[:-2]:
      bshape = tuple(np.broadcast_shapes(s1[:-2], s2[:-2]))
      tensor1 = B200Tensor(tensor1.t.expand(bshape + s1[-2:]), tensor1.code)
      tensor2 = B200Tensor(tensor2.t.expand(bshape + s2[-2:]), tensor2.code)
    if tensor1.shape[-1] != tensor2.shape[-2]:
      raise ValueError("matmul: Input operand 1 has a mismatch in its core dimension 0")
    batch = list(range(nd - 2))
    return self._contract(tensor1, tensor2, [nd - 1], [nd - 2], batch, batch)

  def outer_product(self, tensor1, tensor2):
    """numpy_backend.py:99-100."""
    return self.tensordot(tensor1, tensor2, 0)

  # ------------------------------------------------------------------ a2: metadata ops
  def reshape(self, tensor, shape):
    """numpy_backend.py:56-57 (shape cast to int32).  A view when the strides allow it,
    otherwise one strided-copy kernel (numpy silently copies in the same cases)."""
    self._check_type(tensor)
    shape = tuple(int(s) for s in np.asarray(shape).astype(np.int32).reshape(-1))
    try:
      return B200Tensor(tensor.t.view(shape), tensor.code)
    except RuntimeError:
      pass
    if _prod(shape) != tensor.size and -1 not in shape:
      raise ValueError("cannot reshape array of size {} into shape {}".format(tensor.size, shape))
    return B200Tensor(self.copy(tensor).t.view(shape), tensor.code)

  def transpose(self, tensor, perm=None):
    """numpy_backend.py:59-62 — always a view."""
    self._check_type(tensor)
    if perm is None:
      perm = tuple(reversed(range(tensor.ndim)))
    perm = tuple(int(p) for p in perm)
    if len(perm) != tensor.ndim:
      raise ValueError("axes don't match array")
    return B200Tensor(tensor.t.permute(perm), tensor.code)

  def slice(self, tensor, start_indices, slice_sizes):
    """numpy_backend.py:64-72."""
    if len(start_indices) != len(slice_sizes):
      raise ValueError("Lengths of start_indices and slice_sizes must be"
                       "identical.")
    obj = tuple(slice(int(s), int(s) + int(n)) for s, n in zip(start_indices, slice_sizes))
    return B200Tensor(tensor.t[obj], tensor.code)

  def shape_concat(self, values, axis):
    return np.concatenate(values, axis)

  def shape_tensor(self, tensor):
    return tensor.shape

  def shape_tuple(self, tensor):
    return tensor.shape

  def sparse_shape(self, tensor):
    return self.shape_tuple(tensor)

  def shape_prod(self, values):
    return np.prod(values)

  def convert_to_tensor(self, tensor):
    """numpy_backend.py:92-97: np.ndarray / scalar -> device (H2D); our own handles pass."""
    if isinstance(tensor, B200Tensor):
      return tensor
    torch = self.torch
    if isinstance(tensor, torch.Tensor):
      return B200Tensor(tensor.to(self.device), T.dtype_code(tensor.dtype))
    if not isinstance(tensor, np.ndarray) and not np.isscalar(tensor):
      raise TypeError("Expected a `np.array`, scalar or `B200Tensor`. Got {}".format(type(tensor)))
    arr = np.asarray(tensor)
    code = T.dtype_code(arr.dtype)  # raises TypeError for unsupported dtypes
    if not arr.flags.c_contiguous or not arr.flags.writeable:
      arr = np.array(arr, order="C")
    self._no_capture("convert_to_tensor(host array)")
    return B200Tensor(torch.from_numpy(arr).to(self.device, non_blocking=False), code)

  def from_host(self, array, dtype=None):
    """H2D with an optional dtype (incl. bfloat16, which numpy lacks)."""
    t = self.convert_to_tensor(np.asarray(array))
    return t if dtype is None else self.astype(t, dtype)

  # ------------------------------------------------------------------ a6: elementwise
  def _unary(self, op, tensor, out_code=None):
    self._check_type(tensor)
    out = self._new(tensor.shape, tensor.code if out_code is None else out_code)
    L.check(self.lib.tnb200_unary(op, tensor.ref(), out.ref(), self._stream()))
    return out

  def sqrt(self, tensor):
    return self._unary(L.SQRT, tensor)

  def conj(self, tensor):
    return self._unary(L.CONJ, tensor)

  def abs(self, tensor):
    return self._unary(L.ABS, tensor, T.real_code(tensor.code))

  def sign(self, tensor):
    return self._unary(L.SIGN, tensor)

  def negative(self, tensor):
    return self._unary(L.NEG, tensor)

  def exp(self, tensor):
    return self._unary(L.EXP, tensor)

  def log(self, tensor):
    return self._unary(L.LOG, tensor)

  def sin(self, tensor):
    return self._unary(L.SIN, tensor)

  def cos(self, tensor):
    return self._unary(L.COS, tensor)

  def real(self, tensor):
    return self._unary(L.REAL, tensor, T.real_code(tensor.code))

  def imag(self, tensor):
    return self._unary(L.IMAG, tensor, T.real_code(tensor.code))

  def _binary(self, op, x, y):
    if isinstance(x, B200Tensor):
      y = self._as_tensor(y, x.code)
    elif isinstance(y, B200Tensor):
      x = self._as_tensor(x, y.code)
    else:
      x = self._as_tensor(x)
      y = self._as_tensor(y, x.code)
    code = self._promote(x.code, y.code)
    if op == L.DIV and code in (L.I32, L.I64):
      code = L.F64
    x, y = self.astype(x, code), self.astype(y, code)
    try:
      shape = tuple(np.broadcast_shapes(x.shape, y.shape))
    except ValueError as e:
      raise ValueError("operands could not be broadcast together with shapes {} {}".format(
          x.shape, y.shape)) from e
    xe = x if x.shape == shape else B200Tensor(x.t.expand(shape), code)
    ye = y if y.shape == shape else B200Tensor(y.t.expand(shape), code)
    out = self._new(shape, code)
    L.check(self.lib.tnb200_binary(op, xe.ref(), ye.ref(), out.ref(), self._stream()))
    return out

  def addition(self, tensor1, tensor2):
    return self._binary(L.ADD, tensor1, tensor2)

  def subtraction(self, tensor1, tensor2):
    return self._binary(L.SUB, tensor1, tensor2)

  def multiply(self, tensor1, tensor2):
    return self._binary(L.MUL, tensor1, tensor2)

  def divide(self, tensor1, tensor2):
    return self._binary(L.DIV, tensor1, tensor2)

  def power(self, a, b):
    return self._binary(L.POW, a, b)

  def idivide(self, x, o):
    """x /= o in place (dmrg.py:225,298).  A device scalar is read on the device: no sync."""
    if isinstance(o, B200Tensor):
      if o.size != 1:
        raise ValueError("in-place division is only supported by a scalar")
      if o.code in (L.I32, L.I64):
        o = self.astype(o, L.F64)
      L.check(self.lib.tnb200_scale_by_device_scalar(x.ref(), o.t.data_ptr(), o.code, -1,
                                                     self._stream()))
    else:
      v = 1.0 / complex(o)
      L.check(self.lib.tnb200_affine_inplace(x.ref(), v.real, v.imag, 0.0, 0.0, self._stream()))

  def imultiply(self, x, o):
    if isinstance(o, B200Tensor):
      if o.size != 1:
        raise ValueError("in-place multiplication is only supported by a scalar")
      L.check(self.lib.tnb200_scale_by_device_scalar(x.ref(), o.t.data_ptr(), o.code, 1,
                                                     self._stream()))
    else:
      v = complex(o)
      L.check(self.lib.tnb200_affine_inplace(x.ref(), v.real, v.imag, 0.0, 0.0, self._stream()))

  def iadd(self, y, x, alpha=1.0):
    """y += alpha * x in place."""
    x = self._as_tensor(x, y.code)
    if x.code != y.code:
      x = self.astype(x, y.code)
    if x.shape != y.shape:
      x = B200Tensor(x.t.expand(y.shape), x.code)
    a = complex(alpha)
    L.check(self.lib.tnb200_axpy(x.ref(), y.ref(), a.real, a.imag, None, 1.0, self._stream()))

  def axpy_dev(self, y, x, alpha_dev, sign=1.0):
    """y += sign * (*alpha_dev) * x with the scalar read on the device."""
    if alpha_dev.code != x.code:
      alpha_dev = self.astype(alpha_dev, x.code)
    L.check(self.lib.tnb200_axpy(x.ref(), y.ref(), 0.0, 0.0, alpha_dev.t.data_ptr(), float(sign),
                                 self._stream()))

  def broadcast_right_multiplication(self, tensor1, tensor2):
    """numpy_backend.py:560-565."""
    if len(tensor2.shape) != 1:
      raise ValueError("only order-1 tensors are allowed for `tensor2`,"
                       " found `tensor2.shape = {}`".format(tensor2.shape))
    return self.multiply(tensor1, tensor2)

  def broadcast_left_multiplication(self, tensor1, tensor2):
    """numpy_backend.py:567-575."""
    if len(tensor1.shape) != 1:
      raise ValueError("only order-1 tensors are allowed for `tensor1`,"
                       " found `tensor1.shape = {}`".format(tensor1.shape))
    t1 = self.reshape(tensor1, tensor1.shape + (1,) * (tensor2.ndim - 1))
    return self.multiply(tensor2, t1)

  # ------------------------------------------------------------------ a6: constructors
  def _filled(self, shape, dtype, re, im=0.0):
    out = self._new(tuple(shape) if not isinstance(shape, (int, np.integer)) else (shape,),
                    T.dtype_code(np.float64 if dtype is None else dtype))
    L.check(self.lib.tnb200_fill(out.ref(), re, im, self._stream()))
    return out

  def ones(self, shape, dtype=None):
    return self._filled(shape, dtype, 1.0)

  def zeros(self, shape, dtype=None):
    return self._filled(shape, dtype, 0.0)

  def eye(self, N, dtype=None, M=None):
    out = self._new((N, N if M is None else M), T.dtype_code(np.float64 if dtype is None else dtype))
    L.check(self.lib.tnb200_eye(out.ref(), 0, self._stream()))
    return out

  def _next_seed(self, seed):
    if seed:
      self._seed = int(seed)
    else:
      self._seed = (self._seed * 6364136223846793005 + 1442695040888963407) % (1 << 64)
    return self._seed

  def randn(self, shape, dtype=None, seed=None):
    """numpy_backend.py:132-144 (own Philox stream: values differ from numpy's RNG)."""
    out = self._new(tuple(shape), T.dtype_code(np.float64 if dtype is None else dtype))
    L.check(self.lib.tnb200_randn(out.ref(), self._next_seed(seed), self._stream()))
    return out

  def random_uniform(self, shape, boundaries=(0.0, 1.0), dtype=None, seed=None):
    """numpy_backend.py:146-160."""
    out = self._new(tuple(shape), T.dtype_code(np.float64 if dtype is None else dtype))
    L.check(self.lib.tnb200_uniform(out.ref(), float(boundaries[0]), float(boundaries[1]),
                                    self._next_seed(seed), self._stream()))
    return out

  # ------------------------------------------------------------------ a6: reductions
  def norm(self, tensor):
    """numpy_backend.py:108-109 -> 0-d device tensor (no host sync)."""
    self._check_type(tensor)
    code = tensor.code
    if code in (L.I32, L.I64):
      tensor, code = self.astype(tensor, L.F64), L.F64
    out = self._new((), T.real_code(code))
    L.check(self.lib.tnb200_norm(tensor.ref(), out.t.data_ptr(), self._stream()))
    return out

  def vdot(self, x, y, conj_x=True):
    """sum(conj(x) * y) -> 0-d device tensor (Lanczos, numpy_backend.py:503-504)."""
    out = self._new((), x.code)
    L.check(self.lib.tnb200_dot(x.ref(), y.ref(), 1 if conj_x else 0, out.t.data_ptr(),
                                self._stream()))
    return out

  def sum(self, tensor, axis=None, keepdims=False):
    """numpy_backend.py:603-607."""
    self._check_type(tensor)
    if axis is None:
      axis = tuple(range(tensor.ndim))
    axis = [int(a) + tensor.ndim if int(a) < 0 else int(a) for a in
            ([axis] if isinstance(axis, (int, np.integer)) else axis)]
    shape = [s for i, s in enumerate(tensor.shape) if i not in axis]
    out = self._new(shape, tensor.code)
    L.check(self.lib.tnb200_sum(tensor.ref(), out.ref(), len(axis), _i32arr(axis), self._stream()))
    if keepdims:
      out = self.reshape(out, [1 if i in axis else s for i, s in enumerate(tensor.shape)])
    return out

  def trace(self, tensor, offset=0, axis1=-2, axis2=-1):
    """numpy_backend.py:684-707."""
    self._check_type(tensor)
    nd = tensor.ndim
    if nd < 2:
      raise ValueError("diag requires an array of at least two dimensions")
    a1, a2 = axis1 % nd, axis2 % nd
    if a1 == a2:
      raise ValueError("axis1 and axis2 cannot be the same")
    shape = [s for i, s in enumerate(tensor.shape) if i not in (a1, a2)]
    out = self._new(shape, tensor.code)
    L.check(self.lib.tnb200_trace(tensor.ref(), out.ref(), int(offset), a1, a2, self._stream()))
    return out

  def diagonal(self, tensor, offset=0, axis1=-2, axis2=-1):
    """numpy_backend.py:643-671 — a strided view (no kernel)."""
    self._check_type(tensor)
    return B200Tensor(self.torch.diagonal(tensor.t, offset=offset, dim1=axis1, dim2=axis2),
                      tensor.code)

  def diagflat(self, tensor, k=0):
    """numpy_backend.py:673-682."""
    self._check_type(tensor)
    n = tensor.size + abs(int(k))
    out = self._new((n, n), tensor.code)
    L.check(self.lib.tnb200_diagflat(tensor.ref(), out.ref(), int(k), self._stream()))
    return out

  def item(self, tensor):
    return tensor.item()

  def eps(self, dtype):
    code = T.dtype_code(dtype)
    if code == L.BF16:
      return 2.0**-7
    return np.finfo(T.code_to_np(code)).eps

  def jit(self, fun, *args, **kwargs):
    """abstract_backend.py:798 (numpy's is the identity, numpy_backend.py:600-601): returns a `jit.JitFunction` that
    captures `fun` in a CUDA graph on the second call per (static args, shapes) key and replays it afterwards — this is
    how `tn.ncon` (ncon_interface.py:654-660) and the DMRG `ncon`s reach graph replay without any change to the caller.
    One JitFunction per (fun, static_argnums): `tn.jit`'s wrapper asks for a new one on every call (decorators.py:64-69)."""
    from . import jit as _jit  # pylint: disable=import-outside-toplevel
    static = kwargs.get("static_argnums", ())
    static = (static,) if isinstance(static, int) else tuple(static or ())
    key = (fun, static)
    try:
      jf = self._jit_cache.get(key)
    except TypeError:
      return fun
    if jf is None:
      jf = self._jit_cache[key] = _jit.JitFunction(self, fun, static)
    return jf

  def serialize_tensor(self, tensor):
    import io  # pylint: disable=import-outside-toplevel
    m = io.BytesIO()
    np.save(m, tensor.to_host(), allow_pickle=False)
    m.seek(0)
    return str(m.read(), encoding="latin-1")

  def deserialize_tensor(self, s):
    import io  # pylint: disable=import-outside-toplevel
    m = io.BytesIO()
    m.write(s.encode("latin-1"))
    m.seek(0)
    return self.convert_to_tensor(np.load(m))

  # ------------------------------------------------------------------ a3: einsum
  def einsum(self, expression, *tensors, optimize=True):
    """numpy_backend.py:102-106, lowered onto trace/sum/tensordot kernels."""
    from . import einsum as _einsum  # pylint: disable=import-outside-toplevel
    return _einsum.einsum(self, expression, *tensors)

  # ------------------------------------------------------------------ a4 / a5: split
  def _as_matrix(self, tensor, pivot_axis):
    left = tensor.shape[:pivot_axis]
    right = tensor.shape[pivot_axis:]
    return self.reshape(tensor, (_prod(left), _prod(right))), left, right

  def svd(self, tensor, pivot_axis=-1, max_singular_values=None, max_truncation_error=None,
          relative=False):
    """backends/numpy/decompositions.py:21-74 -> (u, s, vh, s_rest)."""
    self._check_type(tensor)
    self._no_capture("svd")          # (cooperative persistent launch / data-dependent kept count)
    mat, left, right = self._as_matrix(tensor, pivot_axis)
    if mat.code in (L.I32, L.I64, L.F16, L.BF16):
      raise TypeError("svd needs a float32/float64/complex tensor")
    m, n = mat.shape
    r = min(m, n)
    u = self._new((m, r), mat.code)
    s = self._new((r,), T.real_code(mat.code))
    vh = self._new((r, n), mat.code)
    L.check(self.lib.tnb200_svd(mat.ref(), u.ref(), s.ref(), vh.ref(), None, self._stream()))
    if max_singular_values is None:
      max_singular_values = r
    if max_truncation_error is not None:
      keep_dev = self.torch.empty((), dtype=self.torch.int64, device=self.device)
      L.check(self.lib.tnb200_svd_truncation_count(s.ref(), int(max_singular_values), 1,
                                                   float(max_truncation_error),
                                                   1 if relative else 0, keep_dev.data_ptr(),
                                                   self._stream()))
      keep = int(keep_dev.item())  # the one D2H of the split path (data-dependent shape)
    else:
      keep = min(int(max_singular_values), r)
    s = self.astype(s, mat.code)
    s_rest = s[keep:]
    s = s[:keep]
    u = self.reshape(u[:, :keep], list(left) + [keep])
    vh = self.reshape(vh[:keep, :], [keep] + list(right))
    return u, s, vh, s_rest

  def qr(self, tensor, pivot_axis=-1, non_negative_diagonal=False):
    """decompositions.py:77-98."""
    self._check_type(tensor)
    mat, left, right = self._as_matrix(tensor, pivot_axis)
    if mat.code in (L.I32, L.I64, L.F16, L.BF16):
      raise TypeError("qr needs a float32/float64/complex tensor")
    m, n = mat.shape
    r = min(m, n)
    q = self._new((m, r), mat.code)
    rr = self._new((r, n), mat.code)
    L.check(self.lib.tnb200_qr(mat.ref(), q.ref(), rr.ref(), 1 if non_negative_diagonal else 0,
                               self._stream()))
    return self.reshape(q, list(left) + [r]), self.reshape(rr, [r] + list(right))

  def rq(self, tensor, pivot_axis=-1, non_negative_diagonal=False):
    """decompositions.py:101-124: QR of the conjugate transpose, then conjugate back."""
    self._check_type(tensor)
    mat, left, right = self._as_matrix(tensor, pivot_axis)
    ah = self.copy(self.transpose(mat), conj=True)
    q, r = self.qr(ah, 1, non_negative_diagonal)
    rr = self.copy(self.transpose(r), conj=True)
    qq = self.copy(self.transpose(q), conj=True)
    c = rr.shape[1]
    return self.reshape(rr, list(left) + [c]), self.reshape(qq, [c] + list(right))

  # ------------------------------------------------------------------ a13: Lanczos
  def eigsh_lanczos(self, A, args=None, initial_state=None, shape=None, dtype=None,
                    num_krylov_vecs=20, numeig=1, tol=1e-8, delta=1e-8, ndiag=20,
                    reorthogonalize=False):
    from . import lanczos  # pylint: disable=import-outside-toplevel
    return lanczos.eigsh_lanczos(self, A, args, initial_state, shape, dtype, num_krylov_vecs,
                                 numeig, tol, delta, ndiag, reorthogonalize)

  # ------------------------------------------------------------------ InfiniteMPS: eigh / eigs / inv / masks
  def eigh(self, matrix):
    """numpy_backend.py:165-166 (np.linalg.eigh, UPLO='L'): (w ascending, real dtype; v, eigenvectors as columns)."""
    return self._eigh(matrix)

  def _eigh(self, matrix, info=None):
    """eigh with an optional device int32[4] `info` ([0] sweeps, [1] converged flag); None: no host synchronisation."""
    self._check_type(matrix)
    if matrix.ndim < 2:
      raise np.linalg.LinAlgError("{}-dimensional array given. Array must be at least "
                                  "two-dimensional".format(matrix.ndim))
    if matrix.shape[-1] != matrix.shape[-2]:
      raise np.linalg.LinAlgError("Last 2 dimensions of the array must be square")
    if matrix.code not in (L.F32, L.F64, L.C64, L.C128):
      raise TypeError("eigh needs a float32/float64/complex tensor")
    w = self._new(matrix.shape[:-1], T.real_code(matrix.code))
    v = self._new(matrix.shape, matrix.code)
    L.check(self.lib.tnb200_eigh(matrix.ref(), w.ref(), v.ref(), None if info is None else info.data_ptr(),
                                 self._stream()))
    return w, v

  def inv(self, matrix):
    """numpy_backend.py:554-558 (np.linalg.inv).  The one D2H of the singularity word makes it uncapturable."""
    self._check_type(matrix)
    if len(matrix.shape) > 2:
      raise ValueError("input to numpy backend method `inv` has shape {}."
                       " Only matrices are supported.".format(matrix.shape))
    if matrix.ndim < 2:
      raise np.linalg.LinAlgError("{}-dimensional array given. Array must be at least "
                                  "two-dimensional".format(matrix.ndim))
    if matrix.shape[0] != matrix.shape[1]:
      raise np.linalg.LinAlgError("Last 2 dimensions of the array must be square")
    if matrix.code in (L.I32, L.I64):          # np.linalg.inv computes integer input in float64
      matrix = self.astype(matrix, L.F64)
    if matrix.code not in (L.F32, L.F64, L.C64, L.C128):
      raise TypeError("inv needs a float32/float64/complex tensor")
    self._no_capture("inv")
    out = self._new(matrix.shape, matrix.code)
    info = self.torch.empty((), dtype=self.torch.int32, device=self.device)
    L.check(self.lib.tnb200_inv(matrix.ref(), out.ref(), info.data_ptr(), self._stream()))
    if int(info.item()) != 0:
      raise np.linalg.LinAlgError("Singular matrix")
    return out

  def compare(self, op, x, y):
    """x (op) y with numpy broadcasting -> device bool tensor (op: _lib.LT / LE / GT / GE)."""
    if not isinstance(x, B200Tensor):
      x = self._as_tensor(x, y.code)
    y = self._as_tensor(y, x.code)
    code = self._promote(x.code, y.code)
    if T.is_complex_code(code):
      raise TypeError("'<' / '<=' / '>' / '>=' are not supported for complex tensors")
    x, y = self.astype(x, code), self.astype(y, code)
    try:
      shape = tuple(np.broadcast_shapes(x.shape, y.shape))
    except ValueError as e:
      raise ValueError("operands could not be broadcast together with shapes {} {}".format(
          x.shape, y.shape)) from e
    xe = x if x.shape == shape else B200Tensor(x.t.expand(shape), code)
    ye = y if y.shape == shape else B200Tensor(y.t.expand(shape), code)
    out = self._new(shape, L.BOOL)
    L.check(self.lib.tnb200_compare(op, xe.ref(), ye.ref(), out.ref(), self._stream()))
    return out

  def index_update(self, tensor, mask, assignee):
    """numpy_backend.py:548-552: a copy of `tensor` with `assignee` (a scalar, or a size-1 device tensor read on the
    device) at the positions where the boolean `mask` is set.  A host numpy mask is uploaded."""
    self._check_type(tensor)
    if isinstance(mask, np.ndarray):
      mask = self.convert_to_tensor(np.asarray(mask, dtype=np.bool_))
    self._check_type(mask, "mask")
    if mask.code != L.BOOL:
      raise TypeError("index_update needs a boolean mask, got dtype {}".format(mask.dtype))
    if mask.shape != tensor.shape:
      try:
        mask = B200Tensor(mask.t.expand(tensor.shape), L.BOOL)
      except RuntimeError as e:
        raise IndexError("boolean index of shape {} does not match the indexed tensor of shape {}".format(
            mask.shape, tensor.shape)) from e
    out = self._new(tensor.shape, tensor.code)
    if isinstance(assignee, B200Tensor):
      if assignee.size != 1:
        raise ValueError("index_update: the assignee must be a scalar, got shape {}".format(assignee.shape))
      L.check(self.lib.tnb200_masked_fill(tensor.ref(), mask.ref(), out.ref(), 0.0, 0.0, assignee.t.data_ptr(),
                                          assignee.code, self._stream()))
    else:
      v = complex(np.asarray(assignee).item())
      L.check(self.lib.tnb200_masked_fill(tensor.ref(), mask.ref(), out.ref(), v.real, v.imag, None, 0,
                                          self._stream()))
    return out

  def eigs(self, A, args=None, initial_state=None, shape=None, dtype=None, num_krylov_vecs=50, numeig=6,
           tol=1e-8, which='LR', maxiter=None):
    """numpy_backend.py:216-291 (scipy.sparse.linalg.eigs / ARPACK there): thick-restart Arnoldi, arnoldi.py."""
    from . import arnoldi  # pylint: disable=import-outside-toplevel
    return arnoldi.eigs(self, A, args, initial_state, shape, dtype, num_krylov_vecs, numeig, tol, which, maxiter)


def register():
  """Insert the backend into the reference's registry (backend_factory.py:22-28)."""
  if not HAVE_TENSORNETWORK:
    return False
  from tensornetwork.backends import backend_factory  # type: ignore
  backend_factory._BACKENDS["cuda_b200"] = CudaB200Backend  # pylint: disable=protected-access
  return True
