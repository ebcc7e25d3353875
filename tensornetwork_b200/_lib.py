"""ctypes binding of libtnb200.so (the C ABI declared in include/tnb200.h).

There is NO fallback: if the shared library is missing or fails to load, every compute
entry point of the backend raises.  `load()` is lazy so that `import tensornetwork_b200`
stays cheap and does not touch CUDA (the reference requires backends to import their heavy
dependency lazily: tensornetwork/backends/backend_test.py:24-135).
"""
import ctypes
import os

MAX_NDIM = 16
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libtnb200.so")

# dtype codes of tnb200_dtype_t
F64, F32, F16, BF16, C64, C128, I32, I64, BOOL = range(9)
# status codes
OK, ERR_INVALID, ERR_DTYPE, ERR_CUDA, ERR_UNSUPPORTED, ERR_NOCONV = 0, -1, -2, -3, -4, -5
# ops
ADD, SUB, MUL, DIV, POW = range(5)
CONJ, SQRT, ABS, NEG, EXP, LOG, SIN, COS, SIGN, REAL, IMAG = range(11)
LT, LE, GT, GE = range(4)
CONJ_A, CONJ_B = 1, 2
MATH_DEFAULT, MATH_STRICT, MATH_SIMT = 0 << 4, 1 << 4, 2 << 4


class TensorDesc(ctypes.Structure):
  _fields_ = [("data", ctypes.c_void_p), ("dtype", ctypes.c_int32), ("ndim", ctypes.c_int32),
              ("shape", ctypes.c_int64 * MAX_NDIM), ("stride", ctypes.c_int64 * MAX_NDIM)]


class ChainStep(ctypes.Structure):
  """tnb200_chain_step_t"""
  _fields_ = [("a", TensorDesc), ("b", TensorDesc), ("c", TensorDesc), ("naxes", ctypes.c_int32), ("nbatch", ctypes.c_int32),
              ("axes_a", ctypes.c_int32 * MAX_NDIM), ("axes_b", ctypes.c_int32 * MAX_NDIM),
              ("batch_a", ctypes.c_int32 * MAX_NDIM), ("batch_b", ctypes.c_int32 * MAX_NDIM),
              ("dep_a", ctypes.c_int32), ("dep_b", ctypes.c_int32)]


_P = ctypes.POINTER(TensorDesc)
_i32, _i64, _u64, _dbl, _vp = (ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64, ctypes.c_double,
                               ctypes.c_void_p)
_pi32 = ctypes.POINTER(ctypes.c_int32)

# name -> (restype, argtypes): every symbol include/tnb200.h declares
SIGNATURES = {
    "tnb200_last_error": (ctypes.c_char_p, []),
    "tnb200_abi_version": (_i32, []),
    "tnb200_device_info": (_i32, [_pi32, _pi32, _pi32, ctypes.POINTER(_i64)]),
    "tnb200_last_kernel": (ctypes.c_char_p, []),
    "tnb200_launch_count": (_i64, []),
    "tnb200_tensordot": (_i32, [_P, _P, _P, _i32, _pi32, _pi32, _i32, _pi32, _pi32, _i32, _vp]),
    "tnb200_copy": (_i32, [_P, _P, _i32, _vp]),
    "tnb200_binary": (_i32, [_i32, _P, _P, _P, _vp]),
    "tnb200_unary": (_i32, [_i32, _P, _P, _vp]),
    "tnb200_affine_inplace": (_i32, [_P, _dbl, _dbl, _dbl, _dbl, _vp]),
    "tnb200_scale_by_device_scalar": (_i32, [_P, _vp, _i32, _i32, _vp]),
    "tnb200_axpy": (_i32, [_P, _P, _dbl, _dbl, _vp, _dbl, _vp]),
    "tnb200_fill": (_i32, [_P, _dbl, _dbl, _vp]),
    "tnb200_eye": (_i32, [_P, _i64, _vp]),
    "tnb200_randn": (_i32, [_P, _u64, _vp]),
    "tnb200_uniform": (_i32, [_P, _dbl, _dbl, _u64, _vp]),
    "tnb200_norm": (_i32, [_P, _vp, _vp]),
    "tnb200_dot": (_i32, [_P, _P, _i32, _vp, _vp]),
    "tnb200_sum": (_i32, [_P, _P, _i32, _pi32, _vp]),
    "tnb200_trace": (_i32, [_P, _P, _i64, _i32, _i32, _vp]),
    "tnb200_diagflat": (_i32, [_P, _P, _i64, _vp]),
    "tnb200_svd": (_i32, [_P, _P, _P, _P, _vp, _vp]),
    "tnb200_svd_truncation_count": (_i32, [_P, _i64, _i32, _dbl, _i32, _vp, _vp]),
    "tnb200_qr": (_i32, [_P, _P, _P, _i32, _vp]),
    "tnb200_blocksparse_maps": (_i32, [_i32, _vp, _vp, _vp, _vp, _i32, _i32, _i64, _i64, _i32, _vp, _i64, _vp, _vp]),
    "tnb200_svd_batched": (_i32, [_vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _vp]),
    "tnb200_gather": (_i32, [_vp, _vp, _vp, _i64, _i32, _i32, _vp]),
    "tnb200_blocksparse_tensordot": (_i32, [_vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp,
                                            _vp, _vp, _i64, _i64, _i32, _vp]),
    "tnb200_chain_create": (_i32, [_i32, ctypes.POINTER(ChainStep), _pi32, ctypes.POINTER(_vp)]),
    "tnb200_chain_launch": (_i32, [_vp, _vp]),
    "tnb200_chain_destroy": (_i32, [_vp]),
    "tnb200_compare": (_i32, [_i32, _P, _P, _P, _vp]),
    "tnb200_masked_fill": (_i32, [_P, _P, _P, _dbl, _dbl, _vp, _i32, _vp]),
    "tnb200_eigh": (_i32, [_P, _P, _P, _vp, _vp]),
    "tnb200_inv": (_i32, [_P, _P, _vp, _vp]),
    "tnb200_krylov_orth": (_i32, [_P, _P, _i32, _vp, _vp]),
}

_lib = None


def load(path=None):
  """dlopen the library (once) and attach the prototypes.  Raises OSError if it is absent."""
  global _lib
  if _lib is not None:
    return _lib
  path = path or os.environ.get("TNB200_LIB", LIB_PATH)
  if not os.path.exists(path):
    raise OSError("libtnb200.so not found at {} — build it with "
                  "`python -m tensornetwork_b200.build` (there is no CPU fallback)".format(path))
  lib = ctypes.CDLL(path)
  for name, (res, args) in SIGNATURES.items():
    fn = getattr(lib, name)
    fn.restype = res
    fn.argtypes = args
  if lib.tnb200_abi_version() != 1:
    raise OSError("libtnb200.so ABI version mismatch")
  _lib = lib
  return lib


def set_lib(obj):
  """Test hook: install a stand-in object exposing the same tnb200_* callables."""
  global _lib
  _lib = obj


class Tnb200Error(RuntimeError):
  pass


def check(rc):
  """Translate a tnb200_status_t into the reference's exception conventions (SURVEY 8b)."""
  if rc == 0:
    return
  msg = _lib.tnb200_last_error()
  msg = msg.decode() if isinstance(msg, bytes) else str(msg)
  if rc == ERR_INVALID:
    raise ValueError(msg)
  if rc == ERR_DTYPE:
    raise TypeError(msg)
  if rc == ERR_UNSUPPORTED:
    raise NotImplementedError(msg)
  raise Tnb200Error("tnb200 status {}: {}".format(rc, msg))
