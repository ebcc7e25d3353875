// elementwise.cu — the memory-bound helper ops of SURVEY.md 8(a) row a6 (and the strided copy
// that materialises a transpose when reshape() cannot be a view, row a2).
// All kernels are HBM-bound gather/scatter over <= 8 merged modes; no data reuse, so no shared
// memory; grids are sized in multiples of the SM count with a grid-stride loop.
#include "common.cuh"
#include <math.h>

namespace tnb {

// ------------------------------------------------------------------ universal value type
struct ZV { double re, im; };  // every dtype round-trips exactly except |int64| > 2^53

template <typename T> __device__ inline ZV ld(const T* p);
template <> __device__ inline ZV ld<double>(const double* p) { return {*p, 0.0}; }
template <> __device__ inline ZV ld<float>(const float* p) { return {(double)*p, 0.0}; }
template <> __device__ inline ZV ld<__half>(const __half* p) { return {(double)__half2float(*p), 0.0}; }
template <> __device__ inline ZV ld<__nv_bfloat16>(const __nv_bfloat16* p) { return {(double)__bfloat162float(*p), 0.0}; }
template <> __device__ inline ZV ld<cuFloatComplex>(const cuFloatComplex* p) { cuFloatComplex v = *p; return {(double)v.x, (double)v.y}; }
template <> __device__ inline ZV ld<cuDoubleComplex>(const cuDoubleComplex* p) { cuDoubleComplex v = *p; return {v.x, v.y}; }
template <> __device__ inline ZV ld<int32_t>(const int32_t* p) { return {(double)*p, 0.0}; }
template <> __device__ inline ZV ld<long long>(const long long* p) { return {(double)*p, 0.0}; }
template <> __device__ inline ZV ld<bool>(const bool* p) { return {*p ? 1.0 : 0.0, 0.0}; }

template <typename T> __device__ inline void stv(T* p, ZV v);
template <> __device__ inline void stv<double>(double* p, ZV v) { *p = v.re; }
template <> __device__ inline void stv<float>(float* p, ZV v) { *p = (float)v.re; }
template <> __device__ inline void stv<__half>(__half* p, ZV v) { *p = __float2half_rn((float)v.re); }
template <> __device__ inline void stv<__nv_bfloat16>(__nv_bfloat16* p, ZV v) { *p = __float2bfloat16_rn((float)v.re); }
template <> __device__ inline void stv<cuFloatComplex>(cuFloatComplex* p, ZV v) { *p = make_cuFloatComplex((float)v.re, (float)v.im); }
template <> __device__ inline void stv<cuDoubleComplex>(cuDoubleComplex* p, ZV v) { *p = make_cuDoubleComplex(v.re, v.im); }
template <> __device__ inline void stv<int32_t>(int32_t* p, ZV v) { *p = (int32_t)llrint(v.re); }
template <> __device__ inline void stv<long long>(long long* p, ZV v) { *p = llrint(v.re); }
template <> __device__ inline void stv<bool>(bool* p, ZV v) { *p = v.re != 0.0 || v.im != 0.0; }

#define TNB_DISPATCH_DTYPE(dt, FN, ...)                                           \
  switch (dt) {                                                                   \
    case TNB200_F64: return FN<double>(__VA_ARGS__);                              \
    case TNB200_F32: return FN<float>(__VA_ARGS__);                               \
    case TNB200_F16: return FN<__half>(__VA_ARGS__);                              \
    case TNB200_BF16: return FN<__nv_bfloat16>(__VA_ARGS__);                      \
    case TNB200_C64: return FN<cuFloatComplex>(__VA_ARGS__);                      \
    case TNB200_C128: return FN<cuDoubleComplex>(__VA_ARGS__);                    \
    case TNB200_I32: return FN<int32_t>(__VA_ARGS__);                             \
    case TNB200_I64: return FN<long long>(__VA_ARGS__);                           \
    default: set_error("bad dtype %d", dt); return TNB200_ERR_DTYPE;              \
  }

static inline unsigned grid_for(int64_t n, int threads = 256) {
  int64_t blocks = (n + threads - 1) / threads;
  int64_t cap = (int64_t)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

// Build merged modes for up to three same-shape operands (0-strides allowed).
static int build_modes(const tnb200_tensor_t* a, const tnb200_tensor_t* b, const tnb200_tensor_t* c,
                       DevModes& dm, int64_t& total) {
  ModeList m;
  int nops = 1 + (b ? 1 : 0) + (c ? 1 : 0);
  for (int i = 0; i < a->ndim; ++i) {
    if (b && b->shape[i] != a->shape[i]) { set_error("elementwise: shape mismatch on axis %d", i); return TNB200_ERR_INVALID; }
    if (c && c->shape[i] != a->shape[i]) { set_error("elementwise: shape mismatch on axis %d", i); return TNB200_ERR_INVALID; }
    m.push(a->shape[i], a->stride[i], b ? b->stride[i] : 0, c ? c->stride[i] : 0);
  }
  total = m.total();
  merge_modes(m, nops);
  if (!to_dev(m, dm)) { set_error("elementwise: more than %d non-mergeable modes", kDevModes); return TNB200_ERR_UNSUPPORTED; }
  return 0;
}

// ------------------------------------------------------------------------------- copy
template <typename Tin, typename Tout>
__global__ void copy_kernel(const Tin* __restrict__ src, Tout* __restrict__ dst, DevModes m, int64_t total, int conj) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t o0, o1;
    if (m.n == 1) { o0 = i * m.s0[0]; o1 = i * m.s1[0]; } else mode_offsets(m, i, o0, o1);
    ZV v = ld<Tin>(src + o0);
    if (conj) v.im = -v.im;
    stv<Tout>(dst + o1, v);
  }
}
// same-type copy moves raw bits (exact for int64 and NaN payloads)
template <typename T>
__global__ void copy_same_kernel(const T* __restrict__ src, T* __restrict__ dst, DevModes m, int64_t total) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t o0, o1;
    if (m.n == 1) { o0 = i * m.s0[0]; o1 = i * m.s1[0]; } else mode_offsets(m, i, o0, o1);
    dst[o1] = src[o0];
  }
}
// 2-D tiled transpose for the common "swap fastest axis" case: coalesced on both sides.
template <typename T>
__global__ void transpose_tile_kernel(const T* __restrict__ src, T* __restrict__ dst, int64_t rows, int64_t cols,
                                      int64_t s_row, int64_t s_col, int64_t d_row, int64_t d_col,
                                      DevModes outer, int64_t tiles_r, int64_t tiles_c) {
  // src is col-fast (s_col == 1), dst is row-fast (d_row == 1); outer modes: s0 src, s1 dst
  __shared__ T tile[32][33];
  int64_t bid = blockIdx.x;
  int64_t tc = bid % tiles_c; bid /= tiles_c;
  int64_t tr = bid % tiles_r; bid /= tiles_r;
  int64_t o0, o1;
  mode_offsets(outer, bid, o0, o1);
  int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int j = ty; j < 32; j += 8) {
    int64_t r = tr * 32 + j, c = tc * 32 + tx;
    if (r < rows && c < cols) tile[j][tx] = src[o0 + r * s_row + c * s_col];
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    int64_t c = tc * 32 + j, r = tr * 32 + tx;
    if (r < rows && c < cols) dst[o1 + r * d_row + c * d_col] = tile[tx][j];
  }
}

template <typename T>
static int copy_same(const tnb200_tensor_t* src, const tnb200_tensor_t* dst, cudaStream_t st) {
  // try the tiled transpose: find the src-fastest mode and the dst-fastest mode
  ModeList m;
  for (int i = 0; i < src->ndim; ++i) m.push(src->shape[i], src->stride[i], dst->stride[i]);
  int64_t total = m.total();
  merge_modes(m, 2);
  int is = -1, id = -1;
  for (int i = 0; i < m.n; ++i) { if (m.s0[i] == 1) is = i; if (m.s1[i] == 1) id = i; }
  if (is >= 0 && id >= 0 && is != id && m.ext[is] >= 16 && m.ext[id] >= 16 && total >= 4096) {
    ModeList outer;
    for (int i = 0; i < m.n; ++i) if (i != is && i != id) outer.push(m.ext[i], m.s0[i], m.s1[i]);
    DevModes od;
    if (to_dev(outer, od)) {
      int64_t rows = m.ext[id], cols = m.ext[is];  // rows: dst-fast, cols: src-fast
      int64_t tr = (rows + 31) / 32, tc = (cols + 31) / 32;
      int64_t blocks = tr * tc * outer.total();
      if (blocks < (1LL << 31)) {
        transpose_tile_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(
            (const T*)src->data, (T*)dst->data, rows, cols, m.s0[id], m.s0[is], m.s1[id], m.s1[is], od, tr, tc);
        TNB_LAUNCH_CHECK();
        count_launch();
        return 0;
      }
    }
  }
  DevModes dm;
  if (!to_dev(m, dm)) { set_error("copy: more than %d non-mergeable modes", kDevModes); return TNB200_ERR_UNSUPPORTED; }
  copy_same_kernel<T><<<grid_for(total), 256, 0, st>>>((const T*)src->data, (T*)dst->data, dm, total);
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}

template <typename Tin>
static int copy_from(const tnb200_tensor_t* src, const tnb200_tensor_t* dst, int conj, cudaStream_t st) {
  DevModes dm; int64_t total;
  int rc = build_modes(src, dst, nullptr, dm, total);
  if (rc) return rc;
  unsigned g = grid_for(total);
#define TNB_CP(TO) copy_kernel<Tin, TO><<<g, 256, 0, st>>>((const Tin*)src->data, (TO*)dst->data, dm, total, conj)
  switch (dst->dtype) {
    case TNB200_F64: TNB_CP(double); break;
    case TNB200_F32: TNB_CP(float); break;
    case TNB200_F16: TNB_CP(__half); break;
    case TNB200_BF16: TNB_CP(__nv_bfloat16); break;
    case TNB200_C64: TNB_CP(cuFloatComplex); break;
    case TNB200_C128: TNB_CP(cuDoubleComplex); break;
    case TNB200_I32: TNB_CP(int32_t); break;
    case TNB200_I64: TNB_CP(long long); break;
    case TNB200_BOOL: TNB_CP(bool); break;
    default: set_error("copy: bad dtype"); return TNB200_ERR_DTYPE;
  }
#undef TNB_CP
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}

int copy_strided(const tnb200_tensor_t* src, const tnb200_tensor_t* dst, int conj, cudaStream_t st) {
  if (src->ndim != dst->ndim) { set_error("copy: rank mismatch"); return TNB200_ERR_INVALID; }
  for (int i = 0; i < src->ndim; ++i)
    if (src->shape[i] != dst->shape[i]) { set_error("copy: shape mismatch on axis %d", i); return TNB200_ERR_INVALID; }
  if (numel(src) == 0) return 0;
  bool cj = conj && dtype_is_complex(src->dtype);
  if (src->dtype == TNB200_BOOL) return dst->dtype == TNB200_BOOL ? copy_same<bool>(src, dst, st) : copy_from<bool>(src, dst, 0, st);
  if (src->dtype == dst->dtype && !cj) { TNB_DISPATCH_DTYPE(src->dtype, copy_same, src, dst, st); }
  TNB_DISPATCH_DTYPE(src->dtype, copy_from, src, dst, cj ? 1 : 0, st);
}

// ------------------------------------------------------------------------ complex math
__device__ inline ZV zmul(ZV a, ZV b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }
__device__ inline ZV zdiv(ZV a, ZV b) {
  if (b.im == 0.0) return {a.re / b.re, a.im / b.re};
  // Smith's algorithm
  if (fabs(b.re) >= fabs(b.im)) {
    double r = b.im / b.re, d = b.re + b.im * r;
    return {(a.re + a.im * r) / d, (a.im - a.re * r) / d};
  }
  double r = b.re / b.im, d = b.re * r + b.im;
  return {(a.re * r + a.im) / d, (a.im * r - a.re) / d};
}
__device__ inline ZV zsqrt(ZV a, bool is_complex) {
  if (!is_complex || a.im == 0.0) {
    if (a.re >= 0.0 || !is_complex) return {sqrt(a.re), 0.0};
    return {0.0, sqrt(-a.re)};
  }
  double r = hypot(a.re, a.im);
  double sr = sqrt(0.5 * (r + fabs(a.re)));
  double si = a.im / (2.0 * sr);
  if (a.re >= 0.0) return {sr, si};
  return {fabs(si), copysign(sr, a.im)};
}
__device__ inline ZV zexp(ZV a) { double e = exp(a.re); double s, c; sincos(a.im, &s, &c); return {e * c, e * s}; }
__device__ inline ZV zlog(ZV a, bool is_complex) {
  if (!is_complex) return {log(a.re), 0.0};
  return {log(hypot(a.re, a.im)), atan2(a.im, a.re)};
}
__device__ inline ZV zpow(ZV a, ZV b, bool is_complex) {
  if (!is_complex) return {pow(a.re, b.re), 0.0};
  if (a.re == 0.0 && a.im == 0.0) return {(b.re == 0.0 && b.im == 0.0) ? 1.0 : 0.0, 0.0};
  return zexp(zmul(b, zlog(a, true)));
}

// ------------------------------------------------------------------------------ binary
template <typename T>
__global__ void binary_kernel(int op, const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ c,
                              DevModes m, int64_t total, int is_complex, int is_int) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t o0, o1, o2;
    mode_offsets3(m, i, o0, o1, o2);
    ZV x = ld<T>(a + o0), y = ld<T>(b + o1), r;
    switch (op) {
      case TNB200_ADD: r = {x.re + y.re, x.im + y.im}; break;
      case TNB200_SUB: r = {x.re - y.re, x.im - y.im}; break;
      case TNB200_MUL: r = is_complex ? zmul(x, y) : ZV{x.re * y.re, 0.0}; break;
      case TNB200_DIV:
        if (is_int) r = {floor(x.re / y.re), 0.0};
        else r = is_complex ? zdiv(x, y) : ZV{x.re / y.re, 0.0};
        break;
      default: r = zpow(x, y, is_complex); break;
    }
    stv<T>(c + o2, r);
  }
}
// f32 / f64 keep native arithmetic (bit-identical to numpy's ufuncs for + - * /)
template <typename T>
__global__ void binary_native_kernel(int op, const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ c,
                                     DevModes m, int64_t total) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t o0, o1, o2;
    mode_offsets3(m, i, o0, o1, o2);
    T x = a[o0], y = b[o1], r;
    switch (op) {
      case TNB200_ADD: r = x + y; break;
      case TNB200_SUB: r = x - y; break;
      case TNB200_MUL: r = x * y; break;
      default: r = x / y; break;
    }
    c[o2] = r;
  }
}
template <typename T>
static int binary_t(int op, const tnb200_tensor_t* a, const tnb200_tensor_t* b, const tnb200_tensor_t* c, cudaStream_t st) {
  DevModes dm; int64_t total;
  int rc = build_modes(a, b, c, dm, total);
  if (rc) return rc;
  if (total == 0) return 0;
  binary_kernel<T><<<grid_for(total), 256, 0, st>>>(op, (const T*)a->data, (const T*)b->data, (T*)c->data, dm, total,
                                                    dtype_is_complex(a->dtype), a->dtype >= TNB200_I32);
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}
template <typename T>
static int binary_native_t(int op, const tnb200_tensor_t* a, const tnb200_tensor_t* b, const tnb200_tensor_t* c, cudaStream_t st) {
  DevModes dm; int64_t total;
  int rc = build_modes(a, b, c, dm, total);
  if (rc) return rc;
  if (total == 0) return 0;
  binary_native_kernel<T><<<grid_for(total), 256, 0, st>>>(op, (const T*)a->data, (const T*)b->data, (T*)c->data, dm, total);
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------- unary
template <typename Tin, typename Tout>
__global__ void unary_kernel(int op, const Tin* __restrict__ a, Tout* __restrict__ c, DevModes m, int64_t total, int is_complex) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t o0, o1;
    mode_offsets(m, i, o0, o1);
    ZV x = ld<Tin>(a + o0), r;
    switch (op) {
      case TNB200_CONJ: r = {x.re, -x.im}; break;
      case TNB200_SQRT: r = zsqrt(x, is_complex); break;
      case TNB200_ABS: r = {is_complex ? hypot(x.re, x.im) : fabs(x.re), 0.0}; break;
      case TNB200_NEG: r = {-x.re, -x.im}; break;
      case TNB200_EXP: r = is_complex ? zexp(x) : ZV{exp(x.re), 0.0}; break;
      case TNB200_LOG: r = zlog(x, is_complex); break;
      case TNB200_SIN: r = is_complex ? ZV{sin(x.re) * cosh(x.im), cos(x.re) * sinh(x.im)} : ZV{sin(x.re), 0.0}; break;
      case TNB200_COS: r = is_complex ? ZV{cos(x.re) * cosh(x.im), -sin(x.re) * sinh(x.im)} : ZV{cos(x.re), 0.0}; break;
      case TNB200_SIGN:
        if (is_complex) { double n = hypot(x.re, x.im); r = n == 0.0 ? ZV{0.0, 0.0} : ZV{x.re / n, x.im / n}; }
        else r = {x.re > 0.0 ? 1.0 : (x.re < 0.0 ? -1.0 : 0.0), 0.0};
        break;
      case TNB200_REAL: r = {x.re, 0.0}; break;
      default: r = {x.im, 0.0}; break;
    }
    stv<Tout>(c + o1, r);
  }
}
template <typename Tin, typename Tout>
static int unary_tt(int op, const tnb200_tensor_t* a, const tnb200_tensor_t* c, cudaStream_t st) {
  DevModes dm; int64_t total;
  int rc = build_modes(a, c, nullptr, dm, total);
  if (rc) return rc;
  if (total == 0) return 0;
  unary_kernel<Tin, Tout><<<grid_for(total), 256, 0, st>>>(op, (const Tin*)a->data, (Tout*)c->data, dm, total,
                                                           dtype_is_complex(a->dtype));
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}
template <typename T>
static int unary_t(int op, const tnb200_tensor_t* a, const tnb200_tensor_t* c, cudaStream_t st) {
  return unary_tt<T, T>(op, a, c, st);
}

// ------------------------------------------------- in-place affine / device-scalar scale / axpy
template <typename T>
__global__ void affine_kernel(T* x, DevModes m, int64_t total, ZV alpha, ZV beta, const void* alpha_dev, int alpha_dt,
                              int power, int is_complex) {
  if (alpha_dev) {
    ZV s;
    switch (alpha_dt) {
      case TNB200_F64: s = ld<double>((const double*)alpha_dev); break;
      case TNB200_F32: s = ld<float>((const float*)alpha_dev); break;
      case TNB200_F16: s = ld<__half>((const __half*)alpha_dev); break;
      case TNB200_BF16: s = ld<__nv_bfloat16>((const __nv_bfloat16*)alpha_dev); break;
      case TNB200_C64: s = ld<cuFloatComplex>((const cuFloatComplex*)alpha_dev); break;
      default: s = ld<cuDoubleComplex>((const cuDoubleComplex*)alpha_dev); break;
    }
    alpha = power < 0 ? zdiv(ZV{1.0, 0.0}, s) : s;
    if (power < 0 && s.im == 0.0) alpha = {1.0 / s.re, 0.0};
    beta = {0.0, 0.0};
  }
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t o = m.n == 1 ? i * m.s0[0] : mode_offset0(m, i);
    ZV v = ld<T>(x + o);
    ZV r = is_complex ? zmul(v, alpha) : ZV{v.re * alpha.re, 0.0};
    r.re += beta.re; r.im += beta.im;
    stv<T>(x + o, r);
  }
}
// division by a device scalar must be a true division to match numpy's `x /= n`
template <typename T>
__global__ void divide_dev_kernel(T* x, DevModes m, int64_t total, const void* s_dev, int s_dt, int is_complex) {
  ZV s;
  switch (s_dt) {
    case TNB200_F64: s = ld<double>((const double*)s_dev); break;
    case TNB200_F32: s = ld<float>((const float*)s_dev); break;
    case TNB200_F16: s = ld<__half>((const __half*)s_dev); break;
    case TNB200_BF16: s = ld<__nv_bfloat16>((const __nv_bfloat16*)s_dev); break;
    case TNB200_C64: s = ld<cuFloatComplex>((const cuFloatComplex*)s_dev); break;
    default: s = ld<cuDoubleComplex>((const cuDoubleComplex*)s_dev); break;
  }
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t o = m.n == 1 ? i * m.s0[0] : mode_offset0(m, i);
    ZV v = ld<T>(x + o);
    ZV r = (is_complex && s.im != 0.0) ? zdiv(v, s) : ZV{v.re / s.re, v.im / s.re};
    stv<T>(x + o, r);
  }
}
template <typename T>
static int affine_t(const tnb200_tensor_t* x, ZV alpha, ZV beta, const void* alpha_dev, int alpha_dt, int power, cudaStream_t st) {
  DevModes dm; int64_t total;
  int rc = build_modes(x, nullptr, nullptr, dm, total);
  if (rc) return rc;
  if (total == 0) return 0;
  if (alpha_dev && power < 0)
    divide_dev_kernel<T><<<grid_for(total), 256, 0, st>>>((T*)x->data, dm, total, alpha_dev, alpha_dt, dtype_is_complex(x->dtype));
  else
    affine_kernel<T><<<grid_for(total), 256, 0, st>>>((T*)x->data, dm, total, alpha, beta, alpha_dev, alpha_dt, power,
                                                      dtype_is_complex(x->dtype));
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}

template <typename T>
__global__ void axpy_kernel(const T* __restrict__ x, T* y, DevModes m, int64_t total, ZV alpha, const void* alpha_dev,
                            double sign, int is_complex) {
  if (alpha_dev) {
    ZV s = ld<T>((const T*)alpha_dev);
    alpha = {sign * s.re, sign * s.im};
  }
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t o0, o1;
    if (m.n == 1) { o0 = i * m.s0[0]; o1 = i * m.s1[0]; } else mode_offsets(m, i, o0, o1);
    ZV xv = ld<T>(x + o0), yv = ld<T>(y + o1);
    ZV p = is_complex ? zmul(xv, alpha) : ZV{xv.re * alpha.re, 0.0};
    stv<T>(y + o1, ZV{yv.re + p.re, yv.im + p.im});
  }
}
template <typename T>
static int axpy_t(const tnb200_tensor_t* x, const tnb200_tensor_t* y, ZV alpha, const void* alpha_dev, double sign, cudaStream_t st) {
  DevModes dm; int64_t total;
  int rc = build_modes(x, y, nullptr, dm, total);
  if (rc) return rc;
  if (total == 0) return 0;
  axpy_kernel<T><<<grid_for(total), 256, 0, st>>>((const T*)x->data, (T*)y->data, dm, total, alpha, alpha_dev, sign,
                                                  dtype_is_complex(x->dtype));
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}

// ------------------------------------------------------------------ fill / eye / diagflat
template <typename T>
__global__ void fill_kernel(T* c, DevModes m, int64_t total, ZV v) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t o = m.n == 1 ? i * m.s0[0] : mode_offset0(m, i);
    stv<T>(c + o, v);
  }
}
template <typename T>
static int fill_t(const tnb200_tensor_t* c, ZV v, cudaStream_t st) {
  DevModes dm; int64_t total;
  int rc = build_modes(c, nullptr, nullptr, dm, total);
  if (rc) return rc;
  if (total == 0) return 0;
  fill_kernel<T><<<grid_for(total), 256, 0, st>>>((T*)c->data, dm, total, v);
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}
// c[r, q] = (q - r == k) ? src[r - max(-k, 0)] (or 1) : 0
template <typename T>
__global__ void diag_kernel(const T* __restrict__ src, DevModes sm, T* c, int64_t rows, int64_t cols, int64_t sr, int64_t sc, int64_t k) {
  int64_t total = rows * cols;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / cols, q = i - r * cols;
    ZV v = {0.0, 0.0};
    if (q - r == k) {
      if (src) { int64_t j = r - (k < 0 ? -k : 0); v = ld<T>(src + mode_offset0(sm, j)); }
      else v = {1.0, 0.0};
    }
    stv<T>(c + r * sr + q * sc, v);
  }
}
template <typename T>
static int diag_t(const tnb200_tensor_t* a, const tnb200_tensor_t* c, int64_t k, cudaStream_t st) {
  DevModes sm; sm.n = 0;
  if (a) {
    ModeList m;
    for (int i = 0; i < a->ndim; ++i) m.push(a->shape[i], a->stride[i]);
    merge_modes(m, 1);
    if (!to_dev(m, sm)) { set_error("diagflat: too many modes"); return TNB200_ERR_UNSUPPORTED; }
  }
  int64_t total = c->shape[0] * c->shape[1];
  if (total == 0) return 0;
  diag_kernel<T><<<grid_for(total), 256, 0, st>>>(a ? (const T*)a->data : nullptr, sm, (T*)c->data, c->shape[0], c->shape[1],
                                                  c->stride[0], c->stride[1], k);
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------- random
__device__ inline void philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
__device__ inline double u53(uint32_t a, uint32_t b) {  // (0, 1)
  uint64_t x = ((uint64_t)a << 21) ^ (uint64_t)(b >> 11);
  return ((double)(x & ((1ULL << 53) - 1)) + 0.5) * (1.0 / 9007199254740992.0);
}
template <typename T>
__global__ void random_kernel(T* c, DevModes m, int64_t total, uint64_t seed, int normal, double lo, double hi, int is_complex) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    uint32_t r[4];
    philox4x32((uint32_t)i, (uint32_t)(i >> 32), 0x7b200u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
    double u1 = u53(r[0], r[1]), u2 = u53(r[2], r[3]);
    ZV v;
    if (normal) {
      double rad = sqrt(-2.0 * log(u1)), s, co;
      sincospi(2.0 * u2, &s, &co);
      v = {rad * co, is_complex ? rad * s : 0.0};
    } else {
      v = {lo + (hi - lo) * u1, is_complex ? lo + (hi - lo) * u2 : 0.0};
    }
    int64_t o = m.n == 1 ? i * m.s0[0] : mode_offset0(m, i);
    stv<T>(c + o, v);
  }
}
template <typename T>
static int random_t(const tnb200_tensor_t* c, uint64_t seed, int normal, double lo, double hi, cudaStream_t st) {
  DevModes dm; int64_t total;
  int rc = build_modes(c, nullptr, nullptr, dm, total);
  if (rc) return rc;
  if (total == 0) return 0;
  random_kernel<T><<<grid_for(total), 256, 0, st>>>((T*)c->data, dm, total, seed, normal, lo, hi, dtype_is_complex(c->dtype));
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}

// --------------------------------------------------------------------------- reductions
__device__ inline ZV block_reduce(ZV v) {
  __shared__ double sre[32], sim[32];
  for (int o = 16; o > 0; o >>= 1) {
    v.re += __shfl_down_sync(0xffffffffu, v.re, o);
    v.im += __shfl_down_sync(0xffffffffu, v.im, o);
  }
  int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) { sre[w] = v.re; sim[w] = v.im; }
  __syncthreads();
  int nw = (blockDim.x + 31) >> 5;
  if (w == 0) {
    v = l < nw ? ZV{sre[l], sim[l]} : ZV{0.0, 0.0};
    for (int o = 16; o > 0; o >>= 1) {
      v.re += __shfl_down_sync(0xffffffffu, v.re, o);
      v.im += __shfl_down_sync(0xffffffffu, v.im, o);
    }
  }
  return v;  // valid in thread 0
}
// mode 0: sum |x|^2 ; mode 1: sum conj?(x) * y
template <typename T>
__global__ void reduce_partial_kernel(const T* __restrict__ x, const T* __restrict__ y, DevModes m, int64_t total, int mode,
                                      int conj_x, ZV* partial) {
  ZV acc = {0.0, 0.0};
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t o0, o1;
    if (m.n == 1) { o0 = i * m.s0[0]; o1 = i * m.s1[0]; } else mode_offsets(m, i, o0, o1);
    ZV a = ld<T>(x + o0);
    if (mode == 0) acc.re += a.re * a.re + a.im * a.im;
    else {
      ZV b = ld<T>(y + o1);
      if (conj_x) a.im = -a.im;
      ZV p = zmul(a, b);
      acc.re += p.re; acc.im += p.im;
    }
  }
  acc = block_reduce(acc);
  if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}
template <typename Tout>
__global__ void reduce_final_kernel(const ZV* partial, int n, int do_sqrt, Tout* out) {
  ZV acc = {0.0, 0.0};
  for (int i = threadIdx.x; i < n; i += blockDim.x) { acc.re += partial[i].re; acc.im += partial[i].im; }
  acc = block_reduce(acc);
  if (threadIdx.x == 0) {
    if (do_sqrt) acc = {sqrt(acc.re), 0.0};
    stv<Tout>(out, acc);
  }
}
template <typename T>
static int reduce_t(const tnb200_tensor_t* x, const tnb200_tensor_t* y, int mode, int conj_x, void* out, int out_dt, cudaStream_t st) {
  DevModes dm; int64_t total;
  int rc = build_modes(x, y, nullptr, dm, total);
  if (rc) return rc;
  unsigned g = total > 0 ? grid_for(total) : 1;
  if (g > 1024) g = 1024;
  ZV* partial = nullptr;
  rc = ws_alloc((void**)&partial, sizeof(ZV) * g, st);
  if (rc) return rc;
  reduce_partial_kernel<T><<<g, 256, 0, st>>>((const T*)x->data, y ? (const T*)y->data : nullptr, dm, total, mode, conj_x, partial);
  switch (out_dt) {
    case TNB200_F64: reduce_final_kernel<double><<<1, 256, 0, st>>>(partial, g, mode == 0, (double*)out); break;
    case TNB200_F32: reduce_final_kernel<float><<<1, 256, 0, st>>>(partial, g, mode == 0, (float*)out); break;
    case TNB200_F16: reduce_final_kernel<__half><<<1, 256, 0, st>>>(partial, g, mode == 0, (__half*)out); break;
    case TNB200_BF16: reduce_final_kernel<__nv_bfloat16><<<1, 256, 0, st>>>(partial, g, mode == 0, (__nv_bfloat16*)out); break;
    case TNB200_C64: reduce_final_kernel<cuFloatComplex><<<1, 256, 0, st>>>(partial, g, mode == 0, (cuFloatComplex*)out); break;
    case TNB200_C128: reduce_final_kernel<cuDoubleComplex><<<1, 256, 0, st>>>(partial, g, mode == 0, (cuDoubleComplex*)out); break;
    case TNB200_I32: reduce_final_kernel<int32_t><<<1, 256, 0, st>>>(partial, g, mode == 0, (int32_t*)out); break;
    default: reduce_final_kernel<long long><<<1, 256, 0, st>>>(partial, g, mode == 0, (long long*)out); break;
  }
  TNB_LAUNCH_CHECK();
  count_launch(2);
  return ws_free(partial, st);
}

// sum over "reduced" modes: one block per output element
template <typename T>
__global__ void sum_axes_kernel(const T* __restrict__ a, T* c, DevModes keep /*s0 a, s1 c*/, DevModes red /*s0 a*/,
                                int64_t nkeep, int64_t nred, int64_t base_off) {
  for (int64_t o = blockIdx.x; o < nkeep; o += gridDim.x) {
    int64_t oa, oc;
    mode_offsets(keep, o, oa, oc);
    ZV acc = {0.0, 0.0};
    for (int64_t r = threadIdx.x; r < nred; r += blockDim.x) {
      ZV v = ld<T>(a + base_off + oa + mode_offset0(red, r));
      acc.re += v.re; acc.im += v.im;
    }
    acc = block_reduce(acc);
    if (threadIdx.x == 0) stv<T>(c + oc, acc);
    __syncthreads();
  }
}
template <typename T>
static int sum_axes_t(const void* a, void* c, const ModeList& keep, const ModeList& red, int64_t base_off, cudaStream_t st) {
  DevModes dk, dr;
  if (!to_dev(keep, dk) || !to_dev(red, dr)) { set_error("sum: too many modes"); return TNB200_ERR_UNSUPPORTED; }
  int64_t nkeep = keep.total(), nred = red.total();
  if (nkeep == 0) return 0;
  int64_t g = nkeep < (int64_t)num_sms() * 8 ? nkeep : (int64_t)num_sms() * 8;
  int threads = nred >= 128 ? 128 : 32;
  sum_axes_kernel<T><<<(unsigned)g, threads, 0, st>>>((const T*)a, (T*)c, dk, dr, nkeep, nred, base_off);
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}

template <typename T>
__global__ void gather_kernel(const T* __restrict__ src, const long long* __restrict__ idx, T* __restrict__ dst, int64_t n, int scatter) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (scatter) dst[idx[i]] = src[i]; else dst[i] = src[idx[i]];
  }
}
template <typename T>
static int gather_t(const void* src, const int64_t* idx, void* dst, int64_t n, int scatter, cudaStream_t st) {
  if (n == 0) return 0;
  gather_kernel<T><<<grid_for(n), 256, 0, st>>>((const T*)src, (const long long*)idx, (T*)dst, n, scatter);
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}

// ---------------------------------------------------------------------- masks (TNB200_BOOL)
// c = a (op) b elementwise for real dtypes, c bool; 0-strides express broadcasting
template <typename T>
__global__ void compare_kernel(int op, const T* __restrict__ a, const T* __restrict__ b, bool* __restrict__ c, DevModes m, int64_t total) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t o0, o1, o2;
    mode_offsets3(m, i, o0, o1, o2);
    const auto x = to_acc(a[o0]), y = to_acc(b[o1]);
    c[o2] = op == TNB200_LT ? x < y : op == TNB200_LE ? x <= y : op == TNB200_GT ? x > y : x >= y;
  }
}
template <typename T>
static int compare_t(int op, const tnb200_tensor_t* a, const tnb200_tensor_t* b, const tnb200_tensor_t* c, cudaStream_t st) {
  DevModes dm; int64_t total;
  int rc = build_modes(a, b, c, dm, total);
  if (rc) return rc;
  if (total == 0) return 0;
  compare_kernel<T><<<grid_for(total), 256, 0, st>>>(op, (const T*)a->data, (const T*)b->data, (bool*)c->data, dm, total);
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}
__device__ inline ZV ld_any(const void* p, int dt) {
  switch (dt) {
    case TNB200_F64: return ld<double>((const double*)p);
    case TNB200_F32: return ld<float>((const float*)p);
    case TNB200_F16: return ld<__half>((const __half*)p);
    case TNB200_BF16: return ld<__nv_bfloat16>((const __nv_bfloat16*)p);
    case TNB200_C64: return ld<cuFloatComplex>((const cuFloatComplex*)p);
    case TNB200_C128: return ld<cuDoubleComplex>((const cuDoubleComplex*)p);
    case TNB200_I32: return ld<int32_t>((const int32_t*)p);
    case TNB200_I64: return ld<long long>((const long long*)p);
    default: return ld<bool>((const bool*)p);
  }
}
// out = mask ? value : src; the value is given on the host or read on the device (value_dev, value_dt)
template <typename T>
__global__ void masked_fill_kernel(const T* __restrict__ src, const bool* __restrict__ mask, T* __restrict__ out, DevModes m, int64_t total,
                                   ZV value, const void* value_dev, int value_dt) {
  if (value_dev) value = ld_any(value_dev, value_dt);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t o0, o1, o2;
    mode_offsets3(m, i, o0, o1, o2);
    if (mask[o1]) stv<T>(out + o2, value); else out[o2] = src[o0];
  }
}
template <typename T>
static int masked_fill_t(const tnb200_tensor_t* src, const tnb200_tensor_t* mask, const tnb200_tensor_t* out, ZV value, const void* value_dev,
                         int value_dt, cudaStream_t st) {
  DevModes dm; int64_t total;
  int rc = build_modes(src, mask, out, dm, total);
  if (rc) return rc;
  if (total == 0) return 0;
  masked_fill_kernel<T><<<grid_for(total), 256, 0, st>>>((const T*)src->data, (const bool*)mask->data, (T*)out->data, dm, total, value,
                                                         value_dev, value_dt);
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}

static int real_dtype(int dt) {
  if (dt == TNB200_C128) return TNB200_F64;
  if (dt == TNB200_C64) return TNB200_F32;
  return dt;
}

}  // namespace tnb

using namespace tnb;

extern "C" {

int32_t tnb200_copy(const tnb200_tensor_t* src, const tnb200_tensor_t* dst, int32_t conj, void* stream) {
  TNB_REQUIRE(valid_tensor(src) && valid_tensor(dst), TNB200_ERR_INVALID, "copy: invalid tensor descriptor");
  return copy_strided(src, dst, conj, (cudaStream_t)stream);
}

int32_t tnb200_binary(int32_t op, const tnb200_tensor_t* a, const tnb200_tensor_t* b, const tnb200_tensor_t* c, void* stream) {
  TNB_REQUIRE(valid_tensor(a) && valid_tensor(b) && valid_tensor(c), TNB200_ERR_INVALID, "binary: invalid tensor descriptor");
  TNB_REQUIRE(a->ndim == b->ndim && a->ndim == c->ndim, TNB200_ERR_INVALID, "binary: rank mismatch");
  TNB_REQUIRE(a->dtype == b->dtype && a->dtype == c->dtype, TNB200_ERR_DTYPE, "binary: dtype mismatch");
  TNB_REQUIRE(op >= TNB200_ADD && op <= TNB200_POW, TNB200_ERR_INVALID, "binary: bad op %d", op);
  cudaStream_t st = (cudaStream_t)stream;
  if (op != TNB200_POW && a->dtype == TNB200_F64) return binary_native_t<double>(op, a, b, c, st);
  if (op != TNB200_POW && a->dtype == TNB200_F32) return binary_native_t<float>(op, a, b, c, st);
  TNB_DISPATCH_DTYPE(a->dtype, binary_t, op, a, b, c, st);
}

int32_t tnb200_unary(int32_t op, const tnb200_tensor_t* a, const tnb200_tensor_t* c, void* stream) {
  TNB_REQUIRE(valid_tensor(a) && valid_tensor(c), TNB200_ERR_INVALID, "unary: invalid tensor descriptor");
  TNB_REQUIRE(a->ndim == c->ndim, TNB200_ERR_INVALID, "unary: rank mismatch");
  TNB_REQUIRE(op >= TNB200_CONJ && op <= TNB200_IMAG, TNB200_ERR_INVALID, "unary: bad op %d", op);
  TNB_REQUIRE(a->dtype != TNB200_BOOL && c->dtype != TNB200_BOOL, TNB200_ERR_DTYPE, "unary: bool tensors are not supported");
  cudaStream_t st = (cudaStream_t)stream;
  bool to_real = (op == TNB200_ABS || op == TNB200_REAL || op == TNB200_IMAG) && dtype_is_complex(a->dtype);
  if (to_real) {
    TNB_REQUIRE(c->dtype == real_dtype(a->dtype), TNB200_ERR_DTYPE, "unary: abs/real/imag of complex needs a real output");
    if (a->dtype == TNB200_C64) return unary_tt<cuFloatComplex, float>(op, a, c, st);
    return unary_tt<cuDoubleComplex, double>(op, a, c, st);
  }
  TNB_REQUIRE(a->dtype == c->dtype, TNB200_ERR_DTYPE, "unary: dtype mismatch");
  if (a->dtype >= TNB200_I32)
    TNB_REQUIRE(op == TNB200_CONJ || op == TNB200_ABS || op == TNB200_NEG || op == TNB200_SIGN || op == TNB200_REAL,
                TNB200_ERR_UNSUPPORTED, "unary: op %d on integer tensors is not supported", op);
  TNB_DISPATCH_DTYPE(a->dtype, unary_t, op, a, c, st);
}

int32_t tnb200_affine_inplace(const tnb200_tensor_t* x, double ar, double ai, double br, double bi, void* stream) {
  TNB_REQUIRE(valid_tensor(x), TNB200_ERR_INVALID, "affine: invalid tensor descriptor");
  TNB_DISPATCH_DTYPE(x->dtype, affine_t, x, ZV{ar, ai}, ZV{br, bi}, nullptr, 0, 1, (cudaStream_t)stream);
}

int32_t tnb200_scale_by_device_scalar(const tnb200_tensor_t* x, const void* alpha_dev, int32_t alpha_dtype, int32_t power,
                                      void* stream) {
  TNB_REQUIRE(valid_tensor(x) && alpha_dev, TNB200_ERR_INVALID, "scale: invalid arguments");
  TNB_REQUIRE(alpha_dtype >= TNB200_F64 && alpha_dtype <= TNB200_C128, TNB200_ERR_DTYPE, "scale: scalar must be floating");
  TNB_DISPATCH_DTYPE(x->dtype, affine_t, x, ZV{1.0, 0.0}, ZV{0.0, 0.0}, alpha_dev, alpha_dtype, power, (cudaStream_t)stream);
}

int32_t tnb200_axpy(const tnb200_tensor_t* x, const tnb200_tensor_t* y, double ar, double ai, const void* alpha_dev, double sign,
                    void* stream) {
  TNB_REQUIRE(valid_tensor(x) && valid_tensor(y) && x->ndim == y->ndim, TNB200_ERR_INVALID, "axpy: invalid tensors");
  TNB_REQUIRE(x->dtype == y->dtype, TNB200_ERR_DTYPE, "axpy: dtype mismatch");
  TNB_DISPATCH_DTYPE(x->dtype, axpy_t, x, y, ZV{ar, ai}, alpha_dev, sign, (cudaStream_t)stream);
}

int32_t tnb200_fill(const tnb200_tensor_t* c, double re, double im, void* stream) {
  TNB_REQUIRE(valid_tensor(c), TNB200_ERR_INVALID, "fill: invalid tensor descriptor");
  TNB_DISPATCH_DTYPE(c->dtype, fill_t, c, ZV{re, im}, (cudaStream_t)stream);
}

int32_t tnb200_eye(const tnb200_tensor_t* c, int64_t k, void* stream) {
  TNB_REQUIRE(valid_tensor(c) && c->ndim == 2, TNB200_ERR_INVALID, "eye: output must be a matrix");
  TNB_DISPATCH_DTYPE(c->dtype, diag_t, nullptr, c, k, (cudaStream_t)stream);
}

int32_t tnb200_diagflat(const tnb200_tensor_t* a, const tnb200_tensor_t* c, int64_t k, void* stream) {
  TNB_REQUIRE(valid_tensor(a) && valid_tensor(c) && c->ndim == 2, TNB200_ERR_INVALID, "diagflat: invalid tensors");
  TNB_REQUIRE(a->dtype == c->dtype, TNB200_ERR_DTYPE, "diagflat: dtype mismatch");
  int64_t n = numel(a) + (k < 0 ? -k : k);
  TNB_REQUIRE(c->shape[0] == n && c->shape[1] == n, TNB200_ERR_INVALID, "diagflat: output must be %lld x %lld", (long long)n, (long long)n);
  TNB_DISPATCH_DTYPE(a->dtype, diag_t, a, c, k, (cudaStream_t)stream);
}

int32_t tnb200_randn(const tnb200_tensor_t* c, uint64_t seed, void* stream) {
  TNB_REQUIRE(valid_tensor(c), TNB200_ERR_INVALID, "randn: invalid tensor descriptor");
  TNB_REQUIRE(c->dtype <= TNB200_C128, TNB200_ERR_DTYPE, "randn: floating dtypes only");
  TNB_DISPATCH_DTYPE(c->dtype, random_t, c, seed, 1, 0.0, 1.0, (cudaStream_t)stream);
}
int32_t tnb200_uniform(const tnb200_tensor_t* c, double lo, double hi, uint64_t seed, void* stream) {
  TNB_REQUIRE(valid_tensor(c), TNB200_ERR_INVALID, "uniform: invalid tensor descriptor");
  TNB_REQUIRE(c->dtype <= TNB200_C128, TNB200_ERR_DTYPE, "uniform: floating dtypes only");
  TNB_DISPATCH_DTYPE(c->dtype, random_t, c, seed, 0, lo, hi, (cudaStream_t)stream);
}

int32_t tnb200_norm(const tnb200_tensor_t* a, void* out, void* stream) {
  TNB_REQUIRE(valid_tensor(a) && out, TNB200_ERR_INVALID, "norm: invalid arguments");
  TNB_REQUIRE(a->dtype <= TNB200_C128, TNB200_ERR_DTYPE, "norm: floating dtypes only");
  TNB_DISPATCH_DTYPE(a->dtype, reduce_t, a, nullptr, 0, 0, out, real_dtype(a->dtype), (cudaStream_t)stream);
}

int32_t tnb200_dot(const tnb200_tensor_t* x, const tnb200_tensor_t* y, int32_t conj_x, void* out, void* stream) {
  TNB_REQUIRE(valid_tensor(x) && valid_tensor(y) && out && x->ndim == y->ndim, TNB200_ERR_INVALID, "dot: invalid arguments");
  TNB_REQUIRE(x->dtype == y->dtype, TNB200_ERR_DTYPE, "dot: dtype mismatch");
  TNB_DISPATCH_DTYPE(x->dtype, reduce_t, x, y, 1, conj_x, out, x->dtype, (cudaStream_t)stream);
}

int32_t tnb200_sum(const tnb200_tensor_t* a, const tnb200_tensor_t* c, int32_t naxes, const int32_t* axes, void* stream) {
  TNB_REQUIRE(valid_tensor(a) && valid_tensor(c), TNB200_ERR_INVALID, "sum: invalid tensor descriptor");
  TNB_REQUIRE(a->dtype == c->dtype, TNB200_ERR_DTYPE, "sum: dtype mismatch");
  bool red[TNB200_MAX_NDIM] = {false};
  for (int i = 0; i < naxes; ++i) {
    int x = axes[i] < 0 ? axes[i] + a->ndim : axes[i];
    TNB_REQUIRE(x >= 0 && x < a->ndim && !red[x], TNB200_ERR_INVALID, "sum: bad axis");
    red[x] = true;
  }
  TNB_REQUIRE(c->ndim == a->ndim - naxes, TNB200_ERR_INVALID, "sum: output rank mismatch");
  ModeList keep, rm;
  int ca = 0;
  for (int i = 0; i < a->ndim; ++i) {
    if (red[i]) rm.push(a->shape[i], a->stride[i]);
    else {
      TNB_REQUIRE(c->shape[ca] == a->shape[i], TNB200_ERR_INVALID, "sum: output shape mismatch");
      keep.push(a->shape[i], a->stride[i], c->stride[ca]); ++ca;
    }
  }
  merge_modes(keep, 2); merge_modes(rm, 1);
  TNB_DISPATCH_DTYPE(a->dtype, sum_axes_t, a->data, c->data, keep, rm, 0, (cudaStream_t)stream);
}

int32_t tnb200_gather(const void* src, const int64_t* idx_dev, void* dst, int64_t n, int32_t dtype, int32_t scatter, void* stream) {
  TNB_REQUIRE(n >= 0 && (n == 0 || (src && idx_dev && dst)), TNB200_ERR_INVALID, "gather: invalid arguments");
  TNB_DISPATCH_DTYPE(dtype, gather_t, src, idx_dev, dst, n, scatter, (cudaStream_t)stream);
}

int32_t tnb200_trace(const tnb200_tensor_t* a, const tnb200_tensor_t* c, int64_t offset, int32_t axis1, int32_t axis2, void* stream) {
  TNB_REQUIRE(valid_tensor(a) && valid_tensor(c) && a->ndim >= 2, TNB200_ERR_INVALID, "trace: invalid tensor descriptor");
  TNB_REQUIRE(a->dtype == c->dtype, TNB200_ERR_DTYPE, "trace: dtype mismatch");
  if (axis1 < 0) axis1 += a->ndim;
  if (axis2 < 0) axis2 += a->ndim;
  TNB_REQUIRE(axis1 >= 0 && axis1 < a->ndim && axis2 >= 0 && axis2 < a->ndim && axis1 != axis2, TNB200_ERR_INVALID, "trace: bad axes");
  TNB_REQUIRE(c->ndim == a->ndim - 2, TNB200_ERR_INVALID, "trace: output rank mismatch");
  int64_t n1 = a->shape[axis1], n2 = a->shape[axis2];
  int64_t r0 = offset < 0 ? -offset : 0, c0 = offset > 0 ? offset : 0;
  int64_t len = 0;
  if (r0 < n1 && c0 < n2) len = (n1 - r0) < (n2 - c0) ? (n1 - r0) : (n2 - c0);
  ModeList keep, rm;
  int ca = 0;
  for (int i = 0; i < a->ndim; ++i) {
    if (i == axis1 || i == axis2) continue;
    TNB_REQUIRE(c->shape[ca] == a->shape[i], TNB200_ERR_INVALID, "trace: output shape mismatch");
    keep.push(a->shape[i], a->stride[i], c->stride[ca]); ++ca;
  }
  if (len == 0) return tnb200_fill(c, 0.0, 0.0, stream);
  rm.push(len, a->stride[axis1] + a->stride[axis2]);
  int64_t base = r0 * a->stride[axis1] + c0 * a->stride[axis2];
  merge_modes(keep, 2);
  TNB_DISPATCH_DTYPE(a->dtype, sum_axes_t, a->data, c->data, keep, rm, base, (cudaStream_t)stream);
}

int32_t tnb200_compare(int32_t op, const tnb200_tensor_t* a, const tnb200_tensor_t* b, const tnb200_tensor_t* c, void* stream) {
  TNB_REQUIRE(valid_tensor(a) && valid_tensor(b) && valid_tensor(c), TNB200_ERR_INVALID, "compare: invalid tensor descriptor");
  TNB_REQUIRE(a->ndim == b->ndim && a->ndim == c->ndim, TNB200_ERR_INVALID, "compare: rank mismatch");
  TNB_REQUIRE(op >= TNB200_LT && op <= TNB200_GE, TNB200_ERR_INVALID, "compare: bad op %d", op);
  TNB_REQUIRE(a->dtype == b->dtype, TNB200_ERR_DTYPE, "compare: dtype mismatch");
  TNB_REQUIRE(c->dtype == TNB200_BOOL, TNB200_ERR_DTYPE, "compare: the output must be bool");
  cudaStream_t st = (cudaStream_t)stream;
  switch (a->dtype) {
    case TNB200_F64: return compare_t<double>(op, a, b, c, st);
    case TNB200_F32: return compare_t<float>(op, a, b, c, st);
    case TNB200_F16: return compare_t<__half>(op, a, b, c, st);
    case TNB200_BF16: return compare_t<__nv_bfloat16>(op, a, b, c, st);
    case TNB200_I32: return compare_t<int32_t>(op, a, b, c, st);
    case TNB200_I64: return compare_t<long long>(op, a, b, c, st);
    default: set_error("compare: dtype %s has no order", dtype_name(a->dtype)); return TNB200_ERR_DTYPE;
  }
}

int32_t tnb200_masked_fill(const tnb200_tensor_t* src, const tnb200_tensor_t* mask, const tnb200_tensor_t* out, double re, double im,
                           const void* value_dev, int32_t value_dtype, void* stream) {
  TNB_REQUIRE(valid_tensor(src) && valid_tensor(mask) && valid_tensor(out), TNB200_ERR_INVALID, "masked_fill: invalid tensor descriptor");
  TNB_REQUIRE(src->ndim == mask->ndim && src->ndim == out->ndim, TNB200_ERR_INVALID, "masked_fill: rank mismatch");
  TNB_REQUIRE(mask->dtype == TNB200_BOOL, TNB200_ERR_DTYPE, "masked_fill: the mask must be bool");
  TNB_REQUIRE(src->dtype == out->dtype, TNB200_ERR_DTYPE, "masked_fill: dtype mismatch");
  TNB_REQUIRE(!value_dev || (value_dtype >= TNB200_F64 && value_dtype <= TNB200_BOOL), TNB200_ERR_DTYPE, "masked_fill: bad value dtype");
  cudaStream_t st = (cudaStream_t)stream;
  const ZV v{re, im};
  if (src->dtype == TNB200_BOOL) return masked_fill_t<bool>(src, mask, out, v, value_dev, value_dtype, st);
  TNB_DISPATCH_DTYPE(src->dtype, masked_fill_t, src, mask, out, v, value_dev, value_dtype, st);
}

}  // extern "C"
