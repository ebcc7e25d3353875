// common.cuh — shared host/device helpers for libtnb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <cuComplex.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <stdarg.h>
#include <atomic>
#include "../../include/tnb200.h"

namespace tnb {

// ---------------------------------------------------------------- error handling
void set_error(const char* fmt, ...);
void set_kernel_name(const char* name);
extern std::atomic<long long> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

#define TNB_CHECK_CUDA(expr)                                                          \
  do {                                                                                \
    cudaError_t _e = (expr);                                                          \
    if (_e != cudaSuccess) {                                                          \
      tnb::set_error("%s:%d CUDA error %s: %s", __FILE__, __LINE__, #expr,            \
                     cudaGetErrorString(_e));                                         \
      return TNB200_ERR_CUDA;                                                         \
    }                                                                                 \
  } while (0)

#define TNB_REQUIRE(cond, code, ...)                                                  \
  do {                                                                                \
    if (!(cond)) {                                                                    \
      tnb::set_error(__VA_ARGS__);                                                    \
      return (code);                                                                  \
    }                                                                                 \
  } while (0)

#define TNB_LAUNCH_CHECK()                                                            \
  do {                                                                                \
    cudaError_t _e = cudaGetLastError();                                              \
    if (_e != cudaSuccess) {                                                          \
      tnb::set_error("%s:%d kernel launch failed: %s", __FILE__, __LINE__,            \
                     cudaGetErrorString(_e));                                         \
      return TNB200_ERR_CUDA;                                                         \
    }                                                                                 \
  } while (0)

// ---------------------------------------------------------------- dtype helpers
inline int dtype_size(int dt) {
  switch (dt) {
    case TNB200_F64: return 8;
    case TNB200_F32: return 4;
    case TNB200_F16: return 2;
    case TNB200_BF16: return 2;
    case TNB200_C64: return 8;
    case TNB200_C128: return 16;
    case TNB200_I32: return 4;
    case TNB200_I64: return 8;
    case TNB200_BOOL: return 1;
  }
  return 0;
}
inline bool dtype_is_complex(int dt) { return dt == TNB200_C64 || dt == TNB200_C128; }
inline const char* dtype_name(int dt) {
  static const char* n[] = {"f64", "f32", "f16", "bf16", "c64", "c128", "i32", "i64", "bool"};
  return (dt >= 0 && dt < 9) ? n[dt] : "?";
}

inline int num_sms() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  return sms;
}

// ------------------------------------------------ device scalar type <-> enum mapping
template <int DT> struct DType;
template <> struct DType<TNB200_F64> { using T = double; using Acc = double; };
template <> struct DType<TNB200_F32> { using T = float; using Acc = float; };
template <> struct DType<TNB200_F16> { using T = __half; using Acc = float; };
template <> struct DType<TNB200_BF16> { using T = __nv_bfloat16; using Acc = float; };
template <> struct DType<TNB200_C64> { using T = cuFloatComplex; using Acc = cuFloatComplex; };
template <> struct DType<TNB200_C128> { using T = cuDoubleComplex; using Acc = cuDoubleComplex; };
template <> struct DType<TNB200_I32> { using T = int32_t; using Acc = int32_t; };
template <> struct DType<TNB200_I64> { using T = long long; using Acc = long long; };

// accumulate-type arithmetic, overloaded so kernels are written once
__host__ __device__ inline double acc_zero(double*) { return 0.0; }
__host__ __device__ inline float acc_zero(float*) { return 0.f; }
__host__ __device__ inline int32_t acc_zero(int32_t*) { return 0; }
__host__ __device__ inline long long acc_zero(long long*) { return 0; }
__host__ __device__ inline cuFloatComplex acc_zero(cuFloatComplex*) { return make_cuFloatComplex(0.f, 0.f); }
__host__ __device__ inline cuDoubleComplex acc_zero(cuDoubleComplex*) { return make_cuDoubleComplex(0.0, 0.0); }

__device__ inline double to_acc(double x) { return x; }
__device__ inline float to_acc(float x) { return x; }
__device__ inline float to_acc(__half x) { return __half2float(x); }
__device__ inline float to_acc(__nv_bfloat16 x) { return __bfloat162float(x); }
__device__ inline cuFloatComplex to_acc(cuFloatComplex x) { return x; }
__device__ inline cuDoubleComplex to_acc(cuDoubleComplex x) { return x; }
__device__ inline int32_t to_acc(int32_t x) { return x; }
__device__ inline long long to_acc(long long x) { return x; }

template <typename T> __device__ inline T from_acc(double x);
template <> __device__ inline double from_acc<double>(double x) { return x; }
template <typename T, typename A> struct FromAcc;
template <> struct FromAcc<double, double> { __device__ static double f(double x) { return x; } };
template <> struct FromAcc<float, float> { __device__ static float f(float x) { return x; } };
template <> struct FromAcc<__half, float> { __device__ static __half f(float x) { return __float2half_rn(x); } };
template <> struct FromAcc<__nv_bfloat16, float> { __device__ static __nv_bfloat16 f(float x) { return __float2bfloat16_rn(x); } };
template <> struct FromAcc<cuFloatComplex, cuFloatComplex> { __device__ static cuFloatComplex f(cuFloatComplex x) { return x; } };
template <> struct FromAcc<cuDoubleComplex, cuDoubleComplex> { __device__ static cuDoubleComplex f(cuDoubleComplex x) { return x; } };
template <> struct FromAcc<int32_t, int32_t> { __device__ static int32_t f(int32_t x) { return x; } };
template <> struct FromAcc<long long, long long> { __device__ static long long f(long long x) { return x; } };

__device__ inline void fma_acc(double& c, double a, double b) { c = fma(a, b, c); }
__device__ inline void fma_acc(float& c, float a, float b) { c = fmaf(a, b, c); }
__device__ inline void fma_acc(int32_t& c, int32_t a, int32_t b) { c += a * b; }
__device__ inline void fma_acc(long long& c, long long a, long long b) { c += a * b; }
__device__ inline void fma_acc(cuFloatComplex& c, cuFloatComplex a, cuFloatComplex b) {
  c.x = fmaf(a.x, b.x, c.x); c.x = fmaf(-a.y, b.y, c.x);
  c.y = fmaf(a.x, b.y, c.y); c.y = fmaf(a.y, b.x, c.y);
}
__device__ inline void fma_acc(cuDoubleComplex& c, cuDoubleComplex a, cuDoubleComplex b) {
  c.x = fma(a.x, b.x, c.x); c.x = fma(-a.y, b.y, c.x);
  c.y = fma(a.x, b.y, c.y); c.y = fma(a.y, b.x, c.y);
}
__device__ inline double conj_acc(double x) { return x; }
__device__ inline float conj_acc(float x) { return x; }
__device__ inline int32_t conj_acc(int32_t x) { return x; }
__device__ inline long long conj_acc(long long x) { return x; }
__device__ inline cuFloatComplex conj_acc(cuFloatComplex x) { return make_cuFloatComplex(x.x, -x.y); }
__device__ inline cuDoubleComplex conj_acc(cuDoubleComplex x) { return make_cuDoubleComplex(x.x, -x.y); }

// ---------------------------------------------------------------- mode lists
// A "mode" is one (possibly merged) tensor axis: extent + element strides in up to 3 operands.
constexpr int kMaxModes = TNB200_MAX_NDIM;
struct ModeList {
  int n = 0;
  int64_t ext[kMaxModes];
  int64_t s0[kMaxModes];  // stride in first operand
  int64_t s1[kMaxModes];  // stride in second operand (0 if not present)
  int64_t s2[kMaxModes];  // stride in third operand
  void push(int64_t e, int64_t a, int64_t b = 0, int64_t c = 0) {
    ext[n] = e; s0[n] = a; s1[n] = b; s2[n] = c; ++n;
  }
  int64_t total() const { int64_t t = 1; for (int i = 0; i < n; ++i) t *= ext[i]; return t; }
};
// drop extent-1 modes and merge adjacent modes that are contiguous in every operand
// (`nops` operands carry meaningful strides).
inline void merge_modes(ModeList& m, int nops) {
  ModeList r;
  for (int i = 0; i < m.n; ++i) {
    if (m.ext[i] == 1) continue;
    if (r.n > 0) {
      int j = r.n - 1;
      bool ok = r.s0[j] == m.ext[i] * m.s0[i];
      if (nops > 1) ok = ok && r.s1[j] == m.ext[i] * m.s1[i];
      if (nops > 2) ok = ok && r.s2[j] == m.ext[i] * m.s2[i];
      if (ok) {
        r.ext[j] *= m.ext[i]; r.s0[j] = m.s0[i]; r.s1[j] = m.s1[i]; r.s2[j] = m.s2[i];
        continue;
      }
    }
    r.push(m.ext[i], m.s0[i], m.s1[i], m.s2[i]);
  }
  m = r;
}

// Device-side compact form (passed by value inside kernel parameter structs).
constexpr int kDevModes = 12;
struct DevModes {
  int n;
  int64_t ext[kDevModes];
  int64_t s0[kDevModes];
  int64_t s1[kDevModes];
  int64_t s2[kDevModes];
};
inline bool to_dev(const ModeList& m, DevModes& d) {
  if (m.n > kDevModes) return false;
  d.n = m.n;
  for (int i = 0; i < kDevModes; ++i) {
    d.ext[i] = i < m.n ? m.ext[i] : 1;
    d.s0[i] = i < m.n ? m.s0[i] : 0;
    d.s1[i] = i < m.n ? m.s1[i] : 0;
    d.s2[i] = i < m.n ? m.s2[i] : 0;
  }
  return true;
}
// linear index over the mode list (row-major, last mode fastest) -> element offsets
__device__ __forceinline__ void mode_offsets(const DevModes& m, int64_t lin, int64_t& o0, int64_t& o1) {
  o0 = 0; o1 = 0;
#pragma unroll 1
  for (int i = m.n - 1; i > 0; --i) {
    int64_t q = lin / m.ext[i];
    int64_t r = lin - q * m.ext[i];
    o0 += r * m.s0[i]; o1 += r * m.s1[i];
    lin = q;
  }
  if (m.n > 0) { o0 += lin * m.s0[0]; o1 += lin * m.s1[0]; }
}
__device__ __forceinline__ void mode_offsets3(const DevModes& m, int64_t lin, int64_t& o0, int64_t& o1, int64_t& o2) {
  o0 = 0; o1 = 0; o2 = 0;
#pragma unroll 1
  for (int i = m.n - 1; i > 0; --i) {
    int64_t q = lin / m.ext[i];
    int64_t r = lin - q * m.ext[i];
    o0 += r * m.s0[i]; o1 += r * m.s1[i]; o2 += r * m.s2[i];
    lin = q;
  }
  if (m.n > 0) { o0 += lin * m.s0[0]; o1 += lin * m.s1[0]; o2 += lin * m.s2[0]; }
}
__device__ __forceinline__ int64_t mode_offset0(const DevModes& m, int64_t lin) {
  int64_t o0 = 0;
#pragma unroll 1
  for (int i = m.n - 1; i > 0; --i) {
    int64_t q = lin / m.ext[i];
    int64_t r = lin - q * m.ext[i];
    o0 += r * m.s0[i];
    lin = q;
  }
  if (m.n > 0) o0 += lin * m.s0[0];
  return o0;
}

inline bool valid_tensor(const tnb200_tensor_t* t) {
  if (!t || t->ndim < 0 || t->ndim > TNB200_MAX_NDIM) return false;
  if (t->dtype < 0 || t->dtype > TNB200_BOOL) return false;
  for (int i = 0; i < t->ndim; ++i) if (t->shape[i] < 0) return false;
  return true;
}
inline int64_t numel(const tnb200_tensor_t* t) {
  int64_t n = 1;
  for (int i = 0; i < t->ndim; ++i) n *= t->shape[i];
  return n;
}

// stream-ordered scratch memory (graph-capturable); pool keeps memory cached.
int ws_alloc(void** p, size_t bytes, cudaStream_t st);
int ws_free(void* p, cudaStream_t st);

}  // namespace tnb
