// inv.cu — tnb200_inv: the inverse of a square matrix, np.linalg.inv semantics (NumPyBackend.inv,
// backends/numpy/numpy_backend.py:554-558; LAPACK getrf + getri there), by Gauss-Jordan elimination with partial pivoting
// on the augmented matrix [A | I].
//
// The matrix is copied once into row-major n x 2n working storage of the wide type (f64 / c128; f32 and c64 inputs are
// eliminated in double and rounded back).  Step k is two launches:
//   inv_pivot_kernel  one CTA: the pivot row p = argmax_{i >= k} |M[i][k]| (first maximum, like LAPACK's i?amax), swap rows
//                     k and p, divide row k by the pivot, save the multipliers f[i] = M[i][k] (f[k] = 0)
//   inv_elim_kernel   M[i][c] -= f[i] M[k][c] for every row i != k and column c > k (a rank-1 update)
// An exactly zero pivot is singularity: the first such step k writes k + 1 to the device info word and every later launch
// returns at once.  The caller reads that word once (np.linalg.LinAlgError("Singular matrix") when it is not 0).
// The working matrix of n = 2048 in f64 (64 MiB) stays resident in the 126 MB L2 of a B200, so the rank-1 updates run at
// L2 bandwidth; a blocked variant whose trailing update goes through tnb200_tensordot is the next step for larger n.
#include "common.cuh"
#include "cplx.cuh"
#include <math.h>

namespace tnb {

int copy_strided(const tnb200_tensor_t* src, const tnb200_tensor_t* dst, int conj, cudaStream_t st);

template <typename T>
__global__ void inv_init_kernel(T* __restrict__ M, int64_t n, int32_t* info) {
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < n * n; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = idx / n, j = idx % n;
    M[i * 2 * n + n + j] = i == j ? one_<T>() : zero_<T>();
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) *info = 0;
}

template <typename T>
__global__ void __launch_bounds__(1024) inv_pivot_kernel(T* __restrict__ M, int64_t n, int64_t k, T* __restrict__ f, int32_t* info) {
  __shared__ double bv[32];
  __shared__ int64_t bi[32];
  __shared__ T piv_s;
  if (*info) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  const int64_t ld = 2 * n;
  double best = -1.0;
  int64_t besti = n;
  for (int64_t i = k + tid; i < n; i += blockDim.x) {
    const double v = ab2(M[i * ld + k]);
    if (v > best) { best = v; besti = i; }         // ascending i per thread: the first maximum wins
  }
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int64_t oi = __shfl_xor_sync(0xffffffffu, besti, o);
    if (ov > best || (ov == best && oi < besti)) { best = ov; besti = oi; }
  }
  if (lane == 0) { bv[warp] = best; bi[warp] = besti; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < nw; ++w)
      if (bv[w] > bv[0] || (bv[w] == bv[0] && bi[w] < bi[0])) { bv[0] = bv[w]; bi[0] = bi[w]; }
  }
  __syncthreads();
  if (!(bv[0] > 0.0)) {
    if (tid == 0) *info = (int32_t)(k + 1);
    return;
  }
  const int64_t p = bi[0];
  if (p != k)
    for (int64_t c = k + tid; c < ld; c += blockDim.x) {
      const T t = M[k * ld + c]; M[k * ld + c] = M[p * ld + c]; M[p * ld + c] = t;
    }
  __syncthreads();
  if (tid == 0) piv_s = M[k * ld + k];
  __syncthreads();
  const T piv = piv_s;
  for (int64_t c = k + tid; c < ld; c += blockDim.x) M[k * ld + c] = divz(M[k * ld + c], piv);
  for (int64_t i = tid; i < n; i += blockDim.x) f[i] = i == k ? zero_<T>() : M[i * ld + k];
}

template <typename T>
__global__ void inv_elim_kernel(T* __restrict__ M, int64_t n, int64_t k, const T* __restrict__ f, const int32_t* info) {
  if (*info) return;
  const int64_t ld = 2 * n, w = ld - k - 1;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < n * w; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = idx / w, c = k + 1 + idx % w;
    if (i == k) continue;
    const T fi = f[i];
    T x = M[i * ld + c];
    fmacc(x, mulr(fi, -1.0), M[k * ld + c]);
    M[i * ld + c] = x;
  }
}

template <typename T>
static int inv_t(const tnb200_tensor_t* a, const tnb200_tensor_t* out, int wide, int32_t* info, cudaStream_t st) {
  const int64_t n = a->shape[0];
  T *M = nullptr, *f = nullptr;
  int rc;
  if ((rc = ws_alloc((void**)&M, sizeof(T) * (size_t)(2 * n * n), st))) return rc;
  if ((rc = ws_alloc((void**)&f, sizeof(T) * (size_t)n, st))) return rc;
  tnb200_tensor_t left;
  left.data = M; left.dtype = wide; left.ndim = 2;
  left.shape[0] = n; left.shape[1] = n; left.stride[0] = 2 * n; left.stride[1] = 1;
  if ((rc = copy_strided(a, &left, 0, st))) return rc;
  const int64_t cap = 8 * (int64_t)num_sms();
  const unsigned g0 = (unsigned)((n * n + 255) / 256 < cap ? (n * n + 255) / 256 : cap);
  inv_init_kernel<T><<<g0, 256, 0, st>>>(M, n, info);
  count_launch();
  for (int64_t k = 0; k < n; ++k) {
    const int64_t work = n * (2 * n - k - 1);
    const unsigned g = (unsigned)((work + 255) / 256 < cap ? (work + 255) / 256 : cap);
    inv_pivot_kernel<T><<<1, 1024, 0, st>>>(M, n, k, f, info);
    inv_elim_kernel<T><<<g > 0 ? g : 1, 256, 0, st>>>(M, n, k, f, info);
  }
  count_launch((int)(2 * n));
  TNB_LAUNCH_CHECK();
  tnb200_tensor_t right = left;
  right.data = M + n;
  rc = copy_strided(&right, out, 0, st);
  ws_free(M, st); ws_free(f, st);
  return rc;
}

}  // namespace tnb

using namespace tnb;

extern "C" int32_t tnb200_inv(const tnb200_tensor_t* a, const tnb200_tensor_t* out, int32_t* info_dev, void* stream) {
  TNB_REQUIRE(valid_tensor(a) && valid_tensor(out) && info_dev, TNB200_ERR_INVALID, "inv: invalid arguments");
  TNB_REQUIRE(a->ndim == 2 && a->shape[0] == a->shape[1], TNB200_ERR_INVALID, "inv: expects a square matrix");
  TNB_REQUIRE(out->ndim == 2 && out->shape[0] == a->shape[0] && out->shape[1] == a->shape[1], TNB200_ERR_INVALID,
              "inv: output must have the shape of the input");
  const int dt = a->dtype;
  TNB_REQUIRE(dt == TNB200_F64 || dt == TNB200_F32 || dt == TNB200_C64 || dt == TNB200_C128, TNB200_ERR_DTYPE,
              "inv: dtype %s is not supported (f32/f64/c64/c128)", dtype_name(dt));
  TNB_REQUIRE(out->dtype == dt, TNB200_ERR_DTYPE, "inv: output dtype must equal the input dtype");
  TNB_REQUIRE(a->shape[0] < (1LL << 31), TNB200_ERR_UNSUPPORTED, "inv: matrix too large");
  cudaStream_t st = (cudaStream_t)stream;
  set_kernel_name("inv_gauss_jordan");
  if (a->shape[0] == 0) {
    TNB_CHECK_CUDA(cudaMemsetAsync(info_dev, 0, sizeof(int32_t), st));
    return 0;
  }
  if (dtype_is_complex(dt)) return inv_t<zd>(a, out, TNB200_C128, info_dev, st);
  return inv_t<double>(a, out, TNB200_F64, info_dev, st);
}
