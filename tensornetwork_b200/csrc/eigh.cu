// eigh.cu — tnb200_eigh: eigenvalues and eigenvectors of Hermitian matrices, np.linalg.eigh (UPLO='L') semantics
// (NumPyBackend.eigh, backends/numpy/numpy_backend.py:165-166), by cyclic two-sided Jacobi.
//
// The input stack is copied once into contiguous working storage of the wide type (f64 / c128; f32 and c64 inputs
// iterate in double like the SVD).  Only the lower triangle is read and the imaginary part of the diagonal is ignored.
// Convergence is the largest off-diagonal element relative to ||A||_F (Frobenius norm of the Hermitian matrix the lower
// triangle defines, computed on the device): the `scale` measure of the shared Jacobi code (jacobi.cuh).
//
//   n <= EIGH_SMALL_N (64): one CTA per matrix, the whole stack in ONE launch, matrix and rotation in shared memory
//                           (2 x 64 x 65 x 16 B = 133 KB for complex: the shared-memory budget sets the limit).
//   larger n:               blocked two-sided Jacobi on the round-robin block-pair tournament of svd.cu, SB = 16.
//                           Per round: gather A[P,P] of every pair P, diagonalise it in shared memory (svd_eig_kernel),
//                           apply the pair rotations to the columns of A and V (svd_update_kernel), then to the rows of
//                           A (eigh_rowupdate_kernel).  Pairs are disjoint, so a round is one similarity transform.
//                           A fixed number of sweeps is enqueued; a one-thread kernel ends each sweep and sets a device
//                           flag on convergence, after which every remaining launch returns at once.  No host sync.
// Eigenvalues come out ascending (signed), eigenvectors as the columns of v.  info_dev (int32[4], may be NULL):
// [0] the largest number of sweeps any matrix used, [1] 1 if every matrix converged.
#include "common.cuh"
#include "cplx.cuh"
#include "jacobi.cuh"
#include <math.h>

namespace tnb {

int copy_strided(const tnb200_tensor_t* src, const tnb200_tensor_t* dst, int conj, cudaStream_t st);

constexpr int EIGH_SMALL_SB = 32, EIGH_SMALL_N = 2 * EIGH_SMALL_SB;
constexpr int EIGH_SB = 16, EIGH_PB = 2 * EIGH_SB;
constexpr int EIGH_MAX_SWEEPS = 30;

__host__ __device__ inline double eigh_tol(int64_t n) { return 4.0 * sqrt((double)n) * 2.220446049250313e-16; }

// element (i, j) of the Hermitian matrix defined by the lower triangle of the row-major n x n matrix a
template <typename T>
__device__ __forceinline__ T herm_at(const T* a, int64_t n, int64_t i, int64_t j) {
  if (i > j) return a[i * n + j];
  if (i < j) return cj(a[j * n + i]);
  return mk(re_(a[i * n + i]), 0.0, (T*)nullptr);
}
// ||herm(a)||_F^2 contribution of element (i, j), i >= j
template <typename T>
__device__ __forceinline__ double herm_sq(const T* a, int64_t n, int64_t i, int64_t j) {
  return i == j ? re_(a[i * n + i]) * re_(a[i * n + i]) : 2.0 * ab2(a[i * n + j]);
}

// deterministic block sum (any blockDim multiple of 32, <= 1024); red: 32 doubles of shared memory
__device__ double eigh_block_sum(double v, double* red) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (lane == 0) red[warp] = v;
  __syncthreads();
  if (warp == 0) {
    v = lane < nw ? red[lane] : 0.0;
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[0] = v;
  }
  __syncthreads();
  const double r = red[0];
  __syncthreads();
  return r;
}

__global__ void eigh_info_init_kernel(int32_t* info) {
  info[0] = 0; info[1] = 1; info[2] = 0; info[3] = 0;
}

// ---------------------------------------------------------------------------------------------- small path
// One CTA per matrix.  Dynamic shared memory: the eig_smem_bytes<T, 32> layout of svd_eig_kernel.
template <typename T>
__global__ void __launch_bounds__(256) eigh_small_kernel(const T* __restrict__ A, int n, double* __restrict__ W, T* __restrict__ V,
                                                         int32_t* info) {
  constexpr int SB = EIGH_SMALL_SB, PB = 2 * SB, LD = PB + 1;
  extern __shared__ __align__(16) unsigned char es_smem[];
  T* g = reinterpret_cast<T*>(es_smem);
  T* rm = g + PB * LD;
  double* cs = reinterpret_cast<double*>(rm + PB * LD);
  double* sn = cs + SB;
  T* ph = reinterpret_cast<T*>(sn + SB);
  int* pp = reinterpret_cast<int*>(ph + SB);
  int* qq = pp + SB;
  __shared__ float red[8];
  __shared__ float offmax;
  __shared__ double dred[32];
  __shared__ double lam[PB];
  __shared__ int rank[PB];
  const int tid = threadIdx.x;
  const T* a = A + (int64_t)blockIdx.x * n * n;
  double acc = 0.0;
  for (int idx = tid; idx < n * n; idx += blockDim.x) {
    const int i = idx / n, j = idx % n;
    if (i >= j) acc += herm_sq(a, n, i, j);
  }
  const double fro = sqrt(eigh_block_sum(acc, dred));
  for (int idx = tid; idx < PB * PB; idx += blockDim.x) {
    const int i = idx / PB, j = idx % PB;
    g[i * LD + j] = i < n && j < n ? herm_at(a, n, i, j) : zero_<T>();     // padding indices stay decoupled
    rm[i * LD + j] = i == j ? one_<T>() : zero_<T>();
  }
  __syncthreads();
  const int max_sweeps = 40;
  const int sweeps = herm_jacobi_smem<T, SB>(g, rm, cs, sn, ph, pp, qq, red, offmax, nullptr, eigh_tol(n), max_sweeps, fro);
  for (int j = tid; j < n; j += blockDim.x) lam[j] = re_(g[j * LD + j]);
  __syncthreads();
  for (int j = tid; j < n; j += blockDim.x) {
    int r = 0;
    const double lj = lam[j];
    for (int i = 0; i < n; ++i) r += (lam[i] < lj) || (lam[i] == lj && i < j);
    rank[j] = r;
    W[(int64_t)blockIdx.x * n + r] = lj;
  }
  __syncthreads();
  T* v = V + (int64_t)blockIdx.x * n * n;
  for (int idx = tid; idx < n * n; idx += blockDim.x) {
    const int i = idx / n, j = idx % n;
    v[(int64_t)i * n + rank[j]] = rm[i * LD + j];
  }
  if (tid == 0 && info) {
    atomicMax(&info[0], sweeps);
    if (sweeps >= max_sweeps) atomicAnd(&info[1], 0);
  }
}

// ---------------------------------------------------------------------------------------------- large path
// ||herm(a)||_F into *out (one CTA: deterministic)
template <typename T>
__global__ void __launch_bounds__(1024) eigh_fro_kernel(const T* __restrict__ a, int64_t n, double* out) {
  __shared__ double red[32];
  double acc = 0.0;
  for (int64_t idx = threadIdx.x; idx < n * n; idx += blockDim.x) {
    const int64_t i = idx / n, j = idx % n;
    if (i >= j) acc += herm_sq(a, n, i, j);
  }
  acc = eigh_block_sum(acc, red);
  if (threadIdx.x == 0) *out = sqrt(acc);
}
// column-major Cp x Cp working matrices: X = herm(a) (zero padding), V = I
template <typename T>
__global__ void eigh_prep_kernel(const T* __restrict__ a, int64_t n, int64_t Cp, T* __restrict__ X, T* __restrict__ V) {
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < Cp * Cp; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t c = idx / Cp, r = idx % Cp;
    X[idx] = r < n && c < n ? herm_at(a, n, r, c) : zero_<T>();
    V[idx] = r == c ? one_<T>() : zero_<T>();
  }
}
// G[pair] (row-major PB x PB) = X[P, P] of every pair P of the round
template <typename T>
__global__ void __launch_bounds__(256) eigh_gather_kernel(const T* __restrict__ X, int64_t ld, int nb, int round, T* __restrict__ G,
                                                          const int* skip) {
  if (*skip) return;
  int bi, bj;
  rr_pair(nb, round, blockIdx.x, bi, bj);
  T* g = G + (int64_t)blockIdx.x * EIGH_PB * EIGH_PB;
  for (int idx = threadIdx.x; idx < EIGH_PB * EIGH_PB; idx += blockDim.x) {
    const int i = idx / EIGH_PB, j = idx % EIGH_PB;
    g[idx] = X[(int64_t)pair_col<EIGH_SB>(bi, bj, j) * ld + pair_col<EIGH_SB>(bi, bj, i)];
  }
}
// X[P rows, :] <- R^H X[P rows, :] for every pair P of the round (X column-major, ld rows, `cols` columns)
template <typename T>
__global__ void __launch_bounds__(256) eigh_rowupdate_kernel(T* __restrict__ X, int64_t ld, int64_t cols, int nb, int round,
                                                             const T* __restrict__ Rm, const int* skip) {
  constexpr int PB = EIGH_PB, CT = 256 / PB;            // CT columns per tile, one output per thread
  __shared__ T rs[PB][PB + 1];
  __shared__ T tile[CT][PB + 1];
  if (*skip) return;
  int bi, bj;
  rr_pair(nb, round, blockIdx.x, bi, bj);
  const T* rg = Rm + (int64_t)blockIdx.x * PB * PB;
  for (int idx = threadIdx.x; idx < PB * PB; idx += 256) rs[idx / PB][idx % PB] = rg[idx];
  const int k = threadIdx.x % PB, cl = threadIdx.x / PB;
  const int64_t row = pair_col<EIGH_SB>(bi, bj, k);
  for (int64_t cb = (int64_t)blockIdx.y * CT; cb < cols; cb += (int64_t)gridDim.y * CT) {
    const int64_t c = cb + cl;
    __syncthreads();
    tile[cl][k] = c < cols ? X[c * ld + row] : zero_<T>();
    __syncthreads();
    T out = zero_<T>();
#pragma unroll 8
    for (int j = 0; j < PB; ++j) fmacc(out, cj(rs[j][k]), tile[cl][j]);
    if (c < cols) X[c * ld + row] = out;
  }
}
// end of a sweep: count it and raise the done flag once no pair exceeded the tolerance
__global__ void eigh_sweep_kernel(const unsigned int* conv, double tol, int* state) {
  if (state[0]) return;
  state[1] += 1;
  if ((double)__uint_as_float(*conv) <= tol) state[0] = 1;
}
// ascending signed rank of the eigenvalues diag(X); W[rank] = lambda
template <typename T>
__global__ void eigh_rank_kernel(const T* __restrict__ X, int64_t ld, int n, double* __restrict__ W, int* __restrict__ rank,
                                 const int* state, int32_t* info) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j == 0 && info) {
    atomicMax(&info[0], state[1]);
    if (!state[0]) atomicAnd(&info[1], 0);
  }
  if (j >= n) return;
  const double lj = re_(X[(int64_t)j * ld + j]);
  int r = 0;
  for (int i = 0; i < n; ++i) {
    const double li = re_(X[(int64_t)i * ld + i]);
    r += (li < lj) || (li == lj && i < j);
  }
  rank[j] = r;
  W[r] = lj;
}
// row-major n x n eigenvector output: Vout[i][rank[j]] = V[i][j]  (V column-major, ld rows)
template <typename T>
__global__ void eigh_vectors_kernel(const T* __restrict__ V, int64_t ld, int n, const int* __restrict__ rank, T* __restrict__ Vout) {
  const int j = blockIdx.x;
  const int k = rank[j];
  for (int i = threadIdx.x; i < n; i += blockDim.x) Vout[(int64_t)i * n + k] = V[(int64_t)j * ld + i];
}

template <typename T>
static int eigh_large(const T* a, int64_t n, double* W, T* Vout, int32_t* info, cudaStream_t st) {
  constexpr int SB = EIGH_SB, PB = EIGH_PB, RT = Geo<SB>::RT;
  const int64_t Cp = (n + PB - 1) / PB * PB;
  const int nb = (int)(Cp / SB), npairs = nb / 2, rounds = nb - 1;
  T *X = nullptr, *V = nullptr, *G = nullptr, *Rm = nullptr;
  double* fro = nullptr;
  int* rank = nullptr;
  int* state = nullptr;
  unsigned int* conv = nullptr;
  int rc;
  if ((rc = ws_alloc((void**)&X, sizeof(T) * (size_t)(Cp * Cp), st))) return rc;
  if ((rc = ws_alloc((void**)&V, sizeof(T) * (size_t)(Cp * Cp), st))) return rc;
  if ((rc = ws_alloc((void**)&G, sizeof(T) * (size_t)npairs * PB * PB, st))) return rc;
  if ((rc = ws_alloc((void**)&Rm, sizeof(T) * (size_t)npairs * PB * PB, st))) return rc;
  if ((rc = ws_alloc((void**)&fro, sizeof(double), st))) return rc;
  if ((rc = ws_alloc((void**)&rank, sizeof(int) * (size_t)n, st))) return rc;
  if ((rc = ws_alloc((void**)&state, sizeof(int) * 2, st))) return rc;
  if ((rc = ws_alloc((void**)&conv, sizeof(unsigned int) * EIGH_MAX_SWEEPS, st))) return rc;
  TNB_CHECK_CUDA(cudaMemsetAsync(state, 0, sizeof(int) * 2, st));
  TNB_CHECK_CUDA(cudaMemsetAsync(conv, 0, sizeof(unsigned int) * EIGH_MAX_SWEEPS, st));
  const size_t eig_bytes = eig_smem_bytes<T, SB>();
  {
    static bool attr_done = false;      // per T
    if (!attr_done) {
      TNB_CHECK_CUDA(cudaFuncSetAttribute(svd_eig_kernel<T, SB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)eig_bytes));
      attr_done = true;
    }
  }
  eigh_fro_kernel<T><<<1, 1024, 0, st>>>(a, n, fro);
  const unsigned pgrid = (unsigned)((Cp * Cp + 255) / 256 < 4 * num_sms() ? (Cp * Cp + 255) / 256 : 4 * num_sms());
  eigh_prep_kernel<T><<<pgrid, 256, 0, st>>>(a, n, Cp, X, V);
  count_launch(2);
  int split = (4 * num_sms() + npairs - 1) / npairs;
  const int usplit = (int)((Cp + RT - 1) / RT) < split ? (int)((Cp + RT - 1) / RT) : split;
  const int csplit = (int)((Cp + 7) / 8) < split ? (int)((Cp + 7) / 8) : split;
  const double tol = eigh_tol(n);
  for (int sw = 0; sw < EIGH_MAX_SWEEPS; ++sw) {
    for (int r = 0; r < rounds; ++r) {
      eigh_gather_kernel<T><<<npairs, 256, 0, st>>>(X, Cp, nb, r, G, state);
      svd_eig_kernel<T, SB><<<npairs, 256, eig_bytes, st>>>(G, Rm, conv + sw, 1e-15, 10, state, fro);
      svd_update_kernel<T, SB><<<dim3(npairs, usplit), 256, 0, st>>>(X, Cp, nb, r, Rm, state);
      svd_update_kernel<T, SB><<<dim3(npairs, usplit), 256, 0, st>>>(V, Cp, nb, r, Rm, state);
      eigh_rowupdate_kernel<T><<<dim3(npairs, csplit), 256, 0, st>>>(X, Cp, Cp, nb, r, Rm, state);
    }
    eigh_sweep_kernel<<<1, 1, 0, st>>>(conv + sw, tol, state);
    count_launch(5 * rounds + 1);
    TNB_LAUNCH_CHECK();
  }
  eigh_rank_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(X, Cp, (int)n, W, rank, state, info);
  eigh_vectors_kernel<T><<<(unsigned)n, 256, 0, st>>>(V, Cp, (int)n, rank, Vout);
  count_launch(2);
  TNB_LAUNCH_CHECK();
  ws_free(X, st); ws_free(V, st); ws_free(G, st); ws_free(Rm, st); ws_free(fro, st); ws_free(rank, st); ws_free(state, st);
  ws_free(conv, st);
  return 0;
}

template <typename T>
static int eigh_t(const void* a, int64_t batch, int64_t n, double* W, void* V, int32_t* info, cudaStream_t st) {
  if (n <= EIGH_SMALL_N) {
    const size_t smem = eig_smem_bytes<T, EIGH_SMALL_SB>();
    static bool attr_done = false;
    if (!attr_done) {
      TNB_CHECK_CUDA(cudaFuncSetAttribute(eigh_small_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr_done = true;
    }
    set_kernel_name("eigh_small_jacobi");
    eigh_small_kernel<T><<<(unsigned)batch, 256, smem, st>>>((const T*)a, (int)n, W, (T*)V, info);
    TNB_LAUNCH_CHECK();
    count_launch();
    return 0;
  }
  set_kernel_name("eigh_block_jacobi");
  for (int64_t b = 0; b < batch; ++b) {
    int rc = eigh_large<T>((const T*)a + b * n * n, n, W + b * n, (T*)V + b * n * n, info, st);
    if (rc) return rc;
  }
  return 0;
}

}  // namespace tnb

using namespace tnb;

extern "C" int32_t tnb200_eigh(const tnb200_tensor_t* a, const tnb200_tensor_t* w, const tnb200_tensor_t* v, int32_t* info_dev,
                               void* stream) {
  TNB_REQUIRE(valid_tensor(a) && valid_tensor(w) && valid_tensor(v), TNB200_ERR_INVALID, "eigh: invalid tensor descriptor");
  const int nd = a->ndim;
  TNB_REQUIRE(nd >= 2 && a->shape[nd - 1] == a->shape[nd - 2], TNB200_ERR_INVALID, "eigh: expects a stack of square matrices");
  TNB_REQUIRE(v->ndim == nd && w->ndim == nd - 1, TNB200_ERR_INVALID, "eigh: w must be (..., n) and v (..., n, n)");
  for (int i = 0; i < nd; ++i) TNB_REQUIRE(v->shape[i] == a->shape[i], TNB200_ERR_INVALID, "eigh: v must have the shape of a");
  for (int i = 0; i < nd - 1; ++i) TNB_REQUIRE(w->shape[i] == a->shape[i], TNB200_ERR_INVALID, "eigh: w must be (..., n)");
  const int dt = a->dtype;
  TNB_REQUIRE(dt == TNB200_F64 || dt == TNB200_F32 || dt == TNB200_C64 || dt == TNB200_C128, TNB200_ERR_DTYPE,
              "eigh: dtype %s is not supported (f32/f64/c64/c128)", dtype_name(dt));
  const bool cplx = dtype_is_complex(dt), dbl = dt == TNB200_F64 || dt == TNB200_C128;
  TNB_REQUIRE(v->dtype == dt, TNB200_ERR_DTYPE, "eigh: v dtype must equal the input dtype");
  TNB_REQUIRE(w->dtype == (dbl ? TNB200_F64 : TNB200_F32), TNB200_ERR_DTYPE, "eigh: w must have the real dtype of the input");
  const int64_t n = a->shape[nd - 1];
  TNB_REQUIRE(n < (1LL << 31), TNB200_ERR_UNSUPPORTED, "eigh: matrix too large");
  int64_t batch = 1;
  for (int i = 0; i < nd - 2; ++i) batch *= a->shape[i];
  cudaStream_t st = (cudaStream_t)stream;
  if (info_dev) {
    eigh_info_init_kernel<<<1, 1, 0, st>>>(info_dev);
    TNB_LAUNCH_CHECK();
    count_launch();
  }
  if (batch == 0 || n == 0) return 0;
  const int wide = cplx ? TNB200_C128 : TNB200_F64;
  const size_t esz = cplx ? 16 : 8;
  void *da = nullptr, *dv = nullptr;
  double* dw = nullptr;
  int rc;
  if ((rc = ws_alloc(&da, esz * (size_t)(batch * n * n), st))) return rc;
  if ((rc = ws_alloc(&dv, esz * (size_t)(batch * n * n), st))) return rc;
  if ((rc = ws_alloc((void**)&dw, sizeof(double) * (size_t)(batch * n), st))) return rc;
  // contiguous wide views with the caller's shapes
  tnb200_tensor_t ta = *a, tv = *v, tw = *w;
  ta.data = da; ta.dtype = wide; tv.data = dv; tv.dtype = wide; tw.data = dw; tw.dtype = TNB200_F64;
  int64_t s = 1;
  for (int i = nd - 1; i >= 0; --i) { ta.stride[i] = s; tv.stride[i] = s; s *= a->shape[i]; }
  s = 1;
  for (int i = nd - 2; i >= 0; --i) { tw.stride[i] = s; s *= w->shape[i]; }
  rc = copy_strided(a, &ta, 0, st);
  if (rc == 0) rc = cplx ? eigh_t<zd>(da, batch, n, dw, dv, info_dev, st) : eigh_t<double>(da, batch, n, dw, dv, info_dev, st);
  if (rc == 0) rc = copy_strided(&tw, w, 0, st);
  if (rc == 0) rc = copy_strided(&tv, v, 0, st);
  ws_free(da, st); ws_free(dv, st); ws_free(dw, st);
  return rc;
}
