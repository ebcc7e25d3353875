// krylov.cu — tnb200_krylov_orth: one Arnoldi step's orthogonalisation for the restarted Arnoldi eigensolver
// (tensornetwork_b200/arnoldi.py; NumPyBackend.eigs, backends/numpy/numpy_backend.py:216-291, ARPACK there).
//
// Classical Gram-Schmidt with one reorthogonalisation (CGS2) of w against the first k rows of the basis V ((rows, n),
// row-major contiguous), with no host scalar anywhere:
//   krylov_pass1_kernel   row k <- w; partial h1 = V[:k]^H w over this CTA's chunk of the n entries
//   krylov_pass2_kernel   h1 = sum of the partials (fixed CTA order); x -= V[:k]^T h1 on the chunk; partial h2 = V[:k]^H x
//   krylov_pass3_kernel   h2 likewise; x -= V[:k]^T h2; partial |x|^2
//   krylov_norm_kernel    |x| (fixed order); row k <- x / |x|; h[0..k) = h1 + h2, h[k] = |x|
// Every kernel uses the same grid, so a CTA only ever touches its own chunk of row k; the cross-CTA reductions sum the
// per-CTA partials in CTA order (as qr_apply2_kernel does), so results are bit-reproducible.  A zero |x| (breakdown: w
// lies in the span of V[:k]) leaves row k zero and h[k] = 0, which the host detects in H.
// Arithmetic is in double (f64 / complex double) for every storage type.
#include "common.cuh"
#include "cplx.cuh"
#include <math.h>

namespace tnb {

template <typename S> struct KAcc { using A = double; };
template <> struct KAcc<cuFloatComplex> { using A = zd; };
template <> struct KAcc<cuDoubleComplex> { using A = zd; };
__device__ __forceinline__ double kload(double x) { return x; }
__device__ __forceinline__ double kload(float x) { return (double)x; }
__device__ __forceinline__ zd kload(const cuDoubleComplex& x) { const double* p = reinterpret_cast<const double*>(&x); return zd{p[0], p[1]}; }
__device__ __forceinline__ zd kload(cuFloatComplex x) { return zd{(double)x.x, (double)x.y}; }
__device__ __forceinline__ void kstore(double* p, double v) { *p = v; }
__device__ __forceinline__ void kstore(float* p, double v) { *p = (float)v; }
__device__ __forceinline__ void kstore(cuDoubleComplex* p, zd v) { *p = make_cuDoubleComplex(v.x, v.y); }
__device__ __forceinline__ void kstore(cuFloatComplex* p, zd v) { *p = make_cuFloatComplex((float)v.x, (float)v.y); }
__device__ __forceinline__ double kwarp_sum(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ zd kwarp_sum(zd v) { return zd{kwarp_sum(v.x), kwarp_sum(v.y)}; }

constexpr int KT = 256, KJ = 64;   // threads per CTA; basis rows per shared-memory reduction batch

struct KGeo {
  int64_t n, chunk;                // vector length, entries per CTA
  __device__ int64_t lo() const { return (int64_t)blockIdx.x * chunk; }
  __device__ int64_t hi() const { const int64_t h = lo() + chunk; return h < n ? h : n; }
};

// part[blockIdx.x * k + j] = sum over this CTA's chunk of conj(V[j][i]) x[i], j < k
template <typename S, typename A>
__device__ void chunk_dots(const S* __restrict__ V, const S* x, int k, KGeo g, A* __restrict__ part, A* sred) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t i0 = g.lo(), i1 = g.hi();
  for (int j0 = 0; j0 < k; j0 += KJ) {
    const int jn = k - j0 < KJ ? k - j0 : KJ;
    for (int jj = 0; jj < jn; ++jj) {
      const S* v = V + (int64_t)(j0 + jj) * g.n;
      A acc = mk(0.0, 0.0, (A*)nullptr);
      for (int64_t i = i0 + tid; i < i1; i += KT) fmacc(acc, cj(kload(v[i])), kload(x[i]));
      acc = kwarp_sum(acc);
      if (lane == 0) sred[warp * KJ + jj] = acc;
    }
    __syncthreads();
    if (tid < jn) {
      A s = mk(0.0, 0.0, (A*)nullptr);
      for (int w = 0; w < KT / 32; ++w) s = add(s, sred[w * KJ + tid]);
      part[(int64_t)blockIdx.x * k + j0 + tid] = s;
    }
    __syncthreads();
  }
}
// h[j] = sum over CTAs (in order) of part[c * k + j]; x -= V[:k]^T h over this CTA's chunk
template <typename S, typename A>
__device__ void reduce_and_subtract(const S* __restrict__ V, S* x, int k, KGeo g, const A* __restrict__ part, A* h, A* hsave) {
  for (int j = threadIdx.x; j < k; j += KT) {
    A s = mk(0.0, 0.0, (A*)nullptr);
    for (int c = 0; c < (int)gridDim.x; ++c) s = add(s, part[(int64_t)c * k + j]);
    h[j] = s;
    if (blockIdx.x == 0) hsave[j] = s;
  }
  __syncthreads();
  for (int64_t i = g.lo() + threadIdx.x; i < g.hi(); i += KT) {
    A xi = kload(x[i]);
    for (int j = 0; j < k; ++j) xi = sub(xi, mul(kload(V[(int64_t)j * g.n + i]), h[j]));
    kstore(x + i, xi);
  }
  __syncthreads();
}

template <typename S, typename A>
__global__ void __launch_bounds__(KT) krylov_pass1_kernel(S* __restrict__ V, const S* __restrict__ w, int64_t ws, int k, KGeo g,
                                                          A* __restrict__ part) {
  __shared__ A sred[KT / 32 * KJ];
  S* x = V + (int64_t)k * g.n;
  for (int64_t i = g.lo() + threadIdx.x; i < g.hi(); i += KT) x[i] = w[i * ws];
  __syncthreads();
  chunk_dots<S, A>(V, x, k, g, part, sred);
}

template <typename S, typename A>
__global__ void __launch_bounds__(KT) krylov_pass2_kernel(S* __restrict__ V, int k, KGeo g, const A* __restrict__ part_in,
                                                          A* __restrict__ part_out, A* __restrict__ hsave) {
  extern __shared__ __align__(16) unsigned char kr_smem[];
  A* h = reinterpret_cast<A*>(kr_smem);
  __shared__ A sred[KT / 32 * KJ];
  S* x = V + (int64_t)k * g.n;
  reduce_and_subtract<S, A>(V, x, k, g, part_in, h, hsave);
  chunk_dots<S, A>(V, x, k, g, part_out, sred);
}

template <typename S, typename A>
__global__ void __launch_bounds__(KT) krylov_pass3_kernel(S* __restrict__ V, int k, KGeo g, const A* __restrict__ part_in,
                                                          A* __restrict__ hsave, double* __restrict__ nrm_part) {
  extern __shared__ __align__(16) unsigned char kr_smem[];
  A* h = reinterpret_cast<A*>(kr_smem);
  __shared__ double red[KT / 32];
  S* x = V + (int64_t)k * g.n;
  reduce_and_subtract<S, A>(V, x, k, g, part_in, h, hsave);
  double acc = 0.0;
  for (int64_t i = g.lo() + threadIdx.x; i < g.hi(); i += KT) acc += ab2(kload(x[i]));
  acc = kwarp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < KT / 32; ++w) s += red[w];
    nrm_part[blockIdx.x] = s;
  }
}

template <typename S, typename A>
__global__ void __launch_bounds__(KT) krylov_norm_kernel(S* __restrict__ V, int k, KGeo g, const double* __restrict__ nrm_part,
                                                         const A* __restrict__ h1, const A* __restrict__ h2, S* __restrict__ h_out) {
  __shared__ double nrm_s;
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int c = 0; c < (int)gridDim.x; ++c) s += nrm_part[c];
    nrm_s = sqrt(s);
  }
  __syncthreads();
  const double nrm = nrm_s, inv = nrm > 0.0 ? 1.0 / nrm : 0.0;
  S* x = V + (int64_t)k * g.n;
  for (int64_t i = g.lo() + threadIdx.x; i < g.hi(); i += KT) kstore(x + i, mulr(kload(x[i]), inv));
  if (blockIdx.x == 0) {
    for (int j = threadIdx.x; j < k; j += KT) kstore(h_out + j, add(h1[j], h2[j]));
    if (threadIdx.x == 0) kstore(h_out + k, mk(nrm, 0.0, (A*)nullptr));
  }
}

template <typename S>
static int orth_t(const tnb200_tensor_t* basis, const tnb200_tensor_t* w, int k, void* h_dev, cudaStream_t st) {
  using A = typename KAcc<S>::A;
  const int64_t n = basis->shape[1];
  int64_t grid = (n + 4 * KT - 1) / (4 * KT);
  if (grid > 2 * num_sms()) grid = 2 * num_sms();
  if (grid < 1) grid = 1;
  KGeo g{n, (n + grid - 1) / grid};
  const int kk = k > 0 ? k : 1;
  const size_t hbytes = sizeof(A) * (size_t)kk;
  TNB_REQUIRE(hbytes <= 48 * 1024, TNB200_ERR_UNSUPPORTED, "krylov_orth: at most %d basis vectors", (int)(48 * 1024 / sizeof(A)));
  A *p1 = nullptr, *p2 = nullptr, *hs = nullptr;
  double* np = nullptr;
  int rc;
  if ((rc = ws_alloc((void**)&p1, sizeof(A) * (size_t)(grid * kk), st))) return rc;
  if ((rc = ws_alloc((void**)&p2, sizeof(A) * (size_t)(grid * kk), st))) return rc;
  if ((rc = ws_alloc((void**)&hs, sizeof(A) * (size_t)(2 * kk), st))) return rc;
  if ((rc = ws_alloc((void**)&np, sizeof(double) * (size_t)grid, st))) return rc;
  S* V = (S*)basis->data;
  krylov_pass1_kernel<S, A><<<(unsigned)grid, KT, 0, st>>>(V, (const S*)w->data, w->stride[0], k, g, p1);
  krylov_pass2_kernel<S, A><<<(unsigned)grid, KT, hbytes, st>>>(V, k, g, p1, p2, hs);
  krylov_pass3_kernel<S, A><<<(unsigned)grid, KT, hbytes, st>>>(V, k, g, p2, hs + kk, np);
  krylov_norm_kernel<S, A><<<(unsigned)grid, KT, 0, st>>>(V, k, g, np, hs, hs + kk, (S*)h_dev);
  TNB_LAUNCH_CHECK();
  count_launch(4);
  ws_free(p1, st); ws_free(p2, st); ws_free(hs, st); ws_free(np, st);
  return 0;
}

}  // namespace tnb

using namespace tnb;

extern "C" int32_t tnb200_krylov_orth(const tnb200_tensor_t* basis, const tnb200_tensor_t* w, int32_t k, void* h_dev, void* stream) {
  TNB_REQUIRE(valid_tensor(basis) && valid_tensor(w) && h_dev, TNB200_ERR_INVALID, "krylov_orth: invalid arguments");
  TNB_REQUIRE(basis->ndim == 2 && w->ndim == 1 && w->shape[0] == basis->shape[1], TNB200_ERR_INVALID,
              "krylov_orth: basis must be (rows, n) and w (n,)");
  TNB_REQUIRE(basis->stride[1] == 1 && basis->stride[0] == basis->shape[1], TNB200_ERR_INVALID, "krylov_orth: basis must be contiguous");
  TNB_REQUIRE(k >= 0 && k < basis->shape[0], TNB200_ERR_INVALID, "krylov_orth: row %d outside the basis", k);
  TNB_REQUIRE(w->dtype == basis->dtype, TNB200_ERR_DTYPE, "krylov_orth: w dtype must equal the basis dtype");
  if (basis->shape[1] == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  set_kernel_name("krylov_cgs2");
  switch (basis->dtype) {
    case TNB200_F64: return orth_t<double>(basis, w, k, h_dev, st);
    case TNB200_F32: return orth_t<float>(basis, w, k, h_dev, st);
    case TNB200_C128: return orth_t<cuDoubleComplex>(basis, w, k, h_dev, st);
    case TNB200_C64: return orth_t<cuFloatComplex>(basis, w, k, h_dev, st);
    default: set_error("krylov_orth: dtype %s is not supported (f32/f64/c64/c128)", dtype_name(basis->dtype)); return TNB200_ERR_DTYPE;
  }
}
