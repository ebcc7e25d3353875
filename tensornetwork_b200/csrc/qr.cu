// qr.cu — tnb200_qr: reduced Householder QR (decompositions.qr, backends/numpy/decompositions.py:77-98;
// LAPACK geqrf + orgqr there, same reflector convention: beta = -sign(alpha) * |x|, so R's diagonal
// signs match numpy's unless non_negative_diagonal asks for the phase fix of :91-94).
//
// Working storage is column-contiguous so every reflector application is a coalesced
// dot + axpy over one column per CTA.  Per column: one "larfg" launch (norm + scale of the
// reflector) and one "larf" launch over the trailing columns; Q is then formed by applying the
// reflectors in reverse order to the first r columns of the identity.
#include "common.cuh"
#include "cplx.cuh"
#include <math.h>
#include <stdlib.h>

namespace tnb {

int copy_strided(const tnb200_tensor_t* src, const tnb200_tensor_t* dst, int conj, cudaStream_t st);

__device__ inline double block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
  return t;  // every thread gets the total
}
__device__ inline double block_sum_t(double v, double* red) { return block_sum(v, red); }
__device__ inline zd block_sum_t(zd v, double* red) { double a = block_sum(v.x, red); double b = block_sum(v.y, red); return zd{a, b}; }

// LAPACK xLARFG on column j: W[j:, j] -> (beta (real) on the diagonal, v[1:] below it), tau[j]
template <typename T>
__global__ void __launch_bounds__(256) qr_larfg_kernel(T* __restrict__ W, int64_t m, int j, T* __restrict__ tau) {
  __shared__ double red[8];
  T* col = W + (int64_t)j * m;
  double acc = 0.0;
  for (int64_t i = j + 1 + threadIdx.x; i < m; i += blockDim.x) acc += ab2(col[i]);
  const double sigma2 = block_sum(acc, red);
  const T alpha = col[j];
  if (sigma2 == 0.0 && im_(alpha) == 0.0) {
    if (threadIdx.x == 0) tau[j] = zero_<T>();
    return;
  }
  const double nrm = sqrt(ab2(alpha) + sigma2);
  const double beta = re_(alpha) >= 0.0 ? -nrm : nrm;
  const T scale = divz(one_<T>(), sub(alpha, mk(beta, 0.0, (T*)nullptr)));
  for (int64_t i = j + 1 + threadIdx.x; i < m; i += blockDim.x) col[i] = mul(col[i], scale);
  __syncthreads();
  if (threadIdx.x == 0) {
    tau[j] = mk((beta - re_(alpha)) / beta, -im_(alpha) / beta, (T*)nullptr);
    col[j] = mk(beta, 0.0, (T*)nullptr);
  }
}

// apply H_j (conj_tau = 0) or H_j^H (conj_tau = 1), H_j = I - tau v v^H, v = [1; V[j+1:, j]], to the
// columns c0 + blockIdx.x of X (rows j..m-1)
template <typename T>
__global__ void __launch_bounds__(128) qr_larf_kernel(const T* __restrict__ V, T* __restrict__ X, int64_t m, int j, int c0,
                                                      const T* __restrict__ tau, int conj_tau) {
  __shared__ double red[4];
  T t = tau[j];
  if (re_(t) == 0.0 && im_(t) == 0.0) return;
  if (conj_tau) t = cj(t);
  const T* v = V + (int64_t)j * m;
  T* x = X + (int64_t)(c0 + blockIdx.x) * m;
  T acc = threadIdx.x == 0 ? x[j] : zero_<T>();
  for (int64_t i = j + 1 + threadIdx.x; i < m; i += blockDim.x) fmacc(acc, cj(v[i]), x[i]);
  const T w = mul(block_sum_t(acc, red), t);
  if (threadIdx.x == 0) x[j] = sub(x[j], w);
  for (int64_t i = j + 1 + threadIdx.x; i < m; i += blockDim.x) x[i] = sub(x[i], mul(w, v[i]));
}

template <typename T>
__global__ void qr_init_q_kernel(T* Q, int64_t m, int r) {
  int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx < m * r) Q[idx] = (idx % m == idx / m) ? one_<T>() : zero_<T>();
}

// write q (m x r) and r (r x n) with the optional sign fix: phases = sign(diag(R)) (diag is real)
template <typename T>
__global__ void qr_writeout_kernel(const T* __restrict__ W, const T* __restrict__ Q, int64_t m, int64_t n, int r, int nonneg,
                                   T* __restrict__ q, int64_t q_s0, int64_t q_s1, T* __restrict__ rr, int64_t r_s0, int64_t r_s1) {
  const int64_t total_q = m * r, total_r = (int64_t)r * n;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total_q + total_r; idx += (int64_t)gridDim.x * blockDim.x) {
    if (idx < total_q) {
      int64_t c = idx / m, i = idx % m;
      double ph = 1.0;
      if (nonneg) { double d = re_(W[c * m + c]); ph = d > 0.0 ? 1.0 : (d < 0.0 ? -1.0 : 0.0); }
      q[i * q_s0 + c * q_s1] = mulr(Q[c * m + i], ph);
    } else {
      int64_t k = idx - total_q;
      int64_t c = k / r, i = k % r;       // R[i, c]
      T val = i <= c ? W[c * m + i] : zero_<T>();
      if (nonneg) { double d = re_(W[i * m + i]); val = mulr(val, d > 0.0 ? 1.0 : (d < 0.0 ? -1.0 : 0.0)); }
      rr[i * r_s0 + c * r_s1] = val;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Blocked Householder QR for real matrices (compact WY, LAPACK geqrf / orgqr structure): panels of 32 columns.
//   qr_panel_kernel : ONE cluster of 8 CTAs factors a panel.  The panel lives in shared memory, its rows dealt to the CTAs;
//                     per column ONE cluster-wide all-reduce through distributed shared memory carries everything the
//                     reflector needs (sigma^2 = x^T x and the products x^T a_c with all later panel columns come from the
//                     same pass; the pivot-row entries a_jc ride in the same message), then v, tau and the rank-1 update of
//                     the rest of the panel are local.  Ends with T of the compact-WY form (larft) from V^T V.
//   qr_apply_kernel : X[j0:, cols] <- (I - V T' V^T) X for a block of 32 columns per CTA: W1 = V^T X (DMMA), W2 = T' W1,
//                     X -= V W2 (DMMA) — the trailing update (T' = T^T) and, on the identity, the formation of Q (T' = T).
// 3 launches per 32 columns instead of 3 per column; reflector convention unchanged (beta = -sign(alpha) |x|), so the
// factors still agree element-wise with numpy's.
constexpr int QB = 32, QCL = 8, QLD = 68;

__device__ __forceinline__ void qr_dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__device__ __forceinline__ uint32_t qr_cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void qr_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// store a double into the shared memory of CTA `rank` of the cluster at the address corresponding to local pointer p
__device__ __forceinline__ void qr_st_remote(double* p, uint32_t rank, double v) {
  uint32_t a = (uint32_t)__cvta_generic_to_shared(p), r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
  asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(r), "d"(v) : "memory");
}

__global__ void __cluster_dims__(QCL, 1, 1) __launch_bounds__(256, 1)
qr_panel_kernel(double* __restrict__ W, int64_t m, int j0, int b, int rl, double* __restrict__ tau, double* __restrict__ Tout,
                double* __restrict__ Z) {
  extern __shared__ __align__(16) double qsm[];
  const int RLP = rl + (rl & 1);
  double* P = qsm;                               // [QB][RLP]: this CTA's rows of the panel, column-major
  double* part = P + (size_t)QB * RLP;           // [2][QCL][64]
  double* mine = part + 2 * QCL * 64;            // [64]
  double* tot = mine + 64;                       // [64]
  double* taus = tot + 64;                       // [QB]
  double* Ts = taus + QB;                        // [QB][QB + 1]  (rank 0 only)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t rank = qr_cluster_rank();
  const int64_t row0 = (int64_t)j0 + (int64_t)rank * rl;          // first global row of this CTA
  int64_t nl64 = m - row0; if (nl64 > rl) nl64 = rl; if (nl64 < 0) nl64 = 0;
  const int nl = (int)nl64;                                       // local rows
  for (int idx = tid; idx < b * nl; idx += 256) {
    const int c = idx / nl, i = idx - c * nl;
    P[c * RLP + i] = W[(int64_t)(j0 + c) * m + row0 + i];
  }
  if (tid < QB) taus[tid] = 0.0;
  __syncthreads();
  const int nsteps = (int64_t)b < m - j0 ? b : (int)(m - j0);
  for (int j = 0; j < nsteps; ++j) {
    const int64_t gp = (int64_t)j0 + j;                           // global pivot row
    int is = (int)(gp + 1 - row0); if (is < 0) is = 0;            // first local row strictly below the pivot
    const bool own = gp >= row0 && gp < row0 + nl;
    const int jl = (int)(gp - row0);
    if (tid < 64) mine[tid] = 0.0;
    __syncthreads();
    // partial products of column j (rows below the pivot) with columns j .. b-1: one warp per column, strided
    const double* xj = P + j * RLP;
    for (int c = j + warp; c < b; c += 8) {
      const double* ac = P + c * RLP;
      double acc = 0.0;
      for (int i = is + lane; i < nl; i += 32) acc = fma(xj[i], ac[i], acc);
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
      if (lane == 0) mine[c] = acc;
    }
    if (own && tid >= j && tid < b) mine[32 + tid] = P[tid * RLP + jl];      // pivot-row entries a_jc (c = j: alpha)
    __syncthreads();
    const int buf = j & 1;
    if (tid < 64) {
      const double v = mine[tid];
#pragma unroll
      for (uint32_t q = 0; q < QCL; ++q) qr_st_remote(part + ((size_t)buf * QCL + rank) * 64 + tid, q, v);
    }
    qr_cluster_sync();
    if (tid < 64) {
      double t = 0.0;
#pragma unroll
      for (int q = 0; q < QCL; ++q) t += part[((size_t)buf * QCL + q) * 64 + tid];
      tot[tid] = t;
    }
    __syncthreads();
    const double sigma2 = tot[j], alpha = tot[32 + j];
    if (sigma2 != 0.0) {
      const double nrm = sqrt(alpha * alpha + sigma2);
      const double beta = alpha >= 0.0 ? -nrm : nrm;
      const double scale = 1.0 / (alpha - beta);
      const double tj = (beta - alpha) / beta;
      // rank-1 update of the later panel columns with the UNSCALED x (v_i = x_i * scale), then scale column j
      const int nrows = nl - is;
      if (nrows > 0) {
        for (int idx = tid; idx < (b - j - 1) * nrows; idx += 256) {
          const int c = j + 1 + idx / nrows, i = is + idx % nrows;
          const double wc = tj * (tot[32 + c] + tot[c] * scale);
          P[c * RLP + i] -= wc * (xj[i] * scale);
        }
      }
      if (own) {
        for (int c = j + 1 + tid; c < b; c += 256) P[c * RLP + jl] -= tj * (tot[32 + c] + tot[c] * scale);
      }
      __syncthreads();
      for (int i = is + tid; i < nl; i += 256) P[j * RLP + i] *= scale;
      if (own && tid == 0) P[j * RLP + jl] = beta;
      if (tid == 0) taus[j] = tj;
    }
    __syncthreads();
  }
  // write the factored panel back (R above / on the diagonal, V below)
  for (int idx = tid; idx < b * nl; idx += 256) {
    const int c = idx / nl, i = idx - c * nl;
    W[(int64_t)(j0 + c) * m + row0 + i] = P[c * RLP + i];
  }
  // Z = V^T V (strict upper part) for larft: v(i,k) = 0 above the diagonal of the panel, 1 on it, P below
  for (int idx = tid; idx < b * b; idx += 256) {
    const int k = idx / b, jj = idx % b;
    if (k >= jj) continue;
    double acc = 0.0;
    int i0 = (int)((int64_t)j0 + jj - row0); if (i0 < 0) i0 = 0;            // rows >= pivot of the LATER column jj
    for (int i = i0; i < nl; ++i) {
      const int64_t gi = row0 + i;
      const double vk = P[k * RLP + i];                                     // gi >= j0 + jj > j0 + k: below k's pivot
      const double vj = gi == (int64_t)j0 + jj ? 1.0 : P[jj * RLP + i];
      acc = fma(vk, vj, acc);
    }
    if (acc != 0.0) atomicAdd(&Z[k * QB + jj], acc);
  }
  __threadfence();
  qr_cluster_sync();
  if (rank == 0) {
    if (tid < b) tau[tid] = taus[tid];
    for (int idx = tid; idx < QB * (QB + 1); idx += 256) Ts[idx] = 0.0;
    __syncthreads();
    for (int jj = 0; jj < b; ++jj) {                                        // T(0:jj, jj) = -tau_jj T(0:jj, 0:jj) Z(0:jj, jj)
      if (tid < jj) {
        double acc = 0.0;
        for (int l = tid; l < jj; ++l) acc = fma(Ts[tid * (QB + 1) + l], __ldcg(&Z[l * QB + jj]), acc);
        Ts[tid * (QB + 1) + jj] = -taus[jj] * acc;
      }
      if (tid == jj) Ts[jj * (QB + 1) + jj] = taus[jj];
      __syncthreads();
    }
    for (int idx = tid; idx < QB * QB; idx += 256) Tout[idx] = Ts[(idx / QB) * (QB + 1) + idx % QB];
  }
}

// X[j0:, c0 + 32 blockIdx.x ...] <- (I - V T' V^T) X ; V = unit lower trapezoid stored in W[j0:, j0:j0+b], T' = transT ? T^T : T.
// Two kernels over a (column block, row chunk) grid so that a narrow trailing matrix still fills the GPU:
//   qr_apply1_kernel : partial W1 = V^T X over this chunk's row tiles -> w1p[column block][chunk][32 x 32]
//   qr_apply2_kernel : W1 = sum of the partials in chunk order (deterministic), W2 = T' W1, X -= V W2 on this chunk's rows
struct QrApply {
  const double* W; int64_t m; int j0, b; const double* T; int transT; double* X; int64_t ldx; int c0, ncols; int rs; double* w1p;
};
__device__ __forceinline__ void qr_fetch_tile(const QrApply& q, int cb, int nc, int t, int e_c, int e_r, double* pv, double* px) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = e_r + 8 * i;
    const int64_t gi = (int64_t)q.j0 + (int64_t)t * 64 + r;
    double v = 0.0, x = 0.0;
    if (gi < q.m) {
      if (e_c < q.b) {
        const int64_t piv = (int64_t)q.j0 + e_c;
        v = gi > piv ? q.W[(int64_t)(q.j0 + e_c) * q.m + gi] : (gi == piv ? 1.0 : 0.0);
      }
      if (e_c < nc) x = q.X[(int64_t)(cb + e_c) * q.ldx + gi];
    }
    pv[i] = v; px[i] = x;
  }
}

__global__ void __launch_bounds__(256) qr_apply1_kernel(const QrApply q) {
  extern __shared__ __align__(16) double qasm[];
  double (*tv)[QB * QLD] = reinterpret_cast<double (*)[QB * QLD]>(qasm);
  double (*tx)[QB * QLD] = reinterpret_cast<double (*)[QB * QLD]>(qasm + 2 * QB * QLD);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, fr = lane >> 2, fk = lane & 3;
  const int cb = q.c0 + blockIdx.x * QB;
  const int nc = q.ncols - blockIdx.x * QB < QB ? q.ncols - blockIdx.x * QB : QB;
  const int ntiles = (int)((q.m - q.j0 + 63) / 64);
  const int t0 = (int)((int64_t)ntiles * blockIdx.y / q.rs), t1 = (int)((int64_t)ntiles * (blockIdx.y + 1) / q.rs);
  const int e_c = tid >> 3, e_r = tid & 7;
  double pv[8], px[8];
  const int mt = warp >> 1, nt0 = (warp & 1) * 2;
  double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
  if (t0 < t1) {
    qr_fetch_tile(q, cb, nc, t0, e_c, e_r, pv, px);
#pragma unroll
    for (int i = 0; i < 8; ++i) { tv[0][e_c * QLD + e_r + 8 * i] = pv[i]; tx[0][e_c * QLD + e_r + 8 * i] = px[i]; }
    __syncthreads();
    int buf = 0;
    for (int t = t0; t < t1; ++t) {
      if (t + 1 < t1) qr_fetch_tile(q, cb, nc, t + 1, e_c, e_r, pv, px);
      const double* av = tv[buf];
      const double* bx = tx[buf];
#pragma unroll
      for (int k4 = 0; k4 < 64; k4 += 4) {
        const double a = av[(mt * 8 + fr) * QLD + k4 + fk];
#pragma unroll
        for (int j = 0; j < 2; ++j) qr_dmma(acc[j][0], acc[j][1], a, bx[((nt0 + j) * 8 + fr) * QLD + k4 + fk]);
      }
      if (t + 1 < t1) {
#pragma unroll
        for (int i = 0; i < 8; ++i) { tv[buf ^ 1][e_c * QLD + e_r + 8 * i] = pv[i]; tx[buf ^ 1][e_c * QLD + e_r + 8 * i] = px[i]; }
      }
      __syncthreads();
      buf ^= 1;
    }
  }
  double* out = q.w1p + ((size_t)blockIdx.x * q.rs + blockIdx.y) * (QB * QB);
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    out[(mt * 8 + fr) * QB + (nt0 + j) * 8 + 2 * fk] = acc[j][0];
    out[(mt * 8 + fr) * QB + (nt0 + j) * 8 + 2 * fk + 1] = acc[j][1];
  }
}

__global__ void __launch_bounds__(256) qr_apply2_kernel(const QrApply q) {
  extern __shared__ __align__(16) double qasm[];
  double (*tv)[QB * QLD] = reinterpret_cast<double (*)[QB * QLD]>(qasm);
  double (*tx)[QB * QLD] = reinterpret_cast<double (*)[QB * QLD]>(qasm + 2 * QB * QLD);
  double* w1 = qasm + 4 * QB * QLD;
  double* w2 = w1 + QB * (QB + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, fr = lane >> 2, fk = lane & 3;
  const int cb = q.c0 + blockIdx.x * QB;
  const int nc = q.ncols - blockIdx.x * QB < QB ? q.ncols - blockIdx.x * QB : QB;
  const int ntiles = (int)((q.m - q.j0 + 63) / 64);
  const int t0 = (int)((int64_t)ntiles * blockIdx.y / q.rs), t1 = (int)((int64_t)ntiles * (blockIdx.y + 1) / q.rs);
  if (t0 >= t1) return;
  const double* part = q.w1p + (size_t)blockIdx.x * q.rs * (QB * QB);
  for (int idx = tid; idx < QB * QB; idx += 256) {
    double s = 0.0;
    for (int c = 0; c < q.rs; ++c) s += part[(size_t)c * (QB * QB) + idx];
    w1[(idx >> 5) * (QB + 1) + (idx & 31)] = s;
  }
  __syncthreads();
  for (int idx = tid; idx < QB * QB; idx += 256) {
    const int k = idx >> 5, c = idx & 31;
    double s = 0.0;
    if (k < q.b) {
      for (int l = 0; l < q.b; ++l) s = fma(q.transT ? q.T[l * QB + k] : q.T[k * QB + l], w1[l * (QB + 1) + c], s);
    }
    w2[k * (QB + 1) + c] = s;
  }
  __syncthreads();
  const int e_c = tid >> 3, e_r = tid & 7;
  double pv[8], px[8];
  const int ct = warp >> 1, rh = (warp & 1) * 32;
  double wa[8];
#pragma unroll
  for (int k4 = 0; k4 < 8; ++k4) wa[k4] = w2[(k4 * 4 + fk) * (QB + 1) + ct * 8 + fr];
  qr_fetch_tile(q, cb, nc, t0, e_c, e_r, pv, px);
#pragma unroll
  for (int i = 0; i < 8; ++i) { tv[0][e_c * QLD + e_r + 8 * i] = pv[i]; tx[0][e_c * QLD + e_r + 8 * i] = px[i]; }
  __syncthreads();
  int buf = 0;
  for (int t = t0; t < t1; ++t) {
    if (t + 1 < t1) qr_fetch_tile(q, cb, nc, t + 1, e_c, e_r, pv, px);
    const double* av = tv[buf];
    double oc[4][2];
#pragma unroll
    for (int j = 0; j < 4; ++j) { oc[j][0] = 0.0; oc[j][1] = 0.0; }
#pragma unroll
    for (int k4 = 0; k4 < 8; ++k4)
#pragma unroll
      for (int j = 0; j < 4; ++j) qr_dmma(oc[j][0], oc[j][1], wa[k4], av[(k4 * 4 + fk) * QLD + rh + j * 8 + fr]);
    const int c = ct * 8 + fr;
    if (c < nc) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int r = rh + j * 8 + 2 * fk;
        const int64_t gi = (int64_t)q.j0 + (int64_t)t * 64 + r;
        double* dst = q.X + (int64_t)(cb + c) * q.ldx + gi;
        if (gi < q.m) dst[0] = tx[buf][c * QLD + r] - oc[j][0];
        if (gi + 1 < q.m) dst[1] = tx[buf][c * QLD + r + 1] - oc[j][1];
      }
    }
    if (t + 1 < t1) {
#pragma unroll
      for (int i = 0; i < 8; ++i) { tv[buf ^ 1][e_c * QLD + e_r + 8 * i] = pv[i]; tx[buf ^ 1][e_c * QLD + e_r + 8 * i] = px[i]; }
    }
    __syncthreads();
    buf ^= 1;
  }
}

static int qr_apply(const QrApply& q0, double* w1p, size_t w1p_doubles, cudaStream_t st, int* launches) {
  QrApply q = q0;
  const int ncb = (q.ncols + QB - 1) / QB;
  const int ntiles = (int)((q.m - q.j0 + 63) / 64);
  int rs = (2 * num_sms() + ncb - 1) / ncb;
  if (rs > ntiles) rs = ntiles;
  if (rs < 1) rs = 1;
  while ((size_t)ncb * rs * QB * QB > w1p_doubles && rs > 1) --rs;
  q.rs = rs; q.w1p = w1p;
  const size_t smem1 = sizeof(double) * (4 * QB * QLD), smem2 = sizeof(double) * (4 * QB * QLD + 2 * QB * (QB + 1));
  qr_apply1_kernel<<<dim3((unsigned)ncb, (unsigned)rs), 256, smem1, st>>>(q);
  qr_apply2_kernel<<<dim3((unsigned)ncb, (unsigned)rs), 256, smem2, st>>>(q);
  *launches += 2;
  return 0;
}

static int qr_blocked_f64(const tnb200_tensor_t* a, const tnb200_tensor_t* q, const tnb200_tensor_t* r, int nonneg, cudaStream_t st) {
  const int64_t m = a->shape[0], n = a->shape[1];
  const int k = (int)(m < n ? m : n);
  const int npan = (k + QB - 1) / QB;
  double *W = nullptr, *Q = nullptr, *tau = nullptr, *Tb = nullptr, *Z = nullptr;
  int rc;
  if ((rc = ws_alloc((void**)&W, sizeof(double) * (size_t)m * n, st))) return rc;
  if ((rc = ws_alloc((void**)&Q, sizeof(double) * (size_t)m * k, st))) return rc;
  if ((rc = ws_alloc((void**)&tau, sizeof(double) * (size_t)(k + QB), st))) return rc;
  if ((rc = ws_alloc((void**)&Tb, sizeof(double) * (size_t)npan * QB * QB, st))) return rc;
  if ((rc = ws_alloc((void**)&Z, sizeof(double) * (size_t)npan * QB * QB, st))) return rc;
  TNB_CHECK_CUDA(cudaMemsetAsync(Z, 0, sizeof(double) * (size_t)npan * QB * QB, st));
  tnb200_tensor_t dst;
  dst.data = W; dst.dtype = a->dtype; dst.ndim = 2;
  dst.shape[0] = m; dst.shape[1] = n; dst.stride[0] = 1; dst.stride[1] = m;
  if ((rc = copy_strided(a, &dst, 0, st))) return rc;
  const size_t apply_smem = sizeof(double) * (4 * QB * QLD + 2 * QB * (QB + 1));
  static bool attr_done = false;
  if (!attr_done) {
    TNB_CHECK_CUDA(cudaFuncSetAttribute(qr_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 1024));
    TNB_CHECK_CUDA(cudaFuncSetAttribute(qr_apply1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)apply_smem));
    TNB_CHECK_CUDA(cudaFuncSetAttribute(qr_apply2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)apply_smem));
    attr_done = true;
  }
  // partial W1 blocks of the apply kernels: (column blocks) x (row chunks) x 32 x 32, at most ~2 CTAs per SM worth of chunks
  const size_t w1p_doubles = (size_t)(2 * num_sms() + (n + QB - 1) / QB + 8) * QB * QB;
  double* w1p = nullptr;
  if ((rc = ws_alloc((void**)&w1p, sizeof(double) * w1p_doubles, st))) return rc;
  int launches = 0;
  for (int p = 0; p < npan; ++p) {
    const int j0 = p * QB, b = k - j0 < QB ? k - j0 : QB;
    int rl = (int)((m - j0 + QCL - 1) / QCL);
    if (rl < 1) rl = 1;
    const size_t smem = sizeof(double) * ((size_t)QB * (rl + (rl & 1)) + 2 * QCL * 64 + 64 + 64 + QB + QB * (QB + 1)) + 16;
    qr_panel_kernel<<<QCL, 256, smem, st>>>(W, m, j0, b, rl, tau + j0, Tb + (size_t)p * QB * QB, Z + (size_t)p * QB * QB);
    ++launches;
    if (j0 + b < n) {
      QrApply q{W, m, j0, b, Tb + (size_t)p * QB * QB, 1, W, m, j0 + b, (int)(n - j0 - b), 1, nullptr};
      qr_apply(q, w1p, w1p_doubles, st, &launches);
    }
  }
  qr_init_q_kernel<double><<<(unsigned)((m * k + 255) / 256), 256, 0, st>>>(Q, m, k);
  for (int p = npan - 1; p >= 0; --p) {
    const int j0 = p * QB, b = k - j0 < QB ? k - j0 : QB;
    QrApply q{W, m, j0, b, Tb + (size_t)p * QB * QB, 0, Q, m, j0, k - j0, 1, nullptr};
    qr_apply(q, w1p, w1p_doubles, st, &launches);
  }
  int64_t tot = m * k + (int64_t)k * n;
  int64_t blocks = (tot + 255) / 256;
  if (blocks > (int64_t)num_sms() * 16) blocks = (int64_t)num_sms() * 16;
  qr_writeout_kernel<double><<<(unsigned)blocks, 256, 0, st>>>(W, Q, m, n, k, nonneg, (double*)q->data, q->stride[0], q->stride[1],
                                                              (double*)r->data, r->stride[0], r->stride[1]);
  TNB_LAUNCH_CHECK();
  count_launch(launches + 2);
  ws_free(W, st); ws_free(Q, st); ws_free(tau, st); ws_free(Tb, st); ws_free(Z, st); ws_free(w1p, st);
  return 0;
}

template <typename T>
static int qr_real(const tnb200_tensor_t* a, const tnb200_tensor_t* q, const tnb200_tensor_t* r, int nonneg, cudaStream_t st) {
  const int64_t m = a->shape[0], n = a->shape[1];
  const int k = (int)(m < n ? m : n);
  if (m == 0 || n == 0) return 0;
  T *W = nullptr, *Q = nullptr, *tau = nullptr;
  int rc;
  if ((rc = ws_alloc((void**)&W, sizeof(T) * (size_t)m * n, st))) return rc;
  if ((rc = ws_alloc((void**)&Q, sizeof(T) * (size_t)m * k, st))) return rc;
  if ((rc = ws_alloc((void**)&tau, sizeof(T) * (size_t)k, st))) return rc;
  tnb200_tensor_t dst;
  dst.data = W; dst.dtype = a->dtype; dst.ndim = 2;
  dst.shape[0] = m; dst.shape[1] = n; dst.stride[0] = 1; dst.stride[1] = m;
  if ((rc = copy_strided(a, &dst, 0, st))) return rc;
  for (int j = 0; j < k; ++j) {
    qr_larfg_kernel<T><<<1, 256, 0, st>>>(W, m, j, tau);
    if (j + 1 < n) qr_larf_kernel<T><<<(unsigned)(n - j - 1), 128, 0, st>>>(W, W, m, j, j + 1, tau, 1);
  }
  qr_init_q_kernel<T><<<(unsigned)((m * k + 255) / 256), 256, 0, st>>>(Q, m, k);
  for (int j = k - 1; j >= 0; --j) qr_larf_kernel<T><<<(unsigned)(k - j), 128, 0, st>>>(W, Q, m, j, j, tau, 0);
  int64_t tot = m * k + (int64_t)k * n;
  int64_t blocks = (tot + 255) / 256;
  if (blocks > (int64_t)num_sms() * 16) blocks = (int64_t)num_sms() * 16;
  qr_writeout_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(W, Q, m, n, k, nonneg, (T*)q->data, q->stride[0], q->stride[1],
                                                         (T*)r->data, r->stride[0], r->stride[1]);
  TNB_LAUNCH_CHECK();
  count_launch(3 * k + 2);
  ws_free(W, st); ws_free(Q, st); ws_free(tau, st);
  return 0;
}

}  // namespace tnb

using namespace tnb;

extern "C" int32_t tnb200_qr(const tnb200_tensor_t* a, const tnb200_tensor_t* q, const tnb200_tensor_t* r,
                             int32_t non_negative_diagonal, void* stream) {
  TNB_REQUIRE(valid_tensor(a) && valid_tensor(q) && valid_tensor(r), TNB200_ERR_INVALID, "qr: invalid tensor descriptor");
  TNB_REQUIRE(a->ndim == 2 && q->ndim == 2 && r->ndim == 2, TNB200_ERR_INVALID, "qr: expects matrices");
  const int64_t m = a->shape[0], n = a->shape[1], k = m < n ? m : n;
  TNB_REQUIRE(q->shape[0] == m && q->shape[1] == k && r->shape[0] == k && r->shape[1] == n, TNB200_ERR_INVALID,
              "qr: output shapes must be (m,k), (k,n) with k = min(m,n)");
  TNB_REQUIRE(a->dtype != TNB200_BOOL, TNB200_ERR_DTYPE, "qr: bool tensors are not supported");
  TNB_REQUIRE(q->dtype == a->dtype && r->dtype == a->dtype, TNB200_ERR_DTYPE, "qr: dtype mismatch");
  TNB_REQUIRE(m < (1LL << 31) && n < (1LL << 31), TNB200_ERR_UNSUPPORTED, "qr: matrix too large");
  set_kernel_name("qr_householder");
  cudaStream_t st = (cudaStream_t)stream;
  if (a->dtype == TNB200_F64) {
    // blocked path: the panel's rows must fit the shared memory of an 8-CTA cluster (m <= ~6500); TNB200_QR_ALGO=columns keeps the
    // one-launch-per-column kernels
    const char* algo = getenv("TNB200_QR_ALGO");
    const int64_t rl = (m + QCL - 1) / QCL;
    const bool fits = sizeof(double) * ((size_t)QB * (rl + 2) + 2 * QCL * 64 + 128 + QB + QB * (QB + 1)) + 16 <= 226 * 1024;
    if (fits && k >= 16 && !(algo && !strcmp(algo, "columns"))) { set_kernel_name("qr_blocked_wy"); return qr_blocked_f64(a, q, r, non_negative_diagonal, st); }
    return qr_real<double>(a, q, r, non_negative_diagonal, st);
  }
  if (a->dtype == TNB200_C128) return qr_real<zd>(a, q, r, non_negative_diagonal, st);
  if (a->dtype == TNB200_F32 || a->dtype == TNB200_C64) {   // widen, factor, round back
    const bool cplx = a->dtype == TNB200_C64;
    const int wide = cplx ? TNB200_C128 : TNB200_F64;
    const size_t esz = cplx ? 16 : 8;
    void *da = nullptr, *dq = nullptr, *dr = nullptr;
    int rc;
    if ((rc = ws_alloc(&da, esz * (size_t)m * n, st))) return rc;
    if ((rc = ws_alloc(&dq, esz * (size_t)m * k, st))) return rc;
    if ((rc = ws_alloc(&dr, esz * (size_t)k * n, st))) return rc;
    auto mk2 = [&](void* p, int64_t d0, int64_t d1) {
      tnb200_tensor_t t; t.data = p; t.dtype = wide; t.ndim = 2; t.shape[0] = d0; t.shape[1] = d1; t.stride[0] = d1; t.stride[1] = 1; return t;
    };
    tnb200_tensor_t ta = mk2(da, m, n), tq = mk2(dq, m, k), tr = mk2(dr, k, n);
    if ((rc = copy_strided(a, &ta, 0, st))) return rc;
    rc = cplx ? qr_real<zd>(&ta, &tq, &tr, non_negative_diagonal, st) : qr_real<double>(&ta, &tq, &tr, non_negative_diagonal, st);
    if (rc == 0) rc = copy_strided(&tq, q, 0, st);
    if (rc == 0) rc = copy_strided(&tr, r, 0, st);
    ws_free(da, st); ws_free(dq, st); ws_free(dr, st);
    return rc;
  }
  set_error("qr: dtype %s is not supported (f32/f64/c64/c128)", dtype_name(a->dtype));
  return TNB200_ERR_UNSUPPORTED;
}
