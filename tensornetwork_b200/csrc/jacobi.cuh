// jacobi.cuh — the block-pair Jacobi pieces shared by the SVD (svd.cu, one-sided on the Gram matrix of a column pair) and
// the Hermitian eigensolver (eigh.cu, two-sided on the diagonal block of an index pair):
//   rr_pair / pair_col   the round-robin tournament on nb blocks of SB indices
//   herm_jacobi_smem     cyclic two-sided Jacobi of a PB x PB Hermitian matrix held in shared memory
//   svd_eig_kernel       one CTA per pair: diagonalise the pair's PB x PB matrix, write its rotation R
//   svd_update_kernel    X[:, pair columns] <- X[:, pair columns] R for every pair of the round
// T is double or zd (cplx.cuh).  The kernels take an optional device flag `skip`: when it is set they return at once,
// which lets a caller enqueue a fixed number of sweeps and stop work on the device when its convergence test passes.
#pragma once
#include "common.cuh"
#include "cplx.cuh"

namespace tnb {

// Block width SB (columns per block; a pair rotates PB = 2 SB columns) is a template parameter: 16 is the default,
// 32 an experiment (see svd_dispatch): every round streams W and V through HBM once, and doubling the block width
// halves the number of rounds per sweep, but the Gram eigenproblem grows to 64 x 64 (still one CTA).
template <int SB> struct Geo {
  static constexpr int PB = 2 * SB;
  static constexpr int RT = SB == 16 ? 64 : 32;     // rows per shared-memory tile of the gram / update kernels
};

// round-robin tournament on nb (even) players: pair p of round r
__device__ __forceinline__ void rr_pair(int nb, int r, int p, int& i, int& j) {
  const int m = nb - 1;
  if (p == 0) { i = m; j = r % m; }
  else { i = (r + p) % m; j = (r - p + m) % m; }
  if (i > j) { int t = i; i = j; j = t; }
}
template <int SB>
__device__ __forceinline__ int pair_col(int bi, int bj, int c) { return c < SB ? bi * SB + c : bj * SB + (c - SB); }

// Cyclic two-sided Jacobi on the Hermitian PB x PB matrix g (shared memory, leading dimension PB + 1), 256 threads.  The
// rotations are accumulated into rm (initialised by the caller; its columns end up as the eigenvectors).  A sweep first
// measures the largest relative off-diagonal — |g_ij| / scale when scale > 0 (eigh: scale = ||A||_F), otherwise
// |g_ij| / sqrt(g_ii g_jj) over the pairs with a positive diagonal product (the SVD's Gram matrices) — and stops when it
// is <= tol; the measure of the first sweep is atomicMax'ed (float bits) into *conv when conv is not null.
// Returns the number of sweeps that rotated: max_sweeps when the tolerance was not reached.
// Scratch: cs[SB], sn[SB] (double), ph[SB] (T), pp[SB], qq[SB] (int), red[8] (float), offmax (float), all shared.
template <typename T, int SB>
__device__ int herm_jacobi_smem(T* g, T* rm, double* cs, double* sn, T* ph, int* pp, int* qq, float* red, float& offmax,
                                unsigned int* conv, double tol, int max_sweeps, double scale = 0.0) {
  constexpr int PB = Geo<SB>::PB, LD = PB + 1;
  const int tid = threadIdx.x;
  for (int sweep = 0; sweep < max_sweeps; ++sweep) {
    // relative off-diagonal measure
    float loc = 0.f;
    for (int idx = tid; idx < PB * PB; idx += 256) {
      int i = idx / PB, j = idx % PB;
      if (i < j) {
        double d = scale > 0.0 ? scale * scale : re_(g[i * LD + i]) * re_(g[j * LD + j]);
        if (d > 0.0) { float v = (float)(ab2(g[i * LD + j]) / d); loc = fmaxf(loc, v); }     // squared; root taken once below
      }
    }
    for (int o = 16; o > 0; o >>= 1) loc = fmaxf(loc, __shfl_xor_sync(0xffffffffu, loc, o));
    if ((tid & 31) == 0) red[tid >> 5] = loc;
    __syncthreads();
    if (tid == 0) {
      float m = 0.f;
      for (int w = 0; w < 8; ++w) m = fmaxf(m, red[w]);
      m = sqrtf(m);
      offmax = m;
      if (sweep == 0 && conv) atomicMax(conv, __float_as_uint(m));
    }
    __syncthreads();
    if (offmax <= (float)tol) return sweep;
    for (int step = 0; step < PB - 1; ++step) {
      if (tid < SB) {
        const int m = PB - 1;
        int p, q;
        if (tid == 0) { p = m; q = step % m; } else { p = (step + tid) % m; q = (step - tid + m) % m; }
        if (p > q) { int t = p; p = q; q = t; }
        // Hermitian 2x2 [[a, g], [conj g, b]], g = |g| e^{i phi}: rotate (x_p, e^{-i phi} x_q) by the
        // real Jacobi angle of [[a, |g|], [|g|, b]]
        const T gpq = g[p * LD + q];
        const double app = re_(g[p * LD + p]), aqq = re_(g[q * LD + q]);
        const double mag = mag_(gpq);
        double c = 1.0, s = 0.0;
        T e = one_<T>();
        if (mag > 1e-300) {
          e = unit_conj_phase(gpq);
          // t = sign(tau) / (|tau| + sqrt(1 + tau^2)), tau = (aqq - app) / (2 mag), written with one sqrt, one
          // division and one rsqrt (this scalar chain is the latency of every Jacobi step)
          const double dd = aqq - app, m2 = 2.0 * mag;
          const double t = (dd >= 0.0 ? m2 : -m2) / (fabs(dd) + sqrt(fma(dd, dd, m2 * m2)));
          c = rsqrt(fma(t, t, 1.0));
          s = t * c;
        }
        cs[tid] = c; sn[tid] = s; ph[tid] = e; pp[tid] = p; qq[tid] = q;
      }
      __syncthreads();
      // G <- J^H G J with J = the SB disjoint rotations of this step: the 2x2 block (rows p_i,q_i x columns p_j,q_j)
      // of every (row pair, column pair) is touched by exactly one thread, so the column rotation
      //   x_p' = c x_p - s e x_q ,  x_q' = s x_p + c e x_q            (e = e^{-i phi})
      // and the row rotation  r_p' = c r_p - s conj(e) r_q ,  r_q' = s r_p + c conj(e) r_q  are applied back to back
      // in registers, in place (same arithmetic, in the same order, as two separate passes — one barrier less per step)
      for (int blk = tid; blk < SB * SB; blk += 256) {
        const int ki = blk / SB, kj = blk % SB;
        const int pi = pp[ki], qi = qq[ki], pj = pp[kj], qj = qq[kj];
        const double cjj = cs[kj], sjj = sn[kj], cii = cs[ki], sii = sn[ki];
        const T ej = ph[kj], eic = cj(ph[ki]);
        const T a = g[pi * LD + pj], b = mul(ej, g[pi * LD + qj]), c2 = g[qi * LD + pj], d = mul(ej, g[qi * LD + qj]);
        const T a1 = sub(mulr(a, cjj), mulr(b, sjj)), b1 = add(mulr(a, sjj), mulr(b, cjj));
        const T c1 = sub(mulr(c2, cjj), mulr(d, sjj)), d1 = add(mulr(c2, sjj), mulr(d, cjj));
        const T yc = mul(eic, c1), yd = mul(eic, d1);
        g[pi * LD + pj] = sub(mulr(a1, cii), mulr(yc, sii)); g[qi * LD + pj] = add(mulr(a1, sii), mulr(yc, cii));
        g[pi * LD + qj] = sub(mulr(b1, cii), mulr(yd, sii)); g[qi * LD + qj] = add(mulr(b1, sii), mulr(yd, cii));
      }
      // accumulated eigenvector matrix: column rotations only
      for (int idx = tid; idx < SB * PB; idx += 256) {
        int k = idx / PB, i = idx % PB;
        const double c = cs[k], s = sn[k];
        const T e = ph[k];
        int p = pp[k], q = qq[k];
        T x = rm[i * LD + p], y = mul(e, rm[i * LD + q]);
        rm[i * LD + p] = sub(mulr(x, c), mulr(y, s)); rm[i * LD + q] = add(mulr(x, s), mulr(y, c));
      }
      __syncthreads();
    }
  }
  return max_sweeps;
}

// Diagonalise the PB x PB Hermitian matrix of each pair; write the rotation, clear G for the next round,
// record the largest relative off-diagonal seen BEFORE rotating (sweep convergence measure).  `scale` (device, may be null):
// the herm_jacobi_smem scale of the measure.
// Dynamic shared memory: g[PB][PB+1], rm[PB][PB+1] (T), then cs[SB], sn[SB] (double), ph[SB] (T), pp[SB], qq[SB] (int).
template <typename T, int SB>
__global__ void __launch_bounds__(256) svd_eig_kernel(T* __restrict__ G, T* __restrict__ Rout, unsigned int* conv, double tol_inner,
                                                      int max_inner, const int* skip = nullptr, const double* scale = nullptr) {
  constexpr int PB = Geo<SB>::PB, LD = PB + 1;
  if (skip && *skip) return;
  extern __shared__ __align__(16) unsigned char eig_smem[];
  T* g = reinterpret_cast<T*>(eig_smem);
  T* rm = g + PB * LD;
  double* cs = reinterpret_cast<double*>(rm + PB * LD);
  double* sn = cs + SB;
  T* ph = reinterpret_cast<T*>(sn + SB);          // e^{-i phi} of the pivot (real case: its sign is folded into t instead)
  int* pp = reinterpret_cast<int*>(ph + SB);
  int* qq = pp + SB;
  __shared__ float red[8];
  __shared__ float offmax;
  const int pair = blockIdx.x, tid = threadIdx.x;
  T* gg = G + (int64_t)pair * PB * PB;
  for (int idx = tid; idx < PB * PB; idx += 256) {
    int i = idx / PB, j = idx % PB;
    g[i * LD + j] = gg[idx];
    rm[i * LD + j] = i == j ? one_<T>() : zero_<T>();
    gg[idx] = zero_<T>();
  }
  __syncthreads();
  herm_jacobi_smem<T, SB>(g, rm, cs, sn, ph, pp, qq, red, offmax, conv, tol_inner, max_inner, scale ? *scale : 0.0);
  T* ro = Rout + (int64_t)pair * PB * PB;
  for (int idx = tid; idx < PB * PB; idx += 256) ro[idx] = rm[(idx / PB) * LD + idx % PB];
}
template <typename T, int SB>
static size_t eig_smem_bytes() {
  constexpr int PB = Geo<SB>::PB;
  return 2 * sizeof(T) * PB * (PB + 1) + SB * (2 * sizeof(double) + sizeof(T) + 2 * sizeof(int)) + 16;
}

// X[:, pair columns] <- X[:, pair columns] * R   (X = W or V; column-contiguous with `rows` rows)
template <typename T, int SB>
__global__ void __launch_bounds__(256) svd_update_kernel(T* __restrict__ X, int64_t rows, int nb, int round, const T* __restrict__ Rm,
                                                         const int* skip = nullptr) {
  constexpr int PB = Geo<SB>::PB, RT = Geo<SB>::RT, NCG = 256 / RT, CPT = PB / NCG;   // CPT = 8 outputs per thread
  __shared__ T tile[PB][RT];     // read as tile[k][row]: consecutive threads -> consecutive rows (no padding needed)
  __shared__ T rs[PB][PB];       // read as broadcast
  if (skip && *skip) return;
  const int pair = blockIdx.x;
  int bi, bj;
  rr_pair(nb, round, pair, bi, bj);
  const T* rg = Rm + (int64_t)pair * PB * PB;
  for (int idx = threadIdx.x; idx < PB * PB; idx += 256) rs[idx / PB][idx % PB] = rg[idx];
  const int rr = threadIdx.x & (RT - 1), cg = threadIdx.x / RT;   // RT rows x NCG column groups of CPT
  for (int64_t rb = (int64_t)blockIdx.y * RT; rb < rows; rb += (int64_t)gridDim.y * RT) {
    __syncthreads();
    for (int idx = threadIdx.x; idx < PB * RT; idx += 256) {
      int c = idx / RT, r2 = idx % RT;
      int64_t row = rb + r2;
      tile[c][r2] = row < rows ? X[(int64_t)pair_col<SB>(bi, bj, c) * rows + row] : zero_<T>();
    }
    __syncthreads();
    T out[CPT];
#pragma unroll
    for (int c = 0; c < CPT; ++c) out[c] = zero_<T>();
#pragma unroll 8
    for (int k = 0; k < PB; ++k) {
      T x = tile[k][rr];
#pragma unroll
      for (int c = 0; c < CPT; ++c) fmacc(out[c], x, rs[k][cg * CPT + c]);
    }
    int64_t row = rb + rr;
    if (row < rows) {
#pragma unroll
      for (int c = 0; c < CPT; ++c) X[(int64_t)pair_col<SB>(bi, bj, cg * CPT + c) * rows + row] = out[c];
    }
  }
}

}  // namespace tnb
