// svd.cu — tnb200_svd: thin SVD by blocked one-sided (Hestenes) Jacobi, and the truncation
// count of decompositions.svd (backends/numpy/decompositions.py:21-74; LAPACK gesdd there).
//
// The matrix is copied once into column-contiguous working storage W (tall: rows >= cols; a wide
// input is handled through its transpose).  Columns are grouped in blocks of SB; a sweep visits
// every block pair in a round-robin tournament (nb-1 rounds of nb/2 disjoint pairs, all pairs of
// a round processed concurrently):
//   1. gram   : G = [W_I W_J]^T [W_I W_J]           (2SB x 2SB per pair, split over row chunks)
//   2. eig    : cyclic Jacobi eigen-decomposition of G in shared memory -> rotation R
//   3. update : [W_I W_J] <- [W_I W_J] R,  [V_I V_J] <- [V_I V_J] R
// On convergence (all column pairs orthogonal to tol) sigma_j = |w_j|, U = W / sigma, and the
// triplets are sorted in descending order by a rank-counting kernel.  R is orthogonal to working
// precision, so the method is backward stable regardless of how accurately G was formed.
#include "common.cuh"
#include "cplx.cuh"
#include "jacobi.cuh"
#include <math.h>
#include <stdlib.h>
#include <vector>

namespace tnb {

int copy_strided(const tnb200_tensor_t* src, const tnb200_tensor_t* dst, int conj, cudaStream_t st);

template <typename T, int SB>
__global__ void __launch_bounds__(256) svd_gram_kernel(const T* __restrict__ W, int64_t R, int nb, int round, T* __restrict__ G, int rsplit) {
  constexpr int PB = Geo<SB>::PB, RT = Geo<SB>::RT, TPT = PB / 16;   // 16 x 16 threads, TPT x TPT outputs each
  __shared__ T tile[PB][RT + 1];
  const int pair = blockIdx.x, chunk = blockIdx.y;
  int bi, bj;
  rr_pair(nb, round, pair, bi, bj);
  const int64_t rows_per = ((R + rsplit - 1) / rsplit + RT - 1) / RT * RT;
  const int64_t r0 = chunk * rows_per, r1 = min(R, r0 + rows_per);
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  T acc[TPT][TPT];
#pragma unroll
  for (int a = 0; a < TPT; ++a)
#pragma unroll
    for (int b = 0; b < TPT; ++b) acc[a][b] = zero_<T>();
  for (int64_t rb = r0; rb < r1; rb += RT) {
    for (int idx = threadIdx.x; idx < PB * RT; idx += 256) {
      int c = idx / RT, rr = idx % RT;
      int64_t row = rb + rr;
      tile[c][rr] = row < r1 ? W[(int64_t)pair_col<SB>(bi, bj, c) * R + row] : zero_<T>();
    }
    __syncthreads();
#pragma unroll 4
    for (int rr = 0; rr < RT; ++rr) {
      T av[TPT], bv[TPT];
#pragma unroll
      for (int a = 0; a < TPT; ++a) { av[a] = cj(tile[ty * TPT + a][rr]); bv[a] = tile[tx * TPT + a][rr]; }
#pragma unroll
      for (int a = 0; a < TPT; ++a)
#pragma unroll
        for (int b = 0; b < TPT; ++b) fmacc(acc[a][b], av[a], bv[b]);
    }
    __syncthreads();
  }
  T* g = G + (int64_t)pair * PB * PB;     // G = W^H W (Hermitian)
#pragma unroll
  for (int a = 0; a < TPT; ++a)
#pragma unroll
    for (int b = 0; b < TPT; ++b) atomic_add(&g[(ty * TPT + a) * PB + tx * TPT + b], acc[a][b]);
}

template <typename T>
__global__ void svd_colnorm_kernel(const T* __restrict__ W, int64_t R, int64_t ldw, int ncols, double* __restrict__ sig) {
  const int j = blockIdx.x;
  if (j >= ncols) return;
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < R; i += blockDim.x) acc += ab2(W[(int64_t)j * ldw + i]);
  __shared__ double red[32];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    sig[j] = sqrt(t);
  }
}
// descending rank by counting (stable: ties keep column order)
__global__ void svd_rank_kernel(const double* __restrict__ sig, int n, int* __restrict__ rank) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  double sj = sig[j];
  int r = 0;
  for (int i = 0; i < n; ++i) { double si = sig[i]; r += (si > sj) || (si == sj && i < j); }
  rank[j] = r;
}
// scatter the sorted triplets into the caller's u (m x r), s (r), vh (r x n); `tall` = input had m >= n
template <typename T>
__global__ void svd_finalize_kernel(const T* __restrict__ W, const T* __restrict__ V, const double* __restrict__ sig,
                                    const int* __restrict__ rank, int64_t R, int64_t ldw, int Cn, int Cp, int r_out, int tall,
                                    T* __restrict__ u, int64_t u_s0, int64_t u_s1, double* __restrict__ s, int64_t s_s0,
                                    T* __restrict__ vh, int64_t v_s0, int64_t v_s1) {
  const int j = blockIdx.x;          // working column
  const int k = rank[j];
  if (k >= r_out) return;
  const double sg = sig[j];
  const double inv = sg > 0.0 ? 1.0 / sg : 0.0;
  if (threadIdx.x == 0) s[(int64_t)k * s_s0] = sg;
  // WORK = A (tall) or A^H (wide) = Wn S V^H with Wn = W / sigma.
  //   tall: u = Wn, vh = V^H            wide: A = V S Wn^H  ->  u = V, vh = Wn^H
  for (int64_t i = threadIdx.x; i < R; i += blockDim.x) {
    T val = mulr(W[(int64_t)j * ldw + i], inv);
    if (tall) u[i * u_s0 + (int64_t)k * u_s1] = val; else vh[(int64_t)k * v_s0 + i * v_s1] = cj(val);
  }
  for (int64_t i = threadIdx.x; i < Cn; i += blockDim.x) {
    T val = V[(int64_t)j * Cp + i];
    if (tall) vh[(int64_t)k * v_s0 + i * v_s1] = cj(val); else u[i * u_s0 + (int64_t)k * u_s1] = val;
  }
}
template <typename T>
__global__ void svd_eye_kernel(T* V, int Cp) {
  int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx < (int64_t)Cp * Cp) V[idx] = (idx / Cp == idx % Cp) ? one_<T>() : zero_<T>();
}

template <typename T, int SB>
static int svd_real(const tnb200_tensor_t* a, const tnb200_tensor_t* u, const tnb200_tensor_t* s, const tnb200_tensor_t* vh,
                    int32_t* info_dev, cudaStream_t st) {
  constexpr int PB = Geo<SB>::PB, RT = Geo<SB>::RT;
  const int64_t m = a->shape[0], n = a->shape[1];
  const bool tall = m >= n;
  const int64_t R = tall ? m : n;
  const int Cn = (int)(tall ? n : m);
  const int Cp = (Cn + PB - 1) / PB * PB;
  const int nb = Cp / SB, npairs = nb / 2, rounds = nb - 1;
  if (Cn == 0 || R == 0) return 0;
  T *W = nullptr, *V = nullptr, *G = nullptr, *Rm = nullptr;
  double* sig = nullptr;
  int* rank = nullptr;
  unsigned int* conv = nullptr;
  int rc;
  if ((rc = ws_alloc((void**)&W, sizeof(T) * (size_t)Cp * R, st))) return rc;
  if ((rc = ws_alloc((void**)&V, sizeof(T) * (size_t)Cp * Cp, st))) return rc;
  if ((rc = ws_alloc((void**)&G, sizeof(T) * (size_t)npairs * PB * PB, st))) return rc;
  if ((rc = ws_alloc((void**)&Rm, sizeof(T) * (size_t)npairs * PB * PB, st))) return rc;
  if ((rc = ws_alloc((void**)&sig, sizeof(double) * (size_t)Cp, st))) return rc;
  if ((rc = ws_alloc((void**)&rank, sizeof(int) * (size_t)Cp, st))) return rc;
  if ((rc = ws_alloc((void**)&conv, sizeof(unsigned int) * 64, st))) return rc;
  TNB_CHECK_CUDA(cudaMemsetAsync(W, 0, sizeof(T) * (size_t)Cp * R, st));
  TNB_CHECK_CUDA(cudaMemsetAsync(G, 0, sizeof(T) * (size_t)npairs * PB * PB, st));
  // W[j * R + i] = a[i, j] (tall) or a[j, i] (wide)
  tnb200_tensor_t src = *a, dst;
  if (!tall) { src.shape[0] = a->shape[1]; src.shape[1] = a->shape[0]; src.stride[0] = a->stride[1]; src.stride[1] = a->stride[0]; }
  dst.data = W; dst.dtype = a->dtype; dst.ndim = 2;
  dst.shape[0] = R; dst.shape[1] = Cn; dst.stride[0] = 1; dst.stride[1] = R;
  if ((rc = copy_strided(&src, &dst, tall ? 0 : 1, st))) return rc;   // wide: WORK = A^H (conjugated)
  svd_eye_kernel<T><<<(unsigned)(((int64_t)Cp * Cp + 255) / 256), 256, 0, st>>>(V, Cp);
  count_launch();

  const double eps = 2.220446049250313e-16;
  const double tol = 4.0 * sqrt((double)R) * eps;
  // inner (Gram) eigen-solver: tolerance / sweep cap (env knobs for experiments; the outer criterion is unchanged)
  const char* e_tol = getenv("TNB200_SVD_INNER_TOL");
  const char* e_sw = getenv("TNB200_SVD_INNER_SWEEPS");
  const double tol_inner = e_tol ? atof(e_tol) : 1e-15;
  const int max_inner = e_sw ? atoi(e_sw) : 10;
  int rsplit = (4 * num_sms() + npairs - 1) / npairs;
  int max_split = (int)((R + 4 * RT - 1) / (4 * RT));
  if (rsplit > max_split) rsplit = max_split;
  if (rsplit < 1) rsplit = 1;
  int usplit_w = (int)((R + RT - 1) / RT); if (usplit_w > rsplit * 4) usplit_w = rsplit * 4;
  int usplit_v = (Cp + RT - 1) / RT; if (usplit_v > rsplit * 4) usplit_v = rsplit * 4;
  const size_t eig_bytes = eig_smem_bytes<T, SB>();
  {
    static bool attr_done = false;      // per (T, SB) instantiation
    if (!attr_done) {
      TNB_CHECK_CUDA(cudaFuncSetAttribute(svd_eig_kernel<T, SB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)eig_bytes));
      attr_done = true;
    }
  }
  const int max_sweeps = 40;
  int sweeps = 0, converged = 0;
  unsigned int h_conv = 0;
  for (int sw = 0; sw < max_sweeps; ++sw) {
    TNB_CHECK_CUDA(cudaMemsetAsync(conv, 0, sizeof(unsigned int), st));
    for (int r = 0; r < rounds; ++r) {
      svd_gram_kernel<T, SB><<<dim3(npairs, rsplit), 256, 0, st>>>(W, R, nb, r, G, rsplit);
      svd_eig_kernel<T, SB><<<npairs, 256, eig_bytes, st>>>(G, Rm, conv, tol_inner, max_inner);
      svd_update_kernel<T, SB><<<dim3(npairs, usplit_w), 256, 0, st>>>(W, R, nb, r, Rm);
      svd_update_kernel<T, SB><<<dim3(npairs, usplit_v), 256, 0, st>>>(V, Cp, nb, r, Rm);
    }
    count_launch(4 * rounds);
    TNB_LAUNCH_CHECK();
    TNB_CHECK_CUDA(cudaMemcpyAsync(&h_conv, conv, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
    TNB_CHECK_CUDA(cudaStreamSynchronize(st));
    ++sweeps;
    float off;
    memcpy(&off, &h_conv, 4);
    if ((double)off <= tol) { converged = 1; break; }
  }
  svd_colnorm_kernel<T><<<Cp, 256, 0, st>>>(W, R, R, Cp, sig);
  svd_rank_kernel<<<(Cp + 255) / 256, 256, 0, st>>>(sig, Cp, rank);
  svd_finalize_kernel<T><<<Cp, 256, 0, st>>>(W, V, sig, rank, R, R, Cn, Cp, Cn, tall ? 1 : 0, (T*)u->data, u->stride[0], u->stride[1],
                                             (double*)s->data, s->stride[0], (T*)vh->data, vh->stride[0], vh->stride[1]);
  count_launch(3);
  TNB_LAUNCH_CHECK();
  if (info_dev) {
    int32_t h[4] = {sweeps, converged, 0, 0};
    TNB_CHECK_CUDA(cudaMemcpyAsync(info_dev, h, sizeof(h), cudaMemcpyHostToDevice, st));
    TNB_CHECK_CUDA(cudaStreamSynchronize(st));
  }
  ws_free(W, st); ws_free(V, st); ws_free(G, st); ws_free(Rm, st); ws_free(sig, st); ws_free(rank, st); ws_free(conv, st);
  if (!converged) { set_error("svd: Jacobi did not converge in %d sweeps", max_sweeps); return TNB200_ERR_NOCONV; }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Large real matrices: ONE persistent launch for the whole Jacobi iteration (svd_pair_kernel).
//
// Column blocks of 32, pairs of 64 columns.  A pair is owned, for one round, by a TEAM of C CTAs
// (C = SMs / pairs); member c streams its share of the row tiles (64 rows x 64 columns, staged in
// shared memory by a 4-stage cp.async ring):
//   1. Gram     G_c = P_c^T P_c             DMMA (mma.sync.m8n8k4.f64), partial written to global
//   2. team reduction through per-pair arrival counters (red.release / ld.acquire), every member
//      sums the C partials in rank order -> bit-identical G in every member
//   3. eig      one cyclic two-sided Jacobi sweep of the 64 x 64 Gram in shared memory -> J
//               (every member redundantly: identical inputs, identical code, identical J)
//   4. update   P_c <- P_c J for its rows of W and of V   DMMA, J's fragments held in registers
// Rounds are ordered by per-block version counters (block i is touched by exactly one team per round):
// no grid-wide barrier inside a sweep, one per sweep for the device-side convergence flag.  No host
// synchronisation anywhere: the launch is stream-ordered and graph-capturable.
constexpr int PP_SB = 32, PP_PB = 64, PP_RT = 64, PP_LD = 68, PP_GLD = 65, PP_NST = 4, PP_THREADS = 256;

struct PairParams {
  double* W; int64_t ldw; int ntw;       // W: Cp columns of ldw (= padded rows) doubles; ntw row tiles
  double* V; int64_t ldv; int ntv;       // V: Cp x Cp
  double* gpart;                         // [2][npairs][C][64*64] Gram partials (double-buffered by round parity)
  unsigned* gcount;                      // [npairs] arrivals of partials (monotonic)
  unsigned* done;                        // [nb] block versions: C * (rounds completed)
  unsigned* conv;                        // [max_sweeps] float bits of the largest relative off-diagonal seen in a sweep
  unsigned* bar;                         // grid barrier counter
  int32_t* info;                         // [0] sweeps, [1] converged
  int nb, npairs, C, teams, max_sweeps, inner_sweeps, full_every;
  float tol;
};

__device__ __forceinline__ void cp_async16_cg(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void pp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void pp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void pp_dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_add(unsigned* p, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// thread 0 waits until *p >= target; the block then proceeds (acquire for every thread through the barrier)
__device__ __forceinline__ void pp_wait_counter(const unsigned* p, unsigned target) {
  if (threadIdx.x == 0) {
    unsigned ns = 32;
    while ((int)(ld_acquire_u32(p) - target) < 0) { __nanosleep(ns); if (ns < 1024) ns <<= 1; }
  }
  __syncthreads();
}

// pair k (0..31) of step `step` (0..62) of the round-robin tournament on 64 columns, sorted: division-free
// `cross` schedule: only the 32 x 32 pairs between the two blocks of the pair (column k of block i with column
// (k + step) mod 32 of block j, 32 steps) — the pairs INSIDE a block were rotated when the block was last visited by a full schedule
__device__ __forceinline__ void pp_rr(int step, int k, int& a, int& b, bool cross = false) {
  if (cross) { a = k; b = PP_SB + ((k + step) & (PP_SB - 1)); return; }
  if (k == 0) { a = step; b = PP_PB - 1; return; }
  int x = step + k; if (x >= PP_PB - 1) x -= PP_PB - 1;
  int y = step - k + (PP_PB - 1); if (y >= PP_PB - 1) y -= PP_PB - 1;
  a = x < y ? x : y; b = x < y ? y : x;
}

__global__ void __launch_bounds__(PP_THREADS, 1) svd_pair_kernel(const __grid_constant__ PairParams p) {
  extern __shared__ __align__(16) unsigned char pp_smem[];
  double* tiles = reinterpret_cast<double*>(pp_smem);                 // PP_NST x [64 cols][PP_LD]
  double* jt = tiles + PP_NST * PP_PB * PP_LD;                        // [64][PP_LD]: G (ld 65) during eig, then J^T (ld 68)
  double* rm = jt + PP_PB * PP_LD;                                    // [64][65] accumulated rotation J
  double* cs = rm + PP_PB * PP_GLD;                                   // [32] cos, [32] sin
  double* sn = cs + PP_SB;
  __shared__ float red[8];
  __shared__ float s_off;
  double* g = jt;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int fr = lane >> 2, fk = lane & 3;
  const int team = blockIdx.x / p.C, member = blockIdx.x % p.C;
  const int rounds = p.nb - 1;
  // this member's row tiles of W and of V
  const int tw0 = (int)((int64_t)p.ntw * member / p.C), tw1 = (int)((int64_t)p.ntw * (member + 1) / p.C);
  const int tv0 = (int)((int64_t)p.ntv * member / p.C), tv1 = (int)((int64_t)p.ntv * (member + 1) / p.C);
  const int nw = tw1 - tw0, nv = tv1 - tv0;
  unsigned bar_phase = 0;
  int sweeps_done = 0, converged = 0;
  const uint32_t tiles_s = (uint32_t)__cvta_generic_to_shared(tiles);

  for (int sweep = 0; sweep < p.max_sweeps; ++sweep) {
    for (int r = 0; r < rounds; ++r) {
      const unsigned gr = (unsigned)(sweep * rounds + r);             // global round index
      for (int pair = team; pair < p.npairs; pair += p.teams) {
        int bi, bj;
        rr_pair(p.nb, r, pair, bi, bj);
        // tile t of the combined sequence [W tiles | V tiles] of this member -> stage t % NST
        auto issue = [&](int t, int nwt) {
          const double* X; int64_t ld; int64_t rb;
          if (t < nwt) { X = p.W; ld = p.ldw; rb = (int64_t)(tw0 + t) * PP_RT; }
          else { X = p.V; ld = p.ldv; rb = (int64_t)(tv0 + (t - nwt)) * PP_RT; }
          const uint32_t dst0 = tiles_s + (uint32_t)((t % PP_NST) * PP_PB * PP_LD * 8);
#pragma unroll
          for (int i = 0; i < PP_PB * (PP_RT / 2) / PP_THREADS; ++i) {
            const int id = tid + i * PP_THREADS;
            const int c = id >> 5, ch = id & 31;
            const int col = c < PP_SB ? bi * PP_SB + c : bj * PP_SB + (c - PP_SB);
            cp_async16_cg(dst0 + (uint32_t)((c * PP_LD + ch * 2) * 8), X + (int64_t)col * ld + rb + ch * 2);
          }
        };
        // both blocks must carry the previous round's update
        pp_wait_counter(&p.done[bi], (unsigned)p.C * gr);
        pp_wait_counter(&p.done[bj], (unsigned)p.C * gr);

        // ---------------- 1. Gram partial over this member's W tiles
        double acc[2][4][2];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }
        const int gm = (warp >> 1) * 16, gn = (warp & 1) * 32;       // warp tile 16 x 32 of G
#pragma unroll
        for (int s = 0; s < PP_NST - 1; ++s) { if (s < nw) issue(s, nw); pp_commit(); }
        for (int t = 0; t < nw; ++t) {
          pp_wait<PP_NST - 2>();
          __syncthreads();
          if (t + PP_NST - 1 < nw) issue(t + PP_NST - 1, nw);
          pp_commit();
          const double* tl = tiles + (t % PP_NST) * PP_PB * PP_LD;
#pragma unroll 4
          for (int k4 = 0; k4 < PP_RT; k4 += 4) {
            double af[2], bf[4];
#pragma unroll
            for (int i = 0; i < 2; ++i) af[i] = tl[(gm + i * 8 + fr) * PP_LD + k4 + fk];
#pragma unroll
            for (int j = 0; j < 4; ++j) bf[j] = tl[(gn + j * 8 + fr) * PP_LD + k4 + fk];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) pp_dmma(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
          }
        }
        pp_wait<0>();
        __syncthreads();                                              // every stage is free again
        // prefetch the first update tiles (L2 hits) while the team reduces and rotates
        const int nu = nw + nv;
#pragma unroll
        for (int s = 0; s < PP_NST - 1; ++s) { if (s < nu) issue(s, nw); pp_commit(); }
        {
          double* gp = p.gpart + (((size_t)(gr & 1) * p.npairs + pair) * p.C + member) * (PP_PB * PP_PB);
#pragma unroll
          for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
              __stcg(reinterpret_cast<double2*>(gp + (gm + i * 8 + fr) * PP_PB + gn + j * 8 + 2 * fk), make_double2(acc[i][j][0], acc[i][j][1]));
        }
        __threadfence();
        __syncthreads();
        if (tid == 0) red_release_add(&p.gcount[pair], 1u);
        pp_wait_counter(&p.gcount[pair], (unsigned)p.C * (gr + 1));
        // ---------------- 2. G = sum of the partials, in member order
        {
          const double* g0 = p.gpart + ((size_t)(gr & 1) * p.npairs + pair) * p.C * (PP_PB * PP_PB);
          for (int idx = tid; idx < PP_PB * PP_PB; idx += PP_THREADS) {
            double v = 0.0;
            for (int c = 0; c < p.C; ++c) v += __ldcg(g0 + (size_t)c * (PP_PB * PP_PB) + idx);
            const int i = idx >> 6, j = idx & 63;
            g[i * PP_GLD + j] = v;
            rm[i * PP_GLD + j] = i == j ? 1.0 : 0.0;
          }
        }
        __syncthreads();
        // ---------------- 3. cyclic two-sided Jacobi on G
        bool rotate = true;
        for (int isw = 0; isw < p.inner_sweeps; ++isw) {
          float loc = 0.f;
          for (int idx = tid; idx < PP_PB * PP_PB; idx += PP_THREADS) {
            const int i = idx >> 6, j = idx & 63;
            if (i < j) {
              const double d = g[i * PP_GLD + i] * g[j * PP_GLD + j];
              const double x = g[i * PP_GLD + j];
              if (d > 0.0) loc = fmaxf(loc, (float)(x * x / d));
            }
          }
          for (int o = 16; o > 0; o >>= 1) loc = fmaxf(loc, __shfl_xor_sync(0xffffffffu, loc, o));
          if (lane == 0) red[warp] = loc;
          __syncthreads();
          if (tid == 0) {
            float m = 0.f;
            for (int w = 0; w < 8; ++w) m = fmaxf(m, red[w]);
            m = sqrtf(m);
            s_off = m;
            if (isw == 0 && member == 0) atomicMax(&p.conv[sweep], __float_as_uint(m));
          }
          __syncthreads();
          if (s_off <= p.tol) { if (isw == 0) rotate = false; break; }
          // full cyclic schedule (63 steps) every p.full_every-th round, cross-block schedule (32 steps) otherwise
          const bool cross = p.full_every > 1 && (r % p.full_every) != 0;
          const int nsteps = cross ? PP_SB : PP_PB - 1;
          for (int step = 0; step < nsteps; ++step) {
            if (tid < PP_SB) {
              int a, b;
              pp_rr(step, tid, a, b, cross);
              const double gpq = g[a * PP_GLD + b], app = g[a * PP_GLD + a], aqq = g[b * PP_GLD + b];
              double c = 1.0, s = 0.0;
              if (fabs(gpq) > 1e-300) {
                const double dd = aqq - app, m2 = 2.0 * gpq;
                const double t2 = (dd >= 0.0 ? m2 : -m2) / (fabs(dd) + sqrt(fma(dd, dd, m2 * m2)));
                c = rsqrt(fma(t2, t2, 1.0));
                s = t2 * c;
              }
              cs[tid] = c; sn[tid] = s;
            }
            __syncthreads();
            // G <- J^T G J: the 2 x 2 block (rows p_i,q_i x columns p_j,q_j) belongs to one thread.  Every element is in
            // exactly one block, so all loads of a thread are issued before its first store (the compiler cannot prove that
            // the shared-memory stores do not alias the next block's loads and would serialise the four blocks otherwise).
            {
              const int kj = tid & 31;
              int pj, qj;
              pp_rr(step, kj, pj, qj, cross);
              const double cj2 = cs[kj], sj2 = sn[kj];
              int pi[4], qi[4];
              double ci2[4], si2[4], va[4], vb[4], vc[4], vd[4];
#pragma unroll
              for (int it = 0; it < 4; ++it) {
                const int ki = (tid >> 5) + it * 8;
                pp_rr(step, ki, pi[it], qi[it], cross);
                ci2[it] = cs[ki]; si2[it] = sn[ki];
                va[it] = g[pi[it] * PP_GLD + pj]; vb[it] = g[pi[it] * PP_GLD + qj];
                vc[it] = g[qi[it] * PP_GLD + pj]; vd[it] = g[qi[it] * PP_GLD + qj];
              }
              // the accumulated rotation: J[i][a], J[i][b] for 8 of the 32 rotations
              const int ji = tid & 63;
              int ja_[8], jb_[8];
              double jc[8], js[8], jx[8], jy[8];
#pragma unroll
              for (int it = 0; it < 8; ++it) {
                const int k = (tid >> 6) + it * 4;
                pp_rr(step, k, ja_[it], jb_[it], cross);
                jc[it] = cs[k]; js[it] = sn[k];
                jx[it] = rm[ji * PP_GLD + ja_[it]]; jy[it] = rm[ji * PP_GLD + jb_[it]];
              }
#pragma unroll
              for (int it = 0; it < 4; ++it) {
                const double a1 = va[it] * cj2 - vb[it] * sj2, b1 = va[it] * sj2 + vb[it] * cj2;
                const double c1 = vc[it] * cj2 - vd[it] * sj2, d1 = vc[it] * sj2 + vd[it] * cj2;
                g[pi[it] * PP_GLD + pj] = a1 * ci2[it] - c1 * si2[it]; g[qi[it] * PP_GLD + pj] = a1 * si2[it] + c1 * ci2[it];
                g[pi[it] * PP_GLD + qj] = b1 * ci2[it] - d1 * si2[it]; g[qi[it] * PP_GLD + qj] = b1 * si2[it] + d1 * ci2[it];
              }
#pragma unroll
              for (int it = 0; it < 8; ++it) {
                rm[ji * PP_GLD + ja_[it]] = jx[it] * jc[it] - jy[it] * js[it];
                rm[ji * PP_GLD + jb_[it]] = jx[it] * js[it] + jy[it] * jc[it];
              }
            }
            __syncthreads();
          }
        }
        if (rotate) {
          // ---------------- 4. update: X^T[n][row] = sum_k J^T[n][k] X^T[k][row]; this warp owns 16 output columns n
          for (int idx = tid; idx < PP_PB * PP_PB; idx += PP_THREADS) {
            const int n = idx >> 6, k = idx & 63;
            jt[n * PP_LD + k] = rm[k * PP_GLD + n];                   // (G is dead: same storage)
          }
          __syncthreads();
          const int un = (warp >> 1) * 16, ur = (warp & 1) * 32;     // 16 columns x 32 rows of every tile
          double ja[2][16];
#pragma unroll
          for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int k = 0; k < 16; ++k) ja[i][k] = jt[(un + i * 8 + fr) * PP_LD + k * 4 + fk];
          for (int t = 0; t < nu; ++t) {
            pp_wait<PP_NST - 2>();
            __syncthreads();
            if (t + PP_NST - 1 < nu) issue(t + PP_NST - 1, nw);
            pp_commit();
            const double* tl = tiles + (t % PP_NST) * PP_PB * PP_LD;
            double oc[2][4][2];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) { oc[i][j][0] = 0.0; oc[i][j][1] = 0.0; }
#pragma unroll
            for (int k = 0; k < 16; ++k) {
              double bf[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) bf[j] = tl[(k * 4 + fk) * PP_LD + ur + j * 8 + fr];
#pragma unroll
              for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) pp_dmma(oc[i][j][0], oc[i][j][1], ja[i][k], bf[j]);
            }
            double* X; int64_t ld; int64_t rb;
            if (t < nw) { X = p.W; ld = p.ldw; rb = (int64_t)(tw0 + t) * PP_RT; }
            else { X = p.V; ld = p.ldv; rb = (int64_t)(tv0 + (t - nw)) * PP_RT; }
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              const int c = un + i * 8 + fr;
              const int col = c < PP_SB ? bi * PP_SB + c : bj * PP_SB + (c - PP_SB);
#pragma unroll
              for (int j = 0; j < 4; ++j)
                *reinterpret_cast<double2*>(X + (int64_t)col * ld + rb + ur + j * 8 + 2 * fk) = make_double2(oc[i][j][0], oc[i][j][1]);
            }
          }
          pp_wait<0>();
          __threadfence();
        } else {
          pp_wait<0>();                                               // drop the prefetched tiles
        }
        __syncthreads();
        if (tid == 0) { red_release_add(&p.done[bi], 1u); red_release_add(&p.done[bj], 1u); }
      }
    }
    // ---- end of sweep: everyone has added its measure once all blocks carry version C * rounds * (sweep + 1)
    __syncthreads();
    if (tid == 0) {
      __threadfence();
      red_release_add(p.bar, 1u);
      ++bar_phase;
      unsigned ns = 64;
      while ((int)(ld_acquire_u32(p.bar) - bar_phase * gridDim.x) < 0) { __nanosleep(ns); if (ns < 2048) ns <<= 1; }
      s_off = __uint_as_float(ld_acquire_u32(&p.conv[sweep]));
    }
    __syncthreads();
    sweeps_done = sweep + 1;
    // converged when no pair exceeded the tolerance — or when the largest relative off-diagonal seen (BEFORE its rotation)
    // was below 1e-8: Jacobi converges quadratically, the rotations of this sweep left off-diagonals of order 1e-16 and a
    // further, Gram-only sweep would only confirm it
    if (s_off <= p.tol || s_off <= 1e-8f) { converged = 1; break; }
    __syncthreads();
  }
  if (blockIdx.x == 0 && tid == 0 && p.info) { p.info[0] = sweeps_done; p.info[1] = converged; }
}

static int svd_pair_real(const tnb200_tensor_t* a, const tnb200_tensor_t* u, const tnb200_tensor_t* s, const tnb200_tensor_t* vh,
                         int32_t* info_dev, cudaStream_t st) {
  const int64_t m = a->shape[0], n = a->shape[1];
  const bool tall = m >= n;
  const int64_t R = tall ? m : n;
  const int Cn = (int)(tall ? n : m);
  const int Cp = (Cn + PP_PB - 1) / PP_PB * PP_PB;
  const int64_t Rp = (R + PP_RT - 1) / PP_RT * PP_RT;
  const int nb = Cp / PP_SB, npairs = nb / 2;
  const int sms = num_sms();
  int C = sms / npairs; if (C < 1) C = 1;
  const int ntw = (int)(Rp / PP_RT), ntv = Cp / PP_RT;
  if (C > ntw) C = ntw;
  if (C > ntv) C = ntv;
  int teams = sms / C; if (teams > npairs) teams = npairs;
  const int max_sweeps = 60;
  double *W = nullptr, *V = nullptr, *gpart = nullptr, *sig = nullptr;
  int* rank = nullptr;
  unsigned* ctr = nullptr;
  int32_t* info = nullptr;
  int rc;
  const size_t nctr = (size_t)npairs + nb + max_sweeps + 8;
  if ((rc = ws_alloc((void**)&W, sizeof(double) * (size_t)Cp * Rp, st))) return rc;
  if ((rc = ws_alloc((void**)&V, sizeof(double) * (size_t)Cp * Cp, st))) return rc;
  if ((rc = ws_alloc((void**)&gpart, sizeof(double) * 2 * (size_t)npairs * C * PP_PB * PP_PB, st))) return rc;
  if ((rc = ws_alloc((void**)&sig, sizeof(double) * (size_t)Cp, st))) return rc;
  if ((rc = ws_alloc((void**)&rank, sizeof(int) * (size_t)Cp, st))) return rc;
  if ((rc = ws_alloc((void**)&ctr, sizeof(unsigned) * nctr, st))) return rc;
  if ((rc = ws_alloc((void**)&info, sizeof(int32_t) * 4, st))) return rc;
  TNB_CHECK_CUDA(cudaMemsetAsync(W, 0, sizeof(double) * (size_t)Cp * Rp, st));
  TNB_CHECK_CUDA(cudaMemsetAsync(ctr, 0, sizeof(unsigned) * nctr, st));
  TNB_CHECK_CUDA(cudaMemsetAsync(info, 0, sizeof(int32_t) * 4, st));
  tnb200_tensor_t src = *a, dst;
  if (!tall) { src.shape[0] = a->shape[1]; src.shape[1] = a->shape[0]; src.stride[0] = a->stride[1]; src.stride[1] = a->stride[0]; }
  dst.data = W; dst.dtype = a->dtype; dst.ndim = 2;
  dst.shape[0] = R; dst.shape[1] = Cn; dst.stride[0] = 1; dst.stride[1] = Rp;
  if ((rc = copy_strided(&src, &dst, 0, st))) return rc;
  svd_eye_kernel<double><<<(unsigned)(((int64_t)Cp * Cp + 255) / 256), 256, 0, st>>>(V, Cp);
  count_launch();

  PairParams p;
  p.W = W; p.ldw = Rp; p.ntw = ntw; p.V = V; p.ldv = Cp; p.ntv = ntv;
  p.gpart = gpart; p.gcount = ctr; p.done = ctr + npairs; p.conv = ctr + npairs + nb; p.bar = ctr + npairs + nb + max_sweeps;
  p.info = info_dev ? info_dev : info;
  p.nb = nb; p.npairs = npairs; p.C = C; p.teams = teams; p.max_sweeps = max_sweeps;
  const char* e_sw = getenv("TNB200_SVD_INNER_SWEEPS");
  p.inner_sweeps = e_sw ? atoi(e_sw) : 1;
  if (p.inner_sweeps < 1) p.inner_sweeps = 1;
  // rotation schedule inside a pair: the full 64-column cyclic sweep every 4th round, only the 32 x 32 cross-block pairs in
  // between (numpy model of this kernel, n = 1024: 15 sweeps either way; cross-only in ALL but the first round: 16)
  const char* e_fe = getenv("TNB200_SVD_FULL_EVERY");
  p.full_every = e_fe ? atoi(e_fe) : 4;
  if (p.full_every < 1) p.full_every = 1;
  p.tol = (float)(4.0 * sqrt((double)R) * 2.220446049250313e-16);
  const size_t smem = sizeof(double) * ((size_t)PP_NST * PP_PB * PP_LD + PP_PB * PP_LD + PP_PB * PP_GLD + 2 * PP_SB) + sizeof(int) * 2 * PP_SB + 16;
  static bool attr_done = false;
  if (!attr_done) {
    TNB_CHECK_CUDA(cudaFuncSetAttribute(svd_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_done = true;
  }
  int per_sm = 0;
  TNB_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, svd_pair_kernel, PP_THREADS, smem));
  if (per_sm < 1 || teams * C > per_sm * sms) { set_error("svd: persistent kernel does not fit (%d CTAs)", teams * C); return TNB200_ERR_UNSUPPORTED; }
  void* args[] = {(void*)&p};
  // cooperative launch: every CTA must be resident (the teams wait on each other)
  TNB_CHECK_CUDA(cudaLaunchCooperativeKernel((const void*)svd_pair_kernel, dim3((unsigned)(teams * C)), dim3(PP_THREADS), args, smem, st));
  count_launch();
  svd_colnorm_kernel<double><<<Cp, 256, 0, st>>>(W, R, Rp, Cp, sig);
  svd_rank_kernel<<<(Cp + 255) / 256, 256, 0, st>>>(sig, Cp, rank);
  svd_finalize_kernel<double><<<Cp, 256, 0, st>>>(W, V, sig, rank, R, Rp, Cn, Cp, Cn, tall ? 1 : 0, (double*)u->data, u->stride[0], u->stride[1],
                                                  (double*)s->data, s->stride[0], (double*)vh->data, vh->stride[0], vh->stride[1]);
  count_launch(3);
  TNB_LAUNCH_CHECK();
  ws_free(W, st); ws_free(V, st); ws_free(gpart, st); ws_free(sig, st); ws_free(rank, st); ws_free(ctr, st); ws_free(info, st);
  return 0;
}

// decompositions.py:38-57 on the device, in the arithmetic type of `s` (sequential cumsum like numpy)
template <typename T>
__global__ void svd_trunc_kernel(const T* __restrict__ s, int64_t n, int64_t stride, int64_t max_sv, int use_err, double max_err,
                                 int relative, long long* keep) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  long long by_err = max_sv;
  if (use_err) {
    T eps = relative ? (T)((T)max_err * s[0]) : (T)max_err;
    T cum = T(0);
    long long cnt = 0;
    for (int64_t i = n - 1; i >= 0; --i) {
      T v = s[i * stride];
      cum = cum + v * v;
      if (sqrt(cum) > eps) ++cnt;
    }
    by_err = cnt;
  }
  *keep = max_sv < by_err ? max_sv : by_err;
}

}  // namespace tnb

using namespace tnb;

// Block width: 16.  The 32-wide variant (half the rounds per sweep, i.e. half the HBM traffic of the gram / update
// kernels) is kept for real dtypes behind TNB200_SVD_SB=32, but it is SLOWER on B200 — measured 2048^2: 0.57 s vs
// 0.37 s, 4096^2: 2.20 s vs 2.06 s, same sweep counts — because the 64 x 64 Gram eigenproblem (63 dependent Jacobi
// steps per inner sweep in one CTA) then dominates every round.
static int svd_dispatch(bool cplx, const tnb200_tensor_t* a, const tnb200_tensor_t* u, const tnb200_tensor_t* s, const tnb200_tensor_t* vh,
                        int32_t* info_dev, cudaStream_t st) {
  if (cplx) return svd_real<zd, 16>(a, u, s, vh, info_dev, st);
  const int64_t cn = a->shape[0] < a->shape[1] ? a->shape[0] : a->shape[1];
  int sb = 16;
  const char* algo = getenv("TNB200_SVD_ALGO");       // "rounds" = the launch-per-round kernels below
  if (cn >= 256 && !(algo && !strcmp(algo, "rounds"))) {
    set_kernel_name("svd_pair_persistent");
    return svd_pair_real(a, u, s, vh, info_dev, st);
  }
  if (const char* e = getenv("TNB200_SVD_SB")) { const int v = atoi(e); if (v == 16 || v == 32) sb = v; }
  return sb == 32 ? svd_real<double, 32>(a, u, s, vh, info_dev, st) : svd_real<double, 16>(a, u, s, vh, info_dev, st);
}

extern "C" int32_t tnb200_svd(const tnb200_tensor_t* a, const tnb200_tensor_t* u, const tnb200_tensor_t* s, const tnb200_tensor_t* vh,
                              int32_t* info_dev, void* stream) {
  TNB_REQUIRE(valid_tensor(a) && valid_tensor(u) && valid_tensor(s) && valid_tensor(vh), TNB200_ERR_INVALID, "svd: invalid tensor descriptor");
  TNB_REQUIRE(a->ndim == 2 && u->ndim == 2 && vh->ndim == 2 && s->ndim == 1, TNB200_ERR_INVALID, "svd: expects matrix arguments");
  TNB_REQUIRE(a->dtype != TNB200_BOOL, TNB200_ERR_DTYPE, "svd: bool tensors are not supported");
  const int64_t m = a->shape[0], n = a->shape[1], r = m < n ? m : n;
  TNB_REQUIRE(u->shape[0] == m && u->shape[1] == r && vh->shape[0] == r && vh->shape[1] == n && s->shape[0] == r, TNB200_ERR_INVALID,
              "svd: output shapes must be (m,r), (r,), (r,n) with r = min(m,n)");
  TNB_REQUIRE(u->dtype == a->dtype && vh->dtype == a->dtype, TNB200_ERR_DTYPE, "svd: u/vh dtype must equal the input dtype");
  TNB_REQUIRE(m < (1LL << 31) && n < (1LL << 31), TNB200_ERR_UNSUPPORTED, "svd: matrix too large");
  cudaStream_t st = (cudaStream_t)stream;
  set_kernel_name("svd_block_jacobi");
  if (a->dtype == TNB200_F64) { TNB_REQUIRE(s->dtype == TNB200_F64, TNB200_ERR_DTYPE, "svd: s must be f64"); return svd_dispatch(false, a, u, s, vh, info_dev, st); }
  if (a->dtype == TNB200_C128) { TNB_REQUIRE(s->dtype == TNB200_F64, TNB200_ERR_DTYPE, "svd: s must be f64"); return svd_dispatch(true, a, u, s, vh, info_dev, st); }
  if (a->dtype == TNB200_F32 || a->dtype == TNB200_C64) {
    // single precision input: iterate in double (hundreds of accumulated plane rotations cost ~1e-5
    // relative accuracy in fp32, LAPACK's sgesdd delivers ~1e-6), then round the factors back.
    const bool cplx = a->dtype == TNB200_C64;
    TNB_REQUIRE(s->dtype == TNB200_F32, TNB200_ERR_DTYPE, "svd: s must be f32");
    const int wide_dt = cplx ? TNB200_C128 : TNB200_F64;
    const size_t esz = cplx ? 16 : 8;
    void *da = nullptr, *du = nullptr, *dv = nullptr;
    double* ds = nullptr;
    int rc;
    if ((rc = ws_alloc(&da, esz * (size_t)m * n, st))) return rc;
    if ((rc = ws_alloc(&du, esz * (size_t)m * r, st))) return rc;
    if ((rc = ws_alloc((void**)&ds, sizeof(double) * (size_t)r, st))) return rc;
    if ((rc = ws_alloc(&dv, esz * (size_t)r * n, st))) return rc;
    auto mk = [](void* p, int dt, int64_t d0, int64_t d1, int nd) {
      tnb200_tensor_t t; t.data = p; t.dtype = dt; t.ndim = nd;
      t.shape[0] = d0; t.shape[1] = d1; t.stride[0] = nd == 2 ? d1 : 1; t.stride[1] = 1; return t;
    };
    tnb200_tensor_t ta = mk(da, wide_dt, m, n, 2), tu = mk(du, wide_dt, m, r, 2), ts = mk(ds, TNB200_F64, r, 1, 1), tv = mk(dv, wide_dt, r, n, 2);
    if ((rc = copy_strided(a, &ta, 0, st))) return rc;
    rc = svd_dispatch(cplx, &ta, &tu, &ts, &tv, info_dev, st);
    if (rc == 0) rc = copy_strided(&tu, u, 0, st);
    if (rc == 0) rc = copy_strided(&ts, s, 0, st);
    if (rc == 0) rc = copy_strided(&tv, vh, 0, st);
    ws_free(da, st); ws_free(du, st); ws_free(ds, st); ws_free(dv, st);
    return rc;
  }
  set_error("svd: dtype %s is not supported (f32/f64/c64/c128)", dtype_name(a->dtype));
  return TNB200_ERR_UNSUPPORTED;
}

extern "C" int32_t tnb200_svd_truncation_count(const tnb200_tensor_t* s, int64_t max_singular_values, int32_t use_error,
                                               double max_truncation_error, int32_t relative, int64_t* keep_dev, void* stream) {
  TNB_REQUIRE(valid_tensor(s) && s->ndim == 1 && keep_dev, TNB200_ERR_INVALID, "svd_truncation_count: invalid arguments");
  const int64_t n = s->shape[0];
  int64_t max_sv = max_singular_values < 0 ? n : max_singular_values;
  cudaStream_t st = (cudaStream_t)stream;
  if (s->dtype == TNB200_F64)
    svd_trunc_kernel<double><<<1, 32, 0, st>>>((const double*)s->data, n, s->stride[0], max_sv, use_error, max_truncation_error, relative, (long long*)keep_dev);
  else if (s->dtype == TNB200_F32)
    svd_trunc_kernel<float><<<1, 32, 0, st>>>((const float*)s->data, n, s->stride[0], max_sv, use_error, max_truncation_error, relative, (long long*)keep_dev);
  else { set_error("svd_truncation_count: s must be f32/f64"); return TNB200_ERR_DTYPE; }
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}
