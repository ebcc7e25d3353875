// tensordot.cu — tnb200_tensordot: planner (mode classification, operand repacking, kernel
// choice) + the generic strided CUDA-core kernel that serves every dtype and every layout.
//
// Replaces NumPyBackend.tensordot (backends/numpy/numpy_backend.py:35-54) and the batched
// matmul of ncon's _batch_cont (ncon_interface.py:280-354).  np.tensordot materialises
// transposed copies of both operands and calls BLAS; here the operand permutation is folded
// into the kernel's address computation (SIMT path) or into TMA tensor maps (tcgen05 path).
#include "gemm.cuh"
#include <algorithm>
#include <vector>

namespace tnb {

int copy_strided(const tnb200_tensor_t* src, const tnb200_tensor_t* dst, int conj, cudaStream_t st);
int tensordot_thin(int dt, const void* A, const void* B, void* C, const ModeList& mB, const ModeList& mM,
                   const ModeList& mN, const ModeList& mK, bool allow_tf32, cudaStream_t st);
int tensordot_skinny(int dt, const void* A, const void* B, void* C, const ModeList& mB, const ModeList& mM,
                     const ModeList& mN, const ModeList& mK, cudaStream_t st);

// --------------------------------------------------------------------------- SIMT kernel
template <typename T>
struct SimtParams {
  const T* A; const T* B; T* C;
  DevModes mB;  // batch modes : s0 = A, s1 = B, s2 = C
  DevModes mM;  // free A modes: s0 = A, s1 = C
  DevModes mN;  // free B modes: s0 = B, s1 = C
  DevModes mK;  // summed modes: s0 = A, s1 = B
  int64_t M, N, K, batch;
  int conjA, conjB, a_kfast, b_nfast;
  int ksplit;          // > 1: grid.y K-chunks accumulate atomically into `acc_ws` ([batch, M, N] of Acc)
  int64_t kchunk;
  void* acc_ws;
};

constexpr int SBM = 64, SBN = 64, SBK = 16;

__device__ inline void atomic_acc(double* p, double v) { atomicAdd(p, v); }
__device__ inline void atomic_acc(float* p, float v) { atomicAdd(p, v); }
__device__ inline void atomic_acc(int32_t* p, int32_t v) { atomicAdd(p, v); }
__device__ inline void atomic_acc(long long* p, long long v) { atomicAdd((unsigned long long*)p, (unsigned long long)v); }
__device__ inline void atomic_acc(cuFloatComplex* p, cuFloatComplex v) { atomicAdd(&p->x, v.x); atomicAdd(&p->y, v.y); }
__device__ inline void atomic_acc(cuDoubleComplex* p, cuDoubleComplex v) { atomicAdd(&p->x, v.x); atomicAdd(&p->y, v.y); }

template <typename T, typename Acc>
__global__ void __launch_bounds__(256) tensordot_simt_kernel(const __grid_constant__ SimtParams<T> p) {
  __shared__ Acc As[SBK][SBM + 1];
  __shared__ Acc Bs[SBK][SBN + 1];
  const int64_t tilesM = (p.M + SBM - 1) / SBM, tilesN = (p.N + SBN - 1) / SBN;
  int64_t bid = blockIdx.x;
  const int64_t tn = bid % tilesN; bid /= tilesN;
  const int64_t tm = bid % tilesM;
  const int64_t bb = bid / tilesM;
  int64_t offAb, offBb, offCb;
  mode_offsets3(p.mB, bb, offAb, offBb, offCb);
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;

  int am[4], ak[4], bn[4], bk[4];
  int64_t aoff[4], boff[4];
  bool aval[4], bval[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int idx = t + 256 * i;
    if (p.a_kfast) { ak[i] = idx & 15; am[i] = idx >> 4; } else { am[i] = idx & 63; ak[i] = idx >> 6; }
    if (p.b_nfast) { bn[i] = idx & 63; bk[i] = idx >> 6; } else { bk[i] = idx & 15; bn[i] = idx >> 4; }
    int64_t m = tm * SBM + am[i], n = tn * SBN + bn[i];
    aval[i] = m < p.M; bval[i] = n < p.N;
    aoff[i] = aval[i] ? offAb + mode_offset0(p.mM, m) : 0;
    boff[i] = bval[i] ? offBb + mode_offset0(p.mN, n) : 0;
  }
  Acc acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = acc_zero((Acc*)nullptr);

  const int64_t kbeg = p.ksplit > 1 ? (int64_t)blockIdx.y * p.kchunk : 0;
  const int64_t kend = p.ksplit > 1 ? (kbeg + p.kchunk < p.K ? kbeg + p.kchunk : p.K) : p.K;
  for (int64_t k0 = kbeg; k0 < kend; k0 += SBK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      Acc v = acc_zero((Acc*)nullptr);
      int64_t k = k0 + ak[i];
      if (aval[i] && k < kend) {
        int64_t ko, ko1;
        if (p.mK.n <= 1) ko = k * p.mK.s0[0]; else mode_offsets(p.mK, k, ko, ko1);
        v = to_acc(p.A[aoff[i] + ko]);
        if (p.conjA) v = conj_acc(v);
      }
      As[ak[i]][am[i]] = v;
      Acc w = acc_zero((Acc*)nullptr);
      k = k0 + bk[i];
      if (bval[i] && k < kend) {
        int64_t ko, ko1;
        if (p.mK.n <= 1) ko1 = k * p.mK.s1[0]; else mode_offsets(p.mK, k, ko, ko1);
        w = to_acc(p.B[boff[i] + ko1]);
        if (p.conjB) w = conj_acc(w);
      }
      Bs[bk[i]][bn[i]] = w;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < SBK; ++kk) {
      Acc a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[kk][ty + 16 * i]; b[i] = Bs[kk][tx + 16 * i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) fma_acc(acc[i][j], a[i], b[j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int64_t m = tm * SBM + ty + 16 * i;
    if (m >= p.M) continue;
    int64_t oa, ocm;
    mode_offsets(p.mM, m, oa, ocm);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int64_t n = tn * SBN + tx + 16 * j;
      if (n >= p.N) continue;
      int64_t ob, ocn;
      mode_offsets(p.mN, n, ob, ocn);
      if (p.ksplit > 1) atomic_acc((Acc*)p.acc_ws + (bb * p.M + m) * p.N + n, acc[i][j]);
      else p.C[offCb + ocm + ocn] = FromAcc<T, Acc>::f(acc[i][j]);
    }
  }
}

// split-K epilogue: C[...] = convert(acc_ws[b, m, n])
template <typename T, typename Acc>
__global__ void splitk_finalize_kernel(const __grid_constant__ SimtParams<T> p) {
  const int64_t total = p.batch * p.M * p.N;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t n = i % p.N, t = i / p.N, m = t % p.M, bb = t / p.M;
    int64_t oa, ob, oc, o1, ocm, o2, ocn;
    mode_offsets3(p.mB, bb, oa, ob, oc);
    mode_offsets(p.mM, m, o1, ocm);
    mode_offsets(p.mN, n, o2, ocn);
    p.C[oc + ocm + ocn] = FromAcc<T, Acc>::f(((const Acc*)p.acc_ws)[i]);
  }
}

template <int DT>
static int launch_simt(const void* A, const void* B, void* C, const ModeList& mB, const ModeList& mM,
                       const ModeList& mN, const ModeList& mK, bool conjA, bool conjB, cudaStream_t st) {
  using T = typename DType<DT>::T;
  using Acc = typename DType<DT>::Acc;
  SimtParams<T> p;
  p.A = (const T*)A; p.B = (const T*)B; p.C = (T*)C;
  if (!to_dev(mB, p.mB) || !to_dev(mM, p.mM) || !to_dev(mN, p.mN) || !to_dev(mK, p.mK)) {
    set_error("tensordot: more than %d non-mergeable modes in one group", kDevModes);
    return TNB200_ERR_UNSUPPORTED;
  }
  p.M = mM.total(); p.N = mN.total(); p.K = mK.total(); p.batch = mB.total();
  p.conjA = conjA; p.conjB = conjB;
  auto last_stride = [](const ModeList& m, int which) -> int64_t {
    if (m.n == 0) return INT64_MAX;
    int64_t s = which == 0 ? m.s0[m.n - 1] : m.s1[m.n - 1];
    return s < 0 ? -s : s;
  };
  p.a_kfast = last_stride(mK, 0) <= last_stride(mM, 0);
  p.b_nfast = last_stride(mN, 0) <= last_stride(mK, 1);
  int64_t tiles = ((p.M + SBM - 1) / SBM) * ((p.N + SBN - 1) / SBN) * p.batch;
  TNB_REQUIRE(tiles < (1LL << 31), TNB200_ERR_UNSUPPORTED, "tensordot: output too large for one launch");
  // split-K when the output is too small to fill the GPU but the contraction is long
  p.ksplit = 1; p.kchunk = p.K; p.acc_ws = nullptr;
  const int sms = num_sms();
  if (tiles * 2 <= sms && p.K >= 2048) {
    int64_t want = (2 * sms + tiles - 1) / tiles;
    int64_t maxs = p.K / 512;
    int64_t sp = want < maxs ? want : maxs;
    if (sp > 1) {
      p.kchunk = ((p.K + sp - 1) / sp + SBK - 1) / SBK * SBK;
      p.ksplit = (int)((p.K + p.kchunk - 1) / p.kchunk);
    }
  }
  if (p.ksplit > 1) {
    size_t bytes = sizeof(Acc) * (size_t)(p.batch * p.M * p.N);
    int rc = ws_alloc(&p.acc_ws, bytes, st);
    if (rc) return rc;
    TNB_CHECK_CUDA(cudaMemsetAsync(p.acc_ws, 0, bytes, st));
    tensordot_simt_kernel<T, Acc><<<dim3((unsigned)tiles, (unsigned)p.ksplit), 256, 0, st>>>(p);
    int64_t tot = p.batch * p.M * p.N;
    int64_t fb = (tot + 255) / 256; if (fb > sms * 8) fb = sms * 8;
    splitk_finalize_kernel<T, Acc><<<(unsigned)fb, 256, 0, st>>>(p);
    TNB_LAUNCH_CHECK();
    count_launch(2);
    set_kernel_name("simt_splitk");
    return ws_free(p.acc_ws, st);
  }
  tensordot_simt_kernel<T, Acc><<<(unsigned)tiles, 256, 0, st>>>(p);
  TNB_LAUNCH_CHECK();
  count_launch();
  return 0;
}

static int dispatch_simt(int dt, const void* A, const void* B, void* C, const ModeList& mB,
                         const ModeList& mM, const ModeList& mN, const ModeList& mK, bool cA, bool cB,
                         cudaStream_t st) {
  set_kernel_name("simt");
  switch (dt) {
    case TNB200_F64: return launch_simt<TNB200_F64>(A, B, C, mB, mM, mN, mK, cA, cB, st);
    case TNB200_F32: return launch_simt<TNB200_F32>(A, B, C, mB, mM, mN, mK, cA, cB, st);
    case TNB200_F16: return launch_simt<TNB200_F16>(A, B, C, mB, mM, mN, mK, cA, cB, st);
    case TNB200_BF16: return launch_simt<TNB200_BF16>(A, B, C, mB, mM, mN, mK, cA, cB, st);
    case TNB200_C64: return launch_simt<TNB200_C64>(A, B, C, mB, mM, mN, mK, cA, cB, st);
    case TNB200_C128: return launch_simt<TNB200_C128>(A, B, C, mB, mM, mN, mK, cA, cB, st);
    case TNB200_I32: return launch_simt<TNB200_I32>(A, B, C, mB, mM, mN, mK, cA, cB, st);
    case TNB200_I64: return launch_simt<TNB200_I64>(A, B, C, mB, mM, mN, mK, cA, cB, st);
  }
  set_error("tensordot: bad dtype %d", dt);
  return TNB200_ERR_DTYPE;
}

// ------------------------------------------------------------------------------ planner
struct KMode { int64_t ext, sa, sb; };

// collapse one operand's view of a mode group to "single stride or not"
static bool single_mode(const ModeList& in, int which, int64_t& ext, int64_t& stride) {
  ModeList m;
  for (int i = 0; i < in.n; ++i) m.push(in.ext[i], which == 0 ? in.s0[i] : (which == 1 ? in.s1[i] : in.s2[i]));
  merge_modes(m, 1);
  if (m.n > 1) return false;
  ext = m.n ? m.ext[0] : 1;
  stride = m.n ? m.s0[0] : 0;
  return true;
}

static ModeList order_k(const ModeList& mK, int by) {
  std::vector<int> idx(mK.n);
  for (int i = 0; i < mK.n; ++i) idx[i] = i;
  std::stable_sort(idx.begin(), idx.end(), [&](int x, int y) {
    int64_t sx = by == 0 ? mK.s0[x] : mK.s1[x], sy = by == 0 ? mK.s0[y] : mK.s1[y];
    return llabs(sx) > llabs(sy);
  });
  ModeList r;
  for (int i : idx) r.push(mK.ext[i], mK.s0[i], mK.s1[i]);
  return r;
}

// Pack a (batch, free, K) view of one operand into a contiguous row-major [batch, free, K]
// scratch buffer with the strided-copy kernel (the only place a transpose is materialised).
static int pack_operand(int dt, const void* src, const ModeList& mB, int wb, const ModeList& mF,
                        const ModeList& mK, int wk, void** out, int64_t* pitch, cudaStream_t st) {
  tnb200_tensor_t s, d;
  s.data = const_cast<void*>(src); s.dtype = dt; d.dtype = dt;
  int nd = 0;
  auto add = [&](const ModeList& m, int which) -> bool {
    for (int i = 0; i < m.n; ++i) {
      if (nd >= TNB200_MAX_NDIM) return false;
      s.shape[nd] = m.ext[i];
      s.stride[nd] = which == 0 ? m.s0[i] : (which == 1 ? m.s1[i] : m.s2[i]);
      ++nd;
    }
    return true;
  };
  if (!add(mB, wb) || !add(mF, 0) || !add(mK, wk)) {
    set_error("tensordot: too many modes to pack");
    return TNB200_ERR_UNSUPPORTED;
  }
  s.ndim = d.ndim = nd;
  // contiguous [batch, free, K] with the K row padded to a 16-byte multiple (`pitch` elements)
  int64_t ktot = mK.total(), ftot = mF.total();
  const int64_t per16 = 16 / dtype_size(dt) > 0 ? 16 / dtype_size(dt) : 1;
  const int64_t kp = (ktot + per16 - 1) / per16 * per16;
  *pitch = kp;
  int64_t tot = 1;
  {
    // strides of the destination modes: K modes contiguous, free modes over the padded pitch
    int idx = nd - 1;
    int64_t st_ = 1;
    for (int i = mK.n - 1; i >= 0; --i, --idx) { d.shape[idx] = s.shape[idx]; d.stride[idx] = st_; st_ *= s.shape[idx]; }
    st_ = kp;
    for (int i = mF.n - 1; i >= 0; --i, --idx) { d.shape[idx] = s.shape[idx]; d.stride[idx] = st_; st_ *= s.shape[idx]; }
    st_ = kp * ftot;
    for (int i = mB.n - 1; i >= 0; --i, --idx) { d.shape[idx] = s.shape[idx]; d.stride[idx] = st_; st_ *= s.shape[idx]; }
    tot = kp * ftot * mB.total();
  }
  int rc = ws_alloc(out, (size_t)tot * dtype_size(dt), st);
  if (rc) return rc;
  d.data = *out;
  return copy_strided(&s, &d, 0, st);
}

}  // namespace tnb

using namespace tnb;

namespace tnb {
// Validate a contraction request and classify its axes into batch / free-A (M) / free-B (N) / contracted (K)
// mode lists (np.tensordot output order: batch axes, free axes of a, free axes of b).
int build_modes(const tnb200_tensor_t* a, const tnb200_tensor_t* b, const tnb200_tensor_t* c, int32_t naxes,
                const int32_t* axes_a, const int32_t* axes_b, int32_t nbatch, const int32_t* batch_a,
                const int32_t* batch_b, ModeList& mB, ModeList& mM, ModeList& mN, ModeList& mK) {
  TNB_REQUIRE(valid_tensor(a) && valid_tensor(b) && valid_tensor(c), TNB200_ERR_INVALID,
              "tensordot: invalid tensor descriptor");
  TNB_REQUIRE(a->dtype != TNB200_BOOL, TNB200_ERR_DTYPE, "tensordot: bool tensors are not supported");
  TNB_REQUIRE(a->dtype == b->dtype && a->dtype == c->dtype, TNB200_ERR_DTYPE,
              "tensordot: dtype mismatch (%s, %s -> %s)", dtype_name(a->dtype), dtype_name(b->dtype),
              dtype_name(c->dtype));
  TNB_REQUIRE(naxes >= 0 && nbatch >= 0 && naxes + nbatch <= a->ndim && naxes + nbatch <= b->ndim,
              TNB200_ERR_INVALID, "tensordot: too many axes");
  int role_a[TNB200_MAX_NDIM] = {0}, role_b[TNB200_MAX_NDIM] = {0};  // 0 free, 1 summed, 2 batch
  mB = ModeList(); mM = ModeList(); mN = ModeList(); mK = ModeList();
  for (int i = 0; i < naxes; ++i) {
    int x = axes_a[i], y = axes_b[i];
    if (x < 0) x += a->ndim;
    if (y < 0) y += b->ndim;
    TNB_REQUIRE(x >= 0 && x < a->ndim && y >= 0 && y < b->ndim && !role_a[x] && !role_b[y],
                TNB200_ERR_INVALID, "tensordot: bad or repeated axis");
    TNB_REQUIRE(a->shape[x] == b->shape[y], TNB200_ERR_INVALID, "shape-mismatch for sum");
    role_a[x] = 1; role_b[y] = 1;
    mK.push(a->shape[x], a->stride[x], b->stride[y]);
  }
  int cax = 0;
  for (int i = 0; i < nbatch; ++i) {
    int x = batch_a[i], y = batch_b[i];
    if (x < 0) x += a->ndim;
    if (y < 0) y += b->ndim;
    TNB_REQUIRE(x >= 0 && x < a->ndim && y >= 0 && y < b->ndim && !role_a[x] && !role_b[y],
                TNB200_ERR_INVALID, "tensordot: bad or repeated batch axis");
    TNB_REQUIRE(a->shape[x] == b->shape[y], TNB200_ERR_INVALID, "tensordot: batch extent mismatch");
    role_a[x] = 2; role_b[y] = 2;
    TNB_REQUIRE(cax < c->ndim && c->shape[cax] == a->shape[x], TNB200_ERR_INVALID,
                "tensordot: output shape mismatch (batch axis %d)", i);
    mB.push(a->shape[x], a->stride[x], b->stride[y], c->stride[cax]);
    ++cax;
  }
  for (int i = 0; i < a->ndim; ++i)
    if (!role_a[i]) {
      TNB_REQUIRE(cax < c->ndim && c->shape[cax] == a->shape[i], TNB200_ERR_INVALID,
                  "tensordot: output shape mismatch at output axis %d", cax);
      mM.push(a->shape[i], a->stride[i], c->stride[cax]);
      ++cax;
    }
  for (int i = 0; i < b->ndim; ++i)
    if (!role_b[i]) {
      TNB_REQUIRE(cax < c->ndim && c->shape[cax] == b->shape[i], TNB200_ERR_INVALID,
                  "tensordot: output shape mismatch at output axis %d", cax);
      mN.push(b->shape[i], b->stride[i], c->stride[cax]);
      ++cax;
    }
  TNB_REQUIRE(cax == c->ndim, TNB200_ERR_INVALID, "tensordot: output rank mismatch (%d vs %d)", cax,
              c->ndim);

  return 0;
}

// Lower a contraction to a GEMM whose operands are BOTH addressable in place by the TMA / tcgen05 path
// (no repack, no skinny / thin special case).  Used by the chained-GEMM planner (gemm_chain.cu).
int plan_inplace_gemm(const tnb200_tensor_t* a, const tnb200_tensor_t* b, const tnb200_tensor_t* c, int32_t naxes,
                      const int32_t* axes_a, const int32_t* axes_b, int32_t nbatch, const int32_t* batch_a,
                      const int32_t* batch_b, GemmProblem& g) {
  ModeList mB, mM, mN, mK;
  int rc = build_modes(a, b, c, naxes, axes_a, axes_b, nbatch, batch_a, batch_b, mB, mM, mN, mK);
  if (rc) return rc;
  const int dt = a->dtype;
  if (dt != TNB200_F32 && dt != TNB200_F16 && dt != TNB200_BF16) return TNB200_ERR_UNSUPPORTED;
  const int64_t M = mM.total(), N = mN.total(), K = mK.total(), Bt = mB.total();
  if (M == 0 || N == 0 || Bt == 0 || K == 0) return TNB200_ERR_UNSUPPORTED;
  ModeList gB = mB, gM = mM, gN = mN;
  merge_modes(gB, 3); merge_modes(gM, 2); merge_modes(gN, 2);
  if (gB.n > 1) return TNB200_ERR_UNSUPPORTED;
  int64_t cm_ext, cm_s, cn_ext, cn_s;
  ModeList cM, cN;
  for (int i = 0; i < gM.n; ++i) cM.push(gM.ext[i], gM.s1[i]);
  for (int i = 0; i < gN.n; ++i) cN.push(gN.ext[i], gN.s1[i]);
  if (!(single_mode(cM, 0, cm_ext, cm_s) && single_mode(cN, 0, cn_ext, cn_s))) return TNB200_ERR_UNSUPPORTED;
  g = GemmProblem();
  g.dtype = dt; g.M = M; g.N = N; g.K = K; g.batch = Bt;
  g.C = c->data; g.c_sm = cm_s; g.c_sn = cn_s; g.c_sb = gB.n ? gB.s2[0] : 0;
  for (int cand = 0; cand < 2; ++cand) {
    ModeList ko = order_k(mK, cand);
    merge_modes(ko, 2);
    if (ko.n > 4 || gM.n > 4 || gN.n > 4) continue;
    OperandView va, vb;
    va.ptr = a->data; vb.ptr = b->data;
    va.nF = gM.n; for (int i = 0; i < gM.n; ++i) { va.fe[i] = gM.ext[i]; va.fs[i] = gM.s0[i]; }
    vb.nF = gN.n; for (int i = 0; i < gN.n; ++i) { vb.fe[i] = gN.ext[i]; vb.fs[i] = gN.s0[i]; }
    va.nK = vb.nK = ko.n;
    for (int i = 0; i < ko.n; ++i) { va.ke[i] = vb.ke[i] = ko.ext[i]; va.ks[i] = ko.s0[i]; vb.ks[i] = ko.s1[i]; }
    va.sb = gB.n ? gB.s0[0] : 0; vb.sb = gB.n ? gB.s1[0] : 0;
    if (tcgen05_view_ok(dt, va, M, K, Bt) && tcgen05_view_ok(dt, vb, N, K, Bt)) {
      g.A = va; g.B = vb;
      return 0;
    }
  }
  return TNB200_ERR_UNSUPPORTED;
}
}  // namespace tnb

extern "C" int32_t tnb200_tensordot(const tnb200_tensor_t* a, const tnb200_tensor_t* b,
                                    const tnb200_tensor_t* c, int32_t naxes, const int32_t* axes_a,
                                    const int32_t* axes_b, int32_t nbatch, const int32_t* batch_a,
                                    const int32_t* batch_b, int32_t flags, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  ModeList mB, mM, mN, mK;
  {
    int rc = build_modes(a, b, c, naxes, axes_a, axes_b, nbatch, batch_a, batch_b, mB, mM, mN, mK);
    if (rc) return rc;
  }
  const int dt = a->dtype;
  const bool conjA = (flags & TNB200_CONJ_A) && dtype_is_complex(dt);
  const bool conjB = (flags & TNB200_CONJ_B) && dtype_is_complex(dt);
  const int math = (flags >> 4) & 0xF;
  const int64_t M = mM.total(), N = mN.total(), K = mK.total(), Bt = mB.total();
  if (M == 0 || N == 0 || Bt == 0) { set_kernel_name("empty"); return 0; }
  if (K == 0) { set_kernel_name("fill"); return tnb200_fill(c, 0.0, 0.0, stream); }

  ModeList gB = mB, gM = mM, gN = mN;
  merge_modes(gB, 3); merge_modes(gM, 2); merge_modes(gN, 2);

  // ---- degenerate shapes that are pure HBM streaming: dedicated CUDA-core kernels (tensordot_skinny.cu)
  if (math != (TNB200_MATH_SIMT >> 4)) {
    ModeList sK = mK;
    merge_modes(sK, 2);
    int rc = tensordot_thin(dt, a->data, b->data, c->data, gB, gM, gN, sK, math != (TNB200_MATH_STRICT >> 4), st);
    if (rc != TNB200_ERR_UNSUPPORTED) return rc;
    rc = tensordot_skinny(dt, a->data, b->data, c->data, gB, gM, gN, sK, st);
    if (rc != TNB200_ERR_UNSUPPORTED) return rc;
  }

  // ---- try the tensor-core / DMMA GEMM paths
  const bool gemm_dtype = dt == TNB200_F64 || dt == TNB200_F32 || dt == TNB200_F16 || dt == TNB200_BF16;
  const bool want_gemm = gemm_dtype && math != (TNB200_MATH_SIMT >> 4) &&
                         !(dt == TNB200_F32 && math == (TNB200_MATH_STRICT >> 4)) &&
                         (double)M * (double)N * (double)K * (double)Bt >= 32768.0 && gB.n <= 1 &&
                         !(M <= 64 && N <= 64 && Bt * 2 <= num_sms() && K >= 8192);   // skinny, long K: split-K SIMT
  if (want_gemm) {
    int64_t cm_ext, cm_s, cn_ext, cn_s;
    ModeList cM, cN;
    for (int i = 0; i < gM.n; ++i) cM.push(gM.ext[i], gM.s1[i]);
    for (int i = 0; i < gN.n; ++i) cN.push(gN.ext[i], gN.s1[i]);
    bool c_ok = single_mode(cM, 0, cm_ext, cm_s) && single_mode(cN, 0, cn_ext, cn_s);
    if (c_ok) {
      GemmProblem g;
      g.dtype = dt; g.M = M; g.N = N; g.K = K; g.batch = Bt; g.conjA = conjA; g.conjB = conjB; g.math = math;
      g.C = c->data; g.c_sm = cm_s; g.c_sn = cn_s; g.c_sb = gB.n ? gB.s2[0] : 0;
      // Build both operand views under a common ordering of the contracted modes; try the order
      // that sorts them by A's strides and the one that sorts by B's, keep the one under which
      // more operands are addressable in place (TMA for 16/32-bit, 2-stride cp.async for f64).
      auto make_views = [&](int cand, OperandView& va, OperandView& vb) -> bool {
        ModeList ko = order_k(mK, cand);
        merge_modes(ko, 2);                 // joint merge keeps A's and B's k orders identical
        if (ko.n > 4 || gM.n > 4 || gN.n > 4) return false;
        va = OperandView(); vb = OperandView();
        va.ptr = a->data; vb.ptr = b->data;
        va.nF = gM.n; for (int i = 0; i < gM.n; ++i) { va.fe[i] = gM.ext[i]; va.fs[i] = gM.s0[i]; }
        vb.nF = gN.n; for (int i = 0; i < gN.n; ++i) { vb.fe[i] = gN.ext[i]; vb.fs[i] = gN.s0[i]; }
        va.nK = vb.nK = ko.n;
        for (int i = 0; i < ko.n; ++i) { va.ke[i] = vb.ke[i] = ko.ext[i]; va.ks[i] = ko.s0[i]; vb.ks[i] = ko.s1[i]; }
        va.sb = gB.n ? gB.s0[0] : 0; vb.sb = gB.n ? gB.s1[0] : 0;
        return true;
      };
      auto view_ok = [&](const OperandView& v, int64_t ef) -> bool {
        if (dt == TNB200_F64) return v.simple();
        return tcgen05_view_ok(dt, v, ef, K, Bt);
      };
      int best = -1, best_score = -1; bool bestA = false, bestB = false;
      OperandView va, vb;
      for (int cand = 0; cand < 2; ++cand) {
        OperandView xa, xb;
        if (!make_views(cand, xa, xb)) continue;
        bool okA = view_ok(xa, M), okB = view_ok(xb, N);
        int score = (okA ? 1 : 0) + (okB ? 1 : 0);
        if (score > best_score) { best_score = score; best = cand; bestA = okA; bestB = okB; va = xa; vb = xb; }
      }
      if (best >= 0) {
        ModeList ko = order_k(mK, best);
        merge_modes(ko, 2);
        void *packA = nullptr, *packB = nullptr;
        int rc = 0;
        if (!bestA) {   // repack A as a contiguous K-major [batch, M, K] matrix (k in the common order)
          int64_t kp = K;
          rc = pack_operand(dt, a->data, gB, 0, gM, ko, 0, &packA, &kp, st);
          va = OperandView(); va.ptr = packA; va.nF = 1; va.fe[0] = M; va.fs[0] = kp; va.nK = 1; va.ke[0] = K; va.ks[0] = 1; va.sb = M * kp;
        }
        if (rc == 0 && !bestB) {
          ModeList nB;  // free modes of B with B strides in slot 0
          for (int i = 0; i < gN.n; ++i) nB.push(gN.ext[i], gN.s0[i]);
          int64_t kp = K;
          rc = pack_operand(dt, b->data, gB, 1, nB, ko, 1, &packB, &kp, st);
          vb = OperandView(); vb.ptr = packB; vb.nF = 1; vb.fe[0] = N; vb.fs[0] = kp; vb.nK = 1; vb.ke[0] = K; vb.ks[0] = 1; vb.sb = N * kp;
        }
        if (rc == 0) {
          // a packed operand still contracts over ALL of K with one stride: collapse the other
          // operand's view only if it is also single-mode; otherwise both keep `ko`'s mode split
          if ((!bestA || !bestB) && (va.nK != vb.nK)) {
            // the in-place operand has several k modes but the packed one has a single merged mode:
            // give the packed operand the same split (contiguous, so strides are products)
            OperandView& pk = !bestA ? va : vb;
            const OperandView& ip = !bestA ? vb : va;
            pk.nK = ip.nK;
            int64_t st_ = 1;
            for (int i = ip.nK - 1; i >= 0; --i) { pk.ke[i] = ip.ke[i]; pk.ks[i] = st_; st_ *= ip.ke[i]; }
          }
          g.A = va; g.B = vb;
          rc = (dt == TNB200_F64) ? gemm_dmma_f64(g, st) : gemm_tcgen05(g, st);
          if (rc == TNB200_ERR_UNSUPPORTED && (bestA || bestB) && !(packA && packB)) {
            // in-place addressing was rejected at encode time (tile-size dependent): repack everything
            if (!packA) {
              int64_t kp = K;
              rc = pack_operand(dt, a->data, gB, 0, gM, ko, 0, &packA, &kp, st);
              va = OperandView(); va.ptr = packA; va.nF = 1; va.fe[0] = M; va.fs[0] = kp; va.nK = 1; va.ke[0] = K; va.ks[0] = 1; va.sb = M * kp;
            } else { va.nK = 1; va.ke[0] = K; va.ks[0] = 1; }
            if ((rc == 0 || rc == TNB200_ERR_UNSUPPORTED) && !packB) {
              ModeList nB;
              for (int i = 0; i < gN.n; ++i) nB.push(gN.ext[i], gN.s0[i]);
              int64_t kp = K;
              rc = pack_operand(dt, b->data, gB, 1, nB, ko, 1, &packB, &kp, st);
              vb = OperandView(); vb.ptr = packB; vb.nF = 1; vb.fe[0] = N; vb.fs[0] = kp; vb.nK = 1; vb.ke[0] = K; vb.ks[0] = 1; vb.sb = N * kp;
            } else if (packB) { vb.nK = 1; vb.ke[0] = K; vb.ks[0] = 1; }
            if (rc == 0) { g.A = va; g.B = vb; rc = (dt == TNB200_F64) ? gemm_dmma_f64(g, st) : gemm_tcgen05(g, st); }
          }
        }
        if (packA) ws_free(packA, st);
        if (packB) ws_free(packB, st);
        if (rc != TNB200_ERR_UNSUPPORTED) return rc;
      }
    }
  }
  ModeList gK = mK;
  merge_modes(gK, 2);
  return dispatch_simt(dt, a->data, b->data, c->data, gB, gM, gN, gK, conjA, conjB, st);
}

// ------------------------------------------------------------------------------------------ chained contractions
extern "C" int32_t tnb200_chain_create(int32_t nsteps, const tnb200_chain_step_t* steps, int32_t* first_unsupported,
                                       void** handle) {
  TNB_REQUIRE(nsteps >= 1 && steps && handle, TNB200_ERR_INVALID, "chain: bad arguments");
  *handle = nullptr;
  if (first_unsupported) *first_unsupported = -1;
  std::vector<GemmProblem> probs((size_t)nsteps);
  std::vector<int> da((size_t)nsteps), db((size_t)nsteps);
  for (int i = 0; i < nsteps; ++i) {
    const tnb200_chain_step_t& s = steps[i];
    int rc = plan_inplace_gemm(&s.a, &s.b, &s.c, s.naxes, s.axes_a, s.axes_b, s.nbatch, s.batch_a, s.batch_b, probs[i]);
    if (rc) { if (first_unsupported) *first_unsupported = i; return rc; }
    da[i] = s.dep_a; db[i] = s.dep_b;
    TNB_REQUIRE(s.dep_a < i && s.dep_b < i, TNB200_ERR_INVALID, "chain: step %d depends on a later step", i);
    TNB_REQUIRE(s.dep_a < 0 || steps[s.dep_a].c.data == s.a.data, TNB200_ERR_INVALID, "chain: dep_a of step %d does not produce its operand", i);
    TNB_REQUIRE(s.dep_b < 0 || steps[s.dep_b].c.data == s.b.data, TNB200_ERR_INVALID, "chain: dep_b of step %d does not produce its operand", i);
  }
  // tile-shape eligibility is per step: report the first step the chained kernel cannot take
  for (int i = 0; i < nsteps; ++i) {
    const GemmProblem& g = probs[i];
    if (g.M < 256 || g.N < 128 || g.batch != probs[0].batch || g.dtype != probs[0].dtype) {
      if (first_unsupported) *first_unsupported = i;
      return TNB200_ERR_UNSUPPORTED;
    }
  }
  return gemm_chain_create(nsteps, probs.data(), da.data(), db.data(), handle);
}
extern "C" int32_t tnb200_chain_launch(void* handle, void* stream) { return gemm_chain_launch(handle, (cudaStream_t)stream); }
extern "C" int32_t tnb200_chain_destroy(void* handle) { return gemm_chain_destroy(handle); }
