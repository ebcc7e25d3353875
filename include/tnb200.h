/* tnb200.h — C ABI of libtnb200.so, the B200-native (sm_100a) dense contraction + split
 * engine that sits beneath the `cuda_b200` TensorNetwork backend.
 *
 * This is the drop-in boundary of SURVEY.md section 8(b): the reference's plug-in surface is
 * the Python class `AbstractBackend` (tensornetwork/backends/abstract_backend.py:22); the
 * adapter class `tensornetwork_b200.backend.CudaB200Backend` implements that class and
 * forwards every compute method to one of the entry points below through ctypes.
 * No torch / Python types appear here: plain device pointers, sizes, a cudaStream_t passed
 * as void*.  All calls are stream-ordered and asynchronous unless stated; all return 0 on
 * success or a negative tnb200_status_t, with a message available from tnb200_last_error().
 *
 * Each entry point cites the reference method it replaces (file:line relative to the
 * reference repo root).
 */
#ifndef TNB200_H_
#define TNB200_H_

#include <stdint.h>

#if defined(TNB200_BUILD)
#define TNB200_API __attribute__((visibility("default")))
#else
#define TNB200_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define TNB200_MAX_NDIM 16
#define TNB200_ABI_VERSION 1

typedef enum {
  TNB200_OK = 0,
  TNB200_ERR_INVALID = -1,   /* bad argument / shape mismatch  -> Python ValueError   */
  TNB200_ERR_DTYPE = -2,     /* unsupported dtype combination  -> Python TypeError    */
  TNB200_ERR_CUDA = -3,      /* CUDA runtime / driver failure  -> Python RuntimeError */
  TNB200_ERR_UNSUPPORTED = -4,/* valid request this build cannot serve -> NotImplementedError */
  TNB200_ERR_NOCONV = -5     /* iterative kernel did not converge -> RuntimeError */
} tnb200_status_t;

typedef enum {
  TNB200_F64 = 0,
  TNB200_F32 = 1,
  TNB200_F16 = 2,
  TNB200_BF16 = 3,
  TNB200_C64 = 4,   /* interleaved (re, im) float  */
  TNB200_C128 = 5,  /* interleaved (re, im) double */
  TNB200_I32 = 6,
  TNB200_I64 = 7,
  TNB200_BOOL = 8   /* 1 byte, 0 or 1: masks.  Accepted by copy, compare and masked_fill only; every other entry point
                       returns TNB200_ERR_DTYPE for it */
} tnb200_dtype_t;

/* A strided view of device memory.  Strides are in ELEMENTS (like torch), may be 0
 * (broadcast) and need not describe a contiguous block. */
typedef struct tnb200_tensor {
  void* data;
  int32_t dtype;
  int32_t ndim;
  int64_t shape[TNB200_MAX_NDIM];
  int64_t stride[TNB200_MAX_NDIM];
} tnb200_tensor_t;

/* flags for tnb200_tensordot */
#define TNB200_CONJ_A 0x1
#define TNB200_CONJ_B 0x2
/* math mode, bits [4,8): how fp32 / fp64 inputs use the tensor cores */
#define TNB200_MATH_DEFAULT (0 << 4) /* f64: DMMA fp64; f32: TF32 tcgen05 when large; 16-bit: tcgen05 */
#define TNB200_MATH_STRICT (1 << 4)  /* never lower the input precision (f32 -> fp32 FMA path)      */
#define TNB200_MATH_SIMT (2 << 4)    /* force the generic strided CUDA-core kernel (any dtype)     */

TNB200_API const char* tnb200_last_error(void);
TNB200_API int32_t tnb200_abi_version(void);
/* sm count, compute capability and HBM bytes of the current device */
TNB200_API int32_t tnb200_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor,
                           int64_t* total_mem);
/* name of the kernel family the last tnb200_tensordot call on this thread dispatched to
 * ("simt", "dmma_f64", "tcgen05_bf16", ...): used by tests to prove which path ran. */
TNB200_API const char* tnb200_last_kernel(void);
/* number of kernel launches issued by this library since process start (all threads) */
TNB200_API int64_t tnb200_launch_count(void);

/* ---- a1: NumPyBackend.tensordot  (backends/numpy/numpy_backend.py:35-54,
 *          AbstractBackend.tensordot abstract_backend.py:27-38), and the batched form used by
 *          NumPyBackend.matmul (:609-612) / ncon's _batch_cont (ncon_interface.py:280-354).
 * c[batch..., free_a..., free_b...] = sum over contracted axes of a * b.
 * `c` must be a preallocated tensor of that shape (any strides); transposes of a/b are fused:
 * a and b are arbitrary strided views and are never materialised unless the planner has to
 * repack an operand the TMA engine cannot address (see DESIGN.md).
 * batch_a/batch_b list `nbatch` axes of a/b that are carried, not summed (nbatch may be 0). */
TNB200_API int32_t tnb200_tensordot(const tnb200_tensor_t* a, const tnb200_tensor_t* b,
                         const tnb200_tensor_t* c, int32_t naxes, const int32_t* axes_a,
                         const int32_t* axes_b, int32_t nbatch, const int32_t* batch_a,
                         const int32_t* batch_b, int32_t flags, void* stream);

/* ---- a2 helpers: NumPyBackend.transpose/reshape materialisation (numpy_backend.py:56-62).
 * dst[i...] = (conj?) src[i...] with dtype conversion; shapes must match; any strides. */
TNB200_API int32_t tnb200_copy(const tnb200_tensor_t* src, const tnb200_tensor_t* dst, int32_t conj,
                    void* stream);

/* ---- a6: elementwise helpers (numpy_backend.py:536-575 add/sub/mul/div + broadcast_*,
 *          :89-90 sqrt, :162-163 conj, :709-730 abs/sign, :577-589 sin/cos/exp/log, :763-782 power).
 * c = a (op) b with numpy broadcasting expressed by 0-strides; all three same ndim/shape. */
typedef enum { TNB200_ADD = 0, TNB200_SUB = 1, TNB200_MUL = 2, TNB200_DIV = 3,
               TNB200_POW = 4 } tnb200_binop_t;
TNB200_API int32_t tnb200_binary(int32_t op, const tnb200_tensor_t* a, const tnb200_tensor_t* b,
                      const tnb200_tensor_t* c, void* stream);
typedef enum { TNB200_CONJ = 0, TNB200_SQRT = 1, TNB200_ABS = 2, TNB200_NEG = 3,
               TNB200_EXP = 4, TNB200_LOG = 5, TNB200_SIN = 6, TNB200_COS = 7,
               TNB200_SIGN = 8, TNB200_REAL = 9, TNB200_IMAG = 10 } tnb200_unop_t;
TNB200_API int32_t tnb200_unary(int32_t op, const tnb200_tensor_t* a, const tnb200_tensor_t* c,
                     void* stream);
/* x = alpha * x + beta  (in place; `x /= norm` of dmrg.py:225,298 and base_mps.py:172) */
TNB200_API int32_t tnb200_affine_inplace(const tnb200_tensor_t* x, double alpha_re, double alpha_im,
                              double beta_re, double beta_im, void* stream);
/* x = x * (*alpha_dev)^power, alpha read on the device (no host sync): power = -1 divides */
TNB200_API int32_t tnb200_scale_by_device_scalar(const tnb200_tensor_t* x, const void* alpha_dev,
                                      int32_t alpha_dtype, int32_t power, void* stream);
/* y += alpha * x, alpha given on host or (alpha_dev != NULL) as sign * (*alpha_dev) on device */
TNB200_API int32_t tnb200_axpy(const tnb200_tensor_t* x, const tnb200_tensor_t* y, double alpha_re,
                    double alpha_im, const void* alpha_dev, double sign, void* stream);
TNB200_API int32_t tnb200_fill(const tnb200_tensor_t* c, double re, double im, void* stream);
/* c[i, j] = (j - i == k) — NumPyBackend.eye :110-116 */
TNB200_API int32_t tnb200_eye(const tnb200_tensor_t* c, int64_t k, void* stream);
/* standard normal fill (Philox4x32-10 + Box-Muller), NumPyBackend.randn :132-144; complex
 * dtypes get independent re/im parts.  uniform: random_uniform :146-160. */
TNB200_API int32_t tnb200_randn(const tnb200_tensor_t* c, uint64_t seed, void* stream);
TNB200_API int32_t tnb200_uniform(const tnb200_tensor_t* c, double lo, double hi, uint64_t seed,
                       void* stream);

/* ---- a6: reductions.  out is a device scalar/tensor; nothing syncs.
 * norm: Frobenius norm (numpy_backend.py:108-109) -> *out (real dtype of a: f64 for f64/c128,
 *       f32 otherwise).  dot: sum(conj?(x) * y) -> *out in a's dtype (Lanczos :503-504). */
TNB200_API int32_t tnb200_norm(const tnb200_tensor_t* a, void* out, void* stream);
TNB200_API int32_t tnb200_dot(const tnb200_tensor_t* x, const tnb200_tensor_t* y, int32_t conj_x, void* out,
                   void* stream);
/* sum over `naxes` axes (numpy_backend.py:603-607); c has the reduced axes removed */
TNB200_API int32_t tnb200_sum(const tnb200_tensor_t* a, const tnb200_tensor_t* c, int32_t naxes,
                   const int32_t* axes, void* stream);
/* trace over (axis1, axis2) with offset (numpy_backend.py:684-707); c = remaining axes */
TNB200_API int32_t tnb200_trace(const tnb200_tensor_t* a, const tnb200_tensor_t* c, int64_t offset,
                     int32_t axis1, int32_t axis2, void* stream);
/* c (n+|k|, n+|k|) = 0 except the k-th diagonal = ravel(a) (numpy_backend.py:673-682) */
TNB200_API int32_t tnb200_diagflat(const tnb200_tensor_t* a, const tnb200_tensor_t* c, int64_t k,
                        void* stream);

/* ---- masks: NumPyBackend.index_update (numpy_backend.py:548-552) and the elementwise `<=` InfiniteMPS.canonicalize
 * builds its mask with (matrixproductstates/infinite_mps.py:239,273).
 * compare: c = a (op) b for real dtypes, c TNB200_BOOL; a, b, c same shape (0-strides broadcast), a and b one dtype.
 * masked_fill: out = mask ? value : src (one launch); src / out one dtype (bool included), mask TNB200_BOOL, all one shape
 * (0-strides broadcast).  The value is (re, im) from the host, or read on the device from value_dev (dtype value_dtype)
 * when value_dev is not NULL: no host sync either way. */
typedef enum { TNB200_LT = 0, TNB200_LE = 1, TNB200_GT = 2, TNB200_GE = 3 } tnb200_cmpop_t;
TNB200_API int32_t tnb200_compare(int32_t op, const tnb200_tensor_t* a, const tnb200_tensor_t* b, const tnb200_tensor_t* c,
                                  void* stream);
TNB200_API int32_t tnb200_masked_fill(const tnb200_tensor_t* src, const tnb200_tensor_t* mask, const tnb200_tensor_t* out,
                                      double re, double im, const void* value_dev, int32_t value_dtype, void* stream);

/* ---- a4: decompositions.svd (backends/numpy/decompositions.py:21-74).
 * Thin SVD of the m x n matrix view `a` (any strides) by one-sided Jacobi:
 *   u (m x r), s (r, real dtype, DESCENDING), vh (r x n), r = min(m, n); all preallocated and
 *   contiguous.  `info` (device int32[4], may be NULL): [0] sweeps used, [1] converged flag.
 * Truncation is a second call so the data-dependent `keep` needs exactly one D2H of an int. */
TNB200_API int32_t tnb200_svd(const tnb200_tensor_t* a, const tnb200_tensor_t* u, const tnb200_tensor_t* s,
                   const tnb200_tensor_t* vh, int32_t* info_dev, void* stream);
/* decompositions.py:38-57: keep = min(max_singular_values, #{ sqrt(cumsum(s[::-1]^2)) > eps })
 * with eps = max_truncation_error * (relative ? s[0] : 1); max_singular_values < 0 means None,
 * use_error = 0 means max_truncation_error is None.  Writes one int64 to *keep_dev. */
TNB200_API int32_t tnb200_svd_truncation_count(const tnb200_tensor_t* s, int64_t max_singular_values,
                                    int32_t use_error, double max_truncation_error,
                                    int32_t relative, int64_t* keep_dev, void* stream);

/* ---- a5: decompositions.qr / rq (decompositions.py:77-124).  Reduced QR of the m x n view
 * `a`: q (m x r), r (r x n), r = min(m, n), Householder (LAPACK geqrf sign convention) with the
 * optional non_negative_diagonal phase fix (:91-94).  rq is qr of the conjugate transpose and is
 * composed by the adapter. */
TNB200_API int32_t tnb200_qr(const tnb200_tensor_t* a, const tnb200_tensor_t* q, const tnb200_tensor_t* r,
                  int32_t non_negative_diagonal, void* stream);

/* ---- NumPyBackend.eigh (numpy_backend.py:165-166 = np.linalg.eigh, UPLO='L').  a: (..., n, n), any strides, f32 / f64 /
 * c64 / c128; only its lower triangle is read and the imaginary part of its diagonal is ignored.  w (..., n): eigenvalues
 * ascending, in the real dtype; v (..., n, n): eigenvectors as columns, in the input dtype.  Cyclic two-sided Jacobi:
 * n <= 64 -> one CTA per matrix, the whole stack in one launch; larger n -> blocked Jacobi on the block-pair tournament of
 * tnb200_svd, convergence decided on the device.  No host synchronisation (graph-capturable).  `info_dev` (device int32[4],
 * may be NULL): [0] the most sweeps any matrix used, [1] 1 if every matrix converged. */
TNB200_API int32_t tnb200_eigh(const tnb200_tensor_t* a, const tnb200_tensor_t* w, const tnb200_tensor_t* v, int32_t* info_dev,
                               void* stream);
/* ---- NumPyBackend.inv (numpy_backend.py:554-558 = np.linalg.inv).  out = a^-1 for a square n x n view (any strides,
 * f32 / f64 / c64 / c128) by Gauss-Jordan elimination with partial pivoting.  *info_dev (device int32, required) is set to
 * 0, or to k + 1 when the pivot of step k is exactly zero (singular matrix; out is then undefined). */
TNB200_API int32_t tnb200_inv(const tnb200_tensor_t* a, const tnb200_tensor_t* out, int32_t* info_dev, void* stream);
/* ---- the orthogonalisation of one Arnoldi step (NumPyBackend.eigs, numpy_backend.py:216-291; tensornetwork_b200/arnoldi.py).
 * basis: (rows, n) row-major contiguous; w: (n,), any stride, basis dtype (f32 / f64 / c64 / c128); 0 <= k < rows.
 * Classical Gram-Schmidt with one reorthogonalisation of w against basis rows 0..k-1, deterministic reductions; writes
 * w_perp / |w_perp| into basis row k (zeros if |w_perp| = 0) and h_dev[0..k) = <row j, w> (both passes), h_dev[k] = |w_perp|
 * (device, basis dtype).  Four launches, no host sync. */
TNB200_API int32_t tnb200_krylov_orth(const tnb200_tensor_t* basis, const tnb200_tensor_t* w, int32_t k, void* h_dev, void* stream);

/* ---- a11: block_sparse.tensordot per-sector loop (block_sparse/blocksparsetensor.py:1094-1101).
 * For each sector q: C.data[c_map[q]] = A.data[a_map[q]].reshape(m_q,k_q) @ B.data[b_map[q]]
 * .reshape(k_q,n_q), all sectors in ONE launch.  maps are int64 element indices into the flat
 * data vectors, concatenated; *_off[q] is the start of sector q inside the concatenation
 * (nsect+1 entries).  dims holds (m_q, k_q, n_q) triples.  All arrays are device pointers. */
TNB200_API int32_t tnb200_blocksparse_tensordot(const void* a_data, const void* b_data, void* c_data,
                                     int32_t dtype, int32_t nsect, const int64_t* dims_dev,
                                     const int64_t* a_map_dev, const int64_t* a_off_dev,
                                     const int64_t* b_map_dev, const int64_t* b_off_dev,
                                     const int64_t* c_map_dev, const int64_t* c_off_dev,
                                     int64_t max_m, int64_t max_n, int32_t conj_b, void* stream);

/* ---- a12: the per-sector SVDs of backends/symmetric/decompositions.py:54-61 (a Python loop of
 * np.linalg.svd there): `nprob` independent small SVDs in ONE launch, one CTA per matrix, warp-shuffle
 * Jacobi in shared memory.  Problem q: A_q is m_q x n_q, row-major contiguous at a_data + a_off[q]
 * (element offsets); outputs U_q (m x r), S_q (r, real dtype, descending), Vh_q (r x n), r = min(m, n),
 * row-major at the given offsets.  dims holds (m_q, n_q) pairs.  All arrays are device pointers.
 * *status_dev (may be NULL) is set to 1 if any problem failed to converge. */
TNB200_API int32_t tnb200_svd_batched(const void* a_data, int32_t dtype, int32_t nprob, const int64_t* dims_dev,
                                      const int64_t* a_off_dev, void* u_data, const int64_t* u_off_dev, void* s_data,
                                      const int64_t* s_off_dev, void* vh_data, const int64_t* vh_off_dev,
                                      int64_t max_m, int64_t max_n, int32_t* status_dev, void* stream);

/* ---- f3: the int64 element maps of a block-sparse matrix view, built on the device (the reference builds them on the host
 * with numpy unique / intersect: block_sparse/blocksparse_utils.py:330-634, cached only on request, caching.py:22-88).
 * The tensor has `nlegs` stored legs; leg t has dims[t] states with SIGNED charges (flow applied, int64) at
 * charges_dev[leg_off[t] ...].  Matrix view: rows = legs order[0..partition), columns = order[partition..nlegs).
 * Output map_dev[nnz]: sector-major (ascending row charge), inside a sector row-major (rows x columns, both ascending):
 * the position in the data vector of every element — bit-identical to the reference's maps.  `split` cuts the stored legs
 * into the two groups whose states are enumerated; shift = sum of max|charge| over the legs (U(1)), modulus = N for Z_N
 * (0: U(1)); nbins = 2*shift+1 or N; tables_dev = int64 [start_right(nbins) | sect_off(nbins) | ncols(nbins)], the
 * per-charge tables the caller derives from the legs' charge histograms (charge-degeneracy arithmetic).
 * dims / leg_off / order are HOST arrays. */
TNB200_API int32_t tnb200_blocksparse_maps(int32_t nlegs, const int64_t* dims, const int64_t* charges_dev, const int64_t* leg_off,
                                           const int32_t* order, int32_t partition, int32_t split, int64_t modulus, int64_t shift,
                                           int32_t nbins, const int64_t* tables_dev, int64_t nnz, int64_t* map_dev, void* stream);

/* dst[i] = src[idx[i]] (gather) or dst[idx[i]] = src[i] (scatter = 1), i < n; idx is a device int64 array.
 * The fancy-index gathers of block_sparse (blocksparsetensor.py:1094-1101, symmetric decompositions.py:55). */
TNB200_API int32_t tnb200_gather(const void* src, const int64_t* idx_dev, void* dst, int64_t n, int32_t dtype,
                                 int32_t scatter, void* stream);

/* ---- a8/a9: a RUN of dependent pairwise contractions of one path (the sequential `contract_between` loop of
 * contractors/opt_einsum_paths/path_contractors.py:87-90, e.g. the MPS zipper) as ONE persistent launch.
 * Step i is the contraction tnb200_tensordot(a, b, c, ...) would perform; dep_a / dep_b name the earlier step
 * of the chain whose output `c` is this step's operand (or -1 when the operand exists before the launch).
 * Every step must be a tensor-core GEMM addressable in place (M >= 256, N >= 128, 16/32-bit float, one batch
 * mode shared by all steps); otherwise create() returns TNB200_ERR_UNSUPPORTED with *first_unsupported = the
 * offending step and the caller launches the steps one by one.  create() allocates device tables (not
 * capturable); launch() is stream-ordered and capturable; operand addresses are frozen at create(). */
typedef struct {
  tnb200_tensor_t a, b, c;
  int32_t naxes, nbatch;
  int32_t axes_a[TNB200_MAX_NDIM], axes_b[TNB200_MAX_NDIM];
  int32_t batch_a[TNB200_MAX_NDIM], batch_b[TNB200_MAX_NDIM];
  int32_t dep_a, dep_b;
} tnb200_chain_step_t;
TNB200_API int32_t tnb200_chain_create(int32_t nsteps, const tnb200_chain_step_t* steps, int32_t* first_unsupported,
                                       void** handle);
TNB200_API int32_t tnb200_chain_launch(void* handle, void* stream);
TNB200_API int32_t tnb200_chain_destroy(void* handle);

#ifdef __cplusplus
}
#endif
#endif /* TNB200_H_ */
