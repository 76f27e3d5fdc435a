// Host-side mirror of faer::linalg for f64 (the functions SURVEY.md §8a puts on the hot path).
// Names, argument meaning and error behaviour follow the Rust surface; every function launches on `stream`
// and operates on DEVICE views (the C ABI in ffi.cu stages host buffers).
#pragma once
#include "common.cuh"
#include "gemm_f64.cuh"

namespace fb {

// ---- c64 matmul on the f64 DMMA kernel (gemm_c64.cu); views in COMPLEX element units ----
void gemm_c64(cudaStream_t stream, VD dst, int dst_struct, int accum, VCD lhs, int lhs_struct, bool conj_lhs, VCD rhs,
              int rhs_struct, bool conj_rhs, double alpha_re, double alpha_im);

// ---- triangular_solve (reference: faer/src/linalg/triangular_solve.rs:220-419) ----
void solve_lower_triangular_in_place_f64(cudaStream_t stream, VCD tril, bool unit, VD rhs);
void solve_upper_triangular_in_place_f64(cudaStream_t stream, VCD triu, bool unit, VD rhs);

// ---- cholesky::llt::factor (reference: faer/src/linalg/cholesky/llt/factor.rs:68-97) ----
struct LltParams {
  size_t recursion_threshold;  // faer default 64  (ldlt/factor.rs:705-714); GPU path: leaf lives in one CTA
  size_t block_size;           // faer default 128
};
struct LltResult {
  bool ok;
  size_t dynamic_regularization_count;  // valid if ok
  size_t non_positive_pivot_index;      // valid if !ok
};
// ---- c64 triangular solves, LLT and LU (cplx.cu; the c32 twins are declared in gemm_f32.cuh); views in COMPLEX element units ----
void solve_lower_triangular_in_place_c64(cudaStream_t st, VCD tril, bool unit, bool conj, VD rhs);
void solve_upper_triangular_in_place_c64(cudaStream_t st, VCD triu, bool unit, bool conj, VD rhs);
LltResult llt_cholesky_in_place_c64(cudaStream_t st, VD A, double reg_delta, double reg_eps);
void llt_solve_in_place_c64(cudaStream_t st, VCD L, bool conj, VD rhs);
// c64 partial-pivoting LU (perm arrays: HOST int64 of length nrows) and the solve on its factors
size_t lu_partial_piv_in_place_c64(cudaStream_t st, VD A, long long* perm_fwd, long long* perm_inv);
void lu_solve_in_place_c64(cudaStream_t st, VCD L, VCD U, bool conj, const long long* perm_fwd, VD rhs);
void lu_solve_transpose_in_place_c64(cudaStream_t st, VCD L, VCD U, bool conj, const long long* perm_bwd, VD rhs);
// c64 Householder QR without pivoting (returns the rank) and rhs <- Q rhs / Q^H rhs by the block-Householder sequence
i64 qr_in_place_c64(cudaStream_t st, VD A, VD Q_coeff, i64 blocking_threshold);
void apply_householder_sequence_left_c64(cudaStream_t st, VCD basis, VCD factor, bool conj, VD rhs, bool transpose);

// In-place lower Cholesky of the lower triangle of A (strict upper triangle untouched).
// `reg_delta`/`reg_eps`: dynamic regularisation (active iff both > 0), reference llt/factor.rs:85-87.
LltResult llt_cholesky_in_place_f64(cudaStream_t stream, VD A, double reg_delta, double reg_eps, LltParams params);

// reconstruct.cu: `*_reconstruct` / `*_inverse` on the factors (f64); perm arrays are HOST int64
void llt_reconstruct_f64(cudaStream_t st, VD out, VCD L);
void llt_inverse_f64(cudaStream_t st, VD out, VCD L);
void lu_reconstruct_f64(cudaStream_t st, VD out, VCD L, VCD U, const long long* perm_bwd_host);
void lu_inverse_f64(cudaStream_t st, VD out, VCD L, VCD U, const long long* perm_fwd_host);
void qr_inverse_f64(cudaStream_t st, VD out, VCD Q_basis, VCD Q_coeff, VCD R);

// LDLT without pivoting (ldlt_f64.cu; reference cholesky/ldlt/factor.rs:725-767): D on the diagonal, unit-lower L strictly
// below it, strict upper triangle untouched. d_signs: device int8[n] of expected pivot signs, or null.
struct LdltResult {
  bool ok;
  size_t dynamic_regularization_count;  // valid if ok
  size_t zero_pivot_index;              // valid if !ok
};
LdltResult ldlt_in_place_f64(cudaStream_t stream, VD A, double reg_delta, double reg_eps, const signed char* d_signs,
                             LltParams params);
// rhs <- (L D L^T)^-1 rhs (ldlt/solve.rs:11-49); D: device pointer, dstride elements apart
void ldlt_solve_in_place_f64(cudaStream_t stream, VCD L, const double* D, i64 dstride, VD rhs);

// same factorisation, device-only (no sync / read-back); status accumulates in d_info (see llt.cu)
void llt_cholesky_device_f64(cudaStream_t stream, VD A, double reg_delta, double reg_eps, long long* d_info, i64 j0);

// ---- lu::partial_pivoting::factor (reference: faer/src/linalg/lu/partial_pivoting/factor.rs:234-295) ----
struct PartialPivLuParams {
  size_t recursion_threshold;  // faer default 16
  size_t block_size;           // faer default 64 (unused by the reference's recursive code)
  size_t par_threshold;
};
// In-place P A = L U. perm_fwd / perm_inv: DEVICE arrays of nrows indices (u32 if idx_bytes==4 else u64).
// Returns the transposition count.
size_t lu_partial_piv_in_place_f64(cudaStream_t stream, VD A, void* perm_fwd, void* perm_inv, int idx_bytes,
                                   PartialPivLuParams params);

// ---- solves on top of the factors (solve_f64.cu; reference llt/solve.rs:12-35, lu/partial_pivoting/solve.rs:21-54) ----
// one complex element as the C ABI lays it out: (re, im), aligned like R only (faer's c64 / c32 guarantee no more), so that a
// kernel moving it never emits a vector access that would need 2 * sizeof(R) alignment
template <class R>
struct ReIm {
  R re, im;
};
// rhs[i, :] <- rhs[perm_fwd[i], :]; perm_fwd: HOST int64 array of rhs.nrows entries. E: double / float, or ReIm<double> /
// ReIm<float> for a complex view (complex-unit strides on an R* base) reinterpreted as one of (re, im) elements
template <class E>
void permute_rows_in_place(cudaStream_t stream, View<E> rhs, const long long* perm_fwd_host);
// T: double or float
template <class T>
void llt_solve_in_place(cudaStream_t stream, View<const T> L, View<T> rhs);
template <class T>
void lu_solve_in_place(cudaStream_t stream, View<const T> L, View<const T> U, const long long* perm_fwd_host, View<T> rhs);
// rhs <- A^-T rhs (lu/partial_pivoting/solve.rs:55-86); perm_bwd: HOST int64 array, the inverse row permutation
template <class T>
void lu_solve_transpose_in_place(cudaStream_t stream, View<const T> L, View<const T> U, const long long* perm_bwd_host, View<T> rhs);

// workspace-based LU building blocks (used by dist.cu); all work is enqueued on the stream given at creation
struct LuWorkspace;
LuWorkspace* lu_ws_create(cudaStream_t stream, i64 max_window, int sm_limit = 0);
void lu_ws_set_cluster(LuWorkspace* w, int ctas);  // leaves on a thread-block cluster of `ctas` CTAs (0 = off)
void lu_ws_set_big_stream(LuWorkspace* w, cudaStream_t big);  // see lu_rec: offload target for large recursion nodes
void lu_ws_destroy(LuWorkspace* w);
void lu_factor_window_f64(LuWorkspace* w, VD A, i64 start, i64 end, int* d_trans);
void lu_apply_transpositions_f64(LuWorkspace* w, VD cols, const int* d_trans, i64 n);

// ---- multi-GPU (dist.cu): 1-D block-column-cyclic factorizations, one process per GPU, NCCL panel broadcast ----
int dist_unique_id(void* out128);                       // rank 0: 128-byte NCCL unique id
int dist_init(int rank, int nranks, const void* id128);  // all ranks (collective)
void dist_finalize();
bool dist_ready();
int dist_rank();
int dist_nranks();
// A_local: column-major n x (local columns), ld >= n; block column b (width nb) lives on rank b % P.
LltResult dist_llt_f64(double* A_local, i64 ld, i64 n, i64 nb, double reg_delta, double reg_eps, int lookahead);
// LLT of a HOST column-major matrix with the PCIe transfers overlapped with the factorization (dist.cu)
LltResult llt_host_pipelined_f64(double* hostA, i64 host_ld, i64 n, i64 nb, double reg_delta, double reg_eps);
i64 lookahead_min_n();
i64 lookahead_block();
// Distributed P A = L U (square n x n). perm_fwd / perm_inv: HOST arrays of n int64 (identical on every rank).
size_t dist_lu_f64(double* A_local, i64 ld, i64 n, i64 nb, long long* perm_fwd, long long* perm_inv, int lookahead);
// distributed Householder QR (m >= n; block width = Householder block size bs; Q_coeff bs x n on the device, replicated);
// returns n, or -1 when a block turned out rank-deficient
i64 dist_qr_f64(double* A_local, i64 ld, i64 m, i64 n, i64 bs, double* Q_coeff, int flags);
i64 dist_qr_f32(float* A_local, i64 ld, i64 m, i64 n, i64 bs, float* Q_coeff, int flags);

// single-GPU entry points switch to the look-ahead block-column driver above this size (env FAER_B200_LOOKAHEAD_MIN_N,
// default 4096; 0 disables) with this block width (env FAER_B200_NB, default 1024)
i64 lookahead_min_n();
i64 lookahead_block();

// ---- device workspace (grow-only pool, one per process) ----
void* ws_alloc(size_t bytes);  // 256-byte aligned device memory, cached across calls
void ws_free(void* p);
void ws_release_all();
// Per-stream grow-only scratch (split-K partials): work on one stream is ordered, so the buffer is reused call after call
// without host synchronisation; it is re-allocated (after draining the stream) only when a larger size is requested.
void* stream_scratch(cudaStream_t stream, size_t bytes);

}  // namespace fb
