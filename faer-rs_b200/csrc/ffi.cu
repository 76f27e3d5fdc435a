// extern "C" boundary: the symbols declared in include/faer_b200.h. Each entry point mirrors the faer-ffi function of the same name
// (faer-ffi/src/lib.rs, cited per function in the header): same argument order and meaning, by-value PODs, synchronous on return,
// abort() on precondition violations. Host buffers are staged; device buffers are used in place.
//
// This unit holds the families whose drivers are the tensor-core files (matmul, triangular solves, LLT, LU, QR and the Householder
// sequences, written once over the scalar kind <R, CX> with R the real type and CX "complex"), the f64 drivers of their own (LDLT,
// reconstruct / inverse, svd / self_adjoint_evd for real T), the extensions and the global state. ffi_types.cu holds the entry
// points of the flat-map drivers and every default-params / scratch query that is not QR's, LLT's or LU's: that unit also builds
// for the host (tools/emul), this one does not. Helpers shared by both: ffi_common.cuh.
#include "../../include/faer_b200.h"
#include "ffi_common.cuh"
#include "gemm_f32.cuh"
#include "runtime.cuh"
#include "tensor_ops.cuh"

#include <atomic>
#include <cstring>
#include <memory>
#include <type_traits>
#include <vector>

using namespace fb;

namespace {

std::atomic<int> g_par_tag{FaerV0_24_ParTag_Rayon};
std::atomic<size_t> g_par_threads{0};

// ---- the drivers under the families: real T through the f64 / f32 overloads of tensor_ops.cuh and real_llt; complex T through the
// cplx_* overloads (cplx.cu, gemm_c64.cu, gemm_c32.cu; views in complex-unit strides on an R* base, as the complex GEMMs take them) ----
inline LltResult real_llt(cudaStream_t st, View<double> a, double delta, double eps, LltParams p) { return llt_cholesky_in_place_f64(st, a, delta, eps, p); }
inline LltResult real_llt(cudaStream_t st, View<float> a, float delta, float eps, LltParams p) { return llt_cholesky_in_place_f32(st, a, delta, eps, p); }
inline void cplx_gemm(cudaStream_t st, View<double> c, int cs, int acc, View<const double> a, int as, bool ca, View<const double> b, int bs, bool cb, double re, double im) { gemm_c64(st, c, cs, acc, a, as, ca, b, bs, cb, re, im); }
inline void cplx_gemm(cudaStream_t st, View<float> c, int cs, int acc, View<const float> a, int as, bool ca, View<const float> b, int bs, bool cb, float re, float im) { gemm_c32(st, c, cs, acc, a, as, ca, b, bs, cb, re, im); }
inline void cplx_solve_lower(cudaStream_t st, View<const double> t, bool unit, bool conj, View<double> r) { solve_lower_triangular_in_place_c64(st, t, unit, conj, r); }
inline void cplx_solve_lower(cudaStream_t st, View<const float> t, bool unit, bool conj, View<float> r) { solve_lower_triangular_in_place_c32(st, t, unit, conj, r); }
inline void cplx_solve_upper(cudaStream_t st, View<const double> t, bool unit, bool conj, View<double> r) { solve_upper_triangular_in_place_c64(st, t, unit, conj, r); }
inline void cplx_solve_upper(cudaStream_t st, View<const float> t, bool unit, bool conj, View<float> r) { solve_upper_triangular_in_place_c32(st, t, unit, conj, r); }
inline LltResult cplx_llt(cudaStream_t st, View<double> a, double delta, double eps) { return llt_cholesky_in_place_c64(st, a, delta, eps); }
inline LltResult cplx_llt(cudaStream_t st, View<float> a, float delta, float eps) { return llt_cholesky_in_place_c32(st, a, delta, eps); }
inline void cplx_llt_solve(cudaStream_t st, View<const double> l, bool conj, View<double> r) { llt_solve_in_place_c64(st, l, conj, r); }
inline void cplx_llt_solve(cudaStream_t st, View<const float> l, bool conj, View<float> r) { llt_solve_in_place_c32(st, l, conj, r); }
inline size_t cplx_lu(cudaStream_t st, View<double> a, long long* pf, long long* pb) { return lu_partial_piv_in_place_c64(st, a, pf, pb); }
inline size_t cplx_lu(cudaStream_t st, View<float> a, long long* pf, long long* pb) { return lu_partial_piv_in_place_c32(st, a, pf, pb); }
inline void cplx_lu_solve(cudaStream_t st, View<const double> l, View<const double> u, bool conj, const long long* p, View<double> r) { lu_solve_in_place_c64(st, l, u, conj, p, r); }
inline void cplx_lu_solve(cudaStream_t st, View<const float> l, View<const float> u, bool conj, const long long* p, View<float> r) { lu_solve_in_place_c32(st, l, u, conj, p, r); }
inline void cplx_lu_solve_t(cudaStream_t st, View<const double> l, View<const double> u, bool conj, const long long* p, View<double> r) { lu_solve_transpose_in_place_c64(st, l, u, conj, p, r); }
inline void cplx_lu_solve_t(cudaStream_t st, View<const float> l, View<const float> u, bool conj, const long long* p, View<float> r) { lu_solve_transpose_in_place_c32(st, l, u, conj, p, r); }
inline i64 cplx_qr(cudaStream_t st, View<double> a, View<double> q, i64 thr) { return qr_in_place_c64(st, a, q, thr); }
inline i64 cplx_qr(cudaStream_t st, View<float> a, View<float> q, i64 thr) { return qr_in_place_c32(st, a, q, thr); }
inline void cplx_hh_seq(cudaStream_t st, View<const double> b, View<const double> f, bool conj, View<double> r, bool tr) { apply_householder_sequence_left_c64(st, b, f, conj, r, tr); }
inline void cplx_hh_seq(cudaStream_t st, View<const float> b, View<const float> f, bool conj, View<float> r, bool tr) { apply_householder_sequence_left_c32(st, b, f, conj, r, tr); }

// conj?(T) X = rhs with T lower or upper triangular; conj is a no-op for real T
template <bool CX, class R>
void tri_solve(cudaStream_t st, bool lower, View<const R> t, bool unit, bool conj, View<R> r) {
  if constexpr (CX) {
    if (lower) cplx_solve_lower(st, t, unit, conj, r);
    else cplx_solve_upper(st, t, unit, conj, r);
  } else {
    if (lower) solve_lower(st, t, unit, r);
    else solve_upper(st, t, unit, r);
  }
}
// rhs <- op(Q) rhs (transpose = false) or op(Q)^H rhs (transpose = true) for the block-Householder sequence; conj is a no-op for real T
template <bool CX, class R>
void hh_seq(cudaStream_t st, View<const R> basis, View<const R> factor, bool conj, View<R> r, bool transpose) {
  if constexpr (CX) cplx_hh_seq(st, basis, factor, conj, r, transpose);
  else if (transpose) apply_block_householder_sequence_transpose_on_the_left<R>(st, basis, factor, r);
  else apply_block_householder_sequence_on_the_left<R>(st, basis, factor, r);
}
// the leading m x n block of a view: no offset, so the same for real and complex-unit views
template <class V>
V leading(V v, i64 m, i64 n) { return V{v.ptr, m, n, v.rs, v.cs}; }
inline FaerV0_24_MatMut transposed(FaerV0_24_MatMut m) { return FaerV0_24_MatMut{m.ptr, m.ncols, m.nrows, m.col_stride, m.row_stride}; }

// widening / narrowing copies of the f32 LU factorization (below)
template <class TD, class TS>
__global__ void ffi_cast_kernel(TD* __restrict__ dst, i64 drs, i64 dcs, const TS* __restrict__ src, i64 srs, i64 scs, i64 m,
                                i64 c0) {
  const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  const i64 j = c0 + blockIdx.y;
  if (i < m) dst[i * drs + j * dcs] = (TD)src[i * srs + j * scs];
}
template <class TD, class TS>
void ffi_cast(cudaStream_t st, TD* dst, i64 drs, i64 dcs, const TS* src, i64 srs, i64 scs, i64 m, i64 n) {
  if (m == 0 || n == 0) return;
  for (i64 c0 = 0; c0 < n; c0 += 65535) {
    const i64 nc = std::min<i64>(65535, n - c0);
    ffi_cast_kernel<TD, TS><<<dim3((unsigned)((m + 255) / 256), (unsigned)nc), 256, 0, st>>>(dst, drs, dcs, src, srs, scs, m, c0);
    note_launch();
  }
  FB_CUDA_CHECK(cudaGetLastError());
}

// ---- matmul (f64: DMMA, f32: 3xTF32 tensor-core kernel, c64 / c32: the complex GEMMs; `alpha` points to a T-typed scalar) ----
template <class R, bool CX>
void matmul_entry(FaerV0_24_MatMut C, int C_block, FaerV0_24_Accum accum, FaerV0_24_MatRef A, int A_block, FaerV0_24_MatRef B,
                  int B_block, const FaerV0_24_Scalar* alpha, bool conj_a = false, bool conj_b = false) {
  FB_ENTRY();
  FB_ASSERT(C.nrows == A.nrows && C.ncols == B.ncols && A.ncols == B.nrows, "matmul shape mismatch");
  cudaStream_t st = current_stream();
  R a[2] = {0, 0};
  read_scalar(alpha, a, CX ? 2 : 1);
  const size_t es = elem_bytes<R, CX>();
  const int add = accum == FaerV0_24_Accum_Add ? 1 : 0;
  StagedMat c = stage(C, es, add || C_block != FaerV0_24_Block_Rectangular, st), l = stage(A, es, st), r = stage(B, es, st);
  if constexpr (CX)
    cplx_gemm(st, c.view<R>(), C_block, add, l.view<const R>(), A_block, conj_a, r.view<const R>(), B_block, conj_b, a[0], a[1]);
  else
    gemm(st, c.view<R>(), C_block, add, l.view<const R>(), A_block, r.view<const R>(), B_block, a[0]);
  finish_all(st, {&c, &l, &r});
}

// ---- triangular solves (trsm.cu for real T, cplx.cu for complex T) ----
template <class R, bool CX>
void solve_tri_entry(FaerV0_24_MatRef T, FaerV0_24_Conj conj, FaerV0_24_MatMut rhs, bool lower, bool unit) {
  FB_ENTRY();
  FB_ASSERT(T.nrows == T.ncols && rhs.nrows == T.nrows, "triangular solve shape mismatch");
  cudaStream_t st = current_stream();
  const size_t es = elem_bytes<R, CX>();
  StagedMat t = stage(T, es, st), r = stage(rhs, es, true, st);
  tri_solve<CX>(st, lower, t.view<const R>(), unit, CX && conj == FaerV0_24_Conj_Yes, r.view<R>());
  finish_all(st, {&t, &r});
}

// ---- LLT (llt.cu for real T, cplx.cu for complex T) ----
template <class R, bool CX>
FaerV0_24_LltStatus llt_factor_entry(FaerV0_24_MatMut A, FaerV0_24_LltRegularization regularization, FaerV0_24_LltParams params) {
  FB_ENTRY();
  FB_ASSERT(A.nrows == A.ncols, "LLT needs a square matrix");
  cudaStream_t st = current_stream();
  R delta, eps;  // the regularisation parameters are T::Real
  read_regularization(regularization, delta, eps);
  if constexpr (std::is_same<R, double>::value && !CX) {
    // f64 host matrix, column-major and large: upload / factor / download pipelined block column by block column (dist.cu)
    if (A.nrows > 0 && !is_device_pointer(A.ptr) && A.row_stride == 1 && A.col_stride >= (ptrdiff_t)A.nrows &&
        (i64)A.nrows >= lookahead_min_n()) {
      FB_CUDA_CHECK(cudaStreamSynchronize(st));
      const i64 nb = lookahead_block() ? lookahead_block() : 256;
      return llt_status(llt_host_pipelined_f64((double*)A.ptr, (i64)A.col_stride, (i64)A.nrows, nb, delta, eps));
    }
  }
  StagedMat a = stage(A, elem_bytes<R, CX>(), true, st);
  LltResult r;
  if constexpr (CX) r = cplx_llt(st, a.view<R>(), delta, eps);  // the complex driver has no tuning parameters
  else r = real_llt(st, a.view<R>(), delta, eps, LltParams{params.recursion_threshold, params.block_size});
  finish_all(st, {&a});
  return llt_status(r);
}
template <class R, bool CX>
void llt_solve_entry(FaerV0_24_MatRef L, FaerV0_24_Conj A_conj, FaerV0_24_MatMut rhs) {
  FB_ENTRY();
  FB_ASSERT(L.nrows == L.ncols && rhs.nrows == L.nrows, "LLT solve shape mismatch");
  cudaStream_t st = current_stream();
  const size_t es = elem_bytes<R, CX>();
  StagedMat l = stage(L, es, st), r = stage(rhs, es, true, st);
  if constexpr (CX) cplx_llt_solve(st, l.view<const R>(), A_conj == FaerV0_24_Conj_Yes, r.view<R>());
  else llt_solve_in_place(st, l.view<const R>(), r.view<R>());
  finish_all(st, {&l, &r});
}

// ---- partial-pivoting LU (lu_f64.cu for f64 and f32, cplx.cu for complex T) ----
template <class R, bool CX>
FaerV0_24_PartialPivLuStatus lu_factor_entry(FaerV0_24_MatMut A, FaerV0_24_SliceMut perm_fwd, FaerV0_24_SliceMut perm_bwd,
                                             FaerV0_24_PartialPivLuParams params, int idx_bytes) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  // faer.hpp fills SliceMut.len with bytes (ffi_common.cuh): the permutation length is A.nrows
  FB_ASSERT(A.nrows == 0 || (perm_fwd.ptr != nullptr && perm_bwd.ptr != nullptr), "null permutation slice");
  StagedMat a = stage(A, elem_bytes<R, CX>(), true, st);
  const PartialPivLuParams p{params.recursion_threshold, params.block_size, params.par_threshold};
  size_t cnt;
  std::vector<long long> pf, pb;
  double* W = nullptr;
  if constexpr (CX) {
    // the complex driver returns host permutations and has no tuning parameters
    pf.resize(A.nrows);
    pb.resize(A.nrows);
    cnt = cplx_lu(st, a.view<R>(), pf.data(), pb.data());
  } else if constexpr (std::is_same<R, float>::value) {
    // f32 is computed in f64: the matrix is widened on the device, factored by the f64 drivers (fused sub-panel kernel, TMA-fed
    // GEMM, SM partition) and rounded back. The factors carry one f32 rounding instead of an f32 elimination's accumulated ones,
    // and the pivot search sees f64 values (a pivot can differ from an all-f32 elimination's where two candidates agree to f32
    // precision; either choice is a valid partial pivot). The solves run on the native f32 triangular solves.
    const i64 m = (i64)A.nrows, n = (i64)A.ncols;
    VF av = a.view<float>();
    const i64 ld = std::max<i64>(1, (m + 1) & ~(i64)1);
    W = (double*)ws_alloc((size_t)ld * (size_t)std::max<i64>(n, 1) * 8);
    ffi_cast<double, float>(st, W, 1, ld, av.ptr, av.rs, av.cs, m, n);
    cnt = lu_partial_piv_in_place_f64(st, VD{W, m, n, 1, ld}, perm_fwd.ptr, perm_bwd.ptr, idx_bytes, p);
    ffi_cast<float, double>(st, av.ptr, av.rs, av.cs, W, 1, ld, m, n);
  } else {
    cnt = lu_partial_piv_in_place_f64(st, a.view<double>(), perm_fwd.ptr, perm_bwd.ptr, idx_bytes, p);
  }
  finish_all(st, {&a});
  if (W) ws_free(W);
  if constexpr (CX) {
    write_perm(perm_fwd.ptr, pf, idx_bytes);
    write_perm(perm_bwd.ptr, pb, idx_bytes);
  }
  return lu_status(cnt);
}
// transpose = false: perm is perm_fwd (solve.rs:21-54); transpose = true: perm is perm_bwd (solve.rs:55-86)
template <class R, bool CX>
void lu_solve_entry(FaerV0_24_MatRef L, FaerV0_24_MatRef U, FaerV0_24_Conj conj, FaerV0_24_SliceRef perm_slice, FaerV0_24_MatMut rhs,
                    int idx_bytes, bool transpose) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t n = L.nrows;
  FB_ASSERT(L.ncols == n && U.nrows == n && U.ncols == n && rhs.nrows == n, "LU solve shape mismatch");
  const std::vector<long long> perm = read_perm_checked(perm_slice, n, idx_bytes);
  const size_t es = elem_bytes<R, CX>();
  StagedMat l = stage(L, es, st), u = stage(U, es, st), r = stage(rhs, es, true, st);
  if constexpr (CX) {
    const bool cj = conj == FaerV0_24_Conj_Yes;
    if (transpose) cplx_lu_solve_t(st, l.view<const R>(), u.view<const R>(), cj, perm.data(), r.view<R>());
    else cplx_lu_solve(st, l.view<const R>(), u.view<const R>(), cj, perm.data(), r.view<R>());
  } else {
    if (transpose) lu_solve_transpose_in_place(st, l.view<const R>(), u.view<const R>(), perm.data(), r.view<R>());
    else lu_solve_in_place(st, l.view<const R>(), u.view<const R>(), perm.data(), r.view<R>());
  }
  finish_all(st, {&l, &u, &r});
}

// ---- Householder QR (no pivoting), block-Householder sequences and the solves on the QR factors (qr.cu / householder.cu for real
// T, cplx.cu for complex T) ----
template <class R, bool CX>
FaerV0_24_QrStatus qr_factor_entry(FaerV0_24_MatMut A, FaerV0_24_MatMut Q, FaerV0_24_QrParams params) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t size = A.nrows < A.ncols ? A.nrows : A.ncols;
  FB_ASSERT(Q.nrows > 0 && Q.ncols == size, "Q_coeff must be block_size x min(nrows, ncols)");
  const size_t es = elem_bytes<R, CX>();
  StagedMat a = stage(A, es, true, st), q = stage(Q, es, true, st);
  // the reference leaves the strict lower part of each T block untouched and zero-fills nothing for full rank
  i64 rank;
  if constexpr (CX) rank = cplx_qr(st, a.view<R>(), q.view<R>(), (i64)params.blocking_threshold);
  else rank = qr_in_place<R>(st, a.view<R>(), q.view<R>());  // the real driver picks its own blocking
  finish_all(st, {&a, &q});
  return qr_status(CX || rank >= 0, (size_t)rank);  // only the real driver reports an unknown rank (< 0)
}
template <class R, bool CX>
void householder_seq_entry(FaerV0_24_MatRef basis, FaerV0_24_MatRef factor, FaerV0_24_Conj conj, FaerV0_24_MatMut rhs, bool transpose) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t es = elem_bytes<R, CX>();
  StagedMat b = stage(basis, es, st), f = stage(factor, es, st), r = stage(rhs, es, true, st);
  hh_seq<CX>(st, b.view<const R>(), f.view<const R>(), CX && conj == FaerV0_24_Conj_Yes, r.view<R>(), transpose);
  finish_all(st, {&b, &f, &r});
}
// qr/no_pivoting/solve.rs; SURVEY.md §8f rank 1:
// mode 0: solve_lstsq_in_place_with_conj (solve.rs:38-76): rhs <- op(Q)^H rhs, then op(R)[..size, ..] x = rhs[..size, ..]
// mode 1: solve_in_place_with_conj (solve.rs:96-119): the same on a square factorization
// mode 2: solve_transpose_in_place_with_conj (solve.rs:140-176): op(R)^T y = rhs (lower solve on the transposed view), then
//         rhs <- the forward sequence with conj composed with Yes
template <class R, bool CX>
void qr_solve_entry(FaerV0_24_MatRef Qb, FaerV0_24_MatRef Qc, FaerV0_24_MatRef Rm, FaerV0_24_Conj A_conj, FaerV0_24_MatMut rhs, int mode) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t m = Qb.nrows, n = Qb.ncols, size = m < n ? m : n;
  FB_ASSERT(Qc.nrows > 0 && rhs.nrows == m && m >= n && Qc.ncols == size && Rm.nrows >= size && Rm.ncols == n, "QR solve shape mismatch");
  if (mode != 0) FB_ASSERT(m == n && Rm.nrows == n, "QR solve: the factorization must be square");
  if (size == 0 || rhs.ncols == 0) return;
  const bool conj = CX && A_conj == FaerV0_24_Conj_Yes;
  const size_t es = elem_bytes<R, CX>();
  StagedMat b = stage(Qb, es, st), f = stage(Qc, es, st), r = stage(rhs, es, true, st);
  // callers normally pass the packed QR matrix for both Q_basis and R (solve.rs:232-246): stage it once
  const bool alias = Rm.ptr == Qb.ptr && Rm.row_stride == Qb.row_stride && Rm.col_stride == Qb.col_stride;
  std::unique_ptr<StagedMat> rr;
  if (!alias) rr.reset(new StagedMat(Rm.ptr, (i64)size, (i64)n, (i64)Rm.row_stride, (i64)Rm.col_stride, es, true, false, st));
  View<const R> Rv = leading(alias ? b.view<const R>() : rr->view<const R>(), (i64)size, (i64)n);
  View<R> x = r.view<R>();
  if (mode == 2) {
    tri_solve<CX>(st, true, Rv.t(), false, conj, x);
    hh_seq<CX>(st, b.view<const R>(), f.view<const R>(), !conj, x, false);
  } else {
    hh_seq<CX>(st, b.view<const R>(), f.view<const R>(), !conj, x, true);
    tri_solve<CX>(st, false, Rv, false, conj, leading(x, (i64)size, x.ncols));
  }
  finish_all(st, {&b, &f, &r});
  if (rr) rr->finish();
}

// ---- self-adjoint eigendecomposition for real T (evd/mod.rs:270-418): eigenvalues by bisection when U is not wanted, divide and
// conquer + Householder back-transform otherwise. Non-finite input -> EvdStatus::NoConvergence, as the reference ----
template <class T>
FaerV0_24_EvdStatus self_adjoint_evd_entry(FaerV0_24_MatRef A, FaerV0_24_MatMut U, FaerV0_24_VecMut S) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t n = A.nrows;
  FB_ASSERT(A.ncols == n && S.len == n && (n == 0 || S.stride >= 1), "self_adjoint_evd: square A, S of length n, positive stride");
  const bool want_u = U.ncols != 0;
  if (want_u) FB_ASSERT(U.nrows == n && U.ncols == n, "self_adjoint_evd: U must be n x n (or have no columns)");
  if (n == 0) return evd_status(true);
  StagedMat a = stage(A, sizeof(T), st);
  T* s_dev = (T*)ws_alloc(n * sizeof(T));
  bool ok;
  if (want_u) {
    StagedMat u = stage(U, sizeof(T), false, st);
    ok = self_adjoint_evd_with_vectors<T>(st, a.view<const T>(), u.view<T>(), s_dev, 1);
    if (ok) copy_out_vector(S, s_dev, n, sizeof(T), st);
    finish_all(st, {&a, &u});
  } else {
    ok = self_adjoint_eigenvalues<T>(st, a.view<const T>(), s_dev);
    if (ok) copy_out_vector(S, s_dev, n, sizeof(T), st);
    finish_all(st, {&a});
  }
  ws_free(s_dev);
  return evd_status(ok);
}
// ---- SVD for real T (svd/mod.rs:530-672): U.ncols == 0 / V.ncols == 0 mean "do not compute" (faer-ffi/src/lib.rs:2354-2355) ----
template <class T>
FaerV0_24_SvdStatus svd_entry(FaerV0_24_MatRef A, FaerV0_24_MatMut U, FaerV0_24_VecMut S, FaerV0_24_MatMut V,
                              double qr_ratio_threshold) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t size = A.nrows < A.ncols ? A.nrows : A.ncols;
  FB_ASSERT(S.len == size && (size == 0 || S.stride >= 1), "svd: S must have min(nrows, ncols) entries and a positive stride");
  const bool want_u = U.ncols != 0, want_v = V.ncols != 0;
  if (want_u) FB_ASSERT(U.nrows == A.nrows && (U.ncols == A.nrows || U.ncols == size), "svd: U must be nrows x {size, nrows}");
  if (want_v) FB_ASSERT(V.nrows == A.ncols && (V.ncols == A.ncols || V.ncols == size), "svd: V must be ncols x {size, ncols}");
  const double ratio = qr_ratio_threshold > 0.0 ? qr_ratio_threshold : 11.0 / 6.0;
  if (size == 0 && !want_u && !want_v) return svd_status(true);
  StagedMat a = stage(A, sizeof(T), st);
  T* s_dev = (T*)ws_alloc((size + 1) * sizeof(T));
  bool ok;
  if (want_u || want_v) {
    StagedMat u = stage(U, sizeof(T), false, st), v = stage(V, sizeof(T), false, st);
    View<T> uv = want_u ? u.view<T>() : View<T>{nullptr, 0, 0, 1, 1};
    View<T> vv = want_v ? v.view<T>() : View<T>{nullptr, 0, 0, 1, 1};
    ok = svd_with_vectors<T>(st, a.view<const T>(), uv, s_dev, 1, vv, ratio);
    if (ok && size) copy_out_vector(S, s_dev, size, sizeof(T), st);
    finish_all(st, {&a, &u, &v});
  } else {
    ok = singular_values<T>(st, a.view<const T>(), s_dev, ratio);
    if (ok) copy_out_vector(S, s_dev, size, sizeof(T), st);
    finish_all(st, {&a});
  }
  ws_free(s_dev);
  return svd_status(ok);
}

// f64 reconstruct / inverse on the LU factors (reconstruct.cu)
void lu_recon_entry(FaerV0_24_MatMut A, FaerV0_24_MatRef L, FaerV0_24_MatRef U, FaerV0_24_SliceRef perm, int idx_bytes, bool inverse) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const std::vector<long long> p = read_perm_checked(perm, L.nrows, idx_bytes);
  StagedMat a = stage(A, sizeof(double), false, st), l = stage(L, sizeof(double), st), u = stage(U, sizeof(double), st);
  if (inverse) lu_inverse_f64(st, a.view<double>(), l.view<const double>(), u.view<const double>(), p.data());
  else lu_reconstruct_f64(st, a.view<double>(), l.view<const double>(), u.view<const double>(), p.data());
  finish_all(st, {&a, &l, &u});
}

}  // namespace

extern "C" {

// ---- matmul ----
#define FB_MATMUL_FFI(SUF, R, CX)                                                                                               \
  void libfaer_v0_23_matmul_##SUF(FaerV0_24_MatMut C, FaerV0_24_Accum accum, FaerV0_24_MatRef A, FaerV0_24_MatRef B,            \
                                  const FaerV0_24_Scalar* alpha, FaerV0_24_Par par) {                                           \
    (void)par;                                                                                                                  \
    matmul_entry<R, CX>(C, RECT, accum, A, RECT, B, RECT, alpha);                                                               \
  }                                                                                                                             \
  void libfaer_v0_23_matmul_triangular_##SUF(FaerV0_24_MatMut C, FaerV0_24_Block C_block, FaerV0_24_Accum accum,                \
                                             FaerV0_24_MatRef A, FaerV0_24_Block A_block, FaerV0_24_MatRef B,                   \
                                             FaerV0_24_Block B_block, const FaerV0_24_Scalar* alpha, FaerV0_24_Par par) {       \
    (void)par;                                                                                                                  \
    matmul_entry<R, CX>(C, (int)C_block, accum, A, (int)A_block, B, (int)B_block, alpha);                                       \
  }
FB_MATMUL_FFI(f64, double, false)
FB_MATMUL_FFI(f32, float, false)
FB_MATMUL_FFI(c64, double, true)
FB_MATMUL_FFI(c32, float, true)
#undef FB_MATMUL_FFI

// ---- triangular solves ----
#define FB_TRSM_FFI(SUF, R, CX)                                                                                                 \
  void libfaer_v0_23_solve_triangular_lower_in_place_##SUF(FaerV0_24_MatRef L, FaerV0_24_Conj L_conj, FaerV0_24_MatMut rhs,     \
                                                           FaerV0_24_Par par) {                                                 \
    (void)par;                                                                                                                  \
    solve_tri_entry<R, CX>(L, L_conj, rhs, true, false);                                                                        \
  }                                                                                                                             \
  void libfaer_v0_23_solve_triangular_upper_in_place_##SUF(FaerV0_24_MatRef U, FaerV0_24_Conj U_conj, FaerV0_24_MatMut rhs,     \
                                                           FaerV0_24_Par par) {                                                 \
    (void)par;                                                                                                                  \
    solve_tri_entry<R, CX>(U, U_conj, rhs, false, false);                                                                       \
  }                                                                                                                             \
  void libfaer_v0_23_solve_unit_triangular_lower_in_place_##SUF(FaerV0_24_MatRef L, FaerV0_24_Conj L_conj, FaerV0_24_MatMut rhs, \
                                                                FaerV0_24_Par par) {                                            \
    (void)par;                                                                                                                  \
    solve_tri_entry<R, CX>(L, L_conj, rhs, true, true);                                                                         \
  }                                                                                                                             \
  void libfaer_v0_23_solve_unit_triangular_upper_in_place_##SUF(FaerV0_24_MatRef U, FaerV0_24_Conj U_conj, FaerV0_24_MatMut rhs, \
                                                                FaerV0_24_Par par) {                                            \
    (void)par;                                                                                                                  \
    solve_tri_entry<R, CX>(U, U_conj, rhs, false, true);                                                                        \
  }
FB_TRSM_FFI(f64, double, false)
FB_TRSM_FFI(f32, float, false)
FB_TRSM_FFI(c64, double, true)
FB_TRSM_FFI(c32, float, true)
#undef FB_TRSM_FFI

// ---- LLT ----
// the GPU path keeps its (tiny) workspace in the internal device pool, but reports the reference's requirement so callers allocate
// identically
#define FB_LLT_QUERIES(SUF, ES)                                                                                                 \
  FaerV0_24_LltParams libfaer_v0_23_LltParams_##SUF(void) { return FaerV0_24_LltParams{64, 128}; /* ldlt/factor.rs:705-714 */ } \
  FaerV0_24_Layout libfaer_v0_23_llt_factor_in_place_scratch_##SUF(size_t dim, FaerV0_24_Par par, FaerV0_24_LltParams params) { \
    (void)par; (void)params;                                                                                                    \
    return FaerV0_24_Layout{dim * (ES), 64}; /* temp_mat_scratch::<T>(dim, 1), llt/factor.rs:58-66 */                           \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_llt_solve_in_place_scratch_##SUF(size_t dim, size_t rhs_ncols, FaerV0_24_Par par) {            \
    (void)dim; (void)rhs_ncols; (void)par;                                                                                      \
    return FaerV0_24_Layout{0, 1}; /* StackReq::EMPTY (llt/solve.rs:3-10) */                                                    \
  }
#define FB_LLT_FFI(SUF, R, CX)                                                                                                  \
  FaerV0_24_LltStatus libfaer_v0_23_llt_factor_in_place_##SUF(FaerV0_24_MatMut A, FaerV0_24_LltRegularization regularization,   \
                                                              FaerV0_24_Par par, FaerV0_24_MemAlloc mem,                        \
                                                              FaerV0_24_LltParams params) {                                     \
    (void)par; (void)mem;                                                                                                       \
    return llt_factor_entry<R, CX>(A, regularization, params);                                                                  \
  }                                                                                                                             \
  void libfaer_v0_23_llt_solve_in_place_##SUF(FaerV0_24_MatRef L, FaerV0_24_Conj A_conj, FaerV0_24_MatMut rhs,                  \
                                              FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {                                      \
    (void)par; (void)mem;                                                                                                       \
    llt_solve_entry<R, CX>(L, A_conj, rhs);                                                                                     \
  }
FB_LLT_QUERIES(f64, sizeof(double))
FB_LLT_QUERIES(f32, sizeof(float))
FB_LLT_QUERIES(c64, 2 * sizeof(double))
FB_LLT_QUERIES(c32, 2 * sizeof(float))
FB_LLT_FFI(f64, double, false)
FB_LLT_FFI(f32, float, false)
FB_LLT_FFI(c64, double, true)
FB_LLT_FFI(c32, float, true)
#undef FB_LLT_QUERIES
#undef FB_LLT_FFI

// ---- LDLT (no pivoting), f64: ldlt_f64.cu (the other dtypes, reconstruct, inverse and the queries: ffi_types.cu) ----
FaerV0_24_LdltStatus libfaer_v0_23_ldlt_factor_in_place_f64(FaerV0_24_MatMut A, FaerV0_24_LdltRegularization regularization,
                                                            FaerV0_24_Par par, FaerV0_24_MemAlloc mem,
                                                            FaerV0_24_LdltParams params) {
  (void)par; (void)mem;
  FB_ENTRY();
  FB_ASSERT(A.nrows == A.ncols, "LDLT needs a square matrix");
  cudaStream_t st = current_stream();
  double delta, eps;
  read_regularization(regularization, delta, eps);
  const SignsArg signs(regularization.dynamic_regularization_signs, A.nrows, st);
  StagedMat a = stage(A, sizeof(double), true, st);
  const LdltResult r = ldlt_in_place_f64(st, a.view<double>(), delta, eps, signs.ptr,
                                         LltParams{params.recursion_threshold, params.block_size});
  finish_all(st, {&a});
  return ldlt_status(r);
}
void libfaer_v0_23_ldlt_solve_in_place_f64(FaerV0_24_MatRef L, FaerV0_24_VecRef D, FaerV0_24_Conj A_conj, FaerV0_24_MatMut rhs,
                                           FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {
  (void)A_conj; (void)par; (void)mem;
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t n = L.nrows;
  FB_ASSERT(L.ncols == n && D.len == n && rhs.nrows == n, "LDLT solve shape mismatch");
  if (n == 0 || rhs.ncols == 0) return;
  StagedMat l = stage(L, sizeof(double), st), r = stage(rhs, sizeof(double), true, st);
  // D: usually the diagonal of the factored matrix (stride = row_stride + col_stride)
  const DiagArg<double, false> d(D, n, st);
  ldlt_solve_in_place_f64(st, l.view<const double>(), d.ptr, d.stride, r.view<double>());
  finish_all(st, {&l, &r});
}

// ---- partial-pivoting LU ----
#define FB_LU_QUERIES_IT(IT, BYTES, SUF, ES)                                                                                    \
  FaerV0_24_Layout libfaer_v0_23_partial_piv_lu_factor_in_place_scratch_##IT##_##SUF(size_t nrows, size_t ncols, FaerV0_24_Par par, \
                                                                                     FaerV0_24_PartialPivLuParams params) {    \
    (void)par; (void)params;                                                                                                    \
    const size_t size = nrows < ncols ? nrows : ncols; /* StackReq::new::<I>(min(nrows, ncols)) (factor.rs:224-233) */          \
    return FaerV0_24_Layout{size * (BYTES), (BYTES)};                                                                           \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_partial_piv_lu_solve_in_place_scratch_##IT##_##SUF(size_t dim, size_t rhs_ncols, FaerV0_24_Par par) { \
    (void)par;                                                                                                                  \
    return FaerV0_24_Layout{dim * rhs_ncols * (ES), 64}; /* permute_rows_in_place_scratch (perm/mod.rs) */                      \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_partial_piv_lu_solve_transpose_in_place_scratch_##IT##_##SUF(size_t dim, size_t rhs_ncols,     \
                                                                                              FaerV0_24_Par par) {              \
    (void)par;                                                                                                                  \
    return FaerV0_24_Layout{dim * rhs_ncols * (ES), 64};                                                                        \
  }
#define FB_LU_QUERIES(SUF, ES)                                                                                                  \
  FaerV0_24_PartialPivLuParams libfaer_v0_23_PartialPivLuParams_##SUF(void) {                                                   \
    return FaerV0_24_PartialPivLuParams{16, 64, 128 * 128}; /* lu/partial_pivoting/factor.rs:212-222 */                         \
  }                                                                                                                             \
  FB_LU_QUERIES_IT(u32, 4, SUF, ES)                                                                                             \
  FB_LU_QUERIES_IT(u64, 8, SUF, ES)
#define FB_LU_FFI_IT(IT, BYTES, SUF, R, CX)                                                                                     \
  FaerV0_24_PartialPivLuStatus libfaer_v0_23_partial_piv_lu_factor_in_place_##IT##_##SUF(                                       \
      FaerV0_24_MatMut A, FaerV0_24_SliceMut perm_fwd, FaerV0_24_SliceMut perm_bwd, FaerV0_24_Par par, FaerV0_24_MemAlloc mem,   \
      FaerV0_24_PartialPivLuParams params) {                                                                                    \
    (void)par; (void)mem;                                                                                                       \
    return lu_factor_entry<R, CX>(A, perm_fwd, perm_bwd, params, BYTES);                                                        \
  }                                                                                                                             \
  void libfaer_v0_23_partial_piv_lu_solve_in_place_##IT##_##SUF(FaerV0_24_MatRef L, FaerV0_24_MatRef U, FaerV0_24_Conj A_conj,  \
                                                               FaerV0_24_SliceRef perm_fwd, FaerV0_24_SliceRef perm_bwd,        \
                                                               FaerV0_24_MatMut rhs, FaerV0_24_Par par, FaerV0_24_MemAlloc mem) { \
    (void)perm_bwd; (void)par; (void)mem;                                                                                       \
    lu_solve_entry<R, CX>(L, U, A_conj, perm_fwd, rhs, BYTES, false);                                                           \
  }                                                                                                                             \
  void libfaer_v0_23_partial_piv_lu_solve_transpose_in_place_##IT##_##SUF(                                                      \
      FaerV0_24_MatRef L, FaerV0_24_MatRef U, FaerV0_24_Conj A_conj, FaerV0_24_SliceRef perm_fwd, FaerV0_24_SliceRef perm_bwd,   \
      FaerV0_24_MatMut rhs, FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {                                                        \
    (void)perm_fwd; (void)par; (void)mem;                                                                                       \
    lu_solve_entry<R, CX>(L, U, A_conj, perm_bwd, rhs, BYTES, true);                                                            \
  }
#define FB_LU_FFI(SUF, R, CX) FB_LU_FFI_IT(u32, 4, SUF, R, CX) FB_LU_FFI_IT(u64, 8, SUF, R, CX)
FB_LU_QUERIES(f64, sizeof(double))
FB_LU_QUERIES(f32, sizeof(float))
FB_LU_QUERIES(c64, 2 * sizeof(double))
FB_LU_QUERIES(c32, 2 * sizeof(float))
FB_LU_FFI(f64, double, false)
FB_LU_FFI(f32, float, false)
FB_LU_FFI(c64, double, true)
FB_LU_FFI(c32, float, true)
#undef FB_LU_QUERIES_IT
#undef FB_LU_QUERIES
#undef FB_LU_FFI_IT
#undef FB_LU_FFI

// ---- Householder QR (no pivoting), block-Householder sequences and the QR solves ----
// scratch: temp_mat_scratch(block_size, ncols) for the factorization, the block-Householder sequence scratch
// temp_mat_scratch(block_size, rhs_ncols) for the sequences and the solves (solve.rs:3-37)
#define FB_QR_QUERIES(SUF, ES)                                                                                                  \
  FaerV0_24_QrParams libfaer_v0_23_QrParams_##SUF(void) { return FaerV0_24_QrParams{48 * 48, 192 * 256}; }                      \
  size_t libfaer_v0_23_qr_recommended_block_size_##SUF(size_t nrows, size_t ncols) {                                            \
    return (size_t)qr_recommended_block_size((i64)nrows, (i64)ncols);                                                           \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_qr_factor_in_place_scratch_##SUF(size_t nrows, size_t ncols, size_t block_size,                \
                                                                  FaerV0_24_Par par, FaerV0_24_QrParams params) {               \
    (void)nrows; (void)par; (void)params;                                                                                       \
    return FaerV0_24_Layout{block_size * ncols * (ES), 64};                                                                     \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_apply_householder_on_the_left_scratch_##SUF(size_t dim, size_t block_size, size_t rhs_ncols) { \
    (void)dim;                                                                                                                  \
    return FaerV0_24_Layout{block_size * rhs_ncols * (ES), 64};                                                                 \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_apply_householder_transpose_on_the_left_scratch_##SUF(size_t dim, size_t block_size,           \
                                                                                        size_t rhs_ncols) {                     \
    (void)dim;                                                                                                                  \
    return FaerV0_24_Layout{block_size * rhs_ncols * (ES), 64};                                                                 \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_apply_householder_on_the_right_scratch_##SUF(size_t dim, size_t block_size, size_t lhs_nrows) { \
    (void)dim;                                                                                                                  \
    return FaerV0_24_Layout{block_size * lhs_nrows * (ES), 64};                                                                 \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_apply_householder_transpose_on_the_right_scratch_##SUF(size_t dim, size_t block_size,          \
                                                                                         size_t lhs_nrows) {                    \
    (void)dim;                                                                                                                  \
    return FaerV0_24_Layout{block_size * lhs_nrows * (ES), 64};                                                                 \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_qr_solve_lstsq_in_place_scratch_##SUF(size_t nrows, size_t ncols, size_t block_size,           \
                                                                       size_t rhs_ncols, FaerV0_24_Par par) {                   \
    (void)nrows; (void)ncols; (void)par;                                                                                        \
    return FaerV0_24_Layout{block_size * rhs_ncols * (ES), 64};                                                                 \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_qr_solve_in_place_scratch_##SUF(size_t dim, size_t block_size, size_t rhs_ncols,               \
                                                                 FaerV0_24_Par par) {                                           \
    (void)dim; (void)par;                                                                                                       \
    return FaerV0_24_Layout{block_size * rhs_ncols * (ES), 64};                                                                 \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_qr_solve_transpose_in_place_scratch_##SUF(size_t dim, size_t block_size,                       \
                                                                           size_t rhs_ncols, FaerV0_24_Par par) {               \
    (void)dim; (void)par;                                                                                                       \
    return FaerV0_24_Layout{block_size * rhs_ncols * (ES), 64};                                                                 \
  }
#define FB_QR_FFI(SUF, R, CX)                                                                                                   \
  FaerV0_24_QrStatus libfaer_v0_23_qr_factor_in_place_##SUF(FaerV0_24_MatMut A, FaerV0_24_MatMut Q_coeff, FaerV0_24_Par par,    \
                                                            FaerV0_24_MemAlloc mem, FaerV0_24_QrParams params) {                \
    (void)par; (void)mem;                                                                                                       \
    return qr_factor_entry<R, CX>(A, Q_coeff, params);                                                                          \
  }                                                                                                                             \
  void libfaer_v0_23_apply_householder_on_the_left_##SUF(FaerV0_24_MatRef basis, FaerV0_24_MatRef factor, FaerV0_24_Conj conj,  \
                                                         FaerV0_24_MatMut rhs, FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {     \
    (void)par; (void)mem;                                                                                                       \
    householder_seq_entry<R, CX>(basis, factor, conj, rhs, false);                                                              \
  }                                                                                                                             \
  void libfaer_v0_23_apply_householder_transpose_on_the_left_##SUF(FaerV0_24_MatRef basis, FaerV0_24_MatRef factor,             \
                                                                   FaerV0_24_Conj conj, FaerV0_24_MatMut rhs,                   \
                                                                   FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {                 \
    (void)par; (void)mem;                                                                                                       \
    householder_seq_entry<R, CX>(basis, factor, conj, rhs, true);                                                               \
  }                                                                                                                             \
  /* on the right = the transposed sequence on the left of the transposed view, and vice versa (householder.rs:813-854) */     \
  void libfaer_v0_23_apply_householder_on_the_right_##SUF(FaerV0_24_MatRef basis, FaerV0_24_MatRef factor, FaerV0_24_Conj conj, \
                                                          FaerV0_24_MatMut lhs, FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {    \
    (void)par; (void)mem;                                                                                                       \
    householder_seq_entry<R, CX>(basis, factor, conj, transposed(lhs), true);                                                   \
  }                                                                                                                             \
  void libfaer_v0_23_apply_householder_transpose_on_the_right_##SUF(FaerV0_24_MatRef basis, FaerV0_24_MatRef factor,            \
                                                                    FaerV0_24_Conj conj, FaerV0_24_MatMut lhs,                  \
                                                                    FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {                \
    (void)par; (void)mem;                                                                                                       \
    householder_seq_entry<R, CX>(basis, factor, conj, transposed(lhs), false);                                                  \
  }                                                                                                                             \
  void libfaer_v0_23_qr_solve_lstsq_in_place_##SUF(FaerV0_24_MatRef Q_basis, FaerV0_24_MatRef Q_coeff, FaerV0_24_MatRef Rm,     \
                                                   FaerV0_24_Conj A_conj, FaerV0_24_MatMut rhs, FaerV0_24_Par par,              \
                                                   FaerV0_24_MemAlloc mem) {                                                    \
    (void)par; (void)mem;                                                                                                       \
    qr_solve_entry<R, CX>(Q_basis, Q_coeff, Rm, A_conj, rhs, 0);                                                                \
  }                                                                                                                             \
  void libfaer_v0_23_qr_solve_in_place_##SUF(FaerV0_24_MatRef Q_basis, FaerV0_24_MatRef Q_coeff, FaerV0_24_MatRef Rm,           \
                                             FaerV0_24_Conj A_conj, FaerV0_24_MatMut rhs, FaerV0_24_Par par,                    \
                                             FaerV0_24_MemAlloc mem) {                                                          \
    (void)par; (void)mem;                                                                                                       \
    qr_solve_entry<R, CX>(Q_basis, Q_coeff, Rm, A_conj, rhs, 1);                                                                \
  }                                                                                                                             \
  void libfaer_v0_23_qr_solve_transpose_in_place_##SUF(FaerV0_24_MatRef Q_basis, FaerV0_24_MatRef Q_coeff,                      \
                                                       FaerV0_24_MatRef Rm, FaerV0_24_Conj A_conj, FaerV0_24_MatMut rhs,        \
                                                       FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {                             \
    (void)par; (void)mem;                                                                                                       \
    qr_solve_entry<R, CX>(Q_basis, Q_coeff, Rm, A_conj, rhs, 2);                                                                \
  }
FB_QR_QUERIES(f64, sizeof(double))
FB_QR_QUERIES(f32, sizeof(float))
FB_QR_QUERIES(c64, 2 * sizeof(double))
FB_QR_QUERIES(c32, 2 * sizeof(float))
FB_QR_FFI(f64, double, false)
FB_QR_FFI(f32, float, false)
FB_QR_FFI(c64, double, true)
FB_QR_FFI(c32, float, true)
#undef FB_QR_QUERIES
#undef FB_QR_FFI

// ---- SVD / self-adjoint EVD for real T (svd.cu / evd.cu: values by bisection; svd_vectors.cu + tridiag_dc.cu: with vectors) ----
#define FB_SVD_EVD_FFI(SUF, T)                                                                                                  \
  FaerV0_24_SvdStatus libfaer_v0_23_svd_##SUF(FaerV0_24_MatRef A, FaerV0_24_MatMut U, FaerV0_24_VecMut S, FaerV0_24_MatMut V,   \
                                              FaerV0_24_Par par, FaerV0_24_MemAlloc mem, FaerV0_24_SvdParams params) {          \
    (void)par; (void)mem;                                                                                                       \
    return svd_entry<T>(A, U, S, V, params.qr_ratio_threshold);                                                                 \
  }                                                                                                                             \
  FaerV0_24_EvdStatus libfaer_v0_23_self_adjoint_evd_##SUF(FaerV0_24_MatRef A, FaerV0_24_MatMut U, FaerV0_24_VecMut S,          \
                                                           FaerV0_24_Par par, FaerV0_24_MemAlloc mem,                           \
                                                           FaerV0_24_SelfAdjointEvdParams params) {                             \
    (void)par; (void)mem; (void)params;                                                                                         \
    return self_adjoint_evd_entry<T>(A, U, S);                                                                                  \
  }
FB_SVD_EVD_FFI(f64, double)
FB_SVD_EVD_FFI(f32, float)
#undef FB_SVD_EVD_FFI

// ---- reconstruct / inverse on the factors, f64 (reconstruct.cu; qr_reconstruct also f32; the queries: ffi_types.cu) ----
void libfaer_v0_23_llt_reconstruct_f64(FaerV0_24_MatMut A, FaerV0_24_MatRef L, FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {
  (void)par; (void)mem;
  FB_ENTRY();
  cudaStream_t st = current_stream();
  // only the lower triangle is written: the rest of A must survive the round trip
  StagedMat a = stage(A, sizeof(double), true, st), l = stage(L, sizeof(double), st);
  llt_reconstruct_f64(st, a.view<double>(), l.view<const double>());
  finish_all(st, {&a, &l});
}
void libfaer_v0_23_llt_inverse_f64(FaerV0_24_MatMut A_inv, FaerV0_24_MatRef L, FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {
  (void)par; (void)mem;
  FB_ENTRY();
  cudaStream_t st = current_stream();
  StagedMat a = stage(A_inv, sizeof(double), true, st), l = stage(L, sizeof(double), st);
  llt_inverse_f64(st, a.view<double>(), l.view<const double>());
  finish_all(st, {&a, &l});
}
#define FB_LU_RECON_FFI(IT, BYTES)                                                                                              \
  void libfaer_v0_23_partial_piv_lu_reconstruct_##IT##_f64(FaerV0_24_MatMut A, FaerV0_24_MatRef L, FaerV0_24_MatRef U,          \
                                                           FaerV0_24_SliceRef perm_fwd, FaerV0_24_SliceRef perm_bwd,            \
                                                           FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {                         \
    (void)perm_fwd; (void)par; (void)mem;                                                                                       \
    lu_recon_entry(A, L, U, perm_bwd, BYTES, false);                                                                            \
  }                                                                                                                             \
  void libfaer_v0_23_partial_piv_lu_inverse_##IT##_f64(FaerV0_24_MatMut A, FaerV0_24_MatRef L, FaerV0_24_MatRef U,              \
                                                       FaerV0_24_SliceRef perm_fwd, FaerV0_24_SliceRef perm_bwd,                \
                                                       FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {                             \
    (void)perm_bwd; (void)par; (void)mem;                                                                                       \
    lu_recon_entry(A, L, U, perm_fwd, BYTES, true);                                                                             \
  }
FB_LU_RECON_FFI(u32, 4)
FB_LU_RECON_FFI(u64, 8)
#undef FB_LU_RECON_FFI
#define FB_QR_RECON_FFI(SUF, T)                                                                                                 \
  void libfaer_v0_23_qr_reconstruct_##SUF(FaerV0_24_MatMut A, FaerV0_24_MatRef Q_basis, FaerV0_24_MatRef Q_coeff,               \
                                          FaerV0_24_MatRef R, FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {                      \
    (void)par; (void)mem;                                                                                                       \
    FB_ENTRY();                                                                                                                 \
    cudaStream_t st = current_stream();                                                                                         \
    StagedMat a = stage(A, sizeof(T), false, st), b = stage(Q_basis, sizeof(T), st), f = stage(Q_coeff, sizeof(T), st),         \
              r = stage(R, sizeof(T), st);                                                                                      \
    qr_reconstruct<T>(st, a.view<T>(), b.view<const T>(), f.view<const T>(), r.view<const T>());                                \
    finish_all(st, {&a, &b, &f, &r});                                                                                           \
  }
FB_QR_RECON_FFI(f64, double)
FB_QR_RECON_FFI(f32, float)
#undef FB_QR_RECON_FFI
void libfaer_v0_23_qr_inverse_f64(FaerV0_24_MatMut A, FaerV0_24_MatRef Q_basis, FaerV0_24_MatRef Q_coeff, FaerV0_24_MatRef R,
                                  FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {
  (void)par; (void)mem;
  FB_ENTRY();
  cudaStream_t st = current_stream();
  StagedMat a = stage(A, sizeof(double), false, st), b = stage(Q_basis, sizeof(double), st), f = stage(Q_coeff, sizeof(double), st),
            r = stage(R, sizeof(double), st);
  qr_inverse_f64(st, a.view<double>(), b.view<const double>(), f.view<const double>(), r.view<const double>());
  finish_all(st, {&a, &b, &f, &r});
}

// ---- global par / alloc ----
FaerV0_24_Par libfaer_v0_23_get_global_par(void) {
  FaerV0_24_Par p;
  p.tag = (FaerV0_24_ParTag)g_par_tag.load();
  p.nthreads = g_par_threads.load();
  return p;
}
void libfaer_v0_23_set_global_par(FaerV0_24_Par par) {
  g_par_tag.store((int)par.tag);
  g_par_threads.store(par.nthreads);
}
void* libfaer_v0_23_alloc(size_t size, size_t align) {
  // reference: std::alloc::alloc(Layout::from_size_align(size, align)) (faer-ffi/src/lib.rs:2537-2552)
  if (align < sizeof(void*)) align = sizeof(void*);
  void* p = nullptr;
  if (posix_memalign(&p, align, size ? size : 1) != 0) return nullptr;
  return p;
}
void libfaer_v0_23_dealloc(void* ptr, size_t size, size_t align) {
  (void)size; (void)align;
  free(ptr);
}

// ---- extensions ----
int faer_b200_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  return n;
}
void faer_b200_set_stream(void* cuda_stream) { std::lock_guard<std::recursive_mutex> lock(entry_mutex()); set_current_stream((cudaStream_t)cuda_stream); }
unsigned long long faer_b200_launch_count(void) { return g_launch_count; }
void faer_b200_release_workspace(void) { std::lock_guard<std::recursive_mutex> lock(entry_mutex()); ws_release_all(); }
void faer_b200_profile_begin(void) { std::lock_guard<std::recursive_mutex> lock(entry_mutex()); profile_begin(); }
void faer_b200_profile_end(double* flops, double* ms, unsigned long long* count) {
  std::lock_guard<std::recursive_mutex> lock(entry_mutex()); 
  profile_end(flops, ms, count);
}
// ---- multi-GPU extensions (dist.cu) ----
int faer_b200_dist_unique_id(void* out128) { return dist_unique_id(out128); }
int faer_b200_dist_init(int rank, int nranks, const void* id128) {
  std::lock_guard<std::recursive_mutex> lock(entry_mutex()); 
  return dist_init(rank, nranks, id128);
}
void faer_b200_dist_finalize(void) { std::lock_guard<std::recursive_mutex> lock(entry_mutex()); dist_finalize(); }
FaerV0_24_LltStatus faer_b200_dist_llt_factor_in_place_f64(void* A_local, size_t ld, size_t n, size_t nb,
                                                           FaerV0_24_LltRegularization regularization, int lookahead) {
  double delta, eps;
  read_regularization(regularization, delta, eps);
  FB_ASSERT(n == 0 || is_device_pointer(A_local), "distributed entry points take device-resident local matrices");
  return llt_status(dist_llt_f64((double*)A_local, (i64)ld, (i64)n, (i64)nb, delta, eps, lookahead));
}

size_t faer_b200_dist_partial_piv_lu_factor_in_place_f64(void* A_local, size_t ld, size_t n, size_t nb, long long* perm_fwd,
                                                         long long* perm_inv, int lookahead) {
  FB_ASSERT(n == 0 || is_device_pointer(A_local), "distributed entry points take device-resident local matrices");
  return dist_lu_f64((double*)A_local, (i64)ld, (i64)n, (i64)nb, perm_fwd, perm_inv, lookahead);
}

long long faer_b200_dist_qr_factor_in_place_f64(void* A_local, size_t ld, size_t nrows, size_t ncols, size_t block_size, void* Q_coeff,
                                                int flags) {
  FB_ASSERT(ncols == 0 || (is_device_pointer(A_local) && is_device_pointer(Q_coeff)), "distributed entry points take device-resident matrices");
  return dist_qr_f64((double*)A_local, (i64)ld, (i64)nrows, (i64)ncols, (i64)block_size, (double*)Q_coeff, flags);
}
long long faer_b200_dist_qr_factor_in_place_f32(void* A_local, size_t ld, size_t nrows, size_t ncols, size_t block_size, void* Q_coeff,
                                                int flags) {
  FB_ASSERT(ncols == 0 || (is_device_pointer(A_local) && is_device_pointer(Q_coeff)), "distributed entry points take device-resident matrices");
  return dist_qr_f32((float*)A_local, (i64)ld, (i64)nrows, (i64)ncols, (i64)block_size, (float*)Q_coeff, flags);
}


void faer_b200_spicy_matmul_f64(FaerV0_24_MatMut C, FaerV0_24_Block C_block, const unsigned long long* row_idx, size_t nrow_idx,
                                const unsigned long long* col_idx, size_t ncol_idx, FaerV0_24_Accum accum, FaerV0_24_MatRef A,
                                FaerV0_24_MatRef B, const double* D, const FaerV0_24_Scalar* alpha) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  FB_ASSERT(A.ncols == B.nrows, "spicy_matmul shape mismatch");
  FB_ASSERT(!row_idx || nrow_idx == A.nrows, "spicy_matmul: one row index per row of A");
  FB_ASSERT(!col_idx || ncol_idx == B.ncols, "spicy_matmul: one column index per column of B");
  if (row_idx && !is_device_pointer(row_idx))
    for (size_t i = 0; i < nrow_idx; ++i) FB_ASSERT(row_idx[i] < C.nrows, "spicy_matmul: row index out of range");
  if (col_idx && !is_device_pointer(col_idx))
    for (size_t j = 0; j < ncol_idx; ++j) FB_ASSERT(col_idx[j] < C.ncols, "spicy_matmul: column index out of range");
  const double a = read_real<double>(alpha);
  // scattered destinations keep the untouched entries: always stage the old contents
  StagedMat c = stage(C, sizeof(double), true, st), lhs = stage(A, sizeof(double), st), rhs = stage(B, sizeof(double), st);
  // indices and diagonal: device copies of host arrays
  auto to_dev = [&](const void* p, size_t bytes) -> void* {
    if (!p || bytes == 0) return nullptr;
    if (is_device_pointer(p)) return (void*)p;
    void* d = ws_alloc(bytes);
    FB_CUDA_CHECK(cudaMemcpyAsync(d, p, bytes, cudaMemcpyHostToDevice, st));
    return d;
  };
  void* dri = to_dev(row_idx, nrow_idx * 8);
  void* dci = to_dev(col_idx, ncol_idx * 8);
  void* dd = to_dev(D, (size_t)A.ncols * 8);
  spicy_matmul_f64(st, c.view<double>(), (int)C_block, (const long long*)dri, (const long long*)dci,
                   accum == FaerV0_24_Accum_Add ? 1 : 0, lhs.view<const double>(), rhs.view<const double>(), (const double*)dd, 1, a);
  finish_all(st, {&c, &lhs, &rhs});
  if (dri && dri != (void*)row_idx) ws_free(dri);
  if (dci && dci != (void*)col_idx) ws_free(dci);
  if (dd && dd != (void*)D) ws_free(dd);
}

// ---- inner seam: the type-erased product call faer makes in three places (private_gemm_x86::gemm at
// faer/src/linalg/matmul/mod.rs:1373-1411, matmul/triangular.rs:641-680, matmul/internal/mod.rs:143-201), same parameter list.
void faer_b200_gemm(int dtype, int itype, int instr_set, size_t m, size_t n, size_t k, void* dst, ptrdiff_t dst_rs, ptrdiff_t dst_cs,
                    const void* row_idx, const void* col_idx, int dst_kind, int accum, const void* lhs, ptrdiff_t lhs_rs,
                    ptrdiff_t lhs_cs, bool conj_lhs, const void* diag, ptrdiff_t diag_stride, const void* rhs, ptrdiff_t rhs_rs,
                    ptrdiff_t rhs_cs, bool conj_rhs, const void* alpha, size_t n_threads) {
  (void)instr_set; (void)n_threads;
  FB_ASSERT(dtype >= 0 && dtype <= 3, "faer_b200_gemm: dtype must be FaerB200_GemmDType_{F32,F64,C32,C64}");
  FB_ASSERT(dst_kind >= 0 && dst_kind <= 2, "faer_b200_gemm: dst_kind must be FaerB200_GemmDstKind_{Lower,Upper,Full}");
  const FaerV0_24_Accum acc = accum ? FaerV0_24_Accum_Add : FaerV0_24_Accum_Replace;
  const int block = dst_kind == FaerB200_GemmDstKind_Full ? (int)FaerV0_24_Block_Rectangular
                                                          : dst_kind == FaerB200_GemmDstKind_Lower ? (int)FaerV0_24_Block_TriangularLower
                                                                                                   : (int)FaerV0_24_Block_TriangularUpper;
  if (block != (int)FaerV0_24_Block_Rectangular) FB_ASSERT(m == n, "faer_b200_gemm: a triangular destination is square");
  const bool plain = !row_idx && !col_idx && !diag;
  FaerV0_24_MatRef A{lhs, m, k, lhs_rs, lhs_cs}, B{rhs, k, n, rhs_rs, rhs_cs};
  if (plain && dtype != FaerB200_GemmDType_F64) {
    FaerV0_24_MatMut C{dst, m, n, dst_rs, dst_cs};
    const FaerV0_24_Scalar* a = (const FaerV0_24_Scalar*)alpha;
    if (dtype == FaerB200_GemmDType_F32) matmul_entry<float, false>(C, block, acc, A, RECT, B, RECT, a);
    else if (dtype == FaerB200_GemmDType_C64) matmul_entry<double, true>(C, block, acc, A, RECT, B, RECT, a, conj_lhs, conj_rhs);
    else matmul_entry<float, true>(C, block, acc, A, RECT, B, RECT, a, conj_lhs, conj_rhs);
    return;
  }
  FB_ASSERT(dtype == FaerB200_GemmDType_F64, "faer_b200_gemm: scatter indices / diagonal scaling are built for f64 only");
  FB_ENTRY();
  cudaStream_t st = current_stream();
  // index arrays as 64-bit device arrays; the destination's extent is what the indices reach
  auto host_idx = [&](const void* p, size_t cnt) {
    std::vector<unsigned long long> v(cnt);
    if (!p) return v;
    const size_t w = itype == FaerB200_GemmIType_U32 ? 4 : 8;
    std::vector<unsigned char> raw(cnt * w);
    if (is_device_pointer(p)) FB_CUDA_CHECK(cudaMemcpy(raw.data(), p, raw.size(), cudaMemcpyDeviceToHost));
    else memcpy(raw.data(), p, raw.size());
    for (size_t i = 0; i < cnt; ++i) v[i] = w == 4 ? (unsigned long long)((const uint32_t*)raw.data())[i] : ((const uint64_t*)raw.data())[i];
    return v;
  };
  const std::vector<unsigned long long> ri = host_idx(row_idx, m), ci = host_idx(col_idx, n);
  size_t c_rows = m, c_cols = n;
  if (row_idx) { c_rows = 0; for (auto x : ri) c_rows = std::max<size_t>(c_rows, (size_t)x + 1); }
  if (col_idx) { c_cols = 0; for (auto x : ci) c_cols = std::max<size_t>(c_cols, (size_t)x + 1); }
  auto to_dev = [&](const void* p, size_t bytes) -> void* {
    if (bytes == 0) return nullptr;
    void* d = ws_alloc(bytes);
    FB_CUDA_CHECK(cudaMemcpyAsync(d, p, bytes, cudaMemcpyHostToDevice, st));
    return d;
  };
  void* dri = row_idx ? to_dev(ri.data(), m * 8) : nullptr;
  void* dci = col_idx ? to_dev(ci.data(), n * 8) : nullptr;
  // diagonal: device pointers are used in place (with their stride), host ones are gathered into a compact device copy
  const double* dd = (const double*)diag;
  void* dd_own = nullptr;
  i64 dstride = (i64)diag_stride;
  std::vector<double> hd;
  if (diag && !is_device_pointer(diag)) {
    hd.resize(k);
    for (size_t q = 0; q < k; ++q) hd[q] = ((const double*)diag)[(ptrdiff_t)q * diag_stride];
    dd_own = to_dev(hd.data(), k * 8);
    dd = (const double*)dd_own;
    dstride = 1;
  }
  const double a = read_real<double>(alpha);
  FaerV0_24_MatMut C{dst, c_rows, c_cols, dst_rs, dst_cs};
  const bool keep_old = accum != 0 || row_idx || col_idx || block != (int)FaerV0_24_Block_Rectangular;
  StagedMat c = stage(C, sizeof(double), keep_old, st), l = stage(A, sizeof(double), st), r = stage(B, sizeof(double), st);
  if (m > 0 && n > 0)
    spicy_matmul_f64(st, c.view<double>(), block, (const long long*)dri, (const long long*)dci, accum ? 1 : 0,
                     l.view<const double>(), r.view<const double>(), dd, dstride, a);
  finish_all(st, {&c, &l, &r});  // synchronises the stream: the host vectors above may go
  if (dri) ws_free(dri);
  if (dci) ws_free(dci);
  if (dd_own) ws_free(dd_own);
}

int faer_b200_set_option(const char* name, long long value) { return set_option_by_name(name, value) ? 0 : -1; }
long long faer_b200_get_option(const char* name) { return get_option_by_name(name); }

const char* faer_b200_version(void) { return "faer_b200 0.1 (faer-ffi v0_23 ABI subset, sm_100a)"; }

}  // extern "C"
