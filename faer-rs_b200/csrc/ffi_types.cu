// extern "C" boundary, second translation unit: the entry points whose drivers are the flat-map files (reconstruct_types.cu,
// ldlt_types.cu, cplx_condensed.cu) — `*_reconstruct` / `*_inverse` for f32 / c64 / c32, LDLT beyond the f64 factorization, `svd` /
// `self_adjoint_evd` for complex T. Same conventions as ffi.cu (by-value PODs, synchronous on return, abort() on precondition
// violations, host buffers staged, device buffers used in place). Kept apart from ffi.cu so that this unit, runtime.cu and the
// three drivers also build for the host (tools/emul/ffi_types_host.cpp: the staging layer and the drivers end to end on the CPU).
// For the same reason the default-params and scratch queries of svd / self_adjoint_evd, LDLT and the reconstructs / inverses live
// here for every dtype (the Python layer queries them on the host library too); LLT's, LU's and QR's stay with their entry points
// in ffi.cu (qr_recommended_block_size calls into qr.cu).
#include "ffi_common.cuh"
#include "flat_map.cuh"
#include "gemm_f32.cuh"
#include "runtime.cuh"
#include "tensor_ops.cuh"

#include <memory>

using namespace fb;

namespace {

// ---- reconstruct / inverse on the factors for f32 / c64 / c32 (reconstruct_types.cu; scalar kind <R, CX>) ----
template <class R, bool CX>
void llt_recon_entry_t(FaerV0_24_MatMut A, FaerV0_24_MatRef L, bool inverse) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t es = elem_bytes<R, CX>();
  // only the lower triangle is written: the rest of A must survive the round trip
  StagedMat a = stage(A, es, true, st), l = stage(L, es, st);
  if (inverse) llt_inverse_t<R, CX>(st, a.view<R>(), l.view<const R>());
  else llt_reconstruct_t<R, CX>(st, a.view<R>(), l.view<const R>());
  finish_all(st, {&a, &l});
}
template <class R, bool CX>
void lu_recon_entry_t(FaerV0_24_MatMut A, FaerV0_24_MatRef L, FaerV0_24_MatRef U, FaerV0_24_SliceRef perm, int idx_bytes,
                      bool inverse) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t es = elem_bytes<R, CX>();
  const std::vector<long long> p = read_perm_checked(perm, L.nrows, idx_bytes);
  StagedMat a = stage(A, es, false, st), l = stage(L, es, st), u = stage(U, es, st);
  if (inverse) lu_inverse_t<R, CX>(st, a.view<R>(), l.view<const R>(), u.view<const R>(), p.data());
  else lu_reconstruct_t<R, CX>(st, a.view<R>(), l.view<const R>(), u.view<const R>(), p.data());
  finish_all(st, {&a, &l, &u});
}
template <class R, bool CX>
void qr_recon_entry_t(FaerV0_24_MatMut A, FaerV0_24_MatRef Q_basis, FaerV0_24_MatRef Q_coeff, FaerV0_24_MatRef Rm, bool inverse) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t es = elem_bytes<R, CX>();
  StagedMat a = stage(A, es, false, st), b = stage(Q_basis, es, st), f = stage(Q_coeff, es, st), r = stage(Rm, es, st);
  if (inverse) qr_inverse_t<R, CX>(st, a.view<R>(), b.view<const R>(), f.view<const R>(), r.view<const R>());
  else qr_reconstruct_t<R, CX>(st, a.view<R>(), b.view<const R>(), f.view<const R>(), r.view<const R>());
  finish_all(st, {&a, &b, &f, &r});
}

// ---- `svd` / `self_adjoint_evd` for complex T (cplx_condensed.cu); S holds T-typed entries (value, 0), strides in complex units ----
template <class R>
FaerV0_24_EvdStatus self_adjoint_evd_entry_cx(FaerV0_24_MatRef A, FaerV0_24_MatMut U, FaerV0_24_VecMut S) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t n = A.nrows, es = elem_bytes<R, true>();
  FB_ASSERT(A.ncols == n && S.len == n && (n == 0 || S.stride >= 1), "self_adjoint_evd: square A, S of length n, positive stride");
  const bool want_u = U.ncols != 0;
  if (want_u) FB_ASSERT(U.nrows == n && U.ncols == n, "self_adjoint_evd: U must be n x n (or have no columns)");
  if (n == 0) return evd_status(true);
  StagedMat a = stage(A, es, st);
  R* s_dev = (R*)ws_alloc(n * es);
  bool ok;
  if (want_u) {
    StagedMat u = stage(U, es, false, st);
    ok = self_adjoint_evd_cx<R>(st, a.view<const R>(), u.view<R>(), s_dev, 1);
    if (ok) copy_out_vector(S, s_dev, n, es, st);
    finish_all(st, {&a, &u});
  } else {
    ok = self_adjoint_evd_cx<R>(st, a.view<const R>(), View<R>{nullptr, 0, 0, 1, 1}, s_dev, 1);
    if (ok) copy_out_vector(S, s_dev, n, es, st);
    finish_all(st, {&a});
  }
  ws_free(s_dev);
  return evd_status(ok);
}
template <class R>
FaerV0_24_SvdStatus svd_entry_cx(FaerV0_24_MatRef A, FaerV0_24_MatMut U, FaerV0_24_VecMut S, FaerV0_24_MatMut V) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t size = A.nrows < A.ncols ? A.nrows : A.ncols, es = elem_bytes<R, true>();
  FB_ASSERT(S.len == size && (size == 0 || S.stride >= 1), "svd: S must have min(nrows, ncols) entries and a positive stride");
  const bool want_u = U.ncols != 0, want_v = V.ncols != 0;
  if (want_u) FB_ASSERT(U.nrows == A.nrows && (U.ncols == A.nrows || U.ncols == size), "svd: U must be nrows x {size, nrows}");
  if (want_v) FB_ASSERT(V.nrows == A.ncols && (V.ncols == A.ncols || V.ncols == size), "svd: V must be ncols x {size, ncols}");
  if (size == 0 && !want_u && !want_v) return svd_status(true);
  StagedMat a = stage(A, es, st);
  R* s_dev = (R*)ws_alloc((size + 1) * es);
  bool ok;
  if (want_u || want_v) {
    StagedMat u = stage(U, es, false, st), v = stage(V, es, false, st);
    View<R> uv = want_u ? u.view<R>() : View<R>{nullptr, 0, 0, 1, 1};
    View<R> vv = want_v ? v.view<R>() : View<R>{nullptr, 0, 0, 1, 1};
    ok = svd_cx<R>(st, a.view<const R>(), uv, s_dev, 1, vv);
    if (ok && size) copy_out_vector(S, s_dev, size, es, st);
    finish_all(st, {&a, &u, &v});
  } else {
    ok = svd_cx<R>(st, a.view<const R>(), View<R>{nullptr, 0, 0, 1, 1}, s_dev, 1, View<R>{nullptr, 0, 0, 1, 1});
    if (ok && size) copy_out_vector(S, s_dev, size, es, st);
    finish_all(st, {&a});
  }
  ws_free(s_dev);
  return svd_status(ok);
}

// ---- LDLT for the other scalar kinds (ldlt_types.cu); D arrives as a VecRef of T-typed entries ----
template <class R, bool CX>
FaerV0_24_LdltStatus ldlt_factor_entry_t(FaerV0_24_MatMut A, FaerV0_24_LdltRegularization regularization) {
  FB_ENTRY();
  FB_ASSERT(A.nrows == A.ncols, "LDLT needs a square matrix");
  cudaStream_t st = current_stream();
  R delta, eps;
  read_regularization(regularization, delta, eps);
  const SignsArg signs(regularization.dynamic_regularization_signs, A.nrows, st);
  StagedMat a = stage(A, elem_bytes<R, CX>(), true, st);
  const LdltResult r = ldlt_in_place_t<R, CX>(st, a.view<R>(), delta, eps, signs.ptr);
  finish_all(st, {&a});
  return ldlt_status(r);
}
template <class R, bool CX>
void ldlt_solve_entry_t(FaerV0_24_MatRef L, FaerV0_24_VecRef D, FaerV0_24_Conj A_conj, FaerV0_24_MatMut rhs) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t n = L.nrows, es = elem_bytes<R, CX>();
  FB_ASSERT(L.ncols == n && D.len == n && rhs.nrows == n, "LDLT solve shape mismatch");
  if (n == 0 || rhs.ncols == 0) return;
  StagedMat l = stage(L, es, st), r = stage(rhs, es, true, st);
  const DiagArg<R, CX> d(D, n, st);
  ldlt_solve_in_place_t<R, CX>(st, l.view<const R>(), d.ptr, d.stride, A_conj == FaerV0_24_Conj_Yes, r.view<R>());
  finish_all(st, {&l, &r});
}
template <class R, bool CX>
void ldlt_recon_entry_t(FaerV0_24_MatMut A, FaerV0_24_MatRef L, FaerV0_24_VecRef D, bool inverse) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t n = L.nrows, es = elem_bytes<R, CX>();
  FB_ASSERT(L.ncols == n && D.len == n && A.nrows == n && A.ncols == n, "LDLT reconstruct / inverse shape mismatch");
  if (n == 0) return;
  // only the lower triangle is written: the rest of A must survive the round trip
  StagedMat a = stage(A, es, true, st), l = stage(L, es, st);
  const DiagArg<R, CX> d(D, n, st);
  if (inverse) ldlt_inverse_t<R, CX>(st, a.view<R>(), l.view<const R>(), d.ptr, d.stride);
  else ldlt_reconstruct_t<R, CX>(st, a.view<R>(), l.view<const R>(), d.ptr, d.stride);
  finish_all(st, {&a, &l});
}

// ---- reductions to condensed form as extension entry points (svd/bidiag.rs:47-256, evd/tridiag.rs:274-529) ----
// The condensed-form kernels want a column-major matrix (row stride 1). Any other layout (a row-major or strided HOST view keeps
// its layout in the device mirror; a device view is whatever the caller has) goes through a compact column-major copy.
#if defined(__CUDACC__)
#define FT_HD __host__ __device__ __forceinline__
#else
#define FT_HD inline
#endif
template <class T>
struct CopyStrided {
  T* dst; i64 drs, dcs; const T* src; i64 srs, scs, m, n;
  FT_HD void operator()(i64 i, i64 j) const {
    if (i < m && j < n) dst[i * drs + j * dcs] = src[i * srs + j * scs];
  }
};
template <class T>
struct ColMajorWork {
  cudaStream_t st;
  View<T> orig, work;
  T* buf = nullptr;
  ColMajorWork(cudaStream_t st_, View<T> v) : st(st_), orig(v), work(v) {
    if (v.rs != 1 && v.nrows > 0 && v.ncols > 0) {
      buf = (T*)ws_alloc((size_t)v.nrows * (size_t)v.ncols * sizeof(T));
      DevRun run{st};
      run(CopyStrided<T>{buf, 1, v.nrows, v.ptr, v.rs, v.cs, v.nrows, v.ncols}, v.nrows, v.ncols);
      work = View<T>{buf, v.nrows, v.ncols, 1, v.nrows};
    }
  }
  void finish() {
    if (!buf) return;
    DevRun run{st};
    run(CopyStrided<T>{orig.ptr, orig.rs, orig.cs, buf, 1, orig.nrows, orig.nrows, orig.ncols}, orig.nrows, orig.ncols);
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    ws_free(buf);
    buf = nullptr;
  }
};
template <class T>
void bidiag_entry(FaerV0_24_MatMut A, FaerV0_24_MatMut Hl, FaerV0_24_MatMut Hr) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  StagedMat a = stage(A, sizeof(T), true, st);
  StagedMat hl = stage(Hl, sizeof(T), true, st);
  StagedMat hr = stage(Hr, sizeof(T), true, st);
  ColMajorWork<T> w(st, a.view<T>());
  bidiag_in_place<T>(st, w.work, hl.view<T>(), hr.view<T>());
  w.finish();
  finish_all(st, {&a, &hl, &hr});
}
template <class T>
void tridiag_entry(FaerV0_24_MatMut A, FaerV0_24_MatMut H) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  StagedMat a = stage(A, sizeof(T), true, st);
  StagedMat h = stage(H, sizeof(T), true, st);
  ColMajorWork<T> w(st, a.view<T>());
  tridiag_in_place<T>(st, w.work, h.view<T>());
  w.finish();
  finish_all(st, {&a, &h});
}

// ---- triangular inverses (triangular_inverse.rs; faer-ffi/src/lib.rs:938-980) ----
template <class R, bool CX>
void inverse_triangular_entry_t(FaerV0_24_MatMut dst, FaerV0_24_MatRef src, bool lower, bool unit) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t es = elem_bytes<R, CX>();
  FB_ASSERT(dst.nrows == dst.ncols && src.nrows == dst.nrows && src.ncols == dst.ncols, "inverse_triangular shape mismatch");
  if (dst.nrows == 0) return;
  // only the triangle is written: the rest of dst must survive the round trip
  StagedMat d = stage(dst, es, true, st);
  StagedMat s = stage(src, es, st);
  inverse_triangular_t<R, CX>(st, d.view<R>(), s.view<const R>(), lower, unit);
  finish_all(st, {&d, &s});
}

// ---- Hessenberg reduction (extension; evd/hessenberg.rs:549-567) ----
template <class R, bool CX>
void hessenberg_entry_t(FaerV0_24_MatMut A, FaerV0_24_MatMut H) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t es = elem_bytes<R, CX>();
  FB_ASSERT(A.nrows == A.ncols && H.ncols == (A.nrows > 0 ? A.nrows - 1 : 0), "hessenberg_in_place: square A, householder factor bs x (n - 1)");
  StagedMat a = stage(A, es, true, st);
  StagedMat h = stage(H, es, false, st);
  hessenberg_in_place_t<R, CX>(st, a.view<R>(), h.view<R>());
  finish_all(st, {&a, &h});
}

// complex reductions to condensed form (extensions; cplx_condensed.cu)
template <class R>
void bidiag_entry_cx(FaerV0_24_MatMut A, FaerV0_24_MatMut Hl, FaerV0_24_MatMut Hr) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t es = elem_bytes<R, true>();
  StagedMat a = stage(A, es, true, st);
  StagedMat hl = stage(Hl, es, false, st);
  StagedMat hr = stage(Hr, es, false, st);
  bidiag_in_place_cx<R>(st, a.view<R>(), hl.view<R>(), hr.view<R>());
  finish_all(st, {&a, &hl, &hr});
}
template <class R>
void tridiag_entry_cx(FaerV0_24_MatMut A, FaerV0_24_MatMut H) {
  FB_ENTRY();
  cudaStream_t st = current_stream();
  const size_t es = elem_bytes<R, true>();
  StagedMat a = stage(A, es, true, st);
  StagedMat h = stage(H, es, false, st);
  tridiag_in_place_cx<R>(st, a.view<R>(), h.view<R>());
  finish_all(st, {&a, &h});
}

}  // namespace

extern "C" {

// ---- extensions: reductions to condensed form ----
void faer_b200_bidiag_in_place_f64(FaerV0_24_MatMut A, FaerV0_24_MatMut H_left, FaerV0_24_MatMut H_right) {
  bidiag_entry<double>(A, H_left, H_right);
}
void faer_b200_bidiag_in_place_f32(FaerV0_24_MatMut A, FaerV0_24_MatMut H_left, FaerV0_24_MatMut H_right) {
  bidiag_entry<float>(A, H_left, H_right);
}

void faer_b200_bidiag_in_place_c64(FaerV0_24_MatMut A, FaerV0_24_MatMut H_left, FaerV0_24_MatMut H_right) { bidiag_entry_cx<double>(A, H_left, H_right); }
void faer_b200_bidiag_in_place_c32(FaerV0_24_MatMut A, FaerV0_24_MatMut H_left, FaerV0_24_MatMut H_right) { bidiag_entry_cx<float>(A, H_left, H_right); }
void faer_b200_tridiag_in_place_c64(FaerV0_24_MatMut A, FaerV0_24_MatMut householder) { tridiag_entry_cx<double>(A, householder); }
void faer_b200_tridiag_in_place_c32(FaerV0_24_MatMut A, FaerV0_24_MatMut householder) { tridiag_entry_cx<float>(A, householder); }
void faer_b200_tridiag_in_place_f64(FaerV0_24_MatMut A, FaerV0_24_MatMut householder) { tridiag_entry<double>(A, householder); }
void faer_b200_tridiag_in_place_f32(FaerV0_24_MatMut A, FaerV0_24_MatMut householder) { tridiag_entry<float>(A, householder); }

// ---- default params and scratch queries of svd / self_adjoint_evd, the LDLT family and the reconstructs / inverses, every dtype
// (here rather than in ffi.cu so that the host build exports them too). The scratch is the reference's formula with the element
// size ES of T; the GPU path keeps its workspace in the device pool but reports what faer needs, so callers allocate identically.
#define FB_SVD_EVD_QUERIES(SUF, ES)                                                                                             \
  FaerV0_24_BidiagParams libfaer_v0_23_BidiagParams_##SUF(void) { return FaerV0_24_BidiagParams{192 * 256}; }                  \
  FaerV0_24_SvdParams libfaer_v0_23_SvdParams_##SUF(void) {                                                                    \
    /* svd/mod.rs:49-58: recursion_threshold 128, qr_ratio_threshold 11/6 */                                                  \
    return FaerV0_24_SvdParams{FaerV0_24_BidiagParams{192 * 256}, FaerV0_24_QrParams{48 * 48, 192 * 256}, 128, 11.0 / 6.0};    \
  }                                                                                                                            \
  FaerV0_24_Layout libfaer_v0_23_svd_scratch_##SUF(size_t nrows, size_t ncols, FaerV0_24_ComputeSvdVectors compute_U,          \
                                                   FaerV0_24_ComputeSvdVectors compute_V, FaerV0_24_Par par,                   \
                                                   FaerV0_24_SvdParams params) {                                               \
    (void)compute_U; (void)compute_V; (void)par; (void)params;                                                                 \
    return FaerV0_24_Layout{nrows * ncols * (ES), 64}; /* the copy of A */                                                     \
  }                                                                                                                            \
  FaerV0_24_TridiagParams libfaer_v0_23_TridiagParams_##SUF(void) { return FaerV0_24_TridiagParams{192 * 256}; }               \
  FaerV0_24_SelfAdjointEvdParams libfaer_v0_23_SelfAdjointEvdParams_##SUF(void) {                                              \
    return FaerV0_24_SelfAdjointEvdParams{FaerV0_24_TridiagParams{192 * 256}, 128}; /* evd/mod.rs:82-90 */                     \
  }                                                                                                                            \
  FaerV0_24_Layout libfaer_v0_23_self_adjoint_evd_scratch_##SUF(size_t dim, FaerV0_24_ComputeEigenvectors compute_U,           \
                                                                FaerV0_24_Par par, FaerV0_24_SelfAdjointEvdParams params) {    \
    (void)compute_U; (void)par; (void)params;                                                                                  \
    return FaerV0_24_Layout{dim * dim * (ES), 64}; /* the copy of A */                                                         \
  }                                                                                                                            \
  FaerV0_24_HessenbergParams libfaer_v0_23_HessenbergParams_##SUF(void) { return FaerV0_24_HessenbergParams{192 * 256, 256 * 256}; }
#define FB_LDLT_QUERIES(SUF, ES)                                                                                                \
  FaerV0_24_LdltParams libfaer_v0_23_LdltParams_##SUF(void) { return FaerV0_24_LdltParams{64, 128}; /* ldlt/factor.rs:705-714 */ } \
  FaerV0_24_Layout libfaer_v0_23_ldlt_factor_in_place_scratch_##SUF(size_t dim, FaerV0_24_Par par, FaerV0_24_LdltParams params) { \
    (void)par; (void)params;                                                                                                    \
    return FaerV0_24_Layout{dim * (ES), 64}; /* temp_mat_scratch::<T>(dim, 1), ldlt/factor.rs:715-724 */                        \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_ldlt_solve_in_place_scratch_##SUF(size_t dim, size_t rhs_ncols, FaerV0_24_Par par) {           \
    (void)dim; (void)rhs_ncols; (void)par;                                                                                      \
    return FaerV0_24_Layout{0, 1}; /* StackReq::EMPTY (ldlt/solve.rs:3-10) */                                                   \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_ldlt_reconstruct_scratch_##SUF(size_t dim, FaerV0_24_Par par) {                                \
    (void)par;                                                                                                                  \
    return FaerV0_24_Layout{dim * dim * (ES), 64}; /* temp_mat_scratch(dim, dim), ldlt/reconstruct.rs:4-7 */                    \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_ldlt_inverse_scratch_##SUF(size_t dim, FaerV0_24_Par par) {                                    \
    (void)par;                                                                                                                  \
    return FaerV0_24_Layout{dim * dim * (ES), 64}; /* temp_mat_scratch(dim, dim), ldlt/inverse.rs:4-7 */                        \
  }
#define FB_RECON_QUERIES(SUF, ES)                                                                                               \
  FaerV0_24_Layout libfaer_v0_23_llt_reconstruct_scratch_##SUF(size_t dim, FaerV0_24_Par par) {                                 \
    (void)dim; (void)par;                                                                                                       \
    return FaerV0_24_Layout{0, 1}; /* StackReq::EMPTY (llt/reconstruct.rs:3-6) */                                               \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_llt_inverse_scratch_##SUF(size_t dim, FaerV0_24_Par par) {                                     \
    (void)par;                                                                                                                  \
    return FaerV0_24_Layout{dim * dim * (ES), 64}; /* temp_mat_scratch(dim, dim) (llt/inverse.rs:3-8) */                        \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_partial_piv_lu_reconstruct_scratch_u32_##SUF(size_t nrows, size_t ncols, FaerV0_24_Par par) {  \
    (void)par;                                                                                                                  \
    return FaerV0_24_Layout{nrows * ncols * (ES), 64};                                                                          \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_partial_piv_lu_reconstruct_scratch_u64_##SUF(size_t nrows, size_t ncols, FaerV0_24_Par par) {  \
    (void)par;                                                                                                                  \
    return FaerV0_24_Layout{nrows * ncols * (ES), 64};                                                                          \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_partial_piv_lu_inverse_scratch_u32_##SUF(size_t dim, FaerV0_24_Par par) {                      \
    (void)par;                                                                                                                  \
    return FaerV0_24_Layout{dim * dim * (ES), 64};                                                                              \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_partial_piv_lu_inverse_scratch_u64_##SUF(size_t dim, FaerV0_24_Par par) {                      \
    (void)par;                                                                                                                  \
    return FaerV0_24_Layout{dim * dim * (ES), 64};                                                                              \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_qr_reconstruct_scratch_##SUF(size_t nrows, size_t ncols, size_t block_size, FaerV0_24_Par par) { \
    (void)nrows; (void)par;                                                                                                     \
    return FaerV0_24_Layout{block_size * ncols * (ES), 64};                                                                     \
  }                                                                                                                             \
  FaerV0_24_Layout libfaer_v0_23_qr_inverse_scratch_##SUF(size_t dim, size_t block_size, FaerV0_24_Par par) {                   \
    (void)par;                                                                                                                  \
    return FaerV0_24_Layout{block_size * dim * (ES), 64};                                                                       \
  }
#define FB_QUERIES(SUF, ES) FB_SVD_EVD_QUERIES(SUF, ES) FB_LDLT_QUERIES(SUF, ES) FB_RECON_QUERIES(SUF, ES)
FB_QUERIES(f64, sizeof(double))
FB_QUERIES(f32, sizeof(float))
FB_QUERIES(c64, 2 * sizeof(double))
FB_QUERIES(c32, 2 * sizeof(float))
#undef FB_QUERIES
#undef FB_SVD_EVD_QUERIES
#undef FB_LDLT_QUERIES
#undef FB_RECON_QUERIES

// ---- complex `svd` / `self_adjoint_evd` (cplx_condensed.cu: c32 computes in c64) ----
#define FB_SVD_EVD_CPLX_FFI(SUF, R)                                                                                             \
  FaerV0_24_SvdStatus libfaer_v0_23_svd_##SUF(FaerV0_24_MatRef A, FaerV0_24_MatMut U, FaerV0_24_VecMut S, FaerV0_24_MatMut V,  \
                                              FaerV0_24_Par par, FaerV0_24_MemAlloc mem, FaerV0_24_SvdParams params) {         \
    (void)par; (void)mem; (void)params;                                                                                        \
    return svd_entry_cx<R>(A, U, S, V);                                                                                      \
  }                                                                                                                            \
  FaerV0_24_EvdStatus libfaer_v0_23_self_adjoint_evd_##SUF(FaerV0_24_MatRef A, FaerV0_24_MatMut U, FaerV0_24_VecMut S,         \
                                                           FaerV0_24_Par par, FaerV0_24_MemAlloc mem,                          \
                                                           FaerV0_24_SelfAdjointEvdParams params) {                            \
    (void)par; (void)mem; (void)params;                                                                                        \
    return self_adjoint_evd_entry_cx<R>(A, U, S);                                                                            \
  }
FB_SVD_EVD_CPLX_FFI(c64, double)
FB_SVD_EVD_CPLX_FFI(c32, float)
#undef FB_SVD_EVD_CPLX_FFI

// ---- reconstruct / inverse for f32 / c64 / c32 (f64: ffi.cu; qr_reconstruct for f32 too) ----
#define FB_RECON_TYPES_FFI(SUF, R, CX)                                                                                          \
  void libfaer_v0_23_llt_reconstruct_##SUF(FaerV0_24_MatMut A, FaerV0_24_MatRef L, FaerV0_24_Par par, FaerV0_24_MemAlloc mem) { \
    (void)par; (void)mem;                                                                                                       \
    llt_recon_entry_t<R, CX>(A, L, false);                                                                                      \
  }                                                                                                                             \
  void libfaer_v0_23_llt_inverse_##SUF(FaerV0_24_MatMut A_inv, FaerV0_24_MatRef L, FaerV0_24_Par par, FaerV0_24_MemAlloc mem) { \
    (void)par; (void)mem;                                                                                                       \
    llt_recon_entry_t<R, CX>(A_inv, L, true);                                                                                   \
  }                                                                                                                             \
  void libfaer_v0_23_qr_inverse_##SUF(FaerV0_24_MatMut A, FaerV0_24_MatRef Q_basis, FaerV0_24_MatRef Q_coeff, FaerV0_24_MatRef R_, \
                                      FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {                                              \
    (void)par; (void)mem;                                                                                                       \
    qr_recon_entry_t<R, CX>(A, Q_basis, Q_coeff, R_, true);                                                                     \
  }                                                                                                                             \
  FB_LU_RECON_TYPES_FFI(u32, 4, SUF, R, CX)                                                                                     \
  FB_LU_RECON_TYPES_FFI(u64, 8, SUF, R, CX)
#define FB_LU_RECON_TYPES_FFI(IT, BYTES, SUF, R, CX)                                                                            \
  void libfaer_v0_23_partial_piv_lu_reconstruct_##IT##_##SUF(FaerV0_24_MatMut A, FaerV0_24_MatRef L, FaerV0_24_MatRef U,        \
                                                             FaerV0_24_SliceRef perm_fwd, FaerV0_24_SliceRef perm_bwd,          \
                                                             FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {                       \
    (void)perm_fwd; (void)par; (void)mem;                                                                                       \
    lu_recon_entry_t<R, CX>(A, L, U, perm_bwd, BYTES, false);                                                                   \
  }                                                                                                                             \
  void libfaer_v0_23_partial_piv_lu_inverse_##IT##_##SUF(FaerV0_24_MatMut A, FaerV0_24_MatRef L, FaerV0_24_MatRef U,            \
                                                         FaerV0_24_SliceRef perm_fwd, FaerV0_24_SliceRef perm_bwd,              \
                                                         FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {                           \
    (void)perm_bwd; (void)par; (void)mem;                                                                                       \
    lu_recon_entry_t<R, CX>(A, L, U, perm_fwd, BYTES, true);                                                                    \
  }
#define FB_QR_RECON_TYPES_FFI(SUF, R)                                                                                           \
  void libfaer_v0_23_qr_reconstruct_##SUF(FaerV0_24_MatMut A, FaerV0_24_MatRef Q_basis, FaerV0_24_MatRef Q_coeff,               \
                                          FaerV0_24_MatRef R_, FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {                     \
    (void)par; (void)mem;                                                                                                       \
    qr_recon_entry_t<R, true>(A, Q_basis, Q_coeff, R_, false);                                                                  \
  }
FB_RECON_TYPES_FFI(f32, float, false)
FB_RECON_TYPES_FFI(c64, double, true)
FB_RECON_TYPES_FFI(c32, float, true)
FB_QR_RECON_TYPES_FFI(c64, double)
FB_QR_RECON_TYPES_FFI(c32, float)
#undef FB_RECON_TYPES_FFI
#undef FB_QR_RECON_TYPES_FFI
#undef FB_LU_RECON_TYPES_FFI

// ---- LDLT: factor / solve for f32 / c64 / c32, reconstruct / inverse for every dtype (ldlt_types.cu) ----
#define FB_LDLT_FS_FFI(SUF, R, CX)                                                                                              \
  FaerV0_24_LdltStatus libfaer_v0_23_ldlt_factor_in_place_##SUF(FaerV0_24_MatMut A, FaerV0_24_LdltRegularization regularization, \
                                                                FaerV0_24_Par par, FaerV0_24_MemAlloc mem,                      \
                                                                FaerV0_24_LdltParams params) {                                  \
    (void)par; (void)mem; (void)params;                                                                                         \
    return ldlt_factor_entry_t<R, CX>(A, regularization);                                                                       \
  }                                                                                                                             \
  void libfaer_v0_23_ldlt_solve_in_place_##SUF(FaerV0_24_MatRef L, FaerV0_24_VecRef D, FaerV0_24_Conj A_conj,                   \
                                               FaerV0_24_MatMut rhs, FaerV0_24_Par par, FaerV0_24_MemAlloc mem) {               \
    (void)par; (void)mem;                                                                                                       \
    ldlt_solve_entry_t<R, CX>(L, D, A_conj, rhs);                                                                               \
  }
#define FB_LDLT_RI_FFI(SUF, R, CX)                                                                                              \
  void libfaer_v0_23_ldlt_reconstruct_##SUF(FaerV0_24_MatMut A, FaerV0_24_MatRef L, FaerV0_24_VecRef D, FaerV0_24_Par par,      \
                                            FaerV0_24_MemAlloc mem) {                                                           \
    (void)par; (void)mem;                                                                                                       \
    ldlt_recon_entry_t<R, CX>(A, L, D, false);                                                                                  \
  }                                                                                                                             \
  void libfaer_v0_23_ldlt_inverse_##SUF(FaerV0_24_MatMut A_inv, FaerV0_24_MatRef L, FaerV0_24_VecRef D, FaerV0_24_Par par,      \
                                        FaerV0_24_MemAlloc mem) {                                                               \
    (void)par; (void)mem;                                                                                                       \
    ldlt_recon_entry_t<R, CX>(A_inv, L, D, true);                                                                               \
  }
FB_LDLT_FS_FFI(f32, float, false)
FB_LDLT_FS_FFI(c64, double, true)
FB_LDLT_FS_FFI(c32, float, true)
FB_LDLT_RI_FFI(f64, double, false)
FB_LDLT_RI_FFI(f32, float, false)
FB_LDLT_RI_FFI(c64, double, true)
FB_LDLT_RI_FFI(c32, float, true)
#undef FB_LDLT_FS_FFI
#undef FB_LDLT_RI_FFI

// ---- triangular inverses, every dtype ----
#define FB_TRI_INV_FFI(SUF, R, CX)                                                                                              \
  void libfaer_v0_23_inverse_triangular_lower_in_place_##SUF(FaerV0_24_MatMut L_inv, FaerV0_24_MatRef L, FaerV0_24_Par par) {    \
    (void)par;                                                                                                                  \
    inverse_triangular_entry_t<R, CX>(L_inv, L, true, false);                                                                   \
  }                                                                                                                             \
  void libfaer_v0_23_inverse_triangular_upper_in_place_##SUF(FaerV0_24_MatMut L_inv, FaerV0_24_MatRef L, FaerV0_24_Par par) {    \
    (void)par;                                                                                                                  \
    inverse_triangular_entry_t<R, CX>(L_inv, L, false, false);                                                                  \
  }                                                                                                                             \
  void libfaer_v0_23_inverse_unit_triangular_lower_in_place_##SUF(FaerV0_24_MatMut L_inv, FaerV0_24_MatRef L, FaerV0_24_Par par) { \
    (void)par;                                                                                                                  \
    inverse_triangular_entry_t<R, CX>(L_inv, L, true, true);                                                                    \
  }                                                                                                                             \
  void libfaer_v0_23_inverse_unit_triangular_upper_in_place_##SUF(FaerV0_24_MatMut L_inv, FaerV0_24_MatRef L, FaerV0_24_Par par) { \
    (void)par;                                                                                                                  \
    inverse_triangular_entry_t<R, CX>(L_inv, L, false, true);                                                                   \
  }
FB_TRI_INV_FFI(f64, double, false)
FB_TRI_INV_FFI(f32, float, false)
FB_TRI_INV_FFI(c64, double, true)
FB_TRI_INV_FFI(c32, float, true)
#undef FB_TRI_INV_FFI

void faer_b200_hessenberg_in_place_f64(FaerV0_24_MatMut A, FaerV0_24_MatMut householder) { hessenberg_entry_t<double, false>(A, householder); }
void faer_b200_hessenberg_in_place_f32(FaerV0_24_MatMut A, FaerV0_24_MatMut householder) { hessenberg_entry_t<float, false>(A, householder); }
void faer_b200_hessenberg_in_place_c64(FaerV0_24_MatMut A, FaerV0_24_MatMut householder) { hessenberg_entry_t<double, true>(A, householder); }
void faer_b200_hessenberg_in_place_c32(FaerV0_24_MatMut A, FaerV0_24_MatMut householder) { hessenberg_entry_t<float, true>(A, householder); }

}  // extern "C"
