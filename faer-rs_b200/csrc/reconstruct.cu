// `*_reconstruct` / `*_inverse` on the factors (SURVEY.md appendix C, "next" row), f64: compositions of the structured GEMM,
// the triangular solves, the row permutation and the block-Householder sequence that are already on the hot path.
// Reference:
//   cholesky/llt/reconstruct.rs:12-33   out(lower) = L(lower) * L^H(upper)            (only the lower triangle is written)
//   cholesky/llt/inverse.rs:10-39       L_inv = L^-1 (lower), out(lower) = L_inv^H(upper) * L_inv(lower)
//   lu/partial_pivoting/reconstruct.rs:12-80   tmp = L U by structured products (square / tall / wide parts), out = P^-1 tmp
//   lu/partial_pivoting/inverse.rs      A^-1 from the factors; here as the solve applied to the identity (same result up to
//                                       rounding; the reference inverts the triangular factors and multiplies)
//   qr/no_pivoting/reconstruct.rs:13-39 out = [R; 0], then out <- Q out
//   qr/no_pivoting/inverse.rs           A^-1 = R^-1 Q^H; here as the QR solve applied to the identity
// Tests: tests/test_gpu_zz4_reconstruct_inverse.py.
#include "runtime.cuh"
#include "tensor_ops.cuh"

namespace fb {

namespace {

__global__ void set_identity_kernel(double* __restrict__ A, i64 rs, i64 cs, i64 n) {
  const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  const i64 j = blockIdx.y;
  if (i < n && j < n) A[i * rs + j * cs] = i == j ? 1.0 : 0.0;
}
// out (m x n) <- upper trapezoid of R (size x n) in its first `size` rows, zero elsewhere
template <class T>
__global__ void set_upper_trapezoid_kernel(T* __restrict__ out, i64 o_rs, i64 o_cs, i64 m, i64 n, const T* __restrict__ R,
                                           i64 r_rs, i64 r_cs, i64 size) {
  const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  const i64 j = blockIdx.y;
  if (i < m && j < n) out[i * o_rs + j * o_cs] = (i < size && i <= j) ? R[i * r_rs + j * r_cs] : T(0);
}

void set_identity(cudaStream_t st, VD A) {
  const i64 n = A.nrows;
  if (n == 0) return;
  FB_ASSERT(n < 65536, "matrix too wide for one fill launch");
  dim3 grid((unsigned)((n + 255) / 256), (unsigned)n);
  set_identity_kernel<<<grid, 256, 0, st>>>(A.ptr, A.rs, A.cs, n);
  FB_CUDA_CHECK(cudaGetLastError());
  note_launch();
}

}  // namespace

void llt_reconstruct_f64(cudaStream_t st, VD out, VCD L) {
  const i64 n = out.nrows;
  FB_ASSERT(out.ncols == n && L.nrows == n && L.ncols == n, "llt_reconstruct shape mismatch");
  if (n == 0) return;
  gemm_f64(st, out, TRI_LOWER, 0, L, TRI_LOWER, L.t(), TRI_UPPER, 1.0);
}

void llt_inverse_f64(cudaStream_t st, VD out, VCD L) {
  const i64 n = out.nrows;
  FB_ASSERT(out.ncols == n && L.nrows == n && L.ncols == n, "llt_inverse shape mismatch");
  if (n == 0) return;
  double* buf = (double*)ws_alloc((size_t)n * (size_t)n * sizeof(double));
  VD Li{buf, n, n, 1, n};
  set_identity(st, Li);
  solve_lower_triangular_in_place_f64(st, L, false, Li);  // L_inv: lower triangular, exact zeros above the diagonal
  gemm_f64(st, out, TRI_LOWER, 0, cv(Li).t(), TRI_UPPER, cv(Li), TRI_LOWER, 1.0);
  FB_CUDA_CHECK(cudaStreamSynchronize(st));
  ws_free(buf);
}

// perm_bwd: HOST int64[m], the inverse row permutation
void lu_reconstruct_f64(cudaStream_t st, VD out, VCD L, VCD U, const long long* perm_bwd) {
  const i64 m = L.nrows, n = U.ncols, size = std::min(m, n);
  FB_ASSERT(out.nrows == m && out.ncols == n && L.ncols >= size && U.nrows >= size, "lu_reconstruct shape mismatch");
  if (m == 0 || n == 0) return;
  gemm_f64(st, out.sub(0, 0, size, size), RECT, 0, L.sub(0, 0, size, size), UNIT_LOWER, U.sub(0, 0, size, size), TRI_UPPER, 1.0);
  if (m > n)
    gemm_f64(st, out.sub(size, 0, m - size, size), RECT, 0, L.sub(size, 0, m - size, size), RECT, U.sub(0, 0, size, size),
             TRI_UPPER, 1.0);
  if (m < n)
    gemm_f64(st, out.sub(0, size, size, n - size), RECT, 0, L.sub(0, 0, size, size), UNIT_LOWER, U.sub(0, size, size, n - size),
             RECT, 1.0);
  // (P A)[i, :] = A[perm_fwd[i], :]  =>  A[j, :] = (L U)[perm_bwd[j], :]
  permute_rows_in_place(st, out, perm_bwd);
}

void lu_inverse_f64(cudaStream_t st, VD out, VCD L, VCD U, const long long* perm_fwd) {
  const i64 n = out.nrows;
  FB_ASSERT(out.ncols == n && L.nrows == n && L.ncols == n && U.nrows == n && U.ncols == n, "lu_inverse shape mismatch");
  if (n == 0) return;
  set_identity(st, out);
  lu_solve_in_place(st, L, U, perm_fwd, out);
}

template <class T>
void qr_reconstruct(cudaStream_t st, View<T> out, View<const T> Qb, View<const T> Qc, View<const T> R) {
  const i64 m = Qb.nrows, n = R.ncols, size = std::min(m, n);
  FB_ASSERT(out.nrows == m && out.ncols == n && Qb.ncols == size && Qc.ncols == size && R.nrows == size,
            "qr_reconstruct shape mismatch");
  if (m == 0 || n == 0) return;
  FB_ASSERT(n < 65536, "matrix too wide for one fill launch");
  dim3 grid((unsigned)((m + 255) / 256), (unsigned)n);
  set_upper_trapezoid_kernel<T><<<grid, 256, 0, st>>>(out.ptr, out.rs, out.cs, m, n, R.ptr, R.rs, R.cs, size);
  FB_CUDA_CHECK(cudaGetLastError());
  note_launch();
  if (size > 0) apply_block_householder_sequence_on_the_left<T>(st, Qb, Qc, out);
}
template void qr_reconstruct<double>(cudaStream_t, View<double>, View<const double>, View<const double>, View<const double>);
template void qr_reconstruct<float>(cudaStream_t, View<float>, View<const float>, View<const float>, View<const float>);

void qr_inverse_f64(cudaStream_t st, VD out, VCD Qb, VCD Qc, VCD R) {
  const i64 n = out.nrows;
  FB_ASSERT(out.ncols == n && Qb.nrows == n && Qb.ncols == n && Qc.ncols == n && R.nrows == n && R.ncols == n,
            "qr_inverse shape mismatch");
  if (n == 0) return;
  set_identity(st, out);
  apply_block_householder_sequence_transpose_on_the_left<double>(st, Qb, Qc, out);
  solve_upper_triangular_in_place_f64(st, R, false, out);
}

}  // namespace fb
