// Solves on top of the factors (SURVEY.md §8f rank 1): compositions of the kernels already on the hot path, for f64 and f32
// (the triangular solves of tensor_ops.cuh); the row permutation also serves the complex LU solves (cplx.cu).
//
// Reference:
//   cholesky::llt::solve::solve_in_place_with_conj          faer/src/linalg/cholesky/llt/solve.rs:12-35
//       L y = b (lower solve), then L^H x = y (upper solve on the transposed view)
//   lu::partial_pivoting::solve::solve_in_place_with_conj   faer/src/linalg/lu/partial_pivoting/solve.rs:21-54
//       rhs <- P rhs (permute_rows_in_place: dst[i, :] = src[perm_fwd[i], :], perm/mod.rs:256-294),
//       unit-lower solve with L, upper solve with U
//   lu::partial_pivoting::solve::solve_transpose_in_place_with_conj   lu/partial_pivoting/solve.rs:55-86
//       lower solve with U^T, unit-upper solve with L^T, then rhs <- P^-1 rhs (permute_rows_in_place with the inverse
//       permutation, whose forward array is perm_bwd)
#include "runtime.cuh"
#include "tensor_ops.cuh"

namespace fb {

namespace {

// dst (compact column-major, ld = nrows) [i, c] = src[perm[i], c]
template <class E>
__global__ void gather_rows_kernel(E* __restrict__ dst, const E* __restrict__ src, i64 rs, i64 cs, i64 nrows, i64 ncols,
                                   const long long* __restrict__ perm) {
  const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  const i64 c = blockIdx.y;
  if (i < nrows && c < ncols) dst[c * nrows + i] = src[perm[i] * rs + c * cs];
}
template <class E>
__global__ void scatter_back_kernel(E* __restrict__ dst, i64 rs, i64 cs, const E* __restrict__ src, i64 nrows, i64 ncols) {
  const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  const i64 c = blockIdx.y;
  if (i < nrows && c < ncols) dst[i * rs + c * cs] = src[c * nrows + i];
}

}  // namespace

template <class E>
void permute_rows_in_place(cudaStream_t stream, View<E> rhs, const long long* perm_fwd) {
  const i64 n = rhs.nrows, k = rhs.ncols;
  if (n == 0 || k == 0) return;
  FB_ASSERT(k < 65536, "too many right-hand sides for one permutation launch");
  long long* d_perm = (long long*)ws_alloc((size_t)n * 8);
  E* tmp = (E*)ws_alloc((size_t)n * k * sizeof(E));
  FB_CUDA_CHECK(cudaMemcpyAsync(d_perm, perm_fwd, (size_t)n * 8, cudaMemcpyHostToDevice, stream));
  dim3 grid((unsigned)((n + 255) / 256), (unsigned)k);
  gather_rows_kernel<E><<<grid, 256, 0, stream>>>(tmp, rhs.ptr, rhs.rs, rhs.cs, n, k, d_perm);
  FB_CUDA_CHECK(cudaGetLastError());
  note_launch();
  scatter_back_kernel<E><<<grid, 256, 0, stream>>>(rhs.ptr, rhs.rs, rhs.cs, tmp, n, k);
  FB_CUDA_CHECK(cudaGetLastError());
  note_launch();
  FB_CUDA_CHECK(cudaStreamSynchronize(stream));  // perm_fwd (host, pageable) and the pool buffers are released below
  ws_free(tmp);
  ws_free(d_perm);
}
template void permute_rows_in_place<double>(cudaStream_t, View<double>, const long long*);
template void permute_rows_in_place<float>(cudaStream_t, View<float>, const long long*);
template void permute_rows_in_place<ReIm<double>>(cudaStream_t, View<ReIm<double>>, const long long*);
template void permute_rows_in_place<ReIm<float>>(cudaStream_t, View<ReIm<float>>, const long long*);

template <class T>
void llt_solve_in_place(cudaStream_t stream, View<const T> L, View<T> rhs) {
  FB_ASSERT(L.nrows == L.ncols && rhs.nrows == L.nrows, "LLT solve shape mismatch");
  solve_lower(stream, L, false, rhs);
  solve_upper(stream, L.t(), false, rhs);
}

template <class T>
void lu_solve_in_place(cudaStream_t stream, View<const T> L, View<const T> U, const long long* perm_fwd, View<T> rhs) {
  const i64 n = L.nrows;
  FB_ASSERT(L.ncols == n && U.nrows == n && U.ncols == n && rhs.nrows == n, "LU solve shape mismatch");
  permute_rows_in_place(stream, rhs, perm_fwd);
  solve_lower(stream, L, true, rhs);
  solve_upper(stream, U, false, rhs);
}

template <class T>
void lu_solve_transpose_in_place(cudaStream_t stream, View<const T> L, View<const T> U, const long long* perm_bwd, View<T> rhs) {
  const i64 n = L.nrows;
  FB_ASSERT(L.ncols == n && U.nrows == n && U.ncols == n && rhs.nrows == n, "LU solve shape mismatch");
  solve_lower(stream, U.t(), false, rhs);
  solve_upper(stream, L.t(), true, rhs);
  permute_rows_in_place(stream, rhs, perm_bwd);
}

#define FB_SOLVES(T)                                                                                                   \
  template void llt_solve_in_place<T>(cudaStream_t, View<const T>, View<T>);                                           \
  template void lu_solve_in_place<T>(cudaStream_t, View<const T>, View<const T>, const long long*, View<T>);            \
  template void lu_solve_transpose_in_place<T>(cudaStream_t, View<const T>, View<const T>, const long long*, View<T>);
FB_SOLVES(double)
FB_SOLVES(float)
#undef FB_SOLVES

}  // namespace fb
