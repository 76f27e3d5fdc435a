// f32 GEMM / structured GEMM (3xTF32 on the tensor pipe), see gemm_f32.cu.
#pragma once
#include "common.cuh"

namespace fb {

typedef View<float> VF;
typedef View<const float> VCF;
inline VCF cv(const VF& v) { return VCF{v.ptr, v.nrows, v.ncols, v.rs, v.cs}; }

struct GemmF32Params {
  int m, n, k;
  const float* A; i64 a_rs, a_cs; int a_struct;
  const float* B; i64 b_rs, b_cs; int b_struct;
  float* C;       i64 c_rs, c_cs; int c_struct;
  float alpha;
  int accum;
  int tiles_m, tiles_n;
  int k_split_len;       // split-K (see gemm_f64.cuh): 0 = off
  i64 c_split_stride;
};

// dst(struct) = [dst +] alpha * lhs(struct) * rhs(struct); device views, element strides of any sign.
void gemm_f32(cudaStream_t stream, VF dst, int dst_struct, int accum, VCF lhs, int lhs_struct, VCF rhs, int rhs_struct,
              float alpha);
inline void gemm_f32(cudaStream_t stream, VF dst, int accum, VCF lhs, VCF rhs, float alpha) {
  gemm_f32(stream, dst, RECT, accum, lhs, RECT, rhs, RECT, alpha);
}

// c32 (interleaved complex<f32>) product, 4M formulation on the f32 kernels (gemm_c32.cu); views in complex units
void gemm_c32(cudaStream_t stream, VF dst, int dst_struct, int accum, VCF lhs, int lhs_struct, bool conj_lhs, VCF rhs,
              int rhs_struct, bool conj_rhs, float alpha_re, float alpha_im);

// f32 triangular solves (trsm.cu; same algorithm as the f64 ones)
void solve_lower_triangular_in_place_f32(cudaStream_t stream, VCF tril, bool unit, VF rhs);
void solve_upper_triangular_in_place_f32(cudaStream_t stream, VCF triu, bool unit, VF rhs);

// f32 LLT (llt.cu, instantiated for float): same contract as llt_cholesky_in_place_f64 (linalg_f64.cuh)
struct LltResult;
struct LltParams;
LltResult llt_cholesky_in_place_f32(cudaStream_t stream, VF A, float reg_delta, float reg_eps, LltParams params);

// c32 triangular solves, LLT and partial-pivoting LU (cplx.cu, instantiated for float; same contracts as the _c64 functions in
// linalg_f64.cuh); views in COMPLEX element units
void solve_lower_triangular_in_place_c32(cudaStream_t st, VCF tril, bool unit, bool conj, VF rhs);
void solve_upper_triangular_in_place_c32(cudaStream_t st, VCF triu, bool unit, bool conj, VF rhs);
LltResult llt_cholesky_in_place_c32(cudaStream_t st, VF A, float reg_delta, float reg_eps);
void llt_solve_in_place_c32(cudaStream_t st, VCF L, bool conj, VF rhs);
size_t lu_partial_piv_in_place_c32(cudaStream_t st, VF A, long long* perm_fwd, long long* perm_inv);
void lu_solve_in_place_c32(cudaStream_t st, VCF L, VCF U, bool conj, const long long* perm_fwd, VF rhs);
void lu_solve_transpose_in_place_c32(cudaStream_t st, VCF L, VCF U, bool conj, const long long* perm_bwd, VF rhs);
i64 qr_in_place_c32(cudaStream_t st, VF A, VF Q_coeff, i64 blocking_threshold);
void apply_householder_sequence_left_c32(cudaStream_t st, VCF basis, VCF factor, bool conj, VF rhs, bool transpose);

}  // namespace fb
