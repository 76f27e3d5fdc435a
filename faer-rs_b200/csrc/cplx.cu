// c64 / c32 (complex<f64> / complex<f32>) triangular solves, Cholesky LLT, partial-pivoting LU and Householder QR (+ block-Householder
// sequences): faer's recursions on the complex GEMMs (gemm_c64.cu, gemm_c32.cu) with small scalar complex leaf kernels, one source
// templated over the real type R. (The comment blocks at the LU and QR sections cite their reference lines.)
//
// Reference:
//   triangular_solve::solve_[unit_]{lower,upper}_triangular_in_place_with_conj   faer/src/linalg/triangular_solve.rs:220-604
//       recursive split (block_size 200-211): top solve, rhs_bot -= conj?(T10) * rhs_top, bottom solve; leaves multiply by the
//       reciprocal of the diagonal (16-198); upper = lower on reversed views (577-604)
//   cholesky::llt::factor::cholesky_in_place for complex T   cholesky/llt/factor.rs:68-97 -> ldlt/factor.rs:367-498
//       A00 = L00 L00^H (recursion / leaf), conj(L00) X = A10^T, A11(lower) -= A10 A10^H; leaf recurrence
//       a_ij <- a_ij - conj(a_jk) a_ik, d = Re(a_jj), [regularise], fail if !(d > 0), l = sqrt(d), column j (diagonal included)
//       multiplied by recip(l)  (ldlt/factor.rs:7-177, 299-366)
//
// All views are in COMPLEX element units (pointer to the first complex element as R*, strides in complex elements), as in
// gemm_c64.cu / gemm_c32.cu. The leaves are plain scalar kernels (a 32 x 32 block per CTA / one thread per right-hand-side column): O(n^2 leaf)
// work next to the O(n^3) that runs on the DMMA GEMM.
#include <algorithm>
#include <vector>

#include "gemm_f32.cuh"
#include "linalg_f64.cuh"
#include "runtime.cuh"

namespace fb {

namespace {

constexpr int CL = 32;  // leaf order of both recursions

template <class R>
struct CxT {
  R re, im;
};
template <class R>
__device__ __forceinline__ CxT<R> cmul(CxT<R> a, CxT<R> b) {
  return CxT<R>{fma(a.re, b.re, -a.im * b.im), fma(a.re, b.im, a.im * b.re)};
}
template <class R>
__device__ __forceinline__ CxT<R> cld(const R* p, i64 off) {
  return CxT<R>{p[2 * off], p[2 * off + 1]};
}
template <class R>
__device__ __forceinline__ void cst(R* p, i64 off, CxT<R> v) {
  p[2 * off] = v.re;
  p[2 * off + 1] = v.im;
}
// 1 / d without spurious overflow; an infinite d (the +inf diagonal of a skipped reflector, qr factor.rs:287-299) gives 0
template <class R>
__device__ __forceinline__ CxT<R> crecip(CxT<R> d) {
  if (isinf(d.re) || isinf(d.im)) return CxT<R>{R(0), R(0)};
  const R mx = fmax(fabs(d.re), fabs(d.im));
  if (mx == R(0)) {
    const R s = R(1) / fma(d.re, d.re, d.im * d.im);
    return CxT<R>{d.re * s, -d.im * s};
  }
  const R sc = R(1) / mx;
  const R a = d.re * sc, b = d.im * sc;
  const R s = sc / fma(a, a, b * b);
  return CxT<R>{a * s, -b * s};
}

// complex products of the recursions, by scalar type
inline void cgemm(cudaStream_t st, VD dst, int ds, int accum, VCD a, int as, bool ca, VCD b, int bs, bool cb, double ar, double ai) {
  gemm_c64(st, dst, ds, accum, a, as, ca, b, bs, cb, ar, ai);
}
inline void cgemm(cudaStream_t st, VF dst, int ds, int accum, VCF a, int as, bool ca, VCF b, int bs, bool cb, float ar, float ai) {
  gemm_c32(st, dst, ds, accum, a, as, ca, b, bs, cb, ar, ai);
}

// conj?(T) X = B for a lower-triangular leaf T (n <= CL): one thread per column of B, the column in registers
template <class R>
__global__ void __launch_bounds__(64) trsm_leaf_lower_cx_kernel(const R* __restrict__ T, i64 t_rs, i64 t_cs, int n, int unit,
                                                                  int conj, R* __restrict__ B, i64 b_rs, i64 b_cs, i64 ncols) {
  __shared__ R nlr[CL][CL + 1], nli[CL][CL + 1];  // -(conj? l_ik) * inv_i below the diagonal, inv_i on it
  for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
    const int i = e / n, k = e - i * n;
    if (k > i) continue;
    CxT<R> inv{R(1), R(0)};
    if (!unit) {
      inv = crecip(cld(T, (i64)i * t_rs + (i64)i * t_cs));  // 1 / d; 0 for the +inf diagonal of a skipped reflector
      if (conj) inv.im = -inv.im;           // conj(1 / d) = 1 / conj(d)
    }
    CxT<R> v = inv;
    if (k < i) {
      CxT<R> l = cld(T, (i64)i * t_rs + (i64)k * t_cs);
      if (conj) l.im = -l.im;
      v = cmul(CxT<R>{-l.re, -l.im}, inv);
    }
    nlr[i][k] = v.re;
    nli[i][k] = v.im;
  }
  __syncthreads();
  const i64 col = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= ncols) return;
  R yr[CL], yi[CL];
#pragma unroll
  for (int i = 0; i < CL; ++i) {
    if (i < n) {
      CxT<R> v = cld(B, (i64)i * b_rs + col * b_cs);
      v = cmul(v, CxT<R>{nlr[i][i], nli[i][i]});  // * inv_i (1 for a unit diagonal)
#pragma unroll
      for (int k = 0; k < CL; ++k) {
        if (k < i) {
          const CxT<R> t = cmul(CxT<R>{nlr[i][k], nli[i][k]}, CxT<R>{yr[k], yi[k]});
          v.re += t.re;
          v.im += t.im;
        }
      }
      yr[i] = v.re;
      yi[i] = v.im;
      cst(B, (i64)i * b_rs + col * b_cs, v);
    }
  }
}

// in-place lower Cholesky of a <= CL x CL Hermitian block (lower triangle read / written), one CTA, block in shared memory
template <class R>
__global__ void __launch_bounds__(CL * CL) potf2_cx_kernel(R* __restrict__ A, i64 rs, i64 cs, int n, i64 j0, int regularize,
                                                            R eps, R delta, long long* __restrict__ info) {
  __shared__ R Sr[CL][CL + 1], Si[CL][CL + 1];
  __shared__ R s_inv;
  __shared__ int s_fail, s_count;
  if (info[0] >= 0) return;  // an earlier block already failed
  const int i = threadIdx.x % CL, c = threadIdx.x / CL;
  const bool on = i < n && c <= i;
  if (on) {
    const CxT<R> v = cld(A, (i64)i * rs + (i64)c * cs);
    Sr[i][c] = v.re;
    Si[i][c] = v.im;
  }
  if (threadIdx.x == 0) s_count = 0;
  __syncthreads();
  for (int j = 0; j < n; ++j) {
    if (threadIdx.x == 0) {
      R d = Sr[j][j];
      int fail = 0;
      if (regularize && d <= eps) {
        d = delta;
        s_count += 1;
      }
      R inv = R(0);
      if (!(d > R(0))) fail = 1;
      else {
        const R sd = sqrt(d);
        if (sd == R(0) || !isfinite(sd)) fail = 1;
        else inv = R(1) / sd;
      }
      s_inv = inv;
      s_fail = fail;
    }
    __syncthreads();
    if (s_fail) {
      if (threadIdx.x == 0) info[0] = j0 + j;
      return;
    }
    const R inv = s_inv;
    // column j (diagonal included) * recip(l_jj)
    if (c == j && i >= j && i < n) {
      Sr[i][j] *= inv;
      Si[i][j] *= inv;
    }
    __syncthreads();
    // a_ic <- a_ic - conj(l_cj) l_ij for j < c <= i
    if (on && c > j) {
      const CxT<R> lc{Sr[c][j], -Si[c][j]}, li{Sr[i][j], Si[i][j]};
      const CxT<R> t = cmul(lc, li);
      Sr[i][c] -= t.re;
      Si[i][c] -= t.im;
    }
    __syncthreads();
  }
  if (on) cst(A, (i64)i * rs + (i64)c * cs, CxT<R>{Sr[i][c], Si[i][c]});
  if (threadIdx.x == 0 && s_count) info[1] += s_count;
}

template <class R>
inline View<R> csub(View<R> v, i64 i, i64 j, i64 m, i64 n) { return View<R>{v.ptr + 2 * (i * v.rs + j * v.cs), m, n, v.rs, v.cs}; }
template <class R>
inline View<const R> csub(View<const R> v, i64 i, i64 j, i64 m, i64 n) { return View<const R>{v.ptr + 2 * (i * v.rs + j * v.cs), m, n, v.rs, v.cs}; }

template <class R>
void solve_lower_rec_cx(cudaStream_t st, View<const R> T, bool unit, bool conj, View<R> rhs) {
  const i64 n = T.nrows, k = rhs.ncols;
  if (n == 0 || k == 0) return;
  if (n <= CL) {
    trsm_leaf_lower_cx_kernel<R><<<(unsigned)((k + 63) / 64), 64, 0, st>>>(T.ptr, T.rs, T.cs, (int)n, unit ? 1 : 0, conj ? 1 : 0, rhs.ptr,
                                                                         rhs.rs, rhs.cs, k);
    FB_CUDA_CHECK(cudaGetLastError());
    note_launch();
    return;
  }
  const i64 n1 = ((n / 2 + CL - 1) / CL) * CL;
  solve_lower_rec_cx(st, csub(T, 0, 0, n1, n1), unit, conj, csub(rhs, 0, 0, n1, k));
  // rhs_bot -= conj?(T10) * rhs_top
  cgemm(st, csub(rhs, n1, 0, n - n1, k), RECT, 1, csub(T, n1, 0, n - n1, n1), RECT, conj, cv(csub(rhs, 0, 0, n1, k)), RECT, false,
           R(-1), R(0));
  solve_lower_rec_cx(st, csub(T, n1, n1, n - n1, n - n1), unit, conj, csub(rhs, n1, 0, n - n1, k));
}

template <class R>
struct LltCtxC {
  cudaStream_t st;
  int regularize;
  R eps, delta;
  long long* d_info;
};

template <class R>
void llt_rec_cx(const LltCtxC<R>& ctx, View<R> A, i64 j0) {
  const i64 n = A.nrows;
  if (n <= CL) {
    potf2_cx_kernel<R><<<1, CL * CL, 0, ctx.st>>>(A.ptr, A.rs, A.cs, (int)n, j0, ctx.regularize, ctx.eps, ctx.delta, ctx.d_info);
    FB_CUDA_CHECK(cudaGetLastError());
    note_launch();
    return;
  }
  const i64 n1 = ((n / 2 + CL - 1) / CL) * CL, n2 = n - n1;
  View<R> A11 = csub(A, 0, 0, n1, n1), A21 = csub(A, n1, 0, n2, n1), A22 = csub(A, n1, n1, n2, n2);
  llt_rec_cx(ctx, A11, j0);
  // conj(L11) X = A21^T   (ldlt/factor.rs:421-426)
  solve_lower_rec_cx(ctx.st, cv(A11), false, true, A21.t());
  // A22(lower) -= A21 A21^H   (435-446)
  cgemm(ctx.st, A22, TRI_LOWER, 1, cv(A21), RECT, false, cv(A21).t(), RECT, true, R(-1), R(0));
  llt_rec_cx(ctx, A22, j0 + n1);
}


// ---- partial-pivoting LU (lu/partial_pivoting/factor.rs:19-295 for complex T) ---------------------------------------------
constexpr int LU_CW = 16;         // leaf width
constexpr int LU_CT = 1024;       // leaf threads (one CTA walks the panel's rows in global memory)

// Unblocked leaf on the view A (m rows, `ncols_view` columns; local row 0 = first diagonal row of the window [start, start + w)):
// pivot = first row attaining the largest abs1 = |re| + |im| (strict `>` from 0: an all-zero column keeps the diagonal row),
// the swap covers the whole row of the view (factor.rs:46), multipliers by reciprocal-multiply, rank-1 update of the window.
template <class R>
__global__ void __launch_bounds__(LU_CT) lu_leaf_cx_kernel(R* __restrict__ A, i64 rs, i64 cs, int m, int ncols_view, int start,
                                                            int w, int* __restrict__ trans) {
  __shared__ R red_v[LU_CT / 32];
  __shared__ int red_i[LU_CT / 32];
  __shared__ int s_piv;
  __shared__ R s_inv[2];
  __shared__ R s_row[LU_CW][2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int j = 0; j < w && j < m; ++j) {
    const int col = start + j;
    // ---- pivot search over rows >= j ----
    R bv = R(0);
    int bi = j;
    for (int i = j + tid; i < m; i += LU_CT) {
      const CxT<R> a = cld(A, (i64)i * rs + (i64)col * cs);
      const R v = fabs(a.re) + fabs(a.im);
      if (v > bv) {  // rows ascend within a thread: the first maximum is kept
        bv = v;
        bi = i;
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const R ov = __shfl_xor_sync(0xffffffffu, bv, off);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
      if (ov > bv || (ov == bv && oi < bi)) {
        bv = ov;
        bi = oi;
      }
    }
    if (lane == 0) {
      red_v[warp] = bv;
      red_i[warp] = bi;
    }
    __syncthreads();
    if (warp == 0) {
      bv = red_v[lane];
      bi = red_i[lane];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        const R ov = __shfl_xor_sync(0xffffffffu, bv, off);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
        if (ov > bv || (ov == bv && oi < bi)) {
          bv = ov;
          bi = oi;
        }
      }
      if (lane == 0) {
        s_piv = (bv > R(0)) ? bi : j;
        trans[j] = s_piv - j;
      }
    }
    __syncthreads();
    const int piv = s_piv;
    // ---- swap rows j <-> piv over the whole view ----
    if (piv != j) {
      for (int c = tid; c < ncols_view; c += LU_CT) {
        const CxT<R> a = cld(A, (i64)j * rs + (i64)c * cs), b = cld(A, (i64)piv * rs + (i64)c * cs);
        cst(A, (i64)j * rs + (i64)c * cs, b);
        cst(A, (i64)piv * rs + (i64)c * cs, a);
      }
    }
    __syncthreads();
    if (tid == 0) {
      const CxT<R> d = cld(A, (i64)j * rs + (i64)col * cs);
      const R sc = R(1) / fma(d.re, d.re, d.im * d.im);
      s_inv[0] = d.re * sc;
      s_inv[1] = -d.im * sc;
    }
    if (tid < w - j - 1) {
      const CxT<R> u = cld(A, (i64)j * rs + (i64)(col + 1 + tid) * cs);
      s_row[tid][0] = u.re;
      s_row[tid][1] = u.im;
    }
    __syncthreads();
    const CxT<R> inv{s_inv[0], s_inv[1]};
    // ---- multipliers and rank-1 update: one row per thread and iteration ----
    for (int i = j + 1 + tid; i < m; i += LU_CT) {
      const CxT<R> l = cmul(cld(A, (i64)i * rs + (i64)col * cs), inv);
      cst(A, (i64)i * rs + (i64)col * cs, l);
      for (int c = 0; c < w - j - 1; ++c) {
        const CxT<R> t = cmul(l, CxT<R>{s_row[c][0], s_row[c][1]});
        CxT<R> a = cld(A, (i64)i * rs + (i64)(col + 1 + c) * cs);
        a.re -= t.re;
        a.im -= t.im;
        cst(A, (i64)i * rs + (i64)(col + 1 + c) * cs, a);
      }
    }
    __syncthreads();
  }
}

// apply n transpositions (row j <-> row j + trans[j], in order) to every column of the view: one thread per column
template <class R>
__global__ void laswp_cx_kernel(R* __restrict__ A, i64 rs, i64 cs, i64 ncols, const int* __restrict__ trans, int n) {
  const i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncols) return;
  for (int j = 0; j < n; ++j) {
    const int t = trans[j];
    if (t == 0) continue;
    const CxT<R> a = cld(A, (i64)j * rs + c * cs), b = cld(A, (i64)(j + t) * rs + c * cs);
    cst(A, (i64)j * rs + c * cs, b);
    cst(A, (i64)(j + t) * rs + c * cs, a);
  }
}

inline i64 next_pow2_c(i64 n) {
  i64 p = 1;
  while (p < n) p <<= 1;
  return p;
}

// the reference's recursion (factor.rs:68-187): A = current view (all m rows, ncols columns), window [start, end)
template <class R>
void lu_rec_cx(cudaStream_t st, View<R> A, i64 start, i64 end, int* trans) {
  const i64 m = A.nrows, ncols = A.ncols, n = end - start;
  if (n == 0) return;
  if (n <= LU_CW) {
    lu_leaf_cx_kernel<R><<<1, LU_CT, 0, st>>>(A.ptr, A.rs, A.cs, (int)m, (int)ncols, (int)start, (int)n, trans);
    FB_CUDA_CHECK(cudaGetLastError());
    note_launch();
    return;
  }
  const i64 half = n / 2;
  const i64 pw = std::min<i64>(16, next_pow2_c(half));
  const i64 bs = (half + pw - 1) / pw * pw;
  View<R> W = csub(A, 0, start, m, n);
  lu_rec_cx(st, W, 0, bs, trans);
  {
    View<R> A00 = csub(W, 0, 0, bs, bs), A01 = csub(W, 0, bs, bs, n - bs), A10 = csub(W, bs, 0, m - bs, bs), A11 = csub(W, bs, bs, m - bs, n - bs);
    solve_lower_rec_cx(st, cv(A00), true, false, A01);
    cgemm(st, A11, RECT, 1, cv(A10), RECT, false, cv(A01), RECT, false, R(-1), R(0));
    lu_rec_cx(st, csub(W, bs, 0, m - bs, n), bs, n, trans + bs);
  }
  auto swap_cols = [&](View<R> M) {
    if (M.ncols == 0) return;
    laswp_cx_kernel<R><<<(unsigned)((M.ncols + 127) / 128), 128, 0, st>>>(M.ptr, M.rs, M.cs, M.ncols, trans, (int)n);
    FB_CUDA_CHECK(cudaGetLastError());
    note_launch();
  };
  swap_cols(csub(A, 0, 0, m, start));
  swap_cols(csub(A, 0, end, m, ncols - end));
}

// conj?(T) X = rhs, T lower / upper triangular (unit diagonal or not); views in complex units
template <class R>
void solve_lower_triangular_in_place_cx(cudaStream_t st, View<const R> tril, bool unit, bool conj, View<R> rhs) {
  FB_ASSERT(tril.nrows == tril.ncols && rhs.nrows == tril.nrows, "triangular solve shape mismatch");
  solve_lower_rec_cx(st, tril, unit, conj, rhs);
}
template <class R>
void solve_upper_triangular_in_place_cx(cudaStream_t st, View<const R> triu, bool unit, bool conj, View<R> rhs) {
  FB_ASSERT(triu.nrows == triu.ncols && rhs.nrows == triu.nrows, "triangular solve shape mismatch");
  const i64 n = triu.nrows;
  if (n == 0 || rhs.ncols == 0) return;
  // upper = lower on the views with rows and columns reversed (triangular_solve.rs:577-604)
  View<const R> t{triu.ptr + 2 * ((n - 1) * triu.rs + (n - 1) * triu.cs), n, n, -triu.rs, -triu.cs};
  View<R> r{rhs.ptr + 2 * ((n - 1) * rhs.rs), n, rhs.ncols, -rhs.rs, rhs.cs};
  solve_lower_rec_cx(st, t, unit, conj, r);
}

template <class R>
LltResult llt_cholesky_in_place_cx(cudaStream_t st, View<R> A, R reg_delta, R reg_eps) {
  FB_ASSERT(A.nrows == A.ncols, "LLT needs a square matrix");
  LltResult res{true, 0, 0};
  if (A.nrows == 0) return res;
  long long* d_info = (long long*)ws_alloc(2 * sizeof(long long));
  long long h_info[2] = {-1, 0};
  FB_CUDA_CHECK(cudaMemcpyAsync(d_info, h_info, sizeof(h_info), cudaMemcpyHostToDevice, st));
  LltCtxC<R> ctx{st, (reg_delta > R(0) && reg_eps > R(0)) ? 1 : 0, reg_eps, reg_delta, d_info};
  llt_rec_cx(ctx, A, 0);
  FB_CUDA_CHECK(cudaMemcpyAsync(h_info, d_info, sizeof(h_info), cudaMemcpyDeviceToHost, st));
  FB_CUDA_CHECK(cudaStreamSynchronize(st));
  ws_free(d_info);
  if (h_info[0] >= 0) {
    res.ok = false;
    res.non_positive_pivot_index = (size_t)h_info[0];
  } else {
    res.dynamic_regularization_count = (size_t)h_info[1];
  }
  return res;
}

// L y = b, then L^H x = y (cholesky/llt/solve.rs:12-35 for complex L)
template <class R>
void llt_solve_in_place_cx(cudaStream_t st, View<const R> L, bool conj, View<R> rhs) {
  FB_ASSERT(L.nrows == L.ncols && rhs.nrows == L.nrows, "LLT solve shape mismatch");
  solve_lower_triangular_in_place_cx(st, L, false, conj, rhs);
  solve_upper_triangular_in_place_cx(st, L.t(), false, !conj, rhs);
}

// In-place P A = L U of an m x n c64 matrix (views in complex units); perm arrays: HOST int64 of length m. Returns the
// transposition count (lu_in_place, factor.rs:234-295).
template <class R>
size_t lu_partial_piv_in_place_cx(cudaStream_t st, View<R> A, long long* perm_fwd, long long* perm_inv) {
  const i64 m = A.nrows, n = A.ncols, size = std::min(m, n);
  for (i64 i = 0; i < m; ++i) perm_fwd[i] = i;
  size_t n_trans = 0;
  if (size > 0) {
    int* d_trans = (int*)ws_alloc((size_t)size * sizeof(int));
    FB_CUDA_CHECK(cudaMemsetAsync(d_trans, 0, (size_t)size * sizeof(int), st));
    lu_rec_cx(st, A, 0, size, d_trans);
    std::vector<int> h_trans((size_t)size);
    FB_CUDA_CHECK(cudaMemcpyAsync(h_trans.data(), d_trans, (size_t)size * sizeof(int), cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    ws_free(d_trans);
    for (i64 i = 0; i < size; ++i) {
      const int t = h_trans[(size_t)i];
      if (t != 0) {
        std::swap(perm_fwd[i], perm_fwd[i + t]);
        ++n_trans;
      }
    }
    if (m < n) {  // factor.rs:278-285
      solve_lower_rec_cx(st, cv(csub(A, 0, 0, m, size)), true, false, csub(A, 0, size, m, n - size));
      FB_CUDA_CHECK(cudaStreamSynchronize(st));
    }
  }
  for (i64 i = 0; i < m; ++i) perm_inv[perm_fwd[i]] = i;
  return n_trans;
}

// a complex-unit view as a view of (re, im) elements, for the element-generic row permutation of solve_f64.cu; ReIm<R> keeps R's
// alignment, so a device rhs aligned only to sizeof(R) is moved as before
template <class R>
View<ReIm<R>> as_pairs(View<R> v) { return View<ReIm<R>>{(ReIm<R>*)v.ptr, v.nrows, v.ncols, v.rs, v.cs}; }

// rhs <- conj?(A)^-1 rhs from the factors (lu/partial_pivoting/solve.rs:21-54): permute rows, unit-lower solve, upper solve
template <class R>
void lu_solve_in_place_cx(cudaStream_t st, View<const R> L, View<const R> U, bool conj, const long long* perm_fwd, View<R> rhs) {
  const i64 n = L.nrows;
  FB_ASSERT(L.ncols == n && U.nrows == n && U.ncols == n && rhs.nrows == n, "LU solve shape mismatch");
  if (n == 0 || rhs.ncols == 0) return;
  permute_rows_in_place(st, as_pairs(rhs), perm_fwd);
  solve_lower_triangular_in_place_cx(st, L, true, conj, rhs);
  solve_upper_triangular_in_place_cx(st, U, false, conj, rhs);
}

// rhs <- conj?(A)^-T rhs (solve.rs:55-86): lower solve with U^T, unit-upper solve with L^T, then the inverse row permutation
template <class R>
void lu_solve_transpose_in_place_cx(cudaStream_t st, View<const R> L, View<const R> U, bool conj, const long long* perm_bwd, View<R> rhs) {
  const i64 n = L.nrows;
  FB_ASSERT(L.ncols == n && U.nrows == n && U.ncols == n && rhs.nrows == n, "LU solve shape mismatch");
  if (n == 0 || rhs.ncols == 0) return;
  solve_lower_triangular_in_place_cx(st, U.t(), false, conj, rhs);
  solve_upper_triangular_in_place_cx(st, L.t(), true, conj, rhs);
  permute_rows_in_place(st, as_pairs(rhs), perm_bwd);
}

// ---- Householder QR without pivoting for complex T (qr/no_pivoting/factor.rs:11-301; householder.rs:59-107, 132-272, 370-620,
// 724-808) ---------------------------------------------------------------------------------------------------------------------
// The reference's own structure: an unblocked kernel (one CTA) that carries the column-skipping rank logic, and the blocked
// recursion above it on the host with every product on the complex GEMM; the recursion hands blocks of <= QR_LEAF columns to the
// unblocked kernel whole (the reference's `m * n < blocking_threshold` branch), so one host read-back of the new row index per
// leaf. Functional, not tuned: the panels run on a single SM.
constexpr int QR_CT = 1024;
constexpr int QR_LEAF = 16;

template <class R>
struct RealTraits;
template <>
struct RealTraits<double> {
  static constexpr double min_pos = 2.2250738585072014e-308, eps = 2.220446049250313e-16, sml = 0x1p-511, big = 0x1p511;
};
template <>
struct RealTraits<float> {
  static constexpr float min_pos = 1.17549435e-38f, eps = 1.1920929e-7f, sml = 0x1p-63f, big = 0x1p63f;
};

// norm_l2.rs:161-172: selection between the three scaled accumulators
template <class R>
__device__ __forceinline__ R norm_select(R acc_sml, R acc_med, R acc_big) {
  if (acc_sml >= R(1)) return sqrt(acc_sml) * RealTraits<R>::big;
  if (acc_med >= R(1)) return sqrt(acc_med);
  return sqrt(acc_big) * RealTraits<R>::sml;
}

// qr_in_place_unblocked (factor.rs:11-86) on the view A (m x n), reflector coefficients into H[row * h_stride] (complex units),
// starting at (row_start, col_start); the new row index comes back in out_row[0].
template <class R>
__global__ void __launch_bounds__(QR_CT) qr_unblocked_cx_kernel(R* __restrict__ A, i64 rs, i64 cs, int m, int n, R* __restrict__ H,
                                                                i64 h_stride, int h_len, int row_start, int col_start,
                                                                int* __restrict__ out_row) {
  using Tr = RealTraits<R>;
  using Cx = CxT<R>;
  __shared__ R red[6][QR_CT / 32];
  __shared__ R s_inv[2];
  __shared__ R s_tau_inv;
  __shared__ int s_scale, s_action;  // action: 0 = column skipped, 1 = row advances without an update, 2 = update + advance
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int row = row_start, col = col_start;
  const int row_end = h_len < m ? h_len : m;
  while (row < row_end && col < n) {
    const int len = m - row - 1;
    // ---- norm of the column above `row` and of the tail below it (three scaled accumulators each, norm_l2.rs:6-172) ----
    R a0 = 0, a1 = 0, a2 = 0, t0 = 0, t1 = 0, t2 = 0;
    for (int i = tid; i < m; i += QR_CT) {
      if (i == row) continue;
      const Cx x = cld(A, (i64)i * rs + (i64)col * cs);
      const R xs = x.re * Tr::sml, ys = x.im * Tr::sml, xb = x.re * Tr::big, yb = x.im * Tr::big;
      const R q0 = fma(xs, xs, ys * ys), q1 = fma(x.re, x.re, x.im * x.im), q2 = fma(xb, xb, yb * yb);
      if (i < row) {
        a0 += q0; a1 += q1; a2 += q2;
      } else {
        t0 += q0; t1 += q1; t2 += q2;
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      a0 += __shfl_xor_sync(0xffffffffu, a0, off);
      a1 += __shfl_xor_sync(0xffffffffu, a1, off);
      a2 += __shfl_xor_sync(0xffffffffu, a2, off);
      t0 += __shfl_xor_sync(0xffffffffu, t0, off);
      t1 += __shfl_xor_sync(0xffffffffu, t1, off);
      t2 += __shfl_xor_sync(0xffffffffu, t2, off);
    }
    if (lane == 0) {
      red[0][warp] = a0; red[1][warp] = a1; red[2][warp] = a2;
      red[3][warp] = t0; red[4][warp] = t1; red[5][warp] = t2;
    }
    __syncthreads();
    if (tid == 0) {
      R acc[6];
      for (int q = 0; q < 6; ++q) {
        R v = 0;
        for (int w = 0; w < QR_CT / 32; ++w) v += red[q][w];
        acc[q] = v;
      }
      const R norm_above = norm_select(acc[0], acc[1], acc[2]);
      const R tail_norm = norm_select(acc[3], acc[4], acc[5]);
      // make_householder_imp (householder.rs:59-107)
      Cx head = cld(A, (i64)row * rs + (i64)col * cs);
      R head_norm = hypot(head.re, head.im);
      if (head_norm < Tr::min_pos) {
        head = Cx{R(0), R(0)};
        head_norm = R(0);
        cst(A, (i64)row * rs + (i64)col * cs, head);
      }
      R tau, info_norm;
      int scale = 0;
      if (tail_norm < Tr::min_pos) {
        tau = R(INFINITY);
        info_norm = head_norm;
      } else {
        const R norm = hypot(head_norm, tail_norm);
        Cx sign{R(1), R(0)};
        if (head_norm != R(0)) {
          const R hi = R(1) / head_norm;
          sign = Cx{head.re * hi, head.im * hi};
        }
        const Cx signed_norm{sign.re * norm, sign.im * norm};
        const Cx inv = crecip(Cx{head.re + signed_norm.re, head.im + signed_norm.im});
        cst(A, (i64)row * rs + (i64)col * cs, Cx{-signed_norm.re, -signed_norm.im});
        const R t = tail_norm * hypot(inv.re, inv.im);
        tau = R(0.5) * (R(1) + t * t);
        info_norm = norm;
        s_inv[0] = inv.re;
        s_inv[1] = inv.im;
        scale = 1;
      }
      // rank test (factor.rs:41-53)
      const R nrm = hypot(info_norm, norm_above);
      const R threshold = Tr::eps * (R)((double)(m - row) * 16.0) * nrm;
      const R tau_inv = R(1) / tau;
      cst(H, (i64)row * h_stride, Cx{tau, R(0)});
      int action = 0;
      if (tau_inv < Tr::min_pos) {
        if (info_norm > R(0)) action = 1;
      } else if (info_norm > threshold) {
        action = 2;
      }
      s_tau_inv = tau_inv;
      s_scale = scale;
      s_action = action;
    }
    __syncthreads();
    const int action = s_action, scale = s_scale;
    const int vcol = row;  // the essential part always lives below the diagonal of column `row` (== col when nothing was skipped)
    {
      const Cx inv{s_inv[0], s_inv[1]};
      const int z = (col - row) < len ? (col - row) : len;  // rows of column `col` to clear when row != col (factor.rs:33-38)
      for (int i = tid; i < len; i += QR_CT) {
        const i64 r_ = (i64)(row + 1 + i) * rs;
        if (scale) cst(A, r_ + (i64)vcol * cs, cmul(cld(A, r_ + (i64)col * cs), inv));
        if (row != col && i < z) cst(A, r_ + (i64)col * cs, Cx{R(0), R(0)});
      }
    }
    __syncthreads();
    if (action == 2) {
      const R tau_inv = s_tau_inv;
      for (int c = col + 1 + warp; c < n; c += QR_CT / 32) {
        R dr = 0, di = 0;
        for (int i = lane; i < len; i += 32) {
          const i64 r_ = (i64)(row + 1 + i) * rs;
          const Cx v = cld(A, r_ + (i64)vcol * cs), a = cld(A, r_ + (i64)c * cs);
          dr += fma(v.re, a.re, v.im * a.im);   // conj(v) * a
          di += fma(v.re, a.im, -v.im * a.re);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
          dr += __shfl_xor_sync(0xffffffffu, dr, off);
          di += __shfl_xor_sync(0xffffffffu, di, off);
        }
        const Cx a0c = cld(A, (i64)row * rs + (i64)c * cs);
        const Cx k{-(a0c.re + dr) * tau_inv, -(a0c.im + di) * tau_inv};
        if (lane == 0) cst(A, (i64)row * rs + (i64)c * cs, Cx{a0c.re + k.re, a0c.im + k.im});
        for (int i = lane; i < len; i += 32) {
          const i64 r_ = (i64)(row + 1 + i) * rs;
          const Cx t = cmul(k, cld(A, r_ + (i64)vcol * cs));
          Cx a = cld(A, r_ + (i64)c * cs);
          a.re += t.re;
          a.im += t.im;
          cst(A, r_ + (i64)c * cs, a);
        }
      }
    }
    __syncthreads();
    if (action != 0) row += 1;
    col += 1;
  }
  if (tid == 0) out_row[0] = row;
}

// factor.rs:190-203: after a leaf produced `local` reflectors with sub-block size sbs, the s2 x s2 upper-triangular T blocks
// sit in the first rows of H (view Hs: rows from `offset`, columns from `row`); block k moves down to rows [k, k + s2)
template <class R>
__global__ void qr_shift_tblocks_cx_kernel(R* __restrict__ Hs, i64 rs, i64 cs, int local, int sbs) {
  for (int e = threadIdx.x; e < local * sbs; e += blockDim.x) {
    const int col = e / sbs, i = e % sbs;
    const int k = (col / sbs) * sbs, j = col - k;
    if (k == 0 || i > j) continue;
    cst(Hs, (i64)(k + i) * rs + (i64)col * cs, cld(Hs, (i64)i * rs + (i64)col * cs));
  }
}

// factor.rs:283-299: columns >= rank of Q_coeff are zero with +inf on the block diagonals
template <class R>
__global__ void qr_finish_cx_kernel(R* __restrict__ H, i64 rs, i64 cs, int bs, int size, int rank) {
  const i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (i64)bs * (size - rank)) return;
  const int i = (int)(e % bs), j = rank + (int)(e / bs);
  const bool diag = i == j - (j / bs) * bs;
  cst(H, (i64)i * rs + (i64)j * cs, CxT<R>{diag ? R(INFINITY) : R(0), R(0)});
}

template <class R>
struct QrCtx {
  cudaStream_t st;
  int* d_row;
  R* tmp;  // block_size x ncols complex scratch of the block applies
  i64 blocking_threshold;
};

template <class R>
i64 qr_unblocked_cx(const QrCtx<R>& cx, View<R> A, View<R> Hrow, i64 row_start, i64 col_start) {
  if (!(row_start < std::min(Hrow.ncols, A.nrows) && col_start < A.ncols)) return row_start;
  qr_unblocked_cx_kernel<R><<<1, QR_CT, 0, cx.st>>>(A.ptr, A.rs, A.cs, (int)A.nrows, (int)A.ncols, Hrow.ptr, Hrow.cs, (int)Hrow.ncols,
                                                    (int)row_start, (int)col_start, cx.d_row);
  FB_CUDA_CHECK(cudaGetLastError());
  note_launch();
  int h_row = 0;
  FB_CUDA_CHECK(cudaMemcpyAsync(&h_row, cx.d_row, sizeof(int), cudaMemcpyDeviceToHost, cx.st));
  FB_CUDA_CHECK(cudaStreamSynchronize(cx.st));
  return h_row;
}

// upgrade_householder_factor (householder.rs:132-272): T = striu(V^H V), the diagonal (tau) kept
template <class R>
void upgrade_householder_factor_cx(cudaStream_t st, View<R> Tf, View<const R> V, i64 block_size, i64 prev_block_size) {
  if (block_size == prev_block_size || Tf.nrows <= prev_block_size) return;
  const i64 n = V.ncols;
  const i64 block_count = (Tf.nrows + block_size - 1) / block_size;
  if (block_count > 1) {
    const i64 mid = block_count / 2;  // householder.rs:155-157 splits at the block COUNT
    upgrade_householder_factor_cx<R>(st, csub(Tf, 0, 0, mid, mid), csub(V, 0, 0, V.nrows, mid), block_size, prev_block_size);
    upgrade_householder_factor_cx<R>(st, csub(Tf, mid, mid, Tf.nrows - mid, Tf.ncols - mid),
                                     csub(V, mid, mid, V.nrows - mid, V.ncols - mid), block_size, prev_block_size);
    return;
  }
  if (prev_block_size < 8) {
    View<const R> top = csub(V, 0, 0, n, n), bot = csub(V, n, 0, V.nrows - n, n);
    cgemm(st, Tf, UNIT_UPPER, 0, top.t(), UNIT_UPPER, true, top, UNIT_LOWER, false, R(1), R(0));
    if (bot.nrows > 0) cgemm(st, Tf, UNIT_UPPER, 1, bot.t(), RECT, true, bot, RECT, false, R(1), R(0));
  } else {
    const i64 prev_block_count = (Tf.nrows + prev_block_size - 1) / prev_block_size;
    const i64 mid = (prev_block_count / 2) * prev_block_size;
    View<R> tl = csub(Tf, 0, 0, mid, mid), tr = csub(Tf, 0, mid, mid, Tf.ncols - mid), br = csub(Tf, mid, mid, Tf.nrows - mid, Tf.ncols - mid);
    View<const R> left = csub(V, 0, 0, V.nrows, mid), right = csub(V, mid, mid, V.nrows - mid, V.ncols - mid);
    upgrade_householder_factor_cx<R>(st, tl, left, block_size, prev_block_size);
    upgrade_householder_factor_cx<R>(st, br, right, block_size, prev_block_size);
    View<const R> left2 = csub(left, mid, 0, left.nrows - mid, left.ncols);
    const i64 row_mid = right.ncols;
    View<const R> lt = csub(left2, 0, 0, row_mid, left2.ncols), lb = csub(left2, row_mid, 0, left2.nrows - row_mid, left2.ncols);
    View<const R> rt = csub(right, 0, 0, row_mid, right.ncols), rb = csub(right, row_mid, 0, right.nrows - row_mid, right.ncols);
    cgemm(st, tr, RECT, 0, lt.t(), RECT, true, rt, UNIT_LOWER, false, R(1), R(0));
    if (lb.nrows > 0) cgemm(st, tr, RECT, 1, lb.t(), RECT, true, rb, RECT, false, R(1), R(0));
  }
}

// apply_block_householder_on_the_left (householder.rs:370-620): M <- (I - V T^-1 V^H) M (forward = false) or
// (I - V T^-H V^H) M (forward = true), conj_lhs conjugating V and T; tmp: N x K complex scratch
template <class R>
void apply_block_householder_left_cx(cudaStream_t st, View<const R> V, View<const R> Tf, bool conj_lhs, View<R> M, bool forward, R* tmpbuf) {
  const i64 N = V.ncols, m = V.nrows, K = M.ncols;
  if (N == 0 || K == 0) return;
  View<R> tmp{tmpbuf, N, K, 1, N};
  View<const R> Vt = csub(V, 0, 0, N, N), Vb = csub(V, N, 0, m - N, N);
  View<R> top = csub(M, 0, 0, N, K), bot = csub(M, N, 0, m - N, K);
  cgemm(st, tmp, RECT, 0, Vt.t(), UNIT_UPPER, !conj_lhs, View<const R>{top.ptr, N, K, top.rs, top.cs}, RECT, false, R(1), R(0));
  if (m > N) cgemm(st, tmp, RECT, 1, Vb.t(), RECT, !conj_lhs, View<const R>{bot.ptr, m - N, K, bot.rs, bot.cs}, RECT, false, R(1), R(0));
  if (forward) solve_lower_rec_cx<R>(st, Tf.t(), false, !conj_lhs, tmp);
  else {
    // upper = lower on the views with rows and columns reversed
    View<const R> t{Tf.ptr + 2 * ((N - 1) * Tf.rs + (N - 1) * Tf.cs), N, N, -Tf.rs, -Tf.cs};
    View<R> r{tmp.ptr + 2 * ((N - 1) * tmp.rs), N, K, -tmp.rs, tmp.cs};
    solve_lower_rec_cx<R>(st, t, false, conj_lhs, r);
  }
  View<const R> ctmp{tmp.ptr, N, K, tmp.rs, tmp.cs};
  cgemm(st, top, RECT, 1, Vt, UNIT_LOWER, conj_lhs, ctmp, RECT, false, R(-1), R(0));
  if (m > N) cgemm(st, bot, RECT, 1, Vb, RECT, conj_lhs, ctmp, RECT, false, R(-1), R(0));
}

// qr_in_place_blocked (factor.rs:137-256)
template <class R>
i64 qr_blocked_cx(const QrCtx<R>& cx, View<R> A, View<R> H, i64 row_start, i64 col_start) {
  const i64 m = A.nrows, n = A.ncols, size = std::min(m, n);
  const i64 block_size0 = H.nrows;
  if (block_size0 == 1) return qr_unblocked_cx<R>(cx, A, H, row_start, col_start);
  const i64 sub_block_size0 = (block_size0 <= QR_LEAF || m * n < cx.blocking_threshold) ? 1 : block_size0 / 2;
  i64 col = col_start, row = row_start;
  while (row < size && col < n) {
    const i64 block_size = std::min(block_size0, std::min(size - row, n - col));
    const i64 sub_block_size = std::min(block_size, sub_block_size0);
    const i64 start = row;
    i64 offset = 0;
    while (offset < block_size && col < n) {
      const i64 bsz = std::min(n - col, block_size - offset);
      const i64 sbs = std::min(bsz, sub_block_size);
      const i64 new_row = qr_blocked_cx<R>(cx, csub(A, 0, 0, m, col + bsz), csub(H, offset, 0, sbs, H.ncols), row, col);
      const i64 local = new_row - row;
      if (local > 0) {
        if (local > sbs) {
          View<R> Hs = csub(H, offset, row, H.nrows - offset, local);
          qr_shift_tblocks_cx_kernel<R><<<1, 256, 0, cx.st>>>(Hs.ptr, Hs.rs, Hs.cs, (int)local, (int)sbs);
          FB_CUDA_CHECK(cudaGetLastError());
          note_launch();
        }
        View<R> Arr = csub(A, row, row, m - row, local);
        upgrade_householder_factor_cx<R>(cx.st, csub(H, offset, row, local, local), View<const R>{Arr.ptr, Arr.nrows, Arr.ncols, Arr.rs, Arr.cs},
                                         local, sbs);
        if (offset > 0) {
          const i64 w = offset + local;
          View<R> Hh = csub(H, 0, start, w, w);
          View<R> Aa_ = csub(A, start, start, m - start, w);
          View<const R> Aa{Aa_.ptr, Aa_.nrows, Aa_.ncols, Aa_.rs, Aa_.cs};
          View<const R> A0 = csub(Aa, 0, 0, w, w), A1 = csub(Aa, w, 0, Aa.nrows - w, w);
          cgemm(cx.st, Hh, UNIT_UPPER, 0, A0.t(), UNIT_UPPER, true, A0, UNIT_LOWER, false, R(1), R(0));
          if (A1.nrows > 0) cgemm(cx.st, Hh, UNIT_UPPER, 1, A1.t(), RECT, true, A1, RECT, false, R(1), R(0));
        }
      }
      View<R> below = csub(A, row, 0, m - row, n);
      View<R> Q0_ = csub(below, 0, row, m - row, local);
      View<R> A1 = csub(below, 0, col + bsz, m - row, n - (col + bsz));
      View<R> Hq_ = csub(H, offset, row, local, local);
      if (A1.ncols > 0 && local > 0)
        apply_block_householder_left_cx<R>(cx.st, View<const R>{Q0_.ptr, Q0_.nrows, Q0_.ncols, Q0_.rs, Q0_.cs},
                                           View<const R>{Hq_.ptr, Hq_.nrows, Hq_.ncols, Hq_.rs, Hq_.cs}, false, A1, true, cx.tmp);
      offset += local;
      row += local;
      col += bsz;
    }
  }
  return row;
}

// qr_in_place (factor.rs:258-301): returns the rank
template <class R>
i64 qr_in_place_cx(cudaStream_t st, View<R> A, View<R> Q_coeff, i64 blocking_threshold) {
  const i64 m = A.nrows, n = A.ncols, size = std::min(m, n), bs = Q_coeff.nrows;
  FB_ASSERT(bs > 0 && Q_coeff.ncols == size, "Q_coeff must be block_size x min(nrows, ncols)");
  if (size == 0) return 0;
  FB_ASSERT(m < (i64(1) << 31) && n < (i64(1) << 31), "complex QR dimensions limited to 2^31");
  int* d_row = (int*)ws_alloc(sizeof(int));
  R* tmp = (R*)ws_alloc((size_t)bs * (size_t)n * 2 * sizeof(R));
  QrCtx<R> cx{st, d_row, tmp, blocking_threshold};
  const i64 rank = qr_blocked_cx<R>(cx, A, Q_coeff, 0, 0);
  if (rank < size) {
    const i64 cnt = bs * (size - rank);
    qr_finish_cx_kernel<R><<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>(Q_coeff.ptr, Q_coeff.rs, Q_coeff.cs, (int)bs, (int)size, (int)rank);
    FB_CUDA_CHECK(cudaGetLastError());
    note_launch();
  }
  FB_CUDA_CHECK(cudaStreamSynchronize(st));
  ws_free(tmp);
  ws_free(d_row);
  return rank;
}

// apply_block_householder_sequence_[transpose_]on_the_left_in_place_with_conj (householder.rs:724-808): rhs <- Q rhs or Q^H rhs
// (with conj: the conjugated Q), Q given by its basis (unit-lower trapezoid) and block_size x size factor
template <class R>
void apply_householder_sequence_left_cx(cudaStream_t st, View<const R> basis, View<const R> factor, bool conj, View<R> rhs, bool transpose) {
  const i64 bs = factor.nrows, size = factor.ncols, m = basis.nrows, K = rhs.ncols;
  FB_ASSERT(bs > 0 && size == std::min(basis.nrows, basis.ncols) && rhs.nrows == m, "Householder sequence shape mismatch");
  if (size == 0 || K == 0) return;
  R* tmp = (R*)ws_alloc((size_t)bs * (size_t)K * 2 * sizeof(R));
  if (transpose) {
    // householder.rs:768-808: blocks in ascending order, each through transpose_on_the_left = conj composed with Yes, forward
    for (i64 j = 0; j < size;) {
      const i64 b = std::min(bs, size - j);
      apply_block_householder_left_cx<R>(st, csub(basis, j, j, m - j, b), csub(factor, 0, j, b, b), !conj, csub(rhs, j, 0, m - j, K), true, tmp);
      j += b;
    }
  } else {
    // householder.rs:724-765: blocks in descending order (the last block may be short)
    i64 j = size, b = size % bs ? size % bs : bs;
    while (j > 0) {
      const i64 jp = j - b;
      apply_block_householder_left_cx<R>(st, csub(basis, jp, jp, m - jp, b), csub(factor, 0, jp, b, b), conj, csub(rhs, jp, 0, m - jp, K), false, tmp);
      j = jp;
      b = bs;
    }
  }
  FB_CUDA_CHECK(cudaStreamSynchronize(st));
  ws_free(tmp);
}

}  // namespace

// ---- exported entry points (linalg_f64.cuh / gemm_f32.cuh) ------------------------------------------------------------------
#define FB_CPLX_EXPORTS(SUF, R)                                                                                                   \
  void solve_lower_triangular_in_place_##SUF(cudaStream_t st, View<const R> t, bool unit, bool conj, View<R> rhs) {              \
    solve_lower_triangular_in_place_cx<R>(st, t, unit, conj, rhs);                                                               \
  }                                                                                                                               \
  void solve_upper_triangular_in_place_##SUF(cudaStream_t st, View<const R> t, bool unit, bool conj, View<R> rhs) {              \
    solve_upper_triangular_in_place_cx<R>(st, t, unit, conj, rhs);                                                               \
  }                                                                                                                               \
  LltResult llt_cholesky_in_place_##SUF(cudaStream_t st, View<R> A, R reg_delta, R reg_eps) {                                    \
    return llt_cholesky_in_place_cx<R>(st, A, reg_delta, reg_eps);                                                               \
  }                                                                                                                               \
  void llt_solve_in_place_##SUF(cudaStream_t st, View<const R> L, bool conj, View<R> rhs) { llt_solve_in_place_cx<R>(st, L, conj, rhs); } \
  size_t lu_partial_piv_in_place_##SUF(cudaStream_t st, View<R> A, long long* perm_fwd, long long* perm_inv) {                   \
    return lu_partial_piv_in_place_cx<R>(st, A, perm_fwd, perm_inv);                                                             \
  }                                                                                                                               \
  void lu_solve_in_place_##SUF(cudaStream_t st, View<const R> L, View<const R> U, bool conj, const long long* perm_fwd, View<R> rhs) { \
    lu_solve_in_place_cx<R>(st, L, U, conj, perm_fwd, rhs);                                                                      \
  }                                                                                                                               \
  void lu_solve_transpose_in_place_##SUF(cudaStream_t st, View<const R> L, View<const R> U, bool conj, const long long* perm_bwd, \
                                         View<R> rhs) {                                                                           \
    lu_solve_transpose_in_place_cx<R>(st, L, U, conj, perm_bwd, rhs);                                                            \
  }                                                                                                                               \
  i64 qr_in_place_##SUF(cudaStream_t st, View<R> A, View<R> Q_coeff, i64 blocking_threshold) {                                   \
    return qr_in_place_cx<R>(st, A, Q_coeff, blocking_threshold);                                                                \
  }                                                                                                                               \
  void apply_householder_sequence_left_##SUF(cudaStream_t st, View<const R> basis, View<const R> factor, bool conj, View<R> rhs, \
                                             bool transpose) {                                                                    \
    apply_householder_sequence_left_cx<R>(st, basis, factor, conj, rhs, transpose);                                               \
  }
FB_CPLX_EXPORTS(c64, double)
FB_CPLX_EXPORTS(c32, float)
#undef FB_CPLX_EXPORTS

}  // namespace fb
