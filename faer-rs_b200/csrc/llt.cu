// P1 + driver: in-place lower Cholesky (LLT), f64 and f32 (one templated leaf kernel and recursive driver).
//
// Reference: faer/src/linalg/cholesky/llt/factor.rs:68-97 -> ldlt/factor.rs:367-498
// (`cholesky_recursion_right_looking`: for each block column: factor A00, A10 <- A10 * L00^-H,
//  A11(lower) -= A10 * A10^H), leaf recurrence ldlt/factor.rs:7-177 / 299-366:
//     a_ij <- fma(-conj(a_jk), a_ik, a_ij)  for k = 0..j-1 (in k order),
//     d = Re(a_jj); [regularise]; fail with Err(j) if !(d > 0); l_jj = sqrt(d); fail if l_jj == 0 or non-finite;
//     column j (INCLUDING the diagonal entry) is multiplied by recip(l_jj).
//
// B200 mapping: recursive blocked driver on the host stream; the <=128-wide diagonal block is factored by ONE CTA:
//   * 16 "update" warps hold the block in REGISTERS (thread (lane, w) owns rows lane+32a, columns w+16b) and apply the
//     reference's per-element FMA chain (same k order, same reciprocal-multiply, diagonal scaled too) => bit-identical
//     to the reference leaf recurrence;
//   * 4 "pivot" warps keep a redundant copy of the diagonal (updated with the very same FMA sequence, so bit-identical)
//     and do the serial pivot arithmetic (regularise, test, sqrt, reciprocal) of column j+1 WHILE the update warps are
//     still applying column j — the sqrt+divide latency is off the update warps' critical path;
//   * each column costs one __syncthreads; the unscaled pivot column travels through a double-buffered shared vector.
// The panel solve is G3 and the trailing update is the lower-masked DMMA GEMM (G2). A device status word carries the
// first failing column / the regularisation count and is read back once per factorisation.
#include "gemm_f32.cuh"
#include "linalg_f64.cuh"

namespace fb {

namespace {

constexpr int POTF2_MAX = 128;
constexpr int POTF2_UPD_WARPS = 16;
constexpr int POTF2_THREADS = POTF2_UPD_WARPS * 32 + POTF2_MAX;  // 512 update threads + 128 pivot threads
constexpr int POTF2_CB = POTF2_MAX / POTF2_UPD_WARPS;           // column slots per update thread (8)

__device__ __forceinline__ double recip_rn(double x) { return __drcp_rn(x); }
__device__ __forceinline__ float recip_rn(float x) { return __frcp_rn(x); }

// scalar-type dispatch of the two building blocks the recursion calls (G3 solve, lower-masked GEMM)
inline void solve_lower(cudaStream_t st, VCD tri, bool unit, VD rhs) { solve_lower_triangular_in_place_f64(st, tri, unit, rhs); }
inline void solve_lower(cudaStream_t st, VCF tri, bool unit, VF rhs) { solve_lower_triangular_in_place_f32(st, tri, unit, rhs); }
// dst(lower) -= a * a^H
inline void gemm_lower_update(cudaStream_t st, VD dst, VCD a) { gemm_f64(st, dst, TRI_LOWER, 1, a, RECT, a.t(), RECT, -1.0); }
inline void gemm_lower_update(cudaStream_t st, VF dst, VCF a) { gemm_f32(st, dst, TRI_LOWER, 1, a, RECT, a.t(), RECT, -1.0f); }

// info[0]: first failing global column (or -1), info[1]: regularisation count
template <class T>
__global__ void __launch_bounds__(POTF2_THREADS) potf2_kernel(T* __restrict__ A, i64 rs, i64 cs, int n, i64 j0,
                                                               int regularize, T eps, T delta,
                                                               long long* __restrict__ info) {
  __shared__ T colbuf[2][POTF2_MAX];
  __shared__ T s_inv[2];
  __shared__ int s_fail[2];
  __shared__ int s_count;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool is_upd = warp < POTF2_UPD_WARPS;
  const int p = tid - POTF2_UPD_WARPS * 32;  // pivot-thread index (diagonal entry p) when !is_upd
  if (info[0] >= 0) return;  // an earlier block already failed (uniform across the CTA)
  if (tid == 0) s_count = 0;

  // update threads: rows i = lane + 32a, columns c = warp + 16b, kept iff c <= i < n
  T a[4][POTF2_CB];
  T dp = T(0);  // pivot threads: diagonal entry p
  if (is_upd) {
#pragma unroll
    for (int ai = 0; ai < 4; ++ai)
#pragma unroll
      for (int bi = 0; bi < POTF2_CB; ++bi) {
        const int i = lane + 32 * ai, c = warp + POTF2_UPD_WARPS * bi;
        a[ai][bi] = (i < n && c <= i) ? A[(i64)i * rs + (i64)c * cs] : T(0);
      }
  } else if (p < n) {
    dp = A[(i64)p * rs + (i64)p * cs];
  }
  __syncthreads();  // s_count initialised

  // serial pivot arithmetic of column jc (reference ldlt/factor.rs:122-160), done by ONE pivot thread
  auto publish_pivot = [&](int jc, T d) {
    int fail = 0;
    if (regularize) {
      if (d <= eps) {  // LLT: sign == +1
        d = delta;
        s_count += 1;  // single writer per column, ordered by the per-column barrier
      }
    }
    T inv = T(0);
    if (!(d > T(0))) {
      fail = 1;
    } else {
      const T sd = sqrt(d);
      if (sd == T(0) || !isfinite(sd)) fail = 1;
      else inv = recip_rn(sd);  // correctly rounded reciprocal = T(1) / sd bit for bit, without the division's slow path
    }
    s_inv[jc & 1] = inv;
    s_fail[jc & 1] = fail;
  };

  if (is_upd) {
    if (warp == 0) {
#pragma unroll
      for (int ai = 0; ai < 4; ++ai) colbuf[0][lane + 32 * ai] = a[ai][0];
    }
  } else if (p == 0) {
    publish_pivot(0, dp);
  }
  __syncthreads();

  for (int j = 0; j < n; ++j) {
    const T* col = colbuf[j & 1];
    if (s_fail[j & 1]) {
      if (tid == 0) info[0] = j0 + j;
      return;
    }
    const T inv = s_inv[j & 1];
    if (!is_upd) {
      // pivot group: keep the diagonal current with the SAME fma the update threads apply to a_pp, then start the
      // next column's pivot arithmetic immediately
      if (p > j && p < n) {
        const T l = col[p] * inv;
        dp = fma(-l, l, dp);
        if (p == j + 1) publish_pivot(j + 1, dp);
      }
    } else {
      const int jw = j & (POTF2_UPD_WARPS - 1);
      // column j of L goes to global memory (owners: warp jw).
      // NB: like the reference, the stored diagonal is (unregularised a_jj) * recip(l_jj)
      // (ldlt/factor.rs:161-175 scales the whole column, diagonal included, and `diag` is a local copy).
      if (warp == jw) {
#pragma unroll
        for (int ai = 0; ai < 4; ++ai) {
          const int i = lane + 32 * ai;
          if (i >= j && i < n) A[(i64)i * rs + (i64)j * cs] = col[i] * inv;
        }
      }
      // trailing update: a_ic <- fma(-l_cj, l_ij, a_ic) for j < c <= i. The column test depends only on
      // (warp, bi, j): warp-uniform, so dead column slots are BRANCHED over (no predicated-off instruction issue).
      if (warp + POTF2_UPD_WARPS * (POTF2_CB - 1) > j) {
        T li[4];
#pragma unroll
        for (int ai = 0; ai < 4; ++ai) li[ai] = col[lane + 32 * ai] * inv;
#pragma unroll
        for (int bi = 0; bi < POTF2_CB; ++bi) {
          const int c = warp + POTF2_UPD_WARPS * bi;
          if (c > j && c < n) {
            const T lc = col[c] * inv;
#pragma unroll
            for (int ai = 0; ai < 4; ++ai) {
              const int i = lane + 32 * ai;
              if (32 * ai + 31 >= c) {  // warp-uniform: this row slot intersects i >= c
                if (i >= c && i < n) a[ai][bi] = fma(-lc, li[ai], a[ai][bi]);
              }
            }
          }
        }
      }
      // owners of column j+1 publish it (unscaled) into the other buffer
      if (j + 1 < n && warp == ((j + 1) & (POTF2_UPD_WARPS - 1))) {
        const int nbk = (j + 1) / POTF2_UPD_WARPS;
        T* nxt = colbuf[(j + 1) & 1];
#pragma unroll
        for (int ai = 0; ai < 4; ++ai) {
          T v = T(0);
#pragma unroll
          for (int bi = 0; bi < POTF2_CB; ++bi)
            if (bi == nbk) v = a[ai][bi];
          nxt[lane + 32 * ai] = v;
        }
      }
    }
    __syncthreads();
  }
  if (tid == 0 && s_count) info[1] += s_count;
}

template <class T>
struct LltCtx {
  cudaStream_t stream;
  int regularize;
  T eps, delta;
  long long* d_info;
  i64 nb;  // leaf (diagonal block) size, <= POTF2_MAX
};

// Recursive blocked LLT. Same dataflow as the reference's right-looking recursion (factor A00, solve the panel,
// update the trailing lower triangle, continue) but split in HALVES instead of fixed 128-wide steps, so that
// almost all flops are DMMA GEMMs with a large contracted dimension (k = n/2, n/4, ...): the trailing matrix is
// read/written O(log n) times instead of n/128 times. Leaves (<= nb) are the single-CTA potf2 kernel.
template <class T>
void llt_rec(const LltCtx<T>& ctx, View<T> A, i64 j0) {
  const i64 n = A.nrows;
  if (n <= ctx.nb) {
    potf2_kernel<T><<<1, POTF2_THREADS, 0, ctx.stream>>>(A.ptr, A.rs, A.cs, (int)n, j0, ctx.regularize, ctx.eps, ctx.delta,
                                                      ctx.d_info);
    FB_CUDA_CHECK(cudaGetLastError());
    note_launch();
    return;
  }
  // split at a multiple of the leaf size closest to n/2
  i64 n1 = ((n / 2 + ctx.nb - 1) / ctx.nb) * ctx.nb;
  if (n1 >= n) n1 = ((n - 1) / ctx.nb) * ctx.nb;
  const i64 n2 = n - n1;
  View<T> A11 = A.sub(0, 0, n1, n1), A21 = A.sub(n1, 0, n2, n1), A22 = A.sub(n1, n1, n2, n2);
  llt_rec(ctx, A11, j0);
  // conj(L11) X = A21^T   (reference ldlt/factor.rs:421-426)
  solve_lower(ctx.stream, cv(A11), false, A21.t());
  // A22(lower) += -1 * A21 * A21^H   (reference ldlt/factor.rs:435-446)
  gemm_lower_update(ctx.stream, A22, cv(A21));
  llt_rec(ctx, A22, j0 + n1);
}

}  // namespace

namespace {
// the recursive driver with its own status word (one read-back per factorisation)
template <class T>
LltResult llt_recursive_in_place(cudaStream_t stream, View<T> A, T reg_delta, T reg_eps, LltParams params) {
  LltResult res{true, 0, 0};
  const int regularize = (reg_delta > T(0) && reg_eps > T(0)) ? 1 : 0;
  i64 nb = (i64)params.block_size;
  if (nb <= 0 || nb > POTF2_MAX) nb = POTF2_MAX;

  long long* d_info = (long long*)ws_alloc(2 * sizeof(long long));
  long long h_info[2] = {-1, 0};
  FB_CUDA_CHECK(cudaMemcpyAsync(d_info, h_info, sizeof(h_info), cudaMemcpyHostToDevice, stream));

  LltCtx<T> ctx{stream, regularize, reg_eps, reg_delta, d_info, nb};
  llt_rec<T>(ctx, A, 0);

  FB_CUDA_CHECK(cudaMemcpyAsync(h_info, d_info, sizeof(h_info), cudaMemcpyDeviceToHost, stream));
  FB_CUDA_CHECK(cudaStreamSynchronize(stream));
  ws_free(d_info);
  if (h_info[0] >= 0) {
    res.ok = false;
    res.non_positive_pivot_index = (size_t)h_info[0];
  } else {
    res.dynamic_regularization_count = (size_t)h_info[1];
  }
  return res;
}
}  // namespace

// Device-side variant for callers that own the status word (multi-GPU driver): no synchronisation, no read-back.
// d_info[0] must hold -1 (or the first failing column of an earlier block), d_info[1] the regularisation count.
void llt_cholesky_device_f64(cudaStream_t stream, VD A, double reg_delta, double reg_eps, long long* d_info, i64 j0) {
  FB_ASSERT(A.nrows == A.ncols, "LLT needs a square matrix");
  if (A.nrows == 0) return;
  const int regularize = (reg_delta > 0.0 && reg_eps > 0.0) ? 1 : 0;
  LltCtx<double> ctx{stream, regularize, reg_eps, reg_delta, d_info, POTF2_MAX};
  llt_rec<double>(ctx, A, j0);
}

LltResult llt_cholesky_in_place_f64(cudaStream_t stream, VD A, double reg_delta, double reg_eps, LltParams params) {
  FB_ASSERT(A.nrows == A.ncols, "LLT needs a square matrix");
  const i64 n = A.nrows;
  LltResult res{true, 0, 0};
  if (n == 0) return res;
  // Large column-major problems: right-looking block-column driver with two-stream look-ahead (dist.cu run on a
  // single rank): the panel chain (potf2 + solves of block column k+1) overlaps the trailing update of step k.
  // Measured on B200 at n = 16384: 67.5 ms vs 80.8 ms for the purely recursive driver (profiles/r01_lookahead_p1.log).
  if (A.rs == 1 && n >= lookahead_min_n()) {
    // block width: with the trailing update of a step as ONE structured launch the short chain of narrow blocks wins
    // (n = 16384, profiles/r01_nb_sweep2.log): 256 -> 59.3 ms, 512 -> 60.5, 768 -> 67.6, 1024 -> 65.4, 1536 -> 75.4;
    // n = 8192: 256 -> 14.7 ms, 512 -> 17.1. (With one launch per block column it was the other way round,
    // profiles/r01_nb_sweep.log: 512 -> 76.7, 1024 -> 67.3.)
    const i64 nbl = lookahead_block() ? lookahead_block() : 256;
    return dist_llt_f64(A.ptr, A.cs, n, nbl, reg_delta, reg_eps, /*lookahead | local*/ 3);
  }
  return llt_recursive_in_place<double>(stream, A, reg_delta, reg_eps, params);
}

// f32: the same leaf kernel and recursive driver instantiated for float (trailing updates on the 3xTF32 GEMM — tcgen05 for large
// products —, panel solves on the f32 triangular solve). The look-ahead block-column drivers (dist.cu) are f64-only.
LltResult llt_cholesky_in_place_f32(cudaStream_t stream, VF A, float reg_delta, float reg_eps, LltParams params) {
  FB_ASSERT(A.nrows == A.ncols, "LLT needs a square matrix");
  if (A.nrows == 0) return LltResult{true, 0, 0};
  return llt_recursive_in_place<float>(stream, A, reg_delta, reg_eps, params);
}

}  // namespace fb
