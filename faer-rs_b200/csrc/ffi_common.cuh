// Helpers shared by the translation units of the extern "C" boundary (ffi.cu, ffi_types.cu): staging of matrix arguments, scalar /
// permutation / vector arguments that may live on the host or on the device, the status PODs, and the end-of-call sequence of the
// staged matrices. Host code only: ffi_types.cu, and with it this header, also builds with g++ for the host (tools/emul).
#pragma once
#include "../../include/faer_b200.h"
#include "runtime.cuh"

#include <cstdint>
#include <cstring>
#include <initializer_list>
#include <vector>

namespace fb {
// (static, not an anonymous namespace: nvcc's kernel stubs of a unit that also has a global anonymous namespace must stay unambiguous)

// bytes of one T-typed element of the scalar kind <R, complex?>
template <class R, bool CX>
constexpr size_t elem_bytes() { return (CX ? 2 : 1) * sizeof(R); }

// matrix arguments: an input view (copied in, never back) and an output view (copied back; copied in only if its old contents matter)
static inline StagedMat stage(FaerV0_24_MatRef m, size_t elem, cudaStream_t st) {
  return StagedMat(m.ptr, (i64)m.nrows, (i64)m.ncols, (i64)m.row_stride, (i64)m.col_stride, elem, true, false, st);
}
static inline StagedMat stage(FaerV0_24_MatMut m, size_t elem, bool copy_in, cudaStream_t st) {
  return StagedMat(m.ptr, (i64)m.nrows, (i64)m.ncols, (i64)m.row_stride, (i64)m.col_stride, elem, copy_in, true, st);
}

static inline void finish_all(cudaStream_t st, std::initializer_list<StagedMat*> mats) {
  // the compute must be complete before input mirrors return to the pool; calls are synchronous anyway
  FB_CUDA_CHECK(cudaStreamSynchronize(st));
  for (auto* m : mats) m->finish();
}

// `count` consecutive R values behind a scalar argument (host or device): 1 for a real value, 2 for a complex one
template <class R>
static inline void read_scalar(const void* p, R* v, int count) {
  FB_ASSERT(p != nullptr, "null scalar pointer");
  if (is_device_pointer(p)) FB_CUDA_CHECK(cudaMemcpy(v, p, count * sizeof(R), cudaMemcpyDeviceToHost));
  else memcpy(v, p, count * sizeof(R));
}
template <class R>
static inline R read_real(const void* p) {
  R v;
  read_scalar(p, &v, 1);
  return v;
}

// dynamic regularisation of LLT / LDLT: delta and epsilon are T::Real, a null pointer means 0
template <class R, class Reg>
static inline void read_regularization(const Reg& reg, R& delta, R& eps) {
  delta = reg.dynamic_regularization_delta ? read_real<R>(reg.dynamic_regularization_delta) : R(0);
  eps = reg.dynamic_regularization_epsilon ? read_real<R>(reg.dynamic_regularization_epsilon) : R(0);
}

// ---- status PODs (tagged unions: zero the padding and the unused body) ----
static inline FaerV0_24_LltStatus llt_status(const LltResult& r) {
  FaerV0_24_LltStatus out;
  memset(&out, 0, sizeof(out));
  if (r.ok) {
    out.tag = FaerV0_24_LltStatus_Ok;
    out.ok.dynamic_regularization_count = r.dynamic_regularization_count;
  } else {
    out.tag = FaerV0_24_LltStatus_NonPositivePivot;
    out.non_positive_pivot.index = r.non_positive_pivot_index;
  }
  return out;
}
static inline FaerV0_24_LdltStatus ldlt_status(const LdltResult& r) {
  FaerV0_24_LdltStatus out;
  memset(&out, 0, sizeof(out));
  if (r.ok) {
    out.tag = FaerV0_24_LdltStatus_Ok;
    out.ok.dynamic_regularization_count = r.dynamic_regularization_count;
  } else {
    out.tag = FaerV0_24_LdltStatus_ZeroPivot;
    out.zero_pivot.index = r.zero_pivot_index;
  }
  return out;
}
static inline FaerV0_24_PartialPivLuStatus lu_status(size_t transposition_count) {
  FaerV0_24_PartialPivLuStatus out;
  memset(&out, 0, sizeof(out));
  out.tag = FaerV0_24_PartialPivLuStatus_Ok;
  out.ok.transposition_count = transposition_count;
  return out;
}
static inline FaerV0_24_QrStatus qr_status(bool known, size_t rank) {
  FaerV0_24_QrStatus out;
  memset(&out, 0, sizeof(out));
  if (known) {
    out.tag = FaerV0_24_QrStatus_Ok;
    out.ok.rank = rank;
  } else {
    out.tag = FaerV0_24_QrStatus_Unknown;
  }
  return out;
}
static inline FaerV0_24_SvdStatus svd_status(bool ok) {
  FaerV0_24_SvdStatus out;
  memset(&out, 0, sizeof(out));
  out.tag = ok ? FaerV0_24_SvdStatus_Ok : FaerV0_24_SvdStatus_NoConvergence;
  return out;
}
static inline FaerV0_24_EvdStatus evd_status(bool ok) {
  FaerV0_24_EvdStatus out;
  memset(&out, 0, sizeof(out));
  out.tag = ok ? FaerV0_24_EvdStatus_Ok : FaerV0_24_EvdStatus_NoConvergence;
  return out;
}

// ---- index slices (u32 / u64) <-> host int64 ----
// NB: faer.hpp fills SliceMut.len with BYTES while the Rust side reads elements (SURVEY.md appendix A), so callers pass the
// permutation length from a matrix dimension, never from `len`. Every entry must be a row index of that dimension.
static inline std::vector<long long> read_perm_checked(FaerV0_24_SliceRef slice, size_t n, int idx_bytes) {
  std::vector<unsigned char> raw(n * (size_t)idx_bytes);
  if (n) {
    if (is_device_pointer(slice.ptr)) FB_CUDA_CHECK(cudaMemcpy(raw.data(), slice.ptr, raw.size(), cudaMemcpyDeviceToHost));
    else memcpy(raw.data(), slice.ptr, raw.size());
  }
  std::vector<long long> out(n);
  for (size_t i = 0; i < n; ++i) {
    out[i] = idx_bytes == 4 ? (long long)((const uint32_t*)raw.data())[i] : (long long)((const uint64_t*)raw.data())[i];
    FB_ASSERT(out[i] >= 0 && (size_t)out[i] < n, "invalid permutation entry");
  }
  return out;
}
static inline void write_perm(void* dst, const std::vector<long long>& v, int idx_bytes) {
  if (v.empty()) return;
  std::vector<unsigned char> buf(v.size() * (size_t)idx_bytes);
  for (size_t i = 0; i < v.size(); ++i) {
    if (idx_bytes == 4) ((uint32_t*)buf.data())[i] = (uint32_t)v[i];
    else ((uint64_t*)buf.data())[i] = (uint64_t)v[i];
  }
  if (is_device_pointer(dst)) FB_CUDA_CHECK(cudaMemcpy(dst, buf.data(), buf.size(), cudaMemcpyHostToDevice));
  else memcpy(dst, buf.data(), buf.size());
}

// ---- LDLT arguments ----
// expected pivot signs: i8 slice, null = none (faer-ffi/src/lib.rs:838-848); a device slice is used in place, a host slice is
// mirrored on the device
struct SignsArg {
  const signed char* ptr = nullptr;
  signed char* mirror = nullptr;
  SignsArg(FaerV0_24_SliceMut sg, size_t n, cudaStream_t st) {
    if (sg.ptr == nullptr || n == 0) return;
    FB_ASSERT(sg.len >= n, "dynamic_regularization_signs is shorter than the matrix dimension");
    if (is_device_pointer(sg.ptr)) {
      ptr = (const signed char*)sg.ptr;
    } else {
      mirror = (signed char*)ws_alloc(n);
      FB_CUDA_CHECK(cudaMemcpyAsync(mirror, sg.ptr, n, cudaMemcpyHostToDevice, st));
      ptr = mirror;
    }
  }
  ~SignsArg() {
    if (mirror) ws_free(mirror);
  }
  SignsArg(const SignsArg&) = delete;
  SignsArg& operator=(const SignsArg&) = delete;
};
// D, a VecRef of T-typed entries: a device vector is used in place, a host vector is gathered into a compact device copy
template <class R, bool CX>
struct DiagArg {
  const R* ptr;
  i64 stride;
  R* mirror = nullptr;
  DiagArg(FaerV0_24_VecRef D, size_t n, cudaStream_t st) {
    const size_t w = CX ? 2 : 1;
    ptr = (const R*)D.ptr;
    stride = (i64)D.stride;
    if (n > 0 && !is_device_pointer(D.ptr)) {
      std::vector<R> h(n * w);
      for (size_t i = 0; i < n; ++i)
        for (size_t c = 0; c < w; ++c) h[i * w + c] = ((const R*)D.ptr)[((ptrdiff_t)i * D.stride) * (ptrdiff_t)w + (ptrdiff_t)c];
      mirror = (R*)ws_alloc(n * w * sizeof(R));
      FB_CUDA_CHECK(cudaMemcpyAsync(mirror, h.data(), n * w * sizeof(R), cudaMemcpyHostToDevice, st));
      FB_CUDA_CHECK(cudaStreamSynchronize(st));  // `h` is pageable and local
      ptr = mirror;
      stride = 1;
    }
  }
  ~DiagArg() {
    if (mirror) ws_free(mirror);
  }
  DiagArg(const DiagArg&) = delete;
  DiagArg& operator=(const DiagArg&) = delete;
};

// S[i * S.stride] <- s_dev[i] for i < n (elem-byte entries; S on the host or the device), enqueued on st
static inline void copy_out_vector(FaerV0_24_VecMut S, const void* s_dev, size_t n, size_t elem, cudaStream_t st) {
  FB_CUDA_CHECK(cudaMemcpy2DAsync(S.ptr, (size_t)S.stride * elem, s_dev, elem, elem, n, cudaMemcpyDefault, st));
}

}  // namespace fb
