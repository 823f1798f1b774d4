// Host-side dispatch: maps the run-time codes of the C-ABI (dtype, op, flags, vector width) to template arguments,
// and reads the RUA_* measurement knobs (DESIGN.md section 3).  Every launcher goes through these helpers, so a new
// dtype, op or word type is added here once.  The lambdas run on the host only; they launch kernels and return a status.
#pragma once

#include <cstdlib>
#include <type_traits>

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace rua {

template <typename T> struct Type { using type = T; };
template <int N> using Int = std::integral_constant<int, N>;

// f(Type<T>{}) for the storage type of `dtype`; `bad` for a code that names no dtype
template <typename F> inline int with_dtype(int32_t dtype, F&& f, int bad = RUA_ERR_UNSUPPORTED) {
  switch (dtype) {
    case RUA_F32: return f(Type<float>{});
    case RUA_F64: return f(Type<double>{});
    case RUA_F16: return f(Type<__half>{});
    case RUA_BF16: return f(Type<__nv_bfloat16>{});
    default: return bad;
  }
}

// f(Int<OP>{}) for a segment-reduce op code; `bad` for a code that names no op
template <typename F> inline int with_op(int32_t op, F&& f, int bad = RUA_ERR_INVALID) {
  switch (op) {
    case RUA_SUM: return f(Int<RUA_SUM>{});
    case RUA_MEAN: return f(Int<RUA_MEAN>{});
    case RUA_PROD: return f(Int<RUA_PROD>{});
    case RUA_MAX: return f(Int<RUA_MAX>{});
    case RUA_MIN: return f(Int<RUA_MIN>{});
    case RUA_LOGSUMEXP: return f(Int<RUA_LOGSUMEXP>{});
    default: return bad;
  }
}

// f(Int<HE>{}) for a narrow row of HE in {1, 2, 4, 8} elements that fits one 16-byte vector of T
template <typename T, typename F> inline int with_row_elems(int64_t he, F&& f) {
  constexpr int E = 16 / sizeof(T);
  switch (he) {
    case 1: return f(Int<1>{});
    case 2: if constexpr (E >= 2) return f(Int<2>{}); break;
    case 4: if constexpr (E >= 4) return f(Int<4>{}); break;
    case 8: if constexpr (E >= 8) return f(Int<8>{}); break;
  }
  return RUA_ERR_UNSUPPORTED;
}

template <typename F> inline decltype(auto) with_bool(bool b, F&& f) {
  return b ? f(std::true_type{}) : f(std::false_type{});
}

// 32-byte word of the 256-bit global accesses (sm_100: LDG.E.ENL2.256 / STG.E.ENL2.256)
struct alignas(32) V256 {
  unsigned long long x, y, z, w;
};

// f(Type<W>{}) for the row-map word of `bytes` bytes (32, 16, 8, 4, 2; anything else: 1)
template <typename F> inline decltype(auto) with_word(int bytes, F&& f) {
  switch (bytes) {
    case 32: return f(Type<V256>{});
    case 16: return f(Type<uint4>{});
    case 8: return f(Type<uint2>{});
    case 4: return f(Type<unsigned int>{});
    case 2: return f(Type<unsigned short>{});
    default: return f(Type<unsigned char>{});
  }
}

// elements per 16-byte vector (Store<T>::kVec) and accumulator bytes (sizeof(Store<T>::Acc)) of a valid dtype
constexpr int vec_elems(int32_t dtype) { return dtype == RUA_F32 ? 4 : (dtype == RUA_F64 ? 2 : 8); }
constexpr size_t acc_bytes(int32_t dtype) { return dtype == RUA_F64 ? 8 : 4; }

// an integer environment variable, or `dflt` when it is not set; callers keep the value in a function-local static,
// so each knob is read once per process
inline int64_t knob(const char* name, int64_t dflt) {
  const char* e = getenv(name);
  return e ? (int64_t)atoll(e) : dflt;
}

// enough short segments to fill the machine with warps of 32 segments each?  Decides for the warp-per-32-segments
// kernels of the segment reductions, rua_emit_ptr and the narrow L/R -> C, rev and roll row maps alike.
inline bool warpseg_applies(int64_t N, int64_t S) {
  static const int64_t min_s = knob("RUA_WARPSEG_MIN_S", 32768);
  static const int64_t max_avg = knob("RUA_WARPSEG_MAX_AVG", 256);
  return S >= min_s && N <= max_avg * S;
}

}  // namespace rua
