// Shared numeric helpers of the segment-reduce kernels (forward: reduce.cu, backward: reduce_bwd.cu).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <math_constants.h>

#include "common.cuh"
#include "dispatch.cuh"

namespace rua {

constexpr int kRedThreads = 128;
constexpr int kRedUnroll = 8;

// ---------------------------------------------------------------------------------------------
// storage <-> accumulator conversion, 16-byte vectors
// ---------------------------------------------------------------------------------------------
template <typename T> struct Store;
template <> struct Store<float> {
  using Acc = float;
  static constexpr int kVec = 4;
  static constexpr int kMinBlocks = 6;  // CTAs of 128 threads per SM the main kernel is compiled for (<= 85 regs)
  __device__ static void unpack(const uint4& r, Acc* x) {
    x[0] = __uint_as_float(r.x); x[1] = __uint_as_float(r.y); x[2] = __uint_as_float(r.z); x[3] = __uint_as_float(r.w);
  }
  __device__ static uint4 pack(const Acc* x) {
    return make_uint4(__float_as_uint(x[0]), __float_as_uint(x[1]), __float_as_uint(x[2]), __float_as_uint(x[3]));
  }
  __device__ static Acc to_acc(float v) { return v; }
  __device__ static float from_acc(Acc v) { return v; }
};
template <> struct Store<double> {
  using Acc = double;
  static constexpr int kVec = 2;
  static constexpr int kMinBlocks = 4;
  __device__ static void unpack(const uint4& r, Acc* x) {
    x[0] = __hiloint2double((int)r.y, (int)r.x);
    x[1] = __hiloint2double((int)r.w, (int)r.z);
  }
  __device__ static uint4 pack(const Acc* x) {
    return make_uint4((uint32_t)__double2loint(x[0]), (uint32_t)__double2hiint(x[0]),
                      (uint32_t)__double2loint(x[1]), (uint32_t)__double2hiint(x[1]));
  }
  __device__ static Acc to_acc(double v) { return v; }
  __device__ static double from_acc(Acc v) { return v; }
};
template <> struct Store<__half> {
  using Acc = float;
  static constexpr int kVec = 8;
  static constexpr int kMinBlocks = 4;  // half2 -> float2 unpacking needs more registers than the bf16 shift
  __device__ static void unpack(const uint4& r, Acc* x) {
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[k]));
      x[2 * k] = f.x; x[2 * k + 1] = f.y;
    }
  }
  __device__ static uint4 pack(const Acc* x) {
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      __half2 h = __floats2half2_rn(x[2 * k], x[2 * k + 1]);
      w[k] = *reinterpret_cast<uint32_t*>(&h);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
  }
  __device__ static Acc to_acc(__half v) { return __half2float(v); }
  __device__ static __half from_acc(Acc v) { return __float2half_rn(v); }
};
template <> struct Store<__nv_bfloat16> {
  using Acc = float;
  static constexpr int kVec = 8;
  static constexpr int kMinBlocks = 6;
  __device__ static void unpack(const uint4& r, Acc* x) {
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {  // bf16 -> fp32 is a 16-bit shift
      x[2 * k] = __uint_as_float(w[k] << 16);
      x[2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u);
    }
  }
  __device__ static uint4 pack(const Acc* x) {
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      __nv_bfloat162 h = __floats2bfloat162_rn(x[2 * k], x[2 * k + 1]);
      w[k] = *reinterpret_cast<uint32_t*>(&h);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
  }
  __device__ static Acc to_acc(__nv_bfloat16 v) { return __bfloat162float(v); }
  __device__ static __nv_bfloat16 from_acc(Acc v) { return __float2bfloat16_rn(v); }
};

template <int32_t D, typename T> constexpr bool store_matches() {
  return vec_elems(D) == Store<T>::kVec && acc_bytes(D) == sizeof(typename Store<T>::Acc) && Store<T>::kVec * sizeof(T) == 16;
}
static_assert(store_matches<RUA_F32, float>() && store_matches<RUA_F64, double>() && store_matches<RUA_F16, __half>() &&
              store_matches<RUA_BF16, __nv_bfloat16>(), "vec_elems / acc_bytes (dispatch.cuh) disagree with Store<T>");

// ---------------------------------------------------------------------------------------------
// scalar math on the accumulator type
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float max_nan(float a, float b) {  // NaN-propagating, like ATen's segment max
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float min_nan(float a, float b) {
  float r;
  asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ double max_nan(double a, double b) { return (a != a) ? a : ((b != b) ? b : (a < b ? b : a)); }
__device__ __forceinline__ double min_nan(double a, double b) { return (a != a) ? a : ((b != b) ? b : (b < a ? b : a)); }
__device__ __forceinline__ float min_num(float a, float b) { return fminf(a, b); }    // ignores NaN
__device__ __forceinline__ float max_num(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ double min_num(double a, double b) { return fmin(a, b); }
__device__ __forceinline__ double max_num(double a, double b) { return fmax(a, b); }
template <typename A> __device__ __forceinline__ A inf_of();
template <> __device__ __forceinline__ float inf_of<float>() { return CUDART_INF_F; }
template <> __device__ __forceinline__ double inf_of<double>() { return CUDART_INF; }
template <typename A> __device__ __forceinline__ A nan_of();
template <> __device__ __forceinline__ float nan_of<float>() { return CUDART_NAN_F; }
template <> __device__ __forceinline__ double nan_of<double>() { return CUDART_NAN; }
__device__ __forceinline__ float ex2_approx(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float lg2_approx(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// kFast (16-bit storage, 1e-2 contract): one FMUL + one MUFU.  (__expf / __logf are the non-ftz forms: they wrap the
// MUFU in a denormal range check and two rescaling multiplies -- 4-5 instructions per call, which the per-row update
// of short-segment logsumexp pays per element.)
template <bool kFast> __device__ __forceinline__ float exp_acc(float x) {
  return kFast ? ex2_approx(x * 1.4426950408889634f) : expf(x);
}
template <bool kFast> __device__ __forceinline__ double exp_acc(double x) { return exp(x); }
template <bool kFast = false> __device__ __forceinline__ float log_acc(float x) {
  return kFast ? lg2_approx(x) * 0.6931471805599453f : logf(x);
}
template <bool kFast = false> __device__ __forceinline__ double log_acc(double x) { return log(x); }
__device__ __forceinline__ float abs_acc(float x) { return fabsf(x); }
__device__ __forceinline__ double abs_acc(double x) { return fabs(x); }

// order-preserving integer keys so the global extreme can be reduced with integer atomics
__device__ __forceinline__ unsigned long long order_key(float f) {
  uint32_t b = __float_as_uint(f);
  return (unsigned long long)((b & 0x80000000u) ? ~b : (b | 0x80000000u));
}
__device__ __forceinline__ unsigned long long order_key(double d) {
  unsigned long long b = (unsigned long long)__double_as_longlong(d);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ float key_to(float, unsigned long long k) {
  uint32_t b = (uint32_t)k;
  return __uint_as_float((b & 0x80000000u) ? (b & 0x7fffffffu) : ~b);
}
__device__ __forceinline__ double key_to(double, unsigned long long k) {
  return __longlong_as_double((long long)((k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k));
}

// raw (unconverted) register image of V storage elements: keeps the 8-deep load pipeline at 4
// registers per row instead of V accumulator-typed ones
template <typename T, int V> struct Raw { uint4 r; };
template <typename T> struct Raw<T, 1> { T r; };
template <typename T, int V>
__device__ __forceinline__ void load_raw(const T* p, Raw<T, V>& w) {
  if constexpr (V == 1) w.r = *p;
  else w.r = __ldcs(reinterpret_cast<const uint4*>(p));
}
template <typename T, int V>
__device__ __forceinline__ void unpack_raw(const Raw<T, V>& w, typename Store<T>::Acc* x) {
  if constexpr (V == 1) x[0] = Store<T>::to_acc(w.r);
  else Store<T>::unpack(w.r, x);
}
template <typename T, int V>
__device__ __forceinline__ void store_vec(T* p, const typename Store<T>::Acc* x) {
  if constexpr (V == 1) *p = Store<T>::from_acc(x[0]);
  else *reinterpret_cast<uint4*>(p) = Store<T>::pack(x);
}

// ---------------------------------------------------------------------------------------------
// packed 16-bit pairs: max / min are exact in the storage format, so they can run two-at-a-time
// (HMNMX2) on the raw words without unpacking to fp32
// ---------------------------------------------------------------------------------------------
template <typename T> struct Pk {
  static constexpr bool kHas = false;
  static constexpr uint32_t kPosInf = 0u;
};
template <> struct Pk<__nv_bfloat16> {
  static constexpr bool kHas = true;
  static constexpr uint32_t kPosInf = 0x7F807F80u;
  __device__ static __forceinline__ uint32_t max_nan(uint32_t a, uint32_t b) {
    __nv_bfloat162 r = __hmax2_nan(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
    return *reinterpret_cast<uint32_t*>(&r);
  }
  __device__ static __forceinline__ uint32_t min_num(uint32_t a, uint32_t b) {
    __nv_bfloat162 r = __hmin2(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
    return *reinterpret_cast<uint32_t*>(&r);
  }
  __device__ static __forceinline__ void unpack(uint32_t w, float& lo, float& hi) {
    lo = __uint_as_float(w << 16);
    hi = __uint_as_float(w & 0xffff0000u);
  }
};
template <> struct Pk<__half> {
  static constexpr bool kHas = true;
  static constexpr uint32_t kPosInf = 0x7C007C00u;
  __device__ static __forceinline__ uint32_t max_nan(uint32_t a, uint32_t b) {
    __half2 r = __hmax2_nan(*reinterpret_cast<__half2*>(&a), *reinterpret_cast<__half2*>(&b));
    return *reinterpret_cast<uint32_t*>(&r);
  }
  __device__ static __forceinline__ uint32_t min_num(uint32_t a, uint32_t b) {
    __half2 r = __hmin2(*reinterpret_cast<__half2*>(&a), *reinterpret_cast<__half2*>(&b));
    return *reinterpret_cast<uint32_t*>(&r);
  }
  __device__ static __forceinline__ void unpack(uint32_t w, float& lo, float& hi) {
    float2 f = __half22float2(*reinterpret_cast<__half2*>(&w));
    lo = f.x;
    hi = f.y;
  }
};

__device__ __forceinline__ uint32_t word_of(const uint4& w, int j) {
  return j == 0 ? w.x : (j == 1 ? w.y : (j == 2 ? w.z : w.w));
}

template <typename T, int V>
__device__ __forceinline__ typename Store<T>::Acc packed_min_to_acc(const uint32_t* ext2) {
  using A = typename Store<T>::Acc;
  A m = inf_of<A>();
  if constexpr (Pk<T>::kHas && V == 8) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float lo, hi;
      Pk<T>::unpack(ext2[j], lo, hi);
      m = min_num(m, min_num(lo, hi));
    }
  }
  return m;
}


// logsumexp over kRows rows that all belong to the current segment: a[] = running max, s[] = running
// sum of exp(x - a).  One EX2 per element (plus one per column for the rescale).
template <typename T, int V, int kRows>
__device__ __forceinline__ void lse_batch(const Raw<T, V>* raw, typename Store<T>::Acc* a, typename Store<T>::Acc* s,
                                          typename Store<T>::Acc& ext, uint32_t* ext2) {
  using A = typename Store<T>::Acc;
  A bm[V];
  if constexpr (Pk<T>::kHas && V == 8) {
    uint32_t m2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) m2[j] = word_of(raw[0].r, j);
#pragma unroll
    for (int k = 0; k < kRows; ++k) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t w = word_of(raw[k].r, j);
        if (k > 0) m2[j] = Pk<T>::max_nan(m2[j], w);
        ext2[j] = Pk<T>::min_num(ext2[j], w);
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) Pk<T>::unpack(m2[j], bm[2 * j], bm[2 * j + 1]);
  } else {
#pragma unroll
    for (int v = 0; v < V; ++v) bm[v] = -inf_of<A>();
#pragma unroll
    for (int k = 0; k < kRows; ++k) {
      A x[V];
      unpack_raw<T, V>(raw[k], x);
#pragma unroll
      for (int v = 0; v < V; ++v) {
        bm[v] = max_nan(bm[v], x[v]);
        ext = min_num(ext, x[v]);
      }
    }
  }
  // (tried in round 2: exponent arguments formed and exponentiated as PACKED bf16 pairs -- fma.rn.bf16x2 +
  // ex2.approx.ftz.bf16x2.  On sm_100a the packed ex2 is NOT one MUFU: SASS shows two MUFU.EX2.BF16 + PRMT + FMUL per
  // pair, 9 instructions per pair against 8 for the fp32 form below, and cfg3 logsumexp went 84.6 % -> 82.8 % of peak
  // while losing accuracy.  Dropped; profiles/r2_ncu_lse.md has the instruction mix.)
  if constexpr (sizeof(A) == 4) {
    constexpr float kLog2e = 1.4426950408889634f;
    float mb[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
      float m_new = max_nan(a[v], bm[v]);
      s[v] = s[v] == 0.f ? 0.f : s[v] * ex2_approx((a[v] - m_new) * kLog2e);
      a[v] = m_new;
      mb[v] = m_new == -inf_of<A>() ? 0.f : m_new * kLog2e;   // all -inf so far: each adds ex2(-inf) = 0, not ex2(NaN)
    }
#pragma unroll
    for (int k = 0; k < kRows; ++k) {
      A x[V];
      unpack_raw<T, V>(raw[k], x);
#pragma unroll
      for (int v = 0; v < V; ++v) s[v] += ex2_approx(fmaf(x[v], kLog2e, -mb[v]));
    }
  } else {
#pragma unroll
    for (int v = 0; v < V; ++v) {
      A m_new = max_nan(a[v], bm[v]);
      s[v] = s[v] == A(0) ? A(0) : s[v] * exp(a[v] - m_new);
      a[v] = m_new;
    }
#pragma unroll
    for (int k = 0; k < kRows; ++k) {
      A x[V];
      unpack_raw<T, V>(raw[k], x);
#pragma unroll
      for (int v = 0; v < V; ++v) s[v] += exp(x[v] - (a[v] == -inf_of<A>() ? A(0) : a[v]));
    }
  }
}


// ---------------------------------------------------------------------------------------------
// per-op accumulator state shared by the wide-row kernel (reduce.cu) and the flat kernel (reduce_flat.cu)
// ---------------------------------------------------------------------------------------------
struct RedHeader {            // first 64 bytes of the workspace
  unsigned long long ext_key; // global min (max / logsumexp) or global max (min), as an order key
  unsigned int nan_flag;      // a NaN reached an output of max / min / logsumexp
  unsigned int pad[13];
};

template <int OP> struct OpInfo {
  static constexpr bool kIsLse = OP == RUA_LOGSUMEXP;
  static constexpr bool kNeedsExt = OP == RUA_MAX || OP == RUA_MIN || OP == RUA_LOGSUMEXP;
  static constexpr int kParts = kIsLse ? 2 : 1;  // accumulator planes (lse keeps max and sum)
};

// accumulator state for V columns
template <typename A, int V, int OP>
struct State {
  A a[V];   // sum / prod / max / min, or the running max for logsumexp
  A s[OpInfo<OP>::kIsLse ? V : 1];

  __device__ __forceinline__ void reset() {
#pragma unroll
    for (int v = 0; v < V; ++v) {
      if (OP == RUA_SUM || OP == RUA_MEAN) a[v] = A(0);
      else if (OP == RUA_PROD) a[v] = A(1);
      else if (OP == RUA_MIN) a[v] = inf_of<A>();
      else a[v] = -inf_of<A>();
      if (OpInfo<OP>::kIsLse) s[v] = A(0);
    }
  }
  template <bool kFast>
  __device__ __forceinline__ void add(const A* x) {
#pragma unroll
    for (int v = 0; v < V; ++v) {
      if (OP == RUA_SUM || OP == RUA_MEAN) a[v] += x[v];
      else if (OP == RUA_PROD) a[v] *= x[v];
      else if (OP == RUA_MAX) a[v] = max_nan(a[v], x[v]);
      else if (OP == RUA_MIN) a[v] = min_nan(a[v], x[v]);
      else {  // online logsumexp: one exp per element.  A -inf element adds 0, also while the running max is still -inf
              // (-inf - -inf = NaN, clamped to 0 by the fmax); a NaN element still poisons the result through a
        A d = x[v] - a[v];
        A e = exp_acc<kFast>(-abs_acc(d));
        s[v] = d > A(0) ? s[v] * e + A(1) : s[v] + fmax(e, A(0));
        a[v] = max_nan(a[v], x[v]);
      }
    }
  }
  // merge a later piece (b) into this earlier piece, in order
  template <bool kFast>
  __device__ __forceinline__ void merge(const State& b) {
#pragma unroll
    for (int v = 0; v < V; ++v) {
      if (OP == RUA_SUM || OP == RUA_MEAN) a[v] += b.a[v];
      else if (OP == RUA_PROD) a[v] *= b.a[v];
      else if (OP == RUA_MAX) a[v] = max_nan(a[v], b.a[v]);
      else if (OP == RUA_MIN) a[v] = min_nan(a[v], b.a[v]);
      else {
        A m = max_nan(a[v], b.a[v]);
        A s1 = s[v] == A(0) ? A(0) : s[v] * exp_acc<kFast>(a[v] - m);
        A s2 = b.s[v] == A(0) ? A(0) : b.s[v] * exp_acc<kFast>(b.a[v] - m);
        s[v] = s1 + s2;
        a[v] = m;
      }
    }
  }
  // kFast (16-bit storage): lg2.approx instead of the ~25-instruction logf -- with segments of a few rows the logarithm
  // of every OUTPUT element was a third of all instructions of the kernel
  template <bool kFast = false>
  __device__ __forceinline__ void finalize(int64_t len, A* out) const {
#pragma unroll
    for (int v = 0; v < V; ++v) {
      if (OP == RUA_MEAN) out[v] = (a[v] != a[v]) ? a[v] : a[v] / (A)len;
      else if (OP == RUA_LOGSUMEXP) out[v] = log_acc<kFast>(s[v]) + a[v];
      else out[v] = a[v];
    }
  }
  // 16-bit storage, very short segments: one reciprocal per segment instead of a division per element (the result is
  // rounded to 8 / 11 mantissa bits afterwards; the 1e-2 contract of DESIGN.md section 4 has four decimal digits to spare)
  __device__ __forceinline__ void finalize_recip(int64_t len, A* out) const {
    if (OP == RUA_MEAN) {
      const A inv = A(1) / (A)len;
#pragma unroll
      for (int v = 0; v < V; ++v) out[v] = a[v] * inv;
    } else {
      finalize<true>(len, out);
    }
  }
  __device__ __forceinline__ bool any_nan_out(const A* out) const {
    bool n = false;
#pragma unroll
    for (int v = 0; v < V; ++v) n |= (out[v] != out[v]);
    return n;
  }
};

template <typename A, int V, int OP>
__device__ __forceinline__ void store_partial(A* base, int64_t H, int64_t col, const State<A, V, OP>& st) {
#pragma unroll
  for (int v = 0; v < V; ++v) {
    base[col + v] = st.a[v];
    if (OpInfo<OP>::kIsLse) base[H + col + v] = st.s[v];
  }
}
template <typename A, int V, int OP>
__device__ __forceinline__ void load_partial(const A* base, int64_t H, int64_t col, State<A, V, OP>& st) {
#pragma unroll
  for (int v = 0; v < V; ++v) {
    st.a[v] = base[col + v];
    if (OpInfo<OP>::kIsLse) st.s[v] = base[H + col + v];
  }
}

// ---------------------------------------------------------------------------------------------
// host launchers defined in one translation unit and called from another (reduce.cu, reduce_bwd.cu)
// ---------------------------------------------------------------------------------------------
// narrow rows (H * elem <= 16 bytes) run on the rows-on-lanes kernels of reduce_flat.cu
bool flat_supported(int32_t dtype, int64_t H);
int flat_rows_per_tile(int32_t dtype, int64_t H);
int flat_launch(int32_t dtype, int64_t H, int32_t op, const void* data, const int64_t* ridx, const int64_t* off,
                int64_t N, int64_t S, void* out, void* head, void* tail, int64_t* tail_seg, void* hdr,
                int vector_loads, int64_t tiles, cudaStream_t st);
// ... or, with many short segments (warpseg_applies), on the warp-per-32-segments kernels of reduce_warpseg.cu and
// reduce_warpseg_bwd.cu
int warpseg_launch(int32_t dtype, int64_t H, int32_t op, const void* data, const int64_t* off, int64_t N, int64_t S,
                   void* out, void* hdr, cudaStream_t st);
int warpseg_bwd_launch(int32_t dtype, int64_t H, int32_t op, const void* gout, const void* out, const void* data,
                       const int64_t* off, int64_t N, int64_t S, void* grad, cudaStream_t st);
// ... and wide rows in very short segments on the SHORT instance of the main kernel (reduce_short.cu)
bool short_applies(int64_t N, int64_t S, int32_t op);
int short_launch(int32_t dtype, int32_t op, bool gather, bool packed, dim3 grid, int threads, const void* data,
                 const int64_t* ridx, const int64_t* off, int64_t N, int64_t S, int64_t H, int R, void* out, void* head,
                 void* tail, int64_t* tail_seg, void* hdr, int lanes_log2, int64_t chunks, cudaStream_t st);

}  // namespace rua
