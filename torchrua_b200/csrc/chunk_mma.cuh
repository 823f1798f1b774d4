// Warp-tile matrix products over shared memory for the chunked scans (K11 SSD, K12 gated delta rule): m16n8 accumulator
// fragments, mma.sync m16n8k16 with fp32 accumulation for fp16 / bf16 and FMA over the same fragment ownership for
// fp32 / fp64, plus the exponential and the fragment row / column sums both kernels use.
#pragma once

#include "reduce_common.cuh"

namespace rua {

// exponential of the scaled argument: ex2.approx for fp32 (cum is kept in units of log2 e), exp for fp64
__device__ __forceinline__ float ex(float v) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}
__device__ __forceinline__ double ex(double v) { return exp(v); }
template <typename A> __host__ __device__ constexpr A exp_scale() { return sizeof(A) == 4 ? A(1.4426950408889634) : A(1); }
__device__ __forceinline__ float quiet_nan(float) { return __int_as_float(0x7fc00000); }
__device__ __forceinline__ double quiet_nan(double) { return __longlong_as_double(0x7ff8000000000000ll); }

// shared matrix view: element (r, c) at p[r * rs + c * cs]
template <typename T> struct Sm {
  const T* p;
  int rs, cs;
  __device__ __forceinline__ T operator()(int r, int c) const { return p[r * rs + c * cs]; }
};

__device__ __forceinline__ uint32_t pack2(__half lo, __half hi) {
  return (uint32_t)__half_as_ushort(lo) | ((uint32_t)__half_as_ushort(hi) << 16);
}
__device__ __forceinline__ uint32_t pack2(__nv_bfloat16 lo, __nv_bfloat16 hi) {
  return (uint32_t)__bfloat16_as_ushort(lo) | ((uint32_t)__bfloat16_as_ushort(hi) << 16);
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2], __half) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2], __nv_bfloat16) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// fragment element e of the m16n8 accumulator: row gr (+8 for e >= 2), column 2 tg + (e & 1)
__device__ __forceinline__ int frow(int e, int lane) { return (lane >> 2) + (e >= 2 ? 8 : 0); }
__device__ __forceinline__ int fcol(int e, int lane) { return 2 * (lane & 3) + (e & 1); }

// c += A[m0 .. m0 + 16, 0 .. K) B[0 .. K, n0 .. n0 + 8), K a multiple of 16; the one dtype-specific piece
template <typename T, typename Acc>
__device__ __forceinline__ void tile_mma(Acc (&c)[4], Sm<T> a, Sm<T> b, int m0, int n0, int K, int lane) {
  const int gr = lane >> 2, tg = lane & 3;
  if constexpr (sizeof(T) == 2) {
#pragma unroll 4
    for (int k0 = 0; k0 < K; k0 += 16) {
      const int k = k0 + 2 * tg;
      const uint32_t af[4] = {pack2(a(m0 + gr, k), a(m0 + gr, k + 1)), pack2(a(m0 + gr + 8, k), a(m0 + gr + 8, k + 1)),
                              pack2(a(m0 + gr, k + 8), a(m0 + gr, k + 9)),
                              pack2(a(m0 + gr + 8, k + 8), a(m0 + gr + 8, k + 9))};
      const uint32_t bf[2] = {pack2(b(k, n0 + gr), b(k + 1, n0 + gr)), pack2(b(k + 8, n0 + gr), b(k + 9, n0 + gr))};
      mma16816(c, af, bf, T{});
    }
  } else {
#pragma unroll 8
    for (int k = 0; k < K; ++k) {
      const Acc a0 = a(m0 + gr, k), a1 = a(m0 + gr + 8, k), b0 = b(k, n0 + 2 * tg), b1 = b(k, n0 + 2 * tg + 1);
      c[0] = fma(a0, b0, c[0]);
      c[1] = fma(a0, b1, c[1]);
      c[2] = fma(a1, b0, c[2]);
      c[3] = fma(a1, b1, c[3]);
    }
  }
}

// sums over the tile's 8 columns of the rows gr (r0) and gr + 8 (r1): lane tg == 0 ends with them
template <typename Acc> __device__ __forceinline__ void row_sum8(Acc& r0, Acc& r1) {
#pragma unroll
  for (int o = 1; o < 4; o *= 2) {
    r0 += __shfl_xor_sync(kFullMask, r0, o);
    r1 += __shfl_xor_sync(kFullMask, r1, o);
  }
}
// sums over the tile's 16 rows of the columns 2 tg (c0) and 2 tg + 1 (c1): lanes gr == 0 end with them
template <typename Acc> __device__ __forceinline__ void col_sum16(Acc& c0, Acc& c1) {
#pragma unroll
  for (int o = 4; o < 32; o *= 2) {
    c0 += __shfl_xor_sync(kFullMask, c0, o);
    c1 += __shfl_xor_sync(kFullMask, c1, o);
  }
}

}  // namespace rua
