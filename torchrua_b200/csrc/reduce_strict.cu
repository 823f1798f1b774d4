// K4-strict -- segment sum / mean / prod in the REFERENCE'S ORDER OF OPERATIONS (parity mode).
//
// torchrua's segment_sum / segment_mean / segment_prod (torchrua/reduce.py:44-53) call torch.segment_reduce,
// whose kernels accumulate each (segment, column) strictly left to right IN THE STORAGE DTYPE, starting from
// `initial` (0 / 0 / 1): fp32 sums carry fp32 rounding per step, bf16 sums are rounded to bf16 after every add
// (4096 ones -> 256; SURVEY.md 8c hazard 2).  The fast kernels (reduce.cu) accumulate in fp32 across chunks and
// round once -- more accurate, within the stated tolerance, but not bit-identical.  This kernel replays the
// reference's arithmetic exactly: one thread per (segment, column vector), sequential over the rows, one
// rounding to T per step; mean divides by the length converted to T first (c10::BFloat16 / int64_t does that).
// Result: bit-for-bit the output of torch.segment_reduce on the same values.  Coalesced along the hidden
// dimension, 8 independent row loads in flight per thread; HBM-bound when segments are of similar length,
// serial in the longest segment otherwise -- a parity tool, not the default path.
#include "reduce_common.cuh"

namespace rua {

constexpr int kStrictThreads = 128;
constexpr int kStrictUnroll = 8;

// explicit round-to-nearest intrinsics: never contracted into FMAs
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double div_rn(double a, double b) { return __ddiv_rn(a, b); }

template <typename T> __device__ __forceinline__ typename Store<T>::Acc round_to_storage(typename Store<T>::Acc v) {
  return Store<T>::to_acc(Store<T>::from_acc(v));   // identity for fp32 / fp64
}

template <typename T, int V, int OP>
__global__ void __launch_bounds__(kStrictThreads)
segreduce_strict_kernel(const T* __restrict__ data, const int64_t* __restrict__ off, int64_t S, int64_t H,
                        T* __restrict__ out) {
  using A = typename Store<T>::Acc;
  const int64_t hv = H / V;                                  // column vectors per row (H % V == 0 here)
  const int64_t g = (int64_t)blockIdx.x * kStrictThreads + threadIdx.x;
  if (g >= S * hv) return;
  const int64_t s = g / hv;
  const int64_t col = (g - s * hv) * V;
  const int64_t beg = __ldg(off + s), end = __ldg(off + s + 1);
  A acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) acc[v] = OP == RUA_PROD ? A(1) : A(0);
  const T* p = data + beg * H + col;
  for (int64_t r = beg; r < end; r += kStrictUnroll) {
    Raw<T, V> raw[kStrictUnroll];
#pragma unroll
    for (int k = 0; k < kStrictUnroll; ++k)
      if (r + k < end) load_raw<T, V>(p + (int64_t)k * H, raw[k]);
#pragma unroll
    for (int k = 0; k < kStrictUnroll; ++k) {
      if (r + k < end) {
        A x[V];
        unpack_raw<T, V>(raw[k], x);
#pragma unroll
        for (int v = 0; v < V; ++v)   // one rounding to T per step
          acc[v] = round_to_storage<T>(OP == RUA_PROD ? mul_rn(acc[v], x[v]) : add_rn(acc[v], x[v]));
      }
    }
    p += (int64_t)kStrictUnroll * H;
  }
  if (OP == RUA_MEAN && end > beg) {
    const A n = round_to_storage<T>((A)(end - beg));         // the length goes through T first, like c10's operator/
#pragma unroll
    for (int v = 0; v < V; ++v)
      if (acc[v] == acc[v]) acc[v] = div_rn(acc[v], n);
  }
  store_vec<T, V>(out + s * H + col, acc);
}

template <typename T, int V, int OP>
static int strict_launch(const void* data, const int64_t* off, int64_t S, int64_t H, void* out, cudaStream_t st) {
  const int64_t threads = S * (H / V);
  const int64_t blocks = ceil_div(threads, kStrictThreads);
  if (blocks >= (1ll << 31)) return RUA_ERR_UNSUPPORTED;
  segreduce_strict_kernel<T, V, OP><<<(unsigned)blocks, kStrictThreads, 0, st>>>((const T*)data, off, S, H, (T*)out);
  return check_launch();
}

}  // namespace rua

using namespace rua;

extern "C" {

int rua_segment_reduce_strict(const void* data, const int64_t* off, int64_t N, int64_t S, int64_t H, int32_t dtype,
                              int32_t op, void* out, rua_stream_t stream) {
  if (N < 0 || S < 0 || H < 0) return RUA_ERR_INVALID;
  if (S == 0 || H == 0) return RUA_OK;
  if (!off || !out || (N > 0 && !data)) return RUA_ERR_INVALID;
  if (dtype < RUA_F32 || dtype > RUA_BF16) return RUA_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    constexpr int V = Store<T>::kVec;
    const bool vec = H % V == 0 && (((uintptr_t)data | (uintptr_t)out) & 15u) == 0;
    return with_op(op, [&](auto o) {
      constexpr int OP = decltype(o)::value;
      // max / min are order-independent (already bit-exact); logsumexp has no exact replay
      if constexpr (OP == RUA_SUM || OP == RUA_MEAN || OP == RUA_PROD)
        return vec ? strict_launch<T, V, OP>(data, off, S, H, out, st) : strict_launch<T, 1, OP>(data, off, S, H, out, st);
      else
        return (int)RUA_ERR_UNSUPPORTED;
    }, RUA_ERR_UNSUPPORTED);
  });
}

}  // extern "C"
