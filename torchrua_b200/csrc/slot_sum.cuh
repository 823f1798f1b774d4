// Second phase of the backward passes that reduce a small gradient over the whole batch (K8 weight / bias, K9
// transitions / start / end): every CTA of the first phase stored its partial sums in its own slot of the workspace, and
// this kernel sums the slots in slot order.  No atomics, so the result is bit-identical run to run.
#pragma once

#include "reduce_common.cuh"

namespace rua {

// out column i (i < n) = sum over slots sl < S, in slot order, of slots[sl * stride + src], where cols(i, src) sets src
// and returns where the column goes (nullptr: not wanted)
template <typename T, class Cols>
__global__ void slot_sum(const typename Store<T>::Acc* slots, int64_t S, int64_t stride, int64_t n, Cols cols) {
  using A = typename Store<T>::Acc;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t src;
    T* dst = cols(i, src);
    if (!dst) continue;
    const A* p = slots + src;
    A s = 0;
    for (int64_t sl = 0; sl < S; ++sl) s += __ldcg(p + sl * stride);
    *dst = Store<T>::from_acc(s);
  }
}

template <typename T, class Cols>
inline int launch_slot_sum(const typename Store<T>::Acc* slots, int64_t S, int64_t stride, int64_t n, Cols cols,
                           cudaStream_t st) {
  const unsigned blocks = (unsigned)(ceil_div(n, 256) < 4096 ? ceil_div(n, 256) : 4096);
  slot_sum<T><<<blocks, 256, 0, st>>>(slots, S, stride, n, cols);
  return check_launch();
}

}  // namespace rua
