// Closed-form rows of the sequences of a ragged batch, for the kernels that walk one sequence at a time (K9 CRF, K10
// selective scan).  `Args` carries the layout fields: off, poff, sorted, unsorted, layout and Wd (the L / R width).
#pragma once

#include "common.cuh"

namespace rua {

struct Seq {
  int64_t i, o, len, prow;
};

// the sequence of rank `rank` in ragged->sorted (longest first for the package's own sort)
template <class Args> __device__ __forceinline__ Seq seq_of(const Args& a, int64_t rank) {
  Seq s;
  s.i = __ldg(a.sorted + rank);
  s.o = __ldg(a.off + s.i);
  s.len = __ldg(a.off + s.i + 1) - s.o;
  s.prow = a.layout == RUA_PACK ? __ldg(a.unsorted + s.i) : 0;
  return s;
}

// storage row of token t of sequence s: C off[i] + t, L i W + t, R i W + W - len + t, P poff[t] + unsorted[i]
template <class Args> __device__ __forceinline__ int64_t row_of(const Args& a, const Seq& s, int64_t t) {
  switch (a.layout) {
    case RUA_CAT: return s.o + t;
    case RUA_LEFT: return s.i * a.Wd + t;
    case RUA_RIGHT: return s.i * a.Wd + (a.Wd - s.len) + t;
    default: return __ldg(a.poff + t) + s.prow;
  }
}

// f(row) for every row of sequence s's L / R storage that holds no token: rows first, first + step, ... of them
template <class Args, class F>
__device__ __forceinline__ void for_padding_rows(const Args& a, const Seq& s, int first, int step, F&& f) {
  if (a.layout != RUA_LEFT && a.layout != RUA_RIGHT) return;
  const int64_t base = s.i * a.Wd + (a.layout == RUA_LEFT ? s.len : 0);
  for (int64_t q = first; q < a.Wd - s.len; q += step) f(base + q);
}

}  // namespace rua
