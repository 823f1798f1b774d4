// Virtual position -> storage row decode shared by the per-sequence time-axis kernels (K7 scan.cu, K8 conv.cu).
//
// Positions are taken in VIRTUAL order: sequence-major (C order) for C and P, storage order for L / R.  A kernel cuts
// them into chunks of consecutive positions regardless of sequence boundaries; for C and P the sequences that meet a
// chunk are found once per CTA (owner_bounds), after which every position of the chunk decodes with a short search.
#pragma once

#include "common.cuh"

namespace rua {

// sequences [lo, hi) that own the virtual positions jlo .. jhi of a C or P side (jlo <= jhi); lo = hi = 0 for L / R or a
// range that starts at or past the tokens.  Warps 0 and 1 search; every thread of the CTA must call this (one barrier).
template <class Args>
__device__ __forceinline__ void owner_bounds(const Args& a, int64_t n_tok, int64_t jlo, int64_t jhi, int lane, int warp,
                                             int64_t* s_bounds, int64_t& lo, int64_t& hi) {
  const bool search = (a.layout == RUA_CAT || a.layout == RUA_PACK) && jlo < n_tok;
  if (search && warp < 2) {
    const int64_t j = warp == 0 ? jlo : min(jhi, n_tok - 1);
    const int64_t s = warp_owner_search(GlobalOff{a.off}, a.B, j, lane);
    if (lane == 0) s_bounds[warp] = s;
  }
  __syncthreads();
  lo = search ? s_bounds[0] : 0;
  hi = search ? s_bounds[1] + 1 : 0;
}

// virtual position j -> storage row srow and position t within its sequence (srow = j, t = 0 for a row that holds no
// token: L / R padding, C rows at or past n_tok = off[B]); on_token(i, len) runs for a token row only, with i the index of
// its sequence in off (token_sizes order, also for P).  [lo, hi) from owner_bounds.  Row of token (i, t): C off[i] + t,
// L i * W + t, R i * W + (W - len) + t, P poff[t] + unsorted[i].
// `a` is the kernel's argument struct (fields layout, W, off, poff, unsorted), read where it lies.
template <class Args, class OnToken>
__device__ __forceinline__ void decode_position(const Args& a, int64_t j, int64_t n_tok, int64_t lo, int64_t hi,
                                                int64_t& srow, int64_t& t, OnToken&& on_token) {
  srow = j;
  t = 0;
  int64_t i, len;
  if (a.layout == RUA_LEFT || a.layout == RUA_RIGHT) {
    i = j / a.W;
    const int64_t c = j - i * a.W;
    len = __ldg(a.off + i + 1) - __ldg(a.off + i);
    t = a.layout == RUA_LEFT ? c : c - (a.W - len);
    if (t < 0 || t >= len) return;
  } else {
    if (j >= n_tok) return;
    while (hi - lo > 1) {   // owner of j among the sequences [lo, hi) that meet this chunk
      const int64_t mid = (lo + hi) >> 1;
      if (__ldg(a.off + mid) <= j) lo = mid; else hi = mid;
    }
    i = lo;
    const int64_t o = __ldg(a.off + i);
    len = __ldg(a.off + i + 1) - o;
    t = j - o;
    if (a.layout == RUA_PACK) srow = __ldg(a.poff + t) + __ldg(a.unsorted + i);
  }
  on_token(i, len);
}

}  // namespace rua
