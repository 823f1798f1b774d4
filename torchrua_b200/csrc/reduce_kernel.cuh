// K4 main kernel (template): shared by reduce.cu (segments of any length) and reduce_short.cu (the SHORT instantiation
// for batches of very short segments -- sub-word -> word pooling, .seg() pieces: 1..16 rows each).
#pragma once
#include "reduce_common.cuh"

namespace rua {

// ---------------------------------------------------------------------------------------------
// main kernel
// ---------------------------------------------------------------------------------------------
template <typename T, int V, int OP, bool GATHER, bool PACKED, bool SHORT = false>
__global__ void __launch_bounds__(kRedThreads, Store<T>::kMinBlocks)
segreduce_kernel(const T* __restrict__ data, const int64_t* __restrict__ ridx, const int64_t* __restrict__ off,
                 int64_t N, int64_t S, int64_t H, int R, T* __restrict__ out, typename Store<T>::Acc* __restrict__ head,
                 typename Store<T>::Acc* __restrict__ tail, int64_t* __restrict__ tail_seg, RedHeader* hdr,
                 int lanes_log2, int64_t chunks) {
  using A = typename Store<T>::Acc;
  constexpr bool kFast = sizeof(T) == 2;  // 16-bit storage: 1e-2 tolerance, approximate exp is plenty
  constexpr int P = OpInfo<OP>::kParts;
  // 2^lanes_log2 threads span one row (16 bytes each).  Rows of >= 32 vectors: that is the whole CTA (one chunk per
  // CTA, boundaries CTA-uniform).  Shorter rows (32 .. 256 bytes): the CTA hosts blockDim / lanes chunks side by
  // side, one per thread group, so that no lane idles; groups of a warp then diverge at their own boundaries.
  // (a compile-time switch: the extra index arithmetic made the wide-row logsumexp instance spill at its 80 registers)
  const int lanes = PACKED ? 1 << lanes_log2 : (int)blockDim.x;
  const int64_t chunk = PACKED ? (int64_t)blockIdx.x * (blockDim.x >> lanes_log2) + (threadIdx.x >> lanes_log2) : (int64_t)blockIdx.x;
  const int64_t col = PACKED ? ((int64_t)blockIdx.y * lanes + (threadIdx.x & (lanes - 1))) * V
                             : ((int64_t)blockIdx.y * blockDim.x + threadIdx.x) * V;
  const bool active = PACKED ? (col < H && chunk < chunks) : col < H;
  const int64_t row0 = (!PACKED || chunk < chunks) ? chunk * R : N;
  const int64_t row1 = row0 + R < N ? row0 + R : N;

  GlobalOff g{off};
  int64_t s = owner_search(g, S, (!PACKED || row0 < N) ? row0 : (N > 0 ? N - 1 : 0));
  int64_t seg_beg = __ldg(off + s), seg_end = __ldg(off + s + 1);
  // SHORT: a boundary every few rows -- the end of the NEXT segment is fetched one boundary ahead, so the load that the
  // boundary test depends on has a whole segment of rows to land
  constexpr int64_t kNoEnd = 0x7fffffffffffffffll;
  int64_t nxt_end = kNoEnd;
  if constexpr (SHORT) nxt_end = s + 1 < S ? __ldg(off + s + 2) : kNoEnd;
  bool open = seg_beg < row0;   // the segment began in an earlier chunk
  bool pending = false;

  State<A, V, OP> st;
  st.reset();
  A ext = OP == RUA_MIN ? -inf_of<A>() : inf_of<A>();
  uint32_t ext2[4] = {Pk<T>::kPosInf, Pk<T>::kPosInf, Pk<T>::kPosInf, Pk<T>::kPosInf};  // packed running min
  bool saw_nan = false;

  const T* colp = data + col;
  for (int64_t r = row0; r < row1; r += kRedUnroll) {
    Raw<T, V> raw[kRedUnroll];
    if (active) {
#pragma unroll
      for (int k = 0; k < kRedUnroll; ++k)
        if (r + k < row1) load_raw<T, V>(colp + (GATHER ? __ldg(ridx + r + k) : r + k) * H, raw[k]);  // compile-time: row gather (scatter_*)
    }
    // the current segment ends after row `seg_end - 1`: store it and move to the next non-empty one
    auto finish_segment = [&]() {
      if (active) {
        if (open) {
          store_partial<A, V, OP>(head + chunk * P * H, H, col, st);
        } else {
          A o[V];
          if constexpr (SHORT && kFast) st.finalize_recip(seg_end - seg_beg, o);
          else st.template finalize<kFast>(seg_end - seg_beg, o);
          if (OpInfo<OP>::kNeedsExt) saw_nan |= st.any_nan_out(o);
          store_vec<T, V>(out + s * H + col, o);
        }
      }
      st.reset();
      open = false;
      pending = false;
      do {
        ++s;
        seg_beg = seg_end;
        if constexpr (SHORT) {
          seg_end = nxt_end;
          nxt_end = s + 1 < S ? __ldg(off + s + 2) : kNoEnd;
        } else {
          seg_end = s < S ? __ldg(off + s + 1) : kNoEnd;
        }
      } while (s < S && seg_end == seg_beg);
    };

    // Walk the batch run by run: rows [k, e) of the batch belong to the current segment.  Register
    // arrays need static indices, so the per-row code is an unrolled, range-predicated sweep; the
    // (large) segment-finalising code appears once per kernel instead of once per unrolled row.
    const int nrows = (int)(row1 - r < kRedUnroll ? row1 - r : kRedUnroll);
    if constexpr (SHORT) {
      // Segments of a few rows: the run-by-run walk below would sweep the 8 predicated row slots once PER RUN (3-8 times
      // per batch).  Here every row is visited once, in order, with a (uniform) boundary test after it; the finalising
      // code is replicated per slot.  logsumexp uses the one-exponential online update of State::add.
#pragma unroll
      for (int kk = 0; kk < kRedUnroll; ++kk) {
        if (kk < nrows) {
          if (active) {
            A x[V];
            unpack_raw<T, V>(raw[kk], x);
            if (OpInfo<OP>::kIsLse && !pending) {          // first row of a piece: exp(x - x) = 1, no exponential needed
#pragma unroll
              for (int v = 0; v < V; ++v) { st.a[v] = x[v]; st.s[v] = x[v] == -inf_of<A>() ? A(0) : A(1); }   // -inf adds 0
            } else {
              st.template add<kFast>(x);
            }
            if (OpInfo<OP>::kNeedsExt) {
#pragma unroll
              for (int v = 0; v < V; ++v) ext = OP == RUA_MIN ? max_num(ext, x[v]) : min_num(ext, x[v]);
            }
          }
          pending = true;
          if (r + kk + 1 == seg_end) finish_segment();   // uniform across the CTA (or the thread group when PACKED)
        }
      }
      continue;
    }
    int k = 0;
    while (k < nrows) {
      const int64_t left_in_seg = seg_end - r;
      const int e = (int)(left_in_seg < nrows ? left_in_seg : nrows);
      bool done = false;
      if constexpr (OpInfo<OP>::kIsLse) {
        if (k == 0 && e == kRedUnroll) {
          // fast path (uniform): all 8 rows belong to the current segment.  Batch max first, one rescale
          // of the running sum, then exactly one FFMA + EX2 + FADD per element; for 16-bit storage the
          // max and the global-extreme tracking run on packed pairs (HMNMX2), halving their issue cost.
          if (active) lse_batch<T, V, kRedUnroll>(raw, st.a, st.s, ext, ext2);
          done = true;
        }
        // (round 2: batches of 4 rows / 64 registers / 8 CTAs per SM instead of 8 rows / 80 registers / 6 CTAs measured
        // 79.2 % of peak at cfg3 against 85.2 %: the kernel is bound by issue slots and the MUFU pipe -- one EX2 per
        // element is 1.46 ms of SFU time at 16 per clock per SM inside a 2.4 ms kernel -- not by exposed latency.)
        // (round 2: a masked batched form for boundary batches -- rows [k, e) only -- measured 81.3 % of peak at cfg3
        // against 84.6 % for the per-element update below: the kernel sits at its 80-register cap and the extra code
        // costs more than the ~13 % of rows it would speed up.  Dropped.)
      }
      if (!done && active) {
#pragma unroll
        for (int kk = 0; kk < kRedUnroll; ++kk) {
          if (kk >= k && kk < e) {
            A x[V];
            unpack_raw<T, V>(raw[kk], x);
            st.template add<kFast>(x);
            if (OpInfo<OP>::kNeedsExt) {
#pragma unroll
              for (int v = 0; v < V; ++v) ext = OP == RUA_MIN ? max_num(ext, x[v]) : min_num(ext, x[v]);
            }
          }
        }
      }
      pending = true;
      k = e;
      if (r + e == seg_end) finish_segment();  // uniform across the CTA
    }
  }
  if (OpInfo<OP>::kIsLse) ext = min_num(ext, packed_min_to_acc<T, V>(ext2));
  // tell the span kernel which segment (if any) starts in this chunk and runs past its end
  if ((PACKED ? ((threadIdx.x & (lanes - 1)) == 0 && chunk < chunks) : threadIdx.x == 0) && blockIdx.y == 0)
    tail_seg[chunk] = (pending && !open) ? s : -1;
  if (pending && active) {
    // the segment continues in the next chunk: whole-chunk pieces go to `head`, suffix pieces to `tail`
    store_partial<A, V, OP>((open ? head : tail) + chunk * P * H, H, col, st);
    if (OpInfo<OP>::kNeedsExt) {
#pragma unroll
      for (int v = 0; v < V; ++v) saw_nan |= (st.a[v] != st.a[v]);
    }
  }

  if (OpInfo<OP>::kNeedsExt) {
    __shared__ unsigned long long s_key[kRedThreads / 32];
    __shared__ int s_nan;
    if (threadIdx.x == 0) s_nan = 0;
    __syncthreads();
    unsigned long long key = order_key(ext);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      unsigned long long o = __shfl_xor_sync(kFullMask, key, d);
      key = OP == RUA_MIN ? (o > key ? o : key) : (o < key ? o : key);
    }
    if ((threadIdx.x & 31) == 0) s_key[threadIdx.x >> 5] = key;
    if (saw_nan) s_nan = 1;
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int w = 1; w < (int)(blockDim.x >> 5); ++w) {
        unsigned long long o = s_key[w];
        key = OP == RUA_MIN ? (o > key ? o : key) : (o < key ? o : key);
      }
      if (OP == RUA_MIN) atomicMax(&hdr->ext_key, key); else atomicMin(&hdr->ext_key, key);
      if (s_nan) atomicOr(&hdr->nan_flag, 1u);
    }
  }
}

}  // namespace rua
