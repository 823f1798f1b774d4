// K4w' -- backward twin of reduce_warpseg.cu (its own translation unit: the two files are ~160 kernel instances each).
#include "warpseg_common.cuh"

namespace rua {

// ------------------------------------------------------------------------------------------------------------------
// backward twin for the same shape (narrow rows, many short segments): grad[r] = f(g[s], out[s], x[r], #ties) as in
// reduce_bwd.cu, but organised like the forward kernel -- the chunk kernel there gives every THREAD its own run of rows
// when rows are this narrow (13 % of the HBM peak at H = 1: nothing coalesces).  Here lane i owns segment s0 + i, reads
// g / out once (coalesced), rewrites ITS rows inside the warp's shared-memory window (x arrives by TMA bulk copy when the
// op needs it) and the warp then stores the window with coalesced 128-bit stores.  max / min count their ties in a
// first sweep over the same windows (second sweep: L2 hits).
// ------------------------------------------------------------------------------------------------------------------
template <typename T, int HE, int OP>
__global__ void __launch_bounds__(kWsThreads)
segreduce_bwd_warpseg_kernel(const T* __restrict__ gout, const T* __restrict__ out, const T* __restrict__ data,
                             const int64_t* __restrict__ off, int64_t N, int64_t S, T* __restrict__ grad) {
  using A = typename Store<T>::Acc;
  constexpr bool kNeedsX = OP == RUA_MAX || OP == RUA_MIN || OP == RUA_PROD || OP == RUA_LOGSUMEXP;
  constexpr bool kTies = OP == RUA_MAX || OP == RUA_MIN;
  constexpr int E = 16 / (int)sizeof(T);
  constexpr int CE = kWsChunkBytes / (int)sizeof(T);
  constexpr int CR = CE / HE;
  __shared__ __align__(128) uint4 s_buf[kWsWarps][kWsChunkBytes / 16];
  __shared__ __align__(8) uint64_t s_bar[kWsWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t s0 = ((int64_t)blockIdx.x * kWsWarps + warp) * 32;
  const int64_t covered = __ldg(off + S) < N ? __ldg(off + S) : N;
  if (covered < N) {                                  // rows no segment owns (sum of sizes < N): zero gradient, every warp
    const int64_t step = (int64_t)gridDim.x * kWsThreads;   // of the grid takes a strided share of them
    for (int64_t e = covered * HE + (int64_t)blockIdx.x * kWsThreads + threadIdx.x; e < N * HE; e += step)
      grad[e] = Store<T>::from_acc(A(0));
  }
  if (s0 >= S) return;                                // warp-uniform; nothing block-wide below
  const int64_t s = s0 + lane;
  int64_t beg = s < S ? __ldg(off + s) : covered, end = s < S ? __ldg(off + s + 1) : covered;
  const int64_t len = end - beg;
  beg = beg < covered ? beg : covered;
  end = end < covered ? end : covered;
  const int64_t wbeg = shfl_i64(beg, 0), wend = shfl_i64(end, 31);
  const int64_t seg_beg = beg;                        // for prod's exact fallback
  A g[HE], o[HE], c[HE];
  int ties[HE];
#pragma unroll
  for (int h = 0; h < HE; ++h) {
    g[h] = (s < S && len > 0) ? Store<T>::to_acc(gout[s * HE + h]) : A(0);
    o[h] = (kNeedsX && s < S && len > 0) ? Store<T>::to_acc(out[s * HE + h]) : A(0);
    if (OP == RUA_MEAN && len > 0) g[h] = g[h] * (A(1) / (A)len);
    c[h] = g[h];
    ties[h] = 0;
  }
  const int64_t total_e = N * HE;
  const int64_t bulk_e = total_e & ~(int64_t)(E - 1);
  uint4* s_mine = s_buf[warp];
  T* sb = reinterpret_cast<T*>(s_mine);
  uint64_t* bar = &s_bar[warp];
  uint32_t phase = 0;
  if (kNeedsX) {
    if (lane == 0) mbar_init(bar, 1);
    __syncwarp();
  }
  // the rows [r_lo, r_hi) of the window that starts at element e0 are in shared memory after this (x values)
  auto load_window = [&](int64_t e0, int64_t stop_e) {
    const int64_t bulk_stop = stop_e < bulk_e ? stop_e : bulk_e;
    const uint32_t nbytes = bulk_stop > e0 ? (uint32_t)((bulk_stop - e0) * (int64_t)sizeof(T)) : 0u;
    if (nbytes) {
      if (lane == 0) {
        mbar_expect_tx(bar, nbytes);
        bulk_g2s(s_mine, data + e0, nbytes, bar);
      }
      mbar_wait(bar, phase);
      phase ^= 1u;
    }
    if (stop_e > bulk_e) {
      for (int64_t e = (bulk_e > e0 ? bulk_e : e0) + lane; e < total_e && e < stop_e; e += 32) sb[e - e0] = data[e];
      __syncwarp();
    }
  };
  auto one = [&](A x, int h, int64_t row) -> A {      // gradient of one element
    if (OP == RUA_SUM || OP == RUA_MEAN) return g[h];
    if (kTies) return (x != x || x == o[h]) ? c[h] : A(0);
    if (OP == RUA_LOGSUMEXP) return g[h] * exp_acc<false>(x - o[h]);
    if (x != x || x == A(0)) {                         // prod through a zero / NaN: product of the others, exactly
      A ex = A(1);
      for (int64_t q = seg_beg; q < seg_beg + len; ++q)
        if (q != row) ex *= Store<T>::to_acc(data[q * HE + h]);
      return g[h] * ex;
    }
    return g[h] * o[h] / x;
  };

  const int64_t e_first = (wbeg * HE) & ~(int64_t)(E - 1);
  for (int sweep = kTies ? 0 : 1; sweep < 2; ++sweep) {
    for (int64_t e0 = e_first; e0 < wend * HE; e0 += CE) {
      const int64_t want_e = (wend * HE - e0 + (E - 1)) & ~(int64_t)(E - 1);
      const int64_t stop_e = e0 + (want_e < CE ? want_e : CE);
      const int64_t r_lo = e0 / HE;
      const int64_t r_hi = r_lo + CR < wend ? r_lo + CR : wend;
      if (kNeedsX) load_window(e0, stop_e);
      const unsigned who = __ballot_sync(kFullMask, beg <= r_lo && end >= r_lo + CR);
      if (who) {
        // ---- the window lies inside ONE segment: every lane handles its own vectors with the owner's values ----------
        const int own = __ffs(who) - 1;
        A og[HE], oo[HE], oc[HE];
#pragma unroll
        for (int h = 0; h < HE; ++h) {
          og[h] = __shfl_sync(kFullMask, g[h], own);
          oo[h] = __shfl_sync(kFullMask, o[h], own);
          oc[h] = __shfl_sync(kFullMask, c[h], own);
        }
        const int64_t obeg = shfl_i64(seg_beg, own), olen = shfl_i64(len, own);
        int local[HE];
#pragma unroll
        for (int h = 0; h < HE; ++h) local[h] = 0;
#pragma unroll
        for (int j = 0; j < kWsVecPerLane; ++j) {
          const int v = lane + 32 * j;
          A x[E], y[E];
          if (kNeedsX) Store<T>::unpack(s_mine[v], x);
#pragma unroll
          for (int k = 0; k < E; ++k) {
            const int h = k % HE;
            if (sweep == 0) {
              local[h] += (x[k] != x[k] || x[k] == oo[h]) ? 1 : 0;
            } else if (OP == RUA_SUM || OP == RUA_MEAN) {
              y[k] = og[h];
            } else if (kTies) {
              y[k] = (x[k] != x[k] || x[k] == oo[h]) ? oc[h] : A(0);
            } else if (OP == RUA_LOGSUMEXP) {
              y[k] = og[h] * exp_acc<false>(x[k] - oo[h]);
            } else if (x[k] != x[k] || x[k] == A(0)) {
              const int64_t row = r_lo + (int64_t)(v * E + k) / HE;
              A ex = A(1);
              for (int64_t q = obeg; q < obeg + olen; ++q)
                if (q != row) ex *= Store<T>::to_acc(data[q * HE + h]);
              y[k] = og[h] * ex;
            } else {
              y[k] = og[h] * oo[h] / x[k];
            }
          }
          if (sweep == 1) *reinterpret_cast<uint4*>(grad + e0 + (int64_t)v * E) = Store<T>::pack(y);   // window is full: in range
        }
        if (sweep == 0) {
#pragma unroll
          for (int h = 0; h < HE; ++h) {
            int t = local[h];
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) t += __shfl_xor_sync(kFullMask, t, d);
            if (lane == own) ties[h] += t;
          }
        }
      } else {
        // ---- every lane walks its own segment's rows inside the window --------------------------------------------
        const int64_t lo = beg < r_lo ? r_lo : (beg > r_hi ? r_hi : beg), hi = end < r_lo ? r_lo : (end > r_hi ? r_hi : end);
        for (int64_t row = lo; row < hi; ++row) {
          T* cell = sb + (row - r_lo) * HE;
#pragma unroll
          for (int h = 0; h < HE; ++h) {
            const A x = kNeedsX ? Store<T>::to_acc(cell[h]) : A(0);
            if (sweep == 0) ties[h] += (x != x || x == o[h]) ? 1 : 0;
            else cell[h] = Store<T>::from_acc(one(x, h, row));
          }
        }
        if (sweep == 1) {
          __syncwarp();
          // coalesced store of the window: whole vectors inside the warp's range, elements at its two edges
          const int64_t ebeg = wbeg * HE, eend = wend * HE;
#pragma unroll
          for (int j = 0; j < kWsVecPerLane; ++j) {
            const int v = lane + 32 * j;
            const int64_t e = e0 + (int64_t)v * E;
            if (e >= stop_e) continue;
            if (e >= ebeg && e + E <= eend) {
              *reinterpret_cast<uint4*>(grad + e) = s_mine[v];
            } else {
#pragma unroll
              for (int k = 0; k < E; ++k)
                if (e + k >= ebeg && e + k < eend) grad[e + k] = sb[v * E + k];
            }
          }
        }
      }
      __syncwarp();
    }
    if (kTies && sweep == 0) {
#pragma unroll
      for (int h = 0; h < HE; ++h) c[h] = ties[h] > 1 ? g[h] / (A)ties[h] : g[h];
    }
  }
}

// The kernel writes every one of the N rows: the segments' rows [0, off[S]) and zeros on the rows past the last segment.
int warpseg_bwd_launch(int32_t dtype, int64_t H, int32_t op, const void* gout, const void* out, const void* data,
                       const int64_t* off, int64_t N, int64_t S, void* grad, cudaStream_t st) {
  // per-token SCALARS only (H == 1: log-probabilities, losses, scores -- the config-5 shape).  Rows of 2..8 elements
  // keep the chunk kernel of reduce_bwd.cu: instantiating this kernel for them as well costs minutes of compile time
  // for a shape nothing on the path produces.
  if (H != 1) return RUA_ERR_UNSUPPORTED;
  const int64_t blocks = ceil_div(S, (int64_t)kWsWarps * 32);
  if (blocks >= (1ll << 31)) return RUA_ERR_UNSUPPORTED;
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    return with_op(op, [&](auto o) {
      segreduce_bwd_warpseg_kernel<T, 1, decltype(o)::value><<<(unsigned)blocks, kWsThreads, 0, st>>>(
          (const T*)gout, (const T*)out, (const T*)data, off, N, S, (T*)grad);
      return check_launch();
    });
  });
}

}  // namespace rua
