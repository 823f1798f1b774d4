// K4-ws -- segment reduce for NARROW rows (H * elem <= 16 bytes) and MANY SHORT segments: per-token scalars reduced
// per sequence (BASELINE config 5: 1 M segments of 1..64 fp32 values).
//
// Replaces (reference file:line): the same segment_* functions as reduce.cu (torchrua/reduce.py:34-61) on the
// featureless / few-column inputs that mask.py / segment.py style pooling produces.
//
// The rows-on-lanes kernel of reduce_flat.cu spends its time in a per-tile decode chain (two searches, a staged
// offset table, a block scan, three barriers: 49 M warp instructions for 32.5 M rows, 16 % of the HBM peak).  Here a
// WARP owns 32 consecutive SEGMENTS instead:
//   * lane i reads off[s0 + i], off[s0 + i + 1] -- two coalesced loads, no search, no decode, no block barrier;
//   * the rows of those 32 segments are one contiguous range; the warp streams it through a private 4 KB
//     shared-memory window, each window ONE TMA bulk copy (cp.async.bulk global -> shared, completion on a per-warp
//     mbarrier) issued by lane 0: no per-lane load / store instructions, no registers held across the DRAM latency;
//   * every lane then reduces ITS OWN segment out of the window, left to right, four scalars per 128-bit LDS -- all 32
//     lanes busy, about 10x fewer instructions than the tile kernel;
//   * a window that lies entirely inside ONE long segment is reduced by the whole warp (conflict-free reads, shuffle
//     tree), so a long sequence among short ones costs bandwidth, not a serial loop;
//   * every segment is finished by the lane that owns it: no cross-tile pieces, no span kernel, results stored coalesced.
// The launcher picks this kernel when there are enough segments to fill the machine (reduce.cu: plan_reduce).
// Measured and dropped (round 2): 256-thread CTAs (4.4 waves at cfg5: 51 % vs 55 % of peak for 128 threads), and TWO groups of 32
// segments per warp with both first windows in flight (43 %: the extra state costs occupancy, which is what hides the two serial
// DRAM latencies -- offsets, then the window -- of a warp).
#include "warpseg_common.cuh"

namespace rua {

template <typename T, int HE, int OP>
__global__ void __launch_bounds__(kWsThreads)
segreduce_warpseg_kernel(const T* __restrict__ data, const int64_t* __restrict__ off, int64_t N, int64_t S,
                         T* __restrict__ out, RedHeader* hdr) {
  using A = typename Store<T>::Acc;
  using St = State<A, HE, OP>;
  constexpr bool kFast = sizeof(T) == 2;
  constexpr int E = 16 / (int)sizeof(T);            // elements per 16-byte vector
  constexpr int G = E / HE;                         // rows per vector
  constexpr int CE = kWsChunkBytes / (int)sizeof(T);
  constexpr int CR = CE / HE;                       // rows per window
  __shared__ __align__(128) uint4 s_buf[kWsWarps][kWsChunkBytes / 16];
  __shared__ __align__(8) uint64_t s_bar[kWsWarps];

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t s0 = ((int64_t)blockIdx.x * kWsWarps + warp) * 32;
  St acc;
  acc.reset();
  A ext = OP == RUA_MIN ? -inf_of<A>() : inf_of<A>();
  bool saw_nan = false;

  if (s0 < S) {                                     // warp-uniform
    const int64_t covered = __ldg(off + S) < N ? __ldg(off + S) : N;   // rows past the last segment / past N belong to nobody
    const int64_t s = s0 + lane;
    int64_t beg = s < S ? __ldg(off + s) : covered, end = s < S ? __ldg(off + s + 1) : covered;
    const int64_t len = end - beg;
    beg = beg < covered ? beg : covered;
    end = end < covered ? end : covered;
    const int64_t wbeg = shfl_i64(beg, 0), wend = shfl_i64(end, 31);
    const int64_t total_e = N * HE;
    const int64_t bulk_e = total_e & ~(int64_t)(E - 1);   // elements reachable with whole 16-byte vectors
    uint4* s_mine = s_buf[warp];
    const T* sb = reinterpret_cast<const T*>(s_mine);
    uint64_t* bar = &s_bar[warp];
    uint32_t phase = 0;
    if (lane == 0) mbar_init(bar, 1);
    __syncwarp();

    auto add_ext = [&](const A* x) {
      if (OpInfo<OP>::kNeedsExt) {
#pragma unroll
        for (int h = 0; h < HE; ++h) ext = OP == RUA_MIN ? max_num(ext, x[h]) : min_num(ext, x[h]);
      }
    };
    auto add_row = [&](int r) {                      // one row out of the window (row_bytes-wide LDS)
      A x[HE];
      constexpr int kBytes = HE * (int)sizeof(T);
      const T* p = sb + r * HE;
      if constexpr (kBytes == 8) {
        const uint2 w = *reinterpret_cast<const uint2*>(p);
        A y[E];
        Store<T>::unpack(make_uint4(w.x, w.y, 0u, 0u), y);
#pragma unroll
        for (int h = 0; h < HE; ++h) x[h] = y[h];
      } else if constexpr (kBytes == 4) {
        const uint32_t w = *reinterpret_cast<const uint32_t*>(p);
        A y[E];
        Store<T>::unpack(make_uint4(w, 0u, 0u, 0u), y);
#pragma unroll
        for (int h = 0; h < HE; ++h) x[h] = y[h];
      } else {
#pragma unroll
        for (int h = 0; h < HE; ++h) x[h] = Store<T>::to_acc(p[h]);
      }
      acc.template add<kFast>(x);
      add_ext(x);
    };

    for (int64_t e0 = (wbeg * HE) & ~(int64_t)(E - 1); e0 < wend * HE; e0 += CE) {   // e0: a multiple of E (data is 16-byte aligned)
      // ---- the window [e0, e0 + CE) arrives with ONE bulk copy issued by lane 0 --------------------------------
      const int64_t want_e = (wend * HE - e0 + (E - 1)) & ~(int64_t)(E - 1);      // up to the warp's last row, in whole vectors
      const int64_t stop_e = e0 + (want_e < CE ? want_e : CE);
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
      if (stop_e > bulk_e) {                          // the last, partial vector of the whole array: element by element
        T* st_ = reinterpret_cast<T*>(s_mine);
        for (int64_t e = (bulk_e > e0 ? bulk_e : e0) + lane; e < total_e && e < stop_e; e += 32) st_[e - e0] = data[e];
        __syncwarp();
      }
      const int64_t r_lo = e0 / HE;                  // first row of the window (HE divides E)
      const int64_t r_hi = r_lo + CR < wend ? r_lo + CR : wend;
      // does ONE segment cover the whole window?  (at most one lane can say yes)
      const unsigned who = __ballot_sync(kFullMask, beg <= r_lo && end >= r_lo + CR);
      if (who) {                                     // the whole warp reduces it: 8 conflict-free 128-bit reads per lane
        St part;
        part.reset();
#pragma unroll
        for (int j = 0; j < kWsVecPerLane; ++j) {
          A x[E];
          Store<T>::unpack(s_mine[lane + 32 * j], x);
#pragma unroll
          for (int g = 0; g < G; ++g) {
            part.template add<kFast>(&x[g * HE]);
            add_ext(&x[g * HE]);
          }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
          const St other = ws_shfl_xor<A, HE, OP>(part, d);
          part.template merge<kFast>(other);
        }
        if (lane == __ffs(who) - 1) acc.template merge<kFast>(part);
      } else {                                       // every lane reduces its own segment's rows, left to right
        const int64_t lo = beg < r_lo ? r_lo : (beg > r_hi ? r_hi : beg), hi = end < r_lo ? r_lo : (end > r_hi ? r_hi : end);
        int r = (int)(lo - r_lo);
        const int r_end = (int)(hi - r_lo);
        if constexpr (G > 1) {
          for (; r < r_end && (r & (G - 1)); ++r) add_row(r);
        }
#pragma unroll 2
        for (; r + G <= r_end; r += G) {             // G rows per 128-bit LDS
          A x[E];
          Store<T>::unpack(*reinterpret_cast<const uint4*>(sb + r * HE), x);
#pragma unroll
          for (int g = 0; g < G; ++g) {
            acc.template add<kFast>(&x[g * HE]);
            add_ext(&x[g * HE]);
          }
        }
        if constexpr (G > 1) {
          for (; r < r_end; ++r) add_row(r);
        }
      }
      __syncwarp();                                  // everybody is done with the window before it is overwritten
    }

    if (s < S) {
      A o[HE];
      if (len > 0) {
        acc.finalize(OP == RUA_MEAN ? len : 1, o);
        if (OpInfo<OP>::kNeedsExt) saw_nan |= acc.any_nan_out(o);
      } else {                                       // empty: sum / mean -> 0, prod -> 1; max / min / logsumexp are patched
#pragma unroll
        for (int h = 0; h < HE; ++h) o[h] = OP == RUA_PROD ? A(1) : A(0);
      }
      T packed[HE];
#pragma unroll
      for (int h = 0; h < HE; ++h) packed[h] = Store<T>::from_acc(o[h]);
      if constexpr (HE * sizeof(T) == 16) *reinterpret_cast<uint4*>(out + s * HE) = *reinterpret_cast<const uint4*>(packed);
      else if constexpr (HE * sizeof(T) == 8) *reinterpret_cast<uint2*>(out + s * HE) = *reinterpret_cast<const uint2*>(packed);
      else if constexpr (HE * sizeof(T) == 4) *reinterpret_cast<uint32_t*>(out + s * HE) = *reinterpret_cast<const uint32_t*>(packed);
      else {
#pragma unroll
        for (int h = 0; h < HE; ++h) out[s * HE + h] = packed[h];
      }
    }
  }

  if (OpInfo<OP>::kNeedsExt) {                       // global extreme + NaN flag: one atomic per CTA, and only if it can matter
    __shared__ unsigned long long s_key[kWsWarps];
    __shared__ int s_nan;
    if (threadIdx.x == 0) s_nan = 0;
    __syncthreads();
    unsigned long long key = order_key(ext);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const unsigned long long o = __shfl_xor_sync(kFullMask, key, d);
      key = OP == RUA_MIN ? (o > key ? o : key) : (o < key ? o : key);
    }
    if (lane == 0) s_key[warp] = key;
    if (saw_nan) s_nan = 1;
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int w = 1; w < kWsWarps; ++w) {
        const unsigned long long o = s_key[w];
        key = OP == RUA_MIN ? (o > key ? o : key) : (o < key ? o : key);
      }
      const unsigned long long cur = *reinterpret_cast<volatile unsigned long long*>(&hdr->ext_key);
      if (OP == RUA_MIN ? key > cur : key < cur) { if (OP == RUA_MIN) atomicMax(&hdr->ext_key, key); else atomicMin(&hdr->ext_key, key); }
      if (s_nan) atomicOr(&hdr->nan_flag, 1u);
    }
  }
}

int warpseg_launch(int32_t dtype, int64_t H, int32_t op, const void* data, const int64_t* off, int64_t N, int64_t S,
                   void* out, void* hdr, cudaStream_t st) {
  const int64_t blocks = ceil_div(S, (int64_t)kWsWarps * 32);
  if (blocks >= (1ll << 31)) return RUA_ERR_UNSUPPORTED;
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    return with_row_elems<T>(H, [&](auto he) {
      return with_op(op, [&](auto o) {
        segreduce_warpseg_kernel<T, decltype(he)::value, decltype(o)::value><<<(unsigned)blocks, kWsThreads, 0, st>>>(
            (const T*)data, off, N, S, (T*)out, (RedHeader*)hdr);
        return check_launch();
      });
    });
  });
}

}  // namespace rua
