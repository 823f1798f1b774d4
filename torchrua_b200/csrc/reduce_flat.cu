// K4-flat -- segment reduce for NARROW rows (H * elem <= 16 bytes: per-token scalars such as
// log-probabilities, or 2/4/8-wide features), where the wide-row kernel of reduce.cu would leave most
// lanes idle.  This is the "warp shuffles + segmented scan across ragged boundaries" kernel.
//
// Rows map to lanes.  A CTA owns a tile of 256*G consecutive rows (G = 16 / row_bytes: one 128-bit
// load per thread).  The segments that intersect the tile are found with two warp-cooperative 32-ary
// searches and their tile-relative offsets staged in shared memory as 32-bit ints (these kernels are
// issue-bound, so everything inside a tile is 32-bit).  Each thread reduces its G rows locally, cutting
// at segment boundaries: runs that start AND end inside the thread are complete segments and are
// stored directly; the first run may continue one from the threads before, the last may continue into
// the threads after.  Those open ends are stitched by a block-wide SEGMENTED SCAN BY KEY over
// (segment, partial) pairs -- warp shuffles, then one shared-memory hop in which warp 0 scans the 8
// warp totals.  Pieces of segments that cross tile boundaries go to the same head/tail scratch as in
// reduce.cu and are merged in tile order by segreduce_span_kernel: deterministic, no float atomics.
#include "reduce_common.cuh"
#include "tile_decode.cuh"

namespace rua {

constexpr int kFlatThreads = 256;
constexpr int kFlatWarps = kFlatThreads / 32;

template <typename A, int HE, int OP, bool kFast>
__device__ __forceinline__ void flat_merge(State<A, HE, OP>& later, const State<A, HE, OP>& earlier) {
  State<A, HE, OP> t = earlier;
  t.template merge<kFast>(later);
  later = t;
}

template <typename A, int HE, int OP>
__device__ __forceinline__ State<A, HE, OP> flat_shfl_up(const State<A, HE, OP>& v, int d) {
  State<A, HE, OP> o;
#pragma unroll
  for (int h = 0; h < HE; ++h) {
    o.a[h] = __shfl_up_sync(kFullMask, v.a[h], d);
    if constexpr (OpInfo<OP>::kIsLse) o.s[h] = __shfl_up_sync(kFullMask, v.s[h], d);
  }
  if constexpr (!OpInfo<OP>::kIsLse) o.s[0] = A(0);
  return o;
}

// rows per thread: G = rows per 128-bit load, kLoads loads -> GL = 4, 8 or 16 consecutive rows.  The fixed cost
// per thread (segment lookup, block-wide segmented scan, emit) is what made this kernel issue-bound at one
// load per thread (119 instructions per row at fp32 H = 1); it is now amortised over up to 16 rows.
template <typename T, int HE>
struct FlatShape {
  static constexpr int E = 16 / (int)sizeof(T);
  static constexpr int G = E / HE;
  static constexpr int kLoads = G * 4 <= 16 ? 4 : 16 / G;
  static constexpr int GL = G * kLoads;
  static constexpr int R = kFlatThreads * GL;   // rows per tile
};

template <typename T, int HE, int OP>
__global__ void __launch_bounds__(kFlatThreads)
segreduce_flat_kernel(const T* __restrict__ data, const int64_t* __restrict__ ridx, const int64_t* __restrict__ off,
                      int64_t N, int64_t S,
                      T* __restrict__ out, typename Store<T>::Acc* __restrict__ head,
                      typename Store<T>::Acc* __restrict__ tail, int64_t* __restrict__ tail_seg, RedHeader* hdr,
                      int vector_loads) {
  using A = typename Store<T>::Acc;
  using St = State<A, HE, OP>;
  using Shape = FlatShape<T, HE>;
  constexpr bool kFast = sizeof(T) == 2;
  constexpr int E = Shape::E;                  // elements per 128-bit load
  constexpr int G = Shape::G;                  // rows per load
  constexpr int L = Shape::kLoads;             // loads per thread
  constexpr int GL = Shape::GL;                // rows per thread
  constexpr int R = Shape::R;                  // rows per tile
  constexpr int P = OpInfo<OP>::kParts;
  constexpr int SV = OpInfo<OP>::kIsLse ? 2 * HE : HE;   // scalars per partial state
  static_assert(kFlatThreads == kDecThreads, "tile_decode.cuh assumes 256 threads");
  __shared__ TileDecodeSmemT<GL> sm;
  __shared__ int s_wkey[kFlatWarps];
  __shared__ A s_wval[kFlatWarps][SV];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t tile = blockIdx.x;
  const int64_t row0 = tile * R;
  // rows past the last segment (sum of sizes < N) belong to nobody and are not reduced
  const int64_t covered = __ldg(off + S) < N ? __ldg(off + S) : N;
  const int nrows = (int)(row0 + R < covered ? R : covered - row0);
  if (nrows <= 0) {                             // CTA-uniform
    if (tid == 0) tail_seg[tile] = -1;
    return;
  }

  // ---- the thread's GL rows are requested FIRST (256-bit loads: one full sector per lane), so that the DRAM
  // latency overlaps the tile decode and its barriers -----------------------------------------------------
  const int tr0 = tid * GL;                     // tile-relative first row of this thread
  const bool vec = vector_loads && row0 + tr0 + GL <= N && tr0 < nrows;   // rows beyond `nrows` but inside N are ignored
  uint4 raw[L];
  if (vec) {
    const T* base = data + (row0 + tr0) * HE;
    if (vector_loads == 2) {
#pragma unroll
      for (int l = 0; l < L; l += 2)
        asm volatile("ld.global.nc.L1::no_allocate.v4.b64 {%0, %1, %2, %3}, [%4];"
                     : "=l"(*reinterpret_cast<unsigned long long*>(&raw[l].x)), "=l"(*reinterpret_cast<unsigned long long*>(&raw[l].z)),
                       "=l"(*reinterpret_cast<unsigned long long*>(&raw[l + 1].x)), "=l"(*reinterpret_cast<unsigned long long*>(&raw[l + 1].z))
                     : "l"(base + l * E));
    } else {
#pragma unroll
      for (int l = 0; l < L; ++l) raw[l] = __ldg(reinterpret_cast<const uint4*>(base + l * E));
    }
  }

  // ---- which segment owns each row of the tile (tile_decode.cuh) ---------------------------------
  GlobalOff g{off};
  const TileDecode dec = tile_decode<GL>(g, S, row0, nrows, sm);
  const bool staged = dec.staged;
  const int64_t first = dec.first;
  // tile-relative, clamped offsets: rel(k) = off[first + k] - row0 in [-1, R + 1]
  auto rel = [&](int k) -> int {
    if (staged) return sm.rel[k];
    int64_t d = __ldg(off + first + k) - row0;
    return d < -1 ? -1 : (d > R + 1 ? R + 1 : (int)d);
  };

  // ---- thread-local reduction of GL consecutive rows, cut at segment boundaries -----------------
  int sg[GL];                                   // owning segment (relative to `first`) of each row
  if (staged) {
#pragma unroll
    for (int q = 0; q < GL / 4; ++q) {
      const int4 v = reinterpret_cast<const int4*>(sm.seg)[tid * (GL / 4) + q];
      sg[4 * q] = v.x; sg[4 * q + 1] = v.y; sg[4 * q + 2] = v.z; sg[4 * q + 3] = v.w;
    }
  } else {                                      // runs of empty segments overflowed the stage: search per row
#pragma unroll
    for (int k = 0; k < GL; ++k)
      sg[k] = tr0 + k < nrows ? (int)(owner_search(g, S, row0 + tr0 + k) - first) : 0;
  }

  A ext = OP == RUA_MIN ? -inf_of<A>() : inf_of<A>();
  bool saw_nan = false;
  St firstRun, acc;
  acc.reset();
  firstRun.reset();
  int firstLo = -1;                             // the first CLOSED run of this thread (may need a carry-in)
  int closed = 0;
  int lo = -1;                                  // segment of the run being accumulated
  bool have = false;                            // acc holds at least one row
  auto seg_len = [&](int l) -> int64_t { return __ldg(off + first + l + 1) - __ldg(off + first + l); };
  auto close_run = [&]() {
    if (closed == 0) {
      firstRun = acc;
      firstLo = lo;
    } else {  // started and ended inside this thread: a complete segment
      A o[HE];
      acc.finalize(OP == RUA_MEAN ? seg_len(lo) : 1, o);
#pragma unroll
      for (int h = 0; h < HE; ++h) {
        if (OpInfo<OP>::kNeedsExt) saw_nan |= (o[h] != o[h]);
        out[(first + lo) * HE + h] = Store<T>::from_acc(o[h]);
      }
    }
    ++closed;
    acc.reset();
    have = false;
  };
#pragma unroll
  for (int l = 0; l < L; ++l) {
    const int rb = tr0 + l * G;                 // first row of this load
    if (rb < nrows) {
      A x[E];
      if (vec) {
        Store<T>::unpack(raw[l], x);
      } else {
#pragma unroll
        for (int k = 0; k < E; ++k) {
          const int64_t row = row0 + rb + k / HE;                      // optional row gather (scatter_*)
          x[k] = rb + k / HE < nrows ? Store<T>::to_acc(data[(ridx ? __ldg(ridx + row) : row) * HE + k % HE]) : A(0);
        }
      }
#pragma unroll
      for (int k = 0; k < G; ++k) {
        if (rb + k < nrows) {
          const int s_k = sg[l * G + k];
          if (s_k != lo) {
            if (have) close_run();
            lo = s_k;
          }
          acc.template add<kFast>(&x[k * HE]);
          have = true;
          if (OpInfo<OP>::kNeedsExt) {
#pragma unroll
            for (int h = 0; h < HE; ++h) ext = OP == RUA_MIN ? max_num(ext, x[k * HE + h]) : min_num(ext, x[k * HE + h]);
          }
        }
      }
    }
  }
  const int my_end = tr0 + GL < nrows ? tr0 + GL : nrows;  // one past this thread's last row
  if (have && rel(lo + 1) == my_end) close_run();         // the segment ends exactly with this thread
  // what is left in `acc` (if `have`) is an OPEN run of segment first+lo, continuing to the right
  int key = have ? lo : -1;
  St val = acc;

  // ---- block-wide segmented inclusive scan by key -----------------------------------------------
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int k2 = __shfl_up_sync(kFullMask, key, d);
    St v2 = flat_shfl_up<A, HE, OP>(val, d);
    if (lane >= d && k2 == key && key >= 0) flat_merge<A, HE, OP, kFast>(val, v2);
  }
  if (lane == 31) {
    s_wkey[warp] = key;
#pragma unroll
    for (int h = 0; h < HE; ++h) {
      s_wval[warp][h] = val.a[h];
      if constexpr (OpInfo<OP>::kIsLse) s_wval[warp][HE + h] = val.s[h];
    }
  }
  __syncthreads();
  if (warp == 0) {  // warp 0 turns the 8 warp totals into the carries entering each warp
    int wk = lane < kFlatWarps ? s_wkey[lane] : -1;
    St wv;
    wv.reset();
    if (lane < kFlatWarps) {
#pragma unroll
      for (int h = 0; h < HE; ++h) {
        wv.a[h] = s_wval[lane][h];
        if constexpr (OpInfo<OP>::kIsLse) wv.s[h] = s_wval[lane][HE + h];
      }
    }
#pragma unroll
    for (int d = 1; d < kFlatWarps; d <<= 1) {
      const int k2 = __shfl_up_sync(kFullMask, wk, d);
      St v2 = flat_shfl_up<A, HE, OP>(wv, d);
      if (lane >= d && k2 == wk && wk >= 0) flat_merge<A, HE, OP, kFast>(wv, v2);
    }
    // exclusive: warp w receives the inclusive total of warp w-1
    const int ck = __shfl_up_sync(kFullMask, wk, 1);
    St cv = flat_shfl_up<A, HE, OP>(wv, 1);
    if (lane < kFlatWarps) {
      s_wkey[lane] = lane == 0 ? -1 : ck;
#pragma unroll
      for (int h = 0; h < HE; ++h) {
        s_wval[lane][h] = cv.a[h];
        if constexpr (OpInfo<OP>::kIsLse) s_wval[lane][HE + h] = cv.s[h];
      }
    }
  }
  __syncthreads();
  const int ckey = s_wkey[warp];
  St cval;
  cval.reset();
  if (ckey >= 0) {
#pragma unroll
    for (int h = 0; h < HE; ++h) {
      cval.a[h] = s_wval[warp][h];
      if constexpr (OpInfo<OP>::kIsLse) cval.s[h] = s_wval[warp][HE + h];
    }
  }
  // equal keys are contiguous, so every lane whose key equals the carry's key is connected to the warp start
  if (key >= 0 && key == ckey) flat_merge<A, HE, OP, kFast>(val, cval);
  // exclusive value = block-wide inclusive value of the previous thread
  int ekey = __shfl_up_sync(kFullMask, key, 1);
  St eval = flat_shfl_up<A, HE, OP>(val, 1);
  if (lane == 0) {
    ekey = ckey;
    eval = cval;
  }

  // ---- emit -----------------------------------------------------------------------------------
  if (closed > 0) {  // first closed run: fold in what the threads before contributed to the same segment
    St v = firstRun;
    if (ekey == firstLo) flat_merge<A, HE, OP, kFast>(v, eval);
    const int64_t seg = first + firstLo;
    const int64_t beg = __ldg(off + seg);
    if (beg >= row0) {
      A o[HE];
      v.finalize(OP == RUA_MEAN ? __ldg(off + seg + 1) - beg : 1, o);
#pragma unroll
      for (int h = 0; h < HE; ++h) {
        if (OpInfo<OP>::kNeedsExt) saw_nan |= (o[h] != o[h]);
        out[seg * HE + h] = Store<T>::from_acc(o[h]);
      }
    } else {  // the segment began in an earlier tile: this is the tile's head piece
      store_partial<A, HE, OP>(head + tile * P * HE, HE, 0, v);
    }
  }
  const int last_thread = (nrows - 1) / GL;
  if (tid == last_thread) {
    int64_t spans = -1;
    if (key >= 0) {  // the tile ends inside a segment
      const int64_t seg = first + key;
      const int64_t beg = __ldg(off + seg);
      store_partial<A, HE, OP>((beg >= row0 ? tail : head) + tile * P * HE, HE, 0, val);
      if (beg >= row0) spans = seg;
    }
    tail_seg[tile] = spans;  // read by segreduce_span_kernel: the segment that starts here and runs on
  }

  if (OpInfo<OP>::kNeedsExt) {
    __shared__ unsigned long long s_key[kFlatWarps];
    __shared__ int s_nan;
    if (tid == 0) s_nan = 0;
    __syncthreads();
    unsigned long long okey = order_key(ext);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      unsigned long long o = __shfl_xor_sync(kFullMask, okey, d);
      okey = OP == RUA_MIN ? (o > okey ? o : okey) : (o < okey ? o : okey);
    }
    if (lane == 0) s_key[warp] = okey;
    if (saw_nan) s_nan = 1;
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < kFlatWarps; ++w) {
        unsigned long long o = s_key[w];
        okey = OP == RUA_MIN ? (o > okey ? o : okey) : (o < okey ? o : okey);
      }
      if (OP == RUA_MIN) atomicMax(&hdr->ext_key, okey); else atomicMin(&hdr->ext_key, okey);
      if (s_nan) atomicOr(&hdr->nan_flag, 1u);
    }
  }
}

// does a flat kernel exist for rows of `H` elements of this dtype?
bool flat_supported(int32_t dtype, int64_t H) {
  return H >= 1 && H <= vec_elems(dtype) && (H & (H - 1)) == 0;
}

int flat_rows_per_tile(int32_t dtype, int64_t H) {   // == FlatShape<T, H>::R
  const int g = vec_elems(dtype) / (int)H;
  return kFlatThreads * g * (g * 4 <= 16 ? 4 : 16 / g);
}

int flat_launch(int32_t dtype, int64_t H, int32_t op, const void* data, const int64_t* ridx, const int64_t* off,
                int64_t N, int64_t S, void* out, void* head, void* tail, int64_t* tail_seg, void* hdr,
                int vector_loads, int64_t tiles, cudaStream_t st) {
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    using A = typename Store<T>::Acc;
    return with_row_elems<T>(H, [&](auto he) {
      return with_op(op, [&](auto o) {
        segreduce_flat_kernel<T, decltype(he)::value, decltype(o)::value><<<(unsigned)tiles, kFlatThreads, 0, st>>>(
            (const T*)data, ridx, off, N, S, (T*)out, (A*)head, (A*)tail, tail_seg, (RedHeader*)hdr, vector_loads);
        return check_launch();
      });
    });
  });
}

}  // namespace rua
