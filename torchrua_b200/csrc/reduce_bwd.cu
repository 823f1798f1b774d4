// K4' -- segment reduce backward (the `_backward` twin of reduce.cu).
//
// Semantics follow what autograd records for the reference (ATen SegmentReduceBackward0 for
// torchrua/reduce.py:34-53, and the composite graph of segment_logsumexp reduce.py:56-61):
//   sum  : grad[r] = g[s]                     mean : g[s] / len[s]
//   max/min : g[s] / (#ties) for every row equal to the output (NaN rows count as ties), else 0
//   prod : g[s] * out[s] / x  (x != 0, not NaN), else g[s] * product of the other rows
//   logsumexp : g[s] * exp(x - out[s])        (m is detached in the reference, so this is exact)
// Same decomposition as the forward pass: fixed row chunks x 128 column vectors per CTA, segment
// boundaries uniform across the CTA, 16-byte coalesced loads/stores along H.  max/min need the tie
// counts first: one extra read of the data with integer atomics (order independent => deterministic).
// Batches of very short segments (sub-word pieces: N <= 8 S) use the INLINE instances instead: a segment that lies inside
// one chunk is counted by the thread that owns it right before it writes the gradient (a second look at rows that are
// still in L1: no atomics, no S x H counter array to clear, fill and read back), and only segments that CROSS a chunk
// boundary go through the count pass, into one slot of H counters per chunk (at most one crossing segment starts in
// any chunk).  Kept as separate instances: folded into one kernel the extra code cost the long-segment case 5-25 %.
#include "reduce_common.cuh"

namespace rua {

constexpr int kBwdUnroll = 4;
constexpr int kTieInlineAvg = 8;   // max / min backward: average segment length up to which the INLINE instances run

template <typename T, int V>
__device__ __forceinline__ void load_acc(const T* p, typename Store<T>::Acc* x) {
  Raw<T, V> w;
  if constexpr (V == 1) w.r = *p; else w.r = *reinterpret_cast<const uint4*>(p);
  unpack_raw<T, V>(w, x);
}

// walks the chunk's rows and keeps (segment, begin, end) current; uniform across the CTA
struct SegCursor {
  const int64_t* __restrict__ off;
  int64_t S, s, beg, end;
  __device__ __forceinline__ void init(const int64_t* o, int64_t S_, int64_t row) {
    off = o; S = S_;
    GlobalOff g{o};
    s = owner_search(g, S_, row);
    beg = __ldg(o + s);
    end = __ldg(o + s + 1);
    if (row >= end) { s = S_; }  // rows past the last segment (sum of sizes < N)
  }
  // returns true when the segment changed
  __device__ __forceinline__ bool seek(int64_t row) {
    bool moved = false;
    while (s < S && row >= end) {
      ++s;
      beg = end;
      end = s < S ? __ldg(off + s + 1) : beg;
      moved = true;
    }
    return moved;
  }
  __device__ __forceinline__ bool valid() const { return s < S; }
};

// INLINE instance: only the chunk-crossing segments, counters keyed by the chunk the segment starts in
template <typename T, int V, int OP>
__global__ void __launch_bounds__(kRedThreads)
tie_count_crossing_kernel(const T* __restrict__ data, const T* __restrict__ out, const int64_t* __restrict__ off, int64_t N,
                          int64_t S, int64_t H, int R, int* __restrict__ counts, int lanes_log2) {
  using A = typename Store<T>::Acc;
  const int lanes = 1 << lanes_log2;
  const int64_t chunk = (int64_t)blockIdx.x * (blockDim.x >> lanes_log2) + (threadIdx.x >> lanes_log2);
  const int64_t col = ((int64_t)blockIdx.y * lanes + (threadIdx.x & (lanes - 1))) * V;
  const int64_t row0 = chunk * R;
  const bool active = col < H && row0 < N;
  const int64_t row1 = row0 + R < N ? row0 + R : N;
  if (row0 >= N) return;
  SegCursor cur;
  cur.init(off, S, row0);
  int64_t row = row0;
  while (row < row1) {
    cur.seek(row);
    if (!cur.valid()) break;
    const int64_t lo = cur.beg > row0 ? cur.beg : row0, hi = cur.end < row1 ? cur.end : row1;
    if ((cur.beg < row0 || cur.end > row1) && active) {      // this chunk's share of a crossing segment's ties
      A o[V];
      int cnt[V];
      load_acc<T, V>(out + cur.s * H + col, o);
#pragma unroll
      for (int v = 0; v < V; ++v) cnt[v] = 0;
      for (int64_t q = lo; q < hi; ++q) {
        A x[V];
        load_acc<T, V>(data + q * H + col, x);
#pragma unroll
        for (int v = 0; v < V; ++v) cnt[v] += (x[v] != x[v] || x[v] == o[v]) ? 1 : 0;
      }
      int* slot = counts + (cur.beg / R) * H + col;
#pragma unroll
      for (int v = 0; v < V; ++v) if (cnt[v]) atomicAdd(slot + v, cnt[v]);
    }
    row = hi;                                                // segments inside the chunk: counted by the gradient kernel
  }
}

template <typename T, int V, int OP>
__global__ void __launch_bounds__(kRedThreads)
tie_count_kernel(const T* __restrict__ data, const T* __restrict__ out, const int64_t* __restrict__ off, int64_t N,
                 int64_t S, int64_t H, int R, int* __restrict__ counts, int lanes_log2) {
  using A = typename Store<T>::Acc;
  // 2^lanes_log2 threads span one row; short rows: the CTA hosts several chunks side by side (see reduce.cu)
  const int lanes = 1 << lanes_log2;
  const int64_t chunk = (int64_t)blockIdx.x * (blockDim.x >> lanes_log2) + (threadIdx.x >> lanes_log2);
  const int64_t col = ((int64_t)blockIdx.y * lanes + (threadIdx.x & (lanes - 1))) * V;
  const int64_t row0 = chunk * R;
  const bool active = col < H && row0 < N;
  const int64_t row1 = row0 + R < N ? row0 + R : N;
  if (row0 >= N) return;
  SegCursor cur;
  cur.init(off, S, row0);
  A o[V];
  int cnt[V];
#pragma unroll
  for (int v = 0; v < V; ++v) cnt[v] = 0;
  if (active && cur.valid()) load_acc<T, V>(out + cur.s * H + col, o);
  for (int64_t row = row0; row < row1; ++row) {
    int64_t prev = cur.s;
    if (cur.seek(row)) {
      if (active) {
#pragma unroll
        for (int v = 0; v < V; ++v) { if (cnt[v]) atomicAdd(counts + prev * H + col + v, cnt[v]); cnt[v] = 0; }
        if (cur.valid()) load_acc<T, V>(out + cur.s * H + col, o);
      }
    }
    if (!cur.valid()) break;
    if (active) {
      A x[V];
      load_acc<T, V>(data + row * H + col, x);
#pragma unroll
      for (int v = 0; v < V; ++v) cnt[v] += (x[v] != x[v] || x[v] == o[v]) ? 1 : 0;
    }
  }
  if (active && cur.valid()) {
#pragma unroll
    for (int v = 0; v < V; ++v) if (cnt[v]) atomicAdd(counts + cur.s * H + col + v, cnt[v]);
  }
}

template <typename T, int V, int OP, bool INLINE = false>
__global__ void __launch_bounds__(kRedThreads)
segreduce_bwd_kernel(const T* __restrict__ gout, const T* __restrict__ out, const T* __restrict__ data,
                     const int64_t* __restrict__ off, int64_t N, int64_t S, int64_t H, int R,
                     T* __restrict__ grad, const int* __restrict__ counts, int lanes_log2) {
  using A = typename Store<T>::Acc;
  constexpr bool kNeedsX = OP == RUA_MAX || OP == RUA_MIN || OP == RUA_PROD || OP == RUA_LOGSUMEXP;
  constexpr bool kNeedsOut = kNeedsX;
  const int lanes = 1 << lanes_log2;
  const int64_t chunk = (int64_t)blockIdx.x * (blockDim.x >> lanes_log2) + (threadIdx.x >> lanes_log2);
  const int64_t col = ((int64_t)blockIdx.y * lanes + (threadIdx.x & (lanes - 1))) * V;
  const int64_t row0 = chunk * R;
  if (col >= H || row0 >= N) return;
  const int64_t row1 = row0 + R < N ? row0 + R : N;
  SegCursor cur;
  cur.init(off, S, row0);
  A g[V], o[V], c[V];
  // INLINE (segments of a few rows): the gradient / output rows of the NEXT segment are requested while the current one is
  // being written -- otherwise every boundary (one per 2-3 rows) exposes a dependent DRAM load
  Raw<T, V> next_g, next_o;
  int64_t next_s = -1;
  auto load_seg = [&]() {
    if constexpr (INLINE) {
      if (next_s == cur.s) {
        unpack_raw<T, V>(next_g, g);
        unpack_raw<T, V>(next_o, o);
      } else {
        load_acc<T, V>(gout + cur.s * H + col, g);
        load_acc<T, V>(out + cur.s * H + col, o);
      }
      next_s = cur.s + 1;
      if (next_s < S) {
        load_raw<T, V>(gout + next_s * H + col, next_g);
        load_raw<T, V>(out + next_s * H + col, next_o);
      }
    } else {
      load_acc<T, V>(gout + cur.s * H + col, g);
      if (kNeedsOut) load_acc<T, V>(out + cur.s * H + col, o);
    }
    if (OP == RUA_MEAN) {
      A inv = A(1) / (A)(cur.end - cur.beg);
#pragma unroll
      for (int v = 0; v < V; ++v) g[v] *= inv;
    }
    if (OP == RUA_MAX || OP == RUA_MIN) {
      if constexpr (INLINE) {
        int n[V];
        if (cur.end - cur.beg == 1) {                  // a single row is its own extreme
#pragma unroll
          for (int v = 0; v < V; ++v) n[v] = 1;
        } else if (cur.beg >= row0 && cur.end <= row1) {
          // inside this chunk: count the ties here (the loop below reads the same rows again a moment later: L1 hits)
#pragma unroll
          for (int v = 0; v < V; ++v) n[v] = 0;
          for (int64_t q = cur.beg; q < cur.end; ++q) {
            A x[V];
            load_acc<T, V>(data + q * H + col, x);
#pragma unroll
            for (int v = 0; v < V; ++v) n[v] += (x[v] != x[v] || x[v] == o[v]) ? 1 : 0;
          }
        } else {
#pragma unroll
          for (int v = 0; v < V; ++v) n[v] = counts[(cur.beg / R) * H + col + v];
        }
#pragma unroll
        for (int v = 0; v < V; ++v) c[v] = n[v] > 1 ? g[v] / (A)n[v] : g[v];
      } else {
#pragma unroll
        for (int v = 0; v < V; ++v) {
          int n = counts[cur.s * H + col + v];
          c[v] = n > 1 ? g[v] / (A)n : g[v];
        }
      }
    }
  };
  if (cur.valid()) load_seg();
  for (int64_t r = row0; r < row1; r += kBwdUnroll) {
    Raw<T, V> raw[kBwdUnroll];
    if (kNeedsX) {
#pragma unroll
      for (int k = 0; k < kBwdUnroll; ++k)
        if (r + k < row1) load_raw<T, V>(data + (r + k) * H + col, raw[k]);
    }
#pragma unroll
    for (int k = 0; k < kBwdUnroll; ++k) {
      const int64_t row = r + k;
      if (row >= row1) break;
      if (cur.seek(row) && cur.valid()) load_seg();
      A y[V];
      if (!cur.valid()) {
#pragma unroll
        for (int v = 0; v < V; ++v) y[v] = A(0);
      } else if (OP == RUA_SUM || OP == RUA_MEAN) {
#pragma unroll
        for (int v = 0; v < V; ++v) y[v] = g[v];
      } else {
        A x[V];
        unpack_raw<T, V>(raw[k], x);
#pragma unroll
        for (int v = 0; v < V; ++v) {
          if (OP == RUA_MAX || OP == RUA_MIN) {
            y[v] = (x[v] != x[v] || x[v] == o[v]) ? c[v] : A(0);
          } else if (OP == RUA_LOGSUMEXP) {
            y[v] = g[v] * exp_acc<false>(x[v] - o[v]);
          } else {  // prod
            if (x[v] != x[v] || x[v] == A(0)) {
              A ex = A(1);
              for (int64_t q = cur.beg; q < cur.end; ++q)
                if (q != row) ex *= Store<T>::to_acc(data[q * H + col + v]);
              y[v] = g[v] * ex;
            } else {
              y[v] = g[v] * o[v] / x[v];
            }
          }
        }
      }
      store_vec<T, V>(grad + row * H + col, y);
    }
  }
}

template <typename T, int V, int OP>
static int run_bwd(const void* gout, const void* out, const void* data, const int64_t* off, int64_t N, int64_t S,
                   int64_t H, void* grad, void* ws, cudaStream_t st) {
  int64_t hv = H / V;
  int threads = 32;
  while (threads < kRedThreads && threads < hv) threads <<= 1;
  int64_t col_tiles = ceil_div(hv, threads);
  if (col_tiles > 65535) return RUA_ERR_UNSUPPORTED;
  int lanes = threads;
  if (hv < 32) { lanes = 1; while (lanes < hv) lanes <<= 1; threads = kRedThreads; }   // short rows: chunks side by side
  int lg = 0;
  while ((1 << lg) < lanes) ++lg;
  const int cpc = threads / lanes;
  int R = 128;
  while (R > 16 && ceil_div(ceil_div(N, R), cpc) * col_tiles < (int64_t)kNumSMs * 8) R >>= 1;
  dim3 grid((unsigned)ceil_div(ceil_div(N, R), cpc), (unsigned)col_tiles);
  int rc;
  int* counts = nullptr;
  if constexpr (OP == RUA_MAX || OP == RUA_MIN) {
    counts = (int*)ws;
    if (N <= (int64_t)kTieInlineAvg * S) {          // very short segments: ties counted inside the gradient kernel
      const int64_t chunks = ceil_div(N, R);
      if ((rc = check_cuda(cudaMemsetAsync(counts, 0, (size_t)chunks * H * sizeof(int), st)))) return rc;
      tie_count_crossing_kernel<T, V, OP><<<grid, threads, 0, st>>>((const T*)data, (const T*)out, off, N, S, H, R, counts, lg);
      if ((rc = check_launch())) return rc;
      segreduce_bwd_kernel<T, V, OP, true><<<grid, threads, 0, st>>>((const T*)gout, (const T*)out, (const T*)data, off, N,
                                                                     S, H, R, (T*)grad, counts, lg);
      return check_launch();
    }
    if ((rc = check_cuda(cudaMemsetAsync(counts, 0, (size_t)S * H * sizeof(int), st)))) return rc;
    tie_count_kernel<T, V, OP><<<grid, threads, 0, st>>>((const T*)data, (const T*)out, off, N, S, H, R, counts, lg);
    if ((rc = check_launch())) return rc;
  }
  segreduce_bwd_kernel<T, V, OP><<<grid, threads, 0, st>>>((const T*)gout, (const T*)out, (const T*)data, off, N, S,
                                                           H, R, (T*)grad, counts, lg);
  return check_launch();
}

}  // namespace rua

using namespace rua;

extern "C" {

size_t rua_segment_reduce_backward_workspace_bytes(int64_t N, int64_t S, int64_t H, int32_t dtype, int32_t op) {
  (void)dtype;
  if (op == RUA_MAX || op == RUA_MIN) {
    // tie counters: H per segment, or (very short segments) H per chunk of >= 16 rows
    const size_t slots = N <= (int64_t)kTieInlineAvg * S ? (size_t)(N / 16 + 1) : (size_t)S;
    return slots * (size_t)H * sizeof(int) + 16;
  }
  return 16;
}

int rua_segment_reduce_backward(const void* grad_out, const void* out, const void* data, const int64_t* off,
                                int64_t N, int64_t S, int64_t H, int32_t dtype, int32_t op, void* grad_data,
                                void* ws, size_t ws_bytes, rua_stream_t stream) {
  if (N < 0 || S < 0 || H < 0) return RUA_ERR_INVALID;
  if (N == 0 || H == 0) return RUA_OK;
  if (op < RUA_SUM || op > RUA_LOGSUMEXP) return RUA_ERR_INVALID;
  if (dtype < RUA_F32 || dtype > RUA_BF16) return RUA_ERR_UNSUPPORTED;
  if (!grad_data) return RUA_ERR_INVALID;
  if (S == 0)   // no segment owns a row: the gradient is zero, and nothing else is read (the forward's output is empty)
    return check_cuda(cudaMemsetAsync(grad_data, 0, (size_t)N * H * (16 / vec_elems(dtype)), (cudaStream_t)stream));
  if (!grad_out || !out || !data || !off) return RUA_ERR_INVALID;
  if (ws_bytes < rua_segment_reduce_backward_workspace_bytes(N, S, H, dtype, op) - 16) return RUA_ERR_WORKSPACE;
  if ((op == RUA_MAX || op == RUA_MIN) && !ws) return RUA_ERR_INVALID;
  uintptr_t a = (uintptr_t)grad_out | (uintptr_t)out | (uintptr_t)data | (uintptr_t)grad_data;
  bool vec = (H % vec_elems(dtype) == 0) && (a & 15u) == 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (H == 1 && warpseg_applies(N, S) && (((uintptr_t)data | (uintptr_t)grad_data) & 15u) == 0)
    return warpseg_bwd_launch(dtype, H, op, grad_out, out, data, off, N, S, grad_data, st);
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    return with_op(op, [&](auto o) {
      constexpr int OP = decltype(o)::value;
      if (!vec) return run_bwd<T, 1, OP>(grad_out, out, data, off, N, S, H, grad_data, ws, st);
      return run_bwd<T, Store<T>::kVec, OP>(grad_out, out, data, off, N, S, H, grad_data, ws, st);
    });
  });
}

}  // extern "C"
