// K4 -- segment reduce (forward): sum / mean / prod / max / min / logsumexp per contiguous segment.
//
// Replaces (reference file:line): segment_max torchrua/reduce.py:34-36, segment_min :39-41,
// segment_sum :44-45, segment_mean :48-49, segment_prod :52-53, segment_logsumexp :56-61.
// The reference calls ATen segment_reduce (one thread per output, serial walk over the segment,
// accumulation in the storage dtype) and, for logsumexp, ~5 extra passes and 3 N x H temporaries.
//
// Design (HBM-bound: N*D bytes read once, S*D written once):
//   * the N rows are cut into fixed chunks of R rows, whatever the segment lengths -- a Zipf batch
//     (38 % of segments of length 1, 1 % of length 4096) is balanced by construction;
//   * a CTA owns (chunk, 128 column-vectors); a thread owns one 16-byte column vector and walks the
//     chunk's rows top to bottom, 8 independent 128-bit loads in flight, fp32 (fp64) accumulators
//     in registers; lanes map to columns, so every load/store is fully coalesced along H;
//   * segment boundaries are uniform across the CTA (all threads see the same rows): a segment
//     that starts and ends inside the chunk is finalised and stored directly; the pieces of a
//     segment that crosses chunk boundaries go to a small fp32 scratch (at most 2 rows per chunk)
//     and are combined IN CHUNK ORDER by a second tiny kernel -- deterministic, no float atomics;
//   * logsumexp is one pass (online max / rescaled sum, one exp per element);
//   * the reference's `initial` quirks (SURVEY.md 8c hazard 3) cost no extra pass: the global
//     extreme is reduced on the fly (one atomic per CTA) and a NaN is detected at emit time; a
//     third tiny kernel patches empty segments and applies the NaN poisoning.
#include "reduce_kernel.cuh"

namespace rua {

// combine the pieces of every segment that crosses a chunk boundary, in chunk order
template <typename T, int V, int OP>
__global__ void __launch_bounds__(kRedThreads)
segreduce_span_kernel(const int64_t* __restrict__ off, int64_t N, int64_t S, int64_t H, int R,
                      T* __restrict__ out, const typename Store<T>::Acc* __restrict__ head,
                      const typename Store<T>::Acc* __restrict__ tail, const int64_t* __restrict__ tail_seg,
                      RedHeader* hdr) {
  using A = typename Store<T>::Acc;
  constexpr bool kFast = sizeof(T) == 2;
  constexpr int P = OpInfo<OP>::kParts;
  const int64_t b = blockIdx.x;            // boundary between chunk b and b+1
  if ((b + 1) * R >= N) return;
  // the main kernel recorded the segment that starts in chunk b and continues past it (-1: none; a
  // segment that merely passes THROUGH chunk b is finished by the boundary where it started)
  const int64_t s = __ldg(tail_seg + b);
  if (s < 0 || s >= S) return;
  const int64_t beg = __ldg(off + s), end = __ldg(off + s + 1);
  const int64_t col = ((int64_t)blockIdx.y * blockDim.x + threadIdx.x) * V;
  if (col >= H) return;
  State<A, V, OP> acc, piece;
  load_partial<A, V, OP>(tail + b * P * H, H, col, acc);
  for (int64_t c = b + 1;; ++c) {
    load_partial<A, V, OP>(head + c * P * H, H, col, piece);
    acc.template merge<kFast>(piece);
    if (end <= (c + 1) * R) break;
  }
  A o[V];
  acc.template finalize<kFast>(end - beg, o);
  if (OpInfo<OP>::kNeedsExt && acc.any_nan_out(o)) atomicOr(&hdr->nan_flag, 1u);
  store_vec<T, V>(out + s * H + col, o);
}

// empty segments and NaN poisoning (reference `initial` semantics, reduce.py:35,40,57-61).  A lane tests one segment
// (coalesced offset loads: S threads, not S x H / V -- with sub-word pooling S is 40 % of N and the old one-thread-per-
// output-vector form cost a fifth of the whole reduction); the rows that do need a value are then filled by the whole warp.
template <typename T, int V, int OP>
__global__ void __launch_bounds__(256)
segreduce_patch_kernel(const int64_t* __restrict__ off, int64_t S, int64_t H, T* __restrict__ out,
                       const RedHeader* __restrict__ hdr) {
  using A = typename Store<T>::Acc;
  const int lane = threadIdx.x & 31;
  const int64_t s0 = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32;
  if (s0 >= S) return;                                   // warp-uniform
  const bool poison = OpInfo<OP>::kNeedsExt && hdr->nan_flag != 0;
  const int64_t s = s0 + lane;
  const bool flag = s < S && (poison || __ldg(off + s + 1) == __ldg(off + s));
  unsigned todo = __ballot_sync(kFullMask, flag);
  if (todo == 0u) return;
  A val;
  if (poison) val = nan_of<A>();
  else if (OP == RUA_SUM || OP == RUA_MEAN) val = A(0);
  else if (OP == RUA_PROD) val = A(1);
  else val = key_to(A(0), hdr->ext_key);
  A o[V];
#pragma unroll
  for (int v = 0; v < V; ++v) o[v] = val;
  const int64_t hv = H / V;
  if (hv == 1) {                                         // one vector per row: every lane fills its own segment
    if (flag) store_vec<T, V>(out + s * H, o);
    return;
  }
  while (todo) {
    const int b = __ffs(todo) - 1;
    todo &= todo - 1u;
    T* row = out + (s0 + b) * H;
    for (int64_t c = lane; c < hv; c += 32) store_vec<T, V>(row + c * V, o);
  }
}

__global__ void segreduce_init_kernel(RedHeader* hdr, int is_min) {
  hdr->ext_key = is_min ? 0ull : ~0ull;
  hdr->nan_flag = 0u;
}

static inline size_t tail_seg_bytes(int64_t chunks) { return ((size_t)chunks * sizeof(int64_t) + 15) & ~(size_t)15; }

struct RedPlan {
  int R;
  int64_t chunks;
  int threads;
  int64_t col_tiles;
  int vec;
  size_t part_elems;  // per partial array
  bool flat;          // narrow rows: rows-on-lanes kernel
  int vector_loads;
  int32_t dtype;
  int lanes_log2;     // main kernel: 2^lanes_log2 threads per row ...
  int main_threads;   // ... in CTAs of this many threads (several chunks per CTA when rows are short)
};

static RedPlan plan_reduce(int64_t N, int64_t H, int32_t dtype, int32_t op, const void* data, const void* out) {
  RedPlan p;
  p.flat = false;
  p.vector_loads = 0;
  p.dtype = dtype;
  if (flat_supported(dtype, H)) {  // narrow rows: rows map to lanes (reduce_flat.cu)
    p.flat = true;
    p.vector_loads = (((uintptr_t)data) & 31u) == 0 ? 2 : ((((uintptr_t)data) & 15u) == 0 ? 1 : 0);   // 256- / 128-bit loads
    p.vec = 1;
    p.threads = 32;
    p.lanes_log2 = 5;
    p.main_threads = 32;
    p.col_tiles = 1;
    p.R = flat_rows_per_tile(dtype, H);
    p.chunks = N > 0 ? ceil_div(N, p.R) : 0;
    p.part_elems = (size_t)p.chunks * (size_t)H * (op == RUA_LOGSUMEXP ? 2 : 1);
    return p;
  }
  int full = vec_elems(dtype);
  bool aligned = (H % full == 0) && (((uintptr_t)data | (uintptr_t)out) & 15u) == 0;
  p.vec = aligned ? full : 1;
  int64_t hv = H / p.vec;
  int threads = 32;
  while (threads < kRedThreads && threads < hv) threads <<= 1;
  p.threads = threads;
  p.col_tiles = ceil_div(hv, threads);
  // rows shorter than a warp (hv < 32 vectors): pack kRedThreads / lanes chunks into one CTA
  int lanes = threads, lg = 0;
  if (hv < 32 && p.vec > 1) { lanes = 1; while (lanes < hv) lanes <<= 1; }
  while ((1 << lg) < lanes) ++lg;
  p.lanes_log2 = lg;
  p.main_threads = (hv < 32 && p.vec > 1) ? kRedThreads : threads;
  const int cpc = p.main_threads / lanes;   // chunks per CTA
  // largest chunk that still gives every SM ~8 CTAs
  int R = 256;
  while (R > 32 && ceil_div(ceil_div(N, R), cpc) * p.col_tiles < (int64_t)kNumSMs * 8) R >>= 1;
  p.R = R;
  p.chunks = N > 0 ? ceil_div(N, R) : 0;
  p.part_elems = (size_t)p.chunks * (size_t)H * (op == RUA_LOGSUMEXP ? 2 : 1);
  return p;
}

template <typename T, int V, int OP>
static int run_reduce(const RedPlan& p, const void* data, const int64_t* ridx, const int64_t* off, int64_t N, int64_t S,
                      int64_t H, void* out, void* ws, cudaStream_t st) {
  using A = typename Store<T>::Acc;
  RedHeader* hdr = (RedHeader*)ws;
  int64_t* tail_seg = (int64_t*)((char*)ws + sizeof(RedHeader));
  A* head = (A*)((char*)ws + sizeof(RedHeader) + tail_seg_bytes(p.chunks));
  A* tail = head + p.part_elems;
  int rc;
  if (OpInfo<OP>::kNeedsExt) {
    segreduce_init_kernel<<<1, 1, 0, st>>>(hdr, OP == RUA_MIN);
    if ((rc = check_launch())) return rc;
  }
  if (p.flat && !ridx && p.vector_loads >= 1 && warpseg_applies(N, S)) {
    // many short segments of narrow rows: every segment is finished by the lane that owns it (no pieces to merge);
    // empty segments of sum / mean / prod are written inline, so only max / min / logsumexp need the patch pass
    if ((rc = warpseg_launch(p.dtype, H, OP, data, off, N, S, out, hdr, st))) return rc;
    if (!OpInfo<OP>::kNeedsExt) return RUA_OK;
    segreduce_patch_kernel<T, V, OP><<<(unsigned)ceil_div(S, 256), 256, 0, st>>>(off, S, H, (T*)out, hdr);
    return check_launch();
  }
  if (N > 0) {
    if (p.col_tiles > 65535) return RUA_ERR_UNSUPPORTED;
    dim3 grid((unsigned)ceil_div(p.chunks, p.main_threads >> p.lanes_log2), (unsigned)p.col_tiles);
    if (p.flat) {
      rc = flat_launch(p.dtype, H, OP, data, ridx, off, N, S, out, head, tail, tail_seg, hdr, ridx ? 0 : p.vector_loads, p.chunks, st);
      if (rc) return rc;
    } else {
      auto launch = [&](auto gather, auto packed) {
        segreduce_kernel<T, V, OP, decltype(gather)::value, decltype(packed)::value><<<grid, p.main_threads, 0, st>>>(
            (const T*)data, ridx, off, N, S, H, p.R, (T*)out, head, tail, tail_seg, hdr, p.lanes_log2, p.chunks);
      };
      const bool packed = (p.main_threads >> p.lanes_log2) > 1;
      if constexpr (V > 1) {   // packing exists for the vectorised instances only (V = 1 is the odd-alignment fallback)
        if (short_applies(N, S, OP)) {
          rc = short_launch(p.dtype, OP, ridx != nullptr, packed, grid, p.main_threads, data, ridx, off, N, S, H, p.R, out,
                            head, tail, tail_seg, hdr, p.lanes_log2, p.chunks, st);
          if (rc) return rc;
        } else {
          with_bool(ridx != nullptr, [&](auto g) { with_bool(packed, [&](auto pk) { launch(g, pk); }); });
        }
      } else {
        with_bool(ridx != nullptr, [&](auto g) { launch(g, std::false_type{}); });
      }
      if ((rc = check_launch())) return rc;
    }
    if (p.chunks > 1) {
      dim3 g2((unsigned)(p.chunks - 1), (unsigned)p.col_tiles);
      segreduce_span_kernel<T, V, OP><<<g2, p.threads, 0, st>>>(off, N, S, H, p.R, (T*)out, head, tail, tail_seg, hdr);
      if ((rc = check_launch())) return rc;
    }
  }
  segreduce_patch_kernel<T, V, OP><<<(unsigned)ceil_div(S, 256), 256, 0, st>>>(off, S, H, (T*)out, hdr);
  return check_launch();
}

}  // namespace rua

using namespace rua;

extern "C" {

size_t rua_segment_reduce_workspace_bytes(int64_t N, int64_t S, int64_t H, int32_t dtype, int32_t op) {
  (void)S;
  RedPlan p = plan_reduce(N, H, dtype, op, nullptr, nullptr);
  // the vector width may drop to 1 for misaligned views; that only changes threads/tiles, not R... be safe:
  RedPlan q = plan_reduce(N, H, dtype, op, (const void*)1, nullptr);
  size_t elems = p.part_elems > q.part_elems ? p.part_elems : q.part_elems;
  size_t acc = acc_bytes(dtype);
  size_t chunks = p.chunks > q.chunks ? p.chunks : q.chunks;
  return sizeof(RedHeader) + tail_seg_bytes(chunks) + 2 * elems * acc + 64;
}

int rua_segment_reduce(const void* data, const int64_t* off, int64_t N, int64_t S, int64_t H, int32_t dtype,
                       int32_t op, void* out, void* ws, size_t ws_bytes, rua_stream_t stream) {
  return rua_segment_reduce_gather(data, nullptr, off, N, S, H, dtype, op, out, ws, ws_bytes, stream);
}

int rua_segment_reduce_gather(const void* data, const int64_t* row_index, const int64_t* off, int64_t N, int64_t S,
                              int64_t H, int32_t dtype, int32_t op, void* out, void* ws, size_t ws_bytes,
                              rua_stream_t stream) {
  const int64_t* ridx = row_index;
  if (N < 0 || S < 0 || H < 0) return RUA_ERR_INVALID;
  if (S == 0 || H == 0) return RUA_OK;
  if (!off || !out || !ws || (N > 0 && !data)) return RUA_ERR_INVALID;
  if (op < RUA_SUM || op > RUA_LOGSUMEXP) return RUA_ERR_INVALID;
  if (dtype < RUA_F32 || dtype > RUA_BF16) return RUA_ERR_UNSUPPORTED;
  RedPlan p = plan_reduce(N, H, dtype, op, data, out);
  if (ws_bytes < sizeof(RedHeader) + tail_seg_bytes(p.chunks) + 2 * p.part_elems * acc_bytes(dtype)) return RUA_ERR_WORKSPACE;
  if (((uintptr_t)ws & 15u) != 0) return RUA_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    return with_op(op, [&](auto o) {
      constexpr int OP = decltype(o)::value;
      if (p.vec == 1) return run_reduce<T, 1, OP>(p, data, ridx, off, N, S, H, out, ws, st);
      return run_reduce<T, Store<T>::kVec, OP>(p, data, ridx, off, N, S, H, out, ws, st);
    });
  });
}

}  // extern "C"
