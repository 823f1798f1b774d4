// K4s -- the SHORT instantiation of the segment-reduce main kernel (reduce_kernel.cuh): batches whose segments are a few
// rows long on average (sub-word -> word pooling with segment_mean, `.seg()` pieces; reference torchrua/reduce.py:34-61
// called from torchrua/segment.py:6-10).  Same chunking, partial pieces, span / patch kernels and determinism as the
// long-segment instance in reduce.cu; only the walk over the 8 loaded rows differs (one visit per row with a boundary
// test after it instead of one predicated sweep per run).  A separate translation unit so that the two families of
// instantiations compile in parallel.
#include "reduce_kernel.cuh"

namespace rua {

// average segment length (rows) below which the SHORT instance is used; RUA_SEG_SHORT_AVG / RUA_SEG_SHORT_LSE_AVG
// override (0 disables).  Measured on one B200, 1.04 M rows of 2 KB bf16 (profiles/r2_ops.md, "pieces" rows), % of the HBM
// copy peak, run-wise walk -> SHORT: mean U[1,4] 68 -> 86 (with the patch kernel fixed in both), pieces of 8: 87 = 87,
// pieces of 16: 91 > 84; logsumexp U[1,4] 56 -> 62, pieces of 8: 80 > 57 (its per-row online update costs more than
// the batch form of the run-wise walk as soon as whole batches of 8 rows fall inside one segment).
bool short_applies(int64_t N, int64_t S, int32_t op) {
  static const int64_t avg = knob("RUA_SEG_SHORT_AVG", 6);
  static const int64_t avg_lse = knob("RUA_SEG_SHORT_LSE_AVG", 4);
  const int64_t a = op == RUA_LOGSUMEXP ? avg_lse : avg;
  return a > 0 && S > 0 && N < a * S;
}

// vectorised (16-byte column vectors) instances only; the caller keeps the V = 1 fallback on the generic kernel
int short_launch(int32_t dtype, int32_t op, bool gather, bool packed, dim3 grid, int threads, const void* data,
                 const int64_t* ridx, const int64_t* off, int64_t N, int64_t S, int64_t H, int R, void* out, void* head,
                 void* tail, int64_t* tail_seg, void* hdr, int lanes_log2, int64_t chunks, cudaStream_t st) {
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    using A = typename Store<T>::Acc;
    return with_op(op, [&](auto o) {
      with_bool(gather, [&](auto g) {
        with_bool(packed, [&](auto pk) {
          segreduce_kernel<T, Store<T>::kVec, decltype(o)::value, decltype(g)::value, decltype(pk)::value, true>
              <<<grid, threads, 0, st>>>((const T*)data, ridx, off, N, S, H, R, (T*)out, (A*)head, (A*)tail, tail_seg,
                                         (RedHeader*)hdr, lanes_log2, chunks);
        });
      });
      return check_launch();
    });
  });
}

}  // namespace rua
