/*
 * rua_b200.h -- C ABI of the B200-native (sm_100a) ragged-sequence kernels.
 *
 * The reference (speedcell4/torchrua v0.5.1) is pure Python over stock ATen ops and has NO native
 * plugin / FFI interface of its own (SURVEY.md 8b).  This header therefore *defines* the boundary a
 * maintainer would bind: one entry point per kernel family, each citing the reference functions
 * whose bodies it replaces.  The Python mirror of the reference API (package torchrua_b200) calls
 * these through ctypes; INTEGRATION.md shows the stub for binding them from the reference itself.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross the boundary;
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - the caller owns and allocates every buffer, including workspaces (query the *_workspace_bytes
 *     functions); kernels are stateless, enqueue on `stream` and never synchronise;
 *   - return value: 0 on success, <0 on error (rua_error_string); nothing throws across the ABI;
 *   - int64 metadata everywhere, exactly like the reference (torchrua/layout/cat.py:75,
 *     torchrua/core/view.py:15).
 *
 * Notation: B sequences with base lengths len[i]; off = exclusive prefix sum of len (B+1 entries);
 * T = max len; batch_sizes bs[t] = #{i: len[i] > t}; poff = exclusive prefix sum of bs (T+1
 * entries); sorted = argsort-descending permutation, unsorted = its inverse.
 * Row of token (i,t):  C: off[i]+t   L: i*W+t   R: i*W+(W-len[i])+t   P: poff[t]+unsorted[i]
 * (torchrua/core/get.py:21-79, torchrua/layout/{cat,left,right,pack}.py).
 */
#ifndef RUA_B200_H_
#define RUA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* rua_stream_t; /* a cudaStream_t */

enum rua_status {
  RUA_OK = 0,
  RUA_ERR_INVALID = -1,     /* bad argument (null pointer, negative size, bad enum, misalignment) */
  RUA_ERR_WORKSPACE = -2,   /* workspace too small */
  RUA_ERR_UNSUPPORTED = -3, /* size / dtype outside what the kernels implement */
  RUA_ERR_CUDA = -4         /* a CUDA runtime call failed; see rua_last_cuda_error() */
};

enum rua_layout { RUA_CAT = 0, RUA_LEFT = 1, RUA_PACK = 2, RUA_RIGHT = 3 };

/* how one side's per-sequence lengths derive from the base lengths */
enum rua_len_xform {
  RUA_LEN_SAME = 0,  /* len'[i] = len[i]                                   (conversions, rev, roll) */
  RUA_LEN_CONST = 1, /* len'[i] = arg                                      (head(n), last)          */
  RUA_LEN_MINUS = 2  /* len'[i] = len[i] - arg                             (trunc((a,b)), arg=a+b)  */
};

/* token map dst t_d -> src t_s (validity: 0 <= t_s < len_src[i]) */
enum rua_tmap {
  RUA_MAP_SHIFT = 0, /* t_s = t_d + arg                 identity / trunc / head and their inverses */
  RUA_MAP_REV = 1,   /* t_s = len[i] - 1 - t_d          rev, last (torchrua/select/rev.py, last.py) */
  RUA_MAP_ROLL = 2   /* t_s = (t_d - arg) mod len[i]    roll (torchrua/select/roll.py:11)           */
};

enum rua_pad {
  RUA_PAD_FILL = 0, /* padding / unmapped rows receive the fill pattern */
  RUA_PAD_ROW0 = 1, /* ... receive a copy of flat source row 0 (L/R.roll quirk, select/roll.py:19-34) */
  RUA_PAD_WRAP = 2  /* FILL, except that source position -1 wraps like a negative Python index: what
                       last() / segment_last return for an EMPTY sequence (select/last.py:11-13)   */
};

enum rua_dtype { RUA_F32 = 0, RUA_F64 = 1, RUA_F16 = 2, RUA_BF16 = 3 };

enum rua_reduce {
  RUA_SUM = 0, RUA_MEAN = 1, RUA_PROD = 2, RUA_MAX = 3, RUA_MIN = 4, RUA_LOGSUMEXP = 5
};

/* base ragged structure shared by both sides of a row map */
typedef struct {
  int64_t B;               /* number of sequences                                             */
  const int64_t* off;      /* B+1: exclusive prefix sum of the base lengths                   */
  const int64_t* poff;     /* Tp+1: exclusive prefix sum of batch_sizes; NULL if no P side    */
  const int64_t* sorted;   /* B: sorted_indices; NULL if no P side                            */
  const int64_t* unsorted; /* B: unsorted_indices; NULL if no P side                          */
  int64_t Tp;              /* number of time steps in poff (len(batch_sizes)); 0 if no P side */
} rua_ragged_t;

/* one side (source or destination) of a row map */
typedef struct {
  int32_t layout;    /* enum rua_layout                                            */
  int32_t len_xform; /* enum rua_len_xform                                         */
  int64_t len_arg;   /* n for CONST, a+b for MINUS                                 */
  int64_t width;     /* L/R: rows per sequence in storage (data.size(1)); else 0   */
  int64_t rows;      /* total rows in this side's flattened storage (N' or B*W)    */
} rua_side_t;

/* ------------------------------------------------------------------------------------------- */
/* library                                                                                       */
/* ------------------------------------------------------------------------------------------- */
int rua_version(void);
const char* rua_error_string(int status);
int rua_last_cuda_error(void);
/* number of kernel launches issued by this library since load (for bench.py's gpu_launches) */
int64_t rua_launch_count(void);
/* host-only self test of launch-time arithmetic (magic-number division of the narrow-row kernels): 0 = ok.  No GPU. */
int rua_selftest(void);

/* ------------------------------------------------------------------------------------------- */
/* K0  metadata from lengths                                                                     */
/* replaces get_offsets (torchrua/utils.py:16-19), size() (layout/cat.py:61-66),                 */
/* invert_permutation (utils.py:22-26), pack_view (core/view.py:47-58), and the                  */
/* get_mask(...).sum(dim) detours of cat_view/left_view/right_view (core/view.py:11-38,67-71)    */
/* ------------------------------------------------------------------------------------------- */

/* off[0..n] = min(exclusive prefix sum of sizes[0..n), clamp_max); stats[0] = sum, stats[1] =
 * max(sizes) (0 if n==0).  clamp_max = INT64_MAX for the plain scan; C.offsets()/P.offsets() pass N-1
 * (torchrua/layout/cat.py:81, pack.py:45).  ws: rua_scan_workspace_bytes(n) bytes. */
size_t rua_scan_workspace_bytes(int64_t n);
int rua_scan_lengths(const int64_t* sizes, int64_t n, int64_t clamp_max, int64_t* off, int64_t* stats,
                     void* ws, size_t ws_bytes, rua_stream_t stream);

/* the same scan with two optional extras (either may be left out by passing NULL):
 *  - sizes == NULL: the lengths are those of a PackedSequence, len[i] = #{t : bs[t] > unsorted[i]} (core/view.py:21-25
 *    on a P source), computed on the fly and also written to len_out (n entries): P -> token_sizes + offsets in ONE launch;
 *  - notify_host_mapped != NULL: 3 int64 of PINNED HOST memory reachable from the device (UVA).  When the scan is
 *    complete the device writes [sum, max, ticket] there (ticket last, after a system-scope fence), so the host can
 *    learn N = sum and T = max by polling notify[2] == ticket instead of copying stats back and synchronising the
 *    stream.  ws: rua_scan_workspace_bytes(n). */
int rua_scan_lengths_ex(const int64_t* sizes, int64_t n, int64_t clamp_max, int64_t* off, int64_t* stats, void* ws,
                        size_t ws_bytes, const int64_t* bs, const int64_t* unsorted, int64_t Tp, int64_t* len_out,
                        int64_t* notify_host_mapped, int64_t ticket, rua_stream_t stream);

/* pinned host memory a kernel can write to directly (cudaHostAlloc mapped + portable): *device_ptr is what to pass as
 * notify_host_mapped, *host_ptr is where the host polls.  Set-up calls (they synchronise like cudaMalloc / cudaFree). */
int rua_pinned_alloc(size_t bytes, void** host_ptr, void** device_ptr);
int rua_pinned_free(void* host_ptr);

/* stable descending argsort of the lengths (ties by ascending index -- the documented deviation from
 * the reference's non-stable CPU sort, SURVEY.md 8c hazard 1) and its inverse.  T = max length. */
size_t rua_sort_workspace_bytes(int64_t B);
int rua_sort_lengths(const int64_t* len, int64_t B, int64_t T, int64_t* sorted, int64_t* unsorted,
                     void* ws, size_t ws_bytes, rua_stream_t stream);

/* stable ASCENDING argsort of int64 keys in [0, max_key] and its inverse (scatter_* sort their index
 * with this; same workspace as rua_sort_lengths), and the bucket boundaries of the sorted order:
 * off[m] = #{k : keys[k] < m} for m in [0, M]. */
int rua_sort_keys(const int64_t* keys, int64_t n, int64_t max_key, int64_t* sorted, int64_t* unsorted,
                  void* ws, size_t ws_bytes, rua_stream_t stream);
int rua_bucket_offsets(const int64_t* keys, const int64_t* sorted, int64_t n, int64_t M, int64_t* off,
                       rua_stream_t stream);

/* out[perm[j]] = j */
int rua_invert_permutation(const int64_t* perm, int64_t B, int64_t* out, rua_stream_t stream);

/* bs[t] = #{i : len[i] > t}, t in [0,T), given ANY permutation `sorted` that orders len
 * non-increasingly (ours or an injected one). */
int rua_batch_sizes(const int64_t* len, const int64_t* sorted, int64_t B, int64_t T, int64_t* bs,
                    rua_stream_t stream);

/* len[i] = #{t : bs[t] > unsorted[i]}  (P -> token_sizes; core/view.py:21-25 on a P source) */
int rua_lengths_from_pack(const int64_t* bs, const int64_t* unsorted, int64_t B, int64_t T,
                          int64_t* len, rua_stream_t stream);

/* One-launch metadata for B <= rua_meta_fused_max_batch() sequences (a single CTA; bitonic sort in
 * shared memory): off[B+1]; hostbuf[0] = N, hostbuf[1] = T; and, when `sorted` != NULL, the stable
 * descending permutation + inverse, hostbuf[2 + t] = batch_sizes[t] and poff[t] for t < min(T, cap),
 * poff[min(T,cap)] = N (or -1 if T > cap: re-run with a larger cap).  hostbuf has 2 + cap entries so
 * the caller can fetch N, T and batch_sizes with ONE device->host copy (pack_view, core/view.py:47-58). */
int64_t rua_meta_fused_max_batch(void);
int rua_meta_fused(const int64_t* len, int64_t B, int64_t* off, int64_t* sorted, int64_t* unsorted,
                   int64_t* hostbuf, int64_t* poff, int64_t cap, rua_stream_t stream);

/* ------------------------------------------------------------------------------------------- */
/* K1/K2  ragged row map: the 12 layout conversions, the selects and their backward passes       */
/* replaces to_cat / cat_pack_to_left / right_to_left / to_pack / cat_pack_to_right /            */
/* left_to_right (torchrua/core/cast.py:8-71), {cat,left,pack,right}_getitem/_setitem with       */
/* (batch_ptr, token_ptr) keys (core/get.py:21-79, core/set.py:23-92), head / last / rev / roll  */
/* / trunc (torchrua/select/*.py), segment_head / segment_last (reduce.py:64-69)                 */
/* ------------------------------------------------------------------------------------------- */
/* For every row j of the destination storage (dst->rows rows of row_bytes bytes):
 *   decode j -> (i, t_d) in the destination layout; if it is padding -> pad;
 *   t_s = tmap(t_d); if t_s is outside the source's length -> pad;
 *   else copy source row src_row(i, t_s).
 * Every destination byte is written exactly once (padding fill is fused). */
int rua_row_map(const void* src, void* dst, int64_t row_bytes, const rua_ragged_t* ragged,
                const rua_side_t* src_side, const rua_side_t* dst_side, int32_t tmap,
                int64_t tmap_arg, int32_t pad_mode, const void* fill_host, int32_t fill_bytes,
                rua_stream_t stream);

/* fused consumer pattern (SURVEY.md 8f-4): `X.left(fill)` AND `X.mask(zero, one, dtype)` (torchrua/core/cast.py:19-32 +
 * torchrua/mask.py:6-32, e.g. padded activations + the additive attention bias of fmask) from ONE decode of the
 * destination rows: rua_row_map towards a LEFT destination that also writes mask_out[i, t] (dst_side->rows elements of
 * mask_elem_bytes) = one where the row holds a token, zero where it is padding.  Rows of >= 128 bytes only (narrow
 * rows: RUA_ERR_UNSUPPORTED -- launch rua_row_map and rua_mask). */
int rua_row_map_mask(const void* src, void* dst, int64_t row_bytes, const rua_ragged_t* ragged,
                     const rua_side_t* src_side, const rua_side_t* dst_side, const void* fill_host, int32_t fill_bytes,
                     const void* zero_host, const void* one_host, int32_t mask_elem_bytes, void* mask_out,
                     rua_stream_t stream);

/* constructors C/L/P/R.new(list) (torchrua/core/__init__.py:9-36): rua_row_map with an identity token map whose
 * SOURCE is a list -- sequence i is its own contiguous (len[i], row_bytes) allocation src_list[i].  src_list is a
 * DEVICE array of B device pointers; src_align = a power of two that divides every non-null pointer in it (the
 * kernel picks its vector width from it).  Replaces torch.cat + conversion: every payload byte moves once. */
int rua_row_map_list(const void* const* src_list, int32_t src_align, void* dst, int64_t row_bytes,
                     const rua_ragged_t* ragged, const rua_side_t* dst_side, const void* fill_host,
                     int32_t fill_bytes, rua_stream_t stream);

/* compose (torchrua/compose.py:9-33: torch.cat(data)[indices]) without materialising the concatenation: dst[j] = row
 * index[j] of the VIRTUAL concatenation of n_src tensors.  src_list: DEVICE array of n_src device pointers (whole
 * contiguous (rows_k, row_bytes) tensors); bases: DEVICE array of n_src + 1 int64, bases[k] = first row of tensor k in the
 * concatenation, bases[n_src] = total rows; src_align as in rua_row_map_list.  Every payload byte moves once. */
int rua_gather_rows_multi(const void* const* src_list, const int64_t* bases, int32_t n_src, int32_t src_align,
                          const int64_t* index, int64_t n, int64_t row_bytes, void* dst, rua_stream_t stream);

/* dst[j] = src[index[j]] for j < n   (tensor_getitem / Z-keyed getitem, core/get.py:11-31).
 * Negative indices wrap (index + src_rows) like torch advanced indexing; an index that is still out of range is
 * not dereferenced: the row is zero-filled (gather) or skipped (scatter) and counted (rua_index_error_count). */
int rua_gather_rows(const void* src, int64_t src_rows, const int64_t* index, int64_t n,
                    int64_t row_bytes, void* dst, rua_stream_t stream);
/* dst[index[j]] = src[j] for j < n   (tensor_setitem / Z-keyed setitem, core/set.py:10-31) */
int rua_scatter_rows(const void* src, const int64_t* index, int64_t n, int64_t row_bytes, void* dst,
                     int64_t dst_rows, rua_stream_t stream);

/* flat storage rows of layout position keys -- the (batch_ptr, token_ptr) branches of
 * {cat,left,pack,right}_getitem / _setitem (torchrua/core/get.py:21-82, core/set.py:23-92):
 *   C: min(off[b], rows-1) + t     L: b*W + t     R: b*W + (T - len[b]) + t     P: unsorted[b] + min(poff[t], rows-1)
 * with the clamps of C.offsets() / P.offsets() (layout/cat.py:79-81, pack.py:43-45), T = max length for R
 * (layout/right.py:62-67: size()[1], not the storage width W = side->width) and torch's wrap-around of negative
 * indices where the reference's indexing applies it.  batch_ptr == NULL: token_ptr holds flat rows already; they
 * are wrapped and bounds-checked only.  Out-of-range keys yield side->rows (one past the end: rua_gather_rows zero-fills it,
 * rua_scatter_rows skips it, an ascending sort keeps it last) and bump the error counter below.  Feed rows_out to rua_gather_rows / rua_scatter_rows. */
int rua_token_rows(const rua_ragged_t* ragged, const rua_side_t* side, int64_t T, const int64_t* batch_ptr,
                   const int64_t* token_ptr, int64_t n, int64_t* rows_out, rua_stream_t stream);

/* number of out-of-range indices seen by rua_gather_rows / rua_scatter_rows / rua_token_rows on the current device
 * since the last reset.  Those rows were NOT dereferenced (ATen device-asserts in the same situation).  This call
 * synchronises (one 8-byte device->host copy): diagnostics, not data path. */
int rua_index_error_count(int64_t* count_host, int32_t reset);

/* ------------------------------------------------------------------------------------------- */
/* K3  mask / index emit (no payload reads)                                                      */
/* replaces mask / bmask / fmask (torchrua/mask.py:6-32), get_mask (core/view.py:11-18),         */
/* major_sizes_to_ptr (utils.py:7-13), C/L/R.ptr, P.ptr, L.idx, R.idx (layout/*.py)              */
/* ------------------------------------------------------------------------------------------- */
/* out (B, W) elements of elem_bytes in {1,2,4,8}: `one` where t < len[i] else `zero` (left aligned
 * for every layout, mask.py:10). */
int rua_mask(const int64_t* len, int64_t B, int64_t W, const void* zero_host, const void* one_host,
             int32_t elem_bytes, void* out, rua_stream_t stream);

/* enumerate the n = off[S] positions of a segmented range: which[k] = segment id, within[k] = k -
 * off[which[k]].  Either output may be NULL.  If `relabel` is non-NULL, within[k] = relabel[k -
 * off[which[k]]] (P.ptr: segments are time steps, within = sorted_indices[rank]).  With stride != 0 also emits
 * flat[k] = which*stride + within + (align ? (stride - len[which]) : 0)   (L.idx / R.idx). */
int rua_emit_ptr(const int64_t* off, int64_t S, int64_t n, const int64_t* relabel, int64_t* which,
                 int64_t* within, int64_t* flat, int64_t stride, int32_t right_align,
                 rua_stream_t stream);

/* ------------------------------------------------------------------------------------------- */
/* K4  segment reduce                                                                            */
/* replaces segment_max/min/sum/mean/prod/logsumexp (torchrua/reduce.py:34-61)                   */
/* ------------------------------------------------------------------------------------------- */
/* data (N, H) row-major, off (S+1) exclusive prefix of the segment sizes, out (S, H).
 * Accumulates in fp32 (fp64 for RUA_F64) whatever the storage dtype and rounds once.
 * Reference quirks reproduced (SURVEY.md 8c hazard 3): empty segments of max / logsumexp (min)
 * return the global min (max) of the whole tensor; a NaN anywhere poisons every output of
 * max / min / logsumexp; empty sum/mean -> 0, prod -> 1. */
size_t rua_segment_reduce_workspace_bytes(int64_t N, int64_t S, int64_t H, int32_t dtype, int32_t op);
int rua_segment_reduce(const void* data, const int64_t* off, int64_t N, int64_t S, int64_t H,
                       int32_t dtype, int32_t op, void* out, void* ws, size_t ws_bytes,
                       rua_stream_t stream);

/* the same reduction over GATHERED rows: segment s reduces data[row_index[r]] for r in [off[s], off[s+1]);
 * N = off[S] = number of entries of row_index.  scatter_* (torchrua/reduce.py:6-31) = stable sort of the
 * index + rua_bucket_offsets + this. */
int rua_segment_reduce_gather(const void* data, const int64_t* row_index, const int64_t* off, int64_t N,
                              int64_t S, int64_t H, int32_t dtype, int32_t op, void* out, void* ws,
                              size_t ws_bytes, rua_stream_t stream);

/* PARITY MODE for sum / mean / prod: the reference's order of operations replayed exactly -- per (segment,
 * column) strictly left to right in the STORAGE dtype with one rounding per step, mean divides by the length
 * converted to the storage dtype (what torch.segment_reduce computes for torchrua/reduce.py:44-53; SURVEY.md
 * 8c hazard 2).  Bit-identical to the reference for fp32 / fp64 / fp16 / bf16.  No workspace.  Other ops return
 * RUA_ERR_UNSUPPORTED (max / min are bit-exact in rua_segment_reduce already). */
int rua_segment_reduce_strict(const void* data, const int64_t* off, int64_t N, int64_t S, int64_t H,
                              int32_t dtype, int32_t op, void* out, rua_stream_t stream);

/* backward twin (ATen SegmentReduceBackward0 semantics, SURVEY.md 8a): sum -> broadcast, mean ->
 * broadcast / len, max/min -> split evenly among ties, prod -> grad*out/x (exact when x != 0, else
 * product of the others), logsumexp -> softmax weights.  Writes all N rows of grad_data: rows no segment
 * owns (at or past off[S]) get 0.  S == 0: grad_out, out, data and off may be NULL; grad_data is zeroed
 * with cudaMemsetAsync and no kernel runs. */
size_t rua_segment_reduce_backward_workspace_bytes(int64_t N, int64_t S, int64_t H, int32_t dtype,
                                                   int32_t op);
int rua_segment_reduce_backward(const void* grad_out, const void* out, const void* data,
                                const int64_t* off, int64_t N, int64_t S, int64_t H, int32_t dtype,
                                int32_t op, void* grad_data, void* ws, size_t ws_bytes,
                                rua_stream_t stream);

/* ------------------------------------------------------------------------------------------- */
/* K7  per-sequence prefix scans (no counterpart in the reference; replaces the pad -> ATen scan  */
/* along dim 1 -> unpad composition a user would write with to_left / torch.cumsum / to_cat)     */
/* ------------------------------------------------------------------------------------------- */
enum rua_scan { RUA_SCAN_SUM = 0, RUA_SCAN_LOGSUMEXP = 1, RUA_SCAN_MAX = 2, RUA_SCAN_MIN = 3 };

/* workspace of rua_segment_scan (backward = 0) / rua_segment_scan_backward (backward = 1) over side->rows = rows rows of
 * H elements; 0 when there is nothing to do or an argument is invalid. */
size_t rua_segment_scan_workspace_bytes(int64_t rows, int64_t H, int32_t dtype, int32_t op, int32_t backward);

/* src / dst: side->rows rows of H elements in the storage of `side` (C, L, P or R over `ragged`; len_xform must be
 * RUA_LEN_SAME).  For token (i, t) of sequence i with length len[i] (rows from the "Row of token" formulas above):
 *   dst(i, t) = op over src(i, 0..t)             (reverse = 0)
 *   dst(i, t) = op over src(i, t..len[i]-1)      (reverse = 1)
 * op = max / min also writes idx_out (same shape, int64): the position within the sequence of the selected element,
 * ties to the later position in scan order, a NaN sticks with its own position (torch.cummax / cummin).  Rows that hold
 * no token (L / R padding, C rows at or past off[B]) are copied through, with index 0.  max / min: side->rows < 2^31
 * (RUA_ERR_UNSUPPORTED otherwise).  fp32 accumulation (fp64 for
 * RUA_F64), one rounding.  Deterministic: chunk carries are combined in chunk order, never in arrival order.
 * ws: rua_segment_scan_workspace_bytes(side->rows, H, dtype, op, 0) bytes; it is cleared by a memset on `stream`. */
int rua_segment_scan(const void* src, void* dst, int64_t* idx_out, int64_t H, int32_t dtype, int32_t op,
                     int32_t reverse, const rua_ragged_t* ragged, const rua_side_t* side, void* ws, size_t ws_bytes,
                     rua_stream_t stream);

/* gradient of rua_segment_scan with the same op / reverse / ragged / side: grad_in = d(loss)/d(src) from grad_out.
 *   sum: the scan of grad_out in the other direction;
 *   logsumexp: x = the forward input, y = the forward output; grad_in = exp(x - y) * v with v the reverse affine scan
 *              v_k = g_k + exp(y_k - y_next) v_next (exponents <= 0); 0 where x = -inf (torch gives NaN for a leading
 *              -inf);
 *   max / min: idx = the forward indices; grad_in(k) = sum of grad_out(j) over the positions j whose index is k.
 * Arguments an op does not use may be NULL.  Rows that hold no token pass grad_out through.  Every row of grad_in is
 * written.  ws: rua_segment_scan_workspace_bytes(side->rows, H, dtype, op, 1) bytes. */
int rua_segment_scan_backward(const void* grad_out, const void* x, const void* y, const int64_t* idx, void* grad_in,
                              int64_t H, int32_t dtype, int32_t op, int32_t reverse, const rua_ragged_t* ragged,
                              const rua_side_t* side, void* ws, size_t ws_bytes, rua_stream_t stream);

/* per-sequence gated linear recurrence, on the same kernel as the scans (an affine scan with state (m, b)).
 * workspace of rua_segment_linrec (backward = 0) / rua_segment_linrec_backward (backward = 1) over side->rows = rows rows
 * of H elements; 0 when there is nothing to do or an argument is invalid. */
size_t rua_segment_linrec_workspace_bytes(int64_t rows, int64_t H, int32_t dtype, int32_t backward);

/* x / gate / dst: side->rows rows of H elements in the storage of `side` (as rua_segment_scan), all of `dtype`; h0: B rows
 * of H elements in sequence order (for P the index in ragged->off, not the sorted one), or NULL for a zero state.  For
 * token (i, t) of sequence i with length len[i]:
 *   dst(i, t) = gate(i, t) * dst(i, t-1) + x(i, t),  dst(i, -1)     = h0[i]     (reverse = 0)
 *   dst(i, t) = gate(i, t) * dst(i, t+1) + x(i, t),  dst(i, len[i]) = h0[i]     (reverse = 1)
 * Any real gate: 0 resets the state, 1 gives cumsum.  Rows that hold no token are copied through from x.  fp32
 * accumulation (fp64 for RUA_F64), one rounding.  Deterministic: chunk carries are combined in chunk order.  Specified
 * for finite inputs; non-finite values propagate, in a pattern that may differ from a sequential loop (0 * inf).
 * ws: rua_segment_linrec_workspace_bytes(side->rows, H, dtype, 0) bytes; it is cleared by a memset on `stream`. */
int rua_segment_linrec(const void* x, const void* gate, const void* h0, void* dst, int64_t H, int32_t dtype,
                       int32_t reverse, const rua_ragged_t* ragged, const rua_side_t* side, void* ws, size_t ws_bytes,
                       rua_stream_t stream);

/* gradients of rua_segment_linrec with the same gate / h0 / reverse / ragged / side; y = the forward output, g = grad_out.
 * In forward order, with g~(t) = g(t) + gate(t+1) g~(t+1) the whole adjoint of dst(t) (g~ = g at the last position):
 *   grad_x(t)    = g~(t);
 *   grad_gate(t) = g~(t) * y(t-1), with y(-1) = h0[i] (0 when h0 is NULL);
 *   grad_h0[i]   = gate(0) * g~(0), 0 for an empty sequence.
 * The kernel scans z(t) = gate(t) g~(t) against the forward direction; y(t-1) is read from its own row of the same
 * sequence.  grad_x, grad_gate and grad_h0 may each be NULL and are then not computed; y is needed for grad_gate only.
 * Rows that hold no token pass grad_out through to grad_x and get 0 in grad_gate.  Deterministic like the forward.
 * ws: rua_segment_linrec_workspace_bytes(side->rows, H, dtype, 1) bytes. */
int rua_segment_linrec_backward(const void* grad_out, const void* gate, const void* h0, const void* y, void* grad_x,
                                void* grad_gate, void* grad_h0, int64_t H, int32_t dtype, int32_t reverse,
                                const rua_ragged_t* ragged, const rua_side_t* side, void* ws, size_t ws_bytes,
                                rua_stream_t stream);

/* ------------------------------------------------------------------------------------------- */
/* K8  per-sequence depthwise 1-D convolution (no counterpart in the reference; replaces the     */
/* pad -> F.conv1d(groups=H) on (B, H, T) -> unpad composition, and F.conv1d straight on the     */
/* storage, which mixes every sequence's first and last K-1 outputs with its neighbours)         */
/* ------------------------------------------------------------------------------------------- */
/* workspace of rua_segment_conv (backward = 0: always 0) / rua_segment_conv_backward (backward = 1) over rows = side->rows
 * rows of H elements with K taps: a fixed number of per-CTA slots of partial weight / bias gradients, capped whatever
 * rows is (monotone in rows, bounded).  Host only; 0 when an argument is invalid. */
size_t rua_segment_conv_workspace_bytes(int64_t rows, int64_t H, int32_t K, int32_t dtype, int32_t backward);

/* src / dst: side->rows rows of H elements in the storage of `side` (C, L, P or R over `ragged`; len_xform must be
 * RUA_LEN_SAME); weight (H, K) row-major, bias (H) or NULL, both of the payload dtype.  For token (i, t) of sequence i with
 * length len[i] (rows from the "Row of token" formulas above), 1 <= K <= 32, 0 <= pad <= K - 1:
 *   dst(i, t, h) = bias[h] + sum_{k<K} weight[h, k] * src(i, t + k - pad, h),   src(i, s, .) = 0 for s outside [0, len[i])
 * pad = K - 1 is causal (weight[:, K-1] multiplies the current token), pad = (K - 1) / 2 is torch's padding='same'.
 * Rows that hold no token (L / R padding, C rows at or past off[B]) are copied through.  fp32 accumulation (fp64 for
 * RUA_F64), one rounding.  No workspace (ws may be NULL). */
int rua_segment_conv(const void* src, const void* weight, const void* bias, void* dst, int64_t H, int32_t dtype, int32_t K,
                     int32_t pad, const rua_ragged_t* ragged, const rua_side_t* side, void* ws, size_t ws_bytes,
                     rua_stream_t stream);

/* gradients of rua_segment_conv with the same weight / H / dtype / K / pad / ragged / side; x = the forward input.
 *   grad_in: the same convolution of grad_out with the taps flipped and pad' = K - 1 - pad; rows that hold no token pass
 *            grad_out through (every row written);
 *   grad_weight[h, k] = sum over tokens (i, t) with 0 <= t + k - pad < len[i] of grad_out(i, t, h) * x(i, t + k - pad, h);
 *   grad_bias[h] = sum over tokens of grad_out(i, t, h).
 * Any of grad_in / grad_weight / grad_bias may be NULL and is then not computed (x may be NULL without grad_weight).
 * Deterministic: every CTA sums its chunks into its own workspace slot in a fixed order (no atomics), and a second kernel
 * sums the slots in slot order, so grad_weight / grad_bias are bit-identical run to run.  ws:
 * rua_segment_conv_workspace_bytes(side->rows, H, K, dtype, 1) bytes when grad_weight or grad_bias is wanted. */
int rua_segment_conv_backward(const void* grad_out, const void* x, const void* weight, void* grad_in, void* grad_weight,
                              void* grad_bias, int64_t H, int32_t dtype, int32_t K, int32_t pad, const rua_ragged_t* ragged,
                              const rua_side_t* side, void* ws, size_t ws_bytes, rua_stream_t stream);

/* ------------------------------------------------------------------------------------------- */
/* K9  per-sequence linear-chain CRF (no counterpart in the reference; replaces pad -> a Python   */
/* loop over T of logsumexp(alpha[:, :, None] + W + x_t[:, None, :], 1) -> autograd, which keeps */
/* a (B, K, K) temporary per step, and the same loop in max-plus + a backtrack for Viterbi)      */
/* ------------------------------------------------------------------------------------------- */
/* Emissions x: side->rows rows of K tag scores in the storage of `side` (C, L, P or R over `ragged`; len_xform must be
 * RUA_LEN_SAME); W (K, K) row-major, W[a, b] scores tag a at t-1 followed by tag b at t; start, end (K) or NULL for 0; all of
 * `dtype`.  1 <= K <= 64.  For a tag path y of sequence i with length len[i] (rows from the "Row of token" formulas):
 *   score(y) = start[y_0] + sum_t x(i, t)[y_t] + sum_{t>=1} W[y_{t-1}, y_t] + end[y_{len-1}]
 *   log Z_i  = logsumexp over all K^len paths of score(y)
 * Per-sequence outputs (log_z, score, best_score and their gradients grad_log_z, grad_score) are B values of the
 * ACCUMULATOR type (fp32, fp64 for RUA_F64) in sequence order (for P the index in ragged->off).  -inf anywhere means a
 * forbidden tag or transition; behaviour is specified for inputs without NaN.  An empty sequence has log Z = score = best
 * score = 0 and zero gradients.  ragged->sorted is required (B > 0): warp g of a fixed grid of G warps takes the sequences
 * of ranks g, g + G, ... in that order (longest first for the package's own sort), so every result is bit-identical run
 * to run and, for the same sequences, on every layout.  The running state is normalised per step with an fp64 offset. */
enum rua_crf_mode { RUA_CRF_FORWARD = 0, RUA_CRF_BACKWARD = 1, RUA_CRF_DECODE = 2 };

/* workspace of rua_crf_forward (0: none), rua_crf_backward (a fixed number of per-CTA slots of partial transition / start
 * / end gradients: monotone in rows and bounded) and rua_crf_decode (rows x K bytes of uint8 backpointers).  Host only;
 * 0 when an argument is invalid. */
size_t rua_crf_workspace_bytes(int64_t rows, int32_t K, int32_t dtype, int32_t mode);
/* bytes of the state rua_crf_forward keeps for rua_crf_backward: the normalised forward scores (rows x K, accumulator
 * type) and the fp64 offset of every row. */
size_t rua_crf_state_bytes(int64_t rows, int32_t K, int32_t dtype);

/* log_z[i] = log Z_i.  tags != NULL (side->rows int64, read at token rows only): also score[i] = score(tags of i), NaN
 * for a sequence with a tag outside [0, K) (that tag is not dereferenced); tags and score are given together or not at
 * all.  state_out: rua_crf_state_bytes(side->rows, K, dtype) bytes for rua_crf_backward, or NULL.  No workspace. */
int rua_crf_forward(const void* x, const int64_t* tags, const void* W, const void* start, const void* end, void* log_z,
                    void* score, void* state_out, int32_t K, int32_t dtype, const rua_ragged_t* ragged,
                    const rua_side_t* side, void* ws, size_t ws_bytes, rua_stream_t stream);

/* gradients of gZ_i log Z_i + gS_i score_i (gZ = grad_log_z, gS = grad_score or NULL for 0) with the state and log_z of the
 * rua_crf_forward call on the same x / W / start / end / ragged / side:
 *   grad_x(i, t)[b] = gZ mu_t[b] + gS [b = y_t],   mu_t[b] = exp(alpha_t[b] + beta_t[b] - log Z_i) (the tag marginal);
 *   grad_W[a, b]    = sum over tokens t >= 1 of gZ xi_t[a, b] + gS [y_{t-1} = a, y_t = b];
 *   grad_start / grad_end: the same at the first / last token.
 * A sequence with log Z = -inf contributes 0, and so do tags outside [0, K).  Rows that hold no token get 0 in grad_x.  Any
 * of grad_x / grad_W / grad_start / grad_end may be NULL and is then not computed; tags are needed with grad_score only;
 * start is not read (the state holds it).  Deterministic: every CTA sums its sequences into its own workspace slot, and a
 * second kernel sums the slots in slot order.  ws: rua_crf_workspace_bytes(side->rows, K, dtype, RUA_CRF_BACKWARD) bytes
 * when grad_W, grad_start or grad_end is wanted.  No token at all: the gradients are zeroed with cudaMemsetAsync. */
int rua_crf_backward(const void* grad_log_z, const void* grad_score, const void* x, const int64_t* tags, const void* W,
                     const void* start, const void* end, const void* state, const void* log_z, void* grad_x, void* grad_W,
                     void* grad_start, void* grad_end, int32_t K, int32_t dtype, const rua_ragged_t* ragged,
                     const rua_side_t* side, void* ws, size_t ws_bytes, rua_stream_t stream);

/* Viterbi: tags_out (side->rows int64) = the best path of every sequence at its own rows, -1 at rows that hold no token;
 * best_score[i] = its score.  Ties go to the smallest tag index, for the predecessor at every step and for the last tag.
 * ws: rua_crf_workspace_bytes(side->rows, K, dtype, RUA_CRF_DECODE) bytes. */
int rua_crf_decode(const void* x, const void* W, const void* start, const void* end, int64_t* tags_out, void* best_score,
                   int32_t K, int32_t dtype, const rua_ragged_t* ragged, const rua_side_t* side, void* ws,
                   size_t ws_bytes, rua_stream_t stream);

/* ------------------------------------------------------------------------------------------- */
/* K10 per-sequence selective state-space scan, Mamba-1 style (no counterpart in the reference;  */
/* replaces pad -> a Python loop over T that autograd keeps a (B, H, N) state of per step, and   */
/* the linear recurrence over H x N columns, which materialises (tokens, H, N) tensors)          */
/* ------------------------------------------------------------------------------------------- */
/* x, delta, y: side->rows rows of H elements in the storage of `side` (C, L, P or R over `ragged`; len_xform must be
 * RUA_LEN_SAME); Bm, Cm: side->rows rows of N elements in the same storage; all of `dtype`.  A (H, N), h0 / h_final
 * (B, H, N) in sequence order (for P the index in ragged->off) are of the ACCUMULATOR type (fp32, fp64 for RUA_F64).
 * 1 <= N <= 16, H >= 0.  For token (i, t) of sequence i with length len[i] (rows from the "Row of token" formulas),
 * channel h and state n:
 *   dA_t[h, n] = exp(delta_t[h] A[h, n])
 *   h_t[h, n]  = dA_t[h, n] h_{t-1}[h, n] + delta_t[h] Bm_t[n] x_t[h],   h_{-1} = h0[i] (0 when h0 is NULL)
 *   y_t[h]     = sum_n Cm_t[n] h_t[h, n]
 *   h_final[i] = h at the last token (h0[i], or 0, for an empty sequence)
 * reverse = 1 runs from each sequence's end: h_t depends on h_{t+1}, h_{len} = h0[i], h_final[i] is the state at t = 0.
 * fp32 accumulation (fp64 for RUA_F64), one rounding of y.  Rows that hold no token (L / R padding, C rows at or past
 * off[B]) are copied through from x.  ragged->sorted is required (B > 0): CTA (cb, g) of a fixed grid takes channel
 * block cb of the sequences of ranks g, g + G, ... in that order, so every result is bit-identical run to run and, for
 * the same sequences, on every layout.  No float atomics anywhere. */

/* bytes of the state rua_ssm_forward keeps for rua_ssm_backward: the state entering every chunk of 32 steps of every
 * sequence, (rows / 32 + B) x H x N accumulator-type values (at most one H x N state per 32 tokens of each sequence plus
 * one per sequence; with rows >= sum(len)).  Host only; 0 when an argument is invalid. */
size_t rua_ssm_state_bytes(int64_t rows, int64_t B, int64_t H, int32_t N, int32_t dtype);
/* workspace of rua_ssm_backward when grad_A, grad_B or grad_C is wanted (0 when rows, B or H is 0, or an argument is
 * invalid), in accumulator-type values:
 *   G x H x N grad_A slots, G = min(B, ceil(148 c / ceil(H / W))) with c <= 8 CTAs per SM, rounded up to 256 bytes,
 *   + ceil(H / W) x rows x 2N partials of [grad_B | grad_C] per (token, channel block),
 * with W = 128 channels per block (64 for RUA_F64).  Monotone in rows. */
size_t rua_ssm_workspace_bytes(int64_t rows, int64_t B, int64_t H, int32_t N, int32_t dtype);

/* y (and h_final when not NULL) as above.  state_out: rua_ssm_state_bytes(side->rows, B, H, N, dtype) bytes for
 * rua_ssm_backward, or NULL.  No workspace (ws may be NULL). */
int rua_ssm_forward(const void* x, const void* delta, const void* A, const void* Bm, const void* Cm, const void* h0,
                    void* y, void* h_final, void* state_out, int64_t H, int32_t N, int32_t dtype, int32_t reverse,
                    const rua_ragged_t* ragged, const rua_side_t* side, void* ws, size_t ws_bytes, rua_stream_t stream);

/* gradients of sum g y with the state of the rua_ssm_forward call on the same x / delta / A / Bm / Cm / h0 / reverse /
 * ragged / side.  In processing order, with dh_t the adjoint of h_t (0 past the last token):
 *   dh_t[h, n]      = Cm_t[n] g_t[h] + dA_{t+1}[h, n] dh_{t+1}[h, n]
 *   grad_x_t[h]     = delta_t[h] sum_n Bm_t[n] dh_t[h, n]
 *   grad_delta_t[h] = sum_n dh_t[h, n] (A[h, n] dA_t[h, n] h_{t-1}[h, n] + Bm_t[n] x_t[h])
 *   grad_A[h, n]    = sum over all tokens of dh_t[h, n] delta_t[h] dA_t[h, n] h_{t-1}[h, n]
 *   grad_Bm_t[n]    = sum_h dh_t[h, n] delta_t[h] x_t[h]
 *   grad_Cm_t[n]    = sum_h g_t[h] h_t[h, n]
 *   grad_h0[i]      = dA_0 dh_0 (0 for an empty sequence)
 * grad_A and grad_h0 are of the accumulator type, the others of `dtype`.  Any gradient pointer may be NULL and is then not
 * computed.  Rows that hold no token pass grad_out through to grad_x and get 0 in grad_delta, grad_Bm and grad_Cm.  The
 * kernel recomputes each chunk's states from its checkpoint.  Deterministic: grad_A is summed per CTA slot in slot order,
 * grad_Bm / grad_Cm per token in a fixed warp / block order, by a second kernel.  ws: rua_ssm_workspace_bytes(side->rows,
 * B, H, N, dtype) bytes when grad_A, grad_Bm or grad_Cm is wanted.  No token at all: grad_x is copied from grad_out and the
 * other gradients are zeroed on `stream`. */
int rua_ssm_backward(const void* grad_out, const void* x, const void* delta, const void* A, const void* Bm, const void* Cm,
                     const void* state, void* grad_x, void* grad_delta, void* grad_A, void* grad_Bm, void* grad_Cm,
                     void* grad_h0, int64_t H, int32_t N, int32_t dtype, int32_t reverse, const rua_ragged_t* ragged,
                     const rua_side_t* side, void* ws, size_t ws_bytes, rua_stream_t stream);

/* ------------------------------------------------------------------------------------------- */
/* K11 per-sequence Mamba-2 (SSD) state-space scan: a scalar decay per head, a P x N state per   */
/* head, B / C shared by the heads of a group (no counterpart in the reference; replaces pad ->  */
/* a pure-torch chunked einsum that materialises (B, chunks, Q, Q, H) decay tensors)              */
/* ------------------------------------------------------------------------------------------- */
/* x, y: side->rows rows of H x P elements; delta: side->rows rows of H; Bm, Cm: side->rows rows of G x N; all in the
 * storage of `side` (C, L, P or R over `ragged`; len_xform must be RUA_LEN_SAME) and of `dtype`.  A (H), h0 / h_final
 * (B, H, P, N) in sequence order (for P the index in ragged->off) are of the ACCUMULATOR type (fp32, fp64 for RUA_F64).
 * 1 <= P <= 64, 1 <= N <= 128, G >= 1, H >= 0, H % G == 0.  For token (i, t), head h, channel p, state n and group
 * g = h / (H / G):
 *   dA_t      = exp(delta_t[h] A[h])
 *   h_t[p, n] = dA_t h_{t-1}[p, n] + delta_t[h] x_t[h, p] Bm_t[g, n],   h_{-1} = h0[i, h] (0 when h0 is NULL)
 *   y_t[h, p] = sum_n Cm_t[g, n] h_t[p, n]
 *   h_final[i, h] = h at the last token (h0[i, h], or 0, for an empty sequence)
 * reverse = 1 runs from each sequence's end.  Chunked form over Q = 64 tokens of one sequence (16 for RUA_F64); the
 * carried state is kept in the accumulator type and never rounded.  For fp16 / bf16 the operands of the tensor-core
 * products are rounded to `dtype` once each (delta x, the decay-masked scores exp(cum_t - cum_s) (C_t . B_s), the
 * decay-weighted B of the state update and the copy of the state that C reads); fp32 / fp64 round only y.  Rows that
 * hold no token (L / R padding, C rows at or past off[B]) are copied through from x.  ragged->sorted is required
 * (B > 0); the sequence-to-CTA assignment is fixed, so every result is bit-identical run to run and, for the same
 * sequences, on every layout.  No float atomics; every sum runs in a fixed order. */

/* workspace of rua_ssd_backward (0 when rows, B or H is 0, or an argument is invalid), in accumulator-type values, with
 * grid = min(B G, 296), Q = 64 (16 for RUA_F64) and Tmax = ragged->Tp (at least the longest sequence):
 *   grid x H grad_A slots, rounded up to 256 bytes,
 *   + grid x (ceil(Tmax / Q) P N + Tmax 2N): per CTA, the chunk-start states of one head and [grad_B | grad_C] of one
 *     sequence.
 * Host only; monotone in every size argument. */
size_t rua_ssd_workspace_bytes(int64_t rows, int64_t B, int64_t Tmax, int64_t H, int32_t P, int32_t G, int32_t N,
                               int32_t dtype);

/* y (and h_final when not NULL) as above.  No workspace (ws may be NULL), and nothing is kept for the backward, which
 * recomputes the states it needs. */
int rua_ssd_forward(const void* x, const void* delta, const void* A, const void* Bm, const void* Cm, const void* h0,
                    void* y, void* h_final, int64_t H, int32_t P, int32_t G, int32_t N, int32_t dtype, int32_t reverse,
                    const rua_ragged_t* ragged, const rua_side_t* side, void* ws, size_t ws_bytes, rua_stream_t stream);

/* gradients of sum g y for the rua_ssd_forward call on the same x / delta / A / Bm / Cm / h0 / reverse / ragged / side.
 * In processing order, with dh_t the adjoint of h_t (0 past the last token):
 *   dh_t          = Cm_t[g] (x) g_t[h] + dA_{t+1} dh_{t+1}
 *   grad_x_t[h]   = delta_t[h] sum_n Bm_t[g, n] dh_t[., n]
 *   grad_delta_t  = A dA_t <dh_t, h_{t-1}> + <dh_t, x_t[h] (x) Bm_t[g]>
 *   grad_A[h]     = sum over all tokens of delta_t dA_t <dh_t, h_{t-1}>
 *   grad_Bm_t[g]  = sum_{h in g} delta_t[h] sum_p x_t[h, p] dh_t[p, .]
 *   grad_Cm_t[g]  = sum_{h in g} sum_p g_t[h, p] h_t[p, .]
 *   grad_h0[i, h] = dA_0 dh_0 (0 for an empty sequence)
 * grad_A and grad_h0 are of the accumulator type, the others of `dtype`.  Any gradient pointer may be NULL and is then not
 * written.  Rows that hold no token pass grad_out through to grad_x and get 0 in grad_delta, grad_Bm and grad_Cm.  The
 * unit of work is (sequence, group); per head it recomputes the chunk-start states, then walks the chunks from the end.
 * grad_Bm / grad_Cm are summed over a group's heads in head order, grad_A per CTA slot in slot order.  ws:
 * rua_ssd_workspace_bytes(side->rows, B, ragged->Tp, H, P, G, N, dtype) bytes; ragged->Tp must be at least the longest
 * sequence (the lengths live on the device): a longer sequence gets NaN in every gradient it reaches (its rows of
 * grad_x, grad_delta, grad_Bm, grad_Cm, its grad_h0 and grad_A of its heads).  No token at all: grad_x is copied from
 * grad_out and the other gradients are zeroed on `stream`. */
int rua_ssd_backward(const void* grad_out, const void* x, const void* delta, const void* A, const void* Bm, const void* Cm,
                     const void* h0, void* grad_x, void* grad_delta, void* grad_A, void* grad_Bm, void* grad_Cm,
                     void* grad_h0, int64_t H, int32_t P, int32_t G, int32_t N, int32_t dtype, int32_t reverse,
                     const rua_ragged_t* ragged, const rua_side_t* side, void* ws, size_t ws_bytes, rua_stream_t stream);

/* ------------------------------------------------------------------------------------------- */
/* K12 per-sequence gated delta rule (Gated DeltaNet): a scalar log decay and write strength per  */
/* token and value head, a K x V state per value head, q / k shared by the value heads of a key   */
/* group (no counterpart in the reference; replaces pad -> a pure-torch chunked form)             */
/* ------------------------------------------------------------------------------------------- */
/* v, o: side->rows rows of H x V elements; q, k: side->rows rows of G x K; beta: side->rows rows of H; all in the
 * storage of `side` (C, L, P or R over `ragged`; len_xform must be RUA_LEN_SAME) and of `dtype`.  g (side->rows rows of
 * H, the log decay), h0 / h_final (B, H, K, V) in sequence order (for P the index in ragged->off) are of the ACCUMULATOR
 * type (fp32, fp64 for RUA_F64).  1 <= K <= 128, 1 <= V <= 256, G >= 1, H >= 0, H % G == 0.  For token (i, t), value
 * head h and key group c = h / (H / G), with S the K x V state of head h:
 *   S'_t   = exp(g_t[h]) S_{t-1}                              S_{-1} = h0[i, h] (0 when h0 is NULL)
 *   u_t    = beta_t[h] (v_t[h] - S'_t^T k_t[c])
 *   S_t    = S'_t + k_t[c] (x) u_t
 *   o_t[h] = scale S_t^T q_t[c]
 *   h_final[i, h] = S at the last token (h0[i, h], or 0, for an empty sequence)
 * reverse = 1 runs from each sequence's end.  Chunked form over Q tokens of one sequence (64 for fp16 / bf16, 32 for
 * fp32, 16 for RUA_F64) and V blocks of 64 columns (32 for RUA_F64); the carried state, the per-chunk inverse
 * T = (I + strict_tril(diag(beta) (K K^T) o exp(cum_t - cum_s)))^-1, cum and every exponential are kept in the
 * accumulator type.  For fp16 / bf16 each operand of a tensor-core product is rounded to `dtype` once; fp32 / fp64
 * round only o.  Rows that hold no token (L / R padding, C rows at or past off[B]) are copied through from v.
 * ragged->sorted is required (B > 0); the sequence-to-CTA assignment is fixed, so every result is bit-identical run to
 * run and, for the same sequences, on every layout.  No float atomics; every sum runs in a fixed order. */

/* workspace of rua_gdn_backward (0 when rows, B or H is 0, or an argument is invalid), in accumulator-type values, with
 * grid = min(B G, 296), Q and VB as above and Tmax = ragged->Tp (at least the longest sequence):
 *   grid x (ceil(Tmax / Q) K VB + Tmax (2K + 2)): per CTA, the chunk-start states of one (head, V block) and
 *   [grad_q | grad_k | grad_g | grad_beta] of one sequence.
 * Host only; monotone in every size argument. */
size_t rua_gdn_workspace_bytes(int64_t rows, int64_t B, int64_t Tmax, int64_t H, int32_t G, int32_t K, int32_t V,
                               int32_t dtype);

/* o (and h_final when not NULL) as above.  No workspace (ws may be NULL), and nothing is kept for the backward, which
 * recomputes the states it needs. */
int rua_gdn_forward(const void* v, const void* q, const void* k, const void* g, const void* beta, const void* h0, void* o,
                    void* h_final, int64_t H, int32_t G, int32_t K, int32_t V, double scale, int32_t dtype,
                    int32_t reverse, const rua_ragged_t* ragged, const rua_side_t* side, void* ws, size_t ws_bytes,
                    rua_stream_t stream);

/* gradients of sum grad_out o for the rua_gdn_forward call on the same v / q / k / g / beta / h0 / scale / reverse /
 * ragged / side.  In processing order, with dS_t the adjoint of S_t (0 past the last token), p_t = S'_t^T k_t and
 * du_t = dS_t^T k_t after dS_t = scale q_t (x) grad_out_t + exp(g_{t+1}) (I - beta_{t+1} k_{t+1} k_{t+1}^T) dS_{t+1}:
 *   grad_v_t[h]      = beta_t du_t
 *   grad_beta_t[h]   = <du_t, v_t - p_t>
 *   grad_g_t[h]      = <dS_t - beta_t k_t (x) du_t, S'_t>
 *   grad_q_t[c]      = scale sum_{h in c} S_t grad_out_t[h]
 *   grad_k_t[c]      = sum_{h in c} (dS_t u_t - beta_t S'_t du_t)
 *   grad_h0[i, h]    = exp(g_0) (I - beta_0 k_0 k_0^T) dS_0 (0 for an empty sequence)
 * grad_g and grad_h0 are of the accumulator type, the others of `dtype`.  Any gradient pointer may be NULL and is then
 * not written.  Rows that hold no token pass grad_out through to grad_v and get 0 in grad_q, grad_k, grad_g and
 * grad_beta.  The unit of work is (sequence, key group); per (value head, V block) it recomputes the chunk-start states,
 * then walks the chunks from the end.  grad_q / grad_k are summed over a group's heads and V blocks, grad_g / grad_beta
 * over the V blocks, in that order.  ws: rua_gdn_workspace_bytes(side->rows, B, ragged->Tp, H, G, K, V, dtype) bytes;
 * ragged->Tp must be at least the longest sequence (the lengths live on the device): a longer sequence gets NaN in every
 * gradient it reaches (its rows of grad_v, grad_q, grad_k, grad_g, grad_beta and its grad_h0).  No token at all: grad_v
 * is copied from grad_out and the other gradients are zeroed on `stream`. */
int rua_gdn_backward(const void* grad_out, const void* v, const void* q, const void* k, const void* g, const void* beta,
                     const void* h0, void* grad_v, void* grad_q, void* grad_k, void* grad_g, void* grad_beta,
                     void* grad_h0, int64_t H, int32_t G, int32_t K, int32_t V, double scale, int32_t dtype,
                     int32_t reverse, const rua_ragged_t* ragged, const rua_side_t* side, void* ws, size_t ws_bytes,
                     rua_stream_t stream);

/* ------------------------------------------------------------------------------------------- */
/* K5  multi-GPU output gather over NVLink peer memory (SURVEY.md 8e-3; the reference is         */
/* single-device).  One process per GPU; the batch is sharded by sequence; every rank stores its */
/* rows directly into the output buffers ("windows") of all ranks of the node.                   */
/* ------------------------------------------------------------------------------------------- */
#define RUA_MAX_DESTINATIONS 16
#define RUA_PEER_HANDLE_BYTES 64

/* window = device allocation that other processes of the node can map (CUDA IPC).  alloc returns the
 * local pointer and a 64-byte handle to ship to the peers; open maps a peer's window into this
 * process (enables peer access lazily); close unmaps; free releases the local allocation.  These four
 * calls synchronise the device (cudaMalloc / cudaFree semantics); they are set-up, not data path. */
int rua_peer_window_alloc(size_t bytes, void** ptr, void* handle_host);
int rua_peer_window_open(const void* handle_host, void** ptr);
int rua_peer_window_close(void* ptr);
int rua_peer_window_free(void* ptr);

/* fused "local layout -> global C on every rank": the n_tokens tokens of the local shard are walked in cat
 * order; token (i, t) is read ONCE from the local source layout (src_side: C, L, R or P over `ragged`) and
 * stored at row dst_base_host[k][i] + t of destination k, for every k < n_dst <= RUA_MAX_DESTINATIONS.
 * dst_base_host[k] is a DEVICE array of B int64 (first row of local sequence i in destination k), or NULL
 * for "local cat row" (a contiguous local copy).  dst_host[k] are device pointers (local or peer windows);
 * both arrays themselves live on the host.  Replaces to_cat (torchrua/core/cast.py:8-16) + all_gather. */
int rua_row_map_multi(const void* src, int64_t row_bytes, const rua_ragged_t* ragged,
                      const rua_side_t* src_side, int64_t n_tokens, void* const* dst_host,
                      const int64_t* const* dst_base_host, int32_t n_dst, rua_stream_t stream);

/* per-sequence results (segment reductions, last(), head(1)): row j of src (n, row_bytes) is stored at row
 * index[j] of every destination. */
int rua_scatter_rows_multi(const void* src, const int64_t* index, int64_t n, int64_t row_bytes,
                           void* const* dst_host, int32_t n_dst, rua_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RUA_B200_H_ */
