// K1/K2 -- ragged row map: one kernel for the 12 layout conversions, head/last/rev/roll/trunc and
// all of their backward passes.
//
// Replaces (reference file:line): to_cat core/cast.py:8-16, cat_pack_to_left :19-23, right_to_left
// :26-32, to_pack :41-49, cat_pack_to_right :52-56, left_to_right :59-65, the (batch_ptr, token_ptr)
// branches of core/get.py:21-79 and core/set.py:23-92, select/head.py:6-67, last.py:7-13,
// rev.py:6-41, roll.py:6-37, trunc.py:9-62, reduce.py:64-69.
//
// The reference materialises ptr() index tensors (16*N bytes), a BxT int64 mask and a full
// `new_full` of the padded output before a generic aten::index / index_put_ moves the payload.
// Here the destination is walked ONCE in storage order; each warp decodes 32 destination rows in
// parallel (one lane per row: binary search in the L1/L2-resident offset arrays), then the whole
// warp moves those rows with 128-bit coalesced loads/stores, 4 independent vectors in flight per
// lane.  Padding is written by the same pass, so every output byte is stored exactly once and no
// payload byte is read twice: traffic = N*D read + rows_dst*D written (+ metadata).
// HBM-bound; no shared memory (no reuse) and no tensor cores (nothing to contract).
#include <cstring>

#include "common.cuh"
#include "dispatch.cuh"
#include "tile_decode.cuh"
#include "tma.cuh"

namespace rua {

struct RowMapParams {
  const uint8_t* src;
  uint8_t* dst;
  int64_t row_vecs;   // vectors per row
  rua_ragged_t rg;
  rua_side_t s;       // source side
  rua_side_t d;       // destination side
  int32_t tmap;
  int64_t tmap_arg;
  int32_t pad_mode;
  uint4 fill;         // fill pattern replicated to 16 bytes
  int32_t rows_per_warp;   // power of two <= 32
  int32_t lanes_per_row;   // power of two <= 32
  int32_t col_splits;      // gridDim.y
  const int64_t* gather_index;   // explicit source rows (rua_gather_rows) or NULL
  const int64_t* scatter_index;  // explicit destination rows (rua_scatter_rows) or NULL
  unsigned long long* index_errors;   // device counter of out-of-range explicit indices (rows skipped / zero-filled)
  // fused mask (rua_row_map_mask): one element per DESTINATION ROW, `one` where the row holds a token, else `zero`
  void* mask_out;
  int32_t mask_elem;                  // 1, 2, 4 or 8 bytes
  unsigned long long mask_zero, mask_one;
  uint32_t div_wrv_m, div_wrv_s;  // narrow padded destinations: x / (width * row_vecs) for x < 2^31 (FastDiv)
  uint32_t div_rv_m, div_rv_s;    //                             x / row_vecs
};

// unsigned division of x < 2^31 by a divisor fixed at launch: q = (x * m) >> s with m = floor(2^s / d) + 1,
// s = 31 + ceil(log2 d) (Granlund-Montgomery, N = 31); two instructions instead of the ~20 of a runtime
// 32-bit division -- the narrow-row kernels are issue-bound and divide once per 8-byte element
struct FastDiv {
  uint32_t m, s;
  __host__ static FastDiv make(uint64_t d) {
    FastDiv f;
    uint32_t l = 0;
    while ((1ull << l) < d) ++l;
    f.s = 31 + l;
    f.m = (uint32_t)((1ull << f.s) / d + 1);
    return f;
  }
};
__device__ __forceinline__ uint32_t fast_div(uint32_t x, uint32_t m, uint32_t s) {
  return (uint32_t)(((unsigned long long)x * m) >> s);
}

constexpr int kGenericSrc = -1;   // template tag: full generality (selects, transformed lengths, pad quirks)
constexpr int kSrcCatRev = 16;    // C -> C with the token order reversed (C.rev on narrow rows: token ids)
constexpr int kSrcCatRoll = 17;   // C -> C rolled by tmap_arg

// "simple" maps = the 12 layout conversions: identity token map, untransformed lengths, plain fill.  With the
// source layout known at compile time the per-element address is 2-4 instructions and no branches.
template <int SRC>
__device__ __forceinline__ int64_t simple_source_row(const RowMapParams& p, int64_t i, int64_t td, int64_t len) {
  if (SRC == RUA_CAT) return __ldg(p.rg.off + i) + td;
  if (SRC == RUA_LEFT) return i * p.s.width + td;
  if (SRC == RUA_RIGHT) return i * p.s.width + (p.s.width - len) + td;
  return __ldg(p.rg.poff + td) + __ldg(p.rg.unsorted + i);
}

constexpr int64_t kPadRow = -1;
constexpr int64_t kNoRow = -2;

// explicit index tensors follow torch semantics: negative entries wrap around once.  An entry that is still out of
// range is NOT dereferenced (ATen device-asserts there): gathers fill the row with zeros, scatters skip it, and
// the per-device error counter is bumped (rua_index_error_count).
__device__ __forceinline__ int64_t checked_index(const RowMapParams& p, int64_t v, int64_t bad) {
  if (v < 0) v += p.s.rows;
  if (v < 0 || v >= p.s.rows) {
    if (p.index_errors) atomicAdd(p.index_errors, 1ull);
    return bad;
  }
  return v;
}

__device__ __forceinline__ int64_t side_len(const rua_side_t& sd, int64_t base_len) {
  if (sd.len_xform == RUA_LEN_SAME) return base_len;
  if (sd.len_xform == RUA_LEN_CONST) return sd.len_arg;
  return base_len - sd.len_arg;
}

struct CatOff {  // exclusive prefix sum of the transformed lengths, in closed form
  const int64_t* __restrict__ off;
  int32_t xform;
  int64_t arg;
  __device__ __forceinline__ int64_t operator()(int64_t i) const {
    if (xform == RUA_LEN_SAME) return __ldg(off + i);
    if (xform == RUA_LEN_CONST) return arg * i;
    return __ldg(off + i) - arg * i;
  }
};

struct PackOff {  // trunc drops the first `shift` time steps of batch_sizes (select/trunc.py:42)
  const int64_t* __restrict__ poff;
  int64_t shift;
  __device__ __forceinline__ int64_t operator()(int64_t t) const {
    return __ldg(poff + t + shift) - __ldg(poff + shift);
  }
};

__device__ __forceinline__ int64_t pack_shift(const rua_side_t& sd) {
  return sd.len_xform == RUA_LEN_MINUS ? sd.len_arg : 0;
}

__device__ __forceinline__ int64_t source_row(const RowMapParams& p, int64_t i, int64_t td, int64_t base_len);

// destination row j -> source row (or kPadRow)
__device__ __forceinline__ int64_t map_row(const RowMapParams& p, int64_t j) {
  const rua_ragged_t& rg = p.rg;
  int64_t i, td;
  bool have_len = false;
  int64_t base_len = 0;
  if (p.d.layout == RUA_CAT) {
    CatOff f{rg.off, p.d.len_xform, p.d.len_arg};
    i = owner_search(f, rg.B, j);
    td = j - f(i);
  } else if (p.d.layout == RUA_PACK) {
    int64_t sh = pack_shift(p.d);
    PackOff f{rg.poff, sh};
    int64_t steps = p.d.len_xform == RUA_LEN_CONST ? p.d.len_arg : rg.Tp - sh;
    td = owner_search(f, steps, j);
    // rank inside the time step.  A row beyond the step's batch size exists only when poff does not describe `rows`
    // (the speculative C -> P launch of C.pack() whose cap turned out too small, or inconsistent metadata): treat it as
    // padding instead of reading sorted[] out of bounds (the result of such a launch is discarded by the caller).
    const int64_t base = f(td), r = j - base;
    if (r >= f(td + 1) - base) return kPadRow;
    i = __ldg(rg.sorted + r);
  } else {
    int64_t w = p.d.width;
    if (p.d.rows < (1ll << 31)) {
      uint32_t q = (uint32_t)j / (uint32_t)w;
      i = q;
      td = (uint32_t)j - q * (uint32_t)w;
    } else {
      i = j / w;
      td = j - i * w;
    }
    base_len = __ldg(rg.off + i + 1) - __ldg(rg.off + i);
    have_len = true;
    int64_t ld = side_len(p.d, base_len);
    if (p.d.layout == RUA_RIGHT) td -= (w - ld);
    if (td < 0 || td >= ld) return kPadRow;
  }
  if (!have_len) base_len = __ldg(rg.off + i + 1) - __ldg(rg.off + i);
  return source_row(p, i, td, base_len);
}

// token (i, t_d) of the destination -> source row (or kPadRow): token map, validity, source layout
__device__ __forceinline__ int64_t source_row(const RowMapParams& p, int64_t i, int64_t td, int64_t base_len) {
  const rua_ragged_t& rg = p.rg;
  int64_t ts;
  if (p.tmap == RUA_MAP_SHIFT) {
    ts = td + p.tmap_arg;
  } else if (p.tmap == RUA_MAP_REV) {
    ts = base_len - 1 - td;
  } else {
    int64_t m = (td - p.tmap_arg) % base_len;  // base_len > 0 here: a row exists
    ts = m < 0 ? m + base_len : m;
  }
  int64_t ls = side_len(p.s, base_len);
  if (p.pad_mode == RUA_PAD_WRAP && ts == -1) {
    // last() of an EMPTY sequence in the reference indexes position len-1 = -1, which wraps
    // (select/last.py:11-13): C reads row min(off[i], N-1) - 1 (mod N) because C.offsets() is clamped
    // (layout/cat.py:81); L and R read the last column of row i (core/get.py:42,74).
    if (p.s.layout == RUA_CAT) {
      int64_t o = __ldg(rg.off + i);
      o = (o < p.s.rows - 1 ? o : p.s.rows - 1) - 1;
      return o < 0 ? o + p.s.rows : o;
    }
    if (p.s.layout == RUA_LEFT || p.s.layout == RUA_RIGHT) return i * p.s.width + p.s.width - 1;
  }
  if (ts < 0 || ts >= ls) return kPadRow;

  switch (p.s.layout) {
    case RUA_CAT: {
      CatOff f{rg.off, p.s.len_xform, p.s.len_arg};
      const int64_t r = f(i) + ts;
      // lengths that describe more tokens than the storage holds (possible only inside the speculative C -> P launch of
      // C.pack(), before the host has seen N: the caller raises afterwards) must not read past the payload
      return r < p.s.rows ? r : kPadRow;
    }
    case RUA_LEFT:
      return i * p.s.width + ts;
    case RUA_RIGHT:
      return i * p.s.width + (p.s.width - ls) + ts;
    default: {
      int64_t sh = pack_shift(p.s);
      PackOff f{rg.poff, sh};
      return f(ts) + __ldg(rg.unsorted + i);
    }
  }
}

template <typename V> __device__ __forceinline__ V ld_stream(const V* p) { return __ldcs(p); }
template <typename V> __device__ __forceinline__ void st_stream(V* p, V v) { __stcs(p, v); }

// 256-bit global accesses (V256) are new with sm_100 (SASS LDG.E.ENL2.256 / STG.E.ENL2.256): one full 32-byte
// sector per lane and half the LSU instructions of the 128-bit form.  Used when rows are 32-byte multiples.
template <> __device__ __forceinline__ V256 ld_stream<V256>(const V256* p) {
  V256 v;
  asm volatile("ld.global.cs.v4.b64 {%0, %1, %2, %3}, [%4];" : "=l"(v.x), "=l"(v.y), "=l"(v.z), "=l"(v.w) : "l"(p));
  return v;
}
template <> __device__ __forceinline__ void st_stream<V256>(V256* p, V256 v) {
  asm volatile("st.global.cs.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(p), "l"(v.x), "l"(v.y), "l"(v.z), "l"(v.w) : "memory");
}

// the fill pattern is replicated over 16 bytes; a vector narrower than the element (possible only
// for oddly aligned views) picks the slice that matches its byte offset within the row
__device__ __forceinline__ uint32_t fill_word(const uint4& f, int w) {
  return w == 0 ? f.x : (w == 1 ? f.y : (w == 2 ? f.z : f.w));
}
template <typename V> __device__ __forceinline__ V make_fill(const uint4& f, int64_t byte_off);
template <> __device__ __forceinline__ uint4 make_fill<uint4>(const uint4& f, int64_t) { return f; }
template <> __device__ __forceinline__ V256 make_fill<V256>(const uint4& f, int64_t) {
  const unsigned long long lo = ((unsigned long long)f.y << 32) | f.x, hi = ((unsigned long long)f.w << 32) | f.z;
  return V256{lo, hi, lo, hi};
}
template <> __device__ __forceinline__ uint2 make_fill<uint2>(const uint4& f, int64_t o) {
  int w = (int)((o >> 2) & 2);
  return make_uint2(fill_word(f, w), fill_word(f, w + 1));
}
template <> __device__ __forceinline__ unsigned int make_fill<unsigned int>(const uint4& f, int64_t o) {
  return fill_word(f, (int)((o >> 2) & 3));
}
template <> __device__ __forceinline__ unsigned short make_fill<unsigned short>(const uint4& f, int64_t o) {
  return (unsigned short)((fill_word(f, (int)((o >> 2) & 3)) >> (8 * (int)(o & 2))) & 0xffffu);
}
template <> __device__ __forceinline__ unsigned char make_fill<unsigned char>(const uint4& f, int64_t o) {
  return (unsigned char)((fill_word(f, (int)((o >> 2) & 3)) >> (8 * (int)(o & 3))) & 0xffu);
}

constexpr int kRowMapThreads = 128;
constexpr int kUnroll = 4;

template <typename V>
__global__ void __launch_bounds__(kRowMapThreads)
row_map_kernel(const RowMapParams p) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (kRowMapThreads / 32) + (threadIdx.x >> 5);
  const int rpw = p.rows_per_warp;
  const int64_t rows = p.d.rows;
  const int64_t j0 = warp * rpw;
  if (j0 >= rows) return;

  // phase 1: one lane per destination row decodes where its bytes come from
  int64_t srow = kNoRow, drow = kNoRow;
  {
    int64_t j = j0 + lane;
    if (lane < rpw && j < rows) {
      if (p.gather_index) { srow = checked_index(p, __ldg(p.gather_index + j), kPadRow); drow = j; }
      else if (p.scatter_index) {
        drow = checked_index(p, __ldg(p.scatter_index + j), kNoRow);
        srow = drow == kNoRow ? kNoRow : j;
      }
      else { srow = map_row(p, j); drow = j; }
      if (p.mask_out && blockIdx.y == 0) {           // the same decode feeds the mask: coalesced, one element per lane
        const unsigned long long m = srow >= 0 ? p.mask_one : p.mask_zero;
        if (p.mask_elem == 1) reinterpret_cast<uint8_t*>(p.mask_out)[j] = (uint8_t)m;
        else if (p.mask_elem == 2) reinterpret_cast<uint16_t*>(p.mask_out)[j] = (uint16_t)m;
        else if (p.mask_elem == 4) reinterpret_cast<uint32_t*>(p.mask_out)[j] = (uint32_t)m;
        else reinterpret_cast<unsigned long long*>(p.mask_out)[j] = m;
      }
      if (srow == kPadRow && p.pad_mode == RUA_PAD_ROW0) srow = 0;
    }
  }

  // phase 2: the warp moves the rows; `lpr` lanes cooperate on one row, 32/lpr rows at a time
  const int lpr = p.lanes_per_row;
  const int groups = 32 / lpr;
  const int g = lane / lpr, l = lane - g * lpr;
  // column range of this CTA row (gridDim.y splits very wide rows across CTAs)
  const int64_t cols_per = ceil_div(p.row_vecs, (int64_t)p.col_splits);
  const int64_t c0 = (int64_t)blockIdx.y * cols_per;
  const int64_t c1 = c0 + cols_per < p.row_vecs ? c0 + cols_per : p.row_vecs;
  const V* __restrict__ src = reinterpret_cast<const V*>(p.src);
  V* __restrict__ dst = reinterpret_cast<V*>(p.dst);

  for (int r0 = 0; r0 < rpw; r0 += groups) {
    const int r = r0 + g;
    const int64_t s = shfl_i64(srow, r & 31);
    const int64_t dj = shfl_i64(drow, r & 31);
    if (r >= rpw || s == kNoRow) continue;
    V* drow_p = dst + dj * p.row_vecs;
    if (s >= 0) {
      const V* srow_p = src + s * p.row_vecs;
      constexpr int U = sizeof(V) >= 32 ? kUnroll / 2 : kUnroll;   // 64 bytes in flight per lane either way
      int64_t c = c0 + l;
      for (; c + (int64_t)(U - 1) * lpr < c1; c += (int64_t)U * lpr) {
        V v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = ld_stream(srow_p + c + (int64_t)u * lpr);
#pragma unroll
        for (int u = 0; u < U; ++u) st_stream(drow_p + c + (int64_t)u * lpr, v[u]);
      }
      for (; c < c1; c += lpr) st_stream(drow_p + c, ld_stream(srow_p + c));
    } else {
      for (int64_t c = c0 + l; c < c1; c += lpr)
        st_stream(drow_p + c, make_fill<V>(p.fill, c * (int64_t)sizeof(V)));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// constructors (C/L/P/R.new(list_of_tensors), torchrua/core/__init__.py:9-36; SURVEY.md 8f-3): the reference
// concatenates the list (one read + one write of N*D) and then converts (another pass).  Here sequence i stays
// in its own allocation: the destination is walked once and token (i, t) is read from src_list[i] + t * D.
// ------------------------------------------------------------------------------------------------
// destination row j -> (sequence, token) in the destination layout; false = padding
__device__ __forceinline__ bool decode_dst(const RowMapParams& p, int64_t j, int64_t& i, int64_t& td, int64_t& base_len) {
  const rua_ragged_t& rg = p.rg;
  if (p.d.layout == RUA_CAT) {
    GlobalOff f{rg.off};
    i = owner_search(f, rg.B, j);
    td = j - f(i);
    base_len = f(i + 1) - f(i);
    return true;
  }
  if (p.d.layout == RUA_PACK) {
    GlobalOff f{rg.poff};
    td = owner_search(f, rg.Tp, j);
    i = __ldg(rg.sorted + (j - f(td)));
    base_len = __ldg(rg.off + i + 1) - __ldg(rg.off + i);
    return true;
  }
  const int64_t w = p.d.width;
  i = j / w;
  td = j - i * w;
  base_len = __ldg(rg.off + i + 1) - __ldg(rg.off + i);
  if (p.d.layout == RUA_RIGHT) td -= (w - base_len);
  return td >= 0 && td < base_len;
}

// With p.gather_index the list holds n_src whole TENSORS instead (compose, torchrua/compose.py:9-33): destination row j
// copies row index[j] of their virtual concatenation, bases[k] = first row of tensor k in it (bases[n_src] = total).
template <typename V>
__global__ void __launch_bounds__(kRowMapThreads)
row_map_list_kernel(const RowMapParams p, const uint8_t* const* __restrict__ src_list, int64_t row_bytes,
                    const int64_t* __restrict__ bases = nullptr, int n_src = 0) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (kRowMapThreads / 32) + (threadIdx.x >> 5);
  const int rpw = p.rows_per_warp;
  const int64_t rows = p.d.rows;
  const int64_t j0 = warp * rpw;
  if (j0 >= rows) return;
  // phase 1: one lane per destination row finds the ADDRESS its bytes come from (0 = padding, -1 = no row)
  long long saddr = -1;
  {
    const int64_t j = j0 + lane;
    if (lane < rpw && j < rows) {
      if (p.gather_index) {
        const int64_t total = __ldg(bases + n_src);
        int64_t r = __ldg(p.gather_index + j);
        if (r < 0) r += total;
        if (r < 0 || r >= total) {                     // out of range: zero row, counted (see checked_index)
          if (p.index_errors) atomicAdd(p.index_errors, 1ull);
          saddr = 0;
        } else {
          int lo = 0, hi = n_src;
          while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(bases + mid) <= r) lo = mid; else hi = mid;
          }
          saddr = (long long)__ldg(reinterpret_cast<const unsigned long long*>(src_list) + lo) + (r - __ldg(bases + lo)) * row_bytes;
        }
      } else {
        int64_t i, td, len;
        saddr = decode_dst(p, j, i, td, len) ? (long long)__ldg(reinterpret_cast<const unsigned long long*>(src_list) + i) + td * row_bytes : 0;
      }
    }
  }
  const int lpr = p.lanes_per_row;
  const int groups = 32 / lpr;
  const int g = lane / lpr, l = lane - g * lpr;
  const int64_t cols_per = ceil_div(p.row_vecs, (int64_t)p.col_splits);
  const int64_t c0 = (int64_t)blockIdx.y * cols_per;
  const int64_t c1 = c0 + cols_per < p.row_vecs ? c0 + cols_per : p.row_vecs;
  V* __restrict__ dst = reinterpret_cast<V*>(p.dst);
  for (int r0 = 0; r0 < rpw; r0 += groups) {
    const int r = r0 + g;
    const long long sa = shfl_i64(saddr, r & 31);
    if (r >= rpw || sa == -1) continue;
    V* drow_p = dst + (j0 + r) * p.row_vecs;
    if (sa != 0) {
      const V* srow_p = reinterpret_cast<const V*>((uintptr_t)sa);
      constexpr int U = sizeof(V) >= 32 ? kUnroll / 2 : kUnroll;
      int64_t c = c0 + l;
      for (; c + (int64_t)(U - 1) * lpr < c1; c += (int64_t)U * lpr) {
        V v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = ld_stream(srow_p + c + (int64_t)u * lpr);
#pragma unroll
        for (int u = 0; u < U; ++u) st_stream(drow_p + c + (int64_t)u * lpr, v[u]);
      }
      for (; c < c1; c += lpr) st_stream(drow_p + c, ld_stream(srow_p + c));
    } else {
      for (int64_t c = c0 + l; c < c1; c += lpr) st_stream(drow_p + c, make_fill<V>(p.fill, c * (int64_t)sizeof(V)));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K5 -- fused conversion + output gather (multi-GPU, SURVEY.md 8e-3).  The tokens of the LOCAL shard are
// walked in cat order; token (i, t) is read once from the local source layout (C, L, R or P) and stored
// to row base_k[i] + t of EVERY destination k: the windows of all peer GPUs (plain stores through NVLink
// peer mappings: fire-and-forget, coalesced 32-byte sectors) and, optionally, a local contiguous copy
// (base == NULL: row j).  One pass replaces "convert, all_gather padded shards, permute into global order".
// With rows_are_sequences the source is a plain (n, *) matrix of per-sequence results (segment reductions,
// last(), head(1)): row j goes to row base_k[j].
// ------------------------------------------------------------------------------------------------
constexpr int kMaxDst = RUA_MAX_DESTINATIONS;
struct MultiDst {
  uint8_t* dst[kMaxDst];
  const int64_t* base[kMaxDst];
  int32_t n;
  int32_t rows_are_sequences;
};

// The grid may be CAPPED (launch_row_map_multi): with many destinations the kernel is bound by the NVLink wire, not by
// SM issue, so a few CTAs per SM walk the rows in a grid-stride loop and leave the remaining CTA slots of every SM to
// the HBM-bound conversions of the next micro-batch running on another stream (true overlap instead of time slicing).
template <typename V>
__global__ void __launch_bounds__(kRowMapThreads)
row_map_multi_kernel(const RowMapParams p, const MultiDst m) {
  const int lane = threadIdx.x & 31;
  const int rpw = p.rows_per_warp;
  const int64_t rows = p.d.rows;
  const int64_t warps_total = (int64_t)gridDim.x * (kRowMapThreads / 32);
  for (int64_t warp = (int64_t)blockIdx.x * (kRowMapThreads / 32) + (threadIdx.x >> 5); warp * rpw < rows; warp += warps_total) {
  const int64_t j0 = warp * rpw;

  int64_t srow = kNoRow, seq = 0, tok = 0;
  {
    const int64_t j = j0 + lane;
    if (lane < rpw && j < rows) {
      if (m.rows_are_sequences) {
        srow = j; seq = j; tok = 0;
      } else {
        GlobalOff f{p.rg.off};
        seq = owner_search(f, p.rg.B, j);
        const int64_t o = f(seq);
        tok = j - o;
        srow = source_row(p, seq, tok, f(seq + 1) - o);
      }
    }
  }
  const int lpr = p.lanes_per_row;
  const int groups = 32 / lpr;
  const int g = lane / lpr, l = lane - g * lpr;
  const int64_t cols_per = ceil_div(p.row_vecs, (int64_t)p.col_splits);
  const int64_t c0 = (int64_t)blockIdx.y * cols_per;
  const int64_t c1 = c0 + cols_per < p.row_vecs ? c0 + cols_per : p.row_vecs;
  const V* __restrict__ src = reinterpret_cast<const V*>(p.src);
  const int n = m.n;
  const int k0 = (int)(warp % n);   // neighbouring warps start with different peers: all links busy at any instant

  for (int r0 = 0; r0 < rpw; r0 += groups) {
    const int r = r0 + g;
    const int64_t s = shfl_i64(srow, r & 31);
    const int64_t si = shfl_i64(seq, r & 31);
    const int64_t st = shfl_i64(tok, r & 31);
    if (r >= rpw || s < 0) continue;
    const int64_t jl = j0 + r;      // local cat row
    const V* srow_p = src + s * p.row_vecs;
    constexpr int U = sizeof(V) >= 32 ? kUnroll / 2 : kUnroll;
    int64_t c = c0 + l;
    for (; c + (int64_t)(U - 1) * lpr < c1; c += (int64_t)U * lpr) {
      V v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) v[u] = ld_stream(srow_p + c + (int64_t)u * lpr);
      for (int kk = 0; kk < n; ++kk) {
        const int k = k0 + kk < n ? k0 + kk : k0 + kk - n;
        const int64_t dj = m.base[k] ? __ldg(m.base[k] + si) + st : jl;
        V* drow_p = reinterpret_cast<V*>(m.dst[k]) + dj * p.row_vecs;
#pragma unroll
        for (int u = 0; u < U; ++u) st_stream(drow_p + c + (int64_t)u * lpr, v[u]);
      }
    }
    for (; c < c1; c += lpr) {
      const V v = ld_stream(srow_p + c);
      for (int kk = 0; kk < n; ++kk) {
        const int k = k0 + kk < n ? k0 + kk : k0 + kk - n;
        const int64_t dj = m.base[k] ? __ldg(m.base[k] + si) + st : jl;
        st_stream(reinterpret_cast<V*>(m.dst[k]) + dj * p.row_vecs + c, v);
      }
    }
  }
  }   // grid-stride loop over the warps' row groups
}

// ------------------------------------------------------------------------------------------------
// narrow rows (< 128 bytes: token ids, indices, scalars -- BASELINE config 5).  A 20-step binary
// search per 8-byte row would dominate, so here a CTA owns a TILE of consecutive destination
// vectors: one warp-cooperative 32-ary search per tile end finds the segments (sequences or time
// steps) that intersect the tile, their offsets are staged in shared memory, and every thread
// resolves its row with a short shared-memory search.  One thread moves one vector; consecutive
// lanes touch consecutive addresses on the destination side.
// ------------------------------------------------------------------------------------------------
constexpr int kTileThreads = 256;
constexpr int kTileItems = 8;
constexpr int kTileVecs = kTileThreads * kTileItems;  // 2048 destination vectors per CTA
constexpr int kTileCap = kTileVecs + 2;               // staged segment starts
static_assert(kTileThreads == kDecThreads && kTileVecs == kDecTile, "tile_decode.cuh assumes the same tile shape");

template <typename V, int SRC, typename OffFn>
__device__ __forceinline__ void tile_body(const RowMapParams& p, OffFn f, int64_t S, TileDecodeSmem& sm) {
  // Everything inside a tile is 32-bit and tile-relative (a tile spans 2048 vectors): these kernels are
  // ISSUE-bound (ncu: 65 % issue-active at 19 % DRAM), so 64-bit divisions and per-row searches are what
  // they cannot afford.  The tile's destination rows are decoded once (tile_decode.cuh); a row then finds
  // its segment with two shared-memory reads.
  const int tid = threadIdx.x;
  const int64_t total = p.d.rows * p.row_vecs;
  const int64_t e0 = (int64_t)blockIdx.x * kTileVecs;
  const int n_e = (int)(e0 + kTileVecs < total ? kTileVecs : total - e0);  // vectors in this tile
  const uint32_t rv = (uint32_t)p.row_vecs;                                 // < 8 (rows are < 128 bytes)
  const int64_t r0 = rv == 1 ? e0 : e0 / rv;                                // first destination row
  const uint32_t c0 = rv == 1 ? 0u : (uint32_t)(e0 - r0 * rv);              // column of the first vector
  const int64_t r1 = rv == 1 ? e0 + n_e - 1 : (e0 + n_e - 1) / rv;          // last destination row
  const TileDecode dec = tile_decode(f, S, r0, (int)(r1 - r0 + 1), sm);
  const bool staged = dec.staged;
  const int64_t first = dec.first;
  const int* s_rel = sm.rel;

  const V* __restrict__ src = reinterpret_cast<const V*>(p.src);
  V* __restrict__ dst = reinterpret_cast<V*>(p.dst) + e0;
  const bool is_pack = p.d.layout == RUA_PACK;
  const bool len_from_stage = staged && !is_pack && p.d.len_xform == RUA_LEN_SAME;
  int64_t srow[kTileItems];
  uint32_t col[kTileItems];
#pragma unroll
  for (int r = 0; r < kTileItems; ++r) {
    const int e = r * kTileThreads + tid;        // vector index inside the tile
    srow[r] = kNoRow;
    col[r] = 0;
    if (e < n_e) {
      uint32_t jr;                               // tile-relative destination row
      if (rv == 1) { jr = (uint32_t)e; }
      else { const uint32_t q = (uint32_t)e + c0; jr = q / rv; col[r] = q - jr * rv; }
      int64_t s, base;
      int64_t base_len = -1;
      if (staged) {
        const int lo = sm.seg[jr];               // segments first+1 .. first+lo start at or before this row
        s = first + lo;
        base = lo == 0 ? dec.off_first : r0 + s_rel[lo];
        if (len_from_stage && lo > 0 && s_rel[lo + 1] <= kTileVecs) base_len = s_rel[lo + 1] - s_rel[lo];
      } else {
        s = owner_search(f, S, r0 + jr);
        base = f(s);
      }
      const int64_t j = r0 + jr;
      int64_t i, td;
      bool undescribed = false;                  // see map_row: rows of a P that poff does not describe (branch-free: a
      if (is_pack) {                             // `continue` here cost the unrolled decode of EVERY instance 8-16 %)
        td = s;
        undescribed = j - base >= f(s + 1) - base;
        i = __ldg(p.rg.sorted + (undescribed ? 0 : j - base));
      } else { i = s; td = j - base; }
      int64_t sr;
      if (SRC == kGenericSrc) {
        if (base_len < 0) base_len = __ldg(p.rg.off + i + 1) - __ldg(p.rg.off + i);
        sr = source_row(p, i, td, base_len);
        if (sr == kPadRow && p.pad_mode == RUA_PAD_ROW0) sr = 0;
      } else if (SRC == kSrcCatRev || SRC == kSrcCatRoll) {   // same layout on both sides: segment start + mapped token
        if (base_len < 0) base_len = __ldg(p.rg.off + i + 1) - base;
        int64_t ts;
        if (SRC == kSrcCatRev) {
          ts = base_len - 1 - td;
        } else {
          const int64_t m = (td - p.tmap_arg) % base_len;
          ts = m < 0 ? m + base_len : m;
        }
        sr = base + ts;
      } else {                                   // conversions: every destination token of C / P exists in the source
        if (SRC == RUA_RIGHT && base_len < 0) base_len = __ldg(p.rg.off + i + 1) - __ldg(p.rg.off + i);
        sr = simple_source_row<SRC>(p, i, td, base_len);
        if (SRC == RUA_CAT && sr >= p.s.rows) sr = kPadRow;   // see source_row: inconsistent lengths never read past the payload
      }
      srow[r] = undescribed ? kPadRow : sr;
    }
  }
  V val[kTileItems];
#pragma unroll
  for (int r = 0; r < kTileItems; ++r)
    if (srow[r] >= 0) val[r] = ld_stream(src + (rv == 1 ? srow[r] : srow[r] * rv + col[r]));
#pragma unroll
  for (int r = 0; r < kTileItems; ++r) {
    const int e = r * kTileThreads + tid;
    if (srow[r] >= 0) st_stream(dst + e, val[r]);
    else if (srow[r] == kPadRow) st_stream(dst + e, make_fill<V>(p.fill, (int64_t)col[r] * (int64_t)sizeof(V)));
  }
}

// four consecutive vectors as one wide store (256-bit for 8-byte vectors: a full sector per lane)
template <typename V> __device__ __forceinline__ void store4(V* p, const V& a, const V& b, const V& c, const V& d) {
  st_stream(p, a); st_stream(p + 1, b); st_stream(p + 2, c); st_stream(p + 3, d);
}
template <> __device__ __forceinline__ void store4<uint2>(uint2* p, const uint2& a, const uint2& b, const uint2& c, const uint2& d) {
  auto u64 = [](const uint2& v) { return ((unsigned long long)v.y << 32) | v.x; };
  st_stream(reinterpret_cast<V256*>(p), V256{u64(a), u64(b), u64(c), u64(d)});
}
template <> __device__ __forceinline__ void store4<unsigned int>(unsigned int* p, const unsigned int& a, const unsigned int& b,
                                                                 const unsigned int& c, const unsigned int& d) {
  st_stream(reinterpret_cast<uint4*>(p), make_uint4(a, b, c, d));
}
template <> __device__ __forceinline__ void store4<uint4>(uint4* p, const uint4& a, const uint4& b, const uint4& c, const uint4& d) {
  auto u64 = [](unsigned lo, unsigned hi) { return ((unsigned long long)hi << 32) | lo; };
  st_stream(reinterpret_cast<V256*>(p), V256{u64(a.x, a.y), u64(a.z, a.w), u64(b.x, b.y), u64(b.z, b.w)});
  st_stream(reinterpret_cast<V256*>(p) + 1, V256{u64(c.x, c.y), u64(c.z, c.w), u64(d.x, d.y), u64(d.z, d.w)});
}

// L / R -> C, C.rev, C.roll with ONE-VECTOR rows: the same idea as row_map_padded_cat1_kernel on the decoded tile --
// a thread owns four consecutive rows of C, reads their segment indices with one 128-bit shared-memory load, resolves
// the segment once (twice when the group crosses a boundary), loads four vectors and stores them as one wide store.
struct ScaledOff {   // offsets counted in vectors: a sequence of C is one contiguous run of len * rv vectors
  const int64_t* __restrict__ p;
  int64_t rv;
  __device__ __forceinline__ int64_t operator()(int64_t i) const { return __ldg(p + i) * rv; }
};

template <typename V, int SRC>
__global__ void __launch_bounds__(kTileThreads)
row_map_tile_cat1_kernel(const RowMapParams p) {
  __shared__ TileDecodeSmem sm;
  const int tid = threadIdx.x;
  // L / R sources: positions, offsets, lengths and widths are all counted in VECTORS (rows of several vectors are
  // contiguous on both sides); rev / roll permute tokens and run with one vector per row only (rv == 1)
  const int64_t rv = (SRC == RUA_LEFT || SRC == RUA_RIGHT) ? p.row_vecs : 1;
  const int64_t total = p.d.rows * rv;
  const int64_t e0 = (int64_t)blockIdx.x * kTileVecs;
  const int n_e = (int)(e0 + kTileVecs < total ? kTileVecs : total - e0);
  ScaledOff f{p.rg.off, rv};
  const TileDecode dec = tile_decode(f, p.rg.B, e0, n_e, sm);
  const V* __restrict__ src = reinterpret_cast<const V*>(p.src);
  V* __restrict__ dst = reinterpret_cast<V*>(p.dst) + e0;
  const int64_t W = p.s.width * rv;
#pragma unroll
  for (int g = 0; g < kTileItems / 4; ++g) {
    const int eb = (g * kTileThreads + tid) * 4;
    if (eb >= n_e) break;
    int kk[4];
    if (dec.staged) {
      const int4 k4 = reinterpret_cast<const int4*>(sm.seg)[eb >> 2];
      kk[0] = k4.x; kk[1] = k4.y; kk[2] = k4.z; kk[3] = k4.w;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) kk[j] = (int)(owner_search(f, p.rg.B, e0 + (eb + j < n_e ? eb + j : n_e - 1)) - dec.first);
    }
    int64_t srow[4];
    int k_prev = -1;
    int64_t base = 0, len = 0, i = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = kk[j];
      if (k != k_prev) {                       // a group rarely crosses a boundary: one lookup for all four
        k_prev = k;
        i = dec.first + k;
        if (dec.staged && k > 0) {
          const int r = sm.rel[k], nx = sm.rel[k + 1];
          base = e0 + r;
          len = nx <= kTileVecs ? (int64_t)(nx - r) : f(i + 1) - base;
        } else {
          base = f(i);
          len = f(i + 1) - base;
        }
      }
      const int64_t td = e0 + eb + j - base;
      if (SRC == RUA_LEFT) srow[j] = i * W + td;
      else if (SRC == RUA_RIGHT) srow[j] = i * W + (W - len) + td;
      else if (SRC == kSrcCatRev) srow[j] = base + (len - 1 - td);
      else { const int64_t m = (td - p.tmap_arg) % len; srow[j] = base + (m < 0 ? m + len : m); }
    }
    V v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (eb + j < n_e) v[j] = ld_stream(src + srow[j]);
    if (eb + 4 <= n_e) {
      store4<V>(dst + eb, v[0], v[1], v[2], v[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (eb + j < n_e) st_stream(dst + eb + j, v[j]);
    }
  }
}

// L / R -> C, C.rev, C.roll with ONE-VECTOR rows and MANY SHORT sequences (BASELINE config 5: 1 M sequences of 1..64 token
// ids): the decomposition of emit_ptr_warpseg_kernel (emit.cu) with the payload attached.  A warp owns 32 consecutive
// sequences = one contiguous range of C rows; lane i reads off[s0 + i], off[s0 + i + 1] (coalesced: no search, no per-tile
// decode chain, no block barrier), paints its lane number over its sequence's rows in a 2 KB byte window of shared memory,
// and the warp then walks the window four rows per lane: one LDS.32 gives the four owners, a shuffle fetches each owner's
// source constant, four loads, ONE wide store.
constexpr int kWcThreads = 256;
constexpr int kWcWarps = kWcThreads / 32;
constexpr int kWcWin = 2048;   // C rows per window

template <typename V, int SRC>
__global__ void __launch_bounds__(kWcThreads)
row_map_warpseg_cat1_kernel(const RowMapParams p) {
  __shared__ __align__(16) unsigned char s_own[kWcWarps][kWcWin];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t S = p.rg.B, n = p.d.rows;
  const int64_t s0 = ((int64_t)blockIdx.x * kWcWarps + warp) * 32;
  if (s0 >= S) return;                                   // warp-uniform; no block-level synchronisation below
  const int64_t s = s0 + lane;
  int64_t beg = s < S ? __ldg(p.rg.off + s) : n, end = s < S ? __ldg(p.rg.off + s + 1) : n;
  const int64_t len = end - beg;
  beg = beg < n ? beg : n;
  end = end < n ? end : n;
  const int64_t wbeg = shfl_i64(beg, 0), wend = shfl_i64(end, 31);
  const int64_t W = p.s.width;
  // source row of C row q (owned by this lane's sequence):   L: q + c   R: q + c   rev: c - q   roll: beg + (q - beg - sh) mod len
  int64_t c = 0;
  if (SRC == RUA_LEFT) c = s * W - beg;
  else if (SRC == RUA_RIGHT) c = s * W + (W - len) - beg;
  else if (SRC == kSrcCatRev) c = 2 * beg + len - 1;
  int64_t sh = 0;
  if (SRC == kSrcCatRoll && len > 0) { sh = p.tmap_arg % len; if (sh < 0) sh += len; }
  const V* __restrict__ src = reinterpret_cast<const V*>(p.src);
  V* __restrict__ dst = reinterpret_cast<V*>(p.dst);
  unsigned char* own = s_own[warp];
  for (int64_t w0 = wbeg & ~(int64_t)3; w0 < wend; w0 += kWcWin) {
    const int64_t w1 = w0 + kWcWin < wend ? w0 + kWcWin : wend;
    const unsigned who = __ballot_sync(kFullMask, beg <= w0 && end >= w0 + kWcWin);
    if (!who) {
      const int64_t lo64 = beg < w0 ? w0 : (beg > w1 ? w1 : beg), hi64 = end < w0 ? w0 : (end > w1 ? w1 : end);
      int q = (int)(lo64 - w0);
      const int hi = (int)(hi64 - w0);
      for (; q < hi && (q & 3); ++q) own[q] = (unsigned char)lane;
      const unsigned word = (unsigned)lane * 0x01010101u;
      for (; q + 4 <= hi; q += 4) *reinterpret_cast<unsigned*>(own + q) = word;
      for (; q < hi; ++q) own[q] = (unsigned char)lane;
    }
    __syncwarp();
    const int groups = (int)((w1 - w0 + 3) >> 2);
    for (int g0 = 0; g0 < groups; g0 += 32) {
      const int g = g0 + lane;
      int o[4];
      if (who) {
        o[0] = o[1] = o[2] = o[3] = __ffs(who) - 1;
      } else {
        const uchar4 b = reinterpret_cast<const uchar4*>(own)[g < groups ? g : 0];
        o[0] = b.x & 31; o[1] = b.y & 31; o[2] = b.z & 31; o[3] = b.w & 31;   // unpainted bytes: any lane, never loaded
      }
      const int64_t q0 = w0 + 4 * (int64_t)g;
      int64_t from[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int64_t q = q0 + e;
        if (SRC == kSrcCatRoll) {
          const int64_t ob = shfl_i64(beg, o[e]), ol = shfl_i64(len, o[e]), os = shfl_i64(sh, o[e]);
          int64_t u = q - ob - os;
          if (u < 0) u += ol;
          from[e] = ob + u;
        } else {
          const int64_t oc = shfl_i64(c, o[e]);
          from[e] = SRC == kSrcCatRev ? oc - q : q + oc;
        }
      }
      if (g >= groups) continue;
      V v[4];
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (q0 + e >= wbeg && q0 + e < w1) v[e] = ld_stream(src + from[e]);
      if (q0 >= wbeg && q0 + 4 <= w1) {
        store4<V>(dst + q0, v[0], v[1], v[2], v[3]);
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (q0 + e >= wbeg && q0 + e < w1) st_stream(dst + q0 + e, v[e]);
      }
    }
    __syncwarp();
  }
}

// destination C or P: segment search through shared memory
template <typename V, int SRC>
__global__ void __launch_bounds__(kTileThreads)
row_map_tile_kernel(const RowMapParams p) {
  __shared__ TileDecodeSmem sm;
  if (p.d.layout == RUA_CAT) {
    CatOff f{p.rg.off, p.d.len_xform, p.d.len_arg};
    tile_body<V, SRC>(p, f, p.rg.B, sm);
  } else {
    const int64_t sh = pack_shift(p.d);
    PackOff f{p.rg.poff, sh};
    const int64_t steps = p.d.len_xform == RUA_LEN_CONST ? p.d.len_arg : p.rg.Tp - sh;
    tile_body<V, SRC>(p, f, steps, sm);
  }
}

// destination L or R (and the explicit-index gather/scatter): the decode is arithmetic, no staging
template <typename V>
__global__ void __launch_bounds__(kTileThreads)
row_map_flat_kernel(const RowMapParams p) {
  const int64_t total = p.d.rows * p.row_vecs;
  const int64_t e0 = (int64_t)blockIdx.x * kTileVecs;
  const V* __restrict__ src = reinterpret_cast<const V*>(p.src);
  V* __restrict__ dst = reinterpret_cast<V*>(p.dst);
  int64_t srow[kTileItems], drow[kTileItems], col[kTileItems];
#pragma unroll
  for (int r = 0; r < kTileItems; ++r) {
    const int64_t e = e0 + (int64_t)r * kTileThreads + threadIdx.x;
    srow[r] = kNoRow;
    if (e < total) {
      int64_t j;
      if (total < (1ll << 31)) { j = (uint32_t)e / (uint32_t)p.row_vecs; } else { j = e / p.row_vecs; }
      col[r] = e - j * p.row_vecs;
      drow[r] = j;
      int64_t sr;
      if (p.gather_index) { sr = checked_index(p, __ldg(p.gather_index + j), kPadRow); }
      else if (p.scatter_index) {
        const int64_t d = checked_index(p, __ldg(p.scatter_index + j), kNoRow);
        drow[r] = d;
        sr = d == kNoRow ? kNoRow : j;
      }
      else sr = map_row(p, j);
      if (sr == kPadRow && p.pad_mode == RUA_PAD_ROW0) sr = 0;
      srow[r] = sr;
    }
  }
  V val[kTileItems];
#pragma unroll
  for (int r = 0; r < kTileItems; ++r)
    if (srow[r] >= 0) val[r] = ld_stream(src + srow[r] * p.row_vecs + col[r]);
#pragma unroll
  for (int r = 0; r < kTileItems; ++r) {
    if (srow[r] >= 0) st_stream(dst + drow[r] * p.row_vecs + col[r], val[r]);
    else if (srow[r] == kPadRow) st_stream(dst + drow[r] * p.row_vecs + col[r], make_fill<V>(p.fill, col[r] * (int64_t)sizeof(V)));
  }
}

// destination L or R with narrow rows: the decode is arithmetic, but a 64-bit division and two global
// length loads per 8-byte element are still too many instructions.  A CTA owns 2048 consecutive
// destination vectors = a run of consecutive sequences; their offsets are staged once in shared memory
// (tile-relative, 32-bit), and every thread needs one 32-bit division by a CTA-uniform constant.
template <typename V, int SRC>
__global__ void __launch_bounds__(kTileThreads)
row_map_padded_kernel(const RowMapParams p) {
  __shared__ int s_rel[kTileCap];            // off[i0 + k] - off[i0]; clamped only beyond the tile's reach
  const int tid = threadIdx.x;
  const int64_t total = p.d.rows * p.row_vecs;
  const int64_t e0 = (int64_t)blockIdx.x * kTileVecs;
  const int n_e = (int)(e0 + kTileVecs < total ? kTileVecs : total - e0);
  const uint32_t rv = (uint32_t)p.row_vecs;
  const int64_t wrv64 = p.d.width * p.row_vecs;   // vectors per padded sequence
  const int64_t i0 = e0 / wrv64;                  // first sequence of the tile (one 64-bit division per CTA)
  const int64_t i1 = (e0 + n_e - 1) / wrv64;
  const int64_t head64 = e0 - i0 * wrv64;         // offset of the tile's first vector inside sequence i0
  const int cnt = (int)(i1 - i0 + 2);             // <= 2050 because every sequence holds >= 1 vector
  const int64_t base0 = __ldg(p.rg.off + i0);
  for (int k = tid; k < cnt; k += kTileThreads) {
    const int64_t d = __ldg(p.rg.off + i0 + k) - base0;
    s_rel[k] = d > (1 << 30) ? (1 << 30) : (int)d;   // lengths >= 2^30 only matter as "longer than the width"
  }
  __syncthreads();
  // when a padded row is longer than the tile, (head + e) can exceed 32 bits only if wrv64 does: then the
  // tile lies inside ONE sequence and the quotient is 0
  const bool one_seq = wrv64 > (int64_t)(1u << 30);
  const uint32_t wrv = one_seq ? 1u : (uint32_t)wrv64;
  const uint32_t head = one_seq ? 0u : (uint32_t)head64;
  const uint32_t width = (uint32_t)(p.d.width < (1ll << 30) ? p.d.width : (1ll << 30));
  const bool right_dst = p.d.layout == RUA_RIGHT;

  const V* __restrict__ src = reinterpret_cast<const V*>(p.src);
  V* __restrict__ dst = reinterpret_cast<V*>(p.dst) + e0;
  int64_t srow[kTileItems];
  uint32_t col[kTileItems];
#pragma unroll
  for (int r = 0; r < kTileItems; ++r) {
    const int e = r * kTileThreads + tid;
    srow[r] = kNoRow;
    col[r] = 0;
    if (e < n_e) {
      uint32_t q, t, c;
      if (one_seq) {
        const int64_t rem = head64 + e;
        q = 0;
        t = (uint32_t)(rem / rv);
        c = (uint32_t)(rem - (int64_t)t * rv);
      } else {
        const uint32_t x = head + (uint32_t)e;             // < 2^31: head < wrv <= 2^30, e < 2048
        q = fast_div(x, p.div_wrv_m, p.div_wrv_s);
        const uint32_t rem = x - q * wrv;
        if (rv == 1) { t = rem; c = 0; } else { t = fast_div(rem, p.div_rv_m, p.div_rv_s); c = rem - t * rv; }
      }
      col[r] = c;
      int64_t sr = kPadRow;
      if (SRC == kGenericSrc) {
        const int64_t base_len = (int64_t)s_rel[q + 1] - (int64_t)s_rel[q];   // exact unless >= 2^30 (then > width anyway)
        const int64_t ld = side_len(p.d, base_len);
        int64_t td = t;
        if (p.d.layout == RUA_RIGHT) td -= ((int64_t)width - ld);
        if (td >= 0 && td < ld) sr = source_row(p, i0 + q, td, base_len);
        if (sr == kPadRow && p.pad_mode == RUA_PAD_ROW0) sr = 0;
      } else {                                   // conversions: 32-bit, branch-free up to the validity test
        const int sq = s_rel[q];
        const int len = s_rel[q + 1] - sq;       // >= 2^30 only when it exceeds the width anyway
        const int td = (int)t - (right_dst ? (int)width - len : 0);
        if (td >= 0 && td < len)
          sr = SRC == RUA_CAT ? base0 + sq + td : simple_source_row<SRC>(p, i0 + q, td, len);
      }
      srow[r] = sr;
    }
  }
  V val[kTileItems];
#pragma unroll
  for (int r = 0; r < kTileItems; ++r)
    if (srow[r] >= 0) val[r] = ld_stream(src + (rv == 1 ? srow[r] : srow[r] * rv + col[r]));
#pragma unroll
  for (int r = 0; r < kTileItems; ++r) {
    const int e = r * kTileThreads + tid;
    if (srow[r] >= 0) st_stream(dst + e, val[r]);
    else if (srow[r] == kPadRow) st_stream(dst + e, make_fill<V>(p.fill, (int64_t)col[r] * (int64_t)sizeof(V)));
  }
}

// C -> L / R with ONE-VECTOR rows (token ids, per-token scalars: the padded batch every model builds).  The general
// kernel above decodes every 8-byte element on its own (fast division, two shared-memory reads, validity test) and is
// issue-bound at 72 % issue-active.  Here a thread owns FOUR consecutive destination vectors: one division, one pair of
// shared-memory reads (two when the group straddles a row end), four loads, ONE wide store.
template <typename V>
__global__ void __launch_bounds__(kTileThreads)
row_map_padded_cat1_kernel(const RowMapParams p) {
  // A sequence of C is one contiguous run of len * rv vectors and lands in one contiguous run of its padded row, so
  // rows of several vectors are handled by SCALING: widths, lengths and offsets are counted in vectors.
  __shared__ int s_rel[kTileCap];            // (off[i0 + k] - off[i0]) * rv
  const int tid = threadIdx.x;
  const int rv = (int)p.row_vecs;
  const int64_t total = p.d.rows * rv;
  const int64_t e0 = (int64_t)blockIdx.x * kTileVecs;
  const int n_e = (int)(e0 + kTileVecs < total ? kTileVecs : total - e0);
  const uint32_t W = (uint32_t)(p.d.width * rv);   // vectors per padded row: 4 <= W <= 2^30 (checked by the launcher)
  const int64_t i0 = e0 / W;
  const int64_t i1 = (e0 + n_e - 1) / W;
  const uint32_t head = (uint32_t)(e0 - i0 * W);
  const int cnt = (int)(i1 - i0 + 2);
  const int64_t base0 = __ldg(p.rg.off + i0);
  for (int k = tid; k < cnt; k += kTileThreads) {
    const int64_t d = (__ldg(p.rg.off + i0 + k) - base0) * rv;
    s_rel[k] = d > (1 << 30) ? (1 << 30) : (int)d;
  }
  __syncthreads();
  const bool right_dst = p.d.layout == RUA_RIGHT;
  const V* __restrict__ src = reinterpret_cast<const V*>(p.src) + base0 * rv;
  V* __restrict__ dst = reinterpret_cast<V*>(p.dst) + e0;
  const V fill = make_fill<V>(p.fill, 0);    // the launcher checked that the fill pattern has period sizeof(V)
#pragma unroll
  for (int g = 0; g < kTileItems / 4; ++g) {
    const int eb = (g * kTileThreads + tid) * 4;          // tile-relative, 4 consecutive destination vectors
    if (eb >= n_e) break;
    const uint32_t x = head + (uint32_t)eb;               // < 2^31
    const uint32_t q = fast_div(x, p.div_wrv_m, p.div_wrv_s);
    const uint32_t rem = x - q * W;
    int sq = s_rel[q], len = s_rel[q + 1] - sq;
    int shift = right_dst ? (int)W - len : 0;
    V v[4];
    int from[4];                                          // source vector relative to base0 * rv, or -1 = padding
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int t = (int)rem + j;
      if (t >= (int)W && eb + j < n_e) {                  // the group straddles a row end (at most once: W >= 4)
        t -= (int)W;
        if (t == 0) {
          sq = s_rel[q + 1];
          len = s_rel[q + 2] - sq;
          shift = right_dst ? (int)W - len : 0;
        }
      }
      const int td = t - shift;
      from[j] = (td >= 0 && td < len && eb + j < n_e) ? sq + td : -1;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = from[j] >= 0 ? ld_stream(src + from[j]) : fill;
    if (eb + 4 <= n_e) {
      store4<V>(dst + eb, v[0], v[1], v[2], v[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (eb + j < n_e) st_stream(dst + eb + j, v[j]);
    }
  }
}

// P <-> {C, L, R} with narrow rows (< 128 bytes: token ids, scalars, small feature vectors).  P is time-major, the
// other layouts are sequence-major: moving such rows one by one leaves one side with a fraction of each DRAM page
// (8-byte rows: 8 useful bytes per 32-byte sector; 64-byte rows: random 64-byte reads).  This is a ragged TRANSPOSE
// instead: a CTA owns a tile of 32 ranks x TT time steps (TT = 32 / vectors-per-row), touches P along ranks (32
// consecutive rows of one time step are contiguous) and the other layout along time (TT consecutive tokens of one
// sequence are contiguous), and swaps the roles through a padded shared-memory tile.  Tiles that lie entirely
// beyond the ragged frontier (batch_sizes[t0] <= r0) exit at once.
constexpr int kTransposeTileVecs = 32 * 33;   // >= TT * (32 * rv + 1) for every rv in 1..7

template <typename V, bool kFromPack, int RV>       // RV = 1: one-vector rows at compile time; RV = 0: read it from p
__global__ void __launch_bounds__(256)
row_map_transpose_kernel(const RowMapParams p, const int TT_) {
  __shared__ V tile[kTransposeTileVecs];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rv = RV ? RV : (int)p.row_vecs;        // vectors per row, 1..7
  const int TT = RV == 1 ? 32 : TT_;
  const int stride = 32 * rv + 1;                  // shared-memory vectors per time step (+1: bank skew)
  const int64_t r0 = (int64_t)blockIdx.x * 32, t0 = (int64_t)blockIdx.y * TT;
  const rua_side_t& sq = kFromPack ? p.d : p.s;     // the sequence-major side
  const int64_t B = p.rg.B, Tp = p.rg.Tp, W = sq.width;
  const int64_t* __restrict__ poff = p.rg.poff;
  const int64_t* __restrict__ off = p.rg.off;
  const bool padded_dst = kFromPack && sq.layout != RUA_CAT;
  const int64_t bs0 = t0 < Tp ? __ldg(poff + t0 + 1) - __ldg(poff + t0) : 0;
  if (!padded_dst && bs0 <= r0) return;             // CTA-uniform: no token of this tile exists
  const V* __restrict__ src = reinterpret_cast<const V*>(p.src);
  V* __restrict__ dst = reinterpret_cast<V*>(p.dst);

  // Both phases are chains of dependent loads (poff[t] -> rows; sorted[r] -> off[i] -> rows).  A warp owns 4 time
  // steps / 4 ranks of the tile; lanes 0..3 fetch the metadata of all four AT ONCE and broadcast it, so the chain is
  // paid once per warp instead of once per row (this kernel is latency-bound: 94 % warps active, 36 % DRAM).
  auto pack_phase = [&](const bool load) {           // lanes run over (rank, vector): contiguous rows of P
    int64_t my_pt = 0, my_bst = 0;
    {
      const int64_t t = t0 + warp + 8 * lane;
      if (lane < 4 && warp + 8 * lane < TT && t < Tp) { my_pt = __ldg(poff + t); my_bst = __ldg(poff + t + 1) - my_pt; }
    }
    if constexpr (RV == 1) {   // one vector per rank: a single round, all four time steps' loads in flight together
      V val[4];
      bool on[4];
      int64_t at[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int64_t pt = shfl_i64(my_pt, k), bst = shfl_i64(my_bst, k);
        on[k] = t0 + warp + 8 * k < Tp && r0 + lane < bst;
        at[k] = pt + r0 + lane;
        if (load && on[k]) val[k] = ld_stream(src + at[k]);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (!on[k]) continue;
        if (load) tile[(warp + 8 * k) * stride + lane] = val[k];
        else st_stream(dst + at[k], tile[(warp + 8 * k) * stride + lane]);
      }
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int tt = warp + 8 * k;
        const int64_t pt = shfl_i64(my_pt, k), bst = shfl_i64(my_bst, k);
        const int64_t live = bst - r0 < 32 ? bst - r0 : 32;          // ranks of this tile alive at time t
        const int nvec = (tt < TT && t0 + tt < Tp && live > 0) ? (int)live * rv : 0;
        const int64_t base = (pt + r0) * rv;
        for (int q = lane; q < nvec; q += 32) {
          if (load) tile[tt * stride + q] = ld_stream(src + base + q);
          else st_stream(dst + base + q, tile[tt * stride + q]);
        }
      }
    }
  };
  // lanes run over (time, vector): TT consecutive tokens of one sequence are contiguous
  const int tt_l = rv == 1 ? lane : (int)fast_div((uint32_t)lane, p.div_rv_m, p.div_rv_s);
  const int c_l = lane - tt_l * rv;
  const bool lane_on = tt_l < TT;
  auto seq_phase = [&](const bool load) {
    int64_t my_i = 0, my_o = 0, my_len = 0;
    {
      const int64_t r = r0 + warp + 8 * lane;
      if (lane < 4 && r < B) {
        my_i = __ldg(p.rg.sorted + r);
        my_o = __ldg(off + my_i);
        my_len = __ldg(off + my_i + 1) - my_o;
        if (!kFromPack && sq.layout == RUA_CAT && my_o + my_len > sq.rows) my_len = sq.rows > my_o ? sq.rows - my_o : 0;   // see source_row
      }
    }
    const int64_t t = t0 + tt_l;
    V val[RV == 1 ? 4 : 1];
    if constexpr (RV == 1) {   // narrow vectors: the four ranks' row loads go out together (registers are cheap here)
      if (load) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int64_t i = shfl_i64(my_i, k), o = shfl_i64(my_o, k), len = shfl_i64(my_len, k);
          const int64_t row = sq.layout == RUA_CAT ? o + t : (sq.layout == RUA_LEFT ? i * W + t : i * W + (W - len) + t);
          if (r0 + warp + 8 * k < B && t < len) val[k] = ld_stream(src + row);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {                      // the metadata chain was paid once; one round trip per rank here
      const int64_t i = shfl_i64(my_i, k), o = shfl_i64(my_o, k), len = shfl_i64(my_len, k);
      if (r0 + warp + 8 * k >= B) break;               // warp-uniform
      if (!lane_on) continue;
      int64_t row;
      if (sq.layout == RUA_CAT) row = o + t;
      else if (sq.layout == RUA_LEFT) row = i * W + t;
      else row = i * W + (W - len) + t;
      V* cell = tile + tt_l * stride + (warp + 8 * k) * rv + c_l;
      if (load) {
        if (t < len) *cell = RV == 1 ? val[k] : ld_stream(src + row * rv + c_l);
      } else if (t < len) {
        st_stream(dst + row * rv + c_l, *cell);
      } else if (padded_dst && t < W) {              // left-aligned padding (R destinations do not come here)
        st_stream(dst + (i * W + t) * rv + c_l, make_fill<V>(p.fill, (int64_t)c_l * (int64_t)sizeof(V)));
      }
    }
  };
  if (kFromPack) {
    pack_phase(true);
    __syncthreads();
    seq_phase(false);
  } else {
    seq_phase(true);
    __syncthreads();
    pack_phase(false);
  }
}

// The same ragged transpose for ONE-VECTOR rows (token ids, per-token scalars: BASELINE config 5), restructured around
// what bounds it: latency.  ncu on the kernel above (8-byte rows): 94 % warps active, 36 % DRAM -- a CTA lives ~4 us for
// 8 KB in + 8 KB out because its loads form a chain (poff[t] -> rows of P; sorted[r] -> off[i] -> rows of C) and the
// second chain only started after the barrier.  Here (1) BOTH metadata chains are started at kernel entry, and (2) a CTA
// owns KT time-tiles of 32 steps for its 32 ranks and issues the row loads of all of them before the first shared-
// memory store, so the chain is paid once per KT * 8 KB and KT times as many bytes are in flight per thread.
// Round-2 record (profiles/r2_transpose.md): this form reaches 46-48 % (C -> P) / 40 % (P -> C) of the HBM peak on 8-byte rows.
// Two further restructurings were measured and dropped: a per-rank (offset, length) table that turns the chain into
// one coalesced load (no change), and PERSISTENT software-pipelined CTAs that keep the next tile's loads in flight while
// the current one is stored (40 % / 34 %: worse).  ncu shows why: the kernel moves 586 MB of DRAM traffic for 528 MB
// of payload (64-byte DRAM granules around 256-byte runs that start at arbitrary offsets) at 3.4 TB/s -- the runs
// belong to sequences in SORTED order, i.e. scattered over the whole C buffer.  benchmarks/transpose_locality.py then split
// the loss: the scattering costs 6 % (C -> P) / 19 % (P -> C), RAGGEDNESS the rest -- 68 % of the (rank, step) slots of the
// touched tiles hold a token at U[1,64], and constant lengths run at 4.75 TB/s; a compacted variant (lanes over the flattened
// populated slots) gained 10 % / 2 % on ragged batches and lost 22-31 % on uniform ones.  Dropped as well.
template <typename V, bool kFromPack, int KT>
__global__ void __launch_bounds__(256, KT == 1 ? 8 : (KT == 2 ? 5 : 4))
row_map_transpose1_kernel(const RowMapParams p) {
  __shared__ V tile[KT][32][33];                     // [time tile][time step][rank] (+1: bank skew)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t r0 = (int64_t)blockIdx.x * 32, t0 = (int64_t)blockIdx.y * (32 * KT);
  const rua_side_t& sq = kFromPack ? p.d : p.s;     // the sequence-major side
  const int64_t B = p.rg.B, Tp = p.rg.Tp, W = sq.width;
  const int64_t* __restrict__ poff = p.rg.poff;
  const int64_t* __restrict__ off = p.rg.off;
  const bool padded_dst = kFromPack && sq.layout != RUA_CAT;
  const V* __restrict__ src = reinterpret_cast<const V*>(p.src);
  V* __restrict__ dst = reinterpret_cast<V*>(p.dst);

  // ---- both metadata chains start now ---------------------------------------------------------------------------
  // pack side: this warp's time steps are tt = warp + 8 k of every time tile; lane (kt * 4 + k) fetches poff for it
  int64_t my_pt = 0, my_bst = 0;
  if (lane < 4 * KT) {
    const int64_t t = t0 + (lane >> 2) * 32 + warp + 8 * (lane & 3);
    if (t < Tp) { my_pt = __ldg(poff + t); my_bst = __ldg(poff + t + 1) - my_pt; }
  }
  // sequence side: this warp's ranks are r0 + warp + 8 k; lane k fetches sorted -> off for it
  int64_t my_i = 0, my_o = 0, my_len = 0;
  if (lane < 4) {
    const int64_t r = r0 + warp + 8 * lane;
    if (r < B) {
      my_i = __ldg(p.rg.sorted + r);
      my_o = __ldg(off + my_i);
      my_len = __ldg(off + my_i + 1) - my_o;
      if (!kFromPack && sq.layout == RUA_CAT && my_o + my_len > sq.rows) my_len = sq.rows > my_o ? sq.rows - my_o : 0;   // see source_row
    }
  }
  // no token of this CTA exists when the batch size at its first time step does not reach its first rank
  {
    const int64_t bs0 = t0 < Tp ? __ldg(poff + t0 + 1) - __ldg(poff + t0) : 0;
    if (!padded_dst && bs0 <= r0) return;           // CTA-uniform
  }
  auto seq_row = [&](int64_t i, int64_t o, int64_t len, int64_t t) -> int64_t {
    return sq.layout == RUA_CAT ? o + t : (sq.layout == RUA_LEFT ? i * W + t : i * W + (W - len) + t);
  };

  V val[KT][4];
  unsigned on = 0;                                   // bit kt * 4 + k: val[kt][k] holds a row
  if (kFromPack) {   // ---- P -> C / L: read P along ranks ----------------------------------------------------------
#pragma unroll
    for (int kt = 0; kt < KT; ++kt)
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int64_t pt = shfl_i64(my_pt, kt * 4 + k), bst = shfl_i64(my_bst, kt * 4 + k);
        if (r0 + lane < bst) {                       // bst == 0 beyond Tp
          on |= 1u << (kt * 4 + k);
          val[kt][k] = ld_stream(src + pt + r0 + lane);
        }
      }
#pragma unroll
    for (int kt = 0; kt < KT; ++kt)
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (on >> (kt * 4 + k) & 1u) tile[kt][warp + 8 * k][lane] = val[kt][k];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {                    // write the sequence-major side along time
      const int64_t i = shfl_i64(my_i, k), o = shfl_i64(my_o, k), len = shfl_i64(my_len, k);
      if (r0 + warp + 8 * k >= B) break;             // warp-uniform
#pragma unroll
      for (int kt = 0; kt < KT; ++kt) {
        const int64_t t = t0 + kt * 32 + lane;
        if (t < len) st_stream(dst + seq_row(i, o, len, t), tile[kt][lane][warp + 8 * k]);
        else if (padded_dst && t < W) st_stream(dst + i * W + t, make_fill<V>(p.fill, 0));   // left-aligned padding
      }
    }
  } else {           // ---- C / L / R -> P: read the sequence-major side along time ---------------------------------
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int64_t i = shfl_i64(my_i, k), o = shfl_i64(my_o, k), len = shfl_i64(my_len, k);
#pragma unroll
      for (int kt = 0; kt < KT; ++kt) {
        const int64_t t = t0 + kt * 32 + lane;
        if (r0 + warp + 8 * k < B && t < len) {
          on |= 1u << (kt * 4 + k);
          val[kt][k] = ld_stream(src + seq_row(i, o, len, t));
        }
      }
    }
#pragma unroll
    for (int kt = 0; kt < KT; ++kt)
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (on >> (kt * 4 + k) & 1u) tile[kt][lane][warp + 8 * k] = val[kt][k];
    __syncthreads();
#pragma unroll
    for (int kt = 0; kt < KT; ++kt)
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int64_t pt = shfl_i64(my_pt, kt * 4 + k), bst = shfl_i64(my_bst, kt * 4 + k);
        if (r0 + lane < bst) st_stream(dst + pt + r0 + lane, tile[kt][warp + 8 * k][lane]);
      }
  }
}

// can the ragged transpose serve this call?  (identity token map, untransformed lengths, narrow rows)
static bool transpose_applies(const RowMapParams& p, int64_t* grid_y, int* tt) {
  if (p.gather_index || p.scatter_index || p.row_vecs < 1 || p.row_vecs > 7) return false;
  if (p.tmap != RUA_MAP_SHIFT || p.tmap_arg != 0 || p.pad_mode != RUA_PAD_FILL) return false;
  if (p.s.len_xform != RUA_LEN_SAME || p.d.len_xform != RUA_LEN_SAME) return false;
  const bool from_pack = p.s.layout == RUA_PACK && p.d.layout != RUA_PACK;
  const bool to_pack = p.d.layout == RUA_PACK && p.s.layout != RUA_PACK;
  if (!from_pack && !to_pack) return false;
  if (from_pack && p.d.layout == RUA_RIGHT) return false;   // right-aligned padding is not tile-aligned
  int64_t t_extent = p.rg.Tp;
  if (from_pack && p.d.layout == RUA_LEFT && p.d.width > t_extent) t_extent = p.d.width;
  *tt = 32 / (int)p.row_vecs;
  *grid_y = ceil_div(t_extent, *tt);
  return *grid_y >= 1 && *grid_y <= 65535 && ceil_div(p.rg.B, 32) < (1ll << 31);
}

template <typename V>
static void launch_narrow(RowMapParams& p, int64_t rows, cudaStream_t st) {
  int64_t gy = 0;
  int tt = 32;
  if (transpose_applies(p, &gy, &tt)) {
    const FastDiv dv = FastDiv::make((uint64_t)p.row_vecs);
    p.div_rv_m = dv.m; p.div_rv_s = dv.s;
    dim3 grid((unsigned)ceil_div(p.rg.B, 32), (unsigned)gy);
    const bool from_pack = p.s.layout == RUA_PACK;
    if (p.row_vecs == 1) {
      // one-vector rows: KT time tiles of 32 steps per CTA, all of their row loads in flight together
      constexpr int kMaxKT = sizeof(V) >= 16 ? 2 : 4;   // 48 KB of static shared memory
      static const int64_t kt_env = knob("RUA_T1_KT", 0);
      int kt = gy <= 1 ? 1 : ((gy <= 2 || kMaxKT == 2) ? 2 : 4);
      if (sizeof(V) >= 16 && !from_pack) kt = 1;   // 16-byte rows into P: one tile per CTA measured 4.5 vs 4.1 TB/s (T = 512)
      if (kt_env > 0 && kt_env <= kMaxKT) kt = (int)kt_env;
      dim3 g1((unsigned)ceil_div(p.rg.B, 32), (unsigned)ceil_div(gy, kt));
      with_bool(from_pack, [&](auto fp) {
        constexpr bool FP = decltype(fp)::value;
        if (kt == 1) row_map_transpose1_kernel<V, FP, 1><<<g1, 256, 0, st>>>(p);
        else if (kt == 2) row_map_transpose1_kernel<V, FP, 2><<<g1, 256, 0, st>>>(p);
        else row_map_transpose1_kernel<V, FP, kMaxKT><<<g1, 256, 0, st>>>(p);
      });
    } else {
      with_bool(from_pack, [&](auto fp) { row_map_transpose_kernel<V, decltype(fp)::value, 0><<<grid, 256, 0, st>>>(p, tt); });
    }
    return;
  }
  const int64_t blocks = ceil_div(rows * p.row_vecs, kTileVecs);   // tiles of 2048 destination vectors
  const bool indexed = p.gather_index || p.scatter_index;
  const bool searched = !indexed && (p.d.layout == RUA_CAT || p.d.layout == RUA_PACK);
  // the 12 conversions (identity token map, untransformed lengths, plain fill) run source-specialised code
  const bool simple = !indexed && p.tmap == RUA_MAP_SHIFT && p.tmap_arg == 0 && p.pad_mode == RUA_PAD_FILL &&
                      p.s.len_xform == RUA_LEN_SAME && p.d.len_xform == RUA_LEN_SAME;
  const bool cat_select = !indexed && p.s.layout == RUA_CAT && p.d.layout == RUA_CAT && p.pad_mode == RUA_PAD_FILL &&
                          p.s.len_xform == RUA_LEN_SAME && p.d.len_xform == RUA_LEN_SAME &&
                          (p.tmap == RUA_MAP_REV || p.tmap == RUA_MAP_ROLL);
  const int srck = simple ? p.s.layout : (cat_select ? (p.tmap == RUA_MAP_REV ? kSrcCatRev : kSrcCatRoll) : kGenericSrc);
  const unsigned nb = (unsigned)blocks;
  if (searched) {
    // ... with many short sequences: a warp per 32 sequences (no per-tile decode chain)
    if (p.d.layout == RUA_CAT && p.row_vecs == 1 && ((uintptr_t)p.dst & (4 * sizeof(V) - 1)) == 0 &&
        warpseg_applies(rows, p.rg.B) && (srck == RUA_LEFT || srck == RUA_RIGHT || srck == kSrcCatRev || srck == kSrcCatRoll)) {
      const unsigned wb = (unsigned)ceil_div(p.rg.B, (int64_t)kWcWarps * 32);
      switch (srck) {
        case RUA_LEFT: row_map_warpseg_cat1_kernel<V, RUA_LEFT><<<wb, kWcThreads, 0, st>>>(p); break;
        case RUA_RIGHT: row_map_warpseg_cat1_kernel<V, RUA_RIGHT><<<wb, kWcThreads, 0, st>>>(p); break;
        case kSrcCatRev: row_map_warpseg_cat1_kernel<V, kSrcCatRev><<<wb, kWcThreads, 0, st>>>(p); break;
        default: row_map_warpseg_cat1_kernel<V, kSrcCatRoll><<<wb, kWcThreads, 0, st>>>(p); break;
      }
      return;
    }
    // one-vector rows into C from L / R, and C.rev / C.roll: four consecutive rows per thread, one wide store
    if (p.d.layout == RUA_CAT && ((uintptr_t)p.dst & (4 * sizeof(V) - 1)) == 0 &&
        (srck == RUA_LEFT || srck == RUA_RIGHT || (p.row_vecs == 1 && (srck == kSrcCatRev || srck == kSrcCatRoll)))) {
      switch (srck) {
        case RUA_LEFT: row_map_tile_cat1_kernel<V, RUA_LEFT><<<nb, kTileThreads, 0, st>>>(p); break;
        case RUA_RIGHT: row_map_tile_cat1_kernel<V, RUA_RIGHT><<<nb, kTileThreads, 0, st>>>(p); break;
        case kSrcCatRev: row_map_tile_cat1_kernel<V, kSrcCatRev><<<nb, kTileThreads, 0, st>>>(p); break;
        default: row_map_tile_cat1_kernel<V, kSrcCatRoll><<<nb, kTileThreads, 0, st>>>(p); break;
      }
      return;
    }
    switch (srck) {
      case RUA_CAT: row_map_tile_kernel<V, RUA_CAT><<<nb, kTileThreads, 0, st>>>(p); break;
      case RUA_LEFT: row_map_tile_kernel<V, RUA_LEFT><<<nb, kTileThreads, 0, st>>>(p); break;
      case RUA_RIGHT: row_map_tile_kernel<V, RUA_RIGHT><<<nb, kTileThreads, 0, st>>>(p); break;
      case RUA_PACK: row_map_tile_kernel<V, RUA_PACK><<<nb, kTileThreads, 0, st>>>(p); break;
      case kSrcCatRev: row_map_tile_kernel<V, kSrcCatRev><<<nb, kTileThreads, 0, st>>>(p); break;
      case kSrcCatRoll: row_map_tile_kernel<V, kSrcCatRoll><<<nb, kTileThreads, 0, st>>>(p); break;
      default: row_map_tile_kernel<V, kGenericSrc><<<nb, kTileThreads, 0, st>>>(p); break;
    }
  } else if (!indexed) {
    const int64_t wrv = p.d.width * p.row_vecs;
    const FastDiv a = FastDiv::make((uint64_t)(wrv > (1ll << 30) ? 1 : wrv)), b = FastDiv::make((uint64_t)p.row_vecs);
    p.div_wrv_m = a.m; p.div_wrv_s = a.s; p.div_rv_m = b.m; p.div_rv_s = b.s;
    // C into a padded batch (token ids, per-token scalars, small feature rows): four consecutive vectors per thread,
    // one wide store.  Needs a fill pattern that looks the same in every vector of a row.
    bool fill_periodic = true;
    {
      const unsigned char* fb = reinterpret_cast<const unsigned char*>(&p.fill);
      for (size_t k = sizeof(V); k < 16; ++k) fill_periodic &= fb[k] == fb[k % sizeof(V)];
    }
    if (srck == RUA_CAT && fill_periodic && wrv >= 4 && wrv <= (1ll << 30) &&
        ((uintptr_t)p.dst & (4 * sizeof(V) - 1)) == 0) {
      row_map_padded_cat1_kernel<V><<<nb, kTileThreads, 0, st>>>(p);
      return;
    }
    switch (srck) {
      case RUA_CAT: row_map_padded_kernel<V, RUA_CAT><<<nb, kTileThreads, 0, st>>>(p); break;
      case RUA_LEFT: row_map_padded_kernel<V, RUA_LEFT><<<nb, kTileThreads, 0, st>>>(p); break;
      case RUA_RIGHT: row_map_padded_kernel<V, RUA_RIGHT><<<nb, kTileThreads, 0, st>>>(p); break;
      case RUA_PACK: row_map_padded_kernel<V, RUA_PACK><<<nb, kTileThreads, 0, st>>>(p); break;
      default: row_map_padded_kernel<V, kGenericSrc><<<nb, kTileThreads, 0, st>>>(p); break;
    }
  } else {
    row_map_flat_kernel<V><<<nb, kTileThreads, 0, st>>>(p);
  }
}

// widest vector of at most `max_vec` bytes that divides every address and size OR-ed into `align`
static int vec_width(uintptr_t align, int max_vec) {
  int vec = max_vec;
  while (vec > 1 && (align & (uintptr_t)(vec - 1))) vec >>= 1;
  return vec;
}

// Launch plan of the wide-row kernels (row_map / list / multi): the vector width (up to max_vec bytes, 256-bit words only
// for rows of 128 bytes or more), lanes per row (short rows share a warp, 32 / lanes_per_row rows move concurrently),
// and rows per warp / column splits that keep ~32 warps per SM in flight when the problem allows it.  Fills those fields
// of p and returns the vector width in bytes; *blocks gets the number of kRowMapThreads-thread CTAs.
static int plan_wide(RowMapParams& p, uintptr_t align, int64_t row_bytes, int64_t rows, int max_vec, int64_t* blocks) {
  const int vec = vec_width(align, row_bytes >= 128 ? max_vec : 16);
  p.row_vecs = row_bytes / vec;
  int lpr = 1;
  while (lpr < 32 && lpr < p.row_vecs) lpr <<= 1;  // smallest power of two covering the row, <= 32
  p.lanes_per_row = lpr;
  const int64_t target_warps = (int64_t)kNumSMs * 32;
  int rpw = 32;
  while (rpw > 32 / lpr && rpw > 1 && ceil_div(rows, rpw) < target_warps) rpw >>= 1;
  p.rows_per_warp = rpw;
  const int64_t warps = ceil_div(rows, rpw);
  int splits = 1;
  while (warps * splits < target_warps && p.row_vecs / (splits * 2) >= 32 * kUnroll && splits < 64) splits *= 2;
  p.col_splits = splits;
  *blocks = ceil_div(warps, kRowMapThreads / 32);
  return vec;
}

static int launch_row_map(RowMapParams& p, int64_t row_bytes, int64_t rows, cudaStream_t st) {
  if (rows <= 0 || row_bytes <= 0) return RUA_OK;
  // the vector must divide the row size and both base addresses
  const uintptr_t a = (uintptr_t)p.src | (uintptr_t)p.dst | (uintptr_t)row_bytes;

  // C <-> L/R conversions of 128..255-byte rows also take the narrow path: its four-vectors-per-thread kernels treat a
  // sequence as one contiguous run of vectors and beat the row-per-lane-group kernel there (128-byte rows: L -> C
  // 76 % -> 88 % of peak); they need 16-byte vectors and a 64-byte aligned destination
  const bool simple_map = !p.gather_index && !p.scatter_index && p.tmap == RUA_MAP_SHIFT && p.tmap_arg == 0 &&
                          p.pad_mode == RUA_PAD_FILL && p.s.len_xform == RUA_LEN_SAME && p.d.len_xform == RUA_LEN_SAME;
  const bool padded_side = (p.s.layout == RUA_CAT && (p.d.layout == RUA_LEFT || p.d.layout == RUA_RIGHT)) ||
                           (p.d.layout == RUA_CAT && (p.s.layout == RUA_LEFT || p.s.layout == RUA_RIGHT));
  const bool run_copy = simple_map && padded_side && row_bytes < 512 && (a & 15u) == 0 && ((uintptr_t)p.dst & 63u) == 0 &&
                        !p.mask_out;   // the fused mask lives in the wide-row kernel
  if (row_bytes < 128 || run_copy) {  // narrow rows: tile kernels (segment offsets staged in shared memory)
    if (p.mask_out) return RUA_ERR_UNSUPPORTED;   // callers launch rua_mask separately for narrow rows
    const int vec = vec_width(a, 16);
    p.row_vecs = row_bytes / vec;
    if (ceil_div(rows * p.row_vecs, kTileVecs) >= (1ll << 31)) return RUA_ERR_UNSUPPORTED;
    with_word(vec, [&](auto w) {
      using W = typename decltype(w)::type;
      if constexpr (sizeof(W) <= 16) launch_narrow<W>(p, rows, st);   // 256-bit words only in the wide-row kernel
    });
    return check_launch();
  }

  static const bool use256 = knob("RUA_VEC256", 1) != 0;
  int64_t blocks;
  const int vec = plan_wide(p, a, row_bytes, rows, use256 ? 32 : 16, &blocks);
  if (blocks >= (1ll << 31)) return RUA_ERR_UNSUPPORTED;
  const dim3 grid((unsigned)blocks, (unsigned)p.col_splits);
  with_word(vec, [&](auto w) { row_map_kernel<typename decltype(w)::type><<<grid, kRowMapThreads, 0, st>>>(p); });
  return check_launch();
}

static int launch_row_map_list(RowMapParams& p, const uint8_t* const* src_list, int src_align, int64_t row_bytes,
                               int64_t rows, cudaStream_t st, const int64_t* bases = nullptr, int n_src = 0) {
  if (rows <= 0 || row_bytes <= 0) return RUA_OK;
  int64_t blocks;
  const int vec = plan_wide(p, (uintptr_t)p.dst | (uintptr_t)row_bytes | (uintptr_t)src_align, row_bytes, rows, 32, &blocks);
  if (blocks >= (1ll << 31)) return RUA_ERR_UNSUPPORTED;
  const dim3 grid((unsigned)blocks, (unsigned)p.col_splits);
  with_word(vec, [&](auto w) {
    row_map_list_kernel<typename decltype(w)::type><<<grid, kRowMapThreads, 0, st>>>(p, src_list, row_bytes, bases, n_src);
  });
  return check_launch();
}

static int launch_row_map_multi(RowMapParams& p, const MultiDst& m, int64_t row_bytes, int64_t rows, cudaStream_t st) {
  if (rows <= 0 || row_bytes <= 0) return RUA_OK;
  uintptr_t a = (uintptr_t)p.src | (uintptr_t)row_bytes;
  for (int k = 0; k < m.n; ++k) a |= (uintptr_t)m.dst[k];
  // (a TMA bulk-copy variant of this kernel -- one cp.async.bulk per row and destination -- measured 25.6-26.3 ms vs 25.3 ms
  //  at 8 GPUs: the wire, not the store shape, bounds it; profiles/r2_gather_sweep.md)
  int64_t blocks;
  const int vec = plan_wide(p, a, row_bytes, rows, 32, &blocks);
  // wire-bound (>= 4 destinations, i.e. >= 2 peers beside the local window and copy): cap the grid so that other streams'
  // kernels find free CTA slots on every SM; RUA_MULTI_CTAS_PER_SM overrides (0 = no cap)
  static const int64_t cap_per_sm = knob("RUA_MULTI_CTAS_PER_SM", 4);
  if (m.n >= 4 && cap_per_sm > 0 && blocks > (int64_t)kNumSMs * cap_per_sm) blocks = (int64_t)kNumSMs * cap_per_sm;
  if (blocks >= (1ll << 31)) return RUA_ERR_UNSUPPORTED;
  const dim3 grid((unsigned)blocks, (unsigned)p.col_splits);
  with_word(vec, [&](auto w) { row_map_multi_kernel<typename decltype(w)::type><<<grid, kRowMapThreads, 0, st>>>(p, m); });
  return check_launch();
}

static bool valid_side(const rua_side_t* s) {
  if (!s) return false;
  if (s->layout < RUA_CAT || s->layout > RUA_RIGHT) return false;
  if (s->len_xform < RUA_LEN_SAME || s->len_xform > RUA_LEN_MINUS) return false;
  if ((s->layout == RUA_LEFT || s->layout == RUA_RIGHT) && s->width <= 0 && s->rows > 0) return false;
  return s->rows >= 0;
}

// the padding value: fill_bytes = 0 (zeros), or a pattern of 1, 2, 4, 8 or 16 bytes at fill_host that divides the row,
// replicated over 16 bytes into p.fill
static int set_fill(RowMapParams& p, const void* fill_host, int32_t fill_bytes, int64_t row_bytes) {
  if (fill_bytes != 0 && fill_bytes != 1 && fill_bytes != 2 && fill_bytes != 4 && fill_bytes != 8 && fill_bytes != 16)
    return RUA_ERR_INVALID;
  if (fill_bytes > 0 && (!fill_host || row_bytes % fill_bytes != 0)) return RUA_ERR_INVALID;
  uint8_t pat[16] = {0};
  for (int k = 0; fill_bytes > 0 && k < 16; ++k) pat[k] = ((const uint8_t*)fill_host)[k % fill_bytes];
  memcpy(&p.fill, pat, sizeof(pat));
  return RUA_OK;
}

}  // namespace rua

using namespace rua;

extern "C" {

int rua_row_map(const void* src, void* dst, int64_t row_bytes, const rua_ragged_t* ragged,
                const rua_side_t* src_side, const rua_side_t* dst_side, int32_t tmap, int64_t tmap_arg,
                int32_t pad_mode, const void* fill_host, int32_t fill_bytes, rua_stream_t stream) {
  if (!ragged || !valid_side(src_side) || !valid_side(dst_side) || row_bytes < 0) return RUA_ERR_INVALID;
  if (dst_side->rows == 0 || row_bytes == 0) return RUA_OK;
  if (!dst || !ragged->off || ragged->B <= 0) return RUA_ERR_INVALID;
  if (tmap < RUA_MAP_SHIFT || tmap > RUA_MAP_ROLL) return RUA_ERR_INVALID;
  if (pad_mode < RUA_PAD_FILL || pad_mode > RUA_PAD_WRAP) return RUA_ERR_INVALID;
  bool uses_pack = src_side->layout == RUA_PACK || dst_side->layout == RUA_PACK;
  if (uses_pack && (!ragged->poff || !ragged->sorted || !ragged->unsorted)) return RUA_ERR_INVALID;
  if (!src && src_side->rows > 0) return RUA_ERR_INVALID;
  RowMapParams p{};
  if (int rc = set_fill(p, fill_host, fill_bytes, row_bytes)) return rc;
  p.src = (const uint8_t*)src;
  p.dst = (uint8_t*)dst;
  p.rg = *ragged;
  p.s = *src_side;
  p.d = *dst_side;
  p.tmap = tmap;
  p.tmap_arg = tmap_arg;
  p.pad_mode = pad_mode;
  p.gather_index = nullptr;
  p.scatter_index = nullptr;
  return launch_row_map(p, row_bytes, dst_side->rows, (cudaStream_t)stream);
}

int rua_row_map_mask(const void* src, void* dst, int64_t row_bytes, const rua_ragged_t* ragged,
                     const rua_side_t* src_side, const rua_side_t* dst_side, const void* fill_host, int32_t fill_bytes,
                     const void* zero_host, const void* one_host, int32_t mask_elem_bytes, void* mask_out,
                     rua_stream_t stream) {
  if (!ragged || !valid_side(src_side) || !valid_side(dst_side) || row_bytes < 0) return RUA_ERR_INVALID;
  if (dst_side->layout != RUA_LEFT || dst_side->len_xform != RUA_LEN_SAME || src_side->len_xform != RUA_LEN_SAME) return RUA_ERR_INVALID;
  if (mask_elem_bytes != 1 && mask_elem_bytes != 2 && mask_elem_bytes != 4 && mask_elem_bytes != 8) return RUA_ERR_INVALID;
  if (dst_side->rows == 0) return RUA_OK;
  if (!dst || !mask_out || !zero_host || !one_host || !ragged->off || ragged->B <= 0) return RUA_ERR_INVALID;
  if (row_bytes < 128) return RUA_ERR_UNSUPPORTED;
  bool uses_pack = src_side->layout == RUA_PACK;
  if (uses_pack && (!ragged->poff || !ragged->sorted || !ragged->unsorted)) return RUA_ERR_INVALID;
  if (!src && src_side->rows > 0) return RUA_ERR_INVALID;
  RowMapParams p{};
  if (int rc = set_fill(p, fill_host, fill_bytes, row_bytes)) return rc;
  p.src = (const uint8_t*)src;
  p.dst = (uint8_t*)dst;
  p.rg = *ragged;
  p.s = *src_side;
  p.d = *dst_side;
  p.tmap = RUA_MAP_SHIFT;
  p.pad_mode = RUA_PAD_FILL;
  p.mask_out = mask_out;
  p.mask_elem = mask_elem_bytes;
  memcpy(&p.mask_zero, zero_host, mask_elem_bytes);
  memcpy(&p.mask_one, one_host, mask_elem_bytes);
  return launch_row_map(p, row_bytes, dst_side->rows, (cudaStream_t)stream);
}

static int index_rows(const void* src, const int64_t* gidx, const int64_t* sidx, int64_t n, int64_t indexed_rows,
                      int64_t row_bytes, void* dst, rua_stream_t stream) {
  if (n < 0 || row_bytes < 0 || indexed_rows < 0) return RUA_ERR_INVALID;
  if (n == 0 || row_bytes == 0) return RUA_OK;
  if (!src || !dst || (!gidx && !sidx)) return RUA_ERR_INVALID;
  RowMapParams p{};
  p.src = (const uint8_t*)src;
  p.dst = (uint8_t*)dst;
  p.d.rows = n;
  p.s.rows = indexed_rows;  // size of the indexed side, for negative-index wrap-around
  p.gather_index = gidx;
  p.scatter_index = sidx;
  p.index_errors = index_error_counter();
  p.pad_mode = RUA_PAD_FILL;
  return launch_row_map(p, row_bytes, n, (cudaStream_t)stream);
}

int rua_gather_rows(const void* src, int64_t src_rows, const int64_t* index, int64_t n, int64_t row_bytes,
                    void* dst, rua_stream_t stream) {
  return index_rows(src, index, nullptr, n, src_rows, row_bytes, dst, stream);
}

int rua_scatter_rows(const void* src, const int64_t* index, int64_t n, int64_t row_bytes, void* dst,
                     int64_t dst_rows, rua_stream_t stream) {
  return index_rows(src, nullptr, index, n, dst_rows, row_bytes, dst, stream);
}

int rua_row_map_multi(const void* src, int64_t row_bytes, const rua_ragged_t* ragged, const rua_side_t* src_side,
                      int64_t n_tokens, void* const* dst_host, const int64_t* const* dst_base_host, int32_t n_dst,
                      rua_stream_t stream) {
  if (!ragged || !valid_side(src_side) || row_bytes < 0 || n_tokens < 0) return RUA_ERR_INVALID;
  if (n_dst < 0 || n_dst > kMaxDst) return RUA_ERR_INVALID;
  if (n_tokens == 0 || row_bytes == 0 || n_dst == 0) return RUA_OK;
  if (!src || !dst_host || !dst_base_host || !ragged->off || ragged->B <= 0) return RUA_ERR_INVALID;
  if (src_side->len_xform != RUA_LEN_SAME) return RUA_ERR_INVALID;
  if (src_side->layout == RUA_PACK && (!ragged->poff || !ragged->unsorted)) return RUA_ERR_INVALID;
  RowMapParams p{};
  p.src = (const uint8_t*)src;
  p.rg = *ragged;
  p.s = *src_side;
  p.d.layout = RUA_CAT;
  p.d.len_xform = RUA_LEN_SAME;
  p.d.rows = n_tokens;
  p.tmap = RUA_MAP_SHIFT;
  p.pad_mode = RUA_PAD_FILL;
  MultiDst m{};
  m.n = n_dst;
  for (int k = 0; k < n_dst; ++k) {
    if (!dst_host[k]) return RUA_ERR_INVALID;
    m.dst[k] = (uint8_t*)dst_host[k];
    m.base[k] = dst_base_host[k];
  }
  return launch_row_map_multi(p, m, row_bytes, n_tokens, (cudaStream_t)stream);
}

int rua_scatter_rows_multi(const void* src, const int64_t* index, int64_t n, int64_t row_bytes,
                           void* const* dst_host, int32_t n_dst, rua_stream_t stream) {
  if (n < 0 || row_bytes < 0 || n_dst < 0 || n_dst > kMaxDst) return RUA_ERR_INVALID;
  if (n == 0 || row_bytes == 0 || n_dst == 0) return RUA_OK;
  if (!src || !index || !dst_host) return RUA_ERR_INVALID;
  RowMapParams p{};
  p.src = (const uint8_t*)src;
  p.d.rows = n;
  MultiDst m{};
  m.n = n_dst;
  m.rows_are_sequences = 1;
  for (int k = 0; k < n_dst; ++k) {
    if (!dst_host[k]) return RUA_ERR_INVALID;
    m.dst[k] = (uint8_t*)dst_host[k];
    m.base[k] = index;
  }
  return launch_row_map_multi(p, m, row_bytes, n, (cudaStream_t)stream);
}

int rua_row_map_list(const void* const* src_list, int32_t src_align, void* dst, int64_t row_bytes,
                     const rua_ragged_t* ragged, const rua_side_t* dst_side, const void* fill_host, int32_t fill_bytes,
                     rua_stream_t stream) {
  if (!ragged || !valid_side(dst_side) || row_bytes < 0) return RUA_ERR_INVALID;
  if (dst_side->rows == 0 || row_bytes == 0) return RUA_OK;
  if (!src_list || !dst || !ragged->off || ragged->B <= 0) return RUA_ERR_INVALID;
  if (src_align < 1 || (src_align & (src_align - 1))) return RUA_ERR_INVALID;
  if (dst_side->len_xform != RUA_LEN_SAME) return RUA_ERR_INVALID;
  if (dst_side->layout == RUA_PACK && (!ragged->poff || !ragged->sorted)) return RUA_ERR_INVALID;
  RowMapParams p{};
  if (int rc = set_fill(p, fill_host, fill_bytes, row_bytes)) return rc;
  p.dst = (uint8_t*)dst;
  p.rg = *ragged;
  p.d = *dst_side;
  p.s.layout = RUA_CAT;
  return launch_row_map_list(p, (const uint8_t* const*)src_list, src_align, row_bytes, dst_side->rows, (cudaStream_t)stream);
}

int rua_gather_rows_multi(const void* const* src_list, const int64_t* bases, int32_t n_src, int32_t src_align,
                          const int64_t* index, int64_t n, int64_t row_bytes, void* dst, rua_stream_t stream) {
  if (n < 0 || row_bytes < 0 || n_src < 0) return RUA_ERR_INVALID;
  if (n == 0 || row_bytes == 0) return RUA_OK;
  if (!src_list || !bases || !index || !dst || n_src == 0) return RUA_ERR_INVALID;
  if (src_align < 1 || (src_align & (src_align - 1))) return RUA_ERR_INVALID;
  RowMapParams p{};
  p.dst = (uint8_t*)dst;
  p.d.rows = n;
  p.gather_index = index;
  p.index_errors = index_error_counter();
  return launch_row_map_list(p, (const uint8_t* const*)src_list, src_align, row_bytes, n, (cudaStream_t)stream, bases, n_src);
}

/* host-only self test of the launch-time arithmetic (no GPU needed; run by the CPU test-suite): the magic-number
 * division the narrow-row kernels use must be exact for every x < 2^31.  Returns 0, or the failing divisor negated. */
int rua_selftest(void) {
  unsigned long long state = 0x9e3779b97f4a7c15ull;
  auto next = [&state]() { state ^= state << 13; state ^= state >> 7; state ^= state << 17; return state; };
  auto check = [](uint64_t d) -> bool {
    const FastDiv f = FastDiv::make(d);
    const uint64_t xs[] = {0, 1, d - 1, d, d + 1, 2 * d - 1, 2 * d, 3 * d + 1, (1ull << 31) - 1, (1ull << 31) - d,
                           (1ull << 30), (1ull << 30) + d - 1, ((1ull << 31) - 1) / d * d, ((1ull << 31) - 1) / d * d - 1};
    for (uint64_t x : xs) {
      if (x >= (1ull << 31)) continue;
      if ((uint32_t)((x * f.m) >> f.s) != (uint32_t)(x / d)) return false;
    }
    return true;
  };
  for (uint64_t d = 1; d <= 70000; ++d)
    if (!check(d)) return -(int)d;
  for (int b = 1; b <= 30; ++b)
    for (int64_t delta = -2; delta <= 2; ++delta) {
      const int64_t d = (1ll << b) + delta;
      if (d >= 1 && d <= (1ll << 30) && !check((uint64_t)d)) return -(int)d;
    }
  for (int k = 0; k < 200000; ++k) {
    const uint64_t d = 1 + next() % (1ull << 30);
    const FastDiv f = FastDiv::make(d);
    for (int j = 0; j < 8; ++j) {
      const uint64_t x = next() % (1ull << 31);
      if ((uint32_t)((x * f.m) >> f.s) != (uint32_t)(x / d)) return -(int)d;
    }
  }
  return 0;
}

}  // extern "C"
