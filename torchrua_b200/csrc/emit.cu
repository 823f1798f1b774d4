// K3 -- mask / index emit: write-only kernels, no payload reads.
//
// Replaces (reference file:line): mask / bmask / fmask torchrua/mask.py:6-32, get_mask
// core/view.py:11-18, major_sizes_to_ptr utils.py:7-13, C/L/R.ptr layout/cat.py:68-71,
// P.ptr layout/pack.py:23-27, L.idx layout/left.py:73-77, R.idx layout/right.py:74-79.
//
// The reference builds these from repeat_interleave (each an internal cumsum + a .item() sync),
// arange, new_full and index_put_.  Here every output element is a closed form of (segment, within)
// and is stored once with 16-byte coalesced stores.  HBM-write bound.
#include "common.cuh"
#include "dispatch.cuh"
#include "tile_decode.cuh"

namespace rua {

// ------------------------------------------------------------------------------------------------
// mask: out[i, t] = t < len[i] ? one : zero          (left aligned for all layouts, mask.py:10)
// Each thread produces 32 bytes = 32/E consecutive elements of the flattened (B, W) output and stores them
// with one 256-bit store.  When the span lies inside one row (the common case: W is a multiple of the span or
// simply long) the 32 bytes are built word-wise from the count of leading `one`s -- a handful of instructions
// per 8 bytes instead of a compare / select / row-wrap check per element (bool masks: 32 elements per thread).
// ------------------------------------------------------------------------------------------------
template <typename E> __device__ __forceinline__ unsigned long long replicate64(E v) {
  unsigned long long x = (unsigned long long)v;
  if (sizeof(E) < 2) x |= x << 8;
  if (sizeof(E) < 4) x |= x << 16;
  if (sizeof(E) < 8) x |= x << 32;
  return x;
}

constexpr int kMaskIters = 4;   // 32-byte spans per thread (a CTA writes 32 KB: fewer, fatter CTAs than one span per thread)

template <typename E>
__global__ void __launch_bounds__(256)
mask_kernel(const int64_t* __restrict__ len, int64_t B, int64_t W, E zero, E one, E* __restrict__ out, int wide) {
  constexpr int K = 32 / sizeof(E);      // elements per span
  constexpr int EPW = 8 / sizeof(E);     // elements per 64-bit word
  const int64_t total = B * W;
  const unsigned long long ow = replicate64<E>(one), zw = replicate64<E>(zero);
  // all length loads first: the stores below are asm volatile and would serialise load -> store -> load
  int64_t gs[kMaskIters], is[kMaskIters], ts[kMaskIters], ls[kMaskIters];
#pragma unroll
  for (int it = 0; it < kMaskIters; ++it) {
    const int64_t g0 = (((int64_t)blockIdx.x * kMaskIters + it) * blockDim.x + threadIdx.x) * K;
    gs[it] = g0;
    int64_t i = 0, t = 0;
    if (g0 < total) {
      if (total < (1ll << 31)) {
        uint32_t q = (uint32_t)g0 / (uint32_t)W;
        i = q;
        t = (uint32_t)g0 - q * (uint32_t)W;
      } else {
        i = g0 / W;
        t = g0 - i * W;
      }
    }
    is[it] = i;
    ts[it] = t;
    ls[it] = g0 < total ? __ldg(len + i) : 0;
  }
#pragma unroll
  for (int it = 0; it < kMaskIters; ++it) {
    const int64_t g0 = gs[it];
    if (g0 >= total) return;
    int64_t i = is[it], t = ts[it], li = ls[it];
    unsigned long long w0 = 0, w1 = 0, w2 = 0, w3 = 0;   // the 32 output bytes, in registers (no local-memory union)
    if (t + K <= W) {
      const int64_t rest = li - t;
      const int ones = rest <= 0 ? 0 : (rest >= K ? K : (int)rest);   // leading `one`s of this span
      auto word = [&](int w) -> unsigned long long {
        const int n1 = ones - w * EPW;
        const unsigned long long m = n1 >= EPW ? ~0ull : (n1 <= 0 ? 0ull : ((1ull << (n1 * 8 * (int)sizeof(E) & 63)) - 1ull));
        return (ow & m) | (zw & ~m);
      };
      w0 = word(0); w1 = word(1); w2 = word(2); w3 = word(3);
    } else {                                              // the span crosses a row end: element by element
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const unsigned long long e = (unsigned long long)(t < li ? one : zero) << ((k % EPW) * 8 * (int)sizeof(E) & 63);
        if (k / EPW == 0) w0 |= e; else if (k / EPW == 1) w1 |= e; else if (k / EPW == 2) w2 |= e; else w3 |= e;
        if (++t == W) {
          t = 0;
          ++i;
          li = i < B ? __ldg(len + i) : 0;
        }
      }
    }
    if (g0 + K <= total) {
      if (wide) {
        asm volatile("st.global.cs.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(out + g0), "l"(w0), "l"(w1), "l"(w2), "l"(w3) : "memory");
      } else {
        __stcs(reinterpret_cast<ulonglong2*>(out + g0), make_ulonglong2(w0, w1));
        __stcs(reinterpret_cast<ulonglong2*>(out + g0) + 1, make_ulonglong2(w2, w3));
      }
    } else {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const unsigned long long w = k / EPW == 0 ? w0 : (k / EPW == 1 ? w1 : (k / EPW == 2 ? w2 : w3));
        if (g0 + k < total) out[g0 + k] = (E)(w >> ((k % EPW) * 8 * (int)sizeof(E) & 63));
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// ptr / idx emit over a segmented range.  A CTA owns a tile of kDecTile consecutive positions and decodes
// it once (tile_decode.cuh: staged segment starts + a block scan of start counters), after which every
// position resolves its segment with two shared-memory reads.  A thread emits 4 consecutive positions =
// one 256-bit store per output (sm_100: STG.E.ENL2.256, a full 32-byte sector per lane).
// ------------------------------------------------------------------------------------------------
constexpr int kEmitThreads = kDecThreads;
constexpr int kEmitGroup = 4;
constexpr int kEmitRounds = kDecTile / (kEmitThreads * kEmitGroup);  // 2
constexpr int kEmitTile = kDecTile;

__device__ __forceinline__ void st_v4_i64(int64_t* p, const int64_t* v) {
  asm volatile("st.global.cs.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(p), "l"(v[0]), "l"(v[1]), "l"(v[2]), "l"(v[3]) : "memory");
}

__global__ void __launch_bounds__(kEmitThreads)
emit_ptr_kernel(const int64_t* __restrict__ off, int64_t S, int64_t n, const int64_t* __restrict__ relabel,
                int64_t* __restrict__ which, int64_t* __restrict__ within, int64_t* __restrict__ flat,
                int64_t stride, int right_align, int wide_stores) {
  __shared__ TileDecodeSmem sm;
  const int tid = threadIdx.x;
  const int64_t j0 = (int64_t)blockIdx.x * kEmitTile;
  const int nj = (int)(j0 + kEmitTile < n ? kEmitTile : n - j0);
  GlobalOff g{off};
  const TileDecode d = tile_decode(g, S, j0, nj, sm);

#pragma unroll
  for (int r = 0; r < kEmitRounds; ++r) {
    const int jb = (r * kEmitThreads + tid) * kEmitGroup;  // tile-relative, 4 consecutive positions
    if (jb >= nj) break;
    int64_t sv[kEmitGroup], wv[kEmitGroup], fv[kEmitGroup];
    if (d.staged) {
      const int4 k4 = reinterpret_cast<const int4*>(sm.seg)[jb >> 2];
      const int kk[kEmitGroup] = {k4.x, k4.y, k4.z, k4.w};
      int k_prev = -1, rel = 0;
      int64_t shift = 0;   // flat = which * stride + within + shift
#pragma unroll
      for (int e = 0; e < kEmitGroup; ++e) {
        const int k = kk[e];
        if (k != k_prev) {                  // a group rarely crosses a boundary: one lookup for all four
          k_prev = k;
          rel = sm.rel[k];
          if (flat) {
            const int nxt = sm.rel[k + 1];
            const int64_t len = (k > 0 && nxt <= kEmitTile) ? (int64_t)(nxt - rel)
                                                            : __ldg(off + d.first + k + 1) - __ldg(off + d.first + k);
            shift = right_align ? stride - len : 0;
          }
        }
        sv[e] = d.first + k;
        wv[e] = k == 0 ? (j0 + jb + e) - d.off_first : (int64_t)(jb + e - rel);
        fv[e] = sv[e] * stride + wv[e] + shift;
      }
    } else {
#pragma unroll
      for (int k = 0; k < kEmitGroup; ++k) {
        const int64_t j = j0 + jb + k;
        const int64_t jj = j < n ? j : n - 1;
        const int64_t s = owner_search(g, S, jj);
        const int64_t base = __ldg(off + s);
        sv[k] = s;
        wv[k] = jj - base;
        fv[k] = s * stride + wv[k] + (right_align ? stride - (__ldg(off + s + 1) - base) : 0);
      }
    }
    if (relabel) {
#pragma unroll
      for (int k = 0; k < kEmitGroup; ++k)
        if (jb + k < nj) wv[k] = __ldg(relabel + wv[k]);
    }
    const int64_t j = j0 + jb;
    if (wide_stores && jb + kEmitGroup <= nj) {
      if (which) st_v4_i64(which + j, sv);
      if (within) st_v4_i64(within + j, wv);
      if (flat) st_v4_i64(flat + j, fv);
    } else {
      for (int k = 0; k < kEmitGroup && jb + k < nj; ++k) {
        if (which) which[j + k] = sv[k];
        if (within) within[j + k] = wv[k];
        if (flat) flat[j + k] = fv[k];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// ptr / idx emit with MANY SHORT segments (C.ptr / L.idx / R.idx / major_sizes_to_ptr at BASELINE config 5: 1 M
// sequences of 1..64 tokens).  The tile kernel above pays a serial chain per CTA (two searches -> staged offsets ->
// block scan -> emit, three barriers; ncu: 6 of 8 warps idle at the first barrier, 45 % DRAM).  Here a WARP owns 32
// consecutive segments, i.e. one contiguous range of output positions:
//   * lane i reads off[s0 + i], off[s0 + i + 1] (coalesced; no search, no block barrier);
//   * every lane paints ITS OWN lane number over its segment's positions in a 2 KB byte window of shared memory (all
//     lanes busy; a window lying inside one long segment is not painted at all);
//   * the warp then walks the window four positions per lane: one LDS.32 yields the four owners, shuffles fetch the
//     owners' segment starts, and each output array gets one 256-bit store per lane (a full sector).
// ------------------------------------------------------------------------------------------------
constexpr int kEwThreads = 256;
constexpr int kEwWarps = kEwThreads / 32;
constexpr int kEwWin = 2048;   // positions per window

__global__ void __launch_bounds__(kEwThreads)
emit_ptr_warpseg_kernel(const int64_t* __restrict__ off, int64_t S, int64_t n, int64_t* __restrict__ which,
                        int64_t* __restrict__ within, int64_t* __restrict__ flat, int64_t stride, int right_align,
                        int wide_stores) {
  __shared__ __align__(16) unsigned char s_own[kEwWarps][kEwWin];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t s0 = ((int64_t)blockIdx.x * kEwWarps + warp) * 32;
  if (s0 >= S) return;                                   // warp-uniform; no block-level synchronisation below
  const int64_t s = s0 + lane;
  int64_t beg = s < S ? __ldg(off + s) : n, end = s < S ? __ldg(off + s + 1) : n;
  const int64_t shift = right_align ? stride - (end - beg) : 0;   // R.idx: tokens sit at the end of their padded row
  beg = beg < n ? beg : n;
  end = end < n ? end : n;
  const int64_t wbeg = shfl_i64(beg, 0), wend = shfl_i64(end, 31);
  unsigned char* own = s_own[warp];
  // segment starts relative to the warp's first position fit 32 bits unless the warp spans >= 2^30 positions
  const bool small = wend - wbeg < (1ll << 30);
  const int rel_beg = small ? (int)(beg - wbeg) : 0;
  // flat[p] = which * stride + within + shift = (p - wbeg) + flat_c[owner]: one 64-bit shuffle + one add per position
  const int64_t flat_c = flat ? s * stride + shift - (beg - wbeg) : 0;
  for (int64_t w0 = wbeg & ~(int64_t)3; w0 < wend; w0 += kEwWin) {
    const int64_t w1 = w0 + kEwWin < wend ? w0 + kEwWin : wend;
    const unsigned who = __ballot_sync(kFullMask, beg <= w0 && end >= w0 + kEwWin);
    if (!who) {
      const int64_t lo64 = beg < w0 ? w0 : (beg > w1 ? w1 : beg), hi64 = end < w0 ? w0 : (end > w1 ? w1 : end);
      int p = (int)(lo64 - w0);
      const int hi = (int)(hi64 - w0);
      for (; p < hi && (p & 3); ++p) own[p] = (unsigned char)lane;          // head bytes up to a word boundary
      const unsigned word = (unsigned)lane * 0x01010101u;
      for (; p + 4 <= hi; p += 4) *reinterpret_cast<unsigned*>(own + p) = word;   // four positions per store
      for (; p < hi; ++p) own[p] = (unsigned char)lane;
    }
    __syncwarp();
    const int groups = (int)((w1 - w0 + 3) >> 2);        // groups of 4 positions in this window (warp-uniform)
    for (int g0 = 0; g0 < groups; g0 += 32) {
      const int g = g0 + lane;
      int o[4];
      if (who) {
        o[0] = o[1] = o[2] = o[3] = __ffs(who) - 1;
      } else {
        const uchar4 b = reinterpret_cast<const uchar4*>(own)[g < groups ? g : 0];
        o[0] = b.x & 31; o[1] = b.y & 31; o[2] = b.z & 31; o[3] = b.w & 31;   // unpainted bytes: any lane, never stored
      }
      const int64_t p0 = w0 + 4 * (int64_t)g;
      const int64_t q0 = p0 - wbeg;                       // position relative to the warp's first one
      int64_t sv[4], wv[4], fv[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (which) sv[e] = s0 + o[e];
        if (within) {
          if (small) wv[e] = (q0 + e) - (int64_t)__shfl_sync(kFullMask, rel_beg, o[e]);   // warp-uniform branches
          else wv[e] = p0 + e - shfl_i64(beg, o[e]);
        }
        if (flat) fv[e] = (q0 + e) + shfl_i64(flat_c, o[e]);
      }
      if (g >= groups) continue;
      if (wide_stores && p0 >= wbeg && p0 + 4 <= w1) {
        if (which) st_v4_i64(which + p0, sv);
        if (within) st_v4_i64(within + p0, wv);
        if (flat) st_v4_i64(flat + p0, fv);
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int64_t p = p0 + e;
          if (p >= wbeg && p < w1) {
            if (which) which[p] = sv[e];
            if (within) within[p] = wv[e];
            if (flat) flat[p] = fv[e];
          }
        }
      }
    }
    __syncwarp();
  }
}

}  // namespace rua

using namespace rua;

extern "C" {

int rua_mask(const int64_t* len, int64_t B, int64_t W, const void* zero_host, const void* one_host,
             int32_t elem_bytes, void* out, rua_stream_t stream) {
  if (B < 0 || W < 0) return RUA_ERR_INVALID;
  if (B == 0 || W == 0) return RUA_OK;
  if (!len || !zero_host || !one_host || !out) return RUA_ERR_INVALID;
  if (((uintptr_t)out & 15u) != 0) return RUA_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t total = B * W;
  const int64_t per = 32 / elem_bytes;
  const int64_t blocks = ceil_div(ceil_div(total, per), 256 * kMaskIters);
  const int wide = ((uintptr_t)out & 31u) == 0;
  if (blocks >= (1ll << 31)) return RUA_ERR_UNSUPPORTED;
  switch (elem_bytes) {
    case 1: mask_kernel<uint8_t><<<(unsigned)blocks, 256, 0, st>>>(len, B, W, *(const uint8_t*)zero_host, *(const uint8_t*)one_host, (uint8_t*)out, wide); break;
    case 2: mask_kernel<uint16_t><<<(unsigned)blocks, 256, 0, st>>>(len, B, W, *(const uint16_t*)zero_host, *(const uint16_t*)one_host, (uint16_t*)out, wide); break;
    case 4: mask_kernel<uint32_t><<<(unsigned)blocks, 256, 0, st>>>(len, B, W, *(const uint32_t*)zero_host, *(const uint32_t*)one_host, (uint32_t*)out, wide); break;
    case 8: mask_kernel<uint64_t><<<(unsigned)blocks, 256, 0, st>>>(len, B, W, *(const uint64_t*)zero_host, *(const uint64_t*)one_host, (uint64_t*)out, wide); break;
    default: return RUA_ERR_INVALID;
  }
  return check_launch();
}

int rua_emit_ptr(const int64_t* off, int64_t S, int64_t n, const int64_t* relabel, int64_t* which,
                 int64_t* within, int64_t* flat, int64_t stride, int32_t right_align, rua_stream_t stream) {
  if (S < 0 || n < 0) return RUA_ERR_INVALID;
  if (n == 0) return RUA_OK;
  if (!off || S == 0) return RUA_ERR_INVALID;
  if (!which && !within && !flat) return RUA_OK;
  const int64_t blocks = ceil_div(n, kEmitTile);
  if (blocks >= (1ll << 31)) return RUA_ERR_UNSUPPORTED;
  const uintptr_t align = (uintptr_t)which | (uintptr_t)within | (uintptr_t)flat;
  // many short segments (C.ptr / L.idx / R.idx of a large batch): a warp per 32 segments, no per-tile decode chain
  if (!relabel && warpseg_applies(n, S)) {
    const int64_t wblocks = ceil_div(S, (int64_t)kEwWarps * 32);
    if (wblocks >= (1ll << 31)) return RUA_ERR_UNSUPPORTED;
    emit_ptr_warpseg_kernel<<<(unsigned)wblocks, kEwThreads, 0, (cudaStream_t)stream>>>(off, S, n, which, within, flat,
                                                                                       stride, right_align,
                                                                                       (align & 31u) == 0);
    return check_launch();
  }
  emit_ptr_kernel<<<(unsigned)blocks, kEmitThreads, 0, (cudaStream_t)stream>>>(off, S, n, relabel, which, within,
                                                                            flat, stride, right_align,
                                                                            (align & 31u) == 0);
  return check_launch();
}

}  // extern "C"
