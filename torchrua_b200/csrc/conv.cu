// K8 -- per-sequence depthwise 1-D convolution (causal or centred), forward and backward, on every layout.
//
// y(i, t, h) = bias[h] + sum_k w[h, k] x(i, t + k - pad, h), x = 0 outside [0, len_i).  Replaces pad (x.left(0)) ->
// F.conv1d(groups=H) on (B, H, T) -> unpad, which moves the padding twice and transposes the layout both ways.
//
// Design (HBM-bound for small K, like K4 / K7):
//   * positions in the VIRTUAL order of K7 (seq_decode.cuh): sequence-major for C and P, storage order for L / R, cut
//     into chunks of R positions regardless of sequence boundaries.  Tap k of the output at position j reads position
//     j + k - pad, and it is valid exactly when 0 <= t + k - pad < len for the output's own (t, len): then that position
//     is token t + k - pad of the same sequence.  So a chunk needs only its rows plus a halo of pad rows before and
//     K - 1 - pad after, and no sequence lookup beyond the decode of those positions;
//   * a CTA of 256 threads owns a column block (TPC threads x one 16-byte vector, or one element when H is not a multiple
//     of the vector) and walks chunks in a fixed grid stride.  Per chunk it decodes the positions, stages the chunk and
//     its halo in shared memory (each row read once from global, 16-byte loads), and every thread then computes kRG
//     consecutive outputs per pass from the staged rows.  Up to kPasses passes per chunk keep enough loads in flight
//     per stage (a chunk of one pass left the HBM idle through the decode and barriers: 27 % of copy peak at K = 4).
//     A thread whose rows all have every tap valid (the common case) runs the tap loop without per-tap predicates;
//   * taps: K <= reg_taps (8; 4 / none for 16-bit rows) are held in registers (raw storage words, unpacked per tap), larger
//     K are staged once per CTA in shared memory next to the rows;
//   * rows that hold no token (L / R padding, C rows at or past off[B]) are copied through from the staged rows.
// Backward, one pass over grad_out and x:
//   * grad_in is the same convolution of grad_out with flipped taps and pad' = K - 1 - pad;
//   * grad_weight[h, k] = sum grad_out(i, t, h) x(i, t + k - pad, h) over valid taps, grad_bias[h] = sum grad_out.  Each
//     CTA accumulates its chunks in registers (thread = (tap, column vector) pair) and stores one fixed slot; the slots
//     are summed in slot order by slot_sum (slot_sum.cuh).  The grid, and so the number of slots, is a host function of
//     (rows, H, K, dtype) capped at kGridCTAs: fixed assignment, no atomics, bit-identical run to run, bounded workspace.
#include "reduce_common.cuh"
#include "seq_decode.cuh"
#include "slot_sum.cuh"

namespace rua {
namespace {

constexpr int kConvThreads = 256;
constexpr int kMaxTPC = 32;                  // threads across a column block: a 512-byte slab per warp
constexpr int kRG = 4;                       // consecutive output positions per thread and pass
constexpr int kPasses = 4;                   // passes over a chunk: R = kPasses x G x kRG rows staged at once
constexpr size_t kSmemTarget = 100 * 1024;   // fewer passes above this: two CTAs per SM must fit
// taps held in registers for K <= reg_taps: 8, but 4 for the forward of 16-bit rows and none for their backward (next to
// the kRG x 8 fp32 accumulators, and the weight-gradient accumulators of the backward, eight 16-byte tap vectors exceed
// the 128 registers of two CTAs per SM and spill; ptxas -v)
template <int V, bool kBwd> __host__ __device__ constexpr int reg_taps() { return V == 8 ? (kBwd ? 0 : 4) : 8; }
constexpr int kMaxK = 32;
constexpr int kGridCTAs = 8 * kNumSMs;       // CTAs per launch at most (= weight-gradient slots of the backward)
constexpr int kPairs = ((kMaxK + 1) * kMaxTPC + kConvThreads - 1) / kConvThreads;   // (tap, column) pairs per thread

struct ConvArgs {
  const void* in;        // x (forward) / grad_out (backward): also the source of copied-through rows
  const void* x;         // backward: the forward input (grad_weight only)
  const void* weight;    // (H, K) row-major
  const void* bias;      // forward, nullable
  void* out;             // y / grad_in (backward: nullable)
  void* slots;           // backward: per-CTA partial sums of grad_weight / grad_bias
  int64_t H;
  int64_t B;
  const int64_t* off;
  const int64_t* poff;
  const int64_t* unsorted;
  int32_t layout;
  int64_t W;
  int64_t rows;
  int K;
  int pad;               // pad of this launch's convolution (backward: K - 1 - forward pad, taps flipped)
  int fpad;              // forward pad (backward: the grad_weight window)
  int want_gw, want_gb;  // backward
  int tpc_log2;
  int R;
  int ncb;
  int64_t chunks;
};

// shared memory: decoded storage rows (R + 2 (K - 1)), per-output tap bounds, then the staged tiles and taps
struct SmemLayout {
  size_t lo, tile, xtile, taps, total;
};
__host__ __device__ inline SmemLayout smem_layout(int R, int K, int CW, int esz, bool bwd, bool reg_taps) {
  SmemLayout s;
  const size_t eu = (size_t)R + 2 * (K - 1), e = (size_t)R + K - 1, row = (size_t)CW * esz;
  s.lo = eu * 8;
  s.tile = (s.lo + 16 * (size_t)R + 15) / 16 * 16;
  s.xtile = s.tile + e * row;
  s.taps = s.xtile + (bwd ? e * row : 0);
  s.total = s.taps + (reg_taps ? 0 : (size_t)K * row);
  return s;
}

template <typename T, int V> __device__ __forceinline__ Raw<T, V> raw_at(const T* p) {
  Raw<T, V> w;
  if constexpr (V == 1) w.r = *p;
  else w.r = *reinterpret_cast<const uint4*>(p);
  return w;
}
template <typename T, int V> __device__ __forceinline__ void put_raw(T* p, const Raw<T, V>& w) {
  if constexpr (V == 1) *p = w.r;
  else *reinterpret_cast<uint4*>(p) = w.r;
}
template <typename T, int V> __device__ __forceinline__ Raw<T, V> zero_raw() {
  Raw<T, V> w;
  if constexpr (V == 1) w.r = Store<T>::from_acc(0);
  else w.r = make_uint4(0, 0, 0, 0);
  return w;
}

// V taps k of the columns col0 .. col0 + V - 1 (zero past H or K), flipped for the backward
template <typename T, int V, bool kBwd>
__device__ __forceinline__ Raw<T, V> load_taps(const ConvArgs& a, int64_t col0, int k) {
  T v[V];
  const T* w = static_cast<const T*>(a.weight);
  const int kk = kBwd ? a.K - 1 - k : k;
#pragma unroll
  for (int e = 0; e < V; ++e) v[e] = (k < a.K && col0 + e < a.H) ? w[(col0 + e) * a.K + kk] : Store<T>::from_acc(0);
  Raw<T, V> r;
  if constexpr (V == 1) r.r = v[0];
  else memcpy(&r.r, v, 16);
  return r;
}

template <typename T, int V, bool kBwd, bool kReg>
__global__ void __launch_bounds__(kConvThreads, 2) segconv_kernel(ConvArgs a) {
  using A = typename Store<T>::Acc;
  using RawV = Raw<T, V>;
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ int64_t s_bounds[2];
  const int K = a.K, pad = a.pad, R = a.R;
  const int E = R + K - 1, Eu = R + 2 * (K - 1);
  const int TPC = 1 << a.tpc_log2, G = kConvThreads >> a.tpc_log2, CW = TPC * V;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int grp = tid >> a.tpc_log2, lc = tid & (TPC - 1);
  const int cb = (int)(blockIdx.x % (unsigned)a.ncb);
  const int64_t slot = blockIdx.x / (unsigned)a.ncb, nslot = gridDim.x / (unsigned)a.ncb;
  const int64_t col0 = (int64_t)cb * CW + lc * V;
  const bool act = col0 < a.H;
  const SmemLayout L = smem_layout(R, K, CW, sizeof(T), kBwd, kReg);
  int64_t* s_row = reinterpret_cast<int64_t*>(smem);                 // [Eu] storage row of position q0 - (K - 1) + u
  int* s_lo = reinterpret_cast<int*>(smem + L.lo);                    // [R] first valid tap of this launch's conv
  int* s_hi = s_lo + R;                                               // [R] one past the last; < 0: no token (copy)
  int* s_flo = s_hi + R;                                              // [R] backward: forward-pad tap bounds
  int* s_fhi = s_flo + R;
  T* tile = reinterpret_cast<T*>(smem + L.tile);                      // [E][CW] rows from position q0 - pad
  T* xtile = reinterpret_cast<T*>(smem + L.xtile);                    // [E][CW] backward: x from q0 - fpad
  T* taps = reinterpret_cast<T*>(smem + L.taps);                      // [K][CW] taps not in registers
  const T* in = static_cast<const T*>(a.in);
  const bool want_w = kBwd && (a.want_gw || a.want_gb);

  constexpr int kRegTaps = kReg ? reg_taps<V, kBwd>() : 1;
  RawV wr[kReg ? kRegTaps : 1];
  if constexpr (kReg) {
#pragma unroll
    for (int k = 0; k < kRegTaps; ++k) wr[k] = load_taps<T, V, kBwd>(a, col0, k);
  } else {
    for (int i = tid; i < K * TPC; i += kConvThreads) {
      const int k = i >> a.tpc_log2, l = i & (TPC - 1);
      put_raw<T, V>(taps + k * CW + l * V, load_taps<T, V, kBwd>(a, (int64_t)cb * CW + l * V, k));
    }
  }
  A bv[V];
#pragma unroll
  for (int e = 0; e < V; ++e)
    bv[e] = (!kBwd && a.bias && col0 + e < a.H) ? Store<T>::to_acc(static_cast<const T*>(a.bias)[col0 + e]) : A(0);
  A gacc[kBwd ? kPairs : 1][V];
#pragma unroll
  for (int m = 0; m < (kBwd ? kPairs : 1); ++m)
#pragma unroll
    for (int e = 0; e < V; ++e) gacc[m][e] = A(0);

  const int64_t n_tok = __ldg(a.off + a.B);
  for (int64_t c = slot; c < a.chunks; c += nslot) {
    const int64_t q0 = c * R;
    const int nq = a.rows - q0 < R ? (int)(a.rows - q0) : R;
    const int64_t u0 = q0 - (K - 1);
    // ---- decode the chunk's positions and its halo ---------------------------------------------------------------
    int64_t lo, hi;
    owner_bounds(a, n_tok, u0 > 0 ? u0 : 0, min(q0 + nq + K - 2, a.rows - 1), lane, warp, s_bounds, lo, hi);
    for (int u = tid; u < Eu; u += kConvThreads) {
      const int64_t j = u0 + u;
      const int q = u - (K - 1);
      int64_t srow = -1, t;
      int clo = 0, chi = -1, flo = 0, fhi = -1;
      if (j >= 0 && j < a.rows) {
        decode_position(a, j, n_tok, lo, hi, srow, t, [&](int64_t, int64_t len) {
          clo = (int)max((int64_t)0, pad - t);
          chi = (int)min((int64_t)K, len - t + pad);
          flo = (int)max((int64_t)0, a.fpad - t);
          fhi = (int)min((int64_t)K, len - t + a.fpad);
        });
      }
      s_row[u] = srow;
      if (q >= 0 && q < R) {
        s_lo[q] = clo;
        s_hi[q] = chi;
        if constexpr (kBwd) {
          s_flo[q] = flo;
          s_fhi[q] = fhi;
        }
      }
    }
    __syncthreads();
    // ---- stage the rows: each row of the chunk and its halo read once -------------------------------------------
    auto stage = [&](T* dst, const T* src, int base) {   // dst row e = position q0 - (K - 1) + base + e
      for (int e = grp; e < E; e += G) {
        const int64_t j = u0 + base + e;
        RawV v = zero_raw<T, V>();
        if (act && j >= 0 && j < a.rows) load_raw<T, V>(src + s_row[base + e] * a.H + col0, v);
        put_raw<T, V>(dst + e * CW + lc * V, v);
      }
    };
    stage(tile, in, K - 1 - pad);
    if (want_w && a.want_gw) stage(xtile, static_cast<const T*>(a.x), K - 1 - a.fpad);
    __syncthreads();

    // ---- the convolution: kRG consecutive outputs per thread and pass ---------------------------------------------
    for (int qb = grp * kRG; a.out && qb < nq; qb += G * kRG) {
      int rlo[kRG], rhi[kRG];
      bool interior = true;
#pragma unroll
      for (int r = 0; r < kRG; ++r) {
        rlo[r] = s_lo[qb + r];
        rhi[r] = s_hi[qb + r];
        interior &= qb + r >= nq || (rlo[r] == 0 && rhi[r] == K);
      }
      A acc[kRG][V];
#pragma unroll
      for (int r = 0; r < kRG; ++r)
#pragma unroll
        for (int e = 0; e < V; ++e) acc[r][e] = bv[e];
      auto taps_loop = [&](auto all_valid) {
        auto tap = [&](int k, const RawV& wk) {
          A w[V];
          unpack_raw<T, V>(wk, w);
#pragma unroll
          for (int r = 0; r < kRG; ++r) {
            if (decltype(all_valid)::value || (k >= rlo[r] && k < rhi[r])) {
              A x[V];
              unpack_raw<T, V>(raw_at<T, V>(tile + (qb + r + k) * CW + lc * V), x);
#pragma unroll
              for (int e = 0; e < V; ++e) acc[r][e] += w[e] * x[e];
            }
          }
        };
        if constexpr (kReg) {
#pragma unroll
          for (int k = 0; k < kRegTaps; ++k)
            if (k < K) tap(k, wr[k]);
        } else {
          for (int k = 0; k < K; ++k) tap(k, raw_at<T, V>(taps + k * CW + lc * V));
        }
      };
      if (interior) taps_loop(std::true_type{});
      else taps_loop(std::false_type{});
      if (act) {
        T* out = static_cast<T*>(a.out);
#pragma unroll
        for (int r = 0; r < kRG; ++r) {
          const int q = qb + r;
          if (q >= nq) break;
          const int64_t o = s_row[q + K - 1] * a.H + col0;
          if (rhi[r] < 0) put_raw<T, V>(out + o, raw_at<T, V>(tile + (q + pad) * CW + lc * V));
          else store_vec<T, V>(out + o, acc[r]);
        }
      }
    }

    // ---- grad_weight / grad_bias partials: thread = (tap k, column vector) pairs, k = K is the bias ---------------
    if constexpr (kBwd) {
      if (want_w) {
#pragma unroll
        for (int m = 0; m < kPairs; ++m) {
          const int pair = tid + m * kConvThreads;
          const int k = pair >> a.tpc_log2, l = pair & (TPC - 1);
          if (k > K || (k == K ? !a.want_gb : !a.want_gw)) continue;
          for (int q = 0; q < nq; ++q) {
            const int flo = s_flo[q], fhi = s_fhi[q];
            if (k == K ? fhi < 0 : (k < flo || k >= fhi)) continue;
            A g[V];
            unpack_raw<T, V>(raw_at<T, V>(tile + (q + pad) * CW + l * V), g);
            if (k == K) {
#pragma unroll
              for (int e = 0; e < V; ++e) gacc[m][e] += g[e];
            } else {
              A x[V];
              unpack_raw<T, V>(raw_at<T, V>(xtile + (q + k) * CW + l * V), x);
#pragma unroll
              for (int e = 0; e < V; ++e) gacc[m][e] += g[e] * x[e];
            }
          }
        }
      }
    }
    __syncthreads();   // the next chunk overwrites the staged rows
  }

  if constexpr (kBwd) {
    if (want_w) {
      A* slots = static_cast<A*>(a.slots) + (slot * a.ncb + cb) * (int64_t)(K + 1) * CW;
#pragma unroll
      for (int m = 0; m < kPairs; ++m) {
        const int pair = tid + m * kConvThreads;
        const int k = pair >> a.tpc_log2, l = pair & (TPC - 1);
        if (k > K) continue;
#pragma unroll
        for (int e = 0; e < V; ++e) __stcg(slots + (int64_t)k * CW + l * V + e, gacc[m][e]);
      }
    }
  }
}

// columns of the slot sum: grad_weight[h, k] (k < K) and grad_bias[h] (k = K), column i = k * H + h
template <typename T> struct ConvCols {
  T* gw;
  T* gb;
  int64_t H;
  int K, CW;
  __device__ T* operator()(int64_t i, int64_t& src) const {
    const int k = (int)(i / H);
    const int64_t h = i - (int64_t)k * H;
    const int64_t cb = h / CW, c = h - cb * CW;
    src = (cb * (K + 1) + k) * CW + c;
    if (k < K) return gw ? gw + h * K + k : nullptr;
    return gb ? gb + h : nullptr;
  }
};

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
struct Plan {
  int tpc_log2, R, ncb;
  int64_t chunks, S;
  size_t smem, ws;
};

template <typename T, int V> Plan make_plan(int64_t rows, int64_t H, int K, bool bwd) {
  Plan p{};
  const int64_t vecs = ceil_div(H, V);
  int tpc = 1;
  while (tpc < kMaxTPC && tpc < vecs) tpc <<= 1;
  p.tpc_log2 = __builtin_ctz(tpc);
  const bool reg = K <= (bwd ? reg_taps<V, true>() : reg_taps<V, false>());
  for (int passes = kPasses; passes >= 1; passes >>= 1) {
    p.R = passes * (kConvThreads / tpc) * kRG;
    p.smem = smem_layout(p.R, K, tpc * V, sizeof(T), bwd, reg).total;
    if (p.smem <= kSmemTarget) break;
  }
  p.ncb = (int)ceil_div(vecs, tpc);
  p.chunks = ceil_div(rows, p.R);
  const int64_t per_cb = kGridCTAs / p.ncb;
  p.S = p.chunks < per_cb ? p.chunks : (per_cb > 0 ? per_cb : 1);
  p.ws = bwd ? (size_t)p.S * p.ncb * (K + 1) * tpc * V * sizeof(typename Store<T>::Acc) : 0;
  return p;
}

// f(Type<T>{}, Int<V>{}) for `dtype` at the full 16-byte vector when `vec` allows it and H is a multiple of it, else
// one element per thread
template <typename F> int with_conv_type(int32_t dtype, bool vec, int64_t H, F&& f) {
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    constexpr int VV = 16 / sizeof(T);
    if (!vec || H % VV != 0) return f(t, Int<1>{});
    return f(t, Int<VV>{});
  });
}

bool aligned16(const void* p) { return p == nullptr || ((uintptr_t)p & 15) == 0; }

int validate(int64_t H, int32_t dtype, int32_t K, int32_t pad, const rua_ragged_t* rg, const rua_side_t* side) {
  if (H < 1 || dtype < RUA_F32 || dtype > RUA_BF16 || K < 1 || pad < 0 || pad > K - 1) return RUA_ERR_INVALID;
  if (K > kMaxK) return RUA_ERR_UNSUPPORTED;
  if (!rg || !side || rg->B < 0 || !rg->off || side->rows < 0 || side->width < 0) return RUA_ERR_INVALID;
  if (side->len_xform != RUA_LEN_SAME) return RUA_ERR_UNSUPPORTED;
  switch (side->layout) {
    case RUA_CAT: break;
    case RUA_PACK:
      if (!rg->poff || !rg->unsorted) return RUA_ERR_INVALID;
      break;
    case RUA_LEFT: case RUA_RIGHT:
      if (side->rows != rg->B * side->width) return RUA_ERR_INVALID;
      break;
    default: return RUA_ERR_INVALID;
  }
  return RUA_OK;
}

int run(bool bwd, int32_t dtype, int64_t H, int32_t K, int32_t pad, const rua_ragged_t* rg, const rua_side_t* side,
        ConvArgs a, bool vec, void* gw, void* gb, void* ws, size_t ws_bytes, rua_stream_t stream) {
  const int64_t rows = side->rows;
  if (rows == 0) return RUA_OK;
  return with_conv_type(dtype, vec, H, [&](auto t, auto v) {
    using T = typename decltype(t)::type;
    constexpr int V = decltype(v)::value;
    const Plan p = make_plan<T, V>(rows, H, K, bwd);
    if (bwd && (gw || gb) && (!ws || ws_bytes < p.ws)) return (int)RUA_ERR_WORKSPACE;
    if (p.S * p.ncb > 0x7fffffffLL) return (int)RUA_ERR_UNSUPPORTED;
    a.H = H;
    a.B = rg->B;
    a.off = rg->off;
    a.poff = rg->poff;
    a.unsorted = rg->unsorted;
    a.layout = side->layout;
    a.W = side->width;
    a.rows = rows;
    a.K = K;
    a.fpad = pad;
    a.pad = bwd ? K - 1 - pad : pad;
    a.want_gw = gw != nullptr;
    a.want_gb = gb != nullptr;
    a.slots = ws;
    a.tpc_log2 = p.tpc_log2;
    a.R = p.R;
    a.ncb = p.ncb;
    a.chunks = p.chunks;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    auto launch = [&](auto kern) {
      if (p.smem > 48 * 1024) {
        if (int rc = check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem)))
          return rc;
      }
      kern<<<(unsigned)(p.S * p.ncb), kConvThreads, p.smem, st>>>(a);
      return check_launch();
    };
    int rc = with_bool(bwd, [&](auto b) {
      constexpr bool kB = decltype(b)::value;
      if constexpr (reg_taps<V, kB>() > 0) {
        if (K <= reg_taps<V, kB>()) return launch(segconv_kernel<T, V, kB, true>);
      }
      return launch(segconv_kernel<T, V, kB, false>);
    });
    if (rc || !bwd || (!gw && !gb)) return rc;
    const int CW = (1 << p.tpc_log2) * V;
    return launch_slot_sum<T>(static_cast<const typename Store<T>::Acc*>(ws), p.S, (int64_t)p.ncb * (K + 1) * CW,
                              (int64_t)(K + 1) * H, ConvCols<T>{static_cast<T*>(gw), static_cast<T*>(gb), H, K, CW}, st);
  });
}

}  // namespace
}  // namespace rua

using namespace rua;

extern "C" size_t rua_segment_conv_workspace_bytes(int64_t rows, int64_t H, int32_t K, int32_t dtype, int32_t backward) {
  if (rows <= 0 || H < 1 || K < 1 || K > kMaxK || dtype < RUA_F32 || dtype > RUA_BF16 || !backward) return 0;
  size_t total = 0;
  for (bool vec : {true, false})
    with_conv_type(dtype, vec, H, [&](auto t, auto v) {
      const size_t w = make_plan<typename decltype(t)::type, decltype(v)::value>(rows, H, K, true).ws;
      total = w > total ? w : total;
      return RUA_OK;
    });
  return total;
}

extern "C" int rua_segment_conv(const void* src, const void* weight, const void* bias, void* dst, int64_t H,
                                int32_t dtype, int32_t K, int32_t pad, const rua_ragged_t* ragged,
                                const rua_side_t* side, void* ws, size_t ws_bytes, rua_stream_t stream) {
  if (int rc = validate(H, dtype, K, pad, ragged, side)) return rc;
  if (side->rows > 0 && (!src || !weight || !dst)) return RUA_ERR_INVALID;
  ConvArgs a{};
  a.in = src;
  a.weight = weight;
  a.bias = bias;
  a.out = dst;
  const bool vec = aligned16(src) && aligned16(dst);
  return run(false, dtype, H, K, pad, ragged, side, a, vec, nullptr, nullptr, ws, ws_bytes, stream);
}

extern "C" int rua_segment_conv_backward(const void* grad_out, const void* x, const void* weight, void* grad_in,
                                         void* grad_weight, void* grad_bias, int64_t H, int32_t dtype, int32_t K,
                                         int32_t pad, const rua_ragged_t* ragged, const rua_side_t* side, void* ws,
                                         size_t ws_bytes, rua_stream_t stream) {
  if (int rc = validate(H, dtype, K, pad, ragged, side)) return rc;
  if (side->rows > 0) {
    if (!grad_out || !weight || (grad_weight && !x)) return RUA_ERR_INVALID;
    if (!grad_in && !grad_weight && !grad_bias) return RUA_OK;
  }
  ConvArgs a{};
  a.in = grad_out;
  a.x = x;
  a.weight = weight;
  a.out = grad_in;
  const bool vec = aligned16(grad_out) && aligned16(grad_in) && aligned16(grad_weight ? x : nullptr);
  return run(true, dtype, H, K, pad, ragged, side, a, vec, grad_weight, grad_bias, ws, ws_bytes, stream);
}
