// K7 -- per-sequence prefix scans: cumsum / logcumsumexp / cummax / cummin, forward and backward, on every layout.
//
// Replaces the pad -> torch.cumsum(dim=1) -> unpad composition a user would otherwise write (x.left(fill), one ATen
// scan over B x T x D bytes, back to the source layout): N*D bytes are read once and written once, whatever the layout.
//
// Design (HBM-bound, like K4):
//   * positions are taken in VIRTUAL order -- sequence-major (C order) for C and P, storage order for L / R -- and cut
//     into chunks of R consecutive positions regardless of sequence boundaries; the storage row of a position comes from
//     the layout formula of include/rua_b200.h, so P reads the same rows as C.  reverse=True walks the same order
//     backwards.  Rows that hold no token (L / R padding, C rows past off[B]) are copied through in the same pass;
//   * a CTA of 256 threads owns (chunk, column block): G = 256 / TPC groups of TPC threads, every thread one 16-byte
//     column vector (or one element when H is not a multiple of the vector), every group kRG consecutive positions.
//     The rows of a group are loaded at once (kRG loads in flight) and held in registers for both passes below;
//   * pass 1 reduces every group to a segmented aggregate (did a segment start here?, value since the last start);
//     the groups are combined by a Kogge-Stone scan in shared memory (fixed tree: deterministic);
//   * carries between chunks: chunks are taken through a ticket counter, so a predecessor is always scheduled before a
//     successor waits on it (no deadlock at any occupancy).  A chunk publishes its inclusive value at once when a
//     segment starts in it, otherwise its aggregate first and the inclusive value once its own carry is known.  A
//     successor looks back to the nearest published inclusive value and folds the aggregates after it FORWARD, in
//     chunk order: the result is exactly inclusive_c = inclusive_{c-1} (+) aggregate_c, the chained form, however far
//     the look-back had to go -- so floating-point results do not depend on timing.  Only chunks whose last position
//     continues into the next chunk publish anything;
//   * pass 2 replays the held rows with the carry and stores every row once.
//
// Operators (per column; S is the scan state, (+) = compose, applied in scan order):
//   sum        S = x                    a (+) b = a + b
//   logsumexp  S = y                    a (+) b = logaddexp(a, b)   (torch's infinity / NaN rules)
//   max / min  S = (value, index)       b wins when b is NaN or (a is not NaN and b >= a / b <= a): ties and NaN as
//                                       torch.cummax / cummin (the later position wins a tie, a NaN sticks)
//   logcumsumexp backward, in reverse scan order: v_k = g_k + exp(y_k - y_prev) v_prev, grad x_k = exp(x_k - y_k) v_k.
//              S = (v, y of the last position); a (+) b = (exp(b.y - a.y) a.v + b.v, b.y).  The exponent is <= 0
//              (y is monotone in scan order), so nothing overflows
//   cummax / cummin backward, in reverse scan order: grad x_k = sum of g_j over the run of positions whose index is k
//              (the run starts at j = k).  S = (acc, pass) with pass = 0 at a run start: an affine map with slope 0/1.
//   linear recurrence h_t = a_t h_{t-1} + x_t: S = (m, b), the affine map h -> m h + b; an element lifts to (a_t, x_t),
//              (a_t, a_t h0[i] + x_t) at the first position of sequence i when an initial state is given;
//              p (+) q = (p.m q.m, q.m p.b + q.b); the output is b
//   linear recurrence backward, in reverse scan order: with g~_t = g_t + a_{t+1} g~_{t+1} (the whole adjoint of h_t),
//              z_t = a_t g~_t is the same affine scan over the elements (a_t, a_t g_t).  grad x_t = g~_t = g_t + z_{t+1}
//              (the exclusive state), grad a_t = g~_t h_{t-1} (h_{t-1} = the forward output at the previous position, or
//              h0[i] / 0 at the first), grad h0[i] = z at the first position.  h_{t-1} lies at a closed-form row of the
//              same sequence (C / L / R srow -+ 1, P srow -+ the batch size between the two steps), so no halo is staged
#include "reduce_common.cuh"
#include "seq_decode.cuh"

namespace rua {
namespace {

constexpr int kScanThreads = 256;
constexpr int kMaxTPC = 32;   // threads across a row: a 512-byte slab per warp, >= 4 groups per CTA
constexpr uint8_t kTok = 1, kStart = 2, kEnd = 4;

struct ScanArgs {
  const void* in0;          // x (forward) / grad_out (backward): also the source of copied-through rows
  const void* in1;          // logcumsumexp backward: x
  const void* in2;          // logcumsumexp backward: y
  const int64_t* idx_in;    // cummax / cummin backward: indices of the forward pass
  void* out;
  int64_t* idx_out;         // cummax / cummin forward
  int64_t H;
  int64_t B;
  const int64_t* off;
  const int64_t* poff;
  const int64_t* unsorted;
  int32_t layout;
  int32_t reverse;          // scan direction of this launch
  int64_t W;
  int64_t rows;
  int tpc_log2;
  int R;
  int ncb;
  unsigned long long* ticket;
  int* flags;
  void* agg;
  void* inc;
  const void* h0;           // linear recurrence: initial states (B x H), NULL for zero
  void* out_gate;           // linear recurrence backward: grad gate (NULL: not wanted)
  void* out_h0;             // linear recurrence backward: grad h0 (NULL: not wanted)
};

template <typename A> __device__ __forceinline__ bool is_nan(A v) { return v != v; }

// torch's _log_add_exp_helper: equal infinities return themselves instead of inf - inf = NaN
template <bool kFast, typename A> __device__ __forceinline__ A log_add_exp(A a, A b) {
  const A mn = is_nan(b) ? b : (a < b ? a : b);
  const A mx = is_nan(b) ? b : (a < b ? b : a);
  if (mn != mx || isfinite(mn)) return mx + log_acc<kFast>(A(1) + exp_acc<kFast>(mn - mx));
  return a;
}

template <int V> __device__ __forceinline__ void store_i64(int64_t* p, const int64_t* v) {
  if constexpr (V % 2 == 0) {
#pragma unroll
    for (int k = 0; k < V; k += 2) *reinterpret_cast<longlong2*>(p + k) = make_longlong2(v[k], v[k + 1]);
  } else {
#pragma unroll
    for (int k = 0; k < V; ++k) p[k] = v[k];
  }
}

template <typename T, int V> __device__ __forceinline__ void copy_row(const ScanArgs& a, int64_t o, bool idx) {
  Raw<T, V> w;
  load_raw<T, V>(static_cast<const T*>(a.in0) + o, w);
  if constexpr (V == 1) static_cast<T*>(a.out)[o] = w.r;
  else *reinterpret_cast<uint4*>(static_cast<T*>(a.out) + o) = w.r;
  if (idx) {
    int64_t z[V];
#pragma unroll
    for (int k = 0; k < V; ++k) z[k] = 0;
    store_i64<V>(a.idx_out + o, z);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// operators
// ---------------------------------------------------------------------------------------------------------------------
template <typename T, int V_> struct OpSum {
  static constexpr int V = V_, kRG = 16;
  static constexpr int kMinBlocks = 2;
  static constexpr bool kIdx = false, kSeq = false;
  using Tp = T;
  using A = typename Store<T>::Acc;
  struct S { A v; };
  struct E { Raw<T, V> x; };
  __device__ static void load(E& e, const ScanArgs& a, int64_t o, int64_t) { load_raw<T, V>(static_cast<const T*>(a.in0) + o, e.x); }
  __device__ static void lift(const E& e, int64_t, S* s) {
    A x[V];
    unpack_raw<T, V>(e.x, x);
#pragma unroll
    for (int k = 0; k < V; ++k) s[k].v = x[k];
  }
  __device__ static S compose(const S& a, const S& b) { return {a.v + b.v}; }
  __device__ static void emit(const ScanArgs& a, int64_t o, const E&, int64_t, bool, const S*, const S* s) {
    A y[V];
#pragma unroll
    for (int k = 0; k < V; ++k) y[k] = s[k].v;
    store_vec<T, V>(static_cast<T*>(a.out) + o, y);
  }
};

template <typename T, int V_> struct OpLse : OpSum<T, V_> {
  using Base = OpSum<T, V_>;
  using typename Base::S;
  static constexpr bool kFast = sizeof(T) == 2;
  __device__ static S compose(const S& a, const S& b) { return {log_add_exp<kFast>(a.v, b.v)}; }
};

template <typename T, int V_, bool kMax> struct OpExt {
  static constexpr int V = V_, kRG = 8;   // the (value, index) state doubles the registers per column
  static constexpr int kMinBlocks = 2;
  static constexpr bool kIdx = true, kSeq = false;
  using Tp = T;
  using A = typename Store<T>::Acc;
  struct S { A v; int32_t i; };   // a position within a sequence: the host refuses >= 2^31 rows
  struct E { Raw<T, V> x; };
  __device__ static void load(E& e, const ScanArgs& a, int64_t o, int64_t) { load_raw<T, V>(static_cast<const T*>(a.in0) + o, e.x); }
  __device__ static void lift(const E& e, int64_t t, S* s) {
    A x[V];
    unpack_raw<T, V>(e.x, x);
#pragma unroll
    for (int k = 0; k < V; ++k) s[k] = {x[k], (int32_t)t};
  }
  __device__ static S compose(const S& a, const S& b) {
    const bool take = is_nan(b.v) || (!is_nan(a.v) && (kMax ? b.v >= a.v : b.v <= a.v));
    return take ? b : a;
  }
  __device__ static void emit(const ScanArgs& a, int64_t o, const E&, int64_t, bool, const S*, const S* s) {
    A y[V];
    int64_t ix[V];
#pragma unroll
    for (int k = 0; k < V; ++k) { y[k] = s[k].v; ix[k] = s[k].i; }
    store_vec<T, V>(static_cast<T*>(a.out) + o, y);
    store_i64<V>(a.idx_out + o, ix);
  }
};

template <typename T, int V_> struct OpLseBwd {
  static constexpr int V = V_, kRG = 4;   // three inputs held per row
  static constexpr int kMinBlocks = sizeof(T) == 2 ? 1 : 2;   // eight fp32 (v, y) states per thread: 128 registers spill
  static constexpr bool kIdx = false, kSeq = false;
  static constexpr bool kFast = sizeof(T) == 2;
  using Tp = T;
  using A = typename Store<T>::Acc;
  struct S { A v; A y; };
  struct E { Raw<T, V> g, x, y; };
  __device__ static void load(E& e, const ScanArgs& a, int64_t o, int64_t) {
    load_raw<T, V>(static_cast<const T*>(a.in0) + o, e.g);
    load_raw<T, V>(static_cast<const T*>(a.in1) + o, e.x);
    load_raw<T, V>(static_cast<const T*>(a.in2) + o, e.y);
  }
  __device__ static void lift(const E& e, int64_t, S* s) {
    A g[V], y[V];
    unpack_raw<T, V>(e.g, g);
    unpack_raw<T, V>(e.y, y);
#pragma unroll
    for (int k = 0; k < V; ++k) s[k] = {g[k], y[k]};
  }
  __device__ static S compose(const S& a, const S& b) {
    const A f = b.y == a.y ? A(1) : exp_acc<kFast>(b.y - a.y);   // equal (also both -inf): factor 1, not exp(NaN)
    return {f * a.v + b.v, b.y};
  }
  __device__ static void emit(const ScanArgs& a, int64_t o, const E& e, int64_t, bool, const S*, const S* s) {
    A x[V], y[V], r[V];
    unpack_raw<T, V>(e.x, x);
    unpack_raw<T, V>(e.y, y);
#pragma unroll
    for (int k = 0; k < V; ++k) r[k] = x[k] == -inf_of<A>() ? A(0) : exp_acc<kFast>(x[k] - y[k]) * s[k].v;
    store_vec<T, V>(static_cast<T*>(a.out) + o, r);
  }
};

template <typename T, int V_> struct OpRunBwd {
  static constexpr int V = V_, kRG = 8;
  static constexpr int kMinBlocks = 2;
  static constexpr bool kIdx = false, kSeq = false;
  using Tp = T;
  using A = typename Store<T>::Acc;
  struct S { A v; int pass; };
  struct E { Raw<T, V> g; uint32_t start; };   // start bit k: position holds its own forward index (a run starts)
  __device__ static void load(E& e, const ScanArgs& a, int64_t o, int64_t t) {
    load_raw<T, V>(static_cast<const T*>(a.in0) + o, e.g);
    const int64_t* ip = a.idx_in + o;
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < V; ++k) m |= (uint32_t)(__ldcs(reinterpret_cast<const long long*>(ip) + k) == (long long)t) << k;
    e.start = m;
  }
  __device__ static void lift(const E& e, int64_t, S* s) {
    A g[V];
    unpack_raw<T, V>(e.g, g);
#pragma unroll
    for (int k = 0; k < V; ++k) s[k] = ((e.start >> k) & 1) ? S{A(0), 0} : S{g[k], 1};
  }
  __device__ static S compose(const S& a, const S& b) { return {b.pass ? a.v + b.v : b.v, a.pass & b.pass}; }
  __device__ static void emit(const ScanArgs& a, int64_t o, const E& e, int64_t, bool has_before, const S* before, const S*) {
    A g[V], r[V];
    unpack_raw<T, V>(e.g, g);
#pragma unroll
    for (int k = 0; k < V; ++k) r[k] = ((e.start >> k) & 1) ? (has_before ? before[k].v : A(0)) + g[k] : A(0);
    store_vec<T, V>(static_cast<T*>(a.out) + o, r);
  }
};

// Operators with kSeq also receive, per row, the decode flags and the offset ho = i * H + col0 of the row's column vector
// in the per-sequence (B x H) arrays (lift also gets act: a thread past the row end must not read there); their non-token
// rows go through pass() instead of copy_row.
template <typename T, int V> __device__ __forceinline__ Raw<T, V> zero_raw() {
  Raw<T, V> w;
  if constexpr (V == 1) w.r = Store<T>::from_acc(typename Store<T>::Acc(0));
  else w.r = make_uint4(0, 0, 0, 0);
  return w;
}

template <typename T, int V_> struct OpLinRec {
  static constexpr int V = V_, kRG = 6;   // two register images per row: kRG = 8 spills at 128 registers
  static constexpr int kMinBlocks = 2;
  static constexpr bool kSeq = true;
  using Tp = T;
  using A = typename Store<T>::Acc;
  struct S { A m; A b; };
  struct E { Raw<T, V> x, g; };
  __device__ static void load(E& e, const ScanArgs& a, int64_t o, int64_t, uint8_t, int64_t) {
    load_raw<T, V>(static_cast<const T*>(a.in0) + o, e.x);
    load_raw<T, V>(static_cast<const T*>(a.in1) + o, e.g);
  }
  // h0[i] is read here, at a sequence's first position only, rather than held with the row: a third register image per
  // row would force kRG = 4, and chunks that small cost a multiple of the time (the latency chain per chunk)
  __device__ static void lift(const E& e, const ScanArgs& a, bool act, uint8_t fl, int64_t ho, S* s) {
    A x[V], g[V];
    unpack_raw<T, V>(e.x, x);
    unpack_raw<T, V>(e.g, g);
    if (act && (fl & kStart) && a.h0) {   // act: this thread's columns exist (h0 ends at row B-1, column H-1)
      Raw<T, V> w;
      if constexpr (V == 1) w.r = __ldg(static_cast<const T*>(a.h0) + ho);
      else w.r = __ldg(reinterpret_cast<const uint4*>(static_cast<const T*>(a.h0) + ho));
      A h[V];
      unpack_raw<T, V>(w, h);
#pragma unroll
      for (int k = 0; k < V; ++k) x[k] = fma(g[k], h[k], x[k]);
    }
#pragma unroll
    for (int k = 0; k < V; ++k) s[k] = {g[k], x[k]};
  }
  __device__ static S compose(const S& p, const S& q) { return {p.m * q.m, fma(q.m, p.b, q.b)}; }
  __device__ static void emit(const ScanArgs& a, int64_t o, const E&, int64_t, bool, const S*, const S* s, uint8_t,
                              int64_t) {
    A y[V];
#pragma unroll
    for (int k = 0; k < V; ++k) y[k] = s[k].b;
    store_vec<T, V>(static_cast<T*>(a.out) + o, y);
  }
  __device__ static void pass(const ScanArgs& a, int64_t o) { copy_row<T, V>(a, o, false); }
};

template <typename T, int V_> struct OpLinRecBwd {
  static constexpr int V = V_, kRG = 8;   // three inputs held per row: one CTA per SM, but chunks of 8 rows per group
  static constexpr int kMinBlocks = 1;
  static constexpr bool kSeq = true;
  using Tp = T;
  using A = typename Store<T>::Acc;
  struct S { A m; A b; };
  struct E { Raw<T, V> g, a, h; };   // h = h_{t-1}, loaded only when grad gate is wanted
  __device__ static void load(E& e, const ScanArgs& a, int64_t o, int64_t t, uint8_t fl, int64_t ho) {
    load_raw<T, V>(static_cast<const T*>(a.in0) + o, e.g);
    load_raw<T, V>(static_cast<const T*>(a.in1) + o, e.a);
    if (!a.out_gate) return;
    if (fl & kEnd) {   // the first forward position: h_{-1} = h0[i] or 0
      if (a.h0) load_raw<T, V>(static_cast<const T*>(a.h0) + ho, e.h);
      else e.h = zero_raw<T, V>();
      return;
    }
    // the previous forward position of the same sequence; this launch runs against the forward direction
    int64_t d;
    if (a.layout == RUA_PACK) d = a.reverse ? __ldg(a.poff + t - 1) - __ldg(a.poff + t) : __ldg(a.poff + t + 1) - __ldg(a.poff + t);
    else d = a.reverse ? -1 : 1;
    load_raw<T, V>(static_cast<const T*>(a.in2) + o + d * a.H, e.h);
  }
  __device__ static void lift(const E& e, const ScanArgs&, bool, uint8_t, int64_t, S* s) {
    A g[V], m[V];
    unpack_raw<T, V>(e.g, g);
    unpack_raw<T, V>(e.a, m);
#pragma unroll
    for (int k = 0; k < V; ++k) s[k] = {m[k], m[k] * g[k]};
  }
  __device__ static S compose(const S& p, const S& q) { return {p.m * q.m, fma(q.m, p.b, q.b)}; }
  __device__ static void emit(const ScanArgs& a, int64_t o, const E& e, int64_t, bool has_before, const S* before,
                              const S* s, uint8_t fl, int64_t ho) {
    A g[V];
    unpack_raw<T, V>(e.g, g);
#pragma unroll
    for (int k = 0; k < V; ++k) g[k] = has_before ? g[k] + before[k].b : g[k];
    if (a.out) store_vec<T, V>(static_cast<T*>(a.out) + o, g);
    if (a.out_gate) {
      A h[V], r[V];
      unpack_raw<T, V>(e.h, h);
#pragma unroll
      for (int k = 0; k < V; ++k) r[k] = g[k] * h[k];
      store_vec<T, V>(static_cast<T*>(a.out_gate) + o, r);
    }
    if ((fl & kEnd) && a.out_h0) {
      A z[V];
#pragma unroll
      for (int k = 0; k < V; ++k) z[k] = s[k].b;
      store_vec<T, V>(static_cast<T*>(a.out_h0) + ho, z);
    }
  }
  __device__ static void pass(const ScanArgs& a, int64_t o) {   // grad_out passes through, the gate gets 0
    if (a.out) copy_row<T, V>(a, o, false);
    if (a.out_gate) {
      A z[V];
#pragma unroll
      for (int k = 0; k < V; ++k) z[k] = A(0);
      store_vec<T, V>(static_cast<T*>(a.out_gate) + o, z);
    }
  }
};

// ---------------------------------------------------------------------------------------------------------------------
// workspace access: bypass L1 (values are written by other CTAs)
// ---------------------------------------------------------------------------------------------------------------------
template <class S> __device__ __forceinline__ void ws_put(S* p, const S& v) {
  static_assert(sizeof(S) % 4 == 0, "state is stored as 32-bit words");
  const uint32_t* s = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
  for (int i = 0; i < (int)(sizeof(S) / 4); ++i) __stcg(reinterpret_cast<unsigned int*>(p) + i, s[i]);
}
template <class S> __device__ __forceinline__ S ws_get(const S* p) {
  S v;
  uint32_t* d = reinterpret_cast<uint32_t*>(&v);
#pragma unroll
  for (int i = 0; i < (int)(sizeof(S) / 4); ++i) d[i] = __ldcg(reinterpret_cast<const unsigned int*>(p) + i);
  return v;
}
__device__ __forceinline__ int ld_acquire(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// row decode of virtual position j: storage row, position within the sequence, flags (and with kSeq the sequence index)
template <bool kSeq>
__device__ __forceinline__ void decode_row(const ScanArgs& a, int64_t j, int64_t n_tok, int64_t lo, int64_t hi,
                                           int64_t& srow, int64_t& t, uint8_t& fl, int64_t& seq) {
  fl = 0;
  decode_position(a, j, n_tok, lo, hi, srow, t, [&](int64_t i, int64_t len) {
    const int64_t first = a.reverse ? len - 1 : 0, last = a.reverse ? 0 : len - 1;
    fl = kTok | (t == first ? kStart : 0) | (t == last ? kEnd : 0);
    if constexpr (kSeq) seq = i;
  });
}

template <class Op>
__global__ void __launch_bounds__(kScanThreads, Op::kMinBlocks) segscan_kernel(ScanArgs a) {
  using T = typename Op::Tp;
  using S = typename Op::S;
  constexpr int V = Op::V, RG = Op::kRG;
  extern __shared__ __align__(16) unsigned char smem[];
  const int R = a.R;
  int64_t* s_row = reinterpret_cast<int64_t*>(smem);
  int64_t* s_t = s_row + R;
  int64_t* s_seq = s_t + R;                                       // kSeq operators only
  S* s_buf = reinterpret_cast<S*>(s_t + (Op::kSeq ? 2 : 1) * R);  // kScanThreads x V states
  int* s_flag = reinterpret_cast<int*>(s_buf + kScanThreads * V);  // kScanThreads segment-start flags
  uint8_t* s_fl = reinterpret_cast<uint8_t*>(s_flag + kScanThreads);
  __shared__ unsigned long long s_ticket;
  __shared__ int64_t s_bounds[2];
  __shared__ int64_t s_look;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_ticket = atomicAdd(a.ticket, 1ull);
  __syncthreads();
  const int64_t c = (int64_t)(s_ticket / (unsigned)a.ncb);
  const int cb = (int)(s_ticket % (unsigned)a.ncb);
  const int64_t q0 = c * R;
  const int nq = a.rows - q0 < R ? (int)(a.rows - q0) : R;

  // ---- decode the chunk's rows ----------------------------------------------------------------------------------
  const int64_t n_tok = __ldg(a.off + a.B);
  const int64_t jlo = a.reverse ? a.rows - q0 - nq : q0;
  const int64_t jhi = a.reverse ? a.rows - 1 - q0 : q0 + nq - 1;
  int64_t lo, hi;
  owner_bounds(a, n_tok, jlo, jhi, lane, warp, s_bounds, lo, hi);
  for (int q = tid; q < nq; q += kScanThreads) {
    const int64_t j = a.reverse ? a.rows - 1 - (q0 + q) : q0 + q;
    int64_t srow, t;
    uint8_t fl;
    int64_t seq = 0;
    decode_row<Op::kSeq>(a, j, n_tok, lo, hi, srow, t, fl, seq);
    s_row[q] = srow;
    s_t[q] = t;
    s_fl[q] = fl;
    if constexpr (Op::kSeq) s_seq[q] = seq;
  }
  __syncthreads();

  // ---- pass 1: load the group's rows, segmented aggregate per group -----------------------------------------------
  const int TPC = 1 << a.tpc_log2, G = kScanThreads >> a.tpc_log2;
  const int g = tid >> a.tpc_log2, lc = tid & (TPC - 1);
  const int64_t col0 = ((int64_t)cb * TPC + lc) * V;
  const bool act = col0 < a.H;
  const int qb = g * RG;
  typename Op::E e[RG];
#pragma unroll
  for (int r = 0; r < RG; ++r) {
    const int q = qb + r;
    if (act && q < nq && (s_fl[q] & kTok)) {
      if constexpr (Op::kSeq) Op::load(e[r], a, s_row[q] * a.H + col0, s_t[q], s_fl[q], s_seq[q] * a.H + col0);
      else Op::load(e[r], a, s_row[q] * a.H + col0, s_t[q]);
    }
  }
  S s[V];
  bool started = false, have = false;
#pragma unroll
  for (int r = 0; r < RG; ++r) {
    const int q = qb + r;
    if (q < nq) {
      const uint8_t f = s_fl[q];
      if (!(f & kTok)) {
        started = true;
        have = false;
      } else {
        S l[V];
        if constexpr (Op::kSeq) Op::lift(e[r], a, act, f, s_seq[q] * a.H + col0, l);
        else Op::lift(e[r], s_t[q], l);
        if ((f & kStart) || !have) {
#pragma unroll
          for (int k = 0; k < V; ++k) s[k] = l[k];
        } else {
#pragma unroll
          for (int k = 0; k < V; ++k) s[k] = Op::compose(s[k], l[k]);
        }
        have = true;
        started |= (f & kStart) != 0;
      }
    }
  }
  // ---- combine the groups: inclusive segmented scan over g (Kogge-Stone, fixed order) -----------------------------
#pragma unroll
  for (int k = 0; k < V; ++k) s_buf[tid * V + k] = s[k];
  s_flag[tid] = started;
  for (int d = 1; d < G; d <<= 1) {
    __syncthreads();
    S p[V];
    int pf = 1;
    if (g >= d) {
      const int src = tid - d * TPC;
      pf = s_flag[src];
#pragma unroll
      for (int k = 0; k < V; ++k) p[k] = s_buf[src * V + k];
    }
    __syncthreads();
    if (g >= d && !started) {
#pragma unroll
      for (int k = 0; k < V; ++k) s[k] = Op::compose(p[k], s[k]);
      started = pf;
#pragma unroll
      for (int k = 0; k < V; ++k) s_buf[tid * V + k] = s[k];
      s_flag[tid] = started;
    }
  }
  __syncthreads();
  // this group's carry-in from the groups before it, and the whole chunk's aggregate
  S gin[V], tot[V];
  const bool gin_started = g > 0 && s_flag[tid - TPC];
  const bool tot_started = s_flag[(G - 1) * TPC + lc];
#pragma unroll
  for (int k = 0; k < V; ++k) {
    if (g > 0) gin[k] = s_buf[(tid - TPC) * V + k];
    tot[k] = s_buf[((G - 1) * TPC + lc) * V + k];
  }

  // ---- carries between chunks ---------------------------------------------------------------------------------------
  const bool need_carry = (s_fl[0] & kTok) && !(s_fl[0] & kStart);
  const bool need_publish = (s_fl[nq - 1] & kTok) && !(s_fl[nq - 1] & kEnd);
  const int cpb = TPC * V;
  const int64_t slot = (c * a.ncb + cb) * (int64_t)cpb + (int64_t)lc * V;
  S* agg = static_cast<S*>(a.agg);
  S* inc = static_cast<S*>(a.inc);
  int* flag = a.flags + c * a.ncb + cb;
  if (need_publish) {
    S* dst = tot_started ? inc : agg;
#pragma unroll
    for (int k = 0; k < V; ++k) ws_put(dst + slot + k, tot[k]);
    __threadfence();
    __syncthreads();
    if (tid == 0) st_release(flag, tot_started ? 2 : 1);
  }
  S carry[V];
  if (need_carry) {
    if (tid == 0) {
      int64_t k = c - 1;
      while (true) {
        int f;
        do { f = ld_acquire(a.flags + k * a.ncb + cb); } while (f == 0);
        if (f == 2) break;
        --k;
      }
      s_look = k;
    }
    __syncthreads();
    __threadfence();
    const int64_t k0 = s_look;
    const int64_t stride = (int64_t)a.ncb * cpb;
#pragma unroll
    for (int k = 0; k < V; ++k) carry[k] = ws_get(inc + slot - (c - k0) * stride + k);
    for (int64_t m = k0 + 1; m < c; ++m) {
#pragma unroll
      for (int k = 0; k < V; ++k) carry[k] = Op::compose(carry[k], ws_get(agg + slot - (c - m) * stride + k));
    }
    if (need_publish && !tot_started) {
#pragma unroll
      for (int k = 0; k < V; ++k) ws_put(inc + slot + k, Op::compose(carry[k], tot[k]));
      __threadfence();
      __syncthreads();
      if (tid == 0) st_release(flag, 2);
    }
#pragma unroll
    for (int k = 0; k < V; ++k) {
      if (g == 0) gin[k] = carry[k];
      else if (!gin_started) gin[k] = Op::compose(carry[k], gin[k]);
    }
  }

  // ---- pass 2: replay the held rows with the carry, store every row once --------------------------------------------
#pragma unroll
  for (int r = 0; r < RG; ++r) {
    const int q = qb + r;
    if (q < nq) {
      const uint8_t f = s_fl[q];
      const int64_t o = s_row[q] * a.H + col0;
      if (!(f & kTok)) {
        if constexpr (Op::kSeq) {
          if (act) Op::pass(a, o);
        } else {
          if (act) copy_row<T, V>(a, o, Op::kIdx);
        }
      } else {
        S l[V], before[V];
        if constexpr (Op::kSeq) Op::lift(e[r], a, act, f, s_seq[q] * a.H + col0, l);
        else Op::lift(e[r], s_t[q], l);
        const bool hb = !(f & kStart);
#pragma unroll
        for (int k = 0; k < V; ++k) {
          before[k] = gin[k];
          gin[k] = hb ? Op::compose(gin[k], l[k]) : l[k];
        }
        if constexpr (Op::kSeq) {
          if (act) Op::emit(a, o, e[r], s_t[q], hb, before, gin, f, s_seq[q] * a.H + col0);
        } else {
          if (act) Op::emit(a, o, e[r], s_t[q], hb, before, gin);
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
enum Kind { K_SUM, K_LSE, K_MAX, K_MIN, K_LSE_BWD, K_RUN_BWD, K_LINREC, K_LINREC_BWD };

struct Plan {
  int V, tpc_log2, R, ncb;
  int64_t chunks;
  size_t state_bytes, flag_bytes, total;
};

// f(Type<Op>{}) for the operator of `kind` on `dtype`, at the full 16-byte vector when `vec` allows it and H is a
// multiple of it, else one element per thread
template <typename F> int with_scan_op(Kind kind, int32_t dtype, bool vec, int64_t H, F&& f) {
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    auto at = [&](auto v) {
      constexpr int V = decltype(v)::value;
      switch (kind) {
        case K_SUM: return f(Type<OpSum<T, V>>{});
        case K_LSE: return f(Type<OpLse<T, V>>{});
        case K_MAX: return f(Type<OpExt<T, V, true>>{});
        case K_MIN: return f(Type<OpExt<T, V, false>>{});
        case K_LSE_BWD: return f(Type<OpLseBwd<T, V>>{});
        case K_LINREC: return f(Type<OpLinRec<T, V>>{});
        case K_LINREC_BWD: return f(Type<OpLinRecBwd<T, V>>{});
        default: return f(Type<OpRunBwd<T, V>>{});
      }
    };
    constexpr int VV = 16 / sizeof(T);
    if (!vec || H % VV != 0) return at(Int<1>{});
    return at(Int<VV>{});
  });
}

template <class Op> Plan make_plan(int64_t rows, int64_t H) {
  Plan p{};
  p.V = Op::V;
  const int64_t vecs = ceil_div(H, p.V);
  int tpc = 1;
  while (tpc < kMaxTPC && tpc < vecs) tpc <<= 1;
  p.tpc_log2 = __builtin_ctz(tpc);
  p.R = (kScanThreads / tpc) * Op::kRG;
  p.ncb = (int)ceil_div(vecs, tpc);
  p.chunks = ceil_div(rows, p.R);
  p.state_bytes = sizeof(typename Op::S);
  p.flag_bytes = (size_t)ceil_div(16 + 4 * p.chunks * p.ncb, 256) * 256;
  const size_t slots = (size_t)p.chunks * p.ncb * tpc * p.V;
  p.total = p.flag_bytes + 2 * slots * p.state_bytes;
  return p;
}

bool aligned16(const void* p) { return p == nullptr || ((uintptr_t)p & 15) == 0; }

template <class Op> int launch_op(const ScanArgs& a0, const Plan& p, cudaStream_t st) {
  ScanArgs a = a0;
  a.tpc_log2 = p.tpc_log2;
  a.R = p.R;
  a.ncb = p.ncb;
  const size_t smem = (size_t)p.R * (Op::kSeq ? 25 : 17) + sizeof(typename Op::S) * kScanThreads * Op::V + 4 * kScanThreads;
  if (smem > 48 * 1024) {   // narrow rows: up to 4096 positions per chunk (~72 KB)
    if (int rc = check_cuda(cudaFuncSetAttribute(segscan_kernel<Op>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)smem)))
      return rc;
  }
  const int64_t blocks = p.chunks * p.ncb;
  segscan_kernel<Op><<<(unsigned)blocks, kScanThreads, smem, st>>>(a);
  return check_launch();
}

int validate(int64_t H, int32_t dtype, const rua_ragged_t* rg, const rua_side_t* side) {
  if (H < 0 || dtype < RUA_F32 || dtype > RUA_BF16) return RUA_ERR_INVALID;
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
int validate(int64_t H, int32_t dtype, int32_t op, const rua_ragged_t* rg, const rua_side_t* side) {
  if (op < RUA_SCAN_SUM || op > RUA_SCAN_MIN) return RUA_ERR_INVALID;
  return validate(H, dtype, rg, side);
}

int run(Kind kind, int32_t dtype, int64_t H, int32_t reverse, const rua_ragged_t* rg, const rua_side_t* side,
        ScanArgs a, bool vec, void* ws, size_t ws_bytes, rua_stream_t stream) {
  const int64_t rows = side->rows;
  if (rows == 0 || H == 0) return RUA_OK;
  return with_scan_op(kind, dtype, vec, H, [&](auto op) {
    using Op = typename decltype(op)::type;
    const Plan p = make_plan<Op>(rows, H);
    if (!ws || ws_bytes < p.total) return (int)RUA_ERR_WORKSPACE;
    if (p.chunks * p.ncb > 0x7fffffffLL) return (int)RUA_ERR_UNSUPPORTED;
    a.H = H;
    a.B = rg->B;
    a.off = rg->off;
    a.poff = rg->poff;
    a.unsorted = rg->unsorted;
    a.layout = side->layout;
    a.reverse = reverse ? 1 : 0;
    a.W = side->width;
    a.rows = rows;
    unsigned char* w = static_cast<unsigned char*>(ws);
    a.ticket = reinterpret_cast<unsigned long long*>(w);
    a.flags = reinterpret_cast<int*>(w + 16);
    const size_t slots = p.total - p.flag_bytes;
    a.agg = w + p.flag_bytes;
    a.inc = w + p.flag_bytes + slots / 2;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (int rc = check_cuda(cudaMemsetAsync(ws, 0, p.flag_bytes, st))) return rc;
    return launch_op<Op>(a, p, st);
  });
}

Kind forward_kind(int32_t op) {
  return op == RUA_SCAN_SUM ? K_SUM : (op == RUA_SCAN_LOGSUMEXP ? K_LSE : (op == RUA_SCAN_MAX ? K_MAX : K_MIN));
}
Kind backward_kind(int32_t op) {
  return op == RUA_SCAN_SUM ? K_SUM : (op == RUA_SCAN_LOGSUMEXP ? K_LSE_BWD : K_RUN_BWD);
}

// the larger workspace of the two vector widths `kind` may run at
size_t workspace_bytes(Kind kind, int64_t rows, int64_t H, int32_t dtype) {
  size_t total = 0;
  for (bool vec : {true, false})
    with_scan_op(kind, dtype, vec, H, [&](auto o) {
      const size_t t = make_plan<typename decltype(o)::type>(rows, H).total;
      total = t > total ? t : total;
      return RUA_OK;
    });
  return total;
}

}  // namespace
}  // namespace rua

using namespace rua;

extern "C" size_t rua_segment_scan_workspace_bytes(int64_t rows, int64_t H, int32_t dtype, int32_t op,
                                                   int32_t backward) {
  if (rows < 0 || H < 0 || dtype < RUA_F32 || dtype > RUA_BF16 || op < RUA_SCAN_SUM || op > RUA_SCAN_MIN) return 0;
  if (rows == 0 || H == 0) return 0;
  return workspace_bytes(backward ? backward_kind(op) : forward_kind(op), rows, H, dtype);
}

extern "C" int rua_segment_scan(const void* src, void* dst, int64_t* idx_out, int64_t H, int32_t dtype, int32_t op,
                                int32_t reverse, const rua_ragged_t* ragged, const rua_side_t* side, void* ws,
                                size_t ws_bytes, rua_stream_t stream) {
  if (int rc = validate(H, dtype, op, ragged, side)) return rc;
  const bool ext = op == RUA_SCAN_MAX || op == RUA_SCAN_MIN;
  const bool empty = side->rows == 0 || H == 0;
  if (!empty && (!src || !dst || (ext && !idx_out))) return RUA_ERR_INVALID;
  if (ext && side->rows > 0x7fffffffLL) return RUA_ERR_UNSUPPORTED;   // indices are carried as int32
  ScanArgs a{};
  a.in0 = src;
  a.out = dst;
  a.idx_out = ext ? idx_out : nullptr;
  const bool vec = aligned16(src) && aligned16(dst) && aligned16(idx_out);   // idx_out is stored as longlong2 pairs
  return run(forward_kind(op), dtype, H, reverse, ragged, side, a, vec, ws, ws_bytes, stream);
}

extern "C" int rua_segment_scan_backward(const void* grad_out, const void* x, const void* y, const int64_t* idx,
                                         void* grad_in, int64_t H, int32_t dtype, int32_t op, int32_t reverse,
                                         const rua_ragged_t* ragged, const rua_side_t* side, void* ws, size_t ws_bytes,
                                         rua_stream_t stream) {
  if (int rc = validate(H, dtype, op, ragged, side)) return rc;
  const bool empty = side->rows == 0 || H == 0;
  if (!empty) {
    if (!grad_out || !grad_in) return RUA_ERR_INVALID;
    if (op == RUA_SCAN_LOGSUMEXP && (!x || !y)) return RUA_ERR_INVALID;
    if ((op == RUA_SCAN_MAX || op == RUA_SCAN_MIN) && !idx) return RUA_ERR_INVALID;
  }
  ScanArgs a{};
  a.in0 = grad_out;
  a.in1 = x;
  a.in2 = y;
  a.idx_in = idx;
  a.out = grad_in;
  const bool vec = aligned16(grad_out) && aligned16(grad_in) && aligned16(x) && aligned16(y) && aligned16(idx);
  // the gradient runs against the forward scan direction
  return run(backward_kind(op), dtype, H, !reverse, ragged, side, a, vec, ws, ws_bytes, stream);
}

extern "C" size_t rua_segment_linrec_workspace_bytes(int64_t rows, int64_t H, int32_t dtype, int32_t backward) {
  if (rows < 0 || H < 0 || dtype < RUA_F32 || dtype > RUA_BF16) return 0;
  if (rows == 0 || H == 0) return 0;
  return workspace_bytes(backward ? K_LINREC_BWD : K_LINREC, rows, H, dtype);
}

extern "C" int rua_segment_linrec(const void* x, const void* gate, const void* h0, void* dst, int64_t H, int32_t dtype,
                                  int32_t reverse, const rua_ragged_t* ragged, const rua_side_t* side, void* ws,
                                  size_t ws_bytes, rua_stream_t stream) {
  if (int rc = validate(H, dtype, ragged, side)) return rc;
  const bool empty = side->rows == 0 || H == 0;
  if (!empty && (!x || !gate || !dst)) return RUA_ERR_INVALID;
  ScanArgs a{};
  a.in0 = x;
  a.in1 = gate;
  a.h0 = h0;
  a.out = dst;
  const bool vec = aligned16(x) && aligned16(gate) && aligned16(h0) && aligned16(dst);
  return run(K_LINREC, dtype, H, reverse, ragged, side, a, vec, ws, ws_bytes, stream);
}

extern "C" int rua_segment_linrec_backward(const void* grad_out, const void* gate, const void* h0, const void* y,
                                           void* grad_x, void* grad_gate, void* grad_h0, int64_t H, int32_t dtype,
                                           int32_t reverse, const rua_ragged_t* ragged, const rua_side_t* side,
                                           void* ws, size_t ws_bytes, rua_stream_t stream) {
  if (int rc = validate(H, dtype, ragged, side)) return rc;
  const bool empty = side->rows == 0 || H == 0;
  const bool any = grad_x || grad_gate || grad_h0;
  if (!empty && any && (!grad_out || !gate || (grad_gate && !y))) return RUA_ERR_INVALID;
  if (!any || H == 0) return RUA_OK;
  if (!empty && (!ws || ws_bytes < workspace_bytes(K_LINREC_BWD, side->rows, H, dtype))) return RUA_ERR_WORKSPACE;
  // an empty sequence has no first position to write its grad h0 at
  if (grad_h0 && ragged->B > 0) {
    const size_t bytes = (size_t)ragged->B * H * (16 / vec_elems(dtype));
    if (int rc = check_cuda(cudaMemsetAsync(grad_h0, 0, bytes, static_cast<cudaStream_t>(stream)))) return rc;
  }
  ScanArgs a{};
  a.in0 = grad_out;
  a.in1 = gate;
  a.in2 = y;
  a.h0 = h0;
  a.out = grad_x;
  a.out_gate = grad_gate;
  a.out_h0 = grad_h0;
  const bool vec = aligned16(grad_out) && aligned16(gate) && aligned16(h0) && aligned16(y) && aligned16(grad_x) &&
                   aligned16(grad_gate) && aligned16(grad_h0);
  // the gradient runs against the forward scan direction
  return run(K_LINREC_BWD, dtype, H, !reverse, ragged, side, a, vec, ws, ws_bytes, stream);
}
