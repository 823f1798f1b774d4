// K12 -- per-sequence gated delta rule (Gated DeltaNet): a scalar log decay and a write strength per token and value
// head, a (K x V) state per value head, q / k shared by the value heads of a key group; forward and backward on every
// layout, with the per-chunk products on tensor cores.
//
// For token (i, t) of sequence i, value head h < H and key group c = h / (H / G):
//   S'_t = exp(g_t[h]) S_{t-1},   u_t = beta_t[h] (v_t[h] - S'_t^T k_t[c]),   S_t = S'_t + k_t[c] u_t^T
//   o_t[h] = scale S_t^T q_t[c]                                            S_{-1} = h0[i, h] (0 without one)
// (reverse: from each sequence's end.)
//
// Chunked form, chunk = Q tokens of one sequence (never crossing a sequence boundary, the last one partial); with
// cum_t = sum_{r <= t} g_r inside the chunk, gam_t = exp(cum_t), Gam_ts = exp(cum_t - cum_s), w_t = exp(cum_last - cum_t):
//   A     = strict_tril(diag(beta) (K K^T) o Gam)          T = (I + A)^-1 (column forward substitution, accumulator)
//   Z     = diag(beta) (V - diag(gam) K S_in)               V' = T Z         (= U - W S_in of the WY form)
//   O     = scale (diag(gam) Q S_in + (tril(Q K^T) o Gam) V')                 (the mask includes the diagonal)
//   S_out = exp(cum_last) S_in + K^T diag(w) V'
// Every product is a warp-tile loop over m16n8 accumulator fragments (tile_mma, chunk_mma.cuh).
//
// Forward: CTA (h, vb) of a grid (H nvb, Gs) takes V block vb of head h of the sequences of ranks g, g + Gs, ... of
// ragged->sorted.  The K x VB state block lives in the accumulator fragments of the state update for the whole sequence;
// nothing is kept for the backward.
// Backward: the unit is (sequence, key group); CTA c of a 1-D grid takes units c, c + grid, ...  Per (value head, V
// block) of the group, in that order, a forward sweep recomputes the chunk-start states into the CTA's scratch, then a
// reverse sweep carries dS in fragments chunk by chunk from the end.  grad_q / grad_k are summed over the group's heads
// and V blocks, grad_beta / grad_g over the V blocks, in that fixed order in the CTA's scratch, and each is written once.
// No atomics: bit-identical run to run and across layouts.
#include "chunk_mma.cuh"
#include "dispatch.cuh"
#include "seq_rows.cuh"

namespace rua {
namespace {

constexpr int kMaxK = 128, kMaxV = 256;
constexpr int kThr = 256, kWarps = kThr / 32;
constexpr int kBwdCtas = 2 * kNumSMs;  // backward grid: min(B G, kBwdCtas)
constexpr size_t kSmemPerSM = 227 * 1024;

// chunk length Q and V block VB: the backward's operands of one chunk must fit shared memory
// (16-bit: Q 64, VB 64; fp32: Q 32, VB 64; fp64: Q 16, VB 32)
template <typename T> constexpr int chunk_of() { return sizeof(T) == 8 ? 16 : (sizeof(T) == 4 ? 32 : 64); }
template <typename T> constexpr int vblock_of() { return sizeof(T) == 8 ? 32 : 64; }
template <typename T> constexpr int pad_of() { return 16 / (int)sizeof(T); }

struct GdnArgs {
  const void* v;       // rows x H x V
  const void* q;       // rows x G x K
  const void* k;       // rows x G x K
  const void* gl;      // rows x H, accumulator type (log decay)
  const void* beta;    // rows x H
  const void* h0;      // B x H x K x V accumulator type, or NULL
  void* o;             // rows x H x V
  void* hfin;          // B x H x K x V accumulator type, or NULL
  const void* go;      // backward: grad_out, rows x H x V
  void* gv;            // rows x H x V or NULL
  void* gq;            // rows x G x K or NULL
  void* gk;            // rows x G x K or NULL
  void* gg;            // rows x H accumulator type, or NULL
  void* gb;            // rows x H or NULL
  void* gh0;           // B x H x K x V accumulator type, or NULL
  void* scratch;       // grid x (ceil(Tmax / Q) K VB + Tmax (2K + 2)) accumulator type
  double scale;
  int64_t H;
  int G, K, V, reverse;
  int64_t B, Tmax;
  const int64_t* off;
  const int64_t* poff;
  const int64_t* sorted;
  const int64_t* unsorted;
  int32_t layout;
  int64_t Wd;
  int64_t rows;
};

__device__ __forceinline__ int64_t step_row(const GdnArgs& a, const Seq& s, int64_t p) {
  return row_of(a, s, a.reverse ? s.len - 1 - p : p);
}

// shared memory of one chunk; the backward adds its operands and per-token partial sums
template <typename T, int KB, bool kBwd> struct Smem {
  using Acc = typename Store<T>::Acc;
  static constexpr int Q = chunk_of<T>(), VB = vblock_of<T>();
  static constexpr int LDK = KB + pad_of<T>(), LDV = VB + pad_of<T>(), LDQ = Q + pad_of<T>(), LDA = Q + 16 / (int)sizeof(Acc);
  // per token: pA | pW | pB | pBb (VB / 8 each), pF | pFb (Q / 8 each), pFc (Q / 16)
  static constexpr int kPart = kBwd ? 4 * (VB / 8) + 2 * (Q / 8) + Q / 16 : 0;
  static constexpr size_t kAcc = 5 * Q + kWarps + (size_t)Q * kPart;
  static constexpr size_t kAccBytes = (kAcc * sizeof(Acc) + 15) / 16 * 16;
  // the solve's A and T (accumulator) share their bytes with the backward's dT, X, E and Ek (payload), used later
  static constexpr size_t kSolve = 2 * (size_t)Q * LDA * sizeof(Acc), kQQ4 = kBwd ? 4 * (size_t)Q * LDQ * sizeof(T) : 0;
  static constexpr size_t kShared = ((kSolve > kQQ4 ? kSolve : kQQ4) + 15) / 16 * 16;
  static constexpr size_t kT = 2 * (size_t)Q * LDK + (kBwd ? 2 : 1) * (size_t)KB * LDV + (kBwd ? 8 : 2) * (size_t)Q * LDV +
                               2 * (size_t)Q * LDQ;
  static constexpr size_t bytes() { return 8 * Q + kAccBytes + kShared + kT * sizeof(T); }

  int64_t* row;                    // Q storage rows (-1 past the chunk)
  Acc *gl, *be, *cum, *dc, *dw, *wsum;
  Acc *pA, *pW, *pB, *pBb, *pF, *pFb, *pFc;
  Acc *Af, *Tf;                    // Q x LDA
  T *dTs, *Xs, *E, *Ek;            // Q x LDQ, aliasing Af / Tf
  T *Ks, *Qs;                      // Q x LDK
  T *Hs, *DSs;                     // KB x LDV: S_in, dS
  T *Vs, *Vp, *Go, *Gg, *Zs, *Vw, *dVp, *dRs;   // Q x LDV
  T *Pm, *Tt;                      // Q x LDQ

  __device__ explicit Smem(unsigned char* base) {
    row = reinterpret_cast<int64_t*>(base);
    Acc* ac = reinterpret_cast<Acc*>(base + 8 * Q);
    gl = ac;
    be = gl + Q;
    cum = be + Q;
    dc = cum + Q;
    dw = dc + Q;
    wsum = dw + Q;
    pA = wsum + kWarps;
    pW = pA + Q * (VB / 8);
    pB = pW + Q * (VB / 8);
    pBb = pB + Q * (VB / 8);
    pF = pBb + Q * (VB / 8);
    pFb = pF + Q * (Q / 8);
    pFc = pFb + Q * (Q / 8);
    unsigned char* sh = base + 8 * Q + kAccBytes;
    Af = reinterpret_cast<Acc*>(sh);
    Tf = Af + Q * LDA;
    dTs = reinterpret_cast<T*>(sh);
    Xs = dTs + Q * LDQ;
    E = Xs + Q * LDQ;
    Ek = E + Q * LDQ;
    T* t = reinterpret_cast<T*>(sh + kShared);
    Ks = t;
    Qs = Ks + Q * LDK;
    Pm = Qs + Q * LDK;
    Tt = Pm + Q * LDQ;
    Hs = Tt + Q * LDQ;
    Vs = Hs + KB * LDV;
    Vp = Vs + Q * LDV;
    DSs = Vp + Q * LDV;
    Go = DSs + KB * LDV;
    Gg = Go + Q * LDV;
    Zs = Gg + Q * LDV;
    Vw = Zs + Q * LDV;
    dVp = Vw + Q * LDV;
    dRs = dVp + Q * LDV;
  }
};

// f(m0, n0) for the m16n8 tiles of an M x N product, spread over the warps
template <int M, int N, class F> __device__ __forceinline__ void tiles(F&& f) {
  for (int tl = threadIdx.x >> 5; tl < (M / 16) * (N / 8); tl += kWarps) f(tl / (N / 8) * 16, tl % (N / 8) * 8);
}

// dst[t][c] = src[row_t * stride + c0 + c] for c < n (0 elsewhere and past the tokens), all loads before the stores
template <typename T, int R, int C, class S>
__device__ __forceinline__ void stage_mat(T* dst, int ld, const T* src, int64_t stride, int64_t c0, int n, const S& sm) {
  constexpr int kN = R * C / kThr;
  static_assert(R * C % kThr == 0, "stage tile");
  const T zero = Store<T>::from_acc(0);
  T v[kN];
#pragma unroll
  for (int k = 0; k < kN; ++k) {
    const int e = threadIdx.x + k * kThr, t = e / C, c = e - t * C;
    const int64_t r = sm.row[t];
    v[k] = r >= 0 && c < n ? src[r * stride + c0 + c] : zero;
  }
#pragma unroll
  for (int k = 0; k < kN; ++k) {
    const int e = threadIdx.x + k * kThr, t = e / C, c = e - t * C;
    dst[t * ld + c] = v[k];
  }
}

// rows, g, beta, cum (units of log2 e for fp32) and the payload operands of chunk [p0, p0 + steps) of head h, V block vb
template <typename T, int KB, class S>
__device__ __forceinline__ void stage(const GdnArgs& a, const Seq& s, int64_t h, int64_t grp, int v0, int64_t p0,
                                      int steps, S& sm, bool with_q, const T* grad) {
  using Acc = typename S::Acc;
  constexpr int Q = S::Q, VB = S::VB;
  const int tid = threadIdx.x, lane = tid & 31;
  if (tid < Q) {
    const int64_t r = tid < steps ? step_row(a, s, p0 + tid) : -1;
    sm.row[tid] = r;
    sm.gl[tid] = r >= 0 ? static_cast<const Acc*>(a.gl)[r * a.H + h] * exp_scale<Acc>() : Acc(0);
    sm.be[tid] = r >= 0 ? Store<T>::to_acc(static_cast<const T*>(a.beta)[r * a.H + h]) : Acc(0);
  }
  __syncthreads();
  if (tid < 32) {   // lane l holds tokens 2l and 2l + 1, then an inclusive warp scan of the pair sums
    const Acc v0_ = 2 * lane < Q ? sm.gl[2 * lane] : Acc(0);
    const Acc v1 = v0_ + (2 * lane + 1 < Q ? sm.gl[2 * lane + 1] : Acc(0));
    Acc x = v1;
#pragma unroll
    for (int o = 1; o < 32; o *= 2) {
      const Acc u = __shfl_up_sync(kFullMask, x, o);
      if (lane >= o) x += u;
    }
    if (2 * lane < Q) {
      sm.cum[2 * lane] = x - v1 + v0_;
      sm.cum[2 * lane + 1] = x;
    }
  }
  const int64_t G = a.G, H = a.H;
  const int K = a.K, V = a.V, nv = V - v0 < VB ? V - v0 : VB;
  stage_mat<T, Q, KB>(sm.Ks, S::LDK, static_cast<const T*>(a.k), G * K, grp * K, K, sm);
  if (with_q) stage_mat<T, Q, KB>(sm.Qs, S::LDK, static_cast<const T*>(a.q), G * K, grp * K, K, sm);
  stage_mat<T, Q, VB>(sm.Vs, S::LDV, static_cast<const T*>(a.v), H * V, h * V + v0, nv, sm);
  if (grad) stage_mat<T, Q, VB>(sm.Go, S::LDV, grad, H * V, h * V + v0, nv, sm);
}

// Af = strict_tril(diag(beta) (K K^T) o Gam); Pm = tril(Q K^T) o Gam (with_q)
template <typename T, int KB, class S> __device__ __forceinline__ void stage_scores(S& sm, bool with_q) {
  using Acc = typename S::Acc;
  constexpr int Q = S::Q;
  const int lane = threadIdx.x & 31;
  tiles<Q, Q>([&](int m0, int n0) {
    Acc c[4] = {0, 0, 0, 0}, d[4] = {0, 0, 0, 0};
    if (n0 < m0 + 16) {
      tile_mma<T>(c, Sm<T>{sm.Ks, S::LDK, 1}, Sm<T>{sm.Ks, 1, S::LDK}, m0, n0, KB, lane);
      if (with_q) tile_mma<T>(d, Sm<T>{sm.Qs, S::LDK, 1}, Sm<T>{sm.Ks, 1, S::LDK}, m0, n0, KB, lane);
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int t = m0 + frow(e, lane), u = n0 + fcol(e, lane);
      const Acc gam = u <= t ? ex(sm.cum[t] - sm.cum[u]) : Acc(0);
      sm.Af[t * S::LDA + u] = u < t ? sm.be[t] * gam * c[e] : Acc(0);
      if (with_q) sm.Pm[t * S::LDQ + u] = Store<T>::from_acc(gam * d[e]);
    }
  });
}

// T = (I + A)^-1 by forward substitution, one column per thread, in the accumulator type; Tt = T rounded to the payload
template <typename T, class S> __device__ __forceinline__ void solve(S& sm) {
  using Acc = typename S::Acc;
  constexpr int Q = S::Q;
  const int c = threadIdx.x;
  if (c < Q) {
    for (int i = 0; i < Q; ++i) {
      Acc x0 = i == c ? Acc(1) : Acc(0), x1 = 0;
      int j = c;
      for (; j + 1 < i; j += 2) {
        x0 -= sm.Af[i * S::LDA + j] * sm.Tf[j * S::LDA + c];
        x1 -= sm.Af[i * S::LDA + j + 1] * sm.Tf[(j + 1) * S::LDA + c];
      }
      if (j < i) x0 -= sm.Af[i * S::LDA + j] * sm.Tf[j * S::LDA + c];
      const Acc x = x0 + x1;
      sm.Tf[i * S::LDA + c] = x;
      sm.Tt[i * S::LDQ + c] = Store<T>::from_acc(x);
    }
  }
}

// Zd = diag(beta) (V - diag(gam) K S_in)  (Zd may be Vs: each element is read and written by one thread)
template <typename T, int KB, class S> __device__ __forceinline__ void stage_z(S& sm, T* Zd) {
  using Acc = typename S::Acc;
  const int lane = threadIdx.x & 31;
  tiles<S::Q, S::VB>([&](int m0, int n0) {
    Acc c[4] = {0, 0, 0, 0};
    tile_mma<T>(c, Sm<T>{sm.Ks, S::LDK, 1}, Sm<T>{sm.Hs, S::LDV, 1}, m0, n0, KB, lane);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int t = m0 + frow(e, lane), v = n0 + fcol(e, lane);
      const Acc x = Store<T>::to_acc(sm.Vs[t * S::LDV + v]);
      Zd[t * S::LDV + v] = Store<T>::from_acc(sm.be[t] * (x - ex(sm.cum[t]) * c[e]));
    }
  });
}

// V' = T Z
template <typename T, class S> __device__ __forceinline__ void stage_vp(S& sm, const T* Z) {
  using Acc = typename S::Acc;
  const int lane = threadIdx.x & 31;
  tiles<S::Q, S::VB>([&](int m0, int n0) {
    Acc c[4] = {0, 0, 0, 0};
    tile_mma<T>(c, Sm<T>{sm.Tt, S::LDQ, 1}, Sm<T>{Z, S::LDV, 1}, m0, n0, S::Q, lane);
#pragma unroll
    for (int e = 0; e < 4; ++e) sm.Vp[(m0 + frow(e, lane)) * S::LDV + n0 + fcol(e, lane)] = Store<T>::from_acc(c[e]);
  });
}

// state fragment (i, e) of a warp: row k, column v of the K x VB state block
template <int VB> __device__ __forceinline__ void state_pos(int i, int e, int& k, int& v) {
  const int lane = threadIdx.x & 31, tl = (threadIdx.x >> 5) + kWarps * i;
  k = tl / (VB / 8) * 16 + frow(e, lane);
  v = tl % (VB / 8) * 8 + fcol(e, lane);
}

// st = exp(cum_last) st + K^T Vw, Vw = diag(w) V' (in place in Vp)
template <typename T, int KB, class S, typename Acc>
__device__ __forceinline__ void advance_state(Acc (&st)[KB * S::VB / 128 / kWarps][4], S& sm) {
  constexpr int Q = S::Q, VB = S::VB;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const Acc cl = sm.cum[Q - 1];
  for (int e = tid; e < Q * VB; e += kThr) {
    const int t = e / VB, v = e - t * VB;
    T* p = sm.Vp + t * S::LDV + v;
    *p = Store<T>::from_acc(Store<T>::to_acc(*p) * ex(cl - sm.cum[t]));
  }
  __syncthreads();
  const Acc dA = ex(cl);
#pragma unroll
  for (int i = 0; i < KB * VB / 128 / kWarps; ++i) {
    const int tl = warp + kWarps * i, m0 = tl / (VB / 8) * 16, n0 = tl % (VB / 8) * 8;
#pragma unroll
    for (int e = 0; e < 4; ++e) st[i][e] *= dA;
    tile_mma<T>(st[i], Sm<T>{sm.Ks, 1, S::LDK}, Sm<T>{sm.Vp, S::LDV, 1}, m0, n0, Q, lane);
  }
}

// the state block as the payload operand Hs (or DSs)
template <typename T, int KB, int VB, typename Acc>
__device__ __forceinline__ void state_to_smem(const Acc (&st)[KB * VB / 128 / kWarps][4], T* dst, int ld) {
#pragma unroll
  for (int i = 0; i < KB * VB / 128 / kWarps; ++i)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      int k, v;
      state_pos<VB>(i, e, k, v);
      dst[k * ld + v] = Store<T>::from_acc(st[i][e]);
    }
}

// state block from / to global (B x H x K x V, columns v0 ..): 0 past K and V when loading
template <int KB, int VB, typename Acc>
__device__ __forceinline__ void load_state(Acc (&st)[KB * VB / 128 / kWarps][4], const Acc* src, int K, int V, int v0) {
#pragma unroll
  for (int i = 0; i < KB * VB / 128 / kWarps; ++i)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      int k, v;
      state_pos<VB>(i, e, k, v);
      st[i][e] = src && k < K && v0 + v < V ? src[(int64_t)k * V + v0 + v] : Acc(0);
    }
}
template <int KB, int VB, typename Acc>
__device__ __forceinline__ void store_state(const Acc (&st)[KB * VB / 128 / kWarps][4], Acc* dst, int K, int V, int v0) {
#pragma unroll
  for (int i = 0; i < KB * VB / 128 / kWarps; ++i)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      int k, v;
      state_pos<VB>(i, e, k, v);
      if (k < K && v0 + v < V) dst[(int64_t)k * V + v0 + v] = st[i][e];
    }
}

// per-token rows (p0 + t) x K of the CTA's scratch: dst = c on the first (head, V block), dst + c after
template <typename Acc>
__device__ __forceinline__ void accumulate_rows(const Acc (&c)[4], Acc* dst, int m0, int n0, int64_t p0, int steps, int K,
                                                bool first) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int t = m0 + frow(e, lane), k = n0 + fcol(e, lane);
    if (t < steps && k < K) {
      Acc* p = dst + (p0 + t) * K + k;
      *p = first ? c[e] : *p + c[e];
    }
  }
}

template <typename T, int KB>
__global__ void __launch_bounds__(kThr, 1) gdn_forward_kernel(GdnArgs a) {
  using Acc = typename Store<T>::Acc;
  using S = Smem<T, KB, false>;
  constexpr int Q = S::Q, VB = S::VB, TW = KB * VB / 128 / kWarps;
  extern __shared__ __align__(16) unsigned char smem[];
  S sm(smem);
  const int tid = threadIdx.x, lane = tid & 31, K = a.K, V = a.V;
  const int64_t H = a.H, nvb = ceil_div(V, VB), h = blockIdx.x / nvb, grp = h / (H / a.G);
  const int v0 = (int)(blockIdx.x - h * nvb) * VB, nv = V - v0 < VB ? V - v0 : VB;
  const Acc scale = (Acc)a.scale;
  const T* vin = static_cast<const T*>(a.v);
  T* o = static_cast<T*>(a.o);
  auto copy_row = [&](int64_t r) {
    for (int c = tid; c < nv; c += kThr) o[(r * H + h) * V + v0 + c] = vin[(r * H + h) * V + v0 + c];
  };
  if (a.layout == RUA_CAT)   // C rows past the tokens are copied through
    for (int64_t r = __ldg(a.off + a.B) + blockIdx.y; r < a.rows; r += gridDim.y) copy_row(r);

  for (int64_t rank = blockIdx.y; rank < a.B; rank += gridDim.y) {
    const Seq s = seq_of(a, rank);
    for_padding_rows(a, s, 0, 1, copy_row);
    Acc st[TW][4];
    load_state<KB, VB>(st, a.h0 ? static_cast<const Acc*>(a.h0) + (s.i * H + h) * K * V : nullptr, K, V, v0);
    for (int64_t p0 = 0; p0 < s.len; p0 += Q) {
      const int steps = (int)(s.len - p0 < Q ? s.len - p0 : Q);
      __syncthreads();   // the previous chunk's shared data are consumed
      state_to_smem<T, KB, VB>(st, sm.Hs, S::LDV);
      stage<T, KB>(a, s, h, grp, v0, p0, steps, sm, true, nullptr);
      __syncthreads();
      stage_scores<T, KB>(sm, true);
      __syncthreads();
      solve<T>(sm);
      stage_z<T, KB>(sm, sm.Vs);
      __syncthreads();
      stage_vp<T>(sm, sm.Vs);
      __syncthreads();
      // O = scale (diag(gam) Q S_in + Pm V')
      tiles<Q, VB>([&](int m0, int n0) {
        Acc c1[4] = {0, 0, 0, 0}, c2[4] = {0, 0, 0, 0};
        tile_mma<T>(c1, Sm<T>{sm.Qs, S::LDK, 1}, Sm<T>{sm.Hs, S::LDV, 1}, m0, n0, KB, lane);
        tile_mma<T>(c2, Sm<T>{sm.Pm, S::LDQ, 1}, Sm<T>{sm.Vp, S::LDV, 1}, m0, n0, Q, lane);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int t = m0 + frow(e, lane), v = n0 + fcol(e, lane);
          if (t < steps && v < nv)
            o[(sm.row[t] * H + h) * V + v0 + v] = Store<T>::from_acc(scale * (ex(sm.cum[t]) * c1[e] + c2[e]));
        }
      });
      __syncthreads();
      advance_state<T, KB>(st, sm);
    }
    if (a.hfin) store_state<KB, VB>(st, static_cast<Acc*>(a.hfin) + (s.i * H + h) * K * V, K, V, v0);
  }
}

template <typename T, int KB>
__global__ void __launch_bounds__(kThr, 1) gdn_backward_kernel(GdnArgs a) {
  using Acc = typename Store<T>::Acc;
  using S = Smem<T, KB, true>;
  constexpr int Q = S::Q, VB = S::VB, TW = KB * VB / 128 / kWarps;
  extern __shared__ __align__(16) unsigned char smem[];
  S sm(smem);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, gr = lane >> 2, tg = lane & 3, K = a.K, V = a.V;
  const int64_t H = a.H, G = a.G, hpg = H / G, cta = blockIdx.x, rows = a.rows, nvb = ceil_div(V, VB);
  const Acc scale = (Acc)a.scale;
  const T* gout = static_cast<const T*>(a.go);
  T* gv = static_cast<T*>(a.gv);
  T* gq = static_cast<T*>(a.gq);
  T* gk = static_cast<T*>(a.gk);
  Acc* gg = static_cast<Acc*>(a.gg);
  T* gb = static_cast<T*>(a.gb);
  const bool want_qk = gq || gk, want_gb = gg || gb;
  const T zero = Store<T>::from_acc(0);
  const int64_t nch_max = ceil_div(a.Tmax, Q);
  Acc* hsc = static_cast<Acc*>(a.scratch) + cta * (nch_max * K * VB + a.Tmax * (2 * K + 2));   // chunk-start states
  Acc* dqs = hsc + nch_max * K * VB;                                                           // grad_q per token
  Acc* dks = dqs + a.Tmax * K;                                                                 // grad_k per token
  Acc* dgs = dks + a.Tmax * K;                                                                 // grad_g per token
  Acc* dbs = dgs + a.Tmax;                                                                     // grad_beta per token

  // a row that holds no token, heads [h0, h1) and groups [g0, g1): grad_v = grad_out, grad_q = grad_k = grad_g =
  // grad_beta = 0
  auto no_token = [&](int64_t r, int64_t h0, int64_t h1, int64_t g0, int64_t g1) {
    for (int64_t e = tid; e < (h1 - h0) * V; e += kThr) {
      const int64_t x = (r * H + h0) * V + e;
      if (gv) gv[x] = gout[x];
    }
    for (int64_t h = h0 + tid; h < h1; h += kThr) {
      if (gg) gg[r * H + h] = Acc(0);
      if (gb) gb[r * H + h] = zero;
    }
    for (int64_t e = tid; e < (g1 - g0) * K; e += kThr) {
      if (gq) gq[(r * G + g0) * K + e] = zero;
      if (gk) gk[(r * G + g0) * K + e] = zero;
    }
  };
  if (a.layout == RUA_CAT)
    for (int64_t r = __ldg(a.off + a.B) + cta; r < rows; r += gridDim.x) no_token(r, 0, H, 0, G);

  for (int64_t u = cta; u < a.B * G; u += gridDim.x) {
    const int64_t rank = u / G, grp = u - rank * G;
    const Seq s = seq_of(a, rank);
    if (s.len > a.Tmax) {
      // the scratch is sized by ragged->Tp, so a longer sequence cannot be processed: every gradient it reaches is
      // NaN instead (the lengths live on the device, so the host cannot return an error without a synchronisation)
      const Acc nan = quiet_nan(Acc(0));
      const T bad = Store<T>::from_acc(nan);
      for (int64_t e = tid; e < s.len * hpg * V; e += kThr) {
        const int64_t t = e / (hpg * V), x = e - t * hpg * V;
        if (gv) gv[(step_row(a, s, t) * H + grp * hpg) * V + x] = bad;
      }
      for (int64_t e = tid; e < s.len * hpg; e += kThr) {
        const int64_t t = e / hpg, x = e - t * hpg, r = step_row(a, s, t);
        if (gg) gg[r * H + grp * hpg + x] = nan;
        if (gb) gb[r * H + grp * hpg + x] = bad;
      }
      for (int64_t e = tid; e < s.len * K; e += kThr) {
        const int64_t t = e / K, x = e - t * K, r = step_row(a, s, t);
        if (gq) gq[(r * G + grp) * K + x] = bad;
        if (gk) gk[(r * G + grp) * K + x] = bad;
      }
      if (a.gh0)
        for (int64_t e = tid; e < hpg * K * V; e += kThr)
          static_cast<Acc*>(a.gh0)[(s.i * H + grp * hpg) * K * V + e] = nan;
      continue;
    }
    for_padding_rows(a, s, 0, 1, [&](int64_t r) { no_token(r, grp * hpg, (grp + 1) * hpg, grp, grp + 1); });
    const int64_t nch = ceil_div(s.len, Q);
    for (int64_t j = 0; j < hpg; ++j) {
      const int64_t h = grp * hpg + j;
      for (int vb = 0; vb < nvb; ++vb) {
        const int v0 = vb * VB, nv = V - v0 < VB ? V - v0 : VB;
        const bool first_qk = j == 0 && vb == 0, first_gb = vb == 0, last_gb = vb + 1 == nvb;
        // forward sweep: the state entering every chunk
        {
          Acc st[TW][4];
          load_state<KB, VB>(st, a.h0 ? static_cast<const Acc*>(a.h0) + (s.i * H + h) * K * V : nullptr, K, V, v0);
          for (int64_t ch = 0; ch < nch; ++ch) {
            store_state<KB, VB>(st, hsc + ch * K * VB, K, VB, 0);
            if (ch + 1 == nch) break;
            __syncthreads();
            state_to_smem<T, KB, VB>(st, sm.Hs, S::LDV);
            stage<T, KB>(a, s, h, grp, v0, ch * Q, Q, sm, false, nullptr);
            __syncthreads();
            stage_scores<T, KB>(sm, false);
            __syncthreads();
            solve<T>(sm);
            stage_z<T, KB>(sm, sm.Vs);
            __syncthreads();
            stage_vp<T>(sm, sm.Vs);
            __syncthreads();
            advance_state<T, KB>(st, sm);
          }
        }
        // reverse sweep
        Acc ds[TW][4];
#pragma unroll
        for (int i = 0; i < TW; ++i)
#pragma unroll
          for (int e = 0; e < 4; ++e) ds[i][e] = 0;
        for (int64_t ch = nch - 1; ch >= 0; --ch) {
          const int64_t p0 = ch * Q;
          const int steps = (int)(s.len - p0 < Q ? s.len - p0 : Q);
          const Acc* hin = hsc + ch * K * VB;
          __syncthreads();   // the previous chunk's shared data are consumed
          state_to_smem<T, KB, VB>(ds, sm.DSs, S::LDV);
          {
            constexpr int kH = KB * VB / kThr;
            Acc hv[kH];
#pragma unroll
            for (int x = 0; x < kH; ++x) {
              const int e = tid + x * kThr, k = e / VB;
              hv[x] = k < K ? hin[e] : Acc(0);
            }
#pragma unroll
            for (int x = 0; x < kH; ++x) {
              const int e = tid + x * kThr, k = e / VB, v = e - k * VB;
              sm.Hs[k * S::LDV + v] = Store<T>::from_acc(hv[x]);
            }
          }
          // <dS_out, S_in>: the decay term of d(cum_last)
          {
            Acc hd = 0;
#pragma unroll
            for (int i = 0; i < TW; ++i)
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                int k, v;
                state_pos<VB>(i, e, k, v);
                if (k < K) hd += ds[i][e] * hin[k * VB + v];
              }
#pragma unroll
            for (int o = 16; o >= 1; o /= 2) hd += __shfl_xor_sync(kFullMask, hd, o);
            if (lane == 0) sm.wsum[warp] = hd;
          }
          stage<T, KB>(a, s, h, grp, v0, p0, steps, sm, true, gout);
          __syncthreads();
          stage_scores<T, KB>(sm, true);
          __syncthreads();
          solve<T>(sm);
          stage_z<T, KB>(sm, sm.Zs);
          __syncthreads();
          stage_vp<T>(sm, sm.Zs);
          __syncthreads();
          const Acc cl = sm.cum[Q - 1];
          // dV' = scale Pm^T dO + diag(w) K dS; Vw = diag(w) V'; Gg = scale diag(gam) dO; the gam and w terms of dcum
          tiles<Q, VB>([&](int m0, int n0) {
            Acc c1[4] = {0, 0, 0, 0}, c2[4] = {0, 0, 0, 0}, c3[4] = {0, 0, 0, 0};
            tile_mma<T>(c1, Sm<T>{sm.Pm, 1, S::LDQ}, Sm<T>{sm.Go, S::LDV, 1}, m0, n0, Q, lane);
            tile_mma<T>(c2, Sm<T>{sm.Ks, S::LDK, 1}, Sm<T>{sm.DSs, S::LDV, 1}, m0, n0, KB, lane);
            tile_mma<T>(c3, Sm<T>{sm.Qs, S::LDK, 1}, Sm<T>{sm.Hs, S::LDV, 1}, m0, n0, KB, lane);
            Acc ra[4], rw[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int t = m0 + frow(e, lane), v = n0 + fcol(e, lane), x = t * S::LDV + v;
              const Acc w = ex(cl - sm.cum[t]), gm = ex(sm.cum[t]);
              const Acc vp = Store<T>::to_acc(sm.Vp[x]), go = scale * gm * Store<T>::to_acc(sm.Go[x]);
              sm.dVp[x] = Store<T>::from_acc(scale * c1[e] + w * c2[e]);
              sm.Vw[x] = Store<T>::from_acc(w * vp);
              sm.Gg[x] = Store<T>::from_acc(go);
              rw[e] = w * vp * c2[e];
              ra[e] = go * c3[e] - rw[e];
            }
            Acc a0 = ra[0] + ra[1], a1 = ra[2] + ra[3], w0 = rw[0] + rw[1], w1 = rw[2] + rw[3];
            row_sum8(a0, a1);
            row_sum8(w0, w1);
            if (tg == 0) {
              sm.pA[(m0 + gr) * (VB / 8) + n0 / 8] = a0;
              sm.pA[(m0 + gr + 8) * (VB / 8) + n0 / 8] = a1;
              sm.pW[(m0 + gr) * (VB / 8) + n0 / 8] = w0;
              sm.pW[(m0 + gr + 8) * (VB / 8) + n0 / 8] = w1;
            }
          });
          __syncthreads();
          // dZ = T^T dV': grad_v = diag(beta) dZ, dR = -diag(beta gam) dZ, the beta and gam terms; dT = dV' Z^T
          tiles<Q, VB>([&](int m0, int n0) {
            Acc c1[4] = {0, 0, 0, 0}, c2[4] = {0, 0, 0, 0};
            tile_mma<T>(c1, Sm<T>{sm.Tt, 1, S::LDQ}, Sm<T>{sm.dVp, S::LDV, 1}, m0, n0, Q, lane);
            tile_mma<T>(c2, Sm<T>{sm.Ks, S::LDK, 1}, Sm<T>{sm.Hs, S::LDV, 1}, m0, n0, KB, lane);
            Acc rb[4], rc[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int t = m0 + frow(e, lane), v = n0 + fcol(e, lane), x = t * S::LDV + v;
              const Acc b = sm.be[t], gm = ex(sm.cum[t]), dz = c1[e];
              if (gv && t < steps && v < nv) gv[(sm.row[t] * H + h) * V + v0 + v] = Store<T>::from_acc(b * dz);
              sm.dRs[x] = Store<T>::from_acc(-b * gm * dz);
              rb[e] = dz * (Store<T>::to_acc(sm.Vs[x]) - gm * c2[e]);
              rc[e] = -b * gm * dz * c2[e];
            }
            Acc b0 = rb[0] + rb[1], b1 = rb[2] + rb[3], c0 = rc[0] + rc[1], c1_ = rc[2] + rc[3];
            row_sum8(b0, b1);
            row_sum8(c0, c1_);
            if (tg == 0) {
              sm.pBb[(m0 + gr) * (VB / 8) + n0 / 8] = b0;
              sm.pBb[(m0 + gr + 8) * (VB / 8) + n0 / 8] = b1;
              sm.pB[(m0 + gr) * (VB / 8) + n0 / 8] = c0;
              sm.pB[(m0 + gr + 8) * (VB / 8) + n0 / 8] = c1_;
            }
          });
          tiles<Q, Q>([&](int m0, int n0) {
            Acc c[4] = {0, 0, 0, 0};
            if (n0 < m0 + 16) tile_mma<T>(c, Sm<T>{sm.dVp, S::LDV, 1}, Sm<T>{sm.Zs, 1, S::LDV}, m0, n0, VB, lane);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int t = m0 + frow(e, lane), u = n0 + fcol(e, lane);
              sm.dTs[t * S::LDQ + u] = Store<T>::from_acc(u <= t ? c[e] : Acc(0));
            }
          });
          __syncthreads();
          // X = T^T dT
          tiles<Q, Q>([&](int m0, int n0) {
            Acc c[4] = {0, 0, 0, 0};
            tile_mma<T>(c, Sm<T>{sm.Tt, 1, S::LDQ}, Sm<T>{sm.dTs, S::LDQ, 1}, m0, n0, Q, lane);
#pragma unroll
            for (int e = 0; e < 4; ++e)
              sm.Xs[(m0 + frow(e, lane)) * S::LDQ + n0 + fcol(e, lane)] = Store<T>::from_acc(c[e]);
          });
          __syncthreads();
          // dA = -strict_tril(X T^T): Ek = dA o diag(beta) Gam and its beta / cum terms; E = scale tril(dO V'^T) o Gam
          // and its cum terms
          tiles<Q, Q>([&](int m0, int n0) {
            Acc da[4] = {0, 0, 0, 0}, ckk[4] = {0, 0, 0, 0}, cqk[4] = {0, 0, 0, 0}, dp[4] = {0, 0, 0, 0};
            if (n0 < m0 + 16) {
              tile_mma<T>(da, Sm<T>{sm.Xs, S::LDQ, 1}, Sm<T>{sm.Tt, 1, S::LDQ}, m0, n0, Q, lane);
              tile_mma<T>(ckk, Sm<T>{sm.Ks, S::LDK, 1}, Sm<T>{sm.Ks, 1, S::LDK}, m0, n0, KB, lane);
              tile_mma<T>(cqk, Sm<T>{sm.Qs, S::LDK, 1}, Sm<T>{sm.Ks, 1, S::LDK}, m0, n0, KB, lane);
              tile_mma<T>(dp, Sm<T>{sm.Go, S::LDV, 1}, Sm<T>{sm.Vp, 1, S::LDV}, m0, n0, VB, lane);
            }
            Acc f[4], fb[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int t = m0 + frow(e, lane), u = n0 + fcol(e, lane);
              const Acc gam = u <= t ? ex(sm.cum[t] - sm.cum[u]) : Acc(0);
              const Acc dA = u < t ? -da[e] : Acc(0), ek = dA * sm.be[t] * gam, ee = scale * dp[e] * gam;
              sm.Ek[t * S::LDQ + u] = Store<T>::from_acc(ek);
              sm.E[t * S::LDQ + u] = Store<T>::from_acc(ee);
              f[e] = ek * ckk[e] + ee * cqk[e];
              fb[e] = dA * gam * ckk[e];
            }
            Acc r0 = f[0] + f[1], r1 = f[2] + f[3], c0 = f[0] + f[2], c1 = f[1] + f[3], b0 = fb[0] + fb[1],
                b1 = fb[2] + fb[3];
            row_sum8(r0, r1);
            row_sum8(b0, b1);
            col_sum16(c0, c1);
            if (tg == 0) {
              sm.pF[(m0 + gr) * (Q / 8) + n0 / 8] = r0;
              sm.pF[(m0 + gr + 8) * (Q / 8) + n0 / 8] = r1;
              sm.pFb[(m0 + gr) * (Q / 8) + n0 / 8] = b0;
              sm.pFb[(m0 + gr + 8) * (Q / 8) + n0 / 8] = b1;
            }
            if (gr == 0) {
              sm.pFc[(n0 + 2 * tg) * (Q / 16) + m0 / 16] = c0;
              sm.pFc[(n0 + 2 * tg + 1) * (Q / 16) + m0 / 16] = c1;
            }
          });
          __syncthreads();
          // dq = Gg S_in^T + E K, dk = dR S_in^T + Vw dS^T + E^T Q + Ek K + Ek^T K, summed in the CTA's scratch
          if (want_qk) {
            tiles<Q, KB>([&](int m0, int n0) {
              Acc c[4] = {0, 0, 0, 0};
              tile_mma<T>(c, Sm<T>{sm.Gg, S::LDV, 1}, Sm<T>{sm.Hs, 1, S::LDV}, m0, n0, VB, lane);
              tile_mma<T>(c, Sm<T>{sm.E, S::LDQ, 1}, Sm<T>{sm.Ks, S::LDK, 1}, m0, n0, Q, lane);
              accumulate_rows(c, dqs, m0, n0, p0, steps, K, first_qk);
            });
            tiles<Q, KB>([&](int m0, int n0) {
              Acc c[4] = {0, 0, 0, 0};
              tile_mma<T>(c, Sm<T>{sm.dRs, S::LDV, 1}, Sm<T>{sm.Hs, 1, S::LDV}, m0, n0, VB, lane);
              tile_mma<T>(c, Sm<T>{sm.Vw, S::LDV, 1}, Sm<T>{sm.DSs, 1, S::LDV}, m0, n0, VB, lane);
              tile_mma<T>(c, Sm<T>{sm.E, 1, S::LDQ}, Sm<T>{sm.Qs, S::LDK, 1}, m0, n0, Q, lane);
              tile_mma<T>(c, Sm<T>{sm.Ek, S::LDQ, 1}, Sm<T>{sm.Ks, S::LDK, 1}, m0, n0, Q, lane);
              tile_mma<T>(c, Sm<T>{sm.Ek, 1, S::LDQ}, Sm<T>{sm.Ks, S::LDK, 1}, m0, n0, Q, lane);
              accumulate_rows(c, dks, m0, n0, p0, steps, K, first_qk);
            });
          }
          if (tid < Q) {
            const int t = tid;
            Acc v = 0, w = 0;
#pragma unroll
            for (int x = 0; x < VB / 8; ++x) {
              v += sm.pA[t * (VB / 8) + x] + sm.pB[t * (VB / 8) + x];
              w += sm.pW[t * (VB / 8) + x];
            }
#pragma unroll
            for (int x = 0; x < Q / 8; ++x) v += sm.pF[t * (Q / 8) + x];
#pragma unroll
            for (int x = 0; x < Q / 16; ++x) v -= sm.pFc[t * (Q / 16) + x];
            sm.dc[t] = v;
            sm.dw[t] = w;
          }
          // dS_in = exp(cum_last) dS + K^T dR + Q^T Gg
          {
            const Acc dA = ex(cl);
#pragma unroll
            for (int i = 0; i < TW; ++i) {
              const int tl = warp + kWarps * i, m0 = tl / (VB / 8) * 16, n0 = tl % (VB / 8) * 8;
#pragma unroll
              for (int e = 0; e < 4; ++e) ds[i][e] *= dA;
              tile_mma<T>(ds[i], Sm<T>{sm.Ks, 1, S::LDK}, Sm<T>{sm.dRs, S::LDV, 1}, m0, n0, Q, lane);
              tile_mma<T>(ds[i], Sm<T>{sm.Qs, 1, S::LDK}, Sm<T>{sm.Gg, S::LDV, 1}, m0, n0, Q, lane);
            }
          }
          __syncthreads();
          // d(g_r) = sum_{t >= r} dcum_t, with d(cum_last) = exp(cum_last) <dS_out, S_in> + sum_t w_t dw_t at the end
          if (want_gb && tid < steps) {
            const int r = tid;
            Acc dl = 0;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) dl += sm.wsum[w];
            dl *= ex(cl);
            for (int t = 0; t < Q; ++t) dl += sm.dw[t];
            Acc d = dl;
            for (int t = Q - 1; t >= r; --t) d += sm.dc[t];
            Acc b = 0;
#pragma unroll
            for (int x = 0; x < VB / 8; ++x) b += sm.pBb[r * (VB / 8) + x];
#pragma unroll
            for (int x = 0; x < Q / 8; ++x) b += sm.pFb[r * (Q / 8) + x];
            Acc* pg = dgs + p0 + r;
            Acc* pb = dbs + p0 + r;
            if (!first_gb) {
              d += *pg;
              b += *pb;
            }
            if (last_gb) {
              const int64_t row = sm.row[r];
              if (gg) gg[row * H + h] = d;
              if (gb) gb[row * H + h] = Store<T>::from_acc(b);
            } else {
              *pg = d;
              *pb = b;
            }
          }
        }
        if (a.gh0) store_state<KB, VB>(ds, static_cast<Acc*>(a.gh0) + (s.i * H + h) * K * V, K, V, v0);
      }
    }
    if (want_qk) {   // the group's sums over its heads and V blocks, in the sequence's rows
      __syncthreads();
      for (int64_t e = tid; e < s.len * K; e += kThr) {
        const int64_t t = e / K;
        const int k = (int)(e - t * K);
        const int64_t r = step_row(a, s, t);
        if (gq) gq[(r * G + grp) * K + k] = Store<T>::from_acc(dqs[e]);
        if (gk) gk[(r * G + grp) * K + k] = Store<T>::from_acc(dks[e]);
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
bool bad_dtype(int32_t dtype) { return dtype < RUA_F32 || dtype > RUA_BF16; }
int chunk_len(int32_t dtype) { return dtype == RUA_F64 ? 16 : (dtype == RUA_F32 ? 32 : 64); }
int vblock_len(int32_t dtype) { return dtype == RUA_F64 ? 32 : 64; }
size_t esize(int32_t dtype) { return dtype == RUA_F64 ? 8 : (dtype == RUA_F32 ? 4 : 2); }

bool bad_sizes(int64_t H, int32_t G, int32_t K, int32_t V) { return H < 0 || G < 1 || K < 1 || V < 1 || H % G != 0; }

int validate(int64_t H, int32_t G, int32_t K, int32_t V, int32_t dtype, int32_t reverse, const rua_ragged_t* rg,
             const rua_side_t* side) {
  if (bad_dtype(dtype) || bad_sizes(H, G, K, V) || (reverse != 0 && reverse != 1)) return RUA_ERR_INVALID;
  if (K > kMaxK || V > kMaxV) return RUA_ERR_UNSUPPORTED;
  if (!rg || !side || rg->B < 0 || !rg->off || side->rows < 0 || side->width < 0) return RUA_ERR_INVALID;
  if (rg->B > 0 && !rg->sorted) return RUA_ERR_INVALID;
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

void fill_layout(GdnArgs& a, int64_t H, int32_t G, int32_t K, int32_t V, double scale, int32_t reverse,
                 const rua_ragged_t* rg, const rua_side_t* side) {
  a.scale = scale;
  a.H = H;
  a.G = G;
  a.K = K;
  a.V = V;
  a.reverse = reverse;
  a.B = rg->B;
  a.Tmax = rg->Tp;
  a.off = rg->off;
  a.poff = rg->poff;
  a.sorted = rg->sorted;
  a.unsorted = rg->unsorted;
  a.layout = side->layout;
  a.Wd = side->width;
  a.rows = side->rows;
}

int64_t bwd_grid(int64_t B, int64_t G) { return B * G < kBwdCtas ? B * G : kBwdCtas; }

template <typename F> int with_bucket(int32_t K, F&& f) { return K <= 64 ? f(Int<64>{}) : f(Int<128>{}); }

template <class Kern> int set_smem(Kern kern, size_t smem) {
  if (smem <= 48 * 1024) return RUA_OK;
  return check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
}

static_assert(Smem<__nv_bfloat16, 128, true>::bytes() <= kSmemPerSM, "bf16 backward shared memory");
static_assert(Smem<float, 128, true>::bytes() <= kSmemPerSM, "fp32 backward shared memory");
static_assert(Smem<double, 128, true>::bytes() <= kSmemPerSM, "fp64 backward shared memory");

}  // namespace
}  // namespace rua

using namespace rua;

extern "C" size_t rua_gdn_workspace_bytes(int64_t rows, int64_t B, int64_t Tmax, int64_t H, int32_t G, int32_t K,
                                          int32_t V, int32_t dtype) {
  if (rows < 0 || B < 0 || Tmax < 0 || bad_sizes(H, G, K, V) || K > kMaxK || V > kMaxV || bad_dtype(dtype)) return 0;
  if (rows == 0 || B == 0 || H == 0) return 0;
  const size_t grid = (size_t)bwd_grid(B, G);
  const size_t per_cta = (size_t)ceil_div(Tmax, chunk_len(dtype)) * K * vblock_len(dtype) + (size_t)Tmax * (2 * K + 2);
  return grid * per_cta * acc_bytes(dtype);
}

extern "C" int rua_gdn_forward(const void* v, const void* q, const void* k, const void* g, const void* beta,
                               const void* h0, void* o, void* h_final, int64_t H, int32_t G, int32_t K, int32_t V,
                               double scale, int32_t dtype, int32_t reverse, const rua_ragged_t* ragged,
                               const rua_side_t* side, void* ws, size_t ws_bytes, rua_stream_t stream) {
  (void)ws;
  (void)ws_bytes;
  if (int rc = validate(H, G, K, V, dtype, reverse, ragged, side)) return rc;
  const int64_t rows = side->rows, B = ragged->B;
  if (H == 0 || (rows == 0 && B == 0)) return RUA_OK;
  if (rows > 0 && (!v || !o)) return RUA_ERR_INVALID;
  if (B > 0 && rows > 0 && (!q || !k || !g || !beta)) return RUA_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (B == 0)   // C rows with no sequence at all: copied through
    return check_cuda(cudaMemcpyAsync(o, v, (size_t)rows * H * V * esize(dtype), cudaMemcpyDeviceToDevice, st));
  GdnArgs a{};
  fill_layout(a, H, G, K, V, scale, reverse, ragged, side);
  a.v = v;
  a.q = q;
  a.k = k;
  a.gl = g;
  a.beta = beta;
  a.h0 = h0;
  a.o = o;
  a.hfin = h_final;
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    return with_bucket(K, [&](auto kb) {
      constexpr int KB = decltype(kb)::value;
      constexpr size_t smem = Smem<T, KB, false>::bytes();
      auto kern = gdn_forward_kernel<T, KB>;
      if (int rc = set_smem(kern, smem)) return rc;
      // as many sequence strides gs as fit in one wave of resident CTAs: rounding gs up instead would start a second,
      // mostly idle wave whenever H nvb does not divide the resident count (at H nvb = 64: 192 CTAs on 148 SMs)
      const int64_t units = H * ceil_div(V, vblock_of<T>()), resident = kNumSMs * (int64_t)(kSmemPerSM / smem);
      const int64_t gs = resident / units > 1 ? resident / units : 1;
      kern<<<dim3((unsigned)units, (unsigned)(gs < B ? gs : B)), kThr, smem, st>>>(a);
      return check_launch();
    });
  });
}

extern "C" int rua_gdn_backward(const void* grad_out, const void* v, const void* q, const void* k, const void* g,
                                const void* beta, const void* h0, void* grad_v, void* grad_q, void* grad_k, void* grad_g,
                                void* grad_beta, void* grad_h0, int64_t H, int32_t G, int32_t K, int32_t V, double scale,
                                int32_t dtype, int32_t reverse, const rua_ragged_t* ragged, const rua_side_t* side,
                                void* ws, size_t ws_bytes, rua_stream_t stream) {
  if (int rc = validate(H, G, K, V, dtype, reverse, ragged, side)) return rc;
  if (!grad_v && !grad_q && !grad_k && !grad_g && !grad_beta && !grad_h0) return RUA_OK;
  const int64_t rows = side->rows, B = ragged->B;
  if (rows > 0 && H > 0 && !grad_out) return RUA_ERR_INVALID;
  if (rows > 0 && B > 0 && H > 0 && (!v || !q || !k || !g || !beta)) return RUA_ERR_INVALID;
  if (B > 0 && ragged->Tp < 0) return RUA_ERR_INVALID;
  const size_t need = rua_gdn_workspace_bytes(rows, B, ragged->Tp, H, G, K, V, dtype);   // 0 when there is no token
  if (need && (!ws || ws_bytes < need)) return RUA_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t esz = esize(dtype), acc = acc_bytes(dtype);
  if (rows == 0 || B == 0 || H == 0) {   // no token: grad_v passes grad_out through, every other gradient is 0
    if (grad_v && rows > 0 && H > 0)
      if (int rc = check_cuda(cudaMemcpyAsync(grad_v, grad_out, (size_t)rows * H * V * esz, cudaMemcpyDeviceToDevice, st)))
        return rc;
    const struct { void* p; size_t n; } zero[] = {{grad_q, (size_t)rows * G * K * esz}, {grad_k, (size_t)rows * G * K * esz},
                                                  {grad_g, (size_t)rows * H * acc}, {grad_beta, (size_t)rows * H * esz},
                                                  {grad_h0, (size_t)B * H * K * V * acc}};
    for (const auto& z : zero)
      if (z.p && z.n)
        if (int rc = check_cuda(cudaMemsetAsync(z.p, 0, z.n, st))) return rc;
    return RUA_OK;
  }
  GdnArgs a{};
  fill_layout(a, H, G, K, V, scale, reverse, ragged, side);
  a.v = v;
  a.q = q;
  a.k = k;
  a.gl = g;
  a.beta = beta;
  a.h0 = h0;
  a.go = grad_out;
  a.gv = grad_v;
  a.gq = grad_q;
  a.gk = grad_k;
  a.gg = grad_g;
  a.gb = grad_beta;
  a.gh0 = grad_h0;
  a.scratch = ws;
  const int64_t grid = bwd_grid(B, G);
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    return with_bucket(K, [&](auto kb) {
      constexpr int KB = decltype(kb)::value;
      constexpr size_t smem = Smem<T, KB, true>::bytes();
      auto kern = gdn_backward_kernel<T, KB>;
      if (int rc = set_smem(kern, smem)) return rc;
      kern<<<(unsigned)grid, kThr, smem, st>>>(a);
      return check_launch();
    });
  });
}
