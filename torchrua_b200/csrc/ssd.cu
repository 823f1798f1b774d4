// K11 -- per-sequence Mamba-2 (SSD) state-space scan: a scalar decay per head, a (P x N) state per head, B / C shared
// by the heads of a group; forward and backward on every layout, with the per-chunk products on tensor cores.
//
// For token (i, t) of sequence i, head h < H, head channel p < P, state n < N, group g(h) = h / (H / G):
//   dA_t      = exp(delta_t[h] A[h])
//   h_t[p, n] = dA_t h_{t-1}[p, n] + delta_t[h] x_t[h, p] B_t[g, n],     h_{-1} = h0[i, h] (0 without one)
//   y_t[h, p] = sum_n C_t[g, n] h_t[p, n]
// (reverse: from each sequence's end.)
//
// Chunked form, chunk = Q tokens of one sequence (chunks never cross a sequence boundary, the last one is partial);
// with cum_t = sum_{r <= t} delta_r A inside the chunk, u_s = delta_s x_s and w_s = exp(cum_last - cum_s):
//   M     = mask(s <= t) o exp(cum_t - cum_s) o (C B^T)                                (Q x Q)
//   y     = M u + diag(exp(cum)) C h_in^T                                             (Q x P)
//   h_out = exp(cum_last) h_in + (diag(w) u)^T B                                      (P x N)
// Every product is a warp-tile loop over m16n8 accumulator fragments (tile_mma): mma.sync m16n8k16 with fp32
// accumulation for fp16 / bf16, FMA over the same fragment ownership for fp32 / fp64.
//
// Forward: CTA (h, g) of a grid (H, Gs) takes head h of the sequences of ranks g, g + Gs, ... of ragged->sorted.  The
// state lives in the accumulator fragments of the state-update product for the whole sequence (no chunk-state tensor,
// no state-passing kernel) and nothing is kept for the backward.
// Backward: the unit is (sequence, group); CTA c of a 1-D grid takes units c, c + grid, ... (rank-major, so the groups
// of one sequence run side by side).  Per head of the group, a forward sweep recomputes the chunk-start states into the
// CTA's scratch, then a reverse sweep carries dh in fragments chunk by chunk from the end.  grad_B / grad_C are summed
// over the group's heads in head order in the CTA's scratch and written once per sequence; grad_A goes to the CTA's
// slot and slot_sum adds the slots in slot order.  No atomics: bit-identical run to run and across layouts.
#include "dispatch.cuh"
#include "chunk_mma.cuh"
#include "reduce_common.cuh"
#include "seq_rows.cuh"
#include "slot_sum.cuh"

namespace rua {
namespace {

constexpr int kMaxP = 64, kMaxN = 128;
constexpr int kPB = 64;                // P bucket (zero-padded)
constexpr int kThr = 256, kWarps = kThr / 32;
constexpr int kBwdCtas = 2 * kNumSMs;  // backward grid: min(B G, kBwdCtas)
constexpr size_t kSmemPerSM = 227 * 1024;

// chunk length: Q = 64 tokens, 16 for fp64 (whose backward operands would not fit shared memory at 64)
template <typename T> constexpr int chunk_of() { return sizeof(T) == 8 ? 16 : 64; }
// row padding of the shared matrices (16 bytes): the fragment loads of a warp hit 32 different banks
template <typename T> constexpr int pad_of() { return 16 / (int)sizeof(T); }

struct SsdArgs {
  const void* x;       // rows x H x P
  const void* dl;      // rows x H (delta)
  const void* A;       // H, accumulator type
  const void* Bm;      // rows x G x N
  const void* Cm;      // rows x G x N
  const void* h0;      // B x H x P x N accumulator type, or NULL
  void* y;             // rows x H x P
  void* hfin;          // B x H x P x N accumulator type, or NULL
  const void* g;       // backward: grad_out, rows x H x P
  void* gx;            // rows x H x P or NULL
  void* gdl;           // rows x H or NULL
  void* gB;            // rows x G x N or NULL
  void* gC;            // rows x G x N or NULL
  void* gh0;           // B x H x P x N accumulator type, or NULL
  void* ga_slots;      // grid x H accumulator type, or NULL
  void* scratch;       // grid x (ceil(Tmax / Q) P N + Tmax 2N) accumulator type
  int64_t H;
  int P, G, N, reverse;
  int64_t B, Tmax;
  const int64_t* off;
  const int64_t* poff;
  const int64_t* sorted;
  const int64_t* unsorted;
  int32_t layout;
  int64_t Wd;
  int64_t rows;
};

__device__ __forceinline__ int64_t step_row(const SsdArgs& a, const Seq& s, int64_t p) {
  return row_of(a, s, a.reverse ? s.len - 1 - p : p);
}

// shared memory of one chunk
template <typename T, int NB, bool kBwd> struct Smem {
  using Acc = typename Store<T>::Acc;
  static constexpr int Q = chunk_of<T>(), LDU = kPB + pad_of<T>(), LDN = NB + pad_of<T>(), LDQ = Q + pad_of<T>();
  static constexpr int kPartCols = Q / 8 + Q / 16 + NB / 8 + 2 * (kPB / 8);   // pR | pC | pCb | pU | pX per token
  static constexpr size_t kAcc = kBwd ? 4 * Q + kWarps + (size_t)Q * kPartCols : 2 * Q;
  static constexpr size_t kAccBytes = (kAcc * sizeof(Acc) + 15) / 16 * 16;
  static constexpr size_t kT = kBwd ? 2 * (size_t)Q * LDU + 2 * (size_t)Q * LDN + 2 * (size_t)kPB * LDN + 2 * (size_t)Q * LDQ
                                    : (size_t)Q * LDU + 2 * (size_t)Q * LDN + (size_t)kPB * LDN + (size_t)Q * LDQ;
  static constexpr size_t bytes() { return 8 * Q + kAccBytes + kT * sizeof(T); }

  int64_t* row;     // Q storage rows (-1 past the chunk)
  Acc *cum, *dl;    // Q each
  Acc *dc, *ga, *wsum, *pR, *pC, *pCb, *pU, *pX;   // backward only
  T *U, *Bs, *Cs, *M, *Hs;                          // u (Q x LDU), B, C (Q x LDN), M (Q x LDQ), h copy (P x LDN)
  T *G, *DH, *DS;                                   // backward: grad_out, dh copy, dS

  __device__ explicit Smem(unsigned char* base) {
    row = reinterpret_cast<int64_t*>(base);
    Acc* ac = reinterpret_cast<Acc*>(base + 8 * Q);
    cum = ac;
    dl = cum + Q;
    dc = dl + Q;
    ga = dc + Q;
    wsum = ga + Q;
    pR = wsum + kWarps;
    pC = pR + Q * (Q / 8);
    pCb = pC + Q * (Q / 16);
    pU = pCb + Q * (NB / 8);
    pX = pU + Q * (kPB / 8);
    T* t = reinterpret_cast<T*>(base + 8 * Q + kAccBytes);
    U = t;
    Bs = U + Q * LDU;
    Cs = Bs + Q * LDN;
    M = Cs + Q * LDN;
    Hs = M + Q * LDQ;
    G = Hs + kPB * LDN;
    DH = G + Q * LDU;
    DS = DH + kPB * LDN;
  }
};

// rows and delta of the chunk's tokens [p0, p0 + steps) of head h
template <typename T, class S>
__device__ __forceinline__ void stage_rows(const SsdArgs& a, const Seq& s, int64_t h, int64_t p0, int steps, S& sm) {
  const int t = threadIdx.x;
  if (t < S::Q) {
    const int64_t r = t < steps ? step_row(a, s, p0 + t) : -1;
    sm.row[t] = r;
    sm.dl[t] = r >= 0 ? Store<T>::to_acc(static_cast<const T*>(a.dl)[r * a.H + h]) : typename S::Acc(0);
  }
}

// after stage_rows: cum (thread 0), u = delta x rounded to T, B and C of group g, grad_out (when G is set); 0 past the
// tokens, the head channels and the states
template <typename T, int NB, class S>
__device__ __forceinline__ void stage_chunk(const SsdArgs& a, int64_t h, int64_t g, typename S::Acc a2, S& sm, bool want_c,
                                            const T* grad) {
  using Acc = typename S::Acc;
  constexpr int Q = S::Q;
  const int tid = threadIdx.x, lane = tid & 31, P = a.P, N = a.N;
  const int64_t H = a.H, G = a.G;
  if (tid < 32) {   // cum: lane l holds tokens 2l and 2l + 1, then an inclusive warp scan of the pair sums
    const Acc v0 = 2 * lane < Q ? sm.dl[2 * lane] * a2 : Acc(0);
    const Acc v1 = v0 + (2 * lane + 1 < Q ? sm.dl[2 * lane + 1] * a2 : Acc(0));
    Acc s = v1;
#pragma unroll
    for (int o = 1; o < 32; o *= 2) {
      const Acc u = __shfl_up_sync(kFullMask, s, o);
      if (lane >= o) s += u;
    }
    if (2 * lane < Q) {
      sm.cum[2 * lane] = s - v1 + v0;
      sm.cum[2 * lane + 1] = s;
    }
  }
  // every load of a thread is issued before its shared stores: the staging is latency-bound otherwise
  const T* x = static_cast<const T*>(a.x);
  const T zero = Store<T>::from_acc(0);
  constexpr int kU = Q * kPB / kThr;
  T xv[kU], gv[kU];
#pragma unroll
  for (int k = 0; k < kU; ++k) {
    const int e = tid + k * kThr, t = e / kPB, p = e - t * kPB;
    const int64_t r = sm.row[t];
    const bool on = r >= 0 && p < P;
    xv[k] = on ? x[(r * H + h) * P + p] : zero;
    gv[k] = on && grad ? grad[(r * H + h) * P + p] : zero;
  }
#pragma unroll
  for (int k = 0; k < kU; ++k) {
    const int e = tid + k * kThr, t = e / kPB, p = e - t * kPB;
    sm.U[t * S::LDU + p] = Store<T>::from_acc(sm.dl[t] * Store<T>::to_acc(xv[k]));
    if (grad) sm.G[t * S::LDU + p] = gv[k];
  }
  const T* Bm = static_cast<const T*>(a.Bm);
  const T* Cm = static_cast<const T*>(a.Cm);
  constexpr int kB = Q * NB / kThr;
  T bv[kB], cv[kB];
#pragma unroll
  for (int k = 0; k < kB; ++k) {
    const int e = tid + k * kThr, t = e / NB, n = e - t * NB;
    const int64_t r = sm.row[t];
    const bool on = r >= 0 && n < N;
    bv[k] = on ? Bm[(r * G + g) * N + n] : zero;
    cv[k] = on && want_c ? Cm[(r * G + g) * N + n] : zero;
  }
#pragma unroll
  for (int k = 0; k < kB; ++k) {
    const int e = tid + k * kThr, t = e / NB, n = e - t * NB;
    sm.Bs[t * S::LDN + n] = bv[k];
    if (want_c) sm.Cs[t * S::LDN + n] = cv[k];
  }
}

// h = exp(cum_last) h + (diag(w) u)^T B over the staged chunk; scales B by w in place (B is not read afterwards)
template <typename T, int NB, class S, typename Acc>
__device__ __forceinline__ void advance_state(Acc (&st)[NB / 16][4], S& sm) {
  constexpr int Q = S::Q;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const Acc cl = sm.cum[Q - 1];
  for (int e = tid; e < Q * NB; e += kThr) {
    const int t = e / NB, n = e - t * NB;
    T* b = sm.Bs + t * S::LDN + n;
    *b = Store<T>::from_acc(Store<T>::to_acc(*b) * ex(cl - sm.cum[t]));
  }
  __syncthreads();
  const Acc dA = ex(cl);
#pragma unroll
  for (int i = 0; i < NB / 16; ++i) {
    const int tl = warp + kWarps * i, m0 = tl / (NB / 8) * 16, n0 = tl % (NB / 8) * 8;
#pragma unroll
    for (int e = 0; e < 4; ++e) st[i][e] *= dA;
    tile_mma<T>(st[i], Sm<T>{sm.U, 1, S::LDU}, Sm<T>{sm.Bs, S::LDN, 1}, m0, n0, Q, lane);
  }
}

// state fragment (i, e) of a warp: row p, column n of the P x N state
template <int NB> __device__ __forceinline__ void state_pos(int i, int e, int& p, int& n) {
  const int lane = threadIdx.x & 31, tl = (threadIdx.x >> 5) + kWarps * i;
  p = tl / (NB / 8) * 16 + frow(e, lane);
  n = tl % (NB / 8) * 8 + fcol(e, lane);
}

template <typename T, int NB>
__global__ void __launch_bounds__(kThr, 1) ssd_forward_kernel(SsdArgs a) {
  using Acc = typename Store<T>::Acc;
  using S = Smem<T, NB, false>;
  constexpr int Q = S::Q, TW = NB / 16;
  extern __shared__ __align__(16) unsigned char smem[];
  S sm(smem);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, P = a.P, N = a.N;
  const int64_t H = a.H, h = blockIdx.x, g = h / (H / a.G);
  const T* x = static_cast<const T*>(a.x);
  T* y = static_cast<T*>(a.y);
  const Acc a2 = static_cast<const Acc*>(a.A)[h] * exp_scale<Acc>();
  auto copy_row = [&](int64_t r) {
    for (int p = tid; p < P; p += kThr) y[(r * H + h) * P + p] = x[(r * H + h) * P + p];
  };
  if (a.layout == RUA_CAT)   // C rows past the tokens are copied through
    for (int64_t r = __ldg(a.off + a.B) + blockIdx.y; r < a.rows; r += gridDim.y) copy_row(r);

  for (int64_t rank = blockIdx.y; rank < a.B; rank += gridDim.y) {
    const Seq s = seq_of(a, rank);
    for_padding_rows(a, s, 0, 1, copy_row);
    const Acc* h0 = a.h0 ? static_cast<const Acc*>(a.h0) + (s.i * H + h) * P * N : nullptr;
    Acc st[TW][4];
#pragma unroll
    for (int i = 0; i < TW; ++i)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        int p, n;
        state_pos<NB>(i, e, p, n);
        st[i][e] = h0 && p < P && n < N ? h0[p * N + n] : Acc(0);
      }
    for (int64_t p0 = 0; p0 < s.len; p0 += Q) {
      const int steps = (int)(s.len - p0 < Q ? s.len - p0 : Q);
      __syncthreads();   // the previous chunk's shared data are consumed
      stage_rows<T>(a, s, h, p0, steps, sm);
#pragma unroll
      for (int i = 0; i < TW; ++i)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          int p, n;
          state_pos<NB>(i, e, p, n);
          sm.Hs[p * S::LDN + n] = Store<T>::from_acc(st[i][e]);
        }
      __syncthreads();
      stage_chunk<T, NB>(a, h, g, a2, sm, true, nullptr);
      __syncthreads();
      // M = mask o exp(cum_t - cum_s) o C B^T
      for (int tl = warp; tl < (Q / 16) * (Q / 8); tl += kWarps) {
        const int m0 = tl / (Q / 8) * 16, n0 = tl % (Q / 8) * 8;
        Acc c[4] = {0, 0, 0, 0};
        tile_mma<T>(c, Sm<T>{sm.Cs, S::LDN, 1}, Sm<T>{sm.Bs, 1, S::LDN}, m0, n0, NB, lane);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int t = m0 + frow(e, lane), u = n0 + fcol(e, lane);
          sm.M[t * S::LDQ + u] = Store<T>::from_acc(u <= t ? ex(sm.cum[t] - sm.cum[u]) * c[e] : Acc(0));
        }
      }
      __syncthreads();
      // y = M u + diag(exp(cum)) C h_in^T
      for (int tl = warp; tl < (Q / 16) * (kPB / 8); tl += kWarps) {
        const int m0 = tl / (kPB / 8) * 16, n0 = tl % (kPB / 8) * 8;
        Acc c1[4] = {0, 0, 0, 0}, c2[4] = {0, 0, 0, 0};
        tile_mma<T>(c1, Sm<T>{sm.M, S::LDQ, 1}, Sm<T>{sm.U, S::LDU, 1}, m0, n0, Q, lane);
        tile_mma<T>(c2, Sm<T>{sm.Cs, S::LDN, 1}, Sm<T>{sm.Hs, 1, S::LDN}, m0, n0, NB, lane);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int t = m0 + frow(e, lane), p = n0 + fcol(e, lane);
          if (t < steps && p < P) y[(sm.row[t] * H + h) * P + p] = Store<T>::from_acc(c1[e] + ex(sm.cum[t]) * c2[e]);
        }
      }
      advance_state<T, NB>(st, sm);   // B is no longer read by the products above; its first loop only writes B
    }
    if (a.hfin) {
      Acc* hf = static_cast<Acc*>(a.hfin) + (s.i * H + h) * P * N;
#pragma unroll
      for (int i = 0; i < TW; ++i)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          int p, n;
          state_pos<NB>(i, e, p, n);
          if (p < P && n < N) hf[p * N + n] = st[i][e];
        }
    }
  }
}

template <typename T, int NB>
__global__ void __launch_bounds__(kThr, 1) ssd_backward_kernel(SsdArgs a) {
  using Acc = typename Store<T>::Acc;
  using S = Smem<T, NB, true>;
  constexpr int Q = S::Q, TW = NB / 16;
  extern __shared__ __align__(16) unsigned char smem[];
  S sm(smem);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, gr = lane >> 2, tg = lane & 3, P = a.P, N = a.N;
  const int64_t H = a.H, G = a.G, hpg = H / G, cta = blockIdx.x, rows = a.rows;
  const T* x = static_cast<const T*>(a.x);
  const T* gout = static_cast<const T*>(a.g);
  T* gx = static_cast<T*>(a.gx);
  T* gdl = static_cast<T*>(a.gdl);
  T* gB = static_cast<T*>(a.gB);
  T* gC = static_cast<T*>(a.gC);
  const bool want_bc = gB || gC;
  const T zero = Store<T>::from_acc(0);
  Acc* ga = a.ga_slots ? static_cast<Acc*>(a.ga_slots) + cta * H : nullptr;
  if (ga)
    for (int64_t h = tid; h < H; h += kThr) ga[h] = 0;
  const int64_t nch_max = ceil_div(a.Tmax, Q);
  Acc* hsc = static_cast<Acc*>(a.scratch) + cta * (nch_max * P * N + a.Tmax * 2 * N);   // chunk-start states
  Acc* gbc = hsc + nch_max * P * N;                                                   // [grad_B | grad_C] per token

  // a row that holds no token, heads [h0, h1) and groups [g0, g1): grad_x = grad_out, grad_delta = grad_B = grad_C = 0
  auto no_token = [&](int64_t r, int64_t h0, int64_t h1, int64_t g0, int64_t g1) {
    for (int64_t e = tid; e < (h1 - h0) * P; e += kThr) {
      const int64_t k = (r * H + h0) * P + e;
      if (gx) gx[k] = gout[k];
    }
    if (gdl)
      for (int64_t h = h0 + tid; h < h1; h += kThr) gdl[r * H + h] = zero;
    for (int64_t e = tid; e < (g1 - g0) * N; e += kThr) {
      if (gB) gB[(r * G + g0) * N + e] = zero;
      if (gC) gC[(r * G + g0) * N + e] = zero;
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
      __syncthreads();   // thread 0's earlier grad_A slot updates are done
      const T bad = Store<T>::from_acc(quiet_nan(Acc(0)));
      for (int64_t e = tid; e < s.len * hpg * P; e += kThr) {
        const int64_t t = e / (hpg * P), k = e - t * hpg * P;
        const int64_t r = step_row(a, s, t);
        if (gx) gx[(r * H + grp * hpg) * P + k] = bad;
      }
      for (int64_t e = tid; e < s.len * hpg; e += kThr) {
        const int64_t t = e / hpg, k = e - t * hpg;
        if (gdl) gdl[step_row(a, s, t) * H + grp * hpg + k] = bad;
      }
      for (int64_t e = tid; e < s.len * N; e += kThr) {
        const int64_t t = e / N, n = e - t * N;
        const int64_t r = step_row(a, s, t);
        if (gB) gB[(r * G + grp) * N + n] = bad;
        if (gC) gC[(r * G + grp) * N + n] = bad;
      }
      if (a.gh0)
        for (int64_t e = tid; e < hpg * P * N; e += kThr)
          static_cast<Acc*>(a.gh0)[(s.i * H + grp * hpg) * P * N + e] = quiet_nan(Acc(0));
      if (ga)
        for (int64_t k = tid; k < hpg; k += kThr) ga[grp * hpg + k] = quiet_nan(Acc(0));
      __syncthreads();
      continue;
    }
    for_padding_rows(a, s, 0, 1, [&](int64_t r) { no_token(r, grp * hpg, (grp + 1) * hpg, grp, grp + 1); });
    const int64_t nch = ceil_div(s.len, Q);
    for (int64_t j = 0; j < hpg; ++j) {
      const int64_t h = grp * hpg + j;
      const Acc A = static_cast<const Acc*>(a.A)[h], a2 = A * exp_scale<Acc>();
      // forward sweep: the state entering every chunk
      {
        const Acc* h0 = a.h0 ? static_cast<const Acc*>(a.h0) + (s.i * H + h) * P * N : nullptr;
        Acc st[TW][4];
#pragma unroll
        for (int i = 0; i < TW; ++i)
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            int p, n;
            state_pos<NB>(i, e, p, n);
            st[i][e] = h0 && p < P && n < N ? h0[p * N + n] : Acc(0);
          }
        for (int64_t ch = 0; ch < nch; ++ch) {
#pragma unroll
          for (int i = 0; i < TW; ++i)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              int p, n;
              state_pos<NB>(i, e, p, n);
              if (p < P && n < N) hsc[(ch * P + p) * N + n] = st[i][e];
            }
          if (ch + 1 == nch) break;
          __syncthreads();
          stage_rows<T>(a, s, h, ch * Q, Q, sm);
          __syncthreads();
          stage_chunk<T, NB>(a, h, grp, a2, sm, false, nullptr);
          __syncthreads();
          advance_state<T, NB>(st, sm);
        }
      }
      // reverse sweep
      Acc dh[TW][4];
#pragma unroll
      for (int i = 0; i < TW; ++i)
#pragma unroll
        for (int e = 0; e < 4; ++e) dh[i][e] = 0;
      for (int64_t ch = nch - 1; ch >= 0; --ch) {
        const int64_t p0 = ch * Q;
        const int steps = (int)(s.len - p0 < Q ? s.len - p0 : Q);
        __syncthreads();   // the previous chunk's shared data are consumed
        stage_rows<T>(a, s, h, p0, steps, sm);
#pragma unroll
        for (int i = 0; i < TW; ++i)
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            int p, n;
            state_pos<NB>(i, e, p, n);
            sm.DH[p * S::LDN + n] = Store<T>::from_acc(dh[i][e]);
          }
        {
          constexpr int kH = kPB * NB / kThr;
          Acc hv[kH];
#pragma unroll
          for (int k = 0; k < kH; ++k) {
            const int e = tid + k * kThr, p = e / NB, n = e - p * NB;
            hv[k] = p < P && n < N ? hsc[(ch * P + p) * N + n] : Acc(0);
          }
#pragma unroll
          for (int k = 0; k < kH; ++k) {
            const int e = tid + k * kThr, p = e / NB, n = e - p * NB;
            sm.Hs[p * S::LDN + n] = Store<T>::from_acc(hv[k]);
          }
        }
        __syncthreads();
        stage_chunk<T, NB>(a, h, grp, a2, sm, true, gout);
        __syncthreads();
        const Acc cl = sm.cum[Q - 1];
        // M, dS = dM o L with dM = g u^T; the row and column sums of dM o M
        for (int tl = warp; tl < (Q / 16) * (Q / 8); tl += kWarps) {
          const int m0 = tl / (Q / 8) * 16, n0 = tl % (Q / 8) * 8;
          Acc cs[4] = {0, 0, 0, 0}, cm[4] = {0, 0, 0, 0};
          tile_mma<T>(cs, Sm<T>{sm.Cs, S::LDN, 1}, Sm<T>{sm.Bs, 1, S::LDN}, m0, n0, NB, lane);
          tile_mma<T>(cm, Sm<T>{sm.G, S::LDU, 1}, Sm<T>{sm.U, 1, S::LDU}, m0, n0, kPB, lane);
          Acc q[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int t = m0 + frow(e, lane), v = n0 + fcol(e, lane);
            const Acc L = v <= t ? ex(sm.cum[t] - sm.cum[v]) : Acc(0), Mv = L * cs[e];
            sm.M[t * S::LDQ + v] = Store<T>::from_acc(Mv);
            sm.DS[t * S::LDQ + v] = Store<T>::from_acc(cm[e] * L);
            q[e] = cm[e] * Mv;
          }
          Acc r0 = q[0] + q[1], r1 = q[2] + q[3], c0 = q[0] + q[2], c1 = q[1] + q[3];
          row_sum8(r0, r1);
          col_sum16(c0, c1);
          if (tg == 0) {
            sm.pR[(m0 + gr) * (Q / 8) + n0 / 8] = r0;
            sm.pR[(m0 + gr + 8) * (Q / 8) + n0 / 8] = r1;
          }
          if (gr == 0) {
            sm.pC[(n0 + 2 * tg) * (Q / 16) + m0 / 16] = c0;
            sm.pC[(n0 + 2 * tg + 1) * (Q / 16) + m0 / 16] = c1;
          }
        }
        __syncthreads();
        // du = M^T g + diag(w) B dh^T: grad_x, x . du and the decay term of dcum
        for (int tl = warp; tl < (Q / 16) * (kPB / 8); tl += kWarps) {
          const int m0 = tl / (kPB / 8) * 16, n0 = tl % (kPB / 8) * 8;
          Acc c1[4] = {0, 0, 0, 0}, c2[4] = {0, 0, 0, 0};
          tile_mma<T>(c1, Sm<T>{sm.M, 1, S::LDQ}, Sm<T>{sm.G, S::LDU, 1}, m0, n0, Q, lane);
          tile_mma<T>(c2, Sm<T>{sm.Bs, S::LDN, 1}, Sm<T>{sm.DH, 1, S::LDN}, m0, n0, NB, lane);
          Acc xd[4], ud[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int t = m0 + frow(e, lane), p = n0 + fcol(e, lane);
            const int64_t r = sm.row[t];
            const Acc w = ex(cl - sm.cum[t]), du = c1[e] + w * c2[e];
            const bool on = r >= 0 && p < P;
            const Acc xv = on ? Store<T>::to_acc(x[(r * H + h) * P + p]) : Acc(0);
            if (on && gx) gx[(r * H + h) * P + p] = Store<T>::from_acc(sm.dl[t] * du);
            xd[e] = xv * du;
            ud[e] = Store<T>::to_acc(sm.U[t * S::LDU + p]) * w * c2[e];
          }
          Acc x0 = xd[0] + xd[1], x1 = xd[2] + xd[3], u0 = ud[0] + ud[1], u1 = ud[2] + ud[3];
          row_sum8(x0, x1);
          row_sum8(u0, u1);
          if (tg == 0) {
            sm.pX[(m0 + gr) * (kPB / 8) + n0 / 8] = x0;
            sm.pX[(m0 + gr + 8) * (kPB / 8) + n0 / 8] = x1;
            sm.pU[(m0 + gr) * (kPB / 8) + n0 / 8] = u0;
            sm.pU[(m0 + gr + 8) * (kPB / 8) + n0 / 8] = u1;
          }
        }
        // dC = dS B + diag(exp(cum)) g h_in, dB = dS^T C + diag(w) u dh; the inter-chunk term of dcum
        for (int tl = warp; tl < (Q / 16) * (NB / 8); tl += kWarps) {
          const int m0 = tl / (NB / 8) * 16, n0 = tl % (NB / 8) * 8;
          Acc c1[4] = {0, 0, 0, 0}, c2[4] = {0, 0, 0, 0};
          tile_mma<T>(c1, Sm<T>{sm.DS, S::LDQ, 1}, Sm<T>{sm.Bs, S::LDN, 1}, m0, n0, Q, lane);
          tile_mma<T>(c2, Sm<T>{sm.G, S::LDU, 1}, Sm<T>{sm.Hs, S::LDN, 1}, m0, n0, kPB, lane);
          Acc cb[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int t = m0 + frow(e, lane), n = n0 + fcol(e, lane);
            const Acc z = ex(sm.cum[t]) * c2[e];
            cb[e] = Store<T>::to_acc(sm.Cs[t * S::LDN + n]) * z;
            c1[e] += z;
            if (want_bc && t < steps && n < N) {
              Acc* o = gbc + (p0 + t) * 2 * N + N + n;
              *o = j ? *o + c1[e] : c1[e];
            }
          }
          Acc b0 = cb[0] + cb[1], b1 = cb[2] + cb[3];
          row_sum8(b0, b1);
          if (tg == 0) {
            sm.pCb[(m0 + gr) * (NB / 8) + n0 / 8] = b0;
            sm.pCb[(m0 + gr + 8) * (NB / 8) + n0 / 8] = b1;
          }
          if (want_bc) {
            Acc d1[4] = {0, 0, 0, 0}, d2[4] = {0, 0, 0, 0};
            tile_mma<T>(d1, Sm<T>{sm.DS, 1, S::LDQ}, Sm<T>{sm.Cs, S::LDN, 1}, m0, n0, Q, lane);
            tile_mma<T>(d2, Sm<T>{sm.U, S::LDU, 1}, Sm<T>{sm.DH, S::LDN, 1}, m0, n0, kPB, lane);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int t = m0 + frow(e, lane), n = n0 + fcol(e, lane);
              if (t < steps && n < N) {
                const Acc v = d1[e] + ex(cl - sm.cum[t]) * d2[e];
                Acc* o = gbc + (p0 + t) * 2 * N + n;
                *o = j ? *o + v : v;
              }
            }
          }
        }
        // <dh_out, h_out>: the last token's share of dcum
        {
          Acc hd = 0;
          if (ch + 1 < nch) {
#pragma unroll
            for (int i = 0; i < TW; ++i)
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                int p, n;
                state_pos<NB>(i, e, p, n);
                if (p < P && n < N) hd += dh[i][e] * hsc[((ch + 1) * P + p) * N + n];
              }
          }
#pragma unroll
          for (int o = 16; o >= 1; o /= 2) hd += __shfl_xor_sync(kFullMask, hd, o);
          if (lane == 0) sm.wsum[warp] = hd;
        }
        __syncthreads();
        if (tid < Q) {
          const int t = tid;
          Acc v = 0;
#pragma unroll
          for (int k = 0; k < Q / 8; ++k) v += sm.pR[t * (Q / 8) + k];
#pragma unroll
          for (int k = 0; k < Q / 16; ++k) v -= sm.pC[t * (Q / 16) + k];
#pragma unroll
          for (int k = 0; k < NB / 8; ++k) v += sm.pCb[t * (NB / 8) + k];
#pragma unroll
          for (int k = 0; k < kPB / 8; ++k) v -= sm.pU[t * (kPB / 8) + k];
          if (t == steps - 1)
#pragma unroll
            for (int w = 0; w < kWarps; ++w) v += sm.wsum[w];
          sm.dc[t] = v;
        }
        for (int e = tid; e < Q * NB; e += kThr) {   // C scaled by exp(cum_t) for the dh product
          const int t = e / NB, n = e - t * NB;
          T* c = sm.Cs + t * S::LDN + n;
          *c = Store<T>::from_acc(Store<T>::to_acc(*c) * ex(sm.cum[t]));
        }
        __syncthreads();
        // dh_in = exp(cum_last) dh_out + g^T diag(exp(cum)) C
        const Acc dA = ex(cl);
#pragma unroll
        for (int i = 0; i < TW; ++i) {
          const int tl = warp + kWarps * i, m0 = tl / (NB / 8) * 16, n0 = tl % (NB / 8) * 8;
#pragma unroll
          for (int e = 0; e < 4; ++e) dh[i][e] *= dA;
          tile_mma<T>(dh[i], Sm<T>{sm.G, 1, S::LDU}, Sm<T>{sm.Cs, S::LDN, 1}, m0, n0, Q, lane);
        }
        // d(delta_r A) = sum_{k >= r} dcum_k: grad_delta, grad_A
        if (tid < steps) {
          const int r = tid;
          Acc da = 0;
          for (int k = Q - 1; k >= r; --k) da += sm.dc[k];
          Acc xd = 0;
#pragma unroll
          for (int k = 0; k < kPB / 8; ++k) xd += sm.pX[r * (kPB / 8) + k];
          if (gdl) gdl[sm.row[r] * H + h] = Store<T>::from_acc(A * da + xd);
          sm.ga[r] = sm.dl[r] * da;
        }
        if (ga) {
          __syncthreads();
          if (tid == 0) {
            Acc v = ga[h];
            for (int r = 0; r < steps; ++r) v += sm.ga[r];
            ga[h] = v;
          }
        }
      }
      if (a.gh0) {
        Acc* gh = static_cast<Acc*>(a.gh0) + (s.i * H + h) * P * N;
#pragma unroll
        for (int i = 0; i < TW; ++i)
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            int p, n;
            state_pos<NB>(i, e, p, n);
            if (p < P && n < N) gh[p * N + n] = dh[i][e];
          }
      }
    }
    if (want_bc) {   // the group's sums over its heads, in the sequence's rows
      __syncthreads();
      for (int64_t e = tid; e < s.len * N; e += kThr) {
        const int64_t t = e / N;
        const int n = (int)(e - t * N);
        const int64_t r = step_row(a, s, t);
        if (gB) gB[(r * G + grp) * N + n] = Store<T>::from_acc(gbc[t * 2 * N + n]);
        if (gC) gC[(r * G + grp) * N + n] = Store<T>::from_acc(gbc[t * 2 * N + N + n]);
      }
    }
  }
}

template <typename A> struct PlainCols {
  A* out;
  __device__ A* operator()(int64_t i, int64_t& src) const {
    src = i;
    return out + i;
  }
};

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
bool bad_dtype(int32_t dtype) { return dtype < RUA_F32 || dtype > RUA_BF16; }
int chunk_len(int32_t dtype) { return dtype == RUA_F64 ? 16 : 64; }
size_t esize(int32_t dtype) { return dtype == RUA_F64 ? 8 : (dtype == RUA_F32 ? 4 : 2); }
size_t align256(size_t v) { return (v + 255) / 256 * 256; }

bool bad_sizes(int64_t H, int32_t P, int32_t G, int32_t N) { return H < 0 || P < 1 || G < 1 || N < 1 || H % G != 0; }

int validate(int64_t H, int32_t P, int32_t G, int32_t N, int32_t dtype, int32_t reverse, const rua_ragged_t* rg,
             const rua_side_t* side) {
  if (bad_dtype(dtype) || bad_sizes(H, P, G, N) || (reverse != 0 && reverse != 1)) return RUA_ERR_INVALID;
  if (P > kMaxP || N > kMaxN) return RUA_ERR_UNSUPPORTED;
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

void fill_layout(SsdArgs& a, int64_t H, int32_t P, int32_t G, int32_t N, int32_t reverse, const rua_ragged_t* rg,
                 const rua_side_t* side) {
  a.H = H;
  a.P = P;
  a.G = G;
  a.N = N;
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

template <typename F> int with_bucket(int32_t N, F&& f) { return N <= 64 ? f(Int<64>{}) : f(Int<128>{}); }

template <class K> int set_smem(K kern, size_t smem) {
  if (smem <= 48 * 1024) return RUA_OK;
  return check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
}

}  // namespace
}  // namespace rua

using namespace rua;

extern "C" size_t rua_ssd_workspace_bytes(int64_t rows, int64_t B, int64_t Tmax, int64_t H, int32_t P, int32_t G,
                                          int32_t N, int32_t dtype) {
  if (rows < 0 || B < 0 || Tmax < 0 || bad_sizes(H, P, G, N) || P > kMaxP || N > kMaxN || bad_dtype(dtype)) return 0;
  if (rows == 0 || B == 0 || H == 0) return 0;
  const size_t grid = (size_t)bwd_grid(B, G), acc = acc_bytes(dtype);
  const size_t per_cta = (size_t)ceil_div(Tmax, chunk_len(dtype)) * P * N + (size_t)Tmax * 2 * N;
  return align256(grid * H * acc) + grid * per_cta * acc;
}

extern "C" int rua_ssd_forward(const void* x, const void* delta, const void* A, const void* Bm, const void* Cm,
                               const void* h0, void* y, void* h_final, int64_t H, int32_t P, int32_t G, int32_t N,
                               int32_t dtype, int32_t reverse, const rua_ragged_t* ragged, const rua_side_t* side,
                               void* ws, size_t ws_bytes, rua_stream_t stream) {
  (void)ws;
  (void)ws_bytes;
  if (int rc = validate(H, P, G, N, dtype, reverse, ragged, side)) return rc;
  const int64_t rows = side->rows, B = ragged->B;
  if (H == 0 || (rows == 0 && B == 0)) return RUA_OK;
  if (rows > 0 && (!x || !y)) return RUA_ERR_INVALID;
  if (B > 0 && (!A || (rows > 0 && (!delta || !Bm || !Cm)))) return RUA_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (B == 0)   // C rows with no sequence at all: copied through
    return check_cuda(cudaMemcpyAsync(y, x, (size_t)rows * H * P * esize(dtype), cudaMemcpyDeviceToDevice, st));
  SsdArgs a{};
  fill_layout(a, H, P, G, N, reverse, ragged, side);
  a.x = x;
  a.dl = delta;
  a.A = A;
  a.Bm = Bm;
  a.Cm = Cm;
  a.h0 = h0;
  a.y = y;
  a.hfin = h_final;
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    return with_bucket(N, [&](auto nb) {
      constexpr int NB = decltype(nb)::value;
      constexpr size_t smem = Smem<T, NB, false>::bytes();
      auto kern = ssd_forward_kernel<T, NB>;
      if (int rc = set_smem(kern, smem)) return rc;
      const int64_t per_sm = (int64_t)(kSmemPerSM / smem), gs = ceil_div(kNumSMs * per_sm, H);
      kern<<<dim3((unsigned)H, (unsigned)(gs < B ? gs : B)), kThr, smem, st>>>(a);
      return check_launch();
    });
  });
}

extern "C" int rua_ssd_backward(const void* grad_out, const void* x, const void* delta, const void* A, const void* Bm,
                                const void* Cm, const void* h0, void* grad_x, void* grad_delta, void* grad_A,
                                void* grad_Bm, void* grad_Cm, void* grad_h0, int64_t H, int32_t P, int32_t G, int32_t N,
                                int32_t dtype, int32_t reverse, const rua_ragged_t* ragged, const rua_side_t* side,
                                void* ws, size_t ws_bytes, rua_stream_t stream) {
  if (int rc = validate(H, P, G, N, dtype, reverse, ragged, side)) return rc;
  if (!grad_x && !grad_delta && !grad_A && !grad_Bm && !grad_Cm && !grad_h0) return RUA_OK;
  const int64_t rows = side->rows, B = ragged->B;
  if (rows > 0 && H > 0 && !grad_out) return RUA_ERR_INVALID;
  if (rows > 0 && B > 0 && H > 0 && (!x || !delta || !A || !Bm || !Cm)) return RUA_ERR_INVALID;
  if (B > 0 && ragged->Tp < 0) return RUA_ERR_INVALID;
  const size_t need = rua_ssd_workspace_bytes(rows, B, ragged->Tp, H, P, G, N, dtype);   // 0 when there is no token
  if (need && (!ws || ws_bytes < need)) return RUA_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t esz = esize(dtype), acc = acc_bytes(dtype);
  if (rows == 0 || B == 0 || H == 0) {   // no token: grad_x passes grad_out through, every other gradient is 0
    if (grad_x && rows > 0 && H > 0)
      if (int rc = check_cuda(cudaMemcpyAsync(grad_x, grad_out, (size_t)rows * H * P * esz, cudaMemcpyDeviceToDevice, st)))
        return rc;
    const struct { void* p; size_t n; } zero[] = {{grad_delta, (size_t)rows * H * esz}, {grad_A, (size_t)H * acc},
                                                  {grad_Bm, (size_t)rows * G * N * esz}, {grad_Cm, (size_t)rows * G * N * esz},
                                                  {grad_h0, (size_t)B * H * P * N * acc}};
    for (const auto& z : zero)
      if (z.p && z.n)
        if (int rc = check_cuda(cudaMemsetAsync(z.p, 0, z.n, st))) return rc;
    return RUA_OK;
  }
  SsdArgs a{};
  fill_layout(a, H, P, G, N, reverse, ragged, side);
  a.x = x;
  a.dl = delta;
  a.A = A;
  a.Bm = Bm;
  a.Cm = Cm;
  a.h0 = h0;
  a.g = grad_out;
  a.gx = grad_x;
  a.gdl = grad_delta;
  a.gB = grad_Bm;
  a.gC = grad_Cm;
  a.gh0 = grad_h0;
  const int64_t grid = bwd_grid(B, G);
  const size_t sb = align256((size_t)grid * H * acc);
  a.ga_slots = grad_A ? ws : nullptr;
  a.scratch = static_cast<char*>(ws) + sb;
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    using Acc = typename Store<T>::Acc;
    return with_bucket(N, [&](auto nb) {
      constexpr int NB = decltype(nb)::value;
      constexpr size_t smem = Smem<T, NB, true>::bytes();
      auto kern = ssd_backward_kernel<T, NB>;
      if (int rc = set_smem(kern, smem)) return rc;
      kern<<<(unsigned)grid, kThr, smem, st>>>(a);
      if (int rc = check_launch()) return rc;
      if (grad_A)
        return launch_slot_sum<Acc>(static_cast<const Acc*>(a.ga_slots), grid, H, H,
                                    PlainCols<Acc>{static_cast<Acc*>(grad_A)}, st);
      return (int)RUA_OK;
    });
  });
}
