// K9 -- per-sequence linear-chain CRF: log-partition, gold-path score, their gradients, and Viterbi decode, on every
// layout.
//
// Emissions x(i, t) are rows of K tag scores; W[a, b] scores tag a at t - 1 followed by tag b at t; start / end (K,) may be
// NULL (0).  For a tag path y of sequence i (length len):
//   score(y) = start[y_0] + sum_t x(i, t)[y_t] + sum_{t>=1} W[y_{t-1}, y_t] + end[y_{len-1}]
//   log Z_i  = logsumexp over all K^len paths of score(y)
// Replaces pad (x.left(0)) -> a Python loop over T building a (B, K, K) temporary per step, which autograd keeps T of.
//
// Design (the recurrence is sequential in t and independent across sequences; compute-bound: about N K^2 exponentials):
//   * one warp per sequence, J = ceil(K / 32) tags per lane (tag b = lane + 32 j).  Warps take the sequences longest
//     first with a static assignment: warp g of a grid of G warps takes the ranks g, g + G, ... of ragged->sorted, so the
//     result never depends on timing;
//   * row t of sequence i comes from the closed-form row of its layout (C off[i] + t, L i W + t, R i W + W - len + t,
//     P poff[t] + unsorted[i]); the emission row of t + 1 is loaded while step t computes;
//   * W is staged once per CTA in shared memory in the accumulator type (W[a][b] for the forward, its transpose for the
//     backward, so that lanes read consecutive words either way);
//   * the running state is kept normalised, alpha~_t = alpha_t - c_t with max_b alpha~_t[b] = 0, and the offset c_t is
//     accumulated in fp64.  Without it alpha_t reaches 1e4 at T = 4096 and the fp32 rounding of the state alone puts
//     errors of about 0.05 into log Z.  Each column is a log-space logsumexp_a(alpha~[a] + W[a, b]) (two passes: max,
//     then sum of exp), never an exp-space product with exp(W), which underflows on -1e4 / -inf constraints;
//   * the decode is the same kernel on the max-plus semiring: the predecessor argmax (smallest index on ties) goes to a
//     uint8 backpointer per (row, tag) in the workspace, and one lane backtracks the sequence into its own rows.
// Backward (one warp per sequence again, from each sequence's end):
//   * beta~ is normalised like alpha~ (offset d_t in fp64); alpha~_t and c_t come from the state the forward saved per row;
//   * grad_x(t, b) = gZ mu_t[b] + gs [b = y_t],  mu_t[b] = exp(alpha_t[b] + beta_t[b] - log Z);
//   * xi_t[a, b] = exp(alpha_{t-1}[a] + W[a, b] + x_t[b] + beta_t[b] - log Z) = e[a, b] F[a], with e[a, b] the terms of the
//     logsumexp that gives beta_{t-1}[a] and F[a] = exp(max + alpha~_{t-1}[a] + offsets): one exponential per (a, b);
//   * every warp accumulates grad_W (and the start / end terms) in shared memory (K x K does not fit in registers at
//     K = 64), the CTA sums its warps in warp order into its own workspace slot, and slot_sum adds the slots in slot
//     order: no atomics, bit-identical run to run.  The grid is a host function of (B, K, dtype).
#include "reduce_common.cuh"
#include "seq_rows.cuh"
#include "slot_sum.cuh"

namespace rua {
namespace {

constexpr int kMaxTags = 64;
constexpr int kFwdWarps = 8;
constexpr int kBwdWarps = 4;
constexpr int kFwdCtasPerSM = 4;
constexpr int kBwdCtasPerSM = 8;
constexpr size_t kSmemPerSM = 220 * 1024;   // shared memory the CTAs of one SM may use together

struct CrfArgs {
  const void* x;          // rows x K emissions
  const int64_t* tags;    // rows, read at token rows only (forward: gold score; backward: its gradient)
  const void* W;          // K x K
  const void* start;      // K or NULL
  const void* end;        // K or NULL
  void* log_z;            // B, accumulator type
  void* score;            // B, accumulator type (forward with tags)
  void* alpha;            // state: rows x K alpha~ (accumulator type), NULL if not kept
  double* c;              // state: rows offsets c_t
  uint8_t* bp;            // decode: rows x K backpointers
  int64_t* tags_out;      // decode: rows
  const void* g_z;        // backward: B
  const void* g_s;        // backward: B or NULL
  const void* lz_in;      // backward: the forward's log Z
  void* gx;               // backward: rows x K or NULL
  void* slots;            // backward: per-CTA partial sums of [W^T | start | end], NULL if none is wanted
  int want_w;
  int K;
  int64_t B;
  const int64_t* off;
  const int64_t* poff;
  const int64_t* sorted;
  const int64_t* unsorted;
  int32_t layout;
  int64_t Wd;             // L / R width
  int64_t rows;
};

template <typename A> __device__ __forceinline__ A neg_inf() { return (A)(-INFINITY); }
__device__ __forceinline__ float fexp(float v) { return __expf(v); }
__device__ __forceinline__ double fexp(double v) { return exp(v); }
__device__ __forceinline__ float flog(float v) { return __logf(v); }
__device__ __forceinline__ double flog(double v) { return log(v); }

template <typename A> __device__ __forceinline__ A warp_max(A v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    const A w = __shfl_xor_sync(kFullMask, v, o);
    v = w > v ? w : v;
  }
  return v;
}
// butterfly sum: every lane ends with the same bits (each step adds the same two values on both lanes)
template <typename A> __device__ __forceinline__ A warp_sum(A v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
  return v;
}

template <typename T, int J>
__device__ __forceinline__ void load_row(const CrfArgs& a, int64_t row, int lane, typename Store<T>::Acc (&v)[J]) {
  const T* x = static_cast<const T*>(a.x) + row * a.K;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int b = lane + 32 * j;
    v[j] = b < a.K ? Store<T>::to_acc(x[b]) : neg_inf<typename Store<T>::Acc>();
  }
}

// subtract the warp-wide max (0 when it is -inf: every path is forbidden and the state stays -inf) and add it to c
template <typename A, int J> __device__ __forceinline__ void normalise(A (&v)[J], double& c) {
  A m = v[0];
#pragma unroll
  for (int j = 1; j < J; ++j) m = v[j] > m ? v[j] : m;
  m = warp_max(m);
  const A shift = m == neg_inf<A>() ? A(0) : m;
#pragma unroll
  for (int j = 0; j < J; ++j) v[j] -= shift;
  c += (double)m;
}

// value of tag y (valid, same on every lane) from the row held J words per lane
template <typename A, int J> __device__ __forceinline__ A pick(const A (&v)[J], int y) {
  const A w = (J == 2 && y >= 32) ? v[J - 1] : v[0];
  return __shfl_sync(kFullMask, w, y & 31);
}

template <typename T> __device__ __forceinline__ typename Store<T>::Acc opt_at(const void* p, int64_t k) {
  return p ? Store<T>::to_acc(static_cast<const T*>(p)[k]) : typename Store<T>::Acc(0);
}

// kMax = false: forward algorithm (log Z; with kTags also the gold-path score); kMax = true: Viterbi decode
template <typename T, int J, bool kMax, bool kTags>
__global__ void __launch_bounds__(kFwdWarps * 32, 2) crf_forward_kernel(CrfArgs a) {
  using A = typename Store<T>::Acc;
  extern __shared__ __align__(16) unsigned char smem[];
  const int K = a.K, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  A* sW = reinterpret_cast<A*>(smem);          // [a][b]
  A* s_al = sW + K * K + warp * K;             // this warp's alpha~, for the broadcast of a step
  for (int e = threadIdx.x; e < K * K; e += blockDim.x) sW[e] = Store<T>::to_acc(static_cast<const T*>(a.W)[e]);
  if constexpr (kMax) {   // C rows past the tokens hold no tag
    const int64_t n_tok = __ldg(a.off + a.B);
    if (a.layout == RUA_CAT)
      for (int64_t r = n_tok + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < a.rows;
           r += (int64_t)gridDim.x * blockDim.x)
        a.tags_out[r] = -1;
  }
  __syncthreads();
  const A NEG = neg_inf<A>();
  A st[J], en[J];
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int b = lane + 32 * j;
    st[j] = b < K ? opt_at<T>(a.start, b) : A(0);
    en[j] = b < K ? opt_at<T>(a.end, b) : A(0);
  }

  const int64_t G = (int64_t)gridDim.x * kFwdWarps;
  for (int64_t rank = blockIdx.x * (int64_t)kFwdWarps + warp; rank < a.B; rank += G) {
    const Seq s = seq_of(a, rank);
    if constexpr (kMax) for_padding_rows(a, s, lane, 32, [&](int64_t r) { a.tags_out[r] = -1; });
    if (s.len == 0) {
      if (lane == 0) {
        if constexpr (kMax) static_cast<A*>(a.score)[s.i] = A(0);
        else {
          static_cast<A*>(a.log_z)[s.i] = A(0);
          if constexpr (kTags) static_cast<A*>(a.score)[s.i] = A(0);
        }
      }
      continue;
    }
    int64_t rt = row_of(a, s, 0), rn = 0;
    A xc[J], xn[J], al[J];
    load_row<T, J>(a, rt, lane, xc);
#pragma unroll
    for (int j = 0; j < J; ++j) al[j] = lane + 32 * j < K ? st[j] + xc[j] : NEG;
    double c = 0;
    A sc = 0;
    bool bad = false;
    int y = 0;
    if constexpr (kTags) {
      const int64_t y0 = a.tags[rt];
      bad = y0 < 0 || y0 >= K;
      y = bad ? 0 : (int)y0;
      sc = opt_at<T>(a.start, y) + pick(xc, y);
    }
    normalise(al, c);
    auto keep = [&](int64_t r) {
      if (!a.alpha) return;
#pragma unroll
      for (int j = 0; j < J; ++j)
        if (lane + 32 * j < K) static_cast<A*>(a.alpha)[r * K + lane + 32 * j] = al[j];
      if (lane == 0) a.c[r] = c;
    };
    keep(rt);
    if (s.len > 1) {
      rn = row_of(a, s, 1);
      load_row<T, J>(a, rn, lane, xn);
    }
    for (int64_t t = 1; t < s.len; ++t) {
      rt = rn;
#pragma unroll
      for (int j = 0; j < J; ++j) xc[j] = xn[j];
      int64_t yn = 0;
      if constexpr (kTags) yn = a.tags[rt];
      if (t + 1 < s.len) {
        rn = row_of(a, s, t + 1);
        load_row<T, J>(a, rn, lane, xn);
      }
#pragma unroll
      for (int j = 0; j < J; ++j)
        if (lane + 32 * j < K) s_al[lane + 32 * j] = al[j];
      __syncwarp();
#pragma unroll
      for (int j = 0; j < J; ++j) {
        const int b = lane + 32 * j;
        if (b >= K) continue;
        if constexpr (kMax) {
          A best = NEG;
          int arg = 0;
          for (int p = 0; p < K; ++p) {
            const A v = s_al[p] + sW[p * K + b];
            if (v > best) {   // strict: the smallest predecessor wins a tie
              best = v;
              arg = p;
            }
          }
          a.bp[rt * K + b] = (uint8_t)arg;
          al[j] = best + xc[j];
        } else {
          A m = NEG;
          for (int p = 0; p < K; ++p) {
            const A v = s_al[p] + sW[p * K + b];
            m = v > m ? v : m;
          }
          if (m == NEG) {
            al[j] = NEG;
          } else {
            A sum = 0;
            for (int p = 0; p < K; ++p) sum += fexp(s_al[p] + sW[p * K + b] - m);
            al[j] = m + flog(sum) + xc[j];
          }
        }
      }
      __syncwarp();
      normalise(al, c);
      keep(rt);
      if constexpr (kTags) {
        const int yp = y;
        bad |= yn < 0 || yn >= K;
        y = bad ? 0 : (int)yn;
        sc += sW[yp * K + y] + pick(xc, y);
      }
    }

    if constexpr (kMax) {
      A v = NEG;
      int arg = 0;
#pragma unroll
      for (int j = 0; j < J; ++j) {
        const int b = lane + 32 * j;
        const A w = b < K ? al[j] + en[j] : NEG;
        if (w > v) {
          v = w;
          arg = b;
        }
      }
#pragma unroll
      for (int o = 16; o; o >>= 1) {   // max, smallest tag on a tie: the same on every lane
        const A ov = __shfl_xor_sync(kFullMask, v, o);
        const int oa = __shfl_xor_sync(kFullMask, arg, o);
        if (ov > v || (ov == v && oa < arg)) {
          v = ov;
          arg = oa;
        }
      }
      __syncwarp();   // the backpointers of every lane are visible to lane 0
      if (lane == 0) {
        static_cast<A*>(a.score)[s.i] = (A)(c + (double)v);
        int yb = arg;
        for (int64_t t = s.len - 1; t >= 0; --t) {
          const int64_t r = row_of(a, s, t);
          a.tags_out[r] = yb;
          if (t > 0) yb = a.bp[r * K + yb];
        }
      }
    } else {
      A m = NEG;
#pragma unroll
      for (int j = 0; j < J; ++j) {
        al[j] += en[j];
        m = al[j] > m ? al[j] : m;
      }
      m = warp_max(m);
      A sum = 0;
      if (m != NEG) {
#pragma unroll
        for (int j = 0; j < J; ++j) sum += fexp(al[j] - m);
      }
      sum = warp_sum(sum);
      if (lane == 0) {
        const A lz = m == NEG ? NEG : (A)(c + (double)m + (double)flog(sum));
        static_cast<A*>(a.log_z)[s.i] = lz;
        if constexpr (kTags) {
          const A q = sc + opt_at<T>(a.end, y);
          static_cast<A*>(a.score)[s.i] = bad ? (A)NAN : q;
        }
      }
    }
  }
}

template <typename T, int J>
__global__ void __launch_bounds__(kBwdWarps * 32, 4) crf_backward_kernel(CrfArgs a) {
  using A = typename Store<T>::Acc;
  extern __shared__ __align__(16) unsigned char smem[];
  const int K = a.K, KK = K * K, nacc = KK + 2 * K, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  A* sWT = reinterpret_cast<A*>(smem);          // [b][a] = W[a][b]
  A* acc = sWT + KK + warp * (nacc + K);        // this warp's sums: [b][a] transitions, start[K], end[K]
  A* s_u = acc + nacc;                          // [K] x_t[b] + beta~_t[b] of the current step
  for (int e = threadIdx.x; e < KK; e += blockDim.x) {
    const int p = e / K, q = e - p * K;
    sWT[q * K + p] = Store<T>::to_acc(static_cast<const T*>(a.W)[e]);
  }
  for (int e = threadIdx.x; e < kBwdWarps * (nacc + K); e += blockDim.x) sWT[KK + e] = A(0);
  T* gx = static_cast<T*>(a.gx);
  const T zero = Store<T>::from_acc(0);
  if (gx && a.layout == RUA_CAT) {   // C rows past the tokens
    const int64_t n_tok = __ldg(a.off + a.B);
    for (int64_t e = n_tok * K + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < a.rows * K;
         e += (int64_t)gridDim.x * blockDim.x)
      gx[e] = zero;
  }
  __syncthreads();
  const A NEG = neg_inf<A>();
  A en[J];
#pragma unroll
  for (int j = 0; j < J; ++j) en[j] = lane + 32 * j < K ? opt_at<T>(a.end, lane + 32 * j) : A(0);
  const A* alpha = static_cast<const A*>(a.alpha);
  const bool gold = a.g_s && a.tags;
  auto tag_at = [&](int64_t r) -> int {
    if (!gold) return -1;
    const int64_t y = a.tags[r];
    return y >= 0 && y < K ? (int)y : -1;
  };
  auto load_alpha = [&](int64_t r, A (&v)[J]) {
#pragma unroll
    for (int j = 0; j < J; ++j) v[j] = lane + 32 * j < K ? alpha[r * K + lane + 32 * j] : NEG;
  };

  const int64_t G = (int64_t)gridDim.x * kBwdWarps;
  for (int64_t rank = blockIdx.x * (int64_t)kBwdWarps + warp; rank < a.B; rank += G) {
    const Seq s = seq_of(a, rank);
    if (gx) for_padding_rows(a, s, lane, 32, [&](int64_t r) {
      for (int b = 0; b < K; ++b) gx[r * K + b] = zero;
    });
    if (s.len == 0) continue;
    const A gz = static_cast<const A*>(a.g_z)[s.i];
    const A gs = a.g_s ? static_cast<const A*>(a.g_s)[s.i] : A(0);
    const A lz = static_cast<const A*>(a.lz_in)[s.i];
    if (!(lz > NEG) || (gz == A(0) && gs == A(0))) {   // log Z = -inf (or nothing to propagate): zero gradient
      if (gx)
        for (int64_t e = lane; e < s.len * K; e += 32) {
          const int64_t t = e / K;
          gx[row_of(a, s, t) * K + (e - t * K)] = zero;
        }
      continue;
    }
    int64_t rt = row_of(a, s, s.len - 1);
    A xc[J], be[J], alc[J];
    load_row<T, J>(a, rt, lane, xc);
    load_alpha(rt, alc);
    double ct = a.c[rt];
    int y = tag_at(rt);
#pragma unroll
    for (int j = 0; j < J; ++j) be[j] = lane + 32 * j < K ? en[j] : NEG;
    double d = 0;
    normalise(be, d);
    for (int64_t t = s.len - 1;; --t) {
      int64_t rp = 0;
      A xp[J], alp[J];
      double cp = 0;
      int yp = -1;
      if (t > 0) {   // the row of t - 1, loaded while step t computes
        rp = row_of(a, s, t - 1);
        load_row<T, J>(a, rp, lane, xp);
        load_alpha(rp, alp);
        cp = a.c[rp];
        yp = tag_at(rp);
      }
      const A kmu = (A)(ct + d - (double)lz);
#pragma unroll
      for (int j = 0; j < J; ++j) {
        const int b = lane + 32 * j;
        if (b >= K) continue;
        const A g = gz * fexp(alc[j] + be[j] + kmu) + (b == y ? gs : A(0));
        if (gx) gx[rt * K + b] = Store<T>::from_acc(g);
        if (t == s.len - 1) acc[KK + K + b] += g;
        if (t == 0) acc[KK + b] += g;
      }
      if (t == 0) break;
#pragma unroll
      for (int j = 0; j < J; ++j)
        if (lane + 32 * j < K) s_u[lane + 32 * j] = xc[j] + be[j];
      __syncwarp();
      const A kxi = (A)(cp + d - (double)lz);
      A nb[J];
#pragma unroll
      for (int j = 0; j < J; ++j) {
        const int p = lane + 32 * j;   // this lane's tag at t - 1
        nb[j] = NEG;
        if (p >= K) continue;
        A m = NEG;
        for (int q = 0; q < K; ++q) {
          const A v = sWT[q * K + p] + s_u[q];
          m = v > m ? v : m;
        }
        if (m == NEG) continue;
        const A F = a.want_w ? gz * fexp(m + alp[j] + kxi) : A(0);
        A sum = 0;
        for (int q = 0; q < K; ++q) {
          const A e = fexp(sWT[q * K + p] + s_u[q] - m);
          sum += e;
          if (a.want_w) acc[q * K + p] += e * F;
        }
        nb[j] = m + flog(sum);
      }
      if (a.want_w && y >= 0 && yp >= 0 && lane == (yp & 31)) acc[y * K + yp] += gs;
      __syncwarp();
      normalise(nb, d);
#pragma unroll
      for (int j = 0; j < J; ++j) {
        be[j] = nb[j];
        xc[j] = xp[j];
        alc[j] = alp[j];
      }
      rt = rp;
      ct = cp;
      y = yp;
    }
  }

  if (!a.slots) return;
  __syncthreads();
  A* slot = static_cast<A*>(a.slots) + (int64_t)blockIdx.x * nacc;   // [a][b] transitions, start[K], end[K]
  for (int e = threadIdx.x; e < nacc; e += blockDim.x) {
    A v = 0;
    for (int w = 0; w < kBwdWarps; ++w) v += sWT[KK + w * (nacc + K) + e];
    int dst = e;
    if (e < KK) {
      const int q = e / K;
      dst = (e - q * K) * K + q;
    }
    __stcg(slot + dst, v);
  }
}

// columns of the slot sum: [W (K x K) | start | end]
template <typename T> struct CrfCols {
  T* gw;
  T* gs;
  T* ge;
  int K;
  __device__ T* operator()(int64_t i, int64_t& src) const {
    src = i;
    const int64_t KK = (int64_t)K * K;
    if (i < KK) return gw ? gw + i : nullptr;
    if (i < KK + K) return gs ? gs + (i - KK) : nullptr;
    return ge ? ge + (i - KK - K) : nullptr;
  }
};

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
size_t fwd_smem(int K, size_t acc) { return ((size_t)K * K + (size_t)kFwdWarps * K) * acc; }
size_t bwd_smem(int K, size_t acc) { return ((size_t)K * K + (size_t)kBwdWarps * ((size_t)K * K + 3 * K)) * acc; }
int64_t ctas_per_sm(size_t smem, int cap) {
  const int64_t n = (int64_t)(kSmemPerSM / smem);
  return n < 1 ? 1 : (n > cap ? cap : n);
}
int64_t bwd_max_slots(int K, size_t acc) { return kNumSMs * ctas_per_sm(bwd_smem(K, acc), kBwdCtasPerSM); }
int64_t grid_of(int64_t B, int warps, int64_t cap) {
  const int64_t n = ceil_div(B, warps);
  return n < cap ? n : cap;
}

bool bad_dtype(int32_t dtype) { return dtype < RUA_F32 || dtype > RUA_BF16; }

int validate(int32_t K, int32_t dtype, const rua_ragged_t* rg, const rua_side_t* side) {
  if (bad_dtype(dtype) || K < 1) return RUA_ERR_INVALID;
  if (K > kMaxTags) return RUA_ERR_UNSUPPORTED;
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

void fill_layout(CrfArgs& a, int32_t K, const rua_ragged_t* rg, const rua_side_t* side) {
  a.K = K;
  a.B = rg->B;
  a.off = rg->off;
  a.poff = rg->poff;
  a.sorted = rg->sorted;
  a.unsorted = rg->unsorted;
  a.layout = side->layout;
  a.Wd = side->width;
  a.rows = side->rows;
}

template <typename Kern> int launch(Kern kern, int64_t grid, int threads, size_t smem, cudaStream_t st, const CrfArgs& a) {
  if (smem > 48 * 1024) {
    if (int rc = check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem))) return rc;
  }
  kern<<<(unsigned)grid, threads, smem, st>>>(a);
  return check_launch();
}

// kMode: 0 log Z, 1 log Z + gold score, 2 decode
template <int kMode> int run_forward(int32_t dtype, const CrfArgs& a, cudaStream_t st) {
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    const size_t smem = fwd_smem(a.K, sizeof(typename Store<T>::Acc));
    const int64_t grid = grid_of(a.B, kFwdWarps, kNumSMs * ctas_per_sm(smem, kFwdCtasPerSM));
    auto go = [&](auto j) {
      constexpr int J = decltype(j)::value;
      return launch(crf_forward_kernel<T, J, kMode == 2, kMode == 1>, grid, kFwdWarps * 32, smem, st, a);
    };
    return a.K > 32 ? go(Int<2>{}) : go(Int<1>{});
  });
}

}  // namespace
}  // namespace rua

using namespace rua;

extern "C" size_t rua_crf_workspace_bytes(int64_t rows, int32_t K, int32_t dtype, int32_t mode) {
  if (rows <= 0 || K < 1 || K > kMaxTags || bad_dtype(dtype)) return 0;
  switch (mode) {
    case RUA_CRF_BACKWARD: return (size_t)bwd_max_slots(K, acc_bytes(dtype)) * ((size_t)K * K + 2 * K) * acc_bytes(dtype);
    case RUA_CRF_DECODE: return (size_t)rows * K;
    default: return 0;
  }
}

extern "C" size_t rua_crf_state_bytes(int64_t rows, int32_t K, int32_t dtype) {
  if (rows <= 0 || K < 1 || K > kMaxTags || bad_dtype(dtype)) return 0;
  return ((size_t)rows * K * acc_bytes(dtype) + 15) / 16 * 16 + (size_t)rows * 8;
}

extern "C" int rua_crf_forward(const void* x, const int64_t* tags, const void* W, const void* start, const void* end,
                               void* log_z, void* score, void* state_out, int32_t K, int32_t dtype,
                               const rua_ragged_t* ragged, const rua_side_t* side, void* ws, size_t ws_bytes,
                               rua_stream_t stream) {
  (void)ws;
  (void)ws_bytes;
  if (int rc = validate(K, dtype, ragged, side)) return rc;
  if (ragged->B == 0) return RUA_OK;
  if ((side->rows > 0 && !x) || !W || !log_z || (!tags) != (!score)) return RUA_ERR_INVALID;
  CrfArgs a{};
  fill_layout(a, K, ragged, side);
  a.x = x;
  a.tags = tags;
  a.W = W;
  a.start = start;
  a.end = end;
  a.log_z = log_z;
  a.score = score;
  if (state_out && side->rows > 0) {
    a.alpha = state_out;
    a.c = reinterpret_cast<double*>(static_cast<char*>(state_out) +
                                    ((size_t)side->rows * K * acc_bytes(dtype) + 15) / 16 * 16);
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return tags ? run_forward<1>(dtype, a, st) : run_forward<0>(dtype, a, st);
}

extern "C" int rua_crf_decode(const void* x, const void* W, const void* start, const void* end, int64_t* tags_out,
                              void* best_score, int32_t K, int32_t dtype, const rua_ragged_t* ragged,
                              const rua_side_t* side, void* ws, size_t ws_bytes, rua_stream_t stream) {
  if (int rc = validate(K, dtype, ragged, side)) return rc;
  if (ragged->B == 0 && side->rows == 0) return RUA_OK;
  if ((side->rows > 0 && (!x || !tags_out)) || !W || (ragged->B > 0 && !best_score)) return RUA_ERR_INVALID;
  if (side->rows > 0 && (!ws || ws_bytes < rua_crf_workspace_bytes(side->rows, K, dtype, RUA_CRF_DECODE)))
    return RUA_ERR_WORKSPACE;
  CrfArgs a{};
  fill_layout(a, K, ragged, side);
  a.x = x;
  a.W = W;
  a.start = start;
  a.end = end;
  a.score = best_score;
  a.tags_out = tags_out;
  a.bp = static_cast<uint8_t*>(ws);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (ragged->B == 0) {   // C rows with no sequence at all
    if (int rc = check_cuda(cudaMemsetAsync(tags_out, 0xff, (size_t)side->rows * 8, st))) return rc;
    return RUA_OK;
  }
  return run_forward<2>(dtype, a, st);
}

extern "C" int rua_crf_backward(const void* grad_log_z, const void* grad_score, const void* x, const int64_t* tags,
                                const void* W, const void* start, const void* end, const void* state, const void* log_z,
                                void* grad_x, void* grad_W, void* grad_start, void* grad_end, int32_t K, int32_t dtype,
                                const rua_ragged_t* ragged, const rua_side_t* side, void* ws, size_t ws_bytes,
                                rua_stream_t stream) {
  if (int rc = validate(K, dtype, ragged, side)) return rc;
  const bool want_p = grad_W || grad_start || grad_end;
  if (!grad_x && !want_p) return RUA_OK;
  const int64_t rows = side->rows, B = ragged->B;
  if (!W) return RUA_ERR_INVALID;
  if (rows > 0 && B > 0 && (!grad_log_z || !x || !state || !log_z || (grad_score && !tags))) return RUA_ERR_INVALID;
  if (rows > 0 && B > 0 && want_p && (!ws || ws_bytes < rua_crf_workspace_bytes(rows, K, dtype, RUA_CRF_BACKWARD)))
    return RUA_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t esz = dtype == RUA_F64 ? 8 : (dtype == RUA_F32 ? 4 : 2);
  if (rows == 0 || B == 0) {   // no token: every gradient is 0
    if (grad_x && rows > 0)
      if (int rc = check_cuda(cudaMemsetAsync(grad_x, 0, (size_t)rows * K * esz, st))) return rc;
    if (grad_W)
      if (int rc = check_cuda(cudaMemsetAsync(grad_W, 0, (size_t)K * K * esz, st))) return rc;
    if (grad_start)
      if (int rc = check_cuda(cudaMemsetAsync(grad_start, 0, (size_t)K * esz, st))) return rc;
    if (grad_end)
      if (int rc = check_cuda(cudaMemsetAsync(grad_end, 0, (size_t)K * esz, st))) return rc;
    return RUA_OK;
  }
  CrfArgs a{};
  fill_layout(a, K, ragged, side);
  a.x = x;
  a.tags = tags;
  a.W = W;
  a.end = end;
  a.alpha = const_cast<void*>(state);
  a.c = reinterpret_cast<double*>(static_cast<char*>(const_cast<void*>(state)) +
                                  ((size_t)rows * K * acc_bytes(dtype) + 15) / 16 * 16);
  a.g_z = grad_log_z;
  a.g_s = grad_score;
  a.lz_in = log_z;
  a.gx = grad_x;
  a.slots = want_p ? ws : nullptr;
  a.want_w = grad_W != nullptr;
  (void)start;   // alpha~ already holds the start scores
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    using Acc = typename Store<T>::Acc;
    const size_t smem = bwd_smem(K, sizeof(Acc));
    const int64_t grid = grid_of(B, kBwdWarps, bwd_max_slots(K, sizeof(Acc)));
    auto go = [&](auto j) {
      return launch(crf_backward_kernel<T, decltype(j)::value>, grid, kBwdWarps * 32, smem, st, a);
    };
    if (int rc = K > 32 ? go(Int<2>{}) : go(Int<1>{})) return rc;
    if (!want_p) return (int)RUA_OK;
    return launch_slot_sum<T>(static_cast<const Acc*>(ws), grid, (int64_t)K * K + 2 * K, (int64_t)K * K + 2 * K,
                              CrfCols<T>{static_cast<T*>(grad_W), static_cast<T*>(grad_start), static_cast<T*>(grad_end),
                                         K},
                              st);
  });
}
