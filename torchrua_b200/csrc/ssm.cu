// K10 -- per-sequence selective state-space scan (Mamba-1 style, state size N <= 16), forward and backward, on every
// layout.
//
// For token (i, t) of sequence i, channel h < H (the flattened *feat) and state n < N:
//   dA_t[h, n] = exp(delta_t[h] A[h, n])
//   h_t[h, n]  = dA_t[h, n] h_{t-1}[h, n] + delta_t[h] B_t[n] x_t[h],     h_{-1} = h0[i] (0 without one)
//   y_t[h]     = sum_n C_t[n] h_t[h, n]
// (reverse: from each sequence's end, h_{len} = h0[i]).  Replaces pad -> a Python loop over T that keeps a (B, H, N)
// state per step for autograd, and the composition through the linear recurrence that materialises (tokens, H, N)
// gates, inputs and states.
//
// Design (sequential in t, independent across sequences and channels; bound by one exponential per (t, h, n)):
//   * the unit of work is a sequence x a block of kThr channels, one thread per channel holding its N states and
//     A[h, :] (times log2 e) in registers.  CTA (cb, g) of a grid (ceil(H / kThr), G) takes channel block cb of the
//     sequences of ranks g, g + G, ... of ragged->sorted (longest first for the package's own sort), so every thread
//     keeps one channel for the whole launch and the result never depends on timing or on the layout;
//   * row t of sequence i comes from the closed-form row of its layout (seq_rows.cuh);
//   * B_t and C_t of the next kTc steps are staged once per CTA in shared memory and shared by every channel; x and
//     delta of step t + 1 are loaded while step t computes;
//   * each (t, h, n) costs one FMUL + MUFU.EX2 (fp32) for dA;
//   * when a gradient is wanted, the forward stores the state entering every chunk of kTc = 32 steps of a sequence
//     (its slot is off[i] / kTc + i + chunk, so at most rows / 32 + B states of H x N).
// Backward (same units, each sequence from its end, chunk by chunk):
//   * restore the chunk's checkpoint and recompute its states, keeping one sub-checkpoint every kSub steps in shared
//     memory; then per sub-chunk (last first) recompute its kSub states into registers and run the adjoint
//     dh_t = C_t g_t + dA_{t+1} dh_{t+1} backwards over them;
//   * grad_x and grad_delta are per (token, channel) and are written directly;
//   * grad_A is accumulated per thread over all its sequences and stored to the CTA's row of per-g slots, which
//     slot_sum adds in slot order;
//   * grad_B and grad_C are per-token sums over channels: every warp reduces its 32 channels with a transpose-reduce
//     of fixed shape (one for grad_B, one for grad_C), the CTA adds its warps in warp order, writes one partial per
//     (token, channel block), and slot_sum adds the partials in block order.  No atomics anywhere: bit-identical run
//     to run and across layouts.
#include "dispatch.cuh"
#include "reduce_common.cuh"
#include "seq_rows.cuh"
#include "slot_sum.cuh"

namespace rua {
namespace {

constexpr int kMaxState = 16;
constexpr int kTc = 32;                     // checkpoint interval (steps)
constexpr int kFwdThr = 128;
constexpr int kFwdCtasPerSM = 8;
constexpr size_t kSmemPerSM = 220 * 1024;   // shared memory the CTAs of one SM may use together

// backward shape per accumulator type: channels per CTA and the sub-chunk held in registers
template <typename A> struct Bwd;
template <> struct Bwd<float> {
  static constexpr int kThr = 128, kSub = 4;
};
template <> struct Bwd<double> {
  static constexpr int kThr = 64, kSub = 2;
};

// CTAs per SM each instance is compiled for: the register budget that keeps every fp32-accumulated instance free of
// spills without costing the small-N buckets their occupancy
template <typename A, int NB> constexpr int fwd_min_ctas() { return sizeof(A) == 4 && NB == 4 ? 16 : 4; }
template <typename A, int NB> constexpr int bwd_min_ctas() { return sizeof(A) == 8 ? 2 : (NB == 4 ? 5 : (NB == 8 ? 3 : 2)); }

struct SsmArgs {
  const void* x;          // rows x H
  const void* dl;         // rows x H (delta)
  const void* A;          // H x N, accumulator type
  const void* Bm;         // rows x N
  const void* Cm;         // rows x N
  const void* h0;         // B x H x N accumulator type, or NULL
  void* y;                // rows x H
  void* hfin;             // B x H x N accumulator type, or NULL
  void* ck;               // checkpoints: (rows / kTc + B) x H x N accumulator type, or NULL
  const void* g;          // backward: grad_out, rows x H
  void* gx;               // rows x H or NULL
  void* gdl;              // rows x H or NULL
  void* ga_slots;         // G x H x N accumulator type, or NULL
  void* part;             // ceil(H / kThr) x rows x 2N accumulator type: [grad_B | grad_C] partials, or NULL
  void* gh0;              // B x H x N accumulator type, or NULL
  int64_t H;
  int N;
  int reverse;
  int64_t B;
  const int64_t* off;
  const int64_t* poff;
  const int64_t* sorted;
  const int64_t* unsorted;
  int32_t layout;
  int64_t Wd;             // L / R width
  int64_t rows;
};

// exponential of the scaled argument: ex2.approx for fp32 (A is pre-scaled by log2 e), exp for fp64
__device__ __forceinline__ float ssm_exp(float v) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}
__device__ __forceinline__ double ssm_exp(double v) { return exp(v); }
template <typename A> __host__ __device__ constexpr A exp_scale() { return sizeof(A) == 4 ? A(1.4426950408889634) : A(1); }

// storage row of processing step p (p counts from the sequence's end for reverse)
__device__ __forceinline__ int64_t step_row(const SsmArgs& a, const Seq& s, int64_t p) {
  return row_of(a, s, a.reverse ? s.len - 1 - p : p);
}

// stage B_t | C_t of steps [p0, p0 + steps) as sBC[j * 2NB + k] (k < NB: B, else C; 0 for n >= N)
template <typename T, int NB, typename A>
__device__ __forceinline__ void stage_bc(const SsmArgs& a, const Seq& s, int64_t p0, int steps, A* sBC, int nthr) {
  const T* Bm = static_cast<const T*>(a.Bm);
  const T* Cm = static_cast<const T*>(a.Cm);
  for (int e = threadIdx.x; e < steps * 2 * NB; e += nthr) {
    const int j = e / (2 * NB), k = e - j * 2 * NB;
    const int n = k < NB ? k : k - NB;
    A v = 0;
    if (n < a.N) {
      const int64_t r = step_row(a, s, p0 + j);
      v = Store<T>::to_acc((k < NB ? Bm : Cm)[r * a.N + n]);
    }
    sBC[e] = v;
  }
}

// warp sum of V values (V a power of 2, <= 32) per lane: lane l ends with the sum over the warp of v[l % V].  A fixed
// butterfly, so the result is the same bits on every run.
template <typename A, int V> __device__ __forceinline__ A warp_transpose_sum(A (&v)[V], int lane) {
#pragma unroll
  for (int half = V / 2; half >= 1; half /= 2) {
    const bool up = lane & half;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const A send = up ? v[i] : v[i + half];
      const A keep = up ? v[i + half] : v[i];
      v[i] = keep + __shfl_xor_sync(kFullMask, send, half);
    }
  }
  A r = v[0];
#pragma unroll
  for (int o = V; o < 32; o *= 2) r += __shfl_xor_sync(kFullMask, r, o);
  return r;
}

template <typename T, int NB, bool kKeep>
__global__ void __launch_bounds__(kFwdThr, fwd_min_ctas<typename Store<T>::Acc, NB>()) ssm_forward_kernel(SsmArgs a) {
  using A = typename Store<T>::Acc;
  __shared__ A sBC[kTc * 2 * NB];
  const int tid = threadIdx.x, N = a.N;
  const int64_t H = a.H, h = (int64_t)blockIdx.x * kFwdThr + tid;
  const bool on = h < H;
  const T* x = static_cast<const T*>(a.x);
  const T* dl = static_cast<const T*>(a.dl);
  T* y = static_cast<T*>(a.y);
  A a2[NB];
#pragma unroll
  for (int n = 0; n < NB; ++n) a2[n] = on && n < N ? static_cast<const A*>(a.A)[h * N + n] * exp_scale<A>() : A(0);
  if (on && a.layout == RUA_CAT)   // C rows past the tokens are copied through
    for (int64_t r = __ldg(a.off + a.B) + blockIdx.y; r < a.rows; r += gridDim.y) y[r * H + h] = x[r * H + h];

  for (int64_t rank = blockIdx.y; rank < a.B; rank += gridDim.y) {
    const Seq s = seq_of(a, rank);
    if (on) for_padding_rows(a, s, 0, 1, [&](int64_t r) { y[r * H + h] = x[r * H + h]; });
    A st[NB];
    const A* h0 = a.h0 ? static_cast<const A*>(a.h0) + (s.i * H + h) * N : nullptr;
#pragma unroll
    for (int n = 0; n < NB; ++n) st[n] = on && n < N && h0 ? h0[n] : A(0);
    const int64_t base = s.o / kTc + s.i;
    for (int64_t p0 = 0; p0 < s.len; p0 += kTc) {
      const int steps = (int)(s.len - p0 < kTc ? s.len - p0 : kTc);
      __syncthreads();   // the previous chunk's B / C are consumed
      stage_bc<T, NB>(a, s, p0, steps, sBC, kFwdThr);
      __syncthreads();
      if (!on) continue;
      if constexpr (kKeep) {
        A* ck = static_cast<A*>(a.ck) + ((base + p0 / kTc) * H + h) * N;
#pragma unroll
        for (int n = 0; n < NB; ++n)
          if (n < N) ck[n] = st[n];
      }
      int64_t rn = step_row(a, s, p0);
      T xn = x[rn * H + h], dn = dl[rn * H + h];
      for (int j = 0; j < steps; ++j) {
        const int64_t rc = rn;
        const A xv = Store<T>::to_acc(xn), d = Store<T>::to_acc(dn);
        if (j + 1 < steps) {
          rn = step_row(a, s, p0 + j + 1);
          xn = x[rn * H + h];
          dn = dl[rn * H + h];
        }
        const A dx = d * xv;
        const A* bc = sBC + j * 2 * NB;
        A acc = 0;
#pragma unroll
        for (int n = 0; n < NB; ++n) {
          st[n] = ssm_exp(d * a2[n]) * st[n] + dx * bc[n];
          acc += bc[NB + n] * st[n];
        }
        y[rc * H + h] = Store<T>::from_acc(acc);
      }
    }
    if (a.hfin && on) {
      A* hf = static_cast<A*>(a.hfin) + (s.i * H + h) * N;
#pragma unroll
      for (int n = 0; n < NB; ++n)
        if (n < N) hf[n] = st[n];
    }
  }
}

template <typename A, int NB> constexpr size_t bwd_smem_bytes() {
  constexpr int kThr = Bwd<A>::kThr, kSub = Bwd<A>::kSub;
  return sizeof(A) * ((size_t)kTc * 2 * NB                          // sBC
                      + (size_t)(kTc / kSub) * NB * kThr            // sub-checkpoints [q][n][tid]
                      + (size_t)kTc * (kThr / 32) * 2 * NB          // per-warp grad_B | grad_C sums [j][warp][k]
                      + 2 * (size_t)NB * kThr);                     // A[h, :] and the grad_A sums [n][tid]
}

template <typename T, int NB>
__global__ void __launch_bounds__(Bwd<typename Store<T>::Acc>::kThr, bwd_min_ctas<typename Store<T>::Acc, NB>())
ssm_backward_kernel(SsmArgs a) {
  using A = typename Store<T>::Acc;
  constexpr int kThr = Bwd<A>::kThr, kSub = Bwd<A>::kSub, kWarps = kThr / 32, V = 2 * NB;
  extern __shared__ __align__(16) unsigned char smem[];
  A* sBC = reinterpret_cast<A*>(smem);
  A* sSub = sBC + kTc * V;
  A* sRed = sSub + (kTc / kSub) * NB * kThr;
  A* sA = sRed + kTc * kWarps * V;
  A* sGA = sA + NB * kThr;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, N = a.N;
  const int64_t H = a.H, h = (int64_t)blockIdx.x * kThr + tid, rows = a.rows;
  const bool on = h < H;
  const T* x = static_cast<const T*>(a.x);
  const T* dl = static_cast<const T*>(a.dl);
  const T* g = static_cast<const T*>(a.g);
  T* gx = static_cast<T*>(a.gx);
  T* gdl = static_cast<T*>(a.gdl);
  A* part = a.part ? static_cast<A*>(a.part) + (int64_t)blockIdx.x * rows * 2 * N : nullptr;
  A a2[NB];
#pragma unroll
  for (int n = 0; n < NB; ++n) {
    const A av = on && n < N ? static_cast<const A*>(a.A)[h * N + n] : A(0);
    a2[n] = av * exp_scale<A>();
    sA[n * kThr + tid] = av;
    sGA[n * kThr + tid] = A(0);
  }
  const T zero = Store<T>::from_acc(0);
  // a row that holds no token: grad_x = grad_out, grad_delta = 0, grad_B = grad_C = 0
  auto no_token = [&](int64_t r) {
    if (on) {
      if (gx) gx[r * H + h] = g[r * H + h];
      if (gdl) gdl[r * H + h] = zero;
    }
    if (part)
      for (int k = tid; k < 2 * N; k += kThr) part[r * 2 * N + k] = A(0);
  };
  if (a.layout == RUA_CAT)
    for (int64_t r = __ldg(a.off + a.B) + blockIdx.y; r < rows; r += gridDim.y) no_token(r);

  for (int64_t rank = blockIdx.y; rank < a.B; rank += gridDim.y) {
    const Seq s = seq_of(a, rank);
    for_padding_rows(a, s, 0, 1, no_token);
    A c[NB];   // dA_{t+1} dh_{t+1}: the adjoint carried into step t
#pragma unroll
    for (int n = 0; n < NB; ++n) c[n] = A(0);
    const int64_t base = s.o / kTc + s.i;
    for (int64_t p0 = s.len > 0 ? (s.len - 1) / kTc * kTc : -1; p0 >= 0; p0 -= kTc) {
      const int steps = (int)(s.len - p0 < kTc ? s.len - p0 : kTc);
      __syncthreads();   // the previous chunk's B / C and warp sums are consumed
      stage_bc<T, NB>(a, s, p0, steps, sBC, kThr);
      __syncthreads();
      // restore the chunk's checkpoint and recompute its states, keeping the state entering every kSub steps
      A st[NB];
      const A* ck = static_cast<const A*>(a.ck) + ((base + p0 / kTc) * H + h) * N;
#pragma unroll
      for (int n = 0; n < NB; ++n) st[n] = on && n < N ? ck[n] : A(0);
      for (int j = 0; j < steps; ++j) {
        if (j % kSub == 0) {
#pragma unroll
          for (int n = 0; n < NB; ++n) sSub[((j / kSub) * NB + n) * kThr + tid] = st[n];
        }
        const int64_t r = step_row(a, s, p0 + j);
        const A d = on ? Store<T>::to_acc(dl[r * H + h]) : A(0);
        const A dx = on ? d * Store<T>::to_acc(x[r * H + h]) : A(0);
        const A* bc = sBC + j * V;
#pragma unroll
        for (int n = 0; n < NB; ++n) st[n] = ssm_exp(d * a2[n]) * st[n] + dx * bc[n];
      }
      // sub-chunks, last first: recompute kSub states into registers, then the adjoint backwards over them
      for (int q = (steps - 1) / kSub; q >= 0; --q) {
        const int j0 = q * kSub, m = steps - j0 < kSub ? steps - j0 : kSub;
        const A* sub = sSub + q * NB * kThr + tid;   // the state entering step j0, [n * kThr]
        A hs[kSub][NB];   // hs[jj] = the state after step j0 + jj
        A xs[kSub], ds[kSub];
        int64_t rs[kSub];
#pragma unroll
        for (int jj = 0; jj < kSub; ++jj) {
          rs[jj] = jj < m ? step_row(a, s, p0 + j0 + jj) : 0;
          ds[jj] = on && jj < m ? Store<T>::to_acc(dl[rs[jj] * H + h]) : A(0);
          xs[jj] = on && jj < m ? Store<T>::to_acc(x[rs[jj] * H + h]) : A(0);
          const A dx = ds[jj] * xs[jj];
          const A* bc = sBC + (j0 + jj) * V;
#pragma unroll
          for (int n = 0; n < NB; ++n)
            hs[jj][n] = ssm_exp(ds[jj] * a2[n]) * (jj ? hs[jj - 1][n] : sub[n * kThr]) + dx * bc[n];
        }
#pragma unroll
        for (int jj = kSub - 1; jj >= 0; --jj) {
          if (jj >= m) continue;   // m is the same on every thread of the CTA
          const int j = j0 + jj;
          const A d = ds[jj], xv = xs[jj];
          const A gv = on ? Store<T>::to_acc(g[rs[jj] * H + h]) : A(0);
          const A* bc = sBC + j * V;
          A vals[NB];   // grad_B terms of this channel, then its grad_C terms
          A sum_bdh = 0, sum_aq = 0;
#pragma unroll
          for (int n = 0; n < NB; ++n) {
            const A dA = ssm_exp(d * a2[n]);
            const A dh = bc[NB + n] * gv + c[n];
            const A q_ = dh * dA * (jj ? hs[jj - 1][n] : sub[n * kThr]);   // dh_t dA_t h_{t-1}
            sum_bdh += bc[n] * dh;
            sum_aq += sA[n * kThr + tid] * q_;
            sGA[n * kThr + tid] += d * q_;
            c[n] = dA * dh;
            vals[n] = dh * d * xv;
          }
          if (on) {
            if (gx) gx[rs[jj] * H + h] = Store<T>::from_acc(d * sum_bdh);
            if (gdl) gdl[rs[jj] * H + h] = Store<T>::from_acc(sum_aq + xv * sum_bdh);
          }
          if (part) {
            A* red = sRed + (j * kWarps + warp) * V;
            const A wb = warp_transpose_sum<A, NB>(vals, lane);
            if (lane < NB) red[lane] = wb;
#pragma unroll
            for (int n = 0; n < NB; ++n) vals[n] = gv * hs[jj][n];
            const A wc = warp_transpose_sum<A, NB>(vals, lane);
            if (lane < NB) red[NB + lane] = wc;
          }
        }
      }
      if (part) {
        __syncthreads();
        for (int e = tid; e < steps * 2 * N; e += kThr) {
          const int j = e / (2 * N), k = e - j * 2 * N;
          const int kk = k < N ? k : NB + k - N;
          A v = 0;
#pragma unroll
          for (int w = 0; w < kWarps; ++w) v += sRed[(j * kWarps + w) * V + kk];
          part[step_row(a, s, p0 + j) * 2 * N + k] = v;
        }
      }
    }
    if (a.gh0 && on) {
      A* gh = static_cast<A*>(a.gh0) + (s.i * H + h) * N;
#pragma unroll
      for (int n = 0; n < NB; ++n)
        if (n < N) gh[n] = s.len ? c[n] : A(0);
    }
  }
  if (a.ga_slots && on) {
    A* slot = static_cast<A*>(a.ga_slots) + ((int64_t)blockIdx.y * H + h) * N;
#pragma unroll
    for (int n = 0; n < NB; ++n)
      if (n < N) slot[n] = sGA[n * kThr + tid];
  }
}

// columns of the partial sum: rows x [grad_B (N) | grad_C (N)]
template <typename T> struct BCCols {
  T* gb;
  T* gc;
  int N;
  __device__ T* operator()(int64_t i, int64_t& src) const {
    src = i;
    const int64_t r = i / (2 * N), k = i - r * 2 * N;
    if (k < N) return gb ? gb + r * N + k : nullptr;
    return gc ? gc + r * N + (k - N) : nullptr;
  }
};

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
int bwd_threads(int32_t dtype) { return dtype == RUA_F64 ? Bwd<double>::kThr : Bwd<float>::kThr; }
int bucket(int32_t N) { return N <= 4 ? 4 : (N <= 8 ? 8 : 16); }
size_t bwd_smem(int32_t dtype, int32_t N) {
  const int nb = bucket(N);
  if (dtype == RUA_F64)
    return nb == 4 ? bwd_smem_bytes<double, 4>() : (nb == 8 ? bwd_smem_bytes<double, 8>() : bwd_smem_bytes<double, 16>());
  return nb == 4 ? bwd_smem_bytes<float, 4>() : (nb == 8 ? bwd_smem_bytes<float, 8>() : bwd_smem_bytes<float, 16>());
}

// sequence dimension of the grid: enough CTAs for `per_sm` per SM over the channel blocks, at most one per sequence
int64_t seq_grid(int64_t B, int64_t nblk, int64_t per_sm) {
  const int64_t g = ceil_div(kNumSMs * per_sm, nblk);
  return g < B ? g : B;
}
int64_t bwd_ctas_per_sm(int32_t dtype, int32_t N) {
  const int64_t n = (int64_t)(kSmemPerSM / bwd_smem(dtype, N));
  return n < 1 ? 1 : n;
}
int64_t bwd_seq_grid(int64_t B, int64_t H, int32_t N, int32_t dtype) {
  return seq_grid(B, ceil_div(H, bwd_threads(dtype)), bwd_ctas_per_sm(dtype, N));
}

size_t align256(size_t v) { return (v + 255) / 256 * 256; }
// grad_A slots, then the [grad_B | grad_C] partials
size_t slots_bytes(int64_t B, int64_t H, int32_t N, int32_t dtype) {
  return align256((size_t)bwd_seq_grid(B, H, N, dtype) * H * N * acc_bytes(dtype));
}
size_t part_bytes(int64_t rows, int64_t H, int32_t N, int32_t dtype) {
  return (size_t)ceil_div(H, bwd_threads(dtype)) * rows * 2 * N * acc_bytes(dtype);
}

int validate(int64_t H, int32_t N, int32_t dtype, int32_t reverse, const rua_ragged_t* rg, const rua_side_t* side) {
  if (bad_dtype(dtype) || N < 1 || H < 0 || (reverse != 0 && reverse != 1)) return RUA_ERR_INVALID;
  if (N > kMaxState) return RUA_ERR_UNSUPPORTED;
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

void fill_layout(SsmArgs& a, int64_t H, int32_t N, int32_t reverse, const rua_ragged_t* rg, const rua_side_t* side) {
  a.H = H;
  a.N = N;
  a.reverse = reverse;
  a.B = rg->B;
  a.off = rg->off;
  a.poff = rg->poff;
  a.sorted = rg->sorted;
  a.unsorted = rg->unsorted;
  a.layout = side->layout;
  a.Wd = side->width;
  a.rows = side->rows;
}

template <typename F> int with_bucket(int32_t N, F&& f) {
  switch (bucket(N)) {
    case 4: return f(Int<4>{});
    case 8: return f(Int<8>{});
    default: return f(Int<16>{});
  }
}

}  // namespace
}  // namespace rua

using namespace rua;

extern "C" size_t rua_ssm_state_bytes(int64_t rows, int64_t B, int64_t H, int32_t N, int32_t dtype) {
  if (rows < 0 || B < 0 || H < 0 || N < 1 || N > kMaxState || bad_dtype(dtype)) return 0;
  return (size_t)(rows / kTc + B) * H * N * acc_bytes(dtype);
}

extern "C" size_t rua_ssm_workspace_bytes(int64_t rows, int64_t B, int64_t H, int32_t N, int32_t dtype) {
  if (rows < 0 || B < 0 || H < 0 || N < 1 || N > kMaxState || bad_dtype(dtype)) return 0;
  if (rows == 0 || B == 0 || H == 0) return 0;
  return slots_bytes(B, H, N, dtype) + part_bytes(rows, H, N, dtype);
}

extern "C" int rua_ssm_forward(const void* x, const void* delta, const void* A, const void* Bm, const void* Cm,
                               const void* h0, void* y, void* h_final, void* state_out, int64_t H, int32_t N,
                               int32_t dtype, int32_t reverse, const rua_ragged_t* ragged, const rua_side_t* side,
                               void* ws, size_t ws_bytes, rua_stream_t stream) {
  (void)ws;
  (void)ws_bytes;
  if (int rc = validate(H, N, dtype, reverse, ragged, side)) return rc;
  const int64_t rows = side->rows, B = ragged->B;
  if (H == 0 || (rows == 0 && B == 0)) return RUA_OK;
  if (rows > 0 && (!x || !y)) return RUA_ERR_INVALID;
  if (B > 0 && (!A || (rows > 0 && (!delta || !Bm || !Cm)))) return RUA_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t esz = dtype == RUA_F64 ? 8 : (dtype == RUA_F32 ? 4 : 2);
  if (B == 0)   // C rows with no sequence at all: copied through
    return check_cuda(cudaMemcpyAsync(y, x, (size_t)rows * H * esz, cudaMemcpyDeviceToDevice, st));
  SsmArgs a{};
  fill_layout(a, H, N, reverse, ragged, side);
  a.x = x;
  a.dl = delta;
  a.A = A;
  a.Bm = Bm;
  a.Cm = Cm;
  a.h0 = h0;
  a.y = y;
  a.hfin = h_final;
  a.ck = state_out;
  const int64_t nblk = ceil_div(H, kFwdThr);
  const dim3 grid((unsigned)nblk, (unsigned)seq_grid(B, nblk, kFwdCtasPerSM));
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    return with_bucket(N, [&](auto nb) {
      constexpr int NB = decltype(nb)::value;
      if (state_out) ssm_forward_kernel<T, NB, true><<<grid, kFwdThr, 0, st>>>(a);
      else ssm_forward_kernel<T, NB, false><<<grid, kFwdThr, 0, st>>>(a);
      return check_launch();
    });
  });
}

extern "C" int rua_ssm_backward(const void* grad_out, const void* x, const void* delta, const void* A, const void* Bm,
                                const void* Cm, const void* state, void* grad_x, void* grad_delta, void* grad_A,
                                void* grad_B, void* grad_C, void* grad_h0, int64_t H, int32_t N, int32_t dtype,
                                int32_t reverse, const rua_ragged_t* ragged, const rua_side_t* side, void* ws,
                                size_t ws_bytes, rua_stream_t stream) {
  if (int rc = validate(H, N, dtype, reverse, ragged, side)) return rc;
  const bool want_ws = grad_A || grad_B || grad_C;
  if (!grad_x && !grad_delta && !want_ws && !grad_h0) return RUA_OK;
  const int64_t rows = side->rows, B = ragged->B;
  if (rows > 0 && H > 0 && !grad_out) return RUA_ERR_INVALID;
  if (rows > 0 && B > 0 && H > 0 && (!x || !delta || !A || !Bm || !Cm || !state)) return RUA_ERR_INVALID;
  const size_t need = rua_ssm_workspace_bytes(rows, B, H, N, dtype);   // 0 when there is no token
  if (want_ws && need && (!ws || ws_bytes < need)) return RUA_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t esz = dtype == RUA_F64 ? 8 : (dtype == RUA_F32 ? 4 : 2), acc = acc_bytes(dtype);
  if (rows == 0 || B == 0 || H == 0) {   // no token: grad_x passes grad_out through, every other gradient is 0
    if (grad_x && rows > 0 && H > 0)
      if (int rc = check_cuda(cudaMemcpyAsync(grad_x, grad_out, (size_t)rows * H * esz, cudaMemcpyDeviceToDevice, st)))
        return rc;
    const struct { void* p; size_t n; } zero[] = {{grad_delta, (size_t)rows * H * esz}, {grad_A, (size_t)H * N * acc},
                                                  {grad_B, (size_t)rows * N * esz}, {grad_C, (size_t)rows * N * esz},
                                                  {grad_h0, (size_t)B * H * N * acc}};
    for (const auto& z : zero)
      if (z.p && z.n)
        if (int rc = check_cuda(cudaMemsetAsync(z.p, 0, z.n, st))) return rc;
    return RUA_OK;
  }
  SsmArgs a{};
  fill_layout(a, H, N, reverse, ragged, side);
  a.x = x;
  a.dl = delta;
  a.A = A;
  a.Bm = Bm;
  a.Cm = Cm;
  a.ck = const_cast<void*>(state);
  a.g = grad_out;
  a.gx = grad_x;
  a.gdl = grad_delta;
  a.gh0 = grad_h0;
  const size_t sb = slots_bytes(B, H, N, dtype);
  a.ga_slots = grad_A ? ws : nullptr;
  a.part = (grad_B || grad_C) ? static_cast<char*>(ws) + sb : nullptr;
  const int64_t nblk = ceil_div(H, bwd_threads(dtype)), G = bwd_seq_grid(B, H, N, dtype);
  const size_t smem = bwd_smem(dtype, N);
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    using Acc = typename Store<T>::Acc;
    return with_bucket(N, [&](auto nb) {
      constexpr int NB = decltype(nb)::value;
      auto kern = ssm_backward_kernel<T, NB>;
      if (smem > 48 * 1024)
        if (int rc = check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)))
          return rc;
      kern<<<dim3((unsigned)nblk, (unsigned)G), Bwd<Acc>::kThr, smem, st>>>(a);
      if (int rc = check_launch()) return rc;
      if (grad_A)
        if (int rc = launch_slot_sum<Acc>(static_cast<const Acc*>(a.ga_slots), G, H * N, H * N,
                                          PlainCols<Acc>{static_cast<Acc*>(grad_A)}, st))
          return rc;
      if (a.part)
        return launch_slot_sum<T>(static_cast<const Acc*>(a.part), nblk, rows * 2 * N, rows * 2 * N,
                                  BCCols<T>{static_cast<T*>(grad_B), static_cast<T*>(grad_C), N}, st);
      return (int)RUA_OK;
    });
  });
}
