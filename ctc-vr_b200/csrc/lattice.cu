// RNN-T lattice: alpha / beta anti-diagonal wavefront and costs (SURVEY.md §8 A2; the recursion
// torchaudio.functional.rnnt_loss runs inside rnnt_loss_forward, called from
// model/component/transducer.py:180-187).
//
// One CTA per utterance.  Warp 0 walks alpha forward, warp 1 walks beta backward, concurrently.
// Lane l owns lattice columns u = l, l+32, ... (NJ per lane); one anti-diagonal t+u=d per step.
// The neighbour needed from column u-1 (alpha) / u+1 (beta) lives in the adjacent lane one
// diagonal earlier, so the exchange is a single warp shuffle and no barrier is needed.
// lp_blank / lp_label for the utterance are staged once into shared memory with coalesced loads
// (pitch chosen so that a diagonal read is bank-conflict free); utterances whose log-probs do not
// fit in shared memory are read through L2.
//
// Algorithmic HBM bytes: 24 B per cell (2 log-probs read for alpha, again for beta, alpha and beta
// written).  The kernel is bound by the T+U dependent diagonals, not by bandwidth.
#include <stdlib.h>

#include "common.cuh"

namespace ctcvr {

// ---------------------------------------------------------------------------------------------------------------
// Unpadded variant (the whole utterance fits in shared memory four times: lp_blank, lp_label, alpha, beta), used for
// the shapes whose PADDED arrays (next kernel) exceed shared memory.  All of it is aimed at the per-diagonal latency
// (the kernel is a chain of T+U dependent steps, nothing else matters):
//   - base-2 domain: the staged log-probs are pre-multiplied by log2(e), so a step is max / sub / ex2 / add / lg2 / add
//     with no scaling multiplies on the chain; alpha / beta are converted back when they are copied out
//   - alpha / beta are written to shared memory during the sweep (conflict-free diagonal stores) and copied to global
//     memory afterwards with coalesced row stores by all threads (scattered per-diagonal global stores occupy the LSU
//     for ~32 sectors per store)
//   - pointers advance by a constant per diagonal, predicates are selects (no divergent branches in the loop)
constexpr int LAT2_THREADS = 256;
constexpr float kLog2e = 1.4426950408889634f, kLn2 = 0.6931471805599453f;

__device__ __forceinline__ float ex2f(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lg2f(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// log2(2^a + 2^b); -inf safe without a branch: for a = b = -inf, m - m is NaN, so the difference is clamped first
__device__ __forceinline__ float lae2(float a, float b) {
  const float m = fmaxf(a, b), n = fminf(a, b);
  const float d = (n == kNegInf) ? kNegInf : n - m;          // <= 0, -inf if the smaller operand is -inf
  return m + lg2f(1.f + ex2f(d));
}

template <int NJ>
__global__ void __launch_bounds__(LAT2_THREADS) rnnt_lattice2_kernel(
    const float* __restrict__ lp_blank, const float* __restrict__ lp_label, const int32_t* __restrict__ t_len,
    const int32_t* __restrict__ u_len, float* __restrict__ alpha, float* __restrict__ beta,
    float* __restrict__ costs, int T, int U1, int pitch) {
  extern __shared__ float sm[];
  const int b = blockIdx.x;
  const int Tb = max(min(t_len[b], T), 0), Ub = max(min(u_len[b], U1 - 1), 0);
  const size_t base = (size_t)b * T * U1;
  if (Tb <= 0) { if (threadIdx.x == 0) costs[b] = 0.f; return; }
  const int W = Ub + 1;
  float* sb = sm;                               // lp_blank * log2e
  float* sl = sm + (size_t)T * pitch;           // lp_label * log2e
  float* sa = sm + (size_t)2 * T * pitch;       // alpha (base 2)
  float* sc = sm + (size_t)3 * T * pitch;       // beta  (base 2)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = LAT2_THREADS >> 5;
  {
    // flat, 4-deep unrolled staging: the loads of four elements per array are in flight before the first store
    const int n = Tb * U1;                      // rows are contiguous in global memory (row pitch U1)
    const float* gb = lp_blank + base;
    const float* gl = lp_label + base;
    for (int i0 = threadIdx.x; i0 < n; i0 += 4 * LAT2_THREADS) {
      float xb[4], xl[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int i = i0 + k * LAT2_THREADS;
        xb[k] = (i < n) ? __ldg(gb + i) : 0.f;
        xl[k] = (i < n) ? __ldg(gl + i) : 0.f;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int i = i0 + k * LAT2_THREADS;
        if (i < n) {
          const int t = i / U1, u = i - t * U1;
          sb[t * pitch + u] = xb[k] * kLog2e;
          sl[t * pitch + u] = xl[k] * kLog2e;
        }
      }
    }
  }
  __syncthreads();
  const int ndiag = Tb + Ub;
  // Raw 32-bit shared addresses advanced by one row per diagonal: no generic->shared conversion, no index multiply and
  // no divergent branch inside the dependent loop (loads of inactive cells read a safe address and are discarded).
  // The NJ column groups of a lane are processed stage by stage so that their independent dependency chains interleave.
  const uint32_t s_sb = (uint32_t)__cvta_generic_to_shared(sb), s_sl = (uint32_t)__cvta_generic_to_shared(sl);
  const uint32_t s_sa = (uint32_t)__cvta_generic_to_shared(sa), s_sc = (uint32_t)__cvta_generic_to_shared(sc);
  const uint32_t rowb = (uint32_t)pitch * 4u;
  auto lds = [](uint32_t a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; };
  auto sts = [](uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); };
  if (warp == 0) {
    // ---------------- alpha(t,u) = LSE(alpha(t-1,u)+lpb(t-1,u), alpha(t,u-1)+lpl(t,u-1)),  t = d - u
    float prev[NJ], nb[NJ], nl[NJ];
    uint32_t ab[NJ], al[NJ], ao[NJ];            // addresses at diagonal d of lpb[t-1][u], lpl[t][u-1], alpha[t][u]
    int tt[NJ];                                 // t = d - u
    bool col[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int u = lane + 32 * j;
      prev[j] = kNegInf;
      tt[j] = -u;
      col[j] = u <= Ub;
      ab[j] = s_sb + (uint32_t)((-u - 1) * pitch + u) * 4u;
      al[j] = s_sl + (uint32_t)((-u) * pitch + u - 1) * 4u;
      ao[j] = s_sa + (uint32_t)((-u) * pitch + u) * 4u;
    }
    auto fetch = [&](int j, int t, uint32_t pb, uint32_t pl) {
      const bool in = col[j] && (unsigned)t < (unsigned)Tb;
      const bool okb = in && t > 0, okl = in && (lane + 32 * j) > 0;
      const float xb = lds(okb ? pb : s_sb), xl = lds(okl ? pl : s_sl);
      nb[j] = okb ? xb : kNegInf;
      nl[j] = okl ? xl : kNegInf;
    };
#pragma unroll
    for (int j = 0; j < NJ; ++j) fetch(j, tt[j], ab[j], al[j]);
    for (int d = 0; d < ndiag; ++d) {
      float cb[NJ], cl[NJ];
#pragma unroll
      for (int j = 0; j < NJ; ++j) { cb[j] = nb[j]; cl[j] = nl[j]; }
#pragma unroll
      for (int j = 0; j < NJ; ++j) fetch(j, tt[j] + 1, ab[j] + rowb, al[j] + rowb);     // next diagonal
      float cur[NJ], left[NJ], wrap[NJ], xa[NJ], xb[NJ], mm[NJ], dd[NJ];
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        left[j] = __shfl_up_sync(0xffffffffu, prev[j], 1);
        wrap[j] = __shfl_sync(0xffffffffu, prev[j > 0 ? j - 1 : 0], 31);
      }
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        if (lane == 0) left[j] = (j > 0) ? wrap[j] : kNegInf;
        xa[j] = prev[j] + cb[j];
        xb[j] = left[j] + cl[j];
      }
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        mm[j] = fmaxf(xa[j], xb[j]);
        const float n = fminf(xa[j], xb[j]);
        dd[j] = (n == kNegInf) ? kNegInf : n - mm[j];
      }
#pragma unroll
      for (int j = 0; j < NJ; ++j) dd[j] = ex2f(dd[j]);
#pragma unroll
      for (int j = 0; j < NJ; ++j) dd[j] = lg2f(1.f + dd[j]);
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        const bool in = col[j] && (unsigned)tt[j] < (unsigned)Tb;
        float v = mm[j] + dd[j];
        v = (d == 0 && j == 0 && lane == 0) ? 0.f : v;
        v = in ? v : kNegInf;
        if (in) sts(ao[j], v);
        cur[j] = v;
      }
#pragma unroll
      for (int j = 0; j < NJ; ++j) { prev[j] = cur[j]; tt[j] += 1; ab[j] += rowb; al[j] += rowb; ao[j] += rowb; }
    }
  } else if (warp == 1) {
    // ---------------- beta(t,u) = LSE(beta(t+1,u)+lpb(t,u), beta(t,u+1)+lpl(t,u)),  beta(T-1,U) = lpb(T-1,U)
    float prev[NJ], nb[NJ], nl[NJ];
    uint32_t ax[NJ];                            // byte offset of cell (t,u) at diagonal d (same for lpb, lpl, beta)
    int tt[NJ];
    bool col[NJ];
    const int d0 = ndiag - 1;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int u = lane + 32 * j;
      prev[j] = kNegInf;
      tt[j] = d0 - u;
      col[j] = u <= Ub;
      ax[j] = (uint32_t)((d0 - u) * pitch + u) * 4u;
    }
    auto fetch = [&](int j, int t, uint32_t off) {
      const bool in = col[j] && (unsigned)t < (unsigned)Tb;
      const bool okl = in && (lane + 32 * j) < Ub;
      const float xb = lds(s_sb + (in ? off : 0u)), xl = lds(s_sl + (okl ? off : 0u));
      nb[j] = in ? xb : kNegInf;
      nl[j] = okl ? xl : kNegInf;
    };
#pragma unroll
    for (int j = 0; j < NJ; ++j) fetch(j, tt[j], ax[j]);
    for (int d = d0; d >= 0; --d) {
      float cb[NJ], cl[NJ];
#pragma unroll
      for (int j = 0; j < NJ; ++j) { cb[j] = nb[j]; cl[j] = nl[j]; }
#pragma unroll
      for (int j = 0; j < NJ; ++j) fetch(j, tt[j] - 1, ax[j] - rowb);                    // next diagonal (d - 1)
      float cur[NJ], right[NJ], wrap[NJ], xa[NJ], xb[NJ], mm[NJ], dd[NJ];
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        right[j] = __shfl_down_sync(0xffffffffu, prev[j], 1);
        wrap[j] = __shfl_sync(0xffffffffu, prev[(j + 1 < NJ) ? j + 1 : j], 0);
      }
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        if (lane == 31) right[j] = (j + 1 < NJ) ? wrap[j] : kNegInf;
        xa[j] = (tt[j] + 1 < Tb) ? prev[j] + cb[j] : kNegInf;
        xb[j] = right[j] + cl[j];
      }
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        mm[j] = fmaxf(xa[j], xb[j]);
        const float n = fminf(xa[j], xb[j]);
        dd[j] = (n == kNegInf) ? kNegInf : n - mm[j];
      }
#pragma unroll
      for (int j = 0; j < NJ; ++j) dd[j] = ex2f(dd[j]);
#pragma unroll
      for (int j = 0; j < NJ; ++j) dd[j] = lg2f(1.f + dd[j]);
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        const int u = lane + 32 * j;
        const bool in = col[j] && (unsigned)tt[j] < (unsigned)Tb;
        float v = mm[j] + dd[j];
        v = (tt[j] == Tb - 1 && u == Ub) ? cb[j] : v;
        v = in ? v : kNegInf;
        if (in) sts(s_sc + ax[j], v);
        cur[j] = v;
      }
#pragma unroll
      for (int j = 0; j < NJ; ++j) { prev[j] = cur[j]; tt[j] -= 1; ax[j] -= rowb; }
    }
    if (lane == 0) costs[b] = -prev[0] * kLn2;     // beta(0,0)
  }
  __syncthreads();
  for (int t = warp; t < Tb; t += nwarp)
    for (int u = lane; u < W; u += 32) {
      alpha[base + (size_t)t * U1 + u] = sa[t * pitch + u] * kLn2;
      beta[base + (size_t)t * U1 + u] = sc[t * pitch + u] * kLn2;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// v3: the same wavefront with the boundary handling moved out of the dependent loop.  The dependent chain of a
// diagonal is one warp's instruction stream (v2: ~70 instructions = 340 cycles per diagonal, mostly predicates, selects
// and address math).  Here the staged log-prob arrays are PADDED with a large negative sentinel (-1e30, never -inf:
// no NaN from inf - inf, no special cases) - `pad` rows before and after the utterance, one column before, the
// columns beyond U_b - so every lane runs the plain recurrence on every diagonal: cells outside the lattice compute
// sentinel-sized values into padding rows of the alpha/beta arrays and never reach a real cell with a weight above
// 2^-1e30.  Initial conditions are data: lpb[-1][0] = 0 with alpha(-1,0) = 0, and beta(T_b, U_b) = 0.
// Lanes of columns beyond U_b mirror column U_b's addresses and are forced to the sentinel (one select), their
// stores are predicated off by a loop-invariant predicate.
// ---------------------------------------------------------------------------------------------------------------
constexpr float kLatNeg = -1.0e30f;

constexpr int LAT3_THREADS = 1024;               // 2 warps sweep, all 32 stage the log-probs / copy alpha, beta out
template <int NJ>
__global__ void __launch_bounds__(LAT3_THREADS) rnnt_lattice3_kernel(
    const float* __restrict__ lp_blank, const float* __restrict__ lp_label, const int32_t* __restrict__ t_len,
    const int32_t* __restrict__ u_len, float* __restrict__ alpha, float* __restrict__ beta,
    float* __restrict__ costs, int T, int U1, int pitch, int pad) {
  extern __shared__ float sm[];
  const int b = blockIdx.x;
  const int Tb = max(min(t_len[b], T), 0), Ub = max(min(u_len[b], U1 - 1), 0);
  const size_t base = (size_t)b * T * U1;
  if (Tb <= 0) { if (threadIdx.x == 0) costs[b] = 0.f; return; }
  const int W = Ub + 1;
  const int R = T + 2 * pad;                    // rows per array; element (t, u) at (t + pad) * pitch + u + 1
  float* sb = sm;                               // lp_blank * log2e
  float* sl = sm + (size_t)R * pitch;           // lp_label * log2e
  float* sa = sm + (size_t)2 * R * pitch;       // alpha (base 2)
  float* sc = sm + (size_t)3 * R * pitch;       // beta  (base 2)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = LAT3_THREADS >> 5;
  // sentinel fill of the rows the sweeps can touch ([-pad, Tb + pad)), then the utterance's log-probs
  {
    const int nfill = (Tb + 2 * pad) * pitch;
    for (int i = threadIdx.x; i < nfill; i += LAT3_THREADS) { sb[i] = kLatNeg; sl[i] = kLatNeg; }
  }
  __syncthreads();
  {
    const int n = Tb * U1;                      // rows are contiguous in global memory (row pitch U1)
    const float* gb = lp_blank + base;
    const float* gl = lp_label + base;
    for (int i0 = threadIdx.x; i0 < n; i0 += 4 * LAT3_THREADS) {
      float xb[4], xl[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int i = i0 + k * LAT3_THREADS;
        xb[k] = (i < n) ? __ldg(gb + i) : 0.f;
        xl[k] = (i < n) ? __ldg(gl + i) : 0.f;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int i = i0 + k * LAT3_THREADS;
        if (i < n) {
          const int t = i / U1, u = i - t * U1;
          if (u <= Ub) sb[(t + pad) * pitch + u + 1] = fmaxf(xb[k] * kLog2e, kLatNeg);
          if (u < Ub) sl[(t + pad) * pitch + u + 1] = fmaxf(xl[k] * kLog2e, kLatNeg);     // no label leaves column U_b
        }
      }
    }
    if (threadIdx.x == 0) sb[(pad - 1) * pitch + 1] = 0.f;        // lpb[-1][0] = 0: alpha(0,0) = alpha(-1,0) + 0 = 0
  }
  __syncthreads();
  const int ndiag = Tb + Ub;
  const uint32_t s_sb = (uint32_t)__cvta_generic_to_shared(sb), s_sl = (uint32_t)__cvta_generic_to_shared(sl);
  const uint32_t s_sa = (uint32_t)__cvta_generic_to_shared(sa), s_sc = (uint32_t)__cvta_generic_to_shared(sc);
  const uint32_t rowb = (uint32_t)pitch * 4u;
  // opaque to the optimiser: otherwise the shared-window base (S2UR SR_CgaCtaId ...) and the row pitch (LDC) are
  // re-materialised inside the dependent loop
  uint32_t k_sb = s_sb, k_sl = s_sl, k_sa = s_sa, k_sc = s_sc, k_row = rowb;
  asm volatile("" : "+r"(k_sb), "+r"(k_sl), "+r"(k_sa), "+r"(k_sc), "+r"(k_row));
  auto lds = [](uint32_t a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; };
  auto sts = [](uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); };
  auto lse2 = [](float a, float c) {            // log2(2^a + 2^c) for finite operands
    const float m = fmaxf(a, c), n = fminf(a, c);
    return m + lg2f(1.f + ex2f(n - m));
  };
  if (warp == 0) {
    // ---------------- alpha(t,u) = LSE(alpha(t-1,u)+lpb(t-1,u), alpha(t,u-1)+lpl(t,u-1)),  t = d - u
    float prev[NJ], nb[NJ], nl[NJ];
    uint32_t a0[NJ];                            // byte offset of element (t, u) at the current diagonal
    bool col[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int u = lane + 32 * j, uc = min(u, Ub);
      col[j] = u <= Ub;
      prev[j] = (u == 0) ? 0.f : kLatNeg;       // alpha(-1, 0) = 0
      a0[j] = (uint32_t)((0 - uc + pad) * pitch + uc + 1) * 4u;
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) { nb[j] = lds(k_sb + a0[j] - k_row); nl[j] = lds(k_sl + a0[j] - 4u); }
    for (int d = 0; d < ndiag; ++d) {
      float cb[NJ], cl[NJ], left[NJ];
#pragma unroll
      for (int j = 0; j < NJ; ++j) { cb[j] = nb[j]; cl[j] = nl[j]; }
#pragma unroll
      for (int j = 0; j < NJ; ++j) { nb[j] = lds(k_sb + a0[j]); nl[j] = lds(k_sl + a0[j] + k_row - 4u); }   // next diagonal
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        left[j] = __shfl_up_sync(0xffffffffu, prev[j], 1);
        if (j > 0) { const float w = __shfl_sync(0xffffffffu, prev[j - 1], 31); if (lane == 0) left[j] = w; }
        else if (lane == 0) left[j] = kLatNeg;
      }
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        float v = lse2(prev[j] + cb[j], left[j] + cl[j]);
        v = col[j] ? v : kLatNeg;
        if (col[j]) sts(k_sa + a0[j], v);
        prev[j] = v;
        a0[j] += k_row;
      }
    }
  } else if (warp == 1) {
    // ---------------- beta(t,u) = LSE(beta(t+1,u)+lpb(t,u), beta(t,u+1)+lpl(t,u)),  beta(T_b, U_b) = 0
    float prev[NJ], nb[NJ], nl[NJ];
    uint32_t a0[NJ];
    bool col[NJ];
    const int d0 = ndiag - 1;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int u = lane + 32 * j, uc = min(u, Ub);
      col[j] = u <= Ub;
      prev[j] = (u == Ub) ? 0.f : kLatNeg;
      a0[j] = (uint32_t)((d0 - uc + pad) * pitch + uc + 1) * 4u;
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) { nb[j] = lds(k_sb + a0[j]); nl[j] = lds(k_sl + a0[j]); }
    for (int d = d0; d >= 0; --d) {
      float cb[NJ], cl[NJ], right[NJ];
#pragma unroll
      for (int j = 0; j < NJ; ++j) { cb[j] = nb[j]; cl[j] = nl[j]; }
#pragma unroll
      for (int j = 0; j < NJ; ++j) { nb[j] = lds(k_sb + a0[j] - k_row); nl[j] = lds(k_sl + a0[j] - k_row); }   // diagonal d - 1
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        right[j] = __shfl_down_sync(0xffffffffu, prev[j], 1);
        if (j + 1 < NJ) { const float w = __shfl_sync(0xffffffffu, prev[j + 1], 0); if (lane == 31) right[j] = w; }
        else if (lane == 31) right[j] = kLatNeg;
      }
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        float v = lse2(prev[j] + cb[j], right[j] + cl[j]);
        v = col[j] ? v : kLatNeg;
        if (col[j]) sts(k_sc + a0[j], v);
        prev[j] = v;
        a0[j] -= k_row;
      }
    }
    if (lane == 0) costs[b] = -prev[0] * kLn2;     // beta(0,0)
  }
  __syncthreads();
  for (int t = warp; t < Tb; t += nwarp)
    for (int u = lane; u < W; u += 32) {
      alpha[base + (size_t)t * U1 + u] = sa[(t + pad) * pitch + u + 1] * kLn2;
      beta[base + (size_t)t * U1 + u] = sc[(t + pad) * pitch + u + 1] * kLn2;
    }
}

// Fallback for lattices that do not fit shared memory or U1 > 256: one CTA per utterance, block-wide diagonal sweep.
__global__ void rnnt_lattice_generic_kernel(const float* __restrict__ lp_blank, const float* __restrict__ lp_label,
                                            const int32_t* __restrict__ t_len, const int32_t* __restrict__ u_len,
                                            float* __restrict__ alpha, float* __restrict__ beta,
                                            float* __restrict__ costs, int T, int U1) {
  const int b = blockIdx.x;
  const int Tb = max(min(t_len[b], T), 0), Ub = max(min(u_len[b], U1 - 1), 0);
  const size_t base = (size_t)b * T * U1;
  const float* lb = lp_blank + base;
  const float* ll = lp_label + base;
  float* ab = alpha + base;
  float* bb = beta + base;
  if (Tb <= 0) { if (threadIdx.x == 0) costs[b] = 0.f; return; }
  const int ndiag = Tb + Ub;
  for (int d = 0; d < ndiag; ++d) {
    for (int u = threadIdx.x; u <= Ub; u += blockDim.x) {
      int t = d - u;
      if (t < 0 || t >= Tb) continue;
      float v;
      if (d == 0) v = 0.f;
      else {
        float a = (t > 0) ? ab[(t - 1) * U1 + u] + lb[(t - 1) * U1 + u] : kNegInf;
        float c = (u > 0) ? ab[t * U1 + u - 1] + ll[t * U1 + u - 1] : kNegInf;
        v = log_add_exp(a, c);
      }
      ab[t * U1 + u] = v;
    }
    __syncthreads();
  }
  for (int d = ndiag - 1; d >= 0; --d) {
    for (int u = threadIdx.x; u <= Ub; u += blockDim.x) {
      int t = d - u;
      if (t < 0 || t >= Tb) continue;
      float v;
      if (t == Tb - 1 && u == Ub) v = lb[t * U1 + u];
      else {
        float a = (t + 1 < Tb) ? bb[(t + 1) * U1 + u] + lb[t * U1 + u] : kNegInf;
        float c = (u < Ub) ? bb[t * U1 + u + 1] + ll[t * U1 + u] : kNegInf;
        v = log_add_exp(a, c);
      }
      bb[t * U1 + u] = v;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) costs[b] = -bb[0];
}

template <int NJ>
static int launch_lattice(const float* lpb, const float* lpl, const int32_t* t_len, const int32_t* u_len,
                          float* alpha, float* beta, float* costs, int B, int T, int U1, cudaStream_t st) {
  {
    // padded arrays ([T + 2 pad][U1 + 1 rounded up to even]); the unpadded kernel below takes the shapes beyond them
    const int pad3 = U1, pitch3 = (U1 + 2) & ~1;
    const size_t smem3 = (size_t)4 * (T + 2 * pad3) * pitch3 * sizeof(float);
    if (smem3 <= 227 * 1024) {
      CTCVR_CHECK_CUDA(cudaFuncSetAttribute(rnnt_lattice3_kernel<NJ>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)(227 * 1024)));
      rnnt_lattice3_kernel<NJ><<<B, LAT3_THREADS, smem3, st>>>(lpb, lpl, t_len, u_len, alpha, beta, costs, T, U1, pitch3, pad3);
      CTCVR_LAUNCH_CHECK();
      return 0;
    }
  }
  const int pitch = (U1 % 2 == 0) ? U1 : U1 + 1;       // pitch-1 odd => diagonal reads hit distinct banks
  const size_t smem4 = (size_t)4 * T * pitch * sizeof(float);
  if (smem4 <= 220 * 1024) {
    CTCVR_CHECK_CUDA(cudaFuncSetAttribute(rnnt_lattice2_kernel<NJ>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)(220 * 1024)));
    rnnt_lattice2_kernel<NJ><<<B, LAT2_THREADS, smem4, st>>>(lpb, lpl, t_len, u_len, alpha, beta, costs, T, U1, pitch);
    CTCVR_LAUNCH_CHECK();
    return 0;
  }
  // lattices beyond shared memory (T * (U+1) > ~56 k cells): block-wide diagonal sweep on global memory
  rnnt_lattice_generic_kernel<<<B, 256, 0, st>>>(lpb, lpl, t_len, u_len, alpha, beta, costs, T, U1);
  CTCVR_LAUNCH_CHECK();
  return 0;
}

int rnnt_lattice(const float* lpb, const float* lpl, const int32_t* t_len, const int32_t* u_len, float* alpha,
                 float* beta, float* costs, int B, int T, int U1, cudaStream_t st) {
  if (U1 <= 32) return launch_lattice<1>(lpb, lpl, t_len, u_len, alpha, beta, costs, B, T, U1, st);
  if (U1 <= 64) return launch_lattice<2>(lpb, lpl, t_len, u_len, alpha, beta, costs, B, T, U1, st);
  if (U1 <= 128) return launch_lattice<4>(lpb, lpl, t_len, u_len, alpha, beta, costs, B, T, U1, st);
  if (U1 <= 256) return launch_lattice<8>(lpb, lpl, t_len, u_len, alpha, beta, costs, B, T, U1, st);
  rnnt_lattice_generic_kernel<<<B, 256, 0, st>>>(lpb, lpl, t_len, u_len, alpha, beta, costs, T, U1);
  CTCVR_LAUNCH_CHECK();
  return 0;
}

}  // namespace ctcvr
