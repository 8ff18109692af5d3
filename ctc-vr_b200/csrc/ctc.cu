// CTC head tail on B200: log_softmax rows, CTC loss (alpha/beta + gradient wrt logits) and CTC greedy.
//   F.log_softmax(ctc_lo(x)) + nn.CTCLoss(blank, zero_infinity=True):
//     model/rnnt_model.py:52-58, model/online_rnnt_model.py:27-31, model/model.py:289-293
//   ctc_greedy_search: model/rnnt_model.py:188-210, model/online_rnnt_model.py:647-671,
//     wenet/transformer/search.py:107-122
// Algorithmic HBM bytes of the loss: read log-probs once (fwd gather is a subset), write the gradient
// once, alpha scratch written+read: B*T*(2*V + 2*S)*4 B.  The kernel is bound by its T dependent steps.
#include <stdlib.h>

#include "common.cuh"

namespace ctcvr {

// ---------------------------------------------------------------- log_softmax: one warp per row
__global__ void log_softmax_kernel(const float* __restrict__ x, float* __restrict__ y, long rows, int V) {
  long r = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  int lane = threadIdx.x & 31;
  const float* xr = x + r * V;
  float* yr = y + r * V;
  float m = kNegInf;
  for (int v = lane; v < V; v += 32) m = fmaxf(m, xr[v]);
  m = warp_max(m);
  float s = 0.f;
  for (int v = lane; v < V; v += 32) s += expf(xr[v] - m);
  s = warp_sum(s);
  float l = m + logf(s);
  for (int v = lane; v < V; v += 32) yr[v] = xr[v] - l;
}

int log_softmax(const float* x, float* y, long rows, int V, cudaStream_t st) {
  if (rows == 0) return 0;
  log_softmax_kernel<<<cdiv(rows, 8), 256, 0, st>>>(x, y, rows, V);
  CTCVR_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------- CTC loss: one CTA per utterance
// thread s owns extended-label state s (S = 2U+1).  alpha is kept in the workspace [B][T][Sp].
__global__ void ctc_loss_kernel(const float* __restrict__ lp, const int64_t* __restrict__ targets,
                                const int32_t* __restrict__ in_lens, const int32_t* __restrict__ tgt_lens,
                                const float* __restrict__ grad_scale, float* __restrict__ nll_out,
                                float* __restrict__ grad, float* __restrict__ alpha_ws, int T, int V, int Umax,
                                int Sp, int blank, int zero_infinity) {
  extern __shared__ float sm[];
  const int b = blockIdx.x, s = threadIdx.x, nthr = blockDim.x;
  // lengths beyond the tensors cannot index outside them; a negative length behaves exactly like 0
  const int Tb = max(min(in_lens[b], T), 0), Ub = max(min(tgt_lens[b], Umax), 0);
  const int S = 2 * Ub + 1;
  float* cur = sm;                  // [Sp] alpha_{t} / beta_{t} exchange
  float* ab = cur + Sp;             // [Sp] alpha+beta at time t
  float* lc = ab + Sp;              // [Sp] per-leader log-sum of alpha+beta
  float* red = lc + Sp;             // [32]
  int* slot = reinterpret_cast<int*>(red + 32);    // [V] label -> leader state (-1: not in l')
  int* nxt = slot + V;              // [Sp] next state with the same label (-1: none)
  const float* lpb = lp + (size_t)b * T * V;
  float* ga = alpha_ws + (size_t)b * T * Sp;
  float* gb = grad ? grad + (size_t)b * T * V : nullptr;

  // label of odd state q; an out-of-range label (undefined in the reference) is blank: no stray index, and every
  // rule below (skips, label chains) sees the same label the split form does
  auto label = [&](int q) {
    const int l = (int)targets[(size_t)b * Umax + (q >> 1)];
    return (unsigned)l < (unsigned)V ? l : blank;
  };
  const int lab = (s < S && (s & 1)) ? label(s) : blank;
  bool skip_ok = false;             // may take the s-2 transition
  if (s < S && (s & 1) && s >= 2) skip_ok = (lab != label(s - 2));

  // label -> leader map, same-label chains (leader = lowest state carrying the label)
  for (int v = s; v < V; v += nthr) slot[v] = -1;
  if (s < Sp) nxt[s] = -1;
  __syncthreads();
  if (s == 0) {
    slot[blank] = 0;                // all even states: handled by a block reduction, leader 0; odd blank states chain from 0
    for (int q = 1; q < S; q += 2) {
      const int l = label(q);
      if (slot[l] < 0) slot[l] = q;
      else { int p = slot[l]; while (nxt[p] >= 0) p = nxt[p]; nxt[p] = q; }
    }
  }
  __syncthreads();

  float nll;
  if (Tb == 0) {
    nll = (Ub == 0) ? 0.f : INFINITY;
  } else {
    // ---- alpha
    float a = kNegInf;
    if (s < S && s < 2) a = lpb[lab];
    if (s < Sp) { cur[s] = a; ga[s] = a; }
    float lnext = (s < S && Tb > 1) ? lpb[(size_t)V + lab] : 0.f;
    __syncthreads();
    for (int t = 1; t < Tb; ++t) {
      float lcur = lnext;
      if (s < S && t + 1 < Tb) lnext = lpb[(size_t)(t + 1) * V + lab];
      float v = kNegInf;
      if (s < S) {
        v = cur[s];
        if (s >= 1) v = log_add_exp(v, cur[s - 1]);
        if (skip_ok) v = log_add_exp(v, cur[s - 2]);
        v = (v == kNegInf) ? kNegInf : v + lcur;
      }
      __syncthreads();
      if (s < Sp) { cur[s] = v; ga[(size_t)t * Sp + s] = v; }
      __syncthreads();
    }
    float ll = cur[S - 1];
    if (S > 1) ll = log_add_exp(ll, cur[S - 2]);
    nll = -ll;
  }
  bool inf = !(nll < INFINITY);
  if (inf && zero_infinity) nll = 0.f;
  if (s == 0) nll_out[b] = nll;
  if (!gb) return;
  const float scale = grad_scale ? grad_scale[b] : 1.f;
  if (inf || Tb == 0) {            // zero gradient everywhere (ATen zero_infinity semantics)
    for (size_t i = s; i < (size_t)T * V; i += nthr) gb[i] = 0.f;
    return;
  }
  // ---- beta + gradient, t descending
  bool skip_fwd = false;           // may take the s+2 transition
  if (s < S && (s & 1) && s + 2 < S) skip_fwd = (lab != label(s + 2));
  __syncthreads();
  float bprev = kNegInf;
  for (int t = Tb - 1; t >= 0; --t) {
    float lcur = (s < S) ? lpb[(size_t)t * V + lab] : 0.f;
    float v = kNegInf;
    if (s < S) {
      if (t == Tb - 1) v = (s >= S - 2) ? lcur : kNegInf;
      else {
        v = cur[s];
        if (s + 1 < S) v = log_add_exp(v, cur[s + 1]);
        if (skip_fwd) v = log_add_exp(v, cur[s + 2]);
        v = (v == kNegInf) ? kNegInf : v + lcur;
      }
    }
    (void)bprev;
    __syncthreads();                // everyone has read cur (beta_{t+1})
    if (s < Sp) {
      cur[s] = v;
      ab[s] = (s < S) ? ga[(size_t)t * Sp + s] + v : kNegInf;
    }
    __syncthreads();
    // leaders gather log-sum over their label's states
    if (s < S && (s & 1) && slot[lab] == s) {
      float acc = ab[s];
      for (int q = nxt[s]; q >= 0; q = nxt[q]) acc = log_add_exp(acc, ab[q]);
      lc[s] = acc;
    }
    {   // blank: block log-sum-exp over even states, then the odd states labelled blank
      float m = (s < S && !(s & 1)) ? ab[s] : kNegInf;
      float wm = warp_max(m);
      if ((s & 31) == 0) red[s >> 5] = wm;
      __syncthreads();
      float bm = kNegInf;
      for (int w = 0; w < (nthr >> 5); ++w) bm = fmaxf(bm, red[w]);
      __syncthreads();
      float e = (s < S && !(s & 1) && bm != kNegInf) ? expf(ab[s] - bm) : 0.f;
      float ws_ = warp_sum(e);
      if ((s & 31) == 0) red[s >> 5] = ws_;
      __syncthreads();
      if (s == 0) {
        float tot = 0.f;
        for (int w = 0; w < (nthr >> 5); ++w) tot += red[w];
        float acc = (bm == kNegInf) ? kNegInf : bm + logf(tot);
        for (int q = nxt[0]; q >= 0; q = nxt[q]) acc = log_add_exp(acc, ab[q]);
        lc[0] = acc;
      }
      __syncthreads();
    }
    const float* lrow = lpb + (size_t)t * V;
    float* grow = gb + (size_t)t * V;
    for (int vv = s; vv < V; vv += nthr) {
      float l = lrow[vv];
      float g = expf(l);
      int q = slot[vv];
      if (q >= 0 && lc[q] != kNegInf) g -= expf(lc[q] - l + nll);
      grow[vv] = g * scale;
    }
  }
  for (size_t i = (size_t)Tb * V + s; i < (size_t)T * V; i += nthr) gb[i] = 0.f;
}

// ---------------------------------------------------------------- CTC loss, split form (default)
// The kernel above keeps everything of a time step on one CTA's critical path (6 block barriers, a dependent global
// load and the V-wide gradient row per step: 2.9 us per step at T = 500).  Split form:
//   kernel A (one CTA per utterance): the log-probs the DP needs, lp[t][label(s)], are gathered into shared memory
//     once (T x S floats, -1e30 sentinel instead of -inf so the recurrences have no special cases);
//     alpha (warps 0..) and beta (the next warps) then sweep concurrently, one named barrier per step each, and store
//     alpha / beta [T][Sp] to the workspace together with the same-label chains of the extended label sequence;
//   kernel B (one warp per (b, t) row, fully parallel): per-label log-sum of alpha + beta, then the gradient row.
constexpr float kCtcNeg = -1.0e30f;
constexpr float kCtcLog2e = 1.4426950408889634f, kCtcLn2 = 0.6931471805599453f;
__device__ __forceinline__ float ctc_ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float ctc_lg2(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// log(e^a + e^b + e^c) for finite operands.  Natural-log domain on purpose: the log-probs are added exactly (a base-2
// DP would round lp * log2e, an error proportional to |lp|, at every step); the base change multiplies the small
// differences a - m (exact by Sterbenz for the terms that matter), never the large magnitudes.
__device__ __forceinline__ float ctc_lse3(float a, float b, float c) {
  const float m = fmaxf(a, fmaxf(b, c));
  const float e = ctc_ex2((a - m) * kCtcLog2e) + ctc_ex2((b - m) * kCtcLog2e) + ctc_ex2((c - m) * kCtcLog2e);
  return fmaf(ctc_lg2(e), kCtcLn2, m);
}

struct CtcWs {
  float* alpha;   // [B][T][Sp]
  float* beta;    // [B][T][Sp]
  int* meta;      // [B][3][Sp]: label of state s | next state with the same label (-1) | 1 if s is the first of its label
  int* flags;     // [B] 1: no valid alignment (nll = inf) or empty input -> zero gradient
};
static CtcWs carve_ctc_ws(void* ws, int B, int T, int Sp) {
  CtcWs w;
  w.alpha = reinterpret_cast<float*>(ws);
  w.beta = w.alpha + (size_t)B * T * Sp;
  w.meta = reinterpret_cast<int*>(w.beta + (size_t)B * T * Sp);
  w.flags = w.meta + (size_t)B * 3 * Sp;
  return w;
}

// NJ > 0: ONE warp per direction, lane l owns the NJ consecutive states l*NJ .. l*NJ+NJ-1 (Sp = 32 NJ), so the neighbours
// s-1 / s-2 (alpha) and s+1 / s+2 (beta) are registers of the same lane or two shuffles away - no shared-memory exchange and
// no barrier on the T dependent steps (the barrier form below, NJ = 0, spent ~500 cycles per step on a chain of ~170).
// Same operations per state as the barrier form, in the same order: bit-identical alpha / beta.
template <int NJ>
__global__ void ctc_alpha_beta_kernel(const float* __restrict__ lp, const int64_t* __restrict__ targets,
                                      const int32_t* __restrict__ in_lens, const int32_t* __restrict__ tgt_lens,
                                      float* __restrict__ nll_out, float* __restrict__ alpha_ws,
                                      float* __restrict__ beta_ws, int* __restrict__ meta, int* __restrict__ flags,
                                      int T, int V, int Umax, int Sp, int blank, int zero_infinity) {
  extern __shared__ float sm[];
  const int b = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
  // lengths beyond the tensors cannot index outside them; a negative length behaves exactly like 0
  const int Tb = max(min(in_lens[b], T), 0), Ub = max(min(tgt_lens[b], Umax), 0);
  const int S = 2 * Ub + 1;
  float* sel = sm;                               // [Tb][S]  lp[t][label(s)]
  float* ca = sel + (size_t)T * S;               // [2][Sp + 4] alpha exchange, two guard cells on each side
  float* cb = ca + 2 * (Sp + 4);                 // [2][Sp + 4] beta exchange
  int* slot = reinterpret_cast<int*>(cb + 2 * (Sp + 4));   // [V] label -> first state carrying it
  int* lab_s = slot + V;                         // [Sp]
  int* nxt = lab_s + Sp;                         // [Sp]
  const float* lpb = lp + (size_t)b * T * V;
  const int grp = tid / Sp, s = tid - grp * Sp;  // group 0: alpha, group 1: beta
  int* mb = meta + (size_t)b * 3 * Sp;

  for (int i = tid; i < Sp; i += nthr) {
    int l = blank;
    if (i < S && (i & 1)) l = (int)targets[(size_t)b * Umax + (i >> 1)];
    if ((unsigned)l >= (unsigned)V) l = blank;      // out-of-range label (undefined in the reference): no stray index
    lab_s[i] = l;
    nxt[i] = -1;
  }
  for (int v = tid; v < V; v += nthr) slot[v] = -1;
  __syncthreads();
  if (tid == 0) {
    for (int q = 1; q < S; q += 2) {
      const int l = lab_s[q];
      if (slot[l] < 0) slot[l] = q;
      else { int pp = slot[l]; while (nxt[pp] >= 0) pp = nxt[pp]; nxt[pp] = q; }
    }
  }
  // gather: every thread, fully parallel loads
  for (int i = tid; i < Tb * S; i += nthr) {
    const int t = i / S, q = i - t * S;
    sel[i] = fmaxf(lpb[(size_t)t * V + lab_s[q]], kCtcNeg);
  }
  for (int i = tid; i < 2 * (Sp + 4); i += nthr) { ca[i] = kCtcNeg; cb[i] = kCtcNeg; }
  __syncthreads();
  for (int i = tid; i < Sp; i += nthr) {
    mb[i] = lab_s[i];
    mb[Sp + i] = nxt[i];
    mb[2 * Sp + i] = (i < S && (i & 1) && slot[lab_s[i]] == i) ? 1 : 0;
  }
  if (Tb == 0) {
    if (tid == 0) {
      const bool inf = Ub != 0;
      nll_out[b] = inf ? (zero_infinity ? 0.f : INFINITY) : 0.f;
      flags[b] = 1;
    }
    return;
  }
  float* ga = alpha_ws + (size_t)b * T * Sp;
  float* gbt = beta_ws + (size_t)b * T * Sp;
  if (NJ > 0) {
    const int warp = tid >> 5, lane = tid & 31;
    if (warp > 1) return;
    constexpr int NQ = NJ > 0 ? NJ : 1;
    const int s0 = lane * NQ;
    bool live[NQ], skp[NQ];
    float prev[NQ], xn[NQ];
    if (warp == 0) {
      // ---- alpha_t(s) = lse(alpha_{t-1}(s), alpha_{t-1}(s-1), [alpha_{t-1}(s-2)]) + lp_t(label(s))
#pragma unroll
      for (int i = 0; i < NQ; ++i) {
        const int q = s0 + i;
        live[i] = q < S;
        skp[i] = (q < S && (q & 1) && q >= 2) && (lab_s[q] != lab_s[q - 2]);
        prev[i] = (live[i] && q < 2) ? sel[q] : kCtcNeg;
        ga[q] = prev[i];
        xn[i] = (live[i] && Tb > 1) ? sel[S + q] : kCtcNeg;
      }
      for (int t = 1; t < Tb; ++t) {
        float x[NQ];
#pragma unroll
        for (int i = 0; i < NQ; ++i) x[i] = xn[i];
        if (t + 1 < Tb) {
#pragma unroll
          for (int i = 0; i < NQ; ++i) xn[i] = live[i] ? sel[(t + 1) * S + s0 + i] : kCtcNeg;     // next step's log-probs
        }
        // states s0 - 1 and s0 - 2 live in the lane below
        float m1 = __shfl_up_sync(0xffffffffu, prev[NQ - 1], 1);
        float m2 = (NQ >= 2) ? __shfl_up_sync(0xffffffffu, prev[NQ >= 2 ? NQ - 2 : 0], 1) : __shfl_up_sync(0xffffffffu, prev[0], 2);
        if (lane == 0) { m1 = kCtcNeg; m2 = kCtcNeg; }
        if (NQ == 1 && lane == 1) m2 = kCtcNeg;
        float nv[NQ];
#pragma unroll
        for (int i = 0; i < NQ; ++i) {
          const float a1 = (i >= 1) ? prev[i >= 1 ? i - 1 : 0] : m1;
          const float a2 = (i >= 2) ? prev[i >= 2 ? i - 2 : 0] : (i == 1 ? m1 : m2);
          float v = ctc_lse3(prev[i], a1, skp[i] ? a2 : kCtcNeg) + x[i];
          nv[i] = live[i] ? fmaxf(v, kCtcNeg) : kCtcNeg;
        }
#pragma unroll
        for (int i = 0; i < NQ; ++i) { prev[i] = nv[i]; ga[(size_t)t * Sp + s0 + i] = nv[i]; }
      }
      // log-likelihood = lse(alpha_{T-1}(S-1), alpha_{T-1}(S-2)): fetch the two states from their lanes
      float a1 = kCtcNeg, a2 = kCtcNeg;
#pragma unroll
      for (int i = 0; i < NQ; ++i) {
        const float v1 = __shfl_sync(0xffffffffu, prev[i], (S - 1) / NQ);
        const float v2 = __shfl_sync(0xffffffffu, prev[i], S > 1 ? (S - 2) / NQ : 0);
        if ((S - 1) % NQ == i) a1 = v1;
        if (S > 1 && (S - 2) % NQ == i) a2 = v2;
      }
      if (lane == 0) {
        const float ll = ctc_lse3(a1, a2, kCtcNeg);
        const bool inf = ll < -1.0e29f;
        nll_out[b] = inf ? (zero_infinity ? 0.f : INFINITY) : -ll;
        flags[b] = inf ? 1 : 0;
      }
    } else {
      // ---- beta_t(s) = lse(beta_{t+1}(s), beta_{t+1}(s+1), [beta_{t+1}(s+2)]) + lp_t(label(s))
#pragma unroll
      for (int i = 0; i < NQ; ++i) {
        const int q = s0 + i;
        live[i] = q < S;
        skp[i] = (q < S && (q & 1) && q + 2 < S) && (lab_s[q] != lab_s[q + 2]);
        prev[i] = (live[i] && q >= S - 2) ? sel[(Tb - 1) * S + q] : kCtcNeg;
        gbt[(size_t)(Tb - 1) * Sp + q] = prev[i];
        xn[i] = (live[i] && Tb > 1) ? sel[(Tb - 2) * S + q] : kCtcNeg;
      }
      for (int t = Tb - 2; t >= 0; --t) {
        float x[NQ];
#pragma unroll
        for (int i = 0; i < NQ; ++i) x[i] = xn[i];
        if (t >= 1) {
#pragma unroll
          for (int i = 0; i < NQ; ++i) xn[i] = live[i] ? sel[(t - 1) * S + s0 + i] : kCtcNeg;
        }
        float p1 = __shfl_down_sync(0xffffffffu, prev[0], 1);
        float p2 = (NQ >= 2) ? __shfl_down_sync(0xffffffffu, prev[NQ >= 2 ? 1 : 0], 1) : __shfl_down_sync(0xffffffffu, prev[0], 2);
        if (lane == 31) { p1 = kCtcNeg; p2 = kCtcNeg; }
        if (NQ == 1 && lane == 30) p2 = kCtcNeg;
        float nv[NQ];
#pragma unroll
        for (int i = 0; i < NQ; ++i) {
          const float b1 = (i + 1 < NQ) ? prev[i + 1 < NQ ? i + 1 : 0] : p1;
          const float b2 = (i + 2 < NQ) ? prev[i + 2 < NQ ? i + 2 : 0] : (i + 1 < NQ ? p1 : p2);
          float v = ctc_lse3(prev[i], b1, skp[i] ? b2 : kCtcNeg) + x[i];
          nv[i] = live[i] ? fmaxf(v, kCtcNeg) : kCtcNeg;
        }
#pragma unroll
        for (int i = 0; i < NQ; ++i) { prev[i] = nv[i]; gbt[(size_t)t * Sp + s0 + i] = nv[i]; }
      }
    }
    return;
  }
  const int lab = lab_s[s];
  if (grp == 0) {
    // ---- alpha_t(s) = lse(alpha_{t-1}(s), alpha_{t-1}(s-1), [alpha_{t-1}(s-2)]) + lp_t(label(s))
    const bool skip = (s < S && (s & 1) && s >= 2) && (lab != lab_s[s - 2]);
    const bool live = s < S;
    float v = (live && s < 2) ? sel[s] : kCtcNeg;
    int buf = 0;
    ca[buf * (Sp + 4) + 2 + s] = v;
    ga[s] = v;
    asm volatile("bar.sync 1, %0;" ::"r"(Sp));
    for (int t = 1; t < Tb; ++t) {
      const float* c = ca + buf * (Sp + 4) + 2 + s;
      const float x = live ? sel[t * S + s] : kCtcNeg;
      v = ctc_lse3(c[0], c[-1], skip ? c[-2] : kCtcNeg) + x;
      v = live ? fmaxf(v, kCtcNeg) : kCtcNeg;
      buf ^= 1;
      ca[buf * (Sp + 4) + 2 + s] = v;
      ga[(size_t)t * Sp + s] = v;
      asm volatile("bar.sync 1, %0;" ::"r"(Sp));
    }
    if (s == 0) {
      const float* c = ca + buf * (Sp + 4) + 2;
      const float a1 = c[S - 1], a2 = (S > 1) ? c[S - 2] : kCtcNeg;
      const float ll = ctc_lse3(a1, a2, kCtcNeg);
      const bool inf = ll < -1.0e29f;
      nll_out[b] = inf ? (zero_infinity ? 0.f : INFINITY) : -ll;
      flags[b] = inf ? 1 : 0;
    }
  } else if (grp == 1) {
    // ---- beta_t(s) = lse(beta_{t+1}(s), beta_{t+1}(s+1), [beta_{t+1}(s+2)]) + lp_t(label(s))
    const bool skip = (s < S && (s & 1) && s + 2 < S) && (lab != lab_s[s + 2]);
    const bool live = s < S;
    float v = (live && s >= S - 2) ? sel[(Tb - 1) * S + s] : kCtcNeg;
    int buf = 0;
    cb[buf * (Sp + 4) + 2 + s] = v;
    gbt[(size_t)(Tb - 1) * Sp + s] = v;
    asm volatile("bar.sync 2, %0;" ::"r"(Sp));
    for (int t = Tb - 2; t >= 0; --t) {
      const float* c = cb + buf * (Sp + 4) + 2 + s;
      const float x = live ? sel[t * S + s] : kCtcNeg;
      v = ctc_lse3(c[0], c[1], skip ? c[2] : kCtcNeg) + x;
      v = live ? fmaxf(v, kCtcNeg) : kCtcNeg;
      buf ^= 1;
      cb[buf * (Sp + 4) + 2 + s] = v;
      gbt[(size_t)t * Sp + s] = v;
      asm volatile("bar.sync 2, %0;" ::"r"(Sp));
    }
  }
}

constexpr int CTC_GRAD_ROWS = 8;     // rows per CTA (4 warps x 2)
__global__ void __launch_bounds__(128) ctc_grad_kernel(const float* __restrict__ lp, const int32_t* __restrict__ in_lens,
                                                       const int32_t* __restrict__ tgt_lens,
                                                       const float* __restrict__ grad_scale, const float* __restrict__ nll,
                                                       const float* __restrict__ alpha_ws, const float* __restrict__ beta_ws,
                                                       const int* __restrict__ meta, const int* __restrict__ flags,
                                                       float* __restrict__ grad, int T, int V, int Sp, int blank) {
  extern __shared__ float sm[];
  const int b = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int Tb = max(min(in_lens[b], T), 0), S = min(2 * max(tgt_lens[b], 0) + 1, Sp);
  int* mlab = reinterpret_cast<int*>(sm);        // [3][Sp]
  float* abw = sm + 3 * Sp + warp * Sp;          // [4][Sp] alpha + beta of the warp's row
  float* acc = sm + 7 * Sp + warp * V;           // [4][V] per-label log-sum
  const int* mb = meta + (size_t)b * 3 * Sp;
  for (int i = threadIdx.x; i < 3 * Sp; i += 128) mlab[i] = mb[i];
  __syncthreads();
  const bool dead = flags[b] != 0;
  const float scale = grad_scale ? grad_scale[b] : 1.f;
  const float nllb = nll[b];
  for (int r = warp; r < CTC_GRAD_ROWS; r += 4) {
    const int t = blockIdx.x * CTC_GRAD_ROWS + r;
    if (t >= T) break;
    float* grow = grad + ((size_t)b * T + t) * V;
    if (t >= Tb || dead) {
      for (int v = lane; v < V; v += 32) grow[v] = 0.f;
      continue;
    }
    const float* ar = alpha_ws + ((size_t)b * T + t) * Sp;
    const float* br = beta_ws + ((size_t)b * T + t) * Sp;
    float bm = kCtcNeg;
    for (int q = lane; q < Sp; q += 32) {
      const float x = (q < S) ? ar[q] + br[q] : kCtcNeg;
      abw[q] = x;
      if (!(q & 1)) bm = fmaxf(bm, x);
    }
    for (int v = lane; v < V; v += 32) acc[v] = kCtcNeg;
    __syncwarp();
    // blank: log-sum over the even states
    bm = warp_max(bm);
    float be = 0.f;
    for (int q = 2 * lane; q < S; q += 64) be += ctc_ex2((abw[q] - bm) * kCtcLog2e);
    be = warp_sum(be);
    const float lc_blank = fmaf(ctc_lg2(be), kCtcLn2, bm);
    // labels: the first state of every label sums its chain
    for (int q = 1 + 2 * lane; q < S; q += 64) {
      if (mlab[2 * Sp + q]) {
        float m = abw[q];
        for (int k = mlab[Sp + q]; k >= 0; k = mlab[Sp + k]) m = fmaxf(m, abw[k]);
        float e = 0.f;
        for (int k = q; k >= 0; k = mlab[Sp + k]) e += ctc_ex2((abw[k] - m) * kCtcLog2e);
        acc[mlab[q]] = fmaf(ctc_lg2(e), kCtcLn2, m);
      }
    }
    __syncwarp();
    // blank also labels the odd states whose target is blank (or out of range): their chain sum is acc[blank]
    const float lc_blank_all = ctc_lse3(lc_blank, acc[blank], kCtcNeg);
    const float* lrow = lp + ((size_t)b * T + t) * V;
    for (int v = lane; v < V; v += 32) {
      const float l = lrow[v];
      float g = expf(l);
      const float c = (v == blank) ? lc_blank_all : acc[v];
      if (c > -1.0e29f) g -= expf(c - l + nllb);
      grow[v] = g * scale;
    }
    __syncwarp();
  }
}

size_t ctc_loss_ws_bytes(int B, int T, int Umax) {
  int Sp = (2 * Umax + 1 + 31) / 32 * 32;
  return ((size_t)2 * B * T * Sp + (size_t)3 * B * Sp + B) * sizeof(float) + 256;
}

int ctc_loss(const float* lp, const int64_t* targets, const int32_t* in_lens, const int32_t* tgt_lens,
             const float* grad_scale, float* nll, float* grad, int B, int T, int V, int Umax, int blank,
             int zero_infinity, void* ws, size_t ws_bytes, cudaStream_t st) {
  int Sp = (2 * Umax + 1 + 31) / 32 * 32;
  CTCVR_REQUIRE(Sp <= 1024, "ctc_loss: target length %d too long (2U+1 must be <= 1024)", Umax);
  CTCVR_REQUIRE(ws_bytes >= ctc_loss_ws_bytes(B, T, Umax), "ctc_loss: workspace too small");
  const int Smax = 2 * Umax + 1;
  // split form when the gathered log-probs of one utterance fit in shared memory
  const size_t smemA = ((size_t)T * Smax + 4 * (Sp + 4)) * sizeof(float) + (size_t)(V + 2 * Sp) * sizeof(int);
  if (smemA <= 220 * 1024 && 2 * Sp <= 1024) {
    CtcWs W = carve_ctc_ws(ws, B, T, Sp);
    const int threads = 2 * Sp < 256 ? 256 : 2 * Sp;
#define CTCVR_AB_LAUNCH(NJ_)                                                                                                   \
  do {                                                                                                                       \
    CTCVR_CHECK_CUDA(cudaFuncSetAttribute(ctc_alpha_beta_kernel<NJ_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemA)); \
    ctc_alpha_beta_kernel<NJ_><<<B, threads, smemA, st>>>(lp, targets, in_lens, tgt_lens, nll, W.alpha, W.beta, W.meta, W.flags, \
                                                          T, V, Umax, Sp, blank, zero_infinity);                              \
  } while (0)
    switch (Sp / 32) {                       // states per lane of the shuffle form; longer targets take the barrier form
      case 1: CTCVR_AB_LAUNCH(1); break;
      case 2: CTCVR_AB_LAUNCH(2); break;
      case 3: CTCVR_AB_LAUNCH(3); break;
      case 4: CTCVR_AB_LAUNCH(4); break;
      case 5: CTCVR_AB_LAUNCH(5); break;
      case 6: CTCVR_AB_LAUNCH(6); break;
      case 7: CTCVR_AB_LAUNCH(7); break;
      case 8: CTCVR_AB_LAUNCH(8); break;
      default: CTCVR_AB_LAUNCH(0); break;
    }
#undef CTCVR_AB_LAUNCH
    CTCVR_LAUNCH_CHECK();
    if (grad) {
      const size_t smemB = ((size_t)7 * Sp + (size_t)4 * V) * sizeof(float);
      CTCVR_REQUIRE(smemB <= 200 * 1024, "ctc_loss: vocabulary %d too large", V);
      CTCVR_CHECK_CUDA(cudaFuncSetAttribute(ctc_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemB));
      ctc_grad_kernel<<<dim3(cdiv(T, CTC_GRAD_ROWS), B), 128, smemB, st>>>(lp, in_lens, tgt_lens, grad_scale, nll, W.alpha, W.beta,
                                                                            W.meta, W.flags, grad, T, V, Sp, blank);
      CTCVR_LAUNCH_CHECK();
    }
    return 0;
  }
  int threads = Sp < 64 ? 64 : Sp;
  size_t smem = (size_t)(3 * Sp + 32) * sizeof(float) + (size_t)(V + Sp) * sizeof(int);
  CTCVR_REQUIRE(smem <= 200 * 1024, "ctc_loss: vocabulary %d too large", V);
  CTCVR_CHECK_CUDA(cudaFuncSetAttribute(ctc_loss_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ctc_loss_kernel<<<B, threads, smem, st>>>(lp, targets, in_lens, tgt_lens, grad_scale, nll, grad,
                                            reinterpret_cast<float*>(ws), T, V, Umax, Sp, blank, zero_infinity);
  CTCVR_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------- CTC greedy (A10)
// Two launches.  (1) argmax of every frame, one warp per frame, frames of all utterances spread over the whole GPU (one
// CTA per utterance - the first version - left 116 of 148 SMs idle at B = 32 and walked 62 frames per warp in sequence:
// 130 us for 26 MB).  First maximum = lowest index on ties, as torch.argmax / topk(1).  The ids land in the output token
// array itself.  (2) collapse in place, one warp per utterance: keep[t] = id != blank && id != id[t-1], ordered
// compaction by ballot; a 32-frame group is read before anything of it is overwritten and writes only go to positions
// <= the ones already read.
constexpr int GREEDY_FRAMES_PER_CTA = 8;         // 8 warps, one frame each
__global__ void __launch_bounds__(256) ctc_argmax_kernel(const float* __restrict__ scores, const int32_t* __restrict__ lens,
                                                         int32_t* __restrict__ ids, int T, int V) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.y, t = blockIdx.x * GREEDY_FRAMES_PER_CTA + warp;
  if (t >= max(min(lens[b], T), 0)) return;
  const float* x = scores + ((size_t)b * T + t) * V;
  float best = kNegInf;
  int bi = V;
  if ((V & 3) == 0 && ((reinterpret_cast<uintptr_t>(x) & 15u) == 0)) {
    for (int v = 4 * lane; v < V; v += 128) {          // ascending within the lane: the first maximum survives
      const float4 q = __ldg(reinterpret_cast<const float4*>(x + v));
      if (q.x > best) { best = q.x; bi = v; }
      if (q.y > best) { best = q.y; bi = v + 1; }
      if (q.z > best) { best = q.z; bi = v + 2; }
      if (q.w > best) { best = q.w; bi = v + 3; }
    }
  } else {
    for (int v = lane; v < V; v += 32) {
      const float xv = x[v];
      if (xv > best) { best = xv; bi = v; }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  if (lane == 0) ids[(size_t)b * T + t] = bi;
}

__global__ void __launch_bounds__(128) ctc_collapse_kernel(const int32_t* __restrict__ lens, int32_t* __restrict__ tokens,
                                                           int32_t* __restrict__ out_lens, int B, int T, int blank) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  const int Tb = max(min(lens[b], T), 0);
  int32_t* row = tokens + (size_t)b * T;
  int count = 0, carry = -1;                      // carry = id of the frame in front of the group
  for (int t0 = 0; t0 < Tb; t0 += 32) {
    const int t = t0 + lane;
    const int id = (t < Tb) ? row[t] : blank;
    int prev = __shfl_up_sync(0xffffffffu, id, 1);
    if (lane == 0) prev = carry;
    carry = __shfl_sync(0xffffffffu, id, 31);
    const bool keep = (t < Tb) && (id != blank) && (id != prev);
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    __syncwarp();                                 // every lane holds its id before the group is overwritten
    if (keep) row[count + __popc(m & ((1u << lane) - 1))] = id;
    count += __popc(m);
  }
  if (lane == 0) out_lens[b] = count;
}

int ctc_greedy(const float* scores, const int32_t* lens, int32_t* out_tokens, int32_t* out_lens, int B, int T, int V,
               int blank, cudaStream_t st) {
  if (B == 0) return 0;
  ctc_argmax_kernel<<<dim3(cdiv(T, GREEDY_FRAMES_PER_CTA), B), 256, 0, st>>>(scores, lens, out_tokens, T, V);
  CTCVR_LAUNCH_CHECK();
  ctc_collapse_kernel<<<cdiv(B, 4), 128, 0, st>>>(lens, out_tokens, out_lens, B, T, blank);
  CTCVR_LAUNCH_CHECK();
  return 0;
}

}  // namespace ctcvr
