// Forced alignment: the Viterbi (max-plus) forms of the RNN-T lattice and of the CTC alpha recursion, with a backtrace
// on the device.  The recursions are the alpha halves of csrc/lattice.cu and csrc/ctc.cu with log-add replaced by max;
// every step also records which predecessor won, and one thread walks those decisions back from the terminal cell.
//
// Values that cannot be a path: log-probs are clamped to >= -1e30 (a sentinel, never -inf, so no inf - inf and no
// special cases on the dependent chain) and every recursion value to >= -1e30.  A best path scoring below -1e29 runs
// through a -inf log-prob or does not exist (T_b = 0, or a CTC target longer than the frames allow): the utterance gets
// score -inf and -1 in every frame / label / span entry.  Lengths are clamped to the tensor extents (negative = 0) and a
// CTC label outside [0, V) reads as blank, exactly as the loss kernels clamp them.  Nothing is read back on the host.
//
// Tie-breaking (exact fp32 ties):
//   RNN-T: the blank predecessor (t-1, u) wins, so a label is emitted at the earliest frame among equal paths.
//   CTC:   the smaller jump wins (stay over s-1 over s-2); of the two end states, S-1 (final blank) wins.
#include <stdlib.h>

#include "common.cuh"

namespace ctcvr {

constexpr float kAlnNeg = -1.0e30f;     // clamp of log-probs and recursion values
constexpr float kAlnDead = -1.0e29f;    // a best path below this has no finite log-probability
constexpr int VIT_THREADS = 256;        // all threads stage and initialise; one warp runs the recursion (shared forms)

// ---------------------------------------------------------------------------------------------------------------
// RNN-T.  delta(0,0) = 0, delta(t,u) = max(delta(t-1,u) + lpb(t-1,u), delta(t,u-1) + lpl(t,u-1)); score =
// delta(T_b-1,U_b) + lpb(T_b-1,U_b).  Decision bits are packed by anti-diagonal: word dec[d * W + u / 32], bit u % 32,
// is 1 when cell (d - u, u) came from its label predecessor (t, u-1).  Both kernel forms write this layout (the shared
// form has W = NJ, one ballot per column group; the workspace form W = ceil(U1 / 32), one ballot per warp).
// frames[u] = frame at which label u is emitted, token_lp[u] = lpl at that cell; `lpl` / `pitch` address the clamped
// label log-probs (staged rows or the input).
__device__ void rnnt_backtrace(const uint32_t* dec, int W, int Tb, int Ub, const float* lpl, int pitch, int32_t* frames,
                               float* token_lp) {
  int t = Tb - 1, u = Ub;
  while (u > 0) {
    const bool lab = t == 0 || ((dec[(size_t)(t + u) * W + (u >> 5)] >> (u & 31)) & 1u);
    if (lab) {
      --u;
      frames[u] = t;
      token_lp[u] = fmaxf(lpl[(size_t)t * pitch + u], kAlnNeg);
    } else {
      --t;
    }
  }
}

// Shared form, modelled on rnnt_lattice2/3_kernel: one CTA per utterance, the utterance's log-probs staged once into
// shared memory (pitch even: the diagonal reads of a warp hit distinct banks), then warp 0 sweeps the anti-diagonals with
// lane-owned columns u = lane + 32 j; the left neighbour comes from the adjacent lane by shuffle, so no barrier is needed
// per diagonal.  Decisions are ballots stored to shared memory; lane 0 backtraces.
template <int NJ>
__global__ void __launch_bounds__(VIT_THREADS) rnnt_viterbi_kernel(
    const float* __restrict__ lp_blank, const float* __restrict__ lp_label, const int32_t* __restrict__ t_len,
    const int32_t* __restrict__ u_len, int32_t* __restrict__ frames, float* __restrict__ token_lp,
    float* __restrict__ scores, int T, int U1, int pitch) {
  extern __shared__ float sm[];
  const int b = blockIdx.x, U = U1 - 1;
  const int Tb = max(min(t_len[b], T), 0), Ub = max(min(u_len[b], U), 0);
  int32_t* fr = frames + (size_t)b * U;
  float* tk = token_lp + (size_t)b * U;
  for (int u = threadIdx.x; u < U; u += VIT_THREADS) { fr[u] = -1; tk[u] = 0.f; }
  if (Tb == 0) { if (threadIdx.x == 0) scores[b] = kNegInf; return; }
  float* sb = sm;                                             // [T][pitch] lp_blank
  float* sl = sm + (size_t)T * pitch;                         // [T][pitch] lp_label
  uint32_t* dec = reinterpret_cast<uint32_t*>(sl + (size_t)T * pitch);   // [T + U1][NJ]
  const size_t base = (size_t)b * T * U1;
  const int n = Tb * U1;
  for (int i = threadIdx.x; i < n; i += VIT_THREADS) {
    const int t = i / U1, u = i - t * U1;
    if (u <= Ub) sb[t * pitch + u] = fmaxf(__ldg(lp_blank + base + i), kAlnNeg);
    if (u < Ub) sl[t * pitch + u] = fmaxf(__ldg(lp_label + base + i), kAlnNeg);
  }
  __syncthreads();                                            // also orders the -1 fill before the backtrace's stores
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  float prev[NJ];
  bool col[NJ];
#pragma unroll
  for (int j = 0; j < NJ; ++j) { prev[j] = kAlnNeg; col[j] = lane + 32 * j <= Ub; }
  const int nd = Tb + Ub;
  for (int d = 0; d < nd; ++d) {
    float left[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {                            // column u-1 on diagonal d-1 = cell (t, u-1)
      left[j] = __shfl_up_sync(0xffffffffu, prev[j], 1);
      if (j > 0) { const float w = __shfl_sync(0xffffffffu, prev[j > 0 ? j - 1 : 0], 31); if (lane == 0) left[j] = w; }
      else if (lane == 0) left[j] = kAlnNeg;
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int u = lane + 32 * j, t = d - u;
      const bool in = col[j] && (unsigned)t < (unsigned)Tb;
      const bool okb = in && t > 0, okl = in && u > 0;
      const float cb = sb[okb ? (t - 1) * pitch + u : 0], cl = sl[okl ? t * pitch + u - 1 : 0];
      const float xa = okb ? prev[j] + cb : kAlnNeg;
      const float xb = okl ? left[j] + cl : kAlnNeg;
      const bool lab = xb > xa;                               // exact tie: blank predecessor
      float v = lab ? xb : xa;
      v = (d == 0 && u == 0) ? 0.f : v;
      v = in ? fmaxf(v, kAlnNeg) : kAlnNeg;
      const unsigned bits = __ballot_sync(0xffffffffu, lab);
      if (lane == j) dec[d * NJ + j] = bits;
      prev[j] = v;
    }
  }
  float fin = kAlnNeg;                                        // delta(T_b - 1, U_b): column U_b of the last diagonal
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const float x = __shfl_sync(0xffffffffu, prev[j], Ub & 31);
    if (j == (Ub >> 5)) fin = x;
  }
  __syncwarp();
  if (lane != 0) return;
  const float score = fin + sb[(Tb - 1) * pitch + Ub];
  if (!(score >= kAlnDead)) { scores[b] = kNegInf; return; }
  scores[b] = score;
  rnnt_backtrace(dec, NJ, Tb, Ub, sl, pitch, fr, tk);
}

// Workspace form: lattices beyond shared memory or U1 > 256.  One CTA per utterance, block-wide diagonal sweep on the
// input log-probs; the two live diagonals of delta and the decision bits live in the workspace.
__global__ void __launch_bounds__(256) rnnt_viterbi_ws_kernel(
    const float* __restrict__ lp_blank, const float* __restrict__ lp_label, const int32_t* __restrict__ t_len,
    const int32_t* __restrict__ u_len, int32_t* __restrict__ frames, float* __restrict__ token_lp,
    float* __restrict__ scores, int T, int U1, uint32_t* dec_ws, float* ring_ws) {
  const int b = blockIdx.x, U = U1 - 1, W = (U1 + 31) / 32;
  const int Tb = max(min(t_len[b], T), 0), Ub = max(min(u_len[b], U), 0);
  const int lane = threadIdx.x & 31;
  int32_t* fr = frames + (size_t)b * U;
  float* tk = token_lp + (size_t)b * U;
  for (int u = threadIdx.x; u < U; u += blockDim.x) { fr[u] = -1; tk[u] = 0.f; }
  if (Tb == 0) { if (threadIdx.x == 0) scores[b] = kNegInf; return; }
  const float* gb = lp_blank + (size_t)b * T * U1;
  const float* gl = lp_label + (size_t)b * T * U1;
  uint32_t* dec = dec_ws + (size_t)b * (T + U1) * W;
  float* ring = ring_ws + (size_t)b * 2 * U1;                 // [2][U1]: diagonals d-1 and d
  const int nd = Tb + Ub;
  for (int d = 0; d < nd; ++d) {
    const float* rp = ring + ((d + 1) & 1) * U1;
    float* rc = ring + (d & 1) * U1;
    for (int u0 = 0; u0 <= Ub; u0 += blockDim.x) {            // the same trip count for every thread: full-warp ballots
      const int u = u0 + threadIdx.x, t = d - u;
      const bool in = u <= Ub && (unsigned)t < (unsigned)Tb;
      const bool okb = in && t > 0, okl = in && u > 0;
      const float xa = okb ? rp[u] + fmaxf(gb[(size_t)(t - 1) * U1 + u], kAlnNeg) : kAlnNeg;
      const float xb = okl ? rp[u - 1] + fmaxf(gl[(size_t)t * U1 + u - 1], kAlnNeg) : kAlnNeg;
      const bool lab = xb > xa;
      float v = lab ? xb : xa;
      v = (d == 0 && u == 0) ? 0.f : v;
      v = in ? fmaxf(v, kAlnNeg) : kAlnNeg;
      const unsigned bits = __ballot_sync(0xffffffffu, lab);
      if (lane == 0 && (u >> 5) < W) dec[(size_t)d * W + (u >> 5)] = bits;
      if (u <= Ub) rc[u] = v;
    }
    __syncthreads();
  }
  if (threadIdx.x != 0) return;
  const float score = ring[((nd - 1) & 1) * U1 + Ub] + fmaxf(gb[(size_t)(Tb - 1) * U1 + Ub], kAlnNeg);
  if (!(score >= kAlnDead)) { scores[b] = kNegInf; return; }
  scores[b] = score;
  rnnt_backtrace(dec, W, Tb, Ub, gl, U1, fr, tk);
}

// The shared form takes U1 <= 256 when both staged arrays and the decision words fit; NJ column groups per lane.
static bool rnnt_viterbi_shared(int T, int U1, int* nj, int* pitch, size_t* smem) {
  if (U1 > 256) return false;
  *nj = U1 <= 32 ? 1 : U1 <= 64 ? 2 : U1 <= 128 ? 4 : 8;
  *pitch = (U1 + 1) & ~1;
  *smem = (size_t)2 * T * *pitch * sizeof(float) + (size_t)(T + U1) * *nj * sizeof(uint32_t);
  return *smem <= 227 * 1024;
}

size_t rnnt_viterbi_ws_bytes(int B, int T, int U1) {
  int nj, pitch;
  size_t smem;
  if (rnnt_viterbi_shared(T, U1, &nj, &pitch, &smem)) return 0;
  const size_t W = (size_t)(U1 + 31) / 32;
  return ((size_t)B * (T + U1) * W + (size_t)B * 2 * U1) * sizeof(uint32_t);
}

int rnnt_viterbi(const float* lpb, const float* lpl, const int32_t* t_len, const int32_t* u_len, int32_t* frames,
                 float* token_lp, float* scores, int B, int T, int U1, void* ws, size_t ws_bytes, cudaStream_t st) {
  int nj, pitch;
  size_t smem;
  if (rnnt_viterbi_shared(T, U1, &nj, &pitch, &smem)) {
#define CTCVR_VIT_LAUNCH(NJ_)                                                                                           \
  do {                                                                                                                  \
    CTCVR_CHECK_CUDA(cudaFuncSetAttribute(rnnt_viterbi_kernel<NJ_>, cudaFuncAttributeMaxDynamicSharedMemorySize,        \
                                          (int)smem));                                                                  \
    rnnt_viterbi_kernel<NJ_><<<B, VIT_THREADS, smem, st>>>(lpb, lpl, t_len, u_len, frames, token_lp, scores, T, U1, pitch); \
  } while (0)
    switch (nj) {
      case 1: CTCVR_VIT_LAUNCH(1); break;
      case 2: CTCVR_VIT_LAUNCH(2); break;
      case 4: CTCVR_VIT_LAUNCH(4); break;
      default: CTCVR_VIT_LAUNCH(8); break;
    }
#undef CTCVR_VIT_LAUNCH
    CTCVR_LAUNCH_CHECK();
    return 0;
  }
  CTCVR_REQUIRE(ws && ws_bytes >= rnnt_viterbi_ws_bytes(B, T, U1), "rnnt_viterbi: workspace too small");
  const size_t W = (size_t)(U1 + 31) / 32;
  uint32_t* dec = reinterpret_cast<uint32_t*>(ws);
  float* ring = reinterpret_cast<float*>(dec + (size_t)B * (T + U1) * W);
  rnnt_viterbi_ws_kernel<<<B, 256, 0, st>>>(lpb, lpl, t_len, u_len, frames, token_lp, scores, T, U1, dec, ring);
  CTCVR_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// CTC.  Extended labels l' (S = 2 U_b + 1, blank at even s); delta_0(s) = lp_0(l'_s) for s < 2, delta_t(s) =
// max(delta_{t-1}(s), delta_{t-1}(s-1), [delta_{t-1}(s-2)]) + lp_t(l'_s), s-2 allowed when l'_s != blank and
// l'_s != l'_{s-2}.  Two backpointer bits per (t, s) = the jump (0, 1, 2), stored as two ballot words.  The backtrace
// writes per frame the label of the state and its log-prob, and per target token its span [first frame, last + 1)
// (torchaudio.functional.merge_tokens' convention).
__device__ __forceinline__ int ctc_label(const int64_t* targets, int b, int Umax, int V, int blank, int s, int S) {
  if (s >= S || !(s & 1)) return blank;
  const int64_t l = targets[(size_t)b * Umax + (s >> 1)];
  return (l >= 0 && l < V) ? (int)l : blank;
}

// jump(t, s): the bit pair of state s at frame t.  `lp_at(t, s)` gives the (clamped) log-prob of the state's label.
template <class Jump, class Lp>
__device__ void ctc_backtrace(int s, int Tb, const int* lab_s, Jump jump, Lp lp_at, int32_t* labels, float* frame_lp,
                              int32_t* spans) {
  int last = -1;
  for (int t = Tb - 1; t >= 0; --t) {
    labels[t] = lab_s[s];
    frame_lp[t] = lp_at(t, s);
    if (s & 1) {
      if (s != last) { spans[(s >> 1) * 2 + 1] = t + 1; last = s; }
      spans[(s >> 1) * 2] = t;
    }
    if (t > 0) s -= jump(t, s);
  }
}

// Shared form, modelled on ctc_alpha_beta_kernel<NJ>: the log-probs the recursion needs, lp[t][l'_s], are gathered into
// shared memory once; then ONE warp runs the recursion, lane l owning states l NJ .. l NJ + NJ - 1, so s-1 / s-2 are
// registers or two shuffles away and there is no barrier on the T dependent steps.
template <int NJ>
__global__ void __launch_bounds__(VIT_THREADS) ctc_viterbi_kernel(
    const float* __restrict__ lp, const int64_t* __restrict__ targets, const int32_t* __restrict__ in_lens,
    const int32_t* __restrict__ tgt_lens, int32_t* __restrict__ labels, float* __restrict__ frame_lp,
    float* __restrict__ scores, int32_t* __restrict__ spans, int T, int V, int Umax, int blank) {
  constexpr int Sp = 32 * NJ;
  extern __shared__ float sm[];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int Tb = max(min(in_lens[b], T), 0), Ub = max(min(tgt_lens[b], Umax), 0);
  const int S = 2 * Ub + 1;
  float* sel = sm;                                                      // [T_b][S] lp[t][l'_s]
  int* lab_s = reinterpret_cast<int*>(sel + (size_t)T * (2 * Umax + 1)); // [Sp]
  uint32_t* bp = reinterpret_cast<uint32_t*>(lab_s + Sp);               // [T][NJ][2]
  int32_t* lab_out = labels + (size_t)b * T;
  float* flp = frame_lp + (size_t)b * T;
  int32_t* sp = spans + (size_t)b * Umax * 2;
  for (int t = tid; t < T; t += VIT_THREADS) { lab_out[t] = -1; flp[t] = 0.f; }
  for (int i = tid; i < 2 * Umax; i += VIT_THREADS) sp[i] = -1;
  for (int i = tid; i < Sp; i += VIT_THREADS) lab_s[i] = ctc_label(targets, b, Umax, V, blank, i, S);
  if (Tb == 0) { if (tid == 0) scores[b] = kNegInf; return; }
  __syncthreads();
  const float* lpb = lp + (size_t)b * T * V;
  for (int i = tid; i < Tb * S; i += VIT_THREADS) {
    const int t = i / S, q = i - t * S;
    sel[i] = fmaxf(lpb[(size_t)t * V + lab_s[q]], kAlnNeg);
  }
  __syncthreads();
  if (tid >= 32) return;
  const int lane = tid, s0 = lane * NJ;
  bool live[NJ], skp[NJ];
  float prev[NJ];
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    const int q = s0 + i;
    live[i] = q < S;
    skp[i] = live[i] && q >= 2 && lab_s[q] != blank && lab_s[q] != lab_s[q - 2];
    prev[i] = (live[i] && q < 2) ? sel[q] : kAlnNeg;
  }
  for (int t = 1; t < Tb; ++t) {
    float x[NJ];
#pragma unroll
    for (int i = 0; i < NJ; ++i) x[i] = live[i] ? sel[t * S + s0 + i] : kAlnNeg;
    // states s0 - 1 and s0 - 2 live in the lane below
    float m1 = __shfl_up_sync(0xffffffffu, prev[NJ - 1], 1);
    float m2 = (NJ >= 2) ? __shfl_up_sync(0xffffffffu, prev[NJ >= 2 ? NJ - 2 : 0], 1) : __shfl_up_sync(0xffffffffu, prev[0], 2);
    if (lane == 0) { m1 = kAlnNeg; m2 = kAlnNeg; }
    if (NJ == 1 && lane == 1) m2 = kAlnNeg;
    float nv[NJ];
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      const float a1 = (i >= 1) ? prev[i >= 1 ? i - 1 : 0] : m1;
      const float a2 = (i >= 2) ? prev[i >= 2 ? i - 2 : 0] : (i == 1 ? m1 : m2);
      float v = prev[i];
      int jump = 0;
      if (a1 > v) { v = a1; jump = 1; }                       // exact tie: the smaller jump
      if (skp[i] && a2 > v) { v = a2; jump = 2; }
      nv[i] = live[i] ? fmaxf(v + x[i], kAlnNeg) : kAlnNeg;
      const unsigned w0 = __ballot_sync(0xffffffffu, jump & 1), w1 = __ballot_sync(0xffffffffu, jump >> 1);
      if (lane == i) { bp[(t * NJ + i) * 2] = w0; bp[(t * NJ + i) * 2 + 1] = w1; }
    }
#pragma unroll
    for (int i = 0; i < NJ; ++i) prev[i] = nv[i];
  }
  float a1 = kAlnNeg, a2 = kAlnNeg;                           // delta(S-1), delta(S-2)
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    const float v1 = __shfl_sync(0xffffffffu, prev[i], (S - 1) / NJ);
    const float v2 = __shfl_sync(0xffffffffu, prev[i], S > 1 ? (S - 2) / NJ : 0);
    if ((S - 1) % NJ == i) a1 = v1;
    if (S > 1 && (S - 2) % NJ == i) a2 = v2;
  }
  __syncwarp();
  if (lane != 0) return;
  const bool end2 = S > 1 && a2 > a1;                         // exact tie: end on the final blank
  const float score = end2 ? a2 : a1;
  if (!(score >= kAlnDead)) { scores[b] = kNegInf; return; }
  scores[b] = score;
  auto jump = [&](int t, int s) {
    const uint32_t* w = bp + (t * NJ + s % NJ) * 2;
    const int l = s / NJ;
    return (int)((w[0] >> l) & 1u) | (int)(((w[1] >> l) & 1u) << 1);
  };
  auto lp_at = [&](int t, int s) { return sel[t * S + s]; };
  ctc_backtrace(end2 ? S - 2 : S - 1, Tb, lab_s, jump, lp_at, lab_out, flp, sp);
}

// Workspace form: Sp > 256 (U > 127) or log-probs beyond shared memory.  Thread s owns state s; the two live frames of
// delta are exchanged through shared memory with one barrier per frame; backpointer words go to the workspace.
__global__ void __launch_bounds__(1024) ctc_viterbi_ws_kernel(
    const float* __restrict__ lp, const int64_t* __restrict__ targets, const int32_t* __restrict__ in_lens,
    const int32_t* __restrict__ tgt_lens, int32_t* __restrict__ labels, float* __restrict__ frame_lp,
    float* __restrict__ scores, int32_t* __restrict__ spans, int T, int V, int Umax, int blank, uint32_t* bp_ws) {
  extern __shared__ float sm[];
  const int b = blockIdx.x, s = threadIdx.x, Sp = blockDim.x, W = Sp / 32, lane = s & 31, warp = s >> 5;
  const int Tb = max(min(in_lens[b], T), 0), Ub = max(min(tgt_lens[b], Umax), 0);
  const int S = 2 * Ub + 1;
  float* cur = sm;                                            // [2][Sp + 2], two guard cells in front of each
  int* lab_s = reinterpret_cast<int*>(cur + 2 * (Sp + 2));    // [Sp]
  uint32_t* bp = bp_ws + (size_t)b * T * W * 2;               // [T][W][2]
  int32_t* lab_out = labels + (size_t)b * T;
  float* flp = frame_lp + (size_t)b * T;
  int32_t* sp = spans + (size_t)b * Umax * 2;
  for (int t = s; t < T; t += Sp) { lab_out[t] = -1; flp[t] = 0.f; }
  for (int i = s; i < 2 * Umax; i += Sp) sp[i] = -1;
  lab_s[s] = ctc_label(targets, b, Umax, V, blank, s, S);
  if (s < 2) { cur[s] = kAlnNeg; cur[Sp + 2 + s] = kAlnNeg; }
  if (Tb == 0) { if (s == 0) scores[b] = kNegInf; return; }
  __syncthreads();
  const float* lpb = lp + (size_t)b * T * V;
  const int lab = lab_s[s];
  const bool live = s < S;
  const bool skp = live && s >= 2 && lab != blank && lab != lab_s[s - 2];
  float v = (live && s < 2) ? fmaxf(lpb[lab], kAlnNeg) : kAlnNeg;
  float xn = (live && Tb > 1) ? fmaxf(lpb[(size_t)V + lab], kAlnNeg) : kAlnNeg;
  int buf = 0;
  cur[2 + s] = v;
  __syncthreads();
  for (int t = 1; t < Tb; ++t) {
    const float x = xn;
    if (live && t + 1 < Tb) xn = fmaxf(lpb[(size_t)(t + 1) * V + lab], kAlnNeg);     // next frame's log-prob
    const float* c = cur + buf * (Sp + 2) + 2 + s;
    float m = c[0];
    int jump = 0;
    if (c[-1] > m) { m = c[-1]; jump = 1; }
    if (skp && c[-2] > m) { m = c[-2]; jump = 2; }
    v = live ? fmaxf(m + x, kAlnNeg) : kAlnNeg;
    const unsigned w0 = __ballot_sync(0xffffffffu, jump & 1), w1 = __ballot_sync(0xffffffffu, jump >> 1);
    if (lane == 0) { bp[((size_t)t * W + warp) * 2] = w0; bp[((size_t)t * W + warp) * 2 + 1] = w1; }
    buf ^= 1;
    cur[buf * (Sp + 2) + 2 + s] = v;
    __syncthreads();
  }
  if (s != 0) return;
  const float* c = cur + buf * (Sp + 2) + 2;
  const float a1 = c[S - 1], a2 = S > 1 ? c[S - 2] : kAlnNeg;
  const bool end2 = S > 1 && a2 > a1;
  const float score = end2 ? a2 : a1;
  if (!(score >= kAlnDead)) { scores[b] = kNegInf; return; }
  scores[b] = score;
  auto jump = [&](int t, int q) {
    const uint32_t* w = bp + ((size_t)t * W + (q >> 5)) * 2;
    return (int)((w[0] >> (q & 31)) & 1u) | (int)(((w[1] >> (q & 31)) & 1u) << 1);
  };
  auto lp_at = [&](int t, int q) { return fmaxf(lpb[(size_t)t * V + lab_s[q]], kAlnNeg); };
  ctc_backtrace(end2 ? S - 2 : S - 1, Tb, lab_s, jump, lp_at, lab_out, flp, sp);
}

static int ctc_viterbi_sp(int Umax) { return (2 * Umax + 1 + 31) / 32 * 32; }

// The shared form takes Sp <= 256 when the gathered log-probs and the backpointer words fit.
static bool ctc_viterbi_shared(int T, int Umax, size_t* smem) {
  const int Sp = ctc_viterbi_sp(Umax), nj = Sp / 32;
  *smem = ((size_t)T * (2 * Umax + 1) + Sp + (size_t)T * nj * 2) * sizeof(float);
  return nj <= 8 && *smem <= 220 * 1024;
}

size_t ctc_viterbi_ws_bytes(int B, int T, int Umax) {
  size_t smem;
  if (ctc_viterbi_shared(T, Umax, &smem)) return 0;
  return (size_t)B * T * (ctc_viterbi_sp(Umax) / 32) * 2 * sizeof(uint32_t);
}

int ctc_viterbi(const float* lp, const int64_t* targets, const int32_t* in_lens, const int32_t* tgt_lens,
                int32_t* labels, float* frame_lp, float* scores, int32_t* spans, int B, int T, int V, int Umax,
                int blank, void* ws, size_t ws_bytes, cudaStream_t st) {
  const int Sp = ctc_viterbi_sp(Umax);
  CTCVR_REQUIRE(Sp <= 1024, "ctc_viterbi: target length %d too long (2U+1 must be <= 1024)", Umax);
  size_t smem;
  if (ctc_viterbi_shared(T, Umax, &smem)) {
#define CTCVR_VIT_LAUNCH(NJ_)                                                                                           \
  do {                                                                                                                  \
    CTCVR_CHECK_CUDA(cudaFuncSetAttribute(ctc_viterbi_kernel<NJ_>, cudaFuncAttributeMaxDynamicSharedMemorySize,         \
                                          (int)smem));                                                                  \
    ctc_viterbi_kernel<NJ_><<<B, VIT_THREADS, smem, st>>>(lp, targets, in_lens, tgt_lens, labels, frame_lp, scores,     \
                                                          spans, T, V, Umax, blank);                                    \
  } while (0)
    switch (Sp / 32) {
      case 1: CTCVR_VIT_LAUNCH(1); break;
      case 2: CTCVR_VIT_LAUNCH(2); break;
      case 3: CTCVR_VIT_LAUNCH(3); break;
      case 4: CTCVR_VIT_LAUNCH(4); break;
      case 5: CTCVR_VIT_LAUNCH(5); break;
      case 6: CTCVR_VIT_LAUNCH(6); break;
      case 7: CTCVR_VIT_LAUNCH(7); break;
      default: CTCVR_VIT_LAUNCH(8); break;
    }
#undef CTCVR_VIT_LAUNCH
    CTCVR_LAUNCH_CHECK();
    return 0;
  }
  CTCVR_REQUIRE(ws && ws_bytes >= ctc_viterbi_ws_bytes(B, T, Umax), "ctc_viterbi: workspace too small");
  const size_t smem_ws = (size_t)(2 * (Sp + 2) + Sp) * sizeof(float);
  ctc_viterbi_ws_kernel<<<B, Sp, smem_ws, st>>>(lp, targets, in_lens, tgt_lens, labels, frame_lp, scores, spans, T, V,
                                                Umax, blank, reinterpret_cast<uint32_t*>(ws));
  CTCVR_LAUNCH_CHECK();
  return 0;
}

}  // namespace ctcvr
