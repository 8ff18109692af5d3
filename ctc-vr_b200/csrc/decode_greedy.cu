// On-device RNN-T greedy search (SURVEY.md §8 A5 / A6 / A6'):
//   model/component/transducer.py:22-70       basic_greedy_search (n_steps=64, fresh state per utterance)
//   model/online_rnnt_model.py:166-222        streaming greedy (n_steps=10, (h,c)/last token carried across chunks)
//   wenet/transducer/search/greedy_search.py:6-54   same walk
// Semantics kept: the stored state is the LSTM state BEFORE feeding the last token; every step feeds
// (last_token, state); argmax over raw logits; blank -> next frame; non-blank -> emit, token <- id,
// state <- state-after-step; at most n_steps iterations per frame.  Because (token, state) only change
// on an emission, the predictor output is cached between blank frames (identical results).
//
// NB utterances advance in lock-step inside one CTA so that each weight element fetched from L2 feeds
// NB FMAs; there is no host synchronisation per step (the reference has one .item() per step).
#include "decode.cuh"

namespace ctcvr {

constexpr int DEC_THREADS = 512;

template <int NB>
__global__ void __launch_bounds__(DEC_THREADS, 1) rnnt_greedy_kernel(
    ctcvr_decoder_weights w, const float* __restrict__ enc_proj, const int32_t* __restrict__ lens,
    float* __restrict__ h_io, float* __restrict__ c_io, int32_t* __restrict__ last_token,
    int32_t* __restrict__ out_tokens, int32_t* __restrict__ out_lens, int N, int T, int max_out, int blank,
    int n_steps) {
  extern __shared__ __align__(16) float smf[];
  DecodeSmem<NB> s;
  s.carve(smf, w, false);
  float* wred_v = smf + DecodeSmem<NB>::floats(w, false);          // [nwarps][NB]
  int* wred_i = reinterpret_cast<int*>(wred_v + (DEC_THREADS / 32) * NB);
  int* tok = wred_i + (DEC_THREADS / 32) * NB;     // [NB] token fed to the predictor
  int* tcur = tok + NB;                            // [NB] current frame
  int* iter = tcur + NB;                           // [NB] iterations spent on the current frame
  int* nout = iter + NB;                           // [NB] tokens emitted
  int* len = nout + NB;                            // [NB]
  int* commit = len + NB;                          // [NB]
  int* flags = commit + NB;                        // [2]: need_pred, any_active

  const int n0 = blockIdx.x * NB;
  const int H = w.H, L = w.L, D = w.D, V = w.V;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  for (int i = tid; i < L * H * NB; i += DEC_THREADS) {
    int n = i % NB, k = (i / NB) % H, l = i / (NB * H);
    int gn = n0 + n;
    float hv = 0.f, cv = 0.f;
    if (gn < N) { hv = h_io[((size_t)l * N + gn) * H + k]; cv = c_io[((size_t)l * N + gn) * H + k]; }
    s.hs[i] = hv; s.cs[i] = cv;
  }
  if (tid < NB) {
    int gn = n0 + tid;
    tok[tid] = (gn < N) ? last_token[gn] : blank;
    len[tid] = (gn < N) ? min(lens[gn], T) : 0;
    tcur[tid] = 0; iter[tid] = 0; nout[tid] = 0; commit[tid] = 0;
  }
  if (tid == 0) { flags[0] = 1; flags[1] = 1; }
  __syncthreads();

  while (true) {
    if (tid == 0) {
      int any = 0;
      for (int n = 0; n < NB; ++n) any |= (tcur[n] < len[n]);
      flags[1] = any;
    }
    __syncthreads();
    if (!flags[1]) break;
    if (flags[0]) predictor_step<NB>(w, s, tok);
    // joint: z = act(enc_proj[t] + pproj)
    const int act = w.activation >> 8;
    for (int i = tid; i < D * NB; i += DEC_THREADS) {
      int d = i / NB, n = i - d * NB;
      float zz = 0.f;
      if (tcur[n] < len[n]) zz = act_rt(act, enc_proj[((size_t)(n0 + n) * T + tcur[n]) * D + d] + s.pproj[i]);
      s.z[i] = zz;
    }
    __syncthreads();
    // logits + argmax
    float bv[NB];
    int bi[NB];
#pragma unroll
    for (int n = 0; n < NB; ++n) { bv[n] = kNegInf; bi[n] = 0x7fffffff; }
    gemv_t<NB>(w.out_t, V, D, s.z, [&](int j, int n) { return __ldg(w.out_b + j); },
               [&](int j, int n, float v) { argmax_combine(bv[n], bi[n], v, j); });
#pragma unroll
    for (int n = 0; n < NB; ++n) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        float ov = __shfl_xor_sync(0xffffffffu, bv[n], o);
        int oi = __shfl_xor_sync(0xffffffffu, bi[n], o);
        argmax_combine(bv[n], bi[n], ov, oi);
      }
      if (lane == 0) { wred_v[warp * NB + n] = bv[n]; wred_i[warp * NB + n] = bi[n]; }
    }
    __syncthreads();
    if (tid < NB) {
      const int n = tid;
      int need = 0;
      commit[n] = 0;
      if (tcur[n] < len[n]) {
        float v = kNegInf;
        int k = 0x7fffffff;
        for (int wq = 0; wq < DEC_THREADS / 32; ++wq) argmax_combine(v, k, wred_v[wq * NB + n], wred_i[wq * NB + n]);
        if (k == blank) {
          tcur[n] += 1; iter[n] = 0;
        } else {
          if (nout[n] < max_out) out_tokens[(size_t)(n0 + n) * max_out + nout[n]] = k;
          nout[n] += 1;
          tok[n] = k;
          commit[n] = 1;
          need = 1;
          if (++iter[n] >= n_steps) { tcur[n] += 1; iter[n] = 0; }
        }
      }
      unsigned m = __ballot_sync(__activemask(), need);
      if (n == 0) flags[0] = (m != 0);
    }
    __syncthreads();
    if (flags[0]) {
      for (int i = tid; i < L * H * NB; i += DEC_THREADS)
        if (commit[i % NB]) { s.hs[i] = s.hn[i]; s.cs[i] = s.cn[i]; }
      __syncthreads();
    }
  }

  for (int i = tid; i < L * H * NB; i += DEC_THREADS) {
    int n = i % NB, k = (i / NB) % H, l = i / (NB * H);
    int gn = n0 + n;
    if (gn < N) { h_io[((size_t)l * N + gn) * H + k] = s.hs[i]; c_io[((size_t)l * N + gn) * H + k] = s.cs[i]; }
  }
  if (tid < NB && n0 + tid < N) { last_token[n0 + tid] = tok[tid]; out_lens[n0 + tid] = nout[tid]; }
}

template <int NB>
static size_t greedy_smem(const ctcvr_decoder_weights& w) {
  return DecodeSmem<NB>::floats(w, false) * sizeof(float) + (size_t)(DEC_THREADS / 32) * NB * 8 + (6 * NB + 2) * 4;
}

template <int NB>
static int launch_greedy(const ctcvr_decoder_weights& w, const float* enc_proj, const int32_t* lens, float* h,
                         float* c, int32_t* last_token, int32_t* out_tokens, int32_t* out_lens, int N, int T,
                         int max_out, int blank, int n_steps, cudaStream_t st) {
  size_t smem = greedy_smem<NB>(w);
  CTCVR_REQUIRE(smem <= 227 * 1024, "rnnt_greedy: predictor too large for shared memory (H=%d L=%d)", w.H, w.L);
  CTCVR_CHECK_CUDA(cudaFuncSetAttribute(rnnt_greedy_kernel<NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  rnnt_greedy_kernel<NB><<<cdiv(N, NB), DEC_THREADS, smem, st>>>(w, enc_proj, lens, h, c, last_token, out_tokens,
                                                                  out_lens, N, T, max_out, blank, n_steps);
  CTCVR_LAUNCH_CHECK();
  return 0;
}

int rnnt_greedy(const ctcvr_decoder_weights& w, const float* enc_proj, const int32_t* lens, float* h, float* c,
                int32_t* last_token, int32_t* out_tokens, int32_t* out_lens, int N, int T, int max_out, int blank,
                int n_steps, cudaStream_t st) {
  if (N == 0) return 0;
  int per_sm = cdiv(N, 148);
  if (per_sm >= 8 && greedy_smem<8>(w) <= 227 * 1024)
    return launch_greedy<8>(w, enc_proj, lens, h, c, last_token, out_tokens, out_lens, N, T, max_out, blank, n_steps, st);
  if (per_sm >= 3 && greedy_smem<4>(w) <= 227 * 1024)
    return launch_greedy<4>(w, enc_proj, lens, h, c, last_token, out_tokens, out_lens, N, T, max_out, blank, n_steps, st);
  if (per_sm >= 2 && greedy_smem<2>(w) <= 227 * 1024)
    return launch_greedy<2>(w, enc_proj, lens, h, c, last_token, out_tokens, out_lens, N, T, max_out, blank, n_steps, st);
  return launch_greedy<1>(w, enc_proj, lens, h, c, last_token, out_tokens, out_lens, N, T, max_out, blank, n_steps, st);
}

}  // namespace ctcvr
