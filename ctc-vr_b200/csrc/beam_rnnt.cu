// On-device RNN-T beam decoders (SURVEY.md §8 A7, A8), one stream per CTA (grid = streams of the call), hypotheses advancing in
// lock-step inside ONE CTA so that every predictor / joint weight fetched from L2 feeds all of them:
//   A7  OnlineRNNTModel._decode_chunk_beam_search        model/online_rnnt_model.py:389-522
//   A8  PrefixBeamSearch.prefix_beam_search              wenet/transducer/search/prefix_beam_search.py:42-148
// Semantics kept from the reference (see oracle/transducer_oracle.py for the restatement they are checked against):
// fp32 log-softmax, scores accumulated in fp64 (A7: Python float sums; A8: fp32 per frame, fp64 log-add merge),
// stable descending sort, A7 de-duplicates by token sequence keeping the first candidate (no merge), A8 merges
// equal hypotheses with log-add at the first occurrence's position, predictor state stored BEFORE feeding the
// last token.  No host synchronisation inside a chunk (the reference has several .item() per expansion).
#include "decode.cuh"

namespace ctcvr {

constexpr int BM_THREADS = 512;
constexpr int BM_BEAM_MAX = 16;
constexpr int BM_STEPS_MAX = 16;
constexpr int BM_SORT_SMEM = 512;          // candidates whose scores are sorted from shared memory (A7)

// ---- beam state (device, opaque to the caller) ------------------------------------------------------------
// header | per buffer (x2): lens[beam] | scores[beam] (f64) | tokens[beam][max_out] | h[beam][L*H] | c[beam][L*H]
// | state chain [beam][n_steps+1][2][L*H] | candidate arrays
struct BeamLayout {
  size_t off_hdr, off_buf[2], buf_bytes, off_chain, off_cand, total;
  size_t o_len, o_score, o_tok, o_h, o_c;      // offsets inside a buffer
  size_t c_score, c_src, c_extra, c_hash, c_len, c_rank;
  int ncand;
};
__host__ __device__ inline size_t al8(size_t x) { return (x + 7) / 8 * 8; }
__host__ __device__ inline BeamLayout beam_layout(int L, int H, int beam, int n_steps, int max_out) {
  BeamLayout b;
  const size_t LH = (size_t)L * H;
  b.off_hdr = 0;
  size_t o = 64;
  b.o_score = 0;
  b.o_len = al8((size_t)beam * 8);
  b.o_tok = al8(b.o_len + (size_t)beam * 4);
  b.o_h = al8(b.o_tok + (size_t)beam * max_out * 4);
  b.o_c = al8(b.o_h + (size_t)beam * LH * 4);
  b.buf_bytes = al8(b.o_c + (size_t)beam * LH * 4);
  b.off_buf[0] = o; o += b.buf_bytes;
  b.off_buf[1] = o; o += b.buf_bytes;
  b.off_chain = o; o += al8((size_t)beam * (n_steps + 1) * 2 * LH * 4);
  b.ncand = beam * n_steps * (beam + 1);      // fixed slots: (hyp, step, 0 = blank | 1..beam = top-k tokens)
  b.off_cand = o;
  b.c_score = 0;
  b.c_hash = al8((size_t)b.ncand * 8);
  b.c_src = al8(b.c_hash + (size_t)b.ncand * 8);
  b.c_extra = al8(b.c_src + (size_t)b.ncand * 4);
  b.c_len = al8(b.c_extra + (size_t)b.ncand * 4);
  b.c_rank = al8(b.c_len + (size_t)b.ncand * 4);
  o += al8(b.c_rank + (size_t)2 * b.ncand * 4);
  b.total = o;
  return b;
}

__device__ __forceinline__ unsigned long long bm_hash(unsigned long long h, int u) {
  return h * 1099511628211ULL + (unsigned long long)(u + 1);
}

// log-softmax statistics of column n of s.logit ([V][NB]) by the calling warp: max and log(sum exp(x - max))
template <int NB>
__device__ __forceinline__ void warp_lse(const float* logit, int V, int n, float& mx, float& lse) {
  const int lane = threadIdx.x & 31;
  float m = kNegInf;
  for (int v = lane; v < V; v += 32) m = fmaxf(m, logit[v * NB + n]);
  m = warp_max(m);
  float sum = 0.f;
  for (int v = lane; v < V; v += 32) sum += expf(logit[v * NB + n] - m);
  sum = warp_sum(sum);
  mx = m;
  lse = logf(sum);
}

// k largest entries (value desc, lowest index on ties) of x[v] = val(v), v in [0,V) excluding `skip`, by one warp.
// Results in tv/ti (all lanes hold them).  k <= BM_BEAM_MAX.
// Lane l owns v = l + 32 i; for V <= 512 its <= 16 values are read ONCE into registers and a selected entry is struck out
// there (the first version re-evaluated val(v) and searched the selected list - a stack array - for every v in every
// round: 60 k cycles per step, more than the joint GEMV).
template <class F>
__device__ __forceinline__ void warp_topk(F val, int V, int skip, int k, float* tv, int* ti) {
  const int lane = threadIdx.x & 31;
  if (V <= 512) {
    float x[16];
    unsigned alive = 0u;                                     // bit i: entry v = lane + 32 i is a candidate
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int v = lane + 32 * i;
      const bool ok = v < V && v != skip;
      x[i] = ok ? val(v) : 0.f;
      alive |= ok ? (1u << i) : 0u;
    }
    for (int r = 0; r < k; ++r) {
      float bv = kNegInf;
      int bi = 0x7fffffff;
#pragma unroll
      for (int i = 0; i < 16; ++i) {                       // ascending v within the lane: the first maximum survives
        const int v = lane + 32 * i;
        if (((alive >> i) & 1u) && (x[i] > bv || (x[i] == bv && v < bi))) { bv = x[i]; bi = v; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
      }
      tv[r] = bv;
      ti[r] = bi;
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (bi == lane + 32 * i) alive &= ~(1u << i);       // selected: out of the next rounds
    }
    return;
  }
  for (int r = 0; r < k; ++r) {
    float bv = kNegInf;
    int bi = 0x7fffffff;
    for (int v = lane; v < V; v += 32) {
      if (v == skip) continue;
      bool taken = false;
      for (int j = 0; j < r; ++j) taken |= (ti[j] == v);
      if (taken) continue;
      const float x = val(v);
      if (x > bv || (x == bv && v < bi)) { bv = x; bi = v; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    tv[r] = bv;
    ti[r] = bi;
  }
}

// logits of all NB slots for frame vector e (enc_proj row): z = act(e + pproj), logit = out_t^T z + out_b
template <int NB>
__device__ void joint_logits_step(const ctcvr_decoder_weights& w, DecodeSmem<NB>& s, const float* __restrict__ e) {
  const int act = w.activation >> 8;
  for (int i = threadIdx.x; i < w.D * NB; i += blockDim.x) {
    const int d = i / NB;
    s.z[i] = act_rt(act, e[d] + s.pproj[i]);
  }
  __syncthreads();
  gemv_t<NB>(w.out_t, w.V, w.D, s.z, [&](int j, int n) { return __ldg(w.out_b + j); },
             [&](int j, int n, float v) { s.logit[j * NB + n] = v; });
  __syncthreads();
}

// =============================================================================================================
// A7: online beam (model/online_rnnt_model.py:389-522)
// =============================================================================================================
template <int NB>
__global__ void __launch_bounds__(BM_THREADS, 1) rnnt_beam_chunk_kernel(
    ctcvr_decoder_weights w, const float* __restrict__ enc_proj, int T, unsigned char* __restrict__ state, int beam,
    int n_steps, int max_out, int blank, int32_t* __restrict__ out_n, int32_t* __restrict__ out_tokens,
    int32_t* __restrict__ out_lens, double* __restrict__ out_scores, float* __restrict__ out_h,
    float* __restrict__ out_c, const int32_t* __restrict__ chunk_lens, size_t state_stride) {
  extern __shared__ __align__(16) float smf[];
  DecodeSmem<NB> s;
  s.carve(smf, w, true);
  const BeamLayout lay = beam_layout(w.L, w.H, beam, n_steps, max_out);
  {
    // one CTA per stream (grid = number of streams): every per-stream array is offset by the stream index; a stream's
    // chunk may be shorter than T (chunk_lens), its rows beyond that are not read
    const size_t sidx = blockIdx.x;
    enc_proj += sidx * (size_t)T * w.D;
    state += sidx * state_stride;
    out_n += sidx;
    out_tokens += sidx * (size_t)beam * max_out;
    out_lens += sidx * beam;
    out_scores += sidx * beam;
    out_h += sidx * (size_t)beam * w.L * w.H;
    out_c += sidx * (size_t)beam * w.L * w.H;
    if (chunk_lens) T = max(0, min(T, chunk_lens[sidx]));
  }
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = BM_THREADS / 32;
  const int LH = w.L * w.H, V = w.V;
  int* hdr = reinterpret_cast<int*>(state);
  auto b_score = [&](int bf) { return reinterpret_cast<double*>(state + lay.off_buf[bf] + lay.o_score); };
  auto b_len = [&](int bf) { return reinterpret_cast<int*>(state + lay.off_buf[bf] + lay.o_len); };
  auto b_tok = [&](int bf) { return reinterpret_cast<int*>(state + lay.off_buf[bf] + lay.o_tok); };
  auto b_h = [&](int bf) { return reinterpret_cast<float*>(state + lay.off_buf[bf] + lay.o_h); };
  auto b_c = [&](int bf) { return reinterpret_cast<float*>(state + lay.off_buf[bf] + lay.o_c); };
  float* chain = reinterpret_cast<float*>(state + lay.off_chain);       // [beam][n_steps+1][2][LH]
  unsigned char* cb = state + lay.off_cand;
  double* c_score = reinterpret_cast<double*>(cb + lay.c_score);
  unsigned long long* c_hash = reinterpret_cast<unsigned long long*>(cb + lay.c_hash);
  int* c_src = reinterpret_cast<int*>(cb + lay.c_src);       // hyp j | step s << 8
  int* c_extra = reinterpret_cast<int*>(cb + lay.c_extra);   // appended token or -1 (blank candidate)
  int* c_len = reinterpret_cast<int*>(cb + lay.c_len);
  int* c_rank = reinterpret_cast<int*>(cb + lay.c_rank);     // candidate index at sorted position

  __shared__ int sh_tok[NB], sh_active[NB], sh_wlen[NB];
  __shared__ double sh_lp[NB];
  __shared__ unsigned long long sh_hash[NB][BM_STEPS_MAX + 1];    // hash of hyp tokens + walk prefix
  __shared__ int sh_ncand, sh_any, sh_keep[BM_BEAM_MAX], sh_nkeep;
  __shared__ double sh_sc[BM_SORT_SMEM];

  int buf = hdr[1];
  const int k = min(beam, V - 1);
  // candidate slot of (hypothesis j, walk step st, position i): i = 0 blank, 1..k the top-k non-blank tokens.
  // Slot order == the order in which the reference appends candidates (stable-sort tie-break).
  auto slot_of = [&](int j, int st, int i) { return (j * n_steps + st) * (beam + 1) + i; };

  for (int t = 0; t < T; ++t) {
    const int nb = hdr[0];                                   // hypotheses in the beam
    for (int i = tid; i < lay.ncand; i += BM_THREADS) c_len[i] = -1;     // -1 = slot not produced this frame
    __syncthreads();
    for (int g0 = 0; g0 < nb; g0 += NB) {                    // lock-step groups of NB hypotheses
      const int gn = min(NB, nb - g0);
      // load group state
      for (int i = tid; i < LH * NB; i += BM_THREADS) {
        const int n = i % NB, kk = i / NB;
        float hv = 0.f, cv = 0.f;
        if (n < gn) { hv = b_h(buf)[(size_t)(g0 + n) * LH + kk]; cv = b_c(buf)[(size_t)(g0 + n) * LH + kk]; }
        s.hs[i] = hv; s.cs[i] = cv;
      }
      if (tid < NB) {
        const int n = tid;
        sh_active[n] = n < gn;
        sh_wlen[n] = 0;
        if (n < gn) {
          const int len = b_len(buf)[g0 + n];
          sh_tok[n] = len > 0 ? b_tok(buf)[(size_t)(g0 + n) * max_out + len - 1] : blank;
          sh_lp[n] = b_score(buf)[g0 + n];
          unsigned long long h = 1469598103934665603ULL;
          for (int j = 0; j < len; ++j) h = bm_hash(h, b_tok(buf)[(size_t)(g0 + n) * max_out + j]);
          sh_hash[n][0] = h;
        } else {
          sh_tok[n] = blank;
        }
      }
      __syncthreads();
      for (int st = 0; st < n_steps; ++st) {
        if (tid == 0) { int any = 0; for (int n = 0; n < gn; ++n) any |= sh_active[n]; sh_any = any; }
        __syncthreads();
        if (!sh_any) break;
        predictor_step<NB>(w, s, sh_tok);
        joint_logits_step<NB>(w, s, enc_proj + (size_t)t * w.D);
        // state chain: [j][st] = state before this step, [j][st+1] = state after feeding the last token
        for (int i = tid; i < LH * NB; i += BM_THREADS) {
          const int n = i % NB, kk = i / NB;
          if (n < gn && sh_active[n]) {
            float* cj = chain + ((size_t)(g0 + n) * (n_steps + 1) + st) * 2 * LH;
            cj[kk] = s.hs[i]; cj[LH + kk] = s.cs[i];
            cj[2 * LH + kk] = s.hn[i]; cj[3 * LH + kk] = s.cn[i];
          }
        }
        // one warp per hypothesis: log-softmax, blank, top-k non-blank, candidates, continue / break
        for (int n = warp; n < gn; n += nwarp) {
          if (!sh_active[n]) continue;
          float mx, lse;
          warp_lse<NB>(s.logit, V, n, mx, lse);
          const float* lg = s.logit;
          auto lp = [&](int v) { return (lg[v * NB + n] - mx) - lse; };
          float tv[BM_BEAM_MAX];
          int ti[BM_BEAM_MAX];
          warp_topk(lp, V, blank, k, tv, ti);
          if (lane == 0) {
            const float bl = lp(blank);
            const float lmax = fmaxf(bl, tv[0]);                         // = logp.max()
            const int base = slot_of(g0 + n, st, 0);
            const int wl = sh_wlen[n];
            const int hyp_len = b_len(buf)[g0 + n] + wl;
            const double acc = sh_lp[n];
            const unsigned long long h0 = sh_hash[n][wl];
            c_score[base] = acc + (double)bl;
            c_src[base] = (g0 + n) | (st << 8);
            c_extra[base] = -1;
            c_len[base] = hyp_len;
            c_hash[base] = h0;
            for (int i = 0; i < k; ++i) {
              c_score[base + 1 + i] = acc + (double)tv[i];
              c_src[base + 1 + i] = (g0 + n) | (st << 8);
              c_extra[base + 1 + i] = ti[i];
              c_len[base + 1 + i] = hyp_len + 1;
              c_hash[base + 1 + i] = bm_hash(h0, ti[i]);
            }
            if ((double)bl >= (double)lmax - 1e-6) {
              sh_active[n] = 0;
            } else {
              sh_hash[n][wl + 1] = bm_hash(h0, ti[0]);
              sh_wlen[n] = wl + 1;
              sh_lp[n] = acc + (double)tv[0];
              sh_tok[n] = ti[0];
            }
          }
          __syncwarp();
        }
        __syncthreads();
        // commit the walk: state <- state after step for hypotheses that continue
        for (int i = tid; i < LH * NB; i += BM_THREADS) {
          const int n = i % NB;
          if (n < gn && sh_active[n]) { s.hs[i] = s.hn[i]; s.cs[i] = s.cn[i]; }
        }
        __syncthreads();
      }
      __syncthreads();
    }
    // ---- compact the produced slots (slot order = reference append order), then stable sort by score desc
    if (warp == 0) {
      int cnt = 0;
      for (int i0 = 0; i0 < lay.ncand; i0 += 32) {
        const int i = i0 + lane;
        const bool ok = (i < lay.ncand) && (c_len[i] >= 0);
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (ok) c_rank[lay.ncand + cnt + __popc(m & ((1u << lane) - 1u))] = i;    // second half of c_rank: compact list
        cnt += __popc(m);
      }
      if (lane == 0) sh_ncand = cnt;
    }
    __syncthreads();
    const int nc = sh_ncand;
    int* c_list = c_rank + lay.ncand;
    if (nc <= BM_SORT_SMEM) {
      // the scores of the compact list staged in shared memory: the rank loop otherwise makes nc^2 dependent pairs of
      // global loads (c_list -> c_score), 8 % of the kernel in the cycle-counter build
      for (int a = tid; a < nc; a += BM_THREADS) sh_sc[a] = c_score[c_list[a]];
      __syncthreads();
      for (int a = tid; a < nc; a += BM_THREADS) {
        const double sa = sh_sc[a];
        int rank = 0;
        for (int bq = 0; bq < nc; ++bq) {
          const double sb = sh_sc[bq];
          rank += (sb > sa) || (sb == sa && bq < a);
        }
        c_rank[rank] = c_list[a];
      }
    } else {
      for (int a = tid; a < nc; a += BM_THREADS) {
        const double sa = c_score[c_list[a]];
        int rank = 0;
        for (int bq = 0; bq < nc; ++bq) {
          const double sb = c_score[c_list[bq]];
          rank += (sb > sa) || (sb == sa && bq < a);
        }
        c_rank[rank] = c_list[a];
      }
    }
    __syncthreads();
    // ---- de-duplicate by token sequence, first occurrence wins, stop at `beam`
    auto tok_at = [&](int c, int pos) {
      const int j = c_src[c] & 0xff, st = c_src[c] >> 8;
      const int hl = b_len(buf)[j];
      if (pos < hl) return b_tok(buf)[(size_t)j * max_out + pos];
      // walk token p of hypothesis j = the best non-blank token of expansion (j, p)
      const int p = pos - hl;
      if (p < st) return c_extra[slot_of(j, p, 1)];
      return c_extra[c];
    };
    if (warp == 0) {
      int nkeep = 0;
      for (int r = 0; r < nc && nkeep < beam; ++r) {
        const int c = c_rank[r];
        bool dup = false;
        for (int q = 0; q < nkeep && !dup; ++q) {
          const int o = sh_keep[q];
          if (c_hash[o] == c_hash[c] && c_len[o] == c_len[c]) {
            bool same = true;
            for (int pos = lane; pos < c_len[c]; pos += 32) same &= (tok_at(o, pos) == tok_at(c, pos));
            same = __all_sync(0xffffffffu, same);
            dup = same;
          }
        }
        if (!dup) { if (lane == 0) sh_keep[nkeep] = c; ++nkeep; }
        __syncwarp();
      }
      if (lane == 0) sh_nkeep = nkeep;
    }
    __syncthreads();
    // ---- new beam into the other buffer
    const int nk = sh_nkeep, nbuf = buf ^ 1;
    for (int e = warp; e < nk; e += nwarp) {                 // one warp per kept hypothesis: the copies' latencies overlap
      const int c = sh_keep[e];
      const int j = c_src[c] & 0xff, st = c_src[c] >> 8;
      const int len = min(c_len[c], max_out);
      for (int pos = lane; pos < len; pos += 32) b_tok(nbuf)[(size_t)e * max_out + pos] = tok_at(c, pos);
      // blank candidate keeps the state before step st, a token candidate takes the state after it
      const float* cj = chain + ((size_t)j * (n_steps + 1) + st) * 2 * LH + (c_extra[c] >= 0 ? 2 * LH : 0);
      for (int i = lane; i < LH; i += 32) { b_h(nbuf)[(size_t)e * LH + i] = cj[i]; b_c(nbuf)[(size_t)e * LH + i] = cj[LH + i]; }
      if (lane == 0) { b_len(nbuf)[e] = len; b_score(nbuf)[e] = c_score[c]; }
    }
    __syncthreads();
    if (tid == 0) { hdr[0] = nk; hdr[1] = nbuf; }
    buf = nbuf;
    __syncthreads();
  }
  // ---- outputs (beam order = the reference's list order)
  const int nb = hdr[0];
  if (tid == 0) *out_n = nb;
  for (int e = 0; e < nb; ++e) {
    const int len = b_len(buf)[e];
    for (int pos = tid; pos < len; pos += BM_THREADS) out_tokens[(size_t)e * max_out + pos] = b_tok(buf)[(size_t)e * max_out + pos];
    for (int i = tid; i < LH; i += BM_THREADS) { out_h[(size_t)e * LH + i] = b_h(buf)[(size_t)e * LH + i]; out_c[(size_t)e * LH + i] = b_c(buf)[(size_t)e * LH + i]; }
    if (tid == 0) { out_lens[e] = len; out_scores[e] = b_score(buf)[e]; }
  }
}

__global__ void rnnt_beam_reset_kernel(unsigned char* state, int L, int H, int beam, int n_steps, int max_out,
                                       size_t state_stride) {
  state += (size_t)blockIdx.x * state_stride;
  const BeamLayout lay = beam_layout(L, H, beam, n_steps, max_out);
  int* hdr = reinterpret_cast<int*>(state);
  if (threadIdx.x == 0) {
    hdr[0] = 1; hdr[1] = 0;                                   // one empty hypothesis, score 0, zero state
    reinterpret_cast<double*>(state + lay.off_buf[0] + lay.o_score)[0] = 0.0;
    reinterpret_cast<int*>(state + lay.off_buf[0] + lay.o_len)[0] = 0;
  }
  float* h = reinterpret_cast<float*>(state + lay.off_buf[0] + lay.o_h);
  float* c = reinterpret_cast<float*>(state + lay.off_buf[0] + lay.o_c);
  for (int i = threadIdx.x; i < L * H; i += blockDim.x) { h[i] = 0.f; c[i] = 0.f; }
}

template <int NB>
static size_t beam_smem(const ctcvr_decoder_weights& w) { return DecodeSmem<NB>::floats(w, true) * sizeof(float); }

size_t rnnt_beam_state_bytes(const ctcvr_decoder_weights& w, int beam, int n_steps, int max_out) {
  return beam_layout(w.L, w.H, beam, n_steps, max_out).total;
}

int rnnt_beam_reset(void* state, const ctcvr_decoder_weights& w, int S, int beam, int n_steps, int max_out, cudaStream_t st) {
  CTCVR_REQUIRE(state && S >= 1, "rnnt_beam_reset: NULL state or no stream");
  CTCVR_REQUIRE(beam >= 1 && beam <= BM_BEAM_MAX && n_steps >= 1 && n_steps <= BM_STEPS_MAX,
                "rnnt_beam: beam must be within [1,%d] and n_steps within [1,%d]", BM_BEAM_MAX, BM_STEPS_MAX);
  rnnt_beam_reset_kernel<<<S, 256, 0, st>>>(reinterpret_cast<unsigned char*>(state), w.L, w.H, beam, n_steps, max_out,
                                            rnnt_beam_state_bytes(w, beam, n_steps, max_out));
  CTCVR_LAUNCH_CHECK();
  return 0;
}

template <int NB>
static int launch_beam_chunk(const ctcvr_decoder_weights& w, const float* enc_proj, const int32_t* chunk_lens, int S, int T,
                             void* state, int beam, int n_steps, int max_out, int blank, int32_t* out_n,
                             int32_t* out_tokens, int32_t* out_lens, double* out_scores, float* out_h, float* out_c,
                             cudaStream_t st) {
  const size_t smem = beam_smem<NB>(w);
  CTCVR_CHECK_CUDA(cudaFuncSetAttribute(rnnt_beam_chunk_kernel<NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  rnnt_beam_chunk_kernel<NB><<<S, BM_THREADS, smem, st>>>(w, enc_proj, T, reinterpret_cast<unsigned char*>(state), beam,
                                                          n_steps, max_out, blank, out_n, out_tokens, out_lens,
                                                          out_scores, out_h, out_c, chunk_lens,
                                                          rnnt_beam_state_bytes(w, beam, n_steps, max_out));
  CTCVR_LAUNCH_CHECK();
  return 0;
}

int rnnt_beam_chunk(const ctcvr_decoder_weights& w, const float* enc_proj, const int32_t* chunk_lens, int S, int T,
                    void* state, int beam, int n_steps, int max_out, int blank, int32_t* out_n, int32_t* out_tokens,
                    int32_t* out_lens, double* out_scores, float* out_h, float* out_c, cudaStream_t st) {
  CTCVR_REQUIRE(S >= 1, "rnnt_beam: no stream");
  CTCVR_REQUIRE(beam >= 1 && beam <= BM_BEAM_MAX && n_steps >= 1 && n_steps <= BM_STEPS_MAX,
                "rnnt_beam: beam must be within [1,%d] and n_steps within [1,%d]", BM_BEAM_MAX, BM_STEPS_MAX);
  CTCVR_REQUIRE(w.V - 1 >= 1, "rnnt_beam: vocabulary too small");
  const size_t lim = 220 * 1024;
  // one warp per hypothesis inside a group: the candidate append order (hypothesis-major) needs NB <= #warps
  // the lock-step group is as wide as the template: 12 slots for beams of 9..12 (beam 10 of BASELINE.json's cfg5 would
  // otherwise spend 6 of 16 FMA lanes per weight on empty slots)
  if (beam > 12 && beam_smem<16>(w) <= lim)
    return launch_beam_chunk<16>(w, enc_proj, chunk_lens, S, T, state, beam, n_steps, max_out, blank, out_n, out_tokens, out_lens, out_scores, out_h, out_c, st);
  if (beam > 8 && beam_smem<12>(w) <= lim)
    return launch_beam_chunk<12>(w, enc_proj, chunk_lens, S, T, state, beam, n_steps, max_out, blank, out_n, out_tokens, out_lens, out_scores, out_h, out_c, st);
  if (beam > 4 && beam_smem<8>(w) <= lim)
    return launch_beam_chunk<8>(w, enc_proj, chunk_lens, S, T, state, beam, n_steps, max_out, blank, out_n, out_tokens, out_lens, out_scores, out_h, out_c, st);
  if (beam > 1 && beam_smem<4>(w) <= lim)
    return launch_beam_chunk<4>(w, enc_proj, chunk_lens, S, T, state, beam, n_steps, max_out, blank, out_n, out_tokens, out_lens, out_scores, out_h, out_c, st);
  CTCVR_REQUIRE(beam_smem<1>(w) <= lim, "rnnt_beam: predictor too large for shared memory (H=%d L=%d)", w.H, w.L);
  return launch_beam_chunk<1>(w, enc_proj, chunk_lens, S, T, state, beam, n_steps, max_out, blank, out_n, out_tokens, out_lens, out_scores, out_h, out_c, st);
}

// =============================================================================================================
// A8: wenet transducer prefix beam with CTC shallow fusion (wenet/transducer/search/prefix_beam_search.py:42-148)
// =============================================================================================================
// workspace: per buffer (x2): scores[beam] f64 | lens[beam] | tokens[beam][T+1] | h,c [beam][LH]; new states
// [beam][2][LH]; candidates [beam*beam]
struct PrefixLayout {
  size_t off_buf[2], buf_bytes, o_score, o_len, o_tok, o_h, o_c, off_new, off_cand, c_score, c_src, c_tok, c_hash, c_len,
      c_first, total;
};
__host__ __device__ inline PrefixLayout prefix_layout(int L, int H, int beam, int T) {
  PrefixLayout p;
  const size_t LH = (size_t)L * H, ML = (size_t)T + 1;
  p.o_score = 0;
  p.o_len = al8((size_t)beam * 8);
  p.o_tok = al8(p.o_len + (size_t)beam * 4);
  p.o_h = al8(p.o_tok + (size_t)beam * ML * 4);
  p.o_c = al8(p.o_h + (size_t)beam * LH * 4);
  p.buf_bytes = al8(p.o_c + (size_t)beam * LH * 4);
  size_t o = 0;
  p.off_buf[0] = o; o += p.buf_bytes;
  p.off_buf[1] = o; o += p.buf_bytes;
  p.off_new = o; o += al8((size_t)beam * 2 * LH * 4);
  p.off_cand = o;
  const size_t nc = (size_t)beam * beam;
  p.c_score = 0;
  p.c_hash = al8(nc * 8);
  p.c_src = al8(p.c_hash + nc * 8);
  p.c_tok = al8(p.c_src + nc * 4);
  p.c_len = al8(p.c_tok + nc * 4);
  p.c_first = al8(p.c_len + nc * 4);
  o += al8(p.c_first + nc * 4);
  p.total = o;
  return p;
}

template <int NB>
__global__ void __launch_bounds__(BM_THREADS, 1) rnnt_prefix_beam_kernel(
    ctcvr_decoder_weights w, const float* __restrict__ enc_proj, const float* __restrict__ ctc_logp, int T, int beam,
    int blank, float ctc_weight, float tr_weight, int32_t* __restrict__ out_n, int32_t* __restrict__ out_tokens,
    int32_t* __restrict__ out_lens, double* __restrict__ out_scores, unsigned char* __restrict__ ws,
    const int32_t* __restrict__ lens, size_t ws_stride) {
  extern __shared__ __align__(16) float smf[];
  DecodeSmem<NB> s;
  s.carve(smf, w, true);
  const PrefixLayout lay = prefix_layout(w.L, w.H, beam, T);      // sized for the longest utterance of the batch
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = BM_THREADS / 32;
  const int LH = w.L * w.H, V = w.V, ML = T + 1;
  {
    // one CTA per utterance (grid = batch): per-utterance arrays are offset by the utterance index
    const size_t sidx = blockIdx.x;
    enc_proj += sidx * (size_t)T * w.D;
    ctc_logp += sidx * (size_t)T * V;
    ws += sidx * ws_stride;
    out_n += sidx;
    out_tokens += sidx * (size_t)beam * ML;
    out_lens += sidx * beam;
    out_scores += sidx * beam;
    if (lens) T = max(0, min(T, lens[sidx]));
  }
  auto b_score = [&](int bf) { return reinterpret_cast<double*>(ws + lay.off_buf[bf] + lay.o_score); };
  auto b_len = [&](int bf) { return reinterpret_cast<int*>(ws + lay.off_buf[bf] + lay.o_len); };
  auto b_tok = [&](int bf) { return reinterpret_cast<int*>(ws + lay.off_buf[bf] + lay.o_tok); };
  auto b_h = [&](int bf) { return reinterpret_cast<float*>(ws + lay.off_buf[bf] + lay.o_h); };
  auto b_c = [&](int bf) { return reinterpret_cast<float*>(ws + lay.off_buf[bf] + lay.o_c); };
  float* newst = reinterpret_cast<float*>(ws + lay.off_new);          // [beam][2][LH]
  unsigned char* cbp = ws + lay.off_cand;
  double* c_score = reinterpret_cast<double*>(cbp + lay.c_score);
  unsigned long long* c_hash = reinterpret_cast<unsigned long long*>(cbp + lay.c_hash);
  int* c_src = reinterpret_cast<int*>(cbp + lay.c_src);
  int* c_tok = reinterpret_cast<int*>(cbp + lay.c_tok);               // appended token or -1
  int* c_len = reinterpret_cast<int*>(cbp + lay.c_len);
  int* c_first = reinterpret_cast<int*>(cbp + lay.c_first);           // index of the fused entry this one merged into
  __shared__ int sh_tok[NB];
  __shared__ unsigned long long sh_hash[BM_BEAM_MAX];
  __shared__ int sh_nb, sh_sel[BM_BEAM_MAX], sh_nsel;
  __shared__ unsigned long long sh_ch[BM_BEAM_MAX * BM_BEAM_MAX];      // merge keys of the frame's candidates
  __shared__ int sh_cl[BM_BEAM_MAX * BM_BEAM_MAX], sh_cf[BM_BEAM_MAX * BM_BEAM_MAX];

  // initial beam: [blank], score 0, zero state
  if (tid == 0) { b_score(0)[0] = 0.0; b_len(0)[0] = 1; b_tok(0)[0] = blank; sh_nb = 1; sh_hash[0] = bm_hash(1469598103934665603ULL, blank); }
  for (int i = tid; i < LH; i += BM_THREADS) { b_h(0)[i] = 0.f; b_c(0)[i] = 0.f; }
  __syncthreads();
  int buf = 0;

  for (int t = 0; t < T; ++t) {
    const int nb = sh_nb;
    const int k = min(beam, V);
    for (int g0 = 0; g0 < nb; g0 += NB) {
      const int gn = min(NB, nb - g0);
      for (int i = tid; i < LH * NB; i += BM_THREADS) {
        const int n = i % NB, kk = i / NB;
        float hv = 0.f, cv = 0.f;
        if (n < gn) { hv = b_h(buf)[(size_t)(g0 + n) * LH + kk]; cv = b_c(buf)[(size_t)(g0 + n) * LH + kk]; }
        s.hs[i] = hv; s.cs[i] = cv;
      }
      if (tid < NB) sh_tok[tid] = (tid < gn) ? b_tok(buf)[(size_t)(g0 + tid) * ML + b_len(buf)[g0 + tid] - 1] : blank;
      __syncthreads();
      predictor_step<NB>(w, s, sh_tok);
      joint_logits_step<NB>(w, s, enc_proj + (size_t)t * w.D);
      for (int i = tid; i < LH * NB; i += BM_THREADS) {
        const int n = i % NB, kk = i / NB;
        if (n < gn) { newst[(size_t)(g0 + n) * 2 * LH + kk] = s.hn[i]; newst[(size_t)(g0 + n) * 2 * LH + LH + kk] = s.cn[i]; }
      }
      for (int n = warp; n < gn; n += nwarp) {
        float mx, lse;
        warp_lse<NB>(s.logit, V, n, mx, lse);
        const float* lg = s.logit;
        const float* cl = ctc_logp + (size_t)t * V;
        // logp = log(tw * exp(log_softmax) + cw * exp(ctc_logp))   (prefix_beam_search.py:99-101, fp32)
        auto fused = [&](int v) { return logf(tr_weight * expf((lg[v * NB + n] - mx) - lse) + ctc_weight * expf(cl[v])); };
        float tv[BM_BEAM_MAX];
        int ti[BM_BEAM_MAX];
        warp_topk(fused, V, -1, k, tv, ti);
        if (lane == 0) {
          const int j = g0 + n;
          const float sc = (float)b_score(buf)[j];                      // scores tensor is fp32 in the reference
          for (int r = 0; r < k; ++r) {
            const int c = j * beam + r;
            c_score[c] = (double)(sc + tv[r]);
            c_src[c] = j;
            const bool isb = (ti[r] == blank);
            c_tok[c] = isb ? -1 : ti[r];
            c_len[c] = b_len(buf)[j] + (isb ? 0 : 1);
            c_hash[c] = isb ? sh_hash[j] : bm_hash(sh_hash[j], ti[r]);
            c_first[c] = c;
          }
        }
      }
      __syncthreads();
    }
    // ---- merge identical hypotheses (first occurrence accumulates with log-add, in candidate order)
    const int nc = nb * k;
    // candidates of hypothesis j live at j*beam .. j*beam+k-1 (k == beam unless V < beam)
    auto cidx = [&](int i) { return (i / k) * beam + (i % k); };
    auto tok_at = [&](int c, int pos) {
      const int j = c_src[c];
      return (pos < b_len(buf)[j]) ? b_tok(buf)[(size_t)j * ML + pos] : c_tok[c];
    };
    // The order-dependent part (candidate i merges into the FIRST surviving equal candidate q < i) runs on one warp;
    // its search over q is lane-parallel on shared-memory keys (hash, length, survivor flag) and only hash matches
    // are verified token by token.
    for (int i = tid; i < nc; i += BM_THREADS) {
      const int c = cidx(i);
      sh_ch[i] = c_hash[c];
      sh_cl[i] = c_len[c];
      sh_cf[i] = i;
    }
    __syncthreads();
    if (warp == 0) {
      for (int i = 1; i < nc; ++i) {
        const int c = cidx(i);
        const unsigned long long hi = sh_ch[i];
        const int li = sh_cl[i];
        int target = -1;
        for (int q0 = 0; q0 < i && target < 0; q0 += 32) {
          const int q = q0 + lane;
          const bool cand = q < i && sh_cf[q] == q && sh_ch[q] == hi && sh_cl[q] == li;
          unsigned m = __ballot_sync(0xffffffffu, cand);
          while (m && target < 0) {
            const int qq = q0 + __ffs(m) - 1;
            m &= m - 1;
            const int o = cidx(qq);
            bool same = true;
            for (int pos = lane; pos < li; pos += 32) same &= (tok_at(o, pos) == tok_at(c, pos));
            if (__all_sync(0xffffffffu, same)) target = qq;
          }
        }
        if (target >= 0 && lane == 0) {
          const int o = cidx(target);
          const double a = c_score[o], bb = c_score[c];
          double r;
          if (a == -INFINITY && bb == -INFINITY) r = -INFINITY;
          else { const double m2 = fmax(a, bb); r = m2 + log(exp(a - m2) + exp(bb - m2)); }
          c_score[o] = r;
          sh_cf[i] = target;
        }
        __syncwarp();
      }
    }
    __syncthreads();
    for (int i = tid; i < nc; i += BM_THREADS) c_first[cidx(i)] = cidx(sh_cf[i]);
    __syncthreads();
    // ---- stable sort (score desc, candidate order asc) of the fused list, keep `beam`
    for (int i = tid; i < nc; i += BM_THREADS) {
      const int c = cidx(i);
      if (c_first[c] != c) continue;
      int rank = 0;
      for (int q = 0; q < nc; ++q) {
        const int o = cidx(q);
        if (o == c || c_first[o] != o) continue;
        if (c_score[o] > c_score[c] || (c_score[o] == c_score[c] && q < i)) ++rank;
      }
      if (rank < beam) sh_sel[rank] = c;
    }
    if (tid == 0) {
      int cnt = 0;
      for (int i = 0; i < nc; ++i) cnt += (c_first[cidx(i)] == cidx(i));
      sh_nsel = min(cnt, beam);
    }
    __syncthreads();
    const int ns = sh_nsel, nbuf = buf ^ 1;
    for (int e = 0; e < ns; ++e) {
      const int c = sh_sel[e], j = c_src[c], len = c_len[c];
      for (int pos = tid; pos < len; pos += BM_THREADS) b_tok(nbuf)[(size_t)e * ML + pos] = tok_at(c, pos);
      const bool isnew = c_tok[c] >= 0;
      const float* hsrc = isnew ? newst + (size_t)j * 2 * LH : b_h(buf) + (size_t)j * LH;
      const float* csrc = isnew ? newst + (size_t)j * 2 * LH + LH : b_c(buf) + (size_t)j * LH;
      for (int i = tid; i < LH; i += BM_THREADS) { b_h(nbuf)[(size_t)e * LH + i] = hsrc[i]; b_c(nbuf)[(size_t)e * LH + i] = csrc[i]; }
      if (tid == 0) { b_len(nbuf)[e] = len; b_score(nbuf)[e] = c_score[c]; }
    }
    __syncthreads();
    if (tid < ns) sh_hash[tid] = c_hash[sh_sel[tid]];
    if (tid == 0) sh_nb = ns;
    buf = nbuf;
    __syncthreads();
  }
  const int nb = sh_nb;
  if (tid == 0) *out_n = nb;
  for (int e = 0; e < nb; ++e) {
    const int len = b_len(buf)[e];
    for (int pos = tid; pos < len; pos += BM_THREADS) out_tokens[(size_t)e * ML + pos] = b_tok(buf)[(size_t)e * ML + pos];
    if (tid == 0) { out_lens[e] = len; out_scores[e] = b_score(buf)[e]; }
  }
}

size_t rnnt_prefix_beam_ws_bytes(const ctcvr_decoder_weights& w, int beam, int T) {
  return prefix_layout(w.L, w.H, beam, T).total;
}

template <int NB>
static int launch_prefix(const ctcvr_decoder_weights& w, const float* enc_proj, const float* ctc_logp, const int32_t* lens,
                         int S, int T, int beam, int blank, float cw, float tw, int32_t* out_n, int32_t* out_tokens,
                         int32_t* out_lens, double* out_scores, void* ws, cudaStream_t st) {
  const size_t smem = beam_smem<NB>(w);
  CTCVR_CHECK_CUDA(cudaFuncSetAttribute(rnnt_prefix_beam_kernel<NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  rnnt_prefix_beam_kernel<NB><<<S, BM_THREADS, smem, st>>>(w, enc_proj, ctc_logp, T, beam, blank, cw, tw, out_n,
                                                           out_tokens, out_lens, out_scores,
                                                           reinterpret_cast<unsigned char*>(ws), lens,
                                                           rnnt_prefix_beam_ws_bytes(w, beam, T));
  CTCVR_LAUNCH_CHECK();
  return 0;
}

int rnnt_prefix_beam(const ctcvr_decoder_weights& w, const float* enc_proj, const float* ctc_logp, const int32_t* lens,
                     int S, int T, int beam, int blank, float ctc_weight, float transducer_weight, int32_t* out_n,
                     int32_t* out_tokens, int32_t* out_lens, double* out_scores, void* ws, size_t ws_bytes,
                     cudaStream_t st) {
  CTCVR_REQUIRE(beam >= 1 && beam <= BM_BEAM_MAX, "rnnt_prefix_beam: beam must be within [1,%d]", BM_BEAM_MAX);
  CTCVR_REQUIRE(S >= 1, "rnnt_prefix_beam: no utterance");
  CTCVR_REQUIRE(ws && ws_bytes >= (size_t)S * rnnt_prefix_beam_ws_bytes(w, beam, T),
                "rnnt_prefix_beam: workspace too small (%d x ctcvr_rnnt_prefix_beam_ws_bytes)", S);
  const size_t lim = 220 * 1024;
  if (beam > 12 && beam_smem<16>(w) <= lim) return launch_prefix<16>(w, enc_proj, ctc_logp, lens, S, T, beam, blank, ctc_weight, transducer_weight, out_n, out_tokens, out_lens, out_scores, ws, st);
  if (beam > 8 && beam_smem<12>(w) <= lim) return launch_prefix<12>(w, enc_proj, ctc_logp, lens, S, T, beam, blank, ctc_weight, transducer_weight, out_n, out_tokens, out_lens, out_scores, ws, st);
  if (beam > 4 && beam_smem<8>(w) <= lim) return launch_prefix<8>(w, enc_proj, ctc_logp, lens, S, T, beam, blank, ctc_weight, transducer_weight, out_n, out_tokens, out_lens, out_scores, ws, st);
  if (beam > 1 && beam_smem<4>(w) <= lim) return launch_prefix<4>(w, enc_proj, ctc_logp, lens, S, T, beam, blank, ctc_weight, transducer_weight, out_n, out_tokens, out_lens, out_scores, ws, st);
  CTCVR_REQUIRE(beam_smem<1>(w) <= lim, "rnnt_prefix_beam: predictor too large for shared memory (H=%d L=%d)", w.H, w.L);
  return launch_prefix<1>(w, enc_proj, ctc_logp, lens, S, T, beam, blank, ctc_weight, transducer_weight, out_n, out_tokens, out_lens, out_scores, ws, st);
}

}  // namespace ctcvr
