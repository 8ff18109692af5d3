// fp32 SIMT path of the fused transducer joint (the 1e-4 parity path).
//
//   z      = tanh(enc_proj[b,t,:] + pred_proj[b,u,:])          model/component/joint.py:57-67
//   logits = z . W_out^T + b_out                               model/component/joint.py:68
//   fwd : lse, lp_blank, lp_label per lattice cell (log-softmax part of
//         torchaudio.functional.rnnt_loss, model/component/transducer.py:180-187)
//   bwd : recompute logits per utterance chunk, closed-form d cost/d logits (SURVEY.md §8 A2),
//         then dZ = g.W, dW += g^T.z, dH = dZ*(1-z^2), d_enc = sum_u dH, d_pred = sum_t dH.
//   relu / gelu joints: z = act(h) in the z tile, dH = dZ*act'(h) (joint.py:64-67, `activation`).
//
// The forward never writes logits to HBM.  The fp32 backward materialises g and z for a bounded
// chunk of utterances in the caller's workspace (the bf16 tcgen05 path in joint_tc.cu is the
// performance path; this one exists for fp32 parity and as the on-GPU cross-check).
#include "common.cuh"

namespace ctcvr {

constexpr int TM = 64;     // lattice cells per CTA tile
constexpr int TN = 128;    // vocabulary columns per pass
constexpr int TK = 32;     // k-chunk of W staged in smem
constexpr int TMP = TM + 4;   // z tile pitch (floats), keeps float4 alignment
constexpr int TNP = TN + 4;   // W chunk pitch
constexpr int JT_THREADS = 256;

enum { MODE_STATS = 0, MODE_DENSE = 1, MODE_GRAD = 2 };

struct JointTileArgs {
  const float* enc;      // [B,T,D]
  const float* pred;     // [B,U1,D]
  const float* w;        // [V,D]
  const float* bias;     // [V]
  const int32_t* targets;   // [B,U1-1]
  const int32_t* t_len;
  const int32_t* u_len;
  int B, T, U1, D, V, blank;
  int b0;                // first utterance handled by this launch (chunked backward)
  // MODE_STATS outputs
  float* lse;
  float* lp_blank;
  float* lp_label;
  // MODE_DENSE output
  float* logits;         // [B,T,U1,V]
  // MODE_GRAD inputs / outputs
  const float* lse_in;
  const float* alpha;
  const float* beta;
  const float* costs;
  const float* grad_costs;
  float clamp;
  float* g;              // [nb*T*U1, V]
  float* z;              // [nb*T*U1, D]
};

// KIND = MODE | (joint activation << 4): the tanh kernels are joint_tile_kernel<MODE> (ACT_TANH = 0), the relu and gelu
// kernels joint_tile_kernel<MODE + 16> and <MODE + 32>.
template <int KIND>
__global__ void __launch_bounds__(JT_THREADS, 1) joint_tile_kernel(JointTileArgs a) {
  constexpr int MODE = KIND & 15, ACT = KIND >> 4;
  extern __shared__ __align__(16) float smem[];
  float* zs = smem;                         // [D][TMP]
  float* ws = zs + (size_t)a.D * TMP;       // [TK][TNP]
  float* rowc = ws + TK * TNP;              // [4][TM] per-row constants
  int* rowi = reinterpret_cast<int*>(rowc + 4 * TM);   // [3][TM] : label id, t, u (or -1 invalid)

  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int b = a.b0 + blockIdx.y;
  const int D = a.D, V = a.V, U1 = a.U1, T = a.T;
  const int Tb = a.t_len ? max(min(a.t_len[b], T), 0) : T;                    // lengths beyond the tensors cannot index outside them
  const int Ub = a.u_len ? max(min(a.u_len[b], U1 - 1), 0) : U1 - 1;
  const bool dense_enum = (MODE != MODE_STATS);
  const int width = dense_enum ? U1 : (Ub + 1);
  const int ncell = dense_enum ? T * U1 : Tb * (Ub + 1);
  const int c0 = blockIdx.x * TM;
  if (c0 >= ncell) return;

  // ---- per-row bookkeeping
  if (tid < TM) {
    int c = c0 + tid;
    int t = c / width, u = c - t * width;
    bool valid = (c < ncell) && (t < Tb) && (u <= Ub);
    rowi[TM + tid] = valid ? t : -1;
    rowi[2 * TM + tid] = u;
    int lab = -1;
    if (valid && u < Ub && a.targets != nullptr) {
      lab = a.targets[(size_t)b * (U1 - 1) + u];
      if ((unsigned)lab >= (unsigned)V) lab = a.blank;      // out-of-range ids cannot index outside the tile
    }
    rowi[tid] = lab;
    if (MODE == MODE_GRAD) {
      float k_all = kNegInf, k_blank = kNegInf, k_label = kNegInf, scale = 0.f;
      if (valid) {
        size_t cell = ((size_t)b * T + t) * U1 + u;
        float al = a.alpha[cell], be = a.beta[cell], cost = a.costs[b], l = a.lse_in[cell];
        k_all = al + be + cost - l;
        float bnext = kNegInf;
        if (t + 1 < Tb) bnext = a.beta[cell + U1];
        else if (u == Ub) bnext = 0.f;
        k_blank = al + bnext + cost - l;
        if (u < Ub) k_label = al + a.beta[cell + 1] + cost - l;
        scale = a.grad_costs[b];
      }
      rowc[tid] = k_all; rowc[TM + tid] = k_blank; rowc[2 * TM + tid] = k_label; rowc[3 * TM + tid] = scale;
    }
  }
  __syncthreads();

  // ---- z tile: zs[k][row] = act(enc[b,t,k] + pred[b,u,k]); lanes run along k (coalesced)
  for (int r = warp; r < TM; r += JT_THREADS / 32) {
    int t = rowi[TM + r], u = rowi[2 * TM + r];
    if (t >= 0) {
      const float* e = a.enc + ((size_t)b * T + t) * D;
      const float* p = a.pred + ((size_t)b * U1 + u) * D;
      for (int k = lane; k < D; k += 32) zs[(size_t)k * TMP + r] = act_f32<ACT>(e[k] + p[k]);
    } else {
      for (int k = lane; k < D; k += 32) zs[(size_t)k * TMP + r] = 0.f;
    }
  }
  __syncthreads();

  if (MODE == MODE_GRAD) {   // spill z chunk rows (row-major [row][D]) for the dW GEMM
    size_t row0 = (size_t)blockIdx.y * T * U1 + c0;
    for (int r = warp; r < TM; r += JT_THREADS / 32) {
      if (c0 + r < ncell) {
        float* dst = a.z + (row0 + r) * D;
        for (int k = lane; k < D; k += 32) dst[k] = zs[(size_t)k * TMP + r];
      }
    }
  }

  const int rg = tid >> 4, cg = tid & 15;     // rows 4rg..4rg+3, cols 8cg..8cg+7 of the pass
  float run_m[4], run_s[4], pick_b[4], pick_l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) { run_m[i] = kNegInf; run_s[i] = 0.f; pick_b[i] = 0.f; pick_l[i] = 0.f; }

  for (int v0 = 0; v0 < V; v0 += TN) {
    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    for (int k0 = 0; k0 < D; k0 += TK) {
      // stage W[v0..v0+TN)[k0..k0+TK) as ws[kk][col]; lanes along kk (contiguous d)
      for (int col = warp; col < TN; col += JT_THREADS / 32) {
        int v = v0 + col, k = k0 + lane;
        float x = 0.f;
        if (v < V && k < D) x = __ldg(a.w + (size_t)v * D + k);
        ws[lane * TNP + col] = x;
      }
      __syncthreads();
      const int kmax = min(TK, D - k0);
#pragma unroll 8
      for (int kk = 0; kk < kmax; ++kk) {
        float4 zr = *reinterpret_cast<const float4*>(zs + (size_t)(k0 + kk) * TMP + 4 * rg);
        float4 w0 = *reinterpret_cast<const float4*>(ws + kk * TNP + 8 * cg);
        float4 w1 = *reinterpret_cast<const float4*>(ws + kk * TNP + 8 * cg + 4);
        float zv[4] = {zr.x, zr.y, zr.z, zr.w};
        float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(zv[i], wv[j], acc[i][j]);
      }
      __syncthreads();
    }

    // ---- epilogue of this column pass
    const int vbase = v0 + 8 * cg;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float bj = (vbase + j < V) ? __ldg(a.bias + vbase + j) : 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i][j] = (vbase + j < V) ? acc[i][j] + bj : kNegInf;
    }
    if (MODE == MODE_STATS) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int r = 4 * rg + i;
        float m = acc[i][0];
#pragma unroll
        for (int j = 1; j < 8; ++j) m = fmaxf(m, acc[i][j]);
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        float nm = fmaxf(run_m[i], m);
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) s += expf(acc[i][j] - nm);
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        run_s[i] = run_s[i] * expf(run_m[i] - nm) + s;
        run_m[i] = nm;
        int lab = rowi[r];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (vbase + j == a.blank) pick_b[i] = acc[i][j];
          if (vbase + j == lab) pick_l[i] = acc[i][j];
        }
      }
    } else if (MODE == MODE_DENSE) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int c = c0 + 4 * rg + i;
        if (c < ncell) {
          float* dst = a.logits + ((size_t)b * T * U1 + c) * V;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (vbase + j < V) dst[vbase + j] = acc[i][j];
        }
      }
    } else {   // MODE_GRAD
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int r = 4 * rg + i, c = c0 + r;
        if (c >= ncell) continue;
        float k_all = rowc[r], k_blank = rowc[TM + r], k_label = rowc[2 * TM + r], scale = rowc[3 * TM + r];
        int lab = rowi[r];
        float* dst = a.g + ((size_t)blockIdx.y * T * U1 + c) * V;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          int v = vbase + j;
          if (v >= V) continue;
          float gv = 0.f;
          if (k_all != kNegInf) {
            gv = expf(acc[i][j] + k_all);
            if (v == a.blank && k_blank != kNegInf) gv -= expf(acc[i][j] + k_blank);
            if (v == lab && k_label != kNegInf) gv -= expf(acc[i][j] + k_label);
            if (a.clamp > 0.f) gv = fminf(fmaxf(gv, -a.clamp), a.clamp);
            gv *= scale;
          }
          dst[v] = gv;
        }
      }
    }
  }

  if (MODE == MODE_STATS) {
    // pick_b / pick_l live in whichever lane owned the column: reduce over the 16 column lanes
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) {
        pick_b[i] += __shfl_xor_sync(0xffffffffu, pick_b[i], o);
        pick_l[i] += __shfl_xor_sync(0xffffffffu, pick_l[i], o);
      }
      int r = 4 * rg + i;
      int t = rowi[TM + r], u = rowi[2 * TM + r];
      if (cg == 0 && t >= 0) {
        size_t cell = ((size_t)b * T + t) * U1 + u;
        float l = run_m[i] + logf(run_s[i]);
        a.lse[cell] = l;
        a.lp_blank[cell] = pick_b[i] - l;
        a.lp_label[cell] = (rowi[r] >= 0) ? pick_l[i] - l : kNegInf;
      }
    }
  }
}

static size_t joint_tile_smem(int D) {
  return ((size_t)D * TMP + TK * TNP + 4 * TM) * sizeof(float) + 3 * TM * sizeof(int);
}

template <int MODE>
static int launch_joint_tile(const JointTileArgs& a, int nb, cudaStream_t st, int act = ACT_TANH) {
  size_t smem = joint_tile_smem(a.D);
  CTCVR_REQUIRE(smem <= 227 * 1024, "joint fp32 path: join_dim %d too large for one SM's shared memory", a.D);
  const auto kern = act == ACT_RELU ? joint_tile_kernel<MODE | (ACT_RELU << 4)>
                    : act == ACT_GELU ? joint_tile_kernel<MODE | (ACT_GELU << 4)> : joint_tile_kernel<MODE>;
  CTCVR_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(cdiv((long)a.T * a.U1, TM), nb);
  kern<<<grid, JT_THREADS, smem, st>>>(a);
  CTCVR_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------
// plain fp32 GEMM used by the chunked backward: C[M,N] (+)= A(m,k) B(k,n), B row-major [K,N],
// A either row-major [M,K] (A_T=false) or stored [K,M] (A_T=true).  64x64x16 tiles, split-K.
template <bool A_T>
__global__ void __launch_bounds__(256) sgemm_kernel(const float* __restrict__ A, const float* __restrict__ Bm,
                                                    float* __restrict__ C, int M, int N, int K, int lda,
                                                    int ldb, int ldc, int kchunk, int accumulate) {
  __shared__ __align__(16) float As[16][68];
  __shared__ __align__(16) float Bs[16][68];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int kbeg = blockIdx.z * kchunk, kend = min(K, kbeg + kchunk);
  float acc[4][4] = {};
  for (int k0 = kbeg; k0 < kend; k0 += 16) {
    if (A_T) {     // A stored [K][M]: lanes along m
      for (int i = tid; i < 16 * 64; i += 256) {
        int kk = i >> 6, m = i & 63;
        float x = 0.f;
        if (k0 + kk < kend && m0 + m < M) x = A[(size_t)(k0 + kk) * lda + m0 + m];
        As[kk][m] = x;
      }
    } else {       // A stored [M][K]: lanes along k
      for (int i = tid; i < 16 * 64; i += 256) {
        int m = i >> 4, kk = i & 15;
        float x = 0.f;
        if (k0 + kk < kend && m0 + m < M) x = A[(size_t)(m0 + m) * lda + k0 + kk];
        As[kk][m] = x;
      }
    }
    for (int i = tid; i < 16 * 64; i += 256) {
      int kk = i >> 6, n = i & 63;
      float x = 0.f;
      if (k0 + kk < kend && n0 + n < N) x = Bm[(size_t)(k0 + kk) * ldb + n0 + n];
      Bs[kk][n] = x;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float4 av = *reinterpret_cast<const float4*>(&As[kk][4 * ty]);
      float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][4 * tx]);
      float a4[4] = {av.x, av.y, av.z, av.w}, b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a4[i], b4[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int m = m0 + 4 * ty + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + 4 * tx + j;
      if (n >= N) continue;
      if (gridDim.z > 1 || accumulate) atomicAdd(&C[(size_t)m * ldc + n], acc[i][j]);
      else C[(size_t)m * ldc + n] = acc[i][j];
    }
  }
}

// dH = dZ*(1-z^2) in place; d_enc[b,t,:] = sum_u dH.  One CTA per (t, b_local).
__global__ void dh_enc_kernel(float* __restrict__ dz, const float* __restrict__ z, float* __restrict__ d_enc,
                              int b0, int T, int U1, int D) {
  int t = blockIdx.x, bl = blockIdx.y;
  size_t row0 = ((size_t)bl * T + t) * U1;
  for (int k = threadIdx.x; k < D; k += blockDim.x) {
    float s = 0.f;
    for (int u = 0; u < U1; ++u) {
      size_t i = (row0 + u) * D + k;
      float zz = z[i];
      float dh = dz[i] * (1.f - zz * zz);
      dz[i] = dh;
      s += dh;
    }
    d_enc[((size_t)(b0 + bl) * T + t) * D + k] = s;
  }
}
// Other activations: dH = dZ act'(h), h = enc + pred recomputed (gelu's derivative needs h, not z); rows outside the
// utterance (dZ = 0 there) are skipped.
template <int ACT>
__global__ void dh_enc_act_kernel(float* __restrict__ dz, const float* __restrict__ enc, const float* __restrict__ pred,
                                  const int32_t* __restrict__ t_len, const int32_t* __restrict__ u_len,
                                  float* __restrict__ d_enc, int b0, int T, int U1, int D) {
  int t = blockIdx.x, bl = blockIdx.y, b = b0 + bl;
  const int Tb = max(min(t_len[b], T), 0), Ub = max(min(u_len[b], U1 - 1), 0);
  size_t row0 = ((size_t)bl * T + t) * U1;
  for (int k = threadIdx.x; k < D; k += blockDim.x) {
    const float e = enc[((size_t)b * T + t) * D + k];
    float s = 0.f;
    for (int u = 0; u < U1; ++u) {
      size_t i = (row0 + u) * D + k;
      const float dh = (t < Tb && u <= Ub) ? dz[i] * act_grad_f32<ACT>(e + pred[((size_t)b * U1 + u) * D + k]) : 0.f;
      dz[i] = dh;
      s += dh;
    }
    d_enc[((size_t)b * T + t) * D + k] = s;
  }
}
// d_pred[b,u,:] = sum_t dH.  One CTA per (u, b_local).
__global__ void dh_pred_kernel(const float* __restrict__ dh, float* __restrict__ d_pred, int b0, int T, int U1, int D) {
  int u = blockIdx.x, bl = blockIdx.y;
  for (int k = threadIdx.x; k < D; k += blockDim.x) {
    float s = 0.f;
    for (int t = 0; t < T; ++t) s += dh[(((size_t)bl * T + t) * U1 + u) * D + k];
    d_pred[((size_t)(b0 + bl) * U1 + u) * D + k] = s;
  }
}
// d_b[v] += sum_rows g[row][v]
__global__ void colsum_kernel(const float* __restrict__ g, float* __restrict__ out, long rows, int V, long rows_per_cta) {
  long r0 = (long)blockIdx.y * rows_per_cta, r1 = min(rows, r0 + rows_per_cta);
  int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  float s = 0.f;
  for (long r = r0; r < r1; ++r) s += g[r * V + v];
  atomicAdd(out + v, s);
}

static size_t bwd_f32_rows_per_utt(int T, int U1) { return (size_t)T * U1; }
static int bwd_f32_chunk_utts(int B, int T, int U1, int D, int V) {
  size_t per = bwd_f32_rows_per_utt(T, U1) * (size_t)(V + 2 * D) * sizeof(float);
  size_t budget = (size_t)256 << 20;
  int nb = (int)(budget / per);
  if (nb < 1) nb = 1;
  if (nb > B) nb = B;
  return nb;
}

size_t joint_bwd_f32_ws_bytes(int B, int T, int U1, int D, int V) {
  int nb = bwd_f32_chunk_utts(B, T, U1, D, V);
  return (size_t)nb * bwd_f32_rows_per_utt(T, U1) * (size_t)(V + 2 * D) * sizeof(float) + 256;
}

int joint_logits_f32(const float* enc, const float* pred, const float* w, const float* bias, float* logits,
                     int B, int T, int U1, int D, int V, cudaStream_t st) {
  JointTileArgs a{};
  a.enc = enc; a.pred = pred; a.w = w; a.bias = bias; a.logits = logits;
  a.B = B; a.T = T; a.U1 = U1; a.D = D; a.V = V; a.blank = -1;
  return launch_joint_tile<MODE_DENSE>(a, B, st);
}

int joint_fwd_f32(const float* enc, const float* pred, const float* w, const float* bias, const int32_t* targets,
                  const int32_t* t_len, const int32_t* u_len, float* lse, float* lp_blank, float* lp_label,
                  int B, int T, int U1, int D, int V, int blank, int act, cudaStream_t st) {
  JointTileArgs a{};
  a.enc = enc; a.pred = pred; a.w = w; a.bias = bias; a.targets = targets; a.t_len = t_len; a.u_len = u_len;
  a.lse = lse; a.lp_blank = lp_blank; a.lp_label = lp_label;
  a.B = B; a.T = T; a.U1 = U1; a.D = D; a.V = V; a.blank = blank;
  return launch_joint_tile<MODE_STATS>(a, B, st, act);
}

int joint_bwd_f32(const float* enc, const float* pred, const float* w, const float* bias, const int32_t* targets,
                  const int32_t* t_len, const int32_t* u_len, const float* lse, const float* alpha,
                  const float* beta, const float* costs, const float* grad_costs, float clamp, float* d_enc,
                  float* d_pred, float* d_w, float* d_b, int B, int T, int U1, int D, int V, int blank, int act,
                  void* ws, size_t ws_bytes, cudaStream_t st) {
  CTCVR_REQUIRE(ws_bytes >= joint_bwd_f32_ws_bytes(B, T, U1, D, V), "joint_rnnt_bwd fp32: workspace too small");
  const int nb_max = bwd_f32_chunk_utts(B, T, U1, D, V);
  const size_t rpu = bwd_f32_rows_per_utt(T, U1);
  float* g = reinterpret_cast<float*>(ws);
  float* z = g + (size_t)nb_max * rpu * V;
  float* dz = z + (size_t)nb_max * rpu * D;
  CTCVR_CHECK_CUDA(cudaMemsetAsync(d_w, 0, (size_t)V * D * sizeof(float), st));
  CTCVR_CHECK_CUDA(cudaMemsetAsync(d_b, 0, (size_t)V * sizeof(float), st));
  for (int b0 = 0; b0 < B; b0 += nb_max) {
    int nb = min(nb_max, B - b0);
    long R = (long)nb * rpu;
    JointTileArgs a{};
    a.enc = enc; a.pred = pred; a.w = w; a.bias = bias; a.targets = targets; a.t_len = t_len; a.u_len = u_len;
    a.B = B; a.T = T; a.U1 = U1; a.D = D; a.V = V; a.blank = blank; a.b0 = b0;
    a.lse_in = lse; a.alpha = alpha; a.beta = beta; a.costs = costs; a.grad_costs = grad_costs; a.clamp = clamp;
    a.g = g; a.z = z;
    if (int rc = launch_joint_tile<MODE_GRAD>(a, nb, st, act)) return rc;
    // dZ[R,D] = g[R,V] . W[V,D]
    {
      dim3 grid(cdiv(D, 64), cdiv(R, 64), 1);
      sgemm_kernel<false><<<grid, 256, 0, st>>>(g, w, dz, (int)R, D, V, V, D, D, V, 0);
      CTCVR_LAUNCH_CHECK();
    }
    // dW[V,D] += g^T[V,R] . z[R,D]   (split-K over rows, atomic accumulate)
    {
      long sp_ = R / 2048; if (sp_ < 1) sp_ = 1; if (sp_ > 64) sp_ = 64;
      int splits = (int)sp_;
      int kchunk = (int)(((R + splits - 1) / splits + 15) / 16 * 16);
      splits = cdiv(R, kchunk);
      dim3 grid(cdiv(D, 64), cdiv(V, 64), splits);
      sgemm_kernel<true><<<grid, 256, 0, st>>>(g, z, d_w, V, D, (int)R, V, D, D, kchunk, 1);
      CTCVR_LAUNCH_CHECK();
    }
    {
      long rows_per = 1024;
      dim3 grid(cdiv(V, 128), cdiv(R, rows_per));
      colsum_kernel<<<grid, 128, 0, st>>>(g, d_b, R, V, rows_per);
      CTCVR_LAUNCH_CHECK();
    }
    if (act == ACT_RELU)
      dh_enc_act_kernel<ACT_RELU><<<dim3(T, nb), 256, 0, st>>>(dz, enc, pred, t_len, u_len, d_enc, b0, T, U1, D);
    else if (act == ACT_GELU)
      dh_enc_act_kernel<ACT_GELU><<<dim3(T, nb), 256, 0, st>>>(dz, enc, pred, t_len, u_len, d_enc, b0, T, U1, D);
    else
      dh_enc_kernel<<<dim3(T, nb), 256, 0, st>>>(dz, z, d_enc, b0, T, U1, D);
    CTCVR_LAUNCH_CHECK();
    dh_pred_kernel<<<dim3(U1, nb), 256, 0, st>>>(dz, d_pred, b0, T, U1, D);
    CTCVR_LAUNCH_CHECK();
  }
  return 0;
}

}  // namespace ctcvr
