// torchaudio-compatible transducer loss on DENSE logits (the "loss op kept separate" seam):
// torch.ops.torchaudio.rnnt_loss_forward(logits, targets, logit_lengths, target_lengths, blank,
// clamp, fused_log_softmax=True) -> (costs, grads)   site-packages/torchaudio/functional/functional.py:1725
// Used when a caller hands us materialised [B,T,U1,V] logits (e.g. TransducerJoint.forward called
// directly).  The fused op in joint_simt.cu / joint_tc.cu is the hot path; this one reads the logits
// twice (stats, gradient) instead of torchaudio's four passes.
// Lengths are clamped to [0, T] and [0, U1 - 1] exactly as the lattice (lattice.cu) clamps them, and a label outside
// [0, V) is read as blank, so both kernels and the lattice see one utterance and nothing indexes outside the tensors.
#include "common.cuh"

namespace ctcvr {

int rnnt_lattice(const float*, const float*, const int32_t*, const int32_t*, float*, float*, float*, int, int, int,
                 cudaStream_t);

// one warp per lattice cell: lse, lp_blank, lp_label
__global__ void dense_stats_kernel(const float* __restrict__ logits, const int32_t* __restrict__ targets,
                                   const int32_t* __restrict__ t_len, const int32_t* __restrict__ u_len,
                                   float* __restrict__ lse, float* __restrict__ lpb, float* __restrict__ lpl, int B,
                                   int T, int U1, int V, int blank) {
  long cell = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (cell >= (long)B * T * U1) return;
  int lane = threadIdx.x & 31;
  int u = cell % U1;
  int t = (cell / U1) % T;
  int b = cell / ((long)U1 * T);
  const int Tb = max(min(t_len[b], T), 0), Ub = max(min(u_len[b], U1 - 1), 0);
  if (t >= Tb || u > Ub) return;
  const float* x = logits + cell * V;
  float m = kNegInf;
  for (int v = lane; v < V; v += 32) m = fmaxf(m, x[v]);
  m = warp_max(m);
  float s = 0.f;
  for (int v = lane; v < V; v += 32) s += expf(x[v] - m);
  s = warp_sum(s);
  if (lane == 0) {
    float l = m + logf(s);
    lse[cell] = l;
    lpb[cell] = x[blank] - l;
    if (u < Ub) {
      int lab = targets[(long)b * (U1 - 1) + u];
      if ((unsigned)lab >= (unsigned)V) lab = blank;
      lpl[cell] = x[lab] - l;
    } else {
      lpl[cell] = kNegInf;
    }
  }
}

// one warp per lattice cell: dense gradient row (exact zeros at padded cells)
__global__ void dense_grad_kernel(const float* __restrict__ logits, const int32_t* __restrict__ targets,
                                  const int32_t* __restrict__ t_len, const int32_t* __restrict__ u_len,
                                  const float* __restrict__ lse, const float* __restrict__ alpha,
                                  const float* __restrict__ beta, const float* __restrict__ costs,
                                  float* __restrict__ grads, int B, int T, int U1, int V, int blank, float clamp) {
  long cell = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (cell >= (long)B * T * U1) return;
  int lane = threadIdx.x & 31;
  int u = cell % U1;
  int t = (cell / U1) % T;
  int b = cell / ((long)U1 * T);
  float* g = grads + cell * V;
  const int Tb = max(min(t_len[b], T), 0), Ub = max(min(u_len[b], U1 - 1), 0);
  if (t >= Tb || u > Ub) {
    for (int v = lane; v < V; v += 32) g[v] = 0.f;
    return;
  }
  const float* x = logits + cell * V;
  float al = alpha[cell], be = beta[cell], cost = costs[b], l = lse[cell];
  float k_all = al + be + cost - l;
  float bnext = kNegInf;
  if (t + 1 < Tb) bnext = beta[cell + U1];
  else if (u == Ub) bnext = 0.f;
  float k_blank = al + bnext + cost - l;
  float k_label = kNegInf;
  int lab = -1;
  if (u < Ub) {
    k_label = al + beta[cell + 1] + cost - l;
    lab = targets[(long)b * (U1 - 1) + u];
    if ((unsigned)lab >= (unsigned)V) lab = blank;
  }
  for (int v = lane; v < V; v += 32) {
    float xv = x[v];
    float gv = expf(xv + k_all);
    if (v == blank && k_blank != kNegInf) gv -= expf(xv + k_blank);
    if (v == lab) gv -= expf(xv + k_label);
    if (clamp > 0.f) gv = fminf(fmaxf(gv, -clamp), clamp);
    g[v] = gv;
  }
}

int rnnt_loss_dense(const float* logits, const int32_t* targets, const int32_t* t_len, const int32_t* u_len,
                    float* costs, float* grads, int B, int T, int U1, int V, int blank, float clamp, void* ws,
                    size_t ws_bytes, cudaStream_t st) {
  size_t n = (size_t)B * T * U1;
  CTCVR_REQUIRE(ws_bytes >= 5 * n * sizeof(float), "rnnt_loss_dense: workspace too small");
  float* lse = reinterpret_cast<float*>(ws);
  float* lpb = lse + n;
  float* lpl = lpb + n;
  float* alpha = lpl + n;
  float* beta = alpha + n;
  const int warps = 8;
  int grid = cdiv((long)n, warps);
  dense_stats_kernel<<<grid, warps * 32, 0, st>>>(logits, targets, t_len, u_len, lse, lpb, lpl, B, T, U1, V, blank);
  CTCVR_LAUNCH_CHECK();
  if (int rc = rnnt_lattice(lpb, lpl, t_len, u_len, alpha, beta, costs, B, T, U1, st)) return rc;
  if (grads) {
    dense_grad_kernel<<<grid, warps * 32, 0, st>>>(logits, targets, t_len, u_len, lse, alpha, beta, costs, grads, B,
                                                   T, U1, V, blank, clamp);
    CTCVR_LAUNCH_CHECK();
  }
  return 0;
}

}  // namespace ctcvr
