// Forward kernel of the bf16 tcgen05 path (included by joint_tc.cu).
//
//   z      = tanh(enc_proj[b,t,:] + pred_proj[b,u,:])        model/component/joint.py:57-67
//   logits = z . W_out^T + b_out                             model/component/joint.py:68
//   out    : lse, lp_blank, lp_label per lattice cell         log-softmax + gather of torchaudio rnnt_loss
//                                                             (model/component/transducer.py:180-187)
//
// Tiles: 128 lattice cells = nu label columns x (128/nu) consecutive frames of one utterance,
// nu in {4,2,1} (an utterance with W = U_b+1 columns is covered by W/4 groups of 4 columns and the
// binary remainder).  TMEM lane r = 32*q + lane holds cell (t0 + (q/nu)*32 + lane, u0 + q%nu), so the
// label of a cell is uniform across a warp and both gathered logits (blank, label) are one-column
// tcgen05.ld's instead of per-element compares.
//
// One persistent CTA per SM, 896 threads, warp-specialised (role loops run warp-wide, elect.sync around the
// single-thread instructions):
//   warp 0      bulk copies: pre-tiled bf16 W_out k-blocks (two N-halves per k-block) into a smem ring
//   warp 1      MMA issuer: tcgen05.mma M=128, N=Vp/2 (x2), K=16, A from TMEM, B from smem; fp32 accumulators in TMEM
//   warp 2      TMEM allocator
//   warp 3      TMA: slab ring - per k-block the nu pred rows and 128/nu enc rows (bf16, 128B swizzle)
//   warps 4-19  epilogue: tcgen05.ld (thread = cell, 4 column groups), online log-softmax in base 2, gathers, stores
//   warps 20-27 A producers: tanh(e+p) -> packed bf16 -> tcgen05.st into the A stage of TENSOR MEMORY (TS-mode MMA):
//               the A operand costs no shared-memory bandwidth, which is what bounds this kernel
#pragma once
#include "tc_common.cuh"

namespace ctcvr {
namespace tc {

constexpr int F_A_STAGES = 3;                    // A stages in TMEM: 32 columns each (64 k as bf16 pairs)
constexpr int F_EPI_GROUPS = 4;                  // epilogue column groups (4 warps each): more warps hide the TMEM-load and
                                                 // MUFU latencies of the softmax sweep, the phase no MMA overlaps
constexpr int F_EPI_WARPS = 4 * F_EPI_GROUPS;
constexpr int F_PROD_WARP0 = 4 + F_EPI_WARPS;    // first producer warp
constexpr int F_THREADS = (F_PROD_WARP0 + 8) * 32;   // 4 control + epilogue + 8 producer warps
constexpr int F_ACC_COLS = 416;                  // accumulator columns; the A stages follow (416 + 3*32 = 512)
constexpr int F_S_STAGES = 3;
constexpr int F_SLAB_BYTES = 1024 + 128 * 128;   // [pred rows: 1 KB region][128 enc rows x 128 B]
constexpr int F_MAX_W_STAGES = 6;

struct FwdParams {
  const __nv_bfloat16* w_t; // tiled W_out: [KB][2][NH][64] bf16, pre-swizzled (prep_weights3_kernel)
  const float* bias;       // [V]
  const float* bias_l2;    // [Vp] bias * log2(e), -inf beyond V
  const int32_t* targets;  // [B,U1-1]
  const int32_t* t_len;
  const int32_t* u_len;
  const int4* tiles;       // {b, u0, t0, nu}
  const int* ntiles;
  int B, T, U1, D, V, Vp, NH, blank, w_stages;
  float* lse;
  float* lp_blank;
  float* lp_label;
  long long* prof;
  unsigned int* err_host;   // mapped host word for bounded-wait time-outs (tc_common.cuh)
  const float* enc;         // bf16x3 only: the fp32 activations [B,T,D] / [B,U1,D], read in place
  const float* pred;
  // vocabulary tiles (VT kernels only): this launch covers columns [v0, v0 + V) of a vocabulary of Vg entries whose
  // blank is blank_g; bias / w_t / bias_l2 are the tile's, blank is the tile's blank column or -1.  merge: lse holds
  // the log-sum-exp of the earlier tiles (merged in place); lp_blank / lp_label receive raw logit + bias.
  int v0, Vg, blank_g, merge;
};

// vocabulary tiles: a label of the full vocabulary -> its column in the tile [v0, v0 + Vc), -1 when another tile holds
// it.  Ids outside [0, Vg) act as the blank, as in the untiled kernels.
__device__ __forceinline__ int vt_column(int lab, int Vg, int blank_g, int v0, int Vc) {
  if ((unsigned)lab >= (unsigned)Vg) lab = blank_g;
  lab -= v0;
  return ((unsigned)lab < (unsigned)Vc) ? lab : -1;
}

// log(exp(a) + exp(b)) in fp32 (accurate functions: once per cell and tile)
__device__ __forceinline__ float logaddexp_f32(float a, float b) {
  const float m = fmaxf(a, b);
  return (m == kNegInf) ? m : m + log1pf(expf(-fabsf(a - b)));
}

struct FwdSmem {
  uint32_t a_base, w_base, w_bytes, s_base, bar_base;
  float* bias_l2;
  float2* epi_x;            // [groups - 1][128] (max, sum) of epilogue groups 1..
  uint32_t* tmem_ptr;
  __device__ __forceinline__ uint32_t a_stage(int i) const { return a_base + i * A_STAGE_BYTES; }
  __device__ __forceinline__ uint32_t w_stage(int i) const { return w_base + i * w_bytes; }
  __device__ __forceinline__ uint32_t s_stage(int i) const { return s_base + i * F_SLAB_BYTES; }
  __device__ __forceinline__ uint32_t a_full(int i) const { return bar_base + i * 16; }
  __device__ __forceinline__ uint32_t a_empty(int i) const { return bar_base + i * 16 + 8; }
  __device__ __forceinline__ uint32_t s_full(int i) const { return bar_base + 64 + i * 16; }
  __device__ __forceinline__ uint32_t s_empty(int i) const { return bar_base + 64 + i * 16 + 8; }
  __device__ __forceinline__ uint32_t w_full(int i) const { return bar_base + 128 + i * 16; }
  __device__ __forceinline__ uint32_t w_empty(int i) const { return bar_base + 128 + i * 16 + 8; }
  __device__ __forceinline__ uint32_t tmem_full() const { return bar_base + 224; }
  __device__ __forceinline__ uint32_t tmem_empty() const { return bar_base + 232; }
};

__host__ __device__ inline size_t fwd2_smem_bytes(int NH, int Vp, int w_stages) {
  size_t s = 1024;
  s += (size_t)w_stages * NH * 128;
  s = (s + 1023) / 1024 * 1024;
  s += (size_t)F_S_STAGES * F_SLAB_BYTES;
  s += (size_t)Vp * 4 + 1024 * (F_EPI_GROUPS - 1);
  s += 256 + 16;
  return s;
}

__device__ __forceinline__ void carve_fwd2(FwdSmem& L, uint8_t* raw, int NH, int Vp, int w_stages) {
  const uint32_t base = smem_u32(raw);
  uint32_t a = (base + 1023u) & ~1023u;
  L.a_base = a;
  L.w_base = a; L.w_bytes = NH * 128; a += w_stages * NH * 128;
  a = (a + 1023u) & ~1023u;
  L.s_base = a; a += F_S_STAGES * F_SLAB_BYTES;
  L.bias_l2 = reinterpret_cast<float*>(raw + (a - base)); a += Vp * 4;
  a = (a + 15u) & ~15u;
  L.epi_x = reinterpret_cast<float2*>(raw + (a - base)); a += 1024 * (F_EPI_GROUPS - 1);
  L.bar_base = a; a += 256;
  L.tmem_ptr = reinterpret_cast<uint32_t*>(raw + (a - base));
}


// z = act(e + p) in fp32 (tanhf / erff: accurate, the build does not use fast-math) for 8 consecutive k, split into
// hi = bf16_rn(z) and lo = bf16_rn(z - hi) as packed pairs (low half = even k, the TMEM operand layout)
template <int ACT = ACT_TANH>
__device__ __forceinline__ void tanh_split8(const float4& e0, const float4& e1, const float4& p0, const float4& p1,
                                            uint32_t* hi, uint32_t* lo) {
  const float z[8] = {act_f32<ACT>(e0.x + p0.x), act_f32<ACT>(e0.y + p0.y), act_f32<ACT>(e0.z + p0.z),
                      act_f32<ACT>(e0.w + p0.w), act_f32<ACT>(e1.x + p1.x), act_f32<ACT>(e1.y + p1.y),
                      act_f32<ACT>(e1.z + p1.z), act_f32<ACT>(e1.w + p1.w)};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(z[2 * j], z[2 * j + 1]);
    hi[j] = *reinterpret_cast<const uint32_t*>(&h);
    lo[j] = pack_bf16(z[2 * j] - __low2float(h), z[2 * j + 1] - __high2float(h));
  }
}

// SPLIT = false: the bf16 kernel.  SPLIT = true (precision bf16x3): every operand x is hi + lo (bf16 each) and the
// logits accumulate z_hi W_hi + z_lo W_hi + z_hi W_lo, three MMA passes per k-block into the same accumulators.
//   W ring   : per k-block four stages (W_hi half 0, 1, W_lo half 0, 1) from w_t = [KB][hi, lo][2][NH][64]
//   A stages : per k-block two TMEM stages (z_hi, z_lo of its 64 k): the same 3 x 32 columns as bf16
//   producers: read the fp32 enc / pred rows straight from global memory (L2-resident), no slab ring (warp 3 idles)
// ACT: the joint activation (ACT_TANH / ACT_RELU / ACT_GELU), applied by the A producers.
// VT: one vocabulary tile of a larger vocabulary (FwdParams v0 ..): the epilogue merges the tile's log-sum-exp into lse
// and writes the raw blank / label logits of the columns it holds; vt_finalize_kernel subtracts the final lse.
template <bool SPLIT, int ACT = ACT_TANH, bool VT = false>
__device__ __forceinline__ void joint_fwd2_body(const CUtensorMap& tmap_e, const CUtensorMap& tmap_p, const FwdParams& p) {
  extern __shared__ uint8_t smem_raw[];
  FwdSmem L;
  carve_fwd2(L, smem_raw, p.NH, p.Vp, p.w_stages);
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int KB = p.D / BK;
  const int ntiles = *p.ntiles;
  const int WS = p.w_stages;

  if (warp == 0 && lane == 0) {
    g_tc_error_host = p.err_host;
    if (!SPLIT) {                    // the split form gets placeholder tensor maps
      tma_prefetch_desc(&tmap_e);
      tma_prefetch_desc(&tmap_p);
    }
    for (int i = 0; i < F_A_STAGES; ++i) { mbar_init(L.a_full(i), PROD_THREADS / 32); mbar_init(L.a_empty(i), 1); }
    for (int i = 0; i < F_S_STAGES; ++i) { mbar_init(L.s_full(i), 1); mbar_init(L.s_empty(i), PROD_THREADS / 32); }
    for (int i = 0; i < F_MAX_W_STAGES; ++i) { mbar_init(L.w_full(i), 1); mbar_init(L.w_empty(i), 1); }
    mbar_init(L.tmem_full(), 1);
    mbar_init(L.tmem_empty(), F_EPI_WARPS);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_u32(L.tmem_ptr), TMEM_COLS);
  for (int i = tid; i < p.Vp; i += F_THREADS) L.bias_l2[i] = p.bias_l2[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *L.tmem_ptr;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA: W_out k-blocks (warp-wide loop, one lane issues)
    Pipe wp;
    const uint32_t w_bytes = (uint32_t)p.NH * 128u;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
      for (int i = 0; i < (SPLIT ? 4 : 2) * KB; ++i) {
        mbar_wait(L.w_empty(wp.stage), wp.phase ^ 1u, 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(L.w_full(wp.stage), w_bytes);
          bulk_load(L.w_stage(wp.stage), p.w_t + (size_t)i * p.NH * 64, w_bytes, L.w_full(wp.stage));
        }
        __syncwarp();
        wp.advance(WS);
      }
  } else if (warp == 3 && !SPLIT) {
    // ------------------------------------------------------------------ TMA: enc / pred slabs
    Pipe sp;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      const int4 ti = p.tiles[tile];
      const int nbox = 4 / ti.w;                       // 32-frame boxes: 128/nu frames
      const int prow = ti.x * p.U1 + ti.y;
      const int erow = ti.x * p.T + ti.z;
      for (int kb = 0; kb < KB; ++kb) {
        mbar_wait(L.s_empty(sp.stage), sp.phase ^ 1u, 2);
        if (elect_one()) {
          const uint32_t st = L.s_stage(sp.stage);
          mbar_arrive_expect_tx(L.s_full(sp.stage), 512u + (uint32_t)nbox * 4096u);
          tma_load_2d(st, &tmap_p, L.s_full(sp.stage), kb * BK, prow);
          for (int i = 0; i < nbox; ++i)
            tma_load_2d(st + 1024 + i * 4096, &tmap_e, L.s_full(sp.stage), kb * BK, erow + 32 * i);
        }
        __syncwarp();
        sp.advance(F_S_STAGES);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (warp-wide loop, one lane issues)
    Pipe ap, wp;
    uint32_t tphase = 0;
    int prof_n = 0;
    const uint32_t idesc = make_idesc_bf16(BM, p.NH);
    const uint64_t w_desc0 = make_desc_sw128(L.w_stage(0));
    const uint32_t w_step = (uint32_t)p.NH * 8u;         // one ring stage, in 16-byte descriptor units
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      if (lane == 0) TC_PROF(1, 100);
      mbar_wait(L.tmem_empty(), tphase ^ 1u, 3);
      if (lane == 0) TC_PROF(1, 101);
      tc_fence_after();
      if constexpr (SPLIT) {
        for (int kb = 0; kb < KB; ++kb) {
          Pipe al = ap;                                  // z_lo stage follows the z_hi stage
          al.advance(F_A_STAGES);
          mbar_wait(L.a_full(ap.stage), ap.phase, 4);
          mbar_wait(L.a_full(al.stage), al.phase, 4);
          for (int j = 0; j < 4; ++j) {                  // W_hi half 0, 1, W_lo half 0, 1
            const int h = j & 1;
            mbar_wait(L.w_full(wp.stage), wp.phase, 5);
            tc_fence_after();
            if (elect_one()) {
              const uint64_t bd = w_desc0 + (uint64_t)(wp.stage * w_step);
              const uint32_t d = tmem_base + h * p.NH;
              const uint32_t a = tmem_base + F_ACC_COLS + ap.stage * 32;
              const uint32_t a2 = tmem_base + F_ACC_COLS + al.stage * 32;
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4) umma_bf16_ts(d, a + 8 * k4, bd + 2 * k4, idesc, (kb || j >= 2 || k4) ? 1u : 0u);
              if (j < 2) {
#pragma unroll
                for (int k4 = 0; k4 < 4; ++k4) umma_bf16_ts(d, a2 + 8 * k4, bd + 2 * k4, idesc, 1u);
              }
              umma_commit(L.w_empty(wp.stage));
              if (j == 3) { umma_commit(L.a_empty(ap.stage)); umma_commit(L.a_empty(al.stage)); }
            }
            __syncwarp();
            wp.advance(WS);
          }
          ap.advance(F_A_STAGES);
          ap.advance(F_A_STAGES);
        }
      } else
      for (int kb = 0; kb < KB; ++kb) {
        mbar_wait(L.a_full(ap.stage), ap.phase, 4);
        for (int h = 0; h < 2; ++h) {
          mbar_wait(L.w_full(wp.stage), wp.phase, 5);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t bd = w_desc0 + (uint64_t)(wp.stage * w_step);
            const uint32_t d = tmem_base + h * p.NH;
            const uint32_t a = tmem_base + F_ACC_COLS + ap.stage * 32;
            umma_bf16_ts(d, a, bd, idesc, kb ? 1u : 0u);
            umma_bf16_ts(d, a + 8, bd + 2, idesc, 1u);
            umma_bf16_ts(d, a + 16, bd + 4, idesc, 1u);
            umma_bf16_ts(d, a + 24, bd + 6, idesc, 1u);
            umma_commit(L.w_empty(wp.stage));
            if (h == 1) umma_commit(L.a_empty(ap.stage));
          }
          __syncwarp();
          wp.advance(WS);
        }
        ap.advance(F_A_STAGES);
      }
      if (elect_one()) umma_commit(L.tmem_full());
      __syncwarp();
      tphase ^= 1u;
    }
  } else if (warp >= 4 && warp < F_PROD_WARP0) {
    // ------------------------------------------------------------------ epilogue: online log-softmax (base 2)
    // quarter q = TMEM lanes 32q..32q+31 (thread = cell), group eg = which slice of the accumulator columns.
    // The groups keep their own (max, sum); groups 1.. hand their pairs to group 0 through shared memory.
    const int q = warp & 3, eg = (warp - 4) >> 2;
    const int erow = q * 32 + lane;
    const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t tphase = 0;
    int prof_n = 0;
    const float bias_blank = (VT && p.blank < 0) ? 0.f : __ldg(p.bias + p.blank);
    // column chunks of 16, dealt to the groups in contiguous runs
    const int nch = p.Vp / 16;
    const int c_begin = (nch * eg / F_EPI_GROUPS) * 16, c_end = (nch * (eg + 1) / F_EPI_GROUPS) * 16;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      int4 ti = p.tiles[tile];
      pin(ti.x); pin(ti.y); pin(ti.z); pin(ti.w);
      const int b = ti.x, nu = ti.w;
      const int lognu = nu >> 1;                          // 4 -> 2, 2 -> 1, 1 -> 0
      const int u = ti.y + (q & (nu - 1));
      const int t = ti.z + ((q >> lognu) << 5) + lane;
      int Tb = max(min(p.t_len[b], p.T), 0), Ub = max(min(p.u_len[b], p.U1 - 1), 0);
      pin(Tb); pin(Ub);
      const bool valid = t < Tb;
      int lab = -1;
      float bias_lab = 0.f;
      if (eg == 0 && u < Ub) {
        lab = p.targets[(size_t)b * (p.U1 - 1) + u];
        if (VT) lab = vt_column(lab, p.Vg, p.blank_g, p.v0, p.V);
        else if ((unsigned)lab >= (unsigned)p.V) lab = p.blank;    // out-of-range ids cannot index outside the tile
        if (!VT || lab >= 0) bias_lab = __ldg(p.bias + lab);
      }
      pin(lab);
      mbar_wait(L.tmem_full(), tphase, 6);
      if (tid == 128) TC_PROF(2, 1);
      tc_fence_after();
      float xb = 0.f, xl = 0.f;
      if (eg == 0) { xb = tmem_ld1(tq + (VT ? max(p.blank, 0) : p.blank)); xl = tmem_ld1(tq + (lab >= 0 ? lab : 0)); }
      float m = kNegInf, s = 0.f;
      float v[16];
      if (c_begin < c_end) tmem_ld16(tq + c_begin, v);
      for (int c0 = c_begin; c0 < c_end; c0 += 16) {
        tmem_ld_wait();
        float y[16];
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          const float4 bj = *reinterpret_cast<const float4*>(L.bias_l2 + c0 + j);
          y[j] = fmaf(v[j], LOG2E, bj.x);
          y[j + 1] = fmaf(v[j + 1], LOG2E, bj.y);
          y[j + 2] = fmaf(v[j + 2], LOG2E, bj.z);
          y[j + 3] = fmaf(v[j + 3], LOG2E, bj.w);
        }
        if (c0 + 16 < c_end) tmem_ld16(tq + c0 + 16, v);    // next chunk in flight during the math below
        float cm[4] = {kNegInf, kNegInf, kNegInf, kNegInf};
#pragma unroll
        for (int j = 0; j < 16; j += 4)
#pragma unroll
          for (int e = 0; e < 4; ++e) cm[e] = fmaxf(cm[e], y[j + e]);
        const float nm = fmaxf(m, fmaxf(fmaxf(cm[0], cm[1]), fmaxf(cm[2], cm[3])));
        // a group whose columns so far are all padding (bias -inf) has nm = -inf: subtract 0 instead (every term is 0)
        const float nz = (nm == kNegInf) ? 0.f : nm;
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < 16; j += 4)
#pragma unroll
          for (int e = 0; e < 4; ++e) acc[e] += ex2_fast(y[j + e] - nz);
        s = s * ex2_fast(m - nz) + ((acc[0] + acc[1]) + (acc[2] + acc[3]));
        m = nm;
      }
      tc_fence_before();
      warp_arrive(L.tmem_empty());
      if (tid == 128) TC_PROF(2, 2);
      if (eg > 0) { L.epi_x[(eg - 1) * 128 + erow] = make_float2(m, s); }
      named_barrier_sync(3, F_EPI_WARPS * 32);             // the other groups' partials are visible
      if (eg == 0) {
#pragma unroll
        for (int gi = 0; gi < F_EPI_GROUPS - 1; ++gi) {
          const float2 o = L.epi_x[gi * 128 + erow];
          const float nm = fmaxf(m, o.x);
          const float nz = (nm == kNegInf) ? 0.f : nm;
          s = s * ex2_fast(m - nz) + o.y * ex2_fast(o.x - nz);
          m = nm;
        }
        if (valid) {
          const size_t cell = ((size_t)b * p.T + t) * p.U1 + u;
          const float l = (m + lg2_fast(s)) * LN2;
          if constexpr (VT) {
            p.lse[cell] = p.merge ? logaddexp_f32(p.lse[cell], l) : l;
            if (p.blank >= 0) p.lp_blank[cell] = xb + bias_blank;
            if (lab >= 0) p.lp_label[cell] = xl + bias_lab;
          } else {
            p.lse[cell] = l;
            p.lp_blank[cell] = xb + bias_blank - l;
            p.lp_label[cell] = (lab >= 0) ? xl + bias_lab - l : kNegInf;
          }
        }
      }
      named_barrier_sync(3, F_EPI_WARPS * 32);             // partials consumed before the next tile overwrites them
      tphase ^= 1u;
    }
  } else if (warp >= F_PROD_WARP0 && SPLIT) {
    // ------------------------------------------------------------------ bf16x3 A producers: fp32 rows from global
    // thread = tile row 32q + lane, k-half kh: 32 k per k-block -> 16 hi columns (stage a) + 16 lo columns (stage a + 1)
    const int q = warp & 3, kh = (warp - F_PROD_WARP0) >> 2;
    const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16);
    Pipe ap;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      int4 ti = p.tiles[tile];
      pin(ti.x); pin(ti.y); pin(ti.z); pin(ti.w);
      const int lognu = ti.w >> 1;
      const int u = ti.y + (q & (ti.w - 1));
      const int t = min(ti.z + ((q >> lognu) << 5) + lane, p.T - 1);     // rows past the utterance are discarded
      const float4* er = reinterpret_cast<const float4*>(p.enc + ((size_t)ti.x * p.T + t) * p.D + kh * 32);
      const float4* pr = reinterpret_cast<const float4*>(p.pred + ((size_t)ti.x * p.U1 + u) * p.D + kh * 32);
      for (int kb = 0; kb < KB; ++kb) {
        Pipe al = ap;
        al.advance(F_A_STAGES);
        const uint32_t c_hi = (uint32_t)(F_ACC_COLS + ap.stage * 32 + kh * 16), c_lo = (uint32_t)(F_ACC_COLS + al.stage * 32 + kh * 16);
#pragma unroll
        for (int c = 0; c < 2; ++c) {                   // 16 k per round: 8 hi + 8 lo columns
          const float4* e4 = er + kb * 16 + c * 4;
          const float4* p4 = pr + kb * 16 + c * 4;
          const float4 e0 = __ldg(e4), e1 = __ldg(e4 + 1), e2 = __ldg(e4 + 2), e3 = __ldg(e4 + 3);
          const float4 p0 = __ldg(p4), p1 = __ldg(p4 + 1), p2 = __ldg(p4 + 2), p3 = __ldg(p4 + 3);
          uint32_t hi[8], lo[8];
          tanh_split8<ACT>(e0, e1, p0, p1, hi, lo);
          tanh_split8<ACT>(e2, e3, p2, p3, hi + 4, lo + 4);
          if (c == 0) {
            mbar_wait(L.a_empty(ap.stage), ap.phase ^ 1u, 8);
            mbar_wait(L.a_empty(al.stage), al.phase ^ 1u, 8);
            tc_fence_after();
          }
          tmem_st8(tq + c_hi + c * 8, hi);
          tmem_st8(tq + c_lo + c * 8, lo);
        }
        tmem_st_wait();
        tc_fence_before();
        warp_arrive(L.a_full(ap.stage));
        warp_arrive(L.a_full(al.stage));
        ap.advance(F_A_STAGES);
        ap.advance(F_A_STAGES);
      }
    }
  } else if (warp >= F_PROD_WARP0) {
    // ------------------------------------------------------------------ A producers (A operand lives in TMEM)
    // warp = (TMEM lane quarter q, k-half kh): thread = tile row 32q + lane, 32 of the 64 k of a k-block.
    // tanh(e + p) for 32 k -> 16 packed bf16x2 -> one tcgen05.st into the A stage columns of the thread's own lane.
    const int q = warp & 3, kh = (warp - F_PROD_WARP0) >> 2;
    Pipe ap, sp;
    int prof_n = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      int nu = p.tiles[tile].w;
      pin(nu);
      const int lognu = nu >> 1;
      const int ul = q & (nu - 1);
      const int tloc = ((q >> lognu) << 5) + lane;
      const uint32_t e_row = 1024u + (uint32_t)tloc * 128u, e_sw = (uint32_t)(tloc & 7);
      const uint32_t p_row = (uint32_t)ul * 128u, p_sw = (uint32_t)ul;
      for (int kb = 0; kb < KB; ++kb) {
        mbar_wait(L.s_full(sp.stage), sp.phase, 7);
        mbar_wait(L.a_empty(ap.stage), ap.phase ^ 1u, 8);
        if (tid == F_PROD_WARP0 * 32) TC_PROF(3, kb);
        tc_fence_after();
        const uint32_t sb = L.s_stage(sp.stage);
        uint32_t w[16];
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
          const uint32_t c = (uint32_t)(kh * 4 + c4);
          const uint4 ev = lds128(sb + e_row + ((c ^ e_sw) << 4));
          const uint4 pv = lds128(sb + p_row + ((c ^ p_sw) << 4));
          w[4 * c4 + 0] = act_add_bf16x2_packed<ACT>(ev.x, pv.x);
          w[4 * c4 + 1] = act_add_bf16x2_packed<ACT>(ev.y, pv.y);
          w[4 * c4 + 2] = act_add_bf16x2_packed<ACT>(ev.z, pv.z);
          w[4 * c4 + 3] = act_add_bf16x2_packed<ACT>(ev.w, pv.w);
        }
        tmem_st16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(F_ACC_COLS + ap.stage * 32 + kh * 16), w);
        tmem_st_wait();
        tc_fence_before();
        warp_arrive(L.a_full(ap.stage));
        warp_arrive(L.s_empty(sp.stage));
        if (tid == F_PROD_WARP0 * 32) TC_PROF(3, 20 + kb);
        ap.advance(F_A_STAGES);
        sp.advance(F_S_STAGES);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

__global__ void __launch_bounds__(F_THREADS, 1)
joint_fwd2_kernel(const __grid_constant__ CUtensorMap tmap_e, const __grid_constant__ CUtensorMap tmap_p,
                  const FwdParams p) {
  joint_fwd2_body<false>(tmap_e, tmap_p, p);
}
// precision bf16x3 (the tensor maps are unused: the producers read the fp32 rows directly)
__global__ void __launch_bounds__(F_THREADS, 1)
joint_fwd2_x3_kernel(const __grid_constant__ CUtensorMap tmap_e, const __grid_constant__ CUtensorMap tmap_p,
                     const FwdParams p) {
  joint_fwd2_body<true>(tmap_e, tmap_p, p);
}
// relu / gelu joints: the same kernels with the activation of the A producers swapped, named apart for profiler traces
#define CTCVR_FWD2_ACT(name, split, act)                                                                           \
  __global__ void __launch_bounds__(F_THREADS, 1)                                                                   \
  name(const __grid_constant__ CUtensorMap tmap_e, const __grid_constant__ CUtensorMap tmap_p, const FwdParams p) { \
    joint_fwd2_body<split, act>(tmap_e, tmap_p, p);                                                                 \
  }
CTCVR_FWD2_ACT(joint_fwd2_relu_kernel, false, ACT_RELU)
CTCVR_FWD2_ACT(joint_fwd2_gelu_kernel, false, ACT_GELU)
CTCVR_FWD2_ACT(joint_fwd2_x3_relu_kernel, true, ACT_RELU)
CTCVR_FWD2_ACT(joint_fwd2_x3_gelu_kernel, true, ACT_GELU)
#undef CTCVR_FWD2_ACT
// vocabulary tiles (ctcvr_joint_rnnt_fwd_vt): one launch per tile of the vocabulary
#define CTCVR_FWD2_VT(name, split, act)                                                                            \
  __global__ void __launch_bounds__(F_THREADS, 1)                                                                   \
  name(const __grid_constant__ CUtensorMap tmap_e, const __grid_constant__ CUtensorMap tmap_p, const FwdParams p) { \
    joint_fwd2_body<split, act, true>(tmap_e, tmap_p, p);                                                           \
  }
CTCVR_FWD2_VT(joint_fwd2_vt_kernel, false, ACT_TANH)
CTCVR_FWD2_VT(joint_fwd2_vt_relu_kernel, false, ACT_RELU)
CTCVR_FWD2_VT(joint_fwd2_vt_gelu_kernel, false, ACT_GELU)
CTCVR_FWD2_VT(joint_fwd2_x3_vt_kernel, true, ACT_TANH)
CTCVR_FWD2_VT(joint_fwd2_x3_vt_relu_kernel, true, ACT_RELU)
CTCVR_FWD2_VT(joint_fwd2_x3_vt_gelu_kernel, true, ACT_GELU)
#undef CTCVR_FWD2_VT

// Tile table of the forward kernel: per utterance (W/4) groups of 4 label columns x 32-frame blocks, then a
// 2-column group x 64-frame blocks if W & 2, then a 1-column group x 128-frame blocks if W & 1 (64-frame blocks for
// the CTA-pair kernel, joint_tc_fwd_pair.cuh).
__device__ __forceinline__ int fwd_tiles_of(int Tb, int W, int pair) {
  if (Tb <= 0) return 0;
  const int n1 = pair ? ((Tb + 63) >> 6) : ((Tb + 127) >> 7);
  return (W >> 2) * ((Tb + 31) >> 5) + ((W & 2) ? ((Tb + 63) >> 6) : 0) + ((W & 1) ? n1 : 0);
}

}  // namespace tc
}  // namespace ctcvr
