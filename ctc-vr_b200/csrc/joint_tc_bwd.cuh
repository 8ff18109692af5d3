// Backward kernel 1 of the bf16 tcgen05 path (included by joint_tc.cu):
//   recompute logits -> g = d cost / d logits -> dZ^T = W^T g^T -> dH = dZ (1 - z^2) -> d_enc / d_pred partials,
//   d_bias, and the bf16 spill of the G tiles consumed by the dW GEMM (kernel 2, which recomputes z).
//   (model/component/joint.py:57-68 + torchaudio rnnt_loss backward, model/component/transducer.py:180-187)
//
// Tiles are rectangles of TT frames x P label columns of one utterance (row = tloc*P + ul; <21,6> or <16,8>).
// With the transposed second GEMM (TMEM lane = joint dim d, TMEM column = tile row) both reductions are
// thread-local:
//   d_enc[t]  = sum over the P columns of a frame
//   d_pred[u] = sum over the frame slots, kept in registers across the tiles of one (b, u-split) sweep
// TMEM holds 512 columns, so the logits [128 x Vp] and dZ^T [D x 128] cannot coexist: a tile runs its phases on one CTA
//   P1  12 warps : tanh k-half slots -> A operand in TMEM (tcgen05.st) | bulk copies: W_out k-blocks | MMA (TS): logits
//   P2  12 warps : TMEM -> g (bf16) -> smem G tile (K-major over v); the blank / label entries are patched in fp32 from
//                  the forward's lp_blank / lp_label by the thread that wrote the piece (no TMEM gathers, no barrier)
//   P3  bulk copies: W_out^T blocks | MMA (SS): dZ^T[mb] = W^T[mb] . G^T -> TMEM, one commit PER d block |
//                  warp 0 bulk-stores the G tile between the stage loads, warps 12-15 sum its columns (d_bias)
//   P4  warps 4-11, overlapped with P3: as soon as d block mb is committed, dH = dZ * (1 - z^2) with z RECOMPUTED from
//                  the tile's enc / pred rows (a TMA-staged slab of the whole joint dim): one packed tanh per two
//                  elements instead of a z^T round trip through shared memory and L2.  Warp group wg owns d blocks wg, wg+2,
//                  so only the last block's P4 is exposed after the MMAs.
// W_out streams through a ring that spans the (then idle) G region in P1 (up to 6 stages of NH*128 B); W_out^T through
// the first 64 KB of the same memory in P3 (4 x 16 KB).
//
// Roles (512 threads): warp 0 bulk-copy ring | warp 1 MMA issuer | warp 2 TMEM alloc | warp 3 TMA slabs |
// warps 4-15: P1 A producers, P2 workers, (4-11) P4 workers, (12-15) d_bias.  Role loops run warp-wide with
// elect.sync around the single-thread instructions (tc_common.cuh: elect_one).
#pragma once
#include "tc_common.cuh"

#ifndef CTCVR_EXP
#define CTCVR_EXP 0        // tools/exp_build.sh: timing experiments that drop a piece of the kernel (results invalid)
#endif

namespace ctcvr {
namespace tc {

constexpr int B_A_STAGES = 3;
constexpr int B_ACC_COLS = 416;                // TMEM: logits [0, 416) | A stages 416 + 32*stage (P1) ; dZ^T [0, 512) (P3/P4)
constexpr int B_S_STAGES = 2;
constexpr int B_R1_MAX = 6;                    // W_out ring view   (P1): NH x 128 B per stage, over ring + G region
constexpr int B_R3_STAGES = 4;                 // W_out^T ring view (P3): 16 KB per stage
constexpr int B_RING_BYTES = B_R3_STAGES * 16384;
constexpr int B_SLAB_MAX = 4096;               // slab stage of the largest tile geometry: 24 pred rows (3 KB) + 8 enc rows

// Tile geometry of the single-CTA kernel: TT frames x P label columns, row = tloc*P + ul (TT*P <= 128).
//   <16, 8> : 128 rows, u-splits of <= 16 columns          <21, 6> : 126 rows, u-splits of <= 21 columns
// The host picks the variant that wastes fewer rows for the batch's U (U+1 = 41 -> 2 x 21: 2.4% padding vs 14.6%).
template <int P, int TT>
struct BwdGeom {
  int b, Tb, Ub, W, us, t0, ubase;
  __device__ __forceinline__ void init(const int32_t* t_len, const int32_t* u_len, int T, int U1, int4 ti) {
    b = ti.x;
    Tb = max(min(t_len[b], T), 0);
    Ub = max(min(u_len[b], U1 - 1), 0);
    W = Ub + 1;
    const int S = (W + P - 1) / P;
    us = (W + S - 1) / S;
    t0 = ti.z * TT;
    ubase = ti.y * us;
    pin(b); pin(Tb); pin(Ub); pin(W); pin(us); pin(t0); pin(ubase);
  }
  // tile row -> lattice cell; false for padding rows
  __device__ __forceinline__ bool cell(int r, int& t, int& u, int& ul) const {
    const int tloc = r / P;
    ul = r - tloc * P;
    t = t0 + tloc;
    u = ubase + ul;
    return tloc < TT && t < Tb && ul < us && u <= Ub;
  }
};
template <int P>
__host__ __device__ constexpr uint32_t bwd_pred_region() { return (uint32_t)((P * 128 + 1023) / 1024 * 1024); }

constexpr int WORKERS = 384;

struct BwdParams {
  const __nv_bfloat16* w_t;  // tiled W_out   [KB][2][NH][64]     (prep_weights3_kernel)
  const __nv_bfloat16* wt_t; // tiled W_out^T [MB][KBG][128][64]
  const float* bias_l2;     // [Vp] bias*log2e, -inf beyond V
  const int32_t* targets;
  const int32_t* t_len;
  const int32_t* u_len;
  const int4* tiles;        // {b, u-split, frame block, tile index}
  const int* ntiles;
  int B, T, U1, D, V, Vp, NH, blank, r1_stages;
  const float* lse;
  const float* lp_blank;    // forward outputs: logit + bias - lse of the blank / next-label column of every cell
  const float* lp_label;
  const float* alpha;
  const float* beta;
  const float* costs;
  const float* grad_costs;
  float clamp;
  // gt [tile][2][KBG][64 rows][64 v] : the G tile as it lies in shared memory (bulk stores), read MN-major by kernel 2
  __nv_bfloat16* gt;
  float* d_enc_part;        // [S][B,T,D]
  float* d_pred;            // [B,U1,D] atomic accumulate
  float* d_bias;            // [V] atomic accumulate
  long long* prof;
  unsigned int* err_host;   // mapped host word for bounded-wait time-outs (tc_common.cuh)
  // bf16x3 only: the fp32 activations (read in place) and the spill of G_lo = bf16(G - G_hi), laid out as gt
  const float* enc;
  const float* pred;
  __nv_bfloat16* gt_lo;
  // vocabulary tiles (VT kernels only): this launch covers columns [v0, v0 + V) of a vocabulary of Vg entries whose
  // blank is blank_g; w_t / wt_t / bias_l2 / gt / d_bias are the tile's, blank is the tile's blank column or -1, and
  // lse is the full vocabulary's.  accum: add to d_enc_part (an earlier tile stored it) instead of storing.
  int v0, Vg, blank_g, accum;
};

// Shared memory: [weight ring: 4 W^T stages][G tile (P2/P3)]  -- P1 views both as one W ring --
// [P1 slab ring][P4 slab: the tile's enc / pred rows over the whole joint dim][bias][column-sum partials][barriers]
struct Bwd3Smem {
  uint32_t r_base, g_base, r1_bytes, s_base, p4_base, bar_base;
  float* bias_l2;
  float* dbp;               // [4][Vp] column-sum partials
  uint32_t* tmem_ptr;
  __device__ __forceinline__ uint32_t g_kblock(int i) const { return g_base + i * A_STAGE_BYTES; }
  __device__ __forceinline__ uint32_t r1_stage(int i) const { return r_base + i * r1_bytes; }
  __device__ __forceinline__ uint32_t r3_stage(int i) const { return r_base + i * 16384; }
  __device__ __forceinline__ uint32_t s_stage(int i) const { return s_base + i * B_SLAB_MAX; }
  __device__ __forceinline__ uint32_t p4_stage(int kb) const { return p4_base + kb * B_SLAB_MAX; }
  __device__ __forceinline__ uint32_t a_full(int i) const { return bar_base + i * 16; }             // 3
  __device__ __forceinline__ uint32_t a_empty(int i) const { return bar_base + i * 16 + 8; }
  __device__ __forceinline__ uint32_t s_full(int i) const { return bar_base + 48 + i * 16; }        // 2
  __device__ __forceinline__ uint32_t s_empty(int i) const { return bar_base + 48 + i * 16 + 8; }
  __device__ __forceinline__ uint32_t r1_full(int i) const { return bar_base + 80 + i * 16; }       // 6
  __device__ __forceinline__ uint32_t r1_empty(int i) const { return bar_base + 80 + i * 16 + 8; }
  __device__ __forceinline__ uint32_t r3_full(int i) const { return bar_base + 176 + i * 16; }      // 4
  __device__ __forceinline__ uint32_t r3_empty(int i) const { return bar_base + 176 + i * 16 + 8; }
  __device__ __forceinline__ uint32_t dz_full(int mb) const { return bar_base + 240 + mb * 8; }     // 4
  __device__ __forceinline__ uint32_t tmem_full() const { return bar_base + 272; }
  __device__ __forceinline__ uint32_t g_full() const { return bar_base + 280; }
  __device__ __forceinline__ uint32_t tmem_empty() const { return bar_base + 288; }
  __device__ __forceinline__ uint32_t gs_done() const { return bar_base + 296; }   // G spilled and column-summed
  __device__ __forceinline__ uint32_t p4_full() const { return bar_base + 304; }
  // bf16x3 only
  __device__ __forceinline__ uint32_t p3a_done() const { return bar_base + 312; }   // the G_hi MMAs have completed
  __device__ __forceinline__ uint32_t gs_hi_done() const { return bar_base + 320; } // G_hi column-summed
  __device__ __forceinline__ uint32_t glo_full() const { return bar_base + 328; }   // G_lo reloaded into the G tile
};
constexpr uint32_t B_BAR_BYTES = 320;
constexpr uint32_t B_BAR_BYTES_X3 = 352;

__host__ __device__ inline uint32_t bwd3_g_bytes(int Vp) { return (uint32_t)((Vp + 63) / 64) * A_STAGE_BYTES; }
// W_out stages that fit the ring + G region (the G tile is dead during P1)
__host__ __device__ inline int bwd3_r1_stages(int NH, int Vp) {
  const int n = (int)((B_RING_BYTES + bwd3_g_bytes(Vp)) / ((uint32_t)NH * 128u));
  return n > B_R1_MAX ? B_R1_MAX : n;
}

// split = true (bf16x3): no slab regions (the workers read the fp32 rows from global memory), three more barriers
__host__ __device__ inline size_t bwd3_smem_bytes(int NH, int Vp, int D, bool split = false) {
  size_t s = 1024;
  s += B_RING_BYTES + bwd3_g_bytes(Vp);
  if (!split) {
    s += (size_t)B_S_STAGES * B_SLAB_MAX;
    s += (size_t)(D / BK) * B_SLAB_MAX;
  }
  s += (size_t)Vp * 4 + (size_t)4 * Vp * 4;
  s += 16 + (split ? B_BAR_BYTES_X3 : B_BAR_BYTES) + 16;          // alignment + barriers + tmem pointer
  return s;
}

template <bool SPLIT = false>
__device__ __forceinline__ void carve_bwd3(Bwd3Smem& L, uint8_t* raw, int NH, int Vp, int D) {
  const uint32_t base = smem_u32(raw);
  uint32_t a = (base + 1023u) & ~1023u;
  L.r_base = a; L.r1_bytes = (uint32_t)NH * 128u; a += B_RING_BYTES;
  L.g_base = a; a += bwd3_g_bytes(Vp);
  if (!SPLIT) {
    L.s_base = a; a += B_S_STAGES * B_SLAB_MAX;
    L.p4_base = a; a += (uint32_t)(D / BK) * B_SLAB_MAX;
  }
  L.bias_l2 = reinterpret_cast<float*>(raw + (a - base)); a += Vp * 4;
  L.dbp = reinterpret_cast<float*>(raw + (a - base)); a += 4 * Vp * 4;
  a = (a + 15u) & ~15u;
  L.bar_base = a; a += SPLIT ? B_BAR_BYTES_X3 : B_BAR_BYTES;
  L.tmem_ptr = reinterpret_cast<uint32_t*>(raw + (a - base));
}

// rows C0 .. C0+15 (= TMEM columns) of d block values w[]: dH = dZ * (1 - z^2), z = tanh(e[tloc] + p[ul]) recomputed
// as packed bf16 pairs exactly as the P1 producers and the dW GEMM form it.  Every (tloc, ul) is a compile-time constant.
// Other activations (ACT): dH = dZ act'(h) with h the packed bf16 sum the producers form, act' in fp32.
template <int P, int TT, int C0, int ACT = ACT_TANH>
__device__ __forceinline__ void p4_chunk(const float (&w)[16], const uint32_t (&e)[TT], const uint32_t (&pr)[P],
                                         float (&es)[TT], float (&pa)[P]) {
  if constexpr (ACT != ACT_TANH) {
#pragma unroll
    for (int j = 0; j < 16; j += 2) {
      const int c = C0 + j;
      if (c < TT * P) {
        const int tl0 = c / P, u0 = c % P;
        const int c1 = c + 1;
        const int tl1 = (c1 / P < TT) ? c1 / P : TT - 1, u1 = c1 % P;
        const uint32_t hh = add_bf16x2(__byte_perm(e[tl0], e[tl1], 0x5410), __byte_perm(pr[u0], pr[u1], 0x5410));
        const float h0 = w[j] * act_grad_f32<ACT>(__uint_as_float(hh << 16));
        es[tl0] += h0;
        pa[u0] += h0;
        if (c1 < TT * P) {
          const float h1 = w[j + 1] * act_grad_f32<ACT>(__uint_as_float(hh & 0xffff0000u));
          es[tl1] += h1;
          pa[u1] += h1;
        }
      }
    }
    return;
  }
#pragma unroll
  for (int j = 0; j < 16; j += 2) {
    const int c = C0 + j;
    if (c < TT * P) {
      const int tl0 = c / P, u0 = c % P;
      const int c1 = c + 1;
      const int tl1 = (c1 / P < TT) ? c1 / P : TT - 1, u1 = c1 % P;
      const uint32_t ep = __byte_perm(e[tl0], e[tl1], 0x5410);
      const uint32_t pp = __byte_perm(pr[u0], pr[u1], 0x5410);
      const uint32_t zz = tanh_add_bf16x2_packed(ep, pp);
      const float z0 = __uint_as_float(zz << 16), z1 = __uint_as_float(zz & 0xffff0000u);
      const float h0 = w[j] * fmaf(-z0, z0, 1.f);
      es[tl0] += h0;
      pa[u0] += h0;
      if (c1 < TT * P) {
        const float h1 = w[j + 1] * fmaf(-z1, z1, 1.f);
        es[tl1] += h1;
        pa[u1] += h1;
      }
    }
  }
}

// bf16x3 form of p4_chunk: z = tanh(e + p) in fp32 from the fp32 rows (other activations: act'(e + p) in fp32)
template <int P, int TT, int C0, int ACT = ACT_TANH>
__device__ __forceinline__ void p4_chunk(const float (&w)[16], const float (&e)[TT], const float (&pr)[P],
                                             float (&es)[TT], float (&pa)[P]) {
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const int c = C0 + j;
    if (c < TT * P) {
      const int tl = c / P, u = c % P;
      float h;
      if constexpr (ACT == ACT_TANH) {
        const float z = tanhf(e[tl] + pr[u]);
        h = w[j] * fmaf(-z, z, 1.f);
      } else {
        h = w[j] * act_grad_f32<ACT>(e[tl] + pr[u]);
      }
      es[tl] += h;
      pa[u] += h;
    }
  }
}

// SPLIT = false: the bf16 kernel.  SPLIT = true (precision bf16x3), per tile:
//   P1  logits = z_hi W_hi + z_lo W_hi + z_hi W_lo (as the bf16x3 forward; fp32 rows read from global memory)
//   P2  G in fp32 -> G_hi = bf16(G) into the shared G tile, G_lo = bf16(G - G_hi) straight to its global spill (gt_lo)
//   P3  pass 1: dZ^T = W_hi^T G_hi^T + W_lo^T G_hi^T (ring: [MB][KBG][hi, lo] blocks of wt_t); then warp 0 reloads G_lo
//       from the spill (L2) into the G tile and pass 2 adds W_hi^T G_lo^T, committing the d blocks to P4 one by one
//   P4  dH = dZ (1 - z^2) with z = tanh(e + p) in fp32 from the fp32 rows (global memory)
//   d_bias = column sums of G_hi plus column sums of G_lo (after the reload)
// Shared memory: the bf16 layout without the two slab regions (P1 ring / P4 slab).
// ACT: the joint activation of the P1 producers and the P4 derivative (ACT_TANH / ACT_RELU / ACT_GELU).
// VT: one vocabulary tile of a larger vocabulary (BwdParams v0 ..): labels are mapped to the tile's columns, and only
// the columns it holds are patched.
template <int P, int TT, bool SPLIT, int ACT = ACT_TANH, bool VT = false>
__device__ __forceinline__ void joint_bwd3_body(const CUtensorMap& tmap_e, const CUtensorMap& tmap_p, const BwdParams& p) {
  extern __shared__ uint8_t smem_raw[];
  Bwd3Smem L;
  carve_bwd3<SPLIT>(L, smem_raw, p.NH, p.Vp, p.D);
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int KB = p.D / BK;                 // k-blocks of the logits GEMM
  const int KBG = (p.Vp + 63) / 64;        // k-blocks (over v) of the dZ GEMM
  const int MB = p.D / 128;                // 128-lane blocks of dZ^T
  const int R1 = p.r1_stages;
  const int ntiles = *p.ntiles;
  const int tile_begin = (int)(((long)ntiles * blockIdx.x) / gridDim.x);
  const int tile_end = (int)(((long)ntiles * (blockIdx.x + 1)) / gridDim.x);

  if (warp == 0 && lane == 0) {
    g_tc_error_host = p.err_host;
    if (!SPLIT) {                    // the split form gets placeholder tensor maps
      tma_prefetch_desc(&tmap_e);
      tma_prefetch_desc(&tmap_p);
    }
    for (int i = 0; i < B_A_STAGES; ++i) { mbar_init(L.a_full(i), 8); mbar_init(L.a_empty(i), 1); }
    for (int i = 0; i < B_S_STAGES; ++i) { mbar_init(L.s_full(i), 1); mbar_init(L.s_empty(i), 8); }
    for (int i = 0; i < B_R1_MAX; ++i) { mbar_init(L.r1_full(i), 1); mbar_init(L.r1_empty(i), 1); }
    for (int i = 0; i < B_R3_STAGES; ++i) { mbar_init(L.r3_full(i), 1); mbar_init(L.r3_empty(i), 1); }
    for (int i = 0; i < 4; ++i) mbar_init(L.dz_full(i), 1);
    mbar_init(L.tmem_full(), 1);
    mbar_init(L.g_full(), WORKERS / 32);
    mbar_init(L.tmem_empty(), 8);
    mbar_init(L.gs_done(), 1);
    mbar_init(L.p4_full(), 1);
    if (SPLIT) { mbar_init(L.p3a_done(), 1); mbar_init(L.gs_hi_done(), 1); mbar_init(L.glo_full(), 1); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_u32(L.tmem_ptr), TMEM_COLS);
  for (int i = tid; i < p.Vp; i += NTHREADS) L.bias_l2[i] = p.bias_l2[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *L.tmem_ptr;

  if (warp == 0) {
    // ------------------------------------------------------------------ bulk copies: W_out (P1), W_out^T (P3)
    Pipe r1, r3;
    int prof_n = 0;
    uint32_t ph = 0;
    const uint32_t r1_bytes = (uint32_t)p.NH * 128u;
    for (int tile = tile_begin; tile < tile_end; ++tile) {
      if (lane == 0) TC_PROF(0, 1);
      // ring + G region are dead here: the previous tile's last dZ block and its G spill / column sums were observed below
      for (int i = 0; i < (SPLIT ? 4 : 2) * KB; ++i) {
        mbar_wait(L.r1_empty(r1.stage), r1.phase ^ 1u, 11);
        if (elect_one()) {
          mbar_arrive_expect_tx(L.r1_full(r1.stage), r1_bytes);
          bulk_load(L.r1_stage(r1.stage), p.w_t + (size_t)i * p.NH * 64, r1_bytes, L.r1_full(r1.stage));
        }
        __syncwarp();
        r1.advance(R1);
      }
      if (lane == 0) TC_PROF(0, 2);
      mbar_wait(L.tmem_full(), ph, 12);           // every P1 MMA has completed: the W view of the ring is dead
      if (lane == 0) TC_PROF(0, 3);
      // W_out^T stages, with the spill of the finished G tile interleaved (one 8 KB bulk store behind every second
      // stage load): the copy engine serves one queue, and 2*KBG stores issued in one burst at the start of P3 held the
      // stage loads behind them for ~4 k cycles per tile.  k-block i (64 label columns) -> two 8 KB boxes
      // [64 rows][64 v] (rows 0-63 / 64-127), read back MN-major by the dW GEMM.  A stage beyond the preloaded ones
      // is only released by a P3 MMA, i.e. after g_full: the G tile is complete (and fenced) when its store is issued.
      __nv_bfloat16* gdst = p.gt + ((size_t)p.tiles[tile].w * 2) * (size_t)KBG * 4096;
      int ns = 0;                                   // stores issued: store j = (k-block j >> 1, row half j & 1)
      auto spill = [&](int j) {
        if (CTCVR_EXP & 1) return;
        bulk_store(gdst + ((size_t)(j & 1) * KBG + (j >> 1)) * 4096, L.g_kblock(j >> 1) + (uint32_t)(j & 1) * 8192u, 8192u);
      };
      for (int i = 0; i < (SPLIT ? 2 : 1) * MB * KBG; ++i) {
        mbar_wait(L.r3_empty(r3.stage), r3.phase ^ 1u, 13);
        if (elect_one()) {
          mbar_arrive_expect_tx(L.r3_full(r3.stage), 16384u);
          bulk_load(L.r3_stage(r3.stage), p.wt_t + (size_t)i * 8192, 16384u, L.r3_full(r3.stage));
          if (i >= B_R3_STAGES && ((i - B_R3_STAGES) & 1) == 0 && ns < 2 * KBG) spill(ns);
        }
        if (i >= B_R3_STAGES && ((i - B_R3_STAGES) & 1) == 0 && ns < 2 * KBG) ++ns;
        __syncwarp();
        r3.advance(B_R3_STAGES);
      }
      mbar_wait(L.g_full(), ph, 18);
      if (elect_one()) {
        for (int j = ns; j < 2 * KBG; ++j) spill(j);
        bulk_commit();
      }
      __syncwarp();
      if constexpr (SPLIT) {
        // G_lo into the G tile once the pass-1 MMAs, the G_hi column sums and the G_hi spill are done with it.  The
        // P2 threads wrote G_lo with generic stores, fenced for the async proxy before their g_full arrival (seen above)
        const __nv_bfloat16* gsrc = p.gt_lo + ((size_t)p.tiles[tile].w * 2) * (size_t)KBG * 4096;
        mbar_wait(L.p3a_done(), ph, 60);
        mbar_wait(L.gs_hi_done(), ph, 61);
        if (elect_one()) {
          bulk_wait_read<0>();
          mbar_arrive_expect_tx(L.glo_full(), (uint32_t)KBG * 16384u);
          for (int j = 0; j < 2 * KBG; ++j)
            bulk_load(L.g_kblock(j >> 1) + (uint32_t)(j & 1) * 8192u, gsrc + ((size_t)(j & 1) * KBG + (j >> 1)) * 4096, 8192u,
                      L.glo_full());
        }
        __syncwarp();
        for (int i = 0; i < MB * KBG; ++i) {          // pass 2: the W_hi^T blocks again
          mbar_wait(L.r3_empty(r3.stage), r3.phase ^ 1u, 62);
          if (elect_one()) {
            mbar_arrive_expect_tx(L.r3_full(r3.stage), 16384u);
            bulk_load(L.r3_stage(r3.stage), p.wt_t + (size_t)(2 * i) * 8192, 16384u, L.r3_full(r3.stage));
          }
          __syncwarp();
          r3.advance(B_R3_STAGES);
        }
      }
      if (lane == 0) TC_PROF(0, 4);
      mbar_wait(L.dz_full(MB - 1), ph, 14);       // every P3 MMA has completed: G tile and the W^T view are dead
      mbar_wait(L.gs_done(), ph, 16);             // ... the d_bias column sums have read G
      if (elect_one()) bulk_wait_read<0>();       // ... and so have the spill stores
      __syncwarp();
      if (lane == 0) TC_PROF(0, 5);
      ph ^= 1u;
    }
  } else if (warp == 3 && !SPLIT) {
    // ------------------------------------------------------------------ TMA: enc / pred slabs (P1 ring + the P4 slab)
    Pipe sp;
    uint32_t ph = 0;
    for (int tile = tile_begin; tile < tile_end; ++tile) {
      const int4 ti = p.tiles[tile];
      const int b = ti.x;
      const int W = max(min(p.u_len[b], p.U1 - 1), 0) + 1;
      const int S = (W + P - 1) / P, us = (W + S - 1) / S;
      const int prow = b * p.U1 + ti.y * us;
      const int erow = b * p.T + ti.z * TT;
      for (int kb = 0; kb < KB; ++kb) {
        mbar_wait(L.s_empty(sp.stage), sp.phase ^ 1u, 15);
        if (elect_one()) {
          const uint32_t st = L.s_stage(sp.stage);
          mbar_arrive_expect_tx(L.s_full(sp.stage), (uint32_t)(P + TT) * 128u);
          tma_load_2d(st, &tmap_p, L.s_full(sp.stage), kb * BK, prow);
          tma_load_2d(st + bwd_pred_region<P>(), &tmap_e, L.s_full(sp.stage), kb * BK, erow);
        }
        __syncwarp();
        sp.advance(B_S_STAGES);
      }
      // the same rows over the whole joint dim for P4 (its readers of the previous tile are done: tmem_empty)
      mbar_wait(L.tmem_empty(), ph ^ 1u, 17);
      if (elect_one()) {
        mbar_arrive_expect_tx(L.p4_full(), (uint32_t)KB * (uint32_t)(P + TT) * 128u);
        for (int kb = 0; kb < KB; ++kb) {
          const uint32_t st = L.p4_stage(kb);
          tma_load_2d(st, &tmap_p, L.p4_full(), kb * BK, prow);
          tma_load_2d(st + bwd_pred_region<P>(), &tmap_e, L.p4_full(), kb * BK, erow);
        }
      }
      __syncwarp();
      ph ^= 1u;
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (warp-wide loop, one elected lane issues)
    Pipe ap, r1, r3;
    int prof_n = 0;
    uint32_t ph = 0;
    const uint32_t idesc1 = make_idesc_bf16(BM, p.NH);
    const uint32_t idesc2 = make_idesc_bf16(128, BM);
    const uint64_t r1_desc0 = make_desc_sw128(L.r1_stage(0));     // + stage * NH * 8
    const uint64_t r3_desc0 = make_desc_sw128(L.r3_stage(0));     // + stage * 1024
    const uint64_t g_desc0 = make_desc_sw128(L.g_kblock(0));      // + kb * 1024
    const uint32_t r1_step = (uint32_t)p.NH * 8u;
    const int last_nks = (p.Vp - (KBG - 1) * 64) / 16;
    for (int tile = tile_begin; tile < tile_end; ++tile) {
      if (lane == 0) TC_PROF(1, 1);
      mbar_wait(L.tmem_empty(), ph ^ 1u, 20);
      if (lane == 0) TC_PROF(1, 2);
      tc_fence_after();
      if constexpr (SPLIT) {
        for (int kb = 0; kb < KB; ++kb) {
          Pipe al = ap;                                // z_lo stage follows the z_hi stage
          al.advance(B_A_STAGES);
          mbar_wait(L.a_full(ap.stage), ap.phase, 21);
          mbar_wait(L.a_full(al.stage), al.phase, 21);
          for (int j = 0; j < 4; ++j) {                // W_hi half 0, 1, W_lo half 0, 1
            mbar_wait(L.r1_full(r1.stage), r1.phase, 22);
            tc_fence_after();
            if (elect_one()) {
              const uint32_t a = tmem_base + B_ACC_COLS + ap.stage * 32;
              const uint32_t a2 = tmem_base + B_ACC_COLS + al.stage * 32;
              const uint64_t bd = r1_desc0 + (uint64_t)(r1.stage * r1_step);
              const uint32_t d = tmem_base + (j & 1) * p.NH;
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4) umma_bf16_ts(d, a + 8 * k4, bd + 2 * k4, idesc1, (kb || j >= 2 || k4) ? 1u : 0u);
              if (j < 2) {
#pragma unroll
                for (int k4 = 0; k4 < 4; ++k4) umma_bf16_ts(d, a2 + 8 * k4, bd + 2 * k4, idesc1, 1u);
              }
              umma_commit(L.r1_empty(r1.stage));
              if (j == 3) { umma_commit(L.a_empty(ap.stage)); umma_commit(L.a_empty(al.stage)); }
            }
            __syncwarp();
            r1.advance(R1);
          }
          ap.advance(B_A_STAGES);
          ap.advance(B_A_STAGES);
        }
      } else
      for (int kb = 0; kb < KB; ++kb) {
        mbar_wait(L.a_full(ap.stage), ap.phase, 21);
        if (lane == 0) TC_PROF(1, 50 + kb);
        for (int h = 0; h < 2; ++h) {
          mbar_wait(L.r1_full(r1.stage), r1.phase, 22);
          if (lane == 0) TC_PROF(1, 100 + kb * 2 + h);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t a = tmem_base + B_ACC_COLS + ap.stage * 32;
            const uint64_t bd = r1_desc0 + (uint64_t)(r1.stage * r1_step);
            const uint32_t d = tmem_base + h * p.NH;
            umma_bf16_ts(d, a, bd, idesc1, kb ? 1u : 0u);
            umma_bf16_ts(d, a + 8, bd + 2, idesc1, 1u);
            umma_bf16_ts(d, a + 16, bd + 4, idesc1, 1u);
            umma_bf16_ts(d, a + 24, bd + 6, idesc1, 1u);
            umma_commit(L.r1_empty(r1.stage));
            if (h == 1) umma_commit(L.a_empty(ap.stage));
          }
          __syncwarp();
          r1.advance(R1);
        }
        ap.advance(B_A_STAGES);
      }
      if (elect_one()) umma_commit(L.tmem_full());
      __syncwarp();
      if (lane == 0) TC_PROF(1, 3);
      // ---- P3: dZ^T[mb] (128 d x 128 rows) = W^T[mb] (128 x Vp) . G^T (Vp x 128); block mb is handed to P4 on its own
      mbar_wait(L.g_full(), ph, 23);
      if (lane == 0) TC_PROF(1, 4);
      tc_fence_after();
      if constexpr (SPLIT) {
        // pass 1: W_hi^T G_hi^T + W_lo^T G_hi^T into every d block
        for (int mb = 0; mb < MB; ++mb)
          for (int kb = 0; kb < KBG; ++kb)
            for (int hl = 0; hl < 2; ++hl) {
              mbar_wait(L.r3_full(r3.stage), r3.phase, 24);
              tc_fence_after();
              if (elect_one()) {
                const uint64_t ad = r3_desc0 + (uint64_t)(r3.stage * 1024);
                const uint64_t bd = g_desc0 + (uint64_t)(kb * 1024);
                const uint32_t d = tmem_base + mb * 128;
                const int nks = kb == KBG - 1 ? last_nks : 4;
                for (int k4 = 0; k4 < nks; ++k4) umma_bf16(d, ad + 2 * k4, bd + 2 * k4, idesc2, (kb || hl || k4) ? 1u : 0u);
                umma_commit(L.r3_empty(r3.stage));
              }
              __syncwarp();
              r3.advance(B_R3_STAGES);
            }
        if (elect_one()) umma_commit(L.p3a_done());
        __syncwarp();
        // pass 2: + W_hi^T G_lo^T once G_lo is in the tile; d block mb goes to P4 as soon as it is complete
        mbar_wait(L.glo_full(), ph, 63);
        tc_fence_after();
      }
      for (int mb = 0; mb < MB; ++mb) {
        for (int kb = 0; kb < KBG; ++kb) {
          mbar_wait(L.r3_full(r3.stage), r3.phase, 24);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t ad = r3_desc0 + (uint64_t)(r3.stage * 1024);
            const uint64_t bd = g_desc0 + (uint64_t)(kb * 1024);
            const uint32_t d = tmem_base + mb * 128;
            const int nks = kb == KBG - 1 ? last_nks : 4;
            if (nks > 0) umma_bf16(d, ad, bd, idesc2, (kb || SPLIT) ? 1u : 0u);
            if (nks > 1) umma_bf16(d, ad + 2, bd + 2, idesc2, 1u);
            if (nks > 2) umma_bf16(d, ad + 4, bd + 4, idesc2, 1u);
            if (nks > 3) umma_bf16(d, ad + 6, bd + 6, idesc2, 1u);
            umma_commit(L.r3_empty(r3.stage));
            if (kb == KBG - 1) umma_commit(L.dz_full(mb));
          }
          __syncwarp();
          r3.advance(B_R3_STAGES);
        }
        if (lane == 0) TC_PROF(1, 10 + mb);
      }
      if (lane == 0) TC_PROF(1, 5);
      ph ^= 1u;
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ workers (warps 4-15): P1 producers, P2, P4 / spill
    const int q = warp & 3;
    const int wg = (warp - 4) >> 2;            // 0..2
    const int r = q * 32 + lane;               // P2: tile row ; P4: lane of the d block
    const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t ph = 0;
    int prof_n = 0;
    float db[4] = {0.f, 0.f, 0.f, 0.f};        // warp group 2: d_bias of columns r, r + 128, r + 256, r + 384
    float pacc[2][P];                          // warp groups 0/1: d_pred sums of d blocks wg, wg + 2 over one (b, u-split) sweep
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < P; ++j) pacc[i][j] = 0.f;
    int cur_b = -1, cur_ubase = 0;
    auto flush_pred = [&]() {
      if (cur_b < 0 || wg >= 2) return;
      const int Ub = max(min(p.u_len[cur_b], p.U1 - 1), 0);
#pragma unroll
      for (int mbl = 0; mbl < 2; ++mbl) {
        const int mb = wg + 2 * mbl;
        if (mb < MB) {
#pragma unroll
          for (int j = 0; j < P; ++j) {
            const int u = cur_ubase + j;
            if (u <= Ub) atomicAdd(p.d_pred + ((size_t)cur_b * p.U1 + u) * p.D + mb * 128 + r, pacc[mbl][j]);
            pacc[mbl][j] = 0.f;
          }
        }
      }
    };
    // producer addressing (A operand lives in TMEM): thread = tile row r = 32q + lane (its own TMEM lane).  All 12
    // worker warps produce: a k-block is two slots (k-half kh: 32 of its 64 k -> 16 packed bf16x2 -> one tcgen05.st);
    // warp group wg takes the slots s = 2 kb + kh with s % 3 == wg.  rows >= TT*P are padding
    const int p_tloc = min(r / P, TT - 1), p_ul = r % P;
    const uint32_t e_row = bwd_pred_region<P>() + (uint32_t)p_tloc * 128u, e_sw = (uint32_t)(p_tloc & 7);
    const uint32_t p_row = (uint32_t)p_ul * 128u, p_sw = (uint32_t)(p_ul & 7);
    uint32_t kb_base = 0;                       // k-blocks produced before this tile (ring stages follow it)

    for (int tile = tile_begin; tile < tile_end; ++tile) {
      int4 ti = p.tiles[tile];
      pin(ti.x); pin(ti.y); pin(ti.z); pin(ti.w);
      BwdGeom<P, TT> g;
      g.init(p.t_len, p.u_len, p.T, p.U1, ti);
      if (g.b != cur_b || g.ubase != cur_ubase) { flush_pred(); cur_b = g.b; cur_ubase = g.ubase; }

      // ---------------- P1: A k-blocks into TMEM
      {
        // the A columns overlay the dZ^T accumulator of the previous tile: wait until its readers (P4) are done
        mbar_wait(L.tmem_empty(), ph ^ 1u, 40);
        if (tid == 128) TC_PROF(3, 1);
        if constexpr (SPLIT) {
          // slot = 32 k of row r: 16 z_hi columns in A stage 2 kbc, 16 z_lo columns in A stage 2 kbc + 1
          const float4* er = reinterpret_cast<const float4*>(p.enc + ((size_t)g.b * p.T + min(g.t0 + p_tloc, p.T - 1)) * p.D);
          const float4* pr4 = reinterpret_cast<const float4*>(p.pred + ((size_t)g.b * p.U1 + min(g.ubase + p_ul, p.U1 - 1)) * p.D);
          for (int s = wg; s < 2 * KB; s += 3) {
            const int kb = s >> 1, kh = s & 1;
            const uint32_t n_hi = 2u * (kb_base + (uint32_t)kb), n_lo = n_hi + 1u;
            const uint32_t s_hi = n_hi % B_A_STAGES, ph_hi = (n_hi / B_A_STAGES) & 1u;
            const uint32_t s_lo = n_lo % B_A_STAGES, ph_lo = (n_lo / B_A_STAGES) & 1u;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              const float4* e4 = er + kb * 16 + kh * 8 + c * 4;
              const float4* p4 = pr4 + kb * 16 + kh * 8 + c * 4;
              const float4 e0 = __ldg(e4), e1 = __ldg(e4 + 1), e2 = __ldg(e4 + 2), e3 = __ldg(e4 + 3);
              const float4 q0 = __ldg(p4), q1 = __ldg(p4 + 1), q2 = __ldg(p4 + 2), q3 = __ldg(p4 + 3);
              uint32_t hi[8], lo[8];
              tanh_split8<ACT>(e0, e1, q0, q1, hi, lo);
              tanh_split8<ACT>(e2, e3, q2, q3, hi + 4, lo + 4);
              if (c == 0) {
                mbar_wait(L.a_empty(s_hi), ph_hi ^ 1u, 42);
                mbar_wait(L.a_empty(s_lo), ph_lo ^ 1u, 42);
                tc_fence_after();
              }
              tmem_st8(tq + (uint32_t)(B_ACC_COLS + s_hi * 32 + kh * 16 + c * 8), hi);
              tmem_st8(tq + (uint32_t)(B_ACC_COLS + s_lo * 32 + kh * 16 + c * 8), lo);
            }
            tmem_st_wait();
            tc_fence_before();
            warp_arrive(L.a_full(s_hi));
            warp_arrive(L.a_full(s_lo));
          }
        } else
        for (int s = wg; s < 2 * KB; s += 3) {
          const int kb = s >> 1, kh = s & 1;
          const uint32_t kbc = kb_base + (uint32_t)kb;
          const uint32_t a_stg = kbc % B_A_STAGES, a_ph = (kbc / B_A_STAGES) & 1u;
          const uint32_t s_stg = kbc % B_S_STAGES, s_ph = (kbc / B_S_STAGES) & 1u;
          mbar_wait(L.s_full(s_stg), s_ph, 41);
          mbar_wait(L.a_empty(a_stg), a_ph ^ 1u, 42);
          tc_fence_after();
          const uint32_t sb = L.s_stage(s_stg);
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
          tmem_st16(tq + (uint32_t)(B_ACC_COLS + a_stg * 32 + kh * 16), w);
          tmem_st_wait();
          tc_fence_before();
          warp_arrive(L.a_full(a_stg));
          warp_arrive(L.s_empty(s_stg));
        }
        kb_base += (uint32_t)KB;
        if (tid == 128) TC_PROF(3, 2);
      }

      // ---------------- P2: g = d cost / d logits for row r, column chunks wg, wg+3, ...
      int t, u, ul;
      const bool valid = g.cell(r, t, u, ul);
      float k_all = kNegInf, scale = 0.f;
      float a_c = 0.f, be = 0.f, bnext = kNegInf, bl1 = kNegInf, lpb = 0.f, lpl = 0.f;
      int lab = -1;
      if (valid) {
        const size_t cell = ((size_t)g.b * p.T + t) * p.U1 + u;
        const float al = p.alpha[cell], cost = p.costs[g.b], l = p.lse[cell];
        be = p.beta[cell];
        a_c = al + cost;
        k_all = a_c + be - l;
        if (t + 1 < g.Tb) bnext = p.beta[cell + p.U1];
        else if (u == g.Ub) bnext = 0.f;
        lpb = p.lp_blank[cell];
        if (u < g.Ub) {
          bl1 = p.beta[cell + 1];
          lpl = p.lp_label[cell];
          lab = p.targets[(size_t)g.b * (p.U1 - 1) + u];
          if (VT) lab = vt_column(lab, p.Vg, p.blank_g, p.v0, p.V);
          else if ((unsigned)lab >= (unsigned)p.V) lab = p.blank;      // out-of-range ids cannot index outside the tile
        }
        scale = p.grad_costs[g.b];
      }
      // fast path: no clamp and a positive cost gradient (uniform per tile): fold log2(scale) into the exponent
      const float sc_tile = p.grad_costs[g.b];
      const bool fast = !(p.clamp > 0.f) && sc_tile > 0.f;
      const float kr = (valid && fast) ? fmaf(k_all, LOG2E, lg2_fast(scale)) : kNegInf;
      if (tid == 128) TC_PROF(2, 1);
      mbar_wait(L.tmem_full(), ph, 30);
      if (tid == 128) TC_PROF(2, 2);
      tc_fence_after();
      // 16-column pieces wg, wg+3, ..; the next piece's TMEM load is in flight during the math
      // pieces dealt round-robin to the three warp groups (26 pieces at Vp = 416: 9 / 9 / 8; by 32-column chunks it was
      // 10 / 8 / 8 and the phase ended with two groups waiting for the first)
      const int npieces = (p.Vp / 16 - wg + 2) / 3;
      auto piece_col = [&](int i) { return (wg + 3 * i) * 16; };
      float v[16];
      if (npieces > 0) tmem_ld16(tq + piece_col(0), v);
      for (int pi = 0; pi < npieces; ++pi) {
        const int c0 = piece_col(pi);
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
        if (pi + 1 < npieces) tmem_ld16(tq + piece_col(pi + 1), v);
        uint32_t pk[8];
        uint32_t pl[8];                               // bf16x3: G_lo pairs
        if constexpr (SPLIT) {
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            float gg[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              float gv;
              if (fast) {
                gv = ex2_fast(y[j + e] + kr);
              } else {
                gv = ex2_fast(y[j + e] + k_all * LOG2E);
                if (p.clamp > 0.f) gv = fminf(gv, p.clamp);
                gv = valid ? gv * scale : 0.f;
              }
              gg[e] = gv;
            }
            const __nv_bfloat162 h = __floats2bfloat162_rn(gg[0], gg[1]);
            pk[j >> 1] = *reinterpret_cast<const uint32_t*>(&h);
            pl[j >> 1] = pack_bf16(gg[0] - __low2float(h), gg[1] - __high2float(h));
          }
        } else if (fast) {
#pragma unroll
          for (int j = 0; j < 16; j += 2) pk[j >> 1] = pack_bf16(ex2_fast(y[j] + kr), ex2_fast(y[j + 1] + kr));
        } else {
          const float ka2 = k_all * LOG2E;
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            float gg[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              float gv = ex2_fast(y[j + e] + ka2);
              if (p.clamp > 0.f) gv = fminf(gv, p.clamp);
              gg[e] = valid ? gv * scale : 0.f;
            }
            pk[j >> 1] = pack_bf16(gg[0], gg[1]);
          }
        }
        // G tile: k-block c0/64, row r, 16-byte chunks (c0%64)/8, +1, 128B swizzle
        const uint32_t gb = L.g_kblock(c0 >> 6) + r * 128;
        const int ch0 = (c0 & 63) >> 3;
#pragma unroll
        for (int i = 0; i < 2; ++i)
          sts128(gb + (((ch0 + i) ^ (r & 7)) << 4), pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
        if constexpr (SPLIT) {                        // G_lo: the same bytes the G tile's bulk store would write
          uint4* gl = reinterpret_cast<uint4*>(p.gt_lo + (((size_t)ti.w * 2 + (r >> 6)) * KBG + (c0 >> 6)) * 4096 + (r & 63) * 64);
#pragma unroll
          for (int i = 0; i < 2; ++i) gl[(ch0 + i) ^ (r & 7)] = make_uint4(pl[4 * i], pl[4 * i + 1], pl[4 * i + 2], pl[4 * i + 3]);
        }
      }
      // exact (fp32, single rounding) blank and label entries of row r, from the forward's log-probs: the warp group that
      // wrote the 16-column piece of the column patches it (program order within the thread - no barrier needed)
      if (valid) {
        auto entry = [&](float lp, float b1, float b2) {
          float gv = __expf(lp + a_c + be) - __expf(lp + a_c + b1);
          if (b2 != kNegInf) gv -= __expf(lp + a_c + b2);
          if (p.clamp > 0.f) gv = fminf(fmaxf(gv, -p.clamp), p.clamp);
          return gv * scale;
        };
        auto put = [&](int col, float val) {
          const __nv_bfloat16 hb = __float2bfloat16(val);
          const unsigned short h = __bfloat16_as_ushort(hb);
          const uint32_t a = L.g_kblock(col >> 6) + r * 128 + ((((col & 63) >> 3) ^ (r & 7)) << 4) + (col & 7) * 2;
          asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"(h) : "memory");
          if constexpr (SPLIT)                        // after this thread's own 16-byte store of the same chunk
            p.gt_lo[(((size_t)ti.w * 2 + (r >> 6)) * KBG + (col >> 6)) * 4096 + (r & 63) * 64 +
                    ((((col & 63) >> 3) ^ (r & 7)) << 3) + (col & 7)] = __float2bfloat16(val - __bfloat162float(hb));
        };
        if ((!VT || p.blank >= 0) && ((p.blank >> 4) % 3) == wg) put(p.blank, entry(lpb, bnext, (lab == p.blank) ? bl1 : kNegInf));
        if (lab >= 0 && lab != p.blank && ((lab >> 4) % 3) == wg) put(lab, entry(lpl, bl1, kNegInf));
      }
      fence_proxy_async();
      if (SPLIT) asm volatile("fence.proxy.async.global;" ::: "memory");   // G_lo is read back by a bulk copy
      tc_fence_before();
      warp_arrive(L.g_full());
      if (tid == 128) TC_PROF(2, 3);

      if (wg == 2) {
        // ---------------- P3 side work (warps 12-15): spill the G tile, d_bias = its column sums
        mbar_wait(L.g_full(), ph, 31);
        const int nchunk = p.Vp >> 3;
        auto colsum = [&]() {
        for (int it = r; it < ((CTCVR_EXP & 2) ? 0 : 4 * nchunk); it += 128) {
          const int rg = it / nchunk, c = it - rg * nchunk;
          const uint32_t gb = L.g_kblock(c >> 3) + (uint32_t)(rg * 32) * 128u;
          float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
          for (int rr = 0; rr < 32; ++rr) {
            const uint4 x = lds128(gb + rr * 128 + ((((c & 7) ^ (rr & 7))) << 4));
            acc[0] += __uint_as_float(x.x << 16); acc[1] += __uint_as_float(x.x & 0xffff0000u);
            acc[2] += __uint_as_float(x.y << 16); acc[3] += __uint_as_float(x.y & 0xffff0000u);
            acc[4] += __uint_as_float(x.z << 16); acc[5] += __uint_as_float(x.z & 0xffff0000u);
            acc[6] += __uint_as_float(x.w << 16); acc[7] += __uint_as_float(x.w & 0xffff0000u);
          }
          float* o = L.dbp + rg * p.Vp + c * 8;
          *reinterpret_cast<float4*>(o) = make_float4(acc[0], acc[1], acc[2], acc[3]);
          *reinterpret_cast<float4*>(o + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
        }
        named_barrier_sync(2, 128);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int col = r + 128 * i;
          if (col < p.Vp) db[i] += (L.dbp[col] + L.dbp[p.Vp + col]) + (L.dbp[2 * p.Vp + col] + L.dbp[3 * p.Vp + col]);
        }
        named_barrier_sync(2, 128);                   // partials consumed (the next tile overwrites them)
        };
        colsum();
        if constexpr (SPLIT) {                        // + the column sums of G_lo once it is in the tile
          if (r == 0) mbar_arrive(L.gs_hi_done());
          mbar_wait(L.glo_full(), ph, 64);
          colsum();
        }
        if (r == 0) mbar_arrive(L.gs_done());
      } else {
        // ---------------- P4 (warps 4-11), overlapped with P3: dH = dZ * (1 - z^2); reductions.  Warp group wg owns
        // d blocks wg, wg+2.  TMEM column c of a d block = tile row c = (frame slot c / P, label slot c % P): everything
        // is static after unrolling, so any (P, TT) works with aligned 32-column loads.
        if (!SPLIT) mbar_wait(L.p4_full(), ph, 34);
#pragma unroll
        for (int mbl = 0; mbl < 2; ++mbl) {
          const int mb = wg + 2 * mbl;
          if (mb < MB) {
            const int d = mb * 128 + r;
            // this thread's joint dim of the tile's enc / pred rows: slab stage d/64, 16-byte chunk ((d&63)>>3) ^ (row&7)
            // (bf16x3: the fp32 values, coalesced loads from global memory over the lanes = consecutive d)
            std::conditional_t<SPLIT, float, uint32_t> e[TT], pr[P];
            if constexpr (SPLIT) {
#pragma unroll
              for (int i = 0; i < P; ++i) pr[i] = __ldg(p.pred + ((size_t)g.b * p.U1 + min(g.ubase + i, p.U1 - 1)) * p.D + d);
#pragma unroll
              for (int i = 0; i < TT; ++i) e[i] = __ldg(p.enc + ((size_t)g.b * p.T + min(g.t0 + i, p.T - 1)) * p.D + d);
            } else {
              const uint32_t st = L.p4_stage(d >> 6) + (uint32_t)(d & 7) * 2u;
              const uint32_t chn = (uint32_t)((d & 63) >> 3);
#pragma unroll
              for (int i = 0; i < P; ++i) {
                unsigned short x;
                asm volatile("ld.shared.u16 %0, [%1];" : "=h"(x) : "r"(st + i * 128 + ((chn ^ (uint32_t)(i & 7)) << 4)));
                pr[i] = x;
              }
#pragma unroll
              for (int i = 0; i < TT; ++i) {
                unsigned short x;
                asm volatile("ld.shared.u16 %0, [%1];" : "=h"(x) : "r"(st + bwd_pred_region<P>() + i * 128 + ((chn ^ (uint32_t)(i & 7)) << 4)));
                e[i] = x;
              }
            }
            mbar_wait(L.dz_full(mb), ph, 32);
            if (tid == 128) TC_PROF(2, 40 + mb);
            tc_fence_after();
            float es[TT];
#pragma unroll
            for (int i = 0; i < TT; ++i) es[i] = 0.f;
            float v0[16], v1[16];
            const uint32_t tb = tq + mb * 128;
            tmem_ld16(tb, v0);
            tmem_ld_wait();
            tmem_ld16(tb + 16, v1);
            p4_chunk<P, TT, 0, ACT>(v0, e, pr, es, pacc[mbl]);
            tmem_ld_wait();
            tmem_ld16(tb + 32, v0);
            p4_chunk<P, TT, 16, ACT>(v1, e, pr, es, pacc[mbl]);
            tmem_ld_wait();
            tmem_ld16(tb + 48, v1);
            p4_chunk<P, TT, 32, ACT>(v0, e, pr, es, pacc[mbl]);
            tmem_ld_wait();
            tmem_ld16(tb + 64, v0);
            p4_chunk<P, TT, 48, ACT>(v1, e, pr, es, pacc[mbl]);
            tmem_ld_wait();
            tmem_ld16(tb + 80, v1);
            p4_chunk<P, TT, 64, ACT>(v0, e, pr, es, pacc[mbl]);
            tmem_ld_wait();
            tmem_ld16(tb + 96, v0);
            p4_chunk<P, TT, 80, ACT>(v1, e, pr, es, pacc[mbl]);
            tmem_ld_wait();
            tmem_ld16(tb + 112, v1);
            p4_chunk<P, TT, 96, ACT>(v0, e, pr, es, pacc[mbl]);
            tmem_ld_wait();
            p4_chunk<P, TT, 112, ACT>(v1, e, pr, es, pacc[mbl]);
#pragma unroll
            for (int i = 0; i < TT; ++i) {
              const int tt = g.t0 + i;
              if (tt < g.Tb) {
                float& o = p.d_enc_part[(((size_t)ti.y * p.B + g.b) * p.T + tt) * p.D + d];
                if (VT && p.accum) o += es[i]; else o = es[i];
              }
            }
          }
        }
        tc_fence_before();
        warp_arrive(L.tmem_empty());
        if (tid == 128) TC_PROF(2, 5);
      }
      ph ^= 1u;
    }
    flush_pred();
    if (wg == 2 && tile_end > tile_begin) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (r + 128 * i < p.V) atomicAdd(p.d_bias + r + 128 * i, db[i]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

template <int P, int TT>
__global__ void __launch_bounds__(NTHREADS, 1)
joint_bwd3_kernel(const __grid_constant__ CUtensorMap tmap_e, const __grid_constant__ CUtensorMap tmap_p,
                  const BwdParams p) {
  joint_bwd3_body<P, TT, false>(tmap_e, tmap_p, p);
}
// precision bf16x3 (the tensor maps are unused)
template <int P, int TT>
__global__ void __launch_bounds__(NTHREADS, 1)
joint_bwd3_x3_kernel(const __grid_constant__ CUtensorMap tmap_e, const __grid_constant__ CUtensorMap tmap_p,
                     const BwdParams p) {
  joint_bwd3_body<P, TT, true>(tmap_e, tmap_p, p);
}
// relu / gelu joints, named apart for profiler traces
#define CTCVR_BWD3_ACT(name, split, act)                                                                           \
  template <int P, int TT>                                                                                          \
  __global__ void __launch_bounds__(NTHREADS, 1)                                                                    \
  name(const __grid_constant__ CUtensorMap tmap_e, const __grid_constant__ CUtensorMap tmap_p, const BwdParams p) { \
    joint_bwd3_body<P, TT, split, act>(tmap_e, tmap_p, p);                                                          \
  }
CTCVR_BWD3_ACT(joint_bwd3_relu_kernel, false, ACT_RELU)
CTCVR_BWD3_ACT(joint_bwd3_gelu_kernel, false, ACT_GELU)
CTCVR_BWD3_ACT(joint_bwd3_x3_relu_kernel, true, ACT_RELU)
CTCVR_BWD3_ACT(joint_bwd3_x3_gelu_kernel, true, ACT_GELU)
#undef CTCVR_BWD3_ACT
// vocabulary tiles (ctcvr_joint_rnnt_bwd_vt): one launch per tile of the vocabulary
#define CTCVR_BWD3_VT(name, split, act)                                                                            \
  template <int P, int TT>                                                                                          \
  __global__ void __launch_bounds__(NTHREADS, 1)                                                                    \
  name(const __grid_constant__ CUtensorMap tmap_e, const __grid_constant__ CUtensorMap tmap_p, const BwdParams p) { \
    joint_bwd3_body<P, TT, split, act, true>(tmap_e, tmap_p, p);                                                    \
  }
CTCVR_BWD3_VT(joint_bwd3_vt_kernel, false, ACT_TANH)
CTCVR_BWD3_VT(joint_bwd3_vt_relu_kernel, false, ACT_RELU)
CTCVR_BWD3_VT(joint_bwd3_vt_gelu_kernel, false, ACT_GELU)
CTCVR_BWD3_VT(joint_bwd3_x3_vt_kernel, true, ACT_TANH)
CTCVR_BWD3_VT(joint_bwd3_x3_vt_relu_kernel, true, ACT_RELU)
CTCVR_BWD3_VT(joint_bwd3_x3_vt_gelu_kernel, true, ACT_GELU)
#undef CTCVR_BWD3_VT

}  // namespace tc
}  // namespace ctcvr
