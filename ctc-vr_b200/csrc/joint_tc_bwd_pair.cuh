// Backward kernel 1 of the bf16 tcgen05 path on CTA PAIRS (included by joint_tc.cu): the default for D % 256 == 0.
// Same phases, tile geometry and data flow as joint_tc_bwd.cuh (read that header first); what changes is WHO multiplies:
// the two CTAs of a cluster take tiles 2i and 2i+1 (consecutive frame blocks of one (b, u-split) sweep) and one
// tcgen05.mma.cta_group::2 covers both:
//   P1  M = 256 (each CTA's own 128 rows, A in its own TMEM), N = Vp/2 x 2: every W_out stage is loaded HALF by each CTA
//   P3  M = 256 joint dims (CTA r owns d blocks r, r + 2), N = 256 rows: each CTA's G tile is its half of the B
//       operand, and each CTA streams only ITS W_out^T blocks - a quarter of the per-row traffic
//   P4  CTA r reduces its joint dims for both tiles (warp group 0: columns of tile 2i, warp group 1: tile 2i+1);
//       z is recomputed from the enc / pred rows of both tiles, so nothing is exchanged between the CTAs
// Shared-memory bandwidth bounds the single-CTA kernel (P1 at 1.2x, P3 at 1.6x their MMA floors: the tensor core's
// operand reads plus the copy engine's writes exceed 128 B/clk); a pair halves the operand traffic per flop.
// M = 256 keeps a k-block at 832 MMA cycles, which is what hides the ~1 k-cycle cluster hops of the hand-offs (the
// M = 128 pair form, joint_tc_fwd_pair.cuh, has 416-cycle k-blocks and starves on them).
// Only the leader (rank 0) issues MMAs; commits are multicast to both CTAs.  What the leader must know about the peer -
// "my half-stage has landed", "my A stage / G tile is written", "my TMEM is drained" - is forwarded by the peer's
// otherwise idle warp 1 with ONE relaxed remote mbarrier arrive per event, in the order the leader consumes them
// (a release.cluster arrive costs ~1 k cycles, which is what sank the first pair kernel of round 1).
#pragma once
#include "joint_tc_bwd.cuh"

namespace ctcvr {
namespace tc {

constexpr int BP_R1_MAX = 12;                  // W_out half-stages (P1): NH/2 x 128 B, over ring + G region
constexpr int BP_S_STAGES = 2;
constexpr uint32_t BP_ENC_REGION = 2048;       // P4 slab: enc rows of BOTH tiles (2 TT <= 16 rows)

// Shared memory: [weight ring: 4 W^T stages][G tile] -- P1 views both as one W ring of half-stages --
// [P1 slab ring][P4 slab: (D/128) stages of (pred rows | enc rows of both tiles)][bias][column-sum partials][barriers]
struct Bwd4Smem {
  uint32_t r_base, g_base, r1_bytes, s_base, p4_base, p4_bytes, bar_base;
  float* bias_l2;
  float* dbp;
  uint32_t* tmem_ptr;
  __device__ __forceinline__ uint32_t g_kblock(int i) const { return g_base + i * A_STAGE_BYTES; }
  __device__ __forceinline__ uint32_t r1_stage(int i) const { return r_base + i * r1_bytes; }
  __device__ __forceinline__ uint32_t r3_stage(int i) const { return r_base + i * 16384; }
  __device__ __forceinline__ uint32_t s_stage(int i) const { return s_base + i * B_SLAB_MAX; }
  __device__ __forceinline__ uint32_t p4_stage(int i) const { return p4_base + i * p4_bytes; }
  __device__ __forceinline__ uint32_t a_full(int i) const { return bar_base + i * 16; }             // 3
  __device__ __forceinline__ uint32_t a_empty(int i) const { return bar_base + i * 16 + 8; }
  __device__ __forceinline__ uint32_t s_full(int i) const { return bar_base + 416 + i * 16; }       // 3
  __device__ __forceinline__ uint32_t s_empty(int i) const { return bar_base + 416 + i * 16 + 8; }
  __device__ __forceinline__ uint32_t r1_full(int i) const { return bar_base + 80 + i * 16; }       // 12
  __device__ __forceinline__ uint32_t r1_empty(int i) const { return bar_base + 80 + i * 16 + 8; }
  __device__ __forceinline__ uint32_t r3_full(int i) const { return bar_base + 272 + i * 16; }      // 4
  __device__ __forceinline__ uint32_t r3_empty(int i) const { return bar_base + 272 + i * 16 + 8; }
  __device__ __forceinline__ uint32_t dz_full(int mb) const { return bar_base + 336 + mb * 8; }     // 2
  __device__ __forceinline__ uint32_t tmem_full() const { return bar_base + 352; }
  __device__ __forceinline__ uint32_t g_full() const { return bar_base + 360; }
  __device__ __forceinline__ uint32_t tmem_empty() const { return bar_base + 368; }
  __device__ __forceinline__ uint32_t gs_done() const { return bar_base + 376; }
  __device__ __forceinline__ uint32_t p4_full() const { return bar_base + 384; }
  __device__ __forceinline__ uint32_t g_peer() const { return bar_base + 392; }        // leader: the peer's G tile is written
  __device__ __forceinline__ uint32_t te_peer() const { return bar_base + 400; }       // leader: the peer's TMEM is drained
};
constexpr uint32_t BP_BAR_BYTES = 464;

template <int P>
__host__ __device__ constexpr uint32_t bwd4_p4_stage_bytes() { return bwd_pred_region<P>() + BP_ENC_REGION; }
__host__ __device__ inline int bwd4_r1_stages(int NH, int Vp) {
  const int n = (int)((B_RING_BYTES + bwd3_g_bytes(Vp)) / ((uint32_t)(NH / 2) * 128u));
  return n > BP_R1_MAX ? BP_R1_MAX : n;
}
template <int P>
__host__ __device__ inline size_t bwd4_smem_bytes(int NH, int Vp, int D) {
  size_t s = 1024;
  s += B_RING_BYTES + bwd3_g_bytes(Vp);
  s += (size_t)BP_S_STAGES * B_SLAB_MAX;
  s += (size_t)(D / 128) * bwd4_p4_stage_bytes<P>();
  s += (size_t)Vp * 4 + (size_t)4 * Vp * 4;
  s += 16 + BP_BAR_BYTES + 16;
  return s;
}
template <int P>
__device__ __forceinline__ void carve_bwd4(Bwd4Smem& L, uint8_t* raw, int NH, int Vp, int D) {
  const uint32_t base = smem_u32(raw);
  uint32_t a = (base + 1023u) & ~1023u;
  L.r_base = a; L.r1_bytes = (uint32_t)(NH / 2) * 128u; a += B_RING_BYTES;
  L.g_base = a; a += bwd3_g_bytes(Vp);
  L.s_base = a; a += BP_S_STAGES * B_SLAB_MAX;
  L.p4_base = a; L.p4_bytes = bwd4_p4_stage_bytes<P>(); a += (uint32_t)(D / 128) * L.p4_bytes;
  L.bias_l2 = reinterpret_cast<float*>(raw + (a - base)); a += Vp * 4;
  L.dbp = reinterpret_cast<float*>(raw + (a - base)); a += 4 * Vp * 4;
  a = (a + 15u) & ~15u;
  L.bar_base = a; a += BP_BAR_BYTES;
  L.tmem_ptr = reinterpret_cast<uint32_t*>(raw + (a - base));
}

// ACT: the joint activation of the P1 producers and the P4 derivative (ACT_TANH / ACT_RELU / ACT_GELU)
template <int P, int TT, int ACT>
__device__ __forceinline__ void joint_bwd4_body(const CUtensorMap& tmap_e, const CUtensorMap& tmap_e2,
                                                const CUtensorMap& tmap_p, const BwdParams& p) {
  static_assert(2 * TT * 128 <= (int)BP_ENC_REGION, "the enc rows of both tiles share one 2 KB region");
  extern __shared__ uint8_t smem_raw[];
  Bwd4Smem L;
  carve_bwd4<P>(L, smem_raw, p.NH, p.Vp, p.D);
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const int NQ = p.NH >> 1;
  const int KB = p.D / BK;                 // k-blocks of the logits GEMM
  const int KBG = (p.Vp + 63) / 64;        // k-blocks (over v) of the dZ GEMM
  const int MB2 = p.D / 256;               // 256-row blocks of dZ^T: this CTA owns d block 2 mb2 + rank of each
  const int R1 = p.r1_stages;
  const int npairs = (*p.ntiles) >> 1;     // the tile table pads every (b, u-split) sweep to an even number of tiles
  const int ncl = (int)gridDim.x >> 1, cl = (int)blockIdx.x >> 1;
  const int pair_begin = (int)(((long)npairs * cl) / ncl), pair_end = (int)(((long)npairs * (cl + 1)) / ncl);

  if (warp == 0 && lane == 0) {
    g_tc_error_host = p.err_host;
    tma_prefetch_desc(&tmap_e);
    tma_prefetch_desc(&tmap_e2);
    tma_prefetch_desc(&tmap_p);
    const uint32_t fwd = rank == 0 ? 1u : 0u;   // the leader's operand barriers take one forwarded arrival from the peer
    // a_full: the peer's 8 producer warps arrive on the leader's barrier themselves (relaxed remote arrives: one hop less
    // than a forward, and the A stages - 3 k-blocks of TMEM - are the shallowest ring of the kernel)
    for (int i = 0; i < B_A_STAGES; ++i) { mbar_init(L.a_full(i), 8 + 8 * fwd); mbar_init(L.a_empty(i), 1); }
    for (int i = 0; i < BP_S_STAGES; ++i) { mbar_init(L.s_full(i), 1); mbar_init(L.s_empty(i), 8); }
    for (int i = 0; i < BP_R1_MAX; ++i) { mbar_init(L.r1_full(i), 1 + fwd); mbar_init(L.r1_empty(i), 1); }
    for (int i = 0; i < B_R3_STAGES; ++i) { mbar_init(L.r3_full(i), 1 + fwd); mbar_init(L.r3_empty(i), 1); }
    for (int i = 0; i < 2; ++i) mbar_init(L.dz_full(i), 1);
    mbar_init(L.tmem_full(), 1);
    mbar_init(L.g_full(), WORKERS / 32);
    mbar_init(L.tmem_empty(), 8);
    mbar_init(L.gs_done(), 1);
    mbar_init(L.p4_full(), 1);
    mbar_init(L.g_peer(), 1);
    mbar_init(L.te_peer(), 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc2(smem_u32(L.tmem_ptr), TMEM_COLS);
  for (int i = tid; i < p.Vp; i += NTHREADS) L.bias_l2[i] = p.bias_l2[i];
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                       // the peer's barriers exist before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *L.tmem_ptr;

  if (warp == 0) {
    // ------------------------------------------------------------------ bulk copies: this CTA's half of W_out (P1), its
    // W_out^T blocks (P3), and the spill of its G tile
    Pipe r1, r3;
    int prof_n = 0;
    uint32_t ph = 0;
    const uint32_t r1_bytes = (uint32_t)NQ * 128u;
    for (int pi = pair_begin; pi < pair_end; ++pi) {
      const int tile = 2 * pi + (int)rank;
      if (lane == 0) TC_PROF(0, 1);
      // ring + G region are dead here: the previous tile's last dZ block and its G spill / column sums were observed below
      for (int i = 0; i < 2 * KB; ++i) {
        mbar_wait(L.r1_empty(r1.stage), r1.phase ^ 1u, 11);
        if (elect_one()) {
          mbar_arrive_expect_tx(L.r1_full(r1.stage), r1_bytes);
          bulk_load(L.r1_stage(r1.stage), p.w_t + ((size_t)i * p.NH + (size_t)rank * NQ) * 64, r1_bytes, L.r1_full(r1.stage));
        }
        __syncwarp();
        r1.advance(R1);
      }
      if (lane == 0) TC_PROF(0, 2);
      mbar_wait(L.tmem_full(), ph, 12);           // every P1 MMA has completed: the W view of the ring is dead
      if (lane == 0) TC_PROF(0, 3);
      // W_out^T stages of d blocks 2 mb2 + rank, the spill of the finished G tile interleaved (one 8 KB bulk store
      // behind every stage load beyond the preloaded ones; see joint_tc_bwd.cuh)
      __nv_bfloat16* gdst = p.gt + ((size_t)p.tiles[tile].w * 2) * (size_t)KBG * 4096;
      int ns = 0;
      auto spill = [&](int j) {
        bulk_store(gdst + ((size_t)(j & 1) * KBG + (j >> 1)) * 4096, L.g_kblock(j >> 1) + (uint32_t)(j & 1) * 8192u, 8192u);
      };
      for (int mb2 = 0; mb2 < MB2; ++mb2)
        for (int kb = 0; kb < KBG; ++kb) {
          const int i = mb2 * KBG + kb;
          mbar_wait(L.r3_empty(r3.stage), r3.phase ^ 1u, 13);
          const bool st = i >= B_R3_STAGES && ns < 2 * KBG;
          if (elect_one()) {
            mbar_arrive_expect_tx(L.r3_full(r3.stage), 16384u);
            bulk_load(L.r3_stage(r3.stage), p.wt_t + ((size_t)(2 * mb2 + (int)rank) * KBG + kb) * 8192, 16384u, L.r3_full(r3.stage));
            if (st) spill(ns);
          }
          if (st) ++ns;
          __syncwarp();
          r3.advance(B_R3_STAGES);
        }
      mbar_wait(L.g_full(), ph, 18);
      if (elect_one()) {
        for (int j = ns; j < 2 * KBG; ++j) spill(j);
        bulk_commit();
      }
      __syncwarp();
      if (lane == 0) TC_PROF(0, 4);
      mbar_wait(L.dz_full(MB2 - 1), ph, 14);      // every P3 MMA has completed: G tile and the W^T view are dead
      mbar_wait(L.gs_done(), ph, 16);             // ... the d_bias column sums have read G
      if (elect_one()) bulk_wait_read<0>();       // ... and so have the spill stores
      __syncwarp();
      if (lane == 0) TC_PROF(0, 5);
      ph ^= 1u;
    }
  } else if (warp == 3) {
    // ------------------------------------------------------------------ TMA: enc / pred slabs (P1 ring of the CTA's own
    // tile + the P4 slab: the d k-blocks of this CTA's d blocks, pred rows and the enc rows of BOTH tiles)
    Pipe sp;
    uint32_t ph = 0;
    for (int pi = pair_begin; pi < pair_end; ++pi) {
      const int4 ti = p.tiles[2 * pi + (int)rank];
      const int b = ti.x;
      const int W = max(min(p.u_len[b], p.U1 - 1), 0) + 1;
      const int S = (W + P - 1) / P, us = (W + S - 1) / S;
      const int prow = b * p.U1 + ti.y * us;
      const int erow = b * p.T + ti.z * TT;
      const int erow0 = erow - (int)rank * TT;    // first frame of tile 2i (the pair covers 2 TT consecutive frames)
      for (int kb = 0; kb < KB; ++kb) {
        mbar_wait(L.s_empty(sp.stage), sp.phase ^ 1u, 15);
        if (elect_one()) {
          const uint32_t st = L.s_stage(sp.stage);
          mbar_arrive_expect_tx(L.s_full(sp.stage), (uint32_t)(P + TT) * 128u);
          tma_load_2d(st, &tmap_p, L.s_full(sp.stage), kb * BK, prow);
          tma_load_2d(st + bwd_pred_region<P>(), &tmap_e, L.s_full(sp.stage), kb * BK, erow);
        }
        __syncwarp();
        sp.advance(BP_S_STAGES);
      }
      mbar_wait(L.tmem_empty(), ph ^ 1u, 17);     // the P4 readers of the previous pair are done
      if (elect_one()) {
        mbar_arrive_expect_tx(L.p4_full(), (uint32_t)(2 * MB2) * (uint32_t)(P + 2 * TT) * 128u);
        for (int s = 0; s < 2 * MB2; ++s) {       // slab stage s = (mb2, 64-wide half j): k-block (2 mb2 + rank) * 2 + j
          const int kb = (2 * (s >> 1) + (int)rank) * 2 + (s & 1);
          const uint32_t st = L.p4_stage(s);
          tma_load_2d(st, &tmap_p, L.p4_full(), kb * BK, prow);
          tma_load_2d(st + bwd_pred_region<P>(), &tmap_e2, L.p4_full(), kb * BK, erow0);     // 2 TT rows: both tiles' frames
        }
      }
      __syncwarp();
      ph ^= 1u;
    }
  } else if (warp == 1) {
    Pipe ap, r1, r3;
    int prof_n = 0;
    uint32_t ph = 0;
    if (rank == 0) {
      // ---------------------------------------------------------------- MMA issuer (leader; warp-wide loop, one lane issues)
      const uint32_t idesc1 = make_idesc_bf16(256, p.NH);
      const uint32_t idesc2 = make_idesc_bf16(256, 256);
      const uint64_t r1_desc0 = make_desc_sw128(L.r1_stage(0));     // + stage * NQ * 8
      const uint64_t r3_desc0 = make_desc_sw128(L.r3_stage(0));     // + stage * 1024
      const uint64_t g_desc0 = make_desc_sw128(L.g_kblock(0));      // + kb * 1024
      const uint32_t r1_step = (uint32_t)NQ * 8u;
      const int last_nks = (p.Vp - (KBG - 1) * 64) / 16;
      for (int pi = pair_begin; pi < pair_end; ++pi) {
        if (lane == 0) TC_PROF(1, 1);
        mbar_wait(L.tmem_empty(), ph ^ 1u, 20);
        mbar_wait(L.te_peer(), ph ^ 1u, 25);
        if (lane == 0) TC_PROF(1, 2);
        tc_fence_after();
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
              umma2_bf16_ts(d, a, bd, idesc1, kb ? 1u : 0u);
              umma2_bf16_ts(d, a + 8, bd + 2, idesc1, 1u);
              umma2_bf16_ts(d, a + 16, bd + 4, idesc1, 1u);
              umma2_bf16_ts(d, a + 24, bd + 6, idesc1, 1u);
              umma2_commit_mc(L.r1_empty(r1.stage), 3);
              if (h == 1) umma2_commit_mc(L.a_empty(ap.stage), 3);
            }
            __syncwarp();
            r1.advance(R1);
          }
          ap.advance(B_A_STAGES);
        }
        if (elect_one()) umma2_commit_mc(L.tmem_full(), 3);
        __syncwarp();
        if (lane == 0) TC_PROF(1, 3);
        // ---- P3: dZ^T[mb2] (256 d x 256 rows) = W^T[mb2] (256 x Vp) . G^T (Vp x 256); each block is handed to P4 on its own
        mbar_wait(L.g_full(), ph, 23);
        mbar_wait(L.g_peer(), ph, 26);
        if (lane == 0) TC_PROF(1, 4);
        tc_fence_after();
        for (int mb2 = 0; mb2 < MB2; ++mb2) {
          for (int kb = 0; kb < KBG; ++kb) {
            mbar_wait(L.r3_full(r3.stage), r3.phase, 24);
            tc_fence_after();
            if (elect_one()) {
              const uint64_t ad = r3_desc0 + (uint64_t)(r3.stage * 1024);
              const uint64_t bd = g_desc0 + (uint64_t)(kb * 1024);
              const uint32_t d = tmem_base + mb2 * 256;
              const int nks = kb == KBG - 1 ? last_nks : 4;
              if (nks > 0) umma2_bf16(d, ad, bd, idesc2, kb ? 1u : 0u);
              if (nks > 1) umma2_bf16(d, ad + 2, bd + 2, idesc2, 1u);
              if (nks > 2) umma2_bf16(d, ad + 4, bd + 4, idesc2, 1u);
              if (nks > 3) umma2_bf16(d, ad + 6, bd + 6, idesc2, 1u);
              umma2_commit_mc(L.r3_empty(r3.stage), 3);
              if (kb == KBG - 1) umma2_commit_mc(L.dz_full(mb2), 3);
            }
            __syncwarp();
            r3.advance(B_R3_STAGES);
          }
          if (lane == 0) TC_PROF(1, 10 + mb2);
        }
        if (lane == 0) TC_PROF(1, 5);
        ph ^= 1u;
      }
    } else {
      // ---------------------------------------------------------------- peer: forward local readiness to the leader, in
      // the leader's order, one relaxed remote arrive per event
      auto fwd = [&](uint32_t bar) { if (lane == 0) mbar_arrive_remote_relaxed(bar, 0); __syncwarp(); };
      for (int pi = pair_begin; pi < pair_end; ++pi) {
        if (pi != pair_begin) {                    // the leader's first wait on te_peer passes by parity
          mbar_wait(L.tmem_empty(), ph ^ 1u, 30);
          fwd(L.te_peer());
        }
        for (int kb = 0; kb < KB; ++kb) {
          for (int h = 0; h < 2; ++h) {
            mbar_wait(L.r1_full(r1.stage), r1.phase, 32);
            fwd(L.r1_full(r1.stage));
            r1.advance(R1);
          }
          ap.advance(B_A_STAGES);
        }
        mbar_wait(L.g_full(), ph, 33);
        fwd(L.g_peer());
        for (int i = 0; i < MB2 * KBG; ++i) {
          mbar_wait(L.r3_full(r3.stage), r3.phase, 34);
          fwd(L.r3_full(r3.stage));
          r3.advance(B_R3_STAGES);
        }
        ph ^= 1u;
      }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ workers (warps 4-15): P1 producers, P2, P4 / d_bias
    const int q = warp & 3;
    const int wg = (warp - 4) >> 2;            // 0..2
    const int r = q * 32 + lane;               // P2: tile row ; P4: lane of the d block
    const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t ph = 0;
    int prof_n = 0;
    float db[4] = {0.f, 0.f, 0.f, 0.f};        // warp group 2: d_bias of columns r, r + 128, r + 256, r + 384
    float pacc[2][P];                          // warp groups 0/1: d_pred sums of d blocks rank, 2 + rank over one sweep
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < P; ++j) pacc[i][j] = 0.f;
    int cur_b = -1, cur_ubase = 0;
    auto flush_pred = [&]() {
      if (cur_b < 0 || wg >= 2) return;
      const int Ub = max(min(p.u_len[cur_b], p.U1 - 1), 0);
#pragma unroll
      for (int mb2 = 0; mb2 < 2; ++mb2) {
        if (mb2 < MB2) {
          const int d = (2 * mb2 + (int)rank) * 128 + r;
#pragma unroll
          for (int j = 0; j < P; ++j) {
            const int u = cur_ubase + j;
            if (u <= Ub) atomicAdd(p.d_pred + ((size_t)cur_b * p.U1 + u) * p.D + d, pacc[mb2][j]);
            pacc[mb2][j] = 0.f;
          }
        }
      }
    };
    const int p_tloc = min(r / P, TT - 1), p_ul = r % P;
    const uint32_t e_row = bwd_pred_region<P>() + (uint32_t)p_tloc * 128u, e_sw = (uint32_t)(p_tloc & 7);
    const uint32_t p_row = (uint32_t)p_ul * 128u, p_sw = (uint32_t)(p_ul & 7);
    uint32_t kb_base = 0;

    for (int pi = pair_begin; pi < pair_end; ++pi) {
      int4 ti = p.tiles[2 * pi + (int)rank];
      pin(ti.x); pin(ti.y); pin(ti.z); pin(ti.w);
      BwdGeom<P, TT> g;
      g.init(p.t_len, p.u_len, p.T, p.U1, ti);
      if (g.b != cur_b || g.ubase != cur_ubase) { flush_pred(); cur_b = g.b; cur_ubase = g.ubase; }

      // ---------------- P1: A k-blocks of this CTA's tile into its TMEM
      {
        mbar_wait(L.tmem_empty(), ph ^ 1u, 40);
        if (tid == 128) TC_PROF(3, 1);
        for (int s = wg; s < 2 * KB; s += 3) {
          const int kb = s >> 1, kh = s & 1;
          const uint32_t kbc = kb_base + (uint32_t)kb;
          const uint32_t a_stg = kbc % B_A_STAGES, a_ph = (kbc / B_A_STAGES) & 1u;
          const uint32_t s_stg = kbc % BP_S_STAGES, s_ph = (kbc / BP_S_STAGES) & 1u;
          mbar_wait(L.s_full(s_stg), s_ph, 41);
          mbar_wait(L.a_empty(a_stg), a_ph ^ 1u, 42);
          tc_fence_after();
          const uint32_t sb = L.s_stage(s_stg);
          uint32_t w[16];
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const uint32_t c = (uint32_t)(kh * 4 + c4);
            uint4 ev, pv;
            if (CTCVR_EXP & 4) { ev = make_uint4(sb, c, kh, kb); pv = ev; }
            else { ev = lds128(sb + e_row + ((c ^ e_sw) << 4)); pv = lds128(sb + p_row + ((c ^ p_sw) << 4)); }
            if (CTCVR_EXP & 8) { w[4 * c4 + 0] = ev.x ^ pv.y; w[4 * c4 + 1] = ev.y; w[4 * c4 + 2] = ev.z; w[4 * c4 + 3] = ev.w; }
            else {
            w[4 * c4 + 0] = act_add_bf16x2_packed<ACT>(ev.x, pv.x);
            w[4 * c4 + 1] = act_add_bf16x2_packed<ACT>(ev.y, pv.y);
            w[4 * c4 + 2] = act_add_bf16x2_packed<ACT>(ev.z, pv.z);
            w[4 * c4 + 3] = act_add_bf16x2_packed<ACT>(ev.w, pv.w);
            }
          }
          tmem_st16(tq + (uint32_t)(B_ACC_COLS + a_stg * 32 + kh * 16), w);
          tmem_st_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) { if (rank == 0) mbar_arrive(L.a_full(a_stg)); else mbar_arrive_remote_relaxed(L.a_full(a_stg), 0); }
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
          if ((unsigned)lab >= (unsigned)p.V) lab = p.blank;      // out-of-range ids cannot index outside the tile
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
        if (fast) {
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
          const unsigned short h = __bfloat16_as_ushort(__float2bfloat16(val));
          const uint32_t a = L.g_kblock(col >> 6) + r * 128 + ((((col & 63) >> 3) ^ (r & 7)) << 4) + (col & 7) * 2;
          asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"(h) : "memory");
        };
        if (((p.blank >> 4) % 3) == wg) put(p.blank, entry(lpb, bnext, (lab == p.blank) ? bl1 : kNegInf));
        if (lab >= 0 && lab != p.blank && ((lab >> 4) % 3) == wg) put(lab, entry(lpl, bl1, kNegInf));
      }
      fence_proxy_async();
      tc_fence_before();
      warp_arrive(L.g_full());
      if (tid == 128) TC_PROF(2, 3);

      if (wg == 2) {
        // ---------------- P3 side work (warps 12-15): spill the G tile, d_bias = its column sums
        mbar_wait(L.g_full(), ph, 31);
        const int nchunk = p.Vp >> 3;
        for (int it = r; it < 4 * nchunk; it += 128) {
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
        if (r == 0) mbar_arrive(L.gs_done());
      } else {
        // ---------------- P4 (warps 4-11), overlapped with P3: dH = dZ * (1 - z^2); reductions.  TMEM lane = joint dim
        // (2 mb2 + rank) * 128 + r; columns [0,128) are the rows of tile 2i, [128,256) those of tile 2i+1: warp group wg
        // takes the columns (and the enc rows) of tile 2i + wg, for both d blocks of this CTA.
        mbar_wait(L.p4_full(), ph, 34);
        const int zt = ti.z - (int)rank + wg;                       // frame block of the tile this warp group reduces
#pragma unroll
        for (int mb2 = 0; mb2 < 2; ++mb2) {
          if (mb2 < MB2) {
            const int d = (2 * mb2 + (int)rank) * 128 + r;
            uint32_t e[TT], pr[P];
            {
              const uint32_t st = L.p4_stage(mb2 * 2 + (r >> 6)) + (uint32_t)(r & 7) * 2u;
              const uint32_t chn = (uint32_t)((r & 63) >> 3);
#pragma unroll
              for (int i = 0; i < P; ++i) {
                unsigned short x;
                asm volatile("ld.shared.u16 %0, [%1];" : "=h"(x) : "r"(st + i * 128 + ((chn ^ (uint32_t)(i & 7)) << 4)));
                pr[i] = x;
              }
#pragma unroll
              for (int i = 0; i < TT; ++i) {
                const uint32_t row = (uint32_t)(wg * TT + i);      // row within the enc region (both tiles' frames)
                unsigned short x;
                asm volatile("ld.shared.u16 %0, [%1];" : "=h"(x) : "r"(st + bwd_pred_region<P>() + row * 128 + ((chn ^ (row & 7u)) << 4)));
                e[i] = x;
              }
            }
            mbar_wait(L.dz_full(mb2), ph, 32);
            if (tid == 128) TC_PROF(2, 40 + mb2);
            tc_fence_after();
            float es[TT];
#pragma unroll
            for (int i = 0; i < TT; ++i) es[i] = 0.f;
            float v0[16], v1[16];
            const uint32_t tb = tq + (uint32_t)(mb2 * 256 + wg * 128);
            tmem_ld16(tb, v0);
            tmem_ld_wait();
            tmem_ld16(tb + 16, v1);
            p4_chunk<P, TT, 0, ACT>(v0, e, pr, es, pacc[mb2]);
            tmem_ld_wait();
            tmem_ld16(tb + 32, v0);
            p4_chunk<P, TT, 16, ACT>(v1, e, pr, es, pacc[mb2]);
            tmem_ld_wait();
            tmem_ld16(tb + 48, v1);
            p4_chunk<P, TT, 32, ACT>(v0, e, pr, es, pacc[mb2]);
            tmem_ld_wait();
            tmem_ld16(tb + 64, v0);
            p4_chunk<P, TT, 48, ACT>(v1, e, pr, es, pacc[mb2]);
            tmem_ld_wait();
            tmem_ld16(tb + 80, v1);
            p4_chunk<P, TT, 64, ACT>(v0, e, pr, es, pacc[mb2]);
            tmem_ld_wait();
            tmem_ld16(tb + 96, v0);
            p4_chunk<P, TT, 80, ACT>(v1, e, pr, es, pacc[mb2]);
            tmem_ld_wait();
            tmem_ld16(tb + 112, v1);
            p4_chunk<P, TT, 96, ACT>(v0, e, pr, es, pacc[mb2]);
            tmem_ld_wait();
            p4_chunk<P, TT, 112, ACT>(v1, e, pr, es, pacc[mb2]);
#pragma unroll
            for (int i = 0; i < TT; ++i) {
              const int tt = zt * TT + i;
              if (tt < g.Tb) p.d_enc_part[(((size_t)ti.y * p.B + g.b) * p.T + tt) * p.D + d] = es[i];
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
    if (wg == 2 && pair_end > pair_begin) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (r + 128 * i < p.V) atomicAdd(p.d_bias + r + 128 * i, db[i]);
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                       // no MMA / multicast commit / remote arrive may target a CTA that has left
  if (warp == 2) tmem_dealloc2(tmem_base, TMEM_COLS);
}

#define CTCVR_BWD4(name, act)                                                                                      \
  template <int P, int TT>                                                                                          \
  __global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)                                          \
  name(const __grid_constant__ CUtensorMap tmap_e, const __grid_constant__ CUtensorMap tmap_e2,                     \
       const __grid_constant__ CUtensorMap tmap_p, const BwdParams p) {                                             \
    joint_bwd4_body<P, TT, act>(tmap_e, tmap_e2, tmap_p, p);                                                        \
  }
CTCVR_BWD4(joint_bwd4_kernel, ACT_TANH)
CTCVR_BWD4(joint_bwd4_relu_kernel, ACT_RELU)     // relu / gelu joints, named apart for profiler traces
CTCVR_BWD4(joint_bwd4_gelu_kernel, ACT_GELU)
#undef CTCVR_BWD4

}  // namespace tc
}  // namespace ctcvr
