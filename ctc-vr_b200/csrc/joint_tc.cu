// bf16 tcgen05 path of the fused transducer joint (the performance path on B200).
//
//   z      = tanh(enc_proj[b,t,:] + pred_proj[b,u,:])        model/component/joint.py:57-67
//   logits = z . W_out^T + b_out                             model/component/joint.py:68
//   fwd   : per lattice cell lse / lp_blank / lp_label (log-softmax + gather of
//           torchaudio.functional.rnnt_loss, model/component/transducer.py:180-187)
//   bwd   : recompute logits, closed-form d cost/d logits, dZ = g.W, dH = dZ*(1-z^2),
//           d_enc = sum_u dH, d_pred = sum_t dH, dW = g^T.z, db = sum g
//
// Structure (one persistent CTA per SM, 512 threads, warp-specialised):
//   warp 0      TMA producer : streams bf16 W_out k-blocks (128B-swizzled, K-major) into a smem ring
//   warp 1      MMA issuer   : one elected thread issues tcgen05.mma (M=128, N=Vp/2 x2, K=16), fp32
//                              accumulators live in TMEM, commits release smem stages / signal the epilogue
//   warp 2      TMEM allocator
//   warps 4-7   epilogue     : tcgen05.ld (thread = lattice cell), online log-softmax, gathers
//   warps 8-15  A producers  : the A operand is COMPUTED, not loaded: tanh(e+p) -> bf16 -> smem in the
//                              UMMA canonical swizzled layout, fence.proxy.async, mbarrier arrive
// The [B,T,U+1,V] logits only ever exist as TMEM tiles.
#include <algorithm>
#include <stdlib.h>

#include "tc_common.cuh"

namespace ctcvr {
namespace tc {

constexpr int BM = 128;            // lattice cells (rows) per tile
constexpr int BK = 64;             // k-block: 64 bf16 = 128 B = one swizzle row
constexpr int NTHREADS = 512;
constexpr int A_STAGE_BYTES = BM * BK * 2;        // 16 KB
constexpr int PROD_THREADS = 256;
constexpr int TMEM_COLS = 512;
constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;

enum { TILE_FLAT = 0, TILE_RECT = 1 };
constexpr int PROF_CAP = 2048;
// timeline probe for CTA 0 (one lane per role); compiled in always, active only when p.prof != nullptr
#define TC_PROF(role, tag)                                                                         \
  do {                                                                                             \
    if (p.prof != nullptr && blockIdx.x == 0 && blockIdx.y == 0) {                                                   \
      int _n = prof_n++;                                                                           \
      if (_n < PROF_CAP) p.prof[(role)*PROF_CAP + _n] = ((long long)(tag) << 48) | (clock64() & 0xffffffffffffLL); \
    }                                                                                              \
  } while (0)


struct RowMap {
  int b, Tb, Ub, W;
  int t0;        // first frame covered by the tile
  int ubase;     // first label column covered by the tile's pred slab rows
  int np, ne;    // slab rows holding pred / enc vectors
};

// Opaque identity: stops the compiler from re-deriving a per-tile value from global memory inside the
// k-block loops (it otherwise rematerialises the tile-table / length loads there, a chain of two L2
// round trips in front of every operand fetch).
__device__ __forceinline__ void pin(int& x) { asm volatile("" : "+r"(x)); }

// ---- tile geometry ---------------------------------------------------------------------------
template <int TILE>
__device__ __forceinline__ RowMap tile_geometry(const int32_t* t_len, const int32_t* u_len, int T, int U1, int4 ti) {
  RowMap g;
  g.b = ti.x;
  g.Tb = max(min(t_len[g.b], T), 0);
  g.Ub = max(min(u_len[g.b], U1 - 1), 0);
  g.W = g.Ub + 1;
  if (TILE == TILE_FLAT) {
    int ncell = g.Tb * g.W;
    int c0 = ti.y;
    int clast = min(c0 + BM - 1, ncell - 1);
    g.t0 = c0 / g.W;
    g.ubase = 0;
    g.np = g.W;
    g.ne = clast / g.W - g.t0 + 1;
  } else {
    int S = (g.W + 15) >> 4;
    int us = (g.W + S - 1) / S;
    g.t0 = ti.z * 8;
    g.ubase = ti.y * us;
    g.np = 16;
    g.ne = 8;
  }
  pin(g.b); pin(g.Tb); pin(g.Ub); pin(g.W); pin(g.t0); pin(g.ubase); pin(g.np); pin(g.ne);
  return g;
}

// row r of the tile -> lattice cell; returns false for padding rows
template <int TILE>
__device__ __forceinline__ bool row_cell(const RowMap& g, int4 ti, int r, int& t, int& u) {
  if (TILE == TILE_FLAT) {
    int c = ti.y + r;
    t = c / g.W;
    u = c - t * g.W;
    return c < g.Tb * g.W;
  } else {
    int S = (g.W + 15) >> 4;
    int us = (g.W + S - 1) / S;
    int tloc = r >> 4, ul = r & 15;
    t = g.t0 + tloc;
    u = g.ubase + ul;
    return t < g.Tb && ul < us && u <= g.Ub;
  }
}

struct Pipe {
  int stage = 0;
  uint32_t phase = 0;
  __device__ __forceinline__ void advance(int n) {
    if (++stage == n) { stage = 0; phase ^= 1u; }
  }
};

}  // namespace tc
}  // namespace ctcvr
#include "joint_tc_fwd.cuh"
#include "joint_tc_fwd_pair.cuh"
#include "joint_tc_bwd.cuh"
#include "joint_tc_bwd_pair.cuh"
namespace ctcvr {
namespace tc {

// d_enc[b,t,:] = sum over the u-splits of the partial sums (zero for padded frames).  OUT_BF16 (bf16-input entry
// point): d_enc is written as bf16 and blocks B*T.. convert the fp32 d_pred accumulator to bf16 as well.
template <bool OUT_BF16>
__global__ void reduce_denc_kernel(const float* __restrict__ part, const int32_t* __restrict__ t_len,
                                   const int32_t* __restrict__ u_len, void* __restrict__ d_enc_out, int B, int T, int U1,
                                   int D, int P, const float* __restrict__ d_pred_acc, void* __restrict__ d_pred_out) {
  const int bt = blockIdx.x;
  if (bt >= B * T) {                      // d_pred rows (OUT_BF16 only)
    const size_t row = (size_t)(bt - B * T) * D;
    for (int d = threadIdx.x * 4; d < D; d += blockDim.x * 4) {
      const float4 x = *reinterpret_cast<const float4*>(d_pred_acc + row + d);
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(d_pred_out) + row + d) =
          make_uint2(pack_bf16(x.x, x.y), pack_bf16(x.z, x.w));
    }
    return;
  }
  const int b = bt / T, t = bt - b * T;
  const int Tb = max(min(t_len[b], T), 0), W = max(min(u_len[b], U1 - 1), 0) + 1;
  const int S = (W + P - 1) / P;
  const size_t row = ((size_t)b * T + t) * D, step = (size_t)B * T * D;
  for (int d = threadIdx.x * 4; d < D; d += blockDim.x * 4) {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t < Tb)
      for (int i = 0; i < S; ++i) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(part + (size_t)i * step + row + d));
        s.x += x.x; s.y += x.y; s.z += x.z; s.w += x.w;
      }
    if (OUT_BF16)
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(d_enc_out) + row + d) = make_uint2(pack_bf16(s.x, s.y), pack_bf16(s.z, s.w));
    else
      *reinterpret_cast<float4*>(reinterpret_cast<float*>(d_enc_out) + row + d) = s;
  }
}

// =================================================================================================
// Backward kernel 2: dW^T[d][v] = sum_rows z^T[d][row] * g[row][v]  (tcgen05 GEMM, split-K over the row tiles).
// g is read as the row-major G tiles spilled by kernel 1 ([tile][2][KBG][64 rows][64 v], one 1-D bulk copy per 64-row
// stage): the B operand is MN-major (label columns contiguous), N split at a multiple of 64 columns (256 + the rest).
// z^T is RECOMPUTED instead of spilled by kernel 1 and read back: z = tanh(enc + pred) costs one MUFU op per element
// (512 cycles per 64-row stage per SM, under the 832 cycles of the stage's MMAs), whereas a z^T spill is
// D x rows x 2 B = 352 MB at cfg2, written once and read once from HBM.  The A operand lives in TMEM (TS mode):
// lane = d, one 32-bit column per pair of rows.  Producer thread = (d, 32 rows of the stage); it holds the TT enc and
// P pred values of its d for the current row tile in registers, read from a TMA-staged slab once per 128 rows.
// TMEM: accumulators [0, Vp) | A stages 416.. (3 x 32 columns).
// =================================================================================================
constexpr int DW_STAGES = 3;
constexpr int DWR_ROW_PARTS = 4;                 // producer warps per d quarter: each takes 64 / parts rows of a stage
constexpr int DWR_THREADS = (4 + 4 * DWR_ROW_PARTS) * 32;
constexpr int DWR_A_STAGES = 3;
constexpr int DWR_ACC_COLS = 416;

// rows R0 .. R0+2*NP-1 of a tile: NP packed (row 2c, row 2c+1) pairs of tanh(e[tloc] + p[ul]), row = tloc*P + ul
template <int P, int TT, int R0, int NP, int ACT = ACT_TANH>
__device__ __forceinline__ void dwr_rows(const uint32_t (&e)[TT], const uint32_t (&pr)[P], uint32_t (&w)[NP]) {
#pragma unroll
  for (int c = 0; c < NP; ++c) {
    const int r0 = R0 + 2 * c, r1 = r0 + 1;
    const int tl0 = (r0 / P < TT) ? r0 / P : TT - 1, tl1 = (r1 / P < TT) ? r1 / P : TT - 1;
    const int u0 = r0 % P, u1 = r1 % P;
    const uint32_t ep = __byte_perm(e[tl0], e[tl1], 0x5410);
    const uint32_t pp = __byte_perm(pr[u0], pr[u1], 0x5410);
    w[c] = act_add_bf16x2_packed<ACT>(ep, pp);
  }
}

// bf16x3: the same rows as hi / lo pairs of the fp32 act(e + p)
template <int P, int TT, int R0, int NP, int ACT = ACT_TANH>
__device__ __forceinline__ void dwr_rows_x3(const float (&e)[TT], const float (&pr)[P], uint32_t (&hi)[NP], uint32_t (&lo)[NP]) {
#pragma unroll
  for (int c = 0; c < NP; ++c) {
    const int r0 = R0 + 2 * c, r1 = r0 + 1;
    const int tl0 = (r0 / P < TT) ? r0 / P : TT - 1, tl1 = (r1 / P < TT) ? r1 / P : TT - 1;
    const float z0 = act_f32<ACT>(e[tl0] + pr[r0 % P]), z1 = act_f32<ACT>(e[tl1] + pr[r1 % P]);
    const __nv_bfloat162 h = __floats2bfloat162_rn(z0, z1);
    hi[c] = *reinterpret_cast<const uint32_t*>(&h);
    lo[c] = pack_bf16(z0 - __low2float(h), z1 - __high2float(h));
  }
}

constexpr int DWR_S_STAGES = 3;
constexpr int DW_STAGES_X3 = 4;                  // bf16x3: the G_hi and G_lo stages of two k-blocks (no slab ring)
template <int P>
__host__ __device__ constexpr uint32_t dwr_slab_bytes() {          // [d half][pred region | enc region], 1 KB aligned (SW128)
  return 2u * (bwd_pred_region<P>() + 1024u);
}

// SPLIT = true (precision bf16x3): dW^T = z_hi^T G_hi + z_hi^T G_lo + z_lo^T G_hi.  Per 64-row k-block the G loader
// brings a G_hi and a G_lo stage (from the two spills), the producers write a z_hi and a z_lo A stage (z in fp32 from
// the fp32 rows, read straight from global memory: no slab ring, warp 3 idles).
// ACT: the joint activation of the recomputed z (ACT_TANH / ACT_RELU / ACT_GELU).
template <int P, int TT, bool SPLIT, int ACT = ACT_TANH>
__device__ __forceinline__ void dw_gemm_rz_body(const CUtensorMap& tmap_e, const CUtensorMap& tmap_p,
                                                const __nv_bfloat16* __restrict__ gr, const __nv_bfloat16* __restrict__ gr_lo,
                                                const float* __restrict__ enc, const float* __restrict__ pred,
                                                const int4* __restrict__ tile_rows, const int* __restrict__ ntiles_ptr,
                                                float* __restrict__ partials, int D, int Vp, int KBG, int KS) {
  static_assert(TT <= 8, "enc region is one 1 KB swizzle atom");
  constexpr int NS = SPLIT ? DW_STAGES_X3 : DW_STAGES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = smem_u32(smem_raw);
  const uint32_t al = (base + 1023u) & ~1023u;
  const uint32_t b_bytes = (uint32_t)KBG * 8192u;          // one 64-row half of a G tile: [KBG][64 rows][64 v]
  const uint32_t slab = al + NS * b_bytes;                 // DWR_S_STAGES slabs of enc / pred rows (one per row tile)
  const uint32_t bar = slab + (SPLIT ? 0u : DWR_S_STAGES * dwr_slab_bytes<P>());
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem_raw + (bar + (NS + 6) * 16 + 48 - base));
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int mb = blockIdx.x, ks = blockIdx.y;
  const int kblocks = (*ntiles_ptr) * 2;                   // 64-row k-blocks written by kernel 1
  const int kb_begin = (int)(((long)kblocks * ks) / KS), kb_end = (int)(((long)kblocks * (ks + 1)) / KS);
  const int rt_begin = kb_begin >> 1, rt_end = (kb_end + 1) >> 1;
  auto full = [&](int i) { return bar + i * 16; };
  auto empty = [&](int i) { return bar + i * 16 + 8; };
  auto a_full = [&](int i) { return bar + NS * 16 + i * 16; };
  auto a_empty = [&](int i) { return bar + NS * 16 + i * 16 + 8; };
  auto s_full = [&](int i) { return bar + (NS + 3) * 16 + i * 16; };
  auto s_empty = [&](int i) { return bar + (NS + 3) * 16 + i * 16 + 8; };
  const uint32_t done = bar + (NS + 6) * 16;

  if (warp == 0 && lane == 0) {
    if (!SPLIT) {                    // the split form gets placeholder tensor maps
      tma_prefetch_desc(&tmap_e);
      tma_prefetch_desc(&tmap_p);
    }
    for (int i = 0; i < NS; ++i) { mbar_init(full(i), 1); mbar_init(empty(i), 1); }
    for (int i = 0; i < DWR_A_STAGES; ++i) { mbar_init(a_full(i), 4 * DWR_ROW_PARTS); mbar_init(a_empty(i), 1); }
    for (int i = 0; i < DWR_S_STAGES; ++i) { mbar_init(s_full(i), 1); mbar_init(s_empty(i), 4 * DWR_ROW_PARTS); }
    mbar_init(done, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_u32(tmem_ptr), TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ---- G loader: one 1-D bulk copy per stage
    Pipe sp;
    for (int kb = kb_begin; kb < kb_end; ++kb)
      for (int part = 0; part < (SPLIT ? 2 : 1); ++part) {     // bf16x3: G_hi, then G_lo
        mbar_wait(empty(sp.stage), sp.phase ^ 1u, 50);
        if (elect_one()) {
          mbar_arrive_expect_tx(full(sp.stage), b_bytes);
          bulk_load(al + sp.stage * b_bytes, (part ? gr_lo : gr) + (size_t)kb * KBG * 4096, b_bytes, full(sp.stage));
        }
        __syncwarp();
        sp.advance(NS);
      }
  } else if (warp == 3 && !SPLIT) {
    // ---- slab loader: the P pred rows and TT enc rows of each row tile, this CTA's 128 d as two 64-wide boxes
    Pipe ss;
    for (int rt = rt_begin; rt < rt_end; ++rt) {
      mbar_wait(s_empty(ss.stage), ss.phase ^ 1u, 55);
      if (elect_one()) {
        const int4 tr = __ldg(tile_rows + rt);             // {first enc row, first pred row, ..}
        const uint32_t st = slab + ss.stage * dwr_slab_bytes<P>();
        mbar_arrive_expect_tx(s_full(ss.stage), 2u * (uint32_t)(P + TT) * 128u);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint32_t sh = st + h * (bwd_pred_region<P>() + 1024u);
          tma_load_2d(sh, &tmap_p, s_full(ss.stage), mb * 128 + h * 64, tr.y);
          tma_load_2d(sh + bwd_pred_region<P>(), &tmap_e, s_full(ss.stage), mb * 128 + h * 64, tr.x);
        }
      }
      __syncwarp();
      ss.advance(DWR_S_STAGES);
    }
  } else if (warp == 1) {
    // ---- MMA issuer: D[128 d][Vp] += z^T (TMEM) . G (MN-major B, N split 256 + rest)
    Pipe sp, ap;
    const int N0 = min(256, Vp), N1 = Vp - N0;
    const uint32_t idesc0 = make_idesc_bf16_bmn(128, N0);
    const uint32_t idesc1 = make_idesc_bf16_bmn(128, N1 > 0 ? N1 : 16);
    const uint64_t b_desc0 = make_desc_mn_sw128(al, 8192u, 1024u);
    const uint32_t st_step = b_bytes >> 4;
    if constexpr (SPLIT) {
      for (int kb = kb_begin; kb < kb_end; ++kb) {
        Pipe sl = sp, al2 = ap;                              // the lo stages follow the hi stages
        sl.advance(NS);
        al2.advance(DWR_A_STAGES);
        mbar_wait(a_full(ap.stage), ap.phase, 53);
        mbar_wait(a_full(al2.stage), al2.phase, 53);
        mbar_wait(full(sp.stage), sp.phase, 51);
        mbar_wait(full(sl.stage), sl.phase, 51);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a = tmem_base + DWR_ACC_COLS + ap.stage * 32, a2 = tmem_base + DWR_ACC_COLS + al2.stage * 32;
          const uint64_t bh = b_desc0 + (uint64_t)(sp.stage * st_step), bl = b_desc0 + (uint64_t)(sl.stage * st_step);
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4) {
            const uint32_t acc = (kb > kb_begin || k4 > 0) ? 1u : 0u;
            umma_bf16_ts(tmem_base, a + 8 * k4, bh + 128 * k4, idesc0, acc);                       // z_hi G_hi
            if (N1 > 0) umma_bf16_ts(tmem_base + 256, a + 8 * k4, bh + 2048 + 128 * k4, idesc1, acc);
            umma_bf16_ts(tmem_base, a + 8 * k4, bl + 128 * k4, idesc0, 1u);                         // z_hi G_lo
            if (N1 > 0) umma_bf16_ts(tmem_base + 256, a + 8 * k4, bl + 2048 + 128 * k4, idesc1, 1u);
            umma_bf16_ts(tmem_base, a2 + 8 * k4, bh + 128 * k4, idesc0, 1u);                        // z_lo G_hi
            if (N1 > 0) umma_bf16_ts(tmem_base + 256, a2 + 8 * k4, bh + 2048 + 128 * k4, idesc1, 1u);
          }
          umma_commit(empty(sp.stage));
          umma_commit(empty(sl.stage));
          umma_commit(a_empty(ap.stage));
          umma_commit(a_empty(al2.stage));
        }
        __syncwarp();
        sp.advance(NS); sp.advance(NS);
        ap.advance(DWR_A_STAGES); ap.advance(DWR_A_STAGES);
      }
    } else
    for (int kb = kb_begin; kb < kb_end; ++kb) {
      mbar_wait(a_full(ap.stage), ap.phase, 53);
      mbar_wait(full(sp.stage), sp.phase, 51);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t a = tmem_base + DWR_ACC_COLS + ap.stage * 32;
        const uint64_t bd = b_desc0 + (uint64_t)(sp.stage * st_step);
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) {
          const uint32_t acc = (kb > kb_begin || k4 > 0) ? 1u : 0u;
          umma_bf16_ts(tmem_base, a + 8 * k4, bd + 128 * k4, idesc0, acc);
          if (N1 > 0) umma_bf16_ts(tmem_base + 256, a + 8 * k4, bd + 2048 + 128 * k4, idesc1, acc);
        }
        umma_commit(empty(sp.stage));
        umma_commit(a_empty(ap.stage));
      }
      __syncwarp();
      sp.advance(DW_STAGES);
      ap.advance(DWR_A_STAGES);
    }
    if (elect_one()) umma_commit(done);
    __syncwarp();
  } else if (warp >= 4) {
    // ---- producers: warp = (d quarter q, row part rh of the 64-row stage); lane = d
    const int q = warp & 3, rh = (warp - 4) >> 2;          // rh < DWR_ROW_PARTS (2 or 4)
    const int dl = q * 32 + lane;                          // d within the CTA's 128
    const int d = mb * 128 + dl;
    const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16);
    // slab addressing: box half dl>>6, 16-byte chunk ((dl&63)>>3) ^ (row & 7), element dl&7
    const uint32_t s_off = (uint32_t)(dl >> 6) * (bwd_pred_region<P>() + 1024u) + (uint32_t)(dl & 7) * 2u;
    const uint32_t s_chunk = (uint32_t)((dl & 63) >> 3);
    Pipe ap, ss;
    if constexpr (SPLIT) {
      for (int rt = rt_begin; rt < rt_end; ++rt) {
        float e[TT], pr[P];
        {
          const int4 tr = __ldg(tile_rows + rt);           // {first enc row, first pred row, rows readable past them}
#pragma unroll
          for (int i = 0; i < P; ++i) pr[i] = __ldg(pred + (size_t)(tr.y + min(i, tr.w)) * D + d);
#pragma unroll
          for (int i = 0; i < TT; ++i) e[i] = __ldg(enc + (size_t)(tr.x + min(i, tr.z)) * D + d);
        }
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int kb = rt * 2 + hh;
          if (kb < kb_begin || kb >= kb_end) continue;
          constexpr int NP = 32 / DWR_ROW_PARTS;
          uint32_t wh[NP], wl[NP];
          auto rows = [&](auto HH) {
            constexpr int R = decltype(HH)::value * 64;
            if (rh == 0) dwr_rows_x3<P, TT, R, NP, ACT>(e, pr, wh, wl);
            else if (rh == 1) dwr_rows_x3<P, TT, R + 2 * NP, NP, ACT>(e, pr, wh, wl);
            else if (rh == 2) dwr_rows_x3<P, TT, R + 4 * NP, NP, ACT>(e, pr, wh, wl);
            else dwr_rows_x3<P, TT, R + 6 * NP, NP, ACT>(e, pr, wh, wl);
          };
          if (hh == 0) rows(std::integral_constant<int, 0>{}); else rows(std::integral_constant<int, 1>{});
          Pipe al2 = ap;
          al2.advance(DWR_A_STAGES);
          mbar_wait(a_empty(ap.stage), ap.phase ^ 1u, 54);
          mbar_wait(a_empty(al2.stage), al2.phase ^ 1u, 54);
          tc_fence_after();
          if constexpr (NP == 16) {
            tmem_st16(tq + (uint32_t)(DWR_ACC_COLS + ap.stage * 32 + rh * NP), wh);
            tmem_st16(tq + (uint32_t)(DWR_ACC_COLS + al2.stage * 32 + rh * NP), wl);
          } else {
            tmem_st8(tq + (uint32_t)(DWR_ACC_COLS + ap.stage * 32 + rh * NP), wh);
            tmem_st8(tq + (uint32_t)(DWR_ACC_COLS + al2.stage * 32 + rh * NP), wl);
          }
          tmem_st_wait();
          tc_fence_before();
          warp_arrive(a_full(ap.stage));
          warp_arrive(a_full(al2.stage));
          ap.advance(DWR_A_STAGES);
          ap.advance(DWR_A_STAGES);
        }
      }
    } else
    for (int rt = rt_begin; rt < rt_end; ++rt) {
      uint32_t e[TT], pr[P];
      mbar_wait(s_full(ss.stage), ss.phase, 56);
      {
        const uint32_t st = slab + ss.stage * dwr_slab_bytes<P>() + s_off;
#pragma unroll
        for (int i = 0; i < P; ++i) {
          unsigned short v;
          asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(st + i * 128 + ((s_chunk ^ (uint32_t)(i & 7)) << 4)));
          pr[i] = v;
        }
#pragma unroll
        for (int i = 0; i < TT; ++i) {
          unsigned short v;
          asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(st + bwd_pred_region<P>() + i * 128 + ((s_chunk ^ (uint32_t)(i & 7)) << 4)));
          e[i] = v;
        }
      }
      warp_arrive(s_empty(ss.stage));
      ss.advance(DWR_S_STAGES);
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int kb = rt * 2 + hh;
        if (kb < kb_begin || kb >= kb_end) continue;
        constexpr int NP = 32 / DWR_ROW_PARTS;           // row pairs (= TMEM columns) per producer warp and stage
        uint32_t w[NP];
        // rows hh*64 + rh*2*NP ..: one instantiation per (hh, rh) so that every (tloc, ul) is a compile-time constant
        auto rows = [&](auto HH) {
          constexpr int R = decltype(HH)::value * 64;
          if (rh == 0) dwr_rows<P, TT, R, NP, ACT>(e, pr, w);
          else if (rh == 1) dwr_rows<P, TT, R + 2 * NP, NP, ACT>(e, pr, w);
          else if (rh == 2) dwr_rows<P, TT, R + 4 * NP, NP, ACT>(e, pr, w);
          else dwr_rows<P, TT, R + 6 * NP, NP, ACT>(e, pr, w);
        };
        if (hh == 0) rows(std::integral_constant<int, 0>{}); else rows(std::integral_constant<int, 1>{});
        mbar_wait(a_empty(ap.stage), ap.phase ^ 1u, 54);
        tc_fence_after();
        if constexpr (NP == 16) tmem_st16(tq + (uint32_t)(DWR_ACC_COLS + ap.stage * 32 + rh * NP), w);
        else tmem_st8(tq + (uint32_t)(DWR_ACC_COLS + ap.stage * 32 + rh * NP), w);
        tmem_st_wait();
        tc_fence_before();
        warp_arrive(a_full(ap.stage));
        ap.advance(DWR_A_STAGES);
      }
    }
    // ---- epilogue (warps 4-7): accumulators -> split-K partials
    if (rh == 0) {
      float* out = partials + ((size_t)ks * D + d) * Vp;
      if (kb_end > kb_begin) {
        mbar_wait(done, 0, 52);
        tc_fence_after();
        for (int c0 = 0; c0 < Vp; c0 += 32) {
          float v[32];
          tmem_ld32(tq + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(out + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
      } else {
        for (int c0 = 0; c0 < Vp; c0 += 4) *reinterpret_cast<float4*>(out + c0) = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

template <int P, int TT>
__global__ void __launch_bounds__(DWR_THREADS, 1)
dw_gemm_rz_kernel(const __grid_constant__ CUtensorMap tmap_e, const __grid_constant__ CUtensorMap tmap_p,
                  const __nv_bfloat16* __restrict__ gr, const int4* __restrict__ tile_rows,
                  const int* __restrict__ ntiles_ptr, float* __restrict__ partials, int D, int Vp, int KBG, int KS) {
  dw_gemm_rz_body<P, TT, false>(tmap_e, tmap_p, gr, nullptr, nullptr, nullptr, tile_rows, ntiles_ptr, partials, D, Vp, KBG, KS);
}
// precision bf16x3 (the tensor maps are unused)
template <int P, int TT>
__global__ void __launch_bounds__(DWR_THREADS, 1)
dw_gemm_rz_x3_kernel(const __grid_constant__ CUtensorMap tmap_e, const __grid_constant__ CUtensorMap tmap_p,
                     const __nv_bfloat16* __restrict__ gr, const __nv_bfloat16* __restrict__ gr_lo,
                     const float* __restrict__ enc, const float* __restrict__ pred, const int4* __restrict__ tile_rows,
                     const int* __restrict__ ntiles_ptr, float* __restrict__ partials, int D, int Vp, int KBG, int KS) {
  dw_gemm_rz_body<P, TT, true>(tmap_e, tmap_p, gr, gr_lo, enc, pred, tile_rows, ntiles_ptr, partials, D, Vp, KBG, KS);
}
// relu / gelu joints, named apart for profiler traces
#define CTCVR_DWR_ACT(name, act)                                                                                   \
  template <int P, int TT>                                                                                          \
  __global__ void __launch_bounds__(DWR_THREADS, 1)                                                                 \
  name(const __grid_constant__ CUtensorMap tmap_e, const __grid_constant__ CUtensorMap tmap_p,                      \
       const __nv_bfloat16* __restrict__ gr, const int4* __restrict__ tile_rows, const int* __restrict__ ntiles_ptr, \
       float* __restrict__ partials, int D, int Vp, int KBG, int KS) {                                              \
    dw_gemm_rz_body<P, TT, false, act>(tmap_e, tmap_p, gr, nullptr, nullptr, nullptr, tile_rows, ntiles_ptr,        \
                                       partials, D, Vp, KBG, KS);                                                   \
  }
CTCVR_DWR_ACT(dw_gemm_rz_relu_kernel, ACT_RELU)
CTCVR_DWR_ACT(dw_gemm_rz_gelu_kernel, ACT_GELU)
#undef CTCVR_DWR_ACT
#define CTCVR_DWR_X3_ACT(name, act)                                                                                \
  template <int P, int TT>                                                                                          \
  __global__ void __launch_bounds__(DWR_THREADS, 1)                                                                 \
  name(const __grid_constant__ CUtensorMap tmap_e, const __grid_constant__ CUtensorMap tmap_p,                      \
       const __nv_bfloat16* __restrict__ gr, const __nv_bfloat16* __restrict__ gr_lo,                               \
       const float* __restrict__ enc, const float* __restrict__ pred, const int4* __restrict__ tile_rows,           \
       const int* __restrict__ ntiles_ptr, float* __restrict__ partials, int D, int Vp, int KBG, int KS) {          \
    dw_gemm_rz_body<P, TT, true, act>(tmap_e, tmap_p, gr, gr_lo, enc, pred, tile_rows, ntiles_ptr, partials, D, Vp, \
                                      KBG, KS);                                                                     \
  }
CTCVR_DWR_X3_ACT(dw_gemm_rz_x3_relu_kernel, ACT_RELU)
CTCVR_DWR_X3_ACT(dw_gemm_rz_x3_gelu_kernel, ACT_GELU)
#undef CTCVR_DWR_X3_ACT

// dW GEMM shared memory: G stages, slab ring (bf16 only), barriers
template <int P>
static size_t dwr_smem_bytes(int KBG, bool split) {
  return 1024 + (size_t)(split ? DW_STAGES_X3 : DW_STAGES) * ((size_t)KBG * 8192) + (split ? 0 : DWR_S_STAGES * dwr_slab_bytes<P>()) + 256;
}

// d_w[v][d] = sum_ks partials[ks][d][v].  Block = 8 d x 32 v (warp = d row, lanes = consecutive v: coalesced
// reads of every split); the 32 x 8 result is transposed through shared memory for the [V][D] store.
__global__ void __launch_bounds__(256) reduce_dw_kernel(const float* __restrict__ partials, float* __restrict__ d_w,
                                                        int D, int V, int Vp, int KS) {
  __shared__ float tile[8][33];
  const int d0 = blockIdx.x * 8, v0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int d = d0 + ty, v = v0 + tx;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  if (d < D && v < Vp) {
    const float* src = partials + (size_t)d * Vp + v;
    const size_t step = (size_t)D * Vp;
    int k = 0;
    for (; k + 4 <= KS; k += 4) {
      s0 += __ldg(src + (size_t)k * step);
      s1 += __ldg(src + (size_t)(k + 1) * step);
      s2 += __ldg(src + (size_t)(k + 2) * step);
      s3 += __ldg(src + (size_t)(k + 3) * step);
    }
    for (; k < KS; ++k) s0 += __ldg(src + (size_t)k * step);
  }
  tile[ty][tx] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  // thread (vi = tid / 8, di = tid % 8): 8 consecutive d of one v -> 32-byte segments
  const int vi = threadIdx.x >> 3, di = threadIdx.x & 7;
  if (v0 + vi < V && d0 + di < D) d_w[(size_t)(v0 + vi) * D + d0 + di] = tile[di][vi];
}

// =================================================================================================
// Helper kernels: weight conversion, tile tables
// =================================================================================================
// Tile tables.  One CTA per utterance: the CTA sums the tile counts of the utterances before it (block reduction),
// then its threads write the utterance's entries in parallel; the last CTA also writes the total.
template <class Count>
__device__ __forceinline__ int block_prefix(int mine_upto, Count count) {
  __shared__ int s_part[32];
  int acc = 0;
  for (int i = threadIdx.x; i < mine_upto; i += blockDim.x) acc += count(i);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  int tot = 0;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += s_part[i];
  __syncthreads();
  return tot;
}

// Backward tiles: TT frames x P label columns (geom = P | TT << 8 | even << 16), ordered (b, u-split, frame block) so
// that one CTA sweeps consecutive frame blocks of the same (b, u-split).  `even` pads every sweep to an even number of
// frame blocks (the CTA-pair kernel processes tiles 2i, 2i+1 of one sweep together; a padding tile lies beyond T_b).
// Entry = {b, u-split, frame block, tile index}.
__device__ void build_tiles_block(int b, const int32_t* __restrict__ t_len, const int32_t* __restrict__ u_len, int B, int T,
                                  int U1, int geom, int4* __restrict__ tiles, int4* __restrict__ tile_rows,
                                  int* __restrict__ ntiles, int max_tiles) {
  const int P = geom & 0xff, TT = (geom >> 8) & 0xff, even = (geom >> 16) & 1;
  auto ntb_of = [&](int Tb) { const int n = (Tb + TT - 1) / TT; return even ? ((n + 1) & ~1) : n; };
  auto count = [&](int i) {
    const int Tb = max(min(t_len[i], T), 0), W = max(min(u_len[i], U1 - 1), 0) + 1;
    return Tb > 0 ? ((W + P - 1) / P) * ntb_of(Tb) : 0;
  };
  const int off = block_prefix(b, count);
  const int Tb = max(min(t_len[b], T), 0);
  const int n = count(b);
  const int NTB = ntb_of(Tb);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int s = i / NTB, tb = i - s * NTB;
    if (off + i < max_tiles) {
      tiles[off + i] = make_int4(b, s, tb, off + i);
      if (tile_rows) {
        // first enc / pred row of the tile and how many rows may be read past them (kernel 2 recomputes z from these)
        const int W = max(min(u_len[b], U1 - 1), 0) + 1, S = (W + P - 1) / P, us = (W + S - 1) / S;
        const int t0 = tb * TT, ub = s * us;
        tile_rows[off + i] = make_int4(b * T + min(t0, T - 1), b * U1 + min(ub, U1 - 1), max(T - 1 - t0, 0), max(U1 - 1 - ub, 0));
      }
    }
  }
  if (b == B - 1 && threadIdx.x == 0) *ntiles = min(off + n, max_tiles);
}

// fp32 -> bf16 copies of the activations (n4 float4 groups each); the bf16 path rounds enc_proj / pred_proj
// to bf16 (under autocast they already are bf16 values, so this is lossless there).
__device__ void to_bf16_part(long first_i, long stride, const float4* __restrict__ a, uint2* __restrict__ ab, long na4,
                             const float4* __restrict__ b, uint2* __restrict__ bb, long nb4) {
  for (long i = first_i; i < na4 + nb4; i += stride) {
    const bool first = i < na4;
    const float4 v = first ? __ldg(a + i) : __ldg(b + (i - na4));
    const uint2 o = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
    if (first) ab[i] = o; else bb[i - na4] = o;
  }
}

// Tiled, pre-swizzled bf16 copies of W_out for 1-D bulk loads (one contiguous block per smem stage):
//   w_t  [KB][2][NH][64]   stage (kb,h): rows v' = v - h*NH, k' = k - 64 kb; chunk (k'>>3) stored at (k'>>3) ^ (v'&7)
//   wt_t [MB][KBG][128][64] stage (mb,kb): rows d' = d - 128 mb, v' = v - 64 kb; chunk (v'>>3) at (v'>>3) ^ (d'&7)
// plus bias_pad / bias_l2.  One thread per (v, d) of the zero-padded [KBG*64][D] weight.
// SPLIT (bf16x3): x = hi + lo with hi = bf16(x), lo = bf16(x - hi); each stage block is followed by its lo twin:
//   w_t  [KB][hi, lo][2][NH][64]        wt_t [MB][KBG][hi, lo][128][64]
template <bool SPLIT>
__device__ void prep_weights3_part(int i, const float* __restrict__ w, const float* __restrict__ bias,
                                   __nv_bfloat16* __restrict__ w_t, __nv_bfloat16* __restrict__ wt_t,
                                   float* __restrict__ bias_pad, float* __restrict__ bias_l2, int V, int Vp, int D) {
  const int KBG = (Vp + 63) / 64, NH = Vp / 2;
  if (SPLIT && i < KBG * 64 * D) {
    const int v = i / D, d = i - v * D;
    const float xf = (v < V) ? w[(size_t)v * D + d] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16(xf), lo = __float2bfloat16(xf - __bfloat162float(hi));
    if (v < Vp) {
      const int h = v / NH, vl = v - h * NH, kb = d >> 6, kl = d & 63;
      const size_t o = (size_t)vl * 64 + (((kl >> 3) ^ (vl & 7)) << 3) + (kl & 7);
      w_t[(size_t)(kb * 4 + h) * NH * 64 + o] = hi;
      w_t[(size_t)(kb * 4 + 2 + h) * NH * 64 + o] = lo;
    }
    if (wt_t) {
      const int mb = d >> 7, dl = d & 127, kb = v >> 6, vl = v & 63;
      const size_t o = (size_t)(mb * KBG + kb) * 16384 + dl * 64 + (((vl >> 3) ^ (dl & 7)) << 3) + (vl & 7);
      wt_t[o] = hi;
      wt_t[o + 8192] = lo;
    }
  } else if (!SPLIT && i < KBG * 64 * D) {
    const int v = i / D, d = i - v * D;
    const __nv_bfloat16 x = __float2bfloat16((v < V) ? w[(size_t)v * D + d] : 0.f);
    if (v < Vp) {
      const int h = v / NH, vl = v - h * NH, kb = d >> 6, kl = d & 63;
      w_t[(size_t)(kb * 2 + h) * NH * 64 + vl * 64 + (((kl >> 3) ^ (vl & 7)) << 3) + (kl & 7)] = x;
    }
    if (wt_t) {
      const int mb = d >> 7, dl = d & 127, kb = v >> 6, vl = v & 63;
      wt_t[(size_t)(mb * KBG + kb) * 8192 + dl * 64 + (((vl >> 3) ^ (dl & 7)) << 3) + (vl & 7)] = x;
    }
  }
  if (i < Vp) {
    if (bias_pad) bias_pad[i] = (i < V) ? bias[i] : kNegInf;
    if (bias_l2) bias_l2[i] = (i < V) ? bias[i] * LOG2E : kNegInf;
  }
}

// Forward tile table (see joint_tc_fwd.cuh): entry = {b, u0, t0, nu}.
__device__ void build_tiles_fwd_block(int b, const int32_t* __restrict__ t_len, const int32_t* __restrict__ u_len, int B,
                                      int T, int U1, int4* __restrict__ tiles, int* __restrict__ ntiles,
                                      int max_tiles, int pair) {
  const int off = block_prefix(b, [&](int i) { return fwd_tiles_of(max(min(t_len[i], T), 0), max(min(u_len[i], U1 - 1), 0) + 1, pair); });
  const int Tb = max(min(t_len[b], T), 0), W = max(min(u_len[b], U1 - 1), 0) + 1;
  const int n = fwd_tiles_of(Tb, W, pair);
  const int nb32 = (Tb + 31) >> 5, n4 = (W >> 2) * nb32;
  const int n2 = (W & 2) ? ((Tb + 63) >> 6) : 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    int4 e;
    if (i < n4) { const int g = i / nb32; e = make_int4(b, 4 * g, 32 * (i - g * nb32), 4); }
    else if (i < n4 + n2) e = make_int4(b, (W >> 2) * 4, 64 * (i - n4), 2);
    else e = make_int4(b, W - 1, (pair ? 64 : 128) * (i - n4 - n2), 1);
    if (off + i < max_tiles) tiles[off + i] = e;
  }
  if (b == B - 1 && threadIdx.x == 0) *ntiles = min(off + n, max_tiles);
}

// One launch for everything the joint kernels need prepared: tiled weights (blocks [0, nW)), the tile table (blocks
// [nW, nW + B): geom = 0 builds the forward table), and grid-stride zero fills / fp32 -> bf16 activation copies on the
// remaining blocks.  Graph nodes are not free (~3 us each): this replaces up to five of them.
struct PrepArgs {
  const float* w; const float* bias; __nv_bfloat16* w_t; __nv_bfloat16* wt_t; float* bias_pad; float* bias_l2;
  int V, Vp, D, nW;
  const int32_t* t_len; const int32_t* u_len; int B, T, U1, geom, max_tiles, fwd_pair;
  int4* tiles; int4* tile_rows; int* ntiles;
  float* zero0; long n0; float* zero1; long n1;
  const float4* a; uint2* ab; long na4; const float4* b4; uint2* bb; long nb4;
};
template <bool SPLIT>
__global__ void __launch_bounds__(256) prep_kernel(const PrepArgs q) {
  const int blk = blockIdx.x;
  if (blk < q.nW) {
    prep_weights3_part<SPLIT>(blk * 256 + threadIdx.x, q.w, q.bias, q.w_t, q.wt_t, q.bias_pad, q.bias_l2, q.V, q.Vp, q.D);
  } else if (blk < q.nW + q.B) {
    if (q.geom) build_tiles_block(blk - q.nW, q.t_len, q.u_len, q.B, q.T, q.U1, q.geom, q.tiles, q.tile_rows, q.ntiles, q.max_tiles);
    else build_tiles_fwd_block(blk - q.nW, q.t_len, q.u_len, q.B, q.T, q.U1, q.tiles, q.ntiles, q.max_tiles, q.fwd_pair);
  } else {
    const long nb = gridDim.x - q.nW - q.B, first = (long)(blk - q.nW - q.B) * 256 + threadIdx.x, stride = nb * 256;
    for (long i = first; i < q.n0; i += stride) q.zero0[i] = 0.f;
    for (long i = first; i < q.n1; i += stride) q.zero1[i] = 0.f;
    if (q.na4 + q.nb4 > 0) to_bf16_part(first, stride, q.a, q.ab, q.na4, q.b4, q.bb, q.nb4);
  }
}
// Vocabulary tiles: the same launch with the weights of nvt tiles of Vp = Vc columns each (q.V = the full vocabulary,
// q.nW = weight blocks per tile).  Tile c holds rows [c Vc, c Vc + Vc) of W_out; its w_t / wt_t / bias_l2 follow those of
// tile c - 1 without a gap.
template <bool SPLIT>
__global__ void __launch_bounds__(256) prep_vt_kernel(const PrepArgs q, int nvt) {
  const int blk = blockIdx.x;
  if (blk < q.nW * nvt) {
    const int c = blk / q.nW, v0 = c * q.Vp;
    const size_t ws = (size_t)q.Vp * q.D * (SPLIT ? 2 : 1), wts = (size_t)((q.Vp + 63) / 64) * 64 * q.D * (SPLIT ? 2 : 1);
    prep_weights3_part<SPLIT>((blk - c * q.nW) * 256 + threadIdx.x, q.w + (size_t)v0 * q.D, q.bias + v0, q.w_t + c * ws,
                              q.wt_t ? q.wt_t + c * wts : nullptr, nullptr, q.bias_l2 + (size_t)c * q.Vp,
                              min(q.V - v0, q.Vp), q.Vp, q.D);
  } else {                                // the blocks behind the weights: as in prep_kernel
    const int nW = q.nW * nvt;
    if (blk < nW + q.B) {
      if (q.geom) build_tiles_block(blk - nW, q.t_len, q.u_len, q.B, q.T, q.U1, q.geom, q.tiles, q.tile_rows, q.ntiles, q.max_tiles);
      else build_tiles_fwd_block(blk - nW, q.t_len, q.u_len, q.B, q.T, q.U1, q.tiles, q.ntiles, q.max_tiles, q.fwd_pair);
    } else {
      const long nb = gridDim.x - nW - q.B, first = (long)(blk - nW - q.B) * 256 + threadIdx.x, stride = nb * 256;
      for (long i = first; i < q.n0; i += stride) q.zero0[i] = 0.f;
      for (long i = first; i < q.n1; i += stride) q.zero1[i] = 0.f;
      if (q.na4 + q.nb4 > 0) to_bf16_part(first, stride, q.a, q.ab, q.na4, q.b4, q.bb, q.nb4);
    }
  }
}

// Vocabulary tiles, after the last tile's forward: lp_blank / lp_label hold raw logit + bias, lse the merged log-sum-exp
// of the whole vocabulary.  One thread per lattice cell; the cells the untiled forward writes, written the same way.
__global__ void __launch_bounds__(256) vt_finalize_kernel(const float* __restrict__ lse, float* __restrict__ lp_blank,
                                                          float* __restrict__ lp_label, const int32_t* __restrict__ t_len,
                                                          const int32_t* __restrict__ u_len, int B, int T, int U1) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long)B * T * U1) return;
  const int b = (int)(i / ((long)T * U1)), r = (int)(i - (long)b * T * U1), t = r / U1, u = r - t * U1;
  const int Tb = max(min(t_len[b], T), 0), Ub = max(min(u_len[b], U1 - 1), 0);
  if (t >= Tb || u > Ub) return;
  const float l = lse[i];
  lp_blank[i] -= l;
  lp_label[i] = (u < Ub) ? lp_label[i] - l : kNegInf;
}

int make_tmap_bf16_2d(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t pitch_elems,
                      uint32_t box_rows, bool swizzle) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qr;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qr);
    if (e != cudaSuccess || qr != cudaDriverEntryPointSuccess || !sym) {
      set_error("cuTensorMapEncodeTiled is not available from the driver (%s)", cudaGetErrorString(e));
      return 1;
    }
    fn = reinterpret_cast<EncodeTiledFn>(sym);
  }
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {pitch_elems * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%llu cols=%llu box_rows=%u)", (int)r,
              (unsigned long long)rows, (unsigned long long)cols, box_rows);
    return 1;
  }
  return 0;
}

// Mapped pinned host word written by a kernel whose bounded mbarrier wait timed out (a protocol bug or a wedged
// copy): read WITHOUT a host synchronisation at the next tensor-core entry-point call, which then fails loudly.
static unsigned int* tc_error_host_word(unsigned int** dev_ptr) {
  static unsigned int* h = nullptr;
  static unsigned int* d = nullptr;
  if (!h) {
    if (cudaHostAlloc(reinterpret_cast<void**>(&h), sizeof(unsigned int), cudaHostAllocMapped) != cudaSuccess) { h = nullptr; cudaGetLastError(); }
    else { *h = 0u; if (cudaHostGetDevicePointer(reinterpret_cast<void**>(&d), h, 0) != cudaSuccess) { d = nullptr; cudaGetLastError(); } }
  }
  if (dev_ptr) *dev_ptr = d;
  return h;
}
static int check_tc_error(const char* where) {
  unsigned int* h = tc_error_host_word(nullptr);
  if (h && *reinterpret_cast<volatile unsigned int*>(h) != 0u) {
    const unsigned int code = *h;
    *h = 0u;
    set_error("%s: an earlier tcgen05 kernel gave up on a bounded mbarrier wait (flag 0x%08x: site %u, CTA %u); "
              "the results of that call are invalid", where, code, (code >> 16) & 0x7fffu, code & 0xffffu);
    return 1;
  }
  return 0;
}

}  // namespace tc

// =================================================================================================
// Host entry points
// =================================================================================================
using namespace tc;

static long long* g_prof_buf = nullptr;
// dev switch (ctcvr_debug_set_mode(0)): run the experimental CTA-pair forward kernel (joint_tc_fwd_pair.cuh).  It is
// correct (tools/fwd_pair_check.py) but at 200 us against 148 us it is not the default: see DESIGN.md section 5.
static int g_force_single_cta = 1;
static int g_bwd_single_cta = 0;        // ctcvr_debug_set_mode(2): single-CTA backward kernel (A/B timing against the pair kernel)
static int pad_v(int V) { return (V + 31) / 32 * 32; }
static int max_tiles_flat(int B, int T, int U1) { return B * (int)(((long)T * U1 + BM - 1) / BM); }
// Backward tile geometry: P label columns x TT frames.  Pick the variant with fewer tile rows for this (T, U1);
// `even` (pad the frame blocks of an utterance to an even count) is kept in the tile builder but unused.
struct RectGeom { int P, TT, even; };
static RectGeom pick_rect_geom(int T, int U1) {
  auto tiles = [&](int P, int TT) { return (long)((U1 + P - 1) / P) * ((T + TT - 1) / TT); };
  return tiles(21, 6) < tiles(16, 8) ? RectGeom{21, 6, 0} : RectGeom{16, 8, 0};
}
static int max_tiles_rect(int B, int T, int U1) {           // upper bound over both geometries and the even padding
  const long a = (long)((U1 + 15) / 16) * ((((T + 7) / 8) + 1) & ~1), b = (long)((U1 + 20) / 21) * ((T + 5) / 6);
  return B * (int)(a > b ? a : b);
}

// the forward keeps its A stages in the TMEM columns behind the accumulators: Vp + 96 <= 512
bool joint_tc_supported(int U1, int D, int V) { return D % 64 == 0 && D >= 64 && D <= 1024 && pad_v(V) <= 416 && U1 <= 128; }
// the predicate of the bf16 path, both directions (the backward tiles D in 128-lane blocks of dZ^T, at most four)
bool joint_tc_bwd_supported(int U1, int D, int V) { return joint_tc_supported(U1, D, V) && D % 128 == 0 && D <= 512; }

// Vocabulary tiles (ctcvr_joint_rnnt_*_vt): n = ceil(pad32(V) / 416) tiles of Vc = pad32(ceil(V / n)) columns; tile c
// covers [c Vc, min(V, c Vc + Vc)).  Every tile is a vocabulary the untiled kernels take (Vc <= 416), and the last one
// is non-empty for every V up to the cap.
constexpr int VT_MAX_V = 32768;
struct VocabTiles { int n, Vc; };
static VocabTiles vocab_tiles(int V) {
  const int n = cdiv(pad_v(V), 416);
  return {n, pad_v(cdiv(V, n))};
}
bool joint_tc_vt_supported(int U1, int D, int V) {
  return D % 128 == 0 && D >= 128 && D <= 512 && U1 >= 1 && U1 <= 128 && V >= 1 && V <= VT_MAX_V;
}

static int max_tiles_fwd2(int B, int T, int U1) {
  return B * ((U1 >> 2) * ((T + 31) / 32) + (T + 63) / 64 + (T + 63) / 64);
}

struct FwdWs {
  __nv_bfloat16 *wb, *eb, *pb;
  float *bias_pad, *bias_l2;
  int4* tiles;
  int* ntiles;
  size_t bytes;
};
// split (bf16x3): hi and lo copies of W_out; the fp32 activations are read in place (no bf16 copies)
// nvt > 1: vocabulary tiles of V = Vc columns each, their weights back to back
static FwdWs carve_fwd_ws(void* ws, int B, int T, int U1, int D, int V, bool split = false, int nvt = 1) {
  int Vp = pad_v(V);
  uint8_t* p = reinterpret_cast<uint8_t*>(ws);
  size_t off = 0;
  FwdWs w;
  auto take = [&](size_t n) { void* r = p + off; off = align_up(off + n, 1024); return r; };
  w.wb = reinterpret_cast<__nv_bfloat16*>(take((size_t)nvt * Vp * D * 2 * (split ? 2 : 1)));
  w.eb = split ? nullptr : reinterpret_cast<__nv_bfloat16*>(take((size_t)B * T * D * 2));
  w.pb = split ? nullptr : reinterpret_cast<__nv_bfloat16*>(take((size_t)B * U1 * D * 2));
  w.bias_pad = reinterpret_cast<float*>(take((size_t)Vp * 4));
  w.bias_l2 = reinterpret_cast<float*>(take((size_t)nvt * Vp * 4));
  const int mt = max_tiles_flat(B, T, U1) > max_tiles_fwd2(B, T, U1) ? max_tiles_flat(B, T, U1) : max_tiles_fwd2(B, T, U1);
  w.tiles = reinterpret_cast<int4*>(take((size_t)mt * 16));
  w.ntiles = reinterpret_cast<int*>(take(4));
  w.bytes = off;
  return w;
}

size_t joint_fwd_tc_ws_bytes(int B, int T, int U1, int D, int V, int split) {
  if (!joint_tc_bwd_supported(U1, D, V)) return 256;      // the call itself fails with the reason
  return carve_fwd_ws(nullptr, B, T, U1, D, V, split != 0).bytes;
}

static int sm_count() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

int joint_fwd_f32(const float*, const float*, const float*, const float*, const int32_t*, const int32_t*,
                  const int32_t*, float*, float*, float*, int, int, int, int, int, int, cudaStream_t);

// the kernel of a family for the joint activation act (ACT_TANH / ACT_RELU / ACT_GELU)
template <class K>
static K pick_act(int act, K tanh_k, K relu_k, K gelu_k) { return act == ACT_RELU ? relu_k : act == ACT_GELU ? gelu_k : tanh_k; }

// the fields of FwdParams every single-CTA forward launch shares
static FwdParams fwd_params(const FwdWs& W, const float* bias, const int32_t* targets, const int32_t* t_len,
                            const int32_t* u_len, float* lse, float* lp_blank, float* lp_label, int B, int T, int U1,
                            int D, int V, int blank) {
  FwdParams p{};
  p.w_t = W.wb;
  p.bias = bias; p.bias_l2 = W.bias_l2; p.targets = targets; p.t_len = t_len; p.u_len = u_len;
  p.tiles = W.tiles; p.ntiles = W.ntiles;
  p.B = B; p.T = T; p.U1 = U1; p.D = D; p.V = V; p.Vp = pad_v(V); p.NH = p.Vp / 2; p.blank = blank;
  p.lse = lse; p.lp_blank = lp_blank; p.lp_label = lp_label;
  p.prof = g_prof_buf;
  tc_error_host_word(&p.err_host);
  return p;
}

// one launch of the single-CTA forward kernel (joint_fwd2_*): the untiled call, or one vocabulary tile (vt)
static int launch_fwd2(FwdParams& p, const CUtensorMap& tmap_e, const CUtensorMap& tmap_p, bool split, int act, bool vt,
                       int mt, cudaStream_t st) {
  int ws_n = F_MAX_W_STAGES;
  while (ws_n > 2 && fwd2_smem_bytes(p.NH, p.Vp, ws_n) > 232448) --ws_n;
  p.w_stages = ws_n;
  const size_t smem = fwd2_smem_bytes(p.NH, p.Vp, ws_n);
  CTCVR_REQUIRE(smem <= 232448, "joint_rnnt_fwd %s: shared memory budget exceeded (%zu B)", split ? "bf16x3" : "bf16", smem);
  const auto kern = split ? (vt ? pick_act(act, joint_fwd2_x3_vt_kernel, joint_fwd2_x3_vt_relu_kernel, joint_fwd2_x3_vt_gelu_kernel)
                                : pick_act(act, joint_fwd2_x3_kernel, joint_fwd2_x3_relu_kernel, joint_fwd2_x3_gelu_kernel))
                          : (vt ? pick_act(act, joint_fwd2_vt_kernel, joint_fwd2_vt_relu_kernel, joint_fwd2_vt_gelu_kernel)
                                : pick_act(act, joint_fwd2_kernel, joint_fwd2_relu_kernel, joint_fwd2_gelu_kernel));
  CTCVR_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<min(sm_count(), mt), F_THREADS, smem, st>>>(tmap_e, tmap_p, p);
  CTCVR_LAUNCH_CHECK();
  return 0;
}

// split = 1: precision bf16x3 (fp32 inputs, hi / lo operand split, joint_fwd2_x3_kernel); act: the joint activation
int joint_fwd_tc(const void* enc_v, const void* pred_v, int in_bf16, int split, int act, const float* w, const float* bias,
                 const int32_t* targets, const int32_t* t_len, const int32_t* u_len, float* lse, float* lp_blank,
                 float* lp_label, int B, int T, int U1, int D, int V, int blank, void* ws, size_t ws_bytes, cudaStream_t st) {
  const float* enc = reinterpret_cast<const float*>(enc_v);
  const float* pred = reinterpret_cast<const float*>(pred_v);
  // one predicate for both directions, and no silent change of arithmetic: a shape outside the tensor-core tiling is
  // an error here (the fp32 kernels are ~40x slower and round differently - the caller has to ask for them)
  CTCVR_REQUIRE(joint_tc_bwd_supported(U1, D, V), "%s: precision = %s needs D %% 128 == 0, D <= 512, V <= 416 and U+1 <= 128 (got D=%d V=%d U+1=%d); use precision = fp32 for this shape", "joint_rnnt_fwd", split ? "bf16x3" : "bf16", D, V, U1);
  if (check_tc_error("joint_rnnt_fwd")) return 1;
  CTCVR_REQUIRE(ws && ws_bytes >= joint_fwd_tc_ws_bytes(B, T, U1, D, V, split), "joint_rnnt_fwd %s: workspace too small", split ? "bf16x3" : "bf16");
  CTCVR_REQUIRE(((uintptr_t)enc & 15) == 0 && ((uintptr_t)pred & 15) == 0, "joint_rnnt_fwd %s: enc_proj / pred_proj must be 16-byte aligned", split ? "bf16x3" : "bf16");
  const int Vp = pad_v(V), NH = Vp / 2;
  FwdWs W = carve_fwd_ws(ws, B, T, U1, D, V, split != 0);
  const int mt = max_tiles_fwd2(B, T, U1);
  if (split) {
    PrepArgs q{};
    q.w = w; q.bias = bias; q.w_t = W.wb; q.bias_l2 = W.bias_l2; q.V = V; q.Vp = Vp; q.D = D;
    q.nW = cdiv((long)((Vp + 63) / 64) * 64 * D, 256);
    q.t_len = t_len; q.u_len = u_len; q.B = B; q.T = T; q.U1 = U1; q.geom = 0; q.max_tiles = mt;
    q.tiles = W.tiles; q.ntiles = W.ntiles;
    prep_kernel<true><<<q.nW + B, 256, 0, st>>>(q);
    CTCVR_LAUNCH_CHECK();
    FwdParams p = fwd_params(W, bias, targets, t_len, u_len, lse, lp_blank, lp_label, B, T, U1, D, V, blank);
    p.enc = enc; p.pred = pred;
    const CUtensorMap unused{};             // the bf16x3 producers read the fp32 rows directly
    return launch_fwd2(p, unused, unused, true, act, false, mt, st);
  }
  // the parked CTA-pair forward computes tanh only
  const bool use_pair = fwdp_smem_bytes(NH, D) <= 232448 && sm_count() >= 2 && !g_force_single_cta && act == ACT_TANH;
  {
    PrepArgs q{};
    q.fwd_pair = use_pair ? 1 : 0;
    q.w = w; q.bias = bias; q.w_t = W.wb; q.bias_l2 = W.bias_l2; q.V = V; q.Vp = Vp; q.D = D;
    q.nW = cdiv((long)((Vp + 63) / 64) * 64 * D, 256);
    q.t_len = t_len; q.u_len = u_len; q.B = B; q.T = T; q.U1 = U1; q.geom = 0; q.max_tiles = mt;
    q.tiles = W.tiles; q.ntiles = W.ntiles;
    int extra = 0;
    if (in_bf16) {                      // activations already bf16 (autocast): use them in place
      W.eb = const_cast<__nv_bfloat16*>(reinterpret_cast<const __nv_bfloat16*>(enc_v));
      W.pb = const_cast<__nv_bfloat16*>(reinterpret_cast<const __nv_bfloat16*>(pred_v));
    } else {
      q.a = reinterpret_cast<const float4*>(enc); q.ab = reinterpret_cast<uint2*>(W.eb); q.na4 = (long)B * T * D / 4;
      q.b4 = reinterpret_cast<const float4*>(pred); q.bb = reinterpret_cast<uint2*>(W.pb); q.nb4 = (long)B * U1 * D / 4;
      extra = (int)std::min<long>((q.na4 + q.nb4 + 255) / 256, 148L * 8);
    }
    prep_kernel<false><<<q.nW + B + extra, 256, 0, st>>>(q);
    CTCVR_LAUNCH_CHECK();
  }
  if (use_pair) {
    // CTA-pair kernel: W_out resident in shared memory, double-buffered accumulators (joint_tc_fwd_pair.cuh)
    FwdPairParams q{};
    q.w_t = W.wb; q.eb = W.eb; q.pb = W.pb;
    q.bias = bias; q.bias_l2 = W.bias_l2; q.targets = targets; q.t_len = t_len; q.u_len = u_len;
    q.tiles = W.tiles; q.ntiles = W.ntiles;
    q.B = B; q.T = T; q.U1 = U1; q.D = D; q.V = V; q.Vp = Vp; q.NH = NH; q.blank = blank;
    q.lse = lse; q.lp_blank = lp_blank; q.lp_label = lp_label;
    q.prof = g_prof_buf;
    tc_error_host_word(&q.err_host);
    const size_t smem = fwdp_smem_bytes(NH, D);
    CTCVR_CHECK_CUDA(cudaFuncSetAttribute(joint_fwd3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = std::max(2, std::min(sm_count() & ~1, 2 * mt));
    joint_fwd3_kernel<<<grid, FP_THREADS, smem, st>>>(q);
    CTCVR_LAUNCH_CHECK();
    return 0;
  }
  CUtensorMap tmap_e, tmap_p;
  if (make_tmap_bf16_2d(&tmap_e, W.eb, (uint64_t)B * T, D, D, 32)) return 1;
  if (make_tmap_bf16_2d(&tmap_p, W.pb, (uint64_t)B * U1, D, D, 4)) return 1;
  FwdParams p = fwd_params(W, bias, targets, t_len, u_len, lse, lp_blank, lp_label, B, T, U1, D, V, blank);
  return launch_fwd2(p, tmap_e, tmap_p, false, act, false, mt, st);
}

size_t joint_fwd_vt_ws_bytes(int B, int T, int U1, int D, int V, int split) {
  if (!joint_tc_vt_supported(U1, D, V)) return 256;       // the call itself fails with the reason
  const VocabTiles vt = vocab_tiles(V);
  if (vt.n == 1) return joint_fwd_tc_ws_bytes(B, T, U1, D, V, split);
  return carve_fwd_ws(nullptr, B, T, U1, D, vt.Vc, split != 0, vt.n).bytes;
}

// Vocabulary tiles (ctcvr_joint_rnnt_fwd_vt): one prep launch for the weights of every tile, one forward launch per
// tile merging its log-sum-exp into lse, and vt_finalize_kernel.  One tile (pad32(V) <= 416) is the untiled call.
int joint_fwd_vt(const float* enc, const float* pred, int split, int act, const float* w, const float* bias,
                 const int32_t* targets, const int32_t* t_len, const int32_t* u_len, float* lse, float* lp_blank,
                 float* lp_label, int B, int T, int U1, int D, int V, int blank, void* ws, size_t ws_bytes, cudaStream_t st) {
  const char* prec = split ? "bf16x3" : "bf16";
  CTCVR_REQUIRE(joint_tc_vt_supported(U1, D, V), "joint_rnnt_fwd_vt: precision = %s needs D %% 128 == 0, D <= 512, V <= %d and U+1 <= 128 (got D=%d V=%d U+1=%d); use precision = fp32 for this shape", prec, VT_MAX_V, D, V, U1);
  const VocabTiles vt = vocab_tiles(V);
  if (vt.n == 1)
    return joint_fwd_tc(enc, pred, 0, split, act, w, bias, targets, t_len, u_len, lse, lp_blank, lp_label, B, T, U1, D, V,
                        blank, ws, ws_bytes, st);
  if (check_tc_error("joint_rnnt_fwd_vt")) return 1;
  CTCVR_REQUIRE(ws && ws_bytes >= joint_fwd_vt_ws_bytes(B, T, U1, D, V, split), "joint_rnnt_fwd_vt %s: workspace too small", prec);
  CTCVR_REQUIRE(((uintptr_t)enc & 15) == 0 && ((uintptr_t)pred & 15) == 0, "joint_rnnt_fwd_vt %s: enc_proj / pred_proj must be 16-byte aligned", prec);
  const int Vc = vt.Vc;
  FwdWs W = carve_fwd_ws(ws, B, T, U1, D, Vc, split != 0, vt.n);
  const int mt = max_tiles_fwd2(B, T, U1);
  {
    PrepArgs q{};
    q.w = w; q.bias = bias; q.w_t = W.wb; q.bias_l2 = W.bias_l2; q.V = V; q.Vp = Vc; q.D = D;
    q.nW = cdiv((long)((Vc + 63) / 64) * 64 * D, 256);
    q.t_len = t_len; q.u_len = u_len; q.B = B; q.T = T; q.U1 = U1; q.geom = 0; q.max_tiles = mt;
    q.tiles = W.tiles; q.ntiles = W.ntiles;
    int extra = 0;
    if (!split) {
      q.a = reinterpret_cast<const float4*>(enc); q.ab = reinterpret_cast<uint2*>(W.eb); q.na4 = (long)B * T * D / 4;
      q.b4 = reinterpret_cast<const float4*>(pred); q.bb = reinterpret_cast<uint2*>(W.pb); q.nb4 = (long)B * U1 * D / 4;
      extra = (int)std::min<long>((q.na4 + q.nb4 + 255) / 256, 148L * 8);
    }
    if (split) prep_vt_kernel<true><<<q.nW * vt.n + B, 256, 0, st>>>(q, vt.n);
    else prep_vt_kernel<false><<<q.nW * vt.n + B + extra, 256, 0, st>>>(q, vt.n);
    CTCVR_LAUNCH_CHECK();
  }
  CUtensorMap tmap_e{}, tmap_p{};           // bf16x3: unused (the producers read the fp32 rows directly)
  if (!split) {
    if (make_tmap_bf16_2d(&tmap_e, W.eb, (uint64_t)B * T, D, D, 32)) return 1;
    if (make_tmap_bf16_2d(&tmap_p, W.pb, (uint64_t)B * U1, D, D, 4)) return 1;
  }
  const size_t wstride = (size_t)Vc * D * (split ? 2 : 1);
  for (int c = 0; c < vt.n; ++c) {
    const int v0 = c * Vc, Vr = std::min(V - v0, Vc);
    FwdParams p = fwd_params(W, bias + v0, targets, t_len, u_len, lse, lp_blank, lp_label, B, T, U1, D, Vr,
                             (blank >= v0 && blank < v0 + Vr) ? blank - v0 : -1);
    p.w_t = W.wb + c * wstride; p.bias_l2 = W.bias_l2 + (size_t)c * Vc;
    p.Vp = Vc; p.NH = Vc / 2;                 // the tile's padded width (pad_v(Vr) may be smaller in the last tile)
    if (split) { p.enc = enc; p.pred = pred; }
    p.v0 = v0; p.Vg = V; p.blank_g = blank; p.merge = c > 0;
    if (launch_fwd2(p, tmap_e, tmap_p, split != 0, act, true, mt, st)) return 1;
  }
  const long cells = (long)B * T * U1;
  vt_finalize_kernel<<<cdiv(cells, 256), 256, 0, st>>>(lse, lp_blank, lp_label, t_len, u_len, B, T, U1);
  CTCVR_LAUNCH_CHECK();
  return 0;
}

size_t joint_bwd_f32_ws_bytes(int, int, int, int, int);
int joint_bwd_f32(const float*, const float*, const float*, const float*, const int32_t*, const int32_t*,
                  const int32_t*, const float*, const float*, const float*, const float*, const float*, float, float*,
                  float*, float*, float*, int, int, int, int, int, int, void*, size_t, cudaStream_t);


struct BwdWs {
  __nv_bfloat16 *wb, *wtb, *gt, *gt_lo, *eb, *pb;
  float *bias_pad, *bias_l2, *d_enc_part, *partials, *d_pred_acc;
  int4 *tiles, *tile_rows;
  int* ntiles;
  long Rpad;
  int KS, S_max, mt;
  size_t bytes;
};
// split (bf16x3): hi / lo copies of W_out and W_out^T and a second G spill (G_lo); no bf16 activation copies
// nvt > 1: vocabulary tiles of V = Vc columns each: their weights back to back, one tile's G spill and dW partials
static BwdWs carve_bwd_ws(void* ws, int B, int T, int U1, int D, int V, bool split = false, int nvt = 1) {
  const int Vp = pad_v(V);
  uint8_t* p = reinterpret_cast<uint8_t*>(ws);
  size_t off = 0;
  BwdWs w;
  w.mt = max_tiles_rect(B, T, U1);
  w.Rpad = (long)(w.mt + 1) * BM;           // + one scratch row tile for the dummy iterations of the lock-step loop
  w.S_max = (U1 + 15) / 16;               // >= the number of u-splits of either geometry
  const int MB = D / 128;
  w.KS = MB > 0 ? sm_count() / MB : 1;
  if (w.KS < 1) w.KS = 1;
  auto take = [&](size_t n) { void* r = p + off; off = align_up(off + n, 1024); return r; };
  const size_t nw = split ? 2 : 1;
  w.wb = reinterpret_cast<__nv_bfloat16*>(take((size_t)nvt * Vp * D * 2 * nw));
  w.wtb = reinterpret_cast<__nv_bfloat16*>(take((size_t)nvt * ((Vp + 63) / 64) * 64 * D * 2 * nw));
  w.eb = split ? nullptr : reinterpret_cast<__nv_bfloat16*>(take((size_t)B * T * D * 2));
  w.pb = split ? nullptr : reinterpret_cast<__nv_bfloat16*>(take((size_t)B * U1 * D * 2));
  w.bias_pad = reinterpret_cast<float*>(take((size_t)Vp * 4));
  w.bias_l2 = reinterpret_cast<float*>(take((size_t)nvt * Vp * 4));
  w.tiles = reinterpret_cast<int4*>(take((size_t)w.mt * 16));
  w.tile_rows = reinterpret_cast<int4*>(take((size_t)w.mt * 16));
  w.ntiles = reinterpret_cast<int*>(take(4));
  w.gt = reinterpret_cast<__nv_bfloat16*>(take((size_t)((Vp + 63) / 64) * 64 * w.Rpad * 2));
  w.gt_lo = split ? reinterpret_cast<__nv_bfloat16*>(take((size_t)((Vp + 63) / 64) * 64 * w.Rpad * 2)) : nullptr;
  w.d_enc_part = reinterpret_cast<float*>(take((size_t)w.S_max * B * T * D * 4));
  w.partials = reinterpret_cast<float*>(take((size_t)w.KS * D * Vp * 4));
  w.d_pred_acc = nvt > 1 ? nullptr : reinterpret_cast<float*>(take((size_t)B * U1 * D * 4));   // bf16 inputs only
  w.bytes = off;
  return w;
}

size_t joint_bwd_tc_ws_bytes(int B, int T, int U1, int D, int V, int split) {
  if (!joint_tc_bwd_supported(U1, D, V)) return 256;      // the call itself fails with the reason
  return carve_bwd_ws(nullptr, B, T, U1, D, V, split != 0).bytes;
}

// Kernel 1 of the backward for tile geometry (P, TT): the CTA-pair kernel (bf16, use_pair), the single-CTA kernel or its
// bf16x3 form; the untiled call, or one vocabulary tile (vt).  The tensor maps are unused by the bf16x3 form.
template <int P, int TT>
static int launch_bwd_main(BwdParams& p, const BwdWs& W, bool use_pair, bool split, int act, bool vt, cudaStream_t st) {
  const int B = p.B, T = p.T, U1 = p.U1, D = p.D;
  CUtensorMap tmap_e{}, tmap_p{};
  if (!split) {
    if (make_tmap_bf16_2d(&tmap_e, W.eb, (uint64_t)B * T, D, D, TT)) return 1;
    if (make_tmap_bf16_2d(&tmap_p, W.pb, (uint64_t)B * U1, D, D, P)) return 1;
  }
  if (use_pair) {
    CUtensorMap tmap_e2;                 // both tiles' frames in one box (P4 slab)
    if (make_tmap_bf16_2d(&tmap_e2, W.eb, (uint64_t)B * T, D, D, 2 * TT)) return 1;
    p.r1_stages = bwd4_r1_stages(p.NH, p.Vp);
    const size_t smem = bwd4_smem_bytes<P>(p.NH, p.Vp, D);
    const int gridp = std::max(2, std::min(sm_count() & ~1, W.mt & ~1));
    const auto k = vt ? pick_act(act, joint_bwd4_vt_kernel<P, TT>, joint_bwd4_vt_relu_kernel<P, TT>, joint_bwd4_vt_gelu_kernel<P, TT>)
                      : pick_act(act, joint_bwd4_kernel<P, TT>, joint_bwd4_relu_kernel<P, TT>, joint_bwd4_gelu_kernel<P, TT>);
    CTCVR_CHECK_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<gridp, NTHREADS, smem, st>>>(tmap_e, tmap_e2, tmap_p, p);
    CTCVR_LAUNCH_CHECK();
    return 0;
  }
  p.r1_stages = bwd3_r1_stages(p.NH, p.Vp);
  const size_t smem = bwd3_smem_bytes(p.NH, p.Vp, D, split);
  CTCVR_REQUIRE(smem <= 232448 && p.r1_stages >= 2, "joint_rnnt_bwd %s: shared memory budget exceeded (%zu B)", split ? "bf16x3" : "bf16", smem);
  const auto k = split ? (vt ? pick_act(act, joint_bwd3_x3_vt_kernel<P, TT>, joint_bwd3_x3_vt_relu_kernel<P, TT>, joint_bwd3_x3_vt_gelu_kernel<P, TT>)
                             : pick_act(act, joint_bwd3_x3_kernel<P, TT>, joint_bwd3_x3_relu_kernel<P, TT>, joint_bwd3_x3_gelu_kernel<P, TT>))
                       : (vt ? pick_act(act, joint_bwd3_vt_kernel<P, TT>, joint_bwd3_vt_relu_kernel<P, TT>, joint_bwd3_vt_gelu_kernel<P, TT>)
                             : pick_act(act, joint_bwd3_kernel<P, TT>, joint_bwd3_relu_kernel<P, TT>, joint_bwd3_gelu_kernel<P, TT>));
  CTCVR_CHECK_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<min(sm_count(), W.mt), NTHREADS, smem, st>>>(tmap_e, tmap_p, p);
  CTCVR_LAUNCH_CHECK();
  return 0;
}

// Kernel 2 of the backward and its split-K reduction: d_w[v][:] for the V real rows of the Vp-column G spill in gt
// (/ gt_lo), for tile geometry (P, TT).  d_w points at the first row of the vocabulary tile.
template <int P, int TT>
static int launch_bwd_dw(const BwdWs& W, const float* enc, const float* pred, const __nv_bfloat16* gt,
                         const __nv_bfloat16* gt_lo, float* d_w, int B, int T, int U1, int D, int V, int Vp, bool split,
                         int act, cudaStream_t st) {
  const int KBG = (Vp + 63) / 64, MB = D / 128;
  const size_t smem = dwr_smem_bytes<P>(KBG, split);
  CTCVR_REQUIRE(smem <= 232448, "dW GEMM%s: shared memory budget exceeded (%zu B)", split ? " bf16x3" : "", smem);
  if (split) {
    const CUtensorMap unused{};             // the split kernels read the fp32 rows directly
    const auto k = pick_act(act, dw_gemm_rz_x3_kernel<P, TT>, dw_gemm_rz_x3_relu_kernel<P, TT>, dw_gemm_rz_x3_gelu_kernel<P, TT>);
    CTCVR_CHECK_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<dim3(MB, W.KS), DWR_THREADS, smem, st>>>(unused, unused, gt, gt_lo, enc, pred, W.tile_rows, W.ntiles, W.partials, D,
                                                Vp, KBG, W.KS);
  } else {
    CUtensorMap tmap_e, tmap_p;          // the same 64-wide SW128 boxes as kernel 1: TT enc rows / P pred rows
    if (make_tmap_bf16_2d(&tmap_e, W.eb, (uint64_t)B * T, D, D, TT)) return 1;
    if (make_tmap_bf16_2d(&tmap_p, W.pb, (uint64_t)B * U1, D, D, P)) return 1;
    const auto k = pick_act(act, dw_gemm_rz_kernel<P, TT>, dw_gemm_rz_relu_kernel<P, TT>, dw_gemm_rz_gelu_kernel<P, TT>);
    CTCVR_CHECK_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<dim3(MB, W.KS), DWR_THREADS, smem, st>>>(tmap_e, tmap_p, gt, W.tile_rows, W.ntiles, W.partials, D, Vp, KBG, W.KS);
  }
  CTCVR_LAUNCH_CHECK();
  reduce_dw_kernel<<<dim3(cdiv(D, 8), cdiv(Vp, 32)), 256, 0, st>>>(W.partials, d_w, D, V, Vp, W.KS);
  CTCVR_LAUNCH_CHECK();
  return 0;
}

// the fields of BwdParams every kernel-1 launch shares
static BwdParams bwd_params(const BwdWs& W, const float* enc, const float* pred, const int32_t* targets,
                            const int32_t* t_len, const int32_t* u_len, const float* lse, const float* lp_blank,
                            const float* lp_label, const float* alpha, const float* beta, const float* costs,
                            const float* grad_costs, float clamp, float* d_pred, float* d_b, int B, int T, int U1, int D,
                            int V, int blank, bool split) {
  BwdParams p{};
  p.w_t = W.wb; p.wt_t = W.wtb;
  if (split) { p.enc = enc; p.pred = pred; p.gt_lo = W.gt_lo; }
  p.bias_l2 = W.bias_l2; p.targets = targets; p.t_len = t_len; p.u_len = u_len;
  p.tiles = W.tiles; p.ntiles = W.ntiles;
  p.B = B; p.T = T; p.U1 = U1; p.D = D; p.V = V; p.Vp = pad_v(V); p.NH = p.Vp / 2; p.blank = blank;
  p.lse = lse; p.lp_blank = lp_blank; p.lp_label = lp_label;
  p.alpha = alpha; p.beta = beta; p.costs = costs; p.grad_costs = grad_costs; p.clamp = clamp;
  p.gt = W.gt;
  p.d_enc_part = W.d_enc_part; p.d_pred = d_pred; p.d_bias = d_b;
  p.prof = g_prof_buf;
  tc_error_host_word(&p.err_host);
  return p;
}

// the CTA-pair backward kernel takes D % 256 == 0 when its shared memory and ring fit (bf16 only)
static bool bwd_use_pair(const RectGeom& G, int NH, int Vp, int D) {
  const size_t smem_pair = G.P == 21 ? bwd4_smem_bytes<21>(NH, Vp, D) : bwd4_smem_bytes<16>(NH, Vp, D);
  return D % 256 == 0 && smem_pair <= 232448 && sm_count() >= 2 && bwd4_r1_stages(NH, Vp) >= 4 && !g_bwd_single_cta;
}

int joint_bwd_tc(const void* enc_v, const void* pred_v, int in_bf16, int split, int act, const float* w, const float* bias, const int32_t* targets,
                 const int32_t* t_len, const int32_t* u_len, const float* lse, const float* lp_blank, const float* lp_label,
                 const float* alpha, const float* beta,
                 const float* costs, const float* grad_costs, float clamp, float* d_enc, float* d_pred, float* d_w,
                 float* d_b, int B, int T, int U1, int D, int V, int blank, void* ws, size_t ws_bytes, cudaStream_t st) {
  const float* enc = reinterpret_cast<const float*>(enc_v);
  const float* pred = reinterpret_cast<const float*>(pred_v);
  CTCVR_REQUIRE(joint_tc_bwd_supported(U1, D, V), "%s: precision = %s needs D %% 128 == 0, D <= 512, V <= 416 and U+1 <= 128 (got D=%d V=%d U+1=%d); use precision = fp32 for this shape", "joint_rnnt_bwd", split ? "bf16x3" : "bf16", D, V, U1);
  if (check_tc_error("joint_rnnt_bwd")) return 1;
  CTCVR_REQUIRE(ws && ws_bytes >= joint_bwd_tc_ws_bytes(B, T, U1, D, V, split), "joint_rnnt_bwd %s: workspace too small", split ? "bf16x3" : "bf16");
  CTCVR_REQUIRE(((uintptr_t)enc & 15) == 0 && ((uintptr_t)pred & 15) == 0, "joint_rnnt_bwd %s: enc_proj / pred_proj must be 16-byte aligned", split ? "bf16x3" : "bf16");
  const int Vp = pad_v(V), NH = Vp / 2;
  BwdWs W = carve_bwd_ws(ws, B, T, U1, D, V, split != 0);
  const int KBG = (Vp + 63) / 64;
  const int mt = W.mt;
  RectGeom G = pick_rect_geom(T, U1);
  // CTA-pair kernel (joint_tc_bwd_pair.cuh): D in 256-row blocks of dZ^T, tiles paired along the frame axis
  const bool use_pair = !split && bwd_use_pair(G, NH, Vp, D);
  G.even = use_pair ? 1 : 0;
  // bf16 inputs -> bf16 gradients: d_pred is accumulated in fp32 in the workspace and converted by the d_enc reduction
  float* d_pred_acc = in_bf16 ? W.d_pred_acc : d_pred;
  {
    PrepArgs q{};
    q.w = w; q.bias = bias; q.w_t = W.wb; q.wt_t = W.wtb; q.bias_pad = W.bias_pad; q.bias_l2 = W.bias_l2;
    q.V = V; q.Vp = Vp; q.D = D; q.nW = cdiv((long)KBG * 64 * D, 256);
    q.t_len = t_len; q.u_len = u_len; q.B = B; q.T = T; q.U1 = U1; q.geom = G.P | (G.TT << 8) | (G.even << 16);
    q.max_tiles = mt; q.tiles = W.tiles; q.tile_rows = W.tile_rows; q.ntiles = W.ntiles;
    q.zero0 = d_pred_acc; q.n0 = (long)B * U1 * D; q.zero1 = d_b; q.n1 = V;
    if (split) {
      const int extra = (int)std::min<long>((q.n0 + 1023) / 1024, 148L * 8);
      prep_kernel<true><<<q.nW + B + extra, 256, 0, st>>>(q);
    } else {
      if (in_bf16) {
        W.eb = const_cast<__nv_bfloat16*>(reinterpret_cast<const __nv_bfloat16*>(enc_v));
        W.pb = const_cast<__nv_bfloat16*>(reinterpret_cast<const __nv_bfloat16*>(pred_v));
      } else {
        q.a = reinterpret_cast<const float4*>(enc); q.ab = reinterpret_cast<uint2*>(W.eb); q.na4 = (long)B * T * D / 4;
        q.b4 = reinterpret_cast<const float4*>(pred); q.bb = reinterpret_cast<uint2*>(W.pb); q.nb4 = (long)B * U1 * D / 4;
      }
      const int extra = (int)std::min<long>((q.n0 + q.na4 * 4 + q.nb4 * 4 + 1023) / 1024, 148L * 8);
      prep_kernel<false><<<q.nW + B + extra, 256, 0, st>>>(q);
    }
    CTCVR_LAUNCH_CHECK();
  }
  BwdParams p = bwd_params(W, enc, pred, targets, t_len, u_len, lse, lp_blank, lp_label, alpha, beta, costs, grad_costs,
                           clamp, d_pred_acc, d_b, B, T, U1, D, V, blank, split != 0);
  if (G.P == 21 ? launch_bwd_main<21, 6>(p, W, use_pair, split != 0, act, false, st)
                : launch_bwd_main<16, 8>(p, W, use_pair, split != 0, act, false, st)) return 1;
  if (in_bf16)
    reduce_denc_kernel<true><<<B * T + B * U1, 128, 0, st>>>(W.d_enc_part, t_len, u_len, d_enc, B, T, U1, D, G.P, d_pred_acc, d_pred);
  else
    reduce_denc_kernel<false><<<B * T, 128, 0, st>>>(W.d_enc_part, t_len, u_len, d_enc, B, T, U1, D, G.P, nullptr, nullptr);
  CTCVR_LAUNCH_CHECK();
  return G.P == 21 ? launch_bwd_dw<21, 6>(W, enc, pred, W.gt, W.gt_lo, d_w, B, T, U1, D, V, Vp, split != 0, act, st)
                   : launch_bwd_dw<16, 8>(W, enc, pred, W.gt, W.gt_lo, d_w, B, T, U1, D, V, Vp, split != 0, act, st);
}

size_t joint_bwd_vt_ws_bytes(int B, int T, int U1, int D, int V, int split) {
  if (!joint_tc_vt_supported(U1, D, V)) return 256;       // the call itself fails with the reason
  const VocabTiles vt = vocab_tiles(V);
  if (vt.n == 1) return joint_bwd_tc_ws_bytes(B, T, U1, D, V, split);
  return carve_bwd_ws(nullptr, B, T, U1, D, vt.Vc, split != 0, vt.n).bytes;
}

// Vocabulary tiles (ctcvr_joint_rnnt_bwd_vt): one prep launch (every tile's weights, the tile table, the zero fills of
// d_pred and d_bias), then per tile kernel 1 (d_pred / d_bias accumulate; d_enc partials stored by tile 0, added by the
// others), kernel 2 and its reduction into the tile's rows of d_w; the d_enc reduction once at the end.  The G spill
// and the dW partials are one tile's, reused by the next in stream order.  One tile is the untiled call.
int joint_bwd_vt(const float* enc, const float* pred, int split, int act, const float* w, const float* bias,
                 const int32_t* targets, const int32_t* t_len, const int32_t* u_len, const float* lse,
                 const float* lp_blank, const float* lp_label, const float* alpha, const float* beta, const float* costs,
                 const float* grad_costs, float clamp, float* d_enc, float* d_pred, float* d_w, float* d_b, int B, int T,
                 int U1, int D, int V, int blank, void* ws, size_t ws_bytes, cudaStream_t st) {
  const char* prec = split ? "bf16x3" : "bf16";
  CTCVR_REQUIRE(joint_tc_vt_supported(U1, D, V), "joint_rnnt_bwd_vt: precision = %s needs D %% 128 == 0, D <= 512, V <= %d and U+1 <= 128 (got D=%d V=%d U+1=%d); use precision = fp32 for this shape", prec, VT_MAX_V, D, V, U1);
  const VocabTiles vt = vocab_tiles(V);
  if (vt.n == 1)
    return joint_bwd_tc(enc, pred, 0, split, act, w, bias, targets, t_len, u_len, lse, lp_blank, lp_label, alpha, beta,
                        costs, grad_costs, clamp, d_enc, d_pred, d_w, d_b, B, T, U1, D, V, blank, ws, ws_bytes, st);
  if (check_tc_error("joint_rnnt_bwd_vt")) return 1;
  CTCVR_REQUIRE(ws && ws_bytes >= joint_bwd_vt_ws_bytes(B, T, U1, D, V, split), "joint_rnnt_bwd_vt %s: workspace too small", prec);
  CTCVR_REQUIRE(((uintptr_t)enc & 15) == 0 && ((uintptr_t)pred & 15) == 0, "joint_rnnt_bwd_vt %s: enc_proj / pred_proj must be 16-byte aligned", prec);
  const int Vc = vt.Vc, KBG = (Vc + 63) / 64;
  BwdWs W = carve_bwd_ws(ws, B, T, U1, D, Vc, split != 0, vt.n);
  RectGeom G = pick_rect_geom(T, U1);
  const bool use_pair = !split && bwd_use_pair(G, Vc / 2, Vc, D);
  G.even = use_pair ? 1 : 0;
  {
    PrepArgs q{};
    q.w = w; q.bias = bias; q.w_t = W.wb; q.wt_t = W.wtb; q.bias_l2 = W.bias_l2;
    q.V = V; q.Vp = Vc; q.D = D; q.nW = cdiv((long)KBG * 64 * D, 256);
    q.t_len = t_len; q.u_len = u_len; q.B = B; q.T = T; q.U1 = U1; q.geom = G.P | (G.TT << 8) | (G.even << 16);
    q.max_tiles = W.mt; q.tiles = W.tiles; q.tile_rows = W.tile_rows; q.ntiles = W.ntiles;
    q.zero0 = d_pred; q.n0 = (long)B * U1 * D; q.zero1 = d_b; q.n1 = V;
    if (!split) {
      q.a = reinterpret_cast<const float4*>(enc); q.ab = reinterpret_cast<uint2*>(W.eb); q.na4 = (long)B * T * D / 4;
      q.b4 = reinterpret_cast<const float4*>(pred); q.bb = reinterpret_cast<uint2*>(W.pb); q.nb4 = (long)B * U1 * D / 4;
    }
    const int extra = (int)std::min<long>((q.n0 + q.na4 * 4 + q.nb4 * 4 + 1023) / 1024, 148L * 8);
    if (split) prep_vt_kernel<true><<<q.nW * vt.n + B + extra, 256, 0, st>>>(q, vt.n);
    else prep_vt_kernel<false><<<q.nW * vt.n + B + extra, 256, 0, st>>>(q, vt.n);
    CTCVR_LAUNCH_CHECK();
  }
  const size_t wstride = (size_t)Vc * D * (split ? 2 : 1), wtstride = (size_t)KBG * 64 * D * (split ? 2 : 1);
  for (int c = 0; c < vt.n; ++c) {
    const int v0 = c * Vc, Vr = std::min(V - v0, Vc);
    BwdParams p = bwd_params(W, enc, pred, targets, t_len, u_len, lse, lp_blank, lp_label, alpha, beta, costs, grad_costs,
                             clamp, d_pred, d_b + v0, B, T, U1, D, Vr, (blank >= v0 && blank < v0 + Vr) ? blank - v0 : -1,
                             split != 0);
    p.w_t = W.wb + c * wstride; p.wt_t = W.wtb + c * wtstride; p.bias_l2 = W.bias_l2 + (size_t)c * Vc;
    p.Vp = Vc; p.NH = Vc / 2;                 // the tile's padded width (pad_v(Vr) may be smaller in the last tile)
    p.v0 = v0; p.Vg = V; p.blank_g = blank; p.accum = c > 0;
    if (G.P == 21 ? launch_bwd_main<21, 6>(p, W, use_pair, split != 0, act, true, st)
                  : launch_bwd_main<16, 8>(p, W, use_pair, split != 0, act, true, st)) return 1;
    float* dw = d_w + (size_t)v0 * D;
    if (G.P == 21 ? launch_bwd_dw<21, 6>(W, enc, pred, W.gt, W.gt_lo, dw, B, T, U1, D, Vr, Vc, split != 0, act, st)
                  : launch_bwd_dw<16, 8>(W, enc, pred, W.gt, W.gt_lo, dw, B, T, U1, D, Vr, Vc, split != 0, act, st)) return 1;
  }
  reduce_denc_kernel<false><<<B * T, 128, 0, st>>>(W.d_enc_part, t_len, u_len, d_enc, B, T, U1, D, G.P, nullptr, nullptr);
  CTCVR_LAUNCH_CHECK();
  return 0;
}

void tc_set_prof(void* buf) { g_prof_buf = reinterpret_cast<long long*>(buf); }
void tc_set_mode(int mode) {            // bit 0: single-CTA forward (default 1), bit 1: single-CTA backward (default 0)
  g_force_single_cta = mode & 1;
  g_bwd_single_cta = (mode >> 1) & 1;
}

unsigned int tc_error_flag() {
  unsigned int v = 0;
  cudaMemcpyFromSymbol(&v, tc::g_tc_error, sizeof(v));
  unsigned int zero = 0;
  if (v) cudaMemcpyToSymbol(tc::g_tc_error, &zero, sizeof(zero));
  return v;
}

}  // namespace ctcvr
