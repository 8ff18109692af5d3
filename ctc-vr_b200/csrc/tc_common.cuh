// sm_100a primitives used by the tcgen05 kernels: mbarrier, TMA (cp.async.bulk.tensor), TMEM
// allocation, tcgen05.mma / commit / ld, UMMA shared-memory and instruction descriptors.
// Layout conventions (all operands K-major, 128-byte swizzle, bf16):
//   a tile of R rows x 64 k-elements occupies R*128 bytes, 1024-byte aligned; row r lives at
//   r*128, and its 16-byte chunk c (k = 8c..8c+7) is stored at chunk position c ^ (r & 7).
//   This is exactly what TMA writes with CU_TENSOR_MAP_SWIZZLE_128B and what the UMMA descriptor
//   with layout SWIZZLE_128B, SBO = 1024 B expects; advancing k by 16 elements adds 32 B to the
//   descriptor start address.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace ctcvr {
namespace tc {

// ---------------------------------------------------------------------------- debug guard
// Every mbarrier wait is bounded: a protocol bug must not hang the GPU.  On timeout the kernel
// records where, and all later waits return immediately; the host reads the flag after the call.
__device__ unsigned int g_tc_error = 0;
// mapped pinned host word (set by every tcgen05 kernel from its parameters): the host reads it without a
// synchronisation at the next entry-point call and fails that call loudly
__device__ unsigned int* g_tc_error_host = nullptr;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait; `site` identifies the call site in the error flag.  The hot path touches no global
// memory: the error flag is only consulted / written after ~2^20 failed probes (each probe already
// suspends the warp in hardware for a while), so a protocol bug degrades into a slow, flagged exit.
__device__ __noinline__ bool mbar_timeout(uint32_t site) {
  const unsigned int code = 0x80000000u | (site << 16) | (blockIdx.x & 0xffffu);
  atomicCAS(&g_tc_error, 0u, code);
  unsigned int* h = g_tc_error_host;
  if (h != nullptr) { *reinterpret_cast<volatile unsigned int*>(h) = code; __threadfence_system(); }
  return true;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, uint32_t site) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    // every 4096 failed probes: give up if this wait is hopeless or another wait already timed out
    if ((++spins & 4095u) == 0u && (spins > (1u << 20) || *(volatile unsigned int*)&g_tc_error != 0u)) {
      if (mbar_timeout(site)) return;
    }
  }
}

// ---------------------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// 1-D bulk copy global -> shared (contiguous, 16-byte aligned, size multiple of 16), completion on an mbarrier.
// Much cheaper than a 2-D tensor copy of the same bytes (which is issued row by row): operands that this library
// lays out itself (weights, spills) are stored pre-tiled and pre-swizzled so that a stage is one contiguous block.
__device__ __forceinline__ void bulk_load(uint32_t smem_dst, const void* gsrc, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_dst), "l"(gsrc), "r"(bytes), "r"(bar) : "memory");
}
// 1-D bulk copy shared -> global, tracked by the per-thread bulk async-group
__device__ __forceinline__ void bulk_store(void* gdst, uint32_t smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// ---------------------------------------------------------------------------- TMEM / tcgen05
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] . B[smem]^T ; one thread issues for the CTA.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrive once all previously issued MMAs of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}


// ---- cta_group::2 (CTA pair).  The pair kernels use M = 128: 64 rows per CTA at the full tensor rate (N/4 cycles per
// K = 16 step, tools/pair_probe.cu).  D of CTA r: row m (0..63) -> TMEM lane m for columns n < N/2 and lane m + 64 for
// n >= N/2 (column n - N/2): a 64 x N fp32 accumulator takes 128 lanes x N/2 columns - half the columns of the M = 256
// and single-CTA forms, which is what lets two accumulators (or logits and dZ^T) coexist in 512 columns.
// A from tensor memory (TS form): row m of the CTA's 64 rows must be present in lane m AND lane m + 64.
// B: N split, rows [0, N/2) in the leader's shared memory, [N/2, N) in the peer's, at the same offset.
// Only the leader (cluster rank 0) issues MMAs and commits; commits are multicast to both CTAs.
__device__ __forceinline__ void tmem_alloc2(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma2_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once all previously issued MMAs of this thread completed) on the barrier at this offset in every CTA of mask
__device__ __forceinline__ void umma2_commit_mc(uint32_t bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"(mask) : "memory");
}
// arrive on the mbarrier at the same smem offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t rank) {
  uint32_t ra;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(bar), "r"(rank));
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(ra) : "memory");
}
// Same without release semantics (no cluster-scope fence in front of the arrive, which costs ~1 k cycles per call): for
// hand-offs whose payload is tensor memory, already complete (tcgen05.wait::st / ::ld) and fenced
// (tcgen05.fence::before_thread_sync) when the CTA-local barrier that precedes this forward was signalled.
__device__ __forceinline__ void mbar_arrive_remote_relaxed(uint32_t bar, uint32_t rank) {
  uint32_t ra;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(bar), "r"(rank));
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(ra) : "memory");
}
// one arrival per warp on the LEADER's barrier (local arrive on rank 0, remote arrive from rank 1)
__device__ __forceinline__ void warp_arrive_leader(uint32_t bar, uint32_t rank) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) {
    if (rank == 0) mbar_arrive(bar); else mbar_arrive_remote(bar, 0);
  }
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// 32 lanes x 32 columns of fp32: thread i of the warp receives TMEM lane (lane_base + i), columns col..col+31.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// D[tmem] (+)= A[tmem] . B[smem]^T : A is read from tensor memory (lane = row, each 32-bit column = two bf16 along K)
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// thread i of the warp writes 16 consecutive 32-bit columns of TMEM lane (lane_base + i)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
// same, 8 columns
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
// 16 lanes x 16 columns in the MMA-fragment layout: thread t receives, for column group cg = 0..3,
// r[2cg] = (lane t/4, column 4cg + t%4) and r[2cg+1] = (lane 8 + t/4, same column)  (tools/tmem_shape_probe.cu).
// With bf16 pairs in the columns this is exactly the operand layout of stmatrix (8x8 b16 tiles).
__device__ __forceinline__ void tmem_ld_16x128b_x4(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.16x128b.x4.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
// four 8x8 b16 tiles stored TRANSPOSED: threads 8m..8m+7 supply the shared addresses of the 8 rows (16 bytes each) of
// tile m; row j of the stored tile = column j of the fragment held in r[m]
__device__ __forceinline__ void stmatrix_x4_trans(uint32_t row_addr, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
  asm volatile("stmatrix.sync.aligned.m8n8.x4.trans.shared.b16 [%0], {%1, %2, %3, %4};" ::"r"(row_addr), "r"(r0), "r"(r1),
               "r"(r2), "r"(r3) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// one column: thread i of the warp receives TMEM lane (lane_base + i), column col
__device__ __forceinline__ float tmem_ld1(uint32_t taddr) {
  uint32_t r;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr) : "memory");
  return __uint_as_float(r);
}
// 32 contiguous, 32-byte aligned bytes of read-only global memory in one request per lane (LDG.256, sm_100+): half the
// L1 wavefronts of two 16-byte loads when every lane touches a different line
struct U32x8 { uint32_t v[8]; };
__device__ __forceinline__ U32x8 ldg256(const void* p) {
  U32x8 r;
  asm volatile("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]), "=r"(r.v[7])
               : "l"(p));
  return r;
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void sts16(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((unsigned short)v) : "memory");
}
__device__ __forceinline__ float lg2_fast(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---------------------------------------------------------------------------- descriptors
// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
// [0,14) start>>4, [16,30) LBO>>4 (=1, unused for swizzled K-major), [32,46) SBO>>4 (=64: 8 rows x 128 B),
// [46,48) version=1, [61,64) layout=2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// MN-major, SWIZZLE_128B descriptor: the operand's M/N dimension is contiguous in shared memory (64 elements = one
// 128-byte swizzle row), 8 consecutive K rows form a 1024-byte atom.  leading byte offset = distance between atoms
// along M/N (the next 64 elements), stride byte offset = distance between 8-row groups along K
// (cute::UMMA::make_umma_desc<Major::MN>: ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units).
__device__ __forceinline__ uint64_t make_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// instruction descriptor with B given MN-major (bit 16)
__host__ __device__ constexpr uint32_t make_idesc_bf16_bmn(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, N>>3 at [17,23), M>>4 at [24,29).
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// 2^x for x <= 0 on the FMA pipe (no MUFU): round-to-nearest split x = i + f, |f| <= 0.5, degree-4 minimax polynomial
// for 2^f (relative error 3.6e-6), exponent restored by an integer add.  The joint kernels are MUFU-bound (tanh of the
// operand producers + exp of the softmax sweeps); moving the exponentials of a sweep here trades 1 MUFU slot for 9
// FMA/ALU slots per element.  Inputs below -126 return 0.
__device__ __forceinline__ float ex2_poly(float x) {
  x = fmaxf(x, -126.f);
  const float t = x + 12582912.f;                  // 1.5 * 2^23: the integer part lands in the low mantissa bits
  const float f = x - (t - 12582912.f);
  float p = fmaf(0.009676037f, f, 0.055922036f);
  p = fmaf(p, f, 0.24022107f);
  p = fmaf(p, f, 0.69312103f);
  p = fmaf(p, f, 1.0000001f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(t) << 23));
}
// tanh(a + b) on packed bf16 pairs: one packed add and one packed MUFU op per two elements.  The sum is rounded to
// bf16 before the tanh (error <= 2^-9 |x| (1 - z^2) <= 9e-4, below the bf16 rounding of z itself).
__device__ __forceinline__ uint32_t tanh_add_bf16x2_packed(uint32_t a, uint32_t b) {
  uint32_t s, r;
  asm("add.rn.bf16x2 %0, %1, %2;" : "=r"(s) : "r"(a), "r"(b));
  asm("tanh.approx.bf16x2 %0, %1;" : "=r"(r) : "r"(s));
  return r;
}

// act(a + b) on packed bf16 pairs for every activation: the sum is the packed bf16 add of the tanh form; relu is a packed
// max with 0 (exact); gelu is evaluated in fp32 (erff) from the bf16 sum and rounded to bf16.
__device__ __forceinline__ uint32_t add_bf16x2(uint32_t a, uint32_t b) {
  uint32_t s;
  asm("add.rn.bf16x2 %0, %1, %2;" : "=r"(s) : "r"(a), "r"(b));
  return s;
}
template <int ACT>
__device__ __forceinline__ uint32_t act_add_bf16x2_packed(uint32_t a, uint32_t b) {
  if constexpr (ACT == ACT_TANH) {
    return tanh_add_bf16x2_packed(a, b);
  } else if constexpr (ACT == ACT_RELU) {
    uint32_t r;
    asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(add_bf16x2(a, b)), "r"(0u));
    return r;
  } else {
    const uint32_t s = add_bf16x2(a, b);
    return pack_bf16(gelu_f32(__uint_as_float(s << 16)), gelu_f32(__uint_as_float(s & 0xffff0000u)));
  }
}

// Same, pinned in program order (volatile): the producers release a slab stage right behind these - the MUFU issue
// waits for its operands, so every load of the stage has completed by the time the arrive that follows is issued.
// (A plain `asm` may be scheduled below the arrive, which would then overtake the loads.)
__device__ __forceinline__ uint32_t tanh_add_bf16x2_packed_ordered(uint32_t a, uint32_t b) {
  uint32_t s, r;
  asm volatile("add.rn.bf16x2 %0, %1, %2;" : "=r"(s) : "r"(a), "r"(b));
  asm volatile("tanh.approx.bf16x2 %0, %1;" : "=r"(r) : "r"(s));
  return r;
}

// One lane of a converged warp.  Role warps run their loops warp-wide (loop state stays in uniform registers) and
// guard the single-thread instructions (tcgen05.mma/commit, bulk copies) with this: a `lane == 0` branch around the
// whole loop forces every descriptor through R2UR and wraps each UTCHMMA in an ELECT/BRA.U.ANY waterfall, which was
// measured at 2x the MMA time per 4-MMA stage (tools/issue_bench.cu).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .b32 rx;\n.reg .pred px;\nelect.sync rx|px, 0xffffffff;\nselp.u32 %0, 1, 0, px;\n}\n" : "=r"(pred));
  return pred != 0;
}
// One arrival per warp: per-thread arrivals on one mbarrier serialise (256 producer threads x 2 barriers per k-block
// cost ~1500 cycles per k-block in the backward kernel).  Every lane has fenced its own writes before this call.
__device__ __forceinline__ void warp_arrive(uint32_t bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}
// Warp index as a value the compiler knows to be warp-uniform.
__device__ __forceinline__ int uniform_warp_idx() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }
__device__ __forceinline__ void named_barrier_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------------------- host: tensor maps
// cuTensorMapEncodeTiled is fetched through the runtime (no link-time dependency on libcuda).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 2-D bf16 row-major tensor [rows][cols] (cols contiguous, row pitch `pitch_elems`), box [box_rows][64 cols],
// 128-byte swizzle (or none), zero fill out of bounds.
int make_tmap_bf16_2d(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t pitch_elems,
                      uint32_t box_rows, bool swizzle = true);
// 2-D fp32 row-major tensor, box [box_rows][32 cols] (= 128 B), 128-byte swizzle, zero fill out of bounds.
int make_tmap_f32_2d(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t pitch_elems,
                     uint32_t box_rows);

}  // namespace tc
}  // namespace ctcvr
