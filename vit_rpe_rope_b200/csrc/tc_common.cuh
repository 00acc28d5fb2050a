// sm_100a primitives used by the tensor-core kernels: mbarrier, TMA (cp.async.bulk[.tensor]),
// tcgen05 (TMEM alloc / mma / commit / ld / st / fences) and the UMMA shared-memory / instruction
// descriptors.  Inline PTX only; descriptor bit layouts follow the PTX ISA "tcgen05 matrix
// descriptor" / "instruction descriptor" tables (cross-checked against CUTLASS's
// cute/arch/mma_sm100_desc.hpp).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace vrr {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier ----------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ---- TMA ---------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
// 2-D tiled load: coordinates are (c0 = innermost element index, c1 = row index).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// 1-D bulk copy global -> shared (16-byte aligned addresses, size multiple of 16).
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// generic-proxy writes to shared memory -> visible to the async proxy (TMA / tcgen05 operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- TMEM --------------------------------------------------------------------------------------
// One full warp calls alloc; the base address (lane 0, first column) lands in *smem_slot.
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// tcgen05.ld / st, shape 32x32b: thread i of warp w <-> TMEM lane 32*(w%4)+i, register j <-> column +j.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// ---- UMMA descriptors -----------------------------------------------------------------------------
// Shared-memory matrix descriptor, SWIZZLE_128B, 8-row x 128-byte atoms stacked every 1024 bytes.
//   bits [0,14)  start address >> 4        bits [16,30) leading byte offset >> 4
//   bits [32,46) stride byte offset >> 4   bits [46,48) descriptor version (1 on sm_100)
//   bits [61,64) layout type (2 = SWIZZLE_128B)
// The same encoding serves a K-major operand whose rows are 64 bf16 (one swizzle atom wide: Q, K,
// X, W tiles) and an MN-major operand whose rows are 64 contiguous MN elements (V: [key][d]); in
// both cases consecutive 8-row groups are 1024 bytes apart (SBO) and LBO is unused.
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(1024 >> 4) << 32;  // SBO
  d |= (uint64_t)1 << 46;            // version
  d |= (uint64_t)2 << 61;            // SWIZZLE_128B
  return d;
}
// Instruction descriptor for kind::f16 with 16-bit A/B (`fmt`: 0 = f16, 1 = bf16) and fp32 accumulation.
//   [4,6) D fmt (1 = f32)  [7,10) A fmt  [10,13) B fmt
//   [15] A major (0 = K)   [16] B major (0 = K, 1 = MN)   [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t idesc_f16kind(uint32_t fmt, int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] . B[smem]
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] . B[smem]
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// All previously issued tcgen05.mma of this thread arrive on `bar` when they complete
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// One lane of the (converged) warp is elected; returns true for it only.  Keeps the operands of the
// instructions issued under it warp-uniform (uniform registers) - the CUTLASS idiom for TMA / MMA issue.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
      "elect.sync rx|px, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, px;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- thread-block clusters / CTA pairs (cta_group::2) ------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// all threads of every CTA in the cluster (warps converged): release / acquire at cluster scope
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa(uint32_t local_smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_cluster(uint32_t cluster_addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(cluster_addr), "r"(bytes)
               : "memory");
}
// Wait on a barrier that also receives arrivals / complete_tx from the peer CTA.  Deliberately the plain
// CTA-scope try_wait: everything these barriers order moves through the async proxy (TMA -> shared memory ->
// tensor core -> TMEM), no generic-proxy data crosses the CTAs, and an `.acquire.cluster` wait makes ptxas emit
// CCTL.IVALL (an L1 invalidate, ~hundreds of cycles) after EVERY wait - measured at 75 % of this kernel's stall
// samples before it was removed (profiles/r2_gemm_pair_cctl.txt).
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) { mbar_wait(bar, parity); }
// 2-D tiled TMA load issued by one CTA of a pair into its OWN shared memory, completing on an mbarrier that
// may live in the peer CTA (`bar_cluster_addr` from mapa) - the operand feed of tcgen05.mma.cta_group::2.
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0,
                                                 int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
// The same through a 3-D map (box [1][rows][cols]): the packed SwiGLU fc1 weight, plane c2 = gate (0) / value (1).
__device__ __forceinline__ void tma_load_3d_pair(void* smem_dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0,
                                                 int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// TMA stores shared -> global (bulk async-group completion)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint32_t ld_shared_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// TMEM allocation / MMA / commit for a CTA pair
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A[smem, 128 rows per CTA] . B[smem, N/2 rows per CTA]   (M = 256)
__device__ __forceinline__ void mma_ss_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of this thread's cta_group::2 MMAs -> one arrival on the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void mma_commit_pair(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(mask)
               : "memory");
}
// General SWIZZLE_128B shared-memory descriptor: lbo = byte distance between 64-element blocks along MN
// (MN-major operands wider than one swizzle atom; ignored for K-major), sbo = byte distance between 8-row groups.
__device__ __forceinline__ uint64_t smem_desc_sw128_ex(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// Register re-partitioning between the warpgroups of a CTA (warps 4g .. 4g+3 execute it together): the TMA / MMA
// issuing warps give registers back, the compute warpgroups take them.  Counts are multiples of 8.
template <int N>
__device__ __forceinline__ void reg_alloc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void reg_dealloc() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// 2^x for two values WITHOUT the MUFU unit: x = n + f with n = round(x) (magic-number add), f in [-0.5, 0.5];
// 2^f by a degree-3 minimax polynomial (relative error 7.5e-5 - P is rounded right after, to bf16 (unit roundoff
// 3.9e-3, a 50x margin) or to fp16 (4.9e-4, a 6x margin)) and n added into the exponent field.  ~5 FMA-pipe instructions per value on the packed fp32x2 pipe: MUFU.EX2 issues 16
// per clock per SM against 32 softmax elements per clock the tensor pipe could consume at head dim 64, so a share
// of the exponentials computed here raises the kernel's MUFU-bound ceiling.
__device__ __forceinline__ float2 ex2_poly2(float2 x) {
  x = make_float2(fmaxf(x.x, -126.f), fmaxf(x.y, -126.f));
  const float2 magic = make_float2(12582912.f, 12582912.f);  // 1.5 * 2^23: the integer lands in the low mantissa bits
  const float2 t = __fadd2_rn(x, magic);
  const float2 n = __fadd2_rn(t, make_float2(-12582912.f, -12582912.f));
  const float2 f = __fadd2_rn(x, make_float2(-n.x, -n.y));
  float2 q = __ffma2_rn(make_float2(0.0551716685f, 0.0551716685f), f, make_float2(0.2426111251f, 0.2426111251f));
  q = __ffma2_rn(q, f, make_float2(0.6932609677f, 0.6932609677f));
  q = __ffma2_rn(q, f, make_float2(0.9999280572f, 0.9999280572f));
  // (bits(t) << 23) == (n << 23) modulo 2^32: the magic constant's low nine bits are zero
  return make_float2(__int_as_float(__float_as_int(q.x) + (__float_as_int(t.x) << 23)),
                     __int_as_float(__float_as_int(q.y) + (__float_as_int(t.y) << 23)));
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// The 16-bit element type of a tensor-core kernel: bf16 or fp16 operands, P / dS in TMEM, and the 16-bit stores.
// Everything that depends on it goes through this struct, so the two instantiations differ only here.
// The conversions round to nearest and overflow to +-inf (never a clamped finite value): a GradScaler step relies
// on an overflowing fp16 gradient becoming non-finite.
template <typename T>
struct Elem16;
template <>
struct Elem16<__nv_bfloat16> {
  static constexpr uint32_t kFmt = 1;  // instruction-descriptor A/B format
  static constexpr CUtensorMapDataType kTmap = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  static __device__ __forceinline__ uint32_t pack2(float lo, float hi) { return pack_bf16(lo, hi); }
  static __device__ __forceinline__ float2 unpack2(uint32_t w) {
    return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w));
  }
  static __device__ __forceinline__ float round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
};
template <>
struct Elem16<__half> {
  static constexpr uint32_t kFmt = 0;
  static constexpr CUtensorMapDataType kTmap = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  static __device__ __forceinline__ uint32_t pack2(float lo, float hi) {
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  static __device__ __forceinline__ float2 unpack2(uint32_t w) { return __half22float2(*reinterpret_cast<const __half2*>(&w)); }
  static __device__ __forceinline__ float round(float x) { return __half2float(__float2half_rn(x)); }
};
template <typename T>
__host__ __device__ constexpr uint32_t idesc_16(int M, int N, int a_mn_major, int b_mn_major) {
  return idesc_f16kind(Elem16<T>::kFmt, M, N, a_mn_major, b_mn_major);
}

}  // namespace tc

// Host: 2-D tensor map over a row-major [rows][cols] buffer of `dtype` (bf16, fp16 or fp32);
// box = [box_rows][box_cols], box_cols * element bytes <= 128; 128-byte swizzle.
int make_tmap_2d(CUtensorMap* map, const void* base, CUtensorMapDataType dtype, uint64_t rows, uint64_t cols,
                 uint64_t row_stride_bytes, uint32_t box_rows, uint32_t box_cols);

// 3-D map of a 16-bit `dtype` over [d2][d1][d0] (d0 innermost, contiguous), box = [1][box1][box0], box0 * 2 <= 128
// bytes, 128-byte swizzle (or none: plain [box1][box0] staging).  Used for [B][N][E] activations and [planes][N][64]
// head planes: a box never crosses an image / head, rows past N are clipped by the hardware (coordinates must not be
// negative).
int make_tmap_3d(CUtensorMap* map, const void* base, CUtensorMapDataType dtype, uint64_t d0, uint64_t d1, uint64_t d2,
                 uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t box0, uint32_t box1, int swizzle128 = 1);

}  // namespace vrr
