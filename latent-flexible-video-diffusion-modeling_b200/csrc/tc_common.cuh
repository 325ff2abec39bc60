// tcgen05 / TMA / mbarrier PTX wrappers and the tensor-map encoder shared by the tensor-core kernels.  sm_100a only.
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace fdm {

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// barrier initialisation made visible to the async proxy (TMA, tcgen05.commit) and to the other CTAs of the cluster
__device__ __forceinline__ void fence_mbarrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) { asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory"); }
// TMEM columns (a power of two >= 32) for this CTA (CG = 1) or this CTA pair (CG = 2), allocated by one whole warp; the base address
// is written to `slot` in shared memory.  The allocation permit is relinquished at once, so the next CTA on the SM can allocate.
// tmem_dealloc is issued by the same warp with the same column count.  A compile-time count is passed as an immediate: a register
// operand moves the register allocation of the kernels around it.
template <int CG, uint32_t COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot) {
  static_assert(CG == 1 || CG == 2, "cta_group::1 or ::2");
  if constexpr (CG == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "n"(COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  } else {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "n"(COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
}
template <int CG, uint32_t COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t base) {
  static_assert(CG == 1 || CG == 2, "cta_group::1 or ::2");
  if constexpr (CG == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(COLS));
  else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(COLS));
}
// a column count known at run time, single CTA
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols));
}
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 inputs, fp32 accumulate
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major, 128-byte swizzle, rows of 128 bytes, 8-row atoms 1024 bytes apart (SBO); descriptor version 1 (sm_100)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);          // start address, bits [0,14)
  d |= (uint64_t)1 << 16;                            // leading byte offset (unused for swizzled K-major), bits [16,30)
  d |= (uint64_t)(1024 >> 4) << 32;                  // stride byte offset, bits [32,46)
  d |= (uint64_t)1 << 46;                            // version = 1
  d |= (uint64_t)2 << 61;                            // layout type: SWIZZLE_128B
  return d;
}
// The MMA issuer is ONE thread: its scalar instruction stream paces the tensor pipe (measured: ~110 clk per tcgen05.mma with
// 64-bit descriptor arithmetic in the loop vs 32-64 clk of tensor work).  So descriptors are kept as a constant high word
// and a 32-bit low word (start address >> 4 | LBO) that is advanced with plain 32-bit adds.
constexpr uint32_t SMEM_DESC_HI_SW128 = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO = 1024 B, version 1, SWIZZLE_128B
__device__ __forceinline__ uint32_t smem_desc_lo(uint32_t saddr) { return ((saddr & 0x3FFFFu) >> 4) | (1u << 16); }
// D[tmem] (+)= A * B with descriptors given as (lo, constant hi); `accumulate` is a compile-time-foldable flag
__device__ __forceinline__ void umma_bf16_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t"
      "}" ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(SMEM_DESC_HI_SW128) : "memory");
}

// ---------------------------------------------------------------- CTA pairs (cta_group::2): two SMs of one TPC on one M = 256 tile
// The leader (cluster rank 0) issues the MMAs; each CTA stages its own 128 rows of A and HALF of the B tile (N/2 rows), so the
// operand reads per SM and per MMA drop from A + B to A + B/2.  TMA loads of both CTAs complete on the LEADER's barrier, the
// leader's commits are multicast to both CTAs' barriers.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA loads into THIS CTA's shared memory whose bytes complete on a barrier given by its shared::cluster address
__device__ __forceinline__ void tma_load_4d_cg2(void* dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_3d_cg2(void* dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// arrives on the barrier at this shared-memory offset in BOTH CTAs of the pair once the leader's prior MMAs have completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void umma_bf16_lo_pair(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %3, p;\n\t"
      "}" ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(SMEM_DESC_HI_SW128) : "memory");
}
// kind::f16 instruction descriptor with an explicit M (256 for CTA pairs)
__host__ __device__ constexpr uint32_t make_idesc_mn(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, M=128, N=BN
__host__ __device__ constexpr uint32_t make_idesc(int n, int b_mn_major = 0) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}


__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// One lane of a CONVERGED warp.  tcgen05.mma / TMA take their operands from the uniform datapath; issued under a plain
// `if (lane == 0)` the compiler cannot prove uniformity and wraps every instruction in an ELECT/branch "waterfall" loop
// (seen in SASS: ~9 extra instructions per UTCHMMA).  Keeping the issuing warp converged and predicating on elect.sync
// gives straight-line UTCHMMA / UTMALDG sequences.
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t"
      "}" : "=r"(pred));
  return pred != 0;
}

// generic-proxy writes to shared memory (st.shared) must be fenced before the async proxy (tcgen05.mma / TMA) reads them
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Epilogue store helper.  Out of TMEM a lane owns one ROW (tcgen05.ld 32x32b), so a plain per-lane store writes 32 scattered
// 16-byte pieces per instruction (partial 32-byte sectors at the L2: measured 26.5 -> 20.3 us on the cfg4 qkv linear when
// replaced).  Here the warp transposes 64 bytes per lane through a private staging slice (32 rows x 80-byte pitch: conflict-free
// 16-byte accesses) and stores with 4 lanes per row: every instruction writes 8 whole 64-byte row segments.
//   stage      : 2560 bytes of shared memory private to this warp
//   w[4]       : this lane's 64 bytes (row = lane)
//   row_ptr(r) : global address of row r's 64-byte segment, or nullptr to skip the row;  pieces: 16-byte pieces to store (<= 4)
template <class RowPtr>
__device__ __forceinline__ void warp_store_rows64(uint8_t* stage, int lane, const uint4 (&w)[4], RowPtr row_ptr, int pieces = 4) {
#pragma unroll
  for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(stage + lane * 80 + q * 16) = w[q];
  __syncwarp();
  const int piece = lane & 3;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int row = i * 8 + (lane >> 2);
    uint8_t* d = row_ptr(row);
    if (d != nullptr && piece < pieces) *reinterpret_cast<uint4*>(d + piece * 16) = *reinterpret_cast<const uint4*>(stage + row * 80 + piece * 16);
  }
  __syncwarp();
}

__device__ __forceinline__ uint32_t pack2_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// Encodes a TMA tensor map over bf16 elements at `ptr`: `rank` dims (innermost first) and box sizes, no interleave, zero fill out
// of bounds.  `strides` (rank - 1 byte strides of dims 1..rank-1) default to the dense layout of `dims`, `elem_strides` to 1.
// False when the driver has no encoder or rejects the map.  api.cu
bool encode_bf16_map(CUtensorMap* map, const void* ptr, int rank, const cuuint64_t* dims, const cuuint32_t* box,
                     CUtensorMapL2promotion l2, CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B,
                     const cuuint64_t* strides = nullptr, const cuuint32_t* elem_strides = nullptr);

}  // namespace fdm
