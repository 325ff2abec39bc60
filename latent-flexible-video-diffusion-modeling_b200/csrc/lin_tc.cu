// Attention-block linears with the GroupNorm in the operand path (tcgen05.mma, persistent CTAs, weights resident in shared memory,
// outputs written by TMA stores).
//
// Reference call sites (rpe.py:111-113,135-140,170-173): every RPEAttention does
//     x = norm(x);  qkv = self.qkv(x);  ... attention ...;  return x + self.proj_out(h)
// i.e. a GroupNorm, a C -> 3C linear, and a C -> C linear whose residual is the NORMALISED input.  As separate kernels that is a
// normalisation pass (fp32 in, fp32 + bf16 out), a GEMM of 960 one-shot CTAs, and a second GEMM re-reading the fp32 normalised
// tensor.  Here the normalised tensor never exists in memory:
//   * nl_qkv_kernel : A-operand tiles are built IN shared memory from the raw fp32 activations (one TMA box per tile -> GroupNorm
//       scale/shift -> bf16, 128-byte-swizzled K-major rows) and multiplied with W_qkv, which stays resident for the CTA's life.
//       a_mode 1 = per-frame GroupNorm from the (sum, sum of squares) pairs the producing kernel's epilogue left behind;
//       a_mode 2 = the temporal GroupNorm (statistics over C/32 channels x T frames per (video, pixel)) computed in the tile itself:
//       a tile is PL pixels x all T frames, ONE 4-D TMA box of the [B*T][HW][C] tensor, rows ordered (frame, pixel).
//   * proj_out keeps the per-tap conv kernel (conv_tc.cu); its epilogue RECOMPUTES the residual GN(x) from x and the saved
//       statistics (fdm_conv_args.resid_norm 2: the per-(pixel, group) mean / rstd this kernel's a_mode 2 launch writes;
//       3: the per-frame sums).  A persistent proj kernel of this file's design (TMA-fetched residual tile, result formed in
//       place, TMA or row-per-lane stores) was measured at 19-22 us against 13.6 us for the per-tap kernel at the cfg4 16x16
//       shape and was dropped.
// Structure (the first version was warp-specialised — 4 transform + 8 epilogue warps — and every CUDA-core phase was latency-bound:
// 4.5-6 us per tile in the transform, 4 us in the epilogue, profiles/r02_nl_trace_v1.txt): ALL 8 worker warps do the transform, then
// ALL do the epilogue; one elected lane of warp 0 issues the MMAs.  What the per-phase traces (tools/nl_trace.py) showed on the way:
//   * an SM drains its stores at ~15 bytes/clk whatever the instruction (TMA store, coalesced or row-per-lane STG): the 96 KB of
//     a [128 x 384] bf16 tile take ~3.2 us, so the kernel is bound by its OUTPUT and the drain has to overlap everything else;
//   * row-per-lane 16-byte global stores straight from the TMEM registers (32 different lines per instruction) back up the LSU:
//     ~220 clk per STG, 5.7 us per tile;
//   * TMA stores from a 2-deep staging ring serialise on the bulk-group wait: 2.8-3.6 us per tile with nothing overlapped.
// So: the WHOLE output tile has its own staging (6 blocks of [128 rows x 64 columns], SWIZZLE_128B), each block leaves by one
// TMA store as soon as its four warps have written it, and nothing waits for a store of the current tile; the raw rows of the
// next tile are fetched into REGISTERS (coalesced 512-byte rows, in flight under the MMAs and the epilogue) because the staging
// took the shared memory a raw tile would need.
// Shapes: K = C = 128 (two 64-channel chunks; a GroupNorm group = 4 channels = one float4), Cout = 128 / 256 / 384, HW % 16 == 0,
// a_mode 2: T <= 20 (a pixel's T rows live in one warp's registers).
#include "tc_common.cuh"
#include <mutex>

namespace fdm {

constexpr int NL_WORKERS = 256;             // 8 worker warps
constexpr int NL_K = 128;
constexpr int NL_A_BYTES = 2 * 16384;       // [2 chunks][128 rows][128 B]

struct NlParams {
  const float* x;
  const double* stats;
  float* tstats;
  const float* gamma;
  const float* beta;
  const float* bias;
  __nv_bfloat16* y_op;
  int M, B, T, HW, Cout, NS;
  int a_mode;
  int PL, tpv, tiles;  // a_mode 2: pixels per tile, tiles per video
  float eps;
  double inv_cnt;  // 1 / (4 * HW), divided on the host
  long long* trace;  // debug: per-CTA phase timestamps (clock64), NULL in production (fdm_debug_nl_trace)
};

#define NL_TRACE(slot)                                                                        \
  do {                                                                                        \
    if (p.trace != nullptr && (slot) < 64) p.trace[blockIdx.x * 64 + (slot)] = clock64();     \
  } while (0)

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(map), "r"(smem_u32(src)),
               "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(map), "r"(smem_u32(src)),
               "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32_async(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void named_bar(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// per-frame GroupNorm scale / shift of the 4 channels [c, c+4) (= one group at C = 128) from the fp64 sums
__device__ __forceinline__ void nl_frame_coefs(const double* stats, int n, int c, double inv_cnt, float eps, const float4& g4, const float4& b4,
                                               float (&mul)[4], float (&add)[4]) {
  const double2* st = reinterpret_cast<const double2*>(stats + ((size_t)n * NL_K + c) * 2);
  const double2 s0 = st[0], s1 = st[1], s2 = st[2], s3 = st[3];
  const double mean = (s0.x + s1.x + s2.x + s3.x) * inv_cnt;
  const double var = fmax((s0.y + s1.y + s2.y + s3.y) * inv_cnt - mean * mean, 0.0);
  const float mf = (float)mean, rs = rsqrtf((float)var + eps);  // fp64 only for E[x^2] - mean^2
  mul[0] = g4.x * rs; mul[1] = g4.y * rs; mul[2] = g4.z * rs; mul[3] = g4.w * rs;
  add[0] = b4.x - mf * mul[0]; add[1] = b4.y - mf * mul[1]; add[2] = b4.z - mf * mul[2]; add[3] = b4.w - mf * mul[3];
}

// ------------------------------------------------------------------------------------------------------------------------
// qkv: y_op[M][Cout] (bf16) = GN(x) . W^T + bias
// ------------------------------------------------------------------------------------------------------------------------
constexpr int NL_XR = 24;                   // raw rows a transform thread holds in registers (a_mode 1: 16; a_mode 2: T <= 24)
constexpr int NL_STG_BLOCK = 128 * 128;     // bf16 [128 rows][64 cols], SWIZZLE_128B: one TMA store

__global__ void __launch_bounds__(NL_WORKERS, 1) nl_qkv_kernel(const __grid_constant__ CUtensorMap tw, const __grid_constant__ CUtensorMap ty,
                                                              const NlParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t w_bar, a_ready, mma_bar[3];
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(16) float bias_s[384];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w_bytes = p.Cout * NL_K * 2;
  uint8_t* w_s = smem;                     // [2 chunks][Cout rows][128 B]
  uint8_t* a_s = w_s + w_bytes;            // [2 chunks][128 rows][128 B]
  uint8_t* stg_s = a_s + NL_A_BYTES;       // [Cout / 64 blocks][128 rows][128 B]: the whole output tile, drained by TMA stores

  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tw) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&ty) : "memory");
    mbar_init(&w_bar, 1);
    mbar_init(&a_ready, 8);
    for (int i = 0; i < 3; ++i) mbar_init(&mma_bar[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "n"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  for (int i = threadIdx.x; i < p.Cout; i += NL_WORKERS) bias_s[i] = p.bias[i];  // parameters: not written by the previous kernel
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_slot;
  if (threadIdx.x == 0) NL_TRACE(0);

  {
    // weights: issued before griddepcontrol.wait (they do not depend on the previous kernel)
    if (warp == 0 && elect_one_sync()) {
      mbar_expect_tx(&w_bar, (uint32_t)w_bytes);
      for (int c = 0; c < 2; ++c)
        for (int n0 = 0; n0 < p.Cout; n0 += 128) tma_load_3d(w_s + c * p.Cout * 128 + n0 * 128, &tw, &w_bar, c * 64, n0, 0);
    }
    __syncwarp();
    // ===================== workers: transform (raw rows held in registers, fetched one tile ahead), then epilogue
    pdl_wait();
    const int g = warp >> 2, q = warp & 3;
    const int c4 = lane * 4;  // this lane's 4 channels = one GroupNorm group (C = 128)
    const float4 g4 = __ldg(reinterpret_cast<const float4*>(p.gamma + c4));
    const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.beta + c4));
    // destination of this lane's 8 bytes inside an A row: chunk lane/16, 16-byte piece (lane%16)/2 (XOR row%8), half lane%2
    const uint32_t d_chunk = (uint32_t)(lane >> 4) * 16384u, d_piece = (uint32_t)((lane & 15) >> 1), d_half = (uint32_t)(lane & 1) * 8u;
    const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
    const int erow = q * 32 + lane;  // this thread's row of the tile in the epilogue
    const uint32_t e_sw = (uint32_t)(erow & 7);
    const bool leader = (q == 0 && lane == 0);  // issues this group's TMA stores (bulk groups are per thread)
    // a_mode 1: this warp transforms rows [16 warp, 16 warp + 16) (HW % 16 == 0: one frame); a_mode 2: all T rows of pixel `warp`
    const int nrows = p.a_mode == 1 ? 16 : (warp < p.PL ? p.T : 0);
    float4 xr[NL_XR];
    float mul[4] = {0.f, 0.f, 0.f, 0.f}, add[4] = {0.f, 0.f, 0.f, 0.f};
    auto fetch = [&](int tile) {  // this thread's raw values of `tile` (coalesced: a warp reads whole 512-byte rows) + its statistics
      if (p.a_mode == 1) {
        const int m0 = tile * 128 + warp * 16;
        const bool ok = m0 < p.M;
        const float* src = p.x + (size_t)m0 * NL_K + c4;
#pragma unroll
        for (int i = 0; i < 16; ++i) xr[i] = ok ? __ldg(reinterpret_cast<const float4*>(src + i * NL_K)) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok) nl_frame_coefs(p.stats, m0 / p.HW, c4, p.inv_cnt, p.eps, g4, b4, mul, add);
      } else {
        const int vb = tile / p.tpv, px = (tile - vb * p.tpv) * p.PL + warp;
        const bool ok = warp < p.PL && px < p.HW;
        const float* src = p.x + ((size_t)vb * p.T * p.HW + px) * NL_K + c4;
        const size_t fstride = (size_t)p.HW * NL_K;
#pragma unroll
        for (int i = 0; i < NL_XR; ++i)
          xr[i] = (ok && i < p.T) ? __ldg(reinterpret_cast<const float4*>(src + i * fstride)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    // Work items are (tile, 128-column slice) pairs, handed out as contiguous ranges: 320 tiles over 148 CTAs quantise to 3 vs
    // 2.16 tiles (the kernel is bound by what each SM has to store), 960 slices to 7 vs 6.5.  A tile that straddles two CTAs is
    // transformed by both; each computes and stores only its own slices.
    const int items = p.tiles * p.NS;
    const int item_lo = (int)(((long long)blockIdx.x * items) / gridDim.x);
    const int item_hi = (int)(((long long)(blockIdx.x + 1) * items) / gridDim.x);
    const int tile_lo = item_lo / p.NS, tile_hi = (item_hi + p.NS - 1) / p.NS;  // tiles [tile_lo, tile_hi)
    uint32_t mma_ph = 0;  // bit j: parity of the next completion of mma_bar[j]
    if (tile_lo < tile_hi) fetch(tile_lo);
    int it = 0;
    for (int tile = tile_lo; tile < tile_hi; ++tile, ++it) {
      const int j_lo = tile == tile_lo ? item_lo - tile * p.NS : 0;
      const int j_hi = min(p.NS, item_hi - tile * p.NS);
      if (threadIdx.x == 0) NL_TRACE(8 + 8 * it + 0);
      if (p.a_mode == 1) {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int row = warp * 16 + i;
          uint2 o;
          o.x = pack2_bf16(fmaf(xr[i].x, mul[0], add[0]), fmaf(xr[i].y, mul[1], add[1]));
          o.y = pack2_bf16(fmaf(xr[i].z, mul[2], add[2]), fmaf(xr[i].w, mul[3], add[3]));
          *reinterpret_cast<uint2*>(a_s + d_chunk + row * 128 + ((d_piece ^ (uint32_t)(row & 7)) << 4) + d_half) = o;
        }
      } else if (nrows > 0) {
        // statistics of (pixel, group lane) over the T frames around a pivot (the group's first value), two accumulator pairs
        const float pivot = xr[0].x;
        float sa = 0.f, sb = 0.f, qa = 0.f, qb = 0.f;
#pragma unroll
        for (int i = 0; i < NL_XR; i += 2) {
          if (i < p.T) {
            const float d0 = xr[i].x - pivot, d1 = xr[i].y - pivot, d2 = xr[i].z - pivot, d3 = xr[i].w - pivot;
            sa += (d0 + d1) + (d2 + d3);
            qa = fmaf(d0, d0, qa); qa = fmaf(d1, d1, qa); qa = fmaf(d2, d2, qa); qa = fmaf(d3, d3, qa);
          }
          if (i + 1 < p.T) {
            const float e0 = xr[i + 1].x - pivot, e1 = xr[i + 1].y - pivot, e2 = xr[i + 1].z - pivot, e3 = xr[i + 1].w - pivot;
            sb += (e0 + e1) + (e2 + e3);
            qb = fmaf(e0, e0, qb); qb = fmaf(e1, e1, qb); qb = fmaf(e2, e2, qb); qb = fmaf(e3, e3, qb);
          }
        }
        const float cnt = 4.f * (float)p.T;
        const float md = (sa + sb) / cnt;
        const float mean = pivot + md, rstd = rsqrtf(fmaxf((qa + qb) / cnt - md * md, 0.f) + p.eps);
        const int vb = tile / p.tpv, px = (tile - vb * p.tpv) * p.PL + warp;
        if (p.tstats != nullptr && px < p.HW)
          *reinterpret_cast<float2*>(p.tstats + (((size_t)vb * p.HW + px) * 32 + lane) * 2) = make_float2(mean, rstd);
#pragma unroll
        for (int i = 0; i < NL_XR; ++i) {
          if (i < p.T) {
            const int row = i * p.PL + warp;  // rows of the tile are ordered (frame, pixel)
            uint2 o;
            o.x = pack2_bf16((xr[i].x - mean) * rstd * g4.x + b4.x, (xr[i].y - mean) * rstd * g4.y + b4.y);
            o.y = pack2_bf16((xr[i].z - mean) * rstd * g4.z + b4.z, (xr[i].w - mean) * rstd * g4.w + b4.w);
            *reinterpret_cast<uint2*>(a_s + d_chunk + row * 128 + ((d_piece ^ (uint32_t)(row & 7)) << 4) + d_half) = o;
          }
        }
      }
      fence_proxy_async_smem();  // the A tile is read by the tensor core (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(&a_ready);
      if (threadIdx.x == 0) NL_TRACE(8 + 8 * it + 1);

      // the next tile's raw rows: in flight under the MMAs and the epilogue
      if (tile + 1 < tile_hi) fetch(tile + 1);

      if (warp == 0) {
        // MMA issue (one elected lane of warp 0; 8 warps keep the register budget at 255 per thread — a ninth, control-only warp
        // capped it at 168 and the 20 raw rows spilled): once every warp's part of A is in place and the previous tile's
        // accumulators have been drained
        if (it == 0) mbar_wait(&w_bar, 0);
        mbar_wait(&a_ready, it & 1);
        if (lane == 0) NL_TRACE(8 + 8 * it + 2);
        tcgen05_fence_after();
        if (elect_one_sync()) {
          constexpr uint32_t idesc = make_idesc(128);
          const uint32_t a_lo = smem_desc_lo(smem_u32(a_s));
          for (int j = j_lo; j < j_hi; ++j) {
            const uint32_t d = tmem_base + j * 128;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              const uint32_t al = a_lo + c * (16384 >> 4);
              const uint32_t bl = smem_desc_lo(smem_u32(w_s + c * p.Cout * 128 + j * 128 * 128));
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) umma_bf16_lo(d, al + 2 * kk, bl + 2 * kk, idesc, (c | kk) != 0);
            }
            umma_commit(&mma_bar[j]);
          }
        }
        __syncwarp();
        if (lane == 0) NL_TRACE(8 + 8 * it + 3);
      }

      // ---- epilogue: group g takes the 64-column half g of every 128-column slice: + bias -> bf16 -> this thread's 128-byte row
      // of the block (SWIZZLE_128B) -> group barrier -> ONE TMA store of the [128 rows x 64 columns] block.  The whole output
      // tile has its own staging, so nothing here waits for a store of THIS tile; the stores of the previous tile (issued a tile
      // ago) must have been read before the first block is overwritten.
      if (leader) bulk_wait_read0();
      named_bar(1 + g, 128);
      const int vb = p.a_mode == 2 ? tile / p.tpv : 0;
      const int px0 = p.a_mode == 2 ? (tile - vb * p.tpv) * p.PL : 0;
      for (int j = j_lo; j < j_hi; ++j) {
        const int gcol = j * 128 + g * 64;
        mbar_wait(&mma_bar[j], (mma_ph >> j) & 1);
        mma_ph ^= 1u << j;
        if (threadIdx.x == 0 && j == j_lo) NL_TRACE(8 + 8 * it + 4);
        tcgen05_fence_after();
        uint8_t* blk = stg_s + (j * 2 + g) * NL_STG_BLOCK;
        uint8_t* myrow = blk + erow * 128;
#pragma unroll
        for (int h = 0; h < 2; ++h) {  // one 32-column chunk at a time (the TMEM read itself takes ~30 clk: measured)
          uint32_t v[32];
          tmem_ld_32x32b_x32(trow + gcol + 32 * h, v);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float4 b0 = *reinterpret_cast<const float4*>(bias_s + gcol + 32 * h + 8 * k);
            const float4 b1 = *reinterpret_cast<const float4*>(bias_s + gcol + 32 * h + 8 * k + 4);
            uint4 w;
            w.x = pack2_bf16(__uint_as_float(v[8 * k]) + b0.x, __uint_as_float(v[8 * k + 1]) + b0.y);
            w.y = pack2_bf16(__uint_as_float(v[8 * k + 2]) + b0.z, __uint_as_float(v[8 * k + 3]) + b0.w);
            w.z = pack2_bf16(__uint_as_float(v[8 * k + 4]) + b1.x, __uint_as_float(v[8 * k + 5]) + b1.y);
            w.w = pack2_bf16(__uint_as_float(v[8 * k + 6]) + b1.z, __uint_as_float(v[8 * k + 7]) + b1.w);
            *reinterpret_cast<uint4*>(myrow + (((uint32_t)(4 * h + k) ^ e_sw) << 4)) = w;
          }
        }
        fence_proxy_async_smem();
        named_bar(1 + g, 128);
        if (leader) {
          if (p.a_mode == 2) tma_store_4d(&ty, blk, gcol, px0, 0, vb);
          else tma_store_3d(&ty, blk, gcol, tile * 128, 0);
          bulk_commit();
        }
      }
      tcgen05_fence_before();  // orders this tile's TMEM reads before the arrive on a_ready of the next tile
      if (threadIdx.x == 0) NL_TRACE(8 + 8 * it + 5);
    }
    if (leader) bulk_wait_read0();  // shared memory must outlive the stores' reads; grid completion orders the writes themselves
  }
  tcgen05_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) NL_TRACE(3);
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512));
  }
}

// ---------------------------------------------------------------------------------------------------------------- host
static bool nl_encode(CUtensorMap* m, CUtensorMapDataType dt, const void* ptr, int rank, const cuuint64_t* dims,
                      const cuuint64_t* strides, const cuuint32_t* box, CUtensorMapSwizzle swz) {
  EncodeTiledFn enc = get_tensormap_encoder();
  if (!enc) return false;
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return enc(m, dt, rank, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
             CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static long long* g_nl_trace = nullptr;

// pixels per a_mode 2 tile: one pixel per worker warp (its T rows live in that warp's registers), PL * T rows <= 128
static int nl_pixels_per_tile(int T, int HW) {
  if (T > NL_XR) return 0;
  int pl = 128 / T;
  if (pl > 8) pl = 8;
  if (pl > HW) pl = HW;
  return pl;
}

int norm_linear_supported(const fdm_norm_linear_args* a) {
  if (a->K != NL_K || a->Cout % 128 != 0 || a->Cout < 128 || a->Cout > 384) return 0;
  if (a->B <= 0 || a->T <= 0 || a->HW <= 0 || a->HW % 16 != 0) return 0;
  if (a->a_mode != 1 && a->a_mode != 2) return 0;
  if (a->a_mode == 2 && nl_pixels_per_tile(a->T, a->HW) < 1) return 0;
  return 1;
}

}  // namespace fdm

// debug hook (not part of the public header): device buffer of 148 x 64 clock64 stamps filled by the next launches, or NULL
extern "C" void fdm_debug_nl_trace(void* device_buf) { fdm::g_nl_trace = reinterpret_cast<long long*>(device_buf); }

extern "C" int fdm_norm_linear_supported(const fdm_norm_linear_args* a) { return a ? fdm::norm_linear_supported(a) : 0; }

extern "C" int fdm_norm_linear(const fdm_norm_linear_args* a, void* stream) {
  using namespace fdm;
  FDM_REQUIRE(a && a->w && a->bias && a->x && a->gamma && a->beta && a->y_op, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(norm_linear_supported(a), FDM_ERR_UNSUPPORTED);
  if (a->a_mode == 1) FDM_REQUIRE(a->stats != nullptr, FDM_ERR_BAD_ARG);
  NlParams p;
  p.x = a->x; p.stats = a->stats; p.tstats = a->tstats; p.gamma = a->gamma; p.beta = a->beta; p.bias = a->bias;
  p.y_op = reinterpret_cast<__nv_bfloat16*>(a->y_op);
  p.B = a->B; p.T = a->T; p.HW = a->HW; p.Cout = a->Cout; p.NS = a->Cout / 128;
  p.M = a->B * a->T * a->HW;
  p.a_mode = a->a_mode; p.eps = a->eps;
  p.inv_cnt = 1.0 / (4.0 * (double)a->HW);
  p.trace = g_nl_trace;
  p.PL = 1; p.tpv = 1;
  if (a->a_mode == 2) {
    p.PL = nl_pixels_per_tile(a->T, a->HW);
    p.tpv = (a->HW + p.PL - 1) / p.PL;
    p.tiles = a->B * p.tpv;
  } else {
    p.tiles = (p.M + 127) / 128;
  }
  const CUtensorMapDataType BF = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  CUtensorMap tw, ty;
  {
    cuuint64_t dims[3] = {(cuuint64_t)NL_K, (cuuint64_t)a->Cout, 1};
    cuuint64_t strides[2] = {(cuuint64_t)NL_K * 2, (cuuint64_t)a->Cout * NL_K * 2};
    cuuint32_t box[3] = {64, 128, 1};
    FDM_REQUIRE(nl_encode(&tw, BF, a->w, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B), FDM_ERR_UNSUPPORTED);
  }
  if (a->a_mode == 1) {
    cuuint64_t ydims[3] = {(cuuint64_t)a->Cout, (cuuint64_t)p.M, 1};
    cuuint64_t ystrides[2] = {(cuuint64_t)a->Cout * 2, (cuuint64_t)p.M * a->Cout * 2};
    cuuint32_t ybox[3] = {64, 128, 1};
    FDM_REQUIRE(nl_encode(&ty, BF, a->y_op, 3, ydims, ystrides, ybox, CU_TENSOR_MAP_SWIZZLE_128B), FDM_ERR_UNSUPPORTED);
  } else {
    // [B*T][HW][Cout] as (channel, pixel, frame, video): a tile = PL pixels x all T frames of one video, rows ordered (frame, pixel)
    cuuint64_t ydims[4] = {(cuuint64_t)a->Cout, (cuuint64_t)a->HW, (cuuint64_t)a->T, (cuuint64_t)a->B};
    cuuint64_t ystrides[3] = {(cuuint64_t)a->Cout * 2, (cuuint64_t)a->HW * a->Cout * 2, (cuuint64_t)a->T * a->HW * a->Cout * 2};
    cuuint32_t ybox[4] = {64, (cuuint32_t)p.PL, (cuuint32_t)a->T, 1};
    FDM_REQUIRE(nl_encode(&ty, BF, a->y_op, 4, ydims, ystrides, ybox, CU_TENSOR_MAP_SWIZZLE_128B), FDM_ERR_UNSUPPORTED);
  }
  constexpr int SMEM_MAX = 225 * 1024;  // + ~1.6 KB of static shared memory (barriers, bias) <= 227 KB
  const int smem = a->Cout * NL_K * 2 + NL_A_BYTES + (a->Cout / 64) * NL_STG_BLOCK + 1024;
  FDM_REQUIRE(smem <= SMEM_MAX, FDM_ERR_UNSUPPORTED);
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] { attr_err = cudaFuncSetAttribute(nl_qkv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_MAX); });
  if (attr_err != cudaSuccess) {
    set_last_error(attr_err);
    return FDM_ERR_CUDA;
  }
  const int items = p.tiles * p.NS;
  const int grid = items < 148 ? items : 148;
  fdm::launch(nl_qkv_kernel, dim3(grid), dim3(NL_WORKERS), (size_t)smem, reinterpret_cast<cudaStream_t>(stream), tw, ty, p);
  return check_launch();
}
