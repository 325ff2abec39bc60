// 3x3 stride-1 convolution as implicit GEMM on tcgen05 — the "halo" kernel for the feature maps that carry the FLOPs
// (W in {16,32,64,128}: whole image rows per M tile).  Same math / epilogue contract as conv_tc.cu, different data movement.
//
// Why: conv_tc.cu re-loads the A operand once per filter tap (9 x 16 KB per 128-pixel tile) and its B tile once per
// CTA; measured with in-kernel timestamps the main loop runs at the SM's L2->shared-memory ingest rate (~64 B/clk),
// 4-5x slower than the MMAs need.  Here one persistent CTA per SM computes TWO vertically adjacent 128-pixel M tiles:
//   * per (64-channel chunk, filter column s) ONE TMA box of (2*hbox + 2) full image rows is loaded, shifted by s-1
//     in w (hardware zero-fill = padding).  Because the rows are full width, the three filter rows r = 0,1,2 of both
//     M tiles are just 1024-byte-aligned offsets into that box ((j*hbox + r) * W pixels), addressed by the UMMA
//     shared-memory descriptor: 6 A operands from one load (A traffic / 2.4-3.6).
//   * the three weight tiles (r = 0,1,2 for this s) are shared by both M tiles (B traffic / 2).
//   * accumulators: 2 tiles x BN columns, double-buffered in TMEM (up to 512 columns), so the epilogue of work item i
//     overlaps the main loop of item i+1 inside the same CTA (warp-specialised: TMA / MMA / 4 epilogue warps).
//   * GroupNorm statistics: per-warp column sums are combined across the 4 epilogue warps and both tiles in shared
//     memory before the fp64 atomics (8x fewer atomics than one per warp).
//   * nearest x2 upsample + 3x3 conv (unet.py:85-93) WITHOUT the upsampled tensor: output pixel (2y+a, 2x+b) only sees a 2x2
//     neighbourhood of the low-resolution input, with the 3x3 weights that land on the same input pixel pre-summed (fp32, then bf16)
//     per output phase (a, b).  A work item is (tiles, N tile, phase): a 2x2-tap conv over the low-resolution rows whose rows are
//     stored to the phase's pixels of the output — 4/9 of the MMAs of the conv on the upsampled tensor, a 4x smaller operand.
//   * CG = 2 (CTA pairs, `cta_group::2`): the two CTAs of a cluster run two such work items (different rows / frames, SAME output
//     channels) as ONE stream of M = 256 MMAs issued by the leader.  Each CTA stages its own A box and only HALF of the weight
//     tile (BN/2 rows per tap): single-CTA MMAs at N <= 128 are bound by shared-memory operand reads (A + B per MMA, measured
//     86 clk per 128x128x16 against a tensor floor of 64); the pair reads A + B/2 per SM and halves the weight TMA traffic.
// This kernel does not release its dependents after its dependency wait (common.cuh, pdl_wait_only): it is ONE wave of persistent
// CTAs, so the release would come at kernel start and the next kernel's CTAs would sit on the SMs for the whole run (measured: +4 %
// on the cfg5 / cfg3 steps).
#include "tc_common.cuh"
#include <mutex>

namespace fdm {

constexpr int HALO_THREADS = 320;  // TMA warp, MMA warp, 8 epilogue warps
constexpr int HALO_MAX_STAGES = 4;

struct HaloParams {
  const float* bias;
  const float* resid;
  float* y_f32;
  __nv_bfloat16* y_op;
  double* stats;
  int Cout, W, HW, hbox;
  int pairs_per_frame, n_items, ntiles;
  int kchunks0, kchunks1, klast0, klast1;
  int stages, a_bytes, stage_bytes;
  int tpi;       // M tiles per work item: 2 (B shared by two tiles) or 1 (finer items when 2-tile items quantise badly on 148 SMs)
  int a_bytes0;  // bytes of the segment-0 A box ((2*hbox + ks - 1) rows); a_bytes is the slot size
  int ks;  // filter size 3 (row halo of 2), 1 (pointwise: no halo, one 'column', one 'row') or 2 (the per-phase filter of `up`)
  int up, nph, H, log2W;  // up: nearest-x2-upsample mode, nph = 4 output phases per tile set (else 1)
  long long* trace;  // debug (fdm_debug_set_trace): per-CTA cycle counters, NULL in production
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

template <int BN, int TPI, int CG, bool UP>
__global__ void __launch_bounds__(HALO_THREADS, 1) conv_halo_kernel(const __grid_constant__ CUtensorMap ta0,
                                                                   const __grid_constant__ CUtensorMap tw0,
                                                                   const __grid_constant__ CUtensorMap ta1,
                                                                   const __grid_constant__ CUtensorMap tw1,
                                                                   const HaloParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t full_bar[HALO_MAX_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[HALO_MAX_STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_slot;
  constexpr int TMEM_COLS = 4 * BN;  // 2 accumulator buffers x 2 M tiles
  constexpr int B_TAP_BYTES = (BN / CG) * 128;  // a CTA of a pair stages its half of the weight tile's rows
  const uint32_t rank = CG == 2 ? cluster_ctarank() : 0u;
  const int cid = CG == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;        // work-item stream of this CTA (pair)
  const int cstride = CG == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int n_q = p.n_items / CG;
  // work item of this CTA for stream position q: the CTAs of a pair take the item pairs 2k, 2k+1 of the SAME N tile
  // (with `up` an N tile comes in 4 phases: per_pair = ntiles * nph items share the tiles, the pair CTAs take the same one of them)
  const int per_pair = p.ntiles * p.nph;
  auto item_of = [&](int q) { return CG == 2 ? ((2 * (q / per_pair) + (int)rank) * per_pair + q % per_pair) : q; };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* staging = reinterpret_cast<float*>(smem + (size_t)p.stages * p.stage_bytes);  // [8 warps][32][16], XOR-swizzled
  float* statbuf = staging + 8 * 32 * 16;                                              // [2 buffers][2 tiles][4 lane groups][BN][2]

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&ta0) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tw0) : "memory");
    if (p.kchunks1) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&ta1) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tw1) : "memory");
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full_bar[i], 1);
      mbar_init(&tmem_empty_bar[i], 8 * CG);  // one arrival per epilogue warp (of both CTAs: the leader's copy is the live one)
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    if (CG == 2) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "n"(TMEM_COLS));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "n"(TMEM_COLS));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (CG == 2) cluster_sync_all();  // the peer's barriers are initialised before anything signals them
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_base_slot;
  pdl_wait_only();  // everything above (barriers, TMEM, tensor-map prefetch) overlapped the previous kernel's tail

  if (warp == 0) {
    // ===================== TMA producer (whole warp converged; one elected lane issues) =====================
    {
      uint32_t it = 0;
      const uint32_t full0 = CG == 2 ? mapa_u32(smem_u32(&full_bar[0]), 0) : 0u;  // the leader's full barriers (pairs)
      const int b_row = CG == 2 ? (int)rank * (BN / 2) : 0;                         // this CTA's rows of the weight tile
      for (int q = cid; q < n_q; q += cstride) {
        const int item = item_of(q);
        const int pair = item / per_pair, rest = item - pair * per_pair;
        const int phase = rest % p.nph, n_off = (rest / p.nph) * BN;
        const int n = pair / p.pairs_per_frame, h0 = (pair - n * p.pairs_per_frame) * TPI * p.hbox;
        // up: phase (a, b) reads input rows y + {a-1, a} and columns x + {b-1, b}; its 4 taps are rows phase*4 .. +3 of the weights
        const int pad = UP ? 1 - (phase >> 1) : p.ks >> 1, pad_x = UP ? 1 - (phase & 1) : p.ks >> 1;
        const int tap0 = phase * 4;
        for (int kc = 0; kc < p.kchunks0; ++kc) {
          for (int s = 0; s < p.ks; ++s, ++it) {
            const int stage = it % p.stages;
            mbar_wait(&empty_bar[stage], ((it / p.stages) & 1) ^ 1);
            uint8_t* a_dst = smem + (size_t)stage * p.stage_bytes;
            uint8_t* b_dst = a_dst + p.a_bytes;
            if (elect_one_sync()) {
              // weights are packed filter-column major ([s][r][co][ci]): the three filter rows of column s are ONE box
              // (a TMA instruction costs ~450 clk + 0.4 clk/row on this part, measured: tools/tma_bench.cu)
              if (CG == 2) {
                if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * (p.a_bytes0 + p.ks * B_TAP_BYTES));  // both CTAs' bytes
                tma_load_4d_cg2(a_dst, &ta0, full0 + stage * 8, kc * 64, s - pad_x, h0 - pad, n);
                tma_load_3d_cg2(b_dst, &tw0, full0 + stage * 8, kc * 64, n_off + b_row, tap0 + s * p.ks);
              } else {
                mbar_expect_tx(&full_bar[stage], p.a_bytes0 + p.ks * B_TAP_BYTES);
                tma_load_4d(a_dst, &ta0, &full_bar[stage], kc * 64, s - pad_x, h0 - pad, n);
                tma_load_3d(b_dst, &tw0, &full_bar[stage], kc * 64, n_off, tap0 + s * p.ks);
              }
            }
            __syncwarp();
          }
        }
        for (int kc = 0; kc < p.kchunks1; ++kc, ++it) {
          const int stage = it % p.stages;
          mbar_wait(&empty_bar[stage], ((it / p.stages) & 1) ^ 1);
          uint8_t* a_dst = smem + (size_t)stage * p.stage_bytes;
          if (elect_one_sync()) {
            if (CG == 2) {
              if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * (TPI * 128 * 128 + B_TAP_BYTES));
              tma_load_4d_cg2(a_dst, &ta1, full0 + stage * 8, kc * 64, 0, h0, n);
              tma_load_3d_cg2(a_dst + p.a_bytes, &tw1, full0 + stage * 8, kc * 64, n_off + b_row, 0);
            } else {
              mbar_expect_tx(&full_bar[stage], TPI * 128 * 128 + B_TAP_BYTES);
              tma_load_4d(a_dst, &ta1, &full_bar[stage], kc * 64, 0, h0, n);
              tma_load_3d(a_dst + p.a_bytes, &tw1, &full_bar[stage], kc * 64, n_off, 0);
            }
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp converged; one elected lane issues; pairs: the leader CTA only) =====================
    if (CG == 1 || rank == 0) {
      constexpr uint32_t idesc = make_idesc_mn(128 * CG, BN);
      auto mma = [](uint32_t d, uint32_t a_lo, uint32_t b_lo, uint32_t acc) {
        if (CG == 2) umma_bf16_lo_pair(d, a_lo, b_lo, idesc, acc);
        else umma_bf16_lo(d, a_lo, b_lo, idesc, acc);
      };
      auto commit = [](uint64_t* bar) {
        if (CG == 2) umma_commit_pair(bar);
        else umma_commit(bar);
      };
      const uint32_t row16 = ((uint32_t)p.W * 128) >> 4;         // one image row of the A box, in descriptor units (16 B)
      const uint32_t tile_rows16 = (uint32_t)p.hbox * row16;     // second M tile starts hbox rows further down
      uint32_t it = 0, local = 0;
      long long t_wait_tmem = 0, t_wait_full = 0, t_begin = clock64();
      for (int q = cid; q < n_q; q += cstride, ++local) {
        const uint32_t buf = local & 1;
        long long c0 = clock64();
        mbar_wait(&tmem_empty_bar[buf], ((local >> 1) & 1) ^ 1);
        t_wait_tmem += clock64() - c0;
        tcgen05_fence_after();
        const uint32_t acc0 = tmem_base + buf * 2 * BN;
        for (int kc = 0; kc < p.kchunks0; ++kc) {
          const int nk = (kc == p.kchunks0 - 1) ? p.klast0 : 4;
          for (int s = 0; s < p.ks; ++s, ++it) {
            const int stage = it % p.stages;
            long long c1 = clock64();
            mbar_wait(&full_bar[stage], (it / p.stages) & 1);
            t_wait_full += clock64() - c1;
            tcgen05_fence_after();
            const uint32_t a_lo0 = smem_desc_lo(smem_u32(smem + (size_t)stage * p.stage_bytes));
            const uint32_t b_lo0 = a_lo0 + (p.a_bytes >> 4);
            const uint32_t first = (kc | s) != 0;  // 0 only for the very first stage of the item
            if (elect_one_sync()) {
            if (nk == 4) {
              for (int r = 0; r < p.ks; ++r) {
#pragma unroll
                for (int j = 0; j < TPI; ++j) {
                  const uint32_t a_lo = a_lo0 + (j ? tile_rows16 : 0u) + r * row16;
                  const uint32_t b_lo = b_lo0 + r * (B_TAP_BYTES >> 4);
                  mma(acc0 + j * BN, a_lo, b_lo, r == 0 ? first : 1u);
                  mma(acc0 + j * BN, a_lo + 2, b_lo + 2, 1u);
                  mma(acc0 + j * BN, a_lo + 4, b_lo + 4, 1u);
                  mma(acc0 + j * BN, a_lo + 6, b_lo + 6, 1u);
                }
              }
            } else {
              for (int r = 0; r < p.ks; ++r)
                for (int j = 0; j < TPI; ++j)
                  for (int k = 0; k < nk; ++k)
                    mma(acc0 + j * BN, a_lo0 + (j ? tile_rows16 : 0u) + r * row16 + 2 * k,
                        b_lo0 + r * (B_TAP_BYTES >> 4) + 2 * k, (r | k) == 0 ? first : 1u);
            }
            commit(&empty_bar[stage]);
            }
            __syncwarp();
          }
        }
        for (int kc = 0; kc < p.kchunks1; ++kc, ++it) {
          const int nk = (kc == p.kchunks1 - 1) ? p.klast1 : 4;
          const int stage = it % p.stages;
          mbar_wait(&full_bar[stage], (it / p.stages) & 1);
          tcgen05_fence_after();
          const uint32_t a_lo0 = smem_desc_lo(smem_u32(smem + (size_t)stage * p.stage_bytes));
          const uint32_t b_lo0 = a_lo0 + (p.a_bytes >> 4);
          if (elect_one_sync()) {
#pragma unroll
            for (int j = 0; j < TPI; ++j)
              for (int k = 0; k < nk; ++k)
                mma(acc0 + j * BN, a_lo0 + (j ? tile_rows16 : 0u) + 2 * k, b_lo0 + 2 * k, 1u);
            commit(&empty_bar[stage]);
          }
          __syncwarp();
        }
        if (elect_one_sync()) commit(&tmem_full_bar[buf]);
        __syncwarp();
      }
      if (p.trace != nullptr && lane == 0) {
        p.trace[blockIdx.x * 8 + 0] = clock64() - t_begin;
        p.trace[blockIdx.x * 8 + 1] = t_wait_tmem;
        p.trace[blockIdx.x * 8 + 2] = t_wait_full;
      }
    }
  } else {
    // ===================== epilogue (warps 2..9) =====================
    // Two warps per TMEM lane group: warps 2-5 drain M tile 0, warps 6-9 M tile 1 of the item.  16-column chunks:
    // TMEM -> registers -> XOR-swizzled [32][16] staging slice (conflict-free without padding) -> 4 lanes per row (float4),
    // 8 rows per instruction; the residual loads of a chunk are issued before any is used.
    const int e = warp - 2;
    const int g = warp & 3;            // TMEM lane group [32g, 32g+32) this warp may access
    const int hslot = e >> 2;          // second set of four warps: M tile 1 (two-tile items) or the upper half of the columns
    const int j = TPI == 2 ? hslot : 0;
    constexpr int CW = TPI == 2 ? BN : BN / 2;  // columns drained by this warp
    const int c_begin = TPI == 2 ? 0 : hslot * CW;
    float* stg = staging + e * 32 * 16;
    const int sub = lane >> 2, cq4 = lane & 3;
    const int et = threadIdx.x - 64;   // 0..255 among the epilogue threads
    uint32_t local = 0;
    long long e_wait = 0, e_begin = clock64(), e_stats = 0;
    const uint32_t tmem_empty0 = CG == 2 ? mapa_u32(smem_u32(&tmem_empty_bar[0]), 0) : 0u;  // the leader's (pairs)
    for (int q = cid; q < n_q; q += cstride, ++local) {
      const int item = item_of(q);
      const int pair = item / per_pair, rest = item - pair * per_pair;
      const int phase = rest % p.nph, n_off = (rest / p.nph) * BN;
      const uint32_t buf = local & 1;
      const size_t m_pair = (size_t)pair * TPI * 128;
      const size_t m_w = m_pair + j * 128 + g * 32;  // first row of this warp's 32 rows
      float* sbuf = statbuf + (size_t)(local & 1) * (8 * BN * 2);
      // up: this warp's first low-resolution pixel inside its frame, and the offset of the frame's phase-(a, b) origin in the output
      const unsigned fr_up = UP ? (unsigned)(m_pair / (unsigned)p.HW) : 0u;
      const int lp0 = UP ? (int)(m_w - (size_t)fr_up * p.HW) : 0;
      const size_t up_base = UP ? (((size_t)fr_up * 2 * p.H + (phase >> 1)) * (2 * p.W) + (phase & 1)) * p.Cout : 0;
      // bias for this lane's 4 columns of every 16-column chunk: loaded before the accumulator wait (latency hidden)
      float4 biasv[CW / 16];
#pragma unroll
      for (int cc = 0; cc < CW / 16; ++cc) {
        const int col = n_off + c_begin + cc * 16 + cq4 * 4;
        biasv[cc] = (p.bias != nullptr && col < p.Cout) ? __ldg(reinterpret_cast<const float4*>(p.bias + col)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      long long c2 = clock64();
      mbar_wait(&tmem_full_bar[buf], (local >> 1) & 1);
      e_wait += clock64() - c2;
      tcgen05_fence_after();
#pragma unroll
      for (int ci = 0; ci < CW; ci += 16) {
        const int c = c_begin + ci;
        const int col = n_off + c + cq4 * 4;
        const bool col_ok = col < p.Cout;
        float4 res[4];
        if (p.resid != nullptr && col_ok) {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            res[i] = __ldg(reinterpret_cast<const float4*>(p.resid + (m_w + i * 8 + sub) * p.Cout + col));
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i) res[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        uint32_t v[16];
        tmem_ld_32x32b_x16(tmem_base + ((uint32_t)(g * 32) << 16) + buf * 2 * BN + j * BN + c, v);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          *reinterpret_cast<float4*>(stg + lane * 16 + ((q ^ ((lane >> 1) & 3)) << 2)) =
              make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
        __syncwarp();
        const float4 bias = biasv[ci / 16];
        float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int row = i * 8 + sub;
          const float4 a = *reinterpret_cast<const float4*>(stg + row * 16 + ((cq4 ^ ((row >> 1) & 3)) << 2));
          const float o[4] = {a.x + bias.x + res[i].x, a.y + bias.y + res[i].y, a.z + bias.z + res[i].z, a.w + bias.w + res[i].w};
#pragma unroll
          for (int q = 0; q < 4; ++q) { s1[q] += o[q]; s2[q] = fmaf(o[q], o[q], s2[q]); }
          if (col_ok) {
            size_t off = (m_w + row) * p.Cout + col;
            if (UP) {
              // low-resolution pixel (frame, y, x) -> pixel (2y + a, 2x + b) of the output
              const int lp = lp0 + row, yy = lp >> p.log2W, xx = lp & (p.W - 1);
              off = up_base + ((size_t)(2 * yy) * (2 * p.W) + 2 * xx) * p.Cout + col;
            }
            if (p.y_f32 != nullptr) *reinterpret_cast<float4*>(p.y_f32 + off) = make_float4(o[0], o[1], o[2], o[3]);
            if (p.y_op != nullptr) OpType<__nv_bfloat16>::store4(p.y_op + off, make_float4(o[0], o[1], o[2], o[3]));
          }
        }
        if (p.stats != nullptr) {
          // 8 values per lane (4 columns x 2 moments) summed over the 8 lanes that hold the same columns (sub = lane bits 2..4):
          // a transposing butterfly — each step halves the values a lane keeps and exchanges the other half — needs 4 + 2 + 1
          // shuffles instead of 8 x 3, and leaves ONE finished sum in every lane: moment = bit 4, column = bits 3, 2.
          const bool b4 = (lane & 16) != 0, b3 = (lane & 8) != 0, b2 = (lane & 4) != 0;
          float k4[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) k4[q] = (b4 ? s2[q] : s1[q]) + __shfl_xor_sync(0xffffffffu, b4 ? s1[q] : s2[q], 16);
          float k2[2];
#pragma unroll
          for (int q = 0; q < 2; ++q) k2[q] = (b3 ? k4[2 + q] : k4[q]) + __shfl_xor_sync(0xffffffffu, b3 ? k4[q] : k4[2 + q], 8);
          const float k1 = (b2 ? k2[1] : k2[0]) + __shfl_xor_sync(0xffffffffu, b2 ? k2[0] : k2[1], 4);
          const int qcol = (b3 ? 2 : 0) + (b2 ? 1 : 0);
          sbuf[((size_t)(hslot * 4 + g) * BN + c + cq4 * 4 + qcol) * 2 + (b4 ? 1 : 0)] = k1;
        }
        __syncwarp();  // staging is overwritten by the next chunk
      }
      // all TMEM reads of this warp's part of the accumulator buffer are complete (tcgen05.wait::ld inside the load helper)
      tcgen05_fence_before();
      if (lane == 0) {
        if (CG == 2) mbar_arrive_cluster(tmem_empty0 + buf * 8);
        else mbar_arrive(&tmem_empty_bar[buf]);
      }
      long long c3 = clock64();
      if (p.stats != nullptr) {
        // (the partials alternate between two buffers: the next item's partial writes need no second barrier — a thread reaches the
        //  next item's barrier only after its reads below, and this buffer is not written again before that barrier)
        asm volatile("bar.sync 1, 256;" ::: "memory");
        // both tiles lie in one frame (a pair never straddles frames): 8 partials per (column, moment), fixed order
        const int frame = (int)(m_pair / p.HW);
        for (int i = et; i < BN * 2; i += 256) {
          const int cc = i >> 1;
          if (n_off + cc < p.Cout) {
            // two-tile items: 8 partials per column (2 tiles x 4 lane groups); one-tile items: the 4 lane groups of the warp set
            // that drained this half of the columns
            const int k0 = TPI == 2 ? 0 : (cc < BN / 2 ? 0 : 4), k1 = TPI == 2 ? 8 : k0 + 4;
            float acc = 0.f;
            for (int k = k0; k < k1; ++k) acc += sbuf[(size_t)k * BN * 2 + i];
            atomicAdd(p.stats + ((size_t)frame * p.Cout + n_off + cc) * 2 + (i & 1), (double)acc);
          }
        }
      }
      e_stats += clock64() - c3;
    }
    if (p.trace != nullptr && warp == 2 && lane == 0) {
      p.trace[blockIdx.x * 8 + 3] = clock64() - e_begin;
      p.trace[blockIdx.x * 8 + 4] = e_wait;
      p.trace[blockIdx.x * 8 + 5] = e_stats;
      p.trace[blockIdx.x * 8 + 6] = local;
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (CG == 2) cluster_sync_all();  // neither CTA leaves while the other may still signal its barriers or read its shared memory
  if (warp == 2) {
    tcgen05_fence_after();
    if (CG == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
  }
}

// ---------------------------------------------------------------- host side
static bool encode4(CUtensorMap* m, const void* ptr, int N, int H, int W, int C, int rows) {
  EncodeTiledFn enc = get_tensormap_encoder();
  if (!enc) return false;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)W, (cuuint32_t)rows, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
static bool encode3w(CUtensorMap* m, const void* ptr, int taps, int co_pad, int ci_pad, int bn, int box_taps) {
  EncodeTiledFn enc = get_tensormap_encoder();
  if (!enc) return false;
  cuuint64_t dims[3] = {(cuuint64_t)ci_pad, (cuuint64_t)co_pad, (cuuint64_t)taps};
  cuuint64_t strides[2] = {(cuuint64_t)ci_pad * 2, (cuuint64_t)co_pad * ci_pad * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)bn, (cuuint32_t)box_taps};
  cuuint32_t estr[3] = {1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static int g_num_sms = 0;
static long long* g_trace = nullptr;

template <int BN, int TPI, int CG, bool UP>
static int launch_halo_cg(const CUtensorMap& ta0, const CUtensorMap& tw0, const CUtensorMap& ta1, const CUtensorMap& tw1,
                          HaloParams& p, cudaStream_t st) {
  constexpr int SMEM_MAX = 226 * 1024;  // 227 KB per CTA minus the static barriers
  const int extra = 1024 + 8 * 32 * 16 * 4 + 2 * 2 * 4 * BN * 2 * 4;  // alignment slack + staging + statbuf (two buffers)
  p.a_bytes0 = (p.tpi * p.hbox + p.ks - 1) * p.W * 128;
  p.a_bytes = p.a_bytes0 > p.tpi * 128 * 128 ? p.a_bytes0 : p.tpi * 128 * 128;  // the skip segment's box has no halo
  p.stage_bytes = p.a_bytes + p.ks * (BN / CG) * 128;  // a CTA of a pair stages half of the weight tile
  p.stages = (SMEM_MAX - extra) / p.stage_bytes;
  if (p.stages > HALO_MAX_STAGES) p.stages = HALO_MAX_STAGES;
  if (p.stages < 2) return FDM_ERR_UNSUPPORTED;
  const int smem = p.stages * p.stage_bytes + extra;
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] {
    attr_err = cudaFuncSetAttribute(conv_halo_kernel<BN, TPI, CG, UP>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_MAX);
    if (g_num_sms == 0) {
      int dev = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    }
  });
  if (attr_err != cudaSuccess) {
    set_last_error(attr_err);
    return FDM_ERR_CUDA;
  }
  const int sms = g_num_sms > 0 ? g_num_sms : 148;
  if (CG == 2) {
    const int pairs = sms / 2, n_q = p.n_items / 2;
    fdm::launch_cluster(conv_halo_kernel<BN, TPI, CG, UP>, dim3(2 * (n_q < pairs ? n_q : pairs)), dim3(HALO_THREADS), smem, st, 2, ta0, tw0, ta1, tw1, p);
  } else {
    const int grid = p.n_items < sms ? p.n_items : sms;
    fdm::launch(conv_halo_kernel<BN, TPI, CG, UP>, dim3(grid), dim3(HALO_THREADS), smem, st, ta0, tw0, ta1, tw1, p);
  }
  return check_launch();
}

template <int BN, int TPI>
static int launch_halo(const CUtensorMap& ta0, const CUtensorMap& tw0, const CUtensorMap& ta1, const CUtensorMap& tw1,
                       HaloParams& p, bool pair, cudaStream_t st) {
  if (p.up) {
    // upsample convs map C -> C channels of the U-Net's block widths: BN = 32 is not instantiated for them
    if (BN == 32) return FDM_ERR_UNSUPPORTED;
    constexpr int BU = BN == 32 ? 64 : BN;
    if (pair) return launch_halo_cg<BU, TPI, 2, true>(ta0, tw0, ta1, tw1, p, st);
    return launch_halo_cg<BU, TPI, 1, true>(ta0, tw0, ta1, tw1, p, st);
  }
  if (pair) return launch_halo_cg<BN, TPI, 2, false>(ta0, tw0, ta1, tw1, p, st);
  return launch_halo_cg<BN, TPI, 1, false>(ta0, tw0, ta1, tw1, p, st);
}

// FDM_ERR_UNSUPPORTED => the caller falls back to the per-tap kernel of conv_tc.cu
int conv_halo_launch(const fdm_conv_args* a, cudaStream_t st) {
  FDM_REQUIRE(a->a_dtype == FDM_BF16 && (a->ksize == 3 || a->ksize == 1) && a->stride == 1 && !a->out_nchw, FDM_ERR_UNSUPPORTED);
  // upsample: Hin x Win is the LOW-resolution input, the output is 2Hin x 2Win, and w0 holds the 4 x (2x2) per-phase filters
  // ([phase = 2a + b][tap = 2s' + r'][co_pad][ci_pad], see include/fdm_b200.h)
  const int up = a->upsample ? 1 : 0;
  FDM_REQUIRE(!up || (a->ksize == 3 && a->a1 == nullptr && a->resid == nullptr), FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(a->resid_norm == 0, FDM_ERR_UNSUPPORTED);  // the recomputed-GroupNorm residual lives in the per-tap kernel's epilogue
  FDM_REQUIRE(a->C0 % 8 == 0 && (a->a1 == nullptr || a->C1 % 8 == 0) && a->Cout % 4 == 0 && a->Cout >= 32, FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(a->y_op == nullptr || a->op_dtype == FDM_BF16, FDM_ERR_UNSUPPORTED);
  int W = a->Win, H = a->Hin, N = a->N;
  // pointwise layers without per-frame statistics see a flat pixel list: maps the row-halo tiling does not take (8x8, 4x4) run as
  // [N*H*W / 256] "frames" of two 128-pixel rows (the wide qkv linears of the 8x8 levels)
  if (a->ksize == 1 && a->stats == nullptr && !((W == 16 || W == 32 || W == 64 || W == 128) && H % (128 / W) == 0) &&
      ((long)N * H * W) % 256 == 0) {
    N = (int)(((long)N * H * W) / 256);
    H = 2;
    W = 128;
  }
  // W = 128 (the top level of the 128-px model, 40 % of its conv FLOPs): one image row per M tile; the A box of a two-tile item
  // (4 rows = 64 KB) leaves room for one pipeline stage only, so those layers run one-tile items (3 rows = 48 KB, two stages)
  FDM_REQUIRE(W == 16 || W == 32 || W == 64 || W == 128, FDM_ERR_UNSUPPORTED);
  const int hbox = 128 / W;
  FDM_REQUIRE(H % hbox == 0, FDM_ERR_UNSUPPORTED);
  HaloParams p;
  p.bias = a->bias; p.resid = a->resid; p.y_f32 = a->y_f32; p.y_op = reinterpret_cast<__nv_bfloat16*>(a->y_op);
  p.stats = reinterpret_cast<double*>(a->stats);
  p.Cout = a->Cout; p.W = W; p.HW = H * W; p.hbox = hbox;
  p.up = up; p.nph = up ? 4 : 1; p.H = H;
  p.log2W = 0;
  while ((1 << p.log2W) < W) ++p.log2W;
  const int bn = a->Cout % 128 == 0 ? 128 : (a->Cout >= 64 ? 64 : 32);
  p.ntiles = (a->Cout + bn - 1) / bn;
  // items of two M tiles share the weight tiles, but a grid of persistent CTAs finishes with its slowest CTA: pick the item
  // size whose rounds-on-148-SMs x per-item cost is smaller (measured on B200: one-tile items cost ~30 % more per tile —
  // no B sharing, relatively larger halo — so they only pay when two-tile items waste a whole round)
  {
    const long tiles = (long)N * (H / hbox) * p.ntiles * p.nph;
    const long rounds1 = (tiles + 147) / 148, rounds2 = (tiles / 2 + 147) / 148;
    const bool two_ok = H % (2 * hbox) == 0;
    p.tpi = (two_ok && 20 * rounds2 <= 13 * rounds1) ? 2 : 1;
  }
  p.trace = g_trace;
  p.ks = up ? 2 : a->ksize;
  p.kchunks0 = (a->C0 + 63) / 64;
  p.kchunks1 = a->a1 ? (a->C1 + 63) / 64 : 0;
  p.klast0 = (a->C0 - (p.kchunks0 - 1) * 64 + 15) / 16;
  p.klast1 = a->a1 ? (a->C1 - (p.kchunks1 - 1) * 64 + 15) / 16 : 0;
  const int co_pad = (a->Cout + 15) / 16 * 16;
  // CTA pairs (cta_group::2) when the item pairs come out even, so that both CTAs of a pair always have an item; the weight box
  // of a pair CTA holds half of the tile's rows.
  // Measured on B200 (profiles/r02_halo_cta_pairs.txt): 1.10-1.32x on layers with >= 9 pipeline stages per item (Cin >= 192 or a wide
  // skip segment; 384->384 at 32x32 reaches 1474 TFLOP/s), 0.85-1.0x on shallower ones, where the cross-CTA signalling latency of the
  // few stages is not amortised -> pairs only for the deep layers.
  const int stages_per_item = p.kchunks0 * p.ks + p.kchunks1;
  // (W = 128, BN = 128: always worth it, 1.1-1.4x — only pairs can run the two-tile items there, see below)
  bool pair = (stages_per_item >= 9 || (W == 128 && bn == 128)) &&
              ((long)N * (H / (p.tpi * hbox))) % 2 == 0;
  // W = 128 with BN = 128: a single CTA's two-tile stage (64 KB of A + 48 KB of weights) fits only once -> one-tile items (3 image
  // rows loaded per row computed); a pair CTA stages 24 KB of weights, so two stages of two-tile items fit (4 rows per 2 computed)
  if (W == 128 && bn == 128 && !(pair && p.tpi == 2)) {
    p.tpi = 1;
    pair = pair && ((long)N * (H / hbox)) % 2 == 0;
  }
  p.pairs_per_frame = H / (p.tpi * hbox);
  p.n_items = N * p.pairs_per_frame * p.ntiles * p.nph;
  const int brows = pair ? bn / 2 : bn;
  CUtensorMap ta0, tw0, ta1, tw1;
  bool ok = encode4(&ta0, a->a0, N, H, W, a->C0, p.tpi * hbox + p.ks - 1) &&
            encode3w(&tw0, a->w0, up ? 16 : a->ksize * a->ksize, co_pad, p.kchunks0 * 64, brows, p.ks);
  if (ok && a->a1) {
    ok = encode4(&ta1, a->a1, N, H, W, a->C1, p.tpi * hbox) && encode3w(&tw1, a->w1, 1, co_pad, p.kchunks1 * 64, brows, 1);
  } else {
    ta1 = ta0;
    tw1 = tw0;
  }
  FDM_REQUIRE(ok, FDM_ERR_UNSUPPORTED);
  if (p.tpi == 2) {
    if (bn == 128) return launch_halo<128, 2>(ta0, tw0, ta1, tw1, p, pair, st);
    if (bn == 64) return launch_halo<64, 2>(ta0, tw0, ta1, tw1, p, pair, st);
    return launch_halo<32, 2>(ta0, tw0, ta1, tw1, p, pair, st);
  }
  if (bn == 128) return launch_halo<128, 1>(ta0, tw0, ta1, tw1, p, pair, st);
  if (bn == 64) return launch_halo<64, 1>(ta0, tw0, ta1, tw1, p, pair, st);
  return launch_halo<32, 1>(ta0, tw0, ta1, tw1, p, pair, st);
}

}  // namespace fdm

// debug hook (not part of the product ABI): the next conv_halo launches write per-CTA cycle counters to trace[cta][8] =
// {MMA warp total, MMA waiting for a free accumulator, MMA waiting for operands, epilogue total, epilogue waiting for
//  the accumulator, epilogue statistics phase, items}
extern "C" void fdm_debug_set_trace(long long* trace) { fdm::g_trace = trace; }
