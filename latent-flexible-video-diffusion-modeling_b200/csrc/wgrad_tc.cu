// Convolution / linear WEIGHT gradient on tcgen05 (bf16 operands, fp32 accumulation in TMEM), stride 1, 1x1 or 3x3.
//
//   dW[kh][kw][ci][co] = sum over pixels p of  X[p + (kh-1, kw-1)][ci] * dY[p][co]
//
// Per filter tap this is a GEMM whose REDUCTION dimension is the pixel index, and both operands are stored pixel-major with
// the channels contiguous ([N][H][W][C] activations) — i.e. both are "MN-major" UMMA operands and are consumed straight from
// the TMA boxes, no transposition pass:
//   A (M = input channels)  = a TMA box of X:  (hbox + 2) image rows x W pixels x 64 channels, 128-byte swizzle; the three
//                             filter ROWS kh of one filter COLUMN kw are the same box at descriptor offsets of kh*W rows
//                             (the filter column is the box's x offset, zero-filled out of bounds by TMA);
//   B (N = output channels) = a TMA box of dY: hbox rows x W pixels x 64 channels.
// M is always 128: either two 64-channel blocks of X (LBO = block stride) -> one MMA per filter row, or — when only one block
// is staged (C = 64, or very wide rows) — the SAME block at two filter-row offsets (LBO = one image row) -> (kh0, kh1) share
// an MMA and (kh2, unused) the next.  A CTA owns (64|128 input channels) x (<=128 output channels) x (one filter column) x (a
// range of pixel chunks): accumulators stay in TMEM for the whole range (<= 3 x 128 columns), then go to fp32 partials that
// wgrad_reduce_kernel (bwd_conv.cu) sums in a fixed order.  Roofline: tensor (2*9*Cin*Cout FLOP per pixel).
#include "tc_common.cuh"

namespace fdm {

constexpr int WG_MAX_STAGES = 4;
constexpr int WG_TMEM_COLS = 512;

struct WgTcParams {
  float* part;
  int C, Cout, taps, ks;
  int W, hbox, P, hblocks, n_chunks, cps;   // P = hbox*W pixels per chunk; cps = chunks per split
  int nxb, nc, co_chunks;                   // X blocks staged (1|2), output channels per CTA (64|128)
  int stages, stage_bytes, xblk_bytes, x_bytes, dyblk_bytes;
  int n_mma;
  uint32_t a_off16[3], a_lbo16, b_lbo16, acc_col[3];
};

__global__ void __launch_bounds__(128, 1) wgrad_tc_kernel(const __grid_constant__ CUtensorMap tx,
                                                          const __grid_constant__ CUtensorMap tdy, const WgTcParams p) {
  extern __shared__ uint8_t wg_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(wg_smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t full_bar[WG_MAX_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[WG_MAX_STAGES];
  __shared__ __align__(8) uint64_t done_bar;
  __shared__ uint32_t tmem_base_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tx);
    prefetch_tmap(&tdy);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(&done_bar, 1);
    fence_mbarrier_init();
  }
  if (warp == 2) tmem_alloc<1, WG_TMEM_COLS>(&tmem_base_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_base_slot;
  pdl_wait();

  const int ci0 = (blockIdx.x / p.co_chunks) * 64 * p.nxb, co0 = (blockIdx.x % p.co_chunks) * p.nc;
  const int ncols = min(p.nc, p.Cout - co0);
  const int kw = blockIdx.y, pad = p.ks >> 1;
  const int q_begin = blockIdx.z * p.cps;
  const int nq = min(q_begin + p.cps, p.n_chunks) - q_begin;
  const int nxb_valid = min(p.nxb, (p.C - ci0 + 63) / 64);
  const int nyb = ncols / 64;

  if (warp == 0) {
    // ===================== TMA producer =====================
    for (int it = 0; it < nq; ++it) {
      const int q = q_begin + it;
      const int n = q / p.hblocks, h0 = (q - n * p.hblocks) * p.hbox;
      const int stage = it % p.stages;
      mbar_wait(&empty_bar[stage], ((it / p.stages) & 1) ^ 1);
      uint8_t* x_dst = smem + (size_t)stage * p.stage_bytes;
      uint8_t* y_dst = x_dst + p.x_bytes;
      if (elect_one_sync()) {
        mbar_expect_tx(&full_bar[stage], nxb_valid * ((p.hbox + p.ks - 1) * p.W * 128) + nyb * p.dyblk_bytes);
        for (int b = 0; b < nxb_valid; ++b) tma_load_4d(x_dst + (size_t)b * p.xblk_bytes, &tx, &full_bar[stage], ci0 + 64 * b, kw - pad, h0 - pad, n);
        for (int b = 0; b < nyb; ++b) tma_load_4d(y_dst + (size_t)b * p.dyblk_bytes, &tdy, &full_bar[stage], co0 + 64 * b, 0, h0, n);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // instruction descriptor: D = f32, A = B = bf16, BOTH operands MN-major (bits 15, 16), M = 128, N = ncols
    const uint32_t idesc = make_idesc(ncols, 1) | (1u << 15);
    const int ksteps = p.P >> 4;
    for (int it = 0; it < nq; ++it) {
      const int stage = it % p.stages;
      mbar_wait(&full_bar[stage], (it / p.stages) & 1);
      tcgen05_fence_after();
      const uint32_t x_addr16 = (smem_u32(smem + (size_t)stage * p.stage_bytes) & 0x3FFFFu) >> 4;
      const uint32_t a_lo0 = x_addr16 | (p.a_lbo16 << 16);
      const uint32_t b_lo0 = (x_addr16 + ((uint32_t)p.x_bytes >> 4)) | (p.b_lbo16 << 16);
      if (elect_one_sync()) {
        for (int ks = 0; ks < ksteps; ++ks) {
          // 16 pixel rows of 128 bytes per K step = 2048 bytes = 128 descriptor units
#pragma unroll
          for (int j = 0; j < 3; ++j)
            if (j < p.n_mma)
              umma_bf16_lo(tmem_base + p.acc_col[j], a_lo0 + p.a_off16[j] + ks * 128, b_lo0 + ks * 128, idesc, (it | ks) != 0 ? 1u : 0u);
        }
        umma_commit(&empty_bar[stage]);
      }
      __syncwarp();
    }
    if (elect_one_sync()) umma_commit(&done_bar);
    __syncwarp();
  }
  // ===================== epilogue: TMEM lane = accumulator row =====================
  mbar_wait(&done_bar, 0);
  tcgen05_fence_after();
  const int m = threadIdx.x;
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    if (j >= p.n_mma) break;
    int kh, ci;
    if (p.nxb == 2) { kh = j; ci = ci0 + m; }
    else { kh = 2 * j + (m >> 6); ci = ci0 + (m & 63); }
    const bool row_ok = kh < p.ks && ci < p.C && nq > 0;
    const int tap = kh * p.ks + kw;
    float* out = p.part + (((size_t)blockIdx.z * p.taps + (row_ok ? tap : 0)) * p.C + (row_ok ? ci : 0)) * p.Cout + co0;
    for (int c = 0; c < ncols; c += 32) {
      uint32_t r[32];
      tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(warp * 32) << 16) + p.acc_col[j] + c, r);
      if (row_ok) {
#pragma unroll
        for (int i = 0; i < 32; i += 4)
          *reinterpret_cast<float4*>(out + c + i) = make_float4(__uint_as_float(r[i]), __uint_as_float(r[i + 1]), __uint_as_float(r[i + 2]), __uint_as_float(r[i + 3]));
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<1, WG_TMEM_COLS>(tmem_base);
}

struct WgTcGeom {
  bool ok;
  int hbox, P, hblocks, n_chunks, nxb, nc, ci_chunks, co_chunks, stages, stage_bytes, xblk_bytes, x_bytes, dyblk_bytes, splits, cps;
};

static WgTcGeom wg_tc_geom(const fdm_conv_wgrad_args* a) {
  WgTcGeom g{};
  g.ok = false;
  if (a->a_dtype != FDM_BF16 || a->dy_dtype != FDM_BF16 || a->stride != 1) return g;
  if (a->C % 64 || a->Cout % 64) return g;
  const int W = a->Win, H = a->Hin;
  if (W < 8 || W > 128 || (W & (W - 1)) || H < 1) return g;
  int hbox = 128 / W;
  if (hbox < 1) hbox = 1;
  while (hbox > 1 && (H % hbox)) hbox >>= 1;
  if (hbox > H) hbox = H;
  if (H % hbox) return g;
  const int P = hbox * W;
  if (P % 16 || P > 256) return g;
  g.hbox = hbox; g.P = P; g.hblocks = H / hbox; g.n_chunks = a->N * g.hblocks;
  g.nc = a->Cout % 128 == 0 ? 128 : 64;
  g.co_chunks = (a->Cout + g.nc - 1) / g.nc;
  g.dyblk_bytes = P * 128;
  const int limit = 220 * 1024;
  for (int nxb = a->C >= 128 ? 2 : 1; nxb >= 1; --nxb) {
    // pair mode (one block) reads a fourth filter-row offset for the unused half of its second MMA: one extra image row
    const int rows = (hbox + a->ksize - 1 + ((nxb == 1 && a->ksize == 3) ? 1 : 0)) * W;
    if (hbox + a->ksize - 1 > 256) return g;
    g.xblk_bytes = rows * 128;
    g.x_bytes = nxb * g.xblk_bytes;
    g.stage_bytes = g.x_bytes + (g.nc / 64) * g.dyblk_bytes;
    g.stages = limit / g.stage_bytes;
    if (g.stages > WG_MAX_STAGES) g.stages = WG_MAX_STAGES;
    g.nxb = nxb;
    if (g.stages >= 2) break;
  }
  if (g.stages < 2) return g;
  g.ci_chunks = (a->C + 64 * g.nxb - 1) / (64 * g.nxb);
  const long long base = (long long)g.ci_chunks * g.co_chunks * a->ksize;
  // one CTA per SM (shared memory): at most two full waves of 148 CTAs, never a third, nearly empty one
  long long splits = (148LL * 2) / base;
  if (splits > g.n_chunks) splits = g.n_chunks;
  if (splits < 1) splits = 1;
  g.cps = (int)((g.n_chunks + splits - 1) / splits);
  g.splits = (g.n_chunks + g.cps - 1) / g.cps;
  g.ok = g.splits <= 65535;
  return g;
}

size_t conv_wgrad_tc_partial_bytes(const fdm_conv_wgrad_args* a) {
  const WgTcGeom g = wg_tc_geom(a);
  if (!g.ok) return 0;
  return (size_t)g.splits * a->ksize * a->ksize * a->C * a->Cout * sizeof(float);
}

// Runs the tensor-core kernel into `part` ([splits][taps][C][Cout]) and reports the split count for the reduction.
int conv_wgrad_tc(const fdm_conv_wgrad_args* a, float* part, int* splits_out, cudaStream_t st) {
  const WgTcGeom g = wg_tc_geom(a);
  if (!g.ok) return FDM_ERR_UNSUPPORTED;
  // activations [N][H][W][C] as (C, W, H, N) tensors; boxes of 64 channels x W x (hbox + ks - 1 | hbox) rows x 1
  const cuuint64_t xdims[4] = {(cuuint64_t)a->C, (cuuint64_t)a->Win, (cuuint64_t)a->Hin, (cuuint64_t)a->N};
  const cuuint64_t dydims[4] = {(cuuint64_t)a->Cout, (cuuint64_t)a->Win, (cuuint64_t)a->Hin, (cuuint64_t)a->N};
  const cuuint32_t xbox[4] = {64, (cuuint32_t)a->Win, (cuuint32_t)(g.hbox + a->ksize - 1), 1};
  const cuuint32_t dybox[4] = {64, (cuuint32_t)a->Win, (cuuint32_t)g.hbox, 1};
  CUtensorMap tx, tdy;
  if (!encode_bf16_map(&tx, a->a, 4, xdims, xbox, CU_TENSOR_MAP_L2_PROMOTION_L2_128B)) return FDM_ERR_UNSUPPORTED;
  if (!encode_bf16_map(&tdy, a->dy, 4, dydims, dybox, CU_TENSOR_MAP_L2_PROMOTION_L2_128B)) return FDM_ERR_UNSUPPORTED;
  WgTcParams p{};
  p.part = part;
  p.C = a->C; p.Cout = a->Cout; p.ks = a->ksize; p.taps = a->ksize * a->ksize;
  p.W = a->Win; p.hbox = g.hbox; p.P = g.P; p.hblocks = g.hblocks; p.n_chunks = g.n_chunks; p.cps = g.cps;
  p.nxb = g.nxb; p.nc = g.nc; p.co_chunks = g.co_chunks;
  p.stages = g.stages; p.stage_bytes = g.stage_bytes; p.xblk_bytes = g.xblk_bytes; p.x_bytes = g.x_bytes; p.dyblk_bytes = g.dyblk_bytes;
  const uint32_t row16 = (uint32_t)(a->Win * 128) >> 4;  // one image row of the X box in descriptor units
  p.b_lbo16 = (uint32_t)g.dyblk_bytes >> 4;
  if (g.nxb == 2) {
    p.n_mma = a->ksize;
    p.a_lbo16 = (uint32_t)g.xblk_bytes >> 4;
    for (int j = 0; j < a->ksize; ++j) { p.a_off16[j] = j * row16; p.acc_col[j] = j * g.nc; }
  } else {
    p.n_mma = a->ksize == 3 ? 2 : 1;
    p.a_lbo16 = row16;
    for (int j = 0; j < p.n_mma; ++j) { p.a_off16[j] = 2 * j * row16; p.acc_col[j] = j * g.nc; }
  }
  if (p.a_lbo16 >= (1u << 14) || p.b_lbo16 >= (1u << 14)) return FDM_ERR_UNSUPPORTED;
  dim3 grid(g.ci_chunks * g.co_chunks, a->ksize, g.splits);
  const size_t smem = (size_t)g.stages * g.stage_bytes + 1024;
  if (int rc = allow_smem(wgrad_tc_kernel, 226 * 1024)) return rc;
  fdm::launch(wgrad_tc_kernel, grid, dim3(128), smem, st, tx, tdy, p);
  *splits_out = g.splits;
  return check_launch();
}

}  // namespace fdm
