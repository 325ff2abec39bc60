// Head convolution (unet.py:399-403,462-464: 3x3, model_channels -> 3/4 output channels, eps written as NCHW fp32) on tcgen05.
//
// With 4 output channels an implicit GEMM over the 9 filter taps reads every input pixel nine times out of shared memory for
// N = 16 columns of tensor work each (the per-tap kernel ran at 5-8x its HBM floor: 32 / 96 / 201 us at cfg4 / cfg5 / cfg3).  Here
// the filter taps are part of the GEMM's N dimension instead:
//     Z[pixel, (tap, co)] = X[pixel, :] . W[(tap, co), :]          one [pixels x C] x [C x 36] GEMM, every pixel read ONCE
//     y[co, h, x]         = bias[co] + sum_{r,s} Z[(h + r - 1, x + s - 1), (r, s, co)]
// i.e. the convolution's shifts are applied to the (tiny) GEMM OUTPUT in the epilogue.  One CTA = a strip of R image rows of one
// frame: TMA loads the R + 2 rows (zero-filled outside the image: their Z rows are exactly 0, which is the conv's padding), the
// strip's pixels are covered by 128-row MMA tiles whose 48-column accumulators all stay in TMEM, then Z is spilled to shared memory
// (over the dead input tile) and every thread gathers the 9 shifted float4s of its output pixels and writes coalesced NCHW rows.
#include "tc_common.cuh"
#include <mutex>

namespace fdm {

constexpr int HEAD_THREADS = 256;
constexpr int HEAD_NC = 48;      // GEMM columns: 9 taps x 4 output-channel slots = 36, padded to a multiple of 16
constexpr int HEAD_ZW = 36;      // floats of Z kept per pixel
constexpr int HEAD_MAX_CHUNKS = 4;

struct HeadParams {
  const __nv_bfloat16* w;  // packed [tap = kw*3 + kh][co_pad][ci_pad] bf16 (the per-tap kernel's layout)
  const float* bias;
  float* y;                // [N][Cout][H][W]
  int H, W, Cout, co_pad, ci_pad;
  int R;                   // output rows per strip
  int strips_per_frame, nchunks, ntile, tmem_cols;
  uint32_t chunk_stride;   // bytes between the 64-channel chunks of the input strip in shared memory
};

__global__ void __launch_bounds__(HEAD_THREADS) conv_head_kernel(const __grid_constant__ CUtensorMap ta, const HeadParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t load_bar[HEAD_MAX_CHUNKS];
  __shared__ __align__(8) uint64_t mma_bar;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n = blockIdx.x / p.strips_per_frame, h0 = (blockIdx.x - n * p.strips_per_frame) * p.R;
  const int rows = p.R + 2, PS = rows * p.W;
  uint8_t* b_s = smem;                               // [nchunks][48 rows][128 B], K-major, 128-byte swizzle
  uint8_t* a_s = smem + p.nchunks * HEAD_NC * 128;   // [nchunks][ntile * 128 pixels][128 B]; later Z: [pixels][36] fp32
  if (tid == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&ta) : "memory");
    for (int c = 0; c < p.nchunks; ++c) mbar_init(&load_bar[c], 1);
    mbar_init(&mma_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(p.tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  // weight tile: rows (tap, co < 4) of the packed weights, written in the swizzled K-major layout; rows 36..47 are zero.
  // (parameters are never written by the preceding launch of the stream, so this runs before the dependency wait)
  for (int i = tid; i < p.nchunks * HEAD_NC * 8; i += HEAD_THREADS) {
    const int piece = i & 7, row = (i >> 3) % HEAD_NC, c = i / (8 * HEAD_NC);
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    const int tap = row >> 2, co = row & 3;
    if (row < HEAD_ZW && co < p.Cout)
      v = __ldg(reinterpret_cast<const uint4*>(p.w + ((size_t)tap * p.co_pad + co) * p.ci_pad + c * 64) + piece);
    *reinterpret_cast<uint4*>(b_s + c * HEAD_NC * 128 + row * 128 + ((piece ^ (row & 7)) << 4)) = v;
  }
  fence_proxy_async_smem();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  pdl_wait();
  if (warp == 0) {
    if (elect_one_sync()) {
      for (int c = 0; c < p.nchunks; ++c) {
        mbar_expect_tx(&load_bar[c], (uint32_t)PS * 128u);
        tma_load_4d(a_s + (size_t)c * p.chunk_stride, &ta, &load_bar[c], c * 64, 0, h0 - 1, n);
      }
    }
    __syncwarp();
    // chunk-major issue order: the MMAs of chunk 0 run while chunk 1 is still landing
    constexpr uint32_t idesc = make_idesc(HEAD_NC);
    for (int c = 0; c < p.nchunks; ++c) {
      mbar_wait(&load_bar[c], 0);
      tcgen05_fence_after();
      if (elect_one_sync()) {
        const uint32_t a_lo = smem_desc_lo(smem_u32(a_s + (size_t)c * p.chunk_stride));
        const uint32_t b_lo = smem_desc_lo(smem_u32(b_s + c * HEAD_NC * 128));
        for (int t = 0; t < p.ntile; ++t)
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_bf16_lo(tmem + t * HEAD_NC, a_lo + t * (16384 >> 4) + 2 * kk, b_lo + 2 * kk, idesc, (c | kk) != 0);
      }
      __syncwarp();
    }
    if (elect_one_sync()) umma_commit(&mma_bar);
    __syncwarp();
  }
  mbar_wait(&mma_bar, 0);
  tcgen05_fence_after();
  __syncthreads();  // every thread has seen the MMAs complete: the input strip is dead, Z may overwrite it
  float* z_s = reinterpret_cast<float*>(a_s);
  {
    // warp w drains TMEM lane group w % 4 of the tiles w / 4, w / 4 + 2, ...; lane <-> pixel: 9 float4 (144 bytes) per pixel
    const int g = warp & 3;
    for (int t = warp >> 2; t < p.ntile; t += 2) {
      uint32_t v[32], v2[4];
      const uint32_t taddr = tmem + ((uint32_t)(g * 32) << 16) + t * HEAD_NC;
      asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                   : "=r"(v2[0]), "=r"(v2[1]), "=r"(v2[2]), "=r"(v2[3]) : "r"(taddr + 32));
      tmem_ld_32x32b_x32(taddr, v);  // (waits for both loads)
      float4* dst = reinterpret_cast<float4*>(z_s + (size_t)(t * 128 + g * 32 + lane) * HEAD_ZW);
#pragma unroll
      for (int q = 0; q < 8; ++q)
        dst[q] = make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
      dst[8] = make_float4(__uint_as_float(v2[0]), __uint_as_float(v2[1]), __uint_as_float(v2[2]), __uint_as_float(v2[3]));
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(p.tmem_cols));
  }
  float bias[4];
#pragma unroll
  for (int co = 0; co < 4; ++co) bias[co] = (p.bias != nullptr && co < p.Cout) ? __ldg(p.bias + co) : 0.f;
  const int W = p.W, HW = p.H * p.W;
  for (int op = tid; op < p.R * W; op += HEAD_THREADS) {
    const int lr = op / W, x = op - lr * W;  // output row h0 + lr is strip row lr + 1
    float acc[4] = {bias[0], bias[1], bias[2], bias[3]};
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      const int xs = x + s - 1;
      if (xs < 0 || xs >= W) continue;  // left / right padding (top / bottom padding: zero-filled rows -> Z == 0)
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const float4 z = *reinterpret_cast<const float4*>(z_s + (size_t)((lr + r) * W + xs) * HEAD_ZW + (s * 3 + r) * 4);
        acc[0] += z.x; acc[1] += z.y; acc[2] += z.z; acc[3] += z.w;
      }
    }
    float* y = p.y + (size_t)n * p.Cout * HW + (size_t)(h0 + lr) * W + x;
#pragma unroll
    for (int co = 0; co < 4; ++co)
      if (co < p.Cout) y[(size_t)co * HW] = acc[co];
  }
}

static bool head_encode(CUtensorMap* m, const void* ptr, int N, int H, int W, int C, int rows) {
  EncodeTiledFn enc = get_tensormap_encoder();
  if (!enc) return false;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)W, (cuuint32_t)rows, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// FDM_ERR_UNSUPPORTED => the caller falls back to the per-tap kernel
int conv_head_launch(const fdm_conv_args* a, cudaStream_t st) {
  FDM_REQUIRE(a->a_dtype == FDM_BF16 && a->ksize == 3 && a->stride == 1 && !a->upsample && a->out_nchw, FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(a->Cout <= 4 && a->a1 == nullptr && a->y_f32 != nullptr && a->y_op == nullptr && a->resid == nullptr && a->stats == nullptr &&
                  a->resid_norm == 0, FDM_ERR_UNSUPPORTED);
  const int H = a->Hin, W = a->Win;
  FDM_REQUIRE(a->C0 % 64 == 0 && a->C0 <= 64 * HEAD_MAX_CHUNKS && W % 8 == 0 && W <= 256, FDM_ERR_UNSUPPORTED);
  HeadParams p;
  p.w = reinterpret_cast<const __nv_bfloat16*>(a->w0); p.bias = a->bias; p.y = a->y_f32;
  p.H = H; p.W = W; p.Cout = a->Cout; p.co_pad = (a->Cout + 15) / 16 * 16; p.ci_pad = a->C0; p.nchunks = a->C0 / 64;
  // strip height: all R | H whose strip fits (shared memory, <= 10 MMA tiles = 480 TMEM columns, TMA box <= 256 rows); pick the one
  // with the smallest modelled time = rounds over the resident CTA slots x (resident CTAs share the SM's TMA ingest, ~64 B/clk)
  const int sms = 148, smem_cap = 226 * 1024;
  double best = 1e30;
  int bestR = 0;
  for (int R = 1; R <= H; ++R) {
    if (H % R != 0 || R + 2 > 256) continue;
    const int PS = (R + 2) * W, ntile = (PS + 127) / 128;
    if (ntile > 10) continue;
    const long a_bytes = (long)p.nchunks * ntile * 16384, z_bytes = (long)ntile * 128 * HEAD_ZW * 4;
    const long smem = 1024 + p.nchunks * HEAD_NC * 128 + (a_bytes > z_bytes ? a_bytes : z_bytes);
    if (smem > smem_cap) continue;
    int cols = 32;
    while (cols < ntile * HEAD_NC) cols *= 2;
    int k = (int)(smem_cap / smem);
    if (512 / cols < k) k = 512 / cols;
    if (2048 / HEAD_THREADS < k) k = 2048 / HEAD_THREADS;
    const long items = (long)a->N * (H / R);
    const long rounds = (items + (long)sms * k - 1) / ((long)sms * k);
    const double t = (double)rounds * (k * 2.0 * PS * p.nchunks + 3000.0);
    if (t < best) { best = t; bestR = R; }
  }
  FDM_REQUIRE(bestR > 0, FDM_ERR_UNSUPPORTED);
  p.R = bestR;
  p.strips_per_frame = H / p.R;
  const int PS = (p.R + 2) * W;
  p.ntile = (PS + 127) / 128;
  p.chunk_stride = (uint32_t)p.ntile * 16384u;
  p.tmem_cols = 32;
  while (p.tmem_cols < p.ntile * HEAD_NC) p.tmem_cols *= 2;
  const long a_bytes = (long)p.nchunks * p.ntile * 16384, z_bytes = (long)p.ntile * 128 * HEAD_ZW * 4;
  const int smem = 1024 + p.nchunks * HEAD_NC * 128 + (int)(a_bytes > z_bytes ? a_bytes : z_bytes);
  CUtensorMap ta;
  FDM_REQUIRE(head_encode(&ta, a->a0, a->N, H, W, a->C0, p.R + 2), FDM_ERR_UNSUPPORTED);
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] { attr_err = cudaFuncSetAttribute(conv_head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024); });
  if (attr_err != cudaSuccess) {
    set_last_error(attr_err);
    return FDM_ERR_CUDA;
  }
  fdm::launch(conv_head_kernel, dim3(a->N * p.strips_per_frame), dim3(HEAD_THREADS), (size_t)smem, st, ta, p);
  return check_launch();
}

}  // namespace fdm
