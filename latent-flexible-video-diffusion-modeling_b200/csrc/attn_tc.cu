// Spatial self-attention core on tcgen05 (rpe.py:139-144,163-166 with no RPE / no mask): softmax(scale * Q K^T) V per
// (frame, head), sequence = the L = H*W pixels of one frame.  In this U-Net attention only runs on 16x16, 8x8 (and the
// 4x4 middle block of the 32-px model) feature maps, so L is 16, 64 or 256 and a whole score row fits in TMEM:
// no streaming softmax is needed.
//
//   CTA = (128-query tile, head, frame).  128 threads (thread r <-> query row r <-> TMEM lane r) for short rows; for L >= SA_SPLIT_MIN_L
//   256 threads: warps w and w + 4 own the same 32 TMEM lanes and each takes HALF of the score row's columns (the softmax — two TMEM
//   passes, L exp2 and L/8 shared-memory stores per row — is the longest phase of this one-shot CTA and halves; row max and row sum are
//   exchanged through shared memory).
//   1. TMA: Q tile, all K and V rows of this (frame, head) from the packed [N][L][3C] bf16 qkv tensor, 64-channel
//      boxes in the 128B-swizzled K-major layout (head dims 16/32/48 read only their first F/16 k-steps).  V has its own barrier:
//      S = Q K^T starts as soon as Q and K have landed, V is only awaited before O = P V.
//   2. S = Q K^T       tcgen05.mma  M=128, N=L, K=F       -> TMEM columns [0, L)
//   3. softmax         each thread reads its row from TMEM twice (max, then exp2/sum), writes P (bf16, unnormalised)
//                      into shared memory in the swizzled K-major layout (aliasing the dead Q/K tiles)
//   4. O = P V         tcgen05.mma  M=128, N=F, K=L, V consumed as an MN-major operand straight from its [L][F] rows
//                      -> TMEM columns [0, F) (aliasing S, which every thread has finished reading)
//   5. O / rowsum -> bf16 -> out[N][L][C]
#include "tc_common.cuh"
#include <mutex>

namespace fdm {

constexpr int SA_SPLIT_MIN_L = 128;

struct SaTcParams {
  __nv_bfloat16* out;
  int L, C, F, heads;
  int rows;     // TMA box rows = min(L, 128)
  int cf;       // 64-wide channel chunks per head = ceil(F / 64)
  int tmem_cols;
  float scale_log2e;
  float* lse;   // optional [N][heads][L]: natural-log sum-exp of each scaled score row (saved for the backward pass)
  float* attn_mean;  // optional [N][L][L]: += softmax weights / heads (attention-map logging, rpe.py:128-130)
};

// MN-major, 128-byte swizzle: rows (one per K index) of 128 bytes = 64 MN elements; 8-row groups 1024 bytes apart (SBO)
__device__ __forceinline__ uint64_t make_smem_desc_mn(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;            // LBO: stride between 64-element MN blocks — a single block is used (N <= 64)
  d |= (uint64_t)(1024 >> 4) << 32;  // SBO: stride between 8-row K groups
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

__global__ void __launch_bounds__(256) attn_spatial_tc_kernel(const __grid_constant__ CUtensorMap tq, const SaTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t bar_load, bar_v, bar_s, bar_o;
  __shared__ uint32_t tmem_slot;
  __shared__ float xch[2][2][128];  // split rows: [max | sum][column half][row]

  const int tid = threadIdx.x, warp = tid >> 5;
  const bool split = blockDim.x == 256;
  const int hh = warp >> 2;                 // column half of this thread (0 when not split)
  const int row = tid & 127;                // query row inside the tile = TMEM lane
  const int q0 = blockIdx.x * 128, h = blockIdx.y, n = blockIdx.z;
  const int L = p.L, F = p.F, C = p.C;
  const int kv_tile = L * 128;                 // bytes of one 64-channel chunk of K (or V)
  uint8_t* v_s = smem;                         // [cf][L][128 B]
  uint8_t* q_s = v_s + p.cf * kv_tile;         // [cf][128][128 B]
  uint8_t* k_s = q_s + p.cf * 16384;           // [cf][L][128 B]
  uint8_t* p_s = q_s;                          // [ceil(L/64)][128][128 B], aliases Q and K once S is complete

  if (tid == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tq) : "memory");
    mbar_init(&bar_load, 1);
    mbar_init(&bar_v, 1);
    mbar_init(&bar_s, 1);
    mbar_init(&bar_o, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(p.tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  pdl_wait();

  if (tid == 0) {
    const int loads_kv = L / p.rows;
    mbar_expect_tx(&bar_load, (uint32_t)(p.cf * (p.rows * 128 + kv_tile)));
    mbar_expect_tx(&bar_v, (uint32_t)(p.cf * kv_tile));
    for (int c = 0; c < p.cf; ++c) {
      const int ch = h * F + c * 64;
      tma_load_3d(q_s + c * 16384, &tq, &bar_load, ch, q0, n);
      for (int j = 0; j < loads_kv; ++j) tma_load_3d(k_s + c * kv_tile + j * p.rows * 128, &tq, &bar_load, C + ch, j * p.rows, n);
    }
    for (int c = 0; c < p.cf; ++c)
      for (int j = 0; j < loads_kv; ++j)
        tma_load_3d(v_s + c * kv_tile + j * p.rows * 128, &tq, &bar_v, 2 * C + h * F + c * 64, j * p.rows, n);
    mbar_wait(&bar_load, 0);
    tcgen05_fence_after();
    // ---- S = Q K^T
    const uint32_t idesc = make_idesc(L);
    const int ksteps = F / 16;
    for (int ks = 0; ks < ksteps; ++ks) {
      const int c = ks >> 2, kk = ks & 3;
      const uint64_t ad = make_smem_desc(smem_u32(q_s + c * 16384)) + 2 * kk;
      const uint64_t bd = make_smem_desc(smem_u32(k_s + c * kv_tile)) + 2 * kk;
      umma_bf16(tmem, ad, bd, idesc, ks != 0);
    }
    umma_commit(&bar_s);
  }
  __syncwarp();
  mbar_wait(&bar_s, 0);
  tcgen05_fence_after();

  // ---- softmax over this thread's row (split: its half of the row's columns)
  const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);
  const int c_lo = split ? hh * (L >> 1) : 0, c_hi = split ? c_lo + (L >> 1) : L;
  float mx = -INFINITY;
  if (L >= 32) {
    for (int c = c_lo; c < c_hi; c += 32) {
      uint32_t v[32];
      tmem_ld_32x32b_x32(trow + c, v);
#pragma unroll
      for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(v[j]));
    }
  } else {
    uint32_t v[16];
    tmem_ld_32x32b_x16(trow, v);
#pragma unroll
    for (int j = 0; j < 16; ++j) mx = fmaxf(mx, __uint_as_float(v[j]));
  }
  // every thread of the CTA must be done READING Q/K through the tensor core before P overwrites them: S is complete
  // (bar_s), so the MMAs have retired; nothing else reads Q/K.
  if (split) {
    xch[0][hh][row] = mx;
    __syncthreads();
    mx = fmaxf(xch[0][0][row], xch[0][1][row]);
  }
  const float mneg = -mx * p.scale_log2e;
  float sum = 0.f;
  uint8_t* prow = p_s + row * 128;
  const int sw = row & 7;
  if (L >= 32) {
    for (int c = c_lo; c < c_hi; c += 32) {
      uint32_t v[32];
      tmem_ld_32x32b_x32(trow + c, v);
      float e[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        e[j] = exp2f(fmaf(__uint_as_float(v[j]), p.scale_log2e, mneg));
        sum += e[j];
      }
      uint8_t* chunk = prow + (c >> 6) * 16384;
      const int piece0 = (c & 63) >> 3;  // 16-byte piece index inside the 128-byte row
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint4 w = make_uint4(pack_bf16(e[8 * q], e[8 * q + 1]), pack_bf16(e[8 * q + 2], e[8 * q + 3]),
                             pack_bf16(e[8 * q + 4], e[8 * q + 5]), pack_bf16(e[8 * q + 6], e[8 * q + 7]));
        *reinterpret_cast<uint4*>(chunk + (((piece0 + q) ^ sw) << 4)) = w;
      }
    }
  } else {
    uint32_t v[16];
    tmem_ld_32x32b_x16(trow, v);
    float e[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      e[j] = exp2f(fmaf(__uint_as_float(v[j]), p.scale_log2e, mneg));
      sum += e[j];
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      uint4 w = make_uint4(pack_bf16(e[8 * q], e[8 * q + 1]), pack_bf16(e[8 * q + 2], e[8 * q + 3]),
                           pack_bf16(e[8 * q + 4], e[8 * q + 5]), pack_bf16(e[8 * q + 6], e[8 * q + 7]));
      *reinterpret_cast<uint4*>(prow + ((q ^ sw) << 4)) = w;
    }
  }
  if (split) xch[1][hh][row] = sum;  // read after the barrier in front of the PV MMAs (the logging variant syncs here itself)
  if (p.attn_mean != nullptr) {
    // materialising variant (logging path): third pass over the score row while S is still in TMEM — the normalised weights,
    // averaged over the heads by fp32 atomics (the head CTAs of a frame add into the same [L][L] map)
    float tot = sum;
    if (split) {
      __syncthreads();
      tot = xch[1][0][row] + xch[1][1][row];
    }
    const float w = 1.f / (tot * (float)p.heads);
    const int qq = q0 + row;
    float* arow = p.attn_mean + ((size_t)n * L + (qq < L ? qq : 0)) * L;
    if (L >= 32) {
      for (int c = c_lo; c < c_hi; c += 32) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(trow + c, v);
        if (qq < L) {
#pragma unroll
          for (int j = 0; j < 32; ++j) atomicAdd(arow + c + j, exp2f(fmaf(__uint_as_float(v[j]), p.scale_log2e, mneg)) * w);
        }
      }
    } else {
      uint32_t v[16];
      tmem_ld_32x32b_x16(trow, v);
      if (qq < L) {
#pragma unroll
        for (int j = 0; j < 16; ++j) atomicAdd(arow + j, exp2f(fmaf(__uint_as_float(v[j]), p.scale_log2e, mneg)) * w);
      }
    }
  }
  fence_proxy_async_smem();
  tcgen05_fence_before();
  __syncthreads();
  if (split) sum = xch[1][0][row] + xch[1][1][row];
  if (tid == 0) {
    mbar_wait(&bar_v, 0);
    tcgen05_fence_after();
    // ---- O = P V   (N chunks of <= 64 head dims; K = L keys in steps of 16)
    for (int c = 0; c < p.cf; ++c) {
      const int nf = min(64, F - c * 64);
      const uint32_t idesc = make_idesc(nf, /*b_mn_major=*/1);
      for (int ks = 0; ks < L / 16; ++ks) {
        const uint64_t ad = make_smem_desc(smem_u32(p_s + (ks >> 2) * 16384)) + 2 * (ks & 3);
        const uint64_t bd = make_smem_desc_mn(smem_u32(v_s + c * kv_tile + ks * 2048));
        umma_bf16(tmem + c * 64, ad, bd, idesc, ks != 0);
      }
    }
    umma_commit(&bar_o);
  }
  __syncwarp();
  if (hh == 0) {  // the output tile is F <= 128 columns: drained by the first four warps
  mbar_wait(&bar_o, 0);
  tcgen05_fence_after();
  const float inv = 1.f / sum;
  const int q = q0 + row;
  if (p.lse != nullptr && q < L) p.lse[((size_t)n * p.heads + h) * L + q] = mx * p.scale_log2e * 0.6931471805599453f + logf(sum);
  // O / rowsum -> bf16 -> out, 32 head dims (64 bytes per row) at a time through the warp's staging slice (p_s is dead: the PV
  // MMAs have retired), 4 lanes per row (see warp_store_rows64)
  uint8_t* stage = p_s + warp * 2560;
  const int lane = tid & 31;
  const size_t row0 = (size_t)n * L + q0 + warp * 32;
  for (int f = 0; f < F; f += 32) {
    uint32_t v[32];
    const bool two = f + 16 < F;  // F % 32 == 16: the last pass holds 16 head dims (2 pieces)
    {
      uint32_t a[16];
      tmem_ld_32x32b_x16(trow + f, a);
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = a[j];
      if (two) {
        tmem_ld_32x32b_x16(trow + f + 16, a);
#pragma unroll
        for (int j = 0; j < 16; ++j) v[16 + j] = a[j];
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[16 + j] = 0u;
      }
    }
    uint4 w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
      w[k] = make_uint4(pack2_bf16(__uint_as_float(v[8 * k]) * inv, __uint_as_float(v[8 * k + 1]) * inv),
                        pack2_bf16(__uint_as_float(v[8 * k + 2]) * inv, __uint_as_float(v[8 * k + 3]) * inv),
                        pack2_bf16(__uint_as_float(v[8 * k + 4]) * inv, __uint_as_float(v[8 * k + 5]) * inv),
                        pack2_bf16(__uint_as_float(v[8 * k + 6]) * inv, __uint_as_float(v[8 * k + 7]) * inv));
    warp_store_rows64(stage, lane, w, [&](int r) -> uint8_t* {
      return (q0 + warp * 32 + r < L) ? reinterpret_cast<uint8_t*>(p.out + (row0 + r) * C + h * F + f) : nullptr;
    }, two ? 4 : 2);
  }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(p.tmem_cols));
  }
}

static int pow2_at_least(int v, int lo) {
  int r = lo;
  while (r < v) r <<= 1;
  return r;
}

// returns FDM_ERR_UNSUPPORTED for shapes outside the kernel (the caller then uses the CUDA-core kernel)
int attn_spatial_tc_launch(const fdm_attn_spatial_args* a, cudaStream_t st) {
  const int F = a->C / a->heads, L = a->L;
  FDM_REQUIRE(a->qkv_dtype == FDM_BF16 && a->out_dtype == FDM_BF16, FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(F % 16 == 0 && F <= 128 && a->C % 8 == 0, FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(L == 16 || L == 32 || L == 64 || L == 128 || L == 256, FDM_ERR_UNSUPPORTED);
  SaTcParams p;
  p.out = reinterpret_cast<__nv_bfloat16*>(a->out);
  p.L = L; p.C = a->C; p.F = F; p.heads = a->heads;
  p.rows = L < 128 ? L : 128;
  p.cf = (F + 63) / 64;
  p.tmem_cols = pow2_at_least(L > F ? L : F, 32);
  p.scale_log2e = 1.4426950408889634f / sqrtf((float)F);
  p.lse = a->lse;
  p.attn_mean = a->attn_mean;
  EncodeTiledFn enc = get_tensormap_encoder();
  FDM_REQUIRE(enc != nullptr, FDM_ERR_UNSUPPORTED);
  CUtensorMap tq;
  cuuint64_t dims[3] = {(cuuint64_t)3 * a->C, (cuuint64_t)L, (cuuint64_t)a->N};
  cuuint64_t strides[2] = {(cuuint64_t)3 * a->C * 2, (cuuint64_t)L * 3 * a->C * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)p.rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  FDM_REQUIRE(enc(&tq, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(a->qkv), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS, FDM_ERR_UNSUPPORTED);
  const int kv_tile = L * 128;
  const int pbytes = ((L + 63) / 64) * 16384;
  const int qk = p.cf * (16384 + kv_tile);
  const int smem = p.cf * kv_tile + (qk > pbytes ? qk : pbytes) + 1024;
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] {
    attr_err = cudaFuncSetAttribute(attn_spatial_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  });
  if (attr_err != cudaSuccess) {
    set_last_error(attr_err);
    return FDM_ERR_CUDA;
  }
  FDM_REQUIRE(smem <= 200 * 1024, FDM_ERR_UNSUPPORTED);
  dim3 grid((L + 127) / 128, a->heads, a->N);
  // rows of >= SA_SPLIT_MIN_L keys: two threads per query row (256-thread CTAs)
  fdm::launch(attn_spatial_tc_kernel, dim3(grid), dim3(L >= SA_SPLIT_MIN_L ? 256 : 128), smem, st, tq, p);
  return check_launch();
}

}  // namespace fdm
