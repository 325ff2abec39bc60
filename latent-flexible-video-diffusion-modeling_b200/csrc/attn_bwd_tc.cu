// Spatial self-attention BACKWARD on tcgen05 (what autograd runs for rpe.py:139-144,163-166 without RPE / mask), bf16
// operands, fp32 accumulation in TMEM.  Same building blocks as the forward kernel (attn_tc.cu): 128-row tiles, TMA boxes of
// 64 channels in the 128B-swizzled layout, score rows in TMEM, P / dS written by the threads as swizzled K-major bf16 operands,
// the [rows][F] matrices consumed a second time as MN-major operands.
//
//   forward   S = scale Q K^T ; P = exp(S - lse) ; O = P V            (lse saved by the forward kernel)
//   backward  D_i = dO_i . O_i ; dP = dO V^T ; dS = P (dP - D) scale ; dQ = dS K ; dK = dS^T Q ; dV = P^T dO
//
// ONE kernel template, launched twice.  A CTA owns a 128-row tile of the "row" side and walks the "column" side in halves of
// 128 positions; per half:  TMA the two column matrices -> two score MMAs (M=128, N<=128, K=F) into TMEM columns [0,128) and
// [128,256) -> each thread turns its row into P / dS (bf16, swizzled smem) -> output MMAs (M=128, N=F, K=columns of the half)
// accumulate into TMEM columns [256, 256+F) and [384, 384+F) across the halves.
//   KV = false: rows = queries (Q, dO), columns = keys (K, V);   out1 = dS K            -> dQ        (row statistics)
//   KV = true : rows = keys (K, V),    columns = queries (Q, dO); out1 = dS^T Q -> dK, out2 = P^T dO -> dV   (column statistics)
#include "tc_common.cuh"
#include <mutex>

namespace fdm {

struct SaBwdTcParams {
  const __nv_bfloat16* out;   // forward output [N][L][C]
  const __nv_bfloat16* dout;  // [N][L][C]
  __nv_bfloat16* dqkv;        // [N][L][3C]
  float* lse;                 // [N][heads][L] from the forward kernel
  float* dsum;                // [N][heads][L]: written by the row pass (KV = false), read by the column pass
  int L, C, F, heads;
  int rows;  // TMA box rows = min(L, 128)
  int cf;    // 64-channel chunks per head
  float scale, scale_log2e;
};

__device__ __forceinline__ uint64_t sab_desc_mn(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;            // LBO: a single 64-element MN block per MMA (N <= 64)
  d |= (uint64_t)(1024 >> 4) << 32;  // SBO: stride between 8-row K groups
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ uint32_t sab_pack(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

template <bool KV>
__global__ void __launch_bounds__(128) attn_spatial_bwd_tc_kernel(const __grid_constant__ CUtensorMap tq,
                                                                  const __grid_constant__ CUtensorMap td, const SaBwdTcParams p) {
  extern __shared__ uint8_t sab_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(sab_smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t bar_rows, bar_cols, bar_s, bar_o;
  __shared__ uint32_t tmem_slot;
  __shared__ float col_lse[128], col_d[128];

  const int tid = threadIdx.x, warp = tid >> 5;
  const int r0 = blockIdx.x * 128, h = blockIdx.y, n = blockIdx.z;
  const int L = p.L, F = p.F, C = p.C, cf = p.cf;
  const int ncol = L < 128 ? L : 128;           // column positions per half
  const int halves = (L + 127) / 128;
  uint8_t* r1_s = smem;                          // [cf][128][128 B]  row operand of the score MMA #1 (Q | K)
  uint8_t* r2_s = r1_s + cf * 16384;             // row operand of score MMA #2 (dO | V)
  uint8_t* c1_s = r2_s + cf * 16384;             // [cf][128][128 B]  column matrix #1 of the half (K | Q)
  uint8_t* c2_s = c1_s + cf * 16384;             // column matrix #2 (V | dO)
  uint8_t* ds_s = c2_s + cf * 16384;             // [2][128][128 B]   dS tile (K-major over the half's columns)
  uint8_t* p_s = ds_s + 2 * 16384;               // [2][128][128 B]   P tile (KV only)

  if (tid == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tq) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&td) : "memory");
    mbar_init(&bar_rows, 1);
    mbar_init(&bar_cols, 1);
    mbar_init(&bar_s, 1);
    mbar_init(&bar_o, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "n"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  pdl_wait();

  const int row = r0 + tid;                      // this thread's row (TMEM lane tid)
  const bool row_ok = row < L;
  const size_t stat0 = ((size_t)n * p.heads + h) * L;
  float row_lse = 0.f, row_d = 0.f;
  if (!KV) {
    // D_i = dO_i . O_i from global memory (F bf16 values each), lse_i from the forward pass
    if (row_ok) {
      const __nv_bfloat16* o = p.out + ((size_t)n * L + row) * C + h * F;
      const __nv_bfloat16* d = p.dout + ((size_t)n * L + row) * C + h * F;
      float acc = 0.f;
      for (int f = 0; f < F; f += 8) {
        const uint4 a = *reinterpret_cast<const uint4*>(o + f), b = *reinterpret_cast<const uint4*>(d + f);
        const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc = fmaf(__uint_as_float(aw[j] << 16), __uint_as_float(bw[j] << 16), acc);
          acc = fmaf(__uint_as_float(aw[j] & 0xffff0000u), __uint_as_float(bw[j] & 0xffff0000u), acc);
        }
      }
      row_d = acc;
      row_lse = p.lse[stat0 + row];
      p.dsum[stat0 + row] = acc;
    }
  }

  if (tid == 0) {
    // row operands: loaded once
    mbar_expect_tx(&bar_rows, (uint32_t)(2 * cf * p.rows * 128));
    for (int c = 0; c < cf; ++c) {
      const int ch = h * F + c * 64;
      if (KV) {
        tma_load_3d(r1_s + c * 16384, &tq, &bar_rows, C + ch, r0, n);       // K rows
        tma_load_3d(r2_s + c * 16384, &tq, &bar_rows, 2 * C + ch, r0, n);   // V rows
      } else {
        tma_load_3d(r1_s + c * 16384, &tq, &bar_rows, ch, r0, n);           // Q rows
        tma_load_3d(r2_s + c * 16384, &td, &bar_rows, ch, r0, n);           // dO rows
      }
    }
  }
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
  const int sw = tid & 7;
  for (int hf = 0; hf < halves; ++hf) {
    const int c0 = hf * 128;
    if (tid == 0) {
      if (hf > 0) {  // the previous half's output MMAs still read the column matrices and the P / dS tiles
        mbar_wait(&bar_o, (hf - 1) & 1);
        tcgen05_fence_after();
      }
      mbar_expect_tx(&bar_cols, (uint32_t)(2 * cf * p.rows * 128));
      for (int c = 0; c < cf; ++c) {
        const int ch = h * F + c * 64;
        if (KV) {
          tma_load_3d(c1_s + c * 16384, &tq, &bar_cols, ch, c0, n);           // Q
          tma_load_3d(c2_s + c * 16384, &td, &bar_cols, ch, c0, n);           // dO
        } else {
          tma_load_3d(c1_s + c * 16384, &tq, &bar_cols, C + ch, c0, n);       // K
          tma_load_3d(c2_s + c * 16384, &tq, &bar_cols, 2 * C + ch, c0, n);   // V
        }
      }
      if (hf == 0) mbar_wait(&bar_rows, 0);
      mbar_wait(&bar_cols, hf & 1);
      tcgen05_fence_after();
      // ---- scores: S (cols [0,128)) = R1 C1^T, dP (cols [128,256)) = R2 C2^T ; both operands K-major, K = F
      const uint32_t idesc = make_idesc(ncol);
      for (int ks = 0; ks < F / 16; ++ks) {
        const int c = ks >> 2, kk = ks & 3;
        umma_bf16(tmem, make_smem_desc(smem_u32(r1_s + c * 16384)) + 2 * kk, make_smem_desc(smem_u32(c1_s + c * 16384)) + 2 * kk,
                  idesc, ks != 0);
      }
      for (int ks = 0; ks < F / 16; ++ks) {
        const int c = ks >> 2, kk = ks & 3;
        umma_bf16(tmem + 128, make_smem_desc(smem_u32(r2_s + c * 16384)) + 2 * kk, make_smem_desc(smem_u32(c2_s + c * 16384)) + 2 * kk,
                  idesc, ks != 0);
      }
      umma_commit(&bar_s);
    }
    if (KV) {  // column statistics of this half (every thread of the previous half is past its last read: __syncthreads below)
      const int j = c0 + tid;
      col_lse[tid] = (tid < ncol && j < L) ? p.lse[stat0 + j] : 0.f;
      col_d[tid] = (tid < ncol && j < L) ? p.dsum[stat0 + j] : 0.f;
    }
    __syncthreads();
    mbar_wait(&bar_s, hf & 1);
    tcgen05_fence_after();
    // ---- this thread's row of the half: P = exp(S scale - lse), dS = P (dP - D) scale -> swizzled K-major bf16 tiles
    for (int c = 0; c < ncol; c += 16) {
      uint32_t sv[16], dv[16];
      tmem_ld_32x32b_x16(trow + c, sv);
      tmem_ld_32x32b_x16(trow + 128 + c, dv);
      float pv[16], ds[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float lse = KV ? col_lse[c + j] : row_lse;
        const float dd = KV ? col_d[c + j] : row_d;
        const float P = exp2f(fmaf(__uint_as_float(sv[j]), p.scale_log2e, -lse * 1.4426950408889634f));
        pv[j] = P;
        ds[j] = P * (__uint_as_float(dv[j]) - dd) * p.scale;
      }
      const int piece0 = (c & 63) >> 3;
      uint8_t* drow = ds_s + (c >> 6) * 16384 + tid * 128;
#pragma unroll
      for (int q = 0; q < 2; ++q)
        *reinterpret_cast<uint4*>(drow + (((piece0 + q) ^ sw) << 4)) =
            make_uint4(sab_pack(ds[8 * q], ds[8 * q + 1]), sab_pack(ds[8 * q + 2], ds[8 * q + 3]),
                       sab_pack(ds[8 * q + 4], ds[8 * q + 5]), sab_pack(ds[8 * q + 6], ds[8 * q + 7]));
      if (KV) {
        uint8_t* prow = p_s + (c >> 6) * 16384 + tid * 128;
#pragma unroll
        for (int q = 0; q < 2; ++q)
          *reinterpret_cast<uint4*>(prow + (((piece0 + q) ^ sw) << 4)) =
              make_uint4(sab_pack(pv[8 * q], pv[8 * q + 1]), sab_pack(pv[8 * q + 2], pv[8 * q + 3]),
                         sab_pack(pv[8 * q + 4], pv[8 * q + 5]), sab_pack(pv[8 * q + 6], pv[8 * q + 7]));
      }
    }
    fence_proxy_async_smem();
    tcgen05_fence_before();
    __syncthreads();
    if (tid == 0) {
      tcgen05_fence_after();
      // ---- outputs: out1 (cols [256, 256+F)) += dS C1 ; out2 (cols [384, 384+F)) += P C2 ; A K-major over the half's columns,
      //      B = the column matrix read as an MN-major operand (N chunks of <= 64 head dims)
      for (int c = 0; c < cf; ++c) {
        const int nf = min(64, F - c * 64);
        const uint32_t idesc = make_idesc(nf, /*b_mn_major=*/1);
        for (int ks = 0; ks < ncol / 16; ++ks) {
          const uint64_t ad = make_smem_desc(smem_u32(ds_s + (ks >> 2) * 16384)) + 2 * (ks & 3);
          umma_bf16(tmem + 256 + c * 64, ad, sab_desc_mn(smem_u32(c1_s + c * 16384 + ks * 2048)), idesc, (hf | ks) != 0);
        }
        if (KV) {
          for (int ks = 0; ks < ncol / 16; ++ks) {
            const uint64_t ad = make_smem_desc(smem_u32(p_s + (ks >> 2) * 16384)) + 2 * (ks & 3);
            umma_bf16(tmem + 384 + c * 64, ad, sab_desc_mn(smem_u32(c2_s + c * 16384 + ks * 2048)), idesc, (hf | ks) != 0);
          }
        }
      }
      umma_commit(&bar_o);
    }
    __syncwarp();
  }
  mbar_wait(&bar_o, (halves - 1) & 1);
  tcgen05_fence_after();
  // ---- epilogue: this thread's output row(s) -> dqkv (bf16)
  __nv_bfloat16* drow = p.dqkv + ((size_t)n * L + (row_ok ? row : 0)) * 3 * C + h * F;
  for (int f = 0; f < F; f += 16) {
    uint32_t v[16];
    tmem_ld_32x32b_x16(trow + 256 + f, v);
    if (row_ok) {
      __nv_bfloat16* d = drow + (KV ? C : 0) + f;  // dK | dQ
      *reinterpret_cast<uint4*>(d) = make_uint4(sab_pack(__uint_as_float(v[0]), __uint_as_float(v[1])), sab_pack(__uint_as_float(v[2]), __uint_as_float(v[3])),
                                                sab_pack(__uint_as_float(v[4]), __uint_as_float(v[5])), sab_pack(__uint_as_float(v[6]), __uint_as_float(v[7])));
      *reinterpret_cast<uint4*>(d + 8) = make_uint4(sab_pack(__uint_as_float(v[8]), __uint_as_float(v[9])), sab_pack(__uint_as_float(v[10]), __uint_as_float(v[11])),
                                                    sab_pack(__uint_as_float(v[12]), __uint_as_float(v[13])), sab_pack(__uint_as_float(v[14]), __uint_as_float(v[15])));
    }
    if (KV) {
      tmem_ld_32x32b_x16(trow + 384 + f, v);
      if (row_ok) {
        __nv_bfloat16* d = drow + 2 * C + f;  // dV
        *reinterpret_cast<uint4*>(d) = make_uint4(sab_pack(__uint_as_float(v[0]), __uint_as_float(v[1])), sab_pack(__uint_as_float(v[2]), __uint_as_float(v[3])),
                                                  sab_pack(__uint_as_float(v[4]), __uint_as_float(v[5])), sab_pack(__uint_as_float(v[6]), __uint_as_float(v[7])));
        *reinterpret_cast<uint4*>(d + 8) = make_uint4(sab_pack(__uint_as_float(v[8]), __uint_as_float(v[9])), sab_pack(__uint_as_float(v[10]), __uint_as_float(v[11])),
                                                      sab_pack(__uint_as_float(v[12]), __uint_as_float(v[13])), sab_pack(__uint_as_float(v[14]), __uint_as_float(v[15])));
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512));
  }
}

static bool sab_encode(CUtensorMap* m, const void* ptr, int N, int L, int Cs, int rows) {
  EncodeTiledFn enc = get_tensormap_encoder();
  if (!enc) return false;
  cuuint64_t dims[3] = {(cuuint64_t)Cs, (cuuint64_t)L, (cuuint64_t)N};
  cuuint64_t strides[2] = {(cuuint64_t)Cs * 2, (cuuint64_t)L * Cs * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// returns FDM_ERR_UNSUPPORTED for shapes outside the kernel (the caller then uses the CUDA-core kernels)
int attn_spatial_bwd_tc_launch(const fdm_attn_spatial_bwd_args* a, cudaStream_t st) {
  const int F = a->C / a->heads, L = a->L;
  FDM_REQUIRE(a->dtype == FDM_BF16 && a->lse_from_forward, FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(F % 16 == 0 && F <= 128 && a->C % 8 == 0, FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(L == 16 || L == 32 || L == 64 || L == 128 || L == 256, FDM_ERR_UNSUPPORTED);
  SaBwdTcParams p;
  p.out = reinterpret_cast<const __nv_bfloat16*>(a->out);
  p.dout = reinterpret_cast<const __nv_bfloat16*>(a->dout);
  p.dqkv = reinterpret_cast<__nv_bfloat16*>(a->dqkv);
  p.lse = a->lse; p.dsum = a->dsum;
  p.L = L; p.C = a->C; p.F = F; p.heads = a->heads;
  p.rows = L < 128 ? L : 128;
  p.cf = (F + 63) / 64;
  p.scale = 1.0f / sqrtf((float)F);
  p.scale_log2e = 1.4426950408889634f * p.scale;
  CUtensorMap tq, td;
  FDM_REQUIRE(sab_encode(&tq, a->qkv, a->N, L, 3 * a->C, p.rows) && sab_encode(&td, a->dout, a->N, L, a->C, p.rows), FDM_ERR_UNSUPPORTED);
  const int smem = 4 * p.cf * 16384 + 4 * 16384 + 1024;
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] {
    attr_err = cudaFuncSetAttribute(attn_spatial_bwd_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (attr_err == cudaSuccess)
      attr_err = cudaFuncSetAttribute(attn_spatial_bwd_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  });
  if (attr_err != cudaSuccess) {
    set_last_error(attr_err);
    return FDM_ERR_CUDA;
  }
  FDM_REQUIRE(smem <= 200 * 1024, FDM_ERR_UNSUPPORTED);
  dim3 grid((L + 127) / 128, a->heads, a->N);
  fdm::launch(attn_spatial_bwd_tc_kernel<false>, grid, dim3(128), smem, st, tq, td, p);
  fdm::launch(attn_spatial_bwd_tc_kernel<true>, grid, dim3(128), smem, st, tq, td, p);
  return check_launch();
}

}  // namespace fdm
