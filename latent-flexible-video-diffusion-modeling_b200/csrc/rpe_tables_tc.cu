// All RPENet tables of one denoiser forward in ONE launch (rpe.py:20-31; 3 nets per temporal attention, 21 per forward):
//   R[b,t,s,:] = W_o . SiLU( W_t temb[b] + b_t  +  W_d phi(fi[b,t] - fi[b,s]) + b_d ) + b_o
//   phi(d) = [log(1 + max(d, 0)), log(1 + max(-d, 0)), 1[d == 0]]                              (rpe.py:21-26)
// The hidden layer is the A operand of a [B*T*T x C] . [C x C] GEMM per net.  It never goes to memory: each CTA GENERATES its
// 128-row x 64-channel A chunks straight into shared memory in the swizzled K-major layout tcgen05.mma reads (3 features per row,
// C FMAs + SiLU per element), W_o chunks arrive by TMA from a per-net tensor map kept in a DEVICE array, accumulators in TMEM,
// and the epilogue writes the bf16 (and/or fp32) table with coalesced row segments.  Replaces fdm_rpe_hidden + one fdm_conv per
// net (22 launches, the hidden tensors written and re-read) on inference plans.
#include "tc_common.cuh"
#include <string.h>

namespace fdm {

struct RtProblem {  // device-side copy of fdm_rpe_table_problem (32-byte aligned entries after the tensor maps in the blob)
  const float* wd;
  const float* bd;
  const float* bo;
  __nv_bfloat16* out_op;
  float* out_f32;
  int C, te_off;
};

struct RtParams {
  const CUtensorMap* wmaps;  // [count], global memory
  const RtProblem* probs;    // [count]
  const float* te;
  const int64_t* fi;
  int B, T, te_stride, M;
  int wstage;  // bytes of one W_o stage in shared memory: round_up(max_C, 128) * 128
};

// grid (ceil(M/128), 1, nets); 128 threads; thread r <-> table row m0 + r <-> TMEM lane r.  One CTA computes ALL C output channels
// of its 128 rows (accumulators: C <= 512 TMEM columns), so the hidden-layer chunk is generated once per K chunk.
__global__ void __launch_bounds__(128) rpe_tables_kernel(const RtParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t w_full[2], mma_done[2], bar_d;
  __shared__ uint32_t tmem_slot;
  const RtProblem pr = p.probs[blockIdx.z];
  const int C = pr.C;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m0 = blockIdx.x * 128;
  const CUtensorMap* wmap = p.wmaps + blockIdx.z;
  const int Cn = (C + 15) / 16 * 16;           // GEMM N extent (weights beyond C are zero-filled by TMA)
  const int ntiles = (Cn + 127) / 128;         // 128-column accumulator tiles
  const int wstage = p.wstage;                 // bytes of one W stage = round_up(max_C, 128) * 128
  uint8_t* a_s = smem;                         // [2][128][128 B]
  uint8_t* w_s = smem + 2 * 16384;             // [2][ntiles][128][128 B]
  float4* coef_s = reinterpret_cast<float4*>(w_s + 2 * wstage);  // [round_up(C, 64)]: {wd0, wd1, wd2, bd} per hidden channel
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < Cn) tmem_cols <<= 1;
  if (tid == 0) {
    // the tensor map lives in global memory (written by the host before the first launch): make it visible to the TMA unit
    asm volatile("fence.proxy.tensormap::generic.acquire.gpu [%0], 128;" ::"l"(wmap) : "memory");
    prefetch_tmap(wmap);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&w_full[i], 1);
      mbar_init(&mma_done[i], 1);
    }
    mbar_init(&bar_d, 1);
    fence_mbarrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_slot, tmem_cols);
  const int kchunks = (C + 63) / 64;
  for (int c = tid; c < kchunks * 64; c += 128)  // parameters: not produced by the previous kernel, safe before pdl_wait
    coef_s[c] = c < C ? make_float4(__ldg(pr.wd + c * 3), __ldg(pr.wd + c * 3 + 1), __ldg(pr.wd + c * 3 + 2), __ldg(pr.bd + c))
                      : make_float4(0.f, 0.f, 0.f, 0.f);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  pdl_wait();

  // this thread's row m = (b, t, s): the three distance features and the row of W_t temb + b_t it adds
  const int m = m0 + tid;
  const bool row_ok = m < p.M;
  float f0 = 0.f, f1 = 0.f, f2 = 0.f;
  const float* terow = p.te + pr.te_off;
  if (row_ok) {
    const int s = m % p.T, bt = m / p.T;
    const int t = bt % p.T, b = bt / p.T;
    const float d = (float)(p.fi[(size_t)b * p.T + t] - p.fi[(size_t)b * p.T + s]);
    f0 = logf(1.f + fmaxf(d, 0.f));
    f1 = logf(1.f + fmaxf(-d, 0.f));
    f2 = d == 0.f ? 1.f : 0.f;
    terow += (size_t)b * p.te_stride;
  }
  for (int kc = 0; kc < kchunks; ++kc) {
    const int st = kc & 1;
    if (kc >= 2) mbar_wait(&mma_done[st], ((kc >> 1) - 1) & 1);  // the MMAs that read this stage two chunks ago have retired
    if (tid == 0) {
      mbar_expect_tx(&w_full[st], (uint32_t)ntiles * 16384);
      for (int j = 0; j < ntiles; ++j) tma_load_3d(w_s + st * wstage + j * 16384, wmap, &w_full[st], kc * 64, j * 128, 0);
    }
    // generate the hidden-layer chunk: row `tid`, channels [64 kc, 64 kc + 64) -> 8 swizzled 16-byte pieces.  The hidden values are
    // rounded to bf16 right away, so the fast SiLU (ex2.approx / rcp.approx, ~1e-6 relative) is exact at the stored precision.
    uint8_t* arow = a_s + st * 16384 + tid * 128;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int c0 = kc * 64 + q * 8;
      float tev[8];
      if (row_ok && c0 + 8 <= C) {
        const float4 t0 = __ldg(reinterpret_cast<const float4*>(terow + c0)), t1 = __ldg(reinterpret_cast<const float4*>(terow + c0 + 4));
        tev[0] = t0.x; tev[1] = t0.y; tev[2] = t0.z; tev[3] = t0.w; tev[4] = t1.x; tev[5] = t1.y; tev[6] = t1.z; tev[7] = t1.w;
      } else {
#pragma unroll
        for (int u = 0; u < 8; ++u) tev[u] = (row_ok && c0 + u < C) ? __ldg(terow + c0 + u) : 0.f;
      }
      float hv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const float4 cf = coef_s[c0 + u];  // same address for the whole warp: broadcast
        const float e = fmaf(f2, cf.z, fmaf(f1, cf.y, f0 * cf.x)) + cf.w + tev[u];
        hv[u] = (row_ok && c0 + u < C) ? silu_f(e) : 0.f;
      }
      *reinterpret_cast<uint4*>(arow + ((q ^ (tid & 7)) << 4)) =
          make_uint4(pack2_bf16(hv[0], hv[1]), pack2_bf16(hv[2], hv[3]), pack2_bf16(hv[4], hv[5]), pack2_bf16(hv[6], hv[7]));
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
      mbar_wait(&w_full[st], (kc >> 1) & 1);
      tcgen05_fence_after();
      const int nk = min(4, (C - kc * 64 + 15) / 16);
      for (int j = 0; j < ntiles; ++j) {
        const uint32_t idesc = make_idesc(min(128, Cn - j * 128));
        for (int k = 0; k < nk; ++k)
          umma_bf16(tmem + j * 128, make_smem_desc(smem_u32(a_s + st * 16384)) + 2 * k,
                    make_smem_desc(smem_u32(w_s + st * wstage + j * 16384)) + 2 * k, idesc, (kc | k) != 0);
      }
      umma_commit(&mma_done[st]);
      if (kc == kchunks - 1) umma_commit(&bar_d);
    }
    __syncwarp();
  }
  mbar_wait(&bar_d, 0);
  tcgen05_fence_after();
  // ---- epilogue: + b_o, bf16 and/or fp32 table rows, 64-byte row segments with 4 lanes per row (warp_store_rows64)
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
  uint8_t* stage = smem + warp * 2560;  // operand stages are dead
  for (int c0 = 0; c0 < Cn; c0 += 16) {
    uint32_t v[16];
    tmem_ld_32x32b_x16(trow + c0, v);
    float o[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) o[j] = __uint_as_float(v[j]) + (c0 + j < C ? __ldg(pr.bo + c0 + j) : 0.f);
    auto rowp = [&](int r, size_t esz) -> size_t {  // byte offset of row r's first column of this chunk, or ~0 to skip
      const int mm = m0 + warp * 32 + r;
      return mm < p.M ? ((size_t)mm * C + c0) * esz : ~(size_t)0;
    };
    const int cols = min(16, C - c0);  // C % 8 == 0
    if (pr.out_op != nullptr) {
      uint4 w[4];
      w[0] = make_uint4(pack2_bf16(o[0], o[1]), pack2_bf16(o[2], o[3]), pack2_bf16(o[4], o[5]), pack2_bf16(o[6], o[7]));
      w[1] = make_uint4(pack2_bf16(o[8], o[9]), pack2_bf16(o[10], o[11]), pack2_bf16(o[12], o[13]), pack2_bf16(o[14], o[15]));
      w[2] = w[3] = make_uint4(0u, 0u, 0u, 0u);
      warp_store_rows64(stage, lane, w, [&](int r) -> uint8_t* {
        const size_t off = rowp(r, 2);
        return off == ~(size_t)0 ? nullptr : reinterpret_cast<uint8_t*>(pr.out_op) + off;
      }, cols / 8);
    }
    if (pr.out_f32 != nullptr) {
      uint4 w[4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
        w[k] = make_uint4(__float_as_uint(o[4 * k]), __float_as_uint(o[4 * k + 1]), __float_as_uint(o[4 * k + 2]), __float_as_uint(o[4 * k + 3]));
      warp_store_rows64(stage, lane, w, [&](int r) -> uint8_t* {
        const size_t off = rowp(r, 4);
        return off == ~(size_t)0 ? nullptr : reinterpret_cast<uint8_t*>(pr.out_f32) + off;
      }, cols / 4);
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc(tmem, tmem_cols);
  }
}

}  // namespace fdm

using namespace fdm;

extern "C" size_t fdm_rpe_tables_blob_bytes(int32_t count) {
  return count <= 0 ? 0 : (size_t)count * (sizeof(CUtensorMap) + sizeof(RtProblem));
}

// Host-side preparation (once per plan): encode one tensor map per net for its packed W_o (bf16 [1][co_pad16][ci_pad64], the
// FDM_PACK_TC_FWD layout of fdm_pack_weights / the engine's packer) and lay out the device blob = [count tensor maps][count problems].
extern "C" int fdm_rpe_tables_prepare(const fdm_rpe_table_problem* problems, int32_t count, void* host_blob, size_t blob_bytes) {
  FDM_REQUIRE(problems && count > 0 && host_blob, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(blob_bytes >= fdm_rpe_tables_blob_bytes(count), FDM_ERR_BAD_ARG);
  static_assert(sizeof(CUtensorMap) == 128, "CUtensorMap is 128 bytes");
  uint8_t* blob = reinterpret_cast<uint8_t*>(host_blob);
  for (int i = 0; i < count; ++i) {
    const fdm_rpe_table_problem& q = problems[i];
    FDM_REQUIRE(q.wd && q.bd && q.bo && q.w_packed && (q.out_op || q.out_f32) && q.C > 0 && q.C % 8 == 0 && q.te_off % 4 == 0, FDM_ERR_BAD_ARG);
    const int ci_pad = (q.C + 63) / 64 * 64, co_pad = (q.C + 15) / 16 * 16;
    CUtensorMap m;
    const cuuint64_t dims[3] = {(cuuint64_t)ci_pad, (cuuint64_t)co_pad, 1};
    const cuuint32_t box[3] = {64, 128, 1};
    FDM_REQUIRE(encode_bf16_map(&m, q.w_packed, 3, dims, box, CU_TENSOR_MAP_L2_PROMOTION_L2_256B), FDM_ERR_UNSUPPORTED);
    memcpy(blob + (size_t)i * sizeof(CUtensorMap), &m, sizeof(CUtensorMap));
    RtProblem d{q.wd, q.bd, q.bo, reinterpret_cast<__nv_bfloat16*>(q.out_op), q.out_f32, q.C, q.te_off};
    memcpy(blob + (size_t)count * sizeof(CUtensorMap) + (size_t)i * sizeof(RtProblem), &d, sizeof(RtProblem));
  }
  return FDM_OK;
}

extern "C" int fdm_rpe_tables(const fdm_rpe_tables_args* a, void* stream) {
  FDM_REQUIRE(a && a->te && a->frame_indices && a->blob && a->count > 0 && a->B > 0 && a->T > 0 && a->max_C > 0, FDM_ERR_BAD_ARG);
  FDM_REQUIRE((reinterpret_cast<uintptr_t>(a->blob) & 127) == 0, FDM_ERR_BAD_ARG);  // tensor maps need 128-byte alignment
  RtParams p;
  p.wmaps = reinterpret_cast<const CUtensorMap*>(a->blob);
  p.probs = reinterpret_cast<const RtProblem*>(reinterpret_cast<const uint8_t*>(a->blob) + (size_t)a->count * sizeof(CUtensorMap));
  p.te = a->te; p.fi = a->frame_indices; p.B = a->B; p.T = a->T; p.te_stride = a->te_stride;
  p.M = a->B * a->T * a->T;
  FDM_REQUIRE(a->max_C <= 512 && a->te_stride % 4 == 0, FDM_ERR_UNSUPPORTED);  // one CTA holds all C output channels of its rows in TMEM (512 columns)
  p.wstage = (a->max_C + 127) / 128 * 128 * 128;
  const int smem_bytes = 2 * 16384 + 2 * p.wstage + (a->max_C + 63) / 64 * 64 * 16 + 1024;
  dim3 grid((p.M + 127) / 128, 1, a->count);
  if (int rc = allow_smem(rpe_tables_kernel, 200 * 1024)) return rc;
  fdm::launch(rpe_tables_kernel, grid, dim3(128), smem_bytes, (cudaStream_t)stream, p);
  return check_launch();
}
