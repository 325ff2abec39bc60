// Attention cores on CUDA cores (fp32 math, fp32 softmax), used by both precision modes:
//   * temporal attention with the contextual relative-position terms and the two-group mask computed
//     in-kernel (rpe.py:139-170): sequences are T <= 40 frames, far below the tcgen05 tile minimum
//     (M = 64/128), so the QK^T part runs on CUDA cores (SURVEY §7 "hard parts").
//   * spatial attention (rpe.py:139-144,163-166 with no RPE / mask): flash-style streaming softmax.
#include "common.cuh"

namespace fdm {

// =====================================================================================================
// temporal attention
//   grid (ceil(HW/32), heads, B); block 256 = 8 warps; lane <-> pixel, warp <-> query frame t
//   S[t,s] = scale*( q_t.k_s + q_t.Rk[t,s] + k_s.Rq[s,t] );  P = softmax over {s : mask_s == mask_t}
//   O[t]   = sum_s P[t,s] * (v_s + Rv[t,s])
// =====================================================================================================
constexpr int TA_FC = 8;       // head-dim chunk staged in shared memory
constexpr int TA_MAX_WARPS = 12;

struct TAParams {
  const void* qkv; const float* Rq; const float* Rk; const float* Rv; const float* mask; void* out;
  int B, T, HW, C, heads, F, tgroups, nw;
  float scale;
};

// K/V chunk in shared memory as [s][f][32 px]: fp32 for fp32 inputs, packed bf16 pairs for bf16 inputs (half the
// shared-memory traffic: ncu showed this kernel bound by L1/shared bandwidth, not by FMA issue)
template <typename QT>
struct KvTile;
template <>
struct KvTile<float> {
  static constexpr int WORDS_PER_S = TA_FC * 32;
  static __device__ __forceinline__ void stage(float* kv, int s, int fq, int pl, const float* src) {
    float4 v = *reinterpret_cast<const float4*>(src);
    float* d = kv + ((size_t)s * TA_FC + fq * 4) * 32 + pl;
    d[0] = v.x; d[32] = v.y; d[64] = v.z; d[96] = v.w;
  }
  static __device__ __forceinline__ void load(const float* kv, int s, int lane, float (&k)[TA_FC]) {
#pragma unroll
    for (int f = 0; f < TA_FC; ++f) k[f] = kv[((size_t)s * TA_FC + f) * 32 + lane];
  }
};
template <>
struct KvTile<__nv_bfloat16> {
  static constexpr int WORDS_PER_S = (TA_FC / 2) * 32;
  static __device__ __forceinline__ void stage(float* kv, int s, int fq, int pl, const __nv_bfloat16* src) {
    uint2 u = *reinterpret_cast<const uint2*>(src);  // 4 bf16 = 2 pairs
    uint32_t* d = reinterpret_cast<uint32_t*>(kv) + ((size_t)s * (TA_FC / 2) + fq * 2) * 32 + pl;
    d[0] = u.x; d[32] = u.y;
  }
  static __device__ __forceinline__ void load(const float* kv, int s, int lane, float (&k)[TA_FC]) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(kv) + (size_t)s * (TA_FC / 2) * 32 + lane;
#pragma unroll
    for (int fp = 0; fp < TA_FC / 2; ++fp) {
      const uint32_t u = w[fp * 32];
      k[2 * fp] = __uint_as_float(u << 16);
      k[2 * fp + 1] = __uint_as_float(u & 0xffff0000u);
    }
  }
};

// grid (ceil(HW/32), heads, B * tgroups); block = nw warps.  Warp w owns TPW query frames t = (tg*nw + w)*TPW + u for 32
// pixels (lane <-> pixel): every K/V value read from shared memory is used for TPW queries.  Per head-dim chunk of 8:
// K (then V) of ALL T key frames is staged once per block; each warp stages ITS rows Rk[t,:,chunk], Rq[:,t,chunk]
// (then Rv[t,:,chunk]) into a private slice with lane-parallel loads and reads them back as float4 broadcasts.
template <int TP, int TPW, typename QT, typename OT>
__global__ void __launch_bounds__(TA_MAX_WARPS * 32) attn_temporal_kernel(TAParams p) {
  pdl_wait();
  extern __shared__ __align__(16) float ta_smem[];
  using KV = KvTile<QT>;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nthreads = blockDim.x;
  const int T = p.T, C = p.C, F = p.F, HW = p.HW;
  float* kv = ta_smem;                                                     // [T][chunk][32]
  float* ra = ta_smem + (size_t)T * KV::WORDS_PER_S + (size_t)w * 2 * TPW * T * TA_FC;  // [TPW][T][TA_FC]: Rk / Rv
  float* rb = ra + (size_t)TPW * T * TA_FC;                                // [TPW][T][TA_FC]: Rq
  const int px0 = blockIdx.x * 32, h = blockIdx.y;
  const int b = blockIdx.z / p.tgroups, tg = blockIdx.z - b * p.tgroups;
  const int px = min(px0 + lane, HW - 1);
  const bool px_ok = px0 + lane < HW;
  const QT* qkv = reinterpret_cast<const QT*>(p.qkv);
  const size_t tok_stride = (size_t)3 * C;  // per (frame, pixel)
  const float* maskb = p.mask ? p.mask + (size_t)b * T : nullptr;
  int tq[TPW];
  bool act[TPW];
#pragma unroll
  for (int u = 0; u < TPW; ++u) {
    const int t = (tg * p.nw + w) * TPW + u;
    act[u] = t < T;
    tq[u] = act[u] ? t : 0;
  }

  float S[TPW][TP];
#pragma unroll
  for (int u = 0; u < TPW; ++u)
#pragma unroll
    for (int s = 0; s < TP; ++s) S[u][s] = 0.f;
  // ---------------- scores
  for (int f0 = 0; f0 < F; f0 += TA_FC) {
    __syncthreads();
    for (int i = threadIdx.x; i < T * 32 * (TA_FC / 4); i += nthreads) {
      int fq = i % (TA_FC / 4);
      int pl = (i / (TA_FC / 4)) % 32;
      int s = i / (32 * (TA_FC / 4));
      int pp = min(px0 + pl, HW - 1);
      KV::stage(kv, s, fq, pl, qkv + ((size_t)(b * T + s) * HW + pp) * tok_stride + C + h * F + f0 + fq * 4);
    }
    float q[TPW][TA_FC];
#pragma unroll
    for (int u = 0; u < TPW; ++u) {
      for (int i = lane; i < T * TA_FC; i += 32) {
        int s = i / TA_FC, f = i - s * TA_FC;
        ra[u * T * TA_FC + i] = __ldg(p.Rk + (((size_t)(b * T + tq[u]) * T + s) * C + h * F + f0 + f));
        rb[u * T * TA_FC + i] = __ldg(p.Rq + (((size_t)(b * T + s) * T + tq[u]) * C + h * F + f0 + f));
      }
      const QT* qrow = qkv + ((size_t)(b * T + tq[u]) * HW + px) * tok_stride + h * F + f0;
      float4 a = OpType<QT>::load4(qrow), c = OpType<QT>::load4(qrow + 4);
      q[u][0] = a.x; q[u][1] = a.y; q[u][2] = a.z; q[u][3] = a.w; q[u][4] = c.x; q[u][5] = c.y; q[u][6] = c.z; q[u][7] = c.w;
    }
    __syncthreads();
#pragma unroll
    for (int s = 0; s < TP; ++s) {
      if (s < T) {
        float kk[TA_FC];
        KV::load(kv, s, lane, kk);
#pragma unroll
        for (int u = 0; u < TPW; ++u) {
          const float* rka = ra + (u * T + s) * TA_FC;
          const float* rqa = rb + (u * T + s) * TA_FC;
          const float4 rk0 = *reinterpret_cast<const float4*>(rka), rk1 = *reinterpret_cast<const float4*>(rka + 4);
          const float4 rq0 = *reinterpret_cast<const float4*>(rqa), rq1 = *reinterpret_cast<const float4*>(rqa + 4);
          const float rkv[8] = {rk0.x, rk0.y, rk0.z, rk0.w, rk1.x, rk1.y, rk1.z, rk1.w};
          const float rqv[8] = {rq0.x, rq0.y, rq0.z, rq0.w, rq1.x, rq1.y, rq1.z, rq1.w};
          float acc0 = S[u][s], acc1 = 0.f;  // two independent FMA chains
#pragma unroll
          for (int f = 0; f < TA_FC; ++f) {
            acc0 = fmaf(q[u][f], kk[f] + rkv[f], acc0);
            acc1 = fmaf(kk[f], rqv[f], acc1);
          }
          S[u][s] = acc0 + acc1;
        }
      }
    }
  }
  // ---------------- masked softmax (fp32)
#pragma unroll
  for (int u = 0; u < TPW; ++u) {
    const bool gt = maskb ? maskb[tq[u]] > 0.5f : true;
    float mx = -INFINITY;
#pragma unroll
    for (int s = 0; s < TP; ++s) {
      if (s < T) {
        bool ok = maskb ? ((maskb[s] > 0.5f) == gt) : true;
        S[u][s] = ok ? S[u][s] * p.scale : -INFINITY;
        mx = fmaxf(mx, S[u][s]);
      }
    }
    float sum = 0.f;
#pragma unroll
    for (int s = 0; s < TP; ++s) {
      if (s < T) {
        S[u][s] = expf(S[u][s] - mx);
        sum += S[u][s];
      }
    }
    const float inv = 1.f / sum;
#pragma unroll
    for (int s = 0; s < TP; ++s)
      if (s < T) S[u][s] *= inv;
  }
  // ---------------- output
  for (int f0 = 0; f0 < F; f0 += TA_FC) {
    __syncthreads();
    for (int i = threadIdx.x; i < T * 32 * (TA_FC / 4); i += nthreads) {
      int fq = i % (TA_FC / 4);
      int pl = (i / (TA_FC / 4)) % 32;
      int s = i / (32 * (TA_FC / 4));
      int pp = min(px0 + pl, HW - 1);
      KV::stage(kv, s, fq, pl, qkv + ((size_t)(b * T + s) * HW + pp) * tok_stride + 2 * C + h * F + f0 + fq * 4);
    }
#pragma unroll
    for (int u = 0; u < TPW; ++u)
      for (int i = lane; i < T * TA_FC; i += 32) {
        int s = i / TA_FC, f = i - s * TA_FC;
        ra[u * T * TA_FC + i] = __ldg(p.Rv + (((size_t)(b * T + tq[u]) * T + s) * C + h * F + f0 + f));
      }
    __syncthreads();
    float o[TPW][TA_FC];
#pragma unroll
    for (int u = 0; u < TPW; ++u)
#pragma unroll
      for (int f = 0; f < TA_FC; ++f) o[u][f] = 0.f;
#pragma unroll
    for (int s = 0; s < TP; ++s) {
      if (s < T) {
        float vv[TA_FC];
        KV::load(kv, s, lane, vv);
#pragma unroll
        for (int u = 0; u < TPW; ++u) {
          const float* rva = ra + (u * T + s) * TA_FC;
          const float4 r0 = *reinterpret_cast<const float4*>(rva), r1 = *reinterpret_cast<const float4*>(rva + 4);
          const float rvv[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
          const float pr = S[u][s];
#pragma unroll
          for (int f = 0; f < TA_FC; ++f) o[u][f] = fmaf(pr, vv[f] + rvv[f], o[u][f]);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < TPW; ++u) {
      if (act[u] && px_ok) {
        OT* orow = reinterpret_cast<OT*>(p.out) + ((size_t)(b * T + tq[u]) * HW + px) * C + h * F + f0;
        OpType<OT>::store4(orow, make_float4(o[u][0], o[u][1], o[u][2], o[u][3]));
        OpType<OT>::store4(orow + 4, make_float4(o[u][4], o[u][5], o[u][6], o[u][7]));
      }
    }
  }
}

template <int TP, int TPW, typename QT, typename OT>
static int launch_temporal_cfg(TAParams& p, cudaStream_t st) {
  const int slots = (p.T + TPW - 1) / TPW;            // warps needed for all query frames
  // query-frame groups: enough blocks to fill the GPU twice on small feature maps (each group re-stages K/V, which is cheap),
  // at most TA_MAX_WARPS warps per block, at least 2 warps per block
  const int base_blocks = ((p.HW + 31) / 32) * p.heads * p.B;
  int groups = (296 + base_blocks - 1) / base_blocks;
  const int min_groups = (slots + TA_MAX_WARPS - 1) / TA_MAX_WARPS, max_groups = (slots + 1) / 2;
  if (groups < min_groups) groups = min_groups;
  if (groups > max_groups) groups = max_groups;
  if (groups < 1) groups = 1;
  p.nw = (slots + groups - 1) / groups;
  p.tgroups = (slots + p.nw - 1) / p.nw;
  dim3 grid((p.HW + 31) / 32, p.heads, p.B * p.tgroups);
  const size_t smem = ((size_t)p.T * KvTile<QT>::WORDS_PER_S + (size_t)p.nw * 2 * TPW * p.T * TA_FC) * sizeof(float);
  if (smem > 48 * 1024)
    cudaFuncSetAttribute(attn_temporal_kernel<TP, TPW, QT, OT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  fdm::launch(attn_temporal_kernel<TP, TPW, QT, OT>, dim3(grid), dim3(p.nw * 32), smem, st, p);
  return check_launch();
}

template <typename QT, typename OT>
static int launch_temporal(TAParams& p, cudaStream_t st) {
  // one query frame per warp: two per warp halves the shared-memory reads per FMA but costs 161 registers (one block per
  // SM) and measured slower on B200 for T = 20 (567 vs 523 us per step)
  if (p.T <= 8) return launch_temporal_cfg<8, 1, QT, OT>(p, st);
  if (p.T <= 16) return launch_temporal_cfg<16, 1, QT, OT>(p, st);
  if (p.T <= 24) return launch_temporal_cfg<24, 1, QT, OT>(p, st);
  if (p.T <= 32) return launch_temporal_cfg<32, 1, QT, OT>(p, st);
  if (p.T <= 40) return launch_temporal_cfg<40, 1, QT, OT>(p, st);
  return FDM_ERR_UNSUPPORTED;
}

// =====================================================================================================
// spatial attention: grid (ceil(L/64), heads, N); block 256 = 64 queries x 4 lanes (each lane owns F/4 dims)
// =====================================================================================================
constexpr int SA_KC = 32;  // keys per shared-memory chunk
constexpr int SA_QB = 64;  // queries per block

struct SAParams {
  const void* qkv; void* out;
  int N, L, C, heads, F;
  float scale;
};

template <int FQ, typename QT, typename OT>
__global__ void __launch_bounds__(256) attn_spatial_kernel(SAParams p) {
  pdl_wait();
  constexpr int V = (FQ % 4 == 0) ? 4 : 2;   // vector width of shared-memory accesses (F = 24 -> FQ = 6 -> float2)
  constexpr int SUB = FQ + V;                // padded sub-vector stride: lane `sub` starts at sub*SUB
  constexpr int ROW = 4 * SUB;
  __shared__ __align__(16) float ks[SA_KC * ROW];
  __shared__ __align__(16) float vs[SA_KC * ROW];
  const int tid = threadIdx.x, sub = tid & 3, ql = tid >> 2;
  const int n = blockIdx.z, h = blockIdx.y, C = p.C, L = p.L;
  constexpr int F = FQ * 4;
  const int qi = blockIdx.x * SA_QB + ql;
  const bool q_ok = qi < L;
  const QT* base = reinterpret_cast<const QT*>(p.qkv) + (size_t)n * L * 3 * C + h * F;
  float q[FQ], o[FQ];
  {
    const QT* qp = base + (size_t)(q_ok ? qi : 0) * 3 * C + sub * FQ;
#pragma unroll
    for (int f = 0; f < FQ; ++f) {
      q[f] = OpType<QT>::load(qp + f) * p.scale;
      o[f] = 0.f;
    }
  }
  float mrun = -INFINITY, lrun = 0.f;
  for (int j0 = 0; j0 < L; j0 += SA_KC) {
    __syncthreads();
    for (int i = tid; i < SA_KC * (F / V); i += 256) {
      int j = i / (F / V), f = (i - j * (F / V)) * V;
      int jj = min(j0 + j, L - 1);
      const QT* kp = base + (size_t)jj * 3 * C + C + f;
      int off = j * ROW + (f / FQ) * SUB + (f % FQ);
      if constexpr (V == 4) {
        *reinterpret_cast<float4*>(&ks[off]) = OpType<QT>::load4(kp);
        *reinterpret_cast<float4*>(&vs[off]) = OpType<QT>::load4(kp + C);
      } else {
        *reinterpret_cast<float2*>(&ks[off]) = make_float2(OpType<QT>::load(kp), OpType<QT>::load(kp + 1));
        *reinterpret_cast<float2*>(&vs[off]) = make_float2(OpType<QT>::load(kp + C), OpType<QT>::load(kp + C + 1));
      }
    }
    __syncthreads();
    float s[SA_KC];
    float cmax = -INFINITY;
#pragma unroll
    for (int j = 0; j < SA_KC; ++j) {
      const float* kr = &ks[j * ROW + sub * SUB];
      float acc = 0.f;
      if constexpr (V == 4) {
#pragma unroll
        for (int f = 0; f < FQ; f += 4) {
          float4 kk = *reinterpret_cast<const float4*>(kr + f);
          acc = fmaf(q[f], kk.x, acc); acc = fmaf(q[f + 1], kk.y, acc);
          acc = fmaf(q[f + 2], kk.z, acc); acc = fmaf(q[f + 3], kk.w, acc);
        }
      } else {
#pragma unroll
        for (int f = 0; f < FQ; f += 2) {
          float2 kk = *reinterpret_cast<const float2*>(kr + f);
          acc = fmaf(q[f], kk.x, acc); acc = fmaf(q[f + 1], kk.y, acc);
        }
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      acc += __shfl_xor_sync(0xffffffffu, acc, 2);
      s[j] = (j0 + j < L) ? acc : -INFINITY;
      cmax = fmaxf(cmax, s[j]);
    }
    const float mnew = fmaxf(mrun, cmax);
    const float corr = expf(mrun - mnew);  // exp(-inf) = 0 on the first chunk
    lrun *= corr;
#pragma unroll
    for (int f = 0; f < FQ; ++f) o[f] *= corr;
#pragma unroll
    for (int j = 0; j < SA_KC; ++j) {
      const float pj = expf(s[j] - mnew);
      lrun += pj;
      const float* vr = &vs[j * ROW + sub * SUB];
      if constexpr (V == 4) {
#pragma unroll
        for (int f = 0; f < FQ; f += 4) {
          float4 vv = *reinterpret_cast<const float4*>(vr + f);
          o[f] = fmaf(pj, vv.x, o[f]); o[f + 1] = fmaf(pj, vv.y, o[f + 1]);
          o[f + 2] = fmaf(pj, vv.z, o[f + 2]); o[f + 3] = fmaf(pj, vv.w, o[f + 3]);
        }
      } else {
#pragma unroll
        for (int f = 0; f < FQ; f += 2) {
          float2 vv = *reinterpret_cast<const float2*>(vr + f);
          o[f] = fmaf(pj, vv.x, o[f]); o[f + 1] = fmaf(pj, vv.y, o[f + 1]);
        }
      }
    }
    mrun = mnew;
  }
  if (q_ok) {
    const float inv = 1.f / lrun;
    OT* op = reinterpret_cast<OT*>(p.out) + ((size_t)n * L + qi) * C + h * F + sub * FQ;
#pragma unroll
    for (int f = 0; f < FQ; ++f) OpType<OT>::store(op + f, o[f] * inv);
  }
}

template <typename QT, typename OT>
static int launch_spatial(const SAParams& p, cudaStream_t st) {
  dim3 grid((p.L + SA_QB - 1) / SA_QB, p.heads, p.N);
  switch (p.F) {
    case 8: fdm::launch(attn_spatial_kernel<2, QT, OT>, dim3(grid), dim3(256), 0, st, p); break;
    case 16: fdm::launch(attn_spatial_kernel<4, QT, OT>, dim3(grid), dim3(256), 0, st, p); break;
    case 24: fdm::launch(attn_spatial_kernel<6, QT, OT>, dim3(grid), dim3(256), 0, st, p); break;
    case 32: fdm::launch(attn_spatial_kernel<8, QT, OT>, dim3(grid), dim3(256), 0, st, p); break;
    case 48: fdm::launch(attn_spatial_kernel<12, QT, OT>, dim3(grid), dim3(256), 0, st, p); break;
    case 64: fdm::launch(attn_spatial_kernel<16, QT, OT>, dim3(grid), dim3(256), 0, st, p); break;
    case 96: fdm::launch(attn_spatial_kernel<24, QT, OT>, dim3(grid), dim3(256), 0, st, p); break;
    case 128: fdm::launch(attn_spatial_kernel<32, QT, OT>, dim3(grid), dim3(256), 0, st, p); break;
    default: return FDM_ERR_UNSUPPORTED;
  }
  return check_launch();
}

}  // namespace fdm

using namespace fdm;

namespace fdm {
int attn_temporal_tc_launch(const fdm_attn_temporal_args* a, cudaStream_t st);  // attn_temporal_tc.cu
size_t attn_temporal_tc_workspace(const fdm_attn_temporal_args* a);
int tt_row_stride(int T);
}

extern "C" size_t fdm_attn_temporal_workspace(const fdm_attn_temporal_args* a) { return a ? attn_temporal_tc_workspace(a) : 0; }

extern "C" size_t fdm_attn_temporal_attn_offset(const fdm_attn_temporal_args* a) {
  if (!a || attn_temporal_tc_workspace(a) == 0) return 0;
  const size_t rows = (size_t)a->B * a->heads * a->HW * a->T;
  return 2 * rows * (size_t)tt_row_stride(a->T) * sizeof(__nv_bfloat16);  // past the two bf16 score-term tables
}

extern "C" int fdm_attn_temporal(const fdm_attn_temporal_args* a, void* stream) {
  FDM_REQUIRE(a && a->qkv && a->out, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->B > 0 && a->T > 0 && a->HW > 0 && a->heads > 0 && a->C % a->heads == 0, FDM_ERR_BAD_ARG);
  if (a->Rq_op != nullptr && a->Rk_op != nullptr && a->Rv_op != nullptr && a->workspace != nullptr) {
    int rc = attn_temporal_tc_launch(a, (cudaStream_t)stream);
    if (rc != FDM_ERR_UNSUPPORTED) return rc;
  }
  FDM_REQUIRE(a->Rq && a->Rk && a->Rv, FDM_ERR_BAD_ARG);  // the CUDA-core kernel reads the fp32 tables
  FDM_REQUIRE(a->attn_mean == nullptr, FDM_ERR_UNSUPPORTED);
  const int F = a->C / a->heads;
  FDM_REQUIRE(F % TA_FC == 0 && a->T <= 40, FDM_ERR_UNSUPPORTED);
  TAParams p{a->qkv, a->Rq, a->Rk, a->Rv, a->mask, a->out, a->B, a->T, a->HW, a->C, a->heads, F, 1, 1, 1.0f / sqrtf((float)F)};
  cudaStream_t st = (cudaStream_t)stream;
  const bool qb = a->qkv_dtype == FDM_BF16, ob = a->out_dtype == FDM_BF16;
  if (!qb && !ob) return launch_temporal<float, float>(p, st);
  if (!qb && ob) return launch_temporal<float, __nv_bfloat16>(p, st);
  if (qb && !ob) return launch_temporal<__nv_bfloat16, float>(p, st);
  return launch_temporal<__nv_bfloat16, __nv_bfloat16>(p, st);
}

namespace fdm {
int attn_spatial_tc_launch(const fdm_attn_spatial_args* a, cudaStream_t st);  // attn_tc.cu
}

extern "C" int fdm_attn_spatial(const fdm_attn_spatial_args* a, void* stream) {
  FDM_REQUIRE(a && a->qkv && a->out, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->N > 0 && a->L > 0 && a->heads > 0 && a->C % a->heads == 0, FDM_ERR_BAD_ARG);
  if (a->engine == 0 && a->qkv_dtype == FDM_BF16 && a->out_dtype == FDM_BF16) {
    int rc = attn_spatial_tc_launch(a, (cudaStream_t)stream);
    if (rc != FDM_ERR_UNSUPPORTED) return rc;
  }
  FDM_REQUIRE(a->attn_mean == nullptr, FDM_ERR_UNSUPPORTED);  // attention-map logging is served by the tcgen05 kernels only
  const int F = a->C / a->heads;
  SAParams p{a->qkv, a->out, a->N, a->L, a->C, a->heads, F, 1.0f / sqrtf((float)F)};
  cudaStream_t st = (cudaStream_t)stream;
  const bool qb = a->qkv_dtype == FDM_BF16, ob = a->out_dtype == FDM_BF16;
  if (!qb && !ob) return launch_spatial<float, float>(p, st);
  if (!qb && ob) return launch_spatial<float, __nv_bfloat16>(p, st);
  if (qb && !ob) return launch_spatial<__nv_bfloat16, float>(p, st);
  return launch_spatial<__nv_bfloat16, __nv_bfloat16>(p, st);
}
