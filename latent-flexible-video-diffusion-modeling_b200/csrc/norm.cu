// GroupNorm(32) kernels: fused apply (+FiLM)(+SiLU) over a virtual channel concat, and the temporal
// GroupNorm of the attention block whose statistics span (C/32 channels x T frames) per (b, pixel).
// Reference: nn.py:12-19,95-102; unet.py:153-154,165-166,199-203,400-401,460; rpe.py:113,135-137.
// HBM-bound: 128-bit loads/stores, one read of x, one write per requested output.
#include "common.cuh"

namespace fdm {

struct GnParams {
  const void* xa; const float* xb; const double* sa; const double* sb;
  const float* gamma; const float* beta; const float* film;
  void* out_op; float* out_f32; void* raw_op;
  int N, HW, Ca, Cb, C, T, film_stride, film_off, silu, pix_per_block;
  float eps;
  double inv_cnt;  // 1 / (channels per group * HW)
  int film_add;  // 1: use_scale_shift_norm=False (unet.py:204-206): the embedding is ADDED before the norm, h = GN(x + e[n, c])
  DropArgs drop;  // read by the DROP instantiations only
};

__device__ __forceinline__ float4 gn_load4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 gn_load4(const __nv_bfloat16* p) {
  const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
  return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16), __uint_as_float(u.y & 0xffff0000u));
}

// grid: (ceil(HW / pix_per_block), N); block: (C/4) * ppi threads  (ppi pixels per iteration)
// IT = element type of source A (bf16: single-source launches only).  DROP: ResBlock dropout after the SiLU (p.drop).
template <typename OT, typename IT, bool DROP>
__global__ void gn_apply_kernel(GnParams p) {
  pdl_wait();
  __shared__ float s_mean[32], s_rstd[32];
  DropMask dm;
  if constexpr (DROP) dm = load_drop_mask(p.drop);
  const int n = blockIdx.y;
  const int C = p.C, cpg = C / 32;
  const int quads = C / 4;
  const int q = threadIdx.x % quads, pl = threadIdx.x / quads, ppi = blockDim.x / quads;
  const int c = q * 4;
  const bool from_a = c < p.Ca;  // Ca, Cb are multiples of 4: a quad never straddles the concat boundary
  const IT* src = from_a ? reinterpret_cast<const IT*>(p.xa) + (size_t)n * p.HW * p.Ca + c
                         : reinterpret_cast<const IT*>(p.xb) + (size_t)n * p.HW * p.Cb + (c - p.Ca);  // (xb only with IT = float)
  const int sstride = from_a ? p.Ca : p.Cb;
  const int p0 = blockIdx.x * p.pix_per_block;
  const int p1 = min(p0 + p.pix_per_block, p.HW);
  // the first trip's activation loads are in flight while the (latency-bound) statistics prologue runs
  float4 xs[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int pp = p0 + pl + u * ppi;
    if (pp < p1) xs[u] = gn_load4(src + (size_t)pp * sstride);
  }
  if (threadIdx.x < 32) {
    const int g = threadIdx.x;
    double s = 0.0, ss = 0.0;
    for (int j = 0; j < cpg; ++j) {
      int cc = g * cpg + j;
      const double* st = cc < p.Ca ? p.sa + ((size_t)n * p.Ca + cc) * 2 : p.sb + ((size_t)n * p.Cb + (cc - p.Ca)) * 2;
      double s1 = st[0], s2 = st[1];
      if (p.film_add) {
        // statistics of x + e from those of x (e is constant over the pixels of a channel): exact algebra on the fp64 sums
        const double e = (double)p.film[(size_t)(n / p.T) * p.film_stride + p.film_off + cc];
        s2 += 2.0 * e * s1 + (double)p.HW * e * e;
        s1 += (double)p.HW * e;
      }
      s += s1;
      ss += s2;
    }
    // E[x^2] - mean^2 needs the fp64 sums; the final rsqrt does not (bf16-only outputs: two fp64 multiplies and an rsqrtf instead of
    // two fp64 divisions and a square root on the critical path of every block — these launches are latency-bound on
    // the small maps).  Launches that keep an fp32 copy (fp32 parity mode) stay in fp64 throughout.
    if (sizeof(OT) == 2 && p.out_f32 == nullptr) {
      const double inv = p.inv_cnt;  // 1 / (cpg * HW), divided on the host
      const double mean = s * inv;
      const double var = fmax(ss * inv - mean * mean, 0.0);
      s_mean[g] = (float)mean;
      s_rstd[g] = rsqrtf((float)var + p.eps);
    } else {
      const double cnt = (double)cpg * (double)p.HW;
      const double mean = s / cnt;
      const double var = fmax(ss / cnt - mean * mean, 0.0);
      s_mean[g] = (float)mean;
      s_rstd[g] = (float)(1.0 / sqrt(var + (double)p.eps));
    }
  }
  __syncthreads();
  float mul[4], add[4];  // v = x*mul + add, folding mean/rstd/gamma/beta/FiLM
  {
    const int b = n / p.T;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int g = (c + j) / cpg;
      float ga = p.gamma[c + j] * s_rstd[g];
      float be = p.beta[c + j] - s_mean[g] * ga;
      if (p.film != nullptr && p.film_add) {
        be = fmaf(p.film[(size_t)b * p.film_stride + p.film_off + c + j], ga, be);  // (x + e) * ga + be
      } else if (p.film != nullptr) {
        const float* f = p.film + (size_t)b * p.film_stride + p.film_off;
        float sc = 1.f + f[c + j], sh = f[C + c + j];
        ga *= sc;
        be = be * sc + sh;
      }
      mul[j] = ga;
      add[j] = be;
    }
  }
  // 4 pixels per thread per trip, all loads issued before the first use (memory-level parallelism)
  for (int px = p0 + pl; px < p1; px += 4 * ppi) {
    if (px != p0 + pl) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int pp = px + u * ppi;
        if (pp < p1) xs[u] = gn_load4(src + (size_t)pp * sstride);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int pp = px + u * ppi;
      if (pp >= p1) break;
      const float4 x = xs[u];
      float v[4] = {x.x * mul[0] + add[0], x.y * mul[1] + add[1], x.z * mul[2] + add[2], x.w * mul[3] + add[3]};
      if (p.silu) {
        // bf16-only outputs: __expf-based SiLU (rel. error ~1e-6, far below the bf16 rounding of the store);
        // whenever an fp32 copy is written (fp32 parity mode) the precise expf version is used
        if (sizeof(OT) == 2 && p.out_f32 == nullptr) {
#pragma unroll
          for (int j = 0; j < 4; ++j) v[j] = silu_f(v[j]);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) v[j] = silu_precise(v[j]);
        }
      }
      size_t o = ((size_t)n * p.HW + pp) * C + c;
      if constexpr (DROP) dm.apply(o, v);
      float4 v4 = make_float4(v[0], v[1], v[2], v[3]);
      if (p.out_op != nullptr) OpType<OT>::store4(reinterpret_cast<OT*>(p.out_op) + o, v4);
      if (p.out_f32 != nullptr) *reinterpret_cast<float4*>(p.out_f32 + o) = v4;
      if (p.raw_op != nullptr) OpType<OT>::store4(reinterpret_cast<OT*>(p.raw_op) + o, x);
    }
  }
}

struct TgnParams {
  const float* x; const float* gamma; const float* beta; float* out_f32; void* out_op;
  int B, T, HW, C;
  float eps;
};

// Temporal GroupNorm.  A warp handles 8 groups of one (b, pixel): 4 lanes per group split the T frames (lane = 4*group + slice),
// so there are 4 * B * HW warps with T/4-long dependent chains instead of B * HW warps walking all T frames (the first
// version ran at 3.5 warps per SM on the wide models).
// Statistics in ONE pass around a pivot (the group's first value): var = E[(x-p)^2] - (E[x-p])^2 is well conditioned even
// for the tiny groups of this norm (as few as C/32 * T = 2 values), where E[x^2]-mean^2 cancels catastrophically.
// Second pass re-reads the (L1/L2-resident) values, normalises and writes.  V = vector width of the channel accesses.
template <typename OT, int V>
__global__ void __launch_bounds__(256) temporal_gn_kernel(TgnParams p) {
  pdl_wait();
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= p.B * p.HW * 4) return;
  const int gb = warp & 3, pix = warp >> 2;          // group block (8 groups) of pixel `pix`
  const int b = pix / p.HW, px = pix - b * p.HW;
  const int g = gb * 8 + (lane >> 2), ts = lane & 3;  // group, frame slice
  const int cpg = p.C / 32, c0 = g * cpg;
  const size_t fstride = (size_t)p.HW * p.C;
  const float* base = p.x + ((size_t)b * p.T * p.HW + px) * p.C + c0;
  const float pivot = __ldg(base);
  float s = 0.f, ss = 0.f;
#pragma unroll 2
  for (int t = ts; t < p.T; t += 4) {
    const float* r = base + t * fstride;
    for (int j = 0; j < cpg; j += V) {
      float v[V];
      if constexpr (V == 4) { float4 q = __ldg(reinterpret_cast<const float4*>(r + j)); v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w; }
      else if constexpr (V == 2) { float2 q = __ldg(reinterpret_cast<const float2*>(r + j)); v[0] = q.x; v[1] = q.y; }
      else v[0] = __ldg(r + j);
#pragma unroll
      for (int k = 0; k < V; ++k) {
        const float d = v[k] - pivot;
        s += d;
        ss = fmaf(d, d, ss);
      }
    }
  }
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  ss += __shfl_xor_sync(0xffffffffu, ss, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  ss += __shfl_xor_sync(0xffffffffu, ss, 2);
  const float cnt = (float)(cpg * p.T);
  const float md = s / cnt;
  const float mean = pivot + md;
  const float rstd = rsqrtf(fmaxf(ss / cnt - md * md, 0.f) + p.eps);
#pragma unroll 2
  for (int t = ts; t < p.T; t += 4) {
    const float* r = base + t * fstride;
    const size_t o = ((size_t)(b * p.T + t) * p.HW + px) * p.C + c0;
    for (int j = 0; j < cpg; j += V) {
      float v[V];
      if constexpr (V == 4) { float4 q = __ldg(reinterpret_cast<const float4*>(r + j)); v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w; }
      else if constexpr (V == 2) { float2 q = __ldg(reinterpret_cast<const float2*>(r + j)); v[0] = q.x; v[1] = q.y; }
      else v[0] = __ldg(r + j);
#pragma unroll
      for (int k = 0; k < V; ++k) v[k] = (v[k] - mean) * rstd * __ldg(p.gamma + c0 + j + k) + __ldg(p.beta + c0 + j + k);
      if constexpr (V == 4) {
        if (p.out_f32 != nullptr) *reinterpret_cast<float4*>(p.out_f32 + o + j) = make_float4(v[0], v[1], v[2], v[3]);
        if (p.out_op != nullptr) OpType<OT>::store4(reinterpret_cast<OT*>(p.out_op) + o + j, make_float4(v[0], v[1], v[2], v[3]));
      } else {
#pragma unroll
        for (int k = 0; k < V; ++k) {
          if (p.out_f32 != nullptr) p.out_f32[o + j + k] = v[k];
          if (p.out_op != nullptr) OpType<OT>::store(reinterpret_cast<OT*>(p.out_op) + o + j + k, v[k]);
        }
      }
    }
  }
}

}  // namespace fdm

extern "C" int fdm_gn_apply(const fdm_gn_apply_args* a, void* stream) {
  using namespace fdm;
  FDM_REQUIRE(a && a->xa && a->stats_a && a->gamma && a->beta, FDM_ERR_BAD_ARG);
  FDM_REQUIRE((a->xb == nullptr) == (a->stats_b == nullptr), FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->drop_p >= 0.f && a->drop_p <= 1.f, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->drop_philox == nullptr || a->silu == 1, FDM_ERR_BAD_ARG);
  GnParams p{};
  p.xa = a->xa; p.xb = a->xb; p.sa = reinterpret_cast<const double*>(a->stats_a); p.sb = reinterpret_cast<const double*>(a->stats_b); p.gamma = a->gamma; p.beta = a->beta;
  p.film = a->film; p.out_op = a->out_op; p.out_f32 = a->out_f32; p.raw_op = a->raw_op;
  p.N = a->N; p.HW = a->HW; p.Ca = a->Ca; p.Cb = a->xb ? a->Cb : 0; p.C = p.Ca + p.Cb; p.T = a->T > 0 ? a->T : 1;
  p.film_stride = a->film_stride; p.film_off = a->film_off; p.silu = a->silu; p.eps = a->eps;
  p.film_add = (a->film != nullptr && a->film_add) ? 1 : 0;
  p.inv_cnt = 1.0 / ((double)(p.C / 32) * (double)a->HW);
  FDM_REQUIRE(p.C % 32 == 0 && p.Ca % 4 == 0 && p.Cb % 4 == 0 && p.C <= 4096, FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(a->N > 0 && a->HW > 0, FDM_ERR_BAD_ARG);
  const int quads = p.C / 4;
  FDM_REQUIRE(quads <= 1024, FDM_ERR_UNSUPPORTED);
  int ppi = quads >= 256 ? 1 : 256 / quads;
  if (ppi > a->HW) ppi = a->HW;
  const int threads = quads * ppi;
  // aim for >= ~4 waves of 148 SMs when the tensor is large, but keep >= 4 iterations per block
  int ppb = ppi * 4;
  while ((long long)a->N * ((a->HW + ppb - 1) / ppb) > 148LL * 16 && ppb < a->HW) ppb *= 2;
  p.pix_per_block = ppb;
  dim3 grid((a->HW + ppb - 1) / ppb, a->N);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool drop = a->drop_philox != nullptr && a->drop_p > 0.f;
  if (drop) p.drop = drop_args(a->drop_philox, a->drop_p, a->drop_salt);
  if (a->xa_bf16) {
    FDM_REQUIRE(a->xb == nullptr && a->op_dtype == FDM_BF16, FDM_ERR_UNSUPPORTED);
    fdm::launch(drop ? gn_apply_kernel<__nv_bfloat16, __nv_bfloat16, true> : gn_apply_kernel<__nv_bfloat16, __nv_bfloat16, false>,
                dim3(grid), dim3(threads), 0, st, p);
  } else if (a->op_dtype == FDM_BF16) {
    fdm::launch(drop ? gn_apply_kernel<__nv_bfloat16, float, true> : gn_apply_kernel<__nv_bfloat16, float, false>, dim3(grid),
                dim3(threads), 0, st, p);
  } else {
    fdm::launch(drop ? gn_apply_kernel<float, float, true> : gn_apply_kernel<float, float, false>, dim3(grid), dim3(threads), 0, st, p);
  }
  return check_launch();
}

extern "C" int fdm_temporal_gn(const fdm_temporal_gn_args* a, void* stream) {
  using namespace fdm;
  FDM_REQUIRE(a && a->x && a->gamma && a->beta && (a->out_f32 || a->out_op), FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->C % 32 == 0 && a->B > 0 && a->T > 0 && a->HW > 0, FDM_ERR_UNSUPPORTED);
  TgnParams p{a->x, a->gamma, a->beta, a->out_f32, a->out_op, a->B, a->T, a->HW, a->C, a->eps};
  const long long warps = (long long)a->B * a->HW * 4;
  const int threads = 256;
  const int blocks = (int)((warps * 32 + threads - 1) / threads);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int cpg = a->C / 32;
#define FDM_TGN(OT)                                                                    \
  do {                                                                                 \
    if (cpg % 4 == 0) fdm::launch(temporal_gn_kernel<OT, 4>, dim3(blocks), dim3(threads), 0, st, p);         \
    else if (cpg % 2 == 0) fdm::launch(temporal_gn_kernel<OT, 2>, dim3(blocks), dim3(threads), 0, st, p);    \
    else fdm::launch(temporal_gn_kernel<OT, 1>, dim3(blocks), dim3(threads), 0, st, p);                      \
  } while (0)
  if (a->op_dtype == FDM_BF16) FDM_TGN(__nv_bfloat16);
  else FDM_TGN(float);
  return check_launch();
}
