// GroupNorm backward kernels (native_group_norm_backward + silu_backward + the FiLM chain of unet.py:199-203; rpe.py:135-137).
//   fdm_gn_bwd:           per-frame GroupNorm(32) (+FiLM)(+SiLU) over a virtual channel concat — three launches:
//                           stats  : per (n, c)  A = sum_hw du*xhat, B = sum_hw du   (block partials -> fp64 atomics)
//                           apply  : dx = rstd * (du*k_c - mean_g(k B) - xhat * mean_g(k A)),  gx (+)= dx (+ draw)
//                           params : dgamma, dbeta, dscale/dshift (FiLM) from A, B
//   fdm_temporal_gn_bwd:  statistics over (C/32 x T) per (b, pixel)
// HBM/L2-bound: each pass reads x (fp32) and the upstream gradient(s) once with 128-bit accesses.
#include "common.cuh"

namespace fdm {

// silu'(u) = s + u s (1 - s), s = sigmoid(u).  FAST: ex2.approx / rcp.approx (rel. error ~1e-6, far below the bf16 rounding of the
// gradients it multiplies; the kernel was 50 % issue-bound with the precise expf + division); the fp32 mode keeps the precise one.
template <bool FAST>
__device__ __forceinline__ float dsilu_f(float u) {
  const float s = FAST ? __fdividef(1.f, 1.f + __expf(-u)) : 1.f / (1.f + expf(-u));
  return s * (1.f + u * (1.f - s));
}

struct GnBwdParams {
  const float* xa; const float* xb; const double* sa; const double* sb;
  const float* gamma; const float* beta; const float* film;
  const void* dy_op; const float* dy_f32; const void* draw_op;
  float* gxa; float* gxb; double* ab; float* dgamma; float* dbeta; float* dfilm;
  const float* dpass_a; void* gop_a; float* cs_a; float* cs2_a;
  int N, HW, Ca, Cb, C, T, film_stride, film_off, silu, pix_per_block, acc_a, acc_b;
  float eps;
  DropArgs drop;  // read by the DROP instantiations only
};

// group statistics of frame n (threads < 32), as in gn_apply_kernel
__device__ __forceinline__ void gn_group_stats(const GnBwdParams& p, int n, int g, float& mean_o, float& rstd_o) {
  const int cpg = p.C / 32;
  double s = 0.0, ss = 0.0;
  for (int j = 0; j < cpg; ++j) {
    const int cc = g * cpg + j;
    const double* st = cc < p.Ca ? p.sa + ((size_t)n * p.Ca + cc) * 2 : p.sb + ((size_t)n * p.Cb + (cc - p.Ca)) * 2;
    s += st[0];
    ss += st[1];
  }
  const double cnt = (double)cpg * (double)p.HW;
  const double mean = s / cnt;
  const double var = fmax(ss / cnt - mean * mean, 0.0);
  mean_o = (float)mean;
  rstd_o = (float)(1.0 / sqrt(var + (double)p.eps));
}

// MODE 0: statistics pass; MODE 1: apply pass.  grid (ceil(HW / pix_per_block), N); block (C/4) * ppi threads.
// DROP: the forward's dropout mask (p.drop, regenerated) and scale are applied to the upstream gradient before silu'.
template <typename OT, int MODE, bool DROP>
__global__ void __launch_bounds__(256, 3) gn_bwd_kernel(GnBwdParams p) {
  pdl_wait();
  DropMask dm;
  if constexpr (DROP) dm = load_drop_mask(p.drop);
  __shared__ float s_mean[32], s_rstd[32], s_m1[32], s_m2[32];
  __shared__ float s_red[MODE == 0 ? 1024 * 8 : 1024];  // MODE 1: block partials of the fused bias-gradient column sums
  const int n = blockIdx.y, b = n / p.T;
  const int C = p.C, cpg = C / 32, quads = C / 4;
  const int q = threadIdx.x % quads, pl = threadIdx.x / quads, ppi = blockDim.x / quads;
  const int c = q * 4;
  const bool from_a = c < p.Ca;
  const float* src = from_a ? p.xa + (size_t)n * p.HW * p.Ca + c : p.xb + (size_t)n * p.HW * p.Cb + (c - p.Ca);
  const int sstride = from_a ? p.Ca : p.Cb;
  if (threadIdx.x < 32) {
    const int g = threadIdx.x;
    float mean, rstd;
    gn_group_stats(p, n, g, mean, rstd);
    s_mean[g] = mean;
    s_rstd[g] = rstd;
    if (MODE == 1) {
      double m1 = 0.0, m2 = 0.0;
      for (int j = 0; j < cpg; ++j) {
        const int cc = g * cpg + j;
        double k = p.gamma[cc];
        if (p.film != nullptr) k *= 1.0 + (double)p.film[(size_t)b * p.film_stride + p.film_off + cc];
        const double* ab = p.ab + ((size_t)n * C + cc) * 2;
        m2 += k * ab[0];
        m1 += k * ab[1];
      }
      const double cnt = (double)cpg * (double)p.HW;
      s_m1[g] = (float)(m1 / cnt);
      s_m2[g] = (float)(m2 / cnt);
    }
  }
  __syncthreads();
  float mul[4], add[4], kc[4], mean[4], rstd[4], m1[4], m2[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int g = (c + j) / cpg;
    mean[j] = s_mean[g];
    rstd[j] = s_rstd[g];
    float ga = p.gamma[c + j], be = p.beta[c + j], sc = 1.f, sh = 0.f;
    if (p.film != nullptr) {
      const float* f = p.film + (size_t)b * p.film_stride + p.film_off;
      sc = 1.f + f[c + j];
      sh = f[C + c + j];
    }
    kc[j] = ga * sc;
    mul[j] = ga * sc;             // u = xhat*mul + add
    add[j] = be * sc + sh;
    if (MODE == 1) { m1[j] = s_m1[g]; m2[j] = s_m2[g]; }
  }
  float accA[4] = {0.f, 0.f, 0.f, 0.f}, accB[4] = {0.f, 0.f, 0.f, 0.f};
  float accC[4] = {0.f, 0.f, 0.f, 0.f};  // MODE 1: column sums of the final gradient of xa
  const int p0 = blockIdx.x * p.pix_per_block;
  const int p1 = min(p0 + p.pix_per_block, p.HW);
  // GN_U pixels per trip (measured on B200: 2 and 4 are SLOWER than 1 — 111 / 137 registers cut the resident blocks per SM): every load of the trip (x, the upstream gradient(s), the pass-through gradient, the accumulated
  // destination) is issued before the first use — the kernel is HBM/L2-latency bound, not FMA bound
  constexpr int GN_U = 1;
  for (int px0_ = p0 + pl; px0_ < p1; px0_ += GN_U * ppi) {
    float4 x4[GN_U], d_op[GN_U], d_f32[GN_U], d_raw[GN_U], g_old[GN_U];
#pragma unroll
    for (int u = 0; u < GN_U; ++u) {
      const int px = px0_ + u * ppi;
      if (px >= p1) break;
      const size_t o = ((size_t)n * p.HW + px) * C + c;
      x4[u] = __ldg(reinterpret_cast<const float4*>(src + (size_t)px * sstride));
      if (p.dy_op != nullptr) d_op[u] = OpType<OT>::load4(reinterpret_cast<const OT*>(p.dy_op) + o);
      if (p.dy_f32 != nullptr) d_f32[u] = __ldg(reinterpret_cast<const float4*>(p.dy_f32 + o));
      if (MODE == 1) {
        if (p.draw_op != nullptr) d_raw[u] = OpType<OT>::load4(reinterpret_cast<const OT*>(p.draw_op) + o);
        const float* gsrc = from_a ? p.gxa + ((size_t)n * p.HW + px) * p.Ca + c : p.gxb + ((size_t)n * p.HW + px) * p.Cb + (c - p.Ca);
        if (from_a ? p.acc_a : p.acc_b) g_old[u] = *reinterpret_cast<const float4*>(gsrc);
      }
    }
#pragma unroll
    for (int u = 0; u < GN_U; ++u) {
      const int px = px0_ + u * ppi;
      if (px >= p1) break;
      float dy[4] = {0.f, 0.f, 0.f, 0.f};
      if (p.dy_op != nullptr) { dy[0] = d_op[u].x; dy[1] = d_op[u].y; dy[2] = d_op[u].z; dy[3] = d_op[u].w; }
      if (p.dy_f32 != nullptr) { dy[0] += d_f32[u].x; dy[1] += d_f32[u].y; dy[2] += d_f32[u].z; dy[3] += d_f32[u].w; }
      if constexpr (DROP) dm.apply(((size_t)n * p.HW + px) * C + c, dy);
      const float x[4] = {x4[u].x, x4[u].y, x4[u].z, x4[u].w};
      float dx[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float xh = (x[j] - mean[j]) * rstd[j];
        float du = dy[j];
        if (p.silu) du *= dsilu_f<sizeof(OT) == 2>(fmaf(xh, mul[j], add[j]));
        if (MODE == 0) {
          accA[j] = fmaf(du, xh, accA[j]);
          accB[j] += du;
        } else {
          dx[j] = rstd[j] * (du * kc[j] - m1[j] - xh * m2[j]);
        }
      }
      if (MODE == 1) {
        if (p.draw_op != nullptr) { dx[0] += d_raw[u].x; dx[1] += d_raw[u].y; dx[2] += d_raw[u].z; dx[3] += d_raw[u].w; }
        if (from_a && p.dpass_a != nullptr) {
          const float4 d = __ldg(reinterpret_cast<const float4*>(p.dpass_a + ((size_t)n * p.HW + px) * p.Ca + c));
          dx[0] += d.x; dx[1] += d.y; dx[2] += d.z; dx[3] += d.w;
        }
        float* gdst = from_a ? p.gxa + ((size_t)n * p.HW + px) * p.Ca + c : p.gxb + ((size_t)n * p.HW + px) * p.Cb + (c - p.Ca);
        float4 v = make_float4(dx[0], dx[1], dx[2], dx[3]);
        if (from_a ? p.acc_a : p.acc_b) v = make_float4(v.x + g_old[u].x, v.y + g_old[u].y, v.z + g_old[u].z, v.w + g_old[u].w);
        *reinterpret_cast<float4*>(gdst) = v;
        if (from_a && p.gop_a != nullptr) {
          // this launch is the LAST contributor to xa's gradient: emit the operand copy its producer's dgrad / wgrad will read,
          // and the bias gradient (column sums) of that producer — no separate cast pass over the tensor
          OpType<OT>::store4(reinterpret_cast<OT*>(p.gop_a) + ((size_t)n * p.HW + px) * p.Ca + c, v);
          accC[0] += v.x; accC[1] += v.y; accC[2] += v.z; accC[3] += v.w;
        }
      }
    }
  }
  if (MODE == 1 && p.cs_a != nullptr) {
    float* r = s_red + (size_t)threadIdx.x * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) r[j] = accC[j];
    __syncthreads();
    if (pl == 0 && from_a) {
      for (int k = 1; k < ppi; ++k) {
        const float* o = s_red + (size_t)(k * quads + q) * 4;
#pragma unroll
        for (int j = 0; j < 4; ++j) accC[j] += o[j];
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        atomicAdd(p.cs_a + c + j, accC[j]);
        if (p.cs2_a != nullptr) atomicAdd(p.cs2_a + c + j, accC[j]);
      }
    }
  }
  if (MODE == 0) {
    float* r = s_red + (size_t)threadIdx.x * 8;
#pragma unroll
    for (int j = 0; j < 4; ++j) { r[j] = accA[j]; r[4 + j] = accB[j]; }
    __syncthreads();
    if (pl == 0) {
      for (int k = 1; k < ppi; ++k) {
        const float* o = s_red + (size_t)(k * quads + q) * 8;
#pragma unroll
        for (int j = 0; j < 4; ++j) { accA[j] += o[j]; accB[j] += o[4 + j]; }
      }
      double* ab = p.ab + ((size_t)n * C + c) * 2;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        atomicAdd(ab + 2 * j, (double)accA[j]);
        atomicAdd(ab + 2 * j + 1, (double)accB[j]);
      }
    }
  }
}

// parameter gradients from the per-(n, c) sums.  block (32 channels, 8 frame slices): the frames of a video are split over
// threadIdx.y and combined in shared memory (one thread per channel walking all N frames took 45 us per launch at N = 160).
__global__ void __launch_bounds__(256) gn_bwd_params_kernel(GnBwdParams p) {
  pdl_wait();
  __shared__ double redA[8][33], redB[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x, sl = threadIdx.y;
  const bool ok = c < p.C;
  const float ga = ok ? p.gamma[c] : 0.f, be = ok ? p.beta[c] : 0.f;
  const int B = p.N / p.T;
  double dg = 0.0, db = 0.0;
  for (int b = 0; b < B; ++b) {
    double sA = 0.0, sB = 0.0;
    if (ok)
      for (int t = sl; t < p.T; t += 8) {
        const double* ab = p.ab + ((size_t)(b * p.T + t) * p.C + c) * 2;
        sA += ab[0];
        sB += ab[1];
      }
    redA[sl][threadIdx.x] = sA;
    redB[sl][threadIdx.x] = sB;
    __syncthreads();
    if (sl == 0 && ok) {
      for (int k = 1; k < 8; ++k) {
        sA += redA[k][threadIdx.x];
        sB += redB[k][threadIdx.x];
      }
      double sc = 1.0;
      if (p.film != nullptr) {
        sc = 1.0 + (double)p.film[(size_t)b * p.film_stride + p.film_off + c];
        if (p.dfilm != nullptr) {
          p.dfilm[(size_t)b * p.film_stride + p.film_off + c] = (float)((double)ga * sA + (double)be * sB);
          p.dfilm[(size_t)b * p.film_stride + p.film_off + p.C + c] = (float)sB;
        }
      }
      dg += sc * sA;
      db += sc * sB;
    }
    __syncthreads();
  }
  if (sl == 0 && ok) {
    p.dgamma[c] = (float)dg;
    p.dbeta[c] = (float)db;
  }
}

// ---------------- temporal GroupNorm backward -----------------------------------------------------------------------
struct TgnBwdParams {
  const float* x; const float* gamma; const void* dy_op; const float* dy_f32;
  float* gx; float* dgamma; float* dbeta;
  int B, T, HW, C, accumulate;
  float eps;
};

constexpr int TGN_MAX_CPG = 16;

// warp <-> (b, pixel) (grid-stride), lane <-> group.  Three passes over the group's T * C/32 values (L1/L2 resident).
template <typename OT>
__global__ void __launch_bounds__(256) temporal_gn_bwd_kernel(TgnBwdParams p) {
  pdl_wait();
  extern __shared__ float tg_red[];  // [8 warps][2][C]
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int cpg = p.C / 32, c0 = lane * cpg;
  const size_t fstride = (size_t)p.HW * p.C;
  float ga[TGN_MAX_CPG], dg[TGN_MAX_CPG], db[TGN_MAX_CPG];
#pragma unroll
  for (int j = 0; j < TGN_MAX_CPG; ++j) {
    ga[j] = j < cpg ? p.gamma[c0 + j] : 0.f;
    dg[j] = 0.f;
    db[j] = 0.f;
  }
  const float cnt = (float)(cpg * p.T);
  const long long npix = (long long)p.B * p.HW;
  for (long long pix = (long long)blockIdx.x * 8 + w; pix < npix; pix += (long long)gridDim.x * 8) {
    const int b = (int)(pix / p.HW), px = (int)(pix - (long long)b * p.HW);
    const size_t base = ((size_t)b * p.T * p.HW + px) * p.C + c0;
    const float pivot = __ldg(p.x + base);
    float s = 0.f, ss = 0.f;
    for (int t = 0; t < p.T; ++t) {
      const float* r = p.x + base + t * fstride;
#pragma unroll
      for (int j = 0; j < TGN_MAX_CPG; ++j)
        if (j < cpg) {
          const float d = __ldg(r + j) - pivot;
          s += d;
          ss = fmaf(d, d, ss);
        }
    }
    const float md = s / cnt;
    const float mean = pivot + md;
    const float rstd = rsqrtf(fmaxf(ss / cnt - md * md, 0.f) + p.eps);
    float s1 = 0.f, s2 = 0.f;
    for (int t = 0; t < p.T; ++t) {
      const size_t o = base + t * fstride;
#pragma unroll
      for (int j = 0; j < TGN_MAX_CPG; ++j)
        if (j < cpg) {
          float dy = 0.f;
          if (p.dy_op != nullptr) dy = OpType<OT>::load(reinterpret_cast<const OT*>(p.dy_op) + o + j);
          if (p.dy_f32 != nullptr) dy += __ldg(p.dy_f32 + o + j);
          const float xh = (__ldg(p.x + o + j) - mean) * rstd;
          const float dxh = dy * ga[j];
          s1 += dxh;
          s2 = fmaf(dxh, xh, s2);
          dg[j] = fmaf(dy, xh, dg[j]);
          db[j] += dy;
        }
    }
    s1 /= cnt;
    s2 /= cnt;
    for (int t = 0; t < p.T; ++t) {
      const size_t o = base + t * fstride;
#pragma unroll
      for (int j = 0; j < TGN_MAX_CPG; ++j)
        if (j < cpg) {
          float dy = 0.f;
          if (p.dy_op != nullptr) dy = OpType<OT>::load(reinterpret_cast<const OT*>(p.dy_op) + o + j);
          if (p.dy_f32 != nullptr) dy += __ldg(p.dy_f32 + o + j);
          const float xh = (__ldg(p.x + o + j) - mean) * rstd;
          float dx = rstd * (dy * ga[j] - s1 - xh * s2);
          if (p.accumulate) dx += p.gx[o + j];
          p.gx[o + j] = dx;
        }
    }
  }
  // block reduction of the parameter gradients, then one atomic per channel per block
#pragma unroll
  for (int j = 0; j < TGN_MAX_CPG; ++j)
    if (j < cpg) {
      tg_red[(size_t)(w * 2) * p.C + c0 + j] = dg[j];
      tg_red[(size_t)(w * 2 + 1) * p.C + c0 + j] = db[j];
    }
  __syncthreads();
  for (int c = threadIdx.x; c < p.C; c += blockDim.x) {
    float a = 0.f, bsum = 0.f;
    for (int k = 0; k < 8; ++k) {
      a += tg_red[(size_t)(k * 2) * p.C + c];
      bsum += tg_red[(size_t)(k * 2 + 1) * p.C + c];
    }
    atomicAdd(p.dgamma + c, a);
    atomicAdd(p.dbeta + c, bsum);
  }
}

}  // namespace fdm

using namespace fdm;

extern "C" int fdm_gn_bwd(const fdm_gn_bwd_args* a, void* stream) {
  FDM_REQUIRE(a && a->xa && a->stats_a && a->gamma && a->beta && a->gxa && a->ab && a->dgamma && a->dbeta, FDM_ERR_BAD_ARG);
  FDM_REQUIRE((a->xb == nullptr) == (a->stats_b == nullptr), FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->xb == nullptr || a->gxb != nullptr, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->dy_op != nullptr || a->dy_f32 != nullptr, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->drop_p >= 0.f && a->drop_p <= 1.f, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->drop_philox == nullptr || a->silu == 1, FDM_ERR_BAD_ARG);
  GnBwdParams p{};
  p.xa = a->xa; p.xb = a->xb; p.sa = a->stats_a; p.sb = a->stats_b; p.gamma = a->gamma; p.beta = a->beta; p.film = a->film;
  p.dy_op = a->dy_op; p.dy_f32 = a->dy_f32; p.draw_op = a->draw_op; p.gxa = a->gxa; p.gxb = a->gxb; p.ab = a->ab;
  p.dgamma = a->dgamma; p.dbeta = a->dbeta; p.dfilm = a->dfilm;
  p.dpass_a = a->dpass_a;
  p.gop_a = a->gop_a; p.cs_a = a->gop_a ? a->cs_a : nullptr; p.cs2_a = a->gop_a ? a->cs2_a : nullptr;
  p.N = a->N; p.HW = a->HW; p.Ca = a->Ca; p.Cb = a->xb ? a->Cb : 0; p.C = p.Ca + p.Cb; p.T = a->T > 0 ? a->T : 1;
  p.film_stride = a->film_stride; p.film_off = a->film_off; p.silu = a->silu; p.acc_a = a->acc_a; p.acc_b = a->acc_b; p.eps = a->eps;
  FDM_REQUIRE(p.C % 32 == 0 && p.Ca % 4 == 0 && p.Cb % 4 == 0 && p.C <= 4096, FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(a->N > 0 && a->HW > 0 && a->N % p.T == 0, FDM_ERR_BAD_ARG);
  const int quads = p.C / 4;
  FDM_REQUIRE(quads <= 256, FDM_ERR_UNSUPPORTED);  // one thread per channel quad, <= 256 threads (register budget of the apply pass)
  int ppi = quads >= 256 ? 1 : 256 / quads;
  if (ppi > a->HW) ppi = a->HW;
  const int threads = quads * ppi;
  int ppb = ppi * 4;
  while ((long long)a->N * ((a->HW + ppb - 1) / ppb) > 148LL * 16 && ppb < a->HW) ppb *= 2;
  p.pix_per_block = ppb;
  dim3 grid((a->HW + ppb - 1) / ppb, a->N);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int ph = a->phases == 0 ? 7 : a->phases;
  // the sums pass and the apply pass both read du; the parameter-gradient pass reads only the (masked) sums
  const bool drop = a->drop_philox != nullptr && a->drop_p > 0.f;
  if (drop) p.drop = drop_args(a->drop_philox, a->drop_p, a->drop_salt);
  const bool bf = a->op_dtype == FDM_BF16;
  if (ph & 1) {
    fdm::launch(bf ? (drop ? gn_bwd_kernel<__nv_bfloat16, 0, true> : gn_bwd_kernel<__nv_bfloat16, 0, false>)
                   : (drop ? gn_bwd_kernel<float, 0, true> : gn_bwd_kernel<float, 0, false>), grid, dim3(threads), 0, st, p);
  }
  if (ph & 2) fdm::launch(gn_bwd_params_kernel, dim3((p.C + 31) / 32), dim3(32, 8), 0, st, p);
  if (ph & 4) {
    fdm::launch(bf ? (drop ? gn_bwd_kernel<__nv_bfloat16, 1, true> : gn_bwd_kernel<__nv_bfloat16, 1, false>)
                   : (drop ? gn_bwd_kernel<float, 1, true> : gn_bwd_kernel<float, 1, false>), grid, dim3(threads), 0, st, p);
  }
  return check_launch();
}

extern "C" int fdm_temporal_gn_bwd(const fdm_temporal_gn_bwd_args* a, void* stream) {
  FDM_REQUIRE(a && a->x && a->gamma && a->gx && a->dgamma && a->dbeta && (a->dy_op || a->dy_f32), FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->C % 32 == 0 && a->C / 32 <= TGN_MAX_CPG && a->B > 0 && a->T > 0 && a->HW > 0, FDM_ERR_UNSUPPORTED);
  TgnBwdParams p{a->x, a->gamma, a->dy_op, a->dy_f32, a->gx, a->dgamma, a->dbeta, a->B, a->T, a->HW, a->C, a->accumulate, a->eps};
  const long long npix = (long long)a->B * a->HW;
  long long blocks = (npix + 7) / 8;
  if (blocks > 148 * 4) blocks = 148 * 4;
  const size_t smem = (size_t)8 * 2 * a->C * sizeof(float);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (a->op_dtype == FDM_BF16) fdm::launch(temporal_gn_bwd_kernel<__nv_bfloat16>, dim3((unsigned)blocks), dim3(256), smem, st, p);
  else fdm::launch(temporal_gn_bwd_kernel<float>, dim3((unsigned)blocks), dim3(256), smem, st, p);
  return check_launch();
}
