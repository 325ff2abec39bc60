// Backward-pass plumbing kernels: weight (re)packing in one launch, gradient accumulation / 2x2 pooling, layout change of
// the eps gradient, fixed-order partial sums, and the backward of the per-step conditioning path (grouped small linears,
// RPENet hidden layer).  Reference: what torch.autograd runs for nn.Linear (unet.py:304-308,159; rpe.py:12-14), rpe.py:21-30,
// F.interpolate backward (unet.py:85).  All HBM/latency-bound; none is on the FLOP path.
#include "common.cuh"

namespace fdm {

static inline int grid_for_b(long long total, int threads) {
  long long g = (total + threads - 1) / threads;
  long long cap = 148LL * 16;
  return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

// silu'(u) = s + u*s*(1-s), s = sigmoid(u)
__device__ __forceinline__ float dsilu(float u) {
  const float s = 1.f / (1.f + expf(-u));
  return s * (1.f + u * (1.f - s));
}

// ---------------- B0 weight packing ---------------------------------------------------------------------------------
__global__ void pack_weights_kernel(const fdm_pack_problem* __restrict__ probs) {
  pdl_wait();
  const fdm_pack_problem pr = probs[blockIdx.y];
  const int k = pr.k, kk = k * k;
  const long long total = pr.mode == FDM_PACK_SUM2 ? pr.co : (long long)pr.co * pr.ci * kk;
  const int cip64 = (pr.ci + 63) / 64 * 64, cop16 = (pr.co + 15) / 16 * 16;
  const int cop64 = (pr.co + 63) / 64 * 64, cip16 = (pr.ci + 15) / 16 * 16;
  if (pr.mode == FDM_PACK_TC_FWD || pr.mode == FDM_PACK_TC_DGRAD) {
    // tensor-core layouts: a (32 co x 32 ci x taps) tile goes through shared memory so that BOTH the fp32 reads (rows of
    // ci*taps contiguous floats) and the bf16 writes (64-byte runs along ci resp. co) are coalesced.  Writing 2-byte elements
    // straight from the source order cost 1.0 ms per step on the 80 M-parameter model (16x write amplification).
    __shared__ float tile[32][32 * 9 + 1];
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(pr.dst);
    const int tiles_ci = (pr.ci + 31) / 32, ntiles = tiles_ci * ((pr.co + 31) / 32);
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
      const int co0 = (t / tiles_ci) * 32, ci0 = (t % tiles_ci) * 32;
      const int nci = min(32, pr.ci - ci0), nco = min(32, pr.co - co0), nrow = nci * kk;
      for (int i = threadIdx.x; i < nco * nrow; i += blockDim.x) {
        const int r = i / nrow, c = i - r * nrow;
        tile[r][c] = pr.src[((size_t)(co0 + r) * pr.ci + ci0) * kk + c];
      }
      __syncthreads();
      for (int tap = 0; tap < kk; ++tap) {
        const int kh = tap / k, kw = tap - kh * k;
        for (int i = threadIdx.x; i < 32 * 32; i += blockDim.x) {
          const int r = i >> 5, c = i & 31;
          if (pr.mode == FDM_PACK_TC_FWD) {
            if (r < nco && c < nci)
              dst[((size_t)(kw * k + kh) * cop16 + co0 + r) * cip64 + ci0 + c] = __float2bfloat16_rn(tile[r][c * kk + tap]);
          } else {
            if (r < nci && c < nco)
              dst[((size_t)((k - 1 - kw) * k + (k - 1 - kh)) * cip16 + ci0 + r) * cop64 + co0 + c] = __float2bfloat16_rn(tile[c][r * kk + tap]);
          }
        }
      }
      __syncthreads();
    }
    return;
  }
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    if (pr.mode == FDM_PACK_SUM2) {
      reinterpret_cast<float*>(pr.dst)[i] = pr.src[i] + pr.src2[i];
      continue;
    }
    // i indexes the SOURCE [co][ci][kh][kw] (coalesced reads; the packed tensors are small and L2-resident)
    const int kw = (int)(i % k);
    long long r = i / k;
    const int kh = (int)(r % k);
    r /= k;
    const int ci = (int)(r % pr.ci), co = (int)(r / pr.ci);
    const float v = pr.src[i];
    switch (pr.mode) {
      case FDM_PACK_TC_FWD:
        reinterpret_cast<__nv_bfloat16*>(pr.dst)[((size_t)(kw * k + kh) * cop16 + co) * cip64 + ci] = __float2bfloat16_rn(v);
        break;
      case FDM_PACK_TC_DGRAD: {
        const int rr = k - 1 - kh, ss = k - 1 - kw;
        reinterpret_cast<__nv_bfloat16*>(pr.dst)[((size_t)(ss * k + rr) * cip16 + ci) * cop64 + co] = __float2bfloat16_rn(v);
        break;
      }
      case FDM_PACK_SIMT_FWD:
        reinterpret_cast<float*>(pr.dst)[((size_t)(kh * k + kw) * pr.ci + ci) * pr.co + co] = v;
        break;
      default: {  // FDM_PACK_SIMT_DGRAD
        const int rr = k - 1 - kh, ss = k - 1 - kw;
        reinterpret_cast<float*>(pr.dst)[((size_t)(rr * k + ss) * pr.co + co) * pr.ci + ci] = v;
      }
    }
  }
}

// ---------------- B6 accumulate / 2x2 sum-pool ----------------------------------------------------------------------
template <typename ST>
__global__ void accum_kernel(const ST* __restrict__ src, float* __restrict__ dst, int N, int H, int W, int C, int pool, int acc) {
  pdl_wait();
  const int quads = C / 4;
  const long long total = (long long)N * H * W * quads;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int q = (int)(i % quads);
    const long long pix = i / quads;
    float4 v;
    if (pool) {
      const int w = (int)(pix % W);
      const long long r = pix / W;
      const int h = (int)(r % H), n = (int)(r / H);
      const ST* s0 = src + ((((size_t)n * 2 * H + 2 * h) * 2 * W) + 2 * w) * C + q * 4;
      const float4 a = OpType<ST>::load4(s0), b = OpType<ST>::load4(s0 + C);
      const float4 c = OpType<ST>::load4(s0 + (size_t)2 * W * C), d = OpType<ST>::load4(s0 + (size_t)2 * W * C + C);
      v = make_float4(a.x + b.x + c.x + d.x, a.y + b.y + c.y + d.y, a.z + b.z + c.z + d.z, a.w + b.w + c.w + d.w);
    } else {
      v = OpType<ST>::load4(src + (size_t)pix * C + q * 4);
    }
    float4* o = reinterpret_cast<float4*>(dst + (size_t)pix * C + q * 4);
    if (acc) {
      const float4 e = *o;
      v = make_float4(v.x + e.x, v.y + e.y, v.z + e.z, v.w + e.w);
    }
    *o = v;
  }
}

template <typename OT>
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ src, OT* __restrict__ dst, int N, int C, int HW, int Cpad) {
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)N * HW) return;
  const int n = (int)(i / HW), px = (int)(i - (long long)n * HW);
  const float* s = src + (size_t)n * C * HW + px;
  OT* o = dst + (size_t)i * Cpad;
  for (int c = 0; c < Cpad; ++c) OpType<OT>::store(o + c, c < C ? s[(size_t)c * HW] : 0.f);
}

__global__ void sum_parts_kernel(const float* __restrict__ parts, float* __restrict__ out, long long stride, long long n,
                                 int count, int acc) {
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float s = acc ? out[i] : 0.f;
    for (int p = 0; p < count; ++p) s += parts[(size_t)p * stride + i];
    out[i] = s;
  }
}

// ---------------- grouped small linear backward ---------------------------------------------------------------------
// y = act(x) W^T + b with M = a handful of rows.  (1) dW[n][k] = sum_m dy[m][n] act(x[m][k]), db[n] = sum_m dy[m][n]: one thread
// per k (coalesced dW rows), blockIdx.y walks n.  (2) dx_part[m][k] = silu'(x) * sum_n dy[m][n] W[n][k]: one thread per k, the
// n loop streams W rows coalesced; 8 rows of M per pass.
__global__ void __launch_bounds__(128) linear_bwd_w_kernel(const fdm_linear_bwd_problem* __restrict__ probs) {
  pdl_wait();
  const fdm_linear_bwd_problem pr = probs[blockIdx.z];
  const int k = blockIdx.x * 128 + threadIdx.x;
  if (blockIdx.x * 128 >= pr.K) return;
  for (int n = blockIdx.y; n < pr.Nout; n += gridDim.y) {
    float acc = 0.f, bsum = 0.f;
    for (int m = 0; m < pr.M; ++m) {
      const float g = __ldg(pr.dy + (size_t)m * pr.ldy + n);
      bsum += g;
      if (k < pr.K) {
        float xv = __ldg(pr.x + (size_t)m * pr.ldx + k);
        if (pr.silu_in) xv = silu_precise(xv);
        acc = fmaf(g, xv, acc);
      }
    }
    if (k < pr.K) pr.dw[(size_t)n * pr.K + k] = acc;
    if (pr.db != nullptr && blockIdx.x == 0 && threadIdx.x == 0) pr.db[n] = bsum;
  }
}

__global__ void __launch_bounds__(128) linear_bwd_x_kernel(const fdm_linear_bwd_problem* __restrict__ probs) {
  pdl_wait();
  const fdm_linear_bwd_problem pr = probs[blockIdx.y];
  if (pr.dx_part == nullptr) return;
  const int k = blockIdx.x * 128 + threadIdx.x;
  if (k >= pr.K) return;
  for (int m0 = 0; m0 < pr.M; m0 += 8) {
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    int n = 0;
    for (; n + 7 < pr.Nout; n += 8) {  // eight weight rows in flight (a serial chain of Nout DRAM latencies otherwise)
      float w[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) w[u] = __ldg(pr.w + (size_t)(n + u) * pr.K + k);
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (m0 + j < pr.M) acc[j] = fmaf(__ldg(pr.dy + (size_t)(m0 + j) * pr.ldy + n + u), w[u], acc[j]);
    }
    for (; n < pr.Nout; ++n) {
      const float w = __ldg(pr.w + (size_t)n * pr.K + k);
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (m0 + j < pr.M) acc[j] = fmaf(__ldg(pr.dy + (size_t)(m0 + j) * pr.ldy + n), w, acc[j]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (m0 + j < pr.M) {
        float v = acc[j];
        if (pr.silu_in) v *= dsilu(__ldg(pr.x + (size_t)(m0 + j) * pr.ldx + k));
        pr.dx_part[(size_t)(m0 + j) * pr.K + k] = v;
      }
  }
}

// ---------------- RPENet hidden backward ----------------------------------------------------------------------------
// e = te[b][te_off+c] + wd[c]·phi(fi[b,t]-fi[b,s]) + bd[c];  hidden = silu(e).  grid (ceil(C/32), B, nets), block (32, 8):
// threadIdx.x <-> channel (coalesced), threadIdx.y splits the T*T pairs.
template <typename DT>
__global__ void __launch_bounds__(256) rpe_hidden_bwd_kernel(const float* __restrict__ te, const int64_t* __restrict__ fi,
                                                             const fdm_rpe_hidden_bwd_problem* __restrict__ probs,
                                                             float* __restrict__ dte, int T, int te_stride) {
  pdl_wait();
  const fdm_rpe_hidden_bwd_problem pr = probs[blockIdx.z];
  const int c = blockIdx.x * 32 + threadIdx.x, b = blockIdx.y;
  __shared__ float red[8][5][33];
  float s_te = 0.f, s_w0 = 0.f, s_w1 = 0.f, s_w2 = 0.f;
  if (c < pr.C) {
    const float w0 = pr.wd[c * 3], w1 = pr.wd[c * 3 + 1], w2 = pr.wd[c * 3 + 2];
    const float base = pr.bd[c] + te[(size_t)b * te_stride + pr.te_off + c];
    const DT* dh = reinterpret_cast<const DT*>(pr.dhidden) + (size_t)b * T * T * pr.C + c;
    for (int ts = threadIdx.y; ts < T * T; ts += 8) {
      const int t = ts / T, s = ts - t * T;
      const float d = (float)(fi[(size_t)b * T + t] - fi[(size_t)b * T + s]);
      const float f0 = logf(1.f + fmaxf(d, 0.f)), f1 = logf(1.f + fmaxf(-d, 0.f)), f2 = d == 0.f ? 1.f : 0.f;
      const float e = fmaf(f2, w2, fmaf(f1, w1, f0 * w0)) + base;
      const float g = OpType<DT>::load(dh + (size_t)ts * pr.C) * dsilu(e);
      s_te += g;
      s_w0 = fmaf(g, f0, s_w0);
      s_w1 = fmaf(g, f1, s_w1);
      s_w2 = fmaf(g, f2, s_w2);
    }
  }
  red[threadIdx.y][0][threadIdx.x] = s_te;
  red[threadIdx.y][1][threadIdx.x] = s_w0;
  red[threadIdx.y][2][threadIdx.x] = s_w1;
  red[threadIdx.y][3][threadIdx.x] = s_w2;
  __syncthreads();
  if (threadIdx.y == 0 && c < pr.C) {
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    for (int y = 0; y < 8; ++y)
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] += red[y][j][threadIdx.x];
    dte[(size_t)b * te_stride + pr.te_off + c] = v[0];
    atomicAdd(pr.dbd + c, v[0]);
    atomicAdd(pr.dwd + c * 3, v[1]);
    atomicAdd(pr.dwd + c * 3 + 1, v[2]);
    atomicAdd(pr.dwd + c * 3 + 2, v[3]);
  }
}


// ---------------- B7 fused AdamW (+EMA) over flat buffers -----------------------------------------------------------
__global__ void __launch_bounds__(256) adamw_flat_kernel(fdm_adamw_args a) {
  pdl_wait();
  const long long n4 = a.n >> 2;
  const float decay = 1.f - a.lr * a.weight_decay, step = a.lr / a.bias_correction1;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 p4 = reinterpret_cast<float4*>(a.p)[i];
    const float4 g4 = reinterpret_cast<const float4*>(a.g)[i];
    float4 m4 = reinterpret_cast<float4*>(a.m)[i], v4 = reinterpret_cast<float4*>(a.v)[i];
    float p[4] = {p4.x, p4.y, p4.z, p4.w}, m[4] = {m4.x, m4.y, m4.z, m4.w}, v[4] = {v4.x, v4.y, v4.z, v4.w};
    const float g[4] = {g4.x, g4.y, g4.z, g4.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      p[j] *= decay;
      m[j] = m[j] + (g[j] - m[j]) * (1.f - a.beta1);       // lerp, as torch's fused kernel
      v[j] = a.beta2 * v[j] + (1.f - a.beta2) * g[j] * g[j];
      const float denom = sqrtf(v[j]) / a.bias_correction2_sqrt + a.eps;
      p[j] -= step * (m[j] / denom);
    }
    reinterpret_cast<float4*>(a.p)[i] = make_float4(p[0], p[1], p[2], p[3]);
    reinterpret_cast<float4*>(a.m)[i] = make_float4(m[0], m[1], m[2], m[3]);
    reinterpret_cast<float4*>(a.v)[i] = make_float4(v[0], v[1], v[2], v[3]);
    if (a.ema0 != nullptr) {
      float4 e = reinterpret_cast<float4*>(a.ema0)[i];
      const float r = a.ema_rate0;
      reinterpret_cast<float4*>(a.ema0)[i] = make_float4(e.x * r + p[0] * (1.f - r), e.y * r + p[1] * (1.f - r), e.z * r + p[2] * (1.f - r), e.w * r + p[3] * (1.f - r));
    }
    if (a.ema1 != nullptr) {
      float4 e = reinterpret_cast<float4*>(a.ema1)[i];
      const float r = a.ema_rate1;
      reinterpret_cast<float4*>(a.ema1)[i] = make_float4(e.x * r + p[0] * (1.f - r), e.y * r + p[1] * (1.f - r), e.z * r + p[2] * (1.f - r), e.w * r + p[3] * (1.f - r));
    }
  }
}


// ---------------- B8 masked MSE backward: grid (chunks, B*T) ----------------------------------------------------------
__global__ void __launch_bounds__(256) masked_mse_bwd_kernel(fdm_masked_mse_bwd_args a) {
  pdl_wait();
  const int f = blockIdx.y, b = f / a.T;
  float w = 0.f;
  if (a.g_mse != nullptr) w += a.g_mse[b] * (a.m1 ? a.m1[f] : 1.f);
  if (a.g_eval != nullptr) w += a.g_eval[b] * (a.m2 ? a.m2[f] : 1.f);
  w *= 2.f / ((float)a.per_frame * (float)a.T);
  const float* o = a.out + (size_t)f * a.per_frame;
  const float* t = a.target + (size_t)f * a.per_frame;
  float* d = a.d_out + (size_t)f * a.per_frame;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.per_frame; i += (long long)gridDim.x * blockDim.x)
    d[i] = w * (o[i] - t[i]);
}

}  // namespace fdm

using namespace fdm;

extern "C" int fdm_pack_weights(const fdm_pack_weights_args* a, void* stream) {
  FDM_REQUIRE(a && a->problems && a->count > 0 && a->max_elems > 0, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->count <= 65535, FDM_ERR_UNSUPPORTED);
  int gx = (a->max_elems + 255) / 256;
  if (gx > 64) gx = 64;
  fdm::launch(pack_weights_kernel, dim3(gx, a->count), dim3(256), 0, (cudaStream_t)stream, a->problems);
  return check_launch();
}

extern "C" int fdm_accum(const fdm_accum_args* a, void* stream) {
  FDM_REQUIRE(a && a->src && a->dst, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->C % 4 == 0 && a->N > 0 && a->H > 0 && a->W > 0, FDM_ERR_UNSUPPORTED);
  const long long total = (long long)a->N * a->H * a->W * (a->C / 4);
  const int g = grid_for_b(total, 256);
  if (a->src_dtype == FDM_BF16)
    fdm::launch(accum_kernel<__nv_bfloat16>, dim3(g), dim3(256), 0, (cudaStream_t)stream, (const __nv_bfloat16*)a->src, a->dst, a->N, a->H, a->W, a->C, a->pool, a->accumulate);
  else
    fdm::launch(accum_kernel<float>, dim3(g), dim3(256), 0, (cudaStream_t)stream, (const float*)a->src, a->dst, a->N, a->H, a->W, a->C, a->pool, a->accumulate);
  return check_launch();
}

extern "C" int fdm_nchw_to_nhwc(const fdm_nchw_to_nhwc_args* a, void* stream) {
  FDM_REQUIRE(a && a->src && a->dst && a->N > 0 && a->C > 0 && a->Cpad >= a->C, FDM_ERR_BAD_ARG);
  const long long total = (long long)a->N * a->H * a->W;
  const unsigned g = (unsigned)((total + 255) / 256);
  if (a->op_dtype == FDM_BF16)
    fdm::launch(nchw_to_nhwc_kernel<__nv_bfloat16>, dim3(g), dim3(256), 0, (cudaStream_t)stream, a->src, (__nv_bfloat16*)a->dst, a->N, a->C, a->H * a->W, a->Cpad);
  else
    fdm::launch(nchw_to_nhwc_kernel<float>, dim3(g), dim3(256), 0, (cudaStream_t)stream, a->src, (float*)a->dst, a->N, a->C, a->H * a->W, a->Cpad);
  return check_launch();
}

extern "C" int fdm_sum_parts(const fdm_sum_parts_args* a, void* stream) {
  FDM_REQUIRE(a && a->parts && a->out && a->count > 0 && a->n > 0, FDM_ERR_BAD_ARG);
  fdm::launch(sum_parts_kernel, dim3(grid_for_b(a->n, 256)), dim3(256), 0, (cudaStream_t)stream, a->parts, a->out, (long long)a->part_stride, (long long)a->n, a->count, a->accumulate);
  return check_launch();
}

extern "C" int fdm_grouped_linear_bwd(const fdm_grouped_linear_bwd_args* a, void* stream) {
  FDM_REQUIRE(a && a->problems && a->count > 0 && a->max_M > 0 && a->max_Nout > 0 && a->max_K > 0, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->count <= 65535, FDM_ERR_UNSUPPORTED);
  const int kx = (a->max_K + 127) / 128;
  int ny = a->max_Nout < 64 ? a->max_Nout : 64;
  fdm::launch(linear_bwd_w_kernel, dim3(kx, ny, a->count), dim3(128), 0, (cudaStream_t)stream, a->problems);
  fdm::launch(linear_bwd_x_kernel, dim3(kx, a->count), dim3(128), 0, (cudaStream_t)stream, a->problems);
  return check_launch();
}

extern "C" int fdm_rpe_hidden_bwd(const fdm_rpe_hidden_bwd_args* a, void* stream) {
  FDM_REQUIRE(a && a->te && a->frame_indices && a->problems && a->dte && a->count > 0 && a->max_C > 0, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->B <= 65535 && a->count <= 65535, FDM_ERR_UNSUPPORTED);
  dim3 grid((a->max_C + 31) / 32, a->B, a->count);
  if (a->dhidden_dtype == FDM_BF16)
    fdm::launch(rpe_hidden_bwd_kernel<__nv_bfloat16>, grid, dim3(32, 8), 0, (cudaStream_t)stream, a->te, a->frame_indices, a->problems, a->dte, a->T, a->te_stride);
  else
    fdm::launch(rpe_hidden_bwd_kernel<float>, grid, dim3(32, 8), 0, (cudaStream_t)stream, a->te, a->frame_indices, a->problems, a->dte, a->T, a->te_stride);
  return check_launch();
}

extern "C" int fdm_adamw(const fdm_adamw_args* a, void* stream) {
  FDM_REQUIRE(a && a->p && a->g && a->m && a->v && a->n > 0, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->n % 4 == 0, FDM_ERR_UNSUPPORTED);  // flat buffers are laid out in 16-byte slots
  fdm::launch(adamw_flat_kernel, dim3(grid_for_b(a->n / 4, 256)), dim3(256), 0, (cudaStream_t)stream, *a);
  return check_launch();
}

extern "C" int fdm_masked_mse_bwd(const fdm_masked_mse_bwd_args* a, void* stream) {
  FDM_REQUIRE(a && a->out && a->target && a->d_out && (a->g_mse || a->g_eval), FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->B > 0 && a->T > 0 && a->per_frame > 0, FDM_ERR_BAD_ARG);
  int chunks = (int)((a->per_frame + 256 * 4 - 1) / (256 * 4));
  if (chunks > 64) chunks = 64;
  fdm::launch(masked_mse_bwd_kernel, dim3(chunks, a->B * a->T), dim3(256), 0, (cudaStream_t)stream, *a);
  return check_launch();
}
