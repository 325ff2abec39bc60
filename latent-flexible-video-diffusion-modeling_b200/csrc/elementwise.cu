// Elementwise / small kernels: input preparation, casts, the fused DDPM posterior update, q_sample,
// masked MSE, and the per-step conditioning path (timestep embedding, grouped small linears, RPENet hidden).
#include "common.cuh"

namespace fdm {

// ---------------- A1 input prep (unet.py:439-449): NCHW frames -> NHWC (+indicator channel) ----------
__global__ void input_prep_kernel(const float* __restrict__ x, const float* __restrict__ x0,
                                  const float* __restrict__ obs, float* __restrict__ xin,
                                  __nv_bfloat16* __restrict__ xin_bf16, int N, int C, int HW, int Cpad) {
  pdl_wait();
  // one thread per (n, pixel); reads are coalesced across pixels per channel plane
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)N * HW) return;
  int n = (int)(i / HW), px = (int)(i - (long long)n * HW);
  float m = obs[n];
  const float* xs = x + (size_t)n * C * HW + px;
  const float* x0s = x0 + (size_t)n * C * HW + px;
  if (xin != nullptr) {
    float* o = xin + (size_t)i * (C + 1);
    for (int c = 0; c < C; ++c) o[c] = xs[(size_t)c * HW] * (1.f - m) + x0s[(size_t)c * HW] * m;
    o[C] = m;
  }
  if (xin_bf16 != nullptr) {
    __nv_bfloat16* o = xin_bf16 + (size_t)i * Cpad;
    for (int c = 0; c < Cpad; ++c) {
      float v = c < C ? xs[(size_t)c * HW] * (1.f - m) + x0s[(size_t)c * HW] * m : (c == C ? m : 0.f);
      o[c] = __float2bfloat16_rn(v);
    }
  }
}

// ---------------- A6 nearest x2 upsample + cast (unet.py:85) ------------------------------------------
template <typename OT>
__global__ void cast_kernel(const float* __restrict__ x, OT* __restrict__ out, int N, int H, int W, int C, int up) {
  pdl_wait();
  const int Ho = up ? 2 * H : H, Wo = up ? 2 * W : W;
  const int quads = C / 4;
  long long total = (long long)N * Ho * Wo * quads;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int q = (int)(i % quads);
    long long pix = i / quads;
    int ow = (int)(pix % Wo);
    long long r = pix / Wo;
    int oh = (int)(r % Ho), n = (int)(r / Ho);
    int ih = up ? oh >> 1 : oh, iw = up ? ow >> 1 : ow;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    // up == 2: zero insertion (gradient of a stride-2 conv output, laid out for a stride-1 dgrad / wgrad)
    if (up != 2 || ((oh | ow) & 1) == 0) v = *reinterpret_cast<const float4*>(x + (((size_t)n * H + ih) * W + iw) * C + q * 4);
    OpType<OT>::store4(out + (size_t)pix * C + q * 4, v);
  }
}

// bf16 nearest x2 upsample driven by the INPUT: one thread reads 8 channels of one source pixel once (two 16-byte loads) and writes
// them to its four destination pixels with 16-byte stores (the output-driven kernel above re-reads every source value four times,
// pays three 64-bit divisions per element and stores 8 bytes at a time: 27 us for the 16x16 -> 32x32 x 128-channel cast of the cfg4
// shard against 63 MB of traffic)
__global__ void __launch_bounds__(256) upsample2_cast_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ out, int N,
                                                                 int H, int W, int C) {
  pdl_wait();
  const int oct = C >> 3;
  const long long total = (long long)N * H * W * oct;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int o = (int)(i % oct);
    const long long pix = i / oct;  // (n, ih, iw)
    const int iw = (int)(pix % W);
    const long long r = pix / W;
    const int ih = (int)(r % H), n = (int)(r / H);
    const float4 a = __ldg(reinterpret_cast<const float4*>(x + (size_t)pix * C + o * 8));
    const float4 b = __ldg(reinterpret_cast<const float4*>(x + (size_t)pix * C + o * 8 + 4));
    __nv_bfloat162 h0 = __floats2bfloat162_rn(a.x, a.y), h1 = __floats2bfloat162_rn(a.z, a.w);
    __nv_bfloat162 h2 = __floats2bfloat162_rn(b.x, b.y), h3 = __floats2bfloat162_rn(b.z, b.w);
    uint4 w;
    w.x = *reinterpret_cast<uint32_t*>(&h0); w.y = *reinterpret_cast<uint32_t*>(&h1);
    w.z = *reinterpret_cast<uint32_t*>(&h2); w.w = *reinterpret_cast<uint32_t*>(&h3);
    __nv_bfloat16* d = out + (((size_t)n * 2 * H + 2 * ih) * 2 * W + 2 * iw) * C + o * 8;
    *reinterpret_cast<uint4*>(d) = w;
    *reinterpret_cast<uint4*>(d + C) = w;
    *reinterpret_cast<uint4*>(d + (size_t)2 * W * C) = w;
    *reinterpret_cast<uint4*>(d + (size_t)2 * W * C + C) = w;
  }
}

// plain fp32 -> bf16 cast of a flat tensor: 8 elements per thread (two 16-byte loads, one 16-byte store), no index arithmetic
__global__ void __launch_bounds__(256) flat_cast_bf16_kernel(const float4* __restrict__ x, uint4* __restrict__ out, long long n8) {
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const float4 a = __ldg(x + 2 * i), b = __ldg(x + 2 * i + 1);
    __nv_bfloat162 h0 = __floats2bfloat162_rn(a.x, a.y), h1 = __floats2bfloat162_rn(a.z, a.w);
    __nv_bfloat162 h2 = __floats2bfloat162_rn(b.x, b.y), h3 = __floats2bfloat162_rn(b.z, b.w);
    uint4 w;
    w.x = *reinterpret_cast<uint32_t*>(&h0); w.y = *reinterpret_cast<uint32_t*>(&h1);
    w.z = *reinterpret_cast<uint32_t*>(&h2); w.w = *reinterpret_cast<uint32_t*>(&h3);
    out[i] = w;
  }
}

// cast + column sums: the fp32 gradient of a conv output becomes the bf16 operand of its dgrad / wgrad, and its column sums ARE
// the bias gradient — one read instead of a second pass over the tensor (the separate bias-gradient kernels were 7 % of the
// 128-px training step).  block = (C/4 quads) x ppi pixel lanes; block partials -> fp32 atomics (colsum zeroed by the caller).
template <typename OT>
__global__ void __launch_bounds__(256) cast_colsum_kernel(const float* __restrict__ x, OT* __restrict__ out, float* __restrict__ cs,
                                                          float* __restrict__ cs2, long long rows, int C, long long rows_per_block) {
  pdl_wait();
  __shared__ float4 red[256];
  const int quads = C / 4;
  const int q = threadIdx.x % quads, pl = threadIdx.x / quads, ppi = blockDim.x / quads;
  const long long r0 = (long long)blockIdx.x * rows_per_block;
  const long long r1 = r0 + rows_per_block < rows ? r0 + rows_per_block : rows;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  for (long long r = r0 + pl; r < r1; r += 2 * ppi) {
    const bool two = r + ppi < r1;
    const float4 a = *reinterpret_cast<const float4*>(x + (size_t)r * C + q * 4);
    float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
    if (two) b = *reinterpret_cast<const float4*>(x + (size_t)(r + ppi) * C + q * 4);
    OpType<OT>::store4(out + (size_t)r * C + q * 4, a);
    if (two) OpType<OT>::store4(out + (size_t)(r + ppi) * C + q * 4, b);
    s.x += a.x + b.x; s.y += a.y + b.y; s.z += a.z + b.z; s.w += a.w + b.w;
  }
  red[threadIdx.x] = s;
  __syncthreads();
  if (pl == 0) {
    for (int k = 1; k < ppi; ++k) {
      const float4 o = red[k * quads + q];
      s.x += o.x; s.y += o.y; s.z += o.z; s.w += o.w;
    }
    float* d = cs + q * 4;
    atomicAdd(d, s.x); atomicAdd(d + 1, s.y); atomicAdd(d + 2, s.z); atomicAdd(d + 3, s.w);
    if (cs2 != nullptr) {
      d = cs2 + q * 4;
      atomicAdd(d, s.x); atomicAdd(d + 1, s.y); atomicAdd(d + 2, s.z); atomicAdd(d + 3, s.w);
    }
  }
}

// ---------------- A16-A18 fused DDPM posterior update -------------------------------------------------
// (philox4x32_10: common.cuh)
// two standard normals from two 32-bit words (Box-Muller; u1 in (0,1], precise logf / sincosf)
__device__ __forceinline__ float2 box_muller(uint32_t a, uint32_t b) {
  const float u1 = ((float)a + 1.0f) * 2.3283064365386963e-10f;  // (a + 1) / 2^32; a = 2^32-1 rounds to 1.0 -> log = 0
  const float u2 = (float)b * 2.3283064365386963e-10f;
  const float r = sqrtf(-2.0f * logf(u1));
  float sn, cs;
  sincospif(2.0f * u2, &sn, &cs);
  return make_float2(r * cs, r * sn);
}

// x and sample may be the SAME buffer (the graph sampler updates x_t in place): every element is read and then written by
// the same thread, and neither pointer is declared __restrict__ (no ld.global.nc for x).
// noise == nullptr: the step's Gaussian noise is generated in the kernel (perf mode: 12 instead of 16 bytes per element and
// no separate normal_() launch): Philox4x32-10 keyed by philox[0] (seed), counter = (element quad index, t[b], philox[1] (stage
// nonce)) -> an independent stream per (element, diffusion step, stage).  Not bit-compatible with torch's generator.
__global__ void ddpm_step_kernel(const float4* x, const float4* __restrict__ eps,
                                 const float4* __restrict__ noise, const float* __restrict__ coef,
                                 const int64_t* __restrict__ t, float4* sample,
                                 float4* __restrict__ pred, const unsigned long long* __restrict__ philox,
                                 long long per_video4, int B, int clip) {
  pdl_wait();
  long long total = per_video4 * B;
  unsigned long long seed = 0ull, nonce = 0ull;
  if (noise == nullptr) { seed = philox[0]; nonce = philox[1]; }
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int b = (int)(i / per_video4);
    const long long tb = t[b];
    const float* c = coef + (size_t)tb * 8;
    const float ca = c[0], cb = c[1], c1 = c[2], c2 = c[3], sg = c[4];
    float4 xv = x[i], ev = eps[i], nv;
    if (noise != nullptr) {
      nv = noise[i];
    } else {
      const uint4 r = philox4x32_10(make_uint4((uint32_t)i, (uint32_t)((unsigned long long)i >> 32), (uint32_t)tb, (uint32_t)nonce),
                                    make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
      const float2 n0 = box_muller(r.x, r.y), n1 = box_muller(r.z, r.w);
      nv = make_float4(n0.x, n0.y, n1.x, n1.y);
    }
    float xin[4] = {xv.x, xv.y, xv.z, xv.w}, e[4] = {ev.x, ev.y, ev.z, ev.w}, nz[4] = {nv.x, nv.y, nv.z, nv.w};
    float s[4], ps[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      // same association as the reference: (a*x) - (b*eps); c1*xs + c2*x; mean + sigma*noise — no FMA contraction
      float xs = __fsub_rn(__fmul_rn(ca, xin[j]), __fmul_rn(cb, e[j]));
      if (clip) xs = fminf(fmaxf(xs, -1.f), 1.f);
      float mean = __fadd_rn(__fmul_rn(c1, xs), __fmul_rn(c2, xin[j]));
      s[j] = __fadd_rn(mean, __fmul_rn(sg, nz[j]));
      ps[j] = xs;
    }
    sample[i] = make_float4(s[0], s[1], s[2], s[3]);
    if (pred != nullptr) pred[i] = make_float4(ps[0], ps[1], ps[2], ps[3]);
  }
}

// ---------------- A20 q_sample ------------------------------------------------------------------------
__global__ void q_sample_kernel(const float4* __restrict__ x0, const float4* __restrict__ noise,
                                const float* __restrict__ coef2, const int64_t* __restrict__ t,
                                float4* __restrict__ xt, long long per_video4, int B) {
  pdl_wait();
  long long total = per_video4 * B;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int b = (int)(i / per_video4);
    const float a = coef2[(size_t)t[b] * 2], s = coef2[(size_t)t[b] * 2 + 1];
    float4 xv = x0[i], nv = noise[i];
    xt[i] = make_float4(__fadd_rn(__fmul_rn(a, xv.x), __fmul_rn(s, nv.x)), __fadd_rn(__fmul_rn(a, xv.y), __fmul_rn(s, nv.y)),
                        __fadd_rn(__fmul_rn(a, xv.z), __fmul_rn(s, nv.z)), __fadd_rn(__fmul_rn(a, xv.w), __fmul_rn(s, nv.w)));
  }
}

// ---------------- A21 masked MSE means: grid (chunks, B*T) --------------------------------------------
__global__ void masked_mse_kernel(const float* __restrict__ eps, const float* __restrict__ noise,
                                  const float* __restrict__ m1, const float* __restrict__ m2,
                                  float* __restrict__ mse, float* __restrict__ evl, long long per_frame, int T) {
  pdl_wait();
  const int f = blockIdx.y, b = f / T;
  const float* e = eps + (size_t)f * per_frame;
  const float* n = noise + (size_t)f * per_frame;
  float s = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_frame; i += (long long)gridDim.x * blockDim.x) {
    float d = n[i] - e[i];
    s += d * d;
  }
  s = warp_sum(s);
  __shared__ float red[32];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) {
      const float inv = 1.f / ((float)per_frame * (float)T);
      atomicAdd(mse + b, v * (m1 ? m1[f] : 1.f) * inv);
      atomicAdd(evl + b, v * (m2 ? m2[f] : 1.f) * inv);
    }
  }
}

// ---------------- A2 timestep embedding (nn.py:105-123) -----------------------------------------------
__global__ void timestep_embedding_kernel(const float* __restrict__ t, const int64_t* __restrict__ t_index,
                                          const float* __restrict__ t_table, const float* __restrict__ freqs,
                                          float* __restrict__ out, int B, int dim) {
  pdl_wait();
  const int half = dim / 2;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * half) return;
  int b = i / half, k = i - b * half;
  const float tv = t_index != nullptr ? t_table[t_index[b]] : t[b];
  float arg = tv * freqs[k];
  out[(size_t)b * dim + k] = cosf(arg);
  out[(size_t)b * dim + half + k] = sinf(arg);
  if ((dim & 1) && k == 0) out[(size_t)b * dim + dim - 1] = 0.f;
}

// ---------------- grouped small linear: y = act(x) W^T + b -------------------------------------------------------------
// Two kernels.  (1) M <= 8 (the per-step conditioning path: time MLP, FiLM and RPE time projections all have M = B rows):
// one WARP per output column, lanes split K with coalesced reads of the weight row, shuffle reduction — hundreds of
// independent warps instead of a handful of 16x64 tiles walking K serially (these launches sit on the step's critical path).
// (2) general tiled kernel (fp32 mode's RPENet output linear, M = B*T*T rows).
constexpr int GL_SMALL_M = 8;
__global__ void __launch_bounds__(256) grouped_linear_small_kernel(const fdm_linear_problem* __restrict__ probs) {
  extern __shared__ float gl_xs[];  // [M][K]: the (activated) input rows, computed once per block
  pdl_wait();
  const fdm_linear_problem pr = probs[blockIdx.y];
  const int lane = threadIdx.x & 31;
  const int n = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (blockIdx.x * 8 >= pr.Nout) return;  // whole block out of range for this (narrower) problem
  for (int i = threadIdx.x; i < pr.M * pr.K; i += 256) {
    const int m = i / pr.K, k = i - m * pr.K;
    float xv = __ldg(pr.x + (size_t)m * pr.ldx + k);
    gl_xs[i] = pr.silu_in ? silu_precise(xv) : xv;
  }
  __syncthreads();
  if (n >= pr.Nout) return;
  float acc[GL_SMALL_M];
#pragma unroll
  for (int m = 0; m < GL_SMALL_M; ++m) acc[m] = 0.f;
  const float* wrow = pr.w + (size_t)n * pr.K;
  for (int k = lane; k < pr.K; k += 32) {
    const float w = __ldg(wrow + k);
#pragma unroll
    for (int m = 0; m < GL_SMALL_M; ++m)
      if (m < pr.M) acc[m] = fmaf(gl_xs[m * pr.K + k], w, acc[m]);
  }
#pragma unroll
  for (int m = 0; m < GL_SMALL_M; ++m) acc[m] = warp_sum(acc[m]);
  if (lane == 0) {
    const float bias = pr.b ? pr.b[n] : 0.f;
#pragma unroll
    for (int m = 0; m < GL_SMALL_M; ++m)
      if (m < pr.M) pr.y[(size_t)m * pr.ldy + n] = acc[m] + bias;
  }
}

constexpr int GL_TM = 16, GL_TN = 64, GL_TK = 32;
__global__ void __launch_bounds__(256) grouped_linear_kernel(const fdm_linear_problem* __restrict__ probs) {
  pdl_wait();
  const fdm_linear_problem pr = probs[blockIdx.z];
  const int m0 = blockIdx.y * GL_TM, n0 = blockIdx.x * GL_TN;
  if (m0 >= pr.M || n0 >= pr.Nout) return;
  __shared__ float xs[GL_TM][GL_TK + 1];
  __shared__ float ws[GL_TN][GL_TK + 1];
  const int tid = threadIdx.x;
  const int tn = tid & 63, tm = tid >> 6;  // each thread: column tn, rows tm*4 .. tm*4+3
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int k0 = 0; k0 < pr.K; k0 += GL_TK) {
    for (int i = tid; i < GL_TM * GL_TK; i += 256) {
      int r = i / GL_TK, k = i - r * GL_TK;
      float v = 0.f;
      if (m0 + r < pr.M && k0 + k < pr.K) {
        v = pr.x[(size_t)(m0 + r) * pr.ldx + k0 + k];
        if (pr.silu_in) v = silu_precise(v);
      }
      xs[r][k] = v;
    }
    for (int i = tid; i < GL_TN * GL_TK; i += 256) {
      int r = i / GL_TK, k = i - r * GL_TK;
      ws[r][k] = (n0 + r < pr.Nout && k0 + k < pr.K) ? pr.w[(size_t)(n0 + r) * pr.K + k0 + k] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < GL_TK; ++k) {
      float w = ws[tn][k];
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i] = fmaf(xs[tm * 4 + i][k], w, acc[i]);
    }
    __syncthreads();
  }
  if (n0 + tn < pr.Nout) {
    float bias = pr.b ? pr.b[n0 + tn] : 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int m = m0 + tm * 4 + i;
      if (m < pr.M) pr.y[(size_t)m * pr.ldy + n0 + tn] = acc[i] + bias;
    }
  }
}

// ---------------- A9 RPENet hidden layer (rpe.py:21-30) -----------------------------------------------
template <typename OT>
__global__ void rpe_hidden_kernel(const float* __restrict__ te, const int64_t* __restrict__ fi,
                                  const fdm_rpe_hidden_problem* __restrict__ probs, int B, int T, int te_stride) {
  pdl_wait();
  const fdm_rpe_hidden_problem pr = probs[blockIdx.y];
  const int C = pr.C;
  long long total = (long long)B * T * T * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    long long r = i / C;
    int s = (int)(r % T);
    r /= T;
    int t = (int)(r % T), b = (int)(r / T);
    float d = (float)(fi[(size_t)b * T + t] - fi[(size_t)b * T + s]);
    float f0 = logf(1.f + fmaxf(d, 0.f)), f1 = logf(1.f + fmaxf(-d, 0.f)), f2 = d == 0.f ? 1.f : 0.f;
    // embed_distances(feats) = f0*w0 + f1*w1 + f2*w2 + bd, then + (W_t temb + b_t)
    float e = fmaf(f2, pr.wd[c * 3 + 2], fmaf(f1, pr.wd[c * 3 + 1], f0 * pr.wd[c * 3])) + pr.bd[c];
    e += te[(size_t)b * te_stride + pr.te_off + c];
    OpType<OT>::store(reinterpret_cast<OT*>(pr.hidden) + i, silu_precise(e));
  }
}

static inline int grid_for(long long total, int threads) {
  long long g = (total + threads - 1) / threads;
  long long cap = 148LL * 16;
  return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

}  // namespace fdm

using namespace fdm;

extern "C" int fdm_input_prep(const fdm_input_prep_args* a, void* stream) {
  FDM_REQUIRE(a && a->x && a->x0 && a->obs_mask && (a->xin || a->xin_bf16), FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->N > 0 && a->C > 0 && a->H > 0 && a->W > 0, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->xin_bf16 == nullptr || a->Cpad > a->C, FDM_ERR_BAD_ARG);
  long long total = (long long)a->N * a->H * a->W;
  fdm::launch(input_prep_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, a->x, a->x0, a->obs_mask, a->xin, (__nv_bfloat16*)a->xin_bf16, a->N, a->C, a->H * a->W, a->Cpad);
  return check_launch();
}

extern "C" int fdm_cast(const fdm_cast_args* a, void* stream) {
  FDM_REQUIRE(a && a->x && a->out, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->C % 4 == 0 && a->N > 0, FDM_ERR_UNSUPPORTED);
  if (a->colsum != nullptr) {
    FDM_REQUIRE(a->upsample == 0 && a->C / 4 <= 256, FDM_ERR_UNSUPPORTED);
    const long long rows = (long long)a->N * a->H * a->W;
    const int quads = a->C / 4;
    int ppi = 256 / quads;
    if (ppi > rows) ppi = (int)rows;
    long long blocks = (rows + 8 * ppi - 1) / (8 * ppi);  // >= 8 rows per thread
    if (blocks > 148 * 8) blocks = 148 * 8;
    const long long rpb = ((rows + blocks - 1) / blocks + ppi - 1) / ppi * ppi;
    blocks = (rows + rpb - 1) / rpb;
    if (a->op_dtype == FDM_BF16)
      fdm::launch(cast_colsum_kernel<__nv_bfloat16>, dim3((unsigned)blocks), dim3(quads * ppi), 0, (cudaStream_t)stream, a->x, (__nv_bfloat16*)a->out, a->colsum, a->colsum2, rows, a->C, rpb);
    else
      fdm::launch(cast_colsum_kernel<float>, dim3((unsigned)blocks), dim3(quads * ppi), 0, (cudaStream_t)stream, a->x, (float*)a->out, a->colsum, a->colsum2, rows, a->C, rpb);
    return check_launch();
  }
  if (a->upsample == 1 && a->op_dtype == FDM_BF16 && a->C % 8 == 0) {
    const long long tot8 = (long long)a->N * a->H * a->W * (a->C / 8);
    fdm::launch(upsample2_cast_bf16_kernel, dim3(grid_for(tot8, 256)), dim3(256), 0, (cudaStream_t)stream, a->x, (__nv_bfloat16*)a->out, a->N,
                a->H, a->W, a->C);
    return check_launch();
  }
  if (a->upsample == 0 && a->op_dtype == FDM_BF16 && ((long long)a->N * a->H * a->W * a->C) % 8 == 0) {
    const long long n8 = (long long)a->N * a->H * a->W * a->C / 8;
    fdm::launch(flat_cast_bf16_kernel, dim3(grid_for(n8, 256)), dim3(256), 0, (cudaStream_t)stream, (const float4*)a->x, (uint4*)a->out, n8);
    return check_launch();
  }
  long long total = (long long)a->N * a->H * a->W * (a->upsample ? 4 : 1) * (a->C / 4);
  int g = grid_for(total, 256);
  if (a->op_dtype == FDM_BF16)
    fdm::launch(cast_kernel<__nv_bfloat16>, dim3(g), dim3(256), 0, (cudaStream_t)stream, a->x, (__nv_bfloat16*)a->out, a->N, a->H, a->W, a->C, a->upsample);
  else
    fdm::launch(cast_kernel<float>, dim3(g), dim3(256), 0, (cudaStream_t)stream, a->x, (float*)a->out, a->N, a->H, a->W, a->C, a->upsample);
  return check_launch();
}

extern "C" int fdm_ddpm_step(const fdm_ddpm_step_args* a, void* stream) {
  FDM_REQUIRE(a && a->x && a->eps && (a->noise || a->philox) && a->coef && a->t && a->sample, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->per_video % 4 == 0 && a->B > 0, FDM_ERR_UNSUPPORTED);
  long long pv4 = a->per_video / 4;
  fdm::launch(ddpm_step_kernel, dim3(grid_for(pv4 * a->B, 256)), dim3(256), 0, (cudaStream_t)stream, (const float4*)a->x, (const float4*)a->eps, (const float4*)a->noise, a->coef, a->t, (float4*)a->sample,
      (float4*)a->pred_xstart, (const unsigned long long*)a->philox, pv4, a->B, a->clip);
  return check_launch();
}

extern "C" int fdm_q_sample(const fdm_q_sample_args* a, void* stream) {
  FDM_REQUIRE(a && a->x0 && a->noise && a->coef2 && a->t && a->x_t, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->per_video % 4 == 0 && a->B > 0, FDM_ERR_UNSUPPORTED);
  long long pv4 = a->per_video / 4;
  fdm::launch(q_sample_kernel, dim3(grid_for(pv4 * a->B, 256)), dim3(256), 0, (cudaStream_t)stream, (const float4*)a->x0, (const float4*)a->noise, a->coef2, a->t, (float4*)a->x_t, pv4, a->B);
  return check_launch();
}

extern "C" int fdm_masked_mse(const fdm_masked_mse_args* a, void* stream) {
  FDM_REQUIRE(a && a->eps && a->noise && a->mse && a->eval, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->B > 0 && a->T > 0 && a->per_frame > 0, FDM_ERR_BAD_ARG);
  int chunks = (int)((a->per_frame + 256 * 8 - 1) / (256 * 8));
  if (chunks > 64) chunks = 64;
  dim3 grid(chunks, a->B * a->T);
  fdm::launch(masked_mse_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, a->eps, a->noise, a->m1, a->m2, a->mse, a->eval, a->per_frame, a->T);
  return check_launch();
}

extern "C" int fdm_timestep_embedding(const fdm_timestep_embedding_args* a, void* stream) {
  FDM_REQUIRE(a && a->freqs && a->out && a->B > 0 && a->dim >= 2, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->t != nullptr || (a->t_index != nullptr && a->t_table != nullptr), FDM_ERR_BAD_ARG);
  int total = a->B * (a->dim / 2);
  fdm::launch(timestep_embedding_kernel, dim3((total + 127) / 128), dim3(128), 0, (cudaStream_t)stream, a->t, a->t_index, a->t_table, a->freqs, a->out, a->B, a->dim);
  return check_launch();
}

extern "C" int fdm_grouped_linear(const fdm_grouped_linear_args* a, void* stream) {
  FDM_REQUIRE(a && a->problems && a->count > 0 && a->max_M > 0 && a->max_Nout > 0, FDM_ERR_BAD_ARG);
  if (a->max_M <= GL_SMALL_M && a->max_K > 0 && (size_t)a->max_M * a->max_K * sizeof(float) <= 48 * 1024) {
    dim3 grid((a->max_Nout + 7) / 8, a->count);
    FDM_REQUIRE(grid.y <= 65535, FDM_ERR_UNSUPPORTED);
    fdm::launch(grouped_linear_small_kernel, grid, dim3(256), (size_t)a->max_M * a->max_K * sizeof(float), (cudaStream_t)stream,
                a->problems);
    return check_launch();
  }
  dim3 grid((a->max_Nout + GL_TN - 1) / GL_TN, (a->max_M + GL_TM - 1) / GL_TM, a->count);
  FDM_REQUIRE(grid.y <= 65535 && grid.z <= 65535, FDM_ERR_UNSUPPORTED);
  fdm::launch(grouped_linear_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, a->problems);
  return check_launch();
}

extern "C" int fdm_rpe_hidden(const fdm_rpe_hidden_args* a, void* stream) {
  FDM_REQUIRE(a && a->te && a->frame_indices && a->problems && a->count > 0 && a->max_C > 0, FDM_ERR_BAD_ARG);
  long long total = (long long)a->B * a->T * a->T * a->max_C;
  int gx = grid_for(total, 256);
  if (gx > 592) gx = 592;
  dim3 grid(gx, a->count);
  if (a->hidden_dtype == FDM_BF16)
    fdm::launch(rpe_hidden_kernel<__nv_bfloat16>, dim3(grid), dim3(256), 0, (cudaStream_t)stream, a->te, a->frame_indices, a->problems, a->B, a->T, a->te_stride);
  else
    fdm::launch(rpe_hidden_kernel<float>, dim3(grid), dim3(256), 0, (cudaStream_t)stream, a->te, a->frame_indices, a->problems, a->B, a->T, a->te_stride);
  return check_launch();
}
