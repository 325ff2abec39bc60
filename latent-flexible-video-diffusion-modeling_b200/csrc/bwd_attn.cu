// Attention backward on CUDA cores (fp32 math), flash-style: the score matrices are recomputed, never stored.
// Reference: what autograd runs for rpe.py:139-170 (matmul / einsum / softmax / masked_fill backward).
//
//   forward   S = scale*(q.k + q.Rk[t,s] + k.Rq[s,t]) ; P = softmax_s(S | mask) ; O = P (v + Rv[t,s])
//   backward  D_t = dO_t.O_t ; dP = dO.(v + Rv) ; dS = P (dP - D) scale
//             dq_t = sum_s dS (k_s + Rk[t,s]) ; dk_s = sum_t dS (q_t + Rq[s,t]) ; dv_s = sum_t P dO_t
//             dRk[t,s] = sum_px dS q_t ; dRq[s,t] = sum_px dS k_s ; dRv[t,s] = sum_px P dO_t      (temporal only)
// Two kernels per attention: a row-owner pass (log-sum-exp, D, dq, dRk) and a column-owner pass (dk, dv, dRq, dRv) that
// re-forms P from the stored log-sum-exp — no cross-CTA reduction except the pixel sums of the RPE tables (fp32 atomics).
#include "common.cuh"

namespace fdm {

// =====================================================================================================================
// spatial attention backward: per (frame n, head h) sequences of L pixels, head dim F
// =====================================================================================================================
constexpr int SA_KB = 64;   // keys (queries) staged per block iteration
constexpr int SA_RPW = 4;   // rows per warp
constexpr int SA_ROWS = 32; // rows per CTA (8 warps)
constexpr int SA_MAXU = 4;  // F <= 128: up to 4 head-dim elements per lane

struct SABwdParams {
  const void* qkv; const void* out; const void* dout; void* dqkv; float* lse; float* dsum;
  int N, L, C, heads, F;
  float scale;
};

// dst[r][f] (row stride ld) = src[(r0 + r) * row_stride + f], zero for rows >= L
template <typename QT>
__device__ __forceinline__ void sa_stage(float* dst, const QT* src, size_t row_stride, int r0, int L, int F, int ld) {
  const int fq = F >> 2;  // head dims are multiples of 8: four elements per load
  for (int i = threadIdx.x; i < SA_KB * fq; i += blockDim.x) {
    const int r = i / fq, f = (i - r * fq) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r0 + r < L) v = OpType<QT>::load4(src + (size_t)(r0 + r) * row_stride + f);
    float* d = dst + r * ld + f;
    d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
  }
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// grid (ceil(L/32), heads, N), block 256.  Warp w owns query rows i0 + w*4 .. +3.
template <typename QT>
__global__ void __launch_bounds__(256) attn_spatial_bwd_q_kernel(SABwdParams p) {
  pdl_wait();
  extern __shared__ __align__(16) float sa_smem[];
  const int F = p.F, ld = F + 1, L = p.L, C = p.C;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float* Ks = sa_smem;
  float* Vs = Ks + SA_KB * ld;
  float* wq = Vs + SA_KB * ld + w * (SA_RPW * 2 * F + SA_RPW * SA_KB);
  float* wdo = wq + SA_RPW * F;
  float* wds = wdo + SA_RPW * F;
  const int n = blockIdx.z, h = blockIdx.y, i0 = blockIdx.x * SA_ROWS + w * SA_RPW;
  const QT* qkv = reinterpret_cast<const QT*>(p.qkv) + (size_t)n * L * 3 * C + h * F;
  const QT* outp = reinterpret_cast<const QT*>(p.out) + (size_t)n * L * C + h * F;
  const QT* dout = reinterpret_cast<const QT*>(p.dout) + (size_t)n * L * C + h * F;
  float D[SA_RPW];
#pragma unroll
  for (int r = 0; r < SA_RPW; ++r) {
    const int i = i0 + r;
    float part = 0.f;
    for (int f = lane; f < F; f += 32) {
      float qv = 0.f, dv = 0.f, ov = 0.f;
      if (i < L) {
        qv = OpType<QT>::load(qkv + (size_t)i * 3 * C + f);
        dv = OpType<QT>::load(dout + (size_t)i * C + f);
        ov = OpType<QT>::load(outp + (size_t)i * C + f);
      }
      wq[r * F + f] = qv;
      wdo[r * F + f] = dv;
      part = fmaf(dv, ov, part);
    }
    D[r] = warp_sum(part);
  }
  __syncwarp();
  // ---- pass 1: log-sum-exp of every owned row
  float mx[SA_RPW], sm[SA_RPW];
#pragma unroll
  for (int r = 0; r < SA_RPW; ++r) { mx[r] = -INFINITY; sm[r] = 0.f; }
  for (int kb = 0; kb < L; kb += SA_KB) {
    __syncthreads();
    sa_stage(Ks, qkv + C, (size_t)3 * C, kb, L, F, ld);
    __syncthreads();
    float s[SA_RPW][2];
#pragma unroll
    for (int r = 0; r < SA_RPW; ++r) { s[r][0] = 0.f; s[r][1] = 0.f; }
    for (int f = 0; f < F; ++f) {
      const float k0 = Ks[lane * ld + f], k1 = Ks[(lane + 32) * ld + f];
#pragma unroll
      for (int r = 0; r < SA_RPW; ++r) {
        const float qv = wq[r * F + f];
        s[r][0] = fmaf(qv, k0, s[r][0]);
        s[r][1] = fmaf(qv, k1, s[r][1]);
      }
    }
#pragma unroll
    for (int r = 0; r < SA_RPW; ++r)
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (kb + lane + 32 * u < L) {
          const float v = s[r][u] * p.scale;
          if (v > mx[r]) { sm[r] = sm[r] * expf(mx[r] - v) + 1.f; mx[r] = v; }
          else sm[r] += expf(v - mx[r]);
        }
      }
  }
  float lse[SA_RPW];
#pragma unroll
  for (int r = 0; r < SA_RPW; ++r) {
    const float M = warp_max(mx[r]);
    const float t = warp_sum(mx[r] == -INFINITY ? 0.f : sm[r] * expf(mx[r] - M));
    lse[r] = M + logf(t);
  }
  // ---- pass 2: dS and dq
  float dq[SA_RPW][SA_MAXU];
#pragma unroll
  for (int r = 0; r < SA_RPW; ++r)
#pragma unroll
    for (int u = 0; u < SA_MAXU; ++u) dq[r][u] = 0.f;
  for (int kb = 0; kb < L; kb += SA_KB) {
    __syncthreads();
    sa_stage(Ks, qkv + C, (size_t)3 * C, kb, L, F, ld);
    sa_stage(Vs, qkv + 2 * C, (size_t)3 * C, kb, L, F, ld);
    __syncthreads();
    float s[SA_RPW][2], dp[SA_RPW][2];
#pragma unroll
    for (int r = 0; r < SA_RPW; ++r) { s[r][0] = s[r][1] = dp[r][0] = dp[r][1] = 0.f; }
    for (int f = 0; f < F; ++f) {
      const float k0 = Ks[lane * ld + f], k1 = Ks[(lane + 32) * ld + f];
      const float v0 = Vs[lane * ld + f], v1 = Vs[(lane + 32) * ld + f];
#pragma unroll
      for (int r = 0; r < SA_RPW; ++r) {
        const float qv = wq[r * F + f], dv = wdo[r * F + f];
        s[r][0] = fmaf(qv, k0, s[r][0]);
        s[r][1] = fmaf(qv, k1, s[r][1]);
        dp[r][0] = fmaf(dv, v0, dp[r][0]);
        dp[r][1] = fmaf(dv, v1, dp[r][1]);
      }
    }
#pragma unroll
    for (int r = 0; r < SA_RPW; ++r)
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const bool ok = kb + lane + 32 * u < L && i0 + r < L;
        const float P = ok ? expf(s[r][u] * p.scale - lse[r]) : 0.f;
        wds[r * SA_KB + lane + 32 * u] = P * (dp[r][u] - D[r]) * p.scale;
      }
    __syncwarp();
    for (int j = 0; j < SA_KB; ++j) {
      float kv[SA_MAXU];
#pragma unroll
      for (int u = 0; u < SA_MAXU; ++u) kv[u] = (lane + 32 * u < F) ? Ks[j * ld + lane + 32 * u] : 0.f;
#pragma unroll
      for (int r = 0; r < SA_RPW; ++r) {
        const float ds = wds[r * SA_KB + j];
#pragma unroll
        for (int u = 0; u < SA_MAXU; ++u) dq[r][u] = fmaf(ds, kv[u], dq[r][u]);
      }
    }
    __syncwarp();
  }
  QT* dqkv = reinterpret_cast<QT*>(p.dqkv) + (size_t)n * L * 3 * C + h * F;
#pragma unroll
  for (int r = 0; r < SA_RPW; ++r) {
    const int i = i0 + r;
    if (i >= L) continue;
#pragma unroll
    for (int u = 0; u < SA_MAXU; ++u)
      if (lane + 32 * u < F) OpType<QT>::store(dqkv + (size_t)i * 3 * C + lane + 32 * u, dq[r][u]);
    if (lane == 0) {
      p.lse[((size_t)n * p.heads + h) * L + i] = lse[r];
      p.dsum[((size_t)n * p.heads + h) * L + i] = D[r];
    }
  }
}

// grid (ceil(L/32), heads, N), block 256.  Warp w owns key rows j0 + w*4 .. +3; queries are streamed in blocks of 64.
template <typename QT>
__global__ void __launch_bounds__(256) attn_spatial_bwd_kv_kernel(SABwdParams p) {
  pdl_wait();
  extern __shared__ __align__(16) float sa_smem[];
  const int F = p.F, ld = F + 1, L = p.L, C = p.C;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float* Qs = sa_smem;
  float* Ds = Qs + SA_KB * ld;           // dO rows
  float* Ls = Ds + SA_KB * ld;           // [64] lse
  float* Dsum = Ls + SA_KB;              // [64]
  float* wk = Dsum + SA_KB + w * (SA_RPW * 2 * F + 2 * SA_RPW * SA_KB);
  float* wv = wk + SA_RPW * F;
  float* wp = wv + SA_RPW * F;           // [4][64] P
  float* wds = wp + SA_RPW * SA_KB;      // [4][64] dS
  const int n = blockIdx.z, h = blockIdx.y, j0 = blockIdx.x * SA_ROWS + w * SA_RPW;
  const QT* qkv = reinterpret_cast<const QT*>(p.qkv) + (size_t)n * L * 3 * C + h * F;
  const QT* dout = reinterpret_cast<const QT*>(p.dout) + (size_t)n * L * C + h * F;
#pragma unroll
  for (int r = 0; r < SA_RPW; ++r) {
    const int j = j0 + r;
    for (int f = lane; f < F; f += 32) {
      wk[r * F + f] = j < L ? OpType<QT>::load(qkv + (size_t)j * 3 * C + C + f) : 0.f;
      wv[r * F + f] = j < L ? OpType<QT>::load(qkv + (size_t)j * 3 * C + 2 * C + f) : 0.f;
    }
  }
  float dk[SA_RPW][SA_MAXU], dv[SA_RPW][SA_MAXU];
#pragma unroll
  for (int r = 0; r < SA_RPW; ++r)
#pragma unroll
    for (int u = 0; u < SA_MAXU; ++u) { dk[r][u] = 0.f; dv[r][u] = 0.f; }
  const float* lse_g = p.lse + ((size_t)n * p.heads + h) * L;
  const float* dsum_g = p.dsum + ((size_t)n * p.heads + h) * L;
  for (int qb = 0; qb < L; qb += SA_KB) {
    __syncthreads();
    sa_stage(Qs, qkv, (size_t)3 * C, qb, L, F, ld);
    sa_stage(Ds, dout, (size_t)C, qb, L, F, ld);
    if (threadIdx.x < SA_KB) {
      Ls[threadIdx.x] = qb + threadIdx.x < L ? lse_g[qb + threadIdx.x] : 0.f;
      Dsum[threadIdx.x] = qb + threadIdx.x < L ? dsum_g[qb + threadIdx.x] : 0.f;
    }
    __syncthreads();
    float s[SA_RPW][2], dp[SA_RPW][2];
#pragma unroll
    for (int r = 0; r < SA_RPW; ++r) { s[r][0] = s[r][1] = dp[r][0] = dp[r][1] = 0.f; }
    for (int f = 0; f < F; ++f) {
      const float q0 = Qs[lane * ld + f], q1 = Qs[(lane + 32) * ld + f];
      const float d0 = Ds[lane * ld + f], d1 = Ds[(lane + 32) * ld + f];
#pragma unroll
      for (int r = 0; r < SA_RPW; ++r) {
        const float kv = wk[r * F + f], vv = wv[r * F + f];
        s[r][0] = fmaf(q0, kv, s[r][0]);
        s[r][1] = fmaf(q1, kv, s[r][1]);
        dp[r][0] = fmaf(d0, vv, dp[r][0]);
        dp[r][1] = fmaf(d1, vv, dp[r][1]);
      }
    }
#pragma unroll
    for (int r = 0; r < SA_RPW; ++r)
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int il = lane + 32 * u;
        const bool ok = qb + il < L && j0 + r < L;
        const float P = ok ? expf(s[r][u] * p.scale - Ls[il]) : 0.f;
        wp[r * SA_KB + il] = P;
        wds[r * SA_KB + il] = P * (dp[r][u] - Dsum[il]) * p.scale;
      }
    __syncwarp();
    for (int i = 0; i < SA_KB; ++i) {
      float qv[SA_MAXU], dd[SA_MAXU];
#pragma unroll
      for (int u = 0; u < SA_MAXU; ++u) {
        const bool fo = lane + 32 * u < F;
        qv[u] = fo ? Qs[i * ld + lane + 32 * u] : 0.f;
        dd[u] = fo ? Ds[i * ld + lane + 32 * u] : 0.f;
      }
#pragma unroll
      for (int r = 0; r < SA_RPW; ++r) {
        const float P = wp[r * SA_KB + i], ds = wds[r * SA_KB + i];
#pragma unroll
        for (int u = 0; u < SA_MAXU; ++u) {
          dv[r][u] = fmaf(P, dd[u], dv[r][u]);
          dk[r][u] = fmaf(ds, qv[u], dk[r][u]);
        }
      }
    }
    __syncwarp();
  }
  QT* dqkv = reinterpret_cast<QT*>(p.dqkv) + (size_t)n * L * 3 * C + h * F;
#pragma unroll
  for (int r = 0; r < SA_RPW; ++r) {
    const int j = j0 + r;
    if (j >= L) continue;
#pragma unroll
    for (int u = 0; u < SA_MAXU; ++u)
      if (lane + 32 * u < F) {
        OpType<QT>::store(dqkv + (size_t)j * 3 * C + C + lane + 32 * u, dk[r][u]);
        OpType<QT>::store(dqkv + (size_t)j * 3 * C + 2 * C + lane + 32 * u, dv[r][u]);
      }
  }
}

// =====================================================================================================================
// temporal attention backward: per (video b, pixel, head) sequences of T frames; lane <-> pixel, warp <-> frame
// =====================================================================================================================
constexpr int TB_FC = 8;     // head-dim chunk
constexpr int TB_LD = 33;    // padded pixel stride of the staged tiles
constexpr int TB_WARPS = 8;  // frames per CTA (runtime: blockDim.x / 32)

struct TABwdParams {
  const void* qkv; const void* out; const void* dout; const float* Rq; const float* Rk; const float* Rv; const float* mask;
  void* dqkv; float* dRq; float* dRk; float* dRv; float* lse; float* dsum;
  int B, T, HW, C, heads, F;
  float scale;
};

// raw 4-element loads: the conversion to fp32 happens AFTER all loads of a staging step were issued (ncu: 33 % of the stall
// samples of the first version were the bf16 unpack / staging stores waiting on one global load at a time)
template <typename QT>
struct Raw4;
template <>
struct Raw4<float> {
  using T = float4;
  static __device__ __forceinline__ T load(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
  static __device__ __forceinline__ float4 cvt(T v) { return v; }
};
template <>
struct Raw4<__nv_bfloat16> {
  using T = uint2;
  static __device__ __forceinline__ T load(const __nv_bfloat16* p) { return __ldg(reinterpret_cast<const uint2*>(p)); }
  static __device__ __forceinline__ float4 cvt(T u) {
    return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                       __uint_as_float(u.y & 0xffff0000u));
  }
};

// Two tiles staged together (K and V, or Q and dO): tile[(s * 8 + f) * 33 + px] = src[((b*T + s) * HW + px0 + px) * stride + col + f].
// NL = loads per thread and tile at 256 threads (compile-time: all 2*NL loads are in flight before the first store).
template <int NL, typename QT>
__device__ __forceinline__ void tb_stage2(float* tile_a, const QT* src_a, size_t stride_a, int col_a, float* tile_b, const QT* src_b,
                                          size_t stride_b, int col_b, int b, int T, int HW, int px0) {
  typename Raw4<QT>::T ra[NL], rb[NL];
  const int total = T * 32 * (TB_FC / 4);
#pragma unroll
  for (int j = 0; j < NL; ++j) {
    const int i = threadIdx.x + j * blockDim.x;
    if (i < total) {
      const int fq = i % (TB_FC / 4), pl = (i / (TB_FC / 4)) % 32, s = i / (32 * (TB_FC / 4));
      const size_t rowi = (size_t)(b * T + s) * HW + min(px0 + pl, HW - 1);
      ra[j] = Raw4<QT>::load(src_a + rowi * stride_a + col_a + fq * 4);
      if (tile_b != nullptr) rb[j] = Raw4<QT>::load(src_b + rowi * stride_b + col_b + fq * 4);
    }
  }
#pragma unroll
  for (int j = 0; j < NL; ++j) {
    const int i = threadIdx.x + j * blockDim.x;
    if (i < total) {
      const int fq = i % (TB_FC / 4), pl = (i / (TB_FC / 4)) % 32, s = i / (32 * (TB_FC / 4));
      const size_t o = (size_t)(s * TB_FC + fq * 4) * TB_LD + pl;
      const float4 va = Raw4<QT>::cvt(ra[j]);
      tile_a[o] = va.x; tile_a[o + TB_LD] = va.y; tile_a[o + 2 * TB_LD] = va.z; tile_a[o + 3 * TB_LD] = va.w;
      if (tile_b != nullptr) {
        const float4 vb = Raw4<QT>::cvt(rb[j]);
        tile_b[o] = vb.x; tile_b[o + TB_LD] = vb.y; tile_b[o + 2 * TB_LD] = vb.z; tile_b[o + 3 * TB_LD] = vb.w;
      }
    }
  }
}

// tile[(s * 8 + f) * 33 + px] = src[((b*T + s) * HW + px0 + px) * row_stride + col0 + f]   (generic loop: any block size)
template <typename QT>
__device__ __forceinline__ void tb_stage(float* tile, const QT* src, size_t row_stride, int b, int T, int HW, int px0, int col0) {
  for (int i = threadIdx.x; i < T * 32 * (TB_FC / 4); i += blockDim.x) {
    const int fq = i % (TB_FC / 4);
    const int pl = (i / (TB_FC / 4)) % 32;
    const int s = i / (32 * (TB_FC / 4));
    const int pp = min(px0 + pl, HW - 1);
    const float4 v = OpType<QT>::load4(src + ((size_t)(b * T + s) * HW + pp) * row_stride + col0 + fq * 4);
    float* d = tile + (size_t)(s * TB_FC + fq * 4) * TB_LD + pl;
    d[0] = v.x; d[TB_LD] = v.y; d[2 * TB_LD] = v.z; d[3 * TB_LD] = v.w;
  }
}

// out[(x, f)] += sum_px rows[x][px] * cols[f][px]   for x < T, f < 8: lane -> f = lane % 8, x = lane / 8 + 4k.
// rows: [T][33] (per warp), cols: [8][33] with element stride `cs` between f rows.
__device__ __forceinline__ void tb_pixel_gemm(const float* rows, const float* cols, int cstride, int T, int lane, float* dst,
                                              size_t dst_xstride) {
  const int f = lane & 7;
  for (int x = lane >> 3; x < T; x += 4) {
    const float* r = rows + x * TB_LD;
    const float* c = cols + f * cstride;
    float acc = 0.f;
#pragma unroll 8
    for (int px = 0; px < 32; ++px) acc = fmaf(r[px], c[px], acc);
    atomicAdd(dst + (size_t)x * dst_xstride + f, acc);
  }
}

// Row-owner pass.  grid (ceil(HW/32), heads, B), block 256: warp w owns query frames t = w, w+8, ...
template <int TP, typename QT>
__global__ void __launch_bounds__(TB_WARPS * 32, (TP <= 24 ? 2 : 1)) attn_temporal_bwd_q_kernel(TABwdParams p) {
  pdl_wait();
  extern __shared__ __align__(16) float tb_smem[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int T = p.T, C = p.C, F = p.F, HW = p.HW;
  float* ksm = tb_smem;                              // [T][8][33]
  float* vsm = ksm + (size_t)T * TB_FC * TB_LD;      // [T][8][33]
  float* wbase = vsm + (size_t)T * TB_FC * TB_LD + (size_t)w * (3 * T * TB_FC + T * TB_LD + TB_FC * TB_LD);
  float* rk = wbase;                 // [T][8]  Rk[t, s, chunk]
  float* rq = rk + T * TB_FC;        // [T][8]  Rq[s, t, chunk]
  float* rv = rq + T * TB_FC;        // [T][8]  Rv[t, s, chunk]
  float* dsw = rv + T * TB_FC;       // [T][33] dS[s][px]
  float* qw = dsw + T * TB_LD;       // [8][33] q[f][px]
  // one CTA per (32 pixels, head, video, round of 8 query frames): the rounds are independent, and on the small feature maps
  // (8x8: two pixel blocks) they are the only parallelism there is
  const int NW = blockDim.x >> 5;  // frames per CTA
  const int rounds = (T + NW - 1) / NW;
  const int px0 = blockIdx.x * 32, h = blockIdx.y, b = blockIdx.z / rounds;
  const int px = min(px0 + lane, HW - 1);
  const bool px_ok = px0 + lane < HW;
  const QT* qkv = reinterpret_cast<const QT*>(p.qkv);
  const QT* outp = reinterpret_cast<const QT*>(p.out);
  const QT* dout = reinterpret_cast<const QT*>(p.dout);
  QT* dqkv = reinterpret_cast<QT*>(p.dqkv);
  const size_t tok = (size_t)3 * C;
  const float* maskb = p.mask ? p.mask + (size_t)b * T : nullptr;
  {
    const int rd = blockIdx.z - b * rounds;
    const int t_raw = rd * NW + w;
    const bool act = t_raw < T;
    const int t = act ? t_raw : 0;
    const size_t row = (size_t)(b * T + t) * HW + px;
    float S[TP], dP[TP];
#pragma unroll
    for (int s = 0; s < TP; ++s) { S[s] = 0.f; dP[s] = 0.f; }
    float Dt = 0.f;
    for (int f0 = 0; f0 < F; f0 += TB_FC) {
      __syncthreads();
      if (TP >= 32 && blockDim.x == 256) {  // all loads in flight first: pays for T > 24 (measured: cfg5 10.4 -> 8.8 ms; T = 20 got slower)
        tb_stage2<(TP * 64 + 255) / 256, QT>(ksm, qkv, tok, C + h * F + f0, vsm, qkv, tok, 2 * C + h * F + f0, b, T, HW, px0);
      } else {
        tb_stage(ksm, qkv, tok, b, T, HW, px0, C + h * F + f0);
        tb_stage(vsm, qkv, tok, b, T, HW, px0, 2 * C + h * F + f0);
      }
      if constexpr (TP < 32) {
        for (int i = lane; i < T * TB_FC; i += 32) {
          const int s = i / TB_FC, f = i - s * TB_FC;
          rk[i] = __ldg(p.Rk + (((size_t)(b * T + t) * T + s) * C + h * F + f0 + f));
          rq[i] = __ldg(p.Rq + (((size_t)(b * T + s) * T + t) * C + h * F + f0 + f));
          rv[i] = __ldg(p.Rv + (((size_t)(b * T + t) * T + s) * C + h * F + f0 + f));
        }
      } else {
        constexpr int NR = (TP * TB_FC + 31) / 32;
        float r1[NR], r2[NR], r3[NR];
#pragma unroll
        for (int j = 0; j < NR; ++j) {
          const int i = lane + 32 * j;
          if (i < T * TB_FC) {
            const int s = i / TB_FC, f = i - s * TB_FC;
            r1[j] = __ldg(p.Rk + (((size_t)(b * T + t) * T + s) * C + h * F + f0 + f));
            r2[j] = __ldg(p.Rq + (((size_t)(b * T + s) * T + t) * C + h * F + f0 + f));
            r3[j] = __ldg(p.Rv + (((size_t)(b * T + t) * T + s) * C + h * F + f0 + f));
          }
        }
#pragma unroll
        for (int j = 0; j < NR; ++j) {
          const int i = lane + 32 * j;
          if (i < T * TB_FC) { rk[i] = r1[j]; rq[i] = r2[j]; rv[i] = r3[j]; }
        }
      }
      float q[TB_FC], dO[TB_FC];
      {
        const float4 a = OpType<QT>::load4(qkv + row * tok + h * F + f0), c = OpType<QT>::load4(qkv + row * tok + h * F + f0 + 4);
        q[0] = a.x; q[1] = a.y; q[2] = a.z; q[3] = a.w; q[4] = c.x; q[5] = c.y; q[6] = c.z; q[7] = c.w;
        const float4 d0 = OpType<QT>::load4(dout + row * C + h * F + f0), d1 = OpType<QT>::load4(dout + row * C + h * F + f0 + 4);
        dO[0] = d0.x; dO[1] = d0.y; dO[2] = d0.z; dO[3] = d0.w; dO[4] = d1.x; dO[5] = d1.y; dO[6] = d1.z; dO[7] = d1.w;
        const float4 o0 = OpType<QT>::load4(outp + row * C + h * F + f0), o1 = OpType<QT>::load4(outp + row * C + h * F + f0 + 4);
        Dt += dO[0] * o0.x + dO[1] * o0.y + dO[2] * o0.z + dO[3] * o0.w + dO[4] * o1.x + dO[5] * o1.y + dO[6] * o1.z + dO[7] * o1.w;
      }
      __syncthreads();
#pragma unroll
      for (int s = 0; s < TP; ++s) {
        if (s < T) {
          float a0 = S[s], a1 = 0.f, a2 = dP[s];
#pragma unroll
          for (int f = 0; f < TB_FC; ++f) {
            const float kk = ksm[(size_t)(s * TB_FC + f) * TB_LD + lane];
            const float vv = vsm[(size_t)(s * TB_FC + f) * TB_LD + lane];
            a0 = fmaf(q[f], kk + rk[s * TB_FC + f], a0);
            a1 = fmaf(kk, rq[s * TB_FC + f], a1);
            a2 = fmaf(dO[f], vv + rv[s * TB_FC + f], a2);
          }
          S[s] = a0 + a1;
          dP[s] = a2;
        }
      }
    }
    // masked softmax, log-sum-exp, dS (kept in S[])
    const bool gt = maskb ? maskb[t] > 0.5f : true;
    float mx = -INFINITY;
#pragma unroll
    for (int s = 0; s < TP; ++s)
      if (s < T) {
        const bool ok = maskb ? ((maskb[s] > 0.5f) == gt) : true;
        S[s] = ok ? S[s] * p.scale : -INFINITY;
        mx = fmaxf(mx, S[s]);
      }
    float sum = 0.f;
#pragma unroll
    for (int s = 0; s < TP; ++s)
      if (s < T) {
        S[s] = expf(S[s] - mx);
        sum += S[s];
      }
    const float inv = 1.f / sum;
    const float lse = mx + logf(sum);
    __syncwarp();
#pragma unroll
    for (int s = 0; s < TP; ++s)
      if (s < T) {
        const float ds = (act && px_ok) ? S[s] * inv * (dP[s] - Dt) * p.scale : 0.f;
        S[s] = ds;
        dsw[s * TB_LD + lane] = ds;
      }
    if (act && px_ok) {
      const size_t si = (((size_t)b * p.heads + h) * T + t) * HW + px;
      p.lse[si] = lse;
      p.dsum[si] = Dt;
    }
    // dq and dRk
    for (int f0 = 0; f0 < F; f0 += TB_FC) {
      __syncthreads();
      if (TP >= 32 && blockDim.x == 256) {  // all loads in flight first: pays for T > 24 (measured: cfg5 10.4 -> 8.8 ms; T = 20 got slower)
        tb_stage2<(TP * 64 + 255) / 256, QT>(ksm, qkv, tok, C + h * F + f0, nullptr, qkv, tok, 0, b, T, HW, px0);
      } else {
        tb_stage(ksm, qkv, tok, b, T, HW, px0, C + h * F + f0);
      }
      if constexpr (TP < 32) {
        for (int i = lane; i < T * TB_FC; i += 32) {
          const int s = i / TB_FC, f = i - s * TB_FC;
          rk[i] = __ldg(p.Rk + (((size_t)(b * T + t) * T + s) * C + h * F + f0 + f));
        }
      } else {
        float r1[(TP * TB_FC + 31) / 32];
#pragma unroll
        for (int j = 0; j < (TP * TB_FC + 31) / 32; ++j) {
          const int i = lane + 32 * j;
          if (i < T * TB_FC) r1[j] = __ldg(p.Rk + (((size_t)(b * T + t) * T + i / TB_FC) * C + h * F + f0 + (i % TB_FC)));
        }
#pragma unroll
        for (int j = 0; j < (TP * TB_FC + 31) / 32; ++j) {
          const int i = lane + 32 * j;
          if (i < T * TB_FC) rk[i] = r1[j];
        }
      }
      {
        const float4 a = OpType<QT>::load4(qkv + row * tok + h * F + f0), c = OpType<QT>::load4(qkv + row * tok + h * F + f0 + 4);
        const float qv[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
#pragma unroll
        for (int f = 0; f < TB_FC; ++f) qw[f * TB_LD + lane] = qv[f];
      }
      __syncthreads();
      float dq[TB_FC];
#pragma unroll
      for (int f = 0; f < TB_FC; ++f) dq[f] = 0.f;
#pragma unroll
      for (int s = 0; s < TP; ++s)
        if (s < T) {
#pragma unroll
          for (int f = 0; f < TB_FC; ++f)
            dq[f] = fmaf(S[s], ksm[(size_t)(s * TB_FC + f) * TB_LD + lane] + rk[s * TB_FC + f], dq[f]);
        }
      if (act && px_ok) {
        QT* d = dqkv + row * tok + h * F + f0;
        OpType<QT>::store4(d, make_float4(dq[0], dq[1], dq[2], dq[3]));
        OpType<QT>::store4(d + 4, make_float4(dq[4], dq[5], dq[6], dq[7]));
      }
      if (act) tb_pixel_gemm(dsw, qw, TB_LD, T, lane, p.dRk + ((size_t)(b * T + t) * T) * C + h * F + f0, (size_t)C);
    }
  }
}

// Column-owner pass.  warp w owns key frames s = w, w+8, ...
template <int TP, typename QT>
__global__ void __launch_bounds__(TB_WARPS * 32, (TP <= 24 ? 2 : 1)) attn_temporal_bwd_kv_kernel(TABwdParams p) {
  pdl_wait();
  extern __shared__ __align__(16) float tb_smem[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int T = p.T, C = p.C, F = p.F, HW = p.HW;
  float* qsm = tb_smem;                              // [T][8][33]
  float* dosm = qsm + (size_t)T * TB_FC * TB_LD;     // [T][8][33]
  float* wbase = dosm + (size_t)T * TB_FC * TB_LD + (size_t)w * (3 * T * TB_FC + 2 * T * TB_LD + TB_FC * TB_LD);
  float* rk = wbase;                 // [T][8]  Rk[t, s, chunk]  (t runs, s owned)
  float* rq = rk + T * TB_FC;        // [T][8]  Rq[s, t, chunk]
  float* rv = rq + T * TB_FC;        // [T][8]  Rv[t, s, chunk]
  float* dsw = rv + T * TB_FC;       // [T][33] dS[t][px]
  float* pw = dsw + T * TB_LD;       // [T][33] P[t][px]
  float* kw = pw + T * TB_LD;        // [8][33] k[f][px]
  const int NW = blockDim.x >> 5;  // frames per CTA
  const int rounds = (T + NW - 1) / NW;
  const int px0 = blockIdx.x * 32, h = blockIdx.y, b = blockIdx.z / rounds;
  const int px = min(px0 + lane, HW - 1);
  const bool px_ok = px0 + lane < HW;
  const QT* qkv = reinterpret_cast<const QT*>(p.qkv);
  const QT* dout = reinterpret_cast<const QT*>(p.dout);
  QT* dqkv = reinterpret_cast<QT*>(p.dqkv);
  const size_t tok = (size_t)3 * C;
  const float* maskb = p.mask ? p.mask + (size_t)b * T : nullptr;
  {
    const int rd = blockIdx.z - b * rounds;
    const int s_raw = rd * NW + w;
    const bool act = s_raw < T;
    const int s = act ? s_raw : 0;
    const size_t row = (size_t)(b * T + s) * HW + px;
    float S[TP], dP[TP];
#pragma unroll
    for (int t = 0; t < TP; ++t) { S[t] = 0.f; dP[t] = 0.f; }
    for (int f0 = 0; f0 < F; f0 += TB_FC) {
      __syncthreads();
      if (TP >= 32 && blockDim.x == 256) {  // all loads in flight first: pays for T > 24 (measured: cfg5 10.4 -> 8.8 ms; T = 20 got slower)
        tb_stage2<(TP * 64 + 255) / 256, QT>(qsm, qkv, tok, h * F + f0, dosm, dout, (size_t)C, h * F + f0, b, T, HW, px0);
      } else {
        tb_stage(qsm, qkv, tok, b, T, HW, px0, h * F + f0);
        tb_stage(dosm, dout, (size_t)C, b, T, HW, px0, h * F + f0);
      }
      if constexpr (TP < 32) {
        for (int i = lane; i < T * TB_FC; i += 32) {
          const int t = i / TB_FC, f = i - t * TB_FC;
          rk[i] = __ldg(p.Rk + (((size_t)(b * T + t) * T + s) * C + h * F + f0 + f));
          rq[i] = __ldg(p.Rq + (((size_t)(b * T + s) * T + t) * C + h * F + f0 + f));
          rv[i] = __ldg(p.Rv + (((size_t)(b * T + t) * T + s) * C + h * F + f0 + f));
        }
      } else {
        constexpr int NR = (TP * TB_FC + 31) / 32;
        float r1[NR], r2[NR], r3[NR];
#pragma unroll
        for (int j = 0; j < NR; ++j) {
          const int i = lane + 32 * j;
          if (i < T * TB_FC) {
            const int t = i / TB_FC, f = i - t * TB_FC;
            r1[j] = __ldg(p.Rk + (((size_t)(b * T + t) * T + s) * C + h * F + f0 + f));
            r2[j] = __ldg(p.Rq + (((size_t)(b * T + s) * T + t) * C + h * F + f0 + f));
            r3[j] = __ldg(p.Rv + (((size_t)(b * T + t) * T + s) * C + h * F + f0 + f));
          }
        }
#pragma unroll
        for (int j = 0; j < NR; ++j) {
          const int i = lane + 32 * j;
          if (i < T * TB_FC) { rk[i] = r1[j]; rq[i] = r2[j]; rv[i] = r3[j]; }
        }
      }
      float k[TB_FC], v[TB_FC];
      {
        const float4 a = OpType<QT>::load4(qkv + row * tok + C + h * F + f0), c = OpType<QT>::load4(qkv + row * tok + C + h * F + f0 + 4);
        k[0] = a.x; k[1] = a.y; k[2] = a.z; k[3] = a.w; k[4] = c.x; k[5] = c.y; k[6] = c.z; k[7] = c.w;
        const float4 d0 = OpType<QT>::load4(qkv + row * tok + 2 * C + h * F + f0), d1 = OpType<QT>::load4(qkv + row * tok + 2 * C + h * F + f0 + 4);
        v[0] = d0.x; v[1] = d0.y; v[2] = d0.z; v[3] = d0.w; v[4] = d1.x; v[5] = d1.y; v[6] = d1.z; v[7] = d1.w;
      }
      __syncthreads();
#pragma unroll
      for (int t = 0; t < TP; ++t) {
        if (t < T) {
          float a0 = S[t], a1 = 0.f, a2 = dP[t];
#pragma unroll
          for (int f = 0; f < TB_FC; ++f) {
            const float qq = qsm[(size_t)(t * TB_FC + f) * TB_LD + lane];
            const float dd = dosm[(size_t)(t * TB_FC + f) * TB_LD + lane];
            a0 = fmaf(qq, k[f] + rk[t * TB_FC + f], a0);
            a1 = fmaf(k[f], rq[t * TB_FC + f], a1);
            a2 = fmaf(dd, v[f] + rv[t * TB_FC + f], a2);
          }
          S[t] = a0 + a1;
          dP[t] = a2;
        }
      }
    }
    // P[t] (kept in dP[]) and dS[t] (kept in S[]) for the owned key frame s
    const bool gs = maskb ? maskb[s] > 0.5f : true;
    __syncwarp();
#pragma unroll
    for (int t = 0; t < TP; ++t)
      if (t < T) {
        const bool ok = (maskb ? ((maskb[t] > 0.5f) == gs) : true) && act && px_ok;
        const size_t si = (((size_t)b * p.heads + h) * T + t) * HW + px;
        const float P = ok ? expf(S[t] * p.scale - p.lse[si]) : 0.f;
        const float ds = ok ? P * (dP[t] - p.dsum[si]) * p.scale : 0.f;
        S[t] = ds;
        dP[t] = P;
        dsw[t * TB_LD + lane] = ds;
        pw[t * TB_LD + lane] = P;
      }
    // dk, dv, dRq, dRv
    for (int f0 = 0; f0 < F; f0 += TB_FC) {
      __syncthreads();
      if (TP >= 32 && blockDim.x == 256) {  // all loads in flight first: pays for T > 24 (measured: cfg5 10.4 -> 8.8 ms; T = 20 got slower)
        tb_stage2<(TP * 64 + 255) / 256, QT>(qsm, qkv, tok, h * F + f0, dosm, dout, (size_t)C, h * F + f0, b, T, HW, px0);
      } else {
        tb_stage(qsm, qkv, tok, b, T, HW, px0, h * F + f0);
        tb_stage(dosm, dout, (size_t)C, b, T, HW, px0, h * F + f0);
      }
      for (int i = lane; i < T * TB_FC; i += 32) {
        const int t = i / TB_FC, f = i - t * TB_FC;
        rq[i] = __ldg(p.Rq + (((size_t)(b * T + s) * T + t) * C + h * F + f0 + f));
      }
      {
        const float4 a = OpType<QT>::load4(qkv + row * tok + C + h * F + f0), c = OpType<QT>::load4(qkv + row * tok + C + h * F + f0 + 4);
        const float kv[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
#pragma unroll
        for (int f = 0; f < TB_FC; ++f) kw[f * TB_LD + lane] = kv[f];
      }
      __syncthreads();
      float dk[TB_FC], dv[TB_FC];
#pragma unroll
      for (int f = 0; f < TB_FC; ++f) { dk[f] = 0.f; dv[f] = 0.f; }
#pragma unroll
      for (int t = 0; t < TP; ++t)
        if (t < T) {
#pragma unroll
          for (int f = 0; f < TB_FC; ++f) {
            dk[f] = fmaf(S[t], qsm[(size_t)(t * TB_FC + f) * TB_LD + lane] + rq[t * TB_FC + f], dk[f]);
            dv[f] = fmaf(dP[t], dosm[(size_t)(t * TB_FC + f) * TB_LD + lane], dv[f]);
          }
        }
      if (act && px_ok) {
        QT* d = dqkv + row * tok + C + h * F + f0;
        OpType<QT>::store4(d, make_float4(dk[0], dk[1], dk[2], dk[3]));
        OpType<QT>::store4(d + 4, make_float4(dk[4], dk[5], dk[6], dk[7]));
        QT* e = dqkv + row * tok + 2 * C + h * F + f0;
        OpType<QT>::store4(e, make_float4(dv[0], dv[1], dv[2], dv[3]));
        OpType<QT>::store4(e + 4, make_float4(dv[4], dv[5], dv[6], dv[7]));
      }
      if (act) {
        // dRq[s, t, f] += sum_px dS[t][px] k[f][px]
        tb_pixel_gemm(dsw, kw, TB_LD, T, lane, p.dRq + ((size_t)(b * T + s) * T) * C + h * F + f0, (size_t)C);
        // dRv[t, s, f] += sum_px P[t][px] dO[t][f][px]   (the dO row differs per t: cols = dosm + t*8*33)
        const int f = lane & 7;
        for (int t = lane >> 3; t < T; t += 4) {
          const float* r = pw + t * TB_LD;
          const float* c = dosm + (size_t)(t * TB_FC + f) * TB_LD;
          float acc = 0.f;
#pragma unroll 8
          for (int q = 0; q < 32; ++q) acc = fmaf(r[q], c[q], acc);
          atomicAdd(p.dRv + (((size_t)(b * T + t) * T + s) * C + h * F + f0 + f), acc);
        }
      }
    }
  }
}

}  // namespace fdm

using namespace fdm;

namespace fdm {
int attn_spatial_bwd_tc_launch(const fdm_attn_spatial_bwd_args* a, cudaStream_t st);  // attn_bwd_tc.cu
}

extern "C" int fdm_attn_spatial_bwd(const fdm_attn_spatial_bwd_args* a, void* stream) {
  FDM_REQUIRE(a && a->qkv && a->out && a->dout && a->dqkv && a->lse && a->dsum, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->N > 0 && a->L > 0 && a->heads > 0 && a->C % a->heads == 0, FDM_ERR_BAD_ARG);
  if (a->lse_from_forward) {  // tcgen05 kernels (bf16, forward ran on tcgen05 and saved the log-sum-exp)
    const int rc = attn_spatial_bwd_tc_launch(a, reinterpret_cast<cudaStream_t>(stream));
    if (rc != FDM_ERR_UNSUPPORTED) return rc;
    // shapes the tcgen05 kernels do not take: the CUDA-core kernels below recompute the log-sum-exp into `lse` themselves
  }
  const int F = a->C / a->heads;
  FDM_REQUIRE(F <= 32 * SA_MAXU && F % 4 == 0 && a->C % 4 == 0, FDM_ERR_UNSUPPORTED);
  SABwdParams p{a->qkv, a->out, a->dout, a->dqkv, a->lse, a->dsum, a->N, a->L, a->C, a->heads, F, 1.0f / sqrtf((float)F)};
  const int ld = F + 1;
  const size_t smem_q = ((size_t)2 * SA_KB * ld + 8 * (SA_RPW * 2 * F + SA_RPW * SA_KB)) * sizeof(float);
  const size_t smem_kv = ((size_t)2 * SA_KB * ld + 2 * SA_KB + 8 * (SA_RPW * 2 * F + 2 * SA_RPW * SA_KB)) * sizeof(float);
  dim3 grid((a->L + SA_ROWS - 1) / SA_ROWS, a->heads, a->N);
  FDM_REQUIRE(grid.z <= 65535, FDM_ERR_UNSUPPORTED);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
#define FDM_SA_BWD(QT)                                                                                                  \
  do {                                                                                                                  \
    if (int rc = allow_smem(attn_spatial_bwd_q_kernel<QT>, (int)smem_q)) return rc;                                     \
    if (int rc = allow_smem(attn_spatial_bwd_kv_kernel<QT>, (int)smem_kv)) return rc;                                   \
    fdm::launch(attn_spatial_bwd_q_kernel<QT>, grid, dim3(256), smem_q, st, p);                                         \
    fdm::launch(attn_spatial_bwd_kv_kernel<QT>, grid, dim3(256), smem_kv, st, p);                                       \
  } while (0)
  if (a->dtype == FDM_BF16) FDM_SA_BWD(__nv_bfloat16);
  else FDM_SA_BWD(float);
  return check_launch();
}

template <int TP, typename QT>
static int launch_ta_bwd(const TABwdParams& p, cudaStream_t st) {
  const int T = p.T;
  // frames (warps) per CTA.  Fewer warps per CTA (more CTAs on the small feature maps, where 8-warp CTAs number only 48-192) was
  // measured SLOWER on B200 (cfg3: 3.7 -> 4.9 ms per step): every CTA re-stages all T key/value frames, so halving the frames
  // per CTA doubles the staging traffic and the serial stage -> sync -> compute chain stays as long.
  const size_t smem_q = ((size_t)2 * T * TB_FC * TB_LD + (size_t)TB_WARPS * (3 * T * TB_FC + T * TB_LD + TB_FC * TB_LD)) * sizeof(float);
  const size_t smem_kv = ((size_t)2 * T * TB_FC * TB_LD + (size_t)TB_WARPS * (3 * T * TB_FC + 2 * T * TB_LD + TB_FC * TB_LD)) * sizeof(float);
  dim3 grid((p.HW + 31) / 32, p.heads, p.B * ((T + TB_WARPS - 1) / TB_WARPS));
  if (int rc = allow_smem(attn_temporal_bwd_q_kernel<TP, QT>, (int)smem_q)) return rc;
  if (int rc = allow_smem(attn_temporal_bwd_kv_kernel<TP, QT>, (int)smem_kv)) return rc;
  fdm::launch(attn_temporal_bwd_q_kernel<TP, QT>, grid, dim3(TB_WARPS * 32), smem_q, st, p);
  fdm::launch(attn_temporal_bwd_kv_kernel<TP, QT>, grid, dim3(TB_WARPS * 32), smem_kv, st, p);
  return check_launch();
}

extern "C" int fdm_attn_temporal_bwd(const fdm_attn_temporal_bwd_args* a, void* stream) {
  FDM_REQUIRE(a && a->qkv && a->out && a->dout && a->dqkv && a->Rq && a->Rk && a->Rv && a->dRq && a->dRk && a->dRv && a->lse && a->dsum,
              FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->B > 0 && a->T > 0 && a->HW > 0 && a->heads > 0 && a->C % a->heads == 0, FDM_ERR_BAD_ARG);
  const int F = a->C / a->heads;
  FDM_REQUIRE(F % TB_FC == 0 && a->T <= 40 && a->B <= 8000, FDM_ERR_UNSUPPORTED);
  TABwdParams p{a->qkv, a->out, a->dout, a->Rq, a->Rk, a->Rv, a->mask, a->dqkv, a->dRq, a->dRk, a->dRv, a->lse, a->dsum,
                a->B, a->T, a->HW, a->C, a->heads, F, 1.0f / sqrtf((float)F)};
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
#define FDM_TA_BWD(QT)                                      \
  do {                                                      \
    if (a->T <= 8) return launch_ta_bwd<8, QT>(p, st);      \
    if (a->T <= 16) return launch_ta_bwd<16, QT>(p, st);    \
    if (a->T <= 24) return launch_ta_bwd<24, QT>(p, st);    \
    if (a->T <= 32) return launch_ta_bwd<32, QT>(p, st);    \
    return launch_ta_bwd<40, QT>(p, st);                    \
  } while (0)
  if (a->dtype == FDM_BF16) FDM_TA_BWD(__nv_bfloat16);
  FDM_TA_BWD(float);
}
