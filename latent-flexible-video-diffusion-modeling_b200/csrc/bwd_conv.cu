// Convolution / linear WEIGHT gradient and bias gradient (cudnn_convolution_backward_weight / addmm backward at the
// nn.Conv2d sites unet.py:76,108,155,169,176-180,313,402 and nn.Linear sites rpe.py:14,111-112).
//
// GEMM view per filter tap:  dW_tap[ci][co] = sum over output pixels m of  A[pixel(m, tap)][ci] * dY[m][co]
// i.e. M = Cin, N = Cout, K = N*Ho*Wo pixels.  K is split over CTAs into fp32 partials, reduced in a fixed order by a second
// kernel that also writes PyTorch's [co][ci][kh][kw] layout (deterministic; no atomics).
// Engine FDM_CONV_SIMT (this file): CUDA cores, fp32 accumulate, any dtype / shape.  Engine FDM_CONV_TC: wgrad_tc.cu.
#include "common.cuh"

namespace fdm {

// wgrad_tc.cu: tcgen05 engine; FDM_ERR_UNSUPPORTED for shapes / dtypes it does not take (the caller then runs the CUDA-core kernel)
int conv_wgrad_tc(const fdm_conv_wgrad_args* a, float* part, int* splits_out, cudaStream_t st);
size_t conv_wgrad_tc_partial_bytes(const fdm_conv_wgrad_args* a);

constexpr int WG_BM = 64, WG_BN = 64, WG_BK = 16, WG_NT = 256;

struct WgradParams {
  const void* a; const void* dy; float* part;
  int N, Hin, Win, C, Cout, Ho, Wo, ksize, stride;
  long long M;        // output pixels
  long long chunk;    // pixels per split
  int ci_tiles;
};

template <typename AT, typename DT>
__global__ void __launch_bounds__(WG_NT) wgrad_simt_kernel(WgradParams p) {
  pdl_wait();
  __shared__ __align__(16) float As[WG_BK][WG_BM + 4];
  __shared__ __align__(16) float Bs[WG_BK][WG_BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int ci0 = (blockIdx.x % p.ci_tiles) * WG_BM, co0 = (blockIdx.x / p.ci_tiles) * WG_BN;
  const int tap = blockIdx.y, taps = p.ksize * p.ksize;
  const int r = tap / p.ksize, s = tap - r * p.ksize, pad = p.ksize >> 1;
  const long long m_begin = (long long)blockIdx.z * p.chunk;
  const long long m_end = m_begin + p.chunk < p.M ? m_begin + p.chunk : p.M;
  const int HWo = p.Ho * p.Wo;
  const AT* A = reinterpret_cast<const AT*>(p.a);
  const DT* DY = reinterpret_cast<const DT*>(p.dy);
  // load mapping: pixel row lp = tid / 16 (0..15), 4 consecutive channels at (tid % 16) * 4
  const int lp = tid >> 4, lc = (tid & 15) * 4;

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (long long m0 = m_begin; m0 < m_end; m0 += WG_BK) {
    const long long m = m0 + lp;
    float av[4] = {0.f, 0.f, 0.f, 0.f}, bv[4] = {0.f, 0.f, 0.f, 0.f};
    if (m < m_end) {
      const int fn = (int)(m / HWo);
      const int rem = (int)(m - (long long)fn * HWo);
      const int oh = rem / p.Wo, ow = rem - oh * p.Wo;
      const int ih = oh * p.stride + r - pad, iw = ow * p.stride + s - pad;
      if (ih >= 0 && ih < p.Hin && iw >= 0 && iw < p.Win) {
        const AT* arow = A + ((size_t)(fn * p.Hin + ih) * p.Win + iw) * p.C;
        const int c = ci0 + lc;
        if ((p.C & 3) == 0 && c + 3 < p.C) {
          const float4 v = OpType<AT>::load4(arow + c);
          av[0] = v.x; av[1] = v.y; av[2] = v.z; av[3] = v.w;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (c + j < p.C) av[j] = OpType<AT>::load(arow + c + j);
        }
      }
      const DT* drow = DY + (size_t)m * p.Cout;
      const int c = co0 + lc;
      if ((p.Cout & 3) == 0 && c + 3 < p.Cout) {
        const float4 v = OpType<DT>::load4(drow + c);
        bv[0] = v.x; bv[1] = v.y; bv[2] = v.z; bv[3] = v.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (c + j < p.Cout) bv[j] = OpType<DT>::load(drow + c + j);
      }
    }
    *reinterpret_cast<float4*>(&As[lp][lc]) = make_float4(av[0], av[1], av[2], av[3]);
    *reinterpret_cast<float4*>(&Bs[lp][lc]) = make_float4(bv[0], bv[1], bv[2], bv[3]);
    __syncthreads();
#pragma unroll
    for (int k = 0; k < WG_BK; ++k) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  // partial [split][tap][ci][co]
  float* out = p.part + ((size_t)blockIdx.z * taps + tap) * p.C * p.Cout;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int ci = ci0 + ty * 4 + i;
    if (ci >= p.C) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int co = co0 + tx * 4 + j;
      if (co < p.Cout) out[(size_t)ci * p.Cout + co] = acc[i][j];
    }
  }
}

// ---- skinny layers: stem (<= 8 input channels) and head (<= 8 output channels).  The 64x64 tile above would be >= 87 % zeros
// there and, with so few (ci, co) tiles, leaves the split-K CTAs walking ~20k pixels each (measured 4.5 ms per launch on the
// 128-px model).  Here one thread owns a channel of the WIDE side (coalesced global reads) and keeps all taps x narrow-side
// channels in registers; the narrow side is a warp-uniform (broadcast) load.  grid (ceil(wide/128), splits), block 128.
constexpr int WG_NARROW = 8;

template <typename AT, typename DT>
__global__ void __launch_bounds__(128) wgrad_narrow_in_kernel(WgradParams p) {
  pdl_wait();
  const int co = blockIdx.x * 128 + threadIdx.x;
  const bool ok = co < p.Cout;
  const int taps = p.ksize * p.ksize, pad = p.ksize >> 1, HWo = p.Ho * p.Wo;
  const long long m_begin = (long long)blockIdx.y * p.chunk;
  const long long m_end = m_begin + p.chunk < p.M ? m_begin + p.chunk : p.M;
  const AT* A = reinterpret_cast<const AT*>(p.a);
  const DT* DY = reinterpret_cast<const DT*>(p.dy);
  float acc[9][WG_NARROW];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int c = 0; c < WG_NARROW; ++c) acc[t][c] = 0.f;
  int fn = (int)(m_begin / HWo);
  int rem = (int)(m_begin - (long long)fn * HWo);
  int oh = rem / p.Wo, ow = rem - oh * p.Wo;
  for (long long m = m_begin; m < m_end; ++m) {
    const float dy = ok ? OpType<DT>::load(DY + (size_t)m * p.Cout + co) : 0.f;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      if (t < taps) {
        const int r = t / p.ksize, s = t - r * p.ksize;
        const int ih = oh * p.stride + r - pad, iw = ow * p.stride + s - pad;
        if (ih >= 0 && ih < p.Hin && iw >= 0 && iw < p.Win) {  // warp-uniform branch
          const AT* arow = A + ((size_t)(fn * p.Hin + ih) * p.Win + iw) * p.C;
          if (sizeof(AT) == 2 && p.C == 8) {
            const uint4 u = __ldg(reinterpret_cast<const uint4*>(arow));
            const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              acc[t][2 * c] = fmaf(dy, __uint_as_float(w[c] << 16), acc[t][2 * c]);
              acc[t][2 * c + 1] = fmaf(dy, __uint_as_float(w[c] & 0xffff0000u), acc[t][2 * c + 1]);
            }
          } else {
#pragma unroll
            for (int c = 0; c < WG_NARROW; ++c)
              if (c < p.C) acc[t][c] = fmaf(dy, OpType<AT>::load(arow + c), acc[t][c]);
          }
        }
      }
    }
    if (++ow == p.Wo) { ow = 0; if (++oh == p.Ho) { oh = 0; ++fn; } }
  }
  if (!ok) return;
  float* out = p.part + (size_t)blockIdx.y * taps * p.C * p.Cout;
#pragma unroll
  for (int t = 0; t < 9; ++t)
    if (t < taps) {
#pragma unroll
      for (int c = 0; c < WG_NARROW; ++c)
        if (c < p.C) out[((size_t)t * p.C + c) * p.Cout + co] = acc[t][c];
    }
}

template <typename AT, typename DT>
__global__ void __launch_bounds__(128) wgrad_narrow_out_kernel(WgradParams p) {
  pdl_wait();
  const int ci = blockIdx.x * 128 + threadIdx.x;
  const bool ok = ci < p.C;
  const int taps = p.ksize * p.ksize, pad = p.ksize >> 1, HWo = p.Ho * p.Wo;
  const long long m_begin = (long long)blockIdx.y * p.chunk;
  const long long m_end = m_begin + p.chunk < p.M ? m_begin + p.chunk : p.M;
  const AT* A = reinterpret_cast<const AT*>(p.a);
  const DT* DY = reinterpret_cast<const DT*>(p.dy);
  float acc[9][WG_NARROW];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int c = 0; c < WG_NARROW; ++c) acc[t][c] = 0.f;
  int fn = (int)(m_begin / HWo);
  int rem = (int)(m_begin - (long long)fn * HWo);
  int oh = rem / p.Wo, ow = rem - oh * p.Wo;
  for (long long m = m_begin; m < m_end; ++m) {
    float dy[WG_NARROW];
#pragma unroll
    for (int c = 0; c < WG_NARROW; ++c) dy[c] = c < p.Cout ? OpType<DT>::load(DY + (size_t)m * p.Cout + c) : 0.f;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      if (t < taps) {
        const int r = t / p.ksize, s = t - r * p.ksize;
        const int ih = oh * p.stride + r - pad, iw = ow * p.stride + s - pad;
        if (ih >= 0 && ih < p.Hin && iw >= 0 && iw < p.Win) {
          const float x = ok ? OpType<AT>::load(A + ((size_t)(fn * p.Hin + ih) * p.Win + iw) * p.C + ci) : 0.f;
#pragma unroll
          for (int c = 0; c < WG_NARROW; ++c) acc[t][c] = fmaf(x, dy[c], acc[t][c]);
        }
      }
    }
    if (++ow == p.Wo) { ow = 0; if (++oh == p.Ho) { oh = 0; ++fn; } }
  }
  if (!ok) return;
  float* out = p.part + (size_t)blockIdx.y * taps * p.C * p.Cout;
#pragma unroll
  for (int t = 0; t < 9; ++t)
    if (t < taps) {
#pragma unroll
      for (int c = 0; c < WG_NARROW; ++c)
        if (c < p.Cout) out[((size_t)t * p.C + ci) * p.Cout + c] = acc[t][c];
    }
}

// dw[co][ci < Cw][kh][kw] = sum_split part[split][tap = kh*k+kw][ci][co]
__global__ void wgrad_reduce_kernel(const float* __restrict__ part, float* __restrict__ dw, int splits, int taps, int C, int Cw,
                                    int Cout) {
  pdl_wait();
  const long long total = (long long)taps * Cw * Cout;
  const size_t sstride = (size_t)taps * C * Cout;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int co = (int)(i % Cout);
    const long long r = i / Cout;
    const int ci = (int)(r % Cw), tap = (int)(r / Cw);
    const float* src = part + ((size_t)tap * C + ci) * Cout + co;
    // fixed summation order, four independent loads in flight (a serial chain of `splits` DRAM latencies otherwise)
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int k = 0;
    for (; k + 7 < splits; k += 8) {  // eight loads in flight
      const float a0 = src[k * sstride], a1 = src[(k + 1) * sstride], a2 = src[(k + 2) * sstride], a3 = src[(k + 3) * sstride];
      const float a4 = src[(k + 4) * sstride], a5 = src[(k + 5) * sstride], a6 = src[(k + 6) * sstride], a7 = src[(k + 7) * sstride];
      s0 += a0; s1 += a1; s2 += a2; s3 += a3;
      s0 += a4; s1 += a5; s2 += a6; s3 += a7;
    }
    for (; k + 3 < splits; k += 4) {
      s0 += src[k * sstride];
      s1 += src[(k + 1) * sstride];
      s2 += src[(k + 2) * sstride];
      s3 += src[(k + 3) * sstride];
    }
    for (; k < splits; ++k) s0 += src[k * sstride];
    dw[((size_t)co * Cw + ci) * taps + tap] = (s0 + s1) + (s2 + s3);
  }
}

// column sums of dy [rows][C]: stage 1 -> part[block][C], stage 2 -> out (and out2).  C % 4 == 0: a thread owns 4 columns and
// every (256 / (C/4))-th row of the block's range (128/64-bit loads, all lanes busy for any C); other C: one column per thread.
template <typename DT>
__global__ void __launch_bounds__(256) colsum_kernel(const DT* __restrict__ x, float* __restrict__ part, long long rows, int C,
                                                     long long rows_per_block) {
  pdl_wait();
  __shared__ float4 cs_red[256];
  const long long r0 = (long long)blockIdx.x * rows_per_block;
  const long long r1 = r0 + rows_per_block < rows ? r0 + rows_per_block : rows;
  if ((C & 3) == 0) {
    // blockIdx.y walks column chunks of 1024 (qkv gradients have 3C = 1152..1536 columns)
    const int c0 = blockIdx.y * 1024;
    const int quads = min(1024, C - c0) / 4;
    const int q = threadIdx.x % quads, rl = threadIdx.x / quads, nrl = 256 / quads;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    const DT* xc = x + c0 + q * 4;
    if (rl < nrl) {
      long long r = r0 + rl;
      for (; r + 3 * nrl < r1; r += 4 * nrl) {  // four independent loads in flight
        const float4 a = OpType<DT>::load4(xc + (size_t)r * C), b = OpType<DT>::load4(xc + (size_t)(r + nrl) * C);
        const float4 c = OpType<DT>::load4(xc + (size_t)(r + 2 * nrl) * C), d = OpType<DT>::load4(xc + (size_t)(r + 3 * nrl) * C);
        s.x += (a.x + b.x) + (c.x + d.x); s.y += (a.y + b.y) + (c.y + d.y);
        s.z += (a.z + b.z) + (c.z + d.z); s.w += (a.w + b.w) + (c.w + d.w);
      }
      for (; r < r1; r += nrl) {
        const float4 a = OpType<DT>::load4(xc + (size_t)r * C);
        s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
      }
    }
    cs_red[threadIdx.x] = s;
    __syncthreads();
    if (rl == 0) {
      for (int k = 1; k < nrl; ++k) {
        const float4 o = cs_red[k * quads + q];
        s.x += o.x; s.y += o.y; s.z += o.z; s.w += o.w;
      }
      *reinterpret_cast<float4*>(part + (size_t)blockIdx.x * C + c0 + q * 4) = s;
    }
    return;
  }
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s = 0.f;
    for (long long r = r0; r < r1; ++r) s += OpType<DT>::load(x + (size_t)r * C + c);
    part[(size_t)blockIdx.x * C + c] = s;
  }
}
__global__ void colsum_final_kernel(const float* __restrict__ part, float* __restrict__ out, float* __restrict__ out2, int blocks,
                                    int C) {
  pdl_wait();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = 0.f;
  for (int b = 0; b < blocks; ++b) s += part[(size_t)b * C + c];
  if (out != nullptr) out[c] = s;
  if (out2 != nullptr) out2[c] = s;
}

struct WgradGeom {
  int Ho, Wo, taps, splits, ci_tiles, co_tiles, cs_blocks, narrow;
  long long M, chunk, cs_rows;
  size_t part_bytes, cs_bytes;
};

static inline WgradGeom wgrad_geom(const fdm_conv_wgrad_args* a) {
  WgradGeom g;
  const int pad = a->ksize / 2;
  g.Ho = (a->Hin + 2 * pad - a->ksize) / a->stride + 1;
  g.Wo = (a->Win + 2 * pad - a->ksize) / a->stride + 1;
  g.taps = a->ksize * a->ksize;
  g.M = (long long)a->N * g.Ho * g.Wo;
  g.ci_tiles = (a->C + WG_BM - 1) / WG_BM;
  g.co_tiles = (a->Cout + WG_BN - 1) / WG_BN;
  const long long base = (long long)g.ci_tiles * g.co_tiles * g.taps;
  long long want = (148LL * 4 + base - 1) / base;  // ~4 CTAs per SM in total
  const long long max_splits = (g.M + 4 * WG_BK - 1) / (4 * WG_BK);  // at least 64 pixels per split
  if (want > max_splits) want = max_splits;
  if (want < 1) want = 1;
  if (want > 1024) want = 1024;
  g.narrow = (a->C <= WG_NARROW && a->Cout >= 32) ? 1 : ((a->Cout <= WG_NARROW && a->C >= 32) ? 2 : 0);
  if (g.narrow) {
    const long long wide_blocks = ((g.narrow == 1 ? a->Cout : a->C) + 127) / 128;
    want = (148LL * 8 + wide_blocks - 1) / wide_blocks;
    if (want > (g.M + 63) / 64) want = (g.M + 63) / 64;
    if (want < 1) want = 1;
    if (want > 4096) want = 4096;
  }
  g.chunk = ((g.M + want - 1) / want + WG_BK - 1) / WG_BK * WG_BK;
  g.splits = (int)((g.M + g.chunk - 1) / g.chunk);
  g.part_bytes = (size_t)g.splits * g.taps * a->C * a->Cout * sizeof(float);
  if (a->engine == FDM_CONV_TC) {  // either engine may end up running: size for the larger partial buffer
    const size_t tcb = conv_wgrad_tc_partial_bytes(a);
    if (tcb > g.part_bytes) g.part_bytes = tcb;
  }
  g.cs_blocks = (int)(g.M / 64 > 592 ? 592 : (g.M / 64 > 0 ? g.M / 64 : 1));
  g.cs_rows = (g.M + g.cs_blocks - 1) / g.cs_blocks;
  g.cs_blocks = (int)((g.M + g.cs_rows - 1) / g.cs_rows);
  g.cs_bytes = (size_t)g.cs_blocks * a->Cout * sizeof(float);
  return g;
}


}  // namespace fdm

using namespace fdm;

extern "C" size_t fdm_conv_wgrad_workspace(const fdm_conv_wgrad_args* a) {
  if (a == nullptr || a->ksize < 1 || a->stride < 1) return 0;
  const WgradGeom g = wgrad_geom(a);
  return ((g.part_bytes + 255) / 256 * 256) + g.cs_bytes + 256;
}

extern "C" int fdm_conv_wgrad(const fdm_conv_wgrad_args* a, void* stream) {
  FDM_REQUIRE(a && a->dy && a->workspace && (a->dw == nullptr || a->a != nullptr), FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->dw != nullptr || a->dbias != nullptr || a->dbias2 != nullptr, FDM_ERR_BAD_ARG);  // dw == NULL: bias gradient only
  FDM_REQUIRE(a->N > 0 && a->C > 0 && a->Cout > 0 && a->Cw > 0 && a->Cw <= a->C, FDM_ERR_BAD_ARG);
  FDM_REQUIRE((a->ksize == 1 || a->ksize == 3) && (a->stride == 1 || a->stride == 2), FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(a->workspace_bytes >= fdm_conv_wgrad_workspace(a), FDM_ERR_BAD_ARG);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const WgradGeom g = wgrad_geom(a);
  float* part = reinterpret_cast<float*>(a->workspace);
  float* cs_part = reinterpret_cast<float*>(reinterpret_cast<char*>(a->workspace) + (g.part_bytes + 255) / 256 * 256);
  int splits = g.splits;
  bool done = a->dw == nullptr;
  if (!done && a->engine == FDM_CONV_TC) {
    const int rc = conv_wgrad_tc(a, part, &splits, st);
    if (rc == FDM_OK) done = true;
    else if (rc != FDM_ERR_UNSUPPORTED) return rc;
  }
  if (!done) {
    WgradParams p;
    p.a = a->a; p.dy = a->dy; p.part = part;
    p.N = a->N; p.Hin = a->Hin; p.Win = a->Win; p.C = a->C; p.Cout = a->Cout; p.Ho = g.Ho; p.Wo = g.Wo;
    p.ksize = a->ksize; p.stride = a->stride; p.M = g.M; p.chunk = g.chunk; p.ci_tiles = g.ci_tiles;
    dim3 grid(g.ci_tiles * g.co_tiles, g.taps, g.splits);
    dim3 block(WG_NT);
    if (g.narrow) {
      grid = dim3(((g.narrow == 1 ? a->Cout : a->C) + 127) / 128, g.splits, 1);
      block = dim3(128);
    }
    FDM_REQUIRE(grid.z <= 65535 && grid.y <= 65535, FDM_ERR_UNSUPPORTED);
    const bool ab = a->a_dtype == FDM_BF16, db = a->dy_dtype == FDM_BF16;
#define FDM_WG_LAUNCH(K)                                                                     \
  do {                                                                                       \
    if (ab && db) fdm::launch(K<__nv_bfloat16, __nv_bfloat16>, grid, block, 0, st, p);       \
    else if (ab) fdm::launch(K<__nv_bfloat16, float>, grid, block, 0, st, p);                \
    else if (db) fdm::launch(K<float, __nv_bfloat16>, grid, block, 0, st, p);                \
    else fdm::launch(K<float, float>, grid, block, 0, st, p);                                \
  } while (0)
    if (g.narrow == 1) FDM_WG_LAUNCH(wgrad_narrow_in_kernel);
    else if (g.narrow == 2) FDM_WG_LAUNCH(wgrad_narrow_out_kernel);
    else FDM_WG_LAUNCH(wgrad_simt_kernel);
  }
  if (a->dw != nullptr) {
    const long long total = (long long)g.taps * a->Cw * a->Cout;
    long long gr = (total + 255) / 256;
    if (gr > 148 * 8) gr = 148 * 8;
    fdm::launch(wgrad_reduce_kernel, dim3((unsigned)gr), dim3(256), 0, st, (const float*)part, a->dw, splits, g.taps, a->C, a->Cw, a->Cout);
  }
  if (a->dbias != nullptr || a->dbias2 != nullptr) {
    if (a->dy_dtype == FDM_BF16)
      fdm::launch(colsum_kernel<__nv_bfloat16>, dim3(g.cs_blocks, (a->Cout + 1023) / 1024), dim3(256), 0, st, (const __nv_bfloat16*)a->dy, cs_part, g.M, a->Cout, g.cs_rows);
    else
      fdm::launch(colsum_kernel<float>, dim3(g.cs_blocks, (a->Cout + 1023) / 1024), dim3(256), 0, st, (const float*)a->dy, cs_part, g.M, a->Cout, g.cs_rows);
    fdm::launch(colsum_final_kernel, dim3((a->Cout + 127) / 128), dim3(128), 0, st, (const float*)cs_part, a->dbias, a->dbias2, g.cs_blocks, a->Cout);
  }
  return check_launch();
}
