// Generic implicit-GEMM convolution / linear on CUDA cores (fp32 accumulate).
//
// This is the exact-fp32 engine (parity mode, 1e-4 contract) and the engine for the shapes the tcgen05
// kernel does not take (stem conv with C_in = 5, head conv with C_out = 3/4, stride-2 convs).
// Reference call sites: nn.Conv2d at unet.py:76,108,155,169,176-180,313,402; nn.Linear at rpe.py:111-112.
//
// GEMM view:  Y[M = N*Ho*Wo, Cout] = sum over (segment, tap, ci) A[pixel(m, tap), ci] * W[tap][ci][co]
// Tile 64 pixels x 64 channels x 16 k, 256 threads, 4x4 outputs per thread.
#include "common.cuh"

namespace fdm {

constexpr int BM = 64, BN = 64, BK = 16, NT = 256;

struct ConvParams {
  const void* a0;
  const float* w0;
  const void* a1;
  const float* w1;
  const float* bias;
  const float* resid;
  float* y_f32;
  void* y_op;
  double* stats;
  int N, Hin, Win, C0, C1, Cout, Ho, Wo;
  int ksize, stride, upsample, out_nchw;
  int M;  // N*Ho*Wo
};

template <typename AT, typename OT>
__global__ void __launch_bounds__(NT) conv_simt_kernel(ConvParams p) {
  pdl_wait();
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN + 4];

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int HWo = p.Ho * p.Wo;

  // A-load mapping: row lm = tid/4 (0..63), 4 consecutive channels at kq = (tid%4)*4
  const int lm = tid >> 2, lk = (tid & 3) * 4;
  const int gm = m0 + lm;
  const bool row_ok = gm < p.M;
  int fn = 0, oh = 0, ow = 0;
  if (row_ok) {
    fn = gm / HWo;
    int r = gm - fn * HWo;
    oh = r / p.Wo;
    ow = r - oh * p.Wo;
  }
  // B-load mapping: k row = tid/16 (0..15), 4 consecutive co at (tid%16)*4
  const int bk = tid >> 4, bn = (tid & 15) * 4;

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int pad = p.ksize >> 1;
  const int Hlim = p.upsample ? p.Hin * 2 : p.Hin, Wlim = p.upsample ? p.Win * 2 : p.Win;

  for (int seg = 0; seg < 2; ++seg) {
    const AT* A = reinterpret_cast<const AT*>(seg == 0 ? p.a0 : p.a1);
    const float* Wt = seg == 0 ? p.w0 : p.w1;
    if (A == nullptr) continue;
    const int Cin = seg == 0 ? p.C0 : p.C1;
    const int ntaps = seg == 0 ? p.ksize * p.ksize : 1;
    for (int tap = 0; tap < ntaps; ++tap) {
      // source pixel of this thread's A row for this tap
      const AT* arow = nullptr;
      if (row_ok) {
        if (seg == 0) {
          int r = tap / p.ksize, s = tap - r * p.ksize;
          int ih = oh * p.stride + r - pad, iw = ow * p.stride + s - pad;
          if (ih >= 0 && ih < Hlim && iw >= 0 && iw < Wlim) {
            if (p.upsample) { ih >>= 1; iw >>= 1; }
            arow = A + ((size_t)(fn * p.Hin + ih) * p.Win + iw) * Cin;
          }
        } else {
          arow = A + (size_t)gm * Cin;
        }
      }
      const float* wtap = Wt + (size_t)tap * Cin * p.Cout;
      for (int c0 = 0; c0 < Cin; c0 += BK) {
        // ---- load A tile (BM x BK) transposed into As[k][m]
        float av[4] = {0.f, 0.f, 0.f, 0.f};
        if (arow != nullptr) {
          int c = c0 + lk;
          if ((Cin & 3) == 0 && c + 3 < Cin) {
            float4 v = OpType<AT>::load4(arow + c);
            av[0] = v.x; av[1] = v.y; av[2] = v.z; av[3] = v.w;
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (c + j < Cin) av[j] = OpType<AT>::load(arow + c + j);
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) As[lk + j][lm] = av[j];
        // ---- load B tile (BK x BN)
        float bv[4] = {0.f, 0.f, 0.f, 0.f};
        {
          int c = c0 + bk;
          if (c < Cin) {
            const float* wr = wtap + (size_t)c * p.Cout + n0 + bn;
            if ((p.Cout & 3) == 0 && n0 + bn + 3 < p.Cout) {
              float4 v = *reinterpret_cast<const float4*>(wr);
              bv[0] = v.x; bv[1] = v.y; bv[2] = v.z; bv[3] = v.w;
            } else {
#pragma unroll
              for (int j = 0; j < 4; ++j)
                if (n0 + bn + j < p.Cout) bv[j] = wr[j];
            }
          }
        }
        *reinterpret_cast<float4*>(&Bs[bk][bn]) = make_float4(bv[0], bv[1], bv[2], bv[3]);
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
          float4 a4 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
          float4 b4 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
          float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
      }
    }
  }

  // ---- epilogue: bias, residual, stores, GroupNorm statistics
  const int cn = n0 + tx * 4;
  float bias[4] = {0.f, 0.f, 0.f, 0.f};
  if (p.bias != nullptr) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (cn + j < p.Cout) bias[j] = p.bias[cn + j];
  }
  float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
  const bool vec_ok = (p.Cout & 3) == 0 && cn + 3 < p.Cout;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int m = m0 + ty * 4 + i;
    if (m >= p.M) continue;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = acc[i][j] + bias[j];
    if (p.resid != nullptr) {
      const float* rr = p.resid + (size_t)m * p.Cout + cn;
      if (vec_ok) {
        float4 r4 = *reinterpret_cast<const float4*>(rr);
        v[0] += r4.x; v[1] += r4.y; v[2] += r4.z; v[3] += r4.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (cn + j < p.Cout) v[j] += rr[j];
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) { s1[j] += v[j]; s2[j] += v[j] * v[j]; }
    if (p.y_f32 != nullptr) {
      if (p.out_nchw) {
        int f = m / HWo, r = m - f * HWo;
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (cn + j < p.Cout) p.y_f32[((size_t)f * p.Cout + cn + j) * HWo + r] = v[j];
      } else if (vec_ok) {
        *reinterpret_cast<float4*>(p.y_f32 + (size_t)m * p.Cout + cn) = make_float4(v[0], v[1], v[2], v[3]);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (cn + j < p.Cout) p.y_f32[(size_t)m * p.Cout + cn + j] = v[j];
      }
    }
    if (p.y_op != nullptr) {
      OT* yo = reinterpret_cast<OT*>(p.y_op) + (size_t)m * p.Cout + cn;
      if (vec_ok) {
        OpType<OT>::store4(yo, make_float4(v[0], v[1], v[2], v[3]));
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (cn + j < p.Cout) OpType<OT>::store(yo + j, v[j]);
      }
    }
  }
  if (p.stats != nullptr) {
    // HW is a multiple of 16 for every feature map of the U-Net, so the 16-row sub-tile q = ty/4 lies in one frame.
    // Fixed-order reduction (no shared-memory atomics): the statistics must not depend on scheduling.
    __syncthreads();  // As/Bs are dead: reuse As as the [16 ty][64 cols] partial buffers
    float* part1 = &As[0][0];            // 16*64 floats <= BK*(BM+4)
    float* part2 = &Bs[0][0];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      part1[ty * BN + tx * 4 + j] = s1[j];
      part2[ty * BN + tx * 4 + j] = s2[j];
    }
    __syncthreads();
    for (int i = tid; i < 4 * BN; i += NT) {
      int qq = i / BN, c = i - qq * BN;
      int m = m0 + qq * 16;
      if (m < p.M && n0 + c < p.Cout) {
        float a1 = 0.f, a2 = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          a1 += part1[(qq * 4 + k) * BN + c];
          a2 += part2[(qq * 4 + k) * BN + c];
        }
        int f = m / HWo;
        double* dst = p.stats + ((size_t)f * p.Cout + n0 + c) * 2;
        atomicAdd(dst, (double)a1);
        atomicAdd(dst + 1, (double)a2);
      }
    }
  }
}

int conv_tc_launch(const fdm_conv_args* a, cudaStream_t st);    // conv_tc.cu (one TMA box per filter tap)
int conv_halo_launch(const fdm_conv_args* a, cudaStream_t st);  // conv_halo.cu (3x3 s1, row-halo reuse, persistent)
int conv_head_launch(const fdm_conv_args* a, cudaStream_t st);  // conv_head.cu (3x3 head conv, <= 4 output channels, NCHW fp32 out)

static int conv_simt_launch(const fdm_conv_args* a, cudaStream_t st) {
  ConvParams p;
  p.a0 = a->a0; p.w0 = reinterpret_cast<const float*>(a->w0);
  p.a1 = a->a1; p.w1 = reinterpret_cast<const float*>(a->w1);
  p.bias = a->bias; p.resid = a->resid; p.y_f32 = a->y_f32; p.y_op = a->y_op; p.stats = reinterpret_cast<double*>(a->stats);
  p.N = a->N; p.Hin = a->Hin; p.Win = a->Win; p.C0 = a->C0; p.C1 = a->a1 ? a->C1 : 0; p.Cout = a->Cout;
  int Hv = a->upsample ? a->Hin * 2 : a->Hin, Wv = a->upsample ? a->Win * 2 : a->Win;
  int pad = a->ksize / 2;
  p.Ho = (Hv + 2 * pad - a->ksize) / a->stride + 1;
  p.Wo = (Wv + 2 * pad - a->ksize) / a->stride + 1;
  p.ksize = a->ksize; p.stride = a->stride; p.upsample = a->upsample; p.out_nchw = a->out_nchw;
  p.M = a->N * p.Ho * p.Wo;
  if (a->stats != nullptr) FDM_REQUIRE((p.Ho * p.Wo) % 16 == 0, FDM_ERR_UNSUPPORTED);
  dim3 grid((p.M + BM - 1) / BM, (p.Cout + BN - 1) / BN);
  bool abf = a->a_dtype == FDM_BF16, obf = a->op_dtype == FDM_BF16;
  if (!abf && !obf) fdm::launch(conv_simt_kernel<float, float>, dim3(grid), dim3(NT), 0, st, p);
  else if (!abf && obf) fdm::launch(conv_simt_kernel<float, __nv_bfloat16>, dim3(grid), dim3(NT), 0, st, p);
  else if (abf && !obf) fdm::launch(conv_simt_kernel<__nv_bfloat16, float>, dim3(grid), dim3(NT), 0, st, p);
  else fdm::launch(conv_simt_kernel<__nv_bfloat16, __nv_bfloat16>, dim3(grid), dim3(NT), 0, st, p);
  return check_launch();
}

}  // namespace fdm

extern "C" int fdm_conv(const fdm_conv_args* a, void* stream) {
  using namespace fdm;
  FDM_REQUIRE(a != nullptr && a->a0 != nullptr && a->w0 != nullptr, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->N > 0 && a->Hin > 0 && a->Win > 0 && a->C0 > 0 && a->Cout > 0, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->ksize == 1 || a->ksize == 3, FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(a->stride == 1 || a->stride == 2, FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(!(a->upsample && a->stride != 1), FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE((a->a1 == nullptr) == (a->w1 == nullptr), FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->y_f32 != nullptr || a->y_op != nullptr, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(!(a->out_nchw && a->y_f32 == nullptr), FDM_ERR_BAD_ARG);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (a->engine == FDM_CONV_TC) {
    // the halo kernel also has a pointwise mode, but measured slower than the per-tap kernel for the 1x1 qkv / proj_out
    // linears on B200 (35 vs 28 us, 30 vs 17 us: two short K stages cannot amortise the persistent pipeline) -> 3x3 only
    // — but with >= 4 K chunks (Cin >= 256: the wide models' qkv / proj_out) it wins: 43.6 -> 29.2 us for 384 -> 1152 at 16x16
    if (a->out_nchw && a->ksize == 3) {
      const int rh = conv_head_launch(a, st);
      if (rh != FDM_ERR_UNSUPPORTED) return rh;
    }
    const int rc = (a->ksize == 3 || a->C0 >= 256) ? conv_halo_launch(a, st) : FDM_ERR_UNSUPPORTED;
    return rc == FDM_ERR_UNSUPPORTED ? conv_tc_launch(a, st) : rc;
  }
  if (a->engine == FDM_CONV_TC_TAP) return conv_tc_launch(a, st);
  FDM_REQUIRE(a->engine == FDM_CONV_SIMT, FDM_ERR_BAD_ARG);
  FDM_REQUIRE(a->resid_norm == 0, FDM_ERR_UNSUPPORTED);
  return conv_simt_launch(a, st);
}
