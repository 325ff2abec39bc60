// Implicit-GEMM convolution / linear on the 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM, operands fed by TMA).
//
// Replaces the cuDNN/cuBLAS call sites nn.Conv2d (unet.py:76,108,155,169,176-180,313,402) and nn.Linear qkv/proj_out
// (rpe.py:111-112) of the reference for bf16 operands.
//
// GEMM view:   Y[m, co] = sum_{tap, ci} A[pixel(m, tap), ci] * W[tap][co][ci]  (+ second K-segment: 1x1 skip conv)
//   m = (frame n, oh, ow) in NHWC order.  One CTA computes a 128-pixel x BN-channel output tile.
//   A tile  : im2col is done by the TMA engine itself — the activation tensor is described as a 4-D tensor
//             (C, W, H, N) and the 128 pixels of an M tile form a box (64 ch, Wbox, Hbox, Nbox); tap (r,s) is the same
//             box shifted by (s-pad, r-pad), out-of-bounds rows/columns are zero-filled by the hardware (= padding).
//             Stride-2 convs use the tensor map's elementStrides (traversal stride 2 in W and H).
//   B tile  : weights pre-packed [tap][co_pad][ci_pad] bf16 (K-major), box (64 ci, BN co, 1 tap).
//   Both land in shared memory in the canonical 128-byte-swizzled K-major layout that tcgen05.mma reads directly.
//   Pipeline: warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane), warps 2..5 = epilogue
//             (TMEM -> registers -> padded smem staging -> coalesced bias/residual/store/GroupNorm-statistics).
//   The staging buffer aliases the operand ring (all MMAs have retired when the epilogue starts; one tile per CTA),
//   so two CTAs fit per SM and one CTA's epilogue overlaps the other's main loop.
#include "tc_common.cuh"
#include <mutex>

namespace fdm {

constexpr int TC_BM = 128;
constexpr int TC_BK = 64;          // bf16 elements per K chunk = 128 bytes = one swizzle row
constexpr int TC_THREADS = 192;    // 6 warps
constexpr int A_TILE_BYTES = TC_BM * TC_BK * 2;

struct TcParams {
  const float* bias;
  const float* resid;
  float* y_f32;
  __nv_bfloat16* y_op;
  double* stats;
  int M, HWo, Wo, Ho, Cout;
  int wbox, hbox, nbox;  // output-pixel geometry of an M tile
  int taps, ksize, pad, stride;
  int kchunks0, kchunks1;
  int klast0, klast1;  // 16-wide k-steps actually issued in the last 64-channel chunk of each K segment
  int out_nchw;
  int stages;
  int nr;           // filter rows grouped into one pipeline stage: 1, or 3 (one TMA box of weights per filter column)
  int a_slot;       // bytes of the A region of a stage = nr * 16 KB
  int stage_bytes;  // nr * (16 KB + BN * 128)
  // residual = GroupNorm of `resid` recomputed here (0: plain residual; 2: temporal GN from rn_tstats; 3: per-frame GN from rn_stats)
  int resid_norm, rn_T;
  float rn_eps;
  double rn_inv_cnt;  // 1 / (4 * HWo): reciprocal element count of a GroupNorm group, divided on the host
  const float* rn_tstats;
  const double* rn_stats;
  const float* rn_gamma;
  const float* rn_beta;
};

constexpr int TC_MAX_STAGES = 8;
constexpr int TC_STG_ROW = 36;  // floats per staged row (32 columns + 4 pad): conflict-free float4 access

template <int BN>
struct TcSmem {
  static constexpr int B_TILE_BYTES = BN * TC_BK * 2;
  static constexpr int STAGE_BYTES = A_TILE_BYTES + B_TILE_BYTES;
  static constexpr int TMEM_COLS = BN < 32 ? 32 : BN;
  static constexpr int EXTRA_BYTES = 1024;  // alignment slack (the epilogue staging aliases the dead operand ring)
  static_assert(STAGE_BYTES >= 4 * 32 * TC_STG_ROW * 4, "one stage must hold the epilogue staging");
};

// RN: the residual is GroupNorm(resid) recomputed in the epilogue (a separate instantiation: the extra live values cost the plain
// kernel 20-40 registers — its third resident CTA per SM — and 15-35 % when the code was merely predicated; the RN instantiations
// are held to 112 registers so that they keep three CTAs per SM too)
template <int BN, bool RN>
__global__ void __launch_bounds__(TC_THREADS, RN ? 3 : 0) conv_tc_kernel(const __grid_constant__ CUtensorMap ta0,
                                                            const __grid_constant__ CUtensorMap tw0,
                                                            const __grid_constant__ CUtensorMap ta1,
                                                            const __grid_constant__ CUtensorMap tw1, const TcParams p) {
  using S = TcSmem<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t full_bar[TC_MAX_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[TC_MAX_STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar;
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float4 rn_tab[RN ? 4 : 1][2][2][RN ? 32 : 1];  // [epilogue warp][frame half][mul | add][group]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int mt = blockIdx.x, n_off = blockIdx.y * BN;
  const int m0 = mt * TC_BM;
  const int iters0 = (p.taps / p.nr) * p.kchunks0;
  const int iters = iters0 + p.kchunks1;
  const int stages = p.stages;
  constexpr int B_TAP_BYTES = BN * 128;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&ta0) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tw0) : "memory");
    if (p.kchunks1) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&ta1) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tw1) : "memory");
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < stages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(&tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "n"(S::TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_base_slot;
  pdl_wait();  // everything above (barriers, TMEM, tensor-map prefetch) overlapped the previous kernel's tail

  if (warp == 0) {
    // ===================== TMA producer (whole warp converged; one elected lane issues) =====================
    {
      // first output pixel of the tile -> box origin in (w, h, n)
      int w0, h0, n0;
      if (p.nbox > 1) {
        w0 = 0; h0 = 0; n0 = mt * p.nbox;
      } else {
        n0 = m0 / p.HWo;
        int r = m0 - n0 * p.HWo;
        h0 = r / p.Wo;
        w0 = r - h0 * p.Wo;
      }
      for (int it = 0; it < iters; ++it) {
        const int stage = it % stages;
        const uint32_t phase = (it / stages) & 1;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* a_dst = smem + stage * p.stage_bytes;
        uint8_t* b_dst = a_dst + p.a_slot;
        if (elect_one_sync()) {
          if (it < iters0) {
            const int grp = it / p.kchunks0, kc = it - grp * p.kchunks0;
            mbar_expect_tx(&full_bar[stage], p.nr * (A_TILE_BYTES + B_TAP_BYTES));
            if (p.nr == 1) {
              const int s = grp / p.ksize, r = grp - s * p.ksize;  // weights are packed filter-column major: tap = s*k + r
              tma_load_4d(a_dst, &ta0, &full_bar[stage], kc * TC_BK, w0 * p.stride + s - p.pad, h0 * p.stride + r - p.pad, n0);
              tma_load_3d(b_dst, &tw0, &full_bar[stage], kc * TC_BK, n_off, grp);
            } else {
              // grouped stage = one filter column s: three shifted A boxes, ONE weight box covering its three filter rows
              // (a TMA instruction costs ~450 clk + 0.4 clk/row here: 4 instructions per 3 taps instead of 6)
              const int s = grp;
#pragma unroll
              for (int r = 0; r < 3; ++r)
                tma_load_4d(a_dst + r * A_TILE_BYTES, &ta0, &full_bar[stage], kc * TC_BK, w0 * p.stride + s - p.pad,
                            h0 * p.stride + r - p.pad, n0);
              tma_load_3d(b_dst, &tw0, &full_bar[stage], kc * TC_BK, n_off, s * 3);
            }
          } else {
            const int kc = it - iters0;
            mbar_expect_tx(&full_bar[stage], A_TILE_BYTES + B_TAP_BYTES);
            tma_load_4d(a_dst, &ta1, &full_bar[stage], kc * TC_BK, w0, h0, n0);
            tma_load_3d(b_dst, &tw1, &full_bar[stage], kc * TC_BK, n_off, 0);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp converged; one elected lane issues) =====================
    {
      constexpr uint32_t idesc = make_idesc(BN);
      int kc_cnt = 0, stage = 0;
      uint32_t phase = 0;
      for (int it = 0; it < iters; ++it) {
        mbar_wait(&full_bar[stage], phase);
        tcgen05_fence_after();
        const uint32_t a_lo0 = smem_desc_lo(smem_u32(smem + stage * p.stage_bytes));
        const uint32_t b_lo0 = a_lo0 + (p.a_slot >> 4);
        // channels beyond C0/C1 in the last chunk are TMA zero-fill: skip their k-steps
        int nk = TC_BK / 16;
        int rows = 1;
        if (it < iters0) {
          rows = p.nr;
          if (kc_cnt == p.kchunks0 - 1) nk = p.klast0;
          if (++kc_cnt == p.kchunks0) kc_cnt = 0;
        } else if (it == iters - 1) {
          nk = p.klast1;
        }
        // advance 16 bf16 = 32 bytes inside the 128-byte swizzle row: +2 in the (>>4) start-address field
        if (elect_one_sync()) {
        for (int r = 0; r < rows; ++r) {
          const uint32_t a_lo = a_lo0 + r * (A_TILE_BYTES >> 4), b_lo = b_lo0 + r * (B_TAP_BYTES >> 4);
          if (nk == 4) {
            umma_bf16_lo(tmem_base, a_lo, b_lo, idesc, (it | r) != 0);
            umma_bf16_lo(tmem_base, a_lo + 2, b_lo + 2, idesc, 1u);
            umma_bf16_lo(tmem_base, a_lo + 4, b_lo + 4, idesc, 1u);
            umma_bf16_lo(tmem_base, a_lo + 6, b_lo + 6, idesc, 1u);
          } else {
            for (int k = 0; k < nk; ++k) umma_bf16_lo(tmem_base, a_lo + 2 * k, b_lo + 2 * k, idesc, (it | r | k) != 0);
          }
        }
        umma_commit(&empty_bar[stage]);  // frees the smem slot when these MMAs retire
        }
        __syncwarp();
        if (++stage == stages) { stage = 0; phase ^= 1; }
      }
      if (elect_one_sync()) umma_commit(&tmem_full_bar);  // accumulator complete
      __syncwarp();
    }
  } else {
    // ===================== epilogue (warps 2..5) =====================
    // 32-column chunks: TMEM -> registers -> this warp's padded staging slice -> lanes across channels (float4), 4 rows per
    // instruction; the 8 residual loads of a chunk are issued before any is used (memory-level parallelism).
    const int g = warp & 3;  // TMEM lane group this warp may access: lanes [32g, 32g+32)
    // staging aliases the operand ring: every MMA (hence every shared-memory read) has retired once tmem_full fires
    float* stg = reinterpret_cast<float*>(smem) + g * 32 * TC_STG_ROW;
    const int sub = lane >> 3, cq = (lane & 7) * 4;
    const int m_w = m0 + g * 32;  // first row of this warp
    const bool two_frames = p.HWo < 32;  // HWo == 16: rows [0,16) and [16,32) of the warp belong to different frames
    // RN: frame / video of the warp's rows (one integer division per warp instead of two per row and chunk).  Per-frame
    // statistics: lane l computes scale / shift of group l (columns n_off + 4l .. + 3) for the one or two frames of this warp's
    // rows — fp64 arithmetic and a global round trip, done once per warp while the MMAs are still running — into the warp's own
    // slice of a small shared-memory table the chunk loop reads back by column.
    int rn_n[2] = {0, 0}, rn_b[2] = {0, 0};
    if (RN) {
      rn_n[0] = min(m_w, p.M - 1) / p.HWo;
      rn_n[1] = two_frames ? min(m_w + 16, p.M - 1) / p.HWo : rn_n[0];
      rn_b[0] = rn_n[0] / p.rn_T;
      rn_b[1] = rn_n[1] / p.rn_T;
      if (p.resid_norm == 3) {
        const int col = n_off + 4 * lane;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          float4 mu = make_float4(0.f, 0.f, 0.f, 0.f), ad = mu;
          if ((hh == 0 || two_frames) && col < p.Cout && 4 * lane < BN && m_w + hh * 16 < p.M) {
            const float4 gm = __ldg(reinterpret_cast<const float4*>(p.rn_gamma + col));
            const float4 bt = __ldg(reinterpret_cast<const float4*>(p.rn_beta + col));
            const double2* st = reinterpret_cast<const double2*>(p.rn_stats + ((size_t)rn_n[hh] * p.Cout + col) * 2);
            const double2 s0 = st[0], s1_ = st[1], s2_ = st[2], s3 = st[3];
            // fp64 only where it matters (E[x^2] - mean^2); no fp64 division / square root on the epilogue's critical path
            const double mean = (s0.x + s1_.x + s2_.x + s3.x) * p.rn_inv_cnt;
            const double var = fmax((s0.y + s1_.y + s2_.y + s3.y) * p.rn_inv_cnt - mean * mean, 0.0);
            const float mf = (float)mean, rs = rsqrtf((float)var + p.rn_eps);
            mu = make_float4(gm.x * rs, gm.y * rs, gm.z * rs, gm.w * rs);
            ad = make_float4(bt.x - mf * mu.x, bt.y - mf * mu.y, bt.z - mf * mu.z, bt.w - mf * mu.w);
          }
          rn_tab[g][hh][0][lane] = mu;
          rn_tab[g][hh][1][lane] = ad;
        }
        __syncwarp();
      }
    }
    mbar_wait(&tmem_full_bar, 0);
    tcgen05_fence_after();
    // bf16-only outputs without residual / statistics (the qkv linears): each lane owns 32 consecutive channels of its row =
    // 64 contiguous bytes -> packed 16-byte stores straight from the TMEM registers, no shared-memory transpose
    const bool direct = BN >= 32 && p.y_f32 == nullptr && p.y_op != nullptr && p.resid == nullptr && p.stats == nullptr &&
                        !p.out_nchw && (p.Cout & 31) == 0;
#pragma unroll 1
    for (int c = 0; c < BN; c += 32) {
      uint32_t v[32];
      tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(g * 32) << 16) + c, v);
      if (direct) {
        // lane <-> row out of TMEM: pack this lane's 32 channels (64 bytes), transpose through the warp's staging slice (80-byte
        // row pitch: conflict-free 16-byte accesses) and store with 4 lanes per row — every store instruction writes whole
        // 64-byte row segments (8 rows x 64 B) instead of 32 scattered 16-byte pieces (partial-sector writes at the L2)
        uint8_t* sb = reinterpret_cast<uint8_t*>(stg);
        const bool cols_ok = n_off + c < p.Cout;
#pragma unroll
        for (int q = 0; q < 32; q += 8) {
          float4 b0 = make_float4(0.f, 0.f, 0.f, 0.f), b1 = b0;
          if (p.bias != nullptr && cols_ok) {
            b0 = __ldg(reinterpret_cast<const float4*>(p.bias + n_off + c + q));
            b1 = __ldg(reinterpret_cast<const float4*>(p.bias + n_off + c + q + 4));
          }
          __nv_bfloat162 h0 = __floats2bfloat162_rn(__uint_as_float(v[q]) + b0.x, __uint_as_float(v[q + 1]) + b0.y);
          __nv_bfloat162 h1 = __floats2bfloat162_rn(__uint_as_float(v[q + 2]) + b0.z, __uint_as_float(v[q + 3]) + b0.w);
          __nv_bfloat162 h2 = __floats2bfloat162_rn(__uint_as_float(v[q + 4]) + b1.x, __uint_as_float(v[q + 5]) + b1.y);
          __nv_bfloat162 h3 = __floats2bfloat162_rn(__uint_as_float(v[q + 6]) + b1.z, __uint_as_float(v[q + 7]) + b1.w);
          uint4 w;
          w.x = *reinterpret_cast<uint32_t*>(&h0); w.y = *reinterpret_cast<uint32_t*>(&h1);
          w.z = *reinterpret_cast<uint32_t*>(&h2); w.w = *reinterpret_cast<uint32_t*>(&h3);
          *reinterpret_cast<uint4*>(sb + lane * 80 + (q >> 3) * 16) = w;
        }
        __syncwarp();
        if (cols_ok) {
          const int piece = lane & 3;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int row = i * 8 + (lane >> 2);
            const int m = m_w + row;
            if (m < p.M)
              *reinterpret_cast<uint4*>(p.y_op + (size_t)m * p.Cout + n_off + c + piece * 8) =
                  *reinterpret_cast<const uint4*>(sb + row * 80 + piece * 16);
          }
        }
        __syncwarp();
        continue;
      }
#pragma unroll
      for (int q = 0; q < 32; q += 4)
        *reinterpret_cast<float4*>(stg + lane * TC_STG_ROW + q) =
            make_float4(__uint_as_float(v[q]), __uint_as_float(v[q + 1]), __uint_as_float(v[q + 2]), __uint_as_float(v[q + 3]));
      __syncwarp();
      if (p.out_nchw) {
        // narrow head conv (unet.py:402,462-464): eps written as [N][Cout][Ho][Wo] fp32; lane <-> pixel row, few channels
        const int m = m_w + lane;
        if (m < p.M) {
          const int f = m / p.HWo, r = m - f * p.HWo;
          for (int cc = 0; cc < 32 && n_off + c + cc < p.Cout; ++cc) {
            float o = stg[lane * TC_STG_ROW + cc] + (p.bias ? p.bias[n_off + c + cc] : 0.f);
            p.y_f32[((size_t)f * p.Cout + n_off + c + cc) * p.HWo + r] = o;
          }
        }
      } else {
        const int col = n_off + c + cq;
        const bool col_ok = col < p.Cout;  // Cout % 4 == 0
        float4 bias = make_float4(0.f, 0.f, 0.f, 0.f);
        if (col_ok && p.bias != nullptr) bias = __ldg(reinterpret_cast<const float4*>(p.bias + col));
        float4 res[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int m = m_w + i * 4 + sub;
          res[i] = (p.resid != nullptr && col_ok && m < p.M) ? __ldg(reinterpret_cast<const float4*>(p.resid + (size_t)m * p.Cout + col))
                                                             : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (RN && p.resid_norm != 0 && col_ok) {
          // the residual is GroupNorm(resid) (rpe.py:136,173), recomputed from the statistics instead of read from a normalised
          // copy: this lane's 4 channels are one group (Cout = 128)
          if (p.resid_norm == 2) {
            const float4 gm = __ldg(reinterpret_cast<const float4*>(p.rn_gamma + col));
            const float4 bt = __ldg(reinterpret_cast<const float4*>(p.rn_beta + col));
            float2 ms[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int m = m_w + i * 4 + sub;
              const int px = m - rn_n[i >> 2] * p.HWo;
              ms[i] = m < p.M ? __ldg(reinterpret_cast<const float2*>(p.rn_tstats + (((size_t)rn_b[i >> 2] * p.HWo + px) * 32 + (col >> 2)) * 2))
                              : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              res[i].x = (res[i].x - ms[i].x) * ms[i].y * gm.x + bt.x;
              res[i].y = (res[i].y - ms[i].x) * ms[i].y * gm.y + bt.y;
              res[i].z = (res[i].z - ms[i].x) * ms[i].y * gm.z + bt.z;
              res[i].w = (res[i].w - ms[i].x) * ms[i].y * gm.w + bt.w;
            }
          } else {
            const int grp = (c + cq) >> 2;  // this lane's group inside the N tile
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              const float4 mu = rn_tab[g][two_frames ? hh : 0][0][grp], ad = rn_tab[g][two_frames ? hh : 0][1][grp];
#pragma unroll
              for (int i = 4 * hh; i < 4 * hh + 4; ++i) {
                res[i].x = fmaf(res[i].x, mu.x, ad.x);
                res[i].y = fmaf(res[i].y, mu.y, ad.y);
                res[i].z = fmaf(res[i].z, mu.z, ad.z);
                res[i].w = fmaf(res[i].w, mu.w, ad.w);
              }
            }
          }
        }
        float s1[2][4], s2[2][4];
#pragma unroll
        for (int hh = 0; hh < 2; ++hh)
#pragma unroll
          for (int q = 0; q < 4; ++q) s1[hh][q] = s2[hh][q] = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int row = i * 4 + sub;
          const int m = m_w + row;
          const float4 a = *reinterpret_cast<const float4*>(stg + row * TC_STG_ROW + cq);
          const float o[4] = {a.x + bias.x + res[i].x, a.y + bias.y + res[i].y, a.z + bias.z + res[i].z, a.w + bias.w + res[i].w};
          if (m < p.M && col_ok) {
#pragma unroll
            for (int q = 0; q < 4; ++q) { s1[i >> 2][q] += o[q]; s2[i >> 2][q] = fmaf(o[q], o[q], s2[i >> 2][q]); }
            const size_t off = (size_t)m * p.Cout + col;
            if (p.y_f32 != nullptr) *reinterpret_cast<float4*>(p.y_f32 + off) = make_float4(o[0], o[1], o[2], o[3]);
            if (p.y_op != nullptr) OpType<__nv_bfloat16>::store4(p.y_op + off, make_float4(o[0], o[1], o[2], o[3]));
          }
        }
        if (p.stats != nullptr) {
          // combine the 4 row-subgroups (lanes with equal lane%8); one fp64 atomic per (frame, channel, moment) per warp
#pragma unroll
          for (int hh = 0; hh < 2; ++hh)
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              s1[hh][q] += __shfl_xor_sync(0xffffffffu, s1[hh][q], 8);
              s2[hh][q] += __shfl_xor_sync(0xffffffffu, s2[hh][q], 8);
              s1[hh][q] += __shfl_xor_sync(0xffffffffu, s1[hh][q], 16);
              s2[hh][q] += __shfl_xor_sync(0xffffffffu, s2[hh][q], 16);
            }
          if (sub == 0 && col_ok) {
            if (two_frames) {
#pragma unroll
              for (int hh = 0; hh < 2; ++hh) {
                const int mseg = m_w + hh * 16;
                if (mseg < p.M) {
                  double* dst = p.stats + ((size_t)(mseg / p.HWo) * p.Cout + col) * 2;
#pragma unroll
                  for (int q = 0; q < 4; ++q) {
                    atomicAdd(dst + 2 * q, (double)s1[hh][q]);
                    atomicAdd(dst + 2 * q + 1, (double)s2[hh][q]);
                  }
                }
              }
            } else if (m_w < p.M) {
              double* dst = p.stats + ((size_t)(m_w / p.HWo) * p.Cout + col) * 2;
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                atomicAdd(dst + 2 * q, (double)(s1[0][q] + s1[1][q]));
                atomicAdd(dst + 2 * q + 1, (double)(s2[0][q] + s2[1][q]));
              }
            }
          }
        }
      }
      __syncwarp();  // staging slice is overwritten by the next chunk
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(S::TMEM_COLS));
  }
}

// ---------------------------------------------------------------- host side
EncodeTiledFn get_tensormap_encoder() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// activations [N][H][W][C] bf16 as a (C, W, H, N) tensor; box (64, wbox*sw, hbox*sh, nbox) traversed with stride (1, s, s, 1)
static bool encode_act(CUtensorMap* m, const void* ptr, int N, int H, int W, int C, int wbox, int hbox, int nbox, int stride) {
  EncodeTiledFn enc = get_tensormap_encoder();
  if (!enc) return false;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)TC_BK, (cuuint32_t)(wbox * stride), (cuuint32_t)(hbox * stride), (cuuint32_t)nbox};
  cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// weights [taps][co_pad][ci_pad] bf16 as a (ci_pad, co_pad, taps) tensor; box (64, BN, 1)
static bool encode_w(CUtensorMap* m, const void* ptr, int taps, int co_pad, int ci_pad, int bn, int box_taps) {
  EncodeTiledFn enc = get_tensormap_encoder();
  if (!enc) return false;
  cuuint64_t dims[3] = {(cuuint64_t)ci_pad, (cuuint64_t)co_pad, (cuuint64_t)taps};
  cuuint64_t strides[2] = {(cuuint64_t)ci_pad * 2, (cuuint64_t)co_pad * ci_pad * 2};
  cuuint32_t box[3] = {(cuuint32_t)TC_BK, (cuuint32_t)bn, (cuuint32_t)box_taps};
  cuuint32_t estr[3] = {1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int BN, bool RN = false>
static int launch_tc(const CUtensorMap& ta0, const CUtensorMap& tw0, const CUtensorMap& ta1, const CUtensorMap& tw1,
                     TcParams& p, cudaStream_t st) {
  using S = TcSmem<BN>;
  constexpr int SMEM_MAX = (RN ? 216 : 226) * 1024;  // RN: 8.3 KB of static shared memory (the coefficient table)
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] {
    attr_err = cudaFuncSetAttribute(conv_tc_kernel<BN, RN>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_MAX);
  });
  if (attr_err != cudaSuccess) {
    set_last_error(attr_err);
    return FDM_ERR_CUDA;
  }
  dim3 grid((p.M + TC_BM - 1) / TC_BM, (p.Cout + BN - 1) / BN);
  // pipeline depth: a grid that cannot even fill the SMs once is latency-bound -> one CTA per SM with as many operand
  // stages in flight as the K loop has iterations (up to 8); otherwise two CTAs per SM share the shared memory.
  const int budget = (long)grid.x * grid.y <= 148 ? SMEM_MAX : SMEM_MAX / 2;
  p.a_slot = p.nr * A_TILE_BYTES;
  p.stage_bytes = p.nr * S::STAGE_BYTES;
  int stages = (budget - S::EXTRA_BYTES) / p.stage_bytes;
  const int iters = (p.taps / p.nr) * p.kchunks0 + p.kchunks1;
  if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
  if (stages > iters) stages = iters;
  if (stages < 1) return FDM_ERR_UNSUPPORTED;
  p.stages = stages;
  fdm::launch(conv_tc_kernel<BN, RN>, dim3(grid), dim3(TC_THREADS), stages * p.stage_bytes + S::EXTRA_BYTES, st, ta0, tw0, ta1, tw1, p);
  return check_launch();
}

static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

int conv_tc_launch(const fdm_conv_args* a, cudaStream_t st) {
  FDM_REQUIRE(a->a_dtype == FDM_BF16, FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(!a->upsample, FDM_ERR_UNSUPPORTED);
  FDM_REQUIRE(a->C0 % 8 == 0 && (a->a1 == nullptr || a->C1 % 8 == 0), FDM_ERR_UNSUPPORTED);
  if (a->out_nchw) {
    FDM_REQUIRE(a->y_f32 != nullptr && a->y_op == nullptr && a->resid == nullptr && a->stats == nullptr, FDM_ERR_UNSUPPORTED);
  } else {
    FDM_REQUIRE(a->Cout % 4 == 0, FDM_ERR_UNSUPPORTED);
  }
  FDM_REQUIRE(a->y_op == nullptr || a->op_dtype == FDM_BF16, FDM_ERR_UNSUPPORTED);
  const int pad = a->ksize / 2;
  const int Ho = (a->Hin + 2 * pad - a->ksize) / a->stride + 1, Wo = (a->Win + 2 * pad - a->ksize) / a->stride + 1;
  const int HWo = Ho * Wo;
  TcParams p;
  p.bias = a->bias; p.resid = a->resid; p.y_f32 = a->y_f32; p.y_op = reinterpret_cast<__nv_bfloat16*>(a->y_op); p.stats = reinterpret_cast<double*>(a->stats);
  p.M = a->N * HWo; p.HWo = HWo; p.Wo = Wo; p.Ho = Ho; p.Cout = a->Cout;
  // M-tile geometry: 128 consecutive output pixels must form a box in (w, h, n)
  if (Wo >= TC_BM) {
    FDM_REQUIRE(Wo % TC_BM == 0, FDM_ERR_UNSUPPORTED);
    p.wbox = TC_BM; p.hbox = 1; p.nbox = 1;
  } else if (HWo >= TC_BM) {
    FDM_REQUIRE(TC_BM % Wo == 0 && HWo % TC_BM == 0, FDM_ERR_UNSUPPORTED);
    p.wbox = Wo; p.hbox = TC_BM / Wo; p.nbox = 1;
  } else {
    FDM_REQUIRE(TC_BM % HWo == 0, FDM_ERR_UNSUPPORTED);
    p.wbox = Wo; p.hbox = Ho; p.nbox = TC_BM / HWo;
  }
  // GroupNorm statistics are flushed per warp segment: a warp's 32 rows must not straddle frames unevenly
  FDM_REQUIRE(a->stats == nullptr || HWo % 32 == 0 || 32 % HWo == 0, FDM_ERR_UNSUPPORTED);
  p.taps = a->ksize * a->ksize; p.ksize = a->ksize; p.pad = pad; p.stride = a->stride;
  p.kchunks0 = (a->C0 + TC_BK - 1) / TC_BK;
  p.kchunks1 = a->a1 ? (a->C1 + TC_BK - 1) / TC_BK : 0;
  p.klast0 = (a->C0 - (p.kchunks0 - 1) * TC_BK + 15) / 16;
  p.klast1 = a->a1 ? (a->C1 - (p.kchunks1 - 1) * TC_BK + 15) / 16 : 0;
  p.out_nchw = a->out_nchw;
  p.resid_norm = a->resid_norm; p.rn_T = a->rn_T > 0 ? a->rn_T : 1; p.rn_eps = a->rn_eps;
  p.rn_inv_cnt = 1.0 / (4.0 * (double)HWo);
  p.rn_tstats = a->rn_tstats; p.rn_stats = a->rn_stats; p.rn_gamma = a->rn_gamma; p.rn_beta = a->rn_beta;
  if (a->resid_norm != 0) {
    FDM_REQUIRE(a->resid_norm == 2 || a->resid_norm == 3, FDM_ERR_BAD_ARG);
    FDM_REQUIRE(a->resid != nullptr && a->rn_gamma != nullptr && a->rn_beta != nullptr, FDM_ERR_BAD_ARG);
    FDM_REQUIRE(a->resid_norm == 2 ? a->rn_tstats != nullptr : a->rn_stats != nullptr, FDM_ERR_BAD_ARG);
    FDM_REQUIRE(a->Cout == 128 && a->ksize == 1 && !a->out_nchw && (HWo % 32 == 0 || HWo == 16), FDM_ERR_UNSUPPORTED);
  }
  // N tile: as wide as Cout allows, but narrowed while the grid would leave most SMs idle (small feature maps)
  int bn = a->Cout % 128 == 0 ? 128 : (a->Cout >= 64 ? 64 : (a->Cout > 16 ? 32 : 16));
  const int mtiles = (p.M + TC_BM - 1) / TC_BM;
  // (small grids run at the per-SM TMA instruction rate, so more CTAs only help while they land on idle SMs: never exceed 148)
  // (1x1 linears with a short K loop (Cin <= 128: proj_out) are epilogue-bound and light on shared memory — three CTAs per SM are resident —
  //  so they are narrowed up to 3 x 148 CTAs: 8x8 proj_out 10.7 -> 6.2 us with BN = 32; at 16x16 narrower tiles measured slower)
  const int cta_cap = (a->ksize == 1 && a->C0 <= 128 && a->a1 == nullptr) ? 3 * 148 : 148;
  while (bn > 32 && mtiles * ((a->Cout + bn / 2 - 1) / (bn / 2)) <= cta_cap) bn >>= 1;
  const int co_pad = round_up(a->Cout, 16);
  // small grids (one CTA per SM, whole shared memory for the operand ring) run at the TMA INSTRUCTION rate: group the three
  // filter rows of a filter column into one stage so a single weight box serves three taps
  const long ctas = (long)mtiles * ((a->Cout + bn - 1) / bn);
  p.nr = (a->ksize == 3 && ctas <= 148) ? 3 : 1;
  CUtensorMap ta0, tw0, ta1, tw1;
  bool ok = encode_act(&ta0, a->a0, a->N, a->Hin, a->Win, a->C0, p.wbox, p.hbox, p.nbox, a->stride) &&
            encode_w(&tw0, a->w0, p.taps, co_pad, round_up(a->C0, TC_BK), bn, p.nr);
  if (ok && a->a1) {
    ok = encode_act(&ta1, a->a1, a->N, Ho, Wo, a->C1, p.wbox, p.hbox, p.nbox, 1) &&
         encode_w(&tw1, a->w1, 1, co_pad, round_up(a->C1, TC_BK), bn, 1);
  } else {
    ta1 = ta0;
    tw1 = tw0;
  }
  FDM_REQUIRE(ok, FDM_ERR_UNSUPPORTED);
  if (p.resid_norm != 0) {
    if (bn == 128) return launch_tc<128, true>(ta0, tw0, ta1, tw1, p, st);
    if (bn == 64) return launch_tc<64, true>(ta0, tw0, ta1, tw1, p, st);
    return launch_tc<32, true>(ta0, tw0, ta1, tw1, p, st);
  }
  if (bn == 128) return launch_tc<128>(ta0, tw0, ta1, tw1, p, st);
  if (bn == 64) return launch_tc<64>(ta0, tw0, ta1, tw1, p, st);
  if (bn == 32) return launch_tc<32>(ta0, tw0, ta1, tw1, p, st);
  return launch_tc<16>(ta0, tw0, ta1, tw1, p, st);
}

}  // namespace fdm

