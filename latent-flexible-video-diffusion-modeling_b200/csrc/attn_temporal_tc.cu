// Temporal RPE attention on the 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM, operands by TMA).
//
// Reference: RPEAttention._forward, temporal case (rpe.py:133-174), einsums of RPE.forward_qk / forward_v (rpe.py:72-83):
//   S[t,s] = scale * ( q_t.k_s + q_t.Rk[t,s] + k_s.Rq[s,t] )      per (video b, pixel, head)
//   P      = softmax over { s : mask_s == mask_t }                  (two-group mask, rpe.py:156-163)
//   O[t]   = sum_s P[t,s] * ( v_s + Rv[t,s] )
// R*[b,t,s,h,:] depend on (video, frame pair, head) but NOT on the pixel.  That splits the five contractions into two families
// with different GEMM shapes, and each family gets the row order that makes it a dense tensor-core GEMM:
//
//   (A) relative-position terms — for a FIXED frame j they are GEMMs over the pixels:
//         b2[px, s] = Q_j[px, :] . Rk[j, s, :]      b3[px, t] = K_j[px, :] . Rq[j, t, :]      Orv[px, :] = P_j[px, :] . Rv[j, :, :]
//       M = 128 pixels of frame j, N = T (or F), K = F (or T).
//   (B) content terms q.k and P.v — per pixel they are tiny T x T problems.  Rows are ordered (pixel, frame): a 128-row tile holds
//       PL = 128/TP pixels x TP frames, S = Q K^T over the whole tile is ONE 128x128 MMA whose diagonal TP x TP blocks are the
//       per-pixel score matrices (the off-diagonal blocks are wasted tensor work: free at this size), and O = P V with the
//       block-diagonal P written by the softmax threads.
//
//   K1 rpe_bias_kernel   : (A) score terms for every (b, h, frame j): b2[b,h,px,t=j,:] and b3[b,h,px,s=j,:]      (fp32, L2-resident)
//   K2 attn_rows_kernel  : (B): S = QK^T (tcgen05) -> + b2 + b3^T, mask, fp32 softmax from TMEM -> P (bf16) -> O = PV (tcgen05)
//                          also stores the normalised attention weights P[b,h,px,t,:] (consumed by K3; they ARE rpe.py:164's `attn`)
//   K3 rpe_pv_kernel     : (A) value term: out[b,t,px,h,:] += P_t . Rv[t]                                      (tcgen05)
//
// Data never changes layout on the way: the two row orders are two TMA views (tensor maps) of the same [B*T][HW][3C] qkv tensor.
#include "tc_common.cuh"

namespace fdm {

struct TtParams {
  const float* mask;       // [B][T] or nullptr
  __nv_bfloat16* b2;       // [B][heads][HW][T][TS]   q_t . Rk[t,s]      (unscaled; bf16: half the L2 round trip, and K2's tile of both
  __nv_bfloat16* b3;       // [B][heads][HW][T(s)][TS(t)]   k_s . Rq[s,t]  tables shrinks enough for a FOURTH resident CTA per SM)
  __nv_bfloat16* P;        // [B][heads][HW][T][64]   normalised attention weights, zero beyond s >= T
  __nv_bfloat16* out;      // [B*T][HW][C]
  float* attn_mean;        // optional [B*HW][T][T]: += attention weights / heads (attention-map logging, rpe.py:128-130)
  int B, T, HW, C, F, heads;
  int TS;                  // row stride of b2 / b3 in elements: tt_row_stride(T) — a multiple of 4 with TS/4 odd (8-byte aligned rows whose
                           // 8-byte reads by neighbouring threads are bank-conflict free; no padding at T = 20: K2's fourth resident CTA)
  int Tn;                  // GEMM extent of the frame axis = round_up(T, 16)
  int cf;                  // 64-channel chunks per head
  int rows;                // pixels per K1 / K3 tile = min(HW, 128)
  int tmem_cols;
  float scale_log2e;
};

__device__ __forceinline__ uint64_t tt_desc_mn(uint32_t saddr) {  // MN-major, SWIZZLE_128B, single 64-element MN block
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// contiguous global -> shared bulk copy through the TMA engine (bytes % 16 == 0, both addresses 16-byte aligned)
__device__ __forceinline__ void tt_bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ uint32_t tt_pack(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// warp_store_rows64 with 8-byte pieces: rows of the score-term tables are only 8-byte aligned (row stride T rounded up to 4 bf16).
// Consecutive lanes store consecutive pieces of a row: `np` lanes per row segment.
template <class RowPtr>
__device__ __forceinline__ void tt_store_rows8(uint8_t* stage, int lane, const uint4 (&w)[4], RowPtr row_ptr, int np) {
#pragma unroll
  for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(stage + lane * 80 + q * 16) = w[q];
  __syncwarp();
  for (int idx = lane; idx < 32 * np; idx += 32) {
    const int row = idx / np, pc = idx - row * np;
    uint8_t* d = row_ptr(row);
    if (d != nullptr) *reinterpret_cast<uint2*>(d + pc * 8) = *reinterpret_cast<const uint2*>(stage + row * 80 + pc * 8);
  }
  __syncwarp();
}

// ------------------------------------------------------------------------------------------------------------------------
// K1: relative-position score terms.  grid (ceil(HW/128), T, B*heads); 128 threads; thread r <-> pixel row r <-> TMEM lane r
// ------------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) rpe_bias_kernel(const __grid_constant__ CUtensorMap tq, const __grid_constant__ CUtensorMap trk,
                                                       const __grid_constant__ CUtensorMap trq, const TtParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t bar_load, bar_d;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int px0 = blockIdx.x * 128, j = blockIdx.y, bh = blockIdx.z;
  const int b = bh / p.heads, h = bh - b * p.heads;
  const int F = p.F, C = p.C, Tn = p.Tn;
  const int rtile = Tn * 128;
  uint8_t* q_s = smem;                       // [cf][128][128 B]
  uint8_t* k_s = q_s + p.cf * 16384;
  uint8_t* rk_s = k_s + p.cf * 16384;        // [cf][Tn][128 B]
  uint8_t* rq_s = rk_s + p.cf * rtile;
  if (tid == 0) {
    prefetch_tmap(&tq);
    prefetch_tmap(&trk);
    prefetch_tmap(&trq);
    mbar_init(&bar_load, 1);
    mbar_init(&bar_d, 1);
    fence_mbarrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_slot, p.tmem_cols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  pdl_wait();
  if (tid == 0) {
    mbar_expect_tx(&bar_load, (uint32_t)(p.cf * (2 * p.rows * 128 + 2 * rtile)));
    for (int c = 0; c < p.cf; ++c) {
      const int ch = h * F + c * 64;
      tma_load_3d(q_s + c * 16384, &tq, &bar_load, ch, px0, b * p.T + j);
      tma_load_3d(k_s + c * 16384, &tq, &bar_load, C + ch, px0, b * p.T + j);
      tma_load_3d(rk_s + c * rtile, &trk, &bar_load, ch, 0, b * p.T + j);
      tma_load_3d(rq_s + c * rtile, &trq, &bar_load, ch, 0, b * p.T + j);
    }
    mbar_wait(&bar_load, 0);
    tcgen05_fence_after();
    const uint32_t idesc = make_idesc(Tn);
    const int ksteps = F / 16;
    for (int ks = 0; ks < ksteps; ++ks) {
      const int c = ks >> 2, kk = ks & 3;
      umma_bf16(tmem, make_smem_desc(smem_u32(q_s + c * 16384)) + 2 * kk, make_smem_desc(smem_u32(rk_s + c * rtile)) + 2 * kk, idesc, ks != 0);
    }
    for (int ks = 0; ks < ksteps; ++ks) {
      const int c = ks >> 2, kk = ks & 3;
      umma_bf16(tmem + Tn, make_smem_desc(smem_u32(k_s + c * 16384)) + 2 * kk, make_smem_desc(smem_u32(rq_s + c * rtile)) + 2 * kk, idesc, ks != 0);
    }
    umma_commit(&bar_d);
  }
  __syncwarp();
  mbar_wait(&bar_d, 0);
  tcgen05_fence_after();
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
  const int px = px0 + tid;
  const bool ok = tid < p.rows && px < p.HW;
  // 16 fp32 columns (64 bytes per row) at a time through the warp's staging slice (the operand tiles are dead: the MMAs have
  // retired), 4 lanes per row (warp_store_rows64); columns in [T, Tn) come from zero-filled R rows, [Tn, TS) is never read
  uint8_t* stage = smem + warp * 2560;
  const int lane = tid & 31;
  const int r0 = warp * 32;
  (void)ok;
  (void)px;
  for (int c0 = 0; c0 < Tn && c0 < p.TS; c0 += 32) {
    // 32 columns -> 32 bf16 = 64 bytes per row and table
    uint32_t v2[32], v3[32];
    {
      uint32_t a[16];
      tmem_ld_32x32b_x16(trow + c0, a);
#pragma unroll
      for (int k = 0; k < 16; ++k) v2[k] = a[k];
      tmem_ld_32x32b_x16(trow + Tn + c0, a);
#pragma unroll
      for (int k = 0; k < 16; ++k) v3[k] = a[k];
      if (c0 + 16 < Tn) {
        tmem_ld_32x32b_x16(trow + c0 + 16, a);
#pragma unroll
        for (int k = 0; k < 16; ++k) v2[16 + k] = a[k];
        tmem_ld_32x32b_x16(trow + Tn + c0 + 16, a);
#pragma unroll
        for (int k = 0; k < 16; ++k) v3[16 + k] = a[k];
      } else {
#pragma unroll
        for (int k = 0; k < 16; ++k) v2[16 + k] = v3[16 + k] = 0u;
      }
    }
    const int np = min(8, (p.TS - c0) / 4);  // 8-byte pieces of this 64-byte column block that belong to the row
    auto rowp = [&](__nv_bfloat16* base, int r) -> uint8_t* {
      const int rr = r0 + r;
      if (rr >= p.rows || px0 + rr >= p.HW) return nullptr;
      return reinterpret_cast<uint8_t*>(base + (((size_t)bh * p.HW + px0 + rr) * p.T + j) * p.TS + c0);
    };
    uint4 w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
      w[k] = make_uint4(tt_pack(__uint_as_float(v2[8 * k]), __uint_as_float(v2[8 * k + 1])), tt_pack(__uint_as_float(v2[8 * k + 2]), __uint_as_float(v2[8 * k + 3])),
                        tt_pack(__uint_as_float(v2[8 * k + 4]), __uint_as_float(v2[8 * k + 5])), tt_pack(__uint_as_float(v2[8 * k + 6]), __uint_as_float(v2[8 * k + 7])));
    if ((p.TS & 7) == 0) warp_store_rows64(stage, lane, w, [&](int r) { return rowp(p.b2, r); }, np >> 1);
    else tt_store_rows8(stage, lane, w, [&](int r) { return rowp(p.b2, r); }, np);
#pragma unroll
    for (int k = 0; k < 4; ++k)
      w[k] = make_uint4(tt_pack(__uint_as_float(v3[8 * k]), __uint_as_float(v3[8 * k + 1])), tt_pack(__uint_as_float(v3[8 * k + 2]), __uint_as_float(v3[8 * k + 3])),
                        tt_pack(__uint_as_float(v3[8 * k + 4]), __uint_as_float(v3[8 * k + 5])), tt_pack(__uint_as_float(v3[8 * k + 6]), __uint_as_float(v3[8 * k + 7])));
    if ((p.TS & 7) == 0) warp_store_rows64(stage, lane, w, [&](int r) { return rowp(p.b3, r); }, np >> 1);
    else tt_store_rows8(stage, lane, w, [&](int r) { return rowp(p.b3, r); }, np);
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc(tmem, p.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------------------------------
// K2: content terms + softmax.  grid (HW/PL, heads, B); 128 threads; thread r <-> row (pl = r / TP, t = r % TP) <-> TMEM lane r
//     TP = frames per pixel block (8, 16, 32 or 64 >= T), PL = 128 / TP pixels per tile
// ------------------------------------------------------------------------------------------------------------------------
template <int TP>
__global__ void __launch_bounds__(128) attn_rows_kernel(const __grid_constant__ CUtensorMap tq4, const TtParams p) {
  constexpr int PL = 128 / TP;
  constexpr int W = TP < 32 ? 32 : TP;  // score columns a thread reads: the 32-column (or TP-column) window holding its pixel block
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t bar_load, bar_s, bar_o;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int px0 = blockIdx.x * PL, h = blockIdx.y, b = blockIdx.z;
  const int T = p.T, F = p.F, C = p.C, HW = p.HW;
  uint8_t* v_s = smem;                    // [cf][128][128 B]
  uint8_t* q_s = v_s + p.cf * 16384;      // [cf][128][128 B]
  uint8_t* k_s = q_s + p.cf * 16384;      // [cf][128][128 B]
  uint8_t* p_s = q_s;                     // [2][128][128 B]: aliases Q (and K) once S is complete
  if (tid == 0) {
    prefetch_tmap(&tq4);
    mbar_init(&bar_load, 1);
    mbar_init(&bar_s, 1);
    mbar_init(&bar_o, 1);
    fence_mbarrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_slot, 128);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  pdl_wait();
  const int bh = b * p.heads + h;
  const int TS = p.TS;
  // relative-position score terms of this tile's PL pixels: two CONTIGUOUS blocks [PL][T][TS] of b2 / b3 -> shared memory by
  // bulk copies on the same barrier as the operand tiles (scalar per-thread global loads of these rows were 60 % of the kernel)
  __nv_bfloat16* b2_s = reinterpret_cast<__nv_bfloat16*>(smem + p.cf * 3 * 16384);
  __nv_bfloat16* b3_s = b2_s + PL * T * TS;
  if (tid == 0) {
    const uint32_t bias_bytes = (uint32_t)(PL * T * TS * sizeof(__nv_bfloat16));
    mbar_expect_tx(&bar_load, (uint32_t)(p.cf * 3 * 16384) + 2 * bias_bytes);
    for (int c = 0; c < p.cf; ++c) {
      const int ch = h * F + c * 64;
      tma_load_4d(q_s + c * 16384, &tq4, &bar_load, ch, 0, px0, b);
      tma_load_4d(k_s + c * 16384, &tq4, &bar_load, C + ch, 0, px0, b);
      tma_load_4d(v_s + c * 16384, &tq4, &bar_load, 2 * C + ch, 0, px0, b);
    }
    const size_t blk = ((size_t)bh * HW + px0) * T * TS;
    tt_bulk_load(b2_s, p.b2 + blk, bias_bytes, &bar_load);
    tt_bulk_load(b3_s, p.b3 + blk, bias_bytes, &bar_load);
    mbar_wait(&bar_load, 0);
    tcgen05_fence_after();
    const uint32_t idesc = make_idesc(128);
    const int ksteps = F / 16;
    for (int ks = 0; ks < ksteps; ++ks) {
      const int c = ks >> 2, kk = ks & 3;
      umma_bf16(tmem, make_smem_desc(smem_u32(q_s + c * 16384)) + 2 * kk, make_smem_desc(smem_u32(k_s + c * 16384)) + 2 * kk, idesc, ks != 0);
    }
    umma_commit(&bar_s);
  }
  __syncwarp();
  const int pl = tid / TP, t = tid - pl * TP;
  const int px = px0 + pl;
  const bool valid = t < T && px < HW;
  const int sub = TP < 32 ? (pl % (32 / TP)) : 0;     // which TP-block of the 32-column window is this pixel's
  const int col0 = (tid / W) * W;                     // first score column of the window (warp-uniform)
  // two-group mask as bits: bit s = (mask[b, s] > 0.5)
  unsigned long long gbits = ~0ull;
  if (p.mask != nullptr) {
    const int lane = tid & 31;
    const float* maskb = p.mask + (size_t)b * T;
    const unsigned lo = __ballot_sync(0xffffffffu, lane < T && __ldg(maskb + lane) > 0.5f);
    const unsigned hi = __ballot_sync(0xffffffffu, lane + 32 < T && __ldg(maskb + lane + 32) > 0.5f);
    gbits = ((unsigned long long)hi << 32) | lo;
  }
  const bool grp = valid ? ((gbits >> t) & 1ull) != 0 : true;
  mbar_wait(&bar_load, 0);  // bias tiles have landed (the MMA is in flight meanwhile)
  float bias[W];
  {
    float bt[TP];  // this row's bias over its own pixel block: b2[px, t, s] + b3[px, s, t]
    const __nv_bfloat16* b2r = b2_s + (size_t)(pl * T + (valid ? t : 0)) * TS;
    const __nv_bfloat16* b3col = b3_s + (size_t)pl * T * TS + (valid ? t : 0);
    // this row of b2: 16-byte loads when the rows are 16-byte aligned (TS % 8 == 0), else 8-byte loads — both at an odd number of
    // units per row, i.e. free of bank conflicts between the threads of a warp
    auto fin = [&](int s, uint32_t bits) {
      const bool okj = valid && s < T && ((((gbits >> s) & 1ull) != 0) == grp);
      bt[s] = okj ? __uint_as_float(bits) + __bfloat162float(b3col[(size_t)(s < T ? s : 0) * TS]) : -INFINITY;
    };
    if ((TS & 7) == 0) {
#pragma unroll
      for (int k = 0; k < TP / 8; ++k) {
        uint4 r = make_uint4(0u, 0u, 0u, 0u);
        if (valid && 8 * k < T) r = reinterpret_cast<const uint4*>(b2r)[k];
        fin(8 * k, r.x << 16); fin(8 * k + 1, r.x & 0xffff0000u); fin(8 * k + 2, r.y << 16); fin(8 * k + 3, r.y & 0xffff0000u);
        fin(8 * k + 4, r.z << 16); fin(8 * k + 5, r.z & 0xffff0000u); fin(8 * k + 6, r.w << 16); fin(8 * k + 7, r.w & 0xffff0000u);
      }
    } else {
#pragma unroll
      for (int k = 0; k < TP / 4; ++k) {
        uint2 r = make_uint2(0u, 0u);
        if (valid && 4 * k < T) r = reinterpret_cast<const uint2*>(b2r)[k];
        fin(4 * k, r.x << 16); fin(4 * k + 1, r.x & 0xffff0000u); fin(4 * k + 2, r.y << 16); fin(4 * k + 3, r.y & 0xffff0000u);
      }
    }
#pragma unroll
    for (int j = 0; j < W; ++j) {
      const bool own = TP >= 32 ? true : ((j / TP) == sub);
      bias[j] = own ? bt[j % TP] : -INFINITY;
    }
  }
  __syncwarp();
  mbar_wait(&bar_s, 0);
  tcgen05_fence_after();

  // ---- masked softmax over this row's window (fp32)
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
  float e[W];
  float mx = -INFINITY;
#pragma unroll
  for (int c = 0; c < W; c += 32) {
    uint32_t v[32];
    tmem_ld_32x32b_x32(trow + col0 + c, v);
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      e[c + j] = (__uint_as_float(v[j]) + bias[c + j]) * p.scale_log2e;
      mx = fmaxf(mx, e[c + j]);
    }
  }
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < W; ++j) {
    e[j] = valid ? exp2f(e[j] - mx) : 0.f;  // masked entries: exp2(-inf) = 0; rows beyond T: all zero
    sum += e[j];
  }
  const float inv = valid ? 1.f / sum : 0.f;
#pragma unroll
  for (int j = 0; j < W; ++j) e[j] *= inv;
  // ---- P row -> shared memory (K-major, 128-byte swizzle; zero outside the window: P is block diagonal)
  {
    const int sw = tid & 7;
    const int gp0 = col0 >> 3;  // first 16-byte piece of the window among the row's 16 pieces
#pragma unroll
    for (int gp = 0; gp < 16; ++gp) {
      uint8_t* dst = p_s + (gp >> 3) * 16384 + tid * 128 + (((gp & 7) ^ sw) << 4);
      if (gp < gp0 || gp >= gp0 + W / 8) *reinterpret_cast<uint4*>(dst) = make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int q = 0; q < W / 8; ++q) {
      const int gp = gp0 + q;
      uint8_t* dst = p_s + (gp >> 3) * 16384 + tid * 128 + (((gp & 7) ^ sw) << 4);
      *reinterpret_cast<uint4*>(dst) = make_uint4(tt_pack(e[8 * q], e[8 * q + 1]), tt_pack(e[8 * q + 2], e[8 * q + 3]),
                                                  tt_pack(e[8 * q + 4], e[8 * q + 5]), tt_pack(e[8 * q + 6], e[8 * q + 7]));
    }
  }
  fence_proxy_async_smem();
  tcgen05_fence_before();
  __syncthreads();
  if (tid == 0) {
    tcgen05_fence_after();
    // ---- O = P V   (K = the tile's 128 (pixel, frame) rows; N chunks of <= 64 head dims; V is an MN-major operand)
    for (int c = 0; c < p.cf; ++c) {
      const int nf = min(64, F - c * 64);
      const uint32_t idesc = make_idesc(nf, /*b_mn_major=*/1);
      for (int ks = 0; ks < 8; ++ks)
        umma_bf16(tmem + c * 64, make_smem_desc(smem_u32(p_s + (ks >> 2) * 16384)) + 2 * (ks & 3),
                  tt_desc_mn(smem_u32(v_s + c * 16384 + ks * 2048)), idesc, ks != 0);
    }
    umma_commit(&bar_o);
  }
  // ---- attention weights -> global (K3's A operand; also what rpe.py:164 returns as `attn`), while the PV MMAs run.
  // A row's own TP entries are already in this warp's rows of the swizzled P tile: read them back with 8 lanes per row and store
  // whole 128-byte rows (s >= TP zero-filled) — 4 rows per instruction, consecutive (pixel, frame) rows are contiguous in P.
  const int lane = tid & 31;
  if (p.attn_mean != nullptr && valid) {
    float* arow = p.attn_mean + (((size_t)b * HW + px) * T + t) * T;
    const float hw_ = 1.f / (float)p.heads;
#pragma unroll
    for (int j = 0; j < W; ++j) {
      const bool own = TP >= 32 ? true : ((j / TP) == sub);
      if (own && (j % TP) < T) atomicAdd(arow + (j % TP), e[j] * hw_);
    }
  }
  {
    const int k = lane & 7;  // 16-byte piece of the 128-byte output row: entries s = 8k .. 8k+7
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = warp * 32 + i * 4 + (lane >> 3);  // row of the tile
      const int rpl = r / TP, rt = r - rpl * TP;
      if (rt < T && px0 + rpl < HW) {
        uint4 val = make_uint4(0u, 0u, 0u, 0u);
        if (8 * k < TP) {
          const int gp = ((rpl * TP) >> 3) + k;  // piece of the row's 128 columns holding its own block's entries 8k..8k+7
          val = *reinterpret_cast<const uint4*>(p_s + (gp >> 3) * 16384 + r * 128 + (((gp & 7) ^ (r & 7)) << 4));
        }
        *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(p.P + (((size_t)bh * HW + px0 + rpl) * T + rt) * 64) + k * 16) = val;
      }
    }
  }
  __syncwarp();
  mbar_wait(&bar_o, 0);
  tcgen05_fence_after();
  {
    // O -> bf16 -> out: 32 head dims (64 bytes per row) at a time through the warp's staging slice (the P tile is dead: the PV
    // MMAs have retired), 4 lanes per row.  tcgen05.ld is warp-collective: rows beyond T take part and skip the store.
    // (the slice lies inside this warp's OWN 32 rows of the P tile: a slower warp may still be reading its rows for the store above)
    uint8_t* stage = p_s + warp * 4096;
    for (int f = 0; f < F; f += 32) {
      uint32_t v[32];
      const bool two = f + 16 < F;
      {
        uint32_t a[16];
        tmem_ld_32x32b_x16(trow + f, a);
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = a[j];
        if (two) {
          tmem_ld_32x32b_x16(trow + f + 16, a);
#pragma unroll
          for (int j = 0; j < 16; ++j) v[16 + j] = a[j];
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[16 + j] = 0u;
        }
      }
      uint4 w[4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
        w[k] = make_uint4(tt_pack(__uint_as_float(v[8 * k]), __uint_as_float(v[8 * k + 1])), tt_pack(__uint_as_float(v[8 * k + 2]), __uint_as_float(v[8 * k + 3])),
                          tt_pack(__uint_as_float(v[8 * k + 4]), __uint_as_float(v[8 * k + 5])), tt_pack(__uint_as_float(v[8 * k + 6]), __uint_as_float(v[8 * k + 7])));
      warp_store_rows64(stage, lane, w, [&](int rr) -> uint8_t* {
        const int r = warp * 32 + rr;
        const int rpl = r / TP, rt = r - rpl * TP;
        if (rt >= T || px0 + rpl >= HW) return nullptr;
        return reinterpret_cast<uint8_t*>(p.out + ((size_t)(b * T + rt) * HW + px0 + rpl) * C + h * F + f);
      }, two ? 4 : 2);
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc(tmem, 128);
  }
}

// ------------------------------------------------------------------------------------------------------------------------
// K3: relative-position value term.  grid (ceil(HW/128), T, B*heads); 128 threads; thread r <-> pixel row r
//     out[b,t,px,h,:] += P[b,h,px,t,:] . Rv[b,t,:,h,:]
// ------------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) rpe_pv_kernel(const __grid_constant__ CUtensorMap tp4, const __grid_constant__ CUtensorMap trv,
                                                     const __grid_constant__ CUtensorMap to, const TtParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t bar_load, bar_d;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int px0 = blockIdx.x * 128, t = blockIdx.y, bh = blockIdx.z;
  const int b = bh / p.heads, h = bh - b * p.heads;
  const int F = p.F, Tn = p.Tn;
  const int rtile = Tn * 128;
  uint8_t* p_s = smem;               // [128][128 B]  attention weights of frame t, K-major (K = key frame s)
  uint8_t* rv_s = p_s + 16384;       // [cf][Tn][128 B]  Rv[t, s, 64 head dims]: MN-major B operand
  // the content term O_pv of this (frame, head, pixel tile) that K2 left in `out`, fetched by TMA with the operands (a dependent
  // global read-modify-write in the epilogue was 85 % of this kernel's stall samples): [rows][F] bf16, not swizzled
  __nv_bfloat16* o_s = reinterpret_cast<__nv_bfloat16*>(rv_s + p.cf * rtile);
  if (tid == 0) {
    prefetch_tmap(&tp4);
    prefetch_tmap(&trv);
    prefetch_tmap(&to);
    mbar_init(&bar_load, 1);
    mbar_init(&bar_d, 1);
    fence_mbarrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_slot, p.tmem_cols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = tmem_slot;
  pdl_wait();
  if (tid == 0) {
    mbar_expect_tx(&bar_load, (uint32_t)(p.rows * 128 + p.cf * rtile + p.rows * F * 2));
    tma_load_4d(p_s, &tp4, &bar_load, 0, t, px0, bh);
    tma_load_3d(o_s, &to, &bar_load, h * F, px0, b * p.T + t);
    for (int c = 0; c < p.cf; ++c) tma_load_3d(rv_s + c * rtile, &trv, &bar_load, h * F + c * 64, 0, b * p.T + t);
    mbar_wait(&bar_load, 0);
    tcgen05_fence_after();
    for (int c = 0; c < p.cf; ++c) {
      const int nf = min(64, F - c * 64);
      const uint32_t idesc = make_idesc(nf, /*b_mn_major=*/1);
      for (int ks = 0; ks < Tn / 16; ++ks)
        umma_bf16(tmem + c * 64, make_smem_desc(smem_u32(p_s)) + 2 * ks, tt_desc_mn(smem_u32(rv_s + c * rtile + ks * 2048)), idesc, ks != 0);
    }
    umma_commit(&bar_d);
  }
  __syncwarp();
  mbar_wait(&bar_d, 0);
  tcgen05_fence_after();
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
  const int px = px0 + tid;
  const bool ok = tid < p.rows && px < p.HW;
  const __nv_bfloat16* osrc = o_s + (size_t)(ok ? tid : 0) * F;
  uint8_t* stage = p_s + warp * 2560;  // the P tile is dead: the MMAs have retired
  const int lane = tid & 31;
  for (int f = 0; f < F; f += 32) {
    uint32_t v[32];
    const bool two = f + 16 < F;
    {
      uint32_t a[16];
      tmem_ld_32x32b_x16(trow + f, a);
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = a[j];
      if (two) {
        tmem_ld_32x32b_x16(trow + f + 16, a);
#pragma unroll
        for (int j = 0; j < 16; ++j) v[16 + j] = a[j];
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[16 + j] = 0u;
      }
    }
    uint4 w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      uint4 o = make_uint4(0u, 0u, 0u, 0u);
      if (ok && (k < 2 || two)) o = *reinterpret_cast<const uint4*>(osrc + f + 8 * k);
      const uint32_t ow[4] = {o.x, o.y, o.z, o.w};
      uint32_t r[4];
#pragma unroll
      for (int q = 0; q < 4; ++q)
        r[q] = tt_pack(__uint_as_float(ow[q] << 16) + __uint_as_float(v[8 * k + 2 * q]),
                       __uint_as_float(ow[q] & 0xffff0000u) + __uint_as_float(v[8 * k + 2 * q + 1]));
      w[k] = make_uint4(r[0], r[1], r[2], r[3]);
    }
    warp_store_rows64(stage, lane, w, [&](int rr) -> uint8_t* {
      const int r = warp * 32 + rr;
      if (r >= p.rows || px0 + r >= p.HW) return nullptr;
      return reinterpret_cast<uint8_t*>(p.out + ((size_t)(b * p.T + t) * p.HW + px0 + r) * p.C + h * F + f);
    }, two ? 4 : 2);
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc(tmem, p.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------------------------------ host
static int tt_pow2(int v, int lo) {
  int r = lo;
  while (r < v) r <<= 1;
  return r;
}
static inline int tt_round_up(int v, int m) { return (v + m - 1) / m * m; }
// row stride (bf16 elements) of the bias tables: either T rounded up to an ODD number of 16-byte pieces (16-byte row accesses) or to an
// odd number of 8-byte pieces (8-byte accesses), whichever pads less — threads reading their own rows side by side then touch all
// bank groups, and a tile's block of rows stays 16-byte aligned for the bulk copies.  T = 20 -> 20 (K2's smaller tile admits a
// fourth resident CTA), T = 40 -> 40 (16-byte path).
int tt_row_stride(int T) {
  int t16 = tt_round_up(T, 8);
  if (((t16 / 8) & 1) == 0) t16 += 8;
  int t8 = tt_round_up(T, 4);
  if (((t8 / 4) & 1) == 0) t8 += 4;
  return t16 <= t8 ? t16 : t8;
}

static bool tt_shape_ok(const fdm_attn_temporal_args* a) {
  if (a->qkv_dtype != FDM_BF16 || a->out_dtype != FDM_BF16) return false;
  if (a->heads <= 0 || a->C % a->heads) return false;
  const int F = a->C / a->heads;
  if (F % 16 || F > 128 || a->C % 8) return false;
  if (a->T < 1 || a->T > 64) return false;
  const int TP = a->T <= 8 ? 8 : (a->T <= 16 ? 16 : (a->T <= 32 ? 32 : 64));
  if (a->HW % (128 / TP)) return false;
  return true;
}

size_t attn_temporal_tc_workspace(const fdm_attn_temporal_args* a) {
  if (!tt_shape_ok(a)) return 0;
  const size_t rows = (size_t)a->B * a->heads * a->HW * a->T;
  const size_t TS = tt_row_stride(a->T);
  return 2 * rows * TS * sizeof(__nv_bfloat16) + rows * 64 * sizeof(__nv_bfloat16);
}

// returns FDM_ERR_UNSUPPORTED for shapes outside these kernels (the caller then runs the CUDA-core kernel)
int attn_temporal_tc_launch(const fdm_attn_temporal_args* a, cudaStream_t st) {
  if (!tt_shape_ok(a) || !a->Rq_op || !a->Rk_op || !a->Rv_op || !a->workspace) return FDM_ERR_UNSUPPORTED;
  const size_t need = attn_temporal_tc_workspace(a);
  FDM_REQUIRE((size_t)a->workspace_bytes >= need, FDM_ERR_BAD_ARG);
  const int B = a->B, T = a->T, HW = a->HW, C = a->C, heads = a->heads, F = C / heads;
  TtParams p;
  p.mask = a->mask;
  p.B = B; p.T = T; p.HW = HW; p.C = C; p.F = F; p.heads = heads;
  p.TS = tt_row_stride(T);
  p.Tn = tt_round_up(T, 16);
  p.cf = (F + 63) / 64;
  p.rows = HW < 128 ? HW : 128;
  p.scale_log2e = 1.4426950408889634f / sqrtf((float)F);
  const size_t rows = (size_t)B * heads * HW * T;
  p.b2 = reinterpret_cast<__nv_bfloat16*>(a->workspace);
  p.b3 = p.b2 + rows * p.TS;
  p.P = reinterpret_cast<__nv_bfloat16*>(p.b3 + rows * p.TS);
  p.out = reinterpret_cast<__nv_bfloat16*>(a->out);
  p.attn_mean = a->attn_mean;
  const int TP = T <= 8 ? 8 : (T <= 16 ? 16 : (T <= 32 ? 32 : 64));
  const int PL = 128 / TP;

  const CUtensorMapL2promotion L2 = CU_TENSOR_MAP_L2_PROMOTION_L2_128B;
  CUtensorMap tq3, tq4, trq, trk, trv, tp4, to;
  {
    const cuuint64_t dims[3] = {(cuuint64_t)3 * C, (cuuint64_t)HW, (cuuint64_t)B * T};
    const cuuint32_t box[3] = {64, (cuuint32_t)p.rows, 1};
    FDM_REQUIRE(encode_bf16_map(&tq3, a->qkv, 3, dims, box, L2), FDM_ERR_UNSUPPORTED);
  }
  {
    // the same tensor with rows ordered (pixel, frame): dims (channel, frame, pixel, video)
    const cuuint64_t dims[4] = {(cuuint64_t)3 * C, (cuuint64_t)T, (cuuint64_t)HW, (cuuint64_t)B};
    const cuuint64_t strides[3] = {(cuuint64_t)HW * 3 * C * 2, (cuuint64_t)3 * C * 2, (cuuint64_t)T * HW * 3 * C * 2};
    const cuuint32_t box[4] = {64, (cuuint32_t)TP, (cuuint32_t)PL, 1};
    FDM_REQUIRE(encode_bf16_map(&tq4, a->qkv, 4, dims, box, L2, CU_TENSOR_MAP_SWIZZLE_128B, strides), FDM_ERR_UNSUPPORTED);
  }
  {
    const cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)T, (cuuint64_t)B * T};
    const cuuint32_t box[3] = {64, (cuuint32_t)p.Tn, 1};
    FDM_REQUIRE(encode_bf16_map(&trq, a->Rq_op, 3, dims, box, L2) && encode_bf16_map(&trk, a->Rk_op, 3, dims, box, L2) &&
                    encode_bf16_map(&trv, a->Rv_op, 3, dims, box, L2), FDM_ERR_UNSUPPORTED);
  }
  {
    const cuuint64_t dims[4] = {64, (cuuint64_t)T, (cuuint64_t)HW, (cuuint64_t)B * heads};
    const cuuint32_t box[4] = {64, 1, (cuuint32_t)p.rows, 1};
    FDM_REQUIRE(encode_bf16_map(&tp4, p.P, 4, dims, box, L2), FDM_ERR_UNSUPPORTED);
  }
  {
    // `out` as (channel, pixel, frame): box = one head's F channels x the tile's pixels, no swizzle (read by plain ld.shared)
    const cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)HW, (cuuint64_t)B * T};
    const cuuint32_t box[3] = {(cuuint32_t)F, (cuuint32_t)p.rows, 1};
    FDM_REQUIRE(encode_bf16_map(&to, a->out, 3, dims, box, L2, CU_TENSOR_MAP_SWIZZLE_NONE), FDM_ERR_UNSUPPORTED);
  }
  const int smem1 = p.cf * (2 * 16384 + 2 * p.Tn * 128) + 1024;
  const int smem2 = p.cf * 3 * 16384 + 2 * PL * T * p.TS * (int)sizeof(__nv_bfloat16) + 1024;  // P (32 KB) aliases Q + K; + bias tiles
  const int smem3 = 16384 + p.cf * p.Tn * 128 + p.rows * F * 2 + 1024;
  FDM_REQUIRE(smem1 <= 100 * 1024 && smem2 <= 200 * 1024 && smem3 <= 100 * 1024, FDM_ERR_UNSUPPORTED);
  const auto rows_kernel =
      TP == 8 ? attn_rows_kernel<8> : TP == 16 ? attn_rows_kernel<16> : TP == 32 ? attn_rows_kernel<32> : attn_rows_kernel<64>;
  int rc = allow_smem(rpe_bias_kernel, 100 * 1024);
  if (rc == FDM_OK) rc = allow_smem(rows_kernel, 200 * 1024);
  if (rc == FDM_OK) rc = allow_smem(rpe_pv_kernel, 100 * 1024);
  if (rc != FDM_OK) return rc;

  TtParams p1 = p;
  p1.tmem_cols = tt_pow2(2 * p.Tn, 32);
  dim3 gridA((HW + 127) / 128, T, B * heads);
  fdm::launch(rpe_bias_kernel, gridA, dim3(128), smem1, st, tq3, trk, trq, p1);
  rc = check_launch();
  if (rc != FDM_OK) return rc;
  fdm::launch(rows_kernel, dim3(HW / PL, heads, B), dim3(128), smem2, st, tq4, p);
  rc = check_launch();
  if (rc != FDM_OK) return rc;
  TtParams p3 = p;
  p3.tmem_cols = tt_pow2(F, 32);
  fdm::launch(rpe_pv_kernel, gridA, dim3(128), smem3, st, tp4, trv, to, p3);
  return check_launch();
}

}  // namespace fdm
