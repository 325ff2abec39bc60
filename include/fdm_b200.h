/*
 * fdm_b200.h — C-ABI of libfdm_sm100.so: hand-written sm_100a kernels for the FDM latent video
 * denoising hot path (UNetVideoModel.forward + DDPM step math).
 *
 * The reference (plai-group/latent-flexible-video-diffusion-modeling) has NO FFI/plugin boundary:
 * every op below replaces a stock PyTorch call site inside improved_diffusion/{unet,rpe,nn,
 * gaussian_diffusion,respace}.py (cited per entry point, paths relative to the reference root).
 * The Python host in latent-flexible-video-diffusion-modeling_b200/improved_diffusion/ binds these
 * symbols with ctypes (see INTEGRATION.md for the stub).
 *
 * Conventions
 *  - plain pointers and sizes only; all pointers are DEVICE pointers owned by the caller
 *    (PyTorch caching allocator); the library allocates nothing persistent.
 *  - every entry point is asynchronous on `stream` (a cudaStream_t passed as void*), re-entrant, and
 *    never synchronises the device.  Return value: 0 = ok, <0 = FDM_ERR_* (see fdm_status_string).
 *  - activations are channels-last: [N frames][H][W][C]; frame n = b*T + t.
 *  - dtype codes: FDM_F32 = 0, FDM_BF16 = 1 ("operand" tensors feeding tensor-core GEMMs are bf16 in
 *    bf16 mode and fp32 in the exact fp32 mode; residual stream, statistics, softmax are always fp32).
 *  - GroupNorm statistics buffers are [N][C] pairs (sum, sum of squares) of DOUBLES: the producing kernel reduces
 *    each warp's rows in a fixed order in fp32 and adds the partials with fp64 atomics, so the statistics are
 *    reproducible to ~1e-16 run to run (fp32 atomics made the bf16 path chaotic at its rounding-noise level);
 *    the caller zeroes them (one memset per forward).
 */
#ifndef FDM_B200_H_
#define FDM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FDM_ABI_VERSION 2

enum { FDM_F32 = 0, FDM_BF16 = 1 };

enum {
  FDM_OK = 0,
  FDM_ERR_BAD_ARG = -1,      /* null pointer / inconsistent sizes */
  FDM_ERR_UNSUPPORTED = -2,  /* shape or dtype outside what the kernels implement */
  FDM_ERR_CUDA = -3,         /* a CUDA runtime/driver call failed (launch error, bad arch, ...) */
  FDM_ERR_NO_DEVICE = -4     /* no sm_100 device */
};

int fdm_abi_version(void);
const char* fdm_status_string(int status);
/* last CUDA error string seen by this thread inside the library (diagnostics only) */
const char* fdm_last_cuda_error(void);
/* sizeof() of every argument struct, so the host binding can verify its mirror (index = order below) */
size_t fdm_struct_size(int which);

/* ------------------------------------------------------------------------------------------------
 * A1  input preparation — unet.py:439-449
 *   xin[n,h,w,c<C] = x*(1-obs[n]) + x0*obs[n];  xin[n,h,w,C] = obs[n]
 *   x, x0: [N][C][H][W] fp32 (the reference's NCHW frames); xin: [N][H][W][C+1] fp32.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  const float* x;
  const float* x0;
  const float* obs_mask; /* [N] */
  float* xin;      /* fp32 [N][H][W][C+1], or NULL */
  void* xin_bf16;  /* bf16 [N][H][W][Cpad] (channels C+1..Cpad-1 zero: K padding for the tcgen05 stem conv), or NULL */
  int32_t N, C, H, W, Cpad;
} fdm_input_prep_args; /* which = 0 */
int fdm_input_prep(const fdm_input_prep_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * A3/A5/A6/A11  convolution / linear as implicit GEMM — nn.Conv2d call sites unet.py:76,108,155,169,
 * 176-180,313,402 and nn.Linear sites rpe.py:111-112 (qkv, proj_out).
 *   y[n,oh,ow,co] = bias[co] + sum_seg sum_{r,s,ci} A_seg[n, ih, iw, ci] * W_seg[r,s,ci,co]  (+ resid)
 *   segment 0: ksize in {1,3}, stride in {1,2}, optional nearest x2 upsample folded into the gather
 *              (F.interpolate + conv, unet.py:85-87); segment 1 (optional): a 1x1 conv over a second
 *              input with the same spatial size as the output (the ResBlock skip_connection, :180).
 *   Weight layouts:  engine FDM_CONV_SIMT: fp32 [tap = kh*k + kw][ci][co];  engine FDM_CONV_TC: bf16 [tap = kw*k + kh][co_pad][ci_pad]
 *   (filter-column major so one TMA box covers a filter column; ci_pad = ci rounded up to 64, co_pad to 16), both produced by
 *   the host from PyTorch's [co][ci][kh][kw].
 *   FDM_CONV_TC with upsample (3x3, stride 1, Win in {16,32,64,128}): the upsampled tensor is never formed — output pixel
 *   (2y+a, 2x+b) sees input rows y + {a-1, a} and columns x + {b-1, b}; w0 holds the four 2x2 filters of the output phases,
 *   bf16 [phase = 2a + b][tap = 2s' + r'][co_pad][ci_pad], each tap the fp32 SUM of the 3x3 weights that land on that input
 *   pixel (rows: a = 0: {kh 0}, {kh 1, 2};  a = 1: {kh 0, 1}, {kh 2};  columns alike in kw).  4/9 of the FLOPs.
 *   Outputs (any subset): y_f32 [.,Cout] fp32; y_op [.,Cout] in op_dtype; stats (sum,sumsq per frame,
 *   channel); out_nchw: y_f32 is written as [N][Cout][Ho][Wo] (the head conv producing eps).
 * ---------------------------------------------------------------------------------------------- */
/* FDM_CONV_TC: tcgen05; picks the row-halo persistent kernel (conv_halo.cu; CTA pairs / cta_group::2 on deep layers) for 3x3
 * stride-1 convs on 16/32/64/128-wide maps and for wide 1x1 linears (Cin >= 256), the head kernel (conv_head.cu) for the 3x3 conv
 * to <= 4 channels with out_nchw, else the per-tap kernel (conv_tc.cu).  FDM_CONV_TC_TAP forces the per-tap kernel (tests / A-B timing). */
enum { FDM_CONV_SIMT = 0, FDM_CONV_TC = 1, FDM_CONV_TC_TAP = 2 };
typedef struct {
  const void* a0;   /* segment-0 input  [N][Hin][Win][C0], a_dtype */
  const void* w0;   /* segment-0 weights */
  const void* a1;   /* segment-1 input  [N][Ho][Wo][C1] or NULL */
  const void* w1;   /* segment-1 weights (1x1) or NULL */
  const float* bias;  /* [Cout] (sum of both segments' biases) or NULL */
  const float* resid; /* [N][Ho][Wo][Cout] fp32 or NULL */
  float* y_f32;
  void* y_op;
  double* stats;    /* [N][Cout][2] or NULL */
  int32_t N, Hin, Win, C0, C1, Cout;
  int32_t ksize, stride, upsample;
  int32_t a_dtype, op_dtype, out_nchw, engine;
  /* residual = GroupNorm32 of `resid`, recomputed in the epilogue instead of read from a normalised copy (rpe.py:136,173:
   * x = norm(x) ... return x + proj_out(h)).  tcgen05 per-tap engine, ksize 1, Cout = 128 (a group = one float4):
   *   0: `resid` is added as it is;  2: temporal GN, (mean, rstd) per (video, pixel, group) from rn_tstats (written by
   *   fdm_norm_linear a_mode 2);  3: per-frame GN from the (sum, sum of squares) pairs rn_stats */
  int32_t resid_norm;
  int32_t rn_T;            /* frames per video (resid_norm 2) */
  float rn_eps;
  const float* rn_tstats;  /* [B][HW][32][2] */
  const double* rn_stats;  /* [N][Cout][2] */
  const float* rn_gamma;   /* [Cout] */
  const float* rn_beta;
} fdm_conv_args; /* which = 1 */
int fdm_conv(const fdm_conv_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * A4/A5  GroupNorm(32) apply (+FiLM) (+SiLU) — nn.py:12-19, unet.py:153-154,165-166,199-203,400-401,
 * rpe.py:113,136 (spatial attention norm).  The input may be the channel concat of two tensors
 * (th.cat skip connection, unet.py:460) which is never materialised in fp32.
 *   v = (x - mean_g) * rstd_g * gamma + beta;  if film: v = v*(1+film[b][c]) + film[b][C+c];  if silu: v*=sigmoid(v)
 *
 * ResBlock dropout (nn.Dropout between SiLU and the second conv, unet.py:167,203-206), on when drop_philox != NULL and
 * drop_p > 0 (requires silu = 1).  drop_philox is a DEVICE uint64[2] = {seed, nonce}, read at run time (a captured CUDA graph
 * draws a new mask whenever the caller rewrites it).  For the element quad starting at index o of [N][HW][C]:
 *     r    = Philox4x32-10(counter = (lo32(o), hi32(o), drop_salt, lo32(nonce)), key = (lo32(seed), hi32(seed)))
 *     keep = r.{x,y,z,w}[k] >= thr  for element o + k,   thr = min(ceil(drop_p * 2^32), 2^32 - 1)   (i.e. u = r / 2^32 >= p)
 *     out  = keep ? v * s : 0,   s = fp32(1 / (1 - drop_p)), s = 0 for drop_p = 1;  the product is formed in fp32, then rounded
 *                                to op_dtype.
 * fdm_gn_bwd called with the same drop_philox contents, drop_p and drop_salt regenerates the same mask: that is part of this
 * contract (the mask is never stored).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  const void* xa;       /* [N][HW][Ca] fp32, or bf16 when xa_bf16 != 0 */
  const float* xb;      /* [N][HW][Cb] or NULL */
  const double* stats_a; /* [N][Ca][2] */
  const double* stats_b; /* [N][Cb][2] or NULL */
  const float* gamma;   /* [Ca+Cb] */
  const float* beta;
  const float* film;    /* [B][film_stride] rows: scale at [film_off + c], shift at [film_off + C + c]; or NULL */
  void* out_op;         /* [N][HW][C] op_dtype or NULL */
  float* out_f32;       /* [N][HW][C] or NULL */
  void* raw_op;         /* [N][HW][C] op_dtype copy of the un-normalised concat, or NULL */
  int32_t N, HW, Ca, Cb, T;   /* T = frames per video (b = n / T) */
  int32_t film_stride, film_off;
  int32_t silu, op_dtype;
  float eps;
  int32_t xa_bf16;      /* 1: xa holds bf16 (a conv output that only this normalisation reads is stored once, in bf16: inference) */
  int32_t film_add;     /* 1: use_scale_shift_norm=False (unet.py:204-206): film row holds C values e, y = GN(x + e) (statistics of x + e are
                           derived from those of x); 0: scale/shift FiLM, y = GN(x) * (1 + scale) + shift */
  const uint64_t* drop_philox; /* dropout after the SiLU (see above): device {seed, nonce}, or NULL for none */
  float drop_p;         /* 0 <= drop_p <= 1 (FDM_ERR_BAD_ARG otherwise); 0 = no dropout */
  int32_t drop_salt;    /* distinguishes the masks of the launches that share one drop_philox */
} fdm_gn_apply_args; /* which = 2 */
int fdm_gn_apply(const fdm_gn_apply_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * A8(1)  temporal GroupNorm — rpe.py:135-137: statistics over (C/32 channels x T frames) per (b, pixel)
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  const float* x;   /* [B*T][HW][C] */
  const float* gamma;
  const float* beta;
  float* out_f32;   /* [B*T][HW][C] */
  void* out_op;     /* same, op_dtype */
  int32_t B, T, HW, C, op_dtype;
  float eps;
} fdm_temporal_gn_args; /* which = 3 */
int fdm_temporal_gn(const fdm_temporal_gn_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * A2/A5/A9  conditioning path (depends only on t and frame_indices, computed once per step)
 *   fdm_timestep_embedding — nn.py:105-123 (cos | sin)
 *   fdm_grouped_linear     — nn.Linear sites unet.py:304-308 (time_embed), :159 (emb_layers of all
 *                            ResBlocks in one launch), rpe.py:12,14 (RPENet linears of all attention blocks)
 *   fdm_rpe_hidden         — rpe.py:21-30: SiLU(W_t·temb[b]+b_t + W_d·phi(fi[b,t]-fi[b,s]) + b_d)
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  const float* t;         /* [B] model timesteps (already rescaled, respace.py:118-124), or NULL when t_index is given */
  const int64_t* t_index; /* [B] diffusion step index, or NULL */
  const float* t_table;   /* [num_timesteps] model timestep per step index (timestep_map[i]*1000/N), used with t_index */
  const float* freqs;     /* [dim/2] exp(-ln(max_period)*i/half), computed by the host exactly as nn.py:116-118 does (on CPU) */
  float* out;             /* [B][dim] */
  int32_t B, dim;
} fdm_timestep_embedding_args; /* which = 4 */
int fdm_timestep_embedding(const fdm_timestep_embedding_args* a, void* stream);

typedef struct {
  const float* x; /* [M][K] row stride ldx */
  const float* w; /* [Nout][K] (PyTorch Linear layout) */
  const float* b; /* [Nout] or NULL */
  float* y;       /* [M][Nout] row stride ldy */
  int32_t M, K, Nout, ldx, ldy;
  int32_t silu_in; /* apply SiLU to x on load */
} fdm_linear_problem; /* which = 13 */
typedef struct {
  const fdm_linear_problem* problems; /* DEVICE array */
  int32_t count;
  int32_t max_M, max_Nout; /* grid sizing */
  int32_t max_K;           /* largest K of the group (shared-memory sizing of the small-M kernel); 0 = unknown -> tiled kernel */
} fdm_grouped_linear_args; /* which = 5 */
int fdm_grouped_linear(const fdm_grouped_linear_args* a, void* stream);

typedef struct {
  const float* wd;  /* [C][3] embed_distances.weight */
  const float* bd;  /* [C] */
  void* hidden;     /* [B][T][T][C], fp32 or bf16 (hidden_dtype of the launch) */
  int32_t C, te_off; /* this net's W_t·temb + b_t lives at te[b][te_off .. te_off+C) */
} fdm_rpe_hidden_problem; /* which = 14 */
typedef struct {
  const float* te;              /* [B][te_stride] */
  const int64_t* frame_indices; /* [B][T] */
  const fdm_rpe_hidden_problem* problems; /* DEVICE array, one per RPENet */
  int32_t B, T, te_stride, count, max_C;
  int32_t hidden_dtype; /* FDM_F32 (then W_o via fdm_grouped_linear) or FDM_BF16 (then W_o via fdm_conv on tcgen05, 1x1 over B*T*T rows) */
} fdm_rpe_hidden_args; /* which = 6 */
int fdm_rpe_hidden(const fdm_rpe_hidden_args* a, void* stream);

/* A9 (fused)  every RPENet table of a forward in ONE launch (rpe_tables_tc.cu): the hidden layer is generated straight into shared
 *   memory as the A operand of a tcgen05 GEMM with W_o (one tensor map per net, kept in a DEVICE blob), b_o added in the epilogue.
 *   Replaces fdm_rpe_hidden + one fdm_conv per net on inference plans.
 *   fdm_rpe_tables_prepare fills a HOST blob of fdm_rpe_tables_blob_bytes(count) bytes from a HOST array of problems (device
 *   pointers inside); the caller copies it to 128-byte aligned device memory once and passes that to fdm_rpe_tables. */
typedef struct {
  const float* wd;      /* embed_distances.weight [C][3] */
  const float* bd;      /* embed_distances.bias   [C]    */
  const float* bo;      /* out.bias               [C]    */
  const void* w_packed; /* out.weight packed bf16 [1][round_up(C,16)][round_up(C,64)] (FDM_PACK_TC_FWD layout) */
  void* out_op;         /* bf16 table [B][T][T][C] or NULL */
  float* out_f32;       /* fp32 table [B][T][T][C] or NULL */
  int32_t C, te_off;    /* W_t temb + b_t of this net lives at te[b][te_off .. te_off+C) */
} fdm_rpe_table_problem; /* which = 31 */
typedef struct {
  const float* te;              /* [B][te_stride] */
  const int64_t* frame_indices; /* [B][T] */
  const void* blob;             /* DEVICE copy of the prepared blob */
  int32_t count, B, T, te_stride, max_C;
} fdm_rpe_tables_args; /* which = 32 */
size_t fdm_rpe_tables_blob_bytes(int32_t count);
int fdm_rpe_tables_prepare(const fdm_rpe_table_problem* problems, int32_t count, void* host_blob, size_t blob_bytes);
int fdm_rpe_tables(const fdm_rpe_tables_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * A7/A8/A10  the qkv linear of an RPEAttention with its GroupNorm in the operand path (lin_tc.cu) — rpe.py:111-113 (norm, qkv),
 * :135-140 (x = norm(x); qkv = self.qkv(x)).  The normalised tensor is never written:
 *   y_op[m, :] = W . GN(x)[m, :] + bias,  m over the B*T*HW rows of the [B*T][HW][K] activations, K = 128, y_op bf16
 *   a_mode 1: GroupNorm32 per frame, from x (fp32) and the per-(frame, channel) (sum, sum of squares) pairs `stats`;
 *   a_mode 2: the temporal GroupNorm of x (statistics over K/32 channels x T frames per (video, pixel), rpe.py:135-137),
 *             computed inside the tile; the per-(video, pixel, group) (mean, rstd) pairs are written to `tstats` when given.
 *   The matching proj_out (rpe.py:173: return x + proj_out(h) with the NORMALISED x) is fdm_conv with resid = x and
 *   resid_norm = 3 (stats) / 2 (tstats): it recomputes the residual instead of reading a normalised copy.
 *   Persistent CTAs, W resident in shared memory, tcgen05 accumulators in TMEM, the output tile staged whole and drained by TMA
 *   stores.  fdm_norm_linear_supported() tells whether a shape is taken (K = 128, Cout in {128, 256, 384}, HW % 16 == 0,
 *   a_mode 2: T <= 20); callers otherwise run fdm_temporal_gn / fdm_gn_apply + fdm_conv.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  const float* x;       /* [B*T][HW][K] fp32 */
  const double* stats;  /* a_mode 1: [B*T][K][2] */
  float* tstats;        /* a_mode 2: written (may be NULL); [B][HW][32][2] (mean, rstd) */
  const float* gamma;   /* [K] */
  const float* beta;
  const void* w;        /* bf16 [Cout][K] (the packed 1x1 layout of fdm_conv's tcgen05 engine) */
  const float* bias;    /* [Cout] */
  void* y_op;           /* [B*T*HW][Cout] bf16 */
  int32_t B, T, HW, K, Cout;
  int32_t a_mode;
  float eps;
} fdm_norm_linear_args; /* which = 33 */
int fdm_norm_linear(const fdm_norm_linear_args* a, void* stream);
int fdm_norm_linear_supported(const fdm_norm_linear_args* a);

/* ------------------------------------------------------------------------------------------------
 * A8  temporal attention core with in-kernel RPE and the two-group mask — rpe.py:139-170
 *   qkv: [B*T][HW][3C] (q|k|v, each [heads][F]);  Rq,Rk,Rv: [B][T][T][C] fp32 (R[b,t,s,h,f]);
 *   mask: [B][T] (1/0 group id);  out: [B*T][HW][C] op_dtype
 *   Two engines behind the same entry point:
 *     - tcgen05 (attn_temporal_tc.cu; bf16 qkv/out, head dim % 16 == 0, T <= 64): taken when bf16 copies of all three tables
 *       (Rq_op, Rk_op, Rv_op) and a workspace of fdm_attn_temporal_workspace(a) bytes are given.  Three launches: the
 *       relative-position score terms as GEMMs over the pixels of each frame, S = QK^T / softmax / O = PV over rows ordered
 *       (pixel, frame), and the relative-position value term as a GEMM over the pixels.
 *       Workspace layout: bf16 b2[B][heads][HW][T][TS], bf16 b3[B][heads][HW][T][TS] (TS = T rounded up to an odd multiple of 8 or of 4, whichever is smaller), then
 *       bf16 attn[B][heads][HW][T][64] — the NORMALISED attention weights softmax(S)[t, s] (zero for s >= T): what
 *       RPEAttention returns as `attn` (rpe.py:164), readable after the call (fdm_attn_temporal_attn_offset(a) bytes in).
 *     - CUDA cores (attn_simt.cu): fp32 mode and every other shape.
 * A10 spatial attention core — no RPE / no mask; sequence = pixels of one frame.  bf16: S = QK^T and O = PV on tcgen05
 *     (attn_tc.cu: whole score row in TMEM, softmax in fp32 from TMEM); fp32 mode: CUDA-core streaming softmax
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  const void* qkv;
  const float* Rq;
  const float* Rk;
  const float* Rv;
  const float* mask;
  void* out;
  int32_t B, T, HW, C, heads;
  int32_t qkv_dtype, out_dtype;
  const void* Rq_op; /* optional bf16 copies of the three tables ([B][T][T][C]) + workspace: tcgen05 engine */
  const void* Rk_op;
  const void* Rv_op;
  void* workspace;
  int64_t workspace_bytes;
  float* attn_mean; /* optional (tcgen05 engine): [B*HW][T][T] fp32, zeroed by the caller; += softmax(S)[t,s] / heads — the map
                       RPEAttention.forward logs (rpe.py:128-130: mean over heads of `attn`) */
} fdm_attn_temporal_args; /* which = 7 */
int fdm_attn_temporal(const fdm_attn_temporal_args* a, void* stream);
/* bytes of workspace the tcgen05 engine needs for this shape; 0 = the shape is served by the CUDA-core kernel (no workspace) */
size_t fdm_attn_temporal_workspace(const fdm_attn_temporal_args* a);
/* byte offset of the attention-weight tensor inside that workspace */
size_t fdm_attn_temporal_attn_offset(const fdm_attn_temporal_args* a);

typedef struct {
  const void* qkv; /* [N][L][3C] */
  void* out;       /* [N][L][C] */
  int32_t N, L, C, heads;
  int32_t qkv_dtype, out_dtype;
  int32_t engine; /* 0 = auto (tcgen05 kernel for bf16 when L in {16,32,64,128,256} and head dim % 16 == 0, else CUDA cores); 1 = force CUDA cores */
  float* lse;     /* optional output [N][heads][L] (tcgen05 engine only): log-sum-exp of every score row, consumed by fdm_attn_spatial_bwd */
  float* attn_mean; /* optional (tcgen05 engine only): [N][L][L] fp32, zeroed by the caller; += softmax(S)[q,k] / heads (rpe.py:128-130) */
} fdm_attn_spatial_args; /* which = 8 */
int fdm_attn_spatial(const fdm_attn_spatial_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * A6  nearest x2 upsample + cast to operand dtype (F.interpolate, unet.py:85) and plain cast
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  const float* x; /* [N][H][W][C] */
  void* out;      /* [N][H*f][W*f][C], f = upsample ? 2 : 1;  upsample = 2: ZERO-INSERTION (value at even (h,w), zeros
                     elsewhere): the gradient of a stride-2 conv's output prepared for its dgrad/wgrad as stride-1 convs */
  int32_t N, H, W, C, upsample, op_dtype;
  float* colsum;  /* optional (upsample = 0): colsum[c] += sum over all pixels of x[.,c] — the bias gradient of the conv whose output */
  float* colsum2; /* gradient this tensor is (fp32 atomics; zeroed by the caller); colsum2: a second copy (fused 1x1 skip conv bias) */
} fdm_cast_args; /* which = 9 */
int fdm_cast(const fdm_cast_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * A16-A18  fused DDPM posterior update — gaussian_diffusion.py:305-310,341-346,228-231,396-400
 *   coef: DEVICE table [num_timesteps][8] fp32 built once from the float64 numpy tables:
 *     {sqrt_recip_acp, sqrt_recipm1_acp, post_coef1, post_coef2, exp(0.5*log_var)*[t!=0], 0,0,0}
 *   xs = a*x - b*eps; clip; mean = c1*xs + c2*x; sample = mean + sigma*noise
 *   x, eps, noise, sample, pred_xstart: [B][per_video] fp32 (any layout, elementwise); t: [B] int64
 *   sample may alias x (in-place update of the sampler state).
 *   noise == NULL (opt-in perf mode, replaces th.randn_like of gaussian_diffusion.py:396): the noise is drawn inside the
 *   kernel — Philox4x32-10 + Box-Muller, key = philox[0] (seed), counter = (element quad, t[b], philox[1] = stage nonce);
 *   philox: DEVICE uint64[2], read at run time so a captured CUDA graph sees new seeds / nonces.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  const float* x;
  const float* eps;
  const float* noise; /* or NULL with philox != NULL */
  const float* coef;
  const int64_t* t;
  float* sample;
  float* pred_xstart; /* or NULL */
  int64_t per_video;
  int32_t B, clip;
  const uint64_t* philox; /* or NULL */
} fdm_ddpm_step_args; /* which = 10 */
int fdm_ddpm_step(const fdm_ddpm_step_args* a, void* stream);

/* A20/A21  q_sample (gaussian_diffusion.py:200-218) and masked squared-error means (:787-788, nn.py:86-92)
 *   coef2: DEVICE table [num_timesteps][2] = {sqrt_acp, sqrt_one_minus_acp}
 *   mse[b] = mean_{all elems}((noise-eps)^2 * m1[b,frame]); eval[b] likewise with m2;  masks [B][T] or NULL */
typedef struct {
  const float* x0;
  const float* noise;
  const float* coef2;
  const int64_t* t;
  float* x_t;
  int64_t per_video;
  int32_t B;
} fdm_q_sample_args; /* which = 11 */
int fdm_q_sample(const fdm_q_sample_args* a, void* stream);

typedef struct {
  const float* eps;
  const float* noise;
  const float* m1;
  const float* m2;
  float* mse;   /* [B], zeroed by caller */
  float* eval;  /* [B], zeroed by caller */
  int64_t per_frame; /* C*H*W */
  int32_t B, T;
} fdm_masked_mse_args; /* which = 12 */
int fdm_masked_mse(const fdm_masked_mse_args* a, void* stream);


/* ================================================================================================
 * BACKWARD (training) — replaces what torch.autograd runs for the reference's training step
 * (gaussian_diffusion.py:754-796 -> loss.backward() in train_util.py:318-344): cuDNN conv dgrad/wgrad,
 * native_group_norm_backward, softmax/bmm/einsum backward, addmm backward.
 *
 * Gradient conventions: gradients of the fp32 residual stream are fp32 [N][H][W][C]; gradients of GEMM
 * operands (outputs of GroupNorm-apply, qkv, attention outputs) are in the operand dtype.  conv DGRAD is
 * fdm_conv itself over weights packed with mode FDM_PACK_*_DGRAD (a 3x3 pad-1 conv with the filter
 * rotated by 180 degrees and channels swapped; stride-2 dgrad runs over a zero-inserted gradient, see
 * fdm_cast upsample = 2).  Parameter gradients are written in PyTorch's parameter layout, fp32.
 * ============================================================================================== */

/* B0  weight packing: ONE launch re-packs every parameter after an optimizer step (device problem array) */
enum {
  FDM_PACK_TC_FWD = 0,     /* bf16 [tap = kw*k + kh][co_pad16][ci_pad64] = W[co][ci][kh][kw] */
  FDM_PACK_TC_DGRAD = 1,   /* bf16 [tap = s*k + r][ci_pad16][co_pad64]   = W[co][ci][k-1-r][k-1-s] */
  FDM_PACK_SIMT_FWD = 2,   /* fp32 [tap = kh*k + kw][ci][co] */
  FDM_PACK_SIMT_DGRAD = 3, /* fp32 [tap = r*k + s][co][ci]               = W[co][ci][k-1-r][k-1-s] */
  FDM_PACK_SUM2 = 4        /* fp32 [co] = src[co] + src2[co] (bias of a conv fused with its 1x1 skip conv) */
};
typedef struct {
  const float* src;  /* PyTorch parameter: [co][ci][k][k] (Linear: k = 1) */
  const float* src2; /* FDM_PACK_SUM2 only */
  void* dst;         /* padding regions are never written: allocate zeroed */
  int32_t co, ci, k, mode;
} fdm_pack_problem; /* which = 15 */
typedef struct {
  const fdm_pack_problem* problems; /* DEVICE array */
  int32_t count;
  int32_t max_elems; /* largest co*ci*k*k of the group (grid sizing) */
} fdm_pack_weights_args; /* which = 16 */
int fdm_pack_weights(const fdm_pack_weights_args* a, void* stream);

/* B1  conv / linear WGRAD (+ bias gradient) — cudnn_convolution_backward_weight / addmm backward at the nn.Conv2d / nn.Linear
 *     sites listed at fdm_conv.   dw[co][ci][kh][kw] = sum_{n,oh,ow} dy[n,oh,ow,co] * a[n, oh*stride+kh-pad, ow*stride+kw-pad, ci]
 *     split over pixel ranges into fp32 partials (workspace), then reduced in a fixed order (deterministic). */
typedef struct {
  const void* a;    /* forward input operand [N][Hin][Win][C], a_dtype */
  const void* dy;   /* [N][Ho][Wo][Cout], dy_dtype */
  float* dw;        /* [Cout][Cw][k][k] fp32, Cw <= C true input channels (padded operand channels are skipped) */
  float* dbias;     /* [Cout] or NULL: column sums of dy */
  float* dbias2;    /* [Cout] or NULL: a second copy (the 1x1 skip conv's bias sees the same gradient) */
  void* workspace;  /* >= fdm_conv_wgrad_workspace(...) bytes */
  size_t workspace_bytes;
  int32_t N, Hin, Win, C, Cw, Cout, ksize, stride;
  int32_t a_dtype, dy_dtype, engine; /* engine: FDM_CONV_SIMT | FDM_CONV_TC */
} fdm_conv_wgrad_args; /* which = 17 */
int fdm_conv_wgrad(const fdm_conv_wgrad_args* a, void* stream);
size_t fdm_conv_wgrad_workspace(const fdm_conv_wgrad_args* a);

/* B2  GroupNorm(+FiLM)(+SiLU)(+dropout) backward — native_group_norm_backward + silu_backward + the FiLM chain (unet.py:199-203)
 *     du = (dy_op + dy_f32) * m * silu'(u),  m = the dropout factor (keep ? s : 0) of the fdm_gn_apply launch with the same
 *     drop_philox contents / drop_p / drop_salt (1 without dropout);  per (n,c): A = sum_hw du*xhat, B = sum_hw du  (scratch `ab`, fp64 atomics)
 *     dx = rstd * (du*k_c - mean_g(k_c*B) - xhat * mean_g(k_c*A)),  k_c = gamma_c * (1 + scale_c);   gx (+)= dx (+ draw_op)
 *     dgamma_c = sum_n (1+scale) A;  dbeta_c = sum_n (1+scale) B;  dscale[b,c] = sum_{n in b} (gamma A + beta B);  dshift[b,c] = sum B */
typedef struct {
  const float* xa; const float* xb; const double* stats_a; const double* stats_b;
  const float* gamma; const float* beta; const float* film;
  const void* dy_op;    /* gradient wrt out_op (op_dtype) or NULL */
  const float* dy_f32;  /* gradient wrt out_f32 or NULL */
  const void* draw_op;  /* gradient wrt raw_op (op_dtype) or NULL */
  float* gxa; float* gxb; /* gradients wrt xa / xb */
  double* ab;           /* scratch [N][Ca+Cb][2], zeroed by the caller */
  float* dgamma; float* dbeta; /* [Ca+Cb], overwritten */
  float* dfilm;         /* [B][film_stride] rows (scale grads at film_off + c, shift grads at film_off + C + c), overwritten; or NULL */
  int32_t N, HW, Ca, Cb, T, film_stride, film_off, silu, op_dtype;
  int32_t acc_a, acc_b; /* 1: gx += dx, 0: gx = dx */
  float eps;
  const float* dpass_a; /* optional fp32 [N][HW][Ca]: a gradient that reaches xa unchanged (the identity residual of a ResBlock,
                           unet.py:207: out = x + h  =>  g_x += g_out) and is added here instead of by a separate accumulate pass */
  void* gop_a;   /* optional: operand-dtype copy of the FINAL gradient of xa (gxa after this launch's contribution), [N][HW][Ca] — when
                    this GroupNorm is the last contributor to that gradient, the producer's dgrad / wgrad read it without a cast pass */
  float* cs_a;   /* optional (with gop_a): cs_a[c] += column sums of the final gxa = bias gradient of the conv that produced xa (atomics) */
  float* cs2_a;  /* optional second copy (bias of a fused 1x1 skip conv) */
  int32_t phases; /* 0 = all three launches; else a mask: 1 = per-(n,c) sums, 2 = parameter gradients (reads the sums), 4 = apply
                     (reads the sums).  The parameter-gradient launch only feeds parameter gradients, so the training schedule issues it
                     on its side stream (mask 2) and keeps the activation-gradient chain (mask 5) short */
  const uint64_t* drop_philox; /* as fdm_gn_apply_args: the forward's dropout, regenerated (NULL: none; requires silu = 1) */
  float drop_p;
  int32_t drop_salt;
} fdm_gn_bwd_args; /* which = 18 */
int fdm_gn_bwd(const fdm_gn_bwd_args* a, void* stream);

/* B3  temporal GroupNorm backward (rpe.py:135-137) */
typedef struct {
  const float* x; const float* gamma;
  const void* dy_op; const float* dy_f32;
  float* gx;
  float* dgamma; float* dbeta; /* [C], zeroed by the caller (atomic accumulation) */
  int32_t B, T, HW, C, op_dtype, accumulate;
  float eps;
} fdm_temporal_gn_bwd_args; /* which = 19 */
int fdm_temporal_gn_bwd(const fdm_temporal_gn_bwd_args* a, void* stream);

/* B4  attention backward (rpe.py:139-170): recomputes the scores (flash-style), no stored attention matrix.
 *     lse / dsum: scratch [rows] fp32 (log-sum-exp of each score row, and sum_j P_ij dP_ij)
 *     spatial:  rows = N*heads*L;   temporal: rows = B*heads*T*HW;  dRq/dRk/dRv fp32 [B][T][T][C], zeroed by the caller */
typedef struct {
  const void* qkv; const void* out; /* the forward output (D_i = dO_i . O_i) */
  const void* dout; void* dqkv;
  float* lse; float* dsum;
  int32_t N, L, C, heads, dtype;
  int32_t lse_from_forward; /* 1: `lse` holds what fdm_attn_spatial (tcgen05 engine) saved -> the tcgen05 backward kernels may run;
                               0: CUDA-core kernels, which recompute it into `lse` */
} fdm_attn_spatial_bwd_args; /* which = 20 */
int fdm_attn_spatial_bwd(const fdm_attn_spatial_bwd_args* a, void* stream);

typedef struct {
  const void* qkv; const void* out; const float* Rq; const float* Rk; const float* Rv; const float* mask; const void* dout;
  void* dqkv; float* dRq; float* dRk; float* dRv;
  float* lse; float* dsum;
  int32_t B, T, HW, C, heads, dtype;
} fdm_attn_temporal_bwd_args; /* which = 21 */
int fdm_attn_temporal_bwd(const fdm_attn_temporal_bwd_args* a, void* stream);

/* B5  conditioning path backward: RPENet hidden layer (rpe.py:21-30) and the grouped small linears */
typedef struct {
  const float* wd; const float* bd;
  const void* dhidden; /* [B][T][T][C] gradient wrt SiLU(e), dhidden_dtype */
  float* dwd;          /* [C][3], zeroed by the caller */
  float* dbd;          /* [C],    zeroed by the caller */
  int32_t C, te_off;
} fdm_rpe_hidden_bwd_problem; /* which = 22 */
typedef struct {
  const float* te; const int64_t* frame_indices;
  const fdm_rpe_hidden_bwd_problem* problems; /* DEVICE array */
  float* dte; /* [B][te_stride]: d(W_t temb + b_t) written at te_off + c */
  int32_t B, T, te_stride, count, max_C, dhidden_dtype;
} fdm_rpe_hidden_bwd_args; /* which = 23 */
int fdm_rpe_hidden_bwd(const fdm_rpe_hidden_bwd_args* a, void* stream);

typedef struct {
  const float* x; const float* w; const float* dy;
  float* dw;      /* [Nout][K] overwritten */
  float* db;      /* [Nout] overwritten, or NULL */
  float* dx_part; /* [M][K] this problem's contribution to dx (silu' applied when silu_in), or NULL */
  int32_t M, K, Nout, ldx, ldy, silu_in;
} fdm_linear_bwd_problem; /* which = 24 */
typedef struct {
  const fdm_linear_bwd_problem* problems; /* DEVICE array */
  int32_t count, max_M, max_Nout, max_K;
} fdm_grouped_linear_bwd_args; /* which = 25 */
int fdm_grouped_linear_bwd(const fdm_grouped_linear_bwd_args* a, void* stream);

/* out[i] (+)= sum_p parts[p*part_stride + i]  (fixed order) */
typedef struct {
  const float* parts; float* out;
  int64_t part_stride, n;
  int32_t count, accumulate;
} fdm_sum_parts_args; /* which = 26 */
int fdm_sum_parts(const fdm_sum_parts_args* a, void* stream);

/* B6  gradient plumbing: dst (+)= src, optionally summing 2x2 blocks of a twice-larger src (backward of the nearest x2
 *     upsample, unet.py:85);  NCHW fp32 -> NHWC operand with zero channel padding (gradient of eps entering the head conv) */
typedef struct {
  const void* src; float* dst;
  int32_t N, H, W, C; /* dst dims */
  int32_t pool, src_dtype, accumulate;
} fdm_accum_args; /* which = 27 */
int fdm_accum(const fdm_accum_args* a, void* stream);

typedef struct {
  const float* src; void* dst;
  int32_t N, C, H, W, Cpad, op_dtype;
} fdm_nchw_to_nhwc_args; /* which = 28 */
int fdm_nchw_to_nhwc(const fdm_nchw_to_nhwc_args* a, void* stream);


/* B7  fused AdamW over FLAT fp32 buffers — torch.optim.AdamW as constructed by train_util.py:127 (`AdamW(master_params, lr, weight_decay)`),
 *     one launch for the whole model instead of the multi-tensor kernels over 390 tensors (SURVEY §8f-2).  The native backward
 *     already leaves all gradients in one flat buffer; improved_diffusion/optim.py keeps the parameters and both moments flat too.
 *       p *= 1 - lr*wd ;  m = b1 m + (1-b1) g ;  v = b2 v + (1-b2) g^2 ;  p -= (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps)
 *     ema (optional): up to two exponential moving averages of the parameters updated in the same pass (nn.py:55-65) */
typedef struct {
  float* p; const float* g; float* m; float* v;
  float* ema0; float* ema1; /* or NULL */
  int64_t n;
  float lr, beta1, beta2, eps, weight_decay, bias_correction1, bias_correction2_sqrt;
  float ema_rate0, ema_rate1;
} fdm_adamw_args; /* which = 29 */
int fdm_adamw(const fdm_adamw_args* a, void* stream);


/* B8  gradient of the masked squared-error means (fdm_masked_mse) w.r.t. the model output — gaussian_diffusion.py:787-788 backward:
 *     d_out[b,f,i] = (2 / (per_frame*T)) * (out - target) * (g_mse[b]*m1[b,f] + g_eval[b]*m2[b,f]) */
typedef struct {
  const float* out;    /* model output (eps) */
  const float* target; /* noise (or x_start) */
  const float* m1; const float* m2; /* [B][T] masks or NULL (= 1) */
  const float* g_mse; const float* g_eval; /* [B] upstream gradients, either may be NULL (= 0) */
  float* d_out;
  int64_t per_frame;
  int32_t B, T;
} fdm_masked_mse_bwd_args; /* which = 30 */
int fdm_masked_mse_bwd(const fdm_masked_mse_bwd_args* a, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FDM_B200_H_ */
