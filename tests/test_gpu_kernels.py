"""
GPU kernel-level parity (-m gpu): each C-ABI entry point of include/fdm_b200.h against the plain PyTorch op the
reference calls at that site (torch fp32 on the same device).  bf16 tensor-core results are compared with a torch
fp32 op fed the SAME bf16-rounded operands, so the tolerance only has to cover accumulation order (1e-3 rel-L2);
fp32 CUDA-core results are held to 1e-5.
"""
import re

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def pack_tc(w):
    co, ci, kh, kw = w.shape
    cip, cop = (ci + 63) // 64 * 64, (co + 15) // 16 * 16
    out = torch.zeros(kh * kw, cop, cip, dtype=torch.bfloat16, device=w.device)
    out[:, :co, :ci] = w.permute(3, 2, 0, 1).reshape(kh * kw, co, ci).to(torch.bfloat16)  # tap = kw*k + kh
    return out


def pack_simt(w):
    co, ci, kh, kw = w.shape
    return w.permute(2, 3, 1, 0).reshape(kh * kw, ci, co).contiguous().float()


def run_conv(x_nhwc, w, bias, *, stride=1, engine, x1=None, w1=None, resid=None, want_op=False, want_stats=True, want_f32=True):
    """x_nhwc: [N,H,W,C] bf16 (TC) or fp32/bf16 (SIMT).  Returns (y_f32 [N,Ho,Wo,Co], y_op or None, stats or None)."""
    from improved_diffusion import _native as N_
    N, H, W, C0 = x_nhwc.shape
    Co, _, k, _ = w.shape
    pad = k // 2
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    dev = x_nhwc.device
    y = torch.empty(N, Ho, Wo, Co, device=dev)
    yop = torch.empty(N, Ho, Wo, Co, device=dev, dtype=torch.bfloat16) if want_op else None
    stats = torch.zeros(N, Co, 2, device=dev, dtype=torch.float64) if want_stats else None
    pk = pack_simt if engine == N_.CONV_SIMT else pack_tc
    w0p = pk(w)
    w1p = pk(w1) if w1 is not None else None
    a = N_.ConvArgs(a0=x_nhwc.data_ptr(), w0=w0p.data_ptr(), a1=x1.data_ptr() if x1 is not None else None,
                    w1=w1p.data_ptr() if w1p is not None else None, bias=bias.data_ptr() if bias is not None else None,
                    resid=resid.data_ptr() if resid is not None else None, y_f32=y.data_ptr() if want_f32 else None,
                    y_op=yop.data_ptr() if want_op else None, stats=stats.data_ptr() if want_stats else None,
                    N=N, Hin=H, Win=W, C0=C0, C1=x1.shape[-1] if x1 is not None else 0, Cout=Co, ksize=k, stride=stride,
                    upsample=0, a_dtype=N_.BF16 if x_nhwc.dtype == torch.bfloat16 else N_.F32, op_dtype=N_.BF16, out_nchw=0,
                    engine=engine)
    N_.call("fdm_conv", a, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return y, yop, stats


CASES = [
    # N, H, W, C0, Cout, k, stride, C1 (second K segment), resid
    (5, 32, 32, 64, 64, 3, 1, 0, True),
    (5, 32, 32, 64, 128, 3, 1, 64, False),   # ResBlock out-conv with 1x1 skip segment
    (3, 16, 16, 128, 128, 3, 1, 0, True),
    (5, 8, 8, 128, 128, 3, 1, 0, True),      # HW = 64 < 128: two frames per tile, ragged last tile
    (7, 4, 4, 128, 128, 3, 1, 0, False),     # HW = 16: eight frames per tile, half-warp statistics segments
    (2, 16, 16, 64, 192, 1, 1, 0, False),    # qkv linear (1x1), Cout = 3C
    (2, 16, 16, 64, 64, 1, 1, 0, True),      # proj_out + residual
    (2, 32, 32, 32, 32, 3, 1, 0, True),      # nc=32 model: C0 = 32 < the 64-wide K chunk (TMA zero-fill), BN = 32
    (2, 16, 16, 96, 64, 3, 1, 0, False),     # C0 = 96: ragged second K chunk
    (2, 16, 16, 192, 96, 3, 1, 96, False),   # Cout = 96: masked N tile
    (1, 64, 64, 128, 128, 3, 1, 0, True),    # W = 64: two image rows per tile
    (1, 128, 128, 64, 64, 3, 1, 0, False),   # W = 128: one row per tile
    (2, 128, 128, 128, 128, 3, 1, 0, True),  # W = 128 halo, BN = 128: one-tile items, two pipeline stages
    (2, 128, 128, 256, 128, 3, 1, 128, False),  # W = 128 halo with the 1x1 skip segment (decoder ResBlock of the 128-px model)
    (3, 32, 32, 64, 64, 3, 2, 0, False),     # Downsample conv (stride 2) through TMA element strides
    (5, 16, 16, 128, 128, 3, 2, 0, False),   # stride 2 -> 8x8 outputs, two frames per tile
    (40, 32, 32, 64, 64, 3, 1, 0, True),     # > 148 work items: persistent halo CTAs loop, TMEM double buffering wraps
    (24, 16, 16, 256, 128, 3, 1, 128, True), # halo kernel: 4 K chunks + skip segment, BN = 128
    (3, 64, 64, 192, 192, 3, 1, 0, False),   # W = 64 halo (hbox = 2), Cout = 192 -> masked second N tile
    (6, 32, 32, 32, 32, 3, 1, 0, True),      # BN = 32
    (40, 16, 16, 128, 384, 1, 1, 0, False),  # qkv linear through the halo kernel's pointwise mode, 3 N tiles, > 148 items
    (40, 16, 16, 128, 128, 1, 1, 0, True),   # proj_out + residual, pointwise mode
    # CTA pairs (cta_group::2; layers with >= 9 pipeline stages per item and an even number of item pairs)
    (80, 32, 32, 192, 64, 3, 1, 0, False),   # 320 items -> 160 pair items on 74 clusters: the pair loop and the TMEM buffers wrap
    (6, 64, 64, 256, 256, 3, 1, 0, True),    # two N tiles per pair, residual epilogue, W = 64
    (4, 16, 16, 384, 192, 3, 1, 128, False), # Cout = 192 -> BN = 64 pairs (32 weight rows per CTA), 3 N tiles + skip segment
    (2, 16, 16, 192, 96, 3, 1, 0, False),    # Cout = 96: BN = 64, second N tile half masked, 48-row weight boxes cross Cout
    (3, 16, 16, 256, 128, 3, 1, 0, True),    # odd number of item pairs (3): falls back to single CTAs
    (2, 128, 128, 192, 128, 3, 1, 0, False), # W = 128 one-tile items as pairs
]


@pytest.mark.parametrize("engine", [1, 2], ids=["auto", "tap"])
@pytest.mark.parametrize("case", CASES, ids=lambda c: "x".join(map(str, c)))
def test_conv_tc_vs_torch(case, engine):
    from improved_diffusion import _native as N_
    N, H, W, C0, Co, k, stride, C1, use_resid = case
    g = torch.Generator(device="cuda").manual_seed(hash(case) % 1000)
    x = torch.randn(N, H, W, C0, device="cuda", generator=g).to(torch.bfloat16)
    w = (torch.randn(Co, C0, k, k, device="cuda", generator=g) / (C0 * k * k) ** 0.5)
    bias = 0.1 * torch.randn(Co, device="cuda", generator=g)
    pad = k // 2
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    x1 = w1 = None
    if C1:
        x1 = torch.randn(N, Ho, Wo, C1, device="cuda", generator=g).to(torch.bfloat16)
        w1 = torch.randn(Co, C1, 1, 1, device="cuda", generator=g) / C1 ** 0.5
    resid = torch.randn(N, Ho, Wo, Co, device="cuda", generator=g) if use_resid else None
    y, yop, stats = run_conv(x, w, bias, stride=stride, engine=engine, x1=x1, w1=w1, resid=resid, want_op=True)
    wq = w.to(torch.bfloat16).float()
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wq, bias, stride=stride, padding=pad)
    if C1:
        ref = ref + F.conv2d(x1.float().permute(0, 3, 1, 2), w1.to(torch.bfloat16).float())
    ref = ref.permute(0, 2, 3, 1)
    if use_resid:
        ref = ref + resid
    assert rel(y, ref) <= 1e-3, rel(y, ref)
    assert rel(yop.float(), ref) <= 6e-3
    ref_stats = torch.stack([ref.sum(dim=(1, 2)), (ref * ref).sum(dim=(1, 2))], dim=-1)
    assert rel(stats, ref_stats) <= 1e-3
    # and against the CUDA-core engine on the same operands
    y2, _, st2 = run_conv(x, w.to(torch.bfloat16).float(), bias, stride=stride, engine=N_.CONV_SIMT, x1=x1,
                          w1=w1.to(torch.bfloat16).float() if C1 else None, resid=resid)
    assert rel(y, y2) <= 1e-3


@pytest.mark.parametrize("case", [
    # N, H, W, C0, Cout, resid, stats
    (16, 16, 16, 384, 1152, False, False),  # wide qkv linear: halo kernel's pointwise mode (Cin >= 256), 9 N tiles
    (16, 16, 16, 384, 384, True, True),     # wide proj_out + residual + statistics
    (16, 8, 8, 512, 1536, False, False),    # 8x8 map without statistics: runs as a flat pixel list of 128-wide rows
    (12, 4, 4, 512, 512, True, False),      # 4x4, 192 pixels: not a multiple of 256 -> per-tap kernel
    (16, 8, 8, 512, 512, True, True),       # 8x8 with statistics -> per-tap kernel
], ids=lambda c: "x".join(map(str, c)))
def test_wide_pointwise_vs_torch(case):
    from improved_diffusion import _native as N_
    N, H, W, C0, Co, use_resid, want_stats = case
    g = torch.Generator(device="cuda").manual_seed(sum(case[:5]))
    x = torch.randn(N, H, W, C0, device="cuda", generator=g).to(torch.bfloat16)
    w = torch.randn(Co, C0, 1, 1, device="cuda", generator=g) / C0 ** 0.5
    bias = 0.1 * torch.randn(Co, device="cuda", generator=g)
    resid = torch.randn(N, H, W, Co, device="cuda", generator=g) if use_resid else None
    y, yop, stats = run_conv(x, w, bias, engine=N_.CONV_TC, resid=resid, want_op=True, want_stats=want_stats)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), w.to(torch.bfloat16).float(), bias).permute(0, 2, 3, 1)
    if use_resid:
        ref = ref + resid
    assert rel(y, ref) <= 1e-3, rel(y, ref)
    assert rel(yop.float(), ref) <= 6e-3
    if want_stats:
        ref_stats = torch.stack([ref.sum(dim=(1, 2)), (ref * ref).sum(dim=(1, 2))], dim=-1)
        assert rel(stats, ref_stats) <= 1e-3


def run_head_conv(x, w0p, bias, Co, engine):
    """fdm_conv in the head form: 3x3, NCHW fp32 output.  x [N,H,W,C0] bf16, w0p packed by pack_tc.  Returns y [N,Co,H,W]."""
    from improved_diffusion import _native as N_
    N, H, W, C0 = x.shape
    y = torch.full((N, Co, H, W), float("nan"), device="cuda")
    a = N_.ConvArgs(a0=x.data_ptr(), w0=w0p.data_ptr(), a1=None, w1=None, bias=bias.data_ptr(), resid=None, y_f32=y.data_ptr(),
                    y_op=None, stats=None, N=N, Hin=H, Win=W, C0=C0, C1=0, Cout=Co, ksize=3, stride=1, upsample=0,
                    a_dtype=N_.BF16, op_dtype=N_.BF16, out_nchw=1, engine=engine)
    N_.call("fdm_conv", a, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return y


@pytest.mark.parametrize("case", [
    # N, H, W, C0, Cout
    (20, 32, 32, 64, 4),    # cfg4 head
    (3, 64, 64, 128, 4),    # cfg5 head: two 64-channel chunks
    (2, 128, 128, 128, 3),  # cfg3 head: 3 output channels, 128-wide rows
    (5, 16, 16, 192, 4),    # three chunks, whole frame in one strip
    (3, 8, 8, 64, 3),       # small map: partial MMA tile
    (2, 24, 40, 64, 4),     # non-square, W not a power of two
], ids=lambda c: "x".join(map(str, c)))
def test_head_conv_vs_torch(case):
    """conv_head.cu (taps in the GEMM's N dimension, shifts applied to the output) against torch and against the per-tap kernel"""
    from improved_diffusion import _native as N_
    N, H, W, C0, Co = case
    g = torch.Generator(device="cuda").manual_seed(sum(case))
    x = torch.randn(N, H, W, C0, device="cuda", generator=g).to(torch.bfloat16)
    w = torch.randn(Co, C0, 3, 3, device="cuda", generator=g) / (9 * C0) ** 0.5
    bias = 0.1 * torch.randn(Co, device="cuda", generator=g)
    w0p = pack_tc(w)
    outs = []
    for engine in (N_.CONV_TC, N_.CONV_TC_TAP):
        try:
            outs.append(run_head_conv(x, w0p, bias, Co, engine))
        except N_.NativeError:
            assert engine == N_.CONV_TC_TAP  # the per-tap kernel does not take every map shape; the head kernel must
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), w.to(torch.bfloat16).float(), bias, padding=1)
    assert rel(outs[0], ref) <= 1e-3, rel(outs[0], ref)
    if len(outs) > 1:
        assert rel(outs[0], outs[1]) <= 1e-3


@pytest.mark.parametrize("case", [
    # N, H, W, C0, Cout, C1
    (20, 32, 32, 64, 64, 192),      # cfg4 top level: skip_connection over cat([h (128), skip (64)])
    (6, 16, 16, 128, 128, 256),     # 16x16 level
    (4, 64, 64, 128, 128, 384),     # cfg5 / cfg3: deep skip segment, CTA pairs
    (2, 128, 128, 128, 128, 256),   # 128-wide maps, two-tile pair items
    (3, 16, 16, 384, 384, 840),     # ragged last chunk of the skip segment (840 = 13 * 64 + 8)
], ids=lambda c: "x".join(map(str, c)))
def test_conv_wide_skip_segment_vs_torch(case):
    """fdm_conv (halo kernel) with a wide 1x1 skip segment (the ResBlock skip_connection over th.cat of unet.py:460) against torch:
    output and per-frame statistics."""
    from improved_diffusion import _native as N_
    N, H, W, C0, Co, C1 = case
    g = torch.Generator(device="cuda").manual_seed(sum(case))
    x = torch.randn(N, H, W, C0, device="cuda", generator=g).to(torch.bfloat16)
    x1 = torch.randn(N, H, W, C1, device="cuda", generator=g).to(torch.bfloat16)
    w = torch.randn(Co, C0, 3, 3, device="cuda", generator=g) / (9 * C0) ** 0.5
    w1 = torch.randn(Co, C1, 1, 1, device="cuda", generator=g) / C1 ** 0.5
    bias = 0.1 * torch.randn(Co, device="cuda", generator=g)
    w0p, w1p = pack_tc(w), pack_tc(w1)
    y = torch.full((N, H, W, Co), float("nan"), device="cuda")
    stats = torch.zeros(N, Co, 2, device="cuda", dtype=torch.float64)
    a = N_.ConvArgs(a0=x.data_ptr(), w0=w0p.data_ptr(), a1=x1.data_ptr(), w1=w1p.data_ptr(), bias=bias.data_ptr(), resid=None,
                    y_f32=y.data_ptr(), y_op=None, stats=stats.data_ptr(), N=N, Hin=H, Win=W, C0=C0, C1=C1, Cout=Co, ksize=3,
                    stride=1, upsample=0, a_dtype=N_.BF16, op_dtype=N_.BF16, out_nchw=0, engine=N_.CONV_TC)
    N_.call("fdm_conv", a, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), w.to(torch.bfloat16).float(), bias, padding=1)
    ref = ref + F.conv2d(x1.float().permute(0, 3, 1, 2), w1.to(torch.bfloat16).float())
    ref = ref.permute(0, 2, 3, 1)
    assert rel(y, ref) <= 1e-3, rel(y, ref)
    ref_stats = torch.stack([ref.sum(dim=(1, 2)), (ref * ref).sum(dim=(1, 2))], dim=-1)
    assert rel(stats, ref_stats) <= 1e-3, rel(stats, ref_stats)


def pack_tc_up(w):
    """[co][ci][3][3] -> bf16 [phase = 2a + b][tap = 2s' + r'][co_pad][ci_pad]: per-phase 2x2 filters of nearest-x2-upsample + conv"""
    co, ci, _, _ = w.shape
    cip, cop = (ci + 63) // 64 * 64, (co + 15) // 16 * 16
    sets = {0: ([0], [1, 2]), 1: ([0, 1], [2])}
    out = torch.zeros(16, cop, cip, dtype=torch.bfloat16, device=w.device)
    for a in (0, 1):
        for b in (0, 1):
            for sp in (0, 1):
                for rp in (0, 1):
                    ws = w[:, :, sets[a][rp], :][:, :, :, sets[b][sp]].float().sum(dim=(2, 3))
                    out[(2 * a + b) * 4 + 2 * sp + rp, :co, :ci] = ws.to(torch.bfloat16)
    return out


@pytest.mark.parametrize("case", [
    # N, H, W (low resolution), C, Cout
    (20, 16, 16, 128, 128),   # cfg4: 16x16 -> 32x32
    (6, 32, 32, 256, 256),    # cfg5 top: two N tiles
    (4, 64, 64, 128, 128),    # cfg3 top: 64 -> 128
    (5, 16, 16, 384, 384),    # deep: CTA pairs, three N tiles
    (3, 32, 32, 64, 96),      # masked N tile
    (3, 16, 16, 128, 64),     # odd number of tile pairs: single CTAs
], ids=lambda c: "x".join(map(str, c)))
def test_upsample_conv_vs_torch(case):
    """nearest x2 upsample + 3x3 conv as four 2x2-tap phase convs over the low-resolution input (conv_halo.cu, `up` mode)"""
    from improved_diffusion import _native as N_
    N, H, W, C0, Co = case
    g = torch.Generator(device="cuda").manual_seed(sum(case))
    x = torch.randn(N, H, W, C0, device="cuda", generator=g).to(torch.bfloat16)
    w = torch.randn(Co, C0, 3, 3, device="cuda", generator=g) / (9 * C0) ** 0.5
    bias = 0.1 * torch.randn(Co, device="cuda", generator=g)
    wp = pack_tc_up(w)
    y = torch.full((N, 2 * H, 2 * W, Co), float("nan"), device="cuda")
    yop = torch.empty(N, 2 * H, 2 * W, Co, device="cuda", dtype=torch.bfloat16)
    stats = torch.zeros(N, Co, 2, device="cuda", dtype=torch.float64)
    a = N_.ConvArgs(a0=x.data_ptr(), w0=wp.data_ptr(), a1=None, w1=None, bias=bias.data_ptr(), resid=None, y_f32=y.data_ptr(),
                    y_op=yop.data_ptr(), stats=stats.data_ptr(), N=N, Hin=H, Win=W, C0=C0, C1=0, Cout=Co, ksize=3, stride=1,
                    upsample=1, a_dtype=N_.BF16, op_dtype=N_.BF16, out_nchw=0, engine=N_.CONV_TC)
    N_.call("fdm_conv", a, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    xu = F.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2, mode="nearest")
    ref = F.conv2d(xu, w, bias, padding=1).permute(0, 2, 3, 1)              # fp32 weights: the phase filters are summed in fp32
    ref_b = F.conv2d(xu, w.to(torch.bfloat16).float(), bias, padding=1).permute(0, 2, 3, 1)  # what the un-fused bf16 path computes
    err = rel(y, ref)
    assert err <= 4e-3, err
    assert err <= 1.5 * rel(ref_b, ref) + 1e-4, (err, rel(ref_b, ref))      # no worse than rounding each 3x3 weight to bf16
    assert rel(yop.float(), y) <= 6e-3
    yc = y.double()
    ref_stats = torch.stack([yc.sum(dim=(1, 2)), (yc * yc).sum(dim=(1, 2))], dim=-1)
    assert rel(stats, ref_stats) <= 1e-4


def test_conv_simt_fp32_exact():
    from improved_diffusion import _native as N_
    g = torch.Generator(device="cuda").manual_seed(3)
    for (N, H, W, C0, Co, k, stride) in [(2, 32, 32, 5, 32, 3, 1), (2, 16, 16, 64, 4, 3, 1), (3, 32, 32, 64, 64, 3, 2)]:
        x = torch.randn(N, H, W, C0, device="cuda", generator=g)
        w = torch.randn(Co, C0, k, k, device="cuda", generator=g) / (C0 * k * k) ** 0.5
        b = torch.randn(Co, device="cuda", generator=g)
        y, _, stats = run_conv(x, w, b, stride=stride, engine=N_.CONV_SIMT)
        old = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        ref = F.conv2d(x.permute(0, 3, 1, 2), w, b, stride=stride, padding=k // 2).permute(0, 2, 3, 1)
        torch.backends.cudnn.allow_tf32 = old
        assert rel(y, ref) <= 1e-5
        ref_stats = torch.stack([ref.sum(dim=(1, 2)), (ref * ref).sum(dim=(1, 2))], dim=-1)
        assert rel(stats, ref_stats) <= 1e-4


@pytest.mark.parametrize("N,L,C,heads", [(5, 256, 128, 4), (3, 64, 128, 4), (7, 16, 128, 4), (2, 256, 64, 4), (2, 256, 192, 4),
                                         (2, 256, 256, 4), (1, 64, 512, 4), (2, 256, 384, 4), (3, 64, 96, 4)])
@pytest.mark.parametrize("engine", [0, 1])
def test_attn_spatial_vs_torch(N, L, C, heads, engine):
    """fdm_attn_spatial (engine 0: tcgen05 where the shape allows, 1: CUDA cores) vs softmax(q k^T / sqrt(F)) v in torch fp32."""
    from improved_diffusion import _native as N_
    g = torch.Generator(device="cuda").manual_seed(L + C)
    qkv = torch.randn(N, L, 3 * C, device="cuda", generator=g).to(torch.bfloat16)
    out = torch.empty(N, L, C, device="cuda", dtype=torch.bfloat16)
    a = N_.AttnSpatialArgs(qkv=qkv.data_ptr(), out=out.data_ptr(), N=N, L=L, C=C, heads=heads, qkv_dtype=N_.BF16,
                           out_dtype=N_.BF16, engine=engine)
    N_.call("fdm_attn_spatial", a, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    F_ = C // heads
    q, k, v = qkv.float().view(N, L, 3, heads, F_).permute(2, 0, 3, 1, 4)
    ref = (torch.softmax(q @ k.transpose(-1, -2) * F_ ** -0.5, dim=-1) @ v).permute(0, 2, 1, 3).reshape(N, L, C)
    assert rel(out.float(), ref) <= 8e-3, rel(out.float(), ref)  # bf16 output rounding 2^-9 rms + bf16 P


@pytest.mark.parametrize("N,H,W,C0,Co", [(3, 32, 32, 64, 4), (2, 16, 16, 128, 3), (2, 32, 32, 8, 64)])
def test_conv_tc_head_and_stem(N, H, W, C0, Co):
    """Head conv (Cout 3/4, NCHW fp32 output, unet.py:402) and stem conv (5 input channels zero-padded to 8, unet.py:313)."""
    from improved_diffusion import _native as N_
    g = torch.Generator(device="cuda").manual_seed(C0 + Co)
    x = torch.randn(N, H, W, C0, device="cuda", generator=g)
    if C0 == 8:
        x[..., 5:] = 0
    x = x.to(torch.bfloat16)
    w = torch.randn(Co, C0, 3, 3, device="cuda", generator=g) / (C0 * 9) ** 0.5
    bias = 0.1 * torch.randn(Co, device="cuda", generator=g)
    nchw = Co < 16
    y = torch.empty((N, Co, H, W) if nchw else (N, H, W, Co), device="cuda")
    wp = pack_tc(w)
    a = N_.ConvArgs(a0=x.data_ptr(), w0=wp.data_ptr(), a1=None, w1=None, bias=bias.data_ptr(), resid=None, y_f32=y.data_ptr(),
                    y_op=None, stats=None, N=N, Hin=H, Win=W, C0=C0, C1=0, Cout=Co, ksize=3, stride=1, upsample=0,
                    a_dtype=N_.BF16, op_dtype=N_.BF16, out_nchw=int(nchw), engine=N_.CONV_TC)
    N_.call("fdm_conv", a, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), w.to(torch.bfloat16).float(), bias, padding=1)
    if not nchw:
        ref = ref.permute(0, 2, 3, 1)
    assert rel(y, ref) <= 1e-3, rel(y, ref)


def _temporal_reference(qkv, Rq, Rk, Rv, mask, B, T, HW, C, heads):
    """softmax(scale (q k^T + q.Rk + k.Rq) + two-group mask) (v + Rv) in torch fp32 (rpe.py:139-170); returns (out, attn)"""
    F_ = C // heads
    x = qkv.float().view(B, T, HW, 3, heads, F_).permute(3, 0, 2, 4, 1, 5)  # 3 B HW H T F
    q, k, v = x[0], x[1], x[2]
    rq, rk, rv = (r.float().view(B, T, T, heads, F_) for r in (Rq, Rk, Rv))
    w = q @ k.transpose(-1, -2)
    w = w + torch.einsum("bdhtf,btshf->bdhts", q, rk) + torch.einsum("bdhtf,btshf->bdhts", k, rq).transpose(-1, -2)
    w = w * F_ ** -0.5
    allowed = mask.view(B, 1, T) * mask.view(B, T, 1) + (1 - mask.view(B, 1, T)) * (1 - mask.view(B, T, 1))
    w = w.masked_fill((allowed == 0).view(B, 1, 1, T, T), float("-inf"))
    p = torch.softmax(w, dim=-1)
    o = p @ v + torch.einsum("bdhts,btshf->bdhtf", p, rv)
    return o.permute(0, 3, 1, 2, 4).reshape(B * T, HW, C), p  # out [B T HW H F]; attn [B, HW, H, T, T]


@pytest.mark.parametrize("B,T,HW,C,heads", [(2, 5, 256, 64, 4), (1, 20, 64, 128, 4), (2, 7, 16, 128, 4), (1, 40, 256, 384, 4),
                                            (1, 33, 64, 96, 4), (3, 12, 40, 128, 4)])
def test_attn_temporal_vs_torch(B, T, HW, C, heads):
    """fdm_attn_temporal, CUDA-core engine (fp32 tables, no workspace) against torch fp32."""
    from improved_diffusion import _native as N_
    g = torch.Generator(device="cuda").manual_seed(T * 7 + C)
    qkv = torch.randn(B * T, HW, 3 * C, device="cuda", generator=g).to(torch.bfloat16)
    Rq, Rk, Rv = (0.5 * torch.randn(B, T, T, C, device="cuda", generator=g) for _ in range(3))
    mask = (torch.rand(B, T, device="cuda", generator=g) > 0.3).float()
    out = torch.empty(B * T, HW, C, device="cuda", dtype=torch.bfloat16)
    a = N_.AttnTemporalArgs(qkv=qkv.data_ptr(), Rq=Rq.data_ptr(), Rk=Rk.data_ptr(), Rv=Rv.data_ptr(), mask=mask.data_ptr(),
                            out=out.data_ptr(), B=B, T=T, HW=HW, C=C, heads=heads, qkv_dtype=N_.BF16, out_dtype=N_.BF16)
    N_.call("fdm_attn_temporal", a, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ref, _ = _temporal_reference(qkv, Rq, Rk, Rv, mask, B, T, HW, C, heads)
    assert rel(out.float(), ref) <= 6e-3, rel(out.float(), ref)


@pytest.mark.parametrize("B,T,HW,C,heads", [
    (8, 20, 256, 128, 4), (8, 20, 64, 128, 4), (8, 20, 16, 128, 4),      # cfg4's three attention resolutions (F = 32, TP = 32)
    (2, 40, 256, 384, 4), (2, 40, 64, 512, 4),                           # cfg5 (F = 96 / 128, TP = 64, two channel chunks)
    (1, 5, 256, 128, 4), (1, 5, 16, 64, 4),                              # cfg2 / cfg1 (TP = 8, F = 32 / 16)
    (2, 1, 64, 64, 4), (2, 2, 64, 128, 4), (1, 8, 64, 128, 4), (3, 9, 16, 128, 4), (1, 14, 256, 128, 4), (2, 16, 64, 128, 4),
    (1, 17, 64, 256, 4), (1, 32, 64, 128, 4), (1, 33, 16, 384, 4), (1, 64, 64, 128, 2), (2, 12, 64, 192, 4),
])
@pytest.mark.parametrize("masked", [True, False])
def test_attn_temporal_tcgen05_vs_torch(B, T, HW, C, heads, masked):
    """fdm_attn_temporal, tcgen05 engine (attn_temporal_tc.cu: bf16 tables + workspace) against torch fp32 over the SAME
    bf16-rounded operands: the output, and the normalised attention weights it leaves in the workspace (rpe.py:164 `attn`)."""
    from improved_diffusion import _native as N_
    import ctypes as C_
    g = torch.Generator(device="cuda").manual_seed(T * 7 + C + HW)
    qkv = torch.randn(B * T, HW, 3 * C, device="cuda", generator=g).to(torch.bfloat16)
    Rq, Rk, Rv = ((0.5 * torch.randn(B, T, T, C, device="cuda", generator=g)).to(torch.bfloat16) for _ in range(3))
    mask = (torch.rand(B, T, device="cuda", generator=g) > 0.3).float() if masked else None
    out = torch.full((B * T, HW, C), float("nan"), device="cuda", dtype=torch.bfloat16)
    a = N_.AttnTemporalArgs(qkv=qkv.data_ptr(), Rq=None, Rk=None, Rv=None, mask=mask.data_ptr() if masked else None,
                            out=out.data_ptr(), B=B, T=T, HW=HW, C=C, heads=heads, qkv_dtype=N_.BF16, out_dtype=N_.BF16,
                            Rq_op=Rq.data_ptr(), Rk_op=Rk.data_ptr(), Rv_op=Rv.data_ptr())
    need = int(N_.lib().fdm_attn_temporal_workspace(C_.byref(a)))
    assert need > 0, "the tcgen05 engine should take this shape"
    ws = torch.full((need,), 0xFF, device="cuda", dtype=torch.uint8)  # NaN-poisoned: every byte that is read must have been written
    a.workspace, a.workspace_bytes = ws.data_ptr(), need
    N_.call("fdm_attn_temporal", a, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    m = mask if masked else torch.ones(B, T, device="cuda")
    ref, p_ref = _temporal_reference(qkv, Rq, Rk, Rv, m, B, T, HW, C, heads)
    e = rel(out.float(), ref)
    off = int(N_.lib().fdm_attn_temporal_attn_offset(C_.byref(a)))
    attn = ws[off:off + B * heads * HW * T * 64 * 2].view(torch.bfloat16).view(B, heads, HW, T, 64).float()
    e_attn = rel(attn[..., :T].permute(0, 2, 1, 3, 4), p_ref)
    print(f"temporal tcgen05 B={B} T={T} HW={HW} C={C}: out rel-L2 {e:.3e}, attention weights rel-L2 {e_attn:.3e}")
    assert bool(torch.isfinite(out.float()).all())
    assert float(attn[..., T:].abs().max()) == 0.0 if T < 64 else True
    assert e_attn <= 6e-3, e_attn   # P is stored in bf16
    assert e <= 8e-3, e             # bf16 P feeding both value terms, bf16 output


@pytest.mark.parametrize("B,T,Cs", [(8, 20, (128, 128, 128)), (2, 40, (384, 512, 384, 512)), (1, 5, (64,)), (3, 7, (96, 200))])
def test_rpe_tables_fused_vs_torch(B, T, Cs):
    """fdm_rpe_tables (rpe_tables_tc.cu): every RPENet table of a forward in one launch — hidden layer generated in shared memory,
    W_o GEMM on tcgen05 from per-net tensor maps in a device blob — against the torch expression of rpe.py:20-31 over the same
    bf16-rounded hidden values and weights."""
    import ctypes as C_
    from improved_diffusion import _native as N_
    g = torch.Generator(device="cuda").manual_seed(B * 100 + T)
    dev = "cuda"
    te_stride = sum(Cs) + 16
    te = torch.randn(B, te_stride, device=dev, generator=g)
    fi = torch.stack([torch.sort(torch.randperm(300, device=dev, generator=g)[:T]).values for _ in range(B)]).long()
    probs, keep, refs = (N_.RpeTableProblem * len(Cs))(), [], []
    off = 16
    for i, Cc in enumerate(Cs):
        wd, bd, bo = torch.randn(Cc, 3, device=dev, generator=g), torch.randn(Cc, device=dev, generator=g), torch.randn(Cc, device=dev, generator=g)
        w = (torch.randn(Cc, Cc, device=dev, generator=g) / Cc ** 0.5)
        cop, cip = (Cc + 15) // 16 * 16, (Cc + 63) // 64 * 64
        wp = torch.zeros(1, cop, cip, device=dev, dtype=torch.bfloat16)
        wp[0, :Cc, :Cc] = w.to(torch.bfloat16)
        out_op = torch.full((B, T, T, Cc), float("nan"), device=dev, dtype=torch.bfloat16)
        out_f32 = torch.full((B, T, T, Cc), float("nan"), device=dev) if i % 2 == 0 else None
        keep += [wd, bd, bo, wp, out_op, out_f32]
        probs[i] = N_.RpeTableProblem(wd=wd.data_ptr(), bd=bd.data_ptr(), bo=bo.data_ptr(), w_packed=wp.data_ptr(), out_op=out_op.data_ptr(),
                                      out_f32=out_f32.data_ptr() if out_f32 is not None else None, C=Cc, te_off=off)
        d = (fi.unsqueeze(-1) - fi.unsqueeze(-2)).float()
        feats = torch.stack([torch.log(1 + d.clamp(min=0)), torch.log(1 + (-d).clamp(min=0)), (d == 0).float()], dim=-1)
        e = te[:, off:off + Cc].view(B, 1, 1, Cc) + feats @ wd.t() + bd
        hidden = torch.nn.functional.silu(e).to(torch.bfloat16).float()
        refs.append((hidden @ w.to(torch.bfloat16).float().t() + bo, out_op, out_f32))
        off += Cc
    n = int(N_.lib().fdm_rpe_tables_blob_bytes(len(Cs)))
    host = (C_.c_uint8 * n)()
    N_.check(N_.lib().fdm_rpe_tables_prepare(C_.byref(probs), len(Cs), C_.byref(host), n), "prepare")
    raw = torch.zeros(n + 128, dtype=torch.uint8, device=dev)
    blob = raw[(-raw.data_ptr()) % 128:][:n]
    blob.copy_(torch.frombuffer(bytearray(bytes(host)), dtype=torch.uint8))
    a = N_.RpeTablesArgs(te=te.data_ptr(), frame_indices=fi.data_ptr(), blob=blob.data_ptr(), count=len(Cs), B=B, T=T,
                         te_stride=te_stride, max_C=max(Cs))
    N_.call("fdm_rpe_tables", a, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    for ref, out_op, out_f32 in refs:
        assert rel(out_op.float(), ref) <= 4e-3, rel(out_op.float(), ref)
        if out_f32 is not None:
            assert rel(out_f32, ref) <= 2e-4, rel(out_f32, ref)


def _nl_inputs(B, T, HW, Cout, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    C = 128
    dev = "cuda"
    # activations with per-channel offsets and scales, so that the normalisation actually matters
    x = torch.randn(B * T, HW, C, device=dev, generator=g) * (0.5 + torch.rand(C, device=dev, generator=g)) + torch.randn(C, device=dev, generator=g)
    gamma = 1 + 0.3 * torch.randn(C, device=dev, generator=g)
    beta = 0.3 * torch.randn(C, device=dev, generator=g)
    w = torch.randn(Cout, C, device=dev, generator=g) / C ** 0.5
    bias = 0.2 * torch.randn(Cout, device=dev, generator=g)
    return x, gamma, beta, w, bias, g


def _frame_gn(x, gamma, beta, eps):
    # GroupNorm32 per frame over (C/32 channels x HW): x [N][HW][C]
    return F.group_norm(x.permute(0, 2, 1).double(), 32, gamma.double(), beta.double(), eps).permute(0, 2, 1).float()


def _temporal_gn(x, B, T, gamma, beta, eps):
    # rpe.py:135-137: statistics over (C/32 channels x T frames) per (video, pixel)
    N, HW, C = x.shape
    v = x.view(B, T, HW, C).permute(0, 2, 3, 1).reshape(B * HW, C, T).double()
    v = F.group_norm(v, 32, gamma.double(), beta.double(), eps)
    return v.view(B, HW, C, T).permute(0, 3, 1, 2).reshape(N, HW, C).float()


def _frame_stats(x):
    return torch.stack([x.double().sum(1), (x.double() ** 2).sum(1)], dim=-1).contiguous()  # [N][C][2]


NL_SHAPES = [(8, 20, 256), (2, 5, 64), (3, 7, 16), (1, 40, 64), (2, 2, 256), (1, 1, 64), (5, 20, 16)]


@pytest.mark.parametrize("B,T,HW", NL_SHAPES)
@pytest.mark.parametrize("a_mode", [1, 2])
def test_norm_linear_qkv(B, T, HW, a_mode):
    """fdm_norm_linear (lin_tc.cu): GroupNorm (per frame from the producer's sums / temporal, in the tile) in the operand path of
    the C -> 3C linear, against torch group_norm -> bf16 -> linear on the same bf16-rounded weights."""
    import ctypes
    from improved_diffusion import _native as N_
    C, Cout, eps = 128, 384, 1e-5
    x, gamma, beta, w, bias, _ = _nl_inputs(B, T, HW, Cout, seed=B * 1000 + T * 10 + a_mode)
    wp = w.to(torch.bfloat16).contiguous()
    y = torch.full((B * T, HW, Cout), float("nan"), device="cuda", dtype=torch.bfloat16)
    stats = _frame_stats(x)
    tstats = torch.full((B, HW, 32, 2), float("nan"), device="cuda")
    a = N_.NormLinearArgs(x=x.data_ptr(), stats=stats.data_ptr() if a_mode == 1 else None,
                          tstats=tstats.data_ptr() if a_mode == 2 else None, gamma=gamma.data_ptr(), beta=beta.data_ptr(),
                          w=wp.data_ptr(), bias=bias.data_ptr(), y_op=y.data_ptr(),
                          B=B, T=T, HW=HW, K=C, Cout=Cout, a_mode=a_mode, eps=eps)
    if a_mode == 2 and T > 20:
        # the temporal form keeps a pixel's T rows in registers: longer clips run fdm_temporal_gn + fdm_conv
        assert not N_.lib().fdm_norm_linear_supported(ctypes.byref(a))
        return
    assert N_.lib().fdm_norm_linear_supported(ctypes.byref(a))
    N_.call("fdm_norm_linear", a, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    xn = _frame_gn(x, gamma, beta, eps) if a_mode == 1 else _temporal_gn(x, B, T, gamma, beta, eps)
    ref = xn.to(torch.bfloat16).float() @ wp.float().t() + bias
    assert torch.isfinite(y.float()).all()
    e = rel(y.float(), ref)
    assert e <= 5e-3, e   # bf16 output rounding (2^-9) + operand rounding flips at the bf16 boundary
    if a_mode == 2:
        v = x.view(B, T, HW, 32, 4).permute(0, 2, 3, 1, 4).reshape(B, HW, 32, T * 4).double()
        mean, var = v.mean(-1), v.var(-1, unbiased=False)
        assert rel(tstats[..., 0], mean.float()) <= 1e-5
        assert rel(tstats[..., 1], (var + eps).rsqrt().float()) <= 1e-4


def run_proj_recomputed_gn(B, T, HW, resid_norm):
    """fdm_conv in the proj_out form with resid_norm 2 | 3 on the inputs of _nl_inputs.  Returns (y, y_op, stats, torch reference)."""
    from improved_diffusion import _native as N_
    C, eps = 128, 1e-5
    x, gamma, beta, w, bias, g = _nl_inputs(B, T, HW, C, seed=B * 1000 + T * 10 + resid_norm + 5)
    M = B * T * HW
    side = int(HW ** 0.5)
    h = torch.randn(M, C, device="cuda", generator=g).to(torch.bfloat16)
    wp = w.to(torch.bfloat16).contiguous()
    y = torch.full((M, C), float("nan"), device="cuda")
    yop = torch.full((M, C), float("nan"), device="cuda", dtype=torch.bfloat16)
    ostats = torch.zeros(B * T, C, 2, device="cuda", dtype=torch.float64)
    stats = _frame_stats(x)
    r = (_temporal_gn(x, B, T, gamma, beta, eps) if resid_norm == 2 else _frame_gn(x, gamma, beta, eps)).reshape(M, C)
    v = x.view(B, T, HW, 32, 4).permute(0, 2, 3, 1, 4).reshape(B, HW, 32, T * 4).double()
    tstats = torch.stack([v.mean(-1), (v.var(-1, unbiased=False) + eps).rsqrt()], dim=-1).float().contiguous()
    a = N_.ConvArgs(a0=h.data_ptr(), w0=wp.data_ptr(), a1=None, w1=None, bias=bias.data_ptr(), resid=x.data_ptr(), y_f32=y.data_ptr(),
                    y_op=yop.data_ptr(), stats=ostats.data_ptr(), N=B * T, Hin=side, Win=side, C0=C, C1=0, Cout=C, ksize=1, stride=1,
                    upsample=0, a_dtype=N_.BF16, op_dtype=N_.BF16, out_nchw=0, engine=N_.CONV_TC, resid_norm=resid_norm, rn_T=T,
                    rn_eps=eps, rn_tstats=tstats.data_ptr(), rn_stats=stats.data_ptr(), rn_gamma=gamma.data_ptr(),
                    rn_beta=beta.data_ptr())
    N_.call("fdm_conv", a, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return y, yop, ostats, h.float() @ wp.float().t() + bias + r


@pytest.mark.parametrize("B,T,HW", NL_SHAPES)
@pytest.mark.parametrize("resid_norm", [2, 3])
def test_conv_proj_recomputed_groupnorm_residual(B, T, HW, resid_norm):
    """fdm_conv (per-tap tcgen05 engine), proj_out form: the residual is GroupNorm(x) RECOMPUTED in the epilogue — temporal GN from
    the saved (mean, rstd) pairs (resid_norm 2) / per-frame GN from the sums (resid_norm 3) — instead of a normalised fp32 copy
    (rpe.py:136,173); fp32 + bf16 outputs and the GroupNorm statistics of the result."""
    y, yop, ostats, ref = run_proj_recomputed_gn(B, T, HW, resid_norm)
    assert rel(y, ref) <= 2e-5, rel(y, ref)
    assert rel(yop.float(), ref) <= 4e-3
    rs = _frame_stats(ref.view(B * T, HW, -1))
    assert rel(ostats, rs) <= 1e-5, rel(ostats, rs)


def _fdm_kernels(fn):
    """names of the library's kernels (namespace fdm) that torch.profiler records while fn() runs"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if "fdm::" in e.name]


def _run_conv_case(case, **kw):
    """run_conv (tcgen05 engines) on random operands of a (N, H, W, C0, Cout, k) case"""
    from improved_diffusion import _native as N_
    N, H, W, C0, Co, k = case
    g = torch.Generator(device="cuda").manual_seed(sum(case))
    x = torch.randn(N, H, W, C0, device="cuda", generator=g).to(torch.bfloat16)
    w = torch.randn(Co, C0, k, k, device="cuda", generator=g) / (C0 * k * k) ** 0.5
    bias = 0.1 * torch.randn(Co, device="cuda", generator=g)
    return run_conv(x, w, bias, engine=N_.CONV_TC, want_op=True, **kw)


def _run_head_case(case):
    from improved_diffusion import _native as N_
    N, H, W, C0, Co = case
    g = torch.Generator(device="cuda").manual_seed(sum(case))
    x = torch.randn(N, H, W, C0, device="cuda", generator=g).to(torch.bfloat16)
    w = torch.randn(Co, C0, 3, 3, device="cuda", generator=g) / (9 * C0) ** 0.5
    return run_head_conv(x, pack_tc(w), 0.1 * torch.randn(Co, device="cuda", generator=g), Co, N_.CONV_TC)


# route -> (launch, pattern of the demangled kernel name: template arguments <BN, TPI, CG, UP> of the halo kernel, <BN, RN> of the
# per-tap kernel), with case shapes of test_head_conv_vs_torch, test_conv_tc_vs_torch, test_wide_pointwise_vs_torch and
# test_conv_proj_recomputed_groupnorm_residual
CONV_ROUTES = {
    "head": (lambda: _run_head_case((20, 32, 32, 64, 4)), r"\bconv_head_kernel\("),
    "halo": (lambda: _run_conv_case((5, 32, 32, 64, 64, 3)), r"\bconv_halo_kernel<\d+, \d+, 1, false>"),
    "halo_cta_pair": (lambda: _run_conv_case((80, 32, 32, 192, 64, 3)), r"\bconv_halo_kernel<\d+, \d+, 2, false>"),
    "halo_pointwise": (lambda: _run_conv_case((16, 16, 16, 384, 1152, 1), want_stats=False), r"\bconv_halo_kernel<\d+, \d+, 1, false>"),
    "tap_3x3_8x8": (lambda: _run_conv_case((5, 8, 8, 128, 128, 3)), r"\bconv_tc_kernel<\d+, false>"),
    "tap_1x1_resid_norm": (lambda: run_proj_recomputed_gn(8, 20, 256, 2), r"\bconv_tc_kernel<\d+, true>"),
}


@pytest.mark.parametrize("route", list(CONV_ROUTES))
def test_conv_dispatch_runs_the_expected_kernel(route):
    """fdm_conv with engine FDM_CONV_TC picks one of three tcgen05 kernels by shape, and a kernel that refuses a shape (including a
    tensor map the driver rejects) hands it on to the per-tap kernel, which computes the same result more slowly.  The result
    tests cannot tell the kernels apart: this pins which one each route launches, and that it is the only launch."""
    run, kernel = CONV_ROUTES[route]
    names = _fdm_kernels(run)
    assert len(names) == 1 and re.search(kernel, names[0]), names
