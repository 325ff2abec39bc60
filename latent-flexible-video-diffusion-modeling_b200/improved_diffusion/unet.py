"""
UNetVideoModel — the FDM video denoiser with the reference's constructor, parameter names and call
signature (improved_diffusion/unet.py:246-464), executed by the sm_100a kernel schedule of engine.py.

The module tree below is a *parameter layout*: it reproduces the reference's registration order so that
state_dict keys (SURVEY §8b: 390 tensors for the 32-px / num_res_blocks=1 model) and default
initialisation match, and so that reference checkpoints load with strict=True.  `forward` does not walk
the modules; it hands (x, x0, t, frame_indices, masks) to a `DenoiserEngine`, which compiles one flat
kernel schedule per input shape (NHWC activations, fused GroupNorm/SiLU/FiLM, implicit-GEMM convs,
RPE attention kernels) and replays it.
"""
import os

import torch as th
import torch.nn as nn

from .nn import SiLU, conv_nd, linear, normalization, zero_module
from .rpe import RPEAttention


class TimestepBlock(nn.Module):
    """Marker: a block that consumes the timestep embedding (unet.py:24-33)."""


class TimestepEmbedAttnThingsSequential(nn.Sequential, TimestepBlock):
    """Container of one U-Net stage (unet.py:36-57); dispatch happens in the engine's schedule compiler."""


class Upsample(nn.Module):
    def __init__(self, channels, use_conv, dims=2):
        super().__init__()
        self.channels, self.use_conv, self.dims = channels, use_conv, dims
        if use_conv:
            self.conv = conv_nd(dims, channels, channels, 3, padding=1)


class Downsample(nn.Module):
    def __init__(self, channels, use_conv, dims=2):
        super().__init__()
        self.channels, self.use_conv, self.dims = channels, use_conv, dims
        if not use_conv:
            raise NotImplementedError("avg-pool downsampling is never selected by create_model (conv_resample=True)")
        self.op = conv_nd(dims, channels, channels, 3, stride=2 if dims != 3 else (1, 2, 2), padding=1)


class ResBlock(TimestepBlock):
    def __init__(self, channels, emb_channels, dropout, out_channels=None, use_conv=False,
                 use_scale_shift_norm=False, dims=2, use_checkpoint=False):
        super().__init__()
        self.channels, self.emb_channels, self.dropout = channels, emb_channels, dropout
        self.out_channels = out_channels or channels
        self.use_conv, self.use_checkpoint, self.use_scale_shift_norm = use_conv, use_checkpoint, use_scale_shift_norm
        co = self.out_channels
        self.in_layers = nn.Sequential(normalization(channels), SiLU(), conv_nd(dims, channels, co, 3, padding=1))
        self.emb_layers = nn.Sequential(SiLU(), linear(emb_channels, 2 * co if use_scale_shift_norm else co))
        self.out_layers = nn.Sequential(normalization(co), SiLU(), nn.Dropout(p=dropout),
                                        zero_module(conv_nd(dims, co, co, 3, padding=1)))
        if co == channels:
            self.skip_connection = nn.Identity()
        else:
            self.skip_connection = conv_nd(dims, channels, co, 3 if use_conv else 1, padding=1 if use_conv else 0)


class FactorizedAttentionBlock(nn.Module):
    def __init__(self, channels, num_heads, use_rpe_net, time_embed_dim=None, use_checkpoint=False):
        super().__init__()
        self.channels, self.num_heads = channels, num_heads
        self.spatial_attention = RPEAttention(channels=channels, num_heads=num_heads, use_checkpoint=use_checkpoint,
                                              use_rpe_q=False, use_rpe_k=False, use_rpe_v=False)
        self.temporal_attention = RPEAttention(channels=channels, num_heads=num_heads, use_checkpoint=use_checkpoint,
                                               time_embed_dim=time_embed_dim, use_rpe_net=use_rpe_net)


class UNetVideoModel(nn.Module):
    def __init__(self, in_channels, model_channels, out_channels, num_res_blocks, attention_resolutions,
                 image_size=None, dropout=0, channel_mult=(1, 2, 4, 8), conv_resample=True, dims=2,
                 use_checkpoint=False, num_heads=1, num_heads_upsample=-1, use_scale_shift_norm=False,
                 use_rpe_net=False):
        super().__init__()
        if dims != 2:
            raise NotImplementedError("the sm_100a schedule implements the 2-D per-frame U-Net used by FDM")
        if num_heads_upsample == -1:
            num_heads_upsample = num_heads
        self.in_channels = in_channels + 1  # + observed-frame indicator channel
        self.model_channels, self.out_channels = model_channels, out_channels
        self.num_res_blocks, self.attention_resolutions = num_res_blocks, attention_resolutions
        self.dropout, self.channel_mult, self.conv_resample = dropout, channel_mult, conv_resample
        self.use_checkpoint, self.num_heads, self.num_heads_upsample = use_checkpoint, num_heads, num_heads_upsample
        self.use_rpe_net, self.use_scale_shift_norm, self.image_size = use_rpe_net, use_scale_shift_norm, image_size
        mc, ted = model_channels, model_channels * 4
        Seq = TimestepEmbedAttnThingsSequential
        res = lambda ci, co: ResBlock(ci, ted, dropout, out_channels=co, dims=dims, use_checkpoint=use_checkpoint,
                                      use_scale_shift_norm=use_scale_shift_norm)
        att = lambda c, h: FactorizedAttentionBlock(c, use_checkpoint=use_checkpoint, num_heads=h,
                                                    use_rpe_net=use_rpe_net, time_embed_dim=ted)

        self.time_embed = nn.Sequential(linear(mc, ted), SiLU(), linear(ted, ted))
        self.input_blocks = nn.ModuleList([Seq(conv_nd(dims, self.in_channels, mc, 3, padding=1))])
        skip_chans, ch, ds = [mc], mc, 1
        last = len(channel_mult) - 1
        for level, mult in enumerate(channel_mult):
            for _ in range(num_res_blocks):
                stage = [res(ch, mult * mc)]
                ch = mult * mc
                if ds in attention_resolutions:
                    stage.append(att(ch, num_heads))
                self.input_blocks.append(Seq(*stage))
                skip_chans.append(ch)
            if level != last:
                self.input_blocks.append(Seq(Downsample(ch, conv_resample, dims=dims)))
                skip_chans.append(ch)
                ds *= 2
        self.middle_block = Seq(res(ch, ch), att(ch, num_heads), res(ch, ch))
        self.output_blocks = nn.ModuleList([])
        for level in range(last, -1, -1):
            mult = channel_mult[level]
            for i in range(num_res_blocks + 1):
                stage = [res(ch + skip_chans.pop(), mc * mult)]
                ch = mc * mult
                if ds in attention_resolutions:
                    stage.append(att(ch, num_heads_upsample))
                if level and i == num_res_blocks:
                    stage.append(Upsample(ch, conv_resample, dims=dims))
                    ds //= 2
                self.output_blocks.append(Seq(*stage))
        self.out = nn.Sequential(normalization(ch), SiLU(), zero_module(conv_nd(dims, mc, out_channels, 3, padding=1)))
        self._engines = {}
        self.precision = "bf16"  # "bf16": tcgen05 bf16 GEMM operands (2e-2 contract); "fp32": exact CUDA-core path (1e-4)

    # -- dtype plumbing of the reference (unet.py:405-426).  --use_fp16 crashes in the reference (SURVEY §2 #11);
    #    bf16 operand precision is selected with `model.precision` instead.
    def convert_to_fp16(self):
        raise NotImplementedError("use model.precision = 'bf16' (fp16 conversion is broken upstream, fp16_util.py:9-15)")

    def convert_to_fp32(self):
        self.precision = "fp32"

    @property
    def inner_dtype(self):
        return next(self.input_blocks.parameters()).dtype

    def engine(self, precision=None):
        from .engine import DenoiserEngine
        precision = precision or self.precision
        if precision not in self._engines:
            self._engines[precision] = DenoiserEngine(self, precision)
        return self._engines[precision]

    def forward(self, x, *, x0, timesteps, frame_indices=None, obs_mask=None, latent_mask=None,
                return_attn_weights=False):
        """(eps [B,T,C_out,H,W] fp32, attns) — same contract as unet.py:428-464."""
        if return_attn_weights:
            # attention-map logging of TrainLoop.log_samples (train_util.py:451-463).  bf16 mode on CUDA, no gradients: the
            # tcgen05 attention kernels accumulate the head-averaged maps themselves (materialising variants: attn_tc.cu,
            # attn_temporal_tc.cu).  Otherwise (fp32 parity mode, CPU, inside autograd): PyTorch expression of the same network.
            from .engine import NativeShapeError
            if x.is_cuda and self.precision == "bf16" and not th.is_grad_enabled():
                try:
                    return self.engine().forward(x, x0, timesteps, frame_indices, obs_mask, latent_mask, collect_attn=True)
                except NativeShapeError:
                    pass
            from .autograd_path import differentiable_forward
            attns = {"spatial": [], "temporal": [], "mixed": []}
            out = differentiable_forward(self, x, x0, timesteps, frame_indices, obs_mask, latent_mask, attns=attns)
            return out, attns
        needs_grad = th.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters()))
        # the native backward differentiates w.r.t. the PARAMETERS (what training needs); a caller that wants d(eps)/d(x) or
        # d(eps)/d(x0) (guidance-style use) gets the autograd expression below instead of silently missing input gradients
        wants_input_grad = x.requires_grad or (isinstance(x0, th.Tensor) and x0.requires_grad)
        if needs_grad and x.is_cuda and not wants_input_grad and os.environ.get("FDM_TRAIN_ENGINE", "native") != "autograd":
            # training on the GPU: native forward AND backward kernel schedules behind one autograd node (engine._DenoiserFn)
            return self.engine().forward_train(x, x0, timesteps, frame_indices, obs_mask, latent_mask), None
        if needs_grad:
            # NOT a silent fallback: the PyTorch-autograd expression of the same network (autograd_path.py) only runs when asked
            # for — FDM_TRAIN_ENGINE=autograd (the A/B arm of the benchmark and of the parity tests) or FDM_ALLOW_TORCH_TRAIN=1
            # (host-side CPU tests, the drop-in TrainLoop check, gradients w.r.t. the inputs)
            if os.environ.get("FDM_TRAIN_ENGINE") != "autograd" and os.environ.get("FDM_ALLOW_TORCH_TRAIN") != "1":
                why = "on a CPU tensor" if not x.is_cuda else "with gradients w.r.t. the inputs"
                raise RuntimeError(f"UNetVideoModel training {why} is not served by the sm_100a kernels (native training "
                                   "differentiates w.r.t. the parameters, on a CUDA device; there is no silent CPU / PyTorch "
                                   "fallback).  Set FDM_ALLOW_TORCH_TRAIN=1 to run the PyTorch-autograd expression instead.")
            from .autograd_path import differentiable_forward
            return differentiable_forward(self, x, x0, timesteps, frame_indices, obs_mask, latent_mask), None
        if not x.is_cuda:
            raise RuntimeError("UNetVideoModel inference runs on sm_100a kernels only: move the model and inputs to a CUDA "
                               "device (there is no CPU fallback)")
        eps = self.engine().forward(x, x0, timesteps, frame_indices, obs_mask, latent_mask)
        return eps, None
