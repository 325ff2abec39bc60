"""
ResBlock dropout in native training (-m gpu): the nn.Dropout between SiLU and the second conv of every ResBlock
(reference unet.py:167,203-206) is a Philox keep-mask drawn inside the second GroupNorm-apply launch (fdm_gn_apply) and drawn
again inside its backward (fdm_gn_bwd); the mask is never stored.  Checked here: eval mode ignores dropout bit for bit; the
masked operand conv2 reads (`res_a2` in the training plan's arena) has the nn.Dropout semantics; gradients equal those of the
PyTorch-autograd expression of the network with each nn.Dropout replaced by the mask the native forward drew; and the
NativeTrainStep drop-in trains with dropout.
"""
import math

import pytest
import torch
import torch.nn as nn

from oracle import fdm_oracle as O

pytestmark = pytest.mark.gpu
PIXEL = dict(diffusion_space="pixel", pre_encoded=False, pre_encoded_stats_dict=None)
CFG1 = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32)
CFG2 = dict(image_size=32, in_channels=4, num_channels=64, num_res_blocks=1, diffusion_steps=1000)
NRB2 = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=2, diffusion_steps=32)


def build(over, precision, dropout, seed=1):
    from improved_diffusion.script_util import create_model_and_diffusion, model_and_diffusion_defaults
    d = model_and_diffusion_defaults()
    d.update(over)
    d.update(dropout=dropout, diffusion_space_kwargs=dict(PIXEL))
    model, diffusion = create_model_and_diffusion(**d)
    model.load_state_dict(O.init_state_dict(O.make_cfg(**over), seed=seed), strict=True)
    model.to("cuda").train()
    model.precision = precision
    return model, diffusion


def res_blocks(model):
    from improved_diffusion.unet import ResBlock
    return [layer for blk in [*model.input_blocks, model.middle_block, *model.output_blocks] for layer in blk
            if isinstance(layer, ResBlock)]


def set_dropout(model, p):
    model.dropout = p
    for rb in res_blocks(model):
        rb.out_layers[2].p = p


def inputs(over, B, T, n_obs, seed=5):
    inp = O.synthetic_inputs(O.make_cfg(**over), B, T, n_obs, seed=seed, video_len=60)
    return {k: v.cuda() for k, v in inp.items() if k in ("x", "x0", "frame_indices", "obs_mask", "latent_mask")}


def train_forward(model, inp, t):
    eps, _ = model(inp["x"], x0=inp["x0"], timesteps=t, frame_indices=inp["frame_indices"], obs_mask=inp["obs_mask"],
                   latent_mask=inp["latent_mask"])
    return eps


def a2_operands(model):
    """conv2's operand of every ResBlock (NHWC, op dtype) from the training plan's arena, in ResBlock order."""
    P = next(iter(model.engine().train_plans.values()))
    dt = torch.bfloat16 if model.precision == "bf16" else torch.float32
    torch.cuda.synchronize()
    return [P.view(b, (P.B * P.T, H, W, C), dt).clone() for b, C, H, W in P.res_a2]


def zero_conv2(model):
    """ResBlock outputs then do not depend on the dropout: every block's pre-dropout values are the same at any p."""
    with torch.no_grad():
        for rb in res_blocks(model):
            rb.out_layers[3].weight.zero_()
            rb.out_layers[3].bias.zero_()


@pytest.mark.parametrize("over,B,T,n_obs", [(CFG1, 1, 5, 2), (CFG2, 1, 5, 3)], ids=["cfg1", "cfg2"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_eval_mode_ignores_dropout(over, B, T, n_obs, precision):
    """nn.Dropout is the identity in eval mode: eps of a dropout=0.1 model equals that of the same weights built with dropout=0."""
    inp = inputs(over, B, T, n_obs)
    t = torch.tensor([7] * B, device="cuda")
    eps = []
    for p in (0.0, 0.1):
        model, _ = build(over, precision, p)
        model.eval()
        with torch.no_grad():
            eps.append(train_forward(model, inp, t))
    assert torch.equal(eps[0], eps[1])


@pytest.mark.parametrize("p", [0.1, 0.5])
def test_mask_semantics(p):
    """Dropped entries are zero, kept ones are the p = 0 value times 1 / (1 - p), and the dropped fraction over all ResBlocks is
    within 6 binomial sigmas of p (fp32 operands; conv2 zeroed so that dropout upstream does not change a block's input)."""
    model, _ = build(CFG1, "fp32", 0.0)
    zero_conv2(model)
    inp = inputs(CFG1, 1, 5, 2)
    t = torch.tensor([11], device="cuda")
    train_forward(model, inp, t)
    ref = a2_operands(model)
    set_dropout(model, p)
    train_forward(model, inp, t)
    got = a2_operands(model)
    assert len(got) == len(res_blocks(model))
    n = dropped = 0
    for r, g in zip(ref, got):
        live = r != 0
        kept = live & (g != 0)
        assert torch.equal(g[~live], r[~live])
        expect = r[kept].double() / (1 - p)
        assert torch.allclose(g[kept].double(), expect, rtol=5e-7, atol=0), float(((g[kept] - expect) / expect).abs().max())
        n += int(live.sum())
        dropped += int((live & (g == 0)).sum())
    frac, sigma = dropped / n, math.sqrt(p * (1 - p) / n)
    print(f"p = {p}: dropped {dropped} of {n} = {frac:.5f} ({(frac - p) / sigma:+.2f} sigma)")
    assert abs(frac - p) <= 6 * sigma


def test_mask_varies_and_repeats_with_the_seed():
    """Masks differ between two steps and between ResBlocks of the same shape; after torch.manual_seed(s) a fresh model repeats
    them, and another seed does not."""
    inp = inputs(CFG1, 1, 5, 2)
    t = torch.tensor([11], device="cuda")

    def masks(seed, steps=2):
        torch.manual_seed(seed)
        model, _ = build(CFG1, "fp32", 0.5)
        out = []
        for _ in range(steps):  # eager forward, then the captured graph
            train_forward(model, inp, t)
            out.append([a != 0 for a in a2_operands(model)])
        return out

    a, b, c = masks(3), masks(3), masks(4)
    assert all(torch.equal(x, y) for sa, sb in zip(a, b) for x, y in zip(sa, sb))
    differ = lambda x, y: float((x != y).float().mean())
    for k in range(len(a[0])):
        assert 0.4 < differ(a[0][k], a[1][k]) < 0.6, k   # independent masks at p = 0.5 disagree on half the entries
        assert 0.4 < differ(a[0][k], c[0][k]) < 0.6, k
    same_shape = [(i, j) for i in range(len(a[0])) for j in range(i) if a[0][i].shape == a[0][j].shape]
    assert same_shape
    for i, j in same_shape:
        assert 0.4 < differ(a[0][i], a[0][j]) < 0.6, (i, j)


def test_dropout_one_gives_zeros_and_finite_gradients():
    model, diffusion = build(CFG1, "fp32", 1.0)
    inp = inputs(CFG1, 1, 5, 2)
    t = torch.tensor([11], device="cuda")
    terms = diffusion.training_losses(model, inp["x0"], t, model_kwargs={k: inp[k] for k in ("x0", "frame_indices", "obs_mask",
                                                                                              "latent_mask")},
                                      latent_mask=inp["latent_mask"], eval_mask=inp["latent_mask"])
    terms["loss"].mean().backward()
    assert all(int((a != 0).sum()) == 0 for a in a2_operands(model))
    assert all(torch.isfinite(p.grad).all() for p in model.parameters())
    assert all(float(rb.out_layers[3].weight.grad.abs().max()) == 0 for rb in res_blocks(model))


class FixedDropout(nn.Module):
    """nn.Dropout with a given keep mask (NCHW bool), scaled like nn.Dropout in train mode."""

    def __init__(self, keep, p):
        super().__init__()
        self.keep, self.scale = keep, 1.0 / (1.0 - p)

    def forward(self, h):
        return h * (self.keep.to(h.dtype) * self.scale)


def _grad_errors(got, ref):
    """rel-L2 per parameter, denominator floored at 5 % of the median gradient norm (analytically zero gradients carry only
    rounding noise on either side)."""
    floor = 5e-2 * float(torch.stack([v.double().norm() for v in ref.values()]).median())
    return sorted(((float((got[k].double() - ref[k].double()).norm() / max(float(ref[k].double().norm()), floor)), k)
                   for k in ref), reverse=True)


def _train_grads(model, diffusion, inp, t, noise, engine, monkeypatch, precision):
    monkeypatch.setenv("FDM_TRAIN_ENGINE", engine)
    monkeypatch.setattr(model, "precision", precision)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    model.zero_grad(set_to_none=True)
    kw = {k: inp[k] for k in ("x0", "frame_indices", "obs_mask", "latent_mask")}
    terms = diffusion.training_losses(model, inp["x0"], t, model_kwargs=kw, noise=noise, latent_mask=inp["latent_mask"],
                                      eval_mask=inp["latent_mask"])
    terms["loss"].mean().backward()
    torch.cuda.synchronize()
    return terms["loss"].detach().cpu(), {k: p.grad.detach().cpu().clone() for k, p in model.named_parameters()}


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("over,B,T,n_obs", [(CFG2, 1, 5, 3), (NRB2, 2, 5, 2)], ids=["cfg2", "nrb2"])
def test_gradients_match_autograd_with_the_same_masks(over, B, T, n_obs, precision, monkeypatch):
    """Native gradients with dropout = 0.1 against torch.autograd over the PyTorch expression of the network, its nn.Dropout
    modules replaced by the masks the native forward drew.  fp32: the bounds of the dropout-free whole-network parity test
    (test_gpu_parity.py: loss 1e-5, worst parameter 2e-4; a mask that the backward regenerated wrongly shows up as errors of order
    1); bf16: no worse than 1.5x torch's own autocast-bf16 backward (same masks) against the fp32 autograd."""
    p = 0.1
    model, diffusion = build(over, precision, p)
    inp = inputs(over, B, T, n_obs)
    g = torch.Generator().manual_seed(11)
    t = torch.randint(0, diffusion.num_timesteps, (B,), generator=g).cuda()
    noise = torch.randn(inp["x0"].shape, generator=g).cuda()
    loss_n, gn_ = _train_grads(model, diffusion, inp, t, noise, "native", monkeypatch, precision)
    keep = [(a != 0).permute(0, 3, 1, 2).contiguous() for a in a2_operands(model)]
    drop_frac = 1 - sum(float(k.float().sum()) for k in keep) / sum(k.numel() for k in keep)
    assert abs(drop_frac - p) < 0.02, drop_frac
    for rb, k in zip(res_blocks(model), keep):
        rb.out_layers[2] = FixedDropout(k, p)
    loss_a, ga_ = _train_grads(model, diffusion, inp, t, noise, "autograd", monkeypatch, "fp32")
    assert all(torch.isfinite(v).all() for v in gn_.values())
    errs = _grad_errors(gn_, ga_)
    if precision == "fp32":
        print(f"dropout native vs autograd [fp32] worst {errs[0][0]:.3e} at {errs[0][1]}, median {errs[len(errs) // 2][0]:.3e}")
        assert O.rel_l2(loss_n, loss_a) <= 1e-5, O.rel_l2(loss_n, loss_a)
        assert errs[0][0] <= 2e-4, errs[:5]
    else:
        loss_c, gc_ = _train_grads(model, diffusion, inp, t, noise, "autograd", monkeypatch, "bf16")
        cal = _grad_errors(gc_, ga_)
        cal_by = {k: e for e, k in cal}
        worst_c, med_c = cal[0][0], cal[len(cal) // 2][0]
        worst_n, med_n = errs[0][0], errs[len(errs) // 2][0]
        print(f"dropout bf16 vs fp32 autograd: native worst {worst_n:.3e} ({errs[0][1]}) median {med_n:.3e} | autocast worst "
              f"{worst_c:.3e} ({cal[0][1]}) median {med_c:.3e}")
        assert O.rel_l2(loss_n, loss_a) <= max(1.5 * O.rel_l2(loss_c, loss_a), 5e-3)
        assert worst_n <= 1.5 * worst_c, (errs[:3], cal[:3])
        assert med_n <= 1.5 * med_c, (med_n, med_c)
        bad = [(e, k, cal_by[k]) for e, k in errs if e > 1.5 * max(cal_by[k], med_c)]
        assert not bad, bad[:5]


def test_native_train_step_runs_with_dropout(monkeypatch):
    """The NativeTrainStep drop-in (masks, gather, upload, native forward + backward, FlatAdamW) takes two optimizer steps with
    dropout = 0.1; the weights move and every logged value is finite."""
    import numpy as np
    from improved_diffusion.train_step import NativeTrainStep
    monkeypatch.setenv("FDM_TRAIN_ENGINE", "native")
    model, diffusion = build(CFG1, "bf16", 0.1)
    runner = NativeTrainStep(model, diffusion, lr=1e-4, max_frames=5, ema_rate="0.9999")
    torch.manual_seed(7)
    np.random.seed(7)
    g = torch.Generator().manual_seed(3)
    before = [p.detach().clone() for p in model.parameters()]
    logs = [runner.run_step(torch.randn(2, 15, 4, 32, 32, generator=g).clamp(-1, 1),
                            torch.randn(2, 15, 4, 32, 32, generator=g).clamp(-1, 1)) for _ in range(2)]
    assert [r["step"] for r in logs] == [0, 1]
    assert all(math.isfinite(v) for r in logs for v in r.values())
    assert next(iter(model.engine().train_plans.values())).drop_p == 0.1
    assert any(not torch.equal(a, b.detach()) for a, b in zip(before, model.parameters()))
