"""
GPU parity (run with -m gpu on the B200 box): the sm_100a path, called through the reference-shaped Python API
(which binds the C-ABI of include/fdm_b200.h), against (a) the committed reference outputs in tests/golden/ and
(b) the CPU oracle on the same seeded inputs.  Tolerances are north_star's: eps rel-L2 <= 1e-4 in fp32 mode,
<= 2e-2 in bf16 mode.  /root/reference is never read here.
"""
import pytest
import torch

from oracle import fdm_oracle as O

pytestmark = pytest.mark.gpu
PIXEL = dict(diffusion_space="pixel", pre_encoded=False, pre_encoded_stats_dict=None)
TOL = {"fp32": 1e-4, "bf16": 2e-2}


def build(over, precision, seed=1):
    from improved_diffusion.script_util import create_model_and_diffusion, model_and_diffusion_defaults
    d = model_and_diffusion_defaults()
    d.update(over)
    d["diffusion_space_kwargs"] = dict(PIXEL)
    model, diffusion = create_model_and_diffusion(**d)
    cfg = O.make_cfg(**over)
    sd = O.init_state_dict(cfg, seed=seed)
    model.load_state_dict(sd, strict=True)
    model.to("cuda").eval()
    model.precision = precision
    return model, diffusion, cfg, sd


def cuda_kw(inp):
    return {k: inp[k].cuda() for k in ("x0", "frame_indices", "obs_mask", "latent_mask")}


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", ["fwd_cfg1", "fwd_pad", "fwd_img64", "fwd_nc64"])
def test_eps_matches_reference_golden(golden, name, precision):
    g = golden(name)
    model, _, _, _ = build(g["over"], precision)
    inp = g["inputs"]
    with torch.no_grad():
        eps, attn = model(inp["x"].cuda(), timesteps=g["model_t"].cuda(), **cuda_kw(inp))
    assert attn is None and eps.shape == g["eps"].shape and eps.dtype == torch.float32
    e = O.rel_l2(eps.cpu(), g["eps"])
    print(f"{name}[{precision}] eps rel-L2 = {e:.3e}")
    assert e <= TOL[precision]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_inputs_not_mutated_and_repeatable(golden, precision):
    g = golden("fwd_cfg1")
    model, _, _, _ = build(g["over"], precision)
    inp = g["inputs"]
    x, kw = inp["x"].cuda(), cuda_kw(inp)
    snap = [x.clone()] + [v.clone() for v in kw.values()]
    with torch.no_grad():
        a, _ = model(x, timesteps=g["model_t"].cuda(), **kw)
        b, _ = model(x, timesteps=g["model_t"].cuda(), **kw)
    assert torch.equal(x, snap[0]) and all(torch.equal(v, s) for v, s in zip(kw.values(), snap[1:]))
    # GroupNorm statistics: fixed-order fp32 partials per warp + fp64 atomics -> repeat runs agree to ~1e-16 before the
    # fp32 rounding of mean/rstd, i.e. practically bit-for-bit; bf16 mode would otherwise amplify any difference
    assert O.rel_l2(a.cpu(), b.cpu()) <= (1e-6 if precision == "fp32" else 1e-3)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_sample_loop_matches_reference_golden(golden, precision):
    """4-step respaced p_sample_loop with the reference's noise sequence (graph sampler and eager loop)."""
    g = golden("sample_cfg1")
    model, diffusion, cfg, sd = build(g["over"], precision)
    inp = g["inputs"]
    noises = [n.cuda() for n in g["noises"]]
    shape = tuple(inp["x0"].shape)
    for mode in ("graph", "eager"):
        it = iter(noises[1:])
        diffusion._noise_fn = lambda x: next(it)
        if mode == "graph":
            final, attns = diffusion.p_sample_loop(model, shape, noise=noises[0], model_kwargs=cuda_kw(inp),
                                                   latent_mask=inp["latent_mask"].cuda())
            assert attns == {}
        else:
            img = noises[0]
            for out in diffusion.p_sample_loop_progressive(model, shape, noise=noises[0], model_kwargs=cuda_kw(inp)):
                img = out["sample"]
            final = img
        e = O.rel_l2(final.cpu(), g["final"])
        print(f"sample loop [{precision}/{mode}] final rel-L2 = {e:.3e}")
        # 4 chained steps: allow the per-step tolerance to accumulate linearly
        assert e <= 4 * TOL[precision]


def test_per_step_eps_along_the_reference_trajectory(golden):
    """Feed the reference's own x_t at every step (no error accumulation) and compare eps per step."""
    g = golden("sample_cfg1")
    inp = g["inputs"]
    tab = O.Tables(O.make_cfg(**g["over"]))
    xs = [g["noises"][0]] + g["step_samples"][:-1]
    for precision in ("fp32", "bf16"):
        model, diffusion, _, _ = build(g["over"], precision)
        for k, i in enumerate(reversed(range(g["num_timesteps"]))):
            t = torch.tensor([i])
            with torch.no_grad():
                eps, _ = model(xs[k].cuda(), timesteps=O.model_timesteps(tab, t).cuda(), **cuda_kw(inp))
            e = O.rel_l2(eps.cpu(), g["step_eps"][k])
            assert e <= TOL[precision], (precision, i, e)


def test_ddpm_step_kernel_bit_exact_vs_oracle():
    """fdm_ddpm_step / fdm_q_sample reproduce the reference's fp32 association bit-for-bit."""
    _, diffusion = build(dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=1000), "fp32")[:2]
    tab = O.Tables(O.make_cfg(diffusion_steps=1000))
    g = torch.Generator().manual_seed(5)
    B = 3
    x, eps, noise = (torch.randn(B, 5, 4, 32, 32, generator=g) for _ in range(3))
    t = torch.tensor([0, 417, 999])
    ref = O.posterior_from_eps(tab, x, t, eps)
    nz = (t != 0).float().view(-1, 1, 1, 1, 1)
    ref_sample = ref["mean"] + nz * torch.exp(0.5 * ref["log_variance"]) * noise
    diffusion._noise_fn = lambda v: noise.cuda()
    fake = lambda xx, timesteps, **kw: (eps.cuda(), None)
    out = diffusion.p_sample(fake, x.cuda(), t.cuda())
    assert torch.equal(out["pred_xstart"].cpu(), ref["pred_xstart"])
    # sigma = exp(0.5*logvar) is tabulated once in fp32 on the host (same op order), so the sample is bit-exact too
    assert torch.equal(out["sample"].cpu(), ref_sample)
    xt = diffusion.q_sample(x.cuda(), t.cuda(), noise.cuda())
    assert torch.equal(xt.cpu(), O.q_sample(tab, x, t, noise))


def test_ragged_and_odd_shapes():
    """T not a multiple of anything, B > 1 with distinct frame indices per row, all-latent and all-observed rows."""
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=1000)
    model, diffusion, cfg, sd = build(over, "fp32")
    # T = 17 / 25 / 33 / 40 exercise every unrolled key-count variant of the temporal attention kernel (<= 24, 32, 40)
    for (B, T, n_obs, pads) in [(3, 7, 2, (0, 2)), (1, 2, 0, ()), (2, 3, 3, ()), (1, 11, 4, (0,)), (1, 17, 8, ()), (1, 25, 3, (0,)),
                                (1, 33, 30, ()), (1, 40, 20, (0,))]:
        inp = O.synthetic_inputs(cfg, B, T, n_obs, seed=B * 10 + T, video_len=300, pad_rows=pads)
        t = torch.tensor([(37 * (b + 1)) % 1000 for b in range(B)])
        ts = O.model_timesteps(O.Tables(cfg), t)
        with torch.no_grad():
            ref = O.unet_forward(sd, cfg, inp["x"], inp["x0"], ts, inp["frame_indices"], inp["obs_mask"], inp["latent_mask"])
            eps, _ = model(inp["x"].cuda(), timesteps=ts.cuda(), **cuda_kw(inp))
        e = O.rel_l2(eps.cpu(), ref)
        print(f"B={B} T={T} n_obs={n_obs} pads={pads}: rel-L2 {e:.3e}")
        assert e <= 1e-4


def test_single_frame_runs():
    """T == 1: the temporal GroupNorm group is C/32 = 2 values, which makes the REFERENCE itself chaotic (a 1e-6 relative
    input perturbation moves its eps by 1e-1 rel-L2, measured on the CPU oracle), so only shape/finiteness is checked."""
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=1000)
    model, _, cfg, _ = build(over, "fp32")
    inp = O.synthetic_inputs(cfg, 1, 1, 0, seed=11, video_len=300)
    with torch.no_grad():
        eps, _ = model(inp["x"].cuda(), timesteps=torch.tensor([37.0]).cuda(), **cuda_kw(inp))
    assert eps.shape == inp["x"].shape and bool(torch.isfinite(eps).all())


def test_weights_repacked_after_update():
    """load_state_dict / in-place parameter updates invalidate the packed weights (optimizer step, checkpoint resume)."""
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=1000)
    model, _, cfg, _ = build(over, "bf16")
    inp = O.synthetic_inputs(cfg, 1, 4, 2, seed=4)
    ts = torch.tensor([250.0])
    with torch.no_grad():
        a, _ = model(inp["x"].cuda(), timesteps=ts.cuda(), **cuda_kw(inp))
        sd2 = O.init_state_dict(cfg, seed=2)
        model.load_state_dict(sd2)
        b, _ = model(inp["x"].cuda(), timesteps=ts.cuda(), **cuda_kw(inp))
        ref = O.unet_forward(sd2, cfg, inp["x"], inp["x0"], ts, inp["frame_indices"], inp["obs_mask"], inp["latent_mask"])
    assert O.rel_l2(a.cpu(), b.cpu()) > 0.1
    assert O.rel_l2(b.cpu(), ref) <= 2e-2


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_training_losses_on_gpu_match_reference(golden, precision):
    """training_losses + backward on the GPU (fused q_sample kernel + the autograd path) against the reference run."""
    g = golden("train_cfg1")
    model, diffusion, cfg, sd = build(g["over"], precision)
    model.train()
    inp = g["inputs"]
    kw = cuda_kw(inp)
    terms = diffusion.training_losses(model, inp["x0"].cuda(), g["t"].cuda(), model_kwargs=kw, noise=g["noise"].cuda(),
                                      latent_mask=(1 - inp["obs_mask"]).cuda(), eval_mask=inp["latent_mask"].cuda())
    terms["loss"].mean().backward()
    tol = 1e-4 if precision == "fp32" else 3e-2
    for k in ("loss", "mse", "eval-mse"):
        assert O.rel_l2(terms[k].detach().cpu(), g["terms"][k]) <= tol, k
    grads = dict(model.named_parameters())
    assert all(p.grad is not None for p in grads.values())  # DDP find_unused_parameters=False
    for k, ref in g["grads"].items():
        e = O.rel_l2(grads[k].grad.cpu(), ref)
        # fp32: cuDNN/cuBLAS on the GPU vs the reference's CPU run; bf16: autocast gradient noise through ~45 layers
        assert e <= (3e-3 if precision == "fp32" else 2e-1), (k, e)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_wide_model_64px_vs_oracle(precision):
    """cfg5's model family (64-px 4-channel latents, nc = 128 -> C up to 512, head dims 96/128, 64-wide halo convs) on a short
    clip against the CPU oracle computed in the test."""
    over = dict(image_size=64, in_channels=4, num_channels=128, num_res_blocks=1, diffusion_steps=1000)
    model, diffusion, cfg, sd = build(over, precision)
    inp = O.synthetic_inputs(cfg, 1, 3, 1, seed=21, video_len=300, pad_rows=(0,))
    ts = torch.tensor([613.0])
    with torch.no_grad():
        ref = O.unet_forward(sd, cfg, inp["x"], inp["x0"], ts, inp["frame_indices"], inp["obs_mask"], inp["latent_mask"])
        eps, _ = model(inp["x"].cuda(), timesteps=ts.cuda(), **cuda_kw(inp))
    e = O.rel_l2(eps.cpu(), ref)
    print(f"wide 64px [{precision}] eps rel-L2 = {e:.3e}")
    assert e <= TOL[precision]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_pixel_space_128px_vs_oracle(precision):
    """cfg3's model family (128-px RGB frames: 5 resolution levels, channel_mult (1,1,2,3,4), 128-wide per-tap convs at the top,
    64/32/16-wide halo convs below) at reduced width on a 2-frame clip against the CPU oracle."""
    over = dict(image_size=128, in_channels=3, num_channels=32, num_res_blocks=1, diffusion_steps=1000)
    model, diffusion, cfg, sd = build(over, precision)
    inp = O.synthetic_inputs(cfg, 1, 2, 1, seed=31, video_len=40)
    ts = torch.tensor([250.0])
    with torch.no_grad():
        ref = O.unet_forward(sd, cfg, inp["x"], inp["x0"], ts, inp["frame_indices"], inp["obs_mask"], inp["latent_mask"])
        eps, _ = model(inp["x"].cuda(), timesteps=ts.cuda(), **cuda_kw(inp))
    e = O.rel_l2(eps.cpu(), ref)
    print(f"128px [{precision}] eps rel-L2 = {e:.3e}")
    assert eps.shape == (1, 2, 3, 128, 128) and e <= TOL[precision]


def _grad_errors(got, ref):
    """rel-L2 per parameter, with the denominator floored at 5 % of the median gradient norm: several parameters have an
    analytically ZERO gradient (conv biases feeding a GroupNorm, the rpe_k output bias: softmax shift invariance) and only
    carry rounding noise (~1e-10 in fp32, ~1e-5 in bf16 against a median norm of ~2e-3) on either side."""
    floor = 5e-2 * float(torch.stack([v.double().norm() for v in ref.values()]).median())
    return sorted(((float((got[k].double() - ref[k].double()).norm() / max(float(ref[k].double().norm()), floor)), k)
                   for k in ref), reverse=True)


def _train_grads(model, diffusion, inp, t, noise, engine, monkeypatch, precision=None):
    monkeypatch.setenv("FDM_TRAIN_ENGINE", engine)
    if precision is not None:
        monkeypatch.setattr(model, "precision", precision)
    # the autograd side must be true fp32 in BACKWARD too (cuDNN allows TF32 by default; autograd_path only pins the forward)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    model.zero_grad(set_to_none=True)
    terms = diffusion.training_losses(model, inp["x0"].cuda(), t.cuda(), model_kwargs=cuda_kw(inp), noise=noise.cuda(),
                                      latent_mask=inp["latent_mask"].cuda(), eval_mask=inp["latent_mask"].cuda())
    terms["loss"].mean().backward()
    torch.cuda.synchronize()
    return terms["loss"].detach().cpu(), {k: p.grad.detach().cpu().clone() for k, p in model.named_parameters()}


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("case", [
    # model overrides, B, T, n_obs, padded rows
    (dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32), 2, 5, 2, (1,)),
    (dict(image_size=32, in_channels=4, num_channels=64, num_res_blocks=1, diffusion_steps=1000), 1, 7, 3, ()),
    (dict(image_size=64, in_channels=3, num_channels=64, num_res_blocks=1, diffusion_steps=1000), 1, 3, 1, ()),
    # ragged shapes: three videos of four frames with padded rows; an unconditional batch (no observed frames) of 11 frames.
    # (T = 2 is not used: the temporal GroupNorm then normalises 4 values per group and amplifies rounding noise ~100x — fp32
    # gradients still agree to 2e-4, bf16 ones do not; the same ill-conditioning as T = 1 in the forward tests, DESIGN.md §5)
    (dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32), 3, 4, 1, (0, 2)),
    (dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32), 2, 11, 0, ()),
    # cfg5 family: 64-px latents, nc = 128 (C up to 512, head dims 96 / 128), K = 40 frames (the 40-key temporal kernels)
    (dict(image_size=64, in_channels=4, num_channels=128, num_res_blocks=1, diffusion_steps=1000), 1, 40, 10, ()),
    # num_res_blocks = 2 — the reference DEFAULT (script_util.py:14): two ResBlock(+attention) stages per level, three per
    # output level
    (dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=2, diffusion_steps=32), 2, 5, 2, ()),
])
def test_native_backward_matches_autograd(case, precision, monkeypatch):
    """The native backward schedule (engine._DenoiserFn: conv dgrad/wgrad, GroupNorm / attention / RPENet backward kernels) against
    torch.autograd over the PyTorch expression of the same network and parameters, on the same device.  fp32 mode: both sides are
    exact fp32 -> tight; bf16 mode: bf16 GEMM operands / operand gradients on the native side against the exact fp32 autograd."""
    over, B, T, n_obs, pad = case
    model, diffusion, cfg, sd = build(over, precision)
    model.train()
    inp = O.synthetic_inputs(cfg, B, T, n_obs, seed=5, video_len=60, pad_rows=pad)
    g = torch.Generator().manual_seed(11)
    t = torch.randint(0, diffusion.num_timesteps, (B,), generator=g)
    noise = torch.randn(inp["x0"].shape, generator=g)
    loss_n, gn_ = _train_grads(model, diffusion, inp, t, noise, "native", monkeypatch, precision)
    loss_a, ga_ = _train_grads(model, diffusion, inp, t, noise, "autograd", monkeypatch, "fp32")
    assert all(torch.isfinite(v).all() for v in gn_.values())
    errs = _grad_errors(gn_, ga_)
    if precision == "fp32":
        assert O.rel_l2(loss_n, loss_a) <= 1e-5, O.rel_l2(loss_n, loss_a)
        print(f"native vs autograd [fp32] worst grad rel-L2 = {errs[0][0]:.3e} at {errs[0][1]}, median {errs[len(errs) // 2][0]:.3e}")
        assert errs[0][0] <= 2e-4, errs[:5]
    else:
        # CALIBRATED bf16 tolerance: what does torch's own autocast-bf16 backward (cuDNN / cuBLAS bf16 GEMMs, fp32 GroupNorm and
        # softmax — the same numerical recipe) give against exact fp32 autograd on this very case?  The native bf16 gradients must
        # be no worse than 1.5x that, in the worst parameter, in the median parameter, and parameter by parameter (against the
        # larger of that parameter's own autocast error and the autocast median: single small tensors fluctuate).
        loss_c, gc_ = _train_grads(model, diffusion, inp, t, noise, "autograd", monkeypatch, "bf16")
        cal = _grad_errors(gc_, ga_)
        cal_by = {k: e for e, k in cal}
        worst_c, med_c = cal[0][0], cal[len(cal) // 2][0]
        worst_n, med_n = errs[0][0], errs[len(errs) // 2][0]
        print(f"bf16 gradients vs fp32 autograd: native worst {worst_n:.3e} ({errs[0][1]}) median {med_n:.3e} | torch autocast "
              f"worst {worst_c:.3e} ({cal[0][1]}) median {med_c:.3e} | loss err native {O.rel_l2(loss_n, loss_a):.2e} "
              f"autocast {O.rel_l2(loss_c, loss_a):.2e}")
        assert O.rel_l2(loss_n, loss_a) <= max(1.5 * O.rel_l2(loss_c, loss_a), 5e-3)
        assert worst_n <= 1.5 * worst_c, (errs[:3], cal[:3])
        assert med_n <= 1.5 * med_c, (med_n, med_c)
        bad = [(e, k, cal_by[k]) for e, k in errs if e > 1.5 * max(cal_by[k], med_c)]
        assert not bad, bad[:5]
    # a second backward of a fresh forward reproduces the first (buffers are re-zeroed, weights re-packed)
    loss_n2, gn2 = _train_grads(model, diffusion, inp, t, noise, "native", monkeypatch, precision)
    # fp32 atomics (RPE-table pixel sums, temporal-GN parameter sums) make the last bits run-dependent; in bf16 mode a flipped
    # rounding of a gradient operand is a 4e-3 relative step for that element
    rep = _grad_errors(gn2, gn_)[0]
    print(f"   repeat run worst grad rel-L2 = {rep[0]:.3e} at {rep[1]}")
    assert rep[0] <= (1e-4 if precision == "fp32" else 1e-2), rep


def test_native_training_step_follows_weight_updates(monkeypatch):
    """After an optimizer step the training plan must see the new weights (one fdm_pack_weights launch per forward)."""
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32)
    model, diffusion, cfg, sd = build(over, "fp32")
    model.train()
    inp = O.synthetic_inputs(cfg, 1, 5, 2, seed=6)
    t, noise = torch.tensor([17]), torch.randn(inp["x0"].shape, generator=torch.Generator().manual_seed(3))
    opt = torch.optim.SGD(model.parameters(), lr=1e-2)
    _train_grads(model, diffusion, inp, t, noise, "native", monkeypatch)
    opt.step()
    loss_n, gn_ = _train_grads(model, diffusion, inp, t, noise, "native", monkeypatch)
    loss_a, ga_ = _train_grads(model, diffusion, inp, t, noise, "autograd", monkeypatch)
    assert O.rel_l2(loss_n, loss_a) <= 1e-5
    assert _grad_errors(gn_, ga_)[0][0] <= 2e-4


class _AutoregScheme:
    """Minimal autoregressive index scheme with the reference iterator's protocol (set_videos + __next__ returning per-row lists,
    sampling_schemes.py:34-121): condition on the newest `n_ctx` finished frames, generate the next `step` frames."""

    def __init__(self, T, n_obs, B, n_ctx=3, step=2):
        self.T, self.done, self.B, self.n_ctx, self.step = T, n_obs, B, n_ctx, step
        self.videos = None

    def set_videos(self, videos):
        self.videos = videos

    def __iter__(self):
        return self

    def __next__(self):
        if self.done >= self.T:
            raise StopIteration
        lat = list(range(self.done, min(self.done + self.step, self.T)))
        obs = list(range(max(0, self.done - self.n_ctx), self.done))
        self.done += len(lat)
        return [obs] * self.B, [lat] * self.B


def test_device_resident_video_sampler_matches_host_loop():
    """video_sampler.sample_video_with_iterator (buffer on the GPU, one gather / scatter kernel per stage) against the
    reference's host-side procedure (scripts/video_sample.py:28-85 restated: CPU buffer, per-row gather, upload, sample, download,
    per-row scatter) with the same deterministic noise."""
    from improved_diffusion import video_sampler
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32, timestep_respacing="4")
    model, diffusion, cfg, sd = build(over, "fp32")
    diffusion._noise_fn = torch.zeros_like
    B, T, n_obs = 2, 9, 3
    g = torch.Generator().manual_seed(3)
    batch = torch.randn(B, T, 4, 32, 32, generator=g).clamp(-1, 1)
    noise = {}

    def host_loop():
        samples = torch.zeros_like(batch)
        samples[:, :n_obs] = batch[:, :n_obs]
        for obs, lat in _AutoregScheme(T, n_obs, B):
            fi = torch.cat([torch.tensor(obs), torch.tensor(lat)], dim=1).long()
            x0 = torch.stack([samples[i, f] for i, f in enumerate(fi)])
            om = torch.cat([torch.ones_like(torch.tensor(obs)), torch.zeros_like(torch.tensor(lat))], dim=1).view(B, -1, 1, 1, 1).float()
            key = tuple(lat[0])
            noise[key] = torch.randn(x0.shape, generator=torch.Generator().manual_seed(len(noise)))
            out, _ = diffusion.p_sample_loop(model, x0.shape, noise=noise[key].cuda(),
                                             model_kwargs=dict(frame_indices=fi.cuda(), x0=x0.cuda(), obs_mask=om.cuda(),
                                                               latent_mask=(1 - om).cuda()), latent_mask=(1 - om).cuda())
            for i, li in enumerate(lat):
                samples[i, li] = out[i, -len(li):].cpu()
        return samples

    ref = host_loop()
    # same initial noise per stage: patch p_sample_loop's noise through a thin wrapper
    orig = diffusion.p_sample_loop

    def with_noise(model_, shape, **kw):
        lat_n = int(kw["model_kwargs"]["obs_mask"][0].numel() - kw["model_kwargs"]["obs_mask"][0].sum())
        key = tuple(int(v) for v in kw["model_kwargs"]["frame_indices"][0, -lat_n:].tolist())
        return orig(model_, shape, noise=noise[key].cuda(), **kw)
    diffusion.p_sample_loop = with_noise
    try:
        got, used = video_sampler.sample_video_with_iterator(model, diffusion, batch, _AutoregScheme(T, n_obs, B), n_obs)
    finally:
        diffusion.p_sample_loop = orig
    assert got.device == batch.device and len(used) == 3
    assert torch.equal(got[:, :n_obs], batch[:, :n_obs])
    assert O.rel_l2(got, ref) <= 1e-5


def test_flat_adamw_matches_torch_adamw(monkeypatch):
    """optim.FlatAdamW (one fdm_adamw launch over flat parameter / moment / gradient buffers, EMA fused) against torch.optim.AdamW
    + nn.update_ema over several real training steps (native backward: gradients arrive as views of one flat buffer) and one
    step with foreign gradients (gather path); state_dict round trip."""
    import copy
    from improved_diffusion.nn import update_ema
    from improved_diffusion.optim import FlatAdamW
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32)
    model, diffusion, cfg, sd = build(over, "fp32")
    model.train()
    ref = copy.deepcopy(model)
    ref_ema = [p.detach().clone() for p in ref.parameters()]
    opt_ref = torch.optim.AdamW(ref.parameters(), lr=3e-3, weight_decay=0.05)
    opt = FlatAdamW(model.parameters(), lr=3e-3, weight_decay=0.05, ema_rates=(0.9,), model=model, bind=False)
    assert all(torch.equal(a, b) for a, b in zip(model.parameters(), ref.parameters()))  # flattening kept the values
    inp = O.synthetic_inputs(cfg, 1, 5, 2, seed=6)
    noise = torch.randn(inp["x0"].shape, generator=torch.Generator().manual_seed(3))
    for it in range(3):
        t = torch.tensor([5 + 9 * it])
        monkeypatch.setenv("FDM_TRAIN_ENGINE", "native")
        terms = diffusion.training_losses(model, inp["x0"].cuda(), t.cuda(), model_kwargs=cuda_kw(inp), noise=noise.cuda(),
                                          latent_mask=inp["latent_mask"].cuda())
        opt.zero_grad(set_to_none=True)
        terms["loss"].mean().backward()
        # the SAME gradients for both optimizers: Adam's m / sqrt(v) turns the rounding-noise gradients of the analytically
        # zero-gradient parameters into O(lr) steps of random sign, so two separately differentiated copies drift apart
        for p, q in zip(model.parameters(), ref.parameters()):
            q.grad = p.grad.detach().clone()
        base = next(model.parameters()).grad.data_ptr() - 4 * opt._offs[0]
        assert all(p.grad.data_ptr() == base + 4 * o for p, o in zip(model.parameters(), opt._offs)), "gradients are not flat views"
        opt.step()
        opt_ref.step()
        update_ema(ref_ema, list(ref.parameters()), rate=0.9)
    worst = max(O.rel_l2(a.detach().cpu(), b.detach().cpu()) for a, b in zip(model.parameters(), ref.parameters()))
    assert worst <= 1e-5, worst
    assert max(O.rel_l2(a.cpu(), b.cpu()) for a, b in zip(opt.ema_params(0), ref_ema)) <= 1e-5
    # foreign (non-flat) gradients take the gather path; state_dict round trip keeps the moments
    g = torch.Generator(device="cuda").manual_seed(1)
    for p, q in zip(model.parameters(), ref.parameters()):
        p.grad = torch.randn(p.shape, device="cuda", generator=g)
        q.grad = p.grad.clone()
    st = copy.deepcopy(opt.state_dict())
    opt.load_state_dict(st)
    opt.step()
    opt_ref.step()
    worst = max(O.rel_l2(a.detach().cpu(), b.detach().cpu()) for a, b in zip(model.parameters(), ref.parameters()))
    assert worst <= 1e-5, worst
    # the INFERENCE engine (packed weights cached by parameter version) must see every optimizer step
    model.eval()
    x, t5 = inp["x"].cuda(), torch.tensor([5.0]).cuda()
    with torch.no_grad():
        e0, _ = model(x, timesteps=t5, **cuda_kw(inp))
    for p in model.parameters():
        p.grad = torch.randn(p.shape, device="cuda", generator=g)
    opt.step()
    with torch.no_grad():
        e1, _ = model(x, timesteps=t5, **cuda_kw(inp))
        ref.load_state_dict(model.state_dict())
        ref.eval()
        e_ref, _ = ref(x, timesteps=t5, **cuda_kw(inp))
    assert O.rel_l2(e1.cpu(), e0.cpu()) > 1e-4 and O.rel_l2(e1.cpu(), e_ref.cpu()) <= 1e-5
    model.train()
    # the model still runs (its training plan was rebuilt over the flat parameter storage) and checkpoints keep their keys
    assert list(model.state_dict().keys()) == list(ref.state_dict().keys())


def test_flat_gradient_mode_matches_per_parameter_path(monkeypatch):
    """FlatAdamW(..., model=model): one autograd anchor instead of 390 parameter inputs, p.grad as persistent views of the flat
    gradient buffer.  Gradients equal the per-parameter path, two backwards between zero_grad() calls accumulate, and the
    optimizer step equals torch.optim.AdamW on the same gradients."""
    import copy
    from improved_diffusion.optim import FlatAdamW
    monkeypatch.setenv("FDM_TRAIN_ENGINE", "native")
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32)
    model, diffusion, cfg, sd = build(over, "fp32")
    model.train()
    inp = O.synthetic_inputs(cfg, 2, 5, 2, seed=8, pad_rows=(0,))
    noise = torch.randn(inp["x0"].shape, generator=torch.Generator().manual_seed(4))
    t = torch.tensor([3, 21])

    def backward(m_):
        terms = diffusion.training_losses(m_, inp["x0"].cuda(), t.cuda(), model_kwargs=cuda_kw(inp), noise=noise.cuda(),
                                          latent_mask=inp["latent_mask"].cuda())
        terms["loss"].mean().backward()
        return terms["loss"].detach()
    backward(model)
    ref_grads = [p.grad.detach().clone() for p in model.parameters()]
    ref = build(over, "fp32")[0]  # (a model that has run holds compiled plans: build a fresh copy instead of deepcopy)
    ref.load_state_dict(model.state_dict())
    opt_ref = torch.optim.AdamW(ref.parameters(), lr=2e-3, weight_decay=0.01)
    model.zero_grad(set_to_none=True)
    opt = FlatAdamW(model.parameters(), lr=2e-3, weight_decay=0.01, model=model)
    views = [p.grad for p in model.parameters()]
    opt.zero_grad()
    backward(model)
    assert all(p.grad is v for p, v in zip(model.parameters(), views)), "p.grad must stay the persistent view"
    assert _grad_errors({i: g for i, g in enumerate(views)}, {i: g for i, g in enumerate(ref_grads)})[0][0] <= 1e-4
    backward(model)  # second backward without zero_grad: accumulates
    assert _grad_errors({i: g for i, g in enumerate(views)}, {i: 2 * g for i, g in enumerate(ref_grads)})[0][0] <= 1e-4
    opt.zero_grad()
    backward(model)
    for q, g_ in zip(ref.parameters(), views):
        q.grad = g_.detach().clone()
    opt.step()
    opt_ref.step()
    assert max(O.rel_l2(a.detach().cpu(), b.detach().cpu()) for a, b in zip(model.parameters(), ref.parameters())) <= 1e-5


def test_native_training_trajectory_matches_autograd(monkeypatch):
    """Ten SGD steps (fp32 mode, fresh noise / timesteps per step) on two copies of a model — one through the native forward +
    backward schedules (CUDA-graph replays, weight re-packing every step), one through torch.autograd — must stay together:
    the same losses step by step and the same weights at the end."""
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32)
    nat, diffusion, cfg, sd = build(over, "fp32")
    ref = build(over, "fp32")[0]
    nat.train()
    ref.train()
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    inp = O.synthetic_inputs(cfg, 2, 5, 2, seed=12, pad_rows=(1,))
    opts = [torch.optim.SGD(m_.parameters(), lr=0.05) for m_ in (nat, ref)]
    g = torch.Generator().manual_seed(21)
    losses = []
    for it in range(10):
        t = torch.randint(0, 32, (2,), generator=g)
        noise = torch.randn(inp["x0"].shape, generator=g)
        row = []
        for m_, o_, eng in ((nat, opts[0], "native"), (ref, opts[1], "autograd")):
            monkeypatch.setenv("FDM_TRAIN_ENGINE", eng)
            terms = diffusion.training_losses(m_, inp["x0"].cuda(), t.cuda(), model_kwargs=cuda_kw(inp), noise=noise.cuda(),
                                              latent_mask=inp["latent_mask"].cuda())
            o_.zero_grad(set_to_none=True)
            terms["loss"].mean().backward()
            o_.step()
            row.append(float(terms["loss"].detach().mean()))
        losses.append(row)
    print("trajectory: max loss rel diff %.2e" % max(abs(a - b) / abs(b) for a, b in losses))
    for a, b in losses:
        assert abs(a - b) <= 2e-4 * abs(b), losses
    worst = max(O.rel_l2(p.detach().cpu(), q.detach().cpu()) for p, q in zip(nat.parameters(), ref.parameters()))
    print("trajectory: worst weight rel-L2 after 10 steps %.2e" % worst)
    assert worst <= 2e-4, worst


def _video_stream(seed, B=2, T=12):
    g = torch.Generator().manual_seed(seed)
    while True:
        yield torch.randn(B, T, 4, 32, 32, generator=g).clamp(-1, 1)


def test_native_train_step_matches_torch_stack(monkeypatch, tmp_path):
    """train_step.NativeTrainStep (host side of TrainLoop.run_step; on CPU it is bit-identical to the reference's TrainLoop,
    tests/dropin_trainloop.py) over the NATIVE stack — host batch through the pinned staging upload, native forward/backward, flat
    gradient norm, FlatAdamW+EMA, one log read — against the same class over torch.autograd + torch.optim.AdamW from the same
    seeds: same random draws, same logged losses / quartiles / gradient norm for three steps.  (Parameters themselves are not
    compared: Adam turns the rounding-noise gradients of the analytically gradient-free biases into +-lr steps on both sides.)"""
    import numpy as np
    from improved_diffusion.train_step import NativeTrainStep
    from improved_diffusion.sharding import FlatGradDataParallel
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32)

    def run(optimizer, engine, microbatch=-1, wrap=False, steps=3, defer=False):
        model, diffusion, _, _ = build(over, "fp32")
        model.train()
        monkeypatch.setenv("FDM_TRAIN_ENGINE", engine)
        runner = NativeTrainStep(model, diffusion, lr=1e-4, max_frames=5, ema_rate="0.999,0.9999", microbatch=microbatch,
                                 optimizer=optimizer, lr_anneal_steps=100)
        if wrap:
            runner.net = FlatGradDataParallel(model)
        torch.manual_seed(7)
        np.random.seed(7)
        data = _video_stream(3)
        logs = [runner.run_step(next(data), next(data), defer=defer) for _ in range(steps)]
        if defer:  # every call returned the previous step's log; the last one is still in flight
            assert logs[0] is None
            logs = logs[1:] + [runner.flush()]
            assert runner.flush() is None
        tail = (float(torch.rand(())), float(np.random.rand()))
        return logs, tail, model, runner

    nat, tail_n, model_n, runner_n = run("flat", "native")
    ref, tail_r, _, _ = run("torch", "autograd")
    assert tail_n == tail_r  # the same random draws were consumed
    for a, b in zip(nat, ref):
        assert set(a) == set(b), (sorted(a), sorted(b))
        for k in a:
            assert abs(a[k] - b[k]) <= 3e-4 * max(abs(b[k]), 1e-6), (k, a[k], b[k])
    assert nat[2]["lr"] == pytest.approx(1e-4 * (1 - 2 / 100)) and nat[2]["step"] == 2 and nat[2]["samples"] == 6
    assert all(torch.isfinite(e).all() for e in runner_n.ema_params[1])
    assert not torch.equal(runner_n.ema_params[0][0], next(model_n.parameters()).detach())
    late = run("flat", "native", defer=True)[0]  # deferred log reads: the same records, one step later
    for a, b in zip(nat, late):
        assert set(a) == set(b) and a["step"] == b["step"]
        for k in a:
            assert abs(a[k] - b[k]) <= 1e-5 * max(abs(b[k]), 1e-6), (k, a[k], b[k])
    # gradient accumulation over microbatches, with and without the data-parallel wrapper's no_sync() (world size 1: the
    # allreduce is the identity, the deferred-synchronisation bookkeeping is what runs): the same numbers
    acc, _, model_a, _ = run("flat", "native", microbatch=1, steps=2)
    accw, _, model_w, runner_w = run("flat", "native", microbatch=1, wrap=True, steps=2)
    assert runner_w.opt.route.pending is False
    for a, b in zip(acc, accw):  # not bit-identical: the backward's fp32 atomics (RPE tables, split reductions) reorder run to run
        for k in a:
            assert abs(a[k] - b[k]) <= 1e-5 * max(abs(b[k]), 1e-6), (k, a[k], b[k])
    refacc, _, _, _ = run("torch", "autograd", microbatch=1, steps=2)
    for a, b in zip(acc, refacc):
        for k in a:
            assert abs(a[k] - b[k]) <= 3e-4 * max(abs(b[k]), 1e-6), (k, a[k], b[k])
    # checkpoint round trip around the flat buffers: compact files in the reference's layout, identical state after resume()
    path = runner_n.save(str(tmp_path), config={})
    ck = torch.load(path)
    assert list(ck["state_dict"]) == list(model_n.state_dict()) and ck["step"] == 2
    assert all(v.device.type == "cpu" and v.untyped_storage().nbytes() == v.numel() * 4 for v in ck["state_dict"].values())
    model_b = build(over, "fp32", seed=5)[0]
    model_b.train()
    runner_b = NativeTrainStep(model_b, runner_n.diffusion, lr=1e-4, max_frames=5, ema_rate="0.999,0.9999")
    assert runner_b.resume(str(tmp_path)) == 2
    for name in ("flat_p", "flat_m", "flat_v"):
        assert torch.equal(getattr(runner_b.opt, name), getattr(runner_n.opt, name)), name
    assert all(torch.equal(a, b) for a, b in zip(runner_b.opt.flat_ema, runner_n.opt.flat_ema))
    assert runner_b.opt._step == runner_n.opt._step == 3
    assert next(model_b.parameters()).data_ptr() == runner_b.opt.flat_p.data_ptr() + 4 * runner_b.opt._offs[0]  # still flat views


def test_bucketed_backward_segments_match_the_single_graph(monkeypatch):
    """The overlapped gradient exchange runs the backward schedule as one CUDA graph per gradient bucket and hands each bucket to the
    collective as soon as its segment is enqueued (engine.GradRoute.hand_over).  With an identity 'collective' on one GPU the
    segmented path must reproduce the single-graph gradients exactly, bucket views must tile the flat buffer, and every bucket
    must be handed over exactly once, in completion order."""
    from improved_diffusion.engine import grad_route
    from improved_diffusion.optim import FlatAdamW
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32)
    monkeypatch.setenv("FDM_TRAIN_ENGINE", "native")
    model, diffusion, cfg, sd = build(over, "fp32")
    model.train()
    opt = FlatAdamW(model.parameters(), lr=1e-4, weight_decay=0.0, model=model)
    inp = O.synthetic_inputs(cfg, 2, 5, 2, seed=8)
    t, noise = torch.tensor([3, 17]), torch.randn(inp["x0"].shape, generator=torch.Generator().manual_seed(4))

    def grads():
        out = []
        for _ in range(3):  # eager run, graph capture, graph replay
            opt.zero_grad()
            terms = diffusion.training_losses(model, inp["x0"].cuda(), t.cuda(), model_kwargs=cuda_kw(inp), noise=noise.cuda(),
                                              latent_mask=inp["latent_mask"].cuda(), eval_mask=inp["latent_mask"].cuda())
            terms["loss"].mean().backward()
            torch.cuda.synchronize()
            out.append(opt.flat_g.clone())
        return out

    plain = grads()
    seen = []

    def bucket_sync(view):
        seen.append((view.data_ptr(), view.numel()))
        return lambda: None
    route = grad_route(model)
    route.reduce = lambda flat: flat
    route.reduce_async = bucket_sync
    seg = grads()
    P = next(iter(model.engine().train_plans.values()))
    nb = len(P.grad_buckets)
    assert nb >= 3 and len(seen) == 3 * nb
    base = P.pgrad.data_ptr()
    assert [((a - base) // 4, (a - base) // 4 + n) for a, n in seen[:nb]] == [(lo, hi) for lo, hi, _ in P.grad_buckets]
    for a, b in zip(plain, seg):
        # fp32 atomics inside single kernels make the last bits run-dependent in either mode; the segmentation itself adds nothing
        assert O.rel_l2(b.cpu(), a.cpu()) <= 1e-6
    assert any(k[2] is not None for k in P.graphs if k[0] == "train" and k[1] == "bwd"), "segments were not captured as graphs"
