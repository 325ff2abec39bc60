"""
GPU parity at real shapes, and against the UNMODIFIED reference running on the same B200 where a copy of it is present (oracle/_ref):

  * eps at the REAL BASELINE.json shapes (cfg4 shard B=8/K=20/nc=64 — the shape bench.py times —, cfg2, cfg3 128 px/nc=128/K=20/B=2,
    cfg5 64 px/nc=128/K=40 at B = 1, 2, 16, and num_res_blocks=2, the reference default): native fp32 mode <= 1e-4, bf16 mode
    <= 2e-2 against the oracle's network (oracle/fdm_oracle.py, the restatement of the reference's forward that the committed goldens
    of tests/golden pin to the live reference) in PyTorch-eager fp32 on the same GPU (TF32 off) — the GPU-side oracle of SURVEY §8c;
  * with the reference present: its own `sample_video` (scripts/video_sample.py:28-85) driving the native model + diffusion, against
    the same function driving the reference model + diffusion, same seeds; its attention maps; its own `TrainLoop`
    (train_util.py:267-275 run_step) over the native model on the GPU (subprocess helper).  These run the reference's own code, which
    is not part of this repository, and skip without it.
"""
import os
import subprocess
import sys
import types

import pytest
import torch

from oracle import fdm_oracle as O
from oracle import ref_loader as R

pytestmark = pytest.mark.gpu
needs_reference = pytest.mark.skipif(R.find_ref() is None, reason="runs the reference's own code: needs a reference checkout "
                                                                  "(oracle/make_ref.sh copies it into oracle/_ref)")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PIXEL = dict(diffusion_space="pixel", pre_encoded=False, pre_encoded_stats_dict=None)
TOL = {"fp32": 1e-4, "bf16": 2e-2}


@pytest.fixture(autouse=True)
def _exact_fp32_reference():
    """The eager reference is the fp32 oracle on the GPU: no TF32 in cuDNN convs / cuBLAS matmuls."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def build_native(over, seed=1):
    """(native model, native diffusion, oracle cfg, state dict) with deterministic non-zero weights."""
    from improved_diffusion.script_util import create_model_and_diffusion, model_and_diffusion_defaults
    d = model_and_diffusion_defaults()
    d.update(over)
    d["diffusion_space_kwargs"] = dict(PIXEL)
    model, diffusion = create_model_and_diffusion(**d)
    cfg = O.make_cfg(**{**{k: d[k] for k in ("image_size", "in_channels", "num_channels", "num_res_blocks")}, **over})
    sd = O.init_state_dict(cfg, seed=seed)
    model.load_state_dict(sd, strict=True)
    return model.cuda().eval(), diffusion, cfg, sd


def build_pair(over, seed=1):
    """(native model, native diffusion, reference model, reference diffusion) with the same deterministic non-zero weights."""
    model, diffusion, cfg, sd = build_native(over, seed)
    ref_model, ref_diffusion = R.create_reference(over)
    ref_model.load_state_dict(sd, strict=True)  # the reference's own strict load: pins the state-dict contract on the way
    return model, diffusion, ref_model.cuda().eval(), ref_diffusion, cfg, sd


def oracle_eps_on_gpu(sd, cfg, inp, ts):
    """eps of the oracle's network in fp32 on the GPU (the fixture disables TF32): the reference's forward as restated by
    oracle/fdm_oracle.py, held to the live reference's outputs by tests/test_oracle_golden.py."""
    sd_gpu = {k: v.cuda() for k, v in sd.items()}
    return O.unet_forward(sd_gpu, cfg, inp["x"].cuda(), inp["x0"].cuda(), ts.cuda(), inp["frame_indices"].cuda(),
                          inp["obs_mask"].cuda(), inp["latent_mask"].cuda())


def cuda_kw(inp):
    return {k: inp[k].cuda() for k in ("x0", "frame_indices", "obs_mask", "latent_mask")}


LATENT32 = dict(image_size=32, in_channels=4, num_channels=64, num_res_blocks=1, diffusion_steps=1000)
REAL_SHAPES = [
    # name, overrides, B, K, n_obs, padded rows
    ("cfg4-shard-B8-K20", LATENT32, 8, 20, 10, ()),                      # the shape bench.py times (BASELINE configs[3])
    ("cfg4-ragged-last-stage-K14", LATENT32, 8, 14, 7, (3,)),            # hierarchy-2's final stage is ragged (SURVEY §8d)
    ("cfg2-B1-K5", LATENT32, 1, 5, 3, ()),                               # BASELINE configs[1]
    ("cfg3-128px-nc128-B2-K20", dict(image_size=128, in_channels=3, num_channels=128, num_res_blocks=1, diffusion_steps=1000),
     2, 20, 10, ()),                                                     # BASELINE configs[2]
    ("cfg5-B1-K40", dict(image_size=64, in_channels=4, num_channels=128, num_res_blocks=1, diffusion_steps=1000), 1, 40, 20, ()),
    ("cfg5-B2-K40", dict(image_size=64, in_channels=4, num_channels=128, num_res_blocks=1, diffusion_steps=1000), 2, 40, 20, (1,)),
    ("cfg5-B16-K40", dict(image_size=64, in_channels=4, num_channels=128, num_res_blocks=1, diffusion_steps=1000), 16, 40, 20, ()),
    ("nrb2-latent-B2-K8", dict(image_size=32, in_channels=4, num_channels=64, num_res_blocks=2, diffusion_steps=1000), 2, 8, 3, ()),
    ("reference-defaults-64px-nc128-nrb2", dict(diffusion_steps=1000), 1, 6, 2, ()),  # script_util.py:9-36 untouched
]


def _check_eps(label, model, inp, ts, ref):
    """native fp32 and bf16 eps against `ref` (an fp32 eps on the GPU) at the TOL bounds"""
    kw = cuda_kw(inp)
    assert float(ref.abs().mean()) > 1e-2, "vacuous parity: eps ~ 0"
    for precision in ("fp32", "bf16"):
        model.precision = precision
        eps, attn = model(inp["x"].cuda(), timesteps=ts.cuda(), **kw)
        e = O.rel_l2(eps.cpu(), ref.cpu())
        print(f"{label} [{precision}] eps rel-L2 = {e:.3e}")
        assert attn is None and eps.shape == ref.shape
        assert e <= TOL[precision], (label, precision, e)


def _real_shape_inputs(cfg, B, K, n_obs, pads):
    inp = O.synthetic_inputs(cfg, B, K, n_obs, seed=7, video_len=300, pad_rows=pads)
    return inp, O.model_timesteps(O.Tables(cfg), torch.tensor([(97 * (b + 1)) % 1000 for b in range(B)]))


@needs_reference
@pytest.mark.parametrize("name,over,B,K,n_obs,pads", REAL_SHAPES, ids=[c[0] for c in REAL_SHAPES])
def test_eps_at_real_shapes_vs_reference_on_gpu(name, over, B, K, n_obs, pads):
    model, diffusion, ref_model, ref_diffusion, cfg, sd = build_pair(over)
    inp, ts = _real_shape_inputs(cfg, B, K, n_obs, pads)
    with torch.no_grad():
        ref, _ = ref_model(inp["x"].cuda(), timesteps=ts.cuda(), **cuda_kw(inp))
        _check_eps(f"{name} vs reference-on-GPU", model, inp, ts, ref)
    del model, ref_model
    torch.cuda.empty_cache()


@pytest.mark.parametrize("name,over,B,K,n_obs,pads", REAL_SHAPES, ids=[c[0] for c in REAL_SHAPES])
def test_eps_at_real_shapes_vs_oracle_on_gpu(name, over, B, K, n_obs, pads):
    """The same shapes against the oracle's network (oracle/fdm_oracle.py) in fp32 on the GPU: runs without a reference checkout."""
    model, diffusion, cfg, sd = build_native(over)
    inp, ts = _real_shape_inputs(cfg, B, K, n_obs, pads)
    with torch.no_grad():
        _check_eps(f"{name} vs oracle-on-GPU", model, inp, ts, oracle_eps_on_gpu(sd, cfg, inp, ts))
    del model
    torch.cuda.empty_cache()


def test_bench_shape_also_matches_cpu_oracle():
    """The benchmarked shape once more against the CPU oracle (the restatement of the reference's forward that the goldens pin at
    the cfg1 shapes), at B=8, K=20, nc=64."""
    model, diffusion, cfg, sd = build_native(LATENT32)
    inp = O.synthetic_inputs(cfg, 8, 20, 10, seed=0, video_len=300)
    ts = torch.full((8,), 999.0)
    with torch.no_grad():
        ref = O.unet_forward(sd, cfg, inp["x"], inp["x0"], ts, inp["frame_indices"], inp["obs_mask"], inp["latent_mask"])
        for precision in ("fp32", "bf16"):
            model.precision = precision
            eps, _ = model(inp["x"].cuda(), timesteps=ts.cuda(), **cuda_kw(inp))
            e = O.rel_l2(eps.cpu(), ref)
            print(f"bench shape [{precision}] eps rel-L2 vs CPU oracle = {e:.3e}")
            assert e <= TOL[precision]


def _args(scheme, n_obs, max_frames, max_latent):
    return types.SimpleNamespace(n_obs=n_obs, optimality=None, sampling_scheme=scheme, max_frames=max_frames,
                                 max_latent_frames=max_latent, device=torch.device("cuda"), clip_denoised=True, eval_dir=None)


@needs_reference
@pytest.mark.parametrize("scheme,T,n_obs,max_frames,max_latent", [("autoreg", 12, 3, 5, 2), ("hierarchy-2", 20, 4, 8, 4),
                                                                  ("long-range", 11, 2, 6, 3)])
def test_reference_sample_video_runs_over_the_native_model(scheme, T, n_obs, max_frames, max_latent):
    """scripts/video_sample.py::sample_video, UNMODIFIED, (a) over this repo's model + diffusion and (b) over the reference's,
    on the same GPU with the same generator seed: the videos agree (fp32 mode; every stage is a respaced p_sample_loop)."""
    vs = R.load_script("video_sample")
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32, timestep_respacing="4")
    model, diffusion, ref_model, ref_diffusion, cfg, sd = build_pair(over)
    model.precision = "fp32"
    batch = torch.randn(2, T, 4, 32, 32, generator=torch.Generator().manual_seed(3)).clamp(-1, 1)
    torch.manual_seed(11)
    got, used = vs.sample_video(_args(scheme, n_obs, max_frames, max_latent), model, diffusion, batch)
    torch.manual_seed(11)
    want, used_ref = vs.sample_video(_args(scheme, n_obs, max_frames, max_latent), ref_model, ref_diffusion, batch)
    assert used == used_ref and len(used) >= 2
    assert torch.equal(got[:, :n_obs], batch[:, :n_obs])
    e = O.rel_l2(got, want)
    print(f"sample_video[{scheme}] over native vs reference: {len(used)} stages, rel-L2 = {e:.3e}")
    assert e <= 2e-3, e  # 4 chained steps per stage, stages chained through the generated frames
    # and through the device-resident stage driver of this repo (video_sampler): same scheme iterator, same seeds
    from improved_diffusion import video_sampler
    torch.manual_seed(11)
    mine, used_mine = video_sampler.sample_video(_args(scheme, n_obs, max_frames, max_latent), model, diffusion, batch)
    assert [tuple(map(tuple, (o, l))) for o, l in used_mine] == [tuple(map(tuple, (o, l))) for o, l in used_ref]
    e2 = O.rel_l2(mine.cpu(), want)
    print(f"   video_sampler.sample_video vs reference: rel-L2 = {e2:.3e}")
    assert e2 <= 2e-3, e2


class _ContentAdaptiveScheme:
    """Adaptive-style index scheme with the reference iterator's protocol (sampling_schemes.py:241-262: `set_videos` hands the
    current videos to the scheme, which picks per-row observed frames from the finished ones).  lpips (the reference's frame
    embedder) is absent from the image, so the distance here is plain pixel L2 — what matters is that the scheme reads the
    DEVICE-resident buffer every stage and returns per-row DISTINCT index sets."""

    def __init__(self, T, n_obs, B, n_ctx=3, step=2):
        self.T, self.done, self.B, self.n_ctx, self.step = T, n_obs, B, n_ctx, step
        self.videos, self.calls, self.devices = None, 0, set()

    def set_videos(self, videos):
        self.videos = videos
        self.calls += 1
        self.devices.add(videos.device.type)

    def __iter__(self):
        return self

    def __next__(self):
        if self.done >= self.T:
            raise StopIteration
        lat = list(range(self.done, min(self.done + self.step, self.T)))
        obs = []
        for b in range(self.B):
            newest = self.videos[b, self.done - 1]
            d = (self.videos[b, :self.done - 1] - newest).flatten(1).norm(dim=1) if self.done > 1 else torch.zeros(0)
            far = torch.argsort(d, descending=True)[: self.n_ctx - 1].tolist()  # most different finished frames + the newest
            obs.append(sorted(far) + [self.done - 1])
        self.done += len(lat)
        return obs, [lat] * self.B


@needs_reference
def test_adaptive_scheme_on_the_device_resident_buffer():
    """An adaptive scheme (per-row observed sets chosen from the CURRENT samples via set_videos) through video_sampler on the
    device buffer, against the reference's host-loop `sample_video` procedure given the same scheme object type."""
    from improved_diffusion import video_sampler
    vs = R.load_script("video_sample")
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32, timestep_respacing="4")
    model, diffusion, ref_model, ref_diffusion, cfg, sd = build_pair(over)
    model.precision = "fp32"
    B, T, n_obs = 3, 10, 4
    batch = torch.randn(B, T, 4, 32, 32, generator=torch.Generator().manual_seed(5)).clamp(-1, 1)
    mine_scheme = _ContentAdaptiveScheme(T, n_obs, B)
    torch.manual_seed(2)
    got, used = video_sampler.sample_video_with_iterator(model, diffusion, batch, mine_scheme, n_obs)
    assert mine_scheme.devices == {"cuda"} and mine_scheme.calls == len(used) + 1
    assert any(len({tuple(o) for o in obs}) > 1 for obs, _ in used), "rows should pick different observed frames"
    # reference procedure: patch the scheme table so the unmodified sample_video builds the same scheme
    ss = sys.modules[vs.sample_video.__module__].sampling_schemes
    ss["_test_adaptive"] = lambda video_length, num_obs, max_frames, step_size, optimal_schedule_path=None: \
        _ContentAdaptiveScheme(video_length, num_obs, B)
    try:
        torch.manual_seed(2)
        want, used_ref = vs.sample_video(_args("_test_adaptive", n_obs, 5, 2), ref_model, ref_diffusion, batch)
    finally:
        del ss["_test_adaptive"]
    assert [(list(map(list, o)), list(map(list, l))) for o, l in used] == [(list(map(list, o)), list(map(list, l))) for o, l in used_ref]
    e = O.rel_l2(got.cpu(), want)
    print(f"adaptive scheme on the device buffer vs reference sample_video: rel-L2 = {e:.3e}")
    assert e <= 2e-3


@needs_reference
def test_reference_trainloop_runs_over_the_native_model_on_gpu():
    """The reference's unmodified TrainLoop (forward_backward + optimize_normal + log_step, DDP-wrapped on CUDA) over the native
    model, against the same loop over the reference model on the same GPU: see tests/dropin_trainloop_gpu.py."""
    env = dict(os.environ, FDM_TRAIN_ENGINE="native", MASTER_ADDR="127.0.0.1", MASTER_PORT="29631")
    env.pop("FDM_ALLOW_TORCH_TRAIN", None)  # the GPU path must be the native one: no PyTorch-expression fallback allowed
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_trainloop_gpu.py")], env=env, capture_output=True,
                       text=True, timeout=900)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-2000:] + "\n" + r.stderr[-4000:]
    assert "TRAINLOOP_GPU_OK" in r.stdout


def test_philox_noise_mode_statistics_and_determinism():
    """Opt-in perf mode: the step noise drawn inside fdm_ddpm_step (Philox4x32-10 + Box-Muller).  With eps = 0 and coefficients
    a = c1 = c2 = 0, sigma = 1 the kernel's output IS the noise: check moments, independence across steps / stages, determinism."""
    from improved_diffusion import _native as N_
    n, B = 1 << 20, 2
    x = torch.zeros(B, n, device="cuda")
    eps = torch.zeros_like(x)
    coef = torch.zeros(1000, 8, device="cuda")
    coef[:, 4] = 1.0
    out = torch.empty_like(x)

    def draw(seed, nonce, tval):
        t = torch.full((B,), tval, device="cuda", dtype=torch.int64)
        ph = torch.tensor([seed, nonce], device="cuda", dtype=torch.int64)
        a = N_.DdpmStepArgs(x=x.data_ptr(), eps=eps.data_ptr(), noise=None, coef=coef.data_ptr(), t=t.data_ptr(),
                            sample=out.data_ptr(), pred_xstart=None, per_video=n, B=B, clip=1, philox=ph.data_ptr())
        N_.call("fdm_ddpm_step", a, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        return out.clone()

    a = draw(1234, 1, 999)
    assert torch.equal(a, draw(1234, 1, 999))
    flat = a.flatten().double()
    m, v = float(flat.mean()), float(flat.var())
    skew, kurt = float((flat ** 3).mean()), float((flat ** 4).mean())
    print(f"philox normals: mean {m:.2e} var {v:.5f} E[x^3] {skew:.2e} E[x^4] {kurt:.4f}")
    assert abs(m) < 4e-3 and abs(v - 1) < 5e-3 and abs(skew) < 2e-2 and abs(kurt - 3) < 5e-2
    assert float(flat.abs().max()) < 7.0 and bool(torch.isfinite(flat).all())
    for other in (draw(1234, 1, 998), draw(1234, 2, 999), draw(1235, 1, 999)):  # next step / next stage / other seed
        c = float((a.flatten().double() * other.flatten().double()).mean())
        assert abs(c) < 4e-3, c
    assert abs(float((a[0].double() * a[1].double()).mean())) < 5e-3  # the two videos of the batch are independent
    # neighbouring elements uncorrelated (Box-Muller pairs)
    assert abs(float((a[0, :-1].double() * a[0, 1:].double()).mean())) < 5e-3


def test_philox_sampler_matches_torch_noise_sampler_in_distribution():
    """diffusion.noise_mode = 'philox' through p_sample_loop: finite, observed frames untouched, same per-frame statistics as
    the torch-noise sampler on the same weights (different stream, same distribution)."""
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32, timestep_respacing="8")
    model, diffusion, cfg, sd = build_native(over)
    model.precision = "bf16"
    inp = O.synthetic_inputs(cfg, 4, 6, 2, seed=9, video_len=40)
    kw = cuda_kw(inp)
    shape = tuple(inp["x0"].shape)
    torch.manual_seed(0)
    a, _ = diffusion.p_sample_loop(model, shape, model_kwargs=kw, latent_mask=kw["latent_mask"])
    diffusion.noise_mode = "philox"
    torch.manual_seed(0)
    b, _ = diffusion.p_sample_loop(model, shape, model_kwargs=kw, latent_mask=kw["latent_mask"])
    torch.manual_seed(0)
    b2, _ = diffusion.p_sample_loop(model, shape, model_kwargs=kw, latent_mask=kw["latent_mask"])
    diffusion.noise_mode = "torch"
    assert bool(torch.isfinite(b).all()) and b.shape == a.shape
    assert not torch.equal(b, b2), "every stage draws a fresh Philox key"
    sa, sb = float(a[:, 2:].std()), float(b[:, 2:].std())
    print(f"latent-frame std: torch noise {sa:.4f}, philox noise {sb:.4f}")
    assert abs(sa - sb) <= 0.1 * sa


ATTN_CASES = [
    (dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32), 2, 5, 2, (1,)),
    (dict(image_size=32, in_channels=4, num_channels=64, num_res_blocks=1, diffusion_steps=1000), 2, 20, 10, ()),
    (dict(image_size=64, in_channels=4, num_channels=128, num_res_blocks=1, diffusion_steps=1000), 1, 40, 20, ()),
]


def _attn_inputs(cfg, B, T, n_obs, pads):
    inp = O.synthetic_inputs(cfg, B, T, n_obs, seed=3, video_len=300, pad_rows=pads)
    return inp, O.model_timesteps(O.Tables(cfg), torch.tensor([(53 * (b + 1)) % cfg["diffusion_steps"] for b in range(B)]))


def _check_native_maps(label, model, inp, ts, eps_r, attn_r, attn_c):
    """model(..., return_attn_weights=True) in bf16 against fp32 maps `attn_r`; `attn_c` = the same maps with bf16 GEMM operands
    (torch autocast), the calibration of the bound."""
    kw = cuda_kw(inp)
    with torch.no_grad():
        eps_n, attn_n = model(inp["x"].cuda(), timesteps=ts.cuda(), return_attn_weights=True, **kw)
        eps_plain, none = model(inp["x"].cuda(), timesteps=ts.cuda(), **kw)
    assert none is None and O.rel_l2(eps_n.cpu(), eps_plain.cpu()) <= 1e-3  # the logging plan computes the same eps
    assert O.rel_l2(eps_n.cpu(), eps_r.cpu()) <= TOL["bf16"]
    assert set(attn_n) == {"spatial", "temporal", "mixed"} and attn_n["mixed"] == []
    plans = model.engine().plans
    assert any(k[-1] for k in plans), "the maps must come from a collect_attn kernel plan, not from the PyTorch expression"
    worst = worst_c = 0.0
    for key in ("spatial", "temporal"):
        assert len(attn_n[key]) == len(attn_r[key]) == 7
        for a, r, c in zip(attn_n[key], attn_r[key], attn_c[key]):
            assert a.shape == r.shape and a.dtype == torch.float32
            e, e_c = O.rel_l2(a.cpu(), r.cpu()), O.rel_l2(c.float().cpu(), r.cpu())
            worst, worst_c = max(worst, e), max(worst_c, e_c)
            # softmax maps amplify score errors; the bound is what torch's own autocast-bf16 run gives on the same map (x1.5), with
            # north_star's 2e-2 as the floor
            assert e <= max(2e-2, 1.5 * e_c), (key, tuple(a.shape), e, e_c)
            rows = a.sum(dim=-1)
            assert float((rows - 1).abs().max()) <= 2e-3  # every row of a head-averaged softmax sums to 1
    print(f"attention maps vs {label}: worst rel-L2 {worst:.3e} over 14 maps; torch autocast-bf16: {worst_c:.3e}")


@needs_reference
@pytest.mark.parametrize("over,B,T,n_obs,pads", ATTN_CASES)
def test_native_attention_maps_match_the_reference(over, B, T, n_obs, pads):
    """model(..., return_attn_weights=True) (unet.py:454-464, rpe.py:126-131): the head-averaged attention maps of every attention
    block, produced by the materialising variants of the tcgen05 attention kernels, against the unmodified reference on the GPU."""
    model, diffusion, ref_model, ref_diffusion, cfg, sd = build_pair(over)
    model.precision = "bf16"
    inp, ts = _attn_inputs(cfg, B, T, n_obs, pads)
    kw = cuda_kw(inp)
    with torch.no_grad():
        eps_r, attn_r = ref_model(inp["x"].cuda(), timesteps=ts.cuda(), return_attn_weights=True, **kw)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            _, attn_c = ref_model(inp["x"].cuda(), timesteps=ts.cuda(), return_attn_weights=True, **kw)
    assert set(attn_r) == {"spatial", "temporal", "mixed"}
    _check_native_maps("reference-on-GPU", model, inp, ts, eps_r, attn_r, attn_c)


@pytest.mark.parametrize("over,B,T,n_obs,pads", ATTN_CASES)
def test_native_attention_maps_match_the_oracle(over, B, T, n_obs, pads):
    """The same maps against the oracle's network on the GPU (unet_forward(attns=...): mean over heads, absolute value, as
    rpe.py:128-130), fp32 and under autocast-bf16 for the bound: runs without a reference checkout."""
    model, diffusion, cfg, sd = build_native(over)
    model.precision = "bf16"
    inp, ts = _attn_inputs(cfg, B, T, n_obs, pads)
    sd_gpu = {k: v.cuda() for k, v in sd.items()}
    args = (sd_gpu, cfg, inp["x"].cuda(), inp["x0"].cuda(), ts.cuda(), inp["frame_indices"].cuda(), inp["obs_mask"].cuda(),
            inp["latent_mask"].cuda())
    attn_r, attn_c = {}, {}
    with torch.no_grad():
        eps_r = O.unet_forward(*args, attns=attn_r)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            O.unet_forward(*args, attns=attn_c)
    _check_native_maps("oracle-on-GPU", model, inp, ts, eps_r, attn_r, attn_c)


@needs_reference
def test_sample_loop_attention_logging_matches_the_reference():
    """p_sample_loop(return_attn_weights=True): the per-quartile running means of the maps (gaussian_diffusion.py:448-469) through
    the native maps, against the reference loop with the same seeds (TrainLoop.log_samples' path, train_util.py:451-463)."""
    over = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32, timestep_respacing="8")
    model, diffusion, ref_model, ref_diffusion, cfg, sd = build_pair(over)
    model.precision = "bf16"
    inp = O.synthetic_inputs(cfg, 2, 6, 2, seed=4, video_len=40)
    kw = cuda_kw(inp)
    shape = tuple(inp["x0"].shape)
    torch.manual_seed(5)
    s_n, a_n = diffusion.p_sample_loop(model, shape, model_kwargs=kw, latent_mask=kw["latent_mask"], return_attn_weights=True)
    torch.manual_seed(5)
    s_r, a_r = ref_diffusion.p_sample_loop(ref_model, shape, model_kwargs=kw, latent_mask=kw["latent_mask"], return_attn_weights=True)
    assert set(a_n) == set(a_r) and len(a_n) == 8  # 4 quartiles x {spatial, temporal}
    for tag in a_r:
        e = O.rel_l2(a_n[tag].cpu(), a_r[tag].cpu())
        assert a_n[tag].shape == a_r[tag].shape and e <= 3e-2, (tag, e)
    assert O.rel_l2(s_n.cpu(), s_r.cpu()) <= 8 * TOL["bf16"]


def test_sample_loop_attention_logging_matches_reference_golden_on_gpu(golden):
    """p_sample_loop(return_attn_weights=True) on the GPU with the native bf16 map kernels against the reference's own run stored in
    tests/golden/attn_cfg1.pt (same weights, inputs and noises): the final sample and the per-quartile running means of the maps
    (gaussian_diffusion.py:448-469)."""
    g = golden("attn_cfg1")
    model, diffusion, cfg, sd = build_native(g["over"])
    model.precision = "bf16"
    inp = g["inputs"]
    kw = cuda_kw(inp)
    it = iter([n.cuda() for n in g["noises"][1:]])
    diffusion._noise_fn = lambda x: next(it)
    with torch.no_grad():
        final, attns = diffusion.p_sample_loop(model, tuple(inp["x0"].shape), noise=g["noises"][0].cuda(), model_kwargs=kw,
                                               latent_mask=kw["latent_mask"], return_attn_weights=True)
    # calibration, as in the per-forward map tests: what bf16 GEMM operands (torch autocast) cost the oracle's maps of this model on
    # the loop's first-step inputs; the bound is 1.5x that, with 3e-2 as the floor
    tab = O.Tables(cfg)
    ts0 = O.model_timesteps(tab, torch.full((inp["x0"].shape[0],), tab.num_timesteps - 1))
    args = ({k: v.cuda() for k, v in sd.items()}, cfg, g["noises"][0].cuda(), kw["x0"], ts0.cuda(), kw["frame_indices"],
            kw["obs_mask"], kw["latent_mask"])
    a32, a16 = {}, {}
    with torch.no_grad():
        O.unet_forward(*args, attns=a32)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            O.unet_forward(*args, attns=a16)
    e_c = max(O.rel_l2(c.float().cpu(), r.cpu()) for key in ("spatial", "temporal") for c, r in zip(a16[key], a32[key]))
    assert set(attns) == set(g["attns"]) and len(attns) == 8  # 4 quartiles x {spatial, temporal}
    for tag, ref in g["attns"].items():
        e = O.rel_l2(attns[tag].cpu(), ref)
        assert attns[tag].shape == ref.shape and e <= max(3e-2, 1.5 * e_c), (tag, e, e_c)
    print(f"quartile maps vs the reference's stored run: worst rel-L2 "
          f"{max(O.rel_l2(attns[t].cpu(), r) for t, r in g['attns'].items()):.3e}; oracle autocast-bf16 calibration {e_c:.3e}")
    assert O.rel_l2(final.cpu(), g["final"]) <= 8 * TOL["bf16"]


ADDITIVE = dict(image_size=32, in_channels=4, num_channels=64, num_res_blocks=1, diffusion_steps=1000, use_scale_shift_norm=False)


def _additive_inputs(cfg, sd):
    assert sd["input_blocks.1.0.emb_layers.1.weight"].shape[0] == 64  # C outputs, not 2C
    inp = O.synthetic_inputs(cfg, 2, 6, 2, seed=12, video_len=100, pad_rows=(0,))
    return inp, O.model_timesteps(O.Tables(cfg), torch.tensor([17, 803]))


@needs_reference
def test_additive_embedding_resblocks_match_the_reference():
    """use_scale_shift_norm=False (unet.py:204-206): h = out_layers(h + emb_out) — the embedding is added BEFORE the second
    GroupNorm.  Served by fdm_gn_apply's film_add mode (statistics of h + e derived from those of h in fp64); native training of
    this variant raises (the GroupNorm backward kernels implement the scale/shift form)."""
    model, diffusion, ref_model, ref_diffusion, cfg, sd = build_pair(ADDITIVE)
    inp, ts = _additive_inputs(cfg, sd)
    kw = cuda_kw(inp)
    with torch.no_grad():
        ref, _ = ref_model(inp["x"].cuda(), timesteps=ts.cuda(), **kw)
        _check_eps("additive-embedding ResBlocks vs reference-on-GPU", model, inp, ts, ref)
    model.train()
    with pytest.raises(NotImplementedError, match="use_scale_shift_norm"):
        diffusion.training_losses(model, inp["x0"].cuda(), torch.tensor([3, 5]).cuda(), model_kwargs=kw)


def test_additive_embedding_resblocks_match_the_oracle():
    """The additive-embedding ResBlocks against the oracle's network in fp32 on the GPU (res_block(scale_shift=False)), and native
    training of the variant raising: runs without a reference checkout."""
    model, diffusion, cfg, sd = build_native(ADDITIVE)
    inp, ts = _additive_inputs(cfg, sd)
    with torch.no_grad():
        _check_eps("additive-embedding ResBlocks vs oracle-on-GPU", model, inp, ts, oracle_eps_on_gpu(sd, cfg, inp, ts))
    model.train()
    with pytest.raises(NotImplementedError, match="use_scale_shift_norm"):
        diffusion.training_losses(model, inp["x0"].cuda(), torch.tensor([3, 5]).cuda(), model_kwargs=cuda_kw(inp))
