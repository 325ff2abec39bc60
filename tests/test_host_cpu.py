"""CPU: host-side logic of the drop-in package and the C-ABI library surface (no compute calls)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle import fdm_oracle as O
from oracle import ref_loader as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PIXEL = dict(diffusion_space="pixel", pre_encoded=False, pre_encoded_stats_dict=None)


def build(over):
    from improved_diffusion.script_util import create_model_and_diffusion, model_and_diffusion_defaults
    d = model_and_diffusion_defaults()
    d.update(over)
    d["diffusion_space_kwargs"] = dict(PIXEL)
    return create_model_and_diffusion(**d)


def test_library_exports_every_declared_symbol():
    from improved_diffusion import _native
    hdr = open(os.path.join(ROOT, "include", "fdm_b200.h")).read()
    declared = set(re.findall(r"^(?:int|size_t|const char\*)\s+(fdm_\w+)\s*\(", hdr, flags=re.M))
    assert {"fdm_conv", "fdm_ddpm_step", "fdm_attn_temporal", "fdm_abi_version"} <= declared
    lib = ctypes.CDLL(_native.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert set(_native.ENTRY_POINTS) <= declared
    assert _native.lib().fdm_abi_version() == 2
    assert _native.verify_struct_sizes()
    assert _native.lib().fdm_status_string(-2).decode().startswith("unsupported")


def test_defaults_and_factory_contract():
    from improved_diffusion.script_util import model_and_diffusion_defaults, create_model_and_diffusion
    d = model_and_diffusion_defaults()
    assert len(d) == 22 and d["num_heads"] == 4 and d["attention_resolutions"] == "16,8" and d["use_rpe_net"] is True
    assert {k: v for k, v in d.items() if k != "diffusion_space_kwargs"} == \
        {k: v for k, v in O.DEFAULTS.items() if k != "diffusion_space_kwargs"}
    bad = dict(d, image_size=48, diffusion_space_kwargs=dict(PIXEL))
    with pytest.raises(ValueError, match="unsupported image size"):
        create_model_and_diffusion(**bad)
    with pytest.raises(NotImplementedError):
        create_model_and_diffusion(**dict(d, noise_schedule="nope", diffusion_space_kwargs=dict(PIXEL)))
    with pytest.raises(AttributeError, match="beta"):  # rpe.py:50 — the reference's lookup-table branch is broken
        create_model_and_diffusion(**dict(d, use_rpe_net=False, diffusion_space_kwargs=dict(PIXEL)))


@pytest.mark.parametrize("over", [
    dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1),
    dict(image_size=64, in_channels=3, num_channels=32, num_res_blocks=2),
    dict(image_size=128, in_channels=3, num_channels=32, num_res_blocks=1),
])
def test_state_dict_contract(over):
    """Keys, order and shapes equal the reference's (oracle.param_shapes is pinned to the live reference by
    tests/golden/make_golden.py through load_state_dict(strict=True) + key-order assert)."""
    model, _ = build(over)
    shapes = O.param_shapes(O.make_cfg(**over))
    sd = model.state_dict()
    assert list(sd.keys()) == list(shapes.keys())
    for k, s in shapes.items():
        assert tuple(sd[k].shape) == tuple(s), k
    # zero-initialised tensors of the reference (zero_module) are zero here too
    zeros = [k for k in sd if k.endswith(("out_layers.3.weight", "proj_out.weight", "rpe_net.out.weight", "out.2.weight"))]
    assert zeros and all(float(sd[k].abs().sum()) == 0 for k in zeros)
    model.load_state_dict(O.init_state_dict(O.make_cfg(**over), seed=1), strict=True)


@pytest.mark.parametrize("steps,respacing", [(32, ""), (1000, ""), (1000, "250"), (1000, "10,15,20"), (1000, "ddim50"), (32, "4")])
def test_tables_match_oracle(steps, respacing):
    _, diffusion = build(dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=steps,
                              timestep_respacing=respacing))
    tab = O.Tables(O.make_cfg(diffusion_steps=steps, timestep_respacing=respacing))
    assert diffusion.num_timesteps == tab.num_timesteps
    assert diffusion.timestep_map == tab.timestep_map
    for name in ("betas", "alphas_cumprod", "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod",
                 "posterior_mean_coef1", "posterior_mean_coef2", "posterior_variance", "sqrt_alphas_cumprod",
                 "sqrt_one_minus_alphas_cumprod"):
        assert np.array_equal(getattr(diffusion, name), getattr(tab, name)), name
    var, logvar = diffusion._fixed_variance()
    assert np.array_equal(var, tab.model_variance) and np.array_equal(logvar, tab.model_log_variance)


def test_space_timesteps_errors():
    from improved_diffusion.respace import space_timesteps
    assert space_timesteps(100, "ddim10") == O.space_timesteps(100, "ddim10")
    with pytest.raises(ValueError):
        space_timesteps(100, "ddim33")
    with pytest.raises(ValueError):
        space_timesteps(10, "20")
    assert space_timesteps(300, [10, 15, 20]) == O.space_timesteps(300, [10, 15, 20])


def test_cpu_tensor_is_rejected_loudly():
    model, diffusion = build(dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32))
    inp = O.synthetic_inputs(O.make_cfg(image_size=32, in_channels=4), 1, 3, 1)
    with pytest.raises(RuntimeError, match="no CPU fallback"), torch.no_grad():
        model(inp["x"], x0=inp["x0"], timesteps=torch.zeros(1), frame_indices=inp["frame_indices"],
              obs_mask=inp["obs_mask"], latent_mask=inp["latent_mask"])


def test_q_sample_and_losses_host_math_cpu():
    """The torch (non-fused) branches of q_sample / p_mean_variance used for non-CUDA tensors follow the oracle."""
    _, diffusion = build(dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32))
    tab = O.Tables(O.make_cfg(diffusion_steps=32))
    g = torch.Generator().manual_seed(0)
    x0, noise = torch.randn(2, 3, 4, 8, 8, generator=g), torch.randn(2, 3, 4, 8, 8, generator=g)
    t = torch.tensor([5, 31])
    assert torch.equal(diffusion.q_sample(x0, t, noise), O.q_sample(tab, x0, t, noise))
    eps = torch.randn(2, 3, 4, 8, 8, generator=g)
    out = diffusion.p_mean_variance(lambda x, timesteps, **kw: (eps, None), x0, t)
    ref = O.posterior_from_eps(tab, x0, t, eps)
    for k in ("mean", "variance", "log_variance", "pred_xstart"):
        assert torch.equal(out[k], ref[k]), k


def test_training_losses_and_grads_match_reference(golden):
    """training_losses through the public API (autograd path) against the committed reference run: loss terms, parameter
    gradients, and every parameter receiving a gradient (DDP find_unused_parameters=False, train_util.py:124)."""
    g = golden("train_cfg1")
    model, diffusion = build(g["over"])
    model.load_state_dict(O.init_state_dict(O.make_cfg(**g["over"]), seed=1), strict=True)
    model.precision = "fp32"
    model.train()
    inp = g["inputs"]
    kw = dict(frame_indices=inp["frame_indices"], obs_mask=inp["obs_mask"], latent_mask=inp["latent_mask"], x0=inp["x0"])
    terms = diffusion.training_losses(model, inp["x0"], g["t"], model_kwargs=kw, noise=g["noise"],
                                      latent_mask=1 - inp["obs_mask"], eval_mask=inp["latent_mask"])
    terms["loss"].mean().backward()
    for k in ("loss", "mse", "eval-mse"):
        assert O.rel_l2(terms[k].detach(), g["terms"][k]) <= 1e-5, k
    grads = dict(model.named_parameters())
    for k, ref in g["grads"].items():
        assert O.rel_l2(grads[k].grad, ref) <= 1e-4, k
    # analytically-zero gradients (biases in front of a GroupNorm: 1e-10..1e-8 of pure summation-order noise, which differs
    # between hosts / thread counts) are held to an absolute floor relative to the largest gradient of the case
    floor = 1e-7 * max(g["grad_norms"].values())
    for k, nrm in g["grad_norms"].items():
        assert grads[k].grad is not None, k
        assert abs(float(grads[k].grad.norm()) - nrm) <= 1e-3 * nrm + floor, k


def test_drop_in_package_path_resolution(tmp_path):
    """FDM_REFERENCE_PATH: hot-path modules come from this repo, every other improved_diffusion module from the reference
    (INTEGRATION.md §2).  The reference checkout is a stand-in tree: its `unet` / `gaussian_diffusion` refuse to be imported, and its
    `sampling_schemes` replays the hierarchy-2 stages that the live reference's iterator produced (tests/golden/make_stages.py)."""
    import subprocess
    import sys
    pkg = tmp_path / "improved_diffusion"
    pkg.mkdir()
    (pkg / "__init__.py").write_text("")
    for name in ("unet", "gaussian_diffusion"):
        (pkg / f"{name}.py").write_text(f"raise ImportError('{name} must come from the drop-in package')\n")
    (pkg / "sampling_schemes.py").write_text(
        "import json\n"
        f"_fx = json.load(open({os.path.join(ROOT, 'tests', 'golden', 'stages_hierarchy-2_T300.json')!r}))\n"
        "def _hierarchy_2(video_length, num_obs, max_frames, step_size, optimal_schedule_path=None):\n"
        "    assert (video_length, num_obs, max_frames, step_size) == "
        "(_fx['video_length'], _fx['n_obs'], _fx['max_frames'], _fx['step_size'])\n"
        "    return iter([tuple(s) for s in _fx['stages']])\n"
        "sampling_schemes = {'hierarchy-2': _hierarchy_2}\n")
    code = (
        "import sys, improved_diffusion\n"
        "from improved_diffusion import sampling_schemes, unet, gaussian_diffusion\n"
        f"assert sampling_schemes.__file__.startswith({str(tmp_path)!r}), sampling_schemes.__file__\n"
        "assert '_b200' in unet.__file__ and '_b200' in gaussian_diffusion.__file__\n"
        "it = sampling_schemes.sampling_schemes['hierarchy-2'](video_length=300, num_obs=36, max_frames=20, step_size=10)\n"
        "stages = [(len(o), len(l)) for o, l in it]\n"
        "assert len(stages) == 27 and sum(o + l for o, l in stages) == 534, (len(stages), sum(o + l for o, l in stages))\n"
    )
    env = dict(os.environ, FDM_REFERENCE_PATH=str(tmp_path),
               PYTHONPATH=os.path.join(ROOT, "latent-flexible-video-diffusion-modeling_b200"))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]


def test_attention_map_logging_matches_reference(golden):
    """p_sample_loop(return_attn_weights=True) — the path TrainLoop.log_samples takes (train_util.py:451-463): same samples and
    the same per-quartile attention-map averages as the reference (tests/golden/attn_cfg1.pt)."""
    g = golden("attn_cfg1")
    model, diffusion = build(g["over"])
    model.load_state_dict(O.init_state_dict(O.make_cfg(**g["over"]), seed=1), strict=True)
    model.precision = "fp32"
    model.eval()
    inp = g["inputs"]
    kw = dict(frame_indices=inp["frame_indices"], obs_mask=inp["obs_mask"], latent_mask=inp["latent_mask"], x0=inp["x0"])
    it = iter(g["noises"][1:])
    diffusion._noise_fn = lambda x: next(it)
    with torch.no_grad():
        final, attns = diffusion.p_sample_loop(model, tuple(inp["x0"].shape), noise=g["noises"][0], model_kwargs=kw,
                                               latent_mask=inp["latent_mask"], return_attn_weights=True)
    assert O.rel_l2(final, g["final"]) <= 1e-5
    assert set(attns) == set(g["attns"])
    for k, ref in g["attns"].items():
        assert attns[k].shape == ref.shape and O.rel_l2(attns[k], ref) <= 1e-5, k


@pytest.mark.skipif(R.find_ref() is None, reason="runs the reference's own TrainLoop: needs a reference checkout "
                                                "(oracle/make_ref.sh copies it into oracle/_ref)")
def test_drop_in_under_reference_trainloop():
    """The reference's unmodified TrainLoop (train_util.py) runs two optimizer steps over this repo's model + diffusion
    (mask sampling, training_losses, backward, AdamW, EMA, loss logging): tests/dropin_trainloop.py in a subprocess."""
    import socket
    import subprocess
    import sys
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    env = dict(os.environ, FDM_REFERENCE_PATH=R.find_ref(),
               PYTHONPATH=os.path.join(ROOT, "latent-flexible-video-diffusion-modeling_b200"))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_trainloop.py"), str(port)], env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "DROPIN_OK" in r.stdout, (r.stdout[-1000:], r.stderr[-2000:])


def test_device_resident_video_sampler_host_logic_cpu():
    """video_sampler.sample_video_with_iterator on CPU with a row-independent stand-in denoiser: the gather / scatter indexing and
    the iterator protocol against the reference's per-row procedure (scripts/video_sample.py:56-83 restated)."""
    import torch
    from improved_diffusion import video_sampler

    class Fake(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.tensor(0.31))

        def forward(self, x, *, x0, timesteps, frame_indices=None, obs_mask=None, latent_mask=None, return_attn_weights=False):
            fi = frame_indices.float().view(*frame_indices.shape, 1, 1, 1) / 50.0
            return self.w * torch.tanh(x * (1 - obs_mask) + x0 * obs_mask + fi), None

    class Scheme:
        def __init__(self, T, n_obs, B):
            self.T, self.done, self.B = T, n_obs, B

        def set_videos(self, v):
            self.v = v

        def __iter__(self):
            return self

        def __next__(self):
            if self.done >= self.T:
                raise StopIteration
            lat = list(range(self.done, min(self.done + 2, self.T)))
            obs = [0] + list(range(max(1, self.done - 2), self.done))
            self.done += len(lat)
            return [obs] * self.B, [lat] * self.B

    _, diffusion = build(dict(image_size=32, in_channels=2, num_channels=32, num_res_blocks=1, diffusion_steps=32, timestep_respacing="4"))
    diffusion._noise_fn = torch.zeros_like
    model = Fake()
    B, T, n_obs = 3, 8, 3
    batch = torch.randn(B, T, 2, 8, 8, generator=torch.Generator().manual_seed(1)).clamp(-1, 1)
    torch.manual_seed(0)
    got, used = video_sampler.sample_video_with_iterator(model, diffusion, batch, Scheme(T, n_obs, B), n_obs, device="cpu")
    torch.manual_seed(0)
    samples = torch.zeros_like(batch)
    samples[:, :n_obs] = batch[:, :n_obs]
    for obs, lat in Scheme(T, n_obs, B):
        fi = torch.cat([torch.tensor(obs), torch.tensor(lat)], dim=1).long()
        x0 = torch.stack([samples[i, f] for i, f in enumerate(fi)])
        om = torch.cat([torch.ones_like(torch.tensor(obs)), torch.zeros_like(torch.tensor(lat))], dim=1).view(B, -1, 1, 1, 1).float()
        out, _ = diffusion.p_sample_loop(model, x0.shape, model_kwargs=dict(frame_indices=fi, x0=x0, obs_mask=om, latent_mask=1 - om),
                                         latent_mask=1 - om)
        for i, li in enumerate(lat):
            samples[i, li] = out[i, -len(li):]
    assert len(used) == 3 and torch.equal(got, samples)
    just, _ = video_sampler.sample_video_with_iterator(model, diffusion, batch, Scheme(T, n_obs, B), n_obs, device="cpu",
                                                       just_get_indices=True)
    assert torch.equal(just, batch)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("over,B,T", [
    (dict(image_size=32, in_channels=4, num_channels=64, num_res_blocks=1, diffusion_steps=1000), 1, 5),    # cfg2
    (dict(image_size=128, in_channels=3, num_channels=128, num_res_blocks=1, diffusion_steps=1000), 1, 2),  # cfg3 model, short clip
    (dict(image_size=64, in_channels=4, num_channels=128, num_res_blocks=1, diffusion_steps=1000), 1, 3),   # cfg5 model, short clip
])
def test_training_plan_compiles_and_covers_every_parameter(over, B, T, precision):
    """Host logic of the training schedule compiler (no GPU: plans are compiled over a CPU arena, nothing is launched): every
    parameter has a gradient writer in the backward schedule, the weight-packing problems cover every conv / linear weight in
    both layouts, the fused gradient-cast safety check holds, and side-stream launches never write activation gradients."""
    import torch
    from improved_diffusion import _native as N_
    model, _ = build(over)
    model.precision = precision
    S = over["image_size"]
    P = model.engine()._compile(B, T, S, S, torch.device("cpu"), train=True)
    refs = set()
    for fn, cls, f in P.bops:
        refs.update(v.data_ptr() for v in f.values() if isinstance(v, torch.Tensor))
    for dev, cls, items in P.pending:
        for it in items:
            refs.update(v.data_ptr() for v in it.values() if isinstance(v, torch.Tensor))
    base = P.pgrad.data_ptr()
    missing = [name for (name, p), off in zip(model.named_parameters(), P.flat_offs) if base + 4 * off not in refs]
    assert not missing, missing
    # flat layout = gradient-completion order (optim.completion_order): dense 16-byte aligned slots, head first, the conditioning
    # path (time MLP, FiLM projections, RPENets) last; the same layout FlatAdamW uses for parameters / moments / gradients
    from improved_diffusion.optim import model_flat_layout
    params, offs, total, order, n_early = model_flat_layout(model)
    assert offs == P.flat_offs and total == P.pgrad.numel() and sorted(order) == list(range(len(params)))
    names = [n for n, _ in model.named_parameters()]
    pos = 0
    for i in order:
        assert offs[i] == pos
        pos += (params[i].numel() + 3) // 4 * 4
    assert names[order[0]].startswith("out.") and all(
        n.startswith("time_embed.") or ".emb_layers." in n or ".rpe_net." in n for n in (names[i] for i in order[n_early:]))
    # gradient buckets: contiguous cover of the buffer, completion points strictly ascending, the last one = end of the schedule
    bk = P.grad_buckets
    assert len(bk) >= 2 and bk[0][0] == 0 and bk[-1][1] == total and all(a[1] == b[0] for a, b in zip(bk, bk[1:]))
    assert all(a[2] < b[2] for a, b in zip(bk, bk[1:])) and bk[-1][2] == len(P.bops) - 1
    segs = P.backward_segments()
    assert segs[0][0] == 0 and segs[-1][1] == len(P.bops) and all(a[1] == b[0] for a, b in zip(segs, segs[1:]))
    # no launch after a bucket's completion point writes into it
    for (b_lo, b_hi, done) in bk[:-1]:
        for j in range(done + 1, len(P.bops)):
            for v in P.bops[j][2].values():
                if isinstance(v, torch.Tensor) and base <= v.data_ptr() < base + 4 * total:
                    assert not (b_lo <= (v.data_ptr() - base) // 4 < b_hi), (P.bops[j][0], j, done)
    # every >= 2-D weight is packed for the forward and (except the stem: no input gradient) for the dgrad conv
    packed_fwd = {id(s_) for s_, _, _, _, _, _, mode in P.pack_problems if mode in (N_.PACK_TC_FWD, N_.PACK_SIMT_FWD)}
    convs = [p for n_, p in model.named_parameters() if p.dim() == 4 or (p.dim() == 2 and ("qkv" in n_ or "proj_out" in n_ or n_.endswith("rpe_net.out.weight")))]
    assert all(id(p) in packed_fwd for p in convs if p.dim() == 4)
    # side-stream launches only feed parameter gradients
    for i in P.bside:
        fn, _, f = P.bops[i]
        assert fn in ("fdm_conv_wgrad", "fdm_sum_parts") or (fn == "fdm_gn_bwd" and f["phases"] == 2), fn
    assert 0 <= P.bjoin_before <= len(P.bops)
    assert len(P.bops) > 2 * len(P.ops) - 40 and P.bflops > 1.9 * P.flops


@pytest.mark.parametrize("name", ["stages_hierarchy-2_T300", "stages_autoreg_T60"])
def test_stage_fixtures_are_consistent(name):
    """The stage lists generated from the live reference's sampling schemes (tests/golden/make_stages.py): every stage conditions
    only on finished frames, never exceeds max_frames, and the stages cover the video exactly once (SURVEY §8d: hierarchy-2 on a
    300-frame video = 27 stages, 534 model-frames per diffusion step)."""
    import json
    fx = json.load(open(os.path.join(ROOT, "tests", "golden", name + ".json")))
    done, generated = set(range(fx["n_obs"])), []
    for obs, lat in fx["stages"]:
        assert set(obs) <= done and len(obs) + len(lat) <= fx["max_frames"] and not (set(lat) & done)
        done |= set(lat)
        generated += lat
    assert done == set(range(fx["video_length"])) and len(generated) == len(set(generated))
    if name == "stages_hierarchy-2_T300":
        assert len(fx["stages"]) == 27 and sum(len(o) + len(l) for o, l in fx["stages"]) == 534


def test_torch_training_path_is_opt_in(monkeypatch):
    """No silent fallback: differentiating the model on a CPU tensor raises unless the PyTorch-autograd expression is asked for."""
    import torch
    model, _ = build(dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32))
    x = torch.zeros(1, 2, 4, 32, 32)
    kw = dict(x0=x, timesteps=torch.zeros(1), frame_indices=torch.tensor([[0, 1]]), obs_mask=torch.zeros(1, 2, 1, 1, 1),
              latent_mask=torch.ones(1, 2, 1, 1, 1))
    monkeypatch.delenv("FDM_ALLOW_TORCH_TRAIN", raising=False)
    monkeypatch.delenv("FDM_TRAIN_ENGINE", raising=False)
    with pytest.raises(RuntimeError, match="no silent CPU / PyTorch fallback"):
        model(x, **kw)
    monkeypatch.setenv("FDM_ALLOW_TORCH_TRAIN", "1")
    out, _ = model(x, **kw)
    assert out.shape == x.shape and out.requires_grad


def test_mask_sampler_matches_reference_goldens():
    """train_step.sample_all_masks / prepare_training_batch / sample_some_indices against outputs of the reference's TrainLoop
    methods (tests/golden/train_masks.json, made by tests/golden/make_train_masks.py from the live reference): same masks, frame
    indices, gathered frames AND the same RNG positions afterwards (torch + numpy), bit for bit."""
    import json
    import numpy as np
    from improved_diffusion import train_step as ts
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "train_masks.json")))
    for c in gold["cases"]:
        B, T = c["B"], c["T"]
        b1 = (1000 * torch.arange(B).view(B, 1) + torch.arange(T).view(1, T)).float().view(B, T, 1, 1, 1)
        b2 = -b1 - 1
        torch.manual_seed(c["seed"])
        np.random.seed(c["seed"])
        batch, fi, obs, lat = ts.sample_all_masks(b1, b2 if c["second"] else None, max_frames=c["max_frames"],
                                                  pad_with_random_frames=c["pad"])
        tail = [float(torch.rand(())), float(np.random.rand())]
        assert fi.tolist() == c["frame_indices"], c["seed"]
        assert batch.flatten(1).long().tolist() == c["batch"], c["seed"]
        assert obs.flatten(1).long().tolist() == c["obs"] and lat.flatten(1).long().tolist() == c["latent"], c["seed"]
        assert obs.shape == (B, len(c["obs"][0]), 1, 1, 1) and obs.dtype == b1.dtype and fi.dtype == torch.int64
        assert tail == c["tail"], c["seed"]
    torch.manual_seed(123)
    np.random.seed(123)
    draws = [ts.sample_some_indices(n, T) for n, T in [(5, 12), (20, 300), (40, 41), (3, 7), (20, 36)] for _ in range(200)]
    assert draws == gold["draws"]
    # gather=False returns the full-length masks; set_masks overrides the first rows
    torch.manual_seed(0)
    np.random.seed(0)
    b1 = torch.zeros(3, 12, 1, 2, 2)
    preset = {"obs": torch.ones(1, 12, 1, 1, 1), "latent": torch.zeros(1, 12, 1, 1, 1)}
    same, obs, lat = ts.sample_all_masks(b1, max_frames=5, gather=False, set_masks=preset)
    assert same is b1 and obs.shape == (3, 12, 1, 1, 1) and float(obs[0].sum()) == 12 and float(lat[0].sum()) == 0
    assert float((obs[1:] + lat[1:]).flatten(1).sum(1).max()) <= 5
    with pytest.raises(ValueError):
        ts.sample_all_masks(torch.zeros(1, 3, 1, 1, 1), max_frames=5)


def test_train_step_host_logic_cpu(tmp_path):
    """NativeTrainStep on CPU: the flat optimizer refuses (CUDA kernels only, no fallback); the explicit torch arm runs the host
    logic — microbatches, loss weighting, LR annealing, EMA, deferred log reads — and its records are self-consistent.
    (Parity of this arm with the reference's TrainLoop: tests/dropin_trainloop.py.)"""
    import numpy as np
    from improved_diffusion.train_step import NativeTrainStep, UniformTimesteps
    model, diffusion = build(dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32))
    with pytest.raises(RuntimeError):
        NativeTrainStep(model, diffusion, lr=1e-3, max_frames=5)
    with pytest.raises(ValueError):
        NativeTrainStep(model, diffusion, lr=1e-3, max_frames=5, optimizer="sgd")
    np.random.seed(0)
    t, w = UniformTimesteps(diffusion).sample(64, "cpu")
    assert t.dtype == torch.int64 and int(t.min()) >= 0 and int(t.max()) < 32 and torch.all(w == 1) and w.dtype == torch.float32
    runner = NativeTrainStep(model, diffusion, lr=1e-3, max_frames=5, optimizer="torch", microbatch=1, lr_anneal_steps=10,
                             ema_rate="0.5")
    before = [p.detach().clone() for p in model.parameters()]
    torch.manual_seed(1)
    np.random.seed(1)
    g = torch.Generator().manual_seed(2)
    vids = lambda: torch.randn(2, 12, 4, 32, 32, generator=g).clamp(-1, 1)
    first = runner.run_step(vids(), vids(), defer=True)
    second = runner.run_step(vids(), vids(), defer=True)
    last = runner.flush()
    assert first is None and second["step"] == 0 and last["step"] == 1 and runner.flush() is None
    assert second["lr"] == pytest.approx(1e-3) and last["lr"] == pytest.approx(1e-3 * 0.9) and last["samples"] == 4
    for rec in (second, last):
        quart = [k for k in rec if k.startswith("loss_q")]
        assert quart and rec["grad_norm"] > 0 and np.isfinite(rec["loss"])
        assert min(rec[k] for k in quart) - 1e-9 <= rec["loss"] <= max(rec[k] for k in quart) + 1e-9
        assert rec["loss"] == pytest.approx(rec["mse"])
    moved = [i for i, (a, p) in enumerate(zip(before, model.parameters())) if not torch.equal(a, p.detach())]
    assert len(moved) > 50
    i = moved[0]  # EMA with rate 0.5 after two steps sits strictly between the start and the current value
    e, p0, p2 = runner.ema_params[0][i], before[i], list(model.parameters())[i].detach()
    assert not torch.equal(e, p0) and not torch.equal(e, p2)
    # checkpoint files in the reference's layout (names, keys), and back
    path = runner.save(str(tmp_path), config={"max_frames": 5})
    assert sorted(os.listdir(tmp_path)) == ["ema_0.5_000001.pt", "model000001.pt", "opt000001.pt"]
    ck = torch.load(path)
    assert set(ck) == {"state_dict", "config", "step"} and ck["step"] == 1 and list(ck["state_dict"]) == list(model.state_dict())
    model_b, diffusion_b = build(dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32))
    runner_b = NativeTrainStep(model_b, diffusion_b, lr=1e-3, max_frames=5, optimizer="torch", ema_rate="0.5")
    assert runner_b.resume(str(tmp_path)) == 1
    assert all(torch.equal(a.detach(), b.detach()) for a, b in zip(model.parameters(), model_b.parameters()))
    assert all(torch.equal(a, b) for a, b in zip(runner.ema_params[0], runner_b.ema_params[0]))
    sa, sb = runner.opt.state_dict()["state"], runner_b.opt.state_dict()["state"]
    assert all(torch.equal(sa[i]["exp_avg"], sb[i]["exp_avg"]) and float(sa[i]["step"]) == float(sb[i]["step"]) for i in sa)


def test_native_training_refuses_dropout_loudly():
    """The reference applies nn.Dropout inside every ResBlock when --dropout > 0 (unet.py:167,203-206); the native schedules have
    no dropout mask, so training with it must raise instead of silently training without (ADVICE r1)."""
    import pytest as _pt
    from improved_diffusion.script_util import create_model_and_diffusion, model_and_diffusion_defaults
    d = model_and_diffusion_defaults()
    d.update(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32, dropout=0.1,
             diffusion_space_kwargs=dict(PIXEL))
    model, _ = create_model_and_diffusion(**d)
    model.train()
    x = torch.zeros(1, 2, 4, 32, 32)
    kw = dict(x0=x, timesteps=torch.zeros(1), frame_indices=torch.zeros(1, 2, dtype=torch.long), obs_mask=torch.zeros(1, 2, 1, 1, 1),
              latent_mask=torch.ones(1, 2, 1, 1, 1))
    with _pt.raises(NotImplementedError, match="dropout"):
        model.engine().forward_train(x, kw["x0"], kw["timesteps"], kw["frame_indices"], kw["obs_mask"], kw["latent_mask"])
    model.eval()  # dropout is the identity in eval mode: the engine must not object (it then fails later only for lack of a GPU)
    with _pt.raises(Exception) as ei:
        model.engine().forward_train(x, kw["x0"], kw["timesteps"], kw["frame_indices"], kw["obs_mask"], kw["latent_mask"])
    assert "dropout" not in str(ei.value)


def test_decode_denormalises_pre_encoded_latents():
    """gaussian_diffusion.py:933-947: pre-encoded latents are de-normalised (video * std + mean) before the VAE decoder; the VAE
    itself is pluggable (`diffusion.vae_decode`) and stays outside the hot path."""
    import pytest as _pt
    from improved_diffusion.script_util import create_model_and_diffusion, model_and_diffusion_defaults
    mean, std = torch.tensor([0.1, -0.2, 0.3, 0.0]), torch.tensor([1.5, 0.5, 2.0, 1.0])
    d = model_and_diffusion_defaults()
    d.update(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32,
             diffusion_space_kwargs=dict(diffusion_space="latent", pre_encoded=True, pre_encoded_stats_dict=dict(mean=mean, std=std)))
    _, diffusion = create_model_and_diffusion(**d)
    z = torch.randn(2, 3, 4, 8, 8)
    want = z * std.view(1, 1, 4, 1, 1) + mean.view(1, 1, 4, 1, 1)
    assert torch.equal(diffusion.denormalize(z), want)
    assert torch.equal(diffusion.encode(z), z)
    with _pt.raises(NotImplementedError, match="vae_decode"):
        diffusion.decode(z)
    seen = []

    def fake_vae(latents):  # [n, 4, h, w] -> [n, 3, 8h, 8w]
        seen.append(latents.clone())
        return latents[:, :3].repeat_interleave(8, dim=2).repeat_interleave(8, dim=3)
    diffusion.vae_decode = fake_vae
    out = diffusion.decode(z, chunk_size=4)
    assert out.shape == (2, 3, 3, 64, 64) and [s_.shape[0] for s_ in seen] == [4, 2]
    assert torch.equal(torch.cat(seen), want.flatten(0, 1))
    # pixel space: identity, untouched
    d["diffusion_space_kwargs"] = dict(PIXEL)
    _, dp = create_model_and_diffusion(**d)
    assert dp.decode(z) is z and dp.denormalize(z) is z
