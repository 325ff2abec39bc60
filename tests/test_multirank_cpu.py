"""CPU, world_size 2 over gloo: the N > 1 host logic — batch sharding of the sampler (no collective in the loop, one
final all_gather) and the DDP training step (gradient allreduce) through the public API."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import fdm_oracle as O

PIXEL = dict(diffusion_space="pixel", pre_encoded=False, pre_encoded_stats_dict=None)
SMALL = dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32, timestep_respacing="4")


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _build(over):
    from improved_diffusion.script_util import create_model_and_diffusion, model_and_diffusion_defaults
    d = model_and_diffusion_defaults()
    d.update(over)
    d["diffusion_space_kwargs"] = dict(PIXEL)
    model, diffusion = create_model_and_diffusion(**d)
    model.load_state_dict(O.init_state_dict(O.make_cfg(**over), seed=1), strict=True)
    return model, diffusion


class FakeDenoiser(torch.nn.Module):
    """Row-independent stand-in for the denoiser so the sampler's sharding logic can run on CPU."""

    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.tensor(0.37))

    def forward(self, x, *, x0, timesteps, frame_indices=None, obs_mask=None, latent_mask=None, return_attn_weights=False):
        t = timesteps.view(-1, 1, 1, 1, 1) / 1000.0
        fi = frame_indices.float().view(*frame_indices.shape, 1, 1, 1) / 100.0
        return self.w * torch.tanh(x * (1 - obs_mask) + x0 * obs_mask + t + fi), None


def _worker(rank, world, port, what, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    try:
        from improved_diffusion import sharding
        if what == "sample":
            _, diffusion = _build(SMALL)
            model = FakeDenoiser()
            cfg = O.make_cfg(**SMALL)
            B = 5  # ragged over 2 ranks: 3 + 2 rows
            inp = O.synthetic_inputs(cfg, B, 3, 1, seed=4)
            kw = {k: inp[k] for k in ("x0", "frame_indices", "obs_mask", "latent_mask")}
            diffusion._noise_fn = torch.zeros_like
            full = sharding.sample_sharded(diffusion, model, tuple(inp["x0"].shape), kw, noise=inp["x"], latent_mask=inp["latent_mask"])
            local, (lo, hi) = sharding.sample_sharded(diffusion, model, tuple(inp["x0"].shape), kw, noise=inp["x"], gather=False)
            ref, _ = diffusion.p_sample_loop(model, tuple(inp["x0"].shape), noise=inp["x"], model_kwargs=kw)
            assert (lo, hi) == sharding.shard_bounds(B, rank, world)
            assert torch.equal(full, ref), "sharded + gathered sampler differs from the unsharded one"
            assert torch.equal(local, ref[lo:hi])
        elif what == "train":
            over = dict(SMALL, timestep_respacing="")
            model, diffusion = _build(over)
            model.precision = "fp32"
            cfg = O.make_cfg(**over)
            inp = O.synthetic_inputs(cfg, 4, 3, 1, seed=9, pad_rows=(1,))
            t = torch.tensor([3, 11, 19, 27])
            g = torch.Generator().manual_seed(5)
            noise = torch.randn(inp["x0"].shape, generator=g)

            def loss_of(m, sl):
                kw = {k: inp[k][sl] for k in ("x0", "frame_indices", "obs_mask", "latent_mask")}
                terms = diffusion.training_losses(m, inp["x0"][sl], t[sl], model_kwargs=kw, noise=noise[sl],
                                                  latent_mask=1 - inp["obs_mask"][sl], eval_mask=inp["latent_mask"][sl])
                return terms["loss"].mean()

            # reference first (before DDP hooks exist): the same model, whole batch, one process
            loss_of(model, slice(0, 4)).backward()
            ref = {k: p.grad.clone() for k, p in model.named_parameters()}
            model.zero_grad()
            ddp = sharding.wrap_ddp(model)
            lo, hi = sharding.shard_bounds(4, rank, world)
            loss_of(ddp, slice(lo, hi)).backward()  # allreduce(avg) of per-shard mean-loss grads == full-batch mean-loss grads
            assert all(p.grad is not None for p in model.parameters())
            # tensors whose exact gradient is zero (a conv bias in front of a GroupNorm, the softmax-shift rpe_k.out.bias)
            # hold pure rounding noise: compare against a floor tied to the typical gradient norm, not to their own norm
            floor = 5e-2 * sorted(float(v.norm()) for v in ref.values())[len(ref) // 2]
            worst = max(float((p.grad - ref[k]).norm()) / max(float(ref[k].norm()), floor) for k, p in model.named_parameters())
            assert worst <= 1e-4, worst
        elif what == "flat":
            from improved_diffusion.engine import grad_route
            # the collective of FlatGradDataParallel (one mean-allreduce over a flat gradient buffer) and its parameter broadcast
            flat = torch.arange(10, dtype=torch.float32) * (rank + 1)
            sharding.allreduce_mean_(flat)
            assert torch.allclose(flat, torch.arange(10, dtype=torch.float32) * (1 + world) / 2)
            m = FakeDenoiser()
            with torch.no_grad():
                m.w.fill_(float(rank + 3))
            wrapped = sharding.FlatGradDataParallel(m)
            route = grad_route(m)
            assert float(m.w) == 3.0 and callable(route.reduce) and wrapped.module is m and wrapped.route is route
            g = torch.full((4,), float(rank))
            route.reduce(g)
            assert torch.allclose(g, torch.full((4,), (world - 1) / 2))
        elif what == "trainstep":
            # train_step.NativeTrainStep (host side of TrainLoop.run_step) under DDP, torch arm: per-rank data and masks, two
            # microbatches per step (DDP.no_sync() on the first, as train_util.py:311-315), identical weights on both ranks after
            import numpy as np
            from improved_diffusion.train_step import NativeTrainStep
            over = dict(SMALL, timestep_respacing="")
            model, diffusion = _build(over)
            model.precision = "fp32"
            runner = NativeTrainStep(model, diffusion, lr=1e-3, max_frames=4, optimizer="torch", microbatch=1, net=sharding.wrap_ddp(model))
            torch.manual_seed(100 + rank)
            np.random.seed(100 + rank)
            g = torch.Generator().manual_seed(200 + rank)
            recs = [runner.run_step(torch.randn(2, 9, 4, 32, 32, generator=g).clamp(-1, 1),
                                    torch.randn(2, 9, 4, 32, 32, generator=g).clamp(-1, 1)) for _ in range(2)]
            assert recs[1]["samples"] == 2 * 2 * world and recs[1]["step"] == 1 and recs[0]["grad_norm"] > 0
            flat = torch.cat([p.detach().flatten() for p in model.parameters()])
            both = [torch.zeros_like(flat) for _ in range(world)]
            dist.all_gather(both, flat)
            assert torch.equal(both[0], both[1]), "ranks diverged: the gradient exchange of the microbatched step is broken"
            losses = [torch.zeros(1, dtype=torch.float64) for _ in range(world)]
            dist.all_gather(losses, torch.tensor([recs[0]["loss"]], dtype=torch.float64))
            assert float(losses[0]) != float(losses[1])  # different data per rank
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("what", ["sample", "train", "flat", "trainstep"])
def test_two_ranks_gloo(tmp_path, what):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, what, str(tmp_path)), nprocs=2, join=True)
    assert all(os.path.exists(os.path.join(str(tmp_path), f"ok{r}")) for r in range(2))


def test_shard_bounds():
    from improved_diffusion.sharding import shard_bounds
    for n in (0, 1, 5, 8, 64):
        for w in (1, 2, 3, 8):
            b = [shard_bounds(n, r, w) for r in range(w)]
            assert b[0][0] == 0 and b[-1][1] == n and all(b[i][1] == b[i + 1][0] for i in range(w - 1))
            sizes = [hi - lo for lo, hi in b]
            assert max(sizes) - min(sizes) <= 1
