"""
Multi-GPU data parallelism for the hot path (SURVEY §8e), one process per GPU under torchrun:

  * sampling: the videos of a batch are independent through the whole sampler (GroupNorm is per frame / per pixel,
    attention is per (video, pixel) / (video, frame)), so the batch dimension is split across ranks with NO collective
    inside the loop — the reference does the same with SLURM array tasks (scripts/video_sample.py:192-201).  An optional
    one-shot all_gather returns the full batch on every rank.
  * training: torch DistributedDataParallel around the model exactly as train_util.py:118-125 (NCCL gradient allreduce
    over NVLink/NVSwitch, 128 MB buckets, broadcast_buffers=False); `wrap_ddp` is that call with the reference's arguments.
    `FlatGradDataParallel` is the B200-native alternative for the native training path: the backward schedule leaves ALL
    parameter gradients in one flat fp32 buffer, so the exchange is ONE NCCL allreduce over that buffer (no per-parameter
    hooks, no bucket copies) issued from inside the autograd node: the wrapper sets the `reduce` / `reduce_async` of the
    model's `engine.GradRoute`, and `no_sync()` its `synced`.
"""
import contextlib
import os

import torch as th
import torch.distributed as dist

from .engine import grad_route


def shard_bounds(n, rank, world):
    """Contiguous, balanced [lo, hi) of `n` batch rows for `rank`: the first n % world ranks get one extra row."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def _rank_world(group=None):
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def sample_sharded(diffusion, model, shape, model_kwargs, *, noise=None, gather=True, group=None, **kwargs):
    """diffusion.p_sample_loop over this rank's rows of the batch.  Returns the full [B,...] tensor when `gather`
    (ragged shards are padded for the all_gather and trimmed after), else this rank's rows and their (lo, hi)."""
    rank, world = _rank_world(group)
    B = shape[0]
    lo, hi = shard_bounds(B, rank, world)
    cut = lambda v: v[lo:hi] if isinstance(v, th.Tensor) and v.dim() > 0 and v.shape[0] == B else v
    local_kw = {k: cut(v) for k, v in (model_kwargs or {}).items()}
    for k in ("latent_mask",):
        if k in kwargs:
            kwargs[k] = cut(kwargs[k])
    if hi > lo:
        local, _ = diffusion.p_sample_loop(model, (hi - lo,) + tuple(shape[1:]), noise=cut(noise), model_kwargs=local_kw, **kwargs)
    else:
        dev = next(model.parameters()).device
        local = th.empty((0,) + tuple(shape[1:]), device=dev)
    if not gather or world == 1:
        return (local, (lo, hi)) if not gather else local
    width = (B + world - 1) // world
    pad = th.zeros((width,) + tuple(shape[1:]), device=local.device, dtype=local.dtype)
    pad[: hi - lo] = local
    parts = [th.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad, group=group)
    out = []
    for r, part in enumerate(parts):
        a, b = shard_bounds(B, r, world)
        out.append(part[: b - a])
    return th.cat(out, dim=0)


def wrap_ddp(model, device=None):
    """The DDP wrap of train_util.py:118-125 (CPU / gloo processes wrap without device_ids)."""
    from torch.nn.parallel import DistributedDataParallel as DDP
    kw = dict(broadcast_buffers=False, bucket_cap_mb=128, find_unused_parameters=False)
    if device is not None and th.device(device).type == "cuda":
        return DDP(model, device_ids=[device], output_device=device, **kw)
    return DDP(model, **kw)


def allreduce_mean_(flat, group=None):
    """In-place mean over the ranks of `group` (one collective; the NCCL kernel runs on NCCL's stream, ordered after the
    caller's current stream and before its later work)."""
    _, world = _rank_world(group)
    if world > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        flat.div_(world)
    return flat


def allreduce_mean_async(flat, group=None):
    """Start an in-place mean over the ranks of `group` and return a function that makes the CURRENT stream wait for it.  The
    collective runs on the process group's own stream, ordered after everything enqueued on the current stream so far; work
    enqueued on the current stream afterwards (the next backward segment) overlaps it."""
    _, world = _rank_world(group)
    if world <= 1:
        return lambda: None
    backend = dist.get_backend(group)
    if backend == "nccl":
        work = dist.all_reduce(flat, op=dist.ReduceOp.AVG, group=group, async_op=True)
        return work.wait
    work = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group, async_op=True)

    def finish():
        work.wait()
        flat.div_(world)
    return finish


class FlatGradDataParallel(th.nn.Module):
    """Data-parallel wrapper for the NATIVE training path (engine._DenoiserFn): parameters are broadcast from rank 0 once;
    the gradient exchange is a mean-allreduce of the flat parameter-gradient buffer, by default in a few BUCKETS that overlap the
    backward schedule (the buffer is laid out in gradient-completion order: each bucket is launched as soon as the backward has
    passed the point after which it is final); `overlap=False`: ONE allreduce after the whole backward.  Same call signature / state_dict as the wrapped model (`.module`, like DDP)."""

    def __init__(self, model, group=None, overlap=True):
        super().__init__()
        self.module, self.group = model, group
        _, world = _rank_world(group)
        if world > 1:
            for p in model.parameters():
                dist.broadcast(p.data, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
            # p.data writes do not bump the parameters' version counters: drop any packed inference weights / sampler graphs
            for eng in getattr(model, "_engines", {}).values():
                eng.invalidate()
        self.route = route = grad_route(model)
        route.reduce = lambda flat: allreduce_mean_(flat, group)
        # bucketed exchange overlapped with the backward schedule (engine.GradRoute.hand_over); `overlap=False` / FDM_DDP_OVERLAP=0
        # keeps the single allreduce after the whole backward
        if overlap and os.environ.get("FDM_DDP_OVERLAP", "1") != "0":
            route.reduce_async = lambda flat: allreduce_mean_async(flat, group)
        else:
            route.reduce_async = None

    @contextlib.contextmanager
    def no_sync(self):
        """Like DDP.no_sync(): backwards inside the context only accumulate locally; the first backward after it allreduces the
        accumulated gradient once.  Needs the flat-gradient mode (optim.FlatAdamW(..., model=model)), whose flat buffer is what
        gets reduced; as with DDP, do not mix synchronised and unsynchronised backwards between two zero_grad() calls other than
        `no_sync ... no_sync, sync`."""
        if self.route.sink is None:
            raise NotImplementedError("FlatGradDataParallel.no_sync() needs optim.FlatAdamW(..., model=model) (flat-gradient mode)")
        self.route.synced = False
        try:
            yield
        finally:
            self.route.synced = True

    def forward(self, x, **kwargs):
        if not x.is_cuda:
            raise NotImplementedError("FlatGradDataParallel synchronises the native (CUDA) backward; wrap CPU models with wrap_ddp")
        return self.module(x, **kwargs)
