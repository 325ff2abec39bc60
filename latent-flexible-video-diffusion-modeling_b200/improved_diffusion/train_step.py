"""
Host side of one training step — the caller immediately above `training_losses` (SURVEY §8f-2).

Restates, for the non-fp16 path, what `TrainLoop` does per step in improved_diffusion/train_util.py:
  * `sample_some_indices` (:180-191), `sample_all_masks` (:193-221), `prepare_training_batch` (:223-245): which frames of each
    video are observed / latent, and the gather of those frames (padded with random frames of a second batch) into the
    [B, max_frames, C, H, W] training batch;
  * `forward_backward` (:280-333): per microbatch  masks -> encode -> upload -> t, weights -> training_losses -> backward;
  * `optimize_normal` (:346-351), `_log_grad_norm` (:353-357), `_anneal_lr` (:359-365), `log_loss_dict` (:529-535).

The random draws (torch CPU generator, numpy global RNG) are consumed in the reference's order with the reference's dtypes, so a
run seeded like the reference sees the same masks, frame indices and timesteps — tests/dropin_trainloop.py checks two optimizer
steps against the reference's unmodified TrainLoop, tests/golden/train_masks.json pins the mask sampler where the reference is absent.

What changes is the cost once forward+backward takes ~3 ms (cfg2) instead of ~50:
  * the per-row Python gather loops (boolean indexing + 3 copies per video) become ONE index gather per tensor on whatever device
    the batch lives on, and one pinned non-blocking upload;
  * gradient norm = one reduction over the optimizer's flat gradient buffer instead of 390 `.item()` syncs;
  * AdamW + EMA = one launch (`optim.FlatAdamW`); data parallelism = one NCCL allreduce (`sharding.FlatGradDataParallel`), with
    `no_sync()` on all but the last microbatch like the reference's DDP usage;
  * the logged scalars (losses, quartile losses, gradient norm) come back in ONE device->host read after the step instead of
    3 `.item()` + 6 `.cpu()` calls inside it.

This module owns no kernels; it calls the hot path through the same public API a user does.
"""
import contextlib

import numpy as np
import torch as th
import torch.distributed as dist


def _np32(fn, x):
    """numpy's float32 routine `fn` on a 0-d float32 tensor, back as a 0-d float32 tensor (the reference applies np.log / np.exp
    to torch scalars: same routine, same rounding)."""
    return th.tensor(fn(x.numpy()), dtype=th.float32)


def sample_some_indices(max_indices, T):
    """1..max_indices frame indices in [0, T): evenly strided with a log-uniform stride and a uniform start (train_util.py:180-191).
    Draw order per attempt: th.randint (count), np.random.rand (stride), th.rand (start); every intermediate is a 0-d float32
    torch value exactly as upstream (`T / x` is torch's reciprocal(x) * T), so the truncation `int(start + k * stride)` agrees
    bit for bit.  Out-of-range attempts (rounding at the upper edge) are redrawn, as the reference's recursion does."""
    while True:
        count = th.randint(low=1, high=max_indices + 1, size=())
        u = np.random.rand()
        widest = T / (count - 0.999)
        stride = _np32(np.exp, u * _np32(np.log, widest))
        start = th.rand(()) * (T - stride * (count - 1))
        picks = [int(start + k * stride) for k in range(int(count))]
        if 0 <= min(picks) and max(picks) < T:
            return picks


def sample_mask_rows(B, T, max_frames):
    """The observed / latent frame flags of `sample_all_masks` (train_util.py:197-207) as two bool arrays [B, T].
    Per video: one group of latent frames, then groups alternately assigned (fair coin) to observed or latent; frames already
    flagged are dropped from a group; stop at the first group that would exceed `max_frames` flagged frames (that group is discarded)."""
    obs = np.zeros((B, T), dtype=bool)
    lat = np.zeros((B, T), dtype=bool)
    for o, l in zip(obs, lat):
        l[sample_some_indices(max_frames, T)] = True
        while True:
            if int(o.sum()) + int(l.sum()) == T:  # only reachable when T <= max_frames: upstream's loop never terminates from here
                raise ValueError(f"every one of the T={T} frames is flagged with max_frames={max_frames}: the mask sampler "
                                 "needs videos longer than max_frames (the reference hangs in this state)")
            target = o if float(th.rand(())) < 0.5 else l
            group = np.asarray(sample_some_indices(max_frames, T))
            group = group[~(o[group] | l[group])]
            if group.size > max_frames - int(o.sum()) - int(l.sum()):  # duplicates inside a group count, as upstream's len()
                break
            target[group] = True
    return obs, lat


def gather_plan(flags, T, max_frames, pad_with_random_frames):
    """Host-side index table of `prepare_training_batch` (train_util.py:228-241) from the [B, T] bool `flags` (observed | latent):
    returns (indices [B, eff_T] int64, n_real [B]).  Slots below n_real[b] hold the flagged frames in ascending order; the rest are
    padding: uniform random frame numbers (one th.randint per row, row order — the reference's randint_like draws) or 0."""
    B = flags.shape[0]
    n_real = flags.sum(axis=1)
    eff_T = max_frames if pad_with_random_frames else int(n_real.max())
    indices = th.zeros(B, eff_T, dtype=th.int64)
    for b in range(B):
        k = int(n_real[b])
        indices[b, :k] = th.from_numpy(np.flatnonzero(flags[b]))
        if pad_with_random_frames:
            indices[b, k:] = th.randint(high=T, size=(eff_T - k,), dtype=th.int64)
    return indices, n_real


def prepare_training_batch(mask, batch1, batch2, tensors, *, max_frames, pad_with_random_frames=True):
    """Same contract as TrainLoop.prepare_training_batch (train_util.py:223-245): select the frames of `batch1` flagged in `mask`
    [B, T, 1, 1, 1], pad every video to the common length with frames of `batch2` (or `batch1` when it is None) at random
    positions, and select the same positions of every tensor in `tensors` (always from the batch1-aligned tensor, padding
    included, as upstream).  Returns (new_batch, new_tensors, indices).  One gather per tensor instead of a Python loop per row;
    runs on the device the batch lives on (the index table is built on the host: it is B x max_frames integers)."""
    B, T = mask.shape[:2]
    flags = mask.reshape(B, T).cpu().numpy() != 0
    indices, n_real = gather_plan(flags, T, max_frames, pad_with_random_frames)
    dev = batch1.device
    idx = indices.to(dev)
    rows = th.arange(B, device=dev).unsqueeze(1)
    new_batch = batch1[rows, idx]
    if batch2 is not None:
        pad = th.arange(idx.shape[1]).unsqueeze(0) >= th.from_numpy(n_real).unsqueeze(1)  # [B, eff_T], host
        pb, pt = pad.nonzero(as_tuple=True)
        if pb.numel():
            pb, pt = pb.to(dev), pt.to(dev)
            new_batch[pb, pt] = batch2[pb, idx[pb, pt]]
    new_tensors = [t[th.arange(B, device=t.device).unsqueeze(1), indices.to(t.device)] for t in tensors]
    return new_batch, new_tensors, indices.to(mask.device)


def sample_all_masks(batch1, batch2=None, *, max_frames, pad_with_random_frames=True, gather=True, set_masks=None):
    """Same contract as TrainLoop.sample_all_masks (train_util.py:193-221): returns (batch, frame_indices, obs_mask, latent_mask)
    with masks shaped [B, max_frames, 1, 1, 1] in the batch's dtype, or (batch1, obs_mask, latent_mask) over all T frames when
    `gather=False`.  `set_masks={'obs': rows, 'latent': rows}` overrides the first rows (used upstream for logging)."""
    B, T = batch1.shape[:2]
    obs, lat = sample_mask_rows(B, T, max_frames)
    like = dict(dtype=batch1.dtype, device=batch1.device)
    masks = {"obs": th.from_numpy(obs).to(**like).view(B, T, 1, 1, 1), "latent": th.from_numpy(lat).to(**like).view(B, T, 1, 1, 1)}
    if set_masks is not None and len(set_masks["obs"]) > 0:
        for k in masks:
            n = min(len(set_masks[k]), B)
            masks[k][:n] = set_masks[k][:n]
    if not gather:
        return batch1, masks["obs"], masks["latent"]
    any_mask = (masks["obs"] + masks["latent"]).to(th.float32).clip(max=1).to(batch1.dtype)
    batch, (obs_mask, latent_mask), frame_indices = prepare_training_batch(
        any_mask, batch1, batch2, (masks["obs"], masks["latent"]), max_frames=max_frames,
        pad_with_random_frames=pad_with_random_frames)
    return batch, frame_indices, obs_mask, latent_mask


class UniformTimesteps:
    """`UniformSampler` of resample.py:42-67 (the TrainLoop default): t ~ np.random.choice(num_timesteps, p = uniform), weights 1."""

    def __init__(self, diffusion):
        self.n = diffusion.num_timesteps

    def sample(self, batch_size, device):
        p = np.ones([self.n]) / self.n
        t = np.random.choice(self.n, size=(batch_size,), p=p)
        w = 1 / (self.n * p[t])
        return th.from_numpy(t).long().to(device), th.from_numpy(w).float().to(device)


class NativeTrainStep:
    """`TrainLoop.run_step` (train_util.py:272-280) over the native stack: `run_step(batch1, batch2)` does forward_backward +
    optimize_normal and returns the scalars the reference logs (`loss`, `mse`, `eval-mse`, their `_q{0..3}` quartile means,
    `grad_norm`, `lr`, `step`, `samples`) as a dict of Python floats.

    optimizer="flat" (default): optim.FlatAdamW in flat-gradient mode with the EMA rates fused — CUDA only, raises otherwise.
    optimizer="torch": torch.optim.AdamW + per-tensor EMA exactly as upstream (used by the CPU parity test against the
    reference's TrainLoop; also the arm to A/B against).  With an initialised process group of more than one rank the model is
    wrapped in sharding.FlatGradDataParallel ("flat") or left to the caller ("torch": pass an already wrapped `net=`)."""

    def __init__(self, model, diffusion, *, lr, max_frames, weight_decay=0.0, ema_rate="0.9999", microbatch=-1,
                 pad_with_random_frames=True, schedule_sampler=None, lr_anneal_steps=0, optimizer="flat", net=None, device=None):
        self.model, self.diffusion = model, diffusion
        self.lr, self.max_frames, self.microbatch = lr, max_frames, microbatch
        self.pad_with_random_frames, self.lr_anneal_steps = pad_with_random_frames, lr_anneal_steps
        self.ema_rate = [ema_rate] if isinstance(ema_rate, float) else [float(x) for x in str(ema_rate).split(",") if x]
        self.schedule_sampler = schedule_sampler or UniformTimesteps(diffusion)
        self.device = th.device(device) if device is not None else next(model.parameters()).device
        self.world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        self.step = 0
        params = list(model.parameters())
        if optimizer == "flat":
            from .optim import FlatAdamW
            from .sharding import FlatGradDataParallel
            self.opt = FlatAdamW(params, lr=lr, weight_decay=weight_decay, ema_rates=tuple(self.ema_rate), model=model)
            self.net = net if net is not None else (FlatGradDataParallel(model) if self.world > 1 else model)
            self.ema_params = [self.opt.ema_params(i) for i in range(len(self.ema_rate))]
        elif optimizer == "torch":
            self.opt = th.optim.AdamW(params, lr=lr, weight_decay=weight_decay)
            self.net = net if net is not None else model
            self.ema_params = [[p.detach().clone() for p in params] for _ in self.ema_rate]
        else:
            raise ValueError(f"optimizer must be 'flat' or 'torch', got {optimizer!r}")
        self.flat = optimizer == "flat"
        self.params = params
        self._staging = {}
        self._copy_stream = None

    # ---- forward_backward (train_util.py:280-333)
    def forward_backward(self, batch1, batch2=None):
        self.opt.zero_grad()
        dev, pad = self.device, self.pad_with_random_frames
        mb = self.microbatch if self.microbatch > 0 else batch1.shape[0]
        logs = []
        for i in range(0, batch1.shape[0], mb):
            micro, frame_indices, obs_mask, latent_mask = sample_all_masks(
                batch1[i:i + mb], batch2[i:i + mb] if (pad and batch2 is not None) else None, max_frames=self.max_frames,
                pad_with_random_frames=pad)
            micro = self.diffusion.encode(micro) if hasattr(self.diffusion, "encode") else micro
            micro, frame_indices, obs_mask, latent_mask = (self._upload(n, x) for n, x in enumerate(
                (micro, frame_indices, obs_mask, latent_mask)))
            last = i + mb >= batch1.shape[0]
            t, weights = self.schedule_sampler.sample(micro.shape[0], dev)
            no_sync = getattr(self.net, "no_sync", None) if not last else None
            ctx = no_sync() if no_sync is not None else contextlib.nullcontext()
            with ctx:
                losses = self.diffusion.training_losses(
                    self.net, micro, t, model_kwargs=dict(frame_indices=frame_indices, obs_mask=obs_mask, latent_mask=latent_mask,
                                                          x0=micro),
                    latent_mask=(1 - obs_mask) if pad else latent_mask, eval_mask=latent_mask)
                if hasattr(self.schedule_sampler, "update_with_local_losses"):
                    self.schedule_sampler.update_with_local_losses(t, losses["loss"].detach())
                (losses["loss"] * weights).mean().backward()
            logs.append((t, {k: (v * weights).detach() for k, v in losses.items()}))
        return logs

    def _upload(self, slot, x):
        """Host tensor -> device through a persistent pinned staging buffer (allocated once per shape: cudaHostAlloc costs more
        than the step), asynchronous on the current stream; tensors already on the device pass through."""
        dev = self.device
        if x.device == dev or dev.type != "cuda":
            return x.to(dev)
        key = (slot, tuple(x.shape), x.dtype)
        if key not in self._staging:
            self._staging[key] = [th.empty(x.shape, dtype=x.dtype, pin_memory=True), None]
        buf, busy = self._staging[key]
        if busy is not None:
            busy.synchronize()  # the previous upload from this buffer (earlier microbatch) must have left the host
        buf.copy_(x)
        # the copy runs on its own stream so that, with deferred log reads, the upload of step i+1 overlaps the kernels of step i
        # (on the compute stream it would queue behind them and then delay the forward by its own duration)
        if self._copy_stream is None:
            self._copy_stream = th.cuda.Stream(dev)
        main = th.cuda.current_stream(dev)
        done = th.cuda.Event()
        with th.cuda.stream(self._copy_stream):
            y = buf.to(dev, non_blocking=True)
            done.record(self._copy_stream)
        main.wait_event(done)
        y.record_stream(main)
        self._staging[key][1] = done
        return y

    def grad_norm_sq(self):
        """Σ p.grad² as a 0-d device tensor: one reduction over the flat gradient buffer (its alignment padding is zero)."""
        if self.flat:
            return th.linalg.vector_norm(self.opt.flat_g).square()
        return th.stack(th._foreach_norm([p.grad for p in self.params])).square().sum()

    # ---- optimize_normal (train_util.py:346-365)
    def optimize(self):
        gsq = self.grad_norm_sq()
        if self.lr_anneal_steps:
            for group in self.opt.param_groups:
                group["lr"] = self.lr * (1 - self.step / self.lr_anneal_steps)
        self.opt.step()
        if not self.flat:
            with th.no_grad():
                for rate, ema in zip(self.ema_rate, self.ema_params):
                    th._foreach_mul_(ema, rate)
                    th._foreach_add_(ema, [p.detach() for p in self.params], alpha=1 - rate)
        return gsq

    def run_step(self, batch1, batch2=None, defer=False):
        """One optimizer step.  Returns this step's log dict; with `defer=True` the read is left in flight (asynchronous copy
        into pinned memory) and the PREVIOUS step's dict is returned instead (None on the first call; `flush()` returns the last
        one), so that the host side of step i+1 — mask sampling, gather, upload, launches — overlaps the GPU work of step i
        instead of waiting for it as every `.item()` of the reference's logging does."""
        logs = self.forward_backward(batch1, batch2)
        gsq = self.optimize()
        extra = dict(step=self.step, samples=(self.step + 1) * batch1.shape[0] * self.world, lr=self.opt.param_groups[0]["lr"])
        self.step += 1
        previous = self.flush()
        self._pending = self._start_read(logs, gsq, extra)
        return previous if defer else self.flush()

    def flush(self):
        """Finish the log read left in flight by `run_step(..., defer=True)`; None when there is none."""
        pending, self._pending = getattr(self, "_pending", None), None
        if pending is None:
            return None
        host, event, keys, sizes, extra = pending
        if event is not None:
            event.synchronize()
        out = self._reduce_logs(host.numpy().astype(np.float64), keys, sizes)
        out.update(extra)
        return out

    def _start_read(self, logs, gsq, extra):
        """log_loss_dict (train_util.py:529-535) + _log_grad_norm with ONE device->host read: [t | loss terms ...] per microbatch
        and the squared gradient norm are packed into one tensor; means and per-quartile means are formed on the host."""
        keys = list(logs[0][1].keys())
        packed = th.cat([th.cat([t.float()] + [terms[k].float() for k in keys]) for t, terms in logs] + [gsq.float().reshape(1)])
        sizes = [t.shape[0] for t, _ in logs]
        if packed.is_cuda:
            slot = self._log_slot = 1 - getattr(self, "_log_slot", 0)  # two pinned buffers: one in flight, one being read
            key = ("log", slot, packed.numel())
            if key not in self._staging:
                self._staging[key] = [th.empty(packed.numel(), dtype=th.float32, pin_memory=True), None]
            host = self._staging[key][0]
            host.copy_(packed, non_blocking=True)
            event = th.cuda.Event()
            event.record()
            return host, event, keys, sizes, extra
        return packed, None, keys, sizes, extra

    def _reduce_logs(self, host, keys, sizes):
        out, sums, off = {}, {}, 0
        for n in sizes:
            ts = host[off:off + n]
            for j, k in enumerate(keys):
                vals = host[off + (j + 1) * n: off + (j + 2) * n]
                sums.setdefault(k, []).append(vals.mean())  # logkv_mean of the microbatch mean, as upstream
                for tt, v in zip(ts, vals):
                    sums.setdefault(f"{k}_q{int(4 * tt / self.diffusion.num_timesteps)}", []).append(v)
            off += (len(keys) + 1) * n
        for k, v in sums.items():
            out[k] = float(np.mean(v))
        out["grad_norm"] = float(np.sqrt(host[-1]))
        return out


    # ---- checkpoint files in the reference's format (train_util.py:373-402 save, :137-173 resume)
    def save(self, directory, config=None):
        """Writes what TrainLoop.save() writes, under the same names: `model{step:06d}.pt` and `ema_{rate}_{step:06d}.pt`, each
        {"state_dict", "config", "step"}, and `opt{step:06d}.pt` (torch.optim.AdamW state_dict layout — FlatAdamW's is the same).
        `step` is the index of the last completed step, as upstream numbers its files.  Tensors are written as compact CPU copies
        (the parameters / moments / EMA copies are views of flat device buffers here).  Rank 0 writes; returns the model file's path."""
        import os
        step = max(self.step - 1, 0)
        if self.world > 1 and dist.get_rank() != 0:
            dist.barrier()
            return os.path.join(directory, f"model{step:06d}.pt")
        os.makedirs(directory, exist_ok=True)
        compact = lambda t: t.detach().cpu().clone()
        names = [n for n, _ in self.model.named_parameters()]

        def state_dict_of(params):
            sd = {k: compact(v) for k, v in self.model.state_dict().items()}
            sd.update({n: compact(p) for n, p in zip(names, params)})
            return sd

        for rate, params in [(0, self.params)] + list(zip(self.ema_rate, self.ema_params)):
            name = f"model{step:06d}.pt" if not rate else f"ema_{rate}_{step:06d}.pt"
            th.save({"state_dict": state_dict_of(params), "config": dict(config or {}), "step": step}, os.path.join(directory, name))
        osd = self.opt.state_dict()
        osd = {"state": {i: {k: (compact(v) if th.is_tensor(v) else v) for k, v in st.items()} for i, st in osd["state"].items()},
               "param_groups": osd["param_groups"]}
        th.save(osd, os.path.join(directory, f"opt{step:06d}.pt"))
        if self.world > 1:
            dist.barrier()
        return os.path.join(directory, f"model{step:06d}.pt")

    def resume(self, directory):
        """Loads the newest `model*.pt` of `directory` (find_resume_checkpoint, train_util.py:508-517), the matching EMA files
        and optimizer state when present, and continues from that file's step number, as TrainLoop.__init__ does.  Files written
        by the reference's TrainLoop and by `save()` are interchangeable.  Returns the step, or None when there is nothing to resume."""
        import glob
        import os
        found = {int(os.path.basename(f)[5:-3]): f for f in glob.glob(os.path.join(directory, "model*.pt"))}
        if not found:
            return None
        step = max(found)
        dev = self.device
        self.model.load_state_dict(th.load(found[step], map_location=dev)["state_dict"])
        names = [n for n, _ in self.model.named_parameters()]
        with th.no_grad():
            for rate, ema in zip(self.ema_rate, self.ema_params):
                path = os.path.join(directory, f"ema_{rate}_{step:06d}.pt")
                src = th.load(path, map_location=dev)["state_dict"] if os.path.exists(path) else dict(zip(names, self.params))
                for n, e in zip(names, ema):
                    e.copy_(src[n])
        path = os.path.join(directory, f"opt{step:06d}.pt")
        if os.path.exists(path):
            self.opt.load_state_dict(th.load(path, map_location=dev))
        self.step = step
        return step
