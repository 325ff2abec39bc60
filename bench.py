#!/usr/bin/env python
"""
bench.py — denoiser frame-steps/s (sampling) of the FDM hot path on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one diffusion step of the sampler over one batch: UNetVideoModel forward (the whole kernel schedule)
+ the fused posterior update + the step's Gaussian noise draw, i.e. what `diffusion.p_sample` does.  One step
processes B*K frame-steps per GPU.  Multi-GPU = the video batch sharded over ranks, no data-path collective
(weak scaling: B videos per GPU fixed), launched by torchrun (one process per GPU).

Lines printed (rank 0, ONE JSON line): see README/DESIGN.md §measurement for every key.
  value     : whole-job frame-steps/s with inputs resident in HBM (CUDA events, L2 flushed between steps, max over ranks)
  e2e       : same metric through diffusion.p_sample_loop with pinned HOST inputs, H2D + D2H inside the timed region
  roofline  : the dominant kernel class (implicit-GEMM convs) timed alone with CUDA events: algorithmic FLOPs / time
  cpu_baseline : the CPU oracle (port of the reference path) timed on this box's host cores on a bounded sample
  --impl reference : times that CPU path only (rank 0), same workload/metric.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "latent-flexible-video-diffusion-modeling_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch as th  # noqa: E402

PIXEL = dict(diffusion_space="pixel", pre_encoded=False, pre_encoded_stats_dict=None)

# BASELINE.json configs.  `B` is videos PER GPU (weak scaling).
WORKLOADS = {
    # cfg4: hierarchy-2 sampling, 300-frame video, batch 64 sharded over 8 GPUs -> 8 videos/GPU, stage of K=20 frames,
    # Carla-latent model of cfg2 (nc=64, nrb=1, 4x32x32 latents), 1000-step schedule.  The sampling headline.
    "cfg4-sampling": dict(over=dict(image_size=32, in_channels=4, num_channels=64, num_res_blocks=1, diffusion_steps=1000),
                          B=8, K=20, n_obs=10, video_len=300),
    # cfg2 shape (batch 1, K=5): launch-latency bound by construction
    "cfg2-sampling-b1": dict(over=dict(image_size=32, in_channels=4, num_channels=64, num_res_blocks=1, diffusion_steps=1000),
                             B=1, K=5, n_obs=3, video_len=20),
    # cfg1: the reference's own CPU-runnable case
    "cfg1-sampling": dict(over=dict(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32),
                          B=1, K=5, n_obs=3, video_len=20),
    # cfg5: long-context temporal attention stress (nc=128, K=40, 4x64x64 latents)
    "cfg5-sampling": dict(over=dict(image_size=64, in_channels=4, num_channels=128, num_res_blocks=1, diffusion_steps=1000),
                          B=2, K=40, n_obs=20, video_len=300),
    # cfg3's model used as a sampler (pixel space, 128x128x3, nc=128, K=20, 2 videos per GPU): the 128-wide halo convs
    "cfg3-sampling": dict(over=dict(image_size=128, in_channels=3, num_channels=128, num_res_blocks=1, diffusion_steps=1000),
                          B=2, K=20, n_obs=10, video_len=300),
}
DEFAULT_WORKLOAD = "cfg4-sampling"


def random_state_dict(model, seed=1):
    """Random NON-ZERO weights (a freshly constructed model outputs eps == 0: zero_module, reference nn.py:68-74)."""
    g = th.Generator().manual_seed(seed)
    sd = {}
    for k, v in model.state_dict().items():
        if v.dim() > 1:
            sd[k] = th.randn(v.shape, generator=g) / (v[0].numel() ** 0.5)
        elif k.endswith(".weight"):
            sd[k] = 1.0 + 0.1 * th.randn(v.shape, generator=g)
        else:
            sd[k] = 0.1 * th.randn(v.shape, generator=g)
    return sd


def synthetic_batch(cfg_over, B, K, n_obs, video_len, seed):
    g = th.Generator().manual_seed(seed)
    C, S = cfg_over["in_channels"], cfg_over["image_size"]
    x0 = th.randn(B, K, C, S, S, generator=g).clamp(-1, 1)
    fi = th.stack([th.sort(th.randperm(video_len, generator=g)[:K]).values for _ in range(B)]).long()
    obs = th.zeros(B, K, 1, 1, 1)
    obs[:, :n_obs] = 1
    return dict(x0=x0, frame_indices=fi, obs_mask=obs, latent_mask=1 - obs)


def build_native(over, device):
    from improved_diffusion.script_util import create_model_and_diffusion, model_and_diffusion_defaults
    d = model_and_diffusion_defaults()
    d.update(over)
    d["diffusion_space_kwargs"] = dict(PIXEL)
    model, diffusion = create_model_and_diffusion(**d)
    sd = random_state_dict(model)
    model.load_state_dict(sd, strict=True)
    model.to(device).eval()
    return model, diffusion, sd


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe) through NVML on a polling thread
    (5 ms period) that is started >= 0.5 s before the region; only samples inside [mark_begin, mark_end] are reported.  Falls back
    to `nvidia-smi -lms` when the NVML bindings are missing."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.thread = index, [], False, None
        self.t0 = self.t1 = None
        self.nv = self.handle = None
        self.proc = self.path = None

    def _handle(self):
        import pynvml as nv
        nv.nvmlInit()
        try:
            uuid = str(th.cuda.get_device_properties(self.index).uuid)
            h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            h = nv.nvmlDeviceGetHandleByIndex(phys)
        return nv, h

    def start(self):
        try:
            self.nv, self.handle = self._handle()
            self.max_mhz = float(self.nv.nvmlDeviceGetMaxClockInfo(self.handle, self.nv.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            return self._start_smi()

        def poll():
            nv, h = self.nv, self.handle
            while not self.stop_flag:
                try:
                    mhz = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    try:
                        rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                    except Exception:
                        rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                    try:
                        pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                    except Exception:
                        pw = None
                    self.samples.append((time.perf_counter(), mhz, rs, pw))
                except Exception:
                    pass
                time.sleep(0.005)
        self.thread = threading.Thread(target=poll, daemon=True)
        self.thread.start()
        time.sleep(0.5)

    def _start_smi(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=f, stderr=subprocess.DEVNULL)
            time.sleep(1.0)
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": None}
        if self.nv is not None:
            self.stop_flag = True
            if self.thread is not None:
                self.thread.join(timeout=2)
            inside = [x for x in self.samples if self.t0 is not None and self.t0 <= x[0] <= (self.t1 or x[0])]
            use = inside
            if use:
                reasons = sorted({name for _, _, rs, _ in use for name, bit in self.REASONS if rs & bit})
                pw = [x[3] for x in use if x[3] is not None]
                out.update(sm_mhz=statistics.median(x[1] for x in use), sm_min_mhz=min(x[1] for x in use), sm_max_mhz=self.max_mhz,
                           reasons=reasons, samples=len(use), power_w_max=max(pw) if pw else None,
                           source="NVML polled every 5 ms on a thread, samples inside the timed region only",
                           region_ms=1e3 * ((self.t1 or 0) - (self.t0 or 0)))
            return out
        if self.proc is None:
            return out
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 7:
                    continue
                try:
                    sm.append(float(c[0]))
                    mx.append(float(c[1]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm),
                       source="nvidia-smi -lms 20 (NVML bindings unavailable); includes ~1 s before the region")
        return out


def config_dict(workload, wl, world):
    """The workload description both arms print (identical keys and values: the driver compares them)."""
    over = wl["over"]
    return {"workload": workload, "videos_per_gpu": wl["B"], "frames_per_stage": wl["K"], "n_obs": wl["n_obs"],
            "latent": [over["in_channels"], over["image_size"], over["image_size"]], **over,
            "sharding": f"video batch over {world} rank(s), no collective",
            "l2": "flushed between timed steps (192 MB memset outside the event pairs)",
            "weights": "random non-zero init (zero_module tensors re-randomised)"}


DUMP_LIMIT_BYTES = 64_000_000 - 4096  # 64 MB in all, .npy headers (128 bytes each) included


def dump_outputs(directory, arrays):
    """Write each tensor as DIR/<name>.npy in float32, in its own shape.  When all of them together exceed DUMP_LIMIT_BYTES, each
    is cut to a fixed, seeded sample of its flat elements (the same elements on every run for the same shapes)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    total = sum(4 * a.numel() for a in arrays.values())
    for name, a in arrays.items():
        out = a.detach().float().cpu()
        if total > DUMP_LIMIT_BYTES:
            keep = out.numel() * DUMP_LIMIT_BYTES // total
            idx = th.randperm(out.numel(), generator=th.Generator().manual_seed(0))[:keep].sort().values
            out = out.flatten()[idx]
        np.save(os.path.join(directory, name + ".npy"), out.numpy())


def cpu_port_steps(over, B, K, batch, sd, n_steps, warmup, threads):
    """The reference path on host cores through the oracle PORT (oracle/fdm_oracle.py), fp32 torch CPU ops.  Only used when the
    real reference (oracle/_ref) is not available.  Checker/baseline only."""
    from oracle import fdm_oracle as O
    th.set_num_threads(threads)
    cfg = O.make_cfg(**over)
    tab = O.Tables(cfg)
    g = th.Generator().manual_seed(123)
    x = th.randn(batch["x0"].shape, generator=g)
    times = []
    n = tab.num_timesteps
    with th.no_grad():
        for s in range(warmup + n_steps):
            t = th.full((B,), n - 1 - (s % n), dtype=th.int64)
            noise = th.randn(x.shape, generator=g)
            t0 = time.perf_counter()
            out = O.p_sample(tab, sd, cfg, x, t, noise, batch)
            dt = time.perf_counter() - t0
            x = out["sample"]
            if s >= warmup:
                times.append(dt)
    return times


def build_reference(over, sd, device):
    """The UNMODIFIED reference (oracle/_ref, shipped by oracle/make_ref.sh): its own create_model_and_diffusion + strict load."""
    from oracle import ref_loader as R
    model, diffusion = R.create_reference(over)
    model.load_state_dict(sd, strict=True)
    return model.to(device).eval(), diffusion


def reference_sampling_steps(model, diffusion, batch, n_steps, warmup, device, autocast=False):
    """`diffusion.p_sample` of the reference (gaussian_diffusion.py:369-401), one call per diffusion step, stock code path.
    Returns per-step seconds (wall clock around a synchronised call on CUDA)."""
    kw = {k: v.to(device) for k, v in batch.items()}
    B = kw["x0"].shape[0]
    x = th.randn(kw["x0"].shape, generator=th.Generator().manual_seed(123)).to(device)
    n = diffusion.num_timesteps
    cuda = th.device(device).type == "cuda"
    times = []
    ctx = th.autocast("cuda", dtype=th.bfloat16) if autocast else th.autocast("cpu", enabled=False)
    with th.no_grad(), ctx:
        for s in range(warmup + n_steps):
            t = th.full((B,), n - 1 - (s % n), dtype=th.int64, device=device)
            if cuda:
                th.cuda.synchronize()
            t0 = time.perf_counter()
            out = diffusion.p_sample(model, x, t, clip_denoised=True, model_kwargs=kw)
            x = out["sample"].float()
            if cuda:
                th.cuda.synchronize()
            if s >= warmup:
                times.append(time.perf_counter() - t0)
    assert bool(th.isfinite(x).all())
    return times


def cpu_reference(over, B, K, batch, sd, n_steps, warmup):
    """CPU baseline: the real reference when oracle/_ref exists (kind "reference"), else the oracle port (kind "port")."""
    threads = os.cpu_count() or 1
    th.set_num_threads(threads)
    from oracle import ref_loader as R
    sd_cpu = {k: v.detach().cpu() for k, v in sd.items()}
    if R.find_ref() is not None:
        model, diffusion = build_reference(over, sd_cpu, "cpu")
        times = reference_sampling_steps(model, diffusion, batch, n_steps, warmup, "cpu")
        kind, what = "reference", f"UNMODIFIED reference (oracle/_ref), diffusion.p_sample on CPU, fp32, {threads} torch threads"
    else:
        times = cpu_port_steps(over, B, K, batch, sd_cpu, n_steps, warmup, threads)
        kind, what = "port", f"oracle port of the reference path (oracle/_ref absent), fp32 torch CPU ops, {threads} threads"
    total = sum(times)
    return {"value": B * K * len(times) / total, "unit": "frame-steps/s", "cores": threads, "kind": kind,
            "ms_per_step": 1e3 * total / len(times), "ms_per_step_min": 1e3 * min(times), "ms_per_step_max": 1e3 * max(times),
            "sample": f"{len(times)} diffusion steps (after {warmup} warm-up) of the same B={B},K={K} batch: {what}"}


def run_reference(args, wl, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (oracle/_ref: unmodified `diffusion.p_sample` over the
    unmodified `UNetVideoModel`), all host threads, same workload / metric / config.  Rank 0 only."""
    if rank != 0:
        return
    over, B, K = wl["over"], wl["B"], wl["K"]
    from improved_diffusion.script_util import create_model_and_diffusion, model_and_diffusion_defaults
    d = model_and_diffusion_defaults()
    d.update(over)
    d["diffusion_space_kwargs"] = dict(PIXEL)
    model, _ = create_model_and_diffusion(**d)
    sd = random_state_dict(model)
    batch = synthetic_batch(over, B, K, wl["n_obs"], wl["video_len"], seed=0)
    cpu = cpu_reference(over, B, K, batch, sd, max(1, args.steps), max(1, args.warmup))
    v = cpu["value"]
    line = {"impl": "reference", "metric": "denoiser frame-steps/sec (sampling)", "value": v, "unit": "frame-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": cpu["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args.workload, wl, world),
            "cpu_baseline": cpu,
            "e2e": {"value": v, "unit": "frame-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def gpu_eager_sampling(over, batch, sd, dev, B, K, n_steps=10, warmup=3):
    """The kernel set to beat (SURVEY §8d): the UNMODIFIED reference in PyTorch eager on the SAME B200 — fp32 (TF32 off, the
    reference's numerics) and under torch.autocast(bfloat16) (cuDNN / cuBLAS bf16 tensor-core kernels)."""
    from oracle import ref_loader as R
    if R.find_ref() is None:
        return {"unavailable": "oracle/_ref missing (run oracle/make_ref.sh in the build container)"}
    old = (th.backends.cudnn.allow_tf32, th.backends.cuda.matmul.allow_tf32)
    th.backends.cudnn.allow_tf32 = th.backends.cuda.matmul.allow_tf32 = False
    out = {"what": "unmodified reference (oracle/_ref) diffusion.p_sample in PyTorch eager on this GPU, per-step wall clock "
                   f"with synchronisation, {n_steps} steps after {warmup} warm-up"}
    try:
        model, diffusion = build_reference(over, {k: v.detach().cpu() for k, v in sd.items()}, dev)
        for tag, ac in (("fp32", False), ("autocast_bf16", True)):
            ts = reference_sampling_steps(model, diffusion, batch, n_steps, warmup, dev, autocast=ac)
            out[tag] = {"value": B * K * len(ts) / sum(ts), "unit": "frame-steps/s", "ms_per_step": 1e3 * sum(ts) / len(ts)}
        del model
    finally:
        th.backends.cudnn.allow_tf32, th.backends.cuda.matmul.allow_tf32 = old
        th.cuda.empty_cache()
    return out


def gpu_eager_training(over, B, K, dev, sd, n_steps=4, warmup=2):
    """The unmodified reference's training step in PyTorch eager on this GPU: training_losses + backward + torch AdamW."""
    from oracle import ref_loader as R
    if R.find_ref() is None:
        return {"unavailable": "oracle/_ref missing"}
    old = (th.backends.cudnn.allow_tf32, th.backends.cuda.matmul.allow_tf32)
    th.backends.cudnn.allow_tf32 = th.backends.cuda.matmul.allow_tf32 = False
    out = {"what": "unmodified reference (oracle/_ref): diffusion.training_losses + backward + torch.optim.AdamW in PyTorch eager "
                   "on this GPU (CUDA events)"}
    try:
        model, diffusion = build_reference(over, {k: v.detach().cpu() for k, v in sd.items()}, dev)
        model.train()
        opt = th.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.0)
        batch = {k: v.to(dev) for k, v in synthetic_batch(over, B, K, 3, 4 * K, seed=1).items()}
        g = th.Generator(device=dev).manual_seed(0)
        for tag, ac in (("fp32", False), ("autocast_bf16", True)):
            def step():
                t = th.randint(0, diffusion.num_timesteps, (B,), device=dev, generator=g)
                with th.autocast("cuda", dtype=th.bfloat16, enabled=ac):
                    terms = diffusion.training_losses(model, batch["x0"], t, model_kwargs=batch, latent_mask=1 - batch["obs_mask"],
                                                      eval_mask=batch["latent_mask"])
                opt.zero_grad(set_to_none=True)
                terms["loss"].float().mean().backward()
                opt.step()
            for _ in range(warmup):
                step()
            th.cuda.synchronize()
            e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n_steps):
                step()
            e1.record()
            th.cuda.synchronize()
            ms = e0.elapsed_time(e1) / n_steps
            out[tag] = {"value": B / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms}
        del model, opt
    except Exception as ex:  # e.g. out of memory on the eager arm: report, do not hide
        out["error"] = repr(ex)[:300]
    finally:
        th.backends.cudnn.allow_tf32, th.backends.cuda.matmul.allow_tf32 = old
        th.cuda.empty_cache()
    return out


def _peak_tflops():
    """(dense bf16 TFLOP/s, source): the driver-measured cuBLAS number of this pool's B200s, else the profiling recipe's fallback"""
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"]), "measured"
    except Exception:
        return 1590.0, "fallback"


TRAIN_WORKLOADS = {
    # BASELINE.json configs[1]: Carla-latent, nc = 64, K = 5, batch 1, on 1 B200
    "cfg2-train": (dict(image_size=32, in_channels=4, num_channels=64, num_res_blocks=1, diffusion_steps=1000), 1, 5, 20),
    # BASELINE.json configs[2]: Carla pixel-scale, nc = 128, K = 20, 128x128x3 frames, batch 2 PER GPU (DDP over the box)
    "cfg3-train": (dict(image_size=128, in_channels=3, num_channels=128, num_res_blocks=1, diffusion_steps=1000), 2, 20, 6),
    # BASELINE.json configs[4] as a training shape (not part of the default run): long-context model, K = 40, 4x64x64 latents
    "cfg5-train": (dict(image_size=64, in_channels=4, num_channels=128, num_res_blocks=1, diffusion_steps=1000), 2, 40, 6),
    # cfg4's shard shape as a training step (8 videos x 20 frames of 4x32x32 latents, nc = 64)
    "cfg4-train": (dict(image_size=32, in_channels=4, num_channels=64, num_res_blocks=1, diffusion_steps=1000), 8, 20, 10),
}


def bench_train(dev, world, precision, workload="cfg2-train", warmup=3):
    """train samples/s: one training_losses forward + backward (+ DDP gradient allreduce over NCCL when world > 1) + AdamW step
    per iteration, per-GPU batch fixed (weak scaling).  Forward AND backward run on the native kernel schedules
    (engine._DenoiserFn, CUDA-graph replays); the UNMODIFIED reference's training step in PyTorch eager on the same GPU (fp32 and
    autocast-bf16, oracle/_ref) is timed beside it as `gpu_eager` (single-GPU runs only)."""
    import torch.distributed as dist
    over, B, K, steps = TRAIN_WORKLOADS[workload]
    model, diffusion, _ = build_native(over, dev)
    model.precision = precision
    model.train()
    net = model
    if world > 1:
        from improved_diffusion import sharding
        # FDM_DDP=torch: torch DistributedDataParallel exactly as train_util.py:118-125 (drop-in path, per-parameter hooks);
        # default: one allreduce over the native backward's flat gradient buffer
        net = sharding.wrap_ddp(model, dev) if os.environ.get("FDM_DDP", "flat") == "torch" else sharding.FlatGradDataParallel(model)
    # FDM_OPT=torch: torch.optim.AdamW(fused=True) (multi-tensor kernels over the 390 tensors); default: optim.FlatAdamW — the same
    # update rule as ONE fdm_adamw launch over flat parameter / moment / gradient buffers (SURVEY §8f-2)
    if os.environ.get("FDM_OPT", "flat") == "torch":
        opt = th.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.0, fused=True)
    else:
        from improved_diffusion.optim import FlatAdamW
        # flat-gradient mode (model=...) needs the flat data-parallel wrapper, not torch DDP's per-parameter hooks
        opt = FlatAdamW(model.parameters(), lr=1e-4, weight_decay=0.0,
                        model=None if (world > 1 and os.environ.get("FDM_DDP", "flat") == "torch") else model)
    batch = {k: v.to(dev) for k, v in synthetic_batch(over, B, K, 3, 4 * K, seed=1 + int(os.environ.get("RANK", "0"))).items()}
    g = th.Generator(device=dev).manual_seed(0)

    def step():
        t = th.randint(0, diffusion.num_timesteps, (B,), device=dev, generator=g)
        terms = diffusion.training_losses(net, batch["x0"], t, model_kwargs=batch, latent_mask=1 - batch["obs_mask"],
                                          eval_mask=batch["latent_mask"])
        opt.zero_grad(set_to_none=True)
        terms["loss"].mean().backward()
        opt.step()
        return terms["loss"]

    def timed(engine, n):
        os.environ["FDM_TRAIN_ENGINE"] = engine
        for _ in range(warmup):
            step()
        th.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            loss = step()
        e1.record()
        th.cuda.synchronize()
        assert bool(th.isfinite(loss).all()), "training loss is not finite"
        ms = th.tensor([e0.elapsed_time(e1)], device=dev, dtype=th.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / n

    ms = timed("native", steps)
    plan = next(iter(model.engine().train_plans.values()))
    flops = plan.flops + plan.bflops
    out = {"metric": "train samples/sec", "value": world * B / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms,
           "steps": steps,
           "config": {"workload": workload, "batch_per_gpu": B, "frames": K, **over, "optimizer": "AdamW, weight_decay 0 (" + type(opt).__name__ + ")"},
           "launches_per_step": {"forward": plan.n_launches, "backward": plan.n_bwd_launches},
           "roofline": {"bound": "tensor", "achieved": flops / (ms * 1e-3) / 1e12, "unit": "TFLOP/s", "peak": _peak_tflops()[0],
                        "peak_source": _peak_tflops()[1], "frac": flops / (ms * 1e-3) / 1e12 / _peak_tflops()[0],
                        "flops_per_step": flops, "what": "algorithmic fwd + dgrad + wgrad + attention FLOPs of one step / step time "
                                                         "(optimizer, loss and host work included in the time)"},
           "path": "native: forward + backward kernel schedules of libfdm_sm100.so behind one autograd node (conv dgrad and wgrad on "
                   "tcgen05, GroupNorm / attention / RPENet backward kernels); n_gpus > 1: ONE NCCL allreduce over the flat gradient "
                   "buffer per step (sharding.FlatGradDataParallel; FDM_DDP=torch selects torch DDP as in train_util.py:118-125)"}
    del opt, net
    if world == 1:
        sd_host = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
        try:
            out["e2e"] = _train_e2e(model, diffusion, over, B, K, steps)
        except Exception as ex:  # the device-resident number above stands on its own; say what went wrong instead of hiding it
            out["e2e"] = {"error": repr(ex)[:300]}
    del model
    th.cuda.empty_cache()
    if world == 1 and os.environ.get("FDM_BENCH_GPU_EAGER", "1") != "0":
        out["gpu_eager"] = gpu_eager_training(over, B, K, dev, sd_host)
    return out


def _train_e2e(model, diffusion, over, B, K, steps):
    """The same training step end to end through train_step.NativeTrainStep with HOST video batches (3K frames each): per step
    mask sampling (the reference's draw order), frame gather, pinned upload, native forward + backward, gradient norm, FlatAdamW +
    EMA, and one device->host read of the logged scalars (left in flight: `defer=True`).  Wall clock around the loop."""
    import numpy as np
    from improved_diffusion.train_step import NativeTrainStep
    os.environ["FDM_TRAIN_ENGINE"] = "native"
    runner = NativeTrainStep(model, diffusion, lr=1e-4, max_frames=K, ema_rate="0.9999")
    C, S, T = over["in_channels"], over["image_size"], 3 * K
    g = th.Generator().manual_seed(5)
    pool = [th.randn(B, T, C, S, S, generator=g).clamp(-1, 1) for _ in range(4)]
    th.manual_seed(6)
    np.random.seed(6)
    for i in range(3):
        runner.run_step(pool[i % 4], pool[(i + 1) % 4], defer=True)
    runner.flush()
    th.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        runner.run_step(pool[i % 4], pool[(i + 1) % 4], defer=True)
    rec = runner.flush()
    th.cuda.synchronize()
    ms = (time.perf_counter() - t0) / steps * 1e3
    assert np.isfinite(rec["loss"]) and np.isfinite(rec["grad_norm"]), rec
    return {"value": B / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms,
            "h2d_bytes_per_step": B * K * (C * S * S * 4 + 8 + 4 + 4), "d2h_bytes_per_step": (4 * B + 1) * 4,
            "what": f"NativeTrainStep.run_step on host batches [B={B}, T={T}, {C}, {S}, {S}] fp32 (masks, gather, upload, fwd, bwd, "
                    "grad norm, AdamW+EMA, log read)"}


def kernel_classes(P, N_, B, K, Cx, S, osz=2):
    """Forward launches of the plan grouped by kernel class, each with its algorithmic FLOPs and bytes (per step).
    Bytes = every operand read once + every output written once (what a perfectly cached implementation moves through HBM)."""
    def is_halo(st):
        if not (st.engine == N_.CONV_TC and st.ksize == 3 and st.stride == 1 and not st.out_nchw):
            return False
        # (upsample convs run in the halo kernel's phase mode on the LOW-resolution Hin x Win input; their FLOPs are counted as the
        #  3x3 conv over the upsampled tensor — the algorithm the reference runs — although the kernel executes 4/9 of them)
        return st.Win in (16, 32, 64, 128) and st.Hin % max(1, 128 // st.Win) == 0 and st.Cout >= 32 and st.Cout % 4 == 0 and st.C0 % 8 == 0

    def is_halo_pointwise(st):
        # wide 1x1 linears (Cin >= 256) run through the halo kernel's pointwise mode (conv_simt.cu: fdm_conv dispatch)
        if not (st.engine == N_.CONV_TC and st.ksize == 1 and st.stride == 1 and st.C0 >= 256 and not st.out_nchw and not st.resid_norm):
            return False
        if st.Cout < 32 or st.Cout % 4 or st.C0 % 8:
            return False
        tiled = st.Win in (16, 32, 64, 128) and st.Hin % max(1, 128 // st.Win) == 0
        return tiled or (not st.stats and (st.N * st.Hin * st.Win) % 256 == 0)

    def conv_work(st):
        pad = st.ksize // 2
        hv, wv = (2 * st.Hin, 2 * st.Win) if st.upsample else (st.Hin, st.Win)
        ho = (hv + 2 * pad - st.ksize) // st.stride + 1
        wo = (wv + 2 * pad - st.ksize) // st.stride + 1
        fl = 2 * st.N * ho * wo * st.Cout * (st.ksize * st.ksize * st.C0 + st.C1)
        asz = 2 if st.a_dtype == N_.BF16 else 4
        by = st.N * st.Hin * st.Win * st.C0 * asz + st.N * ho * wo * st.C1 * asz + st.ksize * st.ksize * st.C0 * st.Cout * asz
        by += st.N * ho * wo * st.Cout * ((4 if st.y_f32 else 0) + (osz if st.y_op else 0) + (4 if st.resid else 0))
        return fl, by

    classes = {}

    def add(cls, bound, fn, ref, fl, by):
        c = classes.setdefault(cls, {"bound": bound, "calls": [], "flops": 0, "bytes": 0})
        c["calls"].append((fn, ref))
        c["flops"] += fl
        c["bytes"] += by

    for (name, fn, ref), st in zip(P.calls, P._structs):
        if name == "fdm_conv":
            fl, by = conv_work(st)
            if st.engine != N_.CONV_TC:
                add("conv_simt (CUDA-core implicit GEMM)", "fp32", fn, ref, fl, by)
            elif is_halo(st) or is_halo_pointwise(st):
                add("conv_halo (3x3 s1 and wide 1x1, tcgen05; CTA pairs on deep layers)", "tensor", fn, ref, fl, by)
            elif st.Hin == 1 and st.Win == 1:
                add("rpe_out_linear (21 RPENet GEMMs, tcgen05, side stream)", "tensor", fn, ref, fl, by)
            elif st.out_nchw and st.ksize == 3 and st.Cout <= 4 and st.C0 % 64 == 0:
                add("conv_head (3x3 -> eps, filter taps in the GEMM's N, tcgen05)", "hbm", fn, ref, fl, by)
            elif st.ksize == 1:
                add("conv_tc 1x1 (proj_out + residual, per-tap kernel, tcgen05)", "tensor", fn, ref, fl, by)
            elif st.stride == 2:
                add("conv_tc stride-2 (Downsample, per-tap kernel, tcgen05)", "tensor", fn, ref, fl, by)
            else:
                add("conv_tc 3x3 on 8x8 / 4x4 maps (per-tap kernel, tcgen05)", "tensor", fn, ref, fl, by)
        elif name == "fdm_gn_apply":
            el = st.N * st.HW * (st.Ca + st.Cb)
            add("gn_apply (GroupNorm+FiLM+SiLU)", "hbm", fn, ref, 0,
                el * ((2 if st.xa_bf16 else 4) + (osz if st.out_op else 0) + (4 if st.out_f32 else 0) + (osz if st.raw_op else 0)))
        elif name == "fdm_temporal_gn":
            el = st.B * st.T * st.HW * st.C
            add("temporal_gn", "hbm", fn, ref, 0, el * (4 + 4 + osz))
        elif name == "fdm_norm_linear":
            # GroupNorm in the operand path of the qkv linear: fp32 activations read once, bf16 qkv written once (+ weights);
            # bound by the output (an SM drains ~15 B/clk of stores: lin_tc.cu)
            rows = st.B * st.T * st.HW
            add("norm_qkv (GroupNorm in the operand path of the qkv linear, persistent tcgen05)", "hbm", fn, ref,
                2 * rows * st.K * st.Cout, rows * (st.K * 4 + st.Cout * osz) + st.K * st.Cout * 2)
        elif name == "fdm_attn_temporal":
            tok = st.B * st.T * st.HW
            # tcgen05 engine (workspace given): 3 launches per call; bytes = qkv read + out written + bf16 tables + the bf16 score-term
            # tables written and read back + the bf16 attention weights written and read back
            tc = bool(st.workspace)
            extra = 0
            if tc:
                t16 = (st.T + 7) // 8 * 8
                t16 += 8 if (t16 // 8) % 2 == 0 else 0
                t8 = (st.T + 3) // 4 * 4
                t8 += 4 if (t8 // 4) % 2 == 0 else 0
                ts = min(t16, t8)
                rows = st.B * st.heads * st.HW * st.T
                extra = 2 * (2 * rows * ts * 2) + 2 * rows * 64 * 2
            add("attn_temporal (RPE; 3 tcgen05 kernels per call)" if tc else "attn_temporal (RPE, CUDA cores)", "tensor", fn, ref,
                10 * st.T * st.T * st.C * st.B * st.HW,
                tok * st.C * (3 * osz + osz) + 3 * st.B * st.T * st.T * st.C * (2 if tc else 4) + extra)
        elif name == "fdm_attn_spatial":
            add("attn_spatial (tcgen05)", "tensor", fn, ref, 4 * st.L * st.L * st.C * st.N, st.N * st.L * st.C * 4 * osz)
        elif name == "fdm_rpe_tables":
            # every RPENet table in one launch: count x [B*T*T x C] . [C x C] GEMMs; bytes = weights + bf16 tables written
            cs = getattr(P, "rpe_table_channels", [])
            m_rows = st.B * st.T * st.T
            add("rpe_tables (all RPENet tables, one tcgen05 launch, side stream)", "tensor", fn, ref,
                sum(2 * m_rows * c * c for c in cs), sum(c * c * 2 + m_rows * c * 2 for c in cs))
        elif name in ("fdm_cast", "fdm_input_prep"):
            add("cast / input_prep", "hbm", fn, ref, 0, 0)
        else:
            add("conditioning (time MLP, FiLM, RPE hidden)", "latency", fn, ref, 0, 0)
    return classes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override the workload's videos per GPU (cfg5 batch sweep)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write rank 0's sample and eps of the last timed step to DIR/<name>.npy (float32), so that two builds "
                         "run with the same arguments can be compared output for output")
    args = ap.parse_args()
    wl = dict(WORKLOADS[args.workload])
    if args.batch > 0:
        wl["B"] = args.batch
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.no_gpu_eager:
        os.environ["FDM_BENCH_GPU_EAGER"] = "0"

    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what the native timed path computed; --impl reference has no such output")
        run_reference(args, wl, rank, world)
        return

    if args.warmup < 3:
        args.warmup = 3
    import torch.distributed as dist
    if not th.cuda.is_available():
        raise SystemExit("bench.py --impl native needs a CUDA device (no CPU fallback)")
    th.cuda.set_device(local)
    dev = th.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from improved_diffusion import _native as N_
    over, B, K = wl["over"], wl["B"], wl["K"]
    model, diffusion, sd = build_native(over, dev)
    model.precision = args.precision
    batch = synthetic_batch(over, B, K, wl["n_obs"], wl["video_len"], seed=rank)  # each rank its own shard of videos
    shape = tuple(batch["x0"].shape)
    C, S = over["in_channels"], over["image_size"]

    # ------------------------------------------------------------------ device-resident step (value)
    eng = model.engine()
    P = eng.plan_for(B, K, S, S, dev)
    kw_dev = {k: v.to(dev) for k, v in batch.items()}
    eng.load_conditioning(P, kw_dev["x0"], kw_dev["frame_indices"], kw_dev["obs_mask"], kw_dev["latent_mask"])
    tb = diffusion._tables(dev)
    P.set_t_source(tb["model_t"])
    nbuf = th.empty(shape, device=dev)
    step_args = N_.DdpmStepArgs(x=P.ptr(P.x), eps=P.ptr(P.eps), noise=nbuf.data_ptr(), coef=tb["step"].data_ptr(),
                                t=P.ptr(P.t_index), sample=P.ptr(P.x), pred_xstart=None, per_video=K * C * S * S, B=B, clip=1,
                                philox=None)
    stream = th.cuda.current_stream(dev)

    def body():
        s = th.cuda.current_stream(dev).cuda_stream
        P.run(s)
        N_.call("fdm_ddpm_step", step_args, s)

    # ------------------------------------------------------------------ parity of THIS batch (outside every timed region)
    # eps of the benchmarked plan on the benchmarked batch against the CPU oracle (the restatement pinned by the goldens), and —
    # when oracle/_ref travelled — against the unmodified reference run in fp32 on this GPU
    parity = None
    if rank == 0:
        from oracle import fdm_oracle as O
        t_chk = n_chk = None
        g = th.Generator().manual_seed(77)
        x_chk = th.randn(shape, generator=g)
        t_idx = diffusion.num_timesteps // 2
        P.x_view.copy_(x_chk)
        P.t_index_view.fill_(t_idx)
        P.run(stream.cuda_stream)
        stream.synchronize()
        eps_native = P.eps_view.detach().cpu().clone()
        model_t = tb["model_t"][t_idx].item()
        ts = th.full((B,), float(model_t))
        tol = 2e-2 if args.precision == "bf16" else 1e-4
        parity = {"tolerance": tol, "what": f"eps rel-L2 of the benchmarked plan on the benchmarked batch (x_t ~ N(0,1) seed 77, step "
                                            f"index {t_idx}), computed once outside the timed regions"}
        if B * K * S * S * over["num_channels"] <= 8 * 20 * 32 * 32 * 64 * 4:  # bounded CPU work (seconds)
            with th.no_grad():
                sd_cpu = {k: v.detach().cpu() for k, v in model.state_dict().items()}
                ref = O.unet_forward(sd_cpu, O.make_cfg(**over), x_chk, batch["x0"], ts, batch["frame_indices"], batch["obs_mask"],
                                     batch["latent_mask"])
            parity["eps_rel_l2_vs_cpu_oracle"] = O.rel_l2(eps_native, ref)
        try:
            from oracle import ref_loader as R
            if R.find_ref() is not None:
                old = (th.backends.cudnn.allow_tf32, th.backends.cuda.matmul.allow_tf32)
                th.backends.cudnn.allow_tf32 = th.backends.cuda.matmul.allow_tf32 = False
                rm, _ = build_reference(over, {k: v.detach().cpu() for k, v in model.state_dict().items()}, dev)
                with th.no_grad():
                    ref_gpu, _ = rm(x_chk.to(dev), timesteps=ts.to(dev), **kw_dev)
                parity["eps_rel_l2_vs_reference_on_gpu_fp32"] = O.rel_l2(eps_native, ref_gpu.cpu())
                del rm, ref_gpu
                th.backends.cudnn.allow_tf32, th.backends.cuda.matmul.allow_tf32 = old
                th.cuda.empty_cache()
        except Exception as ex:
            parity["reference_on_gpu_error"] = repr(ex)[:200]
        errs = [v for k, v in parity.items() if k.startswith("eps_rel_l2")]
        parity["ok"] = bool(errs) and all(e <= tol for e in errs)

    th.manual_seed(1000 + rank)  # the sampler state and step noise below: the same inputs on every run with the same arguments
    P.x_view.normal_()
    P.t_index_view.fill_(diffusion.num_timesteps - 1)
    nbuf.normal_()
    body()
    stream.synchronize()
    graph = th.cuda.CUDAGraph()
    with th.cuda.graph(graph):
        body()
    flush = th.empty(192 * 1024 * 1024, dtype=th.uint8, device=dev)  # > 126 MB L2

    def one_step(i):
        P.t_index_view.fill_(i)
        nbuf.normal_()
        graph.replay()

    n_t = diffusion.num_timesteps
    P.x_view.normal_()
    for w in range(args.warmup):
        one_step(n_t - 1 - (w % n_t))
    th.cuda.synchronize()
    clocks = ClockSampler(local)
    clocks.start()  # polling starts >= 0.5 s before the timed region
    if world > 1:
        dist.barrier()
    th.cuda.synchronize()
    evs = [(th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    clocks.mark_begin()
    for k in range(args.steps):
        flush.zero_()  # L2 flush between timed iterations (outside the event pair)
        evs[k][0].record()
        one_step(n_t - 1 - ((args.warmup + k) % n_t))
        evs[k][1].record()
    th.cuda.synchronize()
    clocks.mark_end()
    if args.dump_outputs and rank == 0:
        # what p_sample returns for the last timed step, read before the informational passes below reuse the plan's buffers
        dump_outputs(args.dump_outputs, {"sample": P.x_view, "eps": P.eps_view})
    if world > 1:
        dist.barrier()
    th.cuda.synchronize()
    step_ms = [a.elapsed_time(b) for a, b in evs]
    total_ms = th.tensor([sum(step_ms)], device=dev, dtype=th.float64)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    ms_per_step = total_ms / args.steps
    value = world * B * K * args.steps / (total_ms * 1e-3)
    assert bool(th.isfinite(P.x_view).all()), "non-finite sampler state"

    # hot (no L2 flush, back-to-back) for information; long enough (>= 0.3 s) that the clock sampler sees sustained load
    th.cuda.synchronize()
    hot_steps = max(args.steps, int(300.0 / max(ms_per_step, 1e-3)))
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    hot_clocks_t0 = time.perf_counter()
    e0.record()
    for k in range(hot_steps):
        one_step(n_t - 1 - (k % n_t))
    e1.record()
    th.cuda.synchronize()
    hot_clocks_t1 = time.perf_counter()
    hot_ms = e0.elapsed_time(e1) / hot_steps
    clk = clocks.stop()
    if clocks.nv is not None:
        hot = [x for x in clocks.samples if hot_clocks_t0 <= x[0] <= hot_clocks_t1]
        if hot:
            clk["sustained"] = {"sm_mhz": statistics.median(x[1] for x in hot), "samples": len(hot),
                                "what": f"{hot_steps} back-to-back steps right after the timed region"}

    # ------------------------------------------------------------------ roofline: per kernel class, each timed alone
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf, peak_src = (peaks["bf16_tflops"], "measured") if "bf16_tflops" in peaks else (1590.0, "fallback")
    peak_bw, bw_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6500.0, "fallback")
    import ctypes as C_
    sp = C_.c_void_p(stream.cuda_stream)

    def time_calls(calls, reps=20):
        for fn, ref in calls:
            fn(ref, sp)
        th.cuda.synchronize()
        c0, c1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(reps):
            for fn, ref in calls:
                fn(ref, sp)
        c1.record()
        th.cuda.synchronize()
        return c0.elapsed_time(c1) / reps

    # kernels per step: every entry point is one launch, except the tcgen05 temporal attention (3) ; + the statistics memset,
    # the fused posterior update and the two ATen launches of the step (step-index fill, noise draw)
    kernel_launches = sum(3 if (nm == "fdm_attn_temporal" and st_.workspace) else 1 for (nm, _, _), st_ in zip(P.calls, P._structs)) + 4
    classes = kernel_classes(P, N_, B, K, C, S, 2 if args.precision == "bf16" else 4)
    table, conv_ms, conv_fl, n_convs = [], 0.0, 0, 0
    for cls, c in classes.items():
        ms = time_calls(c["calls"])
        row = {"class": cls, "bound": c["bound"], "launches": len(c["calls"]), "us_per_step": 1e3 * ms,
               "share_of_step": ms / hot_ms}
        if c["flops"]:
            tf = c["flops"] / (ms * 1e-3) / 1e12
            row.update(flops=c["flops"], tflops=tf, frac_of_bf16_peak=tf / peak_tf)
        if c["bytes"]:
            gbs = c["bytes"] / (ms * 1e-3) / 1e9
            row.update(bytes=c["bytes"], gbs=gbs, frac_of_hbm_peak=gbs / peak_bw)
        row["frac"] = row.get("frac_of_bf16_peak") if c["bound"] == "tensor" else row.get("frac_of_hbm_peak")
        table.append(row)
        if cls.startswith(("conv_", "rpe_out")):
            conv_ms, conv_fl, n_convs = conv_ms + ms, conv_fl + c["flops"], n_convs + len(c["calls"])
    # K6, the fused posterior update: 16 B per element (x, eps, noise read; x written), HBM-bound
    k6_calls = [(getattr(N_.lib(), "fdm_ddpm_step"), C_.byref(step_args))]
    k6_ms = time_calls(k6_calls, reps=50)
    # cold variant: inputs evicted from L2 first (the number the HBM roofline is about)
    cold = []
    for _ in range(5):
        flush.zero_()
        c0, c1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        c0.record()
        k6_calls[0][0](k6_calls[0][1], sp)
        c1.record()
        th.cuda.synchronize()
        cold.append(c0.elapsed_time(c1))
    k6_bytes = 16 * B * K * C * S * S
    k6_cold = statistics.median(cold)
    table.append({"class": "ddpm_step (K6 fused posterior update)", "bound": "hbm", "launches": 1, "us_per_step": 1e3 * k6_ms,
                  "share_of_step": k6_ms / hot_ms, "bytes": k6_bytes, "gbs": k6_bytes / (k6_ms * 1e-3) / 1e9,
                  "frac_of_hbm_peak": k6_bytes / (k6_ms * 1e-3) / 1e9 / peak_bw, "frac": k6_bytes / (k6_ms * 1e-3) / 1e9 / peak_bw,
                  "cold_l2": {"us": 1e3 * k6_cold, "gbs": k6_bytes / (k6_cold * 1e-3) / 1e9,
                              "frac_of_hbm_peak": k6_bytes / (k6_cold * 1e-3) / 1e9 / peak_bw},
                  "note": f"{k6_bytes / 1e6:.1f} MB per launch: launch latency, not bandwidth, at this size; warm = operands in L2"})
    table.sort(key=lambda r: -r["us_per_step"])
    # `roofline` = the class that takes the most time in the step
    top = next(r for r in table if r.get("frac") is not None)
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_top_kernel_traffic.json")))
        if tj.get("workload") == args.workload and tj.get("class") == top["class"]:
            traffic = tj["dram_bytes_per_launch"]
    except Exception:
        pass
    tensor_bound = top["bound"] == "tensor"
    roofline = {"bound": "tensor" if tensor_bound else "hbm", "kernel": top["class"],
                "achieved": top["tflops"] if tensor_bound else top["gbs"], "peak": peak_tf if tensor_bound else peak_bw,
                "peak_source": peak_src if tensor_bound else bw_src, "unit": "TFLOP/s" if tensor_bound else "GB/s",
                "frac": top["frac"], "traffic": traffic, "launches_per_step": top["launches"],
                "us_per_launch": top["us_per_step"] / top["launches"], "share_of_step": top["share_of_step"],
                "what": "the kernel class with the largest share of the step's time, timed alone (its launches of one step back to "
                        "back, CUDA events on the launching stream); every class is in roofline_table"}
    conv_tf = conv_fl / (conv_ms * 1e-3) / 1e12 if conv_ms else 0.0
    all_convs = {"achieved": conv_tf, "unit": "TFLOP/s", "frac": conv_tf / peak_tf, "launches_per_step": n_convs,
                 "ms_per_step": conv_ms, "share_of_step": conv_ms / hot_ms, "flops_per_step": conv_fl}
    step_tf = P.flops / (ms_per_step * 1e-3) / 1e12
    step_roofline = {"bound": "tensor", "achieved": step_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": step_tf / peak_tf,
                     "frac_of_sustained_peak": step_tf / peaks.get("bf16_tflops_sustained", peak_tf),
                     "flops_per_frame_step": P.flops / (B * K)}

    # ------------------------------------------------------------------ e2e through the public API (host buffers)
    e2e = None
    if not args.no_e2e:
        host = {k: v.pin_memory() for k, v in batch.items()}
        out_host = th.empty(shape, dtype=th.float32).pin_memory()

        def stage():
            kw = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
            final, _ = diffusion.p_sample_loop(model, shape, clip_denoised=True, model_kwargs=kw, latent_mask=kw["latent_mask"])
            out_host.copy_(final, non_blocking=True)
            th.cuda.synchronize()

        stage()  # warm-up (captures the sampler graph)
        th.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        stage()
        if world > 1:
            dist.barrier()
        dt = th.tensor([time.perf_counter() - t0], device=dev, dtype=th.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dt = float(dt.item())
        h2d = sum(v.numel() * v.element_size() for v in host.values())
        d2h = out_host.numel() * 4
        e2e = {"value": world * B * K * n_t / dt, "unit": "frame-steps/s", "h2d_bytes_per_step": h2d / n_t,
               "d2h_bytes_per_step": d2h / n_t, "what": f"diffusion.p_sample_loop, one stage of {n_t} steps, pinned host "
               f"inputs -> device -> pinned host result, wall clock incl. copies", "seconds": dt}

    # ------------------------------------------------------------------ the reference on this box: CPU (all cores) and GPU eager
    cpu = eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference(over, B, K, batch, model.state_dict(), n_steps=int(os.environ.get("FDM_BENCH_CPU_STEPS", "20")), warmup=2)
    if rank == 0 and world == 1 and not args.no_gpu_eager:
        try:
            eager = gpu_eager_sampling(over, batch, model.state_dict(), dev, B, K)
        except Exception as ex:
            eager = {"error": repr(ex)[:300]}

    # ------------------------------------------------------------------ secondary metric: train samples/s (BASELINE cfg2, cfg3)
    train = None
    if not args.no_train:
        del graph
        model._engines.clear()
        th.cuda.empty_cache()
        train = bench_train(dev, world, args.precision, "cfg2-train")
        train["cfg3"] = bench_train(dev, world, args.precision, "cfg3-train")

    if rank == 0:
        line = {"metric": "denoiser frame-steps/sec (sampling)", "value": value, "unit": "frame-steps/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "ms_per_step_hot": hot_ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
                "config": config_dict(args.workload, wl, world),
                "clocks": clk, "e2e": e2e, "gpu_launches": args.steps * kernel_launches,
                "launches_per_step": kernel_launches, "parity": parity, "roofline": roofline, "roofline_table": table,
                "roofline_all_convs": all_convs, "step_roofline": step_roofline,
                "cpu_baseline": cpu, "gpu_eager": eager, "train": train}
        if train is not None:  # promoted copies of the training numbers (BASELINE.json metric part 2: train samples/sec)
            line["train_samples_per_s_cfg2"] = train["value"]
            line["train_ms_per_step_cfg2"] = train["ms_per_step"]
            line["train_samples_per_s_cfg3"] = train["cfg3"]["value"]
            line["train_ms_per_step_cfg3"] = train["cfg3"]["ms_per_step"]
            line["train_frac_of_peak_cfg3"] = train["cfg3"]["roofline"]["frac"]
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
