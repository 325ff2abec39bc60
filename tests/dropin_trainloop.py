"""Helper run as a SUBPROCESS by tests/test_host_cpu.py (needs a reference checkout, named by FDM_REFERENCE_PATH): the reference's own TrainLoop
(improved_diffusion/train_util.py, unmodified) driving THIS repo's model + diffusion for two optimizer steps on CPU.
mpi4py / blobfile / wandb are absent or unwanted here and are stubbed; everything else is the reference's code."""
import os
import sys
import types

import numpy as np
import torch as th
import torch.distributed as dist

# ---- stubs for the process/logging plumbing (SURVEY §2: out of scope)
comm = types.SimpleNamespace(rank=0, size=1, Get_rank=lambda: 0, Get_size=lambda: 1, bcast=lambda x, root=0: x,
                             gather=lambda x, root=0: [x])
sys.modules["mpi4py"] = types.SimpleNamespace(MPI=types.SimpleNamespace(COMM_WORLD=comm))
sys.modules["mpi4py.MPI"] = sys.modules["mpi4py"].MPI
sys.modules["blobfile"] = types.SimpleNamespace(BlobFile=open, join=os.path.join, dirname=os.path.dirname, exists=os.path.exists)
logged = []
sys.modules["wandb"] = types.SimpleNamespace(log=lambda d, **k: logged.append(dict(d)), Video=lambda *a, **k: None,
                                             run=types.SimpleNamespace(id="test"), init=lambda **k: None)

import improved_diffusion  # noqa: E402  (this repo's package; FDM_REFERENCE_PATH appends the reference's modules)
from improved_diffusion import train_util, unet  # noqa: E402
from improved_diffusion.script_util import create_model_and_diffusion, model_and_diffusion_defaults  # noqa: E402

assert train_util.__file__.startswith(os.environ["FDM_REFERENCE_PATH"]), train_util.__file__
assert "_b200" in unet.__file__

os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=sys.argv[1], DIFFUSION_TRAINING_TEST="1")
dist.init_process_group("gloo", rank=0, world_size=1)
th.manual_seed(0)
d = model_and_diffusion_defaults()
d.update(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32,
         diffusion_space_kwargs=dict(diffusion_space="pixel", pre_encoded=False, pre_encoded_stats_dict=None))
model, diffusion = create_model_and_diffusion(**d)
model.precision = "fp32"


def data():
    g = th.Generator().manual_seed(1)
    while True:
        yield th.randn(2, 12, 4, 32, 32, generator=g).clamp(-1, 1), {}


real_save = train_util.TrainLoop.save
train_util.TrainLoop.save = lambda self: None  # no checkpoint files during the training run (checked separately below)
args = types.SimpleNamespace(resume_id="", T=12)
before = [p.detach().clone() for p in model.parameters()]
loop = train_util.TrainLoop(model=model, diffusion=diffusion, data=data(), batch_size=2, microbatch=-1, lr=1e-3, ema_rate="0.9999",
                            log_interval=1, save_interval=10 ** 9, resume_checkpoint="", use_fp16=False,
                            diffusion_space_kwargs=d["diffusion_space_kwargs"], fp16_scale_growth=1e-3, schedule_sampler=None,
                            weight_decay=0.0, lr_anneal_steps=0, sample_interval=None, pad_with_random_frames=True, max_frames=5,
                            enc_dec_chunk_size=10, args=args)
th.manual_seed(5)
np.random.seed(5)
loop.run_loop()
changed = sum(int(not th.equal(a, p.detach())) for a, p in zip(before, model.parameters()))
keys = set().union(*[set(x) for x in logged])
# a freshly built model is mostly zero-initialised (zero_module): only part of the tensors get a non-zero gradient in 2 steps
assert loop.step >= 1 and changed > 50, (loop.step, changed)
assert {"loss", "mse", "grad_norm", "step"} <= keys, keys
assert all(th.isfinite(p).all() for p in model.parameters())

# ---- the same two steps through this repo's train_step.NativeTrainStep (host side of the step restated: mask sampling, gather,
# timestep draw, loss weighting, gradient norm, AdamW, EMA, logging) from the same seeds: identical parameters, EMA and logs
from improved_diffusion.train_step import NativeTrainStep  # noqa: E402

th.manual_seed(0)
model2, diffusion2 = create_model_and_diffusion(**d)
model2.precision = "fp32"
assert all(th.equal(a, p.detach()) for a, p in zip(before, model2.parameters()))
stream = data()
next(stream)  # the reference's constructor takes one batch for visualisation (train_util.py:86-88)
runner = NativeTrainStep(model2, diffusion2, lr=1e-3, max_frames=5, weight_decay=0.0, ema_rate="0.9999", microbatch=-1,
                         pad_with_random_frames=True, optimizer="torch")
th.manual_seed(5)
np.random.seed(5)
mine = [runner.run_step(next(stream)[0], next(stream)[0]) for _ in range(loop.step + 1)]
worst = max(float((a.detach() - b.detach()).abs().max()) for a, b in zip(model.parameters(), model2.parameters()))
worst_ema = max(float((a - b).abs().max()) for a, b in zip(loop.ema_params[0], runner.ema_params[0]))
assert worst <= 1e-6 and worst_ema <= 1e-7, (worst, worst_ema)
ref_logs = [x for x in logged if "loss" in x]
assert len(ref_logs) == len(mine), (len(ref_logs), len(mine))
for r, m in zip(ref_logs, mine):
    for k, v in r.items():
        if k in m and k not in ("step", "samples"):
            assert abs(float(v) - m[k]) <= 1e-5 * max(1.0, abs(m[k])), (k, v, m[k])
    assert {k for k in r if k.startswith(("loss", "mse", "eval-mse", "grad_norm"))} <= set(m), (sorted(r), sorted(m))
    assert int(r["step"]) == m["step"] and int(r["samples"]) == m["samples"]
print("TRAINSTEP_OK worst param diff", worst, "ema", worst_ema, "keys", sorted(mine[0])[:8])

# ---- checkpoint files: NativeTrainStep.save() -> the reference's TrainLoop resumes from them (its own _load_and_sync_parameters,
# _load_optimizer_state, _load_ema_parameters), and the reference's TrainLoop.save() -> NativeTrainStep.resume()
import tempfile  # noqa: E402

work = tempfile.mkdtemp()
os.chdir(work)
os.makedirs("checkpoints")
saved = runner.save(os.path.join("checkpoints", "mine"), config={"T": 12, "max_frames": 5})
assert os.path.basename(saved) == "model000001.pt" and sorted(os.listdir("checkpoints/mine")) == [
    "ema_0.9999_000001.pt", "model000001.pt", "opt000001.pt"]
th.manual_seed(0)
model3, diffusion3 = create_model_and_diffusion(**d)
loop3 = train_util.TrainLoop(model=model3, diffusion=diffusion3, data=data(), batch_size=2, microbatch=-1, lr=1e-3, ema_rate="0.9999",
                             log_interval=1, save_interval=10 ** 9, resume_checkpoint="", use_fp16=False,
                             diffusion_space_kwargs=d["diffusion_space_kwargs"], fp16_scale_growth=1e-3, schedule_sampler=None,
                             weight_decay=0.0, lr_anneal_steps=0, sample_interval=None, pad_with_random_frames=True, max_frames=5,
                             enc_dec_chunk_size=10, args=types.SimpleNamespace(resume_id="mine", T=12))
assert loop3.step == 1
assert all(th.equal(a.detach(), b.detach()) for a, b in zip(model3.parameters(), model2.parameters()))
assert all(th.equal(a.detach(), b) for a, b in zip(loop3.ema_params[0], runner.ema_params[0]))
for pa, pb in zip(loop3.opt.param_groups[0]["params"], runner.opt.param_groups[0]["params"]):
    sa, sb = loop3.opt.state[pa], runner.opt.state[pb]
    assert th.equal(sa["exp_avg"], sb["exp_avg"]) and th.equal(sa["exp_avg_sq"], sb["exp_avg_sq"]) and float(sa["step"]) == float(sb["step"])
train_util.TrainLoop.save = real_save  # the real one from here on (it was stubbed out for the training run above)
loop.args = types.SimpleNamespace(resume_id="theirs", T=12)
loop.step = 1
loop.save()
th.manual_seed(0)
model4, diffusion4 = create_model_and_diffusion(**d)
runner4 = NativeTrainStep(model4, diffusion4, lr=1e-3, max_frames=5, ema_rate="0.9999", optimizer="torch")
assert runner4.resume(os.path.join("checkpoints", "nothing-here")) is None
assert runner4.resume(os.path.join("checkpoints", "theirs")) == 1 and runner4.step == 1
assert all(th.equal(a.detach(), b.detach()) for a, b in zip(model4.parameters(), model.parameters()))
assert all(th.equal(a, b.detach()) for a, b in zip(runner4.ema_params[0], loop.ema_params[0]))
for pa, pb in zip(runner4.opt.param_groups[0]["params"], loop.opt.param_groups[0]["params"]):
    assert th.equal(runner4.opt.state[pa]["exp_avg_sq"], loop.opt.state[pb]["exp_avg_sq"])
print("CHECKPOINT_OK both directions")
print("DROPIN_OK steps", loop.step + 1, "params changed", changed, "logged", sorted(keys)[:6])
dist.destroy_process_group()
