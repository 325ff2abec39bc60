"""Training-step time with ResBlock dropout on one GPU: python tools/dropout_train_bench.py [--rounds R] [--precision P] [workloads]

For each workload (bench.TRAIN_WORKLOADS, default cfg2-train and cfg3-train) two models with the same weights, one built with
dropout = 0 and one with dropout = 0.1, take the step bench.bench_train times (training_losses forward + backward + FlatAdamW) in
interleaved rounds (p = 0, p = 0.1, p = 0, ...), so both see the same machine state; the spread of the p = 0 rounds is the
run-to-run noise the dropout overhead is read against.  bench.bench_train's own p = 0 number is measured beside it in the same
process.  Prints one JSON line per workload, with the GPU's name and power limit."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch as th  # noqa: E402

import bench  # noqa: E402


def gpu_info(dev):
    q = subprocess.run(["nvidia-smi", "-i", str(dev.index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return {"name": th.cuda.get_device_name(dev), "nvidia_smi": q}


def trainer(over, B, K, p, dev, precision):
    from improved_diffusion.optim import FlatAdamW
    model, diffusion, _ = bench.build_native(over, dev)  # same seeded weights for every p
    model.dropout = p
    for m in model.modules():
        if isinstance(m, th.nn.Dropout):
            m.p = p
    model.precision = precision
    model.train()
    opt = FlatAdamW(model.parameters(), lr=1e-4, weight_decay=0.0, model=model)
    batch = {k: v.to(dev) for k, v in bench.synthetic_batch(over, B, K, 3, 4 * K, seed=1).items()}
    g = th.Generator(device=dev).manual_seed(0)

    def step():
        t = th.randint(0, diffusion.num_timesteps, (B,), device=dev, generator=g)
        terms = diffusion.training_losses(model, batch["x0"], t, model_kwargs=batch, latent_mask=1 - batch["obs_mask"],
                                          eval_mask=batch["latent_mask"])
        opt.zero_grad(set_to_none=True)
        terms["loss"].mean().backward()
        opt.step()
        return terms["loss"]
    return model, step


def timed(step, n, warmup):
    for _ in range(warmup):
        step()
    th.cuda.synchronize()
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        loss = step()
    e1.record()
    th.cuda.synchronize()
    assert bool(th.isfinite(loss).all()), "training loss is not finite"
    return e0.elapsed_time(e1) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=["cfg2-train", "cfg3-train"])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    args = ap.parse_args()
    dev = th.device("cuda:0")
    th.cuda.set_device(dev)
    os.environ["FDM_TRAIN_ENGINE"] = "native"
    os.environ.setdefault("FDM_BENCH_GPU_EAGER", "0")
    info = gpu_info(dev)
    for wl in args.workloads:
        over, B, K, steps = bench.TRAIN_WORKLOADS[wl]
        ps = (0.0, 0.1)
        runs = {p: trainer(over, B, K, p, dev, args.precision) for p in ps}
        ms = {p: [] for p in ps}
        for _ in range(args.rounds):
            for p in ps:
                ms[p].append(timed(runs[p][1], steps, warmup=3))
        plans = {p: next(iter(runs[p][0].engine().train_plans.values())) for p in ps}
        assert plans[0.0].drop_philox is None and plans[0.1].drop_p == 0.1
        del runs, plans
        th.cuda.empty_cache()
        ref = bench.bench_train(dev, 1, args.precision, wl)
        med = {p: statistics.median(v) for p, v in ms.items()}
        p0 = ms[0.0]
        print(json.dumps({
            "workload": wl, "precision": args.precision, "gpu": info, "steps_per_round": steps, "rounds": args.rounds,
            "ms_per_step": {str(p): [round(v, 4) for v in ms[p]] for p in ps},
            "median_ms_per_step": {str(p): round(med[p], 4) for p in ps},
            "p0_spread": round((max(p0) - min(p0)) / med[0.0], 4),
            "dropout_0.1_overhead": round(med[0.1] / med[0.0] - 1, 4),
            "bench_train_p0_ms_per_step": round(ref["ms_per_step"], 4),
            "what": "CUDA events around `steps` training steps (forward + backward + FlatAdamW), after 3 warm-up steps, per round; "
                    "rounds alternate p = 0 / p = 0.1; bench_train_p0 is bench.bench_train's p = 0 step in the same process"}))


if __name__ == "__main__":
    main()
