#!/usr/bin/env python
"""What do clipping, non-finite skipping and a per-step learning-rate schedule cost on the graphed training step?

ANPDistractor at bench.py's headline size, tf32x3, one CUDA graph per step.  Two optimizers over two identically built
models, timed alternately in one process: FusedAdam's defaults, and FusedAdam(max_grad_norm, skip_nonfinite) with a
LambdaLR stepped after every replay.  Then the norm pass on its own (b200np_grad_norm over the live gradient), from
CUDA events over many launches.  Prints one JSON line with the card's name and power limit.
usage: tools/bench_optim_control.py [--steps 50] [--rounds 3]"""
import argparse, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "what-matters-for-meta-learning_b200")]
import torch
from bench import NC, NT, TASKS_PER_GPU, make_cfg
from b200np import engine, ops
from b200np.optim import FlatParams, FusedAdam, GraphedStep
from networks.ANPDistractor import ANPDistractor
from oracle import synth
from trainer.losses import LossFunc

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=50)
ap.add_argument("--rounds", type=int, default=3)
args = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("needs a CUDA device")
engine.set_precision("tf32x3")
T = TASKS_PER_GPU
lossf = LossFunc("mse", "distractor")
batches = [[torch.from_numpy(a).cuda() for a in synth.task_batch("distractor", T, NC, NT, seed=100 + i)]
           for i in range(4)]


def arm(controlled):
    model = ANPDistractor(make_cfg(T, "cuda:0")).to("cuda:0")
    kw = dict(max_grad_norm=1.0, skip_nonfinite=True) if controlled else {}
    opt = FusedAdam(FlatParams(model), lr=1e-4, **kw)
    g = GraphedStep(model, lossf, opt, batches[0], warmup=3)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda k: 1.0 / (1 + 1e-3 * k)) if controlled else None

    def run(i):
        g(batches[i % len(batches)])
        if sched is not None:
            sched.step()
    return run, opt


def timed(run, steps):
    for i in range(5):
        run(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        run(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


arms = {"default": arm(False), "clip+skip+schedule": arm(True)}
ms = {k: [] for k in arms}
for _ in range(args.rounds):
    for k, (run, _) in arms.items():
        ms[k].append(round(timed(run, args.steps), 4))

opt = arms["clip+skip+schedule"][1]
f = opt.flat
n_launch = 200
for _ in range(10):
    ops.grad_norm(f.grad, f.n_live, opt.grad_norm, opt._norm_ws)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(n_launch):
    ops.grad_norm(f.grad, f.n_live, opt.grad_norm, opt._norm_ws)
e1.record()
torch.cuda.synchronize()
norm_us = 1e3 * e0.elapsed_time(e1) / n_launch

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                   capture_output=True, text=True).stdout.strip()
print(json.dumps({"workload": f"ANPDistractor graphed step, tf32x3, {T} tasks, nc={NC} nt={NT}",
                  "step_ms": ms, "grad_norm_us": round(norm_us, 2),
                  "grad_norm_note": f"{f.n_live} floats, back-to-back launches (the gradient stays in L2)",
                  "gpu": q or torch.cuda.get_device_name(0)}))
