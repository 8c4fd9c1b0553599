#!/usr/bin/env python
"""What do parameter groups cost the fused Adam step?

1. The kernel alone at 64 M live floats (1.8 GB of traffic per step at 28 B per parameter, beyond the 126 MB L2):
   - `one group`: FusedAdam's default, one group over one run;
   - `alternating`: AdamW over 4096-float parameters that alternate between two groups, the most runs per byte;
   - `decay/no-decay`: AdamW over 1024x1024 weights (decay) and their 1024-float biases (no decay).
   Each is the tick + `b200np_adam_step_groups` pair FusedAdam.step launches, timed with CUDA events over `--launches`
   back-to-back launches, the variants alternating for `--rounds` rounds.  GB/s counts 28 B per updated parameter.
2. The graphed ANPDistractor step at bench.py's headline size (tf32x3): FusedAdam's default against two-group AdamW
   (decay on weights, none on biases), timed alternately in one process.
Prints one JSON line with the card's name and power limit.
usage: tools/bench_adam_groups.py [--launches 100] [--rounds 3] [--steps 50]"""
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
ap.add_argument("--launches", type=int, default=100)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--steps", type=int, default=50)
args = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("needs a CUDA device")
N = 64 << 20


def module(sizes):
    m = torch.nn.Module()
    m.ps = torch.nn.ParameterList([torch.nn.Parameter(torch.empty(k, device="cuda").uniform_(-1, 1)) for k in sizes])
    return m


def adamw_two_groups(flat, decay):
    """AdamW with decay on the parameters `decay(name, p)` selects and none on the rest."""
    named = list(zip(flat.names, flat.params))
    return FusedAdam(flat, lr=1e-4, weight_decay=0.01, decoupled_weight_decay=True,
                     param_groups=[{"params": [p for n, p in named if decay(n, p)]},
                                   {"params": [p for n, p in named if not decay(n, p)], "weight_decay": 0.0}])


def kernel_variants():
    one = FusedAdam(FlatParams(module([4096] * (N // 4096))), lr=1e-4)
    alt_flat = FlatParams(module([4096] * (N // 4096)))
    alt = adamw_two_groups(alt_flat, lambda n, p: int(n.split(".")[-1]) % 2 == 0)
    pairs = N // (1024 * 1024 + 1024)
    split_flat = FlatParams(module([1024 * 1024, 1024] * pairs))
    split = adamw_two_groups(split_flat, lambda n, p: int(n.split(".")[-1]) % 2 == 0)
    out = {}
    for name, opt in (("one group", one), ("alternating", alt), ("decay/no-decay", split)):
        f = opt.flat
        f.grad.normal_()
        out[name] = (opt, f.n_live, int(opt._run_group.numel()))
    return out


def launch(opt):
    f = opt.flat
    ops.adam_step_groups(f.flat, f.grad, opt.m, opt.v, f.n_live, opt._table, opt._run_begin, opt._run_group,
                         opt.t_dev)


def time_kernel(opt, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        launch(opt)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


variants = kernel_variants()
for opt, _, _ in variants.values():
    for _ in range(5):
        launch(opt)
torch.cuda.synchronize()
kernel_us = {k: [] for k in variants}
for _ in range(args.rounds):
    for k, (opt, _, _) in variants.items():
        kernel_us[k].append(round(1e3 * time_kernel(opt, args.launches), 2))
kernel = {k: {"live_floats": n, "runs": runs, "us": kernel_us[k],
              "GB_per_s_best": round(28 * n / (min(kernel_us[k]) * 1e-6) / 1e9, 1)}
          for k, (_, n, runs) in variants.items()}
best_one = kernel["one group"]["GB_per_s_best"]
for k in kernel:
    kernel[k]["rate_vs_one_group"] = round(kernel[k]["GB_per_s_best"] / best_one, 4)
del variants
torch.cuda.empty_cache()

engine.set_precision("tf32x3")
T = TASKS_PER_GPU
lossf = LossFunc("mse", "distractor")
batches = [[torch.from_numpy(a).cuda() for a in synth.task_batch("distractor", T, NC, NT, seed=100 + i)]
           for i in range(4)]


def arm(grouped):
    model = ANPDistractor(make_cfg(T, "cuda:0")).to("cuda:0")
    flat = FlatParams(model)
    opt = adamw_two_groups(flat, lambda n, p: p.dim() > 1) if grouped else FusedAdam(flat, lr=1e-4)
    g = GraphedStep(model, lossf, opt, batches[0], warmup=3)
    return lambda i: g(batches[i % len(batches)])


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


arms = {"default": arm(False), "adamw decay/no-decay": arm(True)}
step_ms = {k: [] for k in arms}
for _ in range(args.rounds):
    for k, run in arms.items():
        step_ms[k].append(round(timed(run, args.steps), 4))

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                   capture_output=True, text=True).stdout.strip()
print(json.dumps({"adam_kernel_64M": kernel, "launches_per_timing": args.launches,
                  "step_workload": f"ANPDistractor graphed step, tf32x3, {T} tasks, nc={NC} nt={NT}",
                  "step_ms": step_ms, "gpu": q or torch.cuda.get_device_name(0)}))
