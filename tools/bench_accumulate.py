#!/usr/bin/env python
"""What does gradient accumulation cost on the fused, graph-captured training step?

1. ANPDistractor at bench.py's headline size (20 tasks per micro-batch, nc=15, nt=21, tf32x3) under GraphedStep with
   `accumulate_steps` k = 1, 2 and 4: time per task over whole windows, CUDA events around `--windows` windows, the
   three configurations alternating for `--rounds` rounds in one process.
2. In the k = 4 run, CUDA events around every call: a micro-step ("first" / "middle" graph: forward, backward and
   the gather) against the window's step ("last" graph: the same plus exchange and Adam).
3. The gradient gather alone over ANPDistractor's live gradients as autograd hands them over (separate tensors):
   `multi_copy` against `multi_accumulate`, captured 20 to a CUDA graph as in the step graphs (so no host time), CUDA
   events over `--launches` calls, alternating.  Both are L2-resident here, as in a step, where the gradients have
   just been written; GB/s counts 8 B (copy) and 12 B (add) per float.
4. With two GPUs or more: two ranks under torch.distributed.run, 20 tasks per rank and micro-batch.  The gradient
   all-reduce calls per window of an eager run (k = 1 and k = 4), and time per task of the graphed step at k = 1 and 4.
Prints one JSON line with the card's name and power limit.
usage: tools/bench_accumulate.py [--rounds 3] [--windows 6] [--launches 200]"""
import argparse, contextlib, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "what-matters-for-meta-learning_b200")]
import torch
from bench import NC, NT, TASKS_PER_GPU, make_cfg
from b200np import dist, engine, ops
from b200np.optim import FlatParams, FusedAdam, GraphedStep
from networks.ANPDistractor import ANPDistractor
from oracle import synth
from trainer.losses import LossFunc

ap = argparse.ArgumentParser()
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--windows", type=int, default=6)
ap.add_argument("--launches", type=int, default=200)
ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)   # one rank of part 4
args = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("needs a CUDA device")
KS = (1, 2, 4)
T = TASKS_PER_GPU
if args.worker:
    dev = torch.device(f"cuda:{int(os.environ['LOCAL_RANK'])}")
    torch.cuda.set_device(dev)
    torch.distributed.init_process_group("nccl", device_id=dev)
else:
    dev = torch.device("cuda:0")
engine.set_precision("tf32x3")
lossf = LossFunc("mse", "distractor")
batches = [[torch.from_numpy(a).to(dev) for a in synth.task_batch("distractor", T, NC, NT, seed=100 + i)]
           for i in range(4)]


def arm(k):
    """A graphed run with accumulate_steps=k whose every role is captured; returns call() -> one micro-batch."""
    model = ANPDistractor(make_cfg(T, str(dev))).to(dev)
    g = GraphedStep(model, lossf, FusedAdam(FlatParams(model), lr=1e-4, accumulate_steps=k), warmup=3)
    n = [0]

    def call():
        n[0] += 1
        return g(batches[n[0] % len(batches)])
    for _ in range(2 * k):
        call()
    torch.cuda.synchronize()
    return call


def ms_per_task(call, k, windows, tasks):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(windows * k):
        call()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (windows * k * tasks)


def gradient_calls(k, windows=2):
    """Gradient all-reduce calls per window of an eager run (the ANP stabiliser's scalar exchanges not counted)."""
    model = ANPDistractor(make_cfg(T, str(dev))).to(dev)
    opt = FusedAdam(FlatParams(model), lr=1e-4, accumulate_steps=k)
    calls, real = [0], dist.all_reduce_sum

    def counting(t):
        calls[0] += t.untyped_storage().data_ptr() == opt.flat.grad.untyped_storage().data_ptr()
        return real(t)
    dist.all_reduce_sum = counting
    try:
        for _ in range(windows):
            opt.zero_grad()
            for i in range(k):
                cx, cy, tx, ty = batches[i % len(batches)]
                with opt.no_sync() if i < k - 1 else contextlib.nullcontext():
                    mu, _, _ = model(cx, cy, tx)
                    lossf.calc_loss(mu, None, ty).backward()
            opt.step()
        torch.cuda.synchronize()
    finally:
        dist.all_reduce_sum = real
    return calls[0] / windows


def worker():
    W = dist.world_size()
    out = {"gradient_allreduce_calls_per_window": {k: gradient_calls(k) for k in (1, 4)}}
    arms = {k: arm(k) for k in (1, 4)}
    us = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, call in arms.items():
            us[k].append(round(1e3 * ms_per_task(call, k, args.windows, T * W), 3))
    out["us_per_task"] = us
    out["ranks"], out["tasks_per_rank_and_micro_batch"] = W, T
    if dist.rank() == 0:
        print("RESULT " + json.dumps(out), flush=True)
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()


if args.worker:
    worker()
    raise SystemExit(0)

# 1 and 2: time per task for k = 1, 2, 4, alternating; per-call times of the k = 4 run
arms = {k: arm(k) for k in KS}
us_per_task = {k: [] for k in KS}
for _ in range(args.rounds):
    for k in KS:
        us_per_task[k].append(round(1e3 * ms_per_task(arms[k], k, args.windows, T), 3))
per_role = {"first": [], "middle": [], "last": []}
evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(4 * args.windows)]
for a, b in evs:
    a.record()
    arms[4]()
    b.record()
torch.cuda.synchronize()
for i, (a, b) in enumerate(evs):
    per_role["first" if i % 4 == 0 else "last" if i % 4 == 3 else "middle"].append(a.elapsed_time(b))
call_ms = {r: round(sum(v) / len(v), 4) for r, v in per_role.items()}
del arms
torch.cuda.empty_cache()

# 3: the gather alone
model = ANPDistractor(make_cfg(T, str(dev))).to(dev)
flat = FlatParams(model)
flat.zero_grad()
cx, cy, tx, ty = batches[0]
mu, _, _ = model(cx, cy, tx)
lossf.calc_loss(mu, None, ty).backward()
segs = [(p.grad.contiguous(), off, k) for _, p, off, k in flat.live]
floats = sum(k for _, _, k in segs)


def gather_us(fn, per_graph=20):
    """us per gather: `per_graph` calls captured in one CUDA graph (as in the step graphs: no host time), replayed."""
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(per_graph):
            fn(flat.grad, segs)
    graph.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.launches // per_graph):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / (args.launches // per_graph * per_graph)


for fn in (ops.multi_copy, ops.multi_accumulate):
    fn(flat.grad, segs)
torch.cuda.synchronize()
gather = {"copy": [], "accumulate": []}
for _ in range(args.rounds):
    gather["copy"].append(round(gather_us(ops.multi_copy), 2))
    gather["accumulate"].append(round(gather_us(ops.multi_accumulate), 2))
gather_GBps = {"copy": round(8 * floats / (min(gather["copy"]) * 1e3), 1),
               "accumulate": round(12 * floats / (min(gather["accumulate"]) * 1e3), 1)}

# 4: two ranks
two = None
if torch.cuda.device_count() >= 2:
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29671", os.path.abspath(__file__), "--worker", "--rounds", str(args.rounds),
           "--windows", str(args.windows)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=1800)
    lines = [l for l in res.stdout.splitlines() if l.startswith("RESULT ")]
    two = json.loads(lines[-1][7:]) if lines else {"error": (res.stdout + res.stderr)[-2000:]}

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                   capture_output=True, text=True).stdout.strip()
print(json.dumps({
    "workload": f"ANPDistractor graphed step, tf32x3, {T} tasks per micro-batch, nc={NC} nt={NT}",
    "us_per_task": us_per_task, "windows_per_timing": args.windows,
    "k4_call_ms": call_ms,
    "micro_step_over_step": round((call_ms["first"] + call_ms["middle"]) / 2 / call_ms["last"], 4),
    "gather_us": gather, "gather_GB_per_s_best": gather_GBps, "gather_live_floats": floats,
    "gather_segments": len(segs),
    "launches_per_timing": args.launches,
    "two_gpus": two, "gpu": q or torch.cuda.get_device_name(0)}))
