#!/usr/bin/env python
"""Benchmark: ANPDistractor meta-train tasks/sec (BASELINE.json's metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--precision tf32x3|tf32|fp32]
                    [--dump-outputs DIR]

One step = zero_grad + forward + loss + backward + (gradient all-reduce) + Adam on a synthetic
Distractor-shaped meta-batch: 20 tasks per GPU (cfg/train/ANP_Distractor.yaml:10), 15 context
and 21 target images of 128x128x1 per task (weak scaling: per-GPU work is fixed).

Prints ONE JSON line (rank 0).  `value` is timed with inputs resident in HBM; `e2e` times the same
step through the public API with pinned HOST inputs copied in and the loss read back every step.
`--impl reference` times the reference's own modules (networks.ANPDistractor + trainer.losses.LossFunc +
torch.optim.Adam, unmodified, from the byte-identical copy oracle/_ref that oracle/make_ref.py materialises;
kind "reference") on the box's host cores, on the FULL 20-task step; without that copy it falls back to the CPU
restatement (oracle/np_oracle.py, kind "port") on a 2-task sample.  `--impl reference-gpu` (internal; run as a
subprocess by the B200 arm) times the same reference modules on the B200 through cuDNN / cuBLAS -- the on-box bar.

Other workloads (BASELINE.json configs 2, 4, 5): --model CNPShapeNet1D|ANP|CNPDistractor|ANPShapeNet1D|CondNeuralProcess,
--nc N (nt follows the dataset's split), --scaling strong --tasks G (global meta-batch G split over the ranks).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "what-matters-for-meta-learning_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

TASKS_PER_GPU, NC, NT = 20, 15, 21
METRIC, UNIT = "ANPDistractor meta-train tasks/sec", "tasks/s"

# model: (task, agg_mode, img_agg, extra config, default tasks/GPU, views per task)   -- cfg/train/*.yaml
MODELS = {
    "ANPDistractor": ("distractor", "attention", "max", dict(dim_w=16), 20, 36),
    "CNPDistractor": ("distractor", "max", "max", dict(dim_w=16), 20, 36),
    "ANP": ("shapenet_3d", "attention", "reshape", dict(), 20, 30),
    "CondNeuralProcess": ("shapenet_3d", "max", "reshape", dict(), 20, 30),
    "CNPShapeNet1D": ("shapenet_1d", "mean", "", dict(dim_w=64, dim_r=100, dim_z=64, n_hidden_units_r=[100, 100]), 10, 30),
    "ANPShapeNet1D": ("shapenet_1d", "attention", "", dict(dim_w=64, dim_r=64, dim_z=64, n_hidden_units_r=[100, 100]), 10, 30),
}
IMG = {"distractor": ([128, 128, 1], 2, 2), "shapenet_1d": ([128, 128, 1], 3, 2), "shapenet_3d": ([64, 64, 4], 4, 4)}


def make_cfg(T, device, model="ANPDistractor"):
    """Namespace with the attributes configs/config.py:33-104 would set from cfg/train/<model>.yaml."""
    task, agg, img_agg, extra, _, _ = MODELS[model]
    img_size, input_dim, output_dim = IMG[task]
    base = dict(method=model, device=device, img_size=img_size, task=task, tasks_per_batch=T, input_dim=input_dim,
                output_dim=output_dim, agg_mode=agg, img_agg=img_agg, dim_w=None, dim_r=None, dim_z=None,
                n_hidden_units_r=None, temperature=0.07, seed=2578, loss_type="mse", beta=0, contrastive=False,
                max_ctx_num=15)
    base.update(extra)
    return types.SimpleNamespace(**base)


def workload(args):
    """(model, task, tasks per rank, nc, nt) of this invocation."""
    task, _, _, _, t_default, views = MODELS[args.model]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.scaling == "strong":
        if args.tasks % world:
            raise SystemExit(f"--tasks {args.tasks} is not divisible by {world} ranks")
        T = args.tasks // world
    else:
        T = args.tasks or t_default
    nc = args.nc if args.nc is not None else 15
    if args.nt is not None:
        nt = args.nt
    elif args.model == "ANPDistractor" or task == "distractor":
        nt = views - nc            # train split of the 36 views (shapenet_distractor.py:287-294)
    else:
        nt = 15
    return args.model, task, T, nc, nt


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], bf16=p["bf16_tflops"], bf16_sustained=p["bf16_tflops_sustained"], src="measured")
    except Exception:
        return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


# --------------------------------------------------------------------------------------------
# reference arms: the reference's own modules (oracle/_ref) on the host cores / on the GPU; oracle port fallback
# --------------------------------------------------------------------------------------------
REF_COPY = os.path.join(ROOT, "oracle", "_ref")


def have_reference_copy():
    return os.path.isfile(os.path.join(REF_COPY, "networks", "ANPDistractor.py"))


def _reference_stepper(model_name, T, nc, nt, device):
    """zero_grad -> forward -> loss -> backward -> Adam with the UNMODIFIED reference classes
    (train.py:41-56,92; trainer/model_trainer.py:59-93), inputs resident on `device`."""
    os.environ["B200NP_REFERENCE_ROOT"] = REF_COPY      # never /root/reference at run time: it is not on the GPU box
    while PKG in sys.path:                              # none of the B200 package on this arm's import path
        sys.path.remove(PKG)
    for k in [k for k in sys.modules if k.split(".")[0] in ("networks", "trainer", "b200np")]:
        del sys.modules[k]
    from oracle import ref_shims, synth
    cfg = make_cfg(T, device, model_name)
    model = ref_shims.reference_class(model_name)(cfg).to(device)
    lossf = ref_shims.reference_lossfunc()(cfg.loss_type, cfg.task)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    batch = [torch.from_numpy(a).to(device) for a in synth.task_batch(cfg.task, T, nc, nt, seed=1)]
    model.train()

    def step():
        cx, cy, tx, ty = batch
        opt.zero_grad()
        mu, var, kl = model(cx, cy, tx)
        loss = lossf.calc_loss(mu, var, ty)
        loss += kl * cfg.beta
        loss.backward()
        opt.step()
        return loss
    return step


def cpu_port_step_time(sample_tasks, steps, warmup):
    from oracle import np_oracle, synth
    from networks.ANPDistractor import ANPDistractor
    torch.set_num_threads(os.cpu_count() or 1)
    model = ANPDistractor(make_cfg(sample_tasks, "cpu"))  # parameter holder only (seeded init)
    ocfg = dict(tasks_per_batch=sample_tasks, agg_mode="attention", img_agg="max", task="distractor")
    tr = np_oracle.OracleTrainer("ANPDistractor", ocfg, model.state_dict(), lr=1e-4)
    batch = [torch.from_numpy(a) for a in synth.task_batch("distractor", sample_tasks, NC, NT, seed=1)]
    for _ in range(warmup):
        tr.step(*batch)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        tr.step(*batch)
        times.append(time.perf_counter() - t0)
    return times


def run_reference_arm(args, rank):
    """CPU arm.  With oracle/_ref: the reference's own modules on the full per-GPU step (same config as the B200 arm).
    Otherwise the oracle port on a 2-task sample."""
    if rank != 0:
        return
    model_name, task, T, nc, nt = workload(args)
    torch.set_num_threads(os.cpu_count() or 1)
    cores = torch.get_num_threads()
    if have_reference_copy():
        kind, sample = "reference", T
        step = _reference_stepper(model_name, T, nc, nt, "cpu")
        for _ in range(args.warmup):
            step()
        times = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            float(step().detach())
            times.append(time.perf_counter() - t0)
        what = (f"the reference's own {model_name} + LossFunc + torch.optim.Adam (oracle/_ref, unmodified), "
                f"full step of {T} tasks (nc={nc}, nt={nt}) per timed step")
    else:
        if model_name != "ANPDistractor":
            raise SystemExit("the oracle-port fallback of the reference arm only covers ANPDistractor")
        kind, sample = "port", 2
        times = cpu_port_step_time(sample, args.steps, args.warmup)
        what = f"{sample} tasks/step (nc={nc}, nt={nt}), full fwd+loss+bwd+Adam, oracle/np_oracle.py"
    total = sum(times)
    value = sample * len(times) / total
    line = {
        "impl": "reference", "metric": metric_name(model_name), "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1, extra={"note": "CPU arm: host cores only; one rank's share of the step"}),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": what},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_reference_gpu_arm(args):
    """On-box bar (SURVEY.md 8d): the reference's own modules on the B200 through cuDNN / cuBLAS / ATen, once with
    PyTorch's defaults (cuDNN convolutions may use TF32, matmuls stay fp32) and once with TF32 disallowed."""
    if not have_reference_copy():
        print(json.dumps({"impl": "reference-gpu", "unavailable": "oracle/_ref not materialised"}))
        return
    model_name, task, T, nc, nt = workload(args)
    out = {"impl": "reference-gpu", "model": model_name, "tasks": T, "nc": nc, "nt": nt}
    for label, tf32 in (("cudnn_tf32_default", True), ("fp32", False)):
        torch.backends.cudnn.allow_tf32 = tf32
        step = _reference_stepper(model_name, T, nc, nt, "cuda:0")
        for _ in range(max(args.warmup, 3)):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        out[label] = {"ms_per_step": ms, "tasks_per_s": T / ms * 1e3}
        del step
        torch.cuda.empty_cache()
    out["peak_mem_GB"] = torch.cuda.max_memory_allocated() / 1e9
    print(json.dumps(out), flush=True)


def _sub_json(argv, timeout):
    """Run `python bench.py <argv>` in a fresh process (the reference's `networks` package and the drop-in one cannot
    share an interpreter) and return its last JSON line, or a dict with the failure."""
    try:
        env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
        r = subprocess.run([sys.executable, os.path.abspath(__file__)] + argv, capture_output=True, text=True,
                           timeout=timeout, env=env)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"unavailable": (r.stderr or "no output").strip().splitlines()[-1][:200]}
    except Exception as e:   # noqa: BLE001
        return {"unavailable": repr(e)[:200]}


def metric_name(model_name):
    return f"{model_name} meta-train tasks/sec"


def workload_config(args, world, extra=None):
    model_name, task, T, nc, nt = workload(args)
    img = "64x64x3" if task == "shapenet_3d" else "128x128x1"
    cfg = {"workload": f"{model_name} meta-train step (fwd+loss+bwd+allreduce+Adam), {T} tasks/GPU, nc={nc} nt={nt}, "
                       f"{img} images, global tasks={T * world}",
           "model_class": model_name, "tasks_per_gpu": T, "global_tasks": T * world, "nc": nc, "nt": nt}
    if extra:
        cfg.update(extra)
    return cfg


# --------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for nme, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------
def run_b200_arm(args, rank, world, local_rank):
    import importlib

    import torch.distributed as td
    from b200np import engine
    from b200np.lib import LIB
    from b200np.optim import FlatParams, FusedAdam, GraphedStep
    from oracle import synth  # input generator only (integer hash); no oracle compute here
    from trainer.losses import LossFunc

    if "B200NP_WGRAD_WAVES" in os.environ:   # diagnostic entry point: pixel chunks per weight-gradient launch
        LIB.b200np_debug_set_wgrad_waves(int(os.environ["B200NP_WGRAD_WAVES"]))
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    if world > 1:
        td.init_process_group("nccl", device_id=dev)
    engine.set_precision(args.precision)
    model_name, task, T, nc, nt = workload(args)
    cls = getattr(importlib.import_module(f"networks.{model_name}"), model_name)
    model = cls(make_cfg(T, str(dev), model_name)).to(dev)
    flat = FlatParams(model)
    opt = FusedAdam(flat, lr=1e-4)
    lossf = LossFunc("mse", task)

    # 4 distinct resident batches per rank (ANPDistractor: 189 MB of inputs > 126 MB L2; a step also streams ~2 GB of
    # activations, far beyond L2), rotated between iterations
    nbatch = 4
    host = [[torch.from_numpy(a).pin_memory() for a in synth.task_batch(task, T, nc, nt, seed=100 * rank + i)]
            for i in range(nbatch)]
    resident = [[t.to(dev) for t in b] for b in host]

    def step(batch):
        cx, cy, tx, ty = batch
        opt.zero_grad()
        mu, _, _ = model(cx, cy, tx)
        loss = lossf.calc_loss(mu, None, ty)
        loss.backward()
        opt.step()
        return loss

    def barrier():
        if world > 1:
            td.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            td.all_reduce(ms, op=td.ReduceOp.MAX)
        return float(ms)

    launches_per_step = None
    if args.graph:
        # the whole step (every kernel of fwd + loss + bwd + all-reduce + Adam) captured once, replayed per step
        l0 = LIB.b200np_launch_count()
        gstep = GraphedStep(model, lossf, opt, resident[0], warmup=max(args.warmup, 3))
        launches_per_step = (LIB.b200np_launch_count() - l0) // (max(args.warmup, 3) + 1)
        run = gstep
    else:
        run = step
    for i in range(args.warmup):
        run(resident[i % nbatch])
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = LIB.b200np_launch_count()
    last = {}

    def timed_step(i):
        last["loss"] = run(resident[i % nbatch])
    ms = timed(timed_step, args.steps)
    launches = launches_per_step * args.steps if args.graph else LIB.b200np_launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # before the e2e leg below trains the same model further
        dump_outputs(args.dump_outputs, loss=last["loss"], params=flat.flat[:flat.n_live], grads=flat.grad)

    # end to end: pinned host inputs -> device every step, loss read back every step
    def e2e_step(i):
        if args.graph:
            # this step's inputs were put on the wire (pinned host -> device, copy stream) while the previous step
            # computed; this call starts the copy of the next step's inputs and reads this step's loss back
            return float(gstep(host[i % nbatch], next_batch=host[(i + 1) % nbatch]))
        b = [t.to(dev, non_blocking=True) for t in host[i % nbatch]]
        return float(step(b).detach())
    e2e_steps = max(3, min(args.steps, 10))
    h2d = sum(t.numel() * 4 for t in host[0])
    if args.profile:
        ms_e2e = float("nan")
    else:
        e2e_step(0)
        ms_e2e = timed(e2e_step, e2e_steps)

    def finish():
        """Common exit: a captured graph holds NCCL kernels, so drop it before the communicator; every rank
        leaves through the same barrier; multi-rank processes then exit without interpreter teardown (an
        orderly NCCL shutdown after graph capture was observed to stall for minutes)."""
        nonlocal run
        if args.graph:
            run = None
        torch.cuda.synchronize()
        if world > 1:
            td.barrier()
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)

    if rank != 0:
        finish()
        return
    extras = {}
    if world == 1 and not args.profile and not args.no_dropin:
        extras["e2e_dropin"] = dropin_loop(args, dev, model_name, task, T, nc, nt)
    is_headline = model_name == "ANPDistractor" and (nc, nt) == (NC, NT)
    roof = dominant_kernel_roofline(args, dev) if (not args.profile and is_headline) else None
    if roof is not None:
        extras["tf32_cublas_peak"] = measured_tf32_peak(dev)
        extras["hbm_kernels"] = hbm_bound_kernels(dev, T, nc, nt, flat.n_live)
    cpu = gpu_ref = None
    if world == 1 and not args.no_cpu_baseline and not args.profile:
        # free this process's GPU memory first: the on-box bar below runs the reference on the same GPU
        fwd = ["--model", model_name, "--nc", str(nc), "--nt", str(nt), "--tasks", str(T)]
        sub = _sub_json(["--impl", "reference", "--steps", "3", "--warmup", "1"] + fwd, timeout=600)
        cpu = sub.get("cpu_baseline") or {"unavailable": sub.get("unavailable", "no cpu_baseline in the sub-run")}
        if "value" in cpu:
            cpu["sample"] = "3 timed steps after 1 warm-up; " + cpu["sample"]
        gpu_ref = _sub_json(["--impl", "reference-gpu", "--steps", "5", "--warmup", "3"] + fwd, timeout=600)
    tasks = T * world
    line = {
        "metric": metric_name(model_name), "value": tasks * args.steps / (ms / 1e3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None,
        "dtype": {"tf32x3": "f32 (3xTF32 split on tcgen05, fp32 accumulate)", "tf32": "tf32", "fp32": "f32"}[args.precision],
        "data": "synthetic",
        "config": workload_config(args, world, extra={
            "precision": args.precision, "cuda_graph": bool(args.graph),
            "l2": "inputs rotate over 4 resident batches (ANPDistractor: 189 MB > 126 MB L2); ~2 GB of activations "
                  "streamed per step"}),
        "e2e": {"value": tasks * e2e_steps / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4, "steps": e2e_steps},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roof,
        "cpu_baseline": cpu,
        "gpu_reference": gpu_ref,
    }
    line.update(extras)
    print(json.dumps(line), flush=True)
    finish()


def dump_outputs(out_dir, **arrays):
    """What the last timed step handed its caller, as float32 `<out_dir>/<name>.npy`: the loss, the flat live
    parameters after the Adam update and the flat gradient they were updated with."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy().reshape(-1))


def dropin_loop(args, dev, model_name, task, T, nc, nt):
    """The reference trainer's own loop (trainer/model_trainer.py:59-93) on the drop-in modules: zero_grad ->
    .to(device) of a pinned host batch -> model -> calc_loss -> `losses += kl * beta` -> backward ->
    torch.optim.Adam.step -> losses.item(), forward / backward replayed as per-shape CUDA graphs behind the nn.Module
    contract (b200np/graphed.py).  Two numbers: the bench's fixed (nc, nt), and `shot ~ U{1..15}` redrawn per step
    like dataset/shapenet_distractor.py:197 (nt = views - nc, so the work per step varies)."""
    import importlib
    import random

    from oracle import synth
    from trainer.losses import LossFunc
    cls = getattr(importlib.import_module(f"networks.{model_name}"), model_name)
    cfg = make_cfg(T, str(dev), model_name)
    model = cls(cfg).to(dev)
    model.enable_cuda_graphs(True)
    lossf = LossFunc("mse", task)
    optimizer = torch.optim.Adam(model.parameters(), lr=1e-4)
    views = nc + nt
    out = {}
    for label, shots in (("fixed_shot", [nc]), ("shot_uniform_1_15", list(range(1, 16)))):
        if label != "fixed_shot" and views - 15 < 1:
            continue
        pool = {k: [torch.from_numpy(a).pin_memory() for a in synth.task_batch(task, T, k, views - k, seed=7 + k)]
                for k in shots}
        rng = random.Random(0)

        def one():
            k = shots[rng.randrange(len(shots))]
            model.train()
            optimizer.zero_grad()
            ctx_x, ctx_y, qry_x, qry_y = (t.to(dev) for t in pool[k])
            pr_mu, pr_var, kl = model(ctx_x, ctx_y, qry_x)
            losses = lossf.calc_loss(pr_mu, pr_var, qry_y)
            losses += kl * cfg.beta
            losses.backward()
            optimizer.step()
            return losses.item()
        for k in shots:          # build every shape's graphs outside the timed region
            rng_state = rng.getstate()
            shots_saved, shots[:] = list(shots), [k]
            one()
            shots[:] = shots_saved
            rng.setstate(rng_state)
        n = max(5, min(args.steps, 20))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n):
            one()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        out[label] = {"value": T * n / dt, "unit": UNIT, "ms_per_step": 1e3 * dt / n, "steps": n}
    out["h2d_bytes_per_step"] = sum(t.numel() * 4 for t in next(iter(pool.values())))
    out["d2h_bytes_per_step"] = 4
    out["what"] = ("reference-style training loop (model_trainer.py:59-93) with torch.optim.Adam on the drop-in modules, "
                   "pinned host batch -> .to(device) and loss.item() every step, wall clock")
    del model, optimizer
    torch.cuda.empty_cache()
    return out


def measured_tf32_peak(dev):
    """cuBLAS TF32 GEMM 8192^3 (torch.matmul with allow_tf32), best of 10 -- measured the way MEASURED_PEAKS.json
    measures bf16 (BASELINE.md section 3 asks for the TF32 figure); context for the roofline's bf16/2 denominator."""
    n = 8192
    a = torch.randn(n, n, device=dev)
    b = torch.randn(n, n, device=dev)
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        for _ in range(3):
            a @ b
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a @ b
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    return {"tflops": 2.0 * n ** 3 / (best * 1e-3) / 1e12, "how": "torch.matmul fp32 8192^3 with allow_tf32, best of 10"}


def hbm_bound_kernels(dev, T, nc, nt, n_params):
    """Achieved HBM GB/s of the HBM-bound class (north_star: aggregation, pooling, loss, Adam), each timed alone on
    buffers larger than L2 where the op's own size allows (Adam; the others are KB-sized at this workload and are
    reported at a 64x scaled batch so that the number is a bandwidth, not a launch latency)."""
    from b200np import ops
    pk = peaks()
    out = {}

    def entry(sec, nbytes, what):
        return {"GBps": nbytes / sec / 1e9, "frac_of_hbm_peak": nbytes / sec / 1e9 / pk["hbm"], "bytes": nbytes,
                "us": sec * 1e6, "what": what}
    # Adam over 64 M parameters (16 B read + 12 B written each; the model's own 3.2 M-parameter launch is 90 MB)
    n = 64 * 1024 * 1024
    p, g, m, v = (torch.randn(n, device=dev) * 0.01 for _ in range(4))
    v.abs_()
    t_dev = torch.zeros(1, device=dev, dtype=torch.int32)
    sec = _time_kernel(lambda: ops.adam_step_dev(p, g, m, v, n, 1e-4, 0.9, 0.999, 1e-8, 0.0, t_dev))
    out["adam"] = entry(sec, 28 * n, "fused Adam, 64 Mi parameters")
    pm, gm, mm, vm = (t[:n_params] for t in (p, g, m, v))
    sec = _time_kernel(lambda: ops.adam_step_dev(pm, gm, mm, vm, n_params, 1e-4, 0.9, 0.999, 1e-8, 0.0, t_dev))
    out["adam_model_size"] = entry(sec, 28 * n_params, f"fused Adam at the model's size ({n_params} parameters, L2-resident)")
    del p, g, m, v
    # context max-aggregation over nc: reads T*nc*256 floats, writes T*256 values + indices
    Tb = T * 2048
    feats = torch.randn(Tb, nc, 256, device=dev)
    sec = _time_kernel(lambda: ops.ctx_aggregate_fwd(feats, 1))
    out["ctx_aggregate_max"] = entry(sec, feats.numel() * 4 + Tb * 256 * 8, f"max over nc={nc}, {Tb} tasks x 256 features")
    del feats
    # adaptive max-pool 2x2 + flatten of the trunk's last map [N,4,4,64] -> [N,256] (+ argmax)
    Nb = T * (nc + nt) * 512
    x = torch.randn(Nb, 4, 4, 64, device=dev)
    sec = _time_kernel(lambda: ops.amp2_flatten_fwd(x))
    out["adaptive_maxpool_flatten"] = entry(sec, x.numel() * 4 + Nb * 256 * 8, f"{Nb} maps of 4x4x64")
    del x
    # loss forward + backward (distractor): reads mu and y, writes d mu
    R = T * nt * 65536
    mu = torch.randn(R, 2, device=dev)
    y = torch.randn(R, 2, device=dev)
    sec = _time_kernel(lambda: ops.loss_fwd_bwd(mu, y, 0))
    out["loss_fwd_bwd"] = entry(sec, R * 2 * 4 * 3, f"distractor loss, {R} rows")
    return out


def ncu_traffic(key, images, precision):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of a roofline kernel, from profiles/ncu_traffic.json
    (filled in from the committed `ncu --set full` captures of `bench.py --roofline-only`); None when the file is
    missing or was captured at another size / precision -- a stale constant must not pass for a measurement."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)
        if t.get("images") != images or t.get("precision") != precision:
            return None
        return float(t[key]["bytes"])
    except Exception:
        return None


def _time_kernel(run, reps=10):
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


def dominant_kernel_roofline(args, dev):
    """Times the dominant kernels of the step alone, with CUDA events on the launching stream (torch's current
    stream, which is the one the C ABI is given).  By CUPTI kernel time (profiles/profile_step_r2.txt) the dominant
    kernel is the TMA-fed halo convolution `tapconv_halo_tma_kernel` (21 % of the step in its 10-tap instance alone, 39 %
    over its three instances); it is timed on its largest instance, the fused `conv2 3x3 + 1x1 s2 skip + bias + ReLU`
    forward of layer1 at the step's own size (all 1140 images of a 20-task ANP step: M = 1140*32*32 pixels, N = 64,
    K = 640).  Algorithmic FLOPs = 2*M*64*640 per launch (SURVEY.md appendix C: 75.5 + 8.4 MFLOP/image); algorithmic
    HBM bytes = input h + every second pixel of every second row of x (the stride-2 skip) + the output.
    Peak = measured dense bf16 / 2 (tf32 issues at half the bf16 rate); the fp32-grade 3xTF32 split spends
    3 MMAs per algorithmic MAC, so its ceiling on this scale is 1/3.  The weight gradient of the same layer
    (`tapwgrad_halo_tma_kernel`, second by time; round 1's dominant kernel) is reported beside it (`second_kernel`)."""
    from b200np import ops
    from b200np.lib import PREC_FP32_SIMT, PREC_TF32, PREC_TF32X3
    prec = {"tf32x3": PREC_TF32X3, "tf32": PREC_TF32, "fp32": PREC_FP32_SIMT}[args.precision]
    N = TASKS_PER_GPU * (NC + NT) + TASKS_PER_GPU * NT
    g = torch.Generator(device="cpu").manual_seed(0)
    x = torch.rand(N, 64, 64, 64, generator=g).to(dev)          # block input  (NHWC)
    h = torch.rand(N, 32, 32, 64, generator=g).to(dev)          # conv1 output (NHWC)
    dy = torch.randn(N, 32, 32, 64, generator=g).to(dev)        # gradient of the block output
    w2 = (torch.randn(64, 64, 3, 3, generator=g) * 0.04).to(dev)
    ws = (torch.randn(64, 64, 1, 1, generator=g) * 0.1).to(dev)
    b = torch.zeros(64, device=dev)
    wf2 = ops.pack_conv_weight(w2)
    wfs = ops.pack_conv_weight(ws)
    flops = 2.0 * N * 32 * 32 * 64 * 640
    # both kernels touch h, every second pixel of every second row of x (the stride-2 skip) and one more
    # 32x32x64 tensor (dY or the output): 3 x 299 MB
    alg_bytes = (h.numel() + x.numel() // 4 + N * 32 * 32 * 64) * 4
    pk = peaks()
    peak = pk["bf16"] / 2.0

    def entry(name, key, sec):
        ach = flops / sec / 1e12
        return {"kernel": name, "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                "frac": ach / peak, "peak_source": f"{pk['src']} bf16 burst {pk['bf16']} TFLOP/s / 2 (tf32 rate)",
                "traffic": ncu_traffic(key, N, args.precision), "launch_ms": sec * 1e3,
                "algorithmic_flop": flops,
                "hbm_view": {"algorithmic_GB": alg_bytes / 1e9, "achieved_GBps": alg_bytes / sec / 1e9,
                             "peak_GBps": pk["hbm"], "frac": alg_bytes / sec / 1e9 / pk["hbm"]}}

    if prec == PREC_FP32_SIMT:
        t_w = _time_kernel(lambda: ops.conv_wgrad(h, dy, 3, 1, prec))
    else:
        t_w = _time_kernel(lambda: ops.conv_wgrad(h, dy, 3, 1, prec, skip=(x, 2)))
    t_f = _time_kernel(lambda: ops.conv_fwd(h, wf2, b, 1, 1, prec, skip=(x, wfs, b, 2)))
    out = entry("tapconv_halo_tma (layer1 conv2 3x3 + 1x1 skip + bias + ReLU forward, implicit GEMM on tcgen05, planes by "
                "TMA tensor maps)", "tapconv_halo", t_f)
    out["second_kernel"] = entry("tapwgrad_halo_tma (layer1 conv2 3x3 + 1x1 skip weight gradient, pixel contraction on "
                                 "tcgen05, operands by TMA tensor maps)", "tapwgrad", t_w)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-gpu"])
    ap.add_argument("--precision", default=os.environ.get("B200NP_PRECISION", "tf32x3"),
                    choices=["tf32x3", "tf32", "fp32"])
    ap.add_argument("--model", default="ANPDistractor", choices=sorted(MODELS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --tasks (default: the YAML's tasks_per_batch) per GPU; strong: --tasks is the GLOBAL "
                         "meta-batch, split over the ranks")
    ap.add_argument("--tasks", type=int, default=0)
    ap.add_argument("--nc", type=int, default=None, help="context images per task (default 15)")
    ap.add_argument("--nt", type=int, default=None, help="target images per task (default: the dataset's train split)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU and on-GPU reference legs")
    ap.add_argument("--no-dropin", action="store_true", help="skip the reference-style training-loop leg (e2e_dropin)")
    ap.add_argument("--no-graph", dest="graph", action="store_false",
                    help="launch every kernel from Python each step instead of replaying the captured CUDA graph")
    ap.add_argument("--roofline-only", action="store_true",
                    help="run only the dominant-kernel timing (the command captured by `ncu --set full`)")
    ap.add_argument("--profile", action="store_true",
                    help="only the resident-input timed loop (for ncu launch lists); skips e2e / roofline / CPU legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's loss, updated parameters and gradient as "
                         "DIR/<name>.npy (float32; same arguments, same inputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.roofline_only):
        ap.error("--dump-outputs dumps the B200 arm's timed step: not with --impl reference* or --roofline-only")
    if args.scaling == "strong" and not args.tasks:
        ap.error("--scaling strong needs --tasks (the global meta-batch)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if args.impl == "reference-gpu":
        run_reference_gpu_arm(args)
        return
    if args.roofline_only:
        print(json.dumps(dominant_kernel_roofline(args, torch.device("cuda:0"))))
        return
    if args.profile:
        args.graph = False  # ncu needs the individual launches
    else:
        args.warmup = max(args.warmup, 3)
    run_b200_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
