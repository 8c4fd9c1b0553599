"""Learning-rate schedules, global-norm gradient clipping and non-finite step skipping on the fused training path.

The total-norm kernel is checked against fp64 torch with guard bands, bitwise repeats and non-finite probes.  With
clipping and skipping off, FusedAdam's step is bit-identical to `adam_step_dev` and launches no norm kernel.  With
them on, it follows `clip_grad_norm_` + `torch.optim.Adam` + a torch LR scheduler; a per-step schedule under CUDA
graphs captures once per shape and never synchronises; a NaN batch leaves the training state untouched; scheduled,
clipped runs checkpoint and resume bit for bit; and two ranks make the same clip and skip decisions.
"""
import copy
import os
import subprocess
import sys
import warnings

import pytest
import torch

from conftest import CASES, build_product_model
from oracle import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LR = 1e-3


def _anp_live_count():
    import bench
    from b200np.optim import FlatParams
    from networks.ANPDistractor import ANPDistractor
    return FlatParams(ANPDistractor(bench.make_cfg(bench.MODELS["ANPDistractor"][4], "cuda")).to("cuda")).n_live


# ------------------------------------------------------------------------------------------------
# the norm kernel
# ------------------------------------------------------------------------------------------------
GUARD = 64     # floats of guard band on either side of every buffer


class Guarded:
    """[guard | payload | guard] in one allocation; the payload starts `off` floats past a 256-B boundary."""

    def __init__(self, n, off=0, dtype=torch.float32, fill=float("nan")):
        self.buf = torch.full((GUARD + off + n + GUARD,), fill, device="cuda", dtype=dtype)
        self.lo, self.hi = GUARD + off, GUARD + off + n
        self.t = self.buf[self.lo:self.hi]
        self.guards = (self.buf[:self.lo].clone(), self.buf[self.hi:].clone())

    def guards_intact(self):
        eq = lambda a, b: torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a,
                                      b.view(torch.int32) if b.dtype == torch.float32 else b)
        return eq(self.buf[:self.lo], self.guards[0]) and eq(self.buf[self.hi:], self.guards[1])


def _norm(g, scale=1.0):
    """Run b200np_grad_norm on a guarded output and workspace; return the float result."""
    from b200np import lib
    from b200np.lib import LIB
    n = g.t.numel()
    out = Guarded(1)
    ws = Guarded(LIB.b200np_grad_norm_workspace(n), dtype=torch.uint8, fill=0xA5)
    lib.check(LIB.b200np_grad_norm(g.t.data_ptr(), n, scale, out.t.data_ptr(), ws.t.data_ptr(), ws.t.numel(),
                                   torch.cuda.current_stream().cuda_stream), "grad_norm")
    torch.cuda.synchronize()
    assert out.guards_intact() and ws.guards_intact() and g.guards_intact()
    return out.t.clone()


@pytest.mark.parametrize("off", [0, 1], ids=["aligned16", "offset4"])
@pytest.mark.parametrize("n", [1, 3, 4, 5, 1023, 148 * 1024 + 1, "anp_live"])
def test_grad_norm_matches_fp64(n, off):
    n = _anp_live_count() if n == "anp_live" else n
    gen = torch.Generator(device="cuda").manual_seed(n)
    g = Guarded(n, off)
    g.t.copy_(torch.randn(n, device="cuda", generator=gen) * torch.logspace(-6, 2, n, device="cuda"))
    before = g.t.clone()
    a, b = _norm(g, 0.5), _norm(g, 0.5)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))          # bitwise repeatable
    assert torch.equal(g.t, before)
    want = 0.5 * float(before.double().norm())
    assert abs(float(a) - want) <= 1e-6 * want, (float(a), want)


@pytest.mark.parametrize("off", [0, 1], ids=["aligned16", "offset4"])
@pytest.mark.parametrize("bad", [float("inf"), float("-inf"), float("nan")], ids=["inf", "-inf", "nan"])
def test_grad_norm_detects_one_nonfinite_element(bad, off):
    n = 4 * 1000 + 3                # 16-B aligned: float4 body and a 3-element scalar tail
    for pos in (0, n // 2, n - 4, n - 1):
        g = Guarded(n, off)
        g.t.copy_(torch.randn(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(pos)))
        g.t[pos] = bad
        r = float(_norm(g)[0])
        assert not (r == r and abs(r) != float("inf")), (pos, r)


# ------------------------------------------------------------------------------------------------
# FusedAdam on a small multi-tensor module
# ------------------------------------------------------------------------------------------------
def _mlp(dtype=torch.float32):
    torch.manual_seed(11)
    return torch.nn.Sequential(torch.nn.Linear(13, 64), torch.nn.Tanh(), torch.nn.Linear(64, 31), torch.nn.Tanh(),
                               torch.nn.Linear(31, 5)).to("cuda", dtype)


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@pytest.mark.parametrize("wd", [0.0, 0.01])
def test_default_path_is_bit_identical_to_adam_step_dev(wd):
    from b200np import ops
    from b200np.optim import FlatParams, FusedAdam
    flat = FlatParams(_mlp())
    opt = FusedAdam(flat, lr=LR, weight_decay=wd)
    n = flat.n_live
    p, m, v, t = flat.flat.clone(), opt.m.clone(), opt.v.clone(), opt.t_dev.clone()
    gen = torch.Generator(device="cuda").manual_seed(3)
    for i in range(5):
        g = torch.randn(n, device="cuda", generator=gen) * (10.0 ** (i - 2))
        opt.zero_grad()
        flat.attach_grads()
        flat.grad.copy_(g)
        if i == 4:
            names = _kernels(opt.step)
            assert any("adam_kernel" in k for k in names) and any("adam_tick_kernel" in k for k in names)
            assert not any("grad_norm" in k for k in names), names
        else:
            opt.step()
        ops.adam_step_dev(p, g, m, v, n, LR, 0.9, 0.999, 1e-8, wd, t)
    torch.cuda.synchronize()
    assert torch.equal(flat.flat[:n], p[:n]) and torch.equal(opt.m, m) and torch.equal(opt.v, v)
    assert torch.equal(opt.t_dev, t) and int(opt.t_dev) == 5


def test_clipped_scheduled_steps_match_torch_fp64():
    """FusedAdam(max_grad_norm=c) + LambdaLR against clip_grad_norm_ + torch.optim.Adam + LambdaLR in fp64."""
    from b200np.optim import FlatParams, FusedAdam
    model, ref = _mlp(), _mlp(torch.float64)
    flat = FlatParams(model)
    w0 = {k: p.detach().double().clone() for k, p in model.named_parameters()}
    gen = torch.Generator(device="cuda").manual_seed(5)
    data = [(torch.randn(32, 13, device="cuda", generator=gen), torch.randn(32, 5, device="cuda", generator=gen),
             50.0 if i % 2 else 0.05) for i in range(20)]

    def loss_of(net, x, y, s):
        return s * ((net(x) - y) ** 2).mean()
    loss_of(ref, data[0][0].double(), data[0][1].double(), 1.0).backward()
    c = float(torch.nn.utils.get_total_norm([p.grad for p in ref.parameters()]))   # between the two loss scales
    ref.zero_grad()
    lam = lambda k: 0.5 ** (k / 7) * (1 + (k % 3))
    opt = FusedAdam(flat, lr=LR, max_grad_norm=c)
    topt = torch.optim.Adam(ref.parameters(), lr=LR)
    sched, tsched = torch.optim.lr_scheduler.LambdaLR(opt, lam), torch.optim.lr_scheduler.LambdaLR(topt, lam)
    clipped = []
    for x, y, s in data:
        opt.zero_grad()
        loss_of(model, x, y, s).backward()
        opt.step()
        want = torch.nn.utils.get_total_norm([p.grad for p in model.parameters()])   # the fp32 gradient's norm
        assert abs(float(opt.grad_norm) - float(want)) <= 1e-6 * float(want)
        assert abs(float(flat.grad.double().norm()) - float(want)) <= 1e-6 * float(want)   # .grad stays unclipped
        topt.zero_grad()
        loss_of(ref, x.double(), y.double(), s).backward()
        clipped.append(float(torch.nn.utils.clip_grad_norm_(ref.parameters(), c)) > c)
        topt.step()
        sched.step(), tsched.step()
        assert opt.lr == topt.param_groups[0]["lr"]
    assert any(clipped) and not all(clipped), clipped
    num = den = 0.0
    for (k, p), q in zip(model.named_parameters(), ref.parameters()):
        num += float(((p.detach().double() - w0[k]) - (q.detach() - w0[k])).pow(2).sum())
        den += float((q.detach() - w0[k]).pow(2).sum())
    assert (num / den) ** 0.5 < 5e-2, (num / den) ** 0.5


# ------------------------------------------------------------------------------------------------
# the product models: schedules under graphs, skipping, checkpoints
# ------------------------------------------------------------------------------------------------
def _batches(case, n, seed=70):
    """`n` batches whose context size alternates between nc and nc + 2 (two graph shapes)."""
    method, task, agg, img_agg, extra, T, nc, nt = CASES[case]
    return [[torch.from_numpy(a).cuda() for a in synth.task_batch(task, T, nc + 2 * (i % 2), nt, seed=seed + i)]
            for i in range(n)]


def _nan_batch(batch):
    bad = [t.clone() for t in batch]
    bad[0][0] = float("nan")                       # the first context image of the first task
    return bad


def _schedule(k):
    return 1.0 / (1 + 0.3 * k) * (1.5 if k % 2 else 1.0)


def _fresh(case, graphed, **opt_kw):
    """(model, opt, GraphedStep or None, step(batch) -> loss clone)."""
    from b200np import engine
    from b200np.optim import FlatParams, FusedAdam, GraphedStep
    from trainer.losses import LossFunc
    engine.set_precision("tf32x3")
    model, _ = build_product_model(case, device="cuda")
    model = model.to("cuda")
    opt = FusedAdam(FlatParams(model), lr=LR, **opt_kw)
    lossf = LossFunc("mse", CASES[case][1])
    if graphed:
        g = GraphedStep(model, lossf, opt, warmup=1)
        return model, opt, g, lambda b: g(b).clone()

    def step(b):
        cx, cy, tx, ty = b
        opt.zero_grad()
        mu, _, _ = model(cx, cy, tx)
        loss = lossf.calc_loss(mu, None, ty)
        loss.backward()
        opt.step()
        return loss.detach().clone()
    return model, opt, None, step


@pytest.mark.parametrize("case", ["anp_distractor", "cnp_distractor_max"])
def test_per_step_schedule_under_graphs(case, monkeypatch):
    from b200np.optim import GraphedStep
    batches = _batches(case, 8)
    captures = []
    real = GraphedStep._capture
    monkeypatch.setattr(GraphedStep, "_capture", lambda self, ent: (captures.append(1), real(self, ent)))
    runs = []
    for graphed in (False, True):
        model, opt, g, step = _fresh(case, graphed, max_grad_norm=0.5)
        sched = torch.optim.lr_scheduler.LambdaLR(opt, _schedule)
        losses, lrs = [], []
        with warnings.catch_warnings():
            warnings.simplefilter("error")
            warnings.filterwarnings("ignore", message="Synchronization debug mode is a prototype")  # torch's own notice
            for i, b in enumerate(batches):
                # from the third step on both shapes are captured: replays and scheduler steps must not synchronise
                torch.cuda.set_sync_debug_mode("error" if graphed and i >= 2 else "default")
                try:
                    losses.append(step(b))
                    sched.step()
                finally:
                    torch.cuda.set_sync_debug_mode("default")
                lrs.append(opt.lr)
        torch.cuda.synchronize()
        runs.append(([float(l) for l in losses], lrs, {k: v.clone() for k, v in model.state_dict().items()}))
    assert len(captures) == 2, captures                          # one per shape, none for the 8 lr changes
    (le, lre, we), (lg, lrg, wg) = runs
    assert lre == lrg and len(set(lre)) == len(lre)
    assert le == pytest.approx(lg, rel=1e-6)
    for k in we:
        assert torch.allclose(we[k], wg[k], rtol=1e-5, atol=1e-7), k


def _state(opt):
    return (opt.flat.flat.clone(), opt.m.clone(), opt.v.clone(), opt.t_dev.clone())


def _same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("graphed", [False, True], ids=["eager", "graphed"])
def test_nonfinite_step_is_skipped(graphed):
    case = "cnp_distractor_max"
    good = _batches(case, 4)
    bad = _nan_batch(good[0])                    # the shape of good[0]: already captured when it arrives
    kw = dict(max_grad_norm=1.0, skip_nonfinite=True)
    model, opt, g, step = _fresh(case, graphed, **kw)
    losses = [step(good[0]), step(good[1])]
    before = _state(opt)
    step(bad)
    torch.cuda.synchronize()
    assert not torch.isfinite(opt.grad_norm)
    assert _same(_state(opt), before) and int(opt.skipped_steps) == 1 and int(opt.t_dev) == 2
    losses += [step(good[2]), step(good[3])]
    got = _state(opt)

    _, ref, _, rstep = _fresh(case, graphed, **kw)
    ref_losses = [rstep(b) for b in good]
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(losses, ref_losses))
    assert _same(got, _state(ref)) and int(ref.skipped_steps) == 0 and int(opt.skipped_steps) == 1


def test_nonfinite_step_propagates_without_skipping():
    case = "cnp_distractor_max"
    _, opt, _, step = _fresh(case, False, max_grad_norm=1.0)
    step(_nan_batch(_batches(case, 1)[0]))
    torch.cuda.synchronize()
    assert not torch.isfinite(opt.flat.flat[:opt.flat.n_live]).all() and int(opt.t_dev) == 1


def test_scheduled_clipped_checkpoint_crosses_to_torch_adam_and_back():
    case = "cnp_distractor_max"
    model, opt, _, step = _fresh(case, False, max_grad_norm=0.5)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, _schedule)
    for b in _batches(case, 3):
        step(b)
        sched.step()
    sd = opt.state_dict()
    assert isinstance(sd["param_groups"][0]["lr"], float) and sd["param_groups"][0]["initial_lr"] == LR
    topt = torch.optim.Adam(model.parameters(), lr=0.5)
    topt.load_state_dict(sd)
    assert topt.param_groups[0]["lr"] == opt.lr and topt.param_groups[0]["initial_lr"] == LR
    _, back, _, _ = _fresh(case, False)
    back.load_state_dict(copy.deepcopy(topt.state_dict()))
    assert back.lr == opt.lr and back.param_groups[0]["initial_lr"] == LR
    assert float(back.param_groups[0].lr_dev) == float(opt.param_groups[0].lr_dev)
    assert torch.equal(back.m, opt.m) and torch.equal(back.v, opt.v) and int(back.t_dev) == 3


@pytest.mark.parametrize("graphed", [False, True], ids=["eager", "graphed"])
def test_resume_with_scheduler_is_bit_exact(graphed, tmp_path):
    case = "anp_distractor"
    batches = _batches(case, 6)
    kw = dict(max_grad_norm=0.5, skip_nonfinite=True)

    def run(resume_at=None):
        model, opt, g, step = _fresh(case, graphed, **kw)
        sched = torch.optim.lr_scheduler.LambdaLR(opt, _schedule)
        losses = []
        for i, b in enumerate(batches):
            if i == resume_at:
                state = g.state_dict() if g else {"model": model.state_dict(), "optimizer": opt.state_dict()}
                torch.save({"train": state, "scheduler": sched.state_dict()}, tmp_path / "ckpt.pt")
                model, opt, g, step = _fresh(case, graphed, **kw)
                if g:
                    step(batches[0]), step(batches[1])       # load over captured graphs
                sched = torch.optim.lr_scheduler.LambdaLR(opt, _schedule)
                sd = torch.load(tmp_path / "ckpt.pt", weights_only=False)
                if g:
                    g.load_state_dict(sd["train"])
                else:
                    model.load_state_dict(sd["train"]["model"])
                    opt.load_state_dict(sd["train"]["optimizer"])
                sched.load_state_dict(sd["scheduler"])
            losses.append(step(b))
            sched.step()
        torch.cuda.synchronize()
        return losses, opt

    ref_losses, ref = run()
    losses, opt = run(resume_at=3)
    assert all(torch.equal(a, b) for a, b in zip(losses, ref_losses))
    assert _same(_state(opt), _state(ref)) and opt.lr == ref.lr
    assert float(opt.param_groups[0].lr_dev) == float(ref.param_groups[0].lr_dev)


# ------------------------------------------------------------------------------------------------
# two GPUs
# ------------------------------------------------------------------------------------------------
_WORKER = r"""
import math, os, sys, torch, torch.distributed as td
ROOT = sys.argv[1]
sys.path[:0] = [ROOT, os.path.join(ROOT, "what-matters-for-meta-learning_b200"), os.path.join(ROOT, "tests")]
from conftest import make_config
from b200np import dist, engine
from b200np.optim import FlatParams, FusedAdam
from networks.ANPDistractor import ANPDistractor
from oracle import synth
from trainer.losses import LossFunc
rank = int(os.environ["RANK"]); dev = torch.device(f"cuda:{int(os.environ['LOCAL_RANK'])}")
torch.cuda.set_device(dev)
td.init_process_group("nccl", device_id=dev)
engine.set_precision("tf32x3")
T, nc, nt, W = 4, 3, 4, td.get_world_size()
batch = [torch.from_numpy(a).to(dev) for a in synth.task_batch("distractor", T, nc, nt, seed=5)]
lossf = LossFunc("mse", "distractor")
lo, hi = dist.shard_tasks(T)
def train(tasks, batches, max_norm):
    torch.manual_seed(0)
    model = ANPDistractor(make_config("ANPDistractor", "distractor", tasks, "attention", "max", device=str(dev),
                                      dim_w=16)).to(dev)
    opt = FusedAdam(FlatParams(model), lr=1e-3, max_grad_norm=max_norm, skip_nonfinite=True)
    out = []
    for b in batches:
        opt.zero_grad()
        mu, _, _ = model(b[0], b[1], b[2]); lossf.calc_loss(mu, None, b[3]).backward(); opt.step()
        torch.cuda.synchronize()
        out.append((opt.flat.flat.clone(), opt.m.clone(), float(opt.grad_norm), int(opt.skipped_steps)))
    return out
# the whole batch on this GPU, no exchange: the reference, and the clip threshold (half the first step's norm)
saved = dist.world_size
dist.world_size = lambda: 1
full = train(T, [batch], 1e30)
c = full[0][2] / 2
full = train(T, [batch], c)
dist.world_size = saved
shard = [t[lo:hi].contiguous() for t in batch]
bad = [t.clone() for t in shard]
if rank == 1:
    bad[0][0] = float("nan")                       # only rank 1 sees the NaN: the all-reduce carries it to rank 0
got = train(T // W, [shard, bad], c)
(w1, m1, n1, s1), (w2, m2, n2, s2) = got
allw = [torch.empty_like(w2) for _ in range(W)]
td.all_gather(allw, w2)
assert all(torch.equal(allw[0], a) for a in allw), "weights differ across ranks"
assert n1 > c and s1 == 0 and s2 == 1 and not math.isfinite(n2), (n1, c, s1, s2, n2)
assert torch.equal(w1, w2), "the skipped step changed the weights"
err_norm = abs(n1 - full[0][2]) / full[0][2]
err_m = float((m1 - full[0][1]).norm() / full[0][1].norm())
if rank == 0:
    print(f"RESULT clip={c:.4e} norm_rel_err={err_norm:.3e} clipped_m_rel_err={err_m:.3e}", flush=True)
assert err_norm < 1e-4 and err_m < 1e-4, (err_norm, err_m)
td.barrier()
td.destroy_process_group()
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_clip_and_skip_agree_across_ranks(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29651", str(script), ROOT]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "RESULT" in out.stdout, out.stdout[-3000:]
    print("\n".join(l for l in out.stdout.splitlines() if l.startswith("RESULT")))
