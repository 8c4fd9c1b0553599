"""Gradient accumulation on the fused training path: `FusedAdam(accumulate_steps=k)`, `no_sync()`, and `GraphedStep`
with one call per micro-batch.

`b200np_multi_accumulate` is checked against torch with guard bands, alignment and tail classes, more than 64
segments, null sources and a bitwise repeat.  `accumulate_steps=1` launches the kernels of the plain step and gives
its bits, eagerly and under graphs.  k equal-shaped CNP micro-batches follow one k-times larger batch and
torch.optim.Adam in fp64 fed the mean gradient, with and without clipping.  The graphed window equals the eager
`no_sync()` window bit for bit, mixed shapes capture once per (shape, role) and never synchronise, a NaN micro-batch
skips its whole window, schedulers step once per window, checkpoints between windows resume bit for bit and are
refused inside one, and a capture mid-window changes nothing.  On two GPUs the window costs one gradient exchange.
"""
import contextlib
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


def _kernels(fn):
    """Names of the CUDA kernels `fn` launches, without their signatures."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name.split("(")[0].replace("void ", "") for e in prof.events()
            if e.device_type == torch.autograd.DeviceType.CUDA]


# ------------------------------------------------------------------------------------------------
# the kernel
# ------------------------------------------------------------------------------------------------
GUARD = 64     # floats of NaN guard band around every buffer


def _segment_specs():
    """(numel, source offset, destination offset mod 4): float4 bodies with 0-3 element scalar tails, sources and
    destinations off 16-byte alignment, an empty segment, grid-stride lengths, and 150 segments in all (3 launches)."""
    specs = [(0, 0, 0), (1, 0, 0), (3, 0, 0), (4, 0, 0), (5, 0, 0), (4096, 0, 0), (4099, 0, 0), (4098, 1, 0),
             (4097, 0, 1), (4100, 2, 3), (300_001, 0, 0), (262_144, 3, 0), (1023, 0, 2)]
    specs += [(37 + 4 * i + i % 4, (i % 5 == 0) * (1 + i % 3), (i % 7 == 0) * 2) for i in range(150 - len(specs))]
    return specs


def _segments(seed):
    """Guarded sources (every 9th one None) and the destination offsets of `_segment_specs`, past a leading guard."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    segs, bufs, cursor = [], [], GUARD
    for j, (n, soff, dmod) in enumerate(_segment_specs()):
        off = (cursor + 3) // 4 * 4 + dmod
        cursor = off + n + 1
        if j % 9 == 4:
            segs.append((None, off, n))
            continue
        buf = torch.full((GUARD + soff + n + GUARD,), float("nan"), device="cuda")
        buf[GUARD + soff:GUARD + soff + n] = torch.randn(n, device="cuda", generator=gen)
        bufs.append(buf)
        segs.append((buf[GUARD + soff:GUARD + soff + n], off, n))
    dst = torch.randn(cursor + GUARD, device="cuda", generator=gen)
    dst[:GUARD] = float("nan")
    dst[cursor:] = float("nan")
    return segs, bufs, dst


def _bits(t):
    return t.view(torch.int32)


def test_multi_accumulate_matches_torch():
    from b200np import ops
    segs, bufs, dst0 = _segments(1)
    assert len(segs) > 128 and any(s is None for s, _, _ in segs)
    assert {(o % 4, s.data_ptr() % 16 if s is not None else 0) for s, o, _ in segs} >= {(0, 0), (1, 0), (2, 0), (0, 4)}
    want = dst0.clone()
    for s, off, n in segs:
        if s is not None:
            want[off:off + n] += s           # torch's fp32 add: the same single rounding per element
    src_before = [b.clone() for b in bufs]
    outs = []
    for _ in range(2):
        dst = dst0.clone()
        names = _kernels(lambda: ops.multi_accumulate(dst, segs))
        assert names == ["multi_accumulate_kernel"] * 3, names
        outs.append(dst)
    assert torch.equal(_bits(outs[0]), _bits(want))   # guards, gaps, null segments and sums, bit for bit
    assert torch.equal(_bits(outs[1]), _bits(outs[0]))
    assert all(torch.equal(_bits(a), _bits(b)) for a, b in zip(bufs, src_before))


def test_multi_copy_keeps_its_kernel_and_zero_fill():
    from b200np import ops
    segs, _, dst0 = _segments(2)
    want = dst0.clone()
    for s, off, n in segs:
        want[off:off + n] = 0.0 if s is None else s
    dst = dst0.clone()
    assert _kernels(lambda: ops.multi_copy(dst, segs)) == ["multi_copy_kernel"] * 3
    assert torch.equal(_bits(dst), _bits(want))


# ------------------------------------------------------------------------------------------------
# the product models
# ------------------------------------------------------------------------------------------------
def _model(case, T=None):
    from b200np import engine
    engine.set_precision("tf32x3")
    model, _ = build_product_model(case, device="cuda", T=T)
    return model.to("cuda")


def _batches(case, n, seed=90, ncs=None, T=None):
    """`n` batches; `ncs`: the context size of each (default: the case's)."""
    method, task, agg, img_agg, extra, T0, nc, nt = CASES[case]
    ncs = ncs or [nc] * n
    return [[torch.from_numpy(a).cuda() for a in synth.task_batch(task, T or T0, c, nt, seed=seed + i)]
            for i, c in enumerate(ncs)]


def _lossf(case):
    from trainer.losses import LossFunc
    return LossFunc("mse", CASES[case][1])


def _fwd_bwd(model, lossf, b):
    mu, _, _ = model(b[0], b[1], b[2])
    loss = lossf.calc_loss(mu, None, b[3])
    loss.backward()
    return loss.detach().clone()


def _eager_window(opt, model, lossf, window):
    """The eager recipe: every backward pass but the last inside no_sync(), then one step."""
    opt.zero_grad()
    losses = []
    for i, b in enumerate(window):
        with opt.no_sync() if i < len(window) - 1 else contextlib.nullcontext():
            losses.append(_fwd_bwd(model, lossf, b))
    opt.step()
    return losses


class Run:
    """A model, its FusedAdam(accumulate_steps=k) and, graphed, its GraphedStep; `call(batch)` is one micro-batch."""

    def __init__(self, case, k, graphed, **kw):
        from b200np.optim import FlatParams, FusedAdam, GraphedStep
        self.model, self.lossf, self.k = _model(case), _lossf(case), k
        self.opt = FusedAdam(FlatParams(self.model), lr=LR, accumulate_steps=k, **kw)
        self.g = GraphedStep(self.model, self.lossf, self.opt, warmup=1) if graphed else None
        self._window = []

    def call(self, b):
        if self.g is not None:
            return [self.g(b).clone()]
        self._window.append(b)
        if len(self._window) < self.k:
            return []
        w, self._window = self._window, []
        return _eager_window(self.opt, self.model, self.lossf, w)

    def run(self, batches):
        losses = []
        for b in batches:
            losses += self.call(b)
        torch.cuda.synchronize()
        return losses

    def state(self):
        o = self.opt
        return (o.flat.flat.clone(), o.m.clone(), o.v.clone(), o.t_dev.clone(), o.skipped_steps.clone())


def _same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


def test_one_step_window_is_the_plain_step():
    """accumulate_steps=1 (explicit) against the default optimizer: the same kernels in the same order and the same
    bits eagerly; under graphs one "last" graph per shape and the eager bits."""
    from b200np.optim import FlatParams, FusedAdam
    case = "anp_distractor"
    batches = _batches(case, 4, ncs=[3, 5, 3, 5])
    lossf = _lossf(case)
    runs, kernels = [], []
    for k in (None, 1):
        model = _model(case)
        opt = FusedAdam(FlatParams(model), lr=LR, **({} if k is None else {"accumulate_steps": k}))
        for i, b in enumerate(batches):
            opt.zero_grad()
            _fwd_bwd(model, lossf, b)
            if i == 3:
                kernels.append(_kernels(opt.step))
            else:
                opt.step()
        torch.cuda.synchronize()
        runs.append((opt.flat.flat.clone(), opt.m.clone(), opt.v.clone(), opt.t_dev.clone()))
    assert kernels[0] == kernels[1], kernels
    assert "multi_accumulate_kernel" not in kernels[1] and "multi_copy_kernel" in kernels[1]
    assert _same(runs[0], runs[1])
    g = Run(case, 1, graphed=True)
    g.run(batches)
    assert [set(e["roles"]) for e in g.g.cache.values()] == [{"last"}, {"last"}]
    assert _same(g.state()[:4], runs[1])


@pytest.mark.parametrize("clip", [False, True], ids=["noclip", "clip"])
def test_accumulated_cnp_matches_big_batch_and_torch_fp64(clip):
    """CNPDistractor (mean aggregation), windows of k = 3 micro-batches of T = 2 tasks.  (a) The window's mean gradient
    equals the gradient of the same model built for T = 6 on the concatenated batch, at the same weights, up to fp32
    rounding.  (b) The update follows torch.optim.Adam over fp64 copies of the parameters fed that mean gradient (with
    clip_grad_norm_ where clipping is on), and `grad_norm` is its norm.  The two together are the big-batch step: the
    updates themselves are not compared with the big batch's, because Adam's first steps move every element by about
    lr * sign(g), so rounding noise on gradients near zero shows up at full size there."""
    from b200np.optim import FlatParams, FusedAdam
    case, k, windows = "cnp_distractor_mean", 3, 4
    lossf = _lossf(case)
    small = _model(case)
    big = _model(case, T=2 * k)
    names = [n for n, _ in small.named_parameters()]
    w0 = {n: p.detach().double().clone() for n, p in small.named_parameters()}
    ref = [p.detach().double().clone().requires_grad_() for p in small.parameters()]
    # loss scales alternate so that a clip threshold between them clips some windows and not others
    scales = [40.0 if w % 2 else 0.05 for w in range(windows)]
    micro = [_batches(case, k, seed=300 + 10 * w) for w in range(windows)]
    cat = [[torch.cat([m[j] for m in mb]) for j in range(4)] for mb in micro]
    c = None
    if clip:
        _fwd_bwd(small, lossf, micro[0][0])
        c = 3.0 * float(torch.nn.utils.get_total_norm([p.grad for p in small.parameters() if p.grad is not None]))
        small.zero_grad(set_to_none=True)
    opt = FusedAdam(FlatParams(small), lr=LR, accumulate_steps=k, max_grad_norm=c if clip else 1e30)
    topt = torch.optim.Adam(ref, lr=LR)
    clipped, grad_errs = [], []
    for w in range(windows):
        s = scales[w]
        opt.zero_grad()
        for i, b in enumerate(micro[w]):
            with opt.no_sync() if i < k - 1 else contextlib.nullcontext():
                mu, _, _ = small(b[0], b[1], b[2])
                (s * lossf.calc_loss(mu, None, b[3])).backward()
        mean = [None if p.grad is None else p.grad.detach().double() / k for p in small.parameters()]
        want_norm = float(torch.nn.utils.get_total_norm([g for g in mean if g is not None]))
        big.load_state_dict(small.state_dict())
        big.zero_grad(set_to_none=True)
        mu, _, _ = big(cat[w][0], cat[w][1], cat[w][2])
        (s * lossf.calc_loss(mu, None, cat[w][3])).backward()
        pairs = [(g, q.grad.double()) for g, q in zip(mean, big.parameters()) if g is not None]
        grad_errs.append(float(sum((g - h).pow(2).sum() for g, h in pairs) ** 0.5
                               / sum(h.pow(2).sum() for _, h in pairs) ** 0.5))
        opt.step()
        assert abs(float(opt.grad_norm) - want_norm) <= 1e-6 * want_norm, (float(opt.grad_norm), want_norm)
        for q, g in zip(ref, mean):
            q.grad = g
        if clip:
            clipped.append(float(torch.nn.utils.clip_grad_norm_(ref, c)) > c)
        topt.step()
    torch.cuda.synchronize()
    if clip:
        assert any(clipped) and not all(clipped), clipped
    num = den = 0.0
    for (n, p), q in zip(small.named_parameters(), ref):
        num += float(((p.detach().double() - w0[n]) - (q.detach() - w0[n])).pow(2).sum())
        den += float((q.detach() - w0[n]).pow(2).sum())
    e_torch = (num / den) ** 0.5
    print(f"\n[cnp mean k={k} {'clip' if clip else 'noclip'}] relative update error vs torch fp64 {e_torch:.2e}; "
          "mean gradient vs the 6-task batch's, per window: " + ", ".join(f"{e:.2e}" for e in grad_errs))
    assert e_torch <= 1e-5 and max(grad_errs) <= 1e-5, (e_torch, grad_errs)
    assert int(opt.t_dev) == windows and opt.t == windows


@pytest.mark.parametrize("case", ["anp_distractor", "cnp_distractor_max"])
def test_graphed_window_equals_eager_no_sync_window(case):
    """k = 3 under GraphedStep against the eager no_sync() recipe, bit for bit: both sum g1 + g2 + g3 in that order.
    The windows mix two shapes."""
    batches = _batches(case, 9, ncs=[3, 5, 3, 5, 5, 3, 3, 3, 5])
    eager, graphed = Run(case, 3, graphed=False), Run(case, 3, graphed=True)
    le, lg = eager.run(batches), graphed.run(batches)
    assert all(torch.equal(a, b) for a, b in zip(le, lg)) and len(lg) == 9
    assert _same(eager.state(), graphed.state()) and int(graphed.opt.t_dev) == 3 and graphed.opt.t == 3
    assert torch.equal(eager.opt.flat.grad, graphed.opt.flat.grad)          # the last window's summed gradient


@pytest.fixture
def captures(monkeypatch):
    from b200np.optim import GraphedStep
    out = []
    real = GraphedStep._capture
    monkeypatch.setattr(GraphedStep, "_capture", lambda self, ent: (out.append(ent["role"]), real(self, ent)))
    return out


def test_mixed_shapes_capture_once_per_shape_and_role(captures):
    """ANPDistractor with a different `shot` per micro-batch: every (shape, role) pair is captured once, later windows
    replay without capturing or synchronising, and the result equals the eager recipe."""
    case, k = "anp_distractor", 3
    ncs = [1, 2, 3, 2, 3, 1, 3, 1, 2] + [2, 1, 3, 3, 2, 1]
    batches = _batches(case, len(ncs), ncs=ncs)
    g = Run(case, k, graphed=True)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        warnings.filterwarnings("ignore", message="Synchronization debug mode is a prototype")  # torch's own notice
        for i, b in enumerate(batches):
            torch.cuda.set_sync_debug_mode("error" if i >= 9 else "default")
            try:
                g.call(b)
            finally:
                torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert sorted(captures) == sorted(["first", "middle", "last"] * 3), captures
    assert all(set(e["roles"]) == {"first", "middle", "last"} for e in g.g.cache.values()) and len(g.g.cache) == 3
    e = Run(case, k, graphed=False)
    e.run(batches)
    assert _same(e.state(), g.state()) and int(g.opt.t_dev) == len(ncs) // k


def _nan_batch(batch):
    bad = [t.clone() for t in batch]
    bad[0][0] = float("nan")                       # the first context image of the first task
    return bad


@pytest.mark.parametrize("graphed", [False, True], ids=["eager", "graphed"])
def test_nan_in_the_middle_micro_batch_skips_the_window(graphed):
    case, k = "cnp_distractor_max", 3
    kw = dict(max_grad_norm=1.0, skip_nonfinite=True)
    good = _batches(case, 2 * k)
    bad = good[:1] + [_nan_batch(good[1])] + good[2:3]
    r = Run(case, k, graphed, **kw)
    r.run(good[:k])
    before = r.state()
    r.run(bad)
    assert not torch.isfinite(r.opt.grad_norm)
    after = r.state()
    assert _same(after[:4], before[:4]) and int(r.opt.skipped_steps) == 1 and int(r.opt.t_dev) == 1
    r.run(good[k:])
    ref = Run(case, k, graphed, **kw)
    ref.run(good)
    assert _same(r.state()[:4], ref.state()[:4]) and int(ref.opt.skipped_steps) == 0


def test_lambda_lr_steps_once_per_window_under_graphs():
    case, k = "cnp_distractor_max", 3
    lam = lambda s: 1.0 / (1 + 0.5 * s)
    batches = _batches(case, 4 * k, ncs=[3, 5, 3] * 4)
    out = []
    for graphed in (False, True):
        r = Run(case, k, graphed)
        sched = torch.optim.lr_scheduler.LambdaLR(r.opt, lam)
        lrs = []
        with warnings.catch_warnings():
            warnings.simplefilter("error")
            for i, b in enumerate(batches):
                r.call(b)
                if i % k == k - 1:
                    sched.step()
                    lrs.append(r.opt.lr)
        torch.cuda.synchronize()
        out.append((lrs, r.state()))
    assert out[0][0] == out[1][0] == [LR * lam(s) for s in range(1, 5)]
    assert _same(out[0][1], out[1][1])


def test_graphed_accumulated_resume_is_bit_exact_and_mid_window_checkpoints_raise(tmp_path):
    case, k = "anp_distractor", 2
    kw = dict(max_grad_norm=0.5, skip_nonfinite=True)
    batches = _batches(case, 4 * k, ncs=[3, 5] * 4)
    lam = lambda s: 0.7 ** s

    def run(resume_at=None):
        r = Run(case, k, True, **kw)
        sched = torch.optim.lr_scheduler.LambdaLR(r.opt, lam)
        losses = []
        for i, b in enumerate(batches):
            if i == resume_at:
                torch.save({"train": r.g.state_dict(), "sched": sched.state_dict()}, tmp_path / "ckpt.pt")
                r = Run(case, k, True, **kw)
                r.run(batches[:k])                     # load over captured graphs
                sched = torch.optim.lr_scheduler.LambdaLR(r.opt, lam)
                ck = torch.load(tmp_path / "ckpt.pt", weights_only=False)
                r.g.load_state_dict(ck["train"])
                sched.load_state_dict(ck["sched"])
            losses += r.call(b)
            if i % k == 0:                             # mid-window: neither saving nor loading is allowed
                with pytest.raises(RuntimeError, match="accumulation window"):
                    r.g.state_dict()
                with pytest.raises(RuntimeError, match="accumulation window"):
                    r.opt.load_state_dict({"state": {}, "param_groups": []})
            else:
                sched.step()
        torch.cuda.synchronize()
        return losses, r

    ref_losses, ref = run()
    losses, r = run(resume_at=2 * k)
    assert all(torch.equal(a, b) for a, b in zip(losses, ref_losses))
    assert _same(r.state(), ref.state()) and r.opt.lr == ref.opt.lr and int(r.opt.t_dev) == 4


def test_eager_mid_window_state_dict_raises():
    case = "cnp_distractor_max"
    r = Run(case, 2, graphed=False)
    b = _batches(case, 2)
    r.opt.zero_grad()
    with r.opt.no_sync():
        _fwd_bwd(r.model, r.lossf, b[0])
    with pytest.raises(RuntimeError, match="accumulation window"):
        r.opt.state_dict()
    _fwd_bwd(r.model, r.lossf, b[1])
    r.opt.step()
    assert sorted(r.opt.state_dict()["state"]) == sorted(r.opt.flat.live_index)


def test_new_shape_mid_window_changes_nothing(captures):
    """A shape first met in the middle of a window (here through prefetch) is captured without touching the window's
    summed gradient, the weights, the moments, the counters or the window position; the run still equals eager."""
    case, k = "anp_distractor", 3
    batches = _batches(case, 2 * k, ncs=[3, 3, 5, 3, 5, 5])
    g = Run(case, k, graphed=True)
    g.call(batches[0])
    g.call(batches[1])
    torch.cuda.synchronize()
    opt = g.opt
    before = g.state() + (opt.flat.grad.clone(), opt.grad_norm.clone())
    n_before = len(captures)
    g.g.prefetch(batches[2])                         # new shape, captured as this window's "last"
    torch.cuda.synchronize()
    assert captures[n_before:] == ["last"]
    assert _same(g.state() + (opt.flat.grad, opt.grad_norm), before) and opt._micro == 2 and opt.t == 0
    g.call(batches[2])
    for b in batches[3:]:
        g.call(b)
    torch.cuda.synchronize()
    e = Run(case, k, graphed=False)
    e.run(batches)
    assert _same(e.state(), g.state())


# ------------------------------------------------------------------------------------------------
# two GPUs
# ------------------------------------------------------------------------------------------------
_WORKER = r"""
import os, sys, torch, torch.distributed as td
ROOT, OUT = sys.argv[1], sys.argv[2]
sys.path[:0] = [ROOT, os.path.join(ROOT, "what-matters-for-meta-learning_b200"), os.path.join(ROOT, "tests")]
from conftest import build_product_model
from b200np import dist, engine
from b200np.optim import FlatParams, FusedAdam
from test_gpu_optim_accumulate import _batches, _lossf, _fwd_bwd
rank = int(os.environ["RANK"]); dev = torch.device(f"cuda:{int(os.environ['LOCAL_RANK'])}")
torch.cuda.set_device(dev)
td.init_process_group("nccl", device_id=dev)
engine.set_precision("tf32x3")
case, T, k, W, windows = "cnp_distractor_mean", 4, 2, td.get_world_size(), 3
per = T // (W * k)
model, _ = build_product_model(case, device=str(dev), T=per)
model = model.to(dev)
lossf = _lossf(case)
opt = FusedAdam(FlatParams(model), lr=1e-3, accumulate_steps=k, max_grad_norm=1e30)
calls, real = [], dist.all_reduce_sum
def counting(t):
    if t.untyped_storage().data_ptr() == opt.flat.grad.untyped_storage().data_ptr():
        calls.append(t.numel())
    return real(t)
dist.all_reduce_sum = counting
per_window = []
for w in range(windows):
    full = [t.to(dev) for t in _batches(case, 1, seed=500 + w, T=T)[0]]
    opt.zero_grad()
    n0 = len(calls)
    for i in range(k):
        lo = (rank * k + i) * per
        b = [t[lo:lo + per].contiguous() for t in full]
        if i < k - 1:
            with opt.no_sync():
                _fwd_bwd(model, lossf, b)
            assert len(calls) == n0, "an exchange started inside no_sync()"
        else:
            _fwd_bwd(model, lossf, b)
    opt.step()
    per_window.append(len(calls) - n0)
torch.cuda.synchronize()
w_ = opt.flat.flat
allw = [torch.empty_like(w_) for _ in range(W)]
td.all_gather(allw, w_)
assert all(torch.equal(allw[0], a) for a in allw), "weights differ across ranks"
assert int(opt.t_dev) == windows
# a second backward pass outside no_sync() would miss the exchange the first one started
opt.zero_grad()
b = [t.to(dev)[:per].contiguous() for t in _batches(case, 1, seed=900, T=T)[0]]
_fwd_bwd(model, lossf, b)
try:
    _fwd_bwd(model, lossf, b)
    raised = False
except RuntimeError as e:
    raised = "no_sync" in str(e)
assert raised, "a second backward outside no_sync() did not raise"
torch.cuda.synchronize()
if rank == 0:
    torch.save({"flat": allw[0].cpu(), "per_window": per_window}, OUT)
    print(f"RESULT ranks={W} gradient all-reduce calls per window={per_window}", flush=True)
td.barrier()
td.destroy_process_group()
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_accumulation_matches_full_batch_with_one_exchange_per_window(tmp_path):
    script, out = tmp_path / "worker.py", tmp_path / "out.pt"
    script.write_text(_WORKER)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29657", str(script), ROOT, str(out)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    print("\n".join(l for l in res.stdout.splitlines() if l.startswith("RESULT")))
    got = torch.load(out)
    # the same three 4-task batches on one GPU, one step each
    from b200np.optim import FlatParams, FusedAdam
    case = "cnp_distractor_mean"
    model, lossf = _model(case, T=4), _lossf(case)
    w0 = {n: p.detach().double().clone() for n, p in model.named_parameters()}
    opt = FusedAdam(FlatParams(model), lr=1e-3, max_grad_norm=1e30)    # the workers' flat layout: independent of T
    for w in range(3):
        opt.zero_grad()
        _fwd_bwd(model, lossf, _batches(case, 1, seed=500 + w, T=4)[0])
        opt.step()
    torch.cuda.synchronize()
    assert opt.flat.flat.numel() == got["flat"].numel()
    num = den = 0.0
    for n, p, off, k in opt.flat.live:
        two = got["flat"][off:off + k].double().view_as(p).cuda()
        num += float(((two - w0[n]) - (p.detach().double() - w0[n])).pow(2).sum())
        den += float((p.detach().double() - w0[n]).pow(2).sum())
    e = (num / den) ** 0.5
    print(f"[2 GPUs, k=2] relative update error against the 4-task batch on one GPU: {e:.2e}")
    assert e <= 1e-5, e
    assert got["per_window"] == [got["per_window"][0]] * 3 and 1 <= got["per_window"][0] <= 2
