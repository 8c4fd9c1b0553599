"""Parameter groups and decoupled weight decay (AdamW) on the fused training path.

Groups carrying identical hyperparameters are bit-identical to the single group, and a parameter in no group stays
bit-identical while its neighbours in the flat buffer move.  Decay / no-decay / own-lr groups under per-group
schedules and clipping follow torch.optim.Adam / AdamW in fp64, fed the same gradients.  Under CUDA graphs, per-group
schedules (OneCycleLR with cycle_momentum=True included) and assignments to betas / weight_decay capture once per
shape and never synchronise.  Multi-group checkpoints cross to torch and back, resume bit for bit, and are refused
without side effects when they do not fit.  Two ranks stay bit-identical.
"""
import copy
import os
import subprocess
import sys
import warnings

import pytest
import torch

from conftest import CASES, build_product_model, rel_l2
from oracle import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LR, WD = 1e-3, 0.05


def _mlp(dtype=torch.float32):
    torch.manual_seed(11)
    return torch.nn.Sequential(torch.nn.Linear(13, 64), torch.nn.Tanh(), torch.nn.Linear(64, 31), torch.nn.Tanh(),
                               torch.nn.Linear(31, 5)).to("cuda", dtype)


def _product(case):
    from b200np import engine
    engine.set_precision("tf32x3")
    model, _ = build_product_model(case, device="cuda")
    return model.to("cuda")


def _groups(params_by_name, wd=WD, trunk_lr=LR / 3):
    """Decay on weights, none on biases, and the CNN trunks' weights (the MLP: its last layer) with their own lr."""
    from b200np.optim import FlatParams
    named = list(params_by_name)
    own = [n for n, p in named if p.dim() > 1 and n.startswith(FlatParams.LATE)] or [named[-2][0]]
    return [{"params": [p for n, p in named if p.dim() > 1 and n not in own], "weight_decay": wd},
            {"params": [p for n, p in named if p.dim() <= 1], "weight_decay": 0.0},
            {"params": [p for n, p in named if n in own], "weight_decay": wd, "lr": trunk_lr}]


def _state(opt):
    return (opt.flat.flat.clone(), opt.m.clone(), opt.v.clone(), opt.t_dev.clone())


def _same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


def _table(opt):
    return opt._table.clone(), [dict((k, v) for k, v in g.items() if k != "params") for g in opt.param_groups]


# ------------------------------------------------------------------------------------------------
# bitwise equivalences
# ------------------------------------------------------------------------------------------------
def _feed(opts, n, steps=5, seed=3):
    """The same gradients, spanning several decades, into every optimizer for `steps` steps."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    for i in range(steps):
        g = torch.randn(n, device="cuda", generator=gen) * (10.0 ** (i - 2))
        for opt in opts:
            opt.zero_grad()
            opt.flat.attach_grads()
            opt.flat.grad.copy_(g)
            opt.step()
    torch.cuda.synchronize()


@pytest.mark.parametrize("wd", [0.0, 0.01])
def test_identical_groups_are_bit_identical_to_one_group(wd):
    from b200np.optim import FlatParams, FusedAdam
    one = FusedAdam(FlatParams(_mlp()), lr=LR, weight_decay=wd)
    model = _mlp()
    ps = list(model.parameters())
    # weights and biases alternate in the flat layout: one run per parameter
    groups = [{"params": ps[0::2]}, {"params": ps[1::2][:2]}, {"params": ps[1::2][2:]}]
    many = FusedAdam(FlatParams(model), lr=LR, weight_decay=wd, param_groups=groups)
    assert many._run_group.numel() == len(ps)
    _feed([one, many], one.flat.n_live)
    assert _same(_state(many), _state(one)) and int(many.t_dev) == 5


def test_frozen_parameters_stay_bit_identical():
    from b200np.optim import FlatParams, FusedAdam
    model = _mlp()
    ps = list(model.parameters())
    frozen = {2, 3}                                  # the middle layer, between two trained ones
    flat = FlatParams(model)
    opt = FusedAdam(flat, lr=LR, weight_decay=0.1, decoupled_weight_decay=True,
                    param_groups=[{"params": [p for i, p in enumerate(ps) if i not in frozen]}])
    w0 = flat.flat.clone()
    _feed([opt], flat.n_live)
    for i, (name, p, off, k) in zip(flat.live_index, flat.live):
        pad = (k + 3) // 4 * 4
        if i in frozen:
            assert torch.equal(flat.flat[off:off + pad], w0[off:off + pad]), name
            assert not opt.m[off:off + pad].any() and not opt.v[off:off + pad].any(), name
        else:
            assert (flat.flat[off:off + k] != w0[off:off + k]).all(), name
    assert sorted(opt.state_dict()["state"]) == [0, 1, 2, 3]       # ids over the group's params: no frozen entries


# ------------------------------------------------------------------------------------------------
# against torch in fp64
# ------------------------------------------------------------------------------------------------
def _lambdas():
    return [lambda k: 0.5 ** (k / 7) * (1 + (k % 3)), lambda k: 1.0 / (1 + 0.3 * k), lambda k: 1.0 + 0.1 * (k % 4)]


def _mlp_loss(model, b, s):
    x, y = b
    return s * ((model(x) - y) ** 2).mean()


def _scheduler(kind, opt, steps):
    if kind == "lambda":
        return torch.optim.lr_scheduler.LambdaLR(opt, _lambdas())
    return torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=[3e-3, 1e-3, 5e-4], total_steps=steps + 1,
                                               base_momentum=[0.8, 0.85, 0.7], max_momentum=[0.95, 0.9, 0.9],
                                               cycle_momentum=True)


def _assign(opt, what):
    """Change one hyperparameter of one group, in place; `what` None: all three below."""
    if what in (None, "weight_decay"):
        opt.param_groups[0]["weight_decay"] = 2 * WD
    if what in (None, "betas"):
        opt.param_groups[1]["betas"] = (0.8, 0.99)
    if what in (None, "decoupled_weight_decay"):
        opt.param_groups[2]["decoupled_weight_decay"] = not opt.param_groups[2]["decoupled_weight_decay"]


@pytest.mark.parametrize("kind", ["lambda", "onecycle"])
@pytest.mark.parametrize("decoupled", [False, True], ids=["adam", "adamw"])
@pytest.mark.parametrize("which", ["mlp", "cnp_distractor_max"])
def test_groups_match_torch_fp64(which, decoupled, kind):
    """The gradients of the fp32 model trained by FusedAdam feed torch.optim.Adam / AdamW over fp64 copies of the
    parameters, with the same groups, per-group schedules (LambdaLR, or OneCycleLR writing every group's betas),
    clip_grad_norm_, and mid-run assignments of weight_decay, betas and decoupled_weight_decay to single groups.
    Each group's update is checked on its own, so a hyperparameter that did not reach the device table fails."""
    from b200np.optim import FlatParams, FusedAdam
    from trainer.losses import LossFunc
    steps = 12
    gen = torch.Generator(device="cuda").manual_seed(5)
    scales = [50.0 if i % 2 else 0.05 for i in range(steps)]
    if which == "mlp":
        model = _mlp()
        data = [(torch.randn(32, 13, device="cuda", generator=gen), torch.randn(32, 5, device="cuda", generator=gen))
                for _ in range(steps)]
        loss_of = _mlp_loss
    else:
        model = _product(which)
        lossf = LossFunc("mse", CASES[which][1])
        data = _batches(which, steps)

        def loss_of(net, b, s):
            mu, _, _ = net(b[0], b[1], b[2])
            return s * lossf.calc_loss(mu, None, b[3])
    names = [n for n, _ in model.named_parameters()]
    ref = [p.detach().double().clone().requires_grad_() for p in model.parameters()]
    flat = FlatParams(model)
    w0 = [p.detach().double().clone() for p in ref]

    # the clip threshold lies between the norms of the two loss scales
    loss_of(model, data[0], 1.0).backward()
    c = float(torch.nn.utils.get_total_norm([p.grad for p in model.parameters() if p.grad is not None]))
    model.zero_grad(set_to_none=True)
    opt = FusedAdam(flat, lr=LR, decoupled_weight_decay=decoupled, max_grad_norm=c,
                    param_groups=_groups(model.named_parameters()))
    topt = (torch.optim.AdamW if decoupled else torch.optim.Adam)(
        [dict(g, params=[ref[names.index(n)] for n in _names(model, g)]) for g in _groups(model.named_parameters())],
        lr=LR, weight_decay=0.0)
    assert [bool(g["decoupled_weight_decay"]) for g in topt.param_groups] == [decoupled] * 3
    sched, tsched = _scheduler(kind, opt, steps), _scheduler(kind, topt, steps)
    clipped = []
    for i, (b, s) in enumerate(zip(data, scales)):
        if i == steps // 2:
            _assign(opt, None), _assign(topt, None)
        opt.zero_grad()
        loss_of(model, b, s).backward()
        grads = [None if p.grad is None else p.grad.detach().double().clone() for p in model.parameters()]
        opt.step()
        for q, g in zip(ref, grads):
            q.grad = g
        clipped.append(float(torch.nn.utils.clip_grad_norm_(ref, c)) > c)
        topt.step()
        sched.step(), tsched.step()
        for key in ("lr", "betas", "weight_decay", "decoupled_weight_decay"):
            assert [g[key] for g in opt.param_groups] == [g[key] for g in topt.param_groups], key
    assert any(clipped) and not all(clipped), clipped
    errs = []
    for g in _groups(model.named_parameters()):
        num = den = 0.0
        for n in _names(model, g):
            j = names.index(n)
            p, q, q0 = model.get_parameter(n), ref[j], w0[j]
            num += float(((p.detach().double() - q0) - (q.detach() - q0)).pow(2).sum())
            den += float((q.detach() - q0).pow(2).sum())
        errs.append((num / den) ** 0.5)
    print(f"\n[{which} {'adamw' if decoupled else 'adam'} {kind}] relative update error per group vs fp64: "
          + ", ".join(f"{e:.2e}" for e in errs))
    assert max(errs) < 2e-4, errs


def _names(model, group):
    ids = {id(p) for p in group["params"]}
    return [n for n, p in model.named_parameters() if id(p) in ids]


# ------------------------------------------------------------------------------------------------
# under graphs
# ------------------------------------------------------------------------------------------------
def _batches(case, n, seed=80):
    """`n` batches whose context size alternates between nc and nc + 2 (two graph shapes)."""
    method, task, agg, img_agg, extra, T, nc, nt = CASES[case]
    return [[torch.from_numpy(a).cuda() for a in synth.task_batch(task, T, nc + 2 * (i % 2), nt, seed=seed + i)]
            for i in range(n)]


def _fresh(case, graphed, **opt_kw):
    """(model, opt, GraphedStep or None, step(batch) -> loss clone), FusedAdam over `_groups`."""
    from b200np.optim import FlatParams, FusedAdam, GraphedStep
    from trainer.losses import LossFunc
    model = _product(case)
    opt = FusedAdam(FlatParams(model), lr=LR, param_groups=_groups(model.named_parameters()), **opt_kw)
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


@pytest.fixture
def captures(monkeypatch):
    from b200np.optim import GraphedStep
    out = []
    real = GraphedStep._capture
    monkeypatch.setattr(GraphedStep, "_capture", lambda self, ent: (out.append(1), real(self, ent)))
    return out


@pytest.mark.parametrize("case", ["anp_distractor", "cnp_distractor_max"])
def test_one_cycle_per_group_under_graphs(case, captures):
    steps = 8
    batches = _batches(case, steps)
    runs = []
    for graphed in (False, True):
        model, opt, g, step = _fresh(case, graphed, decoupled_weight_decay=True, max_grad_norm=0.5)
        sched = torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=[3e-3, 1e-3, 5e-4], total_steps=steps + 1,
                                                    base_momentum=[0.8, 0.85, 0.7], max_momentum=[0.95, 0.9, 0.9],
                                                    cycle_momentum=True)
        losses, hyper = [], []
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
                hyper.append([(gr["lr"], gr["betas"]) for gr in opt.param_groups])
        torch.cuda.synchronize()
        runs.append(([float(l) for l in losses], hyper, {k: v.clone() for k, v in model.state_dict().items()}))
    assert len(captures) == 2, captures                # one per shape, none for 8 x 3 groups' lr and betas changes
    (le, he, we), (lg, hg, wg) = runs
    assert he == hg and len({h[0][1] for h in he}) > 2
    assert le == pytest.approx(lg, rel=1e-6)
    for k in we:
        assert torch.allclose(we[k], wg[k], rtol=1e-5, atol=1e-7), k


@pytest.mark.parametrize("what", ["weight_decay", "betas", "decoupled_weight_decay"])
def test_assignment_between_replays_takes_effect(what, captures):
    """One hyperparameter of one group, assigned between replays, reaches the captured graphs without a recapture:
    the graphed run matches the eager run with the same assignment and differs from the run without it."""
    case = "cnp_distractor_max"
    batches = _batches(case, 5)

    def run(graphed, assign):
        model, opt, g, step = _fresh(case, graphed)
        for i, b in enumerate(batches):
            if i == 2 and assign:
                _assign(opt, what)
            step(b)
        torch.cuda.synchronize()
        return opt.flat.flat.clone(), opt.m.clone(), opt.v.clone()

    graphed = run(True, True)
    assert len(captures) == 2, captures
    eager, plain = run(False, True), run(False, False)
    for a, b in zip(graphed, eager):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-7)
    assert not torch.allclose(graphed[0], plain[0], rtol=1e-5, atol=1e-7)


# ------------------------------------------------------------------------------------------------
# checkpoints
# ------------------------------------------------------------------------------------------------
def _fwd_bwd(model, lossf, batch):
    cx, cy, tx, ty = batch
    mu, _, _ = model(cx, cy, tx)
    lossf.calc_loss(mu, None, ty).backward()


def _params(model):
    return {k: p.detach().clone() for k, p in model.named_parameters()}


def _assert_same_update(got, want):
    for k in want:
        e = rel_l2(got[k].double().cpu().numpy(), want[k].double().cpu().numpy())
        assert e <= 1e-6, (k, e)


def test_state_dict_structure_matches_torch_before_any_step():
    from b200np.optim import FlatParams, FusedAdam
    model = _product("cnp_distractor_max")
    flat = FlatParams(model)
    for decoupled in (False, True):
        groups = lambda: [dict(g, decoupled_weight_decay=decoupled) for g in _groups(model.named_parameters())]
        sd = FusedAdam(flat, lr=LR, param_groups=groups()).state_dict()
        assert sd == torch.optim.Adam(groups(), lr=LR).state_dict()
        assert sd == torch.optim.AdamW(groups(), lr=LR).state_dict()
        ids = [i for g in sd["param_groups"] for i in g["params"]]
        assert ids == list(range(len(ids)))
    # the constructor's value for keys the groups omit, as torch's defaults
    sd = FusedAdam(flat, lr=LR, weight_decay=0.01, decoupled_weight_decay=True,
                   param_groups=[{"params": g["params"]} for g in _groups(model.named_parameters())]).state_dict()
    assert sd == torch.optim.AdamW([{"params": g["params"]} for g in _groups(model.named_parameters())],
                                   lr=LR).state_dict()


@pytest.mark.parametrize("direction", ["torch_to_fused", "fused_to_torch"])
def test_multi_group_checkpoint_crosses_to_torch_and_back(direction):
    from b200np.optim import FlatParams, FusedAdam
    from trainer.losses import LossFunc
    model = _product("cnp_distractor_max")
    flat, lossf = FlatParams(model), LossFunc("mse", "distractor")
    batches = _batches("cnp_distractor_max", 4)
    make_torch = lambda lr: torch.optim.AdamW(_groups(model.named_parameters()), lr=lr)
    make_fused = lambda lr: FusedAdam(flat, lr=lr, decoupled_weight_decay=True,
                                      param_groups=_groups(model.named_parameters()))
    first, second = (make_torch, make_fused) if direction == "torch_to_fused" else (make_fused, make_torch)
    a = first(LR)
    sched = torch.optim.lr_scheduler.LambdaLR(a, _lambdas())
    for b in batches[:3]:
        a.zero_grad()
        _fwd_bwd(model, lossf, b)
        a.step()
        sched.step()
    sd = copy.deepcopy(a.state_dict())
    live = len(flat.live_index)
    assert len(sd["state"]) == live and [len(g["params"]) for g in sd["param_groups"]] == \
        [len(g["params"]) for g in a.param_groups]
    w3 = flat.flat.clone()
    a.zero_grad()
    _fwd_bwd(model, lossf, batches[3])
    a.step()
    want = _params(model)

    flat.flat.copy_(w3)
    b_opt = second(0.5)
    b_opt.load_state_dict(sd)
    assert [g["lr"] for g in b_opt.param_groups] == [g["lr"] for g in a.param_groups]
    assert [g["initial_lr"] for g in b_opt.param_groups] == [g["initial_lr"] for g in a.param_groups]
    b_opt.zero_grad()
    _fwd_bwd(model, lossf, batches[3])
    b_opt.step()
    _assert_same_update(_params(model), want)


def test_multi_group_resume_with_scheduler_is_bit_exact(tmp_path):
    case = "anp_distractor"
    batches = _batches(case, 6)
    kw = dict(decoupled_weight_decay=True, max_grad_norm=0.5, skip_nonfinite=True)

    def run(resume_at=None):
        model, opt, g, step = _fresh(case, True, **kw)
        sched = torch.optim.lr_scheduler.LambdaLR(opt, _lambdas())
        losses = []
        for i, b in enumerate(batches):
            if i == resume_at:
                torch.save({"train": g.state_dict(), "scheduler": sched.state_dict()}, tmp_path / "ckpt.pt")
                model, opt, g, step = _fresh(case, True, **kw)
                step(batches[0]), step(batches[1])       # load over captured graphs
                sched = torch.optim.lr_scheduler.LambdaLR(opt, _lambdas())
                sd = torch.load(tmp_path / "ckpt.pt", weights_only=False)
                g.load_state_dict(sd["train"])
                sched.load_state_dict(sd["scheduler"])
            losses.append(step(b))
            sched.step()
        torch.cuda.synchronize()
        return losses, opt

    ref_losses, ref = run()
    losses, opt = run(resume_at=3)
    assert all(torch.equal(a, b) for a, b in zip(losses, ref_losses))
    assert _same(_state(opt), _state(ref))
    assert torch.equal(opt._table, ref._table)
    assert [g["lr"] for g in opt.param_groups] == [g["lr"] for g in ref.param_groups]


def test_checkpoints_that_do_not_fit_are_refused():
    from b200np.optim import FlatParams, FusedAdam
    from trainer.losses import LossFunc
    model = _product("cnp_distractor_max")
    flat, lossf = FlatParams(model), LossFunc("mse", "distractor")
    opt = FusedAdam(flat, lr=LR, param_groups=_groups(model.named_parameters()))
    for b in _batches("cnp_distractor_max", 2):
        opt.zero_grad()
        _fwd_bwd(model, lossf, b)
        opt.step()
    good = opt.state_dict()
    before = (opt.m.clone(), opt.v.clone(), opt.t_dev.clone()), _table(opt)

    fewer = copy.deepcopy(good)
    fewer["param_groups"] = fewer["param_groups"][:2]
    moved = copy.deepcopy(good)
    moved["param_groups"][1]["params"].append(moved["param_groups"][0]["params"].pop())
    amsgrad = copy.deepcopy(good)
    amsgrad["param_groups"][2]["amsgrad"] = True
    for sd, msg in [(fewer, "group"), (moved, "parameters"), (amsgrad, "amsgrad")]:
        for g in sd["param_groups"]:
            g["lr"], g["betas"], g["weight_decay"], g["decoupled_weight_decay"] = 0.5, (0.1, 0.2), 0.3, True
        with pytest.raises(ValueError, match=msg):
            opt.load_state_dict(sd)
        after = (opt.m, opt.v, opt.t_dev), _table(opt)
        assert _same(after[0], before[0])
        assert torch.equal(after[1][0], before[1][0]) and after[1][1] == before[1][1]
    with pytest.raises(RuntimeError, match="fixed"):
        opt.add_param_group({"params": []})


def test_checkpoint_without_decoupled_key_keeps_each_groups_setting():
    """A checkpoint from a torch older than the `decoupled_weight_decay` key: as torch's Adam and AdamW, FusedAdam
    keeps what each of its groups was built with, in the group dict and in the device table."""
    from b200np.optim import FlatParams, FusedAdam
    model = _product("cnp_distractor_max")
    flat = FlatParams(model)
    old = torch.optim.AdamW(_groups(model.named_parameters()), lr=LR).state_dict()
    for g in old["param_groups"]:
        del g["decoupled_weight_decay"]
    for decoupled in (False, True):
        opt = FusedAdam(flat, lr=0.5, decoupled_weight_decay=decoupled, param_groups=_groups(model.named_parameters()))
        opt.load_state_dict(copy.deepcopy(old))
        assert [g["decoupled_weight_decay"] for g in opt.param_groups] == [decoupled] * 3
        assert opt._table.view(torch.int32)[:, 5].tolist() == [int(decoupled)] * 3 and opt.lr == LR


# ------------------------------------------------------------------------------------------------
# two GPUs
# ------------------------------------------------------------------------------------------------
_WORKER = r"""
import os, sys, torch, torch.distributed as td
ROOT = sys.argv[1]
sys.path[:0] = [ROOT, os.path.join(ROOT, "what-matters-for-meta-learning_b200"), os.path.join(ROOT, "tests")]
from conftest import make_config
from b200np import dist, engine
from b200np.optim import FlatParams, FusedAdam
from networks.ANPDistractor import ANPDistractor
from oracle import synth
from trainer.losses import LossFunc
from test_gpu_optim_groups import _groups
rank = int(os.environ["RANK"]); dev = torch.device(f"cuda:{int(os.environ['LOCAL_RANK'])}")
torch.cuda.set_device(dev)
td.init_process_group("nccl", device_id=dev)
engine.set_precision("tf32x3")
T, nc, nt, W = 4, 3, 4, td.get_world_size()
lo, hi = dist.shard_tasks(T)
lossf = LossFunc("mse", "distractor")
torch.manual_seed(0)
model = ANPDistractor(make_config("ANPDistractor", "distractor", T // W, "attention", "max", device=str(dev),
                                  dim_w=16)).to(dev)
opt = FusedAdam(FlatParams(model), lr=1e-3, decoupled_weight_decay=True, max_grad_norm=1.0,
                param_groups=_groups(model.named_parameters()))
w0 = opt.flat.flat.clone()
for i in range(3):
    b = [torch.from_numpy(a).to(dev)[lo:hi].contiguous() for a in synth.task_batch("distractor", T, nc, nt, seed=5 + i)]
    opt.zero_grad()
    mu, _, _ = model(b[0], b[1], b[2]); lossf.calc_loss(mu, None, b[3]).backward(); opt.step()
torch.cuda.synchronize()
w = opt.flat.flat
allw = [torch.empty_like(w) for _ in range(W)]
td.all_gather(allw, w)
assert all(torch.equal(allw[0], a) for a in allw), "weights differ across ranks"
assert not torch.equal(w, w0) and int(opt.t_dev) == 3
if rank == 0:
    print(f"RESULT ranks={W} moved={float((w - w0).norm()):.4e}", flush=True)
td.barrier()
td.destroy_process_group()
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_groups_stay_identical_across_ranks(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29653", str(script), ROOT]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "RESULT" in out.stdout, out.stdout[-3000:]
    print("\n".join(l for l in out.stdout.splitlines() if l.startswith("RESULT")))
