"""Checkpoint / resume of the fused training path (FlatParams + FusedAdam + GraphedStep).

A run that is saved after 3 steps, rebuilt from scratch, loaded and continued must be bit-identical to the run that
never stopped, eagerly and under CUDA graphs -- including when the fresh GraphedStep has already captured its graphs
(the load must write into the captured buffers).  FusedAdam's state_dict is torch.optim.Adam's, so either optimizer
resumes the other's run; a new learning rate reaches already-captured graphs; checkpoints that do not fit are refused.
"""
import copy

import pytest
import torch

from conftest import CASES, build_product_model, rel_l2
from oracle import synth

pytestmark = pytest.mark.gpu

LR = 1e-3


def _batches(case, n=6):
    """`n` batches whose context size alternates between nc and nc + 2 (two graph shapes)."""
    method, task, agg, img_agg, extra, T, nc, nt = CASES[case]
    return [[torch.from_numpy(a).cuda() for a in synth.task_batch(task, T, nc + 2 * (i % 2), nt, seed=60 + i)]
            for i in range(n)]


def _fresh(case, graphed):
    """A new model, FlatParams, FusedAdam and (graphed) GraphedStep; returns (model, opt, step(batch) -> loss)."""
    from b200np import engine
    from b200np.optim import FlatParams, FusedAdam, GraphedStep
    from trainer.losses import LossFunc
    engine.set_precision("tf32x3")
    model, _ = build_product_model(case, device="cuda")
    model = model.to("cuda")
    opt = FusedAdam(FlatParams(model), lr=LR)
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


def _train(case, batches, graphed, resume_at=None, path=None, step_before_load=False):
    """Train on `batches`.  With `resume_at`: save to `path` after that many steps, build everything anew, load, go
    on.  `step_before_load`: the new objects first take a step on each of the two shapes (graphed: both graphs are
    captured and their state moves on) and the checkpoint is loaded over that."""
    model, opt, g, step = _fresh(case, graphed)
    losses = []
    for i, b in enumerate(batches):
        if i == resume_at:
            torch.save(g.state_dict() if g else {"model": model.state_dict(), "optimizer": opt.state_dict()}, path)
            model, opt, g, step = _fresh(case, graphed)
            if step_before_load:
                step(batches[0]), step(batches[1])
            sd = torch.load(path, weights_only=True)
            if g:
                g.load_state_dict(sd)
            else:
                model.load_state_dict(sd["model"])
                opt.load_state_dict(sd["optimizer"])
        losses.append(step(b))
    torch.cuda.synchronize()
    return losses, opt


@pytest.mark.parametrize("graphed", [False, True], ids=["eager", "graphed"])
@pytest.mark.parametrize("case", ["anp_distractor", "cnp_distractor_max"])
def test_resume_is_bit_exact(case, graphed, tmp_path):
    batches = _batches(case)
    ref_losses, ref = _train(case, batches, graphed)
    runs = [(False, "plain")] + ([(True, "load over captured graphs")] if graphed else [])
    for step_before_load, what in runs:
        losses, opt = _train(case, batches, graphed, resume_at=3, path=tmp_path / "ckpt.pt",
                             step_before_load=step_before_load)
        assert all(torch.equal(a, b) for a, b in zip(losses, ref_losses)), (what, losses, ref_losses)
        assert torch.equal(opt.flat.flat, ref.flat.flat), what
        assert torch.equal(opt.m, ref.m) and torch.equal(opt.v, ref.v), what
        assert int(opt.t_dev) == int(ref.t_dev) == 6 and opt.t == 6, what


def _model(case="cnp_distractor_max"):
    from b200np import engine
    from b200np.optim import FlatParams
    from trainer.losses import LossFunc
    engine.set_precision("tf32x3")
    model, _ = build_product_model(case, device="cuda")
    model = model.to("cuda")
    return model, FlatParams(model), LossFunc("mse", CASES[case][1])


def _fwd_bwd(model, lossf, batch):
    cx, cy, tx, ty = batch
    mu, _, _ = model(cx, cy, tx)
    lossf.calc_loss(mu, None, ty).backward()


def _params(model):
    return {k: p.detach().clone() for k, p in model.named_parameters()}


def _assert_same_update(got, want):
    """Both optimizers take the step from the same state and gradients: only their rounding order differs."""
    for k in want:
        e = rel_l2(got[k].double().cpu().numpy(), want[k].double().cpu().numpy())
        assert e <= 1e-6, (k, e)


def _assert_moments(flat, opt_m, opt_v, state_of):
    for i, (name, p, off, k) in zip(flat.live_index, flat.live):
        st = state_of(i)
        assert torch.equal(opt_m[off:off + k].view_as(p), st["exp_avg"].to(p.device)), name
        assert torch.equal(opt_v[off:off + k].view_as(p), st["exp_avg_sq"].to(p.device)), name


def test_torch_adam_checkpoint_resumes_on_fused_adam():
    from b200np.optim import FusedAdam
    model, flat, lossf = _model()
    batches = _batches("cnp_distractor_max", 4)
    topt = torch.optim.Adam(model.parameters(), lr=LR)
    assert FusedAdam(flat, lr=LR).state_dict() == topt.state_dict()      # same structure, before any step
    for b in batches[:3]:
        topt.zero_grad()
        _fwd_bwd(model, lossf, b)
        topt.step()
    sd = copy.deepcopy(topt.state_dict())
    assert sorted(sd["state"]) == sorted(flat.live_index)                # the dead resnet.fc layers have no entry
    w3 = flat.flat.clone()
    topt.zero_grad()
    _fwd_bwd(model, lossf, batches[3])
    topt.step()
    want = _params(model)

    flat.flat.copy_(w3)
    fopt = FusedAdam(flat, lr=0.5, betas=(0.5, 0.5), eps=1.0)
    fopt.load_state_dict(sd)
    assert (fopt.lr, fopt.betas, fopt.eps, fopt.wd) == (LR, (0.9, 0.999), 1e-8, 0.0)
    assert int(fopt.t_dev) == 3 and fopt.t == 3
    _assert_moments(flat, fopt.m, fopt.v, lambda i: sd["state"][i])
    fopt.zero_grad()
    _fwd_bwd(model, lossf, batches[3])
    fopt.step()
    _assert_same_update(_params(model), want)


def test_fused_adam_checkpoint_resumes_on_torch_adam():
    from b200np.optim import FusedAdam
    model, flat, lossf = _model()
    batches = _batches("cnp_distractor_max", 4)
    fopt = FusedAdam(flat, lr=LR)
    for b in batches[:3]:
        fopt.zero_grad()
        _fwd_bwd(model, lossf, b)
        fopt.step()
    sd = fopt.state_dict()
    assert sorted(sd["state"]) == sorted(flat.live_index)                # the dead resnet.fc layers have no entry
    for s in sd["state"].values():
        step = s["step"]
        assert step.dtype == torch.float32 and step.device.type == "cpu" and step.dim() == 0 and float(step) == 3
    topt = torch.optim.Adam(model.parameters(), lr=0.5)
    topt.load_state_dict(sd)
    assert topt.param_groups[0]["lr"] == LR
    params = list(model.parameters())
    _assert_moments(flat, fopt.m, fopt.v, lambda i: topt.state[params[i]])
    dead = set(range(len(params))) - set(flat.live_index)
    assert dead and all(params[i] not in topt.state for i in dead)
    w3 = flat.flat.clone()
    fopt.zero_grad()
    _fwd_bwd(model, lossf, batches[3])
    fopt.step()
    want = _params(model)

    flat.flat.copy_(w3)
    topt.zero_grad()
    _fwd_bwd(model, lossf, batches[3])
    topt.step()
    _assert_same_update(_params(model), want)


def test_new_hyperparameters_reach_captured_graphs():
    """The graph holds lr as a kernel argument: lr = 0 (assigned, or loaded from a checkpoint) must freeze the
    parameters on the next replay, and the step must still count."""
    model, opt, g, step = _fresh("cnp_distractor_max", graphed=True)
    b = _batches("cnp_distractor_max", 2)
    step(b[0]), step(b[1])                           # both shapes captured with lr = LR
    opt.lr = 0.0
    w, m = opt.flat.flat.clone(), opt.m.clone()
    step(b[0])
    assert torch.equal(opt.flat.flat, w) and not torch.equal(opt.m, m) and int(opt.t_dev) == 3

    opt.lr = LR
    step(b[1])
    assert not torch.equal(opt.flat.flat, w)
    sd = copy.deepcopy(g.state_dict())
    sd["optimizer"]["param_groups"][0]["lr"] = 0.0
    g.load_state_dict(sd)
    assert opt.lr == 0.0
    for batch in b:
        w = opt.flat.flat.clone()
        step(batch)
        assert torch.equal(opt.flat.flat, w)
    assert int(opt.t_dev) == 6


def test_checkpoints_that_do_not_fit_are_refused():
    from b200np.optim import FlatParams, FusedAdam
    model, flat, lossf = _model()
    opt = FusedAdam(flat, lr=LR)
    b = _batches("cnp_distractor_max", 2)
    for batch in b:
        opt.zero_grad()
        _fwd_bwd(model, lossf, batch)
        opt.step()
    good = opt.state_dict()
    before = (opt.m.clone(), opt.v.clone(), int(opt.t_dev), opt.lr)

    other, _ = build_product_model("anp_distractor", device="cuda")
    wrong_model = FusedAdam(FlatParams(other.to("cuda"))).state_dict()
    wrong_shape = copy.deepcopy(good)
    i = flat.live_index[0]
    wrong_shape["state"][i]["exp_avg"] = wrong_shape["state"][i]["exp_avg"][..., :-1]
    uneven = copy.deepcopy(good)
    uneven["state"][flat.live_index[5]]["step"] = torch.tensor(1.0)
    amsgrad = copy.deepcopy(good)
    amsgrad["param_groups"][0]["amsgrad"] = True
    for sd, msg in [(wrong_model, "parameters"), (wrong_shape, "shape"), (uneven, "step counts"),
                    (amsgrad, "amsgrad")]:
        sd["param_groups"][0]["lr"] = 0.5
        with pytest.raises(ValueError, match=msg):
            opt.load_state_dict(sd)
        after = (opt.m, opt.v, int(opt.t_dev), opt.lr)
        assert torch.equal(after[0], before[0]) and torch.equal(after[1], before[1]) and after[2:] == before[2:]
