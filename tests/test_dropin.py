"""The drop-in boundary (SURVEY.md section 8b): with the B200 package first on sys.path and the reference checkout
behind it (what b200_run.py arranges), the reference's own entry scripts import, hot-path names resolve to the B200
classes, everything else to the reference's files -- and the UNMODIFIED `ModelTrainer._train_iter`
(trainer/model_trainer.py:59-93) trains the drop-in modules with `torch.optim.Adam`, tracking the CPU oracle.

The reference tree is /root/reference in the build container and its byte-identical copy oracle/_ref on the GPU box
(oracle/make_ref.py); tests that need it skip when neither exists.
"""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import CASES, ROOT, PKG, make_config, oracle_cfg
from oracle import ref_shims

needs_ref = pytest.mark.skipif(not ref_shims.reference_available(), reason="reference tree not present")

_IMPORT_PROBE = r"""
import importlib, os, sys
root, pkg, ref = sys.argv[1:4]
sys.path.insert(0, root)
from oracle import ref_shims
ref_shims.install()                      # stubs for torchmeta / imgaug / ... (absent from this image)
while ref in sys.path: sys.path.remove(ref)
sys.path.insert(0, pkg)
import b200_run
b200_run.setup_path(ref)
assert sys.path[0] == pkg and sys.path[1] == ref
src = open(os.path.join(ref, "train.py")).read()
exec("\n".join(l for l in src.splitlines() if l.startswith(("import ", "from "))))   # train.py:17-30
inside = lambda m, d: os.path.abspath(sys.modules[m].__file__).startswith(os.path.abspath(d) + os.sep)
assert inside("trainer.model_trainer", ref) and inside("trainer.maml_trainer", ref) and inside("trainer.mmaml_trainer", ref)
assert inside("trainer.losses", pkg) and LossFunc.__mro__[1].__module__ == "trainer._reference_losses"
for method in ("ANPDistractor", "ANP", "ANPShapeNet1D", "CNPDistractor", "CondNeuralProcess", "CNPShapeNet1D"):
    m = importlib.import_module(f"networks.{method}")          # train.py:42-43
    assert inside(m.__name__, pkg), m.__file__
    assert getattr(m, method).__mro__[1].__module__ == "networks._families"
for other in ("models", "ResNet", "fast_attention", "MAMLShapeNet1D", "MMAMLShapeNet1D", "CNPMR"):
    m = importlib.import_module(f"networks.{other}")
    assert inside(m.__name__, ref), m.__file__
# shadowed on purpose, but handing out the reference's own classes unless B200NP_MMAML=1 / B200NP_BBB=1
from networks.gated_conv_net import GatedConvModel
from networks.bbb import BBBConv2d, BBBLinear
assert GatedConvModel.__module__ == "networks._reference_gated_conv_net"
assert BBBConv2d.__module__ == "networks.bbb._reference_BBBConv" and BBBLinear.__module__ == "networks.bbb._reference_BBBLinear"
print("OK")
"""


@needs_ref
def test_train_py_import_block_resolves_under_the_launcher_recipe():
    # other test modules opt into the B200 MMAML / BBB classes through os.environ in this process: the probe checks
    # the DEFAULT resolution, so the child must not inherit those switches
    env = {k: v for k, v in os.environ.items() if k not in ("B200NP_MMAML", "B200NP_BBB")}
    r = subprocess.run([sys.executable, "-c", _IMPORT_PROBE, ROOT, PKG, ref_shims.REFERENCE_ROOT],
                       capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout + r.stderr


@pytest.mark.skipif(not os.path.isfile(os.path.join(ROOT, "oracle", "_ref", "MANIFEST.sha256")),
                    reason="oracle/_ref not materialised")
def test_ref_copy_is_unmodified():
    """oracle/_ref holds byte-identical reference files (sha256 manifest written by oracle/make_ref.py; compared
    with /root/reference itself where that exists)."""
    base = os.path.join(ROOT, "oracle", "_ref")
    n = 0
    for line in open(os.path.join(base, "MANIFEST.sha256")):
        h, rel = line.split()
        assert hashlib.sha256(open(os.path.join(base, rel), "rb").read()).hexdigest() == h, rel
        src = os.path.join("/root/reference", rel)
        if os.path.isfile(src):
            assert hashlib.sha256(open(src, "rb").read()).hexdigest() == h, rel
        n += 1
    assert n >= 50


class _StubData:
    """get_batch like dataset/shapenet_distractor.py:186-207: `shot ~ U{1..max}` context views per batch, the
    remaining views of the 36 as targets; returns (ctx_x, qry_x, ctx_y, qry_y) CPU tensors."""

    def __init__(self, task, views, seed=5):
        self.task, self.views, self.rng, self.calls, self.shots = task, views, np.random.RandomState(seed), 0, []

    def get_batch(self, source, tasks_per_batch, shot):
        from oracle import synth
        nc = int(self.rng.randint(1, shot + 1))            # shapenet_distractor.py:197
        self.shots.append(nc)
        self.calls += 1
        cx, cy, tx, ty = synth.task_batch(self.task, tasks_per_batch, nc, self.views - nc, seed=900 + self.calls)
        return tuple(torch.from_numpy(a) for a in (cx, tx, cy, ty))


def _reference_model_trainer():
    """The unmodified ModelTrainer class out of the reference tree, imported under the launcher's path recipe."""
    ref_shims.install()
    ref = ref_shims.REFERENCE_ROOT
    while ref in sys.path:
        sys.path.remove(ref)
    import b200_run
    b200_run.setup_path(ref)
    import importlib
    mt = importlib.import_module("trainer.model_trainer")
    assert os.path.abspath(mt.__file__).startswith(os.path.abspath(ref))
    return mt.ModelTrainer


class _RestatedTrainer:
    """The training step the reference's ModelTrainer._train_iter takes (trainer/model_trainer.py:59-93), as bench.py's
    e2e_dropin leg times it: zero_grad -> .to(device) of a host batch -> model -> calc_loss -> in-place
    `losses += kl * beta` -> backward -> optimizer.step -> losses.item().  Lets the drop-in's training-loop contract
    be checked without the reference tree."""

    def _train_iter(self, it):
        cfg = self.config
        self.model.train()
        self.optimizer.zero_grad()
        ctx_x, qry_x, ctx_y, qry_y = (t.to(cfg.device)
                                      for t in self.data.get_batch("train", cfg.tasks_per_batch, cfg.max_ctx_num))
        pr_mu, pr_var, kl = self.model(ctx_x, ctx_y, qry_x)
        losses = self.loss.calc_loss(pr_mu, pr_var, qry_y)
        losses += kl * cfg.beta
        losses.backward()
        self.optimizer.step()
        return losses.item()


@needs_ref
@pytest.mark.gpu
@pytest.mark.parametrize("graphs", [False, True])
@pytest.mark.parametrize("case", ["anp_distractor", "cnp_1d_max"])
def test_unmodified_model_trainer_runs_on_the_dropin(case, graphs):
    _check_trainer_on_the_dropin(_reference_model_trainer, case, graphs)


@pytest.mark.gpu
@pytest.mark.parametrize("graphs", [False, True])
@pytest.mark.parametrize("case", ["anp_distractor", "cnp_1d_max"])
def test_restated_training_loop_runs_on_the_dropin(case, graphs):
    _check_trainer_on_the_dropin(lambda: _RestatedTrainer, case, graphs)


def _check_trainer_on_the_dropin(trainer_class, case, graphs):
    """Six `_train_iter` steps of `trainer_class()` on the drop-in modules with torch.optim.Adam and a context size
    redrawn per step track the CPU oracle's loss; then one validation forward."""
    import importlib
    import types
    from b200np import engine
    from oracle import np_oracle
    engine.set_precision("tf32x3")
    ModelTrainer = trainer_class()
    method, task, agg, img_agg, extra, T, _, _ = CASES[case]
    cfg = make_config(method, task, T, agg, img_agg, device="cuda:0", **extra)
    cfg.max_ctx_num, cfg.lr = 15, 1e-3
    model = getattr(importlib.import_module(f"networks.{method}"), method)(cfg).to(cfg.device)
    assert type(model).__mro__[1].__module__ == "networks._families"
    model.enable_cuda_graphs(graphs)
    LossFunc = importlib.import_module("trainer.losses").LossFunc
    optimizer = torch.optim.Adam(model.parameters(), lr=cfg.lr)                    # train.py:52-56
    tr_oracle = np_oracle.OracleTrainer(method, oracle_cfg(cfg), {k: v.cpu() for k, v in model.state_dict().items()},
                                        lr=cfg.lr)
    data = _StubData(task, 36 if task == "distractor" else 30)
    trainer = ModelTrainer.__new__(ModelTrainer)          # BaseTrainer.__init__ only opens a SummaryWriter directory
    trainer.model, trainer.loss, trainer.optimizer = model, LossFunc("mse", task), optimizer
    trainer.config, trainer.data, trainer.writer = cfg, data, None
    seen = []
    orig = trainer.loss.calc_loss

    def spy(mu, var, y, test=False):
        out = orig(mu, var, y, test)
        seen.append(out)
        return out
    trainer.loss.calc_loss = spy
    mirror = _StubData(task, data.views)
    for it in range(1, 7):
        trainer._train_iter(it)                                                     # model_trainer.py:59-93, unmodified
        cx, tx, cy, ty = mirror.get_batch("train", T, cfg.max_ctx_num)
        lo = tr_oracle.step(cx, cy, tx, ty)
        got = float(seen[-1])
        assert abs(got - lo) < 2e-3 * abs(lo), (it, got, lo, data.shots)
    assert len(set(data.shots)) >= 3                     # the context size really changed between steps
    if graphs:
        assert len(model._graphed.cache) == len(set(data.shots))
    # the in-place `losses += kl * beta` of model_trainer.py:80 went through; validation path (no grad, test=True)
    model.eval()
    with torch.no_grad():
        cx, tx, cy, ty = (t.to(cfg.device) for t in mirror.get_batch("val", T, cfg.max_ctx_num))
        mu, var, kl = model(cx, cy, tx, test=True)
        l = trainer.loss.calc_loss(mu, var, ty, test=True)
        assert torch.isfinite(l.view(1)).all()


@pytest.mark.gpu
def test_loss_supports_the_trainers_inplace_add():
    """model_trainer.py:80 does `losses += kl * beta` on the result of calc_loss."""
    from conftest import build_product_model
    from oracle import synth
    from trainer.losses import LossFunc
    model, cfg = build_product_model("cnp_distractor_max", device="cuda")
    model = model.to("cuda")
    cx, cy, tx, ty = (torch.from_numpy(a).cuda() for a in synth.task_batch("distractor", 2, 3, 4, seed=1))
    mu, _, kl = model(cx, cy, tx)
    l = LossFunc("mse", "distractor").calc_loss(mu, None, ty)
    assert l.dim() == 0
    l += kl * 0.5
    l.backward()
    assert model.mu.weight.grad is not None and torch.isfinite(model.mu.weight.grad).all()
