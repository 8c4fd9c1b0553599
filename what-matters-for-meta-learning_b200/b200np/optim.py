"""Flat parameter / gradient buffers and the fused Adam step.

``flatten_module`` re-homes every parameter of a model into one contiguous fp32 buffer (each
``nn.Parameter`` becomes a view, so ``state_dict`` / ``load_state_dict`` / ``parameters()`` keep
working) and gives every parameter a ``.grad`` view into one flat gradient buffer.  That turns
the optimizer step into ONE HBM-bound kernel launch and the data-parallel gradient exchange into
ONE NCCL all-reduce.  Parameters that never receive a gradient (the dead ``resnet.fc`` layers,
SURVEY.md 8a/a14) are placed after the live ones and skipped, exactly like torch.optim.Adam skips
``p.grad is None``.
"""
import torch

from . import dist, ops


class FlatParams:
    """`late(name)`: parameters whose gradients are produced LAST by the backward pass -- the CNN trunks, which are the
    leaves of the backward pass (`img_encoder.*`, the decoder's `conv1` / `resnet`; `encoder_w0.*` for the ShapeNet1D
    family).  They are laid out after all the others, so that the data-parallel exchange can run as two contiguous
    buckets: the dense / attention layers while the encoder CNN's backward is still computing, the CNNs at the end
    (FusedAdam).  `trigger(name)`: the parameter whose trunk starts its backward only after every non-late gradient is
    complete (the ENCODER CNN: the decoder CNN's backward starts right after `fc_mu`, on its own stream)."""

    LATE = ("img_encoder.", "encoder_w0.", "decoder.conv1.", "decoder.resnet.")
    TRIGGER = ("img_encoder.conv1.weight", "encoder_w0.0.weight")

    def __init__(self, module, dead=lambda name: ".resnet.fc." in name, late=lambda name: name.startswith(FlatParams.LATE),
                 trigger=lambda name: name in FlatParams.TRIGGER):
        named = list(module.named_parameters())
        index = {n: i for i, (n, _) in enumerate(named)}
        self.names = [n for n, _ in named]    # in module.parameters() order, the order optimizer checkpoints use
        alive = [(n, p) for n, p in named if not dead(n)]
        live = [(n, p) for n, p in alive if not late(n)] + [(n, p) for n, p in alive if late(n)]
        rest = [(n, p) for n, p in named if dead(n)]
        dev = named[0][1].device
        pad = lambda k: (k + 3) // 4 * 4  # keep every view 16-byte aligned
        self.n_early = sum(pad(p.numel()) for n, p in live if not late(n))
        self.n_live = sum(pad(p.numel()) for _, p in live)
        total = self.n_live + sum(pad(p.numel()) for _, p in rest)
        self.flat = torch.zeros(total, device=dev, dtype=torch.float32)
        self.grad = torch.zeros(self.n_live, device=dev, dtype=torch.float32)
        self.live, self.views, self._keep = [], {}, []
        self.live_index = []                  # position in module.parameters() of each entry of self.live
        off = 0
        for n, p in live + rest:
            k = p.numel()
            view = self.flat[off:off + k].view_as(p)
            view.copy_(p.data)
            p.data = view
            if off < self.n_live:
                self.live.append((n, p, off, k))
                self.live_index.append(index[n])
            off += pad(k)
        self.trigger_ptrs = {p.data_ptr() for n, p, _, _ in self.live if trigger(n)}

    def attach_grads(self):
        """Point every live parameter's .grad at its slice of the flat gradient buffer."""
        for _, p, off, k in self.live:
            p.grad = self.grad[off:off + k].view_as(p)

    def gather_grads(self, lo=0, hi=None, keep=None, skip_missing=False):
        """After autograd: bring every .grad with offset in [lo, hi) into the flat buffer -- ONE launch per 64 parameters
        (`b200np_multi_copy`); parameters without a gradient get zeros (`skip_missing`: are left for a later call).
        Afterwards .grad is the flat view.  `keep`: a list that receives the source tensors (a caller that enqueues the
        copy on another stream keeps them referenced until that stream has joined)."""
        hi = self.n_live if hi is None else hi
        keep = self._keep if keep is None else keep
        segs = []
        for _, p, off, k in self.live:
            if off < lo or off >= hi:
                continue
            view = self.grad[off:off + k].view_as(p)
            g = p.grad
            if g is None:
                if skip_missing:
                    continue
                segs.append((None, off, k))
            elif g.data_ptr() != view.data_ptr():
                if not g.is_contiguous():
                    g = g.contiguous()
                keep.append(g)            # keep the source alive until the copy has been enqueued
                segs.append((g, off, k))
            p.grad = view
        ops.multi_copy(self.grad, segs)
        if keep is self._keep:
            self._keep.clear()

    def zero_grad(self):
        """Drop the gradients: autograd then hands each parameter its gradient tensor by reference (no
        accumulate kernel per parameter); `gather_grads` collects them."""
        for _, p, _, _ in self.live:
            p.grad = None


class FusedAdam:
    """torch.optim.Adam semantics (train.py:52-56: lr from config, betas (0.9, 0.999), eps 1e-8,
    optional L2 weight decay) as one kernel over the flat live-parameter segment.

    Data parallel (world size > 1): the gradient exchange runs as TWO buckets.  When the encoder CNN's backward starts
    (engine.PRE_TRUNK_BACKWARD_HOOKS) every other gradient is complete: they are gathered and all-reduced on a second
    stream while the encoder CNN's data / weight gradients are still being computed; the CNNs' own bucket (~20 % of the
    bytes) follows at the end, and the Adam kernel waits for both.  Inside a captured step this is a graph branch.
    `B200NP_BUCKETS=0`: one all-reduce after the backward pass."""

    def __init__(self, flat: FlatParams, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        import os
        import weakref
        self.flat, self.lr, self.betas, self.eps, self.wd = flat, lr, betas, eps, weight_decay
        self.m = torch.zeros_like(flat.grad)
        self.v = torch.zeros_like(flat.grad)
        self.t = 0
        self.t_dev = torch.zeros(1, device=flat.grad.device, dtype=torch.int32)  # step count for graph replay
        self._early_done, self._early_keep, self._comm = False, [], None
        if os.environ.get("B200NP_BUCKETS", "1") != "0" and flat.n_early and flat.n_early < flat.n_live:
            from . import engine
            ref = weakref.ref(self)

            def hook(ptr):
                me = ref()
                if me is None:
                    engine.PRE_TRUNK_BACKWARD_HOOKS.remove(hook)
                elif ptr in me.flat.trigger_ptrs:
                    me._early_bucket()
            engine.PRE_TRUNK_BACKWARD_HOOKS.append(hook)

    def zero_grad(self, set_to_none=False):
        self.flat.zero_grad()
        self._early_done = False

    def _early_bucket(self):
        """The gradients laid out before the encoder CNN's: gather + all-reduce on the communication stream."""
        if self._early_done or dist.world_size() == 1:
            return
        f = self.flat
        main = torch.cuda.current_stream()
        if self._comm is None:
            self._comm = torch.cuda.Stream(priority=-1)
        self._comm.wait_stream(main)
        with torch.cuda.stream(self._comm):
            f.gather_grads(0, f.n_early, keep=self._early_keep, skip_missing=True)
            dist.all_reduce_sum(f.grad[:f.n_early])
        self._early_done = True

    def step(self):
        from .engine import nvtx_range
        with nvtx_range("b200np.adam.step"):
            self._step()

    def _step(self):
        f = self.flat
        world = dist.world_size()
        if world > 1 and self._early_done:
            # whatever the early bucket did not find (a parameter whose gradient arrived later: none on the shipped
            # models) is exchanged on its own, so the result never depends on the bucket boundary being right
            late_early = [(p, off, k) for _, p, off, k in f.live
                          if off < f.n_early and p.grad is not None and p.grad.data_ptr() != f.grad[off:off + k].data_ptr()]
            torch.cuda.current_stream().wait_stream(self._comm)   # before anything else writes into the early segment
            self._early_keep.clear()
            f.gather_grads()
            dist.all_reduce_sum(f.grad[f.n_early:f.n_live])
            for _, off, k in late_early:
                dist.all_reduce_sum(f.grad[off:off + k])
            self._early_done = False
        else:
            f.gather_grads()
            if world > 1:
                dist.all_reduce_grads(f.grad)
        self.t += 1
        # the step counter is kept on the device so that a captured CUDA graph of the whole step stays valid
        ops.adam_step_dev(f.flat, f.grad, self.m, self.v, f.n_live, self.lr, self.betas[0], self.betas[1], self.eps,
                          self.wd, self.t_dev, 1.0 / world)

    # the rest of a torch.optim.Adam param_group, at the values that describe what the fused kernel computes
    _GROUP_FLAGS = dict(amsgrad=False, maximize=False, foreach=None, capturable=False, differentiable=False, fused=None,
                        decoupled_weight_decay=False)

    def state_dict(self):
        """The optimizer state in exactly the structure `torch.optim.Adam(model.parameters()).state_dict()` has, so
        either optimizer can resume from the other's checkpoint.  `state` is keyed by position in
        `module.parameters()`; each live parameter gets `step` (0-dim float32 CPU tensor) and clones of its slices
        of the moments.  Parameters that never receive a gradient, and every parameter before the first step, get
        no entry, as in torch.  Reading the step count is one 4-byte device-to-host copy."""
        f = self.flat
        t = int(self.t_dev.item())
        state = {}
        if t > 0:
            for i, (_, p, off, k) in sorted(zip(f.live_index, f.live), key=lambda e: e[0]):
                state[i] = {"step": torch.tensor(float(t), dtype=torch.float32),
                            "exp_avg": self.m[off:off + k].view_as(p).clone(),
                            "exp_avg_sq": self.v[off:off + k].view_as(p).clone()}
        group = dict(lr=self.lr, betas=tuple(self.betas), eps=self.eps, weight_decay=self.wd, **self._GROUP_FLAGS,
                     params=list(range(len(f.names))))
        return {"state": state, "param_groups": [group]}

    def load_state_dict(self, state_dict):
        """Resume from a `state_dict()` of this class or of `torch.optim.Adam` over the same model's parameters.

        The moments are written into the existing `m` / `v` (one `multi_copy` launch per 64 parameters) and the step
        count into `t_dev`, all in place, so a CUDA graph captured over these buffers stays valid.  A parameter
        without a state entry gets zero moments.  The hyperparameters are taken from the checkpoint, as torch does.
        The whole checkpoint is checked before anything is written; `ValueError` if it does not fit this model or
        needs something the flat kernel does not do (one step counter, plain Adam)."""
        f = self.flat
        groups = state_dict["param_groups"]
        if len(groups) != 1:
            raise ValueError(f"FusedAdam has one parameter group; the checkpoint has {len(groups)}")
        group = groups[0]
        for flag in ("amsgrad", "maximize", "decoupled_weight_decay"):
            if group.get(flag, False):
                raise ValueError(f"the checkpoint was written with {flag}=True; FusedAdam implements plain Adam only")
        ids = list(group["params"])
        if len(ids) != len(f.names):
            raise ValueError(f"the checkpoint holds {len(ids)} parameters, the model has {len(f.names)}")
        live = dict(zip(f.live_index, f.live))
        found, steps = {}, set()
        for i, pid in enumerate(ids):
            s = state_dict["state"].get(pid)
            if s is None:
                continue
            name = f.names[i]
            if i not in live:
                raise ValueError(f"the checkpoint has Adam state for {name!r}, which never receives a gradient here")
            shape = tuple(live[i][1].shape)
            for key in ("exp_avg", "exp_avg_sq"):
                if tuple(s[key].shape) != shape:
                    raise ValueError(f"{name}: the checkpoint's {key} has shape {tuple(s[key].shape)}, "
                                     f"the parameter {shape}")
            steps.add(float(s["step"]))
            found[i] = s
        if len(steps) > 1:
            raise ValueError(f"the parameters' Adam step counts differ ({sorted(steps)}); the fused kernel keeps one "
                             "step counter for all of them")
        t = steps.pop() if steps else 0.0
        if t < 0 or t != int(t) or t >= 2 ** 31:
            raise ValueError(f"Adam step count {t} is not a valid int32 count")
        dev = f.grad.device
        seg_m, seg_v = [], []
        for i, (_, p, off, k) in zip(f.live_index, f.live):
            s = found.get(i)
            if s is None:
                seg_m.append((None, off, k)), seg_v.append((None, off, k))
            else:
                seg_m.append((s["exp_avg"].detach().to(dev, torch.float32).contiguous(), off, k))
                seg_v.append((s["exp_avg_sq"].detach().to(dev, torch.float32).contiguous(), off, k))
        ops.multi_copy(self.m, seg_m)
        ops.multi_copy(self.v, seg_v)
        self.t_dev.fill_(int(t))
        self.t = int(t)
        self.lr, self.eps, self.wd = float(group["lr"]), float(group["eps"]), float(group["weight_decay"])
        self.betas = tuple(float(b) for b in group["betas"])


class GraphedStep:
    """One meta-train step (zero_grad, forward, loss, backward, all-reduce, Adam) captured in a CUDA graph.

    Every kernel of the path is launched on torch's current stream without host synchronisation or
    allocation outside torch's caching allocator, so the whole step -- a few hundred launches -- can be recorded
    once per (nc, nt) shape and replayed with a single cudaGraphLaunch: no Python / ctypes / autograd time and
    no launch gaps on the GPU.  Inputs are copied into static buffers before each replay.

    Shapes: the reference draws `shot ~ U{1..max_ctx_num}` per batch (dataset/shapenet_distractor.py:197), so the
    context / target split changes from step to step.  Graphs are therefore kept in a cache keyed by the batch's
    shapes (at most `max_ctx_num` entries) and built on first use; all of them share one memory pool, because they
    never run concurrently.

    Building a graph runs `warmup` real steps and the capture itself on the model; parameters, Adam moments and
    the step counter are snapshotted before and restored afterwards, so constructing the object (or meeting a new
    shape) does NOT advance training.  A graph holds the Adam hyperparameters it was captured with; when `opt.lr`,
    `betas`, `eps` or `wd` have changed since (by assignment or `load_state_dict`), the graph is recaptured, in the
    same way, before its next replay.

    Input pipeline: ``step(batch, next_batch=...)`` starts the host-to-device copy of the NEXT batch on a
    second stream into staging buffers while this step computes (the reference gets the same overlap from
    its pinned-memory DataLoader, trainer/model_trainer.py:59-67); the staged batch reaches the graph's
    static inputs with a device-to-device copy (47 MB, ~20 us) at the start of its own step.  A batch handed to
    ``prefetch`` must not be modified until the step that consumes it has been called: the staged copy is
    matched to the step by object identity of its tensors.
    """

    def __init__(self, model, lossf, opt, example_batch=None, warmup=3):
        self.model, self.lossf, self.opt, self.warmup = model, lossf, opt, warmup
        self.copy_stream = torch.cuda.Stream()
        self.ev_ready, self.ev_free = torch.cuda.Event(), torch.cuda.Event()
        self._staged = None          # (graph entry, the prefetched batch's tensors)
        self.cache = {}
        self.pool = torch.cuda.graph_pool_handle()
        from . import engine
        # warm-up and capture run on one high-priority stream: the engine's companion streams (decoder CNN, weight
        # gradients) rank below it, and the captured kernel nodes keep those priorities
        self.side = torch.cuda.Stream(priority=engine.MAIN_PRIORITY if engine.USE_PRIORITIES else 0)
        self.graph = self.loss = None
        if example_batch is not None:
            ent = self._entry(example_batch)
            self.graph, self.loss = ent["graph"], ent["loss"]

    @staticmethod
    def _key(batch):
        return tuple(tuple(t.shape) for t in batch)

    def _hyper(self):
        o = self.opt
        return (o.lr, tuple(o.betas), o.eps, o.wd)

    def _entry(self, batch):
        key = self._key(batch)
        ent = self.cache.get(key)
        if ent is not None:
            return ent
        dev = self.opt.flat.flat.device
        ent = {"static": [torch.empty(t.shape, device=dev, dtype=t.dtype) for t in batch],
               "stage": [torch.empty(t.shape, device=dev, dtype=t.dtype) for t in batch]}
        for s, t in zip(ent["static"], batch):
            s.copy_(t)
        self._capture(ent)
        self.cache[key] = ent
        return ent

    def _capture(self, ent):
        """Warm up and capture the step on `ent`'s static inputs, recording the hyperparameters the graph holds."""
        opt = self.opt
        old = ent.get("graph")
        snap = (opt.flat.flat.clone(), opt.m.clone(), opt.v.clone(), opt.t_dev.clone(), opt.t)
        cur = torch.cuda.current_stream()
        self.side.wait_stream(cur)
        with torch.cuda.stream(self.side):
            for _ in range(self.warmup):
                self._eager(ent["static"])
        cur.wait_stream(self.side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=self.side, pool=self.pool):
            loss = self._eager(ent["static"])
        # neither the warm-up steps nor the capture may advance training
        opt.flat.flat.copy_(snap[0]), opt.m.copy_(snap[1]), opt.v.copy_(snap[2]), opt.t_dev.copy_(snap[3])
        opt.t = snap[4]
        torch.cuda.synchronize()
        ent["graph"], ent["loss"], ent["hyper"] = graph, loss, self._hyper()
        if old is not None and self.graph is old:     # recaptured the example batch's graph
            self.graph, self.loss = graph, loss

    def _eager(self, static):
        cx, cy, tx, ty = static
        self.opt.zero_grad()
        mu, _, _ = self.model(cx, cy, tx)
        loss = self.lossf.calc_loss(mu, None, ty)
        loss.backward()
        self.opt.step()
        return loss.detach()

    def prefetch(self, batch):
        """Start copying `batch` (pinned host or device tensors) into the staging buffers of its shape on the
        copy stream."""
        ent = self._entry(batch)
        cs = self.copy_stream
        cs.wait_event(self.ev_free)            # the previous occupant of the staging buffers has been consumed
        with torch.cuda.stream(cs):
            for s, t in zip(ent["stage"], batch):
                s.copy_(t, non_blocking=True)
            self.ev_ready.record(cs)
        self._staged = (ent, tuple(batch))     # holds the tensors: identity, not addresses, names the batch

    def __call__(self, batch, next_batch=None):
        cur = torch.cuda.current_stream()
        st = self._staged
        if st is not None and len(st[1]) == len(batch) and all(a is b for a, b in zip(st[1], batch)):
            ent = st[0]
            cur.wait_event(self.ev_ready)      # prefetched during the previous step
            for s, t in zip(ent["static"], ent["stage"]):
                s.copy_(t, non_blocking=True)
        else:
            ent = self._entry(batch)
            for s, t in zip(ent["static"], batch):
                if s.data_ptr() != t.data_ptr():
                    s.copy_(t, non_blocking=True)
        if ent["hyper"] != self._hyper():
            # the Adam launch in the graph carries the hyperparameters as kernel arguments: a graph captured before
            # `opt.lr = ...` or `load_state_dict` would silently keep the old values
            self._capture(ent)
        self._staged = None
        self.ev_free.record(cur)
        ent["graph"].replay()
        self.opt.t += 1
        if next_batch is not None:
            self.prefetch(next_batch)
        return ent["loss"]

    def state_dict(self):
        """What a resumed run needs: `{"model": model.state_dict(), "optimizer": opt.state_dict()}`."""
        return {"model": self.model.state_dict(), "optimizer": self.opt.state_dict()}

    def load_state_dict(self, state_dict):
        """Load weights and optimizer state in place (the captured graphs keep their buffers; a graph whose
        hyperparameters changed is recaptured before its next replay).  The optimizer goes first: it checks the
        checkpoint against the model's parameters before anything is written."""
        self.opt.load_state_dict(state_dict["optimizer"])
        self.model.load_state_dict(state_dict["model"])


class GraphedEval:
    """The validation / evaluation forward (evaluator/model_evaluator.py:144-179: no-grad `model(ctx_x, ctx_y,
    tgt_x, test=True)` + `calc_loss(test=True)`) as CUDA graphs, one per (context, target) shape -- the evaluator
    sweeps nc = 1..25 with all views as targets, so a handful of shapes repeat for thousands of tasks.
    Returns `(mu, loss)`; both live in static buffers that the next call with the same shape overwrites."""

    def __init__(self, model, lossf=None, warmup=1):
        self.model, self.lossf, self.warmup = model, lossf, warmup
        self.cache = {}

    def _forward(self, cx, cy, tx, ty):
        mu, _, _ = self.model(cx, cy, tx, test=True)
        loss = self.lossf.calc_loss(mu, None, ty, test=True) if (self.lossf is not None and ty is not None) else None
        return mu, loss

    def __call__(self, ctx_x, ctx_y, tgt_x, tgt_y=None):
        batch = [ctx_x, ctx_y, tgt_x] + ([tgt_y] if tgt_y is not None else [])
        key = tuple(tuple(t.shape) for t in batch)
        ent = self.cache.get(key)
        if ent is None:
            static = [torch.empty(t.shape, device=tgt_x.device if tgt_x.is_cuda else "cuda", dtype=t.dtype) for t in batch]
            for s_, t in zip(static, batch):
                s_.copy_(t)
            args = static + [None] * (4 - len(static))
            with torch.no_grad():
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    for _ in range(self.warmup):
                        self._forward(*args)
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    out = self._forward(*args)
            ent = self.cache[key] = (graph, static, out)
        graph, static, out = ent
        for s_, t in zip(static, batch):
            if s_.data_ptr() != t.data_ptr():
                s_.copy_(t, non_blocking=True)
        graph.replay()
        return out
