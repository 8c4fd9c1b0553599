"""Flat parameter / gradient buffers and the fused Adam step.

``flatten_module`` re-homes every parameter of a model into one contiguous fp32 buffer (each
``nn.Parameter`` becomes a view, so ``state_dict`` / ``load_state_dict`` / ``parameters()`` keep
working) and gives every parameter a ``.grad`` view into one flat gradient buffer.  That turns
the optimizer step into ONE HBM-bound kernel launch and the data-parallel gradient exchange into
ONE NCCL all-reduce.  Parameters that never receive a gradient (the dead ``resnet.fc`` layers,
SURVEY.md 8a/a14) are placed after the live ones and skipped, exactly like torch.optim.Adam skips
``p.grad is None``.
"""
import contextlib

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
        self.params = [p for _, p in named]
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

    def gather_grads(self, lo=0, hi=None, keep=None, skip_missing=False, accumulate=False):
        """After autograd: bring every .grad with offset in [lo, hi) into the flat buffer -- ONE launch per 64 parameters
        (`b200np_multi_copy`); parameters without a gradient get zeros (`skip_missing`: are left for a later call).
        `accumulate`: ADD the gradients to what the flat buffer holds (`b200np_multi_accumulate`; the earlier
        micro-batches of a gradient-accumulation window), and skip parameters without a gradient instead of zeroing.
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
                if not accumulate:
                    segs.append((None, off, k))
            elif g.data_ptr() != view.data_ptr():
                if not g.is_contiguous():
                    g = g.contiguous()
                keep.append(g)            # keep the source alive until the copy has been enqueued
                segs.append((g, off, k))
            p.grad = view
        (ops.multi_accumulate if accumulate else ops.multi_copy)(self.grad, segs)
        if keep is self._keep:
            self._keep.clear()

    def zero_grad(self):
        """Drop the gradients: autograd then hands each parameter its gradient tensor by reference (no
        accumulate kernel per parameter); `gather_grads` collects them."""
        for _, p, _, _ in self.live:
            p.grad = None


class _Group(dict):
    """One of FusedAdam's parameter groups.  Assigning "lr", "betas", "eps", "weight_decay" or
    "decoupled_weight_decay" -- by a torch scheduler, `opt.lr = x` or `load_state_dict` -- also writes the group's
    record of the device table the Adam kernel reads (`row`, see ops.adam_group_table): small fill launches, no
    synchronisation, and captured graphs see the new value on their next replay.  `row` is None while
    torch.optim.Optimizer.__init__ builds the group; FusedAdam fills the table afterwards."""

    _COLUMN = {"lr": 0, "weight_decay": 1, "eps": 4}

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self.row = None

    @property
    def lr_dev(self):
        """The device scalar holding this group's learning rate."""
        return self.row[0]

    def __setitem__(self, key, value):
        if self.row is not None:
            if key in self._COLUMN:
                self.row[self._COLUMN[key]].fill_(float(value))
            elif key == "betas":
                self.row[2].fill_(float(value[0])), self.row[3].fill_(float(value[1]))
            elif key == "decoupled_weight_decay":
                self.row.view(torch.int32)[5].fill_(int(bool(value)))
        super().__setitem__(key, value)


class FusedAdam(torch.optim.Optimizer):
    """torch.optim.Adam / AdamW semantics (train.py:52-56: lr from config, betas (0.9, 0.999), eps 1e-8,
    optional weight decay) as one kernel over the flat live-parameter segment.

    A `torch.optim.Optimizer`, so that the schedulers of `torch.optim.lr_scheduler` drive it.  `param_groups=None`:
    one group over `module.parameters()`.  Otherwise a list of torch-style group dicts (`{"params": [...], "lr": ...,
    "weight_decay": ..., "decoupled_weight_decay": ...}`; keys a group omits take the constructor's values) over
    parameters of the flattened module, matched by identity.  A live parameter in no group is frozen, as in torch:
    never updated, zero moments, no state entry.  The groups are fixed with the flat layout: `add_param_group` after
    construction raises.  Every hyperparameter of every group lives in a device table (see `_Group`), so changing one
    needs no recapture of a graph.  `decoupled_weight_decay=True` is AdamW: `p *= 1 - lr * weight_decay` before the
    update, with the group's current lr.  `opt.lr`, `opt.betas`, `opt.eps` and `opt.wd` are group 0's.

    `max_grad_norm`: clip the gradient to this total norm, as `torch.nn.utils.clip_grad_norm_` between `backward()`
    and `step()` would, but after the data-parallel all-reduce (the norm is that of the averaged gradient, the same on
    every rank).  The norm covers every live parameter, frozen ones included, as `clip_grad_norm_(model.parameters())`
    would.  The clip coefficient is applied inside the Adam kernel, so `.grad` keeps the UNCLIPPED gradient.
    `skip_nonfinite`: a step whose gradient holds an inf or NaN leaves the parameters, both moments and the step count
    unchanged and adds one to `skipped_steps`.  With either set, `grad_norm` is the pre-clip total norm of the last
    step, as `clip_grad_norm_` returns it; both are device tensors, so reading them needs no per-step
    synchronisation.  `max_grad_norm` is a device value too: changing it reaches captured graphs without a recapture.

    Data parallel (world size > 1): the gradient exchange runs as TWO buckets.  When the encoder CNN's backward starts
    (engine.PRE_TRUNK_BACKWARD_HOOKS) every other gradient is complete: they are gathered and all-reduced on a second
    stream while the encoder CNN's data / weight gradients are still being computed; the CNNs' own bucket (~20 % of the
    bytes) follows at the end, and the Adam kernel waits for both.  Inside a captured step this is a graph branch.
    `B200NP_BUCKETS=0`: one all-reduce after the backward pass.

    Gradient accumulation (`accumulate_steps=k`, fixed at construction): one `step()` per window of k backward passes,
    on the SUM of their gradients times 1/(k * world size).  Callers divide the loss by neither k nor the world size.
    Eagerly, run the window's first k-1 backward passes inside `with opt.no_sync():` and the last one outside, then
    `step()`; `GraphedStep` does this per call.  Inside `no_sync()` no gradient exchange starts and the gradients sum
    in `p.grad` under autograd's ordinary rules, so a window costs one exchange whatever k is, and the last backward's
    early bucket still overlaps the encoder CNN's backward.  On world size > 1 a second backward pass outside
    `no_sync()` before `step()` raises `RuntimeError` (its gradients would miss the exchange already started).  The
    norm for clipping and skipping is that of the window's mean gradient, so a NaN in any micro-batch skips the whole
    step; `t`, `t_dev`, schedulers and `skipped_steps` advance once per window.  `state_dict()` / `load_state_dict()`
    raise between a window's backward passes: an open window is not part of the saved state.
    The ANP family's scalar exchanges (the FAVOR+ key stabiliser's MAX in forward, its gradient's SUM in backward) stay
    per micro-batch: each micro-batch is its own meta-batch for the stabiliser, so k accumulated ANP micro-batches
    give the sum of their own gradients, not those of one k-times larger meta-batch (SURVEY.md section 0 #5 puts
    such a difference at 8e-5 relative on the outputs at initialisation).  CNP-family models have independent tasks
    and a mean loss: k equal-shaped micro-batches of T tasks reproduce one batch of k*T tasks up to fp32 rounding."""

    def __init__(self, flat: FlatParams, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0,
                 decoupled_weight_decay=False, max_grad_norm=None, skip_nonfinite=False, param_groups=None,
                 accumulate_steps=1):
        import os
        import weakref
        dev = flat.grad.device
        if int(accumulate_steps) != accumulate_steps or accumulate_steps < 1:
            raise ValueError(f"accumulate_steps={accumulate_steps!r}: needs a whole number of backward passes >= 1")
        defaults = dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay,
                        decoupled_weight_decay=bool(decoupled_weight_decay), **self._GROUP_FLAGS)
        groups = [{"params": flat.params}] if param_groups is None else list(param_groups)
        for g in groups:
            for flag in ("amsgrad", "maximize"):
                if g.get(flag, False):
                    raise ValueError(f"a parameter group sets {flag}=True; FusedAdam implements Adam / AdamW only")
        super().__init__([_Group(g) for g in groups], defaults)
        position = {id(p): i for i, p in enumerate(flat.params)}
        group_of = {}
        for gi, g in enumerate(self.param_groups):
            g["betas"] = tuple(g["betas"])
            for p in g["params"]:
                if id(p) not in position:
                    raise ValueError(f"parameter group {gi} holds a tensor of shape {tuple(p.shape)} that is not a "
                                     "parameter of the flattened module")
                group_of[position[id(p)]] = gi
        # the run table: contiguous ranges of flat.flat[:n_live] and their group (-1: frozen); a parameter's padding
        # belongs to its run, so every run starts at a multiple of 4
        begin, group = [0], [-1]
        for i, (_, _, off, _) in zip(flat.live_index, flat.live):
            gi = group_of.get(i, -1)
            if group[-1] != gi:
                begin.append(off), group.append(gi)
        if len(group) > 1 and begin[1] == 0:      # the first parameter opened a run at 0
            begin, group = begin[1:], group[1:]
        begin.append(flat.n_live)
        self._run_begin = torch.tensor(begin, dtype=torch.int64).to(dev)
        self._run_group = torch.tensor(group, dtype=torch.int32).to(dev)
        self._table = ops.adam_group_table(self.param_groups, dev)
        for g, row in zip(self.param_groups, self._table):
            g.row = row
        self.flat = flat
        self.m = torch.zeros_like(flat.grad)
        self.v = torch.zeros_like(flat.grad)
        self.t = 0                            # host count of step() calls and replays, skipped steps included
        self.t_dev = torch.zeros(1, device=dev, dtype=torch.int32)  # Adam's step count: the kernels read this one
        self._max_norm_dev = torch.zeros((), device=dev)
        self.max_grad_norm, self.skip_nonfinite = max_grad_norm, bool(skip_nonfinite)
        self.grad_norm = torch.zeros((), device=dev)
        self.skipped_steps = torch.zeros((), device=dev, dtype=torch.int32)
        self._norm_ws = ops.grad_norm_workspace(flat.n_live, flat.grad)
        self._early_done, self._early_keep, self._comm = False, [], None
        self._accumulate_steps = int(accumulate_steps)
        self._no_sync = False
        self._micro = 0              # backward passes of the open accumulation window (no_sync blocks / GraphedStep)
        self._gather_adds = False    # the window's earlier gradients are summed in flat.grad (GraphedStep): gathers add
        if os.environ.get("B200NP_BUCKETS", "1") != "0" and flat.n_early and flat.n_early < flat.n_live:
            from . import engine
            ref = weakref.ref(self)

            def hook(ptr):
                me = ref()
                if me is None:
                    engine.PRE_TRUNK_BACKWARD_HOOKS.remove(hook)
                elif ptr in me.flat.trigger_ptrs and not me._no_sync:
                    me._early_bucket()
            engine.PRE_TRUNK_BACKWARD_HOOKS.append(hook)

    def add_param_group(self, param_group):
        if hasattr(self, "_table"):
            raise RuntimeError("FusedAdam's parameter groups are fixed at construction (the kernel's run table is laid "
                               "out with the flat parameters); pass every group to the constructor")
        super().add_param_group(param_group)

    @property
    def accumulate_steps(self):
        """Backward passes per optimizer step (fixed at construction)."""
        return self._accumulate_steps

    @contextlib.contextmanager
    def no_sync(self):
        """As DistributedDataParallel.no_sync(): backward passes inside start no gradient exchange, and their gradients
        sum in `p.grad`.  Run every backward pass of an accumulation window but the last one inside it."""
        prev, self._no_sync = self._no_sync, True
        self._micro += 1
        try:
            yield
        finally:
            self._no_sync = prev

    @property
    def lr(self):
        return self.param_groups[0]["lr"]

    @lr.setter
    def lr(self, value):
        self.param_groups[0]["lr"] = value

    @property
    def betas(self):
        return tuple(self.param_groups[0]["betas"])

    @betas.setter
    def betas(self, value):
        self.param_groups[0]["betas"] = tuple(value)

    @property
    def eps(self):
        return self.param_groups[0]["eps"]

    @eps.setter
    def eps(self, value):
        self.param_groups[0]["eps"] = value

    @property
    def wd(self):
        return self.param_groups[0]["weight_decay"]

    @wd.setter
    def wd(self, value):
        self.param_groups[0]["weight_decay"] = value

    @property
    def max_grad_norm(self):
        return self._max_grad_norm

    @max_grad_norm.setter
    def max_grad_norm(self, value):
        if value is not None:
            self._max_norm_dev.fill_(float(value))
        self._max_grad_norm = value

    def zero_grad(self, set_to_none=False):
        self.flat.zero_grad()
        self._early_done = False
        self._micro, self._gather_adds = 0, False

    def _window_closed(self, what):
        if self._micro:
            raise RuntimeError(f"{what}() between the backward passes of a gradient-accumulation window: the window's "
                               "gradients are not part of the saved state; call it after the window's step()")

    def _early_bucket(self):
        """The gradients laid out before the encoder CNN's: gather + all-reduce on the communication stream."""
        if dist.world_size() == 1:
            return
        if self._early_done:
            raise RuntimeError("a second backward pass before step() outside no_sync(): its gradients would miss the "
                               "exchange the first one started; run all but the last backward pass of a gradient-"
                               "accumulation window inside `with opt.no_sync():`")
        f = self.flat
        main = torch.cuda.current_stream()
        if self._comm is None:
            self._comm = torch.cuda.Stream(priority=-1)
        self._comm.wait_stream(main)
        with torch.cuda.stream(self._comm):
            f.gather_grads(0, f.n_early, keep=self._early_keep, skip_missing=True, accumulate=self._gather_adds)
            dist.all_reduce_sum(f.grad[:f.n_early])
        self._early_done = True

    def step(self):
        from .engine import nvtx_range
        with nvtx_range("b200np.adam.step"):
            self._step()

    def _step(self):
        f = self.flat
        world = dist.world_size()
        acc = self._gather_adds
        if world > 1 and self._early_done:
            # whatever the early bucket did not find (a parameter whose gradient arrived later: none on the shipped
            # models) is exchanged on its own, so the result never depends on the bucket boundary being right
            late_early = [(p, off, k) for _, p, off, k in f.live
                          if off < f.n_early and p.grad is not None and p.grad.data_ptr() != f.grad[off:off + k].data_ptr()]
            torch.cuda.current_stream().wait_stream(self._comm)   # before anything else writes into the early segment
            self._early_keep.clear()
            f.gather_grads(accumulate=acc)
            dist.all_reduce_sum(f.grad[f.n_early:f.n_live])
            for _, off, k in late_early:
                dist.all_reduce_sum(f.grad[off:off + k])
            self._early_done = False
        else:
            f.gather_grads(accumulate=acc)
            if world > 1:
                dist.all_reduce_grads(f.grad)
        self.t += 1
        self._micro, self._gather_adds = 0, False
        scale = 1.0 / (world * self.accumulate_steps)     # the window's mean gradient over every rank
        # the step counter, every hyperparameter and the clip / skip decision are kept on the device so that a
        # captured CUDA graph of the whole step stays valid
        clip = self.max_grad_norm is not None
        if clip or self.skip_nonfinite:
            ops.grad_norm(f.grad, f.n_live, self.grad_norm, self._norm_ws, scale)
        ops.adam_step_groups(f.flat, f.grad, self.m, self.v, f.n_live, self._table, self._run_begin, self._run_group,
                             self.t_dev, scale, max_norm=self._max_norm_dev if clip else None,
                             norm=self.grad_norm, skipped=self.skipped_steps if self.skip_nonfinite else None)

    # the rest of a torch.optim.Adam param_group, at the values that describe what the fused kernel computes
    _GROUP_FLAGS = dict(amsgrad=False, maximize=False, foreach=None, capturable=False, differentiable=False, fused=None)
    _HYPER = ("lr", "betas", "eps", "weight_decay", "decoupled_weight_decay")

    def _ids(self):
        """torch's checkpoint numbering: consecutive over the groups' `params` lists, in group order.  Yields
        (group index, id, position in module.parameters())."""
        position = {id(p): i for i, p in enumerate(self.flat.params)}
        k = 0
        for gi, g in enumerate(self.param_groups):
            for p in g["params"]:
                yield gi, k, position[id(p)]
                k += 1

    def state_dict(self):
        """The optimizer state in exactly the structure `torch.optim.Adam(groups).state_dict()` (or `AdamW`) has, so
        either optimizer can resume from the other's checkpoint.  `state` is keyed by torch's ids (consecutive over
        the groups' `params`, in group order; for the default single group, the position in `module.parameters()`).
        Each live parameter of a group gets `step` (0-dim float32 CPU tensor) and clones of its slices of the
        moments.  Parameters that never receive a gradient, frozen ones, and every parameter before the first step
        get no entry, as in torch.  Each group carries its own hyperparameters and the keys a scheduler added to it
        (`initial_lr`).  Reading the step count is one 4-byte device-to-host copy.  Raises between the backward passes
        of a gradient-accumulation window."""
        self._window_closed("state_dict")
        f = self.flat
        t = int(self.t_dev.item())
        live = dict(zip(f.live_index, f.live))
        state = {}
        if t > 0:
            for _, k, i in self._ids():
                if i in live:
                    _, p, off, n = live[i]
                    state[k] = {"step": torch.tensor(float(t), dtype=torch.float32),
                                "exp_avg": self.m[off:off + n].view_as(p).clone(),
                                "exp_avg_sq": self.v[off:off + n].view_as(p).clone()}
        groups, k = [], 0
        for g in self.param_groups:
            group = {key: v for key, v in g.items() if key != "params"}
            group.update(lr=float(g["lr"]), betas=tuple(g["betas"]), eps=g["eps"], weight_decay=g["weight_decay"],
                         decoupled_weight_decay=bool(g["decoupled_weight_decay"]), **self._GROUP_FLAGS,
                         params=list(range(k, k + len(g["params"]))))
            k += len(g["params"])
            groups.append(group)
        return {"state": state, "param_groups": groups}

    def load_state_dict(self, state_dict):
        """Resume from a `state_dict()` of this class or of `torch.optim.Adam` / `AdamW` over the same parameter
        groups (same count, same sizes, same order).

        The moments are written into the existing `m` / `v` (one `multi_copy` launch per 64 parameters) and the step
        count into `t_dev`, all in place, so a CUDA graph captured over these buffers stays valid.  A parameter
        without a state entry gets zero moments.  Each group's hyperparameters are taken from the checkpoint, as torch
        does, and so are the extra group keys a scheduler keeps there (`initial_lr`).
        The whole checkpoint is checked before anything is written; `ValueError` if it does not fit these groups or
        needs something the flat kernel does not do (one step counter, no amsgrad / maximize).  `RuntimeError` between
        the backward passes of a gradient-accumulation window."""
        self._window_closed("load_state_dict")
        f = self.flat
        groups = state_dict["param_groups"]
        if len(groups) != len(self.param_groups):
            raise ValueError(f"FusedAdam has {len(self.param_groups)} parameter group(s); the checkpoint has "
                             f"{len(groups)}")
        for gi, (group, mine) in enumerate(zip(groups, self.param_groups)):
            for flag in ("amsgrad", "maximize"):
                if group.get(flag, False):
                    raise ValueError(f"the checkpoint was written with {flag}=True; FusedAdam implements Adam / AdamW "
                                     "only")
            if len(group["params"]) != len(mine["params"]):
                raise ValueError(f"parameter group {gi} holds {len(mine['params'])} parameters, the checkpoint's "
                                 f"{len(group['params'])}")
        saved = [pid for group in groups for pid in group["params"]]
        extra = set(state_dict["state"]) - set(saved)
        if extra:
            raise ValueError(f"the checkpoint has state for ids {sorted(extra)}, which are in none of its groups")
        live = dict(zip(f.live_index, f.live))
        found, steps = {}, set()
        for (_, k, i), pid in zip(self._ids(), saved):
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
        own = {"params", "param_names", *self._HYPER, *self._GROUP_FLAGS}
        for g, group in zip(self.param_groups, groups):
            for k in [k for k in g if k not in own]:
                del g[k]
            g.update((k, v) for k, v in group.items() if k not in own)
            g["lr"], g["eps"], g["weight_decay"] = float(group["lr"]), float(group["eps"]), float(group["weight_decay"])
            g["betas"] = tuple(float(b) for b in group["betas"])
            # a checkpoint older than the key leaves the group's own setting, as torch's Adam / AdamW keep their own
            g["decoupled_weight_decay"] = bool(group.get("decoupled_weight_decay", g["decoupled_weight_decay"]))


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

    Building a graph runs `warmup` real steps and the capture itself on the model; parameters, Adam moments, the
    step counter, the skip counter, the flat gradient and the position in an accumulation window are snapshotted
    before and restored afterwards, so constructing the object (or meeting a new shape, mid-window too) does NOT
    advance training.  Every group's hyperparameters and `max_grad_norm` are read from device memory, so a scheduler,
    an assignment or `load_state_dict` changes them without a recapture.  A graph holds only whether clipping and
    skipping are on; when that has changed since the capture, the graph is recaptured, in the same way, before its
    next replay.

    Gradient accumulation (`opt.accumulate_steps` = k > 1, see FusedAdam): each call is one micro-batch and returns
    its loss, and the k-th call of a window is the optimizer step.  Per batch shape up to three graphs ("roles") are
    captured on first use: "first" zeroes the gradients, runs forward, loss and backward and copies the gradients
    into `flat.grad`; "middle" does the same but adds them; "last" runs forward, loss and backward, adds the gradients
    and runs the two-bucket exchange, the norm and Adam.  Shapes may differ within a window.  Only "last" graphs hold
    the clipping / skipping switch, so only they are recaptured when it changes.  With k = 1 the one role is "last",
    the step described above.

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
        self._staged = None          # (shape entry, the prefetched batch's tensors)
        self.cache = {}
        self.pool = torch.cuda.graph_pool_handle()
        from . import engine
        # warm-up and capture run on one high-priority stream: the engine's companion streams (decoder CNN, weight
        # gradients) rank below it, and the captured kernel nodes keep those priorities
        self.side = torch.cuda.Stream(priority=engine.MAIN_PRIORITY if engine.USE_PRIORITIES else 0)
        self.graph = self.loss = None
        if example_batch is not None:
            ent = self._graph(self._entry(example_batch))
            self.graph, self.loss = ent["graph"], ent["loss"]

    @staticmethod
    def _key(batch):
        return tuple(tuple(t.shape) for t in batch)

    def _hyper(self):
        o = self.opt
        return (o.max_grad_norm is not None, o.skip_nonfinite)

    def _role(self):
        """The role of the next call in the accumulation window."""
        o = self.opt
        return "last" if o._micro >= o.accumulate_steps - 1 else "middle" if o._micro else "first"

    def _entry(self, batch):
        """The static and staging inputs of `batch`'s shape, with the graph of the next call's role captured."""
        key = self._key(batch)
        ent = self.cache.get(key)
        if ent is None:
            dev = self.opt.flat.flat.device
            ent = {"static": [torch.empty(t.shape, device=dev, dtype=t.dtype) for t in batch],
                   "stage": [torch.empty(t.shape, device=dev, dtype=t.dtype) for t in batch], "roles": {}}
            for s, t in zip(ent["static"], batch):
                s.copy_(t)
            self.cache[key] = ent
        self._graph(ent)
        return ent

    def _graph(self, ent):
        """The graph of the next call's role on the shape entry `ent`, captured on first use."""
        role = self._role()
        g = ent["roles"].get(role)
        if g is None:
            g = ent["roles"][role] = {"static": ent["static"], "role": role}
            self._capture(g)
        return g

    def _capture(self, ent):
        """Warm up and capture `ent`'s role on its static inputs, recording the hyperparameters a "last" graph holds."""
        opt, f = self.opt, self.opt.flat
        old = ent.get("graph")
        snap = (f.flat.clone(), f.grad.clone(), opt.m.clone(), opt.v.clone(), opt.t_dev.clone(),
                opt.skipped_steps.clone(), opt.grad_norm.clone(), opt.t, opt._micro, opt._gather_adds)
        cur = torch.cuda.current_stream()
        self.side.wait_stream(cur)
        with torch.cuda.stream(self.side):
            for _ in range(self.warmup):
                self._eager(ent["static"], ent["role"])
        cur.wait_stream(self.side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=self.side, pool=self.pool):
            loss = self._eager(ent["static"], ent["role"])
        # neither the warm-up steps nor the capture may advance training or change the open window's gradients
        for t, saved in zip((f.flat, f.grad, opt.m, opt.v, opt.t_dev, opt.skipped_steps, opt.grad_norm), snap):
            t.copy_(saved)
        opt.t, opt._micro, opt._gather_adds = snap[7:]
        torch.cuda.synchronize()
        ent["graph"], ent["loss"] = graph, loss
        ent["hyper"] = self._hyper() if ent["role"] == "last" else None
        if old is not None and self.graph is old:     # recaptured the example batch's graph
            self.graph, self.loss = graph, loss

    def _eager(self, static, role="last"):
        cx, cy, tx, ty = static
        opt = self.opt
        if role == "last" and opt.accumulate_steps == 1:
            opt.zero_grad()
        else:
            # autograd hands over this micro-batch's gradients alone; the window's earlier ones are in flat.grad
            opt.flat.zero_grad()
            opt._gather_adds = role != "first"
        mu, _, _ = self.model(cx, cy, tx)
        loss = self.lossf.calc_loss(mu, None, ty)
        if role == "last":
            loss.backward()
            opt.step()
        else:
            with opt.no_sync():
                loss.backward()
            opt.flat.gather_grads(accumulate=opt._gather_adds)
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
        g = self._graph(ent)
        if g["hyper"] is not None and g["hyper"] != self._hyper():
            # the graph holds whether the norm pass runs and what the Adam launch does with it
            self._capture(g)
        self._staged = None
        self.ev_free.record(cur)
        g["graph"].replay()
        opt = self.opt
        if g["role"] == "last":
            opt.t += 1
            opt._micro, opt._gather_adds = 0, False
            opt._opt_called = True     # a replay of the step is an optimizer step: torch's LR schedulers check for one
        else:
            opt._micro += 1
            opt._gather_adds = True
        if next_batch is not None:
            self.prefetch(next_batch)
        return g["loss"]

    def state_dict(self):
        """What a resumed run needs: `{"model": model.state_dict(), "optimizer": opt.state_dict()}`."""
        return {"model": self.model.state_dict(), "optimizer": self.opt.state_dict()}

    def load_state_dict(self, state_dict):
        """Load weights and optimizer state in place: the captured graphs keep their buffers and read the loaded
        hyperparameters from device memory, so nothing is recaptured.  The optimizer goes first: it checks the
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
