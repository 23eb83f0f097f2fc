"""Training-step drivers for the drop-in models.

`eager_step` is the per-batch body of the reference trainer (FoodRec/common/trainer.py:177-224):
zero_grad, `calculate_loss`, sum, backward, optimizer step.  `GraphedTrainStep` runs the same body
as ONE CUDA-graph replay: the step is ~100 small launches (the propagation kernels are tens of
microseconds each at Allrecipes scale), so without a graph it is bound by CPU launch latency, not
by the GPU.  Numerics are identical to the eager body (same kernels, same order).
"""
from __future__ import annotations

import ctypes as _ctypes
import warnings

import torch


def mark_parameters_updated(model):
    """Invalidate everything cached from the parameter values (propagated evaluation tables, SCHGN's
    user-independent scorer tables).  Needed because a CUDA-graph replay rewrites the parameters in
    place without going through ATen: neither `data_ptr` nor `_version` changes."""
    model._param_generation = getattr(model, "_param_generation", 0) + 1
    if getattr(model, "_eval_cache", None) is not None:
        model._eval_cache = None


def eager_step(model, optimizer, batch, grad_hook=None):
    optimizer.zero_grad()
    losses = model.calculate_loss(batch)
    loss = sum(losses) if isinstance(losses, tuple) else losses
    loss.backward()
    if grad_hook is not None:
        grad_hook(model)
    optimizer.step()
    mark_parameters_updated(model)
    return losses


def allreduce_mean_grads(group=None):
    """Gradient hook for data-parallel replicas: one NCCL all-reduce per dense gradient (capturable)."""
    import torch.distributed as dist
    world = dist.get_world_size(group)

    def hook(model):
        for p in model.parameters():
            if p.grad is not None:
                dist.all_reduce(p.grad, group=group)
                p.grad.div_(world)
    return hook


class OverlappedGradAllReduce:
    """Data-parallel gradient averaging that overlaps the backward: every parameter's gradient is
    all-reduced (NCCL, AVG) on a communication stream as soon as autograd has accumulated it, so the
    user-table gradient (ready after the user-item backward) travels while the item-side graphs are
    still back-propagating.  Call the object between `backward()` and `optimizer.step()` to join the
    streams.  Works under CUDA-graph capture (the communication stream becomes a parallel branch)."""

    def __init__(self, model, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        dev = next(model.parameters()).device
        self.comm = torch.cuda.Stream(device=dev)
        self.handles = [p.register_post_accumulate_grad_hook(self._hook) for p in model.parameters() if p.requires_grad]

    def _hook(self, p):
        cur = torch.cuda.current_stream()
        self.comm.wait_stream(cur)
        with torch.cuda.stream(self.comm):
            self.dist.all_reduce(p.grad, op=self.dist.ReduceOp.AVG, group=self.group)

    def __call__(self, model=None):
        torch.cuda.current_stream().wait_stream(self.comm)

    def remove(self):
        for h in self.handles:
            h.remove()


def _non_negative(cls, **values):
    for k, v in values.items():
        if not float(v) >= 0.0:
            raise ValueError(f"{cls}: invalid {k} {v!r}")


def _unsupported(cls, **options):
    """Options that torch's optimizer has but the reference's optimizer factory never sets: only the default."""
    for k, (v, default) in options.items():
        if v != default:
            raise ValueError(f"{cls}: {k}={v!r} is not supported (only {default!r}, torch's default)")


class _FusedOptimizer(torch.optim.Optimizer):
    """One `fr_optim_step` call per parameter group: dense update of every parameter that has a gradient, in one
    multi-tensor launch per 64 tensors, step counter and learning rate on the device, capturable in a CUDA graph.

    `group["lr"]` stays the source of truth (an lr scheduler writes it).  Its device copy is refreshed by
    `refresh_lr()`, which an eager `step()` calls first and `GraphedTrainStep` calls before each replay; a captured
    `step()` reads the device copy at every replay and never writes it."""

    _rule = None            # FR_OPTIM_* of include/foodrec_b200.h
    _state_keys = ()        # torch's state keys of the learner, in fr_optim_tensor's state0, state1 order
    _has_step = False       # the rule keeps a step counter (Adam, Adagrad)

    def __init__(self, params, defaults):
        _non_negative(type(self).__name__, lr=defaults["lr"], weight_decay=defaults["weight_decay"],
                      eps=defaults.get("eps", 0.0))
        super().__init__(params, defaults)
        self._dev_state = {}

    def _hyper(self, group):
        raise NotImplementedError

    @torch.no_grad()
    def refresh_lr(self):
        """Copy each group's `lr` to its device scalar where it has changed since the last copy.  Asynchronous (one
        fill on the current stream) and nothing at all while the value is unchanged.  Call it outside a capture."""
        for gi, group in enumerate(self.param_groups):
            ds = self._dev_state.get(gi)
            lr = float(group["lr"])
            if ds is None or lr == ds["lr_host"]:
                continue
            _non_negative(type(self).__name__, lr=lr)
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError(f"{type(self).__name__}.refresh_lr() inside a CUDA-graph capture: the write would "
                                   "be frozen into the graph; call it before each replay instead")
            ds["lr"].fill_(lr)
            ds["lr_host"] = lr

    def _group_state(self, gi, group, dev, capturing):
        ds = self._dev_state.get(gi)
        if ds is None:
            if capturing:
                raise RuntimeError(f"{type(self).__name__}: take one eager step() before capturing one, so the device "
                                   "state exists outside the graph")
            lr = float(group["lr"])
            ds = self._dev_state[gi] = dict(
                lr=torch.full((1,), lr, dtype=torch.float64, device=dev), lr_host=lr,
                step=torch.zeros(1, dtype=torch.int32, device=dev) if self._has_step else None,
                scal=torch.zeros(2, dtype=torch.float32, device=dev))
        return ds

    @torch.no_grad()
    def step(self, closure=None):
        from . import _lib
        name = type(self).__name__
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        capturing = torch.cuda.is_current_stream_capturing()
        if not capturing:
            self.refresh_lr()
        for gi, group in enumerate(self.param_groups):
            ps = [p for p in group["params"] if p.grad is not None]
            if not ps:
                continue
            dev = ps[0].device
            if dev.type != "cuda":
                raise _lib.FoodRecError(f"{name} needs CUDA parameters (foodrec_b200 has no CPU path)")
            ds = self._group_state(gi, group, dev, capturing)
            tensors = (_lib.OptimTensor * len(ps))()
            grads = []              # contiguous copies stay alive until the launch is enqueued
            for t, p in zip(tensors, ps):
                if p.dtype != torch.float32 or not p.is_contiguous() or p.grad.is_sparse:
                    raise _lib.FoodRecError(f"{name} handles contiguous fp32 parameters with dense gradients")
                st = self.state[p]
                if not st and self._state_keys:
                    if capturing:
                        raise RuntimeError(f"{name}: a parameter without state inside a CUDA-graph capture; take one "
                                           "eager step() with every parameter's gradient set first")
                    for k in self._state_keys:
                        st[k] = torch.zeros_like(p, memory_format=torch.preserve_format)
                g = p.grad if p.grad.is_contiguous() else p.grad.contiguous()
                grads.append(g)
                s = [st[k].data_ptr() for k in self._state_keys] + [None, None]
                t.param, t.grad, t.state0, t.state1 = p.data_ptr(), g.data_ptr(), s[0], s[1]
                t.n = p.numel()
            hyper = self._hyper(group)
            step = None if ds["step"] is None else ds["step"].data_ptr()
            _lib.check(_lib.lib.fr_optim_step(self._rule, tensors, len(ps), _ctypes.byref(hyper), ds["lr"].data_ptr(),
                                              step, ds["scal"].data_ptr(), _lib.stream_ptr()), "fr_optim_step")
        return loss


class FusedAdam(_FusedOptimizer):
    """`torch.optim.Adam(params, lr, betas, eps, weight_decay)` (amsgrad = False: the reference's optimizer,
    FoodRec/common/trainer.py:142-144) as ONE multi-tensor launch of this library (`fr_optim_step`, the update of
    `fr_adam_step`).  `weight_decay` is torch's L2 term g + wd p, not AdamW's.  State keys (`exp_avg`, `exp_avg_sq`)
    are those of torch's Adam, so optimizer checkpoints carry over except for `step`."""

    _rule, _state_keys, _has_step = 0, ("exp_avg", "exp_avg_sq"), True        # FR_OPTIM_ADAM

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, amsgrad=False, *,
                 maximize=False):
        _unsupported("FusedAdam", amsgrad=(amsgrad, False), maximize=(maximize, False))
        if not (0.0 <= betas[0] < 1.0 and 0.0 <= betas[1] < 1.0):
            raise ValueError(f"FusedAdam: invalid betas {betas!r}")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))

    def _hyper(self, group):
        from . import _lib
        b1, b2 = group["betas"]
        return _lib.OptimHyper(beta1=float(b1), beta2=float(b2), eps=float(group["eps"]),
                               weight_decay=float(group["weight_decay"]))


class FusedSGD(_FusedOptimizer):
    """`torch.optim.SGD(params, lr, weight_decay=weight_decay)` without momentum, as the reference's factory builds it:
    p += -lr (g + wd p).  No state."""

    _rule = 1                                                                   # FR_OPTIM_SGD

    def __init__(self, params, lr=1e-3, momentum=0, dampening=0, weight_decay=0, nesterov=False, *, maximize=False):
        _unsupported("FusedSGD", momentum=(momentum, 0), dampening=(dampening, 0), nesterov=(nesterov, False),
                     maximize=(maximize, False))
        super().__init__(params, dict(lr=lr, weight_decay=weight_decay))

    def _hyper(self, group):
        from . import _lib
        return _lib.OptimHyper(weight_decay=float(group["weight_decay"]))


class FusedAdagrad(_FusedOptimizer):
    """`torch.optim.Adagrad(params, lr, weight_decay=weight_decay)` (lr_decay = 0, initial_accumulator_value = 0), which
    torch cannot capture in a CUDA graph (it reads its step on the host).  State key `sum`; the step counter lives on
    the device."""

    _rule, _state_keys, _has_step = 2, ("sum",), True                           # FR_OPTIM_ADAGRAD

    def __init__(self, params, lr=1e-2, lr_decay=0, weight_decay=0, initial_accumulator_value=0, eps=1e-10, *,
                 maximize=False):
        _unsupported("FusedAdagrad", lr_decay=(lr_decay, 0), initial_accumulator_value=(initial_accumulator_value, 0),
                     maximize=(maximize, False))
        super().__init__(params, dict(lr=lr, eps=eps, weight_decay=weight_decay))

    def _hyper(self, group):
        from . import _lib
        return _lib.OptimHyper(eps=float(group["eps"]), weight_decay=float(group["weight_decay"]))


class FusedRMSprop(_FusedOptimizer):
    """`torch.optim.RMSprop(params, lr, weight_decay=weight_decay)` (momentum = 0, not centred).  State key
    `square_avg`."""

    _rule, _state_keys = 3, ("square_avg",)                                     # FR_OPTIM_RMSPROP

    def __init__(self, params, lr=1e-2, alpha=0.99, eps=1e-8, weight_decay=0, momentum=0, centered=False, *,
                 maximize=False):
        _unsupported("FusedRMSprop", momentum=(momentum, 0), centered=(centered, False), maximize=(maximize, False))
        _non_negative("FusedRMSprop", alpha=alpha)
        super().__init__(params, dict(lr=lr, alpha=alpha, eps=eps, weight_decay=weight_decay))

    def _hyper(self, group):
        from . import _lib
        return _lib.OptimHyper(alpha=float(group["alpha"]), eps=float(group["eps"]),
                               weight_decay=float(group["weight_decay"]))


_LEARNERS = {"adam": FusedAdam, "sgd": FusedSGD, "adagrad": FusedAdagrad, "rmsprop": FusedRMSprop}


def build_optimizer(config, params):
    """The reference trainer's optimizer factory (FoodRec/common/trainer.py:137-154, MMRec's `_build_optimizer`) on
    the fused optimizers: `config["learner"]`, matched case-insensitively, picks Adam, SGD, Adagrad or RMSprop with
    `lr = config["learning_rate"]` and `weight_decay = config["weight_decay"]`, every other option at torch's default.
    An unknown learner gives Adam with `lr` only, as the reference does (it logs a warning)."""
    learner = str(config["learner"]).lower()
    cls = _LEARNERS.get(learner)
    if cls is None:
        warnings.warn(f"unrecognized learner {config['learner']!r}: using Adam", stacklevel=2)
        return FusedAdam(params, lr=config["learning_rate"])
    return cls(params, lr=config["learning_rate"], weight_decay=config["weight_decay"])


class GraphedTrainStep:
    """Capture `zero_grad -> calculate_loss -> backward -> optimizer.step` once, replay per batch.

    `example_batch` fixes the batch shapes (the reference's DataLoader yields a short last batch:
    run that one through `eager_step`).  The optimizer must be capturable: one of the fused
    optimizers of this module (`build_optimizer`), or e.g. `torch.optim.Adam(..., capturable=True)`.
    `__call__(batch)` copies the batch tensors (host pinned or device) into the static inputs,
    replays, and returns the tuple of loss tensors (device, overwritten by the next call).

    Learning-rate schedules: a fused optimizer keeps `lr` on the device, and each call refreshes that
    copy from `group["lr"]` before the replay, so a `LambdaLR` stepped between calls takes effect.
    Any other optimizer froze its float `lr` into the graph at capture: a call after a group's `lr`
    has changed raises instead of silently replaying the old value.
    """

    def __init__(self, model, optimizer, example_batch: dict, keys=None, warmup: int = 3, grad_hook=None):
        self.model, self.optimizer = model, optimizer
        dev = next(model.parameters()).device
        self.keys = list(keys) if keys is not None else list(example_batch.keys())
        self.static = {k: torch.empty_like(example_batch[k], device=dev).copy_(example_batch[k]) for k in self.keys}
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(warmup):  # allocates lazily-created workspaces and optimizer state outside the graph
                eager_step(model, optimizer, self.static, grad_hook)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        optimizer.zero_grad(set_to_none=True)
        with torch.cuda.graph(self.graph):
            losses = model.calculate_loss(self.static)
            loss = sum(losses) if isinstance(losses, tuple) else losses
            loss.backward()
            if grad_hook is not None:
                grad_hook(model)
            optimizer.step()
            self.losses = losses if isinstance(losses, tuple) else (losses,)
            # every term in one device vector (inside the graph), so a trainer reads them with ONE device->host copy
            self.loss_vec = torch.stack([l.detach().reshape(()).float() for l in self.losses])
        # a tensor lr is read on the device at every replay; a float one is what the capture froze
        self.lr_at_capture = [None if torch.is_tensor(g["lr"]) else g["lr"] for g in optimizer.param_groups]

    def _follow_lr(self):
        refresh = getattr(self.optimizer, "refresh_lr", None)
        if refresh is not None:
            refresh()
            return
        for k, (g, lr0) in enumerate(zip(self.optimizer.param_groups, self.lr_at_capture)):
            if lr0 is not None and g["lr"] != lr0:
                raise RuntimeError(
                    f"param group {k}: lr changed from {lr0} to {g['lr']} since the capture, but "
                    f"{type(self.optimizer).__name__} froze it into the graph; use a fused optimizer of "
                    "foodrec_b200.train (its lr lives on the device) or capture again")

    def __call__(self, batch: dict):
        """`batch` tensors may live on the device or in (pinned) host memory: they are copied straight into the
        static inputs of the graph."""
        self._follow_lr()
        for k in self.keys:
            self.static[k].copy_(batch[k], non_blocking=True)
        self.graph.replay()
        mark_parameters_updated(self.model)
        return self.losses

    def loss_values(self):
        """The loss terms of the last replay as python floats: one synchronising device->host copy for all of them
        (the reference trainer's per-term `.item()`, trainer.py:186, costs one round trip per term)."""
        return self.loss_vec.tolist()


class DeviceBatchSampler:
    """Training batches assembled on the device: a shuffled pass over the training interactions with one
    uniformly drawn negative per sample (`fr_sample_negatives`), as `TrainDataLoader` + `DataLoader(shuffle=True)`
    produce them (FoodRec/utils/dataloader.py:50-77,145-151) -- without the per-sample python rejection loop and
    without a host round trip.  Negatives avoid the user's training items and, when the dataset carries them,
    their validation / test items (`validTestRatings`; else `validRatings` mapped through `valid_users`, and
    `testRatings`), like the reference.  Same distribution, a
    different random stream: parity is statistical (SURVEY.md 8f-3)."""

    def __init__(self, dataset, batch_size: int, device, seed: int = 0, drop_last: bool = False):
        import numpy as np
        coo = dataset.train_coo_matrix
        self.n_items, self.batch_size, self.device = int(dataset.n_items), int(batch_size), torch.device(device)
        u = np.asarray(coo.row, dtype=np.int64)
        i = np.asarray(coo.col, dtype=np.int64)
        self.users = torch.from_numpy(u).to(self.device)
        self.items = torch.from_numpy(i).to(self.device)
        eu, ei = [u], [i]
        n_users = int(dataset.n_users)
        vt = getattr(dataset, "validTestRatings", None)
        if vt is not None:
            # the reference's own exclusion structure: dict user -> set of held-out items
            # (FoodRec/utils/dataset.py:35,93-113, read by utils/dataloader.py:145-151)
            us = np.fromiter((uu for uu, items in vt.items() for _ in items), dtype=np.int64)
            it = np.fromiter((j for items in vt.values() for j in items), dtype=np.int64)
            eu.append(us)
            ei.append(it)
        else:
            # `validRatings` is POSITIONAL in the reference (paired with `valid_users`: users without validation
            # rows are skipped, dataset.py:32,115-135); `testRatings` has one list per user
            for name, owners in (("validRatings", "valid_users"), ("testRatings", "test_users")):
                lists = getattr(dataset, name, None)
                if lists is None:
                    continue
                ids = getattr(dataset, owners, None)
                if ids is None:
                    if len(lists) != n_users:
                        raise ValueError(f"dataset.{name} has {len(lists)} lists for {n_users} users and no "
                                         f"dataset.{owners} to map them: cannot attribute held-out items")
                    ids = np.arange(n_users, dtype=np.int64)
                ids = np.asarray(ids, dtype=np.int64)
                if ids.shape[0] != len(lists):
                    raise ValueError(f"dataset.{owners} and dataset.{name} differ in length")
                lens = np.fromiter((len(x) for x in lists), dtype=np.int64, count=len(lists))
                eu.append(np.repeat(ids, lens))
                ei.append(np.fromiter((j for x in lists for j in x), dtype=np.int64, count=int(lens.sum())))
        keys = np.unique(np.concatenate(eu) * self.n_items + np.concatenate(ei))
        ptr = np.zeros(int(dataset.n_users) + 1, dtype=np.int64)
        np.cumsum(np.bincount(keys // self.n_items, minlength=int(dataset.n_users)), out=ptr[1:])
        self.excl_ptr = torch.from_numpy(ptr).to(self.device)
        self.excl_idx = torch.from_numpy((keys % self.n_items).astype(np.int32)).to(self.device)
        self.seed, self.drop_last, self._step = int(seed), drop_last, 0
        self._fail = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._gen = torch.Generator(device=self.device)
        self._gen.manual_seed(self.seed)

    def __len__(self):
        n = self.users.numel()
        return n // self.batch_size if self.drop_last else -(-n // self.batch_size)

    def negatives(self, users: torch.Tensor) -> torch.Tensor:
        from . import _lib
        users = users.to(self.device, torch.int64).contiguous()
        out = torch.empty_like(users)
        self._step += 1
        _lib.check(_lib.lib.fr_sample_negatives(
            self.excl_ptr.data_ptr(), self.excl_idx.data_ptr(), users.data_ptr(), users.numel(), self.n_items,
            self.seed & (2 ** 64 - 1), self._step, out.data_ptr(), self._fail.data_ptr(), _lib.stream_ptr()),
            "fr_sample_negatives")
        return out

    def failures(self) -> int:
        """Samples that found no admissible item so far (a user who interacted with almost every item)."""
        return int(self._fail.item())

    def __iter__(self):
        perm = torch.randperm(self.users.numel(), device=self.device, generator=self._gen)
        for b in range(len(self)):
            sel = perm[b * self.batch_size:(b + 1) * self.batch_size]
            u = self.users[sel]
            yield {"u_id": u, "pos_i_id": self.items[sel], "neg_i_id": self.negatives(u)}
