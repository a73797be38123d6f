"""Training path of the drop-in modules: one autograd bridge for LightweightUNet and OptimizedUNet, and the fused optimizer tail.

Reference call sequence (optimized_train.py:197-236, fp32 branch :220-233):
    optimizer.zero_grad(set_to_none=True); outputs = model(inputs); loss = criterion(outputs, targets)
    loss.backward(); clip_grad_norm_(model.parameters(), 1.0); optimizer.step()
`model(inputs)` lands in `train_forward` when autograd is recording; the gradients autograd asks for (every parameter that
requires one, and the input image when it does) come back through `torch.autograd.Function.backward`, i.e. they land in
`param.grad` / `x.grad` the normal way (wandb.watch hooks keep working).  Frozen parameters cost no kernel work.  The bridge owns
the gradient-delivery policy; each model supplies only its own forward and backward (`_train_forward`, `_train_backward`).
`FusedAdamW` is a `torch.optim.Optimizer` with AdamW's constructor that keeps parameters, gradients and both moments in flat
buffers and runs clip + update as two kernels (dg_adamw_step).

Data parallel (one process per GPU, SURVEY.md section 8e): the ONE collective of a training step -- the mean all-reduce of the
flat gradient (486,409 floats for the shipped LightweightUNet) -- is issued at the END OF BACKWARD (`_TrainFn.backward`), i.e.
between `loss.backward()` and everything the reference does next (optimized_train.py:210-219 / :226-233): `scaler.unscale_` + its
inf check, `clip_grad_norm_`, `optimizer.step()` all see the already-averaged gradient, every rank takes the same skip / clip
decision, and no rank can miss the collective.  `module.ddp_sync = False` turns it off (gradient accumulation over micro-batches).
"""
import contextlib

import torch

from . import _lib


class _TrainCtx:
    """Side channel between the module's autograd node and `L1Loss` below: when the loss of the step is the fused L1, its backward
    leaves (target, dL/dloss) here and the module's backward generates the gradient seed inside the head-backward kernel."""
    __slots__ = ("y", "l1_target", "l1_scale", "l1_marker")

    def __init__(self):
        self.y = self.l1_target = self.l1_scale = self.l1_marker = None


def _on_device_of(t):
    """Make t's GPU the current one for the launches below; a CPU tensor (the bridge over torch stand-ins of the ops) needs none."""
    return torch.cuda.device(t.device) if t.is_cuda else contextlib.nullcontext()


def _alias_grads(flat, params):
    """Make each parameter's `.grad` its consecutive view of `flat`, in order: the layout `_flat_grad_sink` accepts."""
    off = 0
    for p in params:
        p.grad = flat[off:off + p.numel()].view_as(p)
        off += p.numel()


def _zero_grads(flat, params):
    """zero_grad of a flat gradient bucket (FusedAdamW, FlatGradBucket): zero it, stamp it all-zero as of this version -- the
    stamp `_flat_grad_sink` reads, so that backward may write straight into it -- and alias the `.grad`s again."""
    flat.zero_()
    flat._dg_zero_version = flat._version
    _alias_grads(flat, params)


def _flat_grad_sink(params, want=None):
    """The flat fp32 buffer whose consecutive views are the `.grad`s of the parameters flagged in `want` (default: those that
    require a gradient), in parameters() order -- the FusedAdamW / FlatGradBucket layout over the trainable parameters -- if it is
    known to be all-zero since its last `_zero_grads` and nothing else would observe the per-parameter accumulation; else None.
    No other parameter's `.grad` may live in it."""
    if want is None:
        want = [p.requires_grad for p in params]
    sel = [p for p, w in zip(params, want) if w]
    if not sel or sel[0].grad is None:
        return None
    g0 = sel[0].grad
    base = g0._base if g0._base is not None else g0
    if getattr(base, "_dg_zero_version", None) != base._version or base.dtype != torch.float32 or not base.is_contiguous():
        return None
    off = 0
    for p in sel:
        g = p.grad
        if g is None or not p.requires_grad or g.data_ptr() != base.data_ptr() + 4 * off or g.numel() != p.numel():
            return None
        if p._backward_hooks or getattr(p, "_post_accumulate_grad_hooks", None):
            return None     # wandb.watch and friends hook the per-parameter accumulation: keep the ordinary autograd path
        off += p.numel()
    if off != base.numel():
        return None
    storage = base.untyped_storage().data_ptr()
    if any(not w and p.grad is not None and p.grad.untyped_storage().data_ptr() == storage for p, w in zip(params, want)):
        return None
    return base


def _gather_index(module, params, want, device):
    """Positions of the flagged parameters' elements in the full parameters() layout, built once per request and kept on the
    module for its lifetime: a captured step reads the index by address, so no later request may release it."""
    cache = module.__dict__.setdefault("_dg_gather_index", {})
    key = (tuple(want), device)
    if key not in cache:
        idx, off = [], 0
        for p, w in zip(params, want):
            if w:
                idx.append(torch.arange(off, off + p.numel()))
            off += p.numel()
        cache[key] = torch.cat(idx).to(device)
    return cache[key]


class _TrainFn(torch.autograd.Function):
    """The autograd node of a training forward, shared by LightweightUNet and OptimizedUNet.  The model computes:
      module._train_forward(x) -> (y, saved)
      module._train_backward(saved, grad_y, tctx, want_p, grad_x, sink) -> flat
        the parameter gradients flagged in `want_p` (parameters() order) into `sink` when given, else into a buffer of the model's
        own in the full parameters() layout or the compact one over `want_p`; returns the buffer that holds them.  dL/dx into
        `grad_x` (fp32, x's shape) when given.
    This node decides which gradients are wanted and where they land -- the optimizer's flat bucket when `_flat_grad_sink` finds it
    safe (no per-parameter accumulate kernels), else the model's buffer handed to autograd -- and ends with the data-parallel mean
    all-reduce of the parameter gradients."""

    @staticmethod
    def forward(ctx, module, tctx, x, *params):
        with _on_device_of(x):
            y, ctx.saved = module._train_forward(x)
        ctx.module, ctx.tctx, ctx.n_inputs = module, tctx, len(params)
        ctx.x_meta = (x.shape, x.dtype, x.device)
        ctx.direct = getattr(module, "_dg_direct_grads", False)
        if tctx is not None:
            tctx.y = y
        return y

    @staticmethod
    def backward(ctx, grad_y):
        module, tctx = ctx.module, ctx.tctx
        if ctx.saved is None:
            raise RuntimeError(f"{type(module).__name__}: backward through the same forward twice (the saved activations were "
                               "released)")
        params = list(module.parameters())
        # Only what autograd asks for is computed: dL/dx when x needs it, the gradients of parameters that require one.
        # GraphedTrainStep's parameters are not autograd inputs: it wants the trainable ones.
        want_x = ctx.needs_input_grad[2]
        want_p = [p.requires_grad for p in params] if ctx.direct else list(ctx.needs_input_grad[3:])
        shape, x_dtype, dev = ctx.x_meta
        grad_x = torch.empty(shape, dtype=torch.float32, device=dev) if want_x else None
        with _on_device_of(grad_y):
            # the optimizer's flat bucket when it is safe to write into (fresh after zero_grad, no hooks); a fully frozen net gets
            # no gradient buffer at all
            sink = _flat_grad_sink(params, want_p) if any(want_p) else None
            if ctx.direct and sink is None:
                raise RuntimeError("GraphedTrainStep: the gradients must land in the optimizer's flat bucket (FusedAdamW.zero_grad "
                                   "inside the step, no per-parameter hooks)")
            flat = module._train_backward(ctx.saved, grad_y, tctx, want_p, grad_x, sink)
        ctx.saved = None
        if tctx is not None:
            tctx.y = tctx.l1_target = tctx.l1_scale = tctx.l1_marker = None
        if grad_x is not None and grad_x.dtype != x_dtype:
            grad_x = grad_x.to(x_dtype)
        if not any(want_p):
            return (None, None, grad_x) + (None,) * ctx.n_inputs
        sync_gradients(flat, getattr(module, "ddp_sync", True))   # parameter gradients only: dL/dx is per rank's own batch
        if sink is not None:
            sink._dg_zero_version = None      # the bucket now holds a gradient: a second backward must accumulate the ordinary way
            return (None, None, grad_x) + (None,) * ctx.n_inputs
        full = flat.numel() == sum(p.numel() for p in params)
        grads, off = [], 0
        for p, want in zip(params, want_p):
            n = p.numel()
            grads.append(flat[off:off + n].view_as(p) if want else None)   # a frozen range is never written
            off += n if want or full else 0
        return (None, None, grad_x, *grads)


class _FusedL1(torch.autograd.Function):
    @staticmethod
    def forward(ctx, outputs, targets, tctx):
        acc = torch.zeros(1, dtype=torch.float64, device=outputs.device)
        with torch.cuda.device(outputs.device):
            _lib.check(_lib.load().dg_l1_loss_sum(outputs.data_ptr(), targets.data_ptr(), outputs.numel(), acc.data_ptr(),
                                                  torch.cuda.current_stream().cuda_stream))
        ctx.tctx, ctx.targets, ctx.shape = tctx, targets, outputs.shape
        return (acc / outputs.numel()).to(torch.float32).reshape(())

    @staticmethod
    def backward(ctx, grad_loss):
        tctx = ctx.tctx
        scale = grad_loss.detach().float().reshape(1).contiguous()
        tctx.l1_target, tctx.l1_scale = ctx.targets, scale
        tctx.l1_marker = scale.expand(ctx.shape)     # stride-0 view: no kernel; the module's backward recognises it by pointer
        return tctx.l1_marker, None, None


class L1Loss(torch.nn.Module):
    """Drop-in for the `nn.L1Loss()` of optimized_train.py:439.  On an output of this package's module in training it is the fused
    L1 (SURVEY 8a row a10): the loss value is one reduction kernel, and backward never materialises sign(o - t) / numel -- the head
    backward kernel generates it from the forward output and the target.  Anything else (other reductions, other tensors, CPU)
    falls through to torch.nn.functional.l1_loss with identical semantics."""

    def __init__(self, size_average=None, reduce=None, reduction="mean"):
        super().__init__()
        self.reduction = reduction

    def forward(self, outputs, targets):
        tctx = getattr(outputs, "_dg_train_ctx", None)
        if (tctx is None or self.reduction != "mean" or not torch.is_grad_enabled() or not outputs.requires_grad
                or targets.requires_grad or outputs.shape != targets.shape or not targets.is_cuda
                or targets.dtype != torch.float32 or tctx.y is None or outputs.data_ptr() != tctx.y.data_ptr()):
            return torch.nn.functional.l1_loss(outputs, targets, reduction=self.reduction)
        return _FusedL1.apply(outputs, targets.contiguous(), tctx)


def sync_gradients(flat, enabled=True, group=None):
    """Mean all-reduce of the flat gradient over the data-parallel ranks (no-op without an initialised process group).
    NCCL averages inside the collective; backends without AVG (gloo) sum and scale."""
    import torch.distributed as dist
    if not enabled or not (dist.is_available() and dist.is_initialized()):
        return flat
    world = dist.get_world_size(group)
    if world <= 1:
        return flat
    if dist.get_backend(group) == "nccl":
        dist.all_reduce(flat, op=dist.ReduceOp.AVG, group=group)
    else:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        flat.mul_(1.0 / world)
    return flat


def train_forward(module, x):
    """The forward of `module` (LightweightUNet, OptimizedUNet) recorded for autograd through `_TrainFn`.  Only a module whose
    backward consumes `L1Loss`'s seed (class flag `_fused_l1`) gets an output that `L1Loss` fuses: any other module would be handed
    the stride-0 dL/dloss marker as if it were dL/dy."""
    tctx = _TrainCtx() if getattr(module, "_fused_l1", False) else None
    if getattr(module, "_dg_direct_grads", False):
        if x.requires_grad:
            raise NotImplementedError("GraphedTrainStep computes parameter gradients only, not the input image's")
        # GraphedTrainStep: the parameters are NOT autograd inputs -- their AccumulateGrad nodes carry the stream they were created
        # on (the default stream if an eager step's graph is still alive), and the engine would synchronise the capturing stream
        # with it at the end of backward (cudaErrorStreamCaptureIsolation).  A fresh leaf anchors the node instead; the gradients
        # go straight into the optimizer's flat bucket.
        inputs = (torch.zeros((), device=x.device, requires_grad=True),)
    else:
        inputs = tuple(module.parameters())
    y = _TrainFn.apply(module, tctx, x, *inputs)
    if tctx is not None:
        y._dg_train_ctx = tctx
    return y


class FusedAdamW(torch.optim.Optimizer):
    """torch.optim.AdamW (optimized_train.py:440-446) with flat storage and a fused clip + update (dg_adamw_step).

    max_grad_norm > 0 folds `torch.nn.utils.clip_grad_norm_(params, max_grad_norm)` (optimized_train.py:215,230) into the
    step; leave it 0 if the caller clips itself.  All parameters must be fp32 on one CUDA device, in ONE param group.

    Checkpoints: `state_dict()` / `load_state_dict()` use torch.optim.AdamW's own layout (per-parameter `step`, `exp_avg`,
    `exp_avg_sq`), so the `optimizer_state_dict` entry the reference writes into every checkpoint (optimized_train.py:69)
    round-trips with a plain AdamW in either direction.  The data-parallel gradient exchange is NOT here: it happens at the
    end of backward (see the module docstring), before any clipping or inf check."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, max_grad_norm=0.0, capturable=False):
        params = [p for p in params]
        self.capturable = capturable
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, max_grad_norm=max_grad_norm))
        if len(self.param_groups) != 1:
            raise ValueError("FusedAdamW keeps one flat buffer: pass a single param group (per-group hyper-parameters are not supported)")
        ps = [p for g in self.param_groups for p in g["params"] if p.requires_grad]
        if not ps or any(not p.is_cuda or p.dtype != torch.float32 for p in ps):
            raise RuntimeError("FusedAdamW needs fp32 CUDA parameters")
        self._ps = ps
        dev = ps[0].device
        n = sum(p.numel() for p in ps)
        self.flat_p = torch.empty(n, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=dev)
        self._scratch = torch.zeros(1, dtype=torch.float64, device=dev)
        self._step = 0
        # capturable: step count and learning rate in device memory (dg_adamw_step_graph), so that step() can sit inside a CUDA graph
        self._step_dev = torch.zeros(1, dtype=torch.int32, device=dev) if capturable else None
        self._lr_dev = torch.full((1,), float(lr), dtype=torch.float32, device=dev) if capturable else None
        off = 0
        with torch.no_grad():
            for p in ps:
                k = p.numel()
                self.flat_p[off:off + k].copy_(p.reshape(-1))
                p.data = self.flat_p[off:off + k].view_as(p)     # parameters become views of the flat buffer
                off += k
        _alias_grads(self.flat_g, ps)

    def add_param_group(self, param_group):
        if getattr(self, "param_groups", None):
            raise ValueError("FusedAdamW supports a single param group")
        super().add_param_group(param_group)

    def _publish_state(self):
        """Expose the flat moments through `self.state` in torch.optim.AdamW's layout (views, no copies)."""
        off = 0
        for p in self._ps:
            k = p.numel()
            # one `step` tensor PER parameter (torch.optim.AdamW increments each entry in place: a shared tensor would be bumped
            # once per parameter after a reload)
            self.state[p] = {"step": torch.tensor(float(self._step)), "exp_avg": self.exp_avg[off:off + k].view_as(p),
                             "exp_avg_sq": self.exp_avg_sq[off:off + k].view_as(p)}
            off += k

    def _sync_step(self):
        if self.capturable:
            self._step = int(self._step_dev.item())

    def push_hyperparameters(self):
        """capturable only: copy param_groups[0]['lr'] (an LR scheduler writes it on the host) to the device scalar the captured
        step reads.  Call before replaying a graph that contains step()."""
        if self.capturable:
            self._lr_dev.fill_(float(self.param_groups[0]["lr"]))

    def state_dict(self):
        self._sync_step()
        if self._step > 0:
            self._publish_state()
        return super().state_dict()

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)   # validates the groups / sizes and fills self.state with (copied) tensors
        if len(self.param_groups) != 1:
            raise ValueError("FusedAdamW supports a single param group")
        steps = set()
        off = 0
        with torch.no_grad():
            for p in self._ps:
                k = p.numel()
                st = self.state.get(p)
                if st:
                    self.exp_avg[off:off + k].copy_(st["exp_avg"].reshape(-1))
                    self.exp_avg_sq[off:off + k].copy_(st["exp_avg_sq"].reshape(-1))
                    steps.add(int(float(st["step"])))
                else:
                    self.exp_avg[off:off + k].zero_()
                    self.exp_avg_sq[off:off + k].zero_()
                    steps.add(0)
                off += k
        if len(steps) != 1:
            raise ValueError(f"FusedAdamW needs one common step count, checkpoint has {sorted(steps)}")
        self._step = steps.pop()
        if self.capturable:
            self._step_dev.fill_(self._step)
        if self._step > 0:
            self._publish_state()
        else:
            self.state.clear()

    def zero_grad(self, set_to_none=True):
        # the reference calls zero_grad(set_to_none=True) (optimized_train.py:201); keep the flat aliasing instead
        _zero_grads(self.flat_g, self._ps)

    def _gather(self):
        off = 0
        for p in self._ps:
            k = p.numel()
            want = self.flat_g[off:off + k]
            if p.grad is None:
                want.zero_()
            elif p.grad.data_ptr() != want.data_ptr():
                want.copy_(p.grad.reshape(-1))
            off += k

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        self._gather()
        g = self.param_groups[0]
        if self.capturable:
            if not torch.cuda.is_current_stream_capturing():
                self._lr_dev.fill_(float(g["lr"]))
            _lib.check(_lib.load().dg_adamw_step_graph(
                self.flat_p.data_ptr(), self.flat_g.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(),
                self.flat_p.numel(), self._scratch.data_ptr(), float(g["max_grad_norm"]), self._lr_dev.data_ptr(),
                float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]), float(g["weight_decay"]), self._step_dev.data_ptr(),
                1.0, torch.cuda.current_stream().cuda_stream))
            _lib.bump_generation()
            return loss
        self._step += 1
        _lib.check(_lib.load().dg_adamw_step(
            self.flat_p.data_ptr(), self.flat_g.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(),
            self.flat_p.numel(), self._scratch.data_ptr(), float(g["max_grad_norm"]), float(g["lr"]), float(g["betas"][0]),
            float(g["betas"][1]), float(g["eps"]), float(g["weight_decay"]), self._step, 1.0,
            torch.cuda.current_stream().cuda_stream))
        _lib.bump_generation()   # parameters changed behind autograd's back: invalidate packed-weight caches
        return loss

    def grad_norm(self):
        """Total L2 norm of the gradient seen by the last step (the value clip_grad_norm_ returns)."""
        return float(self._scratch.sqrt().item())


def _check_trainable(module, opt_params):
    """The optimizer's parameters must be the module's trainable ones, in parameters() order: the gradients land in its flat
    bucket in that layout."""
    names = {id(p): k for k, p in module.named_parameters()}
    trainable = [p for p in module.parameters() if p.requires_grad]
    if not trainable:
        raise ValueError("GraphedTrainStep: the module has no trainable parameter (requires_grad)")

    def what(p):
        if p is None:
            return "nothing"
        if id(p) not in names:
            return "a tensor that is not a parameter of the module"
        return names[id(p)] + ("" if p.requires_grad else " (frozen)")
    for i in range(max(len(trainable), len(opt_params))):
        a = opt_params[i] if i < len(opt_params) else None
        b = trainable[i] if i < len(trainable) else None
        if a is not b:
            raise ValueError(f"GraphedTrainStep: the optimizer must hold exactly the module's trainable parameters in parameters() "
                             f"order; at position {i} it has {what(a)} where the module's trainable parameters have {what(b)}")


class GraphedTrainStep:
    """One training step of the reference loop (optimized_train.py:201-233: zero_grad, forward, L1, backward -- with the data-parallel
    all-reduce at its end -- clip, AdamW) captured ONCE in a CUDA graph and replayed per batch.

    Why: at the reference's own configuration (global batch 32 = 4 images per GPU on 8 GPUs) a step is ~75 kernels of 10-50 us
    plus the packing kernels of the updated weights; issued from Python the host launch rate bounds it, not the GPU.
    Needs a `FusedAdamW(..., capturable=True)` (step count and learning rate in device memory) and fixed batch shapes.
    Trainable means `requires_grad`: the optimizer must hold exactly the module's trainable parameters, in parameters() order,
    and only their gradients are computed (fine-tuning with frozen layers; the frozen ones cost no kernel work).

        step = GraphedTrainStep(net, opt, criterion, inputs.shape)
        for inputs, targets in loader: loss = step(inputs, targets)      # loss: 0-d device tensor, valid until the next call
    """

    def __init__(self, module, optimizer, criterion, shape, warmup=3, clip_grad_norm=None):
        if not getattr(optimizer, "capturable", False):
            raise RuntimeError("GraphedTrainStep needs FusedAdamW(..., capturable=True)")
        _check_trainable(module, optimizer._ps)
        dev = next(module.parameters()).device
        self.module, self.optimizer, self.criterion, self.clip = module, optimizer, criterion, clip_grad_norm
        # The warm-up steps run with lr = 0 and weight decay 0 against saved moments: they must not train.  Their input is uniform
        # noise, NOT zeros: a bias-free freshly initialised network maps a constant image to constant activations, every GroupNorm
        # then divides by sqrt(eps) (x 316 per layer in the backward), the gradient overflows, and 0 * inf in the AdamW update turns
        # the parameters into NaN before the first real step (measured on a default-initialised OptimizedUNet at 256x256).
        gen = torch.Generator().manual_seed(0)
        self.x = torch.rand(tuple(shape), generator=gen).to(dev)
        self.t = torch.rand((shape[0], module.out_channels) + tuple(shape[2:]), generator=gen).to(dev)
        g = optimizer.param_groups[0]
        saved = (g["lr"], g["weight_decay"], optimizer.exp_avg.clone(), optimizer.exp_avg_sq.clone(), optimizer._step_dev.clone())
        g["lr"], g["weight_decay"] = 0.0, 0.0
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._eager()
        torch.cuda.current_stream().wait_stream(side)
        # restore what the warm-up touched BEFORE capturing: weight decay, betas, eps and the clip norm are launch arguments and are
        # baked into the graph (only the step count and the learning rate are read from device memory)
        g["lr"], g["weight_decay"] = saved[0], saved[1]
        optimizer.exp_avg.copy_(saved[2]); optimizer.exp_avg_sq.copy_(saved[3]); optimizer._step_dev.copy_(saved[4])
        optimizer.push_hyperparameters()
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss = self._eager()

    def _eager(self):
        self.optimizer.zero_grad(set_to_none=True)
        self.module._dg_direct_grads = True
        try:
            loss = self.criterion(self.module(self.x), self.t)
        finally:
            self.module._dg_direct_grads = False
        loss.backward()
        if self.clip:
            torch.nn.utils.clip_grad_norm_(self.module.parameters(), max_norm=self.clip)
        self.optimizer.step()
        return loss.detach()

    def __call__(self, inputs, targets):
        self.x.copy_(inputs, non_blocking=True)
        self.t.copy_(targets, non_blocking=True)
        self.optimizer.push_hyperparameters()
        self.graph.replay()
        _lib.bump_generation()   # the weights changed inside the graph: eager forwards after this must re-pack their caches
        return self.loss
