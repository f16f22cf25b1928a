"""Adam / AdamW over one flat parameter buffer (csrc/adam.cu, include/b2r.h: b2r_adam_flat_step_groups,
b2r_flat_grad_norm).

Mirrors `optim.Adam(net.parameters(), lr=..., weight_decay=...)` of the reference's training
scripts (/root/reference/detection/Votenet/train_Votenet_FSB.py:176-181) and GroupFree3D's
`optim.AdamW` over two parameter groups with `clip_grad_norm_` before every step
(G/train_GF_FSB.py:319-320) for the captured step: parameters become views of ONE contiguous fp32
buffer, the step's gradients are packed into a second one (the buffer the NCCL all-reduce of
dist_utils.FlatGradBucket already works on), the global gradient norm is one deterministic
reduction and the update is a single streaming kernel whose step counter lives on the device, so
it replays from a CUDA graph.  Same arithmetic as torch.optim.Adam / AdamW (amsgrad=False,
maximize=False) and clip_grad_norm_(norm_type=2); checked against them in
tests/test_modules_gpu.py and tests/test_flat_optim_gpu.py.

    opt = FlatAdam(net.parameters(), lr=1e-3)
    loss.backward(); opt.step()             # packs p.grad of every parameter, then updates
    opt.step(grads=list_of_tensors)         # or: gradients given explicitly (p.grad = None scheme)

    opt = FlatAdamW([{"params": enc}, {"params": dec, "lr": 1e-4}], lr=1e-3, weight_decay=5e-4,
                    max_grad_norm=0.1)      # GroupFree3D: AdamW, two groups, global clipping
    sched = torch.optim.lr_scheduler.MultiStepLR(opt, [280, 340])   # any torch scheduler

FlatAdam is a torch.optim.Optimizer: schedulers and hand-written `adjust_learning_rate` loops set
`param_groups[i]["lr"]`.  Each group's lr and weight_decay are read by the kernel from a small
device table.  `step()` refreshes that table before it launches, except inside a CUDA-graph
capture, where it records nothing; a captured step is driven by

    sched.step(); opt.sync_hparams(); graph.replay()

Differences from torch.optim.Adam / AdamW:
  - a parameter without a gradient in a step is treated as having a zero gradient (its moments
    decay and AdamW's decay still applies); torch skips such parameters.  There is one step
    counter for all parameters.
  - `step()` takes the gradients (or reads p.grad) and never modifies p.grad, also when clipping.
"""
import ctypes

import torch
import torch.distributed as dist

from . import _ext, _lib

# options of torch.optim.Adam that select an implementation, not a result: ignored when loading
# a torch checkpoint
_TORCH_IMPL_KEYS = ("foreach", "capturable", "differentiable", "fused")


class FlatAdam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, amsgrad=False,
                 *, maximize=False, decoupled_weight_decay=False, max_grad_norm=None, norm_type=2.0):
        params = list(params)
        if not params:
            raise ValueError("FlatAdam: no parameters")
        if amsgrad or maximize:
            raise ValueError("FlatAdam: amsgrad and maximize are not supported")
        if max_grad_norm is not None and float(norm_type) != 2.0:
            raise ValueError("FlatAdam: only the L2 gradient norm (norm_type=2) is supported, got %r"
                             % (norm_type,))
        defaults = dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay, amsgrad=False,
                        maximize=False, decoupled_weight_decay=bool(decoupled_weight_decay))
        super().__init__(params, defaults)
        self.decoupled = bool(decoupled_weight_decay)
        self.max_grad_norm = None if max_grad_norm is None else float(max_grad_norm)
        g0 = self.param_groups[0]
        self.betas, self.eps = tuple(float(b) for b in g0["betas"]), float(g0["eps"])
        for g in self.param_groups:
            if tuple(float(b) for b in g["betas"]) != self.betas or float(g["eps"]) != self.eps:
                raise ValueError("FlatAdam: every parameter group must use the same betas and eps")
            if g["amsgrad"] or g["maximize"]:
                raise ValueError("FlatAdam: amsgrad and maximize are not supported")
            if bool(g["decoupled_weight_decay"]) != self.decoupled:
                raise ValueError("FlatAdam: decoupled_weight_decay must be the same for every group")
        if len(self.param_groups) > _lib.ADAM_MAX_GROUPS:
            raise ValueError("FlatAdam: at most %d parameter groups" % _lib.ADAM_MAX_GROUPS)

        # the flat layout: parameters in group order; 16-byte aligned slices (every parameter, and
        # so every group, starts at a multiple of 4 floats)
        self.params = [p for g in self.param_groups for p in g["params"]]
        dev = self.params[0].device
        if dev.type != "cuda":
            raise RuntimeError("FlatAdam runs on CUDA only (there is no CPU fallback)")
        for p in self.params:
            if p.dtype != torch.float32 or p.device != dev:
                raise TypeError("FlatAdam: parameters must be fp32 tensors on one device")
        self.offsets, self.group_bounds, n = [], [], 0
        for g in self.param_groups:
            start = n
            for p in g["params"]:
                self.offsets.append(n)
                n += (p.numel() + 3) // 4 * 4
            self.group_bounds.append((start, n))
        self.numel = n
        self.flat_p = torch.zeros(n, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=dev)
        # device step counter { t, 1/(1-b1^t), 1/sqrt(1-b2^t) } (torch's Optimizer.state is the
        # per-parameter dict; FlatAdam keeps its state in the flat buffers)
        self.step_state = torch.zeros(int(_lib.lib().b2r_adam_state_bytes()), dtype=torch.uint8, device=dev)
        # per-group [start, end), lr, weight_decay (b2r_adam_group): read by the kernel at run time
        self.group_table = torch.zeros(len(self.param_groups) * ctypes.sizeof(_lib.AdamGroup),
                                       dtype=torch.uint8, device=dev)
        self._table_host = None          # what the device table holds (skip unchanged rewrites)
        if self.max_grad_norm is not None:
            ws = int(_lib.lib().b2r_flat_grad_norm_workspace_bytes(n))
            self.norm_ws = torch.empty(ws, dtype=torch.uint8, device=dev)
            self._norm_coef = torch.zeros(2, dtype=torch.float32, device=dev)
            # total norm of the last step's (averaged) gradient before clipping: what
            # clip_grad_norm_ returns.  A 0-dim device tensor, overwritten by every step / replay.
            self.last_grad_norm = self._norm_coef[0]
        else:
            self.last_grad_norm = None
        self.g_views = []
        with torch.no_grad():
            for p, off in zip(self.params, self.offsets):
                view = self.flat_p[off:off + p.numel()].view_as(p)
                view.copy_(p)
                p.data = view                       # the module's Parameter now lives in the flat buffer
                self.g_views.append(self.flat_g[off:off + p.numel()].view_as(p))
        self.sync_hparams()

    def add_param_group(self, param_group):
        if hasattr(self, "flat_p"):
            raise RuntimeError("FlatAdam: parameter groups are fixed at construction (the flat "
                               "buffer is laid out then); build a new optimizer instead")
        super().add_param_group(param_group)

    @property
    def lr(self):
        """learning rate of the first group (the one-group optimizer's `lr`)"""
        return self.param_groups[0]["lr"]

    @lr.setter
    def lr(self, value):
        for g in self.param_groups:
            g["lr"] = value

    @property
    def weight_decay(self):
        return self.param_groups[0]["weight_decay"]

    # ---- learning rates that replay from a captured step ----------------------------------------
    def sync_hparams(self):
        """Write every group's lr and weight_decay into the device table, ordered on the current
        stream.  step() calls it outside a capture; a captured step reads whatever the table holds
        when it replays, so call it after changing the rates (scheduler.step()) and before the
        replay.  Never call it inside a capture: a captured write would restore the capture-time
        rates on every replay."""
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("FlatAdam.sync_hparams() inside a CUDA-graph capture would bake the "
                               "current rates into the graph; call it between replays")
        rows = tuple((lo, hi, float(g["lr"]), float(g["weight_decay"]))
                     for (lo, hi), g in zip(self.group_bounds, self.param_groups))
        if rows == self._table_host:
            return
        arr = (_lib.AdamGroup * len(rows))(*[_lib.AdamGroup(*r) for r in rows])
        host = torch.frombuffer(bytearray(arr), dtype=torch.uint8).pin_memory()
        # the caching host allocator keeps `host` alive until the copy has run
        self.group_table.copy_(host, non_blocking=True)
        self._table_host = rows

    # ---- overlapping the gradient all-reduce with the rest of backward (world > 1) --------------
    def set_late(self, n_late):
        """The first `n_late` parameters (in group order) are the ones whose gradients arrive LAST in
        backward (the first layers of the network: backward runs the forward order in reverse).
        `reduce_early` may then be called from a backward hook placed where everything after them
        is done."""
        self.n_late = int(n_late)
        self.off_late = self.offsets[self.n_late] if self.n_late < len(self.params) else self.numel
        self.comm = torch.cuda.Stream(device=self.flat_p.device)
        self._early_done = False

    def reduce_early(self):
        """pack + all-reduce the gradients of params[n_late:] on a side stream, while backward goes
        on with the first layers.  Call when those gradients exist (tensor hook on an activation
        between the two parameter groups).  No-op without a process group."""
        if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
            return
        early = self.params[self.n_late:]
        if any(p.grad is None for p in early):
            return                      # not all there (e.g. a frozen branch): step() does everything
        torch._foreach_copy_(self.g_views[self.n_late:], [p.grad for p in early])
        self.comm.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.comm):
            dist.all_reduce(self.flat_g[self.off_late:])
        self._early_done = True

    def zero_grad(self, set_to_none=True):
        for p in self.params:
            p.grad = None

    def pack(self, grads=None):
        """gradients of this step -> the flat buffer (one multi-tensor copy); parameters without a
        gradient contribute zeros"""
        if grads is None:
            grads = [p.grad for p in self.params]
        have = [(v, g) for v, g in zip(self.g_views, grads) if g is not None]
        if len(have) != len(self.g_views):
            self.flat_g.zero_()
        torch._foreach_copy_([v for v, _ in have], [g for _, g in have])

    def step(self, grads=None, allreduce=True):
        """pack -> (world > 1: one NCCL sum all-reduce of the flat gradient) -> (max_grad_norm:
        global norm + clip coefficient) -> one Adam / AdamW kernel over every group.
        `grads`: one tensor (or None) per parameter in group order; default p.grad."""
        if not torch.cuda.is_current_stream_capturing():
            self.sync_hparams()
        scale = 1.0
        multi = allreduce and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        if multi and getattr(self, "_early_done", False):
            # params[n_late:] are packed and their all-reduce is in flight on the side stream
            self._early_done = False
            if grads is None:
                grads = [p.grad for p in self.params]
            late = [(v, g) for v, g in zip(self.g_views[:self.n_late], grads[:self.n_late]) if g is not None]
            if len(late) != self.n_late:
                self.flat_g[:self.off_late].zero_()
            torch._foreach_copy_([v for v, _ in late], [g for _, g in late])
            if self.off_late > 0:
                dist.all_reduce(self.flat_g[:self.off_late])
            torch.cuda.current_stream().wait_stream(self.comm)
        else:
            self.pack(grads)
            if multi:
                dist.all_reduce(self.flat_g)
        if multi:
            scale = 1.0 / dist.get_world_size()     # averaged inside the kernels (DDP semantics)
        l, stream = _lib.lib(), _ext._stream()
        with _ext._on_device(self.flat_p):
            clip = None
            if self.max_grad_norm is not None:
                clip = self._norm_coef[1:].data_ptr()
                _lib.check(l.b2r_flat_grad_norm(
                    self.flat_g.data_ptr(), self.numel, scale, self.max_grad_norm,
                    self.norm_ws.data_ptr(), self._norm_coef.data_ptr(), clip, stream), "flat_grad_norm")
            desc = _lib.AdamDesc(
                params=self.flat_p.data_ptr(), grads=self.flat_g.data_ptr(),
                exp_avg=self.exp_avg.data_ptr(), exp_avg_sq=self.exp_avg_sq.data_ptr(), n=self.numel,
                state=self.step_state.data_ptr(), groups=self.group_table.data_ptr(),
                n_groups=len(self.param_groups), beta1=self.betas[0], beta2=self.betas[1], eps=self.eps,
                grad_scale=scale, decoupled=int(self.decoupled), clip_coef=clip)
            _lib.check(l.b2r_adam_flat_step_groups(ctypes.byref(desc), stream), "adam_flat_step_groups")
        # the kernel wrote through raw pointers: tell autograd / the weight-image caches
        torch.autograd.graph.increment_version(self.params)

    # ---- checkpoints -----------------------------------------------------------------------------
    def _step_count(self):
        return float(self.step_state.view(torch.float32)[0])

    def state_dict(self):
        """FlatAdam's own format: the flat buffers.  torch_state_dict() writes torch's."""
        return {"flat_p": self.flat_p.clone(), "exp_avg": self.exp_avg.clone(),
                "exp_avg_sq": self.exp_avg_sq.clone(), "state": self.step_state.clone(),
                "lr": self.lr, "betas": self.betas, "eps": self.eps, "weight_decay": self.weight_decay,
                "param_groups": [{k: v for k, v in g.items() if k != "params"} for g in self.param_groups]}

    def _torch_class(self):
        return torch.optim.AdamW if isinstance(self, FlatAdamW) else torch.optim.Adam

    def torch_state_dict(self):
        """Exactly what torch.optim.Adam (FlatAdamW: torch.optim.AdamW) returns from state_dict()
        for the same parameter groups after the same steps: per parameter `step`, `exp_avg`,
        `exp_avg_sq` (copies), and `param_groups` with torch's keys.  Before the first step the
        per-parameter state is empty, as in torch."""
        groups = [{k: v for k, v in g.items() if k != "params"} | {"params": list(g["params"])}
                  for g in self.param_groups]
        sd = self._torch_class()(groups).state_dict()
        t = self._step_count()
        if t > 0:
            for i, (p, off) in enumerate(zip(self.params, self.offsets)):
                sd["state"][i] = {
                    "step": torch.tensor(t, dtype=torch.float32),
                    "exp_avg": self.exp_avg[off:off + p.numel()].view_as(p).clone(),
                    "exp_avg_sq": self.exp_avg_sq[off:off + p.numel()].view_as(p).clone()}
        return sd

    def load_state_dict(self, sd):
        """Accepts state_dict()'s format and torch.optim.Adam / AdamW's (torch_state_dict()).  The
        torch format must have one step count for every parameter (FlatAdam has one device
        counter), or no per-parameter state at all (before the first step)."""
        if "flat_p" in sd:
            self.flat_p.copy_(sd["flat_p"]); self.exp_avg.copy_(sd["exp_avg"])
            self.exp_avg_sq.copy_(sd["exp_avg_sq"]); self.step_state.copy_(sd["state"])
            if "param_groups" in sd:
                for g, s in zip(self.param_groups, sd["param_groups"]):
                    g.update(s)
            else:
                for g in self.param_groups:
                    g["lr"], g["weight_decay"] = sd["lr"], sd["weight_decay"]
            self.sync_hparams()
            return
        saved = sd["param_groups"]
        if len(saved) != len(self.param_groups) or any(
                len(s["params"]) != len(g["params"]) for s, g in zip(saved, self.param_groups)):
            raise ValueError("FlatAdam.load_state_dict: the parameter groups do not match the checkpoint's")
        for s in saved:
            if tuple(float(b) for b in s["betas"]) != self.betas or float(s["eps"]) != self.eps:
                raise ValueError("FlatAdam.load_state_dict: the checkpoint's betas / eps differ from "
                                 "this optimizer's (they are fixed at construction)")
            if s.get("amsgrad") or s.get("maximize"):
                raise ValueError("FlatAdam.load_state_dict: amsgrad and maximize are not supported")
            if bool(s.get("decoupled_weight_decay", self.decoupled)) != self.decoupled:
                raise ValueError("FlatAdam.load_state_dict: the checkpoint's decoupled_weight_decay "
                                 "differs from this optimizer's")
        # state is keyed by the parameter's position over all groups, in group order
        ids = [i for s in saved for i in s["params"]]
        state = sd["state"]
        steps = {float(state[i]["step"]) for i in ids if i in state}
        if state and (len(steps) != 1 or any(i not in state for i in ids)):
            raise ValueError("FlatAdam.load_state_dict: every parameter must have the same step count "
                             "(FlatAdam keeps one device step counter); got %s" % sorted(steps))
        with torch.no_grad():
            for i, p, off in zip(ids, self.params, self.offsets):
                st = state.get(i)
                for buf, key in ((self.exp_avg, "exp_avg"), (self.exp_avg_sq, "exp_avg_sq")):
                    dst = buf[off:off + p.numel()]
                    if st is None:
                        dst.zero_()
                    else:
                        if st[key].numel() != p.numel():
                            raise ValueError("FlatAdam.load_state_dict: %s of parameter %d has %d "
                                             "elements, the parameter %d" % (key, i, st[key].numel(),
                                                                             p.numel()))
                        dst.copy_(st[key].reshape(-1))
            self.step_state.zero_()
            self.step_state.view(torch.float32)[0] = steps.pop() if steps else 0.0
        for g, s in zip(self.param_groups, saved):
            g.update({k: v for k, v in s.items() if k != "params" and k not in _TORCH_IMPL_KEYS})
        self.sync_hparams()


class FlatAdamW(FlatAdam):
    """FlatAdam with torch.optim.AdamW's defaults: decoupled weight decay, weight_decay=0.01."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, amsgrad=False,
                 *, maximize=False, max_grad_norm=None, norm_type=2.0):
        super().__init__(params, lr, betas, eps, weight_decay, amsgrad, maximize=maximize,
                         decoupled_weight_decay=True, max_grad_norm=max_grad_norm, norm_type=norm_type)
