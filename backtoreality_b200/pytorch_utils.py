"""SharedMLP building blocks with the reference's parameter / state-dict layout.

Mirrors the call surface of /root/reference/detection/Votenet/pointnet2/pytorch_utils.py that the
hot path uses: `SharedMLP` (:11-36), `Conv2d` / `Conv1d` (:122-188), the BatchNorm wrappers
(:39-64) and `BNMomentumScheduler` (:262-296).  Module nesting is what fixes the checkpoint keys
(e.g. `sa1.mlp_module.layer0.conv.weight`, `sa1.mlp_module.layer0.bn.bn.running_mean`,
SURVEY.md appendix B), so it is reproduced exactly; reference checkpoints load unchanged.
The unused Conv3d / FC / preact paths of the reference are not carried over.

BatchNorm momentum that follows the scheduler inside a replayed CUDA graph: `sync_bn_momentum(net)`
once before the capture gives every BatchNorm of `net` a slot in a device table of momenta, which
the fused kernels (`bn_finalize` below) and the torch-path BatchNorm read when they run.  After
that, `BNMomentumScheduler.step()` writes the new momenta into the table between replays:

    sync_bn_momentum(net)                        # once, before the capture
    step = CapturedTrainStep(step_fn, batch, snapshot=[net, opt])
    for epoch in range(epochs):
        bnm.step()                               # no recapture
        for batch in loader:
            step(batch)
"""
import ctypes

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib


class _BN(nn.Sequential):
    """`<name>bn` child holding the real BatchNorm; weight=1, bias=0 like the reference (:39-47)."""

    def __init__(self, channels, norm_cls, name=""):
        super().__init__()
        self.add_module(name + "bn", norm_cls(channels))
        nn.init.constant_(self[0].weight, 1.0)
        nn.init.constant_(self[0].bias, 0.0)


class BatchNorm1d(_BN):
    def __init__(self, in_size, *, name=""):
        super().__init__(in_size, nn.BatchNorm1d, name)


class BatchNorm2d(_BN):
    def __init__(self, in_size, name=""):
        super().__init__(in_size, nn.BatchNorm2d, name)


class _ConvBlock(nn.Sequential):
    """conv -> (bn) -> (activation); bias only when there is no BN (reference :67-120)."""

    def __init__(self, conv_cls, bn_cls, in_size, out_size, kernel_size, stride, padding,
                 activation, bn, init, bias, name):
        super().__init__()
        conv = conv_cls(in_size, out_size, kernel_size=kernel_size, stride=stride,
                        padding=padding, bias=bias and not bn)
        init(conv.weight)
        if conv.bias is not None:
            nn.init.constant_(conv.bias, 0.0)
        self.add_module(name + "conv", conv)
        if bn:
            self.add_module(name + "bn", bn_cls(out_size))
        if activation is not None:
            self.add_module(name + "activation", activation)


class Conv1d(_ConvBlock):
    def __init__(self, in_size, out_size, *, kernel_size=1, stride=1, padding=0,
                 activation=nn.ReLU(inplace=True), bn=False, init=nn.init.kaiming_normal_,
                 bias=True, preact=False, name=""):
        assert not preact, "preact blocks are not on the hot path"
        super().__init__(nn.Conv1d, BatchNorm1d, in_size, out_size, kernel_size, stride, padding,
                         activation, bn, init, bias, name)


class Conv2d(_ConvBlock):
    def __init__(self, in_size, out_size, *, kernel_size=(1, 1), stride=(1, 1), padding=(0, 0),
                 activation=nn.ReLU(inplace=True), bn=False, init=nn.init.kaiming_normal_,
                 bias=True, preact=False, name=""):
        assert not preact, "preact blocks are not on the hot path"
        super().__init__(nn.Conv2d, BatchNorm2d, in_size, out_size, kernel_size, stride, padding,
                         activation, bn, init, bias, name)


class SharedMLP(nn.Sequential):
    """Stack of 1x1 Conv2d(+BN)+ReLU named layer0, layer1, ... (reference :11-36)."""

    def __init__(self, args, *, bn=False, activation=nn.ReLU(inplace=True), preact=False,
                 first=False, name=""):
        assert not preact, "preact blocks are not on the hot path"
        super().__init__()
        for i in range(len(args) - 1):
            self.add_module(name + "layer{}".format(i),
                            Conv2d(args[i], args[i + 1], bn=bn, activation=activation))

    def channels(self):
        """[C0, C1, ...] as seen by the fused kernels."""
        convs = [blk.conv for blk in self]
        return [convs[0].in_channels] + [c.out_channels for c in convs]


_BN_TYPES = (nn.BatchNorm1d, nn.BatchNorm2d, nn.BatchNorm3d)


def set_bn_momentum_default(bn_momentum):
    def fn(m):
        if isinstance(m, _BN_TYPES):
            m.momentum = bn_momentum
    return fn


class BNMomentumScheduler(object):
    """Sets BatchNorm momentum from `bn_lambda(epoch)` (reference :271-296)."""

    def __init__(self, model, bn_lambda, last_epoch=-1, setter=set_bn_momentum_default):
        if not isinstance(model, nn.Module):
            raise RuntimeError("Class '{}' is not a PyTorch nn Module".format(type(model).__name__))
        self.model = model
        self.setter = setter
        self.lmbd = bn_lambda
        self.step(last_epoch + 1)
        self.last_epoch = last_epoch

    def step(self, epoch=None):
        if epoch is None:
            epoch = self.last_epoch + 1
        self.last_epoch = epoch
        self.model.apply(self.setter(self.lmbd(epoch)))
        if getattr(self.model, "bn_momentum_table", None) is not None and not _capturing():
            sync_bn_momentum(self.model)


# ---- BatchNorm momentum read from the device ---------------------------------------------------
def _capturing():
    return torch.cuda.is_available() and torch.cuda.is_current_stream_capturing()


def momentum_slot(bn):
    """The one-element device tensor `bn` reads its momentum from (sync_bn_momentum), or None."""
    slot = getattr(bn, "momentum_slot", None)
    if slot is not None and slot.device != bn.running_mean.device:
        raise RuntimeError("BatchNorm momentum slot is on %s, the module's buffers on %s: "
                           "sync_bn_momentum() attached the model before it was moved"
                           % (slot.device, bn.running_mean.device))
    return slot


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def bn_finalize(bn, stats, C, count, scale, shift, mean, invstd, stream):
    """Training-mode BatchNorm bookkeeping of `bn` from the fused kernels' batch statistics
    (b2r_bn_finalize, include/b2r.h).  The momentum comes from `bn`'s slot when the model is
    attached (b2r_bn_finalize_dev, read when the kernel runs), otherwise from `bn.momentum`."""
    lib = _lib.lib()
    slot = momentum_slot(bn)
    common = (_ptr(bn.running_mean), _ptr(bn.running_var), _ptr(scale), _ptr(shift), _ptr(mean),
              _ptr(invstd), _ptr(bn.num_batches_tracked), stream)
    if slot is None:
        status = lib.b2r_bn_finalize(_ptr(stats), C, float(count), _ptr(bn.weight), _ptr(bn.bias),
                                     float(bn.eps), float(bn.momentum), *common)
    else:
        status = lib.b2r_bn_finalize_dev(_ptr(stats), C, float(count), _ptr(bn.weight),
                                         _ptr(bn.bias), float(bn.eps), _ptr(slot), *common)
    _lib.check(status, "bn_finalize")


class _SlotMomentum:
    """forward of an attached torch BatchNorm (the layers the fused kernels do not cover, and the
    BR discriminators): in training mode the running statistics are updated with the momentum in
    `momentum_slot`, read when the kernels run.  Normalisation, output and gradients are those of
    F.batch_norm in training mode."""

    def forward(self, input):
        slot = momentum_slot(self)
        if slot is None or not (self.training and self.track_running_stats):
            return super().forward(input)
        self._check_input_dim(input)
        out = F.batch_norm(input, None, None, self.weight, self.bias, True, 0.0, self.eps)
        with torch.no_grad():
            dims = [0] + list(range(2, input.dim()))
            var, mean = torch.var_mean(input, dim=dims, correction=1)   # unbiased, like torch
            self.running_mean.lerp_(mean, slot)
            self.running_var.lerp_(var, slot)
            self.num_batches_tracked.add_(1)
        return out


class SlotBatchNorm1d(_SlotMomentum, nn.BatchNorm1d):
    pass


class SlotBatchNorm2d(_SlotMomentum, nn.BatchNorm2d):
    pass


class SlotBatchNorm3d(_SlotMomentum, nn.BatchNorm3d):
    pass


_SLOT_CLASSES = {nn.BatchNorm1d: SlotBatchNorm1d, nn.BatchNorm2d: SlotBatchNorm2d,
                 nn.BatchNorm3d: SlotBatchNorm3d}


def sync_bn_momentum(model):
    """Copy the `momentum` of every attached BatchNorm of `model` into its device table, ordered on
    the current stream, and return the table.

    The first call attaches the model: every nn.BatchNorm1d/2d/3d that tracks running statistics
    and has a momentum gets a slot, one element of one fp32 device table (`model.bn_momentum_table`,
    never reallocated, so it outlives every graph that reads it).  The slot is a plain attribute,
    `momentum_slot`, not a buffer: state_dict() keys and values do not change.  Attached modules
    become Slot* subclasses of their torch class, so isinstance checks still hold.
    Later calls skip the copy when no momentum changed.  BNMomentumScheduler.step() calls this
    for an attached model.  Never call it inside a CUDA-graph capture: a captured write would
    restore the capture-time momenta on every replay."""
    if _capturing():
        raise RuntimeError("sync_bn_momentum() inside a CUDA-graph capture would bake the current "
                           "momenta into the graph; call it between replays")
    mods = getattr(model, "_bn_momentum_modules", None)
    if mods is None:
        mods = [m for m in model.modules()
                if isinstance(m, _BN_TYPES) and m.track_running_stats and m.momentum is not None]
        if not mods:
            raise ValueError("sync_bn_momentum: the model has no BatchNorm with running statistics "
                             "and a momentum")
        dev = mods[0].running_mean.device
        if dev.type != "cuda" or any(m.running_mean.device != dev for m in mods):
            raise RuntimeError("sync_bn_momentum: the BatchNorm buffers must be on one CUDA device")
        for m in mods:
            if type(m) not in _SLOT_CLASSES:
                raise TypeError("sync_bn_momentum: cannot attach %s (a subclass of a torch "
                                "BatchNorm with a forward of its own)" % type(m).__name__)
        table = torch.zeros(len(mods), dtype=torch.float32, device=dev)
        for i, m in enumerate(mods):
            m.momentum_slot = table[i:i + 1]
            m.__class__ = _SLOT_CLASSES[type(m)]
        model.bn_momentum_table = table
        model._bn_momentum_modules = mods
        model._bn_momentum_host = None       # what the table holds (skip unchanged rewrites)
    values = []
    for m in mods:
        if m.momentum is None:
            raise ValueError("sync_bn_momentum: momentum=None (cumulative average) is not "
                             "supported for an attached BatchNorm")
        values.append(float(m.momentum))
    values = tuple(values)
    if values != model._bn_momentum_host:
        host = torch.tensor(values, dtype=torch.float32).pin_memory()
        # the caching host allocator keeps `host` alive until the copy has run
        model.bn_momentum_table.copy_(host, non_blocking=True)
        model._bn_momentum_host = values
    return model.bn_momentum_table
