"""BatchNorm momentum read from the device, without a GPU: argument validation of
b2r_bn_finalize_dev (every malformed call returns B2R_ERR_INVALID_ARG before anything is launched)
and the host side of pytorch_utils.sync_bn_momentum.  The kernels and the captured training step
are tested in test_bn_momentum_gpu.py."""
import ctypes
import io

import pytest
import torch
import torch.nn as nn

from test_bn_pool_glue_cpu import INVALID, P, _bn_finalize_args, _rejects

# each of these makes b2r_bn_finalize return B2R_ERR_INVALID_ARG (test_bn_pool_glue_cpu.py)
BAD = (dict(stats=None), dict(scale=None), dict(shift=None), dict(C=0), dict(C=-3),
       dict(count=0.0), dict(count=-1.0), dict(running_mean=None), dict(running_var=None))


def _dev_args(**kw):
    """b2r_bn_finalize_dev's arguments: b2r_bn_finalize's with the momentum as a pointer"""
    kw.setdefault("momentum", P)
    return _bn_finalize_args(**kw)


def test_bn_finalize_dev_rejects_what_the_by_value_entry_rejects():
    for kw in BAD:
        _rejects("b2r_bn_finalize", *_bn_finalize_args(**kw))
        _rejects("b2r_bn_finalize_dev", *_dev_args(**kw))


def test_bn_finalize_dev_rejects_running_statistics_without_a_momentum():
    _rejects("b2r_bn_finalize_dev", *_dev_args(momentum=None))
    # ... also when the call is malformed otherwise
    _rejects("b2r_bn_finalize_dev", *_dev_args(momentum=None, C=0))


def test_bn_finalize_dev_signature_takes_a_pointer():
    from backtoreality_b200 import _lib
    sig = _lib.SIGNATURES["b2r_bn_finalize_dev"]
    assert sig[6] is ctypes.c_void_p
    assert sig[:6] + sig[7:] == _lib.SIGNATURES["b2r_bn_finalize"][:6] + \
        _lib.SIGNATURES["b2r_bn_finalize"][7:]
    assert INVALID == -1


def _attach_on_cpu(m, momentum):
    """what sync_bn_momentum does to one module, with the slot in host memory"""
    from backtoreality_b200 import pytorch_utils
    m.momentum_slot = torch.tensor([momentum], dtype=torch.float32)
    m.__class__ = pytorch_utils._SLOT_CLASSES[type(m)]
    return m


@pytest.mark.parametrize("cls,shape", [(nn.BatchNorm1d, (6, 5)), (nn.BatchNorm1d, (3, 5, 7)),
                                       (nn.BatchNorm2d, (2, 5, 3, 4))])
def test_slot_forward_matches_torch_batchnorm(cls, shape):
    """The torch-path forward of an attached module: output and gradients of F.batch_norm in
    training mode, running statistics updated with the slot's momentum (unbiased variance)."""
    g = torch.Generator().manual_seed(3)
    x = torch.randn(shape, generator=g) * 2 + 0.5
    ref = cls(5, momentum=0.3)
    with torch.no_grad():
        ref.weight.copy_(torch.rand(5, generator=g) + 0.5)
        ref.bias.copy_(torch.randn(5, generator=g))
        ref.running_mean.copy_(torch.randn(5, generator=g))
        ref.running_var.copy_(torch.rand(5, generator=g) + 0.5)
    att = _attach_on_cpu(cls(5, momentum=0.9), 0.3)     # the slot, not .momentum, is read
    att.load_state_dict(ref.state_dict())
    assert isinstance(att, cls)
    xr, xa = x.clone().requires_grad_(), x.clone().requires_grad_()
    yr, ya = ref(xr), att(xa)
    assert torch.equal(yr, ya)
    w = torch.randn(shape, generator=g)
    (yr * w).sum().backward()
    (ya * w).sum().backward()
    for a, b in ((xr.grad, xa.grad), (ref.weight.grad, att.weight.grad), (ref.bias.grad, att.bias.grad)):
        assert torch.equal(a, b)
    for k in ("running_mean", "running_var"):
        a, b = getattr(ref, k), getattr(att, k)
        assert float((a - b).norm() / a.norm()) < 1e-6, k
    assert int(att.num_batches_tracked) == int(ref.num_batches_tracked) == 1
    # eval mode: torch's own forward on the running statistics
    att.load_state_dict(ref.state_dict())
    ref.eval(), att.eval()
    assert torch.equal(ref(x), att(x))


def test_attached_module_keeps_its_state_dict_and_pickles():
    from backtoreality_b200 import pytorch_utils
    net = nn.Sequential(nn.Conv1d(4, 4, 1), nn.BatchNorm1d(4), pytorch_utils.BatchNorm2d(4))
    before = {k: v.clone() for k, v in net.state_dict().items()}
    for m in net.modules():
        if type(m) in pytorch_utils._SLOT_CLASSES:
            _attach_on_cpu(m, 0.1)
    after = net.state_dict()
    assert list(after) == list(before)
    for k in before:
        assert torch.equal(after[k], before[k]), k
    buf = io.BytesIO()
    torch.save(net.state_dict(), buf)
    fresh = nn.Sequential(nn.Conv1d(4, 4, 1), nn.BatchNorm1d(4), pytorch_utils.BatchNorm2d(4))
    buf.seek(0)
    fresh.load_state_dict(torch.load(buf))
    buf = io.BytesIO()
    torch.save(net, buf)                  # the Slot* classes are importable: the module pickles
    buf.seek(0)
    again = torch.load(buf, weights_only=False)
    assert isinstance(again[1], nn.BatchNorm1d) and float(again[1].momentum_slot) == pytest.approx(0.1)


def test_slot_on_another_device_is_refused():
    from backtoreality_b200 import pytorch_utils
    bn = nn.BatchNorm1d(4)
    bn.momentum_slot = torch.zeros(1, device="meta")
    with pytest.raises(RuntimeError, match="slot"):
        pytorch_utils.momentum_slot(bn)


def test_sync_bn_momentum_needs_a_cuda_model():
    from backtoreality_b200 import pytorch_utils
    net = nn.Sequential(nn.BatchNorm1d(4))
    with pytest.raises(RuntimeError, match="CUDA"):
        pytorch_utils.sync_bn_momentum(net)
    with pytest.raises(ValueError, match="no BatchNorm"):
        pytorch_utils.sync_bn_momentum(nn.Sequential(nn.Conv1d(4, 4, 1)))
    assert type(net[0]) is nn.BatchNorm1d          # nothing attached


def test_scheduler_leaves_an_unattached_model_alone():
    from backtoreality_b200 import pytorch_utils
    net = nn.Sequential(nn.BatchNorm1d(4), nn.BatchNorm2d(3))
    bnm = pytorch_utils.BNMomentumScheduler(net, lambda e: max(0.5 * 0.5 ** (e // 20), 0.001))
    assert net[0].momentum == 0.5 and net[1].momentum == 0.5
    bnm.step(20)
    assert net[0].momentum == 0.25
    assert not hasattr(net, "bn_momentum_table") and type(net[0]) is nn.BatchNorm1d
