"""BatchNorm momentum that follows BNMomentumScheduler inside a replayed CUDA graph.

  1. b2r_bn_finalize_dev (momentum read from device memory) against b2r_bn_finalize (by value):
     bit-identical, eagerly and from a replayed graph whose momentum changes between replays.
  2. The captured VoteNet step (CapturedTrainStep, PipelinedTrainStep) of an attached model
     (pytorch_utils.sync_bn_momentum), its momentum changed by the scheduler between replays,
     against an unattached twin run eagerly with the same momenta.
  3. The same on VoteNet_DA (torch BatchNorm in the discriminators) and with the fused kernels
     off (every BatchNorm on the torch path), and the torch-path forward of one attached module
     against torch's own.
  4. Guards: no sync inside a capture, no momentum=None, state_dict unchanged.

The native BatchNorm sites run the same kernel with the same momentum as the twin, so their
running statistics must be bit-identical.  The torch-path update (`lerp_` from torch.var_mean)
rounds differently from cuDNN's, so those are held to a rel-L2 of 1e-6.  Measured errors go to
bn_momentum.log of the run's output directory when it exists (tests/_util.py emu_log).
"""
import ctypes
import io

import numpy as np
import pytest
import torch
import torch.nn as nn

from _util import emu_log, rel_l2
from backtoreality_b200 import scenes

pytestmark = pytest.mark.gpu

EPS = float(np.float32(1e-5))
TORCH_PATH_TOL = 1e-6
# the reference's schedule (train_Votenet_FSB.py: BN_MOMENTUM_INIT 0.5, decay 0.5 every 20 epochs,
# clipped at 0.001) at the epoch of each step: momentum 0.5, 0.5, 0.25, 0.001
EPOCHS = [0, 0, 20, 180]


def bn_lambda(epoch):
    return max(0.5 * 0.5 ** (epoch // 20), 0.001)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _call(name, *args):
    from backtoreality_b200 import _ext, _lib
    _lib.check(getattr(_lib.lib(), name)(*args, _ext._stream()), name)


def _log(name, **errs):
    emu_log(name, log="bn_momentum.log", **errs)


# ---- 1. the entry point ---------------------------------------------------------------------------

class _Finalize:
    """one b2r_bn_finalize problem: fp64 batch sums of z, fresh outputs for every call"""

    def __init__(self, cuda, count=4096, C=300):
        g = torch.Generator().manual_seed(11)
        z = (torch.randn(count, C, generator=g, dtype=torch.float64) * 1.5 + 0.7).to(cuda)
        self.C, self.count = C, float(count)
        self.stats = torch.cat([z.sum(0), (z * z).sum(0)])
        self.gamma = (torch.rand(C, generator=g) + 0.5).to(cuda)
        self.beta = torch.randn(C, generator=g).to(cuda)
        self.rm0 = torch.randn(C, generator=g).to(cuda)
        self.rv0 = (torch.rand(C, generator=g) + 0.25).to(cuda)

    def buffers(self, cuda):
        b = {k: torch.full((self.C,), float("nan"), device=cuda) for k in ("scale", "shift", "mean", "invstd")}
        b.update(rm=self.rm0.clone(), rv=self.rv0.clone(),
                 nbt=torch.tensor([41], dtype=torch.int64, device=cuda))
        return b

    def call(self, b, momentum):
        """momentum: a float (b2r_bn_finalize) or a one-element device tensor (_dev)"""
        dev = isinstance(momentum, torch.Tensor)
        _call("b2r_bn_finalize_dev" if dev else "b2r_bn_finalize", _p(self.stats), self.C, self.count,
              _p(self.gamma), _p(self.beta), EPS, _p(momentum) if dev else momentum,
              _p(b["rm"]), _p(b["rv"]), _p(b["scale"]), _p(b["shift"]), _p(b["mean"]), _p(b["invstd"]),
              _p(b["nbt"]))


def _assert_same(a, b, tag):
    for k in a:
        assert torch.equal(a[k], b[k]), (tag, k)


def test_bn_finalize_dev_equals_by_value(cuda):
    f = _Finalize(cuda)
    for m in (0.0, 0.001, 0.1, 0.5, 1.0):
        want, got = f.buffers(cuda), f.buffers(cuda)
        f.call(want, m)
        f.call(got, torch.tensor([m], dtype=torch.float32, device=cuda))
        torch.cuda.synchronize()
        _assert_same(want, got, m)
        assert int(got["nbt"]) == 42
        if m > 0:
            assert not torch.equal(got["rm"], f.rm0)


def test_bn_finalize_dev_replayed_follows_the_slot(cuda):
    f = _Finalize(cuda)
    slot = torch.tensor([0.5], dtype=torch.float32, device=cuda)
    got = f.buffers(cuda)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g):
            f.call(got, slot)
    torch.cuda.current_stream().wait_stream(side)
    g.replay()
    slot.copy_(torch.tensor([0.001]))
    g.replay()
    want = f.buffers(cuda)
    f.call(want, 0.5)
    f.call(want, 0.001)
    torch.cuda.synchronize()
    _assert_same(want, got, "replay")
    assert int(got["nbt"]) == 43
    # the capture-time momentum would give something else
    frozen = f.buffers(cuda)
    f.call(frozen, 0.5)
    f.call(frozen, 0.5)
    assert not torch.equal(frozen["rm"], got["rm"])


# ---- 2./3. the captured training step -------------------------------------------------------------

def _bns(net):
    return [(n, m) for n, m in net.named_modules() if isinstance(m, nn.modules.batchnorm._BatchNorm)]


def _make(cuda, da=False):
    from backtoreality_b200.votenet import VoteNet, VoteNet_DA
    torch.manual_seed(5)
    net = (VoteNet_DA if da else VoteNet)(4, 1, 4, np.ones((4, 3), np.float32), input_feature_dim=1,
                                          num_proposal=64, vote_factor=1, sampling="vote_fps")
    net = net.to(cuda).train()
    opt = torch.optim.SGD(net.parameters(), lr=0.0)

    def loss_of(pc, geometry):
        ep = net({"point_clouds": pc, "geometry": geometry})
        loss = (ep["proposal_scores_raw"] ** 2).mean() + ((ep["vote_xyz"] - ep["seed_xyz"]) ** 2).mean()
        if da:
            loss = loss + (ep["global_d_pred"] ** 2).mean() + (ep["local_d_pred"] ** 2).mean()
        return loss

    def step(pc, geometry=None):
        for p in net.parameters():
            p.grad = None
        if da:      # the BR step: source forward, then target forward
            half = pc.shape[0] // 2
            loss = loss_of(pc[:half], None) + loss_of(pc[half:], None)
        else:
            loss = loss_of(pc, geometry)
        loss.backward()
        opt.step()
        return loss.detach()
    return net, step


def _batches(cuda, scenes_per_step):
    return [torch.from_numpy(scenes.batch(300 + scenes_per_step * i, scenes_per_step, 8192, C=1,
                                          kind="room", dup=0.2)).to(cuda) for i in range(4)]


def _eager_twin(cuda, batches, da=False):
    """unattached, eager, `momentum` set by the scheduler before each step (the by-value path);
    -> (net, names of the BatchNorms that ran torch's forward)"""
    from backtoreality_b200.pytorch_utils import BNMomentumScheduler
    net, step = _make(cuda, da)
    torch_path = set()
    for name, m in _bns(net):
        m.register_forward_pre_hook(lambda mod, inp, name=name: torch_path.add(name))
    bnm = BNMomentumScheduler(net, bn_lambda)
    for epoch, b in zip(EPOCHS, batches):
        bnm.step(epoch)
        step(b)
    torch.cuda.synchronize()
    return net, torch_path


def _captured(cuda, batches, attach, da=False, pipelined=False):
    from backtoreality_b200.pytorch_utils import BNMomentumScheduler, sync_bn_momentum
    from backtoreality_b200.train_step import CapturedTrainStep, PipelinedTrainStep
    net, step = _make(cuda, da)
    bnm = BNMomentumScheduler(net, bn_lambda)
    if attach:
        sync_bn_momentum(net)
    if pipelined:
        net.pnet.vote_aggregation.sm_limit = (100, 120)
        run = PipelinedTrainStep(net.backbone_net, step, batches[0], warmup=2, fps_cluster=3,
                                 start_after_level=1, snapshot=[net])
        feed = batches[1:] + batches[:1]          # call i submits batch i+1 and trains on batch i
    else:
        run = CapturedTrainStep(step, batches[0], warmup=3, snapshot=[net])
        feed = batches
    for epoch, b in zip(EPOCHS, feed):
        bnm.step(epoch)                           # no recapture
        run(b)
    torch.cuda.synchronize()
    return net


def _compare(tag, twin, torch_path, net, native_exact=True):
    """running statistics of every BatchNorm of `net` against the twin's -> worst rel-L2"""
    worst = {"native": 0.0, "torch": 0.0}
    for (name, a), (name_b, b) in zip(_bns(twin), _bns(net)):
        assert name == name_b
        assert int(a.num_batches_tracked) == int(b.num_batches_tracked), name
        kind = "torch" if name in torch_path else "native"
        for k in ("running_mean", "running_var"):
            x, y = getattr(a, k), getattr(b, k)
            if kind == "native" and native_exact:
                assert torch.equal(x, y), (tag, name, k)
            e = rel_l2(y.cpu().numpy(), x.cpu().numpy())
            worst[kind] = max(worst[kind], e)
            assert e <= TORCH_PATH_TOL, (tag, name, k, e)
    n_torch = sum(1 for n, _ in _bns(net) if n in torch_path)
    _log("%s: %d native, %d torch-path BatchNorms" % (tag, len(_bns(net)) - n_torch, n_torch), **worst)
    return n_torch


def _assert_schedule_mattered(tag, twin, frozen):
    """the capture-time momentum (an unattached captured step) ends somewhere else entirely"""
    diffs = sorted(rel_l2(getattr(b, k).cpu().numpy(), getattr(a, k).cpu().numpy())
                   for (_, a), (_, b) in zip(_bns(twin), _bns(frozen))
                   for k in ("running_mean", "running_var"))
    _log("%s: frozen momentum vs schedule" % tag, median=diffs[len(diffs) // 2], max=diffs[-1])
    assert diffs[len(diffs) // 2] > 1e-2, diffs


def test_captured_votenet_step_follows_the_scheduler(cuda):
    batches = _batches(cuda, 2)
    twin, torch_path = _eager_twin(cuda, batches)
    net = _captured(cuda, batches, attach=True)
    _compare("votenet captured", twin, torch_path, net)
    assert all(int(m.num_batches_tracked) == 4 for _, m in _bns(net))
    _assert_schedule_mattered("votenet captured", twin, _captured(cuda, batches, attach=False))


def test_pipelined_votenet_step_follows_the_scheduler(cuda):
    # capped grids change the summation order of the BatchNorm statistics: rel-L2, not bits
    batches = _batches(cuda, 2)
    twin, torch_path = _eager_twin(cuda, batches)
    net = _captured(cuda, batches, attach=True, pipelined=True)
    _compare("votenet pipelined", twin, torch_path, net, native_exact=False)
    assert all(int(m.num_batches_tracked) == 4 for _, m in _bns(net))


def test_captured_br_step_follows_the_scheduler(cuda):
    batches = _batches(cuda, 4)                     # 2 + 2 scenes: two forwards per step
    twin, torch_path = _eager_twin(cuda, batches, da=True)
    net = _captured(cuda, batches, attach=True, da=True)
    n_torch = _compare("votenet_da captured", twin, torch_path, net)
    assert n_torch >= 4                             # the discriminators' BatchNorm1d
    assert int(net.global_netD1[1].num_batches_tracked) == 8
    _assert_schedule_mattered("votenet_da captured", twin,
                              _captured(cuda, batches, attach=False, da=True))


def test_captured_unfused_step_follows_the_scheduler(cuda, monkeypatch):
    from backtoreality_b200 import fused_sa
    monkeypatch.setattr(fused_sa, "ENABLED", False)
    batches = _batches(cuda, 2)
    twin, torch_path = _eager_twin(cuda, batches)
    net = _captured(cuda, batches, attach=True)
    n_torch = _compare("votenet unfused captured", twin, torch_path, net)
    assert n_torch == len(_bns(net))                # every BatchNorm on the torch path


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({e.key for e in prof.key_averages() if e.device_type.name == "CUDA"})


@pytest.mark.parametrize("cls,shape", [(nn.BatchNorm1d, (8, 256, 1024)),     # global_netD1
                                       (nn.BatchNorm1d, (8, 128, 256)),      # local_netD
                                       (nn.BatchNorm2d, (2, 128, 256, 16))])  # an unfused SA layer
def test_torch_path_forward_matches_torch(cuda, cls, shape):
    """Output and gradients of an attached module against the same unattached module: bit for bit
    when torch runs the same BatchNorm kernels for both, else within 1e-6 (logged with the
    kernels that ran)."""
    from backtoreality_b200.pytorch_utils import sync_bn_momentum
    g = torch.Generator().manual_seed(7)
    x = (torch.randn(shape, generator=g) * 1.3 + 0.4).to(cuda)
    w = torch.randn(shape, generator=g).to(cuda)
    ref = cls(shape[1], momentum=0.3).to(cuda).train()
    with torch.no_grad():
        ref.weight.copy_(torch.rand(shape[1], generator=g) + 0.5)
        ref.bias.copy_(torch.randn(shape[1], generator=g))
    att = cls(shape[1], momentum=0.3).to(cuda).train()
    att.load_state_dict(ref.state_dict())
    sync_bn_momentum(nn.Sequential(att))
    res = {}
    for tag, mod in (("torch", ref), ("attached", att)):
        xi = x.clone().requires_grad_()

        def run():
            y = mod(xi)
            (y * w).sum().backward()
            res[tag] = (y.detach(), xi.grad, mod.weight.grad, mod.bias.grad)
        res[tag + "_kernels"] = [k for k in _kernels(run) if "norm" in k.lower() or "bn_" in k.lower()]
    same_kernels = res["torch_kernels"] == res["attached_kernels"]
    errs = {n: rel_l2(b.cpu().numpy(), a.cpu().numpy())
            for n, a, b in zip(("out", "g_in", "g_weight", "g_bias"), res["torch"], res["attached"])}
    for k in ("running_mean", "running_var"):
        errs[k] = rel_l2(getattr(att, k).cpu().numpy(), getattr(ref, k).cpu().numpy())
    _log("torch path %s%s same_kernels=%s torch=%s attached=%s" % (
        cls.__name__, shape, same_kernels, res["torch_kernels"], res["attached_kernels"]), **errs)
    for n, a, b in zip(("out", "g_in", "g_weight", "g_bias"), res["torch"], res["attached"]):
        if same_kernels:
            assert torch.equal(a, b), n
        else:
            assert errs[n] <= TORCH_PATH_TOL, (n, errs[n])
    assert errs["running_mean"] <= TORCH_PATH_TOL and errs["running_var"] <= TORCH_PATH_TOL, errs
    assert int(att.num_batches_tracked) == 1


# ---- 4. guards ------------------------------------------------------------------------------------

def test_sync_bn_momentum_guards_and_state_dict(cuda):
    from backtoreality_b200.pytorch_utils import BNMomentumScheduler, sync_bn_momentum
    net, _ = _make(cuda, da=True)
    before = {k: v.clone() for k, v in net.state_dict().items()}
    table = sync_bn_momentum(net)
    after = net.state_dict()
    assert list(after) == list(before)
    for k in before:
        assert torch.equal(after[k], before[k]), k
    n = len(_bns(net))
    assert table.shape == (n,) and torch.equal(table, torch.full((n,), 0.1, device=cuda))
    assert all(isinstance(m, (nn.BatchNorm1d, nn.BatchNorm2d)) for _, m in _bns(net))
    # the scheduler writes the same table; it is never reallocated
    bnm = BNMomentumScheduler(net, bn_lambda)
    bnm.step(20)
    assert net.bn_momentum_table is table and sync_bn_momentum(net) is table
    assert torch.equal(table, torch.full((n,), 0.25, device=cuda))
    # save / load round trip: into an unattached model and back into the attached one
    buf = io.BytesIO()
    torch.save(net.state_dict(), buf)
    buf.seek(0)
    sd = torch.load(buf)
    fresh, _ = _make(cuda, da=True)
    fresh.load_state_dict(sd)
    net.load_state_dict(sd)
    # a capture must not record the table write
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError, match="capture"):
        with torch.cuda.stream(side), torch.cuda.graph(g):
            sync_bn_momentum(net)
    torch.cuda.synchronize()
    # momentum=None (cumulative average) is not supported
    net.vgen.bn1.momentum = None
    with pytest.raises(ValueError, match="None"):
        sync_bn_momentum(net)
