"""INTEGRATION.md option A, executed: the reference's UNMODIFIED Python (pointnet2_utils.py,
pointnet2_modules.py, pytorch_utils.py, models/backbone_module.py -- vendored byte for byte under
baseline/_ref by scripts/vendor_reference.py) imported on top of the repo's `pointnet2/_ext.py`
shim, i.e. the nine pybind functions of _ext_src/src/bindings.cpp:11-24 served by libb2r.so
through the C ABI.  The reference's own modules must then reproduce the fixtures that
tests/golden/make_golden.py generated from the same modules on the CPU oracle.

Skipped when baseline/_ref is absent (it is git-ignored; the build container creates it).
"""
import os

import numpy as np
import pytest
import torch

from _util import golden, pattern_like, rel_l2, sub, weight_checksum

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref")


@pytest.fixture(scope="module")
def stacks(cuda):
    from oracle import ref_python
    if not ref_python.available(REF):
        pytest.skip("baseline/_ref not vendored (python scripts/vendor_reference.py)")
    import pointnet2._ext as shim          # the product's drop-in for the reference's extension
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield {f: ref_python.RefStack(f, ref_root=REF, ext=shim) for f in ("votenet", "groupfree3d")}
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@pytest.mark.parametrize("name,flavour,C", [("backbone_votenet_eval.npz", "votenet", 1),
                                           ("backbone_votenet_train.npz", "votenet", 1),
                                           ("backbone_gf3d_train.npz", "groupfree3d", 0)])
def test_reference_backbone_runs_unmodified_on_libb2r(cuda, stacks, name, flavour, C):
    from backtoreality_b200 import _ext, scenes
    g = golden(name)
    rs = stacks[flavour]
    torch.manual_seed(int(g["seed"]))
    net = rs.backbone_module.Pointnet2Backbone(input_feature_dim=C)
    assert abs(weight_checksum(net) - float(g["wsum"])) < 1e-6 * float(g["wsum"])
    net = net.cuda().train(bool(g["train"]))
    pc = torch.from_numpy(scenes.batch(50, int(g["B"]), int(g["N"]), C=C, kind="room", dup=0.2)).cuda()
    before = _ext.LAUNCHES
    ep = net(pc)
    assert _ext.LAUNCHES - before >= 14        # 4 x (FPS, gather, ball query, 2 x group) at least
    assert np.array_equal(ep["sa1_inds"].cpu().numpy(), g["sa1_inds"])
    assert np.array_equal(ep["sa2_inds"].cpu().numpy(), g["sa2_inds"])
    for k in ("sa1_features", "sa2_features", "sa3_features", "sa4_features", "fp2_features"):
        assert rel_l2(sub(ep[k]), g[k]) < 1e-4, k
    (ep["fp2_features"] * pattern_like(ep["fp2_features"])).sum().backward()
    for k, p in (("g_sa1_l0", net.sa1.mlp_module.layer0.conv.weight),
                 ("g_sa2_l0", net.sa2.mlp_module.layer0.conv.weight),
                 ("g_sa4_l2", net.sa4.mlp_module.layer2.conv.weight),
                 ("g_fp1_l0", net.fp1.mlp.layer0.conv.weight),
                 ("g_fp2_l1_bn", net.fp2.mlp.layer1.bn.bn.weight)):
        assert rel_l2(sub(p.grad), g[k]) < 1e-2, k


def test_reference_vote_aggregation_and_fp_module_on_libb2r(cuda, stacks):
    rs = stacks["votenet"]
    g = golden("vote_aggregation.npz")
    torch.manual_seed(int(g["seed"]))
    sa = rs.pointnet2_modules.PointnetSAModuleVotes(npoint=64, radius=0.3, nsample=16,
                                                   mlp=[32, 32, 32, 32], use_xyz=True,
                                                   normalize_xyz=True).cuda()
    gen = torch.Generator().manual_seed(int(g["seed"]) + 1)
    xyz = (torch.rand(2, 256, 3, generator=gen) * 2.0 + 0.5).cuda().requires_grad_(True)
    feats = torch.randn(2, 32, 256, generator=gen).cuda().requires_grad_(True)
    new_xyz, new_feats, inds = sa(xyz, feats)
    assert np.array_equal(inds.cpu().numpy(), g["inds"])
    assert rel_l2(new_feats.detach().cpu().numpy(), g["new_feats"]) < 1e-4
    ((new_feats * pattern_like(new_feats)).sum() + (new_xyz * 0.37).sum()).backward()
    assert rel_l2(xyz.grad.cpu().numpy(), g["g_xyz"]) < 1e-2
    g = golden("fp_module.npz")
    torch.manual_seed(int(g["seed"]))
    fp = rs.pointnet2_modules.PointnetFPModule(mlp=[48 + 16, 32, 24]).cuda()
    gen = torch.Generator().manual_seed(int(g["seed"]) + 1)
    unknown = torch.rand(2, 100, 3, generator=gen)
    known = torch.rand(2, 37, 3, generator=gen)
    known[:, 5] = known[:, 2]
    uf = torch.randn(2, 16, 100, generator=gen).cuda()
    kf = torch.randn(2, 48, 37, generator=gen).cuda()
    y = fp(unknown.cuda(), known.cuda(), uf, kf)
    assert rel_l2(y.detach().cpu().numpy(), g["y"]) < 1e-4


@pytest.fixture
def stack(cuda, monkeypatch):
    """The reference stack as oracle/cpu_modules.py restates it (same `_ext` calls as
    pointnet2_utils.py; held to the same fixtures on the CPU oracle by tests/test_golden_cpu.py)
    with the product's drop-in for the reference's extension as `_ext`: the shim meets the
    reference-generated fixtures on every checkout, also where the reference tree is absent."""
    import pointnet2._ext as shim
    from oracle import cpu_modules
    monkeypatch.setattr(cpu_modules, "_ext", shim)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    return cpu_modules


@pytest.mark.parametrize("name", ["backbone_votenet_eval.npz", "backbone_votenet_train.npz",
                                  "backbone_gf3d_train.npz"])
def test_port_backbone_runs_on_libb2r_shim(cuda, stack, name):
    from backtoreality_b200 import _ext, scenes
    g = golden(name)
    C = int(g["C"])
    torch.manual_seed(int(g["seed"]))
    net = stack.Backbone(input_feature_dim=C, fp2_out=int(g["fp2_out"]))
    assert abs(weight_checksum(net) - float(g["wsum"])) < 1e-6 * float(g["wsum"])
    net = net.cuda().train(bool(g["train"]))
    pc = torch.from_numpy(scenes.batch(50, int(g["B"]), int(g["N"]), C=C, kind="room", dup=0.2)).cuda()
    before = _ext.LAUNCHES
    ep = net(pc)
    assert _ext.LAUNCHES - before >= 14        # 4 x (FPS, gather, ball query, 2 x group) at least
    assert np.array_equal(ep["sa1_inds"].cpu().numpy(), g["sa1_inds"])
    assert np.array_equal(ep["sa2_inds"].cpu().numpy(), g["sa2_inds"])
    for k in ("sa1_features", "sa2_features", "sa3_features", "sa4_features", "fp2_features"):
        assert rel_l2(sub(ep[k]), g[k]) < 1e-4, k
    (ep["fp2_features"] * pattern_like(ep["fp2_features"])).sum().backward()
    for k, p in (("g_sa1_l0", net.sa1.mlp_module.layer0.conv.weight),
                 ("g_sa2_l0", net.sa2.mlp_module.layer0.conv.weight),
                 ("g_sa4_l2", net.sa4.mlp_module.layer2.conv.weight),
                 ("g_fp1_l0", net.fp1.mlp.layer0.conv.weight),
                 ("g_fp2_l1_bn", net.fp2.mlp.layer1.bn.bn.weight)):
        assert rel_l2(sub(p.grad), g[k]) < 1e-2, k


def test_port_vote_aggregation_and_fp_module_on_libb2r_shim(cuda, stack):
    g = golden("vote_aggregation.npz")
    torch.manual_seed(int(g["seed"]))
    sa = stack.SAModuleVotes(npoint=64, radius=0.3, nsample=16, mlp=[32, 32, 32, 32],
                             normalize_xyz=True)
    assert abs(weight_checksum(sa) - float(g["wsum"])) < 1e-6 * float(g["wsum"])
    sa = sa.cuda()
    gen = torch.Generator().manual_seed(int(g["seed"]) + 1)
    xyz = (torch.rand(2, 256, 3, generator=gen) * 2.0 + 0.5).cuda().requires_grad_(True)
    feats = torch.randn(2, 32, 256, generator=gen).cuda().requires_grad_(True)
    new_xyz, new_feats, inds = sa(xyz, feats)
    assert np.array_equal(inds.cpu().numpy(), g["inds"])
    assert rel_l2(new_feats.detach().cpu().numpy(), g["new_feats"]) < 1e-4
    ((new_feats * pattern_like(new_feats)).sum() + (new_xyz * 0.37).sum()).backward()
    assert rel_l2(xyz.grad.cpu().numpy(), g["g_xyz"]) < 1e-2
    g = golden("fp_module.npz")
    torch.manual_seed(int(g["seed"]))
    fp = stack.FPModule(mlp=[48 + 16, 32, 24])
    assert abs(weight_checksum(fp) - float(g["wsum"])) < 1e-6 * float(g["wsum"])
    fp = fp.cuda()
    gen = torch.Generator().manual_seed(int(g["seed"]) + 1)
    unknown = torch.rand(2, 100, 3, generator=gen)
    known = torch.rand(2, 37, 3, generator=gen)
    known[:, 5] = known[:, 2]
    uf = torch.randn(2, 16, 100, generator=gen).cuda()
    kf = torch.randn(2, 48, 37, generator=gen).cuda()
    y = fp(unknown.cuda(), known.cuda(), uf, kf)
    assert rel_l2(y.detach().cpu().numpy(), g["y"]) < 1e-4
