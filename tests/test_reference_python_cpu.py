"""Checks that need the reference tree (oracle/ref_python.py: B2R_REFERENCE_ROOT); skipped without it.

* the reference's ONLY test, pointnet2_test.py:18-30 (gradcheck of three_interpolate), run
  verbatim in spirit on CPU over the oracle `_ext` (double perturbation is applied by gradcheck
  to a float32 op, hence the reference's own loose atol=rtol=1e-1);
* the oracle's module port equals the reference Python modules with IDENTICAL weights
  (state_dict interchange), forward and backward;
* this repo's product modules expose the reference's state-dict layout.
"""
import numpy as np
import pytest
import torch

from _util import pattern_like, rel_l2
from backtoreality_b200 import scenes
from oracle import cpu_modules, ref_python

pytestmark = pytest.mark.skipif(not ref_python.available(), reason="reference tree not present")


def test_reference_interpolation_gradcheck_on_oracle_ext():
    rs = ref_python.RefStack("votenet")
    torch.manual_seed(0)
    feats = torch.randn(1, 2, 4).float().requires_grad_(True)

    def interpolate_func(inputs):
        idx = torch.from_numpy(np.array([[[0, 1, 2], [1, 2, 3]]])).int()
        weight = torch.from_numpy(np.array([[[1, 1, 1], [2, 2, 2]]])).float()
        return rs.pointnet2_utils.three_interpolate(inputs, idx, weight)

    assert torch.autograd.gradcheck(interpolate_func, feats, atol=1e-1, rtol=1e-1)


@pytest.mark.parametrize("flavour,C,fp2_out", [("votenet", 1, 256), ("groupfree3d", 0, 288)])
def test_oracle_port_equals_reference_modules(flavour, C, fp2_out):
    rs = ref_python.RefStack(flavour)
    torch.manual_seed(5)
    ref = rs.backbone_module.Pointnet2Backbone(input_feature_dim=C).train()
    port = cpu_modules.Backbone(input_feature_dim=C, fp2_out=fp2_out).train()
    port.load_state_dict(ref.state_dict())
    pc = torch.from_numpy(scenes.batch(9, 2, 2500, C=C, kind="room", dup=0.2))
    a, b = ref(pc), port(pc)
    for k in a:
        if a[k].dtype == torch.int32:
            assert torch.equal(a[k], b[k]), k
        else:
            assert rel_l2(b[k].detach().numpy(), a[k].detach().numpy()) < 1e-6, k
    (a["fp2_features"] * pattern_like(a["fp2_features"])).sum().backward()
    (b["fp2_features"] * pattern_like(b["fp2_features"])).sum().backward()
    for (n1, p1), (n2, p2) in zip(ref.named_parameters(), port.named_parameters()):
        assert n1 == n2
        assert rel_l2(p2.grad.numpy(), p1.grad.numpy()) < 1e-4, n1


def test_product_modules_have_the_reference_state_dict_layout():
    from backtoreality_b200.backbone_module import Pointnet2Backbone
    for flavour, C, fp2_out in [("votenet", 1, 256), ("groupfree3d", 0, 288)]:
        ref = ref_python.RefStack(flavour).backbone_module.Pointnet2Backbone(input_feature_dim=C)
        mine = Pointnet2Backbone(input_feature_dim=C, fp2_out=fp2_out)
        sd_r, sd_m = ref.state_dict(), mine.state_dict()
        assert list(sd_r.keys()) == list(sd_m.keys())
        for k in sd_r:
            assert sd_r[k].shape == sd_m[k].shape, k
        mine.load_state_dict(sd_r)


def test_nn_distance_oracle_equals_reference_module_on_cpu():
    """The oracle's restatement of utils/nn_distance.py (the checker of the product's arg-min
    kernel in tests/test_ops_gpu.py) against the reference's own module, when the reference tree
    is present (build container); the product itself has no CPU path."""
    import importlib.util
    import os

    import pytest
    import torch
    path = os.path.join(ref_python.REF_ROOT, "detection", "Votenet", "utils", "nn_distance.py")
    if not os.path.isfile(path):
        pytest.skip("reference tree not present")
    spec = importlib.util.spec_from_file_location("ref_nn_distance", path)
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    from backtoreality_b200 import nn_distance as nd
    from oracle import cpu_modules
    g = torch.Generator().manual_seed(4)
    p1, p2 = torch.rand(3, 40, 3, generator=g), torch.rand(3, 17, 3, generator=g)
    for kw in ({}, {"l1": True}, {"l1smooth": True, "delta": 0.25}):
        got, want = cpu_modules.nn_distance(p1, p2, **kw), ref.nn_distance(p1, p2, **kw)
        for a, b in zip(got, want):
            assert torch.equal(a, b)
    e = torch.randn(50, generator=g)
    assert torch.equal(nd.huber_loss(e, 0.4), ref.huber_loss(e, 0.4))
    with pytest.raises(RuntimeError, match="CPU not supported"):
        nd.nn_distance(p1, p2)


def test_gf3d_query_modules_state_dict_matches_reference():
    """backtoreality_b200.gf3d_modules mirrors G/models/modules.py:16-100: same state-dict keys and
    shapes, and (on CPU, where the modules run the reference's own torch formulation) the same
    outputs for the same weights."""
    if not ref_python.available():
        pytest.skip("reference tree not present")
    from backtoreality_b200 import gf3d_modules as ours
    rg = ref_python.RefStack("groupfree3d")
    ref = rg.gf_modules
    for name, args in (("PointsObjClsModule", (288,)), ("PositionEmbeddingLearned", (3, 288)),
                       ("PositionEmbeddingLearned", (6, 64))):
        torch.manual_seed(0)
        a = getattr(ref, name)(*args)
        torch.manual_seed(0)
        b = getattr(ours, name)(*args)
        sa, sb = a.state_dict(), b.state_dict()
        assert list(sa) == list(sb)
        for k in sa:
            assert sa[k].shape == sb[k].shape and torch.equal(sa[k], sb[k]), k
        a.eval(); b.eval()
        x = torch.randn(2, 288, 50) if name == "PointsObjClsModule" else torch.randn(2, 50, args[0])
        assert torch.allclose(a(x), b(x), atol=1e-6)
