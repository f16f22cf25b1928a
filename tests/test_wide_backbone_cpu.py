"""GroupFree3D's width / depth backbone tables and the channel-slice plan of the fused SA layers,
checked without a GPU: module construction, and the library's host-side shape rules."""
import ctypes
import json
import os

import pytest
import torch

from backtoreality_b200 import _lib, fused_sa
from backtoreality_b200.backbone_module import Pointnet2Backbone


def _reference_tables(fdim, fp2_out, width, depth):
    """Channel tables of the GroupFree3D reference constructor (models/backbone_module.py)."""
    w, d = width, depth
    sa = [[fdim] + [64 * w] * d + [128 * w], [128 * w] + [128 * w] * d + [256 * w],
          [256 * w] + [128 * w] * d + [256 * w], [256 * w] + [128 * w] * d + [256 * w]]
    fp = [[512 * w, 256 * w, 256 * w], [512 * w, 256 * w, fp2_out]]
    return sa, fp


def _expected_state(fdim, fp2_out, width, depth):
    sa, fp = _reference_tables(fdim, fp2_out, width, depth)
    want = {}

    def layer(prefix, cin, cout, conv_dims):
        want[prefix + ".conv.weight"] = (cout, cin) + (1,) * conv_dims
        for k in ("weight", "bias", "running_mean", "running_var"):
            want[prefix + ".bn.bn." + k] = (cout,)
        want[prefix + ".bn.bn.num_batches_tracked"] = ()

    for s, mlp in enumerate(sa):
        mlp = [mlp[0] + 3] + mlp[1:]
        for i in range(len(mlp) - 1):
            layer("sa%d.mlp_module.layer%d" % (s + 1, i), mlp[i], mlp[i + 1], 2)
    for f, mlp in enumerate(fp):
        for i in range(len(mlp) - 1):
            layer("fp%d.mlp.layer%d" % (f + 1, i), mlp[i], mlp[i + 1], 2)
    return want


@pytest.mark.parametrize("width,depth", [(1, 2), (2, 2), (1, 3), (2, 3)])
def test_state_dict_follows_reference_formula(width, depth):
    sd = Pointnet2Backbone(input_feature_dim=0, fp2_out=288, width=width, depth=depth).state_dict()
    want = _expected_state(0, 288, width, depth)
    assert {k: tuple(v.shape) for k, v in sd.items()} == want


def test_default_width_depth_builds_todays_module():
    torch.manual_seed(123)
    a = Pointnet2Backbone(input_feature_dim=1, fp2_out=256).state_dict()
    torch.manual_seed(123)
    b = Pointnet2Backbone(input_feature_dim=1, fp2_out=256, width=1, depth=2).state_dict()
    assert list(a) == list(b)
    for k in a:
        assert torch.equal(a[k], b[k]), k
    # the width-1 channel table the project has always built (VoteNet / GF3D defaults)
    assert [blk.conv.out_channels for blk in Pointnet2Backbone(1).sa2.mlp_module] == [128, 128, 256]


@pytest.mark.parametrize("width,depth", [(0, 2), (2, 0), (1.5, 2)])
def test_bad_width_depth_rejected(width, depth):
    with pytest.raises(ValueError):
        Pointnet2Backbone(width=width, depth=depth)


def _sa_layers(fdim, width, depth):
    """(NP, NS, Cin, Cout, gather, last) of every SA layer of the backbone."""
    sa, _ = _reference_tables(fdim, 288, width, depth)
    out = []
    for (NP, NS), mlp in zip([(2048, 64), (1024, 32), (512, 16), (256, 16)], sa):
        L = len(mlp) - 1
        for i in range(L):
            out.append((NP, NS, mlp[i] + (3 if i == 0 else 0), mlp[i + 1], int(i == 0),
                        int(i == L - 1)))
    return out


def _grid(fn, cin, cout, gather, last):
    co, ci = ctypes.c_int(), ctypes.c_int()
    n = getattr(_lib.lib(), fn)(cin, cout, gather, last, ctypes.byref(co), ctypes.byref(ci))
    return n, co.value, ci.value


@pytest.mark.parametrize("B", [2, 4])
@pytest.mark.parametrize("depth", [2, 3])
def test_w2x_backbone_every_layer_covered(B, depth):
    lib = _lib.lib()
    sliced = 0
    for NP, NS, cin, cout, g, last in _sa_layers(0, 2, depth):
        assert lib.b2r_sa_layer_fwd_supported(B, NP, NS, cin, cout, g, last), (cin, cout)
        assert lib.b2r_sa_layer_bwd_supported(B, NP, NS, cin, cout, g, last), (cin, cout)
        for fn in ("b2r_sa_layer_fwd_slices", "b2r_sa_layer_bwd_slices"):
            n, co, ci = _grid(fn, cin, cout, g, last)
            assert n >= 1
            sliced += n > 1
            if n > 1:
                assert co in (128, 256) and (ci == 0 or (g and not last and ci % 8 == 0))
    assert sliced > 0
    # the host's grid tiles every output and feature channel exactly once
    for NP, NS, cin, cout, g, last in _sa_layers(0, 2, depth):
        for bwd in (False, True):
            cover = torch.zeros(cout, max(cin - 3, 1), dtype=torch.int32)
            for co0, co_n, ci0, ci_n in fused_sa.slice_grid(bwd, cin, cout, g, last):
                co_n = co_n or cout
                ci_n = ci_n or max(cin - 3, 1)
                cover[co0:co0 + co_n, ci0:ci0 + ci_n] += 1
            assert bool((cover == 1).all()), (cin, cout, bwd)


_PARENT_TILES = os.path.join(os.path.dirname(__file__), "golden", "sa_layer_tiles_w1.json")


def test_todays_layers_one_launch_same_tile():
    """Every SA layer of the VoteNet, BR and GroupFree3D configurations (backbones with 0 and 1
    input features, vote aggregation, the centre-refine head) runs as ONE unsliced launch with the
    tile recorded before channel slices existed (tests/golden/sa_layer_tiles_w1.json: B, NP, NS,
    Cin, Cout, gather, top, then fwd / bwd tile without and with a plan, bwd tile without dgrad)."""
    lib = _lib.lib()
    with open(_PARENT_TILES) as f:
        rows = json.load(f)
    assert len(rows) > 100
    for r in rows:
        B, NP, NS, cin, cout, g, top = r[:7]
        for fn in ("b2r_sa_layer_fwd_slices", "b2r_sa_layer_bwd_slices"):
            assert _grid(fn, cin, cout, g, top) == (1, cout, 0), (fn, r)
        assert fused_sa.slice_grid(False, cin, cout, g, top) == ((0, 0, 0, 0),)
        got = []
        for cmp in (0, 1):
            got.append(lib.b2r_sa_layer_fwd_tile(B, NP, NS, cin, cout, g, top, cmp))
            got.append(lib.b2r_sa_layer_bwd_tile(B, NP, NS, cin, cout, g, top, 1, cmp))
        got.append(lib.b2r_sa_layer_bwd_tile(B, NP, NS, cin, cout, g, top, 0, 0))
        assert got == r[7:], r


def _fwd_desc(**kw):
    d = _lib.SaLayer()
    d.B, d.N, d.NP, d.NS, d.Cin, d.Cout, d.mode, d.epilogue = 2, 64, 16, 32, 259, 256, 0, 0
    fake = ctypes.c_void_p(4096)   # never dereferenced: validation fails first
    d.xyz = d.new_xyz = d.feat_t = d.idx = d.w_image = d.z = fake
    d.radius = 0.4
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def _bwd_desc(**kw):
    b = _lib.SaLayerBwd()
    b.B, b.N, b.NP, b.NS, b.Cin, b.Cout, b.mode = 2, 64, 16, 32, 259, 256, 0
    fake = ctypes.c_void_p(4096)
    b.xyz = b.new_xyz = b.feat_t = b.idx = b.w_image_bf16 = b.dW = fake
    b.gr = b.z = b.coef_a = b.coef_b = b.coef_c = b.g_feat_t = fake
    b.radius = 0.4
    for k, v in kw.items():
        setattr(b, k, v)
    return b


@pytest.mark.parametrize("kw", [dict(co0=128, co_n=256), dict(co0=-8, co_n=128), dict(co0=8),
                                dict(co_n=-1), dict(ci0=128, ci_n=256), dict(ci0=4, ci_n=128),
                                dict(ci0=8), dict(ci_n=12), dict(accumulate=2),
                                dict(ci_n=128, mode=1, Cin=256)])
def test_fwd_malformed_slice_rejected(kw):
    d = _fwd_desc(**kw)
    assert _lib.lib().b2r_sa_layer_fwd(ctypes.byref(d), None) == -1


def test_fwd_accumulate_on_pooled_layer_rejected():
    d = _fwd_desc(accumulate=1, epilogue=1, zmax=ctypes.c_void_p(4096))
    assert _lib.lib().b2r_sa_layer_fwd(ctypes.byref(d), None) == -1


@pytest.mark.parametrize("kw", [dict(co0=128, co_n=256), dict(co0=4, co_n=128), dict(co0=8),
                                dict(ci0=256, ci_n=128), dict(ci0=4, ci_n=128), dict(ci_n=-8),
                                dict(accumulate=1), dict(accumulate=1, co0=128, co_n=128),
                                dict(ci_n=64, mode=1, Cin=256)])
def test_bwd_malformed_slice_rejected(kw):
    b = _bwd_desc(**kw)
    if kw.get("mode") == 1:
        b.z_prev = b.scale_prev = b.shift_prev = b.gr_prev = ctypes.c_void_p(4096)
    assert _lib.lib().b2r_sa_layer_bwd(ctypes.byref(b), None) == -1
