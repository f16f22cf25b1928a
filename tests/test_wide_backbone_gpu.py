"""Channel-sliced fused SA layers and GroupFree3D's width-2 backbone on the GPU.

Per layer: a sliced launch grid against the operand-rounding emulation (TF32 forward / BF16
backward operands, fp64 products) at test_mlp_gpu.py's bounds, and against the same layer in one
launch where both cover it.  Per block and step: the w2x backbone, fused against the unfused
(QueryAndGroup + cuDNN) arm from the same weights, and its captured / pipelined training step
against the eager one."""
import copy
import ctypes

import numpy as np
import pytest
import torch

from _util import emu_log, rel_l2, round_bf16, round_tf32

pytestmark = pytest.mark.gpu
# test_mlp_gpu.py's bounds: TF32 / BF16 against fp64, and against the operand-rounding emulation
# (the feature slices' partial sums add one fp32 rounding per slice, far below these)
TF32_TOL, BF16_TOL = 2e-3, 1e-2
EMU_TOL_FWD, EMU_TOL_BWD = 3e-6, 5e-5
LOG = "wide_emulation_parity.log"


def _vp(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _fwd(d):
    from backtoreality_b200 import _ext, _lib
    _lib.check(_lib.lib().b2r_sa_layer_fwd(ctypes.byref(d), _ext._stream()), "sa_layer_fwd")


def _bwd(b):
    from backtoreality_b200 import _ext, _lib
    _lib.check(_lib.lib().b2r_sa_layer_bwd(ctypes.byref(b), _ext._stream()), "sa_layer_bwd")


def _geometry(cuda, B, N, C, NP, NS, radius, seed):
    from backtoreality_b200 import pointnet2_utils, scenes
    pc = torch.from_numpy(scenes.batch(seed, B, N, C=1, kind="room", dup=0.2)).to(cuda)
    xyz = pc[..., :3].contiguous()
    g = torch.Generator(device=cuda).manual_seed(seed)
    feat_t = torch.randn(B, N, C, device=cuda, generator=g)
    inds = pointnet2_utils.furthest_point_sample(xyz, NP)
    new_xyz = torch.gather(xyz, 1, inds.long()[..., None].expand(-1, -1, 3)).contiguous()
    idx = pointnet2_utils.ball_query(radius, NS, xyz, new_xyz)
    return xyz, new_xyz, feat_t, idx


@pytest.mark.parametrize("C,NP,NS", [(256, 512, 32), (512, 256, 16)])
def test_sliced_gather_layer_forward_vs_emulation(cuda, C, NP, NS):
    """259 -> 256 (two output slices) and 515 -> 256 (output AND feature slices, partial z)
    gather layers: z against fp64 products of TF32-rounded operands, statistics against z."""
    from backtoreality_b200 import fused_sa
    B, N, Cout, radius = 2, 4096, 256, 0.4
    xyz, new_xyz, feat_t, idx = _geometry(cuda, B, N, C, NP, NS, radius, 7)
    torch.manual_seed(1)
    w = torch.randn(Cout, C + 3, device=cuda) / (C + 3) ** 0.5
    grid = fused_sa.slice_grid(False, C + 3, Cout, True, False)
    assert len(grid) > 1
    images = fused_sa.pack_layer(w, True, "tf32", False)
    M = B * NP * NS
    z = torch.full((M, Cout), float("nan"), device=cuda)
    stats = torch.zeros(2 * Cout, dtype=torch.float64, device=cuda)
    d = fused_sa._lib.SaLayer()
    d.B, d.N, d.NP, d.NS, d.Cin, d.Cout, d.mode, d.epilogue = B, N, NP, NS, C + 3, Cout, 0, 0
    d.xyz, d.new_xyz, d.feat_t, d.idx = _vp(xyz), _vp(new_xyz), _vp(feat_t), _vp(idx)
    d.radius, d.normalize_xyz, d.z = radius, 1, _vp(z)
    for (co0, co_n, ci0, ci_n), img in zip(grid, images):
        d.co0, d.co_n, d.ci0, d.ci_n, d.accumulate = co0, co_n, ci0, ci_n, int(ci0 > 0)
        d.stats = _vp(stats) if ci_n == 0 or ci0 + ci_n >= C else None
        d.w_image = _vp(img)
        _fwd(d)
    torch.cuda.synchronize()
    il = idx.long()
    bi = torch.arange(B, device=cuda)[:, None, None]
    rel = (xyz[bi, il] - new_xyz[:, :, None, :]) / radius
    x = torch.cat([rel, feat_t[bi, il]], -1).reshape(M, C + 3)
    want = round_tf32(x).double() @ round_tf32(w).double().t()
    assert torch.isfinite(z).all()
    assert rel_l2(z.cpu().numpy(), (x.double() @ w.double().t()).cpu().numpy()) < TF32_TOL
    e = rel_l2(z.cpu().numpy(), want.cpu().numpy())
    emu_log("sliced gather fwd %d -> %d, %d launches" % (C + 3, Cout, len(grid)), LOG, z=e)
    assert e < EMU_TOL_FWD, e
    zd = z.double()
    np.testing.assert_allclose(stats[:Cout].cpu().numpy(), zd.sum(0).cpu().numpy(), rtol=1e-6, atol=1e-3)
    np.testing.assert_allclose(stats[Cout:].cpu().numpy(), (zd * zd).sum(0).cpu().numpy(), rtol=1e-6,
                               atol=1e-3)


def _dense_inputs(cuda, M, Cin, Cout, seed):
    g = torch.Generator(device=cuda).manual_seed(seed)
    z_prev = torch.randn(M, Cin, device=cuda, generator=g)
    scale = torch.randn(Cin, device=cuda, generator=g) * 0.5 + 0.8
    shift = torch.randn(Cin, device=cuda, generator=g) * 0.2
    w = torch.randn(Cout, Cin, device=cuda, generator=g) / Cin ** 0.5
    return z_prev, scale, shift, w


@pytest.mark.parametrize("Cin,Cout,NS,pooled", [(256, 256, 32, False), (256, 512, 16, True),
                                                (256, 512, 32, True)])
def test_sliced_dense_layer_forward_vs_emulation(cuda, Cin, Cout, NS, pooled):
    """256 -> 256 and the pooled 256 -> 512 of the w2x SA2-4 blocks, run as their slice grid: z
    against fp64 products of TF32-rounded operands, the statistics against z, and the pooled
    epilogue against the max / min of the same grid's z."""
    from backtoreality_b200 import _lib, fused_sa
    B, NP = 2, 4096 // NS * 4
    M = B * NP * NS
    z_prev, scale, shift, w = _dense_inputs(cuda, M, Cin, Cout, Cin + Cout + NS)
    grid = fused_sa.slice_grid(False, Cin, Cout, False, pooled)
    assert len(grid) > 1
    images = fused_sa.pack_layer(w, False, "tf32", pooled)
    outs = []
    for epi in ((0, 1) if pooled else (0,)):
        d = _lib.SaLayer()
        d.B, d.N, d.NP, d.NS, d.Cin, d.Cout, d.mode, d.epilogue = B, 1, NP, NS, Cin, Cout, 1, epi
        d.z_prev, d.scale_prev, d.shift_prev = _vp(z_prev), _vp(scale), _vp(shift)
        stats = torch.zeros(2 * Cout, dtype=torch.float64, device=cuda)
        d.stats = _vp(stats)
        if epi:
            bufs = [torch.empty(B * NP, Cout, device=cuda) for _ in range(2)] + \
                   [torch.empty(B * NP, Cout, dtype=torch.int32, device=cuda) for _ in range(2)]
            d.zmax, d.zmin, d.amax, d.amin = [_vp(t) for t in bufs]
        else:
            bufs = [torch.full((M, Cout), float("nan"), device=cuda)]
            d.z = _vp(bufs[0])
        for (co0, co_n, ci0, ci_n), img in zip(grid, images):
            d.co0, d.co_n, d.ci0, d.ci_n, d.w_image = co0, co_n, ci0, ci_n, _vp(img)
            _fwd(d)
        torch.cuda.synchronize()
        outs.append((bufs, stats))
    z, stats = outs[0][0][0], outs[0][1]
    x = torch.relu(z_prev.double() * scale.double() + shift.double())
    assert rel_l2(z.cpu().numpy(), (x @ w.double().t()).cpu().numpy()) < TF32_TOL
    want = round_tf32(x.float()).double() @ round_tf32(w).double().t()
    e = rel_l2(z.cpu().numpy(), want.cpu().numpy())
    emu_log("sliced dense fwd %d -> %d, %d launches" % (Cin, Cout, len(grid)), LOG, z=e)
    assert e < EMU_TOL_FWD, e
    zd = z.double()
    np.testing.assert_allclose(stats[:Cout].cpu().numpy(), zd.sum(0).cpu().numpy(), rtol=1e-6, atol=1e-3)
    np.testing.assert_allclose(stats[Cout:].cpu().numpy(), (zd * zd).sum(0).cpu().numpy(), rtol=1e-6,
                               atol=1e-3)
    if pooled:
        (zmax, zmin, amax, amin), st1 = outs[1]
        zz = z.view(B * NP, NS, Cout)
        assert torch.equal(zmax, zz.max(1).values) and torch.equal(zmin, zz.min(1).values)
        assert torch.equal(torch.gather(zz, 1, amax.long()[:, None, :])[:, 0], zmax)
        assert torch.equal(torch.gather(zz, 1, amin.long()[:, None, :])[:, 0], zmin)
        # (fp32 partial sums per tile, fp64 atomics: the two epilogues order them differently)
        assert torch.allclose(stats, st1, rtol=1e-6, atol=1e-3)


@pytest.mark.parametrize("Cin,Cout,src", [(256, 256, "bn"), (256, 256, "direct"), (256, 512, "top")])
def test_sliced_dense_layer_backward_vs_emulation(cuda, Cin, Cout, src):
    """The dense w2x layers' backward as their slice grid (output slices after the first add into
    gr_prev): dW, the masked input gradient and its BatchNorm-backward sums against fp64 and
    against the BF16 operand-rounding emulation, for dz given, (gr, z) + coefficients, and the
    pooled top layer (z recomputed in the kernel)."""
    from backtoreality_b200 import _lib, fused_sa
    NS, M = 16, 16 * 512
    g = torch.Generator(device="cpu").manual_seed(Cin + Cout)
    zp = torch.randn(M, Cin, generator=g).to(cuda)
    sc = (torch.rand(Cin, generator=g) + 0.5).to(cuda)
    sc[::5] *= -1.0
    sh = (torch.randn(Cin, generator=g) * 0.3).to(cuda)
    w = (torch.randn(Cout, Cin, generator=g) / Cin ** 0.5).to(cuda)
    gr = torch.randn(M, Cout, generator=g).to(cuda)
    z = torch.randn(M, Cout, generator=g).to(cuda)
    ca = (torch.rand(Cout, generator=g) + 0.5).to(cuda)
    cb = (torch.randn(Cout, generator=g) * 0.2).to(cuda)
    cc = (torch.randn(Cout, generator=g) * 0.1).to(cuda)
    top = src == "top"
    grid = fused_sa.slice_grid(True, Cin, Cout, False, top)
    assert len(grid) > 1
    images = fused_sa.pack_layer(w, False, "bf16", top)
    b = _lib.SaLayerBwd()
    b.B, b.N, b.NP, b.NS, b.Cin, b.Cout, b.mode = 1, 1, M // NS, NS, Cin, Cout, 1
    b.z_prev, b.scale_prev, b.shift_prev = _vp(zp), _vp(sc), _vp(sh)
    dW = torch.zeros(Cout, Cin, device=cuda)
    gprev = torch.full((M, Cin), float("nan"), device=cuda)
    stats = torch.zeros(2, Cin, dtype=torch.float64, device=cuda)
    b.dW, b.gr_prev, b.stats_prev = _vp(dW), _vp(gprev), _vp(stats)
    x = torch.relu(zp.double() * sc.double() + sh.double())
    w2 = w.double()
    xe, we = round_bf16(x).double(), round_bf16(w2).double()
    keep = []
    if src == "direct":
        dzt = (ca * gr + cb * z + cc).contiguous()
        keep.append(dzt)
        b.dz = _vp(dzt)
        dz = dz_e = dzt.double()
    elif src == "bn":
        b.gr, b.z = _vp(gr), _vp(z)
        b.coef_a, b.coef_b, b.coef_c = _vp(ca), _vp(cb), _vp(cc)
        dz = dz_e = ca.double() * gr.double() + cb.double() * z.double() + cc.double()
    else:
        dysel = torch.randn(M // NS, Cout, generator=g).to(cuda)
        asel = torch.randint(0, NS, (M // NS, Cout), generator=g, dtype=torch.int32).to(cuda)
        keep += [dysel, asel]
        b.dysel, b.asel = _vp(dysel), _vp(asel)
        b.coef_a, b.coef_b, b.coef_c = _vp(ca), _vp(cb), _vp(cc)
        dy = torch.zeros(M // NS, NS, Cout, dtype=torch.float64, device=cuda)
        dy.scatter_(1, asel.long()[:, None, :], dysel.double()[:, None, :])
        dz = ca.double() * dy.reshape(M, Cout) + cb.double() * (x @ w2.t()) + cc.double()
        dz_e = ca.double() * dy.reshape(M, Cout) + cb.double() * (xe @ we.t()) + cc.double()
    dz_e = round_bf16(dz_e).double()
    for j, ((co0, co_n, ci0, ci_n), img) in enumerate(zip(grid, images)):
        b.co0, b.co_n, b.ci0, b.ci_n, b.accumulate = co0, co_n, ci0, ci_n, int(j > 0)
        b.w_image_bf16 = _vp(img)
        _bwd(b)
    torch.cuda.synchronize()
    mask = torch.addcmul(sh, zp, sc) > 0   # as the kernel evaluates it: one fp32 fma
    assert torch.isfinite(gprev).all()
    assert rel_l2(dW.cpu().numpy(), (dz.t() @ x).cpu().numpy()) < BF16_TOL
    assert rel_l2(gprev.cpu().numpy(), ((dz @ w2) * mask).cpu().numpy()) < BF16_TOL
    e_w = rel_l2(dW.cpu().numpy(), (dz_e.t() @ xe).cpu().numpy())
    e_g = rel_l2(gprev.cpu().numpy(), ((dz_e @ we) * mask).cpu().numpy())
    emu_log("sliced dense bwd %s %d -> %d, %d launches" % (src, Cin, Cout, len(grid)), LOG,
            dW=e_w, g_prev=e_g)
    assert e_w < EMU_TOL_BWD and e_g < EMU_TOL_BWD, (e_w, e_g)
    np.testing.assert_allclose(stats[0].cpu().numpy(), gprev.double().sum(0).cpu().numpy(),
                               rtol=1e-5, atol=1e-2)
    np.testing.assert_allclose(stats[1].cpu().numpy(),
                               (gprev.double() * zp.double()).sum(0).cpu().numpy(),
                               rtol=1e-5, atol=1e-2)


@pytest.mark.parametrize("C,N,NP,NS", [(256, 2048, 512, 32), (512, 1024, 256, 16)])
def test_sliced_gather_layer_backward_vs_emulation(cuda, C, N, NP, NS):
    """259 -> 256 (two output slices) and 515 -> 256 (output and feature slices) gather layers
    backward: dW and the scatter-added feature / xyz / centre gradients against autograd in fp64
    and against the BF16 operand-rounding emulation."""
    from backtoreality_b200 import _lib, fused_sa
    B, Cout, r = 2, 256, 0.37
    g = torch.Generator(device="cpu").manual_seed(C + N)
    xyz = torch.rand(B, N, 3, generator=g).to(cuda)
    new_xyz = torch.rand(B, NP, 3, generator=g).to(cuda)
    feats = torch.randn(B, C, N, generator=g).to(cuda)
    idx = torch.randint(0, N, (B, NP, NS), generator=g, dtype=torch.int32).to(cuda)
    w = (torch.randn(Cout, 3 + C, generator=g) / (3 + C) ** 0.5).to(cuda)
    M = B * NP * NS
    dz = torch.randn(M, Cout, generator=g).to(cuda)
    feat_t = fused_sa.to_point_major(feats)
    grid = fused_sa.slice_grid(True, 3 + C, Cout, True, False)
    assert len(grid) > 1
    images = fused_sa.pack_layer(w, True, "bf16", False)
    dW = torch.zeros(Cout, 3 + C, device=cuda)
    g_feat_t = torch.zeros(B, N, C, device=cuda)
    g_xyz = torch.zeros(B, N, 3, device=cuda)
    g_new = torch.zeros(B, NP, 3, device=cuda)
    b = _lib.SaLayerBwd()
    b.B, b.N, b.NP, b.NS, b.Cin, b.Cout, b.mode = B, N, NP, NS, 3 + C, Cout, 0
    b.xyz, b.new_xyz, b.feat_t, b.idx = _vp(xyz), _vp(new_xyz), _vp(feat_t), _vp(idx)
    b.radius, b.normalize_xyz, b.dz, b.dW = r, 1, _vp(dz), _vp(dW)
    b.g_feat_t, b.g_xyz, b.g_new_xyz = _vp(g_feat_t), _vp(g_xyz), _vp(g_new)
    for (co0, co_n, ci0, ci_n), img in zip(grid, images):
        b.co0, b.co_n, b.ci0, b.ci_n, b.accumulate = co0, co_n, ci0, ci_n, 0
        b.w_image_bf16 = _vp(img)
        _bwd(b)
    torch.cuda.synchronize()
    xyz64 = xyz.double().requires_grad_(True)
    new64 = new_xyz.double().requires_grad_(True)
    f64 = feats.double().requires_grad_(True)
    li = idx.long()
    bi = torch.arange(B, device=cuda)[:, None, None].expand_as(li)
    rel = (xyz64[bi, li] - new64[:, :, None, :]) / r
    x = torch.cat([rel, f64.transpose(1, 2)[bi, li]], dim=-1).reshape(M, 3 + C)
    w64 = w.double().requires_grad_(True)
    (x @ w64.t() * dz.double()).sum().backward(retain_graph=True)
    assert rel_l2(dW.cpu().numpy(), w64.grad.cpu().numpy()) < BF16_TOL
    assert rel_l2(g_feat_t.cpu().numpy(), f64.grad.transpose(1, 2).cpu().numpy()) < BF16_TOL
    assert rel_l2(g_xyz.cpu().numpy(), xyz64.grad.cpu().numpy()) < BF16_TOL
    assert rel_l2(g_new.cpu().numpy(), new64.grad.cpu().numpy()) < BF16_TOL
    dz_e = round_bf16(dz).double()
    errs = {"dW": rel_l2(dW.cpu().numpy(), (dz_e.t() @ round_bf16(x).double()).cpu().numpy())}
    for t in (xyz64, new64, f64):
        t.grad = None
    (x @ round_bf16(w).double().t() * dz_e).sum().backward()
    errs["g_feat"] = rel_l2(g_feat_t.cpu().numpy(), f64.grad.transpose(1, 2).cpu().numpy())
    errs["g_xyz"] = rel_l2(g_xyz.cpu().numpy(), xyz64.grad.cpu().numpy())
    errs["g_new"] = rel_l2(g_new.cpu().numpy(), new64.grad.cpu().numpy())
    emu_log("sliced gather bwd %d -> %d, %d launches" % (3 + C, Cout, len(grid)), LOG, **errs)
    for k, e in errs.items():
        assert e < EMU_TOL_BWD, (k, e)


@pytest.mark.parametrize("pooled", [False, True])
def test_output_slices_bit_identical_to_one_launch(cuda, pooled):
    """128 -> 256 is covered by one launch AND by two 128-row output slices: per-channel work is
    the same arithmetic, so z (or the pooled max / min and their samples) match bit for bit."""
    from backtoreality_b200 import _lib, fused_sa
    B, NP, NS, Cin, Cout = 2, 256, 32, 128, 256
    M = B * NP * NS
    z_prev, scale, shift, w = _dense_inputs(cuda, M, Cin, Cout, 3)
    outs = []
    for slices in ([(0, 0)], [(0, 128), (128, 128)]):
        d = _lib.SaLayer()
        d.B, d.N, d.NP, d.NS, d.Cin, d.Cout, d.mode = B, 1, NP, NS, Cin, Cout, 1
        d.epilogue = 1 if pooled else 0
        d.z_prev, d.scale_prev, d.shift_prev = _vp(z_prev), _vp(scale), _vp(shift)
        stats = torch.zeros(2 * Cout, dtype=torch.float64, device=cuda)
        d.stats = _vp(stats)
        if pooled:
            bufs = [torch.empty(B * NP, Cout, device=cuda) for _ in range(2)] + \
                   [torch.empty(B * NP, Cout, dtype=torch.int32, device=cuda) for _ in range(2)]
            d.zmax, d.zmin, d.amax, d.amin = [_vp(t) for t in bufs]
        else:
            bufs = [torch.empty(M, Cout, device=cuda)]
            d.z = _vp(bufs[0])
        keep = []
        for co0, co_n in slices:
            img = fused_sa.pack_weight(w[co0:co0 + co_n] if co_n else w, gather=False)
            keep.append(img)
            d.co0, d.co_n, d.w_image = co0, co_n, _vp(img)
            _fwd(d)
        torch.cuda.synchronize()
        outs.append((bufs, stats))
    (b1, s1), (b2, s2) = outs
    for x, y in zip(b1, b2):
        assert torch.equal(x, y)
    assert torch.allclose(s1, s2, rtol=1e-9, atol=1e-6)


def test_output_slices_backward_matches_one_launch(cuda):
    """Dense 128 -> 256 backward as one launch and as two output slices (the second accumulating
    into gr_prev): the input gradient and its BatchNorm sums agree within fp32 reordering, dW
    rows are the same per-slice arithmetic."""
    from backtoreality_b200 import _lib, fused_sa
    B, NP, NS, Cin, Cout = 2, 256, 32, 128, 256
    M = B * NP * NS
    z_prev, scale, shift, w = _dense_inputs(cuda, M, Cin, Cout, 5)
    g = torch.Generator(device=cuda).manual_seed(9)
    gr = torch.randn(M, Cout, device=cuda, generator=g)
    z = torch.randn(M, Cout, device=cuda, generator=g)
    coef = [torch.randn(Cout, device=cuda, generator=g) * 0.3 for _ in range(3)]
    outs = []
    for slices in ([(0, 0)], [(0, 128), (128, 128)]):
        b = _lib.SaLayerBwd()
        b.B, b.N, b.NP, b.NS, b.Cin, b.Cout, b.mode = B, 1, NP, NS, Cin, Cout, 1
        b.z_prev, b.scale_prev, b.shift_prev = _vp(z_prev), _vp(scale), _vp(shift)
        b.gr, b.z = _vp(gr), _vp(z)
        b.coef_a, b.coef_b, b.coef_c = [_vp(c) for c in coef]
        dW = torch.zeros(Cout, Cin, device=cuda)
        gr_prev = torch.full((M, Cin), float("nan"), device=cuda)
        stats_prev = torch.zeros(2 * Cin, dtype=torch.float64, device=cuda)
        b.dW, b.gr_prev, b.stats_prev = _vp(dW), _vp(gr_prev), _vp(stats_prev)
        keep = []
        for j, (co0, co_n) in enumerate(slices):
            img = fused_sa.pack_weight_bf16(w[co0:co0 + co_n] if co_n else w, gather=False)
            keep.append(img)
            b.co0, b.co_n, b.accumulate, b.w_image_bf16 = co0, co_n, int(j > 0), _vp(img)
            _bwd(b)
        torch.cuda.synchronize()
        outs.append((dW, gr_prev, stats_prev))
    (w1, g1, s1), (w2, g2, s2) = outs
    assert torch.isfinite(g2).all()
    assert rel_l2(g2.cpu().numpy(), g1.cpu().numpy()) < 1e-6
    assert rel_l2(w2.cpu().numpy(), w1.cpu().numpy()) < 1e-6
    assert rel_l2(s2.cpu().numpy(), s1.cpu().numpy()) < 1e-6


def _w2_block(cuda, C, npoint, nsample, radius, depth=2):
    from backtoreality_b200.pointnet2_modules import PointnetSAModuleVotes
    sa = PointnetSAModuleVotes(npoint=npoint, radius=radius, nsample=nsample,
                               mlp=[C] + [256] * depth + [512], use_xyz=True,
                               normalize_xyz=True).to(cuda)
    for blk in sa.mlp_module:
        bn = blk.bn.bn
        bn.weight.data = torch.randn_like(bn.weight) * 0.5 + 0.8
        bn.bias.data = torch.randn_like(bn.bias) * 0.2
    return sa


@pytest.mark.parametrize("cfg", [dict(N=4096, C=256, npoint=1024, radius=0.4, nsample=32),
                                 dict(N=1024, C=512, npoint=512, radius=0.8, nsample=16)])
@pytest.mark.parametrize("compact", [False, True])
def test_w2_block_fused_vs_unfused(cuda, cfg, compact, monkeypatch):
    """SA2 / SA3 of the w2x backbone (259 / 515 -> 256 -> 256 -> 512): fused sliced block against
    the unfused fp32 module, forward and backward, at test_mlp_gpu.py's block tolerances."""
    from backtoreality_b200 import fused_sa, scenes
    monkeypatch.setattr(fused_sa, "COMPACT", compact)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        torch.manual_seed(13)
        sa = _w2_block(cuda, cfg["C"], cfg["npoint"], cfg["nsample"], cfg["radius"]).train()
        ref = copy.deepcopy(sa)
        B = 2
        pc = torch.from_numpy(scenes.batch(71, B, cfg["N"], C=1, kind="room", dup=0.2)).to(cuda)
        outs = []
        for mod, fused in ((sa, True), (ref, False)):
            fused_sa.ENABLED = fused
            try:
                xyz = pc[..., :3].contiguous().clone().requires_grad_(True)
                feats = (torch.randn(B, cfg["C"], cfg["N"], device=cuda,
                                     generator=torch.Generator(device=cuda).manual_seed(5))
                         .requires_grad_(True))
                if fused:
                    assert mod.fusable(xyz)
                new_xyz, y, _ = mod(xyz, feats)
                patt = torch.sin(torch.arange(y.numel(), device=cuda, dtype=torch.float64) * 12.9898)
                ((y * patt.float().view_as(y)).sum() + (new_xyz * 0.37).sum()).backward()
                outs.append((y.detach(), xyz.grad, feats.grad, [p.grad for p in mod.parameters()]))
            finally:
                fused_sa.ENABLED = True
        (y1, gx1, gf1, gp1), (y0, gx0, gf0, gp0) = outs
        assert rel_l2(y1.cpu().numpy(), y0.cpu().numpy()) < 5e-3
        tol = 8e-2
        assert rel_l2(gx1.cpu().numpy(), gx0.cpu().numpy()) < tol
        assert rel_l2(gf1.cpu().numpy(), gf0.cpu().numpy()) < tol
        for (n, _), a, b in zip(sa.named_parameters(), gp1, gp0):
            assert rel_l2(a.cpu().numpy(), b.cpu().numpy()) < tol, n
        for a, b in zip(sa.mlp_module, ref.mlp_module):
            for k in ("running_mean", "running_var"):
                assert rel_l2(getattr(a.bn.bn, k).cpu().numpy(), getattr(b.bn.bn, k).cpu().numpy()) < 5e-3
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _pattern_like(t):
    return torch.sin(torch.arange(t.numel(), device=t.device, dtype=torch.float64) * 12.9898) \
        .float().view_as(t)


def test_w2x_backbone_fused_vs_unfused(cuda, monkeypatch):
    """The whole w2x GroupFree3D backbone (width 2, depth 2, 0 input features, fp2 288), fused vs
    fused_sa.ENABLED = False from the same weights and inputs.  As for width 1
    (test_modules_gpu.py), the fused arm must be no further from the fp32 unfused arm than the
    reference's own cuDNN TF32 arithmetic is: features, every parameter gradient and the running
    statistics.  No SA block may take the unfused path."""
    from backtoreality_b200 import fused_sa, scenes
    from backtoreality_b200.backbone_module import Pointnet2Backbone
    torch.manual_seed(3)
    state = {k: v.clone() for k, v in Pointnet2Backbone(0, 288, width=2, depth=2).state_dict().items()}
    pc = torch.from_numpy(scenes.batch(20, 2, 20000, C=0, kind="room", dup=0.2)).to(cuda)
    feats = ("sa1_features", "sa2_features", "sa3_features", "sa4_features", "fp2_features")
    calls = []
    real_block = fused_sa.sa_block

    def counting_block(*a, **k):
        calls.append(1)
        return real_block(*a, **k)
    monkeypatch.setattr(fused_sa, "sa_block", counting_block)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)

    def run(fused, tf32):
        fused_sa.ENABLED = fused
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = tf32
        net = Pointnet2Backbone(0, 288, width=2, depth=2)
        net.load_state_dict(state)
        net = net.to(cuda).train()
        ep = net(pc)
        (ep["fp2_features"] * _pattern_like(ep["fp2_features"])).sum().backward()
        torch.cuda.synchronize()
        out = {k: ep[k].detach().cpu().numpy() for k in feats}
        out.update({"grad." + n: p.grad.cpu().numpy() for n, p in net.named_parameters()})
        out.update({k: v.cpu().numpy() for k, v in net.state_dict().items() if "running" in k})
        return out

    try:
        ref = run(False, False)
        calls.clear()
        cud = run(False, True)
        assert not calls
        got = run(True, True)
        assert len(calls) == 4          # every SA block ran fused
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
        fused_sa.ENABLED = True
    for k in ref:
        e_f, e_c = rel_l2(got[k], ref[k]), rel_l2(cud[k], ref[k])
        slack = 2e-2 if k.startswith("grad.") else 1e-3
        assert e_f < 1.5 * e_c + slack, (k, e_f, e_c)


def test_w2x_captured_and_pipelined_step_match_eager(cuda):
    """The w2x backbone step (fwd + bwd + FlatAdamW) eagerly, as a captured CUDA graph and
    pipelined (next batch's geometry beside the step): the same loss for each of three batches.
    Learning rate 0 keeps the weights where they are (AdamW's decay is lr-scaled), so the replayed
    forward must reproduce the eager loss up to the order of the statistics' fp64 atomics."""
    from backtoreality_b200 import scenes
    from backtoreality_b200.backbone_module import Pointnet2Backbone
    from backtoreality_b200.flat_adam import FlatAdamW
    from backtoreality_b200.train_step import CapturedTrainStep, PipelinedTrainStep

    def make():
        torch.manual_seed(0)
        net = Pointnet2Backbone(0, 288, width=2, depth=2).to(cuda).train()
        opt = FlatAdamW(net.parameters(), lr=0.0)

        def step(pc, geometry=None):
            for p in net.parameters():
                p.grad = None
            ep = net(pc, geometry=geometry)
            loss = (ep["fp2_features"] ** 2).mean()
            loss.backward()
            opt.step()
            return loss.detach()
        return net, step

    batches = [torch.from_numpy(scenes.batch(500 + 2 * i, 2, 20000, C=0, kind="room", dup=0.2)).to(cuda)
               for i in range(3)]
    _, step_e = make()
    eager = [float(step_e(b)) for b in batches]
    _, step_c = make()
    cap = CapturedTrainStep(step_c, batches[0], warmup=2)
    assert cap.launches_per_step > 50
    captured = [float(cap(b)) for b in batches]
    net_p, step_p = make()
    pipe = PipelinedTrainStep(net_p, step_p, batches[0], warmup=2, fps_cluster=4)
    piped = [float(pipe(batches[(i + 1) % 3])) for i in range(3)]
    for got in (captured, piped):
        for g, e in zip(got, eager):
            assert abs(g - e) <= 2e-5 * abs(e), (got, eager)
    assert len(set(eager)) == 3
