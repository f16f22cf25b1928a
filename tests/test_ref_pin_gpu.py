"""Pins the oracle -- and the product -- against the REFERENCE'S OWN CUDA KERNELS.

tests/golden/ref_kernels.npz holds the reference kernels' outputs on the inputs below (FPS /
ball-query / three_nn indices, three_nn distances, three_interpolate; ball-query rows and
interpolated columns sampled to keep the file small); tests/golden/make_ref_pin.py writes it.
Every test holds the C restatement (oracle) and libb2r bit-identical to those outputs -- this is
what makes the oracle "pinned" rather than merely self-consistent.

Where the reference extension itself is built (oracle/_ref/_ext.so: `make -C oracle ref`, from
the reference's _ext_src compiled for sm_100a), it runs on the B200 as well and must reproduce the
stored outputs bit for bit.
"""
import importlib.util
import os

import numpy as np
import pytest
import torch

from _util import golden
from backtoreality_b200 import scenes
from oracle import cpu_ops

pytestmark = pytest.mark.gpu
_SO = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref",
                   "_ext.so")

FPS_CASES = [(20000, 2048, "room", 0.2), (40000, 2048, "room", 0.2), (50000, 2048, "room", 0.4),
             (2048, 1024, "room_shifted", 0.2), (300, 300, "room", 0.5), (1000, 600, "uniform", 0.0),
             (513, 200, "room", 0.9)]
BQ_CASES = [(40000, 2048, 0.2, 64), (2048, 1024, 0.4, 32), (1024, 256, 0.3, 16)]
BQ_ROW_STEP = 8          # stored ball-query rows: every 8th centre
INTERP_COL_STEP = 8      # stored three_interpolate output: every 8th point


@pytest.fixture(scope="module")
def ref_kernels():
    return golden("ref_kernels.npz")


@pytest.fixture(scope="module")
def ref(cuda):
    """The reference's own extension when it is built, else None (the stored outputs stand in)."""
    if not os.path.isfile(_SO):
        return None
    spec = importlib.util.spec_from_file_location("_ext", _SO)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _scene_xyz(i, B, N, kind="room", dup=0.2):
    return scenes.batch(i, B, N, C=0, kind=kind, dup=dup)[..., :3].copy()


def fps_case(N, npoint, kind, dup):
    return _scene_xyz(1, 2, N, kind, dup)


def fps_hole_case():
    rng = np.random.default_rng(2)
    xyz = (rng.random((2, 5000, 3), dtype=np.float32) - 0.5) * 3
    xyz[:, ::9] *= 0.005
    xyz[0, 0] = 0
    return xyz


def bq_case(N, M):
    xyz = _scene_xyz(4, 2, N)
    new = np.take_along_axis(xyz, cpu_ops.fps(xyz, M)[..., None].astype(np.int64), axis=1)
    return xyz, new


def interp_case():
    xyz = _scene_xyz(6, 2, 4096)
    unk, kn = xyz[:, :1024].copy(), xyz[:, 1024:1536].copy()
    kn[:, 7] = kn[:, 3]
    g = torch.Generator().manual_seed(6)
    f = torch.randn(2, 64, 512, generator=g).numpy()
    w = torch.rand(2, 1024, 3, generator=g).numpy()
    return unk, kn, f, w


@pytest.mark.parametrize("N,npoint,kind,dup", FPS_CASES)
def test_fps_reference_kernel_vs_oracle_vs_product(cuda, ref, ref_kernels, N, npoint, kind, dup):
    from backtoreality_b200 import _ext
    want = ref_kernels["fps_%d_%d_%s_%g" % (N, npoint, kind, dup)]
    xyz = fps_case(N, npoint, kind, dup)
    x = torch.from_numpy(xyz).to(cuda)
    assert np.array_equal(cpu_ops.fps(xyz, npoint), want), "oracle != reference kernel"
    assert np.array_equal(_ext.furthest_point_sampling(x, npoint).cpu().numpy(), want), \
        "libb2r != reference kernel"
    if ref is not None:
        assert np.array_equal(ref.furthest_point_sampling(x, npoint).cpu().numpy(), want)


def test_fps_hole_points_reference_vs_oracle(cuda, ref, ref_kernels):
    xyz = fps_hole_case()
    want = ref_kernels["fps_hole"]
    assert np.array_equal(cpu_ops.fps(xyz, 256), want)
    if ref is not None:
        assert np.array_equal(ref.furthest_point_sampling(torch.from_numpy(xyz).to(cuda), 256).cpu().numpy(),
                              want)


@pytest.mark.parametrize("N,M,r,ns", BQ_CASES)
def test_ball_query_reference_vs_oracle_vs_product(cuda, ref, ref_kernels, N, M, r, ns):
    from backtoreality_b200 import _ext
    want = ref_kernels["bq_%d_%d_%g_%d" % (N, M, r, ns)]
    xyz, new = bq_case(N, M)
    x, q = torch.from_numpy(xyz).to(cuda), torch.from_numpy(new).to(cuda)
    oi = cpu_ops.ball_query(new, xyz, float(np.float32(r)), ns)
    pi = _ext.ball_query(q, x, r, ns).cpu().numpy()
    assert np.array_equal(oi[:, ::BQ_ROW_STEP], want), "oracle != reference kernel"
    assert np.array_equal(pi, oi), "libb2r != oracle"
    if ref is not None:
        assert np.array_equal(ref.ball_query(q, x, r, ns).cpu().numpy(), oi)


def test_three_nn_and_interpolate_reference_vs_oracle_vs_product(cuda, ref, ref_kernels):
    from backtoreality_b200 import _ext
    unk, kn, f_np, w_np = interp_case()
    u, k = torch.from_numpy(unk).to(cuda), torch.from_numpy(kn).to(cuda)
    od, oi = cpu_ops.three_nn(unk, kn)
    assert np.array_equal(oi, ref_kernels["nn_idx"]) and np.array_equal(od, ref_kernels["nn_dist2"])
    pd, pi = _ext.three_nn(u, k)
    assert np.array_equal(pi.cpu().numpy(), oi) and np.array_equal(pd.cpu().numpy(), od)
    f, w = torch.from_numpy(f_np).to(cuda), torch.from_numpy(w_np).to(cuda)
    oo = cpu_ops.interp(f_np, oi, w_np)
    assert np.array_equal(oo[:, :, ::INTERP_COL_STEP], ref_kernels["interp"])
    po = _ext.three_interpolate(f, pi, w)
    assert np.array_equal(po.cpu().numpy(), oo)
    if ref is not None:
        rd, ri = ref.three_nn(u, k)
        assert np.array_equal(ri.cpu().numpy(), oi) and np.array_equal(rd.cpu().numpy(), od)
        assert torch.equal(ref.three_interpolate(f, ri, w), po)


def test_known_answer_on_reference_kernel_and_product(cuda, ref):
    """pointnet2_test.py:18-30 inputs; expected values computed by hand."""
    from backtoreality_b200 import _ext
    feats = torch.tensor([[[1.0, 2.0, 3.0, 4.0], [-1.0, 0.5, 0.25, 8.0]]], device=cuda)
    idx = torch.tensor([[[0, 1, 2], [1, 2, 3]]], dtype=torch.int32, device=cuda)
    w = torch.tensor([[[1.0, 1, 1], [2, 2, 2]]], device=cuda)
    want = torch.tensor([[[6.0, 18.0], [-0.25, 17.5]]], device=cuda)
    assert torch.equal(_ext.three_interpolate(feats, idx, w), want)
    if ref is not None:
        assert torch.equal(ref.three_interpolate(feats, idx, w), want)
