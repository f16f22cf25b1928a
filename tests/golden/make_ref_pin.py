"""Write ref_kernels.npz: the reference kernels' outputs on the inputs of tests/test_ref_pin_gpu.py.

With the reference's own extension built (oracle/_ref/_ext.so, `make -C oracle ref`) and a GPU,
the outputs are taken from the reference kernels, and the oracle must reproduce them bit for bit.
Without it they come from the oracle (oracle/b2r_oracle.c): that C restatement reproduced the
reference kernels bit for bit on these inputs when the reference extension ran on a B200
(profiles/r02/pytest_gpu.log; three_interpolate on features and weights drawn the same way, but
unseeded), and it has not changed since.

    python tests/golden/make_ref_pin.py
"""
import importlib.util
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]

import test_ref_pin_gpu as t  # noqa: E402  (the inputs and sampling steps live with the tests)
from oracle import cpu_ops  # noqa: E402


def reference_ext():
    so = os.path.join(ROOT, "oracle", "_ref", "_ext.so")
    if not (os.path.isfile(so) and torch.cuda.is_available()):
        return None
    spec = importlib.util.spec_from_file_location("_ext", so)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def main():
    ref = reference_ext()
    dev = torch.device("cuda") if ref is not None else None

    def pick(oracle_out, ref_fn):
        if ref is None:
            return oracle_out
        r = ref_fn()
        r = tuple(x.cpu().numpy() for x in r) if isinstance(r, tuple) else r.cpu().numpy()
        for a, b in zip(r if isinstance(r, tuple) else (r,),
                        oracle_out if isinstance(oracle_out, tuple) else (oracle_out,)):
            assert np.array_equal(a, b), "oracle != reference kernel"
        return r

    out = {}
    for N, npoint, kind, dup in t.FPS_CASES:
        xyz = t.fps_case(N, npoint, kind, dup)
        out["fps_%d_%d_%s_%g" % (N, npoint, kind, dup)] = pick(
            cpu_ops.fps(xyz, npoint),
            lambda: ref.furthest_point_sampling(torch.from_numpy(xyz).to(dev), npoint))
    xyz = t.fps_hole_case()
    out["fps_hole"] = pick(cpu_ops.fps(xyz, 256),
                           lambda: ref.furthest_point_sampling(torch.from_numpy(xyz).to(dev), 256))
    for N, M, r, ns in t.BQ_CASES:
        xyz, new = t.bq_case(N, M)
        idx = pick(cpu_ops.ball_query(new, xyz, float(np.float32(r)), ns),
                   lambda: ref.ball_query(torch.from_numpy(new).to(dev), torch.from_numpy(xyz).to(dev), r, ns))
        out["bq_%d_%d_%g_%d" % (N, M, r, ns)] = idx[:, ::t.BQ_ROW_STEP].copy()
    unk, kn, f, w = t.interp_case()
    d2, idx = pick(cpu_ops.three_nn(unk, kn),
                   lambda: ref.three_nn(torch.from_numpy(unk).to(dev), torch.from_numpy(kn).to(dev)))
    out["nn_dist2"], out["nn_idx"] = d2, idx
    y = pick(cpu_ops.interp(f, idx, w),
             lambda: ref.three_interpolate(torch.from_numpy(f).to(dev), torch.from_numpy(idx).to(dev),
                                           torch.from_numpy(w).to(dev)))
    out["interp"] = y[:, :, ::t.INTERP_COL_STEP].copy()
    path = os.path.join(HERE, "ref_kernels.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes;", "reference kernels" if ref is not None else "oracle")


if __name__ == "__main__":
    main()
