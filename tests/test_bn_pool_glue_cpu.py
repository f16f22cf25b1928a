"""Argument validation of the BatchNorm, max-pool and head glue entry points (include/b2r.h): every
call below is malformed and must return B2R_ERR_INVALID_ARG before anything reaches the device,
so this runs without a GPU.  The kernels themselves are tested in test_bn_pool_glue_gpu.py."""
import ctypes

INVALID = -1                    # B2R_ERR_INVALID_ARG
P = ctypes.c_void_p(16)         # never dereferenced: validation fails first


def _lib():
    from backtoreality_b200 import _lib
    return _lib.lib()


def _rejects(fn, *args):
    l = _lib()
    assert getattr(l, fn)(*args, None) == INVALID, (fn, args)
    assert fn.encode() in l.b2r_last_error(), l.b2r_last_error()


def _bn_finalize_args(**kw):
    a = dict(stats=P, C=8, count=64.0, gamma=P, beta=P, eps=1e-5, momentum=0.1, running_mean=P,
             running_var=P, scale=P, shift=P, mean_out=P, invstd_out=P, nbt=P)
    a.update(kw)
    return list(a.values())


def test_bn_finalize_rejects_bad_arguments():
    for kw in (dict(stats=None), dict(scale=None), dict(shift=None), dict(C=0), dict(C=-3),
               dict(count=0.0), dict(count=-1.0),
               # the running statistics are updated together or not at all
               dict(running_mean=None), dict(running_var=None)):
        _rejects("b2r_bn_finalize", *_bn_finalize_args(**kw))


def test_bn_bwd_finalize_rejects_bad_arguments():
    for fn, extra in (("b2r_bn_bwd_finalize", []), ("b2r_bn_bwd_finalize_ex", [P])):
        def args(stats=P, C=8, count=64.0, mean=P, invstd=P):
            return [stats, C, count, P, mean, invstd, 1] + [P] * 8 + extra
        for kw in (dict(stats=None), dict(mean=None), dict(invstd=None), dict(C=0), dict(C=-1),
                   dict(count=0.0), dict(count=-2.0)):
            assert getattr(_lib(), fn)(*args(**kw), None) == INVALID, (fn, kw)


def test_pool_finalize_rejects_bad_arguments():
    def args(zmax=P, zmin=P, scale=P, shift=P, B=2, NP=33, C=31):
        return [zmax, zmin, scale, shift, B, NP, C, P, P]
    for kw in (dict(zmax=None), dict(zmin=None), dict(scale=None), dict(shift=None), dict(B=0),
               dict(NP=0), dict(C=0), dict(B=-1), dict(B=65536)):
        _rejects("b2r_pool_finalize", *args(**kw))


def test_pool_bwd_prep_rejects_bad_arguments():
    def args(dcm=P, dpm=P, zmax=P, zmin=P, amax=P, amin=P, scale=P, shift=P, B=2, NP=33, C=31,
             dysel=P, asel=P, stats=P):
        return [dcm, dpm, zmax, zmin, amax, amin, scale, shift, B, NP, C, dysel, asel, stats]
    for kw in (dict(dcm=None, dpm=None), dict(zmax=None), dict(zmin=None), dict(amax=None),
               dict(amin=None), dict(scale=None), dict(shift=None), dict(dysel=None),
               dict(asel=None), dict(stats=None), dict(B=0), dict(NP=0), dict(C=0),
               dict(C=1025), dict(B=65536)):
        _rejects("b2r_pool_bwd_prep", *args(**kw))


def test_to_point_major_rejects_bad_arguments():
    for args in ((P, -1, 4, 4, P), (P, 2, -1, 4, P), (P, 2, 4, -1, P), (None, 2, 4, 4, P),
                 (P, 2, 4, 4, None)):
        _rejects("b2r_to_point_major", *args)


def test_interp_cat_rejects_bad_arguments():
    def fwd(known=P, skip=P, idx=P, weight=P, B=2, n=5, m=3, C2=8, C1=4, out=P):
        return [known, skip, idx, weight, B, n, m, C2, C1, out]
    for kw in (dict(C2=6), dict(C1=2), dict(C2=0), dict(m=0), dict(B=-1), dict(n=-1),
               dict(known=None), dict(idx=None), dict(weight=None), dict(out=None),
               dict(skip=None)):
        _rejects("b2r_interp_cat_fwd", *fwd(**kw))

    def bwd(g=P, ld_g=12, idx=P, weight=P, B=2, n=5, m=3, C2=8, C1=4):
        return [g, ld_g, idx, weight, B, n, m, C2, C1, P, P]
    for kw in (dict(C2=6), dict(C1=2), dict(ld_g=14), dict(ld_g=8), dict(C2=0), dict(m=0),
               dict(g=None), dict(idx=None), dict(weight=None)):
        _rejects("b2r_interp_cat_bwd", *bwd(**kw))


def test_vote_tail_rejects_bad_arguments():
    def fwd(net=P, ld_net=40, seed_xyz=P, seed_feat=P, M=7, C=33, vote_xyz=P, out=P, norm=P):
        return [net, ld_net, seed_xyz, seed_feat, M, C, vote_xyz, out, norm]
    for kw in (dict(ld_net=35), dict(C=0), dict(M=-1), dict(net=None), dict(seed_xyz=None),
               dict(seed_feat=None), dict(vote_xyz=None), dict(out=None), dict(norm=None)):
        _rejects("b2r_vote_tail_fwd", *fwd(**kw))

    def bwd(out=P, norm=P, M=7, C=33, ld_net=40, g_net=P):
        return [P, P, out, norm, M, C, ld_net, g_net, P]
    for kw in (dict(ld_net=35), dict(C=0), dict(M=-1), dict(out=None), dict(norm=None),
               dict(g_net=None)):
        _rejects("b2r_vote_tail_bwd", *bwd(**kw))
