"""The BatchNorm, max-pool and head glue kernels, each driven directly through the C ABI against a
float64 reference of the same operation:

  b2r_bn_finalize          (csrc/mlp.cu)      batch statistics -> scale / shift, running statistics
  b2r_bn_bwd_finalize_ex   (csrc/mlp_bwd.cu)  BatchNorm-backward sums -> dz = a*g + b*z + c, dgamma,
                                              dbeta, the conv-bias gradient
  b2r_pool_finalize        (csrc/mlp.cu)      relu(scale * (scale >= 0 ? zmax : zmin) + shift)
  b2r_pool_bwd_prep        (csrc/mlp_bwd.cu)  max-pool routing, ReLU mask, BatchNorm-backward sums
  b2r_to_point_major       (csrc/mlp.cu)      (B,C,N) -> (B,N,C)
  b2r_interp_cat_fwd/bwd, b2r_vote_tail_fwd/bwd (csrc/heads.cu)

No GEMM runs here, so there is no TF32 / BF16 noise to absorb: every output is a few fp32 roundings
of exactly known operands and is held to a few ulp of those operands' magnitude.  Where the
kernel takes a decision in fp32 (the ReLU mask, which of zmax / zmin), the reference takes the same
decision the same way (torch.addcmul in fp32 is one fma, like the kernels' fmaf).

Every check records its measured error in glue_errors.log of the run's output directory when that
directory exists (tests/_util.py emu_log); profiles/r04/glue_errors.log has a B200 run.
"""
import ctypes
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from _util import emu_log, pattern_like, rel_l2

pytestmark = pytest.mark.gpu

EPS = float(np.float32(1e-5))     # the kernels take eps as a float
RTOL = 1e-6                       # a few fp32 roundings of fp64 operands (2^-24 = 6e-8 each)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _lib():
    from backtoreality_b200 import _lib
    return _lib.lib()


def _call(name, *args):
    from backtoreality_b200 import _ext, _lib
    _lib.check(getattr(_lib.lib(), name)(*args, _ext._stream()), name)


def _log(name, **errs):
    emu_log(name, log="glue_errors.log", **errs)


def _gen(*key):
    return torch.Generator().manual_seed(zlib.crc32(repr(key).encode()))


def _nan(*shape, dev):
    return torch.full(shape, float("nan"), dtype=torch.float32, device=dev)


def _scaled_err(got, want, mag):
    """max over elements of |got - want| / mag: mag is the magnitude of the operands that produce
    want, so a result that suffers cancellation is judged against what it was computed from."""
    got = torch.as_tensor(got).detach().double().cpu()
    want = torch.as_tensor(want).detach().double().cpu()
    mag = torch.as_tensor(mag).detach().double().cpu()
    assert not torch.isnan(got).any(), "an output element was not written (NaN pre-fill survived)"
    d = (got - want).abs()
    return float(torch.where(d == 0, torch.zeros_like(d), d / mag.clamp_min(1e-300)).max())


def _ulp_err(got, want):
    """max |got - want| in units of the fp32 spacing at want."""
    got = np.asarray(torch.as_tensor(got).cpu(), np.float64)
    want = np.asarray(torch.as_tensor(want).cpu(), np.float64)
    assert not np.isnan(got).any(), "an output element was not written (NaN pre-fill survived)"
    ulp = np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)
    return float((np.abs(got - want) / ulp).max())


# ---- 1. b2r_bn_finalize ---------------------------------------------------------------------------

def _bn_inputs(count, C, g):
    """z (count, C) fp32: channels of mean in [-2, 2] and std in [0.5, 2], channel 0 constant
    (variance 0) and, when C > 1, channel C // 2 at |mean| / std ~ 1e4."""
    mean = torch.rand(C, generator=g, dtype=torch.float64) * 4 - 2
    std = torch.rand(C, generator=g, dtype=torch.float64) * 1.5 + 0.5
    z = (mean + std * torch.randn(count, C, generator=g, dtype=torch.float64)).float()
    z[:, 0] = 0.75
    if C > 1:
        z[:, C // 2] = (1e4 + torch.randn(count, generator=g, dtype=torch.float64)).float()
    return z


def _sums(z):
    zd = z.double()
    return torch.cat([zd.sum(0), (zd * zd).sum(0)])


def _run_bn_finalize(cuda, z, gamma, beta, momentum, rm0, rv0, nbt0=41):
    C = z.shape[1]
    stats = _sums(z).to(cuda)
    stats_before = stats.clone()
    out = {k: _nan(C, dev=cuda) for k in ("scale", "shift", "mean", "invstd")}
    rm = rm0.clone().to(cuda) if rm0 is not None else None
    rv = rv0.clone().to(cuda) if rv0 is not None else None
    nbt = torch.tensor([nbt0], dtype=torch.int64, device=cuda)
    gam = gamma.to(cuda) if gamma is not None else None    # kept alive until the launch
    bet = beta.to(cuda) if beta is not None else None
    _call("b2r_bn_finalize", _p(stats), C, float(z.shape[0]), _p(gam), _p(bet), EPS, momentum,
          _p(rm), _p(rv),
          _p(out["scale"]), _p(out["shift"]), _p(out["mean"]), _p(out["invstd"]), _p(nbt))
    assert torch.equal(stats, stats_before)
    out = {k: v.cpu() for k, v in out.items()}
    return out, (rm.cpu() if rm is not None else None), (rv.cpu() if rv is not None else None), int(nbt)


def _check_bn_finalize(tag, z, gamma, beta, momentum, out, rm0, rv0, rm, rv):
    count = z.shape[0]
    zd = z.double()
    mean = zd.mean(0)
    var = ((zd - mean) ** 2).mean(0)                 # two-pass: no cancellation
    invstd = 1.0 / torch.sqrt(var + EPS)
    gd = gamma.double() if gamma is not None else torch.ones_like(mean)
    bd = beta.double() if beta is not None else torch.zeros_like(mean)
    scale = gd * invstd
    shift = bd - mean * scale
    errs = dict(mean=_scaled_err(out["mean"], mean, mean.abs()),
                invstd=_scaled_err(out["invstd"], invstd, invstd),
                scale=_scaled_err(out["scale"], scale, scale.abs()),
                shift=_scaled_err(out["shift"], shift, bd.abs() + (mean * scale).abs()))
    if rm0 is not None:
        # nn.BatchNorm's own update, in float64, at the float momentum the kernel receives
        m = float(np.float32(momentum))
        rm_ref, rv_ref = rm0.double().clone(), rv0.double().clone()
        F.batch_norm(zd, rm_ref, rv_ref, None, None, True, m, EPS)
        unbiased = var * count / (count - 1)
        errs["running_mean"] = _scaled_err(rm, rm_ref, (1 - m) * rm0.double().abs() + m * mean.abs())
        errs["running_var"] = _scaled_err(rv, rv_ref, (1 - m) * rv0.double().abs() + m * unbiased)
    _log("bn_finalize %s" % tag, **errs)
    for k, e in errs.items():
        assert e <= RTOL, (k, e)


@pytest.mark.parametrize("C", [1, 127, 129, 300])
@pytest.mark.parametrize("count", [2, 3, 64, 4096])
def test_bn_finalize_matches_batchnorm_training(cuda, count, C):
    g = _gen("bn_finalize", count, C)
    z = _bn_inputs(count, C, g)
    gamma = (torch.rand(C, generator=g) + 0.5) * torch.where(torch.arange(C) % 3 == 2, -1.0, 1.0)
    beta = torch.randn(C, generator=g)
    rm0 = torch.randn(C, generator=g)
    rv0 = torch.rand(C, generator=g) * 2 + 0.25
    for momentum in (0.1, 0.3):
        out, rm, rv, nbt = _run_bn_finalize(cuda, z, gamma, beta, momentum, rm0, rv0)
        assert nbt == 42, nbt            # incremented once, whatever the number of blocks
        _check_bn_finalize("count=%d C=%d momentum=%.1f" % (count, C, momentum), z, gamma, beta,
                           momentum, out, rm0, rv0, rm, rv)
        # the constant channel: variance 0 -> invstd = 1 / sqrt(eps) in fp32
        assert out["invstd"][0] == np.float32(1.0) / np.sqrt(np.float32(EPS)), out["invstd"][0]


@pytest.mark.parametrize("count,C", [(3, 300), (64, 129)])
def test_bn_finalize_optional_arguments(cuda, count, C):
    g = _gen("bn_finalize_opt", count, C)
    z = _bn_inputs(count, C, g)
    # no affine parameters: gamma = 1, beta = 0
    rm0, rv0 = torch.randn(C, generator=g), torch.rand(C, generator=g) + 0.5
    out, rm, rv, nbt = _run_bn_finalize(cuda, z, None, None, 0.1, rm0, rv0)
    _check_bn_finalize("no-affine count=%d C=%d" % (count, C), z, None, None, 0.1, out, rm0, rv0, rm, rv)
    assert nbt == 42
    # no running buffers: the batch outputs are unchanged and the counter still advances
    gamma, beta = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g)
    out, _, _, nbt = _run_bn_finalize(cuda, z, gamma, beta, 0.1, None, None, nbt0=7)
    _check_bn_finalize("no-running count=%d C=%d" % (count, C), z, gamma, beta, 0.1, out, None, None,
                       None, None)
    assert nbt == 8
    # no num_batches_tracked / mean / invstd outputs: scale and shift alone
    stats = _sums(z).to(cuda)
    scale, shift = _nan(C, dev=cuda), _nan(C, dev=cuda)
    gam, bet = gamma.to(cuda), beta.to(cuda)
    _call("b2r_bn_finalize", _p(stats), C, float(count), _p(gam), _p(bet), EPS, 0.1, None, None,
          _p(scale), _p(shift), None, None, None)
    assert torch.equal(scale.cpu(), out["scale"]) and torch.equal(shift.cpu(), out["shift"])


# ---- 2. b2r_bn_bwd_finalize_ex ------------------------------------------------------------------

def _bwd_inputs(M, C, g, ratio=None):
    """z (M, C) fp32 with per-channel mean / std; gr = dL/d(BatchNorm output) with a non-zero mean
    and a component along x-hat, so both the S1 and the S2 terms of the backward matter."""
    std = torch.rand(C, generator=g, dtype=torch.float64) + 0.5
    if ratio is None:
        mean = torch.rand(C, generator=g, dtype=torch.float64) * 4 - 2
    else:
        mean = ratio * std * torch.where(torch.arange(C) % 2 == 0, 1.0, -1.0).double()
    xh = torch.randn(M, C, generator=g, dtype=torch.float64)
    z = (mean + std * xh).float()
    gr = (torch.randn(M, C, generator=g, dtype=torch.float64) + 0.3 + 0.5 * xh).float()
    return z, gr, mean, std


def _run_bn_bwd(cuda, z, gr, gamma, mean32, invstd32, training):
    C = z.shape[1]
    zd, gd = z.double(), gr.double()
    stats = torch.cat([gd.sum(0), (gd * zd).sum(0)]).to(cuda)
    names = ("a", "b", "c", "k1", "k2", "gs", "dgamma", "dbeta", "dbias")
    o = {k: _nan(C, dev=cuda) for k in names}
    gam = gamma.to(cuda) if gamma is not None else None    # kept alive until the launch
    mu, inv = mean32.to(cuda), invstd32.to(cuda)
    _call("b2r_bn_bwd_finalize_ex", _p(stats), C, float(z.shape[0]), _p(gam), _p(mu), _p(inv),
          int(training), *[_p(o[k]) for k in names])
    return {k: v.cpu().double() for k, v in o.items()}


def _bn_autograd(z, gr, gamma, bias, training, rm=None, rv=None):
    """fp64 autograd of batch_norm(z0 + bias): dz, dgamma, dbeta, dbias."""
    bd = bias.double().requires_grad_(True)
    zz = z.double() - bias.double() + bd            # z = z0 + bias, with bias a leaf
    zz.retain_grad()
    w = (gamma.double() if gamma is not None else torch.ones(z.shape[1], dtype=torch.float64))
    w.requires_grad_(True)
    bt = torch.zeros(z.shape[1], dtype=torch.float64, requires_grad=True)
    y = F.batch_norm(zz, rm.double() if rm is not None else None,
                     rv.double() if rv is not None else None, w, bt, training, 0.0, EPS)
    y.backward(gr.double())
    return zz.grad, w.grad, bt.grad, bd.grad


@pytest.mark.parametrize("training", [1, 0])
@pytest.mark.parametrize("gamma_kind", ["mixed_sign", "null"])
@pytest.mark.parametrize("M,C", [(2, 3), (333, 129), (4096, 300)])
def test_bn_bwd_finalize_matches_fp64_autograd(cuda, M, C, gamma_kind, training):
    g = _gen("bn_bwd", M, C, gamma_kind, training)
    z, gr, mu, sd = _bwd_inputs(M, C, g)
    gamma = None
    if gamma_kind == "mixed_sign":
        gamma = (torch.rand(C, generator=g) + 0.5) * torch.where(torch.arange(C) % 3 == 1, -1.0, 1.0)
    bias = torch.randn(C, generator=g) * 0.5
    if training:
        zd = z.double()
        mean64, var64 = zd.mean(0), zd.var(0, unbiased=False)
        mean32, invstd32 = mean64.float(), (1.0 / torch.sqrt(var64 + EPS)).float()
        rm = rv = None
    else:
        rm = (mu + 0.2 * torch.randn(C, generator=g, dtype=torch.float64)).float()
        rv = (sd ** 2 * (0.5 + torch.rand(C, generator=g, dtype=torch.float64))).float()
        mean32, invstd32 = rm, (1.0 / torch.sqrt(rv.double() + EPS)).float()
    o = _run_bn_bwd(cuda, z, gr, gamma, mean32, invstd32, training)
    dz_ref, dgamma_ref, dbeta_ref, dbias_ref = _bn_autograd(z, gr, gamma, bias, bool(training), rm, rv)

    zd, gd = z.double(), gr.double()
    mu_k, is_k = mean32.double(), invstd32.double()
    dz = o["a"] * gd + o["b"] * zd + o["c"]           # the kernels' form, evaluated in fp64
    gs_abs = (o["gs"].abs() * gd.abs()).sum(0)
    # c = -gs*k1 - b*mean: its two terms are operands of dz as much as a*g and b*z are
    dz_mag = (o["a"] * gd).abs() + (o["b"] * zd).abs() + (o["gs"] * o["k1"]).abs() + (o["b"] * mu_k).abs()
    errs = dict(
        dz=_scaled_err(dz, dz_ref, dz_mag),
        dgamma=_scaled_err(o["dgamma"], dgamma_ref, (gd * (zd - mu_k) * is_k).abs().sum(0)),
        dbeta=_scaled_err(o["dbeta"], dbeta_ref, gd.abs().sum(0)),
        dbias=_scaled_err(o["dbias"], dbias_ref, gs_abs))
    # the (k1, k2, gs) form and the coefficients describe the same dz
    g64 = gamma.double() if gamma is not None else torch.ones(C, dtype=torch.float64)
    assert torch.equal(o["gs"], o["a"])
    errs["gs"] = _scaled_err(o["gs"], g64 * is_k, (g64 * is_k).abs())
    if training:
        errs["k1"] = _scaled_err(o["k1"], gd.sum(0) / M, gd.abs().sum(0) / M)
        errs["k2"] = _scaled_err(o["k2"], dgamma_ref / M, (gd * (zd - mu_k) * is_k).abs().sum(0) / M)
        errs["b"] = _scaled_err(o["b"], -o["gs"] * o["k2"] * is_k, (o["gs"] * o["k2"] * is_k).abs())
        errs["c"] = _scaled_err(o["c"], -o["gs"] * o["k1"] - o["b"] * mu_k,
                                (o["gs"] * o["k1"]).abs() + (o["b"] * mu_k).abs())
        # with batch statistics the bias in front of BatchNorm has no gradient
        assert dbias_ref.abs().max() <= 1e-12 * gs_abs.max()
    else:
        # running statistics: dz = gamma * invstd * g, the bias gradient is gs * S1
        assert (o["k1"] == 0).all() and (o["k2"] == 0).all()
        assert (o["b"] == 0).all() and (o["c"] == 0).all()
        errs["dbias_gsS1"] = _scaled_err(o["dbias"], o["gs"] * gd.sum(0), gs_abs)
    _log("bn_bwd_finalize M=%d C=%d gamma=%s training=%d" % (M, C, gamma_kind, training), **errs)
    for k, e in errs.items():
        assert e <= RTOL, (k, e)


@pytest.mark.parametrize("ratio", [1, 30, 1000])
def test_bn_bwd_dz_in_fp32_conditioning(cuda, ratio):
    """The SA and dense backward kernels evaluate dz = fmaf(a, g, fmaf(b, z, c)) in fp32, and b*z
    and c cancel when |mean| >> std.  Measures that form against fp64 autograd at |mean| / std =
    ratio (per channel) and holds it below BF16 operand noise (4e-3), the rounding the layer's
    GEMMs apply to dz next."""
    M, C = 4096, 64
    g = _gen("bn_bwd_cond", ratio)
    z, gr, _, _ = _bwd_inputs(M, C, g, ratio=ratio)
    gamma = torch.rand(C, generator=g) + 0.5
    zd = z.double()
    mean32, invstd32 = zd.mean(0).float(), (1.0 / torch.sqrt(zd.var(0, unbiased=False) + EPS)).float()
    o = _run_bn_bwd(cuda, z, gr, gamma, mean32, invstd32, 1)
    dz_ref = _bn_autograd(z, gr, gamma, torch.zeros(C), True)[0]
    a, b, c = (o[k].float().to(cuda) for k in ("a", "b", "c"))
    dz32 = torch.addcmul(torch.addcmul(c, b, z.to(cuda)), a, gr.to(cuda)).double().cpu()
    dz64 = o["a"] * gr.double() + o["b"] * zd + o["c"]
    per_ch32 = [rel_l2(dz32[:, k].numpy(), dz_ref[:, k].numpy()) for k in range(C)]
    per_ch64 = [rel_l2(dz64[:, k].numpy(), dz_ref[:, k].numpy()) for k in range(C)]
    _log("bn_bwd_dz_conditioning |mean|/std=%d" % ratio,
         fp32_form_rel_l2=rel_l2(dz32.numpy(), dz_ref.numpy()), fp32_form_worst_channel=max(per_ch32),
         fp64_form_worst_channel=max(per_ch64))
    assert max(per_ch64) < 1e-6 * max(1, ratio), max(per_ch64)
    assert max(per_ch32) < 4e-3, max(per_ch32)


# ---- 3. / 4. b2r_pool_finalize, b2r_pool_bwd_prep -----------------------------------------------

def _distinct_samples(B, NP, NS, C, g):
    """z (B*NP, NS, C): the NS samples of a (centre, channel) differ by >= 0.18, both signs."""
    perm = torch.rand(B * NP, NS, C, generator=g).argsort(dim=1).float()
    return (perm - NS / 2 + 0.5 * torch.rand(B * NP, NS, C, generator=g)) * 0.37


def _scale_shift(C, g):
    """scale of mixed sign with an exact +0.0 and -0.0 channel (-0.0 >= 0: it selects zmax)."""
    scale = torch.rand(C, generator=g) + 0.25
    scale[0::2] *= -1
    if C >= 2:
        scale[1] = 0.0
    if C >= 4:
        scale[C - 1] = -0.0
    shift = torch.randn(C, generator=g) * 0.5 + 0.05
    return scale, shift


def _pool_inputs(cuda, B, NP, C, NS, g):
    z = _distinct_samples(B, NP, NS, C, g)
    zmax, amax = z.max(dim=1)
    zmin, amin = z.min(dim=1)
    scale, shift = _scale_shift(C, g)
    d = dict(z=z, zmax=zmax, zmin=zmin, amax=amax.int(), amin=amin.int(), scale=scale, shift=shift)
    return {k: v.to(cuda) for k, v in d.items()}


POOL_SHAPES = [(B, NP, C) for B in (1, 3) for NP in (1, 33, 257) for C in (1, 31, 33, 288)]


@pytest.mark.parametrize("B,NP,C", POOL_SHAPES)
def test_pool_finalize_exact(cuda, B, NP, C):
    g = _gen("pool_finalize", B, NP, C)
    t = _pool_inputs(cuda, B, NP, C, 5, g)
    pos = t["scale"] >= 0
    zsel = torch.where(pos, t["zmax"], t["zmin"])
    want = torch.addcmul(t["shift"], zsel, t["scale"]).clamp_min(0)          # the kernel's one fma
    ref = (t["z"].double() * t["scale"].double() + t["shift"].double()).clamp_min(0).amax(dim=1)
    worst = 0.0
    for mode in ("cm", "pm", "both"):
        out_cm = _nan(B, C, NP, dev=cuda) if mode in ("cm", "both") else None
        out_pm = _nan(B * NP, C, dev=cuda) if mode in ("pm", "both") else None
        _call("b2r_pool_finalize", _p(t["zmax"]), _p(t["zmin"]), _p(t["scale"]), _p(t["shift"]),
              B, NP, C, _p(out_cm), _p(out_pm))
        for got in ([out_pm] if out_pm is not None else []) + \
                   ([out_cm.transpose(1, 2).reshape(B * NP, C)] if out_cm is not None else []):
            assert not torch.isnan(got).any(), mode
            assert torch.equal(got, want), (mode, (got - want).abs().max())
            worst = max(worst, _ulp_err(got, ref))
    _log("pool_finalize B=%d NP=%d C=%d" % (B, NP, C), ulp_vs_fp64=worst)
    assert worst <= 1.0, worst


def _prep_reference(t, dout_cm, dout_pm, B, NP, C):
    pos = t["scale"] >= 0
    zsel = torch.where(pos, t["zmax"], t["zmin"])
    asel = torch.where(pos, t["amax"], t["amin"])
    g = torch.zeros(B * NP, C, device=zsel.device)
    if dout_cm is not None:
        g = dout_cm.transpose(1, 2).reshape(B * NP, C).clone()
    if dout_pm is not None:
        g = g + dout_pm if dout_cm is not None else dout_pm.clone()
    mask = torch.addcmul(t["shift"], zsel, t["scale"]) > 0                    # the kernel's one fma
    dysel = torch.where(mask, g, torch.zeros_like(g))
    s1 = dysel.double().sum(0)
    s2 = (dysel.double() * zsel.double()).sum(0)
    m1 = dysel.double().abs().sum(0)
    m2 = (dysel.double() * zsel.double()).abs().sum(0)
    return dysel, asel, torch.cat([s1, s2]), torch.cat([m1, m2])


def _run_prep(cuda, t, dout_cm, dout_pm, B, NP, C, stats0):
    dysel = _nan(B * NP, C, dev=cuda)
    asel = torch.full((B * NP, C), -7, dtype=torch.int32, device=cuda)
    stats = stats0.clone()
    _call("b2r_pool_bwd_prep", _p(dout_cm), _p(dout_pm), _p(t["zmax"]), _p(t["zmin"]),
          _p(t["amax"]), _p(t["amin"]), _p(t["scale"]), _p(t["shift"]), B, NP, C, _p(dysel),
          _p(asel), _p(stats))
    return dysel, asel, stats


@pytest.mark.parametrize("B,NP,C", POOL_SHAPES + [(1, 33, 1024), (3, 257, 1024)])
def test_pool_bwd_prep_exact(cuda, B, NP, C):
    g = _gen("pool_bwd_prep", B, NP, C)
    t = _pool_inputs(cuda, B, NP, C, 6, g)
    dcm = torch.randn(B, C, NP, generator=g).to(cuda)
    dpm = torch.randn(B * NP, C, generator=g).to(cuda)
    stats0 = (torch.randn(2 * C, generator=g, dtype=torch.float64) * 10).to(cuda)   # accumulated
    worst = 0.0
    for cm, pm in ((dcm, None), (None, dpm), (dcm, dpm)):
        dysel, asel, stats = _run_prep(cuda, t, cm, pm, B, NP, C, stats0)
        want_dy, want_as, want_s, mag = _prep_reference(t, cm, pm, B, NP, C)
        assert torch.equal(dysel, want_dy), (cm is not None, pm is not None)
        assert torch.equal(asel, want_as), (cm is not None, pm is not None)
        e = _scaled_err(stats, stats0 + want_s, stats0.abs() + mag)
        worst = max(worst, e)
    _log("pool_bwd_prep B=%d NP=%d C=%d" % (B, NP, C), stats=worst)
    assert worst <= 1e-12, worst


@pytest.mark.parametrize("C", [33, 64])
def test_pool_bwd_prep_dense_output_layer_form(cuda, C):
    """dense_mlp's output layer calls the helper with zmax = zmin = z (B*n, C), NP = n, and one
    int32 scratch buffer as amax, amin and asel: the ReLU mask and the two sums of a plain layer."""
    B, n = 2, 77
    g = _gen("pool_bwd_prep_dense", C)
    z = torch.randn(B * n, C, generator=g).to(cuda)
    scale, shift = (v.to(cuda) for v in _scale_shift(C, g))
    scratch0 = torch.randint(0, 1 << 20, (B * n, C), generator=g, dtype=torch.int32).to(cuda)
    t = dict(zmax=z, zmin=z, amax=scratch0, amin=scratch0, scale=scale, shift=shift)
    stats0 = torch.randn(2 * C, generator=g, dtype=torch.float64).to(cuda)
    dcm = torch.randn(B, C, n, generator=g).to(cuda)
    dpm = torch.randn(B * n, C, generator=g).to(cuda)
    for cm, pm in ((dcm, None), (None, dpm)):
        scratch = scratch0.clone()
        gr = _nan(B * n, C, dev=cuda)
        stats = stats0.clone()
        _call("b2r_pool_bwd_prep", _p(cm), _p(pm), _p(z), _p(z), _p(scratch), _p(scratch),
              _p(scale), _p(shift), B, n, C, _p(gr), _p(scratch), _p(stats))
        want_g, _, want_s, mag = _prep_reference(t, cm, pm, B, n, C)
        assert torch.equal(gr, want_g)
        assert torch.equal(scratch, scratch0)
        assert _scaled_err(stats, stats0 + want_s, stats0.abs() + mag) <= 1e-12


# ---- 5. the pooled top layer's bookkeeping, composed --------------------------------------------

@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("NS", [16, 32, 64])
def test_pooled_top_layer_bookkeeping_matches_fp64_autograd(cuda, NS, training):
    """bn_finalize -> pool_finalize -> pool_bwd_prep -> bn_bwd_finalize on one z against fp64
    autograd of max_pool(relu(batch_norm(z))): everything of the fused top layer but its GEMM.
    The samples of a (centre, channel) are distinct and no pooled pre-activation is within 1e-3 of
    zero, so the argmax and the ReLU mask are the same in fp32 and fp64."""
    B, NP, C = 2, 48, 40
    M = B * NP * NS
    g = _gen("top_layer", NS, training)
    z = _distinct_samples(B, NP, NS, C, g) + (torch.rand(C, generator=g) * 4 - 2)   # (B*NP, NS, C)
    gamma = (torch.rand(C, generator=g) + 0.5) * torch.where(torch.arange(C) % 3 == 2, -1.0, 1.0)
    beta = torch.randn(C, generator=g) * 0.5
    zf = z.reshape(M, C)
    zd_all = zf.double()
    rm = (zd_all.mean(0) + 0.3 * torch.randn(C, generator=g, dtype=torch.float64)).float()
    rv = (zd_all.var(0) * (0.5 + torch.rand(C, generator=g, dtype=torch.float64))).float()

    # fp64 reference in the reference layout (B, C, NP, NS)
    zd = z.double().view(B, NP, NS, C).permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    w = gamma.double().requires_grad_(True)
    bt = beta.double().requires_grad_(True)
    y = F.batch_norm(zd, None if training else rm.double(), None if training else rv.double(), w, bt,
                     training, 0.0, EPS)
    pre = y.detach().amax(dim=3)                     # the pooled pre-activation
    assert pre.abs().min() > 1e-3, "inputs put a pooled pre-activation at the ReLU threshold"
    out_ref = F.max_pool2d(F.relu(y), kernel_size=[1, NS]).squeeze(-1)               # (B, C, NP)
    wts = pattern_like(out_ref.float())
    (out_ref * wts.double()).sum().backward()
    dz_ref = zd.grad.permute(0, 2, 3, 1).reshape(B * NP, NS, C)

    # the kernels
    zc = z.to(cuda)
    gam, bet = gamma.to(cuda), beta.to(cuda)
    if training:
        stats = _sums(zf).to(cuda)
        scale, shift, mean, invstd = (_nan(C, dev=cuda) for _ in range(4))
        _call("b2r_bn_finalize", _p(stats), C, float(M), _p(gam), _p(bet), EPS, 0.1, None, None,
              _p(scale), _p(shift), _p(mean), _p(invstd), None)
    else:                               # running statistics, as fused_sa.py / dense_mlp.py form them
        mean = rm.to(cuda)
        invstd = torch.rsqrt(rv.to(cuda) + EPS)
        scale = gam * invstd
        shift = bet - mean * scale
    zmax, amax = zc.max(dim=1)
    zmin, amin = zc.min(dim=1)
    amax, amin = amax.int(), amin.int()
    out_cm = _nan(B, C, NP, dev=cuda)
    _call("b2r_pool_finalize", _p(zmax), _p(zmin), _p(scale), _p(shift), B, NP, C, _p(out_cm), None)
    dysel = _nan(B * NP, C, dev=cuda)
    asel = torch.empty((B * NP, C), dtype=torch.int32, device=cuda)
    stats2 = torch.zeros(2 * C, dtype=torch.float64, device=cuda)
    wts_c = wts.to(cuda)
    _call("b2r_pool_bwd_prep", _p(wts_c), None, _p(zmax), _p(zmin), _p(amax), _p(amin),
          _p(scale), _p(shift), B, NP, C, _p(dysel), _p(asel), _p(stats2))
    coef = [_nan(C, dev=cuda) for _ in range(3)]
    dgamma, dbeta = _nan(C, dev=cuda), _nan(C, dev=cuda)
    _call("b2r_bn_bwd_finalize", _p(stats2), C, float(M), _p(gam), _p(mean), _p(invstd),
          int(training), _p(coef[0]), _p(coef[1]), _p(coef[2]), None, None, None, _p(dgamma),
          _p(dbeta))
    a, b, c = (v.double().cpu() for v in coef)
    gr = torch.zeros(B * NP, NS, C, dtype=torch.float64)
    gr.scatter_(1, asel.long().cpu()[:, None, :], dysel.double().cpu()[:, None, :])
    dz = a * gr + b * z.double() + c

    errs = dict(out=rel_l2(out_cm.cpu().numpy(), out_ref.detach().numpy()),
                dz=rel_l2(dz.numpy(), dz_ref.numpy()),
                dgamma=rel_l2(dgamma.cpu().numpy(), w.grad.numpy()),
                dbeta=rel_l2(dbeta.cpu().numpy(), bt.grad.numpy()))
    _log("top_layer NS=%d training=%d" % (NS, training), **errs)
    for k, e in errs.items():
        assert e <= 1e-5, (k, e)


# ---- 6. b2r_to_point_major ----------------------------------------------------------------------

@pytest.mark.parametrize("N", [1, 31, 33, 257])
@pytest.mark.parametrize("C", [1, 31, 33, 257])
def test_to_point_major_exact(cuda, C, N):
    B = 3
    x = torch.randn(B, C, N, generator=_gen("tpm", C, N)).to(cuda)
    out = _nan(B, N, C, dev=cuda)
    _call("b2r_to_point_major", _p(x), B, C, N, _p(out))
    assert torch.equal(out, x.transpose(1, 2))


def test_to_point_major_zero_size_is_a_no_op(cuda):
    x = torch.randn(3, 4, 5, device=cuda)
    out = _nan(64, dev=cuda)
    for B, C, N in ((0, 4, 5), (3, 0, 5), (3, 4, 0)):
        assert _lib().b2r_to_point_major(_p(x), B, C, N, _p(out), None) == 0
    assert torch.isnan(out).all()


# ---- 7. csrc/heads.cu ---------------------------------------------------------------------------

def _interp_inputs(B, n, m, g):
    idx = torch.randint(0, m, (B, n, 3), generator=g, dtype=torch.int32)
    idx[:, ::4, 1] = idx[:, ::4, 0]                  # duplicate neighbours inside one row
    idx[:, ::9, 2] = idx[:, ::9, 0]
    w = torch.rand(B, n, 3, generator=g) + 0.05
    w = w / w.sum(-1, keepdim=True)
    return idx, w


@pytest.mark.parametrize("C2,C1", [(4, 0), (132, 36), (256, 4)])
def test_interp_cat_forward_bit_identical_to_oracle(cuda, C2, C1):
    from oracle import cpu_ops
    B, n, m = 3, 37, 19                              # B*n = 111 rows: not a multiple of 8 warps
    g = _gen("interp_fwd", C2, C1)
    known = torch.randn(B, m, C2, generator=g)
    skip = torch.randn(B, n, C1, generator=g) if C1 else None
    idx, w = _interp_inputs(B, n, m, g)
    out = _nan(B * n, C2 + C1, dev=cuda)
    kc, sc, ic, wc = known.to(cuda), skip.to(cuda) if C1 else None, idx.to(cuda), w.to(cuda)
    _call("b2r_interp_cat_fwd", _p(kc), _p(sc), _p(ic), _p(wc), B, n, m, C2, C1, _p(out))
    out = out.cpu().view(B, n, C2 + C1)
    want = cpu_ops.interp(known.transpose(1, 2).numpy(), idx.numpy(), w.numpy())      # (B, C2, n)
    assert np.array_equal(out[..., :C2].transpose(1, 2).numpy(), want)
    if C1:
        assert torch.equal(out[..., C2:], skip)


@pytest.mark.parametrize("outputs", ["both", "known", "skip"])
@pytest.mark.parametrize("C2,C1,pad", [(4, 0, 4), (132, 8, 0), (132, 0, 0), (256, 36, 8)])
def test_interp_cat_backward_matches_fp64(cuda, C2, C1, pad, outputs):
    B, n, m = 3, 37, 19
    g = _gen("interp_bwd", C2, C1, pad, outputs)
    idx, w = _interp_inputs(B, n, m, g)
    ld_g = C2 + C1 + pad
    gg = torch.randn(B * n, ld_g, generator=g)
    gk0 = torch.randn(B, m, C2, generator=g)           # g_known accumulates onto what it holds
    gk = gk0.clone().to(cuda) if outputs in ("both", "known") else None
    gs = _nan(B * n, C1, dev=cuda) if outputs in ("both", "skip") and C1 else None
    gc, ic, wc = gg.to(cuda), idx.to(cuda), w.to(cuda)
    _call("b2r_interp_cat_bwd", _p(gc), ld_g, _p(ic), _p(wc), B, n, m, C2, C1, _p(gk), _p(gs))
    if gk is not None:
        ref = gk0.double().reshape(B * m, C2).clone()
        mag = gk0.double().abs().reshape(B * m, C2).clone()
        rows = (torch.arange(B).repeat_interleave(n) * m)[:, None] + idx.reshape(B * n, 3).long()
        for k in range(3):
            contrib = w.reshape(B * n, 3)[:, k:k + 1].double() * gg[:, :C2].double()
            ref.index_add_(0, rows[:, k], contrib)
            mag.index_add_(0, rows[:, k], contrib.abs())
        e = _scaled_err(gk.cpu().reshape(B * m, C2), ref, mag)
        _log("interp_cat_bwd C2=%d C1=%d ld_g=%d outputs=%s" % (C2, C1, ld_g, outputs), g_known=e)
        assert e <= 1e-5, e
    if gs is not None:
        assert torch.equal(gs.cpu(), gg[:, C2:C2 + C1])


def _vote_inputs(M, C, pad, g):
    ld = 3 + C + pad
    rs = 10.0 ** (torch.rand(M, 1, generator=g) * 6 - 3)         # row norms from 1e-3 to 1e3
    net = torch.randn(M, ld, generator=g)
    net[:, 3:3 + C] *= 0.5 * rs / C ** 0.5
    sf = torch.randn(M, C, generator=g) * rs / C ** 0.5
    sx = torch.rand(M, 3, generator=g)
    return net, sx, sf, ld


def _vote_fwd(cuda, net, sx, sf, C, ld):
    M = net.shape[0]
    vx, out, norm = _nan(M, 3, dev=cuda), _nan(M, C, dev=cuda), _nan(M, dev=cuda)
    nc, sxc, sfc = net.to(cuda), sx.to(cuda), sf.to(cuda)
    _call("b2r_vote_tail_fwd", _p(nc), ld, _p(sxc), _p(sfc), M, C, _p(vx), _p(out), _p(norm))
    return vx.cpu(), out.cpu(), norm.cpu()


@pytest.mark.parametrize("C,pad", [(1, 0), (1, 4), (33, 4), (256, 1), (257, 8)])
def test_vote_tail_forward_matches_fp64(cuda, C, pad):
    M = 8 * 13 + 5
    net, sx, sf, ld = _vote_inputs(M, C, pad, _gen("vote_fwd", C, pad))
    vx, out, norm = _vote_fwd(cuda, net, sx, sf, C, ld)
    assert torch.equal(vx, sx + net[:, :3])
    v = (sf + net[:, 3:3 + C]).double()                # the kernel's one fp32 add, then fp64
    nrm = v.norm(dim=1)
    errs = dict(norm=_scaled_err(norm, nrm, nrm), out=_scaled_err(out, v / nrm[:, None], (v / nrm[:, None]).abs()))
    _log("vote_tail_fwd C=%d ld_net=%d" % (C, ld), **errs)
    for k, e in errs.items():
        assert e <= RTOL, (k, e)


@pytest.mark.parametrize("null", ["none", "g_out", "g_vote_xyz", "g_seed_feat"])
@pytest.mark.parametrize("C,pad", [(1, 4), (33, 4), (256, 1), (257, 8)])
def test_vote_tail_backward_matches_fp64_autograd(cuda, C, pad, null):
    M = 8 * 13 + 5
    g = _gen("vote_bwd", C, pad, null)
    net, sx, sf, ld = _vote_inputs(M, C, pad, g)
    _, out, norm = _vote_fwd(cuda, net, sx, sf, C, ld)
    g_out = torch.randn(M, C, generator=g) if null != "g_out" else None
    g_vx = torch.randn(M, 3, generator=g) if null != "g_vote_xyz" else None
    g_net = _nan(M, ld, dev=cuda)                     # every column, padding included, is written
    g_seed = _nan(M, C, dev=cuda) if null != "g_seed_feat" else None
    goc = g_out.to(cuda) if g_out is not None else None
    gvc = g_vx.to(cuda) if g_vx is not None else None
    oc, nc = out.to(cuda), norm.to(cuda)
    _call("b2r_vote_tail_bwd", _p(goc), _p(gvc), _p(oc), _p(nc), M, C, ld, _p(g_net), _p(g_seed))
    g_net = g_net.cpu()
    assert torch.equal(g_net[:, :3], g_vx if g_vx is not None else torch.zeros(M, 3))
    assert torch.equal(g_net[:, 3 + C:], torch.zeros(M, pad))
    if g_seed is not None:
        assert torch.equal(g_seed.cpu(), g_net[:, 3:3 + C])
    if g_out is None:
        assert torch.equal(g_net[:, 3:3 + C], torch.zeros(M, C))
        return
    v = (sf + net[:, 3:3 + C]).double().requires_grad_(True)
    (v / v.norm(dim=1, keepdim=True)).backward(g_out.double())
    o = out.double()
    mag = (g_out.double().abs() + o.abs() * (g_out.double() * o).abs().sum(1, keepdim=True)) / \
        norm.double()[:, None]
    e = _scaled_err(g_net[:, 3:3 + C], v.grad, mag)
    _log("vote_tail_bwd C=%d ld_net=%d null=%s" % (C, ld, null), g_net=e)
    assert e <= 1e-5, e
