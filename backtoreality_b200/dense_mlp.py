"""Point-major dense MLP heads on tcgen05 (host side of csrc/dense.cu and csrc/heads.cu).

Covers what the reference runs as cuDNN Conv1d / Conv2d(1x1) + BatchNorm + ReLU chains on
(B, C, n) tensors around the set-abstraction path:

    PointnetFPModule.mlp          pointnet2_modules.py:505-514   cat -> SharedMLP [512,256,256]
    VotingModule conv1..3/bn1..2  models/voting_module.py:38-65  (+ votenet.py:93-94 normalise)
    ProposalModule conv1..3/bn1..2 models/proposal_module.py:115-119

A layer here is  z (M, Cout) = x (M, Cin) W^T (+ bias)  on M = B*n positions, point-major, with the
previous layer's BatchNorm + ReLU applied while loading x, BatchNorm batch statistics accumulated
by the GEMM epilogue, and -- in backward -- the ReLU mask and the BatchNorm-backward sums fused
into the input-gradient GEMM.  TF32 operands, FP32 accumulate, forward AND backward (the
precision the reference's cuDNN runs these convolutions at).  Training-mode BatchNorm semantics
(biased batch variance, running statistics with the module's momentum, num_batches_tracked) are
nn.BatchNorm1d/2d's; eval mode uses the running statistics.

No CPU or library fallback inside this module: it raises when libb2r.so is missing.  Callers
(pointnet2_modules.PointnetFPModule, votenet.VotingModule / ProposalModule) keep the reference's
torch formulation for shapes this path does not cover (`supported`) and when ENABLED is False.
"""
import ctypes
import os

import torch

from . import _ext, _lib, pytorch_utils, step_arena

_vp = ctypes.c_void_p

# B2R_DENSE=0 routes the FP / voting / proposal MLPs through torch (cuDNN), as in round 1
ENABLED = os.environ.get("B2R_DENSE", "1") not in ("0", "")


def _ptr(t):
    return _vp(t.data_ptr()) if t is not None else None


def _ceil4(c):
    return (int(c) + 3) & ~3


def _vec(c, dev):
    """A per-channel coefficient vector the kernels may read up to the next multiple of 4."""
    if c % 4 == 0:      # no padding to define: spare the fill kernel (40 of them per VoteNet step)
        return torch.empty(c, dtype=torch.float32, device=dev)
    return torch.zeros(_ceil4(c), dtype=torch.float32, device=dev)


def layer_specs(convs, bns):
    """[(conv, bn or None)] from parallel lists (bn None = plain biased linear layer)."""
    return list(zip(convs, bns))


def enabled():
    """The dense tcgen05 path is on: ENABLED, and the fused SA blocks are (fused_sa.ENABLED = False
    means "the reference's formulation everywhere", e.g. the fp32 comparison arm of the tests)."""
    from . import fused_sa
    return ENABLED and fused_sa.ENABLED


def supported(specs, x):
    if not (enabled() and x.is_cuda and x.dtype == torch.float32):
        return False
    for conv, bn in specs:
        k = conv.kernel_size
        if tuple(k) not in ((1,), (1, 1)) or conv.groups != 1:
            return False
        if bn is not None and (bn.momentum is None or not bn.track_running_stats or not bn.affine):
            return False
    for i, (conv, bn) in enumerate(specs):
        if bn is None and i != len(specs) - 1:
            return False        # only the LAST layer may come without BatchNorm + ReLU
        if bn is not None and i == len(specs) - 1 and conv.out_channels % 4:
            return False
    return specs[0][0].in_channels % 4 == 0


# ---- weight images packed ahead of time, off the critical path -------------------------------
# Every layer needs its weight as a swizzled TF32 operand image (W for forward, W^T for the input
# gradient).  `prepack` issues all of them on a side stream at the start of the step (they depend
# on nothing but the weights); `_DenseMLP` then takes its images instead of packing inline.
_PREPACKED = {}      # id(weight) -> (w_img, wt_img, event, weight._version, weight)
_SIDE = {}           # device -> (pack stream, weight-gradient stream)
_PACK_EVENTS = {}    # device -> event of the last prepack


def _streams(dev):
    st = _SIDE.get(dev)
    if st is None:
        st = _SIDE[dev] = (torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev))
    return st


def _pack(w2, Cout, Cin, need_wt):
    lib = _lib.lib()
    dev = w2.device
    w_img = torch.empty(int(lib.b2r_dense_image_bytes(Cout, Cin)) // 4, dtype=torch.float32, device=dev)
    wt_img = None
    if need_wt:
        wt_img = torch.empty(int(lib.b2r_dense_image_bytes(Cin, Cout)) // 4, dtype=torch.float32,
                             device=dev)
    _lib.check(lib.b2r_dense_pack(_ptr(w2), Cout, Cin, _ptr(w_img), _ptr(wt_img), _ext._stream()),
               "dense_pack")
    _ext.LAUNCHES += 1 if wt_img is None else 2
    return w_img, wt_img


def prepack(convs):
    """Pack the operand images of the given 1x1 convolutions on a side stream (consumed once by
    the next forward through each; a weight modified in between is re-packed inline)."""
    convs = [c for c in convs if c is not None and c.weight.is_cuda]
    if not convs or not enabled():
        return
    dev = convs[0].weight.device
    for key in [k for k, ent in list(_PREPACKED.items()) if ent[4].device == dev]:
        _PREPACKED.pop(key, None)
    main = torch.cuda.current_stream(dev)
    side = _streams(dev)[0]
    side.wait_stream(main)
    want_wt = torch.is_grad_enabled()
    with torch.cuda.stream(side), torch.no_grad():
        ents = []
        for c in convs:
            w = c.weight
            w_img, wt_img = _pack(w.detach().reshape(c.out_channels, c.in_channels), c.out_channels,
                                  c.in_channels, want_wt)
            ents.append((w, w_img, wt_img))
        ev = torch.cuda.Event()
        ev.record(side)
    for w, w_img, wt_img in ents:
        _PREPACKED[id(w)] = (w_img, wt_img, ev, w._version, w)
    _PACK_EVENTS[dev] = ev


def prepack_join():
    """Make the current stream wait for the last `prepack` (a CUDA-graph capture must not end
    with the packing stream un-joined)."""
    if not torch.cuda.is_available():
        return
    dev = torch.device("cuda", torch.cuda.current_device())
    ev = _PACK_EVENTS.pop(dev, None)
    if ev is not None:
        torch.cuda.current_stream().wait_event(ev)


def _take(weight):
    ent = _PREPACKED.pop(id(weight), None)
    if ent is None or ent[4] is not weight or ent[3] != weight._version:
        return None
    main = torch.cuda.current_stream(weight.device)
    main.wait_event(ent[2])
    for t in ent[:2]:
        if t is not None:
            t.record_stream(main)
    return ent[0], ent[1]


class _DenseMLP(torch.autograd.Function):
    """x (M, Cin) point-major -> chain of [conv1x1 (+bias) -> BatchNorm -> ReLU], the last layer
    optionally a plain biased conv.  Returns (out_pm, out_cm):
      last layer with BatchNorm:  out_pm (B, n, C) and out_cm (B, C, n) = relu(bn(z))
      last layer plain:           out_pm (M, ld) raw z with ld = ceil4(C) (columns >= C undefined),
                                  out_cm None
    Parameters are passed flat as (weight, bias | None, gamma | None, beta | None) per layer."""

    @staticmethod
    def forward(ctx, x, specs, training, B, n, *params):
        lib = _lib.lib()
        st = _ext._stream()
        dev = x.device
        M, L = x.shape[0], len(specs)
        assert x.is_contiguous() and x.shape[1] % 4 == 0 and M == B * n
        need = any(ctx.needs_input_grad)
        cur, ld_cur, sc, sh = x, x.shape[1], None, None
        zs, bn_saved, images = [], [], []
        # batch statistics of every layer: ONE zero-filled buffer
        stats_all, s_off = None, 0
        if training:
            stats_all = step_arena.zeros(sum(2 * c.out_channels for c, b in specs if b is not None),
                                    dtype=torch.float64, device=dev)
        for l, (conv, bn) in enumerate(specs):
            w, bias = params[4 * l], params[4 * l + 1]
            Cout, Cin = conv.out_channels, conv.in_channels
            need_wt = need and (l > 0 or ctx.needs_input_grad[0])
            taken = _take(w)
            if taken is None or (need_wt and taken[1] is None):
                taken = _pack(w.detach().reshape(Cout, Cin), Cout, Cin, need_wt)
            w_img, wt_img = taken
            ld_z = _ceil4(Cout)
            z = torch.empty((M, ld_z), dtype=torch.float32, device=dev)
            stats = None
            if bn is not None and training:
                stats = stats_all[s_off:s_off + 2 * Cout]
                s_off += 2 * Cout
            d = _lib.DenseLayer()
            d.M, d.Cin, d.Cout = M, Cin, Cout
            d.in_, d.ld_in, d.sc_in, d.sh_in = _ptr(cur), ld_cur, _ptr(sc), _ptr(sh)
            d.w_img, d.bias = _ptr(w_img), _ptr(bias.detach() if bias is not None else None)
            d.z, d.ld_z, d.stats = _ptr(z), ld_z, _ptr(stats)
            with _ext._timed("dense_fwd"):
                _lib.check(lib.b2r_dense_fwd(ctypes.byref(d), st), "dense_fwd")
            if bn is not None:
                sc, sh = _vec(Cout, dev), _vec(Cout, dev)
                if training:
                    mean = torch.empty(Cout, dtype=torch.float32, device=dev)
                    invstd = torch.empty_like(mean)
                    pytorch_utils.bn_finalize(bn, stats, Cout, M, sc, sh, mean, invstd, st)
                    _ext.LAUNCHES += 1
                else:
                    invstd = torch.rsqrt(bn.running_var + bn.eps)
                    mean = bn.running_mean
                    sc[:Cout] = bn.weight * invstd
                    sh[:Cout] = bn.bias - bn.running_mean * sc[:Cout]
                bn_saved.append((mean, invstd, sc, sh))
            else:
                sc = sh = None
                bn_saved.append(None)
            zs.append(z)
            images.append(wt_img)
            cur, ld_cur = z, ld_z
        last_bn = specs[-1][1] is not None
        if last_bn:
            C = specs[-1][0].out_channels
            out_cm = torch.empty((B, C, n), dtype=torch.float32, device=dev)
            out_pm = torch.empty((B, n, C), dtype=torch.float32, device=dev)
            _lib.check(lib.b2r_pool_finalize(_ptr(cur), _ptr(cur), _ptr(sc), _ptr(sh), B, n, C,
                                             _ptr(out_cm), _ptr(out_pm), st), "pool_finalize")
            _ext.LAUNCHES += 1
        else:
            out_pm, out_cm = cur, None
        ctx.set_materialize_grads(False)
        if need:
            # x and the z's go through save_for_backward: the plain last layer's z IS an output of
            # this node, and an output kept as a ctx attribute is a reference cycle (node -> output
            # -> node) that keeps the whole autograd graph -- AccumulateGrad nodes and their
            # streams included -- alive until the garbage collector runs
            ctx.save_for_backward(x, *zs)
            ctx.saved = (specs, bool(training), B, n, bn_saved, images, params)
        return out_pm, out_cm

    @staticmethod
    def backward(ctx, g_pm, g_cm):
        specs, training, B, n, bn_saved, images, params = ctx.saved
        x, zs = ctx.saved_tensors[0], list(ctx.saved_tensors[1:])
        L = len(specs)
        n_in = 5
        if g_pm is None and g_cm is None:
            return (None,) * (n_in + 4 * L)
        lib = _lib.lib()
        st = _ext._stream()
        dev = x.device
        M = x.shape[0]
        f32 = dict(dtype=torch.float32, device=dev)
        tr = 1 if training else 0
        grads = [None] * (4 * L)
        top = L - 1
        Ct = specs[top][0].out_channels
        coef = None
        # every accumulated output from two zero-filled buffers
        dW_all = step_arena.zeros(sum(c.out_channels * c.in_channels for c, _ in specs), **f32)
        st_all = step_arena.zeros(sum(2 * c.out_channels for c, b in specs if b is not None),
                             dtype=torch.float64, device=dev)
        w_off, s_off = [0], [0]
        for c, b_ in specs:
            w_off.append(w_off[-1] + c.out_channels * c.in_channels)
            s_off.append(s_off[-1] + (2 * c.out_channels if b_ is not None else 0))
        # the weight gradients are off the dependency chain (layer l's input gradient only needs
        # dz and W): they run on a side stream beside the chain and are joined at the end
        main = torch.cuda.current_stream(dev)
        wside = _streams(dev)[1]
        keep = []     # buffers the side stream reads: alive until the join below
        if specs[top][1] is not None:
            # relu / BatchNorm backward of the output layer: mask the incoming gradient with
            # [relu(bn(z)) > 0] and take its two BatchNorm-backward sums (the pooled-output helper
            # with max == min == z)
            mean, invstd, sc, sh = bn_saved[top]
            z = zs[top]
            gr = torch.empty((M, Ct), **f32)
            scratch = torch.empty((M, Ct), dtype=torch.int32, device=dev)
            stats = st_all[s_off[top]:s_off[top + 1]]
            _lib.check(lib.b2r_pool_bwd_prep(
                _ptr(g_cm.contiguous() if g_cm is not None else None),
                _ptr(g_pm.contiguous() if g_pm is not None else None), _ptr(z), _ptr(z),
                _ptr(scratch), _ptr(scratch), _ptr(sc), _ptr(sh), B, n, Ct, _ptr(gr),
                _ptr(scratch), _ptr(stats), st), "pool_bwd_prep")
            _ext.LAUNCHES += 1
            coef = _DenseMLP._bn_bwd(lib, st, stats, specs[top], params, top, mean, invstd, M, tr,
                                     grads, dev)
            ld_g = Ct
        else:
            assert g_cm is None
            gr = g_pm.contiguous()
            ld_g = gr.shape[1]
            if params[4 * top + 1] is not None:
                # bias gradient of the plain last layer: a 14 us column reduction nothing downstream
                # waits for -- on the weight-gradient side stream, off the critical path
                wside.wait_stream(main)
                with torch.cuda.stream(wside):
                    grads[4 * top + 1] = gr[:, :Ct].sum(0)
                gr.record_stream(wside)
                grads[4 * top + 1].record_stream(main)
        g_x = None
        for l in range(L - 1, -1, -1):
            conv, bn = specs[l]
            Cout, Cin = conv.out_channels, conv.in_channels
            b = _lib.DenseLayerBwd()
            b.M, b.Cin, b.Cout = M, Cin, Cout
            if l == 0:
                b.in_, b.ld_in = _ptr(x), x.shape[1]
            else:
                b.in_, b.ld_in = _ptr(zs[l - 1]), zs[l - 1].shape[1]
                b.sc_in, b.sh_in = _ptr(bn_saved[l - 1][2]), _ptr(bn_saved[l - 1][3])
            b.g, b.zz, b.ld_g = _ptr(gr), _ptr(zs[l]), ld_g
            if coef is not None:
                b.ca, b.cb, b.cc = _ptr(coef[0]), _ptr(coef[1]), _ptr(coef[2])
            gin = stats_in = None
            want_gin = l > 0 or ctx.needs_input_grad[0]
            # weight gradient: same descriptor, on the side stream (dz's inputs are ready now)
            dW = dW_all[w_off[l]:w_off[l + 1]].view(Cout, Cin)
            b.dW = _ptr(dW)
            keep += [gr, coef]
            wside.wait_stream(main)
            with _ext._timed("dense_bwd"):
                _lib.check(lib.b2r_dense_bwd(ctypes.byref(b), _vp(wside.cuda_stream)), "dense_bwd")
            b.dW = None
            if want_gin:
                ld_gin = zs[l - 1].shape[1] if l > 0 else x.shape[1]
                gin = torch.empty((M, ld_gin), **f32)
                if ld_gin != Cin:
                    gin[:, Cin:].zero_()
                b.wt_img, b.gin, b.ld_gin = _ptr(images[l]), _ptr(gin), ld_gin
                if l > 0:
                    stats_in = st_all[s_off[l - 1]:s_off[l]]
                    b.stats_in = _ptr(stats_in)
                _lib.check(lib.b2r_dense_bwd(ctypes.byref(b), st), "dense_bwd")
                _ext.LAUNCHES += 1
            grads[4 * l] = dW.view_as(params[4 * l])
            if l > 0:
                mean, invstd, _, _ = bn_saved[l - 1]
                coef = _DenseMLP._bn_bwd(lib, st, stats_in, specs[l - 1], params, l - 1, mean,
                                         invstd, M, tr, grads, dev)
                gr, ld_g = gin, gin.shape[1]
            else:
                g_x = gin
        main.wait_stream(wside)      # join: the weight gradients are complete for what follows
        return (g_x, None, None, None, None) + tuple(grads)

    @staticmethod
    def _bn_bwd(lib, st, stats, spec, params, l, mean, invstd, M, tr, grads, dev):
        """BatchNorm backward bookkeeping of layer l -> (ca, cb, cc); fills dgamma / dbeta / dbias."""
        C = spec[0].out_channels
        coef = [_vec(C, dev) for _ in range(3)]
        dgamma = torch.empty(C, dtype=torch.float32, device=dev)
        dbeta = torch.empty_like(dgamma)
        has_bias = params[4 * l + 1] is not None
        dbias = torch.empty_like(dgamma) if has_bias else None
        _lib.check(lib.b2r_bn_bwd_finalize_ex(
            _ptr(stats), C, float(M), _ptr(params[4 * l + 2].detach()), _ptr(mean), _ptr(invstd), tr,
            _ptr(coef[0]), _ptr(coef[1]), _ptr(coef[2]), None, None, None, _ptr(dgamma),
            _ptr(dbeta), _ptr(dbias), st), "bn_bwd_finalize")
        _ext.LAUNCHES += 1
        grads[4 * l + 1], grads[4 * l + 2], grads[4 * l + 3] = dbias, dgamma, dbeta
        return coef


def dense_mlp(x_pm, specs, training, B, n):
    """x_pm (B*n, Cin) contiguous.  -> (out_pm, out_cm), see _DenseMLP."""
    params = []
    for conv, bn in specs:
        params += [conv.weight, conv.bias, bn.weight if bn is not None else None,
                   bn.bias if bn is not None else None]
    return _DenseMLP.apply(x_pm, specs, training, B, n, *params)


class _InterpCat(torch.autograd.Function):
    """three_interpolate + cat on point-major tensors: known (B,m,C2), skip (B,n,C1) | None,
    idx / weight (B,n,3) -> (B*n, C2 + C1)."""

    @staticmethod
    def forward(ctx, known, skip, idx, weight):
        B, m, C2 = known.shape
        n = idx.shape[1]
        C1 = skip.shape[2] if skip is not None else 0
        out = torch.empty((B * n, C2 + C1), dtype=torch.float32, device=known.device)
        _lib.check(_lib.lib().b2r_interp_cat_fwd(_ptr(known), _ptr(skip), _ptr(idx), _ptr(weight),
                                                 B, n, m, C2, C1, _ptr(out), _ext._stream()),
                   "interp_cat_fwd")
        _ext.LAUNCHES += 1
        ctx.saved = (idx, weight, B, n, m, C2, C1)
        return out

    @staticmethod
    def backward(ctx, g):
        idx, weight, B, n, m, C2, C1 = ctx.saved
        g = g.contiguous()
        g_known = g_skip = None
        if ctx.needs_input_grad[0]:
            g_known = step_arena.zeros((B, m, C2), dtype=torch.float32, device=g.device)
        if C1 and ctx.needs_input_grad[1]:
            g_skip = torch.empty((B, n, C1), dtype=torch.float32, device=g.device)
        _lib.check(_lib.lib().b2r_interp_cat_bwd(_ptr(g), g.shape[1], _ptr(idx), _ptr(weight), B, n,
                                                 m, C2, C1, _ptr(g_known), _ptr(g_skip),
                                                 _ext._stream()), "interp_cat_bwd")
        _ext.LAUNCHES += 1
        return g_known, g_skip, None, None


def interp_cat(known_pm, skip_pm, idx, weight):
    return _InterpCat.apply(known_pm.contiguous(), skip_pm.contiguous() if skip_pm is not None else None,
                            idx.contiguous(), weight.contiguous())


class _VoteTail(torch.autograd.Function):
    """net (M, ld) = [offset(3), residual(C), pad], seed_xyz (B,n,3), seed_feat (B,n,C) point-major
    -> vote_xyz (B,n,3), vote_features (B,n,C) L2-normalised over the channels."""

    @staticmethod
    def forward(ctx, net, seed_xyz, seed_feat):
        B, n, C = seed_feat.shape
        M = B * n
        dev = net.device
        vote_xyz = torch.empty((B, n, 3), dtype=torch.float32, device=dev)
        out = torch.empty((B, n, C), dtype=torch.float32, device=dev)
        norm = torch.empty(M, dtype=torch.float32, device=dev)
        _lib.check(_lib.lib().b2r_vote_tail_fwd(_ptr(net), net.shape[1], _ptr(seed_xyz),
                                                _ptr(seed_feat), M, C, _ptr(vote_xyz), _ptr(out),
                                                _ptr(norm), _ext._stream()), "vote_tail_fwd")
        _ext.LAUNCHES += 1
        ctx.save_for_backward(out, norm)     # `out` is an output: never as a ctx attribute (cycle)
        ctx.ld = net.shape[1]
        ctx.set_materialize_grads(False)
        return vote_xyz, out

    @staticmethod
    def backward(ctx, g_xyz, g_out):
        out, norm = ctx.saved_tensors
        ld = ctx.ld
        B, n, C = out.shape
        if g_xyz is None and g_out is None:
            return None, None, None
        g_xyz = g_xyz.contiguous() if g_xyz is not None else None
        g_out = g_out.contiguous() if g_out is not None else None
        g_net = torch.empty((B * n, ld), dtype=torch.float32, device=out.device)
        g_seed = torch.empty_like(out) if ctx.needs_input_grad[2] else None
        _lib.check(_lib.lib().b2r_vote_tail_bwd(_ptr(g_out), _ptr(g_xyz), _ptr(out), _ptr(norm),
                                                B * n, C, ld, _ptr(g_net), _ptr(g_seed),
                                                _ext._stream()), "vote_tail_bwd")
        _ext.LAUNCHES += 1
        return g_net, (g_xyz if ctx.needs_input_grad[1] else None), g_seed


def vote_tail(net, seed_xyz, seed_feat_pm):
    return _VoteTail.apply(net, seed_xyz.contiguous(), seed_feat_pm.contiguous())
