"""Fused SharedMLP block of a set-abstraction layer on tcgen05 tensor cores (host side).

Drives csrc/mlp.cu through the C ABI (`b2r_mlp_pack_weight`, `b2r_sa_layer_fwd`,
`b2r_bn_finalize`, `b2r_pool_finalize`, include/b2r.h) to compute what the reference computes in
PointnetSAModuleVotes.forward (pointnet2_modules.py:245-267) with
QueryAndGroup -> SharedMLP(3 x [Conv2d 1x1 -> BatchNorm2d -> ReLU]) -> max_pool2d:

    layer 0   gather (idx) + relative/normalised xyz  -> TF32 GEMM -> raw z0 + batch statistics
    layer i   relu(bn(z_{i-1})) applied on load       -> TF32 GEMM -> raw z_i + batch statistics
    last      ... -> TF32 GEMM -> statistics + max/min over nsample (no (B,C,np,ns) tensor)
    finalize  BatchNorm scale/shift (+ running-stat update) and relu(bn(max|min)) -> (B,C,np)

Training-mode BatchNorm uses biased batch statistics over all B*npoint*nsample positions of the
local batch, updates running_mean / running_var (unbiased) with the module's momentum and bumps
num_batches_tracked, exactly like nn.BatchNorm2d (reference pytorch_utils.py:55-58).
Math, FORWARD: TF32 operands (round-to-nearest), FP32 accumulate -- the precision the reference
itself runs at by default (cuDNN TF32 convolutions on sm_80+).
Math, BACKWARD (csrc/mlp_bwd.cu): BF16 operands (X, dz and W rounded to 8 mantissa bits -- NARROWER
than the reference's cuDNN TF32 wgrad / dgrad), FP32 accumulate; the pooled top layer's z is
recomputed in BF16 for the BatchNorm-backward term while the max-pool routing comes from the TF32
forward.  Per layer that is <= 1e-2 rel-L2 against fp64 (measured ~3e-3; tests/test_mlp_gpu.py),
below the 3-4e-2 per-block gradient noise any TF32 forward already causes by flipping ReLU masks /
pool winners (DESIGN.md "Tolerances").  Why BF16: tcgen05 reads the transposed (MN-major) operand
views the weight gradient needs from the same bytes only for 16-bit data (DESIGN.md section 4).
To take the backward out of the comparison, set `fused_sa.ENABLED = False` (or B2R_FUSED=0): the
block then runs QueryAndGroup + torch SharedMLP + max_pool2d, forward and backward, at whatever
precision torch.backends.cudnn.allow_tf32 selects -- the tests' fp32 arm.

Pad-free position space (COMPACT, csrc/compact.cu): blocks with nsample >= 32 do not recompute the
copies of a ball's first hit that the ball query pads with; see `compact_plan`.
"""
import ctypes
import functools
import os

import torch

from . import _ext, _lib, pytorch_utils, step_arena

_vp = ctypes.c_void_p


def _ptr(t):
    return _vp(t.data_ptr()) if t is not None else None


def to_point_major(features):
    """(B,C,N) -> (B,N,C) contiguous."""
    B, C, N = features.shape
    out = torch.empty((B, N, C), dtype=torch.float32, device=features.device)
    _lib.check(_lib.lib().b2r_to_point_major(_ptr(features), B, C, N, _ptr(out), _ext._stream()),
               "to_point_major")
    _ext.LAUNCHES += 1
    return out


def pack_weight(weight, gather):
    """Conv weight (Cout,Cin,1,1) -> packed TF32 swizzled image (1-D float tensor)."""
    Cout, Cin = weight.shape[0], weight.shape[1]
    w = weight.detach().reshape(Cout, Cin).contiguous()
    nbytes = _lib.lib().b2r_mlp_weight_image_bytes(Cout, Cin, 1 if gather else 0)
    image = torch.empty(nbytes // 4, dtype=torch.float32, device=weight.device)
    _lib.check(_lib.lib().b2r_mlp_pack_weight(_ptr(w), Cout, Cin, 1 if gather else 0, _ptr(image),
                                              _ext._stream()), "mlp_pack_weight")
    _ext.LAUNCHES += 1
    return image


# ---- channel slices ----------------------------------------------------------------------------
# A layer too large for one launch (GroupFree3D's width-2 backbone: 259/515 -> 256 gather layers,
# 256 -> 256, 256 -> 512) runs as a fixed grid of launches, each over a slice of the output
# channels and, for gather layers, of the feature channels.  The library chooses the grid
# (b2r_sa_layer_fwd_slices / _bwd_slices); a layer that fits one launch gets the single entry
# (0, 0, 0, 0), i.e. the whole-layer launch with every slice field zero.
@functools.lru_cache(maxsize=None)
def slice_grid(backward, Cin, Cout, gather, last):
    """[(co0, co_n, ci0, ci_n)] in launch order: output slice by output slice, feature slices in
    increasing order inside each."""
    co, ci = ctypes.c_int(), ctypes.c_int()
    fn = _lib.lib().b2r_sa_layer_bwd_slices if backward else _lib.lib().b2r_sa_layer_fwd_slices
    n = fn(Cin, Cout, 1 if gather else 0, 1 if last else 0, ctypes.byref(co), ctypes.byref(ci))
    if n <= 0:
        raise RuntimeError("no fused launch grid for a %d -> %d layer" % (Cin, Cout))
    if n == 1:
        return ((0, 0, 0, 0),)
    C = Cin - 3
    fs = [(c0, min(ci.value, C - c0)) for c0 in range(0, C, ci.value)] if ci.value else [(0, 0)]
    grid = tuple((o0, min(co.value, Cout - o0), c0, cn)
                 for o0 in range(0, Cout, co.value) for c0, cn in fs)
    assert len(grid) == n, (grid, n)
    return grid


def _slice_weight(w, co0, co_n, ci0, ci_n):
    """Weight (Cout,Cin) of one slice: rows co0.., and for a feature slice the columns
    [xyz, features ci0..ci0+ci_n) with the xyz columns zero unless ci0 == 0 (they enter once)."""
    if co_n == 0:
        return w
    w = w[co0:co0 + co_n]
    if ci_n:
        xyz = w[:, :3] if ci0 == 0 else torch.zeros_like(w[:, :3])
        w = torch.cat([xyz, w[:, 3 + ci0:3 + ci0 + ci_n]], 1)
    return w.contiguous()


def pack_layer(weight, gather, kind, last):
    """One operand image per launch of the layer's slice grid: "tf32" (forward) or "bf16"
    (backward)."""
    Cout, Cin = weight.shape[0], weight.shape[1]
    w = weight.detach().reshape(Cout, Cin)
    pack = pack_weight if kind == "tf32" else pack_weight_bf16
    return [pack(_slice_weight(w, *sl), gather)
            for sl in slice_grid(kind == "bf16", Cin, Cout, gather, last)]


# ---- weight images packed ahead of time, off the critical path -------------------------------
# Every fused layer needs its weight as a swizzled operand image (TF32 forward, BF16 backward):
# 29 tiny launches per VoteNet step, each sitting between two dependent kernels on the main
# stream.  `prepack` issues them all on a side stream at the start of the step (they depend on
# nothing but the weights); the layers then `_take` their image instead of packing inline.
_PREPACKED = {}      # (id(weight), kind) -> (image, event, weight._version, weight)
_PACK_STREAMS = {}   # device -> side stream
_PACK_EVENTS = {}    # device -> events recorded by its last prepack (joined by prepack_join)


def prepack(mlp_modules, backward=None):
    """Pack the operand images of every conv of the given SharedMLP modules on a side stream.
    Entries are consumed once (a second forward through the same module in the same step packs
    inline again) and dropped by the next call for the same device; a weight modified in between
    is detected by its version counter and re-packed.  The registry is process-wide on purpose:
    autograd runs the backward nodes -- which take the BF16 images -- on its own threads; entries
    and events are kept per device so that nn.DataParallel replicas (one thread and one device
    each, reference train_Votenet_FSB.py:164-168) do not drop each other's images."""
    mlp_modules = [m for m in mlp_modules if m is not None and len(m) > 0]
    if not mlp_modules or not mlp_modules[0][0].conv.weight.is_cuda:
        if not torch.cuda.is_available():
            return
        dev = torch.device("cuda", torch.cuda.current_device())
    else:
        dev = mlp_modules[0][0].conv.weight.device
    for key in [k for k, ent in list(_PREPACKED.items()) if ent[3].device == dev]:
        _PREPACKED.pop(key, None)
    _PACK_EVENTS[dev] = []
    if not mlp_modules or not mlp_modules[0][0].conv.weight.is_cuda:
        return
    if backward is None:
        backward = torch.is_grad_enabled()
    main = torch.cuda.current_stream(dev)
    side = _PACK_STREAMS.get(dev)
    if side is None:
        side = _PACK_STREAMS[dev] = torch.cuda.Stream(device=dev)
    side.wait_stream(main)
    with torch.cuda.stream(side), torch.no_grad():
        for kind in (("tf32", "bf16") if backward else ("tf32",)):
            for mlp in mlp_modules:
                entries = []
                for i, blk in enumerate(mlp):
                    w = blk.conv.weight
                    if kind == "bf16" and not w.requires_grad:
                        continue
                    images = pack_layer(w, i == 0, kind, i == len(mlp) - 1)
                    # a one-launch layer keeps its single image, a sliced one the list
                    entries.append(((id(w), kind), images[0] if len(images) == 1 else images,
                                    w._version, w))
                ev = torch.cuda.Event()
                ev.record(side)
                _PACK_EVENTS[dev].append(ev)
                for key, image, version, w in entries:
                    _PREPACKED[key] = (image, ev, version, w)


def prepack_join():
    """Make the current stream wait for everything the last `prepack` issued (also needed so that
    a CUDA-graph capture never ends with the packing stream un-joined)."""
    if not torch.cuda.is_available():
        return
    dev = torch.device("cuda", torch.cuda.current_device())
    for ev in _PACK_EVENTS.pop(dev, []):
        torch.cuda.current_stream().wait_event(ev)


def _take(weight, kind):
    ent = _PREPACKED.pop((id(weight), kind), None)
    # the entry holds the Parameter itself: same object (not a recycled id / address) and
    # unmodified since it was packed
    if ent is None or ent[3] is not weight or ent[2] != weight._version:
        return None
    image, ev = ent[0], ent[1]
    main = torch.cuda.current_stream(weight.device)
    main.wait_event(ev)
    for im in _as_list(image):
        im.record_stream(main)
    return image


def _as_list(image):
    """A `_take` result as the list of per-slice images (one entry for a one-launch layer)."""
    return [image] if torch.is_tensor(image) else image


# Pad-free position space (csrc/compact.cu): the ball query pads a centre's unused slots with
# copies of its first hit; the fused block computes each centre on its first 8/16/32/64 >= cnt
# samples only and weights sample 0 by the number of copies it stands for.  Same results up to
# fp32 summation order; on ScanNet-shaped scenes SA1 keeps ~73 % and SA2 ~39 % of its positions.
# Used for blocks with nsample >= COMPACT_MIN_NS (with 16 samples nearly every ball is full).
COMPACT = os.environ.get("B2R_COMPACT", "1") not in ("0", "")
COMPACT_MIN_NS = 32
PLAN_KEYS = ("cidx", "ccen", "cmeta")


def compact_wanted(nsample):
    return COMPACT and nsample in (32, 64) and nsample >= COMPACT_MIN_NS


def compact_plan(idx, N):
    """idx (B,NP,NS) int32 ball-query output (or ANY index tensor: a centre's trailing run of
    copies of its sample 0 is what gets dropped) over N source points per scene ->
    {"cidx", "ccen" (capacity ints each), "cmeta" (16 ints)} for sa_block(..., plan=).  Three tiny
    launches on the current stream; no host synchronisation (sizes stay on the device)."""
    B, NP, NS = idx.shape
    lib = _lib.lib()
    cap = int(lib.b2r_compact_capacity(B, NP, NS))
    dev = idx.device
    cidx = torch.empty(cap, dtype=torch.int32, device=dev)
    ccen = torch.empty(cap, dtype=torch.int32, device=dev)
    cmeta = torch.empty(16, dtype=torch.int32, device=dev)
    ws = torch.empty(int(lib.b2r_compact_workspace_bytes(B, NP)), dtype=torch.uint8, device=dev)
    _lib.check(lib.b2r_compact_plan(_ptr(idx), B, int(N), NP, NS, _ptr(cidx), _ptr(ccen),
                                    _ptr(cmeta), _ptr(ws), _ext._stream()), "compact_plan")
    _ext.LAUNCHES += 3
    return {"cidx": cidx, "ccen": ccen, "cmeta": cmeta}


def supported(mlp_module, xyz, features, idx, pooling="max"):
    """True when the fused kernels cover this block, forward AND backward (otherwise callers use
    the unfused path).  The shape rules live in the library: b2r_sa_layer_fwd_supported /
    b2r_sa_layer_bwd_supported apply exactly the checks the launches apply."""
    if pooling != "max" or not xyz.is_cuda:
        return False
    B, NP, NS = idx.shape
    blocks = list(mlp_module)
    if len(blocks) == 0:
        return False
    lib = _lib.lib()
    for i, blk in enumerate(blocks):
        if not hasattr(blk, "bn") or blk.conv.bias is not None:
            return False
        bn = blk.bn.bn
        if bn.momentum is None or not bn.track_running_stats or not bn.affine:
            return False
        cout, cin = blk.conv.out_channels, blk.conv.in_channels
        gather, top = (1 if i == 0 else 0), (1 if i == len(blocks) - 1 else 0)
        # (both answer for the layer's slice grid when it does not fit one launch)
        if not lib.b2r_sa_layer_fwd_supported(B, NP, NS, cin, cout, gather, top):
            return False
        if not lib.b2r_sa_layer_bwd_supported(B, NP, NS, cin, cout, gather, top):
            return False
    return True


def _layer_work(B, N, NP, NS, Cin, Cout, gather, pooled, backward):
    """ALGORITHMIC work of one fused layer launch as SURVEY.md 8(d) counts it, -> (bytes, flops):
    flops 2 * B*NP*NS * Cin * Cout of the PADDED computation (backward counted 2x forward;
    recomputation not credited, copies of a ball's first hit not discounted); bytes = this
    layer's share of the BLOCK-level compulsory traffic (features in + xyz + idx for the gather
    layer, the pooled output for the top layer, the weights for each; backward 2x) -- the
    inter-layer activations are not compulsory and are not counted."""
    M = B * NP * NS
    flops = 2.0 * M * Cin * Cout
    byts = 4.0 * Cin * Cout
    if gather:
        byts += B * (4.0 * (Cin - 3) * N + 12.0 * N + 4.0 * NP * NS)
    if pooled:
        byts += 4.0 * Cout * B * NP
    if backward:
        flops, byts = 2 * flops, 2 * byts
    return (byts, flops)


def sa_mlp_forward(xyz, new_xyz, feat_t, idx, radius, normalize_xyz, mlp_module, training,
                   want_point_major=True, save=None, sm_limit=0, plan=None):
    """Run the fused block.

    xyz (B,N,3), new_xyz (B,NP,3), feat_t (B,N,C) POINT-major features or None, idx (B,NP,NS).
    Returns (out_cm (B,Cl,NP), out_pm (B,NP,Cl) or None).  When `save` is a dict it receives what
    a backward pass needs (raw z per layer, BN mean/invstd/scale/shift, pooled max/min/arg).
    `plan`: a compact_plan(idx, N) -- the block then runs in its pad-free position space.
    """
    lib = _lib.lib()
    st = _ext._stream()
    dev = xyz.device
    B, N = xyz.shape[0], xyz.shape[1]
    NP, NS = idx.shape[1], idx.shape[2]
    M = B * NP * NS                  # positions of the padded computation (BatchNorm count)
    rows = M if plan is None else int(plan["cidx"].shape[0])   # rows of the z buffers
    blocks = list(mlp_module)
    L = len(blocks)
    z_prev = scale = shift = None
    zs, bn_saved, images = [], [], []
    # batch statistics of every layer: ONE zero-filled buffer (one memset instead of one per layer)
    stats_all = None
    if training:
        stats_all = step_arena.zeros(sum(2 * b.conv.out_channels for b in blocks), dtype=torch.float64,
                                device=dev)
    stats_off = 0
    zmax = zmin = amax = amin = None
    for i, blk in enumerate(blocks):
        conv, bn = blk.conv, blk.bn.bn
        Cin, Cout = conv.in_channels, conv.out_channels
        last = i == L - 1
        image = _take(conv.weight, "tf32")
        image = pack_layer(conv.weight, i == 0, "tf32", last) if image is None else _as_list(image)
        images.append(image)
        stats = None
        if training:
            stats = stats_all[stats_off:stats_off + 2 * Cout]
            stats_off += 2 * Cout
        d = _lib.SaLayer()
        d.B, d.N, d.NP, d.NS, d.Cin, d.Cout = B, N, NP, NS, Cin, Cout
        d.mode = 0 if i == 0 else 1
        d.epilogue = 1 if last else 0
        if i == 0:
            d.xyz, d.new_xyz, d.feat_t, d.idx = _ptr(xyz), _ptr(new_xyz), _ptr(feat_t), _ptr(idx)
            d.radius, d.normalize_xyz = float(radius), 1 if normalize_xyz else 0
        else:
            d.z_prev, d.scale_prev, d.shift_prev = _ptr(z_prev), _ptr(scale), _ptr(shift)
        d.sm_limit = int(sm_limit)
        if plan is not None:
            d.cidx, d.ccen, d.cmeta = _ptr(plan["cidx"]), _ptr(plan["ccen"]), _ptr(plan["cmeta"])
        z = None
        if last:
            zmax = torch.empty((B * NP, Cout), dtype=torch.float32, device=dev)
            zmin = torch.empty_like(zmax)
            amax = torch.empty((B * NP, Cout), dtype=torch.int32, device=dev)
            amin = torch.empty_like(amax)
            d.zmax, d.zmin, d.amax, d.amin = _ptr(zmax), _ptr(zmin), _ptr(amax), _ptr(amin)
        else:
            z = torch.empty((rows, Cout), dtype=torch.float32, device=dev)
            d.z = _ptr(z)
        grid = slice_grid(False, Cin, Cout, i == 0, last)
        with _ext._timed("sa_layer_fwd", _layer_work(B, N, NP, NS, Cin, Cout, i == 0, last, False)):
            for (co0, co_n, ci0, ci_n), img in zip(grid, image):
                # feature slices of one output slice: the first writes z, the others add to it,
                # and the last one takes the BatchNorm sums of the finished z
                d.co0, d.co_n, d.ci0, d.ci_n = co0, co_n, ci0, ci_n
                d.accumulate = 1 if ci0 > 0 else 0
                d.stats = _ptr(stats) if ci0 + ci_n >= Cin - 3 or ci_n == 0 else None
                d.w_image = _ptr(img)
                _lib.check(lib.b2r_sa_layer_fwd(ctypes.byref(d), st), "sa_layer_fwd")
            _ext.LAUNCHES += len(grid) - 1   # (_timed counts one)
        # BatchNorm scale / shift of THIS layer (applied by the next layer's prologue / finalize)
        if training:
            scale = torch.empty(Cout, dtype=torch.float32, device=dev)
            shift = torch.empty_like(scale)
            mean = torch.empty_like(scale)
            invstd = torch.empty_like(scale)
            pytorch_utils.bn_finalize(bn, stats, Cout, M, scale, shift, mean, invstd, st)
            _ext.LAUNCHES += 1
        else:
            invstd = torch.rsqrt(bn.running_var + bn.eps)
            mean = bn.running_mean
            scale = (bn.weight * invstd).contiguous()
            shift = (bn.bias - bn.running_mean * scale).contiguous()
        zs.append(z)
        bn_saved.append((mean, invstd, scale, shift))
        z_prev = z
    Cl = blocks[-1].conv.out_channels
    out_cm = torch.empty((B, Cl, NP), dtype=torch.float32, device=dev)
    out_pm = torch.empty((B, NP, Cl), dtype=torch.float32, device=dev) if want_point_major else None
    _lib.check(lib.b2r_pool_finalize(_ptr(zmax), _ptr(zmin), _ptr(scale), _ptr(shift), B, NP, Cl,
                                     _ptr(out_cm), _ptr(out_pm), st), "pool_finalize")
    _ext.LAUNCHES += 1
    if save is not None:
        save.update(zs=zs, bn=bn_saved, zmax=zmax, zmin=zmin, amax=amax, amin=amin, images=images,
                    plan=plan)
    return out_cm, out_pm


def pack_weight_bf16(weight, gather):
    """Conv weight (Cout,Cin,1,1) -> BF16 swizzled image for the backward kernel (serves the
    top-layer recomputation K-major and dgrad MN-major from the same bytes)."""
    Cout, Cin = weight.shape[0], weight.shape[1]
    w = weight.detach().reshape(Cout, Cin).contiguous()
    nbytes = _lib.lib().b2r_mlp_weight_bf16_image_bytes(Cout, Cin, 1 if gather else 0)
    image = torch.empty(nbytes // 2, dtype=torch.bfloat16, device=weight.device)
    _lib.check(_lib.lib().b2r_mlp_pack_weight_bf16(_ptr(w), Cout, Cin, 1 if gather else 0,
                                                   _ptr(image), _ext._stream()),
               "mlp_pack_weight_bf16")
    _ext.LAUNCHES += 1
    return image


def sa_mlp_backward(g_out_cm, xyz, new_xyz, feat_t, idx, radius, normalize_xyz, weights, gammas,
                    training, saved, need_feat, need_xyz, need_new_xyz, sm_limit=0, versioned=None,
                    g_out_pm=None):
    """Backward of sa_mlp_forward through csrc/mlp_bwd.cu.

    g_out_cm (B,Cl,NP) and/or g_out_pm (B,NP,Cl): gradient of the pooled output in either
    layout (summed when both are given; one of them may be None).  Returns
    (g_feat_t (B,N,C) | None, g_xyz (B,N,3) | None, g_new_xyz (B,NP,3) | None,
     [dW_i (Cout,Cin)], [dgamma_i], [dbeta_i]).
    """
    lib = _lib.lib()
    st = _ext._stream()
    dev = xyz.device
    assert g_out_cm is not None or g_out_pm is not None
    B, N = xyz.shape[0], xyz.shape[1]
    NP, NS = idx.shape[1], idx.shape[2]
    M = B * NP * NS
    plan = saved.get("plan")
    rows = M if plan is None else int(plan["cidx"].shape[0])
    L = len(weights)
    zs, bn, images = saved["zs"], saved["bn"], saved["images"]
    f32 = dict(dtype=torch.float32, device=dev)
    dWs, dgammas, dbetas = [None] * L, [None] * L, [None] * L
    tr = 1 if training else 0

    # --- pooled top layer: route the output gradient to its one sample per (centre, channel)
    top = L - 1
    Ct = weights[top].shape[0]
    mean, invstd, scale, shift = bn[top]
    # every accumulated output of the block from two zero-filled buffers (two memsets in total)
    stats_all = step_arena.zeros(sum(2 * w.shape[0] for w in weights), dtype=torch.float64, device=dev)
    dW_all = step_arena.zeros(sum(w.numel() for w in weights), **f32)
    s_off, w_off = [0], [0]
    for w in weights:
        s_off.append(s_off[-1] + 2 * w.shape[0])
        w_off.append(w_off[-1] + w.numel())
    stats = stats_all[s_off[top]:s_off[top + 1]]
    dysel = torch.empty((B * NP, Ct), **f32)
    asel = torch.empty((B * NP, Ct), dtype=torch.int32, device=dev)
    _lib.check(lib.b2r_pool_bwd_prep(_ptr(g_out_cm), _ptr(g_out_pm), _ptr(saved["zmax"]), _ptr(saved["zmin"]),
                                     _ptr(saved["amax"]), _ptr(saved["amin"]), _ptr(scale),
                                     _ptr(shift), B, NP, Ct, _ptr(dysel), _ptr(asel), _ptr(stats),
                                     st), "pool_bwd_prep")
    coef = [torch.empty(Ct, **f32) for _ in range(3)]
    dgammas[top], dbetas[top] = torch.empty(Ct, **f32), torch.empty(Ct, **f32)
    _lib.check(lib.b2r_bn_bwd_finalize(_ptr(stats), Ct, float(M), _ptr(gammas[top]), _ptr(mean),
                                       _ptr(invstd), tr, _ptr(coef[0]), _ptr(coef[1]),
                                       _ptr(coef[2]), None, None, None, _ptr(dgammas[top]),
                                       _ptr(dbetas[top]), st), "bn_bwd_finalize")
    _ext.LAUNCHES += 2

    g_feat_t = g_xyz = g_new_xyz = None
    gr = None
    for l in range(L - 1, -1, -1):
        Cout, Cin = weights[l].shape[0], weights[l].shape[1]
        b = _lib.SaLayerBwd()
        b.B, b.N, b.NP, b.NS, b.Cin, b.Cout = B, N, NP, NS, Cin, Cout
        b.mode = 0 if l == 0 else 1
        b.sm_limit = int(sm_limit)
        if plan is not None:
            b.cidx, b.ccen, b.cmeta = _ptr(plan["cidx"]), _ptr(plan["ccen"]), _ptr(plan["cmeta"])
        if l == top:   # z is recomputed inside the kernel from the layer's input
            b.dysel, b.asel = _ptr(dysel), _ptr(asel)
        else:
            b.gr, b.z = _ptr(gr), _ptr(zs[l])
        b.coef_a, b.coef_b, b.coef_c = _ptr(coef[0]), _ptr(coef[1]), _ptr(coef[2])
        dWs[l] = dW_all[w_off[l]:w_off[l + 1]].view(Cout, Cin)
        b.dW = _ptr(dWs[l])
        need_dgrad = True
        gr_prev = stats_prev = None
        if l == 0:
            b.xyz, b.new_xyz, b.feat_t, b.idx = _ptr(xyz), _ptr(new_xyz), _ptr(feat_t), _ptr(idx)
            b.radius, b.normalize_xyz = float(radius), 1 if normalize_xyz else 0
            if need_feat and feat_t is not None:
                g_feat_t = step_arena.zeros_like(feat_t)
                b.g_feat_t = _ptr(g_feat_t)
            if need_xyz:
                g_xyz = step_arena.zeros_like(xyz)
                b.g_xyz = _ptr(g_xyz)
            if need_new_xyz:
                g_new_xyz = step_arena.zeros_like(new_xyz)
                b.g_new_xyz = _ptr(g_new_xyz)
            need_dgrad = g_feat_t is not None or need_xyz or need_new_xyz
        else:
            b.z_prev, b.scale_prev, b.shift_prev = _ptr(zs[l - 1]), _ptr(bn[l - 1][2]), _ptr(bn[l - 1][3])
            gr_prev = torch.empty((rows, Cin), **f32)
            stats_prev = stats_all[s_off[l - 1]:s_off[l]]
            b.gr_prev, b.stats_prev = _ptr(gr_prev), _ptr(stats_prev)
        grid = slice_grid(True, Cin, Cout, l == 0, l == top)
        images = [None] * len(grid)
        if need_dgrad or l == top:
            images = _take(versioned[l], "bf16") if versioned is not None else None
            images = (pack_layer(weights[l], l == 0, "bf16", l == top) if images is None
                      else _as_list(images))
        with _ext._timed("sa_layer_bwd", _layer_work(B, N, NP, NS, Cin, Cout, l == 0, l == top, True)):
            for j, ((co0, co_n, ci0, ci_n), img) in enumerate(zip(grid, images)):
                # dense layers: every output slice after the first adds its share of the input
                # gradient (launch order fixes the summation order); gather layers scatter-add
                b.co0, b.co_n, b.ci0, b.ci_n = co0, co_n, ci0, ci_n
                b.accumulate = 1 if (l > 0 and j > 0) else 0
                b.w_image_bf16 = _ptr(img)
                _lib.check(lib.b2r_sa_layer_bwd(ctypes.byref(b), st), "sa_layer_bwd")
            _ext.LAUNCHES += len(grid) - 1
        if l > 0:
            mean, invstd, _, _ = bn[l - 1]
            coef = [torch.empty(Cin, **f32) for _ in range(3)]
            dgammas[l - 1], dbetas[l - 1] = torch.empty(Cin, **f32), torch.empty(Cin, **f32)
            _lib.check(lib.b2r_bn_bwd_finalize(_ptr(stats_prev), Cin, float(M), _ptr(gammas[l - 1]),
                                               _ptr(mean), _ptr(invstd), tr, _ptr(coef[0]),
                                               _ptr(coef[1]), _ptr(coef[2]), None, None, None,
                                               _ptr(dgammas[l - 1]), _ptr(dbetas[l - 1]), st),
                       "bn_bwd_finalize")
            _ext.LAUNCHES += 1
            gr = gr_prev
    return g_feat_t, g_xyz, g_new_xyz, dWs, dgammas, dbetas


class _FusedSABlock(torch.autograd.Function):
    """autograd node of the fused block: QueryAndGroup tail + SharedMLP + max-pool in; out come the
    (B,C,npoint) tensor of the reference and, on request, the same values POINT-major (B,npoint,C)
    -- the layout the next block gathers from.  Consecutive SA blocks hand activations (forward)
    and gradients (backward) to each other point-major, so neither a to_point_major launch nor a
    transposing copy sits between them.  Parameters are passed flat as (W0, gamma0, beta0, ...)."""

    @staticmethod
    def forward(ctx, xyz, new_xyz, features, features_pm, idx, radius, normalize_xyz, mlp_module,
                training, sm_limit, want_pm, plan, *params):
        if features_pm is not None:
            feat_t = features_pm                       # (B,N,C) from the previous block
        elif features is None:
            feat_t = None
        elif features.shape[1] == 1:                   # (B,1,N) and (B,N,1) are the same bytes
            feat_t = features.contiguous().reshape(features.shape[0], features.shape[2], 1)
        else:
            feat_t = to_point_major(features.contiguous())
        need = any(ctx.needs_input_grad)
        save = {} if need else None
        # sm_limit: one cap for both directions, or (forward cap, backward cap)
        fwd_limit, bwd_limit = sm_limit if isinstance(sm_limit, tuple) else (sm_limit, 0)
        out_cm, out_pm = sa_mlp_forward(xyz, new_xyz, feat_t, idx, radius, normalize_xyz,
                                        mlp_module, training, want_point_major=bool(want_pm),
                                        save=save, sm_limit=fwd_limit, plan=plan)
        ctx.set_materialize_grads(False)
        if need:
            ctx.saved = (xyz, new_xyz, feat_t, idx, float(radius), bool(normalize_xyz),
                         bool(training), save, params)
            ctx.bwd_sm_limit = int(bwd_limit)
            ctx.from_pm = features_pm is not None
        if want_pm:
            return out_cm, out_pm
        return out_cm, None

    @staticmethod
    def backward(ctx, g_cm, g_pm):
        xyz, new_xyz, feat_t, idx, radius, normalize_xyz, training, save, params = ctx.saved
        L = len(params) // 3
        n_in = 12
        if g_cm is None and g_pm is None:
            return (None,) * (n_in + 3 * L)
        weights = [params[3 * i].detach().reshape(params[3 * i].shape[0], -1) for i in range(L)]
        gammas = [params[3 * i + 1].detach() for i in range(L)]
        nig = ctx.needs_input_grad
        g_feat_t, g_xyz, g_new_xyz, dWs, dgs, dbs = sa_mlp_backward(
            g_cm.contiguous() if g_cm is not None else None, xyz, new_xyz, feat_t, idx, radius,
            normalize_xyz, weights, gammas, training, save, need_feat=nig[2] or nig[3],
            need_xyz=nig[0], need_new_xyz=nig[1], sm_limit=ctx.bwd_sm_limit,
            versioned=[params[3 * i] for i in range(L)],
            g_out_pm=g_pm.contiguous() if g_pm is not None else None)
        g_features = g_features_pm = None
        if g_feat_t is not None:
            if ctx.from_pm:
                g_features_pm = g_feat_t
            elif g_feat_t.shape[2] == 1:
                g_features = g_feat_t.reshape(g_feat_t.shape[0], 1, g_feat_t.shape[1])
            else:
                g_features = g_feat_t.transpose(1, 2).contiguous()
        out = [g_xyz, g_new_xyz, g_features, g_features_pm] + [None] * (n_in - 4)
        for i in range(L):
            out += [dWs[i].view_as(params[3 * i]), dgs[i], dbs[i]]
        return tuple(out)


def sa_block(xyz, new_xyz, features, idx, radius, normalize_xyz, mlp_module, training,
             sm_limit=0, features_pm=None, want_pm=False, plan=None):
    """Differentiable fused SA block: returns (new_features (B, mlp[-1], npoint), the same
    point-major (B, npoint, mlp[-1]) when `want_pm`, else None).  `features_pm` (B,N,C): the
    input features point-major (a previous block's second output) -- used instead of `features`.
    sm_limit > 0 caps the forward kernels' persistent grid (SMs left to a concurrent geometry
    stream); a tuple (forward cap, backward cap) also caps the backward kernels (the pipelined
    step, where the NEXT batch's geometry runs beside this batch's whole forward and backward).
    plan: compact_plan(idx, N) computed ahead of time (geometry pre-pass); by default one is built
    here when the block qualifies (compact_wanted)."""
    if plan is None and compact_wanted(idx.shape[2]):
        plan = compact_plan(idx, xyz.shape[1])
    params = []
    for blk in mlp_module:
        params += [blk.conv.weight, blk.bn.bn.weight, blk.bn.bn.bias]
    return _FusedSABlock.apply(xyz, new_xyz, features, features_pm, idx, radius, normalize_xyz,
                               mlp_module, training, sm_limit, bool(want_pm), plan, *params)


NUM_SMS = 148   # B200

# Set to False (or B2R_FUSED=0) to route PointnetSAModuleVotes through the unfused path
# (QueryAndGroup kernel + cuDNN SharedMLP + max_pool2d) -- used by the parity tests as the fp32
# comparison arm; it also switches the dense FP / voting / proposal layers off (dense_mlp.enabled).
ENABLED = os.environ.get("B2R_FUSED", "1") not in ("0", "")
