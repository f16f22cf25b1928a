"""flat_adam.FlatAdam / FlatAdamW against torch.optim.Adam / AdamW and clip_grad_norm_ on the same
GPU: parameter groups, decoupled weight decay, global gradient-norm clipping, learning-rate
schedules driving a CUDA-graph-replayed step, and checkpoints in torch's state_dict format.
Parameters are held to the bounds of test_modules_gpu.py::test_flat_adam_matches_torch_adam."""
import ctypes

import pytest
import torch

from backtoreality_b200 import _lib
from backtoreality_b200.flat_adam import FlatAdam, FlatAdamW

pytestmark = pytest.mark.gpu

RTOL, ATOL = 2e-5, 2e-6
# odd sizes: every parameter and every group is padded to 4 floats in the flat buffer
SHAPES = [(64, 33), (7,), (3, 5), (128,), (9, 4, 3), (31,)]
GROUPS = [dict(idx=[0, 1], lr=1e-2, weight_decay=0.05), dict(idx=[2, 3], lr=3e-3, weight_decay=0.0),
          dict(idx=[4, 5], lr=1e-3, weight_decay=0.01)]


def _make(cuda, seed=3):
    torch.manual_seed(seed)
    ref = [torch.nn.Parameter(torch.randn(s, device=cuda)) for s in SHAPES]
    ours = [torch.nn.Parameter(p.detach().clone()) for p in ref]
    return ref, ours


def _groups(params, groups):
    return [{"params": [params[i] for i in g["idx"]], "lr": g["lr"], "weight_decay": g["weight_decay"]}
            for g in groups]


def _order(groups):
    return [i for g in groups for i in g["idx"]]


def _close(ours, ref):
    for a, b in zip(ours, ref):
        torch.testing.assert_close(a, b, rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("kind", ["adamw", "adam_decoupled", "adam_l2"])
@pytest.mark.parametrize("n_groups", [2, 3])
def test_groups_match_torch(cuda, kind, n_groups):
    groups = GROUPS[:n_groups]
    ref, ours = _make(cuda)
    if kind == "adamw":
        o_ref = torch.optim.AdamW(_groups(ref, groups), lr=5e-3)
        o_b2r = FlatAdamW(_groups(ours, groups), lr=5e-3)
    else:
        dec = kind == "adam_decoupled"
        o_ref = torch.optim.Adam(_groups(ref, groups), lr=5e-3, decoupled_weight_decay=dec)
        o_b2r = FlatAdam(_groups(ours, groups), lr=5e-3, decoupled_weight_decay=dec)
    order = _order(groups)
    for it in range(12):
        grads = [torch.randn_like(p) * (it + 1) for p in ref]
        for p, g in zip(ref, grads):
            p.grad = g.clone()
        o_ref.step()
        o_b2r.step([grads[i] for i in order])
        _close(ours, ref)


def _scaled_grads(ref, target_norm, gen):
    g = [torch.randn(p.shape, device=p.device, generator=gen) for p in ref]
    total = torch.linalg.vector_norm(torch.stack([torch.linalg.vector_norm(x) for x in g]))
    return [x * (target_norm / total) for x in g]


def test_clipping_matches_clip_grad_norm(cuda):
    ref, ours = _make(cuda)
    max_norm = 1.0
    o_ref = torch.optim.AdamW(_groups(ref, GROUPS[:2]), lr=5e-3)
    o_b2r = FlatAdamW(_groups(ours, GROUPS[:2]), lr=5e-3, max_grad_norm=max_norm)
    order = _order(GROUPS[:2])
    used = [ref[i] for i in order]
    gen = torch.Generator(device=cuda).manual_seed(5)
    clipped = unclipped = 0
    for it, target in enumerate([0.3, 4.0, 0.9, 25.0, 0.05, 1.7, 0.6, 3.0, 0.2, 9.0, 0.99, 1.01]):
        grads = _scaled_grads(used, target, gen)
        for p, g in zip(used, grads):
            p.grad = g.clone()
        for p, g in zip([ours[i] for i in order], grads):
            p.grad = g.clone()
        total = torch.nn.utils.clip_grad_norm_(used, max_norm)
        o_ref.step()
        o_b2r.step()                     # reads p.grad
        # p.grad is not modified by the clipping
        for i, g in zip(order, grads):
            assert torch.equal(ours[i].grad, g)
        got = float(o_b2r.last_grad_norm)
        assert o_b2r.last_grad_norm.dim() == 0 and o_b2r.last_grad_norm.is_cuda
        assert abs(got - float(total)) <= 1e-5 * float(total), (it, got, float(total))
        clipped += float(total) > max_norm
        unclipped += float(total) <= max_norm
        _close(ours, ref)
    assert clipped >= 3 and unclipped >= 3


def test_grad_norm_kernel_against_fp64_and_nonfinite(cuda):
    """b2r_flat_grad_norm on its own: sizes with a scalar tail and a multi-block grid, grad_scale,
    and torch's handling of infinite / NaN norms."""
    l = _lib.lib()
    out = torch.zeros(2, device=cuda)

    def run(g, scale, max_norm):
        ws = torch.empty(int(l.b2r_flat_grad_norm_workspace_bytes(g.numel())), dtype=torch.uint8, device=cuda)
        _lib.check(l.b2r_flat_grad_norm(g.data_ptr(), g.numel(), scale, max_norm, ws.data_ptr(),
                                        out.data_ptr(), out[1:].data_ptr(),
                                        torch.cuda.current_stream().cuda_stream), "flat_grad_norm")
        return float(out[0]), float(out[1])

    gen = torch.Generator(device=cuda).manual_seed(7)
    for n in (1, 3, 4, 1001, 1_000_003, 14_500_001):
        g = torch.randn(n, device=cuda, generator=gen)
        norm, coef = run(g, 0.5, 2.0)
        want = float(torch.linalg.vector_norm((g * 0.5).double()))
        assert abs(norm - want) <= 1e-6 * want, (n, norm, want)
        # clip_grad_norm_'s expression on the fp32 norm
        want_coef = torch.clamp(2.0 / (torch.tensor(norm) + 1e-6), max=1.0)
        assert coef == float(want_coef)
    g = torch.ones(1000, device=cuda)
    g[17] = float("inf")
    norm, coef = run(g, 1.0, 1.0)
    assert norm == float("inf") and coef == 0.0
    g[17] = float("nan")
    norm, coef = run(g, 1.0, 1.0)
    assert norm != norm and coef != coef


def test_norm_is_bit_identical_over_replays(cuda):
    torch.manual_seed(11)
    params = [torch.nn.Parameter(torch.randn(1_500_000, device=cuda)),
              torch.nn.Parameter(torch.randn(777, device=cuda))]
    opt = FlatAdamW([{"params": params[:1]}, {"params": params[1:], "lr": 1e-4}], lr=1e-3,
                    max_grad_norm=0.1)
    static = [torch.randn_like(p) for p in params]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        opt.step(static)
    torch.cuda.current_stream().wait_stream(s)
    first = opt.last_grad_norm.clone()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        opt.step(static)
    norms = []
    for _ in range(8):
        graph.replay()
        norms.append(opt.last_grad_norm.clone())
    torch.cuda.synchronize()
    for x in norms:
        assert torch.equal(x.view(torch.int32), first.view(torch.int32))


def _lambda_sched(opt):
    return torch.optim.lr_scheduler.LambdaLR(opt, [lambda e: min(1.0, (e + 1) / 6),
                                                   lambda e: min(1.0, (e + 1) / 3)])


def _multistep_sched(opt):
    return torch.optim.lr_scheduler.MultiStepLR(opt, milestones=[5, 12, 17], gamma=0.3)


@pytest.mark.parametrize("make_sched", [_lambda_sched, _multistep_sched], ids=["lambda", "multistep"])
def test_captured_step_follows_lr_schedule(cuda, make_sched):
    """One captured step replayed 20 times while a torch scheduler changes the rates between
    replays (scheduler.step(); opt.sync_hparams()) must equal the same schedule run eagerly with
    torch.optim.AdamW + clip_grad_norm_."""
    ref, ours = _make(cuda, seed=5)
    groups = GROUPS[:2]
    order = _order(groups)
    used_ref, used_ours = [ref[i] for i in order], [ours[i] for i in order]
    o_ref = torch.optim.AdamW(_groups(ref, groups))
    o_b2r = FlatAdamW(_groups(ours, groups), max_grad_norm=0.5)
    s_ref, s_b2r = make_sched(o_ref), make_sched(o_b2r)
    gen = torch.Generator(device=cuda).manual_seed(9)
    targets = [0.2, 3.0, 0.4, 1.5, 0.1, 6.0, 0.45, 0.8, 2.0, 0.3, 5.0]
    grads = [_scaled_grads(used_ref, targets[k % len(targets)], gen) for k in range(21)]
    lrs = []

    def ref_step(k):
        for p, g in zip(used_ref, grads[k]):
            p.grad = g.clone()
        torch.nn.utils.clip_grad_norm_(used_ref, 0.5)
        o_ref.step()

    static = [torch.zeros_like(p) for p in used_ours]
    # step 0: eager warm-up on a side stream (as torch.cuda.graph requires), then capture
    for x, g in zip(static, grads[0]):
        x.copy_(g)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        o_b2r.step(static)
    torch.cuda.current_stream().wait_stream(side)
    ref_step(0)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        o_b2r.step(static)
    for k in range(1, 21):
        s_ref.step()
        s_b2r.step()
        o_b2r.sync_hparams()
        lrs.append(tuple(g["lr"] for g in o_b2r.param_groups))
        assert lrs[-1] == tuple(g["lr"] for g in o_ref.param_groups)
        for x, g in zip(static, grads[k]):
            x.copy_(g)
        graph.replay()
        ref_step(k)
        _close(ours, ref)
    assert len(set(lrs)) >= 3          # the schedule did change the rates between replays


def test_by_value_entry_runs_the_same_kernel(cuda):
    """b2r_adam_flat_step (hyperparameters by value) and b2r_adam_flat_step_groups with one group,
    L2 decay and no clipping compute bit-identical results, and both match torch.optim.Adam."""
    l = _lib.lib()
    n = 100_003
    torch.manual_seed(2)
    p0 = torch.randn(n + 1, device=cuda)[:n].clone()
    bufs = {k: [p0.clone(), torch.zeros(n, device=cuda), torch.zeros(n, device=cuda),
                torch.zeros(l.b2r_adam_state_bytes(), dtype=torch.uint8, device=cuda)] for k in ("v", "t")}
    table = (_lib.AdamGroup * 1)(_lib.AdamGroup(0, n, 1e-2, 0.02))
    dtab = torch.frombuffer(bytearray(table), dtype=torch.uint8).to(cuda)
    ref = torch.nn.Parameter(p0.clone())
    o_ref = torch.optim.Adam([ref], lr=1e-2, weight_decay=0.02)
    stream = torch.cuda.current_stream().cuda_stream
    for it in range(5):
        g = torch.randn(n, device=cuda)
        p, m, v, st = bufs["v"]
        _lib.check(l.b2r_adam_flat_step(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), n,
                                        st.data_ptr(), 1e-2, 0.9, 0.999, 1e-8, 0.02, 0.5, stream), "by value")
        p, m, v, st = bufs["t"]
        d = _lib.AdamDesc(params=p.data_ptr(), grads=g.data_ptr(), exp_avg=m.data_ptr(),
                          exp_avg_sq=v.data_ptr(), n=n, state=st.data_ptr(), groups=dtab.data_ptr(),
                          n_groups=1, beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=0.5, decoupled=0)
        _lib.check(l.b2r_adam_flat_step_groups(ctypes.byref(d), stream), "groups")
        ref.grad = g * 0.5
        o_ref.step()
        for a, b in zip(bufs["v"][:3], bufs["t"][:3]):
            assert torch.equal(a, b)
        torch.testing.assert_close(bufs["v"][0], ref.detach(), rtol=RTOL, atol=ATOL)


def _train(opt, params, gen, steps):
    for _ in range(steps):
        for p in params:
            p.grad = torch.randn(p.shape, device=p.device, generator=gen)
        opt.step()


def test_state_dict_round_trips_with_torch(cuda):
    groups = GROUPS[:2]
    order = _order(groups)
    # torch AdamW -> FlatAdamW
    ref, _ = _make(cuda, seed=21)
    used = [ref[i] for i in order]
    o_ref = torch.optim.AdamW(_groups(ref, groups), lr=5e-3)
    gen = torch.Generator(device=cuda).manual_seed(1)
    _train(o_ref, used, gen, 3)
    sd = o_ref.state_dict()
    ours = [torch.nn.Parameter(p.detach().clone()) for p in ref]
    o_b2r = FlatAdamW(_groups(ours, groups), lr=1.0, weight_decay=0.5)    # overwritten by the load
    o_b2r.load_state_dict(sd)
    assert [g["lr"] for g in o_b2r.param_groups] == [g["lr"] for g in groups]
    # the exported state is what torch itself holds
    back = o_b2r.torch_state_dict()
    assert back["param_groups"] == sd["param_groups"]
    assert sorted(back["state"]) == sorted(sd["state"])
    for i, st in sd["state"].items():
        assert back["state"][i]["step"].device == st["step"].device
        assert float(back["state"][i]["step"]) == float(st["step"])
        torch.testing.assert_close(back["state"][i]["exp_avg"], st["exp_avg"], rtol=0, atol=0)
        torch.testing.assert_close(back["state"][i]["exp_avg_sq"], st["exp_avg_sq"], rtol=0, atol=0)
    used_ours = [ours[i] for i in order]
    for _ in range(5):
        grads = [torch.randn_like(p) for p in used]
        for p, q, g in zip(used, used_ours, grads):
            p.grad, q.grad = g.clone(), g.clone()
        o_ref.step()
        o_b2r.step()
        _close(ours, ref)

    # FlatAdamW -> torch AdamW
    ref, ours = _make(cuda, seed=22)
    used, used_ours = [ref[i] for i in order], [ours[i] for i in order]
    o_b2r = FlatAdamW(_groups(ours, groups), lr=5e-3, max_grad_norm=2.0)
    assert o_b2r.torch_state_dict()["state"] == {}        # torch has no state before the first step
    gen = torch.Generator(device=cuda).manual_seed(2)
    _train(o_b2r, used_ours, gen, 4)
    sd = o_b2r.torch_state_dict()
    assert all(float(s["step"]) == 4.0 for s in sd["state"].values())
    for p, q in zip(ref, ours):
        p.data.copy_(q.detach())
    o_ref = torch.optim.AdamW(_groups(ref, groups), lr=1.0, weight_decay=0.5)
    o_ref.load_state_dict(sd)
    assert o_ref.state_dict()["param_groups"] == sd["param_groups"]
    for _ in range(5):
        grads = [torch.randn_like(p) * 0.1 for p in used]
        for p, q, g in zip(used, used_ours, grads):
            p.grad, q.grad = g.clone(), g.clone()
        torch.nn.utils.clip_grad_norm_(used, 2.0)
        o_ref.step()
        o_b2r.step()
        _close(ours, ref)

    # one device step counter: differing per-parameter steps are refused
    sd["state"][0]["step"] = torch.tensor(3.0)
    with pytest.raises(ValueError, match="same step count"):
        o_b2r.load_state_dict(sd)
