"""Host-side checks of the flat Adam / AdamW optimizer and its C entry points (no GPU needed):
the ctypes mirror of b2r_adam_desc, argument validation before any CUDA call, and the options
FlatAdam refuses."""
import ctypes

import pytest
import torch


def test_adam_desc_mirror_matches_the_library():
    from backtoreality_b200 import _lib
    l = _lib.lib()
    assert l.b2r_struct_bytes(4) == ctypes.sizeof(_lib.AdamDesc)
    assert ctypes.sizeof(_lib.AdamGroup) == 24


def test_new_entries_reject_bad_arguments_before_any_cuda_call():
    from backtoreality_b200 import _lib
    l = _lib.lib()
    assert l.b2r_flat_grad_norm_workspace_bytes(-1) == -1
    assert l.b2r_flat_grad_norm_workspace_bytes(0) > 0
    # the grid, and so the workspace, depends on n only and is bounded
    assert l.b2r_flat_grad_norm_workspace_bytes(1 << 30) == l.b2r_flat_grad_norm_workspace_bytes(1 << 28)
    ws = ctypes.c_void_p(16)      # never dereferenced: validation fails first
    assert l.b2r_flat_grad_norm(None, 8, 1.0, 1.0, ws, ws, ws, None) == -1
    assert l.b2r_flat_grad_norm(ws, -4, 1.0, 1.0, ws, ws, ws, None) == -1
    assert l.b2r_flat_grad_norm(ws, 8, 1.0, 1.0, None, ws, ws, None) == -1
    assert l.b2r_flat_grad_norm(ws, 8, 1.0, 1.0, ws, None, ws, None) == -1
    assert l.b2r_flat_grad_norm(ws, 8, 1.0, 1.0, ws, ws, None, None) == -1
    assert b"b2r_flat_grad_norm" in l.b2r_last_error()
    assert l.b2r_adam_flat_step_groups(None, None) == -1
    d = _lib.AdamDesc(params=16, grads=16, exp_avg=16, exp_avg_sq=16, n=-1, state=16, groups=16,
                      n_groups=1, beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=1.0)
    assert l.b2r_adam_flat_step_groups(ctypes.byref(d), None) == -1
    d.n = 8
    d.groups = None
    assert l.b2r_adam_flat_step_groups(ctypes.byref(d), None) == -1
    d.groups = 16
    for bad in (0, -1, _lib.ADAM_MAX_GROUPS + 1):
        d.n_groups = bad
        assert l.b2r_adam_flat_step_groups(ctypes.byref(d), None) == -1
    d.n_groups = 1
    d.params = 20                 # not 16-byte aligned
    assert l.b2r_adam_flat_step_groups(ctypes.byref(d), None) == -1
    assert b"aligned" in l.b2r_last_error()


def _cpu_params():
    return [torch.nn.Parameter(torch.zeros(4)), torch.nn.Parameter(torch.zeros(3))]


@pytest.mark.parametrize("kwargs, match", [
    (dict(amsgrad=True), "amsgrad"),
    (dict(maximize=True), "maximize"),
    (dict(max_grad_norm=1.0, norm_type=1.0), "norm_type=2"),
    (dict(max_grad_norm=1.0, norm_type=float("inf")), "norm_type=2"),
])
def test_unsupported_options_raise(kwargs, match):
    from backtoreality_b200.flat_adam import FlatAdam, FlatAdamW
    for cls in (FlatAdam, FlatAdamW):
        with pytest.raises(ValueError, match=match):
            cls(_cpu_params(), **kwargs)


@pytest.mark.parametrize("group_opts, match", [
    ({"betas": (0.8, 0.999)}, "same betas and eps"),
    ({"eps": 1e-6}, "same betas and eps"),
    ({"amsgrad": True}, "amsgrad"),
    ({"decoupled_weight_decay": True}, "decoupled_weight_decay"),
])
def test_unsupported_per_group_options_raise(group_opts, match):
    from backtoreality_b200.flat_adam import FlatAdam
    a, b = _cpu_params()
    with pytest.raises(ValueError, match=match):
        FlatAdam([{"params": [a]}, {"params": [b], **group_opts}])


def test_flat_adam_is_a_torch_optimizer_and_refuses_cpu_groups():
    from backtoreality_b200.flat_adam import FlatAdam, FlatAdamW
    assert issubclass(FlatAdam, torch.optim.Optimizer) and issubclass(FlatAdamW, FlatAdam)
    with pytest.raises(ValueError, match="no parameters"):
        FlatAdamW([])
    a, b = _cpu_params()
    with pytest.raises(RuntimeError, match="CUDA only"):
        FlatAdamW([{"params": [a]}, {"params": [b], "lr": 1e-4}])
