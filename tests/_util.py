"""Shared helpers for the parity tests."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    return dict(np.load(os.path.join(GOLDEN, name)))


def weight_checksum(module):
    return float(sum(p.detach().double().abs().sum().cpu() for p in module.parameters()))


def sub(t, n=4096):
    f = t.detach().reshape(-1)
    step = max(1, f.numel() // n)
    return f[::step].cpu().numpy().copy()


def rel_l2(got, want):
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    return float(np.linalg.norm(got - want) / max(np.linalg.norm(want), 1e-30))


def pattern_like(t):
    """Fixed pseudo-random loss weights in [-1, 1] (float64 sine hash -> fp32).

    NOT a linear ramp: a ramp is almost constant along the position axis of every channel, and
    BatchNorm's backward removes exactly that constant, so the surviving gradient is pure
    cancellation residue (measured: the fp32 CPU reference then disagrees with ITSELF by 6e-3
    between 1 and 8 threads)."""
    i = torch.arange(t.numel(), dtype=torch.float64)
    return torch.sin(i * 12.9898 + 0.5 * torch.cos(i * 0.618)).float().reshape(t.shape).to(t.device)


def round_tf32(t):
    """cvt.rna.tf32.f32 of a finite fp32 tensor (csrc/mlp_common.cuh to_tf32): the rounding every
    forward tensor-core operand of the product goes through."""
    bits = t.detach().float().contiguous().view(torch.int32)
    return ((bits + 0x1000) & ~0x1fff).view(torch.float32)


def round_bf16(t):
    """__float2bfloat16_rn: the rounding of the fused SA backward's operands."""
    return t.detach().float().bfloat16().float()


def emu_log(name, log="emulation_parity.log", **errs):
    """Tests that compare a kernel with its operand-rounding emulation record the measured error
    (file `log` in the run's output directory, when that directory exists) so the bounds can be
    audited."""
    d = os.path.join(os.path.dirname(GOLDEN[:-len("/golden")]), "gpurun_out")
    if os.path.isdir(d):
        with open(os.path.join(d, log), "a") as f:
            f.write(name + "  " + "  ".join("%s %.2e" % kv for kv in errs.items()) + "\n")
