"""CUDA-event time of the graph-replayed optimizer step alone (no forward / backward).

Variants over the same parameter set and gradients:
  flat_adam            flat_adam.FlatAdam (Adam, one group): pack + one update kernel
  flat_adamw_2g        flat_adam.FlatAdamW, two groups, no clipping
  flat_adamw_2g_clip   the same with max_grad_norm: pack + norm (2 launches) + update
  torch_adamw          torch.optim.AdamW(fused=True, capturable=True), two groups
  torch_adamw_clip     the same after clip_grad_norm_(foreach=True)
Sizes: the VoteNet parameter set (77 tensors, 956,408 parameters; parameters, gradients and both
moments, ~19 MB, stay in the 126 MB L2 between replays) and 14.5 M parameters (GF3D's
GroupFreeDetector, 14,514,573 parameters = 58 MB of gradient, SURVEY.md section 2b D2: the
VoteNet shapes repeated to that size; ~290 MB per step, streamed from HBM).  Each variant is
captured into its own CUDA graph; the graphs are replayed back to back, `--reps` replays between
two events, `--rounds` rounds interleaved over the variants.  Prints the device name and power
limit first.

    python scripts/optim_step_time.py [--reps 200] [--rounds 7]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from backtoreality_b200.flat_adam import FlatAdam, FlatAdamW  # noqa: E402

GF3D_PARAMS = 14_514_573


def device_line(dev):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = "nvidia-smi unavailable (%s)" % e
    return "device: %s | nvidia-smi name, power limit, max SM clock: %s" % (torch.cuda.get_device_name(dev), q)


def votenet_shapes():
    from backtoreality_b200.votenet import VoteNet
    net = VoteNet(22, 1, 22, np.ones((22, 3), np.float32), input_feature_dim=1, num_proposal=256,
                  vote_factor=1, sampling="vote_fps")
    return [tuple(p.shape) for p in net.parameters()]


def gf3d_shapes(base):
    shapes, n = [], 0
    per = sum(int(np.prod(s)) for s in base)
    while n + per <= GF3D_PARAMS:
        shapes += base
        n += per
    shapes.append((GF3D_PARAMS - n,))
    return shapes


def build(variant, shapes, dev):
    gen = torch.Generator(device=dev).manual_seed(0)
    params = [torch.nn.Parameter(torch.randn(s, device=dev, generator=gen) * 0.1) for s in shapes]
    grads = [torch.randn(s, device=dev, generator=gen) * 1e-3 for s in shapes]
    half = len(params) // 2
    groups = [{"params": params[:half]}, {"params": params[half:], "lr": 1e-4, "weight_decay": 0.0}]
    if variant == "flat_adam":
        opt = FlatAdam(params, lr=1e-3)
    elif variant.startswith("flat_adamw_2g"):
        opt = FlatAdamW(groups, lr=1e-3, weight_decay=5e-4,
                        max_grad_norm=0.1 if variant.endswith("clip") else None)
    else:
        opt = torch.optim.AdamW(groups, lr=1e-3, weight_decay=5e-4, fused=True, capturable=True)
        for p, g in zip(params, grads):
            p.grad = g
    clip = variant == "torch_adamw_clip"

    def step():
        if variant.startswith("flat"):
            opt.step(grads)
        else:
            if clip:
                torch.nn.utils.clip_grad_norm_(params, 0.1, foreach=True)
            opt.step()

    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    return graph, (params, grads, opt)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=7)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "optim_step_time.py measures on the GPU"
    dev = torch.device("cuda", 0)
    print(device_line(dev), flush=True)
    vn = votenet_shapes()
    sizes = [("votenet", vn), ("gf3d_14.5M", gf3d_shapes(vn))]
    variants = ["flat_adam", "flat_adamw_2g", "flat_adamw_2g_clip", "torch_adamw", "torch_adamw_clip"]
    print("reps per timing %d, rounds %d (interleaved); us per optimizer step: median [min, max] of rounds"
          % (a.reps, a.rounds), flush=True)
    for name, shapes in sizes:
        n = sum(int(np.prod(s)) for s in shapes)
        graphs = {v: build(v, shapes, dev) for v in variants}
        for g, _ in graphs.values():       # warm: first replays upload the graphs
            for _ in range(5):
                g.replay()
        torch.cuda.synchronize()
        times = {v: [] for v in variants}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(a.rounds):
            for v in variants:
                g = graphs[v][0]
                e0.record()
                for _ in range(a.reps):
                    g.replay()
                e1.record()
                e1.synchronize()
                times[v].append(e0.elapsed_time(e1) * 1e3 / a.reps)
        print("%s: %d tensors, %d parameters (%.1f MB fp32 per buffer)" % (name, len(shapes), n, n * 4 / 1e6),
              flush=True)
        for v in variants:
            t = sorted(times[v])
            print("  %-20s %8.2f us  [%.2f, %.2f]" % (v, t[len(t) // 2], t[0], t[-1]), flush=True)
        del graphs
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
