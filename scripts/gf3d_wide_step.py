"""Time GroupFree3D's w2x backbone training step (width 2, depth 2, fp2 288) at 4 scenes x 50k
points: fwd + bwd + FlatAdamW, replayed by train_step.PipelinedTrainStep, with the fused SA /
dense layers and with fused_sa.ENABLED = False (QueryAndGroup + cuDNN), alternating in one process.

    python scripts/gf3d_wide_step.py [--out DIR] [--steps 20] [--rounds 3]

Step times: CUDA events around each replay, L2 overwritten (a 256 MB write) before every timed
replay.  Then one profiled replay per arm (torch.profiler, CUDA activities) gives kernel time per
layer class.  Prints the log; with --out DIR also writes DIR/gf3d_wide_step.log."""
import argparse
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from backtoreality_b200 import fused_sa, scenes  # noqa: E402
from backtoreality_b200.backbone_module import Pointnet2Backbone  # noqa: E402
from backtoreality_b200.flat_adam import FlatAdamW  # noqa: E402
from backtoreality_b200.train_step import CapturedTrainStep, PipelinedTrainStep  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "scripts"))
from optim_step_time import device_line  # noqa: E402

# kernel name -> layer class (first match wins)
CLASSES = [("sa_layer_fwd", "fused SA layer fwd"), ("sa_layer_bwd", "fused SA layer bwd"),
           ("thin", "fused SA thin layer"), ("dense", "dense FP layers"),
           ("pack_weight", "weight packing"), ("fps", "FPS"), ("ball_query", "ball query"),
           ("adam", "optimizer"), ("cudnn", "cuDNN conv / BN"), ("conv", "cuDNN conv / BN"),
           ("batch_norm", "cuDNN conv / BN"), ("bn_", "BatchNorm glue"), ("pool", "pool glue"),
           ("group", "grouping movers"), ("gemm", "GEMM (cuBLAS)"), ("sm90", "GEMM (cuBLAS)"),
           ("sm100", "GEMM (cuBLAS)")]


def classify(name):
    low = name.lower()
    for key, cls in CLASSES:
        if key in low:
            return cls
    return "other"


def make_arm(fused, batches):
    fused_sa.ENABLED = fused
    torch.manual_seed(0)
    net = Pointnet2Backbone(input_feature_dim=0, fp2_out=288, width=2, depth=2).cuda().train()
    opt = FlatAdamW(net.parameters(), lr=1e-4)

    def step(pc, geometry=None):
        for p in net.parameters():
            p.grad = None
        ep = net(pc, geometry=geometry)
        loss = (ep["fp2_features"] ** 2).mean()
        loss.backward()
        opt.step()
        return loss.detach()
    try:
        return PipelinedTrainStep(net, step, batches[0], warmup=3, fps_cluster=10,
                                  start_after_level=0), "PipelinedTrainStep"
    except Exception as e:   # reported in the log, never silently
        torch.cuda.synchronize()
        return CapturedTrainStep(step, batches[0], warmup=3), "CapturedTrainStep (pipelined: %s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="", help="directory for gf3d_wide_step.log (default: print only)")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--npoints", type=int, default=50000)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda")
    lines = [device_line(dev),
             "w2x GroupFree3D backbone (width 2, depth 2, fp2 288), %d scenes x %d points, "
             "fwd + bwd + FlatAdamW, PipelinedTrainStep; L2 overwritten before every timed replay"
             % (a.batch, a.npoints)]
    batches = [torch.from_numpy(scenes.batch(900 + a.batch * i, a.batch, a.npoints, C=0, kind="room",
                                             dup=0.2)).to(dev) for i in range(4)]
    arms = {}
    for name, fused in (("fused", True), ("unfused", False)):
        t0 = time.time()
        arms[name], how = make_arm(fused, batches)
        torch.cuda.synchronize()
        lines.append("%s arm: %s, captured in %.1f s" % (name, how, time.time() - t0))
    fused_sa.ENABLED = True
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)   # 256 MB > 126 MB L2
    times = {k: [] for k in arms}
    losses = {k: [] for k in arms}
    i = 0
    for r in range(a.rounds):
        for name, pipe in arms.items():
            for _ in range(a.steps):
                flush.fill_(float(i))
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                loss = pipe(batches[i % len(batches)])
                e.record()
                torch.cuda.synchronize()
                times[name].append(s.elapsed_time(e))
                losses[name].append(float(loss))
                i += 1
    for name in arms:
        t = sorted(times[name])
        lines.append("%-8s step: median %.3f ms, min %.3f, max %.3f over %d replays (%d rounds "
                     "alternating)" % (name, t[len(t) // 2], t[0], t[-1], len(t), a.rounds))
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    lines.append("unfused / fused: %.2fx" % (med["unfused"] / med["fused"]))
    lines.append("first losses fused %s | unfused %s" % (losses["fused"][:2], losses["unfused"][:2]))

    from torch.profiler import ProfilerActivity, profile
    for name, pipe in arms.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                pipe(batches[0])
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            us = getattr(ev, "device_time_total", None)
            if us is None:
                us = ev.cuda_time_total
            if us <= 0:
                continue
            cls = classify(ev.key)
            per[cls] = per.get(cls, 0.0) + us / 3.0
        lines.append("%s arm: kernel time per step by layer class (torch.profiler, 3 replays)" % name)
        for cls, us in sorted(per.items(), key=lambda kv: -kv[1]):
            lines.append("    %-24s %9.1f us" % (cls, us))
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "gf3d_wide_step.log"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
