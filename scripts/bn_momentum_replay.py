"""What a BatchNorm momentum change costs in a replayed training step, and what attaching costs.

  change   the benched VoteNet step (8 scenes x 40000 points, 22 classes, 256 proposals,
           PipelinedTrainStep as bench.py runs it, FlatAdam): host wall time of one momentum change
           done two ways, each ended by a device synchronise:
             sync      bnm.step(epoch) on an attached model (pytorch_utils.sync_bn_momentum):
                       the scheduler writes the device table, the graph is kept
             recapture bnm.step(epoch) on an unattached model, then pipe.recapture() with
                       snapshot=[net, opt] and pipe.prime(batch)
  br       the BR step (VoteNet_DA, 8 + 8 scenes x 40000 points, PipelinedTrainStep with two plans
           per batch as bench.py --workload br runs it): CUDA-event time per replayed step of an
           unattached and an attached model, alternated `--rounds` times, `--steps` replays each.
           Attached, the discriminators' BatchNorm1d update their running statistics from the
           table with torch.var_mean + lerp_ instead of inside cuDNN's kernel.

    python scripts/bn_momentum_replay.py [--steps 30] [--rounds 3] [--changes 10]
"""
import argparse
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from bench import workload_loss  # noqa: E402
from optim_step_time import device_line  # noqa: E402
from backtoreality_b200 import scenes  # noqa: E402
from backtoreality_b200.flat_adam import FlatAdam  # noqa: E402
from backtoreality_b200.pytorch_utils import BNMomentumScheduler, sync_bn_momentum  # noqa: E402
from backtoreality_b200.train_step import PipelinedTrainStep  # noqa: E402
from backtoreality_b200.votenet import VoteNet, VoteNet_DA  # noqa: E402


def bn_lambda(epoch):
    return max(0.5 * 0.5 ** (epoch // 20), 0.001)


def build(dev, workload, attach, first):
    """bench.py's model, optimizer and pipelined step for `workload` ("votenet" or "br")"""
    torch.manual_seed(0)
    net = (VoteNet_DA if workload == "br" else VoteNet)(
        22, 1, 22, np.ones((22, 3), np.float32), input_feature_dim=1, num_proposal=256,
        vote_factor=1, sampling="vote_fps").to(dev).train()
    params = list(net.parameters())
    opt = FlatAdam(params, lr=1e-3)
    bnm = BNMomentumScheduler(net, bn_lambda)
    if attach:
        sync_bn_momentum(net)

    def step(pc, geometry=None):
        for p in params:
            p.grad = None
        loss = workload_loss(workload, net, pc, geometry)
        loss.backward()
        opt.step([p.grad for p in params])
        return loss

    start = None if workload == "br" else 1          # bench.py's --prepass-after defaults
    B = first.shape[0]
    caps, head_cap = PipelinedTrainStep.default_caps(B, 4, start)
    net.pnet.vote_aggregation.sm_limit = head_cap
    pipe = PipelinedTrainStep(net.backbone_net, step, first, fps_cluster=4, sm_caps=caps,
                              start_after_level=start, snapshot=[net, opt],
                              plan_splits=2 if workload == "br" else 1)
    return net, bnm, pipe


def batches(dev, n, count=3):
    return [torch.from_numpy(scenes.batch(n * i, n, 40000, C=1, kind="room", dup=0.2)).to(dev)
            for i in range(count)]


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def momentum_change(dev, a):
    data = batches(dev, 8)
    print("== change: benched VoteNet step (8 x 40000), PipelinedTrainStep + FlatAdam", flush=True)
    res = {}
    for attach in (True, False):
        net, bnm, pipe = build(dev, "votenet", attach, data[0])
        for i in range(3):
            pipe(data[(i + 1) % 3])
        times = []
        n = a.changes if attach else max(a.changes // 3, 2)
        for i in range(n):
            epoch = 20 * (i + 1)                     # a new momentum every time

            def change():
                bnm.step(epoch)
                if not attach:
                    pipe.recapture()
                    pipe.prime(data[0])
            times.append(wall(change))
            pipe(data[1])                            # the graph still runs
        torch.cuda.synchronize()
        res[attach] = times
        print("%-9s %d changes: median %.3f ms, min %.3f, max %.3f" % (
            "sync" if attach else "recapture", n, np.median(times), min(times), max(times)), flush=True)
        del net, bnm, pipe
        torch.cuda.empty_cache()
    print("recapture / sync (medians): %.0fx" % (np.median(res[False]) / np.median(res[True])))


def br_step(dev, a):
    data = batches(dev, 16)
    print("== br: VoteNet_DA step (8 + 8 scenes x 40000), PipelinedTrainStep, plan_splits=2", flush=True)
    arms = {}
    for attach in (False, True):
        arms[attach] = build(dev, "br", attach, data[0])
    for attach, (_, _, pipe) in arms.items():
        for i in range(3):
            pipe(data[(i + 1) % 3])
    ms = {False: [], True: []}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(a.rounds):
        for attach in (False, True):
            pipe = arms[attach][2]
            torch.cuda.synchronize()
            e0.record()
            for i in range(a.steps):
                pipe(data[(i + 1) % 3])
            e1.record()
            torch.cuda.synchronize()
            ms[attach].append(e0.elapsed_time(e1) / a.steps)
            print("round %d %-10s %.4f ms/step" % (r + 1, "attached" if attach else "unattached",
                                                  ms[attach][-1]), flush=True)
    for attach in (False, True):
        print("%-10s median %.4f ms/step over %d rounds of %d replays" % (
            "attached" if attach else "unattached", np.median(ms[attach]), a.rounds, a.steps))
    print("attached - unattached (medians): %+.4f ms/step" % (np.median(ms[True]) - np.median(ms[False])))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--changes", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bn_momentum_replay.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    print(device_line(dev), flush=True)
    momentum_change(dev, a)
    br_step(dev, a)


if __name__ == "__main__":
    main()
