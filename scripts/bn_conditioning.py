"""|mean| / std of every BatchNorm channel in one VoteNet training step (bench.py's model and
batch: 8 scenes of 40000 points).

The fused SA and dense backward kernels evaluate the BatchNorm backward as dz = fmaf(a, g,
fmaf(b, z, c)) in fp32, where b*z and c cancel by a factor of about |mean| / std of the channel
(tests/test_bn_pool_glue_gpu.py::test_bn_bwd_dz_in_fp32_conditioning measures that error at
ratios 1, 30 and 1000).  This prints where the real layers sit.  The batch statistics are read
back from the running statistics after one forward with momentum 1 (running_mean = batch mean,
running_var = unbiased batch variance), so nothing in the product path is instrumented.

    python scripts/bn_conditioning.py
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    from backtoreality_b200 import scenes
    from backtoreality_b200.votenet import VoteNet

    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    net = VoteNet(22, 1, 22, np.ones((22, 3), np.float32), input_feature_dim=1, num_proposal=256,
                  vote_factor=1, sampling="vote_fps").to(dev).train()
    bns = [(n, m) for n, m in net.named_modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)]
    for _, m in bns:
        m.momentum = 1.0
    pc = torch.from_numpy(scenes.batch(0, 8, 40000, C=1, kind="room", dup=0.2)).to(dev)
    net({"point_clouds": pc})
    torch.cuda.synchronize()
    print("%s, %s" % (torch.cuda.get_device_name(dev), torch.__version__))
    print("%-52s %5s %10s %10s %10s" % ("BatchNorm", "C", "median", "p99", "max"))
    worst = 0.0
    for name, m in bns:
        r = (m.running_mean.abs() / m.running_var.clamp_min(1e-30).sqrt()).double().cpu().numpy()
        worst = max(worst, float(r.max()))
        print("%-52s %5d %10.3g %10.3g %10.3g" % (name, r.size, np.median(r), np.percentile(r, 99), r.max()))
    print("largest |mean|/std over all channels: %.3g" % worst)


if __name__ == "__main__":
    main()
