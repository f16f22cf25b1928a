#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: Pointnet2Backbone(+vote head) fwd+bwd scenes/sec @40k pts.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b2r|reference]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one batch of synthetic ScanNet-shaped scenes:
VoteNet FSB (Pointnet2Backbone -> VotingModule -> vote aggregation + proposal head), batch 8 per
GPU, 40k points + height feature, train-mode BatchNorm, forward + backward + (N>1) one NCCL
all-reduce of the flat fp32 gradient + Adam step.  Scenes are sharded across ranks (weak
scaling, no data-path collective).  Prints ONE JSON line on rank 0 (see the task contract):
  value     scenes/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e       the same with the step's input copied from PINNED HOST memory and the loss read back
  roofline  the dominant HBM-bound libb2r kernel (fused QueryAndGroup) timed live with CUDA events
  fps       the FPS cluster kernel (bound by the serial fp32 chain, not by HBM or tensor cores)
  cpu_baseline  the oracle's CPU port of the same step on this box's host cores (N=1 only)
`--impl reference` times that CPU port alone (the reference has no CPU path and is CUDA-only:
"CPU not supported", _ext_src/src/sampling.cpp:38-40; its GPU kernels are timed separately by
scripts/microbench.py).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "Pointnet2Backbone fwd+bwd scenes/sec @40k pts"
UNIT = "scenes/s"


_RESULT_OUT = sys.stdout


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def emit(obj):
    print(json.dumps(obj), file=_RESULT_OUT, flush=True)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b2r", choices=["b2r", "reference"])
    ap.add_argument("--workload", default="votenet", choices=["votenet", "br", "gf3d"],
                    help="votenet: BASELINE.json configs[1] (the metric's config, default); br: configs[2], "
                         "the VoteNet_DA 'Back to Reality' step (source forward + target forward + one "
                         "backward, batch 8+8 per GPU); gf3d: configs[3], the GroupFree3D backbone "
                         "(50k points, batch 4 per GPU, fp2 width 288)")
    ap.add_argument("--batch", type=int, default=0,
                    help="scenes per GPU per step (default: 8; br: 8 source + 8 target; gf3d: 4)")
    ap.add_argument("--npoints", type=int, default=0, help="points per scene (default 40000; gf3d 50000)")
    ap.add_argument("--cpu-scenes", type=int, default=0,
                    help="scenes per CPU step (default: the GPU arm's batch)")
    ap.add_argument("--leg", default="", help=argparse.SUPPRESS)   # internal: subprocess legs
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true",
                    help="launch every kernel from Python instead of replaying the captured step")
    ap.add_argument("--no-pipeline", action="store_true",
                    help="geometry pre-pass of a batch inside its own step (not one step ahead)")
    ap.add_argument("--pipeline-depth", type=int, default=1, choices=[1, 2],
                    help="pipelined step: 1 = whole geometry pre-pass of batch i+1 beside step i; 2 = SA1 "
                         "geometry of batch i+2 and the later levels' of batch i+1 beside step i")
    ap.add_argument("--fps-cluster", type=int, default=None,
                    help="pipelined step: CTAs per scene of the next batch's FPS (default 4; gf3d, with "
                         "4 scenes per GPU: 10)")
    ap.add_argument("--trace", default="",
                    help="after timing, trace 3 steps with torch.profiler (CUPTI) and write a per-kernel "
                         "summary + stream-occupancy analysis of one step to this file")
    ap.add_argument("--prepass-after", type=int, default=None,
                    help="pipelined step: start the next batch's pre-pass after this SA level's forward "
                         "(-1: with the step; default 1, br: -1 -- its step holds two forwards)")
    ap.add_argument("--sm-caps", default="",
                    help="pipelined step: persistent-grid caps 'fwd:bwd' of sa1,sa2,sa3,sa4,vote-agg "
                         "(comma separated, 0 = every SM); default: see PipelinedTrainStep")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, run ONE EXTRA, untimed step of the timed path (same captured "
                         "graph) from the initial weights on the first batch, and write what it produced to "
                         "DIR/<name>.npy (float32): the loss, the gradient of every parameter and the BatchNorm "
                         "running statistics.  Not the last timed step: the timed trajectory does not repeat "
                         "bit for bit (atomics in the fused backward, carried on by Adam)")
    a = ap.parse_args()
    if a.dump_outputs and os.environ.get("B2R_PINGPONG", "0") not in ("0", ""):
        # two captured graphs alternate; the gradient tensors of only one of them are kept
        ap.error("--dump-outputs is not supported with B2R_PINGPONG=1")
    if a.batch <= 0:
        a.batch = 4 if a.workload == "gf3d" else 8
    if a.npoints <= 0:
        a.npoints = 50000 if a.workload == "gf3d" else 40000
    if a.cpu_scenes <= 0:
        a.cpu_scenes = a.batch
    # measured optima (profiles/r02/sweep_*.log): the pre-pass must end with the step, on as few SMs
    # as that allows
    if a.prepass_after is None:
        a.prepass_after = {"br": -1, "gf3d": 0}.get(a.workload, 1)
    if a.fps_cluster is None:
        a.fps_cluster = 10 if a.workload == "gf3d" else 4
    return a


WORKLOADS = {
    "votenet": "VoteNet FSB backbone+vote head fwd/bwd (BASELINE.json configs[1]): "
               "Pointnet2Backbone(input_feature_dim=1) + VotingModule + ProposalModule("
               "vote_aggregation, 256 proposals), train-mode BN, Adam step",
    "br": "VoteNet BR training step (BASELINE.json configs[2]): VoteNet_DA, source forward + target "
          "forward + one backward (train_Votenet_BR.py:277-289), 8 + 8 scenes per GPU, train-mode BN, "
          "Adam step; the domain discriminators stay in torch",
    "gf3d": "GroupFree3D FSB backbone fwd/bwd (BASELINE.json configs[3]): Pointnet2Backbone("
            "input_feature_dim=0, fp2 width 288), num_point 50000, batch 4 per GPU, train-mode BN, Adam step",
}
LOSSES = {
    "votenet": "synthetic scalar: mean(proposal_scores^2) + mean((vote_xyz-seed_xyz)^2)",
    "br": "synthetic scalar: the votenet loss of the source AND the target forward + mean(global_d_pred^2) "
          "+ mean(local_d_pred^2) of both",
    "gf3d": "synthetic scalar: mean(fp2_features^2)",
}


def scenes_per_step(a):
    """scenes one GPU processes per step"""
    return 2 * a.batch if a.workload == "br" else a.batch


def workload_config(a, world):
    return {
        "workload": WORKLOADS[a.workload],
        "scenes_per_gpu": scenes_per_step(a), "global_batch": scenes_per_step(a) * world,
        "points_per_scene": a.npoints,
        "scene_kind": "room (ScanNet-shaped surfaces, 20% duplicate points), seeds 1000+i",
        "loss": LOSSES[a.workload],
        "parallelism": "dp%d (scenes sharded, flat-gradient NCCL all-reduce)" % world,
        "optimizer": ("Adam, lr 1e-3, one streaming kernel over the flat parameter buffer (flat_adam.FlatAdam)"
                      if os.environ.get("B2R_TORCH_ADAM", "0") in ("0", "")
                      else "torch.optim.Adam(fused=True, capturable=True), lr 1e-3"),
        "l2": "160 MB buffer (> the 126 MB L2) written between steps (flush) + 4 rotating input batches",
        "e2e_input": "pinned host -> device on a copy stream, one step ahead (train_step.HostPrefetcher)",
        "launch": ("whole step (fwd+bwd+Adam) captured in one CUDA graph, replayed per batch" if world == 1
                   else ("fwd+bwd replayed from one CUDA graph; NCCL all-reduce + fused Adam eager"
                         if os.environ.get("B2R_EAGER_COLLECTIVE", "0") not in ("0", "")
                         else "whole step (fwd+bwd + gradient pack + NCCL all-reduce + Adam) captured in one "
                              "CUDA graph per rank, replayed per batch")),
        "pipeline": ("none: FPS / ball query of a batch run inside its own step (geometry stream)"
                     if a.no_pipeline or a.no_graph
                     else "geometry pre-pass (FPS, centre gather, ball query, pad-free plans of sa1..sa4) of "
                          "batch i+1 runs beside the step of batch i in the same graph (%d-CTA FPS clusters, "
                          "started after SA level %d's forward; depth %d); every timed step = one pre-pass + "
                          "one fwd/bwd/Adam; e2e copies a later batch from pinned host memory and reads the "
                          "loss of batch i" % (a.fps_cluster, a.prepass_after + 1, a.pipeline_depth)),
        "mlp_math": "SA blocks: fused tcgen05 in the pad-free position space (copies of a ball's first hit "
                    "are not recomputed), forward TF32 / backward BF16 operands, fp32 accumulate; FP / "
                    "voting / proposal MLPs: dense tcgen05 layers, TF32 forward and backward",
    }


def synthetic_loss(ep):
    return (ep["proposal_scores_raw"] ** 2).mean() + ((ep["vote_xyz"] - ep["seed_xyz"]) ** 2).mean()


def workload_loss(workload, net, pc, geometry=None, on_sa2_grad=None):
    """forward + synthetic loss of one step of `workload` (shared by the GPU arm and the CPU port:
    `net` takes {"point_clouds": ..} or, gf3d, the point cloud itself).  on_sa2_grad: called in
    backward once the gradient of SA2's output exists, i.e. when every layer after SA2 has its
    weight gradients (N > 1: the early all-reduce bucket starts there)."""
    def hook(ep):
        if on_sa2_grad is not None and ep["sa2_features"].requires_grad:
            ep["sa2_features"].register_hook(lambda g: on_sa2_grad())

    if workload == "votenet":
        ep = net({"point_clouds": pc, "geometry": geometry} if geometry is not None else {"point_clouds": pc})
        if "seed_xyz" not in ep:
            ep["seed_xyz"] = ep["fp2_xyz"]
        hook(ep)
        return synthetic_loss(ep)
    if workload == "br":
        half = pc.shape[0] // 2
        loss = 0.0
        geo = [None, None]
        if geometry is not None:                  # pre-pass of all 16 scenes, consumed half by half
            from backtoreality_b200.backbone_module import Pointnet2Backbone
            geo = Pointnet2Backbone.split_geometry(geometry, 2)
        for part, g in zip((pc[:half], pc[half:]), geo):      # source forward, then target forward
            ep = net({"point_clouds": part, "geometry": g} if g is not None else {"point_clouds": part})
            if "seed_xyz" not in ep:
                ep["seed_xyz"] = ep["fp2_xyz"]
            loss = loss + synthetic_loss(ep)
            if "global_d_pred" in ep:
                loss = loss + (ep["global_d_pred"] ** 2).mean() + (ep["local_d_pred"] ** 2).mean()
        return loss
    ep = net(pc, geometry=geometry) if geometry is not None else net(pc)
    hook(ep)
    return (ep["fp2_features"] ** 2).mean()


def make_batch(a, index):
    """one step's input for one GPU: (scenes_per_step, N, 3 + C) float32 numpy"""
    from backtoreality_b200 import scenes
    n = scenes_per_step(a)
    return scenes.batch(index * n, n, a.npoints, C=0 if a.workload == "gf3d" else 1, kind="room", dup=0.2)


# ------------------------------------------------------------------------- CPU baseline ----
def port_model(a):
    """The oracle's CPU port (oracle/cpu_modules.py) of the workload's model; also the model the
    `reference_gpu` leg runs over the reference's own CUDA kernels."""
    from oracle import cpu_modules
    if a.workload == "gf3d":
        return cpu_modules.Backbone(input_feature_dim=0, fp2_out=288)
    return cpu_modules.VoteNetCPU(input_feature_dim=1, num_proposal=256)


def cpu_steps(a, steps, warmup, per_step):
    """The oracle's CPU port of the same training step on `per_step` scenes (br: half source,
    half target; its domain discriminators -- 0.1 % of the work -- are not part of the port).
    Returns (scenes/s, ms/step, cores)."""
    from backtoreality_b200 import scenes
    from oracle import cpu_ops
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    net = port_model(a).train()
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    pool = [torch.from_numpy(scenes.batch(100 + i * per_step, per_step, a.npoints,
                                          C=0 if a.workload == "gf3d" else 1, kind="room", dup=0.2))
            for i in range(2)]

    def one(i):
        loss = workload_loss(a.workload, net, pool[i % len(pool)])
        loss.backward()
        opt.step()
        opt.zero_grad()
        return float(loss.detach())

    for i in range(warmup):
        one(i)
    t0 = time.perf_counter()
    for i in range(steps):
        one(i)
    dt = time.perf_counter() - t0
    return per_step * steps / dt, 1e3 * dt / steps, max(cores, cpu_ops.num_threads())


def reference_gpu_steps(a, dev, steps=10, warmup=3):
    """The reference's OWN CUDA kernels (oracle/_ref/_ext.so: its _ext_src compiled for sm_100a by
    oracle/Makefile) under the unfused restatement of its Python stack (oracle/cpu_modules.py:
    group, -=, /=, cat, cuDNN SharedMLP with TF32 allowed, max_pool2d), same model / loss / Adam,
    same batch size, on this GPU.  Reported beside the product arm; returns None when the
    extension was not built."""
    import importlib.util
    path = os.path.join(ROOT, "oracle", "_ref", "_ext.so")
    if not os.path.isfile(path):
        return None
    from backtoreality_b200 import scenes
    from oracle import cpu_modules
    spec = importlib.util.spec_from_file_location("_ext", path)
    ref_ext = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_ext)
    saved = cpu_modules._ext
    cpu_modules._ext = ref_ext
    try:
        torch.manual_seed(0)
        torch.backends.cudnn.benchmark = True
        net = port_model(a).to(dev).train()
        opt = torch.optim.Adam(net.parameters(), lr=1e-3)
        n = scenes_per_step(a)
        pool = [torch.from_numpy(make_batch(a, 100 + i)).to(dev) for i in range(2)]

        def one(i):
            loss = workload_loss(a.workload, net, pool[i % 2])
            loss.backward()
            opt.step()
            opt.zero_grad()

        for i in range(warmup):
            one(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            one(i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        return {"value": n / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps,
                "warmup": warmup,
                "what": "reference CUDA kernels (oracle/_ref/_ext.so, sm_100a build of its "
                        "_ext_src) + unfused Python stack + cuDNN (TF32 allowed, benchmark mode), "
                        "eager, same model/loss/Adam, %d scenes x %d points" % (n, a.npoints)}
    finally:
        cpu_modules._ext = saved


def run_leg(a):
    """Internal (--leg): one of the product arm's reference legs, in its own process."""
    if a.leg == "reference_gpu":
        res = (reference_gpu_steps(a, torch.device("cuda", 0), a.steps, a.warmup)
               if torch.cuda.is_available() else None)
        emit(res or {})
    else:
        per = scenes_per_step(a) if a.cpu_scenes >= a.batch else (
            2 * a.cpu_scenes if a.workload == "br" else a.cpu_scenes)
        val, ms, cores = cpu_steps(a, 3, 1, per)
        emit({"value": val, "unit": UNIT, "cores": cores, "kind": "port", "ms_per_step": ms,
              "sample": "%d scenes of %d points per step, 3 timed steps after 1 warm-up (same model, loss, "
                        "optimizer; oracle/cpu_modules.py + b2r_oracle.c)" % (per, a.npoints)})


def run_reference(a):
    """`--impl reference`: the CPU arm.  Rank 0 only; other ranks exit without work."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    # one step = the GPU arm's per-GPU batch (same BatchNorm batch), fewer scenes only when the
    # requested step count would take more than a few minutes
    per = scenes_per_step(a) if a.cpu_scenes >= a.batch else (2 * a.cpu_scenes if a.workload == "br" else a.cpu_scenes)
    if (a.steps + a.warmup) > 30:
        per = 2 if a.workload == "br" else 1
    val, ms, cores = cpu_steps(a, a.steps, a.warmup, per)
    cfg = {"workload": WORKLOADS[a.workload], "scenes_per_gpu": scenes_per_step(a),
           "global_batch": scenes_per_step(a), "points_per_scene": a.npoints,
           "scene_kind": "room (ScanNet-shaped surfaces, 20% duplicate points), seeds 1000+i",
           "loss": LOSSES[a.workload],
           "parallelism": "host CPU, %d threads (the reference has no CPU path for these ops: this is "
                          "the oracle's port of the same step, oracle/cpu_modules.py + b2r_oracle.c)" % cores,
           "l2": "n/a (CPU)", "launch": "eager torch CPU + OpenMP C oracle ops", "pipeline": "none",
           "mlp_math": "fp32"}
    sample = "%d scenes of %d points per step, %d steps" % (per, a.npoints, a.steps)
    emit({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


# ------------------------------------------------------------------------- clocks ----------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.rows = []
        self.proc = None
        try:
            uuid = str(torch.cuda.get_device_properties(dev).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", uuid, "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception as e:  # nvidia-smi missing: report that instead of clocks
            log("clock sampler unavailable:", e)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def window(self, t0, t1):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            if t < t0 or t > t1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()


def trace_steps(path, fn, steps=3):
    """Kernel timeline of `steps` steps from CUPTI (torch.profiler): per-kernel totals and, for
    the LAST step, how much of the step some kernel was running / only side-stream kernels were
    running / nothing was running.  Evidence for where a graph-replayed step spends its time."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(steps):
            fn(i)
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type is not None and "cuda" in str(e.device_type).lower()
          and e.time_range is not None]
    ev.sort(key=lambda e: e.time_range.start)
    if not ev:
        open(path, "w").write("no CUDA activity records\n")
        return
    t_begin, t_end = ev[0].time_range.start, max(e.time_range.end for e in ev)
    span = (t_end - t_begin) / steps
    last = [e for e in ev if e.time_range.start >= t_end - span]
    agg = {}
    for e in last:
        k = e.name[:90]
        c = agg.setdefault(k, [0, 0.0])
        c[0] += 1
        c[1] += e.time_range.end - e.time_range.start
    # union of busy intervals
    busy, cur_s, cur_e = 0.0, None, None
    for e in last:
        s_, e_ = e.time_range.start, e.time_range.end
        if cur_e is None or s_ > cur_e:
            if cur_e is not None:
                busy += cur_e - cur_s
            cur_s, cur_e = s_, e_
        else:
            cur_e = max(cur_e, e_)
    busy += (cur_e - cur_s) if cur_e is not None else 0.0
    with open(path, "w") as f:
        f.write("CUPTI trace of %d steps; last step analysed: span %.1f us, %d kernels/memcpys, "
                "some kernel running %.1f us (%.1f%%), nothing running %.1f us\n"
                % (steps, span, len(last), busy, 100 * busy / span, span - busy))
        tot = sum(v[1] for v in agg.values())
        f.write("sum of kernel durations %.1f us (overlap across streams counted twice)\n" % tot)
        for k, (n, us) in sorted(agg.items(), key=lambda kv: -kv[1][1])[:60]:
            f.write("%4d %9.1f us %5.1f%%  %s\n" % (n, us, 100 * us / tot, k))
    # time-ordered timeline of the last step with the stream of every record (critical-path view)
    try:
        kev = [k for k in prof.profiler.kineto_results.events()
               if "cuda" in str(k.device_type()).lower() and k.duration_ns() > 0]
        kev.sort(key=lambda k: k.start_ns())
        t1 = max(k.start_ns() + k.duration_ns() for k in kev)
        t0 = t1 - span * 1e3
        streams = {}
        with open(path.replace(".txt", "") + "_timeline.txt", "w") as f:
            f.write("# last traced step: start us (from step begin), duration us, stream, kernel\n")
            for k in kev:
                if k.start_ns() < t0:
                    continue
                sid = streams.setdefault(k.device_resource_id(), len(streams))
                f.write("%9.1f %8.1f  s%d  %s\n" % ((k.start_ns() - t0) / 1e3, k.duration_ns() / 1e3, sid,
                                                  k.name()[:110]))
    except Exception as e:  # the timeline is a diagnostic; the summary above is the artifact
        print("timeline dump failed: %r" % (e,), file=sys.stderr)


def dump_outputs(out_dir, loss, net, grads):
    """What the training step hands its caller: the loss, the gradients (parameter order) and the
    BatchNorm running statistics.  The updated parameters are left out: Adam normalises its update
    per element, which turns rounding noise in a near-zero gradient into a step of up to lr."""
    torch.cuda.synchronize()
    arrays = {"loss": loss}
    for (name, _), g in zip(net.named_parameters(), grads):
        if g is not None:
            arrays["grad." + name] = g
    for name, b in net.named_buffers():
        if b.is_floating_point():
            arrays["buffer." + name] = b
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    assert total <= 64 << 20, "outputs of %d bytes exceed the 64 MB dump limit" % total
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)
    log("wrote %d arrays (%.1f MB) to %s" % (len(arrays), total / 2**20, out_dir))


# ------------------------------------------------------------------------- GPU arm ---------
def run_b2r(a):
    import torch.distributed as dist
    from backtoreality_b200 import _ext, _lib, dist_utils, scenes
    from backtoreality_b200.backbone_module import Pointnet2Backbone
    from backtoreality_b200.votenet import VoteNet, VoteNet_DA

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b2r needs a CUDA device (no CPU fallback exists)")
    _lib.lib()  # loud failure when libb2r.so is missing
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_IB_DISABLE", "1")      # NVLink / NVSwitch only
        os.environ.setdefault("NCCL_P2P_LEVEL", "NVL")
        dist.init_process_group("nccl", device_id=dev)
    assert world == a.gpus or world == 1, "launch with torchrun --nproc-per-node %d" % a.gpus

    # (only the br workload's domain discriminators still run cuDNN convolutions)
    torch.backends.cudnn.benchmark = True
    torch.manual_seed(0)  # identical replicas
    if a.workload == "gf3d":
        net = Pointnet2Backbone(input_feature_dim=0, fp2_out=288).to(dev).train()
        backbone = net
    else:
        cls = VoteNet_DA if a.workload == "br" else VoteNet
        net = cls(22, 1, 22, np.ones((22, 3), np.float32), input_feature_dim=1, num_proposal=256,
                  vote_factor=1, sampling="vote_fps").to(dev).train()
        backbone = net.backbone_net
    params = [p for p in net.parameters()]
    # N > 1: gradients are packed into one flat buffer for a single all-reduce per step
    # optimizer: Adam over one flat buffer (flat_adam.FlatAdam: pack + [all-reduce] + ONE kernel);
    # B2R_TORCH_ADAM=1 keeps torch.optim.Adam(fused) + FlatGradBucket (round 1's arrangement)
    early_hook = None
    use_flat_adam = os.environ.get("B2R_TORCH_ADAM", "0") in ("0", "")
    if use_flat_adam:
        from backtoreality_b200.flat_adam import FlatAdam
        bucket = None
        opt = FlatAdam(params, lr=1e-3)
        if world > 1 and a.workload != "br" and os.environ.get("B2R_OVERLAP", "0") not in ("0", ""):
            # opt-in (measured at 2 GPUs: 3.490 vs 3.492 ms -- the 3.8 MB all-reduce is not what the
            # N > 1 step waits for).  SA1's and SA2's gradients arrive last: everything else is
            # all-reduced on a side stream while their backward runs (sa1, sa2 come first in
            # net.parameters())
            late = list(backbone.sa1.parameters()) + list(backbone.sa2.parameters())
            assert all(x is y for x, y in zip(late, params)), "parameter order: sa1, sa2 first"
            opt.set_late(len(late))
            early_hook = opt.reduce_early
    else:
        bucket = dist_utils.FlatGradBucket(params, as_views=False) if world > 1 else None
        opt = torch.optim.Adam(params, lr=1e-3, fused=True, capturable=True)
    live = {"grads": None}   # the gradient tensors the last backward (or the graph) produced
    # --dump-outputs: the weights and BatchNorm statistics the dumped step starts from
    initial = ([t.detach().clone() for t in list(net.parameters()) + list(net.buffers())]
               if a.dump_outputs else None)

    pool_n = 4
    host = [torch.from_numpy(make_batch(a, rank * pool_n + i)).pin_memory() for i in range(pool_n)]
    resident = [h.to(dev) for h in host]
    flush = torch.empty(160 << 20, dtype=torch.uint8, device=dev)   # > the 126 MB L2

    def fwd_bwd(pc, geometry=None):
        for p in params:          # autograd then ASSIGNS fresh gradients: no accumulate kernels,
            p.grad = None         # nothing to zero
        loss = workload_loss(a.workload, net, pc, geometry, on_sa2_grad=early_hook)
        loss.backward()
        live["grads"] = [p.grad for p in params]
        return loss

    def finish():
        if use_flat_adam:         # pack, (N > 1) the step's only collective, one Adam kernel
            opt.step(live["grads"])
            return
        if bucket is not None:    # the step's only collective: one NCCL sum of the flat gradient
            bucket.reduce_from(live["grads"])
        opt.step()

    def step(pc, geometry=None):
        loss = fwd_bwd(pc, geometry)
        finish()
        return loss

    def stage(msg):
        if world > 1 or os.environ.get("B2R_BENCH_VERBOSE"):
            log("[rank %d] %s" % (rank, msg))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_loop(fn):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for i in range(a.steps):
            flush.zero_()  # L2 flush between steps
            fn(i)
        e1.record()
        barrier()
        t1 = time.perf_counter()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), t0, t1

    stage("model and %d resident batches ready; eager warm-up" % pool_n)
    for i in range(max(a.warmup, 3)):
        step(resident[i % pool_n])
    torch.cuda.synchronize()
    stage("warm-up done")

    # kernel-level timing (roofline / fps blocks): a few eager steps with CUDA events around every
    # libb2r launch on its launching stream -- events cannot be recorded inside a graph replay
    _ext.TIME_OPS.update(["sa_layer_fwd", "sa_layer_bwd", "furthest_point_sampling"])
    _ext.TIMED.clear()
    k_steps = min(a.steps, 5)
    torch.cuda.synchronize()
    l0 = _ext.LAUNCHES
    for i in range(k_steps):
        flush.zero_()
        step(resident[i % pool_n])
    torch.cuda.synchronize()
    launches_per_step = (_ext.LAUNCHES - l0) // k_steps
    timed = {k: list(v) for k, v in _ext.TIMED.items()}
    _ext.TIME_OPS.clear()

    # the step as the user runs it: captured once into a CUDA graph, replayed per batch
    # (N = 1: the optimizer too; N > 1: forward+backward are replayed, the NCCL all-reduce and the
    # 3-kernel fused Adam stay eager so no collective is ever captured)
    graphed = None
    # B2R_EAGER_COLLECTIVE=1: round 1's arrangement (only forward+backward replayed; pack, NCCL
    # all-reduce and Adam launched eagerly after every replay)
    capture_all = world == 1 or os.environ.get("B2R_EAGER_COLLECTIVE", "0") in ("0", "")
    # br runs two forwards per step: one pre-pass over its 16 scenes, pad-free plans per half
    pipelined = not (a.no_graph or a.no_pipeline)
    for attempt in ((0, 1) if not a.no_graph else ()):
        try:
            from backtoreality_b200.train_step import (CapturedTrainStep, PipelinedTrainStep,
                                                       PipelinedTrainStep2, PipelinedTrainStepPP)
            # B2R_PINGPONG=1: two graphs over two static buffer sets, no rotation copies after the
            # optimizer (measured: 3.50 vs 3.48 ms -- the copies were not on the critical path)
            Pipe = PipelinedTrainStepPP if os.environ.get("B2R_PINGPONG", "0") not in ("0", "") \
                else PipelinedTrainStep
            stage("capturing the step into a CUDA graph")
            if pipelined:
                # the vote-aggregation block has no pre-pass level of its own: give its kernels the
                # caps of the levels around it (forward: beside SA1's FPS; backward: it runs first)
                start = None if a.prepass_after < 0 else a.prepass_after
                caps, head_cap = PipelinedTrainStep.default_caps(scenes_per_step(a), a.fps_cluster, start)
                if a.sm_caps:
                    caps = [tuple(int(v) for v in c.split(":")) for c in a.sm_caps.split(",")]
                    caps, head_cap = caps[:4], caps[4]
                if a.workload in ("votenet", "br"):
                    net.pnet.vote_aggregation.sm_limit = head_cap
                if a.pipeline_depth == 2:
                    graphed = PipelinedTrainStep2(backbone, step if capture_all else fwd_bwd,
                                                  resident[0], resident[1], fps_cluster=a.fps_cluster,
                                                  sm_caps=caps,
                                                  after_warmup_step=None if capture_all else finish,
                                                  start_after_level=start)
                else:
                    graphed = Pipe(backbone, step if capture_all else fwd_bwd,
                                   resident[0], fps_cluster=a.fps_cluster, sm_caps=caps,
                                   after_warmup_step=None if capture_all else finish,
                                   start_after_level=start, plan_splits=2 if a.workload == "br" else 1)
            else:
                graphed = CapturedTrainStep(step if capture_all else fwd_bwd, resident[0],
                                            after_warmup_step=None if capture_all else finish)
            stage("captured (%d libb2r launches per step)" % graphed.launches_per_step)
            break
        except Exception as e:
            if capture_all and world > 1 and attempt == 0:
                # the captured collective is the only new ingredient: retry with the all-reduce and
                # the optimizer launched eagerly after every replay (round 1's arrangement)
                log("capture with the NCCL all-reduce inside failed (%s: %s); retrying with an eager "
                    "collective" % (type(e).__name__, e))
                capture_all = False
                torch.cuda.synchronize()
                continue
            # report, then measure the eager loop instead
            log("CUDA-graph capture failed (%s: %s); timing the eager step" % (type(e).__name__, e))
            graphed = None
            pipelined = False
            if a.workload != "gf3d":
                net.pnet.vote_aggregation.sm_limit = 0

    def run_step(pc):
        if graphed is None:
            return step(pc)
        loss = graphed(pc)
        if not capture_all:
            finish()
        return loss

    # pipelined: call i submits batch i+1 (whose geometry pre-pass runs in this call) and trains
    # on batch i; resident[0] was submitted by the constructor
    nxt = (a.pipeline_depth if pipelined else 0)

    def prime():
        if pipelined and a.pipeline_depth == 2:
            graphed.prime(resident[0], resident[1])
        elif pipelined:
            graphed.prime(resident[0])

    for i in range(3):
        run_step(resident[(i + nxt) % pool_n])
    prime()
    sampler = ClockSampler(dev) if rank == 0 else None
    time.sleep(0.3)

    # (1) inputs resident in HBM (graph mode: one device-to-device copy into the static input)
    ms_dev, t0, t1 = timed_loop(lambda i: run_step(resident[(i + nxt) % pool_n]))
    launches = launches_per_step * a.steps
    clocks = sampler.window(t0, t1) if sampler else None

    # (2) end to end: pinned host input -> device each step, loss read back each step.  The
    # upload runs on a copy stream one step ahead of its use (train_step.HostPrefetcher): every
    # timed step uploads ONE batch from pinned host memory, trains on one batch and reads one loss
    from backtoreality_b200.train_step import HostPrefetcher
    pre = HostPrefetcher(host[0], dev) if graphed is not None else None
    state = {"slot": None}

    def e2e_step(i):
        if pre is not None:
            if state["slot"] is None:
                state["slot"] = pre.upload(host[(i + nxt) % pool_n])
            nslot = pre.upload(host[(i + nxt + 1) % pool_n])      # overlaps this step
            loss = run_step(pre.get(state["slot"]))               # device copy into the static input
            pre.release(state["slot"])
            state["slot"] = nslot
            return float(loss.item())
        pc = host[i % pool_n].to(dev, non_blocking=True)
        return float(step(pc).item())

    prime()
    for i in range(2):
        e2e_step(i)
    up0 = pre.bytes_uploaded if pre is not None else 0
    ms_e2e, _, t1e = timed_loop(lambda i: e2e_step(i + 2))
    h2d_per_step = ((pre.bytes_uploaded - up0) // a.steps) if pre is not None else int(host[0].numel() * 4)
    if sampler:
        # clocks over both timed regions (device-resident and end-to-end loops, back to back)
        clocks = sampler.window(t0, t1e)
        sampler.stop()

    if a.dump_outputs:
        # One more step of the same path after the timed ones, from the initial weights and on a
        # fixed batch.  The timed trajectory does not repeat bit for bit (the fused backward sums
        # with atomics) and Adam carries that noise on from step to step; one step from a fixed
        # state repeats to within rounding, so two builds compare array by array.
        with torch.no_grad():
            for t, v in zip(list(net.parameters()) + list(net.buffers()), initial):
                t.copy_(v)
        prime()
        loss = run_step(resident[nxt % pool_n])
        if rank == 0:
            dump_outputs(a.dump_outputs, loss, net, live["grads"])

    if a.trace and rank == 0:
        trace_steps(a.trace, lambda i: run_step(resident[(i + nxt) % pool_n]))

    if rank != 0:
        # leave without tearing NCCL down (see the end of this function): rank 0 still runs its
        # single-GPU timing legs and does not need this rank any more
        torch.cuda.synchronize()
        sys.stderr.flush()
        os._exit(0)

    scenes_total = scenes_per_step(a) * world * a.steps
    out = {
        "metric": METRIC, "value": scenes_total / (ms_dev * 1e-3), "unit": UNIT,
        "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": ms_dev / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "tf32 fwd / bf16 bwd operands, f32 accumulate", "data": "synthetic",
        "config": workload_config(a, world),
        "e2e": {"value": scenes_total / (ms_e2e * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": int(h2d_per_step), "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / a.steps},
        "gpu_launches": launches,
        "clocks": clocks,
    }
    if graphed is None:
        out["config"]["launch"] = "eager: every kernel launched from Python"
    k_div = k_steps

    # roofline of the dominant libb2r kernel class (the fused SA layers), SURVEY.md 8(d): the
    # fused SA MLP is the path's only dense contraction, so it is measured against the TENSOR peak
    # with the algorithmic flops 2*np*ns*sum(C_l*C_l+1) per scene (backward 2x, recomputation not
    # credited, pad copies not discounted), live CUDA events around every launch; the same
    # launches' block-level compulsory bytes against the HBM peak are reported beside it
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    bf16_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = ("measured (MEASURED_PEAKS.json bf16_tflops_sustained / hbm_gbs)" if "hbm_gbs" in peaks
                else "fallback 1400 TFLOP/s, 6650 GB/s")
    cand = {}
    for name, kern in (("sa_layer_fwd", "sa_layer_fwd_kernel"), ("sa_layer_bwd", "sa_layer_bwd_kernel")):
        ev = timed.get(name, [])
        if ev:
            cand[name] = (sum(s_.elapsed_time(e_) for s_, e_, _ in ev), sum(w[0] for _, _, w in ev),
                          sum(w[1] for _, _, w in ev), len(ev), kern)
    if cand:
        name = max(cand, key=lambda k: cand[k][0])
        tot_ms, tot_b, tot_f, n, kern = cand[name]
        tf = tot_f / (tot_ms * 1e-3) / 1e12
        gbs = tot_b / (tot_ms * 1e-3) / 1e9
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
            traffic = (tj.get(name) or tj[kern])["dram_bytes_per_launch"]
        except Exception:
            pass
        # forward operands are TF32 (half the bf16 rate), backward operands BF16
        peak = bf16_peak if name == "sa_layer_bwd" else bf16_peak / 2
        out["roofline"] = {
            "kernel": "%s: all %d launches/step of b2r_%s (fused tcgen05 SA layers of sa1..sa4 and the vote "
                      "aggregation; SA1's thin first layer runs mlp_thin.cu's streaming kernel)"
                      % (kern, n // k_div, name),
            "bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak,
            "traffic": traffic, "peak_source": peak_src,
            "algorithmic_flops_per_launch": tot_f / n, "algorithmic_bytes_per_launch": tot_b / n,
            "avg_launch_us": 1e3 * tot_ms / n, "launches_timed": n, "ms_per_step": tot_ms / k_div,
            "hbm": {"achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                    "what": "SURVEY 8(d) block-level compulsory bytes (features + xyz + idx + weights + "
                            "pooled output; backward 2x) of the same launches / their time"},
            "other": {k: {"ms_per_step": v[0] / k_div, "achieved_tflops": v[2] / (v[0] * 1e-3) / 1e12,
                          "frac_of_tensor_peak": v[2] / (v[0] * 1e-3) / 1e12 /
                          (bf16_peak if k == "sa_layer_bwd" else bf16_peak / 2),
                          "achieved_gbs": v[1] / (v[0] * 1e-3) / 1e9, "launches_per_step": v[3] // k_div}
                      for k, v in cand.items() if k != name}}
    fp = timed.get("furthest_point_sampling", [])
    if fp:
        per_step = len(fp) // k_div
        ms_step = sum(s.elapsed_time(e) for s, e, _ in fp) / k_div
        # SA1 is the first FPS launch of every step: N points -> 2048 samples
        sa1 = [fp[i] for i in range(0, len(fp), per_step)]
        sa1_ms = float(np.mean([s.elapsed_time(e) for s, e, _ in sa1]))
        upd = scenes_per_step(a) * (2048 - 1) * a.npoints  # point-updates per step, 8 flop each
        if a.workload == "br":
            upd //= 2                                           # per launch: one of the two forwards
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6
        out["fps"] = {"kernel": "fps_bucket_kernel (SA1: Morton-sorted buckets + bounding-box skip test, "
                                "indices bit-identical) + fps_small_kernel (later levels), csrc/fps_bucket.cu; "
                                "timed standalone at the lowest-latency cluster width (inside the pipelined "
                                "step SA1 runs on %d-CTA clusters beside the step)" % a.fps_cluster,
                      "bound": "serial fp32 chain (not hbm/tensor)",
                      "note": "algorithmic point-updates (every point, every iteration) / time: the skip test "
                              "executes far fewer",
                      "launches_per_step": per_step, "ms_per_step_all_levels": ms_step,
                      "sa1_ms_per_batch": sa1_ms, "sa1_ms_per_scene": sa1_ms / a.batch,
                      "sa1_point_updates_per_s": upd / (sa1_ms * 1e-3),
                      "sa1_frac_of_fp32_issue_peak": 8 * upd / (sa1_ms * 1e-3) / fp32_peak}

    if world == 1 and not a.no_cpu_baseline:
        # both reference legs run in their own processes (they load oracle/_ref/_ext.so and
        # oracle/liborc.so: checkers, kept out of the product arm's process)
        del graphed
        torch.cuda.empty_cache()
        for leg, key in (("reference_gpu", "reference_gpu"), ("cpu_baseline", "cpu_baseline")):
            log("timing leg %s in a subprocess ..." % leg)
            try:
                cmd = [sys.executable, os.path.abspath(__file__), "--leg", leg, "--workload", a.workload,
                       "--batch", str(a.batch), "--npoints", str(a.npoints), "--cpu-scenes", str(a.cpu_scenes)]
                if leg == "reference_gpu":    # the CPU leg times a fixed 3-step sample (see run_leg)
                    cmd += ["--steps", str(a.steps), "--warmup", str(a.warmup)]
                r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
                line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
                if line:
                    res = json.loads(line[-1])
                    if res:
                        out[key] = res
                else:
                    log("leg %s printed no result: %s" % (leg, r.stderr[-400:]))
            except Exception as e:
                log("leg %s failed: %s: %s" % (leg, type(e).__name__, e))
        # the precision trade of the fused SA backward as a measurement: the SAME step with the SA
        # blocks and the FP / head MLPs on the unfused path (libb2r movers + cuDNN, TF32 forward
        # AND backward -- the reference's own arithmetic), same graph capture and pipelining
        log("timing leg unfused_tf32 in a subprocess ...")
        try:
            cmd = [sys.executable, os.path.abspath(__file__), "--workload", a.workload, "--batch", str(a.batch),
                   "--npoints", str(a.npoints), "--steps", str(a.steps), "--warmup", str(a.warmup),
                   "--no-cpu-baseline"]
            env = dict(os.environ, B2R_FUSED="0", B2R_DENSE="0")
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
            line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            if line:
                res = json.loads(line[-1])
                out["unfused_tf32_arm"] = {
                    "value": res["value"], "unit": UNIT, "ms_per_step": res["ms_per_step"],
                    "what": "B2R_FUSED=0 B2R_DENSE=0: SA blocks and FP / head MLPs through libb2r's "
                            "unfused kernels + cuDNN (TF32 operands forward and backward, FP32 "
                            "accumulate); the product arm's fused SA backward uses BF16 operands"}
            else:
                log("leg unfused_tf32 printed no result: %s" % r.stderr[-400:])
        except Exception as e:
            log("leg unfused_tf32 failed: %s: %s" % (type(e).__name__, e))
    emit(out)
    if world > 1:
        # Leave without tearing NCCL down: destroying a process group whose collectives live
        # inside a CUDA graph blocks in the communicator's destructor (seen on 2 GPUs: the result
        # was printed, the workers never exited).  All timed work is done, the other ranks left
        # the same way after the last timed barrier, and the OS reclaims everything.
        torch.cuda.synchronize()
        _RESULT_OUT.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    a = parse()
    # stdout carries exactly ONE line, the JSON result: anything a library prints to fd 1 (NCCL
    # writes "NCCL version ..." there) is sent to stderr instead
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if a.leg:
        run_leg(a)
    elif a.impl == "reference":
        run_reference(a)
    else:
        run_b2r(a)


if __name__ == "__main__":
    main()
