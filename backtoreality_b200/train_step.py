"""One training step as a replayable CUDA graph.

The hot path issues ~450 small launches per step (libb2r kernels through ctypes, cuDNN for the
FP / vote heads, optimizer); at ~9 ms of GPU work the Python launch overhead leaves the GPU idle
~20 % of the step.  Everything in the step is shape-static and sync-free (no `.item()`, no host
reads), so forward + backward + gradient all-reduce + optimizer are captured ONCE into a CUDA
graph and replayed: one launch per step, no gaps.

Values that are baked in at capture time: tensor addresses (the input is a static buffer that
`__call__` copies into) and the learning rate unless the optimizer reads it from the device
(flat_adam.FlatAdam.sync_hparams).  The BatchNorm momentum, which the reference's
BNMomentumScheduler changes once per epoch (pytorch_utils.py:262-296), replays from a device table
once `pytorch_utils.sync_bn_momentum(model)` has attached the model before the capture;
BNMomentumScheduler.step() then updates that table between replays.  A model that is not
attached keeps its capture-time momentum until `recapture()`.

The warm-up steps that precede a capture are REAL steps on the static batch.  Pass
`snapshot=[model, optimizer, ...]` (anything with state_dict / load_state_dict) and their state
-- weights, BatchNorm running statistics and num_batches_tracked, optimizer moments and step
counts -- is saved before the warm-up and restored after it, so a (re)capture leaves training
exactly where it was (each recapture would otherwise add `warmup` weight updates on duplicated
data).
"""
import copy

import torch
from . import step_arena


def _save_state(objs):
    return [copy.deepcopy(o.state_dict()) for o in (objs or [])]


def _restore_state(objs, saved):
    for o, sd in zip(objs or [], saved):
        o.load_state_dict(sd)


# "thread_local": CUDA calls of OTHER threads (the NCCL watchdog polling its events) neither
# invalidate nor dead-lock a capture -- needed when the step's gradient all-reduce is captured too
CAPTURE_ERROR_MODE = "thread_local"


class CapturedTrainStep:
    """`step_fn(static_input) -> loss tensor` runs fwd + bwd + all-reduce + optimizer, eagerly.
    This wraps it: `loss = captured(batch)` copies `batch` into the static input and replays."""

    def __init__(self, step_fn, example_input, warmup=3, after_warmup_step=None, snapshot=None):
        self.step_fn = step_fn
        self.snapshot = snapshot
        self.after_warmup_step = after_warmup_step   # e.g. the eager optimizer / gradient reset
        self.static_in = example_input.clone()
        self.warmup = warmup
        self.graph = None
        self.static_loss = None
        self.launches_per_step = None
        self.recapture()

    def recapture(self):
        from . import _ext
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        saved = _save_state(self.snapshot)
        with torch.cuda.stream(side):
            for _ in range(self.warmup):
                self._step()
                if self.after_warmup_step is not None:
                    self.after_warmup_step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        _restore_state(self.snapshot, saved)
        saved_ops = set(_ext.TIME_OPS)
        _ext.TIME_OPS.clear()          # timing events cannot be recorded inside a capture
        l0 = _ext.LAUNCHES
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode=CAPTURE_ERROR_MODE):
                loss = self._step()
            self.graph, self.static_loss = g, loss
            self.launches_per_step = _ext.LAUNCHES - l0
        finally:
            _ext.TIME_OPS.update(saved_ops)

    def _step(self):
        # every zero-initialised accumulator of the step comes from one arena, cleared by ONE memset
        step_arena.begin(self.static_in.device)
        try:
            return self.step_fn(self.static_in)
        finally:
            step_arena.end(self.static_in.device)

    def __call__(self, batch, non_blocking=True):
        self.static_in.copy_(batch, non_blocking=non_blocking)
        self.graph.replay()
        return self.static_loss


class PipelinedTrainStep:
    """The captured step, software-pipelined across batches: while the GPU runs forward + backward
    + optimizer of batch i, the geometry pre-pass of batch i+1 (FPS, centre gather and ball query
    of sa1..sa4 -- they depend on xyz alone, never on weights) runs beside it on a side stream
    inside the same CUDA graph.  FPS is a serial chain of 2047+1023+511+255 dependent iterations
    that keeps few SMs busy for 2 ms; here it is off the critical path, on narrow clusters
    (`fps_cluster` CTAs per scene) next to MLP kernels whose persistent grids leave those SMs free.

        pipe = PipelinedTrainStep(net.backbone_net, step_fn, first_batch)
        for nxt in loader:            # the data loader is one batch ahead, as any prefetcher is
            loss_of_previous = pipe(nxt)

    `step_fn(pointcloud, geometry) -> loss` runs forward (passing `geometry` down to
    Pointnet2Backbone.forward), backward and the optimizer.  Every call does one geometry pre-pass
    and one full step, so K calls cost K of each: nothing is skipped, only re-ordered.
    `__call__(next_batch)` returns the loss of the batch submitted by the PREVIOUS call (or by
    the constructor / `prime`).  What is baked in at capture, and what replays from the device
(learning rate, BatchNorm momentum), as for CapturedTrainStep.
    """

    GEO_KEYS = ("inds", "new_xyz", "idx")                       # every level
    FP_KEYS = ("fp1_idx", "fp1_weight", "fp2_idx", "fp2_weight")   # last level: FP interpolation

    @staticmethod
    def default_caps(B, fps_cluster, start_after_level):
        """Persistent-grid caps (forward, backward) of the four SA levels + the cap for fused
        blocks outside the backbone (vote aggregation), for B scenes per step.  SA1's FPS of the
        next batch holds B*fps_cluster SMs for ~2 ms from the moment the pre-pass starts; the
        later levels' FPS hold B SMs (one CTA per scene) for ~1 ms more.
        start_after_level = None: the pre-pass starts with the step -> every forward kernel
        leaves the wide gap, the early backward the narrow one, SA1/SA2 backward run on all SMs.
        start_after_level = k (default 1, measured best: 4.39 vs 4.49 ms per step): levels <= k
        run their forward on every SM, everything up to the backward of level k+1 leaves the
        wide gap (those are the small, latency-bound kernels of the step, which do not care), the
        backward of levels <= k the narrow one."""
        from . import fused_sa
        wide = max(fused_sa.NUM_SMS - B * int(fps_cluster), 32)
        narrow = max(fused_sa.NUM_SMS - B, 32)
        if start_after_level is None:
            return [(wide, 0), (wide, 0), (wide, narrow), (wide, narrow)], (wide, narrow)
        caps = [(0, narrow) if lv <= start_after_level else (wide, wide) for lv in range(4)]
        return caps, (wide, wide)

    PLAN_KEYS = ("cidx", "ccen", "cmeta")    # levels computed pad-free (fused_sa.compact_plan)

    @classmethod
    def _keys(cls, level):
        split_plans = tuple(k for k in level if "#" in k and k.split("#")[0] in cls.PLAN_KEYS)
        return cls.GEO_KEYS + tuple(k for k in cls.PLAN_KEYS + cls.FP_KEYS if k in level) + split_plans

    def __init__(self, backbone, step_fn, first_batch, warmup=3, fps_cluster=4, sm_caps=None,
                 after_warmup_step=None, start_after_level=1, snapshot=None, plan_splits=1):
        self.backbone = backbone
        # > 1: the batch is consumed as that many consecutive forwards over equal slices
        # (Pointnet2Backbone.split_geometry), e.g. the source and target halves of the BR step
        self.plan_splits = int(plan_splits)
        self.step_fn = step_fn
        self.snapshot = snapshot
        self.after_warmup_step = after_warmup_step
        self.fps_cluster = int(fps_cluster)
        if sm_caps is None:
            sm_caps, _ = self.default_caps(first_batch.shape[0], self.fps_cluster, start_after_level)
        self.sm_caps = sm_caps
        # None: the pre-pass of the next batch starts with the step.  k in 0..3: it starts once
        # SA level k's forward has been issued, so that the wide, bandwidth-bound kernels of the
        # first levels run on every SM and SA1's FPS overlaps the small, latency-bound middle of
        # the step instead
        self.start_after_level = start_after_level
        self.warmup = warmup
        self.cur = first_batch.clone()
        self.next = first_batch.clone()
        self.side = torch.cuda.Stream(device=first_batch.device)
        self.geo_cur = None
        self.graph = None
        self.static_loss = None
        self.launches_per_step = None
        self.prime(first_batch)
        self.recapture()

    def _xyz(self, pc):
        return pc[..., 0:3].contiguous()

    def _levels(self, tensors):
        return [dict(t, event=None, fp_event=None, sm_limit=cap)
                for t, cap in zip(tensors, self.sm_caps)]

    def prime(self, batch):
        """(Re)start the pipeline: `batch` becomes the current batch, its geometry is computed
        now, eagerly."""
        self.cur.copy_(batch)
        xyz = self._xyz(self.cur)     # stays referenced until the side stream has been joined
        levels = self.backbone.geometry_prepass(xyz, side=self.side,
                                                plan_splits=getattr(self, "plan_splits", 1))
        torch.cuda.current_stream().wait_stream(self.side)
        fresh = [{k: lv[k] for k in self._keys(lv)} for lv in levels]
        if self.geo_cur is None:
            self.geo_cur = [{k: v.clone() for k, v in lv.items()} for lv in fresh]
        else:
            for dst, src in zip(self.geo_cur, fresh):
                for k in dst:
                    dst[k].copy_(src[k])

    def _pipelined(self):
        """one pipelined step on the static buffers: geometry(next) beside step(cur), then rotate"""
        main = torch.cuda.current_stream()
        # xyz_next is allocated on the main stream and read by the side stream for the whole
        # step: keep the reference until the join, or the allocator hands its memory to the
        # step's own activations while FPS is still reading it
        xyz_next = self._xyz(self.next)
        box = {}
        # the spatial sort of SA1's FPS depends on the coordinates alone: it runs NOW, on the side
        # stream, so that only the sampling itself sits on the pre-pass's dependency chain
        presorted = self._presort(xyz_next)

        def launch_prepass():
            box["nxt"] = self.backbone.geometry_prepass(xyz_next, fps_cluster=self.fps_cluster,
                                                        sm_limit=0, side=self.side,
                                                        plan_splits=self.plan_splits,
                                                        presorted=presorted)

        levels = self._levels(self.geo_cur)
        if self.start_after_level is None:
            launch_prepass()
        else:
            levels[self.start_after_level]["after_forward"] = launch_prepass
        step_arena.begin(self.cur.device)
        try:
            loss = self.step_fn(self.cur, levels)
        finally:
            step_arena.end(self.cur.device)
        if "nxt" not in box:       # the step never reached that level's hook
            launch_prepass()
        nxt = box["nxt"]
        main.wait_stream(self.side)
        del xyz_next
        # rotate: ONE multi-tensor copy launch for all geometry tensors of all levels
        dsts, srcs = [], []
        for dst, src in zip(self.geo_cur, nxt):
            for k in dst:
                dsts.append(dst[k])
                srcs.append(src[k])
        torch._foreach_copy_(dsts + [self.cur], srcs + [self.next])
        return loss

    def _presort(self, xyz_next):
        from . import _ext
        if _ext.FPS_LEGACY or self.start_after_level is None:
            return None       # legacy kernel: no sort; pre-pass from the step's start: nothing to gain
        self.side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.side), torch.no_grad():
            ws = _ext.fps_presort(xyz_next)
        ws.record_stream(torch.cuda.current_stream())
        return ws

    def recapture(self):
        from . import _ext
        warm = torch.cuda.Stream()
        warm.wait_stream(torch.cuda.current_stream())
        saved = _save_state(getattr(self, "snapshot", None))
        with torch.cuda.stream(warm):
            for _ in range(self.warmup):
                self._pipelined()
                if self.after_warmup_step is not None:
                    self.after_warmup_step()
        torch.cuda.current_stream().wait_stream(warm)
        torch.cuda.synchronize()
        _restore_state(getattr(self, "snapshot", None), saved)
        saved_ops = set(_ext.TIME_OPS)
        _ext.TIME_OPS.clear()          # timing events cannot be recorded inside a capture
        l0 = _ext.LAUNCHES
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode=CAPTURE_ERROR_MODE):
                loss = self._pipelined()
            self.graph, self.static_loss = g, loss
            self.launches_per_step = _ext.LAUNCHES - l0
        finally:
            _ext.TIME_OPS.update(saved_ops)

    def __call__(self, next_batch, non_blocking=True):
        self.next.copy_(next_batch, non_blocking=non_blocking)
        self.graph.replay()
        return self.static_loss


class PipelinedTrainStepPP(PipelinedTrainStep):
    """PipelinedTrainStep without the buffer rotation on the critical path ("ping-pong").

    The base class ends every step with a multi-tensor copy of the fresh geometry (and the next
    batch) into the static buffers the captured step reads: ~45 small copy kernels (~70 us) after
    the optimizer, where nothing can overlap them.  Here there are TWO sets of static buffers and
    TWO captured graphs: graph p trains on set p while the pre-pass of the next batch fills set
    1-p -- level by level, on the side streams, as soon as each level exists -- and the next call
    replays graph 1-p.  Same contract as the base class: call i submits batch i+1 and returns the
    loss of batch i; every call runs one complete pre-pass and one complete step."""

    def prime(self, batch):
        self.parity = 0
        if getattr(self, "X", None) is None:
            self.X = [batch.clone(), batch.clone()]
            self.G = [None, None]
        self.X[0].copy_(batch)
        xyz = self._xyz(self.X[0])
        levels = self.backbone.geometry_prepass(xyz, side=self.side)
        torch.cuda.current_stream().wait_stream(self.side)
        fresh = [{k: lv[k] for k in self._keys(lv)} for lv in levels]
        if self.G[0] is None:
            self.G = [[{k: v.clone() for k, v in lv.items()} for lv in fresh] for _ in range(2)]
        else:
            for dst, src in zip(self.G[0], fresh):
                for k in dst:
                    dst[k].copy_(src[k])
        self._alias()

    def _alias(self):   # the attributes the base class (and its tests) expose
        self.cur, self.next = self.X[self.parity], self.X[1 - self.parity]
        self.geo_cur = self.G[self.parity]

    def _pipelined_pp(self, p):
        main = torch.cuda.current_stream()
        xyz_next = self._xyz(self.X[1 - p])   # referenced until the side stream has been joined
        box = {}
        presorted = self._presort(xyz_next)

        def launch_prepass():
            box["nxt"] = self.backbone.geometry_prepass(xyz_next, fps_cluster=self.fps_cluster,
                                                        sm_limit=0, side=self.side, copy_to=self.G[1 - p],
                                                        presorted=presorted)

        levels = self._levels(self.G[p])
        if self.start_after_level is None:
            launch_prepass()
        else:
            levels[self.start_after_level]["after_forward"] = launch_prepass
        step_arena.begin(self.X[p].device)
        try:
            loss = self.step_fn(self.X[p], levels)
        finally:
            step_arena.end(self.X[p].device)
        if "nxt" not in box:
            launch_prepass()
        main.wait_stream(self.side)
        del xyz_next
        return loss

    def _pipelined(self):   # one eager step on the current parity (warm-up)
        loss = self._pipelined_pp(self.parity)
        self.parity ^= 1
        self._alias()
        return loss

    def recapture(self):
        from . import _ext
        warm = torch.cuda.Stream()
        warm.wait_stream(torch.cuda.current_stream())
        saved = _save_state(getattr(self, "snapshot", None))
        self.X[1].copy_(self.X[0])
        with torch.cuda.stream(warm):
            for _ in range((self.warmup + 1) // 2 * 2):     # an even count: parity returns to 0
                self._pipelined()
                if self.after_warmup_step is not None:
                    self.after_warmup_step()
        torch.cuda.current_stream().wait_stream(warm)
        torch.cuda.synchronize()
        _restore_state(getattr(self, "snapshot", None), saved)
        saved_ops = set(_ext.TIME_OPS)
        _ext.TIME_OPS.clear()          # timing events cannot be recorded inside a capture
        self.graphs, self.losses = [None, None], [None, None]
        try:
            for p in (0, 1):
                l0 = _ext.LAUNCHES
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, capture_error_mode=CAPTURE_ERROR_MODE):
                    loss = self._pipelined_pp(p)
                self.graphs[p], self.losses[p] = g, loss
                self.launches_per_step = _ext.LAUNCHES - l0
            self.graph, self.static_loss = self.graphs[0], self.losses[0]
        finally:
            _ext.TIME_OPS.update(saved_ops)

    def __call__(self, next_batch, non_blocking=True):
        p = self.parity
        self.X[1 - p].copy_(next_batch, non_blocking=non_blocking)
        self.graphs[p].replay()
        self.parity ^= 1
        self._alias()
        return self.losses[p]


class PipelinedTrainStep2(PipelinedTrainStep):
    """The pipelined step, two batches deep.  SA1's geometry (FPS of the whole 40k-point scene:
    2047 dependent iterations, ~2 ms on narrow clusters) and the later levels' (FPS 2048 -> 1024
    -> 512 -> 256, ball queries, 3-NN weights: ~1 ms) are independent chains once SA1's centres
    exist, so they run side by side, for DIFFERENT batches: the graph of step i holds

        side stream A   SA1 geometry of batch i+2
        side stream B   SA2..SA4 + FP geometry of batch i+1 (from its SA1 centres, computed by
                        stream A during step i-1)
        main stream     forward + backward + optimizer of batch i

    and then rotates the static buffers.  The longest geometry chain beside a step is ~2 ms
    instead of ~3 ms, which takes the pre-pass off the critical path of a ~3.5 ms step.  Every
    call still does one complete geometry pre-pass (two halves, of two batches) and one complete
    step; the data loader is two batches ahead:

        pipe = PipelinedTrainStep2(net.backbone_net, step_fn, batch0, batch1)
        for b in loader_from_batch2:          # call i submits batch i+2, trains on batch i
            loss_of_batch_i = pipe(b)
    """

    def __init__(self, backbone, step_fn, first_batch, second_batch, warmup=3, fps_cluster=4,
                 sm_caps=None, after_warmup_step=None, start_after_level=1, snapshot=None,
                 b_from_start=False):
        self.backbone = backbone
        # False: both geometry chains start from the same hook (after SA level
        # `start_after_level`'s forward), so the wide first-level kernels keep every SM
        self.b_from_start = bool(b_from_start)
        self.step_fn = step_fn
        self.snapshot = snapshot
        self.after_warmup_step = after_warmup_step
        self.fps_cluster = int(fps_cluster)
        if sm_caps is None:
            sm_caps, _ = self.default_caps(first_batch.shape[0], self.fps_cluster, start_after_level)
        self.sm_caps = sm_caps
        self.start_after_level = start_after_level
        self.warmup = warmup
        self.cur = first_batch.clone()
        self.next = second_batch.clone()
        self.next2 = second_batch.clone()
        self.side = torch.cuda.Stream(device=first_batch.device)     # A: SA1 geometry
        self.side_b = torch.cuda.Stream(device=first_batch.device)   # B: SA2..SA4 + FP geometry
        self.geo_cur = None
        self.geo_a_next = None      # SA1 geometry of `next`
        self.graph = None
        self.static_loss = None
        self.launches_per_step = None
        self.prime(first_batch, second_batch)
        self.recapture()

    def prime(self, batch, batch_after=None):
        """(Re)start the pipeline: `batch` becomes the current batch and `batch_after` the one
        after it; the geometry of the first and SA1's geometry of the second are computed now."""
        if batch_after is None:
            batch_after = batch
        super().prime(batch)
        self.next.copy_(batch_after)
        xyz = self._xyz(self.next)
        lv = self.backbone.geometry_prepass(xyz, side=self.side, first=0, last=0)
        torch.cuda.current_stream().wait_stream(self.side)
        fresh = {k: lv[0][k] for k in self._keys(lv[0])}
        if self.geo_a_next is None:
            self.geo_a_next = {k: v.clone() for k, v in fresh.items()}
        else:
            for k in self.geo_a_next:
                self.geo_a_next[k].copy_(fresh[k])

    def _pipelined(self):
        main = torch.cuda.current_stream()
        xyz_next2 = self._xyz(self.next2)     # referenced until the side streams are joined
        box = {}

        lvl0 = dict(self.geo_a_next, event=None, sm_limit=0)

        def launch_a():
            box["a"] = self.backbone.geometry_prepass(xyz_next2, fps_cluster=self.fps_cluster,
                                                      sm_limit=0, side=self.side, first=0, last=0)
            if not self.b_from_start:
                launch_b()

        def launch_b():   # one-CTA-per-scene FPS launches: 8 SMs + the ball queries
            box["b"] = self.backbone.geometry_prepass(self.geo_a_next["new_xyz"], sm_limit=0,
                                                      side=self.side_b, first=1, last=3, prev=[lvl0])

        if self.b_from_start:
            launch_b()
        levels = self._levels(self.geo_cur)
        if self.start_after_level is None:
            launch_a()
        else:
            levels[self.start_after_level]["after_forward"] = launch_a
        step_arena.begin(self.cur.device)
        try:
            loss = self.step_fn(self.cur, levels)
        finally:
            step_arena.end(self.cur.device)
        if "a" not in box:
            launch_a()
        geo_b = box["b"]
        main.wait_stream(self.side)
        main.wait_stream(self.side_b)
        del xyz_next2
        # rotate: (SA1 geometry of next, fresh later levels) -> current; fresh SA1 geometry -> next
        dsts, srcs = [], []
        for dst, src in zip(self.geo_cur, [self.geo_a_next] + geo_b[1:]):
            for k in dst:
                dsts.append(dst[k])
                srcs.append(src[k])
        torch._foreach_copy_(dsts + [self.cur], srcs + [self.next])
        keys = list(self.geo_a_next)
        torch._foreach_copy_([self.geo_a_next[k] for k in keys] + [self.next],
                             [box["a"][0][k] for k in keys] + [self.next2])
        return loss

    def __call__(self, batch_after_next, non_blocking=True):
        self.next2.copy_(batch_after_next, non_blocking=non_blocking)
        self.graph.replay()
        return self.static_loss


class HostPrefetcher:
    """Input staging (SURVEY.md 8f row 4): batches travel pinned host memory -> device on a COPY
    stream, one step ahead of their use, so the upload of the next batch overlaps the running
    step instead of preceding it on the compute stream (the reference uploads synchronously at
    the top of every iteration, train_Votenet_FSB.py:217-218).

        slot = pre.upload(host_batch)        # asynchronous, returns immediately
        ...
        batch = pre.get(slot)                # compute stream waits for that upload only
        loss = step(batch)
        pre.release(slot)                    # the slot may be overwritten once `step` has read it
    """

    def __init__(self, example, device, depth=2):
        self.stream = torch.cuda.Stream(device=device)
        self.bufs = [torch.empty(example.shape, dtype=example.dtype, device=device)
                     for _ in range(depth)]
        self.ready = [None] * depth
        self.free = [None] * depth
        self.i = 0
        self.bytes_uploaded = 0

    def upload(self, host_batch):
        slot = self.i
        self.i = (self.i + 1) % len(self.bufs)
        if self.free[slot] is not None:
            self.stream.wait_event(self.free[slot])
        with torch.cuda.stream(self.stream):
            self.bufs[slot].copy_(host_batch, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.stream)
        self.ready[slot] = ev
        self.bytes_uploaded += host_batch.numel() * host_batch.element_size()
        return slot

    def get(self, slot):
        torch.cuda.current_stream().wait_event(self.ready[slot])
        return self.bufs[slot]

    def release(self, slot):
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self.free[slot] = ev
