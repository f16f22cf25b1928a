"""Pointnet2Backbone (VoteNet and GroupFree3D flavours) on the B200-native ops.

Mirrors /root/reference/detection/Votenet/models/backbone_module.py:21-133 and
/root/reference/detection/GroupFree3D/models/backbone_module.py:21-138: four
PointnetSAModuleVotes (npoint 2048/1024/512/256, radius 0.2/0.4/0.8/1.2, nsample 64/32/16/16)
and two PointnetFPModule; identical hyper-parameters, end_points keys and state-dict layout
(SURVEY.md appendix B).  The only difference between the two flavours is the width of fp2's last
layer (256 vs 288), selected with `fp2_out`.
"""
import torch
import torch.nn as nn

from . import _ext, fused_sa, pointnet2_utils
from .pointnet2_modules import PointnetFPModule, PointnetSAModuleCenters, PointnetSAModuleVotes

# FPS, centre gather and ball query of ALL four levels depend only on xyz (SURVEY.md 7, step 8):
# run them as a chain on a side stream so that FPS of level l+1 overlaps the MLP of level l.
GEOMETRY_STREAM = True
# FPS runs one CTA (N <= 4096) per scene and cannot share an SM with an MLP CTA (which owns the
# whole register file), so the concurrent MLP kernels leave this many SMs free
GEOMETRY_SMS = 8
_GEO_STREAMS = {}   # device -> side stream (module-level: nn.Module copies stay picklable)
_QUERY_STREAMS = {}  # (device, side stream) -> second side stream (ball queries beside the next level's FPS)


class Pointnet2Backbone(nn.Module):
    """input_feature_dim: channels per point beyond xyz (1 = height for VoteNet, 0 for GF3D).
    fp2_out: 256 (VoteNet) or 288 (GroupFree3D).  width / depth: the GroupFree3D reference's
    channel multiplier and number of hidden layers per SA block (models/backbone_module.py:21-33);
    width=1, depth=2 is the published default and VoteNet's backbone, width=2 the "w2x" models.
    Layers too wide for one fused launch run as channel-slice launches (fused_sa.slice_grid)."""

    def __init__(self, input_feature_dim=0, fp2_out=256, width=1, depth=2):
        super().__init__()
        if int(width) != width or width < 1 or int(depth) != depth or depth < 1:
            raise ValueError("width and depth must be integers >= 1 (got %r, %r)" % (width, depth))
        w, d = int(width), int(depth)
        self.width, self.depth = w, d
        self.sa1 = PointnetSAModuleVotes(npoint=2048, radius=0.2, nsample=64,
                                         mlp=[input_feature_dim] + [64 * w] * d + [128 * w],
                                         use_xyz=True, normalize_xyz=True)
        self.sa2 = PointnetSAModuleVotes(npoint=1024, radius=0.4, nsample=32,
                                         mlp=[128 * w] + [128 * w] * d + [256 * w],
                                         use_xyz=True, normalize_xyz=True)
        self.sa3 = PointnetSAModuleVotes(npoint=512, radius=0.8, nsample=16,
                                         mlp=[256 * w] + [128 * w] * d + [256 * w],
                                         use_xyz=True, normalize_xyz=True)
        self.sa4 = PointnetSAModuleVotes(npoint=256, radius=1.2, nsample=16,
                                         mlp=[256 * w] + [128 * w] * d + [256 * w],
                                         use_xyz=True, normalize_xyz=True)
        self.fp1 = PointnetFPModule(mlp=[512 * w, 256 * w, 256 * w])
        self.fp2 = PointnetFPModule(mlp=[512 * w, 256 * w, fp2_out])

    def _break_up_pc(self, pc):
        xyz = pc[..., 0:3].contiguous()
        features = pc[..., 3:].transpose(1, 2).contiguous() if pc.size(-1) > 3 else None
        return xyz, features

    def geometry_prepass(self, xyz, fps_cluster=0, sm_limit=None, side=None, first=0, last=3,
                         prev=None, copy_to=None, plan_splits=1, presorted=None):
        """inds / new_xyz / ball-query idx of sa1..sa4 for xyz (B,N,3), issued as one chain on a
        side stream with one event per level.  Returns the list of four per-level dicts that
        `forward(..., geometry=)` and `PointnetSAModuleVotes.forward(..., geometry=)` take.

        fps_cluster: CTAs per scene for the FPS launches (0 = lowest latency; a small number when
        the pre-pass belongs to the NEXT batch and runs beside this batch's step,
        train_step.PipelinedTrainStep).  sm_limit: cap of the MLP kernels that will consume each
        level (int, or (forward, backward) tuple); default leaves GEOMETRY_SMS free while a later
        level's FPS may still be running.
        first / last: compute only levels first..last (0-based; default all four).  With first > 0
        `xyz` is the new_xyz of level first-1 and `prev` the list of the earlier levels' dicts
        (returned in front of the new ones); the FP modules' interpolation weights are computed
        with level 3.  Lets a caller run SA1's geometry -- 2047 dependent FPS iterations over the
        whole scene -- and the later levels' as two independent chains
        (train_step.PipelinedTrainStep with depth 2).
        copy_to: optional list of four dicts of preallocated tensors; every level's results are
        also copied into copy_to[level][key] on the side streams as soon as they exist
        (train_step.PipelinedTrainStepPP: the static buffers of the NEXT graph, filled off the
        critical path).
        presorted: `_ext.fps_presort(xyz)` of the same xyz, when the caller ran the first level's
        spatial sort ahead of time (it depends on the coordinates only).
        plan_splits: k > 1 builds the pad-free plans per batch slice (keys "cidx#i", "ccen#i",
        "cmeta#i"): the batch will be consumed as k separate forwards (`split_geometry`; the BR step
        of train_Votenet_BR.py:277-289 runs the source and the target half one after the other)."""
        main = torch.cuda.current_stream()
        if side is None:
            side = _GEO_STREAMS.get(xyz.device)
            if side is None:
                side = _GEO_STREAMS[xyz.device] = torch.cuda.Stream(device=xyz.device)
        side.wait_stream(main)
        # ball query + pad-free plan of a level run on a SECOND side stream, beside the next
        # level's FPS (both only need this level's centres): the serial FPS chain
        # sa1 -> sa2 -> sa3 -> sa4 is the longest dependency chain of the pre-pass
        qkey = (xyz.device, side.cuda_stream)     # one per side stream: independent chains
        query = _QUERY_STREAMS.get(qkey)          # (train_step.PipelinedTrainStep2) stay independent
        if query is None:
            query = _QUERY_STREAMS[qkey] = torch.cuda.Stream(device=xyz.device)
        levels, cur = list(prev) if prev is not None else [], xyz
        assert len(levels) == first
        fp, fp_ev = {}, None
        with torch.cuda.stream(side), torch.no_grad():
            for sa in (self.sa1, self.sa2, self.sa3, self.sa4)[first:last + 1]:
                inds = _ext.furthest_point_sampling(cur, sa.npoint, cluster=fps_cluster,
                                                    presorted=presorted if cur is xyz else None)
                new_xyz = pointnet2_utils.gather_operation(
                    cur.transpose(1, 2).contiguous(), inds).transpose(1, 2).contiguous()
                query.wait_stream(side)
                with torch.cuda.stream(query):
                    idx = pointnet2_utils.ball_query(sa.radius, sa.nsample, cur, new_xyz)
                    # the block's pad-free position space (fused_sa.compact_plan) is geometry too
                    plan = {}
                    if fused_sa.ENABLED and fused_sa.compact_wanted(sa.nsample):
                        if plan_splits <= 1:
                            plan = fused_sa.compact_plan(idx, cur.shape[1])
                        else:
                            per = idx.shape[0] // plan_splits
                            for i in range(plan_splits):
                                part = fused_sa.compact_plan(idx[i * per:(i + 1) * per], cur.shape[1])
                                plan.update({"%s#%d" % (k, i): v for k, v in part.items()})
                    if copy_to is not None:
                        dst = copy_to[len(levels)]
                        keys = [k for k in dst if k in plan or k in ("inds", "new_xyz", "idx")]
                        src = dict(plan, inds=inds, new_xyz=new_xyz, idx=idx)
                        torch._foreach_copy_([dst[k] for k in keys], [src[k] for k in keys])
                    ev = torch.cuda.Event()
                    ev.record(query)
                    # the FP modules' 3-NN indices and inverse-distance weights are geometry too
                    # (fp2 interpolates sa3 -> sa2, fp1 sa4 -> sa3): on THIS stream as soon as their
                    # two levels' centres exist, not at the tail of the FPS chain
                    li = len(levels)
                    if last == 3 and li == 2:
                        fp["fp2_idx"], fp["fp2_weight"] = PointnetFPModule.interpolation_weights(
                            levels[1]["new_xyz"], new_xyz)
                    if last == 3 and li == 3:
                        fp["fp1_idx"], fp["fp1_weight"] = PointnetFPModule.interpolation_weights(
                            levels[2]["new_xyz"], new_xyz)
                        fp_ev = torch.cuda.Event()
                        fp_ev.record(query)
                cur.record_stream(query)
                new_xyz.record_stream(query)
                for t in (inds, new_xyz, idx) + tuple(plan.values()):
                    t.record_stream(main)
                levels.append(dict(plan, inds=inds, new_xyz=new_xyz, idx=idx, event=ev,
                                   sm_limit=(fused_sa.NUM_SMS - GEOMETRY_SMS) if sm_limit is None
                                   else sm_limit))
                cur = new_xyz
            if last == 3:
                for t in fp.values():
                    t.record_stream(main)
                levels[3].update(fp, fp_event=fp_ev)
                if copy_to is not None:
                    with torch.cuda.stream(query):
                        fpk = [k for k in fp if k in copy_to[3]]
                        torch._foreach_copy_([copy_to[3][k] for k in fpk], [fp[k] for k in fpk])
            side.wait_stream(query)       # joining `side` joins the whole pre-pass
        if sm_limit is None:
            levels[-1]["sm_limit"] = 0   # nothing runs beside sa4's MLP
        return levels

    @staticmethod
    def split_geometry(levels, nsplit):
        """The pre-pass of a batch that is consumed as `nsplit` consecutive forwards over equal
        batch slices (geometry_prepass(..., plan_splits=nsplit)) -> one list of four level dicts
        per slice.  Index tensors are leading-dimension views; the `after_forward` hook of a level
        (train_step.PipelinedTrainStep) goes with the FIRST slice."""
        out = []
        for i in range(nsplit):
            part = []
            for lv in levels:
                d = {}
                for k, v in lv.items():
                    if "#" in k:
                        base, j = k.split("#")
                        if int(j) == i:
                            d[base] = v
                    elif torch.is_tensor(v) and k in ("inds", "new_xyz", "idx", "fp1_idx", "fp1_weight",
                                                      "fp2_idx", "fp2_weight"):
                        per = v.shape[0] // nsplit
                        d[k] = v[i * per:(i + 1) * per]
                    elif k == "after_forward":
                        if i == 0:
                            d[k] = v
                    else:
                        d[k] = v
                part.append(d)
            out.append(part)
        return out

    @staticmethod
    def _after_forward(level):
        """hook of a pre-computed geometry level: called once its SA block has been issued
        (train_step.PipelinedTrainStep starts the next batch's pre-pass from here)"""
        if isinstance(level, dict) and level.get("after_forward") is not None:
            level["after_forward"]()

    def forward(self, pointcloud: torch.Tensor, end_points=None, geometry=None):
        """pointcloud (B,N,3+input_feature_dim) -> end_points dict (sa{1..4}_xyz/features,
        sa1_inds, sa2_inds, fp2_features, fp2_xyz, fp2_inds).  `geometry` (not in the reference's
        signature): the result of `geometry_prepass` for this point cloud when it was computed
        ahead of time (e.g. during the previous step)."""
        if not end_points:
            end_points = {}
        xyz, features = self._break_up_pc(pointcloud)
        if xyz.is_cuda and fused_sa.ENABLED and not end_points.get('_prepacked'):
            # weight images of the four SA blocks, packed on a side stream beside the first kernels
            fused_sa.prepack([m.mlp_module for m in (self.sa1, self.sa2, self.sa3, self.sa4)])
        geo = [None] * 4
        if geometry is not None:
            geo = geometry
        elif (GEOMETRY_STREAM and xyz.is_cuda and not xyz.requires_grad
                and all(m.fusable(xyz) for m in (self.sa1, self.sa2, self.sa3, self.sa4))):
            geo = self.geometry_prepass(xyz)

        # consecutive fused blocks hand their activations (and, in backward, their gradients) to
        # each other point-major: no layout-conversion kernels between sa1 -> sa2 -> sa3 -> sa4
        chain = all(isinstance(g, dict) for g in geo)
        if chain:
            geo = [dict(g) for g in geo]            # never mutate the caller's dicts
            for g in geo:
                g["want_pm"] = True
        pm = {}      # point-major copies of sa2..sa4's features, for the dense FP path

        xyz, features, fps_inds = self.sa1(xyz, features, geometry=geo[0])
        end_points['sa1_inds'] = fps_inds
        end_points['sa1_xyz'] = xyz
        end_points['sa1_features'] = features
        self._after_forward(geo[0])
        if chain:
            geo[1]["features_pm"] = geo[0].pop("out_pm", None)

        xyz, features, fps_inds = self.sa2(xyz, features, geometry=geo[1])
        end_points['sa2_inds'] = fps_inds
        end_points['sa2_xyz'] = xyz
        end_points['sa2_features'] = features
        self._after_forward(geo[1])
        if chain:
            pm[2] = geo[2]["features_pm"] = geo[1].pop("out_pm", None)

        xyz, features, fps_inds = self.sa3(xyz, features, geometry=geo[2])
        end_points['sa3_xyz'] = xyz
        end_points['sa3_features'] = features
        self._after_forward(geo[2])
        if chain:
            pm[3] = geo[3]["features_pm"] = geo[2].pop("out_pm", None)

        xyz, features, fps_inds = self.sa4(xyz, features, geometry=geo[3])
        end_points['sa4_xyz'] = xyz
        end_points['sa4_features'] = features
        self._after_forward(geo[3])
        if chain:
            pm[4] = geo[3].pop("out_pm", None)

        interp1 = interp2 = None
        if geo[3] is not None and "fp1_idx" in geo[3]:
            if geo[3].get("fp_event") is not None:
                torch.cuda.current_stream().wait_event(geo[3]["fp_event"])
            interp1 = (geo[3]["fp1_idx"], geo[3]["fp1_weight"])
            interp2 = (geo[3]["fp2_idx"], geo[3]["fp2_weight"])
        fp2_pm = None
        if all(pm.get(k) is not None for k in (2, 3, 4)):
            # dense tcgen05 FP path on the blocks' point-major outputs (no transposes in between)
            r1 = self.fp1.forward_pm(end_points['sa3_xyz'], end_points['sa4_xyz'], pm[3], pm[4],
                                     interp=interp1)
            r2 = None if r1 is None else self.fp2.forward_pm(
                end_points['sa2_xyz'], end_points['sa3_xyz'], pm[2], r1[1], interp=interp2)
            if r2 is not None:
                features, fp2_pm = r2
        if fp2_pm is None:
            features = self.fp1(end_points['sa3_xyz'], end_points['sa4_xyz'],
                                end_points['sa3_features'], end_points['sa4_features'],
                                interp=interp1)
            features = self.fp2(end_points['sa2_xyz'], end_points['sa3_xyz'],
                                end_points['sa2_features'], features, interp=interp2)
        end_points['fp2_features'] = features
        if fp2_pm is not None:
            end_points['fp2_features_pm'] = fp2_pm      # (B,1024,C): for the voting module
        end_points['fp2_xyz'] = end_points['sa2_xyz']
        num_seed = end_points['fp2_xyz'].shape[1]
        end_points['fp2_inds'] = end_points['sa1_inds'][:, 0:num_seed]
        if not end_points.pop('_prepacked', False):
            fused_sa.prepack_join()
        return end_points


class Pointnet2Backbone_jitter(Pointnet2Backbone):
    """The CenterRefine backbone (reference models/backbone_module.py:136-262): Pointnet2Backbone
    plus `ctjt_head`, a PointnetSAModuleCenters(npoint=64, radius=0.8, nsample=16, mlp=[256,128],
    normalize_xyz=False) that pools the fp2 seed features around externally supplied (jittered)
    object centres and appends their one-hot class.  Same sub-module names / state-dict keys.

    forward(pointcloud, center_xyz (B,64,3) | None, center_cls (B,64) int | None, end_points)
        -> end_points (+ 'center_features' (B, 128 + 22, 64) when center_xyz is given)
    """
    NUM_CLASS = 22    # torch.eye(22) in the reference (:260)

    def __init__(self, input_feature_dim=0):
        super().__init__(input_feature_dim=input_feature_dim, fp2_out=256)
        self.ctjt_head = PointnetSAModuleCenters(npoint=64, radius=0.8, nsample=16, mlp=[256, 128],
                                                 use_xyz=True, normalize_xyz=False)

    def forward(self, pointcloud, center_xyz=None, center_cls=None, end_points=None, geometry=None):
        end_points = super().forward(pointcloud, end_points, geometry=geometry)
        if center_xyz is not None:
            center_features = self.ctjt_head(end_points['sa2_xyz'], end_points['fp2_features'],
                                             center_xyz)
            onehot = torch.eye(self.NUM_CLASS, device=center_features.device)[center_cls.long()]
            end_points['center_features'] = torch.cat([center_features, onehot.transpose(1, 2)], dim=1)
        return end_points
