"""Networks on the hot path, mirroring the reference's callers of the SA/FP modules.

PointNet2SemSeg         model/pointnet2.py:131-162              (ScanNet SSG semseg -- the benchmark model)
PointNet2Backbone       model/pointmaskrcnn.py:8-32             (nuScenes backbone `PointNet2`)
PointNet2Multiview2     model/pointnet2multiview.py:61-121      (multi-view semseg, point branch; ENet is out of scope)
PointNet2Multiview2Msg  model/pointnet2multiview.py:179-233     (the MSG semseg stack, point branch)

Attribute names match the reference so its state_dicts load unchanged.  In eval mode under
torch.no_grad() the forward is 17 kernel launches (2 layout transposes, 4 x (FPS+gather, ball
query, fused SA), 4 x (three_nn+weights, fused FP; the head is folded into the last FP block) -- the reference issues ~170
(SURVEY.md 3.2).  Otherwise (training, or eval under autograd) the modules' training paths run: block Functions on
the fused training kernels, each BatchNorm in its own mode (batch or running statistics) as in torch.
"""
import threading

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import pointnet2_utils
from .pointnet_util import (PointNetFeaturePropagation, PointNetSetAbstraction, PointNetSetAbstractionMsg, SpatialGrid, _FoldCache, _fusable, fps_gather_cl, fps_policy,
                            get_mlp_precision, grid_max_points, three_nn_weights_cl,
                            to_channel_last)


def _semseg_head(model, l0_points):
    """conv1 -> bn1 -> ReLU -> dropout -> conv2 -> (B, N, classes) (model/pointnet2.py:158-161).  In training mode, and in
    eval mode under autograd, on the fused training kernels: conv1 + BatchNorm (batch or running statistics, as bn1's mode
    says) + ReLU as one row chain, conv2 as a row GEMM (no 1x1 cuDNN convolutions)."""
    from . import pointnet_util, train_mlp
    if pointnet_util._train_fused(model, l0_points, [model.conv1], [model.bn1]):
        B, C, N = l0_points.shape
        rows = l0_points.permute(0, 2, 1).reshape(B * N, C)
        x = train_mlp.fused_mlp_train(rows, [model.conv1], [model.bn1])
        x = model.drop1(x)
        x = F.linear(x, model.conv2.weight.reshape(model.conv2.out_channels, -1), model.conv2.bias)
        return x.view(B, N, -1)
    x = model.drop1(F.relu(model.bn1(model.conv1(l0_points))))
    x = model.conv2(x)
    return x.permute(0, 2, 1)


class PointNet2SemSeg(nn.Module):
    def __init__(self, num_classes):
        super().__init__()
        self.sa1 = PointNetSetAbstraction(1024, 0.1, 32, 3 + 3, [32, 32, 64], False)
        self.sa2 = PointNetSetAbstraction(256, 0.2, 32, 64 + 3, [64, 64, 128], False)
        self.sa3 = PointNetSetAbstraction(64, 0.4, 32, 128 + 3, [128, 128, 256], False)
        self.sa4 = PointNetSetAbstraction(16, 0.8, 32, 256 + 3, [256, 256, 512], False)
        self.fp4 = PointNetFeaturePropagation(768, [256, 256])
        self.fp3 = PointNetFeaturePropagation(384, [256, 256])
        self.fp2 = PointNetFeaturePropagation(320, [256, 128])
        self.fp1 = PointNetFeaturePropagation(128 + 3, [128, 128, 128])
        self.conv1 = nn.Conv1d(128, 128, 1)
        self.bn1 = nn.BatchNorm1d(128)
        self.drop1 = nn.Dropout(0.5)
        self.conv2 = nn.Conv1d(128, num_classes, 1)
        self._head_fold = _FoldCache()
        self.timers = None  # bench.py: dict name -> [(start_event, end_event)] recorded on the current stream
        self._streams = {}  # device index -> (sampling stream, ball-query stream); shared by DataParallel replicas
        self._streams_lock = threading.Lock()
        self.single_stream = False

    def train(self, mode=True):
        self._head_fold.clear()
        return super().train(mode)

    def __getstate__(self):
        state = self.__dict__.copy()
        state["_streams"], state["_streams_lock"] = {}, None
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)
        self._streams_lock = threading.Lock()

    def __deepcopy__(self, memo):
        import copy
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k == "_streams":
                new.__dict__[k] = {}
            elif k == "_streams_lock":
                new.__dict__[k] = threading.Lock()
            else:
                new.__dict__[k] = copy.deepcopy(v, memo)
        return new

    @property
    def compute_dtype(self):
        return "bf16" if get_mlp_precision() == "bf16" else "f32"

    def _fp1_with_head(self):
        """fp1's three layers + conv1/bn1/relu (+ eval dropout = identity) + conv2 as ONE fused stack."""
        convs = list(self.fp1.mlp_convs) + [self.conv1, self.conv2]
        bns = list(self.fp1.mlp_bns) + [self.bn1, None]
        relus = [True] * len(self.fp1.mlp_convs) + [True, False]
        return self._head_fold.get(self, convs, bns, relus)

    def forward_fused(self, xyz, points, labels=False, logits_dtype=torch.float32):
        """xyz (B, 3, N), points (B, D, N) -> (B, N, num_classes), contiguous; labels=True -> (B, N) uint8 class
        predictions (arg-max fused into the head, see predict()); logits_dtype=torch.bfloat16 (tensor-core path only) stores
        the logits as bf16 -- they carry bf16-MMA precision anyway -- which halves what an evaluation loop reads back.

        The geometry of every level depends on coordinates only, so it runs ahead of the feature path on two side
        streams: FPS chain + 3-NN on one, ball queries on another; the fused SA/FP kernels follow on the caller's
        stream as their indices become ready.  No collective, no host synchronisation."""
        main = torch.cuda.current_stream(xyz.device)
        with self._streams_lock:
            pair = self._streams.get(xyz.device.index)
            if pair is None:
                pair = self._streams[xyz.device.index] = (torch.cuda.Stream(xyz.device), torch.cuda.Stream(xyz.device))
        s_fps, s_bq = pair
        if self.single_stream:  # developer profiling: everything on the caller's stream
            s_fps = s_bq = main
        xyz_cl, feat_cl = to_channel_last(xyz), to_channel_last(points)
        sas = [self.sa1, self.sa2, self.sa3, self.sa4]
        fps_done, bq_done, nn_done = [], [], []
        start = torch.cuda.Event()
        start.record(main)
        keep = []  # tensors produced on side streams and consumed on the main stream

        def use_grid(npts):
            return 2048 <= npts <= grid_max_points()

        grids = {}
        with torch.cuda.stream(s_bq):
            s_bq.wait_event(start)
            if use_grid(xyz_cl.shape[1]):
                # level-0 cell list: independent of the sampling, so it is built while FPS runs
                grids[0] = SpatialGrid(xyz_cl, 1.01 * sas[0].radius)
            g0_done = torch.cuda.Event()
            g0_done.record(s_bq)
        with torch.cuda.stream(s_fps):
            s_fps.wait_event(start)
            levels = [xyz_cl]
            for sa in sas:
                _, new_xyz = fps_gather_cl(levels[-1], sa.npoint)
                levels.append(new_xyz)
                ev = torch.cuda.Event()
                ev.record(s_fps)
                fps_done.append(ev)
        with torch.cuda.stream(s_bq):
            balls = []
            for i, sa in enumerate(sas):
                s_bq.wait_event(fps_done[i])
                if i == 0 and 0 in grids:
                    balls.append(grids[0].ball_query(sa.radius, sa.nsample, levels[1]))
                else:
                    balls.append(pointnet2_utils.BallQuery.brute_force(sa.radius, sa.nsample, levels[i], levels[i + 1]))
                ev = torch.cuda.Event()
                ev.record(s_bq)
                bq_done.append(ev)
        with torch.cuda.stream(s_fps):
            nnw = []
            s_fps.wait_event(g0_done)
            for lvl in (3, 2, 1, 0):  # fp4 .. fp1: fine level `lvl`, coarse level `lvl + 1`
                m_known = levels[lvl + 1].shape[1]
                if m_known <= 1:
                    nnw.append(None)
                elif 512 <= m_known <= grid_max_points():
                    known_grid = SpatialGrid(levels[lvl + 1], 0.0)  # automatic cell: about one point per cell
                    grids["nn%d" % lvl] = known_grid
                    nnw.append(known_grid.three_nn(levels[lvl], query_order=grids[lvl].order if lvl in grids else None))
                else:
                    nnw.append(three_nn_weights_cl(levels[lvl], levels[lvl + 1]))
                ev = torch.cuda.Event()
                ev.record(s_fps)
                nn_done.append(ev)
        for gr in grids.values():
            keep += gr.tensors()
        keep += levels[1:] + balls + [t for pair in nnw if pair is not None for t in pair]
        if not torch.cuda.is_current_stream_capturing():
            # eager mode: these tensors are produced on one stream and read on others; tell the caching allocator
            # about every consumer stream so their memory is not reused while a consumer is still queued
            for t in keep:
                for st in (main, s_fps, s_bq):
                    t.record_stream(st)
            for t in (xyz_cl, feat_cl):
                if t is not None:
                    t.record_stream(s_fps)
                    t.record_stream(s_bq)

        # activations between tensor-core blocks travel as bf16 (they are rounded to bf16 for the MMA operand anyway;
        # halves the gather traffic).  Only when every block of the network runs on the tensor-core path.
        blocks = [sa.folded() for sa in sas] + [self.fp4.folded(), self.fp3.folded(), self.fp2.folded(), self._fp1_with_head()]
        act = torch.bfloat16 if (get_mlp_precision() == "bf16" and all(b.bf16_ok() for b in blocks)) else torch.float32
        feats = [feat_cl]
        for i, sa in enumerate(sas):
            main.wait_event(bq_done[i])
            _, out = sa.forward_cl(levels[i], feats[i], geometry=(levels[i + 1], balls[i]), out_dtype=act)
            feats.append(out)
        l1, l2, l3, l4 = feats[1:]
        main.wait_event(nn_done[0])
        l3 = self.fp4.forward_cl(levels[3], levels[4], l3, l4, nn_weights=nnw[0], out_dtype=act)
        main.wait_event(nn_done[1])
        l2 = self.fp3.forward_cl(levels[2], levels[3], l2, l3, nn_weights=nnw[1], out_dtype=act)
        main.wait_event(nn_done[2])
        l1 = self.fp2.forward_cl(levels[1], levels[2], l1, l2, nn_weights=nnw[2], out_dtype=act)
        main.wait_event(nn_done[3])
        order0 = grids[0].order if 0 in grids else None
        head_dtype = torch.uint8 if labels else logits_dtype
        if self.timers is None:
            return self.fp1.forward_cl(xyz_cl, levels[1], feat_cl, l1, mlp=self._fp1_with_head(), nn_weights=nnw[3],
                                       row_order=order0, out_dtype=head_dtype)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        out = self.fp1.forward_cl(xyz_cl, levels[1], feat_cl, l1, mlp=self._fp1_with_head(), nn_weights=nnw[3],
                                  row_order=order0, out_dtype=head_dtype)
        t1.record()
        self.timers.setdefault("fp1_head", []).append((t0, t1))
        return out

    def can_fuse_labels(self):
        return get_mlp_precision() == "bf16" and self._fp1_with_head().bf16_ok() and self.conv2.out_channels <= 256

    def predict(self, xyz, points):
        """Per-point class predictions (B, N) uint8 = arg-max over the logits, what the reference's evaluation loop
        computes on the host from `pred.cpu().numpy()` (train_scannet_semseg.py:204-205).  In inference on the
        tensor-core path the arg-max is fused into the head kernel: the logits are never written and the result to
        read back is 1 byte per point instead of 84."""
        if _fusable(self, xyz, points) and self.can_fuse_labels():
            return self.forward_fused(xyz, points, labels=True)
        logits = self.forward(xyz, points)
        # first maximum, as numpy.argmax (torch.argmax does not promise an order among ties)
        classes = torch.arange(logits.shape[-1], device=logits.device)
        first = torch.where(logits == logits.max(dim=-1, keepdim=True).values, classes, logits.shape[-1]).min(dim=-1).values
        return first.to(torch.uint8)

    def forward(self, xyz, points):
        if _fusable(self, xyz, points):
            return self.forward_fused(xyz, points)
        l1_xyz, l1_points = self.sa1(xyz, points)
        l2_xyz, l2_points = self.sa2(l1_xyz, l1_points)
        l3_xyz, l3_points = self.sa3(l2_xyz, l2_points)
        l4_xyz, l4_points = self.sa4(l3_xyz, l3_points)
        l3_points = self.fp4(l3_xyz, l4_xyz, l3_points, l4_points)
        l2_points = self.fp3(l2_xyz, l3_xyz, l2_points, l3_points)
        l1_points = self.fp2(l1_xyz, l2_xyz, l1_points, l2_points)
        l0_points = self.fp1(xyz, l1_xyz, points, l1_points)
        return _semseg_head(self, l0_points)


class PointNet2Backbone(nn.Module):
    """The nuScenes backbone (`PointNet2`, model/pointmaskrcnn.py:8-32): xyz (B,3,N), points (B,2,N) ->
    (B, 128, N) per-point features."""

    def __init__(self):
        super().__init__()
        self.sa1 = PointNetSetAbstraction(4096, 1.0, 32, 2 + 3, [32, 32, 64], False)
        self.sa2 = PointNetSetAbstraction(1024, 2.0, 32, 64 + 3, [64, 64, 128], False)
        self.sa3 = PointNetSetAbstraction(256, 4.0, 32, 128 + 3, [128, 128, 256], False)
        self.sa4 = PointNetSetAbstraction(64, 8.0, 32, 256 + 3, [256, 256, 512], False)
        self.fp4 = PointNetFeaturePropagation(768, [256, 256])
        self.fp3 = PointNetFeaturePropagation(384, [256, 256])
        self.fp2 = PointNetFeaturePropagation(320, [256, 128])
        self.fp1 = PointNetFeaturePropagation(128, [128, 128, 128])

    def forward_fused(self, xyz, points):
        """-> (B, N, 128) channel-last.  Cell lists serve the ball queries (clouds up to grid_max_points()), every 3-NN
        whose coarse set has >= 512 points, and the processing order of fp1's rows; activations between tensor-core
        blocks travel as bf16."""
        xyz_cl, feat_cl = to_channel_last(xyz), to_channel_last(points)
        sas = [self.sa1, self.sa2, self.sa3, self.sa4]
        fps_ = [self.fp4, self.fp3, self.fp2, self.fp1]
        blocks = [m.folded() for m in sas + fps_]
        act = torch.bfloat16 if (get_mlp_precision() == "bf16" and all(b.bf16_ok() for b in blocks)) else torch.float32
        levels, feats, grids = [xyz_cl], [feat_cl], {}
        for i, sa in enumerate(sas):
            cur = levels[-1]
            if 2048 <= cur.shape[1] <= grid_max_points():
                grids[i] = SpatialGrid(cur, 1.01 * sa.radius)
            _, new_xyz = fps_gather_cl(cur, sa.npoint)
            ball = (grids[i].ball_query(sa.radius, sa.nsample, new_xyz) if i in grids
                    else pointnet2_utils.ball_query(sa.radius, sa.nsample, cur, new_xyz))
            _, out = sa.forward_cl(cur, feats[-1], geometry=(new_xyz, ball), out_dtype=act)
            levels.append(new_xyz)
            feats.append(out)
        up = feats[4]
        for j, fp in enumerate(fps_):  # fine level 3, 2, 1, 0
            lvl = 3 - j
            fine, coarse = levels[lvl], levels[lvl + 1]
            order = grids[lvl].order if lvl in grids else None
            nnw = None
            # lidar sweeps are far from uniform (rings, dense near the sensor); with ring doubling the cell-list search
            # still beats the brute-force scan: 0.12 vs 1.23 ms at 34720 x 4096, 0.035 (+ 0.017 build) vs 0.066 at 4096 x 1024
            if 512 <= coarse.shape[1] <= grid_max_points():
                nnw = SpatialGrid(coarse, 0.0).three_nn(fine, query_order=order)
            skip = feats[lvl] if lvl > 0 else None
            up = fp.forward_cl(fine, coarse, skip, up, nn_weights=nnw, row_order=order if lvl == 0 else None,
                               out_dtype=act if lvl > 0 else torch.float32)
        return up

    def forward(self, xyz, points):
        if _fusable(self, xyz, points):
            return self.forward_fused(xyz, points).permute(0, 2, 1)
        l1_xyz, l1_points = self.sa1(xyz, points)
        l2_xyz, l2_points = self.sa2(l1_xyz, l1_points)
        l3_xyz, l3_points = self.sa3(l2_xyz, l2_points)
        l4_xyz, l4_points = self.sa4(l3_xyz, l3_points)
        l3_points = self.fp4(l3_xyz, l4_xyz, l3_points, l4_points)
        l2_points = self.fp3(l2_xyz, l3_xyz, l2_points, l3_points)
        l1_points = self.fp2(l1_xyz, l2_xyz, l1_points, l2_points)
        return self.fp1(xyz, l1_xyz, None, l1_points)


_BRANCH_STREAMS = {}  # device index -> side stream of _MultiviewStackBase._two_branches (process-wide, not module state)
_BRANCH_LOCK = threading.Lock()


class _MultiviewStackBase(nn.Module):
    """Shared plumbing of the multi-view networks' point branch (everything after ENet + lifting):
    geometry branch on xyz only, feature branch on the lifted image features, concatenated at level 2."""

    reduce = "max"

    def train(self, mode=True):
        self._head_fold.clear()
        return super().train(mode)

    def _head(self, l0_points):
        return _semseg_head(self, l0_points)

    def _fp1_with_head(self):
        convs = list(self.fp1.mlp_convs) + [self.conv1, self.conv2]
        bns = list(self.fp1.mlp_bns) + [self.bn1, None]
        relus = [True] * len(self.fp1.mlp_convs) + [True, False]
        return self._head_fold.get(self, convs, bns, relus)

    def _blocks(self):
        mods = [self.sa1_geo, self.sa1_feat, self.sa2_geo, self.sa2_feat, self.sa3, self.sa4]
        out = []
        for m in mods:
            out += [m.folded(i) for i in range(len(m.radius_list))] if hasattr(m, "radius_list") else [m.folded()]
        return out + [self.fp4.folded(), self.fp3.folded(), self.fp2.folded(), self._fp1_with_head()]

    def can_fuse_labels(self):
        return get_mlp_precision() == "bf16" and self._fp1_with_head().bf16_ok() and self.conv2.out_channels <= 256

    def forward_fused(self, xyz, image_features, labels=False):
        """Channel-last fused path; the two level-1/level-2 branches share ONE sampling and ball query each
        (the reference recomputes them on identical coordinates, model/pointnet2multiview.py:104-107).  As in
        PointNet2SemSeg.forward_fused: one cell list of the input cloud serves the level-0 ball queries, the 3-NN of fp1
        and the processing order of its rows; activations between tensor-core blocks travel as bf16."""
        xyz_cl = to_channel_last(xyz)
        act = torch.bfloat16 if (get_mlp_precision() == "bf16" and all(b.bf16_ok() for b in self._blocks())) else torch.float32
        # the lifted features are rounded to bf16 for the MMA operand anyway: converting while transposing is bit-identical
        img_cl = image_features.permute(0, 2, 1).to(act).contiguous() if act == torch.bfloat16 else to_channel_last(image_features)
        n0 = xyz_cl.shape[1]
        radii0 = self.sa1_geo.radius_list if hasattr(self.sa1_geo, "radius_list") else [self.sa1_geo.radius]
        g0 = SpatialGrid(xyz_cl, 1.01 * max(radii0)) if 2048 <= n0 <= grid_max_points() else None
        geo1 = self._geometry(self.sa1_geo, xyz_cl, g0)
        l1_xyz, l1g = self.sa1_geo.forward_cl(xyz_cl, None, geometry=geo1, out_dtype=act)
        _, l1f = self.sa1_feat.forward_cl(xyz_cl, img_cl, geometry=geo1, out_dtype=act)
        geo2 = self._geometry(self.sa2_geo, l1_xyz)
        l2_xyz, l2g = self.sa2_geo.forward_cl(l1_xyz, l1g, geometry=geo2, out_dtype=act)
        _, l2f = self.sa2_feat.forward_cl(l1_xyz, l1f, geometry=geo2, out_dtype=act)
        l2 = torch.cat((l2g, l2f), dim=2)
        l3_xyz, l3 = self.sa3.forward_cl(l2_xyz, l2, out_dtype=act)
        l4_xyz, l4 = self.sa4.forward_cl(l3_xyz, l3, out_dtype=act)
        l3 = self.fp4.forward_cl(l3_xyz, l4_xyz, l3, l4, out_dtype=act)
        l2 = self.fp3.forward_cl(l2_xyz, l3_xyz, l2, l3, out_dtype=act)
        l1 = self.fp2.forward_cl(l1_xyz, l2_xyz, l1g, l2, out_dtype=act)
        nnw = None
        if g0 is not None and 512 <= l1_xyz.shape[1] <= grid_max_points():
            nnw = SpatialGrid(l1_xyz, 0.0).three_nn(xyz_cl, query_order=g0.order)
        return self.fp1.forward_cl(xyz_cl, l1_xyz, None, l1, mlp=self._fp1_with_head(), nn_weights=nnw,
                                   row_order=g0.order if g0 is not None else None,
                                   out_dtype=torch.uint8 if labels else torch.float32)

    def predict(self, xyz, image_features):
        """Per-point class predictions (B, N) uint8; see PointNet2SemSeg.predict."""
        if _fusable(self, xyz, image_features) and self.can_fuse_labels():
            return self.forward_fused(xyz, image_features, labels=True)
        logits = self.forward(xyz, image_features)
        classes = torch.arange(logits.shape[-1], device=logits.device)
        return torch.where(logits == logits.max(dim=-1, keepdim=True).values, classes, logits.shape[-1]).min(dim=-1).values.to(torch.uint8)

    @staticmethod
    def _geometry(sa, xyz_cl, grid=None):
        _, new_xyz = fps_gather_cl(xyz_cl, sa.npoint)

        def query(r, k):
            return grid.ball_query(r, k, new_xyz) if grid is not None else pointnet2_utils.ball_query(r, k, xyz_cl, new_xyz)

        if hasattr(sa, "radius_list"):
            return new_xyz, [query(r, k) for r, k in zip(sa.radius_list, sa.nsample_list)]
        return new_xyz, query(sa.radius, sa.nsample)

    def forward(self, xyz, image_features):
        """xyz (B, 3, N), image_features (B, 128, N) (lifted 2-D features) -> (B, N, num_classes)"""
        if _fusable(self, xyz, image_features):
            return self.forward_fused(xyz, image_features)
        if xyz.is_cuda and self.parallel_branches and self.sa1_geo.npoint == self.sa1_feat.npoint and self.sa2_geo.npoint == self.sa2_feat.npoint:
            two_streams = self.parallel_branches is True or (self.parallel_branches == "capture" and torch.cuda.is_current_stream_capturing())
            l1_xyz, l1_points, l2_xyz, l2_points, l2_points_feat = self._two_branches(xyz, image_features, two_streams)
        else:
            l1_xyz, l1_points = self.sa1_geo(xyz, None)
            l2_xyz, l2_points = self.sa2_geo(l1_xyz, l1_points)
            l1_xyz_feat, l1_points_feat = self.sa1_feat(xyz, image_features)
            _, l2_points_feat = self.sa2_feat(l1_xyz_feat, l1_points_feat)
        l2_points = torch.cat((l2_points, l2_points_feat), dim=1)
        l3_xyz, l3_points = self.sa3(l2_xyz, l2_points)
        l4_xyz, l4_points = self.sa4(l3_xyz, l3_points)
        l3_points = self.fp4(l3_xyz, l4_xyz, l3_points, l4_points)
        l2_points = self.fp3(l2_xyz, l3_xyz, l2_points, l3_points)
        l1_points = self.fp2(l1_xyz, l2_xyz, l1_points, l2_points)
        l0_points = self.fp1(xyz, l1_xyz, None, l1_points)
        return self._head(l0_points)

    # composed (training) path: one sampling for the geometry and the image-feature chain, and the two chains on two streams
    # -- "capture": only while a CUDA graph is being captured (GraphedTrainStep), True: always, False: the reference's order.
    # In an eager loop the step is bound by the host (~1000 launches) and the second stream costs host time (measured:
    # 17.1 -> 25.1 ms per eager step), in a replayed graph it shortens the chain of dependent nodes (11.4 -> 9.9 ms).
    parallel_branches = "capture"

    def _two_branches(self, xyz, image_features, two_streams):
        """sa1_geo -> sa2_geo and sa1_feat -> sa2_feat (model/pointnet2multiview.py:99-104) are independent chains that
        sample the SAME clouds: the reference runs them one after the other and samples twice.  Here the two samplings are
        done once (identical indices by construction), the image-feature chain runs on a side stream and the geometry
        chain on the caller's; autograd replays each backward on its forward stream, so the backward overlaps as well
        (the train step at 4 scenes per GPU is a chain of ~1000 small launches, not a throughput problem)."""
        dev = xyz.device
        main = torch.cuda.current_stream(dev)
        with _BRANCH_LOCK:
            side = _BRANCH_STREAMS.get(dev.index)
            if side is None:
                side = _BRANCH_STREAMS[dev.index] = torch.cuda.Stream(dev)
        xyz_c = xyz.permute(0, 2, 1).contiguous()
        fps1 = pointnet2_utils.furthest_point_sample(xyz_c, self.sa1_geo.npoint)
        l1_xyz = pointnet2_utils.gather_operation(xyz.contiguous(), fps1)          # (B, 3, S1) = both modules' new_xyz
        fps2 = pointnet2_utils.furthest_point_sample(l1_xyz.permute(0, 2, 1).contiguous(), self.sa2_geo.npoint)
        if not two_streams:
            side = main
        # (the side stream's chain is enqueued first; the two chains share no tensor that needs a gradient, so the order
        # in which they enter the autograd graph does not change any sum)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            l1_xyz_feat, l1_points_feat = self.sa1_feat(xyz, image_features, fps_idx=fps1)
            _, l2_points_feat = self.sa2_feat(l1_xyz_feat, l1_points_feat, fps_idx=fps2)
        l1_xyz_geo, l1_points = self.sa1_geo(xyz, None, fps_idx=fps1)
        l2_xyz, l2_points = self.sa2_geo(l1_xyz_geo, l1_points, fps_idx=fps2)
        main.wait_stream(side)
        if two_streams and not torch.cuda.is_current_stream_capturing():
            l2_points_feat.record_stream(main)  # allocated on the side stream, consumed on the caller's
        return l1_xyz_geo, l1_points, l2_xyz, l2_points, l2_points_feat

    def forward_views(self, xyz, feats, depth, camera_to_world, intrinsic, depth_min, depth_max, image_dims, accuracy):
        """Lifting + point branch: feats (B, V, 128, H, W) are the 2-D feature maps (ENet output in the reference).
        lift_views is differentiable with respect to feats, so a trainable 2-D stage in front (the reference's
        enet_trainable) receives its gradient through this call."""
        from .projection import lift_views
        points = xyz.permute(0, 2, 1).contiguous()
        image_features = lift_views(points, feats, depth, camera_to_world, intrinsic, depth_min, depth_max, image_dims,
                                    accuracy, reduce=self.reduce)
        return self.forward(xyz, image_features)


class PointNet2Multiview2(_MultiviewStackBase):
    """Point branch of `PointNet2Multiview2` (model/pointnet2multiview.py:61-121; the model the training script
    instantiates, train_scannet_multiview_semseg.py:73).  View reduction: first view, fill all-zero columns (:93-98)."""

    reduce = "first"

    def __init__(self, num_classes):
        super().__init__()
        self.sa1_geo = PointNetSetAbstraction(1024, 0.1, 32, 0 + 3, [32, 32, 64], False)
        self.sa2_geo = PointNetSetAbstraction(256, 0.2, 32, 64 + 3, [64, 64, 128], False)
        self.sa1_feat = PointNetSetAbstraction(1024, 0.1, 32, 128 + 3, [32, 32, 64], False)
        self.sa2_feat = PointNetSetAbstraction(256, 0.2, 32, 64 + 3, [64, 64, 128], False)
        self.sa3 = PointNetSetAbstraction(64, 0.4, 32, 256 + 3, [128, 128, 256], False)
        self.sa4 = PointNetSetAbstraction(16, 0.8, 32, 256 + 3, [256, 256, 512], False)
        self.fp4 = PointNetFeaturePropagation(768, [256, 256])
        self.fp3 = PointNetFeaturePropagation(512, [256, 256])
        self.fp2 = PointNetFeaturePropagation(320, [256, 128])
        self.fp1 = PointNetFeaturePropagation(128, [128, 128, 128])
        self.conv1 = nn.Conv1d(128, 128, 1)
        self.bn1 = nn.BatchNorm1d(128)
        self.drop1 = nn.Dropout(0.5)
        self.conv2 = nn.Conv1d(128, num_classes, 1)
        self._head_fold = _FoldCache()


class PointNet2Multiview2Msg(_MultiviewStackBase):
    """Point branch of `PointNet2Multiview2Msg` (model/pointnet2multiview.py:179-233), the only multi-scale-grouping
    semantic-segmentation stack of the reference (BASELINE config 2).  View reduction: max over views (:210)."""

    reduce = "max"

    def __init__(self, num_classes):
        super().__init__()
        self.sa1_geo = PointNetSetAbstractionMsg(1024, [0.05, 0.1], [16, 32], 0, [[16, 16, 32], [32, 32, 64]])
        self.sa2_geo = PointNetSetAbstractionMsg(256, [0.1, 0.2], [16, 32], 96, [[64, 64, 128], [64, 96, 128]])
        self.sa1_feat = PointNetSetAbstractionMsg(1024, [0.05, 0.1], [16, 32], 128, [[16, 16, 32], [32, 32, 64]])
        self.sa2_feat = PointNetSetAbstractionMsg(256, [0.1, 0.2], [16, 32], 96, [[64, 64, 128], [64, 96, 128]])
        self.sa3 = PointNetSetAbstractionMsg(64, [0.2, 0.4], [16, 32], 512, [[128, 196, 256], [128, 196, 256]])
        self.sa4 = PointNetSetAbstractionMsg(16, [0.4, 0.8], [16, 32], 512, [[256, 256, 512], [256, 384, 512]])
        self.fp4 = PointNetFeaturePropagation(1536, [512, 512])
        self.fp3 = PointNetFeaturePropagation(1024, [512, 512])
        self.fp2 = PointNetFeaturePropagation(608, [256, 256])
        self.fp1 = PointNetFeaturePropagation(256, [128, 128, 128])
        self.conv1 = nn.Conv1d(128, 128, 1)
        self.bn1 = nn.BatchNorm1d(128)
        self.drop1 = nn.Dropout(0.5)
        self.conv2 = nn.Conv1d(128, num_classes, 1)
        self._head_fold = _FoldCache()


class GraphedForward:
    """CUDA-graph replay of a fused forward for a fixed input shape: the ~20 launches on three streams become
    one graph launch (no per-kernel Python / driver overhead).  `run(x)` copies x (device or pinned host, (B, C, N))
    into the static input and returns the static output tensor (valid until the next run)."""

    def __init__(self, model, example_xyz, example_points, warmup=3, labels=False, logits_dtype=None):
        self.model = model
        self.xyz = example_xyz.clone()
        self.points = example_points.clone()
        kw = {"labels": True} if labels else {}  # labels: (B, N) uint8 predictions instead of logits (PointNet2SemSeg.predict)
        if logits_dtype is not None:
            kw["logits_dtype"] = logits_dtype
        side = torch.cuda.Stream(example_xyz.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(warmup):
                model.forward_fused(self.xyz, self.points, **kw)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        from . import _lib
        self.graph = torch.cuda.CUDAGraph()
        n0 = _lib.launch_count()
        with torch.no_grad(), torch.cuda.graph(self.graph):
            self.out = model.forward_fused(self.xyz, self.points, **kw)
        self.kernels_per_replay = _lib.launch_count() - n0  # our kernels captured in the graph

    def run(self, xyz, points):
        self.xyz.copy_(xyz, non_blocking=True)
        self.points.copy_(points, non_blocking=True)
        self.graph.replay()
        return self.out


class PipelinedForward:
    """`depth` graph instances on `depth` streams: consecutive batches overlap on the GPU (the FPS of batch i+1 runs
    on SMs that the latency-bound sampling of a single batch leaves idle).  submit() returns the static output of the
    slot it used together with an event; the output stays valid until that slot is submitted again."""

    def __init__(self, model, example_xyz, example_points, depth=2, labels=False, logits_dtype=None):
        self.depth = depth
        self.streams = [torch.cuda.Stream(example_xyz.device) for _ in range(depth)]
        self.slots = []
        # with several batches in flight the sampling kernel should occupy few SMs rather than finish early
        with fps_policy("throughput" if depth > 1 else "auto"):
            for st in self.streams:
                st.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(st):
                    self.slots.append(GraphedForward(model, example_xyz, example_points, labels=labels, logits_dtype=logits_dtype))
                torch.cuda.current_stream().wait_stream(st)
        self.kernels_per_replay = self.slots[0].kernels_per_replay
        self.i = 0

    def submit(self, xyz, points, after=None):
        """Enqueue one forward; `after` = optional event the slot's stream waits for first (e.g. the H2D copy)."""
        k = self.i % self.depth
        self.i += 1
        st = self.streams[k]
        if after is not None:
            st.wait_event(after)
        else:
            st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            out = self.slots[k].run(xyz, points)
            done = torch.cuda.Event()
            done.record(st)
        return out, done, st

    def join(self):
        for st in self.streams:
            torch.cuda.current_stream().wait_stream(st)


class GraphedViews:
    """CUDA-graph replay of `forward_views` (multi-view lifting + point branch, model/pointnet2multiview.py:83-121) for
    fixed shapes: projection, slab gather and the ~30 launches of the point branch become one graph launch.  `run(...)`
    copies the inputs (device or pinned host) into the static buffers and returns the static logits (valid until the next
    run).  Several instances on several streams overlap consecutive batches like PipelinedForward."""

    def __init__(self, model, xyz, feats, depth, poses, intrinsic, depth_min, depth_max, image_dims, accuracy, warmup=3):
        self.model = model
        self.xyz, self.feats, self.depth, self.poses = xyz.clone(), feats.clone(), depth.clone(), poses.clone()
        self.args = (intrinsic, depth_min, depth_max, image_dims, accuracy)
        side = torch.cuda.Stream(xyz.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(warmup):
                model.forward_views(self.xyz, self.feats, self.depth, self.poses, *self.args)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.no_grad(), torch.cuda.graph(self.graph):
            self.out = model.forward_views(self.xyz, self.feats, self.depth, self.poses, *self.args)

    def run(self, xyz, feats, depth, poses):
        self.xyz.copy_(xyz, non_blocking=True)
        self.feats.copy_(feats, non_blocking=True)
        self.depth.copy_(depth, non_blocking=True)
        self.poses.copy_(poses, non_blocking=True)
        self.graph.replay()
        return self.out


class GraphedTrainStep:
    """One training step -- zero the gradients, forward, loss, backward, optimizer update -- replayed as CUDA graphs for a
    fixed batch shape (the reference's loop: train_scannet_semseg.py:135-146).  An eager MSG step issues ~1500 launches
    and is bound by the host at small per-GPU batches (4 scenes: 18 ms eager, 11 ms replayed on one B200).

    Single process: one graph holds the whole step.  Under torch.distributed (one process per GPU, scenes sharded): the
    gradients of all parameters are views into ONE flat fp32 buffer; graph A = zero + forward + backward, then a single
    all-reduce of that buffer (NCCL, outside the graphs: the only collective of the path), then graph B = the optimizer
    update.  BatchNorm statistics stay per rank, as with the reference's DataParallel replicas.

        stepper = GraphedTrainStep(net, opt, loss_fn, xyz, feats, target)   # opt built with capturable=True
        loss = stepper.step(xyz, feats, target)                             # device tensor; valid until the next step
    """

    def __init__(self, net, opt, loss_fn, example_xyz, example_feats, example_target, group=None, warmup=3):
        from .sharding import FlatGradients
        self.net, self.opt, self.loss_fn = net, opt, loss_fn
        for g in opt.param_groups:
            if not g.get("capturable", False):
                raise ValueError("GraphedTrainStep needs an optimizer built with capturable=True (its step counter lives on the device)")
        self.xyz, self.feats, self.target = example_xyz.clone(), example_feats.clone(), example_target.clone()
        self.grads = FlatGradients(net.parameters(), group)  # gradients accumulate in place into views of one flat buffer
        self.world = self.grads.world
        dev = example_xyz.device
        # the warm-up steps below are real updates: model and optimizer are put back afterwards (in place, because the
        # graphs capture the addresses of the parameters and of the optimizer state)
        net_before = {k: v.clone() for k, v in net.state_dict().items()}
        opt_before = {p: {k: v.clone() for k, v in st.items() if torch.is_tensor(v)} for p, st in opt.state.items()}
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):  # allocates the optimizer state and warms every kernel before capture
                self._fwd_bwd()
                self._reduce()
                opt.step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        with torch.no_grad():
            for k, v in net.state_dict().items():
                v.copy_(net_before[k])
            for p, st in opt.state.items():
                for k, v in st.items():
                    if torch.is_tensor(v):
                        v.copy_(opt_before[p][k]) if p in opt_before else v.zero_()
        self.graph_a = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph_a):
            self.loss = self._fwd_bwd()
            if self.world == 1:
                opt.step()
        self.graph_b = None
        if self.world > 1:
            self.graph_b = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph_b, pool=self.graph_a.pool()):
                opt.step()

    def _fwd_bwd(self):
        self.grads.zero()
        loss = self.loss_fn(self.net(self.xyz, self.feats), self.target)
        loss.backward()
        return loss.detach()

    def _reduce(self):
        self.grads.all_reduce_mean()

    def step(self, xyz, feats, target):
        self.xyz.copy_(xyz, non_blocking=True)
        self.feats.copy_(feats, non_blocking=True)
        self.target.copy_(target, non_blocking=True)
        self.graph_a.replay()
        if self.graph_b is not None:
            self._reduce()
            self.graph_b.replay()
        return self.loss
