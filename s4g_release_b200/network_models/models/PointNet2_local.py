"""PN2_LOCAL — the sibling with a grasp-EVALUATION head (reference: network_models/models/PointNet2_local.py:10-329).

Encoder / decoder as PN2 and PN2_CLS (the same sm_100a operators through pointnet2_utils.modules).  Heads: ``frame_R``
(9 raw values), ``frame_t`` (3-D offset added to the input points, ``t_logit`` zero-initialised :162-164),
``movable_logits`` (2 classes, no sigmoid) and ``local_search_logits``: a SharedMLP(ndim=2) over
[point feature | candidate frame (R 9 + t 3) repeated 4 times = 48 channels] (:86-87, :131-147).  With
``data_batch["local_search_frame"]`` (B, 12, n_frames, n_search) the candidates are given — their translations are made
relative to the point they belong to, IN PLACE like the reference (:135) — else the network's own (R, t) prediction
is the single candidate per point.

Two execution paths share the parameters: the module path (the default, ``fused=None`` or ``fused=False``) and, only
when asked with ``forward(..., fused=True)``, the fused sm_100a engine (``engine.FusedPointNet2Local``): the trunk of
PN2_CLS, the three per-point heads as logits chains, and the evaluation head as one logits chain over bf16 rows
[point feature | candidate x 4] written by one kernel.  The given candidates' translations are updated in place there
too, with the same fp32 subtraction.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from ..nn_utils.functional import smooth_cross_entropy
from ..nn_utils.mlp import SharedMLP
from .PointNet2_tcls import FusedEngineCache, _widths_ok, trunk_fusable
from .pointnet2_utils.modules import PointNetSAModule, PointnetFPModule


class PointNet2(FusedEngineCache, nn.Module):
    _SA_MODULE = PointNetSAModule
    _FP_MODULE = PointnetFPModule
    _ENGINE = "FusedPointNet2Local"

    def __init__(self,
                 score_classes,
                 num_centroids=(10240, 1024, 128, 0),
                 radius=(0.2, 0.3, 0.4, -1.0),
                 num_neighbours=(64, 64, 64, -1),
                 sa_channels=((32, 32, 64), (64, 64, 128), (128, 128, 256), (256, 512, 1024)),
                 fp_channels=((256, 256), (256, 128), (128, 128), (64, 64, 64)),
                 num_fp_neighbours=(0, 3, 3, 3),
                 seg_channels=(128,),
                 dropout_prob=0.5):
        super().__init__()
        n_sa, n_fp = len(num_centroids), len(fp_channels)
        assert len(radius) == n_sa and len(num_neighbours) == n_sa and len(sa_channels) == n_sa
        assert n_sa == n_fp and len(num_fp_neighbours) == n_fp
        self.config = dict(score_classes=score_classes, num_centroids=tuple(num_centroids), radius=tuple(radius),
                           num_neighbours=tuple(num_neighbours), sa_channels=tuple(map(tuple, sa_channels)),
                           fp_channels=tuple(map(tuple, fp_channels)), num_fp_neighbours=tuple(num_fp_neighbours),
                           seg_channels=tuple(seg_channels), dropout_prob=dropout_prob)
        self.sa_modules = nn.ModuleList()
        c = 0
        for i in range(n_sa):
            self.sa_modules.append(self._SA_MODULE(in_channels=c, mlp_channels=sa_channels[i],
                                                   num_centroids=num_centroids[i], radius=radius[i],
                                                   num_neighbours=num_neighbours[i], use_xyz=True))
            c = sa_channels[i][-1]
        skip = [0] + [ch[-1] for ch in sa_channels]
        self.fp_modules = nn.ModuleList()
        c = skip[-1]
        for i in range(n_fp):
            self.fp_modules.append(self._FP_MODULE(in_channels=c + skip[-2 - i], mlp_channels=fp_channels[i],
                                                   num_neighbors=num_fp_neighbours[i]))
            c = fp_channels[i][-1]
        # creation order = the reference's (:86-96): a seeded default init is identical
        self.mlp_grasp_eval = SharedMLP(c + 48, seg_channels, ndim=2, dropout_prob=dropout_prob)
        self.grasp_eval_logit = nn.Conv2d(seg_channels[-1], score_classes, 1, bias=True)
        self.mlp_R = SharedMLP(c, seg_channels, ndim=1)
        self.R_logit = nn.Conv1d(seg_channels[-1], 9, 1, bias=True)
        self.mlp_t = SharedMLP(c, seg_channels, ndim=1)
        self.t_logit = nn.Conv1d(seg_channels[-1], 3, 1, bias=True)
        self.mlp_movable = SharedMLP(c, seg_channels, ndim=1, dropout_prob=dropout_prob)
        self.movable_logit = nn.Conv1d(seg_channels[-1], 2, 1, bias=True)
        self.init_weights()
        self._engine = None
        self._engine_key = None

    def init_weights(self):
        nn.init.zeros_(self.t_logit.weight)
        nn.init.zeros_(self.t_logit.bias)

    def fusable(self, allow_global=False):
        """Whether the fused engine has a plan for this configuration: the trunk rules of PN2_CLS
        (PointNet2_tcls.trunk_fusable, ``allow_global`` as there), head widths that are multiples of 16 and <= 512, at
        most 16 evaluation classes.  ``forward(fused=True)`` asks with ``allow_global=True``."""
        c = self.config
        if not trunk_fusable(c, allow_global):
            return False
        if not _widths_ok(c["seg_channels"]) or any(w > 512 for w in c["seg_channels"]):
            return False
        return c["score_classes"] <= 16

    def forward(self, data_batch, fused=None):
        """``fused``: None / False = the module path; True = the fused engine, for every configuration
        ``fusable(allow_global=True)`` accepts (others raise RuntimeError before any GPU work; given frames that are not
        (B, 12, F, S) contiguous float32 on the points' device with 1 <= F <= N, S >= 1 raise ValueError)."""
        if not fused:
            return self.forward_modules(data_batch)
        points = data_batch["scene_points"]
        if not self.fusable(allow_global=True):
            raise RuntimeError("the fused engine has no plan for this configuration (see PointNet2_local.PointNet2.fusable);"
                               " call with fused=False for the module path")
        frames = data_batch["local_search_frame"] if "local_search_frame" in data_batch else None
        if frames is not None:
            from ...engine import check_local_frames
            check_local_frames(points, frames)
        return self.predictions(self.fused_engine().forward(points, frames), points)

    def predictions(self, raw, points):
        """The engine's raw head outputs -> this model's predictions: ``frame_t`` is the offset added to the points."""
        return {"local_search_logits": raw["local_search_logits"], "frame_R": raw["frame_R"],
                "frame_t": points + raw["frame_t"], "movable_logits": raw["movable_logits"]}

    def forward_modules(self, data_batch):
        points = data_batch["scene_points"]
        xyz, feature = points, None
        level_xyz, level_feature = [xyz], [feature]
        for sa in self.sa_modules:
            xyz, feature = sa(xyz, feature)
            level_xyz.append(xyz)
            level_feature.append(feature)
        sparse_xyz, point_feature = xyz, feature
        for i, fp in enumerate(self.fp_modules):
            dense_xyz = level_xyz[-2 - i]
            point_feature = fp(dense_xyz, sparse_xyz, level_feature[-2 - i], point_feature)
            sparse_xyz = dense_xyz
        R = self.R_logit(self.mlp_R(point_feature))
        t = self.t_logit(self.mlp_t(point_feature))
        mov = self.movable_logit(self.mlp_movable(point_feature))
        if "local_search_frame" in data_batch:
            frames = data_batch["local_search_frame"]          # (B, 12, n_frames, n_search): rows 9.. = translation
            n_frames, n_search = frames.shape[2:]
            anchor = points[:, :, :n_frames].unsqueeze(-1).expand(-1, -1, -1, n_search)
            frames[:, 9:, :, :] = frames[:, 9:, :, :] - anchor   # in place, as the reference does to the caller's tensor
            per_point = point_feature[:, :, :n_frames].unsqueeze(-1).expand(-1, -1, -1, n_search)
        else:
            frames = torch.cat([R, t], dim=1).unsqueeze(-1)   # the prediction itself, one candidate per point
            per_point = point_feature.unsqueeze(-1)
        evaluated = torch.cat([per_point, frames.repeat(1, 4, 1, 1)], dim=1)
        return {"local_search_logits": self.grasp_eval_logit(self.mlp_grasp_eval(evaluated)),
                "frame_R": R, "frame_t": points + t, "movable_logits": mov}


class PointNet2Loss(nn.Module):
    """PointNet2_local.py:167-226: weighted CE over the evaluated candidates and over the 2 movable classes (class-0
    weight 0.4), flip-symmetric rotation MSE (x4: the better of the frame and the frame with its y / z columns negated),
    translation MSE (x20); the normal term is computed by the reference but not returned."""

    def __init__(self, label_smoothing=0, neg_weight=0.1):
        super().__init__()
        self.label_smoothing, self.neg_weight = label_smoothing, neg_weight

    def forward(self, preds, labels):
        logits = preds["local_search_logits"]
        weight = torch.ones(logits.shape[1], device=logits.device)
        weight[0] = self.neg_weight
        mov_weight = torch.ones(2, device=logits.device)
        mov_weight[0] = 0.4
        gt_R = labels["best_frame_R"]
        n = gt_R.shape[2]
        pred_R = preds["frame_R"][:, :, :n]
        flip = gt_R.new_tensor([1, -1, -1, 1, -1, -1, 1, -1, -1]).view(1, 9, 1)
        R_err = torch.minimum(((pred_R - gt_R) ** 2).mean(1), ((pred_R - gt_R * flip) ** 2).mean(1))
        if self.label_smoothing > 0:  # reference :186-195
            eps = float(self.label_smoothing)
            cls_loss = smooth_cross_entropy(logits.permute(0, 2, 3, 1).reshape(-1, logits.shape[1]),
                                            labels["scored_grasp_labels"].reshape(-1), eps, weight=weight)
            mov_loss = smooth_cross_entropy(preds["movable_logits"].transpose(1, 2).reshape(-1, 2),
                                            labels["scene_movable_labels"].reshape(-1), eps, weight=mov_weight)
        else:
            cls_loss = F.cross_entropy(logits, labels["scored_grasp_labels"], weight)
            mov_loss = F.cross_entropy(preds["movable_logits"], labels["scene_movable_labels"], mov_weight)
        return {"cls_loss": cls_loss,
                "R_loss": R_err.mean() * 4.0,
                "t_loss": torch.mean((preds["frame_t"][:, :, :n] - labels["best_frame_t"]) ** 2) * 20.0,
                "mov_loss": mov_loss}


class PointNet2Metric(nn.Module):
    """PointNet2_local.py:229-272: per-candidate / per-point accuracies (unreduced), mean geodesic rotation error under
    the gripper's flip symmetry, mean translation error."""

    def forward(self, preds, labels):
        cls_acc = preds["local_search_logits"].argmax(1).view(-1).eq(labels["scored_grasp_labels"].view(-1)).float()
        mov_acc = preds["movable_logits"].argmax(1).view(-1).eq(labels["scene_movable_labels"].view(-1)).float()
        gt_R = labels["best_frame_R"]
        B, _, n = gt_R.shape
        gt = gt_R.transpose(1, 2).contiguous().view(B * n, 3, 3)
        gt_flipped = gt.clone()
        gt_flipped[:, :, 1:] = -gt_flipped[:, :, 1:]
        pred = preds["frame_R"][:, :, :n].transpose(1, 2).contiguous().view(B * n, 3, 3)

        def geodesic(a):
            m = torch.bmm(a, pred.transpose(1, 2))
            return torch.acos(torch.clamp((m[:, 0, 0] + m[:, 1, 1] + m[:, 2, 2] - 1.0) / 2.0, -1.0, 1.0))

        R_err = torch.stack([geodesic(gt), geodesic(gt_flipped)], dim=1).min(1)[0].mean()
        t_err = torch.mean(torch.sqrt(((labels["best_frame_t"] - preds["frame_t"][:, :, :n]) ** 2).sum(1)))
        return {"cls_acc": cls_acc, "mov_acc": mov_acc, "R_err": R_err, "t_err": t_err}


def build_pointnet2_local(cfg):
    """cfg: the reference's yacs-style node (DATA.SCORE_CLASSES, MODEL.PN2.*) — PointNet2_local.py:275-295."""
    pn2 = cfg.MODEL.PN2
    net = PointNet2(score_classes=cfg.DATA.SCORE_CLASSES, num_centroids=pn2.NUM_CENTROIDS, radius=pn2.RADIUS,
                    num_neighbours=pn2.NUM_NEIGHBOURS, sa_channels=pn2.SA_CHANNELS, fp_channels=pn2.FP_CHANNELS,
                    num_fp_neighbours=pn2.NUM_FP_NEIGHBOURS, seg_channels=pn2.SEG_CHANNELS,
                    dropout_prob=pn2.DROPOUT_PROB)
    return net, PointNet2Loss(label_smoothing=pn2.LABEL_SMOOTHING, neg_weight=pn2.NEG_WEIGHT), PointNet2Metric()
