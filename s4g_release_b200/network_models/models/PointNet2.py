"""PN2 — the sibling of PN2_CLS with a continuous pose head (reference: network_models/models/PointNet2.py:24-153).

Same encoder / decoder as PointNet2_tcls.PointNet2 (so the same sm_100a operators and, for configurations without a
global set-abstraction level, the same fused engine); the heads differ: ``frame_R`` is a 6-D rotation representation
turned into a matrix by ``toRotMatrix`` (functions/functions.py:179-190), ``frame_t`` is a 3-D offset ADDED to the
input points, the score key is ``scene_score_logits``, and ``t_logit`` starts at zero (:150-152).  The reference's
default configuration (4 levels, the last one a global group with num_centroids = 0) runs on the module path unless the
fused engine is asked for with ``fused=True``.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from ..functions.functions import toRotMatrix
from ..nn_utils.functional import smooth_cross_entropy
from . import PointNet2_tcls as _tcls


class PointNet2(_tcls.PointNet2):
    _R_OUT, _T_OUT = 6, 3

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.init_weights()

    def init_weights(self):
        nn.init.zeros_(self.t_logit.weight)
        nn.init.zeros_(self.t_logit.bias)

    def forward(self, data_batch, fused=None):
        """``fused`` routes as PointNet2_tcls.PointNet2.forward (an unsupported configuration with fused=True raises)."""
        return self.predictions(super().forward(data_batch, fused=fused), data_batch["scene_points"])

    def predictions(self, raw, points):
        """raw head outputs -> this model's predictions (PointNet2.py:140-148); shared with train_engine.TrainEngine"""
        return {"scene_score_logits": raw["score"], "frame_R": toRotMatrix(raw["frame_R"]),
                "frame_t": points + raw["frame_t"], "movable_logits": raw["movable_logits"]}


class PointNet2Loss(nn.Module):
    """PointNet2.py:156-213: weighted CE on the score classes, L1 on the movable directions, flip-symmetric rotation
    MSE weighted by the ground-truth score (x5), squared translation error weighted by the score (x20)."""

    def __init__(self, label_smoothing=0, neg_weight=0.1):
        super().__init__()
        self.label_smoothing, self.neg_weight = label_smoothing, neg_weight

    def forward(self, preds, labels):
        logits = preds["scene_score_logits"]
        weight = torch.ones(logits.shape[1], device=logits.device)
        weight[0] = self.neg_weight
        gt_R = labels["best_frame_R"]
        n = gt_R.shape[2]
        pred_R = preds["frame_R"][:, :, :n]
        flip = gt_R.new_tensor([1, -1, -1, 1, -1, -1, 1, -1, -1]).view(1, 9, 1)
        R_err = torch.minimum(((pred_R - gt_R) ** 2).mean(1), ((pred_R - gt_R * flip) ** 2).mean(1))
        gt_score = labels["scene_score"][:, :n]
        t_err = ((preds["frame_t"][:, :, :n] - labels["best_frame_t"]) ** 2).sum(1)
        if self.label_smoothing > 0:  # reference PointNet2.py:174-178
            cls_loss = smooth_cross_entropy(logits.transpose(1, 2).reshape(-1, logits.shape[1]),
                                            labels["scene_score_labels"].reshape(-1), float(self.label_smoothing),
                                            weight=weight)
        else:
            cls_loss = F.cross_entropy(logits, labels["scene_score_labels"], weight)
        return {"cls_loss": cls_loss,
                "R_loss": (R_err * gt_score).mean() * 5.0,
                "t_loss": (t_err * gt_score).mean() * 20.0,
                "mov_loss": F.l1_loss(preds["movable_logits"], labels["scene_movable_labels"])}


class PointNet2Metric(nn.Module):
    """PointNet2.py:216-255: per-point score-class and movable accuracies (unreduced 0/1 tensors), score-weighted geodesic
    angle to the closer of the ground-truth frame and its flip about x, mean translation error."""

    def forward(self, preds, labels):
        cls_acc = (preds["scene_score_logits"].argmax(1).reshape(-1) == labels["scene_score_labels"].reshape(-1)).float()
        mov_acc = ((preds["movable_logits"] > 0.5).reshape(-1).int() ==
                   labels["scene_movable_labels"].reshape(-1).int()).float()
        gt = labels["best_frame_R"]
        b, _, n = gt.shape
        gt = gt.transpose(1, 2).reshape(b * n, 3, 3)
        pred = preds["frame_R"][:, :, :n].transpose(1, 2).reshape(b * n, 3, 3)
        angle = torch.minimum(_tcls._rotation_angle(gt, pred),
                              _tcls._rotation_angle(gt * gt.new_tensor([1.0, -1.0, -1.0]), pred))
        R_err = (labels["scene_score"][:, :n].reshape(-1) * angle).mean()
        t_err = torch.sqrt(((labels["best_frame_t"] - preds["frame_t"][:, :, :n]) ** 2).sum(1)).mean()
        return {"cls_acc": cls_acc, "mov_acc": mov_acc, "R_err": R_err, "t_err": t_err}


def build_pointnet2(cfg):
    """PointNet2.py:258-280 (``MODEL.PN2`` node)."""
    node = cfg.MODEL.PN2
    net = PointNet2(score_classes=cfg.DATA.SCORE_CLASSES, num_centroids=node.NUM_CENTROIDS, radius=node.RADIUS,
                    num_neighbours=node.NUM_NEIGHBOURS, sa_channels=node.SA_CHANNELS, fp_channels=node.FP_CHANNELS,
                    num_fp_neighbours=node.NUM_FP_NEIGHBOURS, seg_channels=node.SEG_CHANNELS,
                    dropout_prob=node.DROPOUT_PROB)
    return net, PointNet2Loss(label_smoothing=node.LABEL_SMOOTHING, neg_weight=node.NEG_WEIGHT), PointNet2Metric()
