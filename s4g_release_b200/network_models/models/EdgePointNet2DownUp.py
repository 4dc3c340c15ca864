"""EDGEPN2DU — EdgeConv encoder AND EdgeConv decoder (reference: network_models/models/EdgePointNet2DownUp.py:8-91).

State of the reference: its constructor (:11-68) builds EdgeSAModule levels, EdgeFPModule levels whose input width is
``2 * sparse + skip`` channels when they interpolate (the edge propagation concatenates [neighbour - centre | centre]),
a skip width of 3 for the finest level (the coordinates themselves), and two heads (``mlp_seg``/``seg_logit`` and
``mlp_frame``/``frame_logit``, 9 channels) — but it uses ``SharedMLP`` without importing it (:65), so the class cannot
be instantiated there, and the forward it would inherit reads heads that this constructor never creates.  Kept here for
the module surface: the same constructor (state_dict keys ``sa_modules.*``, ``fp_modules.*``, ``mlp_seg.*``,
``seg_logit.*``, ``mlp_frame.*``, ``frame_logit.*``), and a forward for the two heads it has — OUR definition, since the
reference has no runnable one: the coordinates are the finest level's skip feature; returns ``scene_score_logits``
(B, score_classes, N) and ``frame_R`` (B, 9, N).

The fused engine (engine.FusedEdgePointNet2DownUp) is opt-in, ``forward(..., fused=True)``: EDGEPN2D's encoder, and
edge propagation levels whose first layer is split into a sparse-row part and a per-point part, so the edge rows are
never built.  Otherwise the model runs on the module path (sm_100a operators + torch autograd), as does its training."""
import torch.nn as nn

from ..nn_utils.mlp import SharedMLP
from . import PointNet2 as _pn2
from .EdgePointNet2Down import edge_levels_fusable
from .PointNet2_tcls import FusedEngineCache, _widths_ok, trunk_fusable
from .pointnet2_utils.modules import EdgeFPModule, EdgeSAModule

PointNet2Loss, PointNet2Metric = _pn2.PointNet2Loss, _pn2.PointNet2Metric


class EdgePointNet2DownUp(FusedEngineCache, nn.Module):
    _SA_MODULE = EdgeSAModule
    _FP_MODULE = EdgeFPModule
    _ENGINE = "FusedEdgePointNet2DownUp"

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
        skip = [3] + [ch[-1] for ch in sa_channels]  # the finest level's skip feature is xyz itself (:46-47)
        self.fp_modules = nn.ModuleList()
        c = skip[-1]
        for i in range(n_fp):
            width = c + skip[-2 - i] if num_fp_neighbours[i] == 0 else 2 * c + skip[-2 - i]  # (:52-61)
            self.fp_modules.append(self._FP_MODULE(in_channels=width, mlp_channels=fp_channels[i],
                                                   num_neighbors=num_fp_neighbours[i]))
            c = fp_channels[i][-1]
        self.mlp_seg = SharedMLP(c, seg_channels, ndim=1, dropout_prob=dropout_prob)
        self.seg_logit = nn.Conv1d(seg_channels[-1], score_classes, 1, bias=True)
        self.mlp_frame = SharedMLP(c, seg_channels, ndim=1)
        self.frame_logit = nn.Conv1d(seg_channels[-1], 9, 1, bias=True)
        self._engine = None
        self._engine_key = None

    def fusable(self, allow_global=False):
        """Whether the fused engine has a plan for this configuration: the trunk rules of ``trunk_fusable``
        (``allow_global`` as there), EDGEPN2D's rule for edge set-abstraction levels (``edge_levels_fusable``), an edge
        propagation level's first layer at most 512 wide (its stacked [U | V] pre-activations, 2 x that width, are one row
        chain's output), and head widths that are multiples of 16, <= 512, with at most 16 score classes."""
        c = self.config
        if not (trunk_fusable(c, allow_global) and edge_levels_fusable(c)):
            return False
        if any(ch[0] > 512 for ch, k in zip(c["fp_channels"], c["num_fp_neighbours"]) if k != 0):
            return False
        return _widths_ok(c["seg_channels"]) and max(c["seg_channels"]) <= 512 and c["score_classes"] <= 16

    def forward(self, data_batch, fused=None):
        """``fused``: None / False = the module path; True = the fused engine, for every configuration
        ``fusable(allow_global=True)`` accepts (others raise RuntimeError before any GPU work)."""
        points = data_batch["scene_points"]
        if not fused:
            return self.forward_modules(points)
        if not self.fusable(allow_global=True):
            raise RuntimeError("the fused engine has no plan for this configuration (see EdgePointNet2DownUp.fusable); "
                               "call with fused=False for the module path")
        return self.fused_engine().forward(points)

    def forward_modules(self, points):
        xyz, feature = points, None
        level_xyz, level_feature = [xyz], [points]
        for sa in self.sa_modules:
            xyz, feature = sa(xyz, feature)
            level_xyz.append(xyz)
            level_feature.append(feature)
        sparse_xyz, sparse_feature = xyz, feature
        for i, fp in enumerate(self.fp_modules):
            dense_xyz, dense_feature = level_xyz[-2 - i], level_feature[-2 - i]
            sparse_feature = fp(dense_xyz, sparse_xyz, dense_feature, sparse_feature)
            sparse_xyz = dense_xyz
        return {"scene_score_logits": self.seg_logit(self.mlp_seg(sparse_feature)),
                "frame_R": self.frame_logit(self.mlp_frame(sparse_feature))}


def build_edgepointnet2downup(cfg):
    node = cfg.MODEL.EDGEPN2DU
    net = EdgePointNet2DownUp(score_classes=cfg.DATA.SCORE_CLASSES, num_centroids=node.NUM_CENTROIDS, radius=node.RADIUS,
                              num_neighbours=node.NUM_NEIGHBOURS, sa_channels=node.SA_CHANNELS,
                              fp_channels=node.FP_CHANNELS, num_fp_neighbours=node.NUM_FP_NEIGHBOURS,
                              seg_channels=node.SEG_CHANNELS, dropout_prob=node.DROPOUT_PROB)
    return net, PointNet2Loss(label_smoothing=node.LABEL_SMOOTHING, neg_weight=node.NEG_WEIGHT), PointNet2Metric()
