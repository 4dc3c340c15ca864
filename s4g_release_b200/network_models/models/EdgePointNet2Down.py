"""EDGEPN2D — PN2 with EdgeConv set-abstraction levels (reference: network_models/models/EdgePointNet2Down.py:9-33).

The reference's class is the PN2 sibling with ``_SA_MODULE = EdgeSAModule`` and the plain PointnetFPModule decoder; the
builder reads the ``MODEL.EDGEPN2D`` node.  An edge level concatenates centroid features to every neighbour; the fused
engine (engine.FusedEdgePointNet2Down) runs it without building those rows, by splitting the level's first layer into a
neighbour part and a centroid part.  The fused engine is opt-in, ``forward(..., fused=True)``; otherwise the model runs
on the module path (sm_100a operators + torch autograd), as does its training."""
from . import PointNet2 as _pn2
from .pointnet2_utils.modules import EdgeSAModule, PointnetFPModule

PointNet2Loss, PointNet2Metric = _pn2.PointNet2Loss, _pn2.PointNet2Metric


def edge_levels_fusable(c):
    """Every edge set-abstraction level (sampled, with input features) of the configuration dict ``c`` is at least two
    layers deep: the centroid term joins the first layer's epilogue, and a one-layer level's first layer is its max-pool."""
    return all(len(ch) > 1 for i, ch in enumerate(c["sa_channels"]) if i > 0 and c["num_centroids"][i] != 0)


class EdgePointNet2Down(_pn2.PointNet2):
    _SA_MODULE = EdgeSAModule
    _FP_MODULE = PointnetFPModule
    _ENGINE = "FusedEdgePointNet2Down"

    def fusable(self, allow_global=False):
        """Whether the fused engine has a plan for this configuration: the PN2 sibling's rules (PointNet2_tcls.PointNet2.
        fusable, ``allow_global`` as there) and every edge level (sampled, with input features) at least two layers deep
        — the centroid term joins the first layer's epilogue, and a one-layer level's first layer is its max-pool."""
        return super().fusable(allow_global) and edge_levels_fusable(self.config)

    def forward(self, data_batch, fused=None):
        """``fused``: None / False = the module path; True = the fused engine, for every configuration
        ``fusable(allow_global=True)`` accepts (others raise RuntimeError before any GPU work)."""
        points = data_batch["scene_points"]
        if not fused:
            return self.predictions(self.forward_modules(points), points)
        if not self.fusable(allow_global=True):
            raise RuntimeError("the fused engine has no plan for this configuration (see EdgePointNet2Down.fusable); "
                               "call with fused=False for the module path")
        return self.predictions(self.fused_engine().forward(points), points)


def build_edgepointnet2down(cfg):
    node = cfg.MODEL.EDGEPN2D
    net = EdgePointNet2Down(score_classes=cfg.DATA.SCORE_CLASSES, num_centroids=node.NUM_CENTROIDS, radius=node.RADIUS,
                            num_neighbours=node.NUM_NEIGHBOURS, sa_channels=node.SA_CHANNELS, fp_channels=node.FP_CHANNELS,
                            num_fp_neighbours=node.NUM_FP_NEIGHBOURS, seg_channels=node.SEG_CHANNELS,
                            dropout_prob=node.DROPOUT_PROB)
    return net, PointNet2Loss(label_smoothing=node.LABEL_SMOOTHING, neg_weight=node.NEG_WEIGHT), PointNet2Metric()
