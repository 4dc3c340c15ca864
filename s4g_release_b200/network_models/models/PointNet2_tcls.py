"""PN2_CLS — the S4G single-shot grasp network (the pretrained "curvature_model").

Module surface of inference/grasp_proposal/network_models/models/PointNet2_tcls.py: same class names,
constructor arguments, dict-in / dict-out ``forward`` (:99-148), parameter creation order (so a seeded
default init is identical) and state_dict keys (``sa_modules.{i}.mlp.{j}.conv.weight`` …,
200 entries / 6 632 213 parameters for the shipped configuration) — reference checkpoints load with
``strict=True``.

Two execution paths share the parameters:
  * module path (``self.training`` or autograd enabled): the nn.Module stack of pointnet2_utils.modules on
    the sm_100a ops — used for training and as the drop-in;
  * fused path (eval + no_grad on CUDA): ``engine.FusedPointNet2`` runs the whole forward with the
    hand-written kernels (geometry in fp32, MLP chains on tcgen05 tensor cores).  A configuration whose last level is
    one global group (this class's default arguments) runs on it only when asked, ``forward(..., fused=True)``.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from ..nn_utils.functional import smooth_cross_entropy
from ..nn_utils.mlp import SharedMLP
from .pointnet2_utils.modules import PointNetSAModule, PointnetFPModule

# configs/curvature_model.yaml:11-22 + yacs defaults (SURVEY.md §5): the shipped PN2_CLS hyper-parameters
PN2_CLS_CONFIG = dict(
    score_classes=3,
    num_centroids=(5120, 1024, 256),
    radius=(0.02, 0.08, 0.32),
    num_neighbours=(64, 64, 64),
    sa_channels=((128, 128, 256), (256, 256, 512), (512, 512, 1024)),
    fp_channels=((1024, 1024), (512, 512), (256, 256, 256)),
    num_fp_neighbours=(3, 3, 3),
    seg_channels=(512, 256, 256, 128),
    num_removal_directions=5,
    dropout_prob=0.5,
)
NUM_INPUT = 25600


def _widths_ok(chans):
    return all(w % 16 == 0 and w >= 16 for w in chans)


def trunk_fusable(c, allow_global=False):
    """Whether the fused engine has a plan for the trunk (encoder + decoder) of the configuration dict ``c``: every level
    samples centroids, neighbourhoods of 8 / 16 / 32 / 64 points, 3-NN propagation, hidden widths that are multiples of
    16 and <= 512 inside a chain (a FP chain is cut after a wider layer, so only its LAST layer may be).

    ``allow_global=True`` also admits a LAST set-abstraction level with one global group (num_centroids = 0,
    num_neighbours = -1) paired with a first propagation level that broadcasts its feature (num_fp_neighbours[0] = 0).
    Shared by the models whose heads the engine runs (PN2_CLS, the PN2 sibling, PN2_LOCAL)."""
    cent, nbrs, fp_nbrs = c["num_centroids"], c["num_neighbours"], c["num_fp_neighbours"]
    if allow_global and cent[-1] == 0 and nbrs[-1] < 0 and fp_nbrs[0] == 0:
        cent, nbrs, fp_nbrs = cent[:-1], nbrs[:-1], fp_nbrs[1:]  # the rules below cover the remaining levels
    if not all(n > 0 for n in cent) or not all(k in (8, 16, 32, 64) for k in nbrs):
        return False
    if not all(k == 3 for k in fp_nbrs):
        return False
    for chans in c["sa_channels"]:
        if not _widths_ok(chans) or any(w > 512 for w in chans[:-1]) or chans[-1] > 1024:
            return False
    for chans in c["fp_channels"]:
        if not _widths_ok(chans) or any(w > 1024 for w in chans):
            return False
    return True


class FusedEngineCache:
    """The fused inference engine of a model, cached and bound to its CURRENT parameters.  ``_ENGINE`` names the engine
    class in engine.py; the model sets ``_engine = _engine_key = None`` in its constructor."""
    _ENGINE = "FusedPointNet2"

    def _param_fingerprint(self):
        """Device + summed version counters of every parameter and buffer: changes on in-place updates under no_grad
        (optimizer steps, EMA), on top of the explicit invalidation in train() / _apply() / load_state_dict().  Writes
        through ``p.data`` bypass the version counter — call ``invalidate_engine()`` after those."""
        tensors = self.__dict__.get("_engine_tensors")
        if tensors is None:
            tensors = list(self.parameters()) + list(self.buffers())
            self.__dict__["_engine_tensors"] = tensors
        return (tensors[0].device, tensors[0].dtype, sum(t._version for t in tensors))

    def invalidate_engine(self):
        self._engine = None
        self._engine_key = None
        self.__dict__.pop("_engine_tensors", None)

    def attach_engine(self, engine):
        """Use an engine built by the caller (e.g. with another MLP backend) for this module's current parameters."""
        self._engine = engine
        self._engine_key = self._param_fingerprint()

    def fused_engine(self, refresh=False):
        """The fused sm_100a inference engine bound to this module's CURRENT parameters (rebuilt when they changed)."""
        key = self._param_fingerprint()
        if self._engine is None or refresh or key != self._engine_key:
            from ... import engine
            self._engine = getattr(engine, self._ENGINE)(self)
            self._engine_key = key
        return self._engine

    def train(self, mode=True):
        self.invalidate_engine()  # parameters may change: re-fold BN on the next eval forward
        return super().train(mode)

    def _apply(self, fn, *args, **kwargs):
        self.invalidate_engine()  # .to() / .cuda() / .half(): the engine's buffers live on the old device
        return super()._apply(fn, *args, **kwargs)

    def load_state_dict(self, *args, **kwargs):
        self.invalidate_engine()
        return super().load_state_dict(*args, **kwargs)

    def __getstate__(self):  # copy.deepcopy / torch.save(model): the engine holds ctypes handles
        state = self.__dict__.copy()
        state["_engine"], state["_engine_key"] = None, None
        state.pop("_engine_tensors", None)
        return state

    def __deepcopy__(self, memo):
        import copy
        clone = self.__class__.__new__(self.__class__)
        memo[id(self)] = clone
        for k, v in self.__getstate__().items():
            clone.__dict__[k] = copy.deepcopy(v, memo)
        return clone


class PointNet2(FusedEngineCache, nn.Module):
    _SA_MODULE = PointNetSAModule
    _FP_MODULE = PointnetFPModule
    _R_OUT, _T_OUT = 9, 4  # frame_R: flattened 3x3; frame_t: 4 approach-offset classes (the PN2 sibling: 6 and 3)

    def __init__(self,
                 score_classes,
                 num_centroids=(10240, 1024, 128, 0),
                 radius=(0.2, 0.3, 0.4, -1.0),
                 num_neighbours=(64, 64, 64, -1),
                 sa_channels=((32, 32, 64), (64, 64, 128), (128, 128, 256), (256, 512, 1024)),
                 fp_channels=((256, 256), (256, 128), (128, 128), (64, 64, 64)),
                 num_fp_neighbours=(0, 3, 3, 3),
                 seg_channels=(128,),
                 num_removal_directions=5,
                 dropout_prob=0.5):
        super().__init__()
        n_sa, n_fp = len(num_centroids), len(fp_channels)
        assert len(radius) == n_sa and len(num_neighbours) == n_sa and len(sa_channels) == n_sa
        assert n_sa == n_fp and len(num_fp_neighbours) == n_fp
        self.config = dict(score_classes=score_classes, num_centroids=tuple(num_centroids), radius=tuple(radius),
                           num_neighbours=tuple(num_neighbours), sa_channels=tuple(map(tuple, sa_channels)),
                           fp_channels=tuple(map(tuple, fp_channels)), num_fp_neighbours=tuple(num_fp_neighbours),
                           seg_channels=tuple(seg_channels), num_removal_directions=num_removal_directions,
                           dropout_prob=dropout_prob)

        # encoder: set abstraction levels (xyz is always concatenated: use_xyz=True)
        self.sa_modules = nn.ModuleList()
        c = 0
        for i in range(n_sa):
            self.sa_modules.append(self._SA_MODULE(in_channels=c, mlp_channels=sa_channels[i],
                                                   num_centroids=num_centroids[i], radius=radius[i],
                                                   num_neighbours=num_neighbours[i], use_xyz=True))
            c = sa_channels[i][-1]
        skip = [0] + [ch[-1] for ch in sa_channels]

        # decoder: feature propagation levels, coarse to fine, with skip links
        self.fp_modules = nn.ModuleList()
        c = skip[-1]
        for i in range(n_fp):
            self.fp_modules.append(self._FP_MODULE(in_channels=c + skip[-2 - i], mlp_channels=fp_channels[i],
                                                   num_neighbors=num_fp_neighbours[i]))
            c = fp_channels[i][-1]

        # four per-point heads
        self.mlp_seg = SharedMLP(c, seg_channels, ndim=1, dropout_prob=dropout_prob)
        self.seg_logit = nn.Conv1d(seg_channels[-1], score_classes, 1, bias=True)
        self.mlp_R = SharedMLP(c, seg_channels, ndim=1)
        self.R_logit = nn.Conv1d(seg_channels[-1], self._R_OUT, 1, bias=True)
        self.mlp_t = SharedMLP(c, seg_channels, ndim=1)
        self.t_logit = nn.Conv1d(seg_channels[-1], self._T_OUT, 1, bias=True)
        self.mlp_movable = SharedMLP(c, seg_channels, ndim=1, dropout_prob=dropout_prob)
        self.movable_logit = nn.Sequential(nn.Conv1d(seg_channels[-1], num_removal_directions, 1, bias=True),
                                           nn.Sigmoid())
        self._engine = None
        self._engine_key = None

    # ------------------------------------------------------------------ module (autograd) path
    def forward_modules(self, points):
        xyz, feature = points, None
        level_xyz, level_feature = [xyz], [feature]
        for sa in self.sa_modules:
            xyz, feature = sa(xyz, feature)
            level_xyz.append(xyz)
            level_feature.append(feature)
        sparse_xyz, sparse_feature = xyz, feature
        for i, fp in enumerate(self.fp_modules):
            dense_xyz, dense_feature = level_xyz[-2 - i], level_feature[-2 - i]
            sparse_feature = fp(dense_xyz, sparse_xyz, dense_feature, sparse_feature)
            sparse_xyz = dense_xyz
        return {
            "score": self.seg_logit(self.mlp_seg(sparse_feature)),
            "frame_R": self.R_logit(self.mlp_R(sparse_feature)),
            "frame_t": self.t_logit(self.mlp_t(sparse_feature)),
            "movable_logits": self.movable_logit(self.mlp_movable(sparse_feature)),
        }

    # ------------------------------------------------------------------ fused (inference) path
    def fusable(self, allow_global=False):
        """Whether the fused engine has a plan for this configuration (engine.py / csrc/chain_plan.cu): the trunk rules of
        ``trunk_fusable``, head widths that are multiples of 16 and <= 512, at most 16 logits per head.  Anything else
        runs on the module path, like the reference.

        ``allow_global=True`` also admits a global last level (see ``trunk_fusable``) — e.g. this class's own default
        constructor arguments.  ``forward(fused=True)`` accepts those; the automatic route (``fused=None``) uses the
        default answer and runs them on the module path, like the reference."""
        c = self.config
        if not trunk_fusable(c, allow_global):
            return False
        if not _widths_ok(c["seg_channels"]) or any(w > 512 for w in c["seg_channels"]):
            return False
        return max(c["score_classes"], self._R_OUT, self._T_OUT, c["num_removal_directions"]) <= 16

    def forward(self, data_batch, fused=None, host_out=None):
        """``fused``: None = the fused engine in eval + no_grad on CUDA when ``fusable()``, else the module path;
        True = the fused engine (also for a global last level, ``fusable(allow_global=True)``); False = the module path.
        ``host_out`` (fused path only): dict of pinned host tensors that receive the predictions while the later
        heads are still computing (engine.FusedPointNet2.forward)."""
        points = data_batch["scene_points"]
        if fused is None:
            fused = (not self.training) and (not torch.is_grad_enabled()) and points.is_cuda and self.fusable()
        if fused:
            if not self.fusable(allow_global=True):
                raise RuntimeError("the fused engine has no plan for this configuration (see PointNet2.fusable); "
                                   "call with fused=False for the module path")
            return self.fused_engine().forward(points, host_out=host_out)
        return self.forward_modules(points)

    def init_weights(self):
        pass

    def predictions(self, raw, points):
        """The prediction dict from the raw head outputs {score, frame_R, frame_t, movable_logits (after the sigmoid)}
        of the trunk + heads (module path, fused engine, training engine).  PN2_CLS emits them as they are; the PN2
        sibling maps them (models/PointNet2.py)."""
        return raw


class PointNet2Loss(nn.Module):
    """Reference PointNet2_tcls.py:156-219: weighted CE on the score classes (class 0 down-weighted),
    L1 on the movable directions, flip-symmetric rotation MSE weighted by the ground-truth score (x5)
    and CE on the 4 approach-offset classes (x0.2).  The reference reads ``preds["scene_score_logits"]``
    although this model's forward emits ``"score"`` (:142,:163); both keys are accepted."""

    def __init__(self, label_smoothing=0, neg_weight=0.1):
        super().__init__()
        self.label_smoothing = label_smoothing
        self.neg_weight = neg_weight

    def forward(self, preds, labels):
        logits = preds["scene_score_logits"] if "scene_score_logits" in preds else preds["score"]
        weight = torch.ones(logits.shape[1], device=logits.device)
        weight[0] = self.neg_weight
        if self.label_smoothing > 0:  # reference :177-180
            cls_loss = smooth_cross_entropy(logits.transpose(1, 2).reshape(-1, logits.shape[1]),
                                            labels["scene_score_labels"].reshape(-1), float(self.label_smoothing),
                                            weight=weight)
        else:
            cls_loss = F.cross_entropy(logits, labels["scene_score_labels"], weight)
        mov_loss = F.l1_loss(preds["movable_logits"], labels["scene_movable_labels"])

        gt_R = labels["best_frame_R"]
        n = gt_R.shape[2]
        pred_R = preds["frame_R"][:, :, :n]
        flip = gt_R.new_tensor([1, -1, -1, 1, -1, -1, 1, -1, -1]).view(1, 9, 1)  # columns 1,2 negated
        loss_a = ((pred_R - gt_R) ** 2).mean(1)
        loss_b = ((pred_R - gt_R * flip) ** 2).mean(1)
        R_loss = (torch.minimum(loss_a, loss_b) * labels["scene_score"][:, :n]).mean() * 5.0
        t_loss = F.cross_entropy(preds["frame_t"][:, :, :n], labels["best_frame_t"]) * 0.2
        return {"cls_loss": cls_loss, "R_loss": R_loss, "t_loss": t_loss, "mov_loss": mov_loss}


def _rotation_angle(gt, pred):
    """Angle of gt · predᵀ from its trace, clamped like the reference (:246-247); gt, pred (n, 3, 3)."""
    tr = torch.einsum("nij,nij->n", gt, pred)  # trace(gt @ pred^T) = sum_ij gt_ij pred_ij
    return torch.acos(torch.clamp((tr - 1.0) / 2.0, -1.0, 1.0))


class PointNet2Metric(nn.Module):
    """Reference PointNet2_tcls.py:222-268: per-point score-class accuracy, movable-direction accuracy (> 0.5),
    score-weighted rotation angle to the closer of the ground-truth frame and its 180-degree flip about x (columns 1, 2
    negated), approach-offset class accuracy.  ``cls_acc`` / ``mov_acc`` / ``t_acc`` are per-element 0/1 tensors (the
    reference's meters average them), ``R_err`` is a scalar.  Accepts the score logits under either key (see the loss)."""

    def forward(self, preds, labels):
        logits = preds["scene_score_logits"] if "scene_score_logits" in preds else preds["score"]
        cls_acc = (logits.argmax(1).reshape(-1) == labels["scene_score_labels"].reshape(-1)).float()
        mov_acc = ((preds["movable_logits"] > 0.5).reshape(-1).int() ==
                   labels["scene_movable_labels"].reshape(-1).int()).float()
        gt = labels["best_frame_R"]
        b, _, n = gt.shape
        gt = gt.transpose(1, 2).reshape(b * n, 3, 3)
        pred = preds["frame_R"][:, :, :n].transpose(1, 2).reshape(b * n, 3, 3)
        gt_flip = gt * gt.new_tensor([1.0, -1.0, -1.0])  # broadcast over the column index
        angle = torch.minimum(_rotation_angle(gt, pred), _rotation_angle(gt_flip, pred))
        R_err = (labels["scene_score"][:, :n].reshape(-1) * angle).mean()
        t_acc = (preds["frame_t"][:, :, :n].argmax(1).reshape(-1) == labels["best_frame_t"].reshape(-1)).float()
        return {"cls_acc": cls_acc, "mov_acc": mov_acc, "R_err": R_err, "t_acc": t_acc}


def build_pointnet2_cls(cfg=None):
    """Reference build_pointnet2_cls (:270-290).  ``cfg`` may be a yacs-style node (MODEL.PN2.*, DATA.*)
    or None for the shipped curvature_model.yaml values."""
    if cfg is None:
        net = PointNet2(**PN2_CLS_CONFIG)
        return net, PointNet2Loss(label_smoothing=0.0, neg_weight=0.5), PointNet2Metric()
    pn2 = cfg.MODEL.PN2
    net = PointNet2(score_classes=cfg.DATA.SCORE_CLASSES, num_centroids=pn2.NUM_CENTROIDS, radius=pn2.RADIUS,
                    num_neighbours=pn2.NUM_NEIGHBOURS, sa_channels=pn2.SA_CHANNELS, fp_channels=pn2.FP_CHANNELS,
                    num_fp_neighbours=pn2.NUM_FP_NEIGHBOURS, seg_channels=pn2.SEG_CHANNELS,
                    num_removal_directions=cfg.DATA.NUM_REMOVAL_DIRECTIONS, dropout_prob=pn2.DROPOUT_PROB)
    return net, PointNet2Loss(label_smoothing=pn2.LABEL_SMOOTHING, neg_weight=pn2.NEG_WEIGHT), PointNet2Metric()
