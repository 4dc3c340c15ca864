"""CPU suite for the fused training step of configurations with a global set-abstraction level (num_centroids = 0) and
broadcast propagation (num_fp_neighbours[0] = 0): which configurations TrainEngine accepts, the PN2 sibling's loss
being separable head by head under its prediction mapping, and the labels of the sibling's translation head.  The
kernels and the step itself: tests/test_global_level_train_gpu.py."""
import hashlib

import numpy as np
import pytest
import torch

from s4g_release_b200 import train_engine as te

# one block per MLP, a global level over 64 points
G_SHALLOW = dict(score_classes=3, num_centroids=(256, 64, 0), radius=(0.1, 0.2, -1.0), num_neighbours=(16, 16, -1),
                 sa_channels=((32,), (64,), (128,)), fp_channels=((128,), (64,), (64,)), num_fp_neighbours=(0, 3, 3),
                 seg_channels=(32,), num_removal_directions=5, dropout_prob=0.0)
# a global level over 1 000 points: more than the 255 rows a uint8 arg-max can address, not a power of two
G_WIDE = dict(G_SHALLOW, num_centroids=(1000, 0), radius=(0.1, -1.0), num_neighbours=(16, -1), sa_channels=((32,), (64,)),
              fp_channels=((64,), (64,)), num_fp_neighbours=(0, 3))


def _tcls(**cfg):
    from s4g_release_b200.network_models.models.PointNet2_tcls import PointNet2
    return PointNet2(**cfg)


def _sibling(**cfg):
    from s4g_release_b200.network_models.models.PointNet2 import PointNet2
    return PointNet2(**cfg)


def _engine(net):
    from s4g_release_b200.network_models.models import PointNet2, PointNet2_tcls
    loss = (PointNet2.PointNet2Loss if isinstance(net, PointNet2.PointNet2) else PointNet2_tcls.PointNet2Loss)()
    return te.TrainEngine(net, loss)


@pytest.mark.parametrize("name, make", [
    ("class defaults", lambda: _tcls(score_classes=3)),
    ("sibling defaults", lambda: _sibling(score_classes=3)),
    ("G_SHALLOW", lambda: _tcls(**G_SHALLOW)),
    ("G_WIDE", lambda: _tcls(**G_WIDE)),
    ("G_SHALLOW sibling", lambda: _sibling(**G_SHALLOW)),
])
def test_engine_accepts(name, make):
    eng = _engine(make())
    assert eng.global_level, name


@pytest.mark.parametrize("overrides, why", [
    (dict(num_centroids=(0,), radius=(-1.0,), num_neighbours=(-1,), sa_channels=((32,),), fp_channels=((64,),),
          num_fp_neighbours=(0,)), "global first level"),
    (dict(num_centroids=(256, 0, 64), radius=(0.1, -1.0, 0.2), num_neighbours=(16, -1, 16)), "global level not last"),
    (dict(num_fp_neighbours=(3, 3, 3)), "global level followed by 3-NN propagation"),
    (dict(num_centroids=(256, 64, 16), radius=(0.1, 0.2, 0.4), num_neighbours=(16, 16, 8)),
     "broadcast propagation without a global level"),
])
def test_engine_refuses(overrides, why):
    for make in (_tcls, _sibling):
        with pytest.raises(RuntimeError, match="no fused plan"):
            _engine(make(**dict(G_SHALLOW, **overrides)))


def test_configurations_without_a_global_level_keep_their_answer():
    from tests.inputs import TINY_CONFIG
    assert not _engine(_tcls(**TINY_CONFIG)).global_level
    with pytest.raises(RuntimeError):
        _engine(_tcls(**dict(TINY_CONFIG, num_neighbours=(16, 16, 12))))


def test_sibling_loss_is_separable_under_its_prediction_mapping():
    """TrainEngine._separable for the PN2 sibling: term k of its PointNet2Loss depends on raw head k only once the raw
    outputs went through the sibling's mapping (toRotMatrix, points + offset), and with the placeholders step_loss
    feeds for the other heads every term keeps its value and stays finite (toRotMatrix(0) would be 0 / 0)."""
    from s4g_release_b200.network_models.models.PointNet2 import PointNet2Loss
    from s4g_release_b200.train import synthetic_labels
    B, N, M = 2, 64, 40
    net = _sibling(**G_SHALLOW)
    eng = _engine(net)
    labels = synthetic_labels(B, N, num_frame=M, first_seed=3, continuous_t=True)
    g = torch.Generator().manual_seed(0)
    points = torch.rand(B, 3, N, generator=g)
    shapes = [(B, 3, N), (B, 6, N), (B, 3, N), (B, 5, N)]
    leaves = [torch.randn(s, generator=g).requires_grad_(True) for s in shapes]

    def preds(ls):
        raw = dict(zip(te.TrainEngine.PRED_KEYS, ls[:3]), movable_logits=torch.sigmoid(ls[3]))
        return net.predictions(raw, points)

    loss_fn = PointNet2Loss(neg_weight=0.5)
    losses = loss_fn(preds(leaves), labels)
    assert tuple(losses) == te.TrainEngine.LOSS_KEYS
    for k, key in enumerate(te.TrainEngine.LOSS_KEYS):
        grads = torch.autograd.grad(losses[key], leaves, retain_graph=True, allow_unused=True)
        for j, gr in enumerate(grads):
            if j == k:
                assert gr is not None and gr.abs().sum() > 0, key
            else:
                assert gr is None or gr.abs().sum() == 0, (key, j)
    eng._batch, eng._n_points = B, N
    holders = [eng._placeholder(k) for k in range(4)]
    assert [tuple(h.shape) for h in holders] == shapes
    for k, key in enumerate(te.TrainEngine.LOSS_KEYS):
        only = loss_fn(preds([leaves[j] if j == k else holders[j] for j in range(4)]), labels)
        assert all(torch.isfinite(v) for v in only.values()), (key, only)
        assert torch.allclose(only[key], losses[key]), key
        assert torch.autograd.grad(only[key], leaves[k])[0].isfinite().all(), key


def test_pn2_cls_placeholders_are_zeros():
    eng = _engine(_tcls(**G_SHALLOW))
    eng._batch, eng._n_points = 2, 10
    assert all(torch.equal(eng._placeholder(k), torch.zeros_like(eng._placeholder(k))) for k in range(4))


def _digest(labels):
    h = hashlib.sha256()
    for k in sorted(labels):
        t = labels[k].numpy()
        h.update(k.encode())
        h.update(str(t.dtype).encode())
        h.update(str(t.shape).encode())
        h.update(np.ascontiguousarray(t).tobytes())
    return h.hexdigest()


def test_synthetic_labels_default_output_is_unchanged():
    from s4g_release_b200.train import synthetic_labels
    # digest of the labels as drawn before continuous_t existed
    assert _digest(synthetic_labels(3, 500, num_frame=200, first_seed=7)) == \
        "d4bed2512325cc8abbd1baaecdd959e821b5dd9d82ada5c50ceb6c4360835224"


def test_continuous_translation_labels():
    from s4g_release_b200.train import synthetic_labels
    a = synthetic_labels(3, 500, num_frame=200, first_seed=7)
    b = synthetic_labels(3, 500, num_frame=200, first_seed=7, continuous_t=True)
    t = b["best_frame_t"]
    assert t.dtype == torch.float32 and tuple(t.shape) == (3, 3, 200)
    assert (t >= 0).all() and (t < 1).all() and len(torch.unique(t)) > 1000
    for k in a:
        if k != "best_frame_t":
            assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, k
    # the draws before best_frame_t are the same
    for k in ("scene_score_labels", "scene_movable_labels", "best_frame_R"):
        assert torch.equal(a[k], b[k]), k
