"""CPU suite for the global set-abstraction level on the fused path: which configurations fusable(allow_global=True)
accepts, and the padded identity neighbour table the engine pools a global level with."""
import numpy as np
import pytest

from tests.inputs import TINY_CONFIG

GLOBAL_CFG = dict(TINY_CONFIG, num_centroids=(256, 64, 16, 0), radius=(0.1, 0.2, 0.4, -1.0),
                  num_neighbours=(16, 16, 8, -1),
                  sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 128, 256)),
                  fp_channels=((64, 64), (64, 32), (32, 32), (32, 32, 16)), num_fp_neighbours=(0, 3, 3, 3),
                  seg_channels=(32,))


def _net(**overrides):
    from s4g_release_b200.network_models.models.PointNet2_tcls import PointNet2
    return PointNet2(**dict(GLOBAL_CFG, **overrides))


def test_class_defaults_are_fusable_only_with_allow_global():
    from s4g_release_b200.network_models.models.PointNet2 import PointNet2 as Sibling
    from s4g_release_b200.network_models.models.PointNet2_tcls import PN2_CLS_CONFIG, PointNet2
    for cls in (PointNet2, Sibling):
        net = cls(score_classes=3)
        assert not net.fusable() and net.fusable(allow_global=True)
        # configurations without a global level: allow_global changes nothing
        assert cls(**PN2_CLS_CONFIG).fusable(allow_global=True) and cls(**TINY_CONFIG).fusable(allow_global=True)
    assert _net().fusable(allow_global=True) and not _net().fusable()


def test_a_single_global_level_is_fusable():
    net = _net(num_centroids=(0,), radius=(-1.0,), num_neighbours=(-1,), sa_channels=((16, 32, 64),),
               fp_channels=((64, 32),), num_fp_neighbours=(0,))
    assert net.fusable(allow_global=True) and not net.fusable()


@pytest.mark.parametrize("overrides, why", [
    (dict(num_centroids=(256, 64, 0, 16), radius=(0.1, 0.2, -1.0, 0.4), num_neighbours=(16, 16, -1, 8)),
     "global level not last"),
    (dict(num_fp_neighbours=(3, 3, 3, 3)), "global level followed by 3-NN propagation"),
    (dict(num_fp_neighbours=(0, 3, 0, 3)), "broadcast propagation on a later level"),
    (dict(num_fp_neighbours=(0, 0, 3, 3)), "two broadcast levels"),
    (dict(num_centroids=(256, 64, 16, 8), radius=(0.1, 0.2, 0.4, 0.8), num_neighbours=(16, 16, 8, 8)),
     "broadcast propagation without a global level"),
    (dict(num_centroids=(256, 64, 16, -1), radius=(0.1, 0.2, 0.4, 0.8), num_neighbours=(16, 16, 8, 8)),
     "num_centroids == -1"),
    (dict(num_neighbours=(16, 16, 12, -1)), "neighbourhood of 12 on a sampled level"),
    (dict(sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 640, 256))), "global hidden width > 512"),
    (dict(sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 128, 2048))), "global output width > 1024"),
    (dict(sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 120, 256))), "global width not a multiple of 16"),
    (dict(fp_channels=((64, 40), (64, 32), (32, 32), (32, 32, 16))), "broadcast level width not a multiple of 16"),
    (dict(seg_channels=(640,)), "head width > 512"),
    (dict(score_classes=17), "more than 16 logits"),
])
def test_allow_global_rejects(overrides, why):
    assert not _net(**overrides).fusable(allow_global=True), why


@pytest.mark.parametrize("n, g, p", [(1, 8, 1), (7, 8, 1), (16, 16, 1), (100, 64, 2), (128, 64, 2), (25600, 64, 400)])
def test_global_group_table(n, g, p):
    from s4g_release_b200.engine import GLOBAL_GROUPS, global_group_table
    got_g, got_p, idx = global_group_table(n)
    assert (got_g, got_p) == (g, p) and got_g in GLOBAL_GROUPS
    assert idx.dtype == np.int32 and idx.shape == (p * g,)
    assert np.array_equal(idx[:n], np.arange(n))  # every point of [0, n) once, in order
    pad = idx[n:]
    assert pad.size == p * g - n < g and ((pad >= 0) & (pad < n)).all()  # padding repeats real points


def test_fused_true_on_an_unsupported_config_raises_before_any_gpu_work():
    import torch
    net = _net(num_fp_neighbours=(3, 3, 3, 3)).eval()
    with torch.no_grad(), pytest.raises(RuntimeError, match="no plan"):
        net({"scene_points": torch.zeros(1, 3, 512)}, fused=True)
