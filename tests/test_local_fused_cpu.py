"""CPU suite for PN2_LOCAL on the fused path: which configurations PointNet2_local.PointNet2.fusable accepts, the errors
fused=True raises before any GPU work, the cached engine's lifetime, and PN2_CLS's answers after the trunk rules moved
into shared code."""
import copy
import pickle

import pytest
import torch

from tests.test_global_level_cpu import GLOBAL_CFG, test_allow_global_rejects as _cls_rejects
from tests.test_pn2_local import CFG as GOLDEN_CFG

# the PN2_CLS reject table of the global-level suite, reused as it stands
CLS_REJECTS = _cls_rejects.pytestmark[0].args[1]


def _local(**overrides):
    from s4g_release_b200.network_models.models.PointNet2_local import PointNet2
    return PointNet2(**dict(GOLDEN_CFG, **overrides))


def test_class_defaults_are_fusable_only_with_allow_global():
    from s4g_release_b200.network_models.models.PointNet2_local import PointNet2
    net = PointNet2(score_classes=3)
    assert not net.fusable() and net.fusable(allow_global=True)


def test_golden_configuration_is_fusable():
    assert _local().fusable(allow_global=True)


def test_configuration_without_global_level_is_fusable():
    net = _local(num_centroids=(256, 64, 16), radius=(0.1, 0.2, 0.4), num_neighbours=(16, 16, 8),
                 sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128)), fp_channels=((64, 64), (32, 32), (32, 32, 16)),
                 num_fp_neighbours=(3, 3, 3))
    assert net.fusable() and net.fusable(allow_global=True)


@pytest.mark.parametrize("overrides, why", [
    (dict(seg_channels=(40,)), "head width not a multiple of 16"),
    (dict(fp_channels=((64, 64), (64, 32), (32, 32), (32, 32, 24))), "point feature width not a multiple of 16"),
    (dict(sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 120, 256))), "global width not a multiple of 16"),
    (dict(seg_channels=(640,)), "head width > 512"),
    (dict(seg_channels=(32, 528)), "head width > 512"),
    (dict(score_classes=17), "more than 16 evaluation classes"),
    (dict(num_centroids=(256, 64, 0, 16), radius=(0.1, 0.2, -1.0, 0.4), num_neighbours=(16, 16, -1, 8)),
     "global level not last"),
    (dict(num_fp_neighbours=(3, 3, 3, 3)), "global level followed by 3-NN propagation"),
    (dict(num_neighbours=(16, 16, 12, -1)), "neighbourhood of 12 on a sampled level"),
])
def test_fusable_rejects(overrides, why):
    net = _local(**overrides)
    assert not net.fusable(allow_global=True) and not net.fusable(), why


def test_fused_true_on_an_unsupported_config_raises_before_any_gpu_work():
    net = _local(num_fp_neighbours=(3, 3, 3, 3)).eval()
    pts = torch.zeros(1, 3, 512)
    for batch in ({"scene_points": pts}, {"scene_points": pts, "local_search_frame": torch.zeros(1, 12, 8, 2)}):
        with torch.no_grad(), pytest.raises(RuntimeError, match="fused=False"):
            net(batch, fused=True)
    assert net._engine is None


@pytest.mark.parametrize("frames, match", [
    (torch.zeros(1, 12, 8), "n_frames, n_search"),
    (torch.zeros(2, 12, 8, 2), "B = 1"),
    (torch.zeros(1, 11, 8, 2), "n_frames, n_search"),
    (torch.zeros(1, 12, 8, 2, dtype=torch.float64), "float32"),
    (torch.zeros(1, 12, 2, 8).transpose(2, 3), "strided"),
    (torch.zeros(1, 12, 513, 2), "n_frames <= 512"),
    (torch.zeros(1, 12, 0, 2), "n_frames <= 512"),
    (torch.zeros(1, 12, 8, 0), "n_search >= 1"),
])
def test_invalid_frames_raise_before_any_gpu_work(frames, match):
    net = _local().eval()
    with torch.no_grad(), pytest.raises(ValueError, match=match):
        net({"scene_points": torch.zeros(1, 3, 512), "local_search_frame": frames}, fused=True)
    assert net._engine is None


def test_engine_cache_is_dropped_by_copies_and_invalidated_by_updates():
    net = _local().eval()
    sentinel = object()
    net.attach_engine(sentinel)
    assert net.fused_engine() is sentinel
    assert copy.deepcopy(net)._engine is None and net._engine is sentinel
    assert pickle.loads(pickle.dumps(net))._engine is None and net._engine is sentinel
    key = net._engine_key
    with torch.no_grad():
        net.grasp_eval_logit.bias.add_(1.0)  # in-place update (optimizer / EMA style)
    assert net._param_fingerprint() != key
    for invalidate in (lambda: net.load_state_dict(net.state_dict()), lambda: net.train(), lambda: net.float()):
        net.attach_engine(sentinel)
        invalidate()
        assert net._engine is None


def test_module_path_stays_the_default():
    """fused=None and fused=False run the module path on the CPU without touching the engine"""
    torch.manual_seed(0)
    net = _local().eval()
    assert net.config["seg_channels"] == GOLDEN_CFG["seg_channels"]
    with torch.no_grad(), pytest.raises(RuntimeError, match="CUDA tensor"):
        net({"scene_points": torch.rand(1, 3, 512)})
    assert net._engine is None


def test_pn2_cls_fusable_answers_unchanged():
    from s4g_release_b200.network_models.models.PointNet2_tcls import PN2_CLS_CONFIG, PointNet2
    from tests.inputs import TINY_CONFIG
    for overrides, why in CLS_REJECTS:
        net = PointNet2(**dict(GLOBAL_CFG, **overrides))
        assert not net.fusable() and not net.fusable(allow_global=True), why
    net = PointNet2(**GLOBAL_CFG)
    assert net.fusable(allow_global=True) and not net.fusable()
    for cfg in (PN2_CLS_CONFIG, TINY_CONFIG):
        assert PointNet2(**cfg).fusable() and PointNet2(**cfg).fusable(allow_global=True)
    assert not PointNet2(**dict(TINY_CONFIG, seg_channels=(64, 32, 40))).fusable()
    assert not PointNet2(**dict(TINY_CONFIG, num_removal_directions=17)).fusable()
