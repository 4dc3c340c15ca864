"""CPU suite for PN2_LOCAL's fused training step: which configurations train_engine.LocalTrainEngine accepts (through
Trainer(fused=True) too), the refusals it shares with the trunk guard, when the loss is separable head by head, the
checks on given candidates before any GPU work, and the seeded batch generator.  The kernels and the step itself:
tests/test_local_train_gpu.py."""
import os

import numpy as np
import pytest
import torch

from s4g_release_b200 import train_engine as te
from tests.test_local_fused_cpu import GOLDEN_CFG, test_fusable_rejects as _local_rejects

LOCAL_REJECTS = _local_rejects.pytestmark[0].args[1]
NO_GLOBAL = dict(GOLDEN_CFG, num_centroids=(256, 64, 16), radius=(0.1, 0.2, 0.4), num_neighbours=(16, 16, 8),
                 sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128)), fp_channels=((64, 64), (32, 32), (32, 32, 16)),
                 num_fp_neighbours=(3, 3, 3))


def _local(**cfg):
    from s4g_release_b200.network_models.models.PointNet2_local import PointNet2
    return PointNet2(**cfg)


def _loss():
    from s4g_release_b200.network_models.models.PointNet2_local import PointNet2Loss
    return PointNet2Loss()


@pytest.mark.parametrize("name, cfg", [("class defaults", dict(score_classes=3)), ("golden", GOLDEN_CFG),
                                       ("no global level", NO_GLOBAL)])
def test_engine_and_trainer_accept(name, cfg):
    from s4g_release_b200.train import Trainer
    net = _local(**cfg)
    eng = te.engine_for(net, _loss())
    assert type(eng) is te.LocalTrainEngine and eng.global_level == (name != "no global level")
    assert te.LocalTrainEngine(net, _loss()).heads[3][1] is net.grasp_eval_logit
    tr = Trainer(net, _loss(), fused=True)
    assert type(tr.engine) is te.LocalTrainEngine
    # heads in PRED_KEYS order; element dropout on movable, channel dropout on the evaluation head, none on R and t
    p = net.config["dropout_prob"]
    drops = [[(b.drop_p, b.channel_drop) for b in blocks] for blocks, _ in eng.heads]
    assert drops[0] == drops[1] == [(0.0, False)] * len(net.mlp_R)
    assert drops[2] == [(p, False)] * len(net.mlp_movable) and drops[3] == [(p, True)] * len(net.mlp_grasp_eval)


def test_plain_train_engine_points_to_the_local_engine():
    with pytest.raises(TypeError, match="LocalTrainEngine"):
        te.TrainEngine(_local(**GOLDEN_CFG), _loss())


@pytest.mark.parametrize("overrides, why", LOCAL_REJECTS)
def test_engine_refuses_what_fusable_rejects(overrides, why):
    net = _local(**dict(GOLDEN_CFG, **overrides))
    assert not net.fusable(allow_global=True), why
    with pytest.raises(RuntimeError, match="no fused plan"):
        te.engine_for(net, _loss())
    from s4g_release_b200.train import Trainer
    with pytest.raises(RuntimeError, match="no fused plan"):
        Trainer(net, _loss(), fused=True)


def test_separable_with_given_frames_only():
    eng = te.engine_for(_local(**GOLDEN_CFG), _loss())
    assert not eng._separable()
    eng._frames = torch.zeros(2, 12, 40, 6)
    assert eng._separable()
    eng.sequential_heads = False
    assert not eng._separable()


def test_given_loss_is_separable_with_the_placeholders():
    """term k of PointNet2_local.PointNet2Loss depends on head k only, and with the placeholders the separable step
    feeds for the other heads (zeros; the evaluation head's in (B, k, F, S)) every term keeps its value"""
    from s4g_release_b200.train import synthetic_local_batch
    B, N, F, S = 2, 64, 10, 3
    eng = te.engine_for(_local(**GOLDEN_CFG), _loss())
    g = torch.Generator().manual_seed(0)
    points = torch.rand(B, 3, N, generator=g)
    frames, labels = synthetic_local_batch(points, F, S)
    shapes = [(B, 9, N), (B, 3, N), (B, 2, N), (B, 3, F, S)]
    leaves = [torch.randn(s, generator=g).requires_grad_(True) for s in shapes]
    eng._points, eng._batch, eng._n_points, eng._frames = points, B, N, frames
    loss_fn = _loss()
    losses = loss_fn(eng._predictions(leaves), labels)
    assert set(losses) == set(te.LocalTrainEngine.LOSS_KEYS)
    holders = [eng._placeholder(k) for k in range(4)]
    assert [tuple(h.shape) for h in holders] == shapes and all((h == 0).all() for h in holders)
    for k, key in enumerate(te.LocalTrainEngine.LOSS_KEYS):
        grads = torch.autograd.grad(losses[key], leaves, retain_graph=True, allow_unused=True)
        assert all((gr is None or gr.abs().sum() == 0) == (j != k) for j, gr in enumerate(grads)), key
        only = loss_fn(eng._predictions([leaves[j] if j == k else holders[j] for j in range(4)]), labels)
        assert torch.allclose(only[key], losses[key]), key


@pytest.mark.parametrize("frames, match", [
    (torch.zeros(1, 12, 8), "n_frames, n_search"),
    (torch.zeros(2, 12, 8, 2), "B = 1"),
    (torch.zeros(1, 12, 8, 2, dtype=torch.float64), "float32"),
    (torch.zeros(1, 12, 2, 8).transpose(2, 3), "strided"),
    (torch.zeros(1, 12, 513, 2), "n_frames <= 512"),
    (torch.zeros(1, 12, 8, 0), "n_search >= 1"),
])
def test_invalid_frames_raise_before_any_gpu_work(frames, match):
    net = _local(**GOLDEN_CFG)
    eng = te.engine_for(net, _loss())
    before = [p.detach().clone() for p in net.parameters()]
    with pytest.raises(ValueError, match=match):
        eng.step_loss({"scene_points": torch.zeros(1, 3, 512), "local_search_frame": frames}, {})
    assert eng.step_count == 0 and all(p.grad is None for p in net.parameters())
    assert all(torch.equal(a, b) for a, b in zip(before, net.parameters()))


def test_synthetic_local_batch():
    from s4g_release_b200.train import synthetic_local_batch
    B, N, F, S = 3, 200, 40, 6
    points = torch.rand(B, 3, N, generator=torch.Generator().manual_seed(1))
    frames, labels = synthetic_local_batch(points, F, S, score_classes=4)
    want = {"scored_grasp_labels": ((B, F, S), torch.int64), "scene_movable_labels": ((B, N), torch.int64),
            "best_frame_R": ((B, 9, F), torch.float32), "best_frame_t": ((B, 3, F), torch.float32)}
    assert {k: (tuple(v.shape), v.dtype) for k, v in labels.items()} == want
    assert tuple(frames.shape) == (B, 12, F, S) and frames.dtype == torch.float32 and frames.is_contiguous()
    assert labels["scored_grasp_labels"].min() >= 0 and labels["scored_grasp_labels"].max() == 3
    assert set(labels["scene_movable_labels"].unique().tolist()) == {0, 1}
    # rotations are orthonormal; translations lie near their point
    R = frames[:, :9].permute(0, 2, 3, 1).reshape(-1, 3, 3).double()
    assert torch.allclose(R @ R.transpose(1, 2), torch.eye(3, dtype=torch.float64).expand_as(R), atol=1e-5)
    Rl = labels["best_frame_R"].permute(0, 2, 1).reshape(-1, 3, 3).double()
    assert torch.allclose(Rl @ Rl.transpose(1, 2), torch.eye(3, dtype=torch.float64).expand_as(Rl), atol=1e-5)
    anchor = points[:, :, :F]
    assert (frames[:, 9:] - anchor.unsqueeze(-1)).abs().max() < 0.15
    assert (labels["best_frame_t"] - anchor).abs().max() < 0.15
    # seeded: the same call gives the same bits, a different seed a different batch
    f2, l2 = synthetic_local_batch(points, F, S, score_classes=4)
    assert torch.equal(frames, f2) and all(torch.equal(labels[k], l2[k]) for k in labels)
    f3, _ = synthetic_local_batch(points, F, S, score_classes=4, first_seed=1)
    assert not torch.equal(frames, f3)
    # matches the golden label layout
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pn2_local.npz"))
    _, lg = synthetic_local_batch(torch.from_numpy(g["points"]), *g["frames"].shape[2:])
    for k, v in lg.items():
        assert tuple(v.shape) == g["label/" + k].shape and str(v.dtype)[6:] == str(g["label/" + k].dtype), k
    with pytest.raises(ValueError):
        synthetic_local_batch(points, N + 1, 1)


def test_kernel_argument_errors_do_not_need_a_gpu():
    """the new entry points refuse bad shapes and rows that are not 16-byte aligned before any CUDA call"""
    import ctypes
    from s4g_release_b200._lib import lib
    a, odd = ctypes.c_void_p(256), ctypes.c_void_p(264)
    for P, rows, p in ((10, 3, 0.5), (10, 0, 0.5), (10, 5, 1.0), (1 << 31, 1 << 30, 0.5)):
        assert lib.s4g_train_bn_act_chdrop_bf16(a, a, a, a, P, 8, 1, rows, 0, p, None) != 0
    assert b"16-byte aligned" in (lib.s4g_train_bn_act_chdrop_bf16(odd, a, a, a, 10, 8, 1, 5, 0, 0.5, None) and
                                  lib.s4g_last_error())
    assert lib.s4g_train_bn_bwd_reduce_chdrop_bf16(a, odd, a, a, 10, 8, 1, 5, 0, 0.5, a, None) != 0
    assert lib.s4g_train_bn_bwd_apply_chdrop_bf16(a, a, a, a, a, a, a, 10, 8, 1, 5, 0, 0.5, odd, None) != 0
    assert lib.s4g_train_bn_act_chdrop_bf16(a, a, a, a, 10, 12, 1, 5, 0, 0.5, None) != 0  # C % 8
    # the row backward: self-mode candidate gradient with F != N, shapes, alignment
    assert lib.s4g_local_eval_rows_bwd_bf16(a, 2, 64, 16, 63, 1, a, a, a, None) != 0
    assert lib.s4g_local_eval_rows_bwd_bf16(a, 2, 64, 16, 10, 2, a, a, a, None) != 0
    assert lib.s4g_local_eval_rows_bwd_bf16(a, 2, 64, 16, 65, 1, a, None, None, None) != 0
    assert lib.s4g_local_eval_rows_bwd_bf16(a, 2, 64, 12, 10, 1, a, None, None, None) != 0
    assert lib.s4g_local_eval_rows_bwd_bf16(odd, 2, 64, 16, 10, 1, a, None, None, None) != 0
    assert lib.s4g_local_eval_rows_bwd_bf16(a, 2, 64, 16, 10, 1, a, a, None, None) != 0
