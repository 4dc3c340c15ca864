"""CPU suite for EDGEPN2DU on the fused path: the split of an edge propagation level's first layer, which configurations
EdgePointNet2DownUp.fusable accepts, the error fused=True raises before any GPU work, the module-path default, the
unchanged state_dict, the cached engine's lifetime, and the argument checks of the two new kernels."""
import copy
import ctypes
import pickle

import pytest
import torch

from tests.test_edge_models import CFG as GOLDEN_CFG

NO_GLOBAL_CFG = dict(GOLDEN_CFG, num_centroids=(256, 64, 16), radius=(0.1, 0.2, 0.4), num_neighbours=(16, 16, 8),
                     sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128)),
                     fp_channels=((64, 32), (32, 32), (32, 32, 16)), num_fp_neighbours=(3, 3, 3))


def _downup(**overrides):
    from s4g_release_b200.network_models.models.EdgePointNet2DownUp import EdgePointNet2DownUp
    return EdgePointNet2DownUp(**dict(GOLDEN_CFG, **overrides))


@pytest.mark.parametrize("c2, c1, cout, weights", [(1, 3, 4, "normalised"), (48, 24, 64, "free"), (128, 3, 64, "free"),
                                                   (32, 64, 16, "normalised")])
def test_edge_fp_split_equals_the_literal_edge_rows(c2, c1, cout, weights):
    """sum_j w_j U[idx_j] + V[idx_k] + T + b == W' [interp | n_k - interp | d] + b per (q, k), in fp64, also for
    interpolation weights that do not sum to one"""
    from s4g_release_b200.engine import FusedEdgePointNet2DownUp
    g = torch.Generator().manual_seed(c2 * 1000 + c1 * 10 + cout)
    f64 = dict(generator=g, dtype=torch.float64)
    Nk, Nq = 50, 300
    w = torch.randn(cout, 2 * c2 + c1, **f64)
    b = torch.randn(cout, **f64)
    S = torch.randn(Nk, c2, **f64)
    d = torch.randn(Nq, c1, **f64)
    idx = torch.randint(0, Nk, (Nq, 3), generator=g)
    wt = torch.rand(Nq, 3, **f64) * 2.0
    if weights == "normalised":
        wt = wt / wt.sum(1, keepdim=True)
    else:
        assert (wt.sum(1) - 1).abs().max() > 0.1
    w_uv, w_d = FusedEdgePointNet2DownUp.split_edge_fp_layer(w, c2)
    assert tuple(w_uv.shape) == (2 * cout, c2) and tuple(w_d.shape) == (cout, c1)
    uv = S @ w_uv.t()
    U, V = uv[:, :cout], uv[:, cout:]
    split = (wt.unsqueeze(-1) * U[idx]).sum(1, keepdim=True) + V[idx] + (d @ w_d.t()).unsqueeze(1) + b  # (Nq, 3, cout)
    interp = (wt.unsqueeze(-1) * S[idx]).sum(1, keepdim=True).expand(-1, 3, -1)
    rows = torch.cat([interp, S[idx] - interp, d.unsqueeze(1).expand(-1, 3, -1)], dim=-1)
    literal = rows @ w.t() + b
    assert (split - literal).abs().max().item() <= 1e-12 * max(1.0, literal.abs().max().item())
    with pytest.raises(AssertionError):
        FusedEdgePointNet2DownUp.split_edge_fp_layer(w[:, :2 * c2], c2)


def test_fusable_answers():
    from s4g_release_b200.network_models.models.EdgePointNet2DownUp import EdgePointNet2DownUp
    net = _downup()
    assert net.fusable(allow_global=True) and not net.fusable()  # the golden configuration has a global level
    assert _downup(**NO_GLOBAL_CFG).fusable()
    defaults = EdgePointNet2DownUp(score_classes=3)
    assert defaults.fusable(allow_global=True) and not defaults.fusable()
    # a one-layer edge set-abstraction level has no plan (EDGEPN2D's rule) ...
    assert not _downup(sa_channels=((16, 16, 32), (32,), (64, 64, 128), (128, 128, 256))).fusable(allow_global=True)
    # ... a one-layer edge propagation level has one: its first layer's rows go straight to the mean
    assert _downup(fp_channels=((64, 64), (64,), (32, 32), (32, 32, 16))).fusable(allow_global=True)
    # the first layer of an edge propagation level at most 512 wide: [U | V] is 2 x that width
    assert _downup(fp_channels=((64, 64), (512, 32), (32, 32), (32, 32, 16))).fusable(allow_global=True)
    assert not _downup(fp_channels=((64, 64), (528, 32), (32, 32), (32, 32, 16))).fusable(allow_global=True)
    assert not _downup(fp_channels=((64, 64), (64, 32), (32, 32), (1024, 32, 16))).fusable(allow_global=True)
    # ... which does not bind the broadcast level (the sibling's, no [U | V])
    assert _downup(fp_channels=((1024, 64), (64, 32), (32, 32), (32, 32, 16))).fusable(allow_global=True)
    assert not _downup(seg_channels=(40,)).fusable(allow_global=True)
    assert not _downup(score_classes=17).fusable(allow_global=True)
    assert not _downup(num_centroids=(256, -1, 16, 0)).fusable(allow_global=True)


def test_fused_true_on_an_unsupported_config_raises_before_any_gpu_work():
    net = _downup(fp_channels=((64, 64), (528, 32), (32, 32), (32, 32, 16))).eval()
    with torch.no_grad(), pytest.raises(RuntimeError, match="no plan"):
        net({"scene_points": torch.zeros(1, 3, 512)}, fused=True)
    assert net._engine is None


def test_module_path_stays_the_default():
    """fused=None and fused=False run the module path (here on the CPU, which the sm_100a operators refuse) for a
    configuration fusable() accepts, without touching the engine"""
    net = _downup(**NO_GLOBAL_CFG).eval()
    assert net.fusable()
    for kwargs in ({}, {"fused": None}, {"fused": False}):
        with torch.no_grad(), pytest.raises(RuntimeError, match="CUDA tensor"):
            net({"scene_points": torch.rand(1, 3, 512)}, **kwargs)
    assert net._engine is None


def test_state_dict_keys_are_unchanged():
    """the config dict and the engine cache are plain attributes: the keys are the reference constructor's, the ones of
    the golden EdgePointNet2Down plus the two heads it has instead of four"""
    import os

    import numpy as np
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "edge_models.npz"))
    ref = [k[3:] for k in gold.files if k.startswith("sd/")]
    keys = list(_downup().state_dict())
    assert [k for k in keys if k.startswith("sa_modules.")] == [k for k in ref if k.startswith("sa_modules.")]
    assert all(k.split(".")[0] in ("sa_modules", "fp_modules", "mlp_seg", "seg_logit", "mlp_frame", "frame_logit")
               for k in keys)
    assert not any("config" in k or "engine" in k for k in keys)
    assert len(keys) == len(set(keys))


def test_engine_cache_is_dropped_by_copies_and_invalidated_by_updates():
    net = _downup().eval()
    sentinel = object()
    net.attach_engine(sentinel)
    assert net.fused_engine() is sentinel
    assert copy.deepcopy(net)._engine is None and net._engine is sentinel
    assert pickle.loads(pickle.dumps(net))._engine is None and net._engine is sentinel
    key = net._engine_key
    with torch.no_grad():
        net.frame_logit.bias.add_(1.0)  # in-place update (optimizer / EMA style)
    assert net._param_fingerprint() != key
    for invalidate in (lambda: net.load_state_dict(net.state_dict()), lambda: net.train(), lambda: net.to(torch.float32)):
        net.attach_engine(sentinel)
        invalidate()
        assert net._engine is None


def test_fused_training_of_edge_models_is_still_refused():
    from s4g_release_b200.network_models.models.PointNet2 import PointNet2Loss
    from s4g_release_b200.train import Trainer
    with pytest.raises(RuntimeError, match="edge set-abstraction"):
        Trainer(_downup(), PointNet2Loss(), fused=True)


def test_new_kernels_argument_errors_need_no_gpu():
    from s4g_release_b200._lib import lib
    d = ctypes.c_void_p(16)
    # (uv, index, weight, t_rows, xyz, w_xyz, shift, B, Nk, Nq, C, out, stream); every call fails its checks before a launch
    assert lib.s4g_edge_interp_rows_bf16(d, d, d, d, d, d, d, 1, 8, 8, 64, d, None) != 0  # both skip kinds
    assert b"exactly one" in lib.s4g_last_error()
    assert lib.s4g_edge_interp_rows_bf16(d, d, d, None, None, None, d, 1, 8, 8, 64, d, None) != 0  # no skip
    assert lib.s4g_edge_interp_rows_bf16(d, d, d, None, d, None, d, 1, 8, 8, 64, d, None) != 0  # cloud without W_d
    assert b"w_xyz" in lib.s4g_last_error()
    assert lib.s4g_edge_interp_rows_bf16(d, d, d, d, None, None, d, 1, 8, 8, 60, d, None) != 0  # C % 8 != 0
    assert lib.s4g_edge_interp_rows_bf16(ctypes.c_void_p(18), d, d, d, None, None, d, 1, 8, 8, 64, d, None) != 0
    assert lib.s4g_edge_interp_rows_bf16(None, d, d, d, None, None, d, 1, 8, 8, 64, d, None) != 0
    assert lib.s4g_rows_group_mean_bf16(d, 4, 12, d, None) != 0  # C % 8 != 0
    assert lib.s4g_rows_group_mean_bf16(ctypes.c_void_p(18), 4, 16, d, None) != 0  # misaligned rows
    assert lib.s4g_rows_group_mean_bf16(None, 4, 16, d, None) != 0
    assert lib.s4g_rows_group_mean_bf16(d, 1 << 28, 64, d, None) != 0  # R * C / 8 >= 2^31
