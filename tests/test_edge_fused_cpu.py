"""CPU suite for EDGEPN2D on the fused path: the edge-level weight split, which configurations
EdgePointNet2Down.fusable accepts, the errors fused=True and the training engine raise before any GPU work, the
module-path default, and the planner / ABI rules of edge chains (in_mode 6)."""
import ctypes

import pytest
import torch

from tests.test_edge_models import CFG as GOLDEN_CFG

IN_GATHER, IN_GATHER_EDGE, IN_ROWS, OUT_ROWS, OUT_MAXPOOL = 1, 6, 0, 2, 3
NO_GLOBAL_CFG = dict(GOLDEN_CFG, num_centroids=(256, 64, 16), radius=(0.1, 0.2, 0.4), num_neighbours=(16, 16, 8),
                     sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128)),
                     fp_channels=((64, 32), (32, 32), (32, 32, 16)), num_fp_neighbours=(3, 3, 3))


def _edge(**overrides):
    from s4g_release_b200.network_models.models.EdgePointNet2Down import EdgePointNet2Down
    return EdgePointNet2Down(**dict(GOLDEN_CFG, **overrides))


@pytest.mark.parametrize("c, cout", [(1, 4), (32, 16), (64, 128)])
def test_edge_weight_split_equals_the_edge_row_product(c, cout):
    """[W_x | W_a + W_b] [x; f_j] + b - W_b f_c == W [x | f_j | f_j - f_c] + b, columns [xyz | neighbour | difference]"""
    from s4g_release_b200.engine import FusedEdgePointNet2Down
    g = torch.Generator().manual_seed(c * 100 + cout)
    w = torch.randn(cout, 3 + 2 * c, generator=g, dtype=torch.float64)
    b = torch.randn(cout, generator=g, dtype=torch.float64)
    x = torch.randn(500, 3, generator=g, dtype=torch.float64)
    f_j = torch.randn(500, c, generator=g, dtype=torch.float64)
    f_c = torch.randn(500, c, generator=g, dtype=torch.float64)
    w_plain, w_u = FusedEdgePointNet2Down.split_edge_layer(w, c)
    assert tuple(w_plain.shape) == (cout, 3 + c) and tuple(w_u.shape) == (cout, c)
    split = torch.cat([x, f_j], 1) @ w_plain.t() + b + f_c @ w_u.t()
    literal = torch.cat([x, f_j, f_j - f_c], 1) @ w.t() + b
    assert (split - literal).abs().max().item() <= 1e-12 * max(1.0, literal.abs().max().item())
    with pytest.raises(AssertionError):
        FusedEdgePointNet2Down.split_edge_layer(w[:, :-1], c)


def test_fusable_answers():
    from s4g_release_b200.network_models.models.EdgePointNet2Down import EdgePointNet2Down
    from s4g_release_b200.network_models.models.PointNet2 import PointNet2
    net = _edge()
    assert net.fusable(allow_global=True) and not net.fusable()  # the golden configuration has a global level
    assert _edge(**NO_GLOBAL_CFG).fusable()
    defaults = EdgePointNet2Down(score_classes=3)
    assert defaults.fusable(allow_global=True) and not defaults.fusable()
    one_layer = dict(sa_channels=((16, 16, 32), (32,), (64, 64, 128), (128, 128, 256)))
    assert PointNet2(**dict(GOLDEN_CFG, **one_layer)).fusable(allow_global=True)  # the sibling has a plan for it ...
    assert not _edge(**one_layer).fusable(allow_global=True)  # ... an edge level of one layer has none
    # a one-layer FIRST level has no input features: it is not an edge level
    assert _edge(sa_channels=((32,), (32, 32, 64), (64, 64, 128), (128, 128, 256))).fusable(allow_global=True)
    assert not _edge(num_centroids=(256, -1, 16, 0)).fusable(allow_global=True)
    assert not _edge(num_fp_neighbours=(3, 3, 3, 3)).fusable(allow_global=True)


def test_fused_true_on_an_unsupported_config_raises_before_any_gpu_work():
    net = _edge(sa_channels=((16, 16, 32), (32,), (64, 64, 128), (128, 128, 256))).eval()
    with torch.no_grad(), pytest.raises(RuntimeError, match="no plan"):
        net({"scene_points": torch.zeros(1, 3, 512)}, fused=True)
    assert net._engine is None


def test_module_path_stays_the_default():
    """fused=None and fused=False run the module path (here on the CPU, which the sm_100a operators refuse) for a
    configuration fusable() accepts, without touching the engine"""
    net = _edge(**NO_GLOBAL_CFG).eval()
    assert net.fusable()
    for fused in (None, False):
        with torch.no_grad(), pytest.raises(RuntimeError, match="CUDA tensor"):
            net({"scene_points": torch.rand(1, 3, 512)}, fused=fused)
    assert net._engine is None


@pytest.mark.parametrize("cfg", [GOLDEN_CFG, NO_GLOBAL_CFG], ids=["global", "no_global"])
def test_fused_training_of_edge_levels_is_refused(cfg):
    from s4g_release_b200.network_models.models.PointNet2 import PointNet2Loss
    from s4g_release_b200.train import Trainer
    from s4g_release_b200.train_engine import TrainEngine
    net = _edge(**cfg)
    with pytest.raises(RuntimeError, match="edge set-abstraction"):
        TrainEngine(net, PointNet2Loss())
    with pytest.raises(RuntimeError, match="edge set-abstraction"):
        Trainer(net, PointNet2Loss(), fused=True)


def _arr(v):
    return (ctypes.c_int * len(v))(*v)


def _create(dims, in_mode, feat_c, out_mode, group):
    from s4g_release_b200._lib import lib
    n = len(dims) - 1
    return lib.s4g_chain_create(n, _arr(dims[:-1]), _arr(dims[1:]), _arr([1] * n), in_mode, feat_c, out_mode, dims[-1],
                                group, 0)


def test_edge_chains_plan_like_gathered_chains():
    """the planner treats an edge chain as the plain gathered chain of the same shape: the same job streams"""
    from s4g_release_b200._lib import lib
    for dims, feat_c, group in (([35, 32, 32, 64], 32, 16), ([67, 64, 64, 128], 64, 16), ([131, 64, 64, 128], 128, 64),
                                ([259, 128, 128, 256], 256, 64)):
        texts = []
        for mode in (IN_GATHER, IN_GATHER_EDGE):
            h = _create(dims, mode, feat_c, OUT_MAXPOOL, group)
            assert h, lib.s4g_last_error()
            buf = ctypes.create_string_buffer(1 << 16)
            lib.s4g_chain_describe(h, buf, len(buf))
            texts.append(buf.value)
            lib.s4g_chain_destroy(h)
        assert texts[0] == texts[1], dims


def test_edge_chain_rules_need_no_gpu():
    from s4g_release_b200._lib import lib
    assert not _create([35, 64], IN_GATHER_EDGE, 32, OUT_MAXPOOL, 16)  # one layer: layer 0 is the max-pool
    assert b"edge chain" in lib.s4g_last_error()
    assert not _create([35, 32, 64], IN_GATHER_EDGE, 32, OUT_ROWS, 1)  # not a max-pool chain
    assert not _create([3, 32, 64], IN_GATHER_EDGE, 0, OUT_MAXPOOL, 16)  # no feature table
    edge = _create([35, 32, 64], IN_GATHER_EDGE, 32, OUT_MAXPOOL, 16)
    plain = _create([35, 32, 64], IN_GATHER, 32, OUT_MAXPOOL, 16)
    assert edge and plain
    d = ctypes.c_void_p(16)
    try:
        assert lib.s4g_chain_run_gather(edge, d, d, d, d, 1, 64, 4, 16, d, None) != 0
        assert b"run_gather_term" in lib.s4g_last_error()
        assert lib.s4g_chain_run_gather_term(plain, d, d, d, d, d, 1, 64, 4, 16, d, None) != 0
        assert b"needs an edge chain" in lib.s4g_last_error()
        assert lib.s4g_chain_run_gather_term(edge, d, d, d, d, None, 1, 64, 4, 16, d, None) != 0
        assert b"group term" in lib.s4g_last_error()
    finally:
        lib.s4g_chain_destroy(edge)
        lib.s4g_chain_destroy(plain)


def test_gather_rows_argument_errors_need_no_gpu():
    from s4g_release_b200._lib import lib
    d = ctypes.c_void_p(16)
    assert lib.s4g_gather_rows_bf16(d, d, 1, 8, 4, 12, d, None) != 0  # C % 8 != 0
    assert lib.s4g_gather_rows_bf16(ctypes.c_void_p(18), d, 1, 8, 4, 16, d, None) != 0  # misaligned rows
    assert lib.s4g_gather_rows_bf16(None, d, 1, 8, 4, 16, d, None) != 0
