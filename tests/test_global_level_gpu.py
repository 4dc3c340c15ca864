"""GPU suite for the fused global set-abstraction level (num_centroids = 0) and the broadcast propagation level
(num_fp_neighbours = 0) paired with it, run with forward(..., fused=True):
  * the two kernels (csrc/fused_ops.cu) are bit-equal to torch;
  * the PN2 sibling with the golden weights is within engine.tolerance() of the reference's own outputs for every MLP
    backend, and the class defaults / a padded global group match the module path;
  * scenes stay independent units, the side-stream 3-NN schedule computes the serial schedule's bits, the automatic
    route is unchanged, and a fused forward launches no torch kernel."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

# the reference PN2 sibling's configuration of tests/golden/pn2_sibling.npz
SIBLING_CFG = dict(score_classes=3, num_centroids=(256, 64, 16, 0), radius=(0.1, 0.2, 0.4, -1.0),
                   num_neighbours=(16, 16, 8, -1),
                   sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 128, 256)),
                   fp_channels=((64, 64), (64, 32), (32, 32), (32, 32, 16)), num_fp_neighbours=(0, 3, 3, 3),
                   seg_channels=(32,), num_removal_directions=5, dropout_prob=0.5)
# a global level over 100 points: two partial groups of 64, the second padded with 28 repeated points
PADDED_CFG = dict(SIBLING_CFG, num_centroids=(400, 100, 0), radius=(0.1, 0.2, -1.0), num_neighbours=(16, 32, -1),
                  sa_channels=((16, 16, 32), (32, 32, 64), (64, 128, 128)), fp_channels=((64, 64), (64, 32), (32, 32)),
                  num_fp_neighbours=(0, 3, 3))
SIBLING_KEYS = ("scene_score_logits", "frame_R", "frame_t", "movable_logits")


def _rel_err(got, want):
    want = torch.as_tensor(want).float().cpu()
    return ((got.float().cpu() - want).abs().max() / max(1.0, want.abs().max().item())).item()


def _seeded(cfg, seed=0, sibling=False):
    """Default init plus non-trivial BatchNorm statistics (so the folded scale / shift are exercised)."""
    from s4g_release_b200.network_models.models.PointNet2 import PointNet2 as Sibling
    from s4g_release_b200.network_models.models.PointNet2_tcls import PointNet2
    torch.manual_seed(seed)
    net = (Sibling if sibling else PointNet2)(**cfg)
    g = torch.Generator().manual_seed(seed)
    for m in net.modules():
        if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
            n = m.num_features
            m.running_mean.copy_(0.1 * torch.randn(n, generator=g))
            m.running_var.copy_(0.5 + torch.rand(n, generator=g))
            m.weight.data.copy_(0.8 + 0.4 * torch.rand(n, generator=g))
            m.bias.data.copy_(0.1 * torch.randn(n, generator=g))
    return net.cuda().eval()


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(os.path.join(os.path.dirname(__file__), "golden", "pn2_sibling.npz")))


@pytest.mark.parametrize("B, P, C", [(1, 1, 8), (3, 1, 256), (2, 2, 1024), (4, 400, 1032), (64, 7, 72)])
def test_rows_segment_max_is_torch_amax(B, P, C):
    from s4g_release_b200.engine import FusedPointNet2
    g = torch.Generator(device="cuda").manual_seed(B * 1000 + P)
    rows = torch.randn(B * P, C, device="cuda", generator=g).to(torch.bfloat16)
    got = FusedPointNet2.rows_segment_max(rows, B)
    assert torch.equal(got, rows.view(B, P, C).amax(dim=1))


@pytest.mark.parametrize("B, Nq, C2, C1", [(1, 1, 8, 0), (3, 100, 256, 0), (2, 128, 1024, 256), (5, 37, 64, 40)])
def test_broadcast_concat_is_expand_cat(B, Nq, C2, C1):
    from s4g_release_b200.engine import FusedPointNet2
    g = torch.Generator(device="cuda").manual_seed(B * 1000 + Nq)
    sparse = torch.randn(B, C2, device="cuda", generator=g).to(torch.bfloat16)
    dense = torch.randn(B * Nq, C1, device="cuda", generator=g).to(torch.bfloat16) if C1 else None
    got = FusedPointNet2.broadcast_concat(sparse, dense, B, Nq)
    want = sparse.view(B, 1, C2).expand(B, Nq, C2)
    if dense is not None:
        want = torch.cat([want, dense.view(B, Nq, C1)], dim=-1)
    assert torch.equal(got, want.reshape(B * Nq, C2 + C1))


@pytest.mark.parametrize("backend", ["tcgen05", "torch", "tf32"])
def test_sibling_golden_every_backend(gold, backend):
    """fused=True against the reference's own PointNet2 outputs, within the backend's stated tolerance"""
    from s4g_release_b200.engine import FusedPointNet2
    from s4g_release_b200.network_models.models.PointNet2 import PointNet2
    torch.backends.cuda.matmul.allow_tf32 = False
    net = PointNet2(**SIBLING_CFG)
    net.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in gold.items() if k.startswith("sd/")}, strict=True)
    net = net.cuda().eval()
    eng = FusedPointNet2(net, mlp_backend=backend)
    net.attach_engine(eng)
    pts = torch.from_numpy(gold["points"]).cuda()
    with torch.no_grad():
        out = net({"scene_points": pts}, fused=True)
        _, trace = eng.forward(pts, return_trace=True)
    assert net._engine is eng
    for k in SIBLING_KEYS:
        assert _rel_err(out[k], gold["out/" + k]) <= eng.tolerance(), (backend, k)
    assert tuple(trace["sa_feature"][-1].shape) == (2, 1, 256)  # the global feature


def test_class_defaults_fused_match_module_path():
    """PointNet2(score_classes=3): 10240 / 1024 / 128 / global, broadcast first propagation level"""
    from tests.inputs import tabletop_batch
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    net = _seeded(dict(score_classes=3), seed=1)
    x = tabletop_batch(2, n_points=12288).cuda()
    with torch.no_grad():
        fused = net({"scene_points": x}, fused=True)
        ref = net({"scene_points": x}, fused=False)
    tol = net.fused_engine().tolerance()
    for k in ref:
        assert _rel_err(fused[k], ref[k]) <= tol, k


@pytest.mark.parametrize("backend", ["tcgen05", "torch"])
def test_padded_global_group_matches_module_path(backend):
    from s4g_release_b200.engine import FusedPointNet2
    from tests.inputs import uniform_cloud
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    net = _seeded(PADDED_CFG, seed=2)
    eng = FusedPointNet2(net, mlp_backend=backend)
    assert net.fusable(allow_global=True)
    x = uniform_cloud(3, 1024, seed=5).cuda()
    with torch.no_grad():
        got = eng.forward(x)
        ref = net({"scene_points": x}, fused=False)
    for k in ref:
        assert _rel_err(got[k], ref[k]) <= eng.tolerance(), (backend, k)


def test_scene_in_batch_equals_scene_alone_and_overlap_is_bit_identical():
    from tests.inputs import tabletop_batch
    net = _seeded(SIBLING_CFG, seed=3, sibling=True)
    x = tabletop_batch(3, first_seed=2000, n_points=4096).cuda()
    eng = net.fused_engine()
    assert eng.global_level and eng.overlap_geometry
    with torch.no_grad():
        a = eng.forward(x)
        one = eng.forward(x[1:2].contiguous())
        eng.overlap_geometry = False
        c = eng.forward(x)
        eng.overlap_geometry = True
        torch.cuda.synchronize()
    for k in a:
        assert torch.equal(a[k][1:2], one[k]), k
        assert torch.equal(a[k], c[k]), k


def test_routing_stays_opt_in():
    from tests.inputs import uniform_cloud
    net = _seeded(SIBLING_CFG, seed=4, sibling=True)
    x = uniform_cloud(1, 1024, seed=6).cuda()
    with torch.no_grad():
        net({"scene_points": x})
    assert net._engine is None  # the automatic route keeps a global level on the module path
    bad = _seeded(dict(SIBLING_CFG, num_fp_neighbours=(3, 3, 3, 3)), seed=4, sibling=True)
    with torch.no_grad(), pytest.raises(RuntimeError, match="no plan"):
        bad({"scene_points": x}, fused=True)


def test_fused_forward_launches_no_torch_kernel():
    from torch.profiler import ProfilerActivity, profile
    from tests.inputs import uniform_cloud
    net = _seeded(SIBLING_CFG, seed=5, sibling=True)
    eng = net.fused_engine()
    x = uniform_cloud(2, 2048, seed=7).cuda()
    with torch.no_grad():
        eng.forward(x)  # first use of this shape: the cached neighbour table and zero centroids are built here
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.forward(x)
            torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert any("rows_segment_max" in n for n in names) and any("broadcast_concat" in n for n in names), names
    assert not [n for n in names if "at::" in n], names
