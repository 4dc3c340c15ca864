"""GPU suite for PN2_LOCAL on the fused engine (forward(..., fused=True), engine.FusedPointNet2Local):
  * the evaluation-row kernel (csrc/fused_ops.cu, s4g_local_eval_rows_bf16) is bit-equal to torch's cat + repeat + bf16
    cast in both modes, and its in-place update of the given frames to the module path's subtraction;
  * the golden weights are within engine.tolerance() of the reference's own outputs on every MLP backend; the class
    defaults and a configuration without a global level match the module path;
  * scenes stay independent, routing stays opt-in and follows weight updates, and a fused forward launches no torch
    kernel;
  * PN2_CLS still launches the 47 kernels per forward that DESIGN.md §1 states."""
import os

import numpy as np
import pytest
import torch

from tests.test_pn2_local import CFG as GOLDEN_CFG

pytestmark = pytest.mark.gpu

KEYS = ("local_search_logits", "frame_R", "frame_t", "movable_logits")
NO_GLOBAL_CFG = dict(GOLDEN_CFG, num_centroids=(256, 64, 16), radius=(0.1, 0.2, 0.4), num_neighbours=(16, 16, 8),
                     sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128)),
                     fp_channels=((64, 64), (32, 32), (32, 32, 16)), num_fp_neighbours=(3, 3, 3))


@pytest.fixture(autouse=True)
def ieee_fp32_module_path():
    """the module path and the torch backend as fp32 references: no TF32 convolutions or matmuls"""
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _rel_err(got, want):
    want = torch.as_tensor(want).float().cpu()
    return ((got.float().cpu() - want).abs().max() / max(1.0, want.abs().max().item())).item()


def _seeded(cfg, seed=0):
    """Default init plus non-trivial BatchNorm statistics (as test_global_level_gpu._seeded) and a non-zero t_logit."""
    from s4g_release_b200.network_models.models.PointNet2_local import PointNet2
    torch.manual_seed(seed)
    net = PointNet2(**cfg)
    g = torch.Generator().manual_seed(seed)
    for m in net.modules():
        if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
            n = m.num_features
            m.running_mean.copy_(0.1 * torch.randn(n, generator=g))
            m.running_var.copy_(0.5 + torch.rand(n, generator=g))
            m.weight.data.copy_(0.8 + 0.4 * torch.rand(n, generator=g))
            m.bias.data.copy_(0.1 * torch.randn(n, generator=g))
    net.t_logit.weight.data.copy_(0.05 * torch.randn(net.t_logit.weight.shape, generator=g))
    return net.cuda().eval()


def _frames(points, F, S, seed):
    """Candidates (B, 12, F, S): random rotation entries, translations near the point they belong to."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    B = points.shape[0]
    rot = torch.randn(B, 9, F, S, device="cuda", generator=g) * 0.5
    t = points[:, :, :F].unsqueeze(-1) + 0.02 * torch.randn(B, 3, F, S, device="cuda", generator=g)
    return torch.cat([rot, t], dim=1).contiguous()


def _want_rows(feat, B, N, cand):
    """torch's cat + repeat + bf16 cast: feat bf16 [B*N, C], cand fp32 (B, 12, F, S) -> bf16 [B*F*S, C + 48]."""
    F, S = cand.shape[2], cand.shape[3]
    per_point = feat.view(B, N, -1)[:, :F].unsqueeze(2).expand(-1, -1, S, -1)
    rep = cand.permute(0, 2, 3, 1).repeat(1, 1, 1, 4).to(torch.bfloat16)
    return torch.cat([per_point, rep], dim=-1).reshape(B * F * S, -1)


@pytest.mark.parametrize("B, N, C", [(1, 1000, 16), (5, 777, 64), (2, 300, 32)])
def test_eval_rows_self_mode_is_cat_repeat_cast(B, N, C):
    from s4g_release_b200.engine import FusedPointNet2Local
    g = torch.Generator(device="cuda").manual_seed(B * 1000 + N)
    feat = torch.randn(B * N, C, device="cuda", generator=g).to(torch.bfloat16)
    xyz = torch.rand(B, 3, N, device="cuda", generator=g)
    R = torch.randn(B, 9, N, device="cuda", generator=g)
    t = torch.randn(B, 3, N, device="cuda", generator=g)
    got = FusedPointNet2Local.local_eval_rows(feat, xyz, None, R, t)
    assert torch.equal(got, _want_rows(feat, B, N, torch.cat([R, t], 1).unsqueeze(-1)))


@pytest.mark.parametrize("B, N, C, F, S", [(1, 100, 16, 100, 1), (5, 300, 64, 37, 6), (2, 257, 32, 200, 64),
                                           (3, 50, 64, 1, 300), (1, 4096, 16, 4096, 3)])
def test_eval_rows_given_mode_is_cat_repeat_cast_and_updates_frames_in_place(B, N, C, F, S):
    from s4g_release_b200.engine import FusedPointNet2Local
    g = torch.Generator(device="cuda").manual_seed(B * 1000 + F * 10 + S)
    feat = torch.randn(B * N, C, device="cuda", generator=g).to(torch.bfloat16)
    xyz = torch.rand(B, 3, N, device="cuda", generator=g)
    frames = torch.randn(B, 12, F, S, device="cuda", generator=g)
    ref = frames.clone()
    ref[:, 9:, :, :] = ref[:, 9:, :, :] - xyz[:, :, :F].unsqueeze(-1).expand(-1, -1, -1, S)  # the module path's update
    got = FusedPointNet2Local.local_eval_rows(feat, xyz, frames)
    assert torch.equal(frames, ref)
    assert torch.equal(got, _want_rows(feat, B, N, ref))


def test_eval_rows_beyond_2_gib():
    """2 x 4096 x 1200 candidates of 112 channels: 2.2 GB of rows, checked on a seeded sample of rows"""
    from s4g_release_b200.engine import FusedPointNet2Local
    B, N, C, F, S = 2, 4096, 64, 4096, 1200
    g = torch.Generator(device="cuda").manual_seed(7)
    feat = torch.randn(B * N, C, device="cuda", generator=g).to(torch.bfloat16)
    xyz = torch.rand(B, 3, N, device="cuda", generator=g)
    frames = torch.randn(B, 12, F, S, device="cuda", generator=g)
    ref = frames.clone()
    ref[:, 9:, :, :] = ref[:, 9:, :, :] - xyz[:, :, :F].unsqueeze(-1).expand(-1, -1, -1, S)
    got = FusedPointNet2Local.local_eval_rows(feat, xyz, frames)
    assert got.numel() * got.element_size() > 2 ** 31
    assert torch.equal(frames, ref)
    rows = torch.randint(0, B * F * S, (8192,), device="cuda", generator=g)
    rows = torch.cat([rows, torch.tensor([0, B * F * S - 1], device="cuda")])
    b, f, s = rows // (F * S), rows % (F * S) // S, rows % S
    cand = ref[b, :, f, s].to(torch.bfloat16).repeat(1, 4)  # (rows, 48)
    want = torch.cat([feat[b * N + f], cand], dim=1)
    assert torch.equal(got[rows], want)


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(os.path.join(os.path.dirname(__file__), "golden", "pn2_local.npz")))


@pytest.mark.parametrize("backend", ["tcgen05", "torch", "tf32"])
def test_golden_every_backend(gold, backend):
    """fused=True against the reference's own PointNet2_local outputs, self and given mode, within the backend's stated
    tolerance; the given frames are updated in place exactly as the module path updates them"""
    from s4g_release_b200.engine import FusedPointNet2Local
    from s4g_release_b200.network_models.models.PointNet2_local import PointNet2
    from tests.test_pn2_local import _reference_weights
    net = PointNet2(**GOLDEN_CFG)
    net.load_state_dict(_reference_weights(gold), strict=True)
    net = net.cuda().eval()
    eng = FusedPointNet2Local(net, mlp_backend=backend)
    net.attach_engine(eng)
    pts = torch.from_numpy(gold["points"]).cuda()
    frames = torch.from_numpy(gold["frames"]).cuda()
    frames_module = frames.clone()
    with torch.no_grad():
        out_self = net({"scene_points": pts}, fused=True)
        out_given = net({"scene_points": pts, "local_search_frame": frames}, fused=True)
        net({"scene_points": pts, "local_search_frame": frames_module}, fused=False)
    assert net._engine is eng
    assert torch.equal(frames, frames_module)
    for tag, out in (("self/", out_self), ("given/", out_given)):
        for k in KEYS:
            want = gold[tag + k]
            assert tuple(out[k].shape) == want.shape, (backend, tag, k)
            assert _rel_err(out[k], want) <= eng.tolerance(), (backend, tag, k)


def _match_module_path(net, x, frames, tol):
    f_fused, f_module = frames.clone(), frames.clone()
    with torch.no_grad():
        for batch_fused, batch_module in (({"scene_points": x}, {"scene_points": x}),
                                          ({"scene_points": x, "local_search_frame": f_fused},
                                           {"scene_points": x, "local_search_frame": f_module})):
            fused = net(batch_fused, fused=True)
            ref = net(batch_module, fused=False)
            for k in KEYS:
                assert fused[k].shape == ref[k].shape, k
                assert _rel_err(fused[k], ref[k]) <= tol, (k, "local_search_frame" in batch_fused)
    assert torch.equal(f_fused, f_module)


def test_class_defaults_fused_match_module_path():
    """PointNet2(score_classes=3): 10240 / 1024 / 128 / global, broadcast first propagation level, 64-channel features"""
    from tests.inputs import tabletop_batch
    net = _seeded(dict(score_classes=3), seed=1)
    x = tabletop_batch(2, n_points=12288).cuda()
    _match_module_path(net, x, _frames(x, 512, 8, seed=1), net.fused_engine().tolerance())


def test_without_global_level_fused_matches_module_path():
    from tests.inputs import uniform_cloud
    net = _seeded(NO_GLOBAL_CFG, seed=2)
    assert net.fusable()
    x = uniform_cloud(2, 1024, seed=5).cuda()
    _match_module_path(net, x, _frames(x, 100, 5, seed=2), net.fused_engine().tolerance())
    assert not net.fused_engine().global_level


def test_scene_in_batch_equals_scene_alone():
    from tests.inputs import tabletop_batch
    net = _seeded(GOLDEN_CFG, seed=3)
    x = tabletop_batch(3, first_seed=2000, n_points=4096).cuda()
    frames = _frames(x, 300, 7, seed=3)
    eng = net.fused_engine()
    with torch.no_grad():
        a = eng.forward(x)
        one = eng.forward(x[1:2].contiguous())
        fa, f1 = frames.clone(), frames[1:2].clone()
        ga = eng.forward(x, fa)
        g1 = eng.forward(x[1:2].contiguous(), f1)
    for k in KEYS:
        assert torch.equal(a[k][1:2], one[k]), k
        assert torch.equal(ga[k][1:2], g1[k]), k
    assert torch.equal(fa[1:2], f1)


def test_routing_stays_opt_in_and_follows_new_weights():
    from tests.inputs import uniform_cloud
    net = _seeded(GOLDEN_CFG, seed=4)
    x = uniform_cloud(2, 1024, seed=6).cuda()
    frames = _frames(x, 64, 4, seed=4)
    with torch.no_grad():
        net({"scene_points": x})
        net({"scene_points": x, "local_search_frame": frames.clone()}, fused=False)
    assert net._engine is None  # fused=None and fused=False keep the module path
    tol = net.fused_engine().tolerance()
    with torch.no_grad():
        before = net({"scene_points": x}, fused=True)["local_search_logits"]
    other = _seeded(GOLDEN_CFG, seed=5)
    net.load_state_dict(other.state_dict())
    _match_module_path(net, x, frames, tol)
    opt = torch.optim.SGD(net.parameters(), lr=0.5)
    for p in net.parameters():
        p.grad = torch.full_like(p, 0.01)
    opt.step()  # in place, under no_grad: only the parameters' version counters tell
    _match_module_path(net, x, frames, tol)
    with torch.no_grad():
        after = net({"scene_points": x}, fused=True)["local_search_logits"]
    assert not torch.equal(before, after)
    for bad, match in ((frames.cpu(), "float32 tensor on cuda"), (frames.double(), "float32"),
                       (_frames(x, 64, 4, seed=4)[:, :, :, :2].transpose(2, 3), "strided"),
                       (torch.zeros(2, 12, 1025, 1, device="cuda"), "n_frames <= 1024")):
        with torch.no_grad(), pytest.raises(ValueError, match=match):
            net({"scene_points": x, "local_search_frame": bad}, fused=True)


@pytest.mark.parametrize("given", [False, True])
def test_fused_forward_launches_no_torch_kernel(given):
    from torch.profiler import ProfilerActivity, profile
    from tests.inputs import uniform_cloud
    net = _seeded(GOLDEN_CFG, seed=6)
    eng = net.fused_engine()
    x = uniform_cloud(2, 2048, seed=7).cuda()
    frames = _frames(x, 256, 16, seed=6) if given else None
    with torch.no_grad():
        eng.forward(x, frames)  # first use of this shape: the global level's tables and the chain plans are made here
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.forward(x, frames)
            torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert any("local_eval_rows" in n for n in names), names
    assert not [n for n in names if "at::" in n], names


def test_pn2_cls_launches_47_kernels_per_forward():
    """DESIGN.md §1: one fused forward of the shipped PN2_CLS configuration launches 47 of the library's kernels"""
    from s4g_release_b200 import _lib
    from s4g_release_b200.engine import FusedPointNet2
    from s4g_release_b200.network_models.models.PointNet2_tcls import NUM_INPUT, PN2_CLS_CONFIG, PointNet2
    from tests.inputs import tabletop_batch
    torch.manual_seed(0)
    net = PointNet2(**PN2_CLS_CONFIG).cuda().eval()
    eng = FusedPointNet2(net)
    x = tabletop_batch(2, n_points=NUM_INPUT).cuda()
    with torch.no_grad():
        eng.forward(x)  # plans made, shapes seen
        torch.cuda.synchronize()
        n0 = _lib.lib.s4g_launch_count()
        eng.forward(x)
        torch.cuda.synchronize()
    assert _lib.lib.s4g_launch_count() - n0 == 47
