"""GPU suite for EDGEPN2DU on the fused engine (forward(..., fused=True), engine.FusedEdgePointNet2DownUp):
  * the edge-row kernel (s4g_edge_interp_rows_bf16) against torch on the same bf16 operands, within one bf16 ulp, with
    both skip kinds (bf16 T rows, the fp32 cloud), with an output over 2 GiB, and on clouds with NaN points;
  * the 3-row mean (s4g_rows_group_mean_bf16) bit-identical to the same expression in torch;
  * the fused edge propagation stage against the reference's own EdgeFPModule (tests/golden/pn2_local.npz, efp/*);
  * the whole model on every MLP backend against the module path, a cancelling split against the torch backend;
  * scenes stay independent, the overlap of the 3-NN searches changes no bit, and a fused forward launches no torch kernel
    and a pinned number of the library's."""
import os

import numpy as np
import pytest
import torch

from tests.test_edge_models import CFG as GOLDEN_CFG

pytestmark = pytest.mark.gpu

KEYS = ("scene_score_logits", "frame_R")


@pytest.fixture(autouse=True)
def ieee_fp32_references():
    """the module path and the torch backend as fp32 references: no TF32 convolutions or matmuls"""
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _rel_err(got, want):
    want = torch.as_tensor(want).float().cpu()
    return ((got.float().cpu() - want).abs().max() / max(1.0, want.abs().max().item())).item()


def _seeded(cfg, seed=0, cls="downup"):
    """Default init plus non-trivial BatchNorm statistics (as test_edge_fused_gpu._seeded)."""
    from s4g_release_b200.network_models.models.EdgePointNet2Down import EdgePointNet2Down
    from s4g_release_b200.network_models.models.EdgePointNet2DownUp import EdgePointNet2DownUp
    torch.manual_seed(seed)
    net = (EdgePointNet2DownUp if cls == "downup" else EdgePointNet2Down)(**cfg)
    g = torch.Generator().manual_seed(seed)
    for m in net.modules():
        if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
            n = m.num_features
            m.running_mean.copy_(0.1 * torch.randn(n, generator=g))
            m.running_var.copy_(0.5 + torch.rand(n, generator=g))
            m.weight.data.copy_(0.8 + 0.4 * torch.rand(n, generator=g))
            m.bias.data.copy_(0.1 * torch.randn(n, generator=g))
    return net.cuda().eval()


# ---------------------------------------------------------------------------------------------------- the edge rows
def _edge_problem(B, Nk, Nq, C, xyz_skip, seed, cloud=None):
    """[U | V] rows, 3-NN of the fused path, T rows or the cloud with W_d, shift"""
    from s4g_release_b200.engine import FusedPointNet2
    g = torch.Generator(device="cuda").manual_seed(seed)
    dense = torch.rand(B, 3, Nq, device="cuda", generator=g) if cloud is None else cloud[0]
    sparse = torch.rand(B, 3, Nk, device="cuda", generator=g) if cloud is None else cloud[1]
    idx, w = FusedPointNet2.three_nn_weights(dense, sparse)
    uv = torch.randn(B * Nk, 2 * C, device="cuda", generator=g).to(torch.bfloat16)
    shift = 0.1 * torch.randn(C, device="cuda", generator=g)
    if xyz_skip:
        return uv, idx, w, None, dense, torch.randn(C, 3, device="cuda", generator=g), shift
    return uv, idx, w, torch.randn(B * Nq, C, device="cuda", generator=g).to(torch.bfloat16), None, None, shift


def _torch_edge_rows(uv, idx, w, t_rows, xyz, w_xyz, shift, B, Nk):
    """fp32 torch on the kernel's operands, the kernel's order of the sums -> (B, Q, 3, C); the ReLU maps NaN to 0 as
    the kernel's fmaxf does.  idx / w / t_rows / xyz may cover a subset of Q queries."""
    C = shift.numel()
    Q = idx.shape[1]
    il = idx.long().reshape(B, Q * 3, 1)
    g = torch.gather(uv.float().reshape(B, Nk, 2 * C), 1, il.expand(-1, -1, 2 * C)).reshape(B, Q, 3, 2 * C)
    U, V = g[..., :C], g[..., C:]
    base = U[:, :, 0] * w[:, :, 0:1]
    base = torch.addcmul(base, U[:, :, 1], w[:, :, 1:2])
    base = torch.addcmul(base, U[:, :, 2], w[:, :, 2:3])
    T = t_rows.float().reshape(B, Q, C) if t_rows is not None else xyz.transpose(1, 2) @ w_xyz.t()
    y = ((base.unsqueeze(2) + V) + T.unsqueeze(2)) + shift
    return torch.where(y > 0, y, torch.zeros_like(y))


def _bf16_ulp(y):
    """the spacing of bf16 numbers at |y| (8 significant bits)"""
    _, e = torch.frexp(y.abs())
    return torch.ldexp(torch.ones_like(y), e - 8)


def _assert_within_one_ulp(got, want, scale):
    """got bf16 vs the fp32 value: one bf16 ulp, plus an absolute floor for fp32 sums that differ in order near 0"""
    err = (got.float() - want).abs()
    tol = torch.maximum(_bf16_ulp(want), torch.full_like(want, 1e-6 * scale))
    bad = err > tol
    assert not bad.any(), "%d elements beyond one ulp, worst %.3e at %.3e" % (
        bad.sum().item(), err[bad].max().item(), want[bad][err[bad].argmax()].item())


@pytest.mark.parametrize("xyz_skip", [False, True], ids=["t_rows", "cloud"])
@pytest.mark.parametrize("B, Nk, Nq, C", [(1, 3, 5, 8), (2, 128, 1024, 64), (3, 1024, 10240, 128), (2, 2000, 3001, 256),
                                          (1, 64, 700, 512), (2, 300, 999, 24)])
def test_edge_rows_match_torch(B, Nk, Nq, C, xyz_skip):
    from s4g_release_b200.engine import FusedEdgePointNet2DownUp
    uv, idx, w, t_rows, xyz, w_xyz, shift = _edge_problem(B, Nk, Nq, C, xyz_skip, seed=Nq + C)
    got = FusedEdgePointNet2DownUp.edge_interp_rows(uv, idx, w, t_rows, xyz, w_xyz, shift, B, Nk, Nq)
    want = _torch_edge_rows(uv, idx, w, t_rows, xyz, w_xyz, shift, B, Nk)
    torch.cuda.synchronize()
    assert tuple(got.shape) == (B * Nq * 3, C)
    assert (want > 0).float().mean() > 0.2
    _assert_within_one_ulp(got.reshape(want.shape), want, uv.float().abs().max().item())


def test_edge_rows_beyond_2_gib():
    """a 2.5 GB output: the second scene's last rows sit past 2 GiB; they and the first scene's first rows are checked"""
    from s4g_release_b200.engine import FusedEdgePointNet2DownUp
    B, Nk, Nq, C = 2, 4096, 820_000, 256
    uv, idx, w, t_rows, xyz, w_xyz, shift = _edge_problem(B, Nk, Nq, C, False, seed=21)
    got = FusedEdgePointNet2DownUp.edge_interp_rows(uv, idx, w, t_rows, xyz, w_xyz, shift, B, Nk, Nq)
    assert got.numel() * got.element_size() > 2 ** 31 + 2 ** 28
    got = got.reshape(B, Nq, 3, C)
    t = t_rows.reshape(B, Nq, C)
    for sel in (slice(0, 3000), slice(Nq - 3000, Nq)):
        want = _torch_edge_rows(uv, idx[:, sel], w[:, sel], t[:, sel].reshape(-1, C), None, None, shift, B, Nk)
        _assert_within_one_ulp(got[:, sel], want, uv.float().abs().max().item())


@pytest.mark.parametrize("xyz_skip", [False, True], ids=["t_rows", "cloud"])
@pytest.mark.parametrize("Nk", [300, 2048])  # the linear 3-NN kernel and the grid one (>= 1024 keys)
def test_edge_rows_on_clouds_with_nan_points(Nk, xyz_skip):
    """NaN queries and NaN keys: the fused 3-NN writes valid rows only (index 0 where the reference has -1), so the
    kernel reads nothing out of bounds and its rows are those of torch on the same indices"""
    from s4g_release_b200.engine import FusedEdgePointNet2DownUp
    B, Nq, C = 2, 5000, 64
    g = torch.Generator(device="cuda").manual_seed(Nk)
    dense = torch.rand(B, 3, Nq, device="cuda", generator=g)
    sparse = torch.rand(B, 3, Nk, device="cuda", generator=g)
    dense[0, :, :100] = float("nan")
    dense[1, 1, 7] = float("nan")
    sparse[1, :, : Nk - 2] = float("nan")  # scene 1: two finite keys only
    sparse[0, 0, 5] = float("nan")
    uv, idx, w, t_rows, xyz, w_xyz, shift = _edge_problem(B, Nk, Nq, C, xyz_skip, seed=Nk + 1, cloud=(dense, sparse))
    assert idx.min().item() >= 0 and idx.max().item() < Nk and torch.isfinite(w).all()
    got = FusedEdgePointNet2DownUp.edge_interp_rows(uv, idx, w, t_rows, xyz, w_xyz, shift, B, Nk, Nq)
    want = _torch_edge_rows(uv, idx, w, t_rows, xyz, w_xyz, shift, B, Nk)
    torch.cuda.synchronize()
    assert torch.isfinite(got.float()).all()
    _assert_within_one_ulp(got.reshape(want.shape), want, uv.float().abs().max().item())


@pytest.mark.parametrize("R, C", [(1, 8), (1000, 64), (65_537, 128), (3001, 512), (7, 1024)])
def test_rows_group_mean_is_the_torch_expression(R, C):
    from s4g_release_b200.engine import FusedEdgePointNet2DownUp
    g = torch.Generator(device="cuda").manual_seed(R + C)
    rows = (3 * torch.randn(3 * R, C, device="cuda", generator=g)).to(torch.bfloat16)
    got = FusedEdgePointNet2DownUp.rows_group_mean(rows)
    x = rows.float().reshape(R, 3, C)
    s = (x[:, 0] + x[:, 1]) + x[:, 2]
    want = (s / torch.full_like(s, 3.0)).to(torch.bfloat16)  # a tensor divisor: IEEE division, no reciprocal
    torch.cuda.synchronize()
    assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------------- the reference's EdgeFPModule
def test_edge_stage_matches_the_reference_edge_fp_module():
    """efp/feature of tests/golden/pn2_local.npz: the reference's own EdgeFPModule(2 x 48 + 24, (64, 32), 3) on 1 024
    dense points with a 24-channel skip and 128 sparse points.  The engine's edge propagation stage (its chains built by
    the same hook as in a model) is run on those inputs: tcgen05 (bf16 operands) and the torch backend's literal rows."""
    from s4g_release_b200.engine import FusedEdgePointNet2DownUp, _fold_mlp
    from s4g_release_b200.network_models.models.pointnet2_utils.modules import EdgeFPModule
    gold = dict(np.load(os.path.join(os.path.dirname(__file__), "golden", "pn2_local.npz")))
    efp = EdgeFPModule(2 * 48 + 24, (64, 32), 3)
    efp.load_state_dict({k[7:]: torch.from_numpy(v) for k, v in gold.items() if k.startswith("efp_sd/")}, strict=True)
    efp = efp.cuda().eval()
    layers = _fold_mlp(efp.mlp)
    dense_xyz = torch.from_numpy(gold["points"]).cuda()
    sparse_xyz = torch.from_numpy(gold["esa/xyz"]).cuda()
    dense = torch.from_numpy(gold["feat"]).cuda().transpose(1, 2).contiguous()  # (B, 1024, 24)
    sparse = torch.from_numpy(gold["esa/feature"]).cuda().transpose(1, 2).contiguous()  # (B, 128, 48)
    want = gold["efp/feature"].transpose(0, 2, 1)  # (B, 1024, 32)
    B, Nq, Nk = dense.shape[0], dense.shape[1], sparse.shape[1]
    net = _seeded(GOLDEN_CFG, seed=2)
    errs = {}
    for backend in ("tcgen05", "torch"):
        eng = FusedEdgePointNet2DownUp(net, mlp_backend=backend)
        i = len(eng.edge_fp)  # one more propagation level, registered as the model's are
        eng.edge_fp.append(True)
        with torch.no_grad():
            if backend == "torch":
                got = eng._fp_reference(i, dense_xyz, sparse_xyz, dense, sparse, layers)
            else:
                # row chains read multiples of 16 channels: the 24-channel skip and W_d get 8 zero channels (exact)
                (w0, b0), rest = layers[0], layers[1:]
                padded = [(torch.cat([w0, w0.new_zeros(w0.shape[0], 8)], dim=1), b0)] + rest
                eng.fp_chains.append(eng._fp_chain(i, padded, 32)[1])
                skip = torch.cat([dense, dense.new_zeros(B, Nq, 8)], dim=-1).reshape(B * Nq, 32)
                idx, w = eng.three_nn_weights(dense_xyz, sparse_xyz)
                got = eng._fp_level(i, sparse.reshape(B * Nk, 48).to(torch.bfloat16), skip.to(torch.bfloat16), dense_xyz,
                                    idx, w, Nk, None)
            torch.cuda.synchronize()
        errs[backend] = _rel_err(got.reshape(B, Nq, 32), want)
    print("EdgeFPModule golden: %s" % errs)
    assert errs["torch"] <= 1e-4, errs
    assert errs["tcgen05"] <= 2e-2, errs


# ---------------------------------------------------------------------------------------------------- the model
@pytest.mark.parametrize("backend", ["tcgen05", "torch", "tf32"])
@pytest.mark.parametrize("which", ["golden_cfg", "class_defaults"])
def test_model_on_every_backend_matches_the_module_path(which, backend):
    from s4g_release_b200.engine import FusedEdgePointNet2DownUp
    from tests.inputs import tabletop_batch
    cfg, n = (GOLDEN_CFG, 4096) if which == "golden_cfg" else (dict(score_classes=3), 12288)
    net = _seeded(cfg, seed=1)
    x = tabletop_batch(2, n_points=n).cuda()
    eng = FusedEdgePointNet2DownUp(net, mlp_backend=backend)
    assert eng.edge_fp == [False, True, True, True] and eng.edge_levels == [False, True, True, False]
    net.attach_engine(eng)
    with torch.no_grad():
        fused = net({"scene_points": x}, fused=True)
        ref = net({"scene_points": x}, fused=False)
    assert net._engine is eng
    errs = {k: _rel_err(fused[k], ref[k]) for k in KEYS}
    print("%s %s vs module path: %s" % (which, backend, errs))
    for k in KEYS:
        assert tuple(fused[k].shape) == tuple(ref[k].shape), k
        assert errs[k] <= eng.tolerance(), (k, errs[k])


@pytest.mark.parametrize("mode", ["wi_is_wn", "wi_is_zero"])
def test_cancelling_split_against_the_torch_backend(mode):
    """Every edge propagation level of the class defaults with a large W_n (x 4) and W_i = W_n + eps (U is tiny) or
    W_i = eps (the layer is W_n (n_k - interp): U and V cancel where n_k ~ interp).  The split's roundings (U, V, T in
    bf16) against the torch backend's literal edge rows in fp32; the error is printed."""
    from s4g_release_b200.engine import FusedEdgePointNet2DownUp
    from tests.inputs import tabletop_batch
    net = _seeded(dict(score_classes=3), seed=6)
    g = torch.Generator().manual_seed(6)
    with torch.no_grad():
        for i in (1, 2, 3):
            w = net.fp_modules[i].mlp[0].conv.weight  # (cout, 2 C2 + C1, 1, 1)
            c2 = net.fp_modules[i - 1].out_channels  # the sparse feature: the previous level's output
            wn = 4.0 * w[:, c2:2 * c2].clone()
            eps = 1e-3 * torch.randn(w.shape[0], c2, 1, 1, generator=g).cuda()
            w[:, c2:2 * c2] = wn
            w[:, :c2] = (wn + eps) if mode == "wi_is_wn" else eps
    x = tabletop_batch(2, n_points=12288).cuda()
    eng = FusedEdgePointNet2DownUp(net)
    with torch.no_grad():
        got = eng.forward(x)
        ref = FusedEdgePointNet2DownUp(net, mlp_backend="torch").forward(x)
    errs = {k: _rel_err(got[k], ref[k]) for k in got}
    print("cancelling split (%s): tcgen05 vs torch backend %s" % (mode, errs))
    for k in got:
        assert errs[k] <= eng.tolerance(), (k, errs[k])


def test_scene_in_batch_equals_scene_alone_and_overlap_is_bit_identical():
    from tests.inputs import tabletop_batch
    net = _seeded(GOLDEN_CFG, seed=3)
    x = tabletop_batch(3, first_seed=2000, n_points=4096).cuda()
    eng = net.fused_engine()
    assert eng.overlap_geometry
    with torch.no_grad():
        a = eng.forward(x)
        one = eng.forward(x[1:2].contiguous())
        eng.overlap_geometry = False
        c = eng.forward(x)
        eng.overlap_geometry = True
        torch.cuda.synchronize()
    for k in KEYS:
        assert torch.equal(a[k][1:2], one[k]), k
        assert torch.equal(a[k], c[k]), k


def test_fused_forward_launches_no_torch_kernel_and_a_pinned_count():
    """Against EDGEPN2D with the same encoder: its plain propagation levels launch 2, 2 and 3 kernels (interpolation +
    chain; at the finest, the first layer on the sparse rows too), an edge propagation level launches its [U | V] chain,
    its T chain (not at the finest level: the cloud enters the row kernel), the row kernel, one chain per later layer
    group and the mean — 5, 5 and 4 here — and there are 2 heads instead of 4: 5 launches more in all."""
    from torch.profiler import ProfilerActivity, profile
    from s4g_release_b200 import _lib
    from tests.inputs import uniform_cloud
    x = uniform_cloud(2, 2048, seed=7).cuda()
    counts = {}
    for cls in ("downup", "down"):
        eng = _seeded(GOLDEN_CFG, seed=5, cls=cls).fused_engine()
        with torch.no_grad():
            eng.forward(x)  # first use of this shape: plans made, the global level's tables built
            torch.cuda.synchronize()
            n0 = _lib.lib.s4g_launch_count()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                eng.forward(x)
                torch.cuda.synchronize()
            counts[cls] = _lib.lib.s4g_launch_count() - n0
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        assert not [n for n in names if "at::" in n], names
        if cls == "downup":
            assert sum("edge_interp_rows" in n for n in names) == 3, names
            assert sum("rows_group_mean" in n for n in names) == 3, names
            assert not [n for n in names if "interp_concat" in n], names
    assert counts["downup"] == counts["down"] + (5 - 2) + (5 - 2) + (4 - 3) - 2, counts
