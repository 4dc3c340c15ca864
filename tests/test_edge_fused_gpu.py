"""GPU suite for EDGEPN2D on the fused engine (forward(..., fused=True), engine.FusedEdgePointNet2Down):
  * the centroid-row kernel (csrc/fused_ops.cu, s4g_gather_rows_bf16) is bit-equal to index_select, also over 2 GiB;
  * the edge chain (in_mode IN_GATHER_EDGE: the gathered max-pool chain whose layer-0 epilogue adds a per-centroid term)
    matches torch on the same bf16 operands, equals the plain chain bit for bit with an all-zero term, and gives the same
    bits under every plan the tuner may pin;
  * the reference's own EDGEPN2D outputs are met within engine.tolerance() on every MLP backend, and the class defaults
    match the module path;
  * scenes stay independent, a fused forward launches no torch kernel and exactly two launches more per edge level than
    the PN2 sibling of the same shape, and a cancelling split (W_a = -W_b + eps, W_a = eps) stays within tolerance."""
import os

import numpy as np
import pytest
import torch

from tests.test_edge_models import CFG as GOLDEN_CFG

pytestmark = pytest.mark.gpu

KEYS = ("scene_score_logits", "frame_R", "frame_t", "movable_logits")


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


def _seeded(cfg, seed=0, cls="edge"):
    """Default init plus non-trivial BatchNorm statistics (as test_global_level_gpu._seeded)."""
    from s4g_release_b200.network_models.models.EdgePointNet2Down import EdgePointNet2Down
    from s4g_release_b200.network_models.models.PointNet2 import PointNet2
    torch.manual_seed(seed)
    net = (EdgePointNet2Down if cls == "edge" else PointNet2)(**cfg)
    g = torch.Generator().manual_seed(seed)
    for m in net.modules():
        if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
            n = m.num_features
            m.running_mean.copy_(0.1 * torch.randn(n, generator=g))
            m.running_var.copy_(0.5 + torch.rand(n, generator=g))
            m.weight.data.copy_(0.8 + 0.4 * torch.rand(n, generator=g))
            m.bias.data.copy_(0.1 * torch.randn(n, generator=g))
    return net.cuda().eval()


# ---------------------------------------------------------------------------------------------------- centroid rows
@pytest.mark.parametrize("B, N, M, C", [(1, 1, 1, 8), (2, 300, 77, 32), (3, 5120, 1024, 64), (64, 1024, 128, 128),
                                        (2, 100, 100, 264)])
def test_gather_rows_is_index_select(B, N, M, C):
    from s4g_release_b200.engine import FusedEdgePointNet2Down
    g = torch.Generator(device="cuda").manual_seed(B * 1000 + M)
    rows = torch.randn(B * N, C, device="cuda", generator=g).to(torch.bfloat16)
    idx = torch.stack([torch.randperm(N, device="cuda", generator=g)[:M] for _ in range(B)]).to(torch.int32)
    got = FusedEdgePointNet2Down.gather_rows(rows, idx)
    flat = (idx.long() + torch.arange(B, device="cuda").view(B, 1) * N).reshape(-1)
    assert torch.equal(got, rows.index_select(0, flat))


def test_gather_rows_beyond_2_gib():
    """a 2.4 GB source table: the last rows sit past 2 GiB of 16-byte pieces' byte offset"""
    from s4g_release_b200.engine import FusedEdgePointNet2Down
    B, N, M, C = 2, 600_000, 4096, 1024
    g = torch.Generator(device="cuda").manual_seed(11)
    rows = torch.randn(B * N, C, device="cuda", generator=g).to(torch.bfloat16)
    assert rows.numel() * rows.element_size() > 2 ** 31
    idx = torch.randint(0, N, (B, M), device="cuda", generator=g, dtype=torch.int32)
    idx[:, -1] = N - 1
    got = FusedEdgePointNet2Down.gather_rows(rows, idx)
    flat = (idx.long() + torch.arange(B, device="cuda").view(B, 1) * N).reshape(-1)
    assert torch.equal(got, rows.index_select(0, flat))


# ---------------------------------------------------------------------------------------------------- the edge chain
def _bf(x):
    return x.to(torch.bfloat16).float()


def _layers(dims, seed, scale=2.0):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(dims[i + 1], dims[i], generator=g) * (scale / np.sqrt(dims[i])),
             torch.randn(dims[i + 1], generator=g) * 0.1, True) for i in range(len(dims) - 1)]


def _problem(feat_c, dims, B, N, M, K, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    xyz = torch.rand(B, 3, N, device="cuda", generator=g)
    ctr = xyz[:, :, :M].contiguous()
    nbr = torch.randint(0, N, (B, M, K), device="cuda", generator=g, dtype=torch.int32)
    feat = torch.randn(B * N, feat_c, device="cuda", generator=g).to(torch.bfloat16)
    term = (0.5 * torch.randn(B * M, dims[0], device="cuda", generator=g)).to(torch.bfloat16)
    return xyz, ctr, nbr, feat, term


def _torch_edge_chain(layers, xyz, ctr, nbr, feat, term):
    """torch fp32 on the chain's bf16 operands: rows [rel xyz | f_j] (the reference's order), layer 0 + term before the
    ReLU, hidden activations rounded to bf16, max over each centroid's K rows"""
    B, M, K = nbr.shape
    C = feat.shape[1]
    idx = nbr.long().reshape(B, M * K)
    gx = torch.gather(xyz.transpose(1, 2), 1, idx.unsqueeze(-1).expand(-1, -1, 3)).reshape(B, M, K, 3)
    rel = _bf(gx - ctr.transpose(1, 2).unsqueeze(2))
    gf = torch.gather(feat.float().reshape(B, -1, C), 1, idx.unsqueeze(-1).expand(-1, -1, C)).reshape(B, M, K, C)
    x = torch.cat([rel, gf], dim=-1).reshape(B * M * K, C + 3)
    for i, (w, b, relu) in enumerate(layers):
        w = _bf(w.cuda())
        x = x @ w.t() + b.cuda()
        if i == 0:
            x = x + term.float().repeat_interleave(K, dim=0)
        x = torch.relu(x) if relu else x
        if i + 1 < len(layers):
            x = _bf(x)
    return _bf(x.reshape(B * M, K, -1).max(dim=1)[0])


@pytest.mark.parametrize("tma", [0, 1])
@pytest.mark.parametrize("feat_c, dims, B, N, M, K", [
    (64, [64, 64, 128], 2, 1024, 65, 8), (64, [32, 32, 64], 3, 700, 100, 16), (128, [128, 128, 256], 2, 2048, 300, 32),
    (128, [64, 64, 128], 2, 4096, 500, 64), (192, [96, 128], 1, 512, 33, 16),
    (64, [48, 64], 2, 1000, 100, 8),  # a 48-wide first layer: the narrow epilogue path
    (64, [64, 64, 128], 2, 8192, 6000, 64),  # 768 000 rows: >= 40 tiles per CTA on 148 SMs
])
def test_edge_chain_matches_torch(feat_c, dims, B, N, M, K, tma):
    from s4g_release_b200.chain import IN_GATHER_EDGE, OUT_MAXPOOL, MlpChain
    layers = _layers([feat_c + 3] + dims, seed=feat_c + M)
    xyz, ctr, nbr, feat, term = _problem(feat_c, dims, B, N, M, K, seed=M + K)
    ch = MlpChain(layers, "cuda", IN_GATHER_EDGE, feat_c, OUT_MAXPOOL, group=K, tma_in=tma)
    got = ch.run_gather(feat, xyz, ctr, nbr, term)
    want = _torch_edge_chain(layers, xyz, ctr, nbr, feat, term)
    torch.cuda.synchronize()
    assert tuple(got.shape) == (B * M, dims[-1])
    err = (got.float() - want).abs().max().item()
    assert err <= 2e-2 * max(want.abs().max().item(), 1e-3), (err, want.abs().max().item())
    if B * M * K >= 148 * 40 * 128:  # the term actually matters: dropping it changes the result
        assert not torch.equal(got, MlpChain(layers, "cuda", IN_GATHER_EDGE, feat_c, OUT_MAXPOOL, group=K, tma_in=tma)
                               .run_gather(feat, xyz, ctr, nbr, torch.zeros_like(term)))


@pytest.mark.parametrize("tma", [0, 1])
@pytest.mark.parametrize("feat_c, dims, K", [(64, [64, 64, 128], 16), (128, [128, 128, 256], 64), (64, [48, 64], 8)])
def test_zero_term_is_the_plain_chain_bit_for_bit(feat_c, dims, K, tma):
    from s4g_release_b200.chain import IN_GATHER, IN_GATHER_EDGE, OUT_MAXPOOL, MlpChain
    layers = _layers([feat_c + 3] + dims, seed=K)
    xyz, ctr, nbr, feat, term = _problem(feat_c, dims, 2, 3000, 777, K, seed=K)
    edge = MlpChain(layers, "cuda", IN_GATHER_EDGE, feat_c, OUT_MAXPOOL, group=K, tma_in=tma)
    plain = MlpChain(layers, "cuda", IN_GATHER, feat_c, OUT_MAXPOOL, group=K, tma_in=tma)
    got = edge.run_gather(feat, xyz, ctr, nbr, torch.zeros_like(term))
    want = plain.run_gather(feat, xyz, ctr, nbr)
    torch.cuda.synchronize()
    assert got.float().abs().max() > 0 and torch.equal(got, want)


def test_every_tunable_plan_of_an_edge_chain_is_bit_identical():
    from s4g_release_b200.chain import IN_GATHER_EDGE, OUT_MAXPOOL, MlpChain
    from s4g_release_b200.engine import candidate_plans
    feat_c, dims, K = 128, [128, 128, 256], 64
    layers = _layers([feat_c + 3] + dims, seed=4)
    xyz, ctr, nbr, feat, term = _problem(feat_c, dims, 2, 4096, 300, K, seed=5)
    want, seen = None, set()
    for slots, pairs, coop, subs, tma in candidate_plans(IN_GATHER_EDGE, feat_c, OUT_MAXPOOL):
        try:
            ch = MlpChain(layers, "cuda", IN_GATHER_EDGE, feat_c, OUT_MAXPOOL, group=K, slots=slots, pairs=pairs, coop=coop,
                          subs=subs, tma_in=tma)
        except RuntimeError:
            continue  # no deadlock-free plan under these constraints
        key = (ch.describe(), tma)
        if key in seen:
            continue
        seen.add(key)
        got = ch.run_gather(feat, xyz, ctr, nbr, term)
        torch.cuda.synchronize()
        if want is None:
            want = got
        assert torch.equal(got, want), "plan %r differs from the planner's default" % ((slots, pairs, coop, subs, tma),)
    assert len(seen) >= 4, "only %d distinct plans were exercised" % len(seen)


# ---------------------------------------------------------------------------------------------------- the model
@pytest.fixture(scope="module")
def gold():
    return dict(np.load(os.path.join(os.path.dirname(__file__), "golden", "edge_models.npz")))


@pytest.mark.parametrize("backend", ["tcgen05", "torch", "tf32"])
def test_golden_every_backend(gold, backend):
    """fused=True against the reference's own EdgePointNet2Down outputs, within the backend's stated tolerance"""
    from s4g_release_b200.engine import FusedEdgePointNet2Down
    from s4g_release_b200.network_models.models.EdgePointNet2Down import EdgePointNet2Down
    net = EdgePointNet2Down(**GOLDEN_CFG)
    net.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in gold.items() if k.startswith("sd/")}, strict=True)
    net = net.cuda().eval()
    eng = FusedEdgePointNet2Down(net, mlp_backend=backend)
    assert eng.edge_levels == [False, True, True, False]
    net.attach_engine(eng)
    with torch.no_grad():
        out = net({"scene_points": torch.from_numpy(gold["points"]).cuda()}, fused=True)
    assert net._engine is eng
    errs = {k: _rel_err(out[k], gold["out/" + k]) for k in KEYS}
    print("golden %s: %s" % (backend, errs))
    for k in KEYS:
        assert tuple(out[k].shape) == gold["out/" + k].shape, k
        assert errs[k] <= eng.tolerance(), (backend, k, errs[k])


def test_class_defaults_fused_match_module_path():
    """EdgePointNet2Down(score_classes=3): 10240 / 1024 / 128 / global; edge levels 1 and 2 over 64 / 128 channels"""
    from tests.inputs import tabletop_batch
    net = _seeded(dict(score_classes=3), seed=1)
    x = tabletop_batch(2, n_points=12288).cuda()
    with torch.no_grad():
        fused = net({"scene_points": x}, fused=True)
        ref = net({"scene_points": x}, fused=False)
    assert net.fused_engine().edge_levels == [False, True, True, False]
    errs = {k: _rel_err(fused[k], ref[k]) for k in KEYS}
    print("class defaults vs module path: %s" % errs)
    for k in KEYS:
        assert errs[k] <= net.fused_engine().tolerance(), (k, errs[k])


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
    for k in a:
        assert torch.equal(a[k][1:2], one[k]), k
        assert torch.equal(a[k], c[k]), k


def test_fused_forward_launches_no_torch_kernel_and_two_more_per_edge_level():
    from torch.profiler import ProfilerActivity, profile
    from s4g_release_b200 import _lib
    from tests.inputs import uniform_cloud
    x = uniform_cloud(2, 2048, seed=7).cuda()
    counts = {}
    for cls in ("edge", "sibling"):
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
        if cls == "edge":
            assert sum("gather_rows" in n for n in names) == 2, names
    # per edge level: the centroid rows and their term chain; everything else launches as in the PN2 sibling
    assert counts["edge"] == counts["sibling"] + 2 * 2, counts


@pytest.mark.parametrize("mode", ["wa_is_minus_wb", "wa_is_zero"])
def test_cancelling_split_against_the_torch_backend(mode):
    """W_a = -W_b + eps (the sum W_a + W_b is tiny) and W_a = eps (the whole layer is W_b (f_j - f_c): the centroid term
    cancels the neighbour term where f_j ~ f_c) on both edge levels of the class defaults.  The split's extra roundings
    (W_a + W_b and u in bf16) against the torch backend's literal edge rows in fp32; the error is printed."""
    from s4g_release_b200.engine import FusedEdgePointNet2Down
    from tests.inputs import tabletop_batch
    net = _seeded(dict(score_classes=3), seed=6)
    g = torch.Generator().manual_seed(6)
    with torch.no_grad():
        for i in (1, 2):
            w = net.sa_modules[i].mlp[0].conv.weight  # (cout, 3 + 2C, 1, 1)
            c = (w.shape[1] - 3) // 2
            eps = 1e-3 * torch.randn(w.shape[0], c, 1, 1, generator=g).cuda()
            w[:, 3:3 + c] = (-w[:, 3 + c:] + eps) if mode == "wa_is_minus_wb" else eps
    x = tabletop_batch(2, n_points=12288).cuda()
    eng = FusedEdgePointNet2Down(net)
    with torch.no_grad():
        got = eng.forward(x)
        ref = FusedEdgePointNet2Down(net, mlp_backend="torch").forward(x)
    errs = {k: _rel_err(got[k], ref[k]) for k in got}
    print("cancelling split (%s): tcgen05 vs torch backend %s" % (mode, errs))
    for k in got:
        assert errs[k] <= eng.tolerance(), (k, errs[k])
