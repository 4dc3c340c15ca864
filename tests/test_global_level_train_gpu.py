"""GPU: the fused training step with a global set-abstraction level (num_centroids = 0) and broadcast propagation
(num_fp_neighbours[0] = 0) — s4g_train_bn_act_segmax_bf16, the int32-routed BatchNorm-backward passes,
s4g_train_rows_segment_sum_bf16 and train_engine.TrainEngine around them.

Kernel level: against torch on the same bf16 operands.  Step level: against autograd of a rounding-matched torch
emulation of the step (bf16 where the fused path stores bf16) and against the fp32 module path, with the tolerances of
tests/test_train_engine_gpu.py."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.test_global_level_train_cpu import G_SHALLOW, G_WIDE

pytestmark = pytest.mark.gpu
BF = torch.bfloat16


def _lib():
    from s4g_release_b200._lib import check, lib, ptr, stream_ptr
    return check, lib, ptr, stream_ptr


def _tied_inputs(B, N, C, seed):
    """bf16 rows with few distinct values (many ties, many ReLU zeros) and scale / shift for which y * scale + shift is
    exact in fp32 — so torch's separate multiply and add give the kernel's fused multiply-add bit for bit"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    y = (torch.randint(-8, 8, (B * N, C), generator=g, device="cuda", dtype=torch.int32).float() / 4).to(BF)
    scale = (torch.rand(C, generator=g, device="cuda") + 0.5).to(BF).float()
    shift = torch.randint(-4, 5, (C,), generator=g, device="cuda").float() / 8
    return y, scale, shift


def _segmax(y, scale, shift, B, N, with_ymax=True):
    check, lib, ptr, stream_ptr = _lib()
    C = y.shape[1]
    out = torch.empty((B, C), dtype=BF, device="cuda")
    arg = torch.empty((B, C), dtype=torch.int32, device="cuda")
    ymax = torch.empty((B, C), dtype=BF, device="cuda") if with_ymax else None
    work = torch.empty((B, C), dtype=torch.int64, device="cuda")
    check(lib.s4g_train_bn_act_segmax_bf16(ptr(y), ptr(scale), ptr(shift), ptr(out), ptr(arg),
                                           ptr(ymax) if with_ymax else None, ptr(work), B, N, C, 1, stream_ptr(y.device)),
          "segmax")
    return out, arg, ymax


SEG_NS = (1, 7, 64, 100, 255, 256, 1000, 25600)
SEG_CS = (8, 72, 1024)
SEG_CASES = [(N, C, (1, 3, 32)[(i + j + 2) % 3]) for i, N in enumerate(SEG_NS) for j, C in enumerate(SEG_CS)]
assert (25600, 1024, 32) in SEG_CASES  # one large-N pool: 32 scenes x 25 600 rows x 1 024 channels


@pytest.mark.parametrize("N,C,B", SEG_CASES)
def test_segmax_against_torch(N, C, B):
    y, scale, shift = _tied_inputs(B, N, C, seed=N + C + B)
    out, arg, ymax = _segmax(y, scale, shift, B, N)
    out2, arg2, ymax2 = _segmax(y, scale, shift, B, N)
    torch.cuda.synchronize()
    assert torch.equal(out, out2) and torch.equal(arg, arg2) and torch.equal(ymax, ymax2)  # bit-identical runs
    t = torch.relu(y.float() * scale + shift).reshape(B, N, C)
    best = t.amax(dim=1)
    rows = torch.arange(N, device="cuda").view(1, N, 1)
    first = torch.where(t == best.unsqueeze(1), rows, N).amin(dim=1)  # the first row holding the maximum
    assert torch.equal(out, best.to(BF))
    assert torch.equal(arg.long(), first)
    assert torch.equal(ymax, torch.gather(y.reshape(B, N, C), 1, first.unsqueeze(1))[:, 0])
    if B * N * C <= 1 << 22:  # and against the CPU argmax (its documented rule: the first maximal value)
        assert torch.equal(arg.long().cpu(), torch.argmax(t.cpu(), dim=1))


def test_segmax_without_ymax_writes_the_same_pool():
    y, scale, shift = _tied_inputs(3, 1000, 72, seed=5)
    a = _segmax(y, scale, shift, 3, 1000)
    b = _segmax(y, scale, shift, 3, 1000, with_ymax=False)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.parametrize("B,N,C", [(3, 1000, 136), (2, 64, 264), (4, 25600, 128), (1, 7, 72), (5, 100, 1024)])
def test_int32_routed_bn_backward_against_torch(B, N, C):
    """apply pass (dy = ka * g + kb * y + kc) and the dense reduce (sum g, sum g * y) with g = the pooled gradient routed
    to row arg[b][c] of scene b and masked by ReLU' — the tolerances of test_bn_bwd_apply_against_torch"""
    check, lib, ptr, stream_ptr = _lib()
    P = B * N
    g = torch.Generator().manual_seed(P + C)
    y = torch.randn(P, C, generator=g).cuda().to(BF)
    scale = (torch.rand(C, generator=g) + 0.5).cuda()
    shift = (torch.randn(C, generator=g) * 0.3).cuda()
    ka, kb, kc = [(torch.randn(C, generator=g) * 0.5).cuda() for _ in range(3)]
    dz = torch.randn(B, C, generator=g).cuda().to(BF)
    _, arg, _ = _segmax(y, scale, shift, B, N)
    pos = (y.float() * scale + shift) > 0
    routed = torch.zeros(B, N, C, device="cuda")
    routed.scatter_(1, arg.long().unsqueeze(1), dz.float().unsqueeze(1))
    gm = torch.where(pos, routed.reshape(P, C), torch.zeros((), device="cuda"))
    st = stream_ptr(y.device)
    dy = torch.empty(P, C, dtype=BF, device="cuda")
    check(lib.s4g_train_bn_bwd_apply_seg_bf16(ptr(dz), ptr(arg), N, ptr(y), ptr(scale), ptr(shift), ptr(ka), ptr(kb),
                                              ptr(kc), P, C, 1, ptr(dy), st), "apply_seg")
    sums = torch.empty(2 * C, dtype=torch.float64, device="cuda")
    check(lib.s4g_train_bn_bwd_reduce_seg_bf16(ptr(dz), ptr(arg), N, ptr(y), ptr(scale), ptr(shift), P, C, 1, ptr(sums), st),
          "reduce_seg")
    torch.cuda.synchronize()
    want = ka * gm + kb * y.float() + kc
    assert (dy.float() - want).abs().max().item() <= 2 ** -7 * max(1.0, want.abs().max().item())
    gd = gm.double()
    np.testing.assert_allclose(sums[:C].cpu().numpy(), gd.sum(0).cpu().numpy(), rtol=1e-4, atol=2e-2)
    np.testing.assert_allclose(sums[C:].cpu().numpy(), (gd * y.double()).sum(0).cpu().numpy(), rtol=1e-4, atol=2e-2)


def _block(cin, cout, seed):
    from s4g_release_b200.network_models.nn_utils.conv import Conv1d
    torch.manual_seed(seed)
    blk = Conv1d(cin, cout, 1)
    blk.bn.weight.data = torch.rand(cout) + 0.5
    blk.bn.bias.data = torch.randn(cout) * 0.2
    return blk.cuda()


@pytest.mark.parametrize("sparse_reduce", [True, False])
@pytest.mark.parametrize("B,N", [(2, 1000), (3, 64)])
def test_global_pool_block_against_autograd(B, N, sparse_reduce, monkeypatch):
    """conv + BatchNorm(train) + ReLU + max over each scene's N rows, forward and backward through Block(global_pool)
    against torch autograd of normalise -> ReLU -> max on the same bf16 rounding; the backward's reduce over the B
    arg-max rows (SPARSE_POOL_REDUCE) and over all rows"""
    from s4g_release_b200 import train_engine as te
    monkeypatch.setattr(te, "SPARSE_POOL_REDUCE", sparse_reduce)
    cin, cout = 72, 96
    blk, ref = _block(cin, cout, seed=3), _block(cin, cout, seed=3)
    ref.load_state_dict(blk.state_dict())
    x = torch.randn(B * N, cin, generator=torch.Generator().manual_seed(5)).to(BF).float().cuda()
    b = te.Block(blk)
    z, arg = b.forward(x.to(BF), pool_k=N, global_pool=True)
    assert arg.dtype == torch.int32 and tuple(z.shape) == (B, cout)
    xr = x.clone().requires_grad_(True)
    ref.train()
    ref.conv.weight.data = ref.conv.weight.data.to(BF).float()
    yr = F.linear(xr, ref.conv.weight.reshape(cout, cin))
    yr = yr + (yr.to(BF).float() - yr).detach()
    zr = torch.relu(ref.bn(yr.t().unsqueeze(0)))[0].t().reshape(B, N, cout).max(dim=1)[0]
    assert (z.float() - zr).abs().max().item() <= 3e-2 * max(1.0, zr.abs().max().item())
    np.testing.assert_allclose(blk.bn.running_mean.cpu().numpy(), ref.bn.running_mean.cpu().numpy(), atol=2e-3)
    np.testing.assert_allclose(blk.bn.running_var.cpu().numpy(), ref.bn.running_var.cpu().numpy(), rtol=2e-2, atol=1e-3)
    dz = torch.randn(zr.shape, generator=torch.Generator().manual_seed(6)).to(BF).float().cuda()
    zr.backward(dz)
    dx = b.backward(dz.to(BF))
    torch.cuda.synchronize()

    def close(got, want, tol):
        rel = (got.float() - want).norm().item() / max(want.norm().item(), 1e-12)
        assert rel <= tol, rel
    close(dx, xr.grad, 3e-2)
    close(blk.conv.weight.grad.reshape(cout, cin), ref.conv.weight.grad.reshape(cout, cin), 3e-2)
    close(blk.bn.weight.grad, ref.bn.weight.grad, 3e-2)
    close(blk.bn.bias.grad, ref.bn.bias.grad, 3e-2)


@pytest.mark.parametrize("B,Nq,c2,ld", [(32, 128, 1024, 1280), (3, 1000, 72, 136), (2, 7, 8, 16), (1, 25600, 256, 512),
                                        (4, 300, 520, 520)])
def test_rows_segment_sum(B, Nq, c2, ld):
    from s4g_release_b200.train_engine import rows_segment_sum
    g = torch.Generator().manual_seed(B + Nq + c2)
    wide = torch.randn(B * Nq, ld, generator=g).cuda().to(BF)
    base = torch.randn(B, c2, generator=g).cuda()
    outs = []
    for _ in range(2):
        out = base.clone()
        rows_segment_sum(wide[:, :c2] if ld > c2 else wide, B, Nq, c2, out)
        outs.append(out)
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])  # fixed order: bit-identical runs
    d = wide[:, :c2].double().reshape(B, Nq, c2)
    want = base.double() + d.sum(1)
    scale = d.abs().sum(1) + base.double().abs()
    assert ((outs[0].double() - want).abs() <= 1e-5 * scale.clamp_min(1e-30)).all()


# ------------------------------------------------------------------------------------------- the step
def _r(x):
    """round to bf16, straight-through for the gradient: the fused path stores this tensor in bf16"""
    return x + (x.to(BF).float() - x).detach()


def _emulated_forward(model, pts):
    """The training forward in plain torch (fp32, autograd) with bf16 rounding where the fused path stores bf16 —
    tests/test_train_engine_gpu.py::_emulated_forward plus the global level (every point of a scene once, absolute
    coordinates, max over the scene) and the broadcast propagation level ([global | skip] rows)."""
    from s4g_release_b200.engine import FusedPointNet2 as E
    cfg = model.config

    def block(x, blk, pool_k=0):
        w = _r(blk.conv.weight.reshape(blk.conv.weight.shape[0], -1))
        y = _r(x @ w.t())
        z = torch.relu(F.batch_norm(y.t().unsqueeze(0), None, None, blk.bn.weight, blk.bn.bias, True, 0.0, blk.bn.eps)[0].t())
        if pool_k:
            z = z.reshape(-1, pool_k, z.shape[1]).max(dim=1)[0]
        return _r(z)

    xyz = pts
    B = xyz.shape[0]
    feat = None
    lv_xyz, lv_feat = [xyz], [None]
    for i, sa in enumerate(model.sa_modules):
        M, K = cfg["num_centroids"][i], cfg["num_neighbours"][i]
        N = xyz.shape[2]
        if M == 0:
            x = torch.cat([_r(xyz.permute(0, 2, 1).reshape(-1, 3)), feat], dim=1)  # [xyz | features], row b * N + n
            ctr, K = xyz.new_zeros(B, 3, 1), N
        else:
            idx = E.fps(xyz, M)
            ctr = E.gather_xyz(xyz, idx)
            nbr = E.ball_query(xyz, ctr, cfg["radius"][i], K).long().reshape(B, M * K)
            rel = torch.gather(xyz, 2, nbr.unsqueeze(1).expand(-1, 3, -1)).reshape(B, 3, M, K) - ctr.unsqueeze(-1)
            x = _r(rel.permute(0, 2, 3, 1).reshape(-1, 3))
            if feat is not None:
                c = feat.shape[1]
                gf = torch.gather(feat.reshape(B, N, c), 1, nbr.unsqueeze(-1).expand(-1, -1, c)).reshape(-1, c)
                x = torch.cat([x, gf], dim=1)
        for j, blk in enumerate(sa.mlp):
            x = block(x, blk, pool_k=K if j == len(sa.mlp) - 1 else 0)
        feat, xyz = x, ctr
        lv_xyz.append(xyz)
        lv_feat.append(feat)
    sparse_xyz, sparse = xyz, feat
    for i, fp in enumerate(model.fp_modules):
        dense_xyz, dense = lv_xyz[-2 - i], lv_feat[-2 - i]
        Nk, Nq, c = sparse_xyz.shape[2], dense_xyz.shape[2], sparse.shape[1]
        if cfg["num_fp_neighbours"][i] == 0:
            x = torch.cat([sparse.reshape(B, 1, c).expand(B, Nq, c).reshape(-1, c), dense], dim=1)
        else:
            idx3, w = E.three_nn_weights(dense_xyz, sparse_xyz)
            g = torch.gather(sparse.reshape(B, Nk, c), 1, idx3.long().reshape(B, Nq * 3, 1).expand(-1, -1, c))
            interp = _r((g.reshape(B, Nq, 3, c) * w.unsqueeze(-1)).sum(2).reshape(-1, c))
            x = interp if dense is None else torch.cat([interp, dense], dim=1)
        for blk in fp.mlp:
            x = block(x, blk)
        sparse_xyz, sparse = dense_xyz, x
    n = sparse_xyz.shape[2]
    outs = []
    for mlp, logit in ((model.mlp_seg, model.seg_logit), (model.mlp_R, model.R_logit), (model.mlp_t, model.t_logit),
                       (model.mlp_movable, model.movable_logit[0])):
        h = sparse
        for blk in mlp:
            h = block(h, blk)
        o = torch.addmm(logit.bias, h, logit.weight.reshape(logit.weight.shape[0], -1).t())
        outs.append(o.reshape(B, n, -1).permute(0, 2, 1))
    raw = {"score": outs[0], "frame_R": outs[1], "frame_t": outs[2], "movable_logits": torch.sigmoid(outs[3])}
    return model.predictions(raw, pts)


def _models(cfg, seed, sibling=False):
    from s4g_release_b200.network_models.models import PointNet2, PointNet2_tcls
    mod = PointNet2 if sibling else PointNet2_tcls
    torch.manual_seed(seed)
    a = mod.PointNet2(**cfg).cuda()
    g = torch.Generator().manual_seed(seed + 1)
    for m in a.modules():  # non-trivial BatchNorm affine parameters
        if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
            m.weight.data = (torch.rand(m.num_features, generator=g) + 0.5).cuda()
            m.bias.data = (torch.randn(m.num_features, generator=g) * 0.1).cuda()
    b = mod.PointNet2(**cfg).cuda()
    b.load_state_dict(a.state_dict())
    pts = torch.rand(2, 3, 2048, generator=g).cuda()
    pts[:, 2] *= 0.3
    from s4g_release_b200.train import synthetic_labels
    labels = synthetic_labels(2, 2048, num_frame=500, first_seed=7, device="cuda", continuous_t=sibling)
    return a, b, pts, labels, mod.PointNet2Loss(neg_weight=0.5)


def _cancelling_bias(model):
    """{name of a gradient that is ZERO in exact arithmetic: name of the gradient that gives its scale}.  The global
    level's pooled output reaches the loss only through the broadcast level's first BatchNorm (train mode), whose input
    gradient sums to zero over all B * Nq rows; so the gradients of the B broadcast global features sum to zero over the
    scenes, and so does the bias gradient of the global level's last BatchNorm, d beta = sum_b d global_b (wherever the
    scene's maximum is positive).  Both paths compute a difference of equal and opposite per-scene sums there — fp32
    rounding in the reference, bf16 rounding of the summed rows in the fused path — so a relative error against the
    reference's ~1e-7 residue measures only the rounding.  It is measured against the scale of the per-scene terms, the
    same BatchNorm's weight gradient, instead."""
    i = len(model.sa_modules) - 1
    j = len(model.sa_modules[i].mlp) - 1
    return {"sa_modules.%d.mlp.%d.bn.bias" % (i, j): "sa_modules.%d.mlp.%d.bn.weight" % (i, j)}


def _grad_stats(a, b):
    """per parameter (relative L2 error of b's gradient against a's, cosine); for a cancelling bias (_cancelling_bias)
    the L2 error over the norm of the same BatchNorm's weight gradient, cosine not defined (1.0)"""
    scale_of = _cancelling_bias(a)
    grads_a = {n: p.grad.flatten().double() for n, p in a.named_parameters()}
    stats = {}
    for (name, pa), (_, pb) in zip(a.named_parameters(), b.named_parameters()):
        assert pb.grad is not None, name
        ga, gb = grads_a[name], pb.grad.flatten().double()
        if name in scale_of:
            stats[name] = ((ga - gb).norm().item() / max(grads_a[scale_of[name]].norm().item(), 1e-12), 1.0)
            continue
        rel = (ga - gb).norm().item() / max(ga.norm().item(), 1e-12)
        cos = torch.dot(ga, gb).item() / max(ga.norm().item() * gb.norm().item(), 1e-30)
        stats[name] = (rel, cos)
    return stats


def test_the_cancelling_bias_gradient_is_rounding_only():
    """the premise of _cancelling_bias, on the fp32 module path: the bias gradient of the global level's last BatchNorm
    is rounding-sized next to its weight gradient, and the per-scene gradients of the broadcast global feature cancel"""
    a, _, pts, labels, loss_fn = _models(G_SHALLOW, seed=0)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    a.train()
    feats = []

    def keep(module, inputs, output):  # output = (centroid xyz, pooled global feature (B, C, 1))
        output[1].retain_grad()
        feats.append(output[1])

    handle = a.sa_modules[-1].register_forward_hook(keep)
    try:
        sum(loss_fn(a({"scene_points": pts}), labels).values()).backward()
    finally:
        handle.remove()
    d_global = feats[0].grad.double()  # (B, C, 1)
    assert d_global.sum(0).norm().item() <= 1e-4 * d_global.norm().item()
    (name, scale), = _cancelling_bias(a).items()
    params = dict(a.named_parameters())
    assert params[name].grad.norm().item() <= 1e-4 * params[scale].grad.norm().item()


def _compare_step(cfg, seed, reference="emulated", sibling=False):
    from s4g_release_b200.train_engine import TrainEngine
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    a, b, pts, labels, loss_fn = _models(cfg, seed, sibling)
    a.train()
    la = loss_fn(_emulated_forward(a, pts) if reference == "emulated" else a({"scene_points": pts}), labels)
    sum(la.values()).backward()
    b.train()
    lb = TrainEngine(b, loss_fn).step_loss({"scene_points": pts}, labels)
    torch.cuda.synchronize()
    return a, b, la, lb, _grad_stats(a, b)


@pytest.mark.parametrize("name", ["G_SHALLOW", "G_WIDE"])
def test_global_step_against_the_rounding_matched_reference(name):
    a, b, la, lb, stats = _compare_step({"G_SHALLOW": G_SHALLOW, "G_WIDE": G_WIDE}[name], seed=0)
    for k in la:
        assert abs(la[k].item() - lb[k].item()) <= 1e-2 * max(abs(la[k].item()), 0.05), (k, la[k].item(), lb[k].item())
    print(name, "vs emulation, worst (rel L2, cos):", max(v[0] for v in stats.values()), min(v[1] for v in stats.values()))
    bad = {n: v for n, v in stats.items() if v[0] > 6e-2 or v[1] < 0.997}
    assert not bad, bad


@pytest.mark.parametrize("name", ["G_SHALLOW", "G_WIDE"])
def test_global_step_against_the_fp32_module_path(name):
    a, b, la, lb, stats = _compare_step({"G_SHALLOW": G_SHALLOW, "G_WIDE": G_WIDE}[name], seed=0, reference="module")
    for k in la:
        assert abs(la[k].item() - lb[k].item()) <= 3e-2 * max(abs(la[k].item()), 0.05), (k, la[k].item(), lb[k].item())
    for (bname, ba), (_, bb) in zip(a.named_buffers(), b.named_buffers()):
        if "running" in bname:
            assert torch.allclose(ba, bb, rtol=3e-2, atol=3e-3), bname
        if "num_batches" in bname:
            assert int(ba) == int(bb) == 1, bname


def test_global_level_counts_every_point_once():
    """A global level over N = 100 points (a partial group of 64 padded to 128 rows would show): its first block's
    grouped rows are exactly the B * N level-1 points, each once, and its running mean / variance after one step are
    torch BatchNorm's over exactly those B * N pre-activation rows."""
    from s4g_release_b200.engine import FusedPointNet2 as E
    from s4g_release_b200.train_engine import TrainEngine
    cfg = dict(G_SHALLOW, num_centroids=(400, 100, 0))
    a, _, pts, _, loss_fn = _models(cfg, seed=2)
    a.train()
    eng = TrainEngine(a, loss_fn)
    with torch.no_grad():
        eng._trunk_forward(pts)
    torch.cuda.synchronize()
    blk = eng.sa[-1][0]
    x, y = blk.saved[0], blk.saved[1]
    B, N, cf = 2, 100, 64
    assert tuple(x.shape) == (B * N, cf + 8) and y.shape[0] == B * N
    l0 = E.gather_xyz(pts, E.fps(pts, 400))
    l1 = E.gather_xyz(l0, E.fps(l0, 100))
    assert torch.equal(x[:, cf:cf + 3], l1.permute(0, 2, 1).reshape(-1, 3).to(BF)) and (x[:, cf + 3:] == 0).all()
    bn = a.sa_modules[-1].mlp[0].bn
    ref = torch.nn.BatchNorm1d(bn.num_features, eps=bn.eps, momentum=bn.momentum).cuda().double().train()
    ref(y.double())
    assert int(bn.num_batches_tracked) == 1
    torch.testing.assert_close(bn.running_mean.double(), ref.running_mean, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(bn.running_var.double(), ref.running_var, rtol=1e-5, atol=1e-6)


def test_sibling_step_against_the_module_path():
    a, b, la, lb, stats = _compare_step(G_SHALLOW, seed=1, reference="module", sibling=True)
    for k in la:
        assert torch.isfinite(lb[k]), k
        assert abs(la[k].item() - lb[k].item()) <= 3e-2 * max(abs(la[k].item()), 0.05), (k, la[k].item(), lb[k].item())
    assert all(np.isfinite(v[0]) for v in stats.values())


def test_sibling_sequential_heads_equal_the_joint_step():
    from s4g_release_b200.train_engine import TrainEngine
    a, b, pts, labels, loss_fn = _models(G_SHALLOW, seed=4, sibling=True)
    a.train()
    b.train()
    ea, eb = TrainEngine(a, loss_fn), TrainEngine(b, loss_fn)
    ea.sequential_heads = False
    assert eb._separable()
    la, lb = ea.step_loss({"scene_points": pts}, labels), eb.step_loss({"scene_points": pts}, labels)
    for k in la:
        assert torch.allclose(la[k], lb[k], rtol=1e-5, atol=1e-6), k
    torch.cuda.synchronize()
    bad = {n: v for n, v in _grad_stats(a, b).items() if v[0] > 2e-2}
    assert not bad, bad


# the sibling's default structure (four levels, the last one global, broadcast first propagation) at reduced width
SIBLING_SMALL = dict(score_classes=3, num_centroids=(512, 128, 32, 0), radius=(0.2, 0.3, 0.4, -1.0),
                     num_neighbours=(32, 32, 16, -1), sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 128, 256)),
                     fp_channels=((128, 128), (128, 64), (64, 64), (32, 32, 32)), num_fp_neighbours=(0, 3, 3, 3),
                     seg_channels=(64,), num_removal_directions=5, dropout_prob=0.5)


@pytest.mark.parametrize("sibling, cfg", [(True, SIBLING_SMALL), (False, dict(G_SHALLOW, dropout_prob=0.5))])
def test_trainer_with_the_fused_step_reduces_the_loss(sibling, cfg):
    from s4g_release_b200.train import Trainer
    _, net, pts, labels, loss_fn = _models(cfg, seed=0, sibling=sibling)
    tr = Trainer(net, loss_fn, lr=2e-3, fused=True)
    first = last = None
    for _ in range(12):
        total = float(sum(tr.step({"scene_points": pts}, labels).values()))
        assert np.isfinite(total)
        first = total if first is None else first
        last = total
    assert last < first, (first, last)
