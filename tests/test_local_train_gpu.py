"""GPU: PN2_LOCAL's fused training step — the channel-dropout BatchNorm passes (s4g_train_bn_act_chdrop_bf16,
s4g_train_bn_bwd_{reduce,apply}_chdrop_bf16), the evaluation-row backward (s4g_local_eval_rows_bwd_bf16) and
train_engine.LocalTrainEngine around them.

Kernel level: against torch on the same bf16 operands.  Step level: against autograd of a rounding-matched torch
emulation (bf16 where the fused path stores bf16) and against the fp32 module path, with the tolerances of
tests/test_global_level_train_gpu.py, in the given and the self mode of the evaluation head."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.test_global_level_train_gpu import _emulated_forward, _grad_stats, _r

pytestmark = pytest.mark.gpu
BF = torch.bfloat16


def _lib():
    from s4g_release_b200._lib import check, lib, ptr, stream_ptr
    return check, lib, ptr, stream_ptr


# ------------------------------------------------------------------------------------------- channel dropout
def _chdrop_act(y, scale, shift, scene_rows, seed, p):
    check, lib, ptr, stream_ptr = _lib()
    P, C = y.shape
    z = torch.empty_like(y)
    check(lib.s4g_train_bn_act_chdrop_bf16(ptr(y), ptr(scale), ptr(shift), ptr(z), P, C, 1, scene_rows, seed, p,
                                           stream_ptr(y.device)), "bn_act_chdrop")
    return z


def _assert_bf16_of(got, want):
    """got (bf16) is want (fp32) rounded once, up to the kernel's fused multiply-add (torch rounds y * scale first)"""
    assert ((got.float() - want).abs() <= 2.0 ** -8 * want.abs()).all()


def _positive_inputs(B, R, C, seed):
    """rows whose pre-activation y * scale + shift is positive everywhere, so a zero in the output is a dropped channel"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    y = (torch.rand(B * R, C, generator=g, device="cuda") + 0.25).to(BF)
    scale = torch.rand(C, generator=g, device="cuda") + 0.5
    shift = torch.rand(C, generator=g, device="cuda") * 0.1
    return y, scale, shift


@pytest.mark.parametrize("B,R,C,p", [(64, 100, 256, 0.5), (7, 1000, 72, 0.3), (3, 1, 8, 0.5), (32, 65536, 32, 0.5)])
def test_channel_dropout_is_per_scene_and_channel(B, R, C, p):
    y, scale, shift = _positive_inputs(B, R, C, seed=B + R + C)
    z = _chdrop_act(y, scale, shift, R, 12345, p)
    torch.cuda.synchronize()
    t = (y.float() * scale + shift).reshape(B, R, C)
    kept = (z.reshape(B, R, C) != 0)
    mask = kept[:, 0]  # (B, C)
    assert torch.equal(kept, mask.unsqueeze(1).expand_as(kept))  # every row of a scene agrees
    want = torch.where(mask.unsqueeze(1), t * (1.0 / (1.0 - p)), torch.zeros((), device="cuda"))
    _assert_bf16_of(z.reshape(B, R, C), want)
    if B * C >= 2000:
        frac = mask.float().mean().item()
        assert abs(frac - (1 - p)) < 4 * np.sqrt(p * (1 - p) / (B * C)) + 1e-3, frac
    assert torch.equal(z, _chdrop_act(y, scale, shift, R, 12345, p))  # same seed, same bits
    if B * C >= 64:
        other = _chdrop_act(y, scale, shift, R, 12346, p)
        assert not torch.equal(other.reshape(B, R, C)[:, 0] != 0, mask)


def test_channel_dropout_off_is_bn_act():
    check, lib, ptr, stream_ptr = _lib()
    y, scale, shift = _positive_inputs(4, 300, 64, seed=3)
    shift -= 1.0  # with ReLU zeros
    z0 = torch.empty_like(y)
    check(lib.s4g_train_bn_act_bf16(ptr(y), ptr(scale), ptr(shift), ptr(z0), y.shape[0], 64, 1, 7, 0.0,
                                    stream_ptr(y.device)), "bn_act")
    assert torch.equal(_chdrop_act(y, scale, shift, 300, 7, 0.0), z0)


@pytest.mark.parametrize("B,R,C,p", [(6, 1000, 136, 0.5), (32, 64, 128, 0.3), (2, 25600, 64, 0.5)])
def test_channel_dropout_backward_against_autograd(B, R, C, p):
    """reduce (sum g, sum g * y) and apply (dy = ka * g + kb * y + kc) with g the autograd gradient of dz through ReLU
    and F.dropout2d's masking and scaling, with the mask the forward drew (read back from its output)"""
    check, lib, ptr, stream_ptr = _lib()
    P = B * R
    gen = torch.Generator().manual_seed(P + C)
    y = torch.randn(P, C, generator=gen).cuda().to(BF)
    scale = (torch.rand(C, generator=gen) + 0.5).cuda()
    shift = (torch.randn(C, generator=gen) * 0.3).cuda()
    ka, kb, kc = [(torch.randn(C, generator=gen) * 0.5).cuda() for _ in range(3)]
    dz = torch.randn(P, C, generator=gen).cuda().to(BF)
    seed = 99
    # the mask: the forward on rows that are positive everywhere (same P, C, scenes, seed)
    ones = torch.ones_like(y)
    mask = (_chdrop_act(ones, torch.ones(C, device="cuda"), torch.zeros(C, device="cuda"), R, seed, p)
            .reshape(B, R, C)[:, 0] != 0).float()  # (B, C)
    assert 0 < mask.mean().item() < 1
    z = _chdrop_act(y, scale, shift, R, seed, p)
    t = (y.float() * scale + shift).requires_grad_(True)
    ref = (torch.relu(t).reshape(B, R, C) * mask.unsqueeze(1) / (1 - p)).reshape(P, C)  # F.dropout2d with that mask
    _assert_bf16_of(z, ref.detach())
    ref.backward(dz.float())
    g = t.grad
    dy = torch.empty(P, C, dtype=BF, device="cuda")
    st = stream_ptr(y.device)
    check(lib.s4g_train_bn_bwd_apply_chdrop_bf16(ptr(dz), ptr(y), ptr(scale), ptr(shift), ptr(ka), ptr(kb), ptr(kc), P, C,
                                                 1, R, seed, p, ptr(dy), st), "apply_chdrop")
    sums = torch.empty(2 * C, dtype=torch.float64, device="cuda")
    check(lib.s4g_train_bn_bwd_reduce_chdrop_bf16(ptr(dz), ptr(y), ptr(scale), ptr(shift), P, C, 1, R, seed, p, ptr(sums),
                                                  st), "reduce_chdrop")
    torch.cuda.synchronize()
    want = ka * g + kb * y.float() + kc
    assert (dy.float() - want).abs().max().item() <= 2 ** -7 * max(1.0, want.abs().max().item())
    gd = g.double()
    np.testing.assert_allclose(sums[:C].cpu().numpy(), gd.sum(0).cpu().numpy(), rtol=1e-4, atol=2e-2)
    np.testing.assert_allclose(sums[C:].cpu().numpy(), (gd * y.double()).sum(0).cpu().numpy(), rtol=1e-4, atol=2e-2)


# ------------------------------------------------------------------------------------------- evaluation-row backward
def _rows_bwd(d, B, N, C, F_, S, dR=None, dt=None):
    check, lib, ptr, stream_ptr = _lib()
    dfeat = torch.empty(B * N, C, dtype=BF, device="cuda")
    check(lib.s4g_local_eval_rows_bwd_bf16(ptr(d), B, N, C, F_, S, ptr(dfeat), ptr(dR) if dR is not None else None,
                                           ptr(dt) if dt is not None else None, stream_ptr(d.device)), "eval_rows_bwd")
    return dfeat


def _assert_rounded_sum(got, parts):
    """got (bf16) = the fp32 sum of the bf16 parts (..., S, C) over S, rounded once: within the rounding of the result
    plus fp32 reassociation"""
    exact = parts.double().sum(-2)
    bound = 2.0 ** -8 * exact.abs() + 1e-5 * parts.double().abs().sum(-2) + 1e-30
    assert ((got.double() - exact).abs() <= bound).all()


@pytest.mark.parametrize("B,N,C,F_,S", [(3, 500, 64, 100, 1), (2, 1024, 128, 40, 6), (2, 300, 16, 300, 64),
                                        (4, 700, 32, 700, 1), (1, 64, 8, 1, 3)])
def test_eval_rows_backward_point_features(B, N, C, F_, S):
    g = torch.Generator(device="cuda").manual_seed(B * N + S)
    d = torch.randn(B * F_ * S, C + 48, generator=g, device="cuda").to(BF)
    dfeat = _rows_bwd(d, B, N, C, F_, S).reshape(B, N, C)
    torch.cuda.synchronize()
    assert torch.equal(dfeat, _rows_bwd(d, B, N, C, F_, S).reshape(B, N, C))  # fixed order: the same bits
    _assert_rounded_sum(dfeat[:, :F_], d.reshape(B, F_, S, C + 48)[..., :C])
    assert (dfeat[:, F_:] == 0).all()


def test_eval_rows_backward_self_mode_candidates():
    """F = N, S = 1: the point features are the rows' first C columns, and the sum over the 4 repeats of the 12
    candidate columns is ADDED to the R (B, 9, N) and t (B, 3, N) gradients already there"""
    B, N, C = 3, 2000, 64
    g = torch.Generator(device="cuda").manual_seed(4)
    d = torch.randn(B * N, C + 48, generator=g, device="cuda").to(BF)
    dR0 = torch.randn(B, 9, N, generator=g, device="cuda")
    dt0 = torch.randn(B, 3, N, generator=g, device="cuda")
    dR, dt = dR0.clone(), dt0.clone()
    dfeat = _rows_bwd(d, B, N, C, N, 1, dR, dt)
    torch.cuda.synchronize()
    assert torch.equal(dfeat, d[:, :C])
    cand = d[:, C:].float().reshape(B, N, 4, 12)
    s = ((cand[:, :, 0] + cand[:, :, 1]) + cand[:, :, 2]) + cand[:, :, 3]  # (B, N, 12), the kernel's order
    assert torch.equal(dR, dR0 + s[..., :9].permute(0, 2, 1))
    assert torch.equal(dt, dt0 + s[..., 9:].permute(0, 2, 1))
    check, lib, ptr, _ = _lib()
    # the candidate gradient exists in self mode only
    assert lib.s4g_local_eval_rows_bwd_bf16(ptr(d), B, N, C, N - 1, 1, ptr(dfeat), ptr(dR), ptr(dt), None) != 0


def test_eval_rows_backward_over_2_gib():
    """a row buffer of 2.3 GB: the last scene's last points, whose rows start beyond 2^31 bytes"""
    B, N, C, F_, S = 2, 4096, 128, 4096, 800
    rows = B * F_ * S
    assert rows * (C + 48) * 2 > 1 << 31
    d = torch.empty(rows, C + 48, dtype=BF, device="cuda")
    d.view(-1)[-(64 * S * (C + 48)):] = torch.randn(64 * S * (C + 48), device="cuda").to(BF)
    d.view(-1)[:-(64 * S * (C + 48))] = 0
    dfeat = _rows_bwd(d, B, N, C, F_, S).reshape(B, N, C)
    torch.cuda.synchronize()
    _assert_rounded_sum(dfeat[1, F_ - 64:], d[-64 * S:].reshape(64, S, C + 48)[..., :C])
    assert (dfeat[0] == 0).all() and (dfeat[1, :F_ - 64] == 0).all()
    del d


# ------------------------------------------------------------------------------------------- the step
# one block per MLP, a global last level: the shallow configuration of the global-level suite with PN2_LOCAL's heads
L_SHALLOW = dict(score_classes=3, num_centroids=(256, 64, 0), radius=(0.1, 0.2, -1.0), num_neighbours=(16, 16, -1),
                 sa_channels=((32,), (64,), (128,)), fp_channels=((128,), (64,), (64,)), num_fp_neighbours=(0, 3, 3),
                 seg_channels=(32,), dropout_prob=0.0)
N_POINTS, N_FRAMES, N_SEARCH = 2048, 500, 4


class _Trunk:
    """the trunk of the emulation in test_global_level_train_gpu: PN2_CLS's heads replaced by an identity 1x1 conv (exact
    in fp32), so its 'score' output is the per-point feature (B, C, N)"""

    def __init__(self, model):
        self.config, self.sa_modules, self.fp_modules = model.config, model.sa_modules, model.fp_modules
        c = model.fp_modules[-1].mlp[-1].conv.weight.shape[0]
        ident = torch.nn.Conv1d(c, c, 1).cuda()
        ident.weight.data = torch.eye(c, device="cuda").reshape(c, c, 1)
        ident.bias.data.zero_()
        self.mlp_seg = self.mlp_R = self.mlp_t = self.mlp_movable = ()
        self.seg_logit = self.R_logit = self.t_logit = ident
        self.movable_logit = [ident]

    def predictions(self, raw, pts):
        return raw["score"]


def _emulated_local(model, pts, frames=None):
    """the training forward of PN2_LOCAL in fp32 torch autograd with bf16 rounding where the fused path stores bf16;
    ``frames`` (given mode) are updated in place, as the reference does"""
    def block(x, blk):
        w = _r(blk.conv.weight.reshape(blk.conv.weight.shape[0], -1))
        y = _r(x @ w.t())
        return _r(torch.relu(F.batch_norm(y.t().unsqueeze(0), None, None, blk.bn.weight, blk.bn.bias, True, 0.0,
                                          blk.bn.eps)[0].t()))

    def head(mlp, logit, x):
        for blk in mlp:
            x = block(x, blk)
        return torch.addmm(logit.bias, x, logit.weight.reshape(logit.weight.shape[0], -1).t())

    B, _, N = pts.shape
    feat = _emulated_forward(_Trunk(model), pts).permute(0, 2, 1).reshape(B * N, -1)
    C = feat.shape[1]
    R, t, mov = [head(m, lg, feat).reshape(B, N, -1).permute(0, 2, 1) for m, lg in (
        (model.mlp_R, model.R_logit), (model.mlp_t, model.t_logit), (model.mlp_movable, model.movable_logit))]
    if frames is not None:
        F_, S = frames.shape[2:]
        frames[:, 9:] = frames[:, 9:] - pts[:, :, :F_].unsqueeze(-1)
        cand = frames.permute(0, 2, 3, 1)
        per_point = feat.reshape(B, N, 1, C)[:, :F_].expand(-1, -1, S, -1)
    else:
        F_, S = N, 1
        cand = torch.cat([R, t], dim=1).permute(0, 2, 1).unsqueeze(2)
        per_point = feat.reshape(B, N, 1, C)
    x = torch.cat([per_point, _r(cand).repeat(1, 1, 1, 4)], dim=-1).reshape(-1, C + 48)
    ev = head(model.mlp_grasp_eval, model.grasp_eval_logit, x).reshape(B, F_, S, -1).permute(0, 3, 1, 2)
    raw = {"local_search_logits": ev, "frame_R": R, "frame_t": t, "movable_logits": mov}
    return model.predictions(raw, pts)


def _local_models(cfg, seed, given):
    from s4g_release_b200.network_models.models.PointNet2_local import PointNet2, PointNet2Loss
    from s4g_release_b200.train import synthetic_local_batch
    torch.manual_seed(seed)
    a = PointNet2(**cfg).cuda()
    g = torch.Generator().manual_seed(seed + 1)
    for m in a.modules():  # non-trivial BatchNorm affine parameters
        if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
            m.weight.data = (torch.rand(m.num_features, generator=g) + 0.5).cuda()
            m.bias.data = (torch.randn(m.num_features, generator=g) * 0.1).cuda()
    a.t_logit.weight.data = (torch.randn(a.t_logit.weight.shape, generator=g) * 0.05).cuda()  # (zero-initialised)
    b = PointNet2(**cfg).cuda()
    b.load_state_dict(a.state_dict())
    pts = torch.rand(2, 3, N_POINTS, generator=g).cuda()
    pts[:, 2] *= 0.3
    frames, labels = synthetic_local_batch(pts, N_FRAMES, N_SEARCH, score_classes=cfg["score_classes"]) if given else \
        synthetic_local_batch(pts, N_POINTS, 1, score_classes=cfg["score_classes"])
    return a, b, pts, (frames if given else None), labels, PointNet2Loss(neg_weight=0.5)


def _batch(pts, frames):
    return {"scene_points": pts} if frames is None else {"scene_points": pts, "local_search_frame": frames}


def _compare_step(cfg, seed, given, reference="emulated"):
    from s4g_release_b200.train_engine import LocalTrainEngine
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    a, b, pts, frames, labels, loss_fn = _local_models(cfg, seed, given)
    a.train()
    fa = None if frames is None else frames.clone()
    preds = _emulated_local(a, pts, fa) if reference == "emulated" else a(_batch(pts, fa))
    la = loss_fn(preds, labels)
    sum(la.values()).backward()
    b.train()
    eng = LocalTrainEngine(b, loss_fn)
    fb = None if frames is None else frames.clone()
    lb = eng.step_loss(_batch(pts, fb), labels)
    torch.cuda.synchronize()
    return a, b, la, lb, _grad_stats(a, b), fa, fb


@pytest.mark.parametrize("given", [True, False], ids=["given", "self"])
def test_step_against_the_rounding_matched_reference(given):
    a, b, la, lb, stats, fa, fb = _compare_step(L_SHALLOW, seed=0, given=given)
    for k in la:
        assert abs(la[k].item() - lb[k].item()) <= 1e-2 * max(abs(la[k].item()), 0.05), (k, la[k].item(), lb[k].item())
    print("given" if given else "self", "vs emulation, worst (rel L2, cos):", max(v[0] for v in stats.values()),
          min(v[1] for v in stats.values()))
    bad = {n: v for n, v in stats.items() if v[0] > 6e-2 or v[1] < 0.997}
    assert not bad, bad
    if given:
        assert torch.equal(fa, fb)


@pytest.mark.parametrize("given", [True, False], ids=["given", "self"])
def test_step_against_the_fp32_module_path(given):
    a, b, la, lb, stats, fa, fb = _compare_step(L_SHALLOW, seed=0, given=given, reference="module")
    for k in la:
        assert abs(la[k].item() - lb[k].item()) <= 3e-2 * max(abs(la[k].item()), 0.05), (k, la[k].item(), lb[k].item())
    for (bname, ba), (_, bb) in zip(a.named_buffers(), b.named_buffers()):
        if "running" in bname:
            assert torch.allclose(ba, bb, rtol=3e-2, atol=3e-3), bname
        if "num_batches" in bname:
            assert int(ba) == int(bb) == 1, bname
    if given:  # one fused step updates the frames exactly as one module-path forward
        assert torch.equal(fa, fb)


def test_self_mode_couples_the_evaluation_head_to_R_and_t():
    """cls_loss reaches the R and t heads through the candidate rows: the step's R_logit gradient is the emulation's
    (R, t and cls terms), not the one of the R and t terms alone"""
    a, b, la, lb, stats, _, _ = _compare_step(L_SHALLOW, seed=3, given=False)
    coupled, fused = a.R_logit.weight.grad.double(), b.R_logit.weight.grad.double()
    _, _, pts, _, labels, loss_fn = _local_models(L_SHALLOW, 3, False)
    a.zero_grad()
    losses = loss_fn(_emulated_local(a, pts), labels)
    (losses["R_loss"] + losses["t_loss"]).backward()
    alone = a.R_logit.weight.grad.double()
    print("R_logit gradient: fused vs coupled %.3e, coupled vs R / t terms alone %.3e"
          % ((fused - coupled).norm() / coupled.norm(), (alone - coupled).norm() / coupled.norm()))
    assert (fused - coupled).norm() < 0.5 * (alone - coupled).norm()


def test_given_sequential_heads_equal_the_joint_step():
    from s4g_release_b200.train_engine import LocalTrainEngine
    a, b, pts, frames, labels, loss_fn = _local_models(L_SHALLOW, seed=4, given=True)
    a.train()
    b.train()
    ea, eb = LocalTrainEngine(a, loss_fn), LocalTrainEngine(b, loss_fn)
    ea.sequential_heads = False
    fa, fb = frames.clone(), frames.clone()
    la, lb = ea.step_loss(_batch(pts, fa), labels), eb.step_loss(_batch(pts, fb), labels)
    for k in la:
        assert torch.allclose(la[k], lb[k], rtol=1e-5, atol=1e-6), k
    torch.cuda.synchronize()
    assert torch.equal(fa, fb)
    bad = {n: v for n, v in _grad_stats(a, b).items() if v[0] > 2e-2}
    assert not bad, bad


@pytest.mark.parametrize("given", [True, False], ids=["given", "self"])
def test_trainer_with_the_fused_step_reduces_the_loss(given):
    from s4g_release_b200.train import Trainer
    _, net, pts, frames, labels, loss_fn = _local_models(dict(L_SHALLOW, dropout_prob=0.5), seed=0, given=given)
    tr = Trainer(net, loss_fn, lr=2e-3, fused=True)
    first = last = None
    for _ in range(12):
        total = float(sum(tr.step(_batch(pts, None if frames is None else frames.clone()), labels).values()))
        assert np.isfinite(total)
        first = total if first is None else first
        last = total
    assert last < first, (first, last)
