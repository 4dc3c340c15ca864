"""The PN2_LOCAL sibling model (network_models/models/PointNet2_local.py) and the Avg / MSG set-abstraction modules against
tests/golden/pn2_local.npz, which holds the outputs of the REFERENCE's own classes (tests/golden/make_pn2_local_golden.py)."""
import os

import numpy as np
import pytest
import torch

CFG = dict(score_classes=3, num_centroids=(256, 64, 16, 0), radius=(0.1, 0.2, 0.4, -1.0), num_neighbours=(16, 16, 8, -1),
           sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 128, 256)),
           fp_channels=((64, 64), (64, 32), (32, 32), (32, 32, 16)), num_fp_neighbours=(0, 3, 3, 3), seg_channels=(32,),
           dropout_prob=0.5)


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(os.path.join(os.path.dirname(__file__), "golden", "pn2_local.npz")))


@pytest.fixture(autouse=True)
def ieee_fp32_convolutions():
    """the goldens are fp32 CPU results: compare with IEEE fp32 convolutions, not torch's default TF32 (3e-4 off here)"""
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _sub(gold, prefix):
    return {k[len(prefix):]: torch.from_numpy(v) for k, v in gold.items() if k.startswith(prefix)}


def _reference_weights(gold):
    """The reference model's seeded weights: the fixture stores their digests, the generator's seeding rebuilds them."""
    from s4g_release_b200.network_models.models.PointNet2_local import PointNet2
    from tests.golden.make_golden import array_digest, seed_reference_weights
    torch.manual_seed(0)
    net = seed_reference_weights(PointNet2(**CFG))
    torch.nn.init.normal_(net.t_logit.weight, std=0.05)
    sd = net.state_dict()
    assert list(sd) == list(gold["sd_keys"])
    for (k, v), want in zip(sd.items(), gold["sd_sha256"]):
        assert array_digest(v) == want, k
    return sd


def test_module_surface_and_seeded_init(gold):
    from s4g_release_b200.network_models.models.PointNet2_local import PointNet2
    torch.manual_seed(0)
    sd = PointNet2(**CFG).state_dict()
    ref = _reference_weights(gold)
    assert list(sd) == list(ref) and all(sd[k].shape == ref[k].shape for k in sd)
    # same parameter creation order => identical default init under the same seed (BN / t_logit were re-seeded later)
    for k in ("sa_modules.0.mlp.0.conv.weight", "fp_modules.3.mlp.2.conv.weight", "mlp_grasp_eval.0.conv.weight",
              "grasp_eval_logit.weight", "R_logit.bias", "movable_logit.weight"):
        assert torch.equal(sd[k], ref[k]), k
    assert float(sd["t_logit.weight"].abs().max()) == 0.0 and float(sd["t_logit.bias"].abs().max()) == 0.0


def test_loss_and_metric_match_reference(gold):
    from s4g_release_b200.network_models.models.PointNet2_local import PointNet2Loss, PointNet2Metric
    preds, labels = _sub(gold, "given/"), _sub(gold, "label/")
    for k, v in PointNet2Loss()(preds, labels).items():
        np.testing.assert_allclose(v.item(), gold["loss/" + k].item(), rtol=1e-6, atol=1e-7)
    metric = PointNet2Metric()(preds, labels)
    assert sorted(metric) == ["R_err", "cls_acc", "mov_acc", "t_err"]
    assert np.array_equal(metric["cls_acc"].numpy(), gold["metric/cls_acc"])
    assert np.array_equal(metric["mov_acc"].numpy(), gold["metric/mov_acc"])
    np.testing.assert_allclose(metric["R_err"].item(), gold["metric/R_err"].item(), rtol=1e-5)
    np.testing.assert_allclose(metric["t_err"].item(), gold["metric/t_err"].item(), rtol=1e-6)


def test_builder_reads_the_reference_config_names():
    from types import SimpleNamespace as NS
    from s4g_release_b200.network_models.models.PointNet2_local import build_pointnet2_local
    pn2 = NS(NUM_CENTROIDS=CFG["num_centroids"], RADIUS=CFG["radius"], NUM_NEIGHBOURS=CFG["num_neighbours"],
             SA_CHANNELS=CFG["sa_channels"], FP_CHANNELS=CFG["fp_channels"], NUM_FP_NEIGHBOURS=CFG["num_fp_neighbours"],
             SEG_CHANNELS=CFG["seg_channels"], DROPOUT_PROB=0.5, LABEL_SMOOTHING=0, NEG_WEIGHT=0.1)
    net, loss, metric = build_pointnet2_local(NS(DATA=NS(SCORE_CLASSES=3), MODEL=NS(PN2=pn2)))
    assert net.grasp_eval_logit.out_channels == 3 and loss.neg_weight == 0.1 and callable(metric)


@pytest.mark.gpu
def test_forward_on_the_sm100a_operators(gold):
    """both branches of the grasp-evaluation head on the GPU operators, incl. the in-place update of the caller's frames"""
    from s4g_release_b200.network_models.models.PointNet2_local import PointNet2
    net = PointNet2(**CFG)
    net.load_state_dict(_reference_weights(gold), strict=True)
    net = net.cuda().eval()
    pts = torch.from_numpy(gold["points"]).cuda()
    frames = torch.from_numpy(gold["frames"]).cuda()
    with torch.no_grad():
        out_self = net({"scene_points": pts})
        out_given = net({"scene_points": pts, "local_search_frame": frames})
    np.testing.assert_allclose(frames.cpu().numpy(), gold["frames_after"], atol=1e-6, rtol=0)
    for tag, out in (("self/", out_self), ("given/", out_given)):
        for k in ("local_search_logits", "frame_R", "frame_t", "movable_logits"):
            want = gold[tag + k]
            assert tuple(out[k].shape) == want.shape
            np.testing.assert_allclose(out[k].cpu().numpy(), want, atol=2e-4 * max(1.0, np.abs(want).max()), rtol=0)


@pytest.mark.gpu
def test_avg_and_msg_set_abstraction_modules(gold):
    from s4g_release_b200.network_models.models.pointnet2_utils.modules import PointNetSAAvgModule, PointNetSAModuleMSG
    pts, feat = torch.from_numpy(gold["points"]).cuda(), torch.from_numpy(gold["feat"]).cuda()
    avg = PointNetSAAvgModule(24, (32, 48), 128, 0.15, 16, True)
    msg = PointNetSAModuleMSG(24, ((16, 32), (32, 64)), 128, (0.1, 0.2), (8, 16), True)
    avg.load_state_dict(_sub(gold, "avg_sd/"), strict=True)
    msg.load_state_dict(_sub(gold, "msg_sd/"), strict=True)
    with torch.no_grad():
        ax, af = avg.cuda().eval()(pts, feat)
        mx, mf = msg.cuda().eval()(pts, feat)
    assert np.array_equal(ax.cpu().numpy(), gold["avg/xyz"]) and np.array_equal(mx.cpu().numpy(), gold["msg/xyz"])  # FPS: bit-exact
    for got, want in ((af, gold["avg/feature"]), (mf, gold["msg/feature"])):
        np.testing.assert_allclose(got.cpu().numpy(), want, atol=2e-4 * max(1.0, np.abs(want).max()), rtol=0)


@pytest.mark.gpu
def test_edge_set_abstraction_and_propagation_modules(gold):
    """EdgeConv variants: edge-feature grouping and the k-NN gather over DENSE queries (dgcnn_ext.gather_knn)"""
    from s4g_release_b200.network_models.models.pointnet2_utils.modules import EdgeFPModule, EdgeSAModule
    pts, feat = torch.from_numpy(gold["points"]).cuda(), torch.from_numpy(gold["feat"]).cuda()
    esa = EdgeSAModule(24, (32, 48), 128, 0.15, 16, True)
    efp = EdgeFPModule(2 * 48 + 24, (64, 32), 3)
    esa.load_state_dict(_sub(gold, "esa_sd/"), strict=True)
    efp.load_state_dict(_sub(gold, "efp_sd/"), strict=True)
    with torch.no_grad():
        ex, ef = esa.cuda().eval()(pts, feat)
        back = efp.cuda().eval()(pts, ex, feat, ef)
    assert np.array_equal(ex.cpu().numpy(), gold["esa/xyz"])
    for got, want in ((ef, gold["esa/feature"]), (back, gold["efp/feature"])):
        assert tuple(got.shape) == want.shape
        np.testing.assert_allclose(got.cpu().numpy(), want, atol=2e-4 * max(1.0, np.abs(want).max()), rtol=0)
