"""GPU: score / SE(3)-pose parity of the fused forward against the fp32 CPU oracle of the reference — BASELINE config 1
(the shipped 2638_view_0 cloud) and 8 synthetic tabletop scenes (config 2).

`north_star`: "per-point grasp scores and SE(3) poses must match within a stated fp32/bf16 tolerance".  The quantities
compared are the ones the reference's consumer derives from the raw heads (grasp_detector.py:137-185, helper
tests/pose_parity.py): expected score, the score > 0.7 decision, the approach-offset class, the Gram-Schmidt'd rotation
(geodesic angle), the gripper translation (mm), the 50 best-scoring points.  Two weight sets, because the pretrained
weights are not in the checkout (tests/conditioned.py explains both):

  "seeded"      the weights of SURVEY.md §8d config 1 (what the golden fixtures use) — a contracting network.  ABSOLUTE
                bounds, stated in BOUNDS_SEEDED, worst case over the 9 scenes.
  "conditioned" He-normal weights + calibrated BatchNorm — a random deep network that amplifies perturbations ~30x, the
                stress case with real decisions (thousands of points above the 0.7 threshold).  Anything but IEEE fp32
                moves its outputs visibly, INCLUDING THE UNMODIFIED REFERENCE: on this GPU torch runs the reference's
                cuDNN convolutions in TF32 by default.  That deviation (reference model + reference CUDA kernels, TF32 on,
                vs the fp32 oracle) is measured in the same test when the reference is staged, else read from
                tests/golden/reference_tf32_floor.json, and is the yardstick: the TF32 tight-parity mode must
                stay within 2x of it, the bf16 throughput path within 16x (8x coarser mantissa, 21 layers) on the mean
                errors, and no decision may flip outside the error band of its own score.

Measured values: profiles/r02/parity.json (written when S4G_PARITY_REPORT is set), DESIGN.md §3 "Precision".

The golden `post/*` arrays of tests/golden/pn2cls_full_2638.npz (reference flow with both thresholds disabled) pin the
candidate count and the per-point scores; its `poses_s` pair point i with the rotation of the i-th best-scoring point
(the reference's indexing quirk, grasp_detector.py:153), a rank permutation that no reduced-precision forward can
reproduce — rotations are therefore compared per point, above.
"""
import json
import os

import numpy as np
import pytest
import torch

from tests import pose_parity

pytestmark = pytest.mark.gpu

N_SYNTH = 8
BOUNDS_SEEDED = {
    "tcgen05": {"score_abs_err_max": 5e-4, "score_abs_err_mean": 1e-4, "t_offset_err_mm_max": 0.05, "rot_err_deg_max": 1.0,
                "rot_err_deg_mean": 0.3, "translation_err_mm_max": 1.0, "translation_err_mm_mean": 0.2,
                "movable_abs_err_max": 1e-3, "logit_rel_err_max": 5e-3, "threshold_flip_frac": 0.0, "t_class_flip_frac": 1e-3},
    "tf32": {"score_abs_err_max": 1e-4, "score_abs_err_mean": 3e-5, "t_offset_err_mm_max": 0.01, "rot_err_deg_max": 0.15,
             "rot_err_deg_mean": 0.05, "translation_err_mm_max": 0.15, "translation_err_mm_mean": 0.03,
             "movable_abs_err_max": 2e-4, "logit_rel_err_max": 1e-3, "threshold_flip_frac": 0.0, "t_class_flip_frac": 1e-3},
}
# conditioned weights: bounds as multiples of the reference's own TF32 deviation (+ a small absolute floor)
MEAN_KEYS = {"score_abs_err_mean": 1e-4, "rot_err_deg_mean": 0.05, "translation_err_mm_mean": 0.05}
FLOOR_FACTOR = {"tf32": 2.0, "tcgen05": 16.0}
REFERENCE_TF32_FLOOR = os.path.join(os.path.dirname(__file__), "golden", "reference_tf32_floor.json")


@pytest.fixture(scope="module")
def scenes(cloud_2638):
    from tests.inputs import tabletop_scene
    return np.stack([cloud_2638] + [tabletop_scene(1000 + i, 25600) for i in range(N_SYNTH)])


@pytest.fixture(scope="module")
def nets(scenes):
    import bench
    from tests.conditioned import calibrate_batchnorm, conditioned_model
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    cond = calibrate_batchnorm(conditioned_model(seed=0).cuda(), torch.from_numpy(scenes[:2]).cuda())
    return {"seeded": bench.seeded_model().cuda(), "conditioned": cond}


@pytest.fixture(scope="module")
def oracle_out(scenes, nets):
    """fp32 CPU oracle forward (reference python modules restated bit-for-bit, tests/golden/make_golden.py)."""
    from oracle import model_cpu
    torch.set_num_threads(min(16, os.cpu_count()))
    out = {}
    with torch.no_grad():
        for name, net in nets.items():
            sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
            out[name] = []
            for s in scenes:
                o = model_cpu.pointnet2_forward(torch.from_numpy(s)[None], sd, model_cpu.PN2_CLS_CONFIG)
                out[name].append({k: v[0].numpy() for k, v in o.items()})
    return out


def _gpu_out(net, scenes, backend):
    from s4g_release_b200.engine import FusedPointNet2
    eng = FusedPointNet2(net.eval(), mlp_backend=backend)
    outs = []
    for s in scenes:  # one scene per call: the tf32 mode materialises grouped tensors
        o = eng.forward(torch.from_numpy(s)[None].cuda())
        torch.cuda.synchronize()
        outs.append({k: v[0].float().cpu().numpy() for k, v in o.items()})
    return outs


def _reference_tf32_out(net, scenes):
    """the UNMODIFIED reference model on its own CUDA kernels with torch's default cuDNN TF32 — None when not staged"""
    from baseline import stage_ref
    from oracle import build_ref
    from oracle.model_cpu import PN2_CLS_CONFIG
    if not stage_ref.available() or not os.path.exists(build_ref.so_path()):
        return None
    RefPointNet2 = stage_ref.import_reference_model(build_ref.load())
    model = RefPointNet2(**PN2_CLS_CONFIG)
    model.load_state_dict({k: v.detach().cpu() for k, v in net.state_dict().items()}, strict=True)
    model = model.cuda().eval()
    keep = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    outs = []
    with torch.no_grad():
        for s in scenes:
            o = model({"scene_points": torch.from_numpy(s)[None].cuda()})
            torch.cuda.synchronize()
            outs.append({k: v[0].float().cpu().numpy() for k, v in o.items()})
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = keep
    return outs


def _report(section, payload):
    path = os.environ.get("S4G_PARITY_REPORT")
    if not path:
        return
    os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
    prev = json.load(open(path)) if os.path.exists(path) else {}
    prev[section] = payload
    json.dump(prev, open(path, "w"), indent=1)


def _worst(scenes, want, got):
    return pose_parity.summarize([pose_parity.scene_metrics(scenes[i], want[i], got[i]) for i in range(len(scenes))])


@pytest.mark.parametrize("backend", ["tcgen05", "tf32"])
def test_seeded_weights_absolute_bounds(scenes, nets, oracle_out, backend):
    worst = _worst(scenes, oracle_out["seeded"], _gpu_out(nets["seeded"], scenes, backend))
    _report("seeded/" + backend, worst)
    print("seeded", backend, json.dumps(worst))
    bad = {k: (worst[k], b) for k, b in BOUNDS_SEEDED[backend].items() if not worst[k] <= b}
    assert not bad, "parity bounds exceeded (measured, bound): %r" % bad


def test_conditioned_weights_against_the_reference_tf32_yardstick(scenes, nets, oracle_out):
    want = oracle_out["conditioned"]
    ref_tf32 = _reference_tf32_out(nets["conditioned"], scenes)
    if ref_tf32 is None:  # the reference is not staged: its deviation as measured when it was (same scenes and weights)
        floor = json.load(open(REFERENCE_TF32_FLOOR))["worst"]
    else:
        floor = _worst(scenes, want, ref_tf32)
        _report("conditioned/reference_cudnn_tf32", floor)
    print("conditioned reference(TF32 default)", json.dumps(floor))
    n_above = min(int((pose_parity.expected_score(o["score"]) > 0.7).sum()) for o in want)
    assert n_above >= 200, "the conditioned weights must produce real candidates"
    for backend in ("tf32", "tcgen05"):
        worst = _worst(scenes, want, _gpu_out(nets["conditioned"], scenes, backend))
        _report("conditioned/" + backend, worst)
        print("conditioned", backend, json.dumps(worst))
        for key, eps in MEAN_KEYS.items():
            assert worst[key] <= FLOOR_FACTOR[backend] * floor[key] + eps, (backend, key, worst[key], floor[key])
        # decisions only flip inside the error band of the quantity they are taken on
        assert worst["threshold_flip_max_margin"] <= worst["score_abs_err_max"] + 1e-12
        assert worst["threshold_flip_frac"] <= 4.0 * worst["score_abs_err_mean"] / 0.1 + 1e-3, worst["threshold_flip_frac"]


def test_reference_flow_goldens_candidate_count_and_scores(cloud_2638, golden_full):
    """`post/n` and `post/scores_s` written by tests/golden/make_golden.py from the reference's post-processing flow
    (both thresholds disabled): the device post-processing of the fused forward keeps every point as a candidate and
    its expected scores agree with the golden to the score tolerance."""
    from s4g_release_b200.network_models.models.PointNet2_tcls import PN2_CLS_CONFIG, PointNet2
    from s4g_release_b200.postprocess import GraspPostProcessor
    from tests.golden.make_golden import seed_reference_weights
    torch.manual_seed(0)
    model = seed_reference_weights(PointNet2(**PN2_CLS_CONFIG)).cuda().eval()
    x = torch.from_numpy(cloud_2638)[None].cuda()
    with torch.no_grad():
        preds = model({"scene_points": x})
    res = GraspPostProcessor(max_candidates=25600).select_and_decode(x, preds, score_threshold=0.0,
                                                                     vertical_degree_threshold=-2.0)
    n = int(res["n"][0])
    assert n == int(golden_full["post/n"]) == 25600
    # with every point kept the candidates stay in cloud order (valid_index = arange), scores are per point
    order = res["point_index"][0, :n].long()
    assert torch.equal(order, torch.arange(n, device=order.device))
    got = res["scores"][0, :n:64].cpu().numpy()
    assert np.abs(got - golden_full["post/scores_s"]).max() <= BOUNDS_SEEDED["tcgen05"]["score_abs_err_max"]


def test_candidate_sets_through_both_post_processings(scenes, nets, oracle_out):
    """Both forwards through the post-processing at the reference's 0.7 threshold (verticalness filter open: it depends
    on the camera pose, not on the forward): the candidate point sets of the TF32 tight-parity mode and of the bf16 path
    against the oracle's — IoU reported; every disagreement lies within the score error band (checked above), so the
    IoU follows the density of points near the threshold on these sensitive weights (measured: 0.81-0.89 for TF32 — the
    reference's own TF32 default gives the same — and 0.3-0.6 for bf16); stated bounds: >= 0.7 (tf32), >= 0.25 (bf16)."""
    from oracle import model_cpu
    from s4g_release_b200.postprocess import GraspPostProcessor
    post = GraspPostProcessor(max_candidates=25600)
    report = {}
    for backend, bound in (("tf32", 0.7), ("tcgen05", 0.25)):
        got = _gpu_out(nets["conditioned"], scenes, backend)
        ious = []
        for i in range(len(scenes)):
            ref_pred = {k: torch.from_numpy(v)[None] for k, v in oracle_out["conditioned"][i].items()}
            _, _, ref_idx, _ = model_cpu.post_processing(scenes[i], ref_pred, 0.7, -2.0, return_index=True)
            dev_pred = {k: torch.from_numpy(v)[None].cuda() for k, v in got[i].items()}
            res = post.select_and_decode(torch.from_numpy(scenes[i])[None].cuda(), dev_pred, 0.7, -2.0)
            n = int(res["n"][0])
            dev_idx = set(res["point_index"][0, :n].cpu().tolist())
            ref_set = set(int(v) for v in ref_idx)
            ious.append(len(dev_idx & ref_set) / max(1, len(dev_idx | ref_set)))
        report[backend] = [round(v, 4) for v in ious]
        print("candidate-set IoU per scene (%s):" % backend, report[backend])
        assert min(ious) >= bound, (backend, ious)
    _report("conditioned/candidate_set_iou", report)
