"""Generate the golden fixtures under tests/golden/ from the REFERENCE's own python modules.

Run in the build container only (needs /root/reference; the GPU box has no copy):

    python tests/golden/make_golden.py

What it does
  1. injects oracle/pn2_ext_cpu.py (the C restatement of the CUDA-only ops) as
     ``grasp_proposal.network_models.models.pointnet2_utils.pn2_ext`` and imports the reference's
     unmodified ``PointNet2_tcls.PointNet2`` (+ modules.py, functions.py, nn_utils/*);
  2. runs it (eval, no_grad, torch-CPU fp32) on
       a. a tiny PN2_CLS-shaped configuration (state_dict stored in the fixture), and
       b. BASELINE config 1: inference/2638_view_0.p, RandomState(0) subsample to 25 600 points, the
          shipped curvature_model.yaml architecture with seeded weights (SURVEY.md §8d);
  3. checks that oracle/model_cpu.py (the functional restatement the GPU tests use as checker)
     reproduces the reference modules' outputs BIT-FOR-BIT on both, and that the product model class
     initialises to an identical state_dict under the same seed;
  4. writes the fixtures.

The ops inside are the C restatement, so these fixtures pin the *python layer* of the oracle
(modules / model / post-process maths).  The ops themselves are pinned against the reference's CUDA
kernels by tests/test_ref_cuda_parity.py (three-way, on the GPU box).
"""
import hashlib
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference/inference"
sys.path.insert(0, ROOT)

from oracle import model_cpu, pn2_ext_cpu  # noqa: E402
from tests.inputs import TINY_CONFIG  # noqa: E402


def import_reference():
    sys.path.insert(0, REF)
    name = "grasp_proposal.network_models.models.pointnet2_utils.pn2_ext"
    mod = types.ModuleType(name)
    for fn in ("farthest_point_sample", "ball_query", "group_points_forward", "group_points_backward",
               "point_search", "interpolate_forward", "interpolate_backward"):
        setattr(mod, fn, getattr(pn2_ext_cpu, fn))
    sys.modules[name] = mod
    import grasp_proposal.network_models.models.pointnet2_utils as pkg
    pkg.pn2_ext = mod
    from grasp_proposal.network_models.models.PointNet2_tcls import PointNet2
    return PointNet2


def seed_reference_weights(model):
    """SURVEY.md §8d config 1: default init under torch.manual_seed(0) happened at construction;
    every BatchNorm then gets non-trivial affine + running statistics from Generator(1)."""
    g = torch.Generator().manual_seed(1)
    for m in model.modules():
        if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
            n = m.num_features
            m.weight.data = torch.rand(n, generator=g) + 0.5
            m.bias.data = torch.randn(n, generator=g) * 0.1
            m.running_mean.data = torch.randn(n, generator=g) * 0.1
            m.running_var.data = torch.rand(n, generator=g) + 0.5
    return model




def sha(t):
    return hashlib.sha256(np.ascontiguousarray(t.numpy() if torch.is_tensor(t) else t).tobytes()).hexdigest()


def array_digest(t):
    """SHA-256 over dtype, shape and bytes: how a fixture stores seeded weights that its test rebuilds."""
    a = np.ascontiguousarray(t.numpy() if torch.is_tensor(t) else t)
    return hashlib.sha256(("%s %s " % (a.dtype, a.shape)).encode() + a.tobytes()).hexdigest()


def run_pair(PointNet2, cfg, points):
    torch.manual_seed(0)
    ref_model = seed_reference_weights(PointNet2(**cfg)).eval()
    with torch.no_grad():
        ref_out = ref_model({"scene_points": points})
    sd = ref_model.state_dict()
    trace = {}
    with torch.no_grad():
        my_out = model_cpu.pointnet2_forward(points, sd, cfg, trace)
    for k in ref_out:
        assert torch.equal(ref_out[k], my_out[k]), f"oracle/model_cpu.py differs from the reference modules on {k}"
    return ref_model, sd, ref_out, trace


def main():
    PointNet2 = import_reference()
    torch.set_num_threads(os.cpu_count())

    # ---- (a) tiny configuration --------------------------------------------------------------
    rs = np.random.RandomState(7)
    pts = rs.rand(2, 3, 1024).astype(np.float32)
    pts[:, 2] *= 0.2
    points = torch.from_numpy(pts)
    _, sd, out, trace = run_pair(PointNet2, TINY_CONFIG, points)
    fix = {"points": pts}
    for k, v in sd.items():
        fix["sd/" + k] = v.numpy()
    for k, v in out.items():
        fix["out/" + k] = v.numpy()
    for i, t in enumerate(trace["sa"]):
        fix[f"sa{i}/fps_index"] = t["fps_index"].numpy().astype(np.int32)
        fix[f"sa{i}/ball_index"] = t["ball_index"].numpy().astype(np.int32)
        fix[f"sa{i}/ball_count"] = t["ball_count"].numpy().astype(np.int32)
        fix[f"sa{i}/new_feature"] = t["new_feature"].numpy()
    for i, t in enumerate(trace["fp"]):
        fix[f"fp{i}/nn_index"] = t["nn_index"].numpy().astype(np.int32)
        fix[f"fp{i}/nn_dist"] = t["nn_dist"].numpy()
        fix[f"fp{i}/fp_feature"] = t["fp_feature"].numpy()
    np.savez_compressed(os.path.join(HERE, "pn2cls_tiny.npz"), **fix)
    print("tiny: ok,", len(fix), "arrays")

    # ---- (b) BASELINE config 1: the shipped fixture, full architecture -------------------------
    pc = np.load(os.path.join(REF, "2638_view_0.p"), allow_pickle=True)["point_cloud"]
    assert pc.shape == (3, 48902) and pc.dtype == np.float32
    sel = np.random.RandomState(0).choice(pc.shape[1], model_cpu.NUM_INPUT, replace=False)
    cloud = np.ascontiguousarray(pc[:, sel])
    np.save(os.path.join(HERE, "cloud_2638_view0_25600.npy"), cloud)
    points = torch.from_numpy(cloud)[None]
    ref_model, sd, out, trace = run_pair(PointNet2, model_cpu.PN2_CLS_CONFIG, points)

    # the product model must initialise identically under the same seed (tests rely on it)
    try:
        from s4g_release_b200.network_models.models.PointNet2_tcls import PointNet2 as MyPointNet2
        torch.manual_seed(0)
        mine = seed_reference_weights(MyPointNet2(**model_cpu.PN2_CLS_CONFIG))
        msd = mine.state_dict()
        assert list(msd.keys()) == list(sd.keys()), "state_dict key order differs"
        for k in sd:
            assert torch.equal(sd[k], msd[k]), f"seeded init differs at {k}"
        print("product model: identical seeded state_dict (%d entries)" % len(sd))
    except ImportError as e:  # product package not built yet
        print("product model check skipped:", e)

    poses, scores = model_cpu.post_processing(cloud, out, score_threshold=0.0, vertical_degree_threshold=-2.0)
    stride = 16
    fix = {"stride": np.int32(stride), "n_params": np.int64(sum(p.numel() for p in ref_model.parameters()))}
    for k, v in out.items():
        fix["out/" + k] = v.numpy()[:, :, ::stride].copy()
        fix["sha/" + k] = np.frombuffer(bytes.fromhex(sha(v)), dtype=np.uint8)
    for i, t in enumerate(trace["sa"]):
        fix[f"sa{i}/fps_index"] = t["fps_index"].numpy().astype(np.int32)
        fix[f"sa{i}/ball_count"] = t["ball_count"].numpy().astype(np.int16)
        fix[f"sa{i}/ball_index_sha"] = np.frombuffer(bytes.fromhex(sha(t["ball_index"])), dtype=np.uint8)
        fix[f"sa{i}/ball_index_sum"] = t["ball_index"].sum(dim=2).numpy().astype(np.int64)
        fix[f"sa{i}/new_feature_s"] = t["new_feature"].numpy()[:, ::8, ::8].copy()
    for i, t in enumerate(trace["fp"]):
        fix[f"fp{i}/nn_index_sha"] = np.frombuffer(bytes.fromhex(sha(t["nn_index"])), dtype=np.uint8)
        fix[f"fp{i}/nn_index_s"] = t["nn_index"].numpy()[:, ::stride].astype(np.int32)
        fix[f"fp{i}/nn_dist_s"] = t["nn_dist"].numpy()[:, ::stride].copy()
    fix["post/poses_s"] = poses[::64].copy()
    fix["post/scores_s"] = scores[::64].copy()
    fix["post/n"] = np.int64(poses.shape[0])
    np.savez_compressed(os.path.join(HERE, "pn2cls_full_2638.npz"), **fix)
    print("full: ok; params", int(fix["n_params"]), "state_dict entries", len(sd))


if __name__ == "__main__":
    main()
