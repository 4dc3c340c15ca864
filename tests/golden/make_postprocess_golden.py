"""Pins oracle/model_cpu.py's post-processing restatements against the REFERENCE'S OWN CODE, executed in the build
container: the method bodies are cut out of /root/reference (grasp_detector.py needs open3d / yacs at import time,
so the module cannot be imported; the functions themselves only need numpy / torch) and run on seeded inputs.
Writes tests/golden/postprocess_ref.npz.   python tests/golden/make_postprocess_golden.py
"""
import ast
import os
import sys
import textwrap
import types

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = "/root/reference/inference/grasp_proposal"
# torch's CPU softmax rounds the last bit of some elements differently with the number of threads that share the work:
# the golden is written, and tests/test_oracle_cpu.py checks it, with this many
TORCH_THREADS = 8


def cut(path, cls, names):
    """Source of the named functions (methods of `cls`, or module level when cls is None), dedented."""
    src = open(path).read()
    tree = ast.parse(src)
    body = tree.body
    if cls:
        body = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == cls).body
    out = {}
    for n in body:
        if isinstance(n, ast.FunctionDef) and n.name in names:
            seg = ast.get_source_segment(src, n)
            lines = src.splitlines()[n.lineno - 1 - len(n.decorator_list): n.end_lineno]
            out[n.name] = textwrap.dedent("\n".join(l for l in lines if not l.strip().startswith("@")))
            del seg
    return out


def main():
    from oracle import model_cpu
    torch.set_num_threads(TORCH_THREADS)
    gd = cut(os.path.join(REF, "grasp_detector.py"), "GraspDetector", {"orthogonalization", "post_processing"})
    cc = cut(os.path.join(REF, "cloud_processor", "view_collision_checker.py"), "CloudCollisionChecker", {"view_non_collision"})
    mu = cut(os.path.join(REF, "utils", "math_utils.py"), None, {"torch_batch_transformation_inv"})

    # --- environment the cut functions expect (values restated from the reference's config files) ---
    realworld = types.SimpleNamespace(camera2base=model_cpu.CAMERA2BASE)
    config = types.SimpleNamespace(FINGER_LENGTH=0.09, BOTTOM_LENGTH=0.16, HALF_HAND_THICKNESS=0.012,
                                   HALF_BOTTOM_WIDTH=0.057, HALF_BOTTOM_SPACE=0.057 - 0.023)
    ns = {"np": np, "torch": torch, "F": F, "os": os, "realworld": realworld, "config": config,
          "BACK_COLLISION_MARGIN": 0.0, "BACK_COLLISION_THRESHOLD": 10 * np.sqrt(8), "FINGER_COLLISION_THRESHOLD": 10,
          "Optional": None}
    for src in list(gd.values()) + list(cc.values()) + list(mu.values()):
        exec(src, ns)
    fake_self = types.SimpleNamespace(_TRAIN2REAL=np.linalg.inv(model_cpu.REAL2TRAIN),
                                      vertical_direction=np.array([[0, 0, 1]], dtype=np.float32), _output_path="/tmp")
    fake_self.orthogonalization = ns["orthogonalization"]

    rs = np.random.RandomState(7)
    n = 4000
    preds = {"score": torch.from_numpy(rs.randn(1, 3, n).astype(np.float32) * 2),
             "frame_R": torch.from_numpy(rs.randn(1, 9, n).astype(np.float32)),
             "frame_t": torch.from_numpy(rs.randn(1, 4, n).astype(np.float32))}
    pts = (rs.rand(3, n) * 0.4 - 0.2).astype(np.float32)
    pts[2] -= 1.0
    fix = {"score": preds["score"].numpy(), "frame_R": preds["frame_R"].numpy(), "frame_t": preds["frame_t"].numpy(),
           "points": pts}
    for tag, (thr, vthr) in {"a": (0.7, 0.2), "b": (0.5, -2.0)}.items():
        poses, scores = ns["post_processing"](fake_self, pts, preds, thr, vthr, False)
        mine_p, mine_s = model_cpu.post_processing(pts, preds, thr, vthr)
        assert np.array_equal(poses, mine_p) and np.array_equal(scores, mine_s), "oracle != reference post_processing"
        fix[f"post_{tag}/thr"] = np.array([thr, vthr])
        fix[f"post_{tag}/poses"] = poses
        fix[f"post_{tag}/scores"] = scores
        print("post_processing %s: %d poses, oracle bit-identical to the reference code" % (tag, poses.shape[0]))

    # --- collision check: reference method on a fake self with the same attributes it builds in __init__ ---
    plane = np.stack([rs.uniform(-0.3, 0.3, 5000), rs.uniform(-0.3, 0.3, 5000), np.full(5000, -1.0)], 1)
    box = np.stack([rs.uniform(-0.03, 0.03, 2000), rs.uniform(-0.02, 0.02, 2000), rs.uniform(-1.0, -0.9, 2000)], 1)
    cloud = np.concatenate([plane, box]).astype(np.float32)
    ct = torch.tensor(cloud).float()
    checker = types.SimpleNamespace(cloud_array=ct, cloud_array_homo=torch.cat([ct.transpose(0, 1), torch.ones(1, ct.shape[0])], 0))
    m = 120
    poses = np.tile(np.eye(4), (m, 1, 1))
    for i in range(m):
        q, _ = np.linalg.qr(rs.randn(3, 3))
        q *= np.sign(np.linalg.det(q))
        poses[i, :3, :3] = q
        poses[i, :3, 3] = [rs.uniform(-0.1, 0.1), rs.uniform(-0.1, 0.1), rs.uniform(-1.05, -0.8)]
    inv = ns["torch_batch_transformation_inv"](torch.tensor(poses, dtype=torch.float32))
    ok = np.array([bool(ns["view_non_collision"](checker, inv[i])) for i in range(m)])
    mine_ok, _ = model_cpu.collision_filter(poses, cloud)
    mask = np.zeros(m, dtype=bool)
    mask[mine_ok] = True
    assert np.array_equal(ok, mask), "oracle != reference view_non_collision"
    assert torch.equal(inv, model_cpu.batch_transformation_inv(poses))
    fix["coll/cloud"] = cloud
    fix["coll/poses"] = poses
    fix["coll/ok"] = ok
    print("collision: %d / %d grasps free, oracle identical to the reference code" % (ok.sum(), m))

    # --- importance sampling: the inline block of GraspDetector.detect (grasp_detector.py:237-246) ---
    src = open(os.path.join(REF, "grasp_detector.py")).read().splitlines()
    start = next(i for i, l in enumerate(src) if "scores_cum = np.cumsum" in l)
    end = next(i for i, l in enumerate(src) if "sampling_indices = np.array(sampling_indices)" in l)
    block = textwrap.dedent("\n".join(l for l in src[start:end + 1] if "np.random.rand" not in l))
    scores = rs.uniform(0.7, 1.0, 300)
    u = np.sort(rs.rand(5))
    env = {"np": np, "scores": scores, "num_selected": 5}
    block = block.replace("scores_cum = np.cumsum(np.exp(5 * scores))",
                          "scores_cum = np.cumsum(np.exp(5 * scores))\nrandom_score = U * scores_cum[-1]")
    env["U"] = u
    exec(block, env)
    assert np.array_equal(env["sampling_indices"], model_cpu.importance_sampling(scores, u))
    fix["samp/scores"] = scores
    fix["samp/u"] = u
    fix["samp/picked"] = env["sampling_indices"]
    print("importance sampling: oracle identical to the reference code")
    np.savez_compressed(os.path.join(HERE, "postprocess_ref.npz"), **fix)


if __name__ == "__main__":
    main()
