"""CPU suite: the oracle (C restatement + python model restatement) against the golden fixtures that
tests/golden/make_golden.py produced from the reference's own python modules, and the closed-form FPS
tie rule against the literal simulation of the reference's block reduction."""
import numpy as np
import pytest
import torch

from tests import inputs
from oracle import model_cpu
from oracle import pn2_ext_cpu as ops
from tests.inputs import TINY_CONFIG


def _sd(golden):
    return {k[3:]: torch.from_numpy(v) for k, v in golden.items() if k.startswith("sd/")}


def test_ops_reproduce_tiny_golden(golden_tiny):
    g = golden_tiny
    pts = torch.from_numpy(g["points"])
    xyz = pts
    for i in range(3):
        idx = ops.farthest_point_sample(xyz, TINY_CONFIG["num_centroids"][i])
        assert np.array_equal(idx.numpy(), g[f"sa{i}/fps_index"])
        new_xyz = ops.gather_points(xyz, idx)
        nbr, cnt = ops.ball_query(xyz, new_xyz, TINY_CONFIG["radius"][i], TINY_CONFIG["num_neighbours"][i])
        assert np.array_equal(nbr.numpy(), g[f"sa{i}/ball_index"])
        assert np.array_equal(cnt.numpy(), g[f"sa{i}/ball_count"])
        xyz = new_xyz


def test_model_reproduces_tiny_golden(golden_tiny):
    g = golden_tiny
    trace = {}
    with torch.no_grad():
        out = model_cpu.pointnet2_forward(torch.from_numpy(g["points"]), _sd(g), TINY_CONFIG, trace)
    for k in ("score", "frame_R", "frame_t", "movable_logits"):
        np.testing.assert_allclose(out[k].numpy(), g["out/" + k], rtol=1e-4, atol=1e-5)
    for i, t in enumerate(trace["fp"]):
        assert np.array_equal(t["nn_index"].numpy(), g[f"fp{i}/nn_index"])
        np.testing.assert_array_equal(t["nn_dist"].numpy(), g[f"fp{i}/nn_dist"])


def test_fps_and_ball_query_on_fixture_cloud(cloud_2638, golden_full):
    """BASELINE config 1 geometry: bit-exact indices on the shipped fixture's 25 600-point subsample."""
    g = golden_full
    xyz = torch.from_numpy(cloud_2638)[None]
    cfg = model_cpu.PN2_CLS_CONFIG
    for i in range(3):
        idx = ops.farthest_point_sample(xyz, cfg["num_centroids"][i])
        assert np.array_equal(idx.numpy(), g[f"sa{i}/fps_index"])
        new_xyz = ops.gather_points(xyz, idx)
        nbr, cnt = ops.ball_query(xyz, new_xyz, cfg["radius"][i], cfg["num_neighbours"][i])
        assert np.array_equal(cnt.numpy(), g[f"sa{i}/ball_count"])
        assert np.array_equal(nbr.sum(dim=2).numpy(), g[f"sa{i}/ball_index_sum"])
        xyz = new_xyz


@pytest.mark.parametrize("gen,N,M", [
    ("lattice", 2000, 600), ("lattice", 700, 700), ("lattice", 200, 150), ("lattice", 40, 40), ("lattice", 13, 9),
    ("dup", 3000, 1500), ("identical", 600, 50), ("uniform", 5120, 1024), ("lattice", 513, 300),
])
def test_fps_tie_rule_closed_form(gen, N, M):
    """The key order (distance desc, bitreverse(j mod BLOCK) asc, j asc) — what the sm_100a kernel
    implements — equals the literal simulation of sampling_kernel.cu:61-118 on tie-heavy inputs."""
    pts = {"lattice": lambda: inputs.lattice_cloud(3, N, N, side=6), "dup": lambda: inputs.duplicated_cloud(3, N, N),
           "identical": lambda: inputs.identical_cloud(2, N), "uniform": lambda: inputs.uniform_cloud(2, N, N)}[gen]()
    a = ops.farthest_point_sample(pts, M)
    b = ops.farthest_point_sample(pts, M, keyed=True)
    assert torch.equal(a, b)
    if gen == "lattice":
        # the rule is NOT "lowest index wins": make sure the input actually exercises ties
        d = (pts[:, :, :, None] - pts[:, :, None, :]).pow(2).sum(1)
        assert (d == d[:, :1, 1:2]).sum() > 4


def test_ball_query_padding_rules():
    pts = inputs.uniform_cloud(2, 500, 3)
    ctr = pts[:, :, ::7].contiguous()
    idx, cnt = ops.ball_query(pts, ctr, 1e-4, 16)  # only the centroid itself (or nothing) is inside
    d2 = ((pts[:, :, None, :] - ctr[:, :, :, None]) ** 2).sum(1)
    for b in range(2):
        for m in range(ctr.shape[2]):
            hits = torch.nonzero(d2[b, m] < np.float32(1e-4) ** 2).flatten()[:16]
            assert cnt[b, m] == len(hits)
            if len(hits) == 0:
                assert (idx[b, m] == 0).all()
            else:
                assert torch.equal(idx[b, m, :len(hits)], hits)
                assert (idx[b, m, len(hits):] == hits[0]).all()
    far = pts + 10.0
    idx, cnt = ops.ball_query(pts, far[:, :, :5].contiguous(), 0.1, 8)
    assert (idx == 0).all() and (cnt == 0).all()


def test_point_search_is_stable_three_smallest():
    q = inputs.lattice_cloud(2, 300, 11, side=4)
    k = inputs.lattice_cloud(2, 64, 12, side=4)
    idx, d2 = ops.point_search(q, k, 3)
    full = ((q[:, :, :, None] - k[:, :, None, :]) ** 2)
    full = torch.from_numpy(np.float32(1) * 0 + (full[:, 0].numpy() + full[:, 1].numpy()) + full[:, 2].numpy())
    ref_d, ref_i = torch.sort(full, dim=2, stable=True)
    # lattice coordinates make every product exact, so the fma order cannot matter here
    assert torch.equal(idx, ref_i[:, :, :3])
    assert torch.equal(d2, ref_d[:, :, :3])
    with pytest.raises(RuntimeError):
        ops.point_search(q, k[:, :, :2].contiguous(), 3)
    with pytest.raises(RuntimeError):
        ops.point_search(q, k, 2)


def test_group_and_interpolate_adjoints():
    rs = np.random.RandomState(0)
    B, C, N, M, K = 2, 5, 40, 9, 4
    x = torch.from_numpy(rs.randn(B, C, N).astype(np.float32))
    idx = torch.from_numpy(rs.randint(0, N, size=(B, M, K)).astype(np.int64))
    y = ops.group_points_forward(x, idx)
    assert torch.equal(y, torch.gather(x[:, :, None, :].expand(B, C, M, N), 3, idx[:, None].expand(B, C, M, K)))
    g = torch.from_numpy(rs.randn(B, C, M, K).astype(np.float32))
    gx = ops.group_points_backward(g, idx, N)
    np.testing.assert_allclose((gx * x).sum().item(), (g * y).sum().item(), rtol=1e-4)
    idx3 = torch.from_numpy(rs.randint(0, N, size=(B, M, 3)).astype(np.int64))
    w = torch.from_numpy(rs.rand(B, M, 3).astype(np.float32))
    z = ops.interpolate_forward(x, idx3, w)
    g2 = torch.from_numpy(rs.randn(B, C, M).astype(np.float32))
    gx2 = ops.interpolate_backward(g2, idx3, w, N)
    np.testing.assert_allclose((gx2 * x).sum().item(), (g2 * z).sum().item(), rtol=1e-4)


def test_post_processing_invariants():
    """grasp_detector.py:137-185 restated: thresholding, orthonormal rotations, homogeneous rows."""
    rs = np.random.RandomState(5)
    n = 2000
    preds = {"score": torch.from_numpy(rs.randn(1, 3, n).astype(np.float32) * 3),
             "frame_R": torch.from_numpy(rs.randn(1, 9, n).astype(np.float32)),
             "frame_t": torch.from_numpy(rs.randn(1, 4, n).astype(np.float32))}
    pts = rs.randn(3, n).astype(np.float32)
    poses, scores = model_cpu.post_processing(pts, preds, 0.5, -2.0)
    assert poses.shape[0] == scores.shape[0] > 0
    assert (scores > 0.5).all()
    R = poses[:, :3, :3]
    RtR = np.einsum("nij,nik->njk", R, R)
    np.testing.assert_allclose(RtR, np.tile(np.eye(3), (R.shape[0], 1, 1)), atol=1e-5)
    assert np.allclose(poses[:, 3], [0, 0, 0, 1])


def test_post_processing_pinned_to_reference_code():
    """oracle/model_cpu.py vs outputs of the reference's OWN post_processing / view_non_collision / importance
    sampling code (cut out of the reference project's source by tests/golden/make_postprocess_golden.py).  Torch's CPU
    softmax rounds the last bit of some elements differently with the number of threads that share the work, so the
    oracle runs with the thread count the golden was written with."""
    import os
    from tests.golden.make_postprocess_golden import TORCH_THREADS
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "postprocess_ref.npz"))
    preds = {k: torch.from_numpy(g[k]) for k in ("score", "frame_R", "frame_t")}
    threads = torch.get_num_threads()
    torch.set_num_threads(TORCH_THREADS)
    try:
        for tag in ("a", "b"):
            thr, vthr = g[f"post_{tag}/thr"]
            poses, scores = model_cpu.post_processing(g["points"], preds, float(thr), float(vthr))
            assert np.array_equal(poses, g[f"post_{tag}/poses"]) and np.array_equal(scores, g[f"post_{tag}/scores"])
    finally:
        torch.set_num_threads(threads)
    ok, _ = model_cpu.collision_filter(g["coll/poses"], g["coll/cloud"])
    assert np.array_equal(ok, np.nonzero(g["coll/ok"])[0])
    assert np.array_equal(model_cpu.importance_sampling(g["samp/scores"], g["samp/u"]), g["samp/picked"])


@pytest.mark.parametrize("kind,N,M", [("lattice", 700, 300), ("dup", 900, 400), ("identical", 100, 20), ("uniform", 1500, 200)])
def test_fp64_oracle_fps_tie_rule(kind, N, M):
    """the double instantiation (sampling_kernel.cu:21 dispatches float and double): closed-form tie rule == literal
    block simulation, and on fp32-representable inputs the double FPS of a lattice picks the same points as fp32
    (all distances exact in both)."""
    from oracle import pn2_ext_cpu as o
    gen = {"lattice": lambda: inputs.lattice_cloud(2, N, 3, side=8), "dup": lambda: inputs.duplicated_cloud(2, N, 3),
           "identical": lambda: inputs.identical_cloud(2, N), "uniform": lambda: inputs.uniform_cloud(2, N, 3)}[kind]
    p32 = gen()
    p64 = p32.double()
    lit = o.farthest_point_sample(p64, M)
    assert torch.equal(o.farthest_point_sample(p64, M, keyed=True), lit)
    if kind in ("lattice", "identical"):
        assert torch.equal(o.farthest_point_sample(p32, M), lit)


def test_fp64_oracle_ops_match_torch():
    from oracle import pn2_ext_cpu as o
    rs = np.random.RandomState(5)
    p = torch.from_numpy(rs.rand(2, 3, 400))
    c = o.gather_points(p, o.farthest_point_sample(p, 40))
    idx, cnt = o.ball_query(p, c, 0.2, 16)
    d = ((p[:, :, None, :] - c[:, :, :, None]) ** 2).sum(1)  # (B,M,N)
    r2 = float(np.float32(0.2)) ** 2
    assert torch.equal(cnt, (d < r2).sum(-1).clamp(max=16))
    nn_i, nn_d = o.point_search(p, c, 3)
    top = torch.topk(((p[:, :, :, None] - c[:, :, None, :]) ** 2).sum(1), 3, dim=-1, largest=False)
    assert torch.equal(nn_i, top.indices)
    np.testing.assert_allclose(nn_d.numpy(), top.values.numpy(), rtol=1e-13, atol=1e-15)
    f = torch.from_numpy(rs.randn(2, 7, 40))
    w = torch.from_numpy(rs.rand(2, 400, 3))
    out = o.interpolate_forward(f, nn_i, w)
    ref = (torch.gather(f[:, :, None, :].expand(-1, -1, 400, -1), 3, nn_i[:, None].expand(-1, 7, -1, -1)) * w[:, None]).sum(-1)
    np.testing.assert_allclose(out.numpy(), ref.numpy(), rtol=1e-13, atol=1e-14)
    g = o.group_points_forward(f, idx.clamp(max=39))
    assert g.dtype == torch.float64 and g.shape == (2, 7, 40, 16)


def test_preprocess_oracle_pinned_to_reference_golden():
    """oracle/model_cpu.py::pre_processing == the reference's own transform_numpy_points + sample_single_cloud
    replay (tests/golden/preprocess_ref.npz, made by tests/golden/make_preprocess_golden.py); the seeded index draw is
    reproduced too."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "preprocess_ref.npz"))
    for name in ("large", "small"):
        cloud, index = g[name + "/cloud"], g[name + "/index"]
        assert np.array_equal(model_cpu.pre_processing(cloud, index), g[name + "/points_f32"])
        rs = np.random.RandomState(17)
        n, m = cloud.shape[1], len(index)
        assert np.array_equal(rs.choice(np.arange(n), m, replace=not (n > m)), index)
