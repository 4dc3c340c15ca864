"""GPU parity suite: every pn2_ext replacement (through the C ABI) against the oracle on the same seeded
inputs — bit-exact for indices / gathers, including the reference's tie-breaking and padding rules —
plus size-independent properties at BASELINE sizes where the oracle would take too long."""
import numpy as np
import pytest
import torch

from tests import inputs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ext():
    from s4g_release_b200.network_models.models.pointnet2_utils import pn2_ext
    return pn2_ext


@pytest.fixture(scope="module")
def ora():
    from oracle import pn2_ext_cpu
    return pn2_ext_cpu


FPS_CASES = [
    # (generator, B, N, M)
    ("uniform", 2, 1024, 256), ("uniform", 3, 5120, 1024), ("uniform", 1, 25600, 5120), ("uniform", 4, 1000, 1000),
    ("uniform", 2, 777, 300), ("uniform", 2, 13, 13), ("uniform", 5, 1, 1), ("uniform", 2, 17, 5),
    ("uniform", 2, 256, 100), ("uniform", 2, 257, 100), ("uniform", 1, 12801, 700), ("uniform", 70, 3000, 64),
    ("lattice", 3, 2000, 600), ("lattice", 2, 700, 700), ("lattice", 2, 200, 150), ("lattice", 2, 40, 40),
    ("lattice", 2, 30000, 2000), ("dup", 2, 3000, 1500), ("dup", 1, 26000, 3000), ("identical", 2, 600, 50),
    ("uniform", 1, 60000, 512), ("lattice", 1, 100000, 600),
    # batches that fill the GPU: two clouds interleaved per cluster (odd batches leave a cluster one cloud)
    ("lattice", 75, 2048, 200), ("dup", 39, 5120, 300), ("uniform", 65, 25600, 80), ("identical", 41, 4000, 20),
]


def _gen(kind, B, N, seed):
    return {"uniform": lambda: inputs.uniform_cloud(B, N, seed), "lattice": lambda: inputs.lattice_cloud(B, N, seed, side=8),
            "dup": lambda: inputs.duplicated_cloud(B, N, seed), "identical": lambda: inputs.identical_cloud(B, N)}[kind]()


@pytest.mark.parametrize("kind,B,N,M", FPS_CASES)
def test_fps_bit_exact(ext, ora, kind, B, N, M):
    pts = _gen(kind, B, N, seed=N + M)
    want = ora.farthest_point_sample(pts, M)
    got = ext.farthest_point_sample(pts.cuda(), M)
    assert got.dtype == torch.int64 and tuple(got.shape) == (B, M)
    assert torch.equal(got.cpu(), want)


def test_fps_fixture_cloud_golden(ext, cloud_2638, golden_full):
    xyz = torch.from_numpy(cloud_2638)[None].cuda()
    for i, m in enumerate((5120, 1024, 256)):
        idx = ext.farthest_point_sample(xyz, m)
        assert np.array_equal(idx.cpu().numpy(), golden_full[f"sa{i}/fps_index"])
        xyz = torch.gather(xyz, 2, idx.unsqueeze(1).expand(-1, 3, -1)).contiguous()


def test_fps_noncontiguous_and_errors(ext, ora):
    base = inputs.uniform_cloud(2, 900, 5)
    nc = base.transpose(1, 2).contiguous().transpose(1, 2)  # (B,3,N) view of a (B,N,3) buffer
    assert not nc.is_contiguous()
    assert torch.equal(ext.farthest_point_sample(nc.cuda(), 100).cpu(), ora.farthest_point_sample(base, 100))
    with pytest.raises(RuntimeError):
        ext.farthest_point_sample(base.cuda(), 901)
    with pytest.raises(RuntimeError):
        ext.farthest_point_sample(base.cuda(), 0)
    with pytest.raises(RuntimeError):
        ext.farthest_point_sample(base[:, :2].cuda(), 10)
    with pytest.raises(RuntimeError):
        ext.farthest_point_sample(base.half().cuda(), 10)  # float32 / float64 only, like AT_DISPATCH_FLOATING_TYPES


def test_fps_full_batch_properties(ext):
    """B = 64 x 25 600 -> 5 120 (BASELINE config 2 shape): properties that do not need the oracle."""
    pts = inputs.tabletop_batch(64).cuda()
    idx = ext.farthest_point_sample(pts, 5120)
    assert (idx[:, 0] == 0).all()
    sel = torch.gather(pts, 2, idx.unsqueeze(1).expand(-1, 3, -1))
    # the distance of each new sample to the already-selected set never increases
    for b in (0, 17, 63):
        s = sel[b].t().double()
        d = torch.cdist(s[:600], s[:600])
        far = torch.stack([d[i, :i].min() for i in range(1, 600)])
        assert (far[1:] <= far[:-1] + 1e-12).all()
    # and a cloud processed alone gives the same answer as inside the batch
    assert torch.equal(ext.farthest_point_sample(pts[5:6].contiguous(), 5120), idx[5:6])


BQ_CASES = [
    ("uniform", 2, 1024, 256, 0.1, 16), ("uniform", 2, 5120, 1024, 0.08, 64), ("uniform", 1, 25600, 700, 0.02, 64),
    ("uniform", 3, 777, 333, 0.2, 7), ("uniform", 2, 100, 100, 0.5, 128), ("uniform", 2, 50, 3, 1e-4, 8),
    ("lattice", 2, 2000, 500, 0.125, 32), ("lattice", 2, 2000, 500, 0.25, 64), ("dup", 2, 3000, 400, 0.05, 32),
    ("identical", 2, 300, 20, 0.1, 16), ("uniform", 2, 33, 33, 10.0, 40), ("uniform", 1, 4099, 517, 0.07, 33),
    # linear-scan kernel (N < 8192) on ties, duplicates, identical points, huge / tiny radii; the 20000-point case runs
    # the grid kernel (N >= 8192), whose edge cases are in test_geometry_edges_gpu.py
    ("lattice", 2, 6000, 700, 0.125, 32), ("lattice", 2, 6000, 300, 0.3, 64), ("dup", 2, 8000, 900, 0.05, 32),
    ("identical", 2, 5000, 40, 0.1, 16), ("uniform", 2, 5000, 300, 10.0, 128), ("uniform", 2, 5000, 300, 1e-4, 8),
    ("uniform", 1, 20000, 1000, 0.05, 200), ("uniform", 3, 4096, 512, 0.11, 64),
]


@pytest.mark.parametrize("kind,B,N,M,r,K", BQ_CASES)
def test_ball_query_bit_exact(ext, ora, kind, B, N, M, r, K):
    pts = _gen(kind, B, N, seed=N + K)
    sel = ora.farthest_point_sample(pts, M)
    ctr = ora.gather_points(pts, sel)
    want_idx, want_cnt = ora.ball_query(pts, ctr, r, K)
    got_idx, got_cnt = ext.ball_query(pts.cuda(), ctr.cuda(), r, K)
    assert got_idx.dtype == torch.int64 and got_cnt.dtype == torch.int64
    assert torch.equal(got_cnt.cpu(), want_cnt)
    assert torch.equal(got_idx.cpu(), want_idx)


@pytest.mark.parametrize("n", [500, 6000])
def test_ball_query_no_hits_and_far_centroids(ext, ora, n):
    pts = inputs.uniform_cloud(2, n, 3)
    far = (pts[:, :, :37] + 10.0).contiguous()
    idx, cnt = ext.ball_query(pts.cuda(), far.cuda(), 0.1, 8)
    assert (idx == 0).all() and (cnt == 0).all()
    mixed = torch.cat([far[:, :, :5], pts[:, :, :6]], dim=2).contiguous()
    w_idx, w_cnt = ora.ball_query(pts, mixed, 0.05, 12)
    g_idx, g_cnt = ext.ball_query(pts.cuda(), mixed.cuda(), 0.05, 12)
    assert torch.equal(g_idx.cpu(), w_idx) and torch.equal(g_cnt.cpu(), w_cnt)


def test_ball_query_fixture_cloud_golden(ext, cloud_2638, golden_full):
    xyz = torch.from_numpy(cloud_2638)[None].cuda()
    for i, (m, r) in enumerate(((5120, 0.02), (1024, 0.08), (256, 0.32))):
        sel = torch.from_numpy(golden_full[f"sa{i}/fps_index"]).long().cuda()
        ctr = torch.gather(xyz, 2, sel.unsqueeze(1).expand(-1, 3, -1)).contiguous()
        idx, cnt = ext.ball_query(xyz, ctr, r, 64)
        assert np.array_equal(cnt.cpu().numpy(), golden_full[f"sa{i}/ball_count"])
        assert np.array_equal(idx.sum(dim=2).cpu().numpy(), golden_full[f"sa{i}/ball_index_sum"])
        xyz = ctr


def test_ball_query_full_batch_properties(ext):
    pts = inputs.tabletop_batch(8).cuda()
    sel = ext.farthest_point_sample(pts, 5120)
    ctr = torch.gather(pts, 2, sel.unsqueeze(1).expand(-1, 3, -1)).contiguous()
    idx, cnt = ext.ball_query(pts, ctr, 0.02, 64)
    assert (cnt >= 1).all()  # every centroid is a point of the cloud, so it finds itself
    k = torch.arange(64, device="cuda")[None, None, :]
    live = k < cnt[:, :, None]
    # ascending index order inside the live part, padding == first neighbour outside
    assert ((idx[:, :, 1:] > idx[:, :, :-1]) | ~live[:, :, 1:]).all()
    assert ((idx == idx[:, :, :1]) | live).all()
    # every listed neighbour is strictly inside the ball (fp32 arithmetic of the reference)
    nb = torch.gather(pts.unsqueeze(2).expand(-1, -1, 5120, -1), 3, idx.unsqueeze(1).expand(-1, 3, -1, -1))
    d = nb - ctr.unsqueeze(-1)
    d2 = torch.addcmul(torch.addcmul(d[:, 1] * d[:, 1], d[:, 0], d[:, 0]), d[:, 2], d[:, 2])
    assert (d2 < np.float32(0.02) * np.float32(0.02) + 1e-9).all()


@pytest.mark.parametrize("B,C,N,M,K", [(2, 3, 500, 60, 16), (3, 131, 1000, 77, 9), (1, 259, 5120, 64, 64), (2, 1, 10, 10, 1)])
def test_group_points_forward_backward(ext, ora, B, C, N, M, K):
    rs = np.random.RandomState(B * C + N)
    x = torch.from_numpy(rs.randn(B, C, N).astype(np.float32))
    idx = torch.from_numpy(rs.randint(0, N, size=(B, M, K)).astype(np.int64))
    got = ext.group_points_forward(x.cuda(), idx.cuda())
    assert torch.equal(got.cpu(), ora.group_points_forward(x, idx))
    g = torch.from_numpy(rs.randn(B, C, M, K).astype(np.float32))
    gi = ext.group_points_backward(g.cuda(), idx.cuda(), N)
    # atomicAdd order is unspecified in the reference too: fp32 tolerance, not bit-exact
    np.testing.assert_allclose(gi.cpu().numpy(), ora.group_points_backward(g, idx, N).numpy(), rtol=1e-4, atol=1e-5)
    # unique indices -> exact
    if M * K <= N:
        perm = torch.stack([torch.from_numpy(rs.permutation(N)[:M * K]) for _ in range(B)]).reshape(B, M, K)
        gi = ext.group_points_backward(g.cuda(), perm.cuda(), N)
        assert torch.equal(gi.cpu(), ora.group_points_backward(g, perm, N))


@pytest.mark.parametrize("kind,B,Nq,Nk", [("uniform", 2, 1024, 256), ("uniform", 2, 5120, 1024), ("uniform", 1, 25600, 5120),
                                          ("lattice", 2, 3000, 300), ("dup", 2, 2000, 900), ("uniform", 3, 101, 3),
                                          ("identical", 2, 50, 10), ("uniform", 1, 300, 2049),
                                          # grid path (Nk >= 1024): ties, duplicates, 3-D clouds (many fall back)
                                          ("lattice", 2, 3000, 1500), ("dup", 2, 2000, 2000), ("identical", 1, 300, 1100),
                                          ("uniform", 2, 4000, 1024)])
def test_point_search_bit_exact(ext, ora, kind, B, Nq, Nk):
    q = _gen(kind, B, Nq, seed=Nq)
    k = _gen(kind, B, Nk, seed=Nk + 1)
    w_idx, w_d = ora.point_search(q, k, 3)
    g_idx, g_d = ext.point_search(q.cuda(), k.cuda(), 3)
    assert torch.equal(g_idx.cpu(), w_idx)
    assert torch.equal(g_d.cpu(), w_d)
    with pytest.raises(RuntimeError):
        ext.point_search(q.cuda(), k.cuda(), 2)
    with pytest.raises(RuntimeError):
        ext.point_search(q.cuda(), k[:, :, :2].contiguous().cuda(), 3)


@pytest.mark.parametrize("B,C,Nk,Nq", [(2, 5, 40, 90), (2, 256, 256, 1024), (1, 512, 1024, 5120)])
def test_interpolate_forward_backward(ext, ora, B, C, Nk, Nq):
    rs = np.random.RandomState(C)
    x = torch.from_numpy(rs.randn(B, C, Nk).astype(np.float32))
    idx = torch.from_numpy(rs.randint(0, Nk, size=(B, Nq, 3)).astype(np.int64))
    w = torch.from_numpy(rs.rand(B, Nq, 3).astype(np.float32))
    got = ext.interpolate_forward(x.cuda(), idx.cuda(), w.cuda())
    assert torch.equal(got.cpu(), ora.interpolate_forward(x, idx, w))  # same fma chain -> bit-exact
    g = torch.from_numpy(rs.randn(B, C, Nq).astype(np.float32))
    gi = ext.interpolate_backward(g.cuda(), idx.cuda(), w.cuda(), Nk)
    np.testing.assert_allclose(gi.cpu().numpy(), ora.interpolate_backward(g, idx, w, Nk).numpy(), rtol=1e-4, atol=1e-4)


def test_autograd_wrappers_match_reference_behaviour(ext):
    from s4g_release_b200.network_models.models.pointnet2_utils import functions as F_
    pts = inputs.uniform_cloud(2, 400, 9).cuda()
    feat = torch.randn(2, 6, 400, device="cuda", requires_grad=True)
    idx = F_.farthest_point_sample(pts, 50)
    ctr = F_.gather_points(pts, idx)
    nbr, _ = F_.ball_query(pts, ctr, 0.3, 8)
    grouped = F_.group_points(feat, nbr)
    grouped.sum().backward()
    want = torch.zeros_like(feat)
    want.scatter_add_(2, nbr.reshape(2, 1, -1).expand(-1, 6, -1), torch.ones(2, 6, 400, device="cuda"))
    assert torch.allclose(feat.grad, want)
    nn_idx, d2 = F_.search_nn_distance(pts, ctr, 3)
    w = torch.softmax(-d2, dim=2)
    feat2 = torch.randn(2, 6, 50, device="cuda", requires_grad=True)
    out = F_.feature_interpolate(feat2, nn_idx, w)
    out.sum().backward()
    assert torch.allclose(feat2.grad.sum(), torch.tensor(6.0 * 2 * 400, device="cuda"), rtol=1e-4)


@pytest.mark.parametrize("kind,B,N,M", [("uniform", 1, 131072, 96), ("uniform", 2, 110000, 64), ("uniform", 1, 262144, 64),
                                        ("lattice", 1, 150000, 48), ("dup", 1, 200000, 40)])
def test_fps_large_clouds_bit_exact(ext, ora, kind, B, N, M):
    """BASELINE config 3 sizes (N up to 262 144): the shared-memory-coordinate variant on 8 / 16-CTA clusters."""
    pts = _gen(kind, B, N, seed=N + M)
    got = ext.farthest_point_sample(pts.cuda(), M)
    assert torch.equal(got.cpu(), ora.farthest_point_sample(pts, M))
    with pytest.raises(RuntimeError):
        ext.farthest_point_sample(torch.zeros(1, 3, 262145, device="cuda"), 4)


@pytest.mark.parametrize("kind,B,N,M", [("uniform", 2, 5120, 1024), ("lattice", 2, 30000, 800), ("dup", 1, 26000, 1200),
                                        ("identical", 2, 6000, 70), ("uniform", 3, 4097, 4097)])
def test_fps_bucket_kernel_bit_exact(ext, ora, kind, B, N, M):
    """the experimental bucket-pruned FPS kernel (s4g_fps_set_bucket_mode) gives the reference's indices too"""
    from s4g_release_b200._lib import lib
    pts = _gen(kind, B, N, seed=21)
    want = ora.farthest_point_sample(pts, M)
    old = lib.s4g_fps_set_bucket_mode(1)
    try:
        got = ext.farthest_point_sample(pts.cuda(), M)
        torch.cuda.synchronize()
    finally:
        lib.s4g_fps_set_bucket_mode(old)
    assert torch.equal(got.cpu(), want)


@pytest.mark.parametrize("B,C,N,K,dtype", [(2, 4, 5, 3, torch.float32), (3, 64, 700, 20, torch.float32), (2, 7, 90, 8, torch.float64)])
def test_gather_knn_like_the_reference_test(B, C, N, K, dtype):
    """the reference's own test of dgcnn_ext (functions/gather_knn.py:27-56, first case = its sizes and seed): forward
    and backward against torch.gather"""
    from s4g_release_b200.network_models.functions.gather_knn import gather_knn
    torch.manual_seed(1)
    feature = torch.rand(B, C, N, dtype=dtype).cuda()
    knn_inds = torch.randint(0, N, [B, N, K]).long().cuda()
    f_ref = feature.clone().requires_grad_(True)
    f_ours = feature.clone().requires_grad_(True)
    want = torch.gather(f_ref.unsqueeze(2).expand(B, C, N, N), 3, knn_inds.unsqueeze(1).expand(B, C, N, K))
    got = gather_knn(f_ours, knn_inds)
    assert torch.equal(got, want)
    want.backward(torch.ones_like(want))
    got.backward(torch.ones_like(got))
    assert f_ref.grad.allclose(f_ours.grad)


@pytest.mark.parametrize("B,N,M,radius,K", [(2, 25600, 5120, 0.02, 64), (3, 5120, 1024, 0.08, 64), (2, 2048, 300, 0.1, 16),
                                             (1, 700, 64, 0.3, 8)])
def test_ball_query_in_two_calls_matches_the_one_call_form(B, N, M, radius, K):
    """index build (s4g_ball_grid_build_f32, here on a second stream) + query = s4g_ball_query_f32_i32, bit for bit"""
    import ctypes
    from s4g_release_b200._lib import check, lib, ptr
    g = torch.Generator().manual_seed(N + M)
    xyz = (torch.rand(B, 3, N, generator=g) * torch.tensor([1.0, 0.8, 0.3]).view(1, 3, 1)).cuda()
    ctr = xyz[:, :, torch.randperm(N, generator=g)[:M]].contiguous()
    want = torch.empty((B, M, K), dtype=torch.int32, device="cuda")
    want_n = torch.empty((B, M), dtype=torch.int32, device="cuda")
    main = torch.cuda.current_stream()
    check(lib.s4g_ball_query_f32_i32(ptr(xyz), ptr(ctr), B, N, M, radius, K, ptr(want), ptr(want_n),
                                     ctypes.c_void_p(main.cuda_stream)), "ball_query")
    side = torch.cuda.Stream()
    side.wait_stream(main)
    grid = lib.s4g_ball_grid_build_f32(ptr(xyz), B, N, radius, ctypes.c_void_p(side.cuda_stream))
    assert grid
    main.wait_stream(side)
    got = torch.empty_like(want)
    got_n = torch.empty_like(want_n)
    check(lib.s4g_ball_query_with_grid_f32_i32(grid, ptr(xyz), ptr(ctr), M, K, ptr(got), ptr(got_n),
                                               ctypes.c_void_p(main.cuda_stream)), "ball_query_with_grid")
    check(lib.s4g_ball_grid_free(grid, ctypes.c_void_p(main.cuda_stream)), "ball_grid_free")
    torch.cuda.synchronize()
    assert torch.equal(got, want) and torch.equal(got_n, want_n)


@pytest.mark.parametrize("B,C,N,M", [(2, 3, 5120, 1024), (3, 64, 777, 300), (1, 1, 10, 10), (2, 259, 1024, 7)])
def test_gather_points_kernel_equals_torch_gather(ext, B, C, N, M):
    """functions.gather_points: the no-autograd path is one s4g_gather_points_f32 launch, bit-identical to the
    torch.gather the reference uses (functions.py:10-25); with autograd it stays torch.gather."""
    from s4g_release_b200.network_models.models.pointnet2_utils import functions as F_
    g = torch.Generator().manual_seed(B * C + M)
    pts = torch.randn(B, C, N, generator=g).cuda()
    idx = torch.randint(0, N, (B, M), generator=g).cuda()
    want = pts.gather(2, idx.unsqueeze(1).expand(B, C, M))
    with torch.no_grad():
        assert torch.equal(F_.gather_points(pts, idx), want)
    assert torch.equal(ext.gather_points(pts.transpose(1, 2).contiguous().transpose(1, 2), idx), want)  # non-contiguous in
    p2 = pts.clone().requires_grad_(True)
    out = F_.gather_points(p2, idx)
    out.sum().backward()
    assert torch.equal(out, want) and p2.grad is not None


@pytest.mark.parametrize("B,C,N,M,K", [(8, 3, 16384, 2048, 32), (4, 40, 5120, 1024, 64), (16, 256, 5120, 1024, 64), (3, 67, 1000, 4096, 8),
                                       (8, 512, 1024, 256, 64), (2, 35, 16386, 2048, 32)])
def test_group_points_forward_staged_equals_plain(ext, B, C, N, M, K):
    """the shared-memory-staged forward (bulk-copied channel planes, gathers from shared memory) and the plain gather kernel
    produce identical tensors (= torch.gather); N % 4 != 0 falls back to the plain kernel"""
    from s4g_release_b200._lib import lib
    g = torch.Generator().manual_seed(N + M)
    x = torch.randn(B, C, N, generator=g).cuda()
    idx = torch.randint(0, N, (B, M, K), generator=g).cuda()
    prev = lib.s4g_group_points_set_staged(0)
    try:
        plain = ext.group_points_forward(x, idx)
        lib.s4g_group_points_set_staged(1)
        staged = ext.group_points_forward(x, idx)
    finally:
        lib.s4g_group_points_set_staged(prev)
    want = torch.gather(x.unsqueeze(2).expand(-1, -1, M, -1), 3, idx.unsqueeze(1).expand(-1, C, -1, -1))
    assert torch.equal(plain, want) and torch.equal(staged, want)
