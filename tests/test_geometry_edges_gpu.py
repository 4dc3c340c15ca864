"""GPU suite: the geometry kernels at the edges where they go wrong, bit for bit against the C oracle.

* Grid ball query (N >= 8192; csrc/grid.cu): ties, duplicates, > 256 hits (linear-scan fallback), one-cell and
  many-cell radii, centroids outside the cloud's box, flat and spread clouds, through the int64 entry point
  (pn2_ext.ball_query), the int32 one-call form and the two-call form.  Every case first asserts which path it takes.
* 3-NN on both sides of the grid threshold (Nk = 1023 / 1024) for pn2_ext.point_search (fp32, fp64) and the fused
  engine's three_nn_weights, including inputs with fewer than three finite distances (NaN points, coordinates whose
  squared distance overflows), where the reference keeps its start values {1e40, 0, 0} / {-1, 0, 0}.
* The fused engine's int32 helpers: interp_concat (plain and ReLU), FPS int32 vs int64, gather_xyz.
"""
import ctypes

import numpy as np
import pytest
import torch

from tests import inputs
from tests.test_ops_gpu import FPS_CASES, _gen

pytestmark = pytest.mark.gpu

NAN = float("nan")


@pytest.fixture(scope="module")
def ext():
    from s4g_release_b200.network_models.models.pointnet2_utils import pn2_ext
    return pn2_ext


@pytest.fixture(scope="module")
def ora():
    from oracle import pn2_ext_cpu
    return pn2_ext_cpu


@pytest.fixture(scope="module")
def abi():
    from s4g_release_b200 import _lib
    return _lib


@pytest.fixture(scope="module")
def engine():
    from s4g_release_b200.engine import FusedPointNet2
    return FusedPointNet2


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


# ------------------------------------------------------------------------------------------------ ball query
def _f32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))


def _pick(pts, M, seed, jitter=0.0):
    """M centroids: points of the cloud (seeded choice), optionally moved by up to `jitter` per axis"""
    B, _, N = pts.shape
    rs = np.random.RandomState(seed)
    sel = np.stack([rs.choice(N, M, replace=M > N) for _ in range(B)])
    ctr = np.take_along_axis(pts.numpy(), sel[:, None, :].repeat(3, 1), 2)
    return _f32(ctr + rs.uniform(-jitter, jitter, ctr.shape))


def _ball_all_forms(ext, ora, abi, pts, ctr, r, K, grid):
    """int64 (pn2_ext), int32 one call with and without count, and the two-call form: all equal to the oracle"""
    lib, ptr = abi.lib, abi.ptr
    B, _, N = pts.shape
    M = ctr.shape[2]
    assert lib.s4g_ball_query_uses_grid(N, K, r) == int(grid)
    want_idx, want_cnt = ora.ball_query(pts, ctr, r, K)
    assert (want_cnt > 0).any() or (ctr.abs() > 5).any()  # the case finds neighbours unless it is about far centroids
    d_pts, d_ctr = pts.cuda(), ctr.cuda()
    got_idx, got_cnt = ext.ball_query(d_pts, d_ctr, r, K)
    assert torch.equal(got_cnt.cpu(), want_cnt)
    assert torch.equal(got_idx.cpu(), want_idx)
    idx = torch.full((B, M, K), -7, dtype=torch.int32, device="cuda")
    cnt = torch.full((B, M), -7, dtype=torch.int32, device="cuda")
    abi.check(lib.s4g_ball_query_f32_i32(ptr(d_pts), ptr(d_ctr), B, N, M, r, K, ptr(idx), ptr(cnt), _stream()),
              "ball_query_i32")
    assert torch.equal(idx.cpu().long(), want_idx) and torch.equal(cnt.cpu().long(), want_cnt)
    idx.fill_(-7)
    abi.check(lib.s4g_ball_query_f32_i32(ptr(d_pts), ptr(d_ctr), B, N, M, r, K, ptr(idx), None, _stream()),
              "ball_query_i32")
    assert torch.equal(idx.cpu().long(), want_idx)
    if K <= 256 and r > 0:  # the two-call form always runs the grid kernel
        g = lib.s4g_ball_grid_build_f32(ptr(d_pts), B, N, r, _stream())
        assert g, lib.s4g_last_error()
        idx.fill_(-7)
        cnt.fill_(-7)
        try:
            abi.check(lib.s4g_ball_query_with_grid_f32_i32(g, ptr(d_pts), ptr(d_ctr), M, K, ptr(idx), ptr(cnt), _stream()),
                      "ball_query_with_grid")
        finally:
            abi.check(lib.s4g_ball_grid_free(g, _stream()), "ball_grid_free")
        assert torch.equal(idx.cpu().long(), want_idx) and torch.equal(cnt.cpu().long(), want_cnt)
    return want_cnt


def _flat(B, N, seed):
    p = inputs.uniform_cloud(B, N, seed)
    p[:, 2] = 0.3
    return p


def _far_point(B, N, seed):
    p = inputs.uniform_cloud(B, N, seed)
    p[:, :, N // 3] = torch.tensor([50.0, 0.5, 0.5])  # one point 50 m away from a 1 m cloud
    return p


def _extents(B, N, seed):
    assert B == 3
    return inputs.uniform_cloud(3, N, seed) * torch.tensor([0.1, 1.0, 10.0]).view(3, 1, 1)


GRID_BQ_CASES = [
    # (cloud, B, N, M, r, K, jitter): N >= 8192, K <= 256 and r > 0 -> grid path
    ("lattice", 2, 10000, 700, 0.125, 32, 0.0),   # only the ~20 duplicates of each lattice site are closer than 0.125
    ("lattice", 2, 10000, 500, 0.3, 64, 0.0),     # 57 sites x ~20 points: > 256 hits -> exact linear-scan fallback
    ("lattice", 2, 8192, 400, 0.2, 256, 0.0),     # K = 256: 19 sites x ~16 points, ties and > 256 hits
    ("dup", 2, 16000, 900, 0.05, 32, 0.01),       # 50 % duplicated points
    ("identical", 2, 8192, 40, 0.1, 16, 0.0),     # every point in one cell, 8192 hits
    ("uniform", 2, 9000, 300, 10.0, 128, 0.0),    # one cell
    ("uniform", 2, 9000, 300, 1e-4, 8, 1e-4),     # 1000 cells per axis at r -> the cell edge grows until the table fits
    ("uniform", 1, 12000, 500, 0.15, 256, 0.0),   # K = 256 on the grid: ~170 hits, buffer not overflowed
    ("flat", 2, 9000, 600, 0.05, 64, 0.02),       # constant z: one cell layer
    ("far_point", 2, 9000, 600, 0.08, 64, 0.01),  # a point 50 m away stretches the box
    ("extents", 3, 9000, 500, 0.05, 64, 0.01),    # one batch, boxes of 0.1, 1 and 10 m: one cell size per cloud
]


@pytest.mark.parametrize("kind,B,N,M,r,K,jitter", GRID_BQ_CASES)
def test_grid_ball_query_edges(ext, ora, abi, kind, B, N, M, r, K, jitter):
    gen = {"flat": _flat, "far_point": _far_point, "extents": _extents}
    pts = gen[kind](B, N, N + K) if kind in gen else _gen(kind, B, N, seed=N + K)
    ctr = _pick(pts, M, seed=M, jitter=jitter)
    if kind == "far_point":
        ctr[:, :, 0] = torch.tensor([50.0, 0.5, 0.5])  # centred on the far point: it finds itself and nothing else
    cnt = _ball_all_forms(ext, ora, abi, pts, ctr, r, K, grid=True)
    if kind == "identical" or (kind == "lattice" and r >= 0.2) or r >= 10:
        assert (cnt == K).any()  # cases built to have more than 256 hits: the linear-scan fallback ran


def test_grid_ball_query_k256_vs_k257(ext, ora, abi):
    """the same cloud and centroids on the grid (K = 256) and on the linear kernel (K = 257)"""
    pts = inputs.uniform_cloud(2, 10000, 31)
    ctr = _pick(pts, 300, seed=32, jitter=0.02)
    for r in (0.12, 0.2):  # ~70 and ~330 hits per centroid: the second overflows the grid's 256-hit buffer
        c256 = _ball_all_forms(ext, ora, abi, pts, ctr, r, 256, grid=True)
        c257 = _ball_all_forms(ext, ora, abi, pts, ctr, r, 257, grid=False)
        assert torch.equal(torch.clamp(c257, max=256), c256)
    assert (c257 == 257).any()


def test_grid_ball_query_8191_vs_8192(ext, ora, abi):
    """N = 8191 runs the linear kernel, N = 8192 the grid: same first 8191 points, same answers where no hit is lost"""
    pts = inputs.tabletop_batch(1, 7, 8192)
    ctr = _pick(pts, 1000, seed=33, jitter=0.01)
    ctr[:, :, 0] = pts[:, :, 8191]  # a centroid on the extra point
    a = _ball_all_forms(ext, ora, abi, pts[:, :, :8191].contiguous(), ctr, 0.03, 64, grid=False)
    b = _ball_all_forms(ext, ora, abi, pts, ctr, 0.03, 64, grid=True)
    assert (a > 0).any() and torch.equal(torch.clamp(b - a, min=0, max=1), b - a)  # one more point: at most one more hit
    assert b[0, 0] == a[0, 0] + 1


def test_grid_ball_query_centroids_outside_the_box(ext, ora, abi):
    r = 0.05
    pts = inputs.uniform_cloud(2, 9000, 34)
    lo, hi = pts.amin(2), pts.amax(2)  # (B,3)
    mid = (lo + hi) / 2
    ctr = []
    for a in range(3):
        for side, sign in ((hi, 1.0), (lo, -1.0)):
            for off in (0.5 * r, 0.99 * r, 1.5 * r, 10.0, 1e6):  # just outside (hits), outside by more than r, far
                c = mid.clone()
                c[:, a] = side[:, a] + sign * off
                ctr.append(c)
                c = side.clone()  # at a corner of the box, pushed out along one axis
                c[:, a] = c[:, a] + sign * off
                ctr.append(c)
    ctr = torch.stack(ctr, 2).contiguous()  # (B,3,60)
    cnt = _ball_all_forms(ext, ora, abi, pts, ctr, r, 32, grid=True)
    assert (cnt > 0).any() and (cnt == 0).any()


def test_grid_ball_query_tabletop_level0(ext, ora, abi):
    """the engine's first level: 2 tabletop scenes, 25 600 -> 5 120 FPS centroids, r = 0.02, K = 64, full index equality"""
    pts = inputs.tabletop_batch(2)
    ctr = ora.gather_points(pts, ora.farthest_point_sample(pts, 5120))
    cnt = _ball_all_forms(ext, ora, abi, pts, ctr, 0.02, 64, grid=True)
    assert (cnt >= 1).all()


# ------------------------------------------------------------------------------------------------ 3-NN
def _ref_weights(d):
    """the kernel's documented arithmetic on the oracle's fp32 distances: v = 1/max(d, 1e-10), w = v / ((v0 + v1) + v2)"""
    d = d.numpy().astype(np.float32)
    v = np.float32(1.0) / np.maximum(d, np.float32(1e-10))
    norm = (v[..., 0] + v[..., 1]) + v[..., 2]
    return torch.from_numpy(v / norm[..., None])


def _check_three_nn(ext, ora, engine, q, k, f64=True):
    """pn2_ext.point_search (fp32) and FusedPointNet2.three_nn_weights against the oracle; fp64 on the same points"""
    Nk = k.shape[2]
    w_idx, w_d = ora.point_search(q, k, 3)
    g_idx, g_d = ext.point_search(q.cuda(), k.cuda(), 3)
    assert torch.equal(g_idx.cpu(), w_idx)
    assert torch.equal(g_d.cpu(), w_d)
    f_idx, f_w = engine.three_nn_weights(q.cuda(), k.cuda())
    f_idx = f_idx.cpu()
    assert f_idx.dtype == torch.int32
    assert ((f_idx >= 0) & (f_idx < Nk)).all(), "fused 3-NN index outside [0, Nk)"
    assert torch.equal(f_idx.long(), torch.clamp(w_idx, min=0))  # the reference's -1 (weight 0) is written as 0
    assert torch.equal(f_w.cpu(), _ref_weights(w_d))
    if f64:
        qd, kd = q.double(), k.double()
        w_idx, w_d = ora.point_search(qd, kd, 3)
        g_idx, g_d = ext.point_search(qd.cuda(), kd.cuda(), 3)
        assert torch.equal(g_idx.cpu(), w_idx) and torch.equal(g_d.cpu(), w_d)
    return w_idx


@pytest.fixture(scope="module")
def tabletop_levels(ext):
    """2 tabletop scenes and their FPS levels 25 600 -> 5 120 -> 1 024 -> 256 (each level's points are a subset of the
    previous one, so many queries are at distance 0 from a key: the 1e-10 clamp)"""
    xyz = inputs.tabletop_batch(2).cuda()
    levels = [xyz]
    for m in (5120, 1024, 256):
        idx = ext.farthest_point_sample(levels[-1], m)
        levels.append(torch.gather(levels[-1], 2, idx.unsqueeze(1).expand(-1, 3, -1)).contiguous())
    return [x.cpu() for x in levels]


@pytest.mark.parametrize("level", [0, 1, 2])
def test_three_nn_tabletop_levels(ext, ora, engine, tabletop_levels, level):
    q, k = tabletop_levels[level], tabletop_levels[level + 1]
    idx = _check_three_nn(ext, ora, engine, q, k)
    assert (idx >= 0).all()


def _nn_cloud(kind, B, Nq, Nk, seed):
    rs = np.random.RandomState(seed)
    q = rs.rand(B, 3, Nq)
    if kind == "uniform":
        k = rs.rand(B, 3, Nk)
    elif kind == "collinear":
        t = rs.rand(B, 1, Nk)
        k = np.concatenate([t, 0.5 * t + 0.25, 0.8 - 0.6 * t], 1)
    elif kind == "coplanar":
        k = rs.rand(B, 3, Nk)
        k[:, 2] = 0.4
    elif kind == "identical":
        k = np.full((B, 3, Nk), 0.25)
    elif kind == "lattice":  # keys and queries on the same 1/8 lattice: distance ties and d = 0
        k = rs.randint(0, 8, (B, 3, Nk)) / 8.0
        q = rs.randint(0, 8, (B, 3, Nq)) / 8.0
    elif kind == "far_queries":  # every query outside the key box: all go to the grid's exact pass
        k = rs.rand(B, 3, Nk)
        q = q + np.array([3.0, -2.0, 10.0])[None, :, None] * rs.choice([1.0, 2.0], (B, 1, Nq))
    elif kind == "outlier":
        k = rs.rand(B, 3, Nk)
        k[:, :, Nk // 2] = [50.0, 0.5, 0.5]
        q[:, :, :4] = np.array([49.0, 0.5, 0.5])[None, :, None]  # a few queries are nearest to it
    else:
        raise ValueError(kind)
    return _f32(q), _f32(k)


@pytest.mark.parametrize("Nk", [1023, 1024])  # linear kernel / grid
@pytest.mark.parametrize("kind", ["uniform", "collinear", "coplanar", "identical", "lattice", "far_queries", "outlier"])
def test_three_nn_geometry(ext, ora, engine, kind, Nk):
    q, k = _nn_cloud(kind, 2, 2000, Nk, seed=Nk)
    idx = _check_three_nn(ext, ora, engine, q, k)
    if kind == "identical":
        assert (idx == torch.tensor([0, 1, 2])).all()  # all tie: earlier key wins


@pytest.mark.parametrize("B,Nq,Nk", [(3, 257, 3), (3, 1, 1023), (3, 1, 1024), (3, 257, 1023), (3, 257, 1024),
                                     (1, 1, 3)])
def test_three_nn_small_shapes(ext, ora, engine, B, Nq, Nk):
    q, k = _nn_cloud("uniform", B, Nq, Nk, seed=Nq + Nk)
    _check_three_nn(ext, ora, engine, q, k)


def _non_finite(case, B, Nq, Nk, seed, dtype):
    """query / key clouds where some queries have fewer than three keys at a finite distance"""
    rs = np.random.RandomState(seed)
    q = rs.rand(B, 3, Nq)
    k = rs.rand(B, 3, Nk)
    big = 3e19 if dtype == np.float32 else 1e21  # squared distance overflows (fp32) / exceeds 1e40 (fp64)
    if case == "nan_query":
        q[:, :, 0] = NAN
        q[:, 0, 5] = NAN  # one coordinate only
        q[:, :, Nq - 1] = NAN
    elif case.startswith("nan_keys_"):  # c keys with finite coordinates, the rest NaN
        c = int(case[-1])
        keep = rs.choice(Nk, c, replace=False)
        mask = np.ones(Nk, bool)
        mask[keep] = False
        k[:, :, mask] = NAN
    elif case == "huge_query":
        q[:, 0, ::3] = big
        q[:, 1, 1::3] = -big
    elif case.startswith("huge_keys_"):  # c keys in the unit box, the rest at +-big
        c = int(case[-1])
        keep = rs.choice(Nk, c, replace=False)
        mask = np.ones(Nk, bool)
        mask[keep] = False
        k[:, 0, mask] = np.where(rs.rand(B, mask.sum()) < 0.5, big, -big)
    else:
        raise ValueError(case)
    q[:, :, 1] = k[:, :, 1]  # a query on a key
    return torch.from_numpy(q.astype(dtype)), torch.from_numpy(k.astype(dtype))


NON_FINITE = ["nan_query", "nan_keys_0", "nan_keys_1", "nan_keys_2", "huge_query", "huge_keys_0", "huge_keys_1",
              "huge_keys_2"]


@pytest.mark.parametrize("Nk", [1023, 1024])  # linear kernel / grid
@pytest.mark.parametrize("case", NON_FINITE)
def test_three_nn_fewer_than_three_finite_f32(ext, ora, engine, case, Nk):
    q, k = _non_finite(case, 2, 300, Nk, seed=Nk, dtype=np.float32)
    idx = _check_three_nn(ext, ora, engine, q, k, f64=False)
    assert (idx == -1).any()  # the case really has queries with fewer than three finite distances


@pytest.mark.parametrize("Nk", [1023, 1024])
@pytest.mark.parametrize("case", NON_FINITE)
def test_three_nn_fewer_than_three_finite_f64(ext, ora, case, Nk):
    q, k = _non_finite(case, 2, 300, Nk, seed=Nk, dtype=np.float64)
    w_idx, w_d = ora.point_search(q, k, 3)
    assert (w_idx == -1).any()
    g_idx, g_d = ext.point_search(q.cuda(), k.cuda(), 3)
    assert torch.equal(g_idx.cpu(), w_idx) and torch.equal(g_d.cpu(), w_d)


def test_three_nn_weights_all_nan_query_contract(engine):
    """an all-NaN query: the reference's distances {1e40, 0, 0} give weights [0, 0.5, 0.5] on rows [0, 0, 0]"""
    for Nk in (1023, 1024):
        k = inputs.uniform_cloud(1, Nk, 5)
        q = torch.full((1, 3, 2), NAN)
        idx, w = engine.three_nn_weights(q.cuda(), k.cuda())
        assert torch.equal(idx.cpu(), torch.zeros(1, 2, 3, dtype=torch.int32))
        assert torch.equal(w.cpu(), torch.tensor([0.0, 0.5, 0.5]).expand(1, 2, 3))


# ------------------------------------------------------------------------------------------------ fused int32 helpers
def _interp_ref(ora, sparse, idx, w, B, Nk, Nq, relu):
    """oracle.interpolate_forward on the fp32 upcast of the bf16 rows, rounded to bf16 (RNE), then ReLU"""
    C2 = sparse.shape[1]
    x = sparse.float().reshape(B, Nk, C2).transpose(1, 2).contiguous()
    out = ora.interpolate_forward(x, idx.long(), w).transpose(1, 2).reshape(B * Nq, C2).to(torch.bfloat16)
    return torch.relu(out) if relu else out


@pytest.mark.parametrize("C1", [0, 8, 128])
@pytest.mark.parametrize("C2", [8, 64, 264, 512])
@pytest.mark.parametrize("weights", ["random", "geometry"])
def test_interp_concat_bit_exact(ora, engine, weights, C2, C1):
    B = 3
    for Nq in (1, 5, 4099):  # 4099 = 1024 warps of 4 rows + a last warp with 3
        Nk = 1000 if weights == "random" else 1024
        g = torch.Generator().manual_seed(C2 * 7 + C1 + Nq)
        if weights == "random":
            idx = torch.randint(0, Nk, (B, Nq, 3), generator=g, dtype=torch.int32)
            w = torch.rand(B, Nq, 3, generator=g) * 2 - 0.5
        else:
            q, k = _nn_cloud("uniform", B, Nq, Nk, seed=Nq)
            idx, w = [t.cpu() for t in engine.three_nn_weights(q.cuda(), k.cuda())]
        sparse = (torch.randn(B * Nk, C2, generator=g) * 3).to(torch.bfloat16)
        dense = (torch.randn(B * Nq, C1, generator=g) * 3).to(torch.bfloat16) if C1 else None
        for relu in (False, True):
            out = engine.interp_concat(sparse.cuda(), idx.cuda(), w.cuda(), dense.cuda() if C1 else None, B, Nk, Nq,
                                       relu=relu).cpu()
            assert out.shape == (B * Nq, C2 + C1)
            assert torch.equal(out[:, :C2], _interp_ref(ora, sparse, idx, w, B, Nk, Nq, relu))
            if C1:
                assert torch.equal(out[:, C2:].view(torch.int16), dense.view(torch.int16))  # byte-equal copy


@pytest.mark.parametrize("kind,B,N,M", FPS_CASES)
def test_fps_int32_equals_int64(ext, abi, kind, B, N, M):
    """the fused engine's int32 FPS returns the int64 entry point's indices (pinned by the oracle in test_ops_gpu),
    with the default kernels and with the bucket kernel"""
    pts = _gen(kind, B, N, seed=N + M).cuda()
    want = ext.farthest_point_sample(pts, M)
    old = abi.lib.s4g_fps_set_bucket_mode(0)
    try:
        for mode in (0, 1):
            abi.lib.s4g_fps_set_bucket_mode(mode)
            got = torch.full((B, M), -7, dtype=torch.int32, device="cuda")
            abi.check(abi.lib.s4g_farthest_point_sample_f32_i32(abi.ptr(pts), B, N, M, abi.ptr(got), _stream()), "fps_i32")
            i64 = ext.farthest_point_sample(pts, M)
            torch.cuda.synchronize()
            assert torch.equal(got.long(), want), "int32 FPS, bucket mode %d" % mode
            assert torch.equal(i64, want), "int64 FPS, bucket mode %d" % mode
    finally:
        abi.lib.s4g_fps_set_bucket_mode(old)


@pytest.mark.parametrize("B,N,M", [(1, 5, 1), (3, 1000, 1), (3, 1000, 257), (3, 25600, 5120), (2, 1, 257)])
def test_gather_xyz_equals_torch_gather(engine, B, N, M):
    g = torch.Generator().manual_seed(N + M)
    xyz = torch.randn(B, 3, N, generator=g).cuda()
    idx = torch.randint(0, N, (B, M), generator=g, dtype=torch.int32)
    idx[:, 0] = N - 1
    idx = idx.cuda()
    got = engine.gather_xyz(xyz, idx)
    assert torch.equal(got, torch.gather(xyz, 2, idx.long().unsqueeze(1).expand(-1, 3, -1)))
