"""GPU suite: the REFERENCE's own CUDA kernels (compiled unmodified for sm_100a into oracle/_ref by
oracle/build_ref.py) side by side with (a) the C oracle, which pins the oracle, and (b) the sm_100a
kernels of this repo.  Bit-exact for FPS / ball query / 3-NN / gathers / interpolation.

The reference kernels' outputs on these seeded inputs are stored in tests/golden/ref_cuda_parity.npz
(tests/golden/make_ref_cuda_parity_golden.py): SHA-256 digests of the bit-exact outputs, a fixed sample of each
atomicAdd backward output.  The C oracle is checked against them on every run, so the comparison with the
reference holds where oracle/_ref is not built (it needs the reference's source tree); where it is built, the
three-way comparison also runs live."""
import os

import numpy as np
import pytest
import torch

from tests import inputs
from tests.golden.make_golden import array_digest

pytestmark = pytest.mark.gpu

FPS_CASES = [("uniform", 2, 5120, 1024), ("lattice", 3, 2000, 600), ("lattice", 2, 200, 150), ("lattice", 2, 40, 40),
             ("dup", 2, 3000, 1500), ("identical", 2, 600, 50), ("scene", 2, 25600, 5120), ("uniform", 2, 13, 9),
             ("lattice", 1, 30000, 1500)]
BALL_CASES = [("uniform", 2, 5120, 1024, 0.08, 64), ("scene", 1, 25600, 5120, 0.02, 64), ("lattice", 2, 2000, 500, 0.125, 32),
              ("dup", 2, 3000, 400, 0.05, 32), ("uniform", 2, 50, 3, 1e-4, 8), ("identical", 2, 300, 20, 0.1, 16)]
NN_CASES = [("uniform", 2, 5120, 1024), ("scene", 1, 25600, 5120), ("lattice", 2, 3000, 300), ("dup", 2, 2000, 900),
            ("uniform", 3, 101, 3)]
GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "ref_cuda_parity.npz")
BWD_SAMPLE = 4096  # elements kept of each atomicAdd backward output


def key(op, case):
    return op + "/" + "-".join(map(str, case))


def bwd_sample(t):
    """The fixed, seeded elements of a backward output that the golden keeps."""
    flat = t.reshape(-1).numpy()
    return flat[np.random.default_rng(0).choice(flat.size, BWD_SAMPLE, replace=False)]


def _gen(kind, B, N, seed):
    return {"uniform": lambda: inputs.uniform_cloud(B, N, seed), "lattice": lambda: inputs.lattice_cloud(B, N, seed, side=8),
            "dup": lambda: inputs.duplicated_cloud(B, N, seed), "identical": lambda: inputs.identical_cloud(B, N),
            "scene": lambda: inputs.tabletop_batch(B, 1000 + seed, N)}[kind]()


def fps_inputs(kind, B, N, M):
    return _gen(kind, B, N, seed=7)


def ball_inputs(kind, B, N, M, rad, K):
    from oracle import pn2_ext_cpu as ora
    pts = _gen(kind, B, N, seed=8)
    return pts, ora.gather_points(pts, ora.farthest_point_sample(pts, M))


def nn_inputs(kind, B, Nq, Nk):
    from oracle import pn2_ext_cpu as ora
    q = _gen(kind, B, Nq, seed=9)
    return q, (ora.gather_points(q, ora.farthest_point_sample(q, Nk)) if kind == "scene" else _gen(kind, B, Nk, seed=10))


def op_inputs():
    """group / interpolate operands: x, idx, grad of the grouped tensor, 3-NN idx, weights, grad of the interpolation"""
    rs = np.random.RandomState(1)
    B, C, N, M, K = 2, 67, 900, 50, 16
    x = torch.from_numpy(rs.randn(B, C, N).astype(np.float32))
    idx = torch.from_numpy(rs.randint(0, N, size=(B, M, K)).astype(np.int64))
    g = torch.from_numpy(rs.randn(B, C, M, K).astype(np.float32))
    idx3 = torch.from_numpy(rs.randint(0, N, size=(B, M, 3)).astype(np.int64))
    w = torch.from_numpy(rs.rand(B, M, 3).astype(np.float32))
    g2 = torch.from_numpy(rs.randn(B, C, M).astype(np.float32))
    return x, idx, g, idx3, w, g2


@pytest.fixture(scope="module")
def ref():
    from oracle import build_ref
    if not os.path.exists(build_ref.so_path()):
        return None
    return build_ref.load()


@pytest.fixture(scope="module")
def ext():
    from s4g_release_b200.network_models.models.pointnet2_utils import pn2_ext
    return pn2_ext


@pytest.fixture(scope="module")
def ora():
    from oracle import pn2_ext_cpu
    return pn2_ext_cpu


@pytest.fixture(scope="module")
def stored():
    return dict(np.load(GOLDEN))


def _digests(*ts):
    return [array_digest(t) for t in ts]


STORED = "C oracle differs from the reference kernel's stored output"
LIVE = "C oracle differs from the reference CUDA kernel"
OURS = "sm_100a kernel differs from the reference kernel's output (matched by the C oracle above)"


@pytest.mark.parametrize("kind,B,N,M", FPS_CASES)
def test_fps_three_way(ref, ext, ora, stored, kind, B, N, M):
    pts = fps_inputs(kind, B, N, M)
    r = ora.farthest_point_sample(pts, M)
    assert _digests(r) == list(stored[key("fps", (kind, B, N, M))]), STORED
    if ref is not None:
        assert torch.equal(ref.farthest_point_sample(pts.cuda(), M).cpu(), r), LIVE
    assert torch.equal(ext.farthest_point_sample(pts.cuda(), M).cpu(), r), OURS


@pytest.mark.parametrize("kind,B,N,M,rad,K", BALL_CASES)
def test_ball_query_three_way(ref, ext, ora, stored, kind, B, N, M, rad, K):
    pts, ctr = ball_inputs(kind, B, N, M, rad, K)
    r_idx, r_cnt = ora.ball_query(pts, ctr, rad, K)
    assert _digests(r_idx, r_cnt) == list(stored[key("ball", (kind, B, N, M, rad, K))]), STORED
    if ref is not None:
        ref_idx, ref_cnt = [t.cpu() for t in ref.ball_query(pts.cuda(), ctr.cuda(), rad, K)]
        assert torch.equal(ref_idx, r_idx) and torch.equal(ref_cnt, r_cnt), LIVE
    g_idx, g_cnt = [t.cpu() for t in ext.ball_query(pts.cuda(), ctr.cuda(), rad, K)]
    assert torch.equal(g_idx, r_idx) and torch.equal(g_cnt, r_cnt), OURS


@pytest.mark.parametrize("kind,B,Nq,Nk", NN_CASES)
def test_point_search_three_way(ref, ext, ora, stored, kind, B, Nq, Nk):
    q, k = nn_inputs(kind, B, Nq, Nk)
    r_idx, r_d = ora.point_search(q, k, 3)
    assert _digests(r_idx, r_d) == list(stored[key("nn", (kind, B, Nq, Nk))]), STORED
    if ref is not None:
        ref_idx, ref_d = [t.cpu() for t in ref.point_search(q.cuda(), k.cuda(), 3)]
        assert torch.equal(ref_idx, r_idx) and torch.equal(ref_d, r_d), LIVE
    g_idx, g_d = [t.cpu() for t in ext.point_search(q.cuda(), k.cuda(), 3)]
    assert torch.equal(g_idx, r_idx) and torch.equal(g_d, r_d), OURS


def test_group_and_interpolate_three_way(ref, ext, ora, stored):
    x, idx, g, idx3, w, g2 = op_inputs()
    N = x.shape[2]
    r = ora.group_points_forward(x, idx)
    assert _digests(r) == list(stored["group_forward"]), STORED
    if ref is not None:
        assert torch.equal(ref.group_points_forward(x.cuda(), idx.cuda()).cpu(), r), LIVE
    assert torch.equal(ext.group_points_forward(x.cuda(), idx.cuda()).cpu(), r), OURS
    r = ora.group_points_backward(g, idx, N)
    np.testing.assert_allclose(bwd_sample(r), stored["group_backward"], rtol=1e-4, atol=1e-5, err_msg=STORED)
    if ref is not None:
        r_ref = ref.group_points_backward(g.cuda(), idx.cuda(), N).cpu()
        np.testing.assert_allclose(r.numpy(), r_ref.numpy(), rtol=1e-4, atol=1e-5, err_msg=LIVE)
        r = r_ref
    got = ext.group_points_backward(g.cuda(), idx.cuda(), N).cpu()
    np.testing.assert_allclose(got.numpy(), r.numpy(), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(bwd_sample(got), stored["group_backward"], rtol=1e-4, atol=1e-5)
    r = ora.interpolate_forward(x, idx3, w)
    assert _digests(r) == list(stored["interpolate_forward"]), STORED
    if ref is not None:
        assert torch.equal(ref.interpolate_forward(x.cuda(), idx3.cuda(), w.cuda()).cpu(), r), LIVE
    assert torch.equal(ext.interpolate_forward(x.cuda(), idx3.cuda(), w.cuda()).cpu(), r), OURS
    r = ora.interpolate_backward(g2, idx3, w, N)
    np.testing.assert_allclose(bwd_sample(r), stored["interpolate_backward"], rtol=1e-4, atol=1e-5, err_msg=STORED)
    if ref is not None:
        r_ref = ref.interpolate_backward(g2.cuda(), idx3.cuda(), w.cuda(), N).cpu()
        np.testing.assert_allclose(r.numpy(), r_ref.numpy(), rtol=1e-4, atol=1e-5, err_msg=LIVE)
        r = r_ref
    got = ext.interpolate_backward(g2.cuda(), idx3.cuda(), w.cuda(), N).cpu()
    np.testing.assert_allclose(got.numpy(), r.numpy(), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(bwd_sample(got), stored["interpolate_backward"], rtol=1e-4, atol=1e-5)
