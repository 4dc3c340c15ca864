"""CPU suite: which ball-query kernel serves a shape.  s4g_ball_query_uses_grid is the host-side rule that both
s4g_ball_query_f32(_i32) and the engine's two-call form follow: the grid kernel for N >= 8192 points, K <= 256
neighbours and a positive radius, the linear scan otherwise.  The GPU edge-case tests assert it before they run, so
pinning it here keeps their cases on the path they are written for."""
import pytest


@pytest.fixture(scope="module")
def lib():
    from s4g_release_b200 import _lib
    return _lib.lib


@pytest.mark.parametrize("N,K,r,grid", [
    (8191, 64, 0.02, 0), (8192, 64, 0.02, 1), (25600, 64, 0.02, 1), (1 << 30, 64, 0.02, 1),
    (8192, 256, 0.02, 1), (8192, 257, 0.02, 0), (25600, 1, 0.02, 1),
    (8192, 64, 1e-30, 1), (8192, 64, 1e30, 1),
    (8192, 64, 0.0, 0), (8192, 64, -0.0, 0), (8192, 64, -1.0, 0), (8192, 64, float("nan"), 0),
    (8192, 64, float("-inf"), 0),
])
def test_ball_query_uses_grid_boundaries(lib, N, K, r, grid):
    assert lib.s4g_ball_query_uses_grid(N, K, r) == grid


def test_ball_grid_build_refuses_what_the_grid_does_not_serve(lib):
    """the two-call form's build rejects a radius the grid cannot serve before touching the device"""
    import ctypes
    dummy = ctypes.c_void_p(16)
    for r in (0.0, -1.0, float("nan")):
        assert not lib.s4g_ball_grid_build_f32(dummy, 1, 8192, r, None)
        assert b"bad cloud or radius" in lib.s4g_last_error()
