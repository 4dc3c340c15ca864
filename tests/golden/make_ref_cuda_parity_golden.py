"""Stores what tests/test_ref_cuda_parity.py compares against: the outputs of the reference's own CUDA kernels
(oracle/_ref, built by oracle/build_ref.py from the reference's source tree) on the test's seeded inputs.  Bit-exact
outputs are stored as SHA-256 digests (tests/golden/make_golden.py::array_digest), the two atomicAdd backward outputs as
a fixed sample of their elements (tests/test_ref_cuda_parity.py::bwd_sample).  On a GPU with oracle/_ref built:

    python tests/golden/make_ref_cuda_parity_golden.py                 -> tests/golden/ref_cuda_parity.npz

`--from-oracle` takes the outputs from the C oracle instead, for when the reference cannot be built: its forward outputs
are bit-identical to the reference kernels' wherever the three-way test has compared them, its backward outputs agree
within the test's tolerance.  The file's `source` entry records which was used.

The committed file was made with `--from-oracle`, from the C oracle as it stood when the three-way test last ran against
oracle/_ref on a B200 and passed every case (profiles/r02/gpu_tests_v8.txt: 366 passed, none of the 5 skips in this
test); neither the oracle nor the test's inputs have changed since, so its digests are those of the reference kernels'
outputs."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from tests import test_ref_cuda_parity as T  # noqa: E402
from tests.golden.make_golden import array_digest  # noqa: E402


def main(from_oracle):
    from oracle import build_ref, pn2_ext_cpu
    if from_oracle:
        impl, dev, source = pn2_ext_cpu, "cpu", "C oracle (oracle/pn2_oracle.c)"
    else:
        impl, dev, source = build_ref.load(), "cuda", "reference CUDA kernels (oracle/_ref)"

    def run(fn, *args):
        out = getattr(impl, fn)(*[a.to(dev) if torch.is_tensor(a) else a for a in args])
        return [t.cpu() for t in out] if isinstance(out, (list, tuple)) else out.cpu()

    def digests(*ts):
        return np.array([array_digest(t) for t in ts])

    fix = {"source": np.array(source)}
    for c in T.FPS_CASES:
        fix[T.key("fps", c)] = digests(run("farthest_point_sample", T.fps_inputs(*c), c[3]))
    for c in T.BALL_CASES:
        pts, ctr = T.ball_inputs(*c)
        fix[T.key("ball", c)] = digests(*run("ball_query", pts, ctr, c[4], c[5]))
    for c in T.NN_CASES:
        q, k = T.nn_inputs(*c)
        fix[T.key("nn", c)] = digests(*run("point_search", q, k, 3))
    x, idx, g, idx3, w, g2 = T.op_inputs()
    N = x.shape[2]
    fix["group_forward"] = digests(run("group_points_forward", x, idx))
    fix["group_backward"] = T.bwd_sample(run("group_points_backward", g, idx, N))
    fix["interpolate_forward"] = digests(run("interpolate_forward", x, idx3, w))
    fix["interpolate_backward"] = T.bwd_sample(run("interpolate_backward", g2, idx3, w, N))
    np.savez_compressed(os.path.join(HERE, "ref_cuda_parity.npz"), **fix)
    print("ref_cuda_parity.npz from", source)


if __name__ == "__main__":
    main("--from-oracle" in sys.argv)
