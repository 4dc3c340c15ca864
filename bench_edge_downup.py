#!/usr/bin/env python
"""Fused inference of EDGEPN2DU (models/EdgePointNet2DownUp.py, default arguments, score_classes=3), run with
``forward(..., fused=True)``, against its module path, with EDGEPN2D (the same encoder, plain propagation levels, four
heads) on the fused engine as the floor.

    python bench_edge_downup.py [--batch 64] [--steps 10] [--warmup 2] [--kernel-iters 20]

Inputs: --batch tabletop scenes of 25 600 points (tests.inputs.tabletop_batch); weights: bench_global.seeded (default
init under manual_seed(0), BatchNorm statistics from Generator(1)) for both models.

After warming up every shape (which includes the one-time plan timing of new chain shapes and the module path's cuDNN
algorithm choice), the EDGEPN2DU fused step, its module-path step (cuDNN's default TF32, as the unmodified reference
runs) and EDGEPN2D's fused step ALTERNATE, each timed with CUDA events after a 256 MB L2 flush.  The module path runs the
largest batch that fits (the fused batch, halved on out-of-memory).  Reported: median ms per step and per scene, peak
memory, per-stage ms of one engine.StageTimer pass (per edge propagation level: fpK.uv, fpK.term, fpK.edge_rows, fpK.mlp,
fpK.mean), the fused-vs-module error of both outputs on the module batch (absolute and over max(1, max|module|)), and per
edge propagation level the two new kernels alone (median over --kernel-iters, L2 flushed before each) on the level's
real 3-NN on the benchmark's scenes and random bf16 rows of its shape, with the bytes each must move at least and the
rate:
  edge_interp_rows  the [U | V] table once (B Nk 2C bf16), per query its indices and weights (24 B) and its T row (C bf16;
                    the finest level reads 12 B of fp32 coordinates instead), and the output (B Nq 3 C bf16);
  rows_group_mean   B Nq 3 C bf16 in, B Nq C bf16 out.
GPU name, power limit and SM clock are read in the same run.  Prints one JSON line; writes nothing to the tree.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench_edge import median, timed  # noqa: E402
from bench_global import L2_FLUSH_BYTES, NUM_POINTS, seeded  # noqa: E402
from bench_train_global import gpu_identity  # noqa: E402


def max_err(model, batch):
    """fused vs module path of every output: absolute and over max(1, max|module|)"""
    got = model(batch, fused=True)
    ref = model(batch, fused=False)
    torch.cuda.synchronize()
    return {k: {"abs": (got[k].float() - ref[k].float()).abs().max().item(),
                "rel": (got[k].float() - ref[k].float()).abs().max().item() / max(1.0, ref[k].abs().max().item())}
            for k in ref}


def edge_kernels_alone(eng, scenes, args, flush):
    """Per edge propagation level: the row kernel and the mean alone, on the level's real 3-NN."""
    with torch.no_grad():
        _, trace = eng.forward(scenes, return_trace=True)
    xyz = [scenes.float().contiguous()]
    for idx in trace["fps"]:
        xyz.append(eng.gather_xyz(xyz[-1], idx))
    n_sa = len(eng.sa)
    g = torch.Generator(device=scenes.device).manual_seed(0)
    out = {}
    for i, edge in enumerate(eng.edge_fp):
        if not edge:
            continue
        dense_xyz, sparse_xyz = xyz[n_sa - 1 - i], xyz[n_sa - i]
        B, Nq, Nk = dense_xyz.shape[0], dense_xyz.shape[2], sparse_xyz.shape[2]
        uv_chain, term_chain, shift, w_xyz = eng._edge_fp[i]
        C = shift.shape[0]
        idx3, w = eng.three_nn_weights(dense_xyz, sparse_xyz)
        uv = torch.randn(B * Nk, 2 * C, device=scenes.device, generator=g).to(torch.bfloat16)
        t_rows = None
        if term_chain is not None:
            t_rows = torch.randn(B * Nq, C, device=scenes.device, generator=g).to(torch.bfloat16)

        def rows():
            return eng.edge_interp_rows(uv, idx3, w, t_rows, dense_xyz if t_rows is None else None, w_xyz, shift, B, Nk,
                                        Nq)

        x = rows()
        eng.rows_group_mean(x)
        rows_ms = median([timed(rows, flush)[0] for _ in range(args.kernel_iters)])
        mean_ms = median([timed(lambda: eng.rows_group_mean(x), flush)[0] for _ in range(args.kernel_iters)])
        rows_bytes = B * Nk * 2 * C * 2 + B * Nq * (24 + (C * 2 if t_rows is not None else 12)) + B * Nq * 3 * C * 2
        mean_bytes = B * Nq * 3 * C * 2 + B * Nq * C * 2
        out["fp%d" % i] = {"B": B, "Nq": Nq, "Nk": Nk, "cout0": C, "edge_rows": B * Nq * 3,
                           "skip": "bf16 rows" if t_rows is not None else "cloud (fp32)",
                           "edge_interp_rows": {"ms": round(rows_ms, 4), "gb": round(rows_bytes / 1e9, 4),
                                                "tb_per_s": round(rows_bytes / rows_ms / 1e9, 3)},
                           "rows_group_mean": {"ms": round(mean_ms, 4), "gb": round(mean_bytes / 1e9, 4),
                                               "tb_per_s": round(mean_bytes / mean_ms / 1e9, 3)}}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--kernel-iters", type=int, default=20)
    args = ap.parse_args()
    if min(args.batch, args.steps, args.warmup, args.kernel_iters) < 1:
        ap.error("every count must be at least 1")
    assert torch.cuda.is_available(), "bench_edge_downup.py needs a CUDA device (there is no CPU path)"
    from s4g_release_b200.engine import StageTimer
    from s4g_release_b200.network_models.models.EdgePointNet2Down import EdgePointNet2Down
    from s4g_release_b200.network_models.models.EdgePointNet2DownUp import EdgePointNet2DownUp
    from tests.inputs import tabletop_batch

    dev = torch.device("cuda", torch.cuda.current_device())
    net = seeded(EdgePointNet2DownUp).to(dev)
    floor = seeded(EdgePointNet2Down).to(dev)
    if not net.fusable(allow_global=True):
        raise RuntimeError("EDGEPN2DU's default configuration has no fused plan")
    scenes = tabletop_batch(args.batch, n_points=NUM_POINTS).to(dev)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    B = scenes.shape[0]
    batch = {"scene_points": scenes}
    with torch.no_grad():
        for _ in range(args.warmup):
            net(batch, fused=True)
            floor(batch, fused=True)
        mb = B
        while True:
            try:
                for _ in range(args.warmup):
                    net({"scene_points": scenes[:mb]}, fused=False)
                torch.cuda.synchronize()
                break
            except torch.cuda.OutOfMemoryError:
                torch.cuda.empty_cache()
                if mb == 1:
                    raise
                mb //= 2
        xm = {"scene_points": scenes[:mb]}
        fused_ms, module_ms, floor_ms, fused_peak, module_peak, floor_peak = [], [], [], 0, 0, 0
        for _ in range(args.steps):
            ms, peak = timed(lambda: net(batch, fused=True), flush)
            fused_ms.append(ms)
            fused_peak = max(fused_peak, peak)
            ms, peak = timed(lambda: net(xm, fused=False), flush)
            module_ms.append(ms)
            module_peak = max(module_peak, peak)
            ms, peak = timed(lambda: floor(batch, fused=True), flush)
            floor_ms.append(ms)
            floor_peak = max(floor_peak, peak)
        eng = net.fused_engine()
        timer = StageTimer()
        eng.forward(scenes, timer=timer)
        torch.cuda.synchronize()
        stages = {k: round(sum(v), 4) for k, v in timer.totals_ms().items()}
        err = max_err(net, xm)
    kernels = edge_kernels_alone(eng, scenes, args, flush)
    fused_step, module_step, floor_step = median(fused_ms), median(module_ms), median(floor_ms)
    result = {"metric": "EDGEPN2DU fused inference vs module path, EDGEPN2D fused as the floor", "gpu": gpu_identity(dev),
              "batch": B, "points_per_scene": NUM_POINTS,
              "fused": {"ms_per_step": round(fused_step, 4), "ms_per_scene": round(fused_step / B, 4),
                        "peak_gb": round(fused_peak / 1e9, 2), "stages_ms": stages, "tolerance": eng.tolerance()},
              "module": {"batch": mb, "ms_per_step": round(module_step, 4), "ms_per_scene": round(module_step / mb, 4),
                         "peak_gb": round(module_peak / 1e9, 2)},
              "edgepn2d_fused": {"ms_per_step": round(floor_step, 4), "ms_per_scene": round(floor_step / B, 4),
                                 "peak_gb": round(floor_peak / 1e9, 2)},
              "speedup_per_scene": round((module_step / mb) / (fused_step / B), 2),
              "downup_over_edgepn2d": round(fused_step / floor_step, 3),
              "max_err": err, "edge_fp_kernels": kernels}
    print(json.dumps(result), flush=True)


if __name__ == "__main__":
    main()
