#!/usr/bin/env python
"""Fused inference of EDGEPN2D (models/EdgePointNet2Down.py, default arguments, score_classes=3), run with
``forward(..., fused=True)``, against its module path, with the PN2 sibling of the same shapes on the fused engine as the
cost floor (the same trunk with plain set-abstraction levels, the same heads).

    python bench_edge.py [--batch 64] [--steps 10] [--warmup 2] [--kernel-iters 20]

Inputs: --batch tabletop scenes of 25 600 points (tests.inputs.tabletop_batch); weights: bench_global.seeded (default
init under manual_seed(0), BatchNorm statistics from Generator(1)) for both models.

After warming up every shape (which includes the one-time plan timing of new chain shapes and the module path's cuDNN
algorithm choice), the EDGEPN2D fused step, its module-path step (cuDNN's default TF32, as the unmodified reference runs)
and the PN2 sibling's fused step ALTERNATE, each timed with CUDA events after a 256 MB L2 flush.  The module path runs
the largest batch that fits (the fused batch, halved on out-of-memory).  Reported: median ms per step and per scene,
peak memory, per-stage ms of one engine.StageTimer pass, the fused-vs-module error of every output on the module batch
(absolute and over max(1, max|module|)), and per edge level its three launches alone (centroid rows, term chain, edge
chain; median over --kernel-iters) next to the plain gathered chain of the same shape and weights (what a level without
the centroid term costs).  The PN2 sibling's fused-vs-module error on the same batch is reported beside EDGEPN2D's: the
error of the bf16 engine without edge levels.  GPU name, power limit and SM clock are read in the same run.  Prints one
JSON line; writes nothing to the tree.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench_global import L2_FLUSH_BYTES, NUM_POINTS, seeded  # noqa: E402
from bench_train_global import gpu_identity  # noqa: E402


def timed(fn, flush):
    """(ms, peak bytes) of one call, CUDA events after an L2 flush"""
    flush.zero_()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), torch.cuda.max_memory_allocated()


def median(v):
    return sorted(v)[len(v) // 2]


def edge_levels_alone(eng, scenes, args, flush):
    """Per edge level: its three launches on the level's real inputs, and the plain gathered chain of the same shape."""
    from s4g_release_b200.chain import IN_GATHER, OUT_MAXPOOL
    with torch.no_grad():
        _, trace = eng.forward(scenes, return_trace=True)
    xyz = [scenes.float().contiguous()]
    for idx in trace["fps"]:
        xyz.append(eng.gather_xyz(xyz[-1], idx))
    out = {}
    for i, edge in enumerate(eng.edge_levels):
        if not edge:
            continue
        f = trace["sa_feature"][i - 1]
        feat = f.reshape(-1, f.shape[-1]).to(torch.bfloat16).contiguous()  # the bf16 rows the level read
        idx, nbr = trace["fps"][i], trace["ball"][i]
        chain, term_chain = eng.sa_chains[i], eng._term_chains[i]
        plain = eng._make_chain(chain_layers(eng, i), IN_GATHER, feat.shape[1], OUT_MAXPOOL,
                                group=eng.cfg["num_neighbours"][i])

        def three():
            term = term_chain.run_rows(eng.gather_rows(feat, idx))
            return chain.run_gather(feat, xyz[i], xyz[i + 1], nbr, term)

        three()
        plain.run_gather(feat, xyz[i], xyz[i + 1], nbr)
        edge_ms = median([timed(three, flush)[0] for _ in range(args.kernel_iters)])
        plain_ms = median([timed(lambda: plain.run_gather(feat, xyz[i], xyz[i + 1], nbr), flush)[0]
                           for _ in range(args.kernel_iters)])
        rows = nbr.numel()
        out["sa%d" % i] = {"rows": rows, "feat_c": feat.shape[1], "edge_three_launches_ms": round(edge_ms, 4),
                           "plain_chain_ms": round(plain_ms, 4), "edge_over_plain": round(edge_ms / plain_ms, 3)}
    return out


def max_err(model, batch):
    """fused vs module path of every output: absolute and over max(1, max|module|)"""
    got = model(batch, fused=True)
    ref = model(batch, fused=False)
    torch.cuda.synchronize()
    return {k: {"abs": (got[k].float() - ref[k].float()).abs().max().item(),
                "rel": (got[k].float() - ref[k].float()).abs().max().item() / max(1.0, ref[k].abs().max().item())}
            for k in ref}


def chain_layers(eng, i):
    """(W, shift, relu) of edge level i's chain as the engine built it: first layer [W_x | W_a + W_b]"""
    (w0, b0), rest = eng.sa[i][0], eng.sa[i][1:]
    w_plain, _ = eng.split_edge_layer(w0, (w0.shape[1] - 3) // 2)
    return [(w_plain, b0, True)] + [(w, b, True) for w, b in rest]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--kernel-iters", type=int, default=20)
    args = ap.parse_args()
    if min(args.batch, args.steps, args.warmup, args.kernel_iters) < 1:
        ap.error("every count must be at least 1")
    assert torch.cuda.is_available(), "bench_edge.py needs a CUDA device (there is no CPU path)"
    from s4g_release_b200.engine import StageTimer
    from s4g_release_b200.network_models.models.EdgePointNet2Down import EdgePointNet2Down
    from s4g_release_b200.network_models.models.PointNet2 import PointNet2
    from tests.inputs import tabletop_batch

    dev = torch.device("cuda", torch.cuda.current_device())
    net = seeded(EdgePointNet2Down).to(dev)
    sibling = seeded(PointNet2).to(dev)
    if not net.fusable(allow_global=True):
        raise RuntimeError("EDGEPN2D's default configuration has no fused plan")
    scenes = tabletop_batch(args.batch, n_points=NUM_POINTS).to(dev)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    B = scenes.shape[0]
    batch = {"scene_points": scenes}
    with torch.no_grad():
        for _ in range(args.warmup):
            net(batch, fused=True)
            sibling(batch, fused=True)
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
        fused_ms, module_ms, sib_ms, fused_peak, module_peak = [], [], [], 0, 0
        for _ in range(args.steps):
            ms, peak = timed(lambda: net(batch, fused=True), flush)
            fused_ms.append(ms)
            fused_peak = max(fused_peak, peak)
            ms, peak = timed(lambda: net(xm, fused=False), flush)
            module_ms.append(ms)
            module_peak = max(module_peak, peak)
            sib_ms.append(timed(lambda: sibling(batch, fused=True), flush)[0])
        eng = net.fused_engine()
        timer = StageTimer()
        eng.forward(scenes, timer=timer)
        torch.cuda.synchronize()
        stages = {k: round(sum(v), 4) for k, v in timer.totals_ms().items()}
        err = {name: max_err(model, xm) for name, model in (("edgepn2d", net), ("pn2_sibling", sibling))}
    levels = edge_levels_alone(eng, scenes, args, flush)
    fused_step, module_step, sib_step = median(fused_ms), median(module_ms), median(sib_ms)
    result = {"metric": "EDGEPN2D fused inference vs module path and the PN2 sibling fused", "gpu": gpu_identity(dev),
              "batch": B, "points_per_scene": NUM_POINTS,
              "fused": {"ms_per_step": round(fused_step, 4), "ms_per_scene": round(fused_step / B, 4),
                        "peak_gb": round(fused_peak / 1e9, 2), "stages_ms": stages, "tolerance": eng.tolerance()},
              "module": {"batch": mb, "ms_per_step": round(module_step, 4), "ms_per_scene": round(module_step / mb, 4),
                         "peak_gb": round(module_peak / 1e9, 2)},
              "pn2_sibling_fused": {"ms_per_step": round(sib_step, 4), "ms_per_scene": round(sib_step / B, 4)},
              "speedup_per_scene": round((module_step / mb) / (fused_step / B), 2),
              "edge_over_sibling": round(fused_step / sib_step, 3),
              "max_err": err, "edge_levels": levels}
    print(json.dumps(result), flush=True)


if __name__ == "__main__":
    main()
