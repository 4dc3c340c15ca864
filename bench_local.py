#!/usr/bin/env python
"""Fused inference of PN2_LOCAL (models/PointNet2_local.py, default arguments, score_classes=3), run with
``forward(..., fused=True)``, against its module path, in the two modes of the grasp-evaluation head:

  * self  — no frame input: each point's own (R, t) prediction is its one candidate (--batch x 25 600 candidates);
  * given — ``local_search_frame`` (B, 12, --frames, --search): --frames points with --search candidates each.  With the
            defaults 64 x 1 024 x 64 = 4.19 M candidate rows, 0.94 GB of bf16 evaluation rows.  The repository records
            no reference training value for n_frames / n_search; these shapes are chosen here.

    python bench_local.py [--batch 64] [--frames 1024] [--search 64] [--steps 10] [--warmup 2] [--kernel-iters 20]

Inputs: --batch tabletop scenes of 25 600 points (tests.inputs.tabletop_batch); weights: bench_global.seeded (default
init under manual_seed(0), BatchNorm statistics from Generator(1)) and t_logit drawn with std 0.05, so the translation
head is not identically zero.  Given candidates: rotation entries N(0, 0.25), translations within 2 cm of their point;
every step starts from the same pristine copy (the head updates the frames in place), restored outside the timed window.

Per mode, after warming up every shape (which includes the one-time plan timing of new chain shapes and the module
path's cuDNN algorithm choice), the fused step and the module-path step (cuDNN's default TF32, as the unmodified
reference runs) ALTERNATE, each timed with CUDA events after a 256 MB L2 flush.  The module path runs the largest batch
that fits (the fused batch, halved on out-of-memory).  Reported: median ms per step and per scene, peak memory
(max_memory_allocated over each path's steps, reset before each), per-stage ms from one engine.StageTimer pass (trunk =
the sum of the set-abstraction and propagation stages), the fused-vs-module error of every output on the module batch
(absolute and over max(1, max|module|)), and the row kernel alone (median over --kernel-iters launches) with the bytes
it must move, computed from the shapes, over its time, next to the HBM figure bench_micro.hbm_peak() reports.  GPU name,
power limit and SM clock are read in the same run.  Prints one JSON line per mode; writes nothing to the tree.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench_global import L2_FLUSH_BYTES, NUM_POINTS, seeded  # noqa: E402
from bench_micro import hbm_peak  # noqa: E402
from bench_train_global import gpu_identity  # noqa: E402


def make_frames(points, F, S, seed=0):
    g = torch.Generator(device=points.device).manual_seed(seed)
    B = points.shape[0]
    rot = 0.5 * torch.randn(B, 9, F, S, device=points.device, generator=g)
    t = points[:, :, :F].unsqueeze(-1) + 0.02 * torch.randn(B, 3, F, S, device=points.device, generator=g)
    return torch.cat([rot, t], dim=1).contiguous()


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


def row_kernel_bytes(B, N, C, F, S, given):
    """HBM bytes the row kernel must move: rows written, features read once per point, candidates read (and the given
    translations written back), the anchoring points read."""
    rows = B * F * S
    out = rows * (C + 48) * 2
    if given:
        return out + B * F * C * 2 + rows * 12 * 4 + rows * 3 * 4 + B * F * 3 * 4
    return out + B * N * C * 2 + B * N * 12 * 4


def bench_mode(net, scenes, frames0, args, flush):
    from s4g_release_b200.engine import FusedPointNet2Local, StageTimer
    eng = net.fused_engine()
    B, _, N = scenes.shape
    given = frames0 is not None
    F, S = (frames0.shape[2], frames0.shape[3]) if given else (N, 1)
    frames = frames0.clone() if given else None

    def batch(x, fr):
        return {"scene_points": x, "local_search_frame": fr} if fr is not None else {"scene_points": x}

    def reset():
        if given:
            frames.copy_(frames0)

    with torch.no_grad():
        # warm-up: the fused shapes, then the largest module batch that fits (and the fused path at that batch)
        for _ in range(args.warmup):
            reset()
            net(batch(scenes, frames), fused=True)
        mb = B
        while True:
            try:
                for _ in range(args.warmup):
                    reset()
                    net(batch(scenes[:mb], frames[:mb] if given else None), fused=False)
                torch.cuda.synchronize()
                break
            except torch.cuda.OutOfMemoryError:
                torch.cuda.empty_cache()
                if mb == 1:
                    raise
                mb //= 2
        xm = scenes[:mb]
        # alternate the two paths
        fused_ms, module_ms, fused_peak, module_peak = [], [], 0, 0
        for _ in range(args.steps):
            reset()
            ms, peak = timed(lambda: net(batch(scenes, frames), fused=True), flush)
            fused_ms.append(ms)
            fused_peak = max(fused_peak, peak)
            reset()
            ms, peak = timed(lambda: net(batch(xm, frames[:mb] if given else None), fused=False), flush)
            module_ms.append(ms)
            module_peak = max(module_peak, peak)
        # per-stage times
        reset()
        timer = StageTimer()
        eng.forward(scenes, frames, timer=timer)
        torch.cuda.synchronize()
        stages = {k: sum(v) for k, v in timer.totals_ms().items()}
        heads = {k: round(v, 4) for k, v in stages.items() if k.startswith("heads.")}
        stage_ms = dict(trunk=round(sum(v for k, v in stages.items() if not k.startswith("heads.")), 4), **heads)
        # fused vs module on the module batch, each from its own copy of the frames
        fa = frames0[:mb].clone() if given else None
        fb = frames0[:mb].clone() if given else None
        got = net(batch(xm, fa), fused=True)
        ref = net(batch(xm, fb), fused=False)
        torch.cuda.synchronize()
        err = {k: {"abs": (got[k].float() - ref[k].float()).abs().max().item(),
                   "rel": (got[k].float() - ref[k].float()).abs().max().item() / max(1.0, ref[k].abs().max().item())}
               for k in ref}
        frames_equal = bool(torch.equal(fa, fb)) if given else None
        del got, ref, fa, fb
        # the row kernel alone, on rows of the trunk's width
        C = eng.head_chains[0].all_cin[0]
        g = torch.Generator(device=scenes.device).manual_seed(2)
        feat = torch.randn(B * N, C, device=scenes.device, generator=g).to(torch.bfloat16)
        R = torch.randn(B, 9, N, device=scenes.device, generator=g)
        t = torch.randn(B, 3, N, device=scenes.device, generator=g)
        run = lambda: FusedPointNet2Local.local_eval_rows(feat, scenes, frames, R, t)  # noqa: E731
        run()
        kernel_ms = median([timed(run, flush)[0] for _ in range(args.kernel_iters)])
    nbytes = row_kernel_bytes(B, N, C, F, S, given)
    peak_gbs, peak_src = hbm_peak()
    fused_step, module_step = median(fused_ms), median(module_ms)
    return {"mode": "given" if given else "self", "batch": B, "points_per_scene": N, "n_frames": F, "n_search": S,
            "candidate_rows": B * F * S, "eval_row_bytes": B * F * S * (C + 48) * 2,
            "fused": {"ms_per_step": round(fused_step, 4), "ms_per_scene": round(fused_step / B, 4),
                      "peak_gb": round(fused_peak / 1e9, 2), "stages_ms": stage_ms, "tolerance": eng.tolerance()},
            "module": {"batch": mb, "ms_per_step": round(module_step, 4), "ms_per_scene": round(module_step / mb, 4),
                       "peak_gb": round(module_peak / 1e9, 2)},
            "speedup_per_scene": round((module_step / mb) / (fused_step / B), 2),
            "max_err": err, "frames_after_equal": frames_equal,
            "row_kernel": {"ms": round(kernel_ms, 4), "bytes": nbytes, "gb_per_s": round(nbytes / kernel_ms / 1e6, 1),
                           "hbm_gb_per_s": peak_gbs, "hbm_source": peak_src,
                           "fraction_of_hbm": round(nbytes / kernel_ms / 1e6 / peak_gbs, 3)}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--search", type=int, default=64)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--kernel-iters", type=int, default=20)
    args = ap.parse_args()
    if min(args.batch, args.frames, args.search, args.steps, args.warmup, args.kernel_iters) < 1:
        ap.error("every count must be at least 1")
    if args.frames > NUM_POINTS:
        ap.error("--frames must be at most %d" % NUM_POINTS)
    assert torch.cuda.is_available(), "bench_local.py needs a CUDA device (there is no CPU path)"
    from s4g_release_b200.network_models.models.PointNet2_local import PointNet2
    from tests.inputs import tabletop_batch

    dev = torch.device("cuda", torch.cuda.current_device())
    net = seeded(PointNet2)
    torch.nn.init.normal_(net.t_logit.weight, std=0.05, generator=torch.Generator().manual_seed(3))
    net = net.to(dev)
    if not net.fusable(allow_global=True):
        raise RuntimeError("PN2_LOCAL's default configuration has no fused plan")
    scenes = tabletop_batch(args.batch, n_points=NUM_POINTS).to(dev)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    for frames in (None, make_frames(scenes, args.frames, args.search)):
        result = bench_mode(net, scenes, frames, args, flush)
        result = dict(metric="PN2_LOCAL fused inference vs module path (%s mode)" % result["mode"],
                      gpu=gpu_identity(dev), **result)
        print(json.dumps(result), flush=True)
        del frames
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
