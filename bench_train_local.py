#!/usr/bin/env python
"""TRAINING step of PN2_LOCAL (models/PointNet2_local.py, default arguments, score_classes=3) with its PointNet2Loss:
fused step (Trainer(fused=True), train_engine.LocalTrainEngine) against the module path, in the two modes of the
grasp-evaluation head:

  * given — ``local_search_frame`` (B, 12, --frames, --search): the shapes of bench_local.py, 1 024 points with 64
            candidates each (2.1 M candidate rows at 32 scenes);
  * self  — no frame input: each point's own (R, t) logits are its one candidate (--batch x 25 600 rows).

    python bench_train_local.py [--batch 32] [--frames 1024] [--search 64] [--steps 5] [--warmup 2] [--kernel-iters 50]

Inputs: --batch tabletop scenes of 25 600 points (tests.inputs.tabletop_batch); candidates and labels from
train.synthetic_local_batch; default init under manual_seed(0), dropout on (p = 0.5: element dropout on the movable
head, channel dropout on the evaluation head).  Per mode, two Trainers from the same weights (Adam): fused and module
(nn.Module stack under autograd, torch's default TF32 convolutions, as the unmodified reference runs).  Their steps
ALTERNATE in one loop, each timed with CUDA events.  Each step edits its frames in place, so it gets a fresh copy of the
pristine frames, made before its timed window.  Peak memory is max_memory_allocated over each path's steps (reset
before every step).  Losses: the first step (same weights, same data: comparable) and the last.  Then the new kernels
alone at the default configuration's shapes (CUDA events over --kernel-iters launches): the channel-dropout BatchNorm
passes over the evaluation head's rows, and the evaluation-row backward in both modes, with the bytes each must move,
computed from the shapes, over its time, next to the HBM figure bench_micro.hbm_peak() reports.  GPU name, power limit
and SM clock are read in the same run.  Prints one JSON line; writes nothing to the tree.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench_train_global import NUM_POINTS, gpu_identity, time_kernel  # noqa: E402

BF = torch.bfloat16


def timed_step(trainer, batch, labels):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    losses = trainer.step(batch, labels)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), torch.cuda.max_memory_allocated(), {k: float(v) for k, v in losses.items()}


def bench_mode(x, frames0, labels, args):
    from s4g_release_b200.network_models.models.PointNet2_local import PointNet2, PointNet2Loss
    from s4g_release_b200.train import Trainer
    B = x.shape[0]
    torch.manual_seed(0)
    fused_net = PointNet2(score_classes=3).to(x.device)
    module_net = PointNet2(score_classes=3).to(x.device)
    module_net.load_state_dict(fused_net.state_dict())
    runs = {"fused": Trainer(fused_net, PointNet2Loss(), fused=True), "module": Trainer(module_net, PointNet2Loss())}
    res = {k: {"ms": [], "peak": 0, "first_loss": None, "last_loss": None, "error": None} for k in runs}
    for i in range(args.warmup + args.steps):
        for name, tr in runs.items():
            r = res[name]
            if r["error"]:
                continue
            batch = {"scene_points": x}
            if frames0 is not None:
                batch["local_search_frame"] = frames0.clone()  # (outside the timed window: the step edits it)
            try:
                ms, peak, losses = timed_step(tr, batch, labels)
            except torch.cuda.OutOfMemoryError as e:
                r["error"] = "out of memory: %s" % str(e).splitlines()[0]
                torch.cuda.empty_cache()
                continue
            if i == 0:
                r["first_loss"] = losses
            r["last_loss"] = losses
            if i >= args.warmup:
                r["ms"].append(ms)
                r["peak"] = max(r["peak"], peak)
    out = {}
    for name, r in res.items():
        ms = sorted(r["ms"])
        med = ms[len(ms) // 2] if ms else None
        out[name] = {"ms_per_step": round(med, 3) if med else None, "ms_all": [round(v, 3) for v in r["ms"]],
                     "scenes_per_s": round(B * 1e3 / med, 2) if med else None,
                     "peak_memory_GB": round(r["peak"] / 2**30, 2), "first_step_loss": r["first_loss"],
                     "last_step_loss": r["last_loss"], "error": r["error"]}
    f, m = out["fused"]["ms_per_step"], out["module"]["ms_per_step"]
    out["speedup"] = round(m / f, 2) if f and m else None
    del runs, fused_net, module_net
    torch.cuda.empty_cache()
    return out


def bench_kernels(dev, B, F, S, iters, peak_gbs):
    """the new kernels at the default configuration's shapes: point features C = 64, evaluation head width 128"""
    from s4g_release_b200._lib import check, lib, ptr, stream_ptr
    st = stream_ptr(dev)
    g = torch.Generator(device=dev).manual_seed(0)
    N, C, H = NUM_POINTS, 64, 128
    out = {}

    def row(ms, nbytes, **shape):
        return dict(shape, us=round(ms * 1e3, 2), bytes=int(nbytes), GB_per_s=round(nbytes / ms / 1e6, 1),
                    frac_of_hbm_figure=round(nbytes / ms / 1e6 / peak_gbs, 3))

    P = B * F * S  # given mode's candidate rows
    y = torch.randn(P, H, generator=g, device=dev).to(BF)
    dz = torch.randn(P, H, generator=g, device=dev).to(BF)
    scale = torch.rand(H, generator=g, device=dev) + 0.5
    shift = torch.randn(H, generator=g, device=dev) * 0.3
    coef = torch.randn(3 * H, generator=g, device=dev)
    z = torch.empty_like(y)
    sums = torch.empty(2 * H, dtype=torch.float64, device=dev)
    ms = time_kernel(lambda: check(lib.s4g_train_bn_act_chdrop_bf16(ptr(y), ptr(scale), ptr(shift), ptr(z), P, H, 1, F * S,
                                                                     7, 0.5, st), "bn_act_chdrop"), iters)
    out["bn_act_chdrop"] = row(ms, 4 * P * H, rows=P, C=H, scene_rows=F * S)
    ms = time_kernel(lambda: check(lib.s4g_train_bn_bwd_reduce_chdrop_bf16(ptr(dz), ptr(y), ptr(scale), ptr(shift), P, H, 1,
                                                                            F * S, 7, 0.5, ptr(sums), st), "reduce_chdrop"),
                     iters)
    out["bn_bwd_reduce_chdrop"] = row(ms, 4 * P * H, rows=P, C=H, scene_rows=F * S)
    ms = time_kernel(lambda: check(lib.s4g_train_bn_bwd_apply_chdrop_bf16(ptr(dz), ptr(y), ptr(scale), ptr(shift), ptr(coef),
                                                                           ptr(coef[H:]), ptr(coef[2 * H:]), P, H, 1, F * S,
                                                                           7, 0.5, ptr(z), st), "apply_chdrop"), iters)
    out["bn_bwd_apply_chdrop"] = row(ms, 6 * P * H, rows=P, C=H, scene_rows=F * S)
    del y, dz, z
    dfeat = torch.empty(B * N, C, dtype=BF, device=dev)
    d = torch.randn(P, C + 48, generator=g, device=dev).to(BF)
    ms = time_kernel(lambda: check(lib.s4g_local_eval_rows_bwd_bf16(ptr(d), B, N, C, F, S, ptr(dfeat), None, None, st),
                                   "eval_rows_bwd"), iters)
    # reads the first C columns of every row, writes every point's feature gradient
    out["local_eval_rows_bwd_given"] = row(ms, 2 * P * C + 2 * B * N * C, B=B, N=N, C=C, F=F, S=S)
    del d
    d = torch.randn(B * N, C + 48, generator=g, device=dev).to(BF)
    dR = torch.zeros(B, 9, N, device=dev)
    dt = torch.zeros(B, 3, N, device=dev)
    ms = time_kernel(lambda: check(lib.s4g_local_eval_rows_bwd_bf16(ptr(d), B, N, C, N, 1, ptr(dfeat), ptr(dR), ptr(dt), st),
                                   "eval_rows_bwd"), iters)
    # reads the rows, writes the feature gradient, reads and writes the R / t gradients
    out["local_eval_rows_bwd_self"] = row(ms, 2 * B * N * (C + 48) + 2 * B * N * C + 2 * 4 * B * N * 12, B=B, N=N, C=C)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--search", type=int, default=64)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--kernel-iters", type=int, default=50)
    args = ap.parse_args()
    if min(args.batch, args.frames, args.search, args.steps, args.warmup, args.kernel_iters) < 1:
        ap.error("--batch, --frames, --search, --steps, --warmup and --kernel-iters must be at least 1")
    if args.frames > NUM_POINTS:
        ap.error("--frames must be at most %d" % NUM_POINTS)
    assert torch.cuda.is_available(), "bench_train_local.py needs a CUDA device (there is no CPU path)"
    from bench_micro import hbm_peak
    from s4g_release_b200.train import synthetic_local_batch
    from tests.inputs import tabletop_batch

    dev = torch.device("cuda", torch.cuda.current_device())
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.benchmark = True
    x = tabletop_batch(args.batch, n_points=NUM_POINTS).to(dev)
    peak_gbs, peak_src = hbm_peak()
    result = {"metric": "PN2_LOCAL training step, fused vs module path (25600 points/scene)",
              "gpu": gpu_identity(dev), "scenes": args.batch, "points_per_scene": NUM_POINTS, "steps": args.steps,
              "warmup": args.warmup, "dropout_prob": 0.5,
              "module_path_precision": "TF32 convolutions / matmuls (torch default for cuDNN), fp32 storage",
              "hbm_figure_GB_per_s": peak_gbs,
              "hbm_figure_source": "bench_micro.hbm_peak(): MEASURED_PEAKS.json when present, else its 6650 GB/s fallback "
                                   "(%s here)" % peak_src}
    frames, labels = synthetic_local_batch(x, args.frames, args.search)
    result["given"] = dict(bench_mode(x, frames, labels, args), n_frames=args.frames, n_search=args.search)
    del frames, labels
    _, labels = synthetic_local_batch(x, NUM_POINTS, 1)
    result["self"] = bench_mode(x, None, labels, args)
    del labels
    result["kernels"] = bench_kernels(dev, args.batch, args.frames, args.search, args.kernel_iters, peak_gbs)
    result["gpu_after"] = gpu_identity(dev)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
