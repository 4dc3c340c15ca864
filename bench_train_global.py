#!/usr/bin/env python
"""TRAINING step of the configurations whose last set-abstraction level is one global group (num_centroids = 0) paired
with a broadcast first propagation level (num_fp_neighbours = 0): fused step against the module path.

  * class_default — PointNet2_tcls.PointNet2(score_classes=3) with PointNet2_tcls.PointNet2Loss;
  * pn2_sibling   — models.PointNet2.PointNet2(score_classes=3) with its PointNet2Loss (continuous translation labels).

    python bench_train_global.py [--batch 32] [--steps 5] [--warmup 2] [--kernel-iters 50]

Inputs: --batch tabletop scenes of 25 600 points (tests.inputs.tabletop_batch), synthetic labels of 4 000 frames
(train.synthetic_labels); default init under manual_seed(0).  Per configuration, two Trainers from the same weights (Adam,
dropout on): fused (train_engine.TrainEngine) and module (nn.Module stack under autograd; torch's default TF32 convolutions,
as the unmodified reference runs).  Their steps ALTERNATE in one loop, each timed with CUDA events; peak memory is
torch's max_memory_allocated over each path's steps (reset before every step, so it includes the other path's
parameters and optimiser state, a few hundred MB).  Losses: the first step (same weights, same data: comparable) and the
last.  Then the new kernels alone (CUDA events over --kernel-iters launches, inputs written before the timed loop) at
the shapes the class defaults produce at this batch, and one large global pool (32 x 25 600 rows x 1 024 channels), with
algorithmic bytes / time next to the HBM figure bench_micro.py uses.  GPU name, power limit and SM clock are read in the
same run.  Prints one JSON line; writes nothing to the tree.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

NUM_POINTS = 25600
BF = torch.bfloat16


def gpu_identity(dev):
    info = {"name": torch.cuda.get_device_name(dev), "power_limit_w": None, "sm_clock_mhz": None, "sm_clock_max_mhz": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=power.limit,clocks.sm,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        p, c, m = [float(v) for v in out.strip().splitlines()[0].split(",")]
        info.update(power_limit_w=p, sm_clock_mhz=c, sm_clock_max_mhz=m)
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def timed_step(trainer, x, y):
    torch.cuda.reset_peak_memory_stats()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    losses = trainer.step({"scene_points": x}, y)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), torch.cuda.max_memory_allocated(), {k: float(v) for k, v in losses.items()}


def bench_config(cls, loss_cls, sibling, x, y, args):
    from s4g_release_b200.train import Trainer
    B = x.shape[0]
    torch.manual_seed(0)
    fused_net = cls(score_classes=3).to(x.device)
    module_net = cls(score_classes=3).to(x.device)
    module_net.load_state_dict(fused_net.state_dict())
    runs = {"fused": Trainer(fused_net, loss_cls(), fused=True), "module": Trainer(module_net, loss_cls())}
    res = {k: {"ms": [], "peak": 0, "first_loss": None, "last_loss": None, "error": None} for k in runs}
    for i in range(args.warmup + args.steps):
        for name, tr in runs.items():
            r = res[name]
            if r["error"]:
                continue
            try:
                ms, peak, losses = timed_step(tr, x, y)
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
    if sibling:
        out["labels"] = "best_frame_t continuous (synthetic_labels(continuous_t=True))"
    del runs, fused_net, module_net
    torch.cuda.empty_cache()
    return out


def time_kernel(fn, iters):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def bench_kernels(dev, B, iters, peak_gbs):
    from s4g_release_b200._lib import check, lib, ptr, stream_ptr
    from s4g_release_b200.train_engine import rows_segment_sum
    st = stream_ptr(dev)
    g = torch.Generator(device=dev).manual_seed(0)
    out = {}

    def row(ms, nbytes, **shape):
        return dict(shape, us=round(ms * 1e3, 2), bytes=int(nbytes), GB_per_s=round(nbytes / ms / 1e6, 1),
                    frac_of_hbm_figure=round(nbytes / ms / 1e6 / peak_gbs, 3))

    # (the class defaults: the global level pools B scenes x 128 points x 1 024 channels; its broadcast level's rows are
    # [global 1 024 | skip 256] wide)
    for name, (Bs, N, C) in (("segmax_class_default", (B, 128, 1024)), ("segmax_large_N", (32, NUM_POINTS, 1024))):
        y = torch.randn(Bs * N, C, generator=g, device=dev).to(BF)
        scale = torch.rand(C, generator=g, device=dev) + 0.5
        shift = torch.randn(C, generator=g, device=dev) * 0.3
        z = torch.empty((Bs, C), dtype=BF, device=dev)
        arg = torch.empty((Bs, C), dtype=torch.int32, device=dev)
        ymax = torch.empty((Bs, C), dtype=BF, device=dev)
        work = torch.empty((Bs, C), dtype=torch.int64, device=dev)
        ms = time_kernel(lambda: check(lib.s4g_train_bn_act_segmax_bf16(ptr(y), ptr(scale), ptr(shift), ptr(z), ptr(arg),
                                                                         ptr(ymax), ptr(work), Bs, N, C, 1, st), "segmax"), iters)
        out[name] = row(ms, 2 * Bs * N * C + Bs * C * (2 + 4 + 2), B=Bs, N=N, C=C)
        dz = torch.randn(Bs, C, generator=g, device=dev).to(BF)
        coef = torch.randn(3 * C, generator=g, device=dev)
        dy = torch.empty_like(y)
        P = Bs * N
        ms = time_kernel(lambda: check(lib.s4g_train_bn_bwd_apply_seg_bf16(ptr(dz), ptr(arg), N, ptr(y), ptr(scale), ptr(shift),
                                                                            ptr(coef), ptr(coef[C:]), ptr(coef[2 * C:]), P, C, 1,
                                                                            ptr(dy), st), "apply_seg"), iters)
        out[name.replace("segmax", "bn_bwd_apply_seg")] = row(ms, 4 * P * C + Bs * C * 6, B=Bs, N=N, C=C)
        sums = torch.empty(2 * C, dtype=torch.float64, device=dev)
        ms = time_kernel(lambda: check(lib.s4g_train_bn_bwd_reduce_seg_bf16(ptr(dz), ptr(arg), N, ptr(y), ptr(scale), ptr(shift),
                                                                             P, C, 1, ptr(sums), st), "reduce_seg"), iters)
        out[name.replace("segmax", "bn_bwd_reduce_seg_dense")] = row(ms, 2 * P * C + Bs * C * 6, B=Bs, N=N, C=C)
        del y, dy
    Nq, c2, c1 = 128, 1024, 256
    dzr = torch.randn(B * Nq, c2 + c1, generator=g, device=dev).to(BF)
    acc = torch.zeros((B, c2), device=dev)
    ms = time_kernel(lambda: rows_segment_sum(dzr, B, Nq, c2, acc), iters)
    out["rows_segment_sum_class_default"] = row(ms, 2 * B * Nq * c2 + 8 * B * c2, B=B, Nq=Nq, c2=c2, ld=c2 + c1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--num-frame", type=int, default=4000)
    ap.add_argument("--kernel-iters", type=int, default=50)
    args = ap.parse_args()
    if min(args.batch, args.steps, args.warmup, args.kernel_iters) < 1:
        ap.error("--batch, --steps, --warmup and --kernel-iters must be at least 1")
    assert torch.cuda.is_available(), "bench_train_global.py needs a CUDA device (there is no CPU path)"
    from bench_micro import hbm_peak
    from s4g_release_b200.network_models.models import PointNet2, PointNet2_tcls
    from s4g_release_b200.train import synthetic_labels
    from tests.inputs import tabletop_batch

    dev = torch.device("cuda", torch.cuda.current_device())
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.benchmark = True
    x = tabletop_batch(args.batch, n_points=NUM_POINTS).to(dev)
    peak_gbs, peak_src = hbm_peak()
    result = {"metric": "training step with a global set-abstraction level, fused vs module path (25600 points/scene)",
              "gpu": gpu_identity(dev), "scenes": args.batch, "points_per_scene": NUM_POINTS, "steps": args.steps,
              "warmup": args.warmup,
              "module_path_precision": "TF32 convolutions / matmuls (torch default for cuDNN), fp32 storage",
              "hbm_figure_GB_per_s": peak_gbs,
              "hbm_figure_source": "bench_micro.hbm_peak(): MEASURED_PEAKS.json when present, else its 6650 GB/s fallback "
                                   "(%s here)" % peak_src}
    for name, cls, loss_cls, sibling in (
            ("class_default", PointNet2_tcls.PointNet2, PointNet2_tcls.PointNet2Loss, False),
            ("pn2_sibling", PointNet2.PointNet2, PointNet2.PointNet2Loss, True)):
        y = synthetic_labels(args.batch, NUM_POINTS, args.num_frame, 2000, device=dev, continuous_t=sibling)
        result[name] = bench_config(cls, loss_cls, sibling, x, y, args)
    result["kernels"] = bench_kernels(dev, args.batch, args.kernel_iters, peak_gbs)
    result["gpu_after"] = gpu_identity(dev)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
