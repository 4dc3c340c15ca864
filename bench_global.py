#!/usr/bin/env python
"""Fused inference of the configurations whose last set-abstraction level is one global group (num_centroids = 0)
paired with a broadcast first propagation level (num_fp_neighbours = 0), run with ``forward(..., fused=True)``:

  * class_default — PointNet2_tcls.PointNet2(score_classes=3): 10240 / 1024 / 128 / global centroids;
  * pn2_sibling   — models.PointNet2.PointNet2(score_classes=3): the same encoder / decoder, 6-D rotation head.

    python bench_global.py [--batch 64] [--steps 20] [--warmup 3] [--module-steps 3]

Inputs: --batch tabletop scenes of 25 600 points (tests.inputs.tabletop_batch); weights: default init under
manual_seed(0), BatchNorm statistics from Generator(1), as bench.py seeds PN2_CLS.  Per configuration:
  fused      ms/step and scenes/s of the engine's forward on device-resident inputs (CUDA events per step, a 256 MB
             buffer written between steps so no step starts with the previous one's data in L2), and per-stage ms
             from a separate pass with engine.StageTimer;
  module     the module path (fused=False, eval, no_grad) at the largest batch that fits — the fused batch, halved on
             out-of-memory — with its ms per scene and scenes/s;
  max_err    max |fused - module| of every output on the module batch's scenes, absolute and over max(1, max|module|).
The GPU's name and power limit are read in the same run.  Prints one JSON line; writes nothing to the tree.
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
L2_FLUSH_BYTES = 256 << 20


def seeded(cls):
    torch.manual_seed(0)
    net = cls(score_classes=3)
    g = torch.Generator().manual_seed(1)
    for m in net.modules():
        if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
            n = m.num_features
            m.weight.data = torch.rand(n, generator=g) + 0.5
            m.bias.data = torch.randn(n, generator=g) * 0.1
            m.running_mean.data = torch.randn(n, generator=g) * 0.1
            m.running_var.data = torch.rand(n, generator=g) + 0.5
    return net.eval()


def gpu_identity(dev):
    info = {"name": torch.cuda.get_device_name(dev), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=power.limit",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        info["power_limit_w"] = float(out.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def time_steps(run, steps, flush):
    ms = []
    for _ in range(steps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return sorted(ms)[len(ms) // 2]


def bench_config(name, cls, scenes, args, flush):
    from s4g_release_b200.engine import StageTimer
    net = seeded(cls).to(scenes.device)
    if not net.fusable(allow_global=True) or net.fusable():
        raise RuntimeError("%s: expected a configuration that is fused only on request" % name)
    B = scenes.shape[0]
    eng = net.fused_engine()
    with torch.no_grad():
        for _ in range(args.warmup):
            eng.forward(scenes)
        torch.cuda.synchronize()
        fused_ms = time_steps(lambda: eng.forward(scenes), args.steps, flush)
        timer = StageTimer()
        eng.forward(scenes, timer=timer)
        torch.cuda.synchronize()
        stages = {k: round(sum(v), 4) for k, v in timer.totals_ms().items()}

        mb, module_ms, ref = B, None, None
        while mb >= 1:
            try:
                x = scenes[:mb]
                ref = net({"scene_points": x}, fused=False)
                torch.cuda.synchronize()
                module_ms = time_steps(lambda: net({"scene_points": x}, fused=False), args.module_steps, flush)
                break
            except torch.cuda.OutOfMemoryError:
                ref = None
                torch.cuda.empty_cache()
                mb //= 2
        if ref is None:
            raise RuntimeError("%s: the module path does not fit one scene" % name)
        got = net({"scene_points": scenes[:mb]}, fused=True)
        torch.cuda.synchronize()
    err = {k: {"abs": (got[k].float() - ref[k].float()).abs().max().item(),
               "rel": (got[k].float() - ref[k].float()).abs().max().item() / max(1.0, ref[k].abs().max().item())}
           for k in ref}
    return {"fused": {"batch": B, "ms_per_step": round(fused_ms, 4), "scenes_per_s": round(B * 1e3 / fused_ms, 1),
                      "stages_ms": stages, "tolerance": eng.tolerance()},
            "module": {"batch": mb, "ms_per_scene": round(module_ms / mb, 4),
                       "scenes_per_s": round(mb * 1e3 / module_ms, 2)},
            "speedup_per_scene": round((module_ms / mb) / (fused_ms / B), 2),
            "max_err": err}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--module-steps", type=int, default=3)
    args = ap.parse_args()
    if min(args.batch, args.steps, args.module_steps) < 1:
        ap.error("--batch, --steps and --module-steps must be at least 1")
    assert torch.cuda.is_available(), "bench_global.py needs a CUDA device (there is no CPU path)"
    from s4g_release_b200.network_models.models.PointNet2 import PointNet2 as Sibling
    from s4g_release_b200.network_models.models.PointNet2_tcls import PointNet2
    from tests.inputs import tabletop_batch

    dev = torch.device("cuda", torch.cuda.current_device())
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    scenes = tabletop_batch(args.batch, n_points=NUM_POINTS).to(dev)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    result = {"metric": "fused inference with a global set-abstraction level, scenes/s (25600 points/scene)",
              "gpu": gpu_identity(dev), "points_per_scene": NUM_POINTS, "steps": args.steps}
    for name, cls in (("class_default", PointNet2), ("pn2_sibling", Sibling)):
        result[name] = bench_config(name, cls, scenes, args, flush)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
