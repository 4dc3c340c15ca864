#!/usr/bin/env python
"""Headline benchmark: S4G (PN2_CLS) inference scenes/s on B200 — BASELINE.json config[1]:
batch 64 synthetic single-view tabletop clouds at the reference's num_points (25 600) per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (the whole PN2_CLS forward: FPS, ball query, fused SA / FP / head
MLP chains) over one batch.  `value` = scenes/s with the inputs already resident in HBM, timed with
CUDA events on the launching stream (per-step event pairs, L2 flushed between steps, max over ranks).
`e2e` = the same metric through the public module API with HOST buffers: pinned host -> device copy of
the clouds, forward, device -> pinned host copy of the four prediction tensors, every step (the public call takes
the pinned result buffers — `model(batch, host_out=...)` — so each head's copy overlaps the next head's compute).
Weak scaling: each rank owns its own 64 scenes, no collective on the data path (SURVEY.md §8e).
`--steps` sets the number of timed steps of the device-resident and the end-to-end loops.  `--dump-outputs DIR` writes the
predictions of the last device-resident step (rank 0) as DIR/<name>.npy in float32: inputs and weights are seeded, so
two builds can be compared output for output.

`--impl reference` times the reference model on the box's HOST cores: the UNMODIFIED reference python modules
(staged under baseline/_ref; the bit-identical oracle restatement when they are not staged) on the C restatement of
its CUDA-only ops (the reference has no CPU implementation of those), each step a bounded sample (1 scene) of the
same workload.  Host threads are pinned (OMP / torch, at most 16: more threads measured SLOWER on this op mix).

Extra blocks in the JSON line (VERDICT r1):
  roofline        the dominant kernel TYPE of the step — mlp_chain_kernel, all its launches — against the measured bf16
                  burst peak, with its DRAM traffic (ncu) and tensor-pipe-active % beside it;
  roofline_fps    the single longest launch (level-0 farthest point sampling): FP32-issue fraction, actual HBM fraction;
  kernels         every stage: `frac` is against the bound that applies (tensor / hbm on THIS implementation's bytes /
                  fp32 issue) and never a scan-bytes figure; `hbm_frac_actual`, `traffic_ratio` from the committed ncu list;
  parity          scene 0 of the batch, fused GPU output vs the fp32 CPU oracle (scores, decisions, rotations, translations);
  reference_cuda  the unmodified reference model on ITS OWN CUDA kernels (oracle/_ref) timed on this GPU: the honest
                  competitor row (SURVEY §8d); the CPU arm is a stated baseline, not the target.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CPU_THREADS = max(1, min(16, os.cpu_count() or 1))
if "--impl" in sys.argv and "reference" in sys.argv:
    # the reference arm is host arithmetic: fix the thread pools BEFORE the OpenMP runtimes load (r1: 32 threads were
    # slower than 16 — two spinning pools, torch's and the oracle's, on one socket)
    os.environ.setdefault("OMP_NUM_THREADS", str(CPU_THREADS))
    os.environ.setdefault("MKL_NUM_THREADS", str(CPU_THREADS))
    os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "S4G scenes/sec (PN2_CLS inference, 25600 points/scene)"
UNIT = "scenes/s"
NUM_POINTS = 25600
L2_FLUSH_BYTES = 256 << 20
DUMP_BYTES = 60_000_000  # array data written by --dump-outputs: under 64 MB with the .npy headers


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "bf16_tflops": d["bf16_tflops"], "sm_max_mhz": d.get("sm_max_mhz", 1965.0),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops_sustained": 1400.0, "bf16_tflops": 1590.0, "sm_max_mhz": 1965.0,
            "source": "fallback (B200_PROFILING.md)"}


def seeded_model():
    """SURVEY.md §8d: default init under manual_seed(0), BatchNorm statistics from Generator(1)."""
    from s4g_release_b200.network_models.models.PointNet2_tcls import PN2_CLS_CONFIG, PointNet2
    torch.manual_seed(0)
    net = PointNet2(**PN2_CLS_CONFIG)
    g = torch.Generator().manual_seed(1)
    for m in net.modules():
        if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
            n = m.num_features
            m.weight.data = torch.rand(n, generator=g) + 0.5
            m.bias.data = torch.randn(n, generator=g) * 0.1
            m.running_mean.data = torch.randn(n, generator=g) * 0.1
            m.running_var.data = torch.rand(n, generator=g) + 0.5
    return net.eval()


def synthetic_scenes(batch, first_seed):
    from tests.inputs import tabletop_scene
    return torch.from_numpy(np.stack([tabletop_scene(first_seed + i, NUM_POINTS) for i in range(batch)]))


def dump_outputs(preds, out_dir, budget=DUMP_BYTES):
    """Writes each (B, C, N) prediction tensor as out_dir/<name>.npy in float32.  When they hold more than `budget`
    bytes, every tensor keeps the same points: a sorted sample drawn from a fixed seed, so dumps stay comparable."""
    n = next(iter(preds.values())).shape[-1]
    total = 4 * sum(v.numel() for v in preds.values())
    keep = None
    if total > budget:
        keep = torch.from_numpy(np.sort(np.random.default_rng(0).choice(n, n * budget // total, replace=False)))
    os.makedirs(out_dir, exist_ok=True)
    for name, v in preds.items():
        if keep is not None:
            v = v.index_select(-1, keep.to(v.device))
        np.save(os.path.join(out_dir, name + ".npy"), v.detach().float().cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,timestamp")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.windows = []  # (t0, t1) wall-clock windows of the timed regions

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def __enter__(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None
        return self

    def __exit__(self, *exc):
        if self.p is not None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.p.kill()
        return False

    def summary(self):
        import datetime
        sm, mx, reasons = [], [], set()
        all_sm, all_mx = [], []
        try:
            self.f.flush()
            for line in open(self.f.name):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 10:
                    continue
                all_sm.append(float(c[1]))
                all_mx.append(float(c[2]))
                try:
                    ts = datetime.datetime.strptime(c[9], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                except ValueError:
                    ts = None
                if self.windows and ts is not None and not any(a - 0.02 <= ts <= b + 0.02 for a, b in self.windows):
                    continue
                sm.append(float(c[1]))
                mx.append(float(c[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.f.name)
        except (OSError, ValueError):
            pass
        if not sm and all_sm:  # no sample fell inside a window: report the whole run, say so
            return {"sm_mhz": statistics.median(all_sm), "sm_max_mhz": max(all_mx), "reasons": sorted(reasons),
                    "samples": len(all_sm), "note": "no sample inside the timed windows; median over the whole run"}
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


FP32_FLOP_PER_EVAL = 10.0  # 3 sub, 1 mul, 2 fma (= 4 flop), 1 min, 1 compare/select: SURVEY.md §8d counts 10 per pair


def stage_model(batch, eng=None):
    """Work per launch for every stage of one step, in THIS implementation's data types (bf16 channel-last features,
    int32 indices, fp32 coordinates): {stage: dict(bound, flops | bytes, note)}.
      tensor      flops = 2 * rows * sum(cin * cout) over the chain's layers (SURVEY.md §8d); min_bytes = what the chain
                  must move through HBM (inputs once, outputs once);
      hbm         bytes = algorithmic minimum (every input read once, every output written once);
      fp32_issue  flops = pair evaluations x 10; for the farthest point sampling the evaluation count is exact
                  (B (M-1) N); the grid-based ball query / 3-NN searches are output-sensitive, their evaluation count is
                  not known without a counter, so only the upper bound is listed and no fraction is derived from it."""
    from s4g_release_b200.network_models.models.PointNet2_tcls import PN2_CLS_CONFIG as C
    B = batch
    n = [NUM_POINTS] + list(C["num_centroids"])
    K = C["num_neighbours"]
    split = eng is not None and getattr(eng, "fp_pre", None) is not None
    st = {}
    cin = 0
    for i in range(3):
        N, M = n[i], n[i + 1]
        st["sa%d.fps" % i] = dict(bound="fp32_issue", flops=B * (M - 1.0) * N * FP32_FLOP_PER_EVAL,
                                  min_bytes=B * (12.0 * N + 4.0 * M), evals="exact")
        st["sa%d.ball_query" % i] = dict(bound="fp32_issue", flops=None, evals_upper_bound=B * float(M) * N,
                                         min_bytes=B * (12.0 * N + 12.0 * M + 4.0 * M * K[i]))
        st["sa%d.gather_xyz" % i] = dict(bound="hbm", bytes=B * M * (4.0 + 12.0 + 12.0))
        dims = [cin + 3] + list(C["sa_channels"][i])
        st["sa%d.mlp" % i] = dict(bound="tensor", flops=2.0 * B * M * K[i] * sum(a * b for a, b in zip(dims[:-1], dims[1:])),
                                  min_bytes=B * (4.0 * M * K[i] + 2.0 * N * cin + 12.0 * N + 12.0 * M + 2.0 * M * dims[-1]))
        cin = dims[-1]
    skip = [0] + [c[-1] for c in C["sa_channels"]]
    c = skip[-1]
    for i in range(3):
        Nq, Nk = n[-2 - i], n[-1 - i]
        st["fp%d.three_nn" % i] = dict(bound="fp32_issue", flops=None, evals_upper_bound=B * float(Nq) * Nk,
                                       min_bytes=B * (12.0 * Nq + 12.0 * Nk + 24.0 * Nq))
        c1 = skip[-2 - i]
        dims = [c + c1] + list(C["fp_channels"][i])
        pre = split and eng.fp_pre[i] is not None
        if pre:  # first conv on the sparse rows, interpolation of its dims[1]-wide output (engine.fp_linear_split)
            st["fp%d.interp_concat" % i] = dict(bound="hbm", bytes=B * (24.0 * Nq + 2.0 * Nk * dims[1] + 2.0 * Nq * dims[1]))
            flops = 2.0 * B * (Nk * dims[0] * dims[1] + Nq * sum(a * b for a, b in zip(dims[1:-1], dims[2:])))
            mb = B * 2.0 * (Nk * (dims[0] + dims[1]) + Nq * (dims[1] + dims[-1]))
        else:
            st["fp%d.interp_concat" % i] = dict(bound="hbm", bytes=B * (24.0 * Nq + 2.0 * Nk * c + 2.0 * Nq * c1 +
                                                                        2.0 * Nq * (c + c1)))
            flops = 2.0 * B * Nq * sum(a * b for a, b in zip(dims[:-1], dims[1:]))
            mb = B * 2.0 * Nq * (dims[0] + dims[-1])
        st["fp%d.mlp" % i] = dict(bound="tensor", flops=flops, min_bytes=mb, reference_flops=2.0 * B * Nq * sum(
            a * b for a, b in zip(dims[:-1], dims[1:])))
        c = dims[-1]
    seg = [c] + list(C["seg_channels"])
    per_head = sum(a * b for a, b in zip(seg[:-1], seg[1:]))
    outs = (C["score_classes"], 9, 4, C["num_removal_directions"])
    st["heads.mlp"] = dict(bound="tensor", flops=2.0 * B * NUM_POINTS * sum(per_head + seg[-1] * o for o in outs),
                           min_bytes=B * NUM_POINTS * (2.0 * c + 4.0 * sum(outs)))
    return st


def reference_state_dict():
    """Seeded weights of SURVEY.md §8d config 1 from the UNMODIFIED reference model class when it is staged (no product
    import on the reference arm), else from the product class (identical under the seed: tests/golden/make_golden.py)."""
    from oracle import pn2_ext_cpu
    from tests.golden.make_golden import seed_reference_weights
    try:
        from baseline import stage_ref
        if not stage_ref.available():
            raise ImportError("baseline/_ref not staged")
        RefPointNet2 = stage_ref.import_reference_model(pn2_ext_cpu)
        from oracle.model_cpu import PN2_CLS_CONFIG
        torch.manual_seed(0)
        model = seed_reference_weights(RefPointNet2(**PN2_CLS_CONFIG)).eval()
        return model, model.state_dict(), "unmodified reference python modules (baseline/_ref)"
    except ImportError:
        net = seeded_model()
        return None, net.state_dict(), "oracle/model_cpu.py (bit-identical restatement of the reference modules)"


def run_reference(args, rank, world):
    """Reference arm: the reference model on the host CPU, rank 0 only."""
    if rank != 0:
        return
    from oracle import model_cpu, pn2_ext_cpu
    torch.set_num_threads(CPU_THREADS)
    model, sd, what = reference_state_dict()
    scenes = synthetic_scenes(1, 1000)
    times = []
    with torch.no_grad():
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            if model is not None:
                out = model({"scene_points": scenes})
            else:
                out = model_cpu.pointnet2_forward(scenes, sd, model_cpu.PN2_CLS_CONFIG)
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    value = 1e3 / ms
    cores = max(pn2_ext_cpu.num_threads(), torch.get_num_threads())
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "PN2_CLS inference, synthetic tabletop clouds, 25600 points/scene (BASELINE config[1])",
                   "sample_per_step": "1 scene of the 64-scene batch"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "1 scene per step: %s on the OpenMP C restatement of the CUDA-only pn2_ext ops "
                                   "(oracle/pn2_oracle.c), torch-CPU fp32 conv/BN; %d threads" % (what, cores)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        dump_outputs(out, args.dump_outputs)


TRAFFIC_FILE = "profiles/r02/ncu_launches.json"
NCU_DETAIL_FILE = "profiles/r02/ncu_kernels.json"


def stage_traffic(eng):
    """Per stage, from the committed ncu launch list of one forward at this workload: DRAM bytes (read + write summed
    over the stage's launches) and the time-weighted tensor-pipe-active %.  Launches are matched by kernel name in
    forward order; returns {} when the list does not match the engine's launch structure."""
    try:
        launches = json.load(open(os.path.join(ROOT, TRAFFIC_FILE)))["launches"]
    except Exception:
        return {}
    def pick(*subs):
        return [l for l in launches if any(x in l["kernel"] for x in subs)]
    fps, interp = pick("fps_kernel"), pick("interp_concat")
    ball = pick("ball_query_grid_kernel", "ball_query_kernel")
    chains = pick("mlp_chain")
    sa = [l for l in chains if ", 3, 1" in l["kernel"]]      # mlp_chain_kernel<.., OUT_MAXPOOL, gather, ..>
    heads = [l for l in chains if ", 4, 0" in l["kernel"]]   # OUT_LOGITS
    rows = [l for l in chains if ", 2, 0" in l["kernel"]]    # OUT_ROWS: the propagation chains, in order
    per_fp = [len(eng.fp_chains[i]) + (1 if eng.fp_pre[i] is not None else 0) for i in range(3)]
    if not (len(fps) == 3 and len(ball) == 3 and len(sa) == 3 and len(heads) == 4 and len(interp) == 3 and
            len(rows) == sum(per_fp)):
        return {}
    def agg(ls):
        ms = sum(l["ms"] for l in ls)
        return {"dram_bytes": sum(l.get("dram_read_MB", 0) + l.get("dram_write_MB", 0) for l in ls) * 1e6,
                "ncu_ms": round(ms, 4),
                "tensor_pipe_active_pct": round(sum(l.get("tensor_active_pct", 0) * l["ms"] for l in ls) / max(ms, 1e-9), 2)}
    out = {}
    r0 = 0
    for i in range(3):
        out["sa%d.fps" % i] = agg([fps[i]])
        out["sa%d.ball_query" % i] = agg([ball[i]])
        out["sa%d.mlp" % i] = agg([sa[i]])
        out["fp%d.interp_concat" % i] = agg([interp[i]])
        out["fp%d.mlp" % i] = agg(rows[r0:r0 + per_fp[i]])
        r0 += per_fp[i]
    out["heads.mlp"] = agg(heads)
    return out


def ncu_details():
    """issue-slot utilisation / L2 hit rate / top stall of the kernels captured with `ncu --set full` (committed summary)."""
    try:
        return json.load(open(os.path.join(ROOT, NCU_DETAIL_FILE)))
    except Exception:
        return {}


def bind_to_gpu_numa_node(gpu_index):
    """Pin this process to the CPUs next to its GPU (8 ranks on one NUMA node cost 4.6 % end to end in r1)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        try:  # CUDA_VISIBLE_DEVICES may renumber the devices: resolve the NVML handle through the UUID
            uuid = "GPU-" + str(torch.cuda.get_device_properties(gpu_index).uuid)
            handle = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
        except Exception:
            handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        before = os.sched_getaffinity(0)
        pynvml.nvmlDeviceSetCpuAffinity(handle)
        after = os.sched_getaffinity(0)
        if len(after) < 4:  # a container cpuset that barely intersects the node: keep what we had
            os.sched_setaffinity(0, before)
            return None
        return sorted(after)
    except Exception:
        return None


def reference_cuda_rows(net_sd, scenes_host, dev):
    """The unmodified reference model (baseline/_ref python) on the reference's own CUDA kernels (oracle/_ref, its .cu
    files compiled unmodified for sm_100a) timed on this GPU — the competitor row of SURVEY.md §8d.  cuDNN TF32 as torch
    defaults it (what a user of the reference gets) and IEEE fp32."""
    rows = {}
    try:
        from baseline import stage_ref
        from oracle import build_ref
        if not stage_ref.available() or not os.path.exists(build_ref.so_path()):
            return {"unavailable": "baseline/_ref or oracle/_ref not staged"}
        RefPointNet2 = stage_ref.import_reference_model(build_ref.load())
        from oracle.model_cpu import PN2_CLS_CONFIG
        model = RefPointNet2(**PN2_CLS_CONFIG)
        model.load_state_dict(net_sd, strict=True)
        model = model.to(dev).eval()
        keep = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        for tf32 in (True, False):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            for b in (1, 8, 64):
                x = scenes_host[:b].to(dev)
                try:
                    with torch.no_grad():
                        model({"scene_points": x})
                        torch.cuda.synchronize()
                        ts = []
                        for _ in range(2 if b == 64 else 3):
                            t0 = time.perf_counter()
                            model({"scene_points": x})
                            torch.cuda.synchronize()  # the reference launches on the legacy default stream
                            ts.append(time.perf_counter() - t0)
                    rows["B%d_%s" % (b, "tf32" if tf32 else "fp32")] = {"ms": round(1e3 * min(ts), 2),
                                                                        "scenes_per_s": round(b / min(ts), 2)}
                except RuntimeError as e:  # out of memory at 64 scenes of unfused fp32 activations
                    rows["B%d_%s" % (b, "tf32" if tf32 else "fp32")] = {"error": str(e)[:80]}
                    torch.cuda.empty_cache()
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = keep
        del model
        torch.cuda.empty_cache()
        rows["what"] = ("unmodified reference PointNet2 + modules.py / functions.py on its own pn2_ext CUDA kernels "
                        "(one CTA per cloud), torch cuDNN convolutions; best wall-clock of 3 (2 at B=64) after 1 warm-up")
    except Exception as e:  # never let the comparison row break the bench line
        rows["unavailable"] = "%s: %s" % (type(e).__name__, str(e)[:120])
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="scenes per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-cuda", action="store_true")
    ap.add_argument("--mlp-backend", default="tcgen05", choices=["tcgen05", "tf32", "torch"])
    ap.add_argument("--no-fp-split", action="store_true", help="A/B: interpolate-then-conv at the finest propagation level")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's predictions to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    from s4g_release_b200 import _lib
    from s4g_release_b200.engine import FusedPointNet2, StageTimer

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path for the product)"
    affinity = bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    B = args.batch
    net = seeded_model().to(dev)
    eng = FusedPointNet2(net, mlp_backend=args.mlp_backend, fp_linear_split=not args.no_fp_split)
    net.attach_engine(eng)
    host_scenes = synthetic_scenes(B, 1000 + rank * B).pin_memory()
    scenes = host_scenes.to(dev)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---------------- device-resident throughput ----------------
    clocks = ClockSampler(local_rank)
    clocks.__enter__()
    for _ in range(args.warmup):
        eng.forward(scenes)
    sync_all()
    launches0 = _lib.lib.s4g_launch_count()
    timers, step_events = [], []
    sync_all()
    t_w0 = time.time()
    for _ in range(args.steps):
        flush.zero_()  # evict L2 between steps (outside the per-step event pair)
        t = StageTimer()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step_out = eng.forward(scenes, timer=t)
        b.record()
        timers.append(t)
        step_events.append((a, b))
    sync_all()
    clocks.window(t_w0, time.time())
    launches = (_lib.lib.s4g_launch_count() - launches0) // args.steps  # kernels launched by libs4g_b200.so
    step_ms = [a.elapsed_time(b) for a, b in step_events]
    ms_local = sum(step_ms) / len(step_ms)

    # ---------------- end to end through the public API with host buffers ----------------
    out_host = None
    e2e_ms = []
    h2d = host_scenes.numel() * 4
    d2h = 0
    for i in range(args.warmup + args.steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        x = host_scenes.to(dev, non_blocking=True)
        with torch.no_grad():
            if out_host is None:  # first (warm-up) step: learn the output shapes
                preds = net({"scene_points": x})
                out_host = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in preds.items()}
                d2h = sum(v.numel() * v.element_size() for v in preds.values())
                for k, v in preds.items():
                    out_host[k].copy_(v, non_blocking=True)
            elif args.mlp_backend == "tcgen05":  # the public call with pinned result buffers: head copies overlap the next head
                preds = net({"scene_points": x}, host_out=out_host)
            else:
                preds = net({"scene_points": x})
                for k, v in preds.items():
                    out_host[k].copy_(v, non_blocking=True)
        torch.cuda.synchronize()
        if i >= args.warmup:
            e2e_ms.append(1e3 * (time.perf_counter() - t0))
            clocks.window(time.time() - e2e_ms[-1] * 1e-3, time.time())
    e2e_local = sum(e2e_ms) / len(e2e_ms)
    # the same public call with bf16 pinned result buffers (the copy converts on the device): half the D2H bytes, for
    # callers that accept bf16 predictions — reported beside the fp32 headline, never instead of it
    e2e16_local = None
    if args.mlp_backend == "tcgen05":
        out16 = {k: torch.empty(v.shape, dtype=torch.bfloat16).pin_memory() for k, v in out_host.items()}
        ts = []
        for i in range(args.warmup + args.steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            x = host_scenes.to(dev, non_blocking=True)
            with torch.no_grad():
                net({"scene_points": x}, host_out=out16)
            torch.cuda.synchronize()
            if i >= args.warmup:
                ts.append(1e3 * (time.perf_counter() - t0))
        e2e16_local = sum(ts) / len(ts)
    time.sleep(0.05)
    clocks.__exit__(None, None, None)
    if args.dump_outputs and rank == 0:
        dump_outputs(step_out, args.dump_outputs)

    # ---------------- reduce over ranks (max time) ----------------
    if world > 1:
        tt = torch.tensor([ms_local, e2e_local, e2e16_local or 0.0], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, e2e, e2e16 = tt[0].item(), tt[1].item(), tt[2].item()
    else:
        ms, e2e, e2e16 = ms_local, e2e_local, e2e16_local or 0.0
    value = world * B / (ms * 1e-3)
    e2e_value = world * B / (e2e * 1e-3)

    if rank == 0:
        peaks = load_peaks()
        clk = clocks.summary()
        n_sms = torch.cuda.get_device_properties(dev).multi_processor_count
        # FP32 issue peak: SMs x 128 lanes x 2 flop (FMA) x the SM clock the step actually ran at
        sm_mhz = clk.get("sm_mhz") or peaks["sm_max_mhz"]
        fp32_peak_tflops = n_sms * 128 * 2 * sm_mhz * 1e6 / 1e12
        tensor_peak = peaks["bf16_tflops"] if args.steps * ms_local < 1000.0 else peaks["bf16_tflops_sustained"]
        tensor_peak_name = "burst" if tensor_peak == peaks["bf16_tflops"] else "sustained"
        model = stage_model(B, eng if args.mlp_backend == "tcgen05" else None)
        traffic = stage_traffic(eng) if (args.mlp_backend == "tcgen05" and B == 64) else {}
        detail = ncu_details()
        per_stage = {}
        for t in timers:
            for name, vals in t.totals_ms().items():
                per_stage.setdefault(name, []).extend(vals)
        kernels = {}
        for name, vals in per_stage.items():
            avg = sum(vals) / args.steps  # a stage may be recorded in two pieces per step (fp2: conv on sparse rows + rest)
            m = model[name]
            k = {"ms": round(avg, 4), "share": round(avg / ms_local, 4), "bound": m["bound"]}
            sec = avg * 1e-3
            if m["bound"] == "tensor":
                ach = m["flops"] / sec / 1e12
                k.update(achieved=round(ach, 2), peak=tensor_peak, unit="TFLOP/s", frac=round(ach / tensor_peak, 4),
                         algorithmic_min_bytes=m["min_bytes"])
            elif m["bound"] == "hbm":
                ach = m["bytes"] / sec / 1e9
                k.update(achieved=round(ach, 2), peak=peaks["hbm_gbs"], unit="GB/s", frac=round(ach / peaks["hbm_gbs"], 4),
                         algorithmic_min_bytes=m["bytes"])
            else:  # fp32 issue (+ dependent-latency) bound geometry
                k.update(peak=round(fp32_peak_tflops, 2), unit="TFLOP/s (fp32 issue: %d SMs x 128 lanes x 2 x %.0f MHz)"
                         % (n_sms, sm_mhz), algorithmic_min_bytes=m["min_bytes"])
                if m.get("flops"):
                    ach = m["flops"] / sec / 1e12
                    k.update(achieved=round(ach, 2), frac=round(ach / fp32_peak_tflops, 4))
                else:
                    k.update(achieved=None, frac=None, evals_upper_bound=m["evals_upper_bound"],
                             note="output-sensitive grid search: evaluations done << upper bound, no rate derived; see "
                                  "issue_active_pct from the ncu capture")
            tr = traffic.get(name)
            if tr:
                k["dram_bytes"] = tr["dram_bytes"]
                k["hbm_frac_actual"] = round(tr["dram_bytes"] / sec / 1e9 / peaks["hbm_gbs"], 4)
                k["traffic_ratio"] = round(tr["dram_bytes"] / k["algorithmic_min_bytes"], 3)
                if m["bound"] == "tensor":
                    k["tensor_pipe_active_pct_ncu"] = tr["tensor_pipe_active_pct"]
            if name in detail:
                k["ncu"] = detail[name]
            if name in ("fp1.three_nn", "fp2.three_nn") and getattr(eng, "overlap_geometry", False):
                # these searches run on a side stream beside the sampling of the next level: the main-stream event pair
                # only sees the wait for them
                k["overlapped"] = "side stream, beside sa%d.fps" % (3 - int(name[2]))
            kernels[name] = k
        if not kernels:  # the torch / tf32 comparison backends run without stage timers
            line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "dtype": {"tf32": "tf32", "torch": "f32"}.get(args.mlp_backend, "bf16"),
                    "data": "synthetic", "config": {"workload": "PN2_CLS inference (comparison backend %s, NOT the product path)"
                                                    % args.mlp_backend, "scenes_per_gpu_per_step": B},
                    "clocks": clk, "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                                           "d2h_bytes_per_step": d2h}, "gpu_launches": int(launches) * args.steps}
            print(json.dumps(line), flush=True)
            if world > 1:
                dist.barrier()
                dist.destroy_process_group()
            return
        # ---- roofline: the dominant kernel TYPE (mlp_chain_kernel, every launch of the step) vs the tensor peak ----
        chain_names = [n for n in kernels if n.endswith(".mlp")]
        chain_ms = sum(kernels[n]["ms"] for n in chain_names)
        chain_flops = sum(model[n]["flops"] for n in chain_names)
        chain_dram = sum(kernels[n].get("dram_bytes", 0) for n in chain_names) if traffic else None
        n_chain = sum(len(c) for c in eng.fp_chains) + sum(p is not None for p in eng.fp_pre) + 3 + 4 \
            if args.mlp_backend == "tcgen05" else None
        ach = chain_flops / (chain_ms * 1e-3) / 1e12
        roof = {"kernel": "mlp_chain_kernel (tcgen05 bf16 fused shared-MLP chains: %s launches per step, sa0-2 / fp0-2 / 4 heads)" % n_chain,
                "bound": "tensor", "achieved": round(ach, 2), "peak": tensor_peak, "unit": "TFLOP/s",
                "frac": round(ach / tensor_peak, 4), "ms_per_step": round(chain_ms, 4), "share_of_step": round(chain_ms / ms_local, 4),
                "flops_per_step": chain_flops, "traffic": chain_dram,
                "traffic_per_launch": (chain_dram / n_chain) if chain_dram and n_chain else None,
                "traffic_source": TRAFFIC_FILE if traffic else None,
                "tensor_pipe_active_pct_ncu": round(sum(kernels[n].get("tensor_pipe_active_pct_ncu", 0) * kernels[n]["ms"]
                                                        for n in chain_names) / chain_ms, 2) if traffic else None,
                "peak_source": peaks["source"] + " — %s bf16 (timed region %.2f s)" % (tensor_peak_name, args.steps * ms_local * 1e-3)}
        f0 = kernels["sa0.fps"]
        roof_fps = {"kernel": "fps_kernel (level 0: %d clouds x 25600 -> 5120; longest single launch)" % B,
                    "ms": f0["ms"], "share_of_step": f0["share"], "bound": "fp32 issue + per-iteration exchange latency",
                    "fp32_issue_frac": f0.get("frac"), "fp32_tflops": f0.get("achieved"), "fp32_issue_peak_tflops": f0["peak"],
                    "hbm_frac_actual": f0.get("hbm_frac_actual"), "dram_bytes": f0.get("dram_bytes"),
                    "us_per_iteration": round(f0["ms"] * 1e3 / 5119.0, 4), "ncu": f0.get("ncu")}
        total_flops = sum(m["flops"] for m in model.values() if m["bound"] == "tensor")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"tcgen05": "bf16", "tf32": "tf32", "torch": "f32"}[args.mlp_backend], "data": "synthetic",
            "config": {"workload": "PN2_CLS inference, synthetic tabletop clouds, 25600 points/scene (BASELINE config[1])",
                       "scenes_per_gpu_per_step": B, "parallelism": "scene-batch sharding, dp%d, no collective" % world,
                       "geometry": "fp32 exact (FPS / ball query / 3-NN)",
                       "mlp": {"tcgen05": "tcgen05 bf16 x bf16 -> fp32 (TMEM), BN folded",
                               "tf32": "tcgen05 kind::tf32 per layer (tight-parity mode, NOT the throughput path)",
                               "torch": "torch fp32 reference MLPs (NOT the product path)"}[args.mlp_backend],
                       "fp_linear_split": bool(getattr(eng, "fp_linear_split", False)),
                       "l2": "flushed between steps (256 MiB memset outside the per-step event pairs)",
                       "cpu_affinity": ("%d CPUs next to GPU %d" % (len(affinity), local_rank)) if affinity else "unchanged"},
            "clocks": clk,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e},
            "e2e_bf16_host_buffers": ({"value": world * B / (e2e16 * 1e-3), "unit": UNIT, "ms_per_step": e2e16,
                                       "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h // 2,
                                       "note": "same public call, caller's pinned result buffers are bf16"}
                                      if e2e16 > 0 else None),
            "gpu_launches": int(launches) * args.steps,
            "gpu_launches_per_step": int(launches),
            "roofline": roof,
            "roofline_fps": roof_fps,
            "model_tflops_per_step": round(total_flops / 1e12, 3),
            "model_tensor_frac": round(total_flops / (ms_local * 1e-3) / 1e12 / tensor_peak, 4),
            "kernels": kernels,
        }
        if world == 1 and not args.no_cpu_baseline:
            from oracle import model_cpu, pn2_ext_cpu
            from tests import pose_parity
            torch.set_num_threads(CPU_THREADS)
            sd = {k: v.cpu() for k, v in net.state_dict().items()}
            one = host_scenes[:1].contiguous()
            with torch.no_grad():
                want = model_cpu.pointnet2_forward(one, sd, model_cpu.PN2_CLS_CONFIG)  # warm-up; also the parity reference
                ts = []
                for _ in range(2):
                    t0 = time.perf_counter()
                    model_cpu.pointnet2_forward(one, sd, model_cpu.PN2_CLS_CONFIG)
                    ts.append(time.perf_counter() - t0)
                got = eng.forward(scenes[:1].contiguous())
                torch.cuda.synchronize()
            line["cpu_baseline"] = {"value": 1.0 / min(ts), "unit": UNIT,
                                    "cores": max(pn2_ext_cpu.num_threads(), torch.get_num_threads()), "kind": "port",
                                    "sample": "1 scene of the batch, best of 2 after 1 warm-up (oracle/model_cpu.py)"}
            # score / pose parity of that scene: fused GPU forward vs the fp32 CPU oracle (tests/pose_parity.py;
            # bounds asserted in tests/test_pose_parity_gpu.py)
            line["parity"] = dict(pose_parity.scene_metrics(one[0].numpy(), {k: v[0].numpy() for k, v in want.items()},
                                                           {k: v[0].float().cpu().numpy() for k, v in got.items()}),
                                  scene="scene 0 of the batch (tabletop_scene(1000))", checker="oracle/model_cpu.py fp32 on the host",
                                  backend=args.mlp_backend)
        if world == 1 and not args.no_reference_cuda:
            line["reference_cuda"] = reference_cuda_rows({k: v.cpu() for k, v in net.state_dict().items()}, host_scenes, dev)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
