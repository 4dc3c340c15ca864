"""Data-parallel training step for PN2_CLS (BASELINE config 4) — one process per GPU.

The reference ships no training loop (SURVEY.md §3.4); this assembles one from its parts only: the model
(module / autograd path on the sm_100a ops), ``PointNet2Loss`` (models/PointNet2_tcls.py:162-219), the
solver defaults Adam lr 1e-3, betas (0.9, 0.999), weight_decay 0 (configs/yacs_config.py:102-118) and
StepLR(step 20, gamma 0.5) (configs/curvature_model.yaml:25-30).  Scenes are sharded contiguously across
ranks; BatchNorm statistics stay per replica (the reference uses plain nn.BatchNorm under DataParallel);
the only collective is ONE flat all-reduce of the 6.63 M fp32 gradients (26.5 MB) per step — NCCL over
NVLink on GPUs, gloo in the CPU tests.
"""
import numpy as np
import torch
import torch.distributed as dist


def shard_range(n_items, rank, world):
    """Contiguous, balanced partition of ``n_items`` scenes: rank r owns [start, stop)."""
    base, extra = divmod(n_items, world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


class GradBucket:
    """One flat fp32 buffer aliasing every parameter's .grad, so the step needs a single all-reduce."""

    def __init__(self, params):
        self.params = [p for p in params if p.requires_grad]
        n = sum(p.numel() for p in self.params)
        dev = self.params[0].device
        self.flat = torch.zeros(n, dtype=torch.float32, device=dev)
        off = 0
        for p in self.params:
            p.grad = self.flat[off:off + p.numel()].view_as(p)
            off += p.numel()

    def zero(self):
        self.flat.zero_()

    def all_reduce_mean(self, group=None):
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group)
            self.flat.div_(dist.get_world_size(group))


def broadcast_parameters(module, src=0, group=None):
    """Replicas start from rank ``src``'s parameters and buffers."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        for t in list(module.parameters()) + list(module.buffers()):
            dist.broadcast(t.data, src=src, group=group)


def synthetic_labels(batch, num_points, num_frame=4000, first_seed=2000, device="cpu", continuous_t=False):
    """SURVEY.md §8d config 4: score labels {0,1,2}, movable {0,1}, random rotations (row-major 9),
    approach-offset class {0..3}, scene_score U[0,1]; M' = 4000 frame points as the reference's smoke block.
    ``continuous_t``: best_frame_t is a float32 (3, M') position in U[0,1)^3 instead of the class index — the label of
    the PN2 sibling's translation head (models/PointNet2.py: frame_t = points + offset)."""
    out = {k: [] for k in ("scene_score_labels", "scene_movable_labels", "best_frame_R", "best_frame_t", "scene_score")}
    for i in range(batch):
        rs = np.random.RandomState(first_seed + i)
        out["scene_score_labels"].append(rs.randint(0, 3, size=num_points))
        out["scene_movable_labels"].append(rs.randint(0, 2, size=(5, num_points)).astype(np.float32))
        q, _ = np.linalg.qr(rs.randn(num_frame, 3, 3))
        out["best_frame_R"].append(q.reshape(num_frame, 9).T.astype(np.float32))
        out["best_frame_t"].append(rs.rand(3, num_frame).astype(np.float32) if continuous_t else
                                   rs.randint(0, 4, size=num_frame))
        out["scene_score"].append(rs.rand(num_points).astype(np.float32))
    return {k: torch.from_numpy(np.stack(v)).to(device) for k, v in out.items()}


class Trainer:
    def __init__(self, model, loss_fn, lr=1e-3, betas=(0.9, 0.999), weight_decay=0.0, step_size=20, gamma=0.5,
                 group=None, fused=False):
        """``fused``: forward + loss + backward on the B200-native training kernels (train_engine.TrainEngine: tcgen05
        GEMMs over bf16 rows, fused BatchNorm / ReLU / max-pool passes) instead of the module path under torch autograd —
        PN2_CLS or the PN2 sibling with its own PointNet2Loss, including a global last level (TrainEngine's guard)."""
        self.model, self.loss_fn, self.group = model, loss_fn, group
        self.engine = None
        if fused:
            from .train_engine import TrainEngine
            self.engine = TrainEngine(model, loss_fn)
        broadcast_parameters(model, 0, group)
        self.bucket = GradBucket(model.parameters())
        self.optimizer = torch.optim.Adam(self.bucket.params, lr=lr, betas=betas, weight_decay=weight_decay)
        self.scheduler = torch.optim.lr_scheduler.StepLR(self.optimizer, step_size=step_size, gamma=gamma)

    def step(self, data_batch, labels):
        """One optimisation step on this rank's shard; returns the loss dict (detached)."""
        self.model.train()
        self.bucket.zero()
        if self.engine is not None:
            losses = self.engine.step_loss(data_batch, labels)
        else:
            preds = self.model(data_batch)
            losses = self.loss_fn(preds, labels)
            total = sum(losses.values())
            total.backward()
        self.bucket.all_reduce_mean(self.group)
        self.optimizer.step()
        return {k: v.detach() for k, v in losses.items()}
