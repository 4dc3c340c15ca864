"""Fused TRAINING step of PN2_CLS on the B200-native kernels (BASELINE config 4).

The module path (pointnet2_utils.modules + torch autograd) materialises every grouped tensor in fp32 channel-first
layout and runs conv / BatchNorm / ReLU / max as separate library kernels: 339 ms and 115 GB for 32 scenes (round 1).
This engine runs the SAME computation — reference PointNet2.forward in training mode (models/PointNet2_tcls.py:99-148),
PointNet2Loss (:162-219) and the backward of all of it — on channel-last bf16 rows:

  geometry        the sm_100a operators of the inference engine (FPS, ball query, 3-NN + weights), exact fp32, no grad
                  (reference functions.py:46-47,76-77,131-132 return None for them too);
  grouping        s4g_train_group_rows_bf16: one gathered row [features | relative xyz] per (centroid, neighbour);
  shared MLP      per block ONE tcgen05 GEMM (csrc/gemm_bf16.cu, fp32 accumulation) + batch statistics (fp64 sums)
                  + one fused normalise / ReLU / dropout pass — for the last block of a set-abstraction level fused with
                  the max over the K neighbours (arg-max kept as uint8);
  heads           the four 4-block MLPs as above; the final biased 1x1 convs (128 -> 3 / 9 / 4 / 5, + sigmoid) and the
                  loss are tiny and stay in torch: autograd hands back d(loss)/d(head features);
  backward        written out by hand — BatchNorm backward in two fused passes (reduce, apply) that also undo ReLU /
                  dropout / max-pool routing on the fly, dX = dY · W on the tcgen05 GEMM, dW = dY^T · X as a plain
                  library GEMM (torch.mm, bf16 operands, fp32 result: the one cuBLAS call per block), scatter-adds of the
                  grouping and interpolation gradients with fp32 vector atomics.

Parameters stay the fp32 master copies of the nn.Module (state_dict / checkpoints unchanged); gradients are written to
``param.grad`` in fp32; BatchNorm running statistics are updated like torch does (momentum, unbiased variance).
Activations are bf16, so this is the numerical regime of bf16 autocast training, not of the fp32 module path: the test
(tests/test_train_engine_gpu.py) states the tolerance.  There is no CPU path.
"""
import torch

from ._lib import check, lib, ptr, stream_ptr
from .engine import FusedPointNet2

BF16 = torch.bfloat16


# ------------------------------------------------------------------------------------------------ kernel wrappers
def gemm(a, b, stats=False):
    """a [P, K] bf16 (row stride % 8 == 0), b [N, K] bf16 -> [P, N] bf16 (N padded to 8 internally when needed).
    ``stats``: also return the fp64 [2N] column sums / sums of squares of the stored result (fused in the epilogue)."""
    assert a.dtype == BF16 and b.dtype == BF16 and a.stride(1) == 1 and b.stride(1) == 1 and a.shape[1] == b.shape[1]
    P, K = a.shape
    N = b.shape[0]
    ldc = (N + 7) // 8 * 8
    c = torch.empty((P, ldc), dtype=BF16, device=a.device)
    if stats:
        sums = torch.empty(2 * N, dtype=torch.float64, device=a.device)
        check(lib.s4g_gemm_bf16_stats(ptr(a), a.stride(0), ptr(b), b.stride(0), ptr(c), ldc, P, N, K, ptr(sums),
                                      stream_ptr(a.device)), "gemm_bf16_stats")
        return (c if ldc == N else c[:, :N]), sums
    check(lib.s4g_gemm_bf16(ptr(a), a.stride(0), ptr(b), b.stride(0), ptr(c), ldc, P, N, K, stream_ptr(a.device)), "gemm_bf16")
    return c if ldc == N else c[:, :N]


def gemm_bwd(a, b, prev_y, prev_scale, prev_shift, relu=True, seed=0, drop_p=0.0):
    """Input-gradient GEMM of block l whose result is the upstream gradient of block l-1 (``prev_*``: that block's
    pre-BatchNorm rows [P, N] and folded scale / shift): returns (g [P, N] bf16, MASKED with block l-1's ReLU' / dropout,
    sums fp64 [2N] = [sum g | sum g * prev_y]) — the first pass of block l-1's BatchNorm backward done in the epilogue."""
    assert a.dtype == BF16 and b.dtype == BF16 and a.stride(1) == 1 and b.stride(1) == 1 and a.shape[1] == b.shape[1]
    P, K = a.shape
    N = b.shape[0]
    assert prev_y.shape == (P, N) and prev_y.stride(1) == 1 and N % 8 == 0
    c = torch.empty((P, N), dtype=BF16, device=a.device)
    sums = torch.empty(2 * N, dtype=torch.float64, device=a.device)
    check(lib.s4g_gemm_bf16_bwd(ptr(a), a.stride(0), ptr(b), b.stride(0), ptr(c), N, P, N, K, ptr(prev_y), prev_y.stride(0),
                                ptr(prev_scale), ptr(prev_shift), 1 if relu else 0, seed, drop_p, ptr(sums),
                                stream_ptr(a.device)), "gemm_bf16_bwd")
    return c, sums


# BatchNorm statistics inside the GEMM epilogue (s4g_gemm_bf16_stats) or as a separate pass over the stored output.
# Measured at 32 scenes (profiles/r02/train_kernels.md): with the statistics fused, the 4 epilogue warps need ~5 800
# cycles per 128 x 128 tile (shuffle butterfly) against ~2 800 cycles of HBM time, so the memory-bound layers run at
# 1.2-3.2 TB/s; the plain GEMM runs at 6.0-6.8 TB/s and the separate pass at ~5 TB/s — cheaper in total.  Kept selectable.
FUSED_STATS = True
# backward, pass 1 of a block's BatchNorm (sum g, sum g*y): (a) for a block whose upstream gradient comes out of the next
# block's input-gradient GEMM, in that GEMM's epilogue (gemm_bwd); (b) for a pooled block, over the G pooled rows only
# (the gradient is zero off the arg-max rows; the forward keeps y at the arg-max).  Both selectable for A/B measurements.
FUSED_BWD_REDUCE = False  # (measured: 79.0 vs 78.6 ms per step — the fused epilogue is instruction-bound, see csrc/gemm_bf16.cu)
SPARSE_POOL_REDUCE = True
# A propagation level WITHOUT skip features (the finest one of PN2_CLS: 512 channels of 5 120 points onto 25 600 points)
# starts with a linear layer on an interpolation whose weights sum to one: W (sum_k w_k f_k) = sum_k w_k (W f_k).  So the
# conv runs on the SPARSE rows (5 x fewer), the 256-wide pre-activations are interpolated instead of the 512-wide
# features (the concat input is never written), and the backward scatters 256-wide gradients; BatchNorm's statistics are
# those of the interpolated rows, as in the reference order (PointNet2_tcls.py:120-128 -> modules.py FeatureInterpolator).
# Measured at 32 scenes: 74.7-75.9 ms with, 75.6 ms without (the saved GEMM / scatter work is paid back by the separate
# statistics pass and the extra casts), 0.6 GB less memory — no gain in training, unlike inference; off by default.
FP_LINEAR_SPLIT = False


def colstats_raw(y):
    P, C = y.shape
    out = torch.empty(2 * C, dtype=torch.float64, device=y.device)
    check(lib.s4g_train_colstats_bf16(ptr(y), y.stride(0), P, C, ptr(out), stream_ptr(y.device)), "train_colstats")
    return out


def colstats(y):
    P, C = y.shape
    out = torch.empty(2 * C, dtype=torch.float64, device=y.device)
    check(lib.s4g_train_colstats_bf16(ptr(y), y.stride(0), P, C, ptr(out), stream_ptr(y.device)), "train_colstats")
    return out[:C], out[C:]


class Block:
    """One conv (bias-free 1x1) + BatchNorm + ReLU block of a SharedMLP in training mode, on rows.
    ``in_perm``: for the first block of a set-abstraction level, the number of gathered feature channels Cf — the input
    rows are [features(Cf) | xyz(3) | 0 x 5] while the reference's weight columns are [xyz(3) | features(Cf)]."""

    def __init__(self, module, grouped_cf=None, drop_p=0.0):
        self.conv, self.bn = module.conv, module.bn
        self.cf = grouped_cf
        self.drop_p = float(drop_p)
        self.cout = self.conv.weight.shape[0]
        self.cin = self.conv.weight.shape[1]
        self.saved = None

    def _weight_rows(self):
        w = self.conv.weight.detach().reshape(self.cout, self.cin)
        if self.cf is None:
            kp = (self.cin + 7) // 8 * 8
            if kp == self.cin:
                return w.to(BF16)
            wb = torch.zeros((self.cout, kp), dtype=BF16, device=w.device)
            wb[:, :self.cin] = w
            return wb
        wb = torch.zeros((self.cout, self.cf + 8), dtype=BF16, device=w.device)
        wb[:, :self.cf] = w[:, 3:]
        wb[:, self.cf:self.cf + 3] = w[:, :3]
        return wb

    def forward(self, x, pool_k=0, seed=0, global_pool=False):
        """x [P, Kp] bf16 -> z [P, cout] bf16, or (pooled [P / pool_k, cout], arg) when pool_k > 0.
        ``global_pool``: pool_k is the N rows of a scene (a global set-abstraction level, any N): the max runs on
        s4g_train_bn_act_segmax_bf16 and arg is int32 (the row inside the scene)."""
        wb = self._weight_rows()
        if FUSED_STATS:
            y, sums = gemm(x, wb, stats=True)  # conv + the BatchNorm batch statistics of its (stored) output
        else:
            y = gemm(x, wb)
            sums = colstats_raw(y)
        return self._normalise(x, y, sums, wb, pool_k, seed, global_pool)

    def forward_pre(self, y, x_rows, wb):
        """the block from its PRE-activations y [P, cout] bf16 (computed elsewhere: FP_LINEAR_SPLIT); x_rows / wb = the rows
        and weights they came from, kept for the caller's backward (backward returns d y, not d x, for such a block)"""
        z = self._normalise(x_rows, y, colstats_raw(y), wb, 0, 0)
        self.saved = self.saved + (True,)
        return z

    def _normalise(self, x, y, sums, wb, pool_k, seed, global_pool=False):
        bn = self.bn
        P = y.shape[0]
        dev = y.device
        C = self.cout
        stat = torch.empty(4 * C, dtype=torch.float32, device=dev)  # [mean | rstd | scale | shift]
        track = bn.track_running_stats and bn.running_mean is not None
        # (momentum None = torch's cumulative moving average: 1 / number of batches seen so far)
        momentum = bn.momentum if bn.momentum is not None else 1.0 / float(int(bn.num_batches_tracked) + 1) if track else 0.0
        check(lib.s4g_train_bn_finalize(ptr(sums), P, C, ptr(bn.weight), ptr(bn.bias), bn.eps, momentum,
                                        ptr(bn.running_mean) if track else None, ptr(bn.running_var) if track else None,
                                        ptr(stat), stream_ptr(dev)), "train_bn_finalize")
        if track:
            bn.num_batches_tracked += 1
        mean_rstd, scale, shift = stat[:2 * C], stat[2 * C:3 * C], stat[3 * C:]
        if global_pool:
            G = P // pool_k
            z = torch.empty((G, self.cout), dtype=BF16, device=dev)
            arg = torch.empty((G, self.cout), dtype=torch.int32, device=dev)
            ymax = torch.empty((G, self.cout), dtype=BF16, device=dev) if SPARSE_POOL_REDUCE else None
            work = torch.empty((G, self.cout), dtype=torch.int64, device=dev)
            check(lib.s4g_train_bn_act_segmax_bf16(ptr(y), ptr(scale), ptr(shift), ptr(z), ptr(arg),
                                                   ptr(ymax) if ymax is not None else None, ptr(work), G, pool_k,
                                                   self.cout, 1, stream_ptr(dev)), "train_bn_act_segmax")
        elif pool_k:
            G = P // pool_k
            z = torch.empty((G, self.cout), dtype=BF16, device=dev)
            arg = torch.empty((G, self.cout), dtype=torch.uint8, device=dev)
            ymax = torch.empty((G, self.cout), dtype=BF16, device=dev) if SPARSE_POOL_REDUCE else None
            check(lib.s4g_train_bn_act_maxpool_bf16(ptr(y), ptr(scale), ptr(shift), ptr(z), ptr(arg),
                                                    ptr(ymax) if ymax is not None else None, G, pool_k, self.cout, 1,
                                                    stream_ptr(dev)), "train_bn_act_maxpool")
        else:
            arg = ymax = None
            z = torch.empty((P, self.cout), dtype=BF16, device=dev)
            check(lib.s4g_train_bn_act_bf16(ptr(y), ptr(scale), ptr(shift), ptr(z), P, self.cout, 1, seed, self.drop_p,
                                            stream_ptr(dev)), "train_bn_act")
        self.saved = (x, y, wb, mean_rstd, scale, shift, arg, pool_k, seed, ymax)
        return (z, arg) if pool_k else z

    def backward(self, dz, need_dx=True, prev=None, pre=None):
        """dz: [P, cout] bf16 (or the pooled gradient [G, cout] when the forward pooled).  Accumulates the parameter
        gradients; returns dx [P, Kp or Cf] bf16 (None when not needed).
        ``pre``: dz is already masked and these are its sums (it came out of gemm_bwd).  ``prev``: the block that produced
        this block's input — dx is then returned as (masked dx, sums) for prev.backward(..., pre=sums)."""
        x, y, wb, mean_rstd, scale, shift, arg, pool_k, seed, ymax = self.saved[:10]
        split = len(self.saved) > 10
        self.saved = None
        P, C = y.shape
        dev = y.device
        drop = 0.0 if pool_k else self.drop_p
        relu = 1
        if pre is not None:
            sums, relu, drop = pre, 0, 0.0
        else:
            sums = torch.empty(2 * C, dtype=torch.float64, device=dev)
            if pool_k and ymax is not None:  # the G arg-max rows carry the whole gradient
                # ReLU' applied ONCE on the G pooled rows (y at the arg-max is ymax); both passes then skip the test
                dzm = torch.empty_like(dz)
                check(lib.s4g_train_relu_mask_rows_bf16(ptr(dz), ptr(ymax), ptr(scale), ptr(shift), P // pool_k, C, ptr(dzm),
                                                        stream_ptr(dev)), "train_relu_mask_rows")
                dz, relu = dzm, 0
                check(lib.s4g_train_bn_bwd_reduce_bf16(ptr(dz), None, 0, ptr(ymax), ptr(scale), ptr(shift), P // pool_k, C, 0,
                                                       seed, 0.0, ptr(sums), stream_ptr(dev)), "train_bn_bwd_reduce")
            elif arg is not None and arg.dtype == torch.int32:  # global pool: dz routed to row arg of its scene
                check(lib.s4g_train_bn_bwd_reduce_seg_bf16(ptr(dz), ptr(arg), pool_k, ptr(y), ptr(scale), ptr(shift), P, C,
                                                           1, ptr(sums), stream_ptr(dev)), "train_bn_bwd_reduce_seg")
            else:
                check(lib.s4g_train_bn_bwd_reduce_bf16(ptr(dz), ptr(arg) if pool_k else None, pool_k, ptr(y), ptr(scale),
                                                       ptr(shift), P, C, 1, seed, drop, ptr(sums), stream_ptr(dev)),
                      "train_bn_bwd_reduce")
        # dgamma += sum g xhat, dbeta += sum g, and dy = ka * g + kb * y + kc folded per channel — one launch
        gw, gb = _grad_buffer(self.bn.weight), _grad_buffer(self.bn.bias)
        coef = torch.empty(3 * C, dtype=torch.float32, device=dev)
        check(lib.s4g_train_bn_bwd_finalize(ptr(sums), P, C, ptr(self.bn.weight), ptr(mean_rstd), ptr(gw), ptr(gb), ptr(coef),
                                            stream_ptr(dev)), "train_bn_bwd_finalize")
        dy = torch.empty((P, C), dtype=BF16, device=dev)
        if arg is not None and arg.dtype == torch.int32:
            check(lib.s4g_train_bn_bwd_apply_seg_bf16(ptr(dz), ptr(arg), pool_k, ptr(y), ptr(scale), ptr(shift), ptr(coef),
                                                      ptr(coef[C:]), ptr(coef[2 * C:]), P, C, relu, ptr(dy), stream_ptr(dev)),
                  "train_bn_bwd_apply_seg")
        else:
            check(lib.s4g_train_bn_bwd_apply_bf16(ptr(dz), ptr(arg) if pool_k else None, pool_k, ptr(y), ptr(scale),
                                                  ptr(shift), ptr(coef), ptr(coef[C:]), ptr(coef[2 * C:]), P, C, relu, seed,
                                                  drop, ptr(dy), stream_ptr(dev)), "train_bn_bwd_apply")
        if split:
            return dy, x, wb  # the caller owns the conv (it ran on other rows)
        # dW = dY^T X: a plain library GEMM (bf16 operands, fp32 result)
        dwb = torch.mm(dy.t(), x, out_dtype=torch.float32)
        if self.cf is None:
            dw = dwb[:, :self.cin]
        else:
            dw = torch.cat([dwb[:, self.cf:self.cf + 3], dwb[:, :self.cf]], dim=1)
        _accumulate(self.conv.weight, dw.reshape(self.conv.weight.shape))
        if not need_dx:
            return None
        cols = self.cf if self.cf is not None else wb.shape[1]
        if cols == 0:
            return None
        wt = wb[:, :cols].t().contiguous()  # dX = dY · W  (B operand = W^T rows)
        if prev is None:
            return gemm(dy, wt)
        py, pscale, pshift, pseed = prev.saved[1], prev.saved[4], prev.saved[5], prev.saved[8]
        return gemm_bwd(dy, wt, py, pscale, pshift, relu=True, seed=pseed, drop_p=prev.drop_p)


def chain_backward(blocks, dz, need_dx=True):
    """backward through the blocks of one shared MLP, last to first; returns the gradient of the chain's input rows"""
    pre = None
    for j in reversed(range(len(blocks))):
        prev = blocks[j - 1] if (j > 0 and FUSED_BWD_REDUCE) else None
        out = blocks[j].backward(dz, need_dx=(j > 0 or need_dx), prev=prev, pre=pre)
        dz, pre = out if prev is not None else (out, None)
    return dz  # ((d y, x rows, weights) when the first block was built from pre-activations: Block.forward_pre)


def _sum_rows(parts):
    """sum of 2-4 equally shaped contiguous bf16 row matrices in one pass (fp32 sums, one rounding)"""
    assert 2 <= len(parts) <= 4 and all(p.dtype == BF16 and p.is_contiguous() and p.shape == parts[0].shape for p in parts)
    out = torch.empty_like(parts[0])
    q = [ptr(p) for p in parts] + [None] * (4 - len(parts))
    check(lib.s4g_train_sum_bf16(q[0], q[1], q[2], q[3], ptr(out), out.numel(), stream_ptr(out.device)), "train_sum_bf16")
    return out


# gradients of the interpolation and of the grouping as gathers over the inverted index (no atomics) or as scatters
INTERP_BWD_GATHER = True


def interp_rows_backward(dz, idx3, w, B, Nk, Nq, c2, want_f32):
    """d(sparse features) [B*Nk, c2] of out[q] = sum_k w[q,k] * sparse[idx3[q,k]] from dz [B*Nq, >= c2] bf16 (its first c2
    columns); fp32 when ``want_f32`` (it is added to another gradient), else bf16 (it feeds the next block's backward)."""
    dev = dz.device
    st = stream_ptr(dev)
    if not INTERP_BWD_GATHER:
        d_sparse = torch.zeros((B * Nk, c2), dtype=torch.float32, device=dev)
        check(lib.s4g_train_interp_rows_bwd(ptr(dz), dz.stride(0), ptr(idx3), ptr(w), B, Nk, Nq, c2, ptr(d_sparse), st),
              "train_interp_rows_bwd")
        return d_sparse if want_f32 else d_sparse.to(BF16)
    lst, end, count = _inverse_index(idx3, B, Nk, Nq * 3)
    out = torch.empty((B * Nk, c2), dtype=torch.float32 if want_f32 else BF16, device=dev)
    check(lib.s4g_train_rows_bwd_gather(ptr(dz), dz.stride(0), ptr(lst), ptr(end), ptr(count), ptr(w), 3, B * Nk, c2, 0,
                                        ptr(out) if want_f32 else None, None if want_f32 else ptr(out), st),
          "train_rows_bwd_gather")
    return out


def _inverse_index(index, B, T, E):
    """index (B, E) int32 with values in [0, T) -> (list [B*E], end [B*T], count [B*T]): per target its entries"""
    dev = index.device
    st = stream_ptr(dev)
    count = torch.empty(B * T, dtype=torch.int32, device=dev)
    check(lib.s4g_train_index_inverse_count(ptr(index), B, T, E, ptr(count), st), "train_index_inverse_count")
    end = torch.cumsum(count, 0, dtype=torch.int32)
    cursor = end - count
    lst = torch.empty(B * E, dtype=torch.int32, device=dev)
    check(lib.s4g_train_index_inverse_fill(ptr(index), B, T, E, ptr(cursor), ptr(lst), st), "train_index_inverse_fill")
    return lst, end, count


def group_rows_backward(dz, nbr, B, N, M, K, cf, dfeat):
    """dfeat[b*N + nbr[b,m,k]] += dz[(b,m,k)][:cf]  (dfeat fp32 [B*N, cf], may already hold the skip connection's gradient)"""
    dev = dz.device
    if not INTERP_BWD_GATHER:
        check(lib.s4g_train_group_rows_bwd(ptr(dz), dz.stride(0), ptr(nbr), B, N, M, K, cf, ptr(dfeat), stream_ptr(dev)),
              "train_group_rows_bwd")
        return
    lst, end, count = _inverse_index(nbr, B, N, M * K)
    check(lib.s4g_train_rows_bwd_gather(ptr(dz), dz.stride(0), ptr(lst), ptr(end), ptr(count), None, 1, B * N, cf, 1,
                                        ptr(dfeat), None, stream_ptr(dev)), "train_rows_bwd_gather")


def rows_segment_sum(dz, B, Nq, c2, out):
    """out [B, c2] fp32 += the sum over each scene's Nq rows of dz's first c2 columns (bf16 [B*Nq, >= c2]); fixed order"""
    check(lib.s4g_train_rows_segment_sum_bf16(ptr(dz), dz.stride(0), B, Nq, c2, ptr(out), stream_ptr(dz.device)),
          "train_rows_segment_sum")


def _grad_buffer(param):
    """param.grad as a contiguous fp32 tensor the kernels can add into (created as zeros when absent)"""
    if param.grad is None:
        param.grad = torch.zeros_like(param)
    assert param.grad.is_contiguous() and param.grad.dtype == torch.float32
    return param.grad


def _accumulate(param, grad):
    grad = grad.to(param.dtype)
    if param.grad is None:
        param.grad = grad.clone().reshape(param.shape)
    else:
        param.grad.add_(grad.reshape(param.shape))


def _has_training_plan(model):
    """PointNet2.fusable(), or for a configuration whose last level is one global group fusable(allow_global=True) —
    as long as a sampled level comes first: a global FIRST level has no input features, and the module path cannot run
    it either (PointNetSAModule.forward unsqueezes the absent feature)."""
    cfg = getattr(model, "config", None)
    if cfg is None or cfg["num_centroids"][-1] != 0:
        return model.fusable()
    return len(cfg["num_centroids"]) > 1 and model.fusable(allow_global=True)


class TrainEngine:
    """forward + loss + backward of PN2_CLS (PointNet2_tcls.PointNet2) or of the PN2 sibling (models.PointNet2) on the
    fused training kernels.  ``model`` on CUDA, a configuration with a training plan (PointNet2.fusable; a global last
    level paired with broadcast propagation after at least one sampled level); ``loss_fn``: the model's PointNet2Loss."""

    def __init__(self, model, loss_fn, seed=0):
        if not _has_training_plan(model):
            raise RuntimeError("TrainEngine: no fused plan for this configuration (PointNet2.fusable)")
        self.model, self.loss_fn = model, loss_fn
        self.cfg = model.config
        # a last level with one global group (num_centroids = 0) and the broadcast first propagation level it pairs with
        self.global_level = self.cfg["num_centroids"][-1] == 0
        self._global_tables = {}  # (B, N) -> (identity neighbour table (B, 1, N) int32, zero centroids (B, 3, 1))
        self.step_count = 0
        self.seed = int(seed)
        self.sequential_heads = True
        cf = 0
        self.sa = []
        for m in model.sa_modules:
            blocks = [Block(b, grouped_cf=cf if j == 0 else None) for j, b in enumerate(m.mlp)]
            self.sa.append(blocks)
            cf = blocks[-1].cout
        self.fp = [[Block(b) for b in m.mlp] for m in model.fp_modules]
        p = self.cfg["dropout_prob"]
        self.heads = [([Block(b, drop_p=dp) for b in mlp], logit) for mlp, logit, dp in (
            (model.mlp_seg, model.seg_logit, p), (model.mlp_R, model.R_logit, 0.0), (model.mlp_t, model.t_logit, 0.0),
            (model.mlp_movable, model.movable_logit[0], p))]

    def _seed(self, k):
        return (self.seed * 1000003 + self.step_count * 7919 + k * 104729 + 1) & 0x7FFFFFFF

    # ------------------------------------------------------------------ forward
    PRED_KEYS = ("score", "frame_R", "frame_t", "movable_logits")
    LOSS_KEYS = ("cls_loss", "R_loss", "t_loss", "mov_loss")  # PointNet2Loss: term k depends on head k only

    def _global_group(self, B, N, dev):
        """(identity neighbour table (B, 1, N) int32, zero centroids (B, 3, 1) fp32) of a global level over N points,
        built once per shape.  Grouped with them, the rows are [features | xyz - 0 | 0]: every point of the scene exactly
        once, with the absolute coordinates the reference concatenates (modules.py:93-98).  (Not the inference engine's
        partial groups padded with repeated points: max ignores repeats, train-mode BatchNorm statistics do not.)"""
        key = (B, N)
        if key not in self._global_tables:
            nbr = torch.arange(N, dtype=torch.int32, device=dev).expand(B, N).reshape(B, 1, N).contiguous()
            self._global_tables[key] = (nbr, torch.zeros((B, 3, 1), dtype=torch.float32, device=dev))
        return self._global_tables[key]

    def _trunk_forward(self, points):
        """set abstraction + feature propagation: points (B,3,N) fp32 -> per-point features [B*N, C] bf16"""
        cfg = self.cfg
        E = FusedPointNet2
        xyz = points.float().contiguous()
        B = xyz.shape[0]
        dev = xyz.device
        feat = None
        lv_xyz, lv_feat, self._sa_ctx = [xyz], [None], []
        for i, blocks in enumerate(self.sa):
            M, K = cfg["num_centroids"][i], cfg["num_neighbours"][i]
            N = xyz.shape[2]
            glob = M == 0
            if glob:  # one group of all N points per scene (the last level, after a sampled one: feat is set)
                M, K = 1, N
                nbr, ctr = self._global_group(B, N, dev)
            else:
                idx = E.fps(xyz, M)
                ctr = E.gather_xyz(xyz, idx)
                nbr = E.ball_query(xyz, ctr, cfg["radius"][i], K)
            cf = 0 if feat is None else feat.shape[1]
            x0 = torch.empty((B * M * K, cf + 8), dtype=BF16, device=dev)
            check(lib.s4g_train_group_rows_bf16(ptr(feat) if feat is not None else None, ptr(xyz), ptr(ctr), ptr(nbr), B, N, M,
                                                K, cf, ptr(x0), stream_ptr(dev)), "train_group_rows")
            h = x0
            for j, blk in enumerate(blocks):
                last = j == len(blocks) - 1
                h = blk.forward(h, pool_k=K if last else 0, global_pool=glob and last)
            feat, _ = h
            self._sa_ctx.append((nbr, B, N, M, K, cf, glob))
            xyz = ctr
            lv_xyz.append(xyz)
            lv_feat.append(feat)
        sparse_xyz, sparse = xyz, feat
        self._fp_ctx = []
        for i, blocks in enumerate(self.fp):
            dense_xyz, dense = lv_xyz[-2 - i], lv_feat[-2 - i]
            Nk, Nq = sparse_xyz.shape[2], dense_xyz.shape[2]
            if i == 0 and self.global_level:  # broadcast propagation: rows [global | skip] (modules.py:131-134)
                self._fp_ctx.append((None, None, B, Nk, Nq, sparse.shape[1], dense.shape[1], False))
                h = E.broadcast_concat(sparse, dense, B, Nq)
                for blk in blocks:
                    h = blk.forward(h)
                sparse_xyz, sparse = dense_xyz, h
                continue
            idx3, w = E.three_nn_weights(dense_xyz, sparse_xyz)
            split = FP_LINEAR_SPLIT and dense is None
            self._fp_ctx.append((idx3, w, B, Nk, Nq, sparse.shape[1], 0 if dense is None else dense.shape[1], split))
            if split:
                wb = blocks[0]._weight_rows()
                y = E.interp_concat(gemm(sparse, wb), idx3, w, None, B, Nk, Nq)
                h = blocks[0].forward_pre(y, sparse, wb)
                rest = blocks[1:]
            else:
                h = E.interp_concat(sparse, idx3, w, dense, B, Nk, Nq)
                rest = blocks
            for blk in rest:
                h = blk.forward(h)
            sparse_xyz, sparse = dense_xyz, h
        self._lv_shapes = [None if f is None else tuple(f.shape) for f in lv_feat]
        self._n_points = sparse_xyz.shape[2]
        self._batch = B
        self._points = points
        return sparse

    def _head_forward(self, k, point_feat):
        """head k: 4 blocks + the biased 1x1 conv -> fp32 logits (B, c, N), an autograd LEAF (the loss runs in torch)"""
        blocks, logit = self.heads[k]
        h = point_feat
        for j, blk in enumerate(blocks):
            h = blk.forward(h, seed=self._seed(10 * k + j))
        B, n = self._batch, self._n_points
        c = logit.weight.shape[0]
        w = logit.weight.detach().reshape(c, -1).contiguous()
        out = torch.empty((B, c, n), dtype=torch.float32, device=h.device)
        check(lib.s4g_train_head_logits_fwd(ptr(h), ptr(w), ptr(logit.bias), ptr(out), h.shape[0], h.shape[1], c, n,
                                            stream_ptr(h.device)), "train_head_logits_fwd")
        self._head_saved[k] = (h, w)
        return out.requires_grad_(True)

    def _head_backward(self, k, leaf):
        """leaf.grad (B, c, N) -> gradients of head k's parameters; returns d(point features) [B*N, C] bf16"""
        blocks, logit = self.heads[k]
        h, w = self._head_saved.pop(k)
        dl = leaf.grad
        B, c, n = dl.shape
        dz = torch.empty_like(h)
        check(lib.s4g_train_head_logits_bwd(ptr(dl), ptr(w), ptr(dz), h.shape[0], h.shape[1], c, n, stream_ptr(h.device)),
              "train_head_logits_bwd")
        # dW [c][C] and dbias [c] of the final conv: one pass over h with fp32 atomics into param.grad (as library calls:
        # four skinny GEMMs of 0.2-0.5 ms each for 0.03 ms of traffic)
        check(lib.s4g_train_head_logits_dw(ptr(dl), ptr(h), ptr(_grad_buffer(logit.weight)), ptr(_grad_buffer(logit.bias)),
                                           h.shape[0], h.shape[1], c, n, stream_ptr(h.device)), "train_head_logits_dw")
        return chain_backward(blocks, dz)

    def _predictions(self, leaves):
        raw = {"score": leaves[0], "frame_R": leaves[1], "frame_t": leaves[2], "movable_logits": torch.sigmoid(leaves[3])}
        return self.model.predictions(raw, self._points)

    def forward(self, points):
        """points (B,3,N) fp32 CUDA -> predictions (fp32 (B, c, N) autograd leaves underneath); keeps what backward needs."""
        self._head_saved = {}
        self._point_feat = self._trunk_forward(points)
        self._head_leaves = [self._head_forward(k, self._point_feat) for k in range(4)]
        return self._predictions(self._head_leaves)

    # ------------------------------------------------------------------ backward
    def backward(self):
        """after ``total_loss.backward()`` filled the head leaves' gradients"""
        dzs = [self._head_backward(k, leaf) for k, leaf in enumerate(self._head_leaves)]
        self._head_leaves = self._point_feat = None
        self._trunk_backward(_sum_rows(dzs))

    def _trunk_backward(self, d_out):
        """d_out: gradient of the per-point features [B*N, C] bf16"""
        dev = d_out.device
        # gradient buffers of the level features (fp32: they receive scatter-adds), index = level
        lv_grad = [None if s is None else torch.zeros(s, dtype=torch.float32, device=dev) for s in self._lv_shapes]
        n_fp = len(self.fp)
        # d_out = gradient of the current propagation level's OUTPUT rows
        for i in reversed(range(n_fp)):
            idx3, w, B, Nk, Nq, c2, c1, split = self._fp_ctx[i]
            if split:
                blk0 = self.fp[i][0]
                dy, x_sparse, wb = chain_backward(self.fp[i], d_out)  # d(pre-activations) of the first block, dense rows
                d_ys = interp_rows_backward(dy, idx3, w, B, Nk, Nq, blk0.cout, want_f32=False)
                del dy
                _accumulate(blk0.conv.weight, torch.mm(d_ys.t(), x_sparse, out_dtype=torch.float32)[:, :blk0.cin]
                            .reshape(blk0.conv.weight.shape))
                d_feat = gemm(d_ys, wb[:, :c2].t().contiguous())  # gradient of the sparse level's features [B*Nk, c2]
                if i == 0:
                    lv_grad[-1].add_(d_feat)
                else:
                    d_out = d_feat
                continue
            dz = chain_backward(self.fp[i], d_out)
            # dz rows = [d interpolated (c2) | d dense skip (c1)]
            if c1:
                lv_grad[-2 - i].add_(dz[:, c2:c2 + c1])
            if idx3 is None:  # broadcast level: the global feature's gradient is the sum over each scene's rows
                rows_segment_sum(dz, B, Nq, c2, lv_grad[-1])
                continue
            d_sparse = interp_rows_backward(dz, idx3, w, B, Nk, Nq, c2, want_f32=(i == 0))
            if i == 0:
                lv_grad[-1].add_(d_sparse)  # the coarsest propagation level interpolates the last SA level's features
            else:
                d_out = d_sparse
        for i in reversed(range(len(self.sa))):
            blocks = self.sa[i]
            nbr, B, N, M, K, cf, glob = self._sa_ctx[i]
            dz = lv_grad[i + 1].to(BF16)  # pooled gradient [B*M, cout]
            lv_grad[i + 1] = None
            dz = chain_backward(blocks, dz, need_dx=cf > 0)
            if cf > 0 and glob:  # identity grouping: row b*N + n of the group is point n of scene b
                lv_grad[i].add_(dz[:, :cf])
            elif cf > 0:
                group_rows_backward(dz, nbr, B, N, M, K, cf, lv_grad[i])
        self._sa_ctx = self._fp_ctx = None

    def _separable(self):
        """PointNet2Loss's four terms depend on one head each (cls <- score, R <- frame_R, t <- frame_t, mov <-
        movable_logits, reference :162-219; the PN2 sibling's loss likewise, through its prediction mapping): the heads
        can then run forward + loss term + backward ONE AFTER THE OTHER, so only one head's activations are alive at a
        time (-13 GB at 32 scenes)."""
        from .network_models.models import PointNet2, PointNet2_tcls
        return self.sequential_heads and type(self.loss_fn) in (PointNet2_tcls.PointNet2Loss, PointNet2.PointNet2Loss)

    def _placeholder(self, k):
        """the value fed for head k's raw output while another head's loss term is computed: zeros, except a 6-D
        rotation representation (the PN2 sibling's frame_R), whose Gram-Schmidt divides 0 by 0 — the identity there"""
        B, n = self._batch, self._n_points
        logit = self.heads[k][1]
        z = torch.zeros((B, logit.weight.shape[0], n), dtype=torch.float32, device=logit.weight.device)
        if k == 1 and z.shape[1] == 6:
            z[:, 0] = 1.0
            z[:, 4] = 1.0
        return z

    def step_loss(self, data_batch, labels):
        """forward + loss + full backward; returns the (detached) loss dict.  Gradients accumulate in param.grad."""
        self.step_count += 1
        points = data_batch["scene_points"]
        with torch.cuda.device(points.device):
            if not self._separable():
                with torch.enable_grad():
                    preds = self.forward(points)
                    losses = self.loss_fn(preds, labels)
                    sum(losses.values()).backward()
                with torch.no_grad():
                    self.backward()
                return {k: v.detach() for k, v in losses.items()}
            self._head_saved = {}
            with torch.no_grad():
                point_feat = self._trunk_forward(points)
            zeros = [self._placeholder(k) for k in range(4)]
            losses, dzs = {}, []
            for k in range(4):
                with torch.no_grad():
                    leaf = self._head_forward(k, point_feat)
                with torch.enable_grad():
                    leaves = [leaf if j == k else zeros[j] for j in range(4)]
                    term = self.loss_fn(self._predictions(leaves), labels)[self.LOSS_KEYS[k]]
                    term.backward()
                losses[self.LOSS_KEYS[k]] = term.detach()
                with torch.no_grad():
                    dzs.append(self._head_backward(k, leaf))  # (bf16 [B*N, C]: 0.4 GB each at 32 scenes)
                del leaf
            with torch.no_grad():
                d_out = _sum_rows(dzs)
                del dzs
                self._trunk_backward(d_out)
        return losses
