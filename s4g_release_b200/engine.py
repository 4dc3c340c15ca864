"""Fused inference engine for PN2_CLS on one B200.

Geometry (FPS, ball query, 3-NN) runs in fp32 with the hand-written sm_100a kernels through the C ABI
(int32 indices, no transposed copies).  The shared MLPs (set abstraction incl. gather + max-pool,
feature propagation, heads) run as fused chains with eval-mode BatchNorm folded into a per-channel
scale/shift (reference nn_utils/conv.py:70-76 → y = relu(W'x + b')).

``mlp_backend``
  * ``"tcgen05"`` — the product path: csrc/mlp_chain.cu (bf16 operands, fp32 accumulation in TMEM);
  * ``"tf32"``    — the tight-parity mode (SURVEY.md §7): every layer is one csrc/linear_tf32.cu launch
    (tcgen05 kind::tf32: 10-bit-mantissa operands rounded to nearest, fp32 accumulation, fp32 activations
    in HBM between layers) — the arithmetic the unmodified reference gets from cuDNN's TF32 default on this
    GPU.  Unfused, so slow; selected explicitly (``FusedPointNet2(model, mlp_backend="tf32")``);
  * ``"torch"``   — plain torch fp32 matmuls on the same folded weights.  Kept ONLY as the on-device
    fp32 reference the numerics tests compare the tcgen05 kernels against; it is not a fallback —
    nothing selects it implicitly.
"""
import json
import os

import numpy as np
import torch

from ._lib import check, lib, ptr, stream_ptr
from .chain import IN_GATHER, IN_GATHER_EDGE, IN_ROWS, OUT_LOGITS, OUT_MAXPOOL, OUT_ROWS, MlpChain

BN_EPS = 1e-5
GLOBAL_GROUPS = (8, 16, 32, 64)  # the max-pool group sizes the chain planner accepts


def global_group_table(n):
    """Neighbour table of a global set-abstraction level over n points (num_centroids = 0: one group of the whole cloud,
    pointnet2_utils/modules.py:93-98).  The gathered max-pool chain pools groups of 8 / 16 / 32 / 64 rows, so the cloud
    is cut into P = ceil(n / g) partial groups of g rows — g the smallest such size >= n, else 64 — and the last group is
    padded with index j % n, a real point of the same scene.  The partial maxima are reduced afterwards; max ignores
    order and repeated rows, so the result is that of one n-wide group.  -> (g, P, int32 indices [P * g])."""
    g = next((k for k in GLOBAL_GROUPS if k >= n), GLOBAL_GROUPS[-1])
    p = -(-n // g)
    return g, p, np.arange(p * g, dtype=np.int32) % n


class StageTimer:
    """CUDA-event stopwatch for the stages of one forward, recorded on the launching stream."""

    def __init__(self):
        self.records = []

    def section(self, name):
        return _Section(self, name)

    def totals_ms(self):
        """{name: [ms per occurrence]} — call after torch.cuda.synchronize()."""
        out = {}
        for name, a, b in self.records:
            out.setdefault(name, []).append(a.elapsed_time(b))
        return out


class _Section:
    def __init__(self, timer, name):
        self.timer, self.name = timer, name

    def __enter__(self):
        if self.timer is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if self.timer is not None:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            self.timer.records.append((self.name, self.a, b))
        return False


def _sec(timer, name):
    return _Section(timer, name)


def _fold_block(block):
    """conv (no bias) + BN(eval) -> (W', b') with y = W' x + b'."""
    w = block.conv.weight.detach().float()
    w = w.reshape(w.shape[0], w.shape[1])
    bn = block.bn
    scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
    shift = bn.bias.detach().float() - bn.running_mean.detach().float() * scale
    return (w * scale[:, None]).contiguous(), shift.contiguous()


def _fold_mlp(mlp):
    return [_fold_block(b) for b in mlp]


# Plan constraints (slots, pairs, coop, subs, tma_in) per chain signature.  Every plan computes the SAME bits (the
# K-blocks of a layer are accumulated in the same order whatever the ring sizes / loop order / pairing:
# tests/test_chain_gpu.py::test_every_tunable_plan_is_bit_identical), so the choice is purely a matter of speed; it is
# still made reproducible: the picks measured on a B200 (148 SMs) are COMMITTED in tuned_plans.json and every process
# uses them; only a signature the table does not know is timed (once per process, ~0.5 s per shape) and remembered in
# the user's cache directory.
_HERE = os.path.dirname(os.path.abspath(__file__))
PLAN_TABLE = os.path.join(_HERE, "tuned_plans.json")
USER_PLAN_TABLE = os.path.join(os.environ.get("XDG_CACHE_HOME", os.path.expanduser("~/.cache")), "s4g_release_b200",
                               "tuned_plans.json")
DEFAULT_PLAN = (0, -1, -1, 1, 0)
_TUNED_SLOTS = {}      # signature -> plan, this process (table entries + what was tuned here)
_TUNED_HERE = {}       # the subset measured by this process (export_tuned_plans)
_TABLES_LOADED = set()


def _chain_signature(layers, in_mode, feat_c, out_mode, group):
    return (tuple((int(w.shape[1]), int(w.shape[0])) for w, _, _ in layers), in_mode, feat_c, out_mode, group)


def _table_key(device):
    props = torch.cuda.get_device_properties(device)
    return "sm%d%d:%d:v%d" % (props.major, props.minor, props.multi_processor_count, lib.s4g_version())


def _load_plan_tables(device):
    key = _table_key(device)
    if key in _TABLES_LOADED:
        return
    _TABLES_LOADED.add(key)
    for path in (PLAN_TABLE, USER_PLAN_TABLE):
        try:
            table = json.load(open(path)).get(key, {})
        except (OSError, ValueError):
            continue
        for sig, plan in table.items():
            _TUNED_SLOTS.setdefault(_sig_from_str(sig), tuple(plan))


def _sig_to_str(sig):
    return json.dumps([list(map(list, sig[0]))] + list(sig[1:]))


def _sig_from_str(text):
    v = json.loads(text)
    return (tuple(tuple(x) for x in v[0]),) + tuple(v[1:])


def export_tuned_plans(device=None):
    """{table key: {signature: plan}} of what THIS process measured (for regenerating tuned_plans.json)."""
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else device
    return {_table_key(device): {_sig_to_str(k): list(v) for k, v in _TUNED_HERE.items()}}


def _remember_plan(device, sig, plan):
    _TUNED_SLOTS[sig] = plan
    _TUNED_HERE[sig] = plan
    try:  # best effort: a read-only home must not break inference
        os.makedirs(os.path.dirname(USER_PLAN_TABLE), exist_ok=True)
        try:
            table = json.load(open(USER_PLAN_TABLE))
        except (OSError, ValueError):
            table = {}
        table.setdefault(_table_key(device), {})[_sig_to_str(sig)] = list(plan)
        tmp = USER_PLAN_TABLE + ".%d.tmp" % os.getpid()
        json.dump(table, open(tmp, "w"), indent=1)
        os.replace(tmp, USER_PLAN_TABLE)
    except OSError:
        pass


def candidate_plans(in_mode, feat_c, out_mode):
    """Every (slots, pairs, coop, subs, tma_in) constraint set the tuner tries (the planner refuses the infeasible ones)."""
    cands = [DEFAULT_PLAN] + [(sl, pr, co, 1, 0) for sl in (3, 4, 5) for pr in (1, 0) for co in (-1, 0, 2)]
    # two row blocks per tile (two 128-row tiles interleaved layer by layer): only narrow chains have the shared
    # memory for it; the planner refuses the others
    cands += [(sl, -1, co, 2, 0) for sl in (0, 3, 4, 5) for co in (-1, 0, 1)]
    # the same plans with the input blocks fetched by TMA: tensor copies for row chains (refused unless
    # cin % 64 == 0), tile::gather4 copies of the neighbours' feature rows for gathered max-pool chains
    if (in_mode == IN_ROWS and out_mode != OUT_MAXPOOL) or (in_mode in (IN_GATHER, IN_GATHER_EDGE) and feat_c > 0):
        cands += [c[:4] + (1,) for c in cands]
    return cands


class FusedPointNet2:
    def __init__(self, model, mlp_backend="tcgen05", autotune=True, fp_linear_split=True):
        self.cfg = model.config
        # autotune: True = committed / cached plan table, time only unknown chain shapes; False = table or the planner's
        # own choice, never time anything; "force" = re-time every shape (to regenerate tuned_plans.json)
        self.autotune = autotune if autotune == "force" else bool(autotune)
        self._copy_stream = None
        self._geom_stream = None
        self.overlap_geometry = True  # 3-NN searches on a side stream beside the next level's sampling
        self.fp_linear_split = fp_linear_split
        self.device = next(model.parameters()).device
        if self.device.type != "cuda":
            raise RuntimeError("FusedPointNet2 needs the model on a CUDA device (there is no CPU path)")
        self.mlp_backend = mlp_backend
        # a last level with one global group (num_centroids = 0) and the broadcast propagation level it pairs with
        # (num_fp_neighbours[0] = 0); PointNet2.fusable(allow_global=True) admits only that pairing
        self.global_level = self.cfg["num_centroids"][-1] == 0
        self._global_tables = {}  # (B, N) -> (g, neighbour table (B,P,g) int32, zero centroids (B,3,P))
        self._global_chains = {}  # g -> max-pool chain of the global level
        self.sa = [_fold_mlp(m.mlp) for m in model.sa_modules]
        self.fp = [_fold_mlp(m.mlp) for m in model.fp_modules]
        heads = []
        for mlp, logit in self._head_modules(model):
            w = logit.weight.detach().float()
            heads.append((_fold_mlp(mlp), w.reshape(w.shape[0], w.shape[1]).contiguous(),
                          logit.bias.detach().float().contiguous()))
        self.heads = heads
        if mlp_backend == "tcgen05":
            self._build_chains()
        elif mlp_backend == "tf32":
            self._prepare_tf32()
        elif mlp_backend != "torch":
            raise ValueError("mlp_backend must be 'tcgen05', 'tf32' or 'torch'")

    _HEAD_SIGMOID = (False, False, False, True)  # per head of _head_modules: the logits epilogue applies a sigmoid

    @staticmethod
    def _head_modules(model):
        """(SharedMLP, logit conv) of each head, in the order of the head stage's outputs."""
        return ((model.mlp_seg, model.seg_logit), (model.mlp_R, model.R_logit), (model.mlp_t, model.t_logit),
                (model.mlp_movable, model.movable_logit[0]))

    def _make_chain(self, layers, in_mode, feat_c, out_mode, group=1, sigmoid=False):
        """Builds one chain.  The planner ranks the shared-memory splits (activation slots vs weight stages) with a
        simulation that is only roughly calibrated, so with ``autotune`` the alternatives (3 / 4 / 5 slots, accumulator
        pairs on / off, cooperative epilogues on / off, one or two row blocks per tile) are timed
        once per chain shape on synthetic rows and the fastest is pinned (set-abstraction level 2: 3.6 -> 2.8 ms)."""
        sig = _chain_signature(layers, in_mode, feat_c, out_mode, group)
        _load_plan_tables(self.device)
        if self.autotune == "force" or (self.autotune and sig not in _TUNED_SLOTS):
            _remember_plan(self.device, sig, self._tune_slots(layers, in_mode, feat_c, out_mode, group, sigmoid))
        slots, pairs, coop, subs, tma = _TUNED_SLOTS.get(sig, DEFAULT_PLAN)
        return MlpChain(layers, self.device, in_mode, feat_c, out_mode, group=group, sigmoid=sigmoid, slots=slots,
                        pairs=pairs, coop=coop, subs=subs, tma_in=tma)

    def _tune_slots(self, layers, in_mode, feat_c, out_mode, group, sigmoid):
        dev = self.device
        g = torch.Generator(device=dev).manual_seed(0)
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        tiles = sms * 48  # 48 tiles per SM: steady state dominates
        rows = tiles * 128
        # the synthetic input + output must fit comfortably beside the caller's tensors (a shared GPU): <= 1/8 of free
        free_bytes = torch.cuda.mem_get_info(dev)[0]
        row_bytes = 2 * (layers[0][0].shape[1] + max(feat_c, 0) + layers[-1][0].shape[0] + 8)
        while rows * row_bytes > free_bytes // 8 and tiles > sms * 4:
            tiles //= 2
            rows = tiles * 128
        if in_mode in (IN_GATHER, IN_GATHER_EDGE):
            K = group
            M = rows // K
            N = 4 * M
            xyz = torch.rand(1, 3, N, device=dev, generator=g)
            ctr = xyz[:, :, :M].contiguous()
            # neighbours are LOCAL in a real scene (ball query): indices near the centroid's own, not uniform over the cloud
            near = torch.randint(0, 512, (1, M, K), device=dev, dtype=torch.int64, generator=g)
            nbr = ((torch.arange(M, device=dev).view(1, M, 1) * (N // M) + near) % N).to(torch.int32)
            feat = torch.randn(N, feat_c, device=dev, generator=g).to(torch.bfloat16) if feat_c else None
            term = None
            if in_mode == IN_GATHER_EDGE:
                term = torch.randn(M, layers[0][0].shape[0], device=dev, generator=g).to(torch.bfloat16)
            run = lambda ch: ch.run_gather(feat, xyz, ctr, nbr, term)
        else:
            x = torch.randn(rows, layers[0][0].shape[1], device=dev, generator=g).to(torch.bfloat16)
            n_points = rows if out_mode == OUT_LOGITS else 0
            run = lambda ch: ch.run_rows(x, n_points=n_points)
        best, best_ms = DEFAULT_PLAN, None
        seen = set()
        candidates = candidate_plans(in_mode, feat_c, out_mode)
        for slots, pairs, coop, subs, tma in candidates:
            try:
                ch = MlpChain(layers, dev, in_mode, feat_c, out_mode, group=group, sigmoid=sigmoid, slots=slots,
                              pairs=pairs, coop=coop, subs=subs, tma_in=tma)
            except RuntimeError:
                continue  # no deadlock-free plan under these constraints
            plan = (ch.describe(), tma)
            if plan in seen:  # different constraints, same job streams
                continue
            seen.add(plan)
            try:
                run(ch)
            except RuntimeError:
                if not tma:
                    raise
                continue  # (a driver without cuTensorMapEncodeTiled: stay on the cp.async input path)
            ts = []
            for _ in range(5):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                run(ch)
                b.record()
                torch.cuda.synchronize(dev)
                ts.append(a.elapsed_time(b))
            ms = min(ts)
            if best_ms is None or ms < best_ms * 0.97:  # keep the planner's choice unless another is clearly faster
                best, best_ms = (slots, pairs, coop, subs, tma), ms
            del ch
        return best

    def _row_chains(self, layers):
        """Split a row chain wherever a hidden activation is too wide to stay on chip (> 512 channels)."""
        chains, cur = [], []
        for i, (w, b) in enumerate(layers):
            cur.append((w, b, True))
            if i + 1 < len(layers) and w.shape[0] > 512:
                chains.append(self._make_chain(cur, IN_ROWS, 0, OUT_ROWS))
                cur = []
        chains.append(self._make_chain(cur, IN_ROWS, 0, OUT_ROWS))
        return chains

    def _build_chains(self):
        cfg = self.cfg
        self.sa_chains = []  # the sampled levels
        feat_c = 0
        for i, layers in enumerate(self.sa[:len(self.sa) - self.global_level]):
            self.sa_chains.append(self._sa_chain(i, layers, feat_c))
            feat_c = layers[-1][0].shape[0]
        self._global_feat_c = feat_c
        if self.global_level and self.sa_chains:  # the global level's cloud size is the previous level's centroid count
            self._global_chain(global_group_table(cfg["num_centroids"][-2])[0])
        # Propagation levels WITHOUT a skip feature (the finest one of PN2_CLS: 25 600 queries from 5 120 keys): the first
        # conv commutes with the interpolation — W (sum_k w_k f_k) + b = sum_k w_k (W f_k + b), the weights sum to one —
        # so it runs on the sparse rows (5x fewer), the interpolation kernel gathers the 256-wide pre-activations
        # instead of the 512-wide features and applies the ReLU, and the 1.6 GB concat input is never written.
        self.fp_pre, self.fp_chains = [], []
        skip_c = [0] + [layers[-1][0].shape[0] for layers in self.sa]
        for i, layers in enumerate(self.fp):
            pre, chains = self._fp_chain(i, layers, skip_c[-2 - i])
            self.fp_pre.append(pre)
            self.fp_chains.append(chains)
        self.head_chains = []
        for k, (layers, w, b) in enumerate(self.heads):
            self.head_chains.append(self._make_chain([(lw, lb, True) for lw, lb in layers] + [(w, b, False)], IN_ROWS, 0,
                                                     OUT_LOGITS, sigmoid=self._HEAD_SIGMOID[k]))

    def _fp_chain(self, i, layers, skip_c):
        """Propagation level i's chains over a skip feature of skip_c channels (0: none) -> (the first layer on the
        sparse rows, or None; the row chains)."""
        broadcast = i == 0 and self.global_level
        if self.fp_linear_split and not broadcast and skip_c == 0 and len(layers) > 1 and layers[0][0].shape[0] <= 512:
            w0, b0 = layers[0]
            return self._make_chain([(w0, b0, False)], IN_ROWS, 0, OUT_ROWS), self._row_chains(layers[1:])
        return None, self._row_chains(layers)

    def _sa_chain(self, i, layers, feat_c):
        """The gathered max-pool chain of sampled level i over a feature table of feat_c channels."""
        return self._make_chain([(w, b, True) for w, b in layers], IN_GATHER, feat_c, OUT_MAXPOOL,
                                group=self.cfg["num_neighbours"][i])

    def _sa_level(self, i, feat, xyz, new_xyz, nbr, idx, timer):
        """Sampled level i's MLP + max-pool on the tcgen05 trunk: bf16 [B*N, C] (or None) -> bf16 [B*M, C'].  ``idx``:
        the level's sampled indices (B, M)."""
        with _sec(timer, "sa%d.mlp" % i):
            return self.sa_chains[i].run_gather(feat, xyz, new_xyz, nbr)

    def _sa_reference(self, i, xyz, feat, new_xyz, nbr, idx, layers):
        """Sampled level i on the torch / tf32 backends: (B, N, C) fp32 (or None) -> (B, M, C')."""
        return self._sa_torch(xyz, feat, new_xyz, nbr, layers)

    def _global_chain(self, g):
        """The global level's max-pool chain for groups of g rows (g follows the cloud size, see global_group_table)."""
        if g not in self._global_chains:
            self._global_chains[g] = self._make_chain([(w, b, True) for w, b in self.sa[-1]], IN_GATHER,
                                                      self._global_feat_c, OUT_MAXPOOL, group=g)
        return self._global_chains[g]

    def _global_group(self, B, n):
        """(g, neighbour table (B,P,g) int32, zero centroids (B,3,P) fp32) of a global level over n points; built once
        per shape from the host, so a forward launches nothing for them.  With zero centroids the chain's relative
        coordinates x - 0 are the absolute coordinates the reference concatenates (modules.py:97-98)."""
        key = (B, n)
        if key not in self._global_tables:
            g, p, idx = global_group_table(n)
            nbr = np.ascontiguousarray(np.broadcast_to(idx.reshape(1, p, g), (B, p, g)))
            self._global_tables[key] = (g, torch.from_numpy(nbr).to(self.device),
                                        torch.from_numpy(np.zeros((B, 3, p), np.float32)).to(self.device))
        return self._global_tables[key]

    def tolerance(self):
        """Max abs error of the head outputs relative to max(|ref|, 1) against the fp32 oracle."""
        return {"torch": 2e-3, "tf32": 4e-3}.get(self.mlp_backend, 6e-2)

    # ---------------------------------------------------------------- tight-parity TF32 layers (csrc/linear_tf32.cu)
    @staticmethod
    def _round_tf32(t):
        """fp32 -> nearest TF32 (10-bit mantissa, ties away from zero = cvt.rna.tf32.f32), kept in fp32 storage."""
        bits = t.contiguous().view(torch.int32)
        return ((bits + 0x1000) & ~0x1FFF).view(torch.float32)

    def _prepare_tf32(self):
        """Weights rounded to TF32 once and padded to a multiple of 4 input channels (16-byte rows for the TMA map)."""
        def prep(w, b):
            k = w.shape[1]
            wp = torch.zeros((w.shape[0], (k + 3) // 4 * 4), dtype=torch.float32, device=self.device)
            wp[:, :k] = self._round_tf32(w.to(self.device))
            return wp, b.to(self.device).contiguous()
        self.sa = [[prep(w, b) for w, b in layers] for layers in self.sa]
        self.fp = [[prep(w, b) for w, b in layers] for layers in self.fp]
        self.heads = [([prep(w, b) for w, b in layers],) + prep(w, b) for layers, w, b in self.heads]

    @staticmethod
    def linear_tf32(x, w, shift, relu=True, round_out=True):
        """x fp32 [P, K'] (K' <= w.shape[1], row stride a multiple of 4), w fp32 [N, K4] -> fp32 [P, N]."""
        P, N, K = x.shape[0], w.shape[0], w.shape[1]
        if x.shape[1] != K or x.stride(1) != 1 or x.stride(0) % 4 != 0 or x.data_ptr() % 16 != 0:
            xp = torch.zeros((P, K), dtype=torch.float32, device=x.device)
            xp[:, :x.shape[1]] = x
            x = xp
        y = torch.empty((P, N), dtype=torch.float32, device=x.device)
        check(lib.s4g_linear_tf32(ptr(x), x.stride(0), ptr(w), w.stride(0), ptr(shift), ptr(y), N, P, N, K,
                                  1 if relu else 0, 1 if round_out else 0, stream_ptr(x.device)), "linear_tf32")
        return y

    def _mlp(self, x, layers):
        """(..., Cin) channel-last through [(W', b')] with ReLU — torch fp32 or one TF32 tensor-core launch per layer."""
        if self.mlp_backend != "tf32":
            return self._chain_torch(x, layers)
        lead = x.shape[:-1]
        h = self._round_tf32(x.reshape(-1, x.shape[-1]))
        for w, b in layers:
            h = self.linear_tf32(h, w, b)
        return h.reshape(*lead, h.shape[-1])

    def _logits(self, h, w, b):
        if self.mlp_backend != "tf32":
            return torch.matmul(h, w.t()) + b
        lead = h.shape[:-1]
        return self.linear_tf32(h.reshape(-1, h.shape[-1]), w, b, relu=False, round_out=False).reshape(*lead, w.shape[0])

    # ---------------------------------------------------------------- geometry (fp32, exact)
    @staticmethod
    def fps(xyz, m):
        B, _, N = xyz.shape
        idx = torch.empty((B, m), dtype=torch.int32, device=xyz.device)
        check(lib.s4g_farthest_point_sample_f32_i32(ptr(xyz), B, N, m, ptr(idx), stream_ptr(xyz.device)), "fps")
        return idx

    @staticmethod
    def ball_query(xyz, new_xyz, radius, k):
        B, _, N = xyz.shape
        M = new_xyz.shape[2]
        idx = torch.empty((B, M, k), dtype=torch.int32, device=xyz.device)
        check(lib.s4g_ball_query_f32_i32(ptr(xyz), ptr(new_xyz), B, N, M, float(radius), k, ptr(idx), None,
                                         stream_ptr(xyz.device)), "ball_query")
        return idx

    @staticmethod
    def three_nn(query, key):
        B, _, Nq = query.shape
        Nk = key.shape[2]
        idx = torch.empty((B, Nq, 3), dtype=torch.int64, device=query.device)
        d2 = torch.empty((B, Nq, 3), dtype=torch.float32, device=query.device)
        check(lib.s4g_point_search_f32(ptr(query), ptr(key), B, Nq, Nk, 3, ptr(idx), ptr(d2),
                                       stream_ptr(query.device)), "point_search")
        return idx, d2

    # ---------------------------------------------------------------- torch fp32 reference MLPs
    @staticmethod
    def _chain_torch(x, layers):
        """x: (..., Cin) channel-last; layers: [(W', b')]."""
        for w, b in layers:
            x = torch.relu(torch.addmm(b, x.reshape(-1, x.shape[-1]), w.t()).reshape(*x.shape[:-1], w.shape[0]))
        return x

    def _sa_torch(self, xyz, feat_cl, new_xyz, nbr, layers, chunk=4, ctr_feat=None):
        """xyz (B,3,N); feat_cl (B,N,C) or None; nbr (B,M,K) -> (B,M,Cout) channel-last.  ``ctr_feat`` (B,M,C): an edge
        level's centroid features; the rows are then EdgeQueryGrouper's [x_j - x_c | f_j | f_j - f_c]."""
        B, M, K = nbr.shape
        out = []
        xyz_cl = xyz.transpose(1, 2)  # (B,N,3)
        ctr_cl = new_xyz.transpose(1, 2)  # (B,M,3)
        for b0 in range(0, B, chunk):
            sl = slice(b0, b0 + chunk)
            idx = nbr[sl].long().reshape(nbr[sl].shape[0], M * K)
            g_xyz = torch.gather(xyz_cl[sl], 1, idx.unsqueeze(-1).expand(-1, -1, 3)).reshape(-1, M, K, 3)
            g = g_xyz - ctr_cl[sl].unsqueeze(2)
            if feat_cl is not None:
                C = feat_cl.shape[-1]
                g_f = torch.gather(feat_cl[sl], 1, idx.unsqueeze(-1).expand(-1, -1, C)).reshape(-1, M, K, C)
                parts = [g, g_f] if ctr_feat is None else [g, g_f, g_f - ctr_feat[sl].unsqueeze(2)]
                g = torch.cat(parts, dim=-1)
            out.append(self._mlp(g, layers).max(dim=2)[0])
        return torch.cat(out, 0)

    def _fp_torch(self, dense_xyz, sparse_xyz, dense_cl, sparse_cl, layers):
        _, interp = self._interp_torch(dense_xyz, sparse_xyz, sparse_cl)
        x = interp if dense_cl is None else torch.cat([interp, dense_cl], dim=-1)
        return self._mlp(x, layers)

    def _interp_torch(self, dense_xyz, sparse_xyz, sparse_cl):
        """FeatureInterpolator's 3-NN interpolation: -> (the neighbours' features (B, Nq, 3, C), interpolated (B, Nq, C))."""
        idx, d2 = self.three_nn(dense_xyz, sparse_xyz)
        inv = 1.0 / torch.clamp(d2, min=1e-10)
        w = inv / inv.sum(dim=2, keepdim=True)
        B, Nq, _ = idx.shape
        C = sparse_cl.shape[-1]
        g = torch.gather(sparse_cl, 1, idx.reshape(B, Nq * 3, 1).expand(-1, -1, C)).reshape(B, Nq, 3, C)
        # reference order of the 3-term sum: fma(in2,w2,fma(in1,w1,in0*w0))
        interp = g[:, :, 0] * w[:, :, 0:1]
        interp = torch.addcmul(interp, g[:, :, 1], w[:, :, 1:2])
        interp = torch.addcmul(interp, g[:, :, 2], w[:, :, 2:3])
        return g, interp

    # ---------------------------------------------------------------- fused-path helpers
    @staticmethod
    def gather_xyz(xyz, idx):
        B, _, N = xyz.shape
        M = idx.shape[1]
        out = torch.empty((B, 3, M), dtype=torch.float32, device=xyz.device)
        check(lib.s4g_gather_xyz_f32_i32(ptr(xyz), ptr(idx), B, N, M, ptr(out), stream_ptr(xyz.device)), "gather_xyz")
        return out

    @staticmethod
    def three_nn_weights(query, key):
        B, _, Nq = query.shape
        Nk = key.shape[2]
        idx = torch.empty((B, Nq, 3), dtype=torch.int32, device=query.device)
        w = torch.empty((B, Nq, 3), dtype=torch.float32, device=query.device)
        check(lib.s4g_three_nn_weights_f32_i32(ptr(query), ptr(key), B, Nq, Nk, ptr(idx), ptr(w),
                                               stream_ptr(query.device)), "three_nn_weights")
        return idx, w

    @staticmethod
    def interp_concat(sparse, idx, w, dense, B, Nk, Nq, relu=False):
        C2 = sparse.shape[1]
        C1 = dense.shape[1] if dense is not None else 0
        out = torch.empty((B * Nq, C2 + C1), dtype=torch.bfloat16, device=sparse.device)
        check(lib.s4g_interp_concat_act_bf16(ptr(sparse), ptr(idx), ptr(w), ptr(dense) if dense is not None else None,
                                             B, Nk, Nq, C2, C1, 1 if relu else 0, ptr(out), stream_ptr(sparse.device)),
              "interp_concat")
        return out

    @staticmethod
    def rows_segment_max(rows, B):
        """bf16 [B*P, C] -> [B, C]: the max over each scene's P rows."""
        C = rows.shape[1]
        out = torch.empty((B, C), dtype=torch.bfloat16, device=rows.device)
        check(lib.s4g_rows_segment_max_bf16(ptr(rows), B, rows.shape[0] // B, C, ptr(out), stream_ptr(rows.device)),
              "rows_segment_max")
        return out

    @staticmethod
    def broadcast_concat(sparse, dense, B, Nq):
        """sparse bf16 [B, C2], dense bf16 [B*Nq, C1] or None -> [B*Nq, C2 + C1] rows [sparse | dense]."""
        C2 = sparse.shape[1]
        C1 = dense.shape[1] if dense is not None else 0
        out = torch.empty((B * Nq, C2 + C1), dtype=torch.bfloat16, device=sparse.device)
        check(lib.s4g_broadcast_concat_bf16(ptr(sparse), ptr(dense) if dense is not None else None, B, Nq, C2, C1,
                                            ptr(out), stream_ptr(sparse.device)), "broadcast_concat")
        return out

    def _side_three_nn(self, pending, early_nn, device):
        """Issues a propagation level's 3-NN search on the side stream once ``pending``'s ready event has fired."""
        dense_p, sparse_p, ready, fp_level = pending
        if self._geom_stream is None:
            self._geom_stream = torch.cuda.Stream(device=device)
        self._geom_stream.wait_event(ready)
        with torch.cuda.stream(self._geom_stream):
            found = self.three_nn_weights(dense_p, sparse_p)
            done = torch.cuda.Event()
            done.record()
        early_nn[fp_level] = (found, done)

    def _trunk_tcgen05(self, points, trace, timer=None):
        """Set abstraction + feature propagation -> (cloud (B,3,N) fp32, per-point features bf16 [B*N, C] channel-last,
        the set-abstraction levels' features).  ``trace``: dict that receives the sampled indices, or None."""
        cfg = self.cfg
        xyz = points.float().contiguous()
        B = xyz.shape[0]
        feat = None  # bf16 [B*N, C] channel-last
        lv_xyz, lv_feat = [xyz], [None]
        # The 3-NN searches of the propagation levels only need coordinates.  Farthest point sampling of levels >= 1 is
        # a latency chain on at most B x cluster SMs, so the search between levels i and i + 1 runs on a side stream
        # beside the sampling of level i + 1 (submitted after it: the sampler's CTAs are placed first): 0.54 + 0.37 ms
        # alone, 0.56 ms together at 64 scenes (profiles/r01/overlap_probe.txt).  A stage timer then sees only the
        # main stream's wait in "fpK.three_nn".
        n_sa = len(self.sa)  # a global level (last, no sampler) has no entry in sa_chains
        overlap = self.overlap_geometry
        main = torch.cuda.current_stream()
        pending, early_nn = None, {}
        for i in range(len(self.sa_chains)):
            ball_grid = None
            # (levels below the one-call form's grid threshold stay on the linear scan: with the build hidden the grid
            # query of the second level, 5 120 points, still measured 0.30 ms against 0.26 ms)
            if overlap and lib.s4g_ball_query_uses_grid(xyz.shape[2], cfg["num_neighbours"][i], float(cfg["radius"][i])):
                cloud_ready = torch.cuda.Event()
                cloud_ready.record()
            else:
                cloud_ready = None
            with _sec(timer, "sa%d.fps" % i):
                idx = self.fps(xyz, cfg["num_centroids"][i])
            if cloud_ready is not None:
                # the ball query's spatial index only needs the cloud: built beside the sampler (submitted after it)
                if self._geom_stream is None:
                    self._geom_stream = torch.cuda.Stream(device=xyz.device)
                self._geom_stream.wait_event(cloud_ready)
                with torch.cuda.stream(self._geom_stream):
                    ball_grid = lib.s4g_ball_grid_build_f32(ptr(xyz), B, xyz.shape[2], float(cfg["radius"][i]),
                                                            stream_ptr(xyz.device))
                    if not ball_grid:
                        raise RuntimeError("s4g_ball_grid_build_f32 failed: " + lib.s4g_last_error().decode())
                    grid_done = torch.cuda.Event()
                    grid_done.record()
            if pending is not None:
                self._side_three_nn(pending, early_nn, xyz.device)
                pending = None
            try:
                with _sec(timer, "sa%d.gather_xyz" % i):
                    new_xyz = self.gather_xyz(xyz, idx)
                with _sec(timer, "sa%d.ball_query" % i):
                    if ball_grid:
                        main.wait_event(grid_done)
                        k = cfg["num_neighbours"][i]
                        nbr = torch.empty((B, new_xyz.shape[2], k), dtype=torch.int32, device=xyz.device)
                        check(lib.s4g_ball_query_with_grid_f32_i32(ball_grid, ptr(xyz), ptr(new_xyz), new_xyz.shape[2], k,
                                                                   ptr(nbr), None, stream_ptr(xyz.device)),
                              "ball_query_with_grid")
                    else:
                        nbr = self.ball_query(xyz, new_xyz, cfg["radius"][i], cfg["num_neighbours"][i])
            finally:
                if ball_grid:  # host struct + stream-ordered arena: released whatever happened in between
                    lib.s4g_ball_grid_free(ball_grid, stream_ptr(xyz.device))
            feat = self._sa_level(i, feat, xyz, new_xyz, nbr, idx, timer)
            if overlap and i + 1 < n_sa and len(self.fp_chains) == n_sa:
                ready = torch.cuda.Event()
                ready.record()  # after this level's chain: the search starts together with the next level's sampling
                pending = (xyz, new_xyz, ready, n_sa - 1 - i)
            xyz = new_xyz
            lv_xyz.append(xyz)
            lv_feat.append(feat)
            if trace is not None:
                trace["fps"].append(idx)
                trace["ball"].append(nbr)
        if self.global_level:
            i = n_sa - 1
            if pending is not None:  # the search below the last sampled level runs beside the global pool
                self._side_three_nn(pending, early_nn, xyz.device)
                pending = None
            g, nbr, ctr = self._global_group(B, xyz.shape[2])
            with _sec(timer, "sa%d.mlp" % i):
                part = self._global_chain(g).run_gather(feat, xyz, ctr, nbr)  # [B*P, C]: one max per partial group
            with _sec(timer, "sa%d.pool" % i):
                feat = self.rows_segment_max(part, B)
            xyz = ctr[:, :, :1]  # the reference's zero centroid (B,3,1)
            lv_xyz.append(xyz)
            lv_feat.append(feat)
        sparse_xyz, sparse = xyz, feat
        for i, chains in enumerate(self.fp_chains):
            dense_xyz, dense = lv_xyz[-2 - i], lv_feat[-2 - i]
            if i == 0 and self.global_level:
                with _sec(timer, "fp0.broadcast"):
                    x = self.broadcast_concat(sparse, dense, B, dense_xyz.shape[2])
                with _sec(timer, "fp0.mlp"):
                    for ch in chains:
                        x = ch.run_rows(x)
                sparse_xyz, sparse = dense_xyz, x
                continue
            with _sec(timer, "fp%d.three_nn" % i):
                if i in early_nn:
                    (idx3, w), done = early_nn.pop(i)
                    main.wait_event(done)
                    idx3.record_stream(main)
                    w.record_stream(main)
                else:
                    idx3, w = self.three_nn_weights(dense_xyz, sparse_xyz)
            sparse = self._fp_level(i, sparse, dense, dense_xyz, idx3, w, sparse_xyz.shape[2], timer)
            sparse_xyz = dense_xyz
        return lv_xyz[0], sparse, lv_feat

    def _fp_level(self, i, sparse, dense, dense_xyz, idx3, w, Nk, timer):
        """Interpolating propagation level i on the tcgen05 trunk: sparse bf16 [B*Nk, C2], skip bf16 [B*Nq, C1] (or None),
        the dense cloud (B,3,Nq), the 3-NN indices / weights -> bf16 [B*Nq, C']."""
        B, Nq = dense_xyz.shape[0], dense_xyz.shape[2]
        if self.fp_pre[i] is not None:
            with _sec(timer, "fp%d.mlp" % i):
                pre = self.fp_pre[i].run_rows(sparse)  # first conv + shift on the sparse rows, no ReLU
            with _sec(timer, "fp%d.interp_concat" % i):
                x = self.interp_concat(pre, idx3, w, None, B, Nk, Nq, relu=True)
        else:
            with _sec(timer, "fp%d.interp_concat" % i):
                x = self.interp_concat(sparse, idx3, w, dense, B, Nk, Nq)
        with _sec(timer, "fp%d.mlp" % i):
            for ch in self.fp_chains[i]:
                x = ch.run_rows(x)
        return x

    def _head_stage(self, xyz, sparse, timer=None, host_out=None):
        """PN2_CLS's four per-point heads on the trunk's features -> {score, frame_R, frame_t, movable_logits (after the
        sigmoid)}, each (B, k, N) fp32."""
        B, n = xyz.shape[0], xyz.shape[2]
        if self.mlp_backend != "tcgen05":
            outs = [self._head_reference(sparse, k) for k in range(4)]
            return {"score": outs[0], "frame_R": outs[1], "frame_t": outs[2], "movable_logits": torch.sigmoid(outs[3])}
        names = ("score", "frame_R", "frame_t", "movable_logits")
        with _sec(timer, "heads.mlp"):
            outs = [None] * 4
            # widest head first: with host_out the copy that cannot hide behind a later head is then the smallest
            order = sorted(range(4), key=lambda k: -self.head_chains[k].out_c)
            for k in order:
                name, ch = names[k], self.head_chains[k]
                if host_out is None:
                    outs[k] = ch.run_rows(sparse, n_points=n)
                    continue
                # stream this head's result to the caller's pinned host tensor while the next head computes; the LAST
                # head has nothing behind it, so it runs as two half-batches: only the second half's copy is exposed
                if self._copy_stream is None:
                    self._copy_stream = torch.cuda.Stream(device=sparse.device)
                o = torch.empty((B, ch.out_c, n), dtype=torch.float32, device=sparse.device)
                cuts = [0, B // 2, B] if (k == order[-1] and B >= 2) else [0, B]
                for b0, b1 in zip(cuts[:-1], cuts[1:]):
                    ch.run_rows(sparse[b0 * n:b1 * n], n_points=n, out=o[b0:b1])
                    ev = torch.cuda.Event()
                    ev.record()
                    self._copy_stream.wait_event(ev)
                    with torch.cuda.stream(self._copy_stream):
                        host_out[name][b0:b1].copy_(o[b0:b1], non_blocking=True)
                o.record_stream(self._copy_stream)
                outs[k] = o
        if host_out is not None:
            torch.cuda.current_stream().wait_stream(self._copy_stream)  # the caller's synchronize covers the copies
        return dict(zip(names, outs))

    def _head_reference(self, sparse, k):
        """Head k on the torch / tf32 backends: (B, N, C) fp32 features -> (B, k_out, N) logits, no sigmoid."""
        layers, w, b = self.heads[k]
        return self._logits(self._mlp(sparse, layers), w, b).transpose(1, 2).contiguous()

    def _trunk_reference(self, points, trace):
        """The trunk on the torch / tf32 backends -> (cloud (B,3,N), per-point features (B, N, C) fp32, the set-abstraction
        levels' features)."""
        cfg = self.cfg
        xyz = points.float().contiguous()
        feat = None
        lv_xyz, lv_feat = [xyz], [None]
        for i, layers in enumerate(self.sa):
            if cfg["num_centroids"][i] == 0:  # global level: the same partial groups as the fused path
                g, nbr, ctr = self._global_group(xyz.shape[0], xyz.shape[2])
                feat = self._sa_torch(xyz, feat, ctr, nbr, layers).amax(dim=1, keepdim=True)  # (B,1,C)
                xyz = ctr[:, :, :1]
                lv_xyz.append(xyz)
                lv_feat.append(feat)
                continue
            idx = self.fps(xyz, cfg["num_centroids"][i])
            new_xyz = torch.gather(xyz, 2, idx.long().unsqueeze(1).expand(-1, 3, -1)).contiguous()
            nbr = self.ball_query(xyz, new_xyz, cfg["radius"][i], cfg["num_neighbours"][i])
            feat = self._sa_reference(i, xyz, feat, new_xyz, nbr, idx, layers)
            xyz = new_xyz
            lv_xyz.append(xyz)
            lv_feat.append(feat)
            if trace is not None:
                trace["fps"].append(idx)
                trace["ball"].append(nbr)
        sparse_xyz, sparse = xyz, feat
        for i, layers in enumerate(self.fp):
            dense_xyz, dense = lv_xyz[-2 - i], lv_feat[-2 - i]
            if i == 0 and self.global_level:  # broadcast propagation, [global | skip] (modules.py:131-134)
                x = sparse.expand(-1, dense_xyz.shape[2], -1)
                sparse = self._mlp(x if dense is None else torch.cat([x, dense], dim=-1), layers)
            else:
                sparse = self._fp_reference(i, dense_xyz, sparse_xyz, dense, sparse, layers)
            sparse_xyz = dense_xyz
        return lv_xyz[0], sparse, lv_feat

    def _fp_reference(self, i, dense_xyz, sparse_xyz, dense, sparse, layers):
        """Interpolating propagation level i on the torch / tf32 backends: (B, Nk, C2), skip (B, Nq, C1) or None ->
        (B, Nq, C')."""
        return self._fp_torch(dense_xyz, sparse_xyz, dense, sparse, layers)

    def _run(self, points, return_trace, timer, head_stage):
        """The trunk on this engine's backend, then ``head_stage(cloud, per-point features)``."""
        if not points.is_cuda:
            raise RuntimeError("scene_points must be a CUDA tensor (there is no CPU path)")
        trace = {"fps": [], "ball": []} if return_trace else None
        with torch.cuda.device(points.device):
            if self.mlp_backend == "tcgen05":
                xyz, sparse, lv_feat = self._trunk_tcgen05(points, trace, timer)
            else:
                xyz, sparse, lv_feat = self._trunk_reference(points, trace)
            preds = head_stage(xyz, sparse)
            if trace is None:
                return preds
            if self.mlp_backend == "tcgen05":
                B, n = xyz.shape[0], xyz.shape[2]
                trace["point_feature"] = sparse.float().reshape(B, n, -1)
                trace["sa_feature"] = [f.float().reshape(B, -1, f.shape[1]) for f in lv_feat[1:]]
            else:
                trace["point_feature"] = sparse
                trace["sa_feature"] = lv_feat[1:]
        return preds, trace

    # ---------------------------------------------------------------- forward
    @torch.no_grad()
    def forward(self, points, return_trace=False, timer=None, host_out=None):
        """points (B,3,N) fp32 CUDA -> the four prediction tensors.  ``host_out``: optional dict of PINNED host tensors
        (same keys / shapes as the result); each head's output is then copied to it on a side stream as soon as that
        head finishes, overlapping the device -> host transfer with the remaining heads (the copies are ordered before
        the current stream's next operation, so one synchronize() after the call makes them visible)."""
        return self._run(points, return_trace, timer, lambda xyz, sparse: self._head_stage(xyz, sparse, timer, host_out))


def check_local_frames(points, frames):
    """The given candidates of PN2_LOCAL's evaluation head: (B, 12, F, S) fp32 contiguous on the points' device with
    1 <= F <= N and S >= 1, else ValueError.  The fused path writes their translations back in place, as the reference
    does, so it takes no copy."""
    B, _, N = points.shape
    if not (isinstance(frames, torch.Tensor) and frames.dim() == 4 and frames.shape[0] == B and frames.shape[1] == 12):
        raise ValueError("local_search_frame must be a (B, 12, n_frames, n_search) tensor with B = %d" % B)
    if frames.device != points.device or frames.dtype != torch.float32 or not frames.is_contiguous():
        raise ValueError("local_search_frame must be a contiguous float32 tensor on %s (got %s %s%s)"
                         % (points.device, frames.dtype, frames.device, "" if frames.is_contiguous() else ", strided"))
    F, S = frames.shape[2], frames.shape[3]
    if not (1 <= F <= N and S >= 1):
        raise ValueError("local_search_frame needs 1 <= n_frames <= %d points and n_search >= 1 (got %d, %d)" % (N, F, S))


class FusedPointNet2Local(FusedPointNet2):
    """PN2_LOCAL (models/PointNet2_local.py): the trunk of FusedPointNet2 unchanged, its own head stage.  Three per-point
    heads (frame_R 9, frame_t 3, movable 2 logits, no sigmoid) and the grasp-evaluation head: one logits chain over the
    rows [point feature | candidate (R 9, t 3) x 4] that ``local_eval_rows`` writes, one row per candidate."""

    _HEAD_SIGMOID = (False, False, False, False)

    @staticmethod
    def _head_modules(model):
        return ((model.mlp_R, model.R_logit), (model.mlp_t, model.t_logit), (model.mlp_movable, model.movable_logit),
                (model.mlp_grasp_eval, model.grasp_eval_logit))

    @staticmethod
    def local_eval_rows(feat, xyz, frames=None, R=None, t=None):
        """feat bf16 [B*N, C]; given: frames (B, 12, F, S) fp32, whose translations become relative to xyz (B,3,N) IN
        PLACE; self: R (B, 9, N), t (B, 3, N) fp32 -> bf16 [B*F*S, C + 48] rows [feature | (R, t) x 4]."""
        B, _, N = xyz.shape
        C = feat.shape[1]
        F, S = (frames.shape[2], frames.shape[3]) if frames is not None else (N, 1)
        out = torch.empty((B * F * S, C + 48), dtype=torch.bfloat16, device=feat.device)
        check(lib.s4g_local_eval_rows_bf16(ptr(feat), B, N, C, ptr(frames) if frames is not None else None, ptr(xyz),
                                           F, S, ptr(R) if R is not None else None, ptr(t) if t is not None else None,
                                           ptr(out), stream_ptr(feat.device)), "local_eval_rows")
        return out

    def _local_head_stage(self, xyz, sparse, frames, timer):
        """-> raw {local_search_logits (B, k, F, S), frame_R (B, 9, N), frame_t (B, 3, N) offset, movable_logits}."""
        B, n = xyz.shape[0], xyz.shape[2]
        F, S = (frames.shape[2], frames.shape[3]) if frames is not None else (n, 1)
        if self.mlp_backend != "tcgen05":
            R, t, mov = [self._head_reference(sparse, k) for k in range(3)]
            if frames is None:  # the prediction itself, one candidate per point
                cand = torch.cat([R, t], dim=1).transpose(1, 2).unsqueeze(2)  # (B, N, 1, 12)
                per_point = sparse.unsqueeze(2)
            else:  # the reference's in-place update of the caller's frames (PointNet2_local.py:135)
                frames[:, 9:] = frames[:, 9:] - xyz[:, :, :F].unsqueeze(-1).expand(-1, -1, -1, S)
                cand = frames.permute(0, 2, 3, 1)  # (B, F, S, 12)
                per_point = sparse[:, :F].unsqueeze(2).expand(-1, -1, S, -1)
            x = torch.cat([per_point, cand.repeat(1, 1, 1, 4)], dim=-1)
            layers, w, b = self.heads[3]
            logits = self._logits(self._mlp(x, layers), w, b).permute(0, 3, 1, 2).contiguous()
        else:
            R_ch, t_ch, mov_ch, eval_ch = self.head_chains
            with _sec(timer, "heads.R"):
                R = R_ch.run_rows(sparse, n_points=n)
            with _sec(timer, "heads.t"):
                t = t_ch.run_rows(sparse, n_points=n)
            with _sec(timer, "heads.movable"):
                mov = mov_ch.run_rows(sparse, n_points=n)
            with _sec(timer, "heads.eval_rows"):
                rows = self.local_eval_rows(sparse, xyz, frames, R, t)
            with _sec(timer, "heads.eval_mlp"):
                logits = eval_ch.run_rows(rows, n_points=F * S).view(B, -1, F, S)
        return {"local_search_logits": logits, "frame_R": R, "frame_t": t, "movable_logits": mov}

    @torch.no_grad()
    def forward(self, points, frames=None, return_trace=False, timer=None):
        """points (B,3,N) fp32 CUDA; ``frames``: None (each point's own (R, t) prediction is its one candidate) or the
        given candidates (B, 12, F, S) fp32 (check_local_frames), whose translation rows are made relative to their
        point IN PLACE, as the reference does.  -> the raw head outputs; the model adds the points to frame_t."""
        if frames is not None:
            check_local_frames(points, frames)
        return self._run(points, return_trace, timer,
                         lambda xyz, sparse: self._local_head_stage(xyz, sparse, frames, timer))


class FusedEdgePointNet2Down(FusedPointNet2):
    """EDGEPN2D (models/EdgePointNet2Down.py): the PN2 sibling whose sampled levels with input features are edge levels
    (EdgeSAModule).  Their first layer sees EdgeQueryGrouper's rows [x_j - x_c | f_j | f_j - f_c] (3 + 2C channels); with
    the folded weight split by those column groups, W' = [W_x | W_a | W_b], it is
        [W_x | W_a + W_b] [x_j - x_c ; f_j] + b' + u_c,   u_c = -W_b f_c,
    so on the tcgen05 trunk an edge level is the plain gathered chain over 3 + C channels with the weights
    [W_x | W_a + W_b], plus the centroid term u: the centroid rows (``gather_rows`` at the level's sampled indices) through
    a one-layer row chain (-W_b, zero shift, no ReLU), added by the edge chain's layer-0 epilogue before the ReLU.  The
    (B, 3 + 2C, M, K) edge tensor never exists.  The torch / tf32 backends build the edge rows literally and use the
    unsplit weights: an independent check of the split.  Level 0 (no input features) and the global level are PN2's."""

    def __init__(self, model, *args, **kwargs):
        from .network_models.models.pointnet2_utils.modules import EdgeSAModule
        c = 0
        self.edge_levels = []  # per set-abstraction level: an edge level (sampled, with input features)
        for m in model.sa_modules:
            self.edge_levels.append(isinstance(m, EdgeSAModule) and m.num_centroids > 0 and c > 0)
            c = m.out_channels
        self._term_chains = {}  # edge level -> the row chain of its centroid term u
        super().__init__(model, *args, **kwargs)

    @staticmethod
    def split_edge_layer(w, c):
        """Folded first-layer weight of an edge level, fp32 [cout, 3 + 2c] with columns [xyz | neighbour | difference]
        -> ([W_x | W_a + W_b] [cout, 3 + c], -W_b [cout, c]), in the input's precision (split before any bf16 cast)."""
        assert w.dim() == 2 and w.shape[1] == 3 + 2 * c, "edge layer expects 3 + 2 x %d input channels" % c
        wx, wa, wb = w[:, :3], w[:, 3:3 + c], w[:, 3 + c:]
        return torch.cat([wx, wa + wb], dim=1).contiguous(), (-wb).contiguous()

    def _sa_chain(self, i, layers, feat_c):
        if not self.edge_levels[i]:
            return super()._sa_chain(i, layers, feat_c)
        (w0, b0), rest = layers[0], layers[1:]
        w_plain, w_u = self.split_edge_layer(w0, feat_c)
        self._term_chains[i] = self._make_chain([(w_u, torch.zeros_like(b0), False)], IN_ROWS, 0, OUT_ROWS)
        return self._make_chain([(w_plain, b0, True)] + [(w, b, True) for w, b in rest], IN_GATHER_EDGE, feat_c,
                                OUT_MAXPOOL, group=self.cfg["num_neighbours"][i])

    @staticmethod
    def gather_rows(rows, idx):
        """bf16 [B*N, C] rows, int32 indices (B, M) -> bf16 [B*M, C], row b*M + m = rows[b*N + idx[b, m]]."""
        B, M = idx.shape
        C = rows.shape[1]
        out = torch.empty((B * M, C), dtype=torch.bfloat16, device=rows.device)
        check(lib.s4g_gather_rows_bf16(ptr(rows), ptr(idx), B, rows.shape[0] // B, M, C, ptr(out),
                                       stream_ptr(rows.device)), "gather_rows")
        return out

    def _sa_level(self, i, feat, xyz, new_xyz, nbr, idx, timer):
        if not self.edge_levels[i]:
            return super()._sa_level(i, feat, xyz, new_xyz, nbr, idx, timer)
        with _sec(timer, "sa%d.term" % i):
            term = self._term_chains[i].run_rows(self.gather_rows(feat, idx))  # u = -W_b f_c, bf16 [B*M, cout0]
        with _sec(timer, "sa%d.mlp" % i):
            return self.sa_chains[i].run_gather(feat, xyz, new_xyz, nbr, term)

    def _sa_reference(self, i, xyz, feat, new_xyz, nbr, idx, layers):
        if not self.edge_levels[i]:
            return super()._sa_reference(i, xyz, feat, new_xyz, nbr, idx, layers)
        ctr_feat = torch.gather(feat, 1, idx.long().unsqueeze(-1).expand(-1, -1, feat.shape[-1]))
        return self._sa_torch(xyz, feat, new_xyz, nbr, layers, ctr_feat=ctr_feat)


class FusedEdgePointNet2DownUp(FusedEdgePointNet2Down):
    """EDGEPN2DU (models/EdgePointNet2DownUp.py): EDGEPN2D's encoder (edge set-abstraction levels, global level), a
    decoder whose interpolating levels are edge levels (EdgeFPModule), and two heads (scene_score_logits, frame_R; no
    sigmoid).  An edge propagation level's first layer sees EdgeFeatureInterpolator's rows [interp_q | n_k - interp_q | d_q]
    for each dense point q and each of its 3 nearest sparse points k (2 C2 + C1 channels), and the level ends with the mean
    over k.  With the folded weight split by those column groups, W' = [W_i | W_n | W_d], and interp_q = sum_j w_qj S_j,
        y0[q,k] = sum_j w_qj U[idx_qj] + V[idx_qk] + T_q + b',   U = (W_i - W_n) S,  V = W_n S,  T = W_d d,
    which needs no assumption on the weights' sum.  So on the tcgen05 trunk an edge propagation level is: one row chain
    over the sparse rows with the stacked weight [W_i - W_n ; W_n] (zero shift, no ReLU) -> bf16 [U | V]; T by a one-layer
    row chain (W_d, zero shift, no ReLU) over the skip rows, or, at the finest level, whose skip is the cloud itself, in
    fp32 inside the row kernel; ``edge_interp_rows`` -> relu(y0) bf16 [B*Nq*3, cout0]; the row chains of the later layers
    over those rows; ``rows_group_mean`` -> [B*Nq, C'].  The (B, 2 C2 + C1, Nq, 3) edge tensor never exists.  The torch /
    tf32 backends build the edge rows literally with the unsplit weights and take the mean: an independent check of the
    split.  The broadcast level (num_fp_neighbours = 0) is the sibling's."""

    _HEAD_SIGMOID = (False, False)

    def __init__(self, model, *args, **kwargs):
        from .network_models.models.pointnet2_utils.modules import EdgeFPModule
        # per propagation level: an edge level (EdgeFPModule that interpolates)
        self.edge_fp = [isinstance(m, EdgeFPModule) and m.interpolator is not None for m in model.fp_modules]
        self._edge_fp = {}  # edge propagation level -> ([U | V] chain, T chain or None, shift b', W_d of the cloud or None)
        super().__init__(model, *args, **kwargs)

    @staticmethod
    def _head_modules(model):
        return ((model.mlp_seg, model.seg_logit), (model.mlp_frame, model.frame_logit))

    @staticmethod
    def split_edge_fp_layer(w, c2):
        """Folded first-layer weight of an edge propagation level, [cout, 2 c2 + c1] with columns [interpolated |
        neighbour - interpolated | skip] -> ([W_i - W_n ; W_n] [2 cout, c2], W_d [cout, c1]), in the input's precision
        (split before any bf16 cast)."""
        assert w.dim() == 2 and w.shape[1] > 2 * c2, "edge propagation layer expects 2 x %d + skip input channels" % c2
        wi, wn, wd = w[:, :c2], w[:, c2:2 * c2], w[:, 2 * c2:]
        return torch.cat([wi - wn, wn], dim=0).contiguous(), wd.contiguous()

    def _fp_chain(self, i, layers, skip_c):
        if not self.edge_fp[i]:
            return super()._fp_chain(i, layers, skip_c)
        (w0, b0), rest = layers[0], layers[1:]
        c1 = skip_c or 3  # no skip feature below the finest level: there it is the cloud (EdgePointNet2DownUp.forward)
        w_uv, w_d = self.split_edge_fp_layer(w0, (w0.shape[1] - c1) // 2)
        cout = w0.shape[0]
        uv = self._make_chain([(w_uv, b0.new_zeros(2 * cout), False)], IN_ROWS, 0, OUT_ROWS)
        if skip_c:
            term, w_xyz = self._make_chain([(w_d, b0.new_zeros(cout), False)], IN_ROWS, 0, OUT_ROWS), None
        else:
            term, w_xyz = None, w_d.to(self.device)
        self._edge_fp[i] = (uv, term, b0.to(self.device).contiguous(), w_xyz)
        return None, self._row_chains(rest) if rest else []

    @staticmethod
    def edge_interp_rows(uv, idx, w, t_rows, xyz, w_xyz, shift, B, Nk, Nq):
        """uv bf16 [B*Nk, 2C] rows [U | V]; 3-NN int32 idx / fp32 w (B,Nq,3); skip: t_rows bf16 [B*Nq, C] or the cloud
        xyz (B,3,Nq) fp32 with w_xyz fp32 [C, 3]; shift fp32 [C] -> bf16 [B*Nq*3, C], relu of the first layer per (q, k)."""
        C = shift.shape[0]
        out = torch.empty((B * Nq * 3, C), dtype=torch.bfloat16, device=uv.device)
        check(lib.s4g_edge_interp_rows_bf16(ptr(uv), ptr(idx), ptr(w), ptr(t_rows) if t_rows is not None else None,
                                            ptr(xyz) if xyz is not None else None,
                                            ptr(w_xyz) if w_xyz is not None else None, ptr(shift), B, Nk, Nq, C, ptr(out),
                                            stream_ptr(uv.device)), "edge_interp_rows")
        return out

    @staticmethod
    def rows_group_mean(rows):
        """bf16 [3R, C] -> [R, C]: the mean of each 3 consecutive rows, ((r0 + r1) + r2) / 3 in fp32, rounded once."""
        R, C = rows.shape[0] // 3, rows.shape[1]
        out = torch.empty((R, C), dtype=torch.bfloat16, device=rows.device)
        check(lib.s4g_rows_group_mean_bf16(ptr(rows), R, C, ptr(out), stream_ptr(rows.device)), "rows_group_mean")
        return out

    def _fp_level(self, i, sparse, dense, dense_xyz, idx3, w, Nk, timer):
        if not self.edge_fp[i]:
            return super()._fp_level(i, sparse, dense, dense_xyz, idx3, w, Nk, timer)
        uv_chain, term_chain, shift, w_xyz = self._edge_fp[i]
        B, Nq = dense_xyz.shape[0], dense_xyz.shape[2]
        with _sec(timer, "fp%d.uv" % i):
            uv = uv_chain.run_rows(sparse)
        t_rows = None
        if term_chain is not None:
            with _sec(timer, "fp%d.term" % i):
                t_rows = term_chain.run_rows(dense)
        with _sec(timer, "fp%d.edge_rows" % i):
            x = self.edge_interp_rows(uv, idx3, w, t_rows, dense_xyz if t_rows is None else None, w_xyz, shift, B, Nk, Nq)
        with _sec(timer, "fp%d.mlp" % i):
            for ch in self.fp_chains[i]:
                x = ch.run_rows(x)
        with _sec(timer, "fp%d.mean" % i):
            return self.rows_group_mean(x)

    def _fp_reference(self, i, dense_xyz, sparse_xyz, dense, sparse, layers):
        if not self.edge_fp[i]:
            return super()._fp_reference(i, dense_xyz, sparse_xyz, dense, sparse, layers)
        g, interp = self._interp_torch(dense_xyz, sparse_xyz, sparse)  # (B, Nq, 3, C2), (B, Nq, C2)
        skip = dense if dense is not None else dense_xyz.transpose(1, 2)
        centre = interp.unsqueeze(2).expand_as(g)
        x = torch.cat([centre, g - centre, skip.unsqueeze(2).expand(-1, -1, g.shape[2], -1)], dim=-1)
        return self._mlp(x, layers).mean(dim=2)

    def _downup_head_stage(self, xyz, sparse, timer):
        """-> {scene_score_logits (B, score_classes, N), frame_R (B, 9, N)} fp32 logits."""
        n = xyz.shape[2]
        if self.mlp_backend != "tcgen05":
            outs = [self._head_reference(sparse, k) for k in range(2)]
        else:
            with _sec(timer, "heads.mlp"):
                outs = [ch.run_rows(sparse, n_points=n) for ch in self.head_chains]
        return {"scene_score_logits": outs[0], "frame_R": outs[1]}

    @torch.no_grad()
    def forward(self, points, return_trace=False, timer=None):
        """points (B,3,N) fp32 CUDA -> {scene_score_logits, frame_R}, as EdgePointNet2DownUp.forward."""
        return self._run(points, return_trace, timer, lambda xyz, sparse: self._downup_head_stage(xyz, sparse, timer))
