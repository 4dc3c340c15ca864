"""Host handle of one fused tcgen05 MLP chain (csrc/mlp_chain.cu) — plans the chain through the C ABI,
packs the BN-folded weights to the kernel's bf16 chunk stream and keeps the device buffers alive."""
import ctypes

import numpy as np
import torch

from ._lib import check, lib, ptr, stream_ptr

IN_ROWS, IN_GATHER, IN_XYZ_MLP, IN_GATHER_EDGE = 0, 1, 5, 6
OUT_ROWS, OUT_MAXPOOL, OUT_LOGITS = 2, 3, 4


def _int_array(values):
    return (ctypes.c_int * len(values))(*[int(v) for v in values])


class MlpChain:
    """layers: list of (W fp32 [cout, cin] BN-folded, shift fp32 [cout], relu: bool).
    ``xyz_layer_on_cuda_cores=True`` plans a gathered chain without features (in_mode IN_GATHER, feat_c 0, first
    layer 3 -> <= 128 channels, more layers behind it) as IN_XYZ_MLP: the kernel evaluates that first layer in fp32 on
    the CUDA cores while it stages the tile.  Off by default — measured on the first set-abstraction level
    (64 x 5120 x 64 rows, 3 -> 128 -> 128 -> 256): 5.57 ms against 4.27 ms with the K = 16 tensor-core layer; the two
    loader warps cannot issue the 49 k FMAs of a tile as fast as the rest of the tile runs.
    ``tma_in=1`` (row chains, cin[0] % 64 == 0): input blocks arrive by TMA tensor copies (s4g_chain_create_tuned_in).
    ``in_mode=IN_GATHER_EDGE``: an edge level's gathered max-pool chain; ``run_gather`` then takes the per-centroid term
    of layer 0 (s4g_chain_run_gather_term)."""

    def __init__(self, layers, device, in_mode=IN_ROWS, feat_c=0, out_mode=OUT_ROWS, group=1, sigmoid=False,
                 xyz_layer_on_cuda_cores=False, slots=0, pairs=-1, coop=-1, subs=1, tma_in=0):
        self.device = torch.device(device)
        self.all_cin = [int(w.shape[1]) for w, _, _ in layers]
        self.all_cout = [int(w.shape[0]) for w, _, _ in layers]
        self._xyz_table = None
        if (xyz_layer_on_cuda_cores and in_mode == IN_GATHER and feat_c == 0 and len(layers) > 1
                and layers[0][0].shape[0] % 16 == 0 and layers[0][0].shape[0] <= 128):
            w0, b0, relu0 = layers[0]
            table = torch.cat([w0.detach().float().reshape(-1, 3), b0.detach().float().reshape(-1, 1)], dim=1)
            self._xyz_table = np.ascontiguousarray(table.cpu().numpy(), dtype=np.float32)
            self._xyz_relu = bool(relu0)
            layers = layers[1:]
            in_mode = IN_XYZ_MLP
        self.n_layers = len(layers)
        self.cin = [int(w.shape[1]) for w, _, _ in layers]
        self.cout = [int(w.shape[0]) for w, _, _ in layers]
        self.in_mode, self.out_mode, self.group = in_mode, out_mode, group
        self.out_c = self.cout[-1]
        relu = [1 if r else 0 for _, _, r in layers]
        self.tma_in = int(tma_in)
        self._h = lib.s4g_chain_create_tuned_in(self.n_layers, _int_array(self.cin), _int_array(self.cout),
                                                _int_array(relu), in_mode, feat_c, out_mode, self.out_c, group,
                                                1 if sigmoid else 0, int(slots), int(pairs), int(coop), int(subs),
                                                self.tma_in)
        if not self._h:
            raise RuntimeError("s4g_chain_create failed: " + lib.s4g_last_error().decode())
        nbytes = lib.s4g_chain_weight_bytes(self._h)
        packed = np.zeros(nbytes, dtype=np.uint8)
        for l, (w, _, _) in enumerate(layers):
            w32 = np.ascontiguousarray(w.detach().float().cpu().numpy())
            check(lib.s4g_chain_pack_weights(self._h, l, w32.ctypes.data_as(ctypes.c_void_p), w32.shape[0],
                                             w32.shape[1], packed.ctypes.data_as(ctypes.c_void_p)), "chain_pack_weights")
        self.weights = torch.from_numpy(packed).to(self.device)
        self.bias = []
        for l, (_, b, _) in enumerate(layers):
            pad = lib.s4g_chain_cout_pad(self._h, l)
            t = torch.zeros(pad, dtype=torch.float32, device=self.device)
            t[: b.numel()] = b.detach().float().to(self.device)
            self.bias.append(t)
        self._bias_ptrs = (ctypes.c_void_p * self.n_layers)(*[t.data_ptr() for t in self.bias])
        check(lib.s4g_chain_set_params(self._h, ptr(self.weights), ctypes.cast(self._bias_ptrs, ctypes.c_void_p)),
              "chain_set_params")
        if self._xyz_table is not None:
            check(lib.s4g_chain_set_xyz_layer(self._h, self._xyz_table.ctypes.data_as(ctypes.c_void_p),
                                              1 if self._xyz_relu else 0),
                  "chain_set_xyz_layer")

    def info(self):
        vals = [ctypes.c_int() for _ in range(7)]
        check(lib.s4g_chain_info(self._h, *[ctypes.byref(v) for v in vals]), "chain_info")
        keys = ("n_jobs", "slots", "stages", "load_depth", "smem_bytes", "sim_cycles", "mma_cycles")
        return {k: v.value for k, v in zip(keys, vals)}

    def describe(self):
        buf = ctypes.create_string_buffer(1 << 16)
        lib.s4g_chain_describe(self._h, buf, len(buf))
        return buf.value.decode()

    def set_profile(self, counters):
        """counters: int64 CUDA tensor [>=148, 16] (or None) — see s4g_chain_set_profile."""
        self._prof = counters
        check(lib.s4g_chain_set_profile(self._h, ptr(counters) if counters is not None else None), "chain_set_profile")

    def flops(self, rows):
        return 2.0 * rows * sum(ci * co for ci, co in zip(self.all_cin, self.all_cout))

    def run_rows(self, x, n_points=0, out=None):
        """x: bf16 [P, stride] channel-last (stride >= cin).  Returns bf16 [P, out_c] or fp32 (B, out_c, n_points);
        ``out``: optional preallocated contiguous result tensor of that shape and dtype (e.g. a slice of a batch)."""
        assert x.is_cuda and x.dtype == torch.bfloat16 and x.dim() == 2 and x.stride(1) == 1
        P = x.shape[0]
        shape, dtype = (((P // n_points, self.out_c, n_points), torch.float32) if self.out_mode == OUT_LOGITS
                        else ((P, self.out_c), torch.bfloat16))
        if out is None:
            out = torch.empty(shape, dtype=dtype, device=x.device)
        else:
            assert tuple(out.shape) == shape and out.dtype == dtype and out.is_contiguous() and out.device == x.device
        check(lib.s4g_chain_run_rows(self._h, ptr(x), x.stride(0), P, ptr(out), n_points, stream_ptr(x.device)),
              "chain_run_rows")
        return out

    def run_gather(self, feat, xyz, ctr, nbr, term=None):
        """feat: bf16 [B*N, C] or None; xyz (B,3,N) fp32; ctr (B,3,M) fp32; nbr (B,M,K) int32; term: an edge chain's
        bf16 [B*M, cout[0]] per-centroid term of layer 0 (required for IN_GATHER_EDGE, refused otherwise)."""
        B, _, N = xyz.shape
        M, K = nbr.shape[1], nbr.shape[2]
        rows = B * M if self.out_mode == OUT_MAXPOOL else B * M * K
        out = torch.empty((rows, self.out_c), dtype=torch.bfloat16, device=xyz.device)
        f = ptr(feat) if feat is not None else None
        if self.in_mode == IN_GATHER_EDGE:
            assert term is not None and term.dtype == torch.bfloat16 and term.is_contiguous()
            assert tuple(term.shape) == (B * M, self.cout[0]) and term.device == xyz.device
            check(lib.s4g_chain_run_gather_term(self._h, f, ptr(xyz), ptr(ctr), ptr(nbr), ptr(term), B, N, M, K, ptr(out),
                                                stream_ptr(xyz.device)), "chain_run_gather_term")
        else:
            assert term is None, "only an IN_GATHER_EDGE chain takes a group term"
            check(lib.s4g_chain_run_gather(self._h, f, ptr(xyz), ptr(ctr), ptr(nbr), B, N, M, K, ptr(out),
                                           stream_ptr(xyz.device)), "chain_run_gather")
        return out

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib.s4g_chain_destroy(h)
