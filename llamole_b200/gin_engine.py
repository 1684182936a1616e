"""Shared host-side engine for the two GIN modules (packs weights, binds graph batches, calls the C ABI)."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import torch
import torch.nn as nn

from . import _cabi


class _Holder(nn.Module):
    """Parameter container (no forward): keeps the reference's module tree so state-dict keys match."""


def mlp4(h_in: int, hidden: int, out: int, drop: float) -> nn.Sequential:
    # Linear, LayerNorm, GELU, Dropout, Linear -> parameter keys .0 .1 .4 (graph_encoder/model.py:111,163)
    return nn.Sequential(nn.Linear(h_in, hidden), nn.LayerNorm(hidden), nn.GELU(), nn.Dropout(drop), nn.Linear(hidden, out))


def gin_trunk_skeleton(num_layer: int, H: int, drop: float, affine_norms: bool) -> nn.Module:
    """Module tree of GNNEncoder (graph_encoder/model.py:82-113) / the trunk of GNNRetrosynthsizer
    (graph_predictor/model.py:231-272)."""
    if num_layer < 2:
        raise ValueError("Number of GNN layers must be greater than 1.")
    t = _Holder()
    t.num_layer = num_layer
    t.atom_encoder = nn.Embedding(118, H)
    t.virtualnode_embedding = nn.Embedding(1, H)
    nn.init.constant_(t.virtualnode_embedding.weight.data, 0)
    convs, norms, vns = [], [], []
    for layer in range(num_layer):
        conv = _Holder()
        conv.mlp = mlp4(H, 4 * H, H, drop)
        conv.eps = nn.Parameter(torch.zeros(1))
        conv.bond_encoder = nn.Embedding(5, H)
        convs.append(conv)
        norms.append(nn.LayerNorm(H, elementwise_affine=affine_norms))
        if layer < num_layer - 1:
            vns.append(mlp4(H, 4 * H, H, drop))
    t.convs = nn.ModuleList(convs)
    t.norms = nn.ModuleList(norms)
    t.mlp_virtualnode_list = nn.ModuleList(vns)
    return t


class GinEngine:
    """One per (module, device).  `trunk_sd` / `head` are fp32 CUDA tensors in the reference key layout."""

    def __init__(self, device: torch.device, H: int, L: int, predictor: bool, out_dim: int, text_dim: int,
                 trunk_sd: Dict[str, torch.Tensor], head: Dict[str, torch.Tensor]):
        if device.type != "cuda":
            raise _cabi.LlamoleB200Error("GIN parameters are on %s; move the module to a B200: there is no CPU path" % device)
        self.device, self.H, self.L, self.predictor, self.out_dim, self.text_dim = device, H, L, predictor, out_dim, text_dim
        self.lib = _cabi.lib()
        self.cfg = _cabi.GinConfig(H, L, int(predictor), int(out_dim), int(text_dim))
        with torch.cuda.device(device):
            _cabi.check(self.lib.llb_arch_check(device.index if device.index is not None else torch.cuda.current_device()),
                        "llb_arch_check")
            nbytes = C.c_size_t()
            _cabi.check(self.lib.llb_gin_packed_bytes(C.byref(self.cfg), C.byref(nbytes)), "llb_gin_packed_bytes")
            self.blob = torch.empty(nbytes.value, dtype=torch.uint8, device=device)
            keep = []

            def arr(fmt, n):
                ts = [trunk_sd[fmt.format(i)] for i in range(n)]
                a = _cabi.ptr_array(ts)
                keep.append(a)
                return C.cast(a, C.POINTER(C.c_void_p))

            null_arr = C.cast(None, C.POINTER(C.c_void_p))
            p = lambda k: _cabi.ptr(trunk_sd[k])  # noqa: E731
            w = _cabi.GinWeights(
                p("atom_encoder.weight"), p("virtualnode_embedding.weight"),
                arr("convs.{}.eps", L), arr("convs.{}.mlp.0.weight", L), arr("convs.{}.mlp.0.bias", L),
                arr("convs.{}.mlp.1.weight", L), arr("convs.{}.mlp.1.bias", L), arr("convs.{}.mlp.4.weight", L),
                arr("convs.{}.mlp.4.bias", L), arr("convs.{}.bond_encoder.weight", L),
                null_arr if predictor else arr("norms.{}.weight", L), null_arr if predictor else arr("norms.{}.bias", L),
                arr("mlp_virtualnode_list.{}.0.weight", L - 1), arr("mlp_virtualnode_list.{}.0.bias", L - 1),
                arr("mlp_virtualnode_list.{}.1.weight", L - 1), arr("mlp_virtualnode_list.{}.1.bias", L - 1),
                arr("mlp_virtualnode_list.{}.4.weight", L - 1), arr("mlp_virtualnode_list.{}.4.bias", L - 1),
                arr("adapters.{}.1.weight", L) if predictor else null_arr, arr("adapters.{}.1.bias", L) if predictor else null_arr,
                p("text_dropping.weight") if predictor else C.c_void_p(None),
                _cabi.ptr(head["w0"]), _cabi.ptr(head["b0"]), _cabi.ptr(head["lnw"]), _cabi.ptr(head["lnb"]),
                _cabi.ptr(head["w4"]), _cabi.ptr(head["b4"]),
            )
            _cabi.check(self.lib.llb_gin_pack_weights(C.byref(self.cfg), C.byref(w), _cabi.ptr(self.blob), self.blob.numel(),
                                                      _cabi.stream_ptr()), "llb_gin_pack_weights")
            torch.cuda.current_stream().synchronize()
            h = C.c_void_p()
            _cabi.check(self.lib.llb_gin_create(C.byref(self.cfg), _cabi.ptr(self.blob), nbytes.value, C.byref(h)), "llb_gin_create")
            self.handle = h
        self.workspace = None
        self.B = 0
        self.n = self.e = 0
        self.grad_blob = None   # transposed weights of the predictor's backward, packed on the first backward

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.llb_gin_destroy(self.handle)
        except Exception:
            pass

    def bind(self, x, edge_index, edge_attr, batch, num_graphs: Optional[int] = None, want_logits: bool = False,
             validate: bool = True):
        """Binds a PyG-layout batch (builds the CSR on the device).  `validate` reads the kernels' input-defect flags back
        (one stream synchronisation, like the reference's own host read of batch[-1]) and raises the IndexError the
        reference's nn.Embedding / scatter raise for ids or indices out of range; pass False inside device-timed loops."""
        dev = self.device
        x = x.to(dev, torch.int64).contiguous()
        edge_index = edge_index.to(dev, torch.int64).contiguous()
        edge_attr = edge_attr.to(dev, torch.int64).contiguous()
        batch = batch.to(dev, torch.int64).contiguous()
        n, e = int(x.numel()), int(edge_attr.numel())
        if n == 0:
            raise ValueError("empty graph batch")
        # the reference reads batch[-1] on the host too (graph_encoder/model.py:127)
        B = int(batch[-1].item()) + 1 if num_graphs is None else int(num_graphs)
        with torch.cuda.device(dev):
            need = C.c_size_t()
            _cabi.check(self.lib.llb_gin_workspace_bytes(C.byref(self.cfg), n, e, B, int(want_logits), C.byref(need)),
                        "llb_gin_workspace_bytes")
            if self.workspace is None or self.workspace.numel() < need.value:
                self.workspace = None
                self.workspace = torch.empty(need.value, dtype=torch.uint8, device=dev)
            self._inputs = (x, edge_index, edge_attr, batch)
            _cabi.check(self.lib.llb_gin_bind(self.handle, _cabi.ptr(self.workspace), need.value, n, e, B, _cabi.ptr(x),
                                              _cabi.ptr(edge_index), _cabi.ptr(edge_attr), _cabi.ptr(batch), _cabi.stream_ptr()),
                        "llb_gin_bind")
            if validate:
                flags = C.c_int32(0)
                _cabi.check(self.lib.llb_gin_input_flags(self.handle, C.byref(flags), _cabi.stream_ptr()), "llb_gin_input_flags")
                if flags.value:
                    names = ((1, "atom id outside [0,118)"), (2, "`batch` not ascending or outside [0,num_graphs)"),
                             (4, "edge endpoint outside [0,num_nodes)"), (8, "bond type outside [0,5)"))
                    what = [msg for bit, msg in names if flags.value & bit]
                    raise IndexError("index out of range in the graph batch: " + "; ".join(what))
        self.B, self.n, self.e = B, n, e
        return B

    def encoder_forward(self, want_pooled: bool = False):
        out = torch.empty((self.B, self.H), dtype=torch.float32, device=self.device)
        pooled = torch.empty((self.B, self.H), dtype=torch.float32, device=self.device) if want_pooled else None
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.llb_gin_encoder_forward(self.handle, _cabi.ptr(out), _cabi.ptr(pooled), _cabi.stream_ptr()),
                        "llb_gin_encoder_forward")
        return (out, pooled) if want_pooled else out

    def predictor_forward(self, c: Optional[torch.Tensor]):
        logits = torch.empty((self.B, self.out_dim), dtype=torch.float32, device=self.device)
        if c is not None:
            c = c.to(self.device, torch.float32).contiguous()
            assert c.shape == (self.B, self.text_dim), (c.shape, self.B, self.text_dim)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.llb_gin_predictor_forward(self.handle, _cabi.ptr(c), _cabi.ptr(logits), _cabi.stream_ptr()),
                        "llb_gin_predictor_forward")
        return logits

    def predictor_forward_saved(self, c: torch.Tensor):
        """predictor_forward (bit-identical logits) that also returns what predictor_backward_c needs: the `saved` buffer and the
        batch sizes it was filled for.  The buffer belongs to this call, so several forwards can be back-propagated in any order."""
        c = c.to(self.device, torch.float32).contiguous()
        assert c.shape == (self.B, self.text_dim), (c.shape, self.B, self.text_dim)
        logits = torch.empty((self.B, self.out_dim), dtype=torch.float32, device=self.device)
        dims = (self.n, self.e, self.B)
        with torch.cuda.device(self.device):
            need = C.c_size_t()
            _cabi.check(self.lib.llb_gin_saved_bytes(C.byref(self.cfg), *dims, C.byref(need)), "llb_gin_saved_bytes")
            saved = torch.empty(need.value, dtype=torch.uint8, device=self.device)
            _cabi.check(self.lib.llb_gin_predictor_forward_saved(self.handle, _cabi.ptr(c), _cabi.ptr(logits), _cabi.ptr(saved), need.value,
                                                                 _cabi.stream_ptr()), "llb_gin_predictor_forward_saved")
        return logits, saved, dims

    def predictor_backward_c(self, c: torch.Tensor, dlogits: torch.Tensor, saved: torch.Tensor, dims) -> torch.Tensor:
        """dL/dc (B, text_dim) fp32 from dL/dlogits of the forward that filled `saved` (c: that forward's condition)."""
        n, e, B = dims
        c = c.to(self.device, torch.float32).contiguous()
        dlogits = dlogits.to(self.device, torch.float32).contiguous()
        assert dlogits.shape == (B, self.out_dim) and c.shape == (B, self.text_dim), (dlogits.shape, c.shape)
        dc = torch.empty((B, self.text_dim), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            if self.grad_blob is None:
                need = C.c_size_t()
                _cabi.check(self.lib.llb_gin_grad_packed_bytes(C.byref(self.cfg), C.byref(need)), "llb_gin_grad_packed_bytes")
                blob = torch.empty(need.value, dtype=torch.uint8, device=self.device)
                _cabi.check(self.lib.llb_gin_pack_grad_weights(self.handle, _cabi.ptr(blob), need.value, _cabi.stream_ptr()),
                            "llb_gin_pack_grad_weights")
                self.grad_blob = blob
            _cabi.check(self.lib.llb_gin_predictor_backward_c(self.handle, n, e, B, _cabi.ptr(c), _cabi.ptr(dlogits), _cabi.ptr(saved),
                                                              saved.numel(), _cabi.ptr(self.grad_blob), self.grad_blob.numel(),
                                                              _cabi.ptr(dc), _cabi.stream_ptr()), "llb_gin_predictor_backward_c")
        return dc

    def predictor_topk(self, c: Optional[torch.Tensor], k: int):
        probs = torch.empty((self.B, k), dtype=torch.float32, device=self.device)
        idx = torch.empty((self.B, k), dtype=torch.int32, device=self.device)
        if c is not None:
            c = c.to(self.device, torch.float32).contiguous()
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.llb_gin_predictor_topk(self.handle, _cabi.ptr(c), int(k), _cabi.ptr(probs), _cabi.ptr(idx),
                                                        _cabi.stream_ptr()), "llb_gin_predictor_topk")
        return probs, idx

    def head_stats(self) -> dict:
        """Rows of the last predictor_topk call that used the fused head kernel / that fell back to the exact path."""
        return {"fused_rows": int(self.lib.llb_gin_stat(self.handle, 0)), "flagged_rows": int(self.lib.llb_gin_stat(self.handle, 1))}

    def launch_count(self) -> int:
        return int(self.lib.llb_gin_launch_count(self.handle))
