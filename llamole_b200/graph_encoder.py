"""GraphCLIP -- drop-in for the reference's src/model/graph_encoder/model.py:GraphCLIP (GIN + virtual node +
projection head).  Same constructor, files and state-dict keys (SURVEY.md section 8b); `forward` runs on the
sm_100a C ABI (CSR segmented aggregation + tcgen05 GEMMs), no PyTorch op on the compute path, no CPU fallback.
With a trainable parameter and grad mode on, `forward` is differentiable with respect to every parameter (backward in CUDA,
csrc/llb_gin_grad.cu)."""
from __future__ import annotations

import json
import os
import warnings

import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import _cabi
from .gin_engine import GinEngine, _Holder, gin_trunk_skeleton


class _EmbeddingsWrtParameters(torch.autograd.Function):
    """Embeddings as a function of the parameters: forward = the engine's saved forward, backward = every parameter's gradient
    on the device.  `params` are the encoder's then the projection head's parameters, in the order of `names`."""

    @staticmethod
    def forward(ctx, eng, names, out_dtype, *params):
        out, saved, dims = eng.encoder_forward_saved()
        ctx.eng, ctx.saved, ctx.dims, ctx.names = eng, saved, dims, names   # the engine (and its blob) stay alive with this graph
        ctx.dtypes = [p.dtype for p in params]
        return out.to(out_dtype)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        trunk, head = ctx.eng.encoder_backward(grad_out.float(), ctx.saved, ctx.dims)
        grads = [(trunk if part == "enc" else head)[key].to(dt) if need else None
                 for (part, key), dt, need in zip(ctx.names, ctx.dtypes, ctx.needs_input_grad[3:])]
        return (None, None, None, *grads)


class GraphCLIP(nn.Module):
    def __init__(self, graph_num_layer, graph_hidden_size, dropout, model_config):
        super().__init__()
        self.model_config = model_config
        self.hidden_size = graph_hidden_size
        self.num_layer = graph_num_layer
        H = graph_hidden_size
        self.molecule_encoder = gin_trunk_skeleton(graph_num_layer, H, dropout, affine_norms=True)
        proj = _Holder()   # ProjectionHead, graph_encoder/model.py:178-197
        proj.fc1 = nn.Linear(H, H)
        proj.norm1 = nn.LayerNorm(H)
        proj.fc2 = nn.Linear(H, H)
        self.molecule_projection = proj
        self.drop_ratio = dropout
        self._engine = None
        self._warned_dropout = False

    def init_model(self, model_path, verbose=True):
        molecule_path = os.path.join(model_path, "model.pt")
        proj_path = os.path.join(model_path, "model_proj.pt")
        if not os.path.exists(molecule_path):
            raise FileNotFoundError(f"Molecule encoder file not found: {molecule_path}")
        if not os.path.exists(proj_path):
            raise FileNotFoundError(f"Molecule projection file not found: {proj_path}")
        self.molecule_encoder.load_state_dict(torch.load(molecule_path, map_location="cpu", weights_only=False))
        self.molecule_projection.load_state_dict(torch.load(proj_path, map_location="cpu", weights_only=False))
        self._engine = None
        if verbose:
            print("GraphCLIP Models initialized.")

    def save_pretrained(self, output_dir):
        os.makedirs(output_dir, exist_ok=True)
        torch.save(self.molecule_encoder.state_dict(), os.path.join(output_dir, "model.pt"))
        torch.save(self.molecule_projection.state_dict(), os.path.join(output_dir, "model_proj.pt"))
        with open(os.path.join(output_dir, "model_config.json"), "w") as f:
            json.dump(self.model_config, f, indent=2)

    def disable_grads(self):
        for p in self.parameters():
            p.requires_grad = False

    def engine(self) -> GinEngine:
        dev = next(self.parameters()).device
        fp = _cabi.params_fingerprint(self)   # repack when a parameter was replaced / cast / written in place
        if self._engine is None or self._engine.device != dev or self._engine.fingerprint != fp:
            self._engine = None
            f32 = lambda sd: {k: v.detach().to(dev, torch.float32).contiguous() for k, v in sd.items()}  # noqa: E731
            trunk = f32(self.molecule_encoder.state_dict())
            pj = f32(self.molecule_projection.state_dict())
            head = {"w0": pj["fc1.weight"], "b0": pj["fc1.bias"], "lnw": pj["norm1.weight"], "lnb": pj["norm1.bias"],
                    "w4": pj["fc2.weight"], "b4": pj["fc2.bias"]}
            self._engine = GinEngine(dev, self.hidden_size, self.num_layer, False, 0, 0, trunk, head)
            self._engine.fingerprint = fp
        return self._engine

    def forward(self, x, edge_index, edge_attr, batch):
        """(B,H) unit-norm embeddings in the parameters' dtype (graph_encoder/model.py:37-41).

        Differentiable with respect to the parameters when grad mode is on, some parameter requires grad and the module is on a
        B200 (the reference loader keeps the graph modules trainable unless disable_graph_model_gradient is set, and the SFT loss
        then trains the encoder through the graph-to-LM connector): the embeddings carry a grad_fn whose backward runs on the
        device.  Otherwise (disable_grads(), torch.no_grad()) no graph is recorded."""
        params = list(self.parameters())
        dtype = params[0].dtype
        if not (torch.is_grad_enabled() and any(p.requires_grad for p in params) and _cabi.arch_ok(params[0].device)):
            with torch.no_grad():
                eng = self.engine()
                eng.bind(x, edge_index, edge_attr, batch)
                return eng.encoder_forward().to(dtype)
        if self.training and self.drop_ratio > 0 and not self._warned_dropout:
            warnings.warn("GraphCLIP: dropout is not applied (the drop-in's forward never applies it), so training-mode "
                          "embeddings and their gradients equal eval-mode ones", stacklevel=2)
            self._warned_dropout = True
        with torch.no_grad():
            eng = self.engine()
            eng.bind(x, edge_index, edge_attr, batch)
        enc = list(self.molecule_encoder.named_parameters())
        proj = list(self.molecule_projection.named_parameters())
        names = [("enc", k) for k, _ in enc] + [("proj", k) for k, _ in proj]
        return _EmbeddingsWrtParameters.apply(eng, names, dtype, *[p for _, p in enc], *[p for _, p in proj])
