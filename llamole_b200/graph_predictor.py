"""GraphPredictor -- drop-in for the reference's src/model/graph_predictor/model.py:GraphPredictor (text-conditioned
GIN template classifier + CostMLP).  The device part (trunk, head, softmax/top-k, cost MLP) runs on the sm_100a
C ABI; the host chemistry (rdchiral template application, Morgan fingerprints) stays the reference's libraries."""
from __future__ import annotations

import ctypes as C
import json
import os
import warnings
from collections import defaultdict

import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import _cabi
from .gin_engine import GinEngine, _Holder, gin_trunk_skeleton, mlp4


_TEMPLATE_BACKEND = None


def set_template_backend(fn) -> None:
    """Override the retro-template application `fn(template, product_smiles) -> list of reactant SMILES`
    (default: rdchiral.main.rdchiralRunText, as graph_predictor/model.py:191).  None restores the default."""
    global _TEMPLATE_BACKEND
    _TEMPLATE_BACKEND = fn


def _template_backend():
    if _TEMPLATE_BACKEND is not None:
        return _TEMPLATE_BACKEND
    from rdchiral.main import rdchiralRunText

    return rdchiralRunText


class _LogitsWrtCondition(torch.autograd.Function):
    """Template logits as a function of c alone: forward = the engine's saved forward, backward = dc on the device."""

    @staticmethod
    def forward(ctx, c, eng, out_dtype):
        logits, saved, dims = eng.predictor_forward_saved(c)
        ctx.eng, ctx.saved, ctx.dims = eng, saved, dims   # the engine (and its blobs) stay alive until this graph is freed
        ctx.save_for_backward(c)
        return logits.to(out_dtype)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_logits):
        (c,) = ctx.saved_tensors
        dc = ctx.eng.predictor_backward_c(c, grad_logits.float(), ctx.saved, ctx.dims)
        return dc.to(c.dtype), None, None


class GraphPredictor(nn.Module):
    def __init__(self, num_layer, hidden_size, drop_ratio, out_dim, model_config, label_to_template, available=None):
        super().__init__()
        self.model_config = model_config
        self.text_input_size = model_config.get("text_input_size", 768)
        self.available = available
        self.text_drop = drop_ratio
        self.hidden_size, self.num_layer, self.out_dim = hidden_size, num_layer, out_dim
        if hasattr(label_to_template, "columns"):   # pandas.DataFrame
            label_to_template = dict(zip(label_to_template["rule_label"], label_to_template["retro_templates"]))
        self.label_to_template = label_to_template
        H = hidden_size
        pred = gin_trunk_skeleton(num_layer, H, drop_ratio, affine_norms=False)    # graph_predictor/model.py:231-272
        pred.adapters = nn.ModuleList(nn.Sequential(nn.SiLU(), nn.Linear(self.text_input_size, 3 * H)) for _ in range(num_layer))
        pred.text_dropping = nn.Embedding(1, self.text_input_size)
        pred.decoder = mlp4(H, 4 * H, out_dim, drop_ratio)
        self.predictor = pred
        self.neural_cost = None
        self._engine = None
        self._warned_param_grads = False

    # ------------------------------------------------------------------ files
    def init_model(self, model_path, verbose=False):
        model_file = os.path.join(model_path, "model.pt")
        if not os.path.exists(model_file):
            raise FileNotFoundError(f"Model file not found: {model_file}")
        self.predictor.load_state_dict(torch.load(model_file, map_location="cpu", weights_only=True))
        self._engine = None

    def init_neural_cost(self, model_path, verbose=False):
        model_file = os.path.join(model_path, "cost_model.pt")
        if not os.path.exists(model_file):
            raise FileNotFoundError(f"Model file not found: {model_file}")
        cost = _Holder()   # CostMLP(n_layers=1, 2048, 128): layers.0, layers.3 (graph_predictor/model.py:355-372)
        cost.layers = nn.Sequential(nn.Linear(2048, 128), nn.ReLU(), nn.Dropout(0.1), nn.Linear(128, 1))
        cost.load_state_dict(torch.load(model_file, map_location="cpu", weights_only=True))
        for p in cost.parameters():
            p.requires_grad = False
        self.neural_cost = cost

    def save_pretrained(self, output_dir):
        import pandas as pd

        os.makedirs(output_dir, exist_ok=True)
        torch.save(self.predictor.state_dict(), os.path.join(output_dir, "model.pt"))
        if self.neural_cost is not None:
            torch.save(self.neural_cost.state_dict(), os.path.join(output_dir, "cost_model.pt"))
        with open(os.path.join(output_dir, "model_config.json"), "w") as f:
            json.dump(self.model_config, f, indent=2)
        pd.DataFrame(list(self.label_to_template.items()), columns=["rule_label", "retro_templates"]).to_csv(
            os.path.join(output_dir, "label_to_template.csv.gz"), index=False, compression="gzip")
        if self.available is not None:
            if isinstance(self.available, list):
                df = pd.DataFrame(self.available, columns=["smiles"])
            elif isinstance(self.available, pd.DataFrame):
                df = self.available
            else:
                raise ValueError("available must be either a list of SMILES strings or a pandas DataFrame")
            df.to_csv(os.path.join(output_dir, "available.csv.gz"), index=False, compression="gzip")

    def disable_grads(self):
        for p in self.predictor.parameters():
            p.requires_grad = False

    # ------------------------------------------------------------------ device path
    def engine(self) -> GinEngine:
        dev = next(self.predictor.parameters()).device
        fp = _cabi.params_fingerprint(self.predictor)   # repack when a parameter was replaced / cast / written in place
        if self._engine is None or self._engine.device != dev or self._engine.fingerprint != fp:
            self._engine = None
            sd = {k: v.detach().to(dev, torch.float32).contiguous() for k, v in self.predictor.state_dict().items()}
            head = {"w0": sd["decoder.0.weight"], "b0": sd["decoder.0.bias"], "lnw": sd["decoder.1.weight"],
                    "lnb": sd["decoder.1.bias"], "w4": sd["decoder.4.weight"], "b4": sd["decoder.4.bias"]}
            self._engine = GinEngine(dev, self.hidden_size, self.num_layer, True, self.out_dim, self.text_input_size, sd, head)
            self._engine.fingerprint = fp
        return self._engine

    def forward(self, x, edge_index, edge_attr, batch, c):
        """Template logits (B,out_dim) (graph_predictor/model.py:306-353); c (B,768) or None.

        Differentiable with respect to c when c requires grad and grad mode is on (Llamole's SFT step back-propagates the retro
        loss through the frozen predictor into the connector): the logits then carry a grad_fn whose backward runs on the
        device.  The predictor's parameters never receive a gradient."""
        dtype = next(self.predictor.parameters()).dtype
        if c is None or not c.requires_grad or not torch.is_grad_enabled():
            with torch.no_grad():
                eng = self.engine()
                eng.bind(x, edge_index, edge_attr, batch)
                return eng.predictor_forward(c).to(dtype)
        if not self._warned_param_grads and any(p.requires_grad for p in self.predictor.parameters()):
            warnings.warn("GraphPredictor: gradients flow to c only; the predictor's parameters receive none "
                          "(call disable_grads() to freeze them, as the reference loader does)", stacklevel=2)
            self._warned_param_grads = True
        with torch.no_grad():
            eng = self.engine()
            eng.bind(x, edge_index, edge_attr, batch)
        return _LogitsWrtCondition.apply(c, eng, dtype)

    @torch.no_grad()
    def topk_templates(self, x, edge_index, edge_attr, batch, c, topk):
        """Batched device part of sample_templates: softmax over out_dim + top-k -> (probs (B,k), indices (B,k))."""
        eng = self.engine()
        eng.bind(x, edge_index, edge_attr, batch, want_logits=True)
        return eng.predictor_topk(c, topk)

    def estimate_cost(self, smiles):
        if self.neural_cost is None:
            raise ValueError("Cost model is not initialized.")
        import numpy as np
        from rdkit import Chem
        from rdkit.Chem import AllChem

        mol = Chem.MolFromSmiles(smiles)
        if mol is None:
            raise ValueError(f"Invalid SMILES string: {smiles}")
        fp = AllChem.GetMorganFingerprintAsBitVect(mol, 2, nBits=2048)
        arr = np.zeros(2048, dtype=np.float32)
        arr[list(fp.GetOnBits())] = 1
        return float(self.cost_from_fingerprints(torch.from_numpy(arr).view(1, -1)).item())

    @torch.no_grad()
    def cost_from_fingerprints(self, fps: torch.Tensor) -> torch.Tensor:
        """CostMLP.forward on (n,2048) fingerprints (graph_predictor/model.py:387-391)."""
        if self.neural_cost is None:
            raise ValueError("Cost model is not initialized.")
        dev = next(self.neural_cost.parameters()).device
        _cabi.require_cuda(next(self.neural_cost.parameters()), "cost model")
        sd = {k: v.detach().to(dev, torch.float32).contiguous() for k, v in self.neural_cost.state_dict().items()}
        fps = fps.to(dev, torch.float32).contiguous()
        out = torch.empty(fps.shape[0], dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _cabi.check(_cabi.lib().llb_cost_mlp(_cabi.ptr(sd["layers.0.weight"]), _cabi.ptr(sd["layers.0.bias"]),
                                                 _cabi.ptr(sd["layers.3.weight"]), _cabi.ptr(sd["layers.3.bias"]), _cabi.ptr(fps),
                                                 fps.shape[0], fps.shape[1], sd["layers.0.weight"].shape[0], _cabi.ptr(out),
                                                 _cabi.stream_ptr()), "llb_cost_mlp")
            torch.cuda.current_stream().synchronize()
        return out.view(-1, 1)

    def sample_templates(self, product_graph, c, product_smiles, topk=10):
        """(reactants, scores, templates) sorted by merged score, scores summing to 1; ([],[],[]) if no template applies
        (graph_predictor/model.py:164-228).  The reference's second, discarded predictor pass (c=None) is dropped."""
        x, edge_index, edge_attr = product_graph.x, product_graph.edge_index, product_graph.edge_attr
        batch = torch.zeros(x.size(0), dtype=torch.long, device=x.device)
        probs, idx = self.topk_templates(x, edge_index, edge_attr, batch, c, topk)
        return self._apply_templates(probs[0].float().cpu().tolist(), idx[0].cpu().tolist(), product_smiles)

    def sample_templates_batch(self, product_graphs, c, product_smiles_list, topk=10):
        """Batched A* expansion (SURVEY.md section 8f-1): `sample_templates` for MANY products with ONE predictor call.

        The reference expands one open node per planner iteration with a B=1 predictor call (planner/molstar.py:24-71,
        modeling_llamole.py:784-889); expanding the k best open nodes together turns that into the batched candidate
        scoring of BASELINE.json configs[3].  `product_graphs` is a list of PyG-like objects (x, edge_index, edge_attr),
        `c` (len, text_dim) or None, `product_smiles_list` the matching SMILES.  Returns one (reactants, scores,
        templates) triple per product, each identical to what `sample_templates` returns for that product alone."""
        if len(product_graphs) != len(product_smiles_list):
            raise ValueError("product_graphs and product_smiles_list differ in length")
        if c is not None and c.shape[0] != len(product_graphs):
            raise ValueError(f"c has {c.shape[0]} rows for {len(product_graphs)} products")
        if not product_graphs:
            return []
        dev = product_graphs[0].x.device
        xs, eis, eas, bs = [], [], [], []
        base = 0
        for gi, g in enumerate(product_graphs):
            n = int(g.x.size(0))
            if n == 0:
                raise ValueError(f"product {gi} has no atoms")
            xs.append(g.x.reshape(-1))
            eis.append(g.edge_index + base)
            eas.append(g.edge_attr.reshape(-1))
            bs.append(torch.full((n,), gi, dtype=torch.long, device=dev))
            base += n
        probs, idx = self.topk_templates(torch.cat(xs), torch.cat(eis, dim=1), torch.cat(eas), torch.cat(bs), c, topk)
        probs, idx = probs.float().cpu().tolist(), idx.cpu().tolist()
        return [self._apply_templates(p, i, smi) for p, i, smi in zip(probs, idx, product_smiles_list)]

    def _apply_templates(self, probs, labels, product_smiles):
        """Host half of sample_templates (graph_predictor/model.py:187-228): apply each of the top-k templates to the
        product, split a template's probability evenly over its outcomes, merge identical reactant sets."""
        run = _template_backend()
        found = defaultdict(list)
        for prob, label in zip(probs, labels):
            template = self.label_to_template[label]
            try:
                outcomes = sorted(run(template, product_smiles))
            except Exception:
                continue
            for reactant in outcomes:
                key = ".".join(sorted(reactant.strip().split("."))) if "." in reactant else reactant
                found[key].append((prob / len(outcomes), template))
        if not found:
            return [], [], []
        merged = sorted(((r, sum(s for s, _ in lst), lst[0][1]) for r, lst in found.items()), key=lambda it: it[1], reverse=True)
        total = sum(s for _, s, _ in merged)
        return [r for r, _, _ in merged], [s / total for _, s, _ in merged], [t for _, _, t in merged]
