"""GraphDiT -- drop-in for the reference's src/model/graph_decoder/diffusion_model.py:GraphDiT.

Same constructor, attributes, files and state-dict keys (SURVEY.md section 8b), but `generate` runs the whole
reverse-diffusion loop in hand-written sm_100a CUDA through the C ABI (include/llamole_b200.h).  The modules
below only HOLD parameters (so `load_state_dict`, `.to(device)`, `.parameters()` and the loader's dtype cast
behave as in the reference); no PyTorch op is on the compute path and there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import json
import os
from types import SimpleNamespace
from typing import Callable, List, Optional, Tuple

import numpy as np
import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import _cabi

X_CLASSES, E_CLASSES, Y_DIM, TEXT_DIM = 16, 5, 10, 768


class _Holder(nn.Module):
    """Parameter container (no forward): keeps the reference's module tree so state-dict keys match."""


def _denoiser_skeleton(max_n_nodes, hidden, depth, heads, mlp_ratio) -> nn.Module:
    # key layout of graph_decoder/transformer.py:26-64, layers.py:25-53,90-109, conditions.py:19-31,60-74,100-106
    H, F, d0 = hidden, int(hidden * mlp_ratio), X_CLASSES + E_CLASSES * max_n_nodes
    den = _Holder()
    den.x_embedder = nn.Sequential(nn.Linear(d0, H, bias=False), nn.LayerNorm(H))
    den.t_embedder = _Holder()
    den.t_embedder.mlp = nn.Sequential(nn.Linear(256, H), nn.SiLU(), nn.Linear(H, H))
    den.y_embedder = _Holder()
    den.y_embedder.embedding_drop = nn.Embedding(Y_DIM, H)
    den.y_embedder.mlps = nn.ModuleList(
        nn.Sequential(nn.Linear(1, H), nn.Softmax(dim=1), nn.Linear(H, H, bias=False)) for _ in range(Y_DIM))
    den.txt_embedder = _Holder()
    den.txt_embedder.embedding_drop = nn.Embedding(1, H)
    den.txt_embedder.linear = nn.Linear(TEXT_DIM, H)
    blocks = []
    for _ in range(depth):
        b = _Holder()
        b.attn = _Holder()
        b.attn.qkv = nn.Linear(H, 3 * H, bias=False)
        b.attn.q_norm = nn.LayerNorm(H // heads)
        b.attn.k_norm = nn.LayerNorm(H // heads)
        b.attn.proj = nn.Linear(H, H)
        b.mlp = _Holder()
        b.mlp.fc1 = nn.Linear(H, F)
        b.mlp.fc2 = nn.Linear(F, H)
        b.adaLN_modulation = nn.Sequential(nn.Linear(H, H), nn.SiLU(), nn.Linear(H, 6 * H), nn.Softsign())
        blocks.append(b)
    den.blocks = nn.ModuleList(blocks)
    den.output_layer = _Holder()
    den.output_layer.xedecoder = _Holder()
    den.output_layer.xedecoder.fc1 = nn.Linear(H, H)
    den.output_layer.xedecoder.fc2 = nn.Linear(H, d0)
    den.output_layer.adaLN_modulation = nn.Sequential(nn.Linear(H, H), nn.SiLU(), nn.Linear(H, 2 * d0))
    return den


def cosine_schedule(T: int, s: float = 0.008) -> Tuple[torch.Tensor, torch.Tensor]:
    """betas / alphas_bar, index 0..T.  Same arithmetic as diffusion_utils.py:364-373 + :172-185 (float64 numpy over
    T+2 linspace points, cast to fp32, then exp(cumsum(log(1-beta))) in fp32) -- the values are looked up by the
    kernels, so they must be bit-identical to the reference's tables."""
    n = T + 2
    grid = np.linspace(0, n, n)
    ac = np.cos(0.5 * np.pi * ((grid / n) + s) / (1 + s)) ** 2
    ac = ac / ac[0]
    betas = torch.from_numpy((1 - ac[1:] / ac[:-1]).squeeze()).float()
    abar = torch.exp(torch.cumsum(torch.log(1 - torch.clamp(betas, min=0, max=1)), dim=0))
    return betas, abar


_SMILES_BACKEND: Optional[Callable] = None


def set_smiles_backend(fn: Optional[Callable]) -> None:
    """fn(molecule_list, atom_decoder) -> List[Optional[str]]; the reference's molecule_utils.graph_to_smiles
    (RDKit valency correction, host side, outside the accelerated path; SURVEY.md section 2)."""
    global _SMILES_BACKEND
    _SMILES_BACKEND = fn


def _smiles_backend() -> Callable:
    if _SMILES_BACKEND is not None:
        return _SMILES_BACKEND
    for mod in ("src.model.graph_decoder.molecule_utils", "graph_decoder.molecule_utils"):
        try:
            m = __import__(mod, fromlist=["graph_to_smiles"])
            return m.graph_to_smiles
        except Exception:
            continue
    raise ImportError(
        "GraphDiT.generate needs the reference's RDKit post-processing (graph_decoder/molecule_utils.graph_to_smiles); "
        "install it with llamole_b200.graph_decoder.set_smiles_backend(fn) or call generate_graphs() for the integer graphs")


class GraphDiT(nn.Module):
    def __init__(self, model_config_path, data_info_path, model_dtype):
        super().__init__()
        if not os.path.exists(model_config_path):
            raise FileNotFoundError(f"Configuration file not found: {model_config_path}")
        if not os.path.exists(data_info_path):
            raise FileNotFoundError(f"Data meta info file not found: {data_info_path}")
        import yaml

        with open(model_config_path, "r") as f:
            cfg = yaml.safe_load(f)
        with open(data_info_path, "r") as f:
            meta = json.load(f)
        self.model_config = SimpleNamespace(**cfg)
        self._meta = meta
        self.T = int(cfg["diffusion_steps"])
        self.guide_scale = cfg["guide_scale"]
        self.Xdim = self.Xdim_output = X_CLASSES
        self.Edim = self.Edim_output = E_CLASSES
        self.ydim = self.ydim_output = Y_DIM
        self.max_n_nodes = int(meta["max_node"])
        self.atom_decoder = meta["active_atoms"]
        self.hidden_size = int(cfg["hidden_size"])
        self.text_input_size = TEXT_DIM
        self.model_dtype = model_dtype
        self.denoiser = _denoiser_skeleton(self.max_n_nodes, self.hidden_size, int(cfg["depth"]), int(cfg["num_heads"]),
                                           cfg["mlp_ratio"])
        # marginal transition statistics (diffusion_model.py:78-93), kept in fp32 (DESIGN.md: the reference's
        # bf16 tables / bf16 time index are a precision defect that is not reproduced)
        atom_dist = torch.tensor(meta["atom_type_dist"], dtype=torch.float32)
        self.active_index = (atom_dist > 0).nonzero().squeeze()
        node_types = atom_dist[self.active_index]
        edge_types = torch.tensor(meta["bond_type_dist"], dtype=torch.float32)
        x_marg = node_types / node_types.sum()
        e_marg = edge_types / edge_types.sum()
        self.x_marginals = x_marg / x_marg.sum()
        self.e_marginals = e_marg / e_marg.sum()
        trans = torch.tensor(meta["transition_E"], dtype=torch.float32)
        xe_raw = trans[self.active_index][:, self.active_index].sum(dim=1)
        self.xe_conditions = xe_raw / xe_raw.sum(dim=-1, keepdim=True)
        ex_raw = xe_raw.t()
        self.ex_conditions = ex_raw / ex_raw.sum(dim=-1, keepdim=True)
        n_hist = torch.tensor(meta["n_atoms_per_mol_dist"], dtype=torch.float32)
        self.node_prob = n_hist / n_hist.sum()
        self.betas, self.alphas_bar = cosine_schedule(self.T)
        self._engine = None
        # worker processes of the graph -> SMILES conversion after sampling (1 = the reference's serial loop on this thread)
        self.smiles_workers = 1

    # ------------------------------------------------------------------ reference surface
    def init_model(self, model_dir, verbose=False):
        model_file = os.path.join(model_dir, "model.pt")
        if not os.path.exists(model_file):
            raise FileNotFoundError(f"Model file not found: {model_file}")
        self.denoiser.load_state_dict(torch.load(model_file, map_location="cpu", weights_only=True))
        self._engine = None
        if verbose:
            print("GraphDiT Denoiser Model initialized.")

    def save_pretrained(self, output_dir):
        import yaml

        os.makedirs(output_dir, exist_ok=True)
        torch.save(self.denoiser.state_dict(), os.path.join(output_dir, "model.pt"))
        with open(os.path.join(output_dir, "model_config.yaml"), "w") as f:
            yaml.dump(vars(self.model_config), f)
        with open(os.path.join(output_dir, "data.meta.json"), "w") as f:
            json.dump(self._meta, f, indent=2)

    def disable_grads(self):
        for p in self.denoiser.parameters():
            p.requires_grad = False

    def check_valid(self, smiles):
        for mod in ("src.model.graph_decoder.molecule_utils", "graph_decoder.molecule_utils"):
            try:
                return __import__(mod, fromlist=["check_valid"]).check_valid(smiles)
            except ImportError:
                continue
        raise ImportError("check_valid needs the reference's RDKit helpers (graph_decoder/molecule_utils.py)")

    def forward(self, x, edge_index, edge_attr, graph_batch, properties, text_embedding, no_label_index):
        """SFT training loss (diffusion_model.py:148-172; called by modeling_llamole.py:371-379); same value as the reference for
        the same torch.manual_seed.  The noisy state, the conditions (dropout, property noise, the text linear) and the
        cross-entropy are eager PyTorch (llamole_b200/dit_train.py), so torch's RNG is consumed in the reference's order.  The
        denoiser c -> masked logits runs on the sm_100a kernels, differentiable with respect to c (so text_embedding, the
        connector and the LLM get their gradient), when the module is on a B200 (`llb_arch_check`), the config is inside the
        engine's limits and no denoiser parameter requires grad -- the frozen decoder Llamole trains with (`disable_grads()`).
        Otherwise (CPU, other GPUs, unsupported shapes, a trainable decoder) the whole loss is eager PyTorch on the module's
        device and the parameters get their gradients too."""
        from .dit_train import graphdit_loss

        return graphdit_loss(self, x, edge_index, edge_attr, graph_batch, properties, text_embedding, no_label_index)

    def device_denoiser_ok(self) -> bool:
        """Whether `forward` runs the denoiser on the sm_100a kernels (see `forward`).  The sampler takes molecules of up to 128
        atoms, the device denoiser's backward up to 64: a checkpoint with a larger max_node trains through the eager loss."""
        params = list(self.denoiser.parameters())
        dev = params[0].device
        if dev.type != "cuda" or any(p.requires_grad for p in params):
            return False
        try:
            lib = _cabi.lib()
        except _cabi.LlamoleB200Error:
            return False
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        nbytes = C.c_size_t()
        cfg = _dit_config(self)
        return lib.llb_arch_check(idx) == _cabi.LLB_OK and \
            lib.llb_dit_packed_bytes(C.byref(cfg), C.byref(nbytes)) == _cabi.LLB_OK and \
            lib.llb_dit_grad_packed_bytes(C.byref(cfg), C.byref(nbytes)) == _cabi.LLB_OK

    def denoise_on_device(self, X_t, E_t, node_mask, c):
        """Masked logits (B,N,16), (B,N,N,5) of the one-hot noisy state (X_t, E_t) at condition c (B,H), in the parameters'
        dtype; differentiable with respect to c when c requires grad."""
        eng = self.engine()
        Xs, Es = state_from_onehot(X_t, E_t)
        n_host = node_mask.sum(dim=1).to("cpu", torch.int32)
        out_dtype = next(self.denoiser.parameters()).dtype
        if torch.is_grad_enabled() and c.requires_grad:
            return _DenoiserWrtCondition.apply(c, eng, Xs, Es, n_host, out_dtype)
        lX, lE, _ = eng.denoise_c(Xs, Es, n_host, c.detach(), want_saved=False)
        return lX.to(out_dtype), lE.to(out_dtype)

    @torch.no_grad()
    def generate(self, properties, text_embedding, no_label_index) -> List[Optional[str]]:
        X, E, n_nodes = self.generate_graphs(properties, text_embedding, no_label_index)
        Xc, Ec, nn_ = X.cpu(), E.cpu(), n_nodes.cpu()
        molecule_list = []
        for i in range(Xc.shape[0]):
            n = int(nn_[i])
            molecule_list.append([Xc[i, :n], Ec[i, :n, :n]])
        if self.smiles_workers > 1:
            from .smiles_io import graphs_to_smiles_parallel

            return graphs_to_smiles_parallel(molecule_list, self.atom_decoder, backend=_smiles_backend(), workers=self.smiles_workers)
        return _smiles_backend()(molecule_list, self.atom_decoder)

    # ------------------------------------------------------------------ accelerated path
    def _device(self) -> torch.device:
        return next(self.denoiser.parameters()).device

    def engine(self) -> "_DitEngine":
        """The packed-weight engine of the current parameters.  It is rebuilt whenever a parameter was replaced, moved or
        written in place since it was packed (`load_state_dict`, the reference loader's `param.data = param.data.to(dtype)`
        cast loop, `.to(device)`, fine-tuning steps): the fingerprint below is every parameter's (data_ptr, _version)."""
        dev = self._device()
        fp = _cabi.params_fingerprint(self.denoiser)
        if self._engine is None or self._engine.device != dev or self._engine.fingerprint != fp:
            self._engine = None   # release the old blob first
            self._engine = _DitEngine(self, dev)
            self._engine.fingerprint = fp
        return self._engine

    def sample_n_nodes(self, batch_size: int, generator: Optional[torch.Generator] = None) -> torch.Tensor:
        """Categorical draw from the node-count histogram (host side like diffusion_utils.py:157-162)."""
        return torch.multinomial(self.node_prob, batch_size, replacement=True, generator=generator)

    @torch.no_grad()
    def generate_graphs(self, properties, text_embedding, no_label_index=-200, n_nodes=None, noise=None, seed: Optional[int] = None,
                        steps: Optional[int] = None, mol_index_base: int = 0):
        """The timed region of `generate`: conditions -> integer graphs.

        Returns X (B,N) int64 (-1 = masked), E (B,N,N) int64 (-1 = masked pair), n_nodes (B,) on the module's device.
        `noise` = dict(qX0,qE0,qX,qE) of pre-drawn Exp(1) tensors reproduces the reference bit for bit given the
        same tensors (oracle parity); otherwise the in-kernel counter RNG keyed by (seed, step, molecule, position).
        `steps` truncates the loop to the first `steps` reverse steps (benchmark sampling only).
        `seed=None` (what `generate` uses) draws a fresh 62-bit seed from torch's global generator on every call, like the
        reference, whose multinomial draws advance the global generator (diffusion_utils.py:376-413): repeated calls with the
        same conditions give different molecules, and `torch.manual_seed` makes a run reproducible.  An explicit seed keys
        the counter RNG by (seed, step, mol_index_base + row, position) and reproduces the same graphs on every call.
        """
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (), dtype=torch.int64).item())
        eng = self.engine()
        dev = eng.device
        B = properties.shape[0]
        if B == 0:   # an empty shard of a sharded batch (sharding.sample_graphs_sharded): nothing to sample
            N = self.max_n_nodes
            z = lambda *shape: torch.zeros(shape, dtype=torch.int64, device=dev)  # noqa: E731
            return z(0, N), z(0, N, N), z(0)
        if n_nodes is None:
            n_nodes = self.sample_n_nodes(B)
        n_host = n_nodes.to("cpu", torch.int32).contiguous()
        props = properties.to(dev, torch.float32)
        props = torch.where(props == no_label_index, torch.full_like(props, float("nan")), props).contiguous()
        txt = text_embedding.to(dev, torch.float32).contiguous()
        eng.begin(n_host, props, txt, mol_index_base)
        if noise is not None:
            q = {k: noise[k].to(dev, torch.float32).contiguous() for k in ("qX0", "qE0", "qX", "qE")}
            eng.init_state(seed, q["qX0"], q["qE0"])
        else:
            q = None
            eng.init_state(seed, None, None)
        t_last = 1 if steps is None else max(1, self.T - steps + 1)
        eng.sample(self.T, t_last, seed, None if q is None else q["qX"], None if q is None else q["qE"])
        X, E = eng.get_state()
        return X.long(), E.long(), n_nodes.to(dev)


def _dit_config(model: GraphDiT, guide_scale: Optional[float] = None) -> _cabi.DitConfig:
    mc = model.model_config
    if guide_scale is None:
        guide_scale = 1.0 if model.guide_scale is None else model.guide_scale
    return _cabi.DitConfig(model.hidden_size, int(mc.depth), int(mc.num_heads), int(model.hidden_size * mc.mlp_ratio),
                           model.max_n_nodes, model.T, Y_DIM, TEXT_DIM, float(guide_scale))


class _DenoiserWrtCondition(torch.autograd.Function):
    """Denoiser logits as a function of c alone: forward = the engine's saved pass, backward = dc on the device."""

    @staticmethod
    def forward(ctx, c, eng, Xs, Es, n_host, out_dtype):
        lX, lE, saved = eng.denoise_c(Xs, Es, n_host, c.detach(), want_saved=True)
        ctx.eng, ctx.saved, ctx.dims = eng, saved, (int(n_host.numel()), int(n_host.sum()))   # one buffer per forward
        ctx.c_dtype = c.dtype
        return lX.to(out_dtype), lE.to(out_dtype)

    @staticmethod
    @once_differentiable
    def backward(ctx, gX, gE):
        B, N = ctx.dims[0], ctx.eng.N
        dev = ctx.eng.device
        gX = torch.zeros((B, N, X_CLASSES), device=dev) if gX is None else gX.float().contiguous()
        gE = torch.zeros((B, N, N, E_CLASSES), device=dev) if gE is None else gE.float().contiguous()
        dc = ctx.eng.backward_c(ctx.saved, ctx.dims, gX, gE)
        return dc.to(ctx.c_dtype), None, None, None, None, None


class _DitEngine:
    """Owns the packed weight blob, the workspace and the C handle for one device."""

    def __init__(self, model: GraphDiT, device: torch.device):
        if device.type != "cuda":
            raise _cabi.LlamoleB200Error(
                "GraphDiT parameters are on %s; move the module to a B200 (`.to('cuda')`): there is no CPU path" % device)
        self.device = device
        self.lib = _cabi.lib()
        self.model = model
        self.N = model.max_n_nodes
        self.cfg = _dit_config(model)
        with torch.cuda.device(device):
            _cabi.check(self.lib.llb_arch_check(device.index if device.index is not None else torch.cuda.current_device()),
                        "llb_arch_check")
            nbytes = C.c_size_t()
            _cabi.check(self.lib.llb_dit_packed_bytes(C.byref(self.cfg), C.byref(nbytes)), "llb_dit_packed_bytes")
            self.blob = torch.empty(nbytes.value, dtype=torch.uint8, device=device)
            self._pack()
            h = C.c_void_p()
            _cabi.check(self.lib.llb_dit_create(C.byref(self.cfg), _cabi.ptr(self.blob), nbytes.value, C.byref(h)), "llb_dit_create")
            self.handle = h
        self.workspace = None
        self.B = 0
        # the SFT loss's denoiser (GraphDiT.forward): its own handle on the same blob with guide_scale = 1 (one pass), so the
        # sampler's binding, workspace and captured graph are never touched; the transposed-weight blob is packed on first use
        self.train_cfg = _dit_config(model, guide_scale=1.0)
        self.train_handle = None
        self.train_workspace = None
        self.grad_blob = None

    def __del__(self):
        try:
            for h in (getattr(self, "handle", None), getattr(self, "train_handle", None)):
                if h:
                    self.lib.llb_dit_destroy(h)
        except Exception:
            pass

    def _pack(self):
        m, dev = self.model, self.device
        sd = {k: v.detach().to(dev, torch.float32).contiguous() for k, v in m.denoiser.state_dict().items()}
        D = int(m.model_config.depth)
        keep = []

        def arr(fmt, n):
            ts = [sd[fmt.format(i)] for i in range(n)]
            a = _cabi.ptr_array(ts)
            keep.append(a)
            return C.cast(a, C.POINTER(C.c_void_p))

        tabs = [t.to(dev, torch.float32).contiguous() for t in
                (m.x_marginals, m.e_marginals, m.xe_conditions, m.ex_conditions, m.betas, m.alphas_bar)]
        p = lambda k: _cabi.ptr(sd[k])  # noqa: E731
        w = _cabi.DitWeights(
            p("x_embedder.0.weight"), p("x_embedder.1.weight"), p("x_embedder.1.bias"),
            p("t_embedder.mlp.0.weight"), p("t_embedder.mlp.0.bias"), p("t_embedder.mlp.2.weight"), p("t_embedder.mlp.2.bias"),
            p("y_embedder.embedding_drop.weight"),
            arr("y_embedder.mlps.{}.0.weight", Y_DIM), arr("y_embedder.mlps.{}.0.bias", Y_DIM), arr("y_embedder.mlps.{}.2.weight", Y_DIM),
            p("txt_embedder.embedding_drop.weight"), p("txt_embedder.linear.weight"), p("txt_embedder.linear.bias"),
            arr("blocks.{}.attn.qkv.weight", D), arr("blocks.{}.attn.q_norm.weight", D), arr("blocks.{}.attn.q_norm.bias", D),
            arr("blocks.{}.attn.k_norm.weight", D), arr("blocks.{}.attn.k_norm.bias", D),
            arr("blocks.{}.attn.proj.weight", D), arr("blocks.{}.attn.proj.bias", D),
            arr("blocks.{}.mlp.fc1.weight", D), arr("blocks.{}.mlp.fc1.bias", D),
            arr("blocks.{}.mlp.fc2.weight", D), arr("blocks.{}.mlp.fc2.bias", D),
            arr("blocks.{}.adaLN_modulation.0.weight", D), arr("blocks.{}.adaLN_modulation.0.bias", D),
            arr("blocks.{}.adaLN_modulation.2.weight", D), arr("blocks.{}.adaLN_modulation.2.bias", D),
            p("output_layer.xedecoder.fc1.weight"), p("output_layer.xedecoder.fc1.bias"),
            p("output_layer.xedecoder.fc2.weight"), p("output_layer.xedecoder.fc2.bias"),
            p("output_layer.adaLN_modulation.0.weight"), p("output_layer.adaLN_modulation.0.bias"),
            p("output_layer.adaLN_modulation.2.weight"), p("output_layer.adaLN_modulation.2.bias"),
            *[_cabi.ptr(t) for t in tabs],
        )
        _cabi.check(self.lib.llb_dit_pack_weights(C.byref(self.cfg), C.byref(w), _cabi.ptr(self.blob), self.blob.numel(),
                                                  _cabi.stream_ptr()), "llb_dit_pack_weights")
        torch.cuda.current_stream().synchronize()   # the fp32 staging copies die with this frame
        del sd, tabs, keep

    # ---- thin wrappers -------------------------------------------------------------------------
    def begin(self, n_nodes_host: torch.Tensor, props: torch.Tensor, txt: torch.Tensor, mol_index_base: int = 0):
        B = int(n_nodes_host.numel())
        with torch.cuda.device(self.device):
            need = C.c_size_t()
            _cabi.check(self.lib.llb_dit_workspace_bytes(C.byref(self.cfg), B, C.byref(need)), "llb_dit_workspace_bytes")
            if self.workspace is None or self.workspace.numel() < need.value:
                self.workspace = None
                self.workspace = torch.empty(need.value, dtype=torch.uint8, device=self.device)
            self._cond = (props, txt)   # keep alive until consumed on the stream
            n_arr = (C.c_int32 * B)(*n_nodes_host.tolist())
            _cabi.check(self.lib.llb_dit_begin(self.handle, _cabi.ptr(self.workspace), self.workspace.numel(), B, n_arr,
                                               _cabi.ptr(props), _cabi.ptr(txt), int(mol_index_base), _cabi.stream_ptr()),
                        "llb_dit_begin")
        self.B = B

    def init_state(self, seed, qX0, qE0):
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.llb_dit_init_state(self.handle, int(seed), _cabi.ptr(qX0), _cabi.ptr(qE0), _cabi.stream_ptr()),
                        "llb_dit_init_state")

    def set_state(self, X: torch.Tensor, E: torch.Tensor):
        X = X.to(self.device, torch.int8).contiguous()
        E = E.to(self.device, torch.int8).contiguous()
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.llb_dit_set_state(self.handle, _cabi.ptr(X), _cabi.ptr(E), _cabi.stream_ptr()), "llb_dit_set_state")
            torch.cuda.current_stream().synchronize()

    def get_state(self):
        X = torch.empty((self.B, self.N), dtype=torch.int8, device=self.device)
        E = torch.empty((self.B, self.N, self.N), dtype=torch.int8, device=self.device)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.llb_dit_get_state(self.handle, _cabi.ptr(X), _cabi.ptr(E), _cabi.stream_ptr()), "llb_dit_get_state")
        return X, E

    def denoise(self, t: int, unconditioned: bool):
        lX = torch.empty((self.B, self.N, X_CLASSES), dtype=torch.float32, device=self.device)
        lE = torch.empty((self.B, self.N, self.N, E_CLASSES), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.llb_dit_denoise(self.handle, int(t), int(bool(unconditioned)), _cabi.ptr(lX), _cabi.ptr(lE),
                                                 _cabi.stream_ptr()), "llb_dit_denoise")
        return lX, lE

    def step(self, t: int, seed=0, qX=None, qE=None, want_probs=False):
        pX = pE = None
        if want_probs:
            pX = torch.zeros((self.B, self.N, X_CLASSES), dtype=torch.float32, device=self.device)
            pE = torch.zeros((self.B, self.N, self.N, E_CLASSES), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.llb_dit_step(self.handle, int(t), int(seed), _cabi.ptr(qX), _cabi.ptr(qE), _cabi.ptr(pX), _cabi.ptr(pE),
                                              _cabi.stream_ptr()), "llb_dit_step")
        return pX, pE

    def sample(self, t_first: int, t_last: int, seed=0, qX_all=None, qE_all=None):
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.llb_dit_sample(self.handle, int(t_first), int(t_last), int(seed), _cabi.ptr(qX_all), _cabi.ptr(qE_all),
                                                _cabi.stream_ptr()), "llb_dit_sample")

    def posterior_sample(self, t, lcX, lcE, luX, luE, seed=0, qX=None, qE=None, want_probs=True):
        pX = pE = None
        if want_probs:
            pX = torch.zeros((self.B, self.N, X_CLASSES), dtype=torch.float32, device=self.device)
            pE = torch.zeros((self.B, self.N, self.N, E_CLASSES), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.llb_dit_posterior_sample(self.handle, int(t), _cabi.ptr(lcX), _cabi.ptr(lcE), _cabi.ptr(luX),
                                                          _cabi.ptr(luE), int(seed), _cabi.ptr(qX), _cabi.ptr(qE), _cabi.ptr(pX),
                                                          _cabi.ptr(pE), _cabi.stream_ptr()), "llb_dit_posterior_sample")
        return pX, pE

    def denoise_c(self, Xs: torch.Tensor, Es: torch.Tensor, n_host: torch.Tensor, c: torch.Tensor, want_saved: bool):
        """Masked logits (fp32) of the int8 states Xs (B,N), Es (B,N,N) of molecules of n_host[b] atoms at condition c (B,H); with
        want_saved also the buffer backward_c needs (None otherwise)."""
        B = int(n_host.numel())
        dev = self.device
        Xs, Es = Xs.to(dev, torch.int8).contiguous(), Es.to(dev, torch.int8).contiguous()
        c = c.to(dev, torch.float32).contiguous()
        lX = torch.zeros((B, self.N, X_CLASSES), dtype=torch.float32, device=dev)
        lE = torch.zeros((B, self.N, self.N, E_CLASSES), dtype=torch.float32, device=dev)
        saved = None
        with torch.cuda.device(dev):
            if self.train_handle is None:
                h = C.c_void_p()
                _cabi.check(self.lib.llb_dit_create(C.byref(self.train_cfg), _cabi.ptr(self.blob), self.blob.numel(), C.byref(h)),
                            "llb_dit_create")
                self.train_handle = h
            need = C.c_size_t()
            _cabi.check(self.lib.llb_dit_workspace_bytes(C.byref(self.train_cfg), B, C.byref(need)), "llb_dit_workspace_bytes")
            if self.train_workspace is None or self.train_workspace.numel() < need.value:
                self.train_workspace = None
                self.train_workspace = torch.empty(need.value, dtype=torch.uint8, device=dev)
            if want_saved:
                sb = C.c_size_t()
                _cabi.check(self.lib.llb_dit_train_saved_bytes(C.byref(self.train_cfg), B, int(n_host.sum()), C.byref(sb)),
                            "llb_dit_train_saved_bytes")
                saved = torch.empty(sb.value, dtype=torch.uint8, device=dev)
            n_arr = (C.c_int32 * B)(*n_host.tolist())
            _cabi.check(self.lib.llb_dit_denoise_c(self.train_handle, _cabi.ptr(self.train_workspace), self.train_workspace.numel(), B,
                                                   n_arr, _cabi.ptr(Xs), _cabi.ptr(Es), _cabi.ptr(c), _cabi.ptr(lX), _cabi.ptr(lE),
                                                   _cabi.ptr(saved), 0 if saved is None else saved.numel(), _cabi.stream_ptr()),
                        "llb_dit_denoise_c")
        return lX, lE, saved

    def backward_c(self, saved: torch.Tensor, dims, dlX: torch.Tensor, dlE: torch.Tensor) -> torch.Tensor:
        """dL/dc (B,H) fp32 from dL/dlogits of the denoise_c call that filled `saved` (dims = (B, total atoms) of that call)."""
        B, M = dims
        dc = torch.empty((B, self.train_cfg.hidden), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            if self.grad_blob is None:
                need = C.c_size_t()
                _cabi.check(self.lib.llb_dit_grad_packed_bytes(C.byref(self.train_cfg), C.byref(need)), "llb_dit_grad_packed_bytes")
                blob = torch.empty(need.value, dtype=torch.uint8, device=self.device)
                _cabi.check(self.lib.llb_dit_pack_grad_weights(self.train_handle, _cabi.ptr(blob), need.value, _cabi.stream_ptr()),
                            "llb_dit_pack_grad_weights")
                self.grad_blob = blob
            _cabi.check(self.lib.llb_dit_backward_c(self.train_handle, B, M, _cabi.ptr(saved), saved.numel(), _cabi.ptr(self.grad_blob),
                                                    self.grad_blob.numel(), _cabi.ptr(dlX), _cabi.ptr(dlE), _cabi.ptr(dc),
                                                    _cabi.stream_ptr()), "llb_dit_backward_c")
        return dc

    def launch_count(self) -> int:
        return int(self.lib.llb_dit_launch_count(self.handle))

    def graph_state(self) -> int:
        """1 when the t-independent launches of a reverse step are replayed as a CUDA graph (small batches), see the header."""
        return int(self.lib.llb_dit_graph_state(self.handle))


def state_from_onehot(X: torch.Tensor, E: torch.Tensor):
    """One-hot (B,N,16)/(B,N,N,5) reference tensors -> int8 class state (-1 where the vector is all zero)."""
    Xs = torch.where(X.sum(-1) > 0, X.argmax(-1), torch.full_like(X.argmax(-1), -1)).to(torch.int8)
    Es = torch.where(E.sum(-1) > 0, E.argmax(-1), torch.full_like(E.argmax(-1), -1)).to(torch.int8)
    return Xs, Es
