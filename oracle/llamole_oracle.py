"""CPU oracle: a restatement of the reference's graph-module hot path in plain torch (CPU, fp32/fp64).

TEST INFRASTRUCTURE ONLY.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
`--impl reference` leg may import this file; the product path (llamole_b200/) never does and fails
loudly when its CUDA library is missing.

Parity status: PINNED.  The reference ships no tests or golden vectors (SURVEY.md section 4), so the
pin is the reference itself: oracle/make_golden.py imports the reference's modules verbatim from
a checkout of the original repository (oracle/ref_import.py), runs them on seeded inputs and
pre-drawn noise, and commits the outputs under tests/golden/; tests/test_oracle.py checks every
function here against those fixtures.

Every function works on a flat `state_dict` (name -> tensor, the reference's checkpoint layout,
SURVEY.md section 8b) instead of nn.Modules, and cites the reference lines it follows.  Paths are relative
to /root/reference/src/model.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor
LN_EPS = 1e-5


# ==============================================================================================
# Tables: noise schedule and marginal transition statistics
# ==============================================================================================
def cosine_schedule(T: int, s: float = 0.008) -> Tuple[Tensor, Tensor]:
    """betas[0..T], alphas_bar[0..T] (fp32).

    graph_decoder/diffusion_utils.py:364-373 (T+2 linspace points, spacing steps/(steps-1)) and
    :172-185 (float() cast, clamp, exp(cumsum(log))).
    """
    steps = T + 2
    x = np.linspace(0, steps, steps)
    ac = np.cos(0.5 * np.pi * ((x / steps) + s) / (1 + s)) ** 2
    ac = ac / ac[0]
    betas = torch.from_numpy((1 - ac[1:] / ac[:-1]).squeeze()).float()
    alphas = 1 - torch.clamp(betas, min=0, max=1)
    alphas_bar = torch.exp(torch.cumsum(torch.log(alphas), dim=0))
    return betas, alphas_bar


@dataclass
class DitTables:
    x_marg: Tensor   # (16,)
    e_marg: Tensor   # (5,)
    xe: Tensor       # (16,5) row-normalised
    ex: Tensor       # (5,16) row-normalised transpose of the raw counts
    n_dist: Tensor   # (max_n+1,) probabilities of the node count
    active_index: Tensor
    max_nodes: int


def dit_tables(meta: dict, dtype=torch.float32) -> DitTables:
    """graph_decoder/diffusion_utils.py:39-57 (DataInfos) and diffusion_model.py:78-93."""
    atom_dist = torch.tensor(meta["atom_type_dist"], dtype=torch.float32)
    active = (atom_dist > 0).nonzero().squeeze()
    node_types = atom_dist[active].to(dtype)
    edge_types = torch.tensor(meta["bond_type_dist"], dtype=torch.float32).to(dtype)
    x_marg = node_types / node_types.sum()
    e_marg = edge_types / edge_types.sum()
    x_marg = x_marg / x_marg.sum()
    e_marg = e_marg / e_marg.sum()
    trans = torch.tensor(meta["transition_E"], dtype=torch.float32).to(dtype)
    xe_raw = trans[active][:, active].sum(dim=1)          # (16,5)
    ex_raw = xe_raw.t()
    xe = xe_raw / xe_raw.sum(dim=-1, keepdim=True)
    ex = ex_raw / ex_raw.sum(dim=-1, keepdim=True)
    n_hist = torch.tensor(meta["n_atoms_per_mol_dist"], dtype=torch.float32)
    return DitTables(x_marg, e_marg, xe, ex, n_hist / n_hist.sum(), active, int(meta["max_node"]))


def union_transition(tb: DitTables) -> Tensor:
    """(d0,d0) joint matrix U, d0 = 16 + 5*max_n.  diffusion_utils.py:287-306."""
    n = tb.max_nodes
    u_x = tb.x_marg.unsqueeze(0).expand(len(tb.x_marg), -1)
    u_e = tb.e_marg.unsqueeze(0).expand(len(tb.e_marg), -1).repeat(n, n)
    u_xe = tb.xe.repeat(1, n)
    u_ex = tb.ex.repeat(n, 1)
    return torch.cat([torch.cat([u_x, u_xe], dim=1), torch.cat([u_ex, u_e], dim=1)], dim=0)


# ==============================================================================================
# Denoiser (graph_decoder/transformer.py, layers.py, conditions.py)
# ==============================================================================================
def _lin(sd, name, x):
    return F.linear(x, sd[name + ".weight"], sd.get(name + ".bias"))


def timestep_features(t_norm: Tensor, dim: int = 256) -> Tensor:
    """conditions.py:33-51: [cos(t f_k), sin(t f_k)], f_k = exp(-ln(1e4) k / half), on NORMALISED t."""
    half = dim // 2
    freqs = torch.exp(-math.log(10000) * torch.arange(half, dtype=torch.float32) / half)
    args = t_norm.reshape(-1, 1).float() * freqs[None]
    return torch.cat([torch.cos(args), torch.sin(args)], dim=-1)


def condition_vector(sd, y: Tensor, txt: Tensor, t_norm: Tensor, unconditioned: bool) -> Tensor:
    """c = t_emb + y_emb + txt_emb, (B,H).  transformer.py:98-101; conditions.py:53-58, 76-98, 108-123 (eval)."""
    dt = sd["t_embedder.mlp.0.weight"].dtype
    h = _lin(sd, "t_embedder.mlp.0", timestep_features(t_norm).to(dt))
    c = _lin(sd, "t_embedder.mlp.2", F.silu(h))
    B = y.shape[0]
    for d in range(y.shape[1]):
        col = y[:, d]
        drop = torch.ones_like(col, dtype=torch.bool) if unconditioned else torch.isnan(col)
        emb = sd["y_embedder.embedding_drop.weight"][d].unsqueeze(0).expand(B, -1).clone()
        keep = ~drop
        if keep.any():
            z = _lin(sd, f"y_embedder.mlps.{d}.0", col[keep].unsqueeze(1).to(dt))
            emb[keep] = F.linear(torch.softmax(z, dim=1), sd[f"y_embedder.mlps.{d}.2.weight"])
        c = c + emb
    drop = torch.ones(B, dtype=torch.bool) if unconditioned else torch.isnan(txt.sum(dim=1))
    emb = sd["txt_embedder.embedding_drop.weight"][0].unsqueeze(0).expand(B, -1).clone()
    keep = ~drop
    if keep.any():
        emb[keep] = _lin(sd, "txt_embedder.linear", txt[keep].to(dt))
    return c + emb


def _attention(sd, p, x, node_mask, heads):
    """layers.py:56-87: qkv (no bias) -> per-head affine LayerNorm on q,k -> masked SDPA -> proj."""
    B, N, H = x.shape
    dh = H // heads
    qkv = _lin(sd, p + "qkv", x).reshape(B, N, 3, heads, dh).permute(2, 0, 3, 1, 4)
    q, k, v = qkv[0], qkv[1], qkv[2]
    q = F.layer_norm(q, (dh,), sd[p + "q_norm.weight"], sd[p + "q_norm.bias"], LN_EPS)
    k = F.layer_norm(k, (dh,), sd[p + "k_norm.weight"], sd[p + "k_norm.bias"], LN_EPS)
    allow = node_mask[:, None, :, None] & node_mask[:, None, None, :]
    allow = allow | (allow.sum(dim=-1, keepdim=True) == 0)      # fully masked query rows see everything
    s = (q @ k.transpose(-1, -2)) * dh ** -0.5
    s = s.masked_fill(~allow, float("-inf"))
    o = torch.softmax(s, dim=-1) @ v
    return _lin(sd, p + "proj", o.transpose(1, 2).reshape(B, N, H))


def denoiser_forward(sd: Dict[str, Tensor], cfg: dict, X_in: Tensor, E_in: Tensor, node_mask: Tensor,
                     y: Tensor, txt: Tensor, t_norm: Tensor, unconditioned: bool,
                     return_hidden: bool = False):
    """Masked logits (X (B,N,16), E (B,N,N,5)).  transformer.py:93-108, 132-145, 163-187."""
    B, N, dx = X_in.shape
    heads, depth = cfg["num_heads"], cfg["depth"]
    tok = torch.cat([X_in, E_in.reshape(B, N, -1)], dim=-1)
    x = F.linear(tok, sd["x_embedder.0.weight"])
    H = x.shape[-1]
    x = F.layer_norm(x, (H,), sd["x_embedder.1.weight"], sd["x_embedder.1.bias"], LN_EPS)
    c = condition_vector(sd, y, txt, t_norm, unconditioned)
    for l in range(depth):
        p = f"blocks.{l}."
        mod = _lin(sd, p + "adaLN_modulation.2", F.silu(_lin(sd, p + "adaLN_modulation.0", c)))
        mod = mod / (1 + mod.abs())                                  # Softsign
        sh_a, sc_a, g_a, sh_m, sc_m, g_m = (m.unsqueeze(1) for m in mod.chunk(6, dim=1))
        a = F.layer_norm(_attention(sd, p + "attn.", x, node_mask, heads), (H,), None, None, LN_EPS)
        x = x + g_a * (a * (1 + sc_a) + sh_a)
        m = _lin(sd, p + "mlp.fc2", F.gelu(_lin(sd, p + "mlp.fc1", x)))
        m = F.layer_norm(m, (H,), None, None, LN_EPS)
        x = x + g_m * (m * (1 + sc_m) + sh_m)
    o = "output_layer."
    out = _lin(sd, o + "xedecoder.fc2", F.gelu(_lin(sd, o + "xedecoder.fc1", x)))
    d0 = out.shape[-1]
    mod = _lin(sd, o + "adaLN_modulation.2", F.silu(_lin(sd, o + "adaLN_modulation.0", c)))
    shift, scale = (m.unsqueeze(1) for m in mod.chunk(2, dim=1))
    out = F.layer_norm(out, (d0,), None, None, LN_EPS) * (1 + scale) + shift
    Xo = X_in + out[:, :, :dx]
    Eo = E_in + out[:, :, dx:].reshape(B, N, N, -1)
    both_invalid = (~node_mask)[:, :, None] & (~node_mask)[:, None, :]
    diag = torch.eye(N, dtype=torch.bool).unsqueeze(0)
    Eo = Eo.masked_fill((both_invalid | diag)[..., None], 0)
    Eo = 0.5 * (Eo + Eo.transpose(1, 2))
    xm = node_mask.unsqueeze(-1)
    Xo = Xo * xm                                                    # PlaceHolder.mask, diffusion_utils.py:93-108
    Eo = Eo * xm.unsqueeze(2) * xm.unsqueeze(1)
    if return_hidden:
        return Xo, Eo, x
    return Xo, Eo


# ==============================================================================================
# Posterior, guidance, sampling (graph_decoder/diffusion_model.py:309-399, diffusion_utils.py)
# ==============================================================================================
def posterior_dense(tb: DitTables, U: Tensor, logits_X: Tensor, logits_E: Tensor, X_t: Tensor, E_t: Tensor,
                    beta_t: float, abar_s: float, abar_t: float) -> Tuple[Tensor, Tensor]:
    """get_prob's tail with the reference's dense (d0,d0) transition matrices.

    diffusion_model.py:332-362; diffusion_utils.py:316-349 (Q = a I + (1-a) U), :476-492 (reverse_diffusion).
    """
    B, N, dx = logits_X.shape
    pX = torch.softmax(logits_X, dim=-1)
    pE = torch.softmax(logits_E, dim=-1)
    d0 = U.shape[0]
    eye = torch.eye(d0, dtype=U.dtype)
    Qt = beta_t * U + (1 - beta_t) * eye
    Qsb = abar_s * eye + (1 - abar_s) * U
    Qtb = abar_t * eye + (1 - abar_t) * U
    xt = torch.cat([X_t, E_t.reshape(B, N, -1)], dim=-1)
    p0 = torch.cat([pX, pE.reshape(B, N, -1)], dim=-1)
    left = xt @ Qt.t()
    right = p0 @ Qsb
    den = (Qtb @ xt.transpose(-1, -2)).transpose(-1, -2)
    un = left * right / den.clamp_min(1e-5)
    uX = un[:, :, :dx].clone()
    uE = un[:, :, dx:].reshape(B, N * N, -1).clone()
    uX[uX.sum(dim=-1) == 0] = 1e-5
    uE[uE.sum(dim=-1) == 0] = 1e-5
    probX = uX / uX.sum(dim=-1, keepdim=True)
    probE = (uE / uE.sum(dim=-1, keepdim=True)).reshape(B, N, N, -1)
    return probX, probE


def guidance(pc: Tensor, pu: Tensor, scale: float) -> Tensor:
    """diffusion_model.py:373-382."""
    p = pu * (pc / pu.clamp_min(1e-5)) ** scale
    return p / p.sum(dim=-1, keepdim=True).clamp_min(1e-5)


def sample_categories(probX: Tensor, probE: Tensor, node_mask: Tensor, qX: Tensor, qE: Tensor):
    """Integer categories (B,N), (B,N,N) given Exp(1) noise.  diffusion_utils.py:376-413 with
    multinomial(1) == argmax(p/q) (SURVEY.md section 8c)."""
    B, N, dx = probX.shape
    pX = probX.clone()
    pX[~node_mask] = 1.0 / dx
    pX = pX.clamp_min(1e-5)
    pX = pX / pX.sum(dim=-1, keepdim=True)
    Xs = (pX / qX).argmax(dim=-1)
    pE = probE.clone()
    de = pE.shape[-1]
    inv = ~(node_mask.unsqueeze(1) & node_mask.unsqueeze(2))
    pE[inv] = 1.0 / de
    pE[torch.eye(N, dtype=torch.bool).unsqueeze(0).expand(B, -1, -1)] = 1.0 / de
    pE = pE.clamp_min(1e-5)
    pE = pE / pE.sum(dim=-1, keepdim=True)
    Es = (pE / qE).argmax(dim=-1)
    Es = torch.triu(Es, diagonal=1)
    Es = Es + Es.transpose(1, 2)
    return Xs, Es


def one_hot_state(Xs: Tensor, Es: Tensor, node_mask: Tensor, dtype) -> Tuple[Tensor, Tensor]:
    """diffusion_model.py:388-399: one-hot then PlaceHolder.mask (diagonal of valid nodes = class 0)."""
    X = F.one_hot(Xs, 16).to(dtype) * node_mask.unsqueeze(-1)
    m = node_mask.unsqueeze(-1)
    E = F.one_hot(Es, 5).to(dtype) * m.unsqueeze(2) * m.unsqueeze(1)
    return X, E


def initial_state(tb: DitTables, node_mask: Tensor, qX0: Tensor, qE0: Tensor, dtype):
    """z_T from the limit marginals; E keeps the strict upper triangle + transpose, so its diagonal is an
    all-zero vector (NOT one-hot).  diffusion_utils.py:495-518."""
    B, N = node_mask.shape
    Xs = (tb.x_marg.to(dtype)[None, None, :] / qX0).argmax(dim=-1)
    Es = (tb.e_marg.to(dtype)[None, None, None, :] / qE0).argmax(dim=-1)
    X = F.one_hot(Xs, 16).to(dtype)
    E = F.one_hot(Es, 5).to(dtype)
    upper = torch.triu(torch.ones(N, N, dtype=dtype), diagonal=1)[None, :, :, None]
    E = E * upper
    E = E + E.transpose(1, 2)
    m = node_mask.unsqueeze(-1)
    return X * m, E * m.unsqueeze(2) * m.unsqueeze(1)


def reverse_step(sd, cfg, tb: DitTables, U: Tensor, sched, X: Tensor, E: Tensor, node_mask: Tensor, y: Tensor,
                 txt: Tensor, t_int: int, qX: Tensor, qE: Tensor, return_probs: bool = False):
    """One reverse step t -> t-1 with classifier-free guidance.  diffusion_model.py:309-399."""
    T = cfg["diffusion_steps"]
    betas, abar = sched
    B = X.shape[0]
    t_norm = torch.full((B, 1), t_int / T, dtype=X.dtype)
    beta_t, abar_s, abar_t = float(betas[t_int]), float(abar[t_int - 1]), float(abar[t_int])
    lX, lE = denoiser_forward(sd, cfg, X, E, node_mask, y, txt, t_norm, False)
    pX, pE = posterior_dense(tb, U, lX, lE, X, E, beta_t, abar_s, abar_t)
    gs = cfg.get("guide_scale")
    if gs is not None and gs != 1:
        luX, luE = denoiser_forward(sd, cfg, X, E, node_mask, y, txt, t_norm, True)
        puX, puE = posterior_dense(tb, U, luX, luE, X, E, beta_t, abar_s, abar_t)
        pX, pE = guidance(pX, puX, gs), guidance(pE, puE, gs)
    Xs, Es = sample_categories(pX, pE, node_mask, qX, qE)
    Xn, En = one_hot_state(Xs, Es, node_mask, X.dtype)
    if return_probs:
        return Xn, En, Xs, Es, pX, pE
    return Xn, En, Xs, Es


def sample_graphs(sd, cfg, meta, props: Tensor, txt: Tensor, n_nodes: Tensor, noise, dtype=torch.float32,
                  no_label_index=-200.0, steps: Optional[int] = None):
    """GraphDiT.generate up to the integer graphs (RDKit conversion is outside the path).

    diffusion_model.py:252-300.  `noise` = dict(qX0 (B,N,16), qE0 (B,N,N,5), qX (T,B,N,16), qE (T,B,N,N,5))
    indexed so that qX[s] is consumed by the step that produces z_s.  `steps` truncates the loop
    (the last `steps` indices are NOT special: it runs t = T .. T-steps+1) for bounded CPU baselines.
    Returns collapsed ints: X (B,N) with -1 at masked nodes, E (B,N,N) with -1 at masked pairs.
    """
    sd = {k: v.to(dtype) for k, v in sd.items()}
    tb = dit_tables(meta, dtype)
    U = union_transition(tb)
    T = cfg["diffusion_steps"]
    sched = cosine_schedule(T)
    N = tb.max_nodes
    y = torch.where(props == no_label_index, torch.full_like(props, float("nan")), props).to(dtype)
    node_mask = torch.arange(N).unsqueeze(0) < n_nodes.unsqueeze(1)
    X, E = initial_state(tb, node_mask, noise["qX0"].to(dtype), noise["qE0"].to(dtype), dtype)
    Xs = Es = None
    last = 0 if steps is None else max(0, T - steps)
    for s in reversed(range(last, T)):
        X, E, Xs, Es = reverse_step(sd, cfg, tb, U, sched, X, E, node_mask, y, txt.to(dtype), s + 1,
                                    noise["qX"][s].to(dtype), noise["qE"][s].to(dtype))
    Xc = Xs.clone()
    Ec = Es.clone()
    Xc[~node_mask] = -1
    Ec[~(node_mask.unsqueeze(1) & node_mask.unsqueeze(2))] = -1
    return Xc, Ec


# ==============================================================================================
# GIN encoder / predictor (graph_encoder/model.py, graph_predictor/model.py)
# ==============================================================================================
def _segment_sum(x: Tensor, seg: Tensor, B: int) -> Tensor:
    return torch.zeros((B, x.shape[1]), dtype=x.dtype).index_add_(0, seg, x)


def _segment_max(x: Tensor, seg: Tensor, B: int) -> Tensor:
    out = torch.full((B, x.shape[1]), float("-inf"), dtype=x.dtype)
    return out.scatter_reduce(0, seg.unsqueeze(1).expand_as(x), x, reduce="amax", include_self=True)


def _mlp4(sd, p, x, names=("0", "1", "4")):
    """Linear(H,4H) -> LayerNorm(4H) -> GELU -> Linear(4H,out) (dropout is identity in eval)."""
    h = _lin(sd, p + names[0], x)
    h = F.layer_norm(h, (h.shape[-1],), sd[p + names[1] + ".weight"], sd[p + names[1] + ".bias"], LN_EPS)
    return _lin(sd, p + names[2], F.gelu(h))


def _gin_conv(sd, p, h, edge_index, edge_attr):
    """graph_encoder/model.py:156-176 == graph_predictor/model.py:394-423.
    agg_i = sum_{j->i} gelu(h_j + bond_emb[e_ji]); mlp((1+eps) h_i + agg_i)."""
    msg = F.gelu(h[edge_index[0]] + sd[p + "bond_encoder.weight"][edge_attr])
    agg = torch.zeros_like(h).index_add_(0, edge_index[1], msg)
    return _mlp4(sd, p + "mlp.", (1 + sd[p + "eps"]) * h + agg)


def gin_trunk(sd, L: int, x, edge_index, edge_attr, batch, c: Optional[Tensor] = None, predictor: bool = False):
    """Node embeddings after L layers, pooled by sum -> (B,H).

    Encoder: graph_encoder/model.py:124-154 (affine LN, no conditioning).
    Predictor: graph_predictor/model.py:306-351 (non-affine LN, per-graph shift/scale/gate from text).
    The virtual-node update pools the layer INPUT h_list[layer] (model.py:148 / :343).
    """
    B = int(batch[-1].item()) + 1
    H = sd["atom_encoder.weight"].shape[1]
    vn = sd["virtualnode_embedding.weight"][0].unsqueeze(0).expand(B, -1)
    h = sd["atom_encoder.weight"][x]
    if predictor and c is None:
        c = sd["text_dropping.weight"].expand(B, -1)
    for l in range(L):
        h_in = h + vn[batch]
        u = _gin_conv(sd, f"convs.{l}.", h_in, edge_index, edge_attr)
        if predictor:
            mod = _lin(sd, f"adapters.{l}.1", F.silu(c))
            shift, scale, gate = (m[batch] for m in mod.chunk(3, dim=1))
            u = F.layer_norm(u, (H,), None, None, LN_EPS) * (1 + scale) + shift
        else:
            u = F.layer_norm(u, (H,), sd[f"norms.{l}.weight"], sd[f"norms.{l}.bias"], LN_EPS)
        if l < L - 1:
            u = F.gelu(u)
        h = (gate * u if predictor else u) + h_in
        if l < L - 1:
            vn = vn + _mlp4(sd, f"mlp_virtualnode_list.{l}.", _segment_max(h_in, batch, B))
    return _segment_sum(h, batch, B)


def gin_encoder_forward(sd_enc, sd_proj, L, x, edge_index, edge_attr, batch) -> Tensor:
    """GraphCLIP.forward: trunk -> ProjectionHead -> L2 normalise.  graph_encoder/model.py:37-41, 199-205."""
    g = gin_trunk(sd_enc, L, x, edge_index, edge_attr, batch)
    z = _mlp4(sd_proj, "", g, names=("fc1", "norm1", "fc2"))
    return z / z.norm(dim=-1, keepdim=True)


def gin_predictor_forward(sd, L, x, edge_index, edge_attr, batch, c: Optional[Tensor]) -> Tensor:
    """GNNRetrosynthsizer.forward -> logits (B,out_dim).  graph_predictor/model.py:306-353."""
    g = gin_trunk(sd, L, x, edge_index, edge_attr, batch, c, predictor=True)
    return _mlp4(sd, "decoder.", g)


def predictor_topk(logits: Tensor, k: int):
    """Device part of sample_templates: softmax over out_dim, top-k.  graph_predictor/model.py:176-179."""
    return torch.topk(torch.softmax(logits, dim=1), k=k, dim=1)


def cost_mlp_forward(sd, fps: Tensor) -> Tensor:
    """CostMLP.forward (n_layers=1): Linear -> ReLU -> Linear -> log(1+exp).  graph_predictor/model.py:387-391."""
    h = torch.relu(_lin(sd, "layers.0", fps))
    return torch.log(1 + torch.exp(_lin(sd, "layers.3", h)))


# ==============================================================================================
# Counter-based noise (host restatement of the device generator; see llamole_b200/csrc/llb_rng.cuh)
# ==============================================================================================
_PHILOX_M0, _PHILOX_M1 = 0xD2511F53, 0xCD9E8D57
_PHILOX_W0, _PHILOX_W1 = 0x9E3779B9, 0xBB67AE85


def philox4x32(counter: np.ndarray, key: np.ndarray) -> np.ndarray:
    """Philox-4x32-10 (Salmon et al. 2011, the published algorithm).  counter (...,4) uint32, key (...,2) uint32."""
    c = counter.astype(np.uint64).copy()
    k0 = key[..., 0].astype(np.uint64).copy()
    k1 = key[..., 1].astype(np.uint64).copy()
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(_PHILOX_M0) * c[..., 0]
        p1 = np.uint64(_PHILOX_M1) * c[..., 2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & mask
        hi1, lo1 = p1 >> np.uint64(32), p1 & mask
        n0 = (hi1 ^ c[..., 1] ^ k0) & mask
        n2 = (hi0 ^ c[..., 3] ^ k1) & mask
        c = np.stack([n0, lo1, n2, lo0], axis=-1)
        k0 = (k0 + np.uint64(_PHILOX_W0)) & mask
        k1 = (k1 + np.uint64(_PHILOX_W1)) & mask
    return c.astype(np.uint32)


def exp1_from_bits(bits: np.ndarray) -> np.ndarray:
    """Exp(1) variate from 32 random bits: u = (bits + 0.5) * 2^-32 in (0,1), q = -log(u) (fp32)."""
    u = (bits.astype(np.float64) + 0.5) * (1.0 / 4294967296.0)
    return (-np.log(u.astype(np.float32))).astype(np.float32)


def counter_noise(seed: int, stream: int, mol: np.ndarray, pos: np.ndarray, n_classes: int) -> np.ndarray:
    """Noise for category slots 0..n_classes-1 of (molecule `mol`, position `pos`) in draw `stream`.

    counter = (pos, mol, stream, group) with group = class // 4; key = (seed lo, seed hi); the 4 output words
    of one Philox call serve 4 consecutive classes.  `stream` = T for the z_T draw, s for the step producing z_s;
    `pos` = node index i for atoms, N + i*N + j for the pair (i<j).
    """
    mol = np.asarray(mol, dtype=np.uint32)
    pos = np.asarray(pos, dtype=np.uint32)
    shape = np.broadcast(mol, pos).shape
    groups = (n_classes + 3) // 4
    out = np.zeros(shape + (groups * 4,), dtype=np.float32)
    key = np.zeros(shape + (2,), dtype=np.uint32)
    key[..., 0] = np.uint32(seed & 0xFFFFFFFF)
    key[..., 1] = np.uint32((seed >> 32) & 0xFFFFFFFF)
    for gidx in range(groups):
        ctr = np.zeros(shape + (4,), dtype=np.uint32)
        ctr[..., 0] = pos
        ctr[..., 1] = mol
        ctr[..., 2] = np.uint32(stream)
        ctr[..., 3] = np.uint32(gidx)
        out[..., 4 * gidx:4 * gidx + 4] = exp1_from_bits(philox4x32(ctr, key))
    return out[..., :n_classes]
