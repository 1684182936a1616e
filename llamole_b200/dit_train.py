"""GraphDiT.forward -- the SFT training loss of the graph decoder (diffusion_model.py:148-250, TrainLossDiscrete :402-438).

The noisy state, the conditions and the cross-entropy always run here in eager PyTorch.  The denoiser runs on the sm_100a
kernels (GraphDiT.denoise_on_device, differentiable with respect to the condition vector) when GraphDiT.device_denoiser_ok()
holds -- a frozen decoder on a B200 -- and as the eager `denoiser_forward` below otherwise.  This module exists so that
the drop-in class keeps the reference's whole surface: `GraphLLMForCausalMLM.forward` calls
`graph_decoder(x, edge_index, edge_attr, graph_batch, properties, text_embedding, no_label_index)` during SFT
(modeling_llamole.py:371-379) and must get the same scalar loss, differentiable with respect to the denoiser's parameters
and to `text_embedding`.  It is plain eager PyTorch on whatever device the module lives on, written from the reference's
semantics (no reference import, no oracle import), and it consumes torch's global RNG in the reference's order -- timestep
draw, the two multinomial noise draws, then per property the condition-dropout uniforms and the N(0,1) embedding noise, then
the text-dropout uniforms -- so that with the same `torch.manual_seed` it reproduces the reference's loss
(checked against the verbatim module when it was written; the repository holds no copy of that module).

Reference behaviours kept on purpose (they define the loss value):
  * padded atom pairs carry the "no bond" class after `encode_no_edge` (diffusion_utils.py:128-141), so they DO enter the bond
    cross-entropy (against logits that `PlaceHolder.mask` zeroed: a constant log 5 each);
  * atoms outside the 16 active types give an all-zero row and drop out of the atom loss;
  * the noisy state is sampled from  [X | E row] @ (abar_t I + (1 - abar_t) U)  over the JOINT 266-vector (:212-216);
  * in training mode every property embedding gets N(0,1) noise added and conditions are dropped with probability
    `drop_condition` (conditions.py:84-96, 116-118); `lowest_t` is 0 in training mode, 1 in eval mode (:199).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

LN_EPS = 1e-5


def union_transition(x_marg, e_marg, xe, ex, n: int) -> torch.Tensor:
    """(d0,d0) joint marginal transition U, d0 = 16 + 5 n (MarginalTransition.get_union_transition, diffusion_utils.py:299-306)."""
    u_x = x_marg.unsqueeze(0).expand(x_marg.numel(), -1)
    u_e = e_marg.unsqueeze(0).expand(e_marg.numel(), -1).repeat(n, n)
    return torch.cat([torch.cat([u_x, xe.repeat(1, n)], dim=1), torch.cat([ex.repeat(n, 1), u_e], dim=1)], dim=0)


def to_dense(data_x, edge_index, data_edge_attr, batch, max_nodes: int):
    """PyG batch -> dense one-hot X (B,N,dx), E (B,N,N,de) with the no-edge class encoded, node_mask (B,N)
    (diffusion_utils.py:111-141: to_dense_batch, remove_self_loops, to_dense_adj, encode_no_edge)."""
    B = int(batch.max().item()) + 1 if batch.numel() else 0
    counts = torch.bincount(batch, minlength=B)
    first = torch.cumsum(counts, 0) - counts
    pos = torch.arange(batch.numel(), device=batch.device) - first[batch]
    fits = pos < max_nodes    # torch_geometric 2.6.1 drops the nodes (and their edges) beyond max_num_nodes without an error
    X = data_x.new_zeros((B, max_nodes, data_x.shape[-1]))
    X[batch[fits], pos[fits]] = data_x[fits]
    node_mask = torch.zeros((B, max_nodes), dtype=torch.bool, device=batch.device)
    node_mask[batch[fits], pos[fits]] = True
    keep = (edge_index[0] != edge_index[1]) & fits[edge_index[0]] & fits[edge_index[1]]
    src, dst, ea = edge_index[0][keep], edge_index[1][keep], data_edge_attr[keep]
    E = data_edge_attr.new_zeros((B, max_nodes, max_nodes, data_edge_attr.shape[-1]))
    E.index_put_((batch[src], pos[src], pos[dst]), ea, accumulate=True)     # duplicate edges add, like to_dense_adj
    no_edge = E.sum(dim=3) == 0
    E[..., 0] = torch.where(no_edge, torch.ones_like(E[..., 0]), E[..., 0])
    diag = torch.eye(max_nodes, dtype=torch.bool, device=E.device)
    E[:, diag] = 0
    return X, E, node_mask


def _lin(mod, x):
    return F.linear(x, mod.weight, mod.bias)


def _conditions(den, y, txt, t, train: bool, unconditioned: bool, drop_prob: float):
    """c = t_embedder(t) + y_embedder(y) + txt_embedder(txt)   (transformer.py:98-101; conditions.py:53-58, 76-98, 108-123)."""
    H = den.x_embedder[0].weight.shape[0]
    half = 128
    freqs = torch.exp(-math.log(10000) * torch.arange(half, dtype=torch.float32) / half).to(t.device)
    args = t.view(-1)[:, None].float() * freqs[None]
    tf = torch.cat([torch.cos(args), torch.sin(args)], dim=-1).to(den.t_embedder.mlp[0].weight.dtype)
    c = _lin(den.t_embedder.mlp[2], F.silu(_lin(den.t_embedder.mlp[0], tf)))
    emb_sum = 0
    for d in range(y.shape[1]):
        label = y[:, d]
        if unconditioned:
            drop = torch.ones_like(label).bool()
        else:
            drop = torch.isnan(label)
            if train:
                drop = drop | (torch.rand(label.shape).type_as(y) < drop_prob)
        emb = torch.zeros((label.shape[0], H)).type_as(y)
        mlp = den.y_embedder.mlps[d]
        out = F.linear(torch.softmax(_lin(mlp[0], label.unsqueeze(1)[~drop]), dim=1), mlp[2].weight)
        emb = emb.index_put((torch.nonzero(~drop).squeeze(1),), out.type_as(emb))
        emb = emb + drop.unsqueeze(1).type_as(emb) * den.y_embedder.embedding_drop.weight[d]
        if train:
            emb = emb + torch.randn_like(emb)
        emb_sum = emb_sum + emb
    if unconditioned:
        drop = torch.ones(txt.shape[0]).bool().to(txt.device)
    else:
        drop = torch.isnan(txt.sum(dim=1))
        if train:
            drop = drop | (torch.rand(txt.shape[0]).type_as(txt) < drop_prob)
    temb = torch.zeros((txt.shape[0], H)).type_as(txt)
    temb = temb.index_put((torch.nonzero(~drop).squeeze(1),), _lin(den.txt_embedder.linear, txt[~drop]).type_as(temb))
    temb = temb + drop.unsqueeze(1).type_as(temb) * den.txt_embedder.embedding_drop.weight[0]
    return c + emb_sum + temb


def denoiser_forward(den, heads: int, X_in, E_in, node_mask, y, txt, t, train: bool, unconditioned: bool, drop_prob: float):
    """Transformer.forward (transformer.py:93-108) on the parameter-holder module tree `den`; returns masked logits."""
    B, N, dx = X_in.shape
    x = F.linear(torch.cat([X_in, E_in.reshape(B, N, -1)], dim=-1), den.x_embedder[0].weight)
    H = x.shape[-1]
    x = F.layer_norm(x, (H,), den.x_embedder[1].weight, den.x_embedder[1].bias, LN_EPS)
    c = _conditions(den, y, txt, t, train, unconditioned, drop_prob)
    dh = H // heads
    allow = node_mask[:, None, :, None] & node_mask[:, None, None, :]
    allow = (allow | (allow.sum(dim=-1, keepdim=True) == 0)).expand(-1, heads, N, N)     # fully masked queries see everything
    for blk in den.blocks:
        mod = F.softsign(_lin(blk.adaLN_modulation[2], F.silu(_lin(blk.adaLN_modulation[0], c))))
        sh_a, sc_a, g_a, sh_m, sc_m, g_m = (m.unsqueeze(1) for m in mod.chunk(6, dim=1))
        qkv = _lin(blk.attn.qkv, x).reshape(B, N, 3, heads, dh).permute(2, 0, 3, 1, 4)
        q = F.layer_norm(qkv[0], (dh,), blk.attn.q_norm.weight, blk.attn.q_norm.bias, LN_EPS)
        k = F.layer_norm(qkv[1], (dh,), blk.attn.k_norm.weight, blk.attn.k_norm.bias, LN_EPS)
        a = F.scaled_dot_product_attention(q, k, qkv[2], attn_mask=allow)
        a = _lin(blk.attn.proj, a.transpose(1, 2).reshape(B, N, H))
        x = x + g_a * (F.layer_norm(a, (H,), None, None, LN_EPS) * (1 + sc_a) + sh_a)
        m = _lin(blk.mlp.fc2, F.gelu(_lin(blk.mlp.fc1, x)))
        x = x + g_m * (F.layer_norm(m, (H,), None, None, LN_EPS) * (1 + sc_m) + sh_m)
    ol = den.output_layer
    out = _lin(ol.xedecoder.fc2, F.gelu(_lin(ol.xedecoder.fc1, x)))
    d0 = out.shape[-1]
    shift, scale = (m.unsqueeze(1) for m in _lin(ol.adaLN_modulation[2], F.silu(_lin(ol.adaLN_modulation[0], c))).chunk(2, dim=1))
    out = F.layer_norm(out, (d0,), None, None, LN_EPS) * (1 + scale) + shift
    Xo = X_in + out[:, :, :dx]
    Eo = E_in + out[:, :, dx:].reshape(B, N, N, -1)
    both_invalid = (~node_mask)[:, :, None] & (~node_mask)[:, None, :]
    diag = torch.eye(N, dtype=torch.bool, device=Eo.device).unsqueeze(0)
    Eo = Eo.masked_fill((both_invalid | diag)[..., None], 0)
    Eo = 0.5 * (Eo + Eo.transpose(1, 2))
    xm = node_mask.unsqueeze(-1)
    return Xo * xm, Eo * xm.unsqueeze(2) * xm.unsqueeze(1)


def sample_noisy_state(model, X, E, node_mask):
    """apply_noise (diffusion_model.py:194-250): draw t per molecule, sample z_t ~ [X | E] Q_t_bar, one-hot, mask."""
    dt = model.model_dtype
    bs, n, _ = X.shape
    lowest_t = 0 if model.training else 1
    t_int = torch.randint(lowest_t, model.T + 1, size=(bs, 1), device=X.device).to(dt)
    t_float = t_int / model.T
    idx = torch.round(t_float * model.T).long()
    abar_t = model.alphas_bar.to(X.device).type_as(t_float)[idx].view(bs, 1, 1)
    U = union_transition(model.x_marginals.to(dt), model.e_marginals.to(dt), model.xe_conditions.to(dt), model.ex_conditions.to(dt), n).to(X.device)
    d0 = U.shape[0]
    Qtb = abar_t * torch.eye(d0, device=X.device, dtype=U.dtype).unsqueeze(0) + (1 - abar_t) * U
    prob_all = torch.cat([X, E.reshape(bs, n, -1)], dim=-1) @ Qtb
    probX = prob_all[:, :, :model.Xdim_output]
    probE = prob_all[:, :, model.Xdim_output:].reshape(bs, n, n, -1)
    # sample_discrete_features (diffusion_utils.py:376-413)
    probX = probX.clone()
    probX[~node_mask] = 1 / probX.shape[-1]
    probX = probX.reshape(bs * n, -1).clamp_min(1e-5)
    probX = probX / probX.sum(dim=-1, keepdim=True)
    X_t = probX.multinomial(1).reshape(bs, n)
    inverse_edge_mask = ~(node_mask.unsqueeze(1) * node_mask.unsqueeze(2))
    diag_mask = torch.eye(n, device=X.device).unsqueeze(0).expand(bs, -1, -1)
    probE = probE.clone()
    probE[inverse_edge_mask] = 1 / probE.shape[-1]
    probE[diag_mask.bool()] = 1 / probE.shape[-1]
    probE = probE.reshape(bs * n * n, -1).clamp_min(1e-5)
    probE = probE / probE.sum(dim=-1, keepdim=True)
    E_t = probE.multinomial(1).reshape(bs, n, n)
    E_t = torch.triu(E_t, diagonal=1)
    E_t = E_t + torch.transpose(E_t, 1, 2)
    X_t = F.one_hot(X_t, num_classes=model.Xdim_output)
    E_t = F.one_hot(E_t, num_classes=model.Edim_output)
    xm = node_mask.unsqueeze(-1)
    return (X_t * xm), (E_t * xm.unsqueeze(2) * xm.unsqueeze(1)), t_float


def train_loss(lambda_train, pred_X, pred_E, true_X, true_E):
    """TrainLossDiscrete.forward (diffusion_model.py:409-438): CE over rows whose true vector is non-zero."""
    true_X = true_X.reshape(-1, true_X.size(-1))
    true_E = true_E.reshape(-1, true_E.size(-1))
    pred_X = pred_X.reshape(-1, pred_X.size(-1))
    pred_E = pred_E.reshape(-1, pred_E.size(-1))
    mask_X = (true_X != 0.0).any(dim=-1)
    mask_E = (true_E != 0.0).any(dim=-1)
    loss_X = F.cross_entropy(pred_X[mask_X, :], torch.argmax(true_X[mask_X, :], dim=-1), reduction="mean")
    loss_E = F.cross_entropy(pred_E[mask_E, :], torch.argmax(true_E[mask_E, :], dim=-1), reduction="mean")
    return lambda_train[0] * loss_X + lambda_train[1] * loss_E


def graphdit_loss(model, x, edge_index, edge_attr, graph_batch, properties, text_embedding, no_label_index):
    """GraphDiT.forward (diffusion_model.py:148-172)."""
    dt = model.model_dtype
    properties = torch.where(properties == no_label_index, float("nan"), properties)
    data_x = F.one_hot(x, num_classes=118).to(dt)[:, model.active_index.to(x.device)]
    data_edge_attr = F.one_hot(edge_attr, num_classes=5).to(dt)
    X, E, node_mask = to_dense(data_x, edge_index, data_edge_attr, graph_batch, model.max_n_nodes)
    X_t, E_t, t = sample_noisy_state(model, X, E, node_mask)
    mc = model.model_config
    den, train, drop = model.denoiser, model.denoiser.training, float(mc.drop_condition)
    y, txt = properties.to(dt).clone(), text_embedding.to(dt)
    if model.device_denoiser_ok():
        # conditions in PyTorch (the token embedding before them draws nothing, so the RNG order is the eager path's), the
        # denoiser c -> logits on the device
        c = _conditions(den, y, txt, t, train, False, drop)
        pX, pE = model.denoise_on_device(X_t.to(dt), E_t.to(dt), node_mask, c)
    else:
        pX, pE = denoiser_forward(den, int(mc.num_heads), X_t.to(dt), E_t.to(dt), node_mask, y, txt, t, train, False, drop)
    return train_loss(mc.lambda_train, pX, pE, X, E)
