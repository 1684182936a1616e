"""GraphCLIP / GraphPredictor at GIN hidden widths that are not multiples of 64.

The library stores every H-wide operand with Hp = round_up(H, 64) columns and every 4H-wide one with I = round_up(4H, 64),
zero-padded (csrc/llb_gin.cu, GinLayout).  The CPU tests check the sizing entries and restate the padded analytic LayerNorm
of the node MLP on the host; the GPU tests hold the padded path to the tolerances of the unpadded one against the CPU oracle:
  embeddings : max |d| <= 3e-3 sqrt(768/H) on unit-norm rows (4096 graphs: min cosine > 0.9995)
  logits     : max |d| <= 0.03, rms <= 0.006;  top-k indices equal to a stable sort of the kernel's own logits
"""
import ctypes
import math

import pytest
import torch

from conftest import record_parity
from llamole_b200 import GraphCLIP, GraphPredictor, _cabi, synth

DEV = "cuda:0"


def _round64(v):
    return (v + 63) // 64 * 64


# ------------------------------------------------------------------------------------------------ sizing (CPU)
@pytest.mark.parametrize("predictor", [0, 1])
@pytest.mark.parametrize("H", [1, 37, 300, 1000])
def test_sizes_for_any_hidden_width(H, predictor):
    lib = _cabi.lib()
    cfg = _cabi.GinConfig(H, 3, predictor, 777 if predictor else 0, 768 if predictor else 0)
    packed, ws = ctypes.c_size_t(), ctypes.c_size_t()
    _cabi.check(lib.llb_gin_packed_bytes(ctypes.byref(cfg), ctypes.byref(packed)), "llb_gin_packed_bytes")
    _cabi.check(lib.llb_gin_workspace_bytes(ctypes.byref(cfg), 500, 1000, 20, 1, ctypes.byref(ws)), "llb_gin_workspace_bytes")
    Hp, I = _round64(H), _round64(4 * H)
    # at least the padded node-MLP weights of every layer: (I,Hp) + (Hp,I) bf16/fp16 + the (Hp,Hp) factor
    assert packed.value >= 3 * (2 * I * Hp * 2 + Hp * Hp * 2)
    # at least the fp32 node rows, their bf16 copy and the aggregation output at the padded width, and the (n, I) intermediate
    assert ws.value >= 500 * (Hp * 4 + 2 * Hp * 2 + I * 2)


@pytest.mark.parametrize("H", [0, -64])
def test_sizes_reject_non_positive_width(H):
    lib = _cabi.lib()
    for predictor in (0, 1):
        cfg = _cabi.GinConfig(H, 3, predictor, 777 if predictor else 0, 768 if predictor else 0)
        n = ctypes.c_size_t()
        assert lib.llb_gin_packed_bytes(ctypes.byref(cfg), ctypes.byref(n)) != 0
        assert lib.llb_gin_workspace_bytes(ctypes.byref(cfg), 10, 10, 2, 0, ctypes.byref(n)) != 0


# ------------------------------------------------------------------------------------------------ padded analytic LayerNorm (CPU)
def _bf(t):
    return t.to(torch.bfloat16).to(torch.float32)


def _pack_node_mlp0(W, b, gamma, beta, Hp, I):
    """What llb_gin_pack_weights stores for the node MLP's first linear at a padded width: the weight centred over its 4H TRUE
    output rows, written into (I, Hp); the Cholesky factor of the TRUE (H+1)x(H+1) Gram block written into (Hp, Hp); and
    mlp_stat = [r (Hp entries, 0 past H) | c0 at index Hp | 0, 0, 0]."""
    rows, H = W.shape
    Wc = _bf(W - W.mean(0, keepdim=True))
    bc = b - b.mean()
    Wt = torch.cat([Wc.double(), bc.double()[:, None]], dim=1)
    Rt = torch.linalg.cholesky(Wt.t() @ Wt, upper=True)
    Wc_p = torch.zeros(I, Hp)
    Wc_p[:rows, :H] = Wc
    pad = lambda v: torch.cat([v, torch.zeros(I - rows)])  # noqa: E731
    R_p = torch.zeros(Hp, Hp)
    R_p[:H, :H] = _bf(Rt[:H, :H].float())
    stat = torch.zeros(Hp + 4)
    stat[:H] = Rt[:H, H].float()
    stat[Hp] = float(Rt[H, H] ** 2)
    return Wc_p, pad(bc), pad(gamma), pad(beta), R_p, stat


def test_padded_analytic_layernorm_matches_the_unpadded_scheme():
    L, H = 2, 300
    Hp, I = _round64(H), _round64(4 * H)
    assert (Hp, I) == (320, 1216)
    enc, _ = synth.gin_encoder_state_dicts(L, H, seed=11)
    x, ei, ea, _ = synth.molecular_graphs(64, seed=0)
    pre = "convs.0."
    h = enc["atom_encoder.weight"][x] + enc["virtualnode_embedding.weight"][0]
    msg = torch.nn.functional.gelu(_bf(h)[ei[0]] + enc[pre + "bond_encoder.weight"][ea])
    a = _bf(((1 + enc[pre + "eps"]) * h).index_add(0, ei[1], msg))          # the bf16 A operand, true width
    a_p = torch.cat([a, torch.zeros(a.shape[0], Hp - H)], dim=1)           # ... and as the kernels hold it (zero-padded)
    W, b = enc[pre + "mlp.0.weight"], enc[pre + "mlp.0.bias"]
    gamma, beta = enc[pre + "mlp.1.weight"], enc[pre + "mlp.1.bias"]
    Wc_p, bc_p, g_p, bt_p, R_p, stat = _pack_node_mlp0(W, b, gamma, beta, Hp, I)
    # c0 sits at index Hp, not H: the statistics epilogue adds r_k to every one of its Hp columns
    assert stat[Hp] > 0 and bool((stat[H:Hp] == 0).all())
    # unpadded scheme (tests/test_analytic_ln_numerics.py)
    R, r, c0 = R_p[:H, :H], stat[:H], float(stat[Hp])
    q_ref = ((a @ R.t() + r) ** 2).sum(1) + c0
    # padded: EpiRowSq over Hp columns with r from stat[:Hp], c0 from stat[Hp]; EpiLnGelu over I columns with 1 / 4H
    q = ((a_p @ R_p.t() + stat[:Hp]) ** 2).sum(1) + stat[Hp]
    assert torch.allclose(q, q_ref, rtol=1e-6, atol=0)
    rstd = torch.rsqrt(q / (4 * H) + 1e-5)
    rstd_ref = torch.rsqrt(q_ref / (4 * H) + 1e-5)
    assert torch.allclose(rstd, rstd_ref, rtol=1e-6, atol=0)
    out = torch.nn.functional.gelu(rstd[:, None] * ((a_p @ Wc_p.t()) * g_p + bc_p * g_p) + bt_p)
    Wc = Wc_p[:4 * H, :H]
    bc = bc_p[:4 * H]
    out_ref = torch.nn.functional.gelu(rstd_ref[:, None] * ((a @ Wc.t()) * gamma + bc * gamma) + beta)
    assert bool((out[:, 4 * H:] == 0).all())                                  # padded columns exactly 0
    assert float((out[:, :4 * H] - out_ref).abs().max()) < 1e-5
    # and the statistics are those of the true 4H-wide pre-activation
    z = a @ Wc.t() + bc
    rel = ((rstd - torch.rsqrt(z.var(1, unbiased=False) + 1e-5)) / rstd).abs().max()
    assert float(rel) < 2e-3


# ------------------------------------------------------------------------------------------------ GPU vs the oracle
def _stats(a, b):
    d = (a.double() - b.double()).abs()
    return float(d.max()), float(d.pow(2).mean().sqrt())


def _ragged_batch(seed):
    """Single atoms, an edge-less fragment, small molecules and a 200-node graph in one batch: (nodes, with edges)."""
    spec = [(1, True), (17, True), (5, False), (200, True), (1, True), (2, True), (3, False), (64, True), (1, True)]
    xs, eis, eas, bs = [], [], [], []
    base = 0
    for gi, (n, edges) in enumerate(spec):
        x, ei, ea, _ = synth.molecular_graphs(1, seed=seed + gi, min_nodes=n, max_nodes=n)
        xs.append(x)
        bs.append(torch.full((n,), gi, dtype=torch.int64))
        if edges:
            eis.append(ei + base)
            eas.append(ea)
        base += n
    return torch.cat(xs), torch.cat(eis, 1), torch.cat(eas), torch.cat(bs)


def _encoder(L, H, seed):
    enc, proj = synth.gin_encoder_state_dicts(L, H, seed=seed)
    g = GraphCLIP(L, H, 0.0, {})
    g.molecule_encoder.load_state_dict(enc)
    g.molecule_projection.load_state_dict(proj)
    return g.to(DEV), enc, proj


@pytest.mark.gpu
@pytest.mark.parametrize("L", [2, 5])
@pytest.mark.parametrize("H", [37, 200, 300, 1000])
def test_encoder_any_width_vs_oracle(H, L):
    from oracle import llamole_oracle as O

    g, enc, proj = _encoder(L, H, seed=21)
    x, ei, ea, b = _ragged_batch(seed=H + L)
    B = int(b[-1]) + 1
    with torch.no_grad():
        ref = O.gin_encoder_forward(enc, proj, L, x, ei, ea, b)
        ref_pooled = O.gin_trunk(enc, L, x, ei, ea, b)
    eng = g.engine()
    eng.bind(x, ei, ea, b)
    emb, pooled = eng.encoder_forward(want_pooled=True)
    torch.cuda.synchronize()
    assert emb.shape == (B, H) and pooled.shape == (B, H)
    assert bool(torch.isfinite(emb).all()) and bool(torch.isfinite(pooled).all())
    mx, rms = _stats(emb.cpu(), ref)
    mx_p, rms_p = _stats(pooled.cpu(), ref_pooled)
    rel_p = rms_p / float(ref_pooled.double().pow(2).mean().sqrt())
    record_parity(f"gin_encoder_any_width[H={H},L={L}]", max_abs=mx, rms=rms, pooled_max_abs=mx_p, pooled_rel_rms=rel_p)
    print(f"\n[parity] GIN encoder H={H} L={L}: max|d|={mx:.2e} rms={rms:.2e}; pooled max|d|={mx_p:.3e} rel rms={rel_p:.2e}")
    assert mx <= 3e-3 * math.sqrt(768 / H), (H, L, mx)
    assert rel_p <= 1e-2, (H, L, rel_p)
    # the module entry: same rows, unit norm, and the parameters' dtype
    out = g(x.to(DEV), ei.to(DEV), ea.to(DEV), b.to(DEV))
    assert out.shape == (B, H) and out.dtype == torch.float32
    assert torch.allclose(out.norm(dim=-1).cpu(), torch.ones(B), atol=1e-4)
    gb = g.to(torch.bfloat16)
    out_b = gb(x.to(DEV), ei.to(DEV), ea.to(DEV), b.to(DEV))
    assert out_b.shape == (B, H) and out_b.dtype == torch.bfloat16


@pytest.mark.gpu
def test_encoder_padded_width_at_the_benchmark_shape():
    """H = 300 (OGB's default GIN width, padded to 320 / 1216), L = 5 over the benchmark's 4096 graphs: the padded operands
    run through the CTA-pair GEMM."""
    from oracle import llamole_oracle as O

    L, H = 5, 300
    g, enc, proj = _encoder(L, H, seed=11)
    x, ei, ea, b = synth.molecular_graphs(4096, seed=0)
    k2 = _cabi.kernel_launches(_cabi.KERN_GEMM_2CTA)
    eng = g.engine()
    eng.bind(x, ei, ea, b)
    emb = eng.encoder_forward()
    torch.cuda.synchronize()
    assert _cabi.kernel_launches(_cabi.KERN_GEMM_2CTA) > k2, "the node MLP must have run on the CTA-pair GEMM"
    with torch.no_grad():
        ref = O.gin_encoder_forward(enc, proj, L, x, ei, ea, b)
    mx, rms = _stats(emb.cpu(), ref)
    cos = float(torch.nn.functional.cosine_similarity(emb.cpu().double(), ref.double(), dim=1).min())
    record_parity("gin_encoder_4096_graphs_H300_L5", nodes=int(x.numel()), edges=int(ea.numel()), max_abs=mx, rms=rms, min_cosine=cos)
    print(f"\n[parity] GIN encoder H=300 L=5, 4096 graphs / {x.numel()} nodes: max|d|={mx:.2e} rms={rms:.2e} min cos={cos:.6f}")
    assert bool(torch.isfinite(emb).all())
    assert mx <= 3e-3 * math.sqrt(768 / H) and cos > 0.9995, (mx, rms, cos)


def _predictor(L, H, D, seed):
    sd = synth.gin_predictor_state_dict(L, H, D, seed=seed)
    gp = GraphPredictor(L, H, 0.0, D, {}, {})
    gp.predictor.load_state_dict(sd)
    return gp.to(DEV), sd


def _check_topk_against_own_logits(gp, inputs, c, lg, k):
    """top-k indices must be a stable sort (value descending, ties to the lower index) of the kernel's own logits"""
    probs, idx = gp.topk_templates(*inputs, c, k)
    torch.cuda.synchronize()
    order = torch.sort(lg, dim=1, descending=True, stable=True).indices[:, :k]
    p_own = torch.softmax(lg.double(), dim=1)
    assert torch.allclose(probs.cpu().double(), torch.gather(p_own, 1, order), rtol=2e-4, atol=1e-7)
    return float((idx.cpu().long() == order).float().mean())


@pytest.mark.gpu
@pytest.mark.parametrize("H", [37, 300])
def test_predictor_any_width_vs_oracle(H):
    from oracle import llamole_oracle as O

    L, D = 2, 777
    gp, sd = _predictor(L, H, D, seed=5)
    x, ei, ea, b = _ragged_batch(seed=3)
    B = int(b[-1]) + 1
    c = synth.text_conditions(B, seed=1)
    inputs = tuple(t.to(DEV) for t in (x, ei, ea, b))
    worst = (0.0, 0.0)
    for cond in (c, None):
        with torch.no_grad():
            ref = O.gin_predictor_forward(sd, L, x, ei, ea, b, cond)
        got = gp(*inputs, None if cond is None else cond.to(DEV))
        torch.cuda.synchronize()
        assert got.shape == (B, D)
        mx, rms = _stats(got.cpu(), ref)
        worst = (max(worst[0], mx), max(worst[1], rms))
        print(f"\n[parity] GIN predictor H={H} ({'text' if cond is not None else 'dropped'}): max|d|={mx:.4f} rms={rms:.5f} (std {float(ref.std()):.2f})")
        assert mx <= 0.03 and rms <= 0.006, (H, mx, rms)
    lg = gp(*inputs, c.to(DEV)).float().cpu()
    same = [_check_topk_against_own_logits(gp, inputs, c.to(DEV), lg, k) for k in (1, 50, D)]
    record_parity(f"gin_predictor_any_width[H={H},D={D}]", logits_max_abs=worst[0], logits_rms=worst[1], topk_positions_equal=min(same))
    assert min(same) == 1.0, same


@pytest.mark.gpu
@pytest.mark.parametrize("H", [37, 300])
def test_predictor_any_width_fused_head(H):
    """16 384 templates over 512 graphs: the fused head + softmax + top-k runs with a padded K (I = round_up(4H, 64))."""
    from oracle import llamole_oracle as O

    L, D, k = 2, 16384, 50
    gp, sd = _predictor(L, H, D, seed=13)
    x, ei, ea, b = synth.molecular_graphs(512, seed=9)
    c = synth.text_conditions(512, seed=4)
    inputs = tuple(t.to(DEV) for t in (x, ei, ea, b))
    got = gp(*inputs, c.to(DEV))
    torch.cuda.synchronize()
    with torch.no_grad():
        ref = O.gin_predictor_forward(sd, L, x, ei, ea, b, c)
    mx, rms = _stats(got.cpu(), ref)
    print(f"\n[parity] GIN predictor H={H} D={D}, 512 graphs: logits max|d|={mx:.4f} rms={rms:.5f}")
    assert mx <= 0.03 and rms <= 0.006, (H, mx, rms)
    same = _check_topk_against_own_logits(gp, inputs, c.to(DEV), got.float().cpu(), k)
    stats = gp.engine().head_stats()
    record_parity(f"gin_predictor_fused_head[H={H},D={D}]", logits_max_abs=mx, logits_rms=rms, topk_positions_equal=same, **stats)
    print(f"[parity] top-{k}: {same:.5f} of positions equal a stable sort of the kernel's logits; head {stats}")
    assert stats["fused_rows"] > 0
    assert same > 0.999, same
