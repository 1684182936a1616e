"""GraphCLIP.forward differentiable with respect to every parameter (csrc/llb_gin_grad.cu, llb_gin_encoder_backward).

Reference gradients come from torch autograd through oracle.gin_encoder_forward in fp64 on the CPU, with loss = <emb, G> for a
fixed random G.  The accuracy gate is the reference's own precision in the loader's compute dtype: for every parameter the
relative L2 error of its gradient against fp64 must not exceed that of the same oracle run in bf16 on the same inputs (the
single-number eps gradients are gated together as one vector over the layers), and every row that carries gradient (norm >= 10 %
of the largest row) must have a cosine >= 0.8 against fp64.  The row floor is set by the reference's own precision: the bf16
oracle's rows of the layer-0 weight gradients at L = 5 reach cosines of 0.86 (every result is printed next to the bf16 oracle's).
"""
import ctypes
import os
import subprocess
import sys
import warnings

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from conftest import ROOT, record_parity
from llamole_b200 import GraphCLIP, _cabi, synth

DEV = "cuda:0"


# ------------------------------------------------------------------------------------------------ helpers
def _G(B, H, seed):
    return torch.randn(B, H, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)


def oracle_grads(enc, proj, L, graph, G, dtype):
    """{("enc"|"proj", key): dL/dparam} for loss = <emb, G> through the oracle, everything in `dtype`; returned as fp64."""
    from oracle import llamole_oracle as O

    e = {k: v.detach().to(dtype).requires_grad_(True) if v.is_floating_point() else v for k, v in enc.items()}
    p = {k: v.detach().to(dtype).requires_grad_(True) for k, v in proj.items()}
    (O.gin_encoder_forward(e, p, L, *graph) * G.to(dtype)).sum().backward()
    out = {("enc", k): v.grad.double() for k, v in e.items() if v.is_floating_point()}
    out.update({("proj", k): v.grad.double() for k, v in p.items()})
    return out


def _rows(t):
    return t.reshape(1, -1) if t.dim() < 2 else t


def _stack_eps(d):
    """the per-layer eps gradients are single numbers: gated together, as one vector over the layers"""
    eps = sorted(k for k in d if k[1].endswith(".eps"))
    out = {k: v for k, v in d.items() if k not in eps}
    if eps:
        out[("enc", "convs.*.eps")] = torch.stack([d[k].reshape(()).double().cpu() for k in eps])
    return out


def _metrics(got, ref64, ref16):
    got, ref64, ref16 = got.double().cpu(), ref64.double(), ref16.double()
    nrm = float(ref64.norm())
    if nrm == 0.0:
        return {"zero": float(got.abs().max()) == 0.0}
    g2, r2, b2 = _rows(got), _rows(ref64), _rows(ref16)
    rn = r2.norm(dim=1)
    keep = rn >= 0.1 * float(rn.max())   # rows that carry gradient
    return {"err": float((got - ref64).norm()) / nrm, "err16": float((ref16 - ref64).norm()) / nrm,
            "cos": float(F.cosine_similarity(got.reshape(1, -1), ref64.reshape(1, -1)).item()),
            "row_cos": float(F.cosine_similarity(g2[keep], r2[keep], dim=1).min()),
            "row_cos16": float(F.cosine_similarity(b2[keep], r2[keep], dim=1).min())}


def _gate(case, got, ref64, ref16):
    """per parameter: rel L2 <= the bf16 oracle's, and per-row cosine >= 0.8 on the rows that carry at least 10 % of the largest
    row's norm (rows far below that are noise-dominated in the bf16 oracle too)"""
    got, ref64, ref16 = _stack_eps(got), _stack_eps(ref64), _stack_eps(ref16)
    res = {"%s.%s" % k: _metrics(got[k], ref64[k], ref16[k]) for k in ref64}
    bad = []
    for name, m in res.items():
        if "zero" in m:
            if not m["zero"]:
                bad.append((name, "reference gradient is 0, ours is not"))
            continue
        print(f"  {case} {name}: rel L2 {m['err']:.3e} (bf16 oracle {m['err16']:.3e}), cos {m['cos']:.6f}, "
              f"min row cos {m['row_cos']:.5f} (bf16 oracle {m['row_cos16']:.5f})")
        if not (m["err"] <= m["err16"] and m["row_cos"] >= 0.8):
            bad.append((name, m))
    full = [m for m in res.values() if "err" in m]
    worst = max(res, key=lambda k: res[k].get("err", 0.0))
    record_parity(case, worst_param=worst, worst_rel_l2=res[worst]["err"], its_bf16_oracle=res[worst]["err16"],
                  min_cos=min(m["cos"] for m in full), min_row_cos=min(m["row_cos"] for m in full))
    print(f"\n[parity] {case}: worst rel L2 {res[worst]['err']:.3e} ({worst}, bf16 oracle {res[worst]['err16']:.3e}), "
          f"min cos {min(m['cos'] for m in full):.6f}, min row cos {min(m['row_cos'] for m in full):.5f}")
    assert not bad, bad


def _encoder(L, H, seed, dtype=torch.float32):
    enc, proj = synth.gin_encoder_state_dicts(L, H, seed=seed)
    g = GraphCLIP(L, H, 0.0, {})
    g.molecule_encoder.load_state_dict(enc)
    g.molecule_projection.load_state_dict(proj)
    return g.to(dtype).to(DEV), enc, proj


def _gpu_grads(g, graph, G):
    for p in g.parameters():
        p.grad = None
    emb = g(*(t.to(DEV) for t in graph))
    assert emb.grad_fn is not None
    (emb.float() * G.to(DEV, torch.float32)).sum().backward()
    out = {("enc", k): p.grad for k, p in g.molecule_encoder.named_parameters()}
    out.update({("proj", k): p.grad for k, p in g.molecule_projection.named_parameters()})
    return out


def _ragged_batch(seed):
    """single atoms, an edge-less fragment, small molecules and a 200-node graph (as tests/test_gin_any_width.py)"""
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


def _star_batch():
    """star graphs with identical leaves: the leaves are automorphic, so the virtual node's max-pool has exact ties"""
    xs, eis, eas, bs = [], [], [], []
    base = 0
    for gi, (leaves, centre, leaf, bond) in enumerate([(3, 5, 5, 0), (4, 6, 7, 1), (6, 5, 8, 0), (2, 14, 7, 2), (5, 6, 16, 0)]):
        xs.append(torch.tensor([centre] + [leaf] * leaves))
        src = torch.arange(1, leaves + 1) + base
        ctr = torch.full((leaves,), base)
        eis.append(torch.stack([torch.cat([src, ctr]), torch.cat([ctr, src])]))
        eas.append(torch.full((2 * leaves,), bond))
        bs.append(torch.full((leaves + 1,), gi))
        base += leaves + 1
    return torch.cat(xs), torch.cat(eis, 1), torch.cat(eas), torch.cat(bs)


# ------------------------------------------------------------------------------------------------ CPU
def test_encoder_saved_sizes():
    lib = _cabi.lib()
    n = ctypes.c_size_t()
    for H in (37, 300, 768):
        enc = _cabi.GinConfig(H, 5, 0, 0, 0)
        _cabi.check(lib.llb_gin_encoder_saved_bytes(ctypes.byref(enc), 3000, 6000, 100, ctypes.byref(n)), "llb_gin_encoder_saved_bytes")
        Hp = (H + 63) // 64 * 64
        assert n.value > 3000 * Hp * (5 * 4 + 5 * 2)   # at least every layer's fp32 input and bf16 aggregation
        # the predictor's c-only entries keep rejecting encoder configs
        assert lib.llb_gin_grad_packed_bytes(ctypes.byref(enc), ctypes.byref(n)) != 0
        assert lib.llb_gin_saved_bytes(ctypes.byref(enc), 10, 10, 2, ctypes.byref(n)) != 0
    for H in (0, -64):
        assert lib.llb_gin_encoder_saved_bytes(ctypes.byref(_cabi.GinConfig(H, 3, 0, 0, 0)), 10, 10, 2, ctypes.byref(n)) != 0
    pred = _cabi.GinConfig(256, 3, 1, 777, 768)
    assert lib.llb_gin_encoder_saved_bytes(ctypes.byref(pred), 10, 10, 2, ctypes.byref(n)) != 0
    enc = _cabi.GinConfig(256, 3, 0, 0, 0)
    assert lib.llb_gin_encoder_saved_bytes(ctypes.byref(enc), 0, 10, 2, ctypes.byref(n)) != 0
    small, big = ctypes.c_size_t(), ctypes.c_size_t()
    _cabi.check(lib.llb_gin_encoder_saved_bytes(ctypes.byref(enc), 500, 1000, 20, ctypes.byref(small)), "llb_gin_encoder_saved_bytes")
    _cabi.check(lib.llb_gin_encoder_saved_bytes(ctypes.byref(enc), 1000, 2000, 20, ctypes.byref(big)), "llb_gin_encoder_saved_bytes")
    assert big.value > small.value
    for name in ("llb_gin_encoder_saved_bytes", "llb_gin_encoder_forward_saved", "llb_gin_encoder_backward"):
        assert name in _cabi.SIGNATURES


def test_oracle_grads_match_finite_differences():
    """the fp64 reference the GPU tests compare against is the derivative of the oracle's loss"""
    from oracle import llamole_oracle as O

    L, H = 2, 4
    enc, proj = synth.gin_encoder_state_dicts(L, H, seed=3)
    enc = {k: v.double() if v.is_floating_point() else v for k, v in enc.items()}
    proj = {k: v.double() for k, v in proj.items()}
    graph = synth.molecular_graphs(3, seed=2, min_nodes=4, max_nodes=7)
    G = _G(3, H, seed=4)
    grads = oracle_grads(enc, proj, L, graph, G, torch.float64)

    def f(e, p):
        with torch.no_grad():
            return float((O.gin_encoder_forward(e, p, L, *graph) * G).sum())

    h = 1e-6
    gen = torch.Generator().manual_seed(0)
    for (part, key), gr in grads.items():
        sd = enc if part == "enc" else proj
        flat = sd[key].view(-1)
        idx = torch.randperm(flat.numel(), generator=gen)[:6]
        for i in idx.tolist():
            keep = float(flat[i])
            flat[i] = keep + h
            fp = f(enc, proj)
            flat[i] = keep - h
            fm = f(enc, proj)
            flat[i] = keep
            fd = (fp - fm) / (2 * h)
            assert abs(fd - float(gr.view(-1)[i])) <= 1e-5 * max(1.0, abs(fd)), (key, i, fd, float(gr.view(-1)[i]))


# ------------------------------------------------------------------------------------------------ GPU: gradients against the oracle
def _case_fused(expect_fused):
    L, H, B = 5, 768, 100
    g, enc, proj = _encoder(L, H, seed=13)
    graph = synth.molecular_graphs(B, seed=7)
    assert graph[0].numel() > 2000
    G = _G(B, H, seed=5)
    k0 = _cabi.kernel_launches(_cabi.KERN_GIN_FUSED_MLP)
    got = _gpu_grads(g, graph, G)
    torch.cuda.synchronize()
    fused = _cabi.kernel_launches(_cabi.KERN_GIN_FUSED_MLP) > k0
    assert fused == expect_fused, fused
    _gate(f"encoder_grads[H=768,L=5,nodes={graph[0].numel()},fused_tail={int(fused)}]", got,
          oracle_grads(enc, proj, L, graph, G, torch.float64), oracle_grads(enc, proj, L, graph, G, torch.bfloat16))


@pytest.mark.gpu
def test_grads_vs_oracle_fused_tail():
    _case_fused(True)


@pytest.mark.gpu
def test_grads_vs_oracle_row_kernel_tail():
    """the same case with the fused layer tail switched off (LLB_GIN_FUSED_TAIL is read once per process: a child process)"""
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_encoder_grad as t; t._case_fused(False)"
            % (ROOT, os.path.join(ROOT, "tests")))
    env = dict(os.environ, LLB_GIN_FUSED_TAIL="0")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.gpu
@pytest.mark.parametrize("L", [2, 5])
@pytest.mark.parametrize("H", [37, 300])
def test_grads_vs_oracle_padded_width(H, L):
    g, enc, proj = _encoder(L, H, seed=5)
    graph = _ragged_batch(seed=H + L)
    B = int(graph[3][-1]) + 1
    G = _G(B, H, seed=6)
    got = _gpu_grads(g, graph, G)
    assert all(bool(torch.isfinite(v).all()) for v in got.values())
    _gate(f"encoder_grads_padded[H={H},L={L}]", got, oracle_grads(enc, proj, L, graph, G, torch.float64),
          oracle_grads(enc, proj, L, graph, G, torch.bfloat16))


@pytest.mark.gpu
def test_grads_vs_oracle_with_max_pool_ties():
    L, H = 4, 256
    g, enc, proj = _encoder(L, H, seed=8)
    graph = _star_batch()
    B = int(graph[3][-1]) + 1
    G = _G(B, H, seed=7)
    got = _gpu_grads(g, graph, G)
    _gate("encoder_grads_star_graphs", got, oracle_grads(enc, proj, L, graph, G, torch.float64),
          oracle_grads(enc, proj, L, graph, G, torch.bfloat16))


# ------------------------------------------------------------------------------------------------ GPU: behaviour
@pytest.mark.gpu
def test_trainable_forward_equals_the_frozen_one():
    L, H = 3, 768
    g, _, _ = _encoder(L, H, seed=5)
    graph = tuple(t.to(DEV) for t in synth.molecular_graphs(12, seed=3))
    eng = g.engine()
    eng.bind(*graph)
    plain = eng.encoder_forward()
    out = g(*graph)
    assert out.grad_fn is not None and torch.equal(out.detach(), plain)
    with torch.no_grad():
        out = g(*graph)
    assert out.grad_fn is None and torch.equal(out, plain)
    g.disable_grads()
    eng = g.engine()
    c0 = eng.launch_count()
    eng.bind(*graph)
    eng.encoder_forward()
    direct = eng.launch_count() - c0
    c0 = eng.launch_count()
    out = g(*graph)
    assert out.grad_fn is None and torch.equal(out, plain)
    assert eng.launch_count() - c0 == direct


@pytest.mark.gpu
def test_backward_is_deterministic_and_per_call():
    L, H = 3, 256
    g, _, _ = _encoder(L, H, seed=5)
    ga, gb = synth.molecular_graphs(10, seed=1), synth.molecular_graphs(7, seed=2)
    Ga, Gb = torch.randn(10, H, device=DEV), torch.randn(7, H, device=DEV)

    def fwd(graph):
        return g(*(t.to(DEV) for t in graph))

    def grads():
        out = [p.grad.clone() for p in g.parameters()]
        for p in g.parameters():
            p.grad = None
        return out

    (fwd(ga) * Ga).sum().backward()
    ref_a = grads()
    (fwd(gb) * Gb).sum().backward()
    ref_b = grads()
    ea = fwd(ga)
    (ea * Ga).sum().backward(retain_graph=True)
    first = grads()
    (ea * Ga).sum().backward()
    again = grads()
    assert all(torch.equal(x, y) and torch.equal(x, r) for x, y, r in zip(first, again, ref_a))
    ea, eb = fwd(ga), fwd(gb)
    (eb * Gb).sum().backward()
    got_b = grads()
    (ea * Ga).sum().backward()
    got_a = grads()
    assert all(torch.equal(x, r) for x, r in zip(got_a, ref_a)) and all(torch.equal(x, r) for x, r in zip(got_b, ref_b))


@pytest.mark.gpu
def test_dropout_warns_once_in_train_mode():
    enc, proj = synth.gin_encoder_state_dicts(2, 64, seed=2)
    g = GraphCLIP(2, 64, 0.1, {})
    g.molecule_encoder.load_state_dict(enc)
    g.molecule_projection.load_state_dict(proj)
    g = g.to(DEV)
    graph = tuple(t.to(DEV) for t in synth.molecular_graphs(3, seed=1))
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        g.eval()
        g(*graph)
        g.train()
        for _ in range(2):
            g(*graph)
    assert sum("dropout is not applied" in str(w.message) for w in rec) == 1, [str(w.message) for w in rec]


# ------------------------------------------------------------------------------------------------ GPU: SFT-shaped step
@pytest.mark.gpu
def test_sft_step_trains_the_encoder():
    """modeling_llamole.py:328: graph embeddings -> graph-to-LM connector -> LM loss, with the loader's bf16 parameters and the
    encoder trainable: the encoder's and the connector's weight gradients against the same pipeline on the oracle, then one SGD
    step and a forward on the stepped parameters"""
    from oracle import llamole_oracle as O

    L, H, B, V = 3, 256, 6, 40
    g, enc, proj = _encoder(L, H, seed=6, dtype=torch.bfloat16)
    graph = synth.molecular_graphs(B, seed=4, min_nodes=3, max_nodes=28)
    torch.manual_seed(0)
    conn = nn.Sequential(nn.Linear(H, V), nn.SiLU())
    labels = torch.randint(0, V, (B,))

    def ref_grads(dtype):
        m = nn.Sequential(nn.Linear(H, V), nn.SiLU()).to(dtype)
        m.load_state_dict({k: v.to(dtype) for k, v in conn.state_dict().items()})
        e = {k: v.detach().to(dtype).requires_grad_(True) if v.is_floating_point() else v for k, v in enc.items()}
        p = {k: v.detach().to(dtype).requires_grad_(True) for k, v in proj.items()}
        F.cross_entropy(m(O.gin_encoder_forward(e, p, L, *graph)).double(), labels).backward()
        out = {("enc", k): v.grad.double() for k, v in e.items() if v.is_floating_point()}
        out.update({("proj", k): v.grad.double() for k, v in p.items()})
        out[("conn", "0.weight")] = m[0].weight.grad.double()
        return out

    conn_gpu = conn.to(torch.bfloat16).to(DEV)
    emb = g(*(t.to(DEV) for t in graph))
    assert emb.dtype == torch.bfloat16 and emb.grad_fn is not None
    F.cross_entropy(conn_gpu(emb).float(), labels.to(DEV)).backward()
    got = {("enc", k): p.grad for k, p in g.molecule_encoder.named_parameters()}
    got.update({("proj", k): p.grad for k, p in g.molecule_projection.named_parameters()})
    got[("conn", "0.weight")] = conn_gpu[0].weight.grad
    assert all(v.dtype == torch.bfloat16 for v in got.values())
    # the weight matrices and embedding tables: the connector's bf16 rounding of dL/d(emb) is shared with the bf16 oracle, and
    # on the single-row vectors (biases, LayerNorm affines) it is most of the bf16 oracle's error as well
    ref64, ref16 = ref_grads(torch.float64), ref_grads(torch.bfloat16)
    mats = [k for k in ref64 if ref64[k].dim() == 2]
    _gate("encoder_sft_step_weight_grads", {k: got[k] for k in mats}, {k: ref64[k] for k in mats}, {k: ref16[k] for k in mats})

    torch.optim.SGD(list(g.parameters()) + list(conn_gpu.parameters()), lr=0.5).step()
    with torch.no_grad():
        after = g(*(t.to(DEV) for t in graph))
    fresh = GraphCLIP(L, H, 0.0, {})
    fresh.molecule_encoder.load_state_dict(g.molecule_encoder.state_dict())
    fresh.molecule_projection.load_state_dict(g.molecule_projection.state_dict())
    fresh = fresh.to(torch.bfloat16).to(DEV)
    fresh.disable_grads()
    ref = fresh(*(t.to(DEV) for t in graph))
    assert torch.equal(after, ref) and not torch.equal(after, emb.detach())
