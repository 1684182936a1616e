"""GraphPredictor.forward differentiable with respect to the text condition c (csrc/llb_gin_grad.cu).

Reference gradients come from torch autograd through oracle.gin_predictor_forward in fp64 on the CPU, with
loss = cross-entropy over fixed labels + <logits, G> for a fixed random G.  The accuracy gate is the reference's own precision
in the shipped configs' compute dtype: for every case the relative L2 error of dc against fp64 must not exceed that of the same
oracle run in bf16 on the same inputs, and every row's cosine against fp64 must be >= 0.999.
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
from llamole_b200 import GraphPredictor, _cabi, synth

DEV = "cuda:0"


# ------------------------------------------------------------------------------------------------ helpers
def _loss(logits, labels, G):
    return F.cross_entropy(logits, labels) + (logits * G).sum()


def _loss_inputs(B, D, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, D, (B,), generator=g), torch.randn(B, D, generator=g, dtype=torch.float64) * 1e-3


def oracle_dc(sd, L, graph, c, labels, G, dtype):
    """dL/dc through the oracle, everything (parameters, c, the loss) in `dtype`; returned as fp64."""
    from oracle import llamole_oracle as O

    sdd = {k: v.to(dtype) if v.is_floating_point() else v for k, v in sd.items()}
    cc = c.detach().to(dtype).requires_grad_(True)
    logits = O.gin_predictor_forward(sdd, L, *graph, cc)
    _loss(logits, labels, G.to(dtype)).backward()
    return cc.grad.double()


def _gate(name, got, ref64, ref16, **extra):
    """rel L2 error of `got` against fp64 <= that of the bf16 oracle; per-row cosine >= 0.999"""
    got, ref64, ref16 = got.double().cpu(), ref64.double(), ref16.double()
    err = float((got - ref64).norm() / ref64.norm())
    err16 = float((ref16 - ref64).norm() / ref64.norm())
    cos = float(F.cosine_similarity(got, ref64, dim=1).min())
    record_parity(name, rel_l2=err, rel_l2_bf16_oracle=err16, min_row_cosine=cos, **extra)
    print(f"\n[parity] {name}: dc rel L2 {err:.3e} (bf16 oracle {err16:.3e}), min row cosine {cos:.6f}")
    assert err <= err16, (name, err, err16)
    assert cos >= 0.999, (name, cos)


def _predictor(L, H, D, seed, dtype=torch.float32):
    sd = synth.gin_predictor_state_dict(L, H, D, seed=seed)
    gp = GraphPredictor(L, H, 0.0, D, {}, {})
    gp.predictor.load_state_dict(sd)
    gp.disable_grads()
    return gp.to(dtype).to(DEV), sd


def _gpu_dc(gp, graph, c, labels, G):
    cg = c.to(DEV, torch.float32).requires_grad_(True)
    logits = gp(*(t.to(DEV) for t in graph), cg)
    assert logits.grad_fn is not None
    _loss(logits.float(), labels.to(DEV), G.to(DEV, torch.float32)).backward()
    return cg.grad


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
    """star graphs with identical leaves (same atom, same bond): the leaves are automorphic, so their rows are equal and the
    virtual node's max-pool has exact ties at every layer"""
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
def test_sizes_of_the_forward_are_unchanged():
    """the forward's blob and workspace do not grow: the backward's weights and buffers have entries of their own"""
    parent = {(1, 0): (168448, 1100288), (1, 1): (1152768, 1234432), (37, 0): (353024, 1233408), (37, 1): (1554176, 1372672),
              (300, 0): (9815296, 3992064), (300, 1): (16524544, 4325888), (1000, 0): (101991936, 11575040),
              (1000, 1): (126551808, 12443904)}
    lib = _cabi.lib()
    for (H, p), want in parent.items():
        cfg = _cabi.GinConfig(H, 3, p, 777 if p else 0, 768 if p else 0)
        packed, ws = ctypes.c_size_t(), ctypes.c_size_t()
        _cabi.check(lib.llb_gin_packed_bytes(ctypes.byref(cfg), ctypes.byref(packed)), "llb_gin_packed_bytes")
        _cabi.check(lib.llb_gin_workspace_bytes(ctypes.byref(cfg), 500, 1000, 20, 1, ctypes.byref(ws)), "llb_gin_workspace_bytes")
        assert (packed.value, ws.value) == want, (H, p)


def test_grad_sizes():
    lib = _cabi.lib()
    n = ctypes.c_size_t()
    for H in (0, -64):
        cfg = _cabi.GinConfig(H, 3, 1, 777, 768)
        assert lib.llb_gin_grad_packed_bytes(ctypes.byref(cfg), ctypes.byref(n)) != 0
        assert lib.llb_gin_saved_bytes(ctypes.byref(cfg), 10, 10, 2, ctypes.byref(n)) != 0
    enc = _cabi.GinConfig(256, 3, 0, 0, 0)
    assert lib.llb_gin_grad_packed_bytes(ctypes.byref(enc), ctypes.byref(n)) != 0
    assert lib.llb_gin_saved_bytes(ctypes.byref(enc), 10, 10, 2, ctypes.byref(n)) != 0
    # the head's transposed copy dominates the grad blob: (4H padded) x (out_dim padded) bf16
    cfg = _cabi.GinConfig(768, 5, 1, 180576, 768)
    _cabi.check(lib.llb_gin_grad_packed_bytes(ctypes.byref(cfg), ctypes.byref(n)), "llb_gin_grad_packed_bytes")
    assert 3072 * 180576 * 2 <= n.value <= 3072 * 180576 * 2 * 1.1
    small, big = ctypes.c_size_t(), ctypes.c_size_t()
    _cabi.check(lib.llb_gin_saved_bytes(ctypes.byref(cfg), 500, 1000, 20, ctypes.byref(small)), "llb_gin_saved_bytes")
    _cabi.check(lib.llb_gin_saved_bytes(ctypes.byref(cfg), 1000, 2000, 20, ctypes.byref(big)), "llb_gin_saved_bytes")
    assert big.value > small.value > 500 * 768 * 4 * 4   # at least the fp32 inputs of layers 1..L-1


def test_oracle_dc_matches_finite_differences():
    """the fp64 reference the GPU tests compare against is the derivative of the oracle's loss"""
    from oracle import llamole_oracle as O

    L, H, D = 3, 16, 11
    sd = {k: v.double() for k, v in synth.gin_predictor_state_dict(L, H, D, text_dim=8, seed=3).items()}
    x, ei, ea, b = synth.molecular_graphs(3, seed=2, min_nodes=4, max_nodes=7)
    c = synth.text_conditions(3, seed=1, text_dim=8).double()
    labels, G = _loss_inputs(3, D, seed=4)
    dc = oracle_dc(sd, L, (x, ei, ea, b), c, labels, G, torch.float64)

    def f(cc):
        with torch.no_grad():
            return float(_loss(O.gin_predictor_forward(sd, L, x, ei, ea, b, cc), labels, G))

    h = 1e-6
    fd = torch.zeros_like(c)
    for i in range(c.shape[0]):
        for j in range(c.shape[1]):
            e = torch.zeros_like(c)
            e[i, j] = h
            fd[i, j] = (f(c + e) - f(c - e)) / (2 * h)
    assert torch.allclose(dc, fd, rtol=1e-5, atol=1e-8), (dc - fd).abs().max()


# ------------------------------------------------------------------------------------------------ GPU: dc against the oracle
def _case_fused(expect_fused):
    L, H, D, B = 5, 768, 16384, 64
    gp, sd = _predictor(L, H, D, seed=13)
    graph = synth.molecular_graphs(B, seed=7)
    c = synth.text_conditions(B, seed=2)
    labels, G = _loss_inputs(B, D, seed=5)
    k0 = _cabi.kernel_launches(_cabi.KERN_GIN_FUSED_MLP)
    got = _gpu_dc(gp, graph, c, labels, G)
    torch.cuda.synchronize()
    fused = _cabi.kernel_launches(_cabi.KERN_GIN_FUSED_MLP) > k0
    assert fused == expect_fused, fused
    ref64 = oracle_dc(sd, L, graph, c, labels, G, torch.float64)
    ref16 = oracle_dc(sd, L, graph, c, labels, G, torch.bfloat16)
    _gate(f"predictor_dc[H=768,L=5,D=16384,fused_tail={int(fused)}]", got, ref64, ref16)


@pytest.mark.gpu
def test_dc_vs_oracle_fused_tail():
    _case_fused(True)


@pytest.mark.gpu
def test_dc_vs_oracle_row_kernel_tail():
    """the same case with the fused layer tail switched off (LLB_GIN_FUSED_TAIL is read once per process: a child process)"""
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_predictor_grad as t; t._case_fused(False)"
            % (ROOT, os.path.join(ROOT, "tests")))
    env = dict(os.environ, LLB_GIN_FUSED_TAIL="0")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.gpu
@pytest.mark.parametrize("L", [2, 5])
@pytest.mark.parametrize("H", [37, 300])
def test_dc_vs_oracle_padded_width(H, L):
    D = 777
    gp, sd = _predictor(L, H, D, seed=5)
    graph = _ragged_batch(seed=H + L)
    B = int(graph[3][-1]) + 1
    c = synth.text_conditions(B, seed=1)
    labels, G = _loss_inputs(B, D, seed=6)
    got = _gpu_dc(gp, graph, c, labels, G)
    assert got.shape == (B, 768) and bool(torch.isfinite(got).all())
    _gate(f"predictor_dc_padded[H={H},L={L}]", got, oracle_dc(sd, L, graph, c, labels, G, torch.float64),
          oracle_dc(sd, L, graph, c, labels, G, torch.bfloat16))


@pytest.mark.gpu
def test_dc_vs_oracle_with_max_pool_ties():
    L, H, D = 4, 256, 333
    gp, sd = _predictor(L, H, D, seed=8)
    graph = _star_batch()
    B = int(graph[3][-1]) + 1
    c = synth.text_conditions(B, seed=3)
    labels, G = _loss_inputs(B, D, seed=7)
    got = _gpu_dc(gp, graph, c, labels, G)
    _gate("predictor_dc_star_graphs", got, oracle_dc(sd, L, graph, c, labels, G, torch.float64),
          oracle_dc(sd, L, graph, c, labels, G, torch.bfloat16))


# ------------------------------------------------------------------------------------------------ GPU: the forward is unchanged
@pytest.mark.gpu
def test_forward_paths_unchanged():
    L, H, D = 3, 256, 777
    gp, sd = _predictor(L, H, D, seed=5)
    graph = tuple(t.to(DEV) for t in synth.molecular_graphs(12, seed=3))
    c = synth.text_conditions(12, seed=1).to(DEV)
    eng = gp.engine()
    eng.bind(*graph)
    plain = eng.predictor_forward(c)          # the path GraphPredictor.forward took before it was differentiable
    plain_none = eng.predictor_forward(None)
    with_grad = gp(*graph, c.clone().requires_grad_(True))
    assert with_grad.grad_fn is not None and torch.equal(with_grad.detach(), plain)
    for out, ref in ((gp(*graph, c), plain), (gp(*graph, None), plain_none)):
        assert out.grad_fn is None and torch.equal(out, ref)
    with torch.no_grad():
        out = gp(*graph, c.clone().requires_grad_(True))
    assert out.grad_fn is None and torch.equal(out, plain)


@pytest.mark.gpu
def test_backward_is_deterministic_and_per_call():
    L, H, D = 3, 256, 777
    gp, _ = _predictor(L, H, D, seed=5)
    ga = synth.molecular_graphs(10, seed=1)
    gb = synth.molecular_graphs(7, seed=2)
    ca, cb = synth.text_conditions(10, seed=1).to(DEV), synth.text_conditions(7, seed=2).to(DEV)
    Ga, Gb = torch.randn(10, D, device=DEV), torch.randn(7, D, device=DEV)

    def fwd(graph, c):
        cg = c.clone().requires_grad_(True)
        return cg, gp(*(t.to(DEV) for t in graph), cg)

    def alone(graph, c, G):
        cg, lg = fwd(graph, c)
        (lg * G).sum().backward()
        return cg.grad.clone()

    ref_a, ref_b = alone(ga, ca, Ga), alone(gb, cb, Gb)
    cg, lg = fwd(ga, ca)
    (lg * Ga).sum().backward(retain_graph=True)
    first = cg.grad.clone()
    cg.grad = None
    (lg * Ga).sum().backward()
    assert torch.equal(first, cg.grad) and torch.equal(first, ref_a)
    cga, la = fwd(ga, ca)
    cgb, lb = fwd(gb, cb)
    (lb * Gb).sum().backward()
    (la * Ga).sum().backward()
    assert torch.equal(cga.grad, ref_a) and torch.equal(cgb.grad, ref_b)


# ------------------------------------------------------------------------------------------------ GPU: SFT-shaped step
@pytest.mark.gpu
def test_sft_step_trains_the_connector():
    """modeling_llamole.py:409-425: c = lm_to_graph_predictor(hidden) in bf16 -> frozen predictor -> CE; the connector's weight
    gradient against the same pipeline on the oracle"""
    from oracle import llamole_oracle as O

    L, H, D, B = 3, 256, 333, 6
    gp, sd = _predictor(L, H, D, seed=6, dtype=torch.bfloat16)
    graph = synth.molecular_graphs(B, seed=4, min_nodes=3, max_nodes=28)
    torch.manual_seed(0)
    conn = nn.Sequential(nn.Linear(896, 768), nn.SiLU())
    hidden = torch.randn(B, 896) * 0.5
    labels = torch.randint(0, D, (B,))

    def ref_grad(dtype):
        m = nn.Sequential(nn.Linear(896, 768), nn.SiLU()).to(dtype)
        m.load_state_dict({k: v.to(dtype) for k, v in conn.state_dict().items()})
        sdd = {k: v.to(dtype) if v.is_floating_point() else v for k, v in sd.items()}
        F.cross_entropy(O.gin_predictor_forward(sdd, L, *graph, m(hidden.to(dtype))), labels).backward()
        return m[0].weight.grad.double()

    conn_gpu = conn.to(torch.bfloat16).to(DEV)
    with warnings.catch_warnings():
        warnings.filterwarnings("error", message=".*receive none")   # frozen with disable_grads(): no parameter warning
        c = conn_gpu(hidden.to(DEV, torch.bfloat16))
        c.retain_grad()
        logits = gp(*(t.to(DEV) for t in graph), c)
    assert logits.dtype == torch.bfloat16
    F.cross_entropy(logits, labels.to(DEV)).backward()
    assert c.grad is not None and c.grad.dtype == torch.bfloat16
    assert all(p.grad is None for p in gp.predictor.parameters())
    _gate("predictor_sft_connector_weight_grad", conn_gpu[0].weight.grad, ref_grad(torch.float64), ref_grad(torch.bfloat16))

    # without disable_grads() the forward warns, once, that the predictor's parameters receive no gradient
    gp2 = GraphPredictor(L, H, 0.0, D, {}, {})
    gp2.predictor.load_state_dict(sd)
    gp2 = gp2.to(DEV)
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        for _ in range(2):
            gp2(*(t.to(DEV) for t in graph), torch.randn(B, 768, device=DEV, requires_grad=True))
    assert sum("receive none" in str(w.message) for w in rec) == 1, [str(w.message) for w in rec]
