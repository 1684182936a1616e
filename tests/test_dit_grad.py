"""GraphDiT.forward with the denoiser on the device, differentiable with respect to the condition vector (csrc/llb_dit_grad.cu).

Reference gradients come from torch autograd through oracle.denoiser_forward in fp64 on the CPU, in eval semantics (no condition
dropout, no property noise), on fixed noisy states and per-molecule t, with loss = the masked cross-entropy of train_loss +
<logits, G> for a fixed random G.  The accuracy gate is the predictor's: the relative L2 error of d text_embedding against fp64
must not exceed that of the same oracle run in bf16, and every row's cosine against fp64 must be >= 0.999 (or, for the
connector's weight gradient, whose rows can nearly cancel over the batch, no lower than the bf16 oracle's own).
"""
import ctypes
import os
import tempfile

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from conftest import record_parity
from llamole_b200 import _cabi, synth
from llamole_b200.dit_train import _conditions, train_loss
from llamole_b200.graph_decoder import GraphDiT

DEV = "cuda:0"


# ------------------------------------------------------------------------------------------------ helpers
def _model(cfg, N, seed, dtype=torch.float32, frozen=True):
    d = tempfile.mkdtemp()
    sd = synth.dit_state_dict(cfg, N, seed=seed)
    synth.write_dit_checkpoint(d, cfg, synth.dit_meta(N, 7, 1), sd)
    m = GraphDiT(os.path.join(d, "config.yaml"), os.path.join(d, "data.meta.json"), dtype)
    m.init_model(d)
    if frozen:
        m.disable_grads()
    for p in m.denoiser.parameters():   # the reference loader's cast: param.data = param.data.to(dtype)
        p.data = p.data.to(dtype)
    return m, sd


def _states(n_nodes, N, seed):
    """one-hot noisy states as sample_noisy_state leaves them: valid atoms one class, valid pairs a symmetric class, class 0 on
    the diagonal of valid atoms, zeros elsewhere"""
    g = torch.Generator().manual_seed(seed)
    B = len(n_nodes)
    mask = torch.arange(N)[None, :] < torch.tensor(n_nodes)[:, None]
    X = F.one_hot(torch.randint(0, 16, (B, N), generator=g), 16).float() * mask[..., None]
    e = torch.randint(0, 5, (B, N, N), generator=g) * (torch.rand(B, N, N, generator=g) < 0.3)
    e = torch.triu(e, 1)
    e = e + e.transpose(1, 2)
    pair = mask[:, :, None] & mask[:, None, :]
    E = F.one_hot(e, 5).float() * pair[..., None]
    return X, E, mask


def _loss(lam, pX, pE, X, E, GX, GE):
    return train_loss(lam, pX, pE, X, E) + (pX * GX).sum() + (pE * GE).sum()


def _inputs(n_nodes, N, seed, t=None, T=500):
    g = torch.Generator().manual_seed(seed)
    B = len(n_nodes)
    X, E, mask = _states(n_nodes, N, seed)
    props, txt = synth.dit_conditions(B, seed=seed)
    y = torch.where(props == -200.0, torch.full_like(props, float("nan")), props)
    t_int = torch.randint(0, T + 1, (B, 1), generator=g) if t is None else torch.tensor(t).view(B, 1)
    GX, GE = torch.randn(B, N, 16, generator=g) * 1e-2, torch.randn(B, N, N, 5, generator=g) * 1e-2
    return X, E, mask, y, txt, t_int.float() / T, GX, GE


def oracle_dtext(sd, cfg, inp, dtype):
    from oracle import llamole_oracle as O

    X, E, mask, y, txt, tn, GX, GE = inp
    sdd = {k: v.to(dtype) for k, v in sd.items()}
    tt = txt.detach().to(dtype).requires_grad_(True)
    pX, pE = O.denoiser_forward(sdd, cfg, X.to(dtype), E.to(dtype), mask, y.to(dtype), tt, tn.to(dtype), False)
    _loss(cfg["lambda_train"], pX, pE, X.to(dtype), E.to(dtype), GX.to(dtype), GE.to(dtype)).backward()
    return tt.grad.double()


def gpu_dtext(m, inp):
    X, E, mask, y, txt, tn, GX, GE = (t.to(DEV) for t in inp)
    tt = txt.clone().requires_grad_(True)
    c = _conditions(m.denoiser, y, tt, tn, False, False, 0.0)
    pX, pE = m.denoise_on_device(X, E, mask, c)
    _loss(m.model_config.lambda_train, pX, pE, X, E, GX, GE).backward()
    return tt.grad


def _gate(name, got, ref64, ref16, **extra):
    """rel L2 error of `got` against fp64 <= that of the bf16 oracle; per-row cosine >= 0.999, or at least the bf16 oracle's own
    where that run cannot reach 0.999 (rows of the connector's weight gradient that nearly cancel over the batch)"""
    got, ref64, ref16 = got.double().cpu(), ref64.double(), ref16.double()
    err = float((got - ref64).norm() / ref64.norm())
    err16 = float((ref16 - ref64).norm() / ref64.norm())
    live = ref64.norm(dim=1) > 0
    cos = float(F.cosine_similarity(got[live], ref64[live], dim=1).min())
    cos16 = float(F.cosine_similarity(ref16[live], ref64[live], dim=1).min())
    record_parity(name, rel_l2=err, rel_l2_bf16_oracle=err16, min_row_cosine=cos, min_row_cosine_bf16_oracle=cos16, **extra)
    print(f"\n[parity] {name}: rel L2 {err:.3e} (bf16 oracle {err16:.3e}), min row cosine {cos:.6f} (bf16 oracle {cos16:.6f})")
    assert err <= err16, (name, err, err16)
    assert cos >= min(0.999, cos16), (name, cos, cos16)


def _graph_batch(m, sizes, seed):
    """PyG-style batch (x atom numbers, edge_index both directions, edge_attr bond classes 1..3, graph_batch): paths"""
    g = torch.Generator().manual_seed(seed)
    act = m.active_index
    xs, eis, eas, bs = [], [], [], []
    off = 0
    for b, n in enumerate(sizes):
        xs.append(act[torch.randint(0, act.numel(), (n,), generator=g)])
        src = torch.arange(n - 1) + off
        ea = torch.randint(1, 4, (n - 1,), generator=g)
        eis.append(torch.stack([torch.cat([src, src + 1]), torch.cat([src + 1, src])]))
        eas.append(torch.cat([ea, ea]))
        bs.append(torch.full((n,), b))
        off += n
    return torch.cat(xs), torch.cat(eis, 1), torch.cat(eas), torch.cat(bs)


# ------------------------------------------------------------------------------------------------ CPU
def test_sizes_of_the_forward_are_unchanged():
    """the sampler's blob and workspace do not grow: the backward's weights and buffers have entries of their own"""
    parent = {(1024, 28, 16, 4096, 50, 500, 2.0): (1151468800, [6358784, 31439872, 228005376]),
              (128, 2, 2, 512, 9, 20, 2.0): (1981696, [709376, 1260800, 6615040]),
              (256, 3, 4, 1024, 64, 100, 1.0): (10559488, [2182400, 9499136, 70046208]),
              (64, 1, 1, 256, 6, 5, 2.0): (404224, [632832, 829184, 2975744])}
    lib = _cabi.lib()
    for (H, D, heads, F_, N, T, gs), (blob, ws) in parent.items():
        cfg = _cabi.DitConfig(H, D, heads, F_, N, T, 10, 768, gs)
        n = ctypes.c_size_t()
        _cabi.check(lib.llb_dit_packed_bytes(ctypes.byref(cfg), ctypes.byref(n)), "llb_dit_packed_bytes")
        assert n.value == blob
        for B, want in zip((1, 6, 64), ws):
            _cabi.check(lib.llb_dit_workspace_bytes(ctypes.byref(cfg), B, ctypes.byref(n)), "llb_dit_workspace_bytes")
            assert n.value == want, (H, B)


def test_grad_sizes():
    lib = _cabi.lib()
    n = ctypes.c_size_t()
    for bad in (_cabi.DitConfig(100, 2, 2, 512, 9, 20, 10, 768, 1.0), _cabi.DitConfig(128, 2, 1, 512, 9, 20, 10, 768, 1.0),
                _cabi.DitConfig(128, 2, 2, 512, 65, 20, 10, 768, 1.0)):
        assert lib.llb_dit_grad_packed_bytes(ctypes.byref(bad), ctypes.byref(n)) != 0
        assert lib.llb_dit_train_saved_bytes(ctypes.byref(bad), 2, 10, ctypes.byref(n)) != 0
    cfg = _cabi.DitConfig(1024, 28, 16, 4096, 50, 500, 10, 768, 1.0)
    assert lib.llb_dit_train_saved_bytes(ctypes.byref(cfg), 0, 0, ctypes.byref(n)) != 0
    assert lib.llb_dit_train_saved_bytes(ctypes.byref(cfg), 2, 101, ctypes.byref(n)) != 0   # more atoms than 2 x 50
    # the transposed operands: per block qkv 3H^2, proj H^2, fc1 + fc2 2HF, adaLN.2 6H^2; adaLN.0 (D+1) H^2; the output layer's
    # fc1 H^2, fc2 H d0, adaLN.2 2 H d0 (bf16)
    H, D, F_, d0 = 1024, 28, 4096, 16 + 5 * 50
    ops = 2 * (D * (10 * H * H + 2 * H * F_) + (D + 1) * H * H + H * H + 3 * H * d0)
    _cabi.check(lib.llb_dit_grad_packed_bytes(ctypes.byref(cfg), ctypes.byref(n)), "llb_dit_grad_packed_bytes")
    assert ops <= n.value <= 1.1 * ops, (n.value, ops)
    small, big = ctypes.c_size_t(), ctypes.c_size_t()
    _cabi.check(lib.llb_dit_train_saved_bytes(ctypes.byref(cfg), 6, 150, ctypes.byref(small)), "llb_dit_train_saved_bytes")
    _cabi.check(lib.llb_dit_train_saved_bytes(ctypes.byref(cfg), 6, 300, ctypes.byref(big)), "llb_dit_train_saved_bytes")
    assert big.value > small.value > (2 * D + 1) * 150 * H * 4   # at least the fp32 residual stream at every block-half boundary


def test_eager_path_is_pinned():
    """CPU, fp32, train mode: the loss and d loss / d text_embedding equal the values of the previous version bit for bit"""
    m, _ = _model(synth.dit_config(128, 2, 2, 4.0, 20, 2.0), 9, seed=3)
    m.train()
    assert not m.device_denoiser_ok()
    x, ei, ea, gb = _graph_batch(m, [3, 9, 1, 5], 1)
    props, txt = synth.dit_conditions(4, seed=5)
    txt = txt.clone().requires_grad_(True)
    torch.manual_seed(11)
    loss = m(x, ei, ea, gb, props, txt, -200)
    loss.backward()
    g = txt.grad
    assert loss.item().hex() == "0x1.291cec0000000p+4"
    assert g.sum().item().hex() == "-0x1.4519080000000p-5"
    assert g.abs().sum().item().hex() == "0x1.b2368a0000000p+2"
    assert [v.hex() for v in g[1, :4].tolist()] == ["0x1.0151360000000p-7", "-0x1.ad613c0000000p-12", "0x1.77ca720000000p-10",
                                                      "-0x1.d16cfc0000000p-9"]
    assert [v.hex() for v in g[3, -3:].tolist()] == ["0x1.f8b6840000000p-11", "0x1.450e5c0000000p-10", "0x1.8d6de20000000p-9"]


def test_oracle_dtext_matches_finite_differences():
    from oracle import llamole_oracle as O

    cfg = synth.dit_config(128, 2, 2, 4.0, 20, 2.0)
    sd = {k: v.double() for k, v in synth.dit_state_dict(cfg, 6, seed=9).items()}
    inp = _inputs([6, 3, 1], 6, seed=2, T=20)
    X, E, mask, y, txt, tn, GX, GE = inp

    def f(tt):
        pX, pE = O.denoiser_forward(sd, cfg, X.double(), E.double(), mask, y.double(), tt, tn.double(), False)
        return _loss(cfg["lambda_train"], pX, pE, X.double(), E.double(), GX.double(), GE.double())

    grad = oracle_dtext(sd, cfg, inp, torch.float64)
    g = torch.Generator().manual_seed(0)
    base = txt.double()
    for _ in range(6):
        b, k = int(torch.randint(0, 3, (1,), generator=g)), int(torch.randint(0, 768, (1,), generator=g))
        e = torch.zeros_like(base)
        e[b, k] = 1e-6
        fd = (f(base + e) - f(base - e)).item() / 2e-6
        assert abs(fd - grad[b, k].item()) <= 1e-6 + 1e-4 * abs(fd), (b, k, fd, grad[b, k].item())


# ------------------------------------------------------------------------------------------------ GPU: accuracy
@pytest.mark.gpu
def test_dtext_vs_oracle_checkpoint_shape():
    """H = 1024, depth 28, 16 heads, N = 50, B = 6: the latency regime (split-K proj and fc2, row kernels)"""
    cfg = synth.dit_config()
    m, sd = _model(cfg, 50, seed=21)
    m = m.to(DEV)
    inp = _inputs([50, 37, 12, 25, 44, 9], 50, seed=3)
    got = gpu_dtext(m, inp)
    _gate("dit_dtext_checkpoint_B6", got, oracle_dtext(sd, cfg, inp, torch.float64), oracle_dtext(sd, cfg, inp, torch.bfloat16))


@pytest.mark.gpu
def test_dtext_vs_oracle_fused_tails():
    """>= 2048 token rows at depth 3: the forward runs the fused CTA-pair GEMM + LayerNorm block tails"""
    cfg = synth.dit_config(depth=3)
    m, sd = _model(cfg, 50, seed=22)
    m = m.to(DEV)
    g = torch.Generator().manual_seed(4)
    sizes = torch.randint(42, 51, (48,), generator=g).tolist()
    assert sum(sizes) >= 2048
    inp = _inputs(sizes, 50, seed=4)
    k0 = _cabi.kernel_launches(_cabi.KERN_GEMM_LN_PAIR)
    got = gpu_dtext(m, inp)
    assert _cabi.kernel_launches(_cabi.KERN_GEMM_LN_PAIR) > k0
    _gate("dit_dtext_fused_tails_depth3", got, oracle_dtext(sd, cfg, inp, torch.float64), oracle_dtext(sd, cfg, inp, torch.bfloat16))


@pytest.mark.gpu
def test_dtext_vs_oracle_ragged_batch():
    """node counts 1, 2, 50 and more; missing properties; one NaN text row (zero gradient); t = 0 and t = T"""
    cfg = synth.dit_config(256, 4, 4, 4.0, 500, 2.0)
    m, sd = _model(cfg, 50, seed=23)
    m = m.to(DEV)
    sizes = [1, 2, 50, 7, 31, 3]
    inp = list(_inputs(sizes, 50, seed=5, t=[0, 500, 250, 1, 499, 77]))
    inp[4] = inp[4].clone()
    inp[4][3, 5] = float("nan")
    inp[3] = inp[3].clone()
    inp[3][0, :] = float("nan")                 # every property of molecule 0 missing
    got = gpu_dtext(m, inp)
    assert torch.all(got[3] == 0)
    ref = oracle_dtext(sd, cfg, inp, torch.float64)
    assert torch.all(ref[3] == 0)
    _gate("dit_dtext_ragged", got, ref, oracle_dtext(sd, cfg, inp, torch.bfloat16))


# ------------------------------------------------------------------------------------------------ GPU: GraphDiT.forward
def _sft_batch(m, B, seed):
    g = torch.Generator().manual_seed(seed)
    sizes = torch.randint(1, m.max_n_nodes + 1, (B,), generator=g).tolist()
    graph = _graph_batch(m, sizes, seed)
    props, txt = synth.dit_conditions(B, seed=seed)
    return graph, props, txt


@pytest.mark.gpu
def test_forward_device_vs_eager_train_mode():
    """same seed, same GPU: the device denoiser against the eager one (a parameter requiring grad routes there), train mode
    with drop_condition = 0.1"""
    cfg = synth.dit_config(512, 4, 8, 4.0, 500, 2.0)
    m, _ = _model(cfg, 30, seed=24)
    m = m.to(DEV).train()
    graph, props, txt = _sft_batch(m, 32, seed=6)
    graph = [t.to(DEV) for t in graph]

    def run(device_path):
        m.denoiser.x_embedder[0].weight.requires_grad_(not device_path)
        assert m.device_denoiser_ok() == device_path
        tt = txt.to(DEV).clone().requires_grad_(True)
        torch.manual_seed(123)
        loss = m(*graph, props.to(DEV), tt, -200)
        loss.backward()
        return loss.item(), tt.grad, torch.cuda.get_rng_state(), torch.get_rng_state()

    ld, gd, cuda_d, cpu_d = run(True)
    le, ge, cuda_e, cpu_e = run(False)
    m.denoiser.x_embedder[0].weight.grad = None
    m.denoiser.x_embedder[0].weight.requires_grad_(False)
    assert torch.equal(cuda_d, cuda_e) and torch.equal(cpu_d, cpu_e)
    assert abs(ld - le) <= 1e-2 * abs(le), (ld, le)
    dropped = ge.norm(dim=1) == 0
    assert dropped.any(), "no text row was dropped: pick another seed"
    assert torch.all(gd[dropped] == 0)
    cos = F.cosine_similarity(gd[~dropped].double(), ge[~dropped].double(), dim=1)
    record_parity("dit_forward_device_vs_eager", loss_device=ld, loss_eager=le, min_row_cosine=float(cos.min()))
    assert float(cos.min()) >= 0.999


@pytest.mark.gpu
def test_sft_step_trains_the_connector():
    """modeling_llamole.py:371-379: text_embedding = lm_to_graph_decoder(hidden) in bf16 -> frozen bf16 GraphDiT -> loss; the
    connector's weight gradient against the same pipeline on the oracle"""
    from oracle import llamole_oracle as O

    cfg = synth.dit_config(256, 3, 4, 4.0, 500, 2.0)
    m, sd = _model(cfg, 40, seed=25, dtype=torch.bfloat16)
    m = m.to(DEV).eval()
    B = 6
    X, E, mask, y, _, tn, GX, GE = _inputs([40, 17, 5, 33, 2, 26], 40, seed=7)
    torch.manual_seed(0)
    conn = nn.Sequential(nn.Linear(896, 768), nn.SiLU())
    hidden = torch.randn(B, 896) * 0.5

    def ref_grad(dtype):
        c2 = nn.Sequential(nn.Linear(896, 768), nn.SiLU()).to(dtype)
        c2.load_state_dict({k: v.to(dtype) for k, v in conn.state_dict().items()})
        sdd = {k: v.to(dtype) for k, v in sd.items()}
        pX, pE = O.denoiser_forward(sdd, cfg, X.to(dtype), E.to(dtype), mask, y.to(dtype), c2(hidden.to(dtype)), tn.to(dtype), False)
        _loss(cfg["lambda_train"], pX, pE, X.to(dtype), E.to(dtype), GX.to(dtype), GE.to(dtype)).backward()
        return c2[0].weight.grad.double()

    conn_gpu = conn.to(torch.bfloat16).to(DEV)
    txt = conn_gpu(hidden.to(DEV, torch.bfloat16))
    Xd, Ed, md, yd, tnd = X.to(DEV, torch.bfloat16), E.to(DEV, torch.bfloat16), mask.to(DEV), y.to(DEV, torch.bfloat16), tn.to(DEV)
    c = _conditions(m.denoiser, yd, txt, tnd, False, False, 0.0)
    pX, pE = m.denoise_on_device(Xd, Ed, md, c)
    assert pX.dtype == torch.bfloat16 and pE.dtype == torch.bfloat16
    _loss(cfg["lambda_train"], pX, pE, Xd, Ed, GX.to(DEV, torch.bfloat16), GE.to(DEV, torch.bfloat16)).backward()
    assert all(p.grad is None for p in m.denoiser.parameters())
    _gate("dit_sft_connector_weight_grad", conn_gpu[0].weight.grad, ref_grad(torch.float64), ref_grad(torch.bfloat16))


# ------------------------------------------------------------------------------------------------ GPU: determinism, ownership
@pytest.mark.gpu
def test_backward_is_deterministic_and_per_call():
    cfg = synth.dit_config(256, 3, 4, 4.0, 500, 2.0)
    m, _ = _model(cfg, 30, seed=26)
    m = m.to(DEV)
    ia = [t.to(DEV) for t in _inputs([30, 12, 5], 30, seed=8)]
    ib = [t.to(DEV) for t in _inputs([7, 30, 30, 1], 30, seed=9)]

    def fwd(inp):
        X, E, mask, y, txt, tn, GX, GE = inp
        tt = txt.clone().requires_grad_(True)
        c = _conditions(m.denoiser, y, tt, tn, False, False, 0.0)
        pX, pE = m.denoise_on_device(X, E, mask, c)
        return tt, _loss(m.model_config.lambda_train, pX, pE, X, E, GX, GE)

    def alone(inp):
        tt, loss = fwd(inp)
        loss.backward()
        return tt.grad

    ref_a, ref_b = alone(ia), alone(ib)
    assert torch.equal(alone(ia), ref_a)                       # run-to-run bit-identical
    ta, la = fwd(ia)
    tb, lb = fwd(ib)
    lb.backward()                                              # reverse order
    la.backward()
    assert torch.equal(ta.grad, ref_a) and torch.equal(tb.grad, ref_b)
    # a sampling run between a forward and its backward changes neither
    X1, E1, _ = m.generate_graphs(*synth.dit_conditions(4, seed=1), n_nodes=torch.tensor([30, 3, 17, 9]), seed=5, steps=3)
    ta, la = fwd(ia)
    X2, E2, _ = m.generate_graphs(*synth.dit_conditions(4, seed=1), n_nodes=torch.tensor([30, 3, 17, 9]), seed=5, steps=3)
    la.backward()
    assert torch.equal(ta.grad, ref_a)
    assert torch.equal(X1, X2) and torch.equal(E1, E2)


@pytest.mark.gpu
def test_routing():
    cfg = synth.dit_config(256, 2, 4, 4.0, 500, 2.0)
    m, _ = _model(cfg, 20, seed=27)
    m = m.to(DEV).train()
    graph, props, txt = _sft_batch(m, 8, seed=10)
    graph = [t.to(DEV) for t in graph]
    props, txt = props.to(DEV), txt.to(DEV)
    # frozen: the device path; under no_grad the same loss bit for bit
    assert m.device_denoiser_ok()
    torch.manual_seed(5)
    l1 = m(*graph, props, txt.clone().requires_grad_(True), -200)
    torch.manual_seed(5)
    with torch.no_grad():
        l2 = m(*graph, props, txt, -200)
    assert torch.equal(l1.detach(), l2)
    # a trainable parameter: the eager path, and the parameter gets its gradient
    w = m.denoiser.blocks[1].mlp.fc2.weight
    w.requires_grad_(True)
    assert not m.device_denoiser_ok()
    torch.manual_seed(5)
    m(*graph, props, txt, -200).backward()
    assert w.grad is not None and w.grad.abs().sum() > 0
    w.requires_grad_(False)
    # the sampler's launches per step are the same before and after training calls on the engine
    eng = m.engine()
    props_s, txt_s = synth.dit_conditions(3, seed=2)
    y = torch.where(props_s == -200.0, torch.full_like(props_s, float("nan")), props_s)

    def step_launches():
        eng.begin(torch.tensor([20, 5, 11], dtype=torch.int32), y.to(DEV).contiguous(), txt_s.to(DEV).contiguous())
        eng.init_state(1, None, None)
        eng.step(500, 1)
        n0 = eng.launch_count()
        eng.step(499, 1)
        return eng.launch_count() - n0

    before = step_launches()
    torch.manual_seed(6)
    m(*graph, props, txt.clone().requires_grad_(True), -200).backward()
    assert step_launches() == before
