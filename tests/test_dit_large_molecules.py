"""GraphDiT sampling with molecules of up to 128 atoms (max_node of the checkpoint's data.meta.json in 65..128).

Above 64 atoms the sampler switches two kernels, from what the host knows about the configuration and the bound batch:
  - attention: the 128-row tile of dit_attention_tma_kernel when a molecule of the batch has more than 64 atoms (a batch of
    smaller molecules keeps the 64-row kernel, whatever the checkpoint's max_node);
  - step kernel: its logit rows T[pass][atom][16 + 5 N] no longer fit a block's shared memory once N > 71 with guidance, and
    live in the raw output-layer rows in global memory.
The training entries (the device SFT denoiser and its backward) stay at 64 atoms: such a checkpoint trains through the eager loss.

Tolerances are those of tests/test_gpu_parity.py and tests/test_gpu_parity_large.py: logits max |d| <= 0.10, rms <= 0.02 against
the fp32 oracle; posterior probabilities within 2e-5 and categories exact (margin >= 1e-3) given the oracle's logits and noise;
teacher-forced categories exact wherever the oracle's margin exceeds 4 (2 s - 1) delta (DESIGN.md 5a).
"""
import ctypes
import os
import subprocess
import sys
import tempfile

import pytest
import torch

from conftest import record_parity
from llamole_b200 import _cabi, synth
from llamole_b200.graph_decoder import GraphDiT, state_from_onehot
from llamole_b200.sharding import pack_graphs, unpack_graphs

DEV = "cuda:0"
HERE = os.path.dirname(os.path.abspath(__file__))


def _child_run(fn, env):
    """the result of this module's function `fn` run in a child process with `env` added to the environment"""
    out = os.path.join(tempfile.mkdtemp(), "child.pt")
    code = f"import sys, torch; sys.path.insert(0, {HERE!r}); from test_dit_large_molecules import {fn}; torch.save({fn}(), {out!r})"
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), cwd=os.path.dirname(HERE), capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    return torch.load(out)


def _stats(a, b):
    d = (a.double() - b.double()).abs()
    return float(d.max()), float(d.pow(2).mean().sqrt())


def _margins(prob, q, valid):
    s = prob.clamp_min(1e-5) / q
    top2 = s.topk(2, dim=-1).values
    return torch.log(top2[..., 0] / top2[..., 1])[valid]


def _al(n):
    return (n + 255) // 256 * 256


def _blob(H, D, heads, F_, N, gs=2.0):
    cfg = _cabi.DitConfig(H, D, heads, F_, N, 20, 10, 768, gs)
    n = ctypes.c_size_t()
    st = _cabi.lib().llb_dit_packed_bytes(ctypes.byref(cfg), ctypes.byref(n))
    return st, n.value, cfg


def _model(cfg, N, seed, on_gpu=True):
    d = tempfile.mkdtemp()
    sd = synth.dit_state_dict(cfg, N, seed=seed)
    meta = synth.dit_meta(N, 7, 1)
    synth.write_dit_checkpoint(d, cfg, meta, sd)
    m = GraphDiT(os.path.join(d, "config.yaml"), os.path.join(d, "data.meta.json"), torch.float32)
    m.init_model(d)
    m.disable_grads()
    return (m.to(DEV) if on_gpu else m), sd, meta


def _conditions(B, seed):
    props, txt = synth.dit_conditions(B, seed=seed)
    props[0, 2] = -200.0   # a missing property in an otherwise complete row
    y = torch.where(props == -200.0, torch.full_like(props, float("nan")), props)
    return props, y, txt


# ------------------------------------------------------------------------------------------------ CPU
def test_sizing_entries_accept_up_to_128_atoms():
    lib = _cabi.lib()
    n = ctypes.c_size_t()
    H, D, heads, F_ = 256, 2, 4, 1024
    for N in (0, 129, 200):
        st, _, cfg = _blob(H, D, heads, F_, N)
        assert st != 0 and b"max_nodes" in lib.llb_last_error(), N
        assert lib.llb_dit_workspace_bytes(ctypes.byref(cfg), 4, ctypes.byref(n)) != 0
    st, base, _ = _blob(H, D, heads, F_, 64)
    assert st == 0
    ws_prev = 0
    for N in (65, 100, 128):
        st, blob, cfg = _blob(H, D, heads, F_, N)
        assert st == 0, lib.llb_last_error()
        # only the x-embedder (H, round_up(d0, 64)) and the output layer's fc2 (d0, H) / adaLN.2 (2 d0, H) weights and biases
        # depend on N; every piece of the blob starts on 256 bytes
        d0, d064 = 16 + 5 * N, 16 + 5 * 64
        k0, k064 = (d0 + 63) // 64 * 64, (d064 + 63) // 64 * 64
        terms = lambda d, k: _al(H * k * 2) + _al(d * H * 2) + _al(2 * d * H * 2) + _al(d * 4) + _al(2 * d * 4)  # noqa: E731
        assert blob - base == terms(d0, k0) - terms(d064, k064), N
        _cabi.check(lib.llb_dit_workspace_bytes(ctypes.byref(cfg), 6, ctypes.byref(n)), "llb_dit_workspace_bytes")
        assert n.value > ws_prev
        ws_prev = n.value
        # the training entries keep their 64-atom limit
        tcfg = _cabi.DitConfig(H, D, heads, F_, N, 20, 10, 768, 1.0)
        assert lib.llb_dit_grad_packed_bytes(ctypes.byref(tcfg), ctypes.byref(n)) != 0
        assert lib.llb_dit_train_saved_bytes(ctypes.byref(tcfg), 2, 10, ctypes.byref(n)) != 0


def test_wire_format_round_trip_at_128_atoms():
    N = 128
    g = torch.Generator().manual_seed(5)
    n = torch.tensor([128, 1, 0, 77, 64])
    B = n.numel()
    valid = torch.arange(N)[None] < n[:, None]
    X = torch.where(valid, torch.randint(0, 16, (B, N), generator=g), torch.full((B, N), -1))
    e = torch.triu(torch.randint(0, 5, (B, N, N), generator=g), 1)
    E = e + e.transpose(1, 2)
    pair = valid[:, :, None] & valid[:, None, :]
    E = torch.where(pair, E, torch.full_like(E, -1))
    wire = pack_graphs(X, E, n)
    assert wire.shape == (B, 2 + 128 + 8256)
    X2, E2, n2 = unpack_graphs(wire, N)
    assert torch.equal(X2, X) and torch.equal(E2, E) and torch.equal(n2, n)


# ------------------------------------------------------------------------------------------------ GPU: H = 256
@pytest.fixture(scope="module")
def dit128():
    cfg = synth.dit_config(256, 2, 4, 4.0, 100, 2.0)
    m, sd, meta = _model(cfg, 128, seed=128)
    return m, cfg, meta, sd


RAGGED = [1, 2, 63, 64, 65, 100, 127, 128]


def _oracle_state(meta, n_nodes, N, seed, sd=None, cfg=None, y=None, txt=None):
    """z_T, then one oracle reverse step (so that the diagonal of valid atoms is one-hot, like every later state)"""
    from oracle import llamole_oracle as O

    B = n_nodes.numel()
    node_mask = torch.arange(N)[None, :] < n_nodes[:, None]
    tb = O.dit_tables(meta)
    g = torch.Generator().manual_seed(seed)
    ex = lambda *s: torch.empty(*s).exponential_(1.0, generator=g)  # noqa: E731
    X, E = O.initial_state(tb, node_mask, ex(B, N, 16), ex(B, N, N, 5), torch.float32)
    if sd is not None:
        U = O.union_transition(tb)
        sched = O.cosine_schedule(cfg["diffusion_steps"])
        with torch.no_grad():
            X, E, _, _ = O.reverse_step(sd, cfg, tb, U, sched, X, E, node_mask, y, txt, cfg["diffusion_steps"], ex(B, N, 16), ex(B, N, N, 5))
    return X, E, node_mask, ex


@pytest.mark.gpu
def test_logits_vs_oracle_ragged_128(dit128):
    from oracle import llamole_oracle as O

    m, cfg, meta, sd = dit128
    N, T = 128, cfg["diffusion_steps"]
    n_nodes = torch.tensor(RAGGED)
    B = n_nodes.numel()
    _, y, txt = _conditions(B, seed=71)
    X, E, node_mask, _ = _oracle_state(meta, n_nodes, N, 1, sd, cfg, y, txt)
    eng = m.engine()
    eng.begin(n_nodes.to(torch.int32), y.to(DEV).contiguous(), txt.to(DEV).contiguous())
    eng.set_state(*state_from_onehot(X, E))
    t = T - 1
    worst = [0.0, 0.0]
    with torch.no_grad():
        for unc in (False, True):
            rX, rE = O.denoiser_forward(sd, cfg, X, E, node_mask, y, txt, torch.full((B, 1), t / T), unc)
            lX, lE = eng.denoise(t, unc)
            torch.cuda.synchronize()
            lX, lE = lX.cpu(), lE.cpu()
            mx, rms = _stats(torch.cat([lX[node_mask].flatten(), lE.flatten()]), torch.cat([rX[node_mask].flatten(), rE.flatten()]))
            worst = [max(worst[0], mx), max(worst[1], rms)]
            assert torch.equal(lE, lE.transpose(1, 2))
            pair = node_mask[:, :, None] & node_mask[:, None, :] & ~torch.eye(N, dtype=torch.bool)[None]
            assert float(lE[~pair].abs().max()) == 0.0 and float(lX[~node_mask].abs().max()) == 0.0
    record_parity("dit_128_atoms_ragged_vs_oracle", n_nodes=RAGGED, hidden=256, depth=2, logits_max_abs=worst[0], logits_rms=worst[1])
    print(f"\n[parity] N=128 ragged batch vs fp32 oracle: max|d|={worst[0]:.4f} rms={worst[1]:.5f}")
    assert worst[0] <= 0.10 and worst[1] <= 0.02, worst


@pytest.mark.gpu
def test_posterior_and_sampling_given_oracle_logits_128(dit128):
    """the global-memory step kernel alone: the oracle's logits in, the oracle's posterior, guidance and categories out"""
    from oracle import llamole_oracle as O

    m, cfg, meta, sd = dit128
    N, T = 128, cfg["diffusion_steps"]
    n_nodes = torch.tensor(RAGGED)
    B = n_nodes.numel()
    _, y, txt = _conditions(B, seed=72)
    X, E, node_mask, ex = _oracle_state(meta, n_nodes, N, 2, sd, cfg, y, txt)
    tb = O.dit_tables(meta)
    U = O.union_transition(tb)
    betas, abar = O.cosine_schedule(T)
    pair = node_mask[:, :, None] & node_mask[:, None, :] & torch.triu(torch.ones(N, N, dtype=torch.bool), 1)
    eng = m.engine()
    eng.begin(n_nodes.to(torch.int32), y.to(DEV).contiguous(), txt.to(DEV).contiguous())
    for t in (T - 1, T // 2, 1):
        with torch.no_grad():
            tn = torch.full((B, 1), t / T)
            lc = O.denoiser_forward(sd, cfg, X, E, node_mask, y, txt, tn, False)
            lu = O.denoiser_forward(sd, cfg, X, E, node_mask, y, txt, tn, True)
            bt, a_s, a_t = float(betas[t]), float(abar[t - 1]), float(abar[t])
            pc = O.posterior_dense(tb, U, lc[0], lc[1], X, E, bt, a_s, a_t)
            pu = O.posterior_dense(tb, U, lu[0], lu[1], X, E, bt, a_s, a_t)
            pX, pE = O.guidance(pc[0], pu[0], cfg["guide_scale"]), O.guidance(pc[1], pu[1], cfg["guide_scale"])
            qX, qE = ex(B, N, 16), ex(B, N, N, 5)
            Xs, Es = O.sample_categories(pX, pE, node_mask, qX, qE)
        eng.set_state(*state_from_onehot(X, E))
        gpX, gpE = eng.posterior_sample(t, lc[0].to(DEV).contiguous(), lc[1].to(DEV).contiguous(), lu[0].to(DEV).contiguous(),
                                        lu[1].to(DEV).contiguous(), 0, qX.to(DEV).contiguous(), qE.to(DEV).contiguous())
        gX, gE = eng.get_state()
        torch.cuda.synchronize()
        gX, gE = gX.cpu().long(), gE.cpu().long()
        assert float((gpX.cpu() - pX)[node_mask].abs().max()) <= 2e-5, t
        assert float((gpE.cpu() - pE)[pair].abs().max()) <= 2e-5, t
        okx = (gX == Xs)[node_mask] | (_margins(pX, qX, node_mask) < 1e-3)
        oke = (gE == Es)[pair] | (_margins(pE, qE, pair) < 1e-3)
        assert bool(okx.all()) and bool(oke.all()), t
        assert torch.equal(gE, gE.transpose(1, 2))
        assert bool((gX[~node_mask] == -1).all()) and bool((gE[~(node_mask[:, :, None] & node_mask[:, None, :])] == -1).all())


TILE_CASES = (([64, 1, 33, 50], "<64>"), ([64, 1, 33, 65], "<128>"))


def _attention_tile_run():
    """for each batch of TILE_CASES: the attention kernels torch.profiler saw in one denoiser pass of the N = 128 checkpoint, and
    the pass's logits"""
    from torch.profiler import ProfilerActivity, profile

    cfg = synth.dit_config(256, 2, 4, 4.0, 100, 2.0)
    m, _, meta = _model(cfg, 128, seed=128)
    out = []
    for sizes, _ in TILE_CASES:
        n_nodes = torch.tensor(sizes)
        _, y, txt = _conditions(n_nodes.numel(), seed=73)
        X, E, _, _ = _oracle_state(meta, n_nodes, 128, 3)
        eng = m.engine()
        eng.begin(n_nodes.to(torch.int32), y.to(DEV).contiguous(), txt.to(DEV).contiguous())
        eng.set_state(*state_from_onehot(X, E))
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            lX, lE = eng.denoise(cfg["diffusion_steps"] - 1, False)
            torch.cuda.synchronize()
        out.append({"names": sorted({e.key for e in prof.key_averages() if "dit_attention" in e.key}), "lX": lX.cpu(), "lE": lE.cpu()})
    return out


@pytest.mark.gpu
def test_attention_tile_follows_the_largest_molecule_of_the_batch(dit128):
    """an N = 128 checkpoint runs today's 64-row attention kernel for a batch of molecules of <= 64 atoms, and the 128-row one
    as soon as one molecule has more; both against the oracle.  The profiler runs in a child process, so that it leaves no
    profiler state behind in this one (tests/test_launch_accounting.py counts kernels with later profiler sessions)."""
    from oracle import llamole_oracle as O

    m, cfg, meta, sd = dit128
    N, T = 128, cfg["diffusion_steps"]
    res = _child_run("_attention_tile_run", {})
    for (sizes, tile), r in zip(TILE_CASES, res):
        assert r["names"] and all(tile in k for k in r["names"]), (sizes, r["names"])
        n_nodes = torch.tensor(sizes)
        B = n_nodes.numel()
        _, y, txt = _conditions(B, seed=73)
        X, E, node_mask, _ = _oracle_state(meta, n_nodes, N, 3)
        with torch.no_grad():
            rX, rE = O.denoiser_forward(sd, cfg, X, E, node_mask, y, txt, torch.full((B, 1), (T - 1) / T), False)
        mx, rms = _stats(torch.cat([r["lX"][node_mask].flatten(), r["lE"].flatten()]), torch.cat([rX[node_mask].flatten(), rE.flatten()]))
        assert mx <= 0.10 and rms <= 0.02, (sizes, mx, rms)


@pytest.mark.gpu
def test_sampling_runs_at_128_atoms(dit128):
    m, cfg, meta, sd = dit128
    N = 128
    B = 10
    props, _, txt = _conditions(B, seed=74)
    n_nodes = torch.tensor([128, 1, 2, 64, 65, 100, 127, 30, 128, 90])
    Xa, Ea, n = m.generate_graphs(props, txt, -200, n_nodes=n_nodes, seed=21)
    torch.cuda.synchronize()
    Xc, Ec = Xa.cpu(), Ea.cpu()
    valid = torch.arange(N)[None] < n.cpu()[:, None]
    pairv = valid[:, :, None] & valid[:, None, :]
    assert bool((Xc[~valid] == -1).all()) and bool((Xc[valid] >= 0).all()) and bool((Xc[valid] < 16).all())
    assert torch.equal(Ec, Ec.transpose(1, 2))
    assert bool((Ec[~pairv] == -1).all()) and bool((Ec[pairv] >= 0).all())
    # run to run
    Xb, Eb, _ = m.generate_graphs(props, txt, -200, n_nodes=n_nodes, seed=21)
    assert torch.equal(Xa, Xb) and torch.equal(Ea, Eb)
    # independent of the batch's composition (the counter RNG is keyed by the global molecule index), for batches on the same
    # kernels: in the latency regime the split-K factor of fc2 follows the row count, so both stay at <= 640 token rows
    n_small = torch.tensor([128, 1, 2, 64, 65, 30])
    assert 2 * int(n_small.sum()) <= 640
    Xa, Ea, _ = m.generate_graphs(props[:6], txt[:6], -200, n_nodes=n_small, seed=22)
    Xs, Es, _ = m.generate_graphs(props[2:6], txt[2:6], -200, n_nodes=n_small[2:], seed=22, mol_index_base=2)
    assert torch.equal(Xa[2:], Xs) and torch.equal(Ea[2:], Es)


@pytest.mark.gpu
def test_small_batch_graph_replay_is_bit_identical_at_128_atoms(dit128):
    """the replayed small-batch pass (128-row attention, global-memory step kernel) against launch-by-launch issue"""
    if os.environ.get("LLB_GRAPH") == "0":
        pytest.skip("graph replay switched off")
    m, cfg, meta, sd = dit128
    T = cfg["diffusion_steps"]
    eng = m.engine()
    B = 6
    _, y, txt = _conditions(B, seed=75)
    n_nodes = torch.tensor([128, 70, 9, 100, 64, 1], dtype=torch.int32)
    res = []
    for eager in (False, True):
        _cabi.profile_enable(eager)
        try:
            eng.begin(n_nodes, y.to(DEV).contiguous(), txt.to(DEV).contiguous())
            eng.init_state(13, None, None)
            l0 = eng.launch_count()
            per_step = []
            for i in range(4):
                eng.step(T - i, 13)
                per_step.append(eng.launch_count() - l0)
                l0 = eng.launch_count()
            lX, lE = eng.denoise(T - 4, False)
            X, E = eng.get_state()
            torch.cuda.synchronize()
            state = eng.graph_state()
        finally:
            _cabi.profile_enable(False)
        assert state == (0 if eager else 1), (eager, state)
        assert len(set(per_step)) == 1, per_step
        res.append((X.clone(), E.clone(), lX.clone(), lE.clone(), per_step[0]))
    g, e = res
    assert all(torch.equal(a, b) for a, b in zip(g[:4], e[:4]))
    assert g[4] == e[4]


# ------------------------------------------------------------------------------------------------ GPU: checkpoint block shape
@pytest.fixture(scope="module")
def dit128_wide():
    cfg = synth.dit_config(hidden=1024, depth=3, heads=16)
    m, sd, meta = _model(cfg, 128, seed=1281)
    return m, cfg, meta, sd


@pytest.mark.gpu
@pytest.mark.parametrize("B,low,regime", [(16, 80, "throughput"), (6, 65, "latency")])
def test_checkpoint_block_shape_vs_oracle_128(dit128_wide, B, low, regime):
    from oracle import llamole_oracle as O

    m, cfg, meta, sd = dit128_wide
    N, T = 128, cfg["diffusion_steps"]
    gen = torch.Generator().manual_seed(13)
    n_nodes = torch.randint(low, N + 1, (B,), generator=gen)
    n_nodes[0], n_nodes[1] = N, low
    rows = 2 * int(n_nodes.sum())
    assert rows >= 2048 if regime == "throughput" else rows < 2048, rows
    _, y, txt = _conditions(B, seed=76)
    node_mask = torch.arange(N)[None, :] < n_nodes[:, None]
    tb = O.dit_tables(meta)
    U = O.union_transition(tb)
    sched = O.cosine_schedule(T)
    ex = lambda *s: torch.empty(*s).exponential_(1.0, generator=gen)  # noqa: E731
    X, E = O.initial_state(tb, node_mask, ex(B, N, 16), ex(B, N, N, 5), torch.float32)
    eng = m.engine()
    eng.begin(n_nodes.to(torch.int32), y.to(DEV).contiguous(), txt.to(DEV).contiguous())
    k2 = _cabi.kernel_launches(_cabi.KERN_GEMM_2CTA)
    kp = _cabi.kernel_launches(_cabi.KERN_GEMM_LN_PAIR)
    t = T - 2
    worst = [0.0, 0.0]
    with torch.no_grad():
        X, E, _, _ = O.reverse_step(sd, cfg, tb, U, sched, X, E, node_mask, y, txt, T, ex(B, N, 16), ex(B, N, N, 5))
        eng.set_state(*state_from_onehot(X, E))
        for unc in (False, True):
            rX, rE = O.denoiser_forward(sd, cfg, X, E, node_mask, y, txt, torch.full((B, 1), t / T), unc)
            lX, lE = eng.denoise(t, unc)
            torch.cuda.synchronize()
            mx, rms = _stats(torch.cat([lX.cpu()[node_mask].flatten(), lE.cpu().flatten()]), torch.cat([rX[node_mask].flatten(), rE.flatten()]))
            worst = [max(worst[0], mx), max(worst[1], rms)]
            assert float((lE.cpu() * (rE == 0)).abs().max()) == 0.0
            assert torch.equal(lE, lE.transpose(1, 2))
        qX, qE = ex(B, N, 16), ex(B, N, N, 5)
        Xn, En, _, _, pX, pE = O.reverse_step(sd, cfg, tb, U, sched, X, E, node_mask, y, txt, t, qX, qE, return_probs=True)
    if regime == "throughput":
        assert _cabi.kernel_launches(_cabi.KERN_GEMM_2CTA) > k2, "qkv / fc1 must have run on the CTA-pair GEMM"
        if os.environ.get("LLB_FUSED_LN") != "0":
            assert _cabi.kernel_launches(_cabi.KERN_GEMM_LN_PAIR) > kp, "the block tails must have run on the fused GEMM + LayerNorm pair kernel"
    else:
        assert _cabi.kernel_launches(_cabi.KERN_GEMM_LN_PAIR) == kp, "the latency regime uses GEMM + row kernel tails"
        if os.environ.get("LLB_GRAPH") != "0" and "LLB_FUSED_LN" not in os.environ:
            assert eng.graph_state() == 1, "the second pass of the binding must have been replayed as a graph"
    print(f"\n[parity] N=128 denoiser at {rows} token rows (H=1024, depth 3) vs fp32 oracle: max|d|={worst[0]:.4f} rms={worst[1]:.5f}")
    assert worst[0] <= 0.10 and worst[1] <= 0.02, worst
    eng.set_state(*state_from_onehot(X, E))
    gpX, gpE = eng.step(t, 0, qX.to(DEV).contiguous(), qE.to(DEV).contiguous(), want_probs=True)
    gX, gE = eng.get_state()
    torch.cuda.synchronize()
    rXc, rEc = state_from_onehot(Xn, En)
    gX, gE = gX.cpu().long(), gE.cpu().long()
    assert torch.equal(gX == -1, rXc.long() == -1) and torch.equal(gE == -1, rEc.long() == -1)
    assert torch.equal(gE, gE.transpose(1, 2))
    gate = 4 * (2 * float(cfg["guide_scale"]) - 1) * worst[0]
    pair = node_mask.unsqueeze(1) & node_mask.unsqueeze(2) & torch.triu(torch.ones(N, N, dtype=torch.bool), 1)
    mX, mE = _margins(pX, qX, node_mask), _margins(pE, qE, pair)
    eqx, eqe = (gX == rXc.long())[node_mask], (gE == rEc.long())[pair]
    assert bool(eqx[mX > gate].all()) and bool(eqe[mE > gate].all()), (gate, float(eqx.float().mean()), float(eqe.float().mean()))
    agree = (int(eqx.sum()) + int(eqe.sum())) / (eqx.numel() + eqe.numel())
    dp = float((gpX.cpu() - pX)[node_mask].abs().max())
    record_parity(f"dit_128_atoms_{regime}_vs_oracle", token_rows=rows, depth=3, hidden=1024, logits_max_abs=worst[0], logits_rms=worst[1],
                  category_gate=gate, category_agreement=agree, max_prob_diff=dp)
    print(f"[parity] teacher-forced step: category agreement {agree:.5f}, gate {gate:.3f}, max |dp| {dp:.4f}")
    assert agree > 0.99


# ------------------------------------------------------------------------------------------------ GPU: switches and routing
def _attn2_run():
    """the sampled graphs and one pass's logits of an N = 100 checkpoint for a batch with molecules above 64 atoms"""
    cfg = synth.dit_config(256, 2, 4, 4.0, 20, 2.0)
    m, _, _ = _model(cfg, 100, seed=100)
    B = 5
    props, y, txt = _conditions(B, seed=77)
    n_nodes = torch.tensor([100, 3, 64, 65, 40])
    X, E, _ = m.generate_graphs(props, txt, -200, n_nodes=n_nodes, seed=5)
    eng = m.engine()
    lX, lE = eng.denoise(7, False)
    torch.cuda.synchronize()
    return {"X": X.cpu(), "E": E.cpu(), "lX": lX.cpu(), "lE": lE.cpu()}


@pytest.mark.gpu
def test_llb_attn_2_keeps_the_default_kernels_above_64_atoms():
    """LLB_ATTN=2 selects the tcgen05 attention only for batches of molecules of <= 64 atoms: here the default results"""
    if os.environ.get("LLB_ATTN"):
        pytest.skip("LLB_ATTN is set for this process")
    child = _child_run("_attn2_run", {"LLB_ATTN": "2"})
    here = _attn2_run()
    for k in here:
        assert torch.equal(here[k], child[k]), k


@pytest.mark.gpu
def test_a_checkpoint_above_64_atoms_trains_through_the_eager_loss():
    cfg = synth.dit_config(256, 2, 4, 4.0, 20, 2.0)
    m, _, _ = _model(cfg, 100, seed=101)
    m.train()
    assert not m.device_denoiser_ok()
    g = torch.Generator().manual_seed(3)
    sizes = [100, 1, 70, 12]
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
    graph = [torch.cat(xs).to(DEV), torch.cat(eis, 1).to(DEV), torch.cat(eas).to(DEV), torch.cat(bs).to(DEV)]
    props, txt = synth.dit_conditions(len(sizes), seed=9)
    txt = txt.to(DEV).requires_grad_(True)
    loss = m(*graph, props.to(DEV), txt, -200)
    loss.backward()
    assert torch.isfinite(loss) and txt.grad is not None and float(txt.grad.abs().sum()) > 0
    m.eval()
    X, E, n = m.generate_graphs(props.to(DEV), txt.detach(), -200, n_nodes=torch.tensor(sizes), seed=3)
    torch.cuda.synchronize()
    valid = torch.arange(100, device=DEV)[None] < n[:, None]
    assert bool((X[valid] >= 0).all()) and bool((X[~valid] == -1).all()) and torch.equal(E, E.transpose(1, 2))
