"""Every C-ABI entry's launch count (llb_gin_launch_count / llb_dit_launch_count: bench.py's gpu_launches) equals the number of
library kernels the CUDA profiler records for that call.  Copies, memsets and PyTorch's own kernels are not counted."""
import os
import tempfile

import pytest
import torch
from torch.autograd import DeviceType
from torch.profiler import ProfilerActivity, profile

from llamole_b200 import GraphCLIP, GraphPredictor, synth
from llamole_b200.graph_decoder import GraphDiT

DEV = "cuda:0"


def _library_kernel(name: str) -> bool:
    return not name.startswith(("Memcpy", "Memset")) and "at::" not in name


def _check(count, fn):
    """Runs fn under the profiler; the handle's launch-count delta must equal the library kernels the profiler saw."""
    torch.cuda.synchronize()
    n0 = count()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA and _library_kernel(e.name)]
    assert names, "the profiler recorded no library kernel"
    assert count() - n0 == len(names), (count() - n0, names)
    return out


def _graphs(num_graphs, seed, **kw):
    return [t.to(DEV) for t in synth.molecular_graphs(num_graphs, seed=seed, **kw)]


@pytest.fixture(scope="module")
def encoder():
    L, H = 3, 256
    enc, proj = synth.gin_encoder_state_dicts(L, H, seed=4)
    clip = GraphCLIP(L, H, 0.0, {})
    clip.molecule_encoder.load_state_dict(enc)
    clip.molecule_projection.load_state_dict(proj)
    return clip.to(DEV).engine()


def _predictor_engine(out_dim, seed):
    L, H = 3, 256
    gp = GraphPredictor(L, H, 0.0, out_dim, {}, {})
    gp.predictor.load_state_dict(synth.gin_predictor_state_dict(L, H, out_dim, seed=seed))
    gp.disable_grads()
    return gp.to(DEV).engine()


@pytest.fixture(scope="module")
def predictor():
    return _predictor_engine(777, seed=13)


@pytest.fixture(scope="module")
def dit():
    cfg = synth.dit_config(256, 2, 4, 4.0, 500, 2.0)
    d = tempfile.mkdtemp()
    synth.write_dit_checkpoint(d, cfg, synth.dit_meta(20, 7, 1), synth.dit_state_dict(cfg, 20, seed=27))
    m = GraphDiT(os.path.join(d, "config.yaml"), os.path.join(d, "data.meta.json"), torch.float32)
    m.init_model(d)
    m.disable_grads()
    return m.to(DEV).engine()


@pytest.mark.gpu
def test_gin_encoder_bind_and_forward(encoder):
    count = encoder.launch_count
    x, ei, ea, b = _graphs(96, seed=6)
    _check(count, lambda: encoder.bind(x, ei, ea, b, num_graphs=96, validate=False))
    _check(count, lambda: encoder.encoder_forward())


@pytest.mark.gpu
def test_gin_bind_without_edges(encoder):
    count = encoder.launch_count
    x, ei, ea, b = _graphs(12, seed=3, min_nodes=1, max_nodes=1)
    assert ea.numel() == 0
    _check(count, lambda: encoder.bind(x, ei, ea, b, num_graphs=12, validate=False))
    _check(count, lambda: encoder.encoder_forward())


@pytest.mark.gpu
def test_predictor_forward(predictor):
    x, ei, ea, b = _graphs(16, seed=7)
    c = synth.dit_conditions(16, seed=5)[1].to(DEV)
    _check(predictor.launch_count, lambda: predictor.bind(x, ei, ea, b, num_graphs=16, validate=False))
    _check(predictor.launch_count, lambda: predictor.predictor_forward(c))


@pytest.mark.gpu
def test_topk_materialised_below_16384_templates(predictor):
    x, ei, ea, b = _graphs(16, seed=8)
    c = synth.dit_conditions(16, seed=6)[1].to(DEV)
    predictor.bind(x, ei, ea, b, num_graphs=16, want_logits=True, validate=False)
    _check(predictor.launch_count, lambda: predictor.predictor_topk(c, 5))


@pytest.mark.gpu
def test_topk_fused_head():
    eng = _predictor_engine(16384, seed=17)
    B = 512
    x, ei, ea, b = _graphs(B, seed=9, min_nodes=5, max_nodes=20)
    c = synth.dit_conditions(B, seed=7)[1].to(DEV)
    eng.bind(x, ei, ea, b, num_graphs=B, want_logits=True, validate=False)
    _check(eng.launch_count, lambda: eng.predictor_topk(c, 10))
    assert eng.head_stats()["fused_rows"] == B


@pytest.mark.gpu
def test_predictor_saved_forward_and_backward(predictor):
    x, ei, ea, b = _graphs(16, seed=10)
    c = synth.dit_conditions(16, seed=8)[1].to(DEV)
    predictor.bind(x, ei, ea, b, num_graphs=16, validate=False)
    dlogits = torch.randn(16, 777, device=DEV)
    assert predictor.grad_blob is None   # the first backward packs the transposed weights too

    def fwd_bwd():
        _, saved, dims = predictor.predictor_forward_saved(c)
        return predictor.predictor_backward_c(c, dlogits, saved, dims)

    _check(predictor.launch_count, fwd_bwd)


@pytest.mark.gpu
def test_dit_begin_init_and_eager_step(dit):
    props, txt = synth.dit_conditions(3, seed=2)
    y = torch.where(props == -200.0, torch.full_like(props, float("nan")), props).to(DEV).contiguous()
    txt = txt.to(DEV).contiguous()
    n_nodes = torch.tensor([20, 5, 11], dtype=torch.int32)
    _check(dit.launch_count, lambda: dit.begin(n_nodes, y, txt))
    _check(dit.launch_count, lambda: dit.init_state(1, None, None))
    _check(dit.launch_count, lambda: dit.step(500, 1))   # the first pass after begin runs eagerly


@pytest.mark.gpu
def test_dit_denoise_c_and_backward_c(dit):
    B, N = 3, dit.N
    n_host = torch.tensor([20, 5, 11], dtype=torch.int32)
    g = torch.Generator().manual_seed(3)
    mask = torch.arange(N)[None, :] < n_host[:, None].long()
    X = torch.where(mask, torch.randint(0, 16, (B, N), generator=g), -1).to(torch.int8)
    e = torch.triu(torch.randint(0, 5, (B, N, N), generator=g), 1)
    pair = mask[:, :, None] & mask[:, None, :]
    E = torch.where(pair, e + e.transpose(1, 2), -1).to(torch.int8)
    c = torch.randn(B, dit.train_cfg.hidden, generator=g).to(DEV)
    dlX = torch.randn(B, N, 16, generator=g).to(DEV)
    dlE = torch.randn(B, N, N, 5, generator=g).to(DEV)
    count = lambda: int(dit.lib.llb_dit_launch_count(dit.train_handle)) if dit.train_handle else 0  # noqa: E731

    def fwd_bwd():
        _, _, saved = dit.denoise_c(X.to(DEV), E.to(DEV), n_host, c, True)
        return dit.backward_c(saved, (B, int(n_host.sum())), dlX, dlE)

    _check(count, fwd_bwd)
