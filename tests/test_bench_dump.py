"""bench.py --dump-outputs: the arrays the timed paths returned, written as float32 / float64 .npy files under a size cap, and the
same files from two runs with the same arguments."""
import importlib.util
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("llb_bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_writes_float_arrays_and_samples_rows_above_the_cap(monkeypatch):
    bench = _bench()
    arrays = {"E": torch.randint(0, 5, (40, 6, 6), dtype=torch.int8), "emb": torch.randn(10, 3),
              "idx": torch.tensor([[0, 2 ** 24 + 1]], dtype=torch.int64)}
    with tempfile.TemporaryDirectory() as d:
        bench.dump_outputs(d, arrays)
        assert sorted(os.listdir(d)) == ["E.npy", "emb.npy", "idx.npy"]
        E, emb, idx = (np.load(os.path.join(d, f"{k}.npy")) for k in ("E", "emb", "idx"))
        assert E.dtype == np.float32 and np.array_equal(E, arrays["E"].float().numpy())
        assert emb.dtype == np.float32 and np.array_equal(emb, arrays["emb"].numpy())
        assert idx.dtype == np.float64 and idx[0, 1] == 2 ** 24 + 1
    cap = 2000
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", cap)
    runs = []
    for _ in range(2):
        with tempfile.TemporaryDirectory() as d:
            bench.dump_outputs(d, arrays)
            files = {f: np.load(os.path.join(d, f)) for f in os.listdir(d)}
            assert sum(a.nbytes for a in files.values()) <= cap and all(a.dtype in (np.float32, np.float64) for a in files.values())
            runs.append(files)
    assert runs[0].keys() == runs[1].keys() and all(np.array_equal(runs[0][f], runs[1][f]) for f in runs[0])
    rows = runs[0]["E_rows.npy"].astype(np.int64)
    assert 0 < len(rows) < 40 and np.all(np.diff(rows) > 0)
    assert np.array_equal(runs[0]["E.npy"], arrays["E"].float().numpy()[rows])


@pytest.mark.gpu
def test_bench_dump_is_what_the_timed_paths_return_and_identical_across_runs():
    B, G, warmup, steps = 64, 256, 3, 2
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--small", "--steps", str(steps), "--warmup", str(warmup), "--dit-batch", str(B),
           "--gin-graphs", str(G)]
    dumps = []
    with tempfile.TemporaryDirectory() as d:
        for i in range(2):
            out = os.path.join(d, str(i))
            r = subprocess.run(cmd + ["--dump-outputs", out], capture_output=True, text=True, timeout=900, cwd=ROOT)
            assert r.returncode == 0, r.stderr[-3000:]
            line = [l for l in r.stdout.splitlines() if l.startswith("{")]
            assert len(line) == 1 and json.loads(line[0])["steps"] == steps
            dumps.append({f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out)})
    a, b = dumps
    assert sorted(a) == ["dit_E", "dit_X", "gin_embedding"]
    assert a["dit_X"].shape == (B, 50) and a["dit_E"].shape == (B, 50, 50) and a["gin_embedding"].shape == (G, 768)
    assert all(v.dtype == np.float32 for v in a.values())
    assert all(np.array_equal(a[k], b[k]) for k in a)

    # the sampled graphs: atom classes 0..15, bond classes 0..4 off the diagonal, symmetric, and exactly the state that the same
    # reverse steps (warm-up, then the timed ones) leave through the product API
    X, E = a["dit_X"], a["dit_E"]
    off = ~np.eye(50, dtype=bool)
    assert X.min() >= 0 and X.max() <= 15 and len(np.unique(X)) > 1
    assert E[:, off].min() >= 0 and E[:, off].max() <= 4 and len(np.unique(E[:, off])) > 1
    assert np.array_equal(E, E.transpose(0, 2, 1))
    from llamole_b200 import synth
    from oracle import llamole_oracle as O

    bench = _bench()
    dev = torch.device("cuda", 0)
    m, cfg, _, _ = bench.build_dit(dev, small=True)
    T, N = cfg["diffusion_steps"], m.max_n_nodes
    props, txt = synth.dit_conditions(B, seed=2024)
    props = torch.where(props == -200.0, torch.full_like(props, float("nan")), props)
    eng = m.engine()
    eng.begin(torch.full((B,), N, dtype=torch.int32), props.to(dev).contiguous(), txt.to(dev).contiguous(), mol_index_base=0)
    eng.init_state(7, None, None)
    for i in range(warmup + steps):
        eng.step(T - i, 7)
    Xs, Es = eng.get_state()
    assert np.array_equal(X, Xs.cpu().float().numpy()) and np.array_equal(E, Es.cpu().float().numpy())

    # the GIN embeddings against the CPU oracle on the benchmark's graphs and weights
    enc, proj = synth.gin_encoder_state_dicts(bench.GIN["layers"], bench.GIN["hidden"], seed=11)
    with torch.no_grad():
        ref = O.gin_encoder_forward(enc, proj, bench.GIN["layers"], *synth.molecular_graphs(G, seed=0))
    emb = torch.from_numpy(a["gin_embedding"])
    cos = float(torch.nn.functional.cosine_similarity(emb.double(), ref.double(), dim=1).min())
    assert float((emb - ref).abs().max()) <= 3e-3 and cos > 0.9995
