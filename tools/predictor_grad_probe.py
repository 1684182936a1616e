"""Times the predictor's backward with respect to c on the B200 (not part of bench.py).

    python tools/predictor_grad_probe.py [--out result.json] [--reps 7] [--inner 5]

At the benchmark's predictor shape (H = 768, L = 5, out_dim = 180 576) and for B = 16 and B = 256 product graphs, reports the
no-grad forward, the saved forward (same logits, plus what the backward needs) and the backward, each the median over `--reps`
alternated repetitions of `--inner` calls timed with CUDA events; the grad blob and saved-buffer sizes; and the GPU's name and
power limit, read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from llamole_b200 import GraphPredictor, synth  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return {"gpu": name, "power_limit": power}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--inner", type=int, default=5)
    ap.add_argument("--out-dim", type=int, default=180576)
    args = ap.parse_args()
    H, L, D = 768, 5, args.out_dim
    dev = torch.device("cuda:0")
    sd = synth.gin_predictor_state_dict(L, H, D, seed=13)
    m = GraphPredictor(L, H, 0.0, D, {"text_input_size": synth.TEXT_DIM}, {}, None)
    m.predictor.load_state_dict(sd)
    m.disable_grads()
    m = m.to(dev)
    del sd
    eng = m.engine()
    result = {"H": H, "L": L, "out_dim": D, **gpu_info(), "cases": []}
    for B in (16, 256):
        x, ei, ea, b = (t.to(dev) for t in synth.molecular_graphs(B, seed=100))
        c = synth.text_conditions(B, seed=7).to(dev)
        dlogits = torch.randn(B, D, device=dev) * 1e-3
        eng.bind(x, ei, ea, b)
        logits, saved, dims = eng.predictor_forward_saved(c)
        eng.predictor_backward_c(c, dlogits, saved, dims)   # packs the grad blob, warms every shape
        eng.predictor_forward(c)
        torch.cuda.synchronize()

        def timed(fn):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.inner):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / args.inner

        t_fwd, t_saved, t_bwd = [], [], []
        for _ in range(args.reps):   # alternated: every repetition times the three calls back to back
            t_fwd.append(timed(lambda: eng.predictor_forward(c)))
            t_saved.append(timed(lambda: eng.predictor_forward_saved(c)))
            t_bwd.append(timed(lambda: eng.predictor_backward_c(c, dlogits, saved, dims)))
        case = {"B": B, "nodes": dims[0], "edges": dims[1], "forward_ms": statistics.median(t_fwd),
                "forward_saved_ms": statistics.median(t_saved), "backward_ms": statistics.median(t_bwd),
                "grad_blob_bytes": int(eng.grad_blob.numel()), "saved_bytes": int(saved.numel()),
                "spread_ms": {"forward": [min(t_fwd), max(t_fwd)], "forward_saved": [min(t_saved), max(t_saved)],
                              "backward": [min(t_bwd), max(t_bwd)]}}
        result["cases"].append(case)
        print(json.dumps(case), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k != "cases"}))


if __name__ == "__main__":
    main()
