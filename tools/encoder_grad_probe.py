"""Times GraphCLIP's forward + backward with respect to its parameters on the B200 (not part of bench.py).

    python tools/encoder_grad_probe.py [--out result.json] [--reps 5] [--inner 3]

At the benchmark's encoder shape (H = 768, L = 5) and for 256 and 4096 synthetic molecular graphs, reports the medians over
`--reps` alternated repetitions (each of `--inner` calls, timed with CUDA events) of
  * the no-grad forward (the path of a frozen encoder),
  * forward + backward through GraphCLIP (saved forward, then every parameter's gradient on the device),
  * forward + backward of the oracle (oracle/llamole_oracle.py) run eagerly on the GPU in bf16 with torch autograd;
the saved-buffer size; and the GPU's name and power limit, read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from llamole_b200 import GraphCLIP, synth  # noqa: E402
from oracle import llamole_oracle as O  # noqa: E402


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
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--inner", type=int, default=3)
    args = ap.parse_args()
    H, L = 768, 5
    dev = torch.device("cuda:0")
    enc, proj = synth.gin_encoder_state_dicts(L, H, seed=11)
    m = GraphCLIP(L, H, 0.0, {})
    m.molecule_encoder.load_state_dict(enc)
    m.molecule_projection.load_state_dict(proj)
    m = m.to(dev)
    # the eager reference in bf16 on the same device, parameters as leaves
    e16 = {k: v.to(dev, torch.bfloat16).requires_grad_(True) if v.is_floating_point() else v.to(dev) for k, v in enc.items()}
    p16 = {k: v.to(dev, torch.bfloat16).requires_grad_(True) for k, v in proj.items()}
    result = {"H": H, "L": L, **gpu_info(), "cases": []}
    for B in (256, 4096):
        graph = tuple(t.to(dev) for t in synth.molecular_graphs(B, seed=100))
        G = torch.randn(B, H, device=dev)
        eng = m.engine()

        def frozen():
            with torch.no_grad():
                eng.bind(*graph, validate=False)
                eng.encoder_forward()

        def ours():
            (m(*graph) * G).sum().backward()

        def oracle():
            with torch.device(dev):   # the oracle allocates its pooling buffers on the default device
                (O.gin_encoder_forward(e16, p16, L, *graph).float() * G).sum().backward()

        for fn in (frozen, ours, oracle):   # warm every shape
            fn()
        torch.cuda.synchronize()

        def timed(fn):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.inner):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / args.inner

        t_f, t_o, t_r = [], [], []
        for _ in range(args.reps):   # alternated: every repetition times the three back to back
            t_f.append(timed(frozen))
            t_o.append(timed(ours))
            t_r.append(timed(oracle))
        eng.bind(*graph)
        _, saved, dims = eng.encoder_forward_saved()
        case = {"graphs": B, "nodes": dims[0], "edges": dims[1], "forward_nograd_ms": statistics.median(t_f),
                "forward_backward_ms": statistics.median(t_o), "oracle_bf16_eager_forward_backward_ms": statistics.median(t_r),
                "saved_bytes": int(saved.numel()),
                "spread_ms": {"forward_nograd": [min(t_f), max(t_f)], "forward_backward": [min(t_o), max(t_o)],
                              "oracle": [min(t_r), max(t_r)]}}
        del saved
        result["cases"].append(case)
        print(json.dumps(case), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k != "cases"}))


if __name__ == "__main__":
    main()
