"""Times GraphDiT.forward + backward (the SFT decoder loss) at the checkpoint shape: the device denoiser against the eager
bf16 one in the same process, alternated.

    python tools/dit_grad_probe.py [--batches 6,16,64] [--reps 5] [--out result.json]

H = 1024, depth 28, 16 heads, N = 50, bf16 parameters (the reference loader's cast), frozen (disable_grads()), train mode;
node counts drawn from the node-count histogram.  One measurement = forward + backward of one loss into text_embedding, ended
by a device synchronise; the median over --reps alternated pairs is reported, with the saved-buffer and grad-blob sizes and the
card's name and power limit read in the same run.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from llamole_b200 import _cabi, synth  # noqa: E402
from llamole_b200.graph_decoder import GraphDiT  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="6,16,64")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    a = ap.parse_args()
    cfg = synth.dit_config()
    d = tempfile.mkdtemp()
    synth.write_dit_checkpoint(d, cfg, synth.dit_meta(50), synth.dit_state_dict(cfg, 50, seed=1))
    m = GraphDiT(os.path.join(d, "config.yaml"), os.path.join(d, "data.meta.json"), torch.bfloat16)
    m.init_model(d)
    m.disable_grads()
    for p in m.denoiser.parameters():
        p.data = p.data.to(torch.bfloat16)
    m = m.to("cuda").train()
    assert m.device_denoiser_ok()
    eager = lambda: False  # noqa: E731

    def batch(B, seed):
        g = torch.Generator().manual_seed(seed)
        sizes = m.sample_n_nodes(B, generator=g).clamp_min(1).tolist()
        act = m.active_index
        xs, eis, eas, bs, off = [], [], [], [], 0
        for b, n in enumerate(sizes):
            xs.append(act[torch.randint(0, act.numel(), (n,), generator=g)])
            src = torch.arange(n - 1) + off
            ea = torch.randint(1, 4, (n - 1,), generator=g)
            eis.append(torch.stack([torch.cat([src, src + 1]), torch.cat([src + 1, src])]))
            eas.append(torch.cat([ea, ea]))
            bs.append(torch.full((n,), b))
            off += n
        props, txt = synth.dit_conditions(B, seed=seed)
        return [t.cuda() for t in (torch.cat(xs), torch.cat(eis, 1), torch.cat(eas), torch.cat(bs), props)], txt.cuda(), sum(sizes)

    def once(graph, txt):
        tt = txt.to(torch.bfloat16).clone().requires_grad_(True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m(*graph, tt, -200).backward()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    res = {"card": card(), "shape": "H=1024 depth=28 heads=16 N=50 bf16", "batches": {}}
    for B in [int(x) for x in a.batches.split(",")]:
        graph, txt, atoms = batch(B, seed=B)
        for _ in range(2):   # warm-up of both paths (grad blob packing, first launches)
            once(graph, txt)
            m.device_denoiser_ok = eager
            once(graph, txt)
            del m.device_denoiser_ok
        dev_ms, eager_ms = [], []
        for _ in range(a.reps):
            dev_ms.append(once(graph, txt))
            m.device_denoiser_ok = eager
            eager_ms.append(once(graph, txt))
            del m.device_denoiser_ok
        sb = ctypes.c_size_t()
        _cabi.check(_cabi.lib().llb_dit_train_saved_bytes(ctypes.byref(m.engine().train_cfg), B, atoms, ctypes.byref(sb)), "saved")
        res["batches"][B] = {"atoms": atoms, "device_ms": statistics.median(dev_ms), "eager_ms": statistics.median(eager_ms),
                             "device_all": dev_ms, "eager_all": eager_ms, "saved_bytes": sb.value}
        print(B, res["batches"][B], flush=True)
    res["grad_blob_bytes"] = m.engine().grad_blob.numel()
    res["card_after"] = card()
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
