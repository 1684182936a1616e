"""Times GraphDiT reverse steps of a checkpoint with molecules of 128 atoms against one with 50, at equal token counts.

    python tools/dit_large_n_probe.py [--reps 5] [--steps 3] [--out result.json]

Checkpoint block shape (H = 1024, depth 28, 16 heads, synthetic weights), guidance scale 2:
  - N = 50:  2048 molecules of 50 atoms (102 400 token rows per pass; the benchmark's throughput shape);
  - N = 128: 800 molecules of 128 atoms (102 400 token rows per pass: 128-row attention tile, step kernel with T in global memory);
  - N = 128: 6 molecules of 128 atoms (the latency regime: graph-replayed passes).
One measurement = --steps consecutive reverse steps ended by a device synchronise; the throughput shapes are alternated and the
median over --reps is reported, as ms per step and ms per 1000 token rows of one pass.  A separate profiled step of each shape
gives the per-slot kernel times of llb_profile_* (attention, dit_step, the GEMM slots).  The card's name and power limit are read
in the same run.
"""
import argparse
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


def model(N, seed):
    cfg = synth.dit_config()
    d = tempfile.mkdtemp()
    synth.write_dit_checkpoint(d, cfg, synth.dit_meta(N), synth.dit_state_dict(cfg, N, seed=seed))
    m = GraphDiT(os.path.join(d, "config.yaml"), os.path.join(d, "data.meta.json"), torch.float32)
    m.init_model(d)
    m.disable_grads()
    return m.to("cuda")


class Shape:
    def __init__(self, name, m, B, n):
        self.name, self.m, self.B, self.n = name, m, B, n
        self.eng = m.engine()
        props, txt = synth.dit_conditions(B, seed=B)
        self.props = torch.where(props == -200.0, torch.full_like(props, float("nan")), props).cuda().contiguous()
        self.txt = txt.cuda().contiguous()
        self.t = m.T

    def bind(self):
        self.eng.begin(torch.full((self.B,), self.n, dtype=torch.int32), self.props, self.txt)
        self.eng.init_state(7, None, None)
        self.t = self.m.T

    def run(self, steps):
        """ms per reverse step over `steps` consecutive steps (rebinding when the schedule runs out)"""
        if self.t - steps < 1:
            self.bind()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.eng.step(self.t, 7)
            self.t -= 1
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    a = ap.parse_args()
    res = {"card": card(), "shape": "H=1024 depth=28 heads=16 guide_scale=2", "shapes": {}}
    m50, m128 = model(50, 1), model(128, 2)
    shapes = [Shape("N=50 B=2048 n=50", m50, 2048, 50), Shape("N=128 B=800 n=128", m128, 800, 128)]
    latency = Shape("N=128 B=6 n=128", m128, 6, 128)
    times = {s.name: [] for s in shapes + [latency]}
    for s in shapes + [latency]:   # one binding per shape at a time: the engines' workspaces are per model
        s.bind()
        s.run(2)   # warm-up: first launches, shared-memory limits, the latency regime's graph capture
    for _ in range(a.reps):
        for s in shapes:   # alternated
            s.bind()
            times[s.name].append(s.run(a.steps))
    latency.bind()
    latency.run(2)
    for _ in range(a.reps):
        times[latency.name].append(latency.run(10 * a.steps))
    for s in shapes + [latency]:
        s.bind()
        s.run(1)
        _cabi.profile_read()
        _cabi.profile_enable(True)
        try:
            s.run(1)
            slots = _cabi.profile_read()
        finally:
            _cabi.profile_enable(False)
        med = statistics.median(times[s.name])
        rows = s.B * s.n
        res["shapes"][s.name] = {"token_rows_per_pass": rows, "ms_per_step": med, "ms_per_1000_rows": med * 1e3 / rows,
                                 "all_ms_per_step": times[s.name], "profiled_slots_ms": {k: v[0] for k, v in slots.items()},
                                 "profiled_slots_launches": {k: v[1] for k, v in slots.items()}}
        print(s.name, json.dumps(res["shapes"][s.name]), flush=True)
    r50, r128 = (res["shapes"][s.name]["ms_per_1000_rows"] for s in shapes)
    res["ratio_ms_per_1000_rows_N128_over_N50"] = r128 / r50
    res["card_after"] = card()
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
