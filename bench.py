#!/usr/bin/env python
"""Benchmark of the hot path: GraphDiT molecules/s (500-step sampling) and GIN graphs/s on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One JSON line on rank 0 (contract in the task statement / DESIGN.md section "Measurement"):
  * headline `value`  = GraphDiT molecules/s, whole job over all N GPUs, BASELINE.json configs[2]
    (multi-conditional 500-step reverse diffusion, batch 2048 per GPU, checkpoint shape H=1024 / depth 28 /
    heads 16 / 50 nodes / guide scale 2, random-init weights, synthetic conditions, every molecule at the full
    50 atoms).  A "step" is ONE reverse-diffusion step over the whole batch (conditional + unconditional denoiser
    pass, posterior, guidance, sampling); molecules/s = batch / (T * seconds per step).
  * `gin` sub-object = GraphCLIP encoder graphs/s over 4096 synthetic molecular graphs per GPU (configs[1]).
  * `e2e`            = the same metric through the public drop-in API with host buffers (H2D + D2H inside the
                       timed region).
  * `roofline`       = dominant kernel (live CUDA-event timing inside the timed region) against the measured peak.
  * `cpu_baseline`   = the CPU oracle (the reference's algorithm in PyTorch fp32) on the box's host cores.
`--impl reference` times that CPU implementation alone with the same metric/config keys.
`--dump-outputs DIR` writes what the timed paths returned in their last timed step (see dump_outputs); every input is seeded, so
two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "GraphDiT molecules/sec (500-step sampling) and GIN graphs/sec at 1/2/4/8 B200"
DIT = dict(hidden=1024, depth=28, heads=16, mlp_ratio=4.0, T=500, guide_scale=2.0, max_nodes=50)
GIN = dict(hidden=768, layers=5)
DUMP_MAX_BYTES = 64 << 20


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def dump_outputs(path, arrays):
    """Writes `arrays` (name -> tensor) as <path>/<name>.npy: float32, or float64 for integers float32 cannot hold exactly.  The
    default workload's outputs come to ~37 MB; when they exceed DUMP_MAX_BYTES in all, each array keeps a fixed, seeded sample of
    its rows (leading dimension), listed in <name>_rows.npy."""
    import numpy as np

    arrays = {k: (v.float() if v.is_floating_point() or int(v.abs().max()) < 2 ** 24 else v.double()) for k, v in arrays.items()}
    frac = min(1.0, 0.9 * DUMP_MAX_BYTES / sum(v.numel() * v.element_size() + 8 * v.shape[0] for v in arrays.values()))
    os.makedirs(path, exist_ok=True)
    for name, v in arrays.items():
        if frac < 1.0:
            rows = torch.randperm(v.shape[0], generator=torch.Generator().manual_seed(0))[: max(1, int(v.shape[0] * frac))].sort().values
            v = v[rows]
            np.save(os.path.join(path, f"{name}_rows.npy"), rows.double().numpy())
        np.save(os.path.join(path, f"{name}.npy"), v.numpy())
    log(f"[bench] wrote {', '.join(sorted(arrays))} to {path}" + (f" (row sample: {frac:.3f} of each)" if frac < 1.0 else ""))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], source="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


def ncu_traffic(slot):
    """DRAM bytes per launch of a kernel from the committed `ncu --set full` capture (profiles/traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))["bytes_per_launch"].get(slot)
    except Exception:
        return None


def dit_flops_per_pass(n_nodes, H=1024, D=28, d0=266):
    """Algorithmic FLOPs of one denoiser pass over molecules with n valid atoms each (SURVEY.md section 8d)."""
    n = n_nodes.double()
    per = D * (n * 24 * H * H + 4 * n * n * H + 14 * H * H) + n * (2 * d0 * H + 2 * H * H + 2 * d0 * H) + 2 * (256 * H + H * H) + 2 * (H * H + 2 * d0 * H)
    return float(per.sum())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(self.rows[0][1]), "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# model construction (synthetic weights of the checkpoint's shapes; no files except two tiny configs)
# ------------------------------------------------------------------------------------------------------
def build_dit(device, small=False):
    import yaml

    from llamole_b200 import GraphDiT, synth

    c = dict(DIT)
    if small:
        c.update(hidden=256, depth=2, heads=4)
    cfg = synth.dit_config(c["hidden"], c["depth"], c["heads"], c["mlp_ratio"], c["T"], c["guide_scale"])
    meta = synth.dit_meta(c["max_nodes"])
    d = tempfile.mkdtemp(prefix="llb_bench_")
    with open(os.path.join(d, "config.yaml"), "w") as f:
        yaml.safe_dump(cfg, f)
    with open(os.path.join(d, "data.meta.json"), "w") as f:
        json.dump(meta, f)
    m = GraphDiT(os.path.join(d, "config.yaml"), os.path.join(d, "data.meta.json"), torch.float32)
    sd = synth.dit_state_dict(cfg, c["max_nodes"], seed=1234)
    m.denoiser.load_state_dict(sd)
    m.disable_grads()
    return m.to(device), cfg, meta, sd


def build_gin(device):
    from llamole_b200 import GraphCLIP, synth

    enc, proj = synth.gin_encoder_state_dicts(GIN["layers"], GIN["hidden"], seed=11)
    g = GraphCLIP(GIN["layers"], GIN["hidden"], 0.0, {})
    g.molecule_encoder.load_state_dict(enc)
    g.molecule_projection.load_state_dict(proj)
    g.disable_grads()
    return g.to(device), enc, proj


# ------------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm on the host cores (oracle port; the verbatim reference when present)
# ------------------------------------------------------------------------------------------------------
def cpu_dit_step_seconds(cfg, meta, sd, B, steps, warmup):
    from llamole_b200 import synth
    from oracle import llamole_oracle as O

    torch.set_num_threads(os.cpu_count() or 1)
    tb = O.dit_tables(meta)
    U = O.union_transition(tb)
    T = cfg["diffusion_steps"]
    sched = O.cosine_schedule(T)
    N = tb.max_nodes
    props, txt = synth.dit_conditions(B)
    y = torch.where(props == -200.0, torch.full_like(props, float("nan")), props)
    node_mask = torch.ones(B, N, dtype=torch.bool)
    g = torch.Generator().manual_seed(5)
    ex = lambda *s: torch.empty(*s).exponential_(1.0, generator=g)  # noqa: E731
    X, E = O.initial_state(tb, node_mask, ex(B, N, 16), ex(B, N, N, 5), torch.float32)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            X, E, _, _ = O.reverse_step(sd, cfg, tb, U, sched, X, E, node_mask, y, txt, T - i, ex(B, N, 16), ex(B, N, N, 5))
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    return sum(times) / len(times)


def cpu_gin_seconds(enc, proj, graphs, reps=1):
    from oracle import llamole_oracle as O

    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        t0 = time.perf_counter()
        for _ in range(reps):
            O.gin_encoder_forward(enc, proj, GIN["layers"], *graphs)
        return (time.perf_counter() - t0) / reps


def run_reference(args, rank, world):
    """--impl reference: the CPU implementation of the path, same metric/config keys, rank 0 only."""
    if rank != 0:
        return
    from llamole_b200 import synth

    cfg = synth.dit_config(DIT["hidden"], DIT["depth"], DIT["heads"], DIT["mlp_ratio"], DIT["T"], DIT["guide_scale"])
    meta = synth.dit_meta(DIT["max_nodes"])
    sd = synth.dit_state_dict(cfg, DIT["max_nodes"], seed=1234)
    B = 16
    sec = cpu_dit_step_seconds(cfg, meta, sd, B, args.steps, args.warmup)
    val = B / (DIT["T"] * sec)
    enc, proj = synth.gin_encoder_state_dicts(GIN["layers"], GIN["hidden"], seed=11)
    graphs = synth.molecular_graphs(512, seed=0)
    gsec = cpu_gin_seconds(enc, proj, graphs, reps=args.steps)
    cores = torch.get_num_threads()
    sample = f"{B} of {args.dit_batch} molecules per step (one reverse step = cond+uncond denoiser pass + posterior + sampling), fp32, {cores} threads"
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "molecules/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": val, "unit": "molecules/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "molecules/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gin": {"value": 512 / gsec, "unit": "graphs/s", "sample": f"512 of 4096 graphs, mean of {args.steps} encoder forwards", "cores": cores},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def workload_config(args):
    return {
        "workload": "BASELINE.json configs[2]: GraphDiT multi-conditional (7 of 10 properties + text embedding) 500-step reverse "
                    "diffusion with classifier-free guidance, batch %d per GPU, all molecules at 50 atoms; a step = one reverse step "
                    "over the batch" % args.dit_batch,
        "dit": {"hidden": DIT["hidden"], "depth": DIT["depth"], "heads": DIT["heads"], "max_nodes": DIT["max_nodes"],
                "timesteps": DIT["T"], "guide_scale": DIT["guide_scale"], "batch_per_gpu": args.dit_batch, "weights": "random-init"},
        "gin_workload": "BASELINE.json configs[1]: GraphCLIP (GIN, H=768, L=5) forward over %d synthetic molecular graphs per GPU" % args.gin_graphs,
        "predictor_workload": "BASELINE.json configs[3]: A* candidate scoring, GIN predictor (H=768, L=5, %d templates) + top-50 over %d synthetic "
                              "reactant graphs per GPU (64k graphs batch-sharded over 8 GPUs)" % (args.pred_out_dim, args.pred_graphs),
        "l2": "activations per step (~7 GB) and GIN node matrices (~375 MB) exceed the 126 MB L2; no explicit flush",
        "parallelism": "dp%d (independent molecule/graph shards, one NCCL all-gather of results)" % args.gpus,
    }


# ------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed iterations of every timed loop, 1..500 (one sampling run has 500 reverse steps): the reverse steps of the "
                         "throughput, ragged and end-to-end DiT sections, the GIN forwards and the predictor passes.  Fixed counts: the "
                         "latency section times 200 steps per batch size, since one step there lasts 1.3-1.8 ms (--no-latency skips it), "
                         "and the CPU baseline of the B200 path samples 3 steps and one GIN forward, as its `sample` strings say")
    ap.add_argument("--warmup", type=int, default=3,
                    help="untimed steps before each timed loop.  The B200 path runs at least 3 (the first launches load modules and fill "
                         "the TMA descriptor cache), logs it when it raises the number and reports the number it ran")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dit-batch", type=int, default=2048)
    ap.add_argument("--gin-graphs", type=int, default=4096)
    ap.add_argument("--pred-graphs", type=int, default=8192, help="A* candidate scoring: reactant graphs per GPU (BASELINE.json configs[3]: 64k over 8 GPUs)")
    ap.add_argument("--pred-out-dim", type=int, default=180576)
    ap.add_argument("--no-predictor", action="store_true")
    ap.add_argument("--small", action="store_true", help="tiny model (debug only; invalid as a benchmark)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true", help="skip the small-batch latency section (profiler captures of the throughput step)")
    ap.add_argument("--only", default="", choices=["", "gin", "predictor"], help="development: time one GIN sub-benchmark alone and print its object")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the timed paths returned in their last step as DIR/<name>.npy (rank 0's shard): "
                         "the sampled graphs dit_X (B, N) and dit_E (B, N, N), gin_embedding, predictor_probs, predictor_indices")
    args = ap.parse_args()
    if not 1 <= args.steps <= DIT["T"] or args.warmup < 0:
        ap.error(f"--steps must be in 1..{DIT['T']} and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if args.warmup < 3:
        log(f"[bench] --warmup {args.warmup} raised to 3: the first launches load modules and fill the TMA descriptor cache")
        args.warmup = 3

    import torch.distributed as dist

    from llamole_b200 import _cabi, synth

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL_DEBUG (e.g. INFO, which the driver uses to count ranks) is left as the caller set it; NCCL prints to stdout by
        # default, which must stay ONE JSON line, so its log goes to stderr unless the caller chose a file
        if os.environ.get("NCCL_DEBUG") and not os.environ.get("NCCL_DEBUG_FILE"):
            os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"
        dist.init_process_group("nccl", device_id=device)
        log(f"[bench] rank {rank}/{world} on cuda:{local_rank}: NCCL process group initialised (nranks={world})")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    pk = peaks()
    T = DIT["T"]
    if args.only:
        fn = bench_gin if args.only == "gin" else bench_predictor
        out = fn(args, device, rank, world, barrier, max_over_ranks, pk)
        outputs = out.pop("_outputs")
        if rank == 0:
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, outputs)
            print(json.dumps(out), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    # ------------------------------------------------------------------ GraphDiT
    m, cfg, meta, sd = build_dit(device, small=args.small)
    eng = m.engine()
    latency = None if args.no_latency else bench_latency(args, m, eng, device, local_rank, pk, T)
    B = args.dit_batch
    N = m.max_n_nodes
    props_h, txt_h = synth.dit_conditions(B, seed=2024 + rank)
    props_h, txt_h = props_h.pin_memory(), txt_h.pin_memory()
    n_nodes = torch.full((B,), N, dtype=torch.int64)
    props_d = props_h.to(device)
    props_d = torch.where(props_d == -200.0, torch.full_like(props_d, float("nan")), props_d).contiguous()
    from llamole_b200 import sharding

    eng.begin(n_nodes.to(torch.int32), props_d, txt_h.to(device).contiguous(), mol_index_base=rank * B)
    eng.init_state(7, None, None)
    for i in range(args.warmup):
        eng.step(T - i, 7)
    n_dev = n_nodes.to(device)
    if world > 1:   # untimed: NCCL communicator / buffers of the one exchange of the path
        Xs, Es = eng.get_state()
        sharding.all_gather_rows(sharding.pack_graphs(Xs, Es, n_dev, check=False), sizes=[B] * world)
    barrier()
    launches0 = eng.launch_count()
    _cabi.profile_enable(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        ev0.record()
        for i in range(args.steps):
            eng.step(T - ((args.warmup + i) % T), 7)
        evc = torch.cuda.Event(enable_timing=True)
        evc.record()
        if world > 1:
            # the path's one exchange (once per sampling run), through the product API: the sampled graphs travel as the
            # packed byte rows of sharding.pack_graphs (1327 B per molecule) in ONE NCCL all-gather and are unpacked on arrival
            Xs, Es = eng.get_state()
            wire = sharding.all_gather_rows(sharding.pack_graphs(Xs, Es, n_dev, check=False), sizes=[B] * world)
            Xg, Eg, ng = sharding.unpack_graphs(wire, N)
            assert Xg.shape[0] == world * B
        ev1.record()
        barrier()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    comm_ms = max_over_ranks(evc.elapsed_time(ev1)) if world > 1 else 0.0
    comm_alone_ms = 0.0
    if world > 1:
        # inside the timed region the gather also absorbs the SKEW between the ranks (GPUs under the power cap differ by a few per cent
        # over a ~0.7 s region); the exchange on its own, from a barrier: pack + all-gather + unpack
        barrier()
        torch.cuda.synchronize()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        Xs, Es = eng.get_state()
        sharding.unpack_graphs(sharding.all_gather_rows(sharding.pack_graphs(Xs, Es, n_dev, check=False), sizes=[B] * world), N)
        eb.record()
        torch.cuda.synchronize()
        comm_alone_ms = max_over_ranks(ea.elapsed_time(eb))
    prof = _cabi.profile_read()
    _cabi.profile_enable(False)
    dit_launches = eng.launch_count() - launches0
    outputs = {}
    if args.dump_outputs:
        Xd, Ed = eng.get_state()    # the sampled graphs after the last timed step, as the step loop's caller reads them
        outputs.update(dit_X=Xd.cpu(), dit_E=Ed.cpu())
    ms_step = ms_total / args.steps
    value = world * B / (T * ms_step / 1e3)
    flops_step = 2 * dit_flops_per_pass(n_nodes, cfg["hidden_size"], cfg["depth"], 16 + 5 * N)
    step_frac = flops_step / (ms_step / 1e3) / (pk["tf_sustained"] * 1e12)
    # dominant kernel by total live time
    M_rows = 2 * int(n_nodes.sum())
    H, F = cfg["hidden_size"], int(cfg["hidden_size"] * cfg["mlp_ratio"])
    gemm_flops = {"gemm_qkv": 2.0 * M_rows * 3 * H * H, "gemm_proj": 2.0 * M_rows * H * H, "gemm_fc1": 2.0 * M_rows * F * H,
                  "gemm_fc2": 2.0 * M_rows * H * F}
    breakdown = {k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[1] / args.steps} for k, v in prof.items()}
    dom = max((k for k in prof if k in gemm_flops), key=lambda k: prof[k][0], default=None)
    roofline = None
    if dom:
        dur = prof[dom][0] / prof[dom][1] / 1e3
        ach = gemm_flops[dom] / dur / 1e12
        roofline = {"bound": "tensor", "kernel": f"gemm_tcgen05_kernel ({dom})", "achieved": ach, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                    "frac": ach / pk["tf_sustained"], "traffic": ncu_traffic(dom), "peak_source": pk["source"] + " (sustained: timed inside a long step)",
                    "launch_ms": dur * 1e3, "flops_per_launch": gemm_flops[dom],
                    "whole_step": {"flops_per_step": flops_step, "achieved": flops_step / (ms_step / 1e3) / 1e12, "frac": step_frac}}
    # the fused posterior + guidance + sampling kernel (K8-K10): HBM-bound by construction, a rounding error of the step.  Bytes per
    # molecule-step as implemented: both passes' raw output rows (2 n x 268 fp32) + the modulation rows + int8 state in and out.
    step_kernel = None
    if "dit_step" in prof:
        d0 = 16 + 5 * N
        sk_bytes = float(sum(2 * int(n) * (d0 + 2) * 4 for n in n_nodes)) + B * (2 * 2 * d0 * 4 + 2 * (N + N * N))
        sk_ms = prof["dit_step"][0] / prof["dit_step"][1]
        step_kernel = {"bound": "hbm", "kernel": "dit_step_kernel", "bytes_per_launch": sk_bytes, "launch_ms": sk_ms, "achieved": sk_bytes / (sk_ms / 1e3) / 1e9,
                       "peak": pk["hbm"], "unit": "GB/s", "frac": sk_bytes / (sk_ms / 1e3) / 1e9 / pk["hbm"], "share_of_step": sk_ms / ms_step,
                       "note": "latency-bound (one CTA per molecule, two 106 KB CTAs per SM), not bandwidth-bound: 1.3 % of the step"}
    # ------------------------------------------------------------------ e2e through the public API (host buffers)
    k_e2e = args.steps
    outX = torch.empty((B, N), dtype=torch.int64).pin_memory()
    outE = torch.empty((B, N, N), dtype=torch.int64).pin_memory()
    if world > 1:
        # every rank holds the conditions of the WHOLE job (world x B molecules, the same seeds on every rank) and calls the
        # product entry point: it samples its own shard and receives everybody's graphs through the packed all-gather
        parts = [synth.dit_conditions(B, seed=2024 + r) for r in range(world)]
        props_all = torch.cat([p for p, _ in parts]).pin_memory()
        txt_all = torch.cat([t for _, t in parts]).pin_memory()
        n_all = torch.full((world * B,), N, dtype=torch.int64)
    barrier()
    t0 = time.perf_counter()
    if world > 1:
        X, E, _ = sharding.sample_graphs_sharded(m.generate_graphs, props_all, txt_all, n_all, seed=7, steps=k_e2e)
        X, E = X[rank * B:(rank + 1) * B], E[rank * B:(rank + 1) * B]
    else:
        X, E, _ = m.generate_graphs(props_h, txt_h, -200, n_nodes=n_nodes, seed=7, steps=k_e2e, mol_index_base=rank * B)
    outX.copy_(X, non_blocking=True)
    outE.copy_(E, non_blocking=True)
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    e2e_val = world * B / (T * (e2e_ms / k_e2e) / 1e3)
    h2d = (props_h.numel() + txt_h.numel()) * 4 + B * 4
    d2h = (outX.numel() + outE.numel()) * 8
    e2e = {"value": e2e_val, "unit": "molecules/s", "h2d_bytes_per_step": h2d / k_e2e, "d2h_bytes_per_step": d2h / k_e2e,
           "note": (f"GraphDiT.generate_graphs(host tensors, steps={k_e2e}) + D2H of the integer graphs; one call's copies amortised over its {k_e2e} reverse steps"
                    if world == 1 else
                    f"sharding.sample_graphs_sharded(GraphDiT.generate_graphs, host tensors of all {world * B} molecules, steps={k_e2e}): own shard sampled, "
                    "all graphs gathered as packed byte rows over NCCL, + D2H of this rank's graphs")}
    del X, E
    # ------------------------------------------------------------------ the same batch size with ragged molecules
    # SURVEY.md section 8d asks for the padded-N figure (the headline above) AND the figure over actual n_i: node counts
    # drawn from the checkpoint's node-count histogram (synthetic: uniform on 5..N), useful FLOPs = valid tokens only.
    ragged = None
    if not args.small:
        n_rag = m.sample_n_nodes(B, generator=torch.Generator().manual_seed(77 + rank))
        eng.begin(n_rag.to(torch.int32), props_d, txt_h.to(device).contiguous(), mol_index_base=rank * B)
        eng.init_state(7, None, None)
        for i in range(args.warmup):
            eng.step(T - i, 7)
        barrier()
        k_rag = args.steps
        ev0.record()
        for i in range(k_rag):
            eng.step(T - ((args.warmup + i) % T), 7)
        ev1.record()
        barrier()
        rag_ms = max_over_ranks(ev0.elapsed_time(ev1)) / k_rag
        rag_flops = 2 * dit_flops_per_pass(n_rag, cfg["hidden_size"], cfg["depth"], 16 + 5 * N)
        ragged = {"value": world * B / (T * rag_ms / 1e3), "unit": "molecules/s", "ms_per_step": rag_ms, "steps": k_rag,
                  "mean_atoms": float(n_rag.double().mean()), "tokens_per_pass": int(n_rag.sum()),
                  "achieved_tflops": rag_flops / (rag_ms / 1e3) / 1e12, "frac_of_sustained": rag_flops / (rag_ms / 1e3) / (pk["tf_sustained"] * 1e12),
                  "note": "node counts ~ the (synthetic) checkpoint histogram, uniform on 5..N; varlen packing: only valid atoms are computed"}
    # ------------------------------------------------------------------ GIN encoder
    gin = bench_gin(args, device, rank, world, barrier, max_over_ranks, pk)
    outputs.update(gin.pop("_outputs"))
    pred = None
    if not args.no_predictor and not args.small:
        pred = bench_predictor(args, device, rank, world, barrier, max_over_ranks, pk)
        outputs.update(pred.pop("_outputs"))
    # ------------------------------------------------------------------ CPU baseline (rank 0, N=1)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.small:
        t0 = time.time()
        sec = cpu_dit_step_seconds(cfg, meta, sd, 16, 3, 1)
        cores = torch.get_num_threads()
        cpu = {"value": 16 / (T * sec), "unit": "molecules/s", "cores": cores, "kind": "port",
               "sample": f"16 of {B} molecules, 3 reverse steps after 1 warm-up ({sec:.2f} s/step), scaled to T={T}; oracle/llamole_oracle.py in fp32"}
        gin["cpu_baseline"] = gin_cpu_baseline(gin)
        if pred is not None:
            pred["cpu_baseline"] = predictor_cpu_baseline(args)
        log(f"cpu baseline took {time.time() - t0:.1f}s")
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        out = {
            "metric": METRIC, "value": value, "unit": "molecules/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": workload_config(args), "clocks": clocks.summary(), "e2e": e2e,
            "comm": {"backend": "nccl" if world > 1 else None, "nranks": world, "comm_ms": comm_ms, "comm_ms_per_step": comm_ms / args.steps,
                     "comm_alone_ms": comm_alone_ms,
                     "what": "one all-gather of the packed sampled graphs (sharding.pack_graphs, 1327 B/molecule) + unpack, once per sampling run; "
                             "comm_ms = from the last step's end to the gathered result inside the timed region (included in ms_per_step; it "
                             "absorbs the skew between the ranks), comm_alone_ms = the same exchange timed from a barrier" if world > 1
                             else "single GPU: no exchange"},
            "latency": latency, "sampling_kernel": step_kernel,
            "gpu_launches": int(dit_launches + gin.pop("_launches") + (pred.pop("_launches") if pred else 0)), "roofline": roofline,
            "cpu_baseline": cpu, "kernel_breakdown": breakdown, "ragged": ragged, "gin": gin, "predictor": pred,
        }
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def gin_cpu_baseline(gin):
    from llamole_b200 import synth

    enc, proj = synth.gin_encoder_state_dicts(GIN["layers"], GIN["hidden"], seed=11)
    graphs = synth.molecular_graphs(512, seed=0)
    sec = cpu_gin_seconds(enc, proj, graphs)
    return {"value": 512 / sec, "unit": "graphs/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": "first 512 of the 4096 graphs, one GraphCLIP forward, oracle/llamole_oracle.py in fp32"}


def predictor_cpu_baseline(args):
    """BASELINE.md section 4: the predictor on a 512-graph subset, oracle port in fp32 on the host cores; the head is evaluated on
    a 16 384-template slice of the weight and its time scaled to out_dim (a Linear's cost is proportional to its rows)."""
    from llamole_b200 import synth
    from oracle import llamole_oracle as O

    torch.set_num_threads(os.cpu_count() or 1)
    H, L, Ds = GIN["hidden"], GIN["layers"], 16384
    sd = synth.gin_predictor_state_dict(L, H, Ds, seed=13)
    x, ei, ea, b = synth.molecular_graphs(512, seed=100)
    c = synth.text_conditions(512, seed=7)
    with torch.no_grad():
        t0 = time.perf_counter()
        logits = O.gin_predictor_forward(sd, L, x, ei, ea, b, c)
        t_all = time.perf_counter() - t0
        hid = torch.randn(512, 4 * H)
        t0 = time.perf_counter()
        torch.nn.functional.linear(hid, sd["decoder.4.weight"], sd["decoder.4.bias"])
        t_head = time.perf_counter() - t0
        t0 = time.perf_counter()
        O.predictor_topk(logits, 50)
        t_topk = time.perf_counter() - t0
    scale = args.pred_out_dim / Ds
    sec = (t_all - t_head) + (t_head + t_topk) * scale
    return {"value": 512 / sec, "unit": "graphs/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"512 of {args.pred_graphs} graphs, one GNNRetrosynthsizer forward + softmax/top-50, oracle/llamole_oracle.py in fp32; head and top-k "
                      f"timed on {Ds} of the {args.pred_out_dim} templates and scaled by {scale:.2f} (trunk {t_all - t_head:.2f} s, head {t_head:.2f} s, top-k {t_topk:.2f} s)"}


def bench_predictor(args, device, rank, world, barrier, max_over_ranks, pk):
    """BASELINE.json configs[3]: reaction-template predictor (GIN trunk with text adapters + 4H head over out_dim templates)
    with the fused softmax/top-50, graphs resident in HBM; weak scaling (the same number of graphs on every GPU)."""
    from llamole_b200 import GraphPredictor, _cabi, synth

    H, L, D, k = GIN["hidden"], GIN["layers"], args.pred_out_dim, 50
    t0 = time.time()
    sd = synth.gin_predictor_state_dict(L, H, D, seed=13)
    m = GraphPredictor(L, H, 0.0, D, {"text_input_size": synth.TEXT_DIM}, {}, None)
    m.predictor.load_state_dict(sd)
    m.disable_grads()
    m = m.to(device)
    del sd
    G = args.pred_graphs
    x, ei, ea, batch = synth.molecular_graphs(G, seed=100 + rank)
    c = synth.text_conditions(G, seed=7 + rank).to(device)
    xd, eid, ead, bd = (t.to(device) for t in (x, ei, ea, batch))
    n, e = int(x.numel()), int(ea.numel())
    eng = m.engine()
    log(f"predictor set-up took {time.time() - t0:.1f}s")
    iters = args.steps
    for _ in range(args.warmup):
        eng.bind(xd, eid, ead, bd, num_graphs=G, want_logits=True, validate=False)
        probs, idx = eng.predictor_topk(c, k)
    barrier()
    l0 = eng.launch_count()
    _cabi.profile_enable(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(iters):
        eng.bind(xd, eid, ead, bd, num_graphs=G, want_logits=True, validate=False)
        probs, idx = eng.predictor_topk(c, k)
    if world > 1:   # the one exchange of the path: gather the candidates' top-k (product helper, one padded all-gather)
        from llamole_b200 import sharding

        sharding.all_gather_rows(torch.cat([probs, idx.to(torch.float32)], dim=1), sizes=[G] * world)
    ev1.record()
    barrier()
    ms = max_over_ranks(ev0.elapsed_time(ev1)) / iters
    prof = _cabi.profile_read()
    _cabi.profile_enable(False)
    launches = eng.launch_count() - l0
    outputs = {"predictor_probs": probs.cpu(), "predictor_indices": idx.cpu()} if args.dump_outputs else {}
    head_stats = eng.head_stats()
    # strong scaling of BASELINE.json configs[3]: 65 536 reactant graphs in total, 65 536 / N per GPU (the local batch repeated with
    # node offsets; same graph statistics), `--steps` timed passes of bind + top-50 + gather
    strong = None
    total_graphs = 65536
    if total_graphs % (world * G) == 0 or total_graphs // world >= G:
        reps_s = max(1, total_graphs // world // G)
        Gs = reps_s * G
        xs = xd.repeat(reps_s)
        eas = ead.repeat(reps_s)
        eis = torch.cat([eid + r * n for r in range(reps_s)], dim=1)
        bs = torch.cat([bd + r * G for r in range(reps_s)])
        cs = c.repeat(reps_s, 1)
        for _ in range(2):
            eng.bind(xs, eis, eas, bs, num_graphs=Gs, want_logits=True, validate=False)
            ps, is_ = eng.predictor_topk(cs, k)
        barrier()
        ev0.record()
        for _ in range(args.steps):
            eng.bind(xs, eis, eas, bs, num_graphs=Gs, want_logits=True, validate=False)
            ps, is_ = eng.predictor_topk(cs, k)
            if world > 1:
                sharding.all_gather_rows(torch.cat([ps, is_.to(torch.float32)], dim=1), sizes=[Gs] * world)
        ev1.record()
        barrier()
        ms_s = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
        strong = {"total_graphs": world * Gs, "graphs_per_gpu": Gs, "ms": ms_s, "value": world * Gs / (ms_s / 1e3), "unit": "graphs/s", "scaling": "strong",
                  "note": "fixed total of 65 536 candidate graphs split over the GPUs; compare `ms` across N"}
        del xs, eas, eis, bs, cs, ps, is_
    # e2e: host graphs + conditions -> top-k on the host
    xp, eip, eap, bp, cp = (t.pin_memory() for t in (x, ei, ea, batch, c.cpu()))
    hp = torch.empty((G, k), dtype=torch.float32).pin_memory()
    hi = torch.empty((G, k), dtype=torch.int32).pin_memory()
    barrier()
    t0 = time.perf_counter()
    reps = args.steps
    for _ in range(reps):
        pr, ix = m.topk_templates(xp.to(device, non_blocking=True), eip.to(device, non_blocking=True), eap.to(device, non_blocking=True),
                                  bp.to(device, non_blocking=True), cp.to(device, non_blocking=True), k)
        hp.copy_(pr, non_blocking=True)
        hi.copy_(ix, non_blocking=True)
        torch.cuda.synchronize()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / reps)
    trunk_flops = 16.0 * n * H * H * L + 16.0 * H * H * (L - 1) * G + 2.0 * G * 768 * 3 * H * L
    head_flops = (8.0 * H * H + 8.0 * H * D) * G
    head_ms = prof.get("gin_gemm_head", (0.0, 0))[0] / iters
    out = {
        "value": world * G / (ms / 1e3), "unit": "graphs/s", "ms_per_batch": ms, "graphs_per_gpu": G, "nodes": n, "directed_edges": e,
        "config": {"hidden": H, "layers": L, "out_dim": D, "topk": k,
                   "timed": "CSR build + predictor trunk + head + softmax/top-50, inputs resident in HBM" + (", + all_gather of the top-k" if world > 1 else "")},
        "e2e": {"value": world * G / (e2e_ms / 1e3), "unit": "graphs/s", "h2d_bytes_per_step": (n * 2 + e * 3) * 8 + G * 768 * 4,
                "d2h_bytes_per_step": G * k * 8},
        "roofline": {"bound": "tensor", "kernel": "gemm_tcgen05 (predictor head, 4H x out_dim)", "achieved": head_flops / (head_ms / 1e3) / 1e12 if head_ms else None,
                     "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": head_flops / (head_ms / 1e3) / 1e12 / pk["tf_sustained"] if head_ms else None,
                     "traffic": None, "peak_source": pk["source"], "flops_per_batch": head_flops, "whole_batch_tflops": (trunk_flops + head_flops) / (ms / 1e3) / 1e12},
        "kernel_breakdown": {k_: {"ms_per_batch": v[0] / iters, "launches": v[1] / iters} for k_, v in prof.items() if k_.startswith("gin_")},
        "strong_scaling": strong, "head": head_stats,
        "_launches": launches, "_outputs": outputs,
    }
    del m, eng
    torch.cuda.empty_cache()
    return out


def bench_latency(args, m, eng, device, local_rank, pk, T):
    """Latency regime (BASELINE.json configs[0]: B = 16; the reference's own call pattern: B = 6 = per_device_eval_batch_size of
    config/generate/*.yaml, modeling_llamole.py:653).  Measured BEFORE the throughput section: a handful of molecules never reaches
    the power cap, so the SM clock of this measurement should not be the capped one the long step leaves behind."""
    from llamole_b200 import synth

    if args.small:
        return None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    weight_bytes = sum(p.numel() for n_, p in m.denoiser.named_parameters() if p.dim() == 2) * 2    # bf16 GEMM operands streamed once per step
    floor_ms = weight_bytes / (pk["hbm"] * 1e9) * 1e3
    latency = {"weight_bytes": weight_bytes, "weight_streaming_floor_ms": floor_ms, "batches": {}}
    for Bl in (6, 16):
        pl, tl = synth.dit_conditions(Bl, seed=900 + Bl)
        pl = torch.where(pl == -200.0, torch.full_like(pl, float("nan")), pl).to(device).contiguous()
        n_l = m.sample_n_nodes(Bl, generator=torch.Generator().manual_seed(5 + Bl)).clamp_(min=10)
        eng.begin(n_l.to(torch.int32), pl, tl.to(device).contiguous(), mol_index_base=0)
        eng.init_state(7, None, None)
        for i in range(20):
            eng.step(T - i, 7)
        torch.cuda.synchronize()
        k_lat = 200
        with ClockSampler(local_rank) as clk:
            ev0.record()
            for i in range(k_lat):
                eng.step(T - 20 - i, 7)
            ev1.record()
            torch.cuda.synchronize()
        ms_l = ev0.elapsed_time(ev1) / k_lat
        latency["batches"][str(Bl)] = {"ms_per_step": ms_l, "molecules_per_s": Bl / (T * ms_l / 1e3), "token_rows": 2 * int(n_l.sum()),
                                       "floor_frac": floor_ms / ms_l, "steps": k_lat, "graph_replay": eng.graph_state() == 1,
                                       "sm_mhz": clk.summary().get("sm_mhz")}
    latency["note"] = ("one reverse step (cond + uncond pass batched, posterior, sampling) at the reference's per-prompt batch sizes, measured "
                       "before the throughput section; floor = streaming the bf16 weights once per step at the measured HBM peak")
    return latency


def bench_gin(args, device, rank, world, barrier, max_over_ranks, pk):
    from llamole_b200 import _cabi, synth

    g, enc, proj = build_gin(device)
    G = args.gin_graphs
    x, ei, ea, batch = synth.molecular_graphs(G, seed=rank)
    xd, eid, ead, bd = (t.to(device) for t in (x, ei, ea, batch))
    n, e = int(x.numel()), int(ea.numel())
    eng = g.engine()
    iters = args.steps
    for _ in range(args.warmup):
        eng.bind(xd, eid, ead, bd, num_graphs=G, validate=False)
        out = eng.encoder_forward()
    barrier()
    l0 = eng.launch_count()
    _cabi.profile_enable(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(iters):
        eng.bind(xd, eid, ead, bd, num_graphs=G, validate=False)
        out = eng.encoder_forward()
    ev1.record()
    barrier()
    ms = max_over_ranks(ev0.elapsed_time(ev1)) / iters
    prof = _cabi.profile_read()
    _cabi.profile_enable(False)
    launches = eng.launch_count() - l0
    outputs = {"gin_embedding": out.cpu()} if args.dump_outputs else {}
    H, L = GIN["hidden"], GIN["layers"]
    agg_bytes = (e + 2 * n) * H * 2      # per layer launch (SURVEY.md section 8d: gathered neighbours + self, bf16, + output)
    agg_ms = prof["gin_aggregate"][0] / prof["gin_aggregate"][1]
    mlp_flops = 16.0 * n * H * H * L + 16.0 * H * H * (L - 1) * G + 4.0 * H * H * G
    gemm_ms = sum(prof[k][0] for k in ("gin_gemm_mlp0", "gin_gemm_mlp4") if k in prof) / iters
    # e2e: host int64 tensors -> embeddings on the host
    xp, eip, eap, bp = (t.pin_memory() for t in (x, ei, ea, batch))
    host_out = torch.empty((G, H), dtype=torch.float32).pin_memory()
    emb = g(xp.to(device, non_blocking=True), eip.to(device, non_blocking=True), eap.to(device, non_blocking=True), bp.to(device, non_blocking=True))
    host_out.copy_(emb)   # one untimed call: allocator / pinned-copy warm-up
    barrier()
    t0 = time.perf_counter()
    reps = args.steps
    for _ in range(reps):
        emb = g(xp.to(device, non_blocking=True), eip.to(device, non_blocking=True), eap.to(device, non_blocking=True), bp.to(device, non_blocking=True))
        host_out.copy_(emb, non_blocking=True)
        torch.cuda.synchronize()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / reps)
    return {
        "value": world * G / (ms / 1e3), "unit": "graphs/s", "ms_per_forward": ms, "graphs_per_gpu": G, "nodes": n, "directed_edges": e,
        "config": {"hidden": H, "layers": L, "timed": "CSR build (llb_gin_bind) + GraphCLIP forward, inputs resident in HBM"},
        "e2e": {"value": world * G / (e2e_ms / 1e3), "unit": "graphs/s", "h2d_bytes_per_step": (n * 2 + e * 3) * 8, "d2h_bytes_per_step": G * H * 4},
        "roofline": {"bound": "hbm", "kernel": "gin_aggregate_wide_kernel", "achieved": agg_bytes / (agg_ms / 1e3) / 1e9, "peak": pk["hbm"],
                     "unit": "GB/s", "frac": agg_bytes / (agg_ms / 1e3) / 1e9 / pk["hbm"], "traffic": ncu_traffic("gin_aggregate"), "launch_ms": agg_ms,
                     "bytes_per_launch": agg_bytes, "peak_source": pk["source"]},
        "mlp_gemms": {"tflops": mlp_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms else None, "frac_of_sustained": mlp_flops / (gemm_ms / 1e3) / 1e12 / pk["tf_sustained"] if gemm_ms else None,
                      "ms_per_forward": gemm_ms,
                      "note": "algorithmic FLOPs of the node / virtual-node / projection MLPs (SURVEY.md 8d) over the time of the mlp0 and mlp4 slots; the "
                              "mlp4 slot is the fused GEMM + layer-tail kernel, the statistics GEMM of the analytic LayerNorm (gin_gemm_stats) is extra work"},
        "whole_forward": {"tflops": mlp_flops / (ms / 1e3) / 1e12, "frac_of_sustained": mlp_flops / (ms / 1e3) / 1e12 / pk["tf_sustained"],
                          "note": "algorithmic MLP FLOPs over the whole forward (CSR build, aggregation, GEMMs, pooling, head)"},
        "kernel_breakdown": {k: {"ms_per_forward": v[0] / iters, "launches": v[1] / iters} for k, v in prof.items()},
        "_launches": launches, "_outputs": outputs,
    }


if __name__ == "__main__":
    main()
