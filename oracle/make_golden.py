"""Generate tests/golden/*.pt by running the UNMODIFIED reference modules (needs LLAMOLE_REFERENCE_ROOT, see oracle/ref_import.py).

TEST INFRASTRUCTURE ONLY.  Usage:  LLAMOLE_REFERENCE_ROOT=<checkout> python -m oracle.make_golden  [--out tests/golden]

The reference has no tests or golden vectors of its own (SURVEY.md section 4), so the pin is made here:
the reference's GraphDiT / GraphCLIP / GraphPredictor are imported verbatim (oracle/ref_import.py),
constructed from a synthetic checkpoint directory (llamole_b200/synth.py), and run on seeded inputs
with pre-drawn Exp(1) noise.  Fixtures hold inputs + outputs + the seeds that regenerate the weights
(plus a checksum of those weights, so that a drift of the generator is detected, not hidden).
"""
from __future__ import annotations

import argparse
import hashlib
import os
import sys
import tempfile

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from llamole_b200 import synth  # noqa: E402
from oracle.ref_import import NoiseTape, load_reference, patched_multinomial  # noqa: E402

DIT_SMALL = dict(hidden=128, depth=2, heads=2, T=12, guide_scale=2.0, max_nodes=12, B=5,
                 n_nodes=[12, 3, 7, 1, 10], w_seed=1234, meta_seed=7, cond_seed=2024, noise_seed=99)
GIN_SMALL = dict(L=3, H=64, out_dim=300, n_graphs=7, graph_seed=3, enc_seed=11, pred_seed=13, c_seed=5)


def checksum(sd) -> float:
    return float(sum(v.double().abs().sum() for v in sd.values()))


def _sha256(t) -> str:
    return hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest()


def pack_meta(meta):
    """Compact form: transition_E (118 x 118 x 5 floats, a third of the fixture) is not stored.  load_fixture regenerates it
    from params["meta_seed"] and checks it against the SHA-256 of its float32 bytes kept here."""
    m = dict(meta)
    m["transition_E_sha256"] = _sha256(torch.tensor(m.pop("transition_E"), dtype=torch.float32))
    return m


def load_fixture(path):
    """A fixture written by this script, with the DiT meta back in the checkpoint's form (transition_E a nested list)."""
    fx = torch.load(path, weights_only=False)
    if "meta" in fx:
        P, m = fx["params"], dict(fx["meta"])
        trans = synth.dit_meta(P["max_nodes"], P["meta_seed"], min_nodes=1)["transition_E"]
        if _sha256(torch.tensor(trans, dtype=torch.float32)) != m.pop("transition_E_sha256"):
            raise AssertionError("synthetic meta generator drifted: transition_E differs from the one the fixture was made with")
        m["transition_E"] = trans
        fx["meta"] = m
    return fx


def exp_noise(g, *shape):
    return torch.empty(*shape).exponential_(1.0, generator=g)


def make_dit(out_dir):
    dm, du, _, _ = load_reference()
    P = DIT_SMALL
    cfg = synth.dit_config(P["hidden"], P["depth"], P["heads"], 4.0, P["T"], P["guide_scale"])
    meta = synth.dit_meta(P["max_nodes"], P["meta_seed"], min_nodes=1)
    sd = synth.dit_state_dict(cfg, P["max_nodes"], P["w_seed"])
    B, N, T = P["B"], P["max_nodes"], P["T"]
    with tempfile.TemporaryDirectory() as d:
        synth.write_dit_checkpoint(d, cfg, meta, sd)
        m = dm.GraphDiT(os.path.join(d, "config.yaml"), os.path.join(d, "data.meta.json"), torch.float32)
        m.init_model(d)
    m.eval()
    props, txt = synth.dit_conditions(B, P["cond_seed"])
    props[1, 5] = -200.0           # one extra missing property
    y = torch.where(props == -200.0, float("nan"), props)
    n_nodes = torch.tensor(P["n_nodes"])
    node_mask = torch.arange(N).unsqueeze(0) < n_nodes.unsqueeze(1)
    g = torch.Generator().manual_seed(P["noise_seed"])
    qX0, qE0 = exp_noise(g, B, N, 16), exp_noise(g, B, N, N, 5)
    qX, qE = exp_noise(g, T, B, N, 16), exp_noise(g, T, B, N, N, 5)

    draws = [qX0.reshape(B * N, 16), qE0.reshape(B * N * N, 5)]
    for s in reversed(range(T)):
        draws += [qX[s].reshape(B * N, 16), qE[s].reshape(B * N * N, 5)]
    tape = NoiseTape(draws)

    rec = {"logits": [], "probs": [], "cats": []}
    orig_forward = m._forward
    orig_sample = du.sample_discrete_features

    def fwd(noisy, text, unconditioned=False):
        pred = orig_forward(noisy, text, unconditioned=unconditioned)
        rec["logits"].append((pred.X.clone(), pred.E.clone()))
        return pred

    def samp(probX, probE, node_mask, step=None, add_nose=True):
        rec["probs"].append((probX.clone(), probE.clone()))
        out = orig_sample(probX, probE, node_mask, step=step, add_nose=add_nose)
        rec["cats"].append((out.X.clone(), out.E.clone()))
        return out

    m._forward = fwd
    du.sample_discrete_features = samp
    try:
        with torch.no_grad(), patched_multinomial(tape):
            z = du.sample_discrete_feature_noise(limit_dist=m.limit_dist, node_mask=node_mask)
            X, E = z.X, z.E
            X0, E0 = X.clone(), E.clone()
            states = []
            for s_int in reversed(range(T)):                     # diffusion_model.py:279-289
                s_arr = s_int * torch.ones((B, 1)).type_as(y)
                t_arr = s_arr + 1
                states.append((X.argmax(-1).to(torch.int8), E.argmax(-1).to(torch.int8)))
                one_hot, disc = m.sample_p_zs_given_zt(s_arr / T, t_arr / T, X, E, y, txt, node_mask)
                X, E = one_hot.X, one_hot.E
            final = one_hot.mask(node_mask, collapse=True)
    finally:
        m._forward = orig_forward
        du.sample_discrete_features = orig_sample
    assert tape.pos == len(draws)
    fx = {
        "params": P, "cfg": cfg, "meta": pack_meta(meta), "weights_checksum": checksum(sd),
        "props": props, "txt": txt, "n_nodes": n_nodes,
        "qX0": qX0, "qE0": qE0, "qX": qX, "qE": qE,
        "X_T": X0, "E_T": E0,
        # per step (in loop order t = T..1): cond logits, uncond logits, guided probs, sampled ints
        "logits_cond_X": torch.stack([rec["logits"][2 * i][0] for i in range(T)]),
        "logits_cond_E": torch.stack([rec["logits"][2 * i][1] for i in range(T)]),
        "logits_unc_X": torch.stack([rec["logits"][2 * i + 1][0] for i in range(T)]),
        "logits_unc_E": torch.stack([rec["logits"][2 * i + 1][1] for i in range(T)]),
        "prob_X": torch.stack([p[0] for p in rec["probs"]]),
        "prob_E": torch.stack([p[1] for p in rec["probs"]]),
        "cat_X": torch.stack([c[0] for c in rec["cats"]]).to(torch.int8),
        "cat_E": torch.stack([c[1] for c in rec["cats"]]).to(torch.int8),
        "final_X": final.X.to(torch.int8), "final_E": final.E.to(torch.int8),
        "schedule_betas": m.noise_schedule.betas.clone(), "schedule_abar": m.noise_schedule.alphas_bar.clone(),
        "x_marg": m.limit_dist.X.clone(), "e_marg": m.limit_dist.E.clone(),
        "xe": m.transition_model.xe_conditions.clone(), "ex": m.transition_model.u_ex[0].clone(),
    }
    torch.save(fx, os.path.join(out_dir, "dit_small.pt"))
    print("dit_small.pt", {k: tuple(v.shape) for k, v in fx.items() if torch.is_tensor(v)})


def make_gin(out_dir):
    _, _, ge, gp = load_reference()
    P = GIN_SMALL
    L, H, out_dim = P["L"], P["H"], P["out_dim"]
    x, ei, ea, batch = synth.molecular_graphs(P["n_graphs"], seed=P["graph_seed"], min_nodes=1, max_nodes=20)
    enc_sd, proj_sd = synth.gin_encoder_state_dicts(L, H, P["enc_seed"])
    pred_sd = synth.gin_predictor_state_dict(L, H, out_dim, seed=P["pred_seed"])
    cost_sd = synth.cost_mlp_state_dict()
    B = int(batch[-1]) + 1
    c = synth.text_conditions(B, P["c_seed"])

    clip = ge.GraphCLIP(L, H, 0.0, {})
    clip.molecule_encoder.load_state_dict(enc_sd)
    clip.molecule_projection.load_state_dict(proj_sd)
    clip.eval()
    pred = gp.GNNRetrosynthsizer(L, H, 768, 0.0, out_dim)
    pred.load_state_dict(pred_sd)
    pred.eval()
    cost = gp.CostMLP(1, 2048, 128, 0.1)
    cost.load_state_dict(cost_sd)
    cost.eval()
    fps = (torch.rand(4, 2048, generator=torch.Generator().manual_seed(1)) < 0.03).float()
    with torch.no_grad():
        emb = clip(x, ei, ea, batch)
        pooled = clip.molecule_encoder(x, ei, ea, batch)
        logits_c = pred(x, ei, ea, batch, c)
        logits_none = pred(x, ei, ea, batch, None)
        topv, topi = torch.topk(torch.softmax(logits_c, dim=1), k=10, dim=1)
        cost_out = cost(fps)
    fx = {
        "params": P, "enc_checksum": checksum(enc_sd) + checksum(proj_sd), "pred_checksum": checksum(pred_sd),
        "x": x, "edge_index": ei, "edge_attr": ea, "batch": batch, "c": c,
        "encoder_pooled": pooled, "encoder_embedding": emb,
        "predictor_logits": logits_c, "predictor_logits_dropped": logits_none,
        "topk_probs": topv, "topk_indices": topi, "fps": fps, "cost": cost_out,
    }
    torch.save(fx, os.path.join(out_dir, "gin_small.pt"))
    print("gin_small.pt", {k: tuple(v.shape) for k, v in fx.items() if torch.is_tensor(v)})


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden"))
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    torch.manual_seed(0)
    make_dit(a.out)
    make_gin(a.out)
