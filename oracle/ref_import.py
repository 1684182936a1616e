"""Import the reference's three hot-path packages VERBATIM from a checkout of the original Llamole repository.

TEST INFRASTRUCTURE ONLY (never imported by the product path).

Works only where LLAMOLE_REFERENCE_ROOT names such a checkout; the repository does not contain one.  Its one user is
oracle/make_golden.py, which writes tests/golden/*.pt (the stored reference outputs the suite compares against).
Nothing under tests/, smoke() or bench.py may call this.

The reference packages have no __init__.py; they import as namespace packages once
<checkout>/src/model is on sys.path (SURVEY.md section 8c).  torch_geometric / rdkit / rdchiral
need not be installed: where they are missing, the stand-ins under oracle/standins are put on sys.path first.
"""
from __future__ import annotations

import os
import sys
from contextlib import contextmanager

import torch

REFERENCE_ROOT = os.environ.get("LLAMOLE_REFERENCE_ROOT", "")
REFERENCE_MODEL_DIR = os.path.join(REFERENCE_ROOT, "src", "model")
_STANDINS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "standins")


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_MODEL_DIR, "graph_decoder"))


_cache = {}


def load_reference():
    """Returns (diffusion_model, diffusion_utils, graph_encoder.model, graph_predictor.model)."""
    if "mods" in _cache:
        return _cache["mods"]
    if not reference_available():
        raise FileNotFoundError(f"reference tree not found under {REFERENCE_ROOT!r}: set LLAMOLE_REFERENCE_ROOT to a checkout of the original Llamole repository")
    for name in ("torch_geometric", "rdkit", "rdchiral"):
        try:
            __import__(name)
        except Exception:
            if _STANDINS not in sys.path:
                sys.path.insert(0, _STANDINS)
    if REFERENCE_MODEL_DIR not in sys.path:
        sys.path.append(REFERENCE_MODEL_DIR)
    import graph_decoder.diffusion_model as dm  # type: ignore
    import graph_decoder.diffusion_utils as du  # type: ignore
    import graph_encoder.model as ge  # type: ignore
    import graph_predictor.model as gp  # type: ignore

    _cache["mods"] = (dm, du, ge, gp)
    return _cache["mods"]


class NoiseTape:
    """Pre-drawn Exp(1) noise consumed by a patched Tensor.multinomial.

    torch's multinomial(1) is argmax(p / q), q ~ Exp(1) (SURVEY.md section 8c, probed); replacing the
    draw of q by a recorded tensor makes the reference sampler a deterministic function of the tape.
    `draws` is a list of tensors consumed in call order; each must match the probability tensor's shape.
    """

    def __init__(self, draws):
        self.draws = list(draws)
        self.pos = 0

    def next(self, like):
        q = self.draws[self.pos]
        self.pos += 1
        assert tuple(q.shape) == tuple(like.shape), (q.shape, like.shape)
        return q.to(like.dtype)


@contextmanager
def patched_multinomial(tape: NoiseTape):
    orig = torch.Tensor.multinomial

    def _mn(self, num_samples, replacement=False, *, generator=None):
        assert num_samples == 1
        q = tape.next(self)
        return (self / q).argmax(dim=-1, keepdim=True)

    torch.Tensor.multinomial = _mn
    try:
        yield tape
    finally:
        torch.Tensor.multinomial = orig
