import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def load_golden(name):
    from oracle.make_golden import load_fixture

    return load_fixture(os.path.join(GOLDEN, name))


@pytest.fixture(scope="session")
def dit_small():
    return load_golden("dit_small.pt")


@pytest.fixture(scope="session")
def gin_small():
    return load_golden("gin_small.pt")


def record_parity(name, **metrics):
    """Append one measured parity result to gpurun_out/parity.json (or $LLB_PARITY_OUT): the numbers DESIGN.md quotes are
    kept as an artefact of the run that produced them (copied to profiles/parity_r*.json)."""
    import json

    path = os.environ.get("LLB_PARITY_OUT", os.path.join(ROOT, "gpurun_out", "parity.json"))
    try:
        os.makedirs(os.path.dirname(path), exist_ok=True)
        data = json.load(open(path)) if os.path.exists(path) else {}
        data[name] = {k: (float(v) if isinstance(v, (int, float)) else v) for k, v in metrics.items()}
        with open(path, "w") as f:
            json.dump(data, f, indent=1, sort_keys=True)
    except Exception:
        pass
