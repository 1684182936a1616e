"""Batched A* expansion (llamole_b200/planner.py, SURVEY.md section 8f-1): with beam = 1 it is the reference's search loop
(planner/molstar.py:11-76) -- checked against a literal restatement of that loop on a stand-in tree; with beam > 1 the
expansions and the value evaluations arrive in batches."""
import hashlib

import numpy as np
import pytest

from llamole_b200.planner import ValueCache, molstar_batched, predictor_expand_batch_fn


def _h(*parts) -> int:
    return int(hashlib.sha256("|".join(str(p) for p in parts).encode()).hexdigest()[:12], 16)


class Network:
    """Synthetic retrosynthesis network: molecule "m<i>" has 0-3 deterministic reactions to molecules with larger indices."""

    def __init__(self, seed, n_mols=60, n_start=14):
        self.seed, self.n = seed, n_mols
        self.starting = {f"m{i}" for i in range(n_mols) if _h(seed, "start", i) % n_mols < n_start and i > 3}
        self.expand_calls, self.value_calls = [], []

    def expand_one(self, mol):
        i = int(mol[1:])
        k = _h(self.seed, "nreact", i) % 4
        if k == 0 or i >= self.n - 1:
            return None
        reactants, scores, templates = [], [], []
        for r in range(k):
            a = min(self.n - 1, i + 1 + _h(self.seed, i, r, "a") % 9)
            b = min(self.n - 1, i + 1 + _h(self.seed, i, r, "b") % 9)
            reactants.append(f"m{a}" if _h(self.seed, i, r, "uni") % 3 == 0 else f"m{a}.m{b}")
            scores.append(0.05 + (_h(self.seed, i, r, "s") % 90) / 100.0)
            templates.append(f"T{i}_{r}")
        tot = sum(scores)
        return {"reactants": reactants, "scores": [s / tot for s in scores], "templates": templates, "analysis": [i]}

    def expand_fn(self, mol):
        self.expand_calls.append([mol])
        return self.expand_one(mol)

    def expand_batch_fn(self, mols):
        self.expand_calls.append(list(mols))
        return [self.expand_one(m) for m in mols]

    def value_one(self, mol):
        return 0.0 if mol in self.starting else 0.5 + (_h(self.seed, "v", mol) % 20) / 10.0

    def value_fn(self, mol, parent=None):
        self.value_calls.append([mol])
        return self.value_one(mol)

    def value_batch_fn(self, mols):
        self.value_calls.append(list(mols))
        return [self.value_one(m) for m in mols]


class _Node:
    def __init__(self, mol, value, known, parent):
        self.mol, self.value, self.known, self.parent = mol, value, known, parent
        self.children, self.open, self.succ = [], not known, known

    def v_target(self):
        return self.value


class StandInTree:
    """Minimal stand-in with MolTree's interface (greedy bookkeeping only, NOT Retro*'s value backup): enough to check the
    call pattern of the search loop on machines without the reference."""

    def __init__(self, target_mol, known_mols, value_fn):
        self.known, self.value_fn = known_mols, value_fn
        self.mol_nodes, self.succ, self.search_status = [], False, 0
        self.root = self._add(target_mol, None)
        self.root.succ_value = np.inf

    def _add(self, mol, parent):
        n = _Node(mol, self.value_fn(mol, parent), mol in self.known, parent)
        self.mol_nodes.append(n)
        return n

    def expand(self, node, reactant_lists, costs, templates, analysis):
        node.open = False
        if costs is None:
            return self.succ
        for mols, c in zip(reactant_lists, costs):
            kids = [self._add(m, node) for m in sorted(mols)]
            node.children.append(kids)
        self._update(self.root)
        self.succ = self.root.succ
        return self.succ

    def _update(self, n):
        if n.known:
            return True
        n.succ = any(all(self._update(k) for k in kids) for kids in n.children)
        return n.succ

    def get_best_route(self):
        return "route"


def _reference_loop(tree_cls, net, iterations):
    """planner/molstar.py:11-76 restated for the stand-in tree."""
    tree = tree_cls("m0", net.starting, net.value_fn)
    i = -1
    if not tree.succ:
        for i in range(iterations):
            scores = np.array([m.v_target() if m.open else np.inf for m in tree.mol_nodes])
            if np.min(scores) == np.inf:
                break
            tree.search_status = np.min(scores)
            m_next = tree.mol_nodes[int(np.argmin(scores))]
            result = net.expand_fn(m_next.mol)
            if result is not None and len(result["scores"]) > 0:
                costs = 0.0 - np.log(np.clip(np.array(result["scores"]), 1e-3, 1.0))
                lists = [list(set(r.split("."))) for r in result["reactants"]]
                if tree.expand(m_next, lists, costs, result["templates"], result["analysis"]):
                    break
                if tree.root.succ_value <= tree.search_status:
                    break
            else:
                tree.expand(m_next, None, None, None, None)
    return tree.succ, i + 1


@pytest.mark.parametrize("seed", range(8))
def test_call_pattern_on_a_stand_in_tree(seed):
    net_a, net_b, net_c = Network(seed), Network(seed), Network(seed)
    want = _reference_loop(StandInTree, net_a, 30)
    got = molstar_batched("m0", 0, net_b.starting, net_b.expand_batch_fn, net_b.value_batch_fn, iterations=30, beam=1, tree_factory=StandInTree)
    assert (got[0], got[2]) == want and [c[0] for c in net_b.expand_calls] == [c[0] for c in net_a.expand_calls]
    stats = {}
    molstar_batched("m0", 0, net_c.starting, net_c.expand_batch_fn, net_c.value_batch_fn, iterations=30, beam=5, tree_factory=StandInTree, stats=stats)
    assert all(1 <= len(c) <= 5 for c in net_c.expand_calls)
    assert stats["expanded"] <= sum(len(c) for c in net_c.expand_calls) <= 30      # a round that solves the target stops applying its batch
    flat = [m for c in net_c.value_calls for m in c]
    assert len(flat) == len(set(flat)), "every molecule is evaluated once"


def test_value_cache_and_predictor_adapter():
    calls = []
    vc = ValueCache(lambda ms: (calls.append(list(ms)), [float(len(m)) for m in ms])[1])
    vc.prefetch(["a", "bb", "a"])
    assert vc("a") == 1.0 and vc("bb") == 2.0 and vc("ccc") == 3.0 and calls == [["a", "bb"], ["ccc"]]

    class FakePredictor:
        def sample_templates_batch(self, graphs, c, smiles, topk=10):
            assert len(graphs) == len(smiles) == c.shape[0]
            return [([f"{s}.x"], [1.0], ["T"]) for s in smiles]

    expand = predictor_expand_batch_fn(FakePredictor(), graph_fn=lambda s: None if s == "bad" else object(),
                                       condition_fn=lambda ms: np.zeros((len(ms), 768)), topk=5)
    out = expand(["a", "bad", "b"])
    assert out[0]["reactants"] == ["a.x"] and out[1]["scores"] == [] and out[2]["templates"] == ["T"]
