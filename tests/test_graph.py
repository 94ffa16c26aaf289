"""Host graph tables vs the reference's getGraphDict (when present) and vs goldens."""
import os

import numpy as np
import pytest
import torch

from sgrl_b200 import graph as G, morphologies as M
from oracle import ref_loader
import parity


def test_morphology_inventory():
    assert len(M.CWHH) == 23 and len(M.ALL) == 27
    for name, par in M.ALL.items():
        assert par[0] == -1 and len(par) <= M.MAX_LIMBS
        assert int(name.split("_")[2]) == len(par)
        assert all(0 <= p < i for i, p in enumerate(par) if i > 0)


def test_hopper5_ranks():
    t = G.traversal_ranks([-1, 0, 1, 2, 3])
    assert t == [[0, 1, 2, 3, 4], [4, 3, 2, 1, 0], [4, 3, 2, 1, 0]]


def test_relation_against_golden():
    gold = parity.load_golden()
    for name, _ in parity.CASES:
        g = G.build_graph(M.ALL[name])
        np.testing.assert_array_equal(torch.stack(g["traversals"]).numpy(), gold[name + "/traversals"])
        np.testing.assert_allclose(g["relation"].numpy(), gold[name + "/relation"], rtol=0, atol=2e-6)
        assert g["relation"].shape == (len(M.ALL[name]),) * 2 + (3,)


def test_graph_tables_against_pins():
    """Every morphology's tables vs tests/golden/pins.npz.  Those were recorded from build_graph itself
    (tests/golden/make_pins.py), not from the reference: they pin the 22 morphologies set_golden.npz does not hold, and the
    single-limb case, where the reference is not available to compare with."""
    pins = np.load(os.path.join(os.path.dirname(parity.GOLDEN), "pins.npz"))
    for name, par in M.ALL.items():
        g = G.build_graph(par)
        np.testing.assert_array_equal(torch.stack(g["traversals"]).numpy(), pins[f"graph/{name}/traversals"], err_msg=name)
        np.testing.assert_allclose(g["relation"].numpy(), pins[f"graph/{name}/relation"], rtol=0, atol=2e-6, err_msg=name)
    assert G.build_graph([-1]) == {"parents": [-1]}


@pytest.mark.skipif(ref_loader.find_reference() is None, reason="reference not on this machine")
def test_graph_against_reference():
    ref = ref_loader.load_reference()
    for name, par in M.ALL.items():
        want = ref.utils.getGraphDict(par, ["pre", "inlcrs", "postlcrs"], device=torch.device("cpu"))
        got = G.build_graph(par)
        for a, b in zip(want["traversals"], got["traversals"]):
            assert torch.equal(a, b), name
        assert torch.equal(want["relation"], got["relation"]), name
    assert G.build_graph([-1]) == {"parents": [-1]}


def test_packed_tables_invariants():
    """Host tables of a packed mixed-morphology batch (SURVEY.md §8f rank 1): ragged graph offsets, per-graph relation
    offsets, loss weights = mean over morphologies of the per-morphology mean, staging rows sized by the largest graph."""
    from sgrl_b200.modules import make_packed_tables, make_tables
    names = ["3d_hopper_3_shin", "3d_humanoid_9_full", "3d_walker_7_full"]
    batches = [4, 2, 3]
    parts = [(G.build_graph(M.ALL[n]), b) for n, b in zip(names, batches)]
    tb = make_packed_tables(parts, "cpu")
    ns = [len(M.ALL[n]) for n in names]
    assert tb.G == sum(batches) and tb.T == sum(b * n for b, n in zip(batches, ns)) and tb.nmax == max(ns)
    cu = tb.cu_limbs.tolist()
    assert cu[0] == 0 and cu[-1] == tb.T and [b - a for a, b in zip(cu, cu[1:])] == [n for b, n in zip(batches, ns) for _ in range(b)]
    assert abs(float(tb.tok_weight.sum()) - 1.0) < 1e-6
    t0 = g0 = ro = 0
    for (graph, b), n, span in zip(parts, ns, tb.parts):
        assert span == (t0, t0 + b * n, g0, g0 + b, n)
        assert tb.rel_off[g0:g0 + b].tolist() == [ro] * b
        assert torch.equal(tb.relation[ro:ro + n * n * 3].view(n, n, 3), graph["relation"])
        one = make_tables(graph, b, "cpu")
        assert torch.equal(tb.rank3[t0:t0 + b * n], one.rank3)
        assert torch.equal(tb.tok_graph[t0:t0 + b * n], one.tok_graph + g0)
        np.testing.assert_allclose(tb.tok_weight[t0:t0 + b * n].numpy(), 1.0 / (len(parts) * b * n), rtol=1e-6)
        t0 += b * n; g0 += b; ro += n * n * 3
    single = make_tables(parts[1][0], 5, "cpu")
    assert single.nmax == 9 and single.tok_weight is None and single.parts == [(0, 45, 0, 5, 9)]
    with pytest.raises(ValueError, match="single-limb"):
        make_tables(G.build_graph([-1]), 1, "cpu")
