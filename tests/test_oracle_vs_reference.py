"""The oracle against the reference's own classes and its create_graph, through what the reference produced and the
fixtures under tests/golden/ keep (tests/golden/make_golden.py ran the reference's ODEfunc / ODEBlock and create_graph):
its default initialisation under a seed, its fp32 rollout outputs BIT FOR BIT, and the adjacency of every shipped graph."""
import os
import pickle

import networkx as nx
import numpy as np
import pytest
import scipy.sparse
import torch

from oracle import gnode_oracle as orc
from _util import GOLDEN_DIR, Golden, golden_threads

# graph, trials, torch seed of the reference's model construction (tests/golden/make_golden.py CASES)
SIM_CASES = [("karate", 1, 0), ("karate", 8, 1), ("dolphins", 4, 2), ("fb-food", 2, 3)]


def check_golden_bit_exact(g, seed):
    """The reference's state_dict is its default init under `seed`, and the oracle's fp32 rollout with it is bitwise the
    reference's outputs."""
    params = orc.default_params(g.H, seed)
    assert list(params) == list(g.params)
    assert all(torch.equal(v, g.params[k]) for k, v in params.items())
    got = orc.forward(g.x, params, orc.batch_coo(g.adjs, g.inst_graph), orc.time_grid(g.maxTime, g.deltaT))
    assert torch.equal(got[:: g.tstride], g.probs32)


@pytest.fixture(autouse=True)
def fixture_thread_count():
    with golden_threads():
        yield


@pytest.mark.parametrize("graph,B,seed", SIM_CASES)
def test_sim_variant_bit_exact(graph, B, seed):
    g = Golden("sim_%s_b%d" % (graph.replace("-", ""), B))
    assert g.variant == "sim" and len(g.inst_graph) == B
    check_golden_bit_exact(g, seed)


def test_ngraphs_variant_bit_exact():
    g = Golden("ng_mixed_b5")
    assert g.variant == "ngraphs" and len(g.adjs) > 1
    check_golden_bit_exact(g, 5)


# largest connected component of the reference's real_graphs/<name>.pkl as its create_graph builds it
GRAPH_CSR = {"karate": "sim_karate_b1", "dolphins": "sim_dolphins_b4", "fb-food": "sim_fbfood_b2",
             "fb-social": "sim_fbsocial_b1", "openflights": "sim_openflights_b2", "wiki-vote": "sim_wikivote_b2",
             "enron": "graphs/enron"}


def stored_csr(name):
    z = np.load(os.path.join(GOLDEN_DIR, GRAPH_CSR[name] + ".npz"))
    indptr, indices = (z["indptr"], z["indices"]) if "indptr" in z else (z["g0_indptr"], z["g0_indices"])
    n = len(indptr) - 1
    return scipy.sparse.csr_matrix((np.ones(len(indices), dtype=np.int64), indices, indptr), shape=(n, n))


def reference_create_graph(path):
    """ode_nn.py:394-414: pickle -> to_undirected -> subgraph of the largest connected component -> adjacency_matrix."""
    with open(path, "rb") as fh:
        G = pickle.load(fh)
    G = G.to_undirected()
    G = G.subgraph(max(nx.connected_components(G), key=len))
    return nx.adjacency_matrix(G)


@pytest.mark.parametrize("name", ["karate", "dolphins", "fb-food", "fb-social", "openflights", "wiki-vote", "enron"])
def test_cached_graph_pipeline_equals_reference_create_graph(name, tmp_path, monkeypatch):
    """N2: pickle -> largest component -> CSR without networkx's adjacency_matrix, and its on-disk cache, give exactly the
    matrix the reference's create_graph builds (ode_nn.py:394-414), for every shipped graph. The pickle is a directed
    graph holding each edge once, with a smaller component whose nodes come first, around the stored component."""
    import gn_ode_sir_b200  # noqa: F401
    from gn_ode_sir_b200 import harness
    want = stored_csr(name)
    want.sort_indices()
    n = want.shape[0]
    G = nx.DiGraph()
    G.add_edges_from([(n, n + 1), (n + 1, n + 2)])
    G.add_nodes_from(range(n))
    coo = scipy.sparse.triu(want).tocoo()
    G.add_edges_from(zip(coo.row.tolist(), coo.col.tolist()))
    (tmp_path / "real_graphs").mkdir()
    label = str(tmp_path / "real_graphs" / name)
    with open(label + ".pkl", "wb") as fh:
        pickle.dump(G, fh)
    ref = reference_create_graph(label + ".pkl").tocsr()
    ref.sort_indices()
    assert ref.shape == want.shape and np.array_equal(ref.indptr, want.indptr) and np.array_equal(ref.indices, want.indices)
    cache = tmp_path / "cache"
    monkeypatch.setenv("GNODE_GRAPH_CACHE", str(cache))
    for attempt in ("built", "cached"):
        G2, A = harness.load_graph(label)
        assert A.shape == want.shape and np.array_equal(A.indptr, want.indptr) and np.array_equal(A.indices, want.indices), attempt
        assert G2.number_of_nodes() == n
    assert len(list(cache.iterdir())) == 1                          # the second load came from the cache file
